"""oracle/pygaussian.py -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

ctypes bindings for oracle/gaussian_oracle.c, the plain-C restatement of the reference's CPU Gaussian blur (window and separable
reflect-101 convolution) that the fn.gaussian_blur tests and tools/bench_gaussian_blur.py --check compare with.  The library is
compiled on first use into a private temporary directory (the source tree may be read-only), with oracle/Makefile's flags.
"""
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "gaussian_oracle.c")
_lib = None


def lib():
    global _lib
    if _lib is None:
        d = tempfile.mkdtemp(prefix="dali_b200_gaussian_oracle_")
        try:
            so = os.path.join(d, "libgaussian_oracle.so")
            subprocess.check_call([os.environ.get("CC", "gcc"), "-O2", "-fPIC", "-ffp-contract=off", "-Wall", "-Wno-unused-function",
                                   "-shared", "-o", so, _SRC, "-lm"])
            _lib = C.CDLL(so)          # the mapping outlives the file
        finally:
            shutil.rmtree(d, ignore_errors=True)
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


# ------------------------------------------------------------------------------------------- Gaussian blur
def gaussian_params(sigma, window_size):
    """(sigma, diameter) of one axis after GaussianBlurParams' rules (gaussian_blur_params.h): window = 2 * ceil(3 sigma) + 1 when
    only sigma is given (3 * sigma in float), sigma = (radius - 1) * 0.3 + 0.8 when only the window is given."""
    sigma, window_size = np.float32(sigma), int(window_size)
    if window_size == 0:
        window_size = 2 * int(np.ceil(np.float32(3) * sigma)) + 1
    if sigma == 0:
        sigma = np.float32(((window_size - 1) // 2 - 1) * 0.3 + 0.8)
    return float(sigma), window_size


def gaussian_window(sigma, diameter):
    w = np.empty(int(diameter), np.float32)
    lib().oracle_gaussian_window(C.c_float(sigma), int(diameter), _p(w))
    return w


def sepconv(x, windows, out_dtype=None, channels=True):
    """Separable reflect-101 convolution of one HW(C) image or DHW(C) volume with per-axis windows (outermost axis first)."""
    x = np.ascontiguousarray(x)
    if not channels:
        x = x[..., None]
    nd = x.ndim - 1
    assert nd in (2, 3) and len(windows) == nd and x.dtype in (np.uint8, np.float32)
    out_dtype = np.dtype(out_dtype or x.dtype)
    out = np.empty(x.shape, out_dtype)
    shape = (C.c_int * 3)(*x.shape[:nd])
    diam = (C.c_int * 3)(*[len(w) for w in windows])
    wcat = np.ascontiguousarray(np.concatenate([np.asarray(w, np.float32) for w in windows]))
    rc = lib().oracle_sepconv(_p(x), 0 if x.dtype == np.uint8 else 1, nd, shape, int(x.shape[-1]), diam, _p(wcat), _p(out),
                              0 if out_dtype == np.uint8 else 1)
    if rc != 0:
        raise RuntimeError(f"sepconv rc={rc}")
    return out if channels else out[..., 0]


def gaussian_blur(x, sigma=0.0, window_size=0, out_dtype=None, channels=True):
    """fn.gaussian_blur of one HW(C) / DHW(C) sample; sigma / window_size: scalar or one value per spatial axis (outermost first)."""
    nd = x.ndim - (1 if channels else 0)
    sig = np.broadcast_to(np.asarray(sigma, np.float32), (nd,))
    ws = np.broadcast_to(np.asarray(window_size), (nd,))
    wins = [gaussian_window(*gaussian_params(s, w)) for s, w in zip(sig, ws)]
    return sepconv(x, wins, out_dtype, channels)

"""ctypes view of the C-ABI in include/dali_b200.h (libdali_b200.so).

This is the binding a maintainer of a Python host would add (see INTEGRATION.md); the C++ operators in
dali_b200/host link the same symbols directly.  Device memory is owned by the caller (torch tensors);
nothing here computes on the CPU -- if the CUDA library is missing the import of `lib()` raises.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libdali_b200.so")

UINT8, INT16, FLOAT16, FLOAT = 0, 5, 8, 9
RGB, BGR, GRAY, YCbCr = 0, 1, 2, 3
FILTER_NN, FILTER_LINEAR, FILTER_TRIANGULAR, FILTER_GAUSSIAN, FILTER_CUBIC, FILTER_LANCZOS3 = range(6)
LAYOUT_HWC, LAYOUT_CHW = 0, 1

EXPORTS = [
    "dalib200GetLastError", "dalib200GetVersion", "dalib200GetLaunchCount", "dalib200ProfilingEnable", "dalib200ProfilingCollect",
    "dalib200JpegGetInfo", "dalib200JpegPlanCreate", "dalib200JpegPlanDestroy", "dalib200JpegPlanSetup",
    "dalib200JpegPlanGetInfo", "dalib200JpegPlanStagedBytes", "dalib200JpegUpload", "dalib200JpegLaunch",
    "dalib200JpegGetStatus", "dalib200JpegDebugGetCoefficients", "dalib200JpegPlanSetupEx", "dalib200JpegPlanGetOutputShape",
    "dalib200JpegStatusAsync", "dalib200JpegStatusFetch", "dalib200JpegPlanGetPlanes", "dalib200JpegPlanSetPlanesOnly",
    "dalib200JpegPlanSetSourceStable", "dalib200JpegPlanLastUploadDirect", "dalib200HostAlloc", "dalib200HostAllocOnDevice", "dalib200HostFree", "dalib200DebugCheckHalfConversion",
    "dalib200ResamplePlanSetupPlanar", "dalib200ResampleLaunchPlanar",
    "dalib200ResamplePlanCreate", "dalib200ResamplePlanDestroy", "dalib200ResamplePlanSetup", "dalib200ResampleLaunch",
    "dalib200ResamplePlanGetOrder",
    "dalib200ResamplePlanGetPath",
    "dalib200Resample3DPlanCreate", "dalib200Resample3DPlanDestroy", "dalib200Resample3DPlanSetup", "dalib200Resample3DLaunch",
    "dalib200Resample3DPlanGetOrder",
    "dalib200CmnPlanCreate", "dalib200CmnPlanDestroy", "dalib200CmnPlanSetup", "dalib200CmnLaunch",
    "dalib200WarpPlanCreate", "dalib200WarpPlanDestroy", "dalib200WarpPlanSetup", "dalib200WarpLaunch", "dalib200WarpPlanGetPath", "dalib200AffineInverse",
    "dalib200PointwisePlanCreate", "dalib200PointwisePlanDestroy", "dalib200LinearTransformSetup", "dalib200ColorSpaceSetup",
    "dalib200PointwiseLaunch", "dalib200ColorTwistMatrix",
    "dalib200SpectrogramPlanCreate", "dalib200SpectrogramPlanDestroy", "dalib200SpectrogramPlanSetup",
    "dalib200SpectrogramNumWindows", "dalib200SpectrogramLaunch", "dalib200HannWindow",
    "dalib200SignalPlanCreate", "dalib200SignalPlanDestroy", "dalib200ToDecibelsSetup", "dalib200MfccSetup", "dalib200SignalOutputRows",
    "dalib200NormalizeSetup", "dalib200SignalLaunch", "dalib200NonsilentSetup", "dalib200NonsilentLaunch", "dalib200AudioResampleSetup",
    "dalib200GenericPlanCreate", "dalib200GenericPlanDestroy", "dalib200MultiplyAddSetup", "dalib200WindowCopySetup", "dalib200GenericLaunch",
    "dalib200MelPlanCreate", "dalib200MelPlanDestroy", "dalib200MelPlanSetup", "dalib200MelLaunch", "dalib200MelPlanSetTensorCores",
    "dalib200SpectrogramMelSupported", "dalib200SpectrogramMelLaunch",
    "dalib200SepConvPlanCreate", "dalib200SepConvPlanDestroy", "dalib200SepConvPlanSetup", "dalib200SepConvLaunch",
    "dalib200SepConvPlanGetPath", "dalib200GaussianWindow",
]


class JpegInfo(C.Structure):
    _fields_ = [("width", C.c_int32), ("height", C.c_int32), ("components", C.c_int32), ("subsampling", C.c_int32),
                ("restart_interval", C.c_int32), ("orientation", C.c_int32)]


class JpegParams(C.Structure):
    _fields_ = [("output_type", C.c_int32), ("fancy_upsampling", C.c_int32), ("dtype", C.c_int32), ("adjust_orientation", C.c_int32)]


class JpegRoi(C.Structure):
    _fields_ = [("use_roi", C.c_int32), ("x0", C.c_int32), ("y0", C.c_int32), ("x1", C.c_int32), ("y1", C.c_int32), ("planes_only", C.c_int32)]


class PlanarImage(C.Structure):
    _fields_ = [("y", C.c_void_p), ("cb", C.c_void_p), ("cr", C.c_void_p), ("pitch_y", C.c_int32), ("pitch_c", C.c_int32),
                ("width", C.c_int32), ("height", C.c_int32), ("crop_x", C.c_int32), ("crop_y", C.c_int32)]


class FilterDesc(C.Structure):
    _fields_ = [("type", C.c_int32), ("antialias", C.c_int32), ("radius", C.c_float)]


class ResampleSample(C.Structure):
    _fields_ = [("in_h", C.c_int32), ("in_w", C.c_int32), ("channels", C.c_int32), ("out_h", C.c_int32), ("out_w", C.c_int32),
                ("use_roi", C.c_int32 * 2), ("roi_start", C.c_float * 2), ("roi_end", C.c_float * 2),
                ("min_filter", FilterDesc * 2), ("mag_filter", FilterDesc * 2)]


class Resample3DSample(C.Structure):
    _fields_ = [("in_shape", C.c_int32 * 3), ("channels", C.c_int32), ("out_shape", C.c_int32 * 3),
                ("use_roi", C.c_int32 * 3), ("roi_start", C.c_float * 3), ("roi_end", C.c_float * 3),
                ("min_filter", FilterDesc * 3), ("mag_filter", FilterDesc * 3)]


class SepConvSample(C.Structure):
    _fields_ = [("ndim", C.c_int32), ("shape", C.c_int32 * 3), ("channels", C.c_int32), ("diameter", C.c_int32 * 3),
                ("window_offset", C.c_int32 * 3)]


class CmnSample(C.Structure):
    _fields_ = [("in_h", C.c_int32), ("in_w", C.c_int32), ("channels", C.c_int32),
                ("anchor_y", C.c_int32), ("anchor_x", C.c_int32), ("crop_h", C.c_int32), ("crop_w", C.c_int32),
                ("mirror", C.c_int32), ("mean", C.c_float * 4), ("inv_std", C.c_float * 4), ("fill", C.c_float * 4)]


class WarpSample(C.Structure):
    _fields_ = [("in_h", C.c_int32), ("in_w", C.c_int32), ("channels", C.c_int32), ("out_h", C.c_int32), ("out_w", C.c_int32),
                ("matrix", C.c_float * 6)]


class ColorSample(C.Structure):
    _fields_ = [("num_pixels", C.c_int64), ("matrix", C.c_float * 9), ("offset", C.c_float * 3)]


class SpectrogramArgs(C.Structure):
    _fields_ = [("nfft", C.c_int32), ("window_length", C.c_int32), ("window_step", C.c_int32), ("power", C.c_int32),
                ("center", C.c_int32), ("reflect", C.c_int32), ("layout_ft", C.c_int32)]


class MelArgs(C.Structure):
    _fields_ = [("nfilter", C.c_int32), ("sample_rate", C.c_float), ("freq_low", C.c_float), ("freq_high", C.c_float),
                ("htk", C.c_int32), ("normalize", C.c_int32)]


class ToDecibelsArgs(C.Structure):
    _fields_ = [("multiplier", C.c_float), ("reference", C.c_float), ("cutoff_db", C.c_float), ("ref_max", C.c_int32)]


class MfccArgs(C.Structure):
    _fields_ = [("n_mfcc", C.c_int32), ("dct_type", C.c_int32), ("normalize", C.c_int32), ("lifter", C.c_float)]


class NormalizeArgs(C.Structure):
    _fields_ = [("mode", C.c_int32), ("ddof", C.c_int32), ("scale", C.c_float), ("shift", C.c_float), ("epsilon", C.c_float)]


class DaliB200Error(RuntimeError):
    pass


_lib = None


def lib():
    """Loads libdali_b200.so; raises (never falls back) when it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise DaliB200Error(f"{LIB_PATH} is missing: run `python -m dali_b200.build` (there is no CPU fallback)")
        _lib = C.CDLL(os.environ.get("DALIB200_LIB", LIB_PATH))      # override: A/B experiments with an older build
        _lib.dalib200GetLastError.restype = C.c_char_p
        _lib.dalib200GetLaunchCount.restype = C.c_uint64
        _lib.dalib200JpegPlanStagedBytes.restype = C.c_size_t
        _lib.dalib200SpectrogramNumWindows.restype = C.c_int64
        _lib.dalib200GaussianWindow.restype = None
        _lib.dalib200GaussianWindow.argtypes = [C.c_float, C.c_int, C.c_void_p]
        _lib.dalib200SepConvPlanSetup.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_int]
    return _lib


class _PinnedBlock:
    def __init__(self, nbytes, device=None):
        p = C.c_void_p()
        if device is None:
            check(lib().dalib200HostAlloc(C.byref(p), C.c_size_t(nbytes)))
        else:
            check(lib().dalib200HostAllocOnDevice(C.byref(p), C.c_size_t(nbytes), int(device)))
        self.ptr, self.nbytes = p.value, nbytes

    def __del__(self):
        try:
            lib().dalib200HostFree(C.c_void_p(self.ptr))
        except Exception:
            pass


def pinned_empty(nbytes, device=None):
    """uint8 numpy array over page-locked host memory (freed with the last view).  Encoded streams held in such memory and fed
    with external_source(no_copy=True) reach the decoder by DMA straight from here (dalib200JpegPlanSetSourceStable).
    device: allocate with that GPU current (for threads whose current device differs, e.g. a reader's read-ahead thread)."""
    import numpy as np
    nbytes = max(1, int(nbytes))
    blk = _PinnedBlock(nbytes, device)
    buf = (C.c_uint8 * nbytes).from_address(blk.ptr)
    buf._blk = blk                      # the numpy array keeps `buf` (its base) alive, `buf` keeps the allocation
    return np.frombuffer(buf, dtype=np.uint8)


def check(rc):
    if rc != 0:
        raise DaliB200Error(lib().dalib200GetLastError().decode("utf-8", "replace") + f" (status {rc})")


def profiling(on):
    check(lib().dalib200ProfilingEnable(int(bool(on))))


def profiling_collect(max_records=65536):
    """[(kernel name, ms)] of every launch since the last collect (device-timed with CUDA events)."""
    names = C.create_string_buffer(max_records * 32)
    ms = (C.c_float * max_records)()
    cnt = C.c_int(0)
    check(lib().dalib200ProfilingCollect(names, 32, ms, max_records, C.byref(cnt)))
    raw = names.raw
    return [(raw[i * 32:(i + 1) * 32].split(b"\0", 1)[0].decode(), float(ms[i])) for i in range(cnt.value)]


def launch_count():
    return int(lib().dalib200GetLaunchCount())


def ptr_array(tensors):
    """void*[] from a list of torch CUDA tensors (or raw ints)."""
    arr = (C.c_void_p * len(tensors))()
    for i, t in enumerate(tensors):
        arr[i] = t if isinstance(t, int) else t.data_ptr()
    return arr


def stream_handle(stream=None):
    import torch
    s = stream if stream is not None else torch.cuda.current_stream()
    return C.c_void_p(s.cuda_stream)


def make_filter(f):
    if isinstance(f, FilterDesc):
        return f
    if isinstance(f, int):
        return FilterDesc(f, 1, 0.0)
    return FilterDesc(int(f[0]), int(f[1]), float(f[2]))


class Plan:
    """RAII holder for a C-ABI plan."""

    def __init__(self, kind, max_batch):
        self._destroy = getattr(lib(), f"dalib200{kind}PlanDestroy")
        self.handle = C.c_void_p()
        check(getattr(lib(), f"dalib200{kind}PlanCreate")(C.byref(self.handle), int(max_batch)))

    def __del__(self):
        try:
            if self.handle:
                self._destroy(self.handle)
                self.handle = C.c_void_p()
        except Exception:
            pass


def np_f32(x, n):
    a = np.zeros(n, np.float32)
    if x is not None:
        x = np.atleast_1d(np.asarray(x, np.float32))
        a[: x.size] = x
        if x.size == 1:
            a[:] = x[0]
    return a

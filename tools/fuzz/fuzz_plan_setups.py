"""Host-side fuzzer of every ...PlanSetup entry point of include/dali_b200.h (see run_setups.sh):
    python fuzz_plan_setups.py <seed> <iterations>      with DALIB200_LIB = the sanitizer build of the library.
Arguments are drawn from plausible values mixed with adversarial ones (zero / negative / huge sizes, windows outside the image, NaN and
infinite floats, invalid enum codes).  Every call must return a status (success or an argument error); a finding is a sanitizer report."""
import ctypes as C
import os
import sys

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", ".."))
from dali_b200 import capi  # noqa: E402

rng = np.random.default_rng(int(sys.argv[1]) if len(sys.argv) > 1 else 0)
N = int(sys.argv[2]) if len(sys.argv) > 2 else 2000
L = capi.lib()
MILD = float(os.environ.get("FUZZ_BAD_SCALE", "1"))      # < 1: fewer adversarial values per call -> more set-ups reach their deep paths
BAD_F = [0.0, -0.0, 1.0, -1.0, 1e-30, 1e30, -1e30, float("nan"), float("inf"), float("-inf"), 0.5, 255.0, 3.4e38]
BAD_I = [0, 1, -1, 2, 3, 7, 8, 16, 17, 255, 256, 4095, 4096, 65535, 65536, 2 ** 31 - 1, -2 ** 31, 10 ** 6]


def dim(lo=1, hi=3000):
    return int(rng.choice(BAD_I)) if rng.random() < 0.08 * MILD else int(rng.integers(lo, hi))


def small(lo, hi):
    return int(rng.choice(BAD_I)) if rng.random() < 0.1 * MILD else int(rng.integers(lo, hi))


def flt(lo=-10.0, hi=10.0):
    return float(rng.choice(BAD_F)) if rng.random() < 0.15 * MILD else float(rng.uniform(lo, hi))


def code(valid):
    return int(rng.choice(BAD_I)) if rng.random() < 0.1 * MILD else int(rng.choice(valid))


def plan(kind, n):
    return capi.Plan(kind, n)


hist = {}


def fake_ptrs(m, base):
    """Device pointers are never dereferenced on the host: aligned fake addresses (sometimes misaligned ones) are enough."""
    return (C.c_void_p * m)(*[base + 0x1000000 * (i + 1) + (int(rng.integers(1, 16)) if rng.random() < 0.1 * MILD else 0) for i in range(m)])


def launch(name, fn, *args):
    """Launch-side host code (descriptor build, arena growth, path selection); the kernels themselves are stubbed out."""
    note(name + "_launch", fn(*args))


TRACE = os.environ.get("FUZZ_TRACE")


def note(name, rc):
    if TRACE:
        print(name, rc, file=sys.stderr, flush=True)
    hist[(name, "ok" if rc == 0 else "err")] = hist.get((name, "ok" if rc == 0 else "err"), 0) + 1


plans = {k: plan(k, 8) for k in ("Resample", "Resample3D", "Cmn", "Warp", "Pointwise", "Spectrogram", "Mel", "Signal", "Generic", "SepConv")}
for it in range(N):
    n = int(rng.integers(0, 9)) if rng.random() < 0.9 else int(rng.choice([9, 100, -1]))
    m = max(n, 1) if n < 64 else 8
    # ---- resample
    S = (capi.ResampleSample * m)()
    for s in S:
        s.in_h, s.in_w, s.channels, s.out_h, s.out_w = dim(), dim(), small(1, 5), dim(0, 600), dim(0, 600)
        for d in range(2):
            s.use_roi[d] = int(rng.integers(0, 2))
            s.roi_start[d], s.roi_end[d] = flt(-50, 3000), flt(-50, 3000)
            s.min_filter[d] = capi.FilterDesc(code(range(6)), int(rng.integers(0, 2)), flt(0, 8))
            s.mag_filter[d] = capi.FilterDesc(code(range(6)), int(rng.integers(0, 2)), flt(0, 8))
    rc = L.dalib200ResamplePlanSetup(plans["Resample"].handle, n, S, code([0, 9]), code([0, 9]))
    note("resample", rc)
    if rc == 0:
        launch("resample", L.dalib200ResampleLaunch, plans["Resample"].handle, fake_ptrs(m, 0x10000000), fake_ptrs(m, 0x7000000000), None)
        for i in range(max(0, min(n, m))):
            L.dalib200ResamplePlanGetOrder(plans["Resample"].handle, i), L.dalib200ResamplePlanGetPath(plans["Resample"].handle, i)
    ok = (C.c_uint8 * m)()
    rc = L.dalib200ResamplePlanSetupPlanar(plans["Resample"].handle, n, S, ok)
    note("resample_planar", rc)
    if rc == 0:
        PI = (capi.PlanarImage * m)()
        for i, q in enumerate(PI):
            q.y, q.cb, q.cr = 0x20000000 + 0x1000000 * i, 0x40000000 + 0x1000000 * i, 0x60000000 + 0x1000000 * i
            q.pitch_y, q.pitch_c = int(rng.choice([16, 64, 1920, 1936, 17])), int(rng.choice([16, 64, 960, 976, 9]))
            q.width, q.height, q.crop_x, q.crop_y = dim(), dim(), small(0, 64), small(0, 64)
        launch("resample_planar", L.dalib200ResampleLaunchPlanar, plans["Resample"].handle, PI, fake_ptrs(m, 0x7000000000), None)
    # ---- resample (volumes)
    V = (capi.Resample3DSample * m)()
    for s in V:
        s.channels = small(1, 5)
        for d in range(3):
            s.in_shape[d], s.out_shape[d] = dim(1, 200), dim(0, 120)
            s.use_roi[d] = int(rng.integers(0, 2))
            s.roi_start[d], s.roi_end[d] = flt(-50, 300), flt(-50, 300)
            s.min_filter[d] = capi.FilterDesc(code(range(6)), int(rng.integers(0, 2)), flt(0, 8))
            s.mag_filter[d] = capi.FilterDesc(code(range(6)), int(rng.integers(0, 2)), flt(0, 8))
    rc = L.dalib200Resample3DPlanSetup(plans["Resample3D"].handle, n, V, code([0, 9]), code([0, 9]))
    note("resample3d", rc)
    if rc == 0:
        launch("resample3d", L.dalib200Resample3DLaunch, plans["Resample3D"].handle, fake_ptrs(m, 0x10000000), fake_ptrs(m, 0x7000000000), None)
        o3 = (C.c_int32 * 3)()
        for i in range(max(0, min(n, m))):
            L.dalib200Resample3DPlanGetOrder(plans["Resample3D"].handle, i, o3)
    # ---- cmn
    Cs = (capi.CmnSample * m)()
    for s in Cs:
        s.in_h, s.in_w, s.channels = dim(), dim(), small(1, 5)
        s.anchor_y, s.anchor_x, s.crop_h, s.crop_w, s.mirror = small(-50, 3000), small(-50, 3000), dim(0, 600), dim(0, 600), int(rng.integers(0, 2))
        for k in range(4):
            s.mean[k], s.inv_std[k], s.fill[k] = flt(0, 255), flt(0, 1), flt(0, 255)
    rc = L.dalib200CmnPlanSetup(plans["Cmn"].handle, n, Cs, code([9, 8, 0]), code([0, 1]), small(1, 5))
    note("cmn", rc)
    if rc == 0:
        launch("cmn", L.dalib200CmnLaunch, plans["Cmn"].handle, fake_ptrs(m, 0x10000000), fake_ptrs(m, 0x7000000000), None)
    # ---- warp
    W = (capi.WarpSample * m)()
    for s in W:
        s.in_h, s.in_w, s.channels, s.out_h, s.out_w = dim(), dim(), small(1, 5), dim(0, 600), dim(0, 600)
        for k in range(6):
            s.matrix[k] = flt(-3, 3)
    rc = L.dalib200WarpPlanSetup(plans["Warp"].handle, n, W, code([0, 1]), int(rng.integers(0, 2)), C.c_float(flt(0, 255)), code([0, 9]))
    note("warp", rc)
    if rc == 0:
        launch("warp", L.dalib200WarpLaunch, plans["Warp"].handle, fake_ptrs(m, 0x10000000), fake_ptrs(m, 0x7000000000), None)
        L.dalib200WarpPlanGetPath(plans["Warp"].handle)
    # ---- pointwise
    P = (capi.ColorSample * m)()
    for s in P:
        s.num_pixels = int(rng.choice([0, -1, 1, 2 ** 40, 2 ** 62])) if rng.random() < 0.1 else int(rng.integers(0, 10 ** 7))
        for k in range(9):
            s.matrix[k] = flt(-2, 2)
        for k in range(3):
            s.offset[k] = flt(-128, 128)
    rc = L.dalib200LinearTransformSetup(plans["Pointwise"].handle, n, P, code([0, 9]))
    note("linear", rc)
    if rc == 0:
        launch("linear", L.dalib200PointwiseLaunch, plans["Pointwise"].handle, fake_ptrs(m, 0x10000000), fake_ptrs(m, 0x7000000000), None)
    npx = (C.c_int64 * m)(*[int(rng.choice([0, -1, 2 ** 40])) if rng.random() < 0.1 else int(rng.integers(0, 10 ** 7)) for _ in range(m)])
    rc = L.dalib200ColorSpaceSetup(plans["Pointwise"].handle, n, npx, code(range(4)), code(range(4)))
    note("csc", rc)
    if rc == 0:
        launch("csc", L.dalib200PointwiseLaunch, plans["Pointwise"].handle, fake_ptrs(m, 0x10000000), fake_ptrs(m, 0x7000000000), None)
    # ---- spectrogram / mel
    a = capi.SpectrogramArgs(code([64, 128, 256, 400, 512, 1000, 1024, 2048, 4096, 8192]), code([16, 64, 400, 512, 1024, 5000]), code([1, 64, 160, 256]),
                             code([1, 2]), int(rng.integers(0, 2)), int(rng.integers(0, 2)), int(rng.integers(0, 2)))
    win = None
    if rng.random() < 0.3 and 0 < a.window_length < 100000:
        win = np.ascontiguousarray(rng.uniform(0, 1, a.window_length), np.float32)
    lens = (C.c_int64 * m)(*[int(rng.choice([0, 1, -1, 2 ** 40])) if rng.random() < 0.1 else int(rng.integers(0, 200000)) for _ in range(m)])
    rc = L.dalib200SpectrogramPlanSetup(plans["Spectrogram"].handle, C.byref(a), None if win is None else win.ctypes.data_as(C.c_void_p), n, lens)
    note("spectrogram", rc)
    if rc == 0:
        launch("spectrogram", L.dalib200SpectrogramLaunch, plans["Spectrogram"].handle, fake_ptrs(m, 0x10000000), fake_ptrs(m, 0x7000000000), None)
        for i in range(max(0, min(n, m))):
            L.dalib200SpectrogramNumWindows(plans["Spectrogram"].handle, i)
    ma = capi.MelArgs(code([1, 40, 80, 128, 1000]), C.c_float(flt(8000, 48000)), C.c_float(flt(0, 4000)), C.c_float(flt(0, 24000)), int(rng.integers(0, 2)),
                      int(rng.integers(0, 2)))
    nwin = (C.c_int64 * m)(*[int(rng.choice([0, -1, 2 ** 40])) if rng.random() < 0.1 else int(rng.integers(0, 2000)) for _ in range(m)])
    rc2 = L.dalib200MelPlanSetup(plans["Mel"].handle, C.byref(ma), code([1, 33, 129, 257, 513, 1025]), n, nwin)
    note("mel", rc2)
    if rc2 == 0:
        L.dalib200MelPlanSetTensorCores(plans["Mel"].handle, int(rng.integers(0, 2)))
        launch("mel", L.dalib200MelLaunch, plans["Mel"].handle, fake_ptrs(m, 0x10000000), fake_ptrs(m, 0x7000000000), None)
    if rc == 0 and rc2 == 0:
        if L.dalib200SpectrogramMelSupported(plans["Spectrogram"].handle, plans["Mel"].handle) == 1:
            launch("spectrogram_mel", L.dalib200SpectrogramMelLaunch, plans["Spectrogram"].handle, plans["Mel"].handle, fake_ptrs(m, 0x10000000),
                   fake_ptrs(m, 0x5000000000) if rng.random() < 0.5 else None, fake_ptrs(m, 0x7000000000), None)
    # ---- signal tail
    db = capi.ToDecibelsArgs(C.c_float(flt(1, 20)), C.c_float(flt(0, 2)), C.c_float(flt(-200, 0)), int(rng.integers(0, 2)))
    vol = (C.c_int64 * m)(*[int(rng.choice([0, -1, 2 ** 40])) if rng.random() < 0.1 else int(rng.integers(0, 10 ** 6)) for _ in range(m)])
    rc = L.dalib200ToDecibelsSetup(plans["Signal"].handle, C.byref(db), n, vol)
    note("todb", rc)
    if rc == 0:
        launch("todb", L.dalib200SignalLaunch, plans["Signal"].handle, fake_ptrs(m, 0x10000000), fake_ptrs(m, 0x7000000000), None)
    shp = (C.c_int64 * (2 * m))(*[int(rng.choice([0, -1, 2 ** 33])) if rng.random() < 0.08 else int(rng.integers(0, 600)) for _ in range(2 * m)])
    mf = capi.MfccArgs(code([1, 13, 40, 128, 1000]), code([1, 2, 3, 4]), int(rng.integers(0, 2)), C.c_float(flt(0, 30)))
    rc = L.dalib200MfccSetup(plans["Signal"].handle, C.byref(mf), n, shp)
    note("mfcc", rc)
    if rc == 0:
        L.dalib200SignalOutputRows(plans["Signal"].handle)
        launch("mfcc", L.dalib200SignalLaunch, plans["Signal"].handle, fake_ptrs(m, 0x10000000), fake_ptrs(m, 0x7000000000), None)
    na = capi.NormalizeArgs(code([0, 1, 2]), small(0, 3), C.c_float(flt(0, 2)), C.c_float(flt(-1, 1)), C.c_float(flt(0, 1e-3)))
    rc = L.dalib200NormalizeSetup(plans["Signal"].handle, C.byref(na), n, shp)
    note("normalize", rc)
    if rc == 0:
        launch("normalize", L.dalib200SignalLaunch, plans["Signal"].handle, fake_ptrs(m, 0x10000000), fake_ptrs(m, 0x7000000000), None)

    class AR(C.Structure):
        _fields_ = [("in_rate", C.c_double), ("out_rate", C.c_double), ("in_length", C.c_int64), ("out_length", C.c_int64), ("channels", C.c_int32)]
    ars = (AR * m)()
    for s in ars:
        s.in_rate, s.out_rate = flt(8000, 48000), flt(8000, 48000)
        s.in_length = int(rng.choice([0, -1, 2 ** 40])) if rng.random() < 0.1 else int(rng.integers(0, 200000))
        s.out_length = int(rng.choice([0, -1, 2 ** 40])) if rng.random() < 0.1 else int(rng.integers(0, 200000))
        s.channels = small(1, 9)
    rc = L.dalib200AudioResampleSetup(plans["Signal"].handle, n, ars, C.c_float(flt(0, 100)))
    note("audio_resample", rc)
    if rc == 0:
        launch("audio_resample", L.dalib200SignalLaunch, plans["Signal"].handle, fake_ptrs(m, 0x10000000), fake_ptrs(m, 0x7000000000), None)

    class NS(C.Structure):
        _fields_ = [("cutoff_db", C.c_float), ("reference_power", C.c_float), ("use_reference_power", C.c_int32)]
    nss = (NS * m)()
    for s in nss:
        s.cutoff_db, s.reference_power, s.use_reference_power = flt(-100, 0), flt(0, 1), int(rng.integers(0, 2))
    rc = L.dalib200NonsilentSetup(plans["Signal"].handle, n, lens, nss, code([1, 512, 2048, 8192]), code([-1, 512, 2048, 8192, 1000]))
    note("nonsilent", rc)
    if rc == 0:
        launch("nonsilent", L.dalib200NonsilentLaunch, plans["Signal"].handle, fake_ptrs(m, 0x10000000), fake_ptrs(m, 0x5000000000), fake_ptrs(m, 0x7000000000), None)
    # ---- generic
    mul = (C.c_float * m)(*[flt() for _ in range(m)])
    add = (C.c_float * m)(*[flt() for _ in range(m)])
    rc = L.dalib200MultiplyAddSetup(plans["Generic"].handle, n, vol, mul, add, code([0, 9]))
    note("multiply_add", rc)
    if rc == 0:
        launch("multiply_add", L.dalib200GenericLaunch, plans["Generic"].handle, fake_ptrs(m, 0x10000000), fake_ptrs(m, 0x7000000000), None)

    class WS(C.Structure):
        _fields_ = [("in_h", C.c_int32), ("in_w", C.c_int32), ("channels", C.c_int32), ("anchor_y", C.c_int32), ("anchor_x", C.c_int32),
                    ("out_h", C.c_int32), ("out_w", C.c_int32), ("flip_x", C.c_int32), ("flip_y", C.c_int32), ("fill", C.c_uint8 * 4)]
    ws = (WS * m)()
    for s in ws:
        s.in_h, s.in_w, s.channels = dim(0, 3000), dim(0, 3000), small(1, 5)
        s.anchor_y, s.anchor_x, s.out_h, s.out_w = small(-50, 3000), small(-50, 3000), dim(0, 3000), dim(0, 3000)
        s.flip_x, s.flip_y = int(rng.integers(0, 2)), int(rng.integers(0, 2))
    rc = L.dalib200WindowCopySetup(plans["Generic"].handle, n, ws)
    note("window_copy", rc)
    if rc == 0:
        launch("window_copy", L.dalib200GenericLaunch, plans["Generic"].handle, fake_ptrs(m, 0x10000000), fake_ptrs(m, 0x7000000000), None)
    # ---- separable convolution: zero / negative / 2^31 extents, even / zero / huge diameters, windows outside the array, NaN / inf taps
    nw = int(rng.choice([0, 1, 7, 64, 300]))
    wins = np.ascontiguousarray(rng.uniform(0, 1, max(nw, 1)), np.float32)
    if nw and rng.random() < 0.1 * MILD:
        wins[int(rng.integers(0, nw))] = float(rng.choice([float("nan"), float("inf"), float("-inf")]))
    SC = (capi.SepConvSample * m)()
    for s in SC:
        s.ndim, s.channels = code([2, 3]), small(1, 5)
        for a in range(3):
            s.shape[a] = dim(0, 300)
            s.diameter[a] = int(rng.choice(BAD_I)) if rng.random() < 0.1 * MILD else 2 * int(rng.integers(0, 12)) + 1
            s.window_offset[a] = int(rng.choice(BAD_I)) if rng.random() < 0.05 * MILD else int(rng.integers(0, max(nw - s.diameter[a], 0) + 1))
    rc = L.dalib200SepConvPlanSetup(plans["SepConv"].handle, n, SC, wins.ctypes.data, nw, code([0, 9]), code([0, 9]))
    note("sepconv", rc)
    # the launch allocates the float temporaries for real (calloc in the stub): only batches of a plausible size are launched
    if rc == 0 and sum(int(np.prod([s.shape[a] for a in range(s.ndim)], dtype=np.int64)) * s.channels for s in SC[:max(n, 0)]) < 2 ** 27:
        launch("sepconv", L.dalib200SepConvLaunch, plans["SepConv"].handle, fake_ptrs(m, 0x10000000), fake_ptrs(m, 0x7000000000), None)
        for i in range(max(0, min(n, m))):
            L.dalib200SepConvPlanGetPath(plans["SepConv"].handle, i)
print("seed", sys.argv[1] if len(sys.argv) > 1 else 0, "iterations", N, "- no sanitizer report;", {f"{k[0]}:{k[1]}": v for k, v in sorted(hist.items())})

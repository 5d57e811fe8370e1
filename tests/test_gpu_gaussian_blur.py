"""-m gpu tests of the separable convolution kernels (csrc/sepconv.cu) and fn.gaussian_blur: bit-exact against the plain-C restatement
(oracle/gaussian_oracle.c oracle_sepconv) through the C-ABI and through the pipeline; both kernel paths, confirmed through
dalib200SepConvPlanGetPath; argument errors; and a tolerance cross-check against torch's reflect-padded depthwise convolution."""
import ctypes as C

import numpy as np
import pytest

from dali_b200 import capi
from oracle import pygaussian as po

pytestmark = pytest.mark.gpu


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint8)


def sepconv(xs, windows, out_dtype=None, ndim=2, plan=None, want_path=False):
    """Samples x[i] of shape (H, W, C) or (D, H, W, C) with per-axis windows windows[i] (outermost first) through dalib200SepConv*."""
    import torch
    n = len(xs)
    samples = (capi.SepConvSample * max(n, 1))()
    flat, offs = [], 0
    for i, (x, ws) in enumerate(zip(xs, windows)):
        s = samples[i]
        s.ndim = ndim
        for a in range(ndim):
            s.shape[a], s.diameter[a], s.window_offset[a] = int(x.shape[a]), len(ws[a]), offs
            flat.append(np.asarray(ws[a], np.float32))
            offs += len(ws[a])
        s.channels = int(x.shape[ndim])
    wcat = np.ascontiguousarray(np.concatenate(flat) if flat else np.zeros(1, np.float32))
    in_dt = capi.UINT8 if xs[0].dtype == np.uint8 else capi.FLOAT
    out_dtype = np.dtype(out_dtype or xs[0].dtype)
    out_dt = capi.UINT8 if out_dtype == np.uint8 else capi.FLOAT
    plan = plan or capi.Plan("SepConv", max(n, 1))
    capi.check(capi.lib().dalib200SepConvPlanSetup(plan.handle, n, samples, wcat.ctypes.data, wcat.size, in_dt, out_dt))
    din = [torch.from_numpy(np.ascontiguousarray(x)).cuda() for x in xs]
    outs = [torch.empty(x.shape, dtype=torch.uint8 if out_dt == capi.UINT8 else torch.float32, device="cuda") for x in xs]
    capi.check(capi.lib().dalib200SepConvLaunch(plan.handle, capi.ptr_array(din), capi.ptr_array(outs), capi.stream_handle()))
    torch.cuda.synchronize()
    res = [o.cpu().numpy() for o in outs]
    if want_path:
        return res, [capi.lib().dalib200SepConvPlanGetPath(plan.handle, i) for i in range(n)]
    return res


def _win(sigma, ws=0):
    return po.gaussian_window(*po.gaussian_params(sigma, ws))


def _img(rng, shape, dt):
    return rng.integers(0, 256, shape, dtype=np.uint8) if dt == np.uint8 else rng.uniform(-50, 300, shape).astype(np.float32)


def test_gaussian_window_host_helper_equals_restatement():
    for sigma, d in [(0.1, 3), (0.5, 5), (1.0, 7), (2.0, 13), (3.8, 23), (0.3, 1), (7.5, 101)]:
        w = np.empty(d, np.float32)
        capi.lib().dalib200GaussianWindow(C.c_float(sigma), d, w.ctypes.data)
        assert np.array_equal(_bits(w), _bits(po.gaussian_window(sigma, d))), (sigma, d)


@pytest.mark.parametrize("in_dt,out_dt", [(np.uint8, np.uint8), (np.uint8, np.float32), (np.float32, np.float32)])
def test_sepconv_2d_ragged_batch_both_paths(in_dt, out_dt):
    """Ragged HW / HWC frames (C 1/3/4; 1x1, 1xN, frames smaller than the window), windows from 3 to 63 taps and one oversize
    vertical window (generic path), every sample against the restatement bit for bit."""
    rng = np.random.default_rng(5)
    shapes = [(224, 224, 3), (1, 1, 3), (1, 37, 1), (29, 1, 4), (5, 7, 3), (100, 300, 4), (64, 48, 1), (17, 250, 3), (480, 640, 3)]
    sig = [(1.3, 0.7), (2.0, 2.0), (0.4, 3.1), (6.0, 0.2), (4.0, 4.0), (0.9, 1.9), (10.0, 0.5), (40.0, 1.0), (3.0, 3.0)]
    xs = [_img(rng, s, in_dt) for s in shapes]
    wins = [(_win(a), _win(b)) for a, b in sig]
    got, paths = sepconv(xs, wins, out_dt, want_path=True)
    for i, x in enumerate(xs):
        want = po.sepconv(x, wins[i], out_dt)
        assert np.array_equal(_bits(got[i]), _bits(want)), (i, shapes[i], sig[i])
    assert paths[7] == 0, "a 241-tap vertical window must take the per-axis passes"
    assert paths[0] == 1 and paths[8] == 1, paths


def test_sepconv_unaligned_rows_take_the_pass_kernel():
    rng = np.random.default_rng(6)
    xs = [_img(rng, (37, 21, 3), np.uint8), _img(rng, (40, 16, 1), np.uint8)]
    wins = [(_win(1.0), _win(2.0))] * 2
    got, paths = sepconv(xs, wins, want_path=True)
    assert paths == [0, 1], paths          # 63-byte rows cannot be bulk-copied; 16-byte rows can
    for i, x in enumerate(xs):
        assert np.array_equal(got[i], po.sepconv(x, wins[i])), i


@pytest.mark.parametrize("in_dt,out_dt", [(np.uint8, np.uint8), (np.float32, np.float32)])
def test_sepconv_volumes(in_dt, out_dt):
    rng = np.random.default_rng(7)
    shapes = [(16, 20, 24, 1), (5, 9, 7, 3), (1, 1, 1, 1), (3, 40, 2, 4)]
    xs = [_img(rng, s, in_dt) for s in shapes]
    wins = [(_win(1.5), _win(0.8), _win(2.5)), (_win(3.0), _win(1.0), _win(0.3)), (_win(1.0),) * 3, (_win(0.6), _win(5.0), _win(2.0))]
    got = sepconv(xs, wins, out_dt, ndim=3)
    for i, x in enumerate(xs):
        assert np.array_equal(_bits(got[i]), _bits(po.sepconv(x, wins[i], out_dt))), (i, shapes[i])


def test_sepconv_plan_reuse_with_growing_shapes():
    rng = np.random.default_rng(8)
    plan = capi.Plan("SepConv", 4)
    for size in (8, 64, 300):
        xs = [_img(rng, (size, size + 3, 1), np.float32) for _ in range(3)]
        wins = [(_win(2.0), _win(1.0))] * 3
        got = sepconv(xs, wins, plan=plan)
        for i, x in enumerate(xs):
            assert np.array_equal(_bits(got[i]), _bits(po.sepconv(x, wins[i]))), (size, i)
        vols = [_img(rng, (size // 4 + 1, 9, 10, 2), np.float32)]
        got = sepconv(vols, [(_win(1.0), _win(1.0), _win(1.0))], ndim=3, plan=plan)
        assert np.array_equal(_bits(got[0]), _bits(po.sepconv(vols[0], [_win(1.0)] * 3))), size


def test_sepconv_setup_rejects_bad_arguments():
    lib = capi.lib()
    plan = capi.Plan("SepConv", 2)
    w = np.ones(9, np.float32)
    bad = np.array([0.2, np.nan, 0.2], np.float32)

    def setup(ndim=2, shape=(8, 8, 0), ch=3, diam=(3, 3, 1), offs=(0, 0, 0), win=w, in_dt=capi.UINT8, out_dt=capi.UINT8):
        s = (capi.SepConvSample * 1)()
        s[0].ndim, s[0].channels = ndim, ch
        for a in range(3):
            s[0].shape[a], s[0].diameter[a], s[0].window_offset[a] = shape[a], diam[a], offs[a]
        return lib.dalib200SepConvPlanSetup(plan.handle, 1, s, win.ctypes.data, win.size, in_dt, out_dt)
    assert setup() == 0
    assert setup(diam=(4, 3, 1)) == 1 and b"odd" in lib.dalib200GetLastError()
    assert setup(diam=(0, 3, 1)) == 1
    assert setup(diam=(9001, 3, 1)) == 1 and b"limit" in lib.dalib200GetLastError()
    assert setup(shape=(-1, 8, 0)) == 1
    assert setup(shape=(1 << 20, 1 << 12, 0)) == 1
    assert setup(offs=(7, 0, 0)) == 1
    assert setup(win=bad) == 1 and b"finite" in lib.dalib200GetLastError()
    assert setup(ndim=4) == 1
    assert setup(in_dt=capi.FLOAT, out_dt=capi.UINT8) == 2
    assert setup(in_dt=capi.INT16, out_dt=capi.INT16) == 2


# ------------------------------------------------------------------------------------------------------------ fn.gaussian_blur
def _run(batch, data, build, layout, extra=()):
    from dali_b200 import fn, pipeline_def

    @pipeline_def(batch_size=batch, num_threads=1, device_id=0, seed=1234)
    def pipe():
        x = fn.external_source(source=lambda i: data, device="gpu", layout=layout)
        ex = [fn.external_source(source=(lambda v: (lambda i: v))(v)) for v in extra]
        return build(fn, x, *ex)
    p = pipe()
    p.build()
    return [o.as_cpu() if hasattr(o, "as_cpu") else o for o in p.run()]


def _blur(x, layout, sigma, ws, out_dtype):
    frames = layout.startswith("F")
    has_c = layout.endswith("C")
    xs = list(x) if frames else [x]
    outs = [po.gaussian_blur(f, sigma, ws, out_dtype, channels=has_c) for f in xs]
    return np.stack(outs) if frames else outs[0]


@pytest.mark.parametrize("layout,shape", [("HW", (45, 61)), ("HWC", (50, 70, 3)), ("HWC", (33, 20, 1)), ("HWC", (40, 40, 4)),
                                          ("FHWC", (3, 24, 31, 3)), ("DHWC", (9, 14, 11, 2)), ("FDHWC", (2, 6, 8, 7, 1)),
                                          ("DHW", (7, 12, 13)), ("FHW", (2, 30, 20))])
def test_gaussian_blur_layouts(layout, shape):
    from dali_b200 import types
    rng = np.random.default_rng(len(layout) * 100 + shape[0])
    data = [rng.integers(0, 256, shape, dtype=np.uint8) for _ in range(3)]
    a, b = _run(3, data, lambda fn, x: (fn.gaussian_blur(x, sigma=1.7), fn.gaussian_blur(x, window_size=5, dtype=types.FLOAT)), layout)
    for i, x in enumerate(data):
        assert np.array_equal(a[i], _blur(x, layout, 1.7, 0, np.uint8)), (layout, i)
        assert np.array_equal(_bits(b[i]), _bits(_blur(x, layout, 0.0, 5, np.float32))), (layout, i)


def test_gaussian_blur_per_sample_and_per_axis_arguments():
    from dali_b200 import types
    rng = np.random.default_rng(11)
    data = [rng.uniform(0, 1, s).astype(np.float32) for s in ((60, 80, 3), (1, 1, 3), (1, 50, 3), (3, 2, 3), (224, 224, 3))]
    n = len(data)
    sig = [np.array(v, np.float32) for v in (0.5, 2.0, 1.1, 3.0, 0.1)]
    win = [np.array(v, np.int32) for v in (0, 23, 0, 7, 0)]
    axes = [np.array(v, np.float32) for v in ((1.0, 3.0), (0.5, 0.5), (2.0, 0.7), (1.5, 1.5), (4.0, 0.2))]
    a, b, c, u = _run(n, data, lambda fn, x, s, w, ax: (
        fn.gaussian_blur(x, sigma=s, window_size=w),
        fn.gaussian_blur(x, sigma=ax),
        fn.gaussian_blur(x, sigma=[0.8, 2.5], window_size=[0, 9]),
        fn.random.uniform(range=[0.1, 2.0])), "HWC", extra=(sig, win, axes))
    # the seeded sigma draw is an output too: the blur of every view with its own sigma
    d, u2 = _run(n, data, lambda fn, x: (lambda s: (fn.gaussian_blur(x, sigma=s), s))(fn.random.uniform(range=[0.1, 2.0], seed=77)), "HWC")
    for i, x in enumerate(data):
        assert np.array_equal(_bits(a[i]), _bits(po.gaussian_blur(x, float(sig[i]), int(win[i])))), i
        assert np.array_equal(_bits(b[i]), _bits(po.gaussian_blur(x, axes[i]))), i
        assert np.array_equal(_bits(c[i]), _bits(po.gaussian_blur(x, [0.8, 2.5], [0, 9]))), i
        assert np.array_equal(_bits(d[i]), _bits(po.gaussian_blur(x, float(np.asarray(u2[i]).reshape(-1)[0])))), i
        assert 0.1 <= float(np.asarray(u[i]).reshape(-1)[0]) <= 2.0


@pytest.mark.parametrize("kwargs,layout,dtype,needle", [
    (dict(window_size=4), "HWC", np.uint8, "odd"),
    (dict(sigma=0.0, window_size=0), "HWC", np.uint8, "shouldn't be 0"),
    (dict(sigma=-1.0), "HWC", np.uint8, "non-negative"),
    (dict(sigma=[1.0, 2.0, 3.0]), "HWC", np.uint8, "must have 2 elements"),
    (dict(sigma=1.0), "CHW", np.uint8, "unsupported layout"),
    (dict(sigma=1.0), "HWC", np.int16, "uint8 and float"),
])
def test_gaussian_blur_rejects_invalid_arguments(kwargs, layout, dtype, needle):
    data = [np.zeros((3, 8, 8) if layout == "CHW" else (8, 8, 3), dtype)]
    with pytest.raises(Exception) as e:
        _run(1, data, lambda fn, x: fn.gaussian_blur(x, **kwargs), layout)
    assert needle in str(e.value), str(e.value)


def test_gaussian_blur_against_torch_reflect_conv():
    """An oracle independent of the restatement: two depthwise fp32 passes of torch with reflect padding (also reflect-101)."""
    import torch
    import torch.nn.functional as F
    rng = np.random.default_rng(12)
    x = rng.integers(0, 256, (4, 96, 128, 3), dtype=np.uint8)
    sig = 1.8
    (out,) = _run(4, list(x), lambda fn, v: (fn.gaussian_blur(v, sigma=sig, dtype=__import__("dali_b200").types.FLOAT),), "HWC")
    w = torch.from_numpy(_win(sig)).cuda()
    r = (w.numel() - 1) // 2
    t = torch.from_numpy(x).cuda().permute(0, 3, 1, 2).float()
    t = F.conv2d(F.pad(t, (r, r, 0, 0), mode="reflect"), w.view(1, 1, 1, -1).repeat(3, 1, 1, 1), groups=3)
    t = F.conv2d(F.pad(t, (0, 0, r, r), mode="reflect"), w.view(1, 1, -1, 1).repeat(3, 1, 1, 1), groups=3)
    want = t.permute(0, 2, 3, 1).cpu().numpy()
    got = np.stack([np.asarray(o) for o in out])
    assert np.abs(got - want).max() <= 1e-3, np.abs(got - want).max()

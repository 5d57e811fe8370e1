"""Gaussian blur on the GPU (dalib200SepConv*, the kernels behind fn.gaussian_blur) on four seeded workloads, with a torch baseline.

    python tools/bench_gaussian_blur.py [--steps 20] [--warmup 3] [--check] [--out FILE]

Workloads: (a) the self-supervised recipes' view blur: 256 x 224x224x3 u8, sigma ~ U[0.1, 2.0] per sample, window from sigma;
(b) the same with window_size = 23; (c) 64 x 1080x1920x3 u8, sigma = 3; (d) 8 x 128^3 x 1 f32 DHW volumes, sigma = 1.5.
Each step is timed with CUDA events around the launch; L2 is flushed (256 MiB write) between steps outside the events; median and
mean are reported.  Lower bounds: bytes (input + output) over 7.7 TB/s, and FP32 operations (a product and a sum per tap, per pass,
per element) over 148 SMs x 128 lanes x the SM clock read through NVML in the same run; the larger one is named.  Baseline: torch,
two (three for volumes) depthwise fp32 convolutions with reflect padding (reflect-101), u8 converted to float inside the timed region.
--check compares a sample of the outputs with the plain-C restatement (oracle/pygaussian.py) bit for bit.  Prints one JSON line."""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

HBM_BYTES_PER_S = 7.7e12


def device_info():
    import pynvml
    import torch
    pynvml.nvmlInit()
    h = pynvml.nvmlDeviceGetHandleByIndex(torch.cuda.current_device())
    name = pynvml.nvmlDeviceGetName(h)
    return {"name": name.decode() if isinstance(name, bytes) else name,
            "power_limit_w": pynvml.nvmlDeviceGetPowerManagementLimit(h) / 1000.0,
            "sm_clock_max_mhz": pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)}, (pynvml, h)


def workloads(rng):
    from oracle import pygaussian as po
    out = []
    sig = rng.uniform(0.1, 2.0, 256).astype(np.float32)
    for tag, ws in (("a_ssl_224_sigma_u0.1_2", 0), ("b_ssl_224_window23", 23)):
        params = [po.gaussian_params(s, ws) for s in sig]
        out.append(dict(name=tag, shape=(224, 224, 3), n=256, dtype=np.uint8, ndim=2, params=[(p, p) for p in params]))
    p = po.gaussian_params(3.0, 0)
    out.append(dict(name="c_1080p_sigma3", shape=(1080, 1920, 3), n=64, dtype=np.uint8, ndim=2, params=[(p, p)] * 64))
    p = po.gaussian_params(1.5, 0)
    out.append(dict(name="d_volume128_f32_sigma1.5", shape=(128, 128, 128, 1), n=8, dtype=np.float32, ndim=3, params=[(p, p, p)] * 8))
    return out


def run(wl, steps, warmup, check, nvml):
    import ctypes as C
    import torch
    import torch.nn.functional as F
    from dali_b200 import capi
    from oracle import pygaussian as po
    lib = capi.lib()
    n, shape, nd = wl["n"], wl["shape"], wl["ndim"]
    g = torch.Generator(device="cuda").manual_seed(1)
    if wl["dtype"] == np.uint8:
        x = torch.randint(0, 256, (n,) + shape, dtype=torch.uint8, device="cuda", generator=g)
    else:
        x = torch.rand((n,) + shape, dtype=torch.float32, device="cuda", generator=g)
    y = torch.empty_like(x)
    wins, offs, key = [], {}, {}
    samples = (capi.SepConvSample * n)()
    for i, pr in enumerate(wl["params"]):
        s = samples[i]
        s.ndim, s.channels = nd, shape[-1]
        for a in range(nd):
            sg, d = pr[a]
            if (sg, d) not in key:
                key[(sg, d)] = sum(len(w) for w in wins)
                wins.append(po.gaussian_window(sg, d))
            s.shape[a], s.diameter[a], s.window_offset[a] = shape[a], d, key[(sg, d)]
    wcat = np.ascontiguousarray(np.concatenate(wins))
    plan = capi.Plan("SepConv", n)
    dt = capi.UINT8 if wl["dtype"] == np.uint8 else capi.FLOAT
    capi.check(lib.dalib200SepConvPlanSetup(plan.handle, n, samples, wcat.ctypes.data, wcat.size, dt, dt))
    ip, op = capi.ptr_array([x[i] for i in range(n)]), capi.ptr_array([y[i] for i in range(n)])
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def ours():
        capi.check(lib.dalib200SepConvLaunch(plan.handle, ip, op, capi.stream_handle()))

    # torch baseline: grouped depthwise convolutions over all samples x channels, windows zero-padded to the batch's longest
    Cn = shape[-1]
    dmax = [max(pr[a][1] for pr in wl["params"]) for a in range(nd)]
    kern = []
    for a in range(nd):
        k = np.zeros((n * Cn, dmax[a]), np.float32)
        for i, pr in enumerate(wl["params"]):
            w = po.gaussian_window(*pr[a])
            o = (dmax[a] - len(w)) // 2
            k[i * Cn:(i + 1) * Cn, o:o + len(w)] = w
        kern.append(torch.from_numpy(k).cuda())

    def baseline():
        t = x.float()
        t = t.permute(0, nd + 1, *range(1, nd + 1)).reshape((1, n * Cn) + shape[:nd])
        conv = F.conv2d if nd == 2 else F.conv3d
        for a in reversed(range(nd)):
            r = (dmax[a] - 1) // 2
            ksh = [1] * nd
            ksh[a] = dmax[a]
            pad = [0] * (2 * nd)
            pad[2 * (nd - 1 - a)] = pad[2 * (nd - 1 - a) + 1] = r
            t = conv(F.pad(t, pad, mode="reflect"), kern[a].view((n * Cn, 1) + tuple(ksh)), groups=n * Cn)
        return t

    def timed(fn):
        for _ in range(warmup):
            fn()
        ts, clocks = [], []
        for _ in range(steps):
            flush.fill_(1)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            b.synchronize()
            ts.append(a.elapsed_time(b))
            clocks.append(nvml[0].nvmlDeviceGetClockInfo(nvml[1], nvml[0].NVML_CLOCK_SM))
        return float(np.median(ts)), float(np.mean(ts)), float(np.median(clocks))

    med, mean, clk = timed(ours)
    tmed, tmean, _ = timed(baseline)
    elems = n * int(np.prod(shape))
    esz = 1 if wl["dtype"] == np.uint8 else 4
    nbytes = 2 * elems * esz
    ops = sum(2 * elems * pr[a][1] for pr in wl["params"] for a in range(nd)) / n
    t_bytes = nbytes / HBM_BYTES_PER_S * 1e3
    t_ops = ops / (148 * 128 * clk * 1e6) * 1e3
    paths = sorted({lib.dalib200SepConvPlanGetPath(plan.handle, i) for i in range(n)})
    res = {"workload": wl["name"], "batch": n, "shape": list(shape), "dtype": str(np.dtype(wl["dtype"])),
           "ms_median": med, "ms_mean": mean, "samples_per_s": n / med * 1e3, "kernel_path": paths,
           "bound_bytes_ms": t_bytes, "bound_fp32_ms": t_ops, "larger_bound": "fp32 operations" if t_ops > t_bytes else "bytes",
           "share_of_larger_bound": max(t_bytes, t_ops) / med, "sm_clock_mhz_median": clk, "algorithmic_bytes": nbytes,
           "fp32_operations": ops, "torch_ms_median": tmed, "torch_ms_mean": tmean}
    if check:
        torch.cuda.synchronize()
        bad = 0
        for i in sorted({0, n // 2, n - 1}):
            xi = x[i].cpu().numpy()
            want = po.sepconv(xi, [po.gaussian_window(*p) for p in wl["params"][i]])
            bad += int(np.count_nonzero(want.view(np.uint8) != y[i].cpu().numpy().view(np.uint8)))
        res["check"] = {"samples": len({0, n // 2, n - 1}), "mismatching_bytes": bad}
        tref = baseline().reshape((n, Cn) + shape[:nd]).permute(0, *range(2, nd + 2), 1).cpu().numpy()
        res["check"]["max_abs_diff_vs_torch"] = float(np.abs(tref - y.float().cpu().numpy()).max())
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--check", action="store_true")
    ap.add_argument("--out", default=None, help="also write the JSON here")
    a = ap.parse_args()
    if a.steps < 1 or a.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    import torch
    if not torch.cuda.is_available():
        sys.exit("bench_gaussian_blur.py needs a CUDA device")
    torch.cuda.set_device(0)
    info, nvml = device_info()
    rng = np.random.default_rng(2024)
    res = {"device": info, "steps": a.steps, "warmup": a.warmup,
           "l2": "flushed between timed steps (256 MiB write), outside the events",
           "workloads": [run(w, a.steps, a.warmup, a.check, nvml) for w in workloads(rng)]}
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()

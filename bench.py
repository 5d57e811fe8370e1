#!/usr/bin/env python
"""bench.py -- images/sec of the C2 hot path: 1080p JPEG decode -> Resize(224x224) -> CropMirrorNormalize fp16 CHW,
batch 256 per GPU (BASELINE.json metric, configs[1]), weak scaling over N GPUs of one node.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
  (N > 1: python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...)

One JSON line on rank 0.  `value` = device-resident throughput (encoded bytes already in HBM when the timed
region starts), `e2e` = the same through the public pipeline API with HOST buffers (header parse + pinned staging
+ H2D inside the timed region, and a D2H read of a result checksum), `roofline` = the dominant kernel timed live
with CUDA events inside the timed region, `cpu_baseline` = the reference CPU path on a bounded sample.
`--impl reference` times the reference's own CPU implementation (libjpeg-turbo via cv2.imdecode for the decode
stage -- the stand-in for nvimgcodec's CPU backend --, then the reference's CPU resample and CMN kernels
compiled from /root/reference into oracle/_ref, or the oracle port when that library is absent).
"""
import argparse
import concurrent.futures as cf
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

BATCH = 256
METRIC = "images/sec decode+resize+CMN (batch 256, 1080p JPEG)"
H, W = 1080, 1920
OUT = 224
ALG_DECODE = H * W * 3            # + J
ALG_RESIZE = H * W * 3 + OUT * OUT * 3
ALG_CMN = OUT * OUT * 3 + OUT * OUT * 3 * 2


def effective_cores():
    """Host cores this process may actually use: the scheduler affinity mask, capped by the cgroup CPU quota (a container
    that reports 128 logical CPUs can be limited to a fraction of them; the stated core count must be the usable one)."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    quota = None
    try:
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max":
            quota = float(q) / float(p)
    except Exception:
        try:
            q = float(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            p = float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                quota = q / p
        except Exception:
            pass
    if quota is not None:
        n = max(1, min(n, int(quota + 0.5)))
    return n, quota


def synth_image(h, w, seed):
    """SURVEY.md 8(d): bicubic-upsampled 34x60 uniform noise + sigma=5 gaussian noise."""
    import cv2
    r = np.random.default_rng(seed)
    lo = r.uniform(0, 255, (max(2, h // 32), max(2, w // 32), 3)).astype(np.float32)
    img = cv2.resize(lo, (w, h), interpolation=cv2.INTER_CUBIC) + r.normal(0, 5, (h, w, 3))
    return np.clip(img, 0, 255).astype(np.uint8)


def make_batch(n, seed0, threads):
    import cv2
    cv2.setNumThreads(1)

    def one(i):
        ok, enc = cv2.imencode(".jpg", synth_image(H, W, seed0 + i), [cv2.IMWRITE_JPEG_QUALITY, 90])
        return np.ascontiguousarray(enc.ravel())
    with cf.ThreadPoolExecutor(threads) as ex:
        return list(ex.map(one, range(n)))


class ClockSampler:
    """SM clock / throttle reasons sampled DURING the timed region (B200_PROFILING.md).  NVML in-process (a sample every ~2 ms: the
    timed region of the default run is only ~70 ms, shorter than the start-up of an `nvidia-smi -lms` child); nvidia-smi as fallback."""
    HW_SLOWDOWN, SW_THERMAL, HW_THERMAL, SW_POWER_CAP = 0x8, 0x20, 0x40, 0x4

    def __init__(self, index):
        self.index, self.samples, self.mx, self.reasons = index, [], None, set()
        self.stop_flag, self.thr, self.nvml, self.handle, self.proc, self.lines = False, None, None, None, None, []
        try:
            import pynvml
            pynvml.nvmlInit()
            h = None
            try:
                import torch
                uuid = str(torch.cuda.get_device_properties(index).uuid)
                h = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid).encode() if not uuid.startswith("GPU-") else uuid.encode())
            except Exception:
                h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.nvml, self.handle = pynvml, h
            self.mx = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nvml = None

    def _sample(self):
        n, h = self.nvml, self.handle
        self.samples.append(float(n.nvmlDeviceGetClockInfo(h, n.NVML_CLOCK_SM)))
        try:
            r = int(n.nvmlDeviceGetCurrentClocksEventReasons(h))
        except Exception:
            r = int(n.nvmlDeviceGetCurrentClocksThrottleReasons(h))
        for bit, nm in ((self.HW_SLOWDOWN, "hw_slowdown"), (self.HW_THERMAL, "hw_thermal_slowdown"), (self.SW_THERMAL, "sw_thermal_slowdown"),
                        (self.SW_POWER_CAP, "sw_power_cap")):
            if r & bit:
                self.reasons.add(nm)

    def _loop(self):
        while not self.stop_flag:
            try:
                self._sample()
            except Exception:
                break
            time.sleep(0.002)

    def start(self):
        if self.nvml is not None:
            self.thr = threading.Thread(target=self._loop, daemon=True)
            self.thr.start()
            return
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thr = threading.Thread(target=self._read, daemon=True)
            self.thr.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if self.nvml is not None:
            self.stop_flag = True
            if self.thr is not None:
                self.thr.join(timeout=1)
            return {"sm_mhz": float(np.median(self.samples)) if self.samples else None, "sm_max_mhz": self.mx, "reasons": sorted(self.reasons),
                    "samples": len(self.samples), "source": "nvml, sampled during the timed region"}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx = float(f[1])
            except ValueError:
                continue
            for k, nm in enumerate(names):
                if f[3 + k].lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm),
                "source": "nvidia-smi -lms 100"}


_CPU_STREAMS = None      # set before the worker processes are forked: they inherit the encoded batch


def _cpu_one(i, mirror_i):
    """One sample through the reference CPU path: libjpeg-turbo decode straight to RGB (cv2.IMREAD_COLOR_RGB: no BGR->RGB
    copy, the reference's decoder emits RGB itself), the reference's CPU resample and CMN kernels (oracle/_ref)."""
    import cv2
    from oracle import pyoracle as po
    from dali_b200.hotpath import IMAGENET_MEAN, IMAGENET_STD
    use_ref = po.have_ref()
    rs = po.ref_resample if use_ref else po.resample
    cm = po.ref_cmn if use_ref else po.cmn
    mean, inv = po.cmn_norm_args(IMAGENET_MEAN, IMAGENET_STD)
    img = cv2.imdecode(_CPU_STREAMS[i], cv2.IMREAD_COLOR_RGB)
    r = rs(img, (OUT, OUT))
    return cm(r, (0, 0), (OUT, OUT), bool(mirror_i), mean, inv, np.float16, "CHW")


def _cpu_worker(args):
    """One worker process: its slice of the sample on a small thread pool (every stage releases the GIL)."""
    idx, mirror, threads, keep = args
    import cv2
    cv2.setNumThreads(1)
    with cf.ThreadPoolExecutor(threads) as ex:
        outs = list(ex.map(_cpu_one, idx, mirror))
    return outs if keep else float(sum(float(o[0, 0, 0]) for o in outs))


class CpuReference:
    """The reference CPU path on the host cores, one sample per task (the reference's own threading model,
    dali/pipeline/operator/operator.h:305-314).  `cores` workers in total: P forked processes x T threads, so that the Python
    glue of one sample never waits for the GIL of another (a single 128-thread pool spent most of its time there)."""

    def __init__(self, streams, cores):
        global _CPU_STREAMS
        import multiprocessing as mp
        from oracle import pyoracle as po
        _CPU_STREAMS = streams
        self.kind = "reference" if po.have_ref() else "port"
        self.cores = cores
        # one single-threaded worker process per usable core (measured on the 16-core-quota B200 host: 16 x 1 = 907 img/s,
        # 2 x 8 threads = 660); beyond 32 cores the process count is capped and threads make up the difference
        self.procs = max(1, min(cores, 32))
        self.threads = max(1, cores // self.procs)
        self.pool = mp.get_context("fork").Pool(self.procs) if self.procs > 1 else None

    def run(self, n, mirror, keep=False):
        """Processes samples [0, n).  Returns (seconds, outputs or None)."""
        idx = list(range(n))
        parts = [(idx[k::self.procs], [int(mirror[i]) for i in idx[k::self.procs]], self.threads, keep) for k in range(self.procs)]
        t0 = time.perf_counter()
        res = self.pool.map(_cpu_worker, parts) if self.pool is not None else [_cpu_worker(parts[0])]
        dt = time.perf_counter() - t0
        if not keep:
            return dt, None
        outs = [None] * n
        for k, part in enumerate(res):
            for i, o in zip(idx[k::self.procs], part):
                outs[i] = o
        return dt, outs

    def single_core(self, n, mirror):
        global _CPU_STREAMS
        t0 = time.perf_counter()
        for i in range(n):
            _cpu_one(i, mirror[i])
        return n / (time.perf_counter() - t0)

    def close(self):
        if self.pool is not None:
            self.pool.close()
            self.pool.join()
            self.pool = None


def dump_sample(batch):
    """Indices of the images `--dump-outputs` keeps: the whole [batch, 3, 224, 224] output as float32 is 154 MB at batch 256,
    so a fixed, seeded sample of whole images is kept (60 MiB: under 64 MB with the index and the .npy headers), sorted."""
    n = min(batch, (60 << 20) // (3 * OUT * OUT * 4))
    return np.sort(np.random.default_rng(0).choice(batch, n, replace=False))


def reference_arm(batch, cores, steps, warmup, dump=None):
    """Times the reference CPU path (bounded sample per step) and returns the JSON fields shared by `--impl reference` and
    the `cpu_baseline` leg of our arm."""
    sample = batch if cores >= 32 else min(batch, max(8, 2 * cores))
    streams = make_batch(sample, 0, min(cores, 16))
    mirror = np.random.default_rng(0).integers(0, 2, sample)
    ref = CpuReference(streams, cores)
    try:
        for _ in range(warmup):
            ref.run(min(sample, max(2, cores)), mirror)
        times = []
        for _ in range(steps):
            dt, _ = ref.run(sample, mirror)
            times.append(dt)
        single = ref.single_core(min(sample, 6), mirror)
        if dump:
            _, outs = ref.run(sample, mirror, keep=True)
            np.save(dump, np.stack(outs))
    finally:
        ref.close()
    t = float(sum(times))
    return {"value": sample * steps / t, "unit": "images/s", "cores": cores, "os_cpu_count": os.cpu_count(), "kind": ref.kind,
            "workers": f"{ref.procs} processes x {ref.threads} threads", "single_core_value": single,
            "sample": f"{sample} images per step (bounded sample of the {batch}-image batch), {steps} steps; decode = cv2.imdecode "
                      "(libjpeg-turbo straight to RGB, stand-in for nvimgcodec's CPU backend), resize + CMN = reference CPU kernels"
                      + (" compiled from the reference sources (oracle/_ref)" if ref.kind == "reference" else " restated (oracle port)"),
            "ms_per_step": 1e3 * t / steps, "median_ms_per_step": 1e3 * float(np.median(times))}, sample


def secondary_workloads(hbm_peak, flush, steps, warmup):
    """BASELINE configs[2] (C3: warp_affine + hsv + CMN over 128 x 16 frames of 720p) and configs[3] (C4: spectrogram + mel over
    64 clips x 10 s @ 16 kHz): device-resident throughput with CUDA events, per-kernel times from the library's own launch
    timing, and an element-wise parity check of one frame / one clip against the CPU oracle (reported, not timed)."""
    import torch
    from dali_b200 import capi
    from dali_b200.hotpath import VideoPipelineC3, AudioPipelineC4, IMAGENET_MEAN, IMAGENET_STD
    from oracle import pyoracle as po
    out = {}

    def timed(fn):
        for _ in range(warmup):
            fn()
        torch.cuda.synchronize()
        capi.profiling(True); capi.profiling_collect()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        for a, b in ev:
            flush.fill_(1)
            a.record(); fn(); b.record()
        torch.cuda.synchronize()
        prof = capi.profiling_collect(); capi.profiling(False)
        agg = {}
        for name, ms in prof:
            agg[name] = agg.get(name, 0.0) + ms / steps
        return float(np.mean([a.elapsed_time(b) for a, b in ev])), agg

    # ---- C3
    nseq, flen, fh, fw = 128, 16, 720, 1280
    nfr = nseq * flen
    rng = np.random.default_rng(3)
    g = torch.Generator(device="cuda"); g.manual_seed(3)
    frames = torch.randint(0, 256, (nfr, fh, fw, 3), dtype=torch.uint8, device="cuda", generator=g)
    inv, hsvp, mir = [], [], []
    for q in range(nseq):
        ang, sc = np.deg2rad(rng.uniform(-10, 10)), rng.uniform(0.95, 1.05)
        cx, cy = fw / 2, fh / 2
        a, b = sc * np.cos(ang), sc * np.sin(ang)
        fwd = np.array([[a, -b, cx - a * cx + b * cy], [b, a, cy - b * cx - a * cy]], np.float32)      # src -> dst (inverse_map=False)
        m = po.affine_inv(fwd)                                                                            # what the kernel consumes
        hp = (rng.uniform(-30, 30), rng.uniform(0.7, 1.3), rng.uniform(0.8, 1.2))
        mr = int(rng.integers(0, 2))
        inv += [m] * flen; hsvp += [hp] * flen; mir += [mr] * flen
    v = VideoPipelineC3(nfr, (fh, fw))
    v.setup(inv, hsvp, mir)
    ms, kern = timed(lambda: v.launch(frames))
    alg = 2 * fh * fw * 3 * 2 + fh * fw * 3 * 3               # warp in+out, hsv in+out, CMN in + fp16 out  (SURVEY 8d: 19 353 600 B)
    i = 5 * flen + 3
    f0 = frames[i].cpu().numpy()
    w0 = po.warp_affine(f0, inv[i], None, 1, 0.0)
    t0 = po.hsv(w0, *hsvp[i])
    mean, istd = po.cmn_norm_args(IMAGENET_MEAN, IMAGENET_STD)
    c0 = po.cmn(t0, (0, 0), (fh, fw), bool(mir[i]), mean, istd, np.float16, "CHW")
    got = v.output[i].cpu().numpy()
    out["c3_video"] = {"workload": "C3: warp_affine(LINEAR, fill 0) -> hsv -> crop_mirror_normalize(fp16 CHW), 128 x 16 frames 720p",
                       "value": nfr / (ms / 1e3), "unit": "frames/s", "ms_per_step": ms, "kernels_ms": kern,
                       "op_boundary_GBps": alg * nfr / (ms / 1e3) / 1e9, "op_boundary_frac_of_hbm": alg * nfr / (ms / 1e3) / 1e9 / hbm_peak,
                       "parity_mismatching_elements": int((got.view(np.uint16) != c0.view(np.uint16)).sum()), "parity_elements": int(c0.size)}
    del v, frames
    torch.cuda.empty_cache()
    # ---- C4
    nclip, clen = 64, 160000
    t = np.arange(clen, dtype=np.float64) / 16000.0
    clips = np.empty((nclip, clen), np.float32)
    for q in range(nclip):
        r = np.random.default_rng(400 + q)
        sig = sum(r.uniform(0.05, 0.2) * np.sin(2 * np.pi * r.uniform(50, 7000) * t + r.uniform(0, 6.28)) for _ in range(5))
        clips[q] = np.clip(sig + r.normal(0, 0.02, clen), -1, 1)
    dclips = torch.from_numpy(clips).cuda()
    au = AudioPipelineC4(nclip, clen)
    ms, kern = timed(lambda: au.launch(dclips))
    nwin = au.nwin
    alg = clen * 4 + 513 * nwin * 4 + 513 * nwin * 4 + 128 * nwin * 4
    spec0 = po.spectrogram(clips[7], 1024, 1024, 256, 2)
    mel0 = po.mel_filter_bank(spec0, 128, 16000.0, 0.0, 8000.0)
    gs, gm = au.spectra[7].cpu().numpy(), au.output[7].cpu().numpy()
    # the same clips through the optional tensor-core mel path (dense TF32x3 GEMM, mma.sync): tolerance path, reported beside the default
    capi.check(capi.lib().dalib200MelPlanSetTensorCores(au.mel.handle, 1))
    ms_tc, kern_tc = timed(lambda: au.launch(dclips))
    gm_tc = au.output[7].cpu().numpy()
    capi.check(capi.lib().dalib200MelPlanSetTensorCores(au.mel.handle, 0))
    # the chain as the executor runs it when only the mel output is consumed: STFT -> mel in ONE kernel, spectrogram never written
    fu = AudioPipelineC4(nclip, clen, fused=True, keep_spectrogram=False)
    ms_f, kern_f = timed(lambda: fu.launch(dclips))
    fused_equal = bool(torch.equal(fu.output.view(torch.int32), au.launch(dclips).view(torch.int32)))
    alg_f = clen * 4 + 128 * nwin * 4
    out["c4_audio"] = {"workload": "C4: spectrogram(nfft 1024, window 1024, step 256, power 2) -> mel_filter_bank(128, sr 16 kHz), 64 clips x 10 s",
                       "value": nclip * nwin / (ms_f / 1e3), "unit": "audio frames/s", "ms_per_step": ms_f, "kernels_ms": kern_f,
                       "path": "fused STFT -> mel kernel (register-resident 32 x 32 FFT, spectrogram not materialised)",
                       "fused_equals_two_kernel_chain_bitwise": fused_equal,
                       "fused_boundary_GBps": alg_f * nclip / (ms_f / 1e3) / 1e9,
                       "two_kernel_chain": {"value": nclip * nwin / (ms / 1e3), "ms_per_step": ms, "kernels_ms": kern},
                       "op_boundary_GBps": alg * nclip / (ms / 1e3) / 1e9, "op_boundary_frac_of_hbm": alg * nclip / (ms / 1e3) / 1e9 / hbm_peak,
                       "stft_max_abs_err_over_max": float(np.abs(gs - spec0).max() / max(1e-30, np.abs(spec0).max())),
                       "stft_stated_tolerance": 2e-4,
                       "mel_max_rel_err": float(np.abs(gm - mel0).max() / max(1e-30, np.abs(mel0).max())),
                       "mel_tensor_core_path": {"kernel_ms": kern_tc.get("mel_filter_bank_mma"), "step_ms": ms_tc,
                                                "max_rel_diff_vs_banded_kernel": float(np.abs(gm_tc - gm).max() / max(1e-30, np.abs(gm).max())),
                                                "note": "mma.sync m16n8k8 TF32, 3-term split, FP32 accumulate; opt-in (dalib200MelPlanSetTensorCores)"}}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3, help="untimed steps in front of every timed leg")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=BATCH)
    ap.add_argument("--no-secondary", action="store_true", help="skip the C3 (video) and C4 (audio) secondary measurements")
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the CPU baseline leg of our arm")
    ap.add_argument("--dump", default=None, help="(reference arm) save the outputs of the sample as .npy")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="after the timed steps, write what the last timed step computed to DIR/*.npy (float32; a fixed, seeded "
                         "sample of the images when the whole batch exceeds 64 MB); --impl ours only: the reference arm "
                         "computes a bounded CPU sample of other size, which --dump saves")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    cores, cpu_quota = effective_cores()
    print(f"host: os.cpu_count()={os.cpu_count()} affinity={len(os.sched_getaffinity(0))} cgroup quota={cpu_quota} -> {cores} usable cores; "
          f"loadavg={os.getloadavg()}", file=sys.stderr)
    batch = args.batch
    config = {"workload": "C2: 1080p JPEG (q90, 4:2:0, baseline) -> decoders.image(mixed) -> resize(224x224, triangular antialias)"
                          " -> crop_mirror_normalize(fp16, CHW, mirror, ImageNet mean/std)",
              "batch_per_gpu": batch, "image": [H, W, 3], "output": [3, OUT, OUT], "sharding": f"independent shard per GPU x{world}"}

    # ------------------------------------------------------------------ reference arm (CPU)
    if args.impl == "reference":
        if rank != 0:
            return 0
        cb, sample = reference_arm(batch, cores, args.steps, args.warmup, dump=args.dump)
        line = {"impl": "reference", "metric": METRIC, "value": cb["value"], "unit": "images/s",
                "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": cb["ms_per_step"],
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
                "config": config, "cpu_baseline": cb,
                "e2e": {"value": cb["value"], "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return 0

    # ---- CPU baseline (rank 0, N == 1 only): the same reference arm on a bounded sample, BEFORE CUDA is initialised (the
    #      worker processes are forked); its outputs are kept for the parity check of the timed configuration
    cpu_baseline, cpu_dump, cpu_sample = None, None, 0
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        import tempfile
        cpu_dump = os.path.join(tempfile.gettempdir(), f"dalib200_cpu_ref_{os.getpid()}.npy")
        cpu_baseline, cpu_sample = reference_arm(batch, cores, args.steps, args.warmup, dump=cpu_dump)

    # ------------------------------------------------------------------ our arm
    import torch
    import torch.distributed as dist
    from dali_b200 import capi
    from dali_b200.hotpath import ImagePipelineC2
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    capi.lib()       # fail loudly if the CUDA library is missing
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json)" if "hbm_gbs" in peaks else "fallback 6.65 TB/s (B200_PROFILING.md)"

    streams = make_batch(batch, 1000 * rank, min(cores, 16))
    # the encoded batch lives in page-locked HOST memory (the contract's "inputs from pinned host memory"), like the buffers of
    # the framework's own file reader; external_source(no_copy=True) lets the decoder DMA them without a host repack
    arena = capi.pinned_empty(sum((s.size + 63) & ~63 for s in streams))
    off, pinned_streams = 0, []
    for s in streams:
        v = arena[off:off + s.size]
        v[:] = s
        pinned_streams.append(v)
        off += (s.size + 63) & ~63
    streams = pinned_streams
    mirror = np.random.default_rng(rank).integers(0, 2, batch)
    J = float(np.mean([s.size for s in streams]))
    pipe = ImagePipelineC2(batch)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")        # > 126 MB L2

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident measurement ("value"): bytes staged and uploaded once, timed region = the kernels
    pipe.setup(streams, mirror)
    pipe.upload()
    for _ in range(args.warmup):
        pipe.launch()
    torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    capi.profiling(True)
    capi.profiling_collect()
    launches0 = capi.launch_count()
    sampler = ClockSampler(local_rank)
    barrier()
    sampler.start()
    t_wall0 = time.perf_counter()
    for a, b in ev:
        flush.fill_(1)                       # L2 flush between timed iterations (outside the per-step events)
        a.record()
        pipe.launch()
        b.record()
    barrier()
    t_wall = time.perf_counter() - t_wall0
    clocks = sampler.stop()
    launches = capi.launch_count() - launches0
    prof = capi.profiling_collect()
    capi.profiling(False)
    step_ms = [a.elapsed_time(b) for a, b in ev]
    # read after the timed steps: the decoder has no status before its first launch (--warmup 0)
    assert all(s == 0 for s in pipe.status()), "decoder reported a truncated stream"
    # the output of the last timed step, read before anything launches the pipeline again
    dumped = None
    if args.dump_outputs and rank == 0:
        keep = dump_sample(batch)
        dumped = {"c2_output": pipe.output[torch.from_numpy(keep).cuda()].float().cpu().numpy(),
                  "c2_output_sample_index": keep.astype(np.float64)}
    total_ms = float(sum(step_ms))
    if world > 1:
        t = torch.tensor([total_ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms = float(t.item())
    ms_per_step = total_ms / args.steps
    value = world * batch / (ms_per_step / 1e3)
    ms_median = float(np.median(step_ms))

    # ---- kernel breakdown (live, from the same timed region)
    agg = {}
    for name, ms in prof:
        a = agg.setdefault(name, [0.0, 0])
        a[0] += ms; a[1] += 1
    kernels = {k: {"ms_per_step": v[0] / args.steps, "launches_per_step": v[1] / args.steps} for k, v in agg.items()}
    dom = max(kernels, key=lambda k: kernels[k]["ms_per_step"]) if kernels else None
    # algorithmic bytes of each kernel per launch (DESIGN.md "kernels"): what the kernel must move at minimum
    coef_bytes = (H // 16 + (H % 16 > 0)) * (W // 16) * 6 * 64 * 2
    plane_bytes = coef_bytes // 2
    alg = {"jpeg_unstuff_count": J, "jpeg_unstuff_scatter": 2 * J, "jpeg_huff_sync_intra": J, "jpeg_huff_sync_walk1": 0.3 * J, "jpeg_huff_sync_walk2": 0.08 * J,
           "jpeg_huff_sync_walk3": 0.03 * J,
           "jpeg_huff_write": J + coef_bytes, "jpeg_dc_scan": 2 * coef_bytes / 64, "jpeg_idct": coef_bytes + plane_bytes,
           "jpeg_upsample_color": plane_bytes + ALG_DECODE, "resample_fused": ALG_RESIZE, "resample_stream": ALG_RESIZE, "cmn_hwc2chw": ALG_CMN,
           # decode -> resize without the RGB image: the 4:2:0 planes in (1.5 bytes per pixel), the resized image out
           "resample_planar": plane_bytes + OUT * OUT * 3}
    roofline = None
    if dom is not None:
        dur = kernels[dom]["ms_per_step"] / max(1.0, kernels[dom]["launches_per_step"]) / 1e3
        per_launch = alg.get(dom, 0) * batch
        ach = per_launch / dur / 1e9 if dur > 0 else 0.0
        traffic, traffic_src = None, None
        try:       # dram__bytes_read.sum + dram__bytes_write.sum of that kernel from the committed `ncu --set full` capture at batch 256
            tj = json.load(open(os.path.join(ROOT, "profiles", "r2_ncu_dram_traffic_batch256.json")))
            if tj.get("batch") == batch:
                traffic = tj["kernels"][dom]["dram_bytes_per_launch"]
                traffic_src = "profiles/r2_ncu_dram_traffic_batch256.json (ncu --set full, --clock-control none, batch 256, per launch)"
        except Exception:
            pass
        roofline = {"kernel": dom, "bound": "hbm", "achieved": ach, "peak": hbm_peak, "unit": "GB/s", "frac": ach / hbm_peak,
                    "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                    "share_of_step": kernels[dom]["ms_per_step"] / ms_per_step, "algorithmic_bytes_per_launch": per_launch}
    op_gbs = (J + ALG_DECODE + ALG_RESIZE + ALG_CMN) * batch / (ms_per_step / 1e3) / 1e9

    # ---- end to end through the PUBLIC API (pipeline_def + fn.*): host buffers in, per step: header parse + pinned staging +
    #      H2D + all kernels + D2H read of a result checksum
    from dali_b200 import fn, types, pipeline_def
    from dali_b200.hotpath import IMAGENET_MEAN, IMAGENET_STD
    mirror_samples = [np.array(m, np.int32) for m in mirror]

    e2e_depth = 3      # prefetch_queue_depth of the public API (reference default 2): three batches in flight hide the H2D copy

    @pipeline_def(batch_size=batch, num_threads=min(cores, 8), device_id=local_rank, prefetch_queue_depth=e2e_depth)
    def c2_pipeline():
        jpegs = fn.external_source(source=lambda i: streams, name="jpegs", no_copy=True)
        mir = fn.external_source(source=lambda i: mirror_samples, name="mirror")
        img = fn.decoders.image(jpegs, device="mixed", output_type=types.RGB)
        img = fn.resize(img, resize_x=OUT, resize_y=OUT)
        return fn.crop_mirror_normalize(img, dtype=types.FLOAT16, output_layout="CHW", crop=(OUT, OUT), mean=IMAGENET_MEAN,
                                        std=IMAGENET_STD, mirror=mir)
    api_pipe = c2_pipeline()
    api_pipe.build()

    def e2e_step():
        (out,) = api_pipe.run()
        t = torch.as_tensor(out.as_tensor(), device="cuda")
        return t, float(t[:, 0, 0, 0].float().sum().item())      # D2H read of a result scalar
    for _ in range(args.warmup):
        api_out, chk = e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        api_out, chk = e2e_step()
    barrier()
    e2e_s = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([e2e_s], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())
    # the public-API result must equal the device-resident path bit for bit
    api_equal = bool(torch.equal(api_out.view(torch.int16), pipe.launch().view(torch.int16)))
    e2e = {"value": world * batch * args.steps / e2e_s, "unit": "images/s", "h2d_bytes_per_step": int(pipe.staged_bytes) + 4 * batch,
           "d2h_bytes_per_step": 4, "ms_per_step": 1e3 * e2e_s / args.steps, "api": "dali_b200.pipeline_def + fn.external_source / "
           "fn.decoders.image(mixed) / fn.resize / fn.crop_mirror_normalize, Pipeline.run()", "prefetch_queue_depth": e2e_depth,
           "equals_device_resident_path": api_equal,
           "host_buffers": "page-locked host arena, fn.external_source(no_copy=True): the samples are copied by DMA from the caller's memory "
                           "(one cudaMemcpyBatchAsync submission per batch, no host repack)",
           "note": "host header parse + H2D + all kernels + D2H of a checksum scalar, per step"}

    # ---- parity of the timed configuration against the CPU reference path (reported, not timed)
    if cpu_baseline is not None:
        want = np.load(cpu_dump)
        os.remove(cpu_dump)
        got = pipe.run(streams, mirror)[:cpu_sample].cpu().numpy()
        cpu_baseline["parity_mismatching_elements"] = int((got.view(np.uint16) != want.view(np.uint16)).sum())
        cpu_baseline["parity_elements"] = int(want.size)

    secondary = None
    if rank == 0 and world == 1 and not args.no_secondary:
        del api_pipe
        try:
            secondary = secondary_workloads(hbm_peak, flush, args.steps, args.warmup)
        except Exception as ex:           # the headline line must not depend on the secondary workloads
            secondary = {"error": repr(ex)}
    # ---- optional consumer-side collective (BASELINE configs[4]): all-gather of the fp16 NCHW output of every rank over NVLink.
    #      Not part of `value` / `e2e` (each rank keeps its shard for training-style consumption); reported for the consumers that
    #      need the full batch.
    allgather = None
    if world > 1:
        from dali_b200.sharding import GatherBuffer
        gb = GatherBuffer((batch, 3, OUT, OUT), torch.float16, torch.device("cuda", local_rank))
        ref_local = pipe.launch().clone()
        pipe.bind_output(gb.local)                   # CMN now writes straight into this rank's slice of the gather buffer
        pipe.setup(streams, mirror); pipe.upload()
        pipe.launch()
        torch.cuda.synchronize()
        for _ in range(2):
            gb.all_gather()
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(5)]
        for a, b in evs:
            a.record(); gb.all_gather(); b.record()
        torch.cuda.synchronize()
        full = gb.full
        inplace_ok = bool(torch.equal(full[rank * batch:(rank + 1) * batch].view(torch.int16), ref_local.view(torch.int16)))
        t = torch.tensor([float(np.median([a.elapsed_time(b) for a, b in evs]))], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        gbytes = full.numel() * full.element_size() / 1e9
        allgather = {"ms": float(t.item()), "bytes_gathered_per_rank": int(full.numel() * full.element_size()),
                     "bus_GBps": gbytes * (world - 1) / world / (float(t.item()) / 1e3), "shape": list(full.shape),
                     "in_place": "CMN writes into recv + rank*count of a persistent buffer; one ncclAllGather, no staging copy",
                     "local_slice_equals_unbound_output": inplace_ok}
    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": "images/s", "n_gpus": world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "u8", "data": "synthetic", "config": config,
                "l2": "flushed between timed iterations (256 MiB write) and working set 1.6 GB > L2", "mean_jpeg_bytes": J,
                "ms_per_step_median": ms_median, "value_at_median": world * batch / (ms_median / 1e3),
                "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu_baseline,
                "kernels": kernels, "op_boundary_GBps": op_gbs, "op_boundary_frac_of_hbm": op_gbs / hbm_peak,
                "wall_s_timed_region": t_wall, "checksum": chk, "secondary": secondary, "allgather_fp16_nchw": allgather}
        print(json.dumps(line))
    if dumped is not None:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, arr in dumped.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), arr)
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())

#!/usr/bin/env python
"""Benchmark of the hot path: SS2D selective scan forward+backward, patch-tokens/s and % of the HBM roofline.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload NAME] [--no-extras] [--dump-outputs DIR]

The metric is quoted at two sequence lengths, so a STEP = one forward + one backward of the selective-scan op at BOTH of them:
L = 196 (224 x 224 images, 14 x 14 tokens; B = 148 / GPU) and L = 6400 (1280 x 1280, 80 x 80 tokens; B = 16 / GPU), with SS2D's
shapes (d_inner 768 -> R = 4 x 768 = 3072 scan rows, G = 4 B/C groups, d_state 1 = R2GenCSR's shipped VMamba config).  One
patch-token = one (image, position) over all R rows; `value` = patch-tokens of both halves / time of both halves (inputs
resident in HBM).  `--workload NAME` times a single workload instead.  `e2e` goes through the same C-ABI calls but starts from
pinned HOST buffers and ends with the results back in host memory (copies inside the timed region).
N > 1 (torchrun): pure data parallelism, per-GPU batch fixed (weak scaling).  The scan itself has no collective; the one
exchange of the path is DDP's gradient all-reduce of the model the scan sits in (VMamba-B / ARM-Base: 84 M parameters = 0.34 GB
fp32, DDP's 25 MB buckets, NCCL all-reduce issued asynchronously through medical_image_analysis_b200.dp).  A bench step is ONE
SS2D layer's scan, and VMamba-B runs 15 layers of exactly the headline shape (stage 3: 14 x 14 tokens, d_inner 768) per training
step, so the gradient set leaves at DDP's cadence: one bucket per step, round robin = 0.34 GB per 14 steps (`config.grad_exchange`).
The line also carries the stress variant -- the WHOLE 0.34 GB set all-reduced after EVERY scan step, 14 x the traffic of a real
step -- measured right after the timed region (`grad_exchange.every_step`) (DESIGN.md, multi-GPU).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

# name -> batch, rows, groups, L, d_state, out_f32 ("oflex": fp32 out / dout)
WORKLOADS = {
    # B = 148 = one image per SM: 148 x 96 = 14208 32-row batches = 12 full waves of the forward's 1184 resident warps
    # (at B = 64 the 5.2 waves of the forward cost 6: -11 %; SURVEY 8d: "B chosen to fill the GPU (e.g. 64-256)")
    "ss2d_m196_n1": dict(B=148, R=3072, G=4, L=196, N=1, out_f32=False),
    "ss2d_m196_n16": dict(B=64, R=3072, G=4, L=196, N=16, out_f32=False),
    "ss2d_m6400_n1": dict(B=16, R=3072, G=4, L=6400, N=1, out_f32=False),
    "ss2d_m6400_n1_b4": dict(B=4, R=3072, G=4, L=6400, N=1, out_f32=False),
    "ss2d_m6400_n16": dict(B=4, R=3072, G=4, L=6400, N=16, out_f32=False),
    "ss2d_m196_n1_o32": dict(B=64, R=3072, G=4, L=196, N=1, out_f32=True),
    "ss2d_m196_n16_o32": dict(B=64, R=3072, G=4, L=196, N=16, out_f32=True),
    # one scan of the ARM mixer at BASELINE configs[1] (MambaXray-VL-Base, SURVEY 8: R = 768 rows, L = 197 = 14 x 14 + cls,
    # one B/C group, d_state 16, z gate; arm/Finetuning/mamba_simple.py:693-704)
    "arm_m197_n16_z": dict(B=64, R=768, G=1, L=197, N=16, out_f32=False, z=True),
}
DEFAULT = "ss2d_m196_n1"
HEADLINE = ("ss2d_m196_n1", "ss2d_m6400_n1")     # the two halves of the metric; the default run times both in every step
GRAD_BUCKET_PARAMS = 84_000_000                  # ARM-Base / VMamba-B size (SURVEY 2.2): the DDP exchange of a real step
GRAD_BUCKET_MB = 25                              # DDP's default bucket_cap_mb -> 13 buckets
# One bench step = the scan of ONE SS2D layer; the model that owns the 84 M parameters runs 15 layers of the headline shape per
# training step (VMamba-B, depths [2, 2, 15, 2]: stage 3 = 14 x 14 tokens, d_model 384 -> d_inner 768;
# R2GenCSR/VMamba/classification/configs/vssm/vmambav2_base_224.yaml), so its gradient set is exchanged once per 15 scan steps,
# bucket by bucket as the backward walks the layers: ceil(13 / 15) = 1 bucket per step.
# The stress variant (all 13 buckets after EVERY scan step = 0.34 GB per 1.66 ms, which no training step of this model asks for)
# is measured too and reported next to it; at N = 2 / 4 it ran 2.04 / 2.54 ms per step with 100 MB buckets (gpurun r2z).
MODEL_SCAN_LAYERS = 15
GRAD_BUCKETS_PER_STEP = 1
METRIC = "patch-tokens/sec SS2D fwd+bwd at L=196/6400 D=768; % HBM roofline"


def bytes_per_token(w, es=2):
    """Algorithmic HBM bytes per patch-token (SURVEY.md 8d): every activation read/written exactly once."""
    R, G, N = w["R"], w["G"], w["N"]
    eso = 4 if w["out_f32"] else es
    fwd = (2 * R + 2 * G * N) * es + R * eso
    bwd = (2 * R + 2 * G * N) * es + R * eso + 2 * R * es + 2 * G * N * es
    if w.get("z"):   # SURVEY 8d: fwd also reads z; bwd also reads z and the saved out, and writes dz
        fwd += R * es
        bwd += 2 * R * es + R * es
    return fwd, bwd


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic(kind, workload, batch):
    """dram__bytes_read.sum + dram__bytes_write.sum of one launch of the `kind` ("fwd" / "bwd") kernel of `workload`, from the
    newest committed `ncu --set full` capture of this same command (profiles/*_ncu_summary.json, written by
    tools/ncu_summary.py); None if no capture is committed.  A capture taken at another per-GPU batch is scaled linearly (the
    traffic of these kernels is proportional to the batch) and says so."""
    import glob
    mult = {"Mbyte": 1e6, "Gbyte": 1e9, "Kbyte": 1e3, "byte": 1.0}
    for f in sorted(glob.glob(os.path.join(ROOT, "profiles", "*_ncu_summary.json")), reverse=True):
        try:
            full = json.load(open(f))
            w = full["workloads"][workload]
            d = full["launches"][w[kind]]
            rd, ru = d["dram__bytes_read.sum"].split()[:2]
            wr, wu = d["dram__bytes_write.sum"].split()[:2]
            cap_b = int(w["B"])
            src = os.path.basename(f) if cap_b == batch else f"{os.path.basename(f)} (captured at B={cap_b}, scaled by {batch}/{cap_b})"
            return (float(rd) * mult[ru] + float(wr) * mult[wu]) * batch / cap_b, src
        except Exception:
            continue
    return None, None


def make_inputs(w, device, seed=0, dtype=torch.bfloat16):
    """Reference generators (test_selective_scan.py:409-444)."""
    g = torch.Generator(device="cpu").manual_seed(seed)
    B, R, G, L, N = w["B"], w["R"], w["G"], w["L"], w["N"]
    A = -0.5 * torch.rand(R, N, generator=g)
    D = torch.randn(R, generator=g)
    bias = 0.5 * torch.rand(R, generator=g)
    gd = torch.Generator(device=device).manual_seed(seed)
    Bm = torch.randn(B, G, N, L, generator=gd, device=device).to(dtype)
    C = torch.randn(B, G, N, L, generator=gd, device=device).to(dtype)
    u = torch.randn(B, R, L, generator=gd, device=device).to(dtype)
    delta = (0.5 * torch.rand(B, R, L, generator=gd, device=device)).to(dtype)
    dout = torch.randn(B, R, L, generator=gd, device=device).to(torch.float32 if w["out_f32"] else dtype)
    z = torch.randn(B, R, L, generator=gd, device=device).to(dtype) if w.get("z") else None
    return dict(u=u, delta=delta, A=A.to(device), B=Bm, C=C, D=D.to(device), bias=bias.to(device), dout=dout, z=z)


DUMP_MAX_ELEMS = 1 << 20       # per array; larger outputs are dumped as a fixed sample (4 MB in float32)
DUMP_MAX_BYTES = 64 << 20      # all arrays of one dump together
GRAD_NAMES = ("du", "ddelta", "dA", "dB", "dC", "dD", "ddelta_bias", "dz")


def dump_outputs(path, names, results):
    """Writes what the caller of each workload's fwd + bwd receives -- out, the last scan state and every gradient -- as
    float32 `path/<workload>.<name>.npy`.  An array of more than DUMP_MAX_ELEMS elements is replaced by the elements at
    DUMP_MAX_ELEMS sorted flat indices drawn with a seed-0 generator, so equal shapes are always sampled at the same places
    and two builds can be compared array for array."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    arrays = {}
    for wname, (out, x, grads) in zip(names, results):
        named = [("out", out), ("last_state", x[:, :, -1, 1::2])] + list(zip(GRAD_NAMES, grads))
        for name, t in named:
            if t is None:
                continue
            flat = t.reshape(-1)
            if flat.numel() > DUMP_MAX_ELEMS:
                idx = torch.randint(flat.numel(), (DUMP_MAX_ELEMS,), generator=torch.Generator().manual_seed(0)).sort().values
                t = flat[idx.to(flat.device)]
            arrays[f"{wname}.{name}"] = t.float().cpu().numpy()
    total = sum(a.nbytes for a in arrays.values())
    assert total <= DUMP_MAX_BYTES, f"output dump of {total} bytes exceeds {DUMP_MAX_BYTES}"
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


class ClockSampler:
    """SM clock / throttle reasons sampled DURING the timed region (B200_PROFILING.md): NVML polled every ~2 ms from a
    background thread (the timed region is only a few ms long, too short for `nvidia-smi -lms`)."""

    def __init__(self, index):
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._stop = False
        self._thread = None

    def _loop(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            # torchrun / CUDA_VISIBLE_DEVICES: map the logical index to the physical device through its UUID
            uuid = torch.cuda.get_device_properties(self.index).uuid
            try:
                h = nv.nvmlDeviceGetHandleByUUID(("GPU-" + str(uuid)).encode())
            except Exception:
                h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
            bits = {"hw_slowdown": nv.nvmlClocksEventReasonHwSlowdown if hasattr(nv, "nvmlClocksEventReasonHwSlowdown") else 0x8,
                    "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}
            while not self._stop:
                self.samples.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for name, bit in bits.items():
                    if r & bit:
                        self.reasons.add(name)
                time.sleep(0.002)
        except Exception as e:   # report, never hide
            self.reasons.add(f"sampler_error:{type(e).__name__}")

    def start(self):
        import threading
        self._thread = threading.Thread(target=self._loop, daemon=True)
        self._thread.start()

    def mark(self):
        """Only samples taken after this call (the start of the timed region) are reported."""
        self._mark = len(self.samples)

    def stop(self):
        self._stop = True
        if self._thread is not None:
            self._thread.join(timeout=2)
        smp = self.samples[getattr(self, "_mark", 0):] or self.samples
        out = {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(smp)}
        if smp:
            out["sm_mhz"] = statistics.median(smp)
        return out


def run_device_steps(inps, steps, warmup, dist_grads=None, last_outputs=None):
    """K timed steps on resident inputs; a step = fwd + bwd of every workload in `inps` (a list), then the gradient exchange.
    Returns (total_ms, [fwd_ms_avg per workload], [bwd_ms_avg per workload]).  If `last_outputs` is a list, the results of
    the last step are appended to it, one (out, x, grads) per workload."""
    from medical_image_analysis_b200 import scan_bwd, scan_fwd
    if isinstance(inps, dict):
        inps = [inps]
    nw = len(inps)

    def one(ev=None, last=False, keep=None):
        g = None
        for wi, inp in enumerate(inps):
            out_f32 = inp["dout"].dtype == torch.float32 and inp["u"].dtype != torch.float32
            if ev:
                ev[3 * wi].record()
            z = inp.get("z")
            out, x, _, hblk = scan_fwd(inp["u"], inp["delta"], inp["A"], inp["B"], inp["C"], inp["D"], z, inp["bias"], True, out_f32,
                                       want_block_states=True)
            if ev:
                ev[3 * wi + 1].record()
            g = scan_bwd(inp["u"], inp["delta"], inp["A"], inp["B"], inp["C"], inp["D"], z, inp["bias"], inp["dout"], x,
                         out if z is not None else None, True, hblk=hblk)
            if ev:
                ev[3 * wi + 2].record()
            if keep is not None:
                keep.append((out, x, g))
        if dist_grads is not None:
            dist_grads(g, last)
        if ev:
            ev[3 * nw].record()

    for k in range(warmup):
        one(None, k == warmup - 1)
    evs = [[torch.cuda.Event(enable_timing=True) for _ in range(3 * nw + 1)] for _ in range(steps)]
    torch.cuda.synchronize()
    for k in range(steps):
        one(evs[k], k == steps - 1, last_outputs if k == steps - 1 else None)
    torch.cuda.synchronize()
    total = evs[0][0].elapsed_time(evs[-1][3 * nw])
    fwd = [sum(e[3 * wi].elapsed_time(e[3 * wi + 1]) for e in evs) / steps for wi in range(nw)]
    bwd = [sum(e[3 * wi + 1].elapsed_time(e[3 * wi + 2]) for e in evs) / steps for wi in range(nw)]
    return total, fwd, bwd


def run_e2e_steps(w, inp, steps, warmup, n_slices=4):
    """Same C-ABI calls, but every step starts from pinned HOST buffers and ends with the results in host memory.
    The batch is cut into slices that flow through three streams (H2D -> fwd+bwd -> D2H) so that the two PCIe
    directions and the kernels overlap; every byte of every step still crosses the bus inside the timed region."""
    from medical_image_analysis_b200 import scan_bwd, scan_fwd
    out_f32 = w["out_f32"]
    names = ("u", "delta", "B", "C", "dout")
    B = w["B"]
    n_slices = max(1, min(n_slices, B))
    bounds = [(i * B // n_slices, (i + 1) * B // n_slices) for i in range(n_slices)]
    host_in = {k: inp[k].cpu().pin_memory() for k in names}
    dev_in = {k: torch.empty_like(inp[k]) for k in names}
    h2d = sum(t.numel() * t.element_size() for t in host_in.values())
    s_in, s_cmp, s_out = torch.cuda.Stream(), torch.cuda.Stream(), torch.cuda.Stream()
    host_out = {}
    d2h = 0
    keep = []
    prev_cmp = [None] * n_slices      # the compute that last read slice i: its inputs may only be overwritten afterwards

    def one(first=False):
        nonlocal d2h
        keep.clear()
        if first:
            d2h = 0
        for si, (lo, hi) in enumerate(bounds):
            ev_in = torch.cuda.Event()
            with torch.cuda.stream(s_in):
                if prev_cmp[si] is not None:
                    s_in.wait_event(prev_cmp[si])
                for k in names:
                    dev_in[k][lo:hi].copy_(host_in[k][lo:hi], non_blocking=True)
                ev_in.record()
            ev_cmp = torch.cuda.Event()
            with torch.cuda.stream(s_cmp):
                s_cmp.wait_event(ev_in)
                sl = {k: dev_in[k][lo:hi] for k in names}
                out, x, _, hblk = scan_fwd(sl["u"], sl["delta"], inp["A"], sl["B"], sl["C"], inp["D"], None, inp["bias"], True, out_f32,
                                           want_block_states=True)
                g = scan_bwd(sl["u"], sl["delta"], inp["A"], sl["B"], sl["C"], inp["D"], None, inp["bias"], sl["dout"], x, None, True, hblk=hblk)
                res = [out] + [t for t in g if t is not None]
                ev_cmp.record()
            prev_cmp[si] = ev_cmp
            keep.append(res)
            with torch.cuda.stream(s_out):
                s_out.wait_event(ev_cmp)
                for j, t in enumerate(res):
                    key = (si, j)
                    if key not in host_out:
                        host_out[key] = torch.empty(t.shape, dtype=t.dtype).pin_memory()
                    if first:
                        d2h += t.numel() * t.element_size()
                    host_out[key].copy_(t, non_blocking=True)
                    t.record_stream(s_out)

    cur = torch.cuda.current_stream()
    one(first=True)
    for _ in range(max(0, warmup - 1)):
        one()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(cur)
    for s_ in (s_in, s_cmp, s_out):
        s_.wait_stream(cur)
    for _ in range(steps):
        one()
    for s_ in (s_in, s_cmp, s_out):
        cur.wait_stream(s_)
    e1.record(cur)
    torch.cuda.synchronize()
    return e0.elapsed_time(e1), h2d, d2h


def aux_kernels(dev, peak_gbs, n=20):
    """The smaller kernels of the path (SURVEY 8f): depth-wise causal conv1d + SiLU of the Mamba mixers and SS2D's
    CrossScan / CrossMerge, timed as `n` back-to-back C-ABI launches on resident bf16 tensors (CUDA events), reported as
    algorithmic GB/s (every tensor read or written once) and fraction of the measured HBM peak."""
    from medical_image_analysis_b200 import _lib
    L_ = _lib.lib()
    st = torch.cuda.current_stream(dev).cuda_stream
    out = []

    def timed(fn):
        for _ in range(3):
            assert fn() == 0
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / n

    B, D, L = 64, 1536, 196                                      # ARM mixer: d_inner 1536, 14 x 14 tokens
    x = torch.randn(B, D, L, device=dev).bfloat16()
    y, dy, dx = torch.empty_like(x), torch.randn_like(x), torch.empty_like(x)
    w, b = torch.randn(D, 4, device=dev), torch.randn(D, device=dev)
    dw, db = torch.empty_like(w), torch.empty_like(b)
    nbytes = x.numel() * 2
    t = timed(lambda: L_.mia_causal_conv1d_fwd(x.data_ptr(), w.data_ptr(), b.data_ptr(), y.data_ptr(), B, D, L, 4, 1, 2, D * L, L, D * L, L, st))
    out.append({"kernel": "causal_conv1d_fwd (B=64, D=1536, L=196, k=4, silu, bf16)", "us": t * 1e3, "gbs": 2 * nbytes / t / 1e6})
    t = timed(lambda: L_.mia_causal_conv1d_bwd(x.data_ptr(), w.data_ptr(), b.data_ptr(), dy.data_ptr(), dx.data_ptr(), dw.data_ptr(),
                                               db.data_ptr(), B, D, L, 4, 1, 2, D * L, L, D * L, L, D * L, L, st))
    out.append({"kernel": "causal_conv1d_bwd (same shape)", "us": t * 1e3, "gbs": 3 * nbytes / t / 1e6})
    B, C, H, W = 64, 768, 14, 14                                 # SS2D: d_inner 768, 14 x 14
    xi = torch.randn(B, C, H, W, device=dev).bfloat16()
    xs = torch.empty(B, 4, C, H * W, device=dev, dtype=torch.bfloat16)
    yo = torch.empty(B, C, H * W, device=dev, dtype=torch.bfloat16)
    nb = xi.numel() * 2
    t = timed(lambda: L_.mia_cross_scan(xi.data_ptr(), xs.data_ptr(), B, C, H, W, 2, st))
    out.append({"kernel": "cross_scan (B=64, C=768, 14x14, bf16)", "us": t * 1e3, "gbs": 5 * nb / t / 1e6})
    t = timed(lambda: L_.mia_cross_merge(xs.data_ptr(), yo.data_ptr(), B, C, H, W, 2, st))
    out.append({"kernel": "cross_merge (same shape)", "us": t * 1e3, "gbs": 5 * nb / t / 1e6})
    w9, dw9 = torch.randn(C, 9, device=dev), torch.empty(C, 9, device=dev)
    bc, dbc = torch.randn(C, device=dev), torch.empty(C, device=dev)
    y2, dy2, dx2 = torch.empty_like(xi), torch.randn_like(xi), torch.empty_like(xi)
    t = timed(lambda: L_.mia_dwconv2d_fwd(xi.data_ptr(), w9.data_ptr(), bc.data_ptr(), y2.data_ptr(), B, C, H, W, 1, 2, st))
    out.append({"kernel": "dwconv2d_3x3_silu_fwd (B=64, C=768, 14x14, bf16)", "us": t * 1e3, "gbs": 2 * nb / t / 1e6})
    t = timed(lambda: L_.mia_dwconv2d_bwd(xi.data_ptr(), w9.data_ptr(), bc.data_ptr(), dy2.data_ptr(), dx2.data_ptr(), dw9.data_ptr(),
                                          dbc.data_ptr(), B, C, H, W, 1, 2, st))
    out.append({"kernel": "dwconv2d_3x3_silu_bwd (same shape)", "us": t * 1e3, "gbs": 3 * nb / t / 1e6})
    try:   # the library path the reference takes for the same op (VERDICT r1 hygiene): cuDNN depth-wise conv + a SiLU kernel
        import torch.nn.functional as F
        w4 = w9.view(C, 1, 3, 3).to(torch.bfloat16)
        b4 = bc.to(torch.bfloat16)
        t = timed(lambda: (F.silu(F.conv2d(xi, w4, b4, padding=1, groups=C)), 0)[1])
        out.append({"kernel": "library: F.silu(F.conv2d(groups=C)) forward, same shape (cuDNN + elementwise)", "us": t * 1e3, "gbs": 2 * nb / t / 1e6})
    except Exception as e:
        out.append({"kernel": "library dwconv2d comparison", "error": repr(e)})
    for o in out:
        if "gbs" not in o:
            continue
        o["hbm_frac"] = o["gbs"] / peak_gbs
    return out


def module_timings(dev, peak_gbs, peak_tf, n=10):
    """Module-level numbers through the autograd surface (VERDICT r1 #5): fwd + bwd under bf16 autocast, loss = out.float().sum()
    like the reference's speed test (test_selective_scan_speed.py:511).  tokens/s = images x tokens / time."""
    from medical_image_analysis_b200.arm import arm_base_pz16
    from medical_image_analysis_b200.mae import SmallPatchEmbed
    from medical_image_analysis_b200.vmamba import SS2D
    out = []

    def timed(step):
        for _ in range(3):
            step()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            step()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / n

    def fb(m, x):
        def step():
            for p in m.parameters():
                p.grad = None
            with torch.autocast("cuda", dtype=torch.bfloat16):
                y = m(x)
            y.float().sum().backward()
        return step

    for name, B, H in (("SS2D(d_model=384, ssm_ratio=2, d_state=1, v3noz) 14x14", 64, 14), ("same, 80x80", 4, 80)):
        try:
            m = SS2D(d_model=384, ssm_ratio=2.0, d_state=1, forward_type="v3noz").to(dev)
            x = torch.randn(B, H, H, 384, device=dev, requires_grad=True)
            ms = timed(fb(m, x))
            out.append({"module": name, "B": B, "ms_fwd_bwd": ms, "patch_tokens_per_s": B * H * H / (ms * 1e-3)})
            del m, x
        except Exception as e:  # report, never hide
            out.append({"module": name, "error": repr(e)})
    try:   # BASELINE configs[1]: MambaXray-VL-Base encoder (12 x (4-direction Mamba mixer + SwiGLU), L = 197, D = 768)
        m = arm_base_pz16(drop_path_rate=0.0).to(dev)
        x = torch.randn(32, 3, 224, 224, device=dev)
        ms = timed(fb(m, x))
        out.append({"module": "arm_base_pz16 encoder fwd+bwd, 224x224 (BASELINE configs[1])", "B": 32, "ms_fwd_bwd": ms,
                    "patch_tokens_per_s": 32 * 196 / (ms * 1e-3), "images_per_s": 32 / (ms * 1e-3)})
        del m, x
    except Exception as e:
        out.append({"module": "arm_base_pz16", "error": repr(e)})
    try:   # BASELINE configs[2] patch encode: 17.6 GFLOP forward per 1280 x 1280 image, x3 with the two backward GEMMs
        B = 8
        m = SmallPatchEmbed(1, 1024, 1024).to(dev)
        x = torch.randn(B, 1, 1280, 1280, device=dev)
        ms = timed(fb(m, x))
        with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):
            ms_f = timed(lambda: m(x))
        fl = 2.0 * B * (6400 * 256 * 1024 + 400 * 16384 * 1024 + 400 * 1024 * 1024)
        out.append({"module": "SmallPatchEmbed(1, 1024, 1024) 1280x1280 (BASELINE configs[2] patch encode)", "B": B, "ms_fwd": ms_f,
                    "ms_fwd_bwd": ms, "patch_tokens_per_s": B * 6400 / (ms * 1e-3), "fwd_tflops": fl / ms_f / 1e9,
                    "fwd_frac_of_measured_bf16_peak": fl / ms_f / 1e9 / peak_tf})
        del m, x
    except Exception as e:
        out.append({"module": "SmallPatchEmbed", "error": repr(e)})
    torch.cuda.empty_cache()
    return out


def cpu_reference_run(w, steps, warmup, budget_s=150.0):
    """The reference's own CPU algorithm (oracle/selective_scan_ref.py = restatement of selective_scan_ref +
    torch autograd, all host threads) on a BOUNDED sample of the workload: one image (B=1), and if K steps of
    that would not fit the time budget, a leading subset of the rows (rows are independent; the figure is
    scaled by rows/R because a patch-token spans all R rows)."""
    from oracle.selective_scan_ref import selective_scan_ref_fwd_bwd
    R, G, L, N = w["R"], w["G"], w["L"], w["N"]
    Ls = min(L, 196 * 2)   # the oracle's autograd backward is O(L^2): cap the sequence, tokens/s stays per token
    g = torch.Generator().manual_seed(0)

    def mk(rows):
        rg = rows // G
        A = -0.5 * torch.rand(rows, N, generator=g)
        Bm = torch.randn(1, G, N, Ls, generator=g)
        C = torch.randn(1, G, N, Ls, generator=g)
        D = torch.randn(rows, generator=g)
        bias = 0.5 * torch.rand(rows, generator=g)
        u = torch.randn(1, rows, Ls, generator=g)
        delta = 0.5 * torch.rand(1, rows, Ls, generator=g)
        dout = torch.randn(1, rows, Ls, generator=g)
        assert rg * G == rows
        return (u, delta, A, Bm, C, D, None, bias, True, dout)

    rows = R
    probe_rows = min(R, 4 * G * 64)
    probe = mk(probe_rows)
    # "all the host threads it can use": torch's intra-op pool scales badly past the physical cores on this op (many small
    # element-wise kernels per token), so time a probe at a few pool sizes and keep the fastest -- the baseline gets its
    # best configuration, not the largest one
    ncpu = os.cpu_count() or 1
    best_t, best_n = None, None
    for n in sorted({ncpu, max(1, ncpu // 2), max(1, ncpu // 4), min(ncpu, 32), min(ncpu, 16), min(ncpu, 8)}, reverse=True):
        torch.set_num_threads(n)
        selective_scan_ref_fwd_bwd(*probe)                        # warms torch's thread pool up
        t0 = time.perf_counter()
        selective_scan_ref_fwd_bwd(*probe)
        t = time.perf_counter() - t0
        if best_t is None or t < best_t:
            best_t, best_n = t, n
    torch.set_num_threads(best_n)
    t_probe = best_t
    est = t_probe * R / probe_rows
    while rows > G * 8 and est * (steps + warmup) * rows / R > budget_s:
        rows //= 2
    args = mk(rows)
    for _ in range(warmup):
        selective_scan_ref_fwd_bwd(*args)
    t0 = time.perf_counter()
    for _ in range(steps):
        selective_scan_ref_fwd_bwd(*args)
    dt = time.perf_counter() - t0
    value = steps * Ls * (rows / R) / dt
    sample = f"B=1, L={Ls}, rows={rows}/{R} (value scaled by rows/R), d_state={N}, fp32, {steps} steps"
    return value, dt * 1e3 / steps, sample, torch.get_num_threads()


def _numa_local_affinity(index):
    """Best effort: run this process (hence first-touch its pinned buffers) on the CPUs of the GPU's NUMA node, so that the e2e
    copies do not cross the inter-socket link (VERDICT r1: 19.6 vs 44 GB/s between boxes).  Returns a description."""
    try:
        bus = None
        try:
            pr = torch.cuda.get_device_properties(index)
            bus = "%04x:%02x:%02x.0" % (int(pr.pci_domain_id), int(pr.pci_bus_id), int(pr.pci_device_id))
        except Exception:
            import pynvml as nv
            nv.nvmlInit()
            uuid = str(torch.cuda.get_device_properties(index).uuid)
            h = nv.nvmlDeviceGetHandleByUUID(("GPU-" + uuid).encode())
            info = nv.nvmlDeviceGetPciInfo(h)
            raw = getattr(info, "busId", None) or getattr(info, "busIdLegacy")
            bus = (raw.decode() if isinstance(raw, bytes) else str(raw)).lower()
            if len(bus.split(":")[0]) == 8:
                bus = bus[4:]
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read().strip())
        if node < 0:
            return "numa_node unknown (-1): affinity unchanged"
        cpus = open(f"/sys/devices/system/node/node{node}/cpulist").read().strip()
        ids = set()
        for part in cpus.split(","):
            a, _, b = part.partition("-")
            ids.update(range(int(a), int(b or a) + 1))
        ids &= os.sched_getaffinity(0)
        if ids:
            os.sched_setaffinity(0, ids)
            return f"pinned to NUMA node {node} ({len(ids)} cpus)"
        return f"NUMA node {node} has no allowed cpu: affinity unchanged"
    except Exception as e:
        return f"affinity unchanged ({type(e).__name__})"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="headline", choices=["headline"] + sorted(WORKLOADS))
    ap.add_argument("--no-extras", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-modules", action="store_true")
    ap.add_argument("--batch", type=int, default=0, help="override the per-GPU batch (single-workload runs)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step to DIR/<workload>.<name>.npy "
                                                          "(float32, large arrays as a fixed sample; rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the CUDA path (--impl b200)")
    names = list(HEADLINE) if args.workload == "headline" else [args.workload]
    ws = [dict(WORKLOADS[n]) for n in names]
    if args.batch > 0 and len(ws) == 1:
        ws[0]["B"] = args.batch
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    bpt = [bytes_per_token(w) for w in ws]
    tokens = [w["B"] * w["L"] for w in ws]                    # per GPU and step
    desc = " + ".join(f"{n} (B={w['B']}/GPU, L={w['L']}, d_state={w['N']}{', z gate' if w.get('z') else ''}, bf16 in, "
                      f"{'fp32' if w['out_f32'] else 'bf16'} out/dout)" for n, w in zip(names, ws))
    config = {"workload": f"selective scan fwd+bwd, R=3072 (K=4 x d_inner 768), G=4: {desc}" if args.workload == "headline" or ws[0]["R"] == 3072
              else f"selective scan fwd+bwd: {desc}, R={ws[0]['R']}, G={ws[0]['G']}",
              "patch_tokens_per_step_per_gpu": sum(tokens), "bytes_per_token": [f + b for f, b in bpt],
              "l2": "working set > L2 (no flush needed)", "parallelism": f"dp{world}",
              "grad_exchange": f"N > 1: DDP gradient set of the model ({GRAD_BUCKET_PARAMS / 1e6:.0f} M fp32 = {GRAD_BUCKET_PARAMS * 4 / 1e9:.2f} GB) in "
                               f"{GRAD_BUCKET_MB} MB buckets, {GRAD_BUCKETS_PER_STEP} bucket per scan step round robin (a step = one of the "
                               f"model's {MODEL_SCAN_LAYERS} SS2D layers of this shape); stress variant (whole set every step) in grad_exchange.every_step",
              "compute": "fp32 scan arithmetic on bf16 activations (dtype key = arithmetic type)"}

    if args.impl == "reference":
        # the reference's CPU path (its selective_scan_ref) on the host cores; rank 0 only
        if rank != 0:
            return
        steps = max(1, args.steps)
        torch.set_num_threads(os.cpu_count() or 1)     # torchrun exports OMP_NUM_THREADS=1: use every host core
        per = []
        for w in ws:
            v, ms, sample, cores = cpu_reference_run(w, steps, max(0, args.warmup), budget_s=150.0 / len(ws))
            per.append((v, ms, sample, cores))
        # the same token mix as the B200 arm: time per step = sum_i tokens_i / value_i
        t_step = sum(t / p[0] for t, p in zip(tokens, per))
        value = sum(tokens) / t_step
        sample = " | ".join(p[2] for p in per)
        line = {"impl": "reference", "metric": METRIC, "value": value, "unit": "patch-tokens/s", "n_gpus": args.gpus, "steps": steps,
                "warmup": max(0, args.warmup), "ms_per_step": t_step * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic", "config": config,
                "cpu_baseline": {"value": value, "unit": "patch-tokens/s", "cores": per[0][3], "kind": "port", "sample": sample},
                "e2e": {"value": value, "unit": "patch-tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return

    assert torch.cuda.is_available(), "bench.py needs a CUDA device (use --impl reference for the CPU arm)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    numa = _numa_local_affinity(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        # NCCL's kernels on a HIGH-priority stream: the scan kernels fill every SM with queued one-warp CTAs, so a collective
        # launched next to them only advances when its CTAs win the block scheduler (without it the 0.34 GB exchange did not
        # overlap at all: gpurun r2z, N = 2, 2.43 ms / step against 1.66 ms at N = 1)
        # (stdout is parked on stderr while NCCL comes up: it prints its version banner there, and this script's stdout is ONE
        # JSON line)
        sys.stdout.flush()
        saved_stdout = os.dup(1)
        os.dup2(2, 1)
        try:
            try:
                opts = dist.ProcessGroupNCCL.Options(is_high_priority_stream=True)
                if os.environ.get("MIA_BENCH_NCCL_MAX_CTAS"):
                    opts.config.max_ctas = int(os.environ["MIA_BENCH_NCCL_MAX_CTAS"])
                dist.init_process_group("nccl", device_id=dev, pg_options=opts)
            except Exception:                                        # older constructor signatures
                dist.init_process_group("nccl", device_id=dev)
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_stdout, 1)
            os.close(saved_stdout)
    from medical_image_analysis_b200 import _lib, dp

    inps = [make_inputs(w, dev, seed=rank + 17 * i) for i, w in enumerate(ws)]
    dist_grads = None
    exchange = None
    if world > 1:
        # DDP's gradient step for the model the scan sits in: ARM-Base-sized fp32 gradients (the scan's own dA / dD / dbias are
        # its first elements) in 25 MB buckets, all-reduced asynchronously so that they overlap the next step (as DDP
        # overlaps its buckets with the rest of the backward); the last step's exchange completes inside the timed region
        exchange = dp.BucketedGradExchange(GRAD_BUCKET_PARAMS, dev, bucket_bytes=int(os.environ.get("MIA_BENCH_BUCKET_MB", str(GRAD_BUCKET_MB))) << 20,
                                           buckets_per_step=GRAD_BUCKETS_PER_STEP)

        def dist_grads(g, last=False):
            exchange.step([g[2], g[5], g[6]], wait=last)
    sampler = ClockSampler(local_rank)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    sampler.start()
    # a dump keeps the last step's outputs alive while the step still allocates; the warm-up keeps its last step's too, so
    # that the memory this takes is already in the caching allocator and the timed step does not have to ask the driver
    dump = rank == 0 and args.dump_outputs
    run_device_steps(inps, max(3, args.warmup), 0, dist_grads, [] if dump else None)   # warm-up (>= 3 steps), also the sustained pre-roll
    time.sleep(0.02)
    sampler.mark()
    launches0 = _lib.launch_count()
    if world > 1:
        dist.barrier()
    last_outputs = [] if dump else None
    total_ms, fwd_ms, bwd_ms = run_device_steps(inps, args.steps, 0, dist_grads, last_outputs)
    launches = _lib.launch_count() - launches0
    clocks = sampler.stop()
    if dump:
        dump_outputs(args.dump_outputs, names, last_outputs)
        del last_outputs
    total_ms = dp.max_over_ranks(total_ms, dev)
    value = sum(tokens) * world * args.steps / (total_ms * 1e-3)

    # ---- end to end: host buffers in, host buffers out (the L = 196 half: the PCIe-bound part is per token the same)
    e2e_steps = max(3, min(args.steps, 10))
    e2e_ms, h2d, d2h = run_e2e_steps(ws[0], inps[0], e2e_steps, 2)
    e2e_ms = dp.max_over_ranks(e2e_ms, dev)
    e2e_value = tokens[0] * world * e2e_steps / (e2e_ms * 1e-3)

    # the exchange alone (outside the timed region, EVERY rank takes part): achieved all-reduce bus bandwidth of this box; and
    # the stress variant: the same K steps with the WHOLE gradient set all-reduced after every scan step (100 MB buckets: the
    # better of the bucket sizes measured for it)
    exchange_alone, stress = {}, {}
    if exchange is not None:
        exchange_alone = exchange.measure_alone(dev)
        ex_all = dp.BucketedGradExchange(GRAD_BUCKET_PARAMS, dev, bucket_bytes=100 << 20)
        exchange.drain()
        run_device_steps(inps, 2, 0, lambda g, last=False: ex_all.step([g[2], g[5], g[6]], wait=last))
        dist.barrier()
        s_ms, _, _ = run_device_steps(inps, args.steps, 0, lambda g, last=False: ex_all.step([g[2], g[5], g[6]], wait=last))
        s_ms = dp.max_over_ranks(s_ms, dev)
        stress = {"every_step": {"value": sum(tokens) * world * args.steps / (s_ms * 1e-3), "ms_per_step": s_ms / args.steps,
                                 "bytes_per_step": ex_all.model_bytes, "bucket_mb": 100,
                                 "note": "whole gradient set all-reduced after EVERY scan step (not the headline: %dx a real step's traffic)"
                                         % exchange.report()["steps_per_gradient_set"]}}
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peak, peak_src = peaks()
    peak_tf = 1671.8
    try:
        peak_tf = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["bf16_tflops"])
    except Exception:
        pass
    per = []
    for n, w, tk, (fb_, bb_), f_ms, b_ms in zip(names, ws, tokens, bpt, fwd_ms, bwd_ms):
        fg, bg = tk * fb_ / (f_ms * 1e-3) / 1e9, tk * bb_ / (b_ms * 1e-3) / 1e9
        per.append({"workload": n, "B": w["B"], "L": w["L"], "d_state": w["N"], "patch_tokens_per_s": tk / ((f_ms + b_ms) * 1e-3),
                    "fwd_ms": f_ms, "bwd_ms": b_ms,
                    "fwd": {"achieved": fg, "frac": fg / peak, "algorithmic_bytes_per_launch": tk * fb_, "traffic": ncu_traffic("fwd", n, w["B"])[0]},
                    "bwd": {"achieved": bg, "frac": bg / peak, "algorithmic_bytes_per_launch": tk * bb_, "traffic": ncu_traffic("bwd", n, w["B"])[0]},
                    "step_frac": tk * (fb_ + bb_) / ((f_ms + b_ms) * 1e-3) / 1e9 / peak})
    dom = max(range(len(ws)), key=lambda i: bwd_ms[i])          # dominant kernel = the backward call with the largest time share
    step_bytes = sum(tk * (f + b) for tk, (f, b) in zip(tokens, bpt))
    step_gbs = step_bytes / (total_ms / args.steps * 1e-3) / 1e9
    bwd_kernel = {1: "ss_bwd_cw_kernel<bf16> (column-walk, scan_bwd_cw.cuh)", 16: "ss_bwd_rowsn_kernel<bf16>"}
    traffic, traffic_src = ncu_traffic("bwd", names[dom], ws[dom]["B"])
    roofline = {"bound": "hbm",
                "kernel": "backward C-ABI call of %s = %s + ss_finalize_kernel (timed together, CUDA events in the timed region)"
                          % (names[dom], bwd_kernel.get(ws[dom]["N"], "ss_bwd_kernel")),
                "achieved": per[dom]["bwd"]["achieved"], "peak": peak, "unit": "GB/s", "frac": per[dom]["bwd"]["frac"],
                "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": per[dom]["bwd"]["algorithmic_bytes_per_launch"],
                "per_workload": per,
                "step": {"achieved": step_gbs, "frac": step_gbs / peak, "roofline_tokens_per_s": peak * 1e9 * sum(tokens) / step_bytes}}
    line = {"metric": METRIC, "value": value, "unit": "patch-tokens/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": config, "clocks": clocks, "gpu_launches": int(launches),
            "e2e": {"value": e2e_value, "unit": "patch-tokens/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "workload": names[0], "host_affinity": numa},
            "roofline": roofline}
    if exchange is not None:
        line["grad_exchange"] = exchange.report()
        line["grad_exchange"].update(exchange_alone)
        line["grad_exchange"].update(stress)

    if not args.no_extras and world == 1:
        extras = []
        for name, ww in WORKLOADS.items():
            if name in names:
                continue
            try:
                i2 = make_inputs(ww, dev, seed=1)
                run_device_steps(i2, 3, 0)
                tms, f_ms, b_ms = run_device_steps(i2, 10, 0)
                fb, bb = bytes_per_token(ww)
                v = ww["B"] * ww["L"] * 10 / (tms * 1e-3)
                extras.append({"workload": name, "B": ww["B"], "value": v, "ms_per_step": tms / 10, "fwd_ms": f_ms[0], "bwd_ms": b_ms[0],
                               "bytes_per_token": fb + bb, "hbm_frac": v * (fb + bb) / 1e9 / peak})
                if ww["N"] > 1:
                    # d_state > 1 is bound by the MUFU (XU) pipe and instruction issue, not by HBM (SURVEY 8d asks for that share next
                    # to the HBM share): the forward needs N exp2 for a = 2^(m A_n) + 2 for the softplus per row-token (+ 2 for
                    # silu(z)), the SM retires 16 MUFU lanes per clock -> floor = row-tokens x MUFU / (16 x SMs x clock)
                    mufu = ww["N"] + 2 + (2 if ww.get("z") else 0)
                    sms = torch.cuda.get_device_properties(dev).multi_processor_count
                    mhz = (clocks or {}).get("sm_mhz") or 1965.0
                    floor_ms = ww["B"] * ww["R"] * ww["L"] * mufu / (16.0 * sms * mhz * 1e6) * 1e3
                    extras[-1].update({"fwd_mufu_per_row_token": mufu, "fwd_mufu_floor_ms": floor_ms, "fwd_xu_pipe_frac": floor_ms / f_ms[0],
                                       "bwd_xu_pipe_frac_ncu": 0.26 if name == "ss2d_m196_n16" else None,
                                       "bwd_xu_source": "profiles/r2b_ncu_bwd_rowsn.json (sm__inst_executed_pipe_xu 26.1 %, issue-active 61.1 %)"
                                       if name == "ss2d_m196_n16" else None})
                del i2
                torch.cuda.empty_cache()
            except Exception as e:  # report, never hide
                extras.append({"workload": name, "error": repr(e)})
        line["extra_workloads"] = extras
        try:
            line["aux_kernels"] = aux_kernels(dev, peak)
        except Exception as e:  # report, never hide
            line["aux_kernels"] = {"error": repr(e)}
    if not args.no_modules and world == 1:
        try:
            line["modules"] = module_timings(dev, peak, peak_tf)
        except Exception as e:  # report, never hide
            line["modules"] = {"error": repr(e)}

    if not args.no_cpu and world == 1:               # (the CPU baseline is a rank-0, N = 1 figure)
        torch.set_num_threads(os.cpu_count() or 1)
        cv, cms, sample, cores = cpu_reference_run(ws[0], 2, 0, budget_s=20.0)
        line["cpu_baseline"] = {"value": cv, "unit": "patch-tokens/s", "cores": cores, "kind": "port", "sample": sample}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()

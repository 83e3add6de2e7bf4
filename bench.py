#!/usr/bin/env python
"""bench.py — view-frames/sec of the V3D denoising hot path (EulerEDMSampler -> VideoUNet -> VideoDecoder).

    python bench.py --gpus N --steps K --warmup W            # B200-native arm (this repo's kernels)
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU path (oracle port) on host cores

One "step" = the whole hot path for one image: T=18 views, 512x512 (latent 4x64x64), 25 Euler-EDM steps with CFG
(B=36 per UNet call) + first-stage decode of the T frames — BASELINE.json configs[1] (V3D_512).  With N GPUs each
rank processes its own image (weak scaling, no data-path collective; the only exchange is the final uint8 frame
gather).  Prints ONE JSON line (rank 0).  Synthetic data, random-init weights of the V3D_512 architecture.

Timed regions (CUDA events on the launching stream, barrier + synchronize on both sides, max over ranks):
  value : inputs already resident in HBM
  e2e   : through the public API with pinned HOST buffers, H2D of noise+conditioning and D2H of the uint8 frames
          inside the timed region.
`roofline` describes the dominant kernel family (the tcgen05 GEMM / implicit conv kernel): algorithmic FLOPs of its
launches in one step / their summed CUDA-event durations, against MEASURED_PEAKS.json.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

# algorithmic FLOPs of the reference modules (BASELINE.md §2; FlopCounterMode on the reference, 2*MAC, CFG-batched)
F_UNET_TF = {14: 35.542, 18: 45.677, 24: 60.884, 25: 63.419}
F_DEC_TF = {14: 42.599, 18: 54.771, 24: 73.028, 25: 76.070}
FALLBACK_PEAKS = {"bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "hbm_gbs": 6650.0}


def work_tf(T: int, S: int, latent: int) -> float:
    fu = F_UNET_TF.get(T, 2.537 * T)
    fd = F_DEC_TF.get(T, 3.043 * T)
    return (S * fu + fd) * (latent / 64.0) ** 2


def load_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            d = json.loads(p.read_text())
            return d, "measured"
        except Exception:
            pass
    return dict(FALLBACK_PEAKS), "fallback"


def csrc_digest() -> str:
    """sha256 over the kernel sources: ties an ncu capture under profiles/ to the build it was taken from."""
    import hashlib

    h = hashlib.sha256()
    for f in sorted((ROOT / "v3d_b200" / "csrc").glob("*.cu*")):
        h.update(f.name.encode())
        h.update(f.read_bytes())
    return h.hexdigest()[:16]


def load_traffic():
    """`roofline.traffic`: dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel from the
    round's `ncu --set full` capture (profiles/traffic_r2.json, written by tools/ncu_summary.py).  DRAM counters cannot
    be read outside a profiler, so the figure comes from that capture - and only while the kernel sources are the ones
    it was taken from (`csrc_digest`); otherwise null."""
    tpath = ROOT / "profiles" / "traffic_r2.json"
    try:
        d = json.loads(tpath.read_text())
        if d.get("csrc_digest") != csrc_digest():
            return None
        return d
    except Exception:
        return None


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled DURING the timed region (B200_PROFILING.md clocks line)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu_index = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                 "-i", str(self.gpu_index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self, t0: float, t1: float) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for ts, line in self.lines:
            if not (t0 <= ts <= t1 + 0.3):
                continue
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the oracle port timed on host cores, on a bounded sample of the same workload
# ---------------------------------------------------------------------------------------------------------------
def _cpu_threads() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


class CpuReference:
    """Oracle port (oracle/, kind "port") of the reference path, fp32, on the host cores.

    mode "real-shape" (default whenever the CPU-time budget allows): one `sample()` runs, AT THE BENCHMARKED SHAPE
    (latent 64 x 64, T frames), the network evaluation of ONE of the two CFG videos (B = T; [uc; c] are independent
    batch items of every operator, so the CFG-batched forward costs twice this) and the first-stage decode of `nd`
    whole frames (the decode's cost is linear in the frame count: the frames only meet in 3-tap temporal convolutions).
        seconds per image = S * 2 * t_unet_half + (T / nd) * t_decode_nd
    Nothing is extrapolated in resolution, so the N^2 attention term and the cache behaviour of the real tensors are in
    the measurement.  The first sample of a run additionally times the full CFG-batched forward (B = 2T) once and
    reports the ratio to 2 * t_unet_half as a check of the batch scaling.

    mode "ladder" (fallback when K samples at the real shape do not fit the budget): round 1's two-size affine
    extrapolation in the latent size.

    The thread count is calibrated once (more threads than the box can really run make the many small ops slower,
    not faster): `cores` in the JSON is the count actually used."""

    LADDER = (((16, 32), (8, 16), 20.0), ((8, 16), (4, 8), 5.5))
    # all timed samples of a run should fit in about this much CPU time (V3D_CPU_BUDGET_S overrides)
    BUDGET_S = float(os.environ.get("V3D_CPU_BUDGET_S", "420"))
    # cost of the real-shape pieces in units of the calibration forward (latent 8, B = 2T), measured on two hosts;
    # only used to decide what fits the budget
    COST_UNET_HALF, COST_DEC_FRAME = 24.0, 5.0

    def __init__(self, T: int, S: int, latent: int, n_samples: int = 1):
        import torch
        from oracle import ref_decoder, ref_unet  # the one place bench.py executes oracle/: the timed baseline

        self.torch, self.ref_unet, self.ref_decoder = torch, ref_unet, ref_decoder
        self.T, self.S, self.latent = T, S, latent
        self.n_samples = max(1, n_samples)
        self.spec_u = ref_unet.UNetSpec()
        self.spec_d = ref_decoder.DecoderSpec()
        g = torch.Generator().manual_seed(0)

        def rnd(shape, key):
            shape = tuple(shape)
            if len(shape) > 1:
                fan = 1
                for d in shape[1:]:
                    fan *= d
                return torch.empty(shape).normal_(0, fan ** -0.5, generator=g)
            if key.endswith(".weight"):
                return torch.ones(shape)
            return torch.zeros(shape)

        self.sd_u = {k: rnd(s, k) for k, s in ref_unet.unet_param_shapes(self.spec_u).items()}
        self.sd_d = {k: rnd(s, k) for k, s in ref_decoder.decoder_param_shapes(self.spec_d).items()}
        self.g = g
        self.xin, self.z = {}, {}
        self.threads, self.thread_trials = self._calibrate_threads()
        torch.set_num_threads(self.threads)
        t_cal = self.thread_trials[self.threads]
        forced = os.environ.get("V3D_CPU_MODE")
        # real-shape samples that fit the budget: as many of the run's steps as possible take one (at least one when a
        # single sample fits at all), the remaining steps repeat the cheap calibration forward as a drift check
        self.nd, self.n_real = 0, 0
        for nd in (T, 6, 3, 2, 1):
            cost = (self.COST_UNET_HALF + nd * self.COST_DEC_FRAME) * t_cal
            if T % nd == 0 and cost * min(self.n_samples, 4) <= self.BUDGET_S:
                self.nd, self.n_real = nd, max(1, min(self.n_samples, int(self.BUDGET_S // cost)))
                break
        if not self.nd and (self.COST_UNET_HALF + self.COST_DEC_FRAME) * t_cal <= self.BUDGET_S:
            self.nd, self.n_real = 1, 1
        per_sample = self.BUDGET_S / max(self.n_real, 1)
        self.mode = forced or ("real-shape" if self.nd else "ladder")
        self.taken = 0
        if self.mode == "real-shape":
            self.nd = self.nd or 1
            self.n_real = self.n_real or 1
            self.full_forward_check = (self.COST_UNET_HALF * 3 + self.nd * self.COST_DEC_FRAME) * t_cal <= per_sample
        else:
            su, sdz = self.LADDER[-1][:2]
            for lu, ldz, cost in self.LADDER:
                if cost * t_cal * self.n_samples <= self.BUDGET_S:
                    su, sdz = lu, ldz
                    break
            self.su = tuple(min(x, latent) for x in su)
            self.sdz = tuple(min(x, latent) for x in sdz)
        self.extra = {}

    def _unet(self, L: int, videos: int = 2) -> float:
        torch = self.torch
        B = videos * self.T
        key = (L, videos)
        if key not in self.xin:
            self.xin[key] = (torch.randn(B, 8, L, L, generator=self.g), torch.full((B,), 0.3),
                             torch.randn(B, 1, 1024, generator=self.g), torch.randn(B, 768, generator=self.g),
                             torch.zeros(videos, self.T))
        x, ts, ctx, y, ind = self.xin[key]
        t0 = time.perf_counter()
        self.ref_unet.unet_forward(self.sd_u, self.spec_u, x, ts, ctx, y, self.T, ind)
        return time.perf_counter() - t0

    def _dec(self, L: int, frames: int = 0) -> float:
        frames = frames or self.T
        key = (L, frames)
        if key not in self.z:
            self.z[key] = self.torch.randn(frames, 4, L, L, generator=self.g)
        t0 = time.perf_counter()
        self.ref_decoder.decoder_forward(self.sd_d, self.spec_d, self.z[key], frames)
        return time.perf_counter() - t0

    def _calibrate_threads(self):
        """Smallest UNet forward (latent 8) at 8, 16, 32, ... threads up to the affinity mask; stop once a step is
        clearly slower than the best so far.  Returns (best, {threads: seconds})."""
        torch = self.torch
        ncpu = _cpu_threads()
        cands = sorted({min(c, ncpu) for c in (8, 16, 32, 64, 128, 256)} | {ncpu})
        trials, best_n, best_t = {}, cands[0], None
        with torch.no_grad():
            torch.set_num_threads(cands[0])
            self._unet(8)  # first call pays allocator / oneDNN primitive setup
            for n in cands:
                torch.set_num_threads(n)
                t = self._unet(8)
                trials[n] = round(t, 3)
                if best_t is None or t < best_t:
                    best_n, best_t = n, t
                elif t > 1.5 * best_t:
                    break
        return best_n, trials

    def warm(self):
        """An untimed warm-up step: the cheap calibration forward (the real-shape pieces run for tens of seconds
        each; their first-call costs - allocator growth, oneDNN primitive creation - are below 1 % of that)."""
        with self.torch.no_grad():
            self._unet(8)

    def sample(self):
        """-> (seconds of one CFG-batched UNet forward at the full size, seconds of the full decode); the raw
        measurements in self.last"""
        L = self.latent
        with self.torch.no_grad():
            if self.mode == "real-shape" and self.taken >= self.n_real:
                t = self._unet(8)                # budget spent: the cheap calibration forward, reported as drift
                self.drift = getattr(self, "drift", []) + [round(t, 3)]
                return None
            if self.mode == "real-shape":
                self.taken += 1
                th = self._unet(L, videos=1)
                tdn = self._dec(L, self.nd)
                self.last = {"unet_half_batch_s": round(th, 3), f"decode_{self.nd}_frames_s": round(tdn, 3)}
                if self.full_forward_check and "full_forward_s" not in self.extra:
                    tf = self._unet(L, videos=2)
                    self.extra = {"full_forward_s": round(tf, 3), "full_over_2x_half": round(tf / (2 * th), 3)}
                return 2.0 * th, tdn * self.T / self.nd
            tu = [self._unet(l) for l in self.su]
            td = [self._dec(l) for l in self.sdz]
        self.last = {"unet_s": dict(zip(self.su, (round(t, 3) for t in tu))),
                     "decode_s": dict(zip(self.sdz, (round(t, 3) for t in td)))}
        return self._affine(self.su, tu), self._affine(self.sdz, td)

    def _affine(self, sizes, times) -> float:
        (l0, l1), (t0, t1) = sizes, times
        full = float(self.latent) ** 2
        if l1 > l0:
            b = (t1 - t0) / (l1 * l1 - l0 * l0)
            a = t0 - b * l0 * l0
            if b > 0 and a >= 0:
                return a + b * full
        return t1 * full / (l1 * l1)  # degenerate fit (noise, or sizes clipped to the latent): plain pixel scaling

    def frames_per_sec(self, t_unet_full: float, t_dec_full: float) -> float:
        return self.T / (self.S * t_unet_full + t_dec_full)

    def describe(self) -> str:
        head = f"oracle port fp32, {self.threads} threads (calibrated over {sorted(self.thread_trials)}), mode {self.mode}: "
        if self.mode == "real-shape":
            return head + (f"per sample, at the benchmarked shape (latent {self.latent}^2, T={self.T}): the network "
                           f"evaluation of one of the two CFG videos (B={self.T}; x2 = the CFG-batched forward) and the "
                           f"decode of {self.nd} of the {self.T} frames (x{self.T // self.nd}); image time = "
                           f"{self.S} x 2 x t_unet_half + {self.T // self.nd} x t_decode; no extrapolation in resolution; "
                           f"{self.n_real} of the run's steps take such a sample (CPU-time budget {self.BUDGET_S:.0f} s), "
                           f"the others repeat the calibration forward as a drift check")
        return head + (f"per sample one CFG-batched UNet forward (B={2 * self.T}, T={self.T}) at latents {self.su[0]}^2 and "
                       f"{self.su[1]}^2 and one decode (T={self.T}) at latents {self.sdz[0]}^2 and {self.sdz[1]}^2; each "
                       f"extrapolated to latent {self.latent}^2 by the affine model t = a + b*pixels through its two "
                       f"sizes, UNet x {self.S} EDM steps (the CPU-time budget did not allow the real shape)")

    def baseline_dict(self, value, tu, td) -> dict:
        return {"value": value, "unit": "view-frames/s", "cores": self.threads, "kind": "port", "mode": self.mode,
                "sample": self.describe(), "t_unet_forward_full_s": tu, "t_decode_full_s": td,
                "last_sample_raw_s": self.last, "batch_scaling_check": self.extra or None,
                "real_shape_samples": getattr(self, "taken", None),
                "calibration_forward_drift_s": getattr(self, "drift", None),
                "thread_calibration_s": self.thread_trials}


def run_reference(args) -> None:
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    ref = CpuReference(args.frames, args.edm_steps, args.latent, n_samples=args.steps)
    for _ in range(args.warmup):
        ref.warm()
    tus, tds = [], []
    t0 = time.perf_counter()
    for _ in range(args.steps):
        r = ref.sample()
        if r is not None:       # a real-shape (or ladder) sample; None = a drift-check step after the budget was spent
            tus.append(r[0])
            tds.append(r[1])
    wall = time.perf_counter() - t0
    tu, td = sum(tus) / len(tus), sum(tds) / len(tds)
    v = ref.frames_per_sec(tu, td)
    base = ref.baseline_dict(v, tu, td)
    base["per_sample_unet_forward_s"] = [round(x, 2) for x in tus]
    base["per_sample_decode_s"] = [round(x, 2) for x in tds]
    line = {
        "impl": "reference", "metric": "view-frames/sec", "value": v, "unit": "view-frames/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000.0 * wall / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, "cpu"),
        "cpu_baseline": base,
        "e2e": {"value": v, "unit": "view-frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def workload_config(args, where: str) -> dict:
    return {"workload": f"V3D_512: 1 image -> {args.frames} views, {args.latent * 8}x{args.latent * 8}, "
                        f"{args.edm_steps} Euler-EDM steps (CFG, B={2 * args.frames}) + first-stage decode; one image per GPU",
            "frames": args.frames, "edm_steps": args.edm_steps, "latent": [4, args.latent, args.latent],
            "cfg_scale": [args.min_cfg, args.max_cfg], "sigma_max": 700.0, "decode_chunk": args.frames,
            # the same dictionary in both arms (the reference arm runs the same workload on rank 0's host cores)
            "parallelism": (f"one image over {args.gpus} ranks, plan '{args.shard}' (views: frame blocks with K|V "
                            "all-gather, conv halos, 3-D GN all-reduce; cfg: the CFG halves on a rank pair)"
                            if getattr(args, "shard", "images") != "images" else f"image-dp{args.gpus}"),
            "l2_policy": "working set per step (3 GB bf16 weights + activations) exceeds the 126 MB L2; no explicit flush",
            "weights": "random-init (per-name seeded, oracle/synth.py), zero-init modules re-randomised"}


def assemble_line(args, *, world, secs, secs_e2e, launches, clocks, h2d_bytes, d2h_bytes, sharded, probe_ms,
                  gemm_records, families, shapes, membound, decode_families=None, decode_shapes=None) -> dict:
    """The JSON line of the native arm from plain numbers (seconds / milliseconds / bytes / FLOPs).
    gemm_records: [(flops, ms)] of every tensor-core GEMM/conv launch of one probed step; families: {op: [ms]};
    shapes: {shape key: [(flops, ms)]}; membound: {family: [(algorithmic bytes, ms)]}."""
    T, S, L = args.frames, args.edm_steps, args.latent
    gemm_flops = sum(f for f, _ in gemm_records)
    gemm_ms = sum(m for _, m in gemm_records)
    breakdown = {k: {"ms": round(sum(v), 3), "launches": len(v)} for k, v in sorted(families.items())}
    def shape_table(table):
        out = []
        for k, v in (table or {}).items():
            sms = sum(m for _, m in v)
            fl = sum(f for f, _ in v)
            out.append({"shape": k, "launches": len(v), "ms": round(sms, 3),
                        "tflops": round(fl / sms / 1e9, 1) if sms > 0 else None})
        out.sort(key=lambda r: -r["ms"])
        return out

    shape_rows = shape_table(shapes)
    decode_breakdown = {k: {"ms": round(sum(v), 3), "launches": len(v)} for k, v in sorted((decode_families or {}).items())}
    decode_breakdown["_sum_of_kernels_ms"] = round(sum(v["ms"] for v in decode_breakdown.values()), 3)
    breakdown["_probed_step_ms"] = round(probe_ms, 3)
    breakdown["_sum_of_kernels_ms"] = round(sum(v["ms"] for k, v in breakdown.items() if isinstance(v, dict)), 3)

    peaks, peak_src = load_peaks()
    peaks_hbm = float(peaks.get("hbm_gbs") or FALLBACK_PEAKS["hbm_gbs"])
    hbm_rows = {}
    for fam, recs in membound.items():
        fms = sum(m for _, m in recs)
        gb = sum(b for b, _ in recs) / 1e9
        if fms > 0:
            hbm_rows[fam] = {"launches": len(recs), "ms": round(fms, 3), "algorithmic_gb": round(gb, 2),
                             "achieved_gbs": round(gb / (fms * 1e-3), 1),
                             "frac_of_hbm_peak": round(gb / (fms * 1e-3) / peaks_hbm, 3)}
    traffic = load_traffic()
    peak_tf = float(peaks.get("bf16_tflops_sustained") or peaks.get("bf16_tflops"))
    n_img = 1 if sharded else world
    value = n_img * T * args.steps / secs
    e2e_value = n_img * T * args.steps / secs_e2e
    model_tf = work_tf(T, S, L)
    achieved = gemm_flops / (gemm_ms * 1e-3) / 1e12 if gemm_ms > 0 else None
    return {
        "metric": "view-frames/sec", "value": value, "unit": "view-frames/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1000.0 * secs / args.steps, "higher_is_better": True,
        "scaling": "strong" if sharded else "weak", "vs_baseline": None, "dtype": "bf16",
        "data": "synthetic",
        "config": workload_config(args, "gpu"),
        "e2e": {"value": e2e_value, "unit": "view-frames/s", "h2d_bytes_per_step": h2d_bytes * world,
                "d2h_bytes_per_step": d2h_bytes * n_img, "ms_per_step": 1000.0 * secs_e2e / args.steps,
                "api": "DiffusionEngine.sample_views + frames_nchw_to_u8 (+ NCCL frame gather when N > 1)"},
        "gpu_launches": launches,
        "clocks": clocks,
        "roofline": {
            "bound": "tensor", "kernel": "gemm_tc_kernel (tcgen05 GEMM / temporal conv / implicit 3x3 conv)",
            "achieved": achieved, "peak": peak_tf,
            "unit": "TFLOP/s", "frac": achieved / peak_tf if achieved is not None else None,
            # DRAM bytes (read + write) of ONE launch of the dominant kernel at its top-level shape - the implicit 3x3
            # conv 36 x 64 x 64, 320 -> 320 (algorithmic: A 94.4 MB + W 1.8 MB + D 94.4 MB = 190.6 MB; part of D is
            # still dirty in L2 at kernel end) - from the round's ncu capture; the other captured kernels in _detail
            "traffic": (traffic["kernels"].get("gemm_tc_kernel<160, 1, 0, 1> #1", {}).get("traffic")
                        if traffic else None),
            "traffic_algorithmic_bytes": 190591488 if traffic else None,
            "traffic_detail": traffic,
            "peak_source": f"{peak_src} bf16_tflops_sustained",
            "launches_per_step": len(gemm_records), "algorithmic_tflop_per_step": gemm_flops / 1e12,
            "kernel_ms_per_step": gemm_ms, "share_of_step": gemm_ms / probe_ms if probe_ms > 0 else None,
            "breakdown_ms_per_step": breakdown,
            "breakdown_decode_only_ms": decode_breakdown,   # the first-stage decode's share of the families above
            "gemm_shapes_top": shape_rows[:30],
            "gemm_shapes_decode": shape_table(decode_shapes)[:20],
            "hbm_bound_families": dict(hbm_rows, peak_gbs=peaks_hbm,
                                       note="algorithmic bytes (each tensor read / written once) over summed CUDA-event "
                                            "durations of one eager step; many of these tensors fit the 126 MB L2"),
            "model": {"reference_accounting_tflop_per_step": model_tf,
                      "achieved_tflops": model_tf / (secs / args.steps), "frac": model_tf / (secs / args.steps) / peak_tf},
        },
    }


# ---------------------------------------------------------------------------------------------------------------
# native arm
# ---------------------------------------------------------------------------------------------------------------
def load_synth_(module, dev, seed: int) -> None:
    """Materialise the parameters of a module built under torch.device("meta") on `dev` with the per-name seeded
    values of the parity fixtures (oracle/synth.py: a seeded generator, no reference arithmetic)."""
    import torch
    from oracle import synth

    for name, p in list(module.named_parameters()):
        val = synth.synth_tensor(name, tuple(p.shape), seed).to(dev)
        mod = module
        parts = name.split(".")
        for part in parts[:-1]:
            mod = mod._modules[part]
        mod._parameters[parts[-1]] = torch.nn.Parameter(val, requires_grad=False)
    module._invalidate()


PARITY_TOL = {"rel_l2": 3e-2, "cosine": 0.999}   # DESIGN.md section 4 (bf16 path vs the fp32 reference)
DUMP_LIMIT_BYTES = 64 * 10 ** 6


def dump_outputs(out_dir, arrays: dict, limit_bytes: int = DUMP_LIMIT_BYTES) -> dict:
    """Write each array as out_dir/<name>.npy in float32, so that two builds can be compared output for output.
    When the arrays together would exceed `limit_bytes`, each is replaced by the same share of its elements: a flat
    sample at indices drawn with a fixed seed and sorted (identical from run to run for the same shapes).
    -> {name: {"shape", "dtype", "sampled_elements" (None: complete)}}"""
    import numpy as np

    out_dir = Path(out_dir)
    out_dir.mkdir(parents=True, exist_ok=True)
    arrays = {k: np.asarray(v, dtype=np.float32) for k, v in arrays.items()}
    total = sum(a.size for a in arrays.values())
    keep = (limit_bytes - 128 * len(arrays)) // 4     # each .npy header takes 128 bytes
    info = {}
    for name, a in arrays.items():
        sampled = None
        flat = a.reshape(-1)
        if total > keep:
            sampled = a.size * keep // total
            flat = flat[np.sort(np.random.default_rng(0).choice(a.size, sampled, replace=False))]
        np.save(out_dir / f"{name}.npy", flat if sampled is not None else a)
        info[name] = {"shape": list(a.shape), "dtype": "float32", "sampled_elements": sampled}
    return info


def parity_check(eng, dev, manifest) -> dict:
    """Before anything is timed: ONE network evaluation and ONE decode at the benchmarked size (T = 18, latent 64 x 64,
    CFG batch 36 / 18 frames -> 512 x 512) against the REAL reference's fp32 outputs on the same weights and inputs
    (tests/golden/unet_v3d512.pt, decoder_v3d512.pt; oracle/make_golden.py).  Raises when out of tolerance."""
    import torch
    from oracle import synth

    gold_dir = ROOT / "tests" / "golden"

    def rel(a, b):
        a, b = a.float(), b.float().to(a.device)
        return ((a - b).norm() / b.norm().clamp_min(1e-12)).item()

    def cos(a, b):
        a, b = a.float().flatten(), b.float().to(a.device).flatten()
        return (a @ b / (a.norm() * b.norm()).clamp_min(1e-12)).item()

    mu = manifest["unet_v3d512"]
    T, hw = mu["T"], mu["latent_hw"]
    gold = torch.load(gold_dir / "unet_v3d512.pt")
    x, c, uc = synth.synth_inputs(T, hw, seed=mu["input_seed"])
    xin = torch.cat([torch.cat([x, x]), torch.cat([uc["concat"], c["concat"]])], 1).to(dev)
    ctx = torch.cat([uc["crossattn"], c["crossattn"]]).to(dev)
    y = torch.cat([uc["vector"], c["vector"]]).to(dev)
    with torch.no_grad():
        out = eng.model.diffusion_model(xin, gold["timesteps"].to(dev), ctx, y, None, T,
                                        torch.zeros(2, T, device=dev))
    st = gold["stride"]
    res = {"unet_forward": {"rel_l2": rel(out[:, :, ::st, ::st], gold["out_sub"]),
                            "cosine": cos(out[:, :, ::st, ::st], gold["out_sub"]),
                            "rel_l2_full_items": rel(out[gold["full_items"]], gold["out_full"]),
                            "finite": bool(torch.isfinite(out).all()), "fixture": "tests/golden/unet_v3d512.pt"}}
    md = manifest["decoder_v3d512"]
    gold = torch.load(gold_dir / "decoder_v3d512.pt")
    z = synth.synth_latents(md["B"], md["latent_hw"], seed=md["z_seed"])
    if not torch.equal(z[:, :, ::16, ::16], gold["z_check"]):
        raise SystemExit("bench.py: the decoder fixture's latents do not regenerate from their seed")
    with torch.no_grad():
        img = eng.first_stage_model.decoder(z.to(dev) / 0.18215, timesteps=md["T"])
    st, crop = gold["stride"], gold["crop"]
    res["decode"] = {"rel_l2": rel(img[:, :, ::st, ::st], gold["out_sub"]),
                     "cosine": cos(img[:, :, ::st, ::st], gold["out_sub"]),
                     "rel_l2_full_frames": rel(img[gold["full_frames"], :, :crop, :crop], gold["out_full"]),
                     "finite": bool(torch.isfinite(img).all()), "fixture": "tests/golden/decoder_v3d512.pt"}
    res["tolerance"] = dict(PARITY_TOL)
    res["against"] = "outputs of the real reference modules (fp32, CPU) on the same seeded weights and inputs"
    for k in ("unet_forward", "decode"):
        r = res[k]
        if not (r["finite"] and r["rel_l2"] <= PARITY_TOL["rel_l2"] and r["cosine"] >= PARITY_TOL["cosine"]):
            raise SystemExit(f"bench.py: parity check failed before timing: {k} {r}")
    return res


def probe_exchanges(plan):
    """Bracket every exchange of a one-image-over-ranks plan with CUDA events (eager step only).
    -> ({kind: [(e0, e1)]}, restore())"""
    import torch

    events, saved = {}, []
    if plan is None:
        return events, lambda: None
    targets = []
    for obj, prefix in ((plan.sample, ""), (plan.decode if plan.decode is not plan.sample else None, "decode_"),
                        (plan.cfg, "")):
        if obj is None:
            continue
        for meth, kind in (("allreduce_stats_", "gn_allreduce"), ("exchange_halos", "halo"), ("gather_rows", "kv_allgather"), ("gather_signal", "kv_allgather_signal"),
                           ("gather_frames", "frame_gather"), ("gather_halves", "cfg_gather")):
            if hasattr(obj, meth):
                targets.append((obj, meth, prefix + kind))
    for obj, meth, kind in targets:
        fn = getattr(obj, meth)

        def wrapped(*a, _fn=fn, _kind=kind, **kw):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            r = _fn(*a, **kw)
            e1.record()
            events.setdefault(_kind, []).append((e0, e1))
            return r

        saved.append((obj, meth))
        setattr(obj, meth, wrapped)

    def restore():
        for obj, meth in saved:
            try:
                delattr(obj, meth)      # instance attribute shadowing the class's method
            except AttributeError:
                pass

    return events, restore


def summarise_exchanges(events, probe_ms: float) -> dict:
    """Per-kind device time of the exchanges of one eager step (CUDA events on the launching stream around each
    torch.distributed call: transfer + the wait for the slowest peer, i.e. load imbalance shows up here)."""
    out = {}
    for kind, evs in sorted(events.items()):
        t = sum(a.elapsed_time(b) for a, b in evs)
        out[kind] = {"calls": len(evs), "ms": round(t, 3)}
    tot = sum(v["ms"] for v in out.values())
    out["_all_exchanges_ms"] = round(tot, 3)
    out["_eager_probed_step_ms"] = round(probe_ms, 3)
    out["_share_of_step"] = round(tot / probe_ms, 4) if probe_ms > 0 else None
    if out and tot > 0:
        out["_limiting"] = max((k for k in out if not k.startswith("_")), key=lambda k: out[k]["ms"])
    return out


def measure_strong(args, eng, dev, rank, world, T, L) -> dict:
    """ONE image over the N ranks (BASELINE.json north_star: the T view-frames sharded over the GPUs of a box with the
    temporal-attention K|V all-gather, plus the CFG-pair split of SURVEY.md 8(e)); every plan that fits N is timed
    (same weights and the same image on every rank, device-resident inputs, CUDA events, max over ranks)."""
    import torch

    from v3d_b200 import ops, parallel
    from v3d_b200.viewshard import ShardPlan

    modes = [m for m in (os.environ.get("V3D_STRONG_PLANS", "views,cfg,cfg+views").split(","))
             if (m == "views" and world <= T) or (m == "cfg" and world == 2) or
             (m == "cfg+views" and world >= 4 and world % 2 == 0 and T // (world // 2) >= 2)]
    g = torch.Generator().manual_seed(23)
    x = torch.randn(T, 4, L, L, generator=g).to(dev)
    c = {"crossattn": torch.randn(1, 1, 1024, generator=g).repeat(T, 1, 1).to(dev),
         "concat": torch.randn(1, 4, L, L, generator=g).repeat(T, 1, 1, 1).to(dev),
         "vector": torch.randn(T, 768, generator=g).to(dev)}
    uc = {"crossattn": torch.zeros_like(c["crossattn"]), "concat": torch.zeros_like(c["concat"]), "vector": c["vector"].clone()}
    k = max(1, min(args.steps, 2))
    out = {"steps": k, "warmup": 1, "unit": "view-frames/s", "plans": {},
           "note": "one image (T view-frames) over all ranks; value = T * steps / max-over-ranks seconds"}
    for mode in modes:
        plan = ShardPlan.create(T, mode)

        def step():
            img = eng.sample_views(x.clone(), c, uc, num_frames=T, decoding_t=T, shard=plan)
            u8 = torch.empty(img.shape[0], 8 * L, 8 * L, 3, device=dev, dtype=torch.uint8)
            ops.frames_nchw_to_u8(img.contiguous(), u8)
            return plan.gather_frames(u8)

        # a plan that fails (an exchange that times out raises in sample_views on the rank that saw it) is reported
        # and skipped on EVERY rank: the ranks agree on the outcome before anything is timed
        ok, err = 1.0, ""
        os.environ["V3D_PEER_CHECK"] = "0"      # no rank may leave the collective sequence early: checked below
        try:
            step()
            torch.cuda.synchronize()
            plan.check_status()
        except Exception as exc:  # noqa: BLE001
            ok, err = 0.0, f"{type(exc).__name__}: {exc}"[:300]
        finally:
            os.environ.pop("V3D_PEER_CHECK", None)
        flag = torch.tensor([ok], device=dev)
        if world > 1:
            torch.distributed.all_reduce(flag, op=torch.distributed.ReduceOp.MIN)
        if flag.item() < 1.0:
            out["plans"][mode] = {"error": err if ok == 0.0 else "failed on another rank"}
            continue
        parallel.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(k):
            step()
        e1.record()
        torch.cuda.synchronize()
        parallel.barrier()
        secs = parallel.max_over_ranks(e0.elapsed_time(e1) / 1000.0, dev)
        # one more step with events around every exchange (rank 0's view)
        events, restore = probe_exchanges(plan)
        p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        unet = eng.model.diffusion_model
        graphs_were, unet.cuda_graphs = unet.cuda_graphs, False   # eager: the events sit between individual launches
        try:
            p0.record()
            step()
            p1.record()
            torch.cuda.synchronize()
        finally:
            unet.cuda_graphs = graphs_were
            restore()
        out["plans"][mode] = {"value": T * k / secs, "ms_per_image": 1000.0 * secs / k,
                              "transport": plan.describe().get("transport"),
                              "blocks": plan.describe().get("sample_blocks") or plan.describe().get("decode_blocks"),
                              "exchanges_ms_per_image": summarise_exchanges(events, p0.elapsed_time(p1))}
    good = {m: v for m, v in out["plans"].items() if "value" in v}
    if good:
        best = max(good, key=lambda m: good[m]["value"])
        out["best_plan"] = best
        out["value"] = out["plans"][best]["value"]
        out["ms_per_image"] = out["plans"][best]["ms_per_image"]
    return out


def run_native(args) -> None:
    import torch

    from v3d_b200 import engine, ops, parallel

    if not torch.cuda.is_available():
        raise SystemExit("bench.py (native arm) needs a CUDA device; there is no CPU fallback for the product path")
    rank, local_rank, world = parallel.init()
    if world != args.gpus:
        if args.gpus > 1:
            raise SystemExit(f"--gpus {args.gpus} needs torchrun with {args.gpus} ranks (WORLD_SIZE={world})")
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    T, S, L = args.frames, args.edm_steps, args.latent

    cfg = engine.v3d_512_config(num_frames=T, num_steps=S, min_cfg=args.min_cfg, max_cfg=args.max_cfg)
    with torch.device("meta"):
        eng = engine.DiffusionEngine(**cfg)
    # --shard views | cfg | cfg+views: ONE image spread over the ranks (strong scaling; SURVEY.md 8(e)): frame blocks
    # (K|V all-gather, conv halos, GroupNorm statistics), the CFG pair on two ranks (one all-gather per network
    # evaluation), or both.  Every rank holds the same weights and the same full-video inputs.
    plan = None
    if args.shard != "images":
        from v3d_b200.viewshard import ShardPlan, ViewShard

        if world > 1:
            plan = ShardPlan.create(T, args.shard)
        else:
            one = ViewShard(num_frames=T, rank=0, world=1)
            plan = ShardPlan("views", T, one, None, one)
    wrank = 0 if plan is not None else rank
    # the weights of the parity fixtures (per-name seeded, bit-identical on every box and rank): the model that is
    # timed below is the model that is checked against the real reference's outputs first
    gold_manifest = json.loads((ROOT / "tests" / "golden" / "MANIFEST.json").read_text())
    load_synth_(eng.model.diffusion_model, dev, gold_manifest["unet_v3d512"]["weight_seed"])
    load_synth_(eng.first_stage_model.decoder, dev, gold_manifest["decoder_v3d512"]["weight_seed"])
    eng.eval()
    parity = None if args.no_parity else parity_check(eng, dev, gold_manifest)

    # synthetic inputs in pinned host memory (one image per rank; the same image on every rank when view-sharded)
    g = torch.Generator().manual_seed(23 + wrank)
    host = {
        "x": torch.randn(T, 4, L, L, generator=g).pin_memory(),
        "c.crossattn": torch.randn(1, 1, 1024, generator=g).repeat(T, 1, 1).pin_memory(),
        "c.concat": torch.randn(1, 4, L, L, generator=g).repeat(T, 1, 1, 1).pin_memory(),
        "c.vector": torch.randn(T, 768, generator=g).pin_memory(),
    }
    host["uc.crossattn"] = torch.zeros_like(host["c.crossattn"]).pin_memory()
    host["uc.concat"] = torch.zeros_like(host["c.concat"]).pin_memory()
    host["uc.vector"] = host["c.vector"].clone().pin_memory()
    h2d_bytes = sum(v.numel() * v.element_size() for v in host.values())
    frames_host = torch.empty(T, 8 * L, 8 * L, 3, dtype=torch.uint8).pin_memory()
    d2h_bytes = frames_host.numel()

    def upload():
        d = {k: v.to(dev, non_blocking=True) for k, v in host.items()}
        c = {k[2:]: d[k] for k in d if k.startswith("c.")}
        uc = {k[3:]: d[k] for k in d if k.startswith("uc.")}
        return d["x"], c, uc

    def hot_path(x, c, uc):
        """The public API call a user makes: sampler loop + decode, then the uint8 THWC wire format."""
        img = eng.sample_views(x, c, uc, num_frames=T, decoding_t=T, shard=plan)  # [T or t_local,3,H,W] fp32
        u8 = torch.empty(img.shape[0], 8 * L, 8 * L, 3, device=dev, dtype=torch.uint8)
        return ops.frames_nchw_to_u8(img.contiguous(), u8)

    x_res, c_res, uc_res = upload()
    torch.cuda.synchronize()

    def step_resident():
        return hot_path(x_res.clone(), c_res, uc_res)

    counts = [1] * world  # one image per rank
    gathered_host = torch.empty(world, T, 8 * L, 8 * L, 3, dtype=torch.uint8).pin_memory() if (world > 1 and rank == 0) else None

    def step_e2e():
        x, c, uc = upload()
        u8 = hot_path(x, c, uc)
        if plan is not None:
            # the decoded-frame gather of the view-sharded path (uint8 THWC over NCCL), then D2H on rank 0
            allf = plan.gather_frames(u8)
            if rank == 0:
                frames_host.copy_(allf, non_blocking=True)
        elif world > 1:
            # the path's only exchange: final decoded-frame gather (uint8 THWC) over NCCL, then D2H on rank 0
            allf = parallel.gather_frames(u8.unsqueeze(0), counts)
            if rank == 0:
                gathered_host.copy_(allf, non_blocking=True)
        else:
            frames_host.copy_(u8, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return frames_host

    def timed(fn, k):
        parallel.barrier()
        torch.cuda.synchronize()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = ops.launch_count() + eng.model.diffusion_model.replayed_launches
        w0 = time.time()
        ev0.record()
        for _ in range(k - 1):
            fn()
        out = fn()      # kept for --dump-outputs; earlier results are dropped at once, as the caching allocator expects
        ev1.record()
        torch.cuda.synchronize()
        w1 = time.time()
        parallel.barrier()
        secs = parallel.max_over_ranks(ev0.elapsed_time(ev1) / 1000.0, dev)
        return secs, ops.launch_count() + eng.model.diffusion_model.replayed_launches - l0, (w0, w1), out

    for _ in range(args.warmup):
        step_resident()
    torch.cuda.synchronize()

    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
        time.sleep(0.3)
    secs, launches, (w0, w1), frames = timed(step_resident, args.steps)
    clk = clocks.stop(w0, w1) if rank == 0 else None
    dumped = None
    if args.dump_outputs and rank == 0:
        # the uint8 THWC frames the hot path returned in the last timed step (rank 0's image or frame block)
        dumped = dump_outputs(args.dump_outputs, {"frames": frames.cpu().numpy()})
    del frames

    step_e2e()  # warm the e2e-only pieces (pinned copies)
    secs_e2e, _, _, _ = timed(step_e2e, args.steps)

    # ---- roofline of the dominant kernel family + per-family breakdown: every launch of ONE step is bracketed
    #      by CUDA events on the launching stream (a separate pass, so the timed region above carries no probes)
    records = []      # (flops, e0, e1) for tensor-core GEMM/conv launches
    families = {}     # op name -> list of (e0, e1)
    shapes = {}       # GEMM shape key -> list of (flops, e0, e1)
    membound = {}     # memory-bound family -> list of (algorithmic bytes, e0, e1)
    decode_families = {}   # the same per-family events, first-stage decode only
    decode_shapes = {}     # GEMM shapes of the decode
    phase = {"name": "sample"}
    host_only = {"launch_count", "pick_block_n", "geglu_perm"}
    saved = {}

    def make_probe(name, fn):
        def probed(*a, **kw):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            r = fn(*a, **kw)
            e1.record()
            fam = name
            if name == "gemm":
                K, N = kw["K"], kw["N"]
                rows = kw["rows_per_batch"] * kw.get("batch", 1)
                taps = 9 if kw.get("conv") is not None else kw.get("ntaps", 1)
                records.append((2.0 * rows * N * K * taps, e0, e1))
                skey = "%s M=%d K=%d N=%d%s%s%s%s" % (
                    "conv3x3" if kw.get("conv") is not None else ("tconv" if taps == 3 else "linear"), rows, K, N,
                    " geglu" if kw.get("act", 0) == ops.ACT_GEGLU else "", " +R1" if kw.get("r1") is not None else "",
                    " +R2" if kw.get("r2") is not None else "", " f32" if kw.get("out_fp32") else "")
                shapes.setdefault(skey, []).append((2.0 * rows * N * K * taps, e0, e1))
                if phase["name"] == "decode":
                    decode_shapes.setdefault(skey, []).append((2.0 * rows * N * K * taps, e0, e1))
                fam = "gemm.conv3x3" if kw.get("conv") is not None else ("gemm.temporal" if taps == 3 else "gemm.linear")
            families.setdefault(fam, []).append((e0, e1))
            if phase["name"] == "decode":
                decode_families.setdefault(fam, []).append((e0, e1))
            try:  # algorithmic HBM bytes of the memory-bound families (DESIGN.md section 3); never fatal
                nbytes = None
                if name == "groupnorm_stats":          # (x, stats, rows_per_sample, nsamples, c): read x once
                    nbytes = 2 * a[2] * a[3] * a[4]
                elif name == "groupnorm_apply":        # (x, y, stats, gamma, beta, rows_per_sample, nsamples, c)
                    nbytes = 2 * 2 * a[5] * a[6] * a[7]
                elif name == "groupnorm":              # one launch (x, y, gamma, beta, rows_per_sample, nsamples, c):
                    nbytes = 2 * 2 * a[4] * a[5] * a[6]    # x read once from HBM (re-read from L2), y written
                elif name == "layernorm":              # (x, y, gamma, beta, rows, c): read + write (+ the fused sum)
                    nbytes = 2 * (3 if kw.get("ysum") is not None else 2) * a[4] * a[5]
                elif name == "attention_temporal":     # (qkv, out, nb, t, s, nheads): q, k, v read, o written
                    nbytes = 2 * 4 * a[2] * a[3] * a[4] * a[5] * 64
                if nbytes is not None:
                    membound.setdefault(name, []).append((float(nbytes), e0, e1))
            except Exception:
                pass
            return r
        return probed

    for name in dir(ops):
        fn = getattr(ops, name)
        if callable(fn) and not name.startswith("_") and name not in host_only and getattr(fn, "__module__", "") == ops.__name__:
            saved[name] = fn
            setattr(ops, name, make_probe(name, fn))
    xchg_events, xchg_restore = probe_exchanges(plan)
    unet = eng.model.diffusion_model
    graphs_were = unet.cuda_graphs
    unet.cuda_graphs = False  # the probe needs eager launches (events between individual kernels)
    first_stage = eng.first_stage_model
    decode_method = first_stage.decode

    def decode_tagged(*a, **kw):   # launches made inside the first-stage decode are also booked under "decode"
        phase["name"] = "decode"
        try:
            return decode_method(*a, **kw)
        finally:
            phase["name"] = "sample"

    first_stage.decode = decode_tagged
    try:
        pe0, pe1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        pe0.record()
        step_resident()
        pe1.record()
        torch.cuda.synchronize()
    finally:
        unet.cuda_graphs = graphs_were
        xchg_restore()
        del first_stage.decode          # back to the class's method
        for name, fn in saved.items():
            setattr(ops, name, fn)
    # CUDA events -> plain milliseconds; everything below is host arithmetic (assemble_line, unit-tested on CPU)
    ms = lambda e0, e1: e0.elapsed_time(e1)
    line = assemble_line(
        args, world=world, secs=secs, secs_e2e=secs_e2e, launches=launches, clocks=clk, h2d_bytes=h2d_bytes,
        d2h_bytes=d2h_bytes, sharded=plan is not None, probe_ms=ms(pe0, pe1),
        gemm_records=[(f, ms(a, b)) for f, a, b in records],
        families={k: [ms(a, b) for a, b in v] for k, v in families.items()},
        shapes={k: [(f, ms(a, b)) for f, a, b in v] for k, v in shapes.items()},
        membound={k: [(nb, ms(a, b)) for nb, a, b in v] for k, v in membound.items()},
        decode_families={k: [ms(a, b) for a, b in v] for k, v in decode_families.items()},
        decode_shapes={k: [(f, ms(a, b)) for f, a, b in v] for k, v in decode_shapes.items()})
    line["parity"] = parity
    if dumped is not None:
        line["dumped_outputs"] = dumped
    if plan is not None:
        line["exchanges_ms_per_step"] = summarise_exchanges(xchg_events, ms(pe0, pe1))
    elif world > 1 and not args.no_strong:
        # BASELINE.json's north_star split next to the image-parallel throughput: ONE image over the N GPUs
        line["strong"] = measure_strong(args, eng, dev, rank, world, T, L)
    line["cuda_graph"] = os.environ.get("V3D_CUDA_GRAPH", "1") != "0"
    if plan is not None:
        line["shard_plan"] = dict(plan.describe(),
                                  cuda_graph_with_collectives=os.environ.get("V3D_VIEWSHARD_GRAPH", "0") == "1")
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        # bounded sample (about a minute of CPU work): one real-shape half-batch forward + a slice of the decode
        os.environ.setdefault("V3D_CPU_BUDGET_S", "45")
        CpuReference.BUDGET_S = float(os.environ["V3D_CPU_BUDGET_S"])
        ref = CpuReference(T, S, L, n_samples=1)
        tu, td = ref.sample()
        line["cpu_baseline"] = ref.baseline_dict(ref.frames_per_sec(tu, td), tu, td)
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        torch.distributed.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["native", "reference"], default="native")
    ap.add_argument("--frames", type=int, default=18)
    ap.add_argument("--edm-steps", type=int, default=25)
    ap.add_argument("--latent", type=int, default=64)
    ap.add_argument("--min-cfg", type=float, default=3.5)
    ap.add_argument("--max-cfg", type=float, default=3.5)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-strong", action="store_true",
                    help="N > 1, image-parallel run: skip the one-image-over-N-GPUs sub-measurement (`strong`)")
    ap.add_argument("--no-parity", action="store_true", help="skip the pre-timing parity check against tests/golden")
    ap.add_argument("--shard", choices=["images", "views", "cfg", "cfg+views"], default="images",
                    help="images (default): one image per GPU, weak scaling.  ONE image over the GPUs (strong scaling): "
                         "views = frame blocks (K|V all-gather, conv halos, 3-D GroupNorm all-reduce); cfg = the [uc; c] "
                         "halves on 2 GPUs (one all-gather per network evaluation); cfg+views = both (>= 4 GPUs)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the timed path returned in its last step (the uint8 frames "
                         "[T, H, W, 3] of rank 0) as DIR/frames.npy in float32; a fixed seeded sample when over 64 MB")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "native":
        ap.error("--dump-outputs needs the native arm: the reference arm times pieces of the path, not the path")
    if args.warmup < 3 and args.impl == "native":
        print("warning: timing rules ask for >= 3 warm-up steps", file=sys.stderr)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_native(args)


if __name__ == "__main__":
    main()

#!/usr/bin/env python
"""bench.py — UNet denoise steps/sec of the DiffSensei sampling loop on B200 (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # this repo's engine (one process per GPU)
    python bench.py --impl reference --gpus N --steps K --warmup W   # the reference's CPU path on the host cores
    python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR  # + the last timed step's latents as DIR/*.npy

A "step" is one iteration of src/pipelines/pipeline_diffsensei.py:310-337 — UNetMangaModel.forward at UNet batch
B = 2*bs under CFG, the CFG blend and the DDIM update — for BASELINE.json configs[1]: 1024x1024 panels, bs = 4 per
GPU (B = 8, latent 128x128), 2 character refs, 50 DDIM steps, bf16, synthetic embeddings and random-init weights
of the SDXL + IP topology (2.9 B params; no checkpoints offline).  N > 1: every rank runs its own bs = 4 shard
(cfg4 = bs 32 over 8 GPUs), no per-step collective; one NCCL all-gather of the final latents outside the timed
region.  Timing: CUDA events on the launching stream, barrier + synchronize on both sides, max over ranks.

Printed JSON line (rank 0): see the contract in the task statement; extra keys `roofline` (dominant kernel: the
tcgen05 GEMM at the FF1/GEGLU shape, timed live with CUDA events, against MEASURED_PEAKS.json), `roofline_family`
(the same kernel time-weighted over the step's real shape census), `roofline_gn` / `roofline_attn` (the two
north-star kernels), `roofline_chain` (the GEMM kernel in chain mode: the four linears between two attention kernels as
one launch), `roofline_cross` (fused text+IP cross-attention against its byte floor), `panel` (MEASURED
panels/sec: whole 50-step panels through DiffSenseiPipeline.denoise, per-panel setup included), `mfu` (with and
without the hoisted K|V projections), `cfg1_gpu` + `cpu_baseline.cfg1_measured` (one same-config CPU/GPU pair),
`gpu_library_baseline` (the torch/cuBLAS/cuDNN/SDPA stack the reference would dispatch — stated, not the product),
`cpu_baseline`, `e2e`, `clocks`.  `--config cfg1|cfg2|cfg3|cfg5` selects the BASELINE workload (default cfg2, the
one the metric is quoted on); the reference arm (`--impl reference`) imports only `oracle/`, never the product.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

METRIC = "unet_denoise_steps_per_sec_1024sq_bs4"
UNIT = "steps/s"
T_STEPS = 50
GUIDANCE, IP_SCALE = 7.5, 0.6
UNET_WEIGHT_SEED = 1234
STEP_TFLOP_CFG2 = 54.8          # analytic 2*MAC count of one cfg2 step, SURVEY.md §8d / BASELINE.md §2


# ------------------------------------------------------------------------------------------------ helpers
def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return {"hbm_gbs": p["hbm_gbs"], "bf16_tflops": p["bf16_tflops"],
                "bf16_tflops_sustained": p.get("bf16_tflops_sustained", p["bf16_tflops"]), "source": "measured"}
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def __exit__(self, *a):
        if self.proc is not None:
            time.sleep(0.15)
            self.proc.terminate()
            self.th.join(timeout=2)

    def summary(self):
        sm, mx, reasons = [], 0, set()
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = max(mx, float(r[1]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx or None,
                "reasons": sorted(reasons), "samples": len(sm)}


# cfg3 (BASELINE configs[2]): var-res buckets of src/datasets/utils.py:6-121 as (height, width) pixels, 2 panels each
# -> bs 8.  864x1216 / 1216x864 have odd feature maps (27 rows or columns at level 2 -> forward_upsample_size path);
# 704x368 is one of the five buckets whose mask geometry (H', W') derived from the token count differs from the true
# feature map (attention_processor.py:131-139; tests/golden/derived_hw_table.pt).
CFG3_BUCKETS = [(864, 1216), (1216, 864), (1536, 672), (704, 368)]
IP_BOXES = [[.05, .10, .50, .95], [.50, .15, .95, .90], [.30, .55, .70, 1.0], [.00, .00, .30, .40]]
DIALOG_BOXES = [[.05, .05, .30, .20], [.70, .05, .95, .22], [.40, .80, .65, .97]]


def config_panels(name):
    """-> list of (bs, latent_h, latent_w, n_chars, dialogs, mllm) groups of same-shape panels making up one batch."""
    if name == "cfg2":
        return [(4, 128, 128, 2, False, False)]
    if name == "cfg1":
        return [(1, 64, 64, 1, False, False)]
    if name == "cfg3":
        return [(2, hh // 8, ww // 8, 4, True, False) for hh, ww in CFG3_BUCKETS]
    if name == "cfg5":
        return [(1, 256, 128, 3, False, True)]
    return [(2, 16, 24, 2, True, False)]          # tiny: plumbing self-test only


def shard_inputs(inp, start, end):
    """Rows [start, end) of a CFG-concatenated global batch [neg(0..bs) ; pos(0..bs)] -> the same layout for the shard."""
    lat, ehs, pooled, time_ids, bbox, dialog = inp
    bs = lat.shape[0]
    pick = lambda t: None if t is None else torch.cat([t[start:end], t[bs + start:bs + end]], 0)
    return lat[start:end], pick(ehs), pick(pooled), pick(time_ids), pick(bbox), pick(dialog)


def synthetic_inputs(cfg, bs, h, w, n_chars, device, dialogs=False, mllm=False):
    """SURVEY.md §8d synthetic conditions (seeds fixed); embeddings stand in for the out-of-scope encoders.
    ``mllm``: the positive image tokens of the real characters are ``0.4 g + 0.6 e`` — MLLM-adapted embeddings g
    pasted over the Resampler output e (pipeline_diffsensei.py:143-145, scripts/demo/gradio.py:108-109)."""
    g = torch.Generator().manual_seed(0)
    lat = torch.randn(bs, 4, h, w, generator=g)
    text = torch.randn(bs, 77, cfg.cross_attention_dim, generator=g)
    neg_text = torch.randn(bs, 77, cfg.cross_attention_dim, generator=torch.Generator().manual_seed(1))
    img = torch.randn(bs, 80, cfg.cross_attention_dim, generator=g)       # Resampler output stand-in (pos)
    neg_img = torch.randn(bs, 80, cfg.cross_attention_dim, generator=g)   # Resampler(zeros) stand-in
    pooled = torch.randn(2 * bs, cfg.pooled_text_dim, generator=g)
    if mllm:
        nv = cfg.num_vision_tokens
        gm = torch.randn(n_chars, nv, cfg.cross_attention_dim, generator=g).reshape(1, n_chars * nv, -1)
        img[:, nv:(1 + n_chars) * nv] = 0.4 * gm + 0.6 * img[:, nv:(1 + n_chars) * nv]
    ehs = torch.cat([torch.cat([neg_text, neg_img], 1), torch.cat([text, img], 1)], 0)
    time_ids = torch.tensor([[h * 8.0, w * 8.0, 0, 0, h * 8.0, w * 8.0]] * (2 * bs))
    pos = IP_BOXES[:n_chars] + [[0.0] * 4] * (4 - n_chars)
    bbox = torch.tensor([[[0.0] * 4] * 4] * bs + [pos] * bs)
    dialog = None
    if dialogs:
        d = DIALOG_BOXES + [[0.0] * 4] * 5
        dialog = torch.tensor([[[0.0] * 4] * 8] * bs + [d] * bs)
    return lat, ehs, pooled, time_ids, bbox, dialog


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, arrays):
    """Write each tensor of ``arrays`` (name -> tensor) as ``out_dir/<name>.npy`` in float32, so that two builds run
    with the same arguments can be compared output for output."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a.float().cpu().numpy())


def event_time_ms(fn, iters, stream_sync=True):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(iters):
        fn(i)
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / iters


# ------------------------------------------------------------------------------------------------ kernel rooflines
def ncu_traffic():
    """DRAM bytes per launch (dram__bytes_read.sum + dram__bytes_write.sum) of the roofline kernels, from the
    committed `ncu --set full` capture of tools/profile_kernels.py (profiles/ncu_traffic.json; null if absent)."""
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            return json.load(f)
    except Exception:
        return {}


def kernel_rooflines(ds, peaks, device):
    """The dominant kernel and the two north-star kernels, each timed alone with CUDA events on the launching
    stream: >= 3 warm-ups, then ROUNDS back-to-back launches that rotate over SETS disjoint input/output buffer
    sets whose total footprint exceeds the 126 MB L2 (so no launch finds its operands cached, and the host's
    per-launch enqueue latency — ~10 us through ctypes — is hidden behind queued work instead of being billed to
    a 30 us kernel).  Reported against the measured BURST peaks (kernel timed alone)."""
    ops = ds.ops
    bf = torch.bfloat16

    def timed(calls, rounds):
        for c in calls:
            c()
        for c in calls[:3]:
            c()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for r in range(rounds):
            for c in calls:
                c()
        e1.record()
        e1.synchronize()
        return e0.elapsed_time(e1) / (rounds * len(calls))

    out = {}
    traffic = ncu_traffic()
    # dominant kernel: gemm_bf16_tcgen05 at the level-2 FF1/GEGLU shape (60 launches per step, 22.5 of 54.8 TFLOP)
    M, N, K = 8192, 10240, 1280
    sets = []
    for i in range(3):                                   # 3 x (21 + 26 + 42 MB) = 267 MB > L2
        a = torch.randn(M, K, device=device).to(bf)
        w = (torch.randn(N, K, device=device) * K ** -0.5).to(bf)
        o = torch.empty(M, N // 2, dtype=bf, device=device)
        sets.append((a, w, o))
    b = torch.zeros(N, device=device)
    ms = timed([(lambda s=s: ops.gemm(s[0], s[1], b, epilogue=ops.EPI_GEGLU, out=s[2])) for s in sets], 4)
    flops = 2.0 * M * N * K
    out["roofline"] = {"kernel": "gemm_bf16_tcgen05<256,2> FF1+GEGLU M8192 N10240 K1280", "bound": "tensor",
                       "achieved": round(flops / ms / 1e9, 1), "peak": peaks["bf16_tflops"], "unit": "TFLOP/s",
                       "frac": round(flops / ms / 1e9 / peaks["bf16_tflops"], 4), "traffic": traffic.get("gemm_ff1"),
                       "ms_per_launch": round(ms, 4), "peak_source": peaks["source"] + " burst (kernel timed alone)",
                       "algorithmic_GFLOP": round(flops / 1e9, 1)}
    del sets
    # the same kernel in chain mode: the four linears between a level-2 block's cross-attention and the next block's
    # self-attention (attn2.to_out -> ff.net.0 -> ff.net.2 -> to_qkv, LayerNorms folded) as ONE launch; 60 per step
    C4 = 1280
    sets = []
    for i in range(3):                                   # 3 x 52 MB of weights + activations > L2
        g = lambda *s_, k=1.0: (torch.randn(*s_, device=device) * k)
        a = g(M, C4).to(bf)
        h = g(M, C4).to(bf)
        st = [torch.zeros(2 * M, dtype=torch.float64, device=device) for _ in range(3)]
        qkv = torch.empty(M, 3 * C4, dtype=bf, device=device)
        f = torch.empty(M, 4 * C4, dtype=bf, device=device)
        W = [(g(C4, C4, k=C4 ** -0.5).to(bf), g(C4)), (g(8 * C4, C4, k=C4 ** -0.5).to(bf), g(8 * C4)),
             (g(C4, 4 * C4, k=(4 * C4) ** -0.5).to(bf), g(C4)), (g(3 * C4, C4, k=C4 ** -0.5).to(bf), g(3 * C4))]
        cs1, csq = g(8 * C4), g(3 * C4)
        sets.append([((a,) + W[0], dict(residual=h, out=h, row_stats_out=st[0], row_stats_zeroed=True)),
                     ((None,) + W[1], dict(epilogue=ops.EPI_GEGLU, ln_stats=st[0], ln_colsum=cs1, zero_rows=st[2],
                                           out=f)),
                     ((None,) + W[2], dict(residual=h, out=h, row_stats_out=st[1], row_stats_zeroed=True)),
                     ((None,) + W[3], dict(ln_stats=st[1], ln_colsum=csq, zero_rows=st[0], out=qkv))])
    ms = timed([(lambda s=s: ops.gemm_chain(s)) for s in sets], 4)
    flops = 2.0 * M * (C4 * C4 + 8 * C4 * C4 + 4 * C4 * C4 + 3 * C4 * C4)
    out["roofline_chain"] = {"kernel": "gemm_bf16_tcgen05<256,2,chain> attn2.to_out>ff.net.0>ff.net.2>to_qkv, M8192 "
                                       "C1280 (4 linears, one launch)", "bound": "tensor",
                             "achieved": round(flops / ms / 1e9, 1), "peak": peaks["bf16_tflops"], "unit": "TFLOP/s",
                             "frac": round(flops / ms / 1e9 / peaks["bf16_tflops"], 4),
                             "traffic": traffic.get("gemm_chain"),
                             "ms_per_launch": round(ms, 4), "algorithmic_GFLOP": round(flops / 1e9, 1)}
    del sets
    # fused GroupNorm+SiLU at (8, 128, 128, 320): algorithmic bytes = read x + write y.  In the step the statistics
    # come from the producing conv's epilogue, so the GroupNorm IS the apply kernel (`roofline_gn`); the stand-alone
    # two-pass form (statistics kernel + apply, what a caller without a producer gets) is reported beside it.
    ga, be = torch.ones(320, device=device), torch.zeros(320, device=device)
    sets = []
    for i in range(4):                                   # 4 x (84 + 84 MB) = 671 MB > L2
        x = torch.randn(8, 128, 128, 320, device=device).to(bf)
        sets.append((x, torch.empty_like(x), ops.channel_stats(x),
                     torch.empty(ops.groupnorm_scratch_floats(8, 320), device=device)))
    gb = 2 * sets[0][0].numel() * 2 / 1e9
    ms = timed([(lambda s=s: ops.groupnorm_apply(s[0], s[2], ga, be, 32, 1e-5, True, out=s[1])) for s in sets], 4)
    out["roofline_gn"] = {"kernel": "gn_apply2_kernel (8,128,128,320) bf16: GroupNorm+SiLU from producer-epilogue "
                                    "channel statistics, one pass", "bound": "hbm",
                          "achieved": round(gb / (ms * 1e-3), 1), "peak": peaks["hbm_gbs"], "unit": "GB/s",
                          "frac": round(gb / (ms * 1e-3) / peaks["hbm_gbs"], 4), "traffic": traffic.get("gn_apply"),
                          "ms_per_launch": round(ms, 4), "algorithmic_MB": round(gb * 1e3, 1)}
    ms2 = timed([(lambda s=s: ops.groupnorm_silu(s[0], ga, be, 32, 1e-5, True, out=s[1], stats=s[3])) for s in sets], 4)
    out["roofline_gn_two_pass"] = {"kernel": "chan_stats_kernel + gn_apply2_kernel (8,128,128,320) bf16, stand-alone",
                                   "bound": "hbm", "achieved": round(gb / (ms2 * 1e-3), 1), "peak": peaks["hbm_gbs"],
                                   "unit": "GB/s", "frac": round(gb / (ms2 * 1e-3) / peaks["hbm_gbs"], 4),
                                   "traffic": traffic.get("gn"), "ms_per_launch": round(ms2, 4),
                                   "algorithmic_MB": round(gb * 1e3, 1)}
    del sets
    # fused self-attention at level 1: B=8, N=4096, 10 heads (4*N^2*C*B flops)
    B, Nn, heads = 8, 4096, 10
    sets = []
    for i in range(2):                                   # 2 x (126 + 42 MB) = 336 MB > L2
        sets.append((torch.randn(B, Nn, 3 * heads * 64, device=device).to(bf),
                     torch.empty(B, Nn, heads * 64, dtype=bf, device=device)))
    ms = timed([(lambda s=s: ops.attention_self(s[0], heads, out=s[1])) for s in sets], 4)
    flops = 4.0 * Nn * Nn * heads * 64 * B
    out["roofline_attn"] = {"kernel": "flash_attn_v5_kernel B8 N4096 h10 d64", "bound": "tensor",
                            "achieved": round(flops / ms / 1e9, 1), "peak": peaks["bf16_tflops"], "unit": "TFLOP/s",
                            "frac": round(flops / ms / 1e9 / peaks["bf16_tflops"], 4), "traffic": traffic.get("flash"),
                            "ms_per_launch": round(ms, 4), "algorithmic_GFLOP": round(flops / 1e9, 1)}
    del sets
    # fused text + masked-IP cross-attention at level 1 (B8 N4096 h10): FLOP-light (157 keys) -> bounded by moving Q in
    # and O out once: 4*B*N*C bytes (K|V of 157 tokens are noise)
    C = heads * 64
    sets = []
    for i in range(4):                                   # 4 x (42 + 42 MB) = 336 MB > L2
        sets.append((torch.randn(B, Nn, C, device=device).to(bf), torch.randn(B, 77, 2 * C, device=device).to(bf),
                     torch.randn(B, 80, 2 * C, device=device).to(bf), torch.empty(B, Nn, C, dtype=bf, device=device)))
    bb = torch.tensor([[[.05, .10, .50, .95], [.50, .15, .95, .90], [0.0] * 4, [0.0] * 4]] * B, device=device)
    ms = timed([(lambda s=s: ops.attention_cross_ip(s[0], s[1], s[2], bb, heads, 1.0, 0.6, 16, 16, out=s[3]))
                for s in sets], 4)
    gb = 4.0 * B * Nn * C / 1e9
    out["roofline_cross"] = {"kernel": "cross_ip_attn kernel B8 N4096 h10 (77 text + 80 IP keys, bbox mask in-kernel)",
                             "bound": "hbm", "achieved": round(gb / (ms * 1e-3), 1), "peak": peaks["hbm_gbs"],
                             "unit": "GB/s", "frac": round(gb / (ms * 1e-3) / peaks["hbm_gbs"], 4),
                             "traffic": traffic.get("cross"), "ms_per_launch": round(ms, 4),
                             "algorithmic_MB": round(gb * 1e3, 1),
                             "flops_frac_of_tensor_peak": round(4.0 * Nn * 157 * C * B / ms / 1e9 / peaks["bf16_tflops"], 4)}
    return out


# ------------------------------------------------------------------------------------------------ CPU reference arm
def pick_host_threads(log=lambda *a: None):
    """Host threads the CPU arm should use.  The affinity mask of a GPU box can advertise far more cores than the
    container's CPU quota grants (128 advertised -> 1.3 GFLOP/s with 128 threads in round 1), so the thread count
    is chosen by measurement: the candidate (affinity, /2, /4, ... >= 4) with the best fp32 GEMM throughput."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    try:                                               # cgroup v2 quota, when visible
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = max(1, min(n, int(int(q) / int(per))))
    except Exception:
        pass
    cands, c = [], n
    while c >= 4:
        cands.append(c)
        c //= 2
    if not cands:
        return max(1, n)
    a, b = torch.randn(1536, 1536), torch.randn(1536, 1536)
    best, best_t = cands[0], float("inf")
    for c in cands:
        torch.set_num_threads(c)
        torch.mm(a, b)
        t0 = time.time()
        for _ in range(3):
            torch.mm(a, b)
        dt = (time.time() - t0) / 3
        log(f"[reference] {c} threads: {2 * 1536 ** 3 / dt / 1e9:.0f} GFLOP/s fp32 GEMM probe")
        if dt < best_t * 0.95:                         # prefer more threads only when clearly faster
            best, best_t = c, dt
    return best


class CpuReference:
    """The reference's CPU path: its processors' arithmetic + the diffusers SDXL blocks as restated by the oracle
    (real diffusers / the reference tree do not exist on the GPU box), fp32, all the host threads the quota grants.
    Imports ONLY ``oracle`` (never the product package: the reference arm must not map libdsengine.so).

    Two measurements, neither of them scaled by a FLOP model:
      * ``cfg1_step``  — BASELINE configs[0] exactly as SURVEY §8d states it: 512x512, bs 1 (UNet batch 2), 1
        character ref, fp32: one full loop iteration (UNet at B = 2, CFG blend, DDIM update);
      * ``cfg2_row``   — the BOUNDED SAMPLE of the cfg2 workload: ONE of the 8 batch rows of a cfg2 step at the full
        128x128 latent (2 character refs).  Every op on the path is per-sample (SURVEY §8e: GroupNorm is per
        sample, attention is per sample), so a cfg2 step is exactly 8 such rows and
        steps/s(cfg2) = 1 / (8 * t_row) — a count of identical units, not a resolution / FLOP extrapolation."""

    def __init__(self, log=lambda *a: None, tiny=False):
        from oracle.config import SDXL, TINY, unet_flops
        from oracle.ddim import DDIMSchedule
        from oracle.unet import OracleUNet
        self.log, self.unet_flops = log, unet_flops
        self.cores = pick_host_threads(log)
        torch.set_num_threads(self.cores)
        self.cfg = TINY if tiny else SDXL
        self.tiny = tiny
        t0 = time.time()
        with torch.device("meta"):
            model = OracleUNet(self.cfg)
        model = model.to_empty(device="cpu")
        with torch.no_grad():
            for name, p in model.named_parameters():      # cheap fill: CPU time does not depend on the values
                if p.dim() == 1 and name.endswith("weight"):
                    p.fill_(1.0)
                elif name.endswith("bias"):
                    p.zero_()
                else:                                      # constant fill: ~10x faster to build than an RNG fill
                    fan_in = p[0].numel() if p.dim() > 1 else p.numel()
                    p.fill_(0.5 * fan_in ** -0.5)
        model.eval()
        model.set_ip_scale(IP_SCALE)
        self.model = model
        self.sch = DDIMSchedule()
        self.ts = self.sch.set_timesteps(T_STEPS)
        log(f"[reference] oracle UNet ({sum(p.numel() for p in model.parameters()) / 1e9:.2f} B params) built in "
            f"{time.time() - t0:.1f}s; {self.cores} host threads")

    @torch.no_grad()
    def cfg1_step(self, steps=3, warmup=1):
        bs, h, w = (1, 64, 64) if not self.tiny else (1, 16, 16)
        lat, ehs, pooled, time_ids, bbox, _ = synthetic_inputs(self.cfg, bs, h, w, 1, "cpu")
        def one(i, lat):
            t = self.ts[i % T_STEPS]
            eps = self.model(torch.cat([lat] * 2), t, ehs, pooled, time_ids, bbox, h / w, None)
            eu, et = eps.chunk(2)
            return self.sch.step(eu + GUIDANCE * (et - eu), t, lat)
        for i in range(warmup):
            lat = one(i, lat)
        times = []
        for i in range(steps):
            t0 = time.time()
            lat = one(warmup + i, lat)
            times.append(time.time() - t0)
        sec = statistics.median(times)
        fl = self.unet_flops(self.cfg, 2 * bs, h, w)
        return {"steps_per_sec": round(1.0 / sec, 5), "sec_per_step": round(sec, 3), "steps": steps, "warmup": warmup,
                "host_gflops": round(fl / sec / 1e9, 1),
                "workload": f"cfg1: {h * 8}x{w * 8} panel, bs={bs} (UNet batch {2 * bs}), 1 character ref, CFG "
                            f"{GUIDANCE}, fp32, full loop iteration (UNet + CFG blend + DDIM)"}

    @torch.no_grad()
    def cfg2_rows(self, steps, warmup):
        """-> (seconds per timed sample list) ; a sample = one batch row of the cfg2 step (see class docstring)."""
        h = w = 128 if not self.tiny else 16
        lat, ehs, pooled, time_ids, bbox, _ = synthetic_inputs(self.cfg, 1, h, w, 2, "cpu")
        ehs, pooled, time_ids, bbox = ehs[1:], pooled[1:], time_ids[1:], bbox[1:]     # the positive CFG row
        times = []
        for i in range(warmup + steps):
            t0 = time.time()
            t = self.ts[i % T_STEPS]
            eps = self.model(lat, t, ehs, pooled, time_ids, bbox, 1.0, None)
            lat = self.sch.step(eps, t, lat)     # DDIM update of the row (the CFG blend needs both rows: 2 FLOP/elt)
            if i >= warmup:
                times.append(time.time() - t0)
        fl = self.unet_flops(self.cfg, 1, h, w)
        return times, fl, (h, w)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    log = lambda *a: print(*a, file=sys.stderr)
    tiny = os.environ.get("DS_BENCH_TINY") == "1"          # plumbing self-test only; never a bench number
    ref = CpuReference(log, tiny)
    # warm-up: the W untimed iterations run the cfg1-size loop step (same modules, threads and allocator; 2.9 s each on
    # the box instead of 13.5 s for a cfg2 row), the last 3 of them are also the timed cfg1 measurement
    cfg1 = ref.cfg1_step(steps=3, warmup=max(1, args.warmup - 3))
    log(f"[reference] cfg1 as stated (B=2, 64x64 latent): {cfg1['sec_per_step']} s/step")
    times, fl, (h, w) = ref.cfg2_rows(args.steps, 0)
    t_row = sum(times) / max(len(times), 1)
    rows_per_step = 8
    value = 1.0 / (rows_per_step * t_row)
    sample = (f"one 'step' of this arm = ONE of the {rows_per_step} batch rows of a cfg2 step (UNet batch 1, latent "
              f"{h}x{w}, 2 character refs, fp32, {fl / 1e12:.3f} TFLOP): every op on the path is per-sample, so "
              f"steps/s = 1 / ({rows_per_step} x seconds per row) — a count of identical rows, no FLOP model; "
              f"{args.steps} timed rows after {max(4, args.warmup)} untimed cfg1-size loop iterations (the warm-up)")
    line = {"impl": "reference", "metric": METRIC, "value": round(value, 6), "unit": UNIT,
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": round(t_row * 1e3, 1), "ms_per_step_is": "one bounded sample (1/8 of a cfg2 step)",
            "sample_fraction_of_step": 1.0 / rows_per_step,
            "ms_per_full_step": round(rows_per_step * t_row * 1e3, 1),
            "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "cfg2: 1024x1024 panels, bs=4 per GPU (UNet batch 8), 2 character refs, 50 DDIM "
                                   f"steps, CFG {GUIDANCE}, ip_scale {IP_SCALE}",
                       "note": "reference CPU path = oracle restatement (diffusers absent on the box); bounded sample"},
            "cpu_baseline": {"value": round(value, 6), "unit": UNIT, "cores": ref.cores, "kind": "port",
                             "sample": sample, "host_gflops": round(fl / t_row / 1e9, 1)},
            "cfg1_measured": cfg1,
            "product_package_imported": "diffsensei_b200" in sys.modules,      # must be False: oracle only
            "e2e": {"value": round(value, 6), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)
    return 0


# ------------------------------------------------------------------------------------------------ GPU-library baseline
@torch.no_grad()
def library_baseline(dev, steps=3, warmup=2, log=lambda *a: None):
    """NOT the product path and not a target: the oracle modules in bf16 on the B200 with
    ``F.scaled_dot_product_attention`` — the cuBLAS / cuDNN / flash-attention kernels the reference itself would
    dispatch on a GPU (SURVEY §2.1), including its Python mask builder with its host syncs — timed for the cfg2 step
    so that "matches or beats the path the reference actually runs" has a measured denominator."""
    from oracle import attention as OA
    from oracle.config import SDXL
    from oracle.ddim import DDIMSchedule
    from oracle.unet import OracleUNet
    with torch.device("meta"):
        model = OracleUNet(SDXL)
    model = model.to_empty(device=dev).to(torch.bfloat16)
    g = torch.Generator(device=dev).manual_seed(5)
    for name, p in model.named_parameters():
        if p.dim() == 1 and name.endswith("weight"):
            p.fill_(1.0)
        elif name.endswith("bias"):
            p.zero_()
        else:
            fan_in = p[0].numel() if p.dim() > 1 else p.numel()
            p.copy_(torch.randn(p.shape, generator=g, device=dev) * fan_in ** -0.5)
    model.eval().set_ip_scale(IP_SCALE)
    OA.USE_SDPA = True
    try:
        lat, ehs, pooled, time_ids, bbox, _ = synthetic_inputs(SDXL, 4, 128, 128, 2, dev)
        lat, ehs, pooled = lat.to(dev), ehs.to(dev, torch.bfloat16), pooled.to(dev, torch.bfloat16)
        time_ids, bbox = time_ids.to(dev), bbox.to(dev)
        sch = DDIMSchedule()
        ts = sch.set_timesteps(T_STEPS)

        def one(i, lat):
            eps = model(torch.cat([lat] * 2).to(torch.bfloat16), ts[i], ehs, pooled, time_ids, bbox, 1.0, None).float()
            eu, et = eps.chunk(2)
            return sch.step(eu + GUIDANCE * (et - eu), ts[i], lat)
        for i in range(warmup):
            lat = one(i, lat)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            lat = one(warmup + i, lat)
        e1.record()
        e1.synchronize()
        ms = e0.elapsed_time(e1) / steps
    finally:
        OA.USE_SDPA = False
    del model
    torch.cuda.empty_cache()
    return {"value": round(1e3 / ms, 4), "unit": UNIT, "ms_per_step": round(ms, 2), "steps": steps, "warmup": warmup,
            "what": "oracle nn.Modules in bf16 on this GPU through torch's library kernels (cuBLAS GEMMs, cuDNN convs, "
                    "F.scaled_dot_product_attention, ATen GroupNorm/LayerNorm) + the reference's Python mask builder "
                    "(host syncs included), eager, no CUDA graph — the stack the reference dispatches; a stated "
                    "baseline, not the product path"}


# ------------------------------------------------------------------------------------------------ our arm
def family_roofline(ds, stepper, peaks, reps=2):
    """Time-weighted roofline of the tcgen05 GEMM family over the REAL shape census of one step: every ds_gemm_bf16 /
    ds_gemm_chain / ds_conv3x3_nhwc launch of an eager step is bracketed by CUDA events; achieved = sum(2*M*N*K) /
    sum(time)."""
    ops = ds.ops
    rec, on = [], [False]
    orig = {"gemm": ops.gemm, "conv3x3": ops.conv3x3}

    def gemm(a, w, *args, **kw):
        if not on[0]:
            return orig["gemm"](a, w, *args, **kw)
        K = a.shape[-1]
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        r = orig["gemm"](a, w, *args, **kw)
        e1.record()
        rec.append((f"gemm M{a.numel() // K} N{w.shape[0]} K{K}", 2.0 * (a.numel() // K) * w.shape[0] * K, e0, e1))
        return r

    def conv3x3(x, w, *args, **kw):
        if not on[0]:
            return orig["conv3x3"](x, w, *args, **kw)
        B, H, W, Cin = x.shape
        st = kw.get("stride", 1)
        up = kw.get("upsample", 1) if "upsample" in kw else 1
        Ho, Wo = ((H * up - 1) // st + 1, (W * up - 1) // st + 1)
        if kw.get("out_hw") is not None:
            Ho, Wo = kw["out_hw"]
        cin_total = Cin + (kw["x2"].shape[-1] if kw.get("x2") is not None else 0)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        r = orig["conv3x3"](x, w, *args, **kw)
        e1.record()
        rec.append((f"conv B{B} {Ho}x{Wo} {cin_total}->{w.shape[0]} s{st}", 2.0 * 9 * cin_total * w.shape[0] * Ho * Wo * B,
                    e0, e1))
        return r

    def gemm_chain(calls, **kw):
        if not on[0]:
            return orig["gemm_chain"](calls, **kw)
        a0 = calls[0][0][0]
        M = a0.numel() // a0.shape[-1]
        ws = [c[0][1] for c in calls]
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        r = orig["gemm_chain"](calls, **kw)
        e1.record()
        rec.append((f"chain M{M} " + ">".join(f"N{w.shape[0]}K{w.shape[1]}" for w in ws),
                    sum(2.0 * M * w.shape[0] * w.shape[1] for w in ws), e0, e1))
        return r

    orig["gemm_chain"] = ops.gemm_chain
    ops.gemm, ops.conv3x3, ops.gemm_chain = gemm, conv3x3, gemm_chain
    try:
        stepper.step(0)
        torch.cuda.synchronize()
        agg = {}
        for r in range(reps):
            rec.clear()
            on[0] = True
            stepper.step(1 + r)
            on[0] = False
            torch.cuda.synchronize()
            for key, fl, e0, e1 in rec:
                d = agg.setdefault(key, [0, 0.0, fl])
                d[0] += 1
                d[1] += e0.elapsed_time(e1)
    finally:
        ops.gemm, ops.conv3x3, ops.gemm_chain = orig["gemm"], orig["conv3x3"], orig["gemm_chain"]
    tot_ms = sum(d[1] for d in agg.values()) / reps
    tot_fl = sum(d[0] * d[2] for d in agg.values()) / reps
    ach = tot_fl / tot_ms / 1e9
    worst = sorted(((k, d[2] / (d[1] / d[0]) / 1e9, d[1] / reps) for k, d in agg.items() if d[1] / reps > 0.25),
                   key=lambda x: x[1])[:4]
    return {"kernel": "gemm_bf16_tcgen05 family (all ds_gemm_bf16 / ds_gemm_chain / ds_conv3x3_nhwc launches of one "
                      "cfg2 step)",
            "bound": "tensor", "achieved": round(ach, 1), "peak": peaks["bf16_tflops"], "unit": "TFLOP/s",
            "frac": round(ach / peaks["bf16_tflops"], 4),
            "frac_of_sustained": round(ach / peaks["bf16_tflops_sustained"], 4),
            "launches_per_step": sum(d[0] for d in agg.values()) // reps, "ms_per_step_in_family": round(tot_ms, 2),
            "TFLOP_per_step_in_family": round(tot_fl / 1e12, 2),
            "how": "per-launch CUDA events in an eager step (events add ~2 us per launch: a lower bound on achieved)",
            "slowest_shapes": [{"shape": k, "TFLOP/s": round(v, 0), "ms_per_step": round(m, 2)} for k, v, m in worst]}


def run_ours(args):
    import diffsensei_b200 as ds
    from diffsensei_b200 import parallel
    from diffsensei_b200.weights import random_state_dict, unet_param_shapes

    rank, world, local = parallel.init_from_env("nccl")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — diffsensei_b200 has no CPU path (use --impl reference)")
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    peaks = measured_peaks()
    cfg = ds.SDXL_MANGA if args.config != "tiny" else ds.TINY
    groups = config_panels(args.config)
    if args.dump_outputs:
        # the dump's size follows from the shapes alone: every rank refuses the same run before any work is timed
        dump_bytes = sum(bs * world * 4 * h * w * 4 for bs, h, w, *_ in groups)
        if dump_bytes > DUMP_LIMIT_BYTES:
            raise SystemExit(f"bench.py: --dump-outputs would write {dump_bytes} bytes, more than {DUMP_LIMIT_BYTES}")

    t0 = time.time()
    engine = ds.UNetMangaEngine(cfg, dev)
    sd = random_state_dict(unet_param_shapes(cfg), seed=UNET_WEIGHT_SEED, device=dev, dtype=torch.bfloat16)
    engine.load_state_dict(sd)
    del sd
    torch.cuda.empty_cache()
    engine.set_ip_scale(IP_SCALE)
    pipe = ds.DiffSenseiPipeline(engine)
    # N > 1 (cfg4 = bs 32 over 8 GPUs): ONE global batch of bs * world panels (every rank builds the same seeded global
    # tensors), sharded contiguously with parallel.shard_range; the final latents are all-gathered in panel order
    inputs, shards = [], []
    for bs, h, w, nc, dlg, ml in groups:
        glob = synthetic_inputs(cfg, bs * world, h, w, nc, dev, dialogs=dlg, mllm=ml)
        s0, s1 = parallel.shard_range(bs * world, world, rank)
        assert s1 - s0 == bs
        shards.append((s0, s1))
        inputs.append(shard_inputs(glob, s0, s1) if world > 1 else glob)
    steppers = [pipe.make_stepper(*inp[:5], g[1] / g[2], inp[5], T_STEPS, GUIDANCE, use_graph=True, chains=args.chains)
                for g, inp in zip(groups, inputs)]
    stepper = steppers[0]
    bs_total = sum(g[0] for g in groups)
    torch.cuda.synchronize()
    if rank == 0:
        print(f"[bench] engine + {len(steppers)} graph(s) ready in {time.time() - t0:.1f}s", file=sys.stderr)

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    def step_all(i):
        for st in steppers:                       # one "step" = one denoise iteration of EVERY panel of the batch
            st.step(i % T_STEPS)

    # ---- value: device-resident loop
    for i in range(args.warmup):
        step_all(i)
    barrier()
    with ClockSampler(local) as clk:
        ms = event_time_ms(lambda i: step_all(args.warmup + i), args.steps)
        barrier()
    ms = parallel.max_over_ranks(ms, dev)
    steps_per_sec = world * 1e3 / ms
    clocks = clk.summary()
    if args.dump_outputs:
        # the latents the last timed step left, taken before the legs below overwrite them
        dump = {f"latents_{g[1] * 8}x{g[2] * 8}": parallel.gather_latents(st.latents_nchw(), [g[0]] * world)
                for g, st in zip(groups, steppers)}
        if rank == 0:
            dump_outputs(args.dump_outputs, dump)

    # ---- e2e: the same call with HOST buffers (pinned), H2D + step + D2H inside the timed region
    hosts = [(torch.randn(g[0], 4, g[1], g[2]).pin_memory(), torch.empty(g[0], 4, g[1], g[2]).pin_memory())
             for g in groups]

    def step_host_all(i):
        for st, (hi, ho) in zip(steppers, hosts):
            st.step_host(i % T_STEPS, hi, ho)
    for i in range(2):
        step_host_all(i)
    barrier()
    e_ms = event_time_ms(step_host_all, args.steps)
    barrier()
    e_ms = parallel.max_over_ranks(e_ms, dev)
    h2d = sum(hi.numel() * 4 for hi, _ in hosts)
    e2e = {"value": round(world * 1e3 / e_ms, 4), "unit": UNIT, "h2d_bytes_per_step": h2d,
           "d2h_bytes_per_step": h2d, "ms_per_step": round(e_ms, 3)}

    # ---- measured panels: whole panels through DiffSenseiPipeline.denoise (per-panel setup INCLUDED: K|V projections
    # of all 70 cross-attention layers, the 50-row time-embedding table, refill of the captured graph's buffers;
    # the graph itself is captured once per shape and re-used), host latents in, host latents out
    panel = None
    if not args.no_panels:
        g0, inp0 = groups[0], inputs[0]
        n_pan = 2

        def run_panel(k):
            lat_h = torch.randn(g0[0], 4, g0[1], g0[2], generator=torch.Generator().manual_seed(100 + k)).pin_memory()
            out = pipe.denoise(lat_h, inp0[1], inp0[2], inp0[3], inp0[4], g0[1] / g0[2], inp0[5], T_STEPS, GUIDANCE,
                               use_graph=True)
            return out.cpu()
        torch.cuda.synchronize()
        t_cap = time.perf_counter()
        run_panel(-1)                                # first panel of this shape: captures (and caches) the graph
        t_cap = time.perf_counter() - t_cap
        st_cached = pipe.stepper_for(inp0[0], inp0[1], inp0[2], inp0[3], inp0[4], g0[1] / g0[2], inp0[5], T_STEPS,
                                     GUIDANCE)
        torch.cuda.synchronize()
        t_set = time.perf_counter()
        st_cached.load_panel(inp0[0], inp0[1], inp0[2], inp0[3], inp0[4], inp0[5])
        torch.cuda.synchronize()
        t_set = time.perf_counter() - t_set
        barrier()
        t_p = time.perf_counter()
        for k in range(n_pan):
            run_panel(k)
        torch.cuda.synchronize()
        t_p = time.perf_counter() - t_p
        t_p = parallel.max_over_ranks(t_p, dev)
        # ... and the step right after the loop (pipeline_diffsensei.py:339-363): latents / scaling_factor -> VAE decode
        # -> post-process, on the SDXL-size decoder (random-init weights), per panel batch
        vae_ms = None
        if args.config in ("cfg2", "cfg1", "tiny"):
            from diffsensei_b200.weights import vae_decoder_param_shapes
            vcfg = ds.SDXL_VAE if args.config != "tiny" else ds.TINY_VAE
            vae = ds.VaeDecoderEngine(vcfg, dev)
            vae.load_state_dict(random_state_dict(vae_decoder_param_shapes(vcfg), seed=99, device=dev, dtype=torch.bfloat16))
            lat_fin = stepper.latents_nchw()
            vae.decode_image(lat_fin)
            torch.cuda.synchronize()
            tv = time.perf_counter()
            img = vae.decode_image(lat_fin)
            img_host = img.cpu()
            vae_ms = (time.perf_counter() - tv) * 1e3
            assert img_host.shape == (g0[0], 3, g0[1] * 8, g0[2] * 8)
            del vae, img
            torch.cuda.empty_cache()
        panel = {"panels_per_sec": round(world * n_pan * g0[0] / t_p, 4), "unit": "panels/s",
                 "panel_batches": n_pan, "panels_per_batch": g0[0], "steps_per_panel": T_STEPS,
                 "sec_per_panel_batch": round(t_p / n_pan, 4),
                 "setup_ms_per_panel_batch": round(t_set * 1e3, 2),
                 "setup_share": round(t_set / (t_p / n_pan), 5),
                 "first_panel_with_graph_capture_s": round(t_cap, 3),
                 "vae_decode_ms_per_panel_batch": None if vae_ms is None else round(vae_ms, 2),
                 "panels_per_sec_incl_vae_decode": None if vae_ms is None else
                 round(world * n_pan * g0[0] / (t_p + n_pan * vae_ms * 1e-3), 4),
                 "how": "wall clock around DiffSenseiPipeline.denoise x panel_batches (host latents in / out, "
                        "prepare_conditions + time-embedding table + graph-buffer refill inside, CUDA graph re-used)"}

    # launches per step: count one eager (non-graph) iteration — graph replays re-issue the same kernels
    per_step = 0
    eager0 = None
    for g, inp in zip(groups, inputs):
        eager = pipe.make_stepper(*inp[:5], g[1] / g[2], inp[5], T_STEPS, GUIDANCE, use_graph=False, chains=args.chains)
        torch.cuda.synchronize()
        n0 = ds.ops.launch_count()
        eager.step(0)
        torch.cuda.synchronize()
        per_step += ds.ops.launch_count() - n0
        eager0 = eager0 or eager

    # one NCCL all-gather of the final latents (outside the timed region): the only collective of the path
    mine = stepper.latents_nchw()
    final = parallel.gather_latents(mine, [groups[0][0]] * world)
    assert final.shape[0] == groups[0][0] * world
    assert torch.equal(final[shards[0][0]:shards[0][1]], mine)       # gathered in global panel order

    extra = {}
    if rank == 0 and args.config == "cfg2" and not args.no_kernel_rooflines:
        extra = kernel_rooflines(ds, peaks, dev)
        try:
            extra["roofline_family"] = family_roofline(ds, eager0, peaks)
        except Exception as e:                                   # never lose the bench line to a diagnostics leg
            extra["roofline_family"] = {"error": repr(e)}
    del eager0
    cfg1_gpu = None
    if rank == 0 and world == 1 and args.config == "cfg2" and not args.no_cpu_baseline:
        i1 = synthetic_inputs(cfg, 1, 64, 64, 1, dev)
        s1 = pipe.make_stepper(*i1[:5], 1.0, None, T_STEPS, GUIDANCE, use_graph=True)
        for i in range(3):
            s1.step(i)
        torch.cuda.synchronize()
        m1 = event_time_ms(lambda i: s1.step((3 + i) % T_STEPS), 10)
        cfg1_gpu = {"steps_per_sec": round(1e3 / m1, 3), "ms_per_step": round(m1, 3),
                    "workload": "cfg1: 512x512 panel, bs=1 (UNet batch 2), 1 character ref, bf16, graph replay"}
        del s1
    lib = None
    if rank == 0 and world == 1 and args.config == "cfg2" and not args.no_library_baseline:
        try:
            lib = library_baseline(dev, log=lambda *a: print(*a, file=sys.stderr))
        except Exception as e:
            lib = {"error": repr(e)}
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        ref = CpuReference(lambda *a: print(*a, file=sys.stderr), tiny=args.config == "tiny")
        c1 = ref.cfg1_step(steps=3, warmup=1)
        times, fl, (hh, ww) = ref.cfg2_rows(2, 0)           # the cfg1 steps above already warmed the process up
        t_row = sum(times) / len(times)
        cpu = {"value": round(1.0 / (8 * t_row), 6), "unit": UNIT, "cores": ref.cores, "kind": "port",
               "sample": f"2 timed batch rows of the cfg2 step (UNet batch 1, latent {hh}x{ww}, fp32, "
                         f"{fl / 1e12:.3f} TFLOP each; a cfg2 step = 8 such rows, no FLOP model), after the cfg1 steps",
               "sec_per_row": round(t_row, 3), "host_gflops": round(fl / t_row / 1e9, 1), "cfg1_measured": c1}
        if cfg1_gpu:
            cpu["cfg1_same_config_ratio"] = round(cfg1_gpu["steps_per_sec"] / c1["steps_per_sec"], 1)
        del ref
    if rank == 0:
        tflop = STEP_TFLOP_CFG2 if args.config == "cfg2" else None
        desc = "; ".join(f"{g[0]}x {g[1] * 8}x{g[2] * 8}" for g in groups)
        line = {"metric": METRIC, "value": round(steps_per_sec, 4), "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": round(ms, 3), "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
                "config": {"workload": f"{args.config}: panels (count x HxW) {desc} per GPU (UNet batch {2 * bs_total}), "
                                       f"{groups[0][3]} character refs, {T_STEPS} DDIM steps, CFG {GUIDANCE}, "
                                       f"ip_scale {IP_SCALE}" + (", dialog boxes" if groups[0][4] else "")
                                       + (", MLLM-adapted image tokens" if groups[0][5] else ""),
                           "weights": "random-init SDXL+IP topology (2.908 B params), bf16",
                           "parallelism": f"dp{world}: one global batch of {bs_total * world} panels, contiguous shards of "
                                          f"{bs_total} per GPU (parallel.shard_range), no per-step collective, final "
                                          "latents all-gathered in panel order",
                           "l2": "working set per step (5.8 GB weights + activations) >> 126 MB L2; no explicit flush",
                           "hoisted": "text/IP K|V projections (0.86 TFLOP/step) and time embeddings are computed "
                                      "once per panel, outside the timed step (inside the measured `panel` leg)"},
                "panels_per_sec": round(world * bs_total * 1e3 / (ms * T_STEPS), 4),
                "panels_per_sec_is": "derived from the step time (bs / (T * ms_per_step)); `panel` is the measurement",
                "panel": panel,
                "gpu_launches": per_step * args.steps, "launches_per_step": per_step,
                "e2e": e2e, "clocks": clocks}
        if tflop:
            hoisted = 0.856
            ach, ach_in = tflop / (ms * 1e-3), (tflop - hoisted) / (ms * 1e-3)
            line["mfu"] = {"model_tflop_per_step": tflop, "tflop_per_step_executed_in_timed_region": tflop - hoisted,
                           "achieved_tflops_per_gpu_model": round(ach, 1),
                           "achieved_tflops_per_gpu_executed": round(ach_in, 1),
                           "frac_of_sustained_peak_model": round(ach / peaks["bf16_tflops_sustained"], 4),
                           "frac_of_sustained_peak_executed": round(ach_in / peaks["bf16_tflops_sustained"], 4),
                           "frac_of_burst_peak_executed": round(ach_in / peaks["bf16_tflops"], 4),
                           "peak": peaks["bf16_tflops_sustained"], "peak_source": peaks["source"] + " sustained",
                           "note": "'model' counts the reference's per-step work incl. the 0.856 TFLOP of text/IP K|V "
                                   "projections this engine hoists out of the loop; 'executed' counts only what the "
                                   "timed step runs (BASELINE.md §2 asks for both)"}
        line.update(extra)
        if "roofline" not in line:
            line["roofline"] = None
        line["cfg1_gpu"] = cfg1_gpu
        line["gpu_library_baseline"] = lib
        if lib and lib.get("value"):
            line["vs_gpu_library_baseline"] = round(steps_per_sec / lib["value"], 2)
        line["cpu_baseline"] = cpu
        emit(line)
    if world > 1:
        torch.distributed.destroy_process_group()
    return 0


_JSON_FD = None


def emit(line: dict) -> None:
    """The ONE JSON line of the contract, on the process's original stdout (see `main`)."""
    data = (json.dumps(line) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_JSON_FD, data)


def main():
    # Libraries write to fd 1 behind Python's back (NCCL prints "NCCL version ..." there on the first collective):
    # keep the original stdout for the JSON line only and send everything else to stderr.
    global _JSON_FD
    sys.stdout.flush()
    _JSON_FD = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--config", choices=["cfg2", "cfg1", "cfg3", "cfg5", "tiny"], default="cfg2")
    ap.add_argument("--no-panels", action="store_true")
    ap.add_argument("--no-library-baseline", action="store_true")
    ap.add_argument("--chains", type=int, default=None,
                    help="concurrent kernel chains per GPU (default: DS_CHAINS env, else 2)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-kernel-rooflines", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the latents of the last timed step to DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to --impl ours")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    return run_reference(args) if args.impl == "reference" else run_ours(args)


if __name__ == "__main__":
    sys.exit(main())

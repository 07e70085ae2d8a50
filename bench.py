#!/usr/bin/env python
"""bench.py -- video-latent tokens/s per denoising step of the Wan DiT forward on B200(s).

  python bench.py --gpus N --steps K --warmup W            (N > 1: launched by torchrun, one rank per GPU)
  python bench.py --impl reference --steps K --warmup W    (the CPU arm: oracle port on the host cores)
  python bench.py ... --dump-outputs DIR                   (also writes the last timed step's output to DIR/*.npy)

Workload (BASELINE.json metric): Wan2.2-T2V-14B architecture (D 5120, 40 heads, ffn 13824, 40 layers), 720p x 81f
latent 16x21x90x160 -> 75 600 tokens, Video-Sparse attention at sparsity 0.9 (top-k 144 of 1440 tiles), synthetic
latents/text and random-init weights, bf16. One "step" = one full transformer forward (the per-denoising-step cost).
N > 1 shards the 75 600 tokens with Ulysses sequence parallelism (strong scaling: the job is one sample).

One JSON line on rank 0; see DESIGN.md "Measurement" for how every field is obtained.
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
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (arch kwargs, latent (C, T, H, W), text_len, vsa_sparsity)
    "wan2.2-t2v-14b_720p_81f_vsa0.9": (dict(hidden_size=5120, num_attention_heads=40, ffn_dim=13824, num_layers=40),
                                        (16, 21, 90, 160), 512, 0.9),
    "fastwan-1.3b_480p_81f_dense": (dict(hidden_size=1536, num_attention_heads=12, ffn_dim=8960, num_layers=30),
                                    (16, 21, 60, 104), 512, None),
}
DEFAULT_WORKLOAD = "wan2.2-t2v-14b_720p_81f_vsa0.9"
METRIC = "video-latent tokens/sec per denoising step"


def load_traffic():
    """Per-launch DRAM bytes of the kernel families from the committed `ncu --set full` capture of this same command
    (profiles/r2_kernel_traffic.json, written by tools/ncu_traffic.py from the .ncu-rep; dram__bytes_read.sum +
    dram__bytes_write.sum averaged over the captured launches of the family)."""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "r2_kernel_traffic.json")))
    except Exception:
        return {}


def measured_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md 'clocks line')."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int = 0):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, pw = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1])); pw.append(float(r[2]))
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        busy = [s for s, p in zip(sm, pw) if p > 300] or sm
        return {"sm_mhz": statistics.median(busy) if busy else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


# ----------------------------------------------------------------------------------------------------------------
# CPU arm: the reference's own PyTorch-CPU path (dense SDPA WanTransformerBlock) timed on the host cores
# ----------------------------------------------------------------------------------------------------------------
CPU_SIZES = (1024, 4096, 9450)  # SURVEY.md section 8d: S in {1024, 4096, 9450} at the true width, then extrapolate


def _reference_root():
    """Where the reference's Python lies: the build container has /root/reference; the GPU box only has what
    oracle/stage_ref_kernels.py staged into oracle/_ref/reference_py (git-ignored, travels with the snapshot)."""
    for cand in (os.environ.get("FVB_REFERENCE_ROOT"), "/root/reference", os.path.join(ROOT, "oracle", "_ref", "reference_py")):
        if cand and os.path.isdir(os.path.join(cand, "fastvideo", "models", "dits")):
            return cand
    return None


class CpuBlock:
    """One transformer block at the workload's true width on the CPU, bf16: the REFERENCE's WanTransformerBlock with its
    torch-SDPA backend when the reference's Python is importable (kind "reference"), else the oracle's restatement of
    it (oracle/wan_ref.py, bit-exact against the reference on CPU -- kind "port"). This is the reference's CPU-runnable
    path (BASELINE.md section 2 "B-CPU"): dense attention; its Triton VSA kernels do not run on a CPU."""

    def __init__(self, arch: dict, threads: int):
        import torch
        from oracle import wan_ref
        torch.set_num_threads(threads)
        self.torch, self.wan_ref = torch, wan_ref
        self.D, self.H, self.F = arch["hidden_size"], arch["num_attention_heads"], arch["ffn_dim"]
        D, H, F_ = self.D, self.H, self.F
        g = torch.Generator().manual_seed(0)
        sd = {}

        def lin(n, o, i):
            sd[n + ".weight"] = (torch.randn(o, i, generator=g) / i ** 0.5).bfloat16()
            sd[n + ".bias"] = torch.zeros(o).bfloat16()

        for n in ["to_q", "to_k", "to_v", "to_out", "attn2.to_q", "attn2.to_k", "attn2.to_v", "attn2.to_out"]:
            lin(n, D, D)
        lin("ffn.fc_in", F_, D)
        lin("ffn.fc_out", D, F_)
        for n in ["norm_q", "norm_k", "attn2.norm_q", "attn2.norm_k", "self_attn_residual_norm.norm"]:
            sd[n + ".weight"] = torch.ones(D).bfloat16()
        sd["self_attn_residual_norm.norm.bias"] = torch.zeros(D).bfloat16()
        sd["scale_shift_table"] = (torch.randn(1, 6, D, generator=g) / D ** 0.5).bfloat16()
        self.sd, self.g = sd, g
        self.kind, self.blk, self.ctxmgr = "port", None, None
        root = _reference_root()
        if root is not None and os.environ.get("FVB_CPU_ARM", "") != "port":
            try:
                os.environ["FVB_REFERENCE_ROOT"] = root
                from oracle import ref_shim
                ref_shim.install()
                from fastvideo.forward_context import set_forward_context
                from fastvideo.models.dits.wanvideo import WanTransformerBlock
                from fastvideo.platforms import AttentionBackendEnum
                blk = WanTransformerBlock(D, F_, H, "rms_norm_across_heads", True, 1e-6, None, (AttentionBackendEnum.TORCH_SDPA, ))
                res = blk.load_state_dict(sd, strict=False)
                assert not res.unexpected_keys and not res.missing_keys, res
                self.blk = blk.to(torch.bfloat16).eval()
                self.ctxmgr = set_forward_context
                self.kind = "reference"
            except Exception as e:  # noqa: BLE001 -- the port is the documented fallback of this arm
                print(f"[bench] reference block not constructible ({type(e).__name__}: {e}); timing the oracle port", file=sys.stderr)

    def grid(self, S: int):
        # a (T, H, W) token grid with T*H*W == S (RoPE tables only; the block's cost does not depend on the shape)
        for t in (21, 16, 8, 4, 2, 1):
            if S % t == 0:
                hw = S // t
                h = int(hw ** 0.5)
                while hw % h:
                    h -= 1
                return (t, h, hw // h)
        return (1, 1, S)

    def time_block(self, S: int) -> float:
        torch, wan_ref = self.torch, self.wan_ref
        D, H = self.D, self.H
        x = torch.randn(1, S, D, generator=self.g).bfloat16()
        ctx = torch.randn(1, 512, D, generator=self.g).bfloat16()
        temb6 = (torch.randn(1, 6, D, generator=self.g) * 0.5).bfloat16()
        d = D // H
        cos, sin = wan_ref.rotary_tables(self.grid(S), [d - 4 * (d // 6), 2 * (d // 6), 2 * (d // 6)])
        with torch.no_grad():
            t0 = time.perf_counter()
            if self.blk is not None:
                with self.ctxmgr(current_timestep=0, attn_metadata=None):
                    self.blk(x, ctx, temb6, (cos, sin), S)
            else:
                wan_ref.wan_block(x, ctx, temb6, self.sd, "", H, cos, sin)
            return time.perf_counter() - t0


def fit_and_extrapolate(points: dict, S_target: int, layers: int):
    """t_block(S) = a*S + b*S^2 (GEMM terms linear, attention quadratic -- SURVEY.md section 8d), least squares through
    the measured (S, seconds) points; returns (tokens/s at S_target for `layers` blocks, a, b, t_block(S_target))."""
    import numpy as np
    Ss = np.array(sorted(points), dtype=np.float64)
    ts = np.array([statistics.median(points[int(S_)]) for S_ in Ss], dtype=np.float64)
    if len(Ss) >= 2:
        A = np.stack([Ss, Ss * Ss], 1)
        (a, b), *_ = np.linalg.lstsq(A / ts[:, None], np.ones_like(ts), rcond=None)  # relative-error weighting
        if b < 0:  # noise on the small sizes: fall back to the linear term alone (an UNDER-estimate of the CPU time)
            a, b = float((ts / Ss).mean()), 0.0
    else:
        a, b = float(ts[0] / Ss[0]), 0.0
    t_target = a * S_target + b * S_target * S_target
    return S_target / (t_target * layers), float(a), float(b), float(t_target)


def cpu_arm_measure(arch: dict, S_target: int, steps: int, warmup: int, threads: int, sizes=CPU_SIZES, big_once: bool = True):
    blk = CpuBlock(arch, threads)
    for _ in range(max(warmup, 1)):
        blk.time_block(sizes[0])
    points = {S: [] for S in sizes}
    step_s = []
    for k in range(steps):
        t_step = 0.0
        for S in sizes:
            if big_once and S == max(sizes) and k > 0:
                continue  # the largest size is timed once: it alone is most of a step's budget
            t = blk.time_block(S)
            points[S].append(t)
            t_step += t
        step_s.append(t_step)
    points = {S: v for S, v in points.items() if v}
    value, a, b, t_target = fit_and_extrapolate(points, S_target, arch["num_layers"])
    spread = {str(S): [round(min(v), 3), round(statistics.median(v), 3), round(max(v), 3)] for S, v in points.items()}
    sample = (f"{'the reference WanTransformerBlock (fastvideo/models/dits/wanvideo.py:361-434, torch-SDPA backend)' if blk.kind == 'reference' else 'oracle/wan_ref.py port of WanTransformerBlock (bit-exact vs the reference on CPU)'}"
              f" at the true width D={arch['hidden_size']}, bf16 torch CPU, {threads} threads, S in {sorted(points)} tokens "
              f"(seconds min/median/max per size: {spread}); t_block(S) = a*S + b*S^2 fitted (a={a:.3e}, b={b:.3e}) and "
              f"extrapolated to S={S_target}: {t_target:.0f} s per block x {arch['num_layers']} layers; dense attention (the "
              f"reference's CPU-runnable path), embedders/head excluded (<1% of FLOPs)")
    return dict(value=value, kind=blk.kind, sample=sample, points=spread, a=a, b=b, t_block_target_s=t_target,
                step_seconds=step_s)


def run_reference_arm(args, rank, world):
    if rank != 0:
        return
    arch, latent, text_len, sparsity = WORKLOADS[args.workload]
    C, T, Hh, Ww = latent
    S_target = T * (Hh // 2) * (Ww // 2)
    threads = os.cpu_count() or 1
    sizes = tuple(int(x) for x in args.cpu_sizes.split(",")) if args.cpu_sizes else CPU_SIZES
    m = cpu_arm_measure(arch, S_target, args.steps, args.warmup, threads, sizes=sizes, big_once=len(sizes) > 2)
    ms_step = statistics.mean(m["step_seconds"]) * 1e3
    line = {"impl": "reference", "metric": METRIC, "value": m["value"], "unit": "tokens/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": args.workload, "tokens": S_target, "latent": list(latent), "text_len": text_len,
                       "model": "Wan2.2-T2V-A14B expert (random init)" if arch["hidden_size"] == 5120 else "Wan2.1-T2V-1.3B (random init)",
                       "layers": arch["num_layers"],
                       "note": "CPU arm: each step times one block on a bounded token sample per size; the value is the fitted cost "
                               "extrapolated to the workload's token count and layer count (ms_per_step = CPU seconds actually spent per step)",
                       "extrapolation": {"model": "t_block(S) = a*S + b*S^2", "a": m["a"], "b": m["b"], "S": S_target,
                                         "t_block_s": m["t_block_target_s"], "sizes_s": m["points"]}},
            "cpu_baseline": {"value": m["value"], "unit": "tokens/s", "cores": threads, "kind": m["kind"], "sample": m["sample"]},
            "e2e": {"value": m["value"], "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)


# HBM-bound row / index kernels of the GPU arm: "work" = algorithmic bytes (every operand row read once, every result row
# written once). Module level so that tests/test_bench_contract.py can call them with the call shapes of both the single-GPU
# and the sequence-parallel forward.
def nbytes(t):
    return float(t.numel() * t.element_size()) if t is not None else 0.0

def ln_bytes(x, *a, **k):
    return nbytes(x) + x.numel() * 2.0 * (2.0 if k.get("want_hidden") else 1.0)

def rope_bytes(x0, w0, x1=None, *a, **k):
    return 2.0 * nbytes(x0) + 2.0 * nbytes(x1)

def rope_scatter_bytes(x0, w0, x1, *a, **k):
    return 2.0 * nbytes(x0) + 2.0 * nbytes(x1)

def mean_bytes(x, nblk, *a, **k):
    return nbytes(x) + x.shape[0] * x.shape[2] * nblk * x.shape[3] * 2.0 * (2.0 if k.get("want_transposed") else 1.0)

def softmax_bytes(x, *a, **k):
    return 2.0 * nbytes(x)

def topk_bytes(scores, *a, **k):
    return nbytes(scores) + scores.numel() * 4.0 + (scores.numel() if k.get("want_mask") else 0.0)

def combine_bytes(out_s, out_c, gate, *a, **k):
    return 2.0 * nbytes(out_s) + nbytes(gate) + nbytes(out_c)


# ----------------------------------------------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------------------------------------------
class KernelTimer:
    """CUDA-event pairs around every launch of one kernel family inside the timed region (torch current stream ==
    the launch stream of every fvb_* call)."""

    def __init__(self):
        self.pairs, self.work, self.enabled = [], 0.0, False

    def wrap(self, fn, work_fn, tag_fn=None):
        import torch

        def inner(*a, **k):
            if not self.enabled:
                return fn(*a, **k)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            r = fn(*a, **k)
            e1.record()
            try:
                w = work_fn(*a, **k)
            except Exception:  # a work model must never take the measurement down; the launch is still timed
                w = 0.0
            self.pairs.append((e0, e1, w, tag_fn(*a, **k) if tag_fn else None))
            self.work += w
            return r
        return inner

    def result(self):
        ms = sum(a.elapsed_time(b) for a, b, _, _ in self.pairs)
        return ms, self.work, len(self.pairs)

    def by_tag(self):
        """Per distinct launch shape: launches, summed ms, achieved TFLOP/s -- shows WHICH GEMM falls off when N grows."""
        agg = {}
        for a, b, w, tag in self.pairs:
            if tag is None:
                continue
            d = agg.setdefault(tag, [0, 0.0, 0.0])
            d[0] += 1
            d[1] += a.elapsed_time(b)
            d[2] += w
        return [{"shape": t, "launches": n, "ms": round(ms, 3), "tflops": round(w / ms / 1e9, 1) if ms else None}
                for t, (n, ms, w) in sorted(agg.items(), key=lambda kv: -kv[1][1])]


def run_gpu_arm(args, rank, world, device):
    import torch
    import torch.distributed as dist
    from fastvideo_b200 import _lib, ops, vsa
    from fastvideo_b200.api import WanDenoiser
    from fastvideo_b200.wan_dit import WanDiT, WanDiTConfig

    arch, latent, text_len, sparsity = WORKLOADS[args.workload]
    arch = dict(arch)
    if args.layers:
        arch["num_layers"] = args.layers  # development only: flagged in the output, never the driver's run
    cfg = WanDiTConfig(vsa=sparsity is not None, **arch)
    t0 = time.time()
    model = WanDiT.random(cfg, device)
    den = WanDenoiser(model, rank, world, vsa_sparsity=sparsity)
    torch.cuda.synchronize()
    if rank == 0:
        print(f"[bench] model built in {time.time() - t0:.1f}s, {torch.cuda.memory_allocated() / 2**30:.1f} GiB", file=sys.stderr)

    g = torch.Generator().manual_seed(1024)
    C, T, Hh, Ww = latent
    lat_h = torch.randn(1, C, T, Hh, Ww, generator=g).bfloat16().pin_memory()
    txt_h = torch.randn(1, text_len, cfg.text_dim, generator=g).bfloat16().pin_memory()
    lat_d, txt_d = lat_h.to(device), txt_h.to(device)
    t_d = torch.full((1,), 500.0, device=device)
    S_tokens = (T // cfg.patch_size[0]) * (Hh // cfg.patch_size[1]) * (Ww // cfg.patch_size[2])

    vsa_topk = model.layout((T // cfg.patch_size[0], Hh // cfg.patch_size[1], Ww // cfg.patch_size[2]), device, sparsity).topk \
        if sparsity is not None else 0

    # kernel-family timers (dominant kernel = the tcgen05 GEMM; second = the attention kernel)
    gemm_t, attn_t, attn_d, rows_t = KernelTimer(), KernelTimer(), KernelTimer(), KernelTimer()

    def gemm_work_linear(x, w, *a, **k):
        return 2.0 * x.numel() / x.shape[-1] * w.shape[0] * w.shape[1]

    def gemm_work_sp(x, M, K, ldx, w, *a, **k):
        return 2.0 * M * K * w.shape[0]

    def gemm_work_batched(a_, b_, *a, **k):
        return 2.0 * a_.shape[0] * a_.shape[1] * b_.shape[1] * a_.shape[2]

    def attn_work(q, k_, v, *a, **kw):
        B, Sq, H, d = q.shape
        if kw.get("sched") is not None:
            nblk = kw["nqb"]
            return 4.0 * B * H * nblk * 64 * vsa_topk * 64 * d  # the reference's FLOP model (bench_vsa.py:84-86)
        return 4.0 * B * H * Sq * k_.shape[1] * d

    def tag_linear(x, w, bias=None, epilogue=0, *a, **k):
        return f"M{x.numel() // x.shape[-1]}xN{w.shape[0]}xK{w.shape[1]}:epi{k.get('epilogue', epilogue)}"

    def tag_sp(x, M, K, ldx, w, bias, out, ldo, epilogue=0, *a, **k):
        kind = "peer-scatter" if k.get("out_col_offsets") is not None else ("kseg" if k.get("x_seg_len") else "plain")
        return f"M{M}xN{w.shape[0]}xK{K}:epi{k.get('epilogue', epilogue)}:{kind}"

    ops.linear = gemm_t.wrap(ops.linear, gemm_work_linear, tag_linear)
    ops.linear_sp = gemm_t.wrap(ops.linear_sp, gemm_work_sp, tag_sp)
    ops.gemm_batched = gemm_t.wrap(ops.gemm_batched, gemm_work_batched)
    def attn_work_bl(q, k_, v, q2k_idx, q2k_num, *a, **kw):
        B, Sq, H, d = q.shape
        return 4.0 * B * H * q2k_idx.shape[2] * 64 * vsa_topk * 64 * d  # the reference's FLOP model (bench_vsa.py:84-86)

    ops.attention = attn_d.wrap(ops.attention, attn_work)
    ops.attention_blocklist = attn_t.wrap(ops.attention_blocklist, attn_work_bl)

    ops.layernorm_modulate = rows_t.wrap(ops.layernorm_modulate, ln_bytes)
    ops.rmsnorm_rope_ = rows_t.wrap(ops.rmsnorm_rope_, rope_bytes)
    ops.rmsnorm_rope_scatter = rows_t.wrap(ops.rmsnorm_rope_scatter, rope_scatter_bytes)
    ops.block_mean = rows_t.wrap(ops.block_mean, mean_bytes)
    ops.softmax_rows = rows_t.wrap(ops.softmax_rows, softmax_bytes)
    ops.topk_index = rows_t.wrap(ops.topk_index, topk_bytes)
    ops.vsa_combine = rows_t.wrap(ops.vsa_combine, combine_bytes)

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- warm-up ----
    for _ in range(args.warmup):
        out = den.forward_device(lat_d, txt_d, t_d)
    sync_all()

    # ---- timed region: K steps, inputs resident in HBM ----
    sampler = ClockSampler(device.index or 0)
    if rank == 0:
        sampler.start()
    gemm_t.enabled = attn_t.enabled = attn_d.enabled = rows_t.enabled = True
    launches0 = _lib.LAUNCHES
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sync_all()
    e0.record()
    for _ in range(args.steps):
        out = den.forward_device(lat_d, txt_d, t_d)
    e1.record()
    sync_all()
    launches = _lib.LAUNCHES - launches0
    gemm_t.enabled = attn_t.enabled = attn_d.enabled = rows_t.enabled = False
    ms_total = torch.tensor([e0.elapsed_time(e1)], device=device)
    if world > 1:
        dist.all_reduce(ms_total, op=dist.ReduceOp.MAX)
    ms_step = ms_total.item() / args.steps

    # ---- end to end through the public API: pinned host in, pinned host out, copies inside the timed region ----
    for _ in range(1):
        res0 = den.step(lat_h, txt_h, 500)  # first call captures the CUDA graph (after its own eager warm-up)
    sync_all()
    # the graph replays the same kernels on the same inputs as the eager forward above: demand the same bits, else run eagerly
    graph_check = None
    if den._graph is not None:
        graph_check = bool(torch.equal(res0.to(device), out))
        if not graph_check:
            print("[bench] CUDA-graph output differs from the eager forward: falling back to eager launches", file=sys.stderr)
            den._graph, den.use_graph, den.graph_status = None, False, "disabled: replay != eager"
    e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e2.record()
    for _ in range(args.steps):
        res_h = den.step(lat_h, txt_h, 500)
    e3.record()
    sync_all()
    clocks = sampler.stop() if rank == 0 else None
    # ---- sequence-parallel parity, driver-visible: the N-rank output against the single-rank engine on rank 0 (every rank
    # holds all weights), bit for bit, on this very workload
    sp_check = None
    if world > 1:
        import hashlib
        out_sp = den.forward_device(lat_d, txt_d, t_d)
        sync_all()
        if rank == 0:
            out_1 = model.forward(lat_d, txt_d, t_d, vsa_sparsity=sparsity)
            torch.cuda.synchronize()
            sha = lambda t: hashlib.sha256(t.contiguous().view(torch.int16).cpu().numpy().tobytes()).hexdigest()[:16]
            sp_check = {"sp_bit_equal": bool(torch.equal(out_sp, out_1)), "sha_sp": sha(out_sp), "sha_single_rank": sha(out_1),
                        "max_abs_diff": float((out_sp.float() - out_1.float()).abs().max()),
                        "comm": den.sp.comm if den.sp is not None else None}
            del out_1
        sync_all()
    ms_e2e = torch.tensor([e2.elapsed_time(e3)], device=device)
    if world > 1:
        dist.all_reduce(ms_e2e, op=dist.ReduceOp.MAX)
    ms_e2e_step = ms_e2e.item() / args.steps
    finite = bool(torch.isfinite(res_h.float()).all())

    if rank != 0:
        return
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"noise_pred": out})
    peaks = measured_peaks()
    peak_tf = (peaks or {}).get("bf16_tflops_sustained", 1400.0)
    peak_src = "MEASURED_PEAKS.json bf16_tflops_sustained (kernel timed inside a long step)" if peaks else "fallback 1.4 PFLOP/s sustained (B200_PROFILING.md)"
    g_ms, g_flop, g_n = gemm_t.result()
    a_ms, a_flop, a_n = attn_t.result()
    d_ms, d_flop, d_n = attn_d.result()
    step_ms_total = ms_step * args.steps
    traffic = load_traffic()

    def fam(name, kernel, ms, flop, n, flop_model):
        ach = flop / ms / 1e9 if ms else None
        t = traffic.get(name, {})
        return {"name": name, "kernel": kernel, "bound": "tensor", "achieved": ach, "peak": peak_tf, "unit": "TFLOP/s",
                "frac": ach / peak_tf if ach else None, "launches_timed": n, "share_of_step": ms / step_ms_total if ms else None,
                "flop_model": flop_model, "traffic": t.get("dram_bytes_per_launch"),
                "algorithmic_bytes": t.get("algorithmic_bytes_per_launch"), "traffic_source": t.get("source")}

    kernels = [fam("gemm", "fvb::gemm_bf16_kernel (every linear of the step)", g_ms, g_flop, g_n, "2*M*N*K"),
               fam("attention_sparse", "fvb::attn_ws_r1_kernel (VSA sparse branch, per-q-block lists; fvb::attn_ws_kernel under FVB_ATTN_IMPL=r2)", a_ms, a_flop, a_n,
                   "4*B*H*S_q*topk*64*d (reference bench_vsa.py:84-86)"),
               fam("attention_dense", "fvb::attn_fwd_kernel (cross attention; self attention of dense workloads)", d_ms, d_flop, d_n,
                   "4*B*H*S_q*S_kv*d")]
    kernels = [k for k in kernels if k["launches_timed"]]
    if kernels and kernels[0]["name"] == "gemm":
        kernels[0]["shapes"] = gemm_t.by_tag()[:8]
    r_ms, r_bytes, r_n = rows_t.result()
    hbm_peak = (peaks or {}).get("hbm_gbs")
    r_gbs = r_bytes / r_ms / 1e6 if r_ms else None
    kernels.append({"name": "rows_and_index",
                    "kernel": "LayerNorm / RMSNorm+RoPE / block means / coarse softmax / top-k + list / gate combine kernels",
                    "bound": "hbm", "share_of_step": r_ms / step_ms_total if r_ms else None, "achieved": r_gbs, "peak": hbm_peak,
                    "unit": "GB/s", "frac": (r_gbs / hbm_peak) if (r_gbs and hbm_peak) else None, "launches_timed": r_n,
                    "bytes_model": "algorithmic: each operand row read once, each result row written once"})
    rest_ms = step_ms_total - sum((k["share_of_step"] or 0) * step_ms_total for k in kernels)
    kernels.append({"name": "other", "kernel": "embedders, head, torch glue between the timed families", "bound": "hbm",
                    "share_of_step": rest_ms / step_ms_total, "achieved": None, "peak": hbm_peak, "unit": "GB/s", "frac": None})
    dom = max((k for k in kernels if k.get("achieved")), key=lambda k: k["share_of_step"] or 0.0, default=None)
    # contract object = the dominant family (largest share of the step); every family sits in roofline.kernels
    roof = {"bound": "tensor", "kernel": dom["kernel"] if dom else None, "achieved": dom["achieved"] if dom else None,
            "peak": peak_tf, "peak_source": peak_src, "unit": "TFLOP/s", "frac": dom["frac"] if dom else None,
            "traffic": dom.get("traffic") if dom else None, "algorithmic_bytes": dom.get("algorithmic_bytes") if dom else None,
            "launches_timed": dom["launches_timed"] if dom else 0, "share_of_step": dom["share_of_step"] if dom else None,
            "kernels": kernels}
    roof_attn = next((k for k in kernels if k["name"] == "attention_sparse"), None) or next(
        (k for k in kernels if k["name"] == "attention_dense"), None)
    line = {"metric": METRIC, "value": S_tokens / (ms_step / 1e3), "unit": "tokens/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "bf16", "data": "synthetic",
            "config": {"workload": args.workload, "model": "Wan2.2-T2V-A14B expert (random init)" if arch["hidden_size"] == 5120 else "Wan2.1-T2V-1.3B (random init)",
                       "layers": arch["num_layers"], "tokens": S_tokens, "latent": list(latent), "text_len": text_len,
                       "vsa_sparsity": sparsity, "global_batch": 1, "parallelism": f"sp{world}",
                       "l2_policy": "inputs exceed L2: one step streams ~30 GB of weights and >10 GB of activations",
                       "full_model": not bool(args.layers)},
            "e2e": {"value": S_tokens / (ms_e2e_step / 1e3), "unit": "tokens/s", "ms_per_step": ms_e2e_step,
                    "h2d_bytes_per_step": den.h2d_bytes_per_step, "d2h_bytes_per_step": den.d2h_bytes_per_step,
                    "api": "fastvideo_b200.api.WanDenoiser.step (pinned host tensors in / out)", "output_finite": finite,
                    "cuda_graph": den.graph_status, "graph_equals_eager": graph_check},
            "gpu_launches": launches, "roofline": roof, "roofline_attention": roof_attn, "clocks": clocks}
    if sp_check is not None:
        line["sp_parity"] = sp_check
        line["config"]["sp_bit_equal"] = sp_check["sp_bit_equal"]
    if world == 1 and not args.no_cpu_baseline:
        # bounded CPU leg in its own process (CUDA hidden, so the reference resolves its CPU platform; own gloo group):
        # one pass over S in {1024, 4096}; the 9450-token point belongs to the `--impl reference` arm
        try:
            r = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", "1", "--warmup", "1",
                                "--cpu-sizes", "1024,4096", "--workload", args.workload],
                               env={**os.environ, "CUDA_VISIBLE_DEVICES": ""}, capture_output=True, text=True, timeout=600)
            ref_line = json.loads(r.stdout.strip().splitlines()[-1])
            line["cpu_baseline"] = ref_line["cpu_baseline"]
        except Exception as e:  # noqa: BLE001
            line["cpu_baseline"] = {"value": None, "unit": "tokens/s", "cores": os.cpu_count(), "kind": "port",
                                    "sample": f"CPU leg failed: {type(e).__name__}: {e}"}
    emit(line)


_REAL_STDOUT = None


def _claim_stdout():
    """The contract is ONE JSON line on stdout. Libraries write there too (NCCL prints its version banner on stdout at
    communicator creation), so file descriptor 1 is pointed at stderr for the whole run and the JSON line is written to
    the saved descriptor."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(line: dict) -> None:
    out = _REAL_STDOUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def dump_outputs(directory: str, arrays: dict) -> None:
    """Writes each tensor as `directory/<name>.npy` in float32, whole: the seeded inputs make two builds of the project
    comparable output for output (the 14B workload's prediction is 4.8 M values, 19 MB)."""
    import numpy as np
    os.makedirs(directory, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(directory, name + ".npy"), t.detach().float().cpu().numpy())


def main():
    _claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD, choices=sorted(WORKLOADS))
    ap.add_argument("--layers", type=int, default=0, help="development only: truncate the model (result is flagged)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-sizes", default="", help="CPU arm: comma-separated token counts of the block samples")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="GPU arm: write the noise prediction of the last timed step to DIR/noise_pred.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs the GPU arm (--impl ours)")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        os.environ.setdefault("CUDA_VISIBLE_DEVICES", "")  # the CPU arm never touches a GPU (before torch is imported)
        run_reference_arm(args, rank, world)
        return
    from fastvideo_b200 import distributed as fdist
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the GPU arm has no CPU fallback; use --impl reference for the CPU arm)")
    rank, world, device = fdist.init_from_env()
    if world != args.gpus and rank == 0:
        print(f"[bench] WORLD_SIZE={world} but --gpus {args.gpus}; using WORLD_SIZE", file=sys.stderr)
    run_gpu_arm(args, rank, world, device)
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()

#!/usr/bin/env python
"""Headline benchmark: tokens/sec of one Long-VITA prefill forward (ViT tower + projector + 48-layer
14B decoder + masked LM head) on synthetic frames, through the HF `forward()` surface.

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--frames F] [--dump-outputs DIR]

A "step" is one full prefill of the configured prompt.  N = 1: BASELINE.json configs[1]
("Long-VITA-16K bf16 single B200, 64 synthetic frames -> 16K tokens").  Launched under torchrun
for N > 1 (one rank per GPU); see DESIGN.md for what each N runs.  Rank 0 prints ONE JSON line.

`--impl reference` times the reference's own CPU implementation of the path - the oracle port
of the HF forward (oracle/model.py; the reference itself cannot be imported here, SURVEY.md 8c) -
on the host cores with all threads, on a bounded sample of the same workload.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "prefill_tokens_per_sec"
UNIT = "tokens/s"


T0 = time.time()


def log(msg: str) -> None:
    sys.stderr.write(f"[bench +{time.time() - T0:7.1f}s] {msg}\n")
    sys.stderr.flush()


def host_threads() -> int:
    """Threads the CPU legs may use: the cores this process is allowed on (cgroup / affinity aware)."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    return max(1, min(n, 64))


def peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))), "measured"
    except Exception:  # noqa: BLE001
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


# ------------------------------------------------------------------------------------------------
# clocks sampler (nvidia-smi during the timed region)
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.rows = []
        self.proc = None
        self.gpu = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200", "-i",
                 str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# CPU baseline (oracle port of the reference HF forward), bounded sample
# ------------------------------------------------------------------------------------------------
_REF_CACHE = {}    # synthetic fp32 weights / inputs of the CPU sample (generated once, outside the timed parts)


def cpu_reference_sample(cfg, total_tokens: int, n_frames: int, threads: int, reduced: bool = False):
    """Time the oracle port of the reference's HF forward on a bounded sample of ONE prefill of `total_tokens`.

    FULL sample (nothing is extrapolated in S):
      * one of the L identical decoder layers on all `total_tokens` tokens: the whole token-wise part (RMSNorm, QKV,
        RoPE, O-proj, SwiGLU MLP) plus the eager causal attention (full S x S scores, then the mask - what the
        reference's HF path computes on a CPU, where flash-attn cannot run) of ONE of the hkv identical kv groups
        (hq / hkv query heads), timed apart inside the same layer call;
      * one of the F identical frames through the whole ViT tower (all layers) + projector.
    REDUCED sample (`reduced=True`, ~3x cheaper; used for the later steps of a many-step run so that it ends within
    minutes): the same layer on the first S/4 query rows only - token-wise operators are row-independent and the eager
    attention computes a full-width (all S keys) score row for every query row, so both parts scale x4 exactly.
    The ViT frame is the same.
    Scaled only by counts of identical units: t_prefill = L * (t_tokenwise + n_heads_or_groups * t_attn) + F * t_frame.
    Returns (tokens_per_sec, seconds_measured, description)."""
    import torch

    from long_vita_b200.weights import global_weights, llm_layer_weights, vit_layer_weights
    from oracle import model as OM
    from oracle import ops as O

    torch.set_num_threads(threads)
    S = total_tokens
    hq, hkv, d = cfg.num_attention_heads, cfg.num_key_value_heads, cfg.head_dim
    grp = hq // hkv
    v = cfg.visual
    if "w" not in _REF_CACHE:
        g = torch.Generator().manual_seed(1)
        _REF_CACHE["w"] = llm_layer_weights(cfg, 0, 1234, "cpu", torch.float32)
        _REF_CACHE["x"] = torch.randn(S, cfg.hidden_size, generator=g)
        wv = global_weights(cfg, 1234, "cpu", torch.float32, with_lm=False)
        for i in range(v.num_hidden_layers):
            wv.update(vit_layer_weights(cfg, i, 1234, "cpu", torch.float32))
        _REF_CACHE["wv"] = wv
        _REF_CACHE["img"] = torch.randn(1, 3, v.image_size, v.image_size, generator=g)
        _REF_CACHE["qkv1"] = [torch.randn(1, S, hkv, d, generator=g) for _ in range(3)]
    w, x, wv, img = (_REF_CACHE[k_] for k_ in ("w", "x", "wv", "img"))
    rows = S // 4 if reduced else S
    pos = torch.arange(rows)
    cos, sin = O.rope_tables(pos, O.rope_inv_freq(cfg.head_dim, cfg.rope_theta), torch.float32)
    t_group = [0.0]

    def attention_hook(q, k, v_, **kw):
        if reduced:      # keys / values of the full sequence (the layer call above only produced S/4 rows of them)
            k, v_ = _REF_CACHE["qkv1"][1], _REF_CACHE["qkv1"][2]
        t0 = time.perf_counter()
        O.attention(q[:, :, :grp], k[:, :, :1], v_[:, :, :1], causal=True, head_chunk=grp, q_chunk=2048,
                    q_pos=torch.arange(q.shape[1]))
        t_group[0] = time.perf_counter() - t0
        return torch.zeros(q.shape, dtype=torch.float32), None      # values are not used by a timing run

    t0 = time.perf_counter()
    with torch.no_grad():
        OM.decoder_layer(cfg, w, 0, x[:rows], cos, sin, attention_fn=attention_hook)
    t_layer = time.perf_counter() - t0
    t_attn = t_group[0]
    t_tok, attn_units, row_scale = max(t_layer - t_attn, 1e-6), hkv, S / rows
    measured_layer = t_layer
    # vision: one frame through the whole tower + projector
    t0 = time.perf_counter()
    with torch.no_grad():
        vit = OM.vit_forward(cfg, wv, img)
        OM.projector_forward(cfg, wv, vit[:, 1:, :])
    t_frame = time.perf_counter() - t0
    measured = measured_layer + t_frame
    L = cfg.num_hidden_layers
    t_full = L * row_scale * (t_tok + attn_units * t_attn) + n_frames * t_frame
    what = (f"the first {rows} of {S} query rows: token-wise part {t_tok:.2f} s + eager causal attention of 1 of {hkv} kv "
            f"groups against all {S} keys {t_attn:.2f} s; rows are independent, x{row_scale:.0f}" if reduced else
            f"token-wise part on all {S} rows {t_tok:.2f} s + eager causal attention of 1 of {hkv} kv groups over the full "
            f"S x S {t_attn:.2f} s")
    desc = (f"oracle port of the reference HF forward (fp32, {threads} threads), S = {S}: 1 of {L} decoder layers ({what}) "
            f"and 1 of {n_frames} frames through all {v.num_hidden_layers} ViT layers + projector ({t_frame:.2f} s); scaled by "
            f"counts of identical units only (x{L} layers, x{attn_units} kv groups, x{n_frames} frames)")
    return total_tokens / t_full, measured, desc


# ------------------------------------------------------------------------------------------------
# probes that ride along with the bench line
# ------------------------------------------------------------------------------------------------
def attn_128k_probe(ops, dev, pk, launches: int = 3):
    """Standalone `lv_attn_fwd` at the length the north-star target is quoted on (S = 131 072, 40:8 heads x 128,
    causal): one warm-up + `launches` timed launches with CUDA events.  FLOPs are the algorithmic causal count
    4 * Hq * d * S (S + 1) / 2 (SURVEY.md 8d).  The kernel is timed alone, so `frac` is against the measured BURST
    cuBLAS bf16 peak; `frac_sustained` is against the sustained figure (the three launches keep the GPU busy ~0.5 s)."""
    import torch

    S, hq, hkv, d = 131072, 40, 8, 128
    g = torch.Generator(device=dev).manual_seed(128)
    q = torch.randn((1, S, hq, d), generator=g, device=dev, dtype=torch.bfloat16)
    k = torch.randn((1, S, hkv, d), generator=g, device=dev, dtype=torch.bfloat16)
    v = torch.randn((1, S, hkv, d), generator=g, device=dev, dtype=torch.bfloat16)
    out = torch.empty_like(q)
    ops.attention_fwd(q, k, v, causal=True, out=out)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(launches):
        ops.attention_fwd(q, k, v, causal=True, out=out)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / launches
    flops = 4.0 * hq * d * (S * (S + 1) / 2)
    ach = flops / (ms / 1000.0) / 1e12
    burst, sust = pk["bf16_tflops"], pk.get("bf16_tflops_sustained", pk["bf16_tflops"])
    return {"bound": "tensor", "kernel": "attn_fwd (standalone, S=131072, 40:8x128 causal)", "achieved": ach, "peak": burst,
            "unit": "TFLOP/s", "frac": ach / burst, "frac_sustained": ach / sust, "frac_of_2250_datasheet": ach / 2250.0,
            "launches": launches, "avg_launch_ms": ms, "flops_per_launch": flops,
            "inputs": "2.7 GB Q+O, 0.5 GB K+V per launch (far beyond the 126 MB L2)"}


def cp_parity_probe(model, runner, S, dev, n_rows: int = 64):
    """Context-parallel parity inside the bench run (N > 1): the fused exchange kernel `lv_attn_cp_fwd` on this rank's
    zig-zag rows of a random [S] problem, for both buffer parities of the exchange protocol, against
      (a) the single-device kernel on the all-gathered K/V with the rank's query segments at their global positions
          (`q_seg_len` / `q_seg_pos`; that path is oracle-validated by the 1-GPU tests at 16K / 128K,
          tests/test_gpu_attention_long.py) - bit-identical in the default (global) key order;
      (b) an fp32 evaluation of `n_rows` sampled query rows per rank (torch matmul / softmax in fp32 on the device - the
          attention definition of oracle.ops.attention) - the error beyond the bf16 output-rounding floor, the quantity
          the parity tests bound by 2e-3.
    Returns (excess over the bf16 floor vs fp32, max |lse - lse_fp32|, rel. difference to the single-device kernel,
    bit-identical?), each the worst over the ranks.  Layout: training/utils.py:329-341."""
    import math

    import torch
    import torch.distributed as dist

    from long_vita_b200 import ops
    from long_vita_b200.cp import zigzag_index

    cfg = model.config
    ctx = runner._context(S, dev)
    hq, hkv, d = cfg.num_attention_heads, cfg.num_key_value_heads, cfg.head_dim
    T, c = ctx.T, S // (2 * ctx.cp)
    g = torch.Generator(device=dev).manual_seed(4321 + ctx.rank)
    gs = torch.Generator().manual_seed(99 + ctx.rank)
    pos_all = zigzag_index(S, ctx.cp, ctx.rank, dev)
    worst = torch.zeros(3, device=dev)
    identical = True
    for _ in range(2):                        # both buffer parities of the exchange protocol
        buf = ctx.qkv_buffer()                # [T, (hq + 2 hkv) d]: the fused QKV GEMM's output lives here in the model
        buf.copy_(torch.randn(buf.shape, generator=g, device=dev, dtype=torch.float32).to(torch.bfloat16))
        q = buf[:, : hq * d].view(T, hq, d)
        k = buf[:, hq * d : (hq + hkv) * d].view(T, hkv, d)
        v = buf[:, (hq + hkv) * d :].view(T, hkv, d)
        K, V = ctx.gather_kv(k, v)            # NCCL all-gather + bit-exact re-order to global positions
        lse_cp = torch.empty((1, hq, T), dtype=torch.float32, device=dev)
        out_cp = ctx.attention(lse=lse_cp).view(T, hq, d)
        out_sd, lse_sd = ops.attention_fwd(q.unsqueeze(0), K.unsqueeze(0), V.unsqueeze(0), causal=True, return_lse=True,
                                           q_seg_len=c, q_seg_pos=(ctx.rank * c, (2 * ctx.cp - 1 - ctx.rank) * c))
        out_sd = out_sd.view(T, hq, d)
        identical = identical and bool(torch.equal(out_cp, out_sd)) and bool(torch.equal(lse_cp, lse_sd))
        rel_sd = (out_cp.float() - out_sd.float()).norm() / out_sd.float().norm()
        # (b) fp32 reference on sampled rows: first / last rows of both segments + random rows
        rows = torch.unique(torch.cat([torch.tensor([0, c - 1, c, T - 1]), torch.randint(0, T, (n_rows - 4,), generator=gs)])).to(dev)
        qs = q[rows].float()                                            # [r, hq, d]
        qpos = pos_all[rows]                                            # global positions
        kpos = torch.arange(S, device=dev)
        ref = torch.empty((rows.numel(), hq, d), dtype=torch.float32, device=dev)
        lse_ref = torch.empty((hq, rows.numel()), dtype=torch.float32, device=dev)
        grp = hq // hkv
        for kh in range(hkv):                                           # one kv group at a time bounds the score matrix
            sc = torch.einsum("rgd,sd->grs", qs[:, kh * grp : (kh + 1) * grp], K[:, kh].float()) / math.sqrt(d)
            sc = sc.masked_fill(kpos[None, None, :] > qpos[None, :, None], float("-inf"))
            lse_ref[kh * grp : (kh + 1) * grp] = torch.logsumexp(sc, dim=-1)
            ref[:, kh * grp : (kh + 1) * grp] = torch.einsum("grs,sd->rgd", torch.softmax(sc, dim=-1), V[:, kh].float())
        got = out_cp[rows].float()
        e_total = (got - ref).norm() / ref.norm()
        e_floor = (ref.to(torch.bfloat16).float() - ref).norm() / ref.norm()
        excess = torch.sqrt(torch.clamp(e_total * e_total - e_floor * e_floor, min=0.0))
        e_lse = (lse_cp[0][:, rows] - lse_ref).abs().max()
        worst = torch.maximum(worst, torch.stack([excess, e_lse, rel_sd]))
    flag = torch.tensor([1.0 if identical else 0.0], device=dev)
    dist.all_reduce(worst, op=dist.ReduceOp.MAX)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    return float(worst[0]), float(worst[1]), float(worst[2]), bool(flag.item() > 0.5)


def ncu_traffic(kind: str):
    """DRAM bytes per launch of the dominant kernel from the committed `ncu --set full` capture of this same command
    (profiles/ncu_traffic.json, written by tools/ncu_summary.py; dram__bytes_read.sum + dram__bytes_write.sum averaged
    over the captured launches).  None when no capture is committed for that kernel."""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
        e = t.get(kind)
        return (e["dram_bytes_per_launch"], e["source"]) if e else (None, None)
    except Exception:  # noqa: BLE001
        return None, None


# ------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--frames", type=int, default=64, help="synthetic frames (64 -> 16K, 512 -> 128K, 4096 -> 1M)")
    ap.add_argument("--text", type=int, default=16)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-cp-parity", action="store_true", help="N > 1: skip the in-run check of the fused exchange kernel")
    ap.add_argument("--no-attn-probe", action="store_true", help="N = 1: skip the standalone 128K attention roofline probe")
    ap.add_argument("--long-run", action="store_true",
                    help="minutes-per-step configs (1M tokens): honour --warmup < 3 and skip the separate e2e pass; "
                         "the printed line is then marked as outside the timing contract")
    ap.add_argument("--layers", type=int, default=None, help="debug: fewer decoder layers (number is then INVALID)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned (the last-position logits) to DIR/logits.npy, float32")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs needs --impl b200 (the reference arm times a sample and computes no outputs)")
    # stdout carries exactly ONE JSON line: everything libraries print meanwhile (e.g. NCCL's
    # "NCCL version ..." banner, written to fd 1 from C) is routed to stderr until the line is emitted
    sys.stdout.flush()
    _stdout_fd = os.dup(1)
    os.dup2(2, 1)

    def emit(line):
        sys.stdout.flush()
        os.dup2(_stdout_fd, 1)
        print(json.dumps(line), flush=True)
        os.dup2(2, 1)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    from long_vita_b200.config import LongVITAConfig
    from long_vita_b200.synthetic import build_prompt

    cfg = LongVITAConfig.long_vita_14b()
    cp = max(world, 1)
    # the SAME prompt at every N: length padded (with text tokens) to a multiple of 2*8*128 so that it
    # shards zig-zag over 1, 2, 4 or 8 ranks in 128-token units
    ids, image_indices = build_prompt(cfg, args.frames, args.text, pad_multiple=2048)
    S = ids.shape[1]
    workload = (f"Long-VITA-{'16K' if args.frames == 64 else str(S)} prefill, {args.frames} synthetic frames "
                f"({args.frames * 256} visual + {2 * args.frames} delimiter tokens) + text, padded to {S} tokens")
    config = {"workload": workload, "frames": args.frames, "tokens": S, "layers": cfg.num_hidden_layers,
              "parallelism": f"cp{cp}" if cp > 1 else "single",
              "l2": "per-step working set (29.5 GB weights + activations) far exceeds the 126 MB L2"}

    if args.impl == "reference":
        if rank != 0:
            return
        threads = host_threads()
        # Step 0 (a warm-up step when W >= 1) always times the FULL sample: a whole decoder layer at the full S.  When
        # that took longer than this run's per-step budget (the whole run should end within a few minutes), the later
        # steps time the REDUCED sample (see cpu_reference_sample); the line reports both so they can be compared.
        budget_s = float(os.environ.get("LV_REF_BUDGET_S", "240")) / max(1, args.warmup + args.steps)
        vals, meas, full, reduced = [], [], None, False
        for i in range(args.warmup + args.steps):
            v, m, desc = cpu_reference_sample(cfg, S, args.frames, threads, reduced=reduced)
            log(f"reference sample {i} ({'reduced' if reduced else 'full'}): {m:.1f} s measured -> {v:.3f} tokens/s for the whole prefill")
            if i == 0:
                full = {"value": v, "seconds_measured": m, "sample": desc}
                reduced = m > budget_s
            if i >= args.warmup:
                vals.append(v)
                meas.append(m)
        value = sum(vals) / len(vals)
        # ms_per_step = what one timed step of THIS arm really took (the bounded sample), so that steps x ms_per_step
        # is the arm's measured time; the whole-prefill time the value corresponds to is ms_per_prefill_scaled.
        line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000.0 * sum(meas) / len(meas),
                "ms_per_prefill_scaled": 1000.0 * S / value,
                "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
                "data": "synthetic", "config": config,
                "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": desc,
                                 "seconds_measured_per_step": sum(meas) / len(meas),
                                 "full_layer_sample_step0": full},
                "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        emit(line)
        return

    import torch
    import torch.distributed as dist

    from long_vita_b200 import ops
    from long_vita_b200.hf.modeling import LongVITAForCausalLM
    from long_vita_b200.synthetic import synthetic_frames

    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback for the product path)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    log("materialising random-init weights on the GPU")
    model = LongVITAForCausalLM.from_synthetic(cfg, seed=1234, device=dev, num_layers=args.layers)
    log("weights ready")
    if world > 1:
        from long_vita_b200 import cp as cpmod

        runner = cpmod.ContextParallelRunner(model, dist.group.WORLD)
        runner.check_faults = False     # the per-forward fault check synchronises the stream; checked once after the timed region
    else:
        runner = None

    # host-side inputs in pinned memory (the e2e region copies them every step)
    # --long-run (no e2e pass): frames are drawn on the device, no pinned host copy of ~5 GB per rank
    images_h = None if args.long_run else synthetic_frames(cfg, args.frames, pin=True)
    ids_h = ids.pin_memory()
    idx_h = image_indices.pin_memory()
    h2d = (0 if images_h is None else images_h.numel() * 2) + ids_h.numel() * 8 + idx_h.numel() * 8
    logits_h = torch.empty((1, 1, cfg.vocab_size), dtype=torch.bfloat16).pin_memory()
    d2h = logits_h.numel() * 2

    def forward_resident(images_d, ids_d, idx_d):
        if runner is not None:
            return runner.forward(ids_d, images_d, idx_d)
        return model(input_ids=ids_d, images=images_d, image_indices=idx_d, num_logits_to_keep=1).logits

    def step_e2e():
        images_d = images_h.to(dev, non_blocking=True)
        ids_d = ids_h.to(dev, non_blocking=True)
        idx_d = idx_h.to(dev, non_blocking=True)
        logits = forward_resident(images_d, ids_d, idx_d)
        logits_h.copy_(logits.view(1, 1, -1), non_blocking=True)

    images_d = synthetic_frames(cfg, args.frames, device=dev) if images_h is None else images_h.to(dev)
    ids_d = ids_h.to(dev)
    idx_d = idx_h.to(dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    n_warm = args.warmup if args.long_run else max(args.warmup, 3)
    for i in range(n_warm):
        forward_resident(images_d, ids_d, idx_d)
        torch.cuda.synchronize()
        log(f"warm-up step {i} done")
    barrier()
    cp_parity = None
    if runner is not None and not args.no_cp_parity:
        cp_parity = cp_parity_probe(model, runner, S, dev)
        log(f"cp parity: excess over the bf16 floor vs fp32 {cp_parity[0]:.3e}, lse {cp_parity[1]:.3e} abs; vs the single-device "
            f"kernel {cp_parity[2]:.3e} rel ({'bit-identical' if cp_parity[3] else 'not bit-identical'})")
        barrier()

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    timer = ops.KernelTimer()
    ops.set_kernel_timer(timer)
    n0 = ops.launch_count()
    last = {}

    def step_resident():
        last["logits"] = forward_resident(images_d, ids_d, idx_d)

    ms_resident = timed(step_resident, args.steps)
    log(f"timed region done: {ms_resident / args.steps:.1f} ms/step")
    launches = ops.launch_count() - n0
    ops.set_kernel_timer(None)
    torch.cuda.synchronize()
    ksum = timer.summary()
    if args.dump_outputs and rank == 0:
        # copied now: later forwards (the e2e pass) may reuse the buffer the logits live in
        os.makedirs(args.dump_outputs, exist_ok=True)
        import numpy as np

        logits = last["logits"].float().cpu().numpy()
        np.save(os.path.join(args.dump_outputs, "logits.npy"), logits)
        log(f"wrote {args.dump_outputs}/logits.npy {logits.shape} float32")
    del last
    # e2e: host buffers, H2D + forward + D2H inside the timed region
    if args.long_run:
        ms_e2e = None
    else:
        step_e2e()
        ms_e2e = timed(step_e2e, args.steps)
    clocks = sampler.stop() if rank == 0 else None
    if runner is not None and runner.ctx is not None:
        runner.ctx.check()      # raises if any in-kernel wait on a peer GPU timed out during the run

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    pk, pk_kind = peaks()
    ms_step = ms_resident / args.steps
    value = S / (ms_step / 1000.0)
    e2e_value = S / (ms_e2e / args.steps / 1000.0) if ms_e2e is not None else None

    def roof(kind):
        d = ksum.get(kind)
        if not d or d["ms"] <= 0:
            return None
        ach = d["flops"] / (d["ms"] / 1000.0) / 1e12
        peak = pk.get("bf16_tflops_sustained", pk["bf16_tflops"])
        return {"bound": "tensor", "kernel": kind, "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak,
                "peak_source": f"{pk_kind} sustained cuBLAS bf16 (kernel timed inside a long step)",
                "launches_per_step": d["launches"] / args.steps, "avg_launch_ms": d["ms"] / d["launches"],
                "share_of_step": d["ms"] / ms_resident, "traffic": ncu_traffic(kind)[0], "traffic_source": ncu_traffic(kind)[1],
                "algorithmic_bytes_or_flops_per_launch": d["flops"] / d["launches"]}

    dominant = max(ksum, key=lambda k_: ksum[k_]["ms"]) if ksum else None
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": n_warm,
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "bf16",
        "data": "synthetic", "config": config, "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
        "gpu_launches": launches,
        "roofline": roof(dominant) if dominant else None,
        "roofline_attn": roof("attn_fwd"),
    }
    if cp_parity is not None:
        # fused in-kernel K/V exchange: error beyond the bf16 output-rounding floor against an fp32 evaluation of sampled
        # rows (the quantity the parity tests bound), worst rank; the run FAILS above 2e-3 (lse above 1e-4)
        line["cp_parity_excess"] = cp_parity[0]
        line["cp_parity"] = {"excess_over_bf16_floor_vs_fp32": cp_parity[0], "lse_max_abs_vs_fp32": cp_parity[1],
                             "rel_fro_vs_single_device_kernel": cp_parity[2], "bit_identical_to_single_device_kernel": cp_parity[3],
                             "sampled_rows_per_rank": 64, "tokens": S, "ranks": world, "bound": 2e-3}
        if not (cp_parity[0] < 2e-3 and cp_parity[1] < 1e-4):
            line["INVALID"] = f"context-parallel parity failed: {cp_parity}"
    if world == 1 and not args.no_attn_probe:
        line["roofline_attn_128k"] = attn_128k_probe(ops, dev, pk)
        log(f"attention @128K standalone: {line['roofline_attn_128k']['achieved']:.0f} TFLOP/s")
    if args.long_run:
        line["note"] = "--long-run: fewer than 3 warm-up steps and no separate e2e pass (minutes per step)"
    if args.layers is not None:
        line["INVALID"] = f"debug run with {args.layers} decoder layers"
    if world == 1 and not args.no_cpu_baseline:
        cores = host_threads()
        log(f"cpu baseline on {cores} threads")
        v, m, desc = cpu_reference_sample(cfg, S, args.frames, cores)
        line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": desc,
                                "seconds_measured": m}
    emit(line)
    if world > 1:
        dist.destroy_process_group()
    if "INVALID" in line and cp_parity is not None and "parity" in line["INVALID"]:
        sys.exit(3)


if __name__ == "__main__":
    main()

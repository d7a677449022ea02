"""Operator layer: PyTorch tensors in / out, arithmetic in liblvb200.so through the C ABI.

PyTorch is used for device memory, streams and autograd plumbing only.  Every function validates
that its tensors are CUDA bf16 (or the stated integer / float type) and raises RuntimeError when
the extension is missing or a call fails - there is no eager fallback.
"""
from __future__ import annotations

import ctypes as C
import math
from typing import Optional, Tuple

import torch

from . import _lib
from ._lib import AttnBwdParams, AttnParams


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _need_cuda_bf16(*ts: Optional[torch.Tensor]) -> None:
    for t in ts:
        if t is None:
            continue
        if not t.is_cuda:
            raise RuntimeError("long_vita_b200 operators run on CUDA tensors only (no CPU fallback)")
        if t.dtype != torch.bfloat16:
            raise RuntimeError(f"expected bfloat16 tensor, got {t.dtype}")


def _need_cuda(t: torch.Tensor, dtype: torch.dtype) -> None:
    if not t.is_cuda or t.dtype != dtype:
        raise RuntimeError(f"expected CUDA {dtype} tensor, got {t.device} {t.dtype}")


class KernelTimer:
    """Optional per-launch device timing of the two tensor-core kernels (CUDA events on the
    launching stream).  bench.py installs one for its roofline numbers; None costs nothing."""

    def __init__(self):
        self.records = []  # (kind, algorithmic flops, start event, end event)

    def start(self):
        ev = torch.cuda.Event(enable_timing=True)
        ev.record()
        return ev

    def stop(self, kind, flops, ev0):
        ev1 = torch.cuda.Event(enable_timing=True)
        ev1.record()
        self.records.append((kind, flops, ev0, ev1))

    def summary(self):
        """kind -> dict(launches, ms, flops); call after a synchronize."""
        out = {}
        for kind, flops, e0, e1 in self.records:
            d = out.setdefault(kind, {"launches": 0, "ms": 0.0, "flops": 0.0})
            d["launches"] += 1
            d["ms"] += e0.elapsed_time(e1)
            d["flops"] += flops
        return out


_TIMER: Optional[KernelTimer] = None


def set_kernel_timer(t: Optional[KernelTimer]) -> None:
    global _TIMER
    _TIMER = t


def launch_count() -> int:
    """Kernels launched by liblvb200.so so far in this process."""
    return int(_lib.lib().lv_launch_count())


# ------------------------------------------------------------------------------------------------
# attention
# ------------------------------------------------------------------------------------------------
def attention_fwd(
    q: torch.Tensor,
    k: torch.Tensor,
    v: torch.Tensor,
    *,
    causal: bool,
    scale: Optional[float] = None,
    layout: str = "bshd",
    return_lse: bool = False,
    q_seg_len: Optional[int] = None,
    q_seg_pos: Optional[Tuple[int, int]] = None,
    kv_pos0: int = 0,
    out: Optional[torch.Tensor] = None,
):
    """softmax(scale * q k^T + mask) v.  `layout` names the dimension order of q/k/v and of the
    returned tensor: "bshd" (flash-attn / HF), "sbhd" (Megatron, dot_product_attention.py:344) or
    "bhsd" (HF AttentionInterface).  Strided views are consumed in place (no .contiguous()) as
    long as the head dimension is contiguous and the other strides are multiples of 8 elements.
    Returns out (same layout as q) or (out, lse[b, hq, sq] float32)."""
    _need_cuda_bf16(q, k, v)
    perm = {"bshd": (0, 1, 2, 3), "sbhd": (1, 0, 2, 3), "bhsd": (0, 2, 1, 3)}[layout]
    qv, kv_, vv = (t.permute(perm) for t in (q, k, v))  # views in b, s, h, d order
    b, sq, hq, d = qv.shape
    _, sk, hkv, _ = kv_.shape

    def ok(t):
        return t.stride(3) == 1 and all(s % 8 == 0 for s in t.stride()[:3])

    if not ok(qv):
        qv = qv.contiguous()
    if not ok(kv_):
        kv_ = kv_.contiguous()
    if not ok(vv):
        vv = vv.contiguous()
    if out is None:
        # allocate in the caller's layout so the result is contiguous there
        out = torch.empty(q.shape, dtype=torch.bfloat16, device=q.device)
    ov = out.permute(perm)
    lse = torch.empty((b, hq, sq), dtype=torch.float32, device=q.device) if return_lse else None

    p = AttnParams()
    p.q, p.k, p.v, p.out = qv.data_ptr(), kv_.data_ptr(), vv.data_ptr(), ov.data_ptr()
    p.lse = _ptr(lse)
    p.batch, p.sq, p.sk, p.hq, p.hkv, p.d = b, sq, sk, hq, hkv, d
    for name, t in (("q_strides", qv), ("k_strides", kv_), ("v_strides", vv), ("o_strides", ov)):
        arr = getattr(p, name)
        arr[0], arr[1], arr[2] = t.stride(0), t.stride(1), t.stride(2)
    p.scale = float(scale if scale is not None else 1.0 / math.sqrt(d))
    p.causal = 1 if causal else 0
    p.q_seg_len = int(q_seg_len if q_seg_len is not None else sq)
    if q_seg_pos is None:
        q_seg_pos = (sk - sq, 0)  # bottom-right aligned causal mask (flash-attn >= 2.1)
    p.q_seg_pos[0], p.q_seg_pos[1] = int(q_seg_pos[0]), int(q_seg_pos[1])
    p.kv_pos0 = int(kv_pos0)
    ev0 = _TIMER.start() if _TIMER is not None else None
    _lib.check(_lib.lib().lv_attn_fwd(C.byref(p), _stream()), "lv_attn_fwd")
    if ev0 is not None:
        if causal and q_seg_len is None and sq == sk:
            fl = 4.0 * b * hq * d * (sq * (sq + 1) / 2)
        else:
            fl = 4.0 * b * hq * d * sq * sk  # upper bound for masked / segmented calls
        _TIMER.stop("attn_fwd", fl, ev0)
    return (out, lse) if return_lse else out


def _fill_attn_params(p, qv, kv_, vv, ov, lse, scale, causal, q_seg_len, q_seg_pos, kv_pos0):
    b, sq, hq, d = qv.shape
    _, sk, hkv, _ = kv_.shape
    p.q, p.k, p.v, p.out = qv.data_ptr(), kv_.data_ptr(), vv.data_ptr(), ov.data_ptr()
    p.lse = _ptr(lse)
    p.batch, p.sq, p.sk, p.hq, p.hkv, p.d = b, sq, sk, hq, hkv, d
    for name, t in (("q_strides", qv), ("k_strides", kv_), ("v_strides", vv), ("o_strides", ov)):
        arr = getattr(p, name)
        arr[0], arr[1], arr[2] = t.stride(0), t.stride(1), t.stride(2)
    p.scale = float(scale if scale is not None else 1.0 / math.sqrt(d))
    p.causal = 1 if causal else 0
    p.q_seg_len = int(q_seg_len if q_seg_len is not None else sq)
    if q_seg_pos is None:
        q_seg_pos = (sk - sq, 0)
    p.q_seg_pos[0], p.q_seg_pos[1] = int(q_seg_pos[0]), int(q_seg_pos[1])
    p.kv_pos0 = int(kv_pos0)


def attention_bwd(d_out, q, k, v, out, lse, *, causal: bool, scale: Optional[float] = None, q_seg_len=None,
                  q_seg_pos=None, kv_pos0: int = 0):
    """Gradients of attention_fwd (layout "bshd").  `out` / `lse` are the forward results.
    Returns (dq, dk, dv) with the shapes of q, k, v."""
    _need_cuda_bf16(d_out, q, k, v, out)
    _need_cuda(lse, torch.float32)

    def fix(t):
        return t if (t.stride(3) == 1 and all(s % 8 == 0 for s in t.stride()[:3])) else t.contiguous()

    q, k, v, out, d_out = fix(q), fix(k), fix(v), fix(out), fix(d_out)
    dq, dk, dv = torch.empty_like(q, memory_format=torch.contiguous_format), \
        torch.empty_like(k, memory_format=torch.contiguous_format), torch.empty_like(v, memory_format=torch.contiguous_format)
    b, sq, hq, _ = q.shape
    delta = torch.empty((b, hq, sq), dtype=torch.float32, device=q.device)
    p = AttnBwdParams()
    _fill_attn_params(p.fwd, q, k, v, out, lse.contiguous(), scale, causal, q_seg_len, q_seg_pos, kv_pos0)
    p.d_out, p.dq, p.dk, p.dv, p.delta_ws = d_out.data_ptr(), dq.data_ptr(), dk.data_ptr(), dv.data_ptr(), delta.data_ptr()
    for name, t in (("do_strides", d_out), ("dq_strides", dq), ("dk_strides", dk), ("dv_strides", dv)):
        arr = getattr(p, name)
        arr[0], arr[1], arr[2] = t.stride(0), t.stride(1), t.stride(2)
    _lib.check(_lib.lib().lv_attn_bwd(C.byref(p), _stream()), "lv_attn_bwd")
    return dq, dk, dv


class _AttentionFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, q, k, v, causal, scale):
        out, lse = attention_fwd(q, k, v, causal=causal, scale=scale, return_lse=True)
        ctx.save_for_backward(q, k, v, out, lse)
        ctx.causal, ctx.scale = causal, scale
        return out

    @staticmethod
    def backward(ctx, d_out):
        q, k, v, out, lse = ctx.saved_tensors
        dq, dk, dv = attention_bwd(d_out.contiguous(), q, k, v, out, lse, causal=ctx.causal, scale=ctx.scale)
        return dq, dk, dv, None, None


def attention(q, k, v, *, causal: bool, scale: Optional[float] = None):
    """Differentiable fused attention, "bshd" layout (the autograd twin of flash_attn_func)."""
    return _AttentionFn.apply(q, k, v, causal, scale)


def _sm_count(device) -> int:
    """SMs of `device`; a B200's 148 for tensors that are not on a GPU (the host tests' oracle-backed operators)."""
    return torch.cuda.get_device_properties(device).multi_processor_count if torch.device(device).type == "cuda" else 148


def attention_decode(q: torch.Tensor, k_cache: torch.Tensor, v_cache: torch.Tensor, length: int, *,
                     scale: Optional[float] = None, n_splits: Optional[int] = None, return_lse: bool = False):
    """One new token against a K/V cache (SURVEY.md 8f-2; the reference has no such path - it re-prefills
    every generated token, long_vita_megatron/inference/text_generation/generation.py:127-135).

    q [hq, d]; k_cache / v_cache [>= length, hkv, d] (post-RoPE rows of the previous tokens, the new token's
    row already appended); returns out [hq, d] (and lse [hq] fp32, natural log - what a context-parallel
    combine across cache shards needs).

    HBM-bound (every K/V row is read once), so the job is to put all SMs on the cache: the G = hq / hkv query
    heads of a kv group become G query ROWS of one head (they share K/V), and the key range is cut into
    `n_splits` chunks that run as the batch dimension of the ordinary fused kernel (`lv_attn_fwd`,
    non-causal, with LSE); the partial results are merged by their log-sum-exp weights (flash-decoding).
    A ragged last chunk is a second launch with sk = remainder."""
    _need_cuda_bf16(q, k_cache, v_cache)
    hq, d = q.shape
    hkv = k_cache.shape[1]
    G = hq // hkv
    if length <= 0 or length > k_cache.shape[0]:
        raise ValueError(f"attention_decode: length {length} outside the cache (capacity {k_cache.shape[0]})")
    if n_splits is None:
        n_splits = max(1, _sm_count(q.device) // hkv)
    per = -(-length // n_splits)
    chunk = max(128, (per + 127) // 128 * 128)                             # keys per split, whole 128-key tiles
    n_full, rem = divmod(length, chunk)
    qp = q.view(hkv, G, d).transpose(0, 1)                                 # [G rows, hkv heads, d]
    outs, lses = [], []
    if n_full:
        qb = qp.unsqueeze(0).expand(n_full, G, hkv, d).contiguous()
        kb = k_cache[: n_full * chunk].view(n_full, chunk, hkv, d)
        vb = v_cache[: n_full * chunk].view(n_full, chunk, hkv, d)
        o, l = attention_fwd(qb, kb, vb, causal=False, scale=scale, return_lse=True)   # [n, G, hkv, d], [n, hkv, G]
        outs.append(o)
        lses.append(l)
    if rem:
        o, l = attention_fwd(qp.unsqueeze(0).contiguous(), k_cache[n_full * chunk : length].unsqueeze(0),
                             v_cache[n_full * chunk : length].unsqueeze(0), causal=False, scale=scale, return_lse=True)
        outs.append(o)
        lses.append(l)
    o = outs[0] if len(outs) == 1 else torch.cat(outs, dim=0)              # [n, G, hkv, d]
    l = lses[0] if len(lses) == 1 else torch.cat(lses, dim=0)              # [n, hkv, G]
    return decode_merge(o, l, return_lse=return_lse)


def decode_merge(o_part: torch.Tensor, lse_part: torch.Tensor, return_lse: bool = False):
    """o_part [n, G, hkv, d] bf16, lse_part [n, hkv, G] fp32 -> out [hq, d] (head h = kvh * G + g) and the
    merged log-sum-exp [hq]: out = sum_s exp(lse_s - LSE) o_s (lv_attn_decode_merge)."""
    _need_cuda_bf16(o_part)
    _need_cuda(lse_part, torch.float32)
    n, G, hkv, d = o_part.shape
    o_part, lse_part = o_part.contiguous(), lse_part.contiguous()
    out = torch.empty((hkv * G, d), dtype=torch.bfloat16, device=o_part.device)
    lse = torch.empty((hkv * G,), dtype=torch.float32, device=o_part.device) if return_lse else None
    _lib.check(_lib.lib().lv_attn_decode_merge(o_part.data_ptr(), lse_part.data_ptr(), out.data_ptr(), _ptr(lse), n, G, hkv, d,
                                               _stream()), "lv_attn_decode_merge")
    return (out, lse) if return_lse else out


# ------------------------------------------------------------------------------------------------
# token-wise operators
# ------------------------------------------------------------------------------------------------
def rmsnorm(x: torch.Tensor, weight: torch.Tensor, eps: float = 1e-6, residual: Optional[torch.Tensor] = None):
    """RMSNorm over the last dim.  With `residual`, returns (norm(x + residual), x + residual)."""
    _need_cuda_bf16(x, weight, residual)
    x2 = x.reshape(-1, x.shape[-1])
    if not x2.is_contiguous():
        x2 = x2.contiguous()
    y = torch.empty_like(x2)
    res2 = None
    s = None
    if residual is not None:
        res2 = residual.reshape(-1, x.shape[-1]).contiguous()
        s = torch.empty_like(x2)
    _lib.check(
        _lib.lib().lv_rmsnorm(x2.data_ptr(), _ptr(res2), weight.data_ptr(), y.data_ptr(), _ptr(s), x2.shape[0],
                              x2.shape[1], float(eps), _stream()),
        "lv_rmsnorm",
    )
    if residual is not None:
        return y.view(x.shape), s.view(x.shape)
    return y.view(x.shape)


def layernorm(x: torch.Tensor, weight: torch.Tensor, bias: Optional[torch.Tensor], eps: float = 1e-6):
    _need_cuda_bf16(x, weight, bias)
    x2 = x.reshape(-1, x.shape[-1])
    if not x2.is_contiguous():
        x2 = x2.contiguous()
    y = torch.empty_like(x2)
    _lib.check(
        _lib.lib().lv_layernorm(x2.data_ptr(), weight.data_ptr(), _ptr(bias), y.data_ptr(), x2.shape[0], x2.shape[1],
                                float(eps), _stream()),
        "lv_layernorm",
    )
    return y.view(x.shape)


def rope_table(pos: torch.Tensor, inv_freq: torch.Tensor):
    """cos, sin tables (bf16 [n, 2 * len(inv_freq)]) for int64 positions `pos` [n]."""
    _need_cuda(pos, torch.int64)
    _need_cuda(inv_freq, torch.float32)
    pos = pos.contiguous().view(-1)
    dim = 2 * inv_freq.numel()
    cos = torch.empty((pos.numel(), dim), dtype=torch.bfloat16, device=pos.device)
    sin = torch.empty_like(cos)
    _lib.check(
        _lib.lib().lv_rope_table(pos.data_ptr(), inv_freq.contiguous().data_ptr(), cos.data_ptr(), sin.data_ptr(),
                                 pos.numel(), dim, _stream()),
        "lv_rope_table",
    )
    return cos, sin


def rope(x: torch.Tensor, cos: torch.Tensor, sin: torch.Tensor, out: Optional[torch.Tensor] = None):
    """Rotate-half RoPE of x[n_tok, heads, dim] (a strided view is fine); returns a new tensor or
    writes `out` (which may be x itself)."""
    _need_cuda_bf16(x, cos, sin)
    assert x.dim() == 3 and x.stride(2) == 1
    n_tok, heads, dim = x.shape
    if out is None:
        out = torch.empty((n_tok, heads, dim), dtype=torch.bfloat16, device=x.device)
    assert out.stride(2) == 1
    _lib.check(
        _lib.lib().lv_rope(x.data_ptr(), out.data_ptr(), cos.data_ptr(), sin.data_ptr(), n_tok, heads, dim, x.stride(0),
                           x.stride(1), out.stride(0), out.stride(1), _stream()),
        "lv_rope",
    )
    return out


def swiglu(gate_up: torch.Tensor):
    _need_cuda_bf16(gate_up)
    inter = gate_up.shape[-1] // 2
    g2 = gate_up.reshape(-1, 2 * inter)
    if not g2.is_contiguous():
        g2 = g2.contiguous()
    out = torch.empty((g2.shape[0], inter), dtype=torch.bfloat16, device=gate_up.device)
    _lib.check(_lib.lib().lv_swiglu(g2.data_ptr(), out.data_ptr(), g2.shape[0], inter, _stream()), "lv_swiglu")
    return out.view(*gate_up.shape[:-1], inter)


def bias_gelu(x: torch.Tensor, bias: Optional[torch.Tensor] = None, approximate: str = "none"):
    _need_cuda_bf16(x, bias)
    x2 = x.reshape(-1, x.shape[-1])
    if not x2.is_contiguous():
        x2 = x2.contiguous()
    y = torch.empty_like(x2)
    _lib.check(
        _lib.lib().lv_bias_gelu(x2.data_ptr(), _ptr(bias), y.data_ptr(), x2.shape[0], x2.shape[1],
                                1 if approximate == "tanh" else 0, _stream()),
        "lv_bias_gelu",
    )
    return y.view(x.shape)


def ls_residual(x: torch.Tensor, y: torch.Tensor, ls: Optional[torch.Tensor] = None,
                bias: Optional[torch.Tensor] = None):
    """x + (y + bias) * ls (layer-scale residual); ls / bias optional."""
    _need_cuda_bf16(x, y, ls, bias)
    x2 = x.reshape(-1, x.shape[-1]).contiguous()
    y2 = y.reshape(-1, x.shape[-1]).contiguous()
    out = torch.empty_like(x2)
    _lib.check(
        _lib.lib().lv_ls_residual(x2.data_ptr(), y2.data_ptr(), _ptr(bias), _ptr(ls), out.data_ptr(), x2.shape[0],
                                  x2.shape[1], _stream()),
        "lv_ls_residual",
    )
    return out.view(x.shape)


def pixel_shuffle(x: torch.Tensor, hw: int, has_cls: bool):
    """[n, (1 +) hw*hw, c] -> [n, (hw/2)^2, 4c]."""
    _need_cuda_bf16(x)
    x = x.contiguous()
    n, _, c = x.shape
    out = torch.empty((n, (hw // 2) ** 2, 4 * c), dtype=torch.bfloat16, device=x.device)
    _lib.check(_lib.lib().lv_pixel_shuffle(x.data_ptr(), out.data_ptr(), n, hw, c, 1 if has_cls else 0, _stream()),
               "lv_pixel_shuffle")
    return out


def embed_scatter(ids: torch.Tensor, table: torch.Tensor, feat: Optional[torch.Tensor] = None,
                  dst_idx: Optional[torch.Tensor] = None, src_idx: Optional[torch.Tensor] = None):
    """out[t] = table[ids[t]]; out[dst_idx[i]] = feat[src_idx[i]] (src_idx None => i)."""
    _need_cuda(ids, torch.int64)
    _need_cuda_bf16(table, feat)
    ids = ids.contiguous().view(-1)
    n_tok, hidden = ids.numel(), table.shape[1]
    out = torch.empty((n_tok, hidden), dtype=torch.bfloat16, device=table.device)
    n_sc = 0
    if feat is not None:
        feat = feat.reshape(-1, hidden).contiguous()
        dst_idx = dst_idx.contiguous().view(-1)
        _need_cuda(dst_idx, torch.int64)
        n_sc = dst_idx.numel()
        if src_idx is not None:
            src_idx = src_idx.contiguous().view(-1)
            _need_cuda(src_idx, torch.int64)
    _lib.check(
        _lib.lib().lv_embed_scatter(ids.data_ptr(), table.data_ptr(), table.shape[0], _ptr(feat), _ptr(src_idx),
                                    _ptr(dst_idx), n_sc, out.data_ptr(), n_tok, hidden, _stream()),
        "lv_embed_scatter",
    )
    return out


def row_gather(x: torch.Tensor, idx: torch.Tensor):
    _need_cuda_bf16(x)
    _need_cuda(idx, torch.int64)
    x = x.contiguous()
    idx = idx.contiguous().view(-1)
    out = torch.empty((idx.numel(), x.shape[1]), dtype=torch.bfloat16, device=x.device)
    _lib.check(_lib.lib().lv_row_gather(x.data_ptr(), idx.data_ptr(), out.data_ptr(), idx.numel(), x.shape[1], _stream()),
               "lv_row_gather")
    return out


def row_scatter_zero(x: torch.Tensor, idx: torch.Tensor, n_rows_out: int):
    _need_cuda_bf16(x)
    _need_cuda(idx, torch.int64)
    x = x.contiguous()
    idx = idx.contiguous().view(-1)
    out = torch.empty((n_rows_out, x.shape[1]), dtype=torch.bfloat16, device=x.device)
    _lib.check(
        _lib.lib().lv_row_scatter_zero(x.data_ptr(), idx.data_ptr(), out.data_ptr(), idx.numel(), n_rows_out, x.shape[1],
                                       _stream()),
        "lv_row_scatter_zero",
    )
    return out


# ------------------------------------------------------------------------------------------------
# dense linears
# ------------------------------------------------------------------------------------------------
_ACT = {None: 0, "none": 0, "gelu": 1, "gelu_tanh": 2, "swiglu": 3}


def linear(x: torch.Tensor, weight: torch.Tensor, bias: Optional[torch.Tensor] = None, act: Optional[str] = None,
           out: Optional[torch.Tensor] = None):
    """act(x @ weight.T + bias); weight is [N, K] (nn.Linear layout)."""
    _need_cuda_bf16(x, weight, bias)
    K = x.shape[-1]
    N = weight.shape[0]
    x2 = x.reshape(-1, K)
    if x2.stride(1) != 1 or x2.stride(0) % 8 != 0:
        x2 = x2.contiguous()
    if weight.stride(1) != 1:
        weight = weight.contiguous()
    M = x2.shape[0]
    n_out = N // 2 if act == "swiglu" else N      # fused SwiGLU: weight rows interleaved (gate_i, up_i)
    if out is None:
        out = torch.empty((M, n_out), dtype=torch.bfloat16, device=x.device)
    if M == 0:      # e.g. a context-parallel rank that owns no answer token (empty logit mask)
        return out.view(*x.shape[:-1], n_out)
    ev0 = _TIMER.start() if _TIMER is not None else None
    _lib.check(
        _lib.lib().lv_gemm_bias_act(x2.data_ptr(), weight.data_ptr(), _ptr(bias), out.data_ptr(), M, N, K, x2.stride(0),
                                    weight.stride(0), out.stride(0), _ACT[act], _stream()),
        "lv_gemm_bias_act",
    )
    if ev0 is not None:
        _TIMER.stop("gemm_bf16", 2.0 * M * N * K, ev0)
    return out.view(*x.shape[:-1], n_out)


def interleave_gate_up(gate_w: torch.Tensor, up_w: torch.Tensor) -> torch.Tensor:
    """[I, H] gate and up projection weights -> [2I, H] with rows (gate_0, up_0, gate_1, up_1, ...):
    the operand layout of linear(..., act="swiglu") (one-time, at load)."""
    return torch.stack([gate_w, up_w], dim=1).reshape(2 * gate_w.shape[0], gate_w.shape[1]).contiguous()


def masked_linear(h: torch.Tensor, weight: torch.Tensor, logit_mask: torch.Tensor, bias: Optional[torch.Tensor] = None):
    """Logit-masked LM head forward: rows of h [s, b, c] selected by logit_mask [b, s] -> [M, b, vocab]
    (LinearWithGradAccumulationAndAsyncCommunication.forward with logit_mask,
    long_vita_megatron/core/tensor_parallel/layers.py:402-409).  b = 1 (the reference's setting when
    logit_mask is used: micro-batch 1).  The row indices are computed by torch (host-side index op)."""
    _need_cuda_bf16(h, weight, bias)
    s, b, c = h.shape
    if b != 1:
        raise NotImplementedError("masked_linear: micro-batch 1")
    idx = logit_mask.reshape(-1).nonzero().view(-1)
    sel = row_gather(h.reshape(s, c), idx)
    return linear(sel, weight, bias).view(idx.numel(), 1, weight.shape[0])


def masked_linear_dgrad(grad_out: torch.Tensor, weight: torch.Tensor, logit_mask: torch.Tensor):
    """dX of masked_linear: masked_scatter(zeros[s, b, c], dY @ W) (layers.py:443-451).  `weight` is
    [vocab, c]; the GEMM needs its transpose as the [N, K] operand, materialised by the caller once
    (weights are frozen in the reference's use of this path: linear_with_frozen_weight, :288-363)."""
    _need_cuda_bf16(grad_out, weight)
    m = grad_out.shape[0]
    s = logit_mask.shape[-1]
    wt = weight.t().contiguous()                      # [c, vocab] = the [N, K] operand of dY @ W
    gi = linear(grad_out.reshape(m, -1), wt)          # [M, c]
    idx = logit_mask.reshape(-1).nonzero().view(-1)
    return row_scatter_zero(gi, idx, s).view(s, 1, -1)


def masked_linear_wgrad(grad_out: torch.Tensor, h: torch.Tensor, logit_mask: torch.Tensor):
    """dW of masked_linear: dY^T . masked_select(h) -> [vocab, c] (layers.py:451-456, 512-520: `grad_output.t()
    .matmul(total_input)`).  Runs on the same tcgen05 GEMM with the contraction over the M selected rows: both
    operands are transposed once ([vocab, M] and [c, M]; M is the number of answer tokens) and M is zero-padded
    to a multiple of 8 (the GEMM's K granularity)."""
    _need_cuda_bf16(grad_out, h)
    s, b, c = h.shape
    m = grad_out.shape[0]
    vocab = grad_out.shape[-1]
    if m == 0:
        return torch.zeros((vocab, c), dtype=torch.bfloat16, device=h.device)
    idx = logit_mask.reshape(-1).nonzero().view(-1)
    sel = row_gather(h.reshape(s, c), idx)                              # [M, c]
    mp = (m + 7) // 8 * 8
    gt = torch.zeros((vocab, mp), dtype=torch.bfloat16, device=h.device)
    gt[:, :m] = grad_out.reshape(m, vocab).t()
    st = torch.zeros((c, mp), dtype=torch.bfloat16, device=h.device)
    st[:, :m] = sel.t()
    return linear(gt, st)                                               # [vocab, c]


class _MaskedLinearFn(torch.autograd.Function):
    """LinearWithGradAccumulationAndAsyncCommunication with `logit_mask` (layers.py:371-456) for tp = 1,
    no sequence parallelism, no gradient-accumulation fusion: forward = gather + GEMM, backward =
    dX = masked_scatter(zeros, dY W) and (when the weight trains) dW = dY^T sel."""

    @staticmethod
    def forward(ctx, h, weight, logit_mask):
        ctx.save_for_backward(h, weight, logit_mask)
        return masked_linear(h, weight, logit_mask)

    @staticmethod
    def backward(ctx, grad_out):
        h, weight, logit_mask = ctx.saved_tensors
        grad_out = grad_out.contiguous()
        gh = gw = None
        if ctx.needs_input_grad[0]:
            if grad_out.shape[0] == 0:
                gh = torch.zeros_like(h)
            else:
                gh = masked_linear_dgrad(grad_out, weight, logit_mask)
        if ctx.needs_input_grad[1]:
            gw = masked_linear_wgrad(grad_out, h, logit_mask)
        return gh, gw, None


def masked_linear_autograd(h: torch.Tensor, weight: torch.Tensor, logit_mask: torch.Tensor):
    """Differentiable logit-masked LM head (SURVEY.md 8a-12)."""
    return _MaskedLinearFn.apply(h, weight, logit_mask)


# ------------------------------------------------------------------------------------------------
# logit-masked LM head fused with the cross-entropy, chunked over the vocabulary (SURVEY.md 8f-3)
# ------------------------------------------------------------------------------------------------
def _ce_chunks(vocab: int, chunk: int):
    chunk = max(8, (chunk // 8) * 8)
    return [(v0, min(vocab, v0 + chunk)) for v0 in range(0, vocab, chunk)]


def ce_accumulate(logits: torch.Tensor, labels: torch.Tensor, run_max: torch.Tensor, run_sum: torch.Tensor, tgt: torch.Tensor,
                  col0: int) -> None:
    """Fold one vocabulary chunk of bf16 logits [M, n] (columns col0 .. col0 + n of the full row) into the running
    fp32 row statistics (in place): max, sum of exp(. - max), and the target logit where labels fall in the chunk."""
    _need_cuda_bf16(logits)
    M, n = logits.shape
    _lib.check(_lib.lib().lv_ce_accumulate(logits.data_ptr(), logits.stride(0), labels.data_ptr(), run_max.data_ptr(),
                                           run_sum.data_ptr(), tgt.data_ptr(), M, n, col0, _stream()), "lv_ce_accumulate")


def ce_grad(logits: torch.Tensor, labels: torch.Tensor, lse: torch.Tensor, dloss: torch.Tensor, col0: int) -> torch.Tensor:
    """In place: logits[M, n] (a vocabulary chunk) -> d_logits = (exp(logits - lse) - onehot) * dloss (bf16)."""
    _need_cuda_bf16(logits)
    M, n = logits.shape
    _lib.check(_lib.lib().lv_ce_grad(logits.data_ptr(), logits.stride(0), logits.data_ptr(), logits.stride(0), labels.data_ptr(),
                                     lse.data_ptr(), dloss.data_ptr(), M, n, col0, _stream()), "lv_ce_grad")
    return logits


def lm_head_ce_fwd(sel: torch.Tensor, weight: torch.Tensor, labels: torch.Tensor, vocab_chunk: int = 16384):
    """Per-row cross-entropy of `sel @ weight.T` against `labels` without materialising the [M, vocab] logits:
    for every chunk of `vocab_chunk` weight rows one GEMM into a [M, chunk] bf16 buffer + `lv_ce_accumulate`.
    sel [M, c] bf16, weight [vocab, c] bf16 (vocab % 8 == 0), labels [M] int64 (negative = ignored -> loss 0).
    Returns (loss [M] fp32, lse [M] fp32).  Same arithmetic as the reference: bf16 logits (the output dtype of its
    ColumnParallelLinear), then the loss in fp32 (gpt_vl_model.py:371-414 -> logits.float())."""
    M, c = sel.shape
    V = weight.shape[0]
    dev = sel.device
    run_max = torch.full((M,), float("-inf"), dtype=torch.float32, device=dev)
    run_sum = torch.zeros((M,), dtype=torch.float32, device=dev)
    tgt = torch.zeros((M,), dtype=torch.float32, device=dev)
    if M == 0:
        return run_sum, run_sum.clone()
    labels = labels.contiguous()
    chunks = _ce_chunks(V, vocab_chunk)
    buf = torch.empty((M, chunks[0][1] - chunks[0][0]), dtype=torch.bfloat16, device=dev)
    for v0, v1 in chunks:
        lg = linear(sel, weight[v0:v1], out=buf[:, : v1 - v0])
        ce_accumulate(lg, labels, run_max, run_sum, tgt, v0)
    lse = torch.log(run_sum) + run_max
    loss = torch.where(labels >= 0, lse - tgt, torch.zeros_like(lse))
    return loss, lse


def lm_head_ce_bwd(sel: torch.Tensor, weight: torch.Tensor, labels: torch.Tensor, lse: torch.Tensor, dloss: torch.Tensor,
                   need_dsel: bool = True, need_dw: bool = False, vocab_chunk: int = 16384):
    """Backward of lm_head_ce_fwd, chunk by chunk: the chunk's logits are recomputed (one GEMM), turned into
    d_logits = (softmax - onehot) * dloss in place (`lv_ce_grad`), and contracted by the same tcgen05 GEMM:
    d_sel += d_logits @ W[chunk] (fp32 accumulation across chunks), dW[chunk] = d_logits^T @ sel
    (layers.py:443-456, 512-520).  Returns (d_sel [M, c] bf16 or None, dW [vocab, c] bf16 or None)."""
    M, c = sel.shape
    V = weight.shape[0]
    dev = sel.device
    dsel = torch.zeros((M, c), dtype=torch.float32, device=dev) if need_dsel else None
    dw = torch.empty((V, c), dtype=torch.bfloat16, device=dev) if need_dw else None
    if M == 0:
        if dw is not None:
            dw.zero_()
        return (None if dsel is None else dsel.to(torch.bfloat16)), dw
    labels = labels.contiguous()
    dloss = dloss.contiguous().float()
    chunks = _ce_chunks(V, vocab_chunk)
    buf = torch.empty((M, chunks[0][1] - chunks[0][0]), dtype=torch.bfloat16, device=dev)
    mp = (M + 7) // 8 * 8
    if need_dw:
        st = torch.zeros((c, mp), dtype=torch.bfloat16, device=dev)        # sel^T, contraction dim padded to 8
        st[:, :M] = sel.t()
    for v0, v1 in chunks:
        n = v1 - v0
        lg = ce_grad(linear(sel, weight[v0:v1], out=buf[:, :n]), labels, lse, dloss, v0)
        if need_dsel:
            wt = weight[v0:v1].t().contiguous()                             # [c, n] = the [N, K] operand of d_logits @ W
            dsel += linear(lg, wt).float()
        if need_dw:
            gt = torch.zeros((n, mp), dtype=torch.bfloat16, device=dev)
            gt[:, :M] = lg.t()
            linear(gt, st, out=dw[v0:v1])
    return (None if dsel is None else dsel.to(torch.bfloat16)), dw


class _MaskedLMHeadCEFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, h, weight, logit_mask, labels, vocab_chunk):
        s, b, c = h.shape
        if b != 1:
            raise NotImplementedError("masked_lm_head_ce: micro-batch 1")
        idx = logit_mask.reshape(-1).nonzero().view(-1)
        sel = row_gather(h.reshape(s, c), idx)
        loss, lse = lm_head_ce_fwd(sel, weight, labels.reshape(-1), vocab_chunk)
        ctx.save_for_backward(sel, weight, idx, labels.reshape(-1), lse)
        ctx.s, ctx.vocab_chunk = s, vocab_chunk
        return loss.view(1, -1)

    @staticmethod
    def backward(ctx, dloss):
        sel, weight, idx, labels, lse = ctx.saved_tensors
        dsel, dw = lm_head_ce_bwd(sel, weight, labels, lse, dloss.reshape(-1), ctx.needs_input_grad[0], ctx.needs_input_grad[1],
                                  ctx.vocab_chunk)
        gh = None
        if dsel is not None:
            gh = row_scatter_zero(dsel, idx, ctx.s).view(ctx.s, 1, -1)
        return gh, dw, None, None, None


def masked_lm_head_ce(h: torch.Tensor, weight: torch.Tensor, logit_mask: torch.Tensor, labels: torch.Tensor,
                      vocab_chunk: int = 16384) -> torch.Tensor:
    """GPTVLModel's training tail in one differentiable op (gpt_vl_model.py:325-339 masked_select of the hidden rows,
    :339 output_layer, :379-382 masked_select of the labels done by the caller, :412 per-token loss): h [s, 1, c],
    weight [vocab, c], logit_mask [1, s] bool, labels [1, M] (the M selected label ids) -> loss [1, M] fp32.  The
    [M, vocab] logits are never materialised (1M tokens x 152 064 would be 318 GB in bf16)."""
    return _MaskedLMHeadCEFn.apply(h, weight, logit_mask, labels, vocab_chunk)


# ------------------------------------------------------------------------------------------------
# differentiable building blocks of the decoder layer (training through the `--spec` layer, SURVEY.md 8f-1)
# ------------------------------------------------------------------------------------------------
def rmsnorm_bwd(x: torch.Tensor, weight: torch.Tensor, dy: torch.Tensor, eps: float = 1e-6,
                add_in: Optional[torch.Tensor] = None):
    """Gradients of rmsnorm(x, weight): returns (dx [+ add_in], dweight).  `x` is the tensor that was normalised."""
    _need_cuda_bf16(x, weight, dy, add_in)
    cols = x.shape[-1]
    x2, dy2 = x.reshape(-1, cols).contiguous(), dy.reshape(-1, cols).contiguous()
    a2 = None if add_in is None else add_in.reshape(-1, cols).contiguous()
    rows = x2.shape[0]
    parts = int(_lib.lib().lv_rmsnorm_bwd_partials(rows, cols))
    dw_part = torch.empty((parts, cols), dtype=torch.float32, device=x.device)
    dx = torch.empty_like(x2)
    _lib.check(_lib.lib().lv_rmsnorm_bwd(x2.data_ptr(), weight.data_ptr(), dy2.data_ptr(), _ptr(a2), dx.data_ptr(),
                                         dw_part.data_ptr(), rows, cols, float(eps), _stream()), "lv_rmsnorm_bwd")
    return dx.view(x.shape), dw_part.sum(dim=0).to(torch.bfloat16)


def swiglu_bwd(gate_up: torch.Tensor, dh: torch.Tensor):
    _need_cuda_bf16(gate_up, dh)
    inter = gate_up.shape[-1] // 2
    g2, d2 = gate_up.reshape(-1, 2 * inter).contiguous(), dh.reshape(-1, inter).contiguous()
    out = torch.empty_like(g2)
    _lib.check(_lib.lib().lv_swiglu_bwd(g2.data_ptr(), d2.data_ptr(), out.data_ptr(), g2.shape[0], inter, _stream()),
               "lv_swiglu_bwd")
    return out.view(gate_up.shape)


class _RMSNormFn(torch.autograd.Function):
    """y = rmsnorm(x [+ residual]); with a residual also returns the sum (the new residual stream)."""

    @staticmethod
    def forward(ctx, x, residual, weight, eps):
        if residual is None:
            y, s = rmsnorm(x, weight, eps), x
        else:
            y, s = rmsnorm(x, weight, eps, residual=residual)
        ctx.save_for_backward(s, weight)
        ctx.eps, ctx.has_res = eps, residual is not None
        return (y, s) if residual is not None else y

    @staticmethod
    def backward(ctx, dy, ds=None):
        s, weight = ctx.saved_tensors
        dx, dw = rmsnorm_bwd(s, weight, dy.contiguous(), ctx.eps, add_in=ds if ctx.has_res else None)
        return dx, (dx if ctx.has_res else None), dw, None


def rmsnorm_autograd(x, weight, eps: float = 1e-6, residual=None):
    return _RMSNormFn.apply(x, residual, weight, eps)


class _SwiGLUFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, gate_up):
        ctx.save_for_backward(gate_up)
        return swiglu(gate_up)

    @staticmethod
    def backward(ctx, dh):
        (gate_up,) = ctx.saved_tensors
        return swiglu_bwd(gate_up, dh.contiguous())


def swiglu_autograd(gate_up):
    return _SwiGLUFn.apply(gate_up)


class _RopeFn(torch.autograd.Function):
    """rotate-half RoPE is linear in x: the gradient is the same rotation with -sin."""

    @staticmethod
    def forward(ctx, x, cos, sin):
        ctx.save_for_backward(cos, sin)
        return rope(x, cos, sin)

    @staticmethod
    def backward(ctx, dy):
        cos, sin = ctx.saved_tensors
        dy = dy if dy.stride(2) == 1 else dy.contiguous()
        return rope(dy, cos, -sin), None, None


def rope_autograd(x, cos, sin):
    return _RopeFn.apply(x, cos, sin)


class _LinearFn(torch.autograd.Function):
    """y = x W^T + b on the tcgen05 GEMM; dX = dY W and dW = dY^T X reuse the same kernel on operands transposed once
    per call (the [N, K] operand of each product must be K-contiguous); the token count is zero-padded to a multiple
    of 8 for the weight gradient (the GEMM's K granularity)."""

    @staticmethod
    def forward(ctx, x, weight, bias):
        ctx.save_for_backward(x, weight)
        ctx.has_bias = bias is not None
        return linear(x, weight, bias)

    @staticmethod
    def backward(ctx, dy):
        x, weight = ctx.saved_tensors
        n_out, k_in = weight.shape
        dy2 = dy.reshape(-1, n_out).contiguous()
        x2 = x.reshape(-1, k_in)
        dx = dw = db = None
        if ctx.needs_input_grad[0]:
            dx = linear(dy2, weight.t().contiguous()).view(x.shape)          # [T, K] = dY [T, N] . (W^T)[K, N]^T
        if ctx.needs_input_grad[1]:
            t = dy2.shape[0]
            tp = (t + 7) // 8 * 8
            dyt = torch.zeros((n_out, tp), dtype=torch.bfloat16, device=dy.device)
            dyt[:, :t] = dy2.t()
            xt = torch.zeros((k_in, tp), dtype=torch.bfloat16, device=dy.device)
            xt[:, :t] = x2.t()
            dw = linear(dyt, xt)                                             # [N, K] = dY^T [N, T] . (X^T)[K, T]^T
        if ctx.has_bias and ctx.needs_input_grad[2]:
            db = dy2.float().sum(dim=0).to(torch.bfloat16)
        return dx, dw, db


def linear_autograd(x, weight, bias=None):
    return _LinearFn.apply(x, weight, bias)


def patch_embed(images: torch.Tensor, w_pad: torch.Tensor, bias: Optional[torch.Tensor], cls: torch.Tensor,
                pos: torch.Tensor, patch: int):
    """images [n,3,S,S] -> [n, 1 + (S/patch)^2, C] (conv-as-GEMM + cls + position embedding).
    `w_pad` is the conv weight flattened to [C, 3*patch*patch] and zero-padded to a multiple of 64."""
    _need_cuda_bf16(images, w_pad, bias, cls, pos)
    images = images.contiguous()
    n, _, size, _ = images.shape
    Cc = w_pad.shape[0]
    P = (size // patch) ** 2
    ws_bytes = int(_lib.lib().lv_patch_embed_ws_bytes(n, size, patch, Cc))
    ws = torch.empty(ws_bytes // 2, dtype=torch.bfloat16, device=images.device)
    out = torch.empty((n, P + (0 if cls is None else 1), Cc), dtype=torch.bfloat16, device=images.device)
    _lib.check(
        _lib.lib().lv_patch_embed(images.data_ptr(), w_pad.contiguous().data_ptr(), _ptr(bias),
                                  None if cls is None else cls.contiguous().data_ptr(), pos.contiguous().data_ptr(), out.data_ptr(),
                                  ws.data_ptr(), n, size, patch, Cc, _stream()),
        "lv_patch_embed",
    )
    return out


def pad_patch_weight(conv_weight: torch.Tensor) -> torch.Tensor:
    """[C, 3, ps, ps] conv weight -> [C, Kpad] GEMM operand (one-time, at load)."""
    Cc = conv_weight.shape[0]
    flat = conv_weight.reshape(Cc, -1)
    k = flat.shape[1]
    kpad = (k + 63) // 64 * 64
    out = torch.zeros((Cc, kpad), dtype=conv_weight.dtype, device=conv_weight.device)
    out[:, :k] = flat
    return out

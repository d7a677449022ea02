"""The attention backward at training scale, against an fp32 reference of the same formulas.

Both passes of the backward (dK/dV per kv tile, dQ per query tile) launch min(items, SMs) persistent CTAs, and every
barrier wait after a CTA's first item depends on phase counters carried over from the items before it.  The parity
tests of test_gpu_attention_bwd.py have at most 144 items per pass, one per CTA on a B200.  Every test here except the
peaked-score one asserts that both passes have more items than the device has SMs, so each CTA walks at least two:
a later change of tile size cannot quietly make a test trivial.

Tolerance: as in test_gpu_attention_bwd.py, the error of each gradient in excess of its bf16 output-rounding floor
< 3e-3 for the whole tensor.  Every 128-row x head tile is also bounded on its own, so that one wrong work item cannot
hide in a norm over a thousand correct ones: < 5e-3, because a tile's estimate is noisier than the whole tensor's (the
ViT's last tiles hold one row: dq per-tile maximum measured 3.0e-3-3.2e-3 at a whole-tensor 1.7e-3, flash-attn 2.8's
2.6e-3 at the same shape; NVIDIA B200, 1000 W power limit).  A wrong item is off by O(1).  Peaked scores have their own bounds (test_peaked_scores_and_scale)."""
import math

import pytest
import torch

from oracle import ops as O
from tests.util import randn_bf16, seeded

TOL, TILE_TOL = 3e-3, 5e-3


def _ref(q, k, v, do, *, causal, scale=None, q_pos=None, kv_pos=None, q_block=512):
    """out, lse, dq, dk, dv of softmax(scale q k^T + mask) v in fp32 on q's device.  q / do [b, sq, hq, d], k / v
    [b, sk, hkv, d]; q_pos / kv_pos global positions (default: the bottom-right aligned mask; kv_pos ascending).
    P is taken from the exact log-sum-exp and delta = rowsum(dO * O) from the fp32 O.  Chunked over kv groups and
    blocks of `q_block` query rows, with the keys no row of a block can see left out, so 32K fits in memory."""
    assert not torch.backends.cuda.matmul.allow_tf32 and torch.backends.cuda.matmul.fp32_precision != "tf32"
    b, sq, hq, d = q.shape
    sk, hkv = k.shape[1], k.shape[2]
    G = hq // hkv
    dev = q.device
    scale = 1.0 / math.sqrt(d) if scale is None else scale
    q_pos = (torch.arange(sq) + (sk - sq) if q_pos is None else q_pos).to(dev)
    kv_pos = (torch.arange(sk) if kv_pos is None else kv_pos).to(dev)
    assert bool((kv_pos[1:] >= kv_pos[:-1]).all())
    out = torch.zeros((b, sq, hq, d), dtype=torch.float32, device=dev)
    lse = torch.empty((b, hq, sq), dtype=torch.float32, device=dev)
    dq, dk, dv = torch.zeros_like(out), torch.zeros((b, sk, hkv, d), device=dev), torch.zeros((b, sk, hkv, d), device=dev)
    for bi in range(b):
        for g in range(hkv):
            heads = slice(g * G, (g + 1) * G)
            kf, vf = k[bi, :, g].float(), v[bi, :, g].float()                        # [sk, d]
            for r0 in range(0, sq, q_block):
                r1 = min(sq, r0 + q_block)
                qp = q_pos[r0:r1]
                n = int(torch.searchsorted(kv_pos, qp.max(), right=True)) if causal else sk
                if n == 0:                     # no row of the block sees a key: out, dq = 0, lse = -inf
                    lse[bi, heads, r0:r1] = -math.inf
                    continue
                qf = q[bi, r0:r1, heads].float().transpose(0, 1)                     # [G, rows, d]
                dof = do[bi, r0:r1, heads].float().transpose(0, 1)
                s = torch.matmul(qf, kf[:n].T) * scale                              # [G, rows, n]
                if causal:
                    s = s.masked_fill(kv_pos[None, None, :n] > qp[None, :, None], -math.inf)
                l = torch.logsumexp(s, dim=-1)                                       # [G, rows]
                p = torch.nan_to_num(torch.exp(s - l[..., None]), nan=0.0)           # rows without a key: 0
                o = torch.matmul(p, vf[:n])
                delta = (dof * o).sum(-1)
                ds = p * (torch.matmul(dof, vf[:n].T) - delta[..., None])
                out[bi, r0:r1, heads] = o.transpose(0, 1)
                lse[bi, heads, r0:r1] = l
                dq[bi, r0:r1, heads] = (torch.matmul(ds, kf[:n]) * scale).transpose(0, 1)
                dk[bi, :n, g] += torch.matmul(ds.transpose(1, 2), qf).sum(0) * scale
                dv[bi, :n, g] += torch.matmul(p.transpose(1, 2), dof).sum(0)
    return out, lse, dq, dk, dv


def test_reference_matches_oracle():
    """_ref against the autograd oracle on the CPU: causal GQA at shifted global positions (a query block whose rows
    see no key, and one with a partial view)."""
    g = seeded(11)
    b, sq, sk, hq, hkv, d = 2, 80, 96, 6, 2, 32
    q, do = randn_bf16((b, sq, hq, d), g), randn_bf16((b, sq, hq, d), g)
    k, v = randn_bf16((b, sk, hkv, d), g), randn_bf16((b, sk, hkv, d), g)
    q_pos = torch.cat([torch.arange(0, 40), torch.arange(130, 170)])
    kv_pos = torch.arange(sk) + 20
    out, lse, dq, dk, dv = _ref(q, k, v, do, causal=True, scale=0.3, q_pos=q_pos, kv_pos=kv_pos, q_block=16)
    ro, rl = O.attention(q, k, v, causal=True, scale=0.3, q_pos=q_pos, kv_pos=kv_pos)
    rq, rk, rv = O.attention_grads(q, k, v, do, causal=True, scale=0.3, q_pos=q_pos, kv_pos=kv_pos)
    assert torch.equal(torch.isinf(lse), torch.isinf(rl)) and bool(torch.isinf(lse[:, :, :20]).all())
    fin = torch.isfinite(rl)
    assert float((lse[fin] - rl[fin]).abs().max() / rl[fin].abs().max()) < 1e-5
    for a, r in ((out, ro), (dq, rq), (dk, rk), (dv, rv)):
        assert float((a - r).norm() / r.norm()) < 1e-5


# ------------------------------------------------------------------------------------------------------------------
def _excess(a, r):
    """(a - r) in excess of the bf16 rounding of r, relative to |r|: whole tensor and max over 128-row x head tiles
    (tiles whose reference is exactly zero are left out; exact zeros are asserted where they are known)."""
    a, r = a.float(), r.float()
    floor = r.to(torch.bfloat16).float() - r
    b, s, h, d = r.shape
    pad = (-s) % 128

    def tiles(x):
        x = torch.nn.functional.pad(x, (0, 0, 0, 0, 0, pad))
        return x.view(b, (s + pad) // 128, 128, h, d).pow(2).sum(dim=(2, 4))       # [b, tiles, h]

    e2, f2, r2 = tiles(a - r), tiles(floor), tiles(r)
    whole = math.sqrt(max(float(e2.sum() - f2.sum()), 0.0) / float(r2.sum()))
    live = r2 > 0
    per = ((e2[live] - f2[live]).clamp_min(0) / r2[live]).sqrt()
    return whole, float(per.max()) if per.numel() else 0.0


def _check_grads(got, ref, tol=TOL, tile_tol=TILE_TOL):
    for name, a, r in zip(("dq", "dk", "dv"), got, ref):
        assert torch.isfinite(a).all(), name
        whole, tile = _excess(a, r)
        assert whole < tol and tile < tile_tol, (name, whole, tile)


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _items(b, sq, sk, hq, hkv):
    """work items of the backward's dK/dV pass and dQ pass (128-row tiles)"""
    return b * hkv * -(-sk // 128), b * hq * -(-sq // 128)


def _assert_many_items(b, sq, sk, hq, hkv):
    a, bq = _items(b, sq, sk, hq, hkv)
    assert a > _sms() and bq > _sms(), (a, bq, _sms())


def _inputs(b, sq, sk, hq, hkv, d, seed):
    g = seeded(seed)
    q, k, v = randn_bf16((b, sq, hq, d), g), randn_bf16((b, sk, hkv, d), g), randn_bf16((b, sk, hkv, d), g)
    do = randn_bf16((b, sq, hq, d), g)
    return tuple(t.cuda() for t in (q, k, v, do))


def _fwd_bwd(q, k, v, do, *, causal, scale=None, **seg):
    from long_vita_b200 import ops

    out, lse = ops.attention_fwd(q, k, v, causal=causal, scale=scale, return_lse=True, **seg)
    dq, dk, dv = ops.attention_bwd(do, q, k, v, out, lse, causal=causal, scale=scale, **seg)
    return out, lse, (dq, dk, dv)


def _cp_rank(S, cp, rank, seed):
    """One context-parallel rank's backward on one device: its zig-zag query chunks {rank, 2cp-1-rank} at their
    global positions against the whole K / V, with the segment arguments cp.CPBackwardMixin passes."""
    c = S // (2 * cp)
    q, k, v, do = _inputs(1, 2 * c, S, 40, 8, 128, seed)
    seg = dict(q_seg_len=c, q_seg_pos=(rank * c, (2 * cp - 1 - rank) * c))
    return (q, k, v, do), seg, O.zigzag_positions(S, cp, rank)


# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("b,S", [(1, 4096), (1, 16384), (3, 2047)])
def test_llm_geometry(lib_built, b, S):
    """40:8 heads x 128, causal: the bench's 16K shape (1024 dK/dV items, 1280 dQ items), 4K, and a ragged batch."""
    _assert_many_items(b, S, S, 40, 8)
    q, k, v, do = _inputs(b, S, S, 40, 8, 128, seed=S + b)
    _, _, got = _fwd_bwd(q, k, v, do, causal=True)
    _check_grads(got, _ref(q, k, v, do, causal=True)[2:])


@pytest.mark.gpu
@pytest.mark.parametrize("S,cp,rank", [(16384, 4, 0), (16384, 4, 3), (32768, 8, 2)])
def test_cp_rank(lib_built, S, cp, rank):
    """A context-parallel rank's backward: dK/dV items past the rank's last visible key are empty (they write zeros)
    and share CTAs with busy ones.  dK/dV must be exactly zero there."""
    (q, k, v, do), seg, pos = _cp_rank(S, cp, rank, seed=S + rank)
    _assert_many_items(1, q.shape[1], S, 40, 8)
    _, _, got = _fwd_bwd(q, k, v, do, causal=True, **seg)
    _check_grads(got, _ref(q, k, v, do, causal=True, q_pos=pos, kv_pos=torch.arange(S))[2:])
    last_visible = int(pos.max()) + 1
    assert not got[1][:, last_visible:].any() and not got[2][:, last_visible:].any()


@pytest.mark.gpu
def test_vit_geometry(lib_built):
    """b = 12, S = 1025, 16:16 x 64, non-causal: 1728 items per pass; each head's last query tile and last kv tile
    hold one valid row."""
    _assert_many_items(12, 1025, 1025, 16, 16)
    q, k, v, do = _inputs(12, 1025, 1025, 16, 16, 64, seed=1025)
    _, _, got = _fwd_bwd(q, k, v, do, causal=False)
    _check_grads(got, _ref(q, k, v, do, causal=False)[2:])


def _schedule_invariance(q, k, v, do, **seg):
    """The backward has no atomics and a fixed order inside each work item, so its result cannot depend on how items
    are spread over CTAs.  Cut the problem into calls with at most one item per CTA and compare bit for bit:
    dK/dV from one call per (batch, kv head) with that head's G query heads, dQ from one call per (batch, query head)."""
    from long_vita_b200 import ops

    b, sq, hq, _ = q.shape
    sk, hkv = k.shape[1], k.shape[2]
    G = hq // hkv
    _assert_many_items(b, sq, sk, hq, hkv)
    assert _items(1, sq, sk, G, 1)[0] <= _sms() and _items(1, sq, sk, 1, 1)[1] <= _sms()
    out, lse, (dq, dk, dv) = _fwd_bwd(q, k, v, do, causal=True, **seg)
    for bi in range(b):
        bs = slice(bi, bi + 1)
        for g in range(hkv):
            hs, gs = slice(g * G, (g + 1) * G), slice(g, g + 1)
            _, dk1, dv1 = ops.attention_bwd(do[bs, :, hs], q[bs, :, hs], k[bs, :, gs], v[bs, :, gs], out[bs, :, hs],
                                            lse[bs, hs], causal=True, **seg)
            assert torch.equal(dk1, dk[bs, :, gs]) and torch.equal(dv1, dv[bs, :, gs]), (bi, g)
        for h in range(hq):
            hs, gs = slice(h, h + 1), slice(h // G, h // G + 1)
            dq1, _, _ = ops.attention_bwd(do[bs, :, hs], q[bs, :, hs], k[bs, :, gs], v[bs, :, gs], out[bs, :, hs],
                                          lse[bs, hs], causal=True, **seg)
            assert torch.equal(dq1, dq[bs, :, hs]), (bi, h)


@pytest.mark.gpu
def test_schedule_invariance_llm_16k(lib_built):
    _schedule_invariance(*_inputs(1, 16384, 16384, 40, 8, 128, seed=7))


@pytest.mark.gpu
def test_schedule_invariance_cp_rank(lib_built):
    (q, k, v, do), seg, _ = _cp_rank(16384, 4, 3, seed=8)
    _schedule_invariance(q, k, v, do, **seg)


@pytest.mark.gpu
def test_megatron_strided_views(lib_built):
    """`core_attention` on the q / k / v Megatron splits off one fused [s, 1, ng, (G + 2) d] projection (k and v
    strided views, q reshaped) in training: the gradient of the fused buffer must be bit-equal to that of the same
    module on contiguous copies, and within tolerance of the reference."""
    from long_vita_b200.megatron import stub
    from long_vita_b200.megatron.core_attention import B200DotProductAttention

    s, ng, G, d = 4096, 8, 5, 128
    _assert_many_items(1, s, s, ng * G, ng)
    attn = B200DotProductAttention(stub.TransformerConfig(hidden_size=ng * G * d, num_attention_heads=ng * G,
                                                          num_query_groups=ng), 1, stub.AttnMaskType.causal)
    g = seeded(12)
    fused0 = randn_bf16((s, 1, ng, (G + 2) * d), g).cuda()
    dout = randn_bf16((s, 1, ng * G * d), g).cuda()

    def grad(contiguous):
        fused = fused0.clone().requires_grad_(True)
        q = fused[..., : G * d].reshape(s, 1, ng * G, d)
        k, v = fused[..., G * d : (G + 1) * d], fused[..., (G + 1) * d :]
        if contiguous:
            q, k, v = q.contiguous(), k.contiguous(), v.contiguous()
        else:
            assert not k.is_contiguous() and not v.is_contiguous()
        attn(q, k, v, None).backward(dout)
        return fused.grad

    strided = grad(False)
    assert torch.equal(strided, grad(True))
    bshd = fused0.permute(1, 0, 2, 3)
    q = bshd[..., : G * d].reshape(1, s, ng * G, d)
    k, v = bshd[..., G * d : (G + 1) * d], bshd[..., (G + 1) * d :]
    rq, rk, rv = _ref(q, k, v, dout.view(s, 1, ng * G, d).permute(1, 0, 2, 3), causal=True)[2:]
    gq = strided[..., : G * d].reshape(s, 1, ng * G, d).permute(1, 0, 2, 3)
    gk, gv = strided[..., G * d : (G + 1) * d].permute(1, 0, 2, 3), strided[..., (G + 1) * d :].permute(1, 0, 2, 3)
    _check_grads((gq, gk, gv), (rq, rk, rv))


@pytest.mark.gpu
@pytest.mark.parametrize("q_mult,scale", [(4.0, None), (1.0, 0.05)])
def test_peaked_scores_and_scale(lib_built, q_mult, scale):
    """Peaked softmax rows (q x 4, default scale) and a non-default scale, S = 2048, 10:2 heads: forward and gradients
    against the reference, and against flash-attn 2's error on the same inputs when it is installed.  Peaked rows put
    more weight on the bf16 rounding of P and dS: at q x 4 dq measured 3.2e-3 (per tile 4.2e-3-4.7e-3), flash-attn
    2.8's 2.9e-3 (per tile 4.3e-3) at the same shape (NVIDIA B200, 1000 W), hence 6e-3 / 1e-2 here; the flash-attn
    comparison is the tight bound."""
    S, hq, hkv, d = 2048, 10, 2, 128
    q, k, v, do = _inputs(1, S, S, hq, hkv, d, seed=int(q_mult * 10) + (scale is not None))
    q = (q.float() * q_mult).to(torch.bfloat16)
    out, lse, got = _fwd_bwd(q, k, v, do, causal=True, scale=scale)
    ro, rl, *ref = _ref(q, k, v, do, causal=True, scale=scale)
    assert _excess(out, ro)[0] < 2e-3 and float((lse - rl).abs().max()) < 1e-4, (_excess(out, ro), float((lse - rl).abs().max()))
    _check_grads(got, ref, tol=6e-3, tile_tol=1e-2)
    try:
        import flash_attn as fa
    except ImportError:
        return
    qf, kf, vf = (t.clone().requires_grad_(True) for t in (q, k, v))
    fa.flash_attn_func(qf, kf, vf, causal=True, softmax_scale=scale).backward(do)
    for a, f, r in zip(got, (qf.grad, kf.grad, vf.grad), ref):
        assert _excess(a, r)[0] < 1.25 * _excess(f, r)[0] + 2e-4, (_excess(a, r), _excess(f, r))

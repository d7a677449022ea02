"""GPU parity of the attention backward (dQ, dK, dV) against fp32 autograd of the oracle attention.
Tolerance: gradients are bf16 outputs of bf16-P / bf16-dS tensor-core GEMMs (as in flash-attn 2's
backward); bound the error in excess of the bf16 output-rounding floor by 3e-3 and require it to be
within 1.25x of flash-attn 2.8's own backward on the same inputs."""
import math

import pytest
import torch

from oracle import ops as O
from tests.util import randn_bf16, rel_fro, seeded

pytestmark = pytest.mark.gpu


def excess(out, ref):
    e, f = rel_fro(out, ref), rel_fro(ref.to(torch.bfloat16), ref)
    return math.sqrt(max(e * e - f * f, 0.0))


def run(sq, sk, hq, hkv, d, causal, b=1, seed=0):
    from long_vita_b200 import ops

    g = seeded(seed)
    q, k, v = randn_bf16((b, sq, hq, d), g), randn_bf16((b, sk, hkv, d), g), randn_bf16((b, sk, hkv, d), g)
    do = randn_bf16((b, sq, hq, d), g)
    rq, rk, rv = O.attention_grads(q, k, v, do, causal=causal)
    qg, kg, vg = (t.cuda().requires_grad_(True) for t in (q, k, v))
    out = ops.attention(qg, kg, vg, causal=causal)
    out.backward(do.cuda())
    return (qg.grad, kg.grad, vg.grad), (rq, rk, rv), (q, k, v, do)


@pytest.mark.parametrize(
    "sq,sk,hq,hkv,d,causal",
    [
        (256, 256, 4, 2, 128, True),
        (512, 512, 10, 2, 128, True),      # GQA 5:1 like the 14B model
        (384, 384, 4, 4, 128, False),
        (1025, 1025, 16, 16, 64, False),   # ViT geometry, ragged tiles
        (300, 300, 2, 1, 64, True),
        (128, 640, 2, 2, 128, True),       # bottom-right aligned causal, sk > sq
        (300, 200, 4, 2, 128, True),       # sq > sk: the first 100 query rows see no key
        (130, 40, 2, 2, 64, True),         # sq > sk: 90 of the 128 rows of the first query tile see no key
    ],
)
def test_attention_backward(lib_built, sq, sk, hq, hkv, d, causal):
    (dq, dk, dv), (rq, rk, rv), _ = run(sq, sk, hq, hkv, d, causal, seed=sq + hq)
    for name, a, r in (("dq", dq, rq), ("dk", dk, rk), ("dv", dv, rv)):
        assert torch.isfinite(a).all(), name
        e = excess(a, r)
        assert e < 3e-3, (name, e, rel_fro(a, r))
    if causal and sq > sk:
        assert not dq[:, : sq - sk].any()


def test_attention_backward_batch(lib_built):
    (dq, dk, dv), (rq, rk, rv), _ = run(260, 260, 4, 2, 128, True, b=3, seed=5)
    assert excess(dq, rq) < 3e-3 and excess(dk, rk) < 3e-3 and excess(dv, rv) < 3e-3


def test_attention_backward_vs_flash_attn(lib_built):
    fa = pytest.importorskip("flash_attn")
    (dq, dk, dv), (rq, rk, rv), (q, k, v, do) = run(1024, 1024, 10, 2, 128, True, seed=9)
    qf, kf, vf = (t.cuda().requires_grad_(True) for t in (q, k, v))
    fa.flash_attn_func(qf, kf, vf, causal=True).backward(do.cuda())
    for a, f, r in ((dq, qf.grad, rq), (dk, kf.grad, rk), (dv, vf.grad, rv)):
        assert excess(a, r) < 1.25 * excess(f, r) + 2e-4, (excess(a, r), excess(f, r))


def test_backward_is_deterministic(lib_built):
    (a1, b1, c1), _, _ = run(640, 640, 10, 2, 128, True, seed=3)
    (a2, b2, c2), _, _ = run(640, 640, 10, 2, 128, True, seed=3)
    assert torch.equal(a1, a2) and torch.equal(b1, b2) and torch.equal(c1, c2)


@pytest.mark.parametrize("cp,rank", [(2, 0), (2, 1), (4, 1)])
def test_backward_of_zigzag_query_segments(lib_built, cp, rank):
    """What one context-parallel rank runs in backward (cp.CPBackwardMixin): its two query chunks at their
    global positions against the whole K/V.  dQ is final; dK/dV are partial sums and must be exactly zero on
    kv rows none of the local queries can see."""
    from long_vita_b200 import ops

    c, hq, hkv, d = 256, 10, 2, 128
    S = 2 * cp * c
    g = seeded(40 + rank)
    q, k, v = randn_bf16((1, S, hq, d), g), randn_bf16((1, S, hkv, d), g), randn_bf16((1, S, hkv, d), g)
    do = randn_bf16((1, S, hq, d), g)
    own = torch.cat([torch.arange(rank * c, (rank + 1) * c), torch.arange((2 * cp - 1 - rank) * c, (2 * cp - rank) * c)])
    ql, dol = q[:, own].contiguous(), do[:, own].contiguous()
    rq, rk, rv = O.attention_grads(ql, k, v, dol, causal=True, q_pos=own, kv_pos=torch.arange(S))
    seg = dict(q_seg_len=c, q_seg_pos=(rank * c, (2 * cp - 1 - rank) * c))
    out, lse = ops.attention_fwd(ql.cuda(), k.cuda(), v.cuda(), causal=True, return_lse=True, **seg)
    dq, dk, dv = ops.attention_bwd(dol.cuda(), ql.cuda(), k.cuda(), v.cuda(), out, lse, causal=True, **seg)
    for name, a, r in (("dq", dq, rq), ("dk", dk, rk), ("dv", dv, rv)):
        assert torch.isfinite(a).all(), name
        assert excess(a, r) < 3e-3, (name, excess(a, r))
    last_visible = (2 * cp - rank) * c
    assert not dk[:, last_visible:].any() and not dv[:, last_visible:].any()

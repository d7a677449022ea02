"""GPU parity: fused tcgen05 attention forward through the C ABI vs the fp32 CPU oracle.

Tolerance (north_star: 1e-3 relative for bf16 activations): inputs are identical bf16 tensors and the
oracle accumulates in fp32.  The kernel's output is bf16, and rounding ANY fp32 result to bf16
already costs ~1.13e-3 relative Frobenius error (uniform rounding, rms 2^-9/sqrt(3)), so the test
measures the error IN EXCESS of that floor: excess = sqrt(e(ours, ref)^2 - e(bf16(ref), ref)^2).
The excess itself has a floor no tensor-core flash attention can beat: P is rounded to bf16 before
the P.V MMA (tcgen05 faults on an fp16 A operand against bf16 V - measured), and for zero-mean random
V that rounding shows up 1:1 in the output (relative rms 2^-9/sqrt(3)..2^-8/sqrt(3) = 1.1e-3..2.3e-3).
flash-attn 2.8 - the kernel the reference runs - measures 1.15e-3..1.49e-3 on these inputs and this
kernel 1.20e-3..1.63e-3 (tools/attn_err.py).  Bound: excess < 2e-3 and <= 1.25x flash-attn's.  The fp32 log-sum-exp, which sees no output rounding, must agree to 1e-4 absolute
(observed ~1e-6).  A live flash-attn 2.8 comparator bounds the same error from the other side."""
import math

import pytest
import torch

from oracle import ops as O
from tests.util import max_rel, randn_bf16, rel_fro, seeded

pytestmark = pytest.mark.gpu

TOL_EXCESS = 2e-3
TOL_LSE = 1e-4


def excess_error(out, ref32):
    """Relative Frobenius error of `out` against the fp32 oracle beyond the bf16 output-rounding floor."""
    e_total = rel_fro(out, ref32)
    e_floor = rel_fro(ref32.to(torch.bfloat16), ref32)
    return math.sqrt(max(e_total * e_total - e_floor * e_floor, 0.0)), e_total, e_floor


@pytest.fixture(scope="module")
def L(lib_built):
    from long_vita_b200 import ops

    return ops


def check(L, b, sq, sk, hq, hkv, d, causal, seed=0, layout="bshd", **kw):
    g = seeded(seed)
    q, k, v = randn_bf16((b, sq, hq, d), g), randn_bf16((b, sk, hkv, d), g), randn_bf16((b, sk, hkv, d), g)
    ref, lse_ref = O.attention(q, k, v, causal=causal, q_pos=kw.get("q_pos"), kv_pos=kw.get("kv_pos_t"))
    perm = {"bshd": (0, 1, 2, 3), "sbhd": (1, 0, 2, 3), "bhsd": (0, 2, 1, 3)}[layout]
    inv = [perm.index(i) for i in range(4)]
    qd, kd, vd = (t.permute(inv).contiguous().cuda() for t in (q, k, v))
    args = {k_: v_ for k_, v_ in kw.items() if k_ in ("q_seg_len", "q_seg_pos", "kv_pos0")}
    out, lse = L.attention_fwd(qd, kd, vd, causal=causal, layout=layout, return_lse=True, **args)
    out = out.permute(perm)
    # rows that see no key (causal sq > sk, keys that start after a query's position): exactly 0 and -inf
    empty = torch.isneginf(lse_ref)
    lse_empty = lse.cpu()[empty]
    assert torch.isneginf(lse_empty).all(), lse_empty.unique()[:4]
    assert not out.cpu()[empty.permute(0, 2, 1)].any()
    e_out, e_total, e_floor = excess_error(out, ref)
    finite = torch.isfinite(lse_ref)
    e_lse = float((lse.cpu()[finite] - lse_ref[finite]).abs().max())
    assert torch.equal(torch.isfinite(lse.cpu()), finite)
    assert e_out < TOL_EXCESS and e_lse < TOL_LSE, (e_out, e_total, e_floor, e_lse, max_rel(out, ref))
    return e_out, e_lse


@pytest.mark.parametrize(
    "sq,hq,hkv,d,causal",
    [
        (512, 8, 2, 128, True),       # SURVEY 8c KAT (1)
        (512, 8, 2, 128, False),
        (1025, 16, 16, 64, False),    # ViT: ragged last tile, 1 valid row
        (4096, 40, 8, 128, True),     # LLM head geometry
        (256, 5, 1, 128, True),       # exactly one work item per head
        (128, 2, 2, 64, True),        # second query tile entirely out of range
        (130, 4, 4, 64, False),
        (1, 2, 1, 128, True),         # single query row / key
        (383, 10, 2, 128, True),      # ragged causal
    ],
)
def test_attention_forward(L, sq, hq, hkv, d, causal):
    check(L, 1, sq, sq, hq, hkv, d, causal, seed=sq + d)


def test_attention_many_items_per_cta_head_dim_64(L):
    """ViT shape with more work items than SMs (12 frames x 16 heads x 5 query blocks = 960 on 148 CTAs): every CTA
    walks several items, with the ragged last one (1 valid row, second tile empty) somewhere in its list."""
    check(L, 12, 1025, 1025, 16, 16, 64, False, seed=77)


def test_attention_batch_and_layouts(L):
    check(L, 3, 300, 300, 4, 2, 128, True, seed=1, layout="bshd")
    check(L, 2, 640, 640, 4, 4, 64, False, seed=2, layout="sbhd")
    check(L, 2, 384, 384, 8, 2, 128, True, seed=3, layout="bhsd")


def test_attention_cross_lengths_bottom_right_causal(L):
    # sk > sq: query i sees keys <= i + (sk - sq)
    check(L, 1, 256, 1024, 4, 2, 128, True, seed=4)
    check(L, 1, 100, 612, 4, 4, 64, True, seed=5)
    # sq > sk: the first sq - sk query rows see no key, inside a query tile whose other rows do
    check(L, 1, 300, 200, 4, 2, 128, True, seed=10)
    check(L, 1, 130, 40, 4, 4, 64, True, seed=11)
    # keys start at position 940: query rows 0-39 (positions 900-939) see none
    check(L, 1, 256, 512, 4, 2, 128, True, seed=12, q_seg_pos=(900, 0), kv_pos0=940,
          q_pos=torch.arange(256) + 900, kv_pos_t=torch.arange(512) + 940)


def test_attention_strided_megatron_views(L):
    # q/k/v as strided views of one fused [s, b, groups, (5+1+1)*d] buffer (dot_product_attention.py:153)
    g = seeded(6)
    s, ng, d = 777, 2, 128
    fused = randn_bf16((s, 1, ng, 7 * d), g)
    fg = fused.cuda()
    q = fused[..., : 5 * d].reshape(s, 1, ng * 5, d)
    k, v = fused[..., 5 * d : 6 * d], fused[..., 6 * d :]
    qg = fg[..., : 5 * d].reshape(s, 1, ng * 5, d)
    kg, vg = fg[..., 5 * d : 6 * d], fg[..., 6 * d :]
    out = L.attention_fwd(qg, kg, vg, causal=True, layout="sbhd")
    ref, _ = O.attention(q.permute(1, 0, 2, 3), k.permute(1, 0, 2, 3), v.permute(1, 0, 2, 3), causal=True)
    assert excess_error(out.permute(1, 0, 2, 3), ref)[0] < TOL_EXCESS


def test_attention_zigzag_segments_match_full_sequence(L):
    # cp-equivalence (SURVEY 8c KAT 2): rank r's queries = chunks {r, 2cp-1-r} against the full K/V
    g = seeded(7)
    S, hq, hkv, d, cp = 2048, 10, 2, 128, 4
    q, k, v = randn_bf16((1, S, hq, d), g), randn_bf16((1, S, hkv, d), g), randn_bf16((1, S, hkv, d), g)
    ref, lse_ref = O.attention(q, k, v, causal=True)
    kd, vd = k.cuda(), v.cuda()
    c = S // (2 * cp)
    parts = []
    for r in range(cp):
        ql = O.zigzag_split(q, cp, r).cuda()
        out = L.attention_fwd(ql, kd, vd, causal=True, q_seg_len=c, q_seg_pos=(r * c, (2 * cp - 1 - r) * c))
        parts.append(out.cpu())
    full = O.zigzag_unsplit(parts)
    assert excess_error(full, ref)[0] < TOL_EXCESS


def test_attention_large_values_lazy_rescale(L):
    # growing row maxima across key tiles exercise the lazy-rescale branch (threshold 2^8)
    g = seeded(8)
    sq, h, d = 1024, 2, 128
    q = randn_bf16((1, sq, h, d), g)
    k = randn_bf16((1, sq, h, d), g)
    ramp = torch.linspace(0.2, 6.0, sq).view(1, sq, 1, 1)
    k = (k.float() * ramp).to(torch.bfloat16)
    v = randn_bf16((1, sq, h, d), g)
    ref, lse_ref = O.attention(q, k, v, causal=False)
    out, lse = L.attention_fwd(q.cuda(), k.cuda(), v.cuda(), causal=False, return_lse=True)
    assert excess_error(out, ref)[0] < TOL_EXCESS
    assert float((lse.cpu() - lse_ref).abs().max() / lse_ref.abs().max()) < 1e-3


def test_attention_vs_flash_attn_comparator(L):
    """Live comparator (the kernel the reference actually runs): our error against the fp32 oracle
    must not be worse than 1.5x flash-attn 2.8's on the same inputs."""
    fa = pytest.importorskip("flash_attn")
    g = seeded(9)
    q, k, v = randn_bf16((1, 2048, 40, 128), g), randn_bf16((1, 2048, 8, 128), g), randn_bf16((1, 2048, 8, 128), g)
    ref, _ = O.attention(q, k, v, causal=True)
    ours = L.attention_fwd(q.cuda(), k.cuda(), v.cuda(), causal=True)
    theirs = fa.flash_attn_func(q.cuda(), k.cuda(), v.cuda(), causal=True)
    e_ours, e_theirs = excess_error(ours, ref)[0], excess_error(theirs, ref)[0]
    assert e_ours < 1.25 * e_theirs, (e_ours, e_theirs)


@pytest.mark.parametrize("length,n_splits", [(1, None), (100, None), (5000, None), (5000, 1), (4096, 4), (33000, None)])
def test_attention_decode(lib_built, length, n_splits):
    """One query token against a K/V cache (LLM geometry 40:8 x 128): GQA heads packed as query rows, key range
    split over the batch dimension of lv_attn_fwd, log-sum-exp merge."""
    from long_vita_b200 import ops

    g = seeded(900 + length)
    hq, hkv, d = 40, 8, 128
    cap = (length + 255) // 128 * 128
    q = randn_bf16((hq, d), g)
    kc, vc = randn_bf16((cap, hkv, d), g), randn_bf16((cap, hkv, d), g)
    out, lse = ops.attention_decode(q.cuda(), kc.cuda(), vc.cuda(), length, n_splits=n_splits, return_lse=True)
    ref, ref_lse = O.attention(q[None, None], kc[None, :length], vc[None, :length], causal=False)
    assert out.shape == (hq, d)
    assert float((lse.cpu() - ref_lse[0, :, 0]).abs().max()) < 1e-4
    # one bf16 rounding of the partial outputs + one of the merged result
    assert rel_fro(out, ref[0, 0]) < 6e-3, rel_fro(out, ref[0, 0])

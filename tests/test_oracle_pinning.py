"""Pin the CPU oracle (tests are CPU-only).

The reference ships no tests or golden vectors, so the oracle is pinned against
  (1) golden outputs generated from the reference's OWN code (tests/golden/make_golden.py, and the outputs the
      tests below store in tests/golden/ref_recorded.pt when run with LV_RECORD_GOLDEN=1 where the reference's
      sources are present - oracle/ref_loader.py):
      InternVisionModel / ResamplerProjector / pixel_shuffle, and the WHOLE LongVITAForCausalLM.forward
      (vision tower -> projector -> embedding scatter -> Qwen2 decoder -> norm -> lm_head),
  (2) the installed third-party modules whose arithmetic the reference delegates to
      (transformers Qwen2DecoderLayer / Qwen2RMSNorm / rotary embedding),
  (3) internal identities: the zig-zag ring schedule equals full causal attention, zig-zag
      split / unsplit round-trips, index_of_a_in_b, masked linear forward/backward vs autograd.
"""
import hashlib
import os
import sys

import pytest
import torch

from long_vita_b200.config import LongVITAConfig
from long_vita_b200.weights import synthetic_state_dict
from oracle import model as OM
from oracle import ops as O
from oracle import ref_loader
from tests.util import digest, recorded

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
sys.path.insert(0, GOLD)


def _tiny_vit_weights(seed):
    cfg = LongVITAConfig.tiny(layers=1, vit_layers=2)
    return cfg, synthetic_state_dict(cfg, seed=seed, dtype=torch.float32, perturb=True, llm_layers=[])


def test_vit_and_projector_match_reference_golden():
    from make_golden import golden_images

    gold = torch.load(os.path.join(GOLD, "ref_vit_tiny.pt"))
    cfg, w = _tiny_vit_weights(gold["seed"])
    images = golden_images(gold["seed"], cfg.visual.image_size)
    assert hashlib.sha256(images.view(torch.int16).numpy().tobytes()).hexdigest() == gold["images_sha256"]
    vit = OM.vit_forward(cfg, w, images.float())
    proj = OM.projector_forward(cfg, w, vit[:, 1:, :])
    proj_s = proj[:, gold["proj_rows"]]                   # the fixture keeps two of every three projector rows
    assert torch.allclose(vit, gold["vit_out"], rtol=1e-4, atol=1e-4), float((vit - gold["vit_out"]).abs().max())
    assert torch.allclose(proj_s, gold["proj_out"], rtol=1e-4, atol=1e-4)


def test_pixel_shuffle_matches_reference_golden_bit_exact():
    gold = torch.load(os.path.join(GOLD, "ref_pixel_shuffle.pt"))
    assert torch.equal(O.pixel_shuffle_half(gold["x"]), gold["y"])


def test_live_reference_modules_agree_with_golden_files():
    """A recorded run of the reference's pixel_shuffle reproduces the committed fixture, and on a second geometry
    (odd batch, wider channels) agrees with the oracle bit for bit."""
    gold = torch.load(os.path.join(GOLD, "ref_pixel_shuffle.pt"))
    x2 = torch.arange(3 * 4 * 4 * 10, dtype=torch.int32).reshape(3, 4, 4, 10)

    def run():
        ref = ref_loader.load()
        return {"y": ref.pixel_shuffle(gold["x"], 0.5).clone(), "y2": ref.pixel_shuffle(x2, 0.5).clone()}

    r = recorded("pixel_shuffle", run)
    assert torch.equal(r["y"], gold["y"])
    assert torch.equal(O.pixel_shuffle_half(x2), r["y2"])


def _sha(t):
    return hashlib.sha256(t.contiguous().view(torch.int32).numpy().tobytes()).hexdigest()


def _long_vita_golden():
    from make_golden import LV_SEED, long_vita_inputs

    gold = torch.load(os.path.join(GOLD, "ref_long_vita_tiny.pt"))
    assert gold["seed"] == LV_SEED
    cfg = LongVITAConfig.tiny(layers=2, vit_layers=1)
    w = synthetic_state_dict(cfg, seed=gold["seed"], dtype=torch.float32, perturb=True)
    ids, images, idx = long_vita_inputs(cfg, gold["seed"])
    # the fixture was produced from these very tensors (guards against RNG drift between torch versions)
    assert _sha(images) == gold["images_sha256"] and _sha(w["model.embed_tokens.weight"]) == gold["embed_sha256"]
    return gold, cfg, w, ids, images, idx


def test_whole_model_oracle_matches_the_references_own_forward():
    """oracle.model.long_vita_forward against outputs of the reference's LongVITAForCausalLM.forward itself
    (modeling_long_vita.py, run from /root/reference by tests/golden/make_golden.py): every decoder layer's
    input, the final normed state and the logits, fp32."""
    gold, cfg, w, ids, images, idx = _long_vita_golden()
    logits, hidden, h_final = OM.long_vita_forward(cfg, w, ids, images, idx, num_logits_to_keep=8, return_hidden=True)
    rows = gold["rows"]
    ref_h = gold["hidden_rows"]                       # [layers + 1 (inputs of each layer ... final norm), 16, H]
    for li in range(cfg.num_hidden_layers):
        assert torch.allclose(hidden[li][rows], ref_h[li], rtol=2e-4, atol=2e-4), (li, float((hidden[li][rows] - ref_h[li]).abs().max()))
    assert torch.allclose(h_final[rows], ref_h[-1], rtol=2e-4, atol=2e-4)
    assert torch.allclose(logits[0], gold["logits_last8"], rtol=2e-4, atol=2e-4), float((logits[0] - gold["logits_last8"]).abs().max())
    assert float((logits[0] - gold["logits_last8"]).norm() / gold["logits_last8"].norm()) < 1e-5
    # the loss the reference returns for `labels` (shifted, -100 ignored) from the oracle's full logits
    from make_golden import golden_labels

    full = OM.long_vita_forward(cfg, w, ids, images, idx)[0]
    labels = golden_labels(ids)[0]
    want = torch.nn.functional.cross_entropy(full[:-1].float(), labels[1:], ignore_index=-100)
    assert abs(float(want) - float(gold["loss"])) < 1e-4


def test_live_reference_forward_reproduces_the_whole_model_golden():
    """A recorded run of the reference's forward reproduces the committed last-8 logits; its logits of every position
    (num_logits_to_keep = 0), at four of the fixture's sampled rows, match the oracle's full forward."""
    gold, cfg, w, ids, images, idx = _long_vita_golden()
    rows = gold["rows"][::4]

    def run():
        model = ref_loader.build_reference_long_vita(cfg, w)
        with torch.no_grad():
            last8 = model(input_ids=ids, images=images, image_indices=idx, num_logits_to_keep=8).logits[0]
            full = model(input_ids=ids, images=images, image_indices=idx).logits[0]
        return {"logits_last8": digest(last8), "logits_rows": full[rows].clone()}

    r = recorded("long_vita_forward", run)
    assert r["logits_last8"] == digest(gold["logits_last8"])
    logits = OM.long_vita_forward(cfg, w, ids, images, idx)[0]
    assert torch.allclose(logits[rows], r["logits_rows"], rtol=2e-4, atol=2e-4), float((logits[rows] - r["logits_rows"]).abs().max())


def test_live_reference_cp_function_reproduces_the_shard_golden():
    """A recorded run of the reference's get_batch_on_this_cp_rank reproduces the committed shards."""
    from make_golden import cp_golden_prompt

    gold = torch.load(os.path.join(GOLD, "ref_cp_shards.pt"))
    ids, idx = cp_golden_prompt()
    S = ids.shape[1]

    def run():
        out = {}
        for (cp, r) in list(gold["shards"])[:3]:
            mod, cpu_placement = ref_loader.load_megatron_training_utils(cp, r, S)
            batch = {"tokens": ids.clone(), "position_ids": torch.arange(S).unsqueeze(0),
                     "external_images": torch.arange(idx.shape[1]).view(-1, 1).clone(), "external_indices": idx.clone(),
                     "attention_mask": None}
            with cpu_placement():
                b = mod.get_batch_on_this_cp_rank(batch)
            out[(cp, r)] = {k: None if v is None else digest(v) for k, v in b.items()}
        assert torch.arange(3, device="cpu").device.type == "cpu" and torch.tensor([1]).sum() == 1   # patches were undone
        return out

    got = recorded("cp_shards", run)
    assert list(got) == list(gold["shards"])[:3]
    for (cp, r), b in got.items():
        want = gold["shards"][(cp, r)]
        assert set(b) == set(want)
        for k, v in want.items():
            assert (v is None and b[k] is None) or b[k] == digest(v), (cp, r, k)


def test_oracle_full_forward_equals_the_references_incremental_decoding():
    """The reference's own KV-cache decoding (three single-token steps after a use_cache prefill,
    tests/golden/ref_long_vita_decode.pt) gives the logits of a full forward over the extended sequence - which is
    what the oracle computes.  This is the fixture the decode path of the build is checked against."""
    from make_golden import decode_new_tokens

    gold, cfg, w, ids, images, idx = _long_vita_golden()
    dec = torch.load(os.path.join(GOLD, "ref_long_vita_decode.pt"))
    new = decode_new_tokens(cfg)
    s = ids.shape[1]
    assert dec["cache_len"] == s + new.shape[1]
    logits = OM.long_vita_forward(cfg, w, torch.cat([ids, new], dim=1), images, idx)[0]
    assert torch.allclose(logits[s - 1], dec["prefill_last"], rtol=2e-4, atol=2e-4)
    for i in range(new.shape[1]):
        assert torch.allclose(logits[s + i], dec["steps"][i], rtol=2e-4, atol=2e-4), i


def test_rope_matches_the_references_own_megatron_rope():
    """oracle rope tables / apply against the reference's Megatron RotaryEmbedding.forward and
    apply_rotary_pos_emb_bshd (rotary_pos_embedding.py:84-122, 181-204) - bit-exact - and the zig-zag slice of the
    table under cp = 2 (:36-47) against the table evaluated at cp.zigzag_index positions."""
    from make_golden import rope_golden_input

    from long_vita_b200 import cp as CP

    gold = torch.load(os.path.join(GOLD, "ref_megatron_rope.pt"))
    S = gold["S"]
    inv = O.rope_inv_freq(128, 1e6)
    freqs = torch.outer(torch.arange(S).float(), inv)
    emb = torch.cat((freqs, freqs), dim=-1)
    assert torch.equal(emb, gold["emb"].view(S, 128))
    t = rope_golden_input()
    cos, sin = O.rope_tables(torch.arange(S), inv, torch.bfloat16)
    assert torch.equal(O.rope_apply(t[:, 0], cos, sin), gold["applied"][:, 0])
    for r in range(2):
        own = CP.zigzag_index(S, 2, r)
        assert torch.equal(emb[own], gold[f"emb_cp2_rank{r}"].view(-1, 128))


def test_embedding_merge_modes_match_the_references_own_embedding():
    """oracle.embed_scatter against the reference's LanguageModelEmbedding.forward (language_model_embedding.py
    :91-174) in its four `external_feature_dict` shapes - bit-exact (index ops)."""
    from make_golden import embedding_golden_inputs

    gold = torch.load(os.path.join(GOLD, "ref_megatron_embedding.pt"))
    table, ids, feat, idx = embedding_golden_inputs()
    s, tpi = ids.shape[1], feat.shape[1]
    assert torch.equal(O.embed_scatter(ids.view(-1), table), gold["none"][:, 0])                    # [s, b, h] -> [s, h]
    assert torch.equal(O.embed_scatter(ids.view(-1), table, feat, idx[1].reshape(-1)), gold["indices"][:, 0])
    assert torch.equal(O.embed_scatter(ids.view(-1), table, feat[:1], 5 + torch.arange(tpi)), gold["pre_len"][:, 0])
    (src_b, src_s), (tgt_b, tgt_s) = gold["src"], gold["tgt"]
    assert torch.equal(O.embed_scatter(ids.view(-1), table, feat, tgt_b * s + tgt_s, src_b * tpi + src_s), gold["src_tgt"][:, 0])


def test_masked_linear_matches_the_references_own_autograd_function():
    """oracle masked_linear_fwd / _bwd against the reference's LinearWithGradAccumulationAndAsyncCommunication with
    logit_mask (layers.py:365-534): output, dX = masked_scatter(zeros, dY W), dW = dY^T sel (fp32)."""
    from make_golden import masked_linear_golden_inputs

    gold = torch.load(os.path.join(GOLD, "ref_megatron_masked_linear.pt"))
    h, w, mask, dy = masked_linear_golden_inputs()
    assert torch.allclose(O.masked_linear_fwd(h, w, mask), gold["out"], rtol=1e-5, atol=1e-5)
    gx, gw = O.masked_linear_bwd(dy, h, w, mask)
    assert torch.allclose(gx, gold["dx"], rtol=1e-5, atol=1e-5) and torch.allclose(gw, gold["dw"], rtol=1e-5, atol=1e-5)
    unmasked = ~mask[0]
    assert not gold["dx"][unmasked].any()


def _hf_qwen2_layer(cfg, w, i=0):
    from transformers import Qwen2Config
    from transformers.models.qwen2 import modeling_qwen2 as Q

    hf = Qwen2Config(vocab_size=cfg.vocab_size, hidden_size=cfg.hidden_size, intermediate_size=cfg.intermediate_size,
                     num_hidden_layers=1, num_attention_heads=cfg.num_attention_heads,
                     num_key_value_heads=cfg.num_key_value_heads, rms_norm_eps=cfg.rms_norm_eps,
                     rope_theta=cfg.rope_theta, max_position_embeddings=1 << 20, attention_dropout=0.0)
    hf._attn_implementation = "eager"
    layer = Q.Qwen2DecoderLayer(hf, 0).eval()
    p = f"model.layers.{i}."
    layer.load_state_dict({k[len(p):]: t for k, t in w.items() if k.startswith(p)}, strict=True)
    return hf, layer, Q


def test_decoder_layer_matches_transformers_qwen2():
    cfg = LongVITAConfig.tiny(layers=1)
    w = synthetic_state_dict(cfg, seed=77, dtype=torch.float32, perturb=True, vit_layers=[])
    hf, layer, Q = _hf_qwen2_layer(cfg, w)
    s = 96
    g = torch.Generator().manual_seed(5)
    x = torch.randn(s, cfg.hidden_size, generator=g)
    pos = torch.arange(s)
    cos, sin = O.rope_tables(pos, O.rope_inv_freq(cfg.head_dim, cfg.rope_theta), torch.float32)
    ours = OM.decoder_layer(cfg, w, 0, x, cos, sin)
    rot = Q.Qwen2RotaryEmbedding(hf)
    hcos, hsin = rot(x[None], pos[None])
    assert torch.allclose(hcos[0], cos, atol=1e-6) and torch.allclose(hsin[0], sin, atol=1e-6)
    mask = torch.full((s, s), float("-inf")).triu(1)[None, None]
    with torch.no_grad():
        theirs = layer(x[None], attention_mask=mask, position_ids=pos[None], position_embeddings=(hcos, hsin))
    theirs = theirs[0] if isinstance(theirs, tuple) else theirs
    assert torch.allclose(ours, theirs.reshape(s, -1), rtol=1e-4, atol=1e-4), float((ours - theirs.reshape(s, -1)).abs().max())


def test_rmsnorm_matches_transformers_bf16_bitwise():
    from transformers.models.qwen2.modeling_qwen2 import Qwen2RMSNorm

    g = torch.Generator().manual_seed(6)
    x = torch.randn(33, 640, generator=g).to(torch.bfloat16)
    m = Qwen2RMSNorm(640, eps=1e-6).to(torch.bfloat16)
    m.weight.data = (1 + 0.1 * torch.randn(640, generator=g)).to(torch.bfloat16)
    assert torch.equal(O.rmsnorm(x, m.weight.data, 1e-6), m(x))


@pytest.mark.parametrize("cp", [2, 4, 8])
def test_zigzag_ring_schedule_equals_full_causal_attention(cp):
    g = torch.Generator().manual_seed(cp)
    S, hq, hkv, d = 64 * cp, 4, 2, 32
    q, k, v = (torch.randn(1, S, h, d, generator=g) for h in (hq, hkv, hkv))
    ref, lse = O.attention(q, k, v, causal=True)
    outs, lses = O.ring_attention_zigzag(q, k, v, cp)
    full = O.zigzag_unsplit(outs)
    full_lse = O.zigzag_unsplit([l.permute(0, 2, 1) for l in lses]).permute(0, 2, 1)
    assert torch.allclose(full, ref, atol=2e-5) and torch.allclose(full_lse, lse, atol=2e-5)


def test_zigzag_split_roundtrip_and_reference_formula():
    x = torch.arange(2 * 48 * 3).reshape(2, 48, 3)
    for cp in (1, 2, 4):
        parts = [O.zigzag_split(x, cp, r) for r in range(cp)]
        assert torch.equal(O.zigzag_unsplit(parts), x)
        for r in range(cp):
            # val.view(.., 2cp, S/2cp, ..).index_select(seq_dim, [r, 2cp-1-r]) (training/utils.py:331-341)
            v = x.view(2, 2 * cp, 48 // (2 * cp), 3).index_select(1, torch.tensor([r, 2 * cp - 1 - r])).reshape(2, -1, 3)
            assert torch.equal(parts[r], v)


def test_index_of_a_in_b():
    g = torch.Generator().manual_seed(3)
    b = torch.randperm(1000, generator=g)[:400]
    a = b[torch.randperm(400, generator=g)[:150]]
    idx = O.index_of_a_in_b(a, b)
    assert torch.equal(b[idx], a)
    # the reference's formulation (training/utils.py:347-350)
    b_idx = torch.where(torch.isin(b, a))[0]
    ref = b_idx[b[b_idx].argsort()[a.argsort().argsort()]]
    assert torch.equal(idx, ref)


def test_masked_linear_forward_backward_match_autograd():
    g = torch.Generator().manual_seed(4)
    s, b, c, vocab = 40, 1, 32, 50
    h = torch.randn(s, b, c, generator=g, requires_grad=True)
    wt = torch.randn(vocab, c, generator=g, requires_grad=True)
    mask = (torch.rand(b, s, generator=g) < 0.3)
    out = O.masked_linear_fwd(h, wt, mask)
    dense = torch.matmul(h, wt.t())[mask.transpose(0, 1)].reshape(-1, b, vocab)
    assert torch.allclose(out, dense, atol=1e-6)
    go = torch.randn(out.shape, generator=g)
    out.backward(go)
    gx, gw = O.masked_linear_bwd(go, h.detach(), wt.detach(), mask)
    assert torch.allclose(gx, h.grad, atol=1e-5) and torch.allclose(gw, wt.grad, atol=1e-5)


def test_whole_model_oracle_runs_and_uses_image_features():
    cfg = LongVITAConfig.tiny(layers=2, vit_layers=1)
    w = synthetic_state_dict(cfg, seed=9, dtype=torch.float32, perturb=True)
    g = torch.Generator().manual_seed(1)
    s = 300
    ids = torch.randint(0, cfg.vocab_size, (1, s), generator=g)
    images = torch.randn(1, 3, 448, 448, generator=g)
    idx = torch.stack([torch.zeros(1, 256, dtype=torch.long), torch.arange(10, 266).view(1, 256)])
    a = OM.long_vita_forward(cfg, w, ids, images, idx, num_logits_to_keep=1)
    b = OM.long_vita_forward(cfg, w, ids, images * 0.5, idx, num_logits_to_keep=1)
    c = OM.long_vita_forward(cfg, w, ids, None, None, num_logits_to_keep=1)
    assert a.shape == (1, 1, cfg.vocab_size)
    assert not torch.allclose(a, b) and not torch.allclose(a, c)


def test_live_megatron_vision_downsample_matches_oracle_bit_exact():
    """The Megatron twin of the projector's front end - MegatronVisionModel.forward_downsample / pixel_shuffle
    (long_vita_megatron/pretrain_long_vita.py:467-483, 572-582), a recorded run of the reference's code: drop the
    class token, view as [n, 32, 32, C], pixel-shuffle x0.5."""
    import types

    x = torch.arange(2 * 17 * 6, dtype=torch.int32).reshape(2, 17, 6)               # 1 class token + 4 x 4 patches

    def run():
        m = ref_loader.load_class_methods("long_vita_megatron/pretrain_long_vita.py", "MegatronVisionModel",
                                          {"forward_downsample", "pixel_shuffle"})
        me = types.SimpleNamespace(add_class_token=True, vision_downsample_ratio=0.5, vision_downsample_stride=1)
        me.pixel_shuffle = lambda x, scale_factor=0.5: m["pixel_shuffle"](me, x, scale_factor)
        return m["forward_downsample"](me, x).clone()

    want = recorded("megatron_vision_downsample", run)
    got = O.pixel_shuffle_half(x[:, 1:].reshape(2, 4, 4, 6)).reshape(2, 4, 24)
    assert torch.equal(got, want)


def test_attention_forward_and_grads_match_transformers_eager_attention():
    """The attention the reference's HF path delegates to when flash-attn is absent - transformers'
    `eager_attention_forward` (repeat_kv + softmax(QK^T * scaling + causal mask) V) - and its autograd, against
    oracle.ops.attention / attention_grads (causal GQA 5:1)."""
    import types

    from transformers.models.qwen2.modeling_qwen2 import eager_attention_forward

    g = torch.Generator().manual_seed(17)
    b, s, hq, hkv, d = 1, 96, 10, 2, 32
    q, k, v = (torch.randn(b, s, h, d, generator=g) for h in (hq, hkv, hkv))
    do = torch.randn(b, s, hq, d, generator=g)
    qq, kk, vv = (t.clone().transpose(1, 2).requires_grad_(True) for t in (q, k, v))          # [b, h, s, d]
    mask = torch.triu(torch.full((s, s), torch.finfo(torch.float32).min), diagonal=1)[None, None]
    mod = types.SimpleNamespace(num_key_value_groups=hq // hkv, training=False)
    out, _ = eager_attention_forward(mod, qq, kk, vv, mask, scaling=d ** -0.5, dropout=0.0)   # [b, s, h, d]
    out.backward(do)
    ref, _ = O.attention(q, k, v, causal=True)
    assert torch.allclose(ref, out.detach(), rtol=1e-5, atol=1e-5)
    dq, dk, dv = O.attention_grads(q, k, v, do, causal=True)
    for a, r in ((dq, qq.grad), (dk, kk.grad), (dv, vv.grad)):
        assert torch.allclose(a, r.transpose(1, 2), rtol=1e-4, atol=1e-5)


def test_siglip_tower_matches_transformers_siglip_encoder():
    """a9: oracle.model.siglip_forward (the Megatron SigLIPViTModel of siglip_vit_model.py:165-228: conv patch embed +
    learned positions, pre-LN blocks with tanh-GELU, no class token, NO final layer norm) against the HF SigLIP vision
    encoder the Megatron weights are converted from - its last hidden state before `post_layernorm`.  The q/k/v
    projections are re-laid into Megatron's per-head interleave [head, (q, k, v), hn]."""
    from types import SimpleNamespace

    from transformers import SiglipVisionConfig, SiglipVisionModel

    torch.manual_seed(3)
    C, I, H, L = 144, 304, 2, 2                       # head_dim 72, as the real SigLIP-so400m
    hf = SiglipVisionModel(SiglipVisionConfig(hidden_size=C, intermediate_size=I, num_hidden_layers=L, num_attention_heads=H,
                                              image_size=448, patch_size=14, hidden_act="gelu_pytorch_tanh",
                                              layer_norm_eps=1e-6, attn_implementation="eager")).eval()
    sd = hf.state_dict()
    e = "vision_model."
    hn = C // H
    w = {"conv1.weight": sd[e + "embeddings.patch_embedding.weight"], "conv1.bias": sd[e + "embeddings.patch_embedding.bias"],
         "position_embeddings.weight": sd[e + "embeddings.position_embedding.weight"]}
    for i in range(L):
        h, m = f"{e}encoder.layers.{i}.", f"decoder.layers.{i}."
        qkv_w = torch.stack([sd[h + f"self_attn.{n}_proj.weight"].view(H, hn, C) for n in "qkv"], dim=1).reshape(3 * C, C)
        qkv_b = torch.stack([sd[h + f"self_attn.{n}_proj.bias"].view(H, hn) for n in "qkv"], dim=1).reshape(3 * C)
        w.update({m + "input_layernorm.weight": sd[h + "layer_norm1.weight"], m + "input_layernorm.bias": sd[h + "layer_norm1.bias"],
                  m + "self_attention.linear_qkv.weight": qkv_w, m + "self_attention.linear_qkv.bias": qkv_b,
                  m + "self_attention.linear_proj.weight": sd[h + "self_attn.out_proj.weight"],
                  m + "self_attention.linear_proj.bias": sd[h + "self_attn.out_proj.bias"],
                  m + "pre_mlp_layernorm.weight": sd[h + "layer_norm2.weight"], m + "pre_mlp_layernorm.bias": sd[h + "layer_norm2.bias"],
                  m + "mlp.linear_fc1.weight": sd[h + "mlp.fc1.weight"], m + "mlp.linear_fc1.bias": sd[h + "mlp.fc1.bias"],
                  m + "mlp.linear_fc2.weight": sd[h + "mlp.fc2.weight"], m + "mlp.linear_fc2.bias": sd[h + "mlp.fc2.bias"]})
    images = torch.randn(2, 3, 448, 448, generator=torch.Generator().manual_seed(4))
    with torch.no_grad():
        ref = hf(pixel_values=images, output_hidden_states=True).hidden_states[-1]
    cfg = SimpleNamespace(hidden_size=C, num_attention_heads=H, kv_channels=hn, num_layers=L, patch_dim=14, layernorm_epsilon=1e-6)
    out = OM.siglip_forward(cfg, w, images)
    assert out.shape == ref.shape == (2, 1024, C)
    assert torch.allclose(out, ref, rtol=1e-4, atol=1e-4), float((out - ref).abs().max())


def test_live_megatron_local_rmsnorm_matches_oracle_bit_exact():
    """a5: the reference's Megatron-local RMSNorm (core/transformer/custom_layers/transformer_engine.py:54-79:
    `_norm(x.float()).type_as(x) * weight`), a recorded run of the reference's code, against oracle.ops.rmsnorm in bf16."""
    import types

    g = torch.Generator().manual_seed(2)
    x = (torch.randn(37, 640, generator=g) * 3).to(torch.bfloat16)
    w = (1 + 0.1 * torch.randn(640, generator=g)).to(torch.bfloat16)

    def run():
        m = ref_loader.load_class_methods("long_vita_megatron/core/transformer/custom_layers/transformer_engine.py", "RMSNorm",
                                          {"_norm", "forward"})
        me = types.SimpleNamespace(eps=1e-6, weight=w)
        me._norm = lambda t: m["_norm"](me, t)
        return digest(m["forward"](me, x))

    assert recorded("megatron_local_rmsnorm", run) == digest(O.rmsnorm(x, w, 1e-6))


# ---- frame preprocessing (SURVEY.md 8f-4): Pillow's fixed-point bicubic resize + normalisation ----
def test_frame_preprocessing_oracle_matches_the_references_own_process_images_fixture():
    """tests/golden/ref_preprocess.pt = outputs of the reference's own ImageProcessor.process_images
    (image_processor.py:183-223, run from /root/reference with Pillow) on seeded frames: wide, tall, square,
    down- and up-scaled.  The numpy restatement of Pillow's 8-bit resample must reproduce them bit for bit."""
    import numpy as np

    from oracle import preprocess as P

    g = torch.load(os.path.join(GOLD, "ref_preprocess.pt"))
    for frames, want in zip(g["frames"], g["out"]):
        got = P.process_frames(list(frames.numpy()), image_size=g["image_size"])
        assert got.dtype == np.float32 and np.array_equal(got, want.numpy()), frames.shape


def test_frame_preprocessing_oracle_matches_the_reference_live_at_448():
    """The reference's ImageProcessor.process_images at the real 448 size (a recorded run: the digest of each output,
    which is too large to store) against the oracle, bit for bit."""
    import sys

    import numpy as np

    sys.path.insert(0, GOLD)
    from make_golden import reference_process_images

    from oracle import preprocess as P

    rng = np.random.default_rng(7)
    shapes = [(360, 640), (500, 333), (448, 448), (100, 100), (448, 600)]
    frames = [rng.integers(0, 256, (2, h, w, 3), dtype=np.uint8) for h, w in shapes]
    want = recorded("process_images_448", lambda: [digest(reference_process_images(f, 448).numpy()) for f in frames])
    assert len(want) == len(frames)
    for f, d in zip(frames, want):
        assert digest(P.process_frames(list(f))) == d, f.shape
    # the product's host-side coefficient tables (long_vita_b200/preprocess.py) are the oracle's
    from long_vita_b200 import preprocess as PP

    for a in (1920, 640, 500, 448, 100):
        xm, cn, kk = P.resample_coeffs(a, 448)
        x2, c2, r2, _ = PP.resample_table(a, 448)
        assert np.array_equal(xm, np.array(x2)) and np.array_equal(cn, np.array(c2)) and np.array_equal(kk, np.array(r2))


def test_dynamic_tiling_oracle_matches_the_references_own_process_dynamic_fixture():
    """tests/golden/ref_preprocess_dynamic.pt = outputs of the reference's own ImageProcessor.process_dynamic
    (image_processor.py:263-285 with dynamic_preprocess :404-448, Pillow's resize) on seeded images at a 28-pixel tile
    (wide, tall, square, tiny; up- and down-scaled; 1 to 12 tiles + thumbnail) - tests/golden/make_golden.py."""
    import numpy as np

    from oracle import preprocess as P

    g = torch.load(os.path.join(GOLD, "ref_preprocess_dynamic.pt"))
    for im, ref, gp in zip(g["images"], g["out"], g["grid_pixels"]):
        got, grid = P.process_dynamic(im.numpy(), g["min_patch_grid"], g["max_patch_grid"], g["image_size"])
        assert grid == tuple(gp)
        assert np.array_equal(got, ref.numpy()), tuple(im.shape)


def test_dynamic_tiling_oracle_matches_the_reference_live_at_448():
    """The same comparison at the real tile size, including a grid that is narrower than the image on one axis and
    wider on the other (a recorded run of the reference: grid and digest of each output)."""
    import numpy as np

    sys.path.insert(0, GOLD)
    from make_golden import reference_process_dynamic

    from oracle import preprocess as P

    rng = np.random.default_rng(5)
    images = [rng.integers(0, 256, (h, w, 3), dtype=np.uint8) for h, w in ((500, 700), (1300, 400), (448, 448), (600, 2100))]

    def run():
        out = []
        for im in images:
            ref, gref = reference_process_dynamic(im, 448)
            out.append((tuple(int(x) for x in gref), digest(ref.numpy())))
        return out

    want = recorded("process_dynamic_448", run)
    assert len(want) == len(images)
    for im, (gref, d) in zip(images, want):
        got, grid = P.process_dynamic(im, 1, 12, 448)
        assert grid == gref, im.shape
        assert digest(got) == d, im.shape

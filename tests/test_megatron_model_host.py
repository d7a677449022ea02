"""CPU tests of the host logic around the Megatron surface (SURVEY.md 8a-15, 8a-11, 8a-12):

* `megatron.checkpoint`: the mcore <-> HF weight layouts are bit-exact permutations, checked against
  an independent restatement of the index description in tools/hf2mcore_long_vita.py:397-414, 488-504.
* `megatron.gpt_vl_model.B200GPTVLModel.forward`: argument handling, the three embedding merge
  modes, logit_mask, labels / loss, `inference_params` overrides - with the operator wrappers
  replaced by the CPU oracle (tests/hostlogic.py), against oracle.model.long_vita_forward.
  This checks composition and indexing only; kernel parity is the `-m gpu` suite.
"""
import types

import pytest
import torch

from long_vita_b200.config import LongVITAConfig
from long_vita_b200.megatron import checkpoint as ck
from long_vita_b200.weights import synthetic_state_dict
from oracle import model as OM
from tests.hostlogic import oracle_ops
from tests.util import digest, recorded, rel_fro


@pytest.fixture(scope="module")
def tiny():
    cfg = LongVITAConfig.tiny(layers=2, vit_layers=1)
    hf = synthetic_state_dict(cfg, seed=77, dtype=torch.bfloat16, perturb=True)
    return cfg, hf, ck.hf_to_mcore(hf, cfg)


def test_checkpoint_roundtrip_is_bit_exact(tiny):
    cfg, hf, mc = tiny
    back = ck.mcore_to_hf(mc, cfg)
    assert set(back) == set(hf)
    for k in hf:
        assert back[k].shape == hf[k].shape and torch.equal(back[k], hf[k]), k
    again = ck.hf_to_mcore(back, cfg)
    assert set(again) == set(mc) and all(torch.equal(again[k], mc[k]) for k in mc)


def test_vit_qkv_index_matches_the_scripts_loops():
    # hf2mcore_long_vita.py:397-414 written out as the script does: q rows of every head, then k, then v
    heads, hn = 16, 64
    idx = []
    for part in range(3):
        for i in range(heads):
            lb = i * hn * 3 + hn * part
            idx.append(torch.arange(lb, lb + hn))
    assert torch.equal(ck.vit_qkv_index(heads, hn), torch.cat(idx))


def test_llm_grouped_qkv_layout(tiny):
    cfg, hf, mc = tiny
    ng, np_, hn, H = cfg.num_key_value_heads, cfg.num_attention_heads, cfg.head_dim, cfg.hidden_size
    w = mc["decoder.layers.0.self_attention.linear_qkv.weight"]
    assert w.shape == ((np_ + 2 * ng) * hn, H)
    # independent statement of :488-498: view(ng, -1, hn, H), split [np/ng, 1, 1] along dim 1
    q, k, v = torch.split(w.view(ng, -1, hn, H), [np_ // ng, 1, 1], dim=1)
    assert torch.equal(q.reshape(-1, H), hf["model.layers.0.self_attn.q_proj.weight"])
    assert torch.equal(k.reshape(-1, H), hf["model.layers.0.self_attn.k_proj.weight"])
    assert torch.equal(v.reshape(-1, H), hf["model.layers.0.self_attn.v_proj.weight"])
    b = mc["decoder.layers.0.self_attention.linear_qkv.bias"].view(ng, -1)
    qb, kb, vb = torch.split(b, [H // ng, hn, hn], dim=1)                      # :495-498
    assert torch.equal(qb.reshape(-1), hf["model.layers.0.self_attn.q_proj.bias"])
    assert torch.equal(kb.reshape(-1), hf["model.layers.0.self_attn.k_proj.bias"])
    assert torch.equal(vb.reshape(-1), hf["model.layers.0.self_attn.v_proj.bias"])
    fc1 = mc["decoder.layers.0.mlp.linear_fc1.weight"]
    g, u = torch.split(fc1, cfg.intermediate_size)                             # :502-504
    assert torch.equal(g, hf["model.layers.0.mlp.gate_proj.weight"]) and torch.equal(u, hf["model.layers.0.mlp.up_proj.weight"])


def _inputs(cfg, s=300, n_img=1, seed=5):
    g = torch.Generator().manual_seed(seed)
    ids = torch.randint(0, cfg.vocab_size, (1, s), generator=g)
    images = torch.randn(n_img, 3, 448, 448, generator=g).to(torch.bfloat16)
    idx_s = torch.stack([torch.arange(7 + i * 270, 7 + i * 270 + 256) for i in range(n_img)])
    return ids, images, torch.stack([torch.zeros_like(idx_s), idx_s])


@pytest.fixture(scope="module")
def model(tiny):
    from long_vita_b200.megatron.gpt_vl_model import B200GPTVLModel

    cfg, hf, mc = tiny
    with oracle_ops():
        return B200GPTVLModel(cfg, mc)


def _oracle_logits(cfg, hf, ids, images, idx, rows):
    w32 = OM.cast_weights(hf, torch.float32)
    logits = OM.long_vita_forward(cfg, w32, ids, None if images is None else images.float(), idx)
    return logits[0][rows]


def test_forward_indices_mode_with_logit_mask(tiny, model):
    cfg, hf, _ = tiny
    ids, images, idx = _inputs(cfg)
    s = ids.shape[1]
    mask = torch.zeros(1, s, dtype=torch.bool)
    mask[0, [10, 299]] = True
    with oracle_ops():
        out = model(ids, torch.arange(s).unsqueeze(0), None, external_inputs={"images": images, "indices": idx},
                    logit_mask=mask)
    assert out.shape == (1, 2, cfg.vocab_size)                     # [b, M, vocab]
    ref = _oracle_logits(cfg, hf, ids, images, idx, [10, 299])
    assert rel_fro(out[0], ref) < 1.5e-2
    assert torch.equal(out[0].float().argmax(-1), ref.argmax(-1))


def test_pre_len_and_src_tgt_modes_equal_indices_mode(tiny, model):
    cfg, hf, _ = tiny
    ids, images, idx = _inputs(cfg)
    s = ids.shape[1]
    pos = torch.arange(s).unsqueeze(0)
    with oracle_ops():
        a = model(ids, pos, None, external_inputs={"images": images, "indices": idx})
        b = model(ids, pos, None, external_inputs={"images": images, "pre_len": 7})
        src = (torch.zeros(256, dtype=torch.long), torch.arange(256))
        tgt = (torch.zeros(256, dtype=torch.long), torch.arange(7, 7 + 256))
        c = model(ids, pos, None, external_inputs={"images": images, "src_indices": src, "tgt_indices": tgt})
        # a partial scatter (what a CP rank owning half of the image's tokens does) must differ
        d = model(ids, pos, None, external_inputs={"images": images, "src_indices": (src[0][:128], src[1][:128]),
                                                   "tgt_indices": (tgt[0][:128], tgt[1][:128])})
    assert a.shape == (1, s, cfg.vocab_size)
    assert torch.equal(a, b) and torch.equal(a, c)
    assert not torch.equal(a, d)
    assert torch.equal(a[0, :7], d[0, :7])                              # causal: rows before the image agree


def test_labels_give_per_token_loss_and_inference_params_override(tiny, model):
    cfg, hf, _ = tiny
    ids, images, idx = _inputs(cfg)
    s = ids.shape[1]
    pos = torch.arange(s).unsqueeze(0)
    mask = torch.zeros(1, s, dtype=torch.bool)
    mask[0, 280:] = True
    labels = torch.randint(0, cfg.vocab_size, (1, s), generator=torch.Generator().manual_seed(9))
    ip = types.SimpleNamespace(external_inputs={"images": images, "indices": idx}, key_value_memory_dict={},
                               logit_mask=mask, use_kv_cache=False)
    with oracle_ops():
        logits = model(ids, pos, None, inference_params=ip)            # both overrides come from inference_params
        loss = model(ids, pos, None, labels=labels, external_inputs={"images": images, "indices": idx}, logit_mask=mask)
    assert logits.shape == (1, 20, cfg.vocab_size)
    assert loss.shape == (1, 20) and loss.dtype == torch.float32
    ref = torch.nn.functional.cross_entropy(logits[0].float(), labels[0, 280:], reduction="none")
    # fused LM head + chunked cross-entropy: the same bf16 logits, the fp32 log-sum-exp summed chunk by chunk
    assert torch.allclose(loss[0], ref, rtol=1e-6, atol=1e-5)
    model.fused_loss = False                                            # the un-fused tail (logits materialised) is exact
    with oracle_ops():
        loss_u = model(ids, pos, None, labels=labels, external_inputs={"images": images, "indices": idx}, logit_mask=mask)
    model.fused_loss = True
    assert torch.allclose(loss_u[0], ref, rtol=0, atol=0)
    full = _oracle_logits(cfg, hf, ids, images, idx, slice(280, 300))
    assert rel_fro(logits[0], full) < 1.5e-2


def test_guards(tiny, model):
    cfg, _, _ = tiny
    ids = torch.zeros(1, 8, dtype=torch.long)
    pos = torch.arange(8).unsqueeze(0)
    with oracle_ops():
        with pytest.raises(AssertionError):
            model(ids, pos, None, packed_seq_params=object())
        with pytest.raises(AssertionError):
            model.embedding(ids, pos, {"features": torch.zeros(1, 256, cfg.hidden_size), "bogus": 1})


def test_product_path_still_refuses_cpu_tensors(tiny):
    """Outside the harness the wrappers are the real ones: no silent CPU fallback."""
    from long_vita_b200 import ops

    with pytest.raises(Exception):
        ops.rmsnorm(torch.zeros(4, 64, dtype=torch.bfloat16), torch.ones(64, dtype=torch.bfloat16))


def test_spec_layer_ungroups_megatron_weights(tiny):
    """B2 (`--spec` layer): TE state-dict names + Megatron's grouped QKV / cat(gate, up) layouts are
    re-ordered correctly - the layer equals the oracle decoder layer on the same (HF-layout) weights."""
    from long_vita_b200.megatron.transformer_layer import B200TransformerLayer
    from oracle import ops as O

    cfg, hf, mc = tiny
    mcfg = types.SimpleNamespace(hidden_size=cfg.hidden_size, num_attention_heads=cfg.num_attention_heads,
                                 num_query_groups=cfg.num_key_value_heads, kv_channels=cfg.head_dim,
                                 ffn_hidden_size=cfg.intermediate_size, layernorm_epsilon=cfg.rms_norm_eps,
                                 hidden_dropout=0.0, attention_dropout=0.0, params_dtype=torch.bfloat16)
    layer = B200TransformerLayer(mcfg, layer_number=1).cpu()       # built on the current GPU where there is one
    sd = {k[len("decoder.layers.0."):]: v for k, v in mc.items() if k.startswith("decoder.layers.0.")}
    missing, unexpected = layer.load_state_dict(sd, strict=True)
    assert not missing and not unexpected
    s = 192
    x = torch.randn(s, 1, cfg.hidden_size, generator=torch.Generator().manual_seed(4)).to(torch.bfloat16)
    inv = O.rope_inv_freq(cfg.head_dim, cfg.rope_theta)
    freqs = torch.outer(torch.arange(s).float(), inv)
    rotary = torch.cat((freqs, freqs), dim=-1).view(s, 1, 1, cfg.head_dim)       # Megatron's `freqs` tensor
    with oracle_ops():
        out, ctx = layer(hidden_states=x, attention_mask=None, context=None, context_mask=None, rotary_pos_emb=rotary,
                         inference_params=None, packed_seq_params=None)
    assert ctx is None and out.shape == (s, 1, cfg.hidden_size)
    cos, sin = O.rope_tables(torch.arange(s), inv, torch.float32)
    ref = OM.decoder_layer(cfg, OM.cast_weights(hf, torch.float32), 0, x[:, 0].float(), cos, sin)
    assert rel_fro(out[:, 0], ref) < 6e-3, rel_fro(out[:, 0], ref)
    # weights updated AFTER the first forward (load_state_dict / an optimizer step) must reach the re-ordered copies
    sd2 = {k_: (v * 0.5 if k_.endswith("linear_fc1.weight") else v) for k_, v in sd.items()}
    layer.load_state_dict(sd2, strict=True)
    hf2 = dict(hf)
    for n_ in ("gate_proj", "up_proj"):
        hf2[f"model.layers.0.mlp.{n_}.weight"] = hf[f"model.layers.0.mlp.{n_}.weight"] * 0.5
    with oracle_ops():
        out2, _ = layer(hidden_states=x, rotary_pos_emb=rotary)
    ref2 = OM.decoder_layer(cfg, OM.cast_weights(hf2, torch.float32), 0, x[:, 0].float(), cos, sin)
    assert rel_fro(out2[:, 0], ref2) < 6e-3 and not torch.equal(out2, out)
    with torch.no_grad():
        layer.self_attention.linear_qkv.bias.add_(0.25)          # in-place update: caught through the version counter
    with oracle_ops():
        out3, _ = layer(hidden_states=x, rotary_pos_emb=rotary)
    assert not torch.equal(out3, out2)
    # whole weights only
    with pytest.raises(NotImplementedError, match="tensor_model_parallel_size"):
        B200TransformerLayer(types.SimpleNamespace(**{**vars(mcfg), "tensor_model_parallel_size": 2}), layer_number=1)


# ------------------------------------------------------------------------------------------------
# context-parallel host logic, world_size 2 over gloo
# ------------------------------------------------------------------------------------------------
class _GlooCPContext:
    """Stand-in for cp.CPContext with the same two methods the layer uses: the K/V exchange is a gloo
    all-gather and the attention is the oracle with this rank's zig-zag query positions."""

    def __init__(self, S, hq, hkv, d):
        import torch.distributed as dist

        from long_vita_b200 import cp as CP

        self.dist, self.CP = dist, CP
        self.cp, self.rank = dist.get_world_size(), dist.get_rank()
        self.S, self.hq, self.hkv, self.d = S, hq, hkv, d
        self.T = S // self.cp
        self.buf = torch.empty(self.T, (hq + 2 * hkv) * d, dtype=torch.bfloat16)

    def qkv_buffer(self):
        return self.buf

    def check(self):
        """cp.CPContext.check reads the exchange's fault word; a gloo all-gather cannot time out silently."""

    def attention(self, out=None, scale=None):
        from oracle import ops as O

        hq, hkv, d, T = self.hq, self.hkv, self.d, self.T
        q = self.buf[:, : hq * d].view(T, hq, d)
        kv = self.buf[:, hq * d :].contiguous()
        parts = [torch.empty_like(kv) for _ in range(self.cp)]
        self.dist.all_gather(parts, kv)
        full = torch.empty(self.S, 2 * hkv * d, dtype=torch.bfloat16)
        for r in range(self.cp):
            full[self.CP.zigzag_index(self.S, self.cp, r)] = parts[r]
        k = full[:, : hkv * d].view(self.S, hkv, d)
        v = full[:, hkv * d :].view(self.S, hkv, d)
        o, _ = O.attention(q[None], k[None], v[None], causal=True, scale=scale,
                           q_pos=self.CP.zigzag_index(self.S, self.cp, self.rank), kv_pos=torch.arange(self.S))
        return o[0].to(torch.bfloat16).reshape(T, hq * d)


def _cp_worker(rank, world, port, tmp):
    import os

    import torch.distributed as dist

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from long_vita_b200 import cp as CP
        from long_vita_b200.megatron.gpt_vl_model import B200GPTVLModel
        from long_vita_b200.synthetic import build_prompt

        torch.set_num_threads(2)
        cfg = LongVITAConfig.tiny(layers=2, vit_layers=1)
        hf = synthetic_state_dict(cfg, seed=77, dtype=torch.bfloat16, perturb=True)
        mc = ck.hf_to_mcore(hf, cfg)
        ids, idx = build_prompt(cfg, 2, n_text=20, pad_multiple=2 * world * 128)
        S = ids.shape[1]
        images = torch.randn(2, 3, 448, 448, generator=torch.Generator().manual_seed(3)).to(torch.bfloat16)
        sh = CP.shard_prompt(ids, idx, world, rank, cfg.visual.tokens_per_image)
        with oracle_ops():
            model = B200GPTVLModel(cfg, mc, cp=_GlooCPContext(S, cfg.num_attention_heads, cfg.num_key_value_heads, cfg.head_dim))
            tpi = cfg.visual.tokens_per_image
            ext = {"images": images[sh.image_sel],
                   "src_indices": (sh.src_idx // tpi, sh.src_idx % tpi),
                   "tgt_indices": (torch.zeros_like(sh.dst_idx), sh.dst_idx)}
            local = model(sh.input_ids, sh.position_ids.unsqueeze(0), None, external_inputs=ext)     # [1, T, vocab]
        parts = [torch.empty_like(local) for _ in range(world)]
        dist.all_gather(parts, local)
        if rank == 0:
            full = torch.cat(parts, dim=1)[:, CP.zigzag_unpermute_index(S, world)]
            torch.save(full, tmp)
    finally:
        dist.destroy_process_group()


def test_two_rank_sharded_forward_equals_unsharded(tiny, model, tmp_path):
    import socket

    import torch.multiprocessing as mp

    from long_vita_b200.synthetic import build_prompt

    cfg, hf, _ = tiny
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    out = str(tmp_path / "sharded.pt")
    mp.spawn(_cp_worker, args=(2, port, out), nprocs=2, join=True)
    sharded = torch.load(out)
    ids, idx = build_prompt(cfg, 2, n_text=20, pad_multiple=2 * 2 * 128)
    images = torch.randn(2, 3, 448, 448, generator=torch.Generator().manual_seed(3)).to(torch.bfloat16)
    with oracle_ops():
        ref = model(ids, torch.arange(ids.shape[1]).unsqueeze(0), None, external_inputs={"images": images, "indices": idx})
    assert sharded.shape == ref.shape
    # identical operator sequence per token; only the attention's reduction order differs
    assert rel_fro(sharded, ref) < 2e-3, rel_fro(sharded, ref)
    assert (sharded[0].float().argmax(-1) == ref[0].float().argmax(-1)).float().mean() > 0.995


def test_masked_lm_head_with_an_empty_mask():
    """A context-parallel rank may own no answer token: the masked head then returns [0, b, vocab]."""
    h = torch.randn(16, 1, 64).to(torch.bfloat16)
    w = torch.randn(96, 64).to(torch.bfloat16)
    with oracle_ops() as ops:
        out = ops.masked_linear(h, w, torch.zeros(1, 16, dtype=torch.bool))
    assert out.shape == (0, 1, 96)


def test_embedding_modes_equal_the_references_own_embedding(tiny):
    """B200GPTVLModel.embedding (index translation to lv_embed_scatter's flat src / dst form) against committed
    outputs of the reference's own LanguageModelEmbedding.forward - bit-exact in all four modes."""
    import os
    import sys

    from long_vita_b200.megatron.gpt_vl_model import B200GPTVLModel

    gold_dir = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
    sys.path.insert(0, gold_dir)
    from make_golden import embedding_golden_inputs

    gold = torch.load(os.path.join(gold_dir, "ref_megatron_embedding.pt"))
    table, ids, feat, idx = embedding_golden_inputs()
    m = B200GPTVLModel.__new__(B200GPTVLModel)              # only the embedding path: no decoder weights needed
    m.word_embeddings = table
    pos = torch.arange(ids.shape[1]).unsqueeze(0)
    with oracle_ops():
        assert torch.equal(m.embedding(ids, pos), gold["none"][:, 0])
        assert torch.equal(m.embedding(ids, pos, {"features": feat, "indices": idx}), gold["indices"][:, 0])
        assert torch.equal(m.embedding(ids, pos, {"features": feat[:1], "pre_len": 5}), gold["pre_len"][:, 0])
        got = m.embedding(ids, pos, {"features": feat, "src_indices": gold["src"], "tgt_indices": gold["tgt"]})
        assert torch.equal(got, gold["src_tgt"][:, 0])


def test_masked_lm_head_forward_and_dgrad_equal_the_references_own_function():
    """ops.masked_linear / masked_linear_dgrad (gather -> GEMM, GEMM -> scatter-with-zeros; kernels replaced by the
    oracle) against committed outputs of the reference's own autograd function (layers.py:365-534)."""
    import os
    import sys

    gold_dir = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
    sys.path.insert(0, gold_dir)
    from make_golden import masked_linear_golden_inputs

    gold = torch.load(os.path.join(gold_dir, "ref_megatron_masked_linear.pt"))
    h, w, mask, dy = masked_linear_golden_inputs()
    bf = torch.bfloat16
    with oracle_ops() as ops:
        out = ops.masked_linear(h.to(bf), w.to(bf), mask)
        dx = ops.masked_linear_dgrad(dy.to(bf), w.to(bf), mask)
    assert out.shape == gold["out"].shape and rel_fro(out, gold["out"]) < 8e-3      # bf16 inputs vs the fp32 fixture
    assert dx.shape == gold["dx"].shape and rel_fro(dx, gold["dx"]) < 8e-3
    assert torch.equal(dx[:, 0].float().abs().sum(-1) == 0, gold["dx"][:, 0].abs().sum(-1) == 0)   # same zero rows


def test_checkpoint_layout_is_the_inverse_of_the_references_own_converter():
    """The reference's `convert_checkpoint_from_megatron_to_transformers` (tools/hf2mcore_long_vita.py:373-510) walks a
    Megatron-shaped module tree and fills the reference's own HF model; applied to `checkpoint.hf_to_mcore(hf)` it
    must give `hf` back, bit for bit - so our mcore names and row orders are exactly the ones the reference's converter
    reads.  The converter only copies, so a recorded run of it is its index map: run on a tree whose every element
    holds its own position in the concatenation of the mcore tensors (sorted by name; low and high digits in two runs,
    each exact in fp32), it fills each HF tensor with the positions it reads, stored as runs of consecutive positions.
    (The converter hard-codes the ViT geometry 1024 / 16 heads, so the vision tower has the real width here.)"""
    from dataclasses import replace

    base = LongVITAConfig.tiny(layers=2, vit_layers=1)
    cfg = replace(base, visual=replace(base.visual, hidden_size=1024, num_attention_heads=16, intermediate_size=64))
    hf = synthetic_state_dict(cfg, seed=404, dtype=torch.float32, perturb=True)
    mc = ck.hf_to_mcore(hf, cfg)
    names = sorted(mc)
    sizes = [mc[k].numel() for k in names]

    def run():
        from oracle import ref_loader

        args = types.SimpleNamespace(
            fp16=False, bf16=False, num_query_groups=cfg.num_key_value_heads, hidden_size=cfg.hidden_size,
            num_attention_heads=cfg.num_attention_heads, transformer_impl="transformer_engine", ffn_hidden_size=cfg.intermediate_size,
            untie_embeddings_and_output_weights=True,
            vit_args=types.SimpleNamespace(hidden_size=1024, num_query_groups=16, num_attention_heads=16))
        convert = ref_loader.load_checkpoint_converter()
        flat_pos = torch.arange(sum(sizes))

        def converted(digits):          # the converter applied to a tree holding `digits` of every position
            hfmodel = ref_loader.build_reference_long_vita(cfg, {k: torch.zeros_like(v) for k, v in hf.items()})
            mg = ref_loader.module_tree_from_state_dict(
                {k: t.to(torch.float32).view(mc[k].shape) for k, t in zip(names, digits.split(sizes))})
            convert(mg, hfmodel, args)  # asserts internally that every parameter was copied exactly once
            return hfmodel.state_dict()

        low, high = converted(flat_pos % 4096), converted(flat_pos // 4096)   # both exact in fp32
        runs = {}
        for k, t in low.items():
            p = high[k].reshape(-1).long() * 4096 + t.reshape(-1).long()
            starts = torch.cat([torch.zeros(1, dtype=torch.long), torch.nonzero(p[1:] != p[:-1] + 1).view(-1) + 1])
            lens = torch.diff(torch.cat([starts, torch.tensor([p.numel()])]))
            runs[k] = (tuple(t.shape), p[starts].clone(), lens)
        return {"names": names, "sizes": sizes, "runs": runs}

    rec = recorded("mcore_to_hf_converter", run)
    assert rec["names"] == names and rec["sizes"] == sizes
    flat = torch.cat([mc[k].reshape(-1) for k in names])
    assert set(rec["runs"]) == set(hf)
    for k, (shape, starts, lens) in rec["runs"].items():
        idx = torch.cat([torch.arange(a, a + n) for a, n in zip(starts.tolist(), lens.tolist())])
        assert torch.equal(flat[idx].view(shape), hf[k]), k


def test_forward_glue_equals_the_references_own_gptvl_forward(tiny, model):
    """The reference's `GPTVLModel.forward` (gpt_vl_model.py:233-416) executed on a stand-in `self` whose sub-modules
    are the reference's OWN LanguageModelEmbedding and RotaryEmbedding, plus this build's vision tower / decoder layers
    / output GEMM for the arithmetic in between.  Everything the two forwards do around those calls - external_inputs
    routing, the embedding merge, rotary table, logit_mask, labels masked_select, [s b h] -> [b s h] - must then agree
    bit for bit with B200GPTVLModel.forward.  The reference's outputs come from a recorded run: per-token losses as
    they are, logits as digests."""
    import os
    import socket

    import torch.distributed as dist

    cfg, hf, mc = tiny
    ids, images, idx = _inputs(cfg)
    s = ids.shape[1]
    args = types.SimpleNamespace(output_multiplier_scale=None, output_logit_softcapping=None, is_instruction_dataset=False)
    mask = torch.zeros(1, s, dtype=torch.bool)
    mask[0, 270:] = True
    labels = torch.randint(0, cfg.vocab_size, (1, s), generator=torch.Generator().manual_seed(1))
    pos = torch.arange(s).unsqueeze(0)
    ext = {"images": images, "indices": idx}
    ip = types.SimpleNamespace(external_inputs=ext, key_value_memory_dict={}, logit_mask=mask, use_kv_cache=False)
    cases = [dict(external_inputs=ext), dict(external_inputs=ext, logit_mask=mask), dict(inference_params=ip),
             dict(external_inputs=ext, logit_mask=mask, labels=labels), dict()]
    # the switches of the training tail (:352-369, :393-395): instruction-dataset shift, logit scale, soft-capping
    variants = [dict(is_instruction_dataset=True), dict(output_multiplier_scale=0.5), dict(output_logit_softcapping=30.0),
                dict(is_instruction_dataset=True, output_multiplier_scale=2.0, output_logit_softcapping=20.0)]
    variant_cases = [dict(external_inputs=ext, logit_mask=mask, labels=labels), dict(external_inputs=ext, logit_mask=mask)]

    def set_variant(variant, on):
        for k_, v_ in variant.items():
            v_ = v_ if on else (False if k_ == "is_instruction_dataset" else None)
            setattr(args, k_, v_)
            setattr(model, k_, v_)

    def keep(out, kw):
        return out.clone() if "labels" in kw else digest(out)

    def same(got, want, kw):
        return torch.equal(got, want) if "labels" in kw else digest(got) == want

    def run():
        from oracle import ref_loader

        ref_forward = ref_loader.load_class_methods(
            "long_vita_megatron/core/models/multimodal/gpt_vl_model.py", "GPTVLModel", {"forward"},
            namespace={"Tensor": torch.Tensor, "InferenceParams": object, "PackedSeqParams": object, "get_args": lambda: args,
                       "os": os})["forward"]
        emb_cls = ref_loader.load_megatron_embedding()
        ecfg = types.SimpleNamespace(hidden_size=cfg.hidden_size, hidden_dropout=0.0, fp32_residual_connection=False,
                                     sequence_parallel=False, init_method=lambda w: None, perform_initialization=False,
                                     clone_scatter_output_in_embedding=False)
        embedding = emb_cls(ecfg, vocab_size=cfg.vocab_size, max_sequence_length=4096, position_embedding_type="rope",
                            parallel_word_embedding=False).eval()
        embedding.word_embeddings.weight.data = model.word_embeddings.clone()
        rope_mod, cpu_placement = ref_loader.load_megatron_rope(1, 0)
        with cpu_placement():
            rotary = rope_mod.RotaryEmbedding(kv_channels=cfg.head_dim, rotary_percent=1.0, rotary_base=int(cfg.rope_theta))
        rotary.get_rotary_seq_len = lambda inference_params, decoder, decoder_input, config: decoder_input.shape[0]

        def decoder(hidden_states, attention_mask, inference_params, rotary_pos_emb, packed_seq_params):
            from long_vita_b200 import ops

            f = rotary_pos_emb.reshape(rotary_pos_emb.shape[0], -1)
            cos, sin = torch.cos(f).to(torch.bfloat16), torch.sin(f).to(torch.bfloat16)
            x, delta = hidden_states[:, 0], None
            for layer in model.layers:
                x, delta = layer.forward(x, delta, cos, sin, {})
            h, _ = ops.rmsnorm(delta, model.final_layernorm, cfg.rms_norm_eps, residual=x)
            return h.unsqueeze(1)

        def output_layer(hidden_states, weight=None, logit_mask=None):
            from long_vita_b200 import ops

            if logit_mask is None:
                return ops.linear(hidden_states, model.output_weight), None
            sel = torch.masked_select(hidden_states, logit_mask.transpose(0, 1).unsqueeze(2)).reshape(-1, 1, hidden_states.shape[2])
            return ops.linear(sel, model.output_weight), None        # same rows the reference's masked linear selects

        def loss_fn(labels, logits):
            lg = logits.float().transpose(0, 1)
            return torch.nn.functional.cross_entropy(lg.reshape(-1, lg.shape[-1]), labels.reshape(-1), reduction="none").view(labels.shape)

        me = types.SimpleNamespace(
            pre_process=True, post_process=True, external_feature_model=lambda **kw: model.external_feature_model(**kw),
            embedding=embedding, position_embedding_type="rope", rotary_pos_emb=rotary, decoder=decoder, config=None,
            unused=torch.zeros(cfg.hidden_size, dtype=torch.bfloat16), share_embeddings_and_output_weights=False,
            output_layer=output_layer, compute_language_model_loss=loss_fn)
        out = {"cases": [], "variants": []}
        with cpu_placement():
            out["cases"] = [keep(ref_forward(me, ids, pos, None, **kw), kw) for kw in cases]
            for variant in variants:
                set_variant(variant, True)
                try:
                    out["variants"].append([keep(ref_forward(me, ids, pos, None, **kw), kw) for kw in variant_cases])
                finally:
                    set_variant(variant, False)
        return out

    with socket.socket() as sock:
        sock.bind(("127.0.0.1", 0))
        port = sock.getsockname()[1]
    dist.init_process_group("gloo", rank=0, world_size=1, init_method=f"tcp://127.0.0.1:{port}")   # forward asks get_rank()
    try:
        with oracle_ops():
            rec = recorded("gptvl_forward", run)
            assert len(rec["cases"]) == len(cases) and len(rec["variants"]) == len(variants)
            for kw, want in zip(cases, rec["cases"]):
                got = model(ids, pos, None, **kw)
                if "labels" in kw:
                    # fused LM head + chunked cross-entropy (8f-3): same bf16 logits, fp32 log-sum-exp summed per chunk
                    assert got.shape == want.shape and torch.allclose(got, want, rtol=1e-6, atol=1e-5), sorted(kw)
                    model.fused_loss = False        # the un-fused tail reproduces the reference's glue bit for bit
                    got = model(ids, pos, None, **kw)
                    model.fused_loss = True
                assert same(got, want, kw), sorted(kw)
            for variant, wants in zip(variants, rec["variants"]):
                set_variant(variant, True)
                try:
                    for kw, want in zip(variant_cases, wants):
                        got = model(ids, pos, None, **kw)
                        if "labels" in kw:
                            assert got.shape == want.shape, (variant, sorted(kw))
                        if "labels" in kw and set(variant) == {"is_instruction_dataset"}:      # the fused tail takes this one
                            assert torch.allclose(got, want, rtol=1e-6, atol=1e-5), variant
                            model.fused_loss = False
                            got = model(ids, pos, None, **kw)
                            model.fused_loss = True
                        assert same(got, want, kw), (variant, sorted(kw))
                finally:
                    set_variant(variant, False)
    finally:
        dist.destroy_process_group()


def test_masked_lm_head_autograd_matches_reference_formulas():
    """a12: dX = masked_scatter(zeros, dY W), dW = dY^T sel (layers.py:443-456) through the product's own
    composition (gather / padded transposes / scatter), kernels replaced by the oracle."""
    from oracle import ops as O

    g = torch.Generator().manual_seed(8)
    s, c, vocab = 40, 64, 96
    h = torch.randn(s, 1, c, generator=g).to(torch.bfloat16).requires_grad_(True)
    w = (torch.randn(vocab, c, generator=g) * 0.1).to(torch.bfloat16).requires_grad_(True)
    mask = torch.zeros(1, s, dtype=torch.bool)
    mask[0, [3, 4, 17, 30, 39]] = True                          # M = 5: exercises the zero padding to 8
    dy = torch.randn(5, 1, vocab, generator=g).to(torch.bfloat16)
    with oracle_ops() as ops:
        out = ops.masked_linear_autograd(h, w, mask)
        out.backward(dy)
        empty = ops.masked_linear_autograd(h.detach().requires_grad_(True), w.detach(), torch.zeros(1, s, dtype=torch.bool))
        assert empty.shape == (0, 1, vocab)
    ref_out = O.masked_linear_fwd(h.detach().float(), w.detach().float(), mask)
    gx, gw = O.masked_linear_bwd(dy.float(), h.detach().float(), w.detach().float(), mask)
    assert rel_fro(out, ref_out) < 5e-3
    assert rel_fro(h.grad, gx) < 5e-3 and rel_fro(w.grad, gw) < 5e-3
    unmasked = torch.ones(s, dtype=torch.bool)
    unmasked[[3, 4, 17, 30, 39]] = False
    assert not h.grad[unmasked].any()                           # rows outside the mask get exactly zero


def _cp_decode_worker(rank, world, port, tmp):
    import os

    import torch.distributed as dist

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from long_vita_b200 import cp as CP
        from long_vita_b200.hf.modeling import LongVITAForCausalLM
        from long_vita_b200.synthetic import build_prompt

        torch.set_num_threads(2)
        cfg = LongVITAConfig.tiny(layers=2, vit_layers=1)
        hf = synthetic_state_dict(cfg, seed=77, dtype=torch.bfloat16, perturb=True)
        ids, idx = build_prompt(cfg, 1, n_text=20, pad_multiple=2 * world * 128)
        S = ids.shape[1]
        images = torch.randn(1, 3, 448, 448, generator=torch.Generator().manual_seed(3)).to(torch.bfloat16)
        new = torch.randint(0, cfg.vocab_size, (3,), generator=torch.Generator().manual_seed(4))
        with oracle_ops():
            model = LongVITAForCausalLM(cfg, hf)
            runner = CP.ContextParallelRunner(model, dist.group.WORLD)
            runner.ctx = _GlooCPContext(S, cfg.num_attention_heads, cfg.num_key_value_heads, cfg.head_dim)
            first = runner.forward(ids, images, idx, use_cache=True, max_new_tokens=8)
            assert len(runner.cache) == S // world and runner.total_len == S
            steps = [runner.decode(new[i]) for i in range(3)]
            # rows went round-robin to rank (S + i) % world
            assert len(runner.cache) == S // world + sum(1 for i in range(3) if (S + i) % world == rank)
        if rank == 0:
            torch.save({"first": first, "steps": torch.cat(steps, dim=1)}, tmp)
    finally:
        dist.destroy_process_group()


def test_two_rank_sharded_cache_decode_equals_full_forward(tiny, tmp_path):
    import socket

    import torch.multiprocessing as mp

    from long_vita_b200.hf.modeling import LongVITAForCausalLM
    from long_vita_b200.synthetic import build_prompt

    cfg, hf, _ = tiny
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    out = str(tmp_path / "decode.pt")
    mp.spawn(_cp_decode_worker, args=(2, port, out), nprocs=2, join=True)
    got = torch.load(out)
    ids, idx = build_prompt(cfg, 1, n_text=20, pad_multiple=2 * 2 * 128)
    images = torch.randn(1, 3, 448, 448, generator=torch.Generator().manual_seed(3)).to(torch.bfloat16)
    new = torch.randint(0, cfg.vocab_size, (3,), generator=torch.Generator().manual_seed(4))
    with oracle_ops():
        full = LongVITAForCausalLM(cfg, hf)(input_ids=torch.cat([ids, new.view(1, 3)], dim=1), images=images,
                                           image_indices=idx).logits
    S = ids.shape[1]
    assert rel_fro(got["first"][0, 0], full[0, S - 1]) < 1e-2
    for i in range(3):     # decode step i consumed new[i] at position S + i
        assert rel_fro(got["steps"][0, i], full[0, S + i]) < 1.5e-2, (i, rel_fro(got["steps"][0, i], full[0, S + i]))
        assert int(got["steps"][0, i].float().argmax()) == int(full[0, S + i].float().argmax())


def test_megatron_kv_cache_protocol_matches_full_forward(tiny, model):
    """Megatron's `--use-kv-cache` loop (generation.py:127-131): the first call carries the prompt and the external
    inputs, later calls only the new tokens and their positions, all sharing one `inference_params`.  The logits
    of every step must equal the full forward over the extended sequence."""
    cfg, hf, _ = tiny
    ids, images, idx = _inputs(cfg)
    s = ids.shape[1]
    new = torch.randint(0, cfg.vocab_size, (1, 3), generator=torch.Generator().manual_seed(12))
    ext = {"images": images, "indices": idx}
    ip = types.SimpleNamespace(external_inputs=ext, key_value_memory_dict={}, logit_mask=None, use_kv_cache=True,
                               max_sequence_length=s + 8)
    with oracle_ops():
        full = model(torch.cat([ids, new], dim=1), torch.arange(s + 3).unsqueeze(0), None, external_inputs=ext)
        first = model(ids, torch.arange(s).unsqueeze(0), None, inference_params=ip)
        cache = ip.key_value_memory_dict["b200_kv_cache"]
        assert len(cache) == s and cache.capacity == s + 8
        assert rel_fro(first[0], full[0, :s]) < 1e-6 or torch.equal(first[0], full[0, :s])
        for i in range(3):
            step = model(new[:, i : i + 1], torch.tensor([[s + i]]), None, inference_params=ip)   # external inputs ignored now
            assert step.shape == (1, 1, cfg.vocab_size) and len(cache) == s + i + 1
            assert rel_fro(step[0, 0], full[0, s + i]) < 1e-2, i
            assert int(step[0, 0].float().argmax()) == int(full[0, s + i].float().argmax())


def test_spec_layer_trains_gradients_match_oracle_autograd(tiny):
    """B2 training path (`_forward_train`): every gradient - input and all seven Megatron-layout parameters - against
    fp32 autograd through the oracle decoder layer on the same weights.  Kernels (forward and backward) are replaced by
    the oracle / torch-autograd formulas here; what is tested is the autograd wiring, the transposed-operand GEMM
    composition for dX / dW, the grouped-QKV slicing and the residual bookkeeping."""
    from long_vita_b200.megatron.transformer_layer import B200TransformerLayer
    from oracle import ops as O

    cfg, hf, mc = tiny
    mcfg = types.SimpleNamespace(hidden_size=cfg.hidden_size, num_attention_heads=cfg.num_attention_heads,
                                 num_query_groups=cfg.num_key_value_heads, kv_channels=cfg.head_dim,
                                 ffn_hidden_size=cfg.intermediate_size, layernorm_epsilon=cfg.rms_norm_eps,
                                 hidden_dropout=0.0, attention_dropout=0.0, params_dtype=torch.bfloat16)
    layer = B200TransformerLayer(mcfg, layer_number=1).cpu()       # built on the current GPU where there is one
    sd = {k[len("decoder.layers.0."):]: v for k, v in mc.items() if k.startswith("decoder.layers.0.")}
    layer.load_state_dict(sd, strict=True)
    for prm in layer.parameters():
        prm.requires_grad_(True)
    s = 160
    g = torch.Generator().manual_seed(21)
    x = torch.randn(s, 1, cfg.hidden_size, generator=g).to(torch.bfloat16).requires_grad_(True)
    dout = (torch.randn(s, 1, cfg.hidden_size, generator=g) * 0.1).to(torch.bfloat16)
    inv = O.rope_inv_freq(cfg.head_dim, cfg.rope_theta)
    freqs = torch.outer(torch.arange(s).float(), inv)
    rotary = torch.cat((freqs, freqs), dim=-1).view(s, 1, 1, cfg.head_dim)
    with oracle_ops():
        out, _ = layer(hidden_states=x, attention_mask=None, rotary_pos_emb=rotary)
        out.backward(dout)
    # fp32 autograd through the oracle layer (HF layout weights)
    w32 = {k: v.float().requires_grad_(True) for k, v in hf.items() if k.startswith("model.layers.0.")}
    xr = x.detach().float()[:, 0].requires_grad_(True)
    cos, sin = O.rope_tables(torch.arange(s), inv, torch.float32)
    ref = OM.decoder_layer(cfg, w32, 0, xr, cos, sin)
    ref.backward(dout.float()[:, 0])
    assert rel_fro(out[:, 0], ref.detach()) < 8e-3
    assert rel_fro(x.grad[:, 0], xr.grad) < 2e-2, rel_fro(x.grad[:, 0], xr.grad)
    # parameter gradients, translated to the Megatron layouts by the (linear, bit-exact) checkpoint re-layout
    ref_mc = ck.hf_to_mcore({k: v.grad for k, v in w32.items()}, cfg)
    for name, prm in layer.named_parameters():
        want = ref_mc["decoder.layers.0." + name]
        assert prm.grad is not None and prm.grad.shape == want.shape, name
        assert rel_fro(prm.grad, want) < 3e-2, (name, rel_fro(prm.grad, want))


def test_fused_masked_lm_head_cross_entropy_host_logic():
    """SURVEY.md 8f-3 host logic on CPU: the chunked LM-head + cross-entropy composition (chunk loop, running softmax
    statistics, gradient chunks, scatter of dX) equals cross_entropy over the materialised logits and its autograd."""
    from long_vita_b200 import ops

    g = torch.Generator().manual_seed(12)
    s, c, V = 40, 64, 200          # 200 = 3 chunks of 64 + a ragged 8
    h = (torch.randn(s, 1, c, generator=g)).to(torch.bfloat16).requires_grad_(True)
    w = (torch.randn(V, c, generator=g) * 0.2).to(torch.bfloat16).requires_grad_(True)
    mask = torch.rand(1, s, generator=g) < 0.4
    M = int(mask.sum())
    labels = torch.randint(0, V, (1, M), generator=g)
    up = torch.randn(1, M, generator=g)
    with oracle_ops():
        loss = ops.masked_lm_head_ce(h, w, mask, labels, vocab_chunk=64)
        loss.backward(up)
    hf, wf = h.detach().float().requires_grad_(True), w.detach().float().requires_grad_(True)
    logits = (hf[mask[0]][:, 0] @ wf.t()).to(torch.bfloat16).float()      # bf16 logits, fp32 loss (the reference's dtypes)
    ref = torch.nn.functional.cross_entropy(logits, labels[0], reduction="none")
    assert loss.shape == (1, M) and loss.dtype == torch.float32
    assert torch.allclose(loss[0], ref, rtol=1e-5, atol=1e-5)
    ref32 = torch.nn.functional.cross_entropy(hf[mask[0]][:, 0] @ wf.t(), labels[0], reduction="none")
    ref32.backward(up[0])
    assert rel_fro(h.grad, hf.grad) < 1e-2 and rel_fro(w.grad, wf.grad) < 1e-2
    assert torch.equal(h.grad[~mask[0]], torch.zeros_like(h.grad[~mask[0]]))           # masked_scatter into zeros
    # ignored rows (negative label): zero loss, zero gradient
    with oracle_ops():
        l2, lse = ops.lm_head_ce_fwd(h.detach()[mask[0]][:, 0], w.detach(), torch.cat([labels[0, :-1], torch.tensor([-1])]), 64)
    assert float(l2[-1]) == 0.0 and torch.allclose(l2[:-1], ref[:-1], rtol=1e-5, atol=1e-5)

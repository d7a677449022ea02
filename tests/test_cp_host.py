"""Host-side context-parallel logic on CPU: zig-zag sharding, image routing and scatter-index
translation (training/utils.py:252-343), checked single-process for cp in {2,4,8} and through a
world_size-2 gloo run (every rank shards the same prompt, the shards are all-gathered, un-permuted
and compared with the unsharded oracle)."""
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from long_vita_b200 import cp as CP
from long_vita_b200.config import LongVITAConfig
from long_vita_b200.synthetic import build_prompt
from oracle import ops as O


def _prompt(n_frames=6, cp=4):
    cfg = LongVITAConfig.tiny()
    ids, idx = build_prompt(cfg, n_frames, n_text=40, pad_multiple=2 * cp * 128)
    return cfg, ids, idx


@pytest.mark.parametrize("cp", [2, 4, 8])
def test_zigzag_index_matches_oracle_and_reference_formula(cp):
    S = 2 * cp * 96
    for r in range(cp):
        own = CP.zigzag_index(S, cp, r)
        assert torch.equal(own, O.zigzag_positions(S, cp, r))
        ref = torch.arange(S).view(2 * cp, S // (2 * cp))[[r, 2 * cp - 1 - r]].view(-1)   # utils.py:279
        assert torch.equal(own, ref)
    inv = CP.zigzag_unpermute_index(S, cp)
    cat = torch.cat([CP.zigzag_index(S, cp, r) for r in range(cp)])
    assert torch.equal(cat[inv], torch.arange(S))


@pytest.mark.parametrize("cp", [2, 4, 8])
def test_shard_prompt_reproduces_unsharded_embedding(cp):
    cfg, ids, idx = _prompt(7, cp)
    S = ids.shape[1]
    H = 16
    g = torch.Generator().manual_seed(0)
    table = torch.randn(cfg.vocab_size, H, generator=g)
    feat = torch.randn(idx.shape[1], 256, H, generator=g)
    full = O.embed_scatter(ids.view(-1), table, feat, idx[1].reshape(-1))
    parts = []
    seen_images = set()
    for r in range(cp):
        sh = CP.shard_prompt(ids, idx, cp, r, 256)
        assert torch.equal(sh.position_ids, CP.zigzag_index(S, cp, r))
        local_feat = feat[sh.image_sel]
        parts.append(O.embed_scatter(sh.input_ids.view(-1), table, local_feat, sh.dst_idx, sh.src_idx))
        seen_images.update(sh.image_sel.tolist())
        # the reference's formulation of the same selection (utils.py:279-289)
        calib = CP.zigzag_index(S, cp, r)
        sel_ref = torch.isin(idx[1], calib).any(dim=1).nonzero().view(-1)
        assert torch.equal(sh.image_sel, sel_ref)
        assert (sh.last_token_local >= 0) == (r == 0)
    assert seen_images == set(range(idx.shape[1]))
    cat = torch.cat(parts)
    assert torch.equal(cat[CP.zigzag_unpermute_index(S, cp)], full)


def _worker(rank, world, port):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        cfg, ids, idx = _prompt(5, world)
        S = ids.shape[1]
        sh = CP.shard_prompt(ids, idx, world, rank, 256)
        # "forward": a token-wise function of (id, position) so that the un-permuted gather is checkable
        local = (sh.input_ids.view(-1) * 3 + sh.position_ids).to(torch.int64)
        gathered = [torch.empty_like(local) for _ in range(world)]
        dist.all_gather(gathered, local)
        full = torch.cat(gathered)[CP.zigzag_unpermute_index(S, world)]
        assert torch.equal(full, ids.view(-1) * 3 + torch.arange(S))
        # CP loss all-reduce pattern (pretrain_long_vita.py:802-803): [loss_sum, n_tok]
        t = torch.tensor([float(local.sum()), float(local.numel())], dtype=torch.float64)
        dist.all_reduce(t)
        assert t[1].item() == S and t[0].item() == float((ids.view(-1) * 3 + torch.arange(S)).sum())
    finally:
        dist.destroy_process_group()


def test_two_rank_gloo_shard_gather_roundtrip():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    mp.spawn(_worker, args=(2, port), nprocs=2, join=True)   # a failed assert in a worker re-raises here


def test_shard_prompt_equals_the_references_own_get_batch_on_this_cp_rank():
    """cp.shard_prompt against committed outputs of the reference's own function (training/utils.py:252-343,
    executed from /root/reference by tests/golden/make_golden.py with Megatron's imports stubbed and device
    placement redirected to the CPU): token and position slices, kept images, (src, tgt) scatter indices -
    bit-exact for cp in {2, 4} and every rank."""
    import sys

    gold_dir = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
    sys.path.insert(0, gold_dir)
    from make_golden import cp_golden_prompt

    gold = torch.load(os.path.join(gold_dir, "ref_cp_shards.pt"))
    ids, idx = cp_golden_prompt()
    assert ids.shape[1] == gold["S"] and idx.shape[1] == gold["n_frames"]
    checked = 0
    for (cp, r), b in gold["shards"].items():
        sh = CP.shard_prompt(ids, idx, cp, r, 256)
        assert torch.equal(sh.input_ids, b["tokens"])
        assert torch.equal(sh.position_ids, b["position_ids"][0])
        assert "external_indices" not in b                       # consumed by the reference function
        if "external_src_indices" in b:
            src_b, src_s = b["external_src_indices"]
            tgt_b, tgt_s = b["external_tgt_indices"]
            assert torch.equal(sh.image_sel, b["external_images"].view(-1))
            assert torch.equal(sh.src_idx, src_b * 256 + src_s)
            assert not tgt_b.any() and torch.equal(sh.dst_idx, tgt_s)
            checked += 1
        else:                                                    # no image token on this rank
            assert sh.image_sel.numel() == 0 and sh.dst_idx.numel() == 0
    assert checked >= 5
    a, b, want = gold["index_of_a_in_b"]
    assert torch.equal(O.index_of_a_in_b(a, b), want)


def _sync_worker(rank, world, port):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from oracle import ref_loader
        from tests.util import digest, recorded

        cfg, ids, idx = _prompt(5, world)
        S = ids.shape[1]
        sh = CP.shard_prompt(ids, idx, world, rank, 256)
        # per-token "logits" [b, s_local, 3] of this rank's shard, as forward_step hands them to sync_output
        local = torch.stack([sh.input_ids[0].float(), sh.position_ids.float(), sh.position_ids.float() * 2], dim=-1).unsqueeze(0)

        def run():
            return digest(ref_loader.load_megatron_generation(world, rank, dist.group.WORLD).sync_output(local))

        full = recorded(f"sync_output_cp{world}", run, store=rank == 0)      # every rank receives the same sequence
        pos = torch.arange(S).float()
        assert full == digest(torch.stack([ids[0].float(), pos, pos * 2], dim=-1).unsqueeze(0))   # global order restored
        # ... which is what zigzag_unpermute_index does with a plain concatenation of the shards
        gathered = [torch.empty_like(local) for _ in range(world)]
        dist.all_gather(gathered, local)
        assert digest(torch.cat(gathered, dim=1)[:, CP.zigzag_unpermute_index(S, world)]) == full
    finally:
        dist.destroy_process_group()


def test_references_own_sync_output_restores_global_order_from_our_shards():
    """2 ranks over gloo: the reference's inference-side gather (generation.py:542-566; a recorded run of it) applied
    to the shards cp.shard_prompt produced returns the sequence in global order, and equals
    cp.zigzag_unpermute_index on the concatenated shards."""
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    mp.spawn(_sync_worker, args=(2, port), nprocs=2, join=True)


# ---- key-tile visiting order of the fused exchange kernel (csrc/attn_fwd.cu: KvWalk, cp_copier) ----
def _order_list(cp, rank, ring):
    """`k.order` as lv_attn_cp_fwd builds it: 2 cp chunk ids, own chunks first then peers by ring distance (ring) or 0..2cp-1."""
    out = []
    for i in range(cp):
        peer = (rank - i + cp) % cp if ring else i
        out += [peer, 2 * cp - 1 - peer] if ring else [2 * i, 2 * i + 1]
    return out


def _walk(n0, n1, order, tc):
    """KvWalk: the tiles [0, lo) both query tiles see first, then [lo, hi), each range in chunk-priority order."""
    lo, hi = min(n0, n1), max(n0, n1)
    seq = []
    for a, b in ((0, lo), (lo, hi)):
        for ch in order:
            seq += list(range(max(a, ch * tc), min(b, (ch + 1) * tc)))
    return seq


def _copier_blocks(nb, order, tc):
    """cp_copier: the i-th staged block in chunk-priority order."""
    out = []
    for i in range(nb):
        j = i
        for ch in order:
            cnt = min(max(nb - ch * tc, 0), tc)
            if j < cnt:
                out.append(ch * tc + j)
                break
            j -= cnt
    return out


def test_visiting_order_model_of_the_exchange_kernel():
    """A restatement of the kernel's index logic (not the kernel - its parity is tests/test_gpu_cp.py): every key tile a
    query tile may see is visited exactly once, the shorter query tile takes part in a PREFIX of the steps, the copier
    stages every needed block once, and in ring order the first blocks are the rank's own."""
    import random

    rnd = random.Random(0)
    for cp in (2, 4, 8):
        for tc in (1, 3, 9):
            for rank in range(cp):
                for ring in (False, True):
                    order = _order_list(cp, rank, ring)
                    assert sorted(order) == list(range(2 * cp))
                    nb = (2 * cp - rank) * tc                      # blocks this rank's queries can see
                    staged = _copier_blocks(nb, order, tc)
                    assert sorted(staged) == list(range(nb))
                    if ring:
                        assert set(staged[:tc]) == set(range(rank * tc, (rank + 1) * tc))     # own first chunk first
                    else:
                        assert staged == list(range(nb))
                    for _ in range(25):
                        n1 = rnd.randint(0, nb)
                        n0 = rnd.randint(0, n1)
                        if rnd.random() < 0.2:
                            n0, n1 = n1, 0                          # second query tile out of range
                        seq = _walk(n0, n1, order, tc)
                        assert sorted(seq) == list(range(max(n0, n1)))
                        assert sorted(seq[: min(n0, n1)]) == list(range(min(n0, n1)))
                        if not ring:
                            assert seq == list(range(max(n0, n1)))  # global order: what the single-device kernel does


def test_shared_context_cache_is_bounded_and_evicts_least_recently_used():
    """CPContext.shared keeps at most MAX_SHARED geometries alive and closes the least recently used one (every rank makes
    the same calls in the same order, so the collective close() lines up).  The peer-mapped buffers need GPUs, so the
    bookkeeping is exercised on a subclass whose constructor / close only record what happened."""
    from long_vita_b200.cp import CPContext

    events = []

    class Fake(CPContext):
        _shared = {}

        def __init__(self, group, seq_total, hq, hkv, d, device, fused_qkv=True):
            self.S = seq_total
            events.append(("open", seq_total))

        def close(self):
            events.append(("close", self.S))

    a = Fake.shared(None, 1024, 8, 2, 64, "cpu")
    b = Fake.shared(None, 2048, 8, 2, 64, "cpu")
    assert Fake.shared(None, 1024, 8, 2, 64, "cpu") is a            # hit: no new buffers, 1024 becomes most recent
    c = Fake.shared(None, 4096, 8, 2, 64, "cpu")                      # third geometry: evicts 2048, not 1024
    assert events == [("open", 1024), ("open", 2048), ("close", 2048), ("open", 4096)]      # closed BEFORE the new one opens
    assert Fake.shared(None, 1024, 8, 2, 64, "cpu") is a and Fake.shared(None, 4096, 8, 2, 64, "cpu") is c
    assert len(Fake._shared) == Fake.MAX_SHARED == 2
    assert Fake.shared(None, 2048, 8, 2, 64, "cpu") is not b        # was closed: a fresh context
    assert Fake.shared(None, 1024, 8, 2, 64, "cpu", fused_qkv=False) is not a     # the layout is part of the key

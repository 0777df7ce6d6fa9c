"""CPU: the host side of the per-hit detail — proposal windows, frame windows of a key clip (engine.moment_frames),
and the detail moving with its hit through the shard exchange (world size 2 and 3 over gloo, numpy stand-in for the
payload merge kernel, which is checked on the GPU in tests/test_gpu_detail.py)."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import oracle as O


@pytest.mark.parametrize("T", [32, 16, 12, 8])
def test_proposal_window_inverts_proposal_index(dkd, T):
    from dkd_b200 import ops
    P = ops.num_proposals(T)
    seen = set()
    for p in range(P):
        w, s = ops.proposal_window(p, T)
        assert 1 <= w <= T and 0 <= s <= T - w
        assert ops.proposal_index(w, s, T) == p
        seen.add((w, s))
    assert len(seen) == P
    with pytest.raises(ValueError):
        ops.proposal_window(P, T)


@pytest.mark.parametrize("T", [32, 12])
def test_moment_frames_is_the_support_of_the_window(dkd, T):
    """For every length 1..128 and every proposal: feed one-hot frames through the reference's own averaging
    (oracle.downsample_clips + oracle.build_proposals); the frames with a non-zero weight in the proposal are exactly
    moment_frames' [first, end)."""
    from dkd_b200 import engine, ops
    P = ops.num_proposals(T)
    Lmax = 128
    lengths = torch.arange(1, Lmax + 1, dtype=torch.int32)
    arg = torch.arange(P, dtype=torch.int32).view(1, P, 1).expand(Lmax, P, 1).contiguous()
    ids = torch.arange(Lmax, dtype=torch.int32).view(Lmax, 1).expand(Lmax, P).contiguous()
    win = engine.moment_frames(arg, ids, lengths, T=T)
    assert win.shape == (Lmax, P, 1, 2) and win.dtype == torch.int32
    for n in range(1, Lmax + 1):
        eye = torch.eye(n).unsqueeze(0)                                    # (1, n frames, n features): one-hot
        props = O.build_proposals(O.downsample_clips(eye, torch.tensor([n]), T))[0]   # (P, n)
        support = props != 0
        f, e = win[n - 1, :, 0, 0].long(), win[n - 1, :, 0, 1].long()
        col = torch.arange(n)[None]
        assert torch.equal(support, (col >= f[:, None]) & (col < e[:, None])), f"length {n}"


def test_moment_frames_frame_head_and_padding(dkd):
    from dkd_b200 import engine
    arg = torch.tensor([[[3, 0], [7, 2]], [[-1, -1], [5, 1]]], dtype=torch.int32)
    ids = torch.tensor([[0, 1], [-1, 1]], dtype=torch.int32)
    lengths = torch.tensor([10, 12], dtype=torch.int32)
    w = engine.moment_frames(arg, ids, lengths, head="frame")
    assert w[0, 0].tolist() == [[3, 4], [0, 1]] and w[1, 1].tolist() == [[5, 6], [1, 2]]
    assert (w[1, 0] == -1).all()
    w2 = engine.moment_frames(arg, ids, lengths)
    assert (w2[1, 0] == -1).all() and (w2[0] >= 0).all()


def test_hit_detail_pack_roundtrip(dkd):
    from dkd_b200 import engine
    g = torch.Generator().manual_seed(0)
    for two in (True, False):
        for nb in (1, 2):
            d = engine.HitDetail(arg=torch.randint(0, 528, (5, 7, nb), generator=g, dtype=torch.int32),
                                 score=torch.randn(5, 7, nb, generator=g),
                                 frame=torch.randn(5, 7, nb, generator=g) if two else None)
            w = d.pack()
            assert w.shape == (5, 7, nb * (3 if two else 2)) and w.dtype == torch.int32
            e = engine.HitDetail.unpack(w, nb, two)
            assert torch.equal(e.arg, d.arg) and torch.equal(e.score, d.score)
            assert (e.frame is None) if not two else torch.equal(e.frame, d.frame)
            p = engine.HitDetail.padding(2, 3, nb, two)
            assert (p.arg == -1).all() and torch.isneginf(p.score).all()
            assert (p.frame is None) if not two else torch.isneginf(p.frame).all()


# ---------------------------------------------------------------------------------------- gloo exchange with detail
def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _np_merge_payload(gs, gi, gw):
    """(G, M, K) lists + (G, M, K, C) words -> (M, K) + (M, K, C): stand-in for dkd_merge_topk_payload."""
    G, M, K = gs.shape
    C = gw.shape[-1]
    s = gs.permute(1, 0, 2).reshape(M, G * K).numpy()
    i = gi.permute(1, 0, 2).reshape(M, G * K).numpy()
    w = gw.permute(1, 0, 2, 3).reshape(M, G * K, C).numpy()
    out_s = np.full((M, K), -np.inf, np.float32)
    out_i = np.full((M, K), -1, np.int32)
    out_w = np.full((M, K, C), -1, np.int32)
    for m in range(M):
        keep = i[m] >= 0
        order = np.lexsort((i[m][keep], -s[m][keep]))[:K]
        out_s[m, : len(order)] = s[m][keep][order]
        out_i[m, : len(order)] = i[m][keep][order]
        out_w[m, : len(order)] = w[m][keep][order]
    return torch.from_numpy(out_s), torch.from_numpy(out_i), torch.from_numpy(out_w)


def _detail_of(ids, m_idx, two):
    """A detail that is a known function of (query, video id): the merge must keep it with its hit."""
    from dkd_b200 import engine
    v = ids.long()
    arg = torch.stack([(v * 7 + m_idx * 3) % 528, (v * 5 + m_idx) % 528], -1).to(torch.int32)
    score = torch.stack([v * 0.25 + m_idx, -v * 0.5 - m_idx], -1).float()
    frame = torch.stack([v * 0.125 - m_idx, v * 1.5 + m_idx], -1).float() if two else None
    d = engine.HitDetail(arg=arg, score=score, frame=frame)
    pad = (ids < 0).unsqueeze(-1)
    d.arg.masked_fill_(pad, -1)
    d.score.masked_fill_(pad, float("-inf"))
    if two:
        d.frame.masked_fill_(pad, float("-inf"))
    return d


def _worker(rank, world, port, Nv, M, K, q, exchange, two):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        import __graft_entry__ as ge
        ge.load_package()
        from dkd_b200 import engine
        from tests.test_dist_gloo import _np_topk
        g = torch.Generator().manual_seed(321)
        scores = torch.randn(M, Nv, generator=g)
        scores[:, 3::7] = 0.5                       # exact ties across shards
        lo, hi = engine.shard_range(Nv, rank, world)
        ls, li = _np_topk(scores[:, lo:hi].numpy(), K, lo)
        m_idx = torch.arange(M).view(M, 1).expand(M, K)
        ld = _detail_of(li, m_idx, two)
        ms, mi, md = engine.merge_shards(ls, li, merge_fn=_np_merge_payload, exchange=exchange, detail=ld)
        ref = O.topk_ids(scores.numpy(), K)
        kk = min(K, Nv)
        ok = np.array_equal(mi.numpy()[:, :kk], ref[:, :kk])
        want = _detail_of(mi, m_idx, two)
        ok = ok and torch.equal(md.arg, want.arg) and torch.equal(md.score, want.score)
        ok = ok and (torch.equal(md.frame, want.frame) if two else md.frame is None)
        if exchange == "query_block":       # the un-gathered form: this rank's query block only
            bs, bi, (q_lo, q_hi), bd = engine.merge_shards(ls, li, merge_fn=_np_merge_payload, gather=False, detail=ld)
            ok = ok and torch.equal(bi, mi[q_lo:q_hi]) and torch.equal(bd.arg, md.arg[q_lo:q_hi])
            ok = ok and torch.equal(bd.score, md.score[q_lo:q_hi])
        q.put((rank, bool(ok)))
    finally:
        dist.destroy_process_group()


def _run(world, Nv, M, K, exchange="query_block", two=True):
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, Nv, M, K, q, exchange, two)) for r in range(world)]
    for p in procs:
        p.start()
    res = [q.get(timeout=180) for _ in procs]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    return sorted(res)


def test_merge_shards_detail_world2_query_block():
    assert all(ok for _, ok in _run(2, Nv=501, M=37, K=100))


def test_merge_shards_detail_world2_all_gather_frame_head():
    assert all(ok for _, ok in _run(2, Nv=501, M=37, K=100, exchange="all_gather", two=False))


def test_merge_shards_detail_world3_short_query_blocks_and_small_shards():
    """3 ranks, 37 queries (blocks of 13 / 13 / 11), shards smaller than K (padding must not survive)."""
    assert all(ok for _, ok in _run(3, Nv=200, M=37, K=100))
    assert all(ok for _, ok in _run(3, Nv=60, M=5, K=30))

"""Deep rankings: top-K up to 4,096 per query (engine.rank(K=...) with K > 256) on every route.

The warp-per-row kernels stop at K = 256 (dense top-K, merges) and Kc = 512 (candidate sort); deeper lists go through
dkd_sort_candidates_deep, dkd_topk_deep and dkd_merge_topk_deep.  Checked here:
  - the three kernels against numpy lexsort (score desc, id asc) bit for bit, with few distinct scores so that exact
    ties happen everywhere, padding, payloads, filters and id_base; where the warp kernels also apply, the deep kernels
    give their output bit for bit;
  - end to end on ~1,500 ragged videos at K = 257 and 600: every route equals precision="exact" and the numpy top-K of
    the exact dense fused matrix, with one and two branches, with and without the detail and a filter; the top-100 of
    a K = 600 ranking is the K = 100 ranking; the certificate's re-rank; shard merges through both exchanges of
    merge_shards; rank_streamed; eval.rank_queries; localize on a deep list;
  - K <= 256 makes the same C-ABI calls as before the deep kernels existed, and none of them.
"""
import numpy as np
import pytest
import torch

from tests import synth
from tests.test_gpu_detail import ROUTES, _lists, _np_ranked, _refuse, _same_detail
from tests.test_gpu_filter import _allowed_rows, _np_topk, _pack, _words

pytestmark = pytest.mark.gpu

DEEP_ENTRIES = {"dkd_sort_candidates_deep", "dkd_topk_deep", "dkd_merge_topk_deep"}
SHALLOW_ENTRIES = {"dkd_topk", "dkd_topk_filtered", "dkd_sort_candidates", "dkd_sort_candidates_payload",
                   "dkd_merge_topk", "dkd_merge_topk_payload"}


def _np_topk_dense(scores, K, id_base=0):
    return _np_topk(scores, np.ones(scores.shape, bool), K, id_base)


def _sorted_lists(rng, G, Mq, K, pad_frac):
    """(G, Mq, K) lists, each sorted (score desc, id asc) with its padding at the end; ids distinct per query across
    the G lists, scores from few values (ties inside and across lists)."""
    s, i = _lists(rng, Mq, G * K, pad_frac)
    s = s.reshape(Mq, G, K).transpose(1, 0, 2).copy()
    i = i.reshape(Mq, G, K).transpose(1, 0, 2).copy()
    i[-1, Mq - 1] = -1                                   # one list all padding
    for g in range(G):
        for m in range(Mq):
            s[g, m], i[g, m], _ = _np_ranked(s[g, m], i[g, m], np.zeros((K, 1), np.int32), K, 1)
    return s, i


# ---------------------------------------------------------------------------------------------------- kernels
@pytest.mark.parametrize("Kc,K_out", [(1, 1), (257, 100), (257, 257), (513, 513), (1000, 300), (1000, 1000),
                                      (4096, 1000), (4096, 4096), (8192, 257), (8192, 4096)])
@pytest.mark.parametrize("C", [None, 1, 6, 8])
def test_sort_candidates_deep_against_numpy(ops, Kc, K_out, C):
    rng = np.random.default_rng(Kc * 10 + (C or 0))
    Mq = 6
    s, i = _lists(rng, Mq, Kc, 0.2)                      # -1 padding at arbitrary positions
    if Kc > 1:
        i[0] = -1                                        # a row without any candidate
    Cw = C or 1
    w = rng.integers(-2 ** 31, 2 ** 31 - 1, (Mq, Kc, Cw), dtype=np.int64).astype(np.int32)
    cs, ci, cw = torch.from_numpy(s).cuda(), torch.from_numpy(i).cuda(), torch.from_numpy(w).cuda()
    pad = torch.full((Cw,), -7, dtype=torch.int32)
    if C is None:
        os_, oi = ops.sort_candidates_deep(cs, ci, K_out)
    else:
        os_, oi, ow = ops.sort_candidates_deep(cs, ci, K_out, payload=cw, pad=pad)
    for m in range(Mq):
        es, ei, ew = _np_ranked(s[m], i[m], w[m], K_out, Cw)
        assert np.array_equal(oi[m].cpu().numpy(), ei) and np.array_equal(os_[m].cpu().numpy(), es), m
        if C is not None:
            assert np.array_equal(ow[m].cpu().numpy(), ew), m
    if Kc <= 512:                                        # where the warp kernel also applies: its output bit for bit
        if C is None:
            rs, ri = ops.sort_candidates(cs, ci, K_out)
        else:
            rs, ri, rw = ops.sort_candidates_payload(cs, ci, cw, K_out, pad)
            assert torch.equal(ow, rw)
        assert torch.equal(os_, rs) and torch.equal(oi, ri)


@pytest.mark.parametrize("K", [1, 100, 256, 257, 1000, 4096])
@pytest.mark.parametrize("Nvk", [5000, 700])
@pytest.mark.parametrize("id_base", [0, 37])
def test_topk_deep_against_numpy(ops, K, Nvk, id_base):
    rng = np.random.default_rng(K + Nvk + id_base)
    Mq = 9
    scores = (rng.integers(-6, 7, (Mq, Nvk)) / 8.0).astype(np.float32)
    scores[1] = 0.5                                      # a row of one value: the K lowest ids
    st = torch.from_numpy(scores).cuda()
    s, i = ops.topk_deep(st, K, id_base)
    ref_s, ref_i = _np_topk_dense(scores, K, id_base)
    assert np.array_equal(i.cpu().numpy(), ref_i) and np.array_equal(s.cpu().numpy(), ref_s)
    if K <= 256:
        rs, ri = ops.topk(st, K, id_base)
        assert torch.equal(s, rs) and torch.equal(i, ri)


@pytest.mark.parametrize("K", [1, 100, 256, 257, 1000, 4096])
@pytest.mark.parametrize("form", ["per_query", "shared_K-1", "shared_K", "shared_K+1", "shared_all"])
def test_topk_deep_filtered_against_numpy(ops, K, form):
    Nvk, id_base = 5000, 37
    rng = np.random.default_rng(K * 7 + len(form))
    counts = [max(K - 1, 0), K, K + 1, Nvk, Nvk // 2]
    Mq = 2 * len(counts)
    scores = (rng.integers(-6, 7, (Mq, Nvk)) / 8.0).astype(np.float32)
    if form == "per_query":
        allowed = _allowed_rows(rng, Mq, Nvk, counts)
    else:
        c = {"shared_K-1": max(K - 1, 0), "shared_K": K, "shared_K+1": K + 1, "shared_all": Nvk}[form]
        allowed = _allowed_rows(rng, 1, Nvk, [c])
    W = (id_base + Nvk + 31) // 32 + 1
    full = rng.random((allowed.shape[0], 32 * W)) < 0.5      # bits outside this corpus's ids: random (ignored)
    full[:, id_base: id_base + Nvk] = allowed
    words = torch.from_numpy(_pack(full)).cuda()
    st = torch.from_numpy(scores).cuda()
    s, i = ops.topk_deep(st, K, id_base, words=words)
    ref_s, ref_i = _np_topk(scores, np.broadcast_to(allowed, (Mq, Nvk)), K, id_base)
    assert np.array_equal(i.cpu().numpy(), ref_i) and np.array_equal(s.cpu().numpy(), ref_s)
    if K <= 256:
        rs, ri = ops.topk_filtered(st, K, words, id_base)
        assert torch.equal(s, rs) and torch.equal(i, ri)


@pytest.mark.parametrize("G", [1, 2, 3, 8])
@pytest.mark.parametrize("Kl", [1, 37, 256, 257, 1000, 4096])
@pytest.mark.parametrize("C", [None, 6])
def test_merge_topk_deep_against_numpy(ops, G, Kl, C):
    rng = np.random.default_rng(G * 10000 + Kl * 10 + (C or 0))
    Mq = 5
    s, i = _sorted_lists(rng, G, Mq, Kl, 0.25)
    Cw = C or 1
    w = rng.integers(-2 ** 31, 2 ** 31 - 1, (G, Mq, Kl, Cw), dtype=np.int64).astype(np.int32)
    gs, gi, gw = torch.from_numpy(s).cuda(), torch.from_numpy(i).cuda(), torch.from_numpy(w).cuda()
    pad = torch.full((Cw,), -7, dtype=torch.int32)
    if C is None:
        ms, mi = ops.merge_topk_deep(gs, gi)
    else:
        ms, mi, mw = ops.merge_topk_deep(gs, gi, payload=gw, pad=pad)
    for m in range(Mq):
        es, ei, ew = _np_ranked(s[:, m].reshape(-1), i[:, m].reshape(-1), w[:, m].reshape(-1, Cw), Kl, Cw)
        assert np.array_equal(mi[m].cpu().numpy(), ei) and np.array_equal(ms[m].cpu().numpy(), es), m
        if C is not None:
            assert np.array_equal(mw[m].cpu().numpy(), ew), m
    if Kl <= 256:
        if C is None:
            rs, ri = ops.merge_topk(gs, gi)
        else:
            rs, ri, rw = ops.merge_topk_payload(gs, gi, gw, pad)
            assert torch.equal(mw, rw)
        assert torch.equal(ms, rs) and torch.equal(mi, ri)


@pytest.mark.parametrize("Kl", [100, 600])
def test_merge_topk_deep_keeps_duplicate_entries_like_the_warp_merge(ops, Kl):
    """The same (score, id) in two lists (no payload): both copies are kept, as the warp merge keeps them."""
    rng = np.random.default_rng(Kl)
    s, i = _sorted_lists(rng, 2, 4, Kl, 0.1)
    s[1], i[1] = s[0], i[0]
    gs, gi = torch.from_numpy(s).cuda(), torch.from_numpy(i).cuda()
    ms, mi = ops.merge_topk_deep(gs, gi)
    es = np.repeat(s[0], 2, axis=1)[:, :Kl]              # padding (-inf, -1) repeats into padding
    ei = np.repeat(i[0], 2, axis=1)[:, :Kl]
    assert np.array_equal(mi.cpu().numpy(), ei) and np.array_equal(ms.cpu().numpy(), es)
    if Kl <= 256:
        rs, ri = ops.merge_topk(gs, gi)
        assert torch.equal(ms, rs) and torch.equal(mi, ri)


# ---------------------------------------------------------------------------------------------------- engine
Nv, L, D, M = 1500, 64, 128, 40
DEPTHS = [257, 600]
_CASES = {}


def _params(nb, seed):
    g = torch.Generator().manual_seed(seed)
    return [(0.05 * torch.randn(D, D, generator=g), 0.01 * torch.randn(D, generator=g),
             0.05 * torch.randn(D, D, generator=g), 0.01 * torch.randn(D, generator=g)) for _ in range(nb)]


def _build(nb):
    """~1,500 ragged videos (lengths 5 .. 64), nb branches, both heads, every precision."""
    from dkd_b200 import engine
    frames, mask, lengths = synth.encoded_corpus(Nv, L, D, seed=71, min_len=5, shared=1.5)
    fr = [frames] + [synth.encoded_corpus(Nv, L, D, seed=72 + b, min_len=5, shared=1.5)[0] * mask[:, :, None]
                     for b in range(1, nb)]
    params = _params(nb, 81)
    qs = [synth.encoded_queries(M, D, seed=90 + b) for b in range(nb)]
    dev = torch.device("cuda")
    prm = [tuple(t.to(dev) for t in p) for p in params]
    pc = engine.prepare_corpus([f.to(dev) for f in fr], mask.to(dev), prm, heads=("frame", "two_scale"),
                               precisions=("exact", "bf16", "fp16", "shortcut"))
    pq = engine.prepare_queries([q.to(dev) for q in qs])
    return dict(nb=nb, frames=fr, mask=mask, lengths=lengths, prm=prm, qs=qs, pc=pc, pq=pq, dense={})


@pytest.fixture(scope="module", params=[1, 2], ids=["1branch", "2branch"])
def case(request, ops):
    nb = request.param
    if nb not in _CASES:
        _CASES[nb] = _build(nb)
    return _CASES[nb]


def _rank(case, head, precision, K, **kw):
    from dkd_b200 import engine
    return engine.rank(case["pc"], case["pq"], K=K, head=head, precision=precision, **kw)


def _dense_exact(case, head):
    if head not in case["dense"]:
        case["dense"][head] = _rank(case, head, "exact", 1, return_dense=True)[2].cpu().numpy()
    return case["dense"][head]


def _filter(seed):
    rng = np.random.default_rng(seed)
    allowed = _allowed_rows(rng, M, Nv, [Nv // 2, 200, 599, 600, 601, Nv])
    return _words(allowed), allowed


@pytest.mark.parametrize("K", DEPTHS)
@pytest.mark.parametrize("head,precision", ROUTES)
def test_deep_rank_equals_exact_and_numpy(case, head, precision, K):
    nb = case["nb"]
    fused = _dense_exact(case, head)
    s_ex, i_ex = _rank(case, head, "exact", K)
    ref_s, ref_i = _np_topk_dense(fused, K)
    assert np.array_equal(i_ex.cpu().numpy(), ref_i) and np.array_equal(s_ex.cpu().numpy(), ref_s)
    s, i = _rank(case, head, precision, K)
    assert torch.equal(i, i_ex) and torch.equal(s, s_ex)
    s, i, det = _rank(case, head, precision, K, return_detail=True)
    assert torch.equal(i, i_ex) and torch.equal(s, s_ex)
    assert det.arg.shape == (M, K, nb) and np.array_equal(_refuse(det, head, nb), s.cpu().numpy())
    if precision != "exact":
        assert _same_detail(det, _rank(case, head, "exact", K, return_detail=True)[2])
    vf, allowed = _filter(K)
    fs_ex, fi_ex = _rank(case, head, "exact", K, video_filter=vf)
    ref_s, ref_i = _np_topk(fused, allowed, K)
    assert np.array_equal(fi_ex.cpu().numpy(), ref_i) and np.array_equal(fs_ex.cpu().numpy(), ref_s)
    fs, fi, fdet = _rank(case, head, precision, K, video_filter=vf, return_detail=True)
    assert torch.equal(fi, fi_ex) and torch.equal(fs, fs_ex)
    assert np.array_equal(_refuse(fdet, head, nb), fs.cpu().numpy())
    assert (fdet.arg[fi < 0] == -1).all()


@pytest.mark.parametrize("head,precision", [("frame", "bf16"), ("two_scale", "bf16"), ("two_scale", "fp16")])
def test_deep_unrescored_route_is_the_top_k_of_its_dense_matrix(case, head, precision):
    s, i, dense = _rank(case, head, precision, 600, rescore=False, return_dense=True)
    ref_s, ref_i = _np_topk_dense(dense.cpu().numpy(), 600)
    assert np.array_equal(i.cpu().numpy(), ref_i) and np.array_equal(s.cpu().numpy(), ref_s)
    s, i, det = _rank(case, head, precision, 600, rescore=False, return_detail=True)
    assert np.array_equal(i.cpu().numpy(), ref_i)
    assert np.array_equal(_refuse(det, head, case["nb"]), s.cpu().numpy())


@pytest.mark.parametrize("head,precision", [("two_scale", "bf16"), ("frame", "bf16"), ("two_scale", "exact"),
                                            ("two_scale", "shortcut")])
def test_top_100_of_a_deep_ranking_is_the_k100_ranking(case, head, precision):
    s6, i6, d6 = _rank(case, head, precision, 600, return_detail=True)
    s1, i1, d1 = _rank(case, head, precision, 100, return_detail=True)
    assert torch.equal(i6[:, :100], i1) and torch.equal(s6[:, :100], s1)
    assert torch.equal(d6.arg[:, :100], d1.arg) and torch.equal(d6.score[:, :100].view(torch.int32),
                                                                d1.score.view(torch.int32))


@pytest.mark.parametrize("head", ["frame", "two_scale"])
@pytest.mark.parametrize("certify", [True, "deferred"])
def test_deep_certificate_fallback_patches_rows(case, head, certify, monkeypatch):
    """A certificate margin larger than any score gap fails every query: all rows are re-ranked by the deep exact
    top-K and patched, scores, ids and detail."""
    from dkd_b200 import engine
    K = 600
    s_ex, i_ex, d_ex = _rank(case, head, "exact", K, return_detail=True)
    vf, _ = _filter(5)
    fs_ex, fi_ex, fd_ex = _rank(case, head, "exact", K, return_detail=True, video_filter=vf)
    monkeypatch.setattr(engine, "CERT_EPS", 10.0)
    for kw, (es, ei, ed) in ((dict(), (s_ex, i_ex, d_ex)), (dict(video_filter=vf), (fs_ex, fi_ex, fd_ex))):
        engine.STATS["certify_fallback_queries"] = 0
        s, i, d = _rank(case, head, "bf16", K, certify=certify, return_detail=True, **kw)
        if certify == "deferred":
            engine.finish()
        assert engine.STATS["certify_fallback_queries"] > 0
        assert torch.equal(i, ei) and torch.equal(s, es) and _same_detail(d, ed)


class _FakeDist:
    """torch.distributed as seen by one rank of `world`, with the other ranks' data given up front: enough of the
    collectives of engine.merge_shards to run both exchanges of G shards in one process."""

    def __init__(self, world, locals_by_rank, rank_=0, blocks_by_rank=None):
        self.world, self.rank_, self.locals, self.blocks = world, rank_, locals_by_rank, blocks_by_rank
        self.n_a2a = self.n_gather = 0

    def install(self, monkeypatch):
        import torch.distributed as dist
        for name in ("get_world_size", "get_rank", "get_backend", "all_gather", "all_to_all_single"):
            monkeypatch.setattr(dist, name, getattr(self, name))

    def get_world_size(self, group=None):
        return self.world

    def get_rank(self, group=None):
        return self.rank_

    def get_backend(self, group=None):
        return "gloo"

    def all_gather(self, outs, t, group=None):
        k = self.n_gather
        self.n_gather += 1
        src = self.blocks if self.blocks is not None else self.locals
        for g, o in enumerate(outs):
            o.copy_(src[g][k].reshape(o.shape))

    def all_to_all_single(self, out, inp, out_split, in_split, group=None):
        k = self.n_a2a
        self.n_a2a += 1
        Mq = inp.shape[0]
        Mb = (Mq + self.world - 1) // self.world
        lo, hi = min(self.rank_ * Mb, Mq), min((self.rank_ + 1) * Mb, Mq)
        if hi == lo:                                    # a rank without queries receives nothing
            return
        rows = out.view(self.world, hi - lo, -1)
        for g in range(self.world):
            rows[g].copy_(self.locals[g][k].reshape(Mq, -1)[lo:hi])


@pytest.mark.parametrize("head,precision", [("two_scale", "bf16"), ("frame", "bf16"), ("two_scale", "exact")])
@pytest.mark.parametrize("exchange", ["all_gather", "query_block"])
def test_deep_shards_merge_to_the_resident_ranking(case, head, precision, exchange, monkeypatch):
    """Shards of 37 videos (ids not aligned to 32, fewer videos than K per shard, more shards than queries), merged by
    engine.merge_shards with and without the detail and a filter."""
    from dkd_b200 import engine
    K, step = 600, 37
    frames = [f.cuda() for f in case["frames"]]
    mask = case["mask"].cuda()
    shards = [engine.prepare_corpus([f[lo: lo + step] for f in frames], mask[lo: lo + step], case["prm"],
                                    heads=(head,), precisions=("exact", precision), id_base=lo)
              for lo in range(0, Nv, step)]
    world = len(shards)
    vf, _ = _filter(9)
    for kw in (dict(), dict(video_filter=vf)):
        s_r, i_r, d_r = _rank(case, head, precision, K, return_detail=True, **kw)
        outs = [engine.rank(pc, case["pq"], K=K, head=head, precision=precision, return_detail=True, **kw)
                for pc in shards]
        for detail in (False, True):
            locs = [[o[0], o[1]] + ([o[2].pack()] if detail else []) for o in outs]
            blocks = None
            if exchange == "query_block":     # every rank's merged block first, then rank 0's all-gather of them
                blocks = []
                for r in range(world):
                    with monkeypatch.context() as mp:
                        _FakeDist(world, locs, r).install(mp)
                        res = engine.merge_shards(outs[r][0], outs[r][1], exchange=exchange, gather=False,
                                                  detail=outs[r][2] if detail else None)
                    blk = [res[0], res[1]] + ([res[3].pack()] if detail else [])
                    Mb = (M + world - 1) // world
                    fills = [float("-inf"), -1, -1]
                    blocks.append([torch.cat([b, b.new_full((Mb - b.shape[0],) + b.shape[1:], f)])
                                   for b, f in zip(blk, fills)])
            with monkeypatch.context() as mp:
                _FakeDist(world, locs, 0, blocks).install(mp)
                res = engine.merge_shards(outs[0][0], outs[0][1], exchange=exchange,
                                          detail=outs[0][2] if detail else None)
            assert torch.equal(res[1], i_r) and torch.equal(res[0], s_r), (kw.keys(), detail)
            if detail:
                assert _same_detail(res[2], d_r)


@pytest.mark.parametrize("head,precision", [("two_scale", "bf16"), ("frame", "bf16"), ("two_scale", "exact")])
def test_deep_streamed_ranking_equals_resident(case, head, precision):
    from dkd_b200 import engine
    K = 600
    frames = [f.cuda() for f in case["frames"]]
    pqs = engine.split_queries([q.cuda() for q in case["qs"]], batch=17)          # 17 + 17 + 6 queries
    assert len(pqs) == 3
    vf, _ = _filter(13)
    for kw in (dict(), dict(video_filter=vf)):
        s_r, i_r, d_r = _rank(case, head, precision, K, return_detail=True, **kw)
        for chunk in (211, 700):       # chunks of fewer videos than K: padded lists fold into the running list
            chunks = engine.iter_chunks(frames, case["mask"].cuda(), chunk_videos=chunk)
            s, i = engine.rank_streamed(chunks, pqs, case["prm"], K=K, head=head, precision=precision, **kw)
            assert torch.equal(i, i_r) and torch.equal(s, s_r), chunk
            chunks = engine.iter_chunks(frames, case["mask"].cuda(), chunk_videos=chunk)
            s, i, d = engine.rank_streamed(chunks, pqs, case["prm"], K=K, head=head, precision=precision,
                                           return_detail=True, **kw)
            assert torch.equal(i, i_r) and torch.equal(s, s_r) and _same_detail(d, d_r), chunk


def test_localize_on_a_deep_list(case):
    from dkd_b200 import engine
    _, ids, _ = _rank(case, "two_scale", "bf16", 600, return_detail=True)
    deep = engine.localize(case["pc"], case["pq"], ids, m=5, iou=0.5)
    head = engine.localize(case["pc"], case["pq"], ids[:, :100].contiguous(), m=5, iou=0.5)
    assert deep.arg.shape == (M, 600, 5)
    assert torch.equal(deep.arg[:, :100], head.arg)
    assert torch.equal(deep.score[:, :100].view(torch.int32), head.score.view(torch.int32))
    assert (deep.arg[:, :, 0] >= 0).all()


@pytest.mark.parametrize("scoring", ["frame", "two_scale"])
def test_rank_queries_deep(ops, dkd, scoring):
    from dkd_b200 import engine, eval as E
    from tests.test_gpu_dropin import _tiny_setup
    _, m, vset, qset, opt = _tiny_setup(dkd)
    opt.scoring, opt.precision, opt.query_chunk = scoring, "bf16", 7
    ctx = E.compute_context_info(m, vset, opt)
    qs, _, _ = E._encode_all_queries(m, qset, opt)
    Kt = 300                                             # more than the videos of the fixture: padded rows
    s, i, _ = E.rank_queries(m, qset, opt, ctx, K=Kt)
    pq = engine.prepare_queries(qs)
    s_ex, i_ex = engine.rank(ctx["prepared"], pq, K=Kt, head=scoring, precision="exact", w_clip=m.clip_scale_w,
                             w_frame=m.frame_scale_w)
    assert s.shape == (len(qset), Kt) and torch.equal(i, i_ex) and torch.equal(s, s_ex)
    assert (i[:, len(vset):] == -1).all()


# ---------------------------------------------------------------------------------------------------- call record
# The C-ABI calls of every shallow route (K <= 256), recorded from the engine before the deep kernels existed: key
# "head/precision/branches/<detail><filter>", value the entry points in call order without their "dkd_" prefix.  The
# list does not depend on K <= 256 and is taken with certify=False (a fallback appends the exact route's calls).
SHALLOW_CALLS = {
    "frame/exact/1/00": "score_max_exact topk",
    "frame/exact/1/01": "score_max_exact topk_filtered",
    "frame/exact/1/10": "score_max_exact topk",
    "frame/exact/1/11": "score_max_exact topk_filtered",
    "frame/bf16/1/00": "score_max_bf16 select_topk candidates_to_csr score_max_exact scatter_fuse sort_candidates",
    "frame/bf16/1/01": ("score_max_bf16 select_topk_filtered candidates_to_csr score_max_exact scatter_fuse "
                        "sort_candidates"),
    "frame/bf16/1/10": ("score_max_bf16 select_topk candidates_to_csr score_max_exact scatter_fuse_detail "
                        "sort_candidates_payload"),
    "frame/bf16/1/11": ("score_max_bf16 select_topk_filtered candidates_to_csr score_max_exact scatter_fuse_detail "
                        "sort_candidates_payload"),
    "frame/fp16/1/00": "score_max_f16 select_topk candidates_to_csr score_max_exact scatter_fuse sort_candidates",
    "frame/fp16/1/01": ("score_max_f16 select_topk_filtered candidates_to_csr score_max_exact scatter_fuse "
                        "sort_candidates"),
    "frame/fp16/1/10": ("score_max_f16 select_topk candidates_to_csr score_max_exact scatter_fuse_detail "
                        "sort_candidates_payload"),
    "frame/fp16/1/11": ("score_max_f16 select_topk_filtered candidates_to_csr score_max_exact scatter_fuse_detail "
                        "sort_candidates_payload"),
    "two_scale/exact/1/00": "clip_score_f32 frame_fuse topk",
    "two_scale/exact/1/01": "clip_score_f32 frame_fuse topk_filtered",
    "two_scale/exact/1/10": "clip_score_f32 frame_fuse topk",
    "two_scale/exact/1/11": "clip_score_f32 frame_fuse topk_filtered",
    "two_scale/bf16/1/00": ("score_max_bf16_lists clip_score_list frame_fuse select_topk candidates_to_csr "
                            "clip_score_f32 frame_fuse_csr sort_candidates"),
    "two_scale/bf16/1/01": ("score_max_bf16_lists clip_score_list frame_fuse select_topk_filtered "
                            "candidates_to_csr clip_score_f32 frame_fuse_csr sort_candidates"),
    "two_scale/bf16/1/10": ("score_max_bf16_lists clip_score_list frame_fuse select_topk candidates_to_csr "
                            "clip_score_f32 frame_fuse_csr_detail sort_candidates_payload"),
    "two_scale/bf16/1/11": ("score_max_bf16_lists clip_score_list frame_fuse select_topk_filtered "
                            "candidates_to_csr clip_score_f32 frame_fuse_csr_detail sort_candidates_payload"),
    "two_scale/fp16/1/00": ("score_max_bf16_lists clip_score_list frame_fuse select_topk candidates_to_csr "
                            "clip_score_f32 frame_fuse_csr sort_candidates"),
    "two_scale/fp16/1/01": ("score_max_bf16_lists clip_score_list frame_fuse select_topk_filtered "
                            "candidates_to_csr clip_score_f32 frame_fuse_csr sort_candidates"),
    "two_scale/fp16/1/10": ("score_max_bf16_lists clip_score_list frame_fuse select_topk candidates_to_csr "
                            "clip_score_f32 frame_fuse_csr_detail sort_candidates_payload"),
    "two_scale/fp16/1/11": ("score_max_bf16_lists clip_score_list frame_fuse select_topk_filtered "
                            "candidates_to_csr clip_score_f32 frame_fuse_csr_detail sort_candidates_payload"),
    "two_scale/shortcut/1/00": ("clip_score_f32 frame_fuse select_topk candidates_to_csr frame_fuse_csr "
                                "sort_candidates"),
    "two_scale/shortcut/1/01": ("clip_score_f32 frame_fuse select_topk_filtered candidates_to_csr frame_fuse_csr "
                                "sort_candidates"),
    "two_scale/shortcut/1/10": ("clip_score_f32 frame_fuse select_topk candidates_to_csr frame_fuse_csr_detail "
                                "sort_candidates_payload"),
    "two_scale/shortcut/1/11": ("clip_score_f32 frame_fuse select_topk_filtered candidates_to_csr "
                                "frame_fuse_csr_detail sort_candidates_payload"),
    "frame/exact/2/00": "score_max_exact score_max_exact fuse_scores topk",
    "frame/exact/2/01": "score_max_exact score_max_exact fuse_scores topk_filtered",
    "frame/exact/2/10": "score_max_exact score_max_exact fuse_scores topk",
    "frame/exact/2/11": "score_max_exact score_max_exact fuse_scores topk_filtered",
    "frame/bf16/2/00": ("score_max_bf16 score_max_bf16 fuse_scores select_topk candidates_to_csr score_max_exact "
                        "score_max_exact scatter_fuse sort_candidates"),
    "frame/bf16/2/01": ("score_max_bf16 score_max_bf16 fuse_scores select_topk_filtered candidates_to_csr "
                        "score_max_exact score_max_exact scatter_fuse sort_candidates"),
    "frame/bf16/2/10": ("score_max_bf16 score_max_bf16 fuse_scores select_topk candidates_to_csr score_max_exact "
                        "score_max_exact scatter_fuse_detail sort_candidates_payload"),
    "frame/bf16/2/11": ("score_max_bf16 score_max_bf16 fuse_scores select_topk_filtered candidates_to_csr "
                        "score_max_exact score_max_exact scatter_fuse_detail sort_candidates_payload"),
    "frame/fp16/2/00": ("score_max_f16 score_max_f16 fuse_scores select_topk candidates_to_csr score_max_exact "
                        "score_max_exact scatter_fuse sort_candidates"),
    "frame/fp16/2/01": ("score_max_f16 score_max_f16 fuse_scores select_topk_filtered candidates_to_csr "
                        "score_max_exact score_max_exact scatter_fuse sort_candidates"),
    "frame/fp16/2/10": ("score_max_f16 score_max_f16 fuse_scores select_topk candidates_to_csr score_max_exact "
                        "score_max_exact scatter_fuse_detail sort_candidates_payload"),
    "frame/fp16/2/11": ("score_max_f16 score_max_f16 fuse_scores select_topk_filtered candidates_to_csr "
                        "score_max_exact score_max_exact scatter_fuse_detail sort_candidates_payload"),
    "two_scale/exact/2/00": "clip_score_f32 frame_fuse clip_score_f32 frame_fuse topk",
    "two_scale/exact/2/01": "clip_score_f32 frame_fuse clip_score_f32 frame_fuse topk_filtered",
    "two_scale/exact/2/10": "clip_score_f32 frame_fuse clip_score_f32 frame_fuse topk",
    "two_scale/exact/2/11": "clip_score_f32 frame_fuse clip_score_f32 frame_fuse topk_filtered",
    "two_scale/bf16/2/00": ("score_max_bf16_lists clip_score_list frame_fuse score_max_bf16_lists clip_score_list "
                            "frame_fuse select_topk candidates_to_csr clip_score_f32 frame_fuse_csr clip_score_f32 "
                            "frame_fuse_csr sort_candidates"),
    "two_scale/bf16/2/01": ("score_max_bf16_lists clip_score_list frame_fuse score_max_bf16_lists clip_score_list "
                            "frame_fuse select_topk_filtered candidates_to_csr clip_score_f32 frame_fuse_csr "
                            "clip_score_f32 frame_fuse_csr sort_candidates"),
    "two_scale/bf16/2/10": ("score_max_bf16_lists clip_score_list frame_fuse score_max_bf16_lists clip_score_list "
                            "frame_fuse select_topk candidates_to_csr clip_score_f32 frame_fuse_csr_detail "
                            "clip_score_f32 frame_fuse_csr_detail sort_candidates_payload"),
    "two_scale/bf16/2/11": ("score_max_bf16_lists clip_score_list frame_fuse score_max_bf16_lists clip_score_list "
                            "frame_fuse select_topk_filtered candidates_to_csr clip_score_f32 "
                            "frame_fuse_csr_detail clip_score_f32 frame_fuse_csr_detail sort_candidates_payload"),
    "two_scale/fp16/2/00": ("score_max_bf16_lists clip_score_list frame_fuse score_max_bf16_lists clip_score_list "
                            "frame_fuse select_topk candidates_to_csr clip_score_f32 frame_fuse_csr clip_score_f32 "
                            "frame_fuse_csr sort_candidates"),
    "two_scale/fp16/2/01": ("score_max_bf16_lists clip_score_list frame_fuse score_max_bf16_lists clip_score_list "
                            "frame_fuse select_topk_filtered candidates_to_csr clip_score_f32 frame_fuse_csr "
                            "clip_score_f32 frame_fuse_csr sort_candidates"),
    "two_scale/fp16/2/10": ("score_max_bf16_lists clip_score_list frame_fuse score_max_bf16_lists clip_score_list "
                            "frame_fuse select_topk candidates_to_csr clip_score_f32 frame_fuse_csr_detail "
                            "clip_score_f32 frame_fuse_csr_detail sort_candidates_payload"),
    "two_scale/fp16/2/11": ("score_max_bf16_lists clip_score_list frame_fuse score_max_bf16_lists clip_score_list "
                            "frame_fuse select_topk_filtered candidates_to_csr clip_score_f32 "
                            "frame_fuse_csr_detail clip_score_f32 frame_fuse_csr_detail sort_candidates_payload"),
    "two_scale/shortcut/2/00": ("clip_score_f32 frame_fuse clip_score_f32 frame_fuse select_topk candidates_to_csr "
                                "frame_fuse_csr frame_fuse_csr sort_candidates"),
    "two_scale/shortcut/2/01": ("clip_score_f32 frame_fuse clip_score_f32 frame_fuse select_topk_filtered "
                                "candidates_to_csr frame_fuse_csr frame_fuse_csr sort_candidates"),
    "two_scale/shortcut/2/10": ("clip_score_f32 frame_fuse clip_score_f32 frame_fuse select_topk candidates_to_csr "
                                "frame_fuse_csr_detail frame_fuse_csr_detail sort_candidates_payload"),
    "two_scale/shortcut/2/11": ("clip_score_f32 frame_fuse clip_score_f32 frame_fuse select_topk_filtered "
                                "candidates_to_csr frame_fuse_csr_detail frame_fuse_csr_detail "
                                "sort_candidates_payload"),
}


def test_shallow_calls_are_unchanged_and_deep_calls_use_the_deep_kernels(case, monkeypatch):
    from dkd_b200 import _lib, engine
    calls = []
    real = _lib.call

    def record(name, *args):
        calls.append(name)
        return real(name, *args)

    monkeypatch.setattr(_lib, "call", record)
    vf, _ = _filter(3)
    nb = case["nb"]

    def pinned(head, precision, detail, filt):
        return ["dkd_" + n for n in SHALLOW_CALLS[f"{head}/{precision}/{nb}/{int(detail)}{int(filt)}"].split()]

    for head, precision in ROUTES:
        for K in (100, 256):
            for detail in (False, True):
                for filt in (False, True):
                    calls.clear()
                    _rank(case, head, precision, K, certify=False, return_detail=detail,
                          video_filter=vf if filt else None)
                    assert calls == pinned(head, precision, detail, filt), (head, precision, K, detail, filt)
        if precision != "exact":
            # Kc = K: the certificate fires, and the re-rank is the exact route's calls on the failed queries
            for detail in (False, True):
                calls.clear()
                engine.STATS["certify_fallback_queries"] = 0
                _rank(case, head, precision, 100, Kc=100, return_detail=detail)
                assert engine.STATS["certify_fallback_queries"] > 0
                assert calls == pinned(head, precision, detail, False) + pinned(head, "exact", detail, False)
    lists = [torch.stack([t, t]) for t in _rank(case, "two_scale", "bf16", 100)]
    calls.clear()
    engine._merge_lists(*lists)
    assert calls == ["dkd_merge_topk"]
    calls.clear()
    for head, precision in ROUTES:
        _rank(case, head, precision, 600)
        _rank(case, head, precision, 600, return_detail=True, video_filter=vf)
    assert {"dkd_topk_deep", "dkd_sort_candidates_deep"} <= set(calls)
    assert not SHALLOW_ENTRIES & set(calls)

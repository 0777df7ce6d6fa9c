"""Filtered ranking (engine.rank(video_filter=...)): each query's top-K restricted to the videos its filter row allows.

The filter acts in the two kernels that choose hits (dkd_topk_filtered on the dense routes, dkd_select_topk_filtered for
the candidates of the bf16 / fp16 / shortcut routes); everything after them is unchanged.  Checked here:
  - both kernels and the filter builder against numpy (allowed counts 0 .. all, id_base not a multiple of 32, shared and
    per-query rows, exact ties at the K-th score with disallowed tied entries at lower ids, too few words);
  - an all-ones filter changes nothing, on every head, precision and branch count, with and without the detail;
  - a filtered ranking equals precision="exact" with the same filter, and the numpy top-K of the exact dense fused
    matrix restricted to the allowed videos;
  - the certificate (immediate and deferred) with a filter, and queries with at most Kc allowed videos are certain;
  - shards with unaligned id_base, rank_streamed over unaligned chunks and query batches, eval.rank_queries;
  - video_filter=None calls none of the new entry points.
"""
import numpy as np
import pytest
import torch

from tests.test_gpu_detail import ROUTES, _build, _refuse, _same_detail

pytestmark = pytest.mark.gpu

Nv, M, K = 300, 64, 32
NEW_ENTRIES = {"dkd_topk_filtered", "dkd_select_topk_filtered", "dkd_build_video_filter"}
_CASES = {}


@pytest.fixture(scope="module", params=[1, 2], ids=["1branch", "2branch"])
def case(request, ops):
    nb = request.param
    if nb not in _CASES:
        _CASES[nb] = _build(nb)
    return _CASES[nb]


# ---------------------------------------------------------------------------------------------------- numpy references
def _pack(allowed):
    """(rows, n) bool -> (rows, ceil(n / 32)) int32 words, bit g & 31 of word g >> 5 = allowed[:, g]."""
    rows, n = allowed.shape
    W = (n + 31) // 32
    bits = np.zeros((rows, 32 * W), np.uint8)
    bits[:, :n] = allowed
    return np.packbits(bits, axis=1, bitorder="little").view("<u4").view(np.int32).reshape(rows, W)


def _words(allowed):
    return torch.from_numpy(_pack(allowed)).cuda()


def _np_topk(scores, allowed, K_, id_base=0):
    """(score desc, id asc) top-K of the allowed entries of every row, padded (-inf, -1)."""
    out_s = np.full((scores.shape[0], K_), -np.inf, np.float32)
    out_i = np.full((scores.shape[0], K_), -1, np.int32)
    for m in range(scores.shape[0]):
        n = np.nonzero(allowed[m])[0]
        order = n[np.lexsort((n, -scores[m, n]))][:K_]
        out_s[m, : len(order)] = scores[m, order]
        out_i[m, : len(order)] = order + id_base
    return out_s, out_i


def _allowed_rows(rng, rows, n, counts):
    """rows x n bool with counts[m % len(counts)] allowed videos in row m, at random positions."""
    a = np.zeros((rows, n), bool)
    for m in range(rows):
        a[m, rng.permutation(n)[: counts[m % len(counts)]]] = True
    return a


# ---------------------------------------------------------------------------------------------------- kernels
KK = 40
COUNTS = [0, 1, KK - 1, KK, KK + 1, Nv // 2, Nv]


def _kernel_inputs(rng, id_base, shared, count=None):
    Mk = len(COUNTS) * 3
    scores = (rng.integers(-6, 7, (Mk, Nv)) / 8.0).astype(np.float32)       # few values: exact ties everywhere
    allowed = _allowed_rows(rng, 1 if shared else Mk, Nv, [count] if shared else COUNTS)
    # the words cover [0, id_base + Nv) and one word more; bits outside this corpus's ids are random (ignored)
    W = (id_base + Nv + 31) // 32 + 1
    full = rng.random((allowed.shape[0], 32 * W)) < 0.5
    full[:, id_base: id_base + Nv] = allowed
    return scores, np.broadcast_to(allowed, (Mk, Nv)), torch.from_numpy(_pack(full)).cuda()


@pytest.mark.parametrize("id_base", [0, 5, 37])
@pytest.mark.parametrize("form", ["per_query"] + [f"shared{c}" for c in COUNTS])
def test_topk_and_select_filtered_against_numpy(ops, id_base, form):
    rng = np.random.default_rng(100 + id_base)
    shared = form != "per_query"
    scores, allowed, words = _kernel_inputs(rng, id_base, shared, int(form[6:]) if shared else None)
    st = torch.from_numpy(scores).cuda()
    ref_s, ref_i = _np_topk(scores, allowed, KK, id_base)
    s, i = ops.topk_filtered(st, KK, words, id_base)
    assert np.array_equal(i.cpu().numpy(), ref_i) and np.array_equal(s.cpu().numpy(), ref_s)
    cand, kth = ops.select_topk_filtered(st, KK, words, id_base)
    cand, kth = cand.cpu().numpy(), kth.cpu().numpy()
    for m in range(scores.shape[0]):
        n_allowed = int(allowed[m].sum())
        if n_allowed <= KK:         # every allowed video in column order, -1 padding, kth -inf
            expect = np.concatenate([np.nonzero(allowed[m])[0] + id_base, np.full(KK - n_allowed, -1)])
            assert np.array_equal(cand[m], expect) and np.isneginf(kth[m]), m
        else:
            assert np.array_equal(np.sort(cand[m]), np.sort(ref_i[m])), m
            assert kth[m] == ref_s[m, KK - 1], m


def test_ties_at_the_kth_score_go_to_the_lower_allowed_ids(ops):
    """Every score equal: the K hits are the K lowest ALLOWED ids, although disallowed ids sit below them."""
    Mk, id_base = 16, 37
    scores = np.full((Mk, Nv), 0.25, np.float32)
    scores[:, 200:] = -1.0
    allowed = np.zeros((Mk, Nv), bool)
    for m in range(Mk):
        allowed[m, 3 + m::2] = True                  # ids 0 .. 2 + m and every other one after: disallowed
    words = torch.from_numpy(_pack(np.pad(allowed, ((0, 0), (id_base, 0))))).cuda()
    st = torch.from_numpy(scores).cuda()
    expect = np.stack([np.nonzero(allowed[m])[0][:KK] for m in range(Mk)]) + id_base
    s, i = ops.topk_filtered(st, KK, words, id_base)
    assert np.array_equal(i.cpu().numpy(), expect) and (s == 0.25).all()
    cand, kth = ops.select_topk_filtered(st, KK, words, id_base)
    assert np.array_equal(cand.cpu().numpy(), expect) and (kth == 0.25).all()


def test_too_few_words_raise(ops):
    from dkd_b200 import _lib
    st = torch.zeros((4, Nv), dtype=torch.float32, device="cuda")
    for id_base in (0, 5, 37):
        short = torch.full((1, (id_base + Nv + 31) // 32 - 1), -1, dtype=torch.int32, device="cuda")
        with pytest.raises(_lib.DkdError):
            ops.topk_filtered(st, KK, short, id_base)
        with pytest.raises(_lib.DkdError):
            ops.select_topk_filtered(st, KK, short, id_base)
        # the C ABI checks it too
        lib = _lib.load()
        out = torch.empty((4, KK), dtype=torch.float32, device="cuda")
        oi = torch.empty((4, KK), dtype=torch.int32, device="cuda")
        assert lib.dkd_topk_filtered(st.data_ptr(), 4, Nv, Nv, KK, id_base, short.data_ptr(), 1, short.shape[1],
                                     out.data_ptr(), oi.data_ptr(), None) == -2
        assert lib.dkd_select_topk_filtered(st.data_ptr(), 4, Nv, Nv, KK, id_base, short.data_ptr(), 1,
                                            short.shape[1], oi.data_ptr(), out.data_ptr(), None) == -2
    rows3 = torch.full((3, 16), -1, dtype=torch.int32, device="cuda")        # neither 1 nor M rows
    with pytest.raises(_lib.DkdError):
        ops.topk_filtered(st, KK, rows3)


# ---------------------------------------------------------------------------------------------------- builder
@pytest.mark.parametrize("n_videos", [300, 64, 33, 1])
def test_build_video_filter_against_numpy(ops, n_videos):
    from dkd_b200 import engine
    rng = np.random.default_rng(n_videos)
    lists = [list(rng.integers(0, n_videos, rng.integers(0, 2 * n_videos + 1))) for _ in range(9)]
    lists[2] = []
    lists[4] = lists[4] + lists[4][:5]                    # duplicates
    per = np.zeros((len(lists), n_videos), bool)
    for m, ids in enumerate(lists):
        per[m, ids] = True
    got = engine.make_video_filter(n_videos, allow=lists)
    assert got.dtype == torch.int32 and got.shape == (len(lists), (n_videos + 31) // 32)
    assert np.array_equal(got.cpu().numpy(), _pack(per))
    assert np.array_equal(engine.make_video_filter(n_videos, deny=lists).cpu().numpy(), _pack(~per))
    # one list: a shared row
    assert np.array_equal(engine.make_video_filter(n_videos, allow=lists[0]).cpu().numpy(), _pack(per[:1]))
    assert np.array_equal(engine.make_video_filter(n_videos, deny=lists[1]).cpu().numpy(), _pack(~per[1:2]))
    assert np.array_equal(engine.make_video_filter(n_videos, allow=[]).cpu().numpy(), _pack(np.zeros((1, n_videos), bool)))
    assert np.array_equal(engine.make_video_filter(n_videos, deny=[]).cpu().numpy(), _pack(np.ones((1, n_videos), bool)))


def test_build_video_filter_rejects_bad_input_before_any_launch(ops, monkeypatch):
    from dkd_b200 import _lib, engine
    calls = []
    real = _lib.call
    monkeypatch.setattr(_lib, "call", lambda name, *a: (calls.append(name), real(name, *a))[1])
    for kw in (dict(allow=[[0, 1], [5, 300]]), dict(deny=[-1]), dict(allow=[3, 300]), dict(), dict(allow=[1], deny=[2])):
        with pytest.raises(ValueError):
            engine.make_video_filter(300, **kw)
    assert calls == []


# ---------------------------------------------------------------------------------------------------- engine.rank
def _rank(case, head, precision, **kw):
    from dkd_b200 import engine
    return engine.rank(case["pc"], case["pq"], K=K, head=head, precision=precision, **kw)


@pytest.mark.parametrize("head,precision", ROUTES)
def test_all_ones_filter_is_a_no_op(case, head, precision):
    from dkd_b200 import engine
    ones = engine.make_video_filter(Nv, deny=[])
    per_query = ones.expand(M, -1).contiguous()
    s0, i0, d0 = _rank(case, head, precision, return_detail=True)
    for vf in (ones, per_query):
        s, i = _rank(case, head, precision, video_filter=vf)
        assert torch.equal(s, s0) and torch.equal(i, i0)
        s, i, d = _rank(case, head, precision, video_filter=vf, return_detail=True)
        assert torch.equal(s, s0) and torch.equal(i, i0) and _same_detail(d, d0)


def _filters(seed):
    """name -> (words, allowed (M, Nv) bool): per-query random (half, and rows with at most Kc allowed videos),
    one shared random row, per-query deny lists of 100 ids."""
    from dkd_b200 import engine
    rng = np.random.default_rng(seed)
    half = rng.random((M, Nv)) < 0.5
    few = _allowed_rows(rng, M, Nv, [0, 1, K - 1, K, K + 1, 100, 128, 129, 200, Nv])
    shared = rng.random((1, Nv)) < 0.4
    deny = [list(rng.permutation(Nv)[:100]) for _ in range(M)]
    denied = np.ones((M, Nv), bool)
    for m, ids in enumerate(deny):
        denied[m, ids] = False
    return {"half": (_words(half), half), "few": (_words(few), few),
            "shared": (_words(shared), np.broadcast_to(shared, (M, Nv))),
            "deny": (engine.make_video_filter(Nv, deny=deny), denied)}


_DENSE = {}


def _dense_exact(case, head):
    key = (case["nb"], head)
    if key not in _DENSE:
        _DENSE[key] = _rank(case, head, "exact", return_dense=True)[2].cpu().numpy()
    return _DENSE[key]


@pytest.mark.parametrize("head,precision", ROUTES)
def test_filtered_rank_equals_the_filtered_exact_ranking(case, head, precision):
    fused = _dense_exact(case, head)
    for name, (vf, allowed) in _filters(7).items():
        s_ex, i_ex = _rank(case, head, "exact", video_filter=vf)
        ref_s, ref_i = _np_topk(fused, allowed, K)
        assert np.array_equal(i_ex.cpu().numpy(), ref_i), name
        assert np.array_equal(s_ex.cpu().numpy(), ref_s), name
        s, i = _rank(case, head, precision, video_filter=vf)
        assert torch.equal(i, i_ex) and torch.equal(s, s_ex), name
        ids = i.cpu().numpy()
        m = np.arange(M)[:, None].repeat(K, 1)
        assert allowed[m, np.maximum(ids, 0)][ids >= 0].all(), name
        s, i, det = _rank(case, head, precision, video_filter=vf, return_detail=True)
        assert torch.equal(i, i_ex) and torch.equal(s, s_ex), name
        assert np.array_equal(_refuse(det, head, case["nb"]), s.cpu().numpy()), name
        assert (det.arg[i < 0] == -1).all(), name


@pytest.mark.parametrize("head", ["frame", "two_scale"])
@pytest.mark.parametrize("certify", [True, "deferred"])
def test_certificate_with_a_filter(case, head, certify):
    """Kc = K leaves no candidate margin, so the certificate fires; the re-rank uses the re-ranked queries' rows.
    Queries with at most Kc allowed videos have all of them as candidates and do not count as fallbacks."""
    from dkd_b200 import engine
    filters = _filters(11)
    for name in ("half", "deny", "shared"):
        vf = filters[name][0]
        s_ex, i_ex, d_ex = _rank(case, head, "exact", video_filter=vf, return_detail=True)
        engine.STATS["certify_fallback_queries"] = 0
        s, i, d = _rank(case, head, "bf16", Kc=K, certify=certify, video_filter=vf, return_detail=True)
        if certify == "deferred":
            engine.finish()
        assert engine.STATS["certify_fallback_queries"] > 0, name
        assert torch.equal(i, i_ex) and torch.equal(s, s_ex) and _same_detail(d, d_ex), name
    few = _allowed_rows(np.random.default_rng(12), M, Nv, [0, 1, K - 1, K])
    vf = _words(few)
    s_ex, i_ex = _rank(case, head, "exact", video_filter=vf)
    engine.STATS["certify_fallback_queries"] = 0
    s, i = _rank(case, head, "bf16", Kc=K, certify=certify, video_filter=vf)
    if certify == "deferred":
        engine.finish()
    assert engine.STATS["certify_fallback_queries"] == 0
    assert torch.equal(i, i_ex) and torch.equal(s, s_ex)


def test_rank_rejects_a_filter_of_the_wrong_shape(case):
    from dkd_b200 import _lib
    vf, _ = _filters(13)["half"]
    with pytest.raises(ValueError):
        _rank(case, "two_scale", "bf16", video_filter=vf[:3])
    with pytest.raises(_lib.DkdError):
        _rank(case, "two_scale", "bf16", video_filter=vf[:, :-1].contiguous())


# ---------------------------------------------------------------------------------------------------- shards, streams
@pytest.mark.parametrize("head,precision", [("two_scale", "bf16"), ("frame", "bf16"), ("two_scale", "exact")])
def test_shards_with_unaligned_id_base_merge_to_the_filtered_ranking(case, head, precision):
    from dkd_b200 import engine, ops
    cut = 147                                                          # shard 1 starts at a bit in the middle of a word
    frames = [f.cuda() for f in case["frames"]]
    mask = case["mask"].cuda()
    shards = [engine.prepare_corpus([f[lo:hi] for f in frames], mask[lo:hi], case["prm"], heads=(head,),
                                    precisions=("exact", precision), id_base=lo) for lo, hi in ((0, cut), (cut, Nv))]
    nb, two = case["nb"], head != "frame"
    for name in ("half", "shared", "deny"):
        vf = _filters(17)[name][0]
        s_r, i_r, d_r = _rank(case, head, precision, video_filter=vf, return_detail=True)
        outs = [engine.rank(pc, case["pq"], K=K, head=head, precision=precision, video_filter=vf, return_detail=True)
                for pc in shards]
        s, i = ops.merge_topk(torch.stack([o[0] for o in outs]), torch.stack([o[1] for o in outs]))
        assert torch.equal(i, i_r) and torch.equal(s, s_r), name
        s, i, w = ops.merge_topk_payload(torch.stack([o[0] for o in outs]), torch.stack([o[1] for o in outs]),
                                         torch.stack([o[2].pack() for o in outs]),
                                         engine.HitDetail.pad_words(nb, two, "cuda"))
        assert torch.equal(i, i_r) and torch.equal(s, s_r) and torch.equal(w, d_r.pack()), name


@pytest.mark.parametrize("head,precision", [("two_scale", "bf16"), ("frame", "bf16"), ("two_scale", "exact")])
def test_streamed_filtered_ranking_equals_resident(case, head, precision):
    from dkd_b200 import engine
    frames = [f.cuda() for f in case["frames"]]
    pqs = engine.split_queries([q.cuda() for q in case["qs"]], batch=24)          # 24 + 24 + 16 queries
    assert len(pqs) == 3
    for name in ("half", "shared", "deny"):
        vf = _filters(19)[name][0]
        s_r, i_r, d_r = _rank(case, head, precision, video_filter=vf, return_detail=True)
        chunks = engine.iter_chunks(frames, case["mask"].cuda(), chunk_videos=70)
        s, i = engine.rank_streamed(chunks, pqs, case["prm"], K=K, head=head, precision=precision, video_filter=vf)
        assert torch.equal(i, i_r) and torch.equal(s, s_r), name
        chunks = engine.iter_chunks(frames, case["mask"].cuda(), chunk_videos=70)
        s, i, d = engine.rank_streamed(chunks, pqs, case["prm"], K=K, head=head, precision=precision,
                                       video_filter=vf, return_detail=True)
        assert torch.equal(i, i_r) and torch.equal(s, s_r) and _same_detail(d, d_r), name


@pytest.mark.parametrize("scoring", ["frame", "two_scale"])
def test_rank_queries_with_a_filter_equals_engine_rank(ops, dkd, scoring):
    from dkd_b200 import engine, eval as E
    from tests.test_gpu_dropin import _tiny_setup
    _, m, vset, qset, opt = _tiny_setup(dkd)
    opt.scoring, opt.precision, opt.query_chunk = scoring, "bf16", 7
    ctx = E.compute_context_info(m, vset, opt)
    qs, metas, _ = E._encode_all_queries(m, qset, opt)
    Nq, Nt, Kt = len(qset), len(vset), 5
    rng = np.random.default_rng(23)
    vf = _words(rng.random((Nq, Nt)) < 0.6)
    s, i, metas2 = E.rank_queries(m, qset, opt, ctx, K=Kt, video_filter=vf)
    assert metas2 == metas and Nq > opt.query_chunk
    pq = engine.prepare_queries(qs)
    s_r, i_r = engine.rank(ctx["prepared"], pq, K=Kt, head=scoring, precision="bf16", w_clip=m.clip_scale_w,
                           w_frame=m.frame_scale_w, video_filter=vf)
    assert torch.equal(i, i_r) and torch.equal(s, s_r)
    s_ex, i_ex = engine.rank(ctx["prepared"], pq, K=Kt, head=scoring, precision="exact", w_clip=m.clip_scale_w,
                             w_frame=m.frame_scale_w, video_filter=vf)
    assert torch.equal(i, i_ex)


# ---------------------------------------------------------------------------------------------------- call record
def test_no_new_entry_point_without_a_filter(case, monkeypatch):
    from dkd_b200 import _lib, engine
    vf = engine.make_video_filter(Nv, deny=[[n % Nv, (7 * n) % Nv] for n in range(M)])
    calls = []
    real = _lib.call

    def record(name, *args):
        calls.append(name)
        return real(name, *args)

    monkeypatch.setattr(_lib, "call", record)
    for head, precision in ROUTES:
        _rank(case, head, precision)
        _rank(case, head, precision, Kc=K, certify=True)
        _rank(case, head, precision, return_detail=True)
    assert calls and not NEW_ENTRIES & set(calls)
    calls.clear()
    for head, precision in ROUTES:
        _rank(case, head, precision, video_filter=vf)
    assert {"dkd_topk_filtered", "dkd_select_topk_filtered"} <= set(calls)
    assert not {"dkd_topk", "dkd_select_topk"} & set(calls)

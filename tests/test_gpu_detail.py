"""The per-hit detail of the ranking (engine.rank(return_detail=True) -> engine.HitDetail): key clip or best frame and
per-branch scores of every returned hit, produced where the hit's score is produced and moved with it through every
sort and merge.

Checked on every route a hit can take (dense exact, candidate rescoring for bf16 / fp16 / shortcut, the certificate's
exact re-rank, immediate and deferred, the streamed chunk fold) and for one- and two-branch models:
  - asking for the detail leaves (scores, ids) bit-identical;
  - the detail of the approximate paths equals the exact path's bit for bit;
  - the fused score recomputed from the detail in numpy float32, in the kernels' rounding order, is the returned score;
  - key clips / best frames are the oracle's first argmax outside its own fp32 ties, scores within 2e-6;
  - exact ties: a window with an identical later copy is reported as the first copy;
  - the payload sort / merge kernels against a numpy reference;
  - return_detail=False calls none of the new entry points.
"""
import numpy as np
import pytest
import torch

from oracle import oracle as O
from tests import synth

pytestmark = pytest.mark.gpu

FP32_TOL = 2e-6
Nv, L, D, M, K = 300, 96, 128, 64, 32
ROUTES = [("frame", "exact"), ("frame", "bf16"), ("frame", "fp16"), ("two_scale", "exact"), ("two_scale", "bf16"),
          ("two_scale", "fp16"), ("two_scale", "shortcut")]
NEW_ENTRIES = {"dkd_frame_fuse_csr_detail", "dkd_scatter_fuse_detail", "dkd_sort_candidates_payload",
               "dkd_merge_topk_payload"}
_CASES = {}


def _params(nb, seed):
    g = torch.Generator().manual_seed(seed)
    return [(0.05 * torch.randn(D, D, generator=g), 0.01 * torch.randn(D, generator=g),
             0.05 * torch.randn(D, D, generator=g), 0.01 * torch.randn(D, generator=g)) for _ in range(nb)]


def _build(nb):
    """Ragged corpus, L < 128, many videos shorter than 32 frames (lengths 5 .. 96), nb branches, both heads."""
    from dkd_b200 import engine
    frames, mask, lengths = synth.encoded_corpus(Nv, L, D, seed=31, min_len=5, shared=1.5)
    fr = [frames] + [synth.encoded_corpus(Nv, L, D, seed=32 + b, min_len=5, shared=1.5)[0] * mask[:, :, None]
                     for b in range(1, nb)]
    params = _params(nb, 41)
    qs = [synth.encoded_queries(M, D, seed=50 + b) for b in range(nb)]
    dev = torch.device("cuda")
    prm = [tuple(t.to(dev) for t in p) for p in params]
    pc = engine.prepare_corpus([f.to(dev) for f in fr], mask.to(dev), prm, heads=("frame", "two_scale"),
                               precisions=("exact", "bf16", "fp16", "shortcut"))
    pq = engine.prepare_queries([q.to(dev) for q in qs])
    assert int((lengths < 32).sum()) > 20
    return dict(nb=nb, frames=fr, mask=mask, lengths=lengths, params=params, prm=prm, qs=qs, pc=pc, pq=pq)


@pytest.fixture(scope="module", params=[1, 2], ids=["1branch", "2branch"])
def case(request, ops):
    nb = request.param
    if nb not in _CASES:
        _CASES[nb] = _build(nb)
    return _CASES[nb]


def _rank(case, head, precision, **kw):
    from dkd_b200 import engine
    return engine.rank(case["pc"], case["pq"], K=K, head=head, precision=precision, **kw)


def _refuse(det, head, nb):
    """The fused score from the detail in numpy float32: fuse_branch per branch, then the sum over branches in order
    (two-scale); fl(0.7 a) + fl(0.3 b) (frame head)."""
    a = det.score.cpu().numpy()
    f32 = np.float32
    if head == "frame":
        return a[..., 0] if nb == 1 else f32(0.7) * a[..., 0] + f32(0.3) * a[..., 1]
    fr = det.frame.cpu().numpy()
    wbs = (0.7, 0.3) if nb == 2 else (1.0,)
    tot = None
    for b in range(nb):
        v = f32(wbs[b]) * (f32(0.7) * a[..., b] + f32(0.3) * fr[..., b])
        tot = v if tot is None else tot + v
    return tot


def _same_detail(a, b):
    same = torch.equal(a.arg, b.arg) and torch.equal(a.score.view(torch.int32), b.score.view(torch.int32))
    if a.frame is not None or b.frame is not None:
        same = same and torch.equal(a.frame.view(torch.int32), b.frame.view(torch.int32))
    return same


@pytest.mark.parametrize("head,precision", ROUTES)
def test_detail_leaves_ranking_unchanged_and_recomputes_the_score(case, head, precision):
    nb = case["nb"]
    s0, i0 = _rank(case, head, precision)
    s1, i1, det = _rank(case, head, precision, return_detail=True)
    assert torch.equal(s0, s1) and torch.equal(i0, i1)
    assert det.arg.shape == (M, K, nb) and det.arg.dtype == torch.int32
    assert det.score.shape == (M, K, nb) and det.score.dtype == torch.float32
    assert (det.frame is None) == (head == "frame")
    hi = L if head == "frame" else O.num_proposals(32)
    assert int(det.arg.min()) >= 0 and int(det.arg.max()) < hi
    assert np.array_equal(_refuse(det, head, nb), s1.cpu().numpy())
    # return_dense + return_detail: the detail comes last
    out = _rank(case, head, precision, return_dense=True, return_detail=True)
    assert len(out) == 4 and out[2].shape == (M, Nv) and _same_detail(out[3], det)


@pytest.mark.parametrize("head,precision", [("frame", "bf16"), ("two_scale", "bf16"), ("two_scale", "fp16")])
def test_detail_of_the_unrescored_dense_route_recomputes_the_score(case, head, precision):
    """rescore=False returns the approximate dense scores: the detail is the approximate pass's, consistently."""
    s, i, det = _rank(case, head, precision, rescore=False, return_detail=True)
    assert np.array_equal(_refuse(det, head, case["nb"]), s.cpu().numpy())


@pytest.mark.parametrize("head,precision", [r for r in ROUTES if r[1] != "exact"])
def test_approximate_paths_give_the_exact_detail(case, head, precision):
    s_ex, i_ex, d_ex = _rank(case, head, "exact", return_detail=True)
    s, i, d = _rank(case, head, precision, return_detail=True)
    assert torch.equal(i, i_ex) and torch.equal(s, s_ex)
    assert _same_detail(d, d_ex)


def _oracle(case):
    if "oracle" not in case:
        nb, mask = case["nb"], case["mask"]
        props, keys, vals = O.two_scale_corpus(case["frames"], mask, case["params"])
        det = O.two_scale_eval_detail(case["qs"], props, keys, vals, mask)
        frame = [O.two_scale_branch(q, f, mask, *p)["frame"].numpy()
                 for q, f, p in zip(case["qs"], case["frames"], case["params"])]
        fh = [O.get_sim_scores(q, f, mask) for q, f in zip(case["qs"], case["frames"])]
        fh_tie = None
        for _, rows, _ in fh:
            top2 = torch.topk(rows, 2, dim=1).values
            t = ((top2[:, 0] - top2[:, 1]) <= FP32_TOL).numpy()
            fh_tie = t if fh_tie is None else fh_tie | t
        case["oracle"] = dict(
            two_scale=dict(arg=det["key_clip"], score=det["clip"], frame=frame, tie=det["tie"]),
            frame=dict(arg=[a.numpy() for _, _, a in fh], score=[s.numpy() for s, _, _ in fh], frame=None, tie=fh_tie))
        assert nb == len(frame)
    return case["oracle"]


@pytest.mark.parametrize("head,precision", ROUTES)
def test_detail_against_the_oracle(case, head, precision):
    ref = _oracle(case)[head]
    _, ids, det = _rank(case, head, precision, return_detail=True)
    ids = ids.cpu().numpy().astype(np.int64)
    m = np.arange(M)[:, None].repeat(K, 1)
    clear = ~ref["tie"][m, ids]
    # videos shorter than 32 frames repeat frames into identical clips, hence identical windows that tie exactly in
    # the oracle: about a quarter of the two-scale hits of this corpus sit on such ties (first-window rule: see
    # test_exact_ties_report_the_first_window and tests/test_gpu_ties.py)
    assert clear.mean() > 0.5
    for b in range(case["nb"]):
        arg = det.arg[..., b].cpu().numpy()
        key_ok = arg == ref["arg"][b][m, ids]
        assert key_ok[clear].all(), f"branch {b}: {int((~key_ok[clear]).sum())} hits off the oracle's first argmax"
        assert np.abs(det.score[..., b].cpu().numpy() - ref["score"][b][m, ids]).max() <= FP32_TOL
        if ref["frame"] is not None:
            err = np.abs(det.frame[..., b].cpu().numpy() - ref["frame"][b][m, ids])[key_ok]
            assert err.max() <= FP32_TOL, f"frame-scale error {err.max():.3g}"


# ---------------------------------------------------------------------------------------- exact ties, two-scale head
def _unit(v):
    return v / v.norm(dim=-1, keepdim=True)


def _tie_frames(Nv_, Dt, seed):
    """Videos of exactly 32 frames, so that clip i is frame i (average_to_fixed_length with n = T).  Video n carries
    one strong window and an identical later copy: even n a single clip (w = 1), odd n a 3-clip pattern (w = 3); every
    other clip is anti-aligned with the queries.  Returns (frames (Nv, 32, D), expected first window, later copy)."""
    g = torch.Generator().manual_seed(seed)
    T = 32
    e = torch.eye(Dt)
    x = torch.empty(Nv_, T, Dt)
    first, copy = [], []
    for n in range(Nv_):
        for i in range(T):
            w = torch.randn(Dt, generator=g)
            w[:4] = 0.0
            x[n, i] = (-0.5 * e[0] + 0.85 * _unit(w)) * (1.0 + torch.rand(1, generator=g))
        s = int(torch.randint(0, T - 10, (1,), generator=g))
        if n % 2 == 0:
            s2 = s + 2 + int(torch.randint(0, T - s - 2, (1,), generator=g))
            x[n, s] = 0.9 * e[0] + 0.43 * e[1]
            x[n, s2] = x[n, s]
            first.append(O.proposal_index(1, s, T))
            copy.append(O.proposal_index(1, s2, T))
        else:
            s2 = s + 4 + int(torch.randint(0, T - s - 6, (1,), generator=g))
            for j in range(3):
                x[n, s + j] = 0.7 * e[0] + 0.714 * e[1 + j]
                x[n, s2 + j] = x[n, s + j]
            first.append(O.proposal_index(3, s, T))
            copy.append(O.proposal_index(3, s2, T))
    return x.contiguous(), torch.tensor(first), torch.tensor(copy)


def test_exact_ties_report_the_first_window(ops):
    from dkd_b200 import engine
    Nt, Dt, Mt, Kt = 30, 128, 40, 10
    frames, first, copy = _tie_frames(Nt, Dt, seed=5)
    mask = torch.ones(Nt, 32)
    g = torch.Generator().manual_seed(6)
    q = torch.zeros(Mt, Dt)
    q[:, 0] = 1.0
    q = _unit(q + 0.01 * torch.randn(Mt, Dt, generator=g))
    # the oracle agrees that the first window is one of the maxima, and that every pair is a tie
    props = O.build_proposals(O.downsample_clips(frames, torch.full((Nt,), 32), 32))
    _, allp, _ = O.clip_scale_scores(q, props)
    top2 = torch.topk(allp, 2, dim=1).values
    assert float((top2[:, 0] - top2[:, 1]).max()) <= 1e-6
    at_first = allp.gather(1, first[None, None, :].expand(Mt, 1, Nt)).squeeze(1)
    assert float((top2[:, 0] - at_first).max()) <= 1e-6
    prm = [tuple(t.cuda() for t in p) for p in _params(1, 7)]
    pc = engine.prepare_corpus([frames.cuda()], mask.cuda(), prm, heads=("two_scale",),
                               precisions=("exact", "bf16", "fp16", "shortcut"))
    pq = engine.prepare_queries([q.cuda()])
    s_ex, i_ex, d_ex = engine.rank(pc, pq, K=Kt, head="two_scale", precision="exact", return_detail=True)
    ids = i_ex.long().cpu()
    for prec in ("exact", "shortcut", "bf16", "fp16"):
        s, i, d = engine.rank(pc, pq, K=Kt, head="two_scale", precision=prec, return_detail=True)
        assert torch.equal(i, i_ex) and torch.equal(s, s_ex), prec
        arg = d.arg[..., 0].long().cpu()
        assert np.array_equal(_refuse(d, "two_scale", 1), s.cpu().numpy()), prec
        if prec in ("exact", "shortcut"):
            assert torch.equal(arg, first[ids]), prec
            assert _same_detail(d, d_ex), prec
        else:
            # the known-key residual (DESIGN §2): a maximal window, i.e. the first window or its identical copy, with
            # the exact maximum as its clip score
            assert ((arg == first[ids]) | (arg == copy[ids])).all(), prec
            assert torch.equal(d.score, d_ex.score), prec


# ---------------------------------------------------------------------------------------- certificate fallback, stream
@pytest.mark.parametrize("head", ["frame", "two_scale"])
@pytest.mark.parametrize("certify", [True, "deferred"])
def test_fallback_patches_the_detail(case, head, certify):
    """Kc = K leaves no candidate margin, so the certificate fires; the re-ranked rows carry the exact detail."""
    from dkd_b200 import engine
    s_ex, i_ex, d_ex = _rank(case, head, "exact", return_detail=True)
    engine.STATS["certify_fallback_queries"] = 0
    s, i, d = _rank(case, head, "bf16", Kc=K, certify=certify, return_detail=True)
    if certify == "deferred":
        engine.finish()
    assert engine.STATS["certify_fallback_queries"] > 0
    assert torch.equal(i, i_ex) and torch.equal(s, s_ex)
    assert _same_detail(d, d_ex)


@pytest.mark.parametrize("head,precision", [("two_scale", "bf16"), ("frame", "bf16"), ("two_scale", "exact")])
def test_streamed_detail_equals_resident(case, head, precision):
    from dkd_b200 import engine
    s_r, i_r, d_r = _rank(case, head, precision, return_detail=True)
    frames = [f.cuda() for f in case["frames"]]
    for chunk in (70, 128):
        chunks = engine.iter_chunks(frames, case["mask"].cuda(), chunk_videos=chunk)
        s, i, d = engine.rank_streamed(chunks, [case["pq"]], case["prm"], K=K, head=head, precision=precision,
                                       return_detail=True)
        assert torch.equal(i, i_r) and torch.equal(s, s_r), chunk
        assert _same_detail(d, d_r), chunk


# ---------------------------------------------------------------------------------------- empty inputs, call record
@pytest.mark.parametrize("head", ["frame", "two_scale"])
def test_empty_queries_and_empty_shard_give_padding_detail(ops, case, head):
    from dkd_b200 import engine
    nb = case["nb"]
    pq0 = engine.prepare_queries([q[:0].cuda() for q in case["qs"]])
    s, i, d = engine.rank(case["pc"], pq0, K=K, head=head, precision="bf16", return_detail=True)
    assert d.arg.shape == (0, K, nb) and d.score.shape == (0, K, nb)
    empty = engine.prepare_corpus([f[:0].cuda() for f in case["frames"]], case["mask"][:0].cuda(), case["prm"],
                                  heads=(head,), id_base=Nv)
    s, i, d = engine.rank(empty, case["pq"], K=K, head=head, precision="bf16", return_detail=True)
    assert (i == -1).all() and (d.arg == -1).all() and torch.isneginf(d.score).all()
    assert (d.frame is None) if head == "frame" else torch.isneginf(d.frame).all()
    # merging the empty shard's padding with a real shard: no padding survives, the real detail is kept
    s_r, i_r, d_r = _rank(case, head, "bf16", return_detail=True)
    pad = engine.HitDetail.pad_words(nb, head != "frame", "cuda")
    ms, mi, mw = ops.merge_topk_payload(torch.stack([s, s_r]), torch.stack([i, i_r]),
                                        torch.stack([d.pack(), d_r.pack()]), pad)
    assert torch.equal(mi, i_r) and torch.equal(ms, s_r) and torch.equal(mw, d_r.pack())


def test_no_new_entry_point_without_detail(case, monkeypatch):
    from dkd_b200 import _lib
    calls = []
    real = _lib.call

    def record(name, *args):
        calls.append(name)
        return real(name, *args)

    monkeypatch.setattr(_lib, "call", record)
    for head, precision in ROUTES:
        _rank(case, head, precision)
        _rank(case, head, precision, Kc=K, certify=True)
    assert calls and not NEW_ENTRIES & set(calls)
    calls.clear()
    for head, precision in ROUTES:
        _rank(case, head, precision, return_detail=True)
    assert {"dkd_sort_candidates_payload", "dkd_frame_fuse_csr_detail", "dkd_scatter_fuse_detail"} <= set(calls)


# ---------------------------------------------------------------------------------------- payload sort / merge kernels
def _np_ranked(s, i, w, K_out, C):
    """(score desc, id asc) of the valid entries (id >= 0) of one query, the first K_out, padded (-inf, -1, pad -7)."""
    keep = i >= 0
    s, i, w = s[keep], i[keep], w[keep]
    order = np.lexsort((i, -s))[:K_out]
    out_s = np.full(K_out, -np.inf, np.float32)
    out_i = np.full(K_out, -1, np.int32)
    out_w = np.full((K_out, C), -7, np.int32)
    out_s[: len(order)], out_i[: len(order)], out_w[: len(order)] = s[order], i[order], w[order]
    return out_s, out_i, out_w


def _lists(rng, rows, n, pad_frac):
    """rows x n entries: distinct ids per row, scores drawn from few values (exact ties across ids), some padding."""
    ids = np.stack([rng.permutation(4 * n)[:n] for _ in range(rows)]).astype(np.int32)
    ids[rng.random((rows, n)) < pad_frac] = -1
    scores = (rng.integers(-6, 7, (rows, n)) / 8.0).astype(np.float32)
    return scores, ids


@pytest.mark.parametrize("Kin,K_out", [(1, 1), (37, 20), (128, 100), (256, 256), (512, 100)])
@pytest.mark.parametrize("C", [1, 6])
def test_sort_candidates_payload_against_numpy(ops, Kin, K_out, C):
    rng = np.random.default_rng(Kin * 10 + C)
    Mq = 45
    s, i = _lists(rng, Mq, Kin, 0.2)
    w = rng.integers(-2 ** 31, 2 ** 31 - 1, (Mq, Kin, C), dtype=np.int64).astype(np.int32)
    cs, ci, cw = torch.from_numpy(s).cuda(), torch.from_numpy(i).cuda(), torch.from_numpy(w).cuda()
    pad = torch.full((C,), -7, dtype=torch.int32)
    os_, oi, ow = ops.sort_candidates_payload(cs, ci, cw, K_out, pad)
    rs, ri = ops.sort_candidates(cs, ci, K_out)
    assert torch.equal(os_, rs) and torch.equal(oi, ri)
    for m in range(Mq):
        es, ei, ew = _np_ranked(s[m], i[m], w[m], K_out, C)
        assert np.array_equal(oi[m].cpu().numpy(), ei) and np.array_equal(os_[m].cpu().numpy(), es)
        assert np.array_equal(ow[m].cpu().numpy(), ew), m


@pytest.mark.parametrize("G", [1, 2, 3, 8])
@pytest.mark.parametrize("Kl", [1, 37, 100, 256])
@pytest.mark.parametrize("C", [1, 6])
def test_merge_topk_payload_against_numpy(ops, G, Kl, C):
    rng = np.random.default_rng(G * 1000 + Kl * 10 + C)
    Mq = 29
    s, i = _lists(rng, Mq, G * Kl, 0.25)           # distinct ids per query across all G lists
    s = s.reshape(Mq, G, Kl).transpose(1, 0, 2).copy()
    i = i.reshape(Mq, G, Kl).transpose(1, 0, 2).copy()
    i[-1, 3] = -1                                    # a query whose last list is all padding
    w = rng.integers(-2 ** 31, 2 ** 31 - 1, (G, Mq, Kl, C), dtype=np.int64).astype(np.int32)
    gs, gi, gw = torch.from_numpy(s).cuda(), torch.from_numpy(i).cuda(), torch.from_numpy(w).cuda()
    pad = torch.full((C,), -7, dtype=torch.int32)
    ms, mi, mw = ops.merge_topk_payload(gs, gi, gw, pad)
    rs, ri = ops.merge_topk(gs, gi)
    assert torch.equal(ms, rs) and torch.equal(mi, ri)
    for m in range(Mq):
        es, ei, ew = _np_ranked(s[:, m].reshape(-1), i[:, m].reshape(-1), w[:, m].reshape(-1, C), Kl, C)
        assert np.array_equal(mi[m].cpu().numpy(), ei) and np.array_equal(ms[m].cpu().numpy(), es)
        assert np.array_equal(mw[m].cpu().numpy(), ew), m


def test_moment_frames_of_ranked_hits(case):
    """engine.moment_frames on the device equals the same call on the host, and every window lies inside its video."""
    from dkd_b200 import engine
    _, ids, det = _rank(case, "two_scale", "bf16", return_detail=True)
    lengths = case["lengths"].int()
    win = engine.moment_frames(det.arg, ids, lengths.cuda())
    host = engine.moment_frames(det.arg.cpu(), ids.cpu(), lengths)
    assert win.shape == (M, K, case["nb"], 2) and torch.equal(win.cpu(), host)
    n = lengths[ids.long().cpu()].unsqueeze(-1)
    assert (host[..., 0] >= 0).all() and (host[..., 0] < host[..., 1]).all() and (host[..., 1] <= n).all()
    _, fids, fdet = _rank(case, "frame", "bf16", return_detail=True)
    fw = engine.moment_frames(fdet.arg, fids, lengths.cuda(), head="frame").cpu()
    assert torch.equal(fw[..., 1] - fw[..., 0], torch.ones_like(fw[..., 0]))
    assert (fw[..., 1] <= lengths[fids.long().cpu()].unsqueeze(-1)).all()

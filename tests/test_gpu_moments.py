"""Moment localization (engine.localize -> engine.Moments): the top-m non-overlapping clip windows of every ranked hit,
from the exact clip-scale curve.

  - dkd_clip_dots_list gives float64-grade per-clip dots, and a numpy float32 window scan of them reproduces
    clip_score_f32's max / first argmax bit for bit;
  - dkd_moment_nms on arbitrary dots and scales is bit-identical to a numpy float32 reference (random curves, exact ties,
    negative curves, whole-video picks at iou = 0, T = 32 and 16);
  - end to end on rank(return_detail=True): with one branch moment 0 is the hit's key clip and clip score; every moment
    is the oracle's fused clip-scale score at its window within 2e-6, moments respect the IoU bound and are ranked;
  - shards, padding, moment_frames on (M, K, m) args, and the entry points localize calls.
"""
import numpy as np
import pytest
import torch

from oracle import oracle as O
from tests import synth

pytestmark = pytest.mark.gpu

FP32_TOL = 2e-6
Nv, L, D, M, K = 300, 96, 128, 64, 32
PRECISIONS = ["exact", "bf16", "shortcut"]
_CASES = {}


def _params(nb, seed):
    g = torch.Generator().manual_seed(seed)
    return [(0.05 * torch.randn(D, D, generator=g), 0.01 * torch.randn(D, generator=g),
             0.05 * torch.randn(D, D, generator=g), 0.01 * torch.randn(D, generator=g)) for _ in range(nb)]


def _build(nb):
    """Ragged corpus, many videos shorter than 32 frames (lengths 5 .. 96), nb branches, two-scale head."""
    from dkd_b200 import engine
    frames, mask, lengths = synth.encoded_corpus(Nv, L, D, seed=61, min_len=5, shared=1.5)
    fr = [frames] + [synth.encoded_corpus(Nv, L, D, seed=62 + b, min_len=5, shared=1.5)[0] * mask[:, :, None]
                     for b in range(1, nb)]
    params = _params(nb, 71)
    qs = [synth.encoded_queries(M, D, seed=80 + b) for b in range(nb)]
    dev = torch.device("cuda")
    prm = [tuple(t.to(dev) for t in p) for p in params]
    pc = engine.prepare_corpus([f.to(dev) for f in fr], mask.to(dev), prm, heads=("two_scale",),
                               precisions=("exact", "bf16", "shortcut"))
    pq = engine.prepare_queries([q.to(dev) for q in qs])
    assert int((lengths < 32).sum()) > 20
    return dict(nb=nb, frames=fr, mask=mask, lengths=lengths, params=params, prm=prm, qs=qs, pc=pc, pq=pq)


@pytest.fixture(scope="module", params=[1, 2], ids=["1branch", "2branch"])
def case(request, ops):
    nb = request.param
    if nb not in _CASES:
        _CASES[nb] = _build(nb)
    return _CASES[nb]


# ---------------------------------------------------------------------------------------------- numpy references
def _windows(T):
    """(w, s) of every proposal p, as int arrays (P,)."""
    ws = np.array([O.proposal_index(w, s, T) for w in range(1, T + 1) for s in range(T - w + 1)])
    assert np.array_equal(ws, np.arange(len(ws)))
    w = np.array([w for w in range(1, T + 1) for s in range(T - w + 1)])
    s = np.array([s for w in range(1, T + 1) for s in range(T - w + 1)])
    return w, s


def np_curve(dots, scale, T):
    """dots (E, 32) fp32, scale (E, P) fp32 -> (E, P) fp32: fl(sequential window sum * scale), the kernels' order."""
    E = dots.shape[0]
    out = np.empty((E, T * (T + 1) // 2), np.float32)
    for s in range(T):
        run = dots[:, s].copy()
        for w in range(1, T - s + 1):
            if w > 1:
                run = run + dots[:, s + w - 1]
            p = O.proposal_index(w, s, T)
            out[:, p] = run * scale[:, p]
    return out


def np_fuse(curves):
    if len(curves) == 1:
        return curves[0]
    return np.float32(0.7) * curves[0] + np.float32(0.3) * curves[1]


def np_iou(w1, s1, w2, s2):
    """fl(inter / union) on clip intervals [s, s + w), float32, elementwise."""
    inter = np.maximum(0, np.minimum(s1 + w1, s2 + w2) - np.maximum(s1, s2))
    union = w1 + w2 - inter
    return inter.astype(np.float32) / union.astype(np.float32)


def np_nms(curve, T, m, iou):
    """Greedy NMS of every row of curve (E, P) fp32 -> (arg (E, m) int32, score (E, m) fp32), padding (-1, -inf)."""
    E, P = curve.shape
    w, s = _windows(T)
    alive = np.ones((E, P), bool)
    arg = np.full((E, m), -1, np.int32)
    score = np.full((E, m), -np.inf, np.float32)
    rows = np.arange(E)
    for j in range(m):
        has = alive.any(axis=1)
        best = np.argmax(np.where(alive, curve, -np.inf), axis=1)       # first maximum: the lower p on ties
        arg[has, j] = best[has]
        score[has, j] = curve[rows, best][has]
        sup = np_iou(w[None, :], s[None, :], w[best][:, None], s[best][:, None]) > np.float32(iou)
        alive &= ~sup
        alive[rows, best] = False
    return arg, score


def _entry_video(vid_ptr):
    """Video of every CSR entry e < vid_ptr[-1]."""
    vp = vid_ptr.cpu().numpy().astype(np.int64)
    return np.repeat(np.arange(len(vp) - 1), np.diff(vp))


# ---------------------------------------------------------------------------------------------- dots pass
def test_clip_dots_list_is_exact_and_reproduces_the_clip_score(case, ops):
    from dkd_b200 import engine
    pc, pq = case["pc"], case["pq"]
    _, ids, _ = engine.rank(pc, pq, K=K, precision="bf16", return_detail=True)
    ids = ids.clone()
    ids[3, :5] = ids[3, 7]                                          # duplicates are separate entries
    csr = ops.candidates_to_csr(ids, pc.Nv, pc.id_base)
    vids = _entry_video(csr[0])
    E = len(vids)
    assert E == M * K
    q_list = csr[1].cpu().numpy()[:E]
    for b, (bd, qn) in enumerate(zip(pc.branches, pq.qn)):
        dots = ops.clip_dots_list(qn, bd.clip_planes, csr)
        assert dots.shape == (M * K, 32)
        got = dots[:E].cpu().numpy()
        q64 = qn.double().cpu().numpy()
        c64 = bd.clips.double().cpu().numpy()
        ref = np.einsum("ed,eid->ei", q64[q_list], c64[vids])
        # clips are means of un-normalised frames: the error bound is 2e-6 on the cosine scale, i.e. x |qn| |clip|
        scale = np.maximum(np.linalg.norm(c64, axis=-1), 1.0)[vids]
        assert (np.abs(got - ref) / scale).max() <= FP32_TOL, b
        sc = bd.prop_scale.cpu().numpy()[vids]
        curve = np_curve(got, sc, 32)
        smax, sarg = ops.clip_score_f32(qn, bd.clip_planes, bd.prop_scale, csr=csr[:2])
        assert np.array_equal(curve.max(axis=1), smax[:E].cpu().numpy()), b
        assert np.array_equal(np.argmax(curve, axis=1), sarg[:E].cpu().numpy().astype(np.int64)), b


# ---------------------------------------------------------------------------------------------- NMS kernel
def _nms_inputs(T, nb, seed):
    """Ids of 12 videos for 24 queries x 7 ranks (some -1), per branch dots (E, 32) in CSR entry order and prop_scale
    (12, P) with: video 0 scale 1 (positive dots: the whole video is the best window), video 1 a scale that depends on
    w only (periodic dots: exact ties at different starts), others random.  Entry kinds by e % 4: random, negative,
    period 4 with one positive clip per period (the best windows are exact ties of single clips in video 1), positive.
    Videos 0 and 1 have at least 4 entries, so every kind occurs in both."""
    from dkd_b200 import ops
    rng = np.random.default_rng(seed)
    Nv_, M_, K_ = 12, 24, 7
    P = T * (T + 1) // 2
    ids = rng.integers(0, Nv_, (M_, K_)).astype(np.int32)
    ids[rng.random((M_, K_)) < 0.1] = -1
    ids[0, :4] = 0
    ids[1, :4] = 1
    ids[5] = -1                                                      # an all-padding row
    csr = ops.candidates_to_csr(torch.from_numpy(ids).cuda(), Nv_, 0)
    E = int(csr[0][-1])
    w, _ = _windows(T)
    dots, scales = [], []
    for _ in range(nb):
        d = rng.standard_normal((M_ * K_, 32)).astype(np.float32)
        kind = np.arange(M_ * K_) % 4
        d[kind == 1] = -np.abs(d[kind == 1]) - 0.05
        per = -rng.uniform(0.6, 1.0, ((kind == 2).sum(), 4)).astype(np.float32)
        per[:, 0] = rng.uniform(0.5, 1.5, (kind == 2).sum())
        d[kind == 2] = np.tile(per, 8)
        d[kind == 3] = np.abs(d[kind == 3]) + 0.1
        d[:, T:] = 0.0
        sc = rng.uniform(0.5, 2.0, (Nv_, P)).astype(np.float32)
        sc[0] = 1.0
        sc[1] = (1.0 / (w * rng.uniform(0.8, 1.2))).astype(np.float32)
        dots.append(torch.from_numpy(d).cuda())
        scales.append(torch.from_numpy(sc).cuda())
    return ids, csr, E, dots, scales


@pytest.mark.parametrize("T", [32, 16])
@pytest.mark.parametrize("nb", [1, 2])
@pytest.mark.parametrize("m", [1, 5, 16])
@pytest.mark.parametrize("iou", [0.0, 0.3, 0.5, 1.0])
def test_moment_nms_matches_numpy(ops, T, nb, m, iou):
    ids, csr, E, dots, scales = _nms_inputs(T, nb, seed=T * 10 + nb)
    M_, K_ = ids.shape
    arg, score = ops.moment_nms(dots, scales, csr, M_, K_, m, iou)
    assert arg.shape == (M_, K_, m) and score.shape == (M_, K_, m)
    vids = _entry_video(csr[0])
    slot = csr[2][:E].cpu().numpy()
    # the entries' dots are stored in CSR order: dots row e belongs to entry e (the kernel never reads slot for input)
    curves = [np_curve(d.cpu().numpy()[:E], s.cpu().numpy()[vids], T) for d, s in zip(dots, scales)]
    curve = np_fuse(curves)
    ra, rs = np_nms(curve, T, m, iou)
    ga = arg.view(M_ * K_, m).cpu().numpy()
    gs = score.view(M_ * K_, m).cpu().numpy()
    assert np.array_equal(ga[slot], ra)
    assert np.array_equal(gs[slot].view(np.int32), rs.view(np.int32))
    # slots without an entry (id -1) stay padding
    pad = np.ones(M_ * K_, bool)
    pad[slot] = False
    assert pad.sum() == (ids == -1).sum() and (ga[pad] == -1).all() and np.isneginf(gs[pad]).all()
    # the inputs really contain exact ties of the maximum at different windows
    top = curve.max(axis=1, keepdims=True)
    assert ((curve == top).sum(axis=1) > 1).any()
    # iou = 0 and a whole-video pick (positive dots at scale 1): every other window overlaps it, the remaining ranks
    # are padding
    if iou == 0.0 and nb == 1:
        rows = np.nonzero((vids == 0) & (np.arange(E) % 4 == 3))[0]
        assert len(rows)
        assert (ga[slot[rows], 0] == O.proposal_index(T, 0, T)).all()
        assert (ga[slot[rows], 1:] == -1).all() and np.isneginf(gs[slot[rows], 1:]).all()


def test_moment_nms_rejects_bad_arguments(ops):
    from dkd_b200 import _lib
    ids, csr, E, dots, scales = _nms_inputs(32, 1, seed=3)
    for m, iou in ((0, 0.5), (17, 0.5), (5, -0.1), (5, float("nan"))):
        with pytest.raises(_lib.DkdError):
            ops.moment_nms(dots, scales, csr, ids.shape[0], ids.shape[1], m, iou)


# ---------------------------------------------------------------------------------------------- end to end
def _oracle_curves(case):
    """Per branch the oracle's float64 clip-scale cosine of every (query, window, video): (M, P, Nv)."""
    if "oracle" not in case:
        props, _, _ = O.two_scale_corpus(case["frames"], case["mask"], case["params"])
        case["oracle"] = [O.clip_scale_scores(q.double(), p.double())[1].numpy() for q, p in zip(case["qs"], props)]
    return case["oracle"]


@pytest.mark.parametrize("precision", PRECISIONS)
def test_localize_ranked_hits(case, precision):
    from dkd_b200 import engine, ops
    nb, pc, pq = case["nb"], case["pc"], case["pq"]
    _, ids, det = engine.rank(pc, pq, K=K, precision=precision, return_detail=True)
    mo = engine.localize(pc, pq, ids, m=5, iou=0.5)
    assert mo.arg.shape == (M, K, 5) and mo.arg.dtype == torch.int32 and mo.score.dtype == torch.float32
    arg, sc = mo.arg.cpu().numpy(), mo.score.cpu().numpy()
    idn = ids.cpu().numpy().astype(np.int64)
    assert (idn >= 0).all() and (arg[..., 0] >= 0).all()
    if nb == 1:
        assert np.array_equal(sc[..., 0].view(np.int32), det.score[..., 0].cpu().numpy().view(np.int32))
        key = det.arg[..., 0].cpu().numpy()
        off = arg[..., 0] != key
        if off.any():
            # only at exact ties: the key clip scores exactly the maximum, at a later window than moment 0's
            csr = ops.candidates_to_csr(ids, pc.Nv, pc.id_base)
            dots = ops.clip_dots_list(pq.qn[0], pc.branches[0].clip_planes, csr)
            vids = _entry_video(csr[0])
            curve = np_curve(dots[: M * K].cpu().numpy(), pc.branches[0].prop_scale.cpu().numpy()[vids], 32)
            slot = csr[2].cpu().numpy()
            by_slot = np.empty_like(curve)
            by_slot[slot] = curve
            flat = np.nonzero(off.reshape(-1))[0]
            assert (by_slot[flat, key.reshape(-1)[flat]] == sc.reshape(-1, 5)[flat, 0]).all()
            assert (key.reshape(-1)[flat] > arg.reshape(-1, 5)[flat, 0]).all()
        if precision != "bf16":
            assert not off.any()
    ref = _oracle_curves(case)
    fused = ref[0] if nb == 1 else 0.7 * ref[0] + 0.3 * ref[1]
    mm = np.arange(M)[:, None, None]
    live = arg >= 0
    err = np.abs(sc - fused[mm, np.where(live, arg, 0), idn[..., None]])[live]
    assert err.max() <= FP32_TOL, f"moment score error {err.max():.3g}"
    assert (np.diff(np.where(live, sc, -np.inf), axis=-1) <= 0).all()
    w, s = _windows(32)
    for i in range(5):
        for j in range(i + 1, 5):
            both = live[..., i] & live[..., j]
            ov = np_iou(w[arg[..., i]], s[arg[..., i]], w[arg[..., j]], s[arg[..., j]])
            assert (ov[both] <= np.float32(0.5)).all()
            assert (arg[..., i] != arg[..., j])[both].all()


def test_localize_shards_compose_by_elementwise_max(case):
    from dkd_b200 import engine
    pc, pq = case["pc"], case["pq"]
    _, ids = engine.rank(pc, pq, K=K, precision="bf16")
    whole = engine.localize(pc, pq, ids, m=4, iou=0.3)
    frames = [f.cuda() for f in case["frames"]]
    mask = case["mask"].cuda()
    parts = []
    for lo, hi in ((0, 37), (37, Nv)):
        sh = engine.prepare_corpus([f[lo:hi] for f in frames], mask[lo:hi], case["prm"], heads=("two_scale",),
                                   precisions=("exact",), id_base=lo)
        parts.append(engine.localize(sh, pq, ids, m=4, iou=0.3))
    assert torch.equal(torch.maximum(parts[0].arg, parts[1].arg), whole.arg)
    assert torch.equal(torch.maximum(parts[0].score, parts[1].score).view(torch.int32), whole.score.view(torch.int32))
    # each hit is owned by one shard: the other one returns padding for it
    assert ((parts[0].arg == -1) | (parts[1].arg == -1)).all()


def test_localize_padding(case):
    from dkd_b200 import engine
    pc, pq = case["pc"], case["pq"]
    _, ids = engine.rank(pc, pq, K=K, precision="bf16")
    ref = engine.localize(pc, pq, ids, m=3, iou=0.5)
    bad = ids.clone()
    bad[0] = -1                                                     # an all-padding row
    bad[1, ::2] = -1
    bad[2, :4] = torch.tensor([Nv, Nv + 5, -7, 2 ** 30], dtype=torch.int32)    # outside the corpus
    mo = engine.localize(pc, pq, bad, m=3, iou=0.5)
    hole = (bad < 0) | (bad >= Nv)
    assert (mo.arg[hole] == -1).all() and torch.isneginf(mo.score[hole]).all()
    keep = ~hole
    assert torch.equal(mo.arg[keep], ref.arg[keep]) and torch.equal(mo.score[keep], ref.score[keep])
    pq0 = engine.prepare_queries([q[:0].cuda() for q in case["qs"]])
    empty = engine.localize(pc, pq0, ids[:0], m=3)
    assert empty.arg.shape == (0, K, 3) and empty.score.shape == (0, K, 3)
    none = engine.localize(pc, pq, ids[:, :0], m=3)
    assert none.arg.shape == (M, 0, 3)
    shard0 = engine.prepare_corpus([f[:0].cuda() for f in case["frames"]], case["mask"][:0].cuda(), case["prm"],
                                   heads=("two_scale",), precisions=("exact",), id_base=Nv)
    mo0 = engine.localize(shard0, pq, ids, m=3)
    assert (mo0.arg == -1).all() and torch.isneginf(mo0.score).all()


def test_moment_frames_of_moments(case):
    from dkd_b200 import engine
    pc, pq = case["pc"], case["pq"]
    _, ids = engine.rank(pc, pq, K=K, precision="bf16")
    ids = ids.clone()
    ids[4, 3:9] = -1
    mo = engine.localize(pc, pq, ids, m=5, iou=0.5)
    lengths = case["lengths"].int().cuda()
    win = engine.moment_frames(mo.arg, ids, lengths)
    assert win.shape == (M, K, 5, 2)
    for j in range(5):
        one = engine.moment_frames(mo.arg[..., j:j + 1].contiguous(), ids, lengths)
        assert torch.equal(win[..., j:j + 1, :], one)
    live = mo.arg >= 0
    assert (win[live][:, 0] < win[live][:, 1]).all() and (win[~live] == -1).all()


def test_localize_calls_only_its_entry_points(case, monkeypatch):
    from dkd_b200 import engine, _lib
    pc, pq = case["pc"], case["pq"]
    _, ids = engine.rank(pc, pq, K=K, precision="bf16")
    calls = []
    real = _lib.call

    def record(name, *args):
        calls.append(name)
        return real(name, *args)

    monkeypatch.setattr(_lib, "call", record)
    engine.localize(pc, pq, ids)
    assert set(calls) == {"dkd_candidates_to_csr", "dkd_clip_dots_list", "dkd_moment_nms"}
    assert calls.count("dkd_clip_dots_list") == case["nb"] and calls.count("dkd_moment_nms") == 1

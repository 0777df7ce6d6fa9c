"""Exact ties in every max / argmax kernel, where the index is known by construction.

Every max / argmax entry point promises the torch.max tie rule: on an exact tie the FIRST maximal index.  The parity
tests elsewhere accept any index within a tolerance of the maximum, so they cannot see that rule.  Here the inputs are
built so that one row (or one window of clips) beats every other by far more than the operand rounding, and an
identical copy of it sits at a later position: the expected index is the first copy, with no near-tie excuse.  The
bf16 / fp16 GEMM keeps a narrower rule (scores carry the column position in their 4 low mantissa bits): it returns one
of the tied rows, with gap 0, so any tau > 0 flags the pair for the exact kernels.  Copies of identical operands must
give identical accumulators; test_copies_score_identically checks that assumption itself.
"""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import oracle as O

pytestmark = pytest.mark.gpu

FP32_TOL = 2e-6
BF16_REF_TOL = 2e-5       # GEMM vs an fp32 evaluation of the same bf16 / fp16 operands (test_gpu_kernels)


def _unit(v):
    return v / v.norm(dim=-1, keepdim=True)


def _queries(M, D, seed):
    """Unit queries close to e0 (the shared direction every score below is built along)."""
    g = torch.Generator().manual_seed(seed)
    q = torch.zeros(M, D)
    q[:, 0] = 1.0
    return _unit(q + 0.01 * torch.randn(M, D, generator=g))


def _row(alpha, g, D):
    """Unit row with cosine alpha to e0, the rest in a random direction orthogonal to e0."""
    w = torch.randn(D, generator=g)
    w[0] = 0.0
    w = _unit(w)
    e = torch.zeros(D)
    e[0] = 1.0
    return alpha * e + (1.0 - alpha * alpha) ** 0.5 * w


def _tie_pairs(R):
    """(first, second) column pairs of one video: same 16-column chunk, later chunk at a smaller in-chunk position,
    across the two column halves of a 176-column tile, across tiles, first and last row."""
    cand = [(3, 7), (10, 18), (2, 26), (0, R - 1), (R - 17, R - 2), (90, 100), (100, 180), (170, 180), (5, 350),
            (60, 70), (40, 120), (20, 140)]
    return [(a, b) for a, b in cand if b < R]


def _tie_corpus(Nv, R, D, seed, masked):
    """Rows (Nv, R, D) and mask (Nv, R) | None.  Video n: rows a_n < b_n are one target row — cosine about +0.7 to the
    queries or about -0.2, alternating so that every pair appears with both signs — and every other row is below it
    by >= 0.3.  With a mask: random masked columns, among them a decoy that would beat the target; video 1 has its
    first copy masked (the second copy is the answer) and the last video is fully masked.  Returns (x, mask, expected index (Nv,))."""
    g = torch.Generator().manual_seed(seed)
    pairs = _tie_pairs(R)
    x = torch.empty(Nv, R, D)
    mask = torch.ones(Nv, R) if masked else None
    want = torch.empty(Nv, dtype=torch.long)
    for n in range(Nv):
        a, b = pairs[n % len(pairs)]
        pos = (n + n // len(pairs)) % 2 == 0        # every pair with both signs when Nv >= 2 len(pairs)
        lo, hi = (-0.4, 0.2) if pos else (-0.95, -0.7)
        for r in range(R):
            x[n, r] = _row(float(lo + (hi - lo) * torch.rand(1, generator=g)), g, D)
        x[n, a] = _row(0.7 if pos else -0.2, g, D)
        x[n, b] = x[n, a]
        want[n] = a
        if masked:
            drop = torch.rand(R, generator=g) < 0.3
            drop[a] = drop[b] = False
            decoy = next(c for c in range(R) if c not in (a, b))
            x[n, decoy] = _row(0.99, g, D)
            drop[decoy] = True
            if n == 1:
                drop[a] = True
                want[n] = b
            mask[n] = (~drop).float()
    if masked:
        mask[Nv - 1] = 0.0
        want[Nv - 1] = 0
    return x, mask, want


def _ref_rows(q, x, mask):
    """(M, R, Nv) float64 scores of the given operands, masked rows at the fill value (elementwise products: identical
    rows give identical scores, which a blocked matrix product does not promise)."""
    qd = q.double()
    rows = torch.stack([(qd[:, None, :] * xn.double()[None]).sum(-1) for xn in x], dim=2)
    if mask is not None:
        rows = torch.where(mask.T[None].bool(), rows, torch.full_like(rows, O.MASK_FILL))
    return rows


# ------------------------------------------------------------------------------------------------ row maxima, GEMM
# (M, Mpad, Nv, R): which of the GEMM's kernels the shape reaches (dkd_score_bf16.cu, score_max_tc)
GEMM_SHAPES = [
    (200, 256, 16, 128),    # pair tiles (R <= 128, Nv >= 2, Mpad % 256 == 0): two videos per N = 256 tile
    (256, 256, 11, 48),     # pair tiles, 3 chunks per video, odd video count
    (200, 256, 18, 144),    # CTA pair, one 144-column tile per video: column halves merged through shared memory
    (200, 256, 24, 528),    # CTA pair, three 176-column tiles per video
    (100, 128, 24, 528),    # single CTA (Mpad = 128)
    (300, 384, 18, 144),    # single CTA (Mpad = 384)
]


def _gemm_operands(ops, M, Mpad, Nv, R, D, masked, half, seed):
    x, mask, want = _tie_corpus(Nv, R, D, seed, masked)
    q = _queries(M, D, seed + 1)
    dt = torch.float16 if half else torch.bfloat16
    qo = torch.zeros(Mpad, D, dtype=dt)
    qo[:M] = q.to(dt)
    xo = x.to(dt).reshape(Nv * R, D)
    rows = _ref_rows(qo[:M].float(), xo.float().view(Nv, R, D), mask)
    mc = None if mask is None else mask.to(torch.uint8).cuda()
    return qo.cuda(), xo.cuda(), mc, rows, want


def _check_gemm_tie_rule(om, oa, rows, want, masked, Nv, R):
    """The GEMM's tie rule (include/dkd_b200.h): out_arg is a row whose score equals the maximum above the 4 low
    mantissa bits — here one of the two copies, which one is unspecified.  Returns the videos that hold a tie."""
    M = om.shape[0]
    pairs = _tie_pairs(R)
    s_ref, a_ref = rows.max(dim=1)
    assert torch.equal(a_ref, want[None].expand(M, Nv))          # the construction: the first copy is the maximum
    oa = oa.cpu().long()
    tied = []
    for n in range(Nv):
        if masked and n == Nv - 1:                                  # fully masked: fill value, index 0
            assert torch.equal(om[:, n].cpu(), torch.full((M,), -1e10)) and bool((oa[:, n] == 0).all())
            continue
        a, b = pairs[n % len(pairs)]
        ok = (oa[:, n] == b) if (masked and n == 1) else ((oa[:, n] == a) | (oa[:, n] == b))
        assert bool(ok.all()), f"video {n} (copies {a}, {b}): got {sorted(set(oa[:, n].tolist()))}"
        if not (masked and n == 1):                                 # masked video 1 keeps one copy only
            tied.append(n)
    # the returned row scores the maximum exactly (the copies are identical operands)
    assert torch.equal(rows.gather(1, oa[:, None, :]).squeeze(1), s_ref)
    assert (om.cpu().double() - s_ref).abs().max() <= BF16_REF_TOL
    return tied


@pytest.mark.parametrize("half", [False, True], ids=["bf16", "f16"])
@pytest.mark.parametrize("masked", [False, True], ids=["nomask", "mask"])
@pytest.mark.parametrize("top2", [False, True], ids=["top1", "top2"])
@pytest.mark.parametrize("M,Mpad,Nv,R", GEMM_SHAPES)
def test_gemm_tie_rule_on_exact_ties(ops, M, Mpad, Nv, R, top2, masked, half):
    """Every exact tie returns one of the tied rows with gap 0, so any tau > 0 flags it."""
    D = 128
    qd, xd, mc, rows, want = _gemm_operands(ops, M, Mpad, Nv, R, D, masked, half, seed=R + Nv)
    if top2:
        om, oa, og, fl = ops.score_max_bf16(qd, M, xd, Nv, R, mc, want_gap=True, flag_tau=1e-3)
    else:
        om, oa = ops.score_max_bf16(qd, M, xd, Nv, R, mc)
    torch.cuda.synchronize()
    tied = _check_gemm_tie_rule(om, oa, rows, want, masked, Nv, R)
    if top2:
        assert torch.equal(og.cpu()[:, tied], torch.zeros(M, len(tied)))     # an exact tie has gap 0 ...
        bits = (fl.cpu().numpy().view(np.uint32)[:, :, None] >> np.arange(32, dtype=np.uint32)) & 1
        assert bits.reshape(M, -1)[:, tied].all()                  # ... so the pair is flagged
        if masked:                                                  # fully masked video: gap <= 0, flagged too
            assert bool((og[:, Nv - 1] <= 0).all()) and bits.reshape(M, -1)[:, Nv - 1].all()


@pytest.mark.parametrize("half", [False, True], ids=["bf16", "f16"])
@pytest.mark.parametrize("masked", [False, True], ids=["nomask", "mask"])
@pytest.mark.parametrize("M,Mpad,Nv,R", [GEMM_SHAPES[0], GEMM_SHAPES[3], GEMM_SHAPES[4]])
def test_gemm_lists_tie_rule_on_exact_ties(ops, M, Mpad, Nv, R, masked, half):
    D = 128
    qd, xd, mc, rows, want = _gemm_operands(ops, M, Mpad, Nv, R, D, masked, half, seed=3 * R + Nv)
    om, oa, cnt, lst = ops.score_max_bf16_lists(qd, M, xd, Nv, R, 1e-3, mask=mc)
    torch.cuda.synchronize()
    tied = _check_gemm_tie_rule(om, oa, rows, want, masked, Nv, R)
    assert torch.equal(cnt.cpu()[tied], torch.full((len(tied),), M, dtype=torch.int32))   # tied pairs listed, once
    assert torch.equal(lst.cpu()[tied].sort(dim=1).values, torch.arange(M, dtype=torch.int32)[None].expand(len(tied), M))


# ------------------------------------------------------------------------------------ row maxima, exact fp32 kernels
@pytest.mark.parametrize("masked", [False, True], ids=["nomask", "mask"])
@pytest.mark.parametrize("M,Nv,R", [(70, 12, 128), (130, 9, 48), (33, 8, 100)])
def test_exact_row_kernels_first_argmax_on_exact_ties(ops, M, Nv, R, masked):
    """score_max_f32 (SIMT) and score_max_exact (tcgen05 kind::tf32, dense and CSR)."""
    D = 128
    x, mask, want = _tie_corpus(Nv, R, D, seed=7 * R + M, masked=masked)
    q = _queries(M, D, seed=M)
    rows = _ref_rows(q, x, mask)
    s_ref, a_ref = rows.max(dim=1)
    assert torch.equal(a_ref, want[None].expand(M, Nv))
    qc, xc = q.cuda(), x.cuda()
    mc = None if mask is None else mask.to(torch.uint8).cuda()
    want_d = want[None].expand(M, Nv)
    om, oa, _ = ops.score_max_f32(qc, xc, mc)
    assert torch.equal(oa.cpu().long(), want_d) and (om.cpu().double() - s_ref).abs().max() <= FP32_TOL
    planes = ops.pack_rows(xc)
    em, ea = ops.score_max_exact(qc, planes, R, mc)
    assert torch.equal(ea.cpu().long(), want_d) and (em.cpu().double() - s_ref).abs().max() <= FP32_TOL
    vid_ptr, q_list, slot = ops.select_pairs_csr(torch.zeros(M, Nv, device="cuda"), 0.5)
    cm, ca = ops.score_max_exact(qc, planes, R, mc, csr=(vid_ptr, q_list))
    sl = slot[: M * Nv].long()
    assert torch.equal(ca, ea.flatten()[sl]) and torch.equal(cm, em.flatten()[sl])


@pytest.mark.parametrize("tensor_cores", [True, False], ids=["tc", "simt"])
@pytest.mark.parametrize("masked", [False, True], ids=["nomask", "mask"])
def test_train_sim_fwd_first_argmax_on_exact_ties(ops, monkeypatch, tensor_cores, masked):
    """dkd_train_sim_fwd (the SIMT forward, reached only with TRAIN_SIM_TENSOR_CORES off) and the tensor-core route:
    cosine and raw maxima both at the first copy.  Raw rows are scaled so that the raw maxima tie too."""
    monkeypatch.setattr(ops, "TRAIN_SIM_TENSOR_CORES", tensor_cores)
    M, Nv, R, D = 40, 12, 64, 128
    x, mask, want = _tie_corpus(Nv, R, D, seed=17, masked=masked)
    x = 2.5 * x
    q = 3.0 * _queries(M, D, seed=18)
    qc, xc = q.cuda(), x.cuda()
    mc = None if mask is None else mask.to(torch.uint8).cuda()
    rq, rx = ops.row_inv_norms(qc), ops.row_inv_norms(xc)
    max_n, arg_n, max_u, arg_u, _ = ops.train_sim_fwd(qc, xc, rq, rx, mc)
    rows = _ref_rows(q, x, mask)
    want_d = want[None].expand(M, Nv)
    assert torch.equal(arg_n.cpu().long(), want_d) and torch.equal(arg_u.cpu().long(), want_d)
    assert (max_u.cpu().double() - rows.max(dim=1).values).abs().max() <= 7.5 * FP32_TOL
    cos = _ref_rows(F.normalize(q, dim=-1), F.normalize(x, dim=-1), mask)
    assert (max_n.cpu().double() - cos.max(dim=1).values).abs().max() <= FP32_TOL


@pytest.mark.parametrize("tensor_cores", [True, False], ids=["tc", "simt"])
def test_train_gradient_of_a_tied_max_reaches_the_first_frame(ops, monkeypatch, tensor_cores):
    """Duplicated frames: the max's gradient goes to the first copy only (torch.max backward), on both forward routes;
    compared with autograd through a float64 restatement of get_sim_scores / get_unnormalized_sim_scores."""
    from dkd_b200 import train
    monkeypatch.setattr(ops, "TRAIN_SIM_TENSOR_CORES", tensor_cores)
    M, Nv, R, D = 24, 8, 32, 64
    x, mask, want = _tie_corpus(Nv, R, D, seed=27, masked=True)
    mask[Nv - 1, 0] = 1.0                        # no fully masked video in a training batch
    want[Nv - 1] = 0
    q = 2.0 * _queries(M, D, seed=28)
    g = torch.Generator().manual_seed(29)
    w_n, w_u = torch.rand(M, Nv, generator=g), torch.rand(M, Nv, generator=g)
    qd = q.cuda().requires_grad_()
    xd = x.cuda().requires_grad_()
    max_n, max_u, _ = train.in_batch_similarity(qd, xd, mask.cuda())
    ((max_n * w_n.cuda()).sum() + (max_u * w_u.cuda()).sum()).backward()
    qr = q.double().requires_grad_()
    xr = x.double().requires_grad_()
    s_n, a_n = _ref_rows(F.normalize(qr, dim=-1), F.normalize(xr, dim=-1), mask).max(dim=1)
    s_u, a_u = _ref_rows(qr, xr, mask).max(dim=1)
    assert torch.equal(a_n, want[None].expand(M, Nv)) and torch.equal(a_u, want[None].expand(M, Nv))
    ((s_n * w_n.double()).sum() + (s_u * w_u.double()).sum()).backward()
    assert (qd.grad.cpu().double() - qr.grad).abs().max() <= 1e-4
    assert (xd.grad.cpu().double() - xr.grad).abs().max() <= 1e-4
    pairs = _tie_pairs(R)
    for n in range(Nv - 1):
        a, b = pairs[n % len(pairs)]
        second = b if n != 1 else a              # video 1: the first copy is masked, the second one wins
        assert bool((xd.grad[n, second] == 0).all()), f"video {n}: gradient reached the second copy"


# ---------------------------------------------------------------------------------------------------- window maxima
def _tie_clips(Nv, T, D, seed):
    """Clips (Nv, T, D) with one exact tie class per video (n % 3) and the expected key clip p(w, s):
      0: two equal strong clips at s1 < s2 - 1 (w = 1 windows tie)           -> p(1, s1)
      1: a 3-clip pattern whose mean beats every window, copied 4+ clips later -> p(3, s)
      2: two equal strong clips at s, s + 1: windows (1, s), (1, s+1), (2, s) tie exactly ((v + v) / 2 = v) -> p(1, s)
    Every other clip is anti-aligned with the queries."""
    g = torch.Generator().manual_seed(seed)
    clips = torch.empty(Nv, T, D)
    want = torch.empty(Nv, dtype=torch.long)
    e = torch.eye(D)
    for n in range(Nv):
        for i in range(T):
            w = torch.randn(D, generator=g)
            w[:4] = 0.0
            clips[n, i] = (-0.5 * e[0] + 0.85 * _unit(w)) * (1.0 + torch.rand(1, generator=g))
        k = n % 3
        span = T - 7
        s = int(torch.randint(0, span + 1, (1,), generator=g))
        if k == 0:
            s2 = s + 2 + int(torch.randint(0, T - s - 2, (1,), generator=g))
            clips[n, s] = 0.9 * e[0] + 0.43 * e[1]
            clips[n, s2] = clips[n, s]
            want[n] = O.proposal_index(1, s, T)
        elif k == 1:
            s2 = s + 4 + int(torch.randint(0, T - s - 6, (1,), generator=g))
            for j in range(3):
                clips[n, s + j] = 0.7 * e[0] + 0.714 * e[1 + j]
                clips[n, s2 + j] = clips[n, s + j]
            want[n] = O.proposal_index(3, s, T)
        else:
            clips[n, s] = 0.9 * e[0] + 0.43 * e[1]
            clips[n, s + 1] = clips[n, s]
            want[n] = O.proposal_index(1, s, T)
    return clips, want


def _clip_case(ops, M, Nv, T, D, seed):
    clips, want = _tie_clips(Nv, T, D, seed)
    q = _queries(M, D, seed + 1)
    props = O.build_proposals(clips)
    s_ref, allp, k_ref = O.clip_scale_scores(q, props)
    top2 = torch.topk(allp, 2, dim=1).values
    assert float((top2[:, 0] - top2[:, 1]).max()) <= 1e-6                  # every pair is a tie (up to CPU rounding)
    at_want = allp.gather(1, want[None, None, :].expand(allp.shape[0], 1, Nv)).squeeze(1)
    assert float((top2[:, 0] - at_want).max()) <= 1e-6                    # ... and the expected window is one of them
    qc, cc = q.cuda(), clips.cuda().contiguous()
    _, ps, _ = ops.build_proposals(cc, want_bf16=False)
    return qc, cc, ps, s_ref, allp, want


@pytest.mark.parametrize("T", [32, 16, 12, 8])
def test_clip_score_first_window_on_exact_ties(ops, T):
    """dkd_clip_score_f32, dense for every T; CSR, run-plus-scatter and dkd_clip_score_list forms for T in {32, 12}."""
    M, Nv, D = 70, 15, 128
    qc, cc, ps, s_ref, allp, want = _clip_case(ops, M, Nv, T, D, seed=T)
    planes = ops.pack_clips(cc)
    om, oa = ops.clip_score_f32(qc, planes, ps)
    torch.cuda.synchronize()
    bad = (oa.cpu().long() != want[None]).nonzero().tolist()
    assert not bad, f"{len(bad)} key clips not the first tied window, e.g. {bad[:3]}: got " \
                    f"{[int(oa[m, n]) for m, n in bad[:3]]}, want {[int(want[n]) for _, n in bad[:3]]}"
    assert (om.cpu() - s_ref).abs().max() <= FP32_TOL
    if T not in (32, 12):
        return
    vid_ptr, q_list, slot = ops.select_pairs_csr(torch.zeros(M, Nv, device="cuda"), 0.5)
    cs, ck = ops.clip_score_f32(qc, planes, ps, csr=(vid_ptr, q_list))
    sl = slot[: M * Nv].long()
    assert torch.equal(cs, om.flatten()[sl]) and torch.equal(ck, oa.flatten()[sl])
    counts = (vid_ptr[1:] - vid_ptr[:-1]).contiguous()
    sm = torch.full((M, Nv), -7.0, device="cuda")
    sa = torch.full((M, Nv), -7, dtype=torch.int32, device="cuda")
    ops.clip_score_f32(qc, planes, ps, csr=(vid_ptr[:-1].contiguous(), q_list, counts), scatter=(slot, sm, sa))
    assert torch.equal(sm, om) and torch.equal(sa, oa)
    lm = torch.full((M, Nv), -7.0, device="cuda")
    la = torch.full((M, Nv), -7, dtype=torch.int32, device="cuda")
    cnt = torch.full((Nv,), M, dtype=torch.int32, device="cuda")
    lst = torch.arange(M, dtype=torch.int32, device="cuda").flip(0)[None].expand(Nv, M).contiguous()
    ops.clip_score_list(qc, planes, ps, cnt, lst, lm, la)
    assert torch.equal(lm, om) and torch.equal(la, oa)


def test_known_key_gives_the_full_search_result(ops):
    """dkd_clip_score_f32 with known_key (T = 32) == the call without it, bit for bit, for the correct key, the
    runner-up, random keys, out-of-range keys and an exactly tied key in a later row (w) of the same video.  The one
    documented residual — a key tied with an EARLIER start of the SAME row keeps the given key — is pinned here."""
    M, Nv, D, T = 64, 15, 128, 32
    qc, cc, ps, s_ref, allp, want = _clip_case(ops, M, Nv, T, D, seed=5)
    planes = ops.pack_clips(cc)
    vid_ptr, q_list, slot = ops.select_pairs_csr(torch.zeros(M, Nv, device="cuda"), 0.5)
    sl = slot[: M * Nv].long()
    csr = (vid_ptr, q_list)
    bm, ba = ops.clip_score_f32(qc, planes, ps, csr=csr)
    assert torch.equal(ba.cpu().long(), want[None].expand(M, Nv).flatten()[sl.cpu()])

    def run(key):
        return ops.clip_score_f32(qc, planes, ps, csr=csr, known_key=key.to(torch.int32).cuda().contiguous())

    g = torch.Generator().manual_seed(6)
    dense_key = ba.new_empty(M * Nv)
    dense_key[sl] = ba
    dense_key = dense_key.view(M, Nv).cpu()
    # runner-up: the best window strictly below the maximum (the tied windows of the maximum are the cases below)
    below = torch.where(allp >= allp.max(dim=1, keepdim=True).values - 1e-6, torch.full_like(allp, -1e30), allp)
    runner = below.argmax(dim=1)
    rnd = torch.randint(0, 528, (M, Nv), generator=g)
    tied = allp.gather(1, rnd[:, None]).squeeze(1) >= allp.max(dim=1).values - 1e-6
    rnd = torch.where(tied, dense_key, rnd)            # a random hit on a tied window would be the residual below
    keys = [dense_key, runner, rnd]
    keys += [torch.full((M, Nv), v) for v in (-1, 528, 10 ** 6)]
    # tied later row: class-2 videos, where p(2, s) ties with p(1, s) = the answer
    later_row = dense_key.clone()
    for n in range(2, Nv, 3):
        s = int(want[n])
        later_row[:, n] = O.proposal_index(2, s, T)
    keys.append(later_row)
    for key in keys:
        km, ka = run(key)
        assert torch.equal(km, bm) and torch.equal(ka, ba)
    # residual: a later start of the same row (class 0: p(1, s2); class 2: p(1, s + 1)) is kept, value identical
    same_row = dense_key.clone()
    expect = dense_key.clone()
    clips = cc.cpu()
    for n in range(Nv):
        if n % 3 == 1:
            continue
        s = int(want[n])
        s2 = next(i for i in range(s + 1, T) if torch.equal(clips[n, i], clips[n, s]))
        same_row[:, n] = s2
        expect[:, n] = s2
    km, ka = run(same_row)
    assert torch.equal(km, bm)
    assert torch.equal(ka.cpu(), expect.flatten()[sl.cpu()].to(torch.int32))


# ------------------------------------------------------------------------------------------ copies score identically
def test_copies_score_identically(ops):
    """Bit-identical outputs for identical operands wherever they sit: a video copied into its pair partner, the next
    16-video work item and the last video; a query copied into the other CTA of a pair and into later query tiles.
    Every tie test above rests on this."""
    g = torch.Generator(device="cuda").manual_seed(3)
    M, Mpad, Nv, D = 2500, 2560, 960, 128
    vid_copies = [1, 15, 16, 17, Nv - 1]
    q_copies = [3 + 128, 3 + 256, 3 + 2304]
    q = F.normalize(torch.randn(M, D, device="cuda", generator=g), dim=-1)
    q[q_copies] = q[3].clone()

    def same_cols(t):
        return all(torch.equal(t[:, 0], t[:, c]) for c in vid_copies)

    def same_rows(t):
        return all(torch.equal(t[3], t[r]) for r in q_copies)

    for R in (528, 128):
        x = F.normalize(torch.randn(Nv, R, D, device="cuda", generator=g), dim=-1)
        x[vid_copies] = x[0].clone()
        mask = (torch.rand(Nv, R, device="cuda", generator=g) > 0.2).to(torch.uint8)
        mask[vid_copies] = mask[0].clone()
        for dt in (torch.bfloat16, torch.float16):
            qo = torch.zeros(Mpad, D, dtype=dt, device="cuda")
            qo[:M] = q.to(dt)
            xo = x.to(dt).reshape(Nv * R, D).contiguous()
            for mk in (None, mask):
                outs = ops.score_max_bf16(qo, M, xo, Nv, R, mk, want_gap=True, flag_tau=1e-3)
                for t in outs[:3]:
                    assert same_cols(t) and same_rows(t), f"R={R} {dt} mask={mk is not None}"
                om, oa, cnt, _ = ops.score_max_bf16_lists(qo, M, xo, Nv, R, 1e-3, mask=mk)
                assert torch.equal(om, outs[0]) and torch.equal(oa, outs[1])
                assert all(int(cnt[0]) == int(cnt[c]) for c in vid_copies)
    # exact kernels (smaller corpus: a copy in the next tile of queries / videos is what matters)
    Nv2, L = 40, 100
    x = F.normalize(torch.randn(Nv2, L, D, device="cuda", generator=g), dim=-1)
    cp = [1, 17, Nv2 - 1]
    x[cp] = x[0].clone()
    mask = (torch.rand(Nv2, L, device="cuda", generator=g) > 0.2).to(torch.uint8)
    mask[cp] = mask[0].clone()
    qs = q[:300].contiguous()
    em, ea = ops.score_max_exact(qs, ops.pack_rows(x), L, mask)
    for t in (em, ea):
        assert all(torch.equal(t[:, 0], t[:, c]) for c in cp) and torch.equal(t[3], t[3 + 128]) and torch.equal(t[3], t[3 + 256])
    clips = torch.randn(Nv2, 32, D, device="cuda", generator=g)
    clips[cp] = clips[0].clone()
    _, ps, _ = ops.build_proposals(clips, want_bf16=False)
    planes = ops.pack_clips(clips)
    cm, ca = ops.clip_score_f32(qs, planes, ps)
    vid_ptr, q_list, slot = ops.select_pairs_csr(torch.zeros(300, Nv2, device="cuda"), 0.5)
    sm, sa = ops.clip_score_f32(qs, planes, ps, csr=(vid_ptr, q_list))
    dm = torch.empty(300 * Nv2, device="cuda")
    da = torch.empty(300 * Nv2, dtype=torch.int32, device="cuda")
    dm[slot.long()] = sm
    da[slot.long()] = sa
    for t in (cm, ca, dm.view(300, Nv2), da.view(300, Nv2)):
        assert all(torch.equal(t[:, 0], t[:, c]) for c in cp) and torch.equal(t[3], t[3 + 128]) and torch.equal(t[3], t[3 + 256])
    lengths = mask.sum(dim=1).to(torch.int32)
    key = torch.randn(Nv2, L, D, device="cuda", generator=g)
    val = torch.randn(Nv2, L, D, device="cuda", generator=g)
    key[cp], val[cp] = key[0].clone(), val[0].clone()
    key, val = key * mask[:, :, None], val * mask[:, :, None]
    tf, th = ops.frame_attn_table(key.contiguous(), val.contiguous(), clips, lengths)
    for t in (tf, th):
        assert all(torch.equal(t[0], t[c]) for c in cp)
    for qq, tab in ((qs, tf), (qs.half(), th)):
        fused, fr = ops.frame_fuse(qq, tab, cm, ca, 0.7, 0.3, 1.0, want_frame=True)
        for t in (fused, fr):
            assert all(torch.equal(t[:, 0], t[:, c]) for c in cp) and torch.equal(t[3], t[3 + 128])
    cand = torch.stack([torch.tensor([0] + cp, dtype=torch.int32)] * 300).cuda()
    cvp, cql, cslot = ops.candidates_to_csr(cand, Nv2)
    ccs, cck = ops.clip_score_f32(qs, planes, ps, csr=(cvp, cql))
    cand_scores = torch.zeros(300, len(cp) + 1, device="cuda")
    ops.frame_fuse_csr(qs, tf, ccs, cck, (cvp, cql, cslot), 0.7, 0.3, 1.0, cand_scores, False)
    assert all(torch.equal(cand_scores[:, 0], cand_scores[:, j]) for j in range(1, len(cp) + 1))
    assert torch.equal(cand_scores[3], cand_scores[3 + 128])


# --------------------------------------------------------------------------------- short videos, two-scale head
def _params(D, seed):
    g = torch.Generator().manual_seed(seed)
    return [tuple(t for t in (0.05 * torch.randn(D, D, generator=g), 0.01 * torch.randn(D, generator=g),
                               0.05 * torch.randn(D, D, generator=g), 0.01 * torch.randn(D, generator=g)))]


@pytest.mark.parametrize("T", [32, 16, 12])
def test_two_scale_short_videos(ops, T):
    """Videos shorter than T clips (average_to_fixed_length copies frames: identical clips, identical windows): clips
    bit-equal to the oracle, exact-path scores within tolerance, key clips the oracle's first argmax wherever its top-2
    gap is resolvable and never a later duplicate of an identical window, and the approximate paths rank identically."""
    from dkd_b200 import engine
    D, L, M = 128, 40, 37
    lens = sorted({1, 2, 3, 5, 15, 16, 17, T - 1, T, L})
    Nv = 2 * len(lens)
    g = torch.Generator().manual_seed(T)
    frames = torch.randn(Nv, L, D, generator=g) + 0.6 * torch.randn(Nv, 1, D, generator=g)
    lengths = torch.tensor(lens + lens, dtype=torch.int32)
    mask = (torch.arange(L)[None] < lengths[:, None].long()).float()
    frames = (frames * mask[:, :, None]).contiguous()
    q = torch.randn(M, D, generator=g)
    kw, kb, vw, vb = _params(D, T + 1)[0]
    ref = O.two_scale_branch(q, frames, mask, kw, kb, vw, vb, T=T)
    clips = ops.downsample_clips(frames.cuda(), lengths.cuda(), T=T).cpu()
    short = lengths <= T
    assert torch.equal(clips[short], ref["clips"][short])
    assert (clips - ref["clips"]).abs().max() <= 1e-6
    prm = [tuple(t.cuda() for t in (kw, kb, vw, vb))]
    pc = engine.prepare_corpus([frames.cuda()], mask.cuda(), prm, T=T, heads=("two_scale",),
                               precisions=("exact", "bf16", "fp16", "shortcut"))
    pq = engine.prepare_queries([q.cuda()])
    fused, per = engine.score_two_scale_head(pc, pq, "exact", want_frame=True)
    s_clip, k_clip = per[0]["clip"].cpu(), per[0]["key_clip"].cpu().long()
    assert (s_clip - ref["clip"]).abs().max() <= FP32_TOL
    allp = O.clip_scale_scores(q, ref["proposals"])[1]
    top2 = torch.topk(allp, 2, dim=1).values
    resolvable = (top2[:, 0] - top2[:, 1]) > 2e-6
    assert torch.equal(k_clip[resolvable], ref["key_clip"][resolvable])
    same = k_clip == ref["key_clip"]
    assert (fused.cpu()[same] - ref["branch"][same]).abs().max() <= 5e-6
    # no identical window (same width, same clip sequence) with a smaller index than the returned one
    P = O.num_proposals(T)
    widths = torch.tensor([w for w in range(1, T + 1) for _ in range(T - w + 1)])
    starts = torch.tensor([s for w in range(1, T + 1) for s in range(T - w + 1)])
    for n in range(Nv):
        c = clips[n]
        for kk in k_clip[:, n].unique().tolist():
            w, s = int(widths[kk]), int(starts[kk])
            for s0 in range(s):
                assert not torch.equal(c[s0:s0 + w], c[s:s + w]), f"video {n}: window {kk} repeats start {s0}"
    assert P == allp.shape[1]
    _, i_ex = engine.rank(pc, pq, K=Nv, head="two_scale", precision="exact")
    for prec in ("bf16", "fp16", "shortcut"):
        _, i_ap = engine.rank(pc, pq, K=Nv, head="two_scale", precision=prec, Kc=Nv)
        assert torch.equal(i_ap, i_ex), prec

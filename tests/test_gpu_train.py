"""Training-step similarity and losses on the GPU (BASELINE.json configs[4]; SURVEY §8f #2): the kernels of
csrc/dkd_train.cu against the oracle (forward values and autograd gradients), and DLDKD.forward of the model
mirror against the loss terms and parameter gradients of the unmodified reference (tests/golden/ref_train_step.npz)."""
import numpy as np
import pytest
import torch

from oracle import oracle as O
from tests import synth
from tests.test_oracle_golden import TRAIN_SETTINGS, TRAIN_TERMS, _stored_entries, _train_fixture

pytestmark = pytest.mark.gpu


def _case(M, N, L, D, seed, caps=None):
    x, mask, lengths = synth.encoded_corpus(N, L, D, seed=seed, min_len=1)
    if N > 2:
        mask[2] = 0                      # one fully masked video: scores exactly -1e10, no gradient
        x[2] = 0
    q = synth.encoded_queries(M, D, seed=seed + 1)
    g = torch.Generator().manual_seed(seed + 2)
    labels = torch.randint(0, N, (M,), generator=g)
    labels[labels == 2] = 0
    return q, x, mask, labels


@pytest.mark.parametrize("M,N,L,D", [(640, 128, 128, 384), (37, 9, 50, 64), (5, 3, 128, 512), (64, 1, 16, 32)])
def test_train_similarity_forward_and_backward(ops, M, N, L, D):
    """One fused pass == get_sim_scores + get_unnormalized_sim_scores + the positive column of the per-frame
    tensor; its backward == autograd through the oracle (fp32 on CPU)."""
    from dkd_b200 import train
    q, x, mask, labels = _case(M, N, L, D, seed=100 + M)
    qr, xr = q.clone().requires_grad_(True), x.clone().requires_grad_(True)
    s, rows, _ = O.get_sim_scores(qr, xr, mask)
    u = O.get_unnormalized_sim_scores(qr, xr, mask)
    curve_ref = rows[torch.arange(M), :, labels]
    qc, xc = q.cuda().requires_grad_(True), x.cuda().requires_grad_(True)
    max_n, max_u, curve = train.in_batch_similarity(qc, xc, mask.cuda(), labels.tolist())
    assert (max_n.detach().cpu() - s.detach()).abs().max() <= 2e-6
    scale = max(1.0, float(u.detach().abs()[u.detach() > -1e9].max()))
    # raw (unnormalised) maxima: relative tolerance 6e-6 — the tensor core's fp32 accumulator truncates (up to one ulp of
    # the running sum per tcgen05.mma: 144 steps at D = 384), which is what separates it from an fp32 FMA chain
    assert (max_u.detach().cpu() - u.detach()).abs().max() <= 6e-6 * scale
    assert (curve.detach().cpu() - curve_ref.detach()).abs().max() <= 2e-6
    # a loss that touches all three outputs with fixed random weights (masked entries weigh 0)
    g = torch.Generator().manual_seed(7)
    wn, wu, wc = torch.randn(M, N, generator=g), torch.randn(M, N, generator=g), torch.randn(M, L, generator=g)
    wc = wc * mask[labels]
    (s * wn).sum().add((u * wu).sum()).add((curve_ref * wc).sum()).backward()
    (max_n * wn.cuda()).sum().add((max_u * wu.cuda()).sum()).add((curve * wc.cuda()).sum()).backward()
    gq, gx = qr.grad, xr.grad
    assert (qc.grad.cpu() - gq).abs().max() <= 2e-5 * max(1.0, float(gq.abs().max()))
    assert (xc.grad.cpu() - gx).abs().max() <= 2e-5 * max(1.0, float(gx.abs().max()))
    assert float(xc.grad[2].abs().max() if N > 2 else 0.0) == 0.0
    # deterministic: a second backward gives the same bits
    qc2, xc2 = q.cuda().requires_grad_(True), x.cuda().requires_grad_(True)
    a, b, c = train.in_batch_similarity(qc2, xc2, mask.cuda(), labels.tolist())
    (a * wn.cuda()).sum().add((b * wu.cuda()).sum()).add((c * wc.cuda()).sum()).backward()
    assert torch.equal(qc2.grad, qc.grad) and torch.equal(xc2.grad, xc.grad)


def test_kl_curve_loss_forward_and_backward(ops):
    from dkd_b200 import train
    M, N, L = 300, 40, 128
    g = torch.Generator().manual_seed(3)
    lengths = torch.randint(1, L + 1, (N,), generator=g)
    lengths[0], lengths[1] = L, 1
    mask = (torch.arange(L)[None] < lengths[:, None]).float()
    labels = torch.randint(0, N, (M,), generator=g)
    pred = (0.3 * torch.randn(M, L, generator=g)).requires_grad_(True)
    tgt = 0.3 * torch.randn(M, L, generator=g)
    ref = 0
    for i in range(M):
        n = int(lengths[labels[i]])
        ref = ref + torch.nn.functional.kl_div(torch.log_softmax(pred[i, :n] / 0.2, -1),
                                               torch.softmax(tgt[i, :n] / 0.2, -1), reduction="sum")
    ref.backward()
    pc = pred.detach().cuda().requires_grad_(True)
    got = train.kl_frame_loss(pc, tgt.cuda(), mask.cuda(), labels.tolist(), 0.2)
    (2.0 * got).backward()
    assert abs(float(got) - float(ref)) <= 1e-5 * max(1.0, abs(float(ref)))
    assert (pc.grad.cpu() - 2.0 * pred.grad).abs().max() <= 1e-5


@pytest.mark.parametrize("style,hard,self_distil", [("soft", True, False), ("soft", False, False), ("hard", True, False),
                                                    ("soft", True, True), ("soft", False, True)])
@pytest.mark.parametrize("M,N,caps", [(640, 128, 5), (21, 7, 3), (9, 9, 1)])
def test_fused_branch_losses_match_oracle_loops(ops, style, hard, self_distil, M, N, caps):
    """The fused triplet + NCE kernel (value and gradient) == the oracle's loop-for-loop restatement of the
    reference with autograd; sampled negatives draw from the same seeded CPU generator in the same order;
    self_distil: the soft targets come from the scores themselves (exploration branch) and carry gradient."""
    from dkd_b200 import train
    g = torch.Generator().manual_seed(11 + M)
    labels = [i // caps for i in range(M)]
    s = 0.2 * torch.randn(M, N, generator=g)
    u = 3.0 * torch.randn(M, N, generator=g)
    sims = 3.0 * torch.randn(M, N, generator=g)
    sr, ur = s.clone().requires_grad_(True), u.clone().requires_grad_(True)
    torch.manual_seed(5)
    trip_ref = O.clip_triplet_loss(sr, labels, 0.1, hard, 20)
    nce_ref = (O.clip_nce_soft(labels, ur, ur if self_distil else sims, 0.8, 0.8) if style == "soft"
               else O.clip_nce(labels, ur))
    (trip_ref + 0.5 * nce_ref).backward()
    sc, uc = s.cuda().requires_grad_(True), u.cuda().requires_grad_(True)
    torch.manual_seed(5)
    trip, nce = train.branch_losses(sc, uc, uc if self_distil else sims.cuda(), labels, 0.1, hard, 20, style == "soft",
                                    0.8, 0.8)
    (trip + 0.5 * nce).backward()
    assert abs(float(trip) - float(trip_ref)) <= 1e-5 * max(1.0, abs(float(trip_ref)))
    assert abs(float(nce) - float(nce_ref)) <= 1e-5 * max(1.0, abs(float(nce_ref)))
    assert (sc.grad.cpu() - sr.grad).abs().max() <= 1e-6
    assert (uc.grad.cpu() - ur.grad).abs().max() <= 1e-6
    # deterministic
    sc2, uc2 = s.cuda().requires_grad_(True), u.cuda().requires_grad_(True)
    torch.manual_seed(5)
    t2, n2 = train.branch_losses(sc2, uc2, uc2 if self_distil else sims.cuda(), labels, 0.1, hard, 20, style == "soft",
                                 0.8, 0.8)
    (t2 + 0.5 * n2).backward()
    assert torch.equal(sc2.grad, sc.grad) and torch.equal(uc2.grad, uc.grad) and float(t2) == float(trip)


@pytest.mark.parametrize("tag", list(TRAIN_SETTINGS))
def test_forward_matches_reference_fixture(ops, dkd, tag):
    """DLDKD.forward(batch) of the mirror (CUDA similarity + KL kernels, hand-written backward) reproduces the
    unmodified reference's loss terms and every parameter gradient."""
    g, m, batch = _train_fixture(dkd, device="cuda")
    style, hard, pool, seed = TRAIN_SETTINGS[tag]
    m.config.label_style = style
    m.set_hard_negative(hard, pool)
    if seed is not None:
        torch.manual_seed(seed)
    loss, terms = m(batch)
    loss.backward()
    ref = dict(zip(TRAIN_TERMS, g[f"{tag}.terms"]))
    for k in TRAIN_TERMS:
        assert abs(float(terms[k]) - ref[k]) <= 5e-6 * max(1.0, abs(ref[k])), (k, float(terms[k]), ref[k])
    for name, p in m.named_parameters():
        if "key_mapping" in name or "val_mapping" in name:
            continue
        want = g[f"{tag}.grad.{name}"]
        got = _stored_entries(g, name, p.grad.cpu().numpy()) if p.grad is not None else np.zeros_like(want)
        assert np.abs(got - want).max() <= 2e-5 * max(1.0, np.abs(want).max()), name


def test_config5_shape_step_runs_and_matches_oracle(ops):
    """BASELINE.json configs[4] at full size from the encoded vectors on: 128 videos x 128 frames, 640 queries,
    D = 384 (teacher 512): loss terms == oracle.train_losses, gradients of the encoded vectors == autograd."""
    from dkd_b200 import train
    N, L, D, Dt, caps = 128, 128, 384, 512, 5
    M = N * caps
    labels = [i // caps for i in range(M)]
    ci, mask, _ = synth.encoded_corpus(N, L, D, seed=51)
    ce, _, _ = synth.encoded_corpus(N, L, D, seed=52)
    ce = ce * mask[:, :, None]
    ct, _, _ = synth.encoded_corpus(N, L, Dt, seed=53)
    ct = ct * mask[:, :, None]
    qi, qe, qt = (synth.encoded_queries(M, d, seed=54 + k) for k, d in enumerate((D, D, Dt)))
    # correlate queries with their positive video so the losses are in a realistic regime
    qi = qi + 0.5 * ci[labels, 0]
    qe = qe + 0.5 * ce[labels, 0]
    qt = qt + 0.5 * ct[labels, 0]
    leaves = [t.clone().requires_grad_(True) for t in (qi, ci, qe, ce)]
    enc = dict(teacher_q=qt, teacher_ctx=ct, inher_q=leaves[0], inher_ctx=leaves[1], explore_q=leaves[2],
               explore_ctx=leaves[3])
    ref, rt = O.train_losses(enc, labels, mask, use_hard_negative=True, hard_pool_size=1, label_style="soft")
    ref.backward()

    class Stub:                                           # the encoders are not under test here
        pass
    dev = "cuda"
    cl = [t.detach().to(dev).requires_grad_(True) for t in (qi, ci, qe, ce)]
    m = Stub()
    m.config = type("C", (), dict(label_style="soft", margin=0.1, use_hard_negative=True, hard_pool_size=1))()
    m.double_branch, m.weight, m.kl_intra_weight, m.inher_nce_weight, m.explore_nce_weight = True, 1, 0.1, 0.04, 0.04
    m.alpha = m.belta = 0.8
    m.encode_context = lambda v, mk: (cl[1], cl[3])
    m.encode_query = lambda t, mk: (cl[0], cl[2])
    batch = dict(text_labels=labels, student_videos=None, student_videos_mask=mask.to(dev), student_text=None,
                 student_text_mask=None, teacher_text=qt.to(dev)[:, None, :], teacher_videos=ct.to(dev))
    loss, terms = train.forward_losses(m, batch)
    loss.backward()
    assert abs(float(loss) - float(ref)) <= 1e-5 * max(1.0, abs(float(ref)))
    for k in ("inher_trip", "inher_nce", "explore_trip", "explore_nce", "kl"):
        assert abs(float(terms[k]) - float(rt[k])) <= 1e-5 * max(1.0, abs(float(rt[k]))), k
    for a, b in zip(cl, leaves):
        assert (a.grad.cpu() - b.grad).abs().max() <= 2e-5 * max(1.0, float(b.grad.abs().max()))

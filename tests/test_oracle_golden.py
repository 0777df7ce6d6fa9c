"""CPU: pin oracle/oracle.py (a-REF functions) and the PyTorch encoder mirror against fixtures that were
produced by RUNNING THE UNMODIFIED REFERENCE (oracle/make_golden.py -> tests/golden/ref_*.npz)."""
import os

import numpy as np
import pytest
import torch

from oracle import oracle as O
from oracle import ref_shim

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _load(name):
    return np.load(os.path.join(GOLD, name))


def test_get_sim_scores_matches_reference_fixture():
    g = _load("ref_sim_scores.npz")
    q, ctx, mask = (torch.from_numpy(g[k]) for k in ("q", "ctx", "mask"))
    s, rows, _ = O.get_sim_scores(q, ctx, mask)
    assert np.array_equal(s.numpy(), g["scores"])          # same torch ops, same order: bit exact
    assert np.array_equal(rows.numpy(), g["rows"])
    s2, rows2, _ = O.get_sim_scores(q, ctx, None)
    assert np.array_equal(s2.numpy(), g["scores_nomask"])
    assert np.array_equal(rows2.numpy(), g["rows_nomask"])
    assert np.array_equal(O.get_unnormalized_sim_scores(q, ctx, mask).numpy(), g["unnorm"])
    assert np.array_equal(O.mask_logits(rows2, mask.T.unsqueeze(0)).numpy(), g["mask_logits"])
    # masked entries are exactly -1e10
    assert (g["rows"][:, mask.numpy().T == 0] == np.float32(-1e10)).all()


def test_average_to_fixed_length_matches_reference_fixture():
    g = _load("ref_avg_fixed.npz")
    for n in (1, 2, 5, 31, 32, 33, 48, 64, 100, 127, 128):
        x = torch.from_numpy(g[f"x_{n}"])
        for T in (32, 8):
            assert np.array_equal(O.average_to_fixed_length(x, T).numpy(), g[f"y_{n}_{T}"]), (n, T)
    assert np.allclose(O.l2_normalize_np_array(g["ufs_x"]), g["l2_y"], rtol=0, atol=0)


def test_metrics_match_reference_fixture():
    g = _load("ref_tiny_eval.npz")
    Nq = int(g["dims"][6])
    t2v = {i: list(g["t2v_ids"][g["t2v_ptr"][i]: g["t2v_ptr"][i + 1]]) for i in range(Nq)}
    assert np.array_equal(O.fuse_branches(g["inher_scores"], g["explore_scores"]), g["fused"])
    for key, sc in (("metrics_inher", g["inher_scores"]), ("metrics_explore", g["explore_scores"]),
                    ("metrics_fused", g["fused"])):
        assert np.allclose(np.array(O.eval_q2m(-1 * sc, t2v)), g[key])
    assert np.isclose(O.t2v_map(-1 * g["fused"], t2v), float(g["map_fused"]))
    # R@K derived from ranked id lists (what the device path returns) agrees with eval_q2m
    top = O.topk_ids(g["fused"], min(100, g["fused"].shape[1]))
    r = O.recall_from_topk(top, t2v, ks=(1, 5))
    assert np.allclose(r, g["metrics_fused"][:2])


def test_get_gt_matches_reference_id_convention():
    vids = [f"vid{n}" for n in range(4)]
    qs = ["vid2#enc#0", "vid0#enc#0", "vid2#enc#1", "nomatch#enc#0"]
    v2t, t2v = O.get_gt(vids, qs)
    assert v2t == [[1], [], [0, 2], []] and t2v == {1: [0], 0: [2], 2: [2]}


def _tiny_model(dkd, g):
    from dkd_b200 import model as M
    Dv, Dq, H, Lc, Lq = (int(v) for v in g["dims"][:5])
    cfg = ref_shim.model_config(Dv, Dq, hidden=H, n_heads=4, max_ctx_l=Lc, max_desc_l=Lq)
    m = M.DLDKD(cfg, ref_shim.options())
    sd = {k[3:]: torch.from_numpy(g[k]) for k in g.files if k.startswith("sd.")}
    missing, unexpected = m.load_state_dict(sd, strict=False)
    assert not unexpected                                     # every reference parameter has a home
    assert all("key_mapping" in k or "val_mapping" in k for k in missing)
    return m.eval()


def test_encoder_mirror_matches_reference_fixture(dkd):
    """encode_context / encode_query (PyTorch, CPU here) with the reference's weights reproduce the
    reference's encoded features."""
    g = _load("ref_tiny_eval.npz")
    m = _tiny_model(dkd, g)
    videos = torch.from_numpy(g["videos"])
    vlen = torch.from_numpy(g["video_len"])
    mask = (torch.arange(videos.shape[1])[None] < vlen[:, None]).float()
    with torch.no_grad():
        fi, fe = m.encode_context(videos, mask)
    assert np.array_equal(mask.numpy(), g["video_mask"])
    # the reference encodes in batches of 4 padded to the batch max length; padding columns differ,
    # valid frames must agree
    valid = mask.bool()
    assert np.allclose(fi[valid].numpy(), g["inher_frame_feat"][valid.numpy()], atol=2e-6)
    assert np.allclose(fe[valid].numpy(), g["explore_frame_feat"][valid.numpy()], atol=2e-6)
    q = torch.from_numpy(g["queries"])
    qmask = (torch.arange(q.shape[1])[None] < torch.from_numpy(g["query_len"])[:, None]).float()
    with torch.no_grad():
        qi, qe = m.encode_query(q, qmask)
    assert np.allclose(qi.numpy(), g["enc_q_inher"], atol=2e-6)
    assert np.allclose(qe.numpy(), g["enc_q_explore"], atol=2e-6)


@pytest.mark.skipif(not ref_shim.available(),
                    reason="the original DL-DKD sources are not present (they are not part of this repository)")
def test_oracle_against_live_reference():
    """Where the original DL-DKD sources are present: the oracle restatements equal the imported reference on fresh
    random inputs."""
    rm, re_, rd = ref_shim.load()
    g = torch.Generator().manual_seed(5)
    q, ctx = torch.randn(33, 48, generator=g), torch.randn(21, 40, 48, generator=g)
    mask = (torch.rand(21, 40, generator=g) > 0.3).float()
    mask[:, 0] = 1
    s_ref, rows_ref = rm.DLDKD.get_sim_scores(q, ctx, mask)
    s, rows, _ = O.get_sim_scores(q, ctx, mask)
    assert torch.equal(s, s_ref) and torch.equal(rows, rows_ref)
    x = np.random.default_rng(3).standard_normal((77, 5)).astype(np.float32)
    assert np.array_equal(O.average_to_fixed_length(torch.from_numpy(x), 32).numpy(), rd.average_to_fixed_length(x, 32))
    sc = np.random.default_rng(4).standard_normal((40, 30)).astype(np.float32)
    gts = {i: [i % 30] for i in range(40)}
    assert np.allclose(O.eval_q2m(-sc, gts), re_.eval_q2m(-sc, gts))
    assert np.isclose(O.t2v_map(-sc, gts), re_.t2v_map(-sc, gts))
    vm = [f"v{i}" for i in range(30)]
    qm = [f"v{i % 30}#enc#{i // 30}" for i in range(40)]
    assert O.get_gt(vm, qm) == re_.get_gt(vm, qm)


TRAIN_TERMS = ["loss_overall", "inher_trip", "inher_nce", "explore_trip", "explore_nce", "kl", "kl_intra"]
TRAIN_SETTINGS = {"soft_hard": ("soft", True, 1, None), "soft_rand": ("soft", False, 20, 123),
                  "hard_hard": ("hard", True, 1, None)}


def _train_fixture(dkd, device="cpu"):
    """The tiny training batch of ref_train_step.npz + the model mirror carrying the reference's weights."""
    from dkd_b200 import model as M
    g = _load("ref_train_step.npz")
    Dv, Dq, H, Lc, Lq = (int(v) for v in g["dims"][:5])
    cfg = ref_shim.model_config(Dv, Dq, hidden=H, n_heads=4, max_ctx_l=Lc, max_desc_l=Lq)
    cfg.input_drop = 0.0
    cfg.drop = 0.0
    m = M.DLDKD(cfg, ref_shim.options())
    sd = {k[3:]: torch.from_numpy(g[k]) for k in g.files if k.startswith("sd.")}
    missing, unexpected = m.load_state_dict(sd, strict=False)
    assert not unexpected and all("key_mapping" in k or "val_mapping" in k for k in missing)
    m = m.to(device).train()
    t = lambda k: torch.from_numpy(g[k]).to(device)
    batch = dict(text_labels=[int(x) for x in g["labels"]], student_videos=t("videos"), student_videos_mask=t("vmask"),
                 student_text=t("text"), student_text_mask=t("qmask"), teacher_text=t("teacher_text"),
                 teacher_videos=t("teacher_videos"))
    return g, m, batch


def _stored_entries(g, name, grad):
    """The entries of a parameter gradient that ref_train_step.npz keeps: all of them, or for a larger parameter the
    fixed sample of flat indices grad_idx.<name> (oracle/make_golden.py sample_grads)."""
    key = f"grad_idx.{name}"
    return grad.reshape(-1)[g[key]] if key in g else grad


@pytest.mark.parametrize("tag", list(TRAIN_SETTINGS))
def test_train_losses_oracle_matches_reference_fixture(dkd, tag):
    """oracle.train_losses on the encoder mirror's outputs reproduces the unmodified reference's DLDKD.forward:
    every loss term, and (through plain autograd) every parameter gradient, for the three fixture settings."""
    g, m, batch = _train_fixture(dkd)
    style, hard, pool, seed = TRAIN_SETTINGS[tag]
    labels, mask = batch["text_labels"], batch["student_videos_mask"]
    ci, ce = m.encode_context(batch["student_videos"], mask)
    qi, qe = m.encode_query(batch["student_text"], batch["student_text_mask"])
    enc = dict(teacher_q=batch["teacher_text"].squeeze(), teacher_ctx=batch["teacher_videos"], inher_q=qi,
               inher_ctx=ci, explore_q=qe, explore_ctx=ce)
    if seed is not None:
        torch.manual_seed(seed)
    loss, terms = O.train_losses(enc, labels, mask, margin=0.1, use_hard_negative=hard, hard_pool_size=pool,
                                 label_style=style)
    ref = dict(zip(TRAIN_TERMS, g[f"{tag}.terms"]))
    assert abs(float(loss) - ref["loss_overall"]) <= 2e-6 * max(1.0, abs(ref["loss_overall"]))
    for k in ("inher_trip", "inher_nce", "explore_trip", "explore_nce", "kl"):
        assert abs(float(terms[k]) - ref[k]) <= 2e-6 * max(1.0, abs(ref[k])), k
    loss.backward()
    for name, p in m.named_parameters():
        if "key_mapping" in name or "val_mapping" in name:
            continue
        want = g[f"{tag}.grad.{name}"]
        got = _stored_entries(g, name, p.grad.numpy()) if p.grad is not None else np.zeros_like(want)
        assert np.abs(got - want).max() <= 1e-5 * max(1.0, np.abs(want).max()), name
    # the similarity intermediates of the fixture
    s, rows, _ = O.get_sim_scores(qi.detach(), ci.detach(), mask)
    assert np.abs(s.numpy() - g["sim_max"]).max() <= 2e-6
    assert np.abs(O.get_unnormalized_sim_scores(qi.detach(), ci.detach(), mask).numpy() - g["sim_unnorm"]).max() <= 2e-5

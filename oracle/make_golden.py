"""Generate tests/golden/ref_*.npz by RUNNING THE UNMODIFIED REFERENCE on CPU.

    DKD_REFERENCE_ROOT=<the reference's source tree> python oracle/make_golden.py
The fixtures pin oracle/oracle.py's (a-REF) functions and the drop-in model/eval mirror.
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path = [p for p in sys.path if os.path.abspath(p or ".") != os.path.join(ROOT, "oracle")]
sys.path.insert(0, ROOT)
from oracle import ref_shim  # noqa: E402
from oracle.datasets import VideoSet, QuerySet  # noqa: E402
from tests import synth  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")
GRAD_SAMPLE = 512      # gradient entries kept per larger parameter of ref_train_step.npz: keeps the file under 1 MB


def sample_grads(out, tags=("soft_hard", "soft_rand", "hard_hard")):
    """In place: every parameter gradient with more than GRAD_SAMPLE entries is cut down to a fixed sample of its flat
    entries (seeded, the same for every tag); the sorted indices are stored once as grad_idx.<name>."""
    rng = np.random.default_rng(0)
    for key in [k for k in out if k.startswith(f"{tags[0]}.grad.")]:
        name = key[len(f"{tags[0]}.grad."):]
        n = out[key].size
        if n <= GRAD_SAMPLE:
            continue
        idx = np.sort(rng.choice(n, GRAD_SAMPLE, replace=False)).astype(np.int32)
        out[f"grad_idx.{name}"] = idx
        for tag in tags:
            out[f"{tag}.grad.{name}"] = out[f"{tag}.grad.{name}"].reshape(-1)[idx]


def golden_sim_scores(M):
    rm, _, _ = M
    g = torch.Generator().manual_seed(1234)
    q = torch.randn(12, 32, generator=g)
    ctx = torch.randn(7, 16, 32, generator=g)
    lengths = torch.tensor([16, 1, 5, 16, 9, 2, 13])
    mask = (torch.arange(16)[None] < lengths[:, None]).float()
    ctx = ctx * mask[:, :, None]
    s, rows = rm.DLDKD.get_sim_scores(q, ctx, mask)
    s_nm, rows_nm = rm.DLDKD.get_sim_scores(q, ctx, None)
    u = rm.DLDKD.get_unnormalized_sim_scores(q, ctx, mask)
    ml = rm.mask_logits(rows_nm, mask.transpose(0, 1).unsqueeze(0))
    np.savez_compressed(os.path.join(OUT, "ref_sim_scores.npz"), q=q.numpy(), ctx=ctx.numpy(), mask=mask.numpy(),
                        scores=s.numpy(), rows=rows.numpy(), scores_nomask=s_nm.numpy(), rows_nomask=rows_nm.numpy(),
                        unnorm=u.numpy(), mask_logits=ml.numpy())


def golden_avg_fixed(M):
    _, _, rd = M
    out = {}
    rng = np.random.default_rng(7)
    for n in (1, 2, 5, 31, 32, 33, 48, 64, 100, 127, 128):
        x = rng.standard_normal((n, 6)).astype(np.float32)
        out[f"x_{n}"] = x
        for T in (32, 8):
            out[f"y_{n}_{T}"] = rd.average_to_fixed_length(x, T)
    # uniform_feature_sampling / l2_normalize mirror (data preprocessing the synthetic generator copies)
    x = rng.standard_normal((300, 6)).astype(np.float32)
    out["ufs_x"] = x
    out["ufs_y"] = rd.uniform_feature_sampling(x, 128).astype(np.float32)
    out["l2_y"] = rd.l2_normalize_np_array(x).astype(np.float32)
    np.savez_compressed(os.path.join(OUT, "ref_avg_fixed.npz"), **out)


def golden_tiny_eval(M):
    rm, re_, rd = M
    Dv, Dq, H, Lc, Lq = 48, 40, 64, 16, 8
    Nv, Nq = 9, 23
    cfg = ref_shim.model_config(Dv, Dq, hidden=H, n_heads=4, max_ctx_l=Lc, max_desc_l=Lq)
    opt = ref_shim.options(eval_query_bsz=5, eval_context_bsz=4)
    torch.manual_seed(0)
    model = rm.DLDKD(cfg, opt)
    # random-init LayerNorm / bias are constants: perturb every parameter so that the fixture
    # exercises all of them
    g = torch.Generator().manual_seed(99)
    with torch.no_grad():
        for p in model.parameters():
            p.add_(0.05 * torch.randn(p.shape, generator=g))
    model.eval()
    vids = synth.raw_videos(Nv, Lc, Dv, seed=11, min_len=3)
    qs = synth.raw_queries(Nq, Dq, seed=12, min_len=2, max_len=Lq)
    vset, qset = VideoSet(vids), QuerySet(qs, Nv)
    with torch.no_grad():
        ctx = re_.compute_context_info(model, vset, opt)
        inher, explore, teacher, qmetas = re_.compute_query2ctx_info(model, qset, opt, ctx)
        # encoded queries in dataset order
        qfeat = torch.zeros(Nq, Lq, Dq)
        qmask = torch.zeros(Nq, Lq)
        for i, f in enumerate(qs):
            qfeat[i, : len(f)] = f
            qmask[i, : len(f)] = 1
        qi, qe = model.encode_query(qfeat, qmask)
    assert teacher is None
    v2t, t2v = re_.get_gt(ctx["video_metas"], qmetas)
    fused = 0.7 * inher + 0.3 * explore
    m_in = re_.eval_q2m(-1 * inher, t2v)
    m_ex = re_.eval_q2m(-1 * explore, t2v)
    m_fu = re_.eval_q2m(-1 * fused, t2v)
    map_fu = re_.t2v_map(-1 * fused, t2v)
    order = np.array([qset.ids.index(m) for m in qmetas], np.int64)  # row r of the scores = dataset query order[r]
    vpad = np.zeros((Nv, Lc, Dv), np.float32)
    vlen = np.zeros((Nv,), np.int32)
    for i, f in enumerate(vids):
        vpad[i, : len(f)] = f.numpy()
        vlen[i] = len(f)
    qlen = np.array([len(f) for f in qs], np.int32)
    sd = {"sd." + k: v.numpy() for k, v in model.state_dict().items()}
    t2v_ptr = np.zeros(Nq + 1, np.int32)
    t2v_ids = []
    for i in range(Nq):
        t2v_ids += t2v[i]
        t2v_ptr[i + 1] = len(t2v_ids)
    np.savez_compressed(
        os.path.join(OUT, "ref_tiny_eval.npz"), dims=np.array([Dv, Dq, H, Lc, Lq, Nv, Nq], np.int64),
        videos=vpad, video_len=vlen, queries=qfeat.numpy(), query_len=qlen,
        inher_frame_feat=ctx["inher_frame_feat"].numpy(), explore_frame_feat=ctx["explore_frame_feat"].numpy(),
        video_mask=ctx["video_mask"].numpy(), inher_scores=inher, explore_scores=explore, order=order,
        enc_q_inher=qi.numpy(), enc_q_explore=qe.numpy(), fused=fused.astype(np.float32),
        metrics_inher=np.array(m_in), metrics_explore=np.array(m_ex), metrics_fused=np.array(m_fu),
        map_fused=np.array(map_fu), t2v_ptr=t2v_ptr, t2v_ids=np.array(t2v_ids, np.int32), **sd)


def golden_train_step(M):
    """DLDKD.forward + backward of the unmodified reference on a tiny batch (BASELINE.json configs[4] in small):
    loss terms and every parameter gradient, for three settings — soft labels + hard negatives (deterministic),
    soft labels + sampled negatives (torch.manual_seed fixes the draws), hard labels + hard negatives."""
    rm, _, _ = M
    Dv, Dq, H, Lc, Lq, Dt = 48, 40, 64, 16, 8, 32
    B, caps = 6, 3
    cfg = ref_shim.model_config(Dv, Dq, hidden=H, n_heads=4, max_ctx_l=Lc, max_desc_l=Lq)
    cfg.input_drop = 0.0
    cfg.drop = 0.0
    opt = ref_shim.options()
    torch.manual_seed(0)
    model = rm.DLDKD(cfg, opt)
    g = torch.Generator().manual_seed(321)
    with torch.no_grad():
        for p in model.parameters():
            p.add_(0.05 * torch.randn(p.shape, generator=g))
    model.train()
    lens = torch.tensor([16, 3, 9, 16, 12, 5])
    vmask = (torch.arange(Lc)[None] < lens[:, None]).float()
    vids = torch.randn(B, Lc, Dv, generator=g) * vmask[:, :, None]
    tv = torch.randn(B, Lc, Dt, generator=g) * vmask[:, :, None]
    labels = [i for i in range(B) for _ in range(caps)]
    nq = len(labels)
    qlen = torch.randint(2, Lq + 1, (nq,), generator=g)
    qmask = (torch.arange(Lq)[None] < qlen[:, None]).float()
    txt = torch.randn(nq, Lq, Dq, generator=g) * qmask[:, :, None]
    tt = torch.randn(nq, 1, Dt, generator=g)
    batch = dict(text_labels=labels, student_videos=vids, student_videos_mask=vmask, student_text=txt,
                 student_text_mask=qmask, teacher_text=tt, teacher_videos=tv)
    out = dict(dims=np.array([Dv, Dq, H, Lc, Lq, Dt, B, caps], np.int64), labels=np.array(labels, np.int64),
               videos=vids.numpy(), vmask=vmask.numpy(), teacher_videos=tv.numpy(), text=txt.numpy(),
               qmask=qmask.numpy(), teacher_text=tt.numpy())
    out.update({"sd." + k: v.detach().numpy().copy() for k, v in model.state_dict().items()})
    terms = ["loss_overall", "inher_trip", "inher_nce", "explore_trip", "explore_nce", "kl", "kl_intra"]
    for tag, style, hard, seed in (("soft_hard", "soft", True, None), ("soft_rand", "soft", False, 123),
                                   ("hard_hard", "hard", True, None)):
        cfg.label_style = style
        model.set_hard_negative(hard, 1 if hard else 20)
        model.zero_grad()
        if seed is not None:
            torch.manual_seed(seed)
        loss, d = model(batch)
        loss.backward()
        out[f"{tag}.terms"] = np.array([float(d[k]) for k in terms], np.float64)
        for k, p in model.named_parameters():
            out[f"{tag}.grad.{k}"] = (p.grad if p.grad is not None else torch.zeros_like(p)).numpy().copy()
    # similarity intermediates of the inheritance branch (encoded features -> scores), for the kernel-level test
    with torch.no_grad():
        ctx_i, _ = model.encode_context(vids, vmask)
        q_i, _ = model.encode_query(txt, qmask)
        s, rows = rm.DLDKD.get_sim_scores(q_i, ctx_i, vmask)
        u = rm.DLDKD.get_unnormalized_sim_scores(q_i, ctx_i, vmask)
    out.update(enc_ctx=ctx_i.numpy(), enc_q=q_i.numpy(), sim_max=s.numpy(), sim_rows=rows.numpy(), sim_unnorm=u.numpy())
    sample_grads(out)
    np.savez_compressed(os.path.join(OUT, "ref_train_step.npz"), **out)


if __name__ == "__main__":
    os.makedirs(OUT, exist_ok=True)
    mods = ref_shim.load()
    golden_sim_scores(mods)
    golden_avg_fixed(mods)
    golden_tiny_eval(mods)
    golden_train_step(mods)
    for f in sorted(os.listdir(OUT)):
        print(f, os.path.getsize(os.path.join(OUT, f)))

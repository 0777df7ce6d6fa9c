"""Drop-in mirror of the reference's eval orchestration (method/eval.py) on the CUDA kernels.

Same names, arguments and return values as the reference:
    compute_context_info(model, eval_dataset, opt)                 method/eval.py:114-175
    compute_query2ctx_info(model, eval_dataset, opt, ctx_info)     method/eval.py:177-219
    eval_q2m(scores, q2m_gts) / t2v_map / get_gt / cal_perf        method/eval.py:43-111, 223-235
    eval_epoch(model, val_video_dataset, val_text_dataset, opt)    method/eval.py:237-263

Extra `opt` fields (all optional; defaults reproduce the reference):
    scoring    "frame" (default: the head the reference ships) | "two_scale" (north_star head)
    precision  "exact" (default: fp32 kernels) | "bf16" (tcgen05 GEMM, scores within 1e-3) | "fp16" | "shortcut"
    ambiguity_tau, candidates   the two empirical constants of the approximate pass (engine.AMBIGUITY_TAU, 128)
Extra entry point: rank_queries(...) -> per-query top-K on the device (the benchmarked hot path).
"""
import logging

import numpy as np
import torch
from torch.utils.data import DataLoader

from . import engine, ops

logger = logging.getLogger(__name__)


def _opt(opt, key, default):
    try:
        return getattr(opt, key)
    except AttributeError:
        if isinstance(opt, dict) and key in opt:
            return opt[key]
        return default


# ---- collate functions: same batch layout as method/data_provider.py:139-170 -----------------
def _pad_stack(seqs):
    lens = [len(s) for s in seqs]
    out = torch.zeros(len(seqs), max(lens), seqs[0].shape[-1])
    mask = torch.zeros(len(seqs), max(lens))
    for i, s in enumerate(seqs):
        out[i, : lens[i]] = s[: lens[i]]
        mask[i, : lens[i]] = 1.0
    return out, mask


def collate_frame_val(data):
    """method/data_provider.py:139-148: items (feat, idx, id) -> (videos, mask, idxs, ids); items that also carry
    teacher features (feat, teacher_feat, idx, id) -> (videos, teacher_videos, mask, idxs, ids)."""
    if len(data[0]) == 3:
        feats, idxs, ids = zip(*data)
        videos, mask = _pad_stack(feats)
        return videos, mask, idxs, ids
    feats, teacher, idxs, ids = zip(*data)
    videos, mask = _pad_stack(feats)
    teacher_videos, _ = _pad_stack(teacher)
    return videos, teacher_videos, mask, idxs, ids


def collate_text_val(data):
    """Each batch is re-ordered by caption length, longest first (method/data_provider.py:152-170);
    query_metas carries the resulting row order.  4-tuple items carry one teacher (CLIP) text vector each."""
    data = sorted(data, key=lambda x: len(x[0]), reverse=True)
    if len(data[0]) == 3:
        feats, idxs, ids = zip(*data)
        target, mask = _pad_stack(feats)
        return target, mask, idxs, ids
    feats, teacher, idxs, ids = zip(*data)
    target, mask = _pad_stack(feats)
    return target, torch.cat([t.reshape(1, -1) for t in teacher], dim=0), mask, idxs, ids


def _cat_padded(tensors):
    """Zero-pad to the longest sequence and concatenate (cat_tensor, method/eval.py:139-155)."""
    if not tensors:
        return None
    Lmax = max(t.shape[1] for t in tensors)
    n = sum(t.shape[0] for t in tensors)
    out = tensors[0].new_zeros((n, Lmax) + tuple(tensors[0].shape[2:]))
    if tensors[0].dim() not in (2, 3):
        raise ValueError("Only support 2/3 dimensional tensors")
    r = 0
    for t in tensors:
        out[r: r + t.shape[0], : t.shape[1]] = t
        r += t.shape[0]
    return out


def compute_context_info(model, eval_dataset, opt):
    """Encode the whole corpus and prepare it on the device.  Returns the reference's dict
    (video_metas, inher_frame_feat, explore_frame_feat, teacher_frame_feat, video_mask) plus
    `prepared`: the engine.PreparedCorpus used by compute_query2ctx_info / rank_queries.

    Datasets whose items carry teacher (CLIP) frame features (5-field batches, method/eval.py:129-132): the teacher
    features are scored raw, like DLDKD.forward does (method/model.py:113-114), so teacher_frame_feat is their padded
    concatenation.  (The reference passes them to encode_context as a third argument, which its own two-argument
    encode_context, method/model.py:215, rejects with a TypeError.)"""
    model.eval()
    loader = DataLoader(eval_dataset, collate_fn=collate_frame_val, batch_size=opt.eval_context_bsz,
                        num_workers=_opt(opt, "num_workers", 0), shuffle=False, pin_memory=_opt(opt, "pin_memory", False))
    metas, inher, explore, teacher, masks = [], [], [], [], []
    with torch.no_grad():
        for batch in loader:
            metas.extend(batch[-1])
            feat = batch[0].to(opt.device, non_blocking=True)
            mask = batch[-3].to(opt.device, non_blocking=True)
            if len(batch) == 5:
                teacher.append(batch[1].to(opt.device, non_blocking=True))
            fi, fe = model.encode_context(feat, mask)
            inher.append(fi)
            explore.append(fe)
            masks.append(mask)
        inher = _cat_padded(inher)
        video_mask = _cat_padded(masks)
        explore = _cat_padded(explore) if model.double_branch else None
        scoring = _opt(opt, "scoring", "frame")
        precision = _opt(opt, "precision", "exact")
        prepared = model.prepare_context(inher, explore, video_mask, heads=(scoring,),
                                         precisions=("exact",) if precision == "exact" else ("exact", precision),
                                         id_base=_opt(opt, "id_base", 0))
    return dict(video_metas=metas, inher_frame_feat=inher, explore_frame_feat=explore,
                teacher_frame_feat=_cat_padded(teacher), video_mask=video_mask, prepared=prepared)


def _encode_all_queries(model, eval_dataset, opt):
    loader = DataLoader(eval_dataset, collate_fn=collate_text_val, batch_size=opt.eval_query_bsz,
                        num_workers=_opt(opt, "num_workers", 0), shuffle=False, pin_memory=_opt(opt, "pin_memory", False))
    metas, qi, qe, qt = [], [], [], []
    with torch.no_grad():
        for batch in loader:
            metas.extend(batch[-1])
            a, b = model.encode_query(batch[0].to(opt.device, non_blocking=True), batch[-3].to(opt.device, non_blocking=True))
            qi.append(a)
            qe.append(b)
            if len(batch) == 5:
                qt.append(batch[1].to(opt.device, non_blocking=True))
    qs = [torch.cat(qi, dim=0)]
    if model.double_branch:
        qs.append(torch.cat(qe, dim=0))
    return qs, metas, (torch.cat(qt, dim=0) if qt else None)


_PRECISIONS = ("exact", "bf16", "fp16", "shortcut")


def compute_query2ctx_info(model, eval_dataset, opt, ctx_info):
    """Score every query against the whole corpus.  Returns (inher_scores, explore_scores | None, teacher_scores |
    None, query_metas) with numpy float32 (Nq, Nv) matrices in DataLoader row order, like the reference.
    With opt.scoring == "two_scale" the matrices are the per-branch two-scale scores
    (w_clip * clip + w_frame * frame).  This is the reference's interface and, like it, ends in a dense
    device->host copy; the ranking-only hot path is rank_queries / eval_epoch(opt.precision != "exact")."""
    model.eval()
    pc = ctx_info["prepared"]
    qs, metas, qt = _encode_all_queries(model, eval_dataset, opt)
    precision = _opt(opt, "precision", "exact")
    scoring = _opt(opt, "scoring", "frame")
    if precision not in _PRECISIONS:
        raise ValueError(f"opt.precision must be one of {_PRECISIONS}, got {precision!r}")
    chunk = int(_opt(opt, "query_chunk", 16384))
    outs = [[] for _ in qs]
    for lo in range(0, qs[0].shape[0], chunk):
        pq = engine.prepare_queries([q[lo: lo + chunk] for q in qs], want_bf16=precision == "bf16")
        if scoring == "frame":
            for o, (s, _) in zip(outs, engine.score_frame_head(pc, pq, precision)):
                o.append(s)
        else:
            for bi in range(len(qs)):  # per-branch two-scale score = fused with branch weight 1
                sub = engine.PreparedCorpus(Nv=pc.Nv, L=pc.L, D=pc.D, T=pc.T, id_base=pc.id_base, mask_u8=pc.mask_u8,
                                            lengths=pc.lengths, branches=[pc.branches[bi]], heads=pc.heads,
                                            Lg=pc.Lg, mask_g=pc.mask_g, Pg=pc.Pg, prop_mask=pc.prop_mask)
                subq = engine.PreparedQueries(M=pq.M, Mpad=pq.Mpad, qn=[pq.qn[bi]], qb=[pq.qb[bi]], qh=[pq.qh[bi]])
                f, _ = engine.score_two_scale_head(sub, subq, precision, model.clip_scale_w, model.frame_scale_w)
                outs[bi].append(f)
    inher = torch.cat(outs[0], dim=0).cpu().numpy().copy()
    explore = torch.cat(outs[1], dim=0).cpu().numpy().copy() if model.double_branch else None
    teacher = None
    if ctx_info.get("teacher_frame_feat") is not None and qt is not None:   # method/eval.py:198-202
        teacher = model.get_sim_scores(qt, ctx_info["teacher_frame_feat"], ctx_info["video_mask"],
                                       want_rows=False)[0].cpu().numpy().copy()
    return inher, explore, teacher, metas


def rank_queries(model, eval_dataset, opt, ctx_info, K=100, return_dense=False, return_detail=False):
    """The hot path: per-query top-K (fused score desc) without materialising anything on the host.
    Returns (scores (Nq, K) fp32 CUDA, ids (Nq, K) int32 CUDA, query_metas) [+ the dense (Nq, Nv) fused device
    matrix of the scoring pass when return_dense] [+ the engine.HitDetail of every hit when return_detail: key clip or
    best frame and per-branch scores; engine.moment_frames turns it into frame windows].  No host synchronisation
    inside: the candidate certificates of the tcgen05 path are resolved once at the end (engine.finish)."""
    model.eval()
    pc = ctx_info["prepared"]
    qs, metas, _ = _encode_all_queries(model, eval_dataset, opt)
    precision = _opt(opt, "precision", "exact")
    scoring = _opt(opt, "scoring", "frame")
    if precision not in _PRECISIONS:
        raise ValueError(f"opt.precision must be one of {_PRECISIONS}, got {precision!r}")
    chunk = int(_opt(opt, "query_chunk", 16384))
    outs = []
    for lo in range(0, qs[0].shape[0], chunk):
        pq = engine.prepare_queries([q[lo: lo + chunk] for q in qs], want_bf16=precision == "bf16")
        outs.append(engine.rank(pc, pq, K=K, head=scoring, precision=precision, w_clip=model.clip_scale_w,
                                w_frame=model.frame_scale_w, certify="deferred", return_dense=return_dense,
                                tau=_opt(opt, "ambiguity_tau", None), Kc=int(_opt(opt, "candidates", 128)),
                                return_detail=return_detail))
    engine.finish()
    res = tuple(engine.HitDetail.cat([o[j] for o in outs]) if isinstance(outs[0][j], engine.HitDetail)
                else torch.cat([o[j] for o in outs]) for j in range(len(outs[0])))
    return res[:2] + (metas,) + res[2:]


def get_gt(video_metas, query_metas):
    """GT lists by id match 'vid#...' -> 'vid' (method/eval.py:43-57), O(Nv + Nq)."""
    pos = {v: i for i, v in enumerate(video_metas)}
    v2t_gt = [[] for _ in video_metas]
    for i, qid in enumerate(query_metas):
        v = pos.get(qid.split('#', 1)[0])
        if v is not None:
            v2t_gt[v].append(i)
    t2v_gt = {}
    for v, qs in enumerate(v2t_gt):
        for q in qs:
            t2v_gt.setdefault(q, []).append(v)
    return v2t_gt, t2v_gt


def _gt_csr(q2m_gts, n_q, first_only=False):
    ptr = np.zeros(n_q + 1, np.int32)
    ids = []
    for i in range(n_q):
        g = list(q2m_gts[i])
        ids += g[:1] if first_only else g
        ptr[i + 1] = len(ids)
    return torch.from_numpy(ptr), torch.tensor(ids, dtype=torch.int32)


def gt_ranks(scores, q2m_gts, first_only=False, device="cuda"):
    """Rank of the best GT per query on the device.  `scores` are NEGATED similarities like the
    reference's eval_q2m argument (numpy or tensor)."""
    s = torch.as_tensor(scores, dtype=torch.float32, device=device)
    zero = torch.zeros_like(s)
    sim = ops.fuse_scores(s.contiguous(), zero, -1.0, 0.0)  # un-negate on the device (exact)
    ptr, ids = _gt_csr(q2m_gts, s.shape[0], first_only)
    return ops.rank_of_gt(sim, ptr.to(device), ids.to(device)).cpu().numpy()


def eval_q2m(scores, q2m_gts):
    """(r1, r5, r10, r100, medr, meanr) from negated scores (method/eval.py:59-94).  Exact-score ties are
    ranked lower-video-index first (the reference's np.argsort leaves them unspecified)."""
    r = gt_ranks(scores, q2m_gts)
    n_q = len(r)
    rk = [100.0 * np.count_nonzero(r <= k) / n_q for k in (1, 5, 10, 100)]
    return (rk[0], rk[1], rk[2], rk[3], np.median(r), r.mean())


def t2v_map(c2i, t2v_gts):
    """mAP with only the first GT relevant => mean(1 / rank) (method/eval.py:97-111)."""
    r = gt_ranks(c2i, t2v_gts, first_only=True)
    return float(np.mean(1.0 / r))


def cal_perf(t2v_all_errors, t2v_gt, test=False):
    r1, r5, r10, r100, medr, meanr = eval_q2m(t2v_all_errors, t2v_gt)
    m = t2v_map(t2v_all_errors, t2v_gt)
    logger.info(" * Text to Video:")
    logger.info(" * r_1_5_10_100: {}".format([round(r1, 1), round(r5, 1), round(r10, 1), round(r100, 1)]))
    logger.info(" * recall sum: {}".format(round(r1 + r5 + r10 + r100, 1)))
    logger.info(" * mAP: {}".format(round(m, 4)))
    return (r1, r5, r10, r100, medr, meanr, m)


def recall_from_topk(top_ids, t2v_gt, ks=(1, 5, 10, 100)):
    """R@K from ranked id lists (host, integer work)."""
    ids = top_ids.cpu().numpy() if isinstance(top_ids, torch.Tensor) else np.asarray(top_ids)
    n_q = ids.shape[0]
    out = []
    for k in ks:
        hit = sum(1 for i in range(n_q) if set(t2v_gt.get(i, ())) & set(ids[i, :k].tolist()))
        out.append(100.0 * hit / n_q)
    return tuple(out)


def metrics_from_ranking(top_ids, dense, t2v_gt, id_base=0):
    """(r1, r5, r10, r100, medr, meanr, mAP) of a device ranking, integer work on the device:
    the GT rank comes from the ranked top-K id lists where a GT video is in them (exact: these are the rescored
    lists) and from dkd_rank_of_gt on the dense fused scores of the scoring pass otherwise (for the tcgen05 path
    those are the approximate scores, |d| <= 1e-3: only ranks beyond K, i.e. medr / meanr / mAP tails, see them;
    R@K for K <= top-K never does)."""
    M, K = top_ids.shape
    dev = top_ids.device
    ptr, gts = _gt_csr(t2v_gt, M)
    ptr1, first = _gt_csr(t2v_gt, M, first_only=True)
    ptr, gts, ptr1, first = ptr.to(dev), gts.to(dev), ptr1.to(dev), first.to(dev)

    def ranks(p, g):
        r_dense = ops.rank_of_gt(dense, p, g).long()
        cnt = (p[1:] - p[:-1]).long()
        owner = torch.repeat_interleave(torch.arange(M, device=dev), cnt)              # query of every GT entry
        hit = top_ids[owner].long() == (g.long() + id_base).unsqueeze(1)               # (n_gt, K)
        pos = torch.where(hit.any(1), hit.float().argmax(1) + 1, torch.full_like(owner, K + 1))
        best = torch.full((M,), K + 1, dtype=torch.long, device=dev).scatter_reduce(0, owner, pos, "amin")
        return torch.where(best <= K, best, torch.maximum(r_dense, torch.full_like(r_dense, K + 1))).cpu().numpy()

    r = ranks(ptr, gts)
    rk = [100.0 * np.count_nonzero(r <= k) / M for k in (1, 5, 10, 100)]
    r1 = ranks(ptr1, first)
    return (rk[0], rk[1], rk[2], rk[3], np.median(r), r.mean(), float(np.mean(1.0 / r1)))


def _log_perf(m):
    logger.info(" * Text to Video:")
    logger.info(" * r_1_5_10_100: {}".format([round(x, 1) for x in m[:4]]))
    logger.info(" * recall sum: {}".format(round(sum(m[:4]), 1)))
    logger.info(" * mAP: {}".format(round(m[6], 4)))


def eval_epoch(model, val_video_dataset, val_text_dataset, opt, test=False):
    """R@1 + R@5 + R@10 + R@100 of the fused score (method/eval.py:237-263).

    opt.precision == "exact" (default): the reference's flow — dense per-branch matrices on the host, the three
    cal_perf reports (inheritance, exploration, fused).
    opt.precision in ("bf16", "fp16", "shortcut"): the hot path — engine.rank on the device (tcgen05 scoring +
    exact rescoring, top-100 identical to the exact path), R@K and the rank statistics computed on the device from
    the ranked lists; nothing of size Nq x Nv crosses to the host.  Only the fused report is produced
    (opt.per_branch_metrics = True adds the two single-branch reports at the cost of two more ranking passes)."""
    model.eval()
    precision = _opt(opt, "precision", "exact")
    if precision == "exact":
        with torch.no_grad():
            ctx = compute_context_info(model, val_video_dataset, opt)
            inher, explore, _, query_metas = compute_query2ctx_info(model, val_text_dataset, opt, ctx)
        _, t2v_gt = get_gt(ctx["video_metas"], query_metas)
        if _opt(opt, "double_branch", model.double_branch) and explore is not None:
            cal_perf(-1 * inher, t2v_gt, test)
            cal_perf(-1 * explore, t2v_gt, test)
            a = torch.from_numpy(inher).to(opt.device)
            b = torch.from_numpy(explore).to(opt.device)
            fused = ops.fuse_scores(a, b, 0.7, 0.3).cpu().numpy()
            r = cal_perf(-1 * fused, t2v_gt, test)
        else:
            r = cal_perf(-1 * inher, t2v_gt, test)
        return r[0] + r[1] + r[2] + r[3]
    with torch.no_grad():
        ctx = compute_context_info(model, val_video_dataset, opt)
        _, top_ids, query_metas, dense = rank_queries(model, val_text_dataset, opt, ctx, K=100, return_dense=True)
    _, t2v_gt = get_gt(ctx["video_metas"], query_metas)
    pc = ctx["prepared"]
    if _opt(opt, "per_branch_metrics", False) and model.double_branch:
        qs, _, _ = _encode_all_queries(model, val_text_dataset, opt)
        for bi in range(2):
            sub = engine.PreparedCorpus(Nv=pc.Nv, L=pc.L, D=pc.D, T=pc.T, id_base=pc.id_base, mask_u8=pc.mask_u8,
                                        lengths=pc.lengths, branches=[pc.branches[bi]], heads=pc.heads,
                                        Lg=pc.Lg, mask_g=pc.mask_g, Pg=pc.Pg, prop_mask=pc.prop_mask)
            pq = engine.prepare_queries([qs[bi]], want_bf16=precision == "bf16")
            _, ids_b, dense_b = engine.rank(sub, pq, K=100, head=_opt(opt, "scoring", "frame"), precision=precision,
                                            w_clip=model.clip_scale_w, w_frame=model.frame_scale_w, return_dense=True)
            _log_perf(metrics_from_ranking(ids_b, dense_b, t2v_gt, pc.id_base))
    m = metrics_from_ranking(top_ids, dense, t2v_gt, pc.id_base)
    _log_perf(m)
    return m[0] + m[1] + m[2] + m[3]

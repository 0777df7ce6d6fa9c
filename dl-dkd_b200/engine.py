"""Scoring engine: prepared corpus (resident in HBM) + per-query-batch scoring and ranking.

Two scoring heads
  "frame"      the head the reference ships: max over frames of cos(q, frame), masked
               (DLDKD.get_sim_scores, method/model.py:307-329), per branch; 0.7/0.3 fusion
               (method/eval.py:254).
  "two_scale"  the head north_star names (SURVEY §8 N1-N6): clip-scale max over the 528 clip
               proposals + key-clip-guided frame-scale score, w_clip/w_frame per branch, then 0.7/0.3.
Two precisions
  "exact"      fp32 SIMT kernels end to end (drop-in parity path).
  "bf16"       tcgen05 bf16 GEMM for the dense contraction (the hot kernel), approximate fused
               scores (<= 1e-3 abs), per-query top-Kc candidates re-scored by the exact fp32 kernels,
               so the returned top-K (ids, scores) equal the exact path's.

HBM layout per branch (Nv videos, L frames, D features, T clips, P = T(T+1)/2 proposals):
  frames_n   (Nv, L, D) fp32   L2-normalised frames          frame head, exact (per-frame output)
  frame_planes (Nv, D/32, 2, L, 32) fp32  tf32 hi/lo planes of frames_n, smem image   frame head, exact + rescoring
  frames_b   (Nv*L, D)  bf16   same, GEMM B operand          frame head, bf16
  clips      (Nv, T, D) fp32   downsampled clips  two-scale, exact + rescoring
  prop_scale (Nv, P)    fp32   1/(w*||mean||)                two-scale, exact + rescoring
  prop_b     (Nv*P, D)  bf16   L2-normalised proposals       two-scale GEMM B operand
  table_f    (Nv, P, D) fp32   normalised attention outputs  frame-scale, exact + rescoring
  table_h    (Nv, P, D) fp16   same                          frame-scale gather of the bf16 path
TVR shape, both branches: 2 x (428 + 214 + 107 + 5 + 884 + 1767 + 884 MB) = 8.6 GB of 180 GB.
"""
import math
from dataclasses import dataclass, field
from typing import List, Optional

import numpy as np
import torch
import torch.nn.functional as F

from . import ops

BRANCH_WEIGHTS = (0.7, 0.3)  # inheritance, exploration: method/eval.py:254


@dataclass
class BranchData:
    frames_n: Optional[torch.Tensor] = None
    frames_b: Optional[torch.Tensor] = None
    frame_planes: Optional[torch.Tensor] = None
    clips: Optional[torch.Tensor] = None
    clip_planes: Optional[torch.Tensor] = None
    prop_scale: Optional[torch.Tensor] = None
    prop_b: Optional[torch.Tensor] = None
    prop_h: Optional[torch.Tensor] = None       # IEEE-half proposals: GEMM B operand of precision="fp16"
    frames_h: Optional[torch.Tensor] = None     # IEEE-half frames: frame head, precision="fp16"
    table_f: Optional[torch.Tensor] = None
    table_h: Optional[torch.Tensor] = None


@dataclass
class PreparedCorpus:
    Nv: int
    L: int
    D: int
    T: int
    id_base: int
    mask_u8: torch.Tensor          # (Nv, L)
    lengths: torch.Tensor          # (Nv,) int32
    branches: List[BranchData] = field(default_factory=list)
    heads: tuple = ("frame", "two_scale")
    # rows per video as the tcgen05 GEMM sees them: the kernel needs R % 16 == 0, so frames / proposals are padded
    # with masked zero rows (frame head: Lg >= L, mask_g (Nv, Lg); two-scale head: Pg >= P, prop_mask (Nv, Pg) | None)
    Lg: int = 0
    mask_g: Optional[torch.Tensor] = None
    Pg: int = 0
    prop_mask: Optional[torch.Tensor] = None

    @property
    def P(self):
        return ops.num_proposals(self.T)

    def nbytes(self):
        tot = 0
        for b in self.branches:
            for t in vars(b).values():
                if t is not None:
                    tot += t.numel() * t.element_size()
        return tot


def prepare_corpus(frames_by_branch, mask, attn_params=None, T=ops.T_CLIPS, heads=("frame", "two_scale"),
                   precisions=("exact", "bf16"), id_base=0) -> PreparedCorpus:
    """Query-independent corpus preparation (run once; hoists the per-call F.normalize of
    method/model.py:319 and builds the two-scale operands).

    frames_by_branch: list of (Nv, L, D) fp32 CUDA tensors from encode_context (1 or 2 branches).
    mask: (Nv, L) {0,1}.  attn_params: per branch (key_w, key_b, val_w, val_b) of the key-clip
    attention (needed for the two_scale head).
    """
    f0 = frames_by_branch[0]
    Nv, L, D = f0.shape
    mask = mask.to(f0.device)
    mask_u8 = (mask > 0).to(torch.uint8).contiguous()
    lengths = mask_u8.sum(dim=1).to(torch.int32).contiguous()
    pc = PreparedCorpus(Nv=Nv, L=L, D=D, T=T, id_base=id_base, mask_u8=mask_u8, lengths=lengths, heads=tuple(heads))
    P = ops.num_proposals(T)
    pc.Lg, pc.Pg = ops.round_up(L, 16), ops.round_up(P, 16)
    pc.mask_g = mask_u8
    if pc.Lg != L:
        pc.mask_g = torch.zeros((Nv, pc.Lg), dtype=torch.uint8, device=f0.device)
        pc.mask_g[:, :L] = mask_u8
    if pc.Pg != P:
        pc.prop_mask = torch.zeros((Nv, pc.Pg), dtype=torch.uint8, device=f0.device)
        pc.prop_mask[:, :P] = 1
    if Nv == 0:  # an empty shard (more ranks than videos): nothing to prepare, rank() returns padding
        pc.branches = [BranchData() for _ in frames_by_branch]
        return pc

    def pad_rows(t, R, Rg):
        """(Nv * R, D) GEMM operand -> (Nv * Rg, D) with zero rows appended to every video (masked in the kernel)."""
        if t is None or Rg == R:
            return t
        out = torch.zeros((Nv, Rg, D), dtype=t.dtype, device=t.device)
        out[:, :R] = t.view(Nv, R, D)
        return out.view(Nv * Rg, D)

    for bi, fr in enumerate(frames_by_branch):
        fr = fr.contiguous().float()
        bd = BranchData()
        if "frame" in heads:
            approx = "bf16" in precisions or "fp16" in precisions
            out = ops.normalize_rows(fr, want_f32="exact" in precisions or approx,
                                     want_bf16="bf16" in precisions, want_f16="fp16" in precisions)
            fn, fb, fh = out if len(out) == 3 else (out[0], out[1], None)
            bd.frames_n = None if fn is None else fn.view(Nv, L, D)
            bd.frames_b = pad_rows(fb, L, pc.Lg)
            bd.frames_h = pad_rows(fh, L, pc.Lg)
            if bd.frames_n is not None and D % 32 == 0:
                bd.frame_planes = ops.pack_rows(bd.frames_n)
        if "two_scale" in heads:
            if attn_params is None:
                raise ValueError("two_scale head needs the key/value projections (attn_params)")
            kw, kb, vw, vb = attn_params[bi]
            bd.clips = ops.downsample_clips(fr, lengths, T)
            bd.clip_planes = ops.pack_clips(bd.clips)
            pb, ps, _ = ops.build_proposals(bd.clips, want_bf16="bf16" in precisions, want_scale=True)
            bd.prop_b = None if pb is None else pad_rows(pb.view(-1, D), P, pc.Pg)
            bd.prop_scale = ps
            if "fp16" in precisions:
                bd.prop_h = pad_rows(ops.build_proposals_f16(bd.clips)[0].view(-1, D), P, pc.Pg)
            # W_k / W_v projections: plain library GEMMs in corpus preparation
            key = F.linear(fr, kw, kb).contiguous()
            val = F.linear(fr, vw, vb).contiguous()
            bd.table_f, bd.table_h = ops.frame_attn_table(key, val, bd.clips, lengths, want_f32=True,
                                                          want_f16=any(x in precisions for x in ("bf16", "fp16", "shortcut")))
            del key, val
        pc.branches.append(bd)
    return pc


@dataclass
class PreparedQueries:
    M: int
    Mpad: int
    qn: List[torch.Tensor]   # per branch (M, D) fp32 normalised
    qb: List[torch.Tensor]   # per branch (Mpad, D) bf16 normalised (or None): GEMM A operand
    qh: List[torch.Tensor]   # per branch (Mpad, D) fp16 normalised (or None): frame-scale gather operand


_PAD_WORDS = {}


@dataclass
class HitDetail:
    """What the ranking knows about each returned hit, aligned with its (scores, ids) (M, K); nb = 1 or 2 branches.
      arg    (M, K, nb) int32   two-scale head: the branch's key clip, a proposal index p in [0, P) (ops.proposal_window
                                gives its (w, s)); frame head: the branch's best frame l in [0, L)
      score  (M, K, nb) fp32    two-scale: the branch's clip-scale score; frame head: its max-over-frames cosine
      frame  (M, K, nb) fp32    two-scale: the branch's frame-scale score; None for the frame head
    Padding hits (id -1) have arg -1 and scores -inf.  These are the values the returned fused score was computed
    from: two-scale, per branch fl(w_b * (fl(w_clip * score) + fl(w_frame * frame))) (w_b = 1 for one branch), summed
    over the branches in order; frame head, fl(0.7 * score_0) + fl(0.3 * score_1), or score_0 for one branch.
    On the device the detail travels as payload words (pack / unpack): per branch (arg, score bits[, frame bits])."""
    arg: torch.Tensor
    score: torch.Tensor
    frame: Optional[torch.Tensor] = None

    @staticmethod
    def pad_words(nb, two_scale, device=None):
        """(C,) int32 payload words of a padding hit: arg -1, scores -inf (cached per device: no copy per call)."""
        key = (nb, bool(two_scale), str(device))
        if key not in _PAD_WORDS:
            ninf = torch.tensor([float("-inf")], dtype=torch.float32).view(torch.int32).item()
            _PAD_WORDS[key] = torch.tensor(([-1, ninf, ninf] if two_scale else [-1, ninf]) * nb, dtype=torch.int32,
                                           device=device)
        return _PAD_WORDS[key]

    @classmethod
    def padding(cls, M, K, nb, two_scale, device=None):
        return cls.unpack(cls.pad_words(nb, two_scale, device).expand(M, K, -1), nb, two_scale)

    def pack(self) -> torch.Tensor:
        """(M, K, C) int32 payload words, C = nb * (3 for two-scale, 2 for the frame head)."""
        M, K, nb = self.arg.shape
        parts = [self.arg, self.score.view(torch.int32)]
        if self.frame is not None:
            parts.append(self.frame.view(torch.int32))
        return torch.stack(parts, dim=-1).reshape(M, K, nb * len(parts))

    @classmethod
    def unpack(cls, words, nb, two_scale):
        M, K, _ = words.shape
        w = words.reshape(M, K, nb, 3 if two_scale else 2)
        return cls(arg=w[..., 0].contiguous(), score=w[..., 1].contiguous().view(torch.float32),
                   frame=w[..., 2].contiguous().view(torch.float32) if two_scale else None)

    @classmethod
    def cat(cls, details):
        return cls(arg=torch.cat([d.arg for d in details]), score=torch.cat([d.score for d in details]),
                   frame=None if details[0].frame is None else torch.cat([d.frame for d in details]))

    def patch(self, idx, other):
        """Overwrite the rows idx (query indices) with other's rows, in place."""
        self.arg[idx] = other.arg
        self.score[idx] = other.score
        if self.frame is not None:
            self.frame[idx] = other.frame


def _gather_detail(ids, id_base, args, scores, frames=None):
    """HitDetail of top-K ids read from the dense per-branch (M, Nv) matrices of the scoring pass."""
    valid = (ids >= 0).unsqueeze(-1)
    n = (ids.long() - id_base).clamp_(min=0)

    def take(mats, fill):
        out = torch.stack([m.gather(1, n) for m in mats], dim=-1)
        return out.masked_fill_(~valid, fill)

    return HitDetail(arg=take(args, -1), score=take(scores, float("-inf")),
                     frame=None if frames is None else take(frames, float("-inf")))


def prepare_queries(q_by_branch, want_bf16=True) -> PreparedQueries:
    M = q_by_branch[0].shape[0]
    Mpad = ops.round_up(max(M, 1), 256)  # 2 x 128: CTA pairs own two query tiles
    qn, qb, qh = [], [], []
    if M == 0:
        return PreparedQueries(M=0, Mpad=Mpad, qn=[q.float() for q in q_by_branch], qb=[None] * len(q_by_branch),
                               qh=[None] * len(q_by_branch))
    for q in q_by_branch:
        f, b, h = ops.normalize_rows(q.contiguous().float(), want_f32=True, want_bf16=want_bf16, rows_pad=Mpad,
                                     want_f16=True)
        qn.append(f[:M])
        qb.append(b)
        qh.append(h)
    return PreparedQueries(M=M, Mpad=Mpad, qn=qn, qb=qb, qh=qh)


def _branch_weights(nb):
    return BRANCH_WEIGHTS[:nb] if nb == 2 else (1.0,)


def _exact_rows(bd: BranchData, qn, pc: PreparedCorpus, csr=None):
    """Exact max/argmax over the frames: tcgen05 kind::tf32 path when the packed planes exist (D % 32 == 0),
    the SIMT fp32 kernel otherwise."""
    if bd.frame_planes is not None:
        return ops.score_max_exact(qn, bd.frame_planes, pc.L, pc.mask_u8, csr=csr)
    s, a, _ = ops.score_max_f32(qn, bd.frames_n, pc.mask_u8, csr=csr)
    return s, a


def score_frame_head(pc: PreparedCorpus, pq: PreparedQueries, precision="exact", want_arg=False):
    """Per-branch dense (M, Nv) scores of the reference head. Returns list of (scores, argmax)."""
    out = []
    for bd, qn, qb, qh in zip(pc.branches, pq.qn, pq.qb, pq.qh):
        if precision == "exact":
            s, a = _exact_rows(bd, qn, pc)
        elif precision == "fp16":
            s, a = ops.score_max_bf16(qh, pq.M, bd.frames_h, pc.Nv, pc.Lg, pc.mask_g)
        else:
            s, a = ops.score_max_bf16(qb, pq.M, bd.frames_b, pc.Nv, pc.Lg, pc.mask_g)
        out.append((s, a))
    return out


AMBIGUITY_TAU = 1.0e-3  # bf16 argmax gaps below this are re-resolved in fp32 (DESIGN.md "bf16 and the key clip")
# precision="fp16": IEEE-half GEMM operands have 11 significant bits instead of 8 — every operand-rounding bound
# shrinks by 8: ambiguity threshold, and the dense-score error bound behind the candidate certificate
AMBIGUITY_TAU_F16 = AMBIGUITY_TAU / 8


def score_two_scale_head(pc: PreparedCorpus, pq: PreparedQueries, precision="exact", w_clip=0.7, w_frame=0.3,
                         want_frame=False, tau=None):
    """Returns (fused (M, Nv), per-branch list of dict(clip, key_clip, frame|None)).

    precision="bf16": the tcgen05 GEMM also flags (one bit per pair) the (query, video) pairs whose gap between
    the best and the runner-up proposal is small.  The key clip steers the frame-scale term discontinuously, so pairs whose
    gap is below `tau` (the bf16 noise floor on score differences) get their clip score and key clip
    recomputed by the exact kernel before the frame-scale gather; tau=0 disables the pass.  Then the key clip of a pair
    whose best windows tie above the 4 low mantissa bits is any one of them (dkd_score_max_bf16's tie rule), not
    necessarily the first; tau > 0 always re-resolves such pairs, whose gap is 0."""
    nb = len(pc.branches)
    wbs = _branch_weights(nb)
    fused = None
    per = []
    if tau is None:
        tau = AMBIGUITY_TAU_F16 if precision == "fp16" else AMBIGUITY_TAU
    for bi, (bd, qn, qb, qh) in enumerate(zip(pc.branches, pq.qn, pq.qb, pq.qh)):
        if precision == "exact":
            s_clip, k_clip = ops.clip_score_f32(qn, bd.clip_planes, bd.prop_scale)
            q, tab = qn, bd.table_f
        elif precision == "shortcut":
            # exact clip scale through the linearity shortcut (32 per-clip dots on tcgen05 kind::tf32 x 3 + window
            # scan): exact key clips for EVERY pair, so no ambiguity pass; only the frame-scale gather is approximate
            s_clip, k_clip = ops.clip_score_f32(qn, bd.clip_planes, bd.prop_scale)
            q, tab = qh, bd.table_h
        else:
            if precision == "fp16":
                qb, prop = qh, bd.prop_h
            else:
                prop = bd.prop_b
            if tau > 0:
                # the GEMM's epilogue appends every ambiguous pair to its video's list; the exact kernel re-resolves
                # the listed pairs and writes them into the dense matrices in place
                s_clip, k_clip, cnt, lst = ops.score_max_bf16_lists(qb, pq.M, prop, pc.Nv, pc.Pg, tau, mask=pc.prop_mask)
                ops.clip_score_list(qn, bd.clip_planes, bd.prop_scale, cnt, lst, s_clip, k_clip)
            else:
                s_clip, k_clip = ops.score_max_bf16(qb, pq.M, prop, pc.Nv, pc.Pg, mask=pc.prop_mask)
            q, tab = qh, bd.table_h
        wb = wbs[bi] if nb == 2 else 1.0
        fused, fr = ops.frame_fuse(q, tab, s_clip, k_clip, w_clip, w_frame, wb, fused=fused, accumulate=bi > 0,
                                   want_frame=want_frame)
        per.append(dict(clip=s_clip, key_clip=k_clip, frame=fr))
    return fused, per


CERT_EPS = 1.0e-3   # bound on |approximate fused score - exact fused score| (north_star tolerance; asserted on dense
                    # scores at full size by tests/test_gpu_configs.py::test_config_dense_error_within_certificate_eps)
CERT_EPS_F16 = 2.5e-4
STATS = {"certify_fallback_queries": 0, "certify_checked_queries": 0}


class PendingCertificate:
    """The device-side outcome of one rank() call's candidate certificate, to be looked at later (certify="deferred"):
    `count` reaches pinned host memory through an asynchronous copy, `resolve()` waits for it and — only if some query
    failed the check — re-ranks those queries by the all-exact path and patches the returned tensors in place."""

    def __init__(self, pc, pq, unsure, out_s, out_i, args, detail=None):
        self.pc, self.pq, self.unsure, self.out_s, self.out_i, self.args = pc, pq, unsure, out_s, out_i, args
        self.detail = detail
        self.host = torch.empty((1,), dtype=torch.int32).pin_memory()
        self.host.copy_(unsure.sum(dtype=torch.int32).reshape(1), non_blocking=True)
        self.event = torch.cuda.Event()
        self.event.record()

    def resolve(self):
        self.event.synchronize()
        return _apply_fallback(self.pc, self.pq, self.unsure, int(self.host[0]), self.out_s, self.out_i, self.args,
                               self.detail)


PENDING: List[PendingCertificate] = []


def finish(keep_last=0):
    """Resolve the deferred certificates (see rank(certify="deferred")), oldest first, all but the `keep_last` most
    recent ones (a pipelined consumer checks call i - 1 while call i is running: that wait never stalls).  Returns the
    number of queries that had to be re-ranked by the exact path."""
    n = 0
    while len(PENDING) > keep_last:
        n += PENDING.pop(0).resolve()
    return n


def poll():
    """Resolve, without blocking, the deferred certificates whose outcome has already reached the host (oldest first).
    rank() calls this on entry, so a stream of deferred calls keeps at most the last few outcomes — and the buffers
    they reference — alive; without it every call would have to allocate fresh device memory."""
    n = 0
    while PENDING and PENDING[0].event.query():
        n += PENDING.pop(0).resolve()
    return n


# ------------------------------------------------------------------------------------------------
# List depth.  The warp-per-row kernels (dkd_topk[_filtered], dkd_merge_topk[_payload], dkd_sort_candidates[_payload])
# hold a whole list in one warp's shared memory and stop at K = 256 / Kc = 512; the block-level deep kernels take
# K <= 4,096 and Kc <= 8,192.  This is the one place that chooses between them: shallow lists keep the warp kernels
# (the same C-ABI calls as before the deep kernels existed), everything else goes deep.
SHALLOW_K = 256
SHALLOW_KC = 512


def candidate_depth(K, Kc):
    """Candidates rank() rescores for a top-K: max(Kc, K) for K <= 256; for deeper lists
    max(Kc, round_up(K + K // 4, 32)), capped at 8,192 — the 25 % slack of K = 100 / Kc = 128.  Measured with it
    (DESIGN.md §8e, 4,096 queries x 16,384 videos, bf16): no query failed the certificate at K = 100, 1,000 or 4,096."""
    if K <= SHALLOW_K:
        return max(Kc, K)
    return max(Kc, min(ops.round_up(K + K // 4, 32), ops.DEEP_KC))


def _check_depth(who, K, Kc):
    """ValueError for a list depth the kernels do not take, before anything runs on the device."""
    if isinstance(K, bool) or not isinstance(K, (int, np.integer)) or not 1 <= K <= ops.DEEP_K:
        raise ValueError(f"{who}: K must be an int in [1, {ops.DEEP_K}], got {K!r}")
    if Kc > ops.DEEP_KC:
        raise ValueError(f"{who}: Kc must be at most {ops.DEEP_KC}, got {Kc}")


def _topk(fused, K, id_base, video_filter=None):
    if K > SHALLOW_K:
        return ops.topk_deep(fused, K, id_base, words=video_filter)
    if video_filter is None:
        return ops.topk(fused, K, id_base)
    return ops.topk_filtered(fused, K, video_filter, id_base)


def _sort(cand_scores, cand, K, words=None, pad=None):
    """The K best of (M, Kc) rescored candidates [+ their (M, Kc, C) payload words]."""
    if K > SHALLOW_K or cand.shape[1] > SHALLOW_KC:
        return ops.sort_candidates_deep(cand_scores, cand, K, payload=words, pad=pad)
    if words is None:
        return ops.sort_candidates(cand_scores, cand, K)
    return ops.sort_candidates_payload(cand_scores, cand, words, K, pad)


def _apply_fallback(pc, pq, unsure, n_unsure, out_s, out_i, args, detail=None):
    STATS["certify_checked_queries"] += pq.M
    STATS["certify_fallback_queries"] += n_unsure
    if n_unsure:
        nb = len(pc.branches)
        idx = unsure.nonzero().squeeze(1)
        sub = PreparedQueries(M=n_unsure, Mpad=ops.round_up(n_unsure, 256), qn=[q[idx].contiguous() for q in pq.qn],
                              qb=[None] * nb, qh=[None] * nb)
        vf = args.get("video_filter")
        if vf is not None and vf.shape[0] != 1:          # per-query filter: the rows of the re-ranked queries
            args = dict(args, video_filter=vf[idx].contiguous())
        if detail is None:
            es, ei = rank(pc, sub, precision="exact", **args)
        else:
            es, ei, ed = rank(pc, sub, precision="exact", return_detail=True, **args)
            detail.patch(idx, ed)
        out_s[idx] = es
        out_i[idx] = ei
    return n_unsure


def make_video_filter(n_videos, allow=None, deny=None, device=None):
    """Video filter words for rank(video_filter=): (Mf, ceil(n_videos / 32)) int32 on `device` (default: the current
    CUDA device), bit (g & 31) of word (g >> 5) of a row set when global video id g may be returned.

    Exactly one of `allow` (only these videos) and `deny` (every video of [0, n_videos) but these) is given, either as
    one list of video ids (a filter shared by every query, Mf = 1) or as a list of per-query id lists (Mf = number of
    queries).  Duplicate ids are harmless; an id outside [0, n_videos) raises ValueError before anything runs on the
    device.  The words cost 4 * ceil(n_videos / 32) bytes per row."""
    if (allow is None) == (deny is None):
        raise ValueError("make_video_filter: give exactly one of allow= and deny=")
    lists = allow if deny is None else deny
    shared = len(lists) == 0 or np.ndim(lists[0]) == 0
    rows = [np.asarray(r, dtype=np.int64).reshape(-1) for r in ([lists] if shared else lists)]
    ids = np.concatenate(rows) if rows else np.zeros(0, np.int64)
    if ids.size and (ids.min() < 0 or ids.max() >= n_videos):
        bad = ids[(ids < 0) | (ids >= n_videos)][0]
        raise ValueError(f"make_video_filter: video id {bad} is outside [0, {n_videos})")
    ptr = np.zeros(len(rows) + 1, np.int64)
    np.cumsum([len(r) for r in rows], out=ptr[1:])
    dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    return ops.build_video_filter(torch.from_numpy(ptr.astype(np.int32)).to(dev),
                                  torch.from_numpy(ids.astype(np.int32)).to(dev), n_videos, deny=deny is not None)


def rank(pc: PreparedCorpus, pq: PreparedQueries, K=100, head="two_scale", precision="bf16", rescore=True,
         Kc=128, w_clip=0.7, w_frame=0.3, tau=None, certify=True, return_dense=False, return_detail=False,
         video_filter=None):
    """Per-query top-K (scores (M,K) fp32, global video ids (M,K) int32) of the fused score
    [+ the dense (M, Nv) fused matrix of the scoring pass when return_dense]
    [+ the HitDetail of every hit when return_detail: key clip / best frame and per-branch scores].

    K: 1 .. 4,096 (ValueError outside).  Lists up to 256 deep use the warp-per-row kernels, deeper ones the block-level
    deep kernels (candidate_depth, DESIGN.md §8e); the result is the same top-K either way.
    precision="bf16" + rescore: bf16 GEMM scores pick candidate_depth(K, Kc) candidates per query: Kc >= K for
    K <= 256, at least round_up(1.25 K, 32) for deeper lists (Kc <= 8,192, ValueError above); the exact fp32
    kernels re-score them, the K best survive.  certify: a query's list is accepted only if its exact K-th
    score exceeds the approximate score of the last candidate by more than CERT_EPS — every non-candidate
    scores at most that approximate value, so (approximation error <= CERT_EPS) none of them can belong in the
    top-K.  The few queries that fail the check are re-ranked by the all-exact path, which makes the result equal
    to precision="exact" for every query instead of "for every query we tested".
      certify=True        the check is read back immediately (one scalar device->host read per call);
      certify="deferred"  no host synchronisation: the outcome is queued in PENDING and engine.finish() — called by
                          the consumer before it reads the lists — applies the (rare) exact re-rank in place; outcomes
                          that have already reached the host are resolved on the next rank() entry (engine.poll()).
    return_detail: the detail is produced where each hit's score is (the candidate rescoring kernels write it beside
    the score, and the sort moves it with its hit; the dense route reads it from the scoring pass at the top-K ids),
    and the certificate's re-rank patches it with the scores.
    video_filter: (1 or M, W) int32 words of make_video_filter, indexed by global video id: only the videos a query's
    row allows can be hits (padding (-inf, -1) when fewer than K are allowed).  The filter acts where the hits are
    chosen (the dense top-K, the candidate selection), so the result equals precision="exact" with the same filter.
    The scoring pass still scores every pair: the dense matrix of return_dense is unfiltered.
    """
    _check_depth("rank", K, Kc)
    nb = len(pc.branches)
    wbs = _branch_weights(nb)
    two = head != "frame"
    if video_filter is not None and (video_filter.dim() != 2 or video_filter.shape[0] not in (1, pq.M)):
        raise ValueError(f"video_filter: expected (1, W) or ({pq.M}, W) words, got {tuple(video_filter.shape)}")
    if PENDING:
        poll()
    if pq.M == 0 or pc.Nv == 0:  # no queries / empty shard: K columns of padding (score -inf, id -1), like dkd_topk
        dev = pc.mask_u8.device
        out = (torch.full((pq.M, K), float("-inf"), dtype=torch.float32, device=dev),
               torch.full((pq.M, K), -1, dtype=torch.int32, device=dev))
        if return_dense:
            out += (torch.empty((pq.M, pc.Nv), dtype=torch.float32, device=dev),)
        return out + (HitDetail.padding(pq.M, K, nb, two, dev),) if return_detail else out
    dense_route = precision == "exact" or not rescore
    per = None
    if head == "frame":
        if precision == "shortcut":
            raise ValueError("precision='shortcut' is a two-scale variant (the frame head has no clip windows)")
        sc = score_frame_head(pc, pq, precision)
        fused = sc[0][0] if nb == 1 else ops.fuse_scores(sc[0][0], sc[1][0], wbs[0], wbs[1])
    else:
        fused, per = score_two_scale_head(pc, pq, precision, w_clip, w_frame, tau=tau,
                                          want_frame=return_detail and dense_route)
    extra = (fused,) if return_dense else ()
    if dense_route:
        out_s, out_i = _topk(fused, K, pc.id_base, video_filter)
        if return_detail:
            if head == "frame":
                det = _gather_detail(out_i, pc.id_base, [a for _, a in sc], [s for s, _ in sc])
            else:
                det = _gather_detail(out_i, pc.id_base, [p["key_clip"] for p in per], [p["clip"] for p in per],
                                     [p["frame"] for p in per])
            extra += (det,)
        return (out_s, out_i) + extra
    Kc = candidate_depth(K, Kc)
    # the candidates are rescored and sorted below: only their SET and the Kc-th approximate score are needed here
    if video_filter is None:
        cand, approx_kth = ops.select_topk(fused, Kc, pc.id_base)
    else:
        cand, approx_kth = ops.select_topk_filtered(fused, Kc, video_filter, pc.id_base)
    csr = ops.candidates_to_csr(cand, pc.Nv, pc.id_base)
    cand_scores = torch.full((pq.M, Kc), float("-inf"), dtype=torch.float32, device=cand.device)
    # payload words of every candidate (HitDetail.pack layout); every valid candidate's slot is written below
    words = torch.empty((pq.M, Kc, nb * (3 if two else 2)), dtype=torch.int32, device=cand.device) if return_detail \
        else None
    if head == "frame":
        ex = [_exact_rows(bd, qn, pc, csr=csr[:2]) for bd, qn in zip(pc.branches, pq.qn)]
        if return_detail:
            b, ab = (ex[1][0], ex[1][1]) if nb == 2 else (None, None)
            ops.scatter_fuse_detail(ex[0][0], b, wbs[0], wbs[1] if nb == 2 else 0.0, ex[0][1], ab, csr, cand_scores,
                                    words)
        elif nb == 2:
            ops.scatter_fuse(ex[0][0], ex[1][0], wbs[0], wbs[1], csr, cand_scores)
        else:
            ops.scatter_fuse(ex[0][0], None, 1.0, 0.0, csr, cand_scores)
    else:
        for bi, (bd, qn) in enumerate(zip(pc.branches, pq.qn)):
            if precision == "shortcut":     # the dense clip scores / key clips are already exact
                cs, ck = per[bi]["clip"], per[bi]["key_clip"]
            else:
                # the dense key clips are final at this point (exact for the flagged pairs, unambiguous for the
                # rest): the exact kernel confirms them against the exact maximum instead of searching all windows
                cs, ck = ops.clip_score_f32(qn, bd.clip_planes, bd.prop_scale, csr=csr[:2],
                                            known_key=per[bi]["key_clip"])
            wb = wbs[bi] if nb == 2 else 1.0
            if return_detail:
                ops.frame_fuse_csr_detail(qn, bd.table_f, cs, ck, csr, w_clip, w_frame, wb, cand_scores, bi > 0,
                                          words, 3 * bi)
            else:
                ops.frame_fuse_csr(qn, bd.table_f, cs, ck, csr, w_clip, w_frame, wb, cand_scores, bi > 0)
    detail = None
    if return_detail:
        out_s, out_i, out_w = _sort(cand_scores, cand, K, words, HitDetail.pad_words(nb, two, cand.device))
        detail = HitDetail.unpack(out_w, nb, two)
    else:
        out_s, out_i = _sort(cand_scores, cand, K)
    if certify and Kc < pc.Nv:
        unsure = out_s[:, K - 1] <= approx_kth + (CERT_EPS if precision == "bf16" else CERT_EPS_F16)
        args = dict(K=K, head=head, w_clip=w_clip, w_frame=w_frame)
        if video_filter is not None:
            # a query with at most Kc allowed videos has all of them as candidates (approx_kth = -inf): certain
            unsure &= ~torch.isneginf(approx_kth)
            args["video_filter"] = video_filter
        if certify == "deferred":
            PENDING.append(PendingCertificate(pc, pq, unsure, out_s, out_i, args, detail))
        else:
            _apply_fallback(pc, pq, unsure, int(unsure.sum()), out_s, out_i, args, detail)
    return (out_s, out_i) + extra + ((detail,) if return_detail else ())


@dataclass
class Moments:
    """The top-m distinct moments of each hit of localize(), aligned with its (M, K) ids.
      arg    (M, K, m) int32   proposal index p in [0, P) of the window (ops.proposal_window gives its (w, s));
                               -1 for padding
      score  (M, K, m) fp32    the window's clip-scale moment score; -inf for padding
    Along m the scores are non-increasing, and no two windows of a hit overlap by an IoU above the call's iou."""
    arg: torch.Tensor
    score: torch.Tensor


def localize(pc: PreparedCorpus, pq: PreparedQueries, ids, m=5, iou=0.5) -> Moments:
    """Where in each hit's video the query matches: the top-m windows of every (query, video) pair of `ids` after
    temporal non-maximum suppression, ranked by the exact clip-scale curve of the two-scale head.

    ids: (pq.M, K) int32 global video ids on the device, normally the ids rank() returned (any list works, duplicates are
    harmless).  Ids of -1 and ids outside [id_base, id_base + Nv) get padding (arg -1, score -inf).
    Moment score of window p(w, s) (DESIGN.md §8d): per branch S_b(p) = fl(fl(d_b[s] + ... + d_b[s+w-1]) *
    prop_scale_b[n, p]), with d_b the query's per-clip dots; one branch: S_0(p); two: fl(0.7 S_0(p)) + fl(0.3 S_1(p))
    (BRANCH_WEIGHTS).  So with one branch the first moment's score is the clip score of HitDetail bit for bit, and its
    window is the hit's key clip (except where the key clip is an exact fp32 tie with an earlier window of the same
    length, the known-key residual); with two branches the fused curve's maximum need not be either branch's key clip.
    NMS: m greedy rounds pick the best unsuppressed window (the lower p on equal scores) and suppress every window
    whose IoU with it, fl(inter / union) over clip intervals [s, s + w), is above iou.  iou >= 1: plain top-m;
    iou = 0: pairwise-disjoint windows.  Ranks left when every window is suppressed are padding.
    Shards: every hit is owned by exactly one shard and padding is (-1, -inf), so when each shard localizes the merged
    global id list, the elementwise maximum of the shards' arg and score is the whole corpus's answer.
    engine.moment_frames(moments.arg, ids, lengths) gives the frame window of every moment."""
    if "two_scale" not in pc.heads:
        raise ValueError("localize: the corpus was prepared without the two-scale head (it has no clip windows)")
    if isinstance(m, bool) or not isinstance(m, int) or not 1 <= m <= 16:
        raise ValueError(f"localize: m must be an int in [1, 16], got {m!r}")
    iou = float(iou)
    if math.isnan(iou) or iou < 0:
        raise ValueError(f"localize: iou must be >= 0, got {iou}")
    if not (isinstance(ids, torch.Tensor) and ids.dtype == torch.int32 and ids.dim() == 2 and ids.shape[0] == pq.M):
        raise ValueError(f"localize: ids must be a ({pq.M}, K) int32 tensor")
    M, K = ids.shape
    if M == 0 or K == 0 or pc.Nv == 0:
        return Moments(arg=torch.full((M, K, m), -1, dtype=torch.int32, device=ids.device),
                       score=torch.full((M, K, m), float("-inf"), dtype=torch.float32, device=ids.device))
    csr = ops.candidates_to_csr(ids.contiguous(), pc.Nv, pc.id_base)
    dots = [ops.clip_dots_list(qn, bd.clip_planes, csr, pc.T) for bd, qn in zip(pc.branches, pq.qn)]
    arg, score = ops.moment_nms(dots, [bd.prop_scale for bd in pc.branches], csr, M, K, m, iou,
                                weights=BRANCH_WEIGHTS)
    return Moments(arg=arg, score=score)


def moment_frames(arg, ids, lengths, T=ops.T_CLIPS, head="two_scale"):
    """Frame windows of the hits: (M, K, nb, 2) int32 [first, end) in the encoded frame sequence of each hit's video.

    arg (M, K, nb) = HitDetail.arg, ids (M, K) global video ids, lengths: valid frames per global video id.
    Two-scale head: the frames whose features were averaged into the key clip's clips s .. s + w - 1 by
    average_to_fixed_length (method/data_provider.py:30-50): clip i of a video of n frames averages frames
    [a_i, a_{i+1}) with a_i = min(round(i * n / T), n - 1), or the single frame a_i when a_i >= a_{i+1}.  The window
    is therefore [a_s, max(a_{s+w}, a_{s+w-1} + 1)) — with the reference's quirks: the clamp to n - 1 means that for
    many lengths the last valid frame is averaged into no clip.  Frame head: [l, l + 1).  Padding hits: (-1, -1)."""
    valid = (ids >= 0).unsqueeze(-1) & (arg >= 0)
    if head == "frame":
        first, end = arg.long(), arg.long() + 1
    else:
        P = ops.num_proposals(T)
        ws = torch.tensor([ops.proposal_window(p, T) for p in range(P)], dtype=torch.long, device=arg.device)
        p = arg.long().clamp(0, P - 1)
        w, s = ws[p, 0], ws[p, 1]
        n = torch.as_tensor(lengths, device=arg.device)[ids.long().clamp(min=0)].unsqueeze(-1).expand_as(arg)
        nf, nl = n.float(), n.long()

        def a(i):   # torch.arange(0, T + 1, 1.0) / T * n, rounded half to even, clamped to n - 1
            return torch.minimum(torch.round(i.float() / T * nf).long(), nl - 1)

        first, end = a(s), torch.maximum(a(s + w), a(s + w - 1) + 1)
    out = torch.stack([first, end], dim=-1).to(torch.int32)
    return out.masked_fill_(~valid.unsqueeze(-1), -1)


def shard_range(Nv: int, rank_: int, world: int):
    """Contiguous video shard [lo, hi) of rank_ (SURVEY §8e)."""
    per = (Nv + world - 1) // world
    lo = min(rank_ * per, Nv)
    return lo, min(lo + per, Nv)


def _merge_lists(scores, ids, words=None, pad=None):
    """(G, M, K) lists [+ (G, M, K, C) payload words] -> the merged (M, K) lists [+ (M, K, C) words].  Every list the
    engine merges comes from rank(), a sort or a merge: sorted, padding at the end, as the deep merge requires."""
    if scores.shape[-1] > SHALLOW_K:
        return ops.merge_topk_deep(scores, ids, payload=words, pad=pad)
    if words is None:
        return ops.merge_topk(scores, ids)
    return ops.merge_topk_payload(scores, ids, words, pad)


def merge_shards(local_scores, local_ids, group=None, merge_fn=None, exchange="query_block", gather=True, detail=None):
    """Global per-query top-K from every rank's local top-K (NCCL over NVLink on the GPU box).

    exchange="query_block" (default; SURVEY §8e's lower-volume alternative): one all-to-all hands rank r every
    rank's lists for query block r (M/G queries), rank r merges only that block with dkd_merge_topk, and — when
    `gather` — one all-gather of the merged blocks gives every rank the full (M, K) result.  Per rank that is
    2 x M*K*8 bytes received and M/G merges instead of G x M*K*8 bytes and M merges for exchange="all_gather"
    (every rank gathers every list and merges every query).  With gather=False the return value is
    (scores, ids, (q_lo, q_hi)): the merged block this rank owns.
    detail: the local HitDetail of the lists (rank(return_detail=True)); it travels with its hits through the same
    exchange (as payload words) and the merged HitDetail is appended to the return value.
    merge_fn overrides the merge kernel (CPU gloo tests): merge_fn(scores (G, M, K), ids) -> (scores, ids), and with
    a detail merge_fn(scores, ids, words (G, M, K, C)) -> (scores, ids, words)."""
    import torch.distributed as dist
    world = dist.get_world_size(group)
    M, K = local_scores.shape
    if detail is None:
        merge = merge_fn or _merge_lists
        local = [local_scores.contiguous(), local_ids.contiguous()]
        finish = tuple
    else:
        nb, two = detail.arg.shape[-1], detail.frame is not None
        pad = HitDetail.pad_words(nb, two, local_scores.device)
        merge = merge_fn or (lambda s, i, w: _merge_lists(s, i, w, pad))
        local = [local_scores.contiguous(), local_ids.contiguous(), detail.pack()]

        def finish(res):
            return (res[0], res[1], HitDetail.unpack(res[2], nb, two))
    if world == 1:
        res = finish(local)
        return res if gather else res[:2] + ((0, M),) + res[2:]
    dev = local_scores.device
    nccl = dist.get_backend(group) == "nccl"
    if exchange == "all_gather":
        gathered = [torch.empty((world,) + t.shape, dtype=t.dtype, device=dev) for t in local]
        for g, t in zip(gathered, local):
            if nccl:
                dist.all_gather_into_tensor(g, t, group=group)
            else:  # gloo (CPU tests): list form
                dist.all_gather(list(g.unbind(0)), t, group=group)
        res = finish(merge(*gathered))
        return res if gather else res[:2] + ((0, M),) + res[2:]
    if exchange != "query_block":
        raise ValueError("exchange must be 'query_block' or 'all_gather'")
    # No packing / padding / reshaping kernels: the (M, K) lists are sent as they are with ROW splits (rank g receives
    # rows [g*Mb, (g+1)*Mb) of every rank), the merge kernel writes this rank's block into a fixed-size (Mb, K)
    # buffer, and the all-gather of those buffers IS the (world*Mb, K) result in query order — [:M] is a view.
    # Payload words ride along as (M, K * C) rows.
    rank_ = dist.get_rank(group)
    Mb = (M + world - 1) // world
    q_lo, q_hi = min(rank_ * Mb, M), min((rank_ + 1) * Mb, M)
    mine = q_hi - q_lo
    in_split = [min((g + 1) * Mb, M) - min(g * Mb, M) for g in range(world)]
    recv = [torch.empty((world, mine) + t.shape[1:], dtype=t.dtype, device=dev) for t in local]
    for r, t in zip(recv, local):
        row = math.prod(t.shape[1:])
        dist.all_to_all_single(r.view(world * mine, row), t.view(M, row), [mine] * world, in_split, group=group)
    if mine:
        block = list(merge(*recv))                                                     # (mine, K): my query block
    else:
        block = [r.new_empty((0,) + r.shape[2:]) for r in recv]
    if not gather:
        res = finish(block)
        return res[:2] + ((q_lo, q_hi),) + res[2:]
    if mine != Mb:       # only the last block(s) can be short: pad to the common size (-inf, -1), sliced away below
        fills = [float("-inf"), -1, -1]
        block = [torch.cat([b, b.new_full((Mb - mine,) + b.shape[1:], f)]) for b, f in zip(block, fills)]
    full = [torch.empty((world * Mb,) + b.shape[1:], dtype=b.dtype, device=dev) for b in block]
    for f, b in zip(full, block):
        if nccl:
            dist.all_gather_into_tensor(f, b.contiguous(), group=group)
        else:
            dist.all_gather(list(f.view((world, Mb) + b.shape[1:]).unbind(0)), b.contiguous(), group=group)
    return finish([f[:M] for f in full])


# ------------------------------------------------------------------------------------------------
# Streamed corpus (BASELINE.json configs[3]: 1 M videos x 32 clips, 100 k queries, 8 GPUs).
# The prepared operands of a 125 k-video shard (prop_b + table_h + table_f: 2.4 MB per video and branch) do
# not fit 180 GB, the encoded clips (49 KB per video and branch) do.  So the shard stays resident as encoded
# frames and is scored chunk by chunk: build the chunk's operands, score every query batch against it, fold
# the chunk's per-query top-K into the running top-K.  Operand building is ~2 % of a chunk's GEMM time at
# 100 k queries, so nothing is gained by keeping more than one chunk of operands alive.
def split_queries(q_by_branch, batch=16384):
    """Encoded query vectors (per branch (Nq, D)) -> list of PreparedQueries of at most `batch` queries."""
    Nq = q_by_branch[0].shape[0]
    return [prepare_queries([q[lo: lo + batch] for q in q_by_branch]) for lo in range(0, max(Nq, 1), batch)]


def iter_chunks(frames_by_branch, mask, chunk_videos=8192, id_base=0):
    """Slice a resident shard of encoded frames into (frames_by_branch, mask, id_base) chunks."""
    Nv = frames_by_branch[0].shape[0]
    for lo in range(0, Nv, chunk_videos):
        hi = min(lo + chunk_videos, Nv)
        yield [f[lo:hi] for f in frames_by_branch], mask[lo:hi], id_base + lo


def rank_streamed(chunks, pqs, attn_params=None, K=100, T=ops.T_CLIPS, head="two_scale", precision="bf16",
                  rescore=True, Kc=128, w_clip=0.7, w_frame=0.3, tau=None, return_detail=False, video_filter=None):
    """Per-query top-K over a corpus presented as successive chunks of videos.

    chunks: iterable of (frames_by_branch, mask, id_base) — e.g. iter_chunks() over a resident shard, or a
    generator that reads / synthesises one chunk at a time.  pqs: list of PreparedQueries (split_queries).
    Returns (scores (Nq, K), ids (Nq, K) int32) [+ HitDetail when return_detail]: identical to rank() over the
    concatenated corpus, because every (query, video) score is produced by the same kernels on the same rows and the
    ordering (score desc, id asc) is total, so a merge of per-chunk top-K lists is the global top-K (the detail moves
    with its hit through that merge).
    video_filter: as for rank(), with one row per query of all the batches together (or one shared row); the words are
    indexed by global id, so every chunk reads the same words."""
    _check_depth("rank_streamed", K, Kc)
    running = [None] * len(pqs)
    offs = np.cumsum([0] + [pq.M for pq in pqs])
    if video_filter is not None and video_filter.shape[0] not in (1, offs[-1]):
        raise ValueError(f"video_filter: expected (1, W) or ({offs[-1]}, W) words, got {tuple(video_filter.shape)}")
    vfs = [video_filter if video_filter is None or video_filter.shape[0] == 1 else video_filter[offs[b]: offs[b + 1]]
           for b in range(len(pqs))]
    precisions = ("exact", precision) if precision != "exact" else ("exact",)
    for frames, mask, id_base in chunks:
        pc = prepare_corpus(frames, mask, attn_params, T=T, heads=(head,), precisions=precisions, id_base=id_base)
        for b, pq in enumerate(pqs):
            out = rank(pc, pq, K=K, head=head, precision=precision, rescore=rescore, Kc=Kc, w_clip=w_clip,
                       w_frame=w_frame, tau=tau, return_detail=return_detail, video_filter=vfs[b])
            if running[b] is None:
                running[b] = out
            elif not return_detail:
                running[b] = _merge_lists(torch.stack([running[b][0], out[0]]), torch.stack([running[b][1], out[1]]))
            else:
                d = out[2]
                s, i, w = _merge_lists(torch.stack([running[b][0], out[0]]), torch.stack([running[b][1], out[1]]),
                                       torch.stack([running[b][2].pack(), d.pack()]),
                                       HitDetail.pad_words(d.arg.shape[-1], d.frame is not None, d.arg.device))
                running[b] = (s, i, HitDetail.unpack(w, d.arg.shape[-1], d.frame is not None))
        del pc
    if any(r is None for r in running):
        raise ValueError("rank_streamed: the corpus has no chunks")
    res = (torch.cat([r[0] for r in running]), torch.cat([r[1] for r in running]))
    return res + (HitDetail.cat([r[2] for r in running]),) if return_detail else res

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
from dataclasses import dataclass, field
from typing import List, Optional

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

    def __init__(self, pc, pq, unsure, out_s, out_i, args):
        self.pc, self.pq, self.unsure, self.out_s, self.out_i, self.args = pc, pq, unsure, out_s, out_i, args
        self.host = torch.empty((1,), dtype=torch.int32).pin_memory()
        self.host.copy_(unsure.sum(dtype=torch.int32).reshape(1), non_blocking=True)
        self.event = torch.cuda.Event()
        self.event.record()

    def resolve(self):
        self.event.synchronize()
        return _apply_fallback(self.pc, self.pq, self.unsure, int(self.host[0]), self.out_s, self.out_i, self.args)


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


def _apply_fallback(pc, pq, unsure, n_unsure, out_s, out_i, args):
    STATS["certify_checked_queries"] += pq.M
    STATS["certify_fallback_queries"] += n_unsure
    if n_unsure:
        nb = len(pc.branches)
        idx = unsure.nonzero().squeeze(1)
        sub = PreparedQueries(M=n_unsure, Mpad=ops.round_up(n_unsure, 256), qn=[q[idx].contiguous() for q in pq.qn],
                              qb=[None] * nb, qh=[None] * nb)
        es, ei = rank(pc, sub, precision="exact", **args)
        out_s[idx] = es
        out_i[idx] = ei
    return n_unsure


def rank(pc: PreparedCorpus, pq: PreparedQueries, K=100, head="two_scale", precision="bf16", rescore=True,
         Kc=128, w_clip=0.7, w_frame=0.3, tau=None, certify=True, return_dense=False):
    """Per-query top-K (scores (M,K) fp32, global video ids (M,K) int32) of the fused score
    [+ the dense (M, Nv) fused matrix of the scoring pass when return_dense].

    precision="bf16" + rescore: bf16 GEMM scores pick Kc >= K candidates per query, the exact fp32
    kernels re-score them, the K best survive.  certify: a query's list is accepted only if its exact K-th
    score exceeds the approximate score of the last candidate by more than CERT_EPS — every non-candidate
    scores at most that approximate value, so (approximation error <= CERT_EPS) none of them can belong in the
    top-K.  The few queries that fail the check are re-ranked by the all-exact path, which makes the result equal
    to precision="exact" for every query instead of "for every query we tested".
      certify=True        the check is read back immediately (one scalar device->host read per call);
      certify="deferred"  no host synchronisation: the outcome is queued in PENDING and engine.finish() — called by
                          the consumer before it reads the lists — applies the (rare) exact re-rank in place; outcomes
                          that have already reached the host are resolved on the next rank() entry (engine.poll()).
    """
    nb = len(pc.branches)
    wbs = _branch_weights(nb)
    if PENDING:
        poll()
    if pq.M == 0 or pc.Nv == 0:  # no queries / empty shard: K columns of padding (score -inf, id -1), like dkd_topk
        dev = pc.mask_u8.device
        out = (torch.full((pq.M, K), float("-inf"), dtype=torch.float32, device=dev),
               torch.full((pq.M, K), -1, dtype=torch.int32, device=dev))
        return out + (torch.empty((pq.M, pc.Nv), dtype=torch.float32, device=dev),) if return_dense else out
    per = None
    if head == "frame":
        if precision == "shortcut":
            raise ValueError("precision='shortcut' is a two-scale variant (the frame head has no clip windows)")
        sc = score_frame_head(pc, pq, precision)
        fused = sc[0][0] if nb == 1 else ops.fuse_scores(sc[0][0], sc[1][0], wbs[0], wbs[1])
    else:
        fused, per = score_two_scale_head(pc, pq, precision, w_clip, w_frame, tau=tau)
    extra = (fused,) if return_dense else ()
    if precision == "exact" or not rescore:
        return ops.topk(fused, K, pc.id_base) + extra
    Kc = max(Kc, K)
    # the candidates are rescored and sorted below: only their SET and the Kc-th approximate score are needed here
    cand, approx_kth = ops.select_topk(fused, Kc, pc.id_base)
    csr = ops.candidates_to_csr(cand, pc.Nv, pc.id_base)
    cand_scores = torch.full((pq.M, Kc), float("-inf"), dtype=torch.float32, device=cand.device)
    if head == "frame":
        ex = [_exact_rows(bd, qn, pc, csr=csr[:2])[0] for bd, qn in zip(pc.branches, pq.qn)]
        if nb == 2:
            ops.scatter_fuse(ex[0], ex[1], wbs[0], wbs[1], csr, cand_scores)
        else:
            ops.scatter_fuse(ex[0], None, 1.0, 0.0, csr, cand_scores)
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
            ops.frame_fuse_csr(qn, bd.table_f, cs, ck, csr, w_clip, w_frame, wb, cand_scores, bi > 0)
    out_s, out_i = ops.sort_candidates(cand_scores, cand, K)
    if certify and Kc < pc.Nv:
        unsure = out_s[:, K - 1] <= approx_kth + (CERT_EPS if precision == "bf16" else CERT_EPS_F16)
        args = dict(K=K, head=head, w_clip=w_clip, w_frame=w_frame)
        if certify == "deferred":
            PENDING.append(PendingCertificate(pc, pq, unsure, out_s, out_i, args))
        else:
            _apply_fallback(pc, pq, unsure, int(unsure.sum()), out_s, out_i, args)
    return (out_s, out_i) + extra


def shard_range(Nv: int, rank_: int, world: int):
    """Contiguous video shard [lo, hi) of rank_ (SURVEY §8e)."""
    per = (Nv + world - 1) // world
    lo = min(rank_ * per, Nv)
    return lo, min(lo + per, Nv)


def merge_shards(local_scores, local_ids, group=None, merge_fn=None, exchange="query_block", gather=True):
    """Global per-query top-K from every rank's local top-K (NCCL over NVLink on the GPU box).

    exchange="query_block" (default; SURVEY §8e's lower-volume alternative): one all-to-all hands rank r every
    rank's lists for query block r (M/G queries), rank r merges only that block with dkd_merge_topk, and — when
    `gather` — one all-gather of the merged blocks gives every rank the full (M, K) result.  Per rank that is
    2 x M*K*8 bytes received and M/G merges instead of G x M*K*8 bytes and M merges for exchange="all_gather"
    (every rank gathers every list and merges every query).  With gather=False the return value is
    (scores, ids, (q_lo, q_hi)): the merged block this rank owns.
    merge_fn overrides the merge kernel (CPU gloo tests)."""
    import torch.distributed as dist
    merge_fn = merge_fn or ops.merge_topk
    world = dist.get_world_size(group)
    M, K = local_scores.shape
    if world == 1:
        return (local_scores, local_ids) if gather else (local_scores, local_ids, (0, M))
    dev = local_scores.device
    if exchange == "all_gather":
        gs = torch.empty((world, M, K), dtype=torch.float32, device=dev)
        gi = torch.empty((world, M, K), dtype=torch.int32, device=dev)
        if dist.get_backend(group) == "nccl":
            dist.all_gather_into_tensor(gs, local_scores.contiguous(), group=group)
            dist.all_gather_into_tensor(gi, local_ids.contiguous(), group=group)
        else:  # gloo (CPU tests): list form
            dist.all_gather(list(gs.unbind(0)), local_scores.contiguous(), group=group)
            dist.all_gather(list(gi.unbind(0)), local_ids.contiguous(), group=group)
        ms, mi = merge_fn(gs, gi)
        return (ms, mi) if gather else (ms, mi, (0, M))
    if exchange != "query_block":
        raise ValueError("exchange must be 'query_block' or 'all_gather'")
    # No packing / padding / reshaping kernels: the (M, K) lists are sent as they are with ROW splits (rank g receives
    # rows [g*Mb, (g+1)*Mb) of every rank), the merge kernel writes this rank's block into a fixed-size (Mb, K)
    # buffer, and the all-gather of those buffers IS the (world*Mb, K) result in query order — [:M] is a view.
    rank_ = dist.get_rank(group)
    Mb = (M + world - 1) // world
    q_lo, q_hi = min(rank_ * Mb, M), min((rank_ + 1) * Mb, M)
    mine = q_hi - q_lo
    in_split = [min((g + 1) * Mb, M) - min(g * Mb, M) for g in range(world)]
    rs = torch.empty((world, mine, K), dtype=torch.float32, device=dev)
    ri = torch.empty((world, mine, K), dtype=torch.int32, device=dev)
    dist.all_to_all_single(rs.view(world * mine, K), local_scores.contiguous(), [mine] * world, in_split, group=group)
    dist.all_to_all_single(ri.view(world * mine, K), local_ids.contiguous(), [mine] * world, in_split, group=group)
    if mine:
        bs, bi = merge_fn(rs, ri)                                                       # (mine, K): my query block
    else:
        bs, bi = rs.new_empty((0, K)), ri.new_empty((0, K))
    if not gather:
        return bs, bi, (q_lo, q_hi)
    if mine != Mb:       # only the last block(s) can be short: pad to the common size (-inf, -1), sliced away below
        bs = torch.cat([bs, bs.new_full((Mb - mine, K), float("-inf"))])
        bi = torch.cat([bi, bi.new_full((Mb - mine, K), -1)])
    fs = torch.empty((world * Mb, K), dtype=torch.float32, device=dev)
    fi = torch.empty((world * Mb, K), dtype=torch.int32, device=dev)
    if dist.get_backend(group) == "nccl":
        dist.all_gather_into_tensor(fs, bs.contiguous(), group=group)
        dist.all_gather_into_tensor(fi, bi.contiguous(), group=group)
    else:
        dist.all_gather(list(fs.view(world, Mb, K).unbind(0)), bs.contiguous(), group=group)
        dist.all_gather(list(fi.view(world, Mb, K).unbind(0)), bi.contiguous(), group=group)
    return fs[:M], fi[:M]


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
                  rescore=True, Kc=128, w_clip=0.7, w_frame=0.3, tau=None):
    """Per-query top-K over a corpus presented as successive chunks of videos.

    chunks: iterable of (frames_by_branch, mask, id_base) — e.g. iter_chunks() over a resident shard, or a
    generator that reads / synthesises one chunk at a time.  pqs: list of PreparedQueries (split_queries).
    Returns (scores (Nq, K), ids (Nq, K) int32): identical to rank() over the concatenated corpus, because every
    (query, video) score is produced by the same kernels on the same rows and the ordering (score desc, id asc)
    is total, so a merge of per-chunk top-K lists is the global top-K."""
    running = [None] * len(pqs)
    precisions = ("exact", precision) if precision != "exact" else ("exact",)
    for frames, mask, id_base in chunks:
        pc = prepare_corpus(frames, mask, attn_params, T=T, heads=(head,), precisions=precisions, id_base=id_base)
        for b, pq in enumerate(pqs):
            s, i = rank(pc, pq, K=K, head=head, precision=precision, rescore=rescore, Kc=Kc, w_clip=w_clip,
                        w_frame=w_frame, tau=tau)
            if running[b] is None:
                running[b] = (s, i)
            else:
                running[b] = ops.merge_topk(torch.stack([running[b][0], s]), torch.stack([running[b][1], i]))
        del pc
    if any(r is None for r in running):
        raise ValueError("rank_streamed: the corpus has no chunks")
    return torch.cat([r[0] for r in running]), torch.cat([r[1] for r in running])

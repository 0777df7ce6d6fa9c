"""Tensor-level wrappers over the C ABI (include/dkd_b200.h).

PyTorch is plumbing here: it allocates device buffers and provides the current stream; every
number is produced by the hand-written kernels in csrc/.  All inputs must be CUDA tensors.
"""
import torch

from . import _lib

T_CLIPS = 32  # clips per video of the two-scale head (map_size); P = T(T+1)/2 = 528


def num_proposals(T: int = T_CLIPS) -> int:
    return T * (T + 1) // 2


def proposal_index(w: int, s: int, T: int = T_CLIPS) -> int:
    """Index of the window (length w, start s): SURVEY §8 N2 ordering."""
    return (w - 1) * T - ((w - 1) * (w - 2)) // 2 + s


def proposal_window(p: int, T: int = T_CLIPS):
    """(w, s) of proposal p: the inverse of proposal_index (window length w = 1..T, start s = 0..T-w)."""
    if not 0 <= p < num_proposals(T):
        raise ValueError(f"proposal {p} out of range for T = {T}")
    w = 1
    while p >= T - w + 1:
        p -= T - w + 1
        w += 1
    return w, p


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _p(t):
    return None if t is None else t.data_ptr()


def _chk(t, dtype, name):
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise _lib.DkdError(f"{name}: expected a CUDA tensor (dkd_b200 has no CPU path)")
    if t.dtype != dtype:
        raise _lib.DkdError(f"{name}: expected dtype {dtype}, got {t.dtype}")
    if not t.is_contiguous():
        raise _lib.DkdError(f"{name}: expected a contiguous tensor")
    return t


def round_up(x: int, m: int) -> int:
    return (x + m - 1) // m * m


def normalize_rows(x, want_f32=True, want_bf16=False, rows_pad=None, eps=1e-12, want_f16=False):
    """F.normalize(x, dim=-1) (method/model.py:318-319) -> (fp32 | None, bf16 | None[, fp16]), each (rows_pad, D).
    The fp16 copy (operand of the frame-scale gather) is returned as a third element when want_f16."""
    _chk(x, torch.float32, "x")
    D = x.shape[-1]
    rows = x.numel() // D
    rows_pad = rows if rows_pad is None else rows_pad
    of = torch.empty((rows_pad, D), dtype=torch.float32, device=x.device) if want_f32 else None
    ob = torch.empty((rows_pad, D), dtype=torch.bfloat16, device=x.device) if want_bf16 else None
    oh = torch.empty((rows_pad, D), dtype=torch.float16, device=x.device) if want_f16 else None
    _lib.call("dkd_normalize_rows", _p(x), rows, D, eps, _p(of), _p(ob), _p(oh), rows_pad, _stream())
    return (of, ob, oh) if want_f16 else (of, ob)


def downsample_clips(frames, lengths, T=T_CLIPS):
    """average_to_fixed_length (method/data_provider.py:30-50) per video: (Nv, L, D) -> (Nv, T, D)."""
    _chk(frames, torch.float32, "frames")
    _chk(lengths, torch.int32, "lengths")
    Nv, L, D = frames.shape
    clips = torch.empty((Nv, T, D), dtype=torch.float32, device=frames.device)
    _lib.call("dkd_downsample_clips", _p(frames), _p(lengths), Nv, L, D, T, _p(clips), _stream())
    return clips


def build_proposals_f16(clips, want_scale=False):
    """(Nv, T, D) clips -> (prop_f16 (Nv,P,D) normalised IEEE-half rows, prop_scale (Nv,P) | None)."""
    _chk(clips, torch.float32, "clips")
    Nv, T, D = clips.shape
    P = num_proposals(T)
    ph = torch.empty((Nv, P, D), dtype=torch.float16, device=clips.device)
    ps = torch.empty((Nv, P), dtype=torch.float32, device=clips.device) if want_scale else None
    _lib.call("dkd_build_proposals_f16", _p(clips), Nv, T, D, _p(ph), _p(ps), _stream())
    return ph, ps


def build_proposals(clips, want_bf16=True, want_scale=True, want_f32=False):
    """(Nv, T, D) clips -> (prop_bf16 (Nv,P,D) normalised, prop_scale (Nv,P), prop_f32 (Nv,P,D) means)."""
    _chk(clips, torch.float32, "clips")
    Nv, T, D = clips.shape
    P = num_proposals(T)
    dev = clips.device
    pb = torch.empty((Nv, P, D), dtype=torch.bfloat16, device=dev) if want_bf16 else None
    ps = torch.empty((Nv, P), dtype=torch.float32, device=dev) if want_scale else None
    pf = torch.empty((Nv, P, D), dtype=torch.float32, device=dev) if want_f32 else None
    _lib.call("dkd_build_proposals", _p(clips), Nv, T, D, _p(pb), _p(ps), _p(pf), _stream())
    return pb, ps, pf


def score_max_f32(qn, xn, mask=None, want_rows=False, csr=None):
    """Exact fp32 get_sim_scores core: qn (M,D), xn (Nv,R,D) normalised -> (max (M,Nv), argmax, rows|None)."""
    _chk(qn, torch.float32, "qn")
    _chk(xn, torch.float32, "xn")
    M, D = qn.shape
    Nv, R, _ = xn.shape
    dev = qn.device
    if mask is not None:
        _chk(mask, torch.uint8, "mask")
    rows = torch.empty((M, R, Nv), dtype=torch.float32, device=dev) if want_rows else None
    if csr is None:
        om = torch.empty((M, Nv), dtype=torch.float32, device=dev)
        oa = torch.empty((M, Nv), dtype=torch.int32, device=dev)
        _lib.call("dkd_score_max_f32", _p(qn), M, _p(xn), Nv, R, D, _p(mask), _p(om), _p(oa), Nv, _p(rows),
                  None, None, _stream())
    else:
        vid_ptr, q_list = csr
        E = q_list.numel()
        om = torch.empty((E,), dtype=torch.float32, device=dev)
        oa = torch.empty((E,), dtype=torch.int32, device=dev)
        _lib.call("dkd_score_max_f32", _p(qn), M, _p(xn), Nv, R, D, _p(mask), _p(om), _p(oa), 0, _p(rows),
                  _p(vid_ptr), _p(q_list), _stream())
    return om, oa, rows


def pack_rows(xn):
    """(Nv, R, D) normalised rows (R <= 128) -> (Nv, D/32, 2, Rpad, 32) fp32: the pre-packed B operand of
    score_max_exact (tf32 hi / lo planes in the shared-memory layout; once per corpus)."""
    _chk(xn, torch.float32, "xn")
    Nv, R, D = xn.shape
    if D % 32 or R > 128:
        raise _lib.DkdError("pack_rows: D must be a multiple of 32 and R <= 128")
    planes = torch.empty((Nv, D // 32, 2, round_up(R, 16), 32), dtype=torch.float32, device=xn.device)
    _lib.call("dkd_pack_rows_tf32", _p(xn), Nv, R, D, _p(planes), _stream())
    return planes


def score_max_exact(qn, planes, R, mask=None, csr=None):
    """Exact get_sim_scores core on the tcgen05 kind::tf32 path: qn (M, D) normalised queries, planes =
    pack_rows(xn) -> (max (M, Nv), first argmax).  csr = (vid_ptr, q_list): listed pairs only, entry order."""
    _chk(qn, torch.float32, "qn")
    _chk(planes, torch.float32, "row_planes")
    M, D = qn.shape
    Nv = planes.shape[0]
    if planes.dim() != 5 or planes.shape[1] * 32 != D or planes.shape[3] != round_up(R, 16):
        raise _lib.DkdError("score_max_exact: row planes do not match (R, D)")
    if mask is not None:
        _chk(mask, torch.uint8, "mask")
    dev = qn.device
    if csr is None:
        om = torch.empty((M, Nv), dtype=torch.float32, device=dev)
        oa = torch.empty((M, Nv), dtype=torch.int32, device=dev)
        _lib.call("dkd_score_max_exact", _p(qn), M, _p(planes), Nv, R, D, _p(mask), _p(om), _p(oa), Nv, None, None,
                  _stream())
    else:
        vid_ptr, q_list = csr
        E = q_list.numel()
        om = torch.empty((E,), dtype=torch.float32, device=dev)
        oa = torch.empty((E,), dtype=torch.int32, device=dev)
        _lib.call("dkd_score_max_exact", _p(qn), M, _p(planes), Nv, R, D, _p(mask), _p(om), _p(oa), 0, _p(vid_ptr),
                  _p(q_list), _stream())
    return om, oa


def pack_clips(clips):
    """(Nv, T, D) clips -> (Nv, D/32, 2, 32, 32) fp32: the pre-packed B operand of the exact clip-scale kernel
    (tf32 hi / lo planes in the shared-memory layout; once per corpus)."""
    _chk(clips, torch.float32, "clips")
    Nv, T, D = clips.shape
    if D % 32:
        raise _lib.DkdError("pack_clips: D must be a multiple of 32")
    planes = torch.empty((Nv, D // 32, 2, 32, 32), dtype=torch.float32, device=clips.device)
    _lib.call("dkd_pack_clips_tf32", _p(clips), Nv, T, D, _p(planes), _stream())
    return planes


def clip_score_f32(qn, clips, prop_scale, csr=None, scatter=None, known_key=None):
    """Exact clip-scale max/argmax over the P proposals via per-clip dots (SURVEY §8 N3) on the tcgen05
    kind::tf32 path.  qn (M, D) normalised queries; clips: (Nv, T, D) fp32 or its pack_clips() form (5-D).
    csr = (vid_ptr, q_list) [CSR by video] or (vid_begin, q_list, vid_cnt) [select_flagged runs]: only the listed
    (query, video) pairs, results in entry order; with scatter = (slot, out_max, out_arg) entry e is written
    into the dense matrices at slot[e] instead.  known_key (list form): dense (M, Nv) int32 key clips to confirm
    instead of searching (same results; see include/dkd_b200.h)."""
    _chk(qn, torch.float32, "qn")
    _chk(prop_scale, torch.float32, "prop_scale")
    planes = clips if clips.dim() == 5 else pack_clips(clips)
    _chk(planes, torch.float32, "clip_planes")
    M, D = qn.shape
    Nv, P = prop_scale.shape
    T = int(round(((8 * P + 1) ** 0.5 - 1) / 2))
    if planes.shape[0] != Nv or planes.shape[1] * 32 != D or T * (T + 1) // 2 != P:
        raise _lib.DkdError("clip_score_f32: clip planes / prop_scale / query shapes do not agree")
    dev = qn.device
    if csr is None:
        om = torch.empty((M, Nv), dtype=torch.float32, device=dev)
        oa = torch.empty((M, Nv), dtype=torch.int32, device=dev)
        _lib.call("dkd_clip_score_f32", _p(qn), M, _p(planes), _p(prop_scale), Nv, T, D, _p(om), _p(oa), Nv,
                  None, None, None, None, None, 0, _stream())
        return om, oa
    vid_ptr, q_list = csr[0], csr[1]
    vid_cnt = csr[2] if len(csr) > 2 else None
    if scatter is not None:
        slot, om, oa = scatter
        _chk(om, torch.float32, "out_max")
        _chk(oa, torch.int32, "out_arg")
    else:
        slot = None
        E = q_list.numel()
        om = torch.empty((E,), dtype=torch.float32, device=dev)
        oa = torch.empty((E,), dtype=torch.int32, device=dev)
    if known_key is not None:
        _chk(known_key, torch.int32, "known_key")
        if T != 32 or known_key.shape != (M, Nv):
            known_key = None            # the confirm-the-key form exists for T = 32 only: full search
    _lib.call("dkd_clip_score_f32", _p(qn), M, _p(planes), _p(prop_scale), Nv, T, D, _p(om), _p(oa), 0,
              _p(vid_ptr), _p(vid_cnt), _p(q_list), _p(slot), _p(known_key), Nv if known_key is not None else 0, _stream())
    return om, oa


def score_max_bf16(q_bf16, M, x_bf16, Nv, R, mask=None, out_max=None, out_arg=None, want_gap=False, flag_tau=None):
    """tcgen05 GEMM + fused max/argmax: q_bf16 (Mpad,D), x_bf16 (Nv*R, D) -> (max (M,Nv), argmax (M,Nv))
    [+ gap (M,Nv) = best - runner-up when want_gap] [+ flags (M, ceil(Nv/32)) uint32 bit matrix of the pairs
    whose gap is below flag_tau].  Both operands bf16, or both IEEE half (dkd_score_max_f16)."""
    half = isinstance(q_bf16, torch.Tensor) and q_bf16.dtype == torch.float16
    _chk(q_bf16, torch.float16 if half else torch.bfloat16, "q_bf16")
    _chk(x_bf16, torch.float16 if half else torch.bfloat16, "x_bf16")
    Mpad, D = q_bf16.shape
    if x_bf16.numel() != Nv * R * D:
        raise _lib.DkdError("x_bf16 does not hold Nv*R rows of D features")
    if mask is not None:
        _chk(mask, torch.uint8, "mask")
    dev = q_bf16.device
    om = out_max if out_max is not None else torch.empty((M, Nv), dtype=torch.float32, device=dev)
    oa = out_arg if out_arg is not None else torch.empty((M, Nv), dtype=torch.int32, device=dev)
    og = torch.empty((M, Nv), dtype=torch.float32, device=dev) if want_gap else None
    fl = torch.zeros((M, (Nv + 31) // 32), dtype=torch.int32, device=dev) if flag_tau is not None else None
    _lib.call("dkd_score_max_f16" if half else "dkd_score_max_bf16", _p(q_bf16), M, Mpad, _p(x_bf16), Nv, R, D,
              _p(mask), _p(om), _p(oa), _p(og), Nv,
              _p(fl), float(flag_tau or 0.0), _stream())
    out = (om, oa)
    if want_gap:
        out += (og,)
    if flag_tau is not None:
        out += (fl,)
    return out


def score_max_bf16_lists(q, M, x, Nv, R, tau, mask=None):
    """The tcgen05 GEMM with the ambiguous-pair lists written by its epilogue: -> (max (M, Nv), argmax (M, Nv),
    flag_cnt (Nv,), flag_list (Nv, M)).  Operands both bf16 or both IEEE half."""
    half = q.dtype == torch.float16
    _chk(q, torch.float16 if half else torch.bfloat16, "q")
    _chk(x, torch.float16 if half else torch.bfloat16, "x")
    Mpad, D = q.shape
    if x.numel() != Nv * R * D:
        raise _lib.DkdError("x does not hold Nv*R rows of D features")
    if mask is not None:
        _chk(mask, torch.uint8, "mask")
    dev = q.device
    om = torch.empty((M, Nv), dtype=torch.float32, device=dev)
    oa = torch.empty((M, Nv), dtype=torch.int32, device=dev)
    cnt = torch.zeros((Nv,), dtype=torch.int32, device=dev)
    lst = torch.empty((Nv, M), dtype=torch.int32, device=dev)
    _lib.call("dkd_score_max_bf16_lists", _p(q), M, Mpad, _p(x), Nv, R, D, _p(mask), _p(om), _p(oa), Nv, float(tau),
              _p(cnt), _p(lst), M, int(half), _stream())
    return om, oa, cnt, lst


def clip_score_list(qn, planes, prop_scale, cnt, lst, out_max, out_arg):
    """Exact clip score / key clip of the listed pairs (score_max_bf16_lists), written in place into the dense
    (M, Nv) matrices."""
    _chk(qn, torch.float32, "qn")
    _chk(planes, torch.float32, "clip_planes")
    _chk(prop_scale, torch.float32, "prop_scale")
    _chk(cnt, torch.int32, "flag_cnt")
    _chk(lst, torch.int32, "flag_list")
    _chk(out_max, torch.float32, "out_max")
    _chk(out_arg, torch.int32, "out_arg")
    M, D = qn.shape
    Nv, P = prop_scale.shape
    T = int(round(((8 * P + 1) ** 0.5 - 1) / 2))
    _lib.call("dkd_clip_score_list", _p(qn), M, _p(planes), _p(prop_scale), Nv, T, D, _p(out_max), _p(out_arg),
              out_max.shape[1], _p(cnt), _p(lst), lst.shape[1], _stream())
    return out_max, out_arg


def select_flagged(flags, Nv, cap=None):
    """Bit matrix of flagged pairs (score_max_bf16 flag_tau) -> (vid_begin, q_list, vid_cnt, slot): per-video
    runs of query indices / dense slots m * Nv + n."""
    _chk(flags, torch.int32, "flags")
    M = flags.shape[0]
    cap = M * Nv if cap is None else cap
    dev = flags.device
    cursor = torch.empty((1,), dtype=torch.int32, device=dev)
    vid_begin = torch.empty((Nv,), dtype=torch.int32, device=dev)
    vid_cnt = torch.empty((Nv,), dtype=torch.int32, device=dev)
    q_list = torch.empty((cap,), dtype=torch.int32, device=dev)
    slot = torch.empty((cap,), dtype=torch.int32, device=dev)
    _lib.call("dkd_select_flagged", _p(flags), M, Nv, Nv, cap, _p(cursor), _p(vid_begin), _p(vid_cnt), _p(q_list),
              _p(slot), _stream())
    return vid_begin, q_list, vid_cnt, slot


def select_pairs_csr(gap, tau, cap=None):
    """CSR by video of the pairs whose bf16 argmax gap is below tau -> (vid_ptr, q_list, slot)."""
    _chk(gap, torch.float32, "gap")
    M, Nv = gap.shape
    cap = M * Nv if cap is None else cap
    dev = gap.device
    counts = torch.empty((Nv,), dtype=torch.int32, device=dev)
    vid_ptr = torch.empty((Nv + 1,), dtype=torch.int32, device=dev)
    q_list = torch.empty((cap,), dtype=torch.int32, device=dev)
    slot = torch.empty((cap,), dtype=torch.int32, device=dev)
    _lib.call("dkd_select_pairs_csr", _p(gap), M, Nv, Nv, tau, cap, _p(counts), _p(vid_ptr), _p(q_list), _p(slot),
              _stream())
    return vid_ptr, q_list, slot


def frame_attn_table(key, val, clips, lengths, want_f32=True, want_f16=True):
    """Key-clip-guided attention outputs for every proposal of every video (SURVEY §8 N4) -> (fp32, fp16) (Nv,P,D)."""
    _chk(key, torch.float32, "key")
    _chk(val, torch.float32, "val")
    _chk(clips, torch.float32, "clips")
    _chk(lengths, torch.int32, "lengths")
    Nv, L, D = key.shape
    T = clips.shape[1]
    P = num_proposals(T)
    dev = key.device
    E = torch.empty((Nv, L, T), dtype=torch.float32, device=dev)
    _lib.call("dkd_key_clip_dots", _p(key), _p(clips), Nv, L, T, D, _p(E), _stream())
    tf = torch.empty((Nv, P, D), dtype=torch.float32, device=dev) if want_f32 else None
    tb = torch.empty((Nv, P, D), dtype=torch.float16, device=dev) if want_f16 else None
    _lib.call("dkd_frame_attn_table", _p(E), _p(val), _p(lengths), Nv, L, T, D, _p(tf), _p(tb), _stream())
    return tf, tb


def frame_fuse(q, table, clip_scores, key_clip, w_clip, w_frame, w_branch, fused=None, accumulate=False,
               want_frame=False):
    """frame[m,n] = q[m].table[n,key_clip[m,n]]; fused (+)= w_branch*(w_clip*clip + w_frame*frame)."""
    is_f16 = q.dtype == torch.float16
    _chk(q, torch.float16 if is_f16 else torch.float32, "q")
    _chk(table, q.dtype, "table")
    _chk(key_clip, torch.int32, "key_clip")
    _chk(clip_scores, torch.float32, "clip_scores")
    M, Nv = key_clip.shape
    _, P, D = table.shape
    dev = key_clip.device
    fr = torch.empty((M, Nv), dtype=torch.float32, device=dev) if want_frame else None
    if fused is None:
        fused = torch.empty((M, Nv), dtype=torch.float32, device=dev)
        accumulate = False
    _lib.call("dkd_frame_fuse", _p(q), _p(table), int(is_f16), _p(clip_scores), _p(key_clip), M, Nv, P, D, Nv,
              w_clip, w_frame, w_branch, int(accumulate), _p(fr), _p(fused), _stream())
    return fused, fr


def fuse_scores(a, b, wa=0.7, wb=0.3):
    """fl(wa*a) + fl(wb*b): the numpy fusion of method/eval.py:254, bit-exact."""
    _chk(a, torch.float32, "a")
    _chk(b, torch.float32, "b")
    out = torch.empty_like(a)
    _lib.call("dkd_fuse_scores", _p(a), _p(b), wa, wb, _p(out), a.numel(), _stream())
    return out


def topk(scores, K, id_base=0):
    """Per-row top-K (score desc, id asc) of a dense (M, Nv) matrix -> (scores (M,K), ids (M,K) int32)."""
    _chk(scores, torch.float32, "scores")
    M, Nv = scores.shape
    os_ = torch.empty((M, K), dtype=torch.float32, device=scores.device)
    oi = torch.empty((M, K), dtype=torch.int32, device=scores.device)
    _lib.call("dkd_topk", _p(scores), M, Nv, Nv, K, id_base, _p(os_), _p(oi), _stream())
    return os_, oi


def select_topk(scores, K, id_base=0):
    """Per-row top-K SET (unsorted ids (M, K) int32, -1 padded) + the K-th best score (M,) of a dense (M, Nv) matrix."""
    _chk(scores, torch.float32, "scores")
    M, Nv = scores.shape
    oi = torch.empty((M, K), dtype=torch.int32, device=scores.device)
    kth = torch.empty((M,), dtype=torch.float32, device=scores.device)
    _lib.call("dkd_select_topk", _p(scores), M, Nv, Nv, K, id_base, _p(oi), _p(kth), _stream())
    return oi, kth


def merge_topk(scores, ids):
    """(G, M, K) shard lists -> merged (M, K)."""
    _chk(scores, torch.float32, "scores")
    _chk(ids, torch.int32, "ids")
    G, M, K = scores.shape
    os_ = torch.empty((M, K), dtype=torch.float32, device=scores.device)
    oi = torch.empty((M, K), dtype=torch.int32, device=scores.device)
    _lib.call("dkd_merge_topk", _p(scores), _p(ids), G, M, K, _p(os_), _p(oi), _stream())
    return os_, oi


def merge_topk_payload(scores, ids, payload, pad):
    """merge_topk + the (G, M, K, C) int32 payload words moved with their entry -> (scores (M, K), ids (M, K),
    payload (M, K, C)); ranks without an entry get the (C,) int32 words `pad`.  Ids must be distinct per query."""
    _chk(scores, torch.float32, "scores")
    _chk(ids, torch.int32, "ids")
    _chk(payload, torch.int32, "payload")
    G, M, K = scores.shape
    C = payload.shape[-1]
    if payload.shape != (G, M, K, C) or pad.shape != (C,):
        raise _lib.DkdError("merge_topk_payload: payload must be (G, M, K, C) and pad (C,)")
    dev = scores.device
    os_ = torch.empty((M, K), dtype=torch.float32, device=dev)
    oi = torch.empty((M, K), dtype=torch.int32, device=dev)
    op = pad.to(device=dev, dtype=torch.int32).expand(M, K, C).contiguous()
    _lib.call("dkd_merge_topk_payload", _p(scores), _p(ids), _p(payload), G, M, K, C, _p(os_), _p(oi), _p(op), _stream())
    return os_, oi, op


def rank_of_gt(scores, gt_ptr, gt_ids):
    """1-based rank of the best-ranked GT video per query (eval_q2m, method/eval.py:73-82)."""
    _chk(scores, torch.float32, "scores")
    _chk(gt_ptr, torch.int32, "gt_ptr")
    _chk(gt_ids, torch.int32, "gt_ids")
    M, Nv = scores.shape
    out = torch.empty((M,), dtype=torch.int32, device=scores.device)
    _lib.call("dkd_rank_of_gt", _p(scores), M, Nv, Nv, _p(gt_ptr), _p(gt_ids), _p(out), _stream())
    return out


def candidates_to_csr(cand_ids, Nv, id_base=0):
    """(M, K) candidate video ids -> per-video CSR (vid_ptr (Nv+1), q_list (M*K), slot (M*K))."""
    _chk(cand_ids, torch.int32, "cand_ids")
    M, K = cand_ids.shape
    dev = cand_ids.device
    counts = torch.empty((Nv,), dtype=torch.int32, device=dev)
    vid_ptr = torch.empty((Nv + 1,), dtype=torch.int32, device=dev)
    q_list = torch.zeros((M * K,), dtype=torch.int32, device=dev)
    slot = torch.zeros((M * K,), dtype=torch.int32, device=dev)
    _lib.call("dkd_candidates_to_csr", _p(cand_ids), M, K, Nv, id_base, _p(counts), _p(vid_ptr), _p(q_list),
              _p(slot), _stream())
    return vid_ptr, q_list, slot


def frame_fuse_csr(q, table, clip_scores, key_clip, csr, w_clip, w_frame, w_branch, cand_scores, accumulate):
    """clip_scores / key_clip: per-entry (E,) arrays, or dense (M, Nv) matrices (read at (query, video) of each entry)."""
    _chk(q, torch.float32, "q")
    _chk(table, torch.float32, "table")
    _chk(clip_scores, torch.float32, "clip_scores")
    _chk(key_clip, torch.int32, "key_clip")
    vid_ptr, q_list, slot = csr
    Nv, P, D = table.shape
    dense_ld = clip_scores.shape[1] if clip_scores.dim() == 2 else 0
    _lib.call("dkd_frame_fuse_csr", _p(q), _p(table), _p(clip_scores), _p(key_clip), _p(vid_ptr), _p(q_list),
              _p(slot), Nv, P, D, w_clip, w_frame, w_branch, int(accumulate), _p(cand_scores), dense_ld, _stream())
    return cand_scores


def sort_candidates(cand_scores, cand_ids, K_out):
    _chk(cand_scores, torch.float32, "cand_scores")
    _chk(cand_ids, torch.int32, "cand_ids")
    M, K = cand_ids.shape
    os_ = torch.empty((M, K_out), dtype=torch.float32, device=cand_ids.device)
    oi = torch.empty((M, K_out), dtype=torch.int32, device=cand_ids.device)
    _lib.call("dkd_sort_candidates", _p(cand_scores), _p(cand_ids), M, K, K_out, _p(os_), _p(oi), _stream())
    return os_, oi


def sort_candidates_payload(cand_scores, cand_ids, payload, K_out, pad):
    """sort_candidates + the (M, K, C) int32 payload words moved with their candidate -> (scores, ids, payload
    (M, K_out, C)); ranks without a candidate get the (C,) int32 words `pad`."""
    _chk(cand_scores, torch.float32, "cand_scores")
    _chk(cand_ids, torch.int32, "cand_ids")
    _chk(payload, torch.int32, "payload")
    M, K = cand_ids.shape
    C = payload.shape[-1]
    if payload.shape != (M, K, C) or pad.shape != (C,):
        raise _lib.DkdError("sort_candidates_payload: payload must be (M, K, C) and pad (C,)")
    dev = cand_ids.device
    os_ = torch.empty((M, K_out), dtype=torch.float32, device=dev)
    oi = torch.empty((M, K_out), dtype=torch.int32, device=dev)
    op = pad.to(device=dev, dtype=torch.int32).expand(M, K_out, C).contiguous()
    _lib.call("dkd_sort_candidates_payload", _p(cand_scores), _p(cand_ids), _p(payload), M, K, K_out, C, _p(os_),
              _p(oi), _p(op), _stream())
    return os_, oi, op


def frame_fuse_csr_detail(q, table, clip_scores, key_clip, csr, w_clip, w_frame, w_branch, cand_scores, accumulate,
                          payload, c0):
    """frame_fuse_csr that also writes (key clip, clip score bits, frame score bits) of every entry to
    payload[slot, c0:c0 + 3] (payload (M, K, C) int32)."""
    _chk(q, torch.float32, "q")
    _chk(table, torch.float32, "table")
    _chk(clip_scores, torch.float32, "clip_scores")
    _chk(key_clip, torch.int32, "key_clip")
    _chk(payload, torch.int32, "payload")
    vid_ptr, q_list, slot = csr
    Nv, P, D = table.shape
    dense_ld = clip_scores.shape[1] if clip_scores.dim() == 2 else 0
    _lib.call("dkd_frame_fuse_csr_detail", _p(q), _p(table), _p(clip_scores), _p(key_clip), _p(vid_ptr), _p(q_list),
              _p(slot), Nv, P, D, w_clip, w_frame, w_branch, int(accumulate), _p(cand_scores), dense_ld, _p(payload),
              payload.shape[-1], c0, _stream())
    return cand_scores


def scatter_fuse_detail(a, b, wa, wb, arg_a, arg_b, csr, cand_scores, payload):
    """scatter_fuse that also writes (arg_a, bits of a[, arg_b, bits of b]) of every entry to payload[slot]
    (payload (M, K, C) int32)."""
    vid_ptr, q_list, slot = csr
    _chk(a, torch.float32, "a")
    _chk(arg_a, torch.int32, "arg_a")
    _chk(payload, torch.int32, "payload")
    _lib.call("dkd_scatter_fuse_detail", _p(a), _p(b), wa, wb, _p(arg_a), _p(arg_b), _p(slot), _p(vid_ptr),
              vid_ptr.numel() - 1, a.numel(), _p(cand_scores), _p(payload), payload.shape[-1], _stream())
    return cand_scores


def scatter_fuse(a, b, wa, wb, csr, cand_scores):
    """cand_scores.flat[slot[e]] = fl(wa*a[e]) + fl(wb*b[e]) over the CSR entries (b may be None)."""
    vid_ptr, q_list, slot = csr
    _chk(a, torch.float32, "a")
    _lib.call("dkd_scatter_fuse", _p(a), _p(b), wa, wb, _p(slot), _p(vid_ptr), vid_ptr.numel() - 1, a.numel(),
              _p(cand_scores), _stream())
    return cand_scores


# ------------------------------------------------------------------------------------------------
# training-step similarity (BASELINE.json configs[4]); see train.py
def row_inv_norms(x, eps=1e-12):
    """1 / max(||row||, eps) for every D-vector of x -> (rows,) fp32."""
    _chk(x, torch.float32, "x")
    D = x.shape[-1]
    rows = x.numel() // D
    out = torch.empty((rows,), dtype=torch.float32, device=x.device)
    _lib.call("dkd_row_inv_norms", _p(x), rows, D, eps, _p(out), _stream())
    return out


TRAIN_SIM_TENSOR_CORES = True   # in-batch similarity forward on tcgen05 kind::tf32 x 3 when the shapes allow


def train_sim_fwd_tc(q, x, mask=None, labels=None, want_unnorm=True):
    """The forward of the in-batch similarity on the tensor cores (fp32 grade): cosine maxima = dkd_score_max_exact on
    the L2-normalised operands (F.normalize then contraction, like method/model.py:318-327), raw maxima = the same
    kernel on the raw operands (:331-350), the positive video's frame curve = dkd_train_curve.  Same outputs as
    train_sim_fwd.  D % 32 == 0, D <= 512, L <= 128."""
    M, D = q.shape
    N, L, _ = x.shape
    qn, _ = normalize_rows(q)
    xn, _ = normalize_rows(x)
    xn = xn.view(N, L, D)
    max_n, arg_n = score_max_exact(qn, pack_rows(xn), L, mask)
    max_u = arg_u = curve = None
    if want_unnorm:
        max_u, arg_u = score_max_exact(q, pack_rows(x), L, mask)
    if labels is not None:
        curve = torch.empty((M, L), dtype=torch.float32, device=q.device)
        _lib.call("dkd_train_curve", _p(qn), _p(xn), _p(mask), _p(labels), M, L, D, _p(curve), _stream())
    return max_n, arg_n, max_u, arg_u, curve


def train_sim_fwd(q, x, rq, rx, mask=None, labels=None, want_unnorm=True):
    """One pass of dots -> (max_n, arg_n, max_u | None, arg_u | None, curve | None); see include/dkd_b200.h."""
    _chk(q, torch.float32, "q")
    _chk(x, torch.float32, "x")
    M, D = q.shape
    N, L, _ = x.shape
    if mask is not None:
        _chk(mask, torch.uint8, "mask")
    if labels is not None:
        _chk(labels, torch.int32, "labels")
    if TRAIN_SIM_TENSOR_CORES and D % 32 == 0 and D <= 512 and L <= 128 and M > 0 and N > 0:
        return train_sim_fwd_tc(q, x, mask, labels, want_unnorm)
    dev = q.device
    max_n = torch.empty((M, N), dtype=torch.float32, device=dev)
    arg_n = torch.empty((M, N), dtype=torch.int32, device=dev)
    max_u = torch.empty((M, N), dtype=torch.float32, device=dev) if want_unnorm else None
    arg_u = torch.empty((M, N), dtype=torch.int32, device=dev) if want_unnorm else None
    curve = torch.empty((M, L), dtype=torch.float32, device=dev) if labels is not None else None
    _lib.call("dkd_train_sim_fwd", _p(q), _p(x), _p(rq), _p(rx), _p(mask), _p(labels), M, N, L, D, _p(max_n),
              _p(arg_n), _p(max_u), _p(arg_u), _p(curve), _stream())
    return max_n, arg_n, max_u, arg_u, curve


def train_sim_bwd(q, x, rq, rx, mask, labels, max_n, arg_n, arg_u, curve, g_n, g_u, g_c, want_q=True, want_x=True):
    M, D = q.shape
    N, L, _ = x.shape
    for name, g in (("g_max_n", g_n), ("g_max_u", g_u), ("g_curve", g_c)):
        if g is not None:
            _chk(g, torch.float32, name)
    gq = torch.empty_like(q) if want_q else None
    gx = torch.empty_like(x) if want_x else None
    _lib.call("dkd_train_sim_bwd", _p(q), _p(x), _p(rq), _p(rx), _p(mask), _p(labels), M, N, L, D, _p(max_n),
              _p(arg_n), _p(arg_u), _p(curve), _p(g_n), _p(g_u), _p(g_c), _p(gq), _p(gx), _stream())
    return gq, gx


def kl_curve_loss(pred, target, lens, temp):
    """Per-query KL(softmax(target/temp) || softmax(pred/temp)) over the first lens[m] frames -> (loss (M,), dpred (M, L))."""
    _chk(pred, torch.float32, "pred")
    _chk(target, torch.float32, "target")
    _chk(lens, torch.int32, "lens")
    M, L = pred.shape
    loss = torch.empty((M,), dtype=torch.float32, device=pred.device)
    dpred = torch.empty((M, L), dtype=torch.float32, device=pred.device)
    _lib.call("dkd_kl_curve_loss", _p(pred), _p(target), _p(lens), M, L, float(temp), _p(loss), _p(dpred), _stream())
    return loss, dpred


def train_losses(s_n, s_u, sims, labels, t2v_draw, v2t_pick, margin, soft, alpha, belta):
    """Fused triplet + NCE losses of one branch -> (terms (2,) [triplet, nce], g_n (M, N), g_u (M, N))."""
    _chk(s_n, torch.float32, "s_n")
    _chk(s_u, torch.float32, "s_u")
    if soft:
        _chk(sims, torch.float32, "sims")
    for name, t in (("labels", labels), ("t2v_draw", t2v_draw), ("v2t_pick", v2t_pick)):
        _chk(t, torch.int32, name)
    M, N = s_n.shape
    dev = s_n.device
    terms = torch.empty((2,), dtype=torch.float32, device=dev)
    g_n = torch.empty((M, N), dtype=torch.float32, device=dev)
    g_u = torch.empty((M, N), dtype=torch.float32, device=dev)
    ws = torch.empty((int(_lib.load().dkd_train_losses_workspace_floats(M, N)),), dtype=torch.float32, device=dev)
    _lib.call("dkd_train_losses", _p(s_n), _p(s_u), _p(sims) if soft else None, _p(labels), _p(t2v_draw), _p(v2t_pick),
              M, N, float(margin), int(bool(soft)), float(alpha), float(belta), _p(terms), _p(g_n), _p(g_u), _p(ws),
              _stream())
    return terms, g_n, g_u


# ------------------------------------------------------------------------------------------------
# corpus-side encoder (SURVEY section 8 f1); see encoder.py
def pack_weight(w):
    """nn.Linear weight (N, K) -> pre-packed tf32 hi / lo planes of dkd_linear_exact (once per model)."""
    _chk(w, torch.float32, "weight")
    N, K = w.shape
    nbytes = int(_lib.load().dkd_weight_planes_bytes(N, K))
    if nbytes < 0:
        raise _lib.DkdError("pack_weight: K must be a multiple of 32")
    planes = torch.empty((nbytes // 4,), dtype=torch.float32, device=w.device)
    _lib.call("dkd_pack_weight_tf32", _p(w), N, K, _p(planes), _stream())
    return planes


def linear_exact(x, w_planes, N, bias=None, relu=False, row_scale_shift=None, out=None):
    """out = act(xh @ W^T + bias) on tcgen05 kind::tf32 x 3 (fp32 grade); xh = x * scale_row + shift_row when
    row_scale_shift ((M, 2), row_stats) is given.  x: (M, K) fp32 contiguous; out: (M, N) (or a given (M, ld) buffer)."""
    _chk(x, torch.float32, "x")
    _chk(w_planes, torch.float32, "w_planes")
    M, K = x.shape
    if bias is not None:
        _chk(bias, torch.float32, "bias")
    if row_scale_shift is not None:
        _chk(row_scale_shift, torch.float32, "row_scale_shift")
    if out is None:
        out = torch.empty((M, N), dtype=torch.float32, device=x.device)
    _chk(out, torch.float32, "out")
    _lib.call("dkd_linear_exact", _p(x), M, K, _p(w_planes), N, _p(bias), int(bool(relu)), _p(row_scale_shift), _p(out),
              out.shape[1], _stream())
    return out


def row_stats(x, eps=1e-5):
    """LayerNorm statistics of every row -> (rows, 2) fp32 (rstd, -mean * rstd)."""
    _chk(x, torch.float32, "x")
    D = x.shape[-1]
    rows = x.numel() // D
    out = torch.empty((rows, 2), dtype=torch.float32, device=x.device)
    _lib.call("dkd_row_stats", _p(x), rows, D, float(eps), _p(out), _stream())
    return out


def layernorm_rows(x, gamma, beta, eps=1e-5, residual=None, pos=None, L=0):
    """LayerNorm(x [+ pos[row % L]] [+ residual]) * gamma + beta.  x / residual: (rows, D) views of wider 2-D matrices
    are accepted (column slices: stride(0) is passed as the leading dimension)."""
    rows, D = x.shape
    for name, t in (("x", x), ("residual", residual)):
        if t is not None and (not t.is_cuda or t.dtype != torch.float32 or t.stride(1) != 1):
            raise _lib.DkdError(f"layernorm_rows: {name} must be an fp32 CUDA matrix with unit column stride")
    _chk(gamma, torch.float32, "gamma")
    _chk(beta, torch.float32, "beta")
    if pos is not None:
        _chk(pos, torch.float32, "pos")
    out = torch.empty((rows, D), dtype=torch.float32, device=x.device)
    _lib.call("dkd_layernorm_rows", _p(x), x.stride(0), rows, D, _p(gamma), _p(beta), float(eps), _p(residual),
              residual.stride(0) if residual is not None else 0, _p(pos), int(L), _p(out), _stream())
    return out


def mha_small(qkv, Nv, L, heads, dh, mask=None, q_off=0, k_off=None, v_off=None):
    """Self-attention per (video, head) over L <= 128 rows from a fused (Nv * L, 3 * heads * dh) QKV matrix."""
    _chk(qkv, torch.float32, "qkv")
    H = heads * dh
    k_off = H if k_off is None else k_off
    v_off = 2 * H if v_off is None else v_off
    if mask is not None:
        _chk(mask, torch.uint8, "mask")
    out = torch.empty((Nv * L, H), dtype=torch.float32, device=qkv.device)
    _lib.call("dkd_mha_small", _p(qkv), qkv.shape[1], q_off, k_off, v_off, _p(mask), Nv, L, heads, dh,
              1.0 / float(dh) ** 0.5, _p(out), H, _stream())
    return out

"""ctypes binding of include/dkd_b200.h.  Fails loudly: there is no CPU or PyTorch fallback.

The library is the product; PyTorch only owns device memory and streams.
"""
import ctypes
import os
from ctypes import c_char_p, c_float, c_int32, c_int64, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libdkd_b200.so")

_P = c_void_p
_I = c_int32
_L = c_int64
_F = c_float

# name -> argument ctypes (return type is int unless listed in _RESTYPES)
PROTOTYPES = {
    "dkd_version": [],
    "dkd_error_string": [_I],
    "dkd_normalize_rows": [_P, _L, _I, _F, _P, _P, _P, _L, _P],
    "dkd_downsample_clips": [_P, _P, _I, _I, _I, _I, _P, _P],
    "dkd_build_proposals": [_P, _I, _I, _I, _P, _P, _P, _P],
    "dkd_score_max_f32": [_P, _I, _P, _I, _I, _I, _P, _P, _P, _L, _P, _P, _P, _P],
    "dkd_row_planes_bytes": [_I, _I, _I],
    "dkd_pack_rows_tf32": [_P, _I, _I, _I, _P, _P],
    "dkd_score_max_exact": [_P, _I, _P, _I, _I, _I, _P, _P, _P, _L, _P, _P, _P],
    "dkd_clip_planes_bytes": [_I, _I],
    "dkd_pack_clips_tf32": [_P, _I, _I, _I, _P, _P],
    "dkd_clip_score_f32": [_P, _I, _P, _P, _I, _I, _I, _P, _P, _L, _P, _P, _P, _P, _P, _L, _P],
    "dkd_clip_dots_list": [_P, _I, _P, _I, _I, _I, _P, _P, _P, _P],
    "dkd_moment_nms": [_P, _P, _P, _P, _F, _F, _P, _P, _I, _I, _I, _F, _P, _P, _P],
    "dkd_score_max_bf16": [_P, _I, _I, _P, _I, _I, _I, _P, _P, _P, _P, _L, _P, _F, _P],
    "dkd_score_max_f16": [_P, _I, _I, _P, _I, _I, _I, _P, _P, _P, _P, _L, _P, _F, _P],
    "dkd_score_max_bf16_lists": [_P, _I, _I, _P, _I, _I, _I, _P, _P, _P, _L, _F, _P, _P, _L, _I, _P],
    "dkd_clip_score_list": [_P, _I, _P, _P, _I, _I, _I, _P, _P, _L, _P, _P, _L, _P],
    "dkd_build_proposals_f16": [_P, _I, _I, _I, _P, _P, _P],
    "dkd_select_flagged": [_P, _I, _I, _L, _L, _P, _P, _P, _P, _P, _P],
    "dkd_select_pairs_csr": [_P, _I, _I, _L, _F, _L, _P, _P, _P, _P, _P],
    "dkd_key_clip_dots": [_P, _P, _I, _I, _I, _I, _P, _P],
    "dkd_frame_attn_table": [_P, _P, _P, _I, _I, _I, _I, _P, _P, _P],
    "dkd_frame_fuse": [_P, _P, _I, _P, _P, _I, _I, _I, _I, _L, _F, _F, _F, _I, _P, _P, _P],
    "dkd_fuse_scores": [_P, _P, _F, _F, _P, _L, _P],
    "dkd_topk": [_P, _I, _I, _L, _I, _I, _P, _P, _P],
    "dkd_select_topk": [_P, _I, _I, _L, _I, _I, _P, _P, _P],
    "dkd_topk_filtered": [_P, _I, _I, _L, _I, _I, _P, _I, _I, _P, _P, _P],
    "dkd_select_topk_filtered": [_P, _I, _I, _L, _I, _I, _P, _I, _I, _P, _P, _P],
    "dkd_build_video_filter": [_P, _P, _I, _I, _I, _I, _P, _P],
    "dkd_merge_topk": [_P, _P, _I, _I, _I, _P, _P, _P],
    "dkd_rank_of_gt": [_P, _I, _I, _L, _P, _P, _P, _P],
    "dkd_candidates_to_csr": [_P, _I, _I, _I, _I, _P, _P, _P, _P, _P],
    "dkd_frame_fuse_csr": [_P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _F, _F, _F, _I, _P, _L, _P],
    "dkd_scatter_fuse": [_P, _P, _F, _F, _P, _P, _I, _L, _P, _P],
    "dkd_sort_candidates": [_P, _P, _I, _I, _I, _P, _P, _P],
    "dkd_sort_candidates_payload": [_P, _P, _P, _I, _I, _I, _I, _P, _P, _P, _P],
    "dkd_merge_topk_payload": [_P, _P, _P, _I, _I, _I, _I, _P, _P, _P, _P],
    "dkd_sort_candidates_deep": [_P, _P, _P, _I, _I, _I, _I, _P, _P, _P, _P],
    "dkd_topk_deep": [_P, _I, _I, _L, _I, _I, _P, _I, _I, _P, _P, _P],
    "dkd_merge_topk_deep": [_P, _P, _P, _I, _I, _I, _I, _P, _P, _P, _P],
    "dkd_frame_fuse_csr_detail": [_P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _F, _F, _F, _I, _P, _L, _P, _I, _I, _P],
    "dkd_scatter_fuse_detail": [_P, _P, _F, _F, _P, _P, _P, _P, _I, _L, _P, _P, _I, _P],
    "dkd_weight_planes_bytes": [_I, _I],
    "dkd_pack_weight_tf32": [_P, _I, _I, _P, _P],
    "dkd_linear_exact": [_P, _L, _I, _P, _I, _P, _I, _P, _P, _L, _P],
    "dkd_row_stats": [_P, _L, _I, _F, _P, _P],
    "dkd_layernorm_rows": [_P, _L, _L, _I, _P, _P, _F, _P, _L, _P, _I, _P, _P],
    "dkd_mha_small": [_P, _L, _I, _I, _I, _P, _I, _I, _I, _I, _F, _P, _L, _P],
    "dkd_row_inv_norms": [_P, _L, _I, _F, _P, _P],
    "dkd_train_curve": [_P, _P, _P, _P, _I, _I, _I, _P, _P],
    "dkd_train_sim_fwd": [_P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _P, _P, _P, _P, _P, _P],
    "dkd_train_sim_bwd": [_P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P],
    "dkd_kl_curve_loss": [_P, _P, _P, _I, _I, _F, _P, _P, _P],
    "dkd_train_losses_workspace_floats": [_I, _I],
    "dkd_train_losses": [_P, _P, _P, _P, _P, _P, _I, _I, _F, _I, _F, _F, _P, _P, _P, _P, _P],
}
_RESTYPES = {"dkd_error_string": c_char_p, "dkd_clip_planes_bytes": c_int64, "dkd_row_planes_bytes": c_int64,
             "dkd_weight_planes_bytes": c_int64,
             "dkd_train_losses_workspace_floats": c_int64}

_lib = None


class DkdError(RuntimeError):
    pass


def load():
    """Load libdkd_b200.so (built by build.py). Raises if it is missing — no fallback path exists."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise DkdError(
            f"{LIB_PATH} not found: build it with `python dl-dkd_b200/build.py` "
            "(nvcc, sm_100a). dkd_b200 has no CPU / PyTorch fallback for the scoring path.")
    lib = ctypes.CDLL(LIB_PATH)
    for name, argtypes in PROTOTYPES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is missing
        fn.argtypes = argtypes
        fn.restype = _RESTYPES.get(name, c_int32)
    _lib = lib
    return lib


def check(code: int, what: str):
    if code != 0:
        msg = load().dkd_error_string(code)
        raise DkdError(f"{what} failed with code {code}: {msg.decode() if msg else '?'}")


# kernels launched per C-ABI call (for bench.py's gpu_launches claim)
KERNELS_PER_CALL = {"dkd_candidates_to_csr": 3, "dkd_select_pairs_csr": 3, "dkd_train_sim_bwd": 2, "dkd_train_losses": 3,
                    "dkd_train_losses_workspace_floats": 0, "dkd_topk_deep": 2, "dkd_merge_topk_deep": 2}  # (memsets are not counted)
_launches = 0
_timed_names = set()
_timed_events = {}


def reset_counters():
    global _launches
    _launches = 0


def launch_count() -> int:
    return _launches


def set_timed(names):
    """bench.py: bracket every call of the named entry points with CUDA events on the current stream."""
    global _timed_names, _timed_events
    _timed_names = set(names)
    _timed_events = {n: [] for n in _timed_names}


def timed_results():
    """name -> list of per-call durations in ms (synchronises)."""
    import torch
    torch.cuda.synchronize()
    return {n: [a.elapsed_time(b) for a, b in evs] for n, evs in _timed_events.items()}


def call(name: str, *args):
    global _launches
    lib = load()
    if name in _timed_names:
        import torch
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        check(getattr(lib, name)(*args), name)
        b.record()
        _timed_events[name].append((a, b))
    else:
        check(getattr(lib, name)(*args), name)
    _launches += KERNELS_PER_CALL.get(name, 1)

"""CPU: deep rankings.  rank() and rank_streamed() reject a K outside [1, 4096] or a Kc above 8192 before anything
reaches the device; the candidate-depth rule, the shape checks of the deep ops wrappers, and the deep entry points' own
argument checks (which come back before any device work)."""
import pytest
import torch


def _corpus(Nv=3):
    from dkd_b200 import engine
    return engine.PreparedCorpus(Nv=Nv, L=4, D=32, T=32, id_base=0, mask_u8=torch.ones((Nv, 4), dtype=torch.uint8),
                                 lengths=torch.full((Nv,), 4, dtype=torch.int32), heads=("frame", "two_scale"))


def _queries(M=2):
    from dkd_b200 import engine
    return engine.PreparedQueries(M=M, Mpad=256, qn=[torch.zeros((M, 32))], qb=[None], qh=[None])


@pytest.fixture
def no_launch(monkeypatch):
    from dkd_b200 import _lib

    def refuse(name, *args):
        raise AssertionError(f"{name} launched")

    monkeypatch.setattr(_lib, "call", refuse)


@pytest.mark.parametrize("kw", [dict(K=0), dict(K=4097), dict(K=-5), dict(K=100.0), dict(K=True),
                                dict(K=1000, Kc=8193), dict(K=100, Kc=10 ** 6)],
                         ids=["K0", "K4097", "K_negative", "K_float", "K_bool", "Kc8193", "Kc_huge"])
@pytest.mark.parametrize("M", [2, 0], ids=["queries", "no_queries"])
def test_rank_rejects_bad_depth_before_any_launch(dkd, no_launch, kw, M):
    from dkd_b200 import engine
    with pytest.raises(ValueError):
        engine.rank(_corpus(), _queries(M), precision="bf16", **kw)


@pytest.mark.parametrize("kw", [dict(K=0), dict(K=4097), dict(K=1000, Kc=8193)], ids=["K0", "K4097", "Kc8193"])
def test_rank_streamed_rejects_bad_depth_before_any_chunk(dkd, no_launch, kw):
    """The check comes before the first chunk's operands are built."""
    from dkd_b200 import engine

    def chunks():
        raise AssertionError("a chunk was requested")
        yield

    with pytest.raises(ValueError):
        engine.rank_streamed(chunks(), [_queries()], **kw)


@pytest.mark.parametrize("K,Kc,want", [(1, 128, 128), (100, 128, 128), (200, 128, 200), (256, 128, 256),
                                       (100, 600, 600), (257, 128, 352), (600, 128, 768), (1000, 128, 1280),
                                       (1000, 2000, 2000), (4096, 128, 5120), (4096, 8192, 8192)])
def test_candidate_depth_rule(dkd, K, Kc, want):
    from dkd_b200 import engine
    assert engine.candidate_depth(K, Kc) == want
    if K > 256:
        assert engine.candidate_depth(K, Kc) >= K + K // 4


def test_deep_entry_points_are_bound(dkd):
    from dkd_b200 import _lib
    P = _lib.PROTOTYPES
    assert len(P["dkd_sort_candidates_deep"]) == len(P["dkd_sort_candidates_payload"])
    assert len(P["dkd_merge_topk_deep"]) == len(P["dkd_merge_topk_payload"])
    assert P["dkd_topk_deep"] == P["dkd_topk_filtered"]
    assert _lib.KERNELS_PER_CALL["dkd_topk_deep"] == 2 and _lib.KERNELS_PER_CALL["dkd_merge_topk_deep"] == 2


def _f(*shape):
    return torch.zeros(shape, dtype=torch.float32)


def _i(*shape):
    return torch.zeros(shape, dtype=torch.int32)


@pytest.mark.parametrize("case", ["Kc0", "Kc8193", "Kout0", "Kout_above_Kc", "Kout4097", "shapes", "C9", "C0",
                                  "payload_rows", "no_pad", "pad_size"])
def test_sort_candidates_deep_checks_shapes(dkd, no_launch, case):
    from dkd_b200 import _lib, ops
    Kc, K_out, payload, pad = 300, 100, None, None
    s, i = _f(2, Kc), _i(2, Kc)
    if case == "Kc0":
        s, i = _f(2, 0), _i(2, 0)
    elif case == "Kc8193":
        s, i = _f(2, 8193), _i(2, 8193)
    elif case == "Kout0":
        K_out = 0
    elif case == "Kout_above_Kc":
        K_out = Kc + 1
    elif case == "Kout4097":
        s, i, K_out = _f(2, 5000), _i(2, 5000), 4097
    elif case == "shapes":
        i = _i(3, Kc)
    elif case == "C9":
        payload, pad = _i(2, Kc, 9), _i(9)
    elif case == "C0":
        payload, pad = _i(2, Kc, 0), _i(0)
    elif case == "payload_rows":
        payload, pad = _i(2, Kc + 1, 4), _i(4)
    elif case == "no_pad":
        payload = _i(2, Kc, 4)
    elif case == "pad_size":
        payload, pad = _i(2, Kc, 4), _i(3)
    with pytest.raises(_lib.DkdError, match="sort_candidates_deep"):
        ops.sort_candidates_deep(s, i, K_out, payload=payload, pad=pad)


@pytest.mark.parametrize("case", ["K0", "K4097", "not_2d"])
def test_topk_deep_checks_shapes(dkd, no_launch, case):
    from dkd_b200 import _lib, ops
    s, K = _f(4, 5000), 100
    if case == "K0":
        K = 0
    elif case == "K4097":
        K = 4097
    else:
        s = _f(4, 50, 2)
    with pytest.raises(_lib.DkdError, match="topk_deep"):
        ops.topk_deep(s, K)


@pytest.mark.parametrize("case", ["K4097", "G0", "shapes", "not_3d", "C9", "no_pad", "payload_lists"])
def test_merge_topk_deep_checks_shapes(dkd, no_launch, case):
    from dkd_b200 import _lib, ops
    s, i, payload, pad = _f(2, 3, 300), _i(2, 3, 300), None, None
    if case == "K4097":
        s, i = _f(2, 3, 4097), _i(2, 3, 4097)
    elif case == "G0":
        s, i = _f(0, 3, 300), _i(0, 3, 300)
    elif case == "shapes":
        i = _i(2, 3, 301)
    elif case == "not_3d":
        s, i = _f(3, 300), _i(3, 300)
    elif case == "C9":
        payload, pad = _i(2, 3, 300, 9), _i(9)
    elif case == "no_pad":
        payload = _i(2, 3, 300, 6)
    elif case == "payload_lists":
        payload, pad = _i(1, 3, 300, 6), _i(6)
    with pytest.raises(_lib.DkdError, match="merge_topk_deep"):
        ops.merge_topk_deep(s, i, payload=payload, pad=pad)


def test_well_formed_cpu_tensors_still_need_the_device(dkd, no_launch):
    """The shape checks pass, then the wrappers refuse host tensors instead of falling back to PyTorch."""
    from dkd_b200 import _lib, ops
    with pytest.raises(_lib.DkdError, match="CUDA"):
        ops.topk_deep(_f(4, 5000), 1000)
    with pytest.raises(_lib.DkdError, match="CUDA"):
        ops.sort_candidates_deep(_f(2, 1280), _i(2, 1280), 1000)
    with pytest.raises(_lib.DkdError, match="CUDA"):
        ops.merge_topk_deep(_f(2, 3, 1000), _i(2, 3, 1000))


def test_deep_entry_points_check_arguments_first(dkd):
    """Shape and argument errors come back before any device work (dummy non-null pointers are never dereferenced)."""
    from dkd_b200 import _lib
    lib = _lib.load()
    p = 256
    topk = lib.dkd_topk_deep
    assert topk(p, 4, 5000, 5000, 0, 0, None, 0, 0, p, p, None) == -2                      # K < 1
    assert topk(p, 4, 5000, 5000, 4097, 0, None, 0, 0, p, p, None) == -2                   # K > 4096
    assert topk(p, 4, 5000, 4999, 100, 0, None, 0, 0, p, p, None) == -1                    # ld < Nv
    assert topk(p, 4, 5000, 5000, 100, 0, p, 3, 157, p, p, None) == -2                     # filter rows neither 1 nor M
    assert topk(p, 4, 5000, 5000, 100, 37, p, 1, 157, p, p, None) == -2                    # words miss ids >= 5024
    assert topk(p, 4, 5000, 5000, 100, -1, p, 1, 157, p, p, None) == -1                    # negative id_base
    assert topk(p, 0, 5000, 5000, 4096, 37, p, 1, 158, p, p, None) == 0                    # no rows: nothing to do
    sort = lib.dkd_sort_candidates_deep
    assert sort(p, p, None, 4, 8193, 100, 0, p, p, None, None) == -2                       # Kc > 8192
    assert sort(p, p, None, 4, 1000, 1001, 0, p, p, None, None) == -2                      # K_out > Kc
    assert sort(p, p, None, 4, 8192, 4097, 0, p, p, None, None) == -2                      # K_out > 4096
    assert sort(p, p, None, 4, 1000, 0, 0, p, p, None, None) == -2                         # K_out < 1
    assert sort(p, p, p, 4, 1000, 100, 9, p, p, p, None) == -2                             # C > 8
    assert sort(p, p, p, 4, 1000, 100, 0, p, p, p, None) == -2                             # C < 1 with a payload
    assert sort(p, p, p, 4, 1000, 100, 6, p, p, None, None) == -1                          # payload without output
    assert sort(p, None, None, 4, 1000, 100, 0, p, p, None, None) == -1
    assert sort(p, p, None, 0, 8192, 4096, 0, p, p, None, None) == 0                       # no rows
    merge = lib.dkd_merge_topk_deep
    assert merge(p, p, None, 0, 4, 1000, 0, p, p, None, None) == -1                        # G < 1
    assert merge(p, p, None, 2, 4, 4097, 0, p, p, None, None) == -2                        # K > 4096
    assert merge(p, p, None, 2, 4, 0, 0, p, p, None, None) == -2                           # K < 1
    assert merge(p, p, p, 2, 4, 1000, 9, p, p, p, None) == -2                              # C > 8
    assert merge(p, p, p, 2, 4, 1000, 6, p, p, None, None) == -1                           # payload without output
    assert merge(p, p, None, 8, 0, 4096, 0, p, p, None, None) == 0                         # no rows

"""CPU: engine.localize rejects malformed input before anything reaches the device and returns padding without a launch
for empty inputs; the moment entry points are bound with the expected arity and check their arguments before any
device work."""
import pytest
import torch


def _corpus(heads=("two_scale",), Nv=3):
    from dkd_b200 import engine
    return engine.PreparedCorpus(Nv=Nv, L=4, D=32, T=32, id_base=0, mask_u8=torch.ones((Nv, 4), dtype=torch.uint8),
                                 lengths=torch.full((Nv,), 4, dtype=torch.int32), heads=heads)


def _queries(M=2):
    from dkd_b200 import engine
    return engine.PreparedQueries(M=M, Mpad=256, qn=[torch.zeros((M, 32))], qb=[None], qh=[None])


@pytest.fixture
def no_launch(monkeypatch):
    from dkd_b200 import _lib

    def refuse(name, *args):
        raise AssertionError(f"{name} launched")

    monkeypatch.setattr(_lib, "call", refuse)


@pytest.mark.parametrize("kw", [dict(m=0), dict(m=17), dict(m=2.0), dict(m=True), dict(iou=-0.1),
                                dict(iou=float("nan")), dict(heads=("frame",)), dict(ids="int64"), dict(ids="rows"),
                                dict(ids="1d"), dict(ids="list")],
                         ids=["m0", "m17", "m_float", "m_bool", "iou_negative", "iou_nan", "frame_head", "ids_int64",
                              "ids_rows", "ids_1d", "ids_list"])
def test_localize_rejects_bad_input_on_the_host(dkd, no_launch, kw):
    from dkd_b200 import engine
    ids = torch.zeros((2, 5), dtype=torch.int32)
    bad = kw.pop("ids", None)
    if bad == "int64":
        ids = ids.long()
    elif bad == "rows":
        ids = torch.zeros((3, 5), dtype=torch.int32)
    elif bad == "1d":
        ids = torch.zeros((10,), dtype=torch.int32)
    elif bad == "list":
        ids = [[0, 1], [2, 0]]
    pc = _corpus(heads=kw.pop("heads", ("two_scale",)))
    with pytest.raises(ValueError):
        engine.localize(pc, _queries(), ids, **kw)


@pytest.mark.parametrize("M,K,Nv", [(0, 5, 3), (2, 0, 3), (2, 5, 0)])
def test_localize_empty_inputs_give_padding_without_a_launch(dkd, no_launch, M, K, Nv):
    from dkd_b200 import engine
    mo = engine.localize(_corpus(Nv=Nv), _queries(M), torch.zeros((M, K), dtype=torch.int32), m=3)
    assert mo.arg.shape == (M, K, 3) and mo.arg.dtype == torch.int32 and (mo.arg == -1).all()
    assert mo.score.shape == (M, K, 3) and mo.score.dtype == torch.float32 and torch.isneginf(mo.score).all()


def test_moment_entry_points_are_bound(dkd):
    from dkd_b200 import _lib
    P = _lib.PROTOTYPES
    assert len(P["dkd_clip_dots_list"]) == 10
    assert len(P["dkd_moment_nms"]) == 15


def test_moment_entry_points_check_arguments_first(dkd):
    """Shape and argument errors come back before any device work (dummy non-null pointers are never dereferenced)."""
    from dkd_b200 import _lib
    lib = _lib.load()
    p = 256
    nms = lib.dkd_moment_nms
    assert nms(p, p, None, None, 0.7, 0.3, p, p, 3, 33, 5, 0.5, p, p, None) == -2        # T > 32
    assert nms(p, p, None, None, 0.7, 0.3, p, p, 3, 32, 0, 0.5, p, p, None) == -2        # m < 1
    assert nms(p, p, None, None, 0.7, 0.3, p, p, 3, 32, 17, 0.5, p, p, None) == -2       # m > 16
    assert nms(p, p, None, None, 0.7, 0.3, p, p, 3, 32, 5, -0.5, p, p, None) == -1       # iou < 0
    assert nms(p, p, None, None, 0.7, 0.3, p, p, 3, 32, 5, float("nan"), p, p, None) == -1
    assert nms(p, p, p, None, 0.7, 0.3, p, p, 3, 32, 5, 0.5, p, p, None) == -1            # dots1 without scale1
    assert nms(p, p, None, None, 0.7, 0.3, p, p, 0, 32, 5, 0.5, p, p, None) == 0          # no videos: nothing to do
    dots = lib.dkd_clip_dots_list
    assert dots(p, 4, p, 3, 33, 64, p, p, p, None) == -2                                    # T > 32
    assert dots(p, 4, p, 3, 32, 48, p, p, p, None) == -2                                    # D % 32
    assert dots(p, 4, p, 3, 32, 64, p, p, 260, None) == -3                                  # misaligned out_dots
    assert dots(p, 4, p, 3, 32, 64, None, p, p, None) == -1                                 # no CSR

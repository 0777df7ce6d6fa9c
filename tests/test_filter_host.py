"""CPU: engine.make_video_filter rejects malformed input before anything reaches the device, and the filtered entry
points are declared with the prototypes the wrappers call them with."""
import pytest


@pytest.mark.parametrize("kw", [dict(allow=[[0, 1], [5, 300]]), dict(allow=[3, 300]), dict(deny=[-1]),
                                dict(deny=[[2], [-3]]), dict(), dict(allow=[1], deny=[2])],
                         ids=["allow_per_query_high", "allow_shared_high", "deny_shared_negative",
                              "deny_per_query_negative", "neither", "both"])
def test_make_video_filter_rejects_bad_input_on_the_host(dkd, kw):
    from dkd_b200 import engine
    with pytest.raises(ValueError):
        engine.make_video_filter(300, **kw)


def test_filtered_entry_points_are_bound(dkd):
    from dkd_b200 import _lib
    P = _lib.PROTOTYPES
    assert len(P["dkd_topk_filtered"]) == len(P["dkd_topk"]) + 3
    assert len(P["dkd_select_topk_filtered"]) == len(P["dkd_select_topk"]) + 3
    assert len(P["dkd_build_video_filter"]) == 8

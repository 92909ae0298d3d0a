"""Host-side grouping of generate_batch / generate_sharded: clips of one output length form one batch whatever their
input rate, with the clips of each (rate, input length) part consecutive."""
import pytest

from flowhigh_b200 import tables
from flowhigh_b200.flowhighsr import FlowHighSR, group_by_output_length


def test_mixed_rates_of_one_output_length_form_one_group():
    srs = [8000, 12000, 16000, 24000, 8000, 12000, 48000, 16000]
    lens = [s // 2 for s in srs]  # 0.5 s each -> 24000 samples at 48 kHz
    groups = group_by_output_length(lens, srs, 48000, "scipy")
    # parts in order of first appearance, caller order inside a part; the 48 kHz clip is its own part
    assert groups == {(24000, "scipy"): [0, 4, 1, 5, 2, 7, 3, 6]}
    idxs = groups[(24000, "scipy")]
    assert FlowHighSR._parts(idxs, srs, lens) == [(8000, 4000, 2), (12000, 6000, 2), (16000, 8000, 2), (24000, 12000, 1),
                                                 (48000, 24000, 1)]
    # a sub-batch split keeps runs of one part together
    assert FlowHighSR._parts(idxs[:3], srs, lens) == [(8000, 4000, 2), (12000, 6000, 1)]


def test_different_output_lengths_stay_apart_and_lengths_are_exact():
    srs = [8000, 16000, 22050, 16000, 48000, 8000]
    lens = [4000, 8000, 11025, 8001, 24000, 3999]
    groups = group_by_output_length(lens, srs, 48000, "soxr_hq")
    assert groups == {(24000, "soxr_hq"): [0, 1, 2, 4], (24003, "soxr_hq"): [3], (23994, "soxr_hq"): [5]}


@pytest.mark.parametrize("sr", [8000, 12000, 16000, 22050, 24000, 44100, 48000])
@pytest.mark.parametrize("n", [393, 4000, 11025, 80001])
def test_output_length_is_what_the_resampler_produces(sr, n):
    """The grouping key is the length resample_normalise returns for either filter design (same up / down ratio)."""
    for method, plan in (("scipy", tables.resample_plan(sr, 48000)), ("soxr_hq", tables.resample_plan_soxr_hq(sr, 48000))):
        want = n if plan is None else tables.resample_out_len(n, plan[1], plan[2])
        assert group_by_output_length([n], [sr], 48000, method) == {(want, method): [0]}

"""CPU tests of the owner-form plan of the adjoint STFT (vr_plan_adjoint_stft): the segments of a sequence cover every sample
exactly once, and each segment's frame range holds every frame whose window reaches one of its samples, directly or
through the reflect padding."""
import numpy as np
import pytest


@pytest.fixture(scope="module")
def cabi():
    import __graft_entry__ as ge
    ge.build_product()
    from skeleton_action_recognition_b200 import _cabi
    return _cabi


def _reflect(t, T):
    t = np.abs(t)
    return np.where(t >= T, 2 * (T - 1) - t, t)


@pytest.mark.parametrize("T", [129, 300, 2100, 75000])
@pytest.mark.parametrize("hop", [8, 16, 100, 300])
@pytest.mark.parametrize("N", [1, 4, 4096])
def test_segments_cover_every_sample_and_every_touching_frame(cabi, N, T, hop):
    plan, segs = cabi.plan_adjoint_stft(N, T, hop)
    assert plan["segments"] == len(segs) >= 1
    assert plan["segment_length"] <= 4096 and plan["smem_bytes"] == 8 * plan["segment_length"]     # ADJ_SEG_MAX
    assert plan["grid"] == min(N * len(segs), 8 * 148)
    owner = np.full(T, -1)
    for k, (s0, s1, _, _) in enumerate(segs):
        assert 0 <= s0 < s1 <= T
        assert (owner[s0:s1] == -1).all()
        owner[s0:s1] = k
    assert (owner >= 0).all()
    if T <= 300:
        assert len(segs) == 1                                      # short sequences: one segment, no halo
    F = T // hop + 1
    f = np.repeat(np.arange(F), 256)
    t = _reflect(f * hop - 128 + np.tile(np.arange(256), F), T)
    pairs = np.unique(np.stack([owner[t], f], 1), axis=0)      # (segment, frame) for every frame that reaches the segment
    for k, (s0, s1, lo, hi) in enumerate(segs):
        fr = pairs[pairs[:, 0] == k, 1]
        assert fr.size == 0 or (lo <= fr.min() and fr.max() <= hi), (k, lo, hi, fr.min(), fr.max())
        assert 0 <= lo and hi <= F - 1
        if fr.size:                                            # and no more than the frames between them
            assert lo == fr.min() and hi == fr.max()


def test_long_sequences_are_cut_and_short_batches_get_more_segments(cabi):
    p1, _ = cabi.plan_adjoint_stft(1, 75000, 16)
    p256, _ = cabi.plan_adjoint_stft(256, 75000, 16)
    assert p1["segments"] > p256["segments"] >= 19
    assert cabi.plan_adjoint_stft(4096, 300, 16)[0]["segments"] == 1


def test_plan_rejects_bad_shapes(cabi):
    with pytest.raises(ValueError):
        cabi.plan_adjoint_stft(1, 128, 16)
    with pytest.raises(ValueError):
        cabi.plan_adjoint_stft(0, 300, 16)
    with pytest.raises(ValueError):
        cabi.plan_adjoint_stft(1, 300, 0)

"""Pin of the oracle against what the unmodified reference computes: oracle/agar_oracle.c replays the recordings of
tests/golden/live/ (tools/gen_golden_live.py, on the inputs of tools/compare_oracle_ref.py) and must reproduce records, events
and observations BIT FOR BIT every frame.  Where the reference's sources are at hand, tools/compare_oracle_ref.py and
tools/fuzz_oracle_ref.py step the two side by side, and tools/gen_golden_live.py --source reference re-records these files."""
import numpy as np
import pytest

import aigar_b200.layout as lay
import gen_golden_live as gl
from golden_util import live, replay_live_rollout


@pytest.mark.parametrize("which,frames,seed", gl.ORACLE_CASES)
def test_oracle_equals_reference(which, frames, seed):
    assert live("oracle_%s_%d" % (which, seed))["actions"].shape[0] == frames
    replay_live_rollout("oracle_%s_%d" % (which, seed))


def test_reset_matches_reference():
    z, got = live("reset"), gl.record_reset("oracle")
    cfg = lay.derive_config(num_nn=1, num_greedy=1, virus=True, split=True, eject=True, event_cap=256)
    L = lay.layout_for_config(cfg)
    d = lay.compare_records(lay.Record(L, z["after_reset"].copy()), lay.Record(L, got["after_reset"]), what="after reset ",
                            check_events=False)
    assert not d, d
    d = lay.compare_records(lay.Record(L, z["after_reset_60"].copy()), lay.Record(L, got["after_reset_60"]),
                            what="after reset+60 ")
    assert not d, d


@pytest.mark.parametrize("kw", gl.VARIATIONS, ids=[str(i) for i in range(len(gl.VARIATIONS))])
def test_config_variations_equal_reference(kw):
    """Flags of networkParameters.py the default configs do not exercise: reward variants, frame-skip, grid sizes,
    channel subsets, bot mixes."""
    i = gl.VARIATIONS.index(kw)
    z = live("variation_%d" % i)
    assert str(z["kw"]) == repr(kw) and z["actions"].shape[0] == gl.variation_frames(kw)
    replay_live_rollout("variation_%d" % i)


def test_views_show_what_the_reference_objects_show():
    """a.i.gar_b200/views.py (SURVEY §8f rank 4): the getters the reference's View reads, over the oracle's env record after 150
    frames of the 1-vs-greedy config, against what the reference objects returned."""
    z, got = live("views"), gl.record_views("oracle")
    assert sorted(z.files) == sorted(list(got) + ["source"])
    for k, v in got.items():
        assert np.array_equal(z[k], v), k


def test_random_configs_equal_reference():
    """tools/fuzz_oracle_ref.py's random flag / bot-mix / grid / frame-skip combinations (6 cases, seed 23) replayed."""
    from fuzz_oracle_ref import cases
    cs = cases(gl.FUZZ_N, gl.FUZZ_SEED)
    assert len(cs) >= 4
    for case, kw, frames, seed in cs:
        z = live("fuzz_%d" % case)
        assert str(z["kw"]) == repr(kw) and int(z["seed"]) == seed and z["actions"].shape[0] == frames
        replay_live_rollout("fuzz_%d" % case)

"""a.i.gar_b200/results.py writes what the reference's own export functions write (src/aigar.py:459-465, 499-519, 609-627)."""
import os

import numpy as np

from aigar_b200 import results as res


def _evals(seed):
    rng = np.random.default_rng(seed)
    return res.episode_evals(rng.uniform(50, 600, 10), rng.uniform(100, 1200, 10), "test", "Test")


def test_episode_evals_is_the_references_reduction():
    means, maxes = [120.5, 130.25, 99.0], [300.0, 410.5, 250.0]
    e = res.episode_evals(means, maxes, "vsGreedy", "Vs_Greedy")
    assert e["meanScore"] == np.mean(means) and e["stdMean"] == np.std(means)
    assert e["meanMaxScore"] == np.mean(maxes) and e["stdMax"] == np.std(maxes) and e["maxScore"] == 410.5


def test_file_formats(tmp_path):
    p = str(tmp_path) + os.sep
    tr = [{"current": _evals(1), "vsGreedy": _evals(2), "virus": _evals(3), "virusGreedy": _evals(4)} for _ in range(3)]
    res.export_test_results(tr, p, {"MULTIPLE_BOTS_PRESENT": True, "VIRUS_SPAWN": True})
    for stem in ("testMassOverTime", "VS_1_GreedyMassOverTime", "Pellet_Collection_Virus_MassOverTime", "VS_1_Greedy_Virus_MassOverTime"):
        lines = open(os.path.join(p, "data", stem + ".txt")).read().splitlines()
        assert len(lines) == 3 and all(float(x) > 0 for x in lines)
    assert open(os.path.join(p, "data", "testMassOverTime.txt")).read() == "".join(str(v["current"]["meanScore"]) + "\n" for v in tr)
    txt = res.write_final_results({"current": _evals(1)}, p, 10)
    e = _evals(1)
    assert txt == ("Number of runs per testing: 10\n" + "test Highscore: %s Mean: %s StdMean: %s Mean_Max_Score: %s Std_Max_Score: %s\n" % (
        round(e["maxScore"], 1), round(e["meanScore"], 1), round(e["stdMean"], 1), round(e["meanMaxScore"], 1), round(e["stdMax"], 1)))
    assert open(os.path.join(p, "final_results.txt")).read() == txt


def test_against_the_reference_functions(tmp_path):
    """The file the reference's own exportResults writes for four fixed values (recorded in tests/golden/live/export_results.npz
    by tools/gen_golden_live.py; the function is pure Python, extracted from aigar.py, which imports Keras at module level)."""
    from golden_util import live
    z = live("export_results")
    b = str(tmp_path) + os.sep + "b_"
    res.export_results([float(v) for v in z["values"]], b, "m")
    assert open(b + "m.txt").read() == str(z["text"])

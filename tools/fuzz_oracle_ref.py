"""Random configurations, C oracle (libm build) vs the UNMODIFIED reference executed through oracle/ref_harness.py, every
field / event / observation every frame (build container only): python tools/fuzz_oracle_ref.py [N] [SEED]"""
import os, sys, random, traceback
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import compare_oracle_ref as cmp  # noqa: E402

FLAGS = ["pellet_grid", "self_grid", "wall_grid", "enemy_grid", "virus_grid", "self_grid_lf", "self_grid_slf", "enemy_grid_lf",
         "enemy_grid_slf", "use_fovsize", "use_last_fovsize", "use_totalmass", "use_last_action", "use_second_last_action"]


def cases(n, seed):
    """The random cases of a run: [(case number, kw, frames, seed)], without those the layout rejects or the reference cannot run
    (frame-skip 0 with a random bot divides by zero, bot.py:244)."""
    import aigar_b200.layout as lay
    rnd = random.Random(seed)
    out = []
    for case in range(n):
        n_nn = rnd.choice([1, 1, 1, 2, 3])
        n_gr = rnd.choice([0, 0, 1, 1, 2, 4])
        n_rd = rnd.choice([0, 0, 0, 1])
        split = rnd.random() < 0.5
        eject = split and rnd.random() < 0.6
        kw = dict(num_nn=n_nn, num_greedy=n_gr, num_random=n_rd, virus=rnd.random() < 0.5, split=split, eject=eject,
                  grid=rnd.choice([3, 5, 8, 11, 11, 14, 16, 19, 25]), frame_skip=rnd.choice([0, 1, 3, 7, 7, 9]),
                  obs_mode=rnd.choice([0, 0, 1]), mass_as_reward=rnd.random() < 0.2,
                  overrides={f: int(rnd.random() < 0.5) for f in rnd.sample(FLAGS, rnd.randint(0, 6))})
        if rnd.random() < 0.15:  # ALL_PLAYER_GRID replaces the self / enemy channels (networkParameters.py:88-91)
            kw["overrides"].update({"all_player_grid": 1, "self_grid": 0, "enemy_grid": 0, "self_grid_lf": 0, "self_grid_slf": 0,
                                    "enemy_grid_lf": 0, "enemy_grid_slf": 0})
        try:
            lay.layout_for_config(lay.derive_config(**kw))
        except ValueError as ex:
            print("case %d rejected by layout (%s)" % (case, ex))
            continue
        if kw["frame_skip"] == 0 and n_rd:
            print("case %d skipped: the reference divides by zero (bot.py:244)" % case)
            continue
        out.append((case, kw, 60 if n_nn + n_gr + n_rd > 3 else 100, rnd.randint(0, 999)))
    return out


if __name__ == "__main__":
    N = int(sys.argv[1]) if len(sys.argv) > 1 else 24
    bad = 0
    for case, kw, frames, seed in cases(N, int(sys.argv[2]) if len(sys.argv) > 2 else 1):
        try:
            ok = cmp.run(kw, frames, seed=seed, verbose=False)
        except Exception:
            ok = False
            traceback.print_exc()
        print("case %d %s: %r" % (case, "OK" if ok else "FAILED", kw), flush=True)
        bad += 0 if ok else 1
    print("%d cases, %d failed" % (N, bad))
    sys.exit(1 if bad else 0)

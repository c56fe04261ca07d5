"""Gumbel search on one GPU: time per simulation of GumbelMCTS / InformationSetGumbelMCTS against their PUCT siblings
(BatchedMCTS / InformationSetMCTS) on the same roots, alternated in one run, and the playing strength of each pair with the
rollout evaluator in StormboundVecEnv, the Gumbel agents playing their returned action, the PUCT agents the arg-max of visits.

Before anything is timed, one search of each kind on 32 trees is checked against the plain-Python model
(tests/sb_gumbel_model.py): action, policy, visits, q and root values must be identical.  Writes the report to --out
(default profiles/r7_bench_gumbel.txt).
"""
import argparse
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests"), os.path.join(ROOT, "tools")]

from bench_ismcts import keys_of  # noqa: E402
from bench_search import LINES, constant_evaluator, gpu_identity, roots_of, say  # noqa: E402
from monsoon_b200.engine import N_ACTIONS, get_engine  # noqa: E402
from monsoon_b200.search import (BatchedMCTS, GumbelMCTS, InformationSetGumbelMCTS, InformationSetMCTS, gumbel_noise,  # noqa: E402
                                 rollout_evaluator, select_actions)
from monsoon_b200.vec_env import StormboundVecEnv  # noqa: E402


def check_against_model(engine, n=32, sims=24, mc=8):
    import sb_determinize_model as D
    import sb_gumbel_model as G
    dev = engine.device
    roots = roots_of(engine, n, 99)
    host = roots.cpu().numpy()
    keys = keys_of(n * (sims + 1), 5, dev)
    hk = keys.cpu().numpy().view(np.uint64)
    hg = gumbel_noise(n, 3)
    gum = torch.from_numpy(hg).to(dev)
    prior = np.full(N_ACTIONS, 1.0 / N_ACTIONS, dtype=np.float32)
    ev = constant_evaluator(n, dev)
    for ism in (False, True):
        models = [G.ISGumbelTreeModel(sims + 1) if ism else G.GumbelTreeModel(host[g], sims + 1) for g in range(n)]

        def evaluate(leaf, k):
            if ism:
                world = [D.determinize(host[g], int(hk[k * n + g])) for g in range(n)]
                want = [t.begin(world[g]) if k == 0 else t.simulate(world[g], prior, np.float32(0), hg[g], k, sims, mc)
                        for g, t in enumerate(models)]
            else:
                want = [t.begin() if k == 0 else t.simulate(prior, np.float32(0), hg[g], k, sims, mc) for g, t in enumerate(models)]
            states = leaf["states"].cpu().numpy()
            assert all(states[g].tobytes() == want[g][0].tobytes() for g in range(n)), k
            return ev(leaf, k)

        mcts = InformationSetGumbelMCTS(n, sims, mc, engine=engine) if ism else GumbelMCTS(n, sims, mc, engine=engine)
        out = mcts.run(roots, evaluate, keys, gum) if ism else mcts.run(roots, evaluate, gum)
        action, policy, visits, q, rv = (t.cpu().numpy() for t in out)
        for g, t in enumerate(models):
            wa, wp, wv, wq, wr = t.end(prior, np.float32(0), hg[g])
            assert action[g] == wa and policy[g].tobytes() == wp.tobytes() and np.array_equal(visits[g], wv), g
            assert np.array_equal(q[g], wq, equal_nan=True) and np.array_equal(rv[g], wr, equal_nan=True), g
        say("model check (%s): %d trees x %d simulations, max_considered %d: every leaf record, action, policy, visits, q and root "
            "value identical to tests/sb_gumbel_model.py" % ("information-set" if ism else "perfect-information", n, sims, mc))


def time_pair(runs, reps):
    """alternate the runs rep by rep; median and min ms of each, CUDA events around each whole search"""
    ms = [[] for _ in runs]
    for _ in range(reps):
        for i, run in enumerate(runs):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            run()
            b.record()
            torch.cuda.synchronize()
            ms[i].append(a.elapsed_time(b))
    return [(float(np.median(m)), min(m)) for m in ms]


def bench_speed(engine, n, sims, reps):
    dev = engine.device
    roots = roots_of(engine, n, 7)
    ev = constant_evaluator(n, dev)
    gum = torch.from_numpy(gumbel_noise(n, 1)).to(dev)
    keys = keys_of(n * (sims + 1), 11, dev)
    for ism in (False, True):
        if ism:
            gm, pm = InformationSetGumbelMCTS(n, sims, engine=engine), InformationSetMCTS(n, sims, engine=engine)
            runs = [lambda: gm.run(roots, ev, keys, gum), lambda: pm.run(roots, ev, keys)]
        else:
            gm, pm = GumbelMCTS(n, sims, engine=engine), BatchedMCTS(n, sims, engine=engine)
            runs = [lambda: gm.run(roots, ev, gum), lambda: pm.run(roots, ev)]
        for r in runs:
            r()  # warm-up
        torch.cuda.synchronize()
        (g_med, g_min), (p_med, p_min) = time_pair(runs, reps)
        say("n=%d sims=%d %-13s Gumbel search %.2f ms (min %.2f) = %.3f ms per simulation; PUCT search %.2f ms (min %.2f) = %.3f ms "
            "per simulation; ratio %.2f" % (n, sims, "information-set" if ism else "perfect-info", g_med, g_min, g_med / sims, p_med,
                                            p_min, p_med / sims, g_med / p_med))
        del gm, pm, runs
        torch.cuda.empty_cache()


def strength(engine, label, mcts, opponent, gumbel, max_moves=600):
    """the first episode of every env of a StormboundVecEnv against `opponent`"""
    n = mcts.n
    env = StormboundVecEnv(n, seed=1234, opponent=opponent, seats=[g % 2 for g in range(n)], engine=engine)
    env.reset()
    ev = rollout_evaluator(engine)
    first = torch.full((n,), -3, dtype=torch.int8, device=engine.device)
    t0 = time.time()
    for _ in range(max_moves):
        out = mcts.run(env.states, ev)
        _o, _m, _r, done, info = env.step(out[0] if gumbel else select_actions(out[0]))
        first = torch.where((first == -3) & done, info["result"], first)
        if not bool((first == -3).any()):
            break
    r = first.cpu().numpy()
    seat = np.arange(n) % 2
    won = int(((r == 0) & (seat == 0)).sum() + ((r == 1) & (seat == 1)).sum())
    lost = int(((r == 1) & (seat == 0)).sum() + ((r == 0) & (seat == 1)).sum())
    drawn = int(((r == -1) | (r == -2)).sum())
    say("strength: %-32s vs %-6s over %d episodes (mixed seats): win %d / draw %d / loss %d (unfinished %d; %.0f s)" % (
        label, opponent, n, won, drawn, lost, int((r == -3).sum()), time.time() - t0))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r7_bench_gumbel.txt"))
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--episodes", type=int, default=1024)
    ap.add_argument("--sizes", default="4096,65536")
    ap.add_argument("--skip-strength", action="store_true")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_gumbel needs a CUDA device")
    engine = get_engine(0)
    name, smi = gpu_identity()
    say("tools/bench_gumbel.py on %s; nvidia-smi name, power limit, max SM clock: %s" % (name, smi))
    check_against_model(engine)
    say("CUDA events around whole 64-simulation searches after one warm-up search of each, Gumbel (max_considered 16, c_visit 50, "
        "c_scale 0.1, caller noise) and PUCT (c_puct 1.25, fpu 0) alternated search by search on the same roots, caller keys for "
        "the information-set searches (their S + 1 sb_determinize calls included), zero-cost evaluator (uniform prior, value 0); "
        "median of %d each; run-to-run spread not measured" % args.reps)
    for n in (int(x) for x in args.sizes.split(",")):
        bench_speed(engine, n, 64, args.reps)
    if not args.skip_strength:
        say("strength: first episode of %d envs, alternating seats, rollout_evaluator; Gumbel agents play the returned action "
            "(max_considered 16, default noise from seed 17), PUCT agents the arg-max of visits (c_puct 1.25, fpu 0); one run each"
            % args.episodes)
        n = args.episodes
        for opp in ("random", "expert"):
            for S in (16, 64):
                strength(engine, "GumbelMCTS S=%d" % S, GumbelMCTS(n, S, seed=17, engine=engine), opp, True)
                strength(engine, "BatchedMCTS S=%d" % S, BatchedMCTS(n, S, engine=engine), opp, False)
                strength(engine, "InformationSetGumbelMCTS S=%d" % S, InformationSetGumbelMCTS(n, S, seed=17, engine=engine), opp, True)
                strength(engine, "InformationSetMCTS S=%d" % S, InformationSetMCTS(n, S, seed=17, engine=engine), opp, False)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write("\n".join(LINES) + "\n")


if __name__ == "__main__":
    main()

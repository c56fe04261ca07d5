"""Batched tree search on one GPU: time per sb_search_simulate against sb_step + sb_observe, time of a rollout search,
workspace bytes, and the playing strength of a BatchedMCTS learner with the rollout evaluator in StormboundVecEnv.

Before anything is timed, one search on a small batch is checked against the plain-Python model (tests/sb_search_model.py):
visits, q and root values must be identical.  Writes the report to --out (default profiles/r4_bench_search.txt).
"""
import argparse
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")]

from monsoon_b200.engine import N_ACTIONS, get_engine  # noqa: E402
from monsoon_b200.search import BatchedMCTS, rollout_evaluator, select_actions  # noqa: E402
from monsoon_b200.vec_env import StormboundVecEnv  # noqa: E402

LINES = []


def say(s):
    print(s, flush=True)
    LINES.append(s)


def gpu_identity():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        q = "nvidia-smi unavailable (%s)" % e
    return name, q


def roots_of(engine, n, seed):
    env = StormboundVecEnv(n, seed=seed, opponent="random", seats=[g % 2 for g in range(n)], engine=engine)
    env.reset()
    return env.states.clone()


def constant_evaluator(n, dev):
    """zero-cost evaluator: preallocated uniform prior over all ids and value 0"""
    prior = torch.full((n, N_ACTIONS), 1.0 / N_ACTIONS, dtype=torch.float32, device=dev)
    value = torch.zeros(n, dtype=torch.float32, device=dev)
    return lambda leaf, k: (prior, value)


def check_against_model(engine, n=32, sims=24):
    import sb_search_model as M
    roots = roots_of(engine, n, 99)
    mcts = BatchedMCTS(n, sims, engine=engine)
    visits, q, rv = (t.cpu().numpy() for t in mcts.run(roots, constant_evaluator(n, engine.device)))
    prior = np.full(N_ACTIONS, 1.0 / N_ACTIONS, dtype=np.float32)
    host = roots.cpu().numpy()
    for g in range(n):
        t = M.TreeModel(host[g], sims + 1)
        t.begin()
        for _ in range(sims):
            t.simulate(prior, np.float32(0), mcts.c_puct, mcts.fpu)
        wv, wq, wr = t.end(prior, np.float32(0))
        assert np.array_equal(visits[g], wv) and np.array_equal(q[g], wq, equal_nan=True) and rv[g] == wr, g
    say("model check: %d trees x %d simulations: visits, q and root value identical to tests/sb_search_model.py" % (n, sims))


def time_events(fn, reps):
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    return float(np.median(ts)), float(np.min(ts))


def bench_speed(engine, n, sims, reps):
    dev = engine.device
    roots = roots_of(engine, n, 7)
    mcts = BatchedMCTS(n, sims, engine=engine)
    ev = constant_evaluator(n, dev)
    mcts.run(roots, ev)
    torch.cuda.synchronize()
    med, best = time_events(lambda: mcts.run(roots, ev), reps)
    actions = select_actions(mcts.out["visits"]).to(torch.uint8)
    st = roots.clone()
    reward = torch.empty(n, dtype=torch.int8, device=dev)
    done, err = torch.empty(n, dtype=torch.uint8, device=dev), torch.empty(n, dtype=torch.uint8, device=dev)

    def step_observe():
        engine.step(st, actions, reward, done, err)
        engine.observe(st)

    steps = []
    for _ in range(max(reps, 5) * 4):
        st.copy_(roots)
        steps.append(time_events(step_observe, 1)[0])
    floor = float(np.median(steps))
    say("n=%d sims=%d  workspace %d bytes (%.1f MB)  search %.2f ms (min %.2f)  per sb_search_simulate %.3f ms  "
        "sb_step+sb_observe %.3f ms  ratio %.2f" % (n, sims, mcts.ws.numel(), mcts.ws.numel() / 1e6, med, best, med / sims, floor,
                                                   med / sims / floor))


def bench_rollout_search(engine, n, sims, reps):
    roots = roots_of(engine, n, 8)
    mcts = BatchedMCTS(n, sims, engine=engine)
    ev = rollout_evaluator(engine)
    mcts.run(roots, ev)
    torch.cuda.synchronize()
    med, best = time_events(lambda: mcts.run(roots, ev), reps)
    say("rollout search n=%d sims=%d: %.1f ms per whole search (min %.1f), %.3f ms per simulation incl. rollout" % (n, sims, med, best,
                                                                                                              med / sims))


def strength(engine, n, sims, opponent, max_moves=600):
    env = StormboundVecEnv(n, seed=1234, opponent=opponent, seats=[g % 2 for g in range(n)], engine=engine)
    env.reset()
    mcts = BatchedMCTS(n, sims, engine=engine)
    ev = rollout_evaluator(engine)
    first = torch.full((n,), -3, dtype=torch.int8, device=engine.device)
    t0 = time.time()
    for _ in range(max_moves):
        visits, _q, _v = mcts.run(env.states, ev)
        _o, _m, _r, done, info = env.step(select_actions(visits))
        new = (first == -3) & done
        first = torch.where(new, info["result"], first)
        if not bool((first == -3).any()):
            break
    r = first.cpu().numpy()
    seat = np.arange(n) % 2
    won = int(((r == 0) & (seat == 0)).sum() + ((r == 1) & (seat == 1)).sum())
    lost = int(((r == 1) & (seat == 0)).sum() + ((r == 0) & (seat == 1)).sum())
    drawn = int(((r == -1) | (r == -2)).sum())
    say("strength: %d sims vs %-6s over %d episodes (mixed seats): win %d / draw %d / loss %d (unfinished %d; %.0f s)" % (
        sims, opponent, n, won, drawn, lost, int((r == -3).sum()), time.time() - t0))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r4_bench_search.txt"))
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--episodes", type=int, default=1024)
    ap.add_argument("--skip-strength", action="store_true")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_search needs a CUDA device")
    engine = get_engine(0)
    name, smi = gpu_identity()
    say("tools/bench_search.py on %s; nvidia-smi name, power limit, max SM clock: %s" % (name, smi))
    say("CUDA events around whole searches (begin + simulations + end) after one warm-up search; median of %d" % args.reps)
    check_against_model(engine)
    for n in (4096, 65536):
        bench_speed(engine, n, 64, args.reps)
    bench_rollout_search(engine, 4096, 64, max(2, args.reps // 2))
    if not args.skip_strength:
        for sims in (16, 64):
            for opp in ("random", "expert"):
                strength(engine, args.episodes, sims, opp)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write("\n".join(LINES) + "\n")


if __name__ == "__main__":
    main()

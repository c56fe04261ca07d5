"""Several leaves per tree per call (sb_search_simulate_batch / sb_search_end_batch, DESIGN.md 8.11) on one GPU: the time of
a whole 64-simulation search at L = 1 and L > 1 leaves per call, the time of each pass, and the playing strength.

Before anything is timed, one batched search of 32 trees is checked against the plain-Python model
(tests/sb_search_batch_model.py): every slot of every call and the read-out must be identical.  Writes the report to --out
(default profiles/r9_bench_search_batch.txt).
"""
import argparse
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests"), os.path.join(ROOT, "tools")]

from bench_reuse import play  # noqa: E402
from bench_search import LINES, gpu_identity, roots_of, say  # noqa: E402
from monsoon_b200.engine import N_ACTIONS, get_engine  # noqa: E402
from monsoon_b200.search import BatchedMCTS  # noqa: E402

KERNELS = ("k_search_simulate", "k_search_batch_select", "k_search_batch_expand", "k_search_end_batch", "k_search_end", "k_search_begin")


def zero_cost():
    """uniform prior over all ids and value 0, one preallocated pair per row count"""
    bufs = {}

    def evaluate(leaf, k):
        n = leaf["states"].shape[0]
        if n not in bufs:
            dev = leaf["states"].device
            bufs[n] = (torch.full((n, N_ACTIONS), 1.0 / N_ACTIONS, dtype=torch.float32, device=dev), torch.zeros(n, dtype=torch.float32, device=dev))
        return bufs[n]

    return evaluate


def check_against_model(engine, n=32, L=8, calls=4):
    from test_gpu_search_batch import run_batch_against_model
    kinds, _models = run_batch_against_model(engine, roots_of(engine, n, 99), L, 1.0, calls)
    say("model check: %d trees, L = %d, %d batch calls: every slot's record, observation, mask, seat and kind, visits, q and "
        "root value identical to tests/sb_search_batch_model.py (slot kinds %s)" % (n, L, calls, dict(sorted(kinds.items()))))


def timed(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def per_kernel(fn):
    """mean device time per launch of each search kernel over one call of fn (torch.profiler, a run of its own)"""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {}
    for evt in prof.key_averages():
        for k in KERNELS:
            if evt.key.startswith(k + "("):
                t = getattr(evt, "device_time_total", None) or getattr(evt, "cuda_time_total", 0)
                out[k] = (t / 1000.0 / max(evt.count, 1), evt.count)
    return out


def speed(engine, n, sims, Ls, reps):
    roots = roots_of(engine, n, 7)
    ev = zero_cost()
    base = BatchedMCTS(n, sims, engine=engine)
    res = {}
    for L in Ls:
        mcts = BatchedMCTS(n, sims, engine=engine, leaves_per_call=L)
        base.run(roots, ev)
        mcts.run(roots, ev)  # warm-up of both
        torch.cuda.synchronize()
        t1, tL = [], []
        for _ in range(reps):  # alternated search by search on the same roots
            t1.append(timed(lambda: base.run(roots, ev)))
            tL.append(timed(lambda: mcts.run(roots, ev)))
        visits = mcts.out["visits"].sum(1).float().mean().item()
        k1, kL = per_kernel(lambda: base.run(roots, ev)), per_kernel(lambda: mcts.run(roots, ev))
        m1, mL = float(np.median(t1)), float(np.median(tL))
        res[L] = (m1, mL)
        say("n=%6d S=%d: L=1 %8.3f ms per search (simulate %.4f ms per call) | L=%-2d %8.3f ms per search (%d calls: select %.4f ms, "
            "expand %.4f ms per call; end %.4f ms) | L=%d / L=1 %.3f | mean root visits at L=%d: %.1f of %d"
            % (n, sims, m1, k1.get("k_search_simulate", (float("nan"),))[0], L, mL, sims // L,
               kL.get("k_search_batch_select", (float("nan"),))[0], kL.get("k_search_batch_expand", (float("nan"),))[0],
               kL.get("k_search_end_batch", (float("nan"),))[0], L, mL / m1, L, visits, sims))
        del mcts
        torch.cuda.empty_cache()
    del base
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r9_bench_search_batch.txt"))
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--episodes", type=int, default=1024)
    ap.add_argument("--sizes", default="1,64,4096,65536")
    ap.add_argument("--leaves", default="4,16,64")
    ap.add_argument("--seeds", default="1234,1235")
    ap.add_argument("--skip-strength", action="store_true")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_search_batch needs a CUDA device")
    engine = get_engine(0)
    name, smi = gpu_identity()
    say("tools/bench_search_batch.py on %s; nvidia-smi name, power limit, max SM clock: %s" % (name, smi))
    check_against_model(engine)
    say("1. speed: CUDA events around whole 64-simulation BatchedMCTS searches (begin, the calls, end), zero-cost evaluator "
        "(uniform prior, value 0, preallocated), roots from StormboundVecEnv; one warm-up of each, then L = 1 and L > 1 "
        "alternated search by search on the same roots, median of %d; per-call pass times from torch.profiler in a separate "
        "run (mean device time per launch)" % args.reps)
    Ls = [int(x) for x in args.leaves.split(",")]
    goal = None
    for n in (int(x) for x in args.sizes.split(",")):
        r = speed(engine, n, 64, Ls, args.reps)
        if n == 4096 and 16 in r:
            goal = r[16]
    if goal:
        say("goal (4,096 trees, L = 16 in under half of L = 1's time): L=1 %.3f ms, L=16 %.3f ms, ratio %.3f: %s"
            % (goal[0], goal[1], goal[1] / goal[0], "met" if goal[1] < 0.5 * goal[0] else "missed"))
    if not args.skip_strength:
        n = args.episodes
        say("2. strength: BatchedMCTS S=64, rollout_evaluator, c_puct 1.25, fpu 0, virtual loss 1, arg-max of visits; first "
            "episode of %d envs, alternating seats, against expert; env seeds %s, one run each" % (n, args.seeds))
        for L in (1, 8, 16):
            for seed in (int(x) for x in args.seeds.split(",")):
                t0 = time.time()
                w, d, l, u, _kept = play(engine, BatchedMCTS(n, 64, engine=engine, leaves_per_call=L), "expert", seed, False)
                say("strength: L=%-2d vs expert seed %d: win %4d / draw %d / loss %4d (unfinished %d; %3.0f s)" % (L, seed, w, d, l, u, time.time() - t0))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write("\n".join(LINES) + "\n")


if __name__ == "__main__":
    main()

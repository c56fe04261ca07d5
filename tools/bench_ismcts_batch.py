"""Several leaves per information-set tree per call (sb_ismcts_simulate_batch / sb_ismcts_end_batch, DESIGN.md 8.12) on one
GPU: the time of a whole 64-simulation InformationSetMCTS search at L = 1 and L > 1 leaves per call, the time of each pass,
and the playing strength.

Before anything is timed, one batched search of 32 trees is checked against the plain-Python model
(tests/sb_ismcts_batch_model.py): every slot of every call and the read-out must be identical.  Writes the report to --out
(default profiles/r10_bench_ismcts_batch.txt).
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
from monsoon_b200.search import InformationSetMCTS  # noqa: E402

KERNELS = ("k_ismcts_simulate", "k_ismcts_simulate_batch", "k_ismcts_end_batch", "k_ismcts_end", "k_ismcts_begin", "k_determinize")


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
    from test_gpu_ismcts_batch import run_batch_against_model
    kinds, _models = run_batch_against_model(engine, roots_of(engine, n, 99), L, 1.0, calls)
    say("model check: %d trees, L = %d, %d batch calls: every slot's record, observation, mask, seat and kind, visits, q and "
        "root value identical to tests/sb_ismcts_batch_model.py (slot kinds %s)" % (n, L, calls, dict(sorted(kinds.items()))))


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
    from test_gpu_determinize import keys_for
    roots = roots_of(engine, n, 7)
    keys = keys_for(n * (sims + 1), 5).to(engine.device)
    ev = zero_cost()
    base = InformationSetMCTS(n, sims, engine=engine)
    res = {}
    for L in Ls:
        mcts = InformationSetMCTS(n, sims, engine=engine, leaves_per_call=L)
        base.run(roots, ev, keys)
        mcts.run(roots, ev, keys)  # warm-up of both
        torch.cuda.synchronize()
        t1, tL = [], []
        for _ in range(reps):  # alternated search by search on the same roots and keys
            t1.append(timed(lambda: base.run(roots, ev, keys)))
            tL.append(timed(lambda: mcts.run(roots, ev, keys)))
        visits = mcts.out["visits"].sum(1).float().mean().item()
        k1, kL = per_kernel(lambda: base.run(roots, ev, keys)), per_kernel(lambda: mcts.run(roots, ev, keys))
        m1, mL = float(np.median(t1)), float(np.median(tL))
        res[L] = (m1, mL)
        nan = (float("nan"),)
        say("n=%6d S=%d: L=1 %8.3f ms per search (simulate %.4f, determinize %.4f ms per call) | L=%-2d %8.3f ms per search "
            "(%d calls: batch %.4f, determinize %.4f ms per call; end %.4f ms) | L=%d / L=1 %.3f | mean root visits at L=%d: %.1f of %d"
            % (n, sims, m1, k1.get("k_ismcts_simulate", nan)[0], k1.get("k_determinize", nan)[0], L, mL, sims // L,
               kL.get("k_ismcts_simulate_batch", nan)[0], kL.get("k_determinize", nan)[0], kL.get("k_ismcts_end_batch", nan)[0],
               L, mL / m1, L, visits, sims))
        del mcts
        torch.cuda.empty_cache()
    del base
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r10_bench_ismcts_batch.txt"))
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--episodes", type=int, default=1024)
    ap.add_argument("--sizes", default="1,64,4096,65536")
    ap.add_argument("--leaves", default="4,16,64")
    ap.add_argument("--seeds", default="1234,1235")
    ap.add_argument("--skip-strength", action="store_true")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_ismcts_batch needs a CUDA device")
    engine = get_engine(0)
    name, smi = gpu_identity()
    say("tools/bench_ismcts_batch.py on %s; nvidia-smi name, power limit, max SM clock: %s" % (name, smi))
    check_against_model(engine)
    say("1. speed: CUDA events around whole 64-simulation InformationSetMCTS searches (the sb_determinize calls, begin, the "
        "calls, end) with caller keys, zero-cost evaluator (uniform prior, value 0, preallocated), roots from StormboundVecEnv; "
        "one warm-up of each, then L = 1 and L > 1 "
        "alternated search by search on the same roots, median of %d; per-call pass times from torch.profiler in a separate "
        "run (mean device time per launch)" % args.reps)
    Ls = [int(x) for x in args.leaves.split(",")]
    res = {}
    for n in (int(x) for x in args.sizes.split(",")):
        res[n] = speed(engine, n, 64, Ls, args.reps)
    for n, want, what in ((1, 0.5, "under half of"), (64, 0.5, "under half of"), (4096, 1.0, "no slower than")):
        if n in res and 16 in res[n]:
            m1, m16 = res[n][16]
            ok = m16 < want * m1 if want < 1 else m16 <= m1
            say("goal (%d trees, L = 16 %s L = 1's time): L=1 %.3f ms, L=16 %.3f ms, ratio %.3f: %s"
                % (n, what, m1, m16, m16 / m1, "met" if ok else "missed"))
    if not args.skip_strength:
        n = args.episodes
        say("2. strength: InformationSetMCTS S=64, rollout_evaluator, c_puct 1.25, fpu 0, virtual loss 1, default keys (seed 17), "
            "arg-max of visits; first "
            "episode of %d envs, alternating seats, against expert; env seeds %s, one run each" % (n, args.seeds))
        for L in (1, 8, 16):
            for seed in (int(x) for x in args.seeds.split(",")):
                t0 = time.time()
                w, d, l, u, _kept = play(engine, InformationSetMCTS(n, 64, seed=17, engine=engine, leaves_per_call=L), "expert", seed, True)
                say("strength: L=%-2d vs expert seed %d: win %4d / draw %d / loss %4d (unfinished %d; %3.0f s)" % (L, seed, w, d, l, u, time.time() - t0))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write("\n".join(LINES) + "\n")


if __name__ == "__main__":
    main()

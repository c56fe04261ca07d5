"""Determinization on one GPU: time of sb_determinize against a copy_ of the same bytes, and the playing strength of a
DeterminizedMCTS learner (Perfect-Information Monte Carlo) beside the perfect-information BatchedMCTS in StormboundVecEnv.

Before anything is timed, sb_determinize on a small batch is checked byte for byte against the plain-Python model
(tests/sb_determinize_model.py).  Writes the report to --out (default profiles/r5_bench_determinize.txt).
"""
import argparse
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests"), os.path.join(ROOT, "tools")]

import bench_search as BS  # noqa: E402
from monsoon_b200.engine import get_engine  # noqa: E402
from monsoon_b200.search import BatchedMCTS, DeterminizedMCTS, rollout_evaluator, select_actions  # noqa: E402
from monsoon_b200.vec_env import StormboundVecEnv, next_seed_array  # noqa: E402

say = BS.say


def keys_of(n, dev, salt=0):
    return torch.from_numpy(next_seed_array(np.arange(n, dtype=np.uint64) + np.uint64(salt))).to(dev)


def check_against_model(engine, n=1024):
    import sb_determinize_model as D
    roots = BS.roots_of(engine, n, 98)
    keys = keys_of(n, engine.device, 5)
    got = engine.determinize(roots, keys).cpu().numpy()
    host, hk = roots.cpu().numpy(), keys.cpu().numpy().view(np.uint64)
    for g in range(n):
        assert got[g].tobytes() == D.determinize(host[g], int(hk[g])).tobytes(), g
    say("model check: %d records: sb_determinize output identical to tests/sb_determinize_model.py" % n)


def bench_kernel(engine, n, reps):
    """records from 4,096 env roots tiled to n (the kernel's work does not depend on which record it gets); out of place, so
    every pass reads n * 512 B and writes n * 512 B, beside a copy_ of the same bytes"""
    dev = engine.device
    base = BS.roots_of(engine, min(n, 4096), 7)
    roots = base.repeat((n + base.shape[0] - 1) // base.shape[0], 1)[:n].contiguous()
    keys = keys_of(n, dev, 1)
    out = torch.empty_like(roots)
    det = lambda: engine.determinize(roots, keys, out=out)  # noqa: E731
    cp = lambda: out.copy_(roots)  # noqa: E731
    for f in (det, cp):
        f()
    torch.cuda.synchronize()
    reps_inner = max(1, 2 ** 22 // n)  # a window of ~4 M records per timed sample
    td = BS.time_events(lambda: [det() for _ in range(reps_inner)], reps)[0] / reps_inner
    tc = BS.time_events(lambda: [cp() for _ in range(reps_inner)], reps)[0] / reps_inner
    gb = n * 1024 / 1e9
    say("n=%d (%.1f MB moved)  sb_determinize %.4f ms = %.0f GB/s  copy_ %.4f ms = %.0f GB/s  ratio %.2f" % (
        n, gb * 1e3, td, gb / (td / 1e3), tc, gb / (tc / 1e3), td / tc))


def strength(engine, n, make, label, opponent, max_moves=600):
    """bench_search.strength's protocol: the first episode of n envs with alternating seats, rollout evaluator, arg-max"""
    env = StormboundVecEnv(n, seed=1234, opponent=opponent, seats=[g % 2 for g in range(n)], engine=engine)
    env.reset()
    mcts = make(n)
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
    say("strength: %-26s vs %-6s over %d episodes (mixed seats): win %d / draw %d / loss %d (unfinished %d; %.0f s)" % (
        label, opponent, n, won, drawn, lost, int((r == -3).sum()), time.time() - t0))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r5_bench_determinize.txt"))
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--episodes", type=int, default=1024)
    ap.add_argument("--skip-strength", action="store_true")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_determinize needs a CUDA device")
    engine = get_engine(0)
    name, smi = BS.gpu_identity()
    say("tools/bench_determinize.py on %s; nvidia-smi name, power limit, max SM clock: %s" % (name, smi))
    say("CUDA events, median of %d samples of back-to-back calls after a warm-up; GB/s counts 1,024 B per record "
        "(512 read + 512 written); at n >= 262,144 the 2 x n x 512 B exceed the 126 MB L2" % args.reps)
    check_against_model(engine)
    for n in (4096, 65536, 1048576):
        bench_kernel(engine, n, args.reps)
    if not args.skip_strength:
        arms = [("DeterminizedMCTS K=%d S=%d" % (k, s), lambda n, k=k, s=s: DeterminizedMCTS(n, k, s, seed=11, engine=engine))
                for k, s in ((4, 16), (8, 8), (4, 64))]
        arms.append(("BatchedMCTS S=64 (perfect)", lambda n: BatchedMCTS(n, 64, engine=engine)))
        for label, make in arms:
            for opp in ("random", "expert"):
                strength(engine, args.episodes, make, label, opp)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write("\n".join(BS.LINES) + "\n")


if __name__ == "__main__":
    main()

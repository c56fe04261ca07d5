"""Tree reuse between moves on one GPU (sb_search_advance / sb_ismcts_advance, DESIGN.md 8.10): the cost of an advance
against a begin and one simulate call, how often the trees are reused in play, and the playing strength with and without
reuse.

Before anything is timed, two moves of both searches on 32 trees are checked against the plain-Python model
(tests/sb_reuse_model.py): every leaf, kept count and read-out must be identical.  Writes the report to --out (default
profiles/r8_bench_reuse.txt).
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
from monsoon_b200.engine import get_engine  # noqa: E402
from monsoon_b200.search import BatchedMCTS, InformationSetMCTS, rollout_evaluator, select_actions  # noqa: E402
from monsoon_b200.vec_env import StormboundVecEnv  # noqa: E402


def check_against_model(engine, n=32, sims=16):
    from test_gpu_reuse import ISPair, SearchPair, stepped
    for ism in (False, True):
        pair = ISPair(engine, n, sims, 2 * sims + 1) if ism else SearchPair(engine, n, sims, 2 * sims + 1)
        roots = roots_of(engine, n, 98)
        _kept, visits = pair.search(roots)
        total = 0
        for _ in range(2):
            a = select_actions(visits)
            roots = stepped(engine, roots, a)
            kept, visits = pair.search(roots, torch.where(a < 156, a, -1).to(torch.int32), sims + 1) if ism else pair.search(roots, sims + 1)
            total += int((kept > 0).sum())
        say("model check (%s): %d trees, a fresh search and two advancing ones of %d simulations (%d advances kept a subtree): "
            "every leaf, kept count, visits, q and root value identical to tests/sb_reuse_model.py"
            % ("information-set" if ism else "perfect-information", n, sims, total))


def cost(engine, n, sims, reps):
    """CUDA events around one advance (its source restored from a copy before each), one begin and one simulate call"""
    dev = engine.device
    ev = constant_evaluator(n, dev)
    roots = roots_of(engine, n, 7)
    keys = keys_of(n * (sims + 1), 11, dev)
    for ism in (False, True):
        mcts = InformationSetMCTS(n, sims, reuse_nodes=sims, engine=engine) if ism else BatchedMCTS(n, sims, reuse_nodes=sims, engine=engine)
        visits = (mcts.run(roots, ev, keys) if ism else mcts.run(roots, ev))[0]
        a = select_actions(visits)
        nxt = roots.clone()
        engine.step(nxt, torch.where(a < 156, a, 155).to(torch.uint8).contiguous())
        played = torch.where(a < 156, a, -1).to(torch.int32)
        m, keep = mcts.max_nodes, sims + 1
        pristine, src, dst = mcts.ws.clone(), mcts.ws, mcts.ws_next
        det = engine.determinize(nxt, keys[:n])
        prior, value = ev(None, 0)
        out = dict(mcts.leaf, kept=mcts.kept)

        def advance():
            if ism:
                engine.ismcts_advance(src, dst, det, played, m, keep, out=out)
            else:
                engine.search_advance(src, dst, nxt, m, keep, out=out)

        def begin():
            (engine.ismcts_begin if ism else engine.search_begin)(src, det if ism else nxt, m, out=mcts.leaf)

        def simulate():
            if ism:
                engine.ismcts_simulate(dst, det, m, prior, value, out=mcts.leaf)
            else:
                engine.search_simulate(dst, n, m, prior, value, out=mcts.leaf)

        times = {"advance": [], "begin": [], "simulate": []}
        for rep in range(reps + 1):  # rep 0 is the warm-up
            for name, fn in (("advance", advance), ("simulate", simulate), ("begin", begin)):
                if name == "advance":
                    src.copy_(pristine)
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                fn()
                e1.record()
                torch.cuda.synchronize()
                if rep:
                    times[name].append(e0.elapsed_time(e1))
            if rep == 0:
                kept = mcts.kept.cpu().numpy()
        med = {k: float(np.median(v)) for k, v in times.items()}
        say("n=%d %-15s trees of a %d-simulation search (max_nodes %d), keep %d: kept > 0 in %.1f %% of trees, mean kept %.1f | "
            "advance %.3f ms (min %.3f), begin %.3f ms (min %.3f), one simulate call %.3f ms (min %.3f); advance / simulate %.2f"
            % (n, "information-set" if ism else "perfect-info", sims, m, keep, 100.0 * (kept > 0).mean(), kept.mean(), med["advance"],
               min(times["advance"]), med["begin"], min(times["begin"]), med["simulate"], min(times["simulate"]),
               med["advance"] / med["simulate"]))
        del mcts, pristine, src, dst, out
        torch.cuda.empty_cache()


def play(engine, mcts, opponent, seed, ism, max_moves=600):
    """the first episode of every env against `opponent` (None: self-play); returns (won, drawn, lost, unfinished, kept list)"""
    n = mcts.n
    env = StormboundVecEnv(n, seed=seed, opponent=opponent, seats=None if opponent is None else [g % 2 for g in range(n)], engine=engine)
    env.reset()
    ev = rollout_evaluator(engine)
    first = torch.full((n,), -3, dtype=torch.int8, device=engine.device)
    played, kept = None, []
    for _ in range(max_moves):
        live = first == -3
        visits = (mcts.run(env.states, ev, played=played) if ism else mcts.run(env.states, ev))[0]
        if mcts.reuse_nodes:
            kept.append(mcts.kept[live].cpu().numpy())
        played = select_actions(visits)
        _o, _m, _r, done, info = env.step(played)
        first = torch.where((first == -3) & done, info["result"], first)
        if not bool((first == -3).any()):
            break
    r = first.cpu().numpy()
    seat = np.arange(n) % 2
    won = int(((r == 0) & (seat == 0)).sum() + ((r == 1) & (seat == 1)).sum())
    lost = int(((r == 1) & (seat == 0)).sum() + ((r == 0) & (seat == 1)).sum())
    return won, int(((r == -1) | (r == -2)).sum()), lost, int((r == -3).sum()), np.concatenate(kept) if kept else None


def make(engine, ism, n, S, reuse):
    return (InformationSetMCTS(n, S, seed=17, reuse_nodes=S if reuse else 0, engine=engine) if ism
            else BatchedMCTS(n, S, reuse_nodes=S if reuse else 0, engine=engine))


def reuse_rate(kept):
    return "decisions with kept > 0: %5.1f %%, mean kept %5.1f" % (100.0 * (kept > 0).mean(), kept.mean())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r8_bench_reuse.txt"))
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--episodes", type=int, default=1024)
    ap.add_argument("--sizes", default="4096,65536")
    ap.add_argument("--seeds", default="1234,1235")
    ap.add_argument("--skip-strength", action="store_true")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_reuse needs a CUDA device")
    engine = get_engine(0)
    name, smi = gpu_identity()
    say("tools/bench_reuse.py on %s; nvidia-smi name, power limit, max SM clock: %s" % (name, smi))
    check_against_model(engine)
    say("1. cost: CUDA events around single calls, after one warm-up of each; the advance reads trees of a real 64-simulation "
        "search (zero-cost evaluator: uniform prior, value 0) and advances to the child of the most visited action; its source "
        "workspace is restored from a copy before each timed advance (not timed); median and min of %d; spread between runs not "
        "measured" % args.reps)
    for n in (int(x) for x in args.sizes.split(",")):
        cost(engine, n, 64, args.reps)
    n = args.episodes
    seeds = [int(x) for x in args.seeds.split(",")]
    say("2. reuse rate and 3. strength: first episode of %d envs (alternating seats against an opponent), rollout_evaluator, "
        "c_puct 1.25, fpu 0, arg-max of visits; reuse_nodes = S when reused; the reuse rate counts decisions of envs still in "
        "their first episode; env seeds %s, one run each" % (n, args.seeds))
    for opp in (None, "random", "expert"):
        for ism in (False, True):
            w, d, l, u, kept = play(engine, make(engine, ism, n, 16, True), opp, seeds[0], ism)
            say("reuse: %-18s S=16 %-9s seed %d: %s" % ("InformationSetMCTS" if ism else "BatchedMCTS", opp or "self-play", seeds[0],
                                                       reuse_rate(kept)))
    if not args.skip_strength:
        for opp in ("random", "expert"):
            for ism in (False, True):
                for S in (16, 64):
                    for reuse in (False, True):
                        for seed in seeds:
                            t0 = time.time()
                            w, d, l, u, kept = play(engine, make(engine, ism, n, S, reuse), opp, seed, ism)
                            say("strength: %-18s S=%-2d reuse %-3s vs %-6s seed %d: win %4d / draw %d / loss %4d (unfinished %d; %3.0f s)%s"
                                % ("InformationSetMCTS" if ism else "BatchedMCTS", S, "yes" if reuse else "no", opp, seed, w, d, l, u,
                                   time.time() - t0, " | " + reuse_rate(kept) if reuse else ""))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write("\n".join(LINES) + "\n")


if __name__ == "__main__":
    main()

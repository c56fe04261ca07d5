"""Information-set tree search on one GPU: time per simulation of InformationSetMCTS (sb_determinize + sb_ismcts_simulate)
against the perfect-information search plus one determinization (sb_search_simulate + sb_determinize), workspace bytes, and
the playing strength of InformationSetMCTS and DeterminizedMCTS learners with the rollout evaluator in StormboundVecEnv.

Before anything is timed, one search on a small batch is checked against the plain-Python model (tests/sb_ismcts_model.py):
every leaf, visits, q and root values must be identical.  Writes the report to --out (default profiles/r6_bench_ismcts.txt).
"""
import argparse
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests"), os.path.join(ROOT, "tools")]

from bench_search import LINES, constant_evaluator, gpu_identity, roots_of, say, time_events  # noqa: E402
from monsoon_b200.engine import N_ACTIONS, get_engine  # noqa: E402
from monsoon_b200.search import BatchedMCTS, DeterminizedMCTS, InformationSetMCTS, rollout_evaluator, select_actions  # noqa: E402
from monsoon_b200.vec_env import StormboundVecEnv  # noqa: E402
from monsoon_b200.vec_env import next_seed_array  # noqa: E402


def keys_of(count, salt, dev):
    return torch.from_numpy(next_seed_array(np.arange(count, dtype=np.uint64) + np.uint64(salt))).to(dev)


def check_against_model(engine, n=32, sims=24):
    import sb_determinize_model as D
    import sb_ismcts_model as I
    roots = roots_of(engine, n, 99)
    keys = keys_of(n * (sims + 1), 5, engine.device)
    host, hk = roots.cpu().numpy(), keys.cpu().numpy().view(np.uint64)
    prior = np.full(N_ACTIONS, 1.0 / N_ACTIONS, dtype=np.float32)
    models = [I.ISTreeModel(sims + 1) for _ in range(n)]
    seen = {}
    ev = constant_evaluator(n, engine.device)

    def evaluate(leaf, k):
        world = [D.determinize(host[g], int(hk[k * n + g])) for g in range(n)]
        want = [t.begin(world[g]) if k == 0 else t.simulate(world[g], prior, np.float32(0), 1.25, 0.0) for g, t in enumerate(models)]
        states = leaf["states"].cpu().numpy()
        assert all(states[g].tobytes() == want[g][0].tobytes() for g in range(n)), k
        seen[k] = True
        return ev(leaf, k)

    mcts = InformationSetMCTS(n, sims, engine=engine)
    visits, q, rv = (t.cpu().numpy() for t in mcts.run(roots, evaluate, keys))
    for g, t in enumerate(models):
        wv, wq, wr = t.end(prior, np.float32(0))
        assert np.array_equal(visits[g], wv) and np.array_equal(q[g], wq, equal_nan=True) and rv[g] == wr, g
    say("model check: %d trees x %d simulations: every leaf record, visits, q and root value identical to tests/sb_ismcts_model.py"
        % (n, len(seen) - 1))


def bench_speed(engine, n, sims, reps):
    dev = engine.device
    roots = roots_of(engine, n, 7)
    ev = constant_evaluator(n, dev)
    keys = keys_of(n * (sims + 1), 11, dev)
    ism = InformationSetMCTS(n, sims, engine=engine)
    ism.run(roots, ev, keys)
    torch.cuda.synchronize()
    med, best = time_events(lambda: ism.run(roots, ev, keys), reps)
    del ism
    torch.cuda.empty_cache()
    pim = BatchedMCTS(n, sims, engine=engine)
    pim.run(roots, ev)
    torch.cuda.synchronize()
    pmed, _pbest = time_events(lambda: pim.run(roots, ev), reps)
    ws_pim = pim.ws.numel()
    del pim
    torch.cuda.empty_cache()
    out = torch.empty_like(roots)
    dmed, _dbest = time_events(lambda: engine.determinize(roots, keys[:n], out=out), max(reps, 5) * 4)
    per, floor = med / sims, pmed / sims + dmed
    say("n=%d sims=%d  workspace %.1f MB (sb_search %.1f MB)  InformationSetMCTS search %.2f ms (min %.2f) = %.3f ms per simulation  "
        "sb_search_simulate %.3f ms + sb_determinize %.4f ms = %.3f ms  ratio %.2f" % (
            n, sims, engine.ismcts_workspace_bytes(n, sims + 1) / 1e6, ws_pim / 1e6, med, best, per, pmed / sims, dmed, floor, per / floor))


def strength(engine, label, mcts, opponent, max_moves=600):
    """the first episode of every env of a StormboundVecEnv against `opponent`, the learner playing the arg-max of mcts's visits"""
    n = mcts.n
    env = StormboundVecEnv(n, seed=1234, opponent=opponent, seats=[g % 2 for g in range(n)], engine=engine)
    env.reset()
    ev = rollout_evaluator(engine)
    first = torch.full((n,), -3, dtype=torch.int8, device=engine.device)
    t0 = time.time()
    for _ in range(max_moves):
        visits, _q, _v = mcts.run(env.states, ev)
        _o, _m, _r, done, info = env.step(select_actions(visits))
        first = torch.where((first == -3) & done, info["result"], first)
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
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r6_bench_ismcts.txt"))
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--episodes", type=int, default=1024)
    ap.add_argument("--skip-strength", action="store_true")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_ismcts needs a CUDA device")
    engine = get_engine(0)
    name, smi = gpu_identity()
    say("tools/bench_ismcts.py on %s; nvidia-smi name, power limit, max SM clock: %s" % (name, smi))
    say("CUDA events around whole 64-simulation searches (the S + 1 sb_determinize calls, begin, simulations, end) after one "
        "warm-up search, caller keys, zero-cost evaluator (uniform prior, value 0); median of %d; the floor is one "
        "sb_search_simulate (a whole BatchedMCTS search / 64, same roots and evaluator) plus one sb_determinize call" % args.reps)
    check_against_model(engine)
    for n in (4096, 65536):
        bench_speed(engine, n, 64, args.reps)
    if not args.skip_strength:
        say("strength: first episode of %d envs, alternating seats, rollout_evaluator, c_puct 1.25, fpu 0, arg-max of visits"
            % args.episodes)
        n = args.episodes
        for opp in ("random", "expert"):
            strength(engine, "InformationSetMCTS S=64", InformationSetMCTS(n, 64, seed=17, engine=engine), opp)
            strength(engine, "InformationSetMCTS S=256", InformationSetMCTS(n, 256, seed=17, engine=engine), opp)
            strength(engine, "DeterminizedMCTS K=4 S=64", DeterminizedMCTS(n, 4, 64, seed=17, engine=engine), opp)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write("\n".join(LINES) + "\n")


if __name__ == "__main__":
    main()

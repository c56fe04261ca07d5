"""GPU: sb_search_begin / sb_search_simulate / sb_search_end (and BatchedMCTS) against the plain-Python search model."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

import sb_oracle as O
import sb_search_model as M
from monsoon_b200 import _lib
from monsoon_b200.search import BatchedMCTS, masked_softmax, rollout_evaluator, select_actions
from monsoon_b200.vec_env import StormboundVecEnv

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LEAF = ("states", "obs", "masks", "obs_err", "to_move", "kind")
FEATURE_W = np.array([0.3, -0.2, 0.1, -0.1, 0.05, -0.05, 0.2, -0.3, 0.15, -0.15])


def env_roots(engine, n, seed, decks=False, plies=5):
    """records of a StormboundVecEnv against the random agent with mixed seats, after a few random learner actions"""
    kw = {}
    if decks:
        seeds = np.arange(n, dtype=np.int64) + 1000 * seed
        fac = np.stack([1 + seeds % 4, 1 + (seeds // 4) % 4], axis=1).astype(np.uint8)
        kw["decks"], kw["factions"] = engine.generate_decks(seeds, 3, 3, factions=fac)
    env = StormboundVecEnv(n, seed=seed, opponent="random", seats=[(g // 2) % 2 for g in range(n)], engine=engine, **kw)
    env.reset()
    rs = np.random.RandomState(seed)
    for k in range(plies):
        mask = env.action_mask().cpu().numpy()
        acts = np.array([rs.choice(np.flatnonzero(m)) if (g + k) % 3 else 255 for g, m in enumerate(mask)])  # 255: stays put
        env.step(torch.from_numpy(acts).to(engine.device))
    return env.states.clone()


def host_eval(leaves):
    """the evaluator on the model's leaves: prior from a hash of (record digest, action), value from the oracle's features"""
    n = len(leaves)
    prior, value = np.empty((n, M.N_ACTIONS), dtype=np.float32), np.empty(n, dtype=np.float32)
    a = np.arange(M.N_ACTIONS, dtype=np.uint64)
    for g, leaf in enumerate(leaves):
        d = O.digest(leaf[0])
        with np.errstate(over="ignore"):
            h = (np.uint64(d) ^ (a * np.uint64(0x9E3779B97F4A7C15))) * np.uint64(0xBF58476D1CE4E5B9)
        prior[g] = ((h >> np.uint64(40)).astype(np.float64) / 2.0**24).astype(np.float32)
        f, _err = O.features(leaf[0].copy())
        value[g] = np.float32(np.tanh(np.clip(np.nan_to_num(f), -50, 50) @ FEATURE_W))
    return prior, value


def compare_leaves(o, want, call):
    got = {k: o[k].cpu().numpy() for k in LEAF}
    for g, (rec, obs, err, mask, to_move, kind) in enumerate(want):
        assert got["states"][g].tobytes() == rec.tobytes(), (call, g)
        assert np.array_equal(got["obs"][g], obs) and int(got["obs_err"][g]) == err, (call, g)
        assert np.array_equal(got["masks"][g], mask), (call, g)
        assert (int(got["to_move"][g]), int(got["kind"][g])) == (to_move, kind), (call, g)


def run_against_model(engine, roots, sims, c_puct, fpu, max_steps=400, rollout=False, max_nodes=None, calls=None):
    """drive the three calls and the model side by side; every call's leaf outputs and the final read-out must be identical"""
    dev = engine.device
    n = roots.shape[0]
    m = max_nodes or sims + 1
    host = roots.cpu().numpy()
    models = [M.TreeModel(host[g], m, max_steps) for g in range(n)]
    ws = torch.empty(engine.search_workspace_bytes(n, m), dtype=torch.uint8, device=dev)
    o = engine.search_begin(ws, roots, m, max_steps)
    want = [t.begin() for t in models]
    kinds = {}
    ev = rollout_evaluator(engine) if rollout else None

    def evaluate():
        for lf in want:
            kinds[lf[5]] = kinds.get(lf[5], 0) + 1
        if not rollout:
            p, v = host_eval(want)
            return torch.from_numpy(p).to(dev), torch.from_numpy(v).to(dev), p, v
        p, v = ev(o, 0)
        pv = [M.rollout_eval(lf) for lf in want]
        wp, wv = np.stack([x[0] for x in pv]), np.array([x[1] for x in pv], dtype=np.float32)
        assert np.array_equal(p.cpu().numpy(), wp) and np.array_equal(v.cpu().numpy(), wv)
        return p, v, wp, wv

    compare_leaves(o, want, 0)
    prior, value, hp, hv = evaluate()
    for k in range(1, (calls if calls is not None else sims) + 1):
        o = engine.search_simulate(ws, n, m, prior, value, c_puct, fpu, out={key: o[key] for key in LEAF})
        want = [t.simulate(hp[g], hv[g], c_puct, fpu) for g, t in enumerate(models)]
        compare_leaves(o, want, k)
        prior, value, hp, hv = evaluate()
    r = engine.search_end(ws, n, m, prior, value)
    ends = [t.end(hp[g], hv[g]) for g, t in enumerate(models)]
    assert np.array_equal(r["visits"].cpu().numpy(), np.stack([e[0] for e in ends]))
    assert np.array_equal(r["q"].cpu().numpy(), np.stack([e[1] for e in ends]), equal_nan=True)
    assert np.array_equal(r["root_value"].cpu().numpy(), np.array([e[2] for e in ends]))
    return kinds, models


@pytest.mark.parametrize("c_puct,fpu,decks", [(1.25, 0.0, False), (2.5, -0.3, True)])
def test_search_matches_model(engine, oracle, c_puct, fpu, decks):
    n = 257
    roots = env_roots(engine, n, 3 if decks else 1, decks)
    finished = roots[::16].clone()
    engine.rollout_random(finished)  # whole games: terminal roots
    roots[::16] = finished
    kinds, models = run_against_model(engine, roots, 48, c_puct, fpu)
    assert kinds.get(M.TERMINAL, 0) > 0 and kinds.get(M.EVAL, 0) > 0, kinds
    assert any(t.nodes[0].terminal for t in models) and any(t.nodes[0].seat for t in models) and not all(t.nodes[0].seat for t in models)


def test_search_matches_model_with_terminal_depth(engine, oracle):
    n = 257
    roots = env_roots(engine, n, 5, plies=8)
    steps = roots[:, 12:14].contiguous().view(torch.int16).to(torch.int32)
    kinds, models = run_against_model(engine, roots, 48, 1.25, 0.0, max_steps=int(steps.min()) + 2)
    assert kinds.get(M.TERMINAL, 0) > n, kinds
    assert any(nd.terminal and nd.parent >= 0 for t in models for nd in t.nodes)


def test_search_matches_model_with_rollout_evaluator(engine, oracle):
    roots = env_roots(engine, 257, 7, plies=10)
    kinds, _ = run_against_model(engine, roots, 48, 1.25, 0.0, rollout=True)
    assert kinds.get(M.EVAL, 0) > 0


def test_full_trees_stop(engine, oracle):
    roots = env_roots(engine, 65, 11)
    kinds, models = run_against_model(engine, roots, 8, 1.25, 0.0, max_nodes=5, calls=8)
    assert kinds.get(M.FULL, 0) >= 4 * 65 and all(len(t.nodes) <= 5 for t in models)


def torch_eval(leaf, k):
    """a zero-cost stand-in for a network: softmax of a fixed function of the observation over the legal set"""
    x = leaf["obs"].view(leaf["obs"].shape[0], -1)[:, :M.N_ACTIONS].to(torch.float32)
    return masked_softmax(x * 0.1, leaf["masks"]), torch.tanh(x[:, :8].sum(1) * 0.05)


def test_launch_count_and_cuda_graph(engine):
    n, sims = 300, 24
    roots = env_roots(engine, n, 13)
    eager = BatchedMCTS(n, sims, engine=engine)
    before = engine.launches
    visits, q, root_value = eager.run(roots, torch_eval)
    torch.cuda.synchronize()
    assert engine.launches == before + sims + 2
    assert bool((visits.sum(1) == sims).all()) and bool((root_value.abs() <= 1).all())
    want = [t.clone() for t in (visits, q, root_value)]
    graphed = BatchedMCTS(n, sims, engine=engine)
    static_roots = roots.clone()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        graphed.run(static_roots, torch_eval)  # warm-up outside the capture
    torch.cuda.current_stream().wait_stream(side)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        outs = graphed.run(static_roots, torch_eval)
    for t in outs:
        t.zero_()
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(outs[0], want[0]) and torch.equal(outs[2], want[2])
    assert torch.equal(torch.nan_to_num(outs[1], nan=7.0), torch.nan_to_num(want[1], nan=7.0))
    other = env_roots(engine, n, 14)
    static_roots.copy_(other)
    g.replay()
    again = eager.run(other, torch_eval)
    torch.cuda.synchronize()
    assert torch.equal(outs[0], again[0]) and torch.equal(outs[2], again[2])
    a = select_actions(outs[0])
    assert bool((a < M.N_ACTIONS).all())


def test_mcts_plays_in_a_vec_env(engine):
    n = 64
    env = StormboundVecEnv(n, seed=21, opponent="expert", seats=[g % 2 for g in range(n)], engine=engine)
    env.reset()
    mcts = BatchedMCTS(n, 8, engine=engine)
    ev = rollout_evaluator(engine)
    for _ in range(20):
        visits, _q, _v = mcts.run(env.states, ev)
        a = select_actions(visits)
        assert bool((a < M.N_ACTIONS).all())
        assert bool(env.action_mask().gather(1, a.unsqueeze(1)).all())
        _o, _m, _r, _d, info = env.step(a)
        assert not bool((info["result"] == -4).any())


def test_empty_batch_and_rejected_arguments(engine):
    dev = engine.device
    lib, h = engine.lib, engine.h
    n, m = 8, 5
    roots = env_roots(engine, n, 17, plies=1)
    ws = torch.empty(engine.search_workspace_bytes(n, m) + 16, dtype=torch.uint8, device=dev)
    o = engine.search_begin(ws, roots, m)
    prior = torch.full((n, M.N_ACTIONS), 0.1, dtype=torch.float32, device=dev)
    value = torch.zeros(n, dtype=torch.float32, device=dev)
    before = engine.launches
    empty = torch.empty((0, 512), dtype=torch.uint8, device=dev)
    engine.search_begin(ws[:0], empty, m)
    engine.search_simulate(ws[:0], 0, m, prior[:0], value[:0])
    engine.search_end(ws[:0], 0, m, prior[:0], value[:0])
    assert engine.launches == before
    p = lambda t: ctypes.c_void_p(t.data_ptr())  # noqa: E731
    nb = ws.numel()
    out6 = [p(o[k]) for k in LEAF]
    vis = torch.empty((n, M.N_ACTIONS), dtype=torch.int32, device=dev)
    qq = torch.empty((n, M.N_ACTIONS), dtype=torch.float64, device=dev)
    rv = torch.empty(n, dtype=torch.float64, device=dev)
    nan, inf = float("nan"), float("inf")
    small = engine.search_workspace_bytes(n, m) - 1

    def begin(n=n, m=m, w=p(ws), b=nb, r=p(roots), ms=400):
        return lib.sb_search_begin(h, n, m, w, b, r, ms, *out6, None)

    def sim(n=n, m=m, w=p(ws), b=nb, pr=p(prior), v=p(value), c=1.0, f=0.0):
        return lib.sb_search_simulate(h, n, m, w, b, pr, v, c, f, *out6, None)

    def end(n=n, m=m, w=p(ws), b=nb, pr=p(prior), v=p(value), outs=(p(vis), p(qq), p(rv))):
        return lib.sb_search_end(h, n, m, w, b, pr, v, *outs, None)

    bad = [begin(n=-1), begin(m=0), begin(m=2**24 + 1), begin(w=None), begin(b=small), begin(w=ctypes.c_void_p(ws.data_ptr() + 8), b=nb - 8),
           begin(r=None), begin(ms=0), begin(ms=65536),
           sim(n=-1), sim(m=0), sim(w=None), sim(b=small), sim(c=-1.0), sim(c=nan), sim(c=inf), sim(f=nan), sim(f=-inf),
           sim(pr=None), sim(v=None),
           end(n=-1), end(m=0), end(w=None), end(b=small), end(pr=None), end(v=None), end(outs=(None, p(qq), p(rv))),
           end(outs=(p(vis), None, p(rv))), end(outs=(p(vis), p(qq), None))]
    assert all(rc == -1 for rc in bad), bad
    assert engine.launches == before
    with pytest.raises(_lib.SbError):
        engine.search_simulate(ws, n, m, prior, value, c_puct=-0.5)
    assert begin() == 0 and sim() == 0 and end() == 0 and engine.launches == before + 3
    torch.cuda.synchronize()


def test_source_names_no_batched_memcpy():
    pat = re.compile("cu(da)?Memcpy(3D)?" + "Batch" + "Async")
    hits = []
    for top in ("monsoon_b200", "include", "oracle", "tests", "tools", "."):
        base = os.path.join(ROOT, top)
        for dirpath, dirs, files in os.walk(base):
            dirs[:] = [] if top == "." else [d for d in dirs if not d.startswith(".") and d != "__pycache__"]
            for f in files:
                if f.endswith((".py", ".cu", ".cuh", ".h", ".c", ".cc", ".cpp", ".sh")) or f == "Makefile":
                    path = os.path.join(dirpath, f)
                    with open(path, errors="replace") as fh:
                        if pat.search(fh.read()):
                            hits.append(path)
    assert not hits, hits

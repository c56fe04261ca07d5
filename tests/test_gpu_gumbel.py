"""GPU: sb_search_simulate_gumbel / sb_search_end_gumbel and sb_ismcts_simulate_gumbel / sb_ismcts_end_gumbel (and
GumbelMCTS / InformationSetGumbelMCTS) against the plain-Python Gumbel model, call for call and byte for byte."""
import ctypes

import numpy as np
import pytest
import torch

import sb_gumbel_model as G
import sb_search_model as M
from monsoon_b200 import _lib
from monsoon_b200.search import GumbelMCTS, InformationSetGumbelMCTS, rollout_evaluator
from monsoon_b200.vec_env import StormboundVecEnv
from test_gpu_determinize import keys_for, mixed_roots
from test_gpu_ismcts import run_against_model as ismcts_puct_against_model, with_copies
from test_gpu_search import LEAF, compare_leaves, env_roots, host_eval, torch_eval
from test_gpu_search import run_against_model as search_puct_against_model

pytestmark = pytest.mark.gpu


def noise(n, seed, nans=False):
    g = (-np.log(-np.log(np.random.default_rng(seed).random((n, M.N_ACTIONS)) * (1 - 2e-12) + 1e-12))).astype(np.float32)
    if nans:
        g[::5, ::11] = np.nan
    return g


def evaluator(engine, rollout, nans):
    """(evaluate(o, want) -> device prior / value and the model's copies); nans: NaN entries in some rows' priors"""
    ev = rollout_evaluator(engine) if rollout else None
    dev = engine.device

    def evaluate(o, want):
        if not rollout:
            p, v = host_eval(want)
            if nans:
                p[::4, ::7] = np.nan
            return torch.from_numpy(p).to(dev), torch.from_numpy(v).to(dev), p, v
        p, v = ev(o, 0)
        pv = [M.rollout_eval(lf) for lf in want]
        wp, wv = np.stack([x[0] for x in pv]), np.array([x[1] for x in pv], dtype=np.float32)
        assert np.array_equal(p.cpu().numpy(), wp) and np.array_equal(v.cpu().numpy(), wv)
        return p, v, wp, wv

    return evaluate


def compare_end(r, ends):
    assert np.array_equal(r["action"].cpu().numpy(), np.array([e[0] for e in ends], dtype=np.int32))
    assert r["policy"].cpu().numpy().tobytes() == np.stack([e[1] for e in ends]).tobytes()
    assert np.array_equal(r["visits"].cpu().numpy(), np.stack([e[2] for e in ends]))
    assert np.array_equal(r["q"].cpu().numpy(), np.stack([e[3] for e in ends]), equal_nan=True)
    assert np.array_equal(r["root_value"].cpu().numpy(), np.array([e[4] for e in ends]), equal_nan=True)


def search_against_model(engine, roots, sims, mc, c_visit=50.0, c_scale=0.1, max_steps=400, rollout=False, max_nodes=None,
                         nans=False, seed=1):
    dev = engine.device
    n = roots.shape[0]
    m = max_nodes or sims + 1
    host = roots.cpu().numpy()
    models = [G.GumbelTreeModel(host[g], m, max_steps) for g in range(n)]
    hg = noise(n, seed, nans)
    gum = torch.from_numpy(hg).to(dev)
    ws = torch.empty(engine.search_workspace_bytes(n, m), dtype=torch.uint8, device=dev)
    evaluate = evaluator(engine, rollout, nans)
    kinds = {}
    o = engine.search_begin(ws, roots, m, max_steps)
    want = [t.begin() for t in models]
    compare_leaves(o, want, 0)
    prior, value, hp, hv = evaluate(o, want)
    for k in range(1, sims + 1):
        o = engine.search_simulate_gumbel(ws, n, m, prior, value, gum, k, sims, mc, c_visit, c_scale, out={key: o[key] for key in LEAF})
        want = [t.simulate(hp[g], hv[g], hg[g], k, sims, mc, c_visit, c_scale) for g, t in enumerate(models)]
        compare_leaves(o, want, k)
        for lf in want:
            kinds[lf[5]] = kinds.get(lf[5], 0) + 1
        prior, value, hp, hv = evaluate(o, want)
    r = engine.search_end_gumbel(ws, n, m, prior, value, gum, c_visit, c_scale)
    compare_end(r, [t.end(hp[g], hv[g], hg[g], c_visit, c_scale) for g, t in enumerate(models)])
    return kinds, models, r


def ismcts_against_model(engine, roots, sims, mc, c_visit=50.0, c_scale=0.1, max_steps=400, rollout=False, max_nodes=None,
                         nans=False, salt=1):
    dev = engine.device
    n = roots.shape[0]
    m = max_nodes or sims + 1
    keys = keys_for(n * (sims + 1), salt).to(dev)
    models = [G.ISGumbelTreeModel(m, max_steps) for _ in range(n)]
    hg = noise(n, salt, nans)
    gum = torch.from_numpy(hg).to(dev)
    ws = torch.empty(engine.ismcts_workspace_bytes(n, m), dtype=torch.uint8, device=dev)
    evaluate = evaluator(engine, rollout, nans)
    kinds = {}

    def world(k):
        det = engine.determinize(roots, keys[k * n:(k + 1) * n])
        return det, det.cpu().numpy()

    det, hd = world(0)
    o = engine.ismcts_begin(ws, det, m, max_steps)
    want = [t.begin(hd[g]) for g, t in enumerate(models)]
    compare_leaves(o, want, 0)
    prior, value, hp, hv = evaluate(o, want)
    for k in range(1, sims + 1):
        det, hd = world(k)
        o = engine.ismcts_simulate_gumbel(ws, det, m, prior, value, gum, k, sims, mc, c_visit, c_scale, out={key: o[key] for key in LEAF})
        want = [t.simulate(hd[g], hp[g], hv[g], hg[g], k, sims, mc, c_visit, c_scale) for g, t in enumerate(models)]
        compare_leaves(o, want, k)
        for lf in want:
            kinds[lf[5]] = kinds.get(lf[5], 0) + 1
        prior, value, hp, hv = evaluate(o, want)
    r = engine.ismcts_end_gumbel(ws, n, m, prior, value, gum, c_visit, c_scale)
    compare_end(r, [t.end(hp[g], hv[g], hg[g], c_visit, c_scale) for g, t in enumerate(models)])
    return kinds, models, r


@pytest.mark.parametrize("mc,sims,nans", [(16, 24, False), (16, 8, True), (2, 12, False), (1, 6, False), (156, 20, True)])
def test_search_matches_model(engine, oracle, mc, sims, nans):
    roots = mixed_roots(engine, 130, 40 + mc)
    kinds, models, r = search_against_model(engine, roots, sims, mc, nans=nans, seed=mc + sims)
    assert kinds.get(M.TERMINAL, 0) > 0 and kinds.get(M.EVAL, 0) > 0, kinds
    assert {t.nodes[0].seat for t in models} == {0, 1}
    act = r["action"].cpu().numpy()
    assert (act == G.NO_ACTION).any() and (act < M.N_ACTIONS).sum() > 100


def test_search_with_rollout_evaluator_small_max_steps_and_full_trees(engine, oracle):
    search_against_model(engine, env_roots(engine, 97, 7, plies=10), 16, 4, rollout=True)
    roots = env_roots(engine, 97, 5, plies=8)
    steps = roots[:, 12:14].contiguous().view(torch.int16).to(torch.int32)
    kinds, _m, _r = search_against_model(engine, roots, 16, 16, max_steps=int(steps.min()) + 2, c_visit=20.0, c_scale=0.5)
    assert kinds.get(M.TERMINAL, 0) > 97, kinds
    kinds, models, _r = search_against_model(engine, env_roots(engine, 65, 11), 8, 16, max_nodes=5)
    assert kinds.get(M.FULL, 0) >= 4 * 65 and all(len(t.nodes) <= 5 for t in models)


@pytest.mark.parametrize("mc,sims,nans", [(16, 16, False), (16, 6, True), (2, 10, False), (1, 5, False), (156, 12, False)])
def test_ismcts_matches_model(engine, oracle, mc, sims, nans):
    roots = with_copies(mixed_roots(engine, 100, 60 + mc))
    kinds, models, r = ismcts_against_model(engine, roots, sims, mc, nans=nans, salt=mc + 3 * sims)
    assert kinds.get(M.TERMINAL, 0) > 0 and kinds.get(M.EVAL, 0) > 0, kinds
    assert {t.nodes[0].seat for t in models} == {0, 1}


def test_ismcts_with_rollout_evaluator_small_max_steps_and_full_trees(engine, oracle):
    ismcts_against_model(engine, env_roots(engine, 65, 9, plies=10), 12, 4, rollout=True, salt=9)
    roots = env_roots(engine, 65, 5, plies=8)
    steps = roots[:, 12:14].contiguous().view(torch.int16).to(torch.int32)
    kinds, _m, _r = ismcts_against_model(engine, roots, 12, 16, max_steps=int(steps.min()) + 2, salt=5)
    assert kinds.get(M.TERMINAL, 0) > 65, kinds
    kinds, models, _r = ismcts_against_model(engine, env_roots(engine, 65, 11), 8, 16, max_nodes=5, salt=11)
    assert kinds.get(M.FULL, 0) >= 4 * 65 and all(len(t.nodes) <= 5 for t in models)


def test_puct_kernels_still_equal_their_models(engine, oracle):
    search_puct_against_model(engine, env_roots(engine, 65, 3), 12, 1.25, 0.0)
    ismcts_puct_against_model(engine, with_copies(mixed_roots(engine, 65, 21)), 12, 1.25, 0.0, salt=2)


def graph_equal(run_eager, run_graphed, engine):
    want = [t.clone() for t in run_eager()]
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        run_graphed()  # warm-up outside the capture
    torch.cuda.current_stream().wait_stream(side)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        outs = run_graphed()
    for t in outs:
        t.zero_()
    g.replay()
    torch.cuda.synchronize()
    for a, b in zip(outs, want):
        assert torch.equal(torch.nan_to_num(a, nan=7.0), torch.nan_to_num(b, nan=7.0))
    return outs


def test_launch_counts_and_cuda_graphs(engine):
    n, sims, dev = 300, 12, engine.device
    roots = env_roots(engine, n, 13)
    gum = torch.from_numpy(noise(n, 3)).to(dev)
    keys = keys_for(n * (sims + 1), 8).to(dev)
    a = GumbelMCTS(n, sims, engine=engine)
    before = engine.launches
    action, policy, visits, q, rv = a.run(roots, torch_eval, gum)
    torch.cuda.synchronize()
    assert engine.launches == before + sims + 2
    assert bool((visits.sum(1) == sims).all()) and bool((action < M.N_ACTIONS).all())
    assert bool(((policy.sum(1) - 1).abs() < 1e-5).all())
    b = InformationSetGumbelMCTS(n, sims, engine=engine)
    before = engine.launches
    b.run(roots, torch_eval, keys, gum)
    torch.cuda.synchronize()
    assert engine.launches == before + 2 * sims + 3
    ga = GumbelMCTS(n, sims, engine=engine)
    graph_equal(lambda: a.run(roots, torch_eval, gum), lambda: ga.run(roots, torch_eval, gum), engine)
    gb = InformationSetGumbelMCTS(n, sims, engine=engine)
    graph_equal(lambda: b.run(roots, torch_eval, keys, gum), lambda: gb.run(roots, torch_eval, keys, gum), engine)
    # default noise: reproducible from the seed, a new draw per call
    x, y = GumbelMCTS(n, sims, seed=5, engine=engine), GumbelMCTS(n, sims, seed=5, engine=engine)
    gx = x.default_gumbel()
    assert np.array_equal(gx, y.default_gumbel()) and not np.array_equal(gx, x.default_gumbel())
    r1 = [t.clone() for t in GumbelMCTS(n, sims, seed=9, engine=engine).run(roots, torch_eval)]
    r2 = GumbelMCTS(n, sims, seed=9, engine=engine).run(roots, torch_eval)
    assert all(torch.equal(torch.nan_to_num(u, nan=7.0), torch.nan_to_num(v, nan=7.0)) for u, v in zip(r1, r2))


def test_actions_play_in_a_vec_env(engine):
    n = 64
    for cls in (GumbelMCTS, InformationSetGumbelMCTS):
        env = StormboundVecEnv(n, seed=23, opponent="expert", seats=[g % 2 for g in range(n)], engine=engine)
        env.reset()
        mcts = cls(n, 8, seed=1, engine=engine)
        ev = rollout_evaluator(engine)
        for _ in range(12):
            action = mcts.run(env.states, ev)[0]
            assert bool((action < M.N_ACTIONS).all())
            assert bool(env.action_mask().gather(1, action.long().unsqueeze(1)).all())
            _o, _m, _r, _d, info = env.step(action)
            assert not bool((info["result"] == -4).any())


def test_empty_batch_and_rejected_arguments(engine):
    dev = engine.device
    lib, h = engine.lib, engine.h
    n, m, S = 8, 5, 4
    roots = env_roots(engine, n, 17, plies=1)
    prior = torch.full((n, M.N_ACTIONS), 0.1, dtype=torch.float32, device=dev)
    value = torch.zeros(n, dtype=torch.float32, device=dev)
    gum = torch.zeros((n, M.N_ACTIONS), dtype=torch.float32, device=dev)
    p = lambda t: ctypes.c_void_p(t.data_ptr())  # noqa: E731
    nan, inf = float("nan"), float("inf")
    act = torch.empty(n, dtype=torch.int32, device=dev)
    pol = torch.empty((n, M.N_ACTIONS), dtype=torch.float32, device=dev)
    vis = torch.empty((n, M.N_ACTIONS), dtype=torch.int32, device=dev)
    qq = torch.empty((n, M.N_ACTIONS), dtype=torch.float64, device=dev)
    rv = torch.empty(n, dtype=torch.float64, device=dev)
    for ism in (False, True):
        wsb = (engine.ismcts_workspace_bytes if ism else engine.search_workspace_bytes)(n, m)
        ws = torch.empty(wsb + 16, dtype=torch.uint8, device=dev)
        o = (engine.ismcts_begin if ism else engine.search_begin)(ws, roots, m)
        out6 = [p(o[k]) for k in LEAF]
        before = engine.launches
        empty = torch.empty((0, 512), dtype=torch.uint8, device=dev)
        if ism:
            engine.ismcts_simulate_gumbel(ws[:0], empty, m, prior[:0], value[:0], gum[:0], 1, S)
            engine.ismcts_end_gumbel(ws[:0], 0, m, prior[:0], value[:0], gum[:0])
        else:
            engine.search_simulate_gumbel(ws[:0], 0, m, prior[:0], value[:0], gum[:0], 1, S)
            engine.search_end_gumbel(ws[:0], 0, m, prior[:0], value[:0], gum[:0])
        assert engine.launches == before
        nb, small = ws.numel(), wsb - 1

        def sim(n=n, m=m, w=p(ws), b=nb, d=p(roots), pr=p(prior), v=p(value), g=p(gum), k=1, s=S, mc=16, cv=50.0, cs=0.1):
            if ism:
                return lib.sb_ismcts_simulate_gumbel(h, n, m, w, b, d, pr, v, g, k, s, mc, cv, cs, *out6, None)
            return lib.sb_search_simulate_gumbel(h, n, m, w, b, pr, v, g, k, s, mc, cv, cs, *out6, None)

        def end(n=n, m=m, w=p(ws), b=nb, pr=p(prior), v=p(value), g=p(gum), cv=50.0, cs=0.1, outs=(p(act), p(pol), p(vis), p(qq), p(rv))):
            f = lib.sb_ismcts_end_gumbel if ism else lib.sb_search_end_gumbel
            return f(h, n, m, w, b, pr, v, g, cv, cs, *outs, None)

        bad = [sim(n=-1), sim(m=0), sim(m=2**24 + 1), sim(w=None), sim(b=small), sim(w=ctypes.c_void_p(ws.data_ptr() + 8), b=nb - 8),
               sim(pr=None), sim(v=None), sim(g=None), sim(k=0), sim(k=S + 1), sim(s=0), sim(s=2**24 + 1, k=1), sim(mc=0), sim(mc=157),
               sim(cv=-1.0), sim(cv=nan), sim(cv=inf), sim(cs=-0.5), sim(cs=nan), sim(cs=inf),
               end(n=-1), end(m=0), end(w=None), end(b=small), end(pr=None), end(v=None), end(g=None), end(cv=-1.0), end(cs=nan),
               end(cs=inf)]
        bad += [end(outs=tuple(None if j == i else x for j, x in enumerate((p(act), p(pol), p(vis), p(qq), p(rv))))) for i in range(5)]
        if ism:
            bad.append(sim(d=None))
        assert all(rc == -1 for rc in bad), bad
        assert "gumbel" in lib.sb_last_error(h).decode()
        assert engine.launches == before
        with pytest.raises(_lib.SbError):
            engine.search_simulate_gumbel(ws, n, m, prior, value, gum, 0, S) if not ism else \
                engine.ismcts_simulate_gumbel(ws, roots, m, prior, value, gum, 0, S)
        assert sim() == 0 and end() == 0 and engine.launches == before + 2
        torch.cuda.synchronize()
        assert int(vis.sum()) == n and bool((act.cpu() < M.N_ACTIONS).all())

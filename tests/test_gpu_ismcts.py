"""GPU: sb_ismcts_begin / sb_ismcts_simulate / sb_ismcts_end (and InformationSetMCTS) against the plain-Python model, and
against the perfect-information search when every world is the root itself."""
import ctypes

import numpy as np
import pytest
import torch

import sb_determinize_model as D
import sb_ismcts_model as I
import sb_oracle as O
import sb_search_model as M
from monsoon_b200 import _lib
from monsoon_b200.search import InformationSetMCTS, rollout_evaluator, select_actions
from monsoon_b200.vec_env import StormboundVecEnv
from test_gpu_determinize import keys_for, mixed_roots
from test_gpu_search import LEAF, compare_leaves, env_roots, host_eval, torch_eval

pytestmark = pytest.mark.gpu


def with_copies(roots, every=7):
    """roots where, every `every` records, the mover's hand slot 1 holds a copy of slot 0's (card, cost, flags)"""
    out = roots.clone()
    host = out.cpu().numpy()
    for g in range(0, host.shape[0], every):
        p = 32 + 104 * int(host[g, 14] != 0)  # pl[local_order]
        if host[g, p + 8] >= 2:               # n_hand
            for off in (12, 16, 20):          # hand card, cost, flags (4 slots each)
                host[g, p + off + 1] = host[g, p + off]
    return torch.from_numpy(host).to(roots.device)


def run_against_model(engine, roots, sims, c_puct, fpu, max_steps=400, rollout=False, max_nodes=None, salt=1):
    """drive the three calls over fresh worlds and the model side by side: every call's leaf outputs and the read-out must be
    identical, and every leaf record must carry its call's key"""
    dev = engine.device
    n = roots.shape[0]
    m = max_nodes or sims + 1
    keys = keys_for(n * (sims + 1), salt).to(dev)
    models = [I.ISTreeModel(m, max_steps) for _ in range(n)]
    ws = torch.empty(engine.ismcts_workspace_bytes(n, m), dtype=torch.uint8, device=dev)
    ev = rollout_evaluator(engine) if rollout else None
    kinds = {}

    def world(k):
        det = engine.determinize(roots, keys[k * n:(k + 1) * n])
        return det, det.cpu().numpy()

    def check(o, want, k):
        compare_leaves(o, want, k)
        got = o["states"].cpu().numpy()
        assert got[:, :8].tobytes() == keys[k * n:(k + 1) * n].cpu().numpy().tobytes(), k  # the call's keys, never the root's
        for lf in want:
            kinds[lf[5]] = kinds.get(lf[5], 0) + 1

    def evaluate(o, want):
        if not rollout:
            p, v = host_eval(want)
            return torch.from_numpy(p).to(dev), torch.from_numpy(v).to(dev), p, v
        p, v = ev(o, 0)
        pv = [M.rollout_eval(lf) for lf in want]
        wp, wv = np.stack([x[0] for x in pv]), np.array([x[1] for x in pv], dtype=np.float32)
        assert np.array_equal(p.cpu().numpy(), wp) and np.array_equal(v.cpu().numpy(), wv)
        return p, v, wp, wv

    det, hd = world(0)
    o = engine.ismcts_begin(ws, det, m, max_steps)
    want = [t.begin(hd[g]) for g, t in enumerate(models)]
    check(o, want, 0)
    prior, value, hp, hv = evaluate(o, want)
    for k in range(1, sims + 1):
        det, hd = world(k)
        o = engine.ismcts_simulate(ws, det, m, prior, value, c_puct, fpu, out={key: o[key] for key in LEAF})
        want = [t.simulate(hd[g], hp[g], hv[g], c_puct, fpu) for g, t in enumerate(models)]
        check(o, want, k)
        prior, value, hp, hv = evaluate(o, want)
    r = engine.ismcts_end(ws, n, m, prior, value)
    ends = [t.end(hp[g], hv[g]) for g, t in enumerate(models)]
    assert np.array_equal(r["visits"].cpu().numpy(), np.stack([e[0] for e in ends]))
    assert np.array_equal(r["q"].cpu().numpy(), np.stack([e[1] for e in ends]), equal_nan=True)
    assert np.array_equal(r["root_value"].cpu().numpy(), np.array([e[2] for e in ends]), equal_nan=True)
    return kinds, models, r


def test_smallest_comparison(engine, oracle):
    roots = env_roots(engine, 24, 2, plies=3)
    kinds, models, r = run_against_model(engine, roots, 4, 1.25, 0.0)
    assert kinds.get(M.EVAL, 0) > 0 and bool((r["visits"].sum(1) == 4).all())


@pytest.mark.parametrize("c_puct,fpu,salt", [(1.25, 0.0, 3), (2.5, -0.3, 4)])
def test_ismcts_matches_model(engine, oracle, c_puct, fpu, salt):
    roots = with_copies(mixed_roots(engine, 258, 20 + salt))
    kinds, models, r = run_against_model(engine, roots, 32, c_puct, fpu, salt=salt)
    assert kinds.get(M.TERMINAL, 0) > 0 and kinds.get(M.EVAL, 0) > 0, kinds
    seats = {t.nodes[0].seat for t in models}
    assert seats == {0, 1}
    host = roots.cpu().numpy()
    assert sum(len(I.representatives(st)) < len(M.legal_ids(O.legal_mask(st.copy()))) for st in host) > 10  # copies in hand
    sums = r["visits"].sum(1).cpu().numpy()
    assert set(sums.tolist()) == {0, 32} and (sums == 32).sum() > 200  # 0: terminal roots


def test_ismcts_matches_model_with_rollout_evaluator(engine, oracle):
    roots = env_roots(engine, 129, 9, plies=10)
    kinds, _models, _r = run_against_model(engine, roots, 24, 1.25, 0.0, rollout=True, salt=9)
    assert kinds.get(M.EVAL, 0) > 0


def test_small_max_steps_and_full_trees(engine, oracle):
    roots = env_roots(engine, 129, 5, plies=8)
    steps = roots[:, 12:14].contiguous().view(torch.int16).to(torch.int32)
    kinds, models, _r = run_against_model(engine, roots, 24, 1.25, 0.0, max_steps=int(steps.min()) + 2, salt=5)
    assert kinds.get(M.TERMINAL, 0) > 129, kinds
    kinds, models, _r = run_against_model(engine, env_roots(engine, 65, 11), 8, 1.25, 0.0, max_nodes=5, salt=11)
    assert kinds.get(M.FULL, 0) >= 4 * 65 and all(len(t.nodes) <= 5 for t in models)


def test_fixed_world_equals_the_perfect_information_search(engine):
    """every world is the root itself (default decks: no card twice in a hand): leaves, visits, q and root value are
    sb_search_*'s"""
    n, sims, dev = 257, 32, engine.device
    roots = env_roots(engine, n, 15, plies=6)
    finished = roots[::16].clone()
    engine.rollout_random(finished)
    roots[::16] = finished
    m = sims + 1
    wa = torch.empty(engine.search_workspace_bytes(n, m), dtype=torch.uint8, device=dev)
    wb = torch.empty(engine.ismcts_workspace_bytes(n, m), dtype=torch.uint8, device=dev)
    a = engine.search_begin(wa, roots, m)
    b = engine.ismcts_begin(wb, roots, m)
    for k in range(sims + 1):
        for key in LEAF:
            assert torch.equal(a[key], b[key]), (k, key)
        prior, value = torch_eval(a, k)
        if k < sims:
            a = engine.search_simulate(wa, n, m, prior, value, 1.25, 0.0, out={key: a[key] for key in LEAF})
            b = engine.ismcts_simulate(wb, roots, m, prior, value, 1.25, 0.0, out={key: b[key] for key in LEAF})
    ra, rb = engine.search_end(wa, n, m, prior, value), engine.ismcts_end(wb, n, m, prior, value)
    assert torch.equal(ra["visits"], rb["visits"]) and torch.equal(ra["root_value"], rb["root_value"])
    assert torch.equal(torch.nan_to_num(ra["q"], nan=7.0), torch.nan_to_num(rb["q"], nan=7.0))
    assert int(rb["visits"].sum()) > n


def test_information_set_mcts_matches_the_model(engine, oracle):
    """the class: worlds from sb_determinize of the roots with the caller's simulation-major keys"""
    n, sims, dev = 40, 10, engine.device
    roots = env_roots(engine, n, 33, plies=7)
    keys = keys_for(n * (sims + 1), 77).to(dev)
    host, hk = roots.cpu().numpy(), keys.cpu().numpy().view(np.uint64)
    models = [I.ISTreeModel(sims + 1) for _ in range(n)]
    state = {}

    def evaluate(leaf, k):
        if k == 0:
            want = [t.begin(D.determinize(host[g], int(hk[g]))) for g, t in enumerate(models)]
        else:
            p, v = state["p"], state["v"]
            want = [t.simulate(D.determinize(host[g], int(hk[k * n + g])), p[g], v[g], 1.25, 0.0) for g, t in enumerate(models)]
        compare_leaves(leaf, want, k)
        state["p"], state["v"] = host_eval(want)
        return torch.from_numpy(state["p"]).to(dev), torch.from_numpy(state["v"]).to(dev)

    mcts = InformationSetMCTS(n, sims, engine=engine)
    before = engine.launches
    visits, q, rv = mcts.run(roots, evaluate, keys)
    torch.cuda.synchronize()
    assert engine.launches == before + 2 * sims + 3
    ends = [t.end(state["p"][g], state["v"][g]) for g, t in enumerate(models)]
    assert np.array_equal(visits.cpu().numpy(), np.stack([e[0] for e in ends]))
    assert np.array_equal(q.cpu().numpy(), np.stack([e[1] for e in ends]), equal_nan=True)
    assert np.array_equal(rv.cpu().numpy(), np.array([e[2] for e in ends]))


def test_launch_count_and_cuda_graph(engine):
    n, sims = 300, 16
    roots = env_roots(engine, n, 13)
    keys = keys_for(n * (sims + 1), 8).to(engine.device)
    eager = InformationSetMCTS(n, sims, engine=engine)
    before = engine.launches
    visits, q, root_value = eager.run(roots, torch_eval, keys)
    torch.cuda.synchronize()
    assert engine.launches == before + 2 * sims + 3
    assert bool((visits.sum(1) == sims).all()) and bool((root_value.abs() <= 1).all())
    want = [t.clone() for t in (visits, q, root_value)]
    graphed = InformationSetMCTS(n, sims, engine=engine)
    static_roots, static_keys = roots.clone(), keys.clone()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        graphed.run(static_roots, torch_eval, static_keys)  # warm-up outside the capture
    torch.cuda.current_stream().wait_stream(side)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        outs = graphed.run(static_roots, torch_eval, static_keys)
    for t in outs:
        t.zero_()
    g.replay()
    torch.cuda.synchronize()
    nan = lambda t: torch.nan_to_num(t, nan=7.0)  # noqa: E731
    assert torch.equal(outs[0], want[0]) and torch.equal(nan(outs[1]), nan(want[1])) and torch.equal(outs[2], want[2])
    static_roots.copy_(env_roots(engine, n, 14))
    static_keys.copy_(keys_for(n * (sims + 1), 9).to(engine.device))
    g.replay()
    again = eager.run(static_roots.clone(), torch_eval, static_keys.clone())
    torch.cuda.synchronize()
    assert torch.equal(outs[0], again[0]) and torch.equal(outs[2], again[2])
    # default keys: reproducible from the seed, a new set per call
    a, b = InformationSetMCTS(n, sims, seed=5, engine=engine), InformationSetMCTS(n, sims, seed=5, engine=engine)
    ka, kb = a.default_keys(), b.default_keys()
    assert np.array_equal(ka, kb) and not np.array_equal(ka, a.default_keys()) and len(set(ka.tolist())) == n * (sims + 1)


def test_ismcts_plays_in_a_vec_env(engine):
    n = 64
    env = StormboundVecEnv(n, seed=23, opponent="expert", seats=[g % 2 for g in range(n)], engine=engine)
    env.reset()
    mcts = InformationSetMCTS(n, 8, seed=1, engine=engine)
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
    ws = torch.empty(engine.ismcts_workspace_bytes(n, m) + 16, dtype=torch.uint8, device=dev)
    o = engine.ismcts_begin(ws, roots, m)
    prior = torch.full((n, M.N_ACTIONS), 0.1, dtype=torch.float32, device=dev)
    value = torch.zeros(n, dtype=torch.float32, device=dev)
    before = engine.launches
    empty = torch.empty((0, 512), dtype=torch.uint8, device=dev)
    engine.ismcts_begin(ws[:0], empty, m)
    engine.ismcts_simulate(ws[:0], empty, m, prior[:0], value[:0])
    engine.ismcts_end(ws[:0], 0, m, prior[:0], value[:0])
    assert engine.launches == before
    p = lambda t: ctypes.c_void_p(t.data_ptr())  # noqa: E731
    nb = ws.numel()
    out6 = [p(o[k]) for k in LEAF]
    vis = torch.empty((n, M.N_ACTIONS), dtype=torch.int32, device=dev)
    qq = torch.empty((n, M.N_ACTIONS), dtype=torch.float64, device=dev)
    rv = torch.empty(n, dtype=torch.float64, device=dev)
    nan, inf = float("nan"), float("inf")
    small = engine.ismcts_workspace_bytes(n, m) - 1

    def begin(n=n, m=m, w=p(ws), b=nb, d=p(roots), ms=400):
        return lib.sb_ismcts_begin(h, n, m, w, b, d, ms, *out6, None)

    def sim(n=n, m=m, w=p(ws), b=nb, d=p(roots), pr=p(prior), v=p(value), c=1.0, f=0.0):
        return lib.sb_ismcts_simulate(h, n, m, w, b, d, pr, v, c, f, *out6, None)

    def end(n=n, m=m, w=p(ws), b=nb, pr=p(prior), v=p(value), outs=(p(vis), p(qq), p(rv))):
        return lib.sb_ismcts_end(h, n, m, w, b, pr, v, *outs, None)

    bad = [begin(n=-1), begin(m=0), begin(m=2**24 + 1), begin(w=None), begin(b=small), begin(w=ctypes.c_void_p(ws.data_ptr() + 8), b=nb - 8),
           begin(d=None), begin(ms=0), begin(ms=65536),
           sim(n=-1), sim(m=0), sim(w=None), sim(b=small), sim(d=None), sim(c=-1.0), sim(c=nan), sim(c=inf), sim(f=nan), sim(f=-inf),
           sim(pr=None), sim(v=None),
           end(n=-1), end(m=0), end(w=None), end(b=small), end(pr=None), end(v=None), end(outs=(None, p(qq), p(rv))),
           end(outs=(p(vis), None, p(rv))), end(outs=(p(vis), p(qq), None))]
    assert all(rc == -1 for rc in bad), bad
    assert "sb_ismcts" in lib.sb_last_error(h).decode()
    assert engine.launches == before
    with pytest.raises(_lib.SbError):
        engine.ismcts_simulate(ws, roots, m, prior, value, c_puct=-0.5)
    assert begin() == 0 and sim() == 0 and end() == 0 and engine.launches == before + 3
    torch.cuda.synchronize()
    assert int(vis.sum()) == n

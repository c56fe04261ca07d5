"""GPU: sb_search_advance / sb_ismcts_advance (and BatchedMCTS / InformationSetMCTS with reuse_nodes) against the
plain-Python statement of tree reuse (tests/sb_reuse_model.py): every advance's leaf outputs and kept counts, every simulate
leaf after it and every read-out must equal the model's byte for byte."""
import ctypes

import numpy as np
import pytest
import torch

import sb_determinize_model as D
import sb_ismcts_model as I
import sb_oracle as O
import sb_reuse_model as R
import sb_search_model as M
from monsoon_b200 import _lib
from monsoon_b200.search import BatchedMCTS, InformationSetMCTS, rollout_evaluator, select_actions
from monsoon_b200.vec_env import StormboundVecEnv
from test_gpu_determinize import keys_for, mixed_roots
from test_gpu_search import LEAF, compare_leaves, env_roots, host_eval, torch_eval

pytestmark = pytest.mark.gpu


class Evaluator:
    """the hashed-prior evaluator, or rollout_evaluator checked against the model's rollouts"""

    def __init__(self, engine, rollout):
        self.dev, self.ev = engine.device, rollout_evaluator(engine) if rollout else None

    def __call__(self, o, want):
        if self.ev is None:
            p, v = host_eval(want)
            return torch.from_numpy(p).to(self.dev), torch.from_numpy(v).to(self.dev), p, v
        p, v = self.ev(o, 0)
        pv = [M.rollout_eval(lf) for lf in want]
        wp, wv = np.stack([x[0] for x in pv]), np.array([x[1] for x in pv], dtype=np.float32)
        assert np.array_equal(p.cpu().numpy(), wp) and np.array_equal(v.cpu().numpy(), wv)
        return p, v, wp, wv


def compare_end(r, ends):
    assert np.array_equal(r["visits"].cpu().numpy(), np.stack([e[0] for e in ends]))
    assert np.array_equal(r["q"].cpu().numpy(), np.stack([e[1] for e in ends]), equal_nan=True)
    assert np.array_equal(r["root_value"].cpu().numpy(), np.array([e[2] for e in ends]), equal_nan=True)


class SearchPair:
    """two workspaces on the device and n TreeModels, searched side by side"""

    def __init__(self, engine, n, sims, max_nodes, max_steps=400, rollout=False):
        self.e, self.n, self.sims, self.m, self.max_steps = engine, n, sims, max_nodes, max_steps
        nb = engine.search_workspace_bytes(n, max_nodes)
        self.ws = [torch.empty(nb, dtype=torch.uint8, device=engine.device) for _ in range(2)]
        self.models = [None] * n
        self.ev = Evaluator(engine, rollout)

    def search(self, roots, keep=None):
        """one search from roots: a begin (keep None) or an advance; returns (kept, visits)"""
        e, n, m = self.e, self.n, self.m
        host = roots.cpu().numpy()
        if keep is None:
            o = e.search_begin(self.ws[0], roots, m, self.max_steps)
            self.models = [M.TreeModel(host[g], m, self.max_steps) for g in range(n)]
            want = [t.begin() for t in self.models]
            kept = np.zeros(n, dtype=np.int32)
        else:
            o = e.search_advance(self.ws[0], self.ws[1], roots, m, keep, self.max_steps)
            self.ws.reverse()
            res = [R.search_advance(self.models[g], host[g], m, keep, self.max_steps) for g in range(n)]
            self.models = [x[0] for x in res]
            want = [x[1] for x in res]
            kept = np.array([x[2] for x in res], dtype=np.int32)
            assert np.array_equal(o["kept"].cpu().numpy(), kept)
        compare_leaves(o, want, "advance")
        prior, value, hp, hv = self.ev(o, want)
        for k in range(1, self.sims + 1):
            o = e.search_simulate(self.ws[0], n, m, prior, value, 1.25, 0.0, out={key: o[key] for key in LEAF})
            want = [t.simulate(hp[g], hv[g], 1.25, 0.0) for g, t in enumerate(self.models)]
            compare_leaves(o, want, k)
            prior, value, hp, hv = self.ev(o, want)
        r = e.search_end(self.ws[0], n, m, prior, value)
        compare_end(r, [t.end(hp[g], hv[g]) for g, t in enumerate(self.models)])
        return kept, r["visits"]


def stepped(engine, roots, a):
    """roots with sb_step(root, a) where a is an action id (the roots with visits), the others unchanged"""
    nxt = roots.clone()
    idx = torch.nonzero(a < 156).squeeze(1)
    sub = roots[idx].contiguous()
    engine.step(sub, a[idx].to(torch.uint8).contiguous())
    nxt[idx] = sub
    return nxt


def next_roots(engine, roots, visits, other):
    """a mix of what an advance meets: the child of the most visited action (most trees), the same root again, an unrelated
    record and a finished game"""
    nxt = stepped(engine, roots, select_actions(visits))
    nxt[1::7] = roots[1::7]
    nxt[2::7] = other[2::7]
    done = nxt[3::11].clone()
    engine.rollout_random(done)
    nxt[3::11] = done
    return nxt


@pytest.mark.parametrize("keep,rollout", [(1, False), (6, False), (10**3, False), (10**3, True)])
def test_search_advance_matches_model(engine, oracle, keep, rollout):
    n, sims = 129 if rollout else 258, 16
    keep = min(keep, sims + 1 + 24)
    pair = SearchPair(engine, n, sims, sims + 1 + 24, rollout=rollout)
    roots = mixed_roots(engine, n, 41)
    _kept, visits = pair.search(roots)
    for move in range(3):
        roots = next_roots(engine, roots, visits, mixed_roots(engine, n, 50 + move))
        kept, visits = pair.search(roots, keep)
        assert (kept > 0).sum() > n // 2 and (kept == 0).any(), kept
        assert kept.max() == keep or keep > 2 * sims


def test_search_advance_small_max_steps_and_full_trees(engine, oracle):
    n, sims = 129, 12
    roots = env_roots(engine, n, 5, plies=8)
    steps = roots[:, 12:14].contiguous().view(torch.int16).to(torch.int32)
    pair = SearchPair(engine, n, sims, sims + 1, max_steps=int(steps.min()) + 3)  # no room to spare: trees fill
    _kept, visits = pair.search(roots)
    roots = next_roots(engine, roots, visits, env_roots(engine, n, 6))
    kept, _visits = pair.search(roots, sims + 1)
    assert (kept > 0).any()
    # another max_steps than the source's: everything starts fresh
    pair.max_steps += 1
    kept, _visits = pair.search(roots, sims + 1)
    assert not kept.any()


class ISPair:
    """two information-set workspaces on the device and n ISTreeModels, with worlds from sb_determinize under caller keys"""

    def __init__(self, engine, n, sims, max_nodes, rollout=False):
        self.e, self.n, self.sims, self.m = engine, n, sims, max_nodes
        nb = engine.ismcts_workspace_bytes(n, max_nodes)
        self.ws = [torch.empty(nb, dtype=torch.uint8, device=engine.device) for _ in range(2)]
        self.models = [None] * n
        self.ev = Evaluator(engine, rollout)
        self.salt = 0

    def search(self, roots, played=None, keep=None):
        e, n, m = self.e, self.n, self.m
        self.salt += 1
        keys = keys_for(n * (self.sims + 1), 1000 + self.salt).to(e.device)
        hk = keys.cpu().numpy().view(np.uint64)
        host = roots.cpu().numpy()
        det = e.determinize(roots, keys[:n])
        worlds = [D.determinize(host[g], int(hk[g])) for g in range(n)]
        if keep is None:
            o = e.ismcts_begin(self.ws[0], det, m)
            self.models = [I.ISTreeModel(m) for _ in range(n)]
            want = [t.begin(worlds[g]) for g, t in enumerate(self.models)]
            kept = np.zeros(n, dtype=np.int32)
        else:
            o = e.ismcts_advance(self.ws[0], self.ws[1], det, played, m, keep)
            self.ws.reverse()
            pl = played.cpu().numpy()
            res = [R.ismcts_advance(self.models[g], worlds[g], int(pl[g]), m, keep) for g in range(n)]
            self.models = [x[0] for x in res]
            want = [x[1] for x in res]
            kept = np.array([x[2] for x in res], dtype=np.int32)
            assert np.array_equal(o["kept"].cpu().numpy(), kept)
        compare_leaves(o, want, "advance")
        prior, value, hp, hv = self.ev(o, want)
        for k in range(1, self.sims + 1):
            det = e.determinize(roots, keys[k * n:(k + 1) * n])
            o = e.ismcts_simulate(self.ws[0], det, m, prior, value, 1.25, 0.0, out={key: o[key] for key in LEAF})
            want = [t.simulate(D.determinize(host[g], int(hk[k * n + g])), hp[g], hv[g], 1.25, 0.0) for g, t in enumerate(self.models)]
            compare_leaves(o, want, k)
            prior, value, hp, hv = self.ev(o, want)
        r = e.ismcts_end(self.ws[0], n, m, prior, value)
        compare_end(r, [t.end(hp[g], hv[g]) for g, t in enumerate(self.models)])
        return kept, r["visits"]


@pytest.mark.parametrize("keep,rollout", [(1, False), (7, False), (10**3, True)])
def test_ismcts_advance_matches_model(engine, oracle, keep, rollout):
    n, sims = 129 if rollout else 258, 16
    keep = min(keep, sims + 1 + 24)
    pair = ISPair(engine, n, sims, sims + 1 + 24, rollout=rollout)
    roots = mixed_roots(engine, n, 61)
    _kept, visits = pair.search(roots)
    for move in range(3):
        a = select_actions(visits)
        nxt = stepped(engine, roots, a)
        played = torch.where(a < 156, a, -1).to(torch.int32)
        played[1::9] = -1                       # nothing played
        played[2::9] = 155                      # PASS: usually the other seat's turn
        played[4::9] = 200                      # not an action id
        played[5::9] = torch.remainder(played[5::9] + 1, 156)  # another action than the one that led here
        roots = nxt
        kept, visits = pair.search(roots, played, keep)
        assert (kept > 0).sum() > n // 5 and (kept == 0).sum() >= n // 3, kept


def episode_models(engine, env, mcts, moves, keep_check):
    """play `moves` decisions of BatchedMCTS(reuse_nodes) in env, checking every call of every move against the model"""
    n, m, keep = mcts.n, mcts.max_nodes, mcts.reuse_nodes + 1
    models, state, stats = [None] * n, {}, []

    def evaluate(leaf, k):
        if k == 0:
            host = state["roots"]
            if state.get("first", True):
                models[:] = [M.TreeModel(host[g], m) for g in range(n)]
                want = [t.begin() for t in models]
                kept = np.zeros(n, dtype=np.int32)
                state["first"] = False
            else:
                res = [R.search_advance(models[g], host[g], m, keep) for g in range(n)]
                models[:] = [x[0] for x in res]
                want, kept = [x[1] for x in res], np.array([x[2] for x in res], dtype=np.int32)
            assert np.array_equal(mcts.kept.cpu().numpy(), kept)
            stats.append(kept)
        else:
            want = [t.simulate(state["p"][g], state["v"][g], mcts.c_puct, mcts.fpu) for g, t in enumerate(models)]
        compare_leaves(leaf, want, k)
        state["p"], state["v"] = host_eval(want)
        return torch.from_numpy(state["p"]).to(engine.device), torch.from_numpy(state["v"]).to(engine.device)

    for _ in range(moves):
        state["roots"] = env.states.cpu().numpy()
        before = engine.launches
        visits, q, rv = mcts.run(env.states, evaluate)
        torch.cuda.synchronize()
        assert engine.launches == before + mcts.num_simulations + 2
        compare_end({"visits": visits, "q": q, "root_value": rv}, [t.end(state["p"][g], state["v"][g]) for g, t in enumerate(models)])
        env.step(select_actions(visits))
    keep_check(np.stack(stats))


@pytest.mark.parametrize("opponent", [None, "random", "expert"])
def test_batched_mcts_reuse_over_episodes(engine, oracle, opponent):
    n, sims = 64, 8
    env = StormboundVecEnv(n, seed=71, opponent=opponent, seats=None if opponent is None else [g % 2 for g in range(n)], engine=engine)
    env.reset()
    mcts = BatchedMCTS(n, sims, reuse_nodes=sims, engine=engine)
    assert mcts.max_nodes == 2 * sims + 1

    def check(kept):
        assert not kept[0].any() and (kept[1:] > 0).mean() > 0.3 and kept.max() <= sims + 1, (kept > 0).mean(1)

    episode_models(engine, env, mcts, 30, check)


def test_information_set_mcts_reuse_over_episodes(engine, oracle):
    n, sims = 64, 8
    env = StormboundVecEnv(n, seed=73, opponent="expert", seats=[g % 2 for g in range(n)], engine=engine)
    env.reset()
    mcts = InformationSetMCTS(n, sims, reuse_nodes=sims, engine=engine)
    m, keep = mcts.max_nodes, sims + 1
    models, state, stats = [None] * n, {}, []
    played = None
    prev = None
    for move in range(30):
        roots = env.states
        host = roots.cpu().numpy()
        keys = keys_for(n * (sims + 1), 500 + move).to(engine.device)
        hk = keys.cpu().numpy().view(np.uint64)
        if played is None:
            eff = None
        else:
            pl = played.cpu().numpy()
            eff = [int(pl[g]) if 0 <= pl[g] < 156 and O.step(prev[g].copy(), int(pl[g])).tobytes() == host[g].tobytes() else -1
                   for g in range(n)]

        def evaluate(leaf, k):
            if k == 0:
                worlds = [D.determinize(host[g], int(hk[g])) for g in range(n)]
                if eff is None:
                    models[:] = [I.ISTreeModel(m) for _ in range(n)]
                    want = [t.begin(worlds[g]) for g, t in enumerate(models)]
                    kept = np.zeros(n, dtype=np.int32)
                else:
                    res = [R.ismcts_advance(models[g], worlds[g], eff[g], m, keep) for g in range(n)]
                    models[:] = [x[0] for x in res]
                    want, kept = [x[1] for x in res], np.array([x[2] for x in res], dtype=np.int32)
                assert np.array_equal(mcts.kept.cpu().numpy(), kept)
                stats.append(kept)
            else:
                want = [t.simulate(D.determinize(host[g], int(hk[k * n + g])), state["p"][g], state["v"][g], 1.25, 0.0)
                        for g, t in enumerate(models)]
            compare_leaves(leaf, want, k)
            state["p"], state["v"] = host_eval(want)
            return torch.from_numpy(state["p"]).to(engine.device), torch.from_numpy(state["v"]).to(engine.device)

        before = engine.launches
        visits, q, rv = mcts.run(roots, evaluate, keys, played=played)
        torch.cuda.synchronize()
        assert engine.launches == before + 2 * sims + (3 if played is None else 4)
        compare_end({"visits": visits, "q": q, "root_value": rv}, [t.end(state["p"][g], state["v"][g]) for g, t in enumerate(models)])
        prev = host.copy()
        played = select_actions(visits)
        env.step(played)
    kept = np.stack(stats)
    assert not kept[0].any() and (kept[1:] > 0).mean() > 0.2 and kept.max() <= sims + 1, (kept > 0).mean(1)


def test_no_reuse_is_todays_search(engine):
    """reuse_nodes = 0: one workspace, begin, S + 2 launches and the outputs of the plain begin / simulate / end calls"""
    n, sims = 200, 12
    roots = env_roots(engine, n, 19)
    mcts = BatchedMCTS(n, sims, engine=engine)
    assert mcts.max_nodes == sims + 1 and mcts.ws_next is None
    for _ in range(2):
        before = engine.launches
        visits, q, rv = [t.clone() for t in mcts.run(roots, torch_eval)]
        assert engine.launches == before + sims + 2
        ws = torch.empty_like(mcts.ws)
        o = engine.search_begin(ws, roots, sims + 1)
        prior, value = torch_eval(o, 0)
        for k in range(1, sims + 1):
            o = engine.search_simulate(ws, n, sims + 1, prior, value, out={key: o[key] for key in LEAF})
            prior, value = torch_eval(o, k)
        r = engine.search_end(ws, n, sims + 1, prior, value)
        assert torch.equal(visits, r["visits"]) and torch.equal(rv, r["root_value"]) and torch.equal(q.nan_to_num(7.0), r["q"].nan_to_num(7.0))
    keys = keys_for(n * (sims + 1), 3).to(engine.device)
    a, b = InformationSetMCTS(n, sims, engine=engine), InformationSetMCTS(n, sims, engine=engine)
    before = engine.launches
    va = a.run(roots, torch_eval, keys)[0].clone()
    vb = b.run(roots, torch_eval, keys, played=torch.zeros(n, dtype=torch.int64, device=engine.device))[0]
    assert engine.launches == before + 2 * (2 * sims + 3) and torch.equal(va, vb)


def test_reset_tree_launch_counts_and_cuda_graph(engine):
    n, sims = 300, 8
    env = StormboundVecEnv(n, seed=29, opponent="random", seats=[g % 2 for g in range(n)], engine=engine)
    env.reset()
    eager = BatchedMCTS(n, sims, reuse_nodes=sims, engine=engine)
    graphed = BatchedMCTS(n, sims, reuse_nodes=sims, engine=engine)
    v0 = eager.run(env.states, torch_eval)[0]
    graphed.run(env.states, torch_eval)
    env.step(select_actions(v0))
    static_roots = env.states.clone()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        outs = graphed.run(static_roots, torch_eval)  # an advancing run, captured: it reads the trees the run above finished
    before = engine.launches
    want = [t.clone() for t in eager.run(env.states, torch_eval)]
    assert engine.launches == before + sims + 2 and bool((eager.kept > 0).any())
    for t in outs:
        t.zero_()
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(outs[0], want[0]) and torch.equal(outs[2], want[2]) and torch.equal(graphed.kept, eager.kept)
    assert torch.equal(outs[1].nan_to_num(7.0), want[1].nan_to_num(7.0))
    # a second replay advances from the workspace the first one consumed: every tree starts fresh, as after reset_tree
    g.replay()
    eager.reset_tree()
    fresh = [t.clone() for t in eager.run(env.states, torch_eval)]
    torch.cuda.synchronize()
    assert not bool(eager.kept.any()) and not bool(graphed.kept.any())
    assert torch.equal(outs[0], fresh[0]) and torch.equal(outs[2], fresh[2])
    # InformationSetMCTS with caller keys: a reusing run is 2S + 4 launches and capturable
    keys = keys_for(n * (sims + 1), 4).to(engine.device)
    ie, ig = InformationSetMCTS(n, sims, reuse_nodes=sims, engine=engine), InformationSetMCTS(n, sims, reuse_nodes=sims, engine=engine)
    r0 = env.states.clone()
    p0 = select_actions(ie.run(r0, torch_eval, keys)[0]).clone()
    ig.run(r0, torch_eval, keys)
    env.step(p0)
    r1, k1 = env.states.clone(), keys_for(n * (sims + 1), 5).to(engine.device)
    g2 = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g2):
        outs = ig.run(r1, torch_eval, k1, played=p0)
    before = engine.launches
    want = [t.clone() for t in ie.run(r1, torch_eval, k1, played=p0)]
    assert engine.launches == before + 2 * sims + 4 and bool((ie.kept > 0).any())
    g2.replay()
    torch.cuda.synchronize()
    assert torch.equal(outs[0], want[0]) and torch.equal(outs[2], want[2]) and torch.equal(ig.kept, ie.kept)


def test_empty_batch_and_rejected_arguments(engine):
    dev = engine.device
    lib, h = engine.lib, engine.h
    n, m = 8, 5
    roots = env_roots(engine, n, 17, plies=1)
    p = lambda t: ctypes.c_void_p(t.data_ptr()) if t is not None else None  # noqa: E731
    kept = torch.empty(n, dtype=torch.int32, device=dev)
    played = torch.zeros(n, dtype=torch.int32, device=dev)
    for kind in ("search", "ismcts"):
        nb = engine.search_workspace_bytes(n, m) if kind == "search" else engine.ismcts_workspace_bytes(n, m)
        wa = torch.empty(nb + 16, dtype=torch.uint8, device=dev)
        wb = torch.empty(nb + 16, dtype=torch.uint8, device=dev)
        big = torch.empty(2 * nb, dtype=torch.uint8, device=dev)
        begin = engine.search_begin if kind == "search" else engine.ismcts_begin
        o = begin(wa, roots, m)
        out6 = [p(o[k]) for k in LEAF]

        def adv(n=n, m=m, src=p(wa), dst=p(wb), b=nb, r=p(roots), ms=400, keep=m, pl=p(played), kd=p(kept)):
            if kind == "search":
                return lib.sb_search_advance(h, n, m, src, dst, b, r, ms, keep, kd, *out6, None)
            return lib.sb_ismcts_advance(h, n, m, src, dst, b, r, pl, ms, keep, kd, *out6, None)

        begin(big[:nb], roots, m)  # every workspace an advance reads here is one the library wrote
        before = engine.launches
        assert adv(n=0, src=None, dst=None, b=0, r=None, pl=None) == 0 and engine.launches == before
        bad = [adv(n=-1), adv(m=0), adv(m=2**24 + 1), adv(keep=0), adv(keep=m + 1), adv(src=None), adv(dst=None),
               adv(src=ctypes.c_void_p(wa.data_ptr() + 8)), adv(dst=ctypes.c_void_p(wb.data_ptr() + 8)), adv(b=nb - 1),
               adv(src=p(wa), dst=p(wa)), adv(src=p(big), dst=ctypes.c_void_p(big.data_ptr() + nb - 16)),
               adv(src=ctypes.c_void_p(big.data_ptr() + nb - 16), dst=p(big)), adv(r=None), adv(ms=0), adv(ms=65536)]
        if kind == "ismcts":
            bad.append(adv(pl=None))
        assert all(rc == -1 for rc in bad), (kind, bad)
        assert ("sb_%s_advance" % kind) in lib.sb_last_error(h).decode()
        assert engine.launches == before
        with pytest.raises(_lib.SbError):
            if kind == "search":
                engine.search_advance(wa[:nb], wb[:nb], roots, m, 0)
            else:
                engine.ismcts_advance(wa[:nb], wb[:nb], roots, played, m, 0)
        # the two adjacent halves of one buffer do not overlap; kept and the leaf outputs are nullable
        assert adv(src=p(big), dst=ctypes.c_void_p(big.data_ptr() + nb), kd=None) == 0 and engine.launches == before + 1
        empty = torch.empty((0, 512), dtype=torch.uint8, device=dev)
        if kind == "search":
            engine.search_advance(wa[:0], wb[:0], empty, m, 1)
        else:
            engine.ismcts_advance(wa[:0], wb[:0], empty, played[:0], m, 1)
        assert engine.launches == before + 1
        torch.cuda.synchronize()

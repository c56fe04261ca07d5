"""GPU: sb_search_simulate_batch / sb_search_end_batch (and BatchedMCTS with leaves_per_call) against the plain-Python
statement of several leaves per tree per call (tests/sb_search_batch_model.py): every slot's leaf outputs of every call and
every read-out must equal the model's byte for byte."""
import ctypes

import numpy as np
import pytest
import torch

import sb_reuse_model as R
import sb_search_batch_model as B
import sb_search_model as M
from monsoon_b200 import _lib
from monsoon_b200.search import BatchedMCTS
from test_gpu_determinize import mixed_roots
from test_gpu_reuse import Evaluator, compare_end, next_roots
from test_gpu_search import LEAF, compare_leaves, env_roots, host_eval, torch_eval

pytestmark = pytest.mark.gpu


def virtual_visits(engine, ws, n, m, L):
    """the V arrays of the n trees' tails (i32[n, max_nodes])"""
    pre = engine.search_workspace_bytes(n, m)
    tail = (engine.search_batch_workspace_bytes(n, m, L) - pre) // n
    t = ws[pre:pre + n * tail].view(n, tail)[:, 8 * L:8 * L + 4 * m].contiguous()
    return t.view(torch.int32).cpu().numpy()


def slot0(n, L, p, v, hp, hv, dev):
    """batch inputs whose slot 0 holds the roots' evaluation (the other slots are not read by the first call)"""
    bp, bv = torch.zeros((n * L, M.N_ACTIONS), dtype=torch.float32, device=dev), torch.zeros(n * L, dtype=torch.float32, device=dev)
    bp.view(n, L, -1)[:, 0] = p
    bv.view(n, L)[:, 0] = v
    hbp, hbv = np.zeros((n * L, M.N_ACTIONS), np.float32), np.zeros(n * L, np.float32)
    hbp.reshape(n, L, -1)[:, 0], hbv.reshape(n, L)[:, 0] = hp, hv
    return bp, bv, hbp, hbv


def run_batch_against_model(engine, roots, L, vl, calls, c_puct=1.25, fpu=0.0, max_steps=400, rollout=False, max_nodes=None):
    """begin, `calls` batch calls and the batch end, with the models side by side; returns (slot kind counts, models)"""
    dev, n = engine.device, roots.shape[0]
    m = max_nodes or 1 + calls * L
    host = roots.cpu().numpy()
    models = [B.BatchTreeModel(host[g], m, L, max_steps) for g in range(n)]
    ws = torch.empty(engine.search_batch_workspace_bytes(n, m, L), dtype=torch.uint8, device=dev)
    ev = Evaluator(engine, rollout)
    o = engine.search_begin(ws, roots, m, max_steps)
    want = [t.begin() for t in models]
    compare_leaves(o, want, 0)
    prior, value, hp, hv = slot0(n, L, *ev(o, want), dev)
    kinds = {}
    for k in range(1, calls + 1):
        before = engine.launches
        o = engine.search_simulate_batch(ws, n, m, L, prior, value, c_puct, fpu, vl)
        assert engine.launches == before + 2
        want = [lf for g, t in enumerate(models) for lf in t.simulate_batch(hp[g * L:(g + 1) * L], hv[g * L:(g + 1) * L], c_puct, fpu, vl)]
        compare_leaves(o, want, k)
        assert not virtual_visits(engine, ws, n, m, L).any(), "virtual visits are zero when a call returns"
        for lf in want:
            kinds[lf[5]] = kinds.get(lf[5], 0) + 1
        prior, value, hp, hv = ev(o, want)
    before = engine.launches
    r = engine.search_end_batch(ws, n, m, L, prior, value)
    assert engine.launches == before + 1
    compare_end(r, [t.end_batch(hp[g * L:(g + 1) * L], hv[g * L:(g + 1) * L]) for g, t in enumerate(models)])
    return kinds, models


@pytest.mark.parametrize("n,L,vl,calls,rollout", [(63, 1, 1.0, 12, False), (64, 2, 0.0, 8, False), (65, 7, 3.5, 4, True),
                                                   (65, 16, 1.0, 4, False), (1, 64, 1.0, 3, False), (63, 64, 3.5, 2, False),
                                                   (4099, 2, 1.0, 3, False)])
def test_batch_matches_model(engine, oracle, n, L, vl, calls, rollout):
    roots = mixed_roots(engine, n, 70 + L) if n > 1 else env_roots(engine, n, 70 + L)
    kinds, models = run_batch_against_model(engine, roots, L, vl, calls, rollout=rollout)
    assert kinds.get(M.EVAL, 0) > 0
    if L >= 16:
        assert kinds.get(B.COLLISION, 0) > 0, kinds
    if n > 60:
        assert any(t.nodes[0].terminal for t in models) and kinds.get(M.TERMINAL, 0) > 0


def test_batch_matches_model_with_small_max_steps(engine, oracle):
    roots = env_roots(engine, 129, 5, plies=8)
    steps = roots[:, 12:14].contiguous().view(torch.int16).to(torch.int32)
    kinds, models = run_batch_against_model(engine, roots, 4, 1.0, 6, c_puct=2.5, fpu=-0.3, max_steps=int(steps.min()) + 2)
    assert kinds.get(M.TERMINAL, 0) > 129, kinds
    assert any(nd.terminal and nd.parent >= 0 for t in models for nd in t.nodes)


def test_full_trees_give_full_slots(engine, oracle):
    roots = env_roots(engine, 65, 11)
    kinds, models = run_batch_against_model(engine, roots, 8, 1.0, 3, max_nodes=6)
    assert kinds.get(M.FULL, 0) >= 2 * 8 * 20 and all(len(t.nodes) <= 6 for t in models)


def test_one_leaf_per_call_is_the_plain_search(engine, oracle):
    """L = 1 through the batch entry points gives sb_search_simulate / sb_search_end's outputs exactly"""
    dev, n, sims, m = engine.device, 257, 24, 25
    roots = mixed_roots(engine, n, 90)
    ws_a = torch.empty(engine.search_workspace_bytes(n, m), dtype=torch.uint8, device=dev)
    ws_b = torch.empty(engine.search_batch_workspace_bytes(n, m, 1), dtype=torch.uint8, device=dev)
    a = engine.search_begin(ws_a, roots, m)
    b = engine.search_begin(ws_b, roots, m)
    for k in range(sims + 1):
        assert all(torch.equal(a[key], b[key]) for key in LEAF), k
        prior, value = torch_eval(a, k)
        if k == sims:
            break
        a = engine.search_simulate(ws_a, n, m, prior, value, 1.25, 0.0)
        b = engine.search_simulate_batch(ws_b, n, m, 1, prior, value, 1.25, 0.0, 1.0)
    ra = engine.search_end(ws_a, n, m, prior, value)
    rb = engine.search_end_batch(ws_b, n, m, 1, prior, value)
    assert torch.equal(ra["visits"], rb["visits"]) and torch.equal(ra["root_value"].nan_to_num(7.0), rb["root_value"].nan_to_num(7.0))
    assert torch.equal(ra["q"].nan_to_num(7.0), rb["q"].nan_to_num(7.0))


class HostEval:
    """BatchedMCTS's evaluate(leaf, k) computing host_eval on the leaf records, so the models can use the same numbers"""

    def __init__(self, dev):
        self.dev = dev

    def __call__(self, leaf, k):
        recs = leaf["states"].cpu().numpy()
        p, v = host_eval([(r,) for r in recs])
        return torch.from_numpy(p).to(self.dev), torch.from_numpy(v).to(self.dev)


@pytest.mark.parametrize("L,R", [(4, 16), (8, 0)])
def test_batched_mcts_with_reuse_matches_models(engine, oracle, L, R):
    dev, n, sims = engine.device, 97, 16
    mcts = BatchedMCTS(n, sims, engine=engine, reuse_nodes=R, leaves_per_call=L, virtual_loss=1.0)
    m = mcts.max_nodes
    roots = mixed_roots(engine, n, 95)
    ev = HostEval(dev)
    models = [None] * n
    for move in range(2):
        host = roots.cpu().numpy()
        before = engine.launches
        visits, q, root_value = mcts.run(roots, ev)
        torch.cuda.synchronize()
        assert engine.launches == before + 2 * (sims // L) + 2
        if move == 0 or not R:
            models = [B.BatchTreeModel(host[g], m, L) for g in range(n)]
            want = [t.begin() for t in models]
            kept = np.zeros(n, np.int32)
        else:
            res = [advance_model(models[g], host[g], m, R + 1) for g in range(n)]
            models, want, kept = [x[0] for x in res], [x[1] for x in res], np.array([x[2] for x in res], np.int32)
        if R:
            assert np.array_equal(mcts.kept.cpu().numpy(), kept)
            if move:
                assert (kept > 0).any() and (kept == 0).any()
        p, v = host_eval(want)
        hp, hv = np.zeros((n * L, M.N_ACTIONS), np.float32), np.zeros(n * L, np.float32)
        hp.reshape(n, L, -1)[:, 0], hv.reshape(n, L)[:, 0] = p, v
        for _ in range(sims // L):
            leaves = [lf for g, t in enumerate(models) for lf in t.simulate_batch(hp[g * L:(g + 1) * L], hv[g * L:(g + 1) * L], 1.25, 0.0, 1.0)]
            hp, hv = host_eval(leaves)
        compare_end({"visits": visits, "q": q, "root_value": root_value},
                    [t.end_batch(hp[g * L:(g + 1) * L], hv[g * L:(g + 1) * L]) for g, t in enumerate(models)])
        roots = next_roots(engine, roots, visits, mixed_roots(engine, n, 96))


def advance_model(src, root, m, keep):
    t, leaf, kept = R.search_advance(src, root, m, keep)
    return B.BatchTreeModel.from_tree(t, src.L), leaf, kept


def test_cuda_graph_replays_a_batched_run(engine):
    n, sims, L = 300, 24, 4
    roots = env_roots(engine, n, 13)
    eager = BatchedMCTS(n, sims, engine=engine, leaves_per_call=L)
    want = [t.clone() for t in eager.run(roots, torch_eval)]
    graphed = BatchedMCTS(n, sims, engine=engine, leaves_per_call=L)
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
    assert bool((outs[0].sum(1) <= sims).all()) and bool((outs[0].sum(1) > 0).any())


def test_leaves_per_call_must_divide_num_simulations(engine):
    with pytest.raises(ValueError):
        BatchedMCTS(4, 10, engine=engine, leaves_per_call=4)
    with pytest.raises(ValueError):
        BatchedMCTS(4, 8, engine=engine, leaves_per_call=4, virtual_loss=-1.0)


def test_empty_batch_and_rejected_arguments(engine):
    dev = engine.device
    lib, h = engine.lib, engine.h
    n, m, L = 8, 9, 4
    roots = env_roots(engine, n, 17, plies=1)
    nb = engine.search_batch_workspace_bytes(n, m, L)
    ws = torch.empty(nb + 16, dtype=torch.uint8, device=dev)
    engine.search_begin(ws, roots, m)
    o = engine._search_outputs(n * L, None, LEAF)
    for t in o.values():
        t.fill_(0x5A)
    prior = torch.full((n * L, M.N_ACTIONS), 0.1, dtype=torch.float32, device=dev)
    value = torch.zeros(n * L, dtype=torch.float32, device=dev)
    vis = torch.full((n, M.N_ACTIONS), 7, dtype=torch.int32, device=dev)
    qq = torch.full((n, M.N_ACTIONS), 7.0, dtype=torch.float64, device=dev)
    rv = torch.full((n,), 7.0, dtype=torch.float64, device=dev)
    torch.cuda.synchronize()
    snapshot = [t.clone() for t in (ws, vis, qq, rv, *o.values())]
    before = engine.launches
    engine.search_simulate_batch(ws[:0], 0, m, L, prior[:0], value[:0])
    engine.search_end_batch(ws[:0], 0, m, L, prior[:0], value[:0])
    assert engine.launches == before
    p = lambda t: ctypes.c_void_p(t.data_ptr())  # noqa: E731
    out6 = [p(o[k]) for k in LEAF]
    nan, inf = float("nan"), float("inf")
    small = nb - 1

    def sim(n=n, m=m, L=L, w=p(ws), b=nb, pr=p(prior), v=p(value), c=1.0, f=0.0, vl=1.0):
        return lib.sb_search_simulate_batch(h, n, m, L, w, b, pr, v, c, f, vl, *out6, None)

    def end(n=n, m=m, L=L, w=p(ws), b=nb, pr=p(prior), v=p(value), outs=(p(vis), p(qq), p(rv))):
        return lib.sb_search_end_batch(h, n, m, L, w, b, pr, v, *outs, None)

    cases = [(sim(L=0), "leaves"), (sim(L=257), "leaves"), (sim(vl=-1.0), "virtual_loss"), (sim(vl=nan), "virtual_loss"),
             (sim(vl=inf), "virtual_loss"), (sim(n=-1), "n must"), (sim(m=0), "max_nodes"), (sim(m=2**24 + 1), "max_nodes"),
             (sim(w=None), "NULL"), (sim(b=small), "too small"), (sim(w=ctypes.c_void_p(ws.data_ptr() + 8), b=nb + 8), "aligned"),
             (sim(c=-1.0), "c_puct"), (sim(c=nan), "c_puct"), (sim(f=nan), "fpu"), (sim(f=-inf), "fpu"),
             (sim(pr=None), "prior"), (sim(v=None), "prior"), (sim(n=2**24, m=2**20, L=256, b=2**62), "n * leaves"),
             (end(L=0), "leaves"), (end(L=257), "leaves"), (end(n=-1), "n must"), (end(m=0), "max_nodes"), (end(w=None), "NULL"),
             (end(b=small), "too small"), (end(pr=None), "prior"), (end(v=None), "prior"),
             (end(outs=(None, p(qq), p(rv))), "visits"), (end(outs=(p(vis), None, p(rv))), "visits"),
             (end(outs=(p(vis), p(qq), None)), "visits")]
    for rc, why in cases:
        assert rc == -1, why
    # the reasons, one call at a time
    for call, why in [(lambda: sim(L=0), "leaves must be 1..256"), (lambda: sim(vl=-1.0), "virtual_loss must be finite"),
                      (lambda: sim(b=small), "sb_search_batch_workspace_bytes"), (lambda: end(L=300), "leaves must be 1..256")]:
        assert call() == -1
        assert why in lib.sb_last_error(h).decode(), (why, lib.sb_last_error(h))
    assert engine.launches == before
    torch.cuda.synchronize()
    assert all(torch.equal(a, b) for a, b in zip(snapshot, (ws, vis, qq, rv, *o.values()))), "a rejected call wrote nothing"
    with pytest.raises(_lib.SbError):
        engine.search_simulate_batch(ws, n, m, L, prior, value, virtual_loss=-0.5)
    assert sim() == 0 and engine.launches == before + 2
    assert end() == 0 and engine.launches == before + 3
    torch.cuda.synchronize()
    assert bool((vis.sum(1) <= L).all())

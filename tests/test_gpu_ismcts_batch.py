"""GPU: sb_ismcts_simulate_batch / sb_ismcts_end_batch (and InformationSetMCTS with leaves_per_call) against the
plain-Python statement of several leaves per information-set tree per call (tests/sb_ismcts_batch_model.py): every slot's
leaf outputs of every call and every read-out must equal the model's byte for byte."""
import ctypes

import numpy as np
import pytest
import torch

import sb_determinize_model as D
import sb_ismcts_batch_model as IB
import sb_reuse_model as R
import sb_search_model as M
from monsoon_b200 import _lib
from monsoon_b200.search import InformationSetMCTS
from test_gpu_determinize import keys_for, mixed_roots
from test_gpu_ismcts import with_copies
from test_gpu_reuse import Evaluator, compare_end, stepped
from test_gpu_search import LEAF, compare_leaves, env_roots, host_eval, torch_eval
from test_gpu_search_batch import slot0

pytestmark = pytest.mark.gpu


def virtual_visits(engine, ws, n, m, L):
    """the V arrays of the n trees' tails (i32[n, max_nodes])"""
    pre = engine.ismcts_workspace_bytes(n, m)
    tail = (engine.ismcts_batch_workspace_bytes(n, m, L) - pre) // n
    t = ws[pre:pre + n * tail].view(n, tail)[:, 16 * L:16 * L + 4 * m].contiguous()
    return t.view(torch.int32).cpu().numpy()


def run_batch_against_model(engine, roots, L, vl, calls, c_puct=1.25, fpu=0.0, max_steps=400, rollout=False, max_nodes=None, salt=1):
    """begin on world 0, `calls` batch calls over fresh worlds and the batch end, with the models side by side; every leaf
    record must carry its own slot's key.  Returns (slot kind counts, models)."""
    dev, n = engine.device, roots.shape[0]
    m = max_nodes or 1 + calls * L
    host = roots.cpu().numpy()
    keys = keys_for(n * (1 + calls * L), salt).to(dev)
    hk = keys.cpu().numpy().view(np.uint64)
    repeated = roots.repeat_interleave(L, 0)
    models = [IB.ISBatchTreeModel(m, L, max_steps) for _ in range(n)]
    ws = torch.empty(engine.ismcts_batch_workspace_bytes(n, m, L), dtype=torch.uint8, device=dev)
    ev = Evaluator(engine, rollout)
    det = engine.determinize(roots, keys[:n])
    o = engine.ismcts_begin(ws, det, m, max_steps)
    want = [t.begin(D.determinize(host[g], int(hk[g]))) for g, t in enumerate(models)]
    compare_leaves(o, want, 0)
    prior, value, hp, hv = slot0(n, L, *ev(o, want), dev)
    kinds = {}
    for k in range(1, calls + 1):
        lo = n + (k - 1) * n * L
        det = engine.determinize(repeated, keys[lo:lo + n * L])
        before = engine.launches
        o = engine.ismcts_simulate_batch(ws, det, m, L, prior, value, c_puct, fpu, vl)
        assert engine.launches == before + 1
        want = [lf for g, t in enumerate(models)
                for lf in t.simulate_batch([D.determinize(host[g], int(hk[lo + g * L + l])) for l in range(L)],
                                           hp[g * L:(g + 1) * L], hv[g * L:(g + 1) * L], c_puct, fpu, vl)]
        compare_leaves(o, want, k)
        got = o["states"].cpu().numpy()
        assert got[:, :8].tobytes() == keys[lo:lo + n * L].cpu().numpy().tobytes(), k  # each slot's own key
        assert not virtual_visits(engine, ws, n, m, L).any(), "virtual visits are zero when a call returns"
        for lf in want:
            kinds[lf[5]] = kinds.get(lf[5], 0) + 1
        prior, value, hp, hv = ev(o, want)
    before = engine.launches
    r = engine.ismcts_end_batch(ws, n, m, L, prior, value)
    assert engine.launches == before + 1
    compare_end(r, [t.end_batch(hp[g * L:(g + 1) * L], hv[g * L:(g + 1) * L]) for g, t in enumerate(models)])
    return kinds, models


@pytest.mark.parametrize("n,L,vl,calls,rollout", [(63, 1, 1.0, 10, False), (64, 2, 0.0, 6, False), (65, 7, 3.5, 3, True),
                                                   (65, 16, 1.0, 3, False), (1, 64, 1.0, 3, False), (63, 64, 3.5, 2, False),
                                                   (4099, 2, 1.0, 2, False), (64, 16, 0.0, 2, True), (1, 7, 0.0, 4, False)])
def test_batch_matches_model(engine, oracle, n, L, vl, calls, rollout):
    roots = with_copies(mixed_roots(engine, n, 70 + L)) if n > 1 else env_roots(engine, n, 70 + L)
    kinds, models = run_batch_against_model(engine, roots, L, vl, calls, rollout=rollout, salt=L + n)
    assert kinds.get(M.EVAL, 0) > 0
    if L >= 16:
        assert kinds.get(IB.COLLISION, 0) > 0, kinds
    if n > 60:
        assert kinds.get(M.TERMINAL, 0) > 0 and {t.nodes[0].seat for t in models} == {0, 1}


def test_batch_matches_model_with_small_max_steps(engine, oracle):
    roots = env_roots(engine, 129, 5, plies=8)
    steps = roots[:, 12:14].contiguous().view(torch.int16).to(torch.int32)
    kinds, models = run_batch_against_model(engine, roots, 4, 1.0, 5, c_puct=2.5, fpu=-0.3, max_steps=int(steps.min()) + 2, salt=5)
    assert kinds.get(M.TERMINAL, 0) > 129, kinds


def test_full_trees_give_full_slots(engine, oracle):
    """trees too small for C * L new nodes: the FULL cut-off falls mid-call, in slot order"""
    roots = env_roots(engine, 65, 11)
    kinds, models = run_batch_against_model(engine, roots, 8, 1.0, 3, max_nodes=6, salt=6)
    assert kinds.get(M.FULL, 0) >= 2 * 8 * 20 and all(len(t.nodes) <= 6 for t in models)
    kinds, models = run_batch_against_model(engine, roots, 16, 0.0, 2, max_nodes=12, salt=7)
    assert kinds.get(M.FULL, 0) > 0 and kinds.get(M.EVAL, 0) > 65


def test_few_actions_at_large_L_collide(engine, oracle):
    """roots late in a game (few legal representatives) with L = 64: slots collide"""
    roots = env_roots(engine, 33, 21, plies=30)
    kinds, _models = run_batch_against_model(engine, roots, 64, 1.0, 2, salt=8)
    assert kinds.get(IB.COLLISION, 0) > 0, kinds


def test_one_leaf_per_call_is_the_plain_search(engine, oracle):
    """L = 1 through the batch entry points gives sb_ismcts_simulate / sb_ismcts_end's outputs exactly"""
    dev, n, sims, m = engine.device, 257, 20, 21
    roots = with_copies(mixed_roots(engine, n, 90))
    keys = keys_for(n * (sims + 1), 3).to(dev)
    ws_a = torch.empty(engine.ismcts_workspace_bytes(n, m), dtype=torch.uint8, device=dev)
    ws_b = torch.empty(engine.ismcts_batch_workspace_bytes(n, m, 1), dtype=torch.uint8, device=dev)
    det = engine.determinize(roots, keys[:n])
    a = engine.ismcts_begin(ws_a, det, m)
    b = engine.ismcts_begin(ws_b, det, m)
    for k in range(sims + 1):
        assert all(torch.equal(a[key], b[key]) for key in LEAF), k
        prior, value = torch_eval(a, k)
        if k == sims:
            break
        det = engine.determinize(roots, keys[(k + 1) * n:(k + 2) * n])
        a = engine.ismcts_simulate(ws_a, det, m, prior, value, 1.25, 0.0)
        b = engine.ismcts_simulate_batch(ws_b, det, m, 1, prior, value, 1.25, 0.0, 1.0)
    ra = engine.ismcts_end(ws_a, n, m, prior, value)
    rb = engine.ismcts_end_batch(ws_b, n, m, 1, prior, value)
    assert torch.equal(ra["visits"], rb["visits"]) and torch.equal(ra["root_value"].nan_to_num(7.0), rb["root_value"].nan_to_num(7.0))
    assert torch.equal(ra["q"].nan_to_num(7.0), rb["q"].nan_to_num(7.0))


@pytest.mark.parametrize("L,vl", [(4, 1.0), (16, 3.5)])
def test_fixed_world_equals_the_perfect_information_batch_search(engine, L, vl):
    """every world is the root itself (default decks): leaves and read-out are sb_search_simulate_batch's"""
    n, calls, dev = 129, 3, engine.device
    roots = env_roots(engine, n, 15, plies=6)
    finished = roots[::16].clone()
    engine.rollout_random(finished)
    roots[::16] = finished
    m = 1 + calls * L
    repeated = roots.repeat_interleave(L, 0)
    wa = torch.empty(engine.search_batch_workspace_bytes(n, m, L), dtype=torch.uint8, device=dev)
    wb = torch.empty(engine.ismcts_batch_workspace_bytes(n, m, L), dtype=torch.uint8, device=dev)
    a = engine.search_begin(wa, roots, m)
    b = engine.ismcts_begin(wb, roots, m)
    for key in LEAF:
        assert torch.equal(a[key], b[key]), key
    p, v = torch_eval(a, 0)
    prior, value = torch.zeros((n * L, M.N_ACTIONS), dtype=torch.float32, device=dev), torch.zeros(n * L, dtype=torch.float32, device=dev)
    prior.view(n, L, -1)[:, 0], value.view(n, L)[:, 0] = p, v
    for k in range(1, calls + 1):
        a = engine.search_simulate_batch(wa, n, m, L, prior, value, 1.25, 0.0, vl)
        b = engine.ismcts_simulate_batch(wb, repeated, m, L, prior, value, 1.25, 0.0, vl)
        for key in LEAF:
            assert torch.equal(a[key], b[key]), (k, key)
        prior, value = torch_eval(a, k)
    ra, rb = engine.search_end_batch(wa, n, m, L, prior, value), engine.ismcts_end_batch(wb, n, m, L, prior, value)
    assert torch.equal(ra["visits"], rb["visits"]) and torch.equal(ra["root_value"], rb["root_value"])
    assert torch.equal(torch.nan_to_num(ra["q"], nan=7.0), torch.nan_to_num(rb["q"], nan=7.0))
    assert int(rb["visits"].sum()) > n


@pytest.mark.parametrize("L,reuse", [(4, 16), (8, 0)])
def test_information_set_mcts_with_reuse_matches_models(engine, oracle, L, reuse):
    """the class over two moves: worlds from sb_determinize of the repeated roots under the caller's keys, and the advance
    of sb_reuse_model composed with the batch model"""
    dev, n, sims = engine.device, 97, 16
    mcts = InformationSetMCTS(n, sims, engine=engine, reuse_nodes=reuse, leaves_per_call=L, virtual_loss=1.0)
    m, C = mcts.max_nodes, sims // L
    roots = with_copies(mixed_roots(engine, n, 95))
    models, played = [None] * n, None
    for move in range(2):
        host = roots.cpu().numpy()
        keys = keys_for(n * (sims + 1), 300 + move).to(dev)
        hk = keys.cpu().numpy().view(np.uint64)
        state = {}

        def evaluate(leaf, k):
            if k == 0:
                worlds = [D.determinize(host[g], int(hk[g])) for g in range(n)]
                if played is None or not reuse:
                    models[:] = [IB.ISBatchTreeModel(m, L) for _ in range(n)]
                    want = [t.begin(worlds[g]) for g, t in enumerate(models)]
                    kept = np.zeros(n, np.int32)
                else:  # the roots are the previous roots stepped with played wherever played is an action id
                    pl = played.cpu().numpy()
                    res = [R.ismcts_advance(models[g], worlds[g], int(pl[g]) if pl[g] < 156 else -1, m, reuse + 1) for g in range(n)]
                    models[:] = [IB.ISBatchTreeModel.from_tree(x[0], L) for x in res]
                    want, kept = [x[1] for x in res], np.array([x[2] for x in res], np.int32)
                if reuse:
                    assert np.array_equal(mcts.kept.cpu().numpy(), kept)
                state["kept"] = kept
                p, v = host_eval(want)
                hp, hv = np.zeros((n * L, M.N_ACTIONS), np.float32), np.zeros(n * L, np.float32)
                hp.reshape(n, L, -1)[:, 0], hv.reshape(n, L)[:, 0] = p, v
            else:
                lo = n + (k - 1) * n * L
                want = [lf for g, t in enumerate(models)
                        for lf in t.simulate_batch([D.determinize(host[g], int(hk[lo + g * L + l])) for l in range(L)],
                                                   state["p"][g * L:(g + 1) * L], state["v"][g * L:(g + 1) * L], 1.25, 0.0, 1.0)]
                p, v = hp, hv = host_eval(want)
            compare_leaves(leaf, want, k)
            state["p"], state["v"] = hp, hv
            return torch.from_numpy(p).to(dev), torch.from_numpy(v).to(dev)

        before = engine.launches
        visits, q, rv = mcts.run(roots, evaluate, keys, played=played)
        torch.cuda.synchronize()
        assert engine.launches == before + 2 * C + 3 + (1 if reuse and played is not None else 0)
        compare_end({"visits": visits, "q": q, "root_value": rv},
                    [t.end_batch(state["p"][g * L:(g + 1) * L], state["v"][g * L:(g + 1) * L]) for g, t in enumerate(models)])
        if reuse and move:
            assert (state["kept"] > 0).any()
        a = torch.argmax(visits, 1)
        a = torch.where(visits.sum(1) > 0, a, torch.full_like(a, 255))
        played = a.to(torch.int32)
        roots = stepped(engine, roots, a)


def test_launch_count_and_cuda_graph(engine):
    n, sims, L = 300, 16, 4
    roots = env_roots(engine, n, 13)
    keys = keys_for(n * (sims + 1), 8).to(engine.device)
    eager = InformationSetMCTS(n, sims, engine=engine, leaves_per_call=L)
    before = engine.launches
    want = [t.clone() for t in eager.run(roots, torch_eval, keys)]
    torch.cuda.synchronize()
    assert engine.launches == before + 2 * (sims // L) + 3
    graphed = InformationSetMCTS(n, sims, engine=engine, leaves_per_call=L)
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
    assert bool((outs[0].sum(1) <= sims).all()) and bool((outs[0].sum(1) > 0).any())
    static_roots.copy_(env_roots(engine, n, 14))
    static_keys.copy_(keys_for(n * (sims + 1), 9).to(engine.device))
    g.replay()
    again = eager.run(static_roots.clone(), torch_eval, static_keys.clone())
    torch.cuda.synchronize()
    assert torch.equal(outs[0], again[0]) and torch.equal(outs[2], again[2])


def test_leaves_per_call_must_divide_num_simulations(engine):
    with pytest.raises(ValueError):
        InformationSetMCTS(4, 10, engine=engine, leaves_per_call=4)
    with pytest.raises(ValueError):
        InformationSetMCTS(4, 8, engine=engine, leaves_per_call=4, virtual_loss=float("nan"))


def test_empty_batch_and_rejected_arguments(engine):
    dev = engine.device
    lib, h = engine.lib, engine.h
    n, m, L = 8, 9, 4
    roots = env_roots(engine, n, 17, plies=1)
    nb = engine.ismcts_batch_workspace_bytes(n, m, L)
    ws = torch.empty(nb + 16, dtype=torch.uint8, device=dev)
    engine.ismcts_begin(ws, roots, m)
    det = roots.repeat_interleave(L, 0)
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
    engine.ismcts_simulate_batch(ws[:0], det[:0], m, L, prior[:0], value[:0])
    engine.ismcts_end_batch(ws[:0], 0, m, L, prior[:0], value[:0])
    assert engine.launches == before
    p = lambda t: ctypes.c_void_p(t.data_ptr())  # noqa: E731
    out6 = [p(o[k]) for k in LEAF]
    nan, inf = float("nan"), float("inf")
    small = nb - 1

    def sim(n=n, m=m, L=L, w=p(ws), b=nb, d=p(det), pr=p(prior), v=p(value), c=1.0, f=0.0, vl=1.0):
        return lib.sb_ismcts_simulate_batch(h, n, m, L, w, b, d, pr, v, c, f, vl, *out6, None)

    def end(n=n, m=m, L=L, w=p(ws), b=nb, pr=p(prior), v=p(value), outs=(p(vis), p(qq), p(rv))):
        return lib.sb_ismcts_end_batch(h, n, m, L, w, b, pr, v, *outs, None)

    cases = [(sim(L=0), "leaves"), (sim(L=257), "leaves"), (sim(vl=-1.0), "virtual_loss"), (sim(vl=nan), "virtual_loss"),
             (sim(vl=inf), "virtual_loss"), (sim(n=-1), "n must"), (sim(m=0), "max_nodes"), (sim(m=2**24 + 1), "max_nodes"),
             (sim(w=None), "NULL"), (sim(b=small), "too small"), (sim(w=ctypes.c_void_p(ws.data_ptr() + 8), b=nb + 8), "aligned"),
             (sim(d=None), "worlds"), (sim(c=-1.0), "c_puct"), (sim(c=nan), "c_puct"), (sim(c=inf), "c_puct"), (sim(f=nan), "fpu"),
             (sim(f=-inf), "fpu"), (sim(pr=None), "prior"), (sim(v=None), "prior"),
             (sim(n=2**24, m=2**10, L=256, b=2**62), "n * leaves"),
             (end(L=0), "leaves"), (end(L=257), "leaves"), (end(n=-1), "n must"), (end(m=0), "max_nodes"), (end(w=None), "NULL"),
             (end(b=small), "too small"), (end(pr=None), "prior"), (end(v=None), "prior"),
             (end(outs=(None, p(qq), p(rv))), "visits"), (end(outs=(p(vis), None, p(rv))), "visits"),
             (end(outs=(p(vis), p(qq), None)), "visits")]
    for rc, why in cases:
        assert rc == -1, why
    for call, why in [(lambda: sim(L=0), "leaves must be 1..256"), (lambda: sim(vl=-1.0), "virtual_loss must be finite"),
                      (lambda: sim(b=small), "sb_ismcts_batch_workspace_bytes"), (lambda: sim(d=None), "worlds (det) are required"),
                      (lambda: sim(n=2**24, m=2**10, L=256, b=2**62), "n * leaves must be below 2^31"),
                      (lambda: end(L=300), "leaves must be 1..256"), (lambda: end(b=small), "sb_ismcts_batch_workspace_bytes")]:
        assert call() == -1
        assert why in lib.sb_last_error(h).decode(), (why, lib.sb_last_error(h))
    assert engine.launches == before
    torch.cuda.synchronize()
    assert all(torch.equal(a, b) for a, b in zip(snapshot, (ws, vis, qq, rv, *o.values()))), "a rejected call wrote nothing"
    with pytest.raises(_lib.SbError):
        engine.ismcts_simulate_batch(ws, det, m, L, prior, value, virtual_loss=-0.5)
    assert sim() == 0 and engine.launches == before + 1
    assert end() == 0 and engine.launches == before + 2
    torch.cuda.synchronize()
    assert bool((vis.sum(1) <= L).all()) and int(vis.sum()) > 0

"""GPU: sb_determinize against the plain-Python model, the observer's view it keeps, and DeterminizedMCTS against PIMC over
the search model."""
import ctypes

import numpy as np
import pytest
import torch

import sb_determinize_model as D
import sb_oracle as O
import sb_search_model as M
from monsoon_b200.search import DeterminizedMCTS, rollout_evaluator
from monsoon_b200.vec_env import next_seed_array
from test_gpu_search import env_roots, host_eval, torch_eval
from test_oracle_golden import chain_of

pytestmark = pytest.mark.gpu


def mixed_roots(engine, n, seed):
    """env records with mixed seats, default and random decks, terminal records and records with an engine status"""
    a = env_roots(engine, n // 2, seed, plies=6)
    b = env_roots(engine, n - n // 2, seed + 1, decks=True, plies=9)
    roots = torch.cat([a, b])
    done = roots[::13].clone()
    engine.rollout_random(done)  # whole games: terminal records
    roots[::13] = done
    roots[5::97, 18] = 3  # an engine status set (SB_ERR_INDEX)
    return roots


def keys_for(n, salt):
    return torch.from_numpy(next_seed_array(np.arange(n, dtype=np.uint64) + np.uint64(salt)) ^ np.int64(-0x3C6EF372FE94F82B))


def test_kernel_matches_model(engine, oracle):
    n = 4099
    dev = engine.device
    roots = mixed_roots(engine, n, 31)
    keys = keys_for(n, 7).to(dev)
    host, hk = roots.cpu().numpy(), keys.cpu().numpy().view(np.uint64)
    assert set(host[:, 14].tolist()) == {0, 1} and (host[:, 18] != 0).any()
    rs = np.random.RandomState(2)
    obs_np = rs.randint(0, 3, n).astype(np.uint8)  # 0 FIRST, any other byte SECOND
    for observer in (None, torch.from_numpy(obs_np).to(dev)):
        got = engine.determinize(roots, keys, observer).cpu().numpy()
        for g in range(n):
            want = D.determinize(host[g], int(hk[g]), None if observer is None else int(obs_np[g]))
            assert got[g].tobytes() == want.tobytes(), (observer is None, g)
        inplace = roots.clone()
        out = engine.determinize(inplace, keys, observer, out=inplace)
        assert out.data_ptr() == inplace.data_ptr() and np.array_equal(inplace.cpu().numpy(), got)
    assert not np.array_equal(got, host)


def test_observer_view_is_kept_at_scale(engine):
    n = 65536
    roots = mixed_roots(engine, n, 41)
    keys = keys_for(n, 11).to(engine.device)
    det = engine.determinize(roots, keys)
    (oa, ea), (ob, eb) = engine.observe(roots), engine.observe(det)
    assert torch.equal(oa, ob) and torch.equal(ea, eb)
    (fa, ea), (fb, eb) = engine.features(roots), engine.features(det)
    assert torch.equal(ea, eb) and torch.equal(fa.view(torch.int64), fb.view(torch.int64))  # bit for bit, NaNs included
    assert torch.equal(engine.legal_mask(roots), engine.legal_mask(det))
    assert not torch.equal(roots, det)


def test_rollouts_of_determinized_records_match_the_oracle(engine, oracle):
    n = 512
    roots = env_roots(engine, n, 51, plies=4)
    det = engine.determinize(roots, keys_for(n, 13).to(engine.device))
    host = det.cpu().numpy()
    chain = torch.zeros(n, dtype=torch.int64, device=engine.device)
    engine.rollout_random(det, 400, chain=chain)
    got, gc = det.cpu().numpy(), chain.cpu().numpy().view(np.uint64)
    clean = 0
    for g in range(n):
        st = host[g].copy()
        _a, dig, _m = O.rollout_random(st, 400)
        assert (st[18] != 0) == (got[g][18] != 0), g
        if st[18] == 0:  # games the rules abort stop at the status; their chains are compared by the golden tests
            assert st.tobytes() == got[g].tobytes() and chain_of(dig) == int(gc[g]), g
            clean += 1
    assert clean > n * 0.9


def pimc_against_model(engine, roots, k, sims, rollout):
    n = roots.shape[0]
    dev = engine.device
    keys = keys_for(n * k, 17 + sims).to(dev)
    mcts = DeterminizedMCTS(n, k, sims, engine=engine)
    host, hk = roots.cpu().numpy(), keys.cpu().numpy().view(np.uint64)
    trees = []
    for t in range(n * k):
        d = D.determinize(host[t // k], int(hk[t]))
        assert np.array_equal(O.legal_mask(d.copy()), O.legal_mask(host[t // k].copy()))  # the same root legal set in all K
        trees.append(M.TreeModel(d, sims + 1))
    want = [t.begin() for t in trees]
    ev = rollout_evaluator(engine) if rollout else None
    last = {}

    def evaluate(leaf, j):
        if rollout:
            p, v = ev(leaf, j)
            pv = [M.rollout_eval(lf) for lf in want]
            hp, hv = np.stack([x[0] for x in pv]), np.array([x[1] for x in pv], dtype=np.float32)
            assert np.array_equal(p.cpu().numpy(), hp) and np.array_equal(v.cpu().numpy(), hv), j
        else:
            assert leaf["states"].cpu().numpy().tobytes() == np.stack([lf[0] for lf in want]).tobytes(), j
            hp, hv = host_eval(want)
            p, v = torch.from_numpy(hp).to(dev), torch.from_numpy(hv).to(dev)
        last["p"], last["v"] = hp, hv
        if j < sims:
            want[:] = [t.simulate(hp[g], hv[g], 1.25, 0.0) for g, t in enumerate(trees)]
        return p, v

    before = engine.launches
    visits, q, rv = mcts.run(roots, evaluate, keys)
    torch.cuda.synchronize()
    assert engine.launches == before + sims + 3 + (sims + 1 if rollout else 0)  # the rollout evaluator launches once per call
    wv, wq, wr = D.pimc_readout(trees, last["p"], last["v"], n, k)
    assert np.array_equal(visits.cpu().numpy(), wv)
    gq = q.cpu().numpy()
    assert np.array_equal(np.isnan(gq), np.isnan(wq)) and np.nanmax(np.abs(gq - wq), initial=0.0) <= 1e-12
    assert np.max(np.abs(rv.cpu().numpy() - wr)) <= 1e-12
    return wv


@pytest.mark.parametrize("rollout", [False, True])
def test_determinized_mcts_matches_pimc_model(engine, oracle, rollout):
    roots = env_roots(engine, 48, 61 if rollout else 62, plies=7)
    visits = pimc_against_model(engine, roots, 4, 12, rollout)
    assert (visits.sum(1) == 4 * 12).sum() > 0


def test_cuda_graph_with_caller_keys(engine):
    n, k, sims = 96, 4, 8
    roots = env_roots(engine, n, 71)
    keys = keys_for(n * k, 3).to(engine.device)
    eager = DeterminizedMCTS(n, k, sims, engine=engine)
    want = [t.clone() for t in eager.run(roots, torch_eval, keys)]
    graphed = DeterminizedMCTS(n, k, sims, engine=engine)
    static_roots, static_keys = roots.clone(), keys.clone()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        graphed.run(static_roots, torch_eval, static_keys)
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
    static_keys.copy_(keys_for(n * k, 4).to(engine.device))
    g.replay()
    again = eager.run(roots, torch_eval, static_keys.clone())
    torch.cuda.synchronize()
    assert torch.equal(outs[0], again[0]) and torch.equal(outs[2], again[2])
    assert not torch.equal(outs[0], want[0])
    # default keys: reproducible from the seed, a new set per call
    a, b = DeterminizedMCTS(n, k, sims, seed=5, engine=engine), DeterminizedMCTS(n, k, sims, seed=5, engine=engine)
    ka, kb = a.default_keys(), b.default_keys()
    assert np.array_equal(ka, kb) and not np.array_equal(ka, a.default_keys()) and len(set(ka.tolist())) == n * k


def test_empty_batch_and_rejected_arguments(engine):
    dev = engine.device
    lib, h = engine.lib, engine.h
    n = 8
    roots = env_roots(engine, n, 81, plies=1)
    keys = keys_for(n, 5).to(dev)
    out = torch.empty_like(roots)
    p = lambda t: ctypes.c_void_p(t.data_ptr())  # noqa: E731
    before = engine.launches
    engine.determinize(roots[:0], keys[:0])
    assert lib.sb_determinize(h, 0, None, None, None, None, None) == 0

    def det(n=n, s=p(roots), o=None, k=p(keys), d=p(out)):
        return lib.sb_determinize(h, n, s, o, k, d, None)

    bad = [det(n=-1), det(s=None), det(k=None), det(d=None)]
    assert all(rc == -1 for rc in bad), bad
    assert "sb_determinize" in lib.sb_last_error(h).decode()
    assert engine.launches == before
    assert det() == 0 and engine.launches == before + 1
    torch.cuda.synchronize()
    assert out.cpu().numpy().tobytes() == np.stack([D.determinize(r, int(k)) for r, k in
                                                    zip(roots.cpu().numpy(), keys.cpu().numpy().view(np.uint64))]).tobytes()

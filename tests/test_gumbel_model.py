"""CPU: the plain-Python Gumbel search model (tests/sb_gumbel_model.py) on the C oracle -- the sequential-halving schedule,
the root's Gumbel-top-k order, the improved policy, the action, the node value, NaN and zero-prior inputs -- and the Gumbel
entry points of the library (symbols, stack frames)."""
import math

import numpy as np
import pytest

import sb_determinize_model as D
import sb_gumbel_model as G
import sb_search_model as SM
from test_determinize_model import ended, keys, records
from test_search_model import hash_eval, position
from test_stack_frames import MAX_STACK, kernel_frames

CHECKS = {(4, 8): [0, 0, 0, 0, 1, 1, 2, 2], (3, 6): [0, 0, 0, 1, 1, 2], (2, 5): [0, 0, 1, 1, 2], (1, 4): [0, 1, 2, 3],
          (16, 16): [0] * 16}


def gumbel_for(seed):
    u = np.random.default_rng(seed).random(SM.N_ACTIONS) * (1 - 2e-12) + 1e-12
    return (-np.log(-np.log(u))).astype(np.float32)


class Recording(G.GumbelTreeModel):
    """records, per call, the root's chosen id, its visit count when chosen and the call's target count"""

    def select(self, nd, c_puct, fpu):
        a = super().select(nd, c_puct, fpu)
        if nd is self.nodes[0]:
            g, sim, S, mc = self._gumbel_call[:4]
            edges = self._edges(nd)
            target = G.seq(min(mc, len(edges)), S)[sim - 1]
            self.log.append((a, dict((e[0], e[1]) for e in edges)[a], target, any(e[1] == target for e in edges)))
        return a


def search(root, sims, mc, gumbel, evaluate=hash_eval, c_visit=50.0, c_scale=0.1, max_nodes=None, cls=Recording):
    t = cls(root, max_nodes or sims + 1)
    t.log, t.evals = [], {}
    leaf = t.begin()
    prior, value = evaluate(leaf)
    t.evals[0] = float(value)
    for k in range(1, sims + 1):
        leaf = t.simulate(prior, value, gumbel, k, sims, mc, c_visit, c_scale)
        prior, value = evaluate(leaf)
        if leaf[5] == SM.EVAL:
            t.evals[t.leaf] = float(value)
    return t, t.end(prior, value, gumbel, c_visit, c_scale)


def roots(oracle, count=12):
    out = [position(oracle, s, p) for s, p in zip(range(40), [4, 9, 15, 22] * 10)]
    return [st for st in out if not SM.over(st, 400)][:count]


def test_seq_check_values_and_its_invariants():
    for (m, S), want in CHECKS.items():
        assert G.seq(m, S) == want
    for m in range(1, 40):
        for S in (1, 2, 5, 16, 31, 64, 200):
            s = G.seq(m, S)
            assert len(s) == S and s[0] == 0
            if m > 1:
                assert s[:min(m, S)] == [0] * min(m, S)  # every considered action once before any second visit


def test_root_visits_follow_sequential_halving(oracle):
    """brute force: at every call the chosen root id had exactly seq(m, S)[k-1] visits when some id had that many"""
    n = 0
    for g, st in enumerate(roots(oracle, 8)):
        for mc, sims in ((16, 32), (4, 16), (2, 7), (1, 5), (156, 24)):
            t, _ = search(st, sims, mc, gumbel_for(g * 10 + mc))
            assert len(t.log) == sims
            for a, na, target, some in t.log:
                assert na == target or not some, (g, mc, sims)
                n += some
    assert n > 300


def test_first_calls_visit_the_top_ids_by_gumbel_plus_logit(oracle):
    for g, st in enumerate(roots(oracle, 8)):
        for mc, sims in ((4, 12), (16, 8), (156, 30)):
            gum = gumbel_for(100 + g)
            t, _ = search(st, sims, mc, gum)
            root = t.nodes[0]
            legal = SM.legal_ids(root.mask)
            m = min(mc, len(legal), sims)
            top = sorted(legal, key=lambda a: (-(float(gum[a]) + G.logit(root.prior[a])), a))[:m]
            assert [a for a, _n, _t, _s in t.log[:m]] == top, (g, mc)
            assert [t.nodes[k].action for k in range(1, m + 1)] == top  # node k is the root child call k expanded


def test_policy_action_and_read_out(oracle):
    for g, st in enumerate(roots(oracle)):
        gum = gumbel_for(7 + g)
        t, (action, policy, visits, q, rv) = search(st, 24, 8, gum)
        legal = SM.legal_ids(t.nodes[0].mask)
        out = np.setdiff1d(np.arange(SM.N_ACTIONS), legal)
        assert (policy[out] == 0).all() and abs(float(policy[legal].astype(np.float64).sum()) - 1.0) < 1e-5
        assert visits.sum() == 24 and action in legal and visits[action] == visits.max()
        assert rv == SM.sign(t.nodes[0].seat) * t.nodes[0].W / t.nodes[0].N


def test_zero_c_scale_gives_the_renormalised_prior(oracle):
    for g, st in enumerate(roots(oracle, 6)):
        t, (_a, policy, _v, _q, _rv) = search(st, 16, 16, gumbel_for(g), c_scale=0.0)
        root = t.nodes[0]
        edges = t._edges(root)
        s = G.Stats(edges, root.prior, root.seat, t.vhat(root), 50.0, 0.0)
        legal = SM.legal_ids(root.mask)
        p = np.array([float(root.prior[a]) for a in legal])
        pi = np.array([s.pi(a, n, w) for a, n, w, _c in edges])
        assert np.abs(pi - p / p.sum()).max() < 1e-12
        assert np.abs(policy[legal] - p / p.sum()).max() < 1e-7


def test_node_value_is_the_node_evaluation(oracle):
    """in 8.6 a node's own evaluation is what remains of W after its children: exact with dyadic values"""

    def dyadic(leaf):
        prior, v = hash_eval(leaf)
        return prior, np.float32(round(float(v) * 8) / 8)

    checked = 0
    for g, st in enumerate(roots(oracle, 6)):
        for ev, exact in ((dyadic, True), (hash_eval, False)):
            t, _ = search(st, 32, 16, gumbel_for(g), evaluate=ev)
            for j, v in t.evals.items():
                nd = t.nodes[j]
                got = t.vhat(nd)
                assert got == v if exact else abs(got - v) < 1e-12, (g, j)
                checked += 1
    assert checked > 300


def test_nan_and_zero_priors_still_select_a_legal_id():
    rs = np.random.RandomState(5)
    nan = float("nan")
    legal = sorted(rs.choice(SM.N_ACTIONS, 12, replace=False).tolist())
    for trial in range(40):
        prior = rs.uniform(0, 1, SM.N_ACTIONS).astype(np.float32)
        gum = rs.gumbel(size=SM.N_ACTIONS).astype(np.float32)
        if trial % 4 == 0:
            prior[:] = nan
        elif trial % 4 == 1:
            prior[legal[::2]] = nan
            gum[legal[1::3]] = nan
        elif trial % 4 == 2:
            prior[:] = 0.0  # a node created terminal in one world (zero prior), reached alive in another
        else:
            gum[:] = nan
        edges = [(a, int(rs.randint(0, 4)) if i % 2 else 0, nan if trial % 8 == 1 and i == 1 else float(rs.uniform(-3, 3)), i + 1)
                 for i, a in enumerate(legal)]
        edges = [(a, n, w if n else 0.0, c if n else None) for a, n, w, c in edges]
        for root in (False, True):
            a, _c = G.select(edges, prior, trial % 2, 0.25, root, gum, 3, 8, 4, 50.0, 0.1)
            assert a in legal, (trial, root)
        action, policy = G.read_out(edges, prior, 0, 0.0, gum, 50.0, 0.1)
        assert action in legal and (policy[np.setdiff1d(np.arange(SM.N_ACTIONS), legal)] == 0).all()
        if trial % 4 == 2:
            s = G.Stats(edges, prior, 0, 0.0, 50.0, 0.1)
            assert not math.isnan(s.vmix) and s.esum >= 1.0 and abs(float(policy.astype(np.float64).sum()) - 1.0) < 1e-5
    assert G.read_out([], prior, 0, 0.0, gum, 50.0, 0.1)[0] == G.NO_ACTION


def test_information_set_model_reads_out_by_root_ids(oracle):
    live = [st for st in records() if not ended(st)][::40][:6]
    for g, st in enumerate(live):
        sims = 16
        t = G.ISGumbelTreeModel(sims + 1)
        gum = gumbel_for(50 + g)
        worlds = [D.determinize(st, k) for k in keys(sims + 1, 900 + g)]
        leaf = t.begin(worlds[0])
        for k in range(1, sims + 1):
            leaf = t.simulate(worlds[k], *hash_eval(leaf), gum, k, sims, 8)
        action, policy, visits, q, rv = t.end(*hash_eval(leaf), gum)
        ids = [a for a in range(SM.N_ACTIONS) if t.root_code[a] != G.NONE_CODE]
        assert visits.sum() == sims and action in ids and visits[action] == visits.max()
        assert (policy[np.setdiff1d(np.arange(SM.N_ACTIONS), ids)] == 0).all()
        assert abs(float(policy.astype(np.float64).sum()) - 1.0) < 1e-5


def test_abi_symbols_and_frames():
    import __graft_entry__ as g
    g.build()
    from monsoon_b200 import _lib
    lib = _lib.load()
    names = ("sb_search_simulate_gumbel", "sb_search_end_gumbel", "sb_ismcts_simulate_gumbel", "sb_ismcts_end_gumbel")
    for nm in names:
        assert hasattr(lib, nm) and nm in _lib.SIGNATURES, nm
    assert lib.sb_abi_version() == 5
    frames = kernel_frames()
    for k in ("k_search_simulate_gumbel", "k_search_end_gumbel", "k_ismcts_simulate_gumbel", "k_ismcts_end_gumbel"):
        got = [v for name, v in frames.items() if k in name]
        assert len(got) == 1 and got[0] <= MAX_STACK, (k, got)


@pytest.mark.parametrize("bad", [dict(num_simulations=0), dict(max_considered=0), dict(max_considered=157), dict(c_visit=-1.0),
                                 dict(c_scale=float("nan"))])
def test_classes_refuse_bad_arguments_without_a_gpu(bad):
    from monsoon_b200.search import _gumbel_args
    kw = dict(num_simulations=8, max_considered=16, c_visit=50.0, c_scale=0.1)
    kw.update(bad)
    with pytest.raises(ValueError):
        _gumbel_args(**kw)

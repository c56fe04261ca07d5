"""GPU: the Gumbel searches' read-out (action and improved policy of GumbelMCTS / InformationSetGumbelMCTS) against an
independent float64 statement of mctx's gumbel_muzero_policy read-out.

test_gpu_gumbel.py compares the kernels with sb_gumbel_model, which restates DESIGN 8.9 with the library's own log and exp;
a formula misread the same way in both would pass there.  The reference below is written from mctx instead
(_compute_mixed_value, qtransform_completed_by_mix_value, the improved policy softmax(logits + sigma(completed q)) and
score_considered for the action), with numpy's log and exp, over what a run exposes: the root's prior and value from the
evaluator's k = 0 call (the node value 8.9 recovers is that evaluation, up to rounding) and the returned visits and q.
Where 8.9 documents a difference from mctx, the reference follows 8.9: min and max of the completed q run over the legal
ids only.
"""
import numpy as np
import pytest
import torch

import sb_oracle as O
import sb_search_model as M
from monsoon_b200.search import GumbelMCTS, InformationSetGumbelMCTS
from sb_ismcts_model import representatives
from test_gpu_determinize import mixed_roots
from test_gpu_search import env_roots

pytestmark = pytest.mark.gpu

NO_ACTION = 255
F32_TINY = float(np.finfo(np.float32).tiny)
F32_MIN_SUBNORMAL = 2.0 ** -149


def mctx_read_out(prior, value, visits, q, legal, gumbel, c_visit, c_scale):
    """float64 (improved policy over the 156 ids, action scores over the legal ids) of mctx's gumbel_muzero_policy at a
    root with legal ids `legal`, raw value `value` and the prior row `prior` as logits log(prior)"""
    p = prior[legal].astype(np.float64)
    n = visits[legal].astype(np.float64)
    with np.errstate(divide="ignore"):
        logits = np.log(p)
    # qtransform_completed_by_mix_value: prior_probs = softmax(logits) over the legal ids, floored at the f32 tiny
    probs = np.maximum(F32_TINY, p / p.sum())
    seen = n > 0
    weighted_q = (probs[seen] * q[legal][seen]).sum() / probs[seen].sum() if seen.any() else 0.0
    mixed = (value + n.sum() * weighted_q) / (n.sum() + 1.0)
    completed = np.where(seen, q[legal], mixed)
    completed = (completed - completed.min()) / max(completed.max() - completed.min(), 1e-8)
    sigma = (c_visit + n.max()) * c_scale * completed
    z = logits + sigma
    e = np.exp(z - z.max())
    policy = np.zeros(M.N_ACTIONS)
    policy[legal] = e / e.sum()
    # score_considered: argmax over the most visited ids of max(-1e9, g + logits - max logits + sigma)
    score = np.maximum(-1e9, gumbel[legal].astype(np.float64) + (logits - logits.max()) + sigma)
    score[n != n.max()] = -np.inf
    return policy, score


def root_legal_sets(roots, max_steps, information_set):
    """A(root): the legal ids (8.6), or the lowest legal id of each move code (8.8); empty for a finished root"""
    out = []
    for rec in roots:
        if M.over(rec, max_steps):
            out.append([])
        else:
            out.append(representatives(rec.copy()) if information_set else M.legal_ids(O.legal_mask(rec.copy())))
    return out


class Evaluator:
    """priors and values from a seeded host stream; the k = 0 call (the roots) gets the edge cases by row:
    0 uniform random, 1 f32 subnormal / 1e-30 / 0 entries at legal ids, 2 unnormalised (sum 7 over the legal ids),
    3 a peaked row, 4 value 0 at every call of the tree (all q equal: the 1e-8 floor of the rescale), 5 like 0"""

    def __init__(self, device, seed):
        self.device, self.rs = device, np.random.default_rng(seed)

    def __call__(self, leaf, k):
        masks = leaf["masks"].cpu().numpy()
        n = masks.shape[0]
        prior = self.rs.uniform(0.01, 1.0, (n, M.N_ACTIONS)).astype(np.float32)
        value = self.rs.uniform(-1.0, 1.0, n).astype(np.float32)
        value[4::6] = 0.0
        if k == 0:
            for i in range(n):
                legal = M.legal_ids(masks[i])
                if i % 6 == 1:
                    specials = np.array([1e-40, 2.0 ** -149, 1e-30, 0.0], dtype=np.float32)
                    prior[i, legal[1::2]] = specials[np.arange(len(legal[1::2])) % 4]
                elif i % 6 == 2 and legal:
                    prior[i, legal] = (7.0 * self.rs.dirichlet(np.ones(len(legal)))).astype(np.float32)
                elif i % 6 == 3:
                    prior[i, legal[len(legal) // 2:]] = 1e-3
            self.root_prior, self.root_value = prior.copy(), value.copy()
        return torch.from_numpy(prior).to(self.device), torch.from_numpy(value).to(self.device)


def noise(n, seed):
    u = np.random.default_rng(seed).uniform(1e-12, 1.0, (n, M.N_ACTIONS))
    return (-np.log(-np.log(u))).astype(np.float32)


@pytest.fixture(scope="module")
def roots(engine):
    r = mixed_roots(engine, 192, 71)
    pool = env_roots(engine, 256, 72, plies=7)
    single = [i for i, a in enumerate(root_legal_sets(pool.cpu().numpy(), 400, False)) if len(a) == 1]
    r = torch.cat([r, pool[single[:16]]])
    host = r.cpu().numpy()
    sizes = [len(a) for a in root_legal_sets(host, 400, False)]
    seats = [M.seat(rec) for rec, s in zip(host, sizes) if s]
    # the cases the read-out must cover: SECOND-to-move roots, one legal id, finished roots
    assert sizes.count(1) >= 5 and sizes.count(0) >= 5 and 0 < sum(seats) < len(seats)
    return r


@pytest.mark.parametrize("information_set", [False, True])
@pytest.mark.parametrize("sims", [1, 8, 32])
@pytest.mark.parametrize("max_considered", [1, 4, 16])
def test_read_out_is_mctx(engine, roots, information_set, sims, max_considered):
    n = roots.shape[0]
    host = roots.cpu().numpy()
    sets = root_legal_sets(host, 400, information_set)
    finished_sets = [representatives(rec.copy()) if not a else None for rec, a in zip(host, sets)]
    gumbel = noise(n, sims * 31 + max_considered)
    g_dev = torch.from_numpy(gumbel).to(engine.device)
    checked = floors = 0
    for c_scale in (0.0, 0.1, 1.0):
        for c_visit in (0.0, 50.0):
            cls = InformationSetGumbelMCTS if information_set else GumbelMCTS
            search = cls(n, sims, max_considered, c_visit, c_scale, seed=sims, engine=engine)
            ev = Evaluator(engine.device, sims + max_considered)
            action, policy, visits, q, _rv = (t.cpu().numpy() for t in search.run(roots, ev, gumbel=g_dev))
            for i in range(n):
                legal = sets[i]
                if not legal:
                    # a finished root, where mctx defines no read-out: 8.9 plays nothing.  8.6 has an empty A, so the policy
                    # is 0.  8.8's A is the stored root codes (the legal representatives); the root keeps a zero prior, so
                    # every logit is -1e9, every sigma 0 and the policy uniform over A.
                    assert action[i] == NO_ACTION, i
                    want = np.zeros(M.N_ACTIONS)
                    if information_set and finished_sets[i]:
                        want[finished_sets[i]] = 1.0 / len(finished_sets[i])
                    assert np.array_equal(policy[i], want.astype(np.float32)), (i, np.flatnonzero(policy[i]), finished_sets[i])
                    continue
                want, score = mctx_read_out(ev.root_prior[i], float(ev.root_value[i]), visits[i], q[i], legal, gumbel[i], c_visit,
                                            c_scale)
                got = policy[i].astype(np.float64)
                assert not np.delete(got, legal).any(), i
                tol = 2.0 * np.spacing(np.float32(want)).astype(np.float64)
                ok = (np.abs(got - want) <= tol) | ((want < F32_MIN_SUBNORMAL) & (got == 0.0))
                assert ok.all(), (i, c_scale, c_visit, np.flatnonzero(~ok)[:5], got[~ok][:5], want[~ok][:5])
                order = np.argsort(-score, kind="stable")
                margin = score[order[0]] - (score[order[1]] if len(order) > 1 else -np.inf)
                if margin > 1e-9:
                    assert action[i] == legal[order[0]], (i, c_scale, c_visit, action[i], legal[order[0]], margin)
                    checked += 1
                vis = visits[i][legal] > 0
                floors += bool(np.ptp(np.where(vis, q[i][legal], 0.0)) == 0.0 and float(ev.root_value[i]) == 0.0)
    live = sum(1 for a in sets if a)
    assert checked >= 3 * live and floors > 0, (checked, live, floors)

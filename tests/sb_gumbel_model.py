"""TEST INFRASTRUCTURE -- plain-Python statement of the Gumbel search (sb_search_simulate_gumbel / sb_search_end_gumbel,
sb_ismcts_simulate_gumbel / sb_ismcts_end_gumbel, include/sb_b200.h, DESIGN.md 8.9) over the tree models of sb_search_model
and sb_ismcts_model, which keep begin, expansion, emission and backup.  Only selection and the read-out are restated.

Python floats are IEEE doubles with correctly rounded + - * /, and log / exp are the oracle's sbo_det_log / sbo_det_exp, the
C statement of the kernels' es_log / es_exp, so every quantity below is the kernel's bit for bit when the sums run in the
kernel's order: 8.6 in increasing id order; 8.8 during simulate over the children newest first (the sibling walk), then
the representative ids without a child in increasing order, and at the end in increasing root id order.  The product
package never imports it.
"""
import numpy as np

import sb_oracle as O
from sb_ismcts_model import NONE_CODE, ISTreeModel, code, hand, representatives
from sb_search_model import N_ACTIONS, TreeModel, legal_ids, sign

NO_ACTION = 255
TINY = 2.0 ** -126
INF = float("inf")


def det_log(x):
    return O.lib().sbo_det_log(x)


def det_exp(y):
    return O.lib().sbo_det_exp(y)


def seq(m, S):
    """mctx's get_sequence_of_considered_visits(m, S), as the loop of sb_gumbel.cuh's header"""
    if m <= 1:
        return list(range(S))
    L = (m - 1).bit_length()  # ceil(log2 m)
    visits, k, out = [0] * m, m, []
    while len(out) < S:
        extra = max(1, S // (L * k))
        for _ in range(extra):
            out += visits[:k]
            for i in range(k):
                visits[i] += 1
        k = max(2, k // 2)
    return out[:S]


def logit(p):
    d = float(np.float32(p))
    return det_log(d) if d > 0.0 else -1e9


def ptilde(p):
    d = float(np.float32(p))
    return d if d > TINY else TINY


class Stats:
    """the per-node quantities of the rule from the edges [(act, n, W, child)] of node nd (prior f32[156], seat), in order"""

    def __init__(self, edges, prior, seat_, vhat, c_visit, c_scale, target=-1):
        self.edges, self.prior, self.sgn = edges, prior, sign(seat_)
        self.sum_n = sum(n for _a, n, _w, _c in edges)
        self.max_n = max([0] + [n for _a, n, _w, _c in edges])
        self.considered = sum(1 for _a, n, _w, _c in edges if n == target)
        sp, spq, visited = 0.0, 0.0, False
        for a, n, w, _c in edges:
            if n > 0:
                pt = ptilde(prior[a])
                visited = True
                sp = sp + pt
                spq = spq + pt * ((self.sgn * w) / float(n))
        mix = float(self.sum_n) * (spq / sp) if visited else 0.0
        self.vmix = (vhat + mix) / float(1 + self.sum_n)
        qmin, qmax = INF, -INF
        for a, n, w, _c in edges:
            q = self.q(n, w)
            if q < qmin:
                qmin = q
            if q > qmax:
                qmax = q
        d = qmax - qmin
        self.qmin, self.qden = qmin, d if d > 1e-8 else 1e-8
        self.sig = (c_visit + float(self.max_n)) * c_scale
        zmax = -INF
        for a, n, w, _c in edges:
            z = self.z(a, n, w)
            if z > zmax:
                zmax = z
        self.zmax = zmax
        esum = 0.0
        for a, n, w, _c in edges:
            esum = esum + self.e(self.z(a, n, w))
        self.esum = esum

    def q(self, n, w):
        return (self.sgn * w) / float(n) if n > 0 else self.vmix

    def sigma(self, n, w):
        return self.sig * ((self.q(n, w) - self.qmin) / self.qden)

    def z(self, a, n, w):
        return logit(self.prior[a]) + self.sigma(n, w)

    def e(self, z):
        d = z - self.zmax
        return det_exp(d) if d >= -700.0 else 0.0

    def pi(self, a, n, w):
        return self.e(self.z(a, n, w)) / self.esum


def argmax(cands):
    """(act, child) of the best (score, act, child), ties to the lower id, NaN never wins; None when nothing scores"""
    best, best_score = None, -INF
    for score, a, c in cands:
        if score > best_score or (score == best_score and best is not None and a < best[0]):
            best, best_score = (a, c), score
    return best


def select(edges, prior, seat_, vhat, root, gumbel, sim, S, max_considered, c_visit, c_scale):
    """(act, child) at a node: the interior rule, or the root's at call sim; (-1, None) when there is no edge"""
    if not edges:
        return -1, None
    lo = min(edges, key=lambda t: t[0])
    if not root:
        s = Stats(edges, prior, seat_, vhat, c_visit, c_scale)
        inv = float(1 + s.sum_n)
        best = argmax((s.pi(a, n, w) - float(n) / inv, a, c) for a, n, w, c in edges)
    else:
        m = min(max_considered, len(edges))
        target = seq(m, S)[sim - 1]
        s = Stats(edges, prior, seat_, vhat, c_visit, c_scale, target)
        pool = [t for t in edges if t[1] == target] if s.considered else edges

        def floor(x):
            return x if x > -1e9 else -1e9
        best = argmax((floor((float(gumbel[a]) + logit(prior[a])) + s.sigma(n, w)), a, c) for a, n, w, c in pool)
    return best if best is not None else (lo[0], lo[3])


def read_out(edges, prior, seat_, vhat, gumbel, c_visit, c_scale):
    """(action, policy f32[156]) at the root after the last backup"""
    policy = np.zeros(N_ACTIONS, dtype=np.float32)
    if not edges:
        return NO_ACTION, policy
    s = Stats(edges, prior, seat_, vhat, c_visit, c_scale)
    for a, n, w, _c in edges:
        policy[a] = np.float32(s.pi(a, n, w))
    top = [t for t in edges if t[1] == s.max_n and t[1] > 0]
    if not top:
        return NO_ACTION, policy
    best = argmax(((float(gumbel[a]) + logit(prior[a])) + s.sigma(n, w), a, c) for a, n, w, c in top)
    return (best[0] if best is not None else min(t[0] for t in top)), policy


class GumbelTreeModel(TreeModel):
    """TreeModel with the Gumbel rule: simulate(prior, value, gumbel, sim, S, max_considered, c_visit, c_scale) returns the
    emitted leaf; end(prior, value, gumbel, c_visit, c_scale) returns (action, policy, visits, q, root_value)."""

    def _edges(self, nd):
        out = []
        for a in legal_ids(nd.mask):
            c = nd.children.get(a)
            out.append((a, self.nodes[c].N, self.nodes[c].W, c) if c is not None else (a, 0, 0.0, None))
        return out

    def vhat(self, nd):
        sn, sw = 0, 0.0
        for a in legal_ids(nd.mask):
            c = nd.children.get(a)
            if c is not None:
                sn += self.nodes[c].N
                sw = sw + self.nodes[c].W
        den = nd.N - sn
        return 0.0 if den < 1 else (sign(nd.seat) * (nd.W - sw)) / float(den)

    def select(self, nd, c_puct, fpu):
        g = self._gumbel_call
        a, _c = select(self._edges(nd), nd.prior, nd.seat, self.vhat(nd), nd is self.nodes[0], *g)
        return a

    def simulate(self, prior, value, gumbel, sim, S, max_considered=16, c_visit=50.0, c_scale=0.1):
        self._gumbel_call = (gumbel, sim, S, max_considered, c_visit, c_scale)
        return super().simulate(prior, value, None, None)

    def end(self, prior, value, gumbel, c_visit=50.0, c_scale=0.1):
        visits, q, rv = super().end(prior, value)
        root = self.nodes[0]
        if root.terminal:
            return NO_ACTION, np.zeros(N_ACTIONS, dtype=np.float32), visits, q, rv
        action, policy = read_out(self._edges(root), root.prior, root.seat, self.vhat(root), gumbel, c_visit, c_scale)
        return action, policy, visits, q, rv


class ISGumbelTreeModel(ISTreeModel):
    """ISTreeModel with the Gumbel rule: simulate(world, prior, value, gumbel, sim, S, max_considered, c_visit, c_scale);
    end(prior, value, gumbel, c_visit, c_scale) returns (action, policy, visits, q, root_value) by the root's action ids."""

    def _children(self, nd):
        """the children of nd in the kernel's sibling-walk order (newest first)"""
        return sorted(nd.children.values(), reverse=True)

    def vhat(self, nd):
        sn, sw = 0, 0.0
        for c in self._children(nd):
            sn += self.nodes[c].N
            sw = sw + self.nodes[c].W
        den = nd.N - sn
        return 0.0 if den < 1 else (sign(nd.seat) * (nd.W - sw)) / float(den)

    def _edges(self, nd, rec):
        h = hand(rec)
        rep = {code(h, a): a for a in representatives(rec)}
        out, seen = [], set()
        for c in self._children(nd):
            a = rep.get(self.nodes[c].code)
            if a is not None and a not in seen:
                seen.add(a)
                out.append((a, self.nodes[c].N, self.nodes[c].W, c))
        out += [(a, 0, 0.0, None) for a in sorted(rep.values()) if a not in seen]
        return out

    def select(self, nd, rec, c_puct, fpu):
        return select(self._edges(nd, rec), nd.prior, nd.seat, self.vhat(nd), nd is self.nodes[0], *self._gumbel_call)

    def simulate(self, world, prior, value, gumbel, sim, S, max_considered=16, c_visit=50.0, c_scale=0.1):
        self._gumbel_call = (gumbel, sim, S, max_considered, c_visit, c_scale)
        return super().simulate(world, prior, value, None, None)

    def end(self, prior, value, gumbel, c_visit=50.0, c_scale=0.1):
        visits, q, rv = super().end(prior, value)
        root = self.nodes[0]
        edges = []
        for a in range(N_ACTIONS):
            if self.root_code[a] == NONE_CODE:
                continue
            c = root.children.get(self.root_code[a])
            edges.append((a, self.nodes[c].N, self.nodes[c].W, c) if c is not None else (a, 0, 0.0, None))
        action, policy = read_out(edges, root.prior, root.seat, self.vhat(root), gumbel, c_visit, c_scale)
        return action, policy, visits, q, rv

"""TEST INFRASTRUCTURE -- plain-Python statement of several leaves per tree per call under virtual loss
(sb_search_simulate_batch / sb_search_end_batch, include/sb_b200.h, DESIGN.md 8.11), one tree at a time, over TreeModel of
sb_search_model (begin and the read-out are its own; sb_reuse_model's advance composes with it through from_tree).

Python floats are IEEE doubles with correctly rounded + - * / and math.sqrt, so the scores below are the kernel's bit for
bit.  The product package never imports it.
"""
import math

import numpy as np

import sb_oracle as O
import sb_search_model as M
from sb_search_model import EVAL, FULL, TERMINAL, legal_ids, sign

COLLISION = 3
BATCH = 3  # tree kind of a batch-form tree: the L slots are pending


class Pending:
    """a node taken by a selection of the current call, before the expansion writes its record"""

    def __init__(self, parent, action):
        self.parent, self.action = parent, action
        self.N, self.W = 0, 0.0
        self.children = {}


class BatchTreeModel(M.TreeModel):
    """One tree of L slots: begin() as TreeModel; simulate_batch(prior f32[L,156], value f32[L], c_puct, fpu, vl) returns
    the L emitted leaves (TreeModel's tuples); end_batch(prior, value) returns (visits, q, root_value).  self.V holds the
    virtual visits (all zero between calls), self.slots the pending (node, kind) pairs."""

    def __init__(self, root, max_nodes, leaves, max_steps=400):
        super().__init__(root, max_nodes, max_steps)
        self.L = leaves
        self.slots = []
        self.V = [0] * max_nodes

    @classmethod
    def from_tree(cls, t, leaves):
        """the batch model of a TreeModel in header form (after begin or sb_reuse_model's advance)"""
        b = cls(t.root, t.max_nodes, leaves, t.max_steps)
        b.nodes, b.leaf, b.kind = t.nodes, t.leaf, t.kind
        return b

    def _add(self, k, v):
        j = k
        while j >= 0:
            self.nodes[j].N += 1
            self.nodes[j].W = self.nodes[j].W + v
            j = self.nodes[j].parent

    def _backup_node(self, k, kind, prior, value):
        nd = self.nodes[k]
        if kind == TERMINAL:
            v = float(nd.tval)
        else:
            nd.prior = np.asarray(prior, dtype=np.float32).copy()
            v = sign(nd.seat) * float(np.float32(value))
        self._add(k, v)

    def _backup_batch(self, prior, value):
        """the header-form leaf from slot 0, or the pending slots in ascending order; the tree is then batch form"""
        if self.kind == FULL:
            return False
        if self.kind in (EVAL, TERMINAL):
            self._backup_node(self.leaf, self.kind, prior[0], value[0])
            self.V = [0] * self.max_nodes
        else:
            for l, (k, kind) in enumerate(self.slots):
                if kind in (EVAL, TERMINAL):
                    self._backup_node(k, kind, prior[l], value[l])
        self.leaf, self.kind = 0, BATCH
        return True

    def _mark(self, j, d):
        while j >= 0:
            self.V[j] = self.V[j] + 1 if d else 0
            j = self.nodes[j].parent

    def select_v(self, j, c_puct, fpu, vl):
        nd, V = self.nodes[j], self.V
        sgn, sq = sign(nd.seat), math.sqrt(float(nd.N + V[j]))
        best, best_score = -1, 0.0
        for a in legal_ids(nd.mask):
            c = nd.children.get(a)
            na = self.nodes[c].N + V[c] if c is not None else 0
            q = ((sgn * self.nodes[c].W) - (float(vl) * float(V[c]))) / float(na) if na else float(fpu)
            u = ((float(c_puct) * float(nd.prior[a])) * sq) / float(1 + na)
            score = q + u
            if best < 0 or score > best_score:
                best, best_score = a, score
        return best

    def _stop(self):
        self.kind = FULL
        self.slots = [(0, FULL)] * self.L
        return [self._emit(0, FULL) for _ in range(self.L)]

    def simulate_batch(self, prior, value, c_puct, fpu, vl):
        if not self._backup_batch(prior, value) or len(self.nodes) >= self.max_nodes:
            return self._stop()
        start = len(self.nodes)
        slots = []
        for _ in range(self.L):
            j, kind = 0, None
            while kind is None:
                if j >= start:
                    kind = COLLISION
                elif self.nodes[j].terminal:
                    kind = TERMINAL
                else:
                    a = self.select_v(j, c_puct, fpu, vl)
                    if a < 0:  # no legal action: the tree stops, the nodes taken in this call are dropped
                        for k in range(start, len(self.nodes)):
                            del self.nodes[self.nodes[k].parent].children[self.nodes[k].action]
                        del self.nodes[start:]
                        return self._stop()
                    c = self.nodes[j].children.get(a)
                    if c is None:
                        if len(self.nodes) >= self.max_nodes:
                            break
                        self.nodes.append(Pending(j, a))
                        c = len(self.nodes) - 1
                        self.nodes[j].children[a] = c
                        kind = EVAL
                    j = c
            if kind is None:
                break
            slots.append((j, kind))
            self._mark(j, 1)
        for k, _kind in slots:
            self._mark(k, 0)
        slots += [(0, FULL)] * (self.L - len(slots))
        out = []
        for l, (k, kind) in enumerate(slots):  # the expansion pass: new records, then every slot's leaf outputs
            if kind == EVAL:
                p = self.nodes[k]
                rec = O.step(self.nodes[p.parent].rec.copy(), p.action)
                self.nodes[k] = M.Node(rec, p.parent, p.action, self.max_steps)
                kind = TERMINAL if self.nodes[k].terminal else EVAL
                slots[l] = (k, kind)
                out.append(self._emit(k, kind))
            elif kind == TERMINAL:
                out.append(self._emit(k, kind))
            else:
                out.append(self._emit(0, kind))
        self.slots = slots
        return out

    def end_batch(self, prior, value):
        self._backup_batch(prior, value)
        self.kind = FULL
        return self.end(None, None)  # TreeModel.end: nothing is pending any more, only the read-out

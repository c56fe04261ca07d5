"""TEST INFRASTRUCTURE -- plain-Python statement of several leaves per tree per call for the information-set search, under
virtual loss (sb_ismcts_simulate_batch / sb_ismcts_end_batch, include/sb_b200.h, DESIGN.md 8.12), one tree at a time, over
ISTreeModel of sb_ismcts_model (begin and the read-out are its own; sb_reuse_model's advance composes with it through
from_tree).

The definition is sequential: slot l walks from the root through its own world l, as ISTreeModel.simulate does, with the
visits of the earlier slots of the same call counted as virtual visits V carrying a loss.  A node taken by an earlier slot
of the call stops a walk that reaches it (COLLISION).  Python floats are IEEE doubles with correctly rounded + - * / and
math.sqrt, so the scores below are the kernel's bit for bit.  The product package never imports it.
"""
import math

import numpy as np

import sb_ismcts_model as I
import sb_oracle as O
from sb_search_model import EVAL, FULL, TERMINAL, first_value, over, seat, sign

COLLISION = 3
BATCH = 3  # tree kind of a batch-form tree: the L slots are pending


class ISBatchTreeModel(I.ISTreeModel):
    """One tree of L slots: begin(world) as ISTreeModel; simulate_batch(worlds u8[L,512], prior f32[L,156], value f32[L],
    c_puct, fpu, vl) returns the L emitted leaves (ISTreeModel's tuples); end_batch(prior, value) returns (visits, q,
    root_value).  self.V holds the virtual visits (all zero between calls), self.slots the pending (node, kind, terminal
    value) triples."""

    def __init__(self, max_nodes, leaves, max_steps=400):
        super().__init__(max_nodes, max_steps)
        self.L = leaves
        self.slots = []
        self.V = [0] * max_nodes

    @classmethod
    def from_tree(cls, t, leaves):
        """the batch model of an ISTreeModel in header form (after begin or sb_reuse_model's ismcts_advance)"""
        b = cls(t.max_nodes, leaves, t.max_steps)
        b.nodes, b.leaf, b.kind, b.tval, b.root_code = t.nodes, t.leaf, t.kind, t.tval, t.root_code
        return b

    def _backup_node(self, k, kind, tval, prior, value):
        nd = self.nodes[k]
        if kind == TERMINAL:
            v = float(tval)
        else:
            nd.prior = np.asarray(prior, dtype=np.float32).copy()
            v = sign(nd.seat) * float(np.float32(value))
        j = k
        while j >= 0:
            self.nodes[j].N += 1
            self.nodes[j].W = self.nodes[j].W + v
            j = self.nodes[j].parent

    def _backup_batch(self, prior, value):
        """the header-form leaf from slot 0, or the pending slots in ascending order; the tree is then batch form"""
        if self.kind == FULL:
            return False
        if self.kind in (EVAL, TERMINAL):
            self._backup_node(self.leaf, self.kind, self.tval, prior[0], value[0])
            self.V = [0] * self.max_nodes
        else:
            for l, (k, kind, tval) in enumerate(self.slots):
                if kind in (EVAL, TERMINAL):
                    self._backup_node(k, kind, tval, prior[l], value[l])
        self.leaf, self.kind = 0, BATCH
        return True

    def _mark(self, j, d):
        while j >= 0:
            self.V[j] = self.V[j] + 1 if d else 0
            j = self.nodes[j].parent

    def select_v(self, j, rec, c_puct, fpu, vl):
        """(action id, child index or None) at node j in the world whose record there is rec: ISTreeModel.select with
        n_a = N + V and q = ((sgn * W) - vl * V) / n_a"""
        nd, V = self.nodes[j], self.V
        sgn, sq = sign(nd.seat), math.sqrt(float(nd.N + V[j]))
        h = I.hand(rec)
        best, best_child, best_score = -1, None, 0.0
        for a in I.representatives(rec):
            c = nd.children.get(I.code(h, a))
            na = self.nodes[c].N + V[c] if c is not None else 0
            q = ((sgn * self.nodes[c].W) - (float(vl) * float(V[c]))) / float(na) if na else float(fpu)
            u = ((float(c_puct) * float(nd.prior[a])) * sq) / float(1 + na)
            score = q + u
            if best < 0 or score > best_score:
                best, best_child, best_score = a, c, score
        return best, best_child

    def _stop(self, worlds):
        self.kind = FULL
        self.slots = [(0, FULL, 0)] * self.L
        return [self._emit(np.asarray(w, dtype=np.uint8), FULL) for w in worlds]

    def simulate_batch(self, worlds, prior, value, c_puct, fpu, vl):
        assert len(worlds) == self.L
        if not self._backup_batch(prior, value) or len(self.nodes) >= self.max_nodes:
            return self._stop(worlds)
        start = len(self.nodes)
        slots, out, ends = [], [], []
        for w in worlds:
            root = np.array(w, dtype=np.uint8, copy=True)
            rec, j, kind, tval = root.copy(), 0, None, 0
            while kind is None:
                if j >= start:
                    kind, rec = COLLISION, root
                elif over(rec, self.max_steps):
                    kind, tval = TERMINAL, first_value(rec)
                else:
                    a, c = self.select_v(j, rec, c_puct, fpu, vl)
                    if a < 0:  # no legal representative: the tree stops, the nodes taken in this call are dropped
                        for k in range(start, len(self.nodes)):
                            del self.nodes[self.nodes[k].parent].children[self.nodes[k].code]
                        del self.nodes[start:]
                        return self._stop(worlds)
                    cd = I.code(I.hand(rec), a)
                    rec = O.step(rec.copy(), a)
                    if c is None:
                        if len(self.nodes) >= self.max_nodes:
                            break
                        self.nodes.append(I.Node(j, cd, seat(rec)))
                        c = len(self.nodes) - 1
                        self.nodes[j].children[cd] = c
                        term = over(rec, self.max_steps)
                        kind, tval = (TERMINAL, first_value(rec)) if term else (EVAL, 0)
                    j = c
            if kind is None:
                break
            slots.append((0 if kind == COLLISION else j, kind, tval))
            out.append(self._emit(rec, kind))
            ends.append(j)
            self._mark(j, 1)
        for j in ends:
            self._mark(j, 0)
        full = len(slots)
        slots += [(0, FULL, 0)] * (self.L - full)
        out += [self._emit(np.asarray(w, dtype=np.uint8), FULL) for w in worlds[full:]]
        self.slots = slots
        return out

    def end_batch(self, prior, value):
        self._backup_batch(prior, value)
        self.kind = FULL
        return self.end(None, None)  # ISTreeModel.end: nothing is pending any more, only the read-out


def tail_bytes(max_nodes, leaves):
    """the per-tree tail after sb_ismcts_workspace_bytes: 16-byte slots {node, kind, terminal value, 0} and i32 V per node"""
    return (16 * leaves + 4 * max_nodes + 15) // 16 * 16


def workspace_bytes(n, max_nodes, leaves):
    """sb_ismcts_batch_workspace_bytes"""
    pre = I.workspace_bytes(n, max_nodes)
    if n < 0 or not 1 <= leaves <= 256 or (n > 0 and pre == 0):
        return 0
    return pre + n * tail_bytes(max_nodes, leaves)

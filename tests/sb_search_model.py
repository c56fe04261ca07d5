"""TEST INFRASTRUCTURE -- plain-Python statement of the batched tree search (sb_search_begin / sb_search_simulate /
sb_search_end, include/sb_b200.h), one tree at a time.

Built only on the pinned C oracle (step, legal_mask, observe, rollout_random).  Python floats are IEEE doubles with correctly
rounded + - * / and math.sqrt, so the PUCT scores below are the kernel's bit for bit.  The product package never imports it.
"""
import math

import numpy as np

import sb_oracle as O
from sb_layout import STATE_DTYPE

N_ACTIONS = 156
EVAL, TERMINAL, FULL = 0, 1, 2


def fields(st):
    return st.view(STATE_DTYPE)[0]


def seat(st):
    return 0 if int(fields(st)["player_sign"]) == 1 else 1


def over(st, max_steps):
    f = fields(st)
    return bool(f["pl"][0]["base"] < 0 or f["pl"][1]["base"] < 0 or f["err"] or f["steps"] >= max_steps)


def first_value(st):
    """game value for FIRST: +1 FIRST won, -1 SECOND won, 0 draw, timeout or engine status"""
    f = fields(st)
    if f["err"]:
        return 0
    l0, l1 = f["pl"][0]["base"] < 0, f["pl"][1]["base"] < 0
    return 1 if (l1 and not l0) else -1 if (l0 and not l1) else 0


def legal_ids(mask):
    return np.flatnonzero(np.unpackbits(np.ascontiguousarray(mask).view(np.uint8), bitorder="little")[:N_ACTIONS]).tolist()


def sign(s):
    return -1.0 if s else 1.0


class Node:
    def __init__(self, rec, parent, action, max_steps):
        self.rec = rec
        self.parent, self.action = parent, action
        self.mask = O.legal_mask(rec)
        self.seat = seat(rec)
        self.terminal = over(rec, max_steps)
        self.tval = first_value(rec) if self.terminal else 0
        self.prior = None
        self.children = {}
        self.N, self.W = 0, 0.0


class TreeModel:
    """One tree: begin() / simulate(prior, value, c_puct, fpu) return the emitted leaf
    (record, obs i32[27,5,4], obs_err, mask i32[5], to_move, kind); end(prior, value) returns (visits, q, root_value)."""

    def __init__(self, root, max_nodes, max_steps=400):
        self.root, self.max_nodes, self.max_steps = root.copy(), max_nodes, max_steps
        self.nodes = []
        self.leaf, self.kind = 0, FULL

    def _emit(self, j, kind):
        nd = self.nodes[j]
        obs, err = O.observe(nd.rec.copy())
        return nd.rec.copy(), obs, err, nd.mask.view(np.int32).copy(), nd.seat, kind

    def begin(self):
        self.nodes = [Node(self.root.copy(), -1, 155, self.max_steps)]
        self.leaf, self.kind = 0, TERMINAL if self.nodes[0].terminal else EVAL
        return self._emit(0, self.kind)

    def _backup(self, prior, value):
        if self.kind == FULL:
            return
        leaf = self.nodes[self.leaf]
        if self.kind == TERMINAL:
            v = float(leaf.tval)
        else:
            leaf.prior = np.asarray(prior, dtype=np.float32).copy()
            v = sign(leaf.seat) * float(np.float32(value))
        j = self.leaf
        while j >= 0:
            self.nodes[j].N += 1
            self.nodes[j].W = self.nodes[j].W + v
            j = self.nodes[j].parent

    def select(self, nd, c_puct, fpu):
        sgn, sq = sign(nd.seat), math.sqrt(float(nd.N))
        best, best_score = -1, 0.0
        for a in legal_ids(nd.mask):
            c = nd.children.get(a)
            na = self.nodes[c].N if c is not None else 0
            q = (sgn * self.nodes[c].W) / float(na) if na else float(fpu)
            u = ((float(c_puct) * float(nd.prior[a])) * sq) / float(1 + na)
            score = q + u
            if best < 0 or score > best_score:
                best, best_score = a, score
        return best

    def simulate(self, prior, value, c_puct, fpu):
        self._backup(prior, value)
        if self.kind == FULL or len(self.nodes) >= self.max_nodes:
            self.kind = FULL
            return self._emit(0, FULL)
        j = 0
        while not self.nodes[j].terminal:
            a = self.select(self.nodes[j], c_puct, fpu)
            c = self.nodes[j].children.get(a)
            if c is None:
                rec = O.step(self.nodes[j].rec.copy(), a)
                self.nodes.append(Node(rec, j, a, self.max_steps))
                k = len(self.nodes) - 1
                self.nodes[j].children[a] = k
                self.leaf, self.kind = k, TERMINAL if self.nodes[k].terminal else EVAL
                return self._emit(k, self.kind)
            j = c
        self.leaf, self.kind = j, TERMINAL
        return self._emit(j, TERMINAL)

    def end(self, prior, value):
        self._backup(prior, value)
        self.kind = FULL
        root = self.nodes[0]
        visits = np.zeros(N_ACTIONS, dtype=np.int32)
        q = np.full(N_ACTIONS, np.nan)
        for a, c in root.children.items():
            visits[a] = self.nodes[c].N
            if self.nodes[c].N:
                q[a] = (sign(root.seat) * self.nodes[c].W) / float(self.nodes[c].N)
        return visits, q, (sign(root.seat) * root.W) / float(root.N)


def rollout_eval(leaf, max_steps=400):
    """the rollout evaluator on one emitted leaf: (prior f32[156], value f32), the record is played out in place"""
    rec, _obs, _err, mask, to_move, _kind = leaf
    ids = legal_ids(mask)
    prior = np.zeros(N_ACTIONS, dtype=np.float32)
    prior[ids] = np.float32(1.0) / np.float32(len(ids))
    O.rollout_random(rec, max_steps)
    return prior, np.float32(first_value(rec) * (1 - 2 * to_move))

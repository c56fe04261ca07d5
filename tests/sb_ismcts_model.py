"""TEST INFRASTRUCTURE -- plain-Python statement of the information-set tree search (sb_ismcts_begin / sb_ismcts_simulate /
sb_ismcts_end, include/sb_b200.h), one tree at a time.

Built on the pinned C oracle (step, legal_mask, observe) and the helpers of sb_search_model.  The worlds are given, as to the
kernels (normally sb_determinize_model.determinize of the root under a fresh key per call).  Selection scans the world's legal
representative ids in increasing order with a strict >, which is the kernel's merged arg-max (children scored in one sibling
walk, then the ids without a child, ties to the lower id).  The product package never imports it.
"""
import math

import numpy as np

import sb_oracle as O
from sb_search_model import EVAL, FULL, N_ACTIONS, TERMINAL, fields, first_value, legal_ids, over, seat, sign

PASS_CODE = 4 << 24
NONE_CODE = 0xFFFFFFFF


def hand(rec):
    """the mover's (local_order's) hand cards, u8[4]"""
    f = fields(rec)
    return [int(c) for c in f["pl"][int(f["local_order"])]["hand_card"]]


def slot(a):
    """(hand slot, first slot of the kind, id distance between slots) of action id a; slot -1 for PASS"""
    if a < 64:
        return a >> 4, 0, 16
    if a < 148:
        return (a - 64) // 21, 0, 21
    if a < 152:
        return a - 148, 0, 1
    if a < 155:
        return a - 151, 1, 1
    return -1, 0, 1


def code(h, a):
    """the move code of action id a for the mover's hand h"""
    if a < 64:
        return h[a >> 4] << 16 | (a & 15)
    if a < 148:
        return 1 << 24 | h[(a - 64) // 21] << 16 | (a - 64) % 21
    if a < 152:
        return 2 << 24 | h[a - 148] << 16
    if a < 155:
        return 3 << 24 | h[a - 151] << 16 | h[0]
    return PASS_CODE


def representatives(rec):
    """the legal ids of rec that represent their code (no lower legal id with the same code), increasing"""
    h = hand(rec)
    legal = legal_ids(O.legal_mask(rec.copy()))
    seen, out = set(), []
    for a in legal:
        c = code(h, a)
        if c not in seen:
            seen.add(c)
            out.append(a)
    return out


class Node:
    def __init__(self, parent, code_, seat_):
        self.parent, self.code, self.seat = parent, code_, seat_
        self.children = {}  # code -> node index
        self.prior = np.zeros(N_ACTIONS, dtype=np.float32)
        self.N, self.W = 0, 0.0


class ISTreeModel:
    """One tree: begin(world) / simulate(world, prior, value, c_puct, fpu) return the emitted leaf
    (record, obs i32[27,5,4], obs_err, mask i32[5], to_move, kind), as sb_search_model.TreeModel; end(prior, value) returns
    (visits, q, root_value) by the root's action ids."""

    def __init__(self, max_nodes, max_steps=400):
        self.max_nodes, self.max_steps = max_nodes, max_steps
        self.nodes = []
        self.leaf, self.kind, self.tval = 0, FULL, 0
        self.root_code = [NONE_CODE] * N_ACTIONS
        self.path = []  # (node, world record) pairs of the last walk, root first

    @staticmethod
    def _emit(rec, kind):
        obs, err = O.observe(rec.copy())
        return rec.copy(), obs, err, O.legal_mask(rec.copy()).view(np.int32).copy(), seat(rec), kind

    def begin(self, world):
        world = np.array(world, dtype=np.uint8, copy=True)
        self.nodes = [Node(-1, NONE_CODE, seat(world))]
        h = hand(world)
        self.root_code = [NONE_CODE] * N_ACTIONS
        for a in representatives(world):
            self.root_code[a] = code(h, a)
        term = over(world, self.max_steps)
        self.leaf, self.kind, self.tval = 0, TERMINAL if term else EVAL, first_value(world) if term else 0
        self.path = [(0, world.copy())]
        return self._emit(world, self.kind)

    def _backup(self, prior, value):
        if self.kind == FULL:
            return
        leaf = self.nodes[self.leaf]
        if self.kind == TERMINAL:
            v = float(self.tval)
        else:
            leaf.prior = np.asarray(prior, dtype=np.float32).copy()
            v = sign(leaf.seat) * float(np.float32(value))
        j = self.leaf
        while j >= 0:
            self.nodes[j].N += 1
            self.nodes[j].W = self.nodes[j].W + v
            j = self.nodes[j].parent

    def select(self, nd, rec, c_puct, fpu):
        """(action id, child index or None) at node nd in the world whose record there is rec"""
        sgn, sq = sign(nd.seat), math.sqrt(float(nd.N))
        h = hand(rec)
        best, best_child, best_score = -1, None, 0.0
        for a in representatives(rec):
            c = nd.children.get(code(h, a))
            na = self.nodes[c].N if c is not None else 0
            q = (sgn * self.nodes[c].W) / float(na) if na else float(fpu)
            u = ((float(c_puct) * float(nd.prior[a])) * sq) / float(1 + na)
            score = q + u
            if best < 0 or score > best_score:
                best, best_child, best_score = a, c, score
        return best, best_child

    def simulate(self, world, prior, value, c_puct, fpu):
        self._backup(prior, value)
        rec = np.array(world, dtype=np.uint8, copy=True)
        self.path = [(0, rec.copy())]
        if self.kind == FULL or len(self.nodes) >= self.max_nodes:
            self.kind = FULL
            return self._emit(rec, FULL)
        j = 0
        while True:
            if over(rec, self.max_steps):
                self.leaf, self.kind, self.tval = j, TERMINAL, first_value(rec)
                return self._emit(rec, TERMINAL)
            a, c = self.select(self.nodes[j], rec, c_puct, fpu)
            cd = code(hand(rec), a)
            rec = O.step(rec.copy(), a)
            if c is None:
                self.nodes.append(Node(j, cd, seat(rec)))
                k = len(self.nodes) - 1
                self.nodes[j].children[cd] = k
                self.path.append((k, rec.copy()))
                term = over(rec, self.max_steps)
                self.leaf, self.kind, self.tval = k, TERMINAL if term else EVAL, first_value(rec) if term else 0
                return self._emit(rec, self.kind)
            j = c
            self.path.append((j, rec.copy()))

    def end(self, prior, value):
        self._backup(prior, value)
        self.kind = FULL
        root = self.nodes[0]
        visits = np.zeros(N_ACTIONS, dtype=np.int32)
        q = np.full(N_ACTIONS, np.nan)
        for a in range(N_ACTIONS):
            c = root.children.get(self.root_code[a]) if self.root_code[a] != NONE_CODE else None
            if c is not None and self.nodes[c].N:
                visits[a] = self.nodes[c].N
                q[a] = (sign(root.seat) * self.nodes[c].W) / float(self.nodes[c].N)
        return visits, q, (sign(root.seat) * root.W) / float(root.N)


def workspace_bytes(n, max_nodes):
    """sb_ismcts_workspace_bytes: a 656-byte header and max_nodes 656-byte nodes per tree"""
    return n * 656 * (1 + max_nodes) if n >= 0 and 1 <= max_nodes <= 1 << 24 else 0

"""TEST INFRASTRUCTURE -- plain-Python statement of tree reuse between moves (sb_search_advance / sb_ismcts_advance,
include/sb_b200.h, DESIGN.md 8.10) over the tree models of sb_search_model and sb_ismcts_model, one tree at a time.

An advance returns a new model, the tree the advance leaves in ws_dst, with the leaf it emits and the number of nodes kept.
The source model is the tree the finished search left in ws_src; it is not changed (the kernel consumes ws_src, the model
need not).  The product package never imports it.
"""
import copy

import numpy as np

import sb_ismcts_model as I
import sb_search_model as M
from sb_search_model import EVAL, FULL, N_ACTIONS, TERMINAL, over, seat


def kept_order(nodes, j, keep):
    """the first `keep` of node j and its descendants in creation order (increasing index): [old index], j first"""
    inside, order = {j}, [j]
    for k in range(j + 1, len(nodes)):
        if len(order) >= keep:
            break
        if nodes[k].parent in inside:
            inside.add(k)
            order.append(k)
    return order


def _carry(nodes, order):
    """copies of the kept nodes, renumbered: parent remapped (-1 at the root), children dicts keep only kept children"""
    new_index = {old: new for new, old in enumerate(order)}
    out = []
    for old in order:
        nd = copy.copy(nodes[old])
        nd.parent = new_index.get(nodes[old].parent, -1) if old != order[0] else -1
        nd.children = {key: new_index[c] for key, c in nodes[old].children.items() if c in new_index}
        if nd.prior is not None:
            nd.prior = nd.prior.copy()
        out.append(nd)
    return out


def search_match(src, root):
    """8.6: the lowest-index node of the finished tree src whose record equals root byte for byte, -1 if none (or src is
    not finished)"""
    if src is None or src.kind != FULL:
        return -1
    for k, nd in enumerate(src.nodes):
        if nd.rec.tobytes() == np.asarray(root, dtype=np.uint8).tobytes():
            return k
    return -1


def search_advance(src, root, max_nodes, keep, max_steps=400):
    """(new TreeModel, emitted leaf, kept) of sb_search_advance on one tree; src is the source TreeModel or None (a
    workspace that holds no finished tree)"""
    t = M.TreeModel(root, max_nodes, max_steps)
    j = search_match(src, root) if src is not None and src.max_steps == max_steps else -1
    if j < 0:
        return t, t.begin(), 0
    t.nodes = _carry(src.nodes, kept_order(src.nodes, j, keep))
    t.leaf, t.kind = 0, TERMINAL if t.nodes[0].terminal else EVAL
    return t, t._emit(0, t.kind), len(t.nodes)


def ismcts_match(src, world, played, max_steps):
    """8.8: the source root's child for root action id `played`, -1 when the rule does not hold (the world's seat to move
    must be the child's and the source root's: one observer)"""
    if src is None or src.kind != FULL or src.max_steps != max_steps or not 0 <= played < N_ACTIONS:
        return -1
    code = src.root_code[played]
    if code == I.NONE_CODE or code not in src.nodes[0].children:
        return -1
    c = src.nodes[0].children[code]
    if over(world, max_steps) or src.nodes[c].seat != seat(world) or src.nodes[0].seat != seat(world):
        return -1
    return c


def ismcts_advance(src, world, played, max_nodes, keep, max_steps=400):
    """(new ISTreeModel, emitted leaf, kept) of sb_ismcts_advance on one tree: world is world 0 of the new root"""
    t = I.ISTreeModel(max_nodes, max_steps)
    leaf = t.begin(world)
    j = ismcts_match(src, np.asarray(world, dtype=np.uint8), int(played), max_steps)
    if j < 0:
        return t, leaf, 0
    t.nodes = _carry(src.nodes, kept_order(src.nodes, j, keep))
    t.nodes[0].code = I.NONE_CODE
    return t, leaf, len(t.nodes)

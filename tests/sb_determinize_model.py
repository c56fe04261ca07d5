"""TEST INFRASTRUCTURE -- plain-Python statement of sb_determinize (include/sb_b200.h) over the packed bytes, and of the
PIMC read-out of monsoon_b200.search.DeterminizedMCTS over the search model's trees.  The product package never imports it.
"""
import math

import numpy as np

import sb_search_model as SM
from ref_harness import philox4x32_10
from sb_layout import CF_OBJ, DECK_MAX, HAND_MAX, STATE_DTYPE

TAG = 0xDE7E
M32 = 0xFFFFFFFF
M64 = (1 << 64) - 1


def movable_slots(f, r):
    """[(in_deck, index)] of pl[r]'s movable card records: hand, then deck, without SB_CF_OBJ records"""
    p = f["pl"][r]
    out = [(0, h) for h in range(min(int(p["n_hand"]), HAND_MAX)) if not int(p["hand_flags"][h]) & CF_OBJ]
    return out + [(1, d) for d in range(min(int(p["n_deck"]), DECK_MAX)) if not int(p["deck_flags"][d]) & CF_OBJ]


def determinize(st, key, observer=None):
    """the record st (u8[512]) as sb_determinize rewrites it for observer (None = its local_order) and key (u64)"""
    out = np.array(st, dtype=np.uint8, copy=True)
    f = out.view(STATE_DTYPE)[0]
    o = int(f["local_order"] != 0) if observer is None else int(observer != 0)
    r = 1 - o
    key = int(key) & M64
    k_lo, k_hi = key & M32, key >> 32
    slots = movable_slots(f, r)
    p = f["pl"][r]
    names = (("hand_card", "hand_cost", "hand_flags"), ("deck_card", "deck_cost", "deck_flags"))
    trip = [tuple(int(p[nm][i]) for nm in names[d]) for d, i in slots]
    m = len(trip)
    for t, i in enumerate(range(m - 1, 0, -1)):
        w0 = philox4x32_10(t, 0, TAG, 0, k_lo, k_hi)[0]
        j = (w0 * (i + 1)) >> 32
        trip[i], trip[j] = trip[j], trip[i]
    for (d, i), tr in zip(slots, trip):
        for nm, v in zip(names[d], tr):
            p[nm][i] = v
    f["seed_lo"], f["seed_hi"] = k_lo, k_hi
    return out


def pimc_readout(trees, prior, value, n, k):
    """DeterminizedMCTS's read-out from n * k search-model trees (tree t = i * k + s) after their last evaluation:
    (visits i32[n,156] summed over s, q f64[n,156] visit-weighted mean of the per-tree q, NaN where the sum is 0,
    root_value f64[n] mean of the per-tree root values)"""
    ends = [t.end(prior[g], value[g]) for g, t in enumerate(trees)]
    vis = np.stack([e[0] for e in ends]).reshape(n, k, SM.N_ACTIONS)
    q = np.stack([e[1] for e in ends]).reshape(n, k, SM.N_ACTIONS)
    rv = np.array([e[2] for e in ends]).reshape(n, k)
    visits = vis.sum(1, dtype=np.int32)
    wsum = np.where(vis > 0, np.nan_to_num(q) * vis, 0.0).sum(1)
    with np.errstate(invalid="ignore", divide="ignore"):
        qq = np.where(visits > 0, wsum / visits, math.nan)
    return visits, qq, rv.mean(1)

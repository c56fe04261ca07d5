"""BatchedMCTS: n independent Monte-Carlo tree searches (PUCT) on the GPU with a caller-supplied evaluator.

The tree lives in a workspace on the device (sb_search_begin / sb_search_simulate / sb_search_end, include/sb_b200.h); one
simulation is one launch that backs up the last leaf, selects a new leaf, expands it with the engine's own step and emits
what the evaluator needs.  The evaluator stays in Python, usually a torch network:

    mcts = BatchedMCTS(env.n, num_simulations=64)
    visits, q, root_value = mcts.run(env.states, evaluate)   # evaluate(leaf, k) -> (prior f32[n,156], value f32[n])
    obs, masks, reward, done, info = env.step(select_actions(visits))

BatchedMCTS sees both hands and the future draws of the game's own random stream (the child of (s, a) is exactly the record
sb_step(s, a) gives), i.e. it is a perfect-information search, like the reference agent's forks.  DeterminizedMCTS is the fair
agent (Perfect-Information Monte Carlo): it searches K determinizations of each root (sb_determinize: the opponent's hand /
deck assignment and the random stream resampled, everything the player to move sees kept) and sums the root visits:

    mcts = DeterminizedMCTS(env.n, num_determinizations=8, num_simulations=8)
    visits, q, root_value = mcts.run(env.states, rollout_evaluator())

InformationSetMCTS is the information-set search (single-observer ISMCTS, sb_ismcts_*): one tree per root over what the
player to move sees, every simulation walking it through a fresh determinization, so the simulations are not split into K
separate trees that each believe their own world:

    mcts = InformationSetMCTS(env.n, num_simulations=64)
    visits, q, root_value = mcts.run(env.states, rollout_evaluator())

With reuse_nodes = R > 0, BatchedMCTS and InformationSetMCTS keep the subtree of the position reached between moves
(sb_search_advance / sb_ismcts_advance, DESIGN.md 8.10): a search of S simulations then starts from the visits the last
search already spent below the new root, up to R + 1 nodes of it:

    mcts = BatchedMCTS(env.n, num_simulations=64, reuse_nodes=64)
    for move in range(moves):
        visits, q, root_value = mcts.run(env.states, evaluate)   # mcts.kept: nodes carried over per tree
        obs, masks, reward, done, info = env.step(select_actions(visits))

GumbelMCTS and InformationSetGumbelMCTS run the same two trees with Gumbel MuZero's selection (sb_*_simulate_gumbel,
DESIGN.md 8.9): Gumbel-top-k with sequential halving at the root instead of exploration noise, and an improved policy
softmax(logits + sigma(completed q)) to train on, next to the action to play:

    mcts = GumbelMCTS(env.n, num_simulations=16)
    action, policy, visits, q, root_value = mcts.run(env.states, evaluate)
    obs, masks, reward, done, info = env.step(action)

With leaves_per_call = L > 1, BatchedMCTS selects L leaves per tree per call under virtual loss (sb_search_simulate_batch,
DESIGN.md 8.11), so the evaluator sees n * L rows per call and is called S / L times instead of S:

    mcts = BatchedMCTS(env.n, num_simulations=64, leaves_per_call=16)
    visits, q, root_value = mcts.run(env.states, evaluate)   # evaluate(leaf, k): n rows at k = 0, n * 16 rows at k = 1..4

InformationSetMCTS takes leaves_per_call too (sb_ismcts_simulate_batch, DESIGN.md 8.12): each of the L leaves of a tree is
walked through a world of its own, so the fair search gets the same larger evaluator batches:

    mcts = InformationSetMCTS(env.n, num_simulations=64, leaves_per_call=16)
    visits, q, root_value = mcts.run(env.states, rollout_evaluator())
"""
import math

import numpy as np
import torch

from .engine import N_ACTIONS, STATE_BYTES, get_engine
from .vec_env import next_seed, next_seed_array

_PLAYER_SIGN, _ERR = 16, 18     # byte offsets in SbState (include/sb_state.h)
_BASE_I16 = (16, 68)            # pl[0].base and pl[1].base as int16 indices (byte offsets 32 and 136)
LEAF_KEYS = ("states", "obs", "masks", "obs_err", "to_move", "kind")
_bits = {}


def legal_actions(masks):
    """bool[n,156] from legal masks i32[n,5] (u32 words, bit a of the mask = action id a)."""
    dev = masks.device
    if dev not in _bits:
        _bits[dev] = torch.arange(32, dtype=torch.int32, device=dev)
    return ((masks.unsqueeze(-1) >> _bits[dev]) & 1).reshape(masks.shape[0], -1)[:, :N_ACTIONS].bool()


def masked_softmax(logits, masks):
    """softmax of logits [n,156] over the legal set of masks i32[n,5]: f32, 0 at illegal action ids."""
    x = logits.float().masked_fill(~legal_actions(masks), float("-inf"))
    return torch.softmax(x, dim=-1).nan_to_num_(0.0)


def rollout_evaluator(engine=None, max_steps=400):
    """evaluate(leaf, k) with a uniform prior over the legal set (1/popcount in f32) and the value of one uniform-random
    rollout (sb_rollout_random, at most max_steps steps) run in place on leaf["states"]: +1 / -1 when the seat to move at the
    leaf wins / loses by the bases, 0 for a draw, an engine status or a rollout that hit max_steps."""
    engine = engine if engine is not None else get_engine()
    bufs = {}  # row count -> (prior, value): a batched search asks for n rows at k = 0 and n * L rows after

    def evaluate(leaf, k):
        states = leaf["states"]
        n = states.shape[0]
        if n not in bufs:
            bufs[n] = (torch.empty((n, N_ACTIONS), dtype=torch.float32, device=states.device),
                       torch.empty(n, dtype=torch.float32, device=states.device))
        prior, value = bufs[n]
        legal = legal_actions(leaf["masks"])
        inv = torch.reciprocal(legal.sum(1, keepdim=True, dtype=torch.int32).to(torch.float32))
        torch.where(legal, inv, torch.zeros((), dtype=torch.float32, device=states.device), out=prior)
        engine.rollout_random(states, max_steps)
        bases = states.view(torch.int16)[:, list(_BASE_I16)]
        lost = bases < 0
        first = (lost[:, 1] & ~lost[:, 0]).to(torch.float32) - (lost[:, 0] & ~lost[:, 1]).to(torch.float32)
        first.masked_fill_(states[:, _ERR] != 0, 0.0)
        torch.mul(first, 1.0 - 2.0 * leaf["to_move"].to(torch.float32), out=value)
        return prior, value

    return evaluate


def select_actions(visits, temperature=0.0, generator=None):
    """One action id per row of visits i32[n,156] (int64[n]): the arg-max (ties to the lowest id) at temperature 0, else a
    sample proportional to visits^(1/temperature).  A row without visits gives 255, which is never a legal action id.
    visits may come from BatchedMCTS (perfect information: the search saw the opponent's cards and future draws) or from
    DeterminizedMCTS / InformationSetMCTS (only what the player to move sees)."""
    has = visits.sum(1) > 0
    if temperature == 0:
        a = torch.argmax(visits, dim=1)
    else:
        v = visits.to(torch.float64)
        w = (v / v.amax(1, keepdim=True).clamp_min(1.0)) ** (1.0 / float(temperature))
        w = torch.where(has.unsqueeze(1), w, torch.ones_like(w))
        a = torch.multinomial(w, 1, generator=generator).squeeze(1)
    return torch.where(has, a, torch.full_like(a, 255))


class BatchedMCTS:
    """n trees of num_simulations + 1 nodes in one workspace, with every output buffer allocated once.

    run(roots, evaluate) -> (visits i32[n,156], q f64[n,156] NaN where unvisited, root_value f64[n]), q and root_value for
    the seat to move at the root.  evaluate(leaf, k) receives the leaf buffers (dict of states u8[n,512], obs i32[n,27,5,4],
    masks i32[n,5], obs_err u8[n], to_move u8[n], kind u8[n]: 0 evaluate, 1 terminal, 2 full) and the simulation index k
    (0 = the roots; add exploration noise to the prior there) and returns (prior f32[n,156], value f32[n]) on the device,
    the value from the point of view of to_move.  A run is exactly num_simulations + 2 library launches; with an evaluator
    that only uses torch it synchronises nothing with the host and can be captured in a torch.cuda.CUDAGraph.  The returned
    tensors are buffers of this object, overwritten by the next run.

    reuse_nodes = R > 0 keeps trees between runs: the trees have num_simulations + 1 + R nodes (so S simulations always
    fit), in two workspaces that take turns.  The first run, and the first after reset_tree(), begins fresh trees; every
    later run starts with sb_search_advance, which carries over the subtree of the lowest node whose record is the new root
    (the child of the action played, or an opponent position the search expanded), at most R + 1 nodes of it.  Still
    num_simulations + 2 launches.  self.kept i32[n] holds the nodes each tree carried over in the last run (0: a fresh root).
    Root noise added at k = 0 applies to a carried-over root too: the prior of k = 0 replaces its stored one.  A captured
    advancing run reads the trees the run before it finished, and an advance consumes the trees it reads (their node
    counts become 0): replaying one captured run a second time starts every tree fresh (self.kept all 0).  To replay a
    reusing loop, capture two consecutive runs in one graph, so that the workspaces take turns as they do eagerly.

    leaves_per_call = L > 1 selects L leaves per tree per call under virtual loss (sb_search_simulate_batch, DESIGN.md
    8.11): each selection counts the earlier paths of the same call as extra visits, each carrying virtual_loss, so the
    leaves spread out, and all n * L are expanded in parallel and evaluated as one batch.  num_simulations = S must be a
    multiple of L.  A run is the begin (or advance), C = S / L batch calls and the batch end: 2C + 2 library launches.
    evaluate(leaf, k) gets the n roots at k = 0 and n * L rows at k = 1..C, tree-major (row g * L + l is leaf l of tree g),
    with kind 3 for a collision (the walk reached a leaf another selection of the same call had just taken; the root is
    emitted and its evaluation is not used).  The read-out is the same triple; a root's child visits then add up to its
    slots that were neither a collision nor full, so they can sum to less than S.  L = 1 is the plain search exactly.
    """

    def __init__(self, n, num_simulations, c_puct=1.25, fpu=0.0, max_steps=400, engine=None, device=None, reuse_nodes=0,
                 leaves_per_call=1, virtual_loss=1.0):
        if int(num_simulations) < 0:
            raise ValueError("num_simulations must be >= 0")
        if not (math.isfinite(c_puct) and c_puct >= 0) or not math.isfinite(fpu):
            raise ValueError("c_puct must be finite and >= 0, fpu finite")
        if int(reuse_nodes) < 0:
            raise ValueError("reuse_nodes must be >= 0")
        if not 1 <= int(leaves_per_call) <= 256 or int(num_simulations) % int(leaves_per_call):
            raise ValueError("leaves_per_call must be 1..256 and divide num_simulations")
        if not (math.isfinite(virtual_loss) and virtual_loss >= 0):
            raise ValueError("virtual_loss must be finite and >= 0")
        self.engine = e = engine if engine is not None else get_engine(device)
        self.n, self.num_simulations, self.reuse_nodes = int(n), int(num_simulations), int(reuse_nodes)
        self.c_puct, self.fpu, self.max_steps = float(c_puct), float(fpu), int(max_steps)
        self.leaves, self.virtual_loss = int(leaves_per_call), float(virtual_loss)
        self.max_nodes = self.num_simulations + 1 + self.reuse_nodes
        L = self.leaves
        nb = e.search_workspace_bytes(self.n, self.max_nodes) if L == 1 else e.search_batch_workspace_bytes(self.n, self.max_nodes, L)
        self.ws = torch.empty(nb, dtype=torch.uint8, device=e.device)
        self.ws_next = torch.empty(nb, dtype=torch.uint8, device=e.device) if self.reuse_nodes else None
        self.kept = torch.zeros(self.n, dtype=torch.int32, device=e.device)
        self.fresh = True
        self.leaf = e._search_outputs(self.n, None, LEAF_KEYS)
        self.out = e._search_outputs(self.n, None, ("visits", "q", "root_value"))
        if L > 1:
            self.batch_leaf = e._search_outputs(self.n * L, None, LEAF_KEYS)
            self.batch_prior = torch.empty((self.n * L, N_ACTIONS), dtype=torch.float32, device=e.device)
            self.batch_value = torch.empty(self.n * L, dtype=torch.float32, device=e.device)

    def reset_tree(self):
        """the next run begins fresh trees (kept 0), e.g. after new episodes were dealt"""
        self.fresh = True

    def run(self, roots, evaluate):
        e, n, m = self.engine, self.n, self.max_nodes
        assert roots.shape[0] == n, "roots are u8[n, 512] with n = %d" % n
        if self.reuse_nodes and not self.fresh:
            e.search_advance(self.ws, self.ws_next, roots, m, self.reuse_nodes + 1, self.max_steps, out=dict(self.leaf, kept=self.kept))
            self.ws, self.ws_next = self.ws_next, self.ws
        else:
            e.search_begin(self.ws, roots, m, self.max_steps, out=self.leaf)
            if self.reuse_nodes:
                self.kept.zero_()
        self.fresh = False
        prior, value = evaluate(self.leaf, 0)
        L = self.leaves
        if L == 1:
            for k in range(1, self.num_simulations + 1):
                e.search_simulate(self.ws, n, m, prior, value, self.c_puct, self.fpu, out=self.leaf)
                prior, value = evaluate(self.leaf, k)
            e.search_end(self.ws, n, m, prior, value, out=self.out)
            return self.out["visits"], self.out["q"], self.out["root_value"]
        # the first batch call backs up the roots from slot 0 of each tree's rows; the other slots are not read
        self.batch_prior.view(n, L, N_ACTIONS)[:, 0].copy_(prior)
        self.batch_value.view(n, L)[:, 0].copy_(value)
        prior, value = self.batch_prior, self.batch_value
        for k in range(1, self.num_simulations // L + 1):
            e.search_simulate_batch(self.ws, n, m, L, prior, value, self.c_puct, self.fpu, self.virtual_loss, out=self.batch_leaf)
            prior, value = evaluate(self.batch_leaf, k)
        e.search_end_batch(self.ws, n, m, L, prior, value, out=self.out)
        return self.out["visits"], self.out["q"], self.out["root_value"]


class DeterminizedMCTS:
    """Perfect-Information Monte Carlo over BatchedMCTS: n roots, K determinizations each, num_simulations per tree.

    Tree t = i * K + k searches root i under determinization k: the roots are repeated into a preallocated u8[n*K,512]
    buffer and determinized in place for each root's own local_order (the seat to move, whose hand sb_observe shows), so
    every tree sees the root player's cards as they are and a resampled assignment of the opponent's cards to hand and
    deck slots, with a resampled random stream.  One inner BatchedMCTS(n*K, num_simulations) runs over them and
    evaluate(leaf, k) sees n*K leaves in that layout (rollout_evaluator works unchanged).

    run(roots, evaluate, keys=None) -> (visits i32[n,156] summed over the K trees, q f64[n,156] the visit-weighted mean of
    the trees' q, NaN where the summed visits are 0, root_value f64[n] the mean of the trees' root values), for the seat to
    move at the root.  The root player is the observer, so the root's legal set is the same in all K trees.
    keys: device i64[n*K], the Philox keys of the determinizations.  When None they come from `seed` and a per-object
    call counter on the host (next_seed mix) and are copied to the device: that run is reproducible but not capture-safe.
    With caller keys (and a capture-safe evaluator) a run synchronises nothing with the host and can be captured in a
    torch.cuda.CUDAGraph.  A run is exactly num_simulations + 3 library launches.  The returned tensors are buffers of this
    object, overwritten by the next run.
    """

    def __init__(self, n, num_determinizations, num_simulations, c_puct=1.25, fpu=0.0, max_steps=400, seed=0, engine=None,
                 device=None):
        if int(num_determinizations) < 1:
            raise ValueError("num_determinizations must be >= 1")
        self.n, self.k = int(n), int(num_determinizations)
        self.inner = BatchedMCTS(self.n * self.k, num_simulations, c_puct, fpu, max_steps, engine, device)
        self.engine = e = self.inner.engine
        self.seed, self.calls = int(seed), 0
        self.states = torch.empty((self.n * self.k, STATE_BYTES), dtype=torch.uint8, device=e.device)
        self.out = e._search_outputs(self.n, None, ("visits", "q", "root_value"))

    def default_keys(self):
        """the keys of the next run without caller keys: next_seed(base + t) for tree t, base = next_seed(next_seed(seed) +
        call index)"""
        base = next_seed(next_seed(self.seed) + self.calls)
        self.calls += 1
        return next_seed_array(np.arange(self.n * self.k, dtype=np.uint64) + np.uint64(base))

    def run(self, roots, evaluate, keys=None):
        e, n, k = self.engine, self.n, self.k
        assert roots.shape == (n, STATE_BYTES), "roots are u8[n, 512] with n = %d" % n
        if keys is None:
            keys = torch.from_numpy(self.default_keys()).to(e.device)
        assert keys.shape == (n * k,), "keys are i64[n * K] with n * K = %d" % (n * k)
        self.states.view(n, k, STATE_BYTES).copy_(roots.unsqueeze(1).expand(n, k, STATE_BYTES))
        e.determinize(self.states, keys, out=self.states)
        visits, q, root_value = self.inner.run(self.states, evaluate)
        vis = visits.view(n, k, N_ACTIONS)
        total = vis.sum(1)
        wsum = (torch.nan_to_num(q.view(n, k, N_ACTIONS), nan=0.0) * vis).sum(1)
        self.out["visits"].copy_(total)
        torch.div(wsum, total, out=self.out["q"])
        self.out["q"].masked_fill_(total == 0, float("nan"))
        torch.mean(root_value.view(n, k), 1, out=self.out["root_value"])
        return self.out["visits"], self.out["q"], self.out["root_value"]


class InformationSetMCTS:
    """Information-set MCTS: n roots, one tree each over the root player's information set, num_simulations per tree.

    Every call of the search gets a fresh world per root: sb_determinize(roots, keys_k) for the root's own local_order (the
    seat to move) into one preallocated u8[n,512] buffer, then sb_ismcts_begin (k = 0) or sb_ismcts_simulate (k = 1..S)
    walks the tree through it.  Edges are keyed by move codes (card and target, not hand slot), so the tree is shared by
    every world.  evaluate(leaf, k) receives the leaf buffers as in BatchedMCTS; leaf["states"] holds the world's record at
    the leaf, never the root's hidden cards or key, so rollout_evaluator works unchanged.

    run(roots, evaluate, keys=None) -> (visits i32[n,156], q f64[n,156] NaN where unvisited, root_value f64[n]), for the seat
    to move at the root, by the root's action ids (an id that plays the same card as a lower legal id reads 0 / NaN).
    keys: device i64[(S+1)*n], simulation-major (keys[k*n:(k+1)*n] are the worlds of call k).  When None they come from
    `seed` and a per-object call counter on the host (next_seed mix) and are copied to the device: reproducible but not
    capture-safe.  With caller keys (and a capture-safe evaluator) a run synchronises nothing with the host and can be
    captured in a torch.cuda.CUDAGraph.  A run is exactly 2 * num_simulations + 3 library launches (S + 1 sb_determinize,
    begin, S simulate, end).  The returned tensors are buffers of this object, overwritten by the next run.

    reuse_nodes = R > 0 keeps trees between runs, as BatchedMCTS's (num_simulations + 1 + R nodes, two workspaces,
    reset_tree(), self.kept): a later run passes played, the id played at the previous run's roots (e.g.
    select_actions(visits)), and starts with sb_ismcts_advance, which carries over the subtree of that root action's child
    (at most R + 1 nodes) where the new root is exactly the record sb_step(previous root, played) gives.  The run checks
    that on the device: it keeps a copy of the previous roots, steps it with played (one sb_step) and compares it byte for
    byte with the new roots; where they differ (an episode that ended and was redealt, a rejected action, an opponent turn
    in between) the tree starts fresh.  Such a run is 2 * num_simulations + 4 library launches (2S + 3 with played None,
    which starts every tree fresh), and with caller keys still capturable, with BatchedMCTS's caveat on replaying one
    captured advancing run.  With R = 0, played is ignored.

    leaves_per_call = L > 1 selects L leaves per tree per call under virtual loss (sb_ismcts_simulate_batch, DESIGN.md
    8.12), each walked through a world of its own: the roots are repeated once per run into a u8[n*L,512] buffer, which each
    call determinizes with its n * L keys into a preallocated world buffer.  num_simulations = S must be a multiple of L.
    The keys keep their shape, i64[(S+1)*n]: the first n are world 0, and call c = 1..S/L uses the n * L keys after the
    first n + (c-1) * n * L, tree-major (key n + (c-1) * n * L + g * L + l is the world of leaf l of tree g), so
    default_keys is unchanged.  A run is the world-0 determinization and begin (or advance), C = S / L determinizations and
    batch calls and the batch end: 2C + 3 library launches (one more with an advance's played check).  evaluate(leaf, k) gets
    the n roots at k = 0 and n * L rows at k = 1..C, tree-major, with kind 3 for a collision (the world's root is emitted and
    its evaluation is not used); a root's child visits then add up to its slots that were neither a collision nor full.
    L = 1 is the plain search exactly.  It combines with reuse_nodes (two batch-sized workspaces).
    """

    def __init__(self, n, num_simulations, c_puct=1.25, fpu=0.0, max_steps=400, seed=0, engine=None, device=None, reuse_nodes=0,
                 leaves_per_call=1, virtual_loss=1.0):
        if int(num_simulations) < 0:
            raise ValueError("num_simulations must be >= 0")
        if not (math.isfinite(c_puct) and c_puct >= 0) or not math.isfinite(fpu):
            raise ValueError("c_puct must be finite and >= 0, fpu finite")
        if int(reuse_nodes) < 0:
            raise ValueError("reuse_nodes must be >= 0")
        if not 1 <= int(leaves_per_call) <= 256 or int(num_simulations) % int(leaves_per_call):
            raise ValueError("leaves_per_call must be 1..256 and divide num_simulations")
        if not (math.isfinite(virtual_loss) and virtual_loss >= 0):
            raise ValueError("virtual_loss must be finite and >= 0")
        self.engine = e = engine if engine is not None else get_engine(device)
        self.n, self.num_simulations, self.reuse_nodes = int(n), int(num_simulations), int(reuse_nodes)
        self.c_puct, self.fpu, self.max_steps = float(c_puct), float(fpu), int(max_steps)
        self.leaves, self.virtual_loss = int(leaves_per_call), float(virtual_loss)
        self.max_nodes = self.num_simulations + 1 + self.reuse_nodes
        self.seed, self.calls = int(seed), 0
        L = self.leaves
        nb = e.ismcts_workspace_bytes(self.n, self.max_nodes) if L == 1 else e.ismcts_batch_workspace_bytes(self.n, self.max_nodes, L)
        self.ws = torch.empty(nb, dtype=torch.uint8, device=e.device)
        self.world = torch.empty((self.n, STATE_BYTES), dtype=torch.uint8, device=e.device)
        self.kept = torch.zeros(self.n, dtype=torch.int32, device=e.device)
        self.fresh = True
        if self.reuse_nodes:
            self.ws_next = torch.empty(nb, dtype=torch.uint8, device=e.device)
            self.prev = torch.empty((self.n, STATE_BYTES), dtype=torch.uint8, device=e.device)
            self.stepped = torch.empty((self.n, STATE_BYTES), dtype=torch.uint8, device=e.device)
            self.played = torch.empty(self.n, dtype=torch.int32, device=e.device)
            self.step_out = [torch.empty(self.n, dtype=d, device=e.device) for d in (torch.uint8, torch.int8, torch.uint8, torch.uint8)]
        self.leaf = e._search_outputs(self.n, None, LEAF_KEYS)
        self.out = e._search_outputs(self.n, None, ("visits", "q", "root_value"))
        if L > 1:
            self.repeated = torch.empty((self.n * L, STATE_BYTES), dtype=torch.uint8, device=e.device)
            self.worlds = torch.empty((self.n * L, STATE_BYTES), dtype=torch.uint8, device=e.device)
            self.batch_leaf = e._search_outputs(self.n * L, None, LEAF_KEYS)
            self.batch_prior = torch.empty((self.n * L, N_ACTIONS), dtype=torch.float32, device=e.device)
            self.batch_value = torch.empty(self.n * L, dtype=torch.float32, device=e.device)

    def default_keys(self):
        """the keys of the next run without caller keys: next_seed(base + t) for t < (S+1)*n, base = next_seed(next_seed(seed)
        + call index).  The count is (num_simulations + 1) * n whatever reuse_nodes is."""
        base = next_seed(next_seed(self.seed) + self.calls)
        self.calls += 1
        return next_seed_array(np.arange((self.num_simulations + 1) * self.n, dtype=np.uint64) + np.uint64(base))

    def reset_tree(self):
        """the next run begins fresh trees (kept 0), e.g. after new episodes were dealt"""
        self.fresh = True

    def _played(self, roots, played):
        """played i32[n] where sb_step(previous root, played) is the new root byte for byte, else -1"""
        if played is None:
            return self.played.fill_(-1)
        played = torch.as_tensor(played).to(self.engine.device, torch.int64)
        assert tuple(played.shape) == (self.n,), "played is one action id per root, [n]"
        act, reward, done, err = self.step_out
        ok = (played >= 0) & (played < N_ACTIONS)
        act.copy_(torch.where(ok, played, N_ACTIONS - 1))
        self.stepped.copy_(self.prev)
        self.engine.step(self.stepped, act, reward=reward, done=done, err=err)
        ok &= (self.stepped == roots).all(1)
        return self.played.copy_(torch.where(ok, played, -1))

    def run(self, roots, evaluate, keys=None, played=None):
        e, n, m, S = self.engine, self.n, self.max_nodes, self.num_simulations
        assert roots.shape == (n, STATE_BYTES), "roots are u8[n, 512] with n = %d" % n
        if keys is None:
            keys = torch.from_numpy(self.default_keys()).to(e.device)
        assert keys.shape == ((S + 1) * n,), "keys are i64[(S + 1) * n] with (S + 1) * n = %d" % ((S + 1) * n)
        e.determinize(roots, keys[:n], out=self.world)
        if self.reuse_nodes and not self.fresh:
            e.ismcts_advance(self.ws, self.ws_next, self.world, self._played(roots, played), m, self.reuse_nodes + 1, self.max_steps,
                             out=dict(self.leaf, kept=self.kept))
            self.ws, self.ws_next = self.ws_next, self.ws
        else:
            e.ismcts_begin(self.ws, self.world, m, self.max_steps, out=self.leaf)
            if self.reuse_nodes:
                self.kept.zero_()
        if self.reuse_nodes:
            self.prev.copy_(roots)
        self.fresh = False
        prior, value = evaluate(self.leaf, 0)
        L = self.leaves
        if L == 1:
            for k in range(1, self.num_simulations + 1):
                e.determinize(roots, keys[k * n:(k + 1) * n], out=self.world)
                e.ismcts_simulate(self.ws, self.world, m, prior, value, self.c_puct, self.fpu, out=self.leaf)
                prior, value = evaluate(self.leaf, k)
            e.ismcts_end(self.ws, n, m, prior, value, out=self.out)
            return self.out["visits"], self.out["q"], self.out["root_value"]
        # the first batch call backs up the roots from slot 0 of each tree's rows; the other slots are not read
        self.repeated.view(n, L, STATE_BYTES).copy_(roots.unsqueeze(1).expand(n, L, STATE_BYTES))
        self.batch_prior.view(n, L, N_ACTIONS)[:, 0].copy_(prior)
        self.batch_value.view(n, L)[:, 0].copy_(value)
        prior, value = self.batch_prior, self.batch_value
        for k in range(1, S // L + 1):
            lo = n + (k - 1) * n * L
            e.determinize(self.repeated, keys[lo:lo + n * L], out=self.worlds)
            e.ismcts_simulate_batch(self.ws, self.worlds, m, L, prior, value, self.c_puct, self.fpu, self.virtual_loss, out=self.batch_leaf)
            prior, value = evaluate(self.batch_leaf, k)
        e.ismcts_end_batch(self.ws, n, m, L, prior, value, out=self.out)
        return self.out["visits"], self.out["q"], self.out["root_value"]


def gumbel_noise(n, seed):
    """f32[n,156] of -log(-log u), u uniform on (0, 1) in steps of 2^-53, from numpy's default_rng(seed) (host)"""
    u = np.random.default_rng(seed).integers(1, 1 << 53, size=(n, N_ACTIONS), dtype=np.int64).astype(np.float64) / float(1 << 53)
    return (-np.log(-np.log(u))).astype(np.float32)


def _gumbel_args(num_simulations, max_considered, c_visit, c_scale):
    if not 1 <= int(num_simulations) <= 1 << 24:
        raise ValueError("num_simulations must be 1..2^24")
    if not 1 <= int(max_considered) <= N_ACTIONS:
        raise ValueError("max_considered must be 1..156")
    if not (math.isfinite(c_visit) and c_visit >= 0 and math.isfinite(c_scale) and c_scale >= 0):
        raise ValueError("c_visit and c_scale must be finite and >= 0")


class GumbelMCTS:
    """Gumbel MuZero search over BatchedMCTS's perfect-information trees: n trees of num_simulations + 1 nodes.

    run(roots, evaluate, gumbel=None) -> (action i32[n], policy f32[n,156], visits i32[n,156], q f64[n,156], root_value
    f64[n]).  action is the id to play (the root id with the most visits and the best g + logit + sigma among those; 255
    when the root has no visit, e.g. a finished game) and feeds StormboundVecEnv.step directly; policy is the improved
    policy softmax(logit + sigma(completed q)) over the legal set, the training target; visits, q and root_value are
    BatchedMCTS's.  evaluate(leaf, k) is BatchedMCTS's contract (rollout_evaluator works unchanged); the root needs no noise.
    gumbel: device f32[n,156], the Gumbel noise of the search.  When None it is -log(-log u) drawn on the host from `seed`
    and a per-object call counter (next_seed mix) and copied to the device: reproducible but not capture-safe.  With caller
    noise (and a capture-safe evaluator) a run synchronises nothing with the host and can be captured in a
    torch.cuda.CUDAGraph.  A run is exactly num_simulations + 2 library launches.  The returned tensors are buffers of this
    object, overwritten by the next run.
    """

    def __init__(self, n, num_simulations, max_considered=16, c_visit=50.0, c_scale=0.1, max_steps=400, seed=0, engine=None,
                 device=None):
        _gumbel_args(num_simulations, max_considered, c_visit, c_scale)
        self.engine = e = engine if engine is not None else get_engine(device)
        self.n, self.num_simulations, self.max_considered = int(n), int(num_simulations), int(max_considered)
        self.c_visit, self.c_scale, self.max_steps = float(c_visit), float(c_scale), int(max_steps)
        self.max_nodes = self.num_simulations + 1
        self.seed, self.calls = int(seed), 0
        self.ws = torch.empty(e.search_workspace_bytes(self.n, self.max_nodes), dtype=torch.uint8, device=e.device)
        self.gumbel = torch.empty((self.n, N_ACTIONS), dtype=torch.float32, device=e.device)
        self.leaf = e._search_outputs(self.n, None, LEAF_KEYS)
        self.out = e._search_outputs(self.n, None, ("action", "policy", "visits", "q", "root_value"))

    def default_gumbel(self):
        """the noise of the next run without caller noise: gumbel_noise(n, next_seed(next_seed(seed) + call index))"""
        base = next_seed(next_seed(self.seed) + self.calls)
        self.calls += 1
        return gumbel_noise(self.n, base)

    def _noise(self, gumbel):
        if gumbel is None:
            self.gumbel.copy_(torch.from_numpy(self.default_gumbel()))
            return self.gumbel
        assert tuple(gumbel.shape) == (self.n, N_ACTIONS), "gumbel is f32[n, 156] with n = %d" % self.n
        return gumbel

    def _result(self):
        o = self.out
        return o["action"], o["policy"], o["visits"], o["q"], o["root_value"]

    def run(self, roots, evaluate, gumbel=None):
        e, n, m, S = self.engine, self.n, self.max_nodes, self.num_simulations
        assert roots.shape[0] == n, "roots are u8[n, 512] with n = %d" % n
        g = self._noise(gumbel)
        e.search_begin(self.ws, roots, m, self.max_steps, out=self.leaf)
        prior, value = evaluate(self.leaf, 0)
        for k in range(1, S + 1):
            e.search_simulate_gumbel(self.ws, n, m, prior, value, g, k, S, self.max_considered, self.c_visit, self.c_scale, out=self.leaf)
            prior, value = evaluate(self.leaf, k)
        e.search_end_gumbel(self.ws, n, m, prior, value, g, self.c_visit, self.c_scale, out=self.out)
        return self._result()


class InformationSetGumbelMCTS(GumbelMCTS):
    """Gumbel MuZero search over InformationSetMCTS's information-set trees: one tree per root over what the player to move
    sees, every call walking it through a fresh determinization.

    run(roots, evaluate, keys=None, gumbel=None) -> (action, policy, visits, q, root_value) as GumbelMCTS, by the root's
    action ids (an id that plays the same card as a lower legal id reads 0 visits, NaN q and 0 policy).  keys are
    InformationSetMCTS's (device i64[(S+1)*n], simulation-major; None: from `seed` and a call counter on the host), gumbel
    GumbelMCTS's.  With caller keys and noise (and a capture-safe evaluator) a run can be captured in a torch.cuda.CUDAGraph.
    A run is exactly 2 * num_simulations + 3 library launches (S + 1 sb_determinize, begin, S simulate, end).
    """

    def __init__(self, n, num_simulations, max_considered=16, c_visit=50.0, c_scale=0.1, max_steps=400, seed=0, engine=None,
                 device=None):
        _gumbel_args(num_simulations, max_considered, c_visit, c_scale)
        self.engine = e = engine if engine is not None else get_engine(device)
        self.n, self.num_simulations, self.max_considered = int(n), int(num_simulations), int(max_considered)
        self.c_visit, self.c_scale, self.max_steps = float(c_visit), float(c_scale), int(max_steps)
        self.max_nodes = self.num_simulations + 1
        self.seed, self.calls, self.key_calls = int(seed), 0, 0
        self.ws = torch.empty(e.ismcts_workspace_bytes(self.n, self.max_nodes), dtype=torch.uint8, device=e.device)
        self.world = torch.empty((self.n, STATE_BYTES), dtype=torch.uint8, device=e.device)
        self.gumbel = torch.empty((self.n, N_ACTIONS), dtype=torch.float32, device=e.device)
        self.leaf = e._search_outputs(self.n, None, LEAF_KEYS)
        self.out = e._search_outputs(self.n, None, ("action", "policy", "visits", "q", "root_value"))

    def default_keys(self):
        """InformationSetMCTS.default_keys, with a call counter of its own"""
        base = next_seed(next_seed(self.seed) + self.key_calls)
        self.key_calls += 1
        return next_seed_array(np.arange(self.max_nodes * self.n, dtype=np.uint64) + np.uint64(base))

    def run(self, roots, evaluate, keys=None, gumbel=None):
        e, n, m, S = self.engine, self.n, self.max_nodes, self.num_simulations
        assert roots.shape == (n, STATE_BYTES), "roots are u8[n, 512] with n = %d" % n
        if keys is None:
            keys = torch.from_numpy(self.default_keys()).to(e.device)
        assert keys.shape == (m * n,), "keys are i64[(S + 1) * n] with (S + 1) * n = %d" % (m * n)
        g = self._noise(gumbel)
        e.determinize(roots, keys[:n], out=self.world)
        e.ismcts_begin(self.ws, self.world, m, self.max_steps, out=self.leaf)
        prior, value = evaluate(self.leaf, 0)
        for k in range(1, S + 1):
            e.determinize(roots, keys[k * n:(k + 1) * n], out=self.world)
            e.ismcts_simulate_gumbel(self.ws, self.world, m, prior, value, g, k, S, self.max_considered, self.c_visit, self.c_scale,
                                     out=self.leaf)
            prior, value = evaluate(self.leaf, k)
        e.ismcts_end_gumbel(self.ws, n, m, prior, value, g, self.c_visit, self.c_scale, out=self.out)
        return self._result()

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

GumbelMCTS and InformationSetGumbelMCTS run the same two trees with Gumbel MuZero's selection (sb_*_simulate_gumbel,
DESIGN.md 8.9): Gumbel-top-k with sequential halving at the root instead of exploration noise, and an improved policy
softmax(logits + sigma(completed q)) to train on, next to the action to play:

    mcts = GumbelMCTS(env.n, num_simulations=16)
    action, policy, visits, q, root_value = mcts.run(env.states, evaluate)
    obs, masks, reward, done, info = env.step(action)
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
    bufs = {}

    def evaluate(leaf, k):
        states = leaf["states"]
        n = states.shape[0]
        if bufs.get("n") != n:
            bufs.update(n=n, prior=torch.empty((n, N_ACTIONS), dtype=torch.float32, device=states.device),
                        value=torch.empty(n, dtype=torch.float32, device=states.device))
        prior, value = bufs["prior"], bufs["value"]
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
    """

    def __init__(self, n, num_simulations, c_puct=1.25, fpu=0.0, max_steps=400, engine=None, device=None):
        if int(num_simulations) < 0:
            raise ValueError("num_simulations must be >= 0")
        if not (math.isfinite(c_puct) and c_puct >= 0) or not math.isfinite(fpu):
            raise ValueError("c_puct must be finite and >= 0, fpu finite")
        self.engine = engine if engine is not None else get_engine(device)
        self.n, self.num_simulations = int(n), int(num_simulations)
        self.c_puct, self.fpu, self.max_steps = float(c_puct), float(fpu), int(max_steps)
        self.max_nodes = self.num_simulations + 1
        self.ws = torch.empty(self.engine.search_workspace_bytes(self.n, self.max_nodes), dtype=torch.uint8, device=self.engine.device)
        self.leaf = self.engine._search_outputs(self.n, None, LEAF_KEYS)
        self.out = self.engine._search_outputs(self.n, None, ("visits", "q", "root_value"))

    def run(self, roots, evaluate):
        e, n, m = self.engine, self.n, self.max_nodes
        assert roots.shape[0] == n, "roots are u8[n, 512] with n = %d" % n
        e.search_begin(self.ws, roots, m, self.max_steps, out=self.leaf)
        prior, value = evaluate(self.leaf, 0)
        for k in range(1, self.num_simulations + 1):
            e.search_simulate(self.ws, n, m, prior, value, self.c_puct, self.fpu, out=self.leaf)
            prior, value = evaluate(self.leaf, k)
        e.search_end(self.ws, n, m, prior, value, out=self.out)
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
    """

    def __init__(self, n, num_simulations, c_puct=1.25, fpu=0.0, max_steps=400, seed=0, engine=None, device=None):
        if int(num_simulations) < 0:
            raise ValueError("num_simulations must be >= 0")
        if not (math.isfinite(c_puct) and c_puct >= 0) or not math.isfinite(fpu):
            raise ValueError("c_puct must be finite and >= 0, fpu finite")
        self.engine = e = engine if engine is not None else get_engine(device)
        self.n, self.num_simulations = int(n), int(num_simulations)
        self.c_puct, self.fpu, self.max_steps = float(c_puct), float(fpu), int(max_steps)
        self.max_nodes = self.num_simulations + 1
        self.seed, self.calls = int(seed), 0
        self.ws = torch.empty(e.ismcts_workspace_bytes(self.n, self.max_nodes), dtype=torch.uint8, device=e.device)
        self.world = torch.empty((self.n, STATE_BYTES), dtype=torch.uint8, device=e.device)
        self.leaf = e._search_outputs(self.n, None, LEAF_KEYS)
        self.out = e._search_outputs(self.n, None, ("visits", "q", "root_value"))

    def default_keys(self):
        """the keys of the next run without caller keys: next_seed(base + t) for t < (S+1)*n, base = next_seed(next_seed(seed)
        + call index)"""
        base = next_seed(next_seed(self.seed) + self.calls)
        self.calls += 1
        return next_seed_array(np.arange(self.max_nodes * self.n, dtype=np.uint64) + np.uint64(base))

    def run(self, roots, evaluate, keys=None):
        e, n, m = self.engine, self.n, self.max_nodes
        assert roots.shape == (n, STATE_BYTES), "roots are u8[n, 512] with n = %d" % n
        if keys is None:
            keys = torch.from_numpy(self.default_keys()).to(e.device)
        assert keys.shape == (m * n,), "keys are i64[(S + 1) * n] with (S + 1) * n = %d" % (m * n)
        e.determinize(roots, keys[:n], out=self.world)
        e.ismcts_begin(self.ws, self.world, m, self.max_steps, out=self.leaf)
        prior, value = evaluate(self.leaf, 0)
        for k in range(1, self.num_simulations + 1):
            e.determinize(roots, keys[k * n:(k + 1) * n], out=self.world)
            e.ismcts_simulate(self.ws, self.world, m, prior, value, self.c_puct, self.fpu, out=self.leaf)
            prior, value = evaluate(self.leaf, k)
        e.ismcts_end(self.ws, n, m, prior, value, out=self.out)
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

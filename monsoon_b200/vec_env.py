"""StormboundVecEnv: n Stormbound games as one batched, auto-resetting environment on the GPU.

Each step is one launch of sb_env_step (include/sb_b200.h): check and apply the learner's actions, let the opponent play until
the learner is to move again, deal the next game of every env whose episode ended, and emit observations and legal masks.
Nothing is synchronised with the host and every output is preallocated, so `step` can be captured in a torch.cuda.CUDAGraph.
"""
import numpy as np
import torch

from .engine import N_ACTIONS, get_engine
from .evo import FitnessEvaluator

OPPONENTS = {None: 0, "none": 0, "random": 1, "expert": 2, "heuristic": 3}
_M64 = (1 << 64) - 1
_PLAYER_SIGN = 16  # byte offset of SbState.player_sign (include/sb_state.h): 1 = FIRST to move


def next_seed(s):
    """Seed of an env's next episode from the Philox key `s` of the finished one (splitmix64 finaliser, 63 bits)."""
    z = (int(s) + 0x9E3779B97F4A7C15) & _M64
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & _M64
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & _M64
    z ^= z >> 31
    return z & 0x7FFFFFFFFFFFFFFF


def next_seed_array(s):
    """Vectorised next_seed: uint64 wrap-around arithmetic on an integer array; returns int64."""
    z = np.asarray(s).astype(np.uint64)
    with np.errstate(over="ignore"):
        z = z + np.uint64(0x9E3779B97F4A7C15)
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    z ^= z >> np.uint64(31)
    return (z & np.uint64(0x7FFFFFFFFFFFFFFF)).astype(np.int64)


class StormboundVecEnv:
    """n envs, one packed 512-byte record each (`states`).

    opponent: None (self-play: the caller acts for both seats), "random" (uniform legal agent), "expert"
    (Stormbound.expert_action) or "heuristic" (HeuristicAgent with rows of `opponent_weights`, a f64[P,10] tensor or a list
    of WeightVectors, chosen per env by `opponent_index` i32[n], default row g).  seats: the learner's seat per env, an int or
    a sequence of 0 (FIRST) / 1 (SECOND); default FIRST.  decks / factions: u8[2,k] + u8[2] shared by all envs, or
    u8[n,2,k] + u8[n,2] per env, kept by the env across its episodes; default the reference's two decks.  The first seeds are
    next_seed(seed + g), or `seeds` i64[n]; episode e + 1 of an env is dealt from next_seed of episode e's key.

    reset() -> (obs i32[n,27,5,4], masks i32[n,5]); step(actions) -> (obs, masks, reward f32[n], done bool[n], info) with
    reward +1 / -1 when an episode ended in this call with the learner (in self-play: the seat that acted) winning / losing,
    else 0, and info = {result, length, final_states (valid where done), obs_err} as device tensors.  Every returned tensor
    is a buffer of the env, overwritten by the next call.
    """

    def __init__(self, n, seed=0, opponent=None, seats=None, opponent_weights=None, opponent_index=None, decks=None, factions=None,
                 max_steps=400, device=None, engine=None, seeds=None):
        if opponent not in OPPONENTS:
            raise ValueError("opponent must be one of %s" % sorted(k for k in OPPONENTS if k))
        self.engine = engine if engine is not None else get_engine(device)
        dev = self.engine.device
        self.n = n
        self.opponent = OPPONENTS[opponent]
        self.max_steps = int(max_steps)
        if seeds is None:
            seeds = next_seed_array(np.arange(n, dtype=np.uint64) + np.uint64(int(seed) & _M64))
        self.seeds = torch.as_tensor(np.asarray(seeds, dtype=np.int64) if not torch.is_tensor(seeds) else seeds).to(dev, torch.int64).contiguous()
        assert self.seeds.numel() == n
        if seats is None or isinstance(seats, int):
            seat = torch.full((n,), int(seats or 0), dtype=torch.uint8, device=dev)
        else:
            seat = torch.as_tensor(np.asarray(seats) if not torch.is_tensor(seats) else seats).to(dev, torch.uint8).contiguous()
        assert seat.numel() == n and int(seat.max()) <= 1 if n else True
        self.seat = seat if self.opponent else None
        self._learner = seat.to(torch.int8)  # seat of the reward: the learner's, or in self-play the seat that acted (set per step)
        self.w_opp = self.idx_opp = None
        if self.opponent == 3:
            if opponent_weights is None:
                raise ValueError("opponent='heuristic' needs opponent_weights")
            self.w_opp = FitnessEvaluator._weight_table(opponent_weights, dev)
            if opponent_index is not None:
                self.idx_opp = torch.as_tensor(opponent_index).to(dev, torch.int32).contiguous()
        self.decks = None if decks is None else torch.as_tensor(decks).to(dev, torch.uint8).contiguous()
        self.factions = None if factions is None else torch.as_tensor(factions).to(dev, torch.uint8).contiguous()
        self.states = self.engine.empty_states(n)
        self.actions = torch.zeros(n, dtype=torch.uint8, device=dev)
        self._out = self.engine._env_outputs(n, {"states": self.states}, ("states", "obs", "masks", "obs_err", "result", "length", "final_states"))
        self.reward = torch.zeros(n, dtype=torch.float32, device=dev)
        self.done = torch.zeros(n, dtype=torch.bool, device=dev)
        self._decided = torch.zeros(n, dtype=torch.bool, device=dev)
        self._bits = torch.arange(32, dtype=torch.int32, device=dev)

    def _env_kw(self):
        return dict(opponent=self.opponent, seat=self.seat, w_opp=self.w_opp, idx_opp=self.idx_opp, max_steps=self.max_steps,
                    decks=self.decks, factions=self.factions)

    def reset(self):
        """Deal every env's first game from `seeds`; the opponent opens where the learner is SECOND."""
        o = self._out
        self.engine.env_reset(self.seeds, out={k: o[k] for k in ("states", "obs", "masks", "obs_err")}, **self._env_kw())
        return o["obs"], o["masks"]

    def step(self, actions):
        """actions: one action id per env (any integer dtype, on the device or the host)."""
        o = self._out
        actions = actions if torch.is_tensor(actions) else torch.as_tensor(np.asarray(actions))
        # ids outside 0..255 become 255, which is never legal: the env rejects them (-4) instead of playing a wrapped u8 id
        self.actions.copy_(torch.where((actions < 0) | (actions > 255), 255, actions))
        if self.opponent == 0:  # self-play: the reward is relative to the seat that acts now
            torch.ne(self.states[:, _PLAYER_SIGN].view(torch.int8), 1, out=self.done)
            self._learner.copy_(self.done)
        self.engine.env_step(self.states, self.actions, out={k: o[k] for k in ("result", "length", "final_states", "obs", "masks", "obs_err")},
                             **self._env_kw())
        r = o["result"]
        torch.eq(r, self._learner, out=self.done)  # result 0 / 1 = the seat that won
        torch.ge(r, 0, out=self._decided)
        self.reward.copy_(self.done).mul_(2).sub_(1).mul_(self._decided)
        torch.gt(r, -3, out=self.done)
        info = {"result": r, "length": o["length"], "final_states": o["final_states"], "obs_err": o["obs_err"]}
        return o["obs"], o["masks"], self.reward, self.done, info

    def to_play(self):
        """u8[n]: the seat to move in each env (0 FIRST, 1 SECOND)."""
        return (self.states[:, _PLAYER_SIGN].view(torch.int8) != 1).to(torch.uint8)

    def action_mask(self):
        """bool[n,156]: the legal actions of the last returned observation."""
        m = self._out["masks"]
        return ((m.unsqueeze(-1) >> self._bits) & 1).reshape(self.n, -1)[:, :N_ACTIONS].bool()

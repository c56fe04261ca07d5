"""TEST INFRASTRUCTURE -- plain-Python statement of the batched environment (sb_env_reset / sb_env_step, include/sb_b200.h).

Built only from the pinned C oracle's primitives (new_game, step, legal_mask, observe, expert_action, select_action and
lib().sbo_agent_pick), one env at a time.  The product package never imports it; the tests compare the kernels against it.
"""
import numpy as np

import sb_oracle as O
from sb_layout import STATE_DTYPE

N_ACTIONS = 156
CONTINUES, REJECTED = -3, -4


def next_seed(s):
    """splitmix64's output function of s + golden gamma, top bit cleared (restated here, not imported from the product)."""
    m = (1 << 64) - 1
    z = (s + 0x9E3779B97F4A7C15) & m
    z ^= z >> 30
    z = (z * 0xBF58476D1CE4E5B9) & m
    z ^= z >> 27
    z = (z * 0x94D049BB133111EB) & m
    z ^= z >> 31
    return z & ((1 << 63) - 1)


def fields(st):
    return st.view(STATE_DTYPE)[0]


def key(st):
    f = fields(st)
    return int(f["seed_lo"]) | (int(f["seed_hi"]) << 32)


def to_move(st):
    return 0 if int(fields(st)["player_sign"]) == 1 else 1


def legal_actions(st):
    bits = np.unpackbits(O.legal_mask(st).view(np.uint8), bitorder="little")[:N_ACTIONS]
    return np.flatnonzero(bits).tolist()


class EnvModel:
    """One env: decks (deck0, deck1) and factions (f0, f1) of its games; opponent 0 none, 1 random, 2 expert, 3 heuristic
    with weight row w_opp; seat = the learner's (0 FIRST, 1 SECOND)."""

    def __init__(self, decks, factions, opponent, seat=0, w_opp=None, max_steps=400):
        self.decks, self.factions = decks, factions
        self.opponent, self.seat, self.w_opp, self.max_steps = opponent, seat, w_opp, max_steps

    def over(self, st):
        f = fields(st)
        return bool(f["pl"][0]["base"] < 0 or f["pl"][1]["base"] < 0 or f["err"] or f["steps"] >= self.max_steps)

    @staticmethod
    def result(st):
        f = fields(st)
        if f["err"]:
            return -2
        l0, l1 = f["pl"][0]["base"] < 0, f["pl"][1]["base"] < 0
        return 0 if (l1 and not l0) else 1 if (l0 and not l1) else -1

    def _opponent_action(self, st):
        if self.opponent == 1:
            legal = legal_actions(st)
            return legal[O.lib().sbo_agent_pick(key(st), int(fields(st)["steps"]), len(legal))]
        if self.opponent == 2:
            return O.expert_action(st)  # draws from the game's stream: st changes before the step
        return O.select_action(st, self.w_opp)[0]

    def _opponent_plays(self, st):
        while self.opponent and to_move(st) != self.seat and not self.over(st):
            O.step(st, self._opponent_action(st))

    def reset(self, seed):
        st = O.new_game(seed, self.decks[0], self.decks[1], int(self.factions[0]), int(self.factions[1]))
        self._opponent_plays(st)
        return st

    def step(self, st, action):
        """-> (record, result, length, finished record or None); `st` itself is left alone."""
        if action >= N_ACTIONS or action not in legal_actions(st):
            return st.copy(), REJECTED, 0, None
        st = st.copy()
        O.step(st, action)
        self._opponent_plays(st)
        if not self.over(st):
            return st, CONTINUES, 0, None
        return self.reset(next_seed(key(st))), self.result(st), int(fields(st)["steps"]), st

    @staticmethod
    def outputs(st):
        """(observation i32[27,5,4], observe()'s error code, legal mask as i32[5])"""
        obs, err = O.observe(st)
        return obs, err, O.legal_mask(st).view(np.int32)

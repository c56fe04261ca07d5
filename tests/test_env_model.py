"""CPU: the environment's seed chain and the plain-Python env model (tests/sb_env_model.py) against the oracle's own game loops."""
import numpy as np
import pytest

import sb_oracle
from sb_env_model import CONTINUES, REJECTED, EnvModel, legal_actions, next_seed
from monsoon_b200.engine import DEFAULT_DECKS, DEFAULT_FACTIONS, deck_indices
from monsoon_b200 import vec_env

DECKS = [np.array(deck_indices(d), dtype=np.uint8) for d in DEFAULT_DECKS]


def test_next_seed_scalar_numpy_and_model_agree():
    rs = np.random.RandomState(11)
    seeds = rs.randint(0, 2**63, size=10000, dtype=np.int64).astype(np.uint64)
    seeds[:5000] |= np.uint64(1 << 63)  # the whole 64-bit key range, not only what next_seed itself returns
    seeds[:4] = np.array([0, 1, 2**64 - 1, 2**63], dtype=np.uint64)
    got = vec_env.next_seed_array(seeds)
    assert got.dtype == np.int64 and (got >= 0).all()
    for s, g in zip(seeds.tolist(), got.tolist()):
        assert vec_env.next_seed(s) == next_seed(s) == g, s


def play(model, seed, w_learner):
    """the learner plays oracle.select_action until the first episode ends -> (result, length, finished record)"""
    st = model.reset(seed)
    while True:
        st, res, length, final = model.step(st, sb_oracle.select_action(st, w_learner)[0])
        if res != CONTINUES:
            return res, length, final


@pytest.mark.parametrize("seat", [0, 1])
def test_model_reproduces_play_heuristic(oracle, seat):
    rs = np.random.RandomState(5 + seat)
    for seed in range(40):
        wl, wo = rs.uniform(-1, 1, 10), rs.uniform(-1, 1, 10)
        for opponent, w_opp in ((3, wo), (2, None)):
            model = EnvModel(DECKS, DEFAULT_FACTIONS, opponent, seat, w_opp)
            res, length, final = play(model, seed, wl)
            st = oracle.new_game(seed, DECKS[0], DECKS[1], *DEFAULT_FACTIONS)
            wf, ws = (wl, w_opp) if seat == 0 else (w_opp, wl)
            r, acts = oracle.play_heuristic(st, wf, ws, 400)
            assert (res, length) == (r, len(acts)), (opponent, seat, seed)
            assert final.tobytes() == st.tobytes(), (opponent, seat, seed)


def test_illegal_action_is_rejected_and_leaves_the_record(oracle):
    for opponent in range(4):
        model = EnvModel(DECKS, DEFAULT_FACTIONS, opponent, 1, np.full(10, 0.5))
        st = model.reset(7)
        legal = set(legal_actions(st))
        illegal = [a for a in range(156) if a not in legal][:3] + [156, 255]
        for a in illegal:
            out, res, length, final = model.step(st, a)
            assert (res, length, final) == (REJECTED, 0, None) and out.tobytes() == st.tobytes()


def test_max_steps_ends_the_episode_as_a_timeout(oracle):
    model = EnvModel(DECKS, DEFAULT_FACTIONS, 0, max_steps=5)
    st = model.reset(3)
    for k in range(5):
        st, res, length, final = model.step(st, legal_actions(st)[0])
        assert res == (CONTINUES if k < 4 else -1)
    assert length == 5 and final is not None
    assert st.tobytes() == oracle.new_game(next_seed(int(final.view(np.uint32)[0]) | int(final.view(np.uint32)[1]) << 32),
                                           DECKS[0], DECKS[1], *DEFAULT_FACTIONS).tobytes()

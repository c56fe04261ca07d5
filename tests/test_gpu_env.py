"""GPU: sb_env_reset / sb_env_step (and StormboundVecEnv) against the plain-Python env model and the pinned entry points."""
import numpy as np
import pytest
import torch

from sb_env_model import CONTINUES, EnvModel, next_seed
from monsoon_b200 import _lib
from monsoon_b200.engine import DEFAULT_DECKS, DEFAULT_FACTIONS, deck_indices
from monsoon_b200.vec_env import StormboundVecEnv, next_seed_array

pytestmark = pytest.mark.gpu

DECKS = np.array([deck_indices(d) for d in DEFAULT_DECKS], dtype=np.uint8)


def pick(mask_words, g, call):
    """the learner: a fixed hash of (env, call) over the legal set; every 13th choice is an illegal action (rejected, -4)"""
    h = ((g * 0x9E3779B1) ^ (call * 0x85EBCA77)) & 0xFFFFFFFF
    h = (h ^ (h >> 15)) * 0x2C1B3C6D & 0xFFFFFFFF
    bits = np.unpackbits(np.ascontiguousarray(mask_words).view(np.uint8), bitorder="little")[:156]
    if h % 13 == 0:
        illegal = np.flatnonzero(bits == 0)
        return int(illegal[0]) if len(illegal) else 200
    legal = np.flatnonzero(bits)
    return int(legal[(h >> 4) % len(legal)])


def run_against_model(engine, opponent, n, seeds, seats, decks, factions, w_opp=None, idx_opp=None, max_steps=400):
    dev = engine.device
    per_env = decks.ndim == 3
    models = [EnvModel(decks[g] if per_env else decks, factions[g] if per_env else factions, opponent, int(seats[g]),
                       None if w_opp is None else w_opp[g if idx_opp is None else idx_opp[g]], max_steps) for g in range(n)]
    kw = dict(opponent=opponent, seat=torch.from_numpy(seats).to(dev), max_steps=max_steps, decks=torch.from_numpy(decks).to(dev),
              factions=torch.from_numpy(np.ascontiguousarray(factions)).to(dev),
              w_opp=None if w_opp is None else torch.from_numpy(w_opp).to(dev),
              idx_opp=None if idx_opp is None else torch.from_numpy(idx_opp).to(dev))
    o = engine.env_reset(torch.from_numpy(seeds).to(dev), **kw)
    states = o["states"]
    want = [m.reset(int(seeds[g])) for g, m in enumerate(models)]

    def compare(o, call):
        got = states.cpu().numpy()
        obs, masks, oerr = o["obs"].cpu().numpy(), o["masks"].cpu().numpy(), o["obs_err"].cpu().numpy()
        for g in range(n):
            assert got[g].tobytes() == want[g].tobytes(), (opponent, call, g)
            wo, we, wm = EnvModel.outputs(want[g])
            assert np.array_equal(obs[g], wo) and int(oerr[g]) == we and np.array_equal(masks[g], wm), (opponent, call, g)
        return masks

    masks = compare(o, -1)
    episodes = np.zeros(n, dtype=np.int64)
    counts = {}
    call = 0
    while episodes.min() < 2:
        actions = np.array([pick(masks[g], g, call) for g in range(n)], dtype=np.uint8)
        o = engine.env_step(states, torch.from_numpy(actions).to(dev), **kw)
        res, length, final = o["result"].cpu().numpy(), o["length"].cpu().numpy(), o["final_states"].cpu().numpy()
        for g in range(n):
            want[g], r, ln, fin = models[g].step(want[g], int(actions[g]))
            assert (int(res[g]), int(length[g])) == (r, ln), (opponent, call, g)
            if fin is not None:
                assert final[g].tobytes() == fin.tobytes(), (opponent, call, g)
                episodes[g] += 1
            counts[r] = counts.get(r, 0) + 1
        masks = compare(o, call)
        call += 1
    return counts


def opponent_table(n, p=5):
    rs = np.random.RandomState(17)
    return rs.uniform(-1, 1, (p, 10)), (np.arange(n) % p).astype(np.int32)


@pytest.mark.parametrize("opponent", [0, 1, 2, 3])
def test_env_matches_model_default_decks(engine, oracle, opponent):
    n = 257
    seeds = next_seed_array(np.arange(n) + 1000 * opponent)
    seats = (np.arange(n) % 2).astype(np.uint8)
    w, idx = opponent_table(n) if opponent == 3 else (None, None)
    counts = run_against_model(engine, opponent, n, seeds, seats, DECKS, np.array(DEFAULT_FACTIONS, dtype=np.uint8), w, idx)
    assert counts.get(-4, 0) > 0 and counts.get(0, 0) > 0 and counts.get(1, 0) > 0, counts


@pytest.mark.parametrize("opponent", [0, 1, 2])
def test_env_matches_model_random_decks(engine, oracle, opponent):
    n = 257
    seeds = next_seed_array(np.arange(n) + 5000 + 1000 * opponent)
    fac = np.stack([1 + seeds % 4, 1 + (seeds // 4) % 4], axis=1).astype(np.uint8)
    decks, _ = engine.generate_decks(seeds, 3, 3, factions=fac)
    seats = ((np.arange(n) // 3) % 2).astype(np.uint8)
    counts = run_against_model(engine, opponent, n, seeds, seats, decks.cpu().numpy(), fac)
    assert counts.get(-2, 0) > 0, counts  # these seeds reach engine statuses (unsupported / overflow) in every opponent kind


def _first_episodes(engine, n, seeds, seats, learner_w, **kw):
    """the learner plays sb_select_action with rows of learner_w until every env has finished one episode"""
    dev = engine.device
    o = engine.env_reset(seeds, seat=seats, **kw)
    states = o["states"]
    res = torch.full((n,), -3, dtype=torch.int8, device=dev)
    length = torch.zeros(n, dtype=torch.int32, device=dev)
    final = torch.zeros((n, 512), dtype=torch.uint8, device=dev)
    after = torch.zeros((n, 512), dtype=torch.uint8, device=dev)
    for _ in range(2000):
        a, _s = engine.select_action(states, learner_w)
        o = engine.env_step(states, a, seat=seats, **kw)
        first = (res == CONTINUES) & (o["result"] != CONTINUES)
        res = torch.where(first, o["result"], res)
        length = torch.where(first, o["length"], length)
        final = torch.where(first[:, None], o["final_states"], final)
        after = torch.where(first[:, None], states, after)
        if not bool((res == CONTINUES).any()):
            break
    return res.cpu().numpy(), length.cpu().numpy(), final.cpu().numpy(), after.cpu().numpy()


def test_env_cross_checks_against_rollout_heuristic(engine):
    n = 1024
    dev = engine.device
    seeds = torch.from_numpy(next_seed_array(np.arange(n) + 77)).to(dev)
    seats_np = (np.arange(n) % 2).astype(np.uint8)
    seats = torch.from_numpy(seats_np).to(dev)
    rs = np.random.RandomState(23)
    wl, wo = torch.from_numpy(rs.uniform(-1, 1, (n, 10))).to(dev), torch.from_numpy(rs.uniform(-1, 1, (n, 10))).to(dev)
    first_seat = torch.from_numpy(seats_np == 0).to(dev)[:, None]
    for opponent in (3, 2):
        kw = dict(opponent=opponent, w_opp=wo if opponent == 3 else None)
        res, length, final, after = _first_episodes(engine, n, seeds, seats, wl, **kw)
        states = engine.reset(seeds)
        if opponent == 3:
            rr, rl = engine.rollout_heuristic(states, torch.where(first_seat, wl, wo).contiguous(), torch.where(first_seat, wo, wl).contiguous())
        else:  # the expert plays the seat without a table
            rr, rl = torch.empty(n, dtype=torch.int8, device=dev), torch.empty(n, dtype=torch.int32, device=dev)
            for s in (0, 1):
                sel = torch.nonzero(seats == s).flatten()
                sub = states[sel].contiguous()
                w = wl[sel].contiguous()
                r, l = engine.rollout_heuristic(sub, w if s == 0 else None, None if s == 0 else w)
                states[sel], rr[sel], rl[sel] = sub, r, l
        assert np.array_equal(res, rr.cpu().numpy()) and np.array_equal(length, rl.cpu().numpy()), opponent
        assert np.array_equal(final, states.cpu().numpy()), opponent
        # the second episode of env g is dealt from next_seed of the first episode's key, i.e. next_seed(seed_g)
        nxt = torch.from_numpy(next_seed_array(seeds.cpu().numpy())).to(dev)
        want = engine.env_reset(nxt, seat=seats, **kw)["states"].cpu().numpy()
        assert np.array_equal(after, want), opponent
        plain = engine.reset(nxt).cpu().numpy()
        assert np.array_equal(after[seats_np == 0], plain[seats_np == 0]), opponent
    assert next_seed(int(seeds[0])) == int(nxt[0])


def test_env_launches_nullable_outputs_and_rejected_arguments(engine):
    dev = engine.device
    n = 300
    seeds = torch.from_numpy(next_seed_array(np.arange(n))).to(dev)
    w = torch.rand((4, 10), dtype=torch.float64, device=dev)
    idx = (torch.arange(n, device=dev) % 4).to(torch.int32)
    for opponent in range(4):
        kw = dict(opponent=opponent, w_opp=w, idx_opp=idx, seat=(torch.arange(n, device=dev) % 2).to(torch.uint8))
        o = engine.env_reset(seeds, **kw)
        st = o["states"]
        before = engine.launches
        a = torch.full((n,), 155, dtype=torch.uint8, device=dev)  # PASS (legal or rejected, both are outputs)
        st2 = st.clone()
        full = engine.env_step(st, a, **kw)
        torch.cuda.synchronize()
        assert engine.launches == before + 1
        bare = engine.env_step(st2, a, out={"obs": None, "masks": None, "obs_err": None, "final_states": None}, **kw)
        assert torch.equal(st, st2) and torch.equal(full["result"], bare["result"]) and torch.equal(full["length"], bare["length"])
        half = engine.env_step(st.clone(), a, out={"obs": None}, **kw)  # obs_err without obs
        full2 = engine.env_step(st2, a, **kw)
        assert torch.equal(half["obs_err"], full2["obs_err"]) and torch.equal(half["masks"], full2["masks"])
        before = engine.launches
        empty = engine.env_step(st[:0], a[:0], **dict(kw, seat=None, idx_opp=None))
        engine.env_reset(seeds[:0], **dict(kw, seat=None, idx_opp=None))
        assert engine.launches == before and empty["result"].numel() == 0
    bad = [dict(opponent=4), dict(opponent=-1), dict(opponent=3, w_opp=None), dict(max_steps=0), dict(max_steps=65536),
           dict(decks=torch.ones((2, 17), dtype=torch.uint8, device=dev), factions=torch.zeros(2, dtype=torch.uint8, device=dev)),
           dict(decks=torch.ones((2, 0), dtype=torch.uint8, device=dev), factions=torch.zeros(2, dtype=torch.uint8, device=dev))]
    st = engine.env_reset(seeds)["states"]
    a = torch.zeros(n, dtype=torch.uint8, device=dev)
    for b in bad:
        before = engine.launches
        with pytest.raises(_lib.SbError):
            engine.env_step(st, a, **b)
        with pytest.raises(_lib.SbError):
            engine.env_reset(seeds, **b)
        assert engine.launches == before, b


@pytest.mark.parametrize("opponent", [None, "expert", "heuristic"])
def test_vec_env_step_in_a_cuda_graph(engine, opponent):
    n = 512
    kw = dict(seed=9, opponent=opponent, seats=[g % 2 for g in range(n)], opponent_weights=torch.rand((n, 10), dtype=torch.float64),
              engine=engine)
    eager, graphed = StormboundVecEnv(n, **kw), StormboundVecEnv(n, **kw)
    eager.reset()
    graphed.reset()
    static_actions = torch.zeros(n, dtype=torch.int64, device=engine.device)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        graphed.step(static_actions)  # warm-up outside the capture
    torch.cuda.current_stream().wait_stream(side)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        outs = graphed.step(static_actions)
    graphed.states.copy_(eager.states)
    graphed._out["masks"].copy_(eager._out["masks"])
    rs = np.random.RandomState(4)
    seen_done = 0
    for call in range(150):
        mask = eager.action_mask().cpu().numpy()
        acts = np.array([rs.choice(np.flatnonzero(m)) for m in mask])
        static_actions.copy_(torch.from_numpy(acts))
        g.replay()
        obs, masks, reward, done, info = eager.step(torch.from_numpy(acts).to(engine.device))
        torch.cuda.synchronize()
        assert torch.equal(graphed.states, eager.states), call
        for x, y in zip(outs[:4], (obs, masks, reward, done)):
            assert torch.equal(x, y), call
        for k in info:
            assert torch.equal(outs[4][k][done], info[k][done]) if k == "final_states" else torch.equal(outs[4][k], info[k]), (call, k)
        assert torch.equal(graphed.to_play(), eager.to_play())
        r = info["result"].cpu().numpy()
        seat = eager._learner.cpu().numpy()
        rw = reward.cpu().numpy()
        for i in np.flatnonzero(r >= 0):
            assert rw[i] == (1.0 if r[i] == seat[i] else -1.0)
        assert (rw[r < 0] == 0).all()
        seen_done += int(done.sum())
    assert seen_done > 0


def test_out_of_range_actions_and_seat_bytes(engine):
    n = 64
    env = StormboundVecEnv(n, seed=1, opponent="random", engine=engine)
    env.reset()
    legal = env.action_mask().to(torch.int32).argmax(1).to(torch.int64)  # one legal id per env
    before = env.states.clone()
    _o, _m, reward, done, info = env.step(legal + 256)  # would wrap to a legal id in a u8 cast
    assert (info["result"] == -4).all() and torch.equal(env.states, before) and not done.any() and not reward.any()
    _o, _m, _r, _d, info = env.step(torch.full((n,), -1, dtype=torch.int64, device=engine.device))
    assert (info["result"] == -4).all() and torch.equal(env.states, before)
    seeds = env.seeds
    second = engine.env_reset(seeds, opponent=2, seat=torch.ones(n, dtype=torch.uint8, device=engine.device))["states"]
    other = engine.env_reset(seeds, opponent=2, seat=torch.full((n,), 7, dtype=torch.uint8, device=engine.device))["states"]
    assert torch.equal(second, other)  # any non-zero seat byte is SECOND

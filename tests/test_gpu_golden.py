"""GPU vs the golden fixtures produced by the reference itself (no oracle in between)."""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def load(name):
    p = os.path.join(G, name)
    if not os.path.exists(p):
        pytest.skip("fixture %s not generated" % name)
    return np.load(p)


def test_10k_default_games_rollout_kernel(engine):
    z = load("default_chain_10k.npz")
    ok = z["err"] == 0
    seeds = torch.from_numpy(z["seeds"].astype(np.int64)).to(engine.device)
    st = engine.reset(seeds)
    chain = torch.zeros(len(seeds), dtype=torch.int64, device=engine.device)
    steps = engine.rollout_random(st, 400, chain=chain)
    steps, chain = steps.cpu().numpy(), chain.cpu().numpy().view(np.uint64)
    assert np.array_equal(steps[ok], z["steps"][ok])
    assert np.array_equal(chain[ok], z["chain"][ok])
    host = st.cpu().numpy()
    assert (host[~ok][:, 18] != 0).all()  # games where the reference raised are flagged


def test_10k_default_games_lane_refill(engine):
    """Same fixture through the persistent-lane schedule (finished lanes take the next game from a counter):
    1,024 lanes play 10,000 games, results must not depend on which lane played which game."""
    z = load("default_chain_10k.npz")
    ok = z["err"] == 0
    seeds = torch.from_numpy(z["seeds"].astype(np.int64)).to(engine.device)
    try:
        for bs, grid, dense in ((128, 8, 0), (256, 5, 0), (512, 4, 0), (1024, 2, 0), (1024, 3, 1)):  # dense = the 32-register, two-CTAs-per-SM variant
            engine.set_option("refill", 1)
            engine.set_option("block_sync", bs)
            engine.set_option("refill_grid", grid)
            engine.set_option("dense", dense)
            engine.set_option("games_per_warp", 32)
            st = engine.reset(seeds)
            chain = torch.zeros(len(seeds), dtype=torch.int64, device=engine.device)
            steps = engine.rollout_random(st, 400, chain=chain)
            steps, chain = steps.cpu().numpy(), chain.cpu().numpy().view(np.uint64)
            assert np.array_equal(steps[ok], z["steps"][ok]), bs
            assert np.array_equal(chain[ok], z["chain"][ok]), bs
            assert (st.cpu().numpy()[~ok][:, 18] != 0).all()
    finally:
        for k, v in (("refill", -1), ("block_sync", -1), ("refill_grid", 0), ("games_per_warp", 0), ("dense", -1)):
            engine.set_option(k, v)


def test_random_deck_games_rollout_kernel(engine):
    z = load("randdeck_chain.npz")
    dev = engine.device
    st = engine.reset(torch.from_numpy(z["seeds"].astype(np.int64)).to(dev), torch.from_numpy(z["decks"]).to(dev),
                      torch.from_numpy(z["factions"]).to(dev))
    chain = torch.zeros(len(z["seeds"]), dtype=torch.int64, device=dev)
    steps = engine.rollout_random(st, 400, chain=chain)
    host = st.cpu().numpy()
    steps, chain = steps.cpu().numpy(), chain.cpu().numpy().view(np.uint64)
    unsupported = (host[:, 18] == 5) | ((host[:, 18] == 6) & ((z["err"] != 2) | (steps <= z["steps"])))
    clean = (z["err"] == 0) & ~unsupported
    assert np.array_equal(steps[clean], z["steps"][clean]) and np.array_equal(chain[clean], z["chain"][clean])
    raised = (z["err"] != 0) & ~unsupported
    assert (host[raised][:, 18] != 0).all() and np.array_equal(steps[raised], z["steps"][raised] + 1)
    assert unsupported.sum() <= len(unsupported) * 3 // 200


def test_card_focus_games_rollout_kernel(engine):
    """card_focus.npz: all 112 cards (S203 and UP01-03 included) in decks stacked toward each card, reference tapes."""
    z = load("card_focus.npz")
    dev = engine.device
    st = engine.reset(torch.from_numpy(z["seeds"].astype(np.int64)).to(dev), torch.from_numpy(z["decks"]).to(dev),
                      torch.from_numpy(z["factions"]).to(dev))
    chain = torch.zeros(len(z["seeds"]), dtype=torch.int64, device=dev)
    steps = engine.rollout_random(st, 400, chain=chain)
    host = st.cpu().numpy()
    steps, chain = steps.cpu().numpy(), chain.cpu().numpy().view(np.uint64)
    unsupported = (host[:, 18] == 5) | ((host[:, 18] == 6) & ((z["err"] != 2) | (steps <= z["steps"])))
    clean = (z["err"] == 0) & ~unsupported
    assert np.array_equal(steps[clean], z["steps"][clean]) and np.array_equal(chain[clean], z["chain"][clean])
    raised = (z["err"] != 0) & ~unsupported
    assert (host[raised][:, 18] != 0).all() and np.array_equal(steps[raised], z["steps"][raised] + 1)
    assert unsupported.sum() <= len(unsupported) * 3 // 200


def test_observation_and_features_vs_reference(engine):
    """sb_observe / sb_features against the reference's own get_observation / StateFeatures (rows a11, a12): exact."""
    z = load("obs_features.npz")
    st = torch.from_numpy(z["states"]).to(engine.device)
    obs, err = engine.observe(st)
    assert int(err.max()) == 0 and np.array_equal(obs.cpu().numpy(), z["obs"])
    f, err = engine.features(st)
    assert int(err.max()) == 0
    f = f.cpu().numpy()
    assert np.array_equal(f, z["feat"]), np.abs(f - z["feat"]).max()


def test_deck_generation_kernel(engine):
    """sb_generate_decks against the decks the reference's utils.py produced (every schedule phase, both
    random.sample call shapes), batched by identical parameters."""
    z = load("deck_generation.npz")
    key = np.stack([z["generation"], z["mode"], z["n_preserve"], (z["q"] * 1000).astype(np.uint32)], axis=1)
    done = 0
    for u in np.unique(key, axis=0):
        sel = np.nonzero((key == u).all(axis=1))[0]
        mode = int(u[1])
        if mode == 3:
            decks, fout = engine.generate_decks(z["seeds"][sel].astype(np.int64), int(u[0]), 3, factions=z["factions"][sel])
        else:
            i0 = sel[0]
            assert (z["archetypes"][sel] == z["archetypes"][i0]).all()
            decks, fout = engine.generate_decks(z["seeds"][sel].astype(np.int64), int(u[0]), mode, int(u[2]), float(z["q"][i0]),
                                                z["archetypes"][i0], z["factions"][i0])
        assert np.array_equal(decks.cpu().numpy().reshape(len(sel), 24), z["decks"][sel]), u
        assert np.array_equal(fout.cpu().numpy(), z["factions"][sel])
        done += len(sel)
    assert done == len(z["seeds"])


def fnv1a64_rows(rows):
    """fnv1a64 of every 512-byte row (the digest the fixtures store), vectorised over games"""
    h = np.full(rows.shape[0], 0xCBF29CE484222325, dtype=np.uint64)
    prime = np.uint64(0x100000001B3)
    with np.errstate(over="ignore"):
        for b in range(rows.shape[1]):
            h = (h ^ rows[:, b].astype(np.uint64)) * prime
    return h


def test_expert_games_step_api(engine):
    """sb_expert_action + sb_step against the reference's expert-vs-expert tapes: every action, every state digest."""
    z = load("expert_tapes.npz")
    dev = engine.device
    n = len(z["seeds"])
    st = engine.reset(torch.from_numpy(z["seeds"].astype(np.int64)).to(dev), torch.from_numpy(z["decks"]).to(dev),
                      torch.from_numpy(z["factions"]).to(dev))
    assert np.array_equal(st.cpu().numpy(), z["init"])
    steps, lengths = z["steps"].astype(np.int64), z["lengths"].astype(np.int64)
    aoff = np.concatenate([[0], np.cumsum(lengths)[:-1]])
    doff = np.concatenate([[0], np.cumsum(steps)[:-1]])
    tolerated = np.zeros(n, dtype=bool)
    raised = np.zeros(n, dtype=bool)
    for k in range(int(lengths.max()) + 1):
        # games still inside their tape; a game the reference aborted gets its aborting action (or expert call) too
        live = np.nonzero(((k < steps) | ((k == steps) & (z["err"] != 0))) & ~tolerated)[0]
        if live.size == 0:
            break
        idx = torch.from_numpy(live).to(dev)
        sub = st.index_select(0, idx).contiguous()
        act = engine.expert_action(sub)
        a = act.cpu().numpy()
        expert_err = sub[:, 18].cpu().numpy() != 0
        _r, _d, err = engine.step(sub, act)
        st.index_copy_(0, idx, sub)
        host, err = sub.cpu().numpy(), err.cpu().numpy()
        inside = k < steps[live]
        tolerated[live[inside & ((err == 5) | (err == 6))]] = True
        chk = inside & (err != 5) & (err != 6)
        g = live[chk]
        assert np.array_equal(a[chk], z["actions"][aoff[g] + k]), k
        assert np.array_equal(fnv1a64_rows(host[chk]), z["digests"][doff[g] + k]), k
        last = live[~inside]
        kinds = z["err"][last]
        same_action = (kinds == 3) | (a[~inside] == z["actions"][np.minimum(aoff[last] + k, len(z["actions"]) - 1)])
        assert same_action.all(), k
        raised[last] = (err[~inside] != 0) | expert_err[~inside]
    assert raised[(z["err"] != 0) & ~tolerated].all()
    assert tolerated.sum() <= n * 3 // 200


def test_heuristic_decisions(engine):
    z = load("heuristic_decisions.npz")
    st = torch.from_numpy(z["states"]).to(engine.device)
    w = torch.from_numpy(z["weights"]).to(engine.device)
    actions, scores = engine.select_action(st, w, want_scores=True)
    actions, scores = actions.cpu().numpy(), scores.cpu().numpy()
    for i in range(len(actions)):
        ref = z["scores"][i]
        legal = ~np.isnan(ref)
        assert np.array_equal(legal, ~np.isnan(scores[i]))
        np.testing.assert_allclose(scores[i][legal], ref[legal], rtol=1e-5, atol=1e-9)
        top = np.sort(ref[legal])[::-1]
        if len(top) == 1 or top[0] - top[1] > 1e-5 * max(1.0, abs(top[0])):
            assert int(actions[i]) == int(z["chosen"][i]), i


def test_heuristic_whole_games(engine):
    z = load("heuristic_decisions.npz")
    dev = engine.device
    st = engine.reset(torch.from_numpy(z["game_seeds"].astype(np.int64)).to(dev))
    res, steps = engine.rollout_heuristic(st, torch.from_numpy(z["w_first"]).to(dev), torch.from_numpy(z["w_second"]).to(dev), max_steps=400)
    assert np.array_equal(steps.cpu().numpy(), z["game_lengths"])
    assert np.array_equal(res.cpu().numpy(), z["game_result"])


def test_heuristic_vs_expert_games(engine):
    """sb_rollout_heuristic with one seat handed to the scripted opponent, against the reference's own games
    (HeuristicAgent vs Stormbound.expert_action, both seatings): winner, length and final state."""
    z = load("heuristic_vs_expert.npz")
    dev = engine.device
    for seat in (0, 1):
        sel = np.nonzero(z["seat"] == seat)[0]
        st = engine.reset(torch.from_numpy(z["seeds"][sel].astype(np.int64)).to(dev))
        w = torch.from_numpy(z["weights"][sel]).to(dev)
        res, steps = engine.rollout_heuristic(st, w if seat == 0 else None, w if seat == 1 else None, max_steps=400)
        res, steps, host = res.cpu().numpy(), steps.cpu().numpy(), st.cpu().numpy()
        assert np.array_equal(res, z["result"][sel])
        ok = z["result"][sel] != -2
        assert np.array_equal(steps[ok], z["lengths"][sel][ok])
        host[:, 19] = 0  # the fixture's final state was packed without the done/reward byte
        assert np.array_equal(fnv1a64_rows(host[ok]), z["final"][sel][ok])


def test_heuristic_games_at_scale(engine):
    """BASELINE config 1 on the GPU: the 1,024 reference HeuristicAgent-vs-HeuristicAgent games in one launch."""
    z = load("heuristic_games.npz")
    dev = engine.device
    st = engine.reset(torch.from_numpy(z["seeds"].astype(np.int64)).to(dev))
    res, steps = engine.rollout_heuristic(st, torch.from_numpy(z["w_first"]).to(dev), torch.from_numpy(z["w_second"]).to(dev), max_steps=400)
    res, steps, host = res.cpu().numpy(), steps.cpu().numpy(), st.cpu().numpy()
    assert np.array_equal(res, z["result"])
    ok = z["result"] != -2
    assert np.array_equal(steps[ok], z["lengths"][ok])
    host[:, 19] = 0
    assert np.array_equal(fnv1a64_rows(host[ok]), z["final"][ok])



@pytest.mark.parametrize("iw,grid", [(4, 6), (8, 5), (16, 3), (8, 0)])
def test_heuristic_games_with_warp_refill(engine, iw, grid):
    """The persistent shape of the heuristic rollout (a warp whose game ended takes the next game from a counter) on a grid
    much smaller than the batch: the same 1,024 reference games, same winners, lengths and final states."""
    z = load("heuristic_games.npz")
    dev = engine.device
    try:
        engine.set_option("heur_refill", 1)
        engine.set_option("heur_iw", iw)
        engine.set_option("heur_grid", grid)
        st = engine.reset(torch.from_numpy(z["seeds"].astype(np.int64)).to(dev))
        res, steps = engine.rollout_heuristic(st, torch.from_numpy(z["w_first"]).to(dev), torch.from_numpy(z["w_second"]).to(dev), max_steps=400)
        res, steps, host = res.cpu().numpy(), steps.cpu().numpy(), st.cpu().numpy()
    finally:
        for k, v in (("heur_refill", -1), ("heur_iw", -1), ("heur_grid", 0)):
            engine.set_option(k, v)
    assert np.array_equal(res, z["result"])
    ok = z["result"] != -2
    assert np.array_equal(steps[ok], z["lengths"][ok])
    host[:, 19] = 0
    assert np.array_equal(fnv1a64_rows(host[ok]), z["final"][ok])


def test_heuristic_vs_expert_with_warp_refill(engine):
    """Refill shape with one seat handed to the scripted opponent: identical to the one-wave shape."""
    dev = engine.device
    seeds = torch.arange(3000, dtype=torch.int64, device=dev) + 777
    w = torch.from_numpy(np.random.RandomState(5).uniform(0, 1, (3000, 10))).to(dev)
    out = []
    for refill, grid in ((0, 0), (1, 7)):
        try:
            engine.set_option("heur_refill", refill)
            engine.set_option("heur_grid", grid)
            st = engine.reset(seeds)
            res, steps = engine.rollout_heuristic(st, w, None, max_steps=400)
            out.append((res.cpu().numpy(), steps.cpu().numpy(), st.cpu().numpy()))
        finally:
            engine.set_option("heur_refill", -1)
            engine.set_option("heur_grid", 0)
    for a, b in zip(out[0], out[1]):
        assert np.array_equal(a, b)


@pytest.mark.parametrize("pack,grid", [(1, 0), (2, 0), (3, 0), (4, 0), (8, 0), (4, 3), (8, 5), (1, 7)])
def test_heuristic_games_packed_warps(engine, pack, grid):
    """K games per warp (k_rollout_heuristic_packed: candidates of K games dealt to the 32 lanes, segmented arg-max, the owner
    lane re-applies the winner): the 1,024 whole reference HeuristicAgent games again, also from a grid far smaller than the batch."""
    z = load("heuristic_games.npz")
    dev = engine.device
    try:
        engine.set_option("heur_pack", pack)
        engine.set_option("heur_grid", grid)
        st = engine.reset(torch.from_numpy(z["seeds"].astype(np.int64)).to(dev))
        res, steps = engine.rollout_heuristic(st, torch.from_numpy(z["w_first"]).to(dev), torch.from_numpy(z["w_second"]).to(dev), max_steps=400)
        res, steps, host = res.cpu().numpy(), steps.cpu().numpy(), st.cpu().numpy()
    finally:
        for k, v in (("heur_pack", -1), ("heur_grid", 0)):
            engine.set_option(k, v)
    assert np.array_equal(res, z["result"])
    ok = z["result"] != -2
    assert np.array_equal(steps[ok], z["lengths"][ok])
    host[:, 19] = 0
    assert np.array_equal(fnv1a64_rows(host[ok]), z["final"][ok])


def test_heuristic_vs_expert_packed_warps(engine):
    """Packed shape with one seat handed to the scripted opponent, and random decks (all cards): identical to the one-game-per-warp kernel."""
    dev = engine.device
    seeds = torch.arange(3000, dtype=torch.int64, device=dev) + 777
    w = torch.from_numpy(np.random.RandomState(5).uniform(0, 1, (3000, 10))).to(dev)
    fac = torch.from_numpy(np.random.RandomState(9).randint(1, 5, (3000, 2)).astype(np.uint8)).to(dev)
    decks, factions = engine.generate_decks(seeds, 0, 3, factions=fac)
    out = []
    for pack in (0, 1, 2, 4, 8):
        try:
            engine.set_option("heur_pack", pack)
            st = engine.reset(seeds)
            res, steps = engine.rollout_heuristic(st, w, None, max_steps=400)
            st2 = engine.reset(seeds, decks, factions)
            res2, steps2 = engine.rollout_heuristic(st2, w, w, max_steps=150)
            out.append(tuple(x.cpu().numpy() for x in (res, steps, st, res2, steps2, st2)))
        finally:
            engine.set_option("heur_pack", -1)
    for other in out[1:]:
        for a, b in zip(out[0], other):
            assert np.array_equal(a, b)

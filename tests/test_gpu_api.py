"""GPU: the drop-in Python layer (reference class contracts) behaves like the oracle / the reference's callers expect."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


class Cfg:
    games_per_pairing = 2
    max_turns = 400
    seed = 11
    num_workers = 128


def test_game_contract(engine, oracle):
    from monsoon_b200.games import Game
    from monsoon_b200.engine import DEFAULT_DECKS, deck_indices
    d0, d1 = (deck_indices(d) for d in DEFAULT_DECKS)
    g = Game(seed=5, engine=engine)
    st = oracle.new_game(5, d0, d1, 3, 2)
    obs = g.reset()
    assert obs.shape == (27, 5, 4) and obs.dtype == np.int32 and np.array_equal(obs, oracle.observe(st)[0])
    for step in range(60):
        legal = g.legal_actions()
        m = oracle.legal_mask(st)
        assert legal == [a for a in range(156) if m[a >> 5] >> (a & 31) & 1] and legal == sorted(legal)
        a = legal[step % len(legal)]
        obs, reward, done = g.step(a)
        oracle.step(st, a)
        assert np.array_equal(obs, oracle.observe(st)[0]) and reward in (0, 10) and done == bool(st[19] & 1)
        assert g.to_play() == (0 if np.int8(st[16]) == 1 else 1)
        bases = np.frombuffer(st[32:34].tobytes() + st[136:138].tobytes(), dtype='<i2')
        assert g.env.have_winner() == bool((bases < 0).any())  # `done` is evaluated BEFORE the PASS turn pipeline (Q2)
        if done:
            break
    assert g.action_to_string(155) == "Pass the turn" and len(g.env.actions) == 156


def test_adapter_and_agent(engine, oracle):
    from monsoon_b200.evo import HeuristicAgent, StormboundAdapter, WeightVector, play_game
    from monsoon_b200.games import Game
    np.random.seed(4)
    w1, w2 = WeightVector(10), WeightVector(10)
    ad = StormboundAdapter(Game(seed=9, engine=engine))
    before = ad.game.state.clone()
    a1 = HeuristicAgent(w1, 0)
    legal = ad.get_legal_actions()
    nxt = ad.apply_action(legal[0])
    assert torch.equal(ad.game.state, before) and not torch.equal(nxt.game.state, before)  # functional apply
    f = ad.extract_features()
    assert f.get_feature_vector().shape == (10,) and f.get_feature_names()[0] == "mana_efficiency"
    host = before[0].cpu().numpy()
    a, scores, _m = oracle.select_action(host.copy(), w1.weights)
    assert a1.select_action(ad) == a
    assert abs(a1.score_action(ad, legal[-1]) - scores[legal[-1]]) <= 1e-5 * max(1.0, abs(scores[legal[-1]]))
    end, turns = play_game(ad, a1, HeuristicAgent(w2, 1), max_turns=400)
    r, acts = oracle.play_heuristic(host.copy(), w1.weights, w2.weights, 400)
    assert turns == len(acts) and end.get_result() == r and end.is_terminal() == (r != -1 or turns < 400)


def test_fitness_evaluator_matches_oracle(engine, oracle):
    from monsoon_b200.evo import FitnessEvaluator, WeightVector, game_seed
    from monsoon_b200.engine import DEFAULT_DECKS, deck_indices
    d0, d1 = (deck_indices(d) for d in DEFAULT_DECKS)
    np.random.seed(8)
    pop = [WeightVector(10) for _ in range(4)]
    ev = FitnessEvaluator(Cfg(), engine=engine)
    fit = ev.evaluate_population(pop, generation=2)
    want = np.zeros(4)
    for i in range(4):
        for j in range(4):
            if i == j:
                continue
            for k in range(2):
                st = oracle.new_game(game_seed(11, 2, i, j, k), d0, d1, 3, 2)
                r, _ = oracle.play_heuristic(st, pop[i].weights, pop[j].weights, 400)
                want[i] += 1.0 if r == 0 else 0.5 if r < 0 else 0.0
    assert np.allclose(fit, want / (3 * 2)) and len(fit) == 4 and all(0 <= x <= 1 for x in fit)
    assert len(ev.hall_of_fame) == 4 and ev.get_stats()["total_games"] == 24


def test_fitness_evaluator_with_deck_schedule(engine, oracle):
    """evo/fitness.py:136-141: with a deck_config every game is dealt its own generation-aware decks."""
    from monsoon_b200.evo import DeckEvolutionConfig, FitnessEvaluator, WeightVector, game_seed
    from monsoon_b200.engine import DEFAULT_DECKS
    cfg = DeckEvolutionConfig(DEFAULT_DECKS[0], DEFAULT_DECKS[1], exploit_generations=1, explore_generations=4,
                              max_random_ratio=1.0, balance_archetype_ratio=0.5)
    np.random.seed(9)
    pop = [WeightVector(10) for _ in range(3)]
    arch, fac = [cfg.player1_archetype, cfg.player2_archetype], [cfg.player1_faction, cfg.player2_faction]
    for generation in (0, 3, 7):  # exploit, explore, balance
        ev = FitnessEvaluator(Cfg(), deck_config=cfg, engine=engine)
        fit = ev.evaluate_population(pop, generation=generation)
        mode, keep, q = cfg.phase_parameters(generation)
        want, flagged = np.zeros(3), 0
        for i in range(3):
            for j in range(3):
                if i == j:
                    continue
                for k in range(2):
                    seed = game_seed(11, generation, i, j, k)
                    d = oracle.generate_decks(seed, generation, mode, keep, q, arch, fac)
                    st = oracle.new_game(seed, d[0], d[1], fac[0], fac[1])
                    r, _ = oracle.play_heuristic(st, pop[i].weights, pop[j].weights, 400)
                    flagged += r == -2
                    want[i] += 1.0 if r == 0 else 0.5 if r < 0 else 0.0  # an aborted game (-2) is a draw, like a timeout
        assert np.allclose(fit, want / (2 * 2)), (generation, fit, want, flagged)
        # none of these games aborts, so the draw scoring of -2 is not exercised here (tests/test_gpu_fitness.py does)
        assert flagged == 0 and ev.last_aborted == (0, 0), (generation, flagged, ev.last_aborted)


def test_deck_generation_matches_oracle_at_scale(engine, oracle):
    seeds = (np.arange(6000, dtype=np.int64) * 2654435761) % (1 << 40)
    arch = np.arange(1, 25, dtype=np.uint8).reshape(2, 12)
    for mode, keep, q in ((1, 3, 0.0), (1, 9, 0.0), (2, 0, 0.35), (3, 0, 0.0)):
        fac = np.stack([1 + seeds % 4, 1 + (seeds // 4) % 4], axis=1).astype(np.uint8)
        if mode == 3:
            decks, _ = engine.generate_decks(seeds, 17, 3, factions=fac)
        else:
            decks, _ = engine.generate_decks(seeds, 17, mode, keep, q, arch, [2, 4])
        decks = decks.cpu().numpy()
        for i in range(0, 6000, 7):
            want = oracle.generate_decks(int(seeds[i]), 17, mode, keep, q, arch, fac[i] if mode == 3 else [2, 4])
            assert np.array_equal(decks[i], want), (mode, i)



def test_empty_ragged_and_rejected_inputs(engine):
    """Empty batches are no-ops, a batch that is not a multiple of any CTA / warp size is handled exactly, finished
    games are left alone by the rollouts, and malformed calls fail loudly instead of launching."""
    from monsoon_b200 import _lib
    dev = engine.device
    empty = torch.empty((0, 512), dtype=torch.uint8, device=dev)
    assert engine.legal_mask(empty).shape == (0, 5)
    assert engine.rollout_random(empty, 400).numel() == 0
    assert engine.expert_action(empty).numel() == 0
    res, steps = engine.rollout_heuristic(empty, torch.zeros((0, 10), dtype=torch.float64, device=dev),
                                          torch.zeros((0, 10), dtype=torch.float64, device=dev))
    assert res.numel() == 0 and steps.numel() == 0
    d, f = engine.generate_decks(np.zeros(0, dtype=np.int64), 0, 0, 12, 0.0, np.arange(1, 25, dtype=np.uint8), [1, 2])
    assert d.shape == (0, 2, 12) and f.shape == (0, 2)
    # ragged: 37 and 1 games through every per-game kernel shape; results do not depend on the batch they ran in
    seeds = torch.arange(37, dtype=torch.int64, device=dev) + 9000
    st37 = engine.reset(seeds)
    s37 = engine.rollout_random(st37, 400)
    st1 = engine.reset(seeds[36:37])
    s1 = engine.rollout_random(st1, 400)
    assert int(s1[0]) == int(s37[36]) and torch.equal(st1[0], st37[36])
    # finished games: a second rollout takes zero steps and leaves the records untouched
    before = st37.clone()
    again = engine.rollout_random(st37, 400)
    assert int(again.sum()) == 0 and torch.equal(before, st37)
    w = torch.rand((37, 10), dtype=torch.float64, device=dev)
    res, steps = engine.rollout_heuristic(st37, w, w)
    assert int(steps.sum()) == 0 and torch.equal(before, st37)
    # rejected calls
    with pytest.raises(_lib.SbError):
        engine.generate_decks(seeds, 0, 3)  # fully random decks need per-game factions
    big = torch.zeros((8, 65), dtype=torch.float64, device=dev)
    with pytest.raises(_lib.SbError):
        engine.es_offspring(1, 0, 4, 4, 0.1, 0.01, 1e-5, big, big.clone())  # more than 64 features
    with pytest.raises(_lib.SbError):
        engine.es_select(9, np.zeros(8), big[:, :10].contiguous(), big[:, :10].contiguous())  # mu > rows


def test_evaluate_vs_expert_matches_oracle(engine, oracle):
    from monsoon_b200.evo import FitnessEvaluator, WeightVector, game_seed
    from monsoon_b200.engine import DEFAULT_DECKS, deck_indices
    d0, d1 = (deck_indices(d) for d in DEFAULT_DECKS)
    np.random.seed(12)
    pop = [WeightVector(10) for _ in range(5)]
    ev = FitnessEvaluator(Cfg(), engine=engine)
    fit = ev.evaluate_vs_expert(pop, generation=4, games=3)
    want = np.zeros(5)
    for i in range(5):
        for k in range(3):
            st = oracle.new_game(game_seed(11, 4, i, i, k), d0, d1, 3, 2)
            r, _ = oracle.play_heuristic(st, pop[i].weights, None, 400)
            want[i] += 1.0 if r == 0 else 0.5 if r == -1 else 0.0
    assert np.allclose(fit, want / 3) and ev.get_stats()["total_games"] == 15


def test_dense_variants_give_identical_states(engine):
    """The 32-register (2,048 resident threads per SM) build k_step<true> is normally chosen for batches that fill the
    chip; forced here on a small batch, with 8, 16 and 32 games per warp, it must give the records, rewards, done flags,
    errors and next masks of the default build k_step<false>.  The thread-per-game engine is forced: at this batch size the
    policy picks the warp engine, which has no dense build."""
    dev = engine.device
    n = 300
    seeds = torch.arange(n, dtype=torch.int64, device=dev) + 4242
    outs = {}
    try:
        engine.set_option("engine", 0)
        for dense in (0, 1):
            for gpw in (8, 16, 32):
                engine.set_option("dense", dense)
                engine.set_option("games_per_warp", gpw)
                st = engine.reset(seeds)
                for lo, depth in zip(range(0, n, 75), (15, 45, 65, 85)):  # late records: some games end during the steps
                    engine.rollout_random(st[lo:lo + 75], depth)
                trace = []
                for _ in range(8):
                    masks = engine.legal_mask(st).cpu().numpy().view(np.uint32)
                    acts = np.array([next(a for a in range(156) if m[a >> 5] >> (a & 31) & 1) for m in masks], dtype=np.uint8)
                    nm = torch.empty((n, 5), dtype=torch.int32, device=dev)
                    trace += [t.cpu().numpy() for t in engine.step(st, torch.from_numpy(acts).to(dev), next_masks=nm)] + [nm.cpu().numpy()]
                outs[dense, gpw] = trace + [st.cpu().numpy()]
    finally:
        for k, v in (("engine", -1), ("dense", -1), ("games_per_warp", 0)):
            engine.set_option(k, v)
    want = outs[0, 8]
    assert any(r.any() for r in want[0:-1:4]), "no step gave a reward: the comparison of rewards would be vacuous"
    for key, got in outs.items():
        assert all(np.array_equal(u, v) for u, v in zip(got, want)), key


def test_evolutionary_stormbound(engine):
    """EvolutionaryStormbound mirror (games/evolutionary_stormbound.py:21-232): exploit-phase decks are the archetypes, the
    game steps like Game on the same stream key, reset() re-deals, there is no `.env` (Q17)."""
    from monsoon_b200.games import EvolutionaryStormbound, Game
    from monsoon_b200.engine import DEFAULT_DECKS, DEFAULT_FACTIONS
    g = EvolutionaryStormbound(seed=11, generation=0, engine=engine)
    assert not hasattr(g, "env")
    assert g.player1_deck == list(DEFAULT_DECKS[0]) and g.player2_deck == list(DEFAULT_DECKS[1])
    # utils.py:152-153: the faction is the one of the archetype's first card (UA07 is NEUTRAL), not DEFAULT_FACTIONS
    ref = Game(seed=11, decks=DEFAULT_DECKS, factions=(g.deck_config.player1_faction, g.deck_config.player2_faction), engine=engine)
    rs = np.random.RandomState(0)
    for _ in range(40):
        la = g.legal_actions()
        assert la == ref.legal_actions() and g.to_play() == ref.to_play()
        a = int(la[rs.randint(len(la))])
        obs, reward, done = g.step(a)
        obs2, reward2, done2 = ref.step(a)
        assert np.array_equal(obs, obs2) and reward * 10 == reward2 and done == done2  # Game.step multiplies by 10 (:140)
        if g.have_winner():
            break
    first = g.state.clone()
    g.reset()
    assert not torch.equal(first, g.state) and g.to_play() == 0
    g.set_generation(45)  # explore phase of the default schedule: part of each deck is random
    g.reset()
    assert g.get_phase_info()["phase"] == "Explore" and len(g.player1_deck) == 12
    assert isinstance(g.expert_agent(), int) and g.action_to_string(155) == "Pass the turn"


@pytest.mark.gpu
def test_device_schedule_matches_host_pairings(engine):
    """sb_eval_schedule == the reference-shaped pairing lists (evo/fitness.py:52-59) + the scalar seed hash, for every mode and any shard"""
    import sys, os
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    from test_host_logic import OracleEngine
    for mode, n_ind, n_total, g in (("round_robin", 5, 5, 3), ("round_robin", 4, 9, 2), ("round_robin", 1, 3, 4), ("versus", 6, 8, 3), ("solo", 7, 7, 5)):
        n_pairs = {"round_robin": n_ind * (n_total - 1), "versus": n_ind * (n_total - n_ind), "solo": n_ind}[mode]
        for lo, n in ((0, n_pairs * g), (3, n_pairs * g - 4)):
            i1, i2, seeds = engine.eval_schedule(mode, n_ind, n_total, g, 123456789, 7, lo, n)
            w1, w2, ws = OracleEngine.host_schedule(mode, n_ind, n_total, g, 123456789, 7, lo, n)
            assert np.array_equal(i1.cpu().numpy(), w1) and np.array_equal(i2.cpu().numpy(), w2) and np.array_equal(seeds.cpu().numpy(), ws), (mode, lo)


@pytest.mark.gpu
def test_eval_population_entry_matches_stepwise_calls(engine):
    """sb_eval_population (one call, chunked, device-side schedule) == schedule + reset + rollout + accumulate issued one by one"""
    rs = np.random.RandomState(11)
    w = torch.from_numpy(rs.uniform(0, 1, (7, 10))).to(engine.device)
    for mode, n_ind in (("round_robin", 7), ("versus", 5), ("solo", 7)):
        n_games = {"round_robin": 7 * 6, "versus": 5 * 2, "solo": 7}[mode] * 3
        counts, aborted = engine.eval_population(mode, n_ind, w, 3, 99, 2, 1, n_games - 2, chunk_games=16)
        i1, i2, seeds = engine.eval_schedule(mode, n_ind, 7, 3, 99, 2, 1, n_games - 3)
        st = engine.reset(seeds)
        res, _ = engine.rollout_heuristic(st, w, None if mode == "solo" else w, i1, None if mode == "solo" else i2)
        want = engine.accumulate_fitness(res, i1, torch.zeros((n_ind, 3), dtype=torch.int32, device=engine.device))
        assert torch.equal(counts, want) and int(counts.sum()) == n_games - 3


def test_bench_dump_outputs_end_to_end(oracle, tmp_path):
    """`bench.py --dump-outputs` on the GPU: states.npy / steps.npy are the final records and env-step counts of the LAST timed
    step (not a warm-up pass), equal to the oracle's rollouts of the same seeds.  Rank 0's pass k (warm-up passes first,
    max(--warmup, 3) of them) plays seeds k * games + i."""
    import json
    import os
    import subprocess
    import sys
    from monsoon_b200.engine import DEFAULT_DECKS, DEFAULT_FACTIONS, deck_indices
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    n, steps, warmup = 256, 2, 3
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--games", str(n), "--steps", str(steps), "--warmup", "0",
                          "--no-saturated", "--no-evo", "--no-cpu-baseline", "--dump-outputs", str(tmp_path / "dump")],
                         capture_output=True, text=True, timeout=600, cwd=root, env=dict(os.environ, RANK="0", WORLD_SIZE="1"))
    assert out.returncode == 0, out.stderr[-2000:]
    d = json.loads([l for l in out.stdout.splitlines() if l.strip()][-1])
    assert d["steps"] == steps and d["warmup"] == warmup
    assert sorted(os.listdir(tmp_path / "dump")) == ["states.npy", "steps.npy"]
    states, counts = np.load(tmp_path / "dump" / "states.npy"), np.load(tmp_path / "dump" / "steps.npy")
    assert states.dtype == np.float32 and states.shape == (n, 512) and counts.dtype == np.float32 and counts.shape == (n,)
    d0, d1 = (deck_indices(x) for x in DEFAULT_DECKS)
    last = warmup + steps - 1
    for i in range(n):
        st = oracle.new_game(last * n + i, d0, d1, *DEFAULT_FACTIONS)
        actions, _dig, _masks = oracle.rollout_random(st, 400)
        assert np.array_equal(states[i], st.astype(np.float32)) and counts[i] == len(actions), i

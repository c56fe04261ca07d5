"""The fitness evaluation on the device against the oracle's own games.

The evaluation's output is, per individual, {wins, draws, losses} of the games it played as FIRST, and the aborted games split by
cause.  The scoring rule (evo/fitness.py:208-210): result 0 is a win, 1 a loss, -1 (a draw or a timeout) and -2 (an aborted game)
are draws.  An aborted game counts in aborted[0] when the reference raises too (state.err 1..4) and in aborted[1] when a limit of
this engine stopped it (state.err 5..7, SB_ERR_UNSUPPORTED and up).

  * sb_accumulate_fitness and sb_count_aborted against numpy, at batch sizes around the 256-thread CTA and far beyond it;
  * sb_eval_population for the three schedules against the oracle playing the same games, over a deck pair whose games end in
    every way (wins, losses, draws, timeouts, and both causes of abort), for any shard, chunk size and step cap;
  * FitnessEvaluator end to end on both device paths (sb_eval_population, and the step-by-step path that a deck schedule takes),
    with its aborted-game counters and its capacity warning.
The last test runs without a GPU: it pins that the fixture decks, seeds and weights still produce every outcome, so that a change
of the oracle or of the decks fails loudly instead of leaving the GPU tests vacuous."""
import functools
import os
import sys
import warnings

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from test_host_logic import OracleEngine  # noqa: E402

SB_ERR_UNSUPPORTED = 5  # include/sb_state.h: err codes from here on are limits of this engine
RESULTS = (-2, -1, 0, 1)

# One deck pair for every game of an evaluation (sb_eval_population shares it).  Random legal decks of factions 1 and 2 with the
# neutral UA20 in both: its copies grow hands and decks beyond the packed layout, so some games stop at an engine limit (err 5 / 6),
# others at an exception the reference raises too (err 1..4).  The first card of each deck carries the deck's faction, so a
# DeckEvolutionConfig with these archetypes deals exactly this pair in its exploit phase (utils.py:152-153).
DECKS = (["UT12", "UA20", "U017", "U026", "UE03", "U117", "U021", "S021", "UE04", "S003", "U020", "S007"],
         ["B203", "U026", "U027", "B007", "U030", "U002", "B008", "UT01", "UE03", "U019", "U212", "UA20"])
FACTIONS = (1, 2)
BASE_SEED, GENERATION = 2024, 3
SCHEDULES = {  # mode: (n_ind, n_total, games_per_pair); rows n_ind.. of the round robin are hall-of-fame opponents
    "round_robin": (6, 9, 8),
    "versus": (6, 9, 16),
    "solo": (8, 8, 30),
}
STEP_CAP = 120  # short enough that a third of the games time out, long enough that all other outcomes still occur


class Cfg:
    games_per_pairing = 4
    max_turns = 400
    seed = 11
    num_workers = 1


def weight_table(n_total):
    return np.random.RandomState(1).uniform(0, 1, (9, 10))[:n_total]


def n_games(mode):
    n_ind, n_total, g = SCHEDULES[mode]
    return {"round_robin": n_ind * (n_total - 1), "versus": n_ind * (n_total - n_ind), "solo": n_ind}[mode] * g


def deck_ids():
    from monsoon_b200.engine import deck_indices
    return [deck_indices(d) for d in DECKS]


def play(oracle, i1, i2, seeds, weights, decks, factions, max_steps, expert_second):
    """the oracle's games: (result, final err byte, env steps) of each"""
    out = np.zeros((len(seeds), 3), dtype=np.int64)
    for t, (a, b, s) in enumerate(zip(i1.tolist(), i2.tolist(), seeds.tolist())):
        st = oracle.new_game(s, decks[0], decks[1], factions[0], factions[1])
        r, acts = oracle.play_heuristic(st, weights[a], None if expert_second else weights[b], max_steps)
        out[t] = r, st[18], len(acts)
    return out


@functools.lru_cache(maxsize=None)
def schedule_games(oracle, mode, max_steps=400):
    """(FIRST row, result, err, steps) of every game of SCHEDULES[mode] over DECKS, in game-index order"""
    n_ind, n_total, g = SCHEDULES[mode]
    i1, i2, seeds = OracleEngine.host_schedule(mode, n_ind, n_total, g, BASE_SEED, GENERATION, 0, n_games(mode))
    games = play(oracle, i1, i2, seeds, weight_table(n_total), deck_ids(), FACTIONS, max_steps, mode == "solo")
    return i1, games[:, 0], games[:, 1], games[:, 2]


def tally(i1, res, err, n_ind, lo=0, hi=None):
    """counts i64[n_ind, 3] and aborted i64[2] of the games [lo, hi), by the scoring rule of the module docstring"""
    i1, res, err = i1[lo:hi], res[lo:hi], err[lo:hi]
    counts = np.zeros((n_ind, 3), dtype=np.int64)
    np.add.at(counts, (i1, np.where(res == 0, 0, np.where(res == 1, 2, 1))), 1)
    ab = res == -2
    return counts, np.array([np.sum(ab & (err < SB_ERR_UNSUPPORTED)), np.sum(ab & (err >= SB_ERR_UNSUPPORTED))], dtype=np.int64)


def assert_every_outcome(counts, aborted, what):
    """non-vacuity: the reference side has wins, draws, losses and both causes of abort"""
    tot = counts.sum(axis=0)
    assert tot[0] > 0 and tot[1] > 0 and tot[2] > 0 and aborted[0] > 0 and aborted[1] > 0, (what, tot, aborted)


def fixture_tensors(engine):
    return (torch.tensor(deck_ids(), dtype=torch.uint8, device=engine.device),
            torch.tensor(FACTIONS, dtype=torch.uint8, device=engine.device))


def eval_population(engine, mode, lo, hi, counts=None, aborted=None, chunk_games=0, max_steps=400):
    n_ind, n_total, g = SCHEDULES[mode]
    w = torch.from_numpy(weight_table(n_total)).to(engine.device)
    decks, factions = fixture_tensors(engine)
    counts, aborted = engine.eval_population(mode, n_ind, w, g, BASE_SEED, GENERATION, lo, hi, max_steps=max_steps, counts=counts,
                                             aborted=aborted, chunk_games=chunk_games, decks=decks, factions=factions)
    return counts.cpu().numpy().astype(np.int64), aborted.cpu().numpy().astype(np.int64)


# ---------------------------------------------------------------- a. the two reductions against numpy
BATCHES = (1, 255, 256, 257, 100_003, 1 << 20)


@pytest.mark.gpu
@pytest.mark.parametrize("n", BATCHES)
@pytest.mark.parametrize("rows", [1, 4096, None], ids=["P1", "P4096", "row_g"])
def test_accumulate_fitness_matches_numpy(engine, n, rows):
    """counts[idx_first[g]] += one of {win, draw, loss} per game, added to what the table held; idx_first = None is row g.
    P = 1 sends every game's atomic to one of three counters."""
    rs = np.random.RandomState(n % 9973 + (rows or 7))
    result = rs.choice(np.array(RESULTS, dtype=np.int8), n)
    result[:min(n, 4)] = RESULTS[:min(n, 4)]
    p = n if rows is None else rows
    idx = np.arange(n, dtype=np.int32) if rows is None else rs.randint(0, rows, n).astype(np.int32)
    start = rs.randint(1, 1000, (p, 3)).astype(np.int32)
    want = start.astype(np.int64)
    np.add.at(want, (idx, np.where(result == 0, 0, np.where(result == 1, 2, 1))), 1)
    dev = engine.device
    counts = torch.from_numpy(start).to(dev)
    engine.accumulate_fitness(torch.from_numpy(result).to(dev), None if rows is None else torch.from_numpy(idx).to(dev), counts)
    assert np.array_equal(counts.cpu().numpy(), want)


@pytest.mark.gpu
@pytest.mark.parametrize("n", BATCHES)
def test_count_aborted_matches_numpy(engine, n):
    """out += {aborted games with err below SB_ERR_UNSUPPORTED, aborted games with err SB_ERR_UNSUPPORTED and up}, read from
    byte 18 of each record; a game whose result is not -2 never counts, whatever its err byte holds."""
    rs = np.random.RandomState(n % 9973)
    err = rs.randint(0, 8, n).astype(np.uint8)
    result = rs.choice(np.array(RESULTS, dtype=np.int8), n)
    k = min(n, 32)  # every (err, result) pair once, when the batch is large enough
    err[:k], result[:k] = np.arange(32)[:k] % 8, np.array(RESULTS, dtype=np.int8).repeat(8)[:k]
    dev = engine.device
    gen = torch.Generator(device=dev).manual_seed(n)
    states = torch.randint(0, 256, (n, 512), dtype=torch.uint8, device=dev, generator=gen)  # neighbouring bytes hold noise
    states[:, 18] = torch.from_numpy(err).to(dev)
    out = torch.tensor([123456, 7890], dtype=torch.int32, device=dev)
    engine.count_aborted(states, torch.from_numpy(result).to(dev), out)
    ab = result == -2
    want = [123456 + np.sum(ab & (err < SB_ERR_UNSUPPORTED)), 7890 + np.sum(ab & (err >= SB_ERR_UNSUPPORTED))]
    assert out.cpu().tolist() == want, (n, want)


@pytest.mark.gpu
def test_empty_reductions_launch_nothing(engine):
    dev = engine.device
    counts = torch.full((SCHEDULES["versus"][0], 3), 5, dtype=torch.int32, device=dev)
    out = torch.full((2,), 9, dtype=torch.int32, device=dev)
    before = engine.launches
    engine.accumulate_fitness(torch.empty(0, dtype=torch.int8, device=dev), torch.empty(0, dtype=torch.int32, device=dev), counts)
    engine.count_aborted(torch.empty((0, 512), dtype=torch.uint8, device=dev), torch.empty(0, dtype=torch.int8, device=dev), out)
    engine.eval_schedule("round_robin", 3, 4, 2, 1, 0, 5, 0)
    eval_population(engine, "versus", 17, 17, counts=counts, aborted=out)
    assert engine.launches == before
    assert counts.eq(5).all() and out.eq(9).all()


# ---------------------------------------------------------------- b. sb_eval_population against the oracle
@pytest.mark.gpu
@pytest.mark.parametrize("mode", list(SCHEDULES))
def test_eval_population_matches_oracle(engine, oracle, mode):
    """The whole schedule in one call == the oracle's games counted by hand; a second call adds the same again."""
    i1, res, err, _ = schedule_games(oracle, mode)
    want_c, want_a = tally(i1, res, err, SCHEDULES[mode][0])
    assert_every_outcome(want_c, want_a, mode)
    dev = engine.device
    counts = torch.zeros((SCHEDULES[mode][0], 3), dtype=torch.int32, device=dev)
    aborted = torch.zeros(2, dtype=torch.int32, device=dev)
    got_c, got_a = eval_population(engine, mode, 0, n_games(mode), counts=counts, aborted=aborted)
    assert np.array_equal(got_c, want_c) and np.array_equal(got_a, want_a), (mode, got_c, want_c, got_a, want_a)
    got_c, got_a = eval_population(engine, mode, 0, n_games(mode), counts=counts, aborted=aborted)
    assert np.array_equal(got_c, 2 * want_c) and np.array_equal(got_a, 2 * want_a), mode


@pytest.mark.gpu
@pytest.mark.parametrize("mode", list(SCHEDULES))
def test_eval_population_chunks_and_shards(engine, oracle, mode):
    """Any chunk size gives the single-call counts; shards [lo, hi) give the counts of their own games, also when they cut a
    pairing in the middle, and the shards of world sizes 1, 2, 3 and 8 sum to the whole."""
    from monsoon_b200.evo import FitnessEvaluator
    n_ind, _n_total, g = SCHEDULES[mode]
    i1, res, err, _ = schedule_games(oracle, mode)
    n = n_games(mode)
    want_c, want_a = tally(i1, res, err, n_ind)
    for chunk in (1, 7, 16, n, n + 5):
        got_c, got_a = eval_population(engine, mode, 0, n, chunk_games=chunk)
        assert np.array_equal(got_c, want_c) and np.array_equal(got_a, want_a), (mode, chunk)
    lo, hi = g // 2 + 1, n - g // 2 - 1
    assert lo % g and hi % g  # both ends inside a pairing
    for chunk in (0, 7):
        got_c, got_a = eval_population(engine, mode, lo, hi, chunk_games=chunk)
        ref_c, ref_a = tally(i1, res, err, n_ind, lo, hi)
        assert np.array_equal(got_c, ref_c) and np.array_equal(got_a, ref_a), (mode, lo, hi, chunk)
    for world in (1, 2, 3, 8):
        sum_c, sum_a = np.zeros_like(want_c), np.zeros_like(want_a)
        for rank in range(world):
            lo, hi = FitnessEvaluator.shard(n, rank, world)
            got_c, got_a = eval_population(engine, mode, lo, hi, chunk_games=16)
            ref_c, ref_a = tally(i1, res, err, n_ind, lo, hi)
            assert np.array_equal(got_c, ref_c) and np.array_equal(got_a, ref_a), (mode, world, rank)
            sum_c, sum_a = sum_c + got_c, sum_a + got_a
        assert np.array_equal(sum_c, want_c) and np.array_equal(sum_a, want_a), (mode, world)


@pytest.mark.gpu
def test_eval_population_step_cap_and_no_aborted_buffer(engine, oracle):
    """A step cap that many games reach: the timeouts are draws.  aborted_d = NULL (the C ABI allows it) leaves the counts as
    they are with the buffer."""
    mode = "round_robin"
    n_ind, n_total, g = SCHEDULES[mode]
    n = n_games(mode)
    i1, res, err, steps = schedule_games(oracle, mode, STEP_CAP)
    want_c, want_a = tally(i1, res, err, n_ind)
    assert_every_outcome(want_c, want_a, "step cap")
    assert np.sum((res == -1) & (steps == STEP_CAP)) > n // 4  # timeouts, not only drawn games
    got_c, got_a = eval_population(engine, mode, 0, n, chunk_games=50, max_steps=STEP_CAP)
    assert np.array_equal(got_c, want_c) and np.array_equal(got_a, want_a)
    counts = torch.zeros((n_ind, 3), dtype=torch.int32, device=engine.device)
    w = torch.from_numpy(weight_table(n_total)).to(engine.device)
    decks, factions = fixture_tensors(engine)
    P = engine._p
    rc = engine.lib.sb_eval_population(engine.h, engine.SCHEDULES[mode], n_ind, n_total, g, BASE_SEED, GENERATION, 0, n, P(w), P(decks),
                                       decks.shape[1], P(factions), STEP_CAP, 50, P(counts), None, engine._stream())
    assert rc == 0
    assert np.array_equal(counts.cpu().numpy(), want_c)


BAD_SCHEDULES = (  # (mode, n_ind, n_total, games_per_pair): one per condition sb_eval_schedule rejects
    (-1, 2, 4, 2),   # mode below 0
    (3, 2, 4, 2),    # mode above 2
    (0, 0, 4, 2),    # no individual
    (2, -1, 4, 2),
    (0, 2, 4, 0),    # no game per pairing
    (1, 2, 4, -3),
    (2, 5, 4, 2),    # fewer rows than individuals
    (0, 1, 1, 2),    # a round robin of one row
    (1, 3, 3, 2),    # versus without an opponent row
)


@pytest.mark.gpu
@pytest.mark.parametrize("bad", BAD_SCHEDULES, ids=lambda b: "m%d_i%d_t%d_g%d" % b)
def test_bad_schedule_is_rejected(engine, bad):
    """-1, the reason in sb_last_error, nothing launched and nothing written: through sb_eval_schedule and sb_eval_population."""
    mode, n_ind, n_total, g = bad
    dev, P = engine.device, engine._p
    i1 = torch.full((8,), -7, dtype=torch.int32, device=dev)
    i2 = torch.full((8,), -7, dtype=torch.int32, device=dev)
    seeds = torch.full((8,), -7, dtype=torch.int64, device=dev)
    counts = torch.full((8, 3), 11, dtype=torch.int32, device=dev)
    aborted = torch.full((2,), 13, dtype=torch.int32, device=dev)
    w = torch.zeros((8, 10), dtype=torch.float64, device=dev)
    decks, factions = fixture_tensors(engine)
    reason = "(mode %d, %d individuals, %d rows, %d games per pairing)" % bad
    before = engine.launches
    rc = engine.lib.sb_eval_schedule(engine.h, mode, n_ind, n_total, g, 1, 0, 0, 8, P(i1), P(i2), P(seeds), engine._stream())
    msg = engine.lib.sb_last_error(engine.h).decode()
    assert rc < 0 and "sb_eval_schedule" in msg and reason in msg, (rc, msg)
    rc = engine.lib.sb_eval_population(engine.h, mode, n_ind, n_total, g, 1, 0, 0, 8, P(w), P(decks), decks.shape[1], P(factions), 400,
                                       0, P(counts), P(aborted), engine._stream())
    msg = engine.lib.sb_last_error(engine.h).decode()
    assert rc < 0 and reason in msg, (rc, msg)
    assert engine.launches == before
    torch.cuda.synchronize(dev)
    assert i1.eq(-7).all() and i2.eq(-7).all() and seeds.eq(-7).all() and counts.eq(11).all() and aborted.eq(13).all()


# ---------------------------------------------------------------- c. FitnessEvaluator end to end
def evaluator_calls(oracle, decks, factions):
    """What FitnessEvaluator must return for the sequence of calls in test_fitness_evaluator_matches_oracle_games, from the oracle:
    [(call, generation, fitness, counts, aborted, n_games)].  The round robin of generation 1 also plays the hall of fame of
    generation 0 (the top five by fitness, evo/fitness.py:247-259)."""
    from monsoon_b200.evo import WeightVector
    rs = np.random.RandomState(21)
    pop, opp = rs.uniform(0, 1, (4, 10)), rs.uniform(0, 1, (2, 10))
    g, out = Cfg.games_per_pairing, []

    def run(call, generation, mode, table, n_ind, g, per):
        n = {"round_robin": n_ind * (len(table) - 1), "versus": n_ind * (len(table) - n_ind), "solo": n_ind}[mode] * g
        i1, i2, seeds = OracleEngine.host_schedule(mode, n_ind, len(table), g, Cfg.seed, generation, 0, n)
        games = play(oracle, i1, i2, seeds, table, decks, factions, Cfg.max_turns, mode == "solo")
        counts, aborted = tally(i1, games[:, 0], games[:, 1], n_ind)
        fitness = (counts[:, 0] + 0.5 * counts[:, 1]) / per
        out.append((call, generation, fitness, counts, aborted, n))
        return fitness

    fit0 = run("evaluate_population", 0, "round_robin", pop, 4, g, 3 * g)
    hof = pop[[i for _f, i in sorted(zip(fit0, range(4)), key=lambda x: x[0], reverse=True)[:5]]]
    run("evaluate_population", 1, "round_robin", np.concatenate([pop, hof]), 4, g, 7 * g)
    run("evaluate_vs", 2, "versus", np.concatenate([pop, opp]), 4, 3, 2 * 3)
    run("evaluate_vs_expert", 3, "solo", pop, 4, 5, 5)
    vectors = []
    for row in list(pop) + list(opp):
        v = WeightVector(10)
        v.weights = row.copy()
        vectors.append(v)
    return out, vectors[:4], vectors[4:]


def deck_schedule():
    """a DeckEvolutionConfig that stays in its exploit phase, where every game is dealt the archetypes: DECKS"""
    from monsoon_b200.evo import DeckEvolutionConfig
    return DeckEvolutionConfig(DECKS[0], DECKS[1], exploit_generations=1000, explore_generations=10)


@pytest.mark.gpu
@pytest.mark.parametrize("path", ["eval_population", "stepwise"])
def test_fitness_evaluator_matches_oracle_games(engine, oracle, path):
    """evaluate_population (with and without hall-of-fame rows), evaluate_vs and evaluate_vs_expert == the oracle's games scored by
    hand, aborted games as draws: fitness, counts, last_aborted and get_aborted(); the capacity warning fires exactly for the
    calls in which more than 1 % of the games stopped at an engine limit.  "eval_population": no deck schedule, one
    sb_eval_population call over the default decks.  "stepwise": a deck schedule dealing DECKS, so the evaluator takes the
    schedule / generate_decks / reset / rollout / accumulate / count calls one chunk of 7 games at a time."""
    from monsoon_b200.engine import DEFAULT_DECKS, DEFAULT_FACTIONS, deck_indices
    from monsoon_b200.evo import FitnessEvaluator
    if path == "stepwise":
        calls, pop, opp = evaluator_calls(oracle, deck_ids(), FACTIONS)
        ev = FitnessEvaluator(Cfg(), deck_config=deck_schedule(), engine=engine, chunk_games=7)
    else:
        calls, pop, opp = evaluator_calls(oracle, [deck_indices(d) for d in DEFAULT_DECKS], DEFAULT_FACTIONS)
        ev = FitnessEvaluator(Cfg(), engine=engine)
    total = np.zeros(2, dtype=np.int64)
    for call, generation, fitness, counts, aborted, n in calls:
        with warnings.catch_warnings(record=True) as caught:
            warnings.simplefilter("always")
            if call == "evaluate_population":
                got = ev.evaluate_population(pop, generation)
            elif call == "evaluate_vs":
                got = ev.evaluate_vs(pop, opp, generation, games_per_opponent=3)
            else:
                got = ev.evaluate_vs_expert(pop, generation, games=5)
        what = (path, call, generation)
        assert np.array_equal(ev.last_counts, counts), (what, ev.last_counts, counts)
        assert np.allclose(got, fitness, rtol=0, atol=1e-12), (what, got, fitness)
        assert ev.last_aborted == tuple(aborted.tolist()), (what, ev.last_aborted, aborted)
        capacity = [w for w in caught if "capacity limit" in str(w.message)]
        assert len(capacity) == (1 if aborted[1] * 100 > n else 0), (what, aborted, n, [str(w.message) for w in caught])
        total += aborted
    assert ev.get_aborted() == {"aborted_like_reference": int(total[0]), "aborted_by_engine_limit": int(total[1])}
    if path == "stepwise":
        assert_every_outcome(sum(c[3] for c in calls), total, "evaluator, stepwise")


WARNING_CASES = {7: (1, 100), 11: (2, 100)}  # generation: (games stopped at an engine limit, games) of warning_case


def warning_case():
    """5 individuals x 20 games against the expert seat: 100 games, so 1 % of them is exactly one game"""
    from monsoon_b200.evo import WeightVector
    vectors = []
    for row in np.random.RandomState(0).uniform(0, 1, (5, 10)):
        v = WeightVector(10)
        v.weights = row
        vectors.append(v)
    return vectors, 20


@pytest.mark.gpu
@pytest.mark.parametrize("generation", sorted(WARNING_CASES))
def test_capacity_warning_at_one_percent(engine, generation):
    """One game in 100 stopped at an engine limit is not above the 1 % line (no warning); two are (one warning)."""
    from monsoon_b200.evo import FitnessEvaluator
    pop, games = warning_case()
    limit, n = WARNING_CASES[generation]
    ev = FitnessEvaluator(Cfg(), deck_config=deck_schedule(), engine=engine)
    with warnings.catch_warnings(record=True) as caught:
        warnings.simplefilter("always")
        ev.evaluate_vs_expert(pop, generation, games=games)
    assert ev.last_aborted[1] == limit and len(pop) * games == n
    capacity = [w for w in caught if "capacity limit" in str(w.message)]
    assert len(capacity) == (1 if limit * 100 > n else 0), [str(w.message) for w in caught]


# ---------------------------------------------------------------- d. the fixture itself (CPU)
def test_fixture_decks_play_every_outcome(oracle):
    """The oracle alone: the fixture decks, seeds and weights give every outcome and both causes of abort in every schedule, at the
    step cap, and in the evaluator's stepwise calls; the deck schedule deals exactly DECKS; the warning cases hold 1 and 2
    engine-limit aborts in 100 games."""
    from monsoon_b200._card_table import CARDS
    from monsoon_b200.evo import game_seed
    for mode in SCHEDULES:
        i1, res, err, _ = schedule_games(oracle, mode)
        assert_every_outcome(*tally(i1, res, err, SCHEDULES[mode][0]), mode)
        assert set(err[res == -2].tolist()) <= set(range(1, 8)) and not err[res != -2].any(), mode
    i1, res, err, steps = schedule_games(oracle, "round_robin", STEP_CAP)
    assert_every_outcome(*tally(i1, res, err, SCHEDULES["round_robin"][0]), "step cap")
    assert np.sum((res == -1) & (steps == STEP_CAP)) > n_games("round_robin") // 4
    calls, _pop, _opp = evaluator_calls(oracle, deck_ids(), FACTIONS)
    assert_every_outcome(sum(c[3] for c in calls), sum(c[4] for c in calls), "evaluator, stepwise")
    cfg = deck_schedule()
    assert (cfg.player1_faction, cfg.player2_faction) == FACTIONS == tuple(int(CARDS[d[0]]["faction"]) for d in deck_ids())
    mode, keep, q = cfg.phase_parameters(11)
    for seed in (0, 1, 2 ** 40 + 3):
        got = oracle.generate_decks(seed, 11, mode, keep, q, [cfg.player1_archetype, cfg.player2_archetype], FACTIONS)
        assert got.tolist() == deck_ids()
    pop, games = warning_case()
    for generation, (limit, n) in WARNING_CASES.items():
        ab = np.zeros(2, dtype=np.int64)
        for i, v in enumerate(pop):
            for k in range(games):
                st = oracle.new_game(game_seed(Cfg.seed, generation, i, i, k), *deck_ids(), *FACTIONS)
                r, _ = oracle.play_heuristic(st, v.weights, None, Cfg.max_turns)
                ab[int(st[18]) >= SB_ERR_UNSUPPORTED] += r == -2
        assert ab[1] == limit and len(pop) * games == n, (generation, ab)

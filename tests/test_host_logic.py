"""CPU: host-side logic of the drop-in layer (no kernels): pairing schedule, sharding, seeds, the
reference-faithful evaluator, hall of fame, and the N>1 reduction path over gloo (world_size 2)."""
import json
import os
import socket
import subprocess
import sys

import numpy as np
import pytest


class Cfg:
    games_per_pairing = 3
    max_turns = 60
    seed = 7
    num_workers = 4


def test_pairings_match_reference_schedule():
    from monsoon_b200.evo import FitnessEvaluator
    p = FitnessEvaluator.pairings(3, 5)  # 3 individuals + 2 hall-of-fame opponents
    assert p == [(0, 1), (0, 2), (0, 3), (0, 4), (1, 0), (1, 2), (1, 3), (1, 4), (2, 0), (2, 1), (2, 3), (2, 4)]


def test_shard_is_a_partition():
    from monsoon_b200.evo import FitnessEvaluator
    for n in (0, 1, 7, 65536, 1000003):
        for world in (1, 2, 3, 8):
            blocks = [FitnessEvaluator.shard(n, r, world) for r in range(world)]
            assert blocks[0][0] == 0 and blocks[-1][1] == n
            assert all(blocks[i][1] == blocks[i + 1][0] for i in range(world - 1))
            sizes = [b - a for a, b in blocks]
            assert max(sizes) - min(sizes) <= 1


def test_game_seed_is_deterministic_and_spread():
    from monsoon_b200.evo import game_seed
    s = {game_seed(7, g, i, j, k) for g in range(3) for i in range(8) for j in range(8) for k in range(4)}
    assert len(s) == 3 * 8 * 8 * 4
    assert game_seed(7, 1, 2, 3, 4) == game_seed(7, 1, 2, 3, 4) and all(0 <= x < 2 ** 63 for x in s)


def test_mask_to_actions_sorted():
    from monsoon_b200.games import mask_to_actions
    m = np.zeros(5, dtype=np.uint32)
    for a in (0, 31, 32, 64, 148, 155):
        m[a >> 5] |= np.uint32(1 << (a & 31))
    assert mask_to_actions(m) == [0, 31, 32, 64, 148, 155]


def test_reference_faithful_evaluator_reproduces_degenerate_fitness():
    """SURVEY fact 7: the reference's evaluate_population returns 1.0 for everybody (no game is stepped)."""
    from monsoon_b200.evo import FitnessEvaluator, WeightVector
    np.random.seed(0)
    pop = [WeightVector(10) for _ in range(4)]
    ev = FitnessEvaluator(Cfg(), reference_faithful=True)
    assert ev.evaluate_population(pop, 0) == [1.0] * 4
    assert len(ev.hall_of_fame) == 4  # top-5 copies of a population of 4
    assert ev.evaluate_population(pop, 1) == [1.0] * 4  # now with hall-of-fame opponents: still (n_total-1)*g / ((n_total-1)*g)
    st = ev.get_stats()
    assert st["total_games"] == (4 * 3 + 4 * 7) * 3 and set(st) == {"total_games", "total_time", "avg_time_per_game", "games_per_second"}
    assert ev.hall_of_fame[0] is not pop[0] and np.array_equal(ev.hall_of_fame[0].weights, pop[0].weights)


class OracleEngine:
    """Test double with the Engine surface FitnessEvaluator._play uses, computing on the CPU with the oracle.
    Lets the sharding + collective logic run under gloo without a GPU."""

    def __init__(self):
        import torch
        import sb_oracle
        self.o, self.device = sb_oracle, torch.device("cpu")
        from monsoon_b200.engine import DEFAULT_DECKS, deck_indices
        self.d = [deck_indices(x) for x in DEFAULT_DECKS]

    def reset(self, seeds, decks=None, factions=None):
        import torch
        if decks is None:
            return torch.from_numpy(np.stack([self.o.new_game(int(s), self.d[0], self.d[1], 3, 2) for s in seeds.tolist()]))
        d, f = decks.numpy(), factions.numpy()
        return torch.from_numpy(np.stack([self.o.new_game(int(s), d[i][0], d[i][1], int(f[i][0]), int(f[i][1]))
                                          for i, s in enumerate(seeds.tolist())]))

    def generate_decks(self, seeds, generation, mode, n_preserve=0, q=0.0, archetypes=None, arch_factions=None, factions=None):
        import torch
        d = np.stack([self.o.generate_decks(int(s), generation, mode, n_preserve, q, archetypes, arch_factions) for s in seeds.tolist()])
        return torch.from_numpy(d), torch.from_numpy(np.tile(np.asarray(arch_factions, dtype=np.uint8), (len(d), 1)))

    def rollout_heuristic(self, states, w_first, w_second, idx_first, idx_second, max_steps=400):
        import torch
        st = states.numpy()
        _tot, res, steps = self.o.batch_heuristic(st, w_first.numpy(), w_second.numpy(), idx_first.numpy(), idx_second.numpy(),
                                                  max_steps, 2)
        return torch.from_numpy(res.astype(np.int8)), torch.from_numpy(steps)

    def accumulate_fitness(self, result, idx_first, counts):
        for r, i in zip(result.tolist(), idx_first.tolist()):
            counts[i, 0 if r == 0 else 2 if r == 1 else 1] += 1
        return counts

    def count_aborted(self, states, result, out):
        for r, st in zip(result.tolist(), states.numpy()):
            if r == -2:
                out[1 if st[18] >= 5 else 0] += 1
        return out

    @staticmethod
    def host_schedule(mode, n_ind, n_total, g, base_seed, generation, lo, n):
        """what sb_eval_schedule computes, from the reference-shaped pairing LISTS and the scalar seed hash"""
        from monsoon_b200.evo import FitnessEvaluator, game_seed
        pairs = {"round_robin": FitnessEvaluator.pairings(n_ind, n_total), "versus": [(i, n_ind + b) for i in range(n_ind) for b in range(n_total - n_ind)],
                 "solo": [(i, i) for i in range(n_ind)]}[mode]
        rows = [(pairs[gi // g][0], pairs[gi // g][1], game_seed(base_seed, generation, pairs[gi // g][0], pairs[gi // g][1], gi % g)) for gi in range(lo, lo + n)]
        return (np.array([r[0] for r in rows], dtype=np.int32), np.array([r[1] for r in rows], dtype=np.int32), np.array([r[2] for r in rows], dtype=np.int64))

    def eval_schedule(self, mode, n_ind, n_total, g, base_seed, generation, lo, n):
        import torch
        return tuple(torch.from_numpy(a) for a in self.host_schedule(mode, n_ind, n_total, g, base_seed, generation, lo, n))

    def eval_population(self, mode, n_ind, weights, g, base_seed, generation, lo, hi, max_steps=400, counts=None, aborted=None, chunk_games=0):
        chunk = chunk_games or 262144
        for c0 in range(lo, hi, chunk):
            i1, i2, seeds = self.eval_schedule(mode, n_ind, weights.shape[0], g, base_seed, generation, c0, min(hi, c0 + chunk) - c0)
            states = self.reset(seeds)
            res, _ = self.rollout_heuristic(states, weights, weights, i1, i2, max_steps)
            self.accumulate_fitness(res, i1, counts)
            self.count_aborted(states, res, aborted)
        return counts, aborted


def _deck_schedule():
    from monsoon_b200.evo import DeckEvolutionConfig
    from monsoon_b200.engine import DEFAULT_DECKS
    return DeckEvolutionConfig(DEFAULT_DECKS[0], DEFAULT_DECKS[1], exploit_generations=0, explore_generations=2, max_random_ratio=1.0,
                               balance_archetype_ratio=0.5)


def _rank_main(rank, world, port, q):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    sys.path[:0] = [os.path.dirname(os.path.dirname(os.path.abspath(__file__))), os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle")]
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from monsoon_b200.evo import FitnessEvaluator, WeightVector
    np.random.seed(3)
    pop = [WeightVector(10) for _ in range(3)]
    if rank != 0:  # only rank 0's weights count: the broadcast must overwrite these
        for v in pop:
            v.weights = np.zeros(10)
    ev = FitnessEvaluator(Cfg(), engine=OracleEngine(), chunk_games=5)
    fit = ev.evaluate_population(pop, 0)
    ev2 = FitnessEvaluator(Cfg(), deck_config=_deck_schedule(), engine=OracleEngine(), chunk_games=7)  # per-game decks, balance phase
    fit2 = ev2.evaluate_population(pop, 5)
    # the versus schedule over a RESIDENT weight table (device-side schedule, one collective for counts + aborted counters)
    import torch
    table = torch.from_numpy(np.stack([v.weights for v in pop]))
    ev3 = FitnessEvaluator(Cfg(), engine=OracleEngine(), chunk_games=4)
    fit3 = ev3.evaluate_vs(table, [pop[0]], 2, games_per_opponent=2)
    q.put((rank, fit, ev.last_counts.tolist(), fit2, ev2.last_counts.tolist(), fit3, ev3.last_counts.tolist()))
    dist.destroy_process_group()


def test_two_rank_gloo_matches_single_rank():
    import torch.multiprocessing as mp
    from monsoon_b200.evo import FitnessEvaluator, WeightVector
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle"))
    np.random.seed(3)
    pop = [WeightVector(10) for _ in range(3)]
    single = FitnessEvaluator(Cfg(), engine=OracleEngine(), chunk_games=1000)
    want = single.evaluate_population(pop, 0)
    assert single.last_counts.sum() == 3 * 2 * 3
    single2 = FitnessEvaluator(Cfg(), deck_config=_deck_schedule(), engine=OracleEngine(), chunk_games=1000)
    want2 = single2.evaluate_population(pop, 5)
    single3 = FitnessEvaluator(Cfg(), engine=OracleEngine(), chunk_games=1000)
    want3 = single3.evaluate_vs(pop, [pop[0]], 2, games_per_opponent=2)
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_rank_main, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    got = [q.get(timeout=300) for _ in procs]
    for p in procs:
        p.join(60)
    for _rank, fit, counts, fit2, counts2, fit3, counts3 in got:
        assert fit == want and counts == single.last_counts.tolist()
        assert fit2 == want2 and counts2 == single2.last_counts.tolist()  # decks derive from the game seed: partition-invariant
        assert fit3 == want3 and counts3 == single3.last_counts.tolist()


# ---------------------------------------------------------------- f4: checkpoint / log formats
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def test_reads_reference_checkpoint():
    """A pickle written by the reference's Population.save_population (evo/population.py:281-296)."""
    from monsoon_b200.training import EvolutionaryConfig, load_checkpoint
    from monsoon_b200.evo import WeightVector
    d = load_checkpoint(os.path.join(GOLDEN, "ref_population.pkl"))
    z = np.load(os.path.join(GOLDEN, "es_operators.npz"))
    assert d["generation"] == 5 and len(d["individuals"]) == 12 and isinstance(d["config"], EvolutionaryConfig)
    assert all(isinstance(v, WeightVector) for v in d["individuals"])
    assert np.array_equal(np.array([v.weights for v in d["individuals"]]), z["normal_sur_w"][-1])
    assert np.array_equal(np.array([v.sigmas for v in d["individuals"]]), z["normal_sur_s"][-1])
    assert d["fitness_scores"] == z["normal_sur_f"][-1].tolist() and d["config"].mu == 12 and d["config"].lambda_ == 20


def test_checkpoint_round_trip_and_reference_class_paths(tmp_path):
    import pickletools
    from monsoon_b200.training import EvolutionaryConfig, dump_checkpoint, load_checkpoint
    from monsoon_b200.evo import WeightVector
    np.random.seed(3)
    data = {"generation": 9, "individuals": [WeightVector(10) for _ in range(4)], "fitness_scores": [0.5, 0.25, 0.125, 0.0],
            "config": EvolutionaryConfig(mu=4, lambda_=4, seed=1)}
    path = tmp_path / "ours.pkl"
    dump_checkpoint(data, str(path))
    ops = [(op.name, arg) for op, arg, _pos in pickletools.genops(path.read_bytes())]
    names = {arg for name, arg in ops if name in ("SHORT_BINUNICODE", "BINUNICODE")}
    assert {"evo.weights", "WeightVector", "evo.config", "EvolutionaryConfig"} <= names  # what the reference will import
    assert not any("monsoon_b200" in str(arg) for _n, arg in ops)
    back = load_checkpoint(str(path))
    assert back["generation"] == 9 and back["fitness_scores"] == data["fitness_scores"] and back["config"] == data["config"]
    for a, b in zip(back["individuals"], data["individuals"]):
        assert np.array_equal(a.weights, b.weights) and np.array_equal(a.sigmas, b.sigmas) and a.size == b.size
    assert "evo" not in sys.modules or not hasattr(sys.modules["evo"], "__path__") or sys.modules["evo"].__path__ != []


def test_reference_loads_our_checkpoint(tmp_path):
    """The other direction: the reference's Population.load_population (evo/population.py) is a plain pickle.load of
    evo.weights.WeightVector / evo.config.EvolutionaryConfig objects.  A fresh interpreter, with stand-in `evo` modules in place
    of the reference's and without monsoon_b200, loads our file, and every object carries the attributes, with the types (and
    for arrays the dtype and shape), of the same object in the checkpoint the reference itself wrote (golden/ref_population.pkl)."""
    from monsoon_b200.training import EvolutionaryConfig, dump_checkpoint
    from monsoon_b200.evo import WeightVector
    np.random.seed(4)
    vecs = [WeightVector(10) for _ in range(3)]
    path = tmp_path / "ours.pkl"
    dump_checkpoint({"generation": 2, "individuals": vecs, "fitness_scores": [0.9, 0.8, 0.7], "config": EvolutionaryConfig(mu=3, lambda_=3)}, str(path))
    evo = tmp_path / "standin" / "evo"
    evo.mkdir(parents=True)
    (evo / "__init__.py").write_text("")
    (evo / "weights.py").write_text("class WeightVector:\n    pass\n")
    (evo / "config.py").write_text("class EvolutionaryConfig:\n    pass\n")
    code = ("import sys, json, pickle; sys.path.insert(0, %r)\n"
            "from evo.weights import WeightVector; from evo.config import EvolutionaryConfig\n"
            "def shape(p):\n"
            "    d = pickle.load(open(p, 'rb'))\n"
            "    assert type(d['config']) is EvolutionaryConfig and all(type(v) is WeightVector for v in d['individuals'])\n"
            "    attrs = lambda o: sorted((k, type(v).__name__, str(getattr(v, 'dtype', '')), tuple(getattr(v, 'shape', ())))\n"
            "                             for k, v in vars(o).items())\n"
            "    return {'keys': sorted(d), 'vectors': sorted({tuple(attrs(v)) for v in d['individuals']}), 'config': attrs(d['config'])}\n"
            "ours = pickle.load(open(%r, 'rb'))\n"
            "assert 'monsoon_b200' not in sys.modules\n"
            "print(json.dumps([shape(%r), shape(%r), ours['generation'], ours['config'].mu, ours['individuals'][1].weights.tolist()]))"
            % (str(evo.parent), str(path), str(path), os.path.join(GOLDEN, "ref_population.pkl")))
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, cwd=str(tmp_path))
    assert out.returncode == 0, out.stderr[-2000:]
    ours, ref, generation, mu, weights = json.loads(out.stdout.strip().splitlines()[-1])
    assert ours == ref
    assert generation == 2 and mu == 3 and weights == vecs[1].weights.tolist()


def test_training_log_rows_match_reference_format(tmp_path):
    from monsoon_b200.training import append_generation_log
    z = np.load(os.path.join(GOLDEN, "es_operators.npz"))
    keys = ("generation", "best_fitness", "mean_fitness", "std_fitness", "diversity", "avg_mutation_strength")
    st = dict(zip(keys, z["log_stats"].tolist()))
    st["generation"] = int(st["generation"])
    log = tmp_path / "training_log.csv"
    append_generation_log(str(log), st, {"games_per_second": 1234.56}, 7.891)
    append_generation_log(str(log), dict(st, generation=st["generation"] + 1, best_fitness=0.75), {"games_per_second": 99.0}, 0.004)
    assert log.read_text() == open(os.path.join(GOLDEN, "ref_training_log.csv")).read()


def test_config_mirror_matches_reference_defaults():
    from monsoon_b200.training import EvolutionaryConfig, load_checkpoint
    ref_cfg = load_checkpoint(os.path.join(GOLDEN, "ref_population.pkl"))["config"]
    ours = EvolutionaryConfig(mu=12, lambda_=20, tau=0.1, tau_prime=0.01, min_sigma=1e-5, initial_sigma=0.1)
    assert vars(ref_cfg).keys() == vars(ours).keys()  # the reference's dataclass fields, all of them
    assert vars(ref_cfg) == vars(ours)
    with pytest.raises(ValueError):
        EvolutionaryConfig(mu=0)



def test_bench_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` (the CPU arm: the reference's own Python engine when its staged copy is at hand, else the
    oracle port, on all host cores; the port always printed beside it) runs without a GPU and prints ONE JSON line with the
    keys the driver reads; both legs time exactly --steps steps and report them; ranks other than 0 print nothing."""
    import json
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, RANK="0", WORLD_SIZE="1")
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "5", "--warmup", "1"],
                         capture_output=True, text=True, timeout=600, env=env, cwd=root)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "env_steps_per_sec" and d["unit"] == "env_steps/s"
    assert d["value"] > 0 and d["higher_is_better"] is True and d["steps"] == 5 and d["warmup"] == 1
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["cpu_baseline_port"]["kind"] == "port" and d["cpu_baseline_port"]["value"] > 0
    for leg in (d["cpu_baseline"], d["cpu_baseline_port"]):
        assert leg["timed_steps"] == 5 and leg["seconds"] > 0 and leg["value"] == leg["env_steps"] / leg["seconds"]
    port = d["cpu_baseline_port"]
    assert port["env_steps"] > 5 * 4096  # every timed step plays all 4,096 games to completion
    assert d["ms_per_step"] == 1e3 * d["cpu_baseline"]["seconds"] / 5
    if d["cpu_baseline"]["kind"] == "reference":  # the Python engine is two to three orders of magnitude slower than its C restatement
        assert d["cpu_baseline_port"]["value"] > 50 * d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "env_steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "model" not in d["config"]
    env["RANK"] = "1"
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=600, env=env, cwd=root)
    assert out.returncode == 0 and out.stdout.strip() == ""
    for bad in (["--steps", "0"], ["--steps", "1", "--dump-outputs", "unused"]):  # refused, not silently changed or ignored
        out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference"] + bad,
                             capture_output=True, text=True, timeout=600, env=env, cwd=root)
        assert out.returncode == 2 and out.stdout.strip() == "", bad
    assert not os.path.exists(os.path.join(root, "unused"))


def test_bench_dump_outputs(tmp_path, monkeypatch):
    """`bench.py --dump-outputs`: float32 copies of the arrays, exact for u8 records and int32 counts; above the size limit the
    same seeded rows of every array, with their indices, and the same files from run to run."""
    import torch
    monkeypatch.setattr(sys, "path", list(sys.path))
    monkeypatch.setattr(sys, "dont_write_bytecode", sys.dont_write_bytecode)
    import bench
    states = torch.arange(64 * 32, dtype=torch.int64).remainder(251).to(torch.uint8).view(64, 32)
    steps = torch.arange(64, dtype=torch.int32) * 7
    assert bench.dump_outputs(str(tmp_path / "all"), {"states": states, "steps": steps}) == ["states", "steps"]
    got = np.load(tmp_path / "all" / "states.npy")
    assert got.dtype == np.float32 and np.array_equal(got, states.numpy())
    assert np.array_equal(np.load(tmp_path / "all" / "steps.npy"), steps.numpy())
    assert bench.DUMP_LIMIT == 64_000_000
    monkeypatch.setattr(bench, "DUMP_LIMIT", 8192)
    for d in ("a", "b"):
        assert bench.dump_outputs(str(tmp_path / d), {"states": states, "steps": steps}) == ["rows", "states", "steps"]
    rows = np.load(tmp_path / "a" / "rows.npy").astype(np.int64)
    assert 0 < len(rows) < 64 and np.array_equal(rows, np.unique(rows))
    assert sum(os.path.getsize(tmp_path / "a" / (k + ".npy")) for k in ("rows", "states", "steps")) <= 8192  # the files, headers too
    for k in ("rows", "states", "steps"):
        assert (tmp_path / "a" / (k + ".npy")).read_bytes() == (tmp_path / "b" / (k + ".npy")).read_bytes()
    assert np.array_equal(np.load(tmp_path / "a" / "states.npy"), states.numpy()[rows])
    assert np.array_equal(np.load(tmp_path / "a" / "steps.npy"), steps.numpy()[rows])


def test_evolutionary_stormbound_mirror_surface():
    """games/evolutionary_stormbound.py:21-232: same public members, and -- like the reference (SURVEY Q17) -- no `.env`,
    which is what makes the reference's adapter / evaluator fall into their AttributeError branches with this class.
    `want` is the public callable member list read off the reference class itself (it has no `env` attribute)."""
    from monsoon_b200.games import EvolutionaryStormbound as Mirror
    want = {"to_play", "reset", "set_generation", "get_phase_info", "step", "legal_actions", "get_observation", "have_winner",
            "render", "close", "expert_agent", "action_to_string"}
    have = {n for n in vars(Mirror) if not n.startswith("_") and callable(getattr(Mirror, n))}
    assert want <= have, want - have
    assert "env" not in vars(Mirror) and "env" not in Mirror.__init__.__code__.co_names


def test_resident_weight_tables_give_the_same_evaluation():
    """FitnessEvaluator fed the rows of a resident weight table (what training.Population hands it since round 2) == fed the
    WeightVector list: fitness, counts and hall of fame, for the round robin (with hall-of-fame opponents in the second
    generation), the versus schedule and the expert-seat schedule."""
    import torch
    from monsoon_b200.evo import FitnessEvaluator, WeightVector
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle"))
    np.random.seed(5)
    pop = [WeightVector(10) for _ in range(3)]
    table = torch.from_numpy(np.stack([v.weights for v in pop]))
    a = FitnessEvaluator(Cfg(), engine=OracleEngine(), chunk_games=4)
    b = FitnessEvaluator(Cfg(), engine=OracleEngine(), chunk_games=1000)
    for gen in range(2):  # the second generation plays the hall of fame of the first
        fa, fb = a.evaluate_population(pop, gen), b.evaluate_population(table, gen)
        assert fa == fb and np.array_equal(a.last_counts, b.last_counts)
        assert len(a.hall_of_fame) == len(b.hall_of_fame) == 3
        assert all(np.array_equal(x.weights, y.weights) for x, y in zip(a.hall_of_fame, b.hall_of_fame))
    opp = [WeightVector(10)]
    assert a.evaluate_vs(pop, opp, 3, games_per_opponent=2) == b.evaluate_vs(table, opp, 3, games_per_opponent=2)
    assert np.array_equal(a.last_counts, b.last_counts) and a.last_counts.sum() == 3 * 2


def test_state_bridge_round_trip_and_layout(oracle):
    """monsoon_b200.state (the sb_pack / sb_unpack host bridge of SURVEY 8b): the product's own structured dtype == the oracle-side mirror
    of include/sb_state.h field by field, unpack -> pack is the identity on records of real games, and the dict says what the record says."""
    import sb_layout
    from monsoon_b200 import state as S
    assert S.STATE_DTYPE.itemsize == 512
    for name in S.STATE_DTYPE.names:
        assert S.STATE_DTYPE.fields[name][1] == sb_layout.STATE_DTYPE.fields[name][1], name
    for name in S.PLAYER_DTYPE.names:
        assert S.PLAYER_DTYPE.fields[name][1] == sb_layout.PLAYER_DTYPE.fields[name][1], name
    from test_oracle_golden import default_decks
    d0, d1 = default_decks()
    for seed in range(12):
        st = oracle.new_game(seed, d0, d1, 3, 2)
        for k in range(60):
            d = S.unpack_state(st)
            assert S.pack_state(d).tobytes() == st.tobytes(), (seed, k)
            r = st.view(sb_layout.STATE_DTYPE)[0]
            assert d["players"][0]["strength"] == int(r["pl"][0]["base"]) and d["steps"] == k
            assert sum(e is not None for row in d["board"] for e in row) == int((r["tile"]["card"] != 0).sum())
            m = oracle.legal_mask(st)
            legal = [a for a in range(156) if m[a >> 5] >> (a & 31) & 1]
            oracle.step(st, legal[(seed * 7 + k * 13) % len(legal)])
            if st[19] & 1 or st[18]:
                break
        assert "order 0" in S.render_state(st)

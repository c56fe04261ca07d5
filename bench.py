#!/usr/bin/env python3
"""bench.py -- env-steps/s and games/s of the batched Stormbound hot path on N B200s.

Workload (BASELINE.json configs[1]): 4,096 parallel games per GPU, uniform-random legal agents,
default decks, every game played to completion (max 400 env steps).  One bench "step" = one pass:
sb_reset (new seeds) + sb_rollout_random over the 4,096 games of each rank.  Weak scaling: every rank
plays its own 4,096 games (disjoint seeds), no data-path collective (SURVEY 8e).

  python bench.py --gpus 1 --steps 20 --warmup 3
  python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N --steps K --warmup W
  python bench.py --impl reference ...     # CPU arm: the oracle port on all host threads
  python bench.py ... --dump-outputs DIR   # also write the last timed step's results as DIR/<name>.npy (float32)

JSON keys follow the driver contract; `roofline` and `cpu_baseline` are described in DESIGN.md.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path[:0] = [ROOT]
sys.dont_write_bytecode = True  # the bench leaves the source tree as it found it (it may be read-only)

B_STEP = 2 * 512 + 1 + 20 + 2  # algorithmic bytes per env step (SURVEY 8d): state in+out, action, mask, reward/done
METRIC = "env_steps_per_sec"
WORKLOAD = "4096 parallel games/GPU, uniform-random legal agents, default decks, played to completion (max 400 steps)"
# What ncu measured for ONE launch of the kernels behind the three legs (profiles/r2_summary.md; `--set full`, one capture
# each).  Static facts of the kernels (instructions per env step, lanes per instruction, DRAM bytes per launch): the live
# part of `roofline` is the CUDA-event duration measured in this run.
NCU = {
    # named workload, 4,096 games: kw_rollout_random<32,1,true> (one game per warp, turn-synchronous 32-warp CTAs)
    "rollout_4096": {"kernel": "kw_rollout_random<32,1,true>", "capture": "profiles/r2_w4096_s5_metrics.txt", "dram_bytes": None,
                     "warp_inst_per_env_step": None, "threads_per_inst": None, "issue_active_pct": None},
    # saturated leg, 262,144 games: k_rollout_random<false,1024,true,2> (one game per thread, lane refill, 32-register build)
    "rollout_262144": {"kernel": "k_rollout_random<false,1024,true,2>", "capture": "profiles/r1_rollout_262144_final_metrics.txt",
                       "dram_bytes": 82.7e9, "warp_inst_per_env_step": 8.95e9 / 18.8e6, "threads_per_inst": 4.41, "issue_active_pct": 17.9},
    # evo leg, 65,536 heuristic games: k_rollout_heuristic<8,false> (warp per game, lane per candidate, warp refill)
    "heuristic_65536": {"kernel": "k_rollout_heuristic<8,false>", "capture": "profiles/r1_heur_65536_s2_refill_metrics.txt",
                        "dram_bytes": 1060e9, "warp_inst_per_env_step": None, "threads_per_inst": 11.2, "issue_active_pct": 15.8},
}


def load_ncu_constants():
    """profiles/r2_ncu_constants.json (written by tools/ncu_constants.py from the committed captures) overrides the table above"""
    try:
        with open(os.path.join(ROOT, "profiles", "r2_ncu_constants.json")) as f:
            for k, v in json.load(f).items():
                NCU.setdefault(k, {}).update(v)
    except Exception:  # noqa: BLE001
        pass


def bench_config(n_games_per_gpu=4096):
    """the SAME dict in both arms (the driver compares them); everything else about a run is a top-level key"""
    return {"workload": WORKLOAD, "games_per_gpu": n_games_per_gpu}


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:  # noqa: BLE001
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler(threading.Thread):
    """SM clock / throttle reasons sampled DURING the timed region (NVML every 5 ms; nvidia-smi fallback)."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    BITS = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.sm, self.mx, self.reasons, self.stop_flag, self.how = index, [], [], set(), False, "nvml"

    def prepare(self):
        """NVML handle set up BEFORE the timed region, so that even a few-millisecond region gets its samples."""
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nv = pynvml
            self._h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self._mx = pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM)
        except Exception:  # noqa: BLE001
            self._nv = None

    def sample_once(self):
        """One NVML sample; also called from the main thread right after the launches, while the GPU is busy."""
        if getattr(self, "_nv", None) is None:
            return
        self.sm.append(self._nv.nvmlDeviceGetClockInfo(self._h, self._nv.NVML_CLOCK_SM))
        self.mx.append(self._mx)
        r = self._nv.nvmlDeviceGetCurrentClocksEventReasons(self._h)
        for name, bit in self.BITS.items():
            if r & bit:
                self.reasons.add(name)

    def _nvml(self):
        if getattr(self, "_nv", None) is None:
            raise RuntimeError("nvml unavailable")
        while not self.stop_flag:
            self.sample_once()
            time.sleep(0.005)

    def _smi(self):
        self.how = "nvidia-smi"
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                f = [x.strip() for x in out.split(",")]
                if f and f[0].isdigit():
                    self.sm.append(int(f[0]))
                    self.mx.append(int(f[1]))
                    for i in range(4):
                        if len(f) > 2 + i and f[2 + i].lower().startswith("active"):
                            self.reasons.add(names[i])
            except Exception:  # noqa: BLE001
                pass
            time.sleep(0.05)

    def run(self):
        try:
            self._nvml()
        except Exception:  # noqa: BLE001
            self._smi()

    def summary(self):
        sm = sorted(self.sm)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(self.mx) if self.mx else None,
                "reasons": sorted(self.reasons), "samples": len(sm), "how": self.how}


def issue_roofline(key, env_steps_per_launch, seconds_per_launch, sm_count, sm_mhz):
    """issue-slot roofline of a rollout kernel: warp instructions per second against sm_count x 4 schedulers x clock"""
    c = NCU.get(key, {})
    peak = sm_count * 4 * sm_mhz * 1e6
    out = {"peak_warp_inst_per_s": peak, "threads_per_inst": c.get("threads_per_inst"), "issue_active_pct": c.get("issue_active_pct"),
           "warp_inst_per_env_step": c.get("warp_inst_per_env_step"), "source": c.get("capture")}
    if c.get("warp_inst_per_env_step"):
        out["achieved_warp_inst_per_s"] = c["warp_inst_per_env_step"] * env_steps_per_launch / seconds_per_launch
        out["frac"] = out["achieved_warp_inst_per_s"] / peak
    return out


DUMP_LIMIT = 64_000_000  # bytes of the files written by --dump-outputs in all, .npy headers included
NPY_HEADER_MAX = 1024  # allowance per file for its .npy header (numpy writes 128 bytes for these shapes)


def dump_outputs(out_dir, arrays, seed=0):
    """Writes each array as out_dir/<name>.npy in float32 (exact for the u8 records and int32 step counts).  When the files
    would exceed DUMP_LIMIT, the same seeded sample of rows is taken from every array and its indices are written as
    rows.npy, so that two builds run with the same arguments write the same rows."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    host = {k: v.detach().cpu().numpy().astype(np.float32) for k, v in arrays.items()}
    n = len(next(iter(host.values())))
    row_bytes = sum(a[:1].nbytes for a in host.values())
    if n * row_bytes + len(host) * NPY_HEADER_MAX > DUMP_LIMIT:  # sample rows; one more file, rows.npy (8 bytes a row)
        keep = (DUMP_LIMIT - (len(host) + 1) * NPY_HEADER_MAX) // (row_bytes + 8)
        rows = np.sort(np.random.default_rng(seed).choice(n, keep, replace=False))
        host = {k: a[rows] for k, a in host.items()}
        host["rows"] = rows.astype(np.float64)
    for k, a in host.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)
    return sorted(host)


def cpu_port(n_games, threads, seed0=10_000_000):
    """The oracle port (plain C restatement of the reference engine) on `threads` host threads."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import numpy as np
    import sb_oracle as oracle
    from monsoon_b200.engine import DEFAULT_DECKS, DEFAULT_FACTIONS, deck_indices
    d0, d1 = (deck_indices(d) for d in DEFAULT_DECKS)
    # dealing the games is a single-threaded Python loop over the C oracle: kept OUT of the CPU arm's clock (the GPU
    # arm's clock includes its reset kernel), so the comparison errs in the CPU's favour
    states = np.stack([oracle.new_game(seed0 + i, d0, d1, *DEFAULT_FACTIONS) for i in range(n_games)])
    t0 = time.perf_counter()
    total, _steps = oracle.batch_random(states, 400, threads)
    dt = time.perf_counter() - t0
    return total, dt


def python_reference_leg(n_games=256):
    """BASELINE.md section 3: the reference's own Python engine, unmodified, multiprocessing.Pool(os.cpu_count()) on the
    box's host cores, a bounded sample (256 whole games) of the same workload.  None when no copy of the reference is at hand."""
    try:
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import ref_python_baseline
        r = ref_python_baseline.run(n_games)
        return None if r is None else {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")}
    except Exception as e:  # noqa: BLE001 -- a reported baseline must never take the bench line down
        return {"unavailable": "%s: %s" % (type(e).__name__, e)}


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path on all host cores.  The reference is pure Python; its
    unmodified engine travels to the GPU box as the staged copy oracle/_ref/monsoon (oracle/stage_ref.py) and is what this arm times
    (kind "reference": games/stormbound.py, multiprocessing.Pool(os.cpu_count()), a bounded sample of the job's games per step).
    The plain-C oracle port on all host threads is printed beside it (`cpu_baseline_port`); it is the arm itself only when no copy
    of the reference is at hand."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    n_games = 4096 * max(args.gpus, 1)  # the job's games per step: 4,096 per GPU, like the GPU arm at this N
    # the port: every step plays all n_games; exactly args.warmup untimed steps, then exactly args.steps timed ones
    for _ in range(args.warmup):
        cpu_port(n_games, threads)
    tot_steps, tot_t = 0, 0.0
    for k in range(args.steps):
        s, dt = cpu_port(n_games, threads, seed0=20_000_000 + k * n_games)
        tot_steps += s
        tot_t += dt
    port = {"value": tot_steps / tot_t, "unit": "env_steps/s", "cores": threads, "kind": "port", "timed_steps": args.steps,
            "env_steps": int(tot_steps), "seconds": tot_t,
            "sample": "%d games (default decks, random agents, to completion) per step, %d steps; dealing excluded from the clock" % (n_games, args.steps)}
    # the reference itself: a bounded sample of the same games per step (whole games; ~500 env steps/s per core), exactly
    # args.warmup untimed and args.steps timed steps like the port
    py, py_steps, py_t, sample_games = None, 0, 0.0, max(64, 2 * threads)
    try:
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import ref_python_baseline
        if ref_python_baseline.reference_dir() is not None:
            for k in range(args.warmup + args.steps):
                r = ref_python_baseline.run(sample_games, seed0=30_000_000 + k * 100_000)
                if k >= args.warmup:
                    py_steps += r["steps"]
                    py_t += r["seconds"]
            py = {"value": py_steps / py_t, "unit": "env_steps/s", "cores": threads, "kind": "reference", "timed_steps": args.steps,
                  "env_steps": int(py_steps), "seconds": py_t,
                  "sample": "%d of the job's %d games per step (default decks, random agents, to completion, %d env steps in %.1f s in all): the "
                            "reference's unmodified Python engine (games/stormbound.py) under multiprocessing.Pool(%d)"
                            % (sample_games, n_games, py_steps, py_t, threads)}
    except Exception as e:  # noqa: BLE001 -- fall back to the port rather than lose the arm
        py = None
        port["reference_unavailable"] = "%s: %s" % (type(e).__name__, e)
    arm = py or port
    line = {
        "impl": "reference", "metric": METRIC, "value": arm["value"], "unit": "env_steps/s", "n_gpus": args.gpus, "steps": arm["timed_steps"],
        "warmup": args.warmup, "ms_per_step": 1e3 * arm["seconds"] / arm["timed_steps"],
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": bench_config(),
        "notes": "CPU arm = the reference's own Python engine on all host cores (kind reference) when its staged copy travelled with the "
                 "snapshot, else the plain-C oracle port; the port (about 1,000x faster per core than the Python) is printed in cpu_baseline_port",
        "cpu_baseline": arm,
        "cpu_baseline_port": port,
        "e2e": {"value": arm["value"], "unit": "env_steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--games", type=int, default=4096, help="parallel games per GPU (the named workload is 4096)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-saturated", action="store_true")
    ap.add_argument("--no-evo", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the final game records and env-step counts of the last timed step "
                                                          "(rank 0) as DIR/states.npy and DIR/steps.npy, float32")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 0:
        ap.error("--warmup must not be negative")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what the GPU path computed: not available with --impl reference")
    if args.impl == "reference":
        return run_reference(args)
    load_ncu_constants()

    import numpy as np
    import torch
    import torch.distributed as dist
    from monsoon_b200.engine import Engine

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    torch.cuda.set_device(local_rank)
    eng = Engine(local_rank)
    dev = eng.device
    n = args.games
    warmup = max(args.warmup, 3)

    seeds = torch.empty(n, dtype=torch.int64, device=dev)
    base = torch.arange(n, dtype=torch.int64, device=dev)
    states = eng.empty_states(n)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)  # > 126 MB L2
    steps_total = torch.zeros((), dtype=torch.int64, device=dev)
    last_steps = []

    def one_pass(k, timed):
        seeds.copy_(base + (rank * 1_000_003 + k) * n)
        flush.fill_(k & 255)  # L2 flush between timed iterations (outside the event-bracketed region)
        e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        e0.record()
        eng.reset(seeds, out=states)
        e1.record()
        st = eng.rollout_random(states, max_steps=400)
        e2.record()
        if timed:
            steps_total.add_(st.sum())
            last_steps[:] = [st]
        return e0, e1, e2

    for k in range(warmup):
        one_pass(k, False)
    torch.cuda.synchronize()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.prepare()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    launches0 = eng.launches
    if rank == 0:
        sampler.start()
    events = [one_pass(warmup + k, True) for k in range(args.steps)]
    if rank == 0:
        sampler.sample_once()  # launches are asynchronous: the GPU is inside the timed work here
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    launches = eng.launches - launches0
    sampler.stop_flag = True
    if args.dump_outputs and rank == 0:  # after the timed region: what the caller of reset + rollout_random received last
        dump_outputs(args.dump_outputs, {"states": states, "steps": last_steps[0]})
    t_ms = sum(e0.elapsed_time(e2) for e0, _e1, e2 in events)
    t_roll_ms = sum(e1.elapsed_time(e2) for _e0, e1, e2 in events)
    tt = torch.tensor([t_ms, t_roll_ms], dtype=torch.float64, device=dev)
    tot = steps_total.clone()
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
    t_ms, t_roll_ms = (float(x) for x in tt.cpu())
    total_steps = int(tot.cpu())
    value = total_steps / (t_ms * 1e-3)

    # end to end through the C ABI with HOST buffers (sb_rollout_random_host: H2D seeds/decks, both kernels,
    # D2H final states + step counts, stream sync), wall clock around the call
    # The step's inputs (seeds) and results (final states, step counts) live in PINNED host memory.
    seeds_pin = torch.empty(n, dtype=torch.int64, pin_memory=True)
    states_pin = torch.empty((n, 512), dtype=torch.uint8, pin_memory=True)
    steps_pin = torch.empty(n, dtype=torch.int32, pin_memory=True)
    seeds_h = np.arange(n, dtype=np.uint64)
    sh = seeds_pin.numpy().view(np.uint64)
    e2e_steps, e2e_t = 0, 0.0
    for k in range(warmup + args.steps):
        sh[:] = seeds_h + np.uint64((rank * 1_000_003 + 50_000 + k) * n)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        _st, steps_h, _ = eng.rollout_random_host(sh, max_steps=400, want_states=True, out_states=states_pin.numpy(), out_steps=steps_pin.numpy())
        dt = time.perf_counter() - t0
        if k >= warmup:
            e2e_steps += int(steps_h.sum())
            e2e_t += dt
    e2 = torch.tensor([e2e_t], dtype=torch.float64, device=dev)
    es = torch.tensor([e2e_steps], dtype=torch.int64, device=dev)
    if world > 1:
        dist.all_reduce(e2, op=dist.ReduceOp.MAX)
        dist.all_reduce(es, op=dist.ReduceOp.SUM)
    e2e_value = int(es.cpu()) / float(e2.cpu())

    # capacity figure beside the named workload: the same kernels on a batch that fills the chip (one rank's number)
    sat = None
    if not args.no_saturated:
        ns = 262144
        sseeds = torch.arange(ns, dtype=torch.int64, device=dev) + 900_000_000 + rank * 10_000_000
        sstates = eng.empty_states(ns)
        best, ssteps = None, 0
        for rep in range(3):
            eng.reset(sseeds + rep * ns, out=sstates)
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a0.record()
            st = eng.rollout_random(sstates, max_steps=400)
            a1.record()
            torch.cuda.synchronize()
            ms = a0.elapsed_time(a1)
            if rep and (best is None or ms < best):
                best, ssteps = ms, int(st.sum())
        sv = torch.tensor([best, float(ssteps)], dtype=torch.float64, device=dev)
        if world > 1:  # whole-job figure: total steps over the slowest rank's time
            mx = sv.clone()
            dist.all_reduce(mx, op=dist.ReduceOp.MAX)
            dist.all_reduce(sv, op=dist.ReduceOp.SUM)
            best, ssteps = float(mx[0]), float(sv[1])
        sat = {"games_per_gpu": ns, "value": ssteps / (best * 1e-3), "unit": "env_steps/s", "ms": best,
               "games_per_sec": ns * world / (best * 1e-3), "hbm_equiv_gbs": B_STEP * ssteps / (best * 1e-3) / 1e9,
               "roofline": {"kernel": NCU["rollout_262144"]["kernel"], "traffic": NCU["rollout_262144"]["dram_bytes"],
                            "traffic_unit": "bytes per launch (ncu, %s)" % NCU["rollout_262144"]["capture"],
                            "issue": issue_roofline("rollout_262144", ssteps / world, best * 1e-3, eng.sm_count, 1965)}}
        del sstates

    # the third part of BASELINE.json's metric: wall time of one evo fitness evaluation (config 3: population
    # 256 x 256 games/individual as FIRST vs one heuristic baseline, heuristic agents on both sides, 65,536 games
    # sharded over the ranks; weights broadcast + int32 count all-reduce over NCCL), through the public
    # FitnessEvaluator API (host seed derivation and H2D of seeds/indices inside the timed region)
    evo = None
    if not args.no_evo:
        from monsoon_b200.evo import FitnessEvaluator, WeightVector

        class _Cfg:
            games_per_pairing, max_turns, seed, num_workers = 256, 400, 1, 1

        def _vec(w):
            v = WeightVector(10)
            v.weights = np.asarray(w, dtype=np.float64)
            return v
        pop = [_vec(w) for w in np.random.RandomState(42).uniform(0, 1, (256, 10))]
        opp = [_vec(np.random.RandomState(7).uniform(0, 1, 10))]
        ev = FitnessEvaluator(_Cfg(), engine=eng)
        walls = []
        for gen in range(2):
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()
            t0 = time.perf_counter()
            fit = ev.evaluate_vs(pop, opp, generation=gen, games_per_opponent=256)
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()
            walls.append(time.perf_counter() - t0)
        evo = {"config": "pop 256 x 256 games vs heuristic baseline (65,536 games, max 400 steps)", "generation_wall_s": walls[-1],
               "games_per_sec": 65536 / walls[-1], "mean_fitness": float(np.mean(fit)),
               "aborted_games": {"like_reference": ev.last_aborted[0], "engine_limit": ev.last_aborted[1]},
               "roofline": {"kernel": NCU["heuristic_65536"]["kernel"], "traffic": NCU["heuristic_65536"]["dram_bytes"],
                            "traffic_unit": "bytes per 65,536-game launch on one GPU (ncu, %s)" % NCU["heuristic_65536"]["capture"],
                            "threads_per_inst": NCU["heuristic_65536"]["threads_per_inst"],
                            "issue_active_pct": NCU["heuristic_65536"]["issue_active_pct"]}}

    if rank == 0:
        peak, peak_src = measured_peak()
        steps_per_launch = total_steps / world / max(args.steps, 1)
        achieved = B_STEP * steps_per_launch / (t_roll_ms / args.steps * 1e-3) / 1e9
        out = {
            "metric": METRIC, "value": value, "unit": "env_steps/s", "n_gpus": world, "steps": args.steps, "warmup": warmup,
            "ms_per_step": t_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u8", "data": "synthetic",
            "config": bench_config(n),
            "notes": {"l2": "flushed between timed iterations (256 MiB fill)",
                      "timing": "CUDA events on the launch stream, reset+rollout kernels, max over ranks",
                      "e2e": "sb_rollout_random_host: pinned host seeds in, final states + step counts out, H2D + both kernels + D2H + "
                             "stream sync inside a host wall clock; other seeds than the event-timed passes, no L2 flush between calls",
                      "engine": "default policy: one game per warp (kw_rollout_random, turn-synchronous 32-warp CTAs) while the batch fits "
                                "one wave, one game per thread (k_rollout_random) beyond; both bit-identical (tests/test_gpu_engines.py)"},
            "games_per_sec": n * world * args.steps / (t_ms * 1e-3),
            "env_steps_per_game": total_steps / (n * world * args.steps),
            "gpu_launches": launches,
            "e2e": {"value": e2e_value, "unit": "env_steps/s", "h2d_bytes_per_step": n * 8 + 24 + 2,
                    "d2h_bytes_per_step": n * 512 + n * 4},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": NCU["rollout_4096"]["dram_bytes"] if n == 4096 else None,
                         "traffic_unit": "bytes per launch (ncu --set full, %s)" % NCU["rollout_4096"]["capture"],
                         "kernel": NCU["rollout_4096"]["kernel"], "peak_source": peak_src, "algorithmic_bytes_per_env_step": B_STEP,
                         # what actually bounds a whole-game rollout (SURVEY 8d): warp-instruction issue, not HBM
                         "issue": issue_roofline("rollout_4096", steps_per_launch, t_roll_ms / args.steps * 1e-3, eng.sm_count,
                                                 (sampler.summary().get("sm_max_mhz") or 1965))},
            "clocks": sampler.summary(),
        }
        if sat:
            out["saturated"] = sat
        if evo:
            out["evo_generation"] = evo
        if world == 1 and not args.no_cpu_baseline:
            threads = os.cpu_count() or 1
            ng = 131072  # ~20 core-seconds of rollouts
            s, dt = cpu_port(ng, threads)
            port = {"value": s / dt, "unit": "env_steps/s", "cores": threads, "kind": "port",
                    "sample": "%d games of the same workload (%d env steps), rollouts only, in %.2f s wall on %d threads" % (ng, s, dt, threads)}
            py = python_reference_leg()
            # the reference's own Python engine when its staged copy is at hand (BASELINE.md section 3), the plain-C port beside it
            out["cpu_baseline"] = py if (py and "value" in py) else port
            out["cpu_baseline_port"] = port
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()

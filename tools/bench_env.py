"""GPU: the batched environment (sb_env_step, one launch per call) at n = 4,096 and 65,536 for each opponent kind, and beside
it, for opponents 0 and 2, the loop a user writes without it: torch gather / scatter of the finished envs + sb_reset, rounds of
sb_expert_action / sb_step on the envs where the opponent is to move (one host synchronisation per round), then sb_observe and
sb_legal_mask.  Both paths start from the same records and get the same actions; the script asserts that they return identical
records, observations, masks and results before it times them.

Timing: CUDA events around the env call (or the whole composed call) only, summed over windows of at least --seconds seconds after
--warmup calls.  The learner is a uniform-random legal policy drawn on the device by torch (outside the timed region).
Reports ms per call, learner steps/s (n / call time) and total env steps/s (both seats, from the records' step counters).
Usage: python tools/bench_env.py [--sizes 4096 65536] [--seconds 1.0] [--out FILE]"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT]
import torch  # noqa: E402

from monsoon_b200.engine import Engine  # noqa: E402
from monsoon_b200.state import PLAYER_DTYPE, STATE_DTYPE  # noqa: E402
from monsoon_b200.vec_env import next_seed_array  # noqa: E402

F = STATE_DTYPE.fields
OFF_STEPS, OFF_SIGN, OFF_ERR = F["steps"][1], F["player_sign"][1], F["err"][1]
OFF_BASE = [F["pl"][1] + o * PLAYER_DTYPE.itemsize + PLAYER_DTYPE.fields["base"][1] for o in range(2)]
MAX_STEPS = 400


def i16(states, off):
    return states[:, off:off + 2].contiguous().view(torch.int16).flatten().to(torch.int32)


def gpu_identity():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True,
                           timeout=30)
        power = q.stdout.strip() or "unknown"
    except (OSError, subprocess.SubprocessError):
        power = "unknown"
    return name, power


class Composed:
    """The hand-written environment loop over the pinned entry points (opponent 0 or 2)."""

    def __init__(self, eng, opponent, seat, decks, factions):
        self.eng, self.opponent, self.seat, self.decks, self.factions = eng, opponent, seat.to(torch.int32), decks, factions

    def over(self, st):
        return (i16(st, OFF_BASE[0]) < 0) | (i16(st, OFF_BASE[1]) < 0) | (st[:, OFF_ERR] != 0) | (i16(st, OFF_STEPS) >= MAX_STEPS)

    def to_move(self, st):
        return (st[:, OFF_SIGN].view(torch.int8) != 1).to(torch.int32)

    def opponent_rounds(self, st, seat):
        if self.opponent == 0:
            return
        while True:
            idx = torch.nonzero((self.to_move(st) != seat) & ~self.over(st)).flatten()
            if idx.numel() == 0:  # host synchronisation: one per round
                return
            sub = st[idx]
            a = self.eng.expert_action(sub)
            self.eng.step(sub, a)
            st[idx] = sub

    def next_seeds(self, st):
        key = st[:, 0:8].contiguous().view(torch.int64).flatten()

        def shr(z, k):  # logical shift of the int64 bit pattern
            return (z >> k) & ((1 << (64 - k)) - 1)
        z = key + (0x9E3779B97F4A7C15 - (1 << 64))
        z = (z ^ shr(z, 30)) * (0xBF58476D1CE4E5B9 - (1 << 64))
        z = (z ^ shr(z, 27)) * (0x94D049BB133111EB - (1 << 64))
        z = z ^ shr(z, 31)
        return z & 0x7FFFFFFFFFFFFFFF

    def step(self, st, actions):
        e = self.eng
        m = e.legal_mask(st)
        a = actions.to(torch.int64)
        word = torch.gather(m, 1, (a.clamp(max=155) >> 5)[:, None]).flatten()
        legal = (a < 156) & (((word >> (a & 31)) & 1) != 0)
        before = st.clone()
        e.step(st, actions)
        self.opponent_rounds(st, self.seat)
        ended = self.over(st) & legal
        l0, l1 = i16(st, OFF_BASE[0]) < 0, i16(st, OFF_BASE[1]) < 0
        res = torch.where(l1 & ~l0, 0, torch.where(l0 & ~l1, 1, -1))
        res = torch.where(st[:, OFF_ERR] != 0, -2, res)
        res = torch.where(ended, res, torch.where(legal, -3, -4)).to(torch.int8)
        length = torch.where(ended, i16(st, OFF_STEPS), 0)
        final = st.clone()
        idx = torch.nonzero(ended).flatten()
        if idx.numel():
            fresh = e.reset(self.next_seeds(st)[idx].contiguous(), self.decks, self.factions)
            self.opponent_rounds(fresh, self.seat[idx])
            st[idx] = fresh
        st.copy_(torch.where(legal[:, None], st, before))
        obs, oerr = e.observe(st)
        masks = e.legal_mask(st)
        return {"result": res, "length": length, "final_states": final, "obs": obs, "masks": masks, "obs_err": oerr}


def random_legal(masks, gen):
    bits = ((masks.unsqueeze(-1) >> torch.arange(32, dtype=torch.int32, device=masks.device)) & 1).reshape(masks.shape[0], -1)[:, :156]
    return (torch.rand(bits.shape, device=masks.device, generator=gen) * bits).argmax(1).to(torch.uint8)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", type=int, nargs="+", default=[4096, 65536])
    ap.add_argument("--seconds", type=float, default=1.0)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_env.py needs a CUDA device")
    eng = Engine(0)
    dev = eng.device
    name, power = gpu_identity()
    print("GPU: %s, power limit %s" % (name, power), flush=True)
    decks, factions = eng._default_deck_tensors()
    lines = []
    for n in args.sizes:
        seeds = torch.from_numpy(next_seed_array(range(n))).to(dev)
        seat = (torch.arange(n, device=dev) % 2).to(torch.uint8)
        w = torch.rand((64, 10), dtype=torch.float64, device=dev, generator=torch.Generator(device=dev).manual_seed(1))
        idx = (torch.arange(n, device=dev) % 64).to(torch.int32)
        for opponent in range(4):
            kw = dict(opponent=opponent, seat=seat, w_opp=w, idx_opp=idx, max_steps=MAX_STEPS)
            gen = torch.Generator(device=dev).manual_seed(n + opponent)
            o = eng.env_reset(seeds, **kw)
            st = o["states"]
            out = eng._env_outputs(n, None, ("result", "length", "final_states", "obs", "masks", "obs_err"))
            masks = o["masks"]
            composed = Composed(eng, opponent, seat, decks, factions) if opponent in (0, 2) else None
            if composed is not None:  # identity before timing: same records, same actions, episodes ending and restarting
                st2 = st.clone()
                for _ in range(150 if opponent == 0 else 40):
                    a = random_legal(masks, gen)
                    a[::97] = 200  # a few rejected actions
                    eng.env_step(st, a, out=out, **kw)
                    c = composed.step(st2, a)
                    assert torch.equal(st, st2), (n, opponent)
                    for k in ("result", "length", "obs", "masks", "obs_err"):
                        assert torch.equal(out[k].to(c[k].dtype), c[k]), (n, opponent, k)
                    done = out["result"] > -3
                    assert torch.equal(out["final_states"][done], c["final_states"][done]), (n, opponent)
                    masks = out["masks"]
            arms = [("env_step", None)] + ([("composed", composed)] if composed is not None else [])
            for arm, comp in arms:
                work = st.clone()
                m = masks.clone()
                total_steps = torch.zeros((), dtype=torch.int64, device=dev)
                ms, calls, k = 0.0, 0, 0
                while k < args.warmup or ms < args.seconds * 1e3:
                    a = random_legal(m, gen)
                    s0 = i16(work, OFF_STEPS)
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    r = eng.env_step(work, a, out=out, **kw) if comp is None else comp.step(work, a)
                    e1.record()
                    m = r["masks"]
                    if k >= args.warmup:
                        total_steps += (i16(work, OFF_STEPS) - s0 + r["length"]).sum()
                        e1.synchronize()
                        ms += e0.elapsed_time(e1)
                        calls += 1
                    k += 1
                tot = int(total_steps)
                rec = {"n": n, "opponent": opponent, "path": arm, "calls": calls, "ms_per_call": ms / calls,
                       "learner_steps_per_s": n * calls / (ms / 1e3), "env_steps_per_s": tot / (ms / 1e3), "gpu": name, "power_limit": power}
                lines.append(rec)
                print(json.dumps(rec), flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write("# tools/bench_env.py on %s, power limit %s\n" % (name, power))
            for r in lines:
                f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()

"""CPU-only measure of the hot instruction footprint of a warp-engine kernel (default: the bench's kw_rollout_random<32,1,1>).

Execution counts come from the host twin of the warp engine (tests/wsim/wsim.cpp, the same sbw_*.cuh source) built with
gcc --coverage and made to play the bench's workload: default decks, uniform-random legal agents, every game to
completion (max 400 env steps), dealt by the oracle from seeds 0..N-1.  Every SASS instruction of the kernel (its own code
and its private copies of the callees, read from the library built by monsoon_b200/build.py with -lineinfo) gets the
count of its source line, per WARP:
  * a uniform line counts once per execution;
  * a line inside FOR_LANES ... END_LANES or a lane lambda of the collectives runs 32 times on the host per entry of the
    section and counts as (its host count / 32), rounded up;
  * an instruction of an inlined helper gets the count of the outermost call site in the device function it sits in,
    times the helper line's executions per call of the helper (both from the host counts), frame by frame;
  * the kernel's own lines (sbw_kernels.cu, not part of the host twin) count once per env step inside the turn-synchronous
    rounds, once per game elsewhere, and not at all on the chain-digest path (the bench passes no chain).
Counts are per source line, so every instruction of a line gets the line's count: instructions of a line that branches
or loops within itself are over-weighted (the weighted total runs ~3x the measured 1.7 k warp instructions per env step).
The footprint is a ranking of the instructions by heat, not an instruction count; compare it between builds.
The report: the bytes of SASS that cover 90 / 99 / 99.9 % of the weighted instructions, the same per function, and how
many distinct 128-byte lines of the kernel image those hot instructions touch.  No GPU is needed.

  python tools/hot_footprint.py [--games 4096] [--lib monsoon_b200/libsb_b200.so | --cubin FILE] [--json OUT]
"""
import argparse
import bisect
import collections
import ctypes
import json
import math
import os
import re
import shutil
import subprocess
import sys
import tempfile

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(REPO, "monsoon_b200", "csrc")
WSIM = os.path.join(REPO, "tests", "wsim", "wsim.cpp")
CUDA = os.environ.get("CUDA_HOME", "/usr/local/cuda")
LEVELS = (0.90, 0.99, 0.999)
LINE_BYTES = 128


# ---------------------------------------------------------------- host execution counts
def play(so, n_games, max_steps):
    """child process: the bench's games through the coverage build; the counts are written when the process exits"""
    sys.path.insert(0, os.path.join(REPO, "oracle"))
    sys.path.insert(0, REPO)
    import numpy as np
    import sb_oracle
    from monsoon_b200.engine import DEFAULT_DECKS, DEFAULT_FACTIONS, deck_indices
    sb_oracle.build()
    d0, d1 = (deck_indices(d) for d in DEFAULT_DECKS)
    L = ctypes.CDLL(so)
    L.wsim_rollout_random.restype = ctypes.c_int
    steps = 0
    for seed in range(n_games):
        st = sb_oracle.new_game(seed, d0, d1, *DEFAULT_FACTIONS)
        steps += L.wsim_rollout_random(st.ctypes.data_as(ctypes.c_void_p), max_steps, None, None)
    print(json.dumps({"games": n_games, "env_steps": steps}))


def host_counts(tmp, n_games, max_steps):
    """{(basename, line): host count}, {basename: [(start, end, calls, name)]}, env steps"""
    obj = os.path.join(tmp, "wsim.o")
    so = os.path.join(tmp, "libwsim_cov.so")
    flags = ["-O0", "--coverage", "-std=c++17", "-fPIC", "-ffp-contract=off", "-fno-strict-aliasing", "-w"]
    subprocess.check_call(["g++"] + flags + ["-c", "-x", "c++", WSIM, "-o", obj])
    subprocess.check_call(["g++", "-shared", "--coverage", obj, "-o", so])
    out = subprocess.run([sys.executable, os.path.abspath(__file__), "--play", so, "--games", str(n_games), "--max-steps", str(max_steps)],
                         check=True, capture_output=True, text=True).stdout
    played = json.loads(out.strip().splitlines()[-1])
    js = subprocess.run(["gcov", "--json-format", "--stdout", "-o", tmp, os.path.join(tmp, "wsim.gcda")], check=True, capture_output=True,
                        text=True, cwd=tmp).stdout
    counts, funcs = collections.Counter(), collections.defaultdict(list)
    for doc in js.splitlines():
        if not doc.strip():
            continue
        for f in json.loads(doc)["files"]:
            base = os.path.basename(f["file"])
            if not (base.startswith("sbw_") or base.startswith("sb_")):
                continue
            for ln in f["lines"]:
                counts[(base, ln["line_number"])] += ln["count"]
            for fn in f["functions"]:
                funcs[base].append((fn["start_line"], fn["end_line"], fn["execution_count"], fn["demangled_name"]))
    return counts, funcs, played["env_steps"]


def lane_lines(path):
    """line numbers that belong to a FOR_LANES ... END_LANES section or to the body of a lane lambda ([&](int ...) { ... })"""
    src = open(path).read()
    starts = [0] + [m.end() for m in re.finditer("\n", src)]
    line_of = lambda pos: bisect.bisect_right(starts, pos)
    out = set()
    for m in re.finditer(r"FOR_LANES\(", src):
        e = src.find("END_LANES", m.end())
        out.update(range(line_of(m.start()), line_of(e) + 1))
    for m in re.finditer(r"\[&\]\(int \w+\)[^{]*\{", src):
        depth, i = 1, m.end()
        while depth:
            depth += {"{": 1, "}": -1}.get(src[i], 0)
            i += 1
        out.update(range(line_of(m.start()), line_of(i) + 1))
    return out


class Weights:
    def __init__(self, counts, funcs, env_steps, games):
        self.counts, self.env_steps, self.games, self.kernel_src = counts, env_steps, games, None
        self.lanes = {b: lane_lines(os.path.join(CSRC, b)) for b in funcs if os.path.exists(os.path.join(CSRC, b))}
        calls = collections.defaultdict(lambda: [0, False])  # (base, start, end) -> [calls, is lambda]
        for b, fl in funcs.items():
            for s, e, c, name in fl:
                k = calls[(b, s, e)]
                k[0] += c
                k[1] = k[1] or "lambda" in name
        self.funcs = collections.defaultdict(list)
        for (b, s, e), (c, lam) in calls.items():
            self.funcs[b].append((s, e, math.ceil(c / 32) if lam else c))

    def kernel_line(self, ln):
        """the kernel's own lines: once per env step in the turn-synchronous rounds (phase A loop, phase B block), once per
        game elsewhere; the chain-digest lines not at all (the bench passes no chain)"""
        if self.kernel_src is None:
            src = open(os.path.join(CSRC, "sbw_kernels.cu")).read().split("\n")
            a = next(i for i, l in enumerate(src) if "phase A" in l)
            b = next(i for i, l in enumerate(src) if "phase B" in l)
            depth, e = 0, b
            for e in range(b, len(src)):
                depth += src[e].count("{") - src[e].count("}")
                if depth <= 0:
                    break
            self.kernel_src = (src, a + 1, e + 1)
        src, a, e = self.kernel_src
        if "digest" in src[ln - 1]:
            return 0
        return self.env_steps if a <= ln <= e else self.games

    def line(self, base, ln):
        """per-warp count of a source line, or None when the host twin has no code on it"""
        c = self.counts.get((base, ln))
        if c is None:
            return None
        return math.ceil(c / 32) if ln in self.lanes.get(base, ()) else c

    def enclosing_calls(self, base, ln):
        best = None
        for s, e, c in self.funcs.get(base, ()):
            if s <= ln <= e and (best is None or e - s < best[1] - best[0]):
                best = (s, e, c)
        return None if best is None else best[2]

    def instruction(self, chain):
        """chain: [(base, line)] innermost first, outermost = the device function the instruction sits in"""
        base, ln = chain[-1]
        if base == "sbw_kernels.cu":
            w = float(self.kernel_line(ln))
        else:
            w = self.line(base, ln)
            if w is None:
                w = self.enclosing_calls(base, ln)
            if w is None:
                return None
            w = float(w)
        for b, l in reversed(chain[:-1]):  # per-call ratio of each inlined frame, outermost first
            c, calls = self.line(b, l), self.enclosing_calls(b, l)
            if c is None or not calls:
                continue
            w *= c / calls
        return w


# ---------------------------------------------------------------- SASS with inline line info
def mangled_prefix(kernel):
    m = re.fullmatch(r"(\w+)<([\d,\s]+)>", kernel)
    if not m:
        return "_Z%d%s" % (len(kernel), kernel)
    args = "".join("Li%dE" % int(a) for a in m.group(2).split(","))
    return "_Z%d%sI%sE" % (len(m.group(1)), m.group(1), args)


def cubin_of(lib, tmp, prefix):
    """the sm_100a cubin of `lib` that holds the kernel"""
    d = os.path.join(tmp, "elf")
    os.makedirs(d, exist_ok=True)
    subprocess.run([os.path.join(CUDA, "bin", "cuobjdump"), "-xelf", "all", os.path.abspath(lib)], check=True, capture_output=True, cwd=d)
    for f in sorted(os.listdir(d)):
        p = os.path.join(d, f)
        syms = subprocess.run([os.path.join(CUDA, "bin", "cuobjdump"), "-elf", p], check=True, capture_output=True, text=True).stdout
        if ".text." + prefix in syms:
            return p
    raise SystemExit("no cubin of %s holds %s" % (lib, prefix))


FILE_RE = re.compile(r'File "([^"]+)", line (\d+)')
INS_RE = re.compile(r"^\s+/\*([0-9a-f]{4,})\*/\s+(.*?)\s*;")


def sass(cubin, prefix):
    """[(offset, function, chain, text)] of the kernel's text section"""
    txt = subprocess.run([os.path.join(CUDA, "bin", "nvdisasm"), "-c", "-gi", cubin], check=True, capture_output=True, text=True).stdout
    out, inside, func, chain, block = [], False, "(kernel)", [], []
    for line in txt.splitlines():
        if line.startswith("\t.section"):
            inside = line.split()[1].rstrip(",").startswith(".text." + prefix)
            continue
        if not inside:
            continue
        if line.startswith("$") and line.endswith(":"):
            m = re.search(r"\$_Z(\d+)(\w+)", line[line.index("$", 1):])
            func = m.group(2)[:int(m.group(1))] if m else line
            continue
        if line.startswith("\t//## File"):
            block.append(line)
            continue
        m = INS_RE.match(line)
        if not m:
            continue
        if block:  # one annotation line per frame, innermost first ('File A, line x inlined at B, line y' ... 'File Z, line z')
            chain = [(os.path.basename(f), int(n)) for f, n in (FILE_RE.search(b).groups() for b in block)]
            block = []
        out.append((int(m.group(1), 16), func, list(chain), m.group(2)))
    if not out:
        raise SystemExit("kernel %s not found" % prefix)
    return out


# ---------------------------------------------------------------- report
def report(ins, wts):
    weights = [wts.instruction(c) if c else None for _, _, c, _ in ins]
    unmapped = sum(1 for w in weights if w is None)
    weights = [w or 0.0 for w in weights]
    total = sum(weights)
    order = sorted(range(len(ins)), key=lambda i: -weights[i])
    levels, acc, k = {}, 0.0, 0
    for lv in LEVELS:
        while acc < lv * total:
            acc += weights[order[k]]
            k += 1
        hot = order[:k]
        per = collections.Counter(ins[i][1] for i in hot)
        levels[lv] = {"instructions": k, "bytes": 16 * k, "lines_128B": len({ins[i][0] // LINE_BYTES for i in hot}),
                      "per_function_bytes": {f: 16 * n for f, n in per.most_common()}}
    size = collections.Counter(f for _, f, _, _ in ins)
    fw = collections.Counter()
    for (_, f, _, _), w in zip(ins, weights):
        fw[f] += w
    span = {}
    for off, f, _, _ in ins:
        lo, hi = span.get(f, (off, off))
        span[f] = (min(lo, off), max(hi, off))
    return {"instructions": len(ins), "bytes": 16 * len(ins), "weighted_instructions": total, "unmapped_instructions": unmapped,
            "levels": {"%g" % lv: v for lv, v in levels.items()},
            "functions": {f: {"bytes": 16 * size[f], "offset": span[f][0], "weight_share": fw[f] / total if total else 0.0} for f in size}}


def text(r, kernel, games, env_steps):
    o = ["hot footprint of %s: %d games, %d env steps (host twin, gcov); %d SASS instructions = %d bytes; %.4g weighted warp "
         "instructions = %.0f per env step; %d instructions without a count" %
         (kernel, games, env_steps, r["instructions"], r["bytes"], r["weighted_instructions"], r["weighted_instructions"] / max(env_steps, 1),
          r["unmapped_instructions"]), ""]
    o.append("%-8s %10s %10s %14s" % ("cover", "instr", "bytes", "128 B lines"))
    for lv, v in r["levels"].items():
        o.append("%-8s %10d %10d %14d" % ("%.1f %%" % (100 * float(lv)), v["instructions"], v["bytes"], v["lines_128B"]))
    o.append("")
    o.append("%-24s %8s %8s %8s %8s %8s %8s" % ("function", "offset", "bytes", "weight", "90 %", "99 %", "99.9 %"))
    fn = sorted(r["functions"].items(), key=lambda kv: -kv[1]["weight_share"])
    for f, v in fn:
        hot = [r["levels"][lv]["per_function_bytes"].get(f, 0) for lv in r["levels"]]
        if not any(hot) and v["weight_share"] == 0:
            continue
        o.append("%-24s %8x %8d %7.2f%% %8d %8d %8d" % (f[:24], v["offset"], v["bytes"], 100 * v["weight_share"], *hot))
    cold = [f for f, v in fn if v["weight_share"] == 0 and not any(r["levels"][lv]["per_function_bytes"].get(f, 0) for lv in r["levels"])]
    o.append("never executed: %s" % ", ".join(cold))
    return "\n".join(o) + "\n"


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--games", type=int, default=4096)
    ap.add_argument("--max-steps", type=int, default=400)
    ap.add_argument("--kernel", default="kw_rollout_random<32,1,1>")
    ap.add_argument("--lib", default=os.path.join(REPO, "monsoon_b200", "libsb_b200.so"))
    ap.add_argument("--cubin", help="a cubin of sbw_kernels.cu instead of the library")
    ap.add_argument("--json", help="write the full report here as JSON")
    ap.add_argument("--play", help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.play:
        return play(a.play, a.games, a.max_steps)
    prefix = mangled_prefix(a.kernel)
    tmp = tempfile.mkdtemp(prefix="hot_footprint_")
    try:
        counts, funcs, env_steps = host_counts(tmp, a.games, a.max_steps)
        ins = sass(a.cubin or cubin_of(a.lib, tmp, prefix), prefix)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    r = report(ins, Weights(counts, funcs, env_steps, a.games))
    r.update(kernel=a.kernel, games=a.games, env_steps=env_steps)
    sys.stdout.write(text(r, a.kernel, a.games, env_steps))
    if a.json:
        with open(a.json, "w") as f:
            json.dump(r, f, indent=1)


if __name__ == "__main__":
    main()

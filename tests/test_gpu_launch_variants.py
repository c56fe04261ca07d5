"""GPU: every kernel variant the launch policy picks, run at the batch sizes that pick it.

sb_kernels.cu does not run one kernel per entry point: it chooses the engine (one game per thread or per warp), the games
per warp, the CTA-synchronous block size, lane refill and the 32-register builds from the batch size and the SM count, and
the sbw_* launchers turn into persistent grid-stride loops once a batch exceeds one grid.  Every setting must give the
same results.  Here each variant runs at a batch size that selects it by default, against the oracle and against another
variant of the same call.

`expected_kernel` restates the policy as a table.  Each call is recorded with torch.profiler (CUDA activity, CUPTI), and
the kernel the table names must be among the kernels launched, with its template arguments and its grid: a policy change
that moves a size to another variant fails here and names the variant that is no longer reached.  Batch sizes are derived
from the SM count; the sizes in comments are the ones of a 148-SM B200.
"""
import contextlib
import json
import os
import re
import tempfile

import numpy as np
import pytest
import torch
from torch.profiler import ProfilerActivity, profile

from monsoon_b200.engine import CARD_INDEX, DEFAULT_DECKS, DEFAULT_FACTIONS, MASK_WORDS, PASS, deck_indices

pytestmark = pytest.mark.gpu

TPB_GAME = 64  # sb_kernels.cu: threads per CTA of the thread-per-game kernels
WARPS_PER_CTA = 4  # sb_kernels.cu: CTA size (in warps) of k_select_action
FNV = 0x100000001B3
AUTO = {"engine": -1, "block_sync": -1, "refill": -1, "dense": -1, "games_per_warp": 0, "refill_grid": 0, "w_grid": 0,
        "refill_ctas": 0, "w_shape": -1, "turn_sync": 1}


# ---------------------------------------------------------------- the launch policy as a table
def _cdiv(a, b):
    return (a + b - 1) // b


def _warp_engine(entry, n, sm, opt):
    """sb_kernels.cu use_warp_engine"""
    if opt["engine"] >= 0:
        return opt["engine"] != 0
    return {"rollout_random": n <= sm * 32, "step": n <= 8192, "legal_mask": True, "observe": True, "features": n <= 65536,
            "expert_action": n <= 16384, "select_action": False}[entry]


def _games_per_warp(n, sm, opt):
    """sb_kernels.cu games_per_warp"""
    if 0 < opt["games_per_warp"] <= 32:
        return opt["games_per_warp"]
    per_warp = _cdiv(2 * n, sm * 7)
    return 32 if per_warp > 16 else 16 if per_warp > 8 else 8


def expected_kernel(entry, n, sm_count, options):
    """(kernel name with its template arguments, grid) of the launch that `entry` makes for n records.  options: the
    handle's options (AUTO with overrides) plus "chain" for rollout_random (the digest chain was passed).  Restates
    use_warp_engine, games_per_warp, launch_rollout_random and sb_step (sb_kernels.cu), query_grid and the sbw_*
    launchers (sbw_kernels.cu); only the default CTA shapes of the warp engine (w_shape -1, w_grid 0) are covered."""
    opt = dict(AUTO, **options)
    sm = sm_count
    if _warp_engine(entry, n, sm, opt):
        if entry == "rollout_random":  # sbw_rollout_random, shape 5 (32 warps x 1) or 2 (8 warps x 8 per SM)
            wpc, per_sm, sync = (32, 1, 1) if n <= sm * 32 else (8, 8, 0)
            return "kw_rollout_random<%d,%d,%d>" % (wpc, per_sm, sync), min(_cdiv(n, wpc), sm * per_sm)
        if entry in ("legal_mask", "observe", "features"):  # kw_stream: 8 CTAs of 8 warps per SM
            mode = {"legal_mask": 0, "observe": 1, "features": 2}[entry]
            return "kw_stream<8,%d>" % mode, min(_cdiv(n, 8), sm * 8)
        if entry == "step":
            return "kw_step<8>", min(_cdiv(n, 8), sm * 32)
        if entry == "expert_action":
            return "kw_query<8,3>", min(_cdiv(n, 8), sm * 32)
        return "kw_select_action<4>", min(_cdiv(n, 4), sm * 32)
    gpw = _games_per_warp(n, sm, opt)
    dense = opt["dense"] if opt["dense"] >= 0 else int(n >= sm * 1536)
    if entry == "rollout_random":
        digest = "true" if opt.get("chain") else "false"
        bs = opt["block_sync"]
        if bs < 0:
            bs = 1024 if n >= 90000 else 512 if n >= 57000 else 128 if n >= 30000 else 0
        refill = opt["refill"] if opt["refill"] >= 0 else int(n > sm * 1024)
        queue = bool(refill) and bs >= 128 and gpw == 32
        tpb = 1024 if bs >= 1024 else 512 if bs >= 512 else 256 if bs >= 256 else 128
        qgrid = sm * (1024 // tpb)
        if bs >= 1024 and queue and dense:
            return "k_rollout_random<%s,1024,true,2>" % digest, 2 * sm
        for t in (1024, 512, 256, 128):
            if bs >= t:
                return "k_rollout_random<%s,%d,true,1>" % (digest, t), qgrid if queue else _cdiv(n, gpw * t // 32)
        return "k_rollout_random<%s,%d,false,1>" % (digest, TPB_GAME), _cdiv(n, gpw * TPB_GAME // 32)
    if entry == "step":
        return "k_step<%s>" % ("true" if dense else "false"), _cdiv(n, gpw * TPB_GAME // 32)
    if entry == "select_action":
        return "k_select_action", _cdiv(n, WARPS_PER_CTA)
    return {"legal_mask": "k_legal_mask", "observe": "k_observe", "features": "k_features",
            "expert_action": "k_expert_action"}[entry], _cdiv(n, TPB_GAME)


# ---------------------------------------------------------------- vacuity guard: which kernels a call launched
def _kernel_name(raw):
    """'void k_rollout_random<(bool)0, 1024, (bool)1, 2>(int, ...)' -> 'k_rollout_random<false,1024,true,2>'"""
    s = raw.replace("(bool)0", "false").replace("(bool)1", "true").replace("(int)", "")
    s = re.sub(r"^void\s+", "", s.strip())
    depth = 0
    for i, c in enumerate(s):
        depth += c == "<"
        depth -= c == ">"
        if c == "(" and depth == 0:
            s = s[:i]
            break
    return re.sub(r"\s+", "", s)


def _launched(fn):
    """fn() under torch.profiler: (its result, [(kernel name, (grid x, y, z))] of the library kernels it launched)"""
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as f:
            events = json.load(f).get("traceEvents", [])
    names = [(_kernel_name(e["name"]), tuple(e.get("args", {}).get("grid", (-1, -1, -1)))) for e in events if e.get("cat") == "kernel"]
    return out, [(k, g) for k, g in names if k.startswith(("k_", "kw_"))]


def run_checked(engine, entry, n, options, fn, again):
    """fn() (one library call of `entry` on n records) must launch the kernel and grid that expected_kernel names.
    A short profiling session now and then records no kernel at all; then again() (the same call on copies of its inputs)
    is recorded instead, up to twice.  If none of the sessions records a library kernel, the check fails."""
    name, grid = expected_kernel(entry, n, engine.sm_count, options)
    out, ours = _launched(fn)
    for _ in range(2):
        if ours:
            break
        _, ours = _launched(again)
    assert ours, ("torch.profiler recorded none of the library's kernels during %s(n=%d) in three sessions: without CUDA "
                  "activity tracing this test cannot tell which variant ran" % (entry, n))
    print("%-14s n=%-8d profiler: %s" % (entry, n, "; ".join("%s grid=%d" % (k, g[0]) for k, g in ours)))
    assert (name, (grid, 1, 1)) in ours, ("%s(n=%d, %s) should launch %s with grid %d; the profiler saw %s"
                                          % (entry, n, {k: v for k, v in options.items() if AUTO.get(k) != v}, name, grid, ours))
    return out


@contextlib.contextmanager
def options(handle, **overrides):
    """every option of the launch policy at its auto value, then the overrides; auto again afterwards"""
    for k, v in AUTO.items():
        handle.set_option(k, v)
    try:
        for k, v in overrides.items():
            handle.set_option(k, v)
        yield dict(AUTO, **overrides)
    finally:
        for k, v in AUTO.items():
            handle.set_option(k, v)


# ---------------------------------------------------------------- helpers
def sample(n):
    """oracle sample positions: the first and the last 256 records and every 211th"""
    return np.unique(np.r_[np.arange(min(n, 256)), np.arange(max(0, n - 256), n), np.arange(0, n, 211)])


def _chain(digests):
    ch = 0
    for d in digests:
        ch = ((ch ^ int(d)) * FNV) & 0xFFFFFFFFFFFFFFFF
    return ch


def _mix(x):
    x = (x ^ (x >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
    x = (x ^ (x >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    return x ^ (x >> np.uint64(31))


def pick_actions(masks, seed, rnd):
    """one legal action per record from its mask u32[n,5], by a fixed hash of (seed, round, record); about one in eight is
    PASS where PASS is legal, and PASS where nothing is"""
    n = masks.shape[0]
    bits = np.unpackbits(np.ascontiguousarray(masks).view(np.uint8).reshape(n, 4 * MASK_WORDS), axis=1, bitorder="little")[:, :156]
    h = _mix(np.arange(n, dtype=np.uint64) * np.uint64(0x9E3779B97F4A7C15) + np.uint64((seed * 1000003 + rnd) & 0xFFFFFFFF))
    cnt = bits.sum(axis=1).astype(np.int64)
    k = (h % np.maximum(cnt, 1).astype(np.uint64)).astype(np.int64)
    a = np.argmax(np.cumsum(bits, axis=1) > k[:, None], axis=1)
    a = np.where(((h >> np.uint64(61)) == 0) & (bits[:, PASS] == 1), PASS, a)
    return np.where(cnt == 0, PASS, a).astype(np.uint8)


def _alive(rec):
    return not (rec[19] & 1) and not rec[18]


def _default_deck_arrays(n):
    decks = np.empty((n, 2, 12), dtype=np.uint8)
    decks[:, 0], decks[:, 1] = deck_indices(DEFAULT_DECKS[0]), deck_indices(DEFAULT_DECKS[1])
    return decks, np.tile(np.array(DEFAULT_FACTIONS, dtype=np.uint8), (n, 1))


def _start_records(engine, n, seed0, random_deck_games=False):
    seeds = torch.arange(n, dtype=torch.int64, device=engine.device) + seed0
    if not random_deck_games:
        return engine.reset(seeds)
    from test_gpu_parity import random_decks
    decks, factions = zip(*(random_decks(seed0 + i, exclude=("UP01", "UP02", "UP03", "S203")) for i in range(n)))
    return engine.reset(seeds, torch.tensor(np.array(decks, dtype=np.uint8), device=engine.device),
                        torch.tensor(np.array(factions, dtype=np.uint8), device=engine.device))


# ---------------------------------------------------------------- (c) random rollouts at every auto shape
ROLLOUT_CASES = [  # id: the variant at 148 SMs; n from the SM count; forced options; random decks
    ("warp-shape5", lambda sm: 32 * sm, {}, False),                  # 4,736: kw_rollout_random<32,1,1>
    ("gpw16-bsync0", lambda sm: 41 * sm, {}, False),                 # 6,068: k_rollout_random<D,64,false,1>, gpw 16
    ("gpw32-bsync0", lambda sm: 20000, {}, False),                   # k_rollout_random<D,64,false,1>, gpw 32
    ("bsync128", lambda sm: 40000, {}, False),
    ("bsync256-forced", lambda sm: 40000, {"block_sync": 256}, False),
    ("bsync512", lambda sm: 60000, {}, False),
    ("bsync1024-one-wave", lambda sm: 100000, {}, False),
    ("refill-grid-sm", lambda sm: 1080 * sm, {}, True),              # 159,840: refill, 148 CTAs; every card effect
    ("refill-dense", lambda sm: max(262144, 1536 * sm), {}, False),  # bench.py's saturated workload, 296 CTAs
]


@pytest.mark.parametrize("case", ROLLOUT_CASES, ids=[c[0] for c in ROLLOUT_CASES])
def test_rollout_random_variants(engine, oracle, case):
    """the whole batch with and without the digest chain (the DIGEST=true / false builds) against each other and against
    the oracle's rollouts: final records byte for byte and step counts; digest chains on a sample"""
    _id, size, forced, random_deck_games = case
    n = size(engine.sm_count)
    start = _start_records(engine, n, 500000 + n, random_deck_games)
    with options(engine, **forced) as opt:
        st_chain = start.clone()
        chain = torch.zeros(n, dtype=torch.int64, device=engine.device)
        steps_chain = run_checked(engine, "rollout_random", n, dict(opt, chain=True),
                                  lambda: engine.rollout_random(st_chain, 400, chain=chain),
                                  lambda: engine.rollout_random(start.clone(), 400, chain=torch.zeros_like(chain)))
        st_plain = start.clone()
        steps_plain = run_checked(engine, "rollout_random", n, dict(opt, chain=False), lambda: engine.rollout_random(st_plain, 400),
                                  lambda: engine.rollout_random(start.clone(), 400))
    assert torch.equal(st_chain, st_plain) and torch.equal(steps_chain, steps_plain)
    host0 = start.cpu().numpy()
    want = host0.copy()
    _tot, want_steps = oracle.batch_random(want, 400, nthreads=os.cpu_count())
    got, steps, chain = st_chain.cpu().numpy(), steps_chain.cpu().numpy(), chain.cpu().numpy().view(np.uint64)
    bad = np.nonzero((got != want).any(axis=1) | (steps != want_steps))[0]
    assert bad.size == 0, "%d of %d games differ from the oracle, first %s" % (bad.size, n, bad[:10])
    for i in sample(n):
        _a, digests, _m = oracle.rollout_random(host0[i].copy(), 400)
        assert _chain(digests) == int(chain[i]), i


# ---------------------------------------------------------------- (d) sb_step across its variants
STEP_CASES = [
    ("kw_step", lambda sm: 8192, {}),
    ("k_step-gpw16", lambda sm: 8200, {}),
    ("k_step-gpw32", lambda sm: 50000, {}),
    ("k_step-dense", lambda sm: max(230000, 1536 * sm), {}),
    ("kw_step-grid-stride", lambda sm: max(40000, 256 * sm + 1), {"engine": 1}),  # one grid = 32 CTAs x 8 warps per SM
]


@pytest.mark.parametrize("case", STEP_CASES, ids=[c[0] for c in STEP_CASES])
def test_step_variants(engine, oracle, case):
    """8 rounds of legal_mask + step on mid-game records of mixed depths: the whole batch against the same records stepped
    in chunks of 4,096 (the warp engine), a sample against the oracle after every round"""
    _id, size, forced = case
    n = size(engine.sm_count)
    dev = engine.device
    st = _start_records(engine, n, 800000 + n)
    bounds = np.linspace(0, n, 9).astype(int)
    for k, depth in enumerate((0, 1, 3, 7, 15, 31, 63, 90)):
        if depth:
            engine.rollout_random(st[bounds[k]:bounds[k + 1]], depth)
    idx = sample(n)
    for rnd in range(8):
        masks = engine.legal_mask(st)
        acts = torch.from_numpy(pick_actions(masks.cpu().numpy().view(np.uint32), n, rnd)).to(dev)
        before = st.clone()
        ref = st.clone()
        r_ref = torch.empty(n, dtype=torch.int8, device=dev)
        d_ref, e_ref = (torch.empty(n, dtype=torch.uint8, device=dev) for _ in range(2))
        m_ref = torch.empty((n, MASK_WORDS), dtype=torch.int32, device=dev)
        with options(engine):
            for lo in range(0, n, 4096):
                hi = min(n, lo + 4096)
                engine.step(ref[lo:hi], acts[lo:hi], r_ref[lo:hi], d_ref[lo:hi], e_ref[lo:hi], m_ref[lo:hi])
        nm = torch.empty((n, MASK_WORDS), dtype=torch.int32, device=dev)
        with options(engine, **forced) as opt:
            reward, done, err = run_checked(engine, "step", n, opt, lambda: engine.step(st, acts, next_masks=nm),
                                            lambda: engine.step(before.clone(), acts, next_masks=torch.empty_like(nm)))
        for name, got, want in (("records", st, ref), ("reward", reward, r_ref), ("done", done, d_ref), ("err", err, e_ref),
                                ("next masks", nm, m_ref)):
            assert torch.equal(got, want), "round %d: %s differ from the chunked warp-engine step" % (rnd, name)
        pre, post, a = before[idx].cpu().numpy(), st[idx].cpu().numpy(), acts[idx].cpu().numpy()
        r, d, e, m = (t[idx].cpu().numpy() for t in (reward, done, err, nm))
        for j, i in enumerate(idx):
            if not _alive(pre[j]):
                continue
            h = pre[j].copy()
            oracle.step(h, int(a[j]))
            assert h.tobytes() == post[j].tobytes(), (rnd, i, int(a[j]))
            assert (int(r[j]), int(d[j]), int(e[j])) == ((h[19] >> 1) & 1, h[19] & 1, h[18]), (rnd, i)
            assert np.array_equal(oracle.legal_mask(h), m[j].view(np.uint32)), (rnd, i)


# ---------------------------------------------------------------- (e) record queries past one persistent wave
@pytest.fixture(scope="module")
def records(engine):
    """1,000,003 distinct records: reset + random rollouts of 0..400 steps, finished games among them; every 100th game
    holds one of UP01-03, which have no observation id (SB_ERR_OBS_ID); every 997th game then plays action 64 (the spell
    of hand slot 0), which sets err (SB_ERR_INDEX) where that card is not a spell"""
    n = 1000003
    dev = engine.device
    decks, factions = _default_deck_arrays(n)
    up = np.arange(0, n, 100)
    decks[up, up % 2, up % 12] = np.array([CARD_INDEX["UP01"], CARD_INDEX["UP02"], CARD_INDEX["UP03"]], dtype=np.uint8)[(up // 100) % 3]
    with options(engine):
        st = engine.reset(torch.arange(n, dtype=torch.int64, device=dev) + 3000000, torch.from_numpy(decks).to(dev),
                          torch.from_numpy(factions).to(dev))
        bounds = np.linspace(0, n, 9).astype(int)
        for k, depth in enumerate((0, 1, 3, 8, 20, 50, 120, 400)):
            if depth:
                engine.rollout_random(st[bounds[k]:bounds[k + 1]], depth)
        bad = torch.arange(5, n, 997, device=dev)
        sub = st[bad]
        engine.step(sub, torch.full((sub.shape[0],), 64, dtype=torch.uint8, device=dev))
        st[bad] = sub
    assert int((st[:, 19] & 1).sum()) > 1000 and int((st[:, 18] != 0).sum()) > 0
    yield st
    del st
    torch.cuda.empty_cache()


def test_queries_past_one_wave(engine, oracle, records):
    """legal_mask / observe / features at one persistent wave of kw_stream, one record past it, both sides of the features
    engine switch and 1 M records, against the other engine (forced) on the whole batch and the oracle on a sample"""
    sm = engine.sm_count
    big = records.shape[0]
    with options(engine, engine=0):  # thread engine: unpack + query
        t_mask = engine.legal_mask(records)
        t_obs, t_oerr = engine.observe(records)
        t_feat, t_ferr = engine.features(records)
    with options(engine, engine=1):  # warp engine: streams the packed record
        w_feat, w_ferr = engine.features(records)
    assert torch.equal(t_feat.view(torch.int64), w_feat.view(torch.int64)) and torch.equal(t_ferr, w_ferr)
    del w_feat, w_ferr
    assert int((t_oerr != 0).sum()) > big // 400, "the observation error path did not run"
    with options(engine) as opt:
        for n in (64 * sm, 64 * sm + 1, 65536, 65537, big):
            sub = records[:n]
            m = run_checked(engine, "legal_mask", n, opt, lambda: engine.legal_mask(sub), lambda: engine.legal_mask(sub))
            assert torch.equal(m, t_mask[:n]), n
            o, oe = run_checked(engine, "observe", n, opt, lambda: engine.observe(sub), lambda: engine.observe(sub))
            assert torch.equal(o, t_obs[:n]) and torch.equal(oe, t_oerr[:n]), n
            del o, oe
            f, fe = run_checked(engine, "features", n, opt, lambda: engine.features(sub), lambda: engine.features(sub))
            assert torch.equal(f.view(torch.int64), t_feat[:n].view(torch.int64)) and torch.equal(fe, t_ferr[:n]), n
    idx = np.unique(np.concatenate([sample(n) for n in (64 * sm, 64 * sm + 1, 65536, 65537, big)]))
    it = torch.from_numpy(idx).to(engine.device)
    host, mask, obs, oerr, feat, ferr = (t[it].cpu().numpy() for t in (records, t_mask, t_obs, t_oerr, t_feat, t_ferr))
    for j, i in enumerate(idx):
        assert np.array_equal(oracle.legal_mask(host[j]), mask[j].view(np.uint32)), i
        o, e = oracle.observe(host[j])
        assert np.array_equal(o, obs[j]) and e == int(oerr[j]), i
        f, e = oracle.features(host[j])
        assert np.array_equal(f.view(np.int64), feat[j].view(np.int64)) and e == int(ferr[j]), i


def test_expert_action_variants(engine, oracle, records):
    """kw_query at its largest default batch, k_expert_action one record later, and kw_query's grid-stride loop (forced);
    actions and the records (stream position) against the other engine and the oracle"""
    sm = engine.sm_count
    for n, forced in ((16384, {}), (16385, {}), (max(40000, 256 * sm + 1), {"engine": 1})):
        base = records[:n]
        with options(engine, **forced) as opt:
            st = base.clone()
            acts = run_checked(engine, "expert_action", n, opt, lambda: engine.expert_action(st),
                               lambda: engine.expert_action(base.clone()))
            other = 0 if _warp_engine("expert_action", n, sm, opt) else 1
        with options(engine, engine=other):
            st_o = base.clone()
            acts_o = engine.expert_action(st_o)
        assert torch.equal(acts, acts_o) and torch.equal(st, st_o), n
        idx = sample(n)
        it = torch.from_numpy(idx).to(engine.device)
        pre, post, a = base[it].cpu().numpy(), st[it].cpu().numpy(), acts[it].cpu().numpy()
        for j, i in enumerate(idx):
            if not _alive(pre[j]):
                continue
            h = pre[j].copy()
            assert oracle.expert_action(h) == int(a[j]) and h.tobytes() == post[j].tobytes(), (n, i)


def test_select_action_grid_stride(engine, oracle, records):
    """kw_select_action past one grid (forced): actions and scores exactly equal to the thread engine's and the oracle's
    (both engines and the oracle evaluate the same operations in the same order)"""
    sm = engine.sm_count
    n = max(20000, 4 * 32 * sm + 1)
    sub = records[:n]
    w = torch.from_numpy(np.random.RandomState(21).uniform(0, 1, (n, 10))).to(engine.device)
    with options(engine, engine=1) as opt:
        acts, scores = run_checked(engine, "select_action", n, opt, lambda: engine.select_action(sub, w, want_scores=True),
                                   lambda: engine.select_action(sub, w, want_scores=True))
    with options(engine, engine=0):
        acts_t, scores_t = engine.select_action(sub, w, want_scores=True)
    assert torch.equal(acts, acts_t)
    assert np.array_equal(scores.cpu().numpy(), scores_t.cpu().numpy(), equal_nan=True)
    idx = sample(n)
    it = torch.from_numpy(idx).to(engine.device)
    host, wn, a, sc = (t[it].cpu().numpy() for t in (sub, w, acts, scores))
    for j, i in enumerate(idx):
        if not _alive(host[j]):
            continue
        oa, osc, _m = oracle.select_action(host[j].copy(), wn[j])
        assert oa == int(a[j]) and np.array_equal(osc, sc[j], equal_nan=True), i


# ---------------------------------------------------------------- (f) host-buffer entry points
def test_host_buffer_entry_points(engine):
    """sb_rollout_random_host and sb_step_host give the bytes of the device calls; the staging buffer grows (4,096 ->
    262,144) and is reused for a smaller batch (1,000)"""
    dev = engine.device
    with options(engine) as opt:
        for n in (4096, 262144, 1000):
            seeds = np.arange(n, dtype=np.uint64) * np.uint64(7) + np.uint64(123457 + n)
            for want_chain in (True, False):
                h_states, h_steps, h_chain = run_checked(
                    engine, "rollout_random", n, dict(opt, chain=want_chain),
                    lambda: engine.rollout_random_host(seeds, want_chain=want_chain),
                    lambda: engine.rollout_random_host(seeds, want_chain=want_chain))
                st = engine.reset(torch.from_numpy(seeds.view(np.int64)).to(dev))
                chain = torch.zeros(n, dtype=torch.int64, device=dev) if want_chain else None
                steps = engine.rollout_random(st, 400, chain=chain)
                assert np.array_equal(h_states, st.cpu().numpy()) and np.array_equal(h_steps, steps.cpu().numpy()), (n, want_chain)
                if want_chain:
                    assert np.array_equal(h_chain, chain.cpu().numpy().view(np.uint64)), n
            st = engine.reset(torch.from_numpy(seeds.view(np.int64)).to(dev))
            engine.rollout_random(st, 25)
            acts = pick_actions(engine.legal_mask(st).cpu().numpy().view(np.uint32), n, 99)
            for want_masks in (True, False):
                d_st = st.clone()
                nm = torch.empty((n, MASK_WORDS), dtype=torch.int32, device=dev) if want_masks else None
                r, d, e = engine.step(d_st, torch.from_numpy(acts).to(dev), next_masks=nm)
                h_st = st.cpu().numpy()
                hr, hd, he, hm = run_checked(engine, "step", n, opt, lambda: engine.step_host(h_st, acts, want_masks),
                                             lambda: engine.step_host(st.cpu().numpy(), acts, want_masks))
                assert np.array_equal(h_st, d_st.cpu().numpy()), (n, want_masks)
                assert np.array_equal(hr, r.cpu().numpy()) and np.array_equal(hd, d.cpu().numpy()) and np.array_equal(he, e.cpu().numpy())
                if want_masks:
                    assert np.array_equal(hm, nm.cpu().numpy().view(np.uint32)), n

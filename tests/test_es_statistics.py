"""The evolution-strategy operators (sb_es_* on the device, sbo_es_* in the oracle) at the edges of the ABI, and the
distributions they draw from, on the oracle (CPU) and on the device.

test_gpu_training.py checks the kernels against the oracle at three shapes with one seed whose high word is 0, and
es_operators.npz pins the oracle to the reference through a restatement of the same normal sampler.  So a wrong sampler
shared by both, or a key that drops its high word in both, would pass there.  Here the draws are tested against the
distributions WeightVector.mutate and Population.select_from_combined specify, and the seed's high word must change the
draws.  Every statistical test runs on fixed seeds, so it is deterministic; the p-values of those seeds are recorded
beside each test (the device's draws are the oracle's bit for bit, so they hold on both backends), and a test asserts
p > 1e-3.
"""
import numpy as np
import pytest
from scipy import stats

P_MIN = 1e-3
SEED = 0xDEADBEEF00000007
SEEDS = (SEED, (1 << 64) - 1)
GENERATIONS = (0, 0xFFFFFFFF)


class OracleES:
    """the four operators on host arrays, in place, as sb_oracle states them"""

    def __init__(self, oracle):
        self.o = oracle

    def offspring(self, seed, gen, mu, lam, tau, tau_prime, min_sigma, w, s):
        return self.o.es_offspring(seed, gen, mu, lam, tau, tau_prime, min_sigma, w, s)

    def select(self, mu, fitness, w, s):
        return self.o.es_select(mu, fitness, w, s)

    def reset_sigmas(self, seed, gen, initial_sigma, s):
        self.o.es_reset_sigmas(seed, gen, initial_sigma, s)

    def inject(self, seed, gen, tau, tau_prime, min_sigma, initial_sigma, w, s):
        return self.o.es_inject_diversity(seed, gen, tau, tau_prime, min_sigma, initial_sigma, w, s)


class DeviceES:
    """the same operators through the library's kernels: host arrays in, results copied back into them"""

    def __init__(self, engine):
        import torch
        self.torch, self.e = torch, engine

    def _dev(self, a):
        return self.torch.from_numpy(np.ascontiguousarray(a)).to(self.e.device)

    def offspring(self, seed, gen, mu, lam, tau, tau_prime, min_sigma, w, s):
        dw, ds = self._dev(w), self._dev(s)
        parents = self.torch.empty(lam, dtype=self.torch.int32, device=self.e.device)
        self.e.es_offspring(seed, gen, mu, lam, tau, tau_prime, min_sigma, dw, ds, parents)
        w[...], s[...] = dw.cpu().numpy(), ds.cpu().numpy()
        return parents.cpu().numpy()

    def select(self, mu, fitness, w, s):
        out = self.e.es_select(mu, fitness, self._dev(w), self._dev(s), want_order=True)
        return tuple(t.cpu().numpy() for t in out)

    def reset_sigmas(self, seed, gen, initial_sigma, s):
        ds = self._dev(s)
        self.e.es_reset_sigmas(seed, gen, initial_sigma, ds)
        s[...] = ds.cpu().numpy()

    def inject(self, seed, gen, tau, tau_prime, min_sigma, initial_sigma, w, s):
        dw, ds = self._dev(w), self._dev(s)
        chosen = self.torch.empty(max(1, w.shape[0] // 2), dtype=self.torch.int32, device=self.e.device)
        self.e.es_inject_diversity(seed, gen, tau, tau_prime, min_sigma, initial_sigma, dw, ds, chosen)
        w[...], s[...] = dw.cpu().numpy(), ds.cpu().numpy()
        return chosen.cpu().numpy()


@pytest.fixture(params=["oracle", pytest.param("device", marks=pytest.mark.gpu)])
def es(request, oracle):
    return OracleES(oracle) if request.param == "oracle" else DeviceES(request.getfixturevalue("engine"))


def population(mu, lam, nf, seed):
    rs = np.random.RandomState(seed)
    w = np.concatenate([rs.uniform(0, 1, (mu, nf)), np.zeros((lam, nf))])
    s = np.concatenate([rs.uniform(1e-4, 0.3, (mu, nf)), np.zeros((lam, nf))])
    return w, s


# ---------------------------------------------------------------- edges of the ABI, the kernels against the oracle bit for bit
def same(a, b):
    return np.asarray(a).tobytes() == np.asarray(b).tobytes()


@pytest.mark.gpu
@pytest.mark.parametrize("mu,lam,nf", [(1, 1, 1), (1, 7, 64), (3, 5, 1), (13, 29, 64), (4096, 4096, 10), (4096, 1, 64)])
def test_kernels_equal_the_oracle_at_the_edges(engine, oracle, mu, lam, nf):
    dev, ref = DeviceES(engine), OracleES(oracle)
    for seed in SEEDS:
        for gen in GENERATIONS:
            w, s = population(mu, lam, nf, mu * 7 + lam + nf)
            W, S = w.copy(), s.copy()
            assert same(dev.offspring(seed, gen, mu, lam, 0.1, 0.01, 1e-5, w, s), ref.offspring(seed, gen, mu, lam, 0.1, 0.01, 1e-5, W, S))
            assert same(w, W) and same(s, S), (seed, gen)
            fitness = np.round(np.random.RandomState(gen & 0xFF).uniform(0, 1, mu + lam), 1)  # ties
            got, want = dev.select(mu, fitness, w, s), ref.select(mu, fitness, W, S)
            assert all(same(a, b) for a, b in zip(got, want)), (seed, gen)
            s2, S2 = got[1].copy(), want[1].copy()
            dev.reset_sigmas(seed, gen, 0.1, s2)
            ref.reset_sigmas(seed, gen, 0.1, S2)
            assert same(s2, S2)
            w2, W2 = got[0].copy(), want[0].copy()
            assert same(dev.inject(seed, gen, 0.1, 0.01, 1e-5, 0.1, w2, s2), ref.inject(seed, gen, 0.1, 0.01, 1e-5, 0.1, W2, S2))
            assert same(w2, W2) and same(s2, S2), (seed, gen)


def test_select_ties_signed_zeros_and_infinities(es):
    """top-mu by fitness descending, ties in original order (Python's stable sorted(..., reverse=True)); -0.0 == +0.0"""
    inf = float("inf")
    fitness = np.array([0.0, -0.0, inf, 0.5, -inf, 0.5, -0.0, inf, 0.0, -inf, 0.25, 0.5])
    total, nf = len(fitness), 3
    w = np.arange(total * nf, dtype=np.float64).reshape(total, nf)
    s = w + 0.5
    want = sorted(range(total), key=lambda i: fitness[i], reverse=True)
    for mu in (1, 5, total):
        wo, so, fo, order = es.select(mu, fitness, w, s)
        assert order.tolist() == want[:mu]
        assert same(fo, fitness[want[:mu]]) and same(wo, w[want[:mu]]) and same(so, s[want[:mu]])


@pytest.mark.gpu
@pytest.mark.parametrize("mu", [1, 3, 13, 4096])
def test_inject_diversity_equals_the_oracle(engine, oracle, mu):
    """one CTA of 256 threads: at mu = 4,096 the 2,048 chosen rows take eight passes"""
    nf = 10
    for seed in SEEDS:
        w, s = population(mu, 0, nf, mu)
        W, S = w.copy(), s.copy()
        chosen = DeviceES(engine).inject(seed, 5, 0.1, 0.01, 1e-5, 0.1, w, s)
        assert same(chosen, OracleES(oracle).inject(seed, 5, 0.1, 0.01, 1e-5, 0.1, W, S))
        assert same(w, W) and same(s, S)
        k = max(1, mu // 2)
        assert len(set(chosen.tolist())) == k and chosen.min() >= 0 and chosen.max() < mu
        changed = np.flatnonzero((w != population(mu, 0, nf, mu)[0]).any(1))
        assert set(changed.tolist()) <= set(chosen.tolist()) and len(changed) > 0.9 * k


def test_the_seed_high_word_keys_every_stream(es):
    """Philox's key is (seed low word, seed high word): seeds that differ only in the high word must draw differently"""
    mu, lam, nf = 37, 64, 8
    a, b = 0x0000000100000007, 0x0000000200000007
    outs = []
    for seed in (a, b):
        w, s = population(mu, lam, nf, 1)
        parents = es.offspring(seed, 3, mu, lam, 0.1, 0.01, 1e-5, w, s)
        r = s[:mu].copy()
        es.reset_sigmas(seed, 3, 0.1, r)
        chosen = es.inject(seed, 3, 0.1, 0.01, 1e-5, 0.1, w[:mu].copy(), s[:mu].copy())
        outs.append((parents, w[mu:], r, chosen))
    (pa, ca, ra, xa), (pb, cb, rb, xb) = outs
    assert not np.array_equal(pa, pb) and not np.array_equal(ca, cb) and not np.array_equal(ra, rb) and not np.array_equal(xa, xb)


# ---------------------------------------------------------------- distributions
def mutation_normals(es, seed):
    """tau = tau' = 0 keeps sigma, so each child's (w - 0.5) / sigma is the mutation's normal draw (parents at 0.5), to about
    1e-12: 0.5 + sigma z rounds to a multiple of 2^-54, an error of 2^-42 in z"""
    mu, lam, nf, sig = 37, 4096, 64, 2.0 ** -12
    w, s = np.zeros((mu + lam, nf)), np.zeros((mu + lam, nf))
    w[:mu], s[:mu] = 0.5, sig
    parents = es.offspring(seed, 3, mu, lam, 0.0, 0.0, 1e-300, w, s)
    assert np.all(s[mu:] == sig)
    return ((w[mu:] - 0.5) / sig).ravel(), parents


def test_mutation_normals_are_standard_normal(es):
    # seed 0xDEADBEEF00000007, 262,144 draws: KS p = 0.77; variance 1.00016, p = 0.95; |z| > 3: 725 draws, p = 0.51;
    # |z| > 4: 10 draws, p = 0.11
    z, _parents = mutation_normals(es, SEED)
    assert stats.kstest(z, "norm").pvalue > P_MIN
    n = z.size
    # the variance of n standard normals: (n - 1) s^2 is chi-square with n - 1 degrees of freedom
    chi = (n - 1) * z.var(ddof=1)
    assert min(stats.chi2.cdf(chi, n - 1), stats.chi2.sf(chi, n - 1)) * 2 > P_MIN
    for t in (3.0, 4.0):
        k = int((np.abs(z) > t).sum())
        assert stats.binomtest(k, n, 2 * stats.norm.sf(t)).pvalue > P_MIN, (t, k)


def test_parent_choice_is_uniform(es):
    # mu 37, lambda 4,096, seed 0xDEADBEEF00000007: chi-square p = 0.56
    _z, parents = mutation_normals(es, SEED)
    assert parents.min() >= 0 and parents.max() < 37
    assert stats.chisquare(np.bincount(parents, minlength=37)).pvalue > P_MIN


def test_sigma_update_is_log_normal(es):
    """sigma' = sigma exp(tau' g + tau n_i): with tau' = 0 the log ratio / tau is an iid N(0, 1) per feature; with tau = 0
    it is one N(0, 1) per row, the same in every feature of the row"""
    # seed 12345: KS p = 0.62 (per feature, 262,144 values), 0.24 (per row, 4,096 values)
    mu, lam, nf, sig = 37, 4096, 64, 0.01
    for tau, tau_prime in ((0.1, 0.0), (0.0, 0.1)):
        w, s = np.full((mu + lam, nf), 0.5), np.full((mu + lam, nf), sig)
        es.offspring(12345, 4, mu, lam, tau, tau_prime, 1e-300, w, s)
        r = np.log(s[mu:] / sig) / (tau + tau_prime)
        if tau_prime:
            assert np.allclose(r, r[:, :1], rtol=0, atol=1e-12)
            r = r[:, 0]
        assert stats.kstest(r.ravel(), "norm").pvalue > P_MIN, (tau, tau_prime)


def test_reset_sigmas_are_uniform(es):
    # seed 0xDEADBEEF00000007, 1,024 x 64 values: KS p = 0.35
    sigma0 = 0.1
    s = np.zeros((1024, 64))
    es.reset_sigmas(SEED, 9, sigma0, s)
    assert s.min() >= 0.5 * sigma0 and s.max() < 1.5 * sigma0
    assert stats.kstest(s.ravel(), "uniform", args=(0.5 * sigma0, sigma0)).pvalue > P_MIN


def test_inject_diversity_chooses_uniformly(es):
    """choice(mu, mu // 2, replace=False): over 2,000 generations at mu = 37 every row is chosen with frequency 18 / 37.

    Each generation draws k = 18 distinct rows, so a row's count has variance G p (1 - p) and the counts are negatively
    correlated; Pearson's statistic is then (mu - k) / (mu - 1) times chi-square(mu - 1), not chi-square(mu - 1), and is
    rescaled before the test.  Uncorrected it would pass a shuffle as biased as Sattolo's (j drawn below i instead of i + 1)."""
    # seed 0xDEADBEEF00000007, generations 0..1999: corrected chi-square p = 0.73
    mu, k, gens = 37, 18, 2000
    w, s = np.full((mu, 1), 0.5), np.full((mu, 1), 0.1)
    counts = np.zeros(mu, dtype=np.int64)
    for gen in range(gens):
        chosen = es.inject(SEED, gen, 0.1, 0.01, 1e-5, 0.1, w, s)
        assert len(chosen) == k and len(set(chosen.tolist())) == k and chosen.min() >= 0 and chosen.max() < mu
        counts += np.bincount(chosen, minlength=mu)
    expected = gens * k / mu
    statistic = ((counts - expected) ** 2 / expected).sum() * (mu - 1) / (mu - k)
    assert stats.chi2.sf(statistic, mu - 1) > P_MIN

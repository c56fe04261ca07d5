"""The library's deterministic log and exp (device es_log / es_exp in sb_es.cuh, the oracle's sbo_det_log / sbo_det_exp)
against the exact values, computed with decimal at 60 digits, and the device functions against the oracle bit for bit.

The other tests compare these functions only with restatements that share their arithmetic (the oracle, ref_harness,
sb_gumbel_model), so a truncated series or a missing ln2 correction would pass there.  Errors are in ulps of the exact
value.  Inputs: for log every f32 binade (subnormals included: es_log takes every f32 prior), log-uniform doubles over the
normal range, the region near 1 and the branch points; for exp the range the Gumbel softmax uses ([-700, 0]), the range of
the mutation step ([-20, 20]), the region near 0 and the points where the reduction's k changes.
"""
import ctypes
import math
import os
import subprocess
from decimal import Decimal, getcontext

import numpy as np
import pytest

import ref_harness

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HERE = os.path.dirname(os.path.abspath(__file__))

# Measured maxima of the oracle over the inputs below (the device equals it bit for bit): log 2.71 ulp at x = 1.000948, where
# log x is small and the result is the series term alone; exp 1.09 ulp at y = 91.842.  The bounds leave about one ulp of room.
LOG_MAX_ULP = 4.0
EXP_MAX_ULP = 2.0
F32_TINY = 2.0 ** -126


def _f32_bits(bits):
    return np.asarray(bits, dtype=np.uint32).view(np.float32).astype(np.float64)


def log_inputs():
    rng = np.random.default_rng(20261021)
    xs = []
    # every f32 binade [2^e, 2^(e+1)), e = -149 .. 127, with random mantissas (the subnormal binades hold 2^(e+149) values)
    for e in range(-149, 128):
        if e < -126:
            lo = 1 << (e + 149)
            xs.append(_f32_bits(rng.integers(lo, 2 * lo, size=min(lo, 40))))
        else:
            xs.append(_f32_bits(((e + 127) << 23) | rng.integers(0, 1 << 23, size=40)))
    xs.append(np.exp2(rng.uniform(-1022.0, 1024.0, size=8000)))  # log-uniform doubles over the normal range
    xs.append(1.0 + rng.uniform(-1e-3, 1e-3, size=4000))
    half = math.sqrt(0.5)
    branch = [half, 1.0 - 2.0 ** -53, 1.0 + 2.0 ** -52, F32_TINY, 1.0 - 2.0 ** -24, 1.0 + 2.0 ** -23]
    for k in (1, 2):
        branch += [half - k * math.ulp(half), half + k * math.ulp(half)]
    branch += [2.0 ** e for e in range(-1022, 1024)]
    branch += [math.nextafter(2.0 ** e, 0.0) for e in range(-1021, 1024)]
    xs.append(np.array(branch))
    return np.concatenate(xs)


def exp_inputs():
    rng = np.random.default_rng(1021)
    ys = [rng.uniform(-700.0, 0.0, size=8000), rng.uniform(-20.0, 20.0, size=8000), rng.uniform(-1e-6, 1e-6, size=2000)]
    # odd multiples of ln2 / 2, where the rounding of y / ln2 to k changes, +- 3 ulp
    mid = (2.0 * np.arange(-1010, 1010) + 1.0) * (math.log(2.0) / 2.0)
    mid = mid[np.abs(mid) < 700.0]
    for k in range(-3, 4):
        ys.append(mid + k * np.spacing(mid))
    ys.append(np.array([-700.0, 0.0, 2.0 ** -60, -(2.0 ** -60)]))
    return np.concatenate(ys)


def _ulp_errors(got, xs, exact):
    getcontext().prec = 60
    err = np.empty(len(xs))
    for i, (g, x) in enumerate(zip(got.tolist(), xs.tolist())):
        ex = exact(Decimal(x))
        err[i] = float(abs(Decimal(g) - ex) / Decimal(math.ulp(float(ex))))
    return err


def _oracle(fn, xs):
    return np.array([fn(float(x)) for x in xs])


def test_inputs_cover_the_issue_points():
    xs = log_inputs()
    f32 = xs[(xs >= 2.0 ** -149) & (xs < 2.0 ** 128)]
    assert 2.0 ** -149 in xs and F32_TINY in xs and (1.0 - 2.0 ** -53) in xs and (1.0 + 2.0 ** -52) in xs
    assert len(np.unique(np.frexp(f32)[1])) == 277  # every f32 binade
    assert -700.0 in exp_inputs() and np.abs(exp_inputs()).max() <= 700.0


def test_det_log_within_bound_of_exact(oracle):
    xs = log_inputs()
    got = _oracle(oracle.lib().sbo_det_log, xs)
    one = xs == 1.0
    assert np.all(got[one] == 0.0)
    err = _ulp_errors(got[~one], xs[~one], lambda d: d.ln())
    worst = int(np.argmax(err))
    assert err[worst] <= LOG_MAX_ULP, "sbo_det_log(%r): %.3f ulp" % (xs[~one][worst], err[worst])


def test_det_exp_within_bound_of_exact(oracle):
    ys = exp_inputs()
    got = _oracle(oracle.lib().sbo_det_exp, ys)
    err = _ulp_errors(got, ys, lambda d: d.exp())
    worst = int(np.argmax(err))
    assert err[worst] <= EXP_MAX_ULP, "sbo_det_exp(%r): %.3f ulp" % (ys[worst], err[worst])


def test_ref_harness_det_log_is_the_oracle_bit_for_bit(oracle):
    """oracle/ref_harness.py drives the reference's Population with det_log in the Marsaglia normal (es_operators.npz)"""
    xs = log_inputs()
    want = _oracle(oracle.lib().sbo_det_log, xs)
    got = np.array([ref_harness.det_log(float(x)) for x in xs])
    assert got.tobytes() == want.tobytes()


def build_probe(tmp):
    from monsoon_b200.build import CSRC, NVCC_FLAGS
    so = os.path.join(str(tmp), "libes_math_probe.so")
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    subprocess.check_call([nvcc] + NVCC_FLAGS + ["-I", CSRC, "-o", so, os.path.join(HERE, "es_math_probe.cu")], cwd=str(tmp))
    lib = ctypes.CDLL(so)
    lib.es_math_probe.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]
    lib.es_math_probe.restype = ctypes.c_int
    return lib


@pytest.mark.gpu
def test_device_log_and_exp_equal_the_oracle_bit_for_bit(engine, oracle, tmp_path):
    probe = build_probe(tmp_path)
    for op, xs, fn in ((0, log_inputs(), oracle.lib().sbo_det_log), (1, exp_inputs(), oracle.lib().sbo_det_exp)):
        x = np.ascontiguousarray(xs, dtype=np.float64)
        y = np.zeros_like(x)
        assert probe.es_math_probe(len(x), op, x.ctypes.data, y.ctypes.data) == 0
        want = _oracle(fn, x)
        bad = np.flatnonzero(y.view(np.uint64) != want.view(np.uint64))
        assert bad.size == 0, (op, x[bad[:5]], y[bad[:5]], want[bad[:5]])

"""Shared by tests/test_random_edges.py (CPU) and tests/test_gpu_random_edges.py (GPU): the reference's draws of cmb_random_* at
its edge parameters (tests/golden/random_edges.json, written by tests/golden/make_random_edges.py) and the high-precision
bracket for the kinds whose variate is itself a log or pow result.

Excluded, on purpose (also in the header of cimba_b200/csrc/distributions.cuh):
* geometric with p = 0, or with p so small that the count exceeds 2^32 (and the negative binomial built on it): the reference
  converts an out-of-range double to unsigned, which C leaves undefined - x86 wraps where sm_100 saturates;
* hyper-exponential and loaded dice whose probabilities sum to less than 1: the reference indexes past its table."""
import json
import sys
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
sys.path.insert(0, str(HERE / "golden"))
from make_random_edges import digest, draws  # noqa: E402,F401

FIXTURE = json.loads((HERE / "golden/random_edges.json").read_text())
RECORDS = FIXTURE["cases"]

EXCLUDED = [
    ("geometric, p = 0", "-log(1 - 0) = 0: the count is inf, converted to unsigned - undefined in C (x86 wraps, sm_100 saturates)"),
    ("geometric, p < ~1e-9", "counts beyond 2^32 converted to unsigned - undefined in C (x86 wraps, sm_100 saturates)"),
    ("negative binomial / pascal on such a geometric", "the same conversion, summed"),
    ("hyper-exponential with probabilities summing to < 1", "the reference reads the mean past the end of its table"),
    ("loaded dice with probabilities summing to < 1", "returns n, one past the last outcome, in the reference"),
]

# the variate IS a libm result: log (logistic) or pow (weibull, pareto) of an argument formed from one stream's draw
BRACKETED = {11: "log", 18: "pow", 19: "pow"}


def params_of(rec):
    return [float.fromhex(p) for p in rec["params"]]


def rec_id(rec):
    return f"k{rec['kind']}-" + "_".join(f"{v:.3g}" for v in params_of(rec)) + f"-s{rec['seed'] & 0xffff:04x}"


def gamma_pow_kind(kind, p):
    """Kinds whose variate goes through rnd_gamma's pow(u, 1 / shape) (shape < 1), interleaved with other draws."""
    return ((kind == 15 and p[0] < 1.0) or (kind == 20 and p[0] < 2.0) or (kind == 21 and min(p[0], p[1]) < 2.0)
            or (kind == 22 and p[2] < 2.0))


def same(a, b):
    """Bit for bit, with every NaN equal to every NaN."""
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    na, nb = np.isnan(a), np.isnan(b)
    return (na == nb) & (na | (a.view(np.uint64) == b.view(np.uint64)))


def check_first8_and_digest(values, rec, what):
    want = np.array([float.fromhex(h) for h in rec["first8"]])
    ok = same(values[:8], want)
    assert ok.all(), (what, rec_id(rec), values[:8][~ok], want[~ok])
    assert digest(values) == rec["sha256"], (what, rec_id(rec))


def ulp_distance(a, b):
    """How many doubles lie between a and b (NaN vs NaN = 0, NaN vs number = huge)."""
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)

    def ordered(x):                                     # exact integers: a float64 difference would round to 2^10 steps
        i = np.ascontiguousarray(x).view(np.int64)
        return np.where(i < 0, np.int64(-2**63) - i, i).tolist()
    d = np.array([abs(x - y) for x, y in zip(ordered(a), ordered(b))], dtype=np.float64)
    na, nb = np.isnan(a), np.isnan(b)
    return np.where(na & nb, 0.0, np.where(na | nb, np.inf, d))


def _neighbours(t, k):
    """The doubles within k ulp of the real number t (an mpmath mpf): round to nearest, then k steps either way."""
    import mpmath
    if mpmath.isinf(t):
        return {float(t)}
    if t == 0:
        return {0.0, -0.0}
    d = float(t)
    out = {d}
    lo = hi = d
    for _ in range(k):
        lo, hi = float(np.nextafter(lo, -np.inf)), float(np.nextafter(hi, np.inf))
        out |= {lo, hi}
    return out


def bracket_violations(kind, p, values, stream, k):
    """Indices where `values` (kind 11, 18 or 19 with params p) is not the formula of distributions.cuh evaluated with some libm
    result within k ulp of the exact log / pow of the argument formed, with the same double operations, from `stream` - uniform01
    (kind 3) for logistic and pareto, exponential(1) (kind 1) for weibull, at the same seed."""
    import mpmath
    mpmath.mp.prec = 256
    bad = []
    for i, (v, x) in enumerate(zip(np.asarray(values, dtype=np.float64).tolist(), np.asarray(stream, dtype=np.float64).tolist())):
        if kind == 11:                                  # m + s * log(x / (1.0 - x))
            m, s = p
            arg = x / (1.0 - x)
            libm = _neighbours(mpmath.log(mpmath.mpf(arg)) if arg > 0 else mpmath.ninf, k)
            cands = {m + s * L for L in libm}
        elif kind == 18:                                # scale * pow(u, 1.0 / shape)
            shape, scale = p
            e = 1.0 / shape
            libm = _neighbours(mpmath.power(mpmath.mpf(x), mpmath.mpf(e)), k)
            cands = {scale * L for L in libm}
        else:                                           # mode / pow(u, 1.0 / shape)
            shape, mode = p
            e = 1.0 / shape
            libm = _neighbours(mpmath.power(mpmath.mpf(x), mpmath.mpf(e)), k)
            with np.errstate(divide="ignore", over="ignore", invalid="ignore"):
                cands = {float(np.float64(mode) / np.float64(L)) for L in libm}
        if not any((c == v) or (np.isnan(c) and np.isnan(v)) for c in cands):
            bad.append(i)
    return bad


def bracket_stream(lib, prefix, kind, seed, n):
    """The draws the variates of a bracketed kind consume, one per variate: uniform01 (kind 3) or exponential(1) (kind 1)."""
    if kind == 18:
        return draws(lib, prefix, seed, 1, [1.0, 0.0], n)
    return draws(lib, prefix, seed, 3, [0.0, 0.0], n)

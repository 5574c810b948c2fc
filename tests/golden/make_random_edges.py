"""What the UNMODIFIED reference build (oracle/_ref/librefdrv.so) draws for cmb_random_* at its edge parameters: the
domain's corners (lo == hi, p = 0 and 1, mode == min or max, a shape of exactly 1, one degree of freedom) and the results
that overflow, underflow to subnormals or come out NaN.

    make -C oracle ref && python tests/golden/make_random_edges.py      -> tests/golden/random_edges.json

Every case is drawn at two seeds, N variates each (a multiple of 64, so that the reference's coin-flip cache is empty
between calls).  A record holds the kind, its parameters, the seed, N, the first 8 values as hex and the SHA-256 of all N
as little-endian f64 with every NaN replaced by one pattern: x86 makes the NaN 0xfff8..., sm_100 0x7fff..., and a NaN is
compared as a NaN, not by its bits.  Kinds 1..8 go through ref_rng_draws(p0, p1), 9..33 through ref_rng_draws_ex(params).

Running it again writes the same file byte for byte."""
import hashlib
import json
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT / "tests"))
from oracle_libs import load_ref, rng_draws, rng_draws_ex  # noqa: E402

SEEDS = [0x34F05C64D7AD598F, 0x0123456789ABCDEF]
N = 65_536
CANONICAL_NAN = 0x7FF8000000000000

# kind, params.  Kinds 1..8 take (p0, p1).
CASES = [
    (1, [5e-324, 0.0]), (1, [1e-300, 0.0]), (1, [1e300, 0.0]),
    (4, [0.0, 0.0]), (4, [1.0, -2.0]), (4, [1e16, 1.0]),
    (5, [1, 1.5]), (5, [64, 0.25]),
    (6, [2.0, 2.0]), (6, [3.0, -1.0]), (6, [-1e308, 1e308]),
    (7, [5, 5]), (7, [-2.0**61, 2.0**61 - 1024]),
    (8, [0.0, 0.0]), (8, [1.0, 0.0]), (8, [1e-18, 0.0]),
    (9, [1.0, 1.0, 3.0]), (9, [1.0, 3.0, 3.0]),
    (10, [0.5, 0.0]), (10, [710.0, 1.0]), (10, [-740.0, 1.0]),
    (11, [1.0, -2.0]), (11, [1e6, 1.5]),
    (18, [0.1, 1.0]), (18, [1.0, 2.0]), (18, [50.0, 1.0]),
    (19, [0.1, 1.0]), (19, [1e3, 2.0]),
    (15, [1.0, 1.0]), (15, [1.0 - 2.0**-53, 1.0]), (15, [0.05, 1.0]), (15, [1e3, 1.0]), (15, [2.5, 1e-300]),
    (31, [1.0]), (31, [1.0 - 2.0**-53]), (31, [0.05]), (31, [1e3]),
    (16, [1.0, 1.0, 0.0, 1.0]), (16, [0.5, 2.0, 0.0, 1.0]),
    (17, [0.0, 0.0, 1.0]), (17, [0.0, 1.0, 1.0]),
    (32, [0.0, 0.0, 1.0, 4.0]), (32, [0.0, 1.0, 1.0, 4.0]), (32, [0.0, 0.3, 1.0, 0.0]),
    (20, [1.0]), (20, [2.0]), (20, [1e4]), (20, [0.02]),
    (21, [1.0, 1.0]), (21, [2.0, 1e4]),
    (22, [0.0, 1.0, 1.0]), (22, [0.0, 1.0, 2.0]), (22, [0.0, 1.0, 0.02]),
    (23, [0.0]), (12, [0.0, 0.0]), (12, [1.0, 0.0]),
    (25, [1.0]), (25, [0.5]), (25, [1e-6]),
    (26, [0, 0.5]), (26, [10, 1.0]), (26, [10, 0.5]), (26, [10, 1e-6]),
    (27, [0, 0.5]), (27, [3, 1.0]), (27, [3, 0.5]), (27, [2, 1e-6]),
    (33, [0, 0.5]), (33, [3, 1.0]), (33, [3, 0.5]),
    (28, [1e-3]), (28, [500.0]),
    (29, [1, 1.0]), (29, [3, 0.5, 0.0, 0.5]),
    (30, [1, 1.0]), (30, [3, 0.5, 0.0, 0.5]),
]


def digest(values) -> str:
    u = np.ascontiguousarray(values, dtype=np.float64).view(np.uint64).copy()
    u[np.isnan(np.asarray(values, dtype=np.float64))] = CANONICAL_NAN
    return hashlib.sha256(u.astype("<u8").tobytes()).hexdigest()


def draws(lib, prefix, seed, kind, params, n=N):
    if kind <= 8:
        return np.asarray(rng_draws(lib, prefix, seed, kind, float(params[0]), float(params[1]), n), dtype=np.float64)
    return np.asarray(rng_draws_ex(lib, prefix, seed, kind, params, n), dtype=np.float64)


def main():
    ref = load_ref()
    if ref is None:
        sys.exit("oracle/_ref/librefdrv.so is missing: make -C oracle ref")
    out = []
    for kind, params in CASES:
        for seed in SEEDS:
            v = draws(ref, "ref", seed, kind, params)
            out.append({"kind": kind, "params": [float(p).hex() for p in params], "seed": seed, "n": N,
                        "first8": [float(x).hex() for x in v[:8]], "sha256": digest(v)})
    path = ROOT / "tests/golden/random_edges.json"
    path.write_text(json.dumps({"n": N, "seeds": SEEDS, "canonical_nan": CANONICAL_NAN, "cases": out}, indent=1) + "\n")
    print("wrote", path, len(out), "records")


if __name__ == "__main__":
    main()

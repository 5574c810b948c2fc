"""Loaders for the two CPU checkers (test infrastructure; never imported by cimba_b200).

* ``load_port()``  - oracle/liboracle_port.so, the plain-C restatement
  (built on demand with gcc; travels to the GPU box as a prebuilt .so too).
* ``load_ref()``   - oracle/_ref/librefdrv.so, model drivers linked against the
  unmodified reference library.  Present wherever `make -C oracle ref` has run
  (needs /root/reference); returns None otherwise.

What the reference build returned for the runs the tests compare with is stored in
tests/golden/reference_runs.json (tests/golden/make_reference_runs.py), so the
comparisons hold wherever the suite runs.
"""
from __future__ import annotations

import ctypes as C
import hashlib
import json
import subprocess
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
ORACLE = ROOT / "oracle"
REFERENCE_RUNS = ROOT / "tests/golden/reference_runs.json"


def reference_runs():
    return json.loads(REFERENCE_RUNS.read_text())


def result_digest(rows):
    """SHA-256 of result rows as tests/golden/reference_runs.json records them: one line per row, integers as unsigned
    64-bit decimals, floating-point values (float32 widened exactly) as hex floats."""
    text = "\n".join(" ".join(float(v).hex() if isinstance(v, (float, np.floating)) else str(int(v) & (2**64 - 1)) for v in row)
                     for row in rows)
    return hashlib.sha256(text.encode()).hexdigest()


def trial_rows(results):
    """run_trials results as digest rows: events, objects, t_end, sum_wait, max_fel, max_queue, the eight counters."""
    return [(*r.key(), r.max_fel, r.max_queue, *r.counters()) for r in results]


class Result(C.Structure):
    _fields_ = [("events", C.c_uint64), ("objects", C.c_uint64), ("t_end", C.c_double),
                ("sum_wait", C.c_double), ("max_fel", C.c_uint64), ("max_queue", C.c_uint64),
                ("counter", C.c_uint64 * 8)]

    def key(self):
        return (self.events, self.objects, self.t_end, self.sum_wait)

    def counters(self):
        return list(self.counter)


_DP = C.POINTER(C.c_double)
_UP = C.POINTER(C.c_uint64)


def _bind(lib, prefix):
    run = getattr(lib, f"{prefix}_run_trials")
    run.restype = C.c_int
    run.argtypes = [C.c_int, C.c_int, C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint64,
                    C.c_double, C.c_double, C.c_int, C.POINTER(Result)]
    tr = getattr(lib, f"{prefix}_trace_trial")
    tr.restype = C.c_int
    tr.argtypes = [C.c_int, C.c_int, C.c_uint64, C.c_uint64, C.c_double, C.c_double,
                   C.c_uint64, _UP, _DP, C.POINTER(Result)]
    dr = getattr(lib, f"{prefix}_rng_draws")
    dr.restype = C.c_int
    dr.argtypes = [C.c_uint64, C.c_int, C.c_double, C.c_double, C.c_uint64, _DP]
    fm = getattr(lib, f"{prefix}_fmix64")
    fm.restype = C.c_uint64
    fm.argtypes = [C.c_uint64, C.c_uint64]
    for name, nargs in (("datasummary_of", 2), ("datasummary_split_merge", 3)):
        f = getattr(lib, f"{prefix}_{name}")
        f.restype = C.c_int
        f.argtypes = [_DP] + [C.c_uint64] * (nargs - 1) + [_DP]
    f = getattr(lib, f"{prefix}_wtdsummary_of")
    f.restype = C.c_int
    f.argtypes = [_DP, _DP, C.c_uint64, _DP]
    f = getattr(lib, f"{prefix}_wtdsummary_split_merge")
    f.restype = C.c_int
    f.argtypes = [_DP, _DP, C.c_uint64, C.c_uint64, _DP]
    return lib


def load_port():
    so = ORACLE / "liboracle_port.so"
    src = [ORACLE / "port/cimba_port.c", ORACLE / "port/awacs_port.c", ORACLE / "port/cimba_port.h",
           ORACLE / "port/zig_tables.h"]
    if not so.exists() or so.stat().st_mtime < max(p.stat().st_mtime for p in src):
        subprocess.run(["make", "-C", str(ORACLE), "port"], check=True, capture_output=True)
    lib = _bind(C.CDLL(str(so)), "port")
    lib.port_heap_script.restype = C.c_int
    lib.port_heap_script.argtypes = [C.c_uint64, C.POINTER(C.c_int), _DP,
                                     C.POINTER(C.c_int64), _UP]
    return lib


def load_ref():
    so = ORACLE / "_ref/librefdrv.so"
    if not so.exists():
        return None
    lib = _bind(C.CDLL(str(so)), "ref")
    lib.ref_cpu_cores.restype = C.c_int
    return lib


def trace_trial(lib, prefix, model, servers, seed, nobj, arr, srv, cap):
    r = Result()
    keys = (C.c_uint64 * max(cap, 1))()
    times = (C.c_double * max(cap, 1))()
    getattr(lib, f"{prefix}_trace_trial")(model, servers, seed, nobj, arr, srv, cap, keys, times, C.byref(r))
    n = min(cap, r.events)
    return r, list(keys)[:n], list(times)[:n]


def run_trials(lib, prefix, model, servers, master, first, count, nobj, arr, srv, par=0):
    res = (Result * count)()
    getattr(lib, f"{prefix}_run_trials")(model, servers, master, first, count, nobj, arr, srv, par, res)
    return res


def rng_draws(lib, prefix, seed, kind, p0, p1, n):
    out = np.empty(n, dtype=np.float64)
    rc = getattr(lib, f"{prefix}_rng_draws")(seed, kind, p0, p1, n, out.ctypes.data_as(_DP))
    assert rc == 0
    return out


# kinds 9..33 of *_rng_draws_ex: one parameter set per distribution (+ a few extra corners)
DIST_CASES = [
    (9, [1.0, 2.5, 7.0]), (10, [0.5, 0.75]), (11, [1.0, 2.0]), (12, [0.0, 1.5]), (13, [3, 0.5, 1.0, 2.0]),
    (14, [3, 0.5, 1.0, 4.0, 0.2, 0.5, 0.3]), (15, [2.5, 1.5]), (16, [2.0, 3.5, 1.0, 4.0]), (17, [1.0, 2.0, 6.0]),
    (18, [1.7, 2.0]), (19, [2.5, 1.0]), (20, [3.0]), (21, [4.0, 7.0]), (22, [1.0, 2.0, 5.0]), (23, [1.3]), (24, []),
    (25, [0.3]), (26, [12, 0.35]), (27, [4, 0.4]), (28, [3.5]), (29, [4, 0.1, 0.2, 0.3, 0.4]),
    (30, [5, 0.05, 0.25, 0.4, 0.1, 0.2]), (31, [4.2]), (32, [1.0, 2.0, 6.0, 2.5]), (33, [3, 0.6]),
    (15, [0.6, 2.0]), (20, [1.0]), (31, [1.0]), (9, [0.0, 0.0, 1.0]), (28, [0.2]),
]
# the variate IS a log / pow result: CUDA's libm vs glibc may differ in the last places (lognormal, kind 10, is an
# exp result and exact: csrc/glibc_exp.cuh restates glibc's exp)
DIST_LIBM_KINDS = {11, 18, 19}


def rng_draws_ex(lib, prefix, seed, kind, params, n):
    """n variates of kind 9..33 from {ref,port}_rng_draws_ex (n % 64 == 0 keeps the reference's
    thread-local coin-flip cache empty between calls)."""
    f = getattr(lib, f"{prefix}_rng_draws_ex")
    f.restype = C.c_int
    f.argtypes = [C.c_uint64, C.c_int, C.POINTER(C.c_double), C.c_uint32, C.c_uint64, C.POINTER(C.c_double)]
    out = (C.c_double * n)()
    par = (C.c_double * max(1, len(params)))(*[float(v) for v in params])
    rc = f(seed, kind, par, len(params), n, out)
    assert rc == 0, (prefix, kind, rc)
    return list(out)


# ---------------------------------------------------------------- AWACS (tutorial/tut_5_1.c, BASELINE config 5)
class AwacsOut(C.Structure):
    _fields_ = [("events", C.c_uint64), ("t_end", C.c_double), ("num_found", C.c_uint32), ("tds_count", C.c_uint32 * 6),
                ("mode_count", C.c_uint32 * 4), ("pad", C.c_uint32), ("sum_x", C.c_double), ("sum_y", C.c_double)]

    def key(self):
        return (self.events, self.t_end, self.num_found, list(self.tds_count), list(self.mode_count),
                self.sum_x, self.sum_y)

    def row(self):
        return (self.events, self.t_end, self.num_found, *self.tds_count, *self.mode_count, self.sum_x, self.sum_y)


AWACS_TARGETS = 1000
AWACS_TERRAIN_SEED = 0x34F05C64D7AD598F


def load_awacs_ref():
    """oracle/_ref/libawacs_ref.so = the UNMODIFIED tutorial source behind a stub hdf5.h; None when not built."""
    so = ORACLE / "_ref/libawacs_ref.so"
    if not so.exists():
        return None
    lib = C.CDLL(str(so))
    lib.awacs_ref_map.restype = C.POINTER(C.c_float)
    return lib


def awacs_terrain(lib, prefix, seed, width_nm, height_nm, threads=1):
    """(map float32 [rows*cols], cols, rows, geom[6]) from the reference build ('ref') or the port ('port');
    `threads` > 1 lets the port compute the noise part of the cells in parallel (same map)."""
    cols, rows, geom = C.c_uint32(), C.c_uint32(), (C.c_float * 6)()
    if prefix == "ref":
        lib.awacs_ref_terrain(C.c_uint64(seed), C.c_float(width_nm), C.c_float(height_nm), C.c_float(30.0),
                              C.c_float(-10.0), C.byref(cols), C.byref(rows), geom)
        n = cols.value * rows.value
        m = np.ctypeslib.as_array(lib.awacs_ref_map(), shape=(n,)).copy()
    else:
        lib.port_awacs_grid(C.c_float(width_nm), C.c_float(height_nm), C.byref(cols), C.byref(rows))
        m = np.empty(cols.value * rows.value, dtype=np.float32)
        lib.port_awacs_terrain_mt(C.c_uint64(seed), C.c_float(width_nm), C.c_float(height_nm), C.c_float(30.0),
                                  C.c_float(-10.0), m.ctypes.data_as(C.POINTER(C.c_float)), geom, None, C.c_int(threads))
    return m, cols.value, rows.value, np.array(list(geom), dtype=np.float32)


def awacs_trial(lib, prefix, seed, duration_h, terrain=None, trace_cap=0):
    """One trial: (AwacsOut, keys, times, per-target dict).  `terrain` = awacs_terrain(...) for the port; the
    reference build uses the terrain its last awacs_ref_terrain call made."""
    out = AwacsOut()
    keys = (C.c_uint64 * max(1, trace_cap))()
    times = (C.c_double * max(1, trace_cap))()
    x, y = (C.c_float * AWACS_TARGETS)(), (C.c_float * AWACS_TARGETS)()
    mode, tds, det = (C.c_int * AWACS_TARGETS)(), (C.c_int * AWACS_TARGETS)(), (C.c_int * AWACS_TARGETS)()
    if prefix == "ref":
        rc = lib.awacs_ref_trial(C.c_uint64(seed), C.c_double(duration_h), C.c_uint64(trace_cap), keys, times,
                                 C.byref(out), x, y, mode, tds, det)
    else:
        m, cols, rows, geom = terrain
        rc = lib.port_awacs_trial(C.c_uint64(seed), C.c_double(duration_h), m.ctypes.data_as(C.POINTER(C.c_float)),
                                  C.c_uint32(cols), C.c_uint32(rows), geom.ctypes.data_as(C.POINTER(C.c_float)),
                                  C.c_uint64(trace_cap), keys, times, C.byref(out), x, y, mode, tds, det)
    assert rc == 0
    n = min(trace_cap, out.events)
    per = dict(x=np.array(x[:], dtype=np.float32), y=np.array(y[:], dtype=np.float32), mode=list(mode), tds=list(tds),
               detected=list(det))
    return out, list(keys)[:n], list(times)[:n], per


def awacs_ref_experiment(lib, master_seed, first, count, duration_h):
    """`count` trials of the unmodified tutorial model through the reference's own cimba_run_experiment (all host
    cores), seeds cmb_random_fmix64(master_seed, first + i); uses the terrain of the last awacs_ref_terrain call."""
    out = (AwacsOut * count)()
    rc = lib.awacs_ref_experiment(C.c_uint64(master_seed), C.c_uint64(first), C.c_uint64(count), C.c_double(duration_h), out)
    assert rc == 0
    return list(out)

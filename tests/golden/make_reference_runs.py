"""What the UNMODIFIED reference build (oracle/_ref: librefdrv.so, libawacs_ref.so, libtut3_ref.so) returns for the runs the
tests compare the plain-C port, the engine's host build and the device with, beyond the vectors of the other make_*.py here.

    make -C oracle ref && python tests/golden/make_reference_runs.py      -> tests/golden/reference_runs.json

Each record holds a run's inputs, its per-trial event counts and the SHA-256 of its result rows (oracle_libs.result_digest);
a test repeats the run on the code under test and compares the digest.  Where the reference is run through its own pthread
executive (cimba_run_experiment), the same trials are also run one at a time here and must agree."""
import ctypes as C
import json
import random
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT / "tests"))
from oracle_libs import (DIST_CASES, REFERENCE_RUNS, awacs_ref_experiment, awacs_terrain, awacs_trial,  # noqa: E402
                         load_awacs_ref, load_ref, result_digest, rng_draws_ex, run_trials, trace_trial,
                         trial_rows)

MASTER = 0x34F05C64D7AD598F

# test_oracle_port.py::test_port_equals_live_reference: model, arr_mean, srv_mean, servers
PORT_CASES = [(0, 1 / 0.9, 1.0, 1), (0, 1.25, 1.0, 1), (1, 1.25, 1.0, 1), (2, 1 / 6.4, 1.0, 8), (2, 0.5, 1.0, 3),
              (3, 1.0, 1.0, 10), (3, 0.5, 1.0, 2), (3, 0.7, 0.7, 1), (4, 1.0, 1.0, 20), (4, 1.0, 1.0, 5),
              (5, 1.0, 1.0, 10), (5, 0.5, 1.0, 2), (6, 1.0, 1.0, 8), (6, 0.5, 1.0, 2), (7, 1.0, 1.0, 500), (7, 0.5, 1.0, 5),
              (8, 1.0, 0.6, 1), (8, 0.4, 1.2, 1), (9, 1 / 0.9, 1.0, 1), (9, 2.0, 1.0, 1),
              (10, 2.0, 8.0, 10), (10, 1.2, 8.0, 4), (10, 0.9, 8.0, 3), (11, 1.0, 1.0, 10), (11, 0.5, 1.0, 2),
              (12, 1.0, 1.0, 10), (12, 0.5, 1.0, 4), (13, 1.0, 1.0, 10), (13, 0.5, 1.0, 3), (14, 1.0, 1.0, 1)]

# test_cmb_engine.py::test_engine_matches_the_live_reference_build: model, servers, num_objects, arr_mean, srv_mean, params
ENGINE_CASES = [(0, 1, 7000, 1.0, 1.0, []), (2, 5, 7000, 0.22, 1.0, []), (16, 300, 25, 2.5, 1.0, [0.9]), (17, 2, 7000, 1.2, 1.0, [])]


def record(rows, **inputs):
    return dict(inputs, events=[int(r[0]) for r in rows], sha256=result_digest(rows))


def engine_case(model, servers, nobj, arr, srv, params, first, count):
    return {"model": model, "servers": servers, "num_objects": nobj, "arr_mean": float(arr).hex(), "srv_mean": float(srv).hex(),
            "params": params, "first": first, "count": count}


def engine_runs(ref, case, counters):
    """The reference's trials of an engine case, as (events, objects, t_end, sum_wait, counters[:counters])."""
    ref.ref_set_param(0, case["params"][0] if case["params"] else 0.0)
    res = run_trials(ref, "ref", case["model"], case["servers"], MASTER, case["first"], case["count"], case["num_objects"],
                     float.fromhex(case["arr_mean"]), float.fromhex(case["srv_mean"]), par=0)
    ref.ref_set_param(0, 0.0)
    return record([(*r.key(), *r.counters()[:counters]) for r in res], **case)


def drawn_engine_cases():
    """test_cmb_engine.py::test_engine_against_the_live_reference_on_drawn_parameters: the reference's test worlds and tutorial 1
    on drawn parameters - capacities 1..40, durations, means, warm-up times (not model 18: its cmb_random_flip calls leave cached
    bits in the reference's thread-local cache for the trials after it)."""
    rnd = random.Random(7)
    cases = []
    for model in (3, 4, 5, 6, 8, 9, 11, 12, 13, 14, 19):
        for _ in range(3):
            servers = 1 if model in (8, 9, 14, 19) else rnd.randint(1, 40)
            nobj = rnd.randint(150, 1500)
            arr, srv = rnd.choice([0.4, 0.7, 1.0, 1.6]), rnd.choice([0.6, 1.0, 1.4])
            params = [rnd.uniform(0.0, 100.0)] if model == 19 else []
            cases.append(engine_case(model, servers, nobj, arr, srv, params, rnd.randint(0, 5000), 4))
    return cases


class Tut3Out(C.Structure):
    _fields_ = [("events", C.c_uint64), ("t_end", C.c_double), ("park", C.c_double), ("riding", C.c_double),
                ("waiting", C.c_double), ("walking", C.c_double), ("rides", C.c_double)]


def main():
    ref, aref = load_ref(), load_awacs_ref()
    assert ref is not None and aref is not None, "oracle/_ref is not built (make -C oracle ref)"
    ref.ref_set_param.argtypes = [C.c_int, C.c_double]
    out = {"master": MASTER}

    out["distributions"] = []
    for kind, par in DIST_CASES:
        for seed in (1, 0xC0FFEE):
            v = rng_draws_ex(ref, "ref", seed, kind, par, 8192)
            out["distributions"].append({"kind": kind, "params": par, "seed": seed, "n": len(v),
                                         "sha256": result_digest([(x,) for x in v])})

    out["port_cases"] = []
    for model, arr, srv, servers in PORT_CASES:
        size = 20_000 if model in (0, 1, 2, 9) else (30 if model == 7 else 1500)     # models 3..8: duration in time units
        res = run_trials(ref, "ref", model, servers, 0xC0FFEE, 100, 48, size, arr, srv, par=0)
        tsize = 3000 if model in (0, 1, 2, 9) else (15 if model == 7 else 800)
        r, keys, times = trace_trial(ref, "ref", model, servers, 99, tsize, arr, srv, 9000)
        out["port_cases"].append(dict(record(trial_rows(res), model=model, arr=arr, srv=srv, servers=servers, master=0xC0FFEE,
                                             first=100, count=48, num_objects=size),
                                      trace_seed=99, trace_objects=tsize, trace_cap=9000,
                                      trace_sha256=result_digest([r.key(), *zip(keys, times)])))

    # the reference's pthread executive (cimba_run_experiment, all cores) against the same trials one at a time
    par = run_trials(ref, "ref", 0, 1, MASTER, 0, 32, 5000, 1 / 0.9, 1.0, par=1)
    assert trial_rows(par) == trial_rows(run_trials(ref, "ref", 0, 1, MASTER, 0, 32, 5000, 1 / 0.9, 1.0, par=0))
    out["executive"] = record([r.key() for r in par], model=0, servers=1, first=0, count=32, num_objects=5000, arr=1 / 0.9, srv=1.0)

    m, cols, rows, geom = awacs_terrain(aref, "ref", 77, 8.0, 6.0)
    out["awacs_terrain"] = {"seed": 77, "width_nm": 8.0, "height_nm": 6.0, "cols": cols, "rows": rows,
                            "geom": [float(v).hex() for v in geom], "map_sha256": result_digest([m.view("<u4")])}
    out["awacs_trials"] = []
    for seed in (5, 6):
        o, keys, times, per = awacs_trial(aref, "ref", seed, 0.03, trace_cap=3000)
        targets = list(zip(per["tds"], per["detected"], per["mode"], per["x"].view("<u4")))
        out["awacs_trials"].append(dict(record([o.row()], seed=seed, hours=0.03), trace_cap=3000,
                                        trace_sha256=result_digest(zip(keys, times)), targets_sha256=result_digest(targets)))
    outs = awacs_ref_experiment(aref, MASTER, 3, 6, 0.02)
    assert [o.key() for o in outs] == [awacs_trial(aref, "ref", ref.ref_fmix64(MASTER, 3 + i), 0.02)[0].key() for i in range(6)]
    out["awacs_executive"] = record([o.row() for o in outs], first=3, count=6, hours=0.02)

    out["engine_cases"] = [engine_runs(ref, engine_case(*c, first=11, count=5), 4) for c in ENGINE_CASES]
    out["engine_drawn_cases"] = [engine_runs(ref, c, 8) for c in drawn_engine_cases()]

    # test_gpu_cmb_engine.py: the reneging model with 1200 processes, through the reference's pthread executive
    renege = engine_case(16, 1200, 30, 3.0, 1.0, [0.8], 100, 24)
    ref.ref_set_param(0, 0.8)
    res = run_trials(ref, "ref", 16, 1200, MASTER, 100, 24, 30, 3.0, 1.0, par=1)
    ref.ref_set_param(0, 0.0)
    out["renege"] = record([(r.events, r.t_end, r.sum_wait, *r.counters()[:4]) for r in res], **renege)

    # tutorial/tut_1_7.c's experiment: 39 utilisations x 2 replications, warm-up 100, 2000 time units; trial i is seeded (MASTER, i)
    arr_means = [1.0 / (0.025 * (k // 2 + 1)) for k in range(78)]
    ref.ref_set_param(0, 100.0)
    res = [run_trials(ref, "ref", 19, 1, MASTER, i, 1, 2000, a, 1.0, par=0)[0] for i, a in enumerate(arr_means)]
    ref.ref_set_param(0, 0.0)
    out["tutorial1"] = record([(r.events, r.t_end, *r.counters()) for r in res], arr_means=[a.hex() for a in arr_means],
                              warmup=100.0, num_objects=2000)

    # tutorial/tut_3_1.c, trials 1000..1299
    lib = C.CDLL(str(ROOT / "oracle/_ref/libtut3_ref.so"))
    lib.tut3_ref_trial.argtypes = [C.c_uint64, C.POINTER(Tut3Out)]
    park = []
    for i in range(1000, 1300):
        o = Tut3Out()
        assert lib.tut3_ref_trial(ref.ref_fmix64(MASTER, i), C.byref(o)) == 0
        park.append((o.events, o.t_end, o.park, o.riding, o.waiting, o.walking, o.rides))
    out["park"] = record(park, first=1000, count=300)

    REFERENCE_RUNS.write_text(json.dumps(out, indent=1) + "\n")
    print(REFERENCE_RUNS, REFERENCE_RUNS.stat().st_size, "bytes")


if __name__ == "__main__":
    main()

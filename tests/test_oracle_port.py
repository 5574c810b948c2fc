"""CPU tests: pin the plain-C oracle (oracle/port) to the reference.

Two anchors, both generated from the unmodified reference build: (1) the golden
vectors of tests/golden/make_golden.py; (2) the reference's results for more
seeds and models (tests/golden/make_reference_runs.py).
"""
import ctypes as C

import numpy as np
import pytest

from oracle_libs import reference_runs, result_digest, rng_draws, run_trials, trace_trial, trial_rows

KAT_SEED = 0x34F05C64D7AD598F
RUNS = reference_runs()


def _u64(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.uint64)


def test_fmix64_golden(port, golden):
    for seed, vals in golden["fmix64"].items():
        assert [port.port_fmix64(int(seed), k) for k in range(4)] == vals
    # SURVEY.md section 8c known answers
    assert port.port_fmix64(KAT_SEED, 0) == 0xA9668314774003F8
    assert port.port_fmix64(KAT_SEED, 1) == 0x3A4431CFB7782955


def test_sfc64_known_answer(port):
    """First four sfc64 outputs after cmb_random_initialize(KAT seed), SURVEY.md 8c."""
    v = _u64(rng_draws(port, "port", KAT_SEED, 0, 0, 0, 4))
    assert [int(x) for x in v] == [0xF02D5E84CDE20D15, 0x77AC3D6A1A0CEA15,
                                   0x899343477AF13C7A, 0x5075D2DA64199B6E]


def test_exponential_normal_known_answers(port):
    e = rng_draws(port, "port", KAT_SEED, 1, 1.0, 0, 4)
    assert list(e) == [3.8042282138002448, 1.8955281505704349, 0.92997109312110893, 0.59381178361121356]
    z = rng_draws(port, "port", KAT_SEED, 2, 0, 0, 4)
    assert list(z) == [-0.3168921584334039, 2.3967586040326996, -1.4514249997250523, 1.0383410708137473]


@pytest.mark.parametrize("kind", range(9))
def test_rng_streams_match_golden_checksums(port, golden, kind):
    """10^5..10^6 draws per (seed, distribution): first 16 verbatim + checksums of all bits."""
    for seed, per in golden["rng"].items():
        g = per[str(kind)]
        v = rng_draws(port, "port", int(seed), kind, g["p0"], g["p1"], g["n"])
        u = _u64(v)
        if kind == 0:
            assert [int(x) for x in u[:16]] == g["first"]
        else:
            assert [float.hex(float(x)) for x in v[:16]] == g["first"]
        assert int(np.bitwise_xor.reduce(u)) == g["xor"]
        assert int(np.add.reduce(u, dtype=np.uint64)) == g["sum"]


def test_remaining_distributions_match_golden(port, golden):
    """Kinds 9..33 (triangular ... pascal): the restatement against streams drawn from the reference."""
    from oracle_libs import rng_draws_ex
    assert len(golden["distributions"]) >= 25
    for g in golden["distributions"]:
        v = np.array(rng_draws_ex(port, "port", KAT_SEED, g["kind"], g["params"], g["n"]))
        u = _u64(v)
        tag = (g["kind"], g["params"])
        assert [float.hex(float(x)) for x in v[:8]] == g["first"], tag
        assert int(np.bitwise_xor.reduce(u)) == g["xor"], tag
        assert int(np.add.reduce(u, dtype=np.uint64)) == g["sum"], tag


def test_remaining_distributions_match_live_reference(port):
    """Kinds 9..33, two more seeds: every one of 8192 variates as the reference drew it."""
    from oracle_libs import DIST_CASES, rng_draws_ex
    assert [(g["kind"], g["params"]) for g in RUNS["distributions"][::2]] == [(k, list(p)) for k, p in DIST_CASES]
    for g in RUNS["distributions"]:
        b = rng_draws_ex(port, "port", g["seed"], g["kind"], g["params"], g["n"])
        assert result_digest([(x,) for x in b]) == g["sha256"], (g["kind"], g["params"], g["seed"])


def test_trials_match_golden(port, golden):
    """Every committed single-trial record: counts exact, clock and sums bit-exact,
    and the first 512 pops (key, time) of the 1000-object runs."""
    for t in golden["trials"]:
        if t["num_objects"] > 100_000:
            continue
        cap = len(t.get("trace_key", []))
        r, keys, times = trace_trial(port, "port", t["model"], t["servers"], t["seed"], t["num_objects"],
                                     float.fromhex(t["arr_mean"]), float.fromhex(t["srv_mean"]), cap)
        tag = (t["model"], hex(t["seed"]), t["num_objects"])
        assert (r.events, r.objects) == (t["events"], t["objects"]), tag
        assert float.hex(r.t_end) == t["t_end"], tag
        assert float.hex(r.sum_wait) == t["sum_wait"], tag
        assert (r.max_fel, r.max_queue) == (t["max_fel"], t["max_queue"]), tag
        assert r.counters() == t["counters"], tag
        if cap:
            assert keys == t["trace_key"], tag
            assert [float.hex(x) for x in times] == t["trace_time"], tag


@pytest.mark.parametrize("model", [0, 1, 2, 9])
def test_full_size_known_answer(port, golden, model):
    """The 10^6-object known answers (SURVEY.md 8c: M/M/1 2 099 622 events, ...)."""
    t = [x for x in golden["trials"] if x["num_objects"] == 1_000_000 and x["model"] == model][0]
    r, _, _ = trace_trial(port, "port", model, t["servers"], t["seed"], 1_000_000,
                          float.fromhex(t["arr_mean"]), float.fromhex(t["srv_mean"]), 0)
    assert (r.events, r.objects) == (t["events"], t["objects"])
    assert float.hex(r.t_end) == t["t_end"] and float.hex(r.sum_wait) == t["sum_wait"]
    assert r.counters() == t["counters"]            # model 9: the time-weighted queue-length cmb_wtdsummary
    if model == 0:
        assert r.events == 2_099_622 and r.t_end == 1109668.9795469602 and r.sum_wait == 9895522.5628889836


def test_harbor_reproduces_the_reference_golden_file(port, golden):
    """test/reference/condition.txt (the reference's own golden output for its harbor model, seed
    0x34f05c64d7ad598f, 100 simulated years): N 328781 small / 109454 large ships, mean system times
    10.91 / 17.48, tug history N 1736975 mean 0.8025, berth histories N 645947 / 217380."""
    import struct
    t = [x for x in golden["trials"] if x["model"] == 10 and x["num_objects"] == 873_600][0]
    r, _, _ = trace_trial(port, "port", 10, 10, KAT_SEED, 873_600, 2.0, 8.0, 0)
    assert (r.events, r.objects, float.hex(r.t_end), float.hex(r.sum_wait)) == \
           (t["events"], t["objects"], t["t_end"], t["sum_wait"])
    assert r.counters() == t["counters"] and (r.max_fel, r.max_queue) == (t["max_fel"], t["max_queue"])
    c = r.counters()
    f = lambda u: struct.unpack("<d", struct.pack("<Q", u))[0]
    assert (c[0], c[1]) == (328781, 109454)
    assert ("%.4g" % f(c[2]), "%.4g" % f(c[3])) == ("10.91", "17.48")
    assert (c[4], "%.4g" % f(c[5])) == (1736975, "0.8025")
    assert (c[6] & 0xffffffff, c[6] >> 32) == (645947, 217380)


@pytest.mark.parametrize("model", [11, 13])
def test_objectqueue_and_priorityqueue_reproduce_the_reference_golden_files(port, golden, model):
    """test/reference/objectqueue.txt and priorityqueue.txt (test/test_objectqueue.c / test_priorityqueue.c, seed
    0x34f05c64d7ad598f, 1e6 time units): queue-length history N 5689021, time-weighted mean 5.008."""
    import struct
    t = [x for x in golden["trials"] if x["model"] == model and x["num_objects"] == 1_000_000][0]
    r, _, _ = trace_trial(port, "port", model, 10, KAT_SEED, 1_000_000, 1.0, 1.0, 0)
    assert (r.events, r.objects, float.hex(r.t_end), float.hex(r.sum_wait)) == \
           (t["events"], t["objects"], t["t_end"], t["sum_wait"])
    assert r.counters() == t["counters"] and (r.max_fel, r.max_queue) == (t["max_fel"], t["max_queue"])
    mean = struct.unpack("<d", struct.pack("<Q", r.counters()[6]))[0]
    assert r.max_queue == 5689021 and "%.4g" % mean == "5.008"


def test_buffer_reproduces_the_reference_golden_file(port, golden):
    """test/reference/buffer.txt (test/test_buffer.c, seed 0x34f05c64d7ad598f, 10 000 time units):
    level history N 41876, time-weighted mean 4.980."""
    import struct
    t = [x for x in golden["trials"] if x["model"] == 12 and x["num_objects"] == 10_000 and x["seed"] == KAT_SEED][-1]
    r, _, _ = trace_trial(port, "port", 12, 10, KAT_SEED, 10_000, 1.0, 1.0, 0)
    assert (r.events, float.hex(r.t_end)) == (t["events"], t["t_end"])
    assert r.counters() == t["counters"] and (r.max_fel, r.max_queue) == (t["max_fel"], t["max_queue"])
    mean = struct.unpack("<d", struct.pack("<Q", r.counters()[4]))[0]
    assert r.max_queue == 41876 and "%.3f" % mean == "4.980"


def test_resource_reproduces_the_reference_golden_file(port, golden):
    """test/reference/resource.txt (test/test_resource.c, seed 0x34f05c64d7ad598f, 25 time units): usage history
    N 30, time-weighted mean 0.9816, and the one logged pre-emption: Target_3 at t = 6.3280."""
    import struct
    t = [x for x in golden["trials"] if x["model"] == 14 and x["num_objects"] == 25 and x["seed"] == KAT_SEED][-1]
    r, _, _ = trace_trial(port, "port", 14, 1, KAT_SEED, 25, 1.0, 1.0, 0)
    assert (r.events, float.hex(r.t_end), float.hex(r.sum_wait)) == (t["events"], t["t_end"], t["sum_wait"])
    assert r.counters() == t["counters"] and r.max_queue == t["max_queue"] == 30
    f = lambda u: struct.unpack("<d", struct.pack("<Q", u))[0]
    c = r.counters()
    assert "%.4f" % f(c[3]) == "0.9816" and "%.4f" % f(c[4]) == "6.3280" and c[5] == 3 and c[1] == 1


def test_experiment_seeding_matches_golden(port, golden):
    g = golden["experiment_mm1"]
    res = run_trials(port, "port", 0, 1, g["master_seed"], 0, len(g["trials"]), g["num_objects"], 1 / 0.9, 1.0)
    for r, t in zip(res, g["trials"]):
        assert (r.events, r.objects, float.hex(r.t_end), float.hex(r.sum_wait)) == \
               (t["events"], t["objects"], t["t_end"], t["sum_wait"])
    # sharding: trials [40, 64) run on their own give the same answers (seed = f(global index))
    part = run_trials(port, "port", 0, 1, g["master_seed"], 40, 24, g["num_objects"], 1 / 0.9, 1.0)
    assert [p.key() for p in part] == [r.key() for r in list(res)[40:]]
    # the pthread executive of the port gives the same per-trial results
    par = run_trials(port, "port", 0, 1, g["master_seed"], 0, 64, g["num_objects"], 1 / 0.9, 1.0, par=4)
    assert [p.key() for p in par] == [r.key() for r in res]


def test_summaries_match_golden(port, golden):
    s = golden["summary"]
    x = np.array([float.fromhex(v) for v in s["x"]])
    w = np.array([float.fromhex(v) for v in s["w"]])
    dp = C.POINTER(C.c_double)
    xs, wsp = x.ctypes.data_as(dp), w.ctypes.data_as(dp)
    o = (C.c_double * 8)()
    port.port_datasummary_of(xs, 1000, o)
    assert [float.hex(v) for v in o[:7]] == s["data_all"]
    port.port_wtdsummary_of(xs, wsp, 1000, o)
    assert [float.hex(v) for v in o[:8]] == s["wtd_all"]
    for na in (1, 333, 500, 999):
        port.port_datasummary_split_merge(xs, na, 1000, o)
        assert [float.hex(v) for v in o[:7]] == s[f"data_merge_{na}"]
        port.port_wtdsummary_split_merge(xs, wsp, na, 1000, o)
        assert [float.hex(v) for v in o[:8]] == s[f"wtd_merge_{na}"]


def test_heap_script_orders_like_the_comparator(port):
    """cmi_hashheap order = (time asc, priority desc, key asc) under push/pop/cancel churn."""
    g = np.random.default_rng(5)
    n = 4000
    ops = np.zeros(n, dtype=np.int32)
    vd = np.zeros(n)
    vi = np.zeros(n, dtype=np.int64)
    live = {}            # key -> (time, prio)
    model_out = []
    next_key = 0
    for s in range(n):
        r = g.random()
        if r < 0.55 or not live:
            ops[s] = 0
            vd[s] = float(g.integers(0, 40))          # many ties
            vi[s] = int(g.integers(-2, 3))
            next_key += 1
            live[next_key] = (vd[s], vi[s])
            model_out.append(next_key)
        elif r < 0.85:
            ops[s] = 1
            k = min(live, key=lambda k: (live[k][0], -live[k][1], k))
            del live[k]
            model_out.append(k)
        else:
            ops[s] = 2
            k = int(g.integers(1, next_key + 1))
            vi[s] = k
            model_out.append(1 if k in live else 0)
            live.pop(k, None)
    out = np.zeros(n, dtype=np.uint64)
    rc = port.port_heap_script(n, ops.ctypes.data_as(C.POINTER(C.c_int)), vd.ctypes.data_as(C.POINTER(C.c_double)),
                               vi.ctypes.data_as(C.POINTER(C.c_int64)), out.ctypes.data_as(C.POINTER(C.c_uint64)))
    assert rc == 0
    assert [int(v) for v in out] == model_out


# ------------------------------------------------------------------ live reference

@pytest.mark.parametrize("case", RUNS["port_cases"],
                         ids=lambda c: f"{c['model']}-{c['arr']}-{c['srv']}-{c['servers']}")
def test_port_equals_live_reference(port, case):
    """48 trials per model and load (keys, max_fel / max_queue and counters) and one pop trace of up to 9000 pops,
    as the reference computed them."""
    model, servers, arr, srv = case["model"], case["servers"], case["arr"], case["srv"]
    b = run_trials(port, "port", model, servers, case["master"], case["first"], case["count"], case["num_objects"], arr, srv)
    assert [x.events for x in b] == case["events"]
    assert result_digest(trial_rows(b)) == case["sha256"]
    rb, kb, tb = trace_trial(port, "port", model, servers, case["trace_seed"], case["trace_objects"], arr, srv, case["trace_cap"])
    assert result_digest([rb.key(), *zip(kb, tb)]) == case["trace_sha256"]


def test_reference_pthread_executive_equals_serial(port):
    """cimba_run_experiment (all cores) - the multi-thread path the reference itself only smoke-tests (SURVEY.md
    section 4), checked against the same trials run serially when the vectors were made - against the port's trials,
    serial and on its own pthread executive."""
    g = RUNS["executive"]
    for par in (0, 4):
        b = run_trials(port, "port", g["model"], g["servers"], RUNS["master"], g["first"], g["count"], g["num_objects"],
                       g["arr"], g["srv"], par=par)
        assert result_digest([x.key() for x in b]) == g["sha256"]

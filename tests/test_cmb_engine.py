"""CPU tests of the general engine (cimba_b200/csrc/cmb_device.cuh) and of the models written against its authoring
surface (cimba_b200/models/*.cuh, examples/tandem_model.cuh): the SAME source text compiled for the host
(tests/cmb_engine_host.cpp) must reproduce, trial for trial, what the unmodified reference produced for the same
models written against its own API (tests/golden/cmb_engine_vectors.json, tests/golden/reference_runs.json): event
count, clock, sums, counters and the pop trace - M/M/1 (also in heavy traffic and overload, where the
queue grows without bound), G/G/1, M/M/c (3, 8 and 64 servers, overload), the reneging model with 40, 1000 and 1500
processes (timers, cancels by handle, wait-list removals, the stop cascade) and the tandem model with a blocking put."""
import ctypes as C
import subprocess
from pathlib import Path

import pytest

from cmb_cases import GOLD, MASTER, RESOURCEPOOL_GOLDEN_LINE, TRACE, case_id, check_trial, inverse_fmix64, wtdsummary_line
from oracle_libs import reference_runs, result_digest

ROOT = Path(__file__).resolve().parents[1]
RUNS = reference_runs()


class HostResult(C.Structure):
    _fields_ = [("events", C.c_uint64), ("objects", C.c_uint64), ("t_end", C.c_double), ("sum_wait", C.c_double),
                ("max_fel", C.c_uint64), ("max_queue", C.c_uint64), ("counter", C.c_uint64 * 8), ("status", C.c_uint32),
                ("pad", C.c_uint32)]


@pytest.fixture(scope="module")
def host(tmp_path_factory):
    so = tmp_path_factory.mktemp("cmb") / "libcmb_engine_host.so"
    subprocess.run(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-Wall", "-Wno-unknown-pragmas", "-Wno-unused-function",
                    "-shared", "-fPIC", str(ROOT / "tests/cmb_engine_host.cpp"), "-o", str(so)], check=True, capture_output=True)
    lib = C.CDLL(str(so))
    f = lib.host_cmb_run_trials
    f.restype = C.c_int
    f.argtypes = [C.c_int, C.c_int, C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint64, C.c_double, C.c_double,
                  C.POINTER(C.c_double), C.c_uint32, C.c_uint64, C.c_uint64, C.POINTER(C.c_uint64), C.POINTER(C.c_double),
                  C.POINTER(HostResult)]
    return f


def run_host(f, c, n, arena=1 << 26, first=0, master=MASTER):
    out = (HostResult * n)()
    par = (C.c_double * max(1, len(c["params"])))(*c["params"])
    keys = (C.c_uint64 * (n * TRACE))()
    times = (C.c_double * (n * TRACE))()
    rc = f(c["model"], c["servers"], master, first, n, c["num_objects"], float.fromhex(c["arr_mean"]),
           float.fromhex(c["srv_mean"]), par, len(c["params"]), arena, TRACE, keys, times, out)
    assert rc == 0
    return out, keys, times


@pytest.mark.parametrize("case", GOLD["cases"], ids=case_id)
def test_engine_source_on_the_cpu_matches_the_reference_vectors(host, case):
    n = len(case["trials"])
    out, keys, times = run_host(host, case, n)
    for i, want in enumerate(case["trials"]):
        assert out[i].status == 0
        check_trial(want, out[i].events, out[i].objects, out[i].t_end, out[i].sum_wait, list(out[i].counter),
                    keys[i * TRACE:(i + 1) * TRACE], times[i * TRACE:(i + 1) * TRACE], f"trial {i}")
        if case["model"] == 2:
            assert out[i].max_queue == want["max_queue"]        # process structs ever created
        if case["model"] in (11, 12, 13, 14):
            assert out[i].max_queue == want["max_queue"]        # samples in the recorded history
        if case["model"] in (3, 4, 5, 6, 8):
            assert out[i].max_queue == want["max_fel"]          # the deepest the event list was at a pop


def check_reference_run(host, case, counters):
    """A case of tests/golden/reference_runs.json on the engine's host build: events, objects, t_end, sum_wait and the
    first `counters` counters of every trial as the reference computed them."""
    out, _, _ = run_host(host, case, case["count"], first=case["first"])
    assert all(o.status == 0 for o in out), case
    assert [o.events for o in out] == case["events"], case
    assert result_digest([(o.events, o.objects, o.t_end, o.sum_wait, *list(o.counter)[:counters]) for o in out]) == case["sha256"], case


def test_engine_matches_the_live_reference_build(host):
    for case in RUNS["engine_cases"]:
        check_reference_run(host, case, 4)


def test_a_small_arena_is_reported_not_survived_silently(host):
    """The event list of a 1000-process trial cannot grow out of 4 KB: the trial must say so in its status word."""
    case = next(c for c in GOLD["cases"] if c["model"] == 16 and c["servers"] == 1000)
    out, _, _ = run_host(host, case, 1, arena=4096)
    assert out[0].status & 64           # CIMBA_B200_TRIAL_ARENA_EXHAUSTED


def test_hashheap_growth_and_key_map(host):
    """M/M/c with 64 servers grows the event list from 8 to 128 slots; the reneging model activates the key map."""
    c64 = next(c for c in GOLD["cases"] if c["model"] == 2 and c["servers"] == 64)
    out, _, _ = run_host(host, c64, 1)
    assert out[0].max_fel == 128
    rn = next(c for c in GOLD["cases"] if c["model"] == 16 and c["servers"] == 1500)
    out, _, _ = run_host(host, rn, 1)
    assert out[0].counter[5] >= 11 and out[0].counter[6] == 1 and out[0].counter[7] == 1500


def test_engine_reproduces_the_reference_resourcepool_golden_file(host):
    """test/reference/resourcepool.txt - the golden file round 1 left open (its result depends on the holders' tie-break by
    process address): the reference's own pool test written against the authoring surface (cimba_b200/models/cheese_model.cuh),
    seeded like the test (cmb_random_initialize(0x34f05c64d7ad598f)), 20 units, 100 time units, gives the file's summary line."""
    import cimba_b200 as cb
    case = {"model": 18, "servers": 20, "num_objects": 100, "arr_mean": (1.0).hex(), "srv_mean": (1.0).hex(), "params": []}
    out, _, _ = run_host(host, case, 1, master=inverse_fmix64(0x34F05C64D7AD598F))
    assert out[0].status == 0 and out[0].counter[0] == 120
    assert wtdsummary_line(cb.lib, list(out[0].counter)) == RESOURCEPOOL_GOLDEN_LINE


def test_engine_reproduces_the_reference_condition_golden_file(host):
    """test/reference/condition.txt: the reference's harbor (test/test_condition.c = tutorial/tut_4_1.c) written against the
    authoring surface (cimba_b200/models/harbor_general_model.cuh), seeded like the test, 100 simulated years: 4 579 051 events,
    the file's ship counts (:8, :35), mean system times, tug (:85) and berth (:62, :75) history sizes and the tug mean."""
    import struct
    case = {"model": 10, "servers": 10, "num_objects": 873600, "arr_mean": (2.0).hex(), "srv_mean": (8.0).hex(), "params": []}
    out, _, _ = run_host(host, case, 1, master=inverse_fmix64(0x34F05C64D7AD598F))
    o = out[0]
    f = lambda u: struct.unpack("<d", struct.pack("<Q", u))[0]
    c = list(o.counter)
    assert o.status == 0 and o.events == 4579051
    assert (c[0], c[1]) == (328781, 109454) and ("%.4g" % f(c[2]), "%.4g" % f(c[3])) == ("10.91", "17.48")
    assert c[4] == 1736975 and "%.4g" % f(c[5]) == "0.8025"
    assert (c[6] & 0xffffffff, c[6] >> 32) == (645947, 217380)


def _double(u):
    import struct
    return struct.unpack("<d", struct.pack("<Q", int(u) & (2**64 - 1)))[0]


@pytest.mark.parametrize("model", [11, 13])
def test_engine_reproduces_the_reference_queue_golden_files(host, model):
    """test/reference/objectqueue.txt (model 11, cmb_objectqueue) and priorityqueue.txt (model 13, cmb_priorityqueue): the
    reference's queue tests written against the authoring surface (cimba_b200/models/guarded_model.cuh), seeded like the
    tests, capacity 10, 1e6 time units: length history N 5689021, time-weighted mean 5.008."""
    case = {"model": model, "servers": 10, "num_objects": 1_000_000, "arr_mean": (1.0).hex(), "srv_mean": (1.0).hex(), "params": []}
    out, _, _ = run_host(host, case, 1, master=inverse_fmix64(0x34F05C64D7AD598F))
    assert out[0].status == 0 and out[0].max_queue == 5689021 and "%.4g" % _double(out[0].counter[6]) == "5.008"


def test_engine_reproduces_the_reference_buffer_golden_file(host):
    """test/reference/buffer.txt: test/test_buffer.c on the engine's cmb_buffer (cimba_b200/models/workshop_model.cuh), capacity 10,
    10 000 time units: level history N 41876, time-weighted mean 4.980."""
    case = {"model": 12, "servers": 10, "num_objects": 10_000, "arr_mean": (1.0).hex(), "srv_mean": (1.0).hex(), "params": []}
    out, _, _ = run_host(host, case, 1, master=inverse_fmix64(0x34F05C64D7AD598F))
    assert out[0].status == 0 and out[0].max_queue == 41876 and "%.3f" % _double(out[0].counter[4]) == "4.980"


def test_engine_reproduces_the_reference_resource_golden_file(host):
    """test/reference/resource.txt: test/test_resource.c on the engine's cmb_resource with pre-emption: history N 30, mean 0.9816,
    one pre-emption - Target_3 loses the resource at t = 6.3280 - in a run of 85 events."""
    case = {"model": 14, "servers": 1, "num_objects": 25, "arr_mean": (1.0).hex(), "srv_mean": (1.0).hex(), "params": []}
    out, _, _ = run_host(host, case, 1, master=inverse_fmix64(0x34F05C64D7AD598F))
    c = list(out[0].counter)
    assert out[0].status == 0 and out[0].events == 85 and out[0].max_queue == 30
    assert "%.4f" % _double(c[3]) == "0.9816" and "%.4f" % _double(c[4]) == "6.3280" and c[5] == 3 and c[1] == 1


@pytest.mark.parametrize("case", [c for c in GOLD["cases"] if c["model"] in (0, 1, 9, 17, 19)], ids=case_id)
def test_static_tier_source_on_the_cpu_matches_the_reference_vectors(host, case):
    """csrc/cmb_static.cuh: the same model templates (mm1_model.cuh, gg1_model.cuh, examples/tandem_model.cuh) compiled against
    cmb::StaticSim - one event slot per process, guards as a bit per process, queues as rings - on the CPU.  With a ring of 512
    entries behind the 32-entry window an overloaded trial is flagged (and would be re-run by the general engine on the device);
    with a ring sized for it the tier itself gives the reference's answer."""
    n = len(case["trials"])
    static_case = dict(case, model=case["model"] + 100)
    for ring in (512, 1 << 17):
        out, keys, times = run_host(host, static_case, n, arena=ring)
        for i, want in enumerate(case["trials"]):
            if ring == 512 and out[i].status:
                assert out[i].status == 1               # CIMBA_B200_TRIAL_QUEUE_OVERFLOW: the repair pass's business
                continue
            assert out[i].status == 0
            check_trial(want, out[i].events, out[i].objects, out[i].t_end, out[i].sum_wait,
                        list(out[i].counter) if case["model"] in (9, 19) else None,    # the history's eight summary words
                        keys[i * TRACE:(i + 1) * TRACE], times[i * TRACE:(i + 1) * TRACE], f"trial {i}")


def test_theme_park_tutorial_on_the_engine_matches_the_unmodified_tutorial_source(host):
    """tutorial/tut_3_1.c (nine attractions, priority queues, batch servers, visitors that balk, jockey and renege on timers) written
    against the authoring surface (cimba_b200/models/park_model.cuh): events executed, final clock and the tutorial's five averages
    of 64 trials, bit for bit, against vectors the UNMODIFIED tutorial source produced (tests/golden/make_park_golden.py)."""
    import json
    import struct
    gold = json.loads((ROOT / "tests/golden/park_vectors.json").read_text())
    n = len(gold["trials"])
    case = {"model": 20, "servers": 1, "num_objects": 0, "arr_mean": (1.0).hex(), "srv_mean": (1.0).hex(), "params": []}
    out, _, _ = run_host(host, case, n, master=gold["master"])
    for i, want in enumerate(gold["trials"]):
        d = [struct.unpack("<d", struct.pack("<Q", v))[0].hex() for v in list(out[i].counter)[:5]]
        assert out[i].status == 0 and (out[i].events, float(out[i].t_end).hex(), d) == (want["events"], want["t_end"], want["means"]), i


def test_second_tutorial_on_the_engine_matches_the_unmodified_tutorial_source(host):
    """tutorial/tut_2_1.c (mice acquire, rats pre-empt, a cat interrupts; ~670 000 events per trial) written against the authoring
    surface (cimba_b200/models/tutorial2_model.cuh): events executed, final clock and the random stream's position after the run,
    against the UNMODIFIED tutorial source run as a program (tests/golden/make_tutorial2_golden.py)."""
    import json
    gold = json.loads((ROOT / "tests/golden/tutorial2_vectors.json").read_text())
    n = 12
    case = {"model": 21, "servers": 1, "num_objects": 0, "arr_mean": (1.0).hex(), "srv_mean": (1.0).hex(), "params": []}
    out, _, _ = run_host(host, case, n, master=gold["master"])
    for i, want in enumerate(gold["trials"][:n]):
        assert out[i].status == 0
        assert (out[i].events, float(out[i].t_end).hex(), out[i].counter[0]) == (want["events"], want["t_end"], want["next_raw"]), i


def test_static_tier_and_general_engine_agree_on_parameters_no_vector_covers(host):
    """The same model templates compiled against cmb::StaticSim and cmb::Sim, run side by side on parameter sets drawn here (no
    stored vector knows them): events executed, final clock, sums, counters and the first pops must be the same for every trial."""
    import random
    rnd = random.Random(20260921)
    for model, servers_of, params_of in ((0, lambda: 1, lambda: []), (1, lambda: 1, lambda: []), (9, lambda: 1, lambda: []),
                                         (17, lambda: rnd.randint(1, 6), lambda: []), (19, lambda: 1, lambda: [rnd.uniform(0.0, 300.0)])):
        for _ in range(4):
            rho = rnd.uniform(0.3, 1.02)
            case = {"model": model, "servers": servers_of(), "num_objects": rnd.randint(500, 4000), "arr_mean": (1.0 / rho).hex(),
                    "srv_mean": rnd.choice([1.0, 0.7, 1.3]).hex(), "params": params_of()}
            first = rnd.randint(0, 10_000)
            general, gk, gt = run_host(host, case, 3, first=first)
            static, sk, st = run_host(host, dict(case, model=model + 100), 3, arena=1 << 16, first=first)
            for i in range(3):
                assert general[i].status == 0 and static[i].status == 0, (case, i)
                assert (general[i].events, general[i].objects, general[i].t_end, general[i].sum_wait, list(general[i].counter)) == \
                       (static[i].events, static[i].objects, static[i].t_end, static[i].sum_wait, list(static[i].counter)), (case, i)
                n = min(int(general[i].events), TRACE)
                assert list(gk[i * TRACE:i * TRACE + n]) == list(sk[i * TRACE:i * TRACE + n]), (case, i)
                assert list(gt[i * TRACE:i * TRACE + n]) == list(st[i * TRACE:i * TRACE + n]), (case, i)


def test_engine_against_the_live_reference_on_drawn_parameters(host):
    """Beyond the vectors of cmb_engine_vectors.json: the reference's test worlds and tutorial 1 on the engine's host build
    against the reference's results on drawn parameters - capacities 1..40, durations, means, warm-up times
    (tests/golden/make_reference_runs.py draws them), all eight counters."""
    assert len(RUNS["engine_drawn_cases"]) == 33
    for case in RUNS["engine_drawn_cases"]:
        check_reference_run(host, case, 8)

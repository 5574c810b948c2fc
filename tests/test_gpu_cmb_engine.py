"""GPU parity of the general engine (cimba_b200/csrc/cmb_device.cuh) and of everything built on it, through the C-ABI:

* the models written against the authoring surface (M/M/1, G/G/1, M/M/c, the 1000-process reneging model) against the
  vectors the unmodified reference produced for the same models written against its own API
  (tests/golden/cmb_engine_vectors.json, tests/golden/reference_runs.json);
* the repair pass: trials the fixed-capacity fast kernels flag (rho = 0.99, rho > 1, a wait list that outgrows its
  ring) come back with the reference's answer and a clean status word - the drop-in has no capacity the reference lacks;
* MODEL_MMC with 64 servers (the fast kernel's event list holds 16 entries);
* model libraries of one's own: examples/*.cu built with scripts/build_model.py, loaded with cimba_b200_model_load
  and run through cimba_b200_run_experiment like any built-in model."""
import sys
from pathlib import Path

import numpy as np
import pytest
import torch

import cimba_b200 as cb
from cmb_cases import GOLD, MASTER, RESOURCEPOOL_GOLDEN_LINE, TRACE, case_id, check_trial, inverse_fmix64, wtdsummary_line
from oracle_libs import load_port, reference_runs, result_digest, run_trials

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parents[1]
RUNS = reference_runs()
BUILTIN = {0: cb.MODEL_MM1, 1: cb.MODEL_GG1, 2: cb.MODEL_MMC, 7: cb.MODEL_HOLD, 10: cb.MODEL_HARBOR, 16: cb.MODEL_RENEGE,
           18: cb.MODEL_POOL_RECORDED, 19: cb.MODEL_TUTORIAL1,
           # the reference's own test worlds: since round 2 they run on the general engine by default
           9: cb.MODEL_MM1_RECORDED, 3: cb.MODEL_GUARDED, 4: cb.MODEL_PREEMPT, 5: cb.MODEL_BUFFER, 6: cb.MODEL_PRIOQ, 8: cb.MODEL_TIMERS,
           11: cb.MODEL_GUARDED_RECORDED, 12: cb.MODEL_BUFFER_RECORDED, 13: cb.MODEL_PRIOQ_RECORDED, 14: cb.MODEL_RESOURCE_RECORDED}
COVERAGE = (3, 4, 5, 6, 8, 9, 11, 12, 13, 14)


def run_case(case, model_id, variant, n, trace=True, spill=0):
    return cb.run_trials(n, arr_mean=float.fromhex(case["arr_mean"]), srv_mean=float.fromhex(case["srv_mean"]),
                         num_objects=case["num_objects"], master_seed=MASTER, model=model_id, servers=case["servers"],
                         variant=variant, trace_cap=TRACE if trace else 0, params=case["params"], queue_spill_cap=spill)


def compare(case, res, n):
    ev, ob = res.events.cpu().numpy(), res.objects.cpu().numpy()
    te, sw = res.t_end.cpu().numpy(), res.sum_wait.cpu().numpy()
    cnt = res.counters.cpu().numpy()
    tk = res.trace_key.cpu().numpy() if res.trace_key is not None else None
    tt = res.trace_time.cpu().numpy() if res.trace_time is not None else None
    assert (res.status.cpu().numpy()[:n] == 0).all(), res.status.cpu().numpy()[:n]
    for i, want in enumerate(case["trials"][:n]):
        check_trial(want, ev[i], ob[i], te[i], sw[i], cnt[i] if case["model"] in (7, 10, 16, 18, 19) + COVERAGE else None,
                    tk[i] if tk is not None else None, tt[i] if tt is not None else None, f"trial {i}",
                    max_queue=int(res.max_queue[i]) if case["model"] in (11, 12, 13, 14) else None)
        if case["model"] in (3, 4, 5, 6, 8):
            assert int(res.max_queue[i]) == want["max_fel"]


@pytest.mark.parametrize("case", [c for c in GOLD["cases"] if c["model"] in BUILTIN], ids=case_id)
def test_models_on_the_general_engine_match_the_reference_vectors(case):
    n = len(case["trials"])
    res = run_case(case, BUILTIN[case["model"]], cb.VARIANT_GENERAL if case["model"] not in (16, 18) else 0, n)
    compare(case, res, n)


@pytest.mark.parametrize("case", [c for c in GOLD["cases"] if c["model"] in (0, 1, 2, 9)], ids=case_id)
def test_default_kernels_with_their_repair_pass_match_the_reference_vectors(case):
    """variant 0 = the fast kernel; whatever it flags the repair pass re-runs.  The heavy-traffic, overload and
    64-server cases cannot be served by the fixed tables alone."""
    n = len(case["trials"])
    res = run_case(case, BUILTIN[case["model"]], 0, n)
    compare(case, res, n)


@pytest.mark.parametrize("case", [c for c in GOLD["cases"] if c["model"] == 0], ids=case_id)
def test_producer_consumer_variant_of_the_headline_kernel_matches_the_reference_vectors(case):
    """variant 2 of MODEL_MM1 (csrc/mm1_pc.cuh): the variates come from producer warps through shared-memory rings - same stream,
    same answers, pop traces included; flagged trials go to the repair pass like the default kernel's."""
    n = len(case["trials"])
    compare(case, run_case(case, cb.MODEL_MM1, 2, n), n)


def test_the_repair_pass_is_what_answers_in_overload():
    """At rho = 1.05 every trial outgrows the 32 + 512 entry queue: the diag counter shows the repair pass re-ran
    them all, and with a ring sized for the traffic the fast kernel keeps them (same answers either way)."""
    case = next(c for c in GOLD["cases"] if c["model"] == 0 and float.fromhex(c["arr_mean"]) < 1.0)
    n = len(case["trials"])
    dev = torch.device("cuda", torch.cuda.current_device())
    arr = torch.full((n,), float.fromhex(case["arr_mean"]), dtype=torch.float64, device=dev)
    srv = torch.full((n,), float.fromhex(case["srv_mean"]), dtype=torch.float64, device=dev)
    for spill, want_repairs in ((0, n), (4096, 0)):
        diag = torch.zeros(4, dtype=torch.int64, device=dev)
        res = cb.launch_trials(arr, srv, num_objects=case["num_objects"], master_seed=MASTER, queue_spill_cap=spill, diag=diag)
        torch.cuda.synchronize()
        assert int(diag[2].item()) == want_repairs
        compare(case, res, n)


def test_host_buffer_entry_point_returns_the_reference_answer_in_heavy_traffic():
    """cimba_b200_run_experiment at rho = 0.99: rc 0, no status bits, results as the reference's."""
    case = next(c for c in GOLD["cases"] if c["model"] == 0 and c["num_objects"] == 60000)
    n = len(case["trials"])
    exp = np.zeros(n, dtype=cb.TRIAL_DTYPE)
    exp["arr_mean"], exp["srv_mean"] = float.fromhex(case["arr_mean"]), float.fromhex(case["srv_mean"])
    cb.cimba_run_experiment(exp, num_objects=case["num_objects"], master_seed=MASTER)
    for i, want in enumerate(case["trials"]):
        assert (int(exp["events"][i]), int(exp["obj_cnt"][i])) == (want["events"], want["objects"])
        assert float(exp["t_end"][i]).hex() == want["t_end"] and float(exp["sum_wait"][i]).hex() == want["sum_wait"]
        assert exp["status"][i] == 0


def test_general_engine_against_the_oracle_at_other_sizes():
    """Beyond the stored vectors: ragged trial counts, a few thousand trials taken grid-stride, against the C oracle."""
    port = load_port()
    for model, servers, arr, srv, nobj, n in ((0, 1, 1 / 0.9, 1.0, 700, 3000), (2, 8, 1 / 6.4, 1.0, 500, 2500),
                                               (1, 1, 1.25, 1.0, 600, 1111)):
        res = cb.run_trials(n, arr_mean=arr, srv_mean=srv, num_objects=nobj, master_seed=MASTER, first_trial=5,
                            model=BUILTIN[model], servers=servers, variant=cb.VARIANT_GENERAL)
        want = run_trials(port, "port", model, servers, MASTER, 5, n, nobj, arr, srv)
        ev, te, sw = res.events.cpu().tolist(), res.t_end.cpu().tolist(), res.sum_wait.cpu().tolist()
        assert res.status.abs().sum().item() == 0
        for i, w in enumerate(want):
            assert (ev[i], te[i], sw[i]) == (w.events, w.t_end, w.sum_wait), (model, i)


@pytest.mark.parametrize("model,servers", [(3, 40), (3, 1000), (13, 64), (6, 33), (11, 200)])
def test_queue_capacities_the_round_one_tables_could_not_hold(model, servers):
    """Capacities beyond 16 (15 for the priority queue) used to be refused; they go to the general engine now."""
    port = load_port()
    n, dur = 64, 300
    res = cb.run_trials(n, arr_mean=0.5, srv_mean=1.0, num_objects=dur, master_seed=MASTER, model=BUILTIN[model], servers=servers)
    want = run_trials(port, "port", model, servers, MASTER, 0, n, dur, 0.5, 1.0)
    assert res.status.abs().sum().item() == 0
    ev, te, sw, cnt = res.events.cpu().tolist(), res.t_end.cpu().tolist(), res.sum_wait.cpu().tolist(), res.counters.cpu().numpy()
    for i, w in enumerate(want):
        assert (ev[i], te[i], sw[i]) == (w.events, w.t_end, w.sum_wait), (model, i)
        assert [int(v) & (2**64 - 1) for v in cnt[i]] == list(w.counter), (model, i)


def test_reneging_model_against_the_live_reference_build():
    """1200 processes per trial: events, clock, sums and counters as the reference's pthread executive computed them
    (tests/golden/reference_runs.json)."""
    g = RUNS["renege"]
    servers = g["servers"]
    res = cb.run_trials(g["count"], arr_mean=float.fromhex(g["arr_mean"]), srv_mean=float.fromhex(g["srv_mean"]),
                        num_objects=g["num_objects"], master_seed=MASTER, first_trial=g["first"], model=cb.MODEL_RENEGE,
                        servers=servers, params=g["params"])
    assert res.status.abs().sum().item() == 0
    ev, te, sw, cnt = res.events.cpu().tolist(), res.t_end.cpu().tolist(), res.sum_wait.cpu().tolist(), res.counters.cpu().tolist()
    assert ev == g["events"]
    assert result_digest([(ev[i], te[i], sw[i], *cnt[i][:4]) for i in range(g["count"])]) == g["sha256"]
    for i in range(g["count"]):
        assert cnt[i][6] == 1 and cnt[i][7] == servers          # the key map was in use; every process was created


def _model_library(stem):
    sys.path.insert(0, str(ROOT / "scripts"))
    so = ROOT / "cimba_b200/lib/models" / f"lib{stem}.so"
    if not so.exists():                                 # built by __graft_entry__.build(); nvcc is on the GPU box too
        import build_model
        build_model.build(ROOT / "examples" / f"{stem}.cu")
    return so


def test_a_user_built_model_library_loads_and_matches_the_builtin_model():
    mid = cb.load_model(_model_library("mm1_user_model"))
    assert mid >= cb.MODEL_USER_BASE and cb.lib.cimba_b200_model_name(mid) == b"mm1 (user build)"
    case = GOLD["cases"][0]
    n = len(case["trials"])
    compare(case, run_case(case, mid, 0, n), n)
    # ... and through the host-buffer entry point, like any built-in model
    exp = np.zeros(n, dtype=cb.TRIAL_DTYPE)
    exp["arr_mean"], exp["srv_mean"] = float.fromhex(case["arr_mean"]), float.fromhex(case["srv_mean"])
    cb.cimba_run_experiment(exp, model=mid, num_objects=case["num_objects"], master_seed=MASTER)
    assert [int(v) for v in exp["events"]] == [t["events"] for t in case["trials"]]


def test_a_model_that_exists_only_as_a_user_library_matches_the_reference():
    """examples/tandem_model.cuh: two stations, a bounded buffer, a put that blocks - nowhere in the library."""
    mid = cb.load_model(_model_library("tandem_user_model"))
    for case in [c for c in GOLD["cases"] if c["model"] == 17]:
        n = len(case["trials"])
        compare(case, run_case(case, mid, 0, n), n)


@pytest.mark.parametrize("case", [c for c in GOLD["cases"] if c["model"] in (0, 1, 9, 19)], ids=case_id)
def test_static_tier_matches_the_reference_vectors(case):
    """CIMBA_B200_VARIANT_STATIC: mm1_model.cuh / gg1_model.cuh - the text the general engine runs - compiled against
    cmb::StaticSim<2, 1> (registers + shared memory).  Heavy traffic and overload outgrow its 32 + 512 entry queue: those trials
    come back through the general engine from the same template, with the reference's answer."""
    n = len(case["trials"])
    compare(case, run_case(case, BUILTIN[case["model"]], cb.VARIANT_STATIC, n), n)
    compare(case, run_case(case, BUILTIN[case["model"]], cb.VARIANT_STATIC, n, spill=8192), n)


def test_static_tier_against_the_oracle_at_other_sizes():
    port = load_port()
    for model, arr, srv, nobj, n in ((0, 1 / 0.9, 1.0, 900, 3000), (1, 1.25, 1.0, 700, 1111), (0, 1 / 0.97, 1.0, 3000, 257)):
        res = cb.run_trials(n, arr_mean=arr, srv_mean=srv, num_objects=nobj, master_seed=MASTER, first_trial=9,
                            model=BUILTIN[model], variant=cb.VARIANT_STATIC)
        want = run_trials(port, "port", model, 1, MASTER, 9, n, nobj, arr, srv)
        ev, te, sw = res.events.cpu().tolist(), res.t_end.cpu().tolist(), res.sum_wait.cpu().tolist()
        assert res.status.abs().sum().item() == 0
        for i, w in enumerate(want):
            assert (ev[i], te[i], sw[i]) == (w.events, w.t_end, w.sum_wait), (model, i)


def test_user_built_static_tier_libraries_match_the_reference():
    """examples/tandem_static_user_model.cu (three processes, two queues, a put that blocks on the bounded one) and
    examples/mm1_static_user_model.cu: CMB_EXPORT_STATIC_MODEL, scripts/build_model.py, cimba_b200_model_load."""
    mid = cb.load_model(_model_library("tandem_static_user_model"))
    assert b"static tier" in cb.lib.cimba_b200_model_name(mid)
    for case in [c for c in GOLD["cases"] if c["model"] == 17]:
        n = len(case["trials"])
        compare(case, run_case(case, mid, 0, n), n)             # servers = 1, rho > 1: queue 1 outgrows the ring -> repaired
    mm1 = cb.load_model(_model_library("mm1_static_user_model"))
    case = GOLD["cases"][0]
    n = len(case["trials"])
    compare(case, run_case(case, mm1, 0, n), n)
    exp = np.zeros(n, dtype=cb.TRIAL_DTYPE)
    exp["arr_mean"], exp["srv_mean"] = float.fromhex(case["arr_mean"]), float.fromhex(case["srv_mean"])
    cb.cimba_run_experiment(exp, model=mm1, num_objects=case["num_objects"], master_seed=MASTER)
    assert [int(v) for v in exp["events"]] == [t["events"] for t in case["trials"]]


def test_tutorial_one_as_an_experiment_through_the_host_buffer_entry():
    """tutorial/tut_1_7.c: 39 utilisations x replications in ONE trial array, cimba_run_experiment over it, each trial's result
    the time-weighted mean queue length.  Here: the same array through cimba_b200_run_experiment (MODEL_TUTORIAL1, warm-up time in
    the descriptor's params), every trial's avg_queue_length bit-identical to the unmodified reference running the tutorial's trial
    (tests/golden/reference_runs.json: 39 utilisations x 2 replications, warm-up 100, 2000 time units)."""
    g = RUNS["tutorial1"]
    dt = np.dtype([("arr_mean", "<f8"), ("srv_mean", "<f8"), ("events", "<u8"), ("t_end", "<f8"), ("status", "<u4"), ("pad", "<u4"),
                   ("counters", "<u8", (8,))])
    exp = np.zeros(len(g["arr_means"]), dtype=dt)
    exp["arr_mean"], exp["srv_mean"] = [float.fromhex(a) for a in g["arr_means"]], 1.0
    cb.cimba_run_experiment(exp, model=cb.MODEL_TUTORIAL1, num_objects=g["num_objects"], master_seed=MASTER, params=[g["warmup"]])
    assert not exp["status"].any()
    assert [int(v) for v in exp["events"]] == g["events"]
    assert result_digest([(exp["events"][i], exp["t_end"][i], *exp["counters"][i]) for i in range(len(exp))]) == g["sha256"]
    mean_len = exp["counters"][:, 3].copy().view("<f8")
    assert mean_len[-1] > mean_len[0]                   # rho 0.975 queues more than rho 0.025


def test_theme_park_tutorial_on_device_matches_the_unmodified_tutorial_source():
    """MODEL_PARK = tutorial/tut_3_1.c on the general engine: 64 trials against the vectors of the unmodified tutorial source
    (tests/golden/park_vectors.json), and 300 more against the tutorial's results for them (tests/golden/reference_runs.json)."""
    import json
    gold = json.loads((ROOT / "tests/golden/park_vectors.json").read_text())
    n = len(gold["trials"])
    res = cb.run_trials(n, arr_mean=1.0, srv_mean=1.0, num_objects=0, master_seed=gold["master"], model=cb.MODEL_PARK)
    assert res.status.abs().sum().item() == 0
    ev, te, cnt = res.events.cpu().tolist(), res.t_end.cpu().tolist(), res.counters.cpu().numpy()
    for i, want in enumerate(gold["trials"]):
        means = [float(v).hex() for v in cnt[i][:5].copy().view("<f8")]
        assert (ev[i], float(te[i]).hex(), means) == (want["events"], want["t_end"], want["means"]), i
    g = RUNS["park"]
    res = cb.run_trials(g["count"], arr_mean=1.0, srv_mean=1.0, num_objects=0, master_seed=MASTER, first_trial=g["first"],
                        model=cb.MODEL_PARK)
    assert res.status.abs().sum().item() == 0
    ev, te, cnt = res.events.cpu().tolist(), res.t_end.cpu().tolist(), res.counters.cpu().numpy()
    assert ev == g["events"]
    assert result_digest([(ev[i], te[i], *cnt[i][:5].copy().view("<f8")) for i in range(g["count"])]) == g["sha256"]


def test_second_tutorial_on_device_matches_the_unmodified_tutorial_source():
    """MODEL_TUTORIAL2 = tutorial/tut_2_1.c on the general engine, trials of ~670 000 events each (the tutorial's length is hard-coded)
    against the vectors of the unmodified tutorial source: events executed, final clock, the random stream's position after the
    run.  Four trials here (one lane each of one warp: ~30 s); tests/test_cmb_engine.py holds the engine's host build to twelve."""
    import json
    gold = json.loads((ROOT / "tests/golden/tutorial2_vectors.json").read_text())
    n = 4
    res = cb.run_trials(n, arr_mean=1.0, srv_mean=1.0, num_objects=0, master_seed=gold["master"], model=cb.MODEL_TUTORIAL2)
    assert res.status.abs().sum().item() == 0
    ev, te, cnt = res.events.cpu().tolist(), res.t_end.cpu().tolist(), res.counters.cpu().numpy()
    for i, want in enumerate(gold["trials"][:n]):
        assert (ev[i], float(te[i]).hex(), int(cnt[i][0]) & (2**64 - 1)) == (want["events"], want["t_end"], want["next_raw"]), i


def test_unknown_model_ids_and_bad_libraries_are_refused():
    with pytest.raises(cb.CimbaError):
        cb.run_trials(4, arr_mean=1.0, srv_mean=1.0, num_objects=10, master_seed=1, model=cb.MODEL_USER_BASE + 999)
    with pytest.raises(cb.CimbaError):
        cb.load_model(ROOT / "oracle/liboracle_port.so")        # a library, but not a model


def test_resourcepool_golden_file_reproduced_on_device():
    """test/reference/resourcepool.txt on the GPU: the reference's own pool test (pre-emption, priority changes, interrupts,
    the holders' tie-break) on the general engine, seed 0x34f05c64d7ad598f, 20 units, 100 time units: the usage history's
    summary line as the reference prints it."""
    res = cb.run_trials(1, arr_mean=1.0, srv_mean=1.0, num_objects=100, master_seed=inverse_fmix64(0x34F05C64D7AD598F),
                        model=cb.MODEL_POOL_RECORDED, servers=20)
    assert int(res.status[0]) == 0
    counters = [int(v) & (2**64 - 1) for v in res.counters[0].cpu().tolist()]
    assert counters[0] == 120 and int(res.max_queue[0]) == 120
    assert wtdsummary_line(cb.lib, counters) == RESOURCEPOOL_GOLDEN_LINE

"""GPU tests of cmb_random_* at its edge parameters, and of the samplers a model writes with them, on both engines.

* cimba_b200_rng_draws / _ex on the device against what the unmodified reference drew (tests/golden/random_edges.json): bit
  for bit, NaN compared as NaN, wherever the variate is exact by construction.  Logistic, weibull and pareto, whose variate IS a
  log or pow result, are held to the high-precision bracket instead: the formula of distributions.cuh evaluated with a libm
  result within CUDA's documented bound of the exact value (1 ulp for log, 2 for pow), from the stream the variate consumes.
  Gamma with shape < 1 and what builds on it (chi-squared with k < 2, F, t) interleave the pow with other draws: compared with
  the port within a few ulp of the result, over all 65 536 variates - a stream that fell out of step (a different number of
  draws for one variate, a zero-valued chi-squared redrawn on one side only) would miss that by far from then on.
* tests/sampler_model.cuh built with scripts/build_model.py as a general-engine library and as a static-tier library: every
  sampler case at 1, 31, 33, 65 and 4096 trials from trial 5 (lanes park at different steps; both branches of the parked batch
  are taken), and through cimba_run_experiment.  The pop trace equals the engine's host build (held to the port's stream by
  tests/test_random_edges.py), and for the first trials the port's stream directly.

Nothing is launched before the host build has run every sampler case to the end, in a subprocess with a timeout: a sampler
that does not terminate there fails this module instead of running on the device.  Not compared, on purpose: see
tests/random_edges.py (out-of-range conversions to unsigned, probability tables that sum to less than 1)."""
import json
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

import sampler_cases as sc
from random_edges import BRACKETED, RECORDS, bracket_stream, bracket_violations, check_first8_and_digest, draws, \
    gamma_pow_kind, params_of, rec_id, same, ulp_distance

pytestmark = pytest.mark.gpu
COUNTS = (1, 31, 33, 65, 4096)


@pytest.fixture(scope="module", autouse=True)
def host_results(tmp_path_factory):
    """Every sampler case through the host build of the same text, both engines, every trial a device run below uses; the
    module stops here - before any launch - if that does not finish."""
    d = tmp_path_factory.mktemp("sampler_host")
    so = sc.build_host(d)
    out = d / "host.json"
    try:
        p = subprocess.run([sys.executable, "-s", str(sc.HERE / "sampler_cases.py"), str(so), str(out)],
                           timeout=sc.HOST_TIMEOUT_S, capture_output=True, text=True)
    except subprocess.TimeoutExpired:
        pytest.fail(f"a sampler did not terminate on the host build within {sc.HOST_TIMEOUT_S} s: not launched on the device")
    if p.returncode != 0:
        pytest.fail("the host build of the samplers failed; nothing launched on the device:\n" + p.stderr[-2000:])
    return json.loads(out.read_text())


# ---------------------------------------------------------------------------------------------------------- the stream kernels
def _device_draws(cb, rec):
    p = params_of(rec)
    if rec["kind"] <= 8:
        return cb.rng_draws(rec["seed"], rec["kind"], rec["n"], p[0], p[1]).cpu().numpy()
    return cb.rng_draws_ex(rec["seed"], rec["kind"], rec["n"], p).cpu().numpy()


@pytest.mark.parametrize("rec", RECORDS, ids=rec_id)
def test_device_streams_at_edge_parameters(cb, port, rec):
    kind, p = rec["kind"], params_of(rec)
    if kind in (26, 27, 33) and p[0] == 0:
        # n = 0 trials / m = 0 successes: the C-ABI takes params[0] as a count >= 1 and refuses the launch
        with pytest.raises(Exception):
            _device_draws(cb, rec)
        return
    dev = _device_draws(cb, rec)
    if kind in BRACKETED:
        stream = cb.rng_draws(rec["seed"], 1 if kind == 18 else 3, rec["n"], 1.0 if kind == 18 else 0.0, 0.0).cpu().numpy()
        assert same(stream, bracket_stream(port, "port", kind, rec["seed"], rec["n"])).all()
        bad = bracket_violations(kind, p, dev, stream, 1 if BRACKETED[kind] == "log" else 2)
        assert not bad, (rec_id(rec), bad[:5], dev[bad[:3]], stream[bad[:3]])
    elif gamma_pow_kind(kind, p):
        cpu = draws(port, "port", rec["seed"], kind, p, rec["n"])
        d = ulp_distance(dev, cpu)
        if kind == 22 and p[2] < 0.1:
            # t with v << 1: chi-squared(v) is often subnormal or zero (the t loop redraws it), so its few-ulp pow difference is
            # a large relative one after the division; a stream out of step would still differ by O(1)
            with np.errstate(invalid="ignore", divide="ignore"):
                rel = np.where(d == 0, 0.0, np.abs(dev - cpu) / np.maximum(np.abs(cpu), 1e-300))
            assert np.nanmax(rel) < 1e-2, (rec_id(rec), float(np.nanmax(rel)))
        else:
            assert d.max() <= 16, (rec_id(rec), float(d.max()), np.flatnonzero(d > 16)[:5])
        assert np.mean(d == 0) > 0.5, rec_id(rec)
    else:
        check_first8_and_digest(dev, rec, "device")


def test_the_zero_valued_chi_squared_loop_is_exercised(port):
    """t with v = 0.02 redraws its chi-squared while it is 0: make sure the fixture's case actually meets such zeros."""
    chi = draws(port, "port", RECORDS[0]["seed"], 20, [0.02], 65_536)
    assert (chi == 0.0).sum() >= 10


# ------------------------------------------------------------------------------------------------ samplers through cmb_device.cuh
@pytest.fixture(scope="module")
def sampler_libs(cb, tmp_path_factory):
    """tests/sampler_model.cuh as a user library twice: CMB_EXPORT_MODEL (general engine) and CMB_EXPORT_STATIC_MODEL with one
    process and no queue (static tier), built by scripts/build_model.py into a temporary directory."""
    sys.path.insert(0, str(sc.ROOT / "scripts"))
    import build_model
    d = tmp_path_factory.mktemp("sampler_dev")
    head = (f'#include "{sc.ROOT}/cimba_b200/csrc/cmb_launch.cuh"\n'
            f'#include "{sc.ROOT}/tests/sampler_model.cuh"\n')
    srcs = {"general": head + 'CMB_EXPORT_MODEL(cimba_b200::tests::SamplerT<cimba_b200::cmb::Sim>, "sampler test model")\n',
            "static": head + 'CMB_EXPORT_STATIC_MODEL(cimba_b200::tests::SamplerT, 1, 0, "sampler test model, static tier")\n'}
    for name, text in srcs.items():
        (d / f"sampler_{name}.cu").write_text(text)
    with ThreadPoolExecutor(2) as ex:
        libs = dict(zip(srcs, ex.map(lambda n: build_model.build(d / f"sampler_{n}.cu", d / f"libsampler_{n}.so"), srcs)))
    return {name: cb.load_model(path) for name, path in libs.items()}


def _device_trials(cb, mid, c, n):
    cap = c[3] + 1
    res = cb.run_trials(n, arr_mean=1.0, srv_mean=1.0, num_objects=c[3], master_seed=sc.MASTER, first_trial=sc.FIRST, model=mid,
                        trace_cap=cap, params=sc.model_params(c))
    st, ev, ob = res.status.cpu().numpy(), res.events.cpu().numpy(), res.objects.cpu().numpy()
    te, tt = res.t_end.cpu().numpy(), res.trace_time.cpu().numpy()
    return [[int(st[i]), int(ev[i]), int(ob[i]), float(te[i]).hex(), [float(x).hex() for x in tt[i][:min(cap, int(ev[i]))]]]
            for i in range(n)]


@pytest.mark.parametrize("case", sc.CASES, ids=sc.case_id)
def test_samplers_on_both_engines_match_the_host_build_and_the_port(cb, port, sampler_libs, host_results, case):
    want = host_results[case[0]]["0"]                   # the general engine's host build ...
    assert want == host_results[case[0]]["1"]           # ... which its static tier equals
    for n in COUNTS:
        for engine, mid in sampler_libs.items():
            got = _device_trials(cb, mid, case, n)
            bad = [i for i in range(n) if got[i] != want[i]]
            assert not bad, (case[0], engine, n, bad[:3], got[bad[0]][:4], want[bad[0]][:4])
    if case[4] is not None:                             # and the port's stream itself, for the first trials
        for i in range(33):
            ev, ob, t_end, trace = sc.expected_trial(port, case, port.port_fmix64(sc.MASTER, sc.FIRST + i))
            assert want[i] == [0, ev, ob, t_end.hex(), [t.hex() for t in trace]], (case[0], i)


@pytest.mark.parametrize("case", [c for c in sc.CASES if c[0] in ("exp_below_half_mean", "normal_m1_redrawn_while_negative",
                                                                   "normal_tail_only", "exp_tail_only", "composite_exp_plus_gamma",
                                                                   "poisson_500")], ids=sc.case_id)
def test_samplers_through_cimba_run_experiment(cb, sampler_libs, host_results, case):
    want = host_results[case[0]]["0"]
    n = 4096
    for engine, mid in sampler_libs.items():
        exp = np.zeros(n, dtype=cb.TRIAL_DTYPE)
        exp["arr_mean"], exp["srv_mean"] = 1.0, 1.0
        cb.cimba_run_experiment(exp, model=mid, num_objects=case[3], master_seed=sc.MASTER, first_trial=sc.FIRST,
                                params=sc.model_params(case))
        assert [int(v) for v in exp["status"]] == [0] * n, (case[0], engine)
        assert [int(v) for v in exp["events"]] == [w[1] for w in want], (case[0], engine)
        assert [float(v).hex() for v in exp["t_end"]] == [w[3] for w in want], (case[0], engine)

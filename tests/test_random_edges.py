"""CPU tests of cmb_random_* at its edge parameters, and of the samplers a model writes with them.

* The port (oracle/port) against what the unmodified reference drew at the same parameters (tests/golden/random_edges.json):
  every kind, two seeds, 65 536 variates, bit for bit with NaN compared as NaN.  Shapes of exactly 1 (where rnd_gamma changes
  branch), chi-squared with k < 2, F and t with one degree of freedom, a subnormal mean, lo == hi, p = 0 and 1, mode == min or
  max, a lognormal deep in glibc exp's underflow path, results that overflow to inf.
* Logistic, weibull and pareto, whose variate IS a log or pow result: each value is the formula of distributions.cuh evaluated
  with a libm result within 1 ulp of the exact one (mpmath), from the stream the variate consumes.
* tests/sampler_model.cuh, a process that holds for CMB_PROCESS_HOLD_SAMPLED, compiled for the CPU on the general engine and the
  static tier (tests/sampler_host.cpp): every pop time equals the running sum of the port's variates, truncated samplers
  included.  The static tier first tries a sampler with the ziggurats' rectangles only; a truncated sampler that rejects
  whatever such a failed try returned, or that can only be satisfied by a tail draw, used to loop forever there - run in a
  subprocess with a timeout, so that such a hang fails the test instead of stalling the suite.

Not compared, on purpose (see tests/random_edges.py and the header of cimba_b200/csrc/distributions.cuh): geometric with p = 0
or with p so small that the count exceeds 2^32, and the negative binomial on it - the reference converts an out-of-range double
to unsigned, undefined in C, where x86 wraps and sm_100 saturates; hyper-exponential and loaded dice whose probabilities sum to
less than 1 - the reference indexes past its table."""
import json
import subprocess
import sys

import numpy as np
import pytest

import sampler_cases as sc
from random_edges import BRACKETED, EXCLUDED, FIXTURE, RECORDS, bracket_stream, bracket_violations, check_first8_and_digest, \
    draws, params_of, rec_id
from oracle_libs import load_port


def test_fixture_covers_two_seeds_per_case_and_lists_its_exclusions():
    assert FIXTURE["n"] % 64 == 0 and len(FIXTURE["seeds"]) == 2
    per = {}
    for r in RECORDS:
        per.setdefault((r["kind"], tuple(r["params"])), set()).add(r["seed"])
    assert all(s == set(FIXTURE["seeds"]) for s in per.values())
    kinds = {k for k, _ in per}
    assert {1, 4, 5, 6, 7, 8, 9, 10, 11, 12, 15, 16, 17, 18, 19, 20, 21, 22, 23, 25, 26, 27, 28, 29, 30, 31, 32, 33} <= kinds
    # no case of the fixture is one of the documented exclusions
    for (kind, par) in per:
        p = [float.fromhex(v) for v in par]
        if kind == 25:
            assert 1e-9 < p[0] <= 1.0
        if kind in (27, 33):
            assert 1e-9 < p[1] <= 1.0
        if kind == 29:
            assert sum(p[1:1 + int(p[0])]) == 1.0
    assert len(EXCLUDED) == 5


@pytest.mark.parametrize("rec", RECORDS, ids=rec_id)
def test_port_matches_the_reference_at_edge_parameters(port, rec):
    v = draws(port, "port", rec["seed"], rec["kind"], params_of(rec), rec["n"])
    check_first8_and_digest(v, rec, "port")


@pytest.mark.parametrize("rec", [r for r in RECORDS if r["kind"] in BRACKETED], ids=rec_id)
def test_port_log_and_pow_variates_within_one_ulp_of_the_exact_value(port, rec):
    """glibc's log and pow are within 1 ulp (the port links them): the bracket must hold for every variate."""
    p = params_of(rec)
    v = draws(port, "port", rec["seed"], rec["kind"], p, rec["n"])
    stream = bracket_stream(port, "port", rec["kind"], rec["seed"], rec["n"])
    bad = bracket_violations(rec["kind"], p, v, stream, 1)
    assert not bad, (rec_id(rec), bad[:5], v[bad[:3]], stream[bad[:3]])


def test_bracket_rejects_a_variate_two_ulp_off(port):
    """The bracket is tight enough to notice: move one pareto variate by 2 ulp and it fails there."""
    rec = [r for r in RECORDS if r["kind"] == 19 and params_of(r)[0] == 1e3][0]
    p = params_of(rec)
    v = draws(port, "port", rec["seed"], 19, p, 64)
    stream = bracket_stream(port, "port", 19, rec["seed"], 64)
    v[7] = np.nextafter(np.nextafter(v[7], np.inf), np.inf)
    assert bracket_violations(19, p, v, stream, 1) == [7]


# ------------------------------------------------------------------------------------------ samplers on the engine's host build
@pytest.fixture(scope="module")
def host_so(tmp_path_factory):
    return sc.build_host(tmp_path_factory.mktemp("sampler"))


def _run_in_subprocess(so, out, timeout):
    return subprocess.run([sys.executable, "-s", str(sc.HERE / "sampler_cases.py"), str(so), str(out)], timeout=timeout,
                          capture_output=True, text=True)


@pytest.fixture(scope="module")
def host_results(host_so, tmp_path_factory):
    """Every case on both engines of the host build, trials FIRST .. FIRST + 4095, in a subprocess: a sampler that does not
    terminate fails here, by the timeout."""
    out = tmp_path_factory.mktemp("sampler_out") / "host.json"
    try:
        p = _run_in_subprocess(host_so, out, sc.HOST_TIMEOUT_S)
    except subprocess.TimeoutExpired:
        pytest.fail(f"the host build did not finish every sampler case within {sc.HOST_TIMEOUT_S} s")
    assert p.returncode == 0, p.stderr[-2000:]
    return json.loads(out.read_text())


def test_truncated_samplers_terminate_on_the_static_tier(host_so, tmp_path):
    """The static tier's host build must finish truncated samplers - exponential redrawn while > mean / 2, normal(-1, 0.5) redrawn
    while negative, and two that only a ziggurat tail can satisfy - as the reference does.  Before the fix it never finished the
    first trial of any of them (a failed rectangles-only try returned a constant the sampler rejected, forever)."""
    code = ("import sys; sys.path.insert(0, %r); import sampler_cases as sc\n"
            "f = sc.load_host(%r)\n"
            "for c in sc.TRUNCATED:\n"
            "    r = sc.run_host(f, 1, c, sc.FIRST, 64)\n"
            "    assert all(x[0] == 0 and x[1] == c[3] + 1 for x in r), c[0]\n") % (str(sc.HERE), str(host_so))
    try:
        p = subprocess.run([sys.executable, "-s", "-c", code], timeout=60, capture_output=True, text=True)
    except subprocess.TimeoutExpired:
        pytest.fail("a truncated sampler did not terminate on the static tier's host build within 60 s")
    assert p.returncode == 0, p.stderr[-2000:]


def test_tail_thresholds_lie_beyond_the_rectangles():
    """The tail-only samplers' thresholds are just above the largest value each ziggurat's rectangles can give, and below what its
    tail gives (the exponential tail starts at ZIG_EXP_TAIL, the normal one at ZIG_NOR_TAIL)."""
    assert sc.EXP_HOT_MAX < sc.EXP_TAIL_R < sc.EXP_HOT_MAX * (1 + 1e-9)
    assert sc.NOR_HOT_MAX < sc.NOR_TAIL_R < sc.NOR_HOT_MAX * (1 + 1e-9)
    assert abs(sc.EXP_HOT_MAX - 7.56927469414779) < 1e-12 and abs(sc.NOR_HOT_MAX - 3.6360066255010701) < 1e-12


@pytest.mark.parametrize("case", [c for c in sc.CASES if c[4] is not None], ids=sc.case_id)
def test_sampler_pop_times_are_the_running_sums_of_the_port_stream(host_results, case):
    port = load_port()
    res = host_results[case[0]]
    for i in list(range(65)) + list(range(4031, 4096)):
        seed = port.port_fmix64(sc.MASTER, sc.FIRST + i)
        ev, ob, t_end, trace = sc.expected_trial(port, case, seed)
        want = [0, ev, ob, t_end.hex(), [t.hex() for t in trace]]
        for engine in ("0", "1"):
            assert res[engine][i] == want, (case[0], "engine", engine, "trial", sc.FIRST + i)


def test_composite_sampler_static_tier_equals_general_engine(host_results):
    """exponential(a) + gamma(2, b): a rectangles-only draw, then one with its slow paths inline.  No single port stream gives
    it, so the general engine (pinned to the reference elsewhere) is the oracle here."""
    res = host_results["composite_exp_plus_gamma"]
    assert all(r[0] == 0 and r[1] == 25 for r in res["0"])
    assert res["1"] == res["0"]


def test_every_case_ran_on_both_engines_without_a_flag(host_results):
    for c in sc.CASES:
        for engine in ("0", "1"):
            assert len(host_results[c[0]][engine]) == sc.HOST_TRIALS
            assert all(r[0] == 0 and r[1] == c[3] + 1 for r in host_results[c[0]][engine]), (c[0], engine)

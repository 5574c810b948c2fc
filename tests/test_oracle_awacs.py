"""CPU tests of the AWACS oracle (tutorial/tut_5_1.c, BASELINE config 5): the plain-C restatement
(oracle/port/awacs_port.c) against vectors the UNMODIFIED tutorial source compiled behind a stub hdf5.h
(oracle/_ref/libawacs_ref.so) produced (tests/golden/awacs_vectors.json, tests/golden/make_golden.py --only-awacs;
tests/golden/reference_runs.json, tests/golden/make_reference_runs.py)."""
import ctypes as C
import hashlib
import json
from pathlib import Path

import numpy as np
import pytest

from oracle_libs import (AWACS_TERRAIN_SEED, awacs_terrain, awacs_trial, load_port, reference_runs, result_digest)

GOLD = json.loads((Path(__file__).parent / "golden/awacs_vectors.json").read_text())
RUNS = reference_runs()


@pytest.fixture(scope="module")
def port():
    return load_port()


@pytest.fixture(scope="module")
def port_terrain(port):
    g = GOLD["terrain"]
    return awacs_terrain(port, "port", AWACS_TERRAIN_SEED, g["width_nm"], g["height_nm"])


def test_port_terrain_matches_the_reference_vectors(port_terrain):
    m, cols, rows, geom = port_terrain
    g = GOLD["terrain"]
    assert (cols, rows) == (g["cols"], g["rows"])
    assert [float(v).hex() for v in geom] == g["geom"]
    assert hashlib.sha256(m.tobytes()).hexdigest() == g["map_sha256"]


def test_threaded_terrain_generation_gives_the_same_map(port, port_terrain):
    g = GOLD["terrain"]
    m, cols, rows, geom = awacs_terrain(port, "port", AWACS_TERRAIN_SEED, g["width_nm"], g["height_nm"], threads=5)
    assert (cols, rows) == port_terrain[1:3] and np.array_equal(geom, port_terrain[3])
    assert np.array_equal(m.view(np.uint32), port_terrain[0].view(np.uint32))


@pytest.mark.parametrize("case", GOLD["trials"], ids=lambda c: f"seed{c['seed']}")
def test_port_trial_matches_the_reference_vectors(port, port_terrain, case):
    out, keys, times, per = awacs_trial(port, "port", case["seed"], GOLD["duration_h"], port_terrain, trace_cap=4000)
    assert out.events == case["events"] and out.t_end.hex() == case["t_end"] and out.num_found == case["num_found"]
    assert list(out.tds_count) == case["tds_count"] and list(out.mode_count) == case["mode_count"]
    assert out.sum_x.hex() == case["sum_x"] and out.sum_y.hex() == case["sum_y"]
    trace = hashlib.sha256(np.array(keys, dtype=np.uint64).tobytes() + np.array(times, dtype=np.float64).tobytes())
    assert trace.hexdigest() == case["trace_sha256"]
    assert hashlib.sha256(np.array(per["tds"], dtype=np.int32).tobytes()).hexdigest() == case["tds_sha256"]


def test_port_platform_state_matches_the_reference_vectors(port):
    six, r = (C.c_float * 6)(), C.c_float()
    for t, want in GOLD["platform"].items():
        port.port_awacs_platform_state(C.c_double(float(t)), six, C.byref(r))
        assert [float(v).hex() for v in six] + [float(r.value).hex()] == want


@pytest.fixture(scope="module")
def small_terrain(port):
    g = RUNS["awacs_terrain"]
    return awacs_terrain(port, "port", g["seed"], g["width_nm"], g["height_nm"])


def test_port_matches_the_live_reference_build(port, small_terrain):
    """A second terrain and two more trials (pop traces, every target's detect state, mode and position) as the
    reference computed them (tests/golden/make_reference_runs.py)."""
    m, cols, rows, geom = small_terrain
    g = RUNS["awacs_terrain"]
    assert (cols, rows) == (g["cols"], g["rows"]) and [float(v).hex() for v in geom] == g["geom"]
    assert result_digest([m.view(np.uint32)]) == g["map_sha256"]
    for want in RUNS["awacs_trials"]:
        po, pk, ptm, pper = awacs_trial(port, "port", want["seed"], want["hours"], small_terrain, trace_cap=want["trace_cap"])
        assert po.events == want["events"][0] and result_digest([po.row()]) == want["sha256"]
        assert result_digest(zip(pk, ptm)) == want["trace_sha256"]
        targets = zip(pper["tds"], pper["detected"], pper["mode"], pper["x"].view(np.uint32))
        assert result_digest(targets) == want["targets_sha256"]


def test_reference_executive_runs_awacs_trials_in_parallel(port, small_terrain):
    """cimba_run_experiment over the tutorial's run_trial (all host cores) gave what one-at-a-time runs give when the
    vectors were made; the port's trials give the same."""
    g = RUNS["awacs_executive"]
    outs = [awacs_trial(port, "port", port.port_fmix64(RUNS["master"], g["first"] + i), g["hours"], small_terrain)[0]
            for i in range(g["count"])]
    assert [o.events for o in outs] == g["events"] and result_digest([o.row() for o in outs]) == g["sha256"]

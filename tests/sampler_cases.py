"""Shared by tests/test_random_edges.py (CPU) and tests/test_gpu_random_edges.py (GPU): the samplers of tests/sampler_model.cuh,
their host build (tests/sampler_host.cpp) and what each trial must produce.

The oracle is the port's variate stream (oracle/port): every hold of a trial lasts |the next variate of one kind| at the trial's
seed fmix64(master, first + i), or for a truncated sampler the next one its acceptance test passes.  So the pop trace of a trial
is the running sum t_k = t_(k-1) + d_k, t_0 = 0 (the process's start), and the trial ends at t_N after N + 1 pops.

Run as a program (`python sampler_cases.py LIB OUT.json`), it runs every case through the host build's static tier and general
engine and writes what they returned: the GPU module runs that in a subprocess with a timeout before it launches anything, so that a
sampler that does not terminate on the CPU is never launched on a device."""
import ctypes as C
import json
import re
import subprocess
import sys
from pathlib import Path

HERE = Path(__file__).resolve().parent
ROOT = HERE.parent
MASTER = 0x34F05C64D7AD598F
FIRST = 5                       # trials FIRST .. FIRST + HOST_TRIALS - 1 cover every device run
HOST_TRIALS = 4096
HOST_TIMEOUT_S = 300            # what the host build needs for all of them is a few seconds

# tests/sampler_model.cuh SAMPLER_*
EXP_BELOW, NORMAL_ABOVE, EXP_ABOVE, EXPONENTIAL, NORMAL, ERLANG, GAMMA, BETA, PERT, LOGNORMAL, POISSON, TRIANGULAR, RAYLEIGH, \
    UNIFORM, DICE, BERNOULLI, COMPOSITE = range(17)


def _zig_hot_bounds():
    """The largest variate the rectangles of each ziggurat can give (rng.cuh exp_hot, draw_std_normal's hot branch): a bound
    times the widest layer, the full 64-bit (exponential) or signed 63-bit (normal) integer converted to double."""
    text = (ROOT / "cimba_b200/csrc/zig_tables.cuh").read_text()

    def table(name):
        body = re.search(name + r"\[256\] = \{([^}]*)\}", text).group(1)
        return [float(v) for v in body.replace("\n", " ").split(",") if v.strip()]

    exp_max = int(re.search(r"#define ZIG_EXP_MAX (\d+)u", text).group(1))
    nor_max = int(re.search(r"#define ZIG_NOR_MAX (\d+)u", text).group(1))
    e = max(x * float(2**64 - 1) for x in table("zig_exp_x")[:exp_max + 1])
    n = max(x * float(2**63 - 1) for x in table("zig_nor_x")[:nor_max + 1])
    return e, n


EXP_HOT_MAX, NOR_HOT_MAX = _zig_hot_bounds()
# just beyond the last rectangle: only a slow-path draw (the tail) can pass these
EXP_TAIL_R = EXP_HOT_MAX * (1 + 2**-40)
NOR_TAIL_R = NOR_HOT_MAX * (1 + 2**-40)

# name, sampler params (params[1..] of the model), holds per trial, port stream (kind, params), acceptance test
# port kinds 1..8 go through *_rng_draws(p0, p1), 9..33 through *_rng_draws_ex(params)
CASES = [
    ("exp_below_half_mean", EXP_BELOW, [3.0, 0.5], 24, (1, [3.0, 0.0]), lambda v: not (v > 0.5 * 3.0)),
    ("normal_m1_redrawn_while_negative", NORMAL_ABOVE, [-1.0, 0.5, 0.0], 16, (4, [-1.0, 0.5]), lambda v: not (v < 0.0)),
    ("normal_tail_only", NORMAL_ABOVE, [0.0, 1.0, NOR_TAIL_R], 3, (4, [0.0, 1.0]), lambda v: not (v < NOR_TAIL_R)),
    ("exp_tail_only", EXP_ABOVE, [1.0, EXP_TAIL_R], 3, (1, [1.0, 0.0]), lambda v: not (v < EXP_TAIL_R)),
    ("exponential_1e-300", EXPONENTIAL, [1e-300], 24, (1, [1e-300, 0.0]), None),
    ("exponential_1e300", EXPONENTIAL, [1e300], 24, (1, [1e300, 0.0]), None),
    ("normal_sigma0", NORMAL, [2.5, 0.0], 24, (4, [2.5, 0.0]), None),
    ("normal_sigma_negative", NORMAL, [1.0, -2.0], 24, (4, [1.0, -2.0]), None),
    ("erlang_k1", ERLANG, [1, 0.75], 24, (5, [1, 0.75]), None),
    ("erlang_k7", ERLANG, [7, 0.25], 24, (5, [7, 0.25]), None),
    ("gamma_shape1", GAMMA, [1.0, 2.0], 24, (15, [1.0, 2.0]), None),
    ("gamma_shape3", GAMMA, [3.0, 0.5], 24, (15, [3.0, 0.5]), None),
    ("gamma_scale_1e-300", GAMMA, [1e3, 1e-300], 24, (15, [1e3, 1e-300]), None),
    ("beta_a1_b1", BETA, [1.0, 1.0, 0.0, 2.0], 24, (16, [1.0, 1.0, 0.0, 2.0]), None),
    ("beta_a_half", BETA, [0.5, 2.0, 1.0, 3.0], 24, (16, [0.5, 2.0, 1.0, 3.0]), None),
    ("pert_mode_min", PERT, [1.0, 1.0, 4.0], 24, (17, [1.0, 1.0, 4.0]), None),
    ("pert_mode_max", PERT, [1.0, 4.0, 4.0], 24, (17, [1.0, 4.0, 4.0]), None),
    ("lognormal", LOGNORMAL, [0.25, 0.5], 24, (10, [0.25, 0.5]), None),
    ("lognormal_s0", LOGNORMAL, [0.75, 0.0], 24, (10, [0.75, 0.0]), None),
    ("lognormal_m_minus740", LOGNORMAL, [-740.0, 1.0], 24, (10, [-740.0, 1.0]), None),
    ("poisson_1e-3", POISSON, [1e-3], 24, (28, [1e-3]), None),
    ("poisson_500", POISSON, [500.0], 8, (28, [500.0]), None),
    ("triangular_mode_min", TRIANGULAR, [0.5, 0.5, 2.0], 24, (9, [0.5, 0.5, 2.0]), None),
    ("triangular_mode_max", TRIANGULAR, [0.5, 2.0, 2.0], 24, (9, [0.5, 2.0, 2.0]), None),
    ("rayleigh", RAYLEIGH, [1.5], 24, (23, [1.5]), None),
    ("rayleigh_scale0", RAYLEIGH, [0.0], 24, (23, [0.0]), None),
    ("uniform", UNIFORM, [0.25, 3.0], 24, (6, [0.25, 3.0]), None),
    ("uniform_lo_eq_hi", UNIFORM, [1.5, 1.5], 24, (6, [1.5, 1.5]), None),
    ("uniform_lo_gt_hi", UNIFORM, [3.0, -1.0], 24, (6, [3.0, -1.0]), None),
    ("dice", DICE, [1, 6], 24, (7, [1, 6]), None),
    ("dice_lo_eq_hi", DICE, [4, 4], 24, (7, [4, 4]), None),
    ("bernoulli_p0", BERNOULLI, [0.0], 24, (8, [0.0, 0.0]), None),
    ("bernoulli_p1", BERNOULLI, [1.0], 24, (8, [1.0, 0.0]), None),
    ("bernoulli_half", BERNOULLI, [0.5], 24, (8, [0.5, 0.0]), None),
    # the rectangles-only exponential, then a gamma with its slow paths inline: no single port stream; the general engine is the oracle
    ("composite_exp_plus_gamma", COMPOSITE, [1.0, 0.5], 24, None, None),
]
TRUNCATED = [c for c in CASES if c[5] is not None]


def case_id(c):
    return c[0]


def model_params(c):
    return [float(c[1]), *[float(v) for v in c[2]]]


class HostResult(C.Structure):
    _fields_ = [("events", C.c_uint64), ("objects", C.c_uint64), ("t_end", C.c_double), ("sum_wait", C.c_double),
                ("max_fel", C.c_uint64), ("max_queue", C.c_uint64), ("counter", C.c_uint64 * 8), ("status", C.c_uint32),
                ("pad", C.c_uint32)]


def build_host(out_dir: Path) -> Path:
    so = Path(out_dir) / "libsampler_host.so"
    subprocess.run(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-Wall", "-Wno-unknown-pragmas", "-Wno-unused-function",
                    "-shared", "-fPIC", str(HERE / "sampler_host.cpp"), "-o", str(so)], check=True, capture_output=True)
    return so


def load_host(so):
    f = C.CDLL(str(so)).host_sampler_run_trials
    f.restype = C.c_int
    f.argtypes = [C.c_int, C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint64, C.POINTER(C.c_double), C.c_uint32, C.c_uint64,
                  C.POINTER(C.c_uint64), C.POINTER(C.c_double), C.POINTER(HostResult)]
    return f


def run_host(f, engine, c, first, count, master=MASTER):
    """engine 0 = general, 1 = static tier: [(status, events, objects, t_end, [trace times])] per trial"""
    nobj = c[3]
    cap = nobj + 1
    par = model_params(c)
    out = (HostResult * count)()
    keys = (C.c_uint64 * (count * cap))()
    times = (C.c_double * (count * cap))()
    rc = f(engine, master, first, count, nobj, (C.c_double * len(par))(*par), len(par), cap, keys, times, out)
    assert rc == 0
    return [(o.status, o.events, o.objects, o.t_end, list(times[i * cap:i * cap + min(cap, o.events)])) for i, o in enumerate(out)]


def port_durations(port, c, seed):
    """The hold durations of one trial: |variate| for the first num_objects variates of the case's port stream that its
    acceptance test passes."""
    from oracle_libs import rng_draws, rng_draws_ex
    kind, kp = c[4]
    nobj, accept = c[3], c[5]
    n = 64 * max(1, (nobj + 63) // 64)
    while True:
        if kind <= 8:
            vals = rng_draws(port, "port", seed, kind, float(kp[0]), float(kp[1]), n)
        else:
            vals = rng_draws_ex(port, "port", seed, kind, kp, n)
        kept = [float(v) for v in vals if accept is None or accept(float(v))]
        if len(kept) >= nobj:
            return [abs(v) for v in kept[:nobj]]
        n *= 4


def expected_trial(port, c, seed):
    """(events, objects, t_end, trace times) of one trial, from the port's stream"""
    t, trace = 0.0, [0.0]
    for d in port_durations(port, c, seed):
        t = t + d
        trace.append(t)
    return c[3] + 1, c[3], t, trace


def main(argv):
    so, out = argv[1], argv[2]
    f = load_host(so)
    res = {}
    for c in CASES:
        res[c[0]] = {str(engine): [[s, e, o, t.hex(), [x.hex() for x in tr]] for s, e, o, t, tr in run_host(f, engine, c, FIRST, HOST_TRIALS)]
                     for engine in (0, 1)}
    Path(out).write_text(json.dumps(res))
    return 0


if __name__ == "__main__":
    sys.exit(main(sys.argv))

#!/usr/bin/env python3
"""bench.py - M/M/1 replication benchmark (BASELINE.json metric) on N B200s, plus the other BASELINE configs.

One "step" = one pass of the hot path over one batch: every rank runs `--trials` independent M/M/1 replications of
`--objects` customers each (benchmark/MM1_multi.c with NUM_TRIALS = 65536, rho = 0.9 as the reference file has it) in
ONE launch of the persistent simulation kernel (+ the repair pass behind it, which finds nothing to do at this load).
Weak scaling: per-GPU work is fixed, rank r runs global trial indices [r T, (r + 1) T); no data-path collective.
Every step runs the same seeds (cmb_random_fmix64(master, global trial index)): the answer of step k is the answer of
step 0, which is what lets the same trials be checked against the CPU reference inside this run.

  value     FEL pops ("events" = cmb_event_execute_next() calls) per second, all ranks, device-resident inputs,
            CUDA-event timed, max over ranks.
  e2e       the same through the host-buffer C-ABI entry (cimba_b200_run_experiment: pinned staging, H2D, kernel,
            D2H inside the timed region) and, at N > 1, the NCCL all-gather + cmb_datasummary merge of the per-rank
            summaries inside it too.
  roofline  bound = "issue": this kernel keeps a trial's whole state on chip (DRAM traffic ~0.1 B/event, reported as
            `traffic`), so what binds it is SM instruction issue.  achieved = warp-instructions issued per second =
            the kernel's own count of event-loop iterations (job.diag, added up by the kernel in this very run) x the
            loop's instruction count (calibrated once against ncu smsp__inst_executed.sum,
            profiles/issue_calibration.json) / the launch's CUDA-event time; peak = 4 schedulers x SMs x the SM clock
            nvidia-smi reported DURING the timed region.  The HBM figure SURVEY.md section 8d defines (72 B/event
            algorithmic against the measured copy peak) stays beside it under "hbm".
  cpu_baseline / --impl reference
            the reference's own pthread executive (oracle/_ref, unmodified sources) running the STOCK benchmark
            bodies (no per-event bookkeeping: oracle/ref_build/ref_driver.c ref_bench_trials) on this box's host
            cores, on a bounded sample of the same trials.  `cores` is what the process may actually use
            (scheduler affinity and the cgroup CPU quota), `threads` what cimba_run_experiment starts (one per
            logical CPU it sees, src/cimba.c:171) - on a quota-limited box they differ and the line says so.
  secondary one entry per other BASELINE configuration (rho = 0.8; config 3 M/M/c c = 8; config 4 G/G/1 at
            1 048 576 replications; config 5 AWACS, short; the hold model; M/M/1 and G/G/1 from their authoring-surface
            source on the static tier; M/M/1 on the general engine), each timed
            the same way on this run's GPUs with its own parity sample against the reference build, and the
            single-core benchmark/MM1_single.c row.
  --dump-outputs DIR
            the per-trial results of the last timed step (what launch_trials returns: events, objects, t_end, sum_wait,
            status, max_queue, counters) as DIR/<name>.npy in float64.  The same arguments give the same inputs on
            every run, so two builds of the project can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.dont_write_bytecode = True                 # the benchmark writes nothing into the tree it runs from
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))

MASTER_SEED = 0x34F05C64D7AD598F
ARRIVAL_RATE, SERVICE_RATE = 0.9, 1.0          # benchmark/MM1_multi.c:27-28
BYTES_PER_EVENT = 72.0                         # SURVEY.md section 8d (packed layout)
BYTES_PER_EVENT_REFLAYOUT = 150.9              # same, reference record layout


def parse_args():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=3)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--impl", default="native", choices=["native", "reference"])
    p.add_argument("--trials", type=int, default=65536, help="replications per GPU per step")
    p.add_argument("--objects", type=int, default=1_000_000, help="customers per replication")
    p.add_argument("--mapping", type=int, default=1, choices=[1, 32], help="1 lane/trial or 32 (warp/trial)")
    p.add_argument("--variant", type=int, default=0, help="0 default kernel, 1 unfused formulation, 16 general engine, 17 static tier (A/B)")
    p.add_argument("--ref-trials", type=int, default=0, help="CPU sample size (0 = 16 per usable core)")
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--no-e2e", action="store_true")
    p.add_argument("--no-secondary", action="store_true")
    p.add_argument("--single-process", action="store_true",
                   help="time cimba_b200_run_experiment_all_gpus (one host thread per GPU in THIS process) over --gpus GPUs")
    p.add_argument("--dump-outputs", metavar="DIR",
                   help="write the per-trial results of the last timed step to DIR/<name>.npy (float64)")
    return p.parse_args()


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(res, out_dir: str, rank: int, world: int) -> None:
    """The arrays launch_trials hands its caller (TrialResults), as float64 .npy files, so that two builds can be
    compared output for output.  Above DUMP_LIMIT_BYTES in all, a fixed seeded sample of trials is written, with
    the trial indices beside it (trial_index.npy)."""
    import numpy as np
    arrays = {name: getattr(res, name).double().cpu().numpy()
              for name in ("events", "objects", "t_end", "sum_wait", "status", "max_queue", "counters")}
    n = len(arrays["events"])
    per_trial = sum(a[0].nbytes for a in arrays.values())
    if n * per_trial > DUMP_LIMIT_BYTES:
        keep = np.sort(np.random.default_rng(0).choice(n, (DUMP_LIMIT_BYTES - 65536) // (per_trial + 8), replace=False))
        arrays = {name: a[keep] for name, a in arrays.items()}
        arrays["trial_index"] = keep.astype(np.float64)
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    suffix = f"_rank{rank}" if world > 1 else ""
    for name, a in arrays.items():
        np.save(out / f"{name}{suffix}.npy", a)


# ------------------------------------------------------------------------------------------------ host facts
def usable_cpus():
    """What this process may actually use: scheduler affinity capped by the cgroup CPU quota (v2 cpu.max, v1 cfs)."""
    try:
        affinity = len(os.sched_getaffinity(0))
    except Exception:
        affinity = os.cpu_count() or 1
    quota = None
    try:
        q, per = Path("/sys/fs/cgroup/cpu.max").read_text().split()
        if q != "max":
            quota = int(q) / int(per)
    except Exception:
        try:
            q = int(Path("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read_text())
            per = int(Path("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read_text())
            if q > 0:
                quota = q / per
        except Exception:
            pass
    cores = affinity if quota is None else max(1, min(affinity, int(round(quota))))
    return {"cores": cores, "logical": os.cpu_count() or 1, "affinity": affinity, "cgroup_quota": quota}


def measured_traffic():
    """DRAM bytes per event of the timed kernel from the committed ncu capture (profiles/traffic.json:
    dram__bytes_read.sum + dram__bytes_write.sum of the bench's own launch); None if absent."""
    try:
        return json.loads((ROOT / "profiles" / "traffic.json").read_text())
    except Exception:
        return None


def issue_calibration():
    """warp-instructions per event-loop iteration of each fast kernel, calibrated against ncu
    (scripts/calibrate_issue.py -> profiles/issue_calibration.json)."""
    try:
        return json.loads((ROOT / "profiles" / "issue_calibration.json").read_text())
    except Exception:
        return {}


def measured_peak_gbs():
    f = ROOT / "MEASURED_PEAKS.json"
    if f.exists():
        try:
            return float(json.loads(f.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                 "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm = sorted(int(float(r[1])) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit())
        mx = [int(float(r[2])) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            if len(r) >= 9:
                for nm, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------ the CPU reference
def cpu_reference_run(trials: int, objects: int, first: int = 0, model: int = 0, servers: int = 1,
                      arr_mean: float = 1.0 / ARRIVAL_RATE, srv_mean: float = 1.0 / SERVICE_RATE, threads: int = 0):
    """Time the reference's own CPU path on `trials` replications of model 0 (M/M/1), 1 (G/G/1) or 2 (M/M/c): the
    stock benchmark bodies through cimba_run_experiment (threads = 0: all logical cores) or serially (threads = 1);
    falls back to the plain-C oracle port where oracle/_ref did not travel."""
    import ctypes as C
    from oracle_libs import Result, load_port, load_ref, run_trials
    ref = load_ref()
    host = usable_cpus()
    if ref is not None and hasattr(ref, "ref_bench_trials"):
        f = ref.ref_bench_trials
        f.restype = C.c_int
        f.argtypes = [C.c_int, C.c_int, C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint64, C.c_double, C.c_double, C.c_int,
                      C.POINTER(Result)]
        res = (Result * trials)()
        t0 = time.perf_counter()
        rc = f(model, servers, MASTER_SEED, first, trials, objects, arr_mean, srv_mean, threads, res)
        dt = time.perf_counter() - t0
        assert rc == 0
        kind = "reference"
        nthreads = 1 if threads == 1 else ref.ref_cpu_cores()
        body = "stock benchmark bodies + cmb_event_queue_execute() (oracle/ref_build/ref_driver.c ref_bench_trials)"
    else:
        port = load_port()
        nthreads = 1 if threads == 1 else host["cores"]
        t0 = time.perf_counter()
        res = run_trials(port, "port", model, servers, MASTER_SEED, first, trials, objects, arr_mean, srv_mean, par=nthreads)
        dt = time.perf_counter() - t0
        kind = "port"
        body = "plain-C restatement (oracle/port): oracle/_ref did not travel with this snapshot"
    events = sum(r.events for r in res)
    return {"events": events, "seconds": dt, "cores": 1 if threads == 1 else host["cores"], "threads": nthreads,
            "kind": kind, "results": res, "body": body, "host": host}


def single_core_rows(objects: int):
    """benchmark/MM1_single.c (BASELINE config 1): one replication on one core, rho = 0.9 (the reference file) and 0.8."""
    rows = []
    for rho in (0.9, 0.8):
        cpu_reference_run(1, min(objects, 100_000), arr_mean=1.0 / rho, threads=1)                 # warm-up
        r = cpu_reference_run(2, objects, arr_mean=1.0 / rho, threads=1)
        rows.append({"workload": f"benchmark/MM1_single (rho={rho}, {objects} objects, 1 core)", "rho": rho,
                     "value": r["events"] / r["seconds"], "unit": "events/s", "cores": 1, "kind": r["kind"],
                     "events_per_trial": r["events"] // 2, "seconds_per_trial": r["seconds"] / 2})
    return rows


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    host = usable_cpus()
    trials = args.ref_trials or 16 * host["cores"]
    for _ in range(args.warmup):
        cpu_reference_run(max(host["cores"], 1), min(args.objects, 100_000))
    t_total, ev_total, last = 0.0, 0, None
    for k in range(args.steps):
        last = cpu_reference_run(trials, args.objects, first=k * trials)
        t_total += last["seconds"]
        ev_total += last["events"]
    value = ev_total / t_total
    sample = f"{trials} of {args.trials} replications x {args.objects} objects per step"
    line = {
        "impl": "reference", "metric": "M/M/1 simulated events/sec (FEL pops/s)", "value": value,
        "unit": "events/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * t_total / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "benchmark/MM1_multi (rho=0.9, 1e6 objects/trial, 65536 trials/GPU)",
                   "sample": sample, "seeding": "cmb_random_fmix64(master, trial)", "body": last["body"]},
        "cpu_baseline": {"value": value, "unit": "events/s", "cores": last["cores"], "threads": last["threads"],
                         "kind": last["kind"], "sample": sample, "host": last["host"]},
        "e2e": {"value": value, "unit": "events/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "events_convention_4_per_object": 4.0 * trials * args.objects * args.steps / t_total,
    }
    try:
        line["single_core"] = single_core_rows(args.objects)
    except Exception as e:                              # never lose the line over an extra
        line["single_core"] = {"error": repr(e)}
    emit(line)


_REAL_STDOUT = None


def emit(line):
    out = _REAL_STDOUT if _REAL_STDOUT is not None else sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


# ------------------------------------------------------------------------------------------------ secondary configurations
def secondary_configs(args, cb, torch, dist, dev, rank, world, barrier):
    """The other BASELINE.json configurations on this run's GPUs: one warm-up + one timed step each (CUDA events, max
    over ranks, trials sharded over ranks like the primary), a parity sample against the reference build on rank 0."""
    import numpy as np
    from oracle_libs import load_ref, run_trials
    ref = load_ref() if rank == 0 else None
    out = []

    def timed(launch, merge=None):
        launch(True)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        res = launch(False)
        merged = merge(res) if merge is not None else None   # the config's cross-GPU step, inside the timed region
        e1.record()
        barrier()
        return res, merged, e0.elapsed_time(e1)

    def gather(ms, events, bad):
        t = torch.tensor([ms, float(events), float(bad)], dtype=torch.float64, device=dev)
        if world > 1:
            mx, sm = t.clone(), t.clone()
            dist.all_reduce(mx, op=dist.ReduceOp.MAX)
            dist.all_reduce(sm, op=dist.ReduceOp.SUM)
            return float(mx[0]), int(sm[1]), int(sm[2])
        return ms, int(events), int(bad)

    def queue_like(name, model, servers, arr, srv, total_trials, per_gpu_fixed, parity_model, merge_nccl=False,
                   variant=0, objects=None):
        nobj = objects or args.objects
        trials = per_gpu_fixed if per_gpu_fixed else max(1, total_trials // world)
        first = rank * trials
        am = torch.full((trials,), arr, dtype=torch.float64, device=dev)
        sm = torch.full((trials,), srv, dtype=torch.float64, device=dev)
        bufs = cb.TrialBuffers(trials, dev, 0, model, servers, variant, 0, nobj)

        def launch(warm):
            if warm:
                return cb.launch_trials(am[:1024], sm[:1024], num_objects=min(nobj, 2000), master_seed=MASTER_SEED, first_trial=first,
                                        model=model, servers=servers, variant=variant)
            return cb.launch_trials(am, sm, num_objects=nobj, master_seed=MASTER_SEED, first_trial=first, model=model,
                                    servers=servers, variant=variant, buffers=bufs)

        merge = (lambda res: cb.merge_across_ranks(cb.summarize_on_device(res.sum_wait, res.objects))) if merge_nccl else None
        res, merged, ms = timed(launch, merge)
        ms, events, bad = gather(ms, int(res.events.sum().item()), int((res.status != 0).sum().item()))
        row = {"workload": name, "trials_total": trials * world, "trials_per_gpu": trials, "objects_per_trial": nobj,
               "ms": ms, "value": events / ms * 1e3, "unit": "events/s", "events": events, "failed_trials": bad}
        if merged is not None:
            row["summary"] = {"n": merged.count(), "mean_time_in_system": merged.mean(), "ci95_half_width": merged.half_width_95(),
                              "merge": "cmb_datasummary per GPU, NCCL all-gather + merge in rank order, inside the timed region"}
        if rank == 0 and parity_model is not None:
            n = 16
            r = cpu_reference_run(n, nobj, model=parity_model, servers=servers, arr_mean=arr, srv_mean=srv)
            ev, te, sw = res.events[:n].cpu().tolist(), res.t_end[:n].cpu().tolist(), res.sum_wait[:n].cpu().tolist()
            row["parity"] = {"kind": r["kind"], "trials": n, "bit_identical": all(
                (ev[i], te[i], sw[i]) == (w.events, w.t_end, w.sum_wait) for i, w in enumerate(r["results"])),
                "cpu_events_per_s": r["events"] / r["seconds"], "cpu_cores": r["cores"]}
        del bufs, am, sm
        return row

    def guarded(fn):
        try:
            row = fn()
        except Exception as e:                          # a secondary entry must never cost the primary line
            row = {"error": repr(e)}
        if rank == 0:
            out.append(row)
        torch.cuda.empty_cache()

    guarded(lambda: queue_like("MM1_multi rho=0.8 (BASELINE.json's rho), 65536 replications per GPU", cb.MODEL_MM1, 1,
                               1.0 / 0.8, 1.0, 0, args.trials, 0))
    guarded(lambda: queue_like("config 3: M/M/c c=8 via cmb_resourcepool, 32768 replications per GPU (262144 over 8), "
                               "per-GPU cmb_datasummary merged over NCCL", cb.MODEL_MMC, 8, 1.0 / 6.4, 1.0, 0, 32768, 2,
                               merge_nccl=True))
    guarded(lambda: queue_like("config 4: G/G/1 (Erlang-2 arrivals, ziggurat-normal service), 1048576 replications in all",
                               cb.MODEL_GG1, 1, 1.25, 1.0, 1048576, 0, 1))
    guarded(lambda: queue_like("M/M/1 written against the device authoring surface (cimba_b200/models/mm1_model.cuh, 50 lines), on the STATIC "
                               "tier (CIMBA_B200_VARIANT_STATIC: registers + shared memory, general engine as repair pass), "
                               "65536 replications per GPU at full length", cb.MODEL_MM1, 1, 1.0 / ARRIVAL_RATE, 1.0, 0, args.trials, 0,
                               variant=cb.VARIANT_STATIC))
    guarded(lambda: queue_like("G/G/1 (config 4's model) from its authoring-surface source (gg1_model.cuh: Erlang-2 and redrawn-normal holds as "
                               "CMB_PROCESS_HOLD_SAMPLED) on the static tier, 1048576 replications in all x 1e5 objects",
                               cb.MODEL_GG1, 1, 1.25, 1.0, 1048576, 0, 1, variant=cb.VARIANT_STATIC, objects=min(args.objects, 100_000)))
    guarded(lambda: queue_like("M/M/1 written against the device authoring surface, on the general engine (CIMBA_B200_VARIANT_GENERAL), "
                               "65536 replications per GPU x 1e5 objects", cb.MODEL_MM1, 1, 1.0 / ARRIVAL_RATE, 1.0, 0, args.trials, 0,
                               variant=cb.VARIANT_GENERAL, objects=min(args.objects, 100_000)))

    def hold_model():
        trials, workers, duration = max(1, 4096 // world), 1000, 200
        am = torch.full((trials,), 1.0, dtype=torch.float64, device=dev)
        bufs = cb.TrialBuffers(trials, dev, 0, cb.MODEL_HOLD, workers, 0)

        def launch(warm):
            return cb.launch_trials(am, am, num_objects=5 if warm else duration, master_seed=MASTER_SEED, first_trial=rank * trials,
                                    model=cb.MODEL_HOLD, servers=workers, buffers=bufs)
        res, _, ms = timed(launch)
        ms, events, bad = gather(ms, int(res.events.sum().item()), int((res.status != 0).sum().item()))
        row = {"workload": "hold model: 1000 processes per trial in cmb_process_hold loops (AWACS' event-list shape), 4096 trials in all",
               "trials_total": trials * world, "ms": ms, "value": events / ms * 1e3, "unit": "events/s", "events": events,
               "failed_trials": bad}
        if rank == 0 and ref is not None:
            want = run_trials(ref, "ref", 7, workers, MASTER_SEED, 0, 4, duration, 1.0, 1.0, par=1)
            ev, sw = res.events[:4].cpu().tolist(), res.sum_wait[:4].cpu().tolist()
            row["parity"] = {"kind": "reference", "trials": 4,
                             "bit_identical": all((ev[i], sw[i]) == (w.events, w.sum_wait) for i, w in enumerate(want))}
        return row
    guarded(hold_model)

    def awacs_short():
        from oracle_libs import AWACS_TERRAIN_SEED, awacs_terrain, awacs_ref_experiment, load_awacs_ref, load_port
        import ctypes as C
        trials, seconds = max(1, 4096 // world), 300
        host = usable_cpus()
        m, cols, rows, geom = awacs_terrain(load_port(), "port", AWACS_TERRAIN_SEED, 100.0, 100.0, max(1, host["cores"] // max(1, world)))
        cb.awacs_set_terrain(torch.from_numpy(m).to(dev), cols, rows, geom)
        cb.awacs_run(trials, duration_s=5, master_seed=1, device=dev)     # warm-up at full width (buffers, clocks)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        res, _ = cb.awacs_run(trials, duration_s=seconds, master_seed=MASTER_SEED, first_trial=rank * trials, device=dev)
        e1.record()
        barrier()
        ms, events, bad = gather(e0.elapsed_time(e1), int(res.events.sum().item()), int((res.status != 0).sum().item()))
        row = {"workload": f"config 5: AWACS tutorial/tut_5_1.c, 4096 replications in all, {seconds} simulated seconds each "
                           f"(the tutorial runs 24 h: profiles/r02_awacs.md), 100 x 100 nm terrain ({cols} x {rows} cells)",
               "trials_total": trials * world, "ms": ms, "value": events / ms * 1e3, "unit": "events/s", "events": events,
               "target_sweeps_per_s": trials * world * seconds * 1000 / ms * 1e3, "failed_trials": bad}
        aref = load_awacs_ref() if rank == 0 else None
        if aref is not None:
            aref.awacs_ref_adopt_terrain(m.ctypes.data_as(C.POINTER(C.c_float)), C.c_uint32(cols), C.c_uint32(rows),
                                         geom.ctypes.data_as(C.POINTER(C.c_float)))
            n = max(1, min(8, host["cores"]))
            t0 = time.perf_counter()
            outs = awacs_ref_experiment(aref, MASTER_SEED, 0, n, seconds / 3600.0)
            dt = time.perf_counter() - t0
            ev, found, sx = res.events[:n].cpu().tolist(), res.objects[:n].cpu().tolist(), res.sum_wait[:n].cpu().tolist()
            row["parity"] = {"kind": "reference (unmodified tutorial source, glibc libm)", "trials": n,
                             "bit_identical": all((ev[i], found[i], sx[i]) == (o.events, o.num_found, o.sum_x) for i, o in enumerate(outs)),
                             "cpu_target_sweeps_per_s": n * seconds * 1000 / dt, "cpu_cores": host["cores"]}
        return row
    guarded(awacs_short)
    return out


# ------------------------------------------------------------------------------------------------ one process, all GPUs
def run_single_process(args):
    """cimba_b200_run_experiment_all_gpus: the executive's one-host-thread-per-GPU form, timed from the outside."""
    import numpy as np
    import torch
    import cimba_b200 as cb
    n_gpus = min(args.gpus, torch.cuda.device_count())
    T, NOBJ = args.trials * n_gpus, args.objects
    exp = np.zeros(T, dtype=cb.TRIAL_DTYPE)
    exp["arr_mean"], exp["srv_mean"] = 1.0 / ARRIVAL_RATE, 1.0 / SERVICE_RATE
    for _ in range(max(1, args.warmup)):
        cb.cimba_run_experiment(exp, num_objects=min(NOBJ, 2000), master_seed=MASTER_SEED, all_gpus=True, max_gpus=n_gpus)
    samplers = [ClockSampler(g) for g in range(n_gpus)]
    for s in samplers:
        s.start()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        cb.cimba_run_experiment(exp, num_objects=NOBJ, master_seed=MASTER_SEED, all_gpus=True, max_gpus=n_gpus)
    dt = time.perf_counter() - t0
    clocks = [s.stop() for s in samplers]
    events = int(exp["events"].sum())
    emit({"metric": "M/M/1 simulated events/sec (FEL pops/s)", "value": events * args.steps / dt, "unit": "events/s",
          "n_gpus": n_gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
          "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
          "config": {"workload": "benchmark/MM1_multi (rho=0.9, 1e6 objects/trial, 65536 trials/GPU)",
                     "mode": "single process: cimba_b200_run_experiment_all_gpus, one host thread per GPU; wall clock around the call "
                             "(host staging, H2D, kernels, D2H, scatter inside)"},
          "e2e": {"value": events * args.steps / dt, "unit": "events/s", "h2d_bytes_per_step": 16 * T, "d2h_bytes_per_step": 40 * T},
          "gpu_launches": int(cb.lib.cimba_b200_launch_count()), "clocks": clocks[0], "per_gpu_clocks": clocks,
          "failed_trials": int((exp["status"] != 0).sum())})


def main():
    args = parse_args()
    # The contract is ONE JSON line on stdout.  Libraries print there too (NCCL's version banner under
    # NCCL_DEBUG=VERSION, for one), so file descriptor 1 is pointed at stderr for the whole run and the
    # line goes to the saved descriptor at the end.
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    if args.impl == "reference":
        run_reference_arm(args)
        return
    if args.single_process:
        run_single_process(args)
        return

    import numpy as np
    import torch
    import torch.distributed as dist
    import cimba_b200 as cb
    from cimba_b200.experiment import TrialBuffers

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU path exists)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    T, NOBJ = args.trials, args.objects
    first = rank * T
    arr = torch.full((T,), 1.0 / ARRIVAL_RATE, dtype=torch.float64, device=dev)
    srv = torch.full((T,), 1.0 / SERVICE_RATE, dtype=torch.float64, device=dev)
    bufs = TrialBuffers(T, dev, 0, cb.MODEL_MM1, 1, args.variant)
    diag = torch.zeros(4, dtype=torch.int64, device=dev)

    def step():
        return cb.launch_trials(arr, srv, num_objects=NOBJ, master_seed=MASTER_SEED, first_trial=first,
                                mapping=args.mapping, buffers=bufs, variant=args.variant, diag=diag)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    for _ in range(args.warmup):
        step()
    barrier()
    diag.zero_()

    sampler = ClockSampler(local)
    sampler.start()                                     # every rank watches its own GPU
    launches0 = cb.lib.cimba_b200_launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    per_launch = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
                  for _ in range(args.steps)]
    barrier()
    ev0.record()
    for k in range(args.steps):
        per_launch[k][0].record()
        res = step()
        per_launch[k][1].record()
    ev1.record()
    barrier()
    launches = cb.lib.cimba_b200_launch_count() - launches0
    ms_total = ev0.elapsed_time(ev1)
    kernel_ms = [a.elapsed_time(b) for a, b in per_launch]
    clocks = sampler.stop()
    diag_host = diag.cpu().tolist()
    if args.dump_outputs:
        dump_outputs(res, args.dump_outputs, rank, world)

    events_rank = int(res.events.sum().item())
    bad = int((res.status != 0).sum().item())
    t = torch.tensor([ms_total, float(events_rank), float(bad)], dtype=torch.float64, device=dev)
    if world > 1:
        tmax = t.clone()
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        tsum = t.clone()
        dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
        ms_total, events_all, bad = float(tmax[0]), int(tsum[1]), int(tsum[2])
    else:
        events_all = events_rank
    per_rank = None
    if world > 1:
        # the slowest rank sets the number; record every rank's own time and clocks beside it
        mine = {"rank": rank, "ms_per_step": float(t[0]) / args.steps, "sm_mhz": clocks.get("sm_mhz"),
                "reasons": clocks.get("reasons")}
        gathered = [None] * world
        dist.all_gather_object(gathered, mine)
        per_rank = gathered
    ms_per_step = ms_total / args.steps
    value = events_all / (ms_per_step * 1e-3)

    # cross-GPU statistics merge, reported with the line (the e2e leg below has it INSIDE its timed region)
    local_summary = cb.summarize_on_device(res.sum_wait, res.objects)
    merged = cb.merge_across_ranks(local_summary)

    # ---- end to end through the host-buffer C-ABI (pinned staging + H2D + kernel + D2H) + the NCCL summary merge
    e2e = None
    if not args.no_e2e:
        exp = np.zeros(T, dtype=cb.TRIAL_DTYPE)
        exp["arr_mean"], exp["srv_mean"] = 1.0 / ARRIVAL_RATE, 1.0 / SERVICE_RATE
        n_e2e = max(1, min(args.steps, 10))
        cb.cimba_run_experiment(exp, num_objects=min(NOBJ, 1000), master_seed=MASTER_SEED,
                                first_trial=first, mapping=args.mapping, device=local, variant=args.variant)     # warm-up
        barrier()
        t0 = time.perf_counter()
        for _ in range(n_e2e):
            cb.cimba_run_experiment(exp, num_objects=NOBJ, master_seed=MASTER_SEED,
                                    first_trial=first, mapping=args.mapping, device=local, variant=args.variant)
            if world > 1:
                # benchmark/MM1_multi.c:143-148 across GPUs: per-rank cmb_datasummary of the results just written into
                # the host array, all-gathered over NCCL and merged in rank order
                sw = torch.from_numpy(exp["sum_wait"].copy()).to(dev)
                ob = torch.from_numpy(exp["obj_cnt"].astype(np.int64)).to(dev)
                e2e_merged = cb.merge_across_ranks(cb.summarize_on_device(sw, ob))
        torch.cuda.synchronize(dev)
        dt = time.perf_counter() - t0
        te = torch.tensor([dt, float(exp["events"].sum())], dtype=torch.float64, device=dev)
        if world > 1:
            tm = te.clone()
            dist.all_reduce(tm, op=dist.ReduceOp.MAX)
            ts = te.clone()
            dist.all_reduce(ts, op=dist.ReduceOp.SUM)
            dt, ev_e2e = float(tm[0]), float(ts[1])
        else:
            ev_e2e = float(te[1])
        e2e = {"value": ev_e2e * n_e2e / dt, "unit": "events/s", "steps": n_e2e,
               "h2d_bytes_per_step": 16 * T + (16 * T if world > 1 else 0), "d2h_bytes_per_step": 40 * T,
               "api": "cimba_b200_run_experiment (host trial-struct array, results in place)"
                      + ("; then the per-rank cmb_datasummary, NCCL all-gather and merge, all inside the timed region" if world > 1 else ""),
               "bit_identical_to_device_path": bool(
                   np.array_equal(exp["events"], res.events.cpu().numpy().astype(np.uint64)))}
        if world > 1:
            e2e["merged_mean_time_in_system"] = e2e_merged.mean()

    secondary = None
    if not args.no_secondary:
        del bufs
        torch.cuda.empty_cache()
        secondary = secondary_configs(args, cb, torch, dist, dev, rank, world, barrier)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peak, peak_src = measured_peak_gbs()
    kernel_s = sum(kernel_ms) / len(kernel_ms) * 1e-3
    kname = {0: "mm1_kernel", 1: "queue_kernel<0>", 16: "trial_kernel<MM1> (general engine)", 17: "static_trial_kernel<MM1T, 2, 1> (static tier)"}.get(args.variant, "mm1_kernel")
    cal = issue_calibration().get(kname if args.mapping == 1 else "", {})
    tr = measured_traffic()
    sms = torch.cuda.get_device_properties(dev).multi_processor_count
    sm_mhz = clocks.get("sm_mhz")
    hbm_gbs = events_rank * BYTES_PER_EVENT / kernel_s / 1e9
    roofline = {"bound": "issue", "achieved": None, "peak": None, "unit": "Gwarp-inst/s", "frac": None, "traffic": None,
                "kernel": kname, "kernel_ms": kernel_s * 1e3,
                "loop_iterations_per_launch": diag_host[0] / args.steps, "warps": diag_host[1] / args.steps,
                "repaired_trials": diag_host[2],
                "note": "per-trial state is on chip by design (DRAM traffic ~0.1 B/event): SM instruction issue binds, not HBM",
                "hbm": {"algorithmic_bytes_per_event": BYTES_PER_EVENT, "achieved_gbs": hbm_gbs, "peak_gbs": peak,
                        "frac_of_hbm_peak": hbm_gbs / peak, "peak_source": peak_src,
                        "reference_layout_gbs": events_rank * BYTES_PER_EVENT_REFLAYOUT / kernel_s / 1e9,
                        "note": "SURVEY.md section 8d's figure; > 1 because the records never leave the SM, not because work is skipped"}}
    if cal.get("warp_instructions_per_iteration") and sm_mhz and diag_host[0] > 0:
        inst = diag_host[0] / args.steps * cal["warp_instructions_per_iteration"]
        roofline["achieved"] = inst / kernel_s / 1e9
        roofline["peak"] = 4.0 * sms * sm_mhz * 1e6 / 1e9
        roofline["frac"] = roofline["achieved"] / roofline["peak"]
        roofline["warp_instructions_per_iteration"] = cal["warp_instructions_per_iteration"]
        roofline["calibration"] = cal.get("source")
        roofline["peak_source"] = f"4 warp schedulers x {sms} SMs x {sm_mhz} MHz (nvidia-smi median during the timed region)"
        roofline["warp_instructions_per_event"] = inst / max(1, events_rank)
        roofline["issue_active_pct_ncu"] = cal.get("issue_active_pct_under_ncu")
        roofline["alu_pipe_pct_ncu"] = cal.get("alu_pipe_pct_under_ncu")
        roofline["frac_note"] = ("frac = executed warp-instructions / (schedulers x clock x time), measured in this run; ncu's own "
                                 "smsp__issue_active of the calibration launch is beside it (it counts issue-port cycles, which "
                                 "the half-rate FP64 and ALU instructions of this loop hold for more than one)")
    if tr and args.variant == 0 and args.mapping == 1:
        roofline["traffic"] = tr["dram_bytes_per_event"] * events_rank
        roofline["traffic_source"] = tr["source"]

    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        host = usable_cpus()
        trials = args.ref_trials or 32 * host["cores"]
        r = cpu_reference_run(trials, NOBJ)
        # parity on the very same trials, at full per-trial size
        gpu_ev = res.events[:trials].cpu().tolist()
        gpu_te = res.t_end[:trials].cpu().tolist()
        gpu_sw = res.sum_wait[:trials].cpu().tolist()
        same = all((gpu_ev[i], gpu_te[i], gpu_sw[i]) == (w.events, w.t_end, w.sum_wait)
                   for i, w in enumerate(r["results"]))
        cpu = {"value": r["events"] / r["seconds"], "unit": "events/s", "cores": r["cores"], "threads": r["threads"],
               "kind": r["kind"], "body": r["body"], "host": r["host"],
               "sample": f"{trials} of {T} replications x {NOBJ} objects (same seeds as GPU trials 0..{trials - 1})",
               "seconds": r["seconds"], "gpu_results_bit_identical_on_sample": bool(same)}
        if r["host"]["cores"] != r["host"]["logical"]:
            cpu["note"] = (f"this process may use {r['host']['cores']} CPUs (cgroup quota / affinity) of the {r['host']['logical']} the "
                           f"box shows; cimba_run_experiment still starts {r['threads']} worker threads")
        try:
            cpu["single_core"] = single_core_rows(NOBJ)
        except Exception as e:
            cpu["single_core"] = {"error": repr(e)}

    line = {
        "metric": "M/M/1 simulated events/sec (FEL pops/s)", "value": value, "unit": "events/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "benchmark/MM1_multi (rho=0.9, 1e6 objects/trial, 65536 trials/GPU)",
                   "trials_per_gpu": T, "objects_per_trial": NOBJ, "rho": ARRIVAL_RATE / SERVICE_RATE,
                   "mapping": "lane-per-trial" if args.mapping == 1 else "warp-per-trial",
                   "seeding": "cmb_random_fmix64(0x34f05c64d7ad598f, global trial index); every step runs the same trials",
                   "l2": "no input re-use between steps: 1 MB of inputs, all state regenerated on chip"},
        "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks, "per_rank": per_rank, "roofline": roofline,
        "cpu_baseline": cpu, "secondary": secondary,
        "events_per_step": events_all, "failed_trials": bad,
        "events_convention_4_per_object": 4.0 * T * world * NOBJ / (ms_per_step * 1e-3),
        "summary": {"n": merged.count(), "mean_time_in_system": merged.mean(),
                    "ci95_half_width": merged.half_width_95(), "expected": 1.0 / (SERVICE_RATE - ARRIVAL_RATE)},
    }
    emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()

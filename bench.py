#!/usr/bin/env python
"""bench.py -- phonons traced per second on the BASELINE.json workloads (see DESIGN.md "Measurement").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W

One "step" = one pass of the propagate path over one batch of phonons: per_gpu phonons on every GPU (weak scaling).
The default workload is BASELINE.json configs[1], the one the metric is quoted on: the Halfspace near-source model
(do-halfspace-nearsrc50.sh) at the scripted take-off-angle degree 9, 1.25e8 phonons per GPU and step (its 1e9 phonons over
the 8 GPUs it is quoted on).  --workload selects any of the five BASELINE configs (halfspace, halfspace_nearsrc50,
crustpinch, lopnor, spherical), each with its own batch size.  The model is built by radiative3d_b200/workload_model.py
(the workload's geometry as the reference built it, its take-off-angle set, source and scatterer tables at the degree).

  value    device-timed (CUDA events on the launching stream, max over ranks): model resident in HBM, K steps plus
           the end-of-run NCCL reduction of the bins (two collectives: the f64 block and the i64 block).
  e2e      the same batch through the C ABI with HOST buffers.  One GPU: r3d_create (H2D of the pinned model tables) +
           r3d_run + r3d_fetch (D2H of bins and counters) + r3d_destroy.  N GPUs: rank 0 uploads the large tables once and
           broadcasts them over NVLink (NCCL), every rank runs its share, the bins are reduced to rank 0, rank 0 fetches.
  roofline the propagate kernel (one launch per step and GPU) timed with CUDA events on its stream over one more step;
           `roofline` is the HBM bound (SURVEY 8d bytes), `roofline_issue` the instruction-issue bound the kernel actually
           runs against (warp instructions per loop event from the committed ncu captures, profiles/kernel_counters.json).
  cpu_baseline  the unmodified reference binary (oracle/_ref/r3d_ref_main) on one host core, bounded sample.

--dump-outputs DIR writes what the last timed step computed, as a caller of the path receives it (bins and counters summed
over ranks), to DIR/energies.npy (f64 [n_seis, n_bins, 5]), DIR/counts.npy and DIR/counters.npy (as f64): that step's
phonons are traced once more after the timing (phonon i always draws from stream (seed, i)), so two builds run with the
same arguments can be compared output for output.

--impl reference times the reference's own CPU implementation with all host threads it can use (independent
processes, the reference's own way of scaling: scripts/do-parallel.sh), on a bounded sample per step.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOAD = "halfspace_nearsrc50"          # BASELINE.json configs[1]: the configuration the metric is quoted on (the default)
TOA_DEGREE = int(os.environ.get("R3D_BENCH_TOA_DEGREE", "9"))      # the scripted degree (do-fundamentals.sh:82); the override is for the test-suite
SEED = 20261018
# The five BASELINE.json configs (radiative3d_b200/workloads.py holds their command lines).  per_gpu = phonons per GPU per
# step, sized so that a step is 50-350 ms of device time and at least ~150 phonons pass through every slot of the kernel (a
# step is one launch: its ramp-up and its tail - the last, longest-lived phonons - cost about as much as ~20 phonons per
# slot, which a production run of 1e9 phonons does not notice); ref_per_proc / ref_one_core = the bounded samples of the CPU arms
# (the reference does 2e5 / 6e3 / 3e3 / 3e2 phonons per second and core on halfspace / crust pinch / Lop Nor / whole-Earth).
WORKLOADS = {
    "halfspace": dict(script="do-halfspace.sh", per_gpu=125_000_000, ref_per_proc=400_000, ref_one_core=1_500_000,
                      what="Halfspace model, 144 seismometers x 400 bins"),
    "halfspace_nearsrc50": dict(script="do-halfspace-nearsrc50.sh", per_gpu=125_000_000, ref_per_proc=400_000, ref_one_core=1_500_000,
                                what="Halfspace model, 144 seismometers x 1250 bins"),
    "crustpinch": dict(script="do-crustpinch.sh", per_gpu=30_000_000, ref_per_proc=20_000, ref_one_core=60_000,
                       what="crust-pinch model (2275 tetrahedra, interfaces with mode conversion), 480 seismometers x 300 bins"),
    "lopnor": dict(script="do-lopnor.sh", per_gpu=40_000_000, ref_per_proc=10_000, ref_one_core=30_000,
                   what="Lop Nor model (21 tilted layers, heterogeneous scattering), 320 seismometers x 300 bins"),
    "spherical": dict(script="do-spherical.sh", per_gpu=4_000_000, ref_per_proc=1_000, ref_one_core=3_000,
                      what="whole-Earth shells (quadratic-velocity layers), 480 seismometers x 400 bins"),
}
PER_GPU = WORKLOADS[WORKLOAD]["per_gpu"]
REF_MAIN = os.path.join(ROOT, "oracle", "_ref", "r3d_ref_main")
# SURVEY 8(d): bytes per table draw = ceil(log2 nTOA)*8 + 16, per catch = 96
BYTES_PER_CATCH = 96


def algorithmic_bytes_per_draw(n_toa):
    return (max(1, (n_toa - 1).bit_length())) * 8 + 16


# ---------------------------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock, throttle reasons and power sampled every 10 ms through NVML while the timed region runs (nvidia-smi every
    200 ms when the NVML binding is missing)."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap,power.draw")
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, index):
        self.rows, self.proc, self.nvml, self.halt, self.how = [], None, None, False, None
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
            ids = [v for v in vis.split(",") if v.strip()]
            phys = int(ids[index]) if ids and all(v.strip().isdigit() for v in ids) and index < len(ids) else index
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_sm = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self.nvml, self.how = pynvml, "nvml every 10 ms"
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.how = "nvidia-smi every 200 ms"
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _poll(self):
        n = self.nvml
        bits = [(getattr(n, "nvmlClocksEventReasonHwSlowdown", 0x8), 0), (getattr(n, "nvmlClocksEventReasonHwThermalSlowdown", 0x40), 1),
                (getattr(n, "nvmlClocksEventReasonSwThermalSlowdown", 0x20), 2), (getattr(n, "nvmlClocksEventReasonSwPowerCap", 0x4), 3)]
        reasons_of = getattr(n, "nvmlDeviceGetCurrentClocksEventReasons", None) or n.nvmlDeviceGetCurrentClocksThrottleReasons
        while not self.halt:
            try:
                sm = float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM))
                mask = int(reasons_of(self.handle))
                pw = n.nvmlDeviceGetPowerUsage(self.handle) / 1000.0
                row = [str(sm), str(self.max_sm)] + ["Not Active"] * 4 + [str(pw)]
                for b, k in bits:
                    if mask & b:
                        row[2 + k] = "Active"
                self.rows.append((time.perf_counter(), row))
            except Exception:
                pass
            time.sleep(0.01)

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [x.strip() for x in line.split(",")]))

    def stop(self, t0, t1):
        if not self.proc and not self.nvml:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["neither NVML nor nvidia-smi available"]}
        if self.nvml:
            self.halt = True
            self.thread.join(timeout=1.0)
        else:
            time.sleep(0.25)
            self.proc.terminate()
        rows = [r for t, r in self.rows if t0 <= t <= t1] or [r for _, r in self.rows[-3:]]
        sm = [float(r[0]) for r in rows if r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in rows if r[1].replace(".", "").isdigit()]
        reasons = sorted({n for r in rows for n, v in zip(self.NAMES, r[2:6]) if v.lower().startswith("active")})
        pw = [float(r[6]) for r in rows if len(r) > 6 and r[6].replace(".", "").isdigit()]
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(rows), "power_w_max": max(pw) if pw else None, "how": self.how}


class ReferenceRun:
    """One run of the UNMODIFIED reference program on a workload.  The simulation part is timed inside the process: from the
    reference's own "@@ __BEGINNING_SIMULATION__" line (model.cpp:609) to process exit, so that model-build time - which
    stretches when many processes build their tables at once - is not estimated from another run."""

    def __init__(self, workload, n_phonons, outdir):
        from radiative3d_b200 import workloads
        os.makedirs(outdir, exist_ok=True)
        self.t_start = time.perf_counter()
        self.t_sim = None
        self.proc = subprocess.Popen([REF_MAIN] + workloads.cmdline(workload, n_phonons, TOA_DEGREE, outdir), cwd=outdir,
                                     stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        self.thread = threading.Thread(target=self._watch, daemon=True)
        self.thread.start()

    def _watch(self):
        for line in self.proc.stdout:
            if self.t_sim is None and "__BEGINNING_SIMULATION__" in line:
                self.t_sim = time.perf_counter()

    def wait(self):
        """-> (seconds of model build, seconds of simulation + output)"""
        rc = self.proc.wait()
        t_end = time.perf_counter()
        self.thread.join(timeout=5.0)
        if rc != 0 or self.t_sim is None:
            raise RuntimeError(f"reference binary failed (rc {rc})")
        return self.t_sim - self.t_start, t_end - self.t_sim


def cpu_baseline_one_core(workload):
    """The reference binary on ONE host core: (sample phonons) / (seconds after its model build)."""
    sample = WORKLOADS[workload]["ref_one_core"]
    if not os.path.exists(REF_MAIN):
        return cpu_baseline_port(workload, max(sample // 10, 100), 1)
    with tempfile.TemporaryDirectory() as tmp:
        t_init, t_run = ReferenceRun(workload, sample, os.path.join(tmp, "run")).wait()
    return {"value": sample / max(t_run, 1e-9), "unit": "phonons/s", "cores": 1, "kind": "reference",
            "sample": f"{sample} phonons of {workload} at TOA degree {TOA_DEGREE} through oracle/_ref/r3d_ref_main "
                      f"(unmodified reference, -O3): {t_run:.1f} s from its __BEGINNING_SIMULATION__ line to exit, after {t_init:.1f} s of model build"}


def cpu_baseline_port(workload, sample, threads):
    """Fallback when the reference binary did not travel: the C oracle (a port), on `threads` host threads."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_binding as ob
    from radiative3d_b200 import workload_model
    m = workload_model.build_model(workload, TOA_DEGREE)
    ob.run(m, 0, min(1000, sample), SEED, nthreads=threads)
    t = time.perf_counter()
    ob.run(m, 0, sample, SEED, nthreads=threads)
    dt = time.perf_counter() - t
    return {"value": sample / dt, "unit": "phonons/s", "cores": threads, "kind": "port",
            "sample": f"{sample} phonons of {workload} at TOA degree {TOA_DEGREE} through oracle/liboracle.so"}


# ---------------------------------------------------------------------------------------------------------------
def reference_arm(args):
    """bench.py --impl reference: the reference's CPU implementation on all host cores (independent processes)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    wl = args.workload
    cores = int(os.environ.get("R3D_BENCH_REF_CORES", "0")) or max(1, min(os.cpu_count() or 1, 32))      # (overrides: test-suite)
    per_proc = int(os.environ.get("R3D_BENCH_REF_PER_PROC", "0")) or WORKLOADS[wl]["ref_per_proc"]
    base = {"metric": "phonons traced/sec", "unit": "phonons/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "impl": "reference", "gpu_launches": 0,
            "config": {"workload": f"{wl} ({WORKLOADS[wl]['script']}), TOA degree {TOA_DEGREE}",
                       "phonons_per_step": cores * per_proc, "note": "bounded sample of the GPU arm's batch"}}
    if not os.path.exists(REF_MAIN):
        cb = cpu_baseline_port(wl, cores * max(per_proc // 20, 50), cores)
        base.update(value=cb["value"], ms_per_step=None, cpu_baseline=cb,
                    e2e={"value": cb["value"], "unit": "phonons/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0})
        print(json.dumps(base))
        return 0
    with tempfile.TemporaryDirectory() as tmp:
        def step(i):       # (the reference seeds with time(NULL): equal seeds duplicate phonons, not cost)
            runs = [ReferenceRun(wl, per_proc, os.path.join(tmp, f"s{i}_{c}")) for c in range(cores)]
            res = [r.wait() for r in runs]
            return max(t for t, _ in res), max(t for _, t in res)       # slowest model build, slowest simulation

        for i in range(min(args.warmup, 1)):          # one warm-up pass is enough for a CPU process farm
            step(-1 - i)
        times = [step(i) for i in range(args.steps)]
    sim = [max(t, 1e-9) for _, t in times]
    value = cores * per_proc * len(sim) / sum(sim)
    cb = {"value": value, "unit": "phonons/s", "cores": cores, "kind": "reference",
          "sample": f"{cores} independent processes x {per_proc} phonons per step through oracle/_ref/r3d_ref_main; per step the "
                    f"slowest process's time from its own __BEGINNING_SIMULATION__ line to exit (model build, "
                    f"{sum(t for t, _ in times) / len(times):.1f} s with all processes building at once, is not counted)"}
    base.update(value=value, ms_per_step=1e3 * sum(sim) / len(sim), cpu_baseline=cb,
                e2e={"value": value, "unit": "phonons/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0})
    print(json.dumps(base))
    return 0


# ---------------------------------------------------------------------------------------------------------------
def issue_roofline(workload, events_per_second, sm_mhz, n_sm=148):
    """The bound the kernel actually runs against: warp instructions issued.  achieved = loop events per second (live) x warp
    instructions per event (ncu, profiles/kernel_counters.json); peak = SMs x 4 schedulers x SM clock (1 instruction per
    scheduler and cycle)."""
    try:
        kc = json.load(open(os.path.join(ROOT, "profiles", "kernel_counters.json")))[workload]
    except (OSError, ValueError, KeyError):
        return None
    mhz = sm_mhz or 1965.0
    peak = n_sm * 4 * mhz * 1e6
    achieved = events_per_second * kc["warp_inst_per_event"]
    return {"bound": "issue", "kernel": "propagate_kernel", "achieved": achieved / 1e9, "peak": peak / 1e9, "unit": "G warp-inst/s",
            "frac": achieved / peak, "warp_inst_per_event": kc["warp_inst_per_event"], "thread_inst_per_event": kc["thread_inst_per_event"],
            "active_lanes_per_inst": kc.get("lanes_per_inst"), "ncu_issue_active_pct": kc.get("issue_active_pct"),
            "ncu_fp64_pipe_pct": kc.get("fp64_pipe_pct"), "ncu_warps_per_sm": kc.get("warps_per_sm"),
            "peak_source": f"{n_sm} SMs x 4 schedulers x {mhz:.0f} MHz (SM clock sampled during the timed region)",
            "counters_source": kc.get("source")}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=WORKLOAD, choices=sorted(WORKLOADS))
    ap.add_argument("--per-gpu", type=int, default=None, help="phonons per GPU per step (default: the workload's)")
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None, help="write the last timed step's bins and counters as .npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return reference_arm(args)
    args.warmup = max(args.warmup, 3)
    wl = args.workload
    # stdout carries ONE JSON line: whatever libraries print to fd 1 meanwhile (NCCL's version banner) goes to stderr
    json_fd = os.dup(1)
    os.dup2(2, 1)

    import numpy as np
    import torch
    import torch.distributed as dist
    from radiative3d_b200 import abi, distributed, engine, workload_model
    from radiative3d_b200.model import _ARRAYS

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the propagate path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    if world != args.gpus and rank == 0:
        print(f"bench.py: --gpus {args.gpus} but WORLD_SIZE {world}; using {world}", file=sys.stderr)

    # ---- the model: built for the workload at the TOA degree, pinned --------------------------------------------
    model = workload_model.build_model(wl, TOA_DEGREE, device=local)
    keep = []
    for name, _ in _ARRAYS:
        t = torch.from_numpy(getattr(model, name)).pin_memory()
        keep.append(t)
        setattr(model, name, t.numpy())
    per, K, W = (args.per_gpu or WORKLOADS[wl]["per_gpu"]), args.steps, args.warmup
    eng = engine.Engine(model, devices=(local,))

    def enqueue(i):
        first, n = distributed.shard_range(i * per * world, per * world, rank, world)
        eng.run_simulation(n, seed=SEED, first_phonon=first)

    fblk, iblk, k_at = eng.device_accumulator_blocks(0)
    fblk, iblk = torch.as_tensor(fblk, device=dev), torch.as_tensor(iblk, device=dev)
    for i in range(W):
        enqueue(i)
    eng.sync()
    distributed.all_reduce_blocks(fblk, iblk, k_at)   # warm-up of the collectives too (NCCL sets its channels up lazily)
    torch.cuda.synchronize()
    eng.reset()

    # ---- timed region: K steps + the reduction of the bins (two collectives) ----------------------------------
    sampler = ClockSampler(local) if rank == 0 else None
    launches0 = eng.launch_count
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i in range(K):
        enqueue(W + i)
    dev_s = eng.sync()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    distributed.all_reduce_blocks(fblk, iblk, k_at)
    ev1.record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t1 = time.perf_counter()
    dev_s += ev0.elapsed_time(ev1) * 1e-3
    launches = eng.launch_count - launches0          # our kernels only (the two NCCL collectives are the library's)
    clocks = sampler.stop(t0, t1) if sampler else None
    tt = torch.tensor([dev_s, t1 - t0, float(launches)], dtype=torch.float64, device=dev)
    if world > 1:
        mx = tt.clone()
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        dist.all_reduce(tt, op=dist.ReduceOp.SUM)
        dev_s, wall_s, launches = float(mx[0]), float(mx[1]), int(tt[2])
    else:
        wall_s = t1 - t0
    total = K * per * world
    counters = iblk[k_at:k_at + abi.R3D_NCOUNTERS].cpu().numpy().astype(np.uint64)
    if int(counters[abi.R3D_CNT_PHONONS]) != total:
        raise SystemExit(f"bench.py: traced {int(counters[abi.R3D_CNT_PHONONS])} phonons, expected {total}")
    events_total = int(counters[abi.R3D_CNT_EVENTS])

    # ---- roofline of the propagate kernel (the only kernel of the path): CUDA events on its launching stream, live,
    # over one extra step of the same size (rank 0's GPU; the kernels are per GPU)
    roofline, roofline_issue = None, None
    eng.reset()
    eng.set_profiling(True)
    enqueue(W + K)
    eng.sync()
    kt = eng.kernel_times()
    kt["phonons"] = per
    eng.set_profiling(False)
    if rank == 0:
        bytes_draw = algorithmic_bytes_per_draw(model.n_toa)
        alg = kt["draws"] * bytes_draw + kt["catches"] * BYTES_PER_CATCH          # SURVEY 8(d)
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except OSError:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        traffic, traffic_note = None, None
        try:
            tj = json.load(open(os.path.join(ROOT, "profiles", "kernel_counters.json")))[wl]
            traffic = tj["dram_bytes_per_phonon"] * kt["phonons"] / max(kt["launches"], 1)
            traffic_note = tj.get("source")
        except (OSError, ValueError, KeyError):
            pass
        sec, nl = kt["seconds"], max(kt["launches"], 1)
        achieved = alg / sec / 1e9
        ph = kt["phase1_seconds"] + kt["phase2_seconds"]
        roofline = {"bound": "hbm", "kernel": "propagate_kernel", "achieved": achieved, "peak": peak, "unit": "GB/s",
                    "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_note,
                    "peak_source": "MEASURED_PEAKS.json hbm_gbs (measured)" if peaks else "fallback 6650 GB/s (B200_PROFILING.md)",
                    "avg_launch_ms": 1e3 * sec / nl, "algorithmic_bytes_per_launch": alg / nl,
                    "algorithmic_bytes": f"{bytes_draw} B per table draw + {BYTES_PER_CATCH} B per bin update (SURVEY 8d)",
                    "share_of_step": {"propagate_kernel": 1.0},
                    "phase_share": {"advance": kt["phase1_seconds"] / ph if ph else None,
                                    "draw+face+bend": kt["phase2_seconds"] / ph if ph else None},
                    "units": {"phonons": per, "loop_events": kt["events"], "table_draws": kt["draws"], "bin_updates": kt["catches"]},
                    "ctas": kt["ctas"], "iterations_of_busiest_cta": kt["iterations"],
                    "note": "the kernel is latency / issue bound, not HBM bound: see roofline_issue"}
        roofline_issue = issue_roofline(wl, kt["events"] / sec, clocks.get("sm_mhz") if clocks else None, kt["ctas"])

    if args.dump_outputs:
        eng.reset()
        enqueue(W + K - 1)
        eng.sync()
        distributed.all_reduce_blocks(fblk, iblk, k_at)
        torch.cuda.synchronize()
        if rank == 0:
            e, c, k = eng.fetch()
            os.makedirs(args.dump_outputs, exist_ok=True)
            for name, a in (("energies", e), ("counts", c), ("counters", k)):
                np.save(os.path.join(args.dump_outputs, f"{name}.npy"), a.astype(np.float64))

    # ---- e2e: host model in, host bins out, through the C ABI ---------------------------------------------------
    eng.close()
    del fblk, iblk
    e2e_times = []
    big = sum(getattr(model, n).nbytes for n in distributed.BIG_TABLES)
    small = model.table_bytes() - big
    h2d = model.table_bytes() if world == 1 else big + world * small       # large tables once per node, small ones per rank
    d2h = model.n_seis * model.n_bins * (abi.R3D_BIN_NF64 * 8 + abi.R3D_BIN_NCNT * 8) + abi.R3D_NCOUNTERS * 8
    host_e = torch.zeros((model.n_seis, model.n_bins, abi.R3D_BIN_NF64), dtype=torch.float64).pin_memory()      # the caller's result buffers
    host_c = torch.zeros((model.n_seis, model.n_bins, abi.R3D_BIN_NCNT), dtype=torch.int64).pin_memory()
    host_out = (host_e.numpy(), host_c.numpy().view(np.uint64))
    e2e_phonons = None
    for i in range(args.e2e_steps + 1 if args.e2e_steps > 0 else 0):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t = time.perf_counter()
        first, n = distributed.shard_range((W + K + 1 + i) * per * world, per * world, rank, world)
        if world == 1:
            with engine.Engine(model, devices=(local,)) as e2:
                e2.run_simulation(n, seed=SEED, first_phonon=first)
                e2.sync()
                ee, cc, kk = e2.fetch(out=host_out)
        else:
            # host model on rank 0 -> one H2D of the large tables + NCCL broadcast over NVLink -> every rank's share ->
            # reduction of the bins to rank 0 -> rank 0's host buffers
            tables = distributed.broadcast_model_tables(model, dev, src=0)
            torch.cuda.synchronize()
            with engine.Engine(model, devices=(local,), device_tables=tables) as e2:
                e2.run_simulation(n, seed=SEED, first_phonon=first)
                e2.sync()
                fb, ib, at = e2.device_accumulator_blocks(0)
                fb, ib = torch.as_tensor(fb, device=dev), torch.as_tensor(ib, device=dev)
                distributed.all_reduce_blocks(fb, ib, at, dst=0)
                torch.cuda.synchronize()
                if rank == 0:
                    ee, cc, kk = e2.fetch(out=host_out)
                del fb, ib
            del tables
            dist.barrier()
        dt = time.perf_counter() - t
        if rank == 0:
            e2e_phonons = int(kk[abi.R3D_CNT_PHONONS])
        if i > 0:                                   # first pass warms the allocator / context
            e2e_times.append(dt)
    e2e_s = sum(e2e_times) / len(e2e_times) if e2e_times else float("nan")
    if world > 1:
        tmx = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
        dist.all_reduce(tmx, op=dist.ReduceOp.MAX)
        e2e_s = float(tmx[0])
    if rank == 0 and e2e_times and e2e_phonons != per * world:
        raise SystemExit(f"bench.py: the end-to-end leg returned {e2e_phonons} phonons on rank 0, expected {per * world}")

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu = cpu_baseline_one_core(wl)

    if rank == 0:
        guide_gb = None
        out = {
            "metric": "phonons traced/sec", "value": total / dev_s, "unit": "phonons/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": 1e3 * dev_s / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"{wl} ({WORKLOADS[wl]['script']}): {model.n_cells} cells, {model.n_seis} seismometers x {model.n_bins} bins, "
                                   f"TOA degree {TOA_DEGREE} ({model.n_toa} take-off angles, {model.table_bytes() / 1e9:.2f} GB of tables)",
                       "phonons_per_gpu_per_step": per, "global_phonons_per_step": per * world, "parallelism": f"phonon-index sharding x{world}, "
                       "bins reduced once at the end (NCCL, 2 collectives: f64 block, i64 block)",
                       "cache": f"inputs larger than L2: {model.table_bytes() / 1e9:.2f} GB of CDF tables plus guide tables, gathered at random, vs 126 MB L2",
                       "timing": "CUDA events on the launching stream (r3d_sync) + torch events around the reduction, max over ranks",
                       "wall_ms_per_step": 1e3 * wall_s / K,
                       "loop_events_per_second": events_total / dev_s, "events_per_phonon": events_total / total,
                       "model_built_by": "radiative3d_b200/workload_model.py"},
            "clocks": clocks, "gpu_launches": launches,
            "e2e": {"value": per * world / e2e_s, "unit": "phonons/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "what": ("r3d_create(pinned host model) + r3d_run + r3d_fetch(pinned host bins) + r3d_destroy, wall clock" if world == 1 else
                             "rank 0: H2D of the large tables from pinned memory + NCCL broadcast over NVLink; every rank: r3d_create(device "
                             "tables) + r3d_run of its share + reduction of the bins to rank 0 (2 NCCL collectives) + r3d_destroy; rank 0: "
                             "r3d_fetch into pinned host bins; wall clock, max over ranks")},
            "roofline": roofline, "roofline_issue": roofline_issue,
        }
        if cpu:
            out["cpu_baseline"] = cpu
        sys.stdout.flush()
        os.write(json_fd, (json.dumps(out) + "\n").encode())
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())

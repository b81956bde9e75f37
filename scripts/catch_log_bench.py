"""Cost of the catch log and of replaying the logged phonons.  On halfspace_nearsrc50 (1.25e8 phonons per step) and spherical
(4e6 per step), both at take-off-angle degree 9, steps alternate in one session between
  off       no log,
  all       every seismometer, every bin,
  distant   the seismometer farthest from the source, the later half of the bins,
each step over a new index range.  Step times are device seconds (CUDA events, r3d_sync).  Then the phonons of the last
"distant" step and of the last "all" step (at most 2^18 and 2^14 of each on the two models) are replayed with all event reports, timed on the host
around the call (it ends in a device synchronisation).  Prints one JSON line with the card's name and power limit; writes
nothing to the repository (optional --out FILE).

    python scripts/catch_log_bench.py [--steps 4] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from radiative3d_b200 import abi, engine, workload_model  # noqa: E402

SEED = 20261018


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    except OSError:
        return "unknown"
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def distant_seismometer(m):
    loc = m.seis.reshape(-1, abi.R3D_SEIS_NPARAM)[:, :3]
    return int(np.argmax(np.linalg.norm(loc - np.asarray(m.src_loc)[None, :], axis=1)))


def replay(eng, phonons, per_phonon_cap):
    t0 = time.perf_counter()
    try:
        ev = eng.trace_events_indices(phonons, SEED, capacity=max(4096, per_phonon_cap * phonons.size))
    except engine.R3DError as e:          # more events than room: reported, not retried
        return {"phonons": int(phonons.size), "error": str(e)}
    s = time.perf_counter() - t0
    return {"phonons": int(phonons.size), "events": int(ev.size), "seconds": s,
            "phonons_per_second": phonons.size / s if s > 0 else None}


def one_workload(name, per_step, steps, capacity, replay_max, events_per_phonon):
    m = workload_model.build_model(name, 9)
    far = distant_seismometer(m)
    modes = {"off": None, "all": dict(seismometers=None, bins=None),
             "distant": dict(seismometers=[far], bins=(m.n_bins // 2, m.n_bins))}
    secs = {k: [] for k in modes}
    records = {k: [] for k in modes}
    first = 0
    last = {}
    with engine.Engine(m) as eng:
        for warm in (True, False):
            for _ in range(1 if warm else steps):
                for mode, sel in modes.items():
                    if sel is None:
                        eng.set_catch_log(capacity=None)
                    else:
                        eng.set_catch_log(sel["seismometers"], sel["bins"], capacity)
                    eng.sync()
                    eng.run_simulation(per_step, seed=SEED, first_phonon=first)
                    s = eng.sync()
                    first += per_step
                    if sel is not None:
                        rec, matched = eng.fetch_catch_log()
                        last[mode] = rec
                        if not warm:
                            records[mode].append(matched)
                    if not warm:
                        secs[mode].append(s)
        eng.set_catch_log(capacity=None)
        ph_far = np.unique(last["distant"]["phonon"])[:replay_max]
        ph_all = np.unique(last["all"]["phonon"])[:replay_max]
        rep = {"distant": replay(eng, ph_far, events_per_phonon), "all_first": replay(eng, ph_all, events_per_phonon)}
    med = {k: float(np.median(v)) for k, v in secs.items()}
    return {"workload": name, "toa_degree": 9, "phonons_per_step": per_step, "distant_seismometer": far,
            "distant_bins": [m.n_bins // 2, m.n_bins], "capacity_per_device": capacity,
            "seconds": secs, "median_seconds": med,
            "overhead_all": med["all"] / med["off"] - 1.0, "overhead_distant": med["distant"] / med["off"] - 1.0,
            "records_per_step": {k: v for k, v in records.items() if v},
            "catches_per_phonon": float(np.mean(records["all"])) / per_step,
            "record_bytes_per_step_all": float(np.mean(records["all"])) * abi.CATCH_DTYPE.itemsize,
            "replay": rep}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=4, help="timed steps of each kind")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    out = {"card": card(), "workloads": [
        one_workload("halfspace_nearsrc50", 125_000_000, a.steps, 1 << 23, 1 << 18, 128),
        one_workload("spherical", 4_000_000, a.steps, 1 << 25, 1 << 14, 2048),
    ]}
    line = json.dumps(out)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()

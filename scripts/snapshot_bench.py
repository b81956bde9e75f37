"""Cost of energy snapshots on the benchmark workload: halfspace_nearsrc50 at take-off-angle degree 9, 1.25e8 phonons per
step, steps alternating between snapshots off and K = 16 times over [0, ttl] on a 128^3 grid over the box the
seismometers and the source span.  Prints one JSON line: device seconds of each step kind (CUDA events, r3d_sync), their
ratio, the card's name and power limit.  Writes nothing to the repository (optional --out FILE).

    python scripts/snapshot_bench.py [--steps 4] [--per-step 125000000] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from radiative3d_b200 import engine, workload_model  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=4, help="timed steps of each kind")
    ap.add_argument("--per-step", type=int, default=125000000)
    ap.add_argument("--dim", type=int, default=128)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    m = workload_model.build_model("halfspace_nearsrc50", 9)
    pts = np.vstack([np.asarray(m.src_loc)[None, :], m.seis.reshape(-1, 18)[:, :3]])
    lo, hi = pts.min(axis=0), pts.max(axis=0)
    ext = np.maximum(hi - lo, 1.0)
    lo, hi = lo - 0.05 * ext, hi + 0.05 * ext
    dims = (a.dim,) * 3
    voxel = (hi - lo) / a.dim
    times = np.linspace(0.0, m.ttl, 16)
    t_off, t_on = [], []
    first = 0
    with engine.Engine(m) as eng:
        for warm in (True, False):
            for step in range(1 if warm else a.steps):
                for on in (False, True):
                    eng.set_snapshots(times if on else None, lo, voxel, dims)
                    eng.sync()
                    eng.run_simulation(a.per_step, seed=20261018, first_phonon=first)
                    s = eng.sync()
                    first += a.per_step
                    if not warm:
                        (t_on if on else t_off).append(s)
        eng.set_snapshots(times, lo, voxel, dims)
        eng.run_simulation(a.per_step, seed=20261018)
        e, c, oe, oc = eng.fetch_snapshots()
    rec = c.reshape(16, -1).sum(axis=1) + oc.sum(axis=1)
    occupied = (c.reshape(16, -1, 2).sum(axis=2) > 0).sum(axis=1)
    out = {"workload": "halfspace_nearsrc50", "toa_degree": 9, "phonons_per_step": a.per_step, "snapshot_times": 16,
           "grid": list(dims), "grid_origin": lo.tolist(), "voxel": voxel.tolist(), "card": card(),
           "seconds_off": t_off, "seconds_on": t_on, "median_off": float(np.median(t_off)), "median_on": float(np.median(t_on)),
           "ratio_on_off": float(np.median(t_on) / np.median(t_off)),
           "records_per_snapshot": rec.tolist(), "outside_per_snapshot": oc.sum(axis=1).tolist(),
           "occupied_voxels_per_snapshot": occupied.tolist()}
    line = json.dumps(out)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()

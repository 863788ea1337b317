"""Cost of per-micrograph CTF groups at the cfg 2 shape (N = 224, DISPLACE_CENTER 40 1) with C = 8 CTFs per group.

Reports, on the GPU it runs on (card name and power limit are printed with the numbers):
  * ns per likelihood of the fused kernel, grouped variant against the ungrouped one (CUDA events around every launch);
  * the front end's share of a step (projection, FFT, conv sums: step wall time less fused-kernel time) at
    G = 1, 100 and 1000 groups of M = 1000 particles (G = 1000: one particle per group);
  * the wall time of the same work as G separate ungrouped runs (one handle per group, set-up excluded).

    python tools/ctf_groups_time.py [--orient 192] [--particles 1000] [--out results.json]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from bioem_b200 import api, synth  # noqa: E402
from bioem_b200.cases import Case, build_case  # noqa: E402

GRID = dict(synth.PRODUCTION_GRID, CTF_B_ENV=(2.0, 300.0, 1), CTF_DEFOCUS=(0.5, 2.5, 8))  # C = 8, 2 micro-m wide


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def timed_run(e, reps=2):
    """(wall ms of run() + synchronize, fused-kernel ms) of the best of reps full runs after one warm-up"""
    e.set_kernel_timing(True)
    e.run()
    e.synchronize()
    e.kernel_time()
    best = None
    for _ in range(reps):
        e.reset()
        t0 = time.perf_counter()
        e.run()
        e.synchronize()
        wall = (time.perf_counter() - t0) * 1e3
        lik = e.kernel_time()[0]
        if best is None or wall < best[0]:
            best = (wall, lik)
    return best


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--orient", type=int, default=192)
    ap.add_argument("--particles", type=int, default=1000)
    ap.add_argument("--groups", default="1,100,1000")
    ap.add_argument("--out", default=None, help="also write the numbers as JSON to this file")
    a = ap.parse_args()
    if api.lib().bioem_b200_device_count() == 0:
        raise SystemExit("ctf_groups_time: no CUDA device")
    M, O = a.particles, a.orient
    case = Case("cfg2g", 224, 1.0, 1000, M, 4608, O, GRID, 40, 1, particle_format="mrc", bulk_particles=16)
    cd = build_case(case)
    hi, parts = api.inputs_for_case(cd)
    C = hi.C
    res = dict(card=card(), N=224, C=C, M=M, O=O, rows=[])
    print(f"card: {res['card']}  N=224 C={C} M={M} O={O}", flush=True)

    def engine(cfg, ctf=None, grouped=None, particles=parts):
        e = api.Engine(cfg)
        e.upload_model(hi.points, hi.NormDen)
        e.upload_orientations(hi.angles)
        if grouped is not None:
            e.upload_ctf_groups(*grouped[0])
        else:
            e.upload_ctf(*ctf)
        e.upload_particles(particles)
        if grouped is not None:
            e.set_particle_groups(grouped[1])
        return e

    e = engine(hi.cfg, ctf=(hi.refCTF, hi.CtfParam))
    wall, lik = timed_run(e)
    e.close()
    n = O * C * M
    res["ungrouped"] = dict(wall_ms=wall, lik_ms=lik, ns_per_lik=lik * 1e6 / n, front_share=(wall - lik) / wall)
    print(f"ungrouped: step {wall:.1f} ms, fused kernel {lik:.1f} ms = {lik * 1e6 / n:.2f} ns/likelihood, "
          f"front end {100 * (wall - lik) / wall:.2f} %", flush=True)
    rng = np.random.default_rng(0)
    for G in (int(x) for x in a.groups.split(",")):
        defs = np.round(np.linspace(1.1, 5.9, G), 4).astype(np.float32)
        tables = hi.ctf_groups(defs, GRID)
        group = np.repeat(np.arange(G, dtype=np.int32), -(-M // G))[:M]
        group = group[rng.permutation(M)]  # interleaved in the stack, as micrographs come
        e = engine(hi.cfg, grouped=(tables, group))
        wall, lik = timed_run(e)
        e.close()
        # the same work as G separate runs (uploads outside the clock)
        sep = 0.0
        for g in range(G):
            idx = np.flatnonzero(group == g)
            cfg = api.Config.from_buffer_copy(hi.cfg)
            cfg.Priordefcent = tables[2][g]
            s = engine(cfg, ctf=(tables[0][g], tables[1][g]), particles=parts[idx])
            s.run()  # warm-up of this handle
            s.synchronize()
            s.reset()
            t0 = time.perf_counter()
            s.run()
            s.synchronize()
            sep += (time.perf_counter() - t0) * 1e3
            s.close()
        row = dict(G=G, wall_ms=wall, lik_ms=lik, ns_per_lik=lik * 1e6 / n, front_share=(wall - lik) / wall,
                   separate_runs_ms=sep)
        res["rows"].append(row)
        print(f"G={G}: step {wall:.1f} ms, fused kernel {lik * 1e6 / n:.2f} ns/likelihood, front end "
              f"{100 * row['front_share']:.2f} %, {G} separate runs {sep:.1f} ms", flush=True)
    if a.out:
        os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()

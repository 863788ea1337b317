"""Cost of rendering calculated images (Engine.render_maps) at the production shapes.

    python tools/render_time.py [--reps 5] [--json out.json]

cfg 2 shape: 1000 records of 224 x 224 with 1000 distinct orientations of the 4608-orientation list, 32 CTFs.
cfg 4 shape: 2000 records of 360 x 360, the 48^3-voxel model (110,592 points), 4608 orientations (about 1600 distinct).
Per shape it prints the wall time of the synchronous call (after one warm-up call), maps per second, the split between
the front end (projection, forward FFT, convolution) and the inverse transform from a separate torch.profiler run, and
the inverse transform's ns per map next to its memory bound (8 F bytes read, F = N (N/2 + 1), 4 N^2 bytes written, at
7.7 TB/s) and its FLOP count (2.5 N^2 log2 N^2).  The card's name and power limit are read in the same call.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))

import numpy as np  # noqa: E402

from bioem_b200 import api  # noqa: E402
from bioem_b200.cases import build_case  # noqa: E402

FRONT = ("project_kernel", "fft_rows_kernel", "fft_cols_kernel", "ctf_conv_kernel", "gen_dft_rows_kernel",
         "gen_dft_cols_kernel", "gen_conv_kernel")
INVERSE = ("render_cols_kernel", "render_rows_kernel", "gen_render_cols_kernel", "gen_render_rows_kernel")
HBM = 7.7e12


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return r.stdout.strip() if r.returncode == 0 else "unknown (nvidia-smi failed)"


def engine_for(name: str, n_records: int, seed: int):
    cd = build_case(name, n_particles=2)
    hi, parts = api.inputs_for_case(cd)
    e = api.Engine(hi.cfg, 0)
    e.upload_model(hi.points, hi.NormDen)
    e.upload_orientations(hi.angles)
    if hi.use_psf:
        e.upload_ctf_real(hi.psf_kernels, hi.CtfParam)
    else:
        e.upload_ctf(hi.refCTF, hi.CtfParam)
    e.upload_particles(parts)
    rng = np.random.default_rng(seed)
    rec = np.zeros(n_records, dtype=api.PROB_MAP_DTYPE)
    rec["orient"] = rng.choice(e.O, n_records, replace=n_records > e.O)
    rec["conv"] = rng.integers(0, e.C, n_records)
    rec["cent_x"] = rng.integers(-40, 41, n_records)
    rec["cent_y"] = rng.integers(-40, 41, n_records)
    rec["norm"] = rng.uniform(0.5, 2.0, n_records)
    rec["mu"] = rng.normal(0.0, 1.0, n_records)
    return hi, e, rec


def kernel_split(e, rec):
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.init()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        e.render_maps(rec)
        torch.cuda.synchronize()
    front = inverse = copies = 0.0
    per = {}
    for ev in prof.key_averages():
        us = getattr(ev, "device_time_total", None)
        if us is None:
            us = ev.cuda_time_total
        name = ev.key
        if not us or name.startswith("cuda"):  # (host-side runtime calls)
            continue
        per[name] = per.get(name, 0.0) + us
        if any(k in name for k in INVERSE):
            inverse += us
        elif any(k in name for k in FRONT):
            front += us
        elif "Memcpy" in name or "memcpy" in name:
            copies += us
    return front / 1e3, inverse / 1e3, copies / 1e3, {k: v / 1e3 for k, v in per.items()}


def measure(name: str, n_records: int, reps: int, seed: int) -> dict:
    hi, e, rec = engine_for(name, n_records, seed)
    try:
        N = hi.N
        e.render_maps(rec)  # warm-up: module load, batch buffers, memory pool
        times = []
        for _ in range(reps):
            t = time.perf_counter()
            e.render_maps(rec)
            times.append(time.perf_counter() - t)
        wall = float(np.median(times))
        front, inverse, copies, per = kernel_split(e, rec)
        F = N * (N // 2 + 1)
        flop = 2.5 * N * N * math.log2(N * N)
        byts = 8 * F + 4 * N * N
        ns_map = inverse * 1e6 / n_records
        bound_ns = byts / HBM * 1e9
        return dict(case=name, N=N, records=n_records, distinct_orientations=int(len(np.unique(rec["orient"]))),
                    C=e.C, model_points=int(len(hi.points)), wall_ms=wall * 1e3, wall_ms_all=[t * 1e3 for t in times],
                    maps_per_s=n_records / wall, front_ms=front, inverse_ms=inverse, copy_ms=copies,
                    inverse_ns_per_map=ns_map, inverse_bound_ns_per_map=bound_ns,
                    inverse_gflops=flop / ns_map, inverse_gbytes_per_s=byts / ns_map, kernels_ms=per)
    finally:
        e.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--json", default=None)
    a = ap.parse_args()
    if api.lib().bioem_b200_device_count() == 0:
        raise SystemExit("render_time.py: no CUDA device")
    out = dict(card=card(), shapes=[measure("cfg2", 1000, a.reps, 1), measure("cfg4", 2000, a.reps, 2)])
    print(f"card: {out['card']}")
    for r in out["shapes"]:
        print(f"{r['case']}: N={r['N']} records={r['records']} distinct orientations={r['distinct_orientations']} "
              f"C={r['C']} model points={r['model_points']}")
        print(f"  synchronous call {r['wall_ms']:.2f} ms (median of {len(r['wall_ms_all'])}), {r['maps_per_s']:.0f} maps/s")
        print(f"  profiled: front end {r['front_ms']:.2f} ms, inverse transform {r['inverse_ms']:.3f} ms, "
              f"device copies {r['copy_ms']:.2f} ms")
        print(f"  inverse transform {r['inverse_ns_per_map']:.0f} ns/map; memory bound {r['inverse_bound_ns_per_map']:.0f} "
              f"ns/map; {r['inverse_gflops']:.0f} GFLOP/s, {r['inverse_gbytes_per_s']:.0f} GB/s")
    if a.json:
        with open(a.json, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()

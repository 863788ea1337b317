#!/usr/bin/env python3
"""bench.py — throughput of the BioEM likelihood hot path on B200.

  python bench.py --gpus N --steps K --warmup W            (our arm, C ABI -> sm_100a kernels)
  python bench.py --impl reference --gpus N --steps K --warmup W   (reference CPU code on host cores)

Workload (BASELINE.json configs[1], "cfg2"): synthetic ~1k-point model vs 1000 synthetic
224x224 particles, QUATERNION_LIST_4608_Orient, production CTF grid (4 x 8 x 1 = 32 kernels),
DISPLACE_CENTER 40 1  ->  4608 * 32 * 1000 = 147,456,000 likelihoods per step.
A step = one full pass of the hot path (projection .. log-sum-exp/arg-max merge) over the whole
orientation grid.  With N GPUs the orientation grid is sharded in contiguous blocks (one process
per GPU), partial results are merged with one NCCL all-gather per step (strong scaling).

metric  likelihoods/s  = image x orientation x CTF triples per second (whole job, all GPUs)
value   inputs resident in HBM before the timed region (CUDA events on the library's stream)
e2e     the same job through the public API from pinned HOST buffers: upload (H2D) + device
        particle FFTs + run + download (D2H) inside the timed region
roofline  dominant kernel = likelihood_kernel<224>; algorithmic bytes per likelihood = 8*F =
        202,496 B (one streamed read of the particle half-spectrum, SURVEY §8d) over the kernel's
        CUDA-event time, against the measured HBM copy bandwidth (MEASURED_PEAKS.json)
cpu_baseline  the unmodified reference (oracle/_ref/bioEM_ref = reference sources + FFTW-API
        shim) on the host cores, on a bounded slice of the same workload
"""
from __future__ import annotations

import argparse
import json
import os
import re
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

WORKLOADS = {
    # name: (case name, particles, orientations) -- BASELINE.json configs[0..4]
    "cfg1": ("cfg1", 10, 576),
    "cfg2": ("cfg2", 1000, 4608),       # the headline: the configuration the metric is quoted on
    "cfg3": ("cfg3", 10000, 36864),     # 36864 orientations x 10k particles, orientation-sharded over the GPUs
    "cfg4": ("cfg4", 2000, 4608),       # 48^3 MRC voxel model (--ReadModelMRC), 360 x 360, dense CTF grid (256)
    "cfg5": ("cfg5", 5000, 4608),       # WRITE_PROB_ANGLES 10: per-orientation posterior table + top-K
}
# measured on this pool's B200 by tools/ubench/fp32x2.cu (gpurun_out/ubench_fp32x2.txt): FP32 FMA issue rate
FMA_OPS_PER_CLK_SM = 124.4


def _ncu_record(kernel: str) -> dict:
    """what the committed ncu --set full capture of the dominant kernel measured (profiles/ncu_traffic.json)"""
    p = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    try:
        return json.load(open(p)).get(kernel, {})
    except Exception:
        return {}


def _traffic(kernel: str, likelihoods_per_launch: float):
    """dram bytes per (average) launch of the dominant kernel, from the committed ncu capture
    (bytes per likelihood x likelihoods per launch), or None."""
    try:
        return int(float(_ncu_record(kernel)["dram_bytes_per_likelihood"]) * likelihoods_per_launch)
    except Exception:
        return None


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region."""

    def __init__(self, gpu_index: int):
        self.rows = []
        self.proc = None
        self.gpu = gpu_index

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self) -> dict:
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
                for k, nme in enumerate(names):
                    if r[3 + k].lower().startswith("active"):
                        reasons.add(nme)
            except Exception:
                pass
        # samples under load = upper half (the region is bracketed by idle moments)
        sm_sorted = sorted(sm)
        load = sm_sorted[len(sm_sorted) // 2:] if sm_sorted else []
        med = load[len(load) // 2] if load else None
        return {"sm_mhz": med, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def build_workload(name: str, n_particles: int | None = None, n_orient: int | None = None):
    from bioem_b200 import api
    from bioem_b200.cases import build_case
    cname, m, o = WORKLOADS[name]
    cd = build_case(cname, n_particles=n_particles, n_orient=n_orient)
    hi, parts = api.inputs_for_case(cd)
    return cd, hi, parts


def build_workload_shared(name, n_particles, n_orient, rank, world, barrier):
    """One rank of the box synthesises the particle stack (seconds of numpy per thousand images), the others
    load it from /dev/shm: every rank holds ALL particles (only the orientation grid is sharded)."""
    if world == 1:
        return build_workload(name, n_particles, n_orient)
    from bioem_b200 import api
    from bioem_b200.cases import build_case
    path = f"/dev/shm/bioem_b200_bench_{name}_{n_particles}_{n_orient}_{os.environ.get('MASTER_PORT', '0')}.npy"
    cname = WORKLOADS[name][0]
    if rank == 0:
        cd, hi, parts = build_workload(name, n_particles, n_orient)
        np.save(path, parts)
        barrier()
    else:
        barrier()
        parts = np.load(path)
        cd = build_case(cname, n_particles=1, n_orient=n_orient)  # model, orientations, CTF grid (cheap)
        hi, _ = api.inputs_for_case(cd)
    barrier()
    if rank == 0:
        try:
            os.remove(path)
        except OSError:
            pass
    return cd, hi, parts


def run_ours(args):
    import torch
    import torch.distributed as dist
    from bioem_b200 import api

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the hot path has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        # stdout carries exactly one JSON line: NCCL's own output (the version banner it prints at
        # NCCL_DEBUG=VERSION / WARN, warnings) goes to stderr
        # (NCCL honours NCCL_DEBUG_FILE only above the VERSION level)
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() in ("VERSION", "NONE", ""):
            os.environ["NCCL_DEBUG"] = "WARN"
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    cname, m_full, o_full = WORKLOADS[args.workload]
    n_or = min(args.orientations, o_full) if args.orientations else None
    n_pa = min(args.particles, m_full) if args.particles else None
    cd, hi, parts = build_workload_shared(args.workload, n_pa, n_or, rank, world, barrier)
    case = cd.case
    O, Cn, M, N = hi.O, hi.C, parts.shape[0], hi.N
    K = int(case.write_angles)
    o_lo, o_hi = rank * O // world, (rank + 1) * O // world  # reference bioem.cpp:748-753
    likelihoods_step = O * Cn * M

    eng = api.Engine(hi.cfg, local)
    eng.upload_all(hi, parts)
    eng.set_kernel_timing(True)  # CUDA events around every launch of the fused kernel (roofline accounting)
    stream = torch.cuda.ExternalStream(api.lib().bioem_b200_stream(eng._h), device=local)
    if world > 1:
        # the library's own NCCL communicator: rank 0 makes the id, torch.distributed only carries it (plumbing)
        idt = torch.zeros(128, dtype=torch.uint8, device="cuda")
        if rank == 0:
            idt.copy_(torch.frombuffer(bytearray(api.nccl_unique_id()), dtype=torch.uint8))
        dist.broadcast(idt, 0)
        eng.nccl_init(world, rank, bytes(idt.cpu().numpy().tobytes()))

    def step(e=eng, lo=o_lo, hi_=o_hi):
        e.reset()
        e.run(lo, hi_)
        if world > 1:
            # ONE ncclAllGather of the per-image (max, sum, arg-max) partials + the fold, on the library's stream
            e.merge_nccl()

    for _ in range(args.warmup):
        step()
    barrier()
    eng.kernel_time()  # drain the warm-up launches
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)
    eng.reset()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    t_wall0 = time.perf_counter()
    total_launches = 0
    for _ in range(args.steps):
        step()
        total_launches += eng.stats()[0]
    e1.record(stream)
    barrier()
    t_wall = time.perf_counter() - t_wall0
    ms_dev = e0.elapsed_time(e1)
    lik_ms, lik_launches = eng.kernel_time()  # every launch of the fused kernel inside the timed region
    clocks = sampler.stop() if rank == 0 else None
    t = torch.tensor([ms_dev], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total = float(t.item())
    pm, _ = eng.download(out_angles=False)
    refine = eng.exact_argmax_info()
    if args.dump_outputs:
        top = None
        if K:  # every rank takes part in the selection of the K most probable orientations
            top = eng.top_angles_nccl(K, o_lo, o_hi) if world > 1 else eng.download_top_angles(K)
        if rank == 0:
            dump_outputs(args.dump_outputs, pm, top)

    # ---- correctness behind the multi-GPU number: the sharded + NCCL-merged result of an orientation prefix
    # against ONE rank evaluating the same prefix alone (bit-identical records expected)
    result_check = None
    if world > 1:
        op = min(O, max(world, 64))
        eng.reset()
        eng.run(rank * op // world, (rank + 1) * op // world)
        eng.merge_nccl()
        sharded, _ = eng.download(out_angles=False)
        top_sh = eng.top_angles_nccl(K, rank * op // world, (rank + 1) * op // world) if K else None
        if rank == 0:
            eng.reset()
            eng.run(0, op)
            single, _ = eng.download(out_angles=False)
            same = sum(int(all(sharded[m][k] == single[m][k] for k in ("orient", "conv", "cent_x", "cent_y")))
                       for m in range(M))
            lp_s = np.log(sharded["Total"]) + sharded["Constoadd"]
            lp_1 = np.log(single["Total"]) + single["Constoadd"]
            result_check = {"orientations": op, "argmax_identical": f"{same}/{M}",
                            "max_rel_dlogp": float(np.max(np.abs(lp_s - lp_1) / np.abs(lp_1))),
                            "const_identical": bool((sharded["Constoadd"] == single["Constoadd"]).all())}
            if K:
                top_1 = eng.download_top_angles(K, 0, op)
                result_check["top_angles_identical"] = bool((top_sh["orient"] == top_1["orient"]).all())
        barrier()

    # ---- end to end through the public API, host buffers, copies inside the timed region
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory().numpy()  # noqa: E731
    h_parts, h_ctf, h_ang = pin(parts), pin(hi.refCTF), pin(hi.angles)
    h2d = h_parts.nbytes + h_ctf.nbytes + h_ang.nbytes + hi.points.nbytes + hi.CtfParam.nbytes
    out_maps = np.zeros(M, dtype=api.PROB_MAP_DTYPE)
    d2h = out_maps.nbytes + (M * K * api.TOP_ANGLE_DTYPE.itemsize if K else 0)
    e2e_steps = max(1, min(2, args.steps))

    def e2e_step():
        e = api.Engine(hi.cfg, local)
        e.upload_model(hi.points, hi.NormDen)
        e.upload_orientations(h_ang)
        e.upload_ctf(h_ctf, hi.CtfParam)
        e.upload_particles(h_parts)
        if world > 1:
            e.nccl_attach(eng.nccl_comm())  # the process's communicator is built once, like any NCCL application's
        e.reset()
        e.run(o_lo, o_hi)
        if world > 1:
            e.merge_nccl()
        e.download(out_maps, out_angles=False)
        if K:  # WRITE_PROB_ANGLES: the K most probable orientations per particle, selected on the device
            (e.top_angles_nccl(K, o_lo, o_hi) if world > 1 else e.download_top_angles(K))
        e.close()

    e2e_val = None
    if not args.no_e2e:
        e2e_step()  # warm
        barrier()
        t0 = time.perf_counter()
        for k in range(e2e_steps):
            e2e_step()
        barrier()
        te = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        e2e_val = likelihoods_step * e2e_steps / float(te.item())

    kmode = eng.cached_product()
    if rank == 0:
        hbm_peak, peak_src = _peaks()
        F = N * (N // 2 + 1)
        value = likelihoods_step * args.steps / (ms_total / 1e3)
        kname = f"likelihood_kernel<{N}>"
        roof = None
        if lik_launches:
            # per-rank kernel time covers this rank's share of the likelihoods
            per_rank_lik = (o_hi - o_lo) * Cn * M * args.steps
            ach = per_rank_lik * 8.0 * F / (lik_ms / 1e3) / 1e9
            flop = 2.5 * N * N * np.log2(N * N)
            mhz = clocks.get("sm_mhz") or clocks.get("sm_max_mhz") or 1965.0
            fp32_peak = 148 * 128 * 2 * mhz / 1e6
            fp32_ach = per_rank_lik * flop / (lik_ms / 1e3) / 1e12
            rec = _ncu_record(kname)
            roof = {"bound": "hbm", "achieved": round(ach, 1), "peak": hbm_peak, "unit": "GB/s",
                    "frac": round(ach / hbm_peak, 4), "traffic": _traffic(kname, per_rank_lik / lik_launches),
                    "peak_source": peak_src,
                    "kernel": kname, "launches": int(lik_launches),
                    "avg_launch_ms": round(lik_ms / lik_launches, 3),
                    "ns_per_likelihood": round(1e6 * lik_ms / per_rank_lik, 2),
                    "algorithmic_bytes_per_likelihood": 8 * F,
                    # "frac" is the ALGORITHMIC ratio SURVEY 8(d) defines (8F streamed bytes per likelihood over the
                    # kernel time, against the HBM copy peak): the operands are served by L2, so it is not measured
                    # DRAM utilisation -- that, and the units that actually bind, come from the ncu capture:
                    "measured_units_ncu": {k: rec[k] for k in ("dram_pct_of_peak", "lsu_data_pipe_pct", "fma_pipe_pct",
                                                                "issue_slot_pct", "l2_to_sm_bytes_per_likelihood",
                                                                "capture") if k in rec} or None,
                    "fp32_algorithmic_tflops": round(fp32_ach, 2),
                    # compute side of the two-sided FFT roofline (SURVEY 8d): 148 SMs x 128 FP32 lanes x 2 x SM clock
                    "fp32_peak_tflops": round(fp32_peak, 1), "fp32_frac": round(fp32_ach / fp32_peak, 4),
                    # the FMA issue rate tools/ubench/fp32x2.cu measured on this GPU (124.4 of 128 lanes per clock per SM)
                    "fp32_measured_peak_tflops": round(148 * FMA_OPS_PER_CLK_SM * 2 * mhz / 1e6, 1),
                    "fp32_frac_of_measured": round(fp32_ach / (148 * FMA_OPS_PER_CLK_SM * 2 * mhz / 1e6), 4),
                    "kernel_share_of_step": round(lik_ms / (ms_total), 4)}
        sliced = (n_or is not None and n_or < o_full) or (n_pa is not None and n_pa < m_full)
        line = {
            "metric": "likelihoods/s", "value": round(value, 1), "unit": "likelihoods/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": round(ms_total / args.steps, 3), "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"{args.workload}: {O} orientations x {Cn} CTF x {M} particles "
                                   f"{N}x{N}, DISPLACE_CENTER {case.max_disp} {case.grid_space}"
                                   + (f", WRITE_PROB_ANGLES {K}" if K else "")
                                   + (f", model = {case.voxel_model}^3 MRC volume ({hi.points.shape[0]} points)" if case.voxel_model else "")
                                   + (f" [slice of the named {o_full} x {m_full} shape]" if sliced else ""),
                       "likelihoods_per_step": likelihoods_step,
                       "parallelism": f"orientation-sharded x{world}, merge = one ncclAllGather inside the library" if world > 1 else "single GPU",
                       # which operands the fused kernel streams (bioem_b200_cached_product): real CTF kernels -> the
                       # product projection x conj(particle), cached per resident CTA, and the real CTF tables
                       "kernel_mode": {1: "cached product (real CTF kernels)", 0: "complex conv spectra"}.get(kmode, "undecided"),
                       "l2": f"inputs larger than L2 (particle spectra {M * 8 * F / 1e6:.0f} MB re-streamed per orientation group"
                             + (" + one scratch map per resident CTA)" if kmode == 1 else
                                " + up to 1.07 GB of conv spectra per launch)")},
            "clocks": clocks,
            "e2e": {"value": round(e2e_val, 1) if e2e_val else None, "unit": "likelihoods/s", "h2d_bytes_per_step": int(h2d),
                    "d2h_bytes_per_step": int(d2h), "steps": e2e_steps},
            "gpu_launches": int(total_launches),
            "roofline": roof,
            # the pass that evaluates the arg-max displacement of every particle's winning likelihood with the reference's
            # first-of-ties rule (exact_argmax_kernel): records evaluated / re-evaluations that did not reproduce the logpro
            "exact_argmax_pass": {"records": refine[0], "disagreed": refine[2]},
            "wall_s_timed_region": round(t_wall, 3),
        }
        if result_check is not None:
            line["result_check"] = result_check
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline(args.workload, budget_s=args.cpu_seconds)
            line["reference_gpu"] = reference_gpu(args.workload) if args.workload in ("cfg1", "cfg2") else None
        print(json.dumps(line), flush=True)
    eng.close()
    if world > 1:
        dist.destroy_process_group()


def dump_outputs(out_dir: str, pm: np.ndarray, top: np.ndarray | None) -> None:
    """Write what a caller of the timed path receives after its last step, one DIR/<field>.npy per field, so that two
    builds can be compared output for output on the same seeded inputs: the per-particle records (float64, exact for
    the integer fields; norm and mu as the float32 they are) and, with WRITE_PROB_ANGLES, the K most probable
    orientations per particle as top_<field>.npy.  At most 10,000 particles x 10 orientations: a few MB in all."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {k: pm[k].astype(np.float32 if pm.dtype[k] == np.float32 else np.float64) for k in pm.dtype.names}
    if top is not None:
        arrays.update({f"top_{k}": top[k].astype(np.float64) for k in ("orient", "forAngles", "ConstAngle")})
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, f"{k}.npy"), a)


def _mkl_lib() -> str:
    """PyTorch's libtorch_cpu.so is linked against Intel oneMKL and exports its DFTI entry points: the FFTW-API shim of
    the reference build (oracle/fftw_shim) binds them at run time when BIOEM_FFT_MKL_LIB names the file."""
    if os.environ.get("BIOEM_REF_FFT", "mkl") != "mkl":
        return ""
    try:
        import importlib.util
        spec = importlib.util.find_spec("torch")
        path = os.path.join(os.path.dirname(spec.origin), "lib", "libtorch_cpu.so")
        return path if os.path.exists(path) else ""
    except Exception:
        return ""


FFT_LABEL = {"mkl": "Intel oneMKL DFTI (the copy PyTorch bundles, bound at run time by oracle/fftw_shim; FFTW 3 is not in the image)",
             "builtin": "built-in engine of the FFTW-API shim (oracle/fft_core.hpp, builder code; FFTW 3 is not in the image)"}
_LAST_FFT = {"engine": "builtin"}


def _ref_slice(workload: str, n_orient: int, n_part: int, workdir: str, threads: int, stages: dict | None = None):
    """Run oracle/_ref/bioEM_ref on the first n_orient orientations x all CTFs x n_part particles
    of the workload; returns (likelihoods, seconds of the reference's own run() timer)."""
    from bioem_b200.cases import build_case, reference_cli
    cname, _, _ = WORKLOADS[workload]
    cd = build_case(cname, workdir, n_particles=n_part, n_orient=n_orient)
    refbin = os.path.join(ROOT, "oracle", "_ref", "bioEM_ref")
    env = {**os.environ, "OMP_NUM_THREADS": str(threads), "BIOEM_FFT_MKL_LIB": _mkl_lib()}
    env.pop("GPU", None)
    if stages is not None:
        env["BIOEM_DEBUG_OUTPUT"] = "1"  # the reference's own stage timers (timer.cpp:156-165)
    r = subprocess.run([refbin] + reference_cli(cd), cwd=workdir, env=env, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("reference binary failed: " + r.stdout[-500:] + r.stderr[-500:])
    sec = None
    for ln in r.stdout.splitlines():
        if ln.startswith("FFT engine:"):
            _LAST_FFT["engine"] = "mkl" if "oneMKL" in ln else "builtin"
        if "The code ran for" in ln:
            sec = float(ln.split("for")[1].split("seconds")[0])
        if stages is not None:
            mm = re.match(r"SUMMARY -> (.*?): Total ([0-9.eE+-]+) sec", ln)
            if mm:
                stages[mm.group(1).strip()] = float(mm.group(2))
    return cd.case.likelihoods, sec


def cpu_baseline(workload: str, budget_s: float = 15.0) -> dict:
    refbin = os.path.join(ROOT, "oracle", "_ref", "bioEM_ref")
    threads = os.cpu_count() or 1
    if not os.path.exists(refbin):
        return {"value": None, "unit": "likelihoods/s", "cores": threads, "kind": "reference",
                "sample": "oracle/_ref/bioEM_ref not present"}
    with tempfile.TemporaryDirectory() as d:
        cname, m_full, o_full = WORKLOADS[workload]
        # the reference parallelises over images (bioem.cpp:1392): give every thread some
        n_part = min(m_full, max(64, 4 * threads))
        n, s = _ref_slice(workload, 2, n_part, os.path.join(d, "probe"), threads)
        rate = n / max(s, 1e-6)
        # scale the slice to ~budget_s of CPU work (orientations first, then particles)
        per_orient = rate and (n / 2) / rate
        n_or = int(max(2, min(o_full, budget_s / max(per_orient, 1e-9))))
        if n_or > 64 and n_part < m_full:
            n_part = min(m_full, n_part * max(1, n_or // 64))
            n_or = 64
        n, s = _ref_slice(workload, n_or, n_part, os.path.join(d, "run"), threads)
        stages = {}
        try:  # a second, shorter run with the reference's stage timers on (they serialise some of its loops)
            _ref_slice(workload, max(2, n_or // 4), n_part, os.path.join(d, "stages"), threads, stages)
        except Exception:
            stages = {}
    from bioem_b200.cases import CASES
    return {"value": round(n / s, 1), "unit": "likelihoods/s", "cores": threads, "kind": "reference",
            # FFTW is not in this image: the reference's 9 FFTW symbols are served by oracle/fftw_shim, which hands the
            # transforms to Intel oneMKL when it can (else to its built-in engine)
            "fft": FFT_LABEL[_LAST_FFT["engine"]],
            "fft_microbench": _fft_microbench(CASES[WORKLOADS[workload][0]].n_pixels),
            "reference_stage_totals_s": stages or None,
            "sample": f"unmodified reference ({_LAST_FFT['engine']} FFT behind the FFTW-API shim, Algo 1, OpenMP {threads} threads) on the first "
                      f"{n_or} orientations x all CTFs x {n_part} particles of {workload} = {n} likelihoods in {s:.2f} s "
                      f"(reference's own run() timer)"}


def _fft_microbench(n: int) -> dict | None:
    """How much of the CPU baseline is the builder's FFT shim: one N x N c2r transform by the shim's engine
    (oracle/fft_core.hpp through liboracle.so) against numpy's pocketfft on the same core."""
    try:
        from oracle import pyoracle
        L = pyoracle.lib()
        rng = np.random.default_rng(0)
        X = np.ascontiguousarray(rng.normal(size=(n, n // 2 + 1, 2)).astype(np.float32))
        y = np.zeros((n, n), dtype=np.float32)
        reps = max(4, int(2e6 / (n * n)))
        Xc = X.copy()
        L.oracle_fft_c2r(n, pyoracle._fp(Xc), pyoracle._fp(y))
        t0 = time.perf_counter()
        for _ in range(reps):
            Xc[:] = X
            L.oracle_fft_c2r(n, pyoracle._fp(Xc), pyoracle._fp(y))
        t_shim = (time.perf_counter() - t0) / reps
        Z = (X[..., 0] + 1j * X[..., 1]).astype(np.complex64)
        np.fft.irfft2(Z, s=(n, n))
        t0 = time.perf_counter()
        for _ in range(reps):
            np.fft.irfft2(Z, s=(n, n))
        t_np = (time.perf_counter() - t0) / reps
        out = {"n": n, "builtin_shim_c2r_us": round(1e6 * t_shim, 1), "numpy_pocketfft_c2r_us": round(1e6 * t_np, 1),
               "note": "one core, one N x N c2r transform = the FFT work of one likelihood"}
        try:  # torch.fft on CPU is the same oneMKL the reference arm uses
            import torch
            torch.set_num_threads(1)
            zt = torch.from_numpy(Z)
            torch.fft.irfft2(zt, s=(n, n))
            t0 = time.perf_counter()
            for _ in range(reps):
                torch.fft.irfft2(zt, s=(n, n))
            out["mkl_c2r_us"] = round(1e6 * (time.perf_counter() - t0) / reps, 1)
        except Exception:
            pass
        return out
    except Exception as e:  # a side number
        return {"error": str(e)[:200]}


def reference_gpu(workload: str, n_orient: int = 8) -> dict:
    """The reference's own CUDA path (bioem_cuda.cu + cuFFT rebuilt for sm_100a, oracle/_ref/bioEM_ref_cuda,
    GPU=1 GPUWORKLOAD=100) on the first n_orient orientations of the workload on this box's GPU 0:
    likelihoods/s from its own per-orientation timer (SURVEY 8d, "reference GPU on the same box").
    Reported beside the CPU baseline; never part of a timed region of ours."""
    refbin = os.path.join(ROOT, "oracle", "_ref", "bioEM_ref_cuda")
    if not os.path.exists(refbin):
        return {"value": None, "unit": "likelihoods/s", "sample": "oracle/_ref/bioEM_ref_cuda not present"}
    from bioem_b200.cases import build_case, reference_cli
    cname, m_full, _ = WORKLOADS[workload]
    try:
        with tempfile.TemporaryDirectory() as d:
            cd = build_case(cname, d, n_particles=m_full, n_orient=n_orient)
            env = {**os.environ, "GPU": "1", "GPUWORKLOAD": "100", "GPUDEVICE": "0", "BIOEM_DEBUG_OUTPUT": "1",
                   "OMP_NUM_THREADS": str(os.cpu_count() or 1)}
            r = subprocess.run([refbin] + reference_cli(cd), cwd=d, env=env, capture_output=True, text=True,
                               timeout=300)
        if r.returncode != 0:
            raise RuntimeError((r.stdout[-300:] + r.stderr[-300:]).replace("\n", " | "))
        mean = None
        for ln in r.stdout.splitlines():
            if "Total time of projection" in ln:
                mean = float(ln.split("Mean")[1].split("sec")[0])
        per_or = cd.case.n_ctf * cd.case.n_particles
        return {"value": round(per_or / mean, 1), "unit": "likelihoods/s",
                "sample": f"unmodified reference CUDA path (bioem_cuda.cu + cuFFT, nvcc sm_100a, GPU=1 GPUWORKLOAD=100) "
                          f"on 1 GPU: mean {mean * 1e3:.1f} ms per orientation over the first {n_orient} orientations x "
                          f"{cd.case.n_ctf} CTFs x {cd.case.n_particles} particles of {workload} (its own timer)"}
    except Exception as e:  # a reported side number: never fail the bench for it
        return {"value": None, "unit": "likelihoods/s", "sample": f"failed: {e}"[:300]}


def run_reference(args):
    """Reference arm: the reference's own CPU implementation of the path on the host cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    refbin = os.path.join(ROOT, "oracle", "_ref", "bioEM_ref")
    if not os.path.exists(refbin):
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/bioEM_ref was not built"}))
        return
    cname, m_full, o_full = WORKLOADS[args.workload]
    from bioem_b200.cases import CASES
    case = CASES[cname]
    with tempfile.TemporaryDirectory() as d:
        n_part = min(m_full, max(64, 4 * threads))
        n, s = _ref_slice(args.workload, 2, n_part, os.path.join(d, "probe"), threads)
        per_orient = s / 2
        # every step is one run of the reference on a slice; the slice is sized so that warm-up + steps stay within
        # about three minutes of CPU work in total
        per_step = min(args.cpu_seconds, 180.0 / max(1, args.steps + args.warmup))
        n_or = int(max(2, min(o_full, per_step / max(per_orient, 1e-9))))
        times = []
        for k in range(args.warmup + args.steps):
            n, s = _ref_slice(args.workload, n_or, n_part, os.path.join(d, f"s{k}"), threads)
            if k >= args.warmup:
                times.append(s)
    total = sum(times)
    value = n * len(times) / total
    sample = (f"each step = unmodified reference (oracle/_ref/bioEM_ref: reference sources + FFTW-API shim, FFT engine = "
              f"{_LAST_FFT['engine']}, Algo 1, OpenMP {threads} threads) on the first {n_or} orientations x {case.n_ctf} CTFs x {n_part} "
              f"particles of {args.workload} = {n} likelihoods; time = the reference's own run() timer")
    line = {
        "impl": "reference", "metric": "likelihoods/s", "value": round(value, 1), "unit": "likelihoods/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": round(1e3 * total / len(times), 3), "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{args.workload}: {o_full} orientations x {case.n_ctf} CTF x {m_full} particles "
                               f"{case.n_pixels}x{case.n_pixels}, DISPLACE_CENTER {case.max_disp} {case.grid_space}",
                   "likelihoods_per_step": n, "parallelism": f"host OpenMP x{threads}"},
        "cpu_baseline": {"value": round(value, 1), "unit": "likelihoods/s", "cores": threads, "kind": "reference",
                         "fft": FFT_LABEL[_LAST_FFT["engine"]],
                         "sample": sample},
        "e2e": {"value": round(value, 1), "unit": "likelihoods/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2,
                    help="timed steps of the measurement (the end-to-end leg, which rebuilds every input per step, times "
                         "min(2, steps) of its own; e2e.steps reports them)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg2", choices=sorted(WORKLOADS))
    ap.add_argument("--orientations", type=int, default=0,
                    help="use only the first K orientations of the workload's list (bounded runs of cfg3 / cfg4; stated in config.workload)")
    ap.add_argument("--particles", type=int, default=0, help="use only the first M particles of the workload (stated in config.workload)")
    ap.add_argument("--cpu-seconds", type=float, default=15.0, help="CPU work budget of one reference sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true", help="skip the end-to-end leg (profiling runs only)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step as DIR/<name>.npy (inputs are seeded: same arguments, "
                         "same inputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of --impl ours; the reference arm times the reference binary")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()

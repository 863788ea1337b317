"""GPU test of the measurement contract: bench.py prints exactly one JSON line on stdout with the keys
the driver reads (on the small cfg1 workload, without the CPU legs, so that it runs in seconds)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from bioem_b200 import api
from bioem_b200.cases import build_case

pytestmark = pytest.mark.gpu
ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))


def test_bench_line_has_the_contract_keys():
    if api.lib().bioem_b200_device_count() == 0:
        pytest.fail("no CUDA device visible: the gpu-marked tests must run on the B200 box")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "cfg1", "--steps", "5", "--warmup", "3",
                        "--no-cpu-baseline"], capture_output=True, text=True, cwd=ROOT, timeout=600)
    assert r.returncode == 0, r.stderr[-800:]
    lines = [ln for ln in r.stdout.split("\n") if ln.strip()]
    assert len(lines) == 1, r.stdout[:500]
    d = json.loads(lines[0])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "clocks", "e2e", "gpu_launches", "roofline"):
        assert k in d, k
    assert d["metric"] == "likelihoods/s" and d["unit"] == "likelihoods/s" and d["higher_is_better"] is True
    assert d["n_gpus"] == 1 and d["steps"] == 5 and d["warmup"] == 3 and d["vs_baseline"] is None
    assert "workload" in d["config"] and d["data"] == "synthetic"
    assert d["value"] > 0 and d["gpu_launches"] > 0
    assert d["e2e"]["value"] > 0 and d["e2e"]["h2d_bytes_per_step"] > 0 and d["e2e"]["d2h_bytes_per_step"] > 0
    # the driver runs --steps 20: the roofline must not depend on the number of steps
    assert d["roofline"] is not None and d["roofline"]["launches"] >= 5
    for k in ("bound", "achieved", "peak", "unit", "frac", "traffic"):
        assert k in d["roofline"], k
    assert abs(d["roofline"]["frac"] - d["roofline"]["achieved"] / d["roofline"]["peak"]) < 1e-3
    for k in ("sm_mhz", "sm_max_mhz", "reasons"):
        assert k in d["clocks"], k


def test_bench_dumps_what_the_last_timed_step_computed(tmp_path):
    """--dump-outputs: the per-particle records and the WRITE_PROB_ANGLES top-K table of the last timed step, as
    float32 / float64 .npy files, equal to what the library returns for the same seeded inputs outside bench.py."""
    if api.lib().bioem_b200_device_count() == 0:
        pytest.fail("no CUDA device visible: the gpu-marked tests must run on the B200 box")
    out = tmp_path / "dump"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "cfg5", "--particles", "8",
                        "--orientations", "64", "--steps", "2", "--warmup", "1", "--no-cpu-baseline", "--no-e2e",
                        "--dump-outputs", str(out)], capture_output=True, text=True, cwd=ROOT, timeout=600)
    assert r.returncode == 0, r.stderr[-800:]
    got = {p.stem: np.load(p) for p in out.glob("*.npy")}
    fields = list(api.PROB_MAP_DTYPE.names)
    assert set(got) == set(fields) | {"top_orient", "top_forAngles", "top_ConstAngle"}
    assert all(a.dtype in (np.float32, np.float64) for a in got.values())
    assert sum(a.nbytes for a in got.values()) <= 64 << 20
    cd = build_case("cfg5", n_particles=8, n_orient=64)
    hi, parts = api.inputs_for_case(cd)
    eng = api.Engine(hi.cfg)
    try:
        eng.upload_all(hi, parts)
        eng.run()
        pm, _ = eng.download(out_angles=False)
        top = eng.download_top_angles(cd.case.write_angles)
    finally:
        eng.close()
    for k in fields:
        np.testing.assert_array_equal(got[k], pm[k])
    for k in ("orient", "forAngles", "ConstAngle"):
        np.testing.assert_array_equal(got["top_" + k], top[k])

"""Per-micrograph CTF groups (bioem_b200_upload_ctf_groups / bioem_b200_set_particle_groups, bioEM_b200
--DefocusPerParticle).

Contract: a grouped run over G groups of C rows gives what G separate ungrouped runs give -- run g with group g's
table, prior centre and particles only -- with max_prob_conv mapped to the row of the whole table, g*C + c.  These tests
pin the batch geometry (BIOEM_B200_OB / BIOEM_B200_OG) on both sides and assert every record field, Total included,
bit for bit; the angle table and the top-K rows likewise.  A grouped table always runs the cached-product mode, so the
separate runs are pinned to it too (BIOEM_B200_CACHED_PRODUCT=1).
"""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from bioem_b200 import api, synth
from bioem_b200.cases import CFG1_CTF, Case, build_case, reference_cli
from oracle import pyoracle
from tests import likmodel
from tests.test_gpu_likelihoods import EPS32, TOTAL_RTOL, VALUE_K
from tests.test_gpu_parity import LOGP_ATOL, _need_gpu

pytestmark = pytest.mark.gpu

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
EXE = os.path.join(ROOT, "bioem_b200", "bin", "bioEM_b200")

# 12 real CTFs over a 1 micro-m defocus window (every group then has >= 4 rows: the cached-product mode's own choice)
GRID32 = dict(CTF_DEFOCUS=(1.0, 2.0, 3), CTF_B_ENV=(2.0, 300.0, 2), CTF_AMPLITUDE=(0.05, 0.25, 2))
SHAPES = {
    32: Case("grp32", 32, 1.5, 60, 24, 576, 10, GRID32, 4, 1, write_angles=3, model_sigma=5.0, model_rmax=12.0),
    64: Case("grp64", 64, 1.5, 200, 20, 576, 8, synth.PRODUCTION_GRID, 10, 1, write_angles=4, model_sigma=10.0,
             model_rmax=26.0, particle_format="mrc"),
    224: Case("grp224", 224, 1.0, 1000, 7, 4608, 6, synth.PRODUCTION_GRID, 40, 1, write_angles=2,
              particle_format="mrc"),
}
_DATA = {}


def _inputs(N):
    if N not in _DATA:
        cd = build_case(SHAPES[N])
        _DATA[N] = (cd,) + api.inputs_for_case(cd)
    return _DATA[N]


def _groups(M, G):
    """uneven, interleaved groups with one group of a single particle (the last); G = M: one group per particle"""
    if G == 1:
        return np.zeros(M, np.int32)
    if G == M:
        return np.random.default_rng(5).permutation(M).astype(np.int32)
    g = np.array([(m * 7 + m // 3) % (G - 1) for m in range(M)], np.int32)
    g[M // 2] = G - 1
    assert set(g) == set(range(G))
    return g


def _defocus(ctf, G):
    """one defocus value [micro-m] per group inside the allowed range of the grid's width"""
    d0, d1, _ = ctf["CTF_DEFOCUS"]
    half = 0.5 * (d1 - d0)
    return np.linspace(half + 0.1, min(8.0 - half, half + 4.0), G).astype(np.float32)


def _pin(monkeypatch, ob=3, og=2):
    monkeypatch.setenv("BIOEM_B200_OB", str(ob))
    monkeypatch.setenv("BIOEM_B200_OG", str(og))
    monkeypatch.setenv("BIOEM_B200_CACHED_PRODUCT", "1")


def _engine(hi, cfg, parts):
    e = api.Engine(cfg)
    e.upload_model(hi.points, hi.NormDen)
    e.upload_orientations(hi.angles)
    return e


def _grouped(hi, parts, tables, group, cfg=None):
    ref, par, cen = tables
    e = _engine(hi, cfg or hi.cfg, parts)
    e.upload_ctf_groups(ref, par, cen)
    e.upload_particles(parts)
    e.set_particle_groups(group)
    return e


def _separate(hi, parts, tables, group, g):
    ref, par, cen = tables
    cfg = api.Config.from_buffer_copy(hi.cfg)
    cfg.Priordefcent = cen[g]
    e = _engine(hi, cfg, parts)
    e.upload_ctf(ref[g], par[g])
    idx = np.flatnonzero(group == g)
    e.upload_particles(parts[idx])
    return e, idx


def _assert_records(got, want, C, g, tag):
    w = want.copy()
    w["conv"] += g * C
    for k in PROB_FIELDS:
        np.testing.assert_array_equal(got[k], w[k], err_msg=f"{tag}: {k}")


PROB_FIELDS = ("Total", "Constoadd", "cent_x", "cent_y", "orient", "conv", "norm", "mu")


# ----------------------------------------------------------------------------- 1. equivalence with separate runs

EQUIV = [(32, 1), (32, 3), (32, 17), (32, 24), (64, 3), (64, 20), (224, 3)]


@pytest.mark.parametrize("N,G", EQUIV, ids=[f"N{n}-G{g}" for n, g in EQUIV])
@pytest.mark.parametrize("angles", [0, 1], ids=["noangles", "angles"])
def test_grouped_run_equals_separate_runs(monkeypatch, N, G, angles):
    _need_gpu()
    _pin(monkeypatch)
    cd, hi, parts = _inputs(N)
    cfg = api.Config.from_buffer_copy(hi.cfg)
    if not angles:
        cfg.writeAngles = 0
    hi2 = api.HostInputs.__new__(api.HostInputs)
    hi2.__dict__.update(hi.__dict__)
    hi2.cfg = cfg
    M, K = len(parts), max(1, int(cfg.writeAngles))
    group = _groups(M, G)
    tables = hi.ctf_groups(_defocus(cd.case.ctf, G), cd.case.ctf)
    e = _grouped(hi2, parts, tables, group, cfg)
    e.run()
    pm, pa = e.download()
    assert e.cached_product() == 1
    top = e.download_top_angles(K) if angles else None
    _, n_lik = e.stats()
    assert n_lik == e.O * hi.C * M
    for g in range(G):
        s, idx = _separate(hi2, parts, tables, group, g)
        s.run()
        spm, spa = s.download()
        _assert_records(pm[idx], spm, hi.C, g, f"N={N} G={G} group {g}")
        if angles:
            np.testing.assert_array_equal(pa[:, idx], spa)
            np.testing.assert_array_equal(top[idx], s.download_top_angles(K))
        s.close()
    e.close()


def test_one_group_equals_upload_ctf(monkeypatch):
    """G = 1 with the config's prior centre: bit for bit the ungrouped upload_ctf run"""
    _need_gpu()
    _pin(monkeypatch)
    cd, hi, parts = _inputs(64)
    e = _grouped(hi, parts, (hi.refCTF[None], hi.CtfParam[None], None), np.zeros(len(parts), np.int32))
    e.run()
    pm, pa = e.download()
    u = _engine(hi, hi.cfg, parts)
    u.upload_ctf(hi.refCTF, hi.CtfParam)
    u.upload_particles(parts)
    u.run()
    upm, upa = u.download()
    for k in PROB_FIELDS:
        np.testing.assert_array_equal(pm[k], upm[k], err_msg=k)
    np.testing.assert_array_equal(pa, upa)
    # the conv parameters of the grouped front end (ctf_sums_kernel) equal ctf_conv_kernel's
    for o, c in ((0, 0), (e.O - 1, hi.C - 1)):
        assert e.debug_convolved(o, c)[1:] == u.debug_convolved(o, c)[1:]
    e.close()
    u.close()


# ----------------------------------------------------------------------------- 2. every likelihood

@pytest.mark.parametrize("N,G", [(32, 3), (64, 20)], ids=["N32-G3", "N64-G20"])
def test_every_captured_likelihood_of_a_grouped_run(monkeypatch, N, G):
    """run_capture of a grouped run: every window entry written, every value within FP32-FFT error of the float64
    window of the particle's own group CTF, download() equal to the fold of the captured values"""
    _need_gpu()
    for v in ("BIOEM_B200_OB", "BIOEM_B200_OG", "BIOEM_B200_CACHED_PRODUCT"):
        monkeypatch.delenv(v, raising=False)
    cd, hi, parts = _inputs(N)
    group = _groups(len(parts), G)
    tables = hi.ctf_groups(_defocus(cd.case.ctf, G), cd.case.ctf)
    e = _grouped(hi, parts, tables, group)
    cap = e.run_capture()
    pm, pa = e.download()
    O, Cn, M = e.O, hi.C, e.M
    assert cap.shape[:3] == (O, Cn, M)
    assert not np.isnan(cap).any(), np.argwhere(np.isnan(cap))[:8]
    xs = likmodel.window(hi.N, hi.cfg.maxDisplaceCenter, hi.cfg.GridSpaceCenter)
    refs, sR, ssR = zip(*(e.debug_particle(m) for m in range(M)))
    refs, sR, ssR = np.stack(refs), np.array(sR, np.float32), np.array(ssR, np.float32)
    a = 0.5 * (3.0 - hi.cfg.Ntotpi)
    worst = 0.0
    for g in range(G):
        idx = np.flatnonzero(group == g)
        cfg = api.Config.from_buffer_copy(hi.cfg)
        cfg.Priordefcent = tables[2][g]
        pri = [likmodel.prior(type("H", (), {"cfg": cfg}), tables[1][g, c]) for c in range(Cn)]
        lp = np.empty((O, Cn, len(idx), cap.shape[-1] ** 2))
        for o in range(O):
            for c in range(Cn):
                conv, sC, ssC = e.debug_convolved(o, g * Cn + c)
                win, rms = likmodel.corr_windows(conv[None], refs[idx], hi.N, xs)
                got = cap[o, c, idx]
                scale = EPS32 * np.log2(hi.N ** 2) * np.maximum(rms[0] * np.sqrt(hi.N), np.abs(win[0]).max(axis=(-1, -2)))
                worst = max(worst, float((np.abs(got - win[0]).max(axis=(-1, -2)) / scale).max()))
                lp[o, c] = likmodel.logpro(got.reshape(len(idx), -1), sR[idx, None], ssR[idx, None], sC, ssC,
                                           hi.cfg.Ntotpi, pri[c])
        for j, m in enumerate(idx):
            want = likmodel.fold(lp[:, :, j], kernel=True, a=a)
            r = pm[m]
            assert r["Constoadd"] == want["Constoadd"], (g, m)
            assert (r["orient"], r["conv"]) == (want["orient"], g * Cn + want["conv"]), (g, m)
            assert (r["cent_x"], r["cent_y"]) == likmodel.centre(hi.N, hi.cfg.maxDisplaceCenter,
                                                                 hi.cfg.GridSpaceCenter, want["lin"])
            assert abs(r["Total"] / want["Total"] - 1) <= TOTAL_RTOL + want["err"] / want["Total"], (g, m)
            if pa is not None:
                np.testing.assert_array_equal(pa[:, m]["ConstAngle"], want["ConstAngle"])
                arel = np.abs(pa[:, m]["forAngles"] / want["forAngles"] - 1)
                assert np.all(arel <= TOTAL_RTOL + want["err_angles"] / want["forAngles"]), (g, m)
    assert worst <= VALUE_K, worst
    e.close()


# ----------------------------------------------------------------------------- 3. oracle pin

def test_three_groups_match_the_oracle_per_group(monkeypatch):
    _need_gpu()
    monkeypatch.delenv("BIOEM_B200_CACHED_PRODUCT", raising=False)
    case = Case("grp32o", 32, 1.5, 60, 9, 576, 12, dict(CFG1_CTF, CTF_DEFOCUS=(1.0, 2.0, 4)), 4, 1,
                model_sigma=5.0, model_rmax=12.0)
    cd = build_case(case)
    hi, parts = api.inputs_for_case(cd)
    defs = np.array([1.25, 2.5, 3.75], np.float32)
    group = np.array([0, 1, 2, 2, 0, 1, 1, 0, 2], np.int32)
    e = _grouped(hi, parts, hi.ctf_groups(defs, case.ctf), group)
    e.run()
    pm, _ = e.download()
    Cn = hi.C
    for g, d in enumerate(defs):
        idx = np.flatnonzero(group == g)
        half = np.float32(0.5) * (np.float32(2.0) - np.float32(1.0))
        ctf = dict(case.ctf, CTF_DEFOCUS=(float(d - half), float(d + half), 4), PRIOR_DEFOCUS_CENTER=float(d))
        P = pyoracle.Prepared(Case(**{**case.__dict__, "ctf": ctf, "n_particles": len(idx)}), cd.model, cd.quats,
                              cd.particles[idx])
        ref = P.run()["prob"]
        for j, m in enumerate(idx):
            lg = hi.final_logprob(pm[m]["Total"], pm[m]["Constoadd"])
            lo = P.final_logprob(ref[j]["Total"], ref[j]["Constoadd"])
            assert abs(lg - lo) <= LOGP_ATOL[32] and abs(lg - lo) <= 1e-4 * abs(lo), (g, m, lg, lo)
            same = (pm[m]["orient"], pm[m]["conv"], pm[m]["cent_x"], pm[m]["cent_y"]) == \
                (ref[j]["orient"], g * Cn + ref[j]["conv"], ref[j]["cent_x"], ref[j]["cent_y"])
            # a near-tie may pick another maximum: then the oracle's logpro there is within the parity tolerance
            if not same:
                alt = P.logpro_at(j, int(pm[m]["orient"]), int(pm[m]["conv"]) - g * Cn, int(pm[m]["cent_x"]),
                                  int(pm[m]["cent_y"]))
                assert abs(alt - ref[j]["Constoadd"]) <= LOGP_ATOL[32], (g, m)
    e.close()


# ----------------------------------------------------------------------------- 4. consumers, refusals

def test_render_and_merge_peers_of_grouped_runs(monkeypatch):
    _need_gpu()
    _pin(monkeypatch)
    cd, hi, parts = _inputs(32)
    G = 3
    group = _groups(len(parts), G)
    tables = hi.ctf_groups(_defocus(cd.case.ctf, G), cd.case.ctf)
    e = _grouped(hi, parts, tables, group)
    e.run()
    pm, pa = e.download()
    maps = e.render_maps(pm)
    for g in range(G):
        s, idx = _separate(hi, parts, tables, group, g)
        s.run()
        spm, _ = s.download()
        np.testing.assert_array_equal(maps[idx], s.render_maps(spm))
        s.close()
    # two grouped handles over orientation blocks, merged on the device == one grouped handle
    h = [_grouped(hi, parts, tables, group) for _ in range(2)]
    cut = e.O // 2
    h[0].run(0, cut)
    h[1].run(cut, e.O)
    for x in h:
        x.synchronize()
    api.merge_peers(h)
    mpm, _ = h[0].download(out_angles=False)
    for k in ("Constoadd", "cent_x", "cent_y", "orient", "conv", "norm", "mu"):
        np.testing.assert_array_equal(mpm[k], pm[k], err_msg=k)
    np.testing.assert_allclose(mpm["Total"], pm["Total"], rtol=1e-12)
    for x in h + [e]:
        x.close()


def _rc(fn, *args):
    return getattr(api.lib(), fn)(*args)


def test_grouped_refusals_and_invalidation(monkeypatch):
    _need_gpu()
    monkeypatch.delenv("BIOEM_B200_CACHED_PRODUCT", raising=False)
    cd, hi, parts = _inputs(32)
    fp = ctypes.POINTER(ctypes.c_float)
    ip = ctypes.POINTER(ctypes.c_int)
    ref, par, cen = hi.ctf_groups(_defocus(cd.case.ctf, 2), cd.case.ctf)
    e = _engine(hi, hi.cfg, parts)
    h = e._h
    r, p = np.ascontiguousarray(ref), np.ascontiguousarray(par)
    # G < 1, C < 1, a complex kernel
    assert _rc("bioem_b200_upload_ctf_groups", h, r.ctypes.data_as(fp), p.ctypes.data_as(fp), None, 0, hi.C) == 1
    assert _rc("bioem_b200_upload_ctf_groups", h, r.ctypes.data_as(fp), p.ctypes.data_as(fp), None, 2, 0) == 1
    rc = r.copy()
    rc[1, 2, 5, 1] = 1e-3
    assert _rc("bioem_b200_upload_ctf_groups", h, rc.ctypes.data_as(fp), p.ctypes.data_as(fp), None, 2, hi.C) == 1
    assert "imaginary" in api.lib().bioem_b200_last_error().decode()
    # the list before a grouped table / particles
    g = np.zeros(len(parts), np.int32)
    assert _rc("bioem_b200_set_particle_groups", h, g.ctypes.data_as(ip), len(g)) == 3
    e.upload_ctf_groups(ref, par, cen)
    e.upload_particles(parts)
    # no list: run refuses; wrong count / group out of range
    assert _rc("bioem_b200_run", h, 0, e.O) == 3
    assert _rc("bioem_b200_set_particle_groups", h, g.ctypes.data_as(ip), len(g) - 1) == 1
    bad = g.copy()
    bad[3] = 2
    assert _rc("bioem_b200_set_particle_groups", h, bad.ctypes.data_as(ip), len(g)) == 1
    e.set_particle_groups(g)
    e.run()
    first, _ = e.download()
    # a new list invalidates the running state: a second run does not fold into the first
    e.set_particle_groups(g)
    e.run()
    again, _ = e.download()
    np.testing.assert_array_equal(again["Total"], first["Total"])
    # the cached-product mode cannot be switched off for a grouped table
    monkeypatch.setenv("BIOEM_B200_CACHED_PRODUCT", "0")
    e.upload_ctf_groups(ref, par, cen)  # (keeps the list: its groups exist)
    assert _rc("bioem_b200_run", h, 0, e.O) == 1
    monkeypatch.delenv("BIOEM_B200_CACHED_PRODUCT")
    # new particles drop the list; upload_ctf drops the grouped table (and with it the list)
    e.upload_particles(parts)
    assert _rc("bioem_b200_run", h, 0, e.O) == 3
    e.upload_ctf(hi.refCTF, hi.CtfParam)
    assert _rc("bioem_b200_set_particle_groups", h, g.ctypes.data_as(ip), len(g)) == 3
    e.run()
    e.close()
    # direct-DFT edges and USE_PSF take no grouped table
    for name, N in (("toy33", 33), ("toy32psf", 32)):
        cd2 = build_case(name)
        hi2, parts2 = api.inputs_for_case(cd2)
        e2 = _engine(hi2, hi2.cfg, parts2)
        F = N * (N // 2 + 1)
        t = np.zeros((2, 3, F, 2), np.float32)
        q = np.zeros((2, 3, 4), np.float32)
        assert _rc("bioem_b200_upload_ctf_groups", e2._h, t.ctypes.data_as(fp), q.ctypes.data_as(fp), None, 2, 3) == 1
        e2.close()


# ----------------------------------------------------------------------------- 5. binary

def _tokens(path):
    return [ln.split(" ") for ln in open(path, encoding="utf-8").read().split("\n")]


@pytest.mark.parametrize("gpus", [1, 2])
def test_binary_defocus_per_particle_equals_per_group_runs(tmp_path, gpus):
    """--DefocusPerParticle with 3 groups == bioEM_b200 once per group (shifted CTF_DEFOCUS, PRIOR_DEFOCUS_CENTER =
    the value, that group's particles), RefMap numbers mapped back: Output_Probabilities and ANG_PROB token for token"""
    _need_gpu()
    if not os.path.exists(EXE):
        subprocess.check_call(["make", "-C", os.path.join(ROOT, "bioem_b200", "csrc", "host")])
    case = SHAPES[32]
    cd = build_case(case, str(tmp_path / "all"))
    defs = np.array([1.5, 2.25, 3.0], np.float32)
    group = _groups(case.n_particles, 3)
    (tmp_path / "all" / "defocus.txt").write_text("\n".join(f"{defs[g]:.9g}" for g in group) + "\n")
    env = {**os.environ, "BIOEM_B200_OVERSUBSCRIBE": "1"} if gpus > 1 else dict(os.environ)
    cli = reference_cli(cd) + ["--DefocusPerParticle", "defocus.txt", "--Gpus", str(gpus)]
    r = subprocess.run([EXE] + cli, cwd=tmp_path / "all", capture_output=True, text=True, env=env)
    assert r.returncode == 0, r.stdout[-800:] + r.stderr[-800:]
    got_p, got_a = _tokens(tmp_path / "all" / "Output_Probabilities"), _tokens(tmp_path / "all" / "ANG_PROB")
    f32 = np.float32
    half = f32(0.5) * (f32(case.ctf["CTF_DEFOCUS"][1]) - f32(case.ctf["CTF_DEFOCUS"][0]))
    want_p, want_a = {}, {}
    for g, d in enumerate(defs):
        idx = np.flatnonzero(group == g)
        wd = tmp_path / f"g{g}"
        wd.mkdir()
        ctf = dict(case.ctf, CTF_DEFOCUS=(f"{d - half:.9g}", f"{d + half:.9g}", case.ctf["CTF_DEFOCUS"][2]),
                   PRIOR_DEFOCUS_CENTER=f"{d:.9g}")
        synth.write_param_file(str(wd / "param.txt"), case.n_pixels, case.pixel_size, case.max_disp, case.grid_space,
                               ctf, True, case.write_angles)
        synth.write_particles_text(str(wd / "particles.txt"), cd.particles[idx])
        r = subprocess.run([EXE, "--Modelfile", cd.paths["model"], "--Particlesfile", "particles.txt", "--Inputfile",
                            "param.txt", "--ReadOrientation", cd.paths["orient"], "--Gpus", "1"],
                           cwd=wd, capture_output=True, text=True)
        assert r.returncode == 0, r.stdout[-800:] + r.stderr[-800:]
        for src, dst in ((_tokens(wd / "Output_Probabilities"), want_p), (_tokens(wd / "ANG_PROB"), want_a)):
            for t in src:
                if len(t) > 2 and (t[0] == "RefMap:" or (t[0] == "" and t[1].isdigit())):
                    m = int(idx[int(t[1])])
                    dst.setdefault(m, []).append(t[:1] + [str(m)] + t[2:])
    hdr = next(i for i, t in enumerate(got_p) if t[0] == "RefMap:")
    body = [t for t in got_p[hdr:] if len(t) > 2]
    assert body == [t for m in range(case.n_particles) for t in want_p[m]]
    rows = [t for t in got_a if len(t) > 2 and t[0] == "" and t[1].isdigit()]
    assert rows == [t for m in range(case.n_particles) for t in want_a[m]]

"""Calculated particle images: bioem_b200_render_maps, Engine.render_maps and bioEM_b200 --WriteBestMaps.

A rendered map is norm * R0 shifted by the record's displacement, plus mu, where R0 = c2r(V) / N^2 is the convolved
projection of the record's orientation and CTF.  Checks:
  1. every map against a float64 model built from the GPU's own conv spectrum (debug_convolved: numpy irfft2, which
     sees only the Hermitian part of the self-conjugate columns as any c2r does, quirk Q1), in FP32-FFT error units;
  2. identities with the library's own numbers: sum R0 = sumC; sum R0^2 = sumsquareC less the anti-Hermitian energy of
     the self-conjugate columns (sumsquareC is the reference's Parseval sum over the whole half-spectrum, which a real
     image cannot carry); the window value debug_correlation at the record's displacement is sum R0_shifted * I; the
     records' norm / mu solve the least-squares normal equations of I ~ norm * R0 + mu with sumsquareC in place of
     sum R0^2 (what the reference's formula does);
  3. planted images made from the oracle's convolved projection: the record names the planted orientation, CTF and
     displacement, and rendering the planted parameters gives back the planted image;
  4. the running state, batching and refusals; 5. the binary's MRC stack.
"""
import os
import subprocess

import numpy as np
import pytest

from bioem_b200 import api
from bioem_b200.cases import build_case, reference_cli
from oracle import pyoracle
from tests import likmodel
from tests.test_gpu_likelihoods import EPS32, _case, _case_inputs, _custom
from tests.test_gpu_parity import _all_edges, _engine_with, _need_gpu

pytestmark = pytest.mark.gpu

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
EXE = os.path.join(ROOT, "bioem_b200", "bin", "bioEM_b200")
# rendered - float64 model <= VALUE_K * EPS32 * log2(N^2) * max(|norm| rms(R0) sqrt(N), max |model|)
VALUE_K = 4.0
# sums over the image against the library's FP32 numbers, relative to the magnitudes involved
SUM_K = 32.0


def _env(monkeypatch, mode=None, ob=None):
    for var, val in (("BIOEM_B200_CACHED_PRODUCT", mode), ("BIOEM_B200_OB", ob), ("BIOEM_B200_OG", None)):
        if val is None:
            monkeypatch.delenv(var, raising=False)
        else:
            monkeypatch.setenv(var, str(val))


def _engine(monkeypatch, spec, mode=None, ob=None):
    _need_gpu()
    _env(monkeypatch, mode, ob)
    hi, parts, ctf, cfg = _case_inputs(spec)
    return hi, parts, ctf, _engine_with(hi, parts, ctf=ctf, cfg=cfg)


def _records(n, O, C, N, seed):
    """random records: any orientation, CTF, |cent| < N, norm and mu"""
    rng = np.random.default_rng(seed)
    r = np.zeros(n, dtype=api.PROB_MAP_DTYPE)
    r["orient"] = rng.integers(0, O, n)
    r["conv"] = rng.integers(0, C, n)
    r["cent_x"] = rng.integers(-N + 1, N, n)
    r["cent_y"] = rng.integers(-N + 1, N, n)
    r["norm"] = rng.uniform(-3.0, 3.0, n)
    r["mu"] = rng.normal(0.0, 2.0, n)
    return r


def _r0(e, o, c, cache):
    """float64 R0 = c2r(V) / N^2 from the GPU's own conv spectrum, with the GPU's sumC / sumsquareC"""
    if (o, c) not in cache:
        N = e.cfg.NumberPixels
        conv, s, ss = e.debug_convolved(o, c)
        V = (conv[:, 0].astype(np.float64) + 1j * conv[:, 1]).reshape(N, N // 2 + 1)
        cache[(o, c)] = (np.fft.irfft2(V, s=(N, N)), s, ss)
    return cache[(o, c)]


def _model(e, rec, cache):
    """float64 maps of the records and their error units"""
    N = e.cfg.NumberPixels
    out = np.empty((len(rec), N, N))
    unit = np.empty(len(rec))
    for i, r in enumerate(rec):
        R0 = _r0(e, int(r["orient"]), int(r["conv"]), cache)[0]
        nm, mu = float(r["norm"]), float(r["mu"])
        out[i] = nm * np.roll(R0, (int(r["cent_x"]), int(r["cent_y"])), axis=(0, 1)) + mu
        unit[i] = EPS32 * np.log2(N * N) * max(abs(nm) * np.sqrt((R0 ** 2).mean()) * np.sqrt(N), np.abs(out[i]).max())
    return out, unit


def _check_model(tag, e, rec, got, cache):
    want, unit = _model(e, rec, cache)
    ratio = np.abs(got - want).max(axis=(1, 2)) / unit
    worst = float(ratio.max())
    assert worst <= VALUE_K, (tag, worst, rec[int(np.argmax(ratio))])
    return worst


def _anti_energy(hi, ctf, e, o, c):
    """(1/N^2) sum over the self-conjugate columns of |(V[kx] - conj V[-kx]) / 2|^2: what sumsquareC counts and no
    real image carries.  V = P conj(K) from the GPU's projection and the uploaded CTF table, in float64."""
    N = hi.N
    P = np.fft.rfft2(e.debug_projection(o).astype(np.float64))
    if ctf is not None:
        tab = ctf[0][c]
    elif hi.use_psf:
        K = np.fft.rfft2(hi.psf_kernels[c].astype(np.float64))
        tab = None
    else:
        tab = hi.refCTF[c]
    if tab is not None:
        K = (tab[:, 0].astype(np.float64) + 1j * tab[:, 1]).reshape(N, N // 2 + 1)
    V = P * np.conj(K)
    cols = [0] + ([N // 2] if N % 2 == 0 else [])
    d = 0.0
    for k in cols:
        v = V[:, k]
        a = 0.5 * (v - np.conj(np.roll(v[::-1], 1)))
        d += float((np.abs(a) ** 2).sum())
    return d / (N * N)


def _lin(N, maxd, G, cx, cy):
    nw = maxd // G + 1 + (maxd + G - 1) // G
    for lin in range(nw * nw):
        if likmodel.centre(N, maxd, G, lin) == (cx, cy):
            return lin // nw, lin % nw
    raise AssertionError((cx, cy))


# ----------------------------------------------------------------------------- 1 + 2: float64 model, identities

MODEL_CASES = [
    ("toy32", _case("toy32"), 0), ("toy32", _case("toy32"), 1), ("toy36g2", _case("toy36g2"), None),
    ("toy32psf", _case("toy32psf"), None), ("toy32euler", _case("toy32euler"), None),
    ("cfg2_slice", _case("cfg2_slice"), 0), ("cfg2_slice", _case("cfg2_slice"), 1),
    ("cfg4_slice", _case("cfg4_slice", ctf=8), None),  # N = 360: one CTA per SM for the likelihood
    ("toy33", _case("toy33"), None), ("toy26", _case("toy26"), None),  # direct-DFT path
]


@pytest.mark.parametrize("name,spec,mode", [pytest.param(n, s, m, id=n if m is None else f"{n}-mode{m}")
                                            for n, s, m in MODEL_CASES])
def test_rendered_maps_match_float64_model_and_identities(monkeypatch, name, spec, mode):
    hi, parts, ctf, e = _engine(monkeypatch, spec, mode)
    try:
        e.run()
        pm, _ = e.download()
        if mode is not None:
            assert e.cached_product() == mode
        N, maxd, G = hi.N, hi.cfg.maxDisplaceCenter, hi.cfg.GridSpaceCenter
        rec = np.concatenate([pm, _records(24, e.O, e.C, N, seed=N)])
        got = e.render_maps(rec)
        assert got.shape == (len(rec), N, N) and got.dtype == np.float32
        cache = {}
        worst = _check_model(name, e, rec, got, cache)
        # identities at norm = 1, mu = 0, every particle's record
        unit_rec = pm.copy()
        unit_rec["norm"], unit_rec["mu"] = 1.0, 0.0
        S = e.render_maps(unit_rec).astype(np.float64)
        gap = 0.0
        for m in range(e.M):
            o, c = int(pm[m]["orient"]), int(pm[m]["conv"])
            _, sC, ssC = _r0(e, o, c, cache)
            Sm, Im = S[m], parts[m].astype(np.float64)
            absS = np.abs(Sm).sum()
            assert abs(Sm.sum() - sC) <= SUM_K * EPS32 * np.log2(N * N) * absS, (name, m, Sm.sum(), sC)
            delta = _anti_energy(hi, ctf, e, o, c)
            sq = (Sm ** 2).sum()
            assert abs(sq - (ssC - delta)) <= SUM_K * EPS32 * np.log2(N * N) * ssC, (name, m, sq, ssC, delta)
            gap = max(gap, ssC / sq - 1)
            wx, wy = _lin(N, maxd, G, int(pm[m]["cent_x"]), int(pm[m]["cent_y"]))
            v = float(e.debug_correlation(o, c, m)[wx, wy])
            mag = np.sqrt(sq * (Im ** 2).sum())
            assert abs((Sm * Im).sum() - v) <= SUM_K * EPS32 * np.log2(N * N) * mag, (name, m, (Sm * Im).sum(), v)
            # normal equations of the record's fit: residual orthogonal to the constant image, and to R0 up to norm * delta
            nm, mu = float(pm[m]["norm"]), float(pm[m]["mu"])
            res = Im - nm * Sm - mu
            scale = np.abs(Im).sum() + abs(nm) * absS + abs(mu) * N * N
            assert abs(res.sum()) <= 64 * EPS32 * scale, (name, m, res.sum(), scale)
            lhs = (Sm * res).sum()
            assert abs(lhs - nm * delta) <= 64 * EPS32 * (mag + abs(nm) * ssC + abs(mu) * absS), (name, m, lhs, nm * delta)
        print(f"\n[render] {name} mode {e.cached_product()}: N={N} records={len(rec)} value/FFT-bound {worst:.3f}"
              f"  sumsquareC / sum R0^2 - 1 up to {gap:.2e} (quirk Q1)")
    finally:
        e.close()


@pytest.mark.parametrize("n", _all_edges())
def test_every_fused_edge_renders_a_random_record_before_any_run(monkeypatch, n):
    """one random record per instantiated fused edge, on a handle that has never run"""
    hi, parts, ctf, e = _engine(monkeypatch, _custom(n, min(10, n // 4), n_orient=2))
    try:
        rec = _records(2, e.O, e.C, n, seed=n)
        got = e.render_maps(rec)
        _check_model(f"edge{n}", e, rec, got, {})
    finally:
        e.close()


# ----------------------------------------------------------------------------- 3: planted images

PLANT = [(5, 1, 3, -2, 2.5, 0.7), (11, 2, -4, 1, 0.8, -1.5), (0, 0, 0, 4, 1.3, 0.1)]  # o, c, cent_x, cent_y, norm, mu


@pytest.mark.parametrize("name,mode", [("toy32", 0), ("toy32", 1), ("toy32psf", None), ("toy33", None)])
def test_planted_images_pinned_to_the_oracle(monkeypatch, name, mode):
    """Particles norm * shift(R0, cent) + mu made in float64 from the oracle's convolved projection, plus a 1 % noise
    orthogonal to the planted image and to the constant image (so that the fit is well defined).  The record names the
    planted orientation, CTF and displacement -- asymmetric in x and y, so the axes and the sign are pinned -- and
    rendering the planted parameters gives back the planted image.  The records' own norm / mu equal the planted ones
    only where the CTF kernels are Hermitian (PSF): for the reference's CTF table the sumsquareC in their formula
    carries the quirk-Q1 energy that the image does not."""
    _need_gpu()
    _env(monkeypatch, mode)
    cd = build_case(name)
    P = pyoracle.Prepared(cd.case, cd.model, cd.quats, cd.particles)
    N = P.N
    rng = np.random.default_rng(11)
    signal, imgs = [], []
    for o, c, cx, cy, nm, mu in PLANT:
        conv = P.convolve(P.projection(o), c)[0]
        V = (conv[:, 0].astype(np.float64) + 1j * conv[:, 1]).reshape(N, N // 2 + 1)
        S = np.roll(np.fft.irfft2(V, s=(N, N)), (cx, cy), axis=(0, 1))
        s = nm * S + mu
        noise = rng.normal(size=(N, N)) * 0.01 * abs(nm) * S.std()
        noise -= noise.mean()
        S0 = S - S.mean()
        noise -= (noise * S0).sum() / (S0 * S0).sum() * S0
        signal.append(s)
        imgs.append(s + noise)
    signal = np.array(signal)
    hi, _ = api.inputs_for_case(cd)
    e = _engine_with(hi, np.array(imgs, np.float32))
    try:
        e.run()
        pm, _ = e.download()
        want = np.zeros(len(PLANT), dtype=api.PROB_MAP_DTYPE)
        for k, name_ in enumerate(("orient", "conv", "cent_x", "cent_y", "norm", "mu")):
            want[name_] = [p[k] for p in PLANT]
        for m in range(len(PLANT)):
            assert (pm[m]["orient"], pm[m]["conv"], pm[m]["cent_x"], pm[m]["cent_y"]) == tuple(PLANT[m][:4]), (m, pm[m])
        got = e.render_maps(want).astype(np.float64)
        rms = np.sqrt(((signal - signal.mean(axis=(1, 2), keepdims=True)) ** 2).mean(axis=(1, 2)))
        err = np.abs(got - signal).max(axis=(1, 2)) / rms
        assert err.max() <= 64 * EPS32 * np.log2(N * N) * np.sqrt(N), err
        if hi.use_psf:
            np.testing.assert_allclose(pm["norm"], want["norm"], rtol=1e-4)
            best = e.render_maps(pm).astype(np.float64)
            assert (np.abs(best - signal).max(axis=(1, 2)) / rms).max() <= 1e-3
        print(f"\n[render] planted {name}: rendered - planted up to {err.max():.2e} x rms")
    finally:
        e.close()


# ----------------------------------------------------------------------------- 4: state, batching, refusals

def test_rendering_leaves_the_running_state_untouched(monkeypatch):
    spec = _case("toy32", angles=3)
    outs = []
    for render in (False, True):
        hi, parts, ctf, e = _engine(monkeypatch, spec, mode=1)
        try:
            e.run()
            before = e.stats()
            if render:
                e.render_maps(_records(40, e.O, e.C, hi.N, seed=1))
                assert e.stats() == before
            pm, pa = e.download()
            outs.append((pm.tobytes(), pa.tobytes(), e.exact_argmax_info(), e.out_of_frame()[0].tobytes(),
                         e.out_of_frame()[1], e.stats()))
        finally:
            e.close()
    assert outs[0] == outs[1]


def test_batches_of_many_orientations_equal_one_record_at_a_time(monkeypatch):
    """1000 records over several hundred distinct orientations under a small OB: the same bits as one call per record"""
    spec = _custom(32, 4, n_orient=400)
    hi, parts, ctf, e = _engine(monkeypatch, spec, ob=7)
    try:
        rec = _records(1000, e.O, e.C, hi.N, seed=3)
        assert len(np.unique(rec["orient"])) >= 300
        got = e.render_maps(rec)
        for i in range(len(rec)):
            np.testing.assert_array_equal(e.render_maps(rec[i:i + 1])[0], got[i], err_msg=str(i))
        _check_model("ob7", e, rec[:50], got[:50], {})
        assert e.render_maps(rec[:0]).shape == (0, hi.N, hi.N)
    finally:
        e.close()


def test_invalid_records_are_refused(monkeypatch):
    hi, parts, ctf, e = _engine(monkeypatch, _case("toy32"))
    L = api.lib()
    N = hi.N
    try:
        good = _records(3, e.O, e.C, N, seed=2)
        out = np.zeros((3, N, N), np.float32)
        for field, val, msg in (("orient", e.O, "orientation"), ("orient", -1, "orientation"), ("conv", e.C, "CTF"),
                                ("cent_x", N, "displacement"), ("cent_y", -N, "displacement")):
            bad = good.copy()
            bad[1][field] = val
            assert L.bioem_b200_render_maps(e._h, bad.ctypes.data, 3, api._fp(out)) == 1  # BIOEM_B200_ERR_INVALID
            err = L.bioem_b200_last_error().decode()
            assert msg in err and "record 1" in err, err
        assert L.bioem_b200_render_maps(e._h, good.ctypes.data, -1, api._fp(out)) == 1
        assert "negative" in L.bioem_b200_last_error().decode()
        assert L.bioem_b200_render_maps(e._h, None, 3, api._fp(out)) == 1
        assert L.bioem_b200_render_maps(e._h, good.ctypes.data, 3, None) == 1
        assert "null" in L.bioem_b200_last_error().decode()
        assert L.bioem_b200_render_maps(e._h, None, 0, None) == 0
    finally:
        e.close()
    # missing uploads
    bare = api.Engine(hi.cfg)
    try:
        assert L.bioem_b200_render_maps(bare._h, good.ctypes.data, 3, api._fp(out)) == 3  # BIOEM_B200_ERR_STATE
        assert "uploaded" in L.bioem_b200_last_error().decode()
        with pytest.raises(api.BioemError):
            bare.render_maps(good)
    finally:
        bare.close()


# ----------------------------------------------------------------------------- 5: the binary

def _run_binary(name, tmp_path, extra=(), env=None):
    if not os.path.exists(EXE):
        subprocess.check_call(["make", "-C", os.path.join(ROOT, "bioem_b200", "csrc", "host")])
    cd = build_case(name, str(tmp_path))
    r = subprocess.run([EXE] + reference_cli(cd) + list(extra), cwd=tmp_path, capture_output=True, text=True,
                       env={**os.environ, **(env or {})})
    assert r.returncode == 0, r.stdout[-800:] + r.stderr[-800:]
    return cd


def _read_stack(path, N):
    """the MRC reader's layout: maps[i][x][y] = file[j = y][i = x] per image"""
    raw = open(path, "rb").read()
    hdr = np.frombuffer(raw[:1024], np.int32)
    assert (hdr[0], hdr[1], hdr[3]) == (N, N, 2)
    data = np.frombuffer(raw[1024 + int(hdr[23]):], np.float32).reshape(int(hdr[2]), N, N)
    return np.ascontiguousarray(np.transpose(data, (0, 2, 1)))


@pytest.mark.parametrize("name", ["toy32", "cfg2_slice"])
def test_binary_writes_the_best_fit_maps(name, tmp_path):
    _need_gpu()
    plain, best = tmp_path / "plain", tmp_path / "best"
    plain.mkdir()
    best.mkdir()
    _run_binary(name, plain)
    cd = _run_binary(name, best, ["--WriteBestMaps", "best.mrc"])
    assert open(plain / "Output_Probabilities").read() == open(best / "Output_Probabilities").read()
    hi, parts = api.inputs_for_case(cd)
    e = _engine_with(hi, parts)
    try:
        e.run()
        pm, _ = e.download()
        want = e.render_maps(pm)
    finally:
        e.close()
    got = _read_stack(best / "best.mrc", hi.N)
    assert got.shape == want.shape
    np.testing.assert_array_equal(got, want)
    if name == "toy32":
        # the same stack when the orientation grid is split over two handles and merged on the device
        two = tmp_path / "two"
        two.mkdir()
        _run_binary(name, two, ["--WriteBestMaps", "best.mrc", "--Gpus", "2"], env={"BIOEM_B200_OVERSUBSCRIBE": "1"})
        assert open(two / "best.mrc", "rb").read() == open(best / "best.mrc", "rb").read()

"""Every likelihood of a production run against a float64 model (tests/likmodel.py).

Engine.run_capture (bioem_b200_debug_run_values) runs what run() runs -- batches of OB orientations, OG orientations per
CTA, the kernel mode the inputs select -- and returns every correlation window the fused kernel (or the direct-DFT
path) computed on the way.  For every case:
  1. coverage: every window entry of every (orientation, CTF, particle) was written (the capture is prefilled with NaN);
  2. values: every captured value against the window computed in double from the GPU's own operands, in units of the
     error of an FP32 FFT;
  3. inspection path: debug_correlation returns the captured window bit for bit;
  4. epilogue: download() against the fold of the GPU's own captured values in the path's semantics.
Geometry: captures of different (OB, OG) are bit-identical.  Pure-noise particles give flat posteriors: there every
likelihood carries about 1/(O*C) of Total, so a likelihood that is lost or wrong shows in Total and the angle table.

The tests at the top need no GPU: they rehearse the model against the oracle.
"""
import numpy as np
import pytest

from bioem_b200 import api, synth
from bioem_b200.cases import CASES, DENSE_CTF, Case, build_case
from oracle import pyoracle
from tests import likmodel
from tests.test_gpu_parity import _engine_with, _need_gpu

EPS32 = 2.0 ** -24
# captured value - float64 window <= VALUE_K * EPS32 * log2(N^2) * max(rms(map) * sqrt(N), max |window|)
VALUE_K = 4.0
# Total and the angle table against the fold of the captured values, relative, on top of the model's own bound
# (likmodel.fold "err": the fused kernel's cubic for a*log1p(t); on the direct-DFT path the terms whose logpro may narrow
# to the neighbouring float).  Fused kernel: the terms of the sum of exp carry ex2.approx (2 ulps) and rcp.approx (1 ulp)
# in the argument, the FP32 partial sums over a thread, a warp and the CTA about ten roundings.  Direct-DFT path: sums in
# double.
TOTAL_RTOL = 16 * EPS32
DOUBLE_RTOL = 1e-12


# ----------------------------------------------------------------------------- model rehearsal (no GPU)

@pytest.mark.parametrize("name", ["toy32", "toy36g2", "toy33"])
def test_float64_window_matches_oracle_correlation(name):
    """likmodel.corr_windows against the oracle's FP32 cross-correlation: layout, window order and sign"""
    cd = build_case(name)
    P = pyoracle.Prepared(cd.case, cd.model, cd.quats, cd.particles)
    N = P.N
    xs = likmodel.window(N, P.case.max_disp, P.case.grid_space)
    worst = 0.0
    for o, c in ((0, 0), (P.O - 1, P.C - 1)):
        conv = P.convolve(P.projection(o), c)[0]
        win, rms = likmodel.corr_windows(conv, P.RefMapsFFT, N, xs)
        for m in range(P.M):
            want = P.cross_correlation(conv, m) / np.float32(N * N)
            bound = EPS32 * np.log2(N * N) * max(rms[m] * np.sqrt(N), np.abs(win[m]).max())
            worst = max(worst, np.abs(want[np.ix_(xs, xs)] - win[m]).max() / bound)
    assert worst <= VALUE_K, worst


@pytest.mark.parametrize("name", ["toy32", "toy36g2", "toy33", "toy35g2"])
def test_reference_fold_reproduces_oracle(name):
    """The reference-semantics fold over the oracle's own per-displacement logpro reproduces its records.  logpro of
    the traced correlation values: without the multiply-add (the oracle is compiled with -ffp-contract=off) it is the
    oracle's bit for bit; with it, as the library computes, firstele moves by at most two ulps of its largest term."""
    cd = build_case(name)
    P = pyoracle.Prepared(cd.case, cd.model, cd.quats, cd.particles)
    sums = [[P.convolve(P.projection(o), c)[1:] for c in range(P.C)] for o in range(P.O)]
    pri = [likmodel.prior(P, P.CtfParam[c]) for c in range(P.C)]
    for m in range(P.M):
        res = P.run(trace_image=m)
        tl, tv = res["trace_logpro"], res["trace_value"]
        for o in range(P.O):
            for c in range(P.C):
                args = (tv[o, c], P.sumRef[m], P.sumsqRef[m], *sums[o][c], P.cfg.Ntotpi)
                np.testing.assert_array_equal(likmodel.logpro(*args, pri[c], fused=False).astype(np.float32), tl[o, c])
                fe, big = likmodel.firstele(*args)
                # one rounding of the product less, and the three roundings after it: within 2 ulps of the largest term
                assert np.all(np.abs(fe - likmodel.firstele(*args, fused=False)[0]) <= 2 * np.spacing(big)), (m, o, c)
        got = likmodel.fold(tl, kernel=False)
        want = res["prob"][m]
        assert got["Constoadd"] == want["Constoadd"]
        cx, cy = likmodel.centre(P.N, P.case.max_disp, P.case.grid_space, got["lin"])
        assert (got["orient"], got["conv"], cx, cy) == (want["orient"], want["conv"], want["cent_x"], want["cent_y"])
        assert abs(got["Total"] / want["Total"] - 1) <= 1e-12
        if res["angle"] is not None:
            np.testing.assert_array_equal(got["ConstAngle"], res["angle"][:, m]["ConstAngle"])
            np.testing.assert_allclose(got["forAngles"], res["angle"][:, m]["forAngles"], rtol=1e-12)
        # the kernel's semantics moves each term by at most one ulp of logpro (see _check)
        k = likmodel.fold(tl.astype(np.float64), kernel=True)
        assert abs(np.log(k["Total"] / got["Total"])) <= np.spacing(np.float32(np.abs(tl).max()))


# ----------------------------------------------------------------------------- GPU: capture and check

def _case_inputs(spec):
    """(HostInputs, particles, ctf or None, cfg) of one case spec"""
    base = spec["case"]
    case = CASES[base] if isinstance(base, str) else base
    if "o" in spec or "m" in spec:
        case = Case(**{**case.__dict__, "n_orient": spec.get("o", case.n_orient), "n_particles": spec.get("m", case.n_particles)})
    cd = build_case(case)
    hi, parts = api.inputs_for_case(cd)
    if spec.get("noise"):
        # normalised Gaussian images: after marginalising over normalisation and offset their logpro varies by O(1) nats
        # only, the posterior is flat; plus one clean particle whose terms nearly all underflow
        rng = np.random.default_rng(7)
        noise = rng.normal(size=(spec["noise"], hi.N, hi.N))
        ctfp = synth.ctf_grid_params(case.ctf)
        clean, _ = synth.make_particles(cd.model, cd.quats, hi.N, case.pixel_size, 1, case.max_disp, ctfp, snr=1e12,
                                        seed=3)
        parts = api.HostInputs.normalise_particles(np.concatenate([noise, clean]).astype(np.float32))
    ctf = None
    if "ctf" in spec:
        ctf = (np.ascontiguousarray(hi.refCTF[:spec["ctf"]]), np.ascontiguousarray(hi.CtfParam[:spec["ctf"]]))
    cfg = api.Config.from_buffer_copy(hi.cfg)
    if "angles" in spec:
        cfg.writeAngles = spec["angles"]
    return hi, parts, ctf, cfg


def _capture(monkeypatch, spec, ob=None, og=None, mode=None):
    """Engine of the case under the given geometry / kernel mode: (engine, capture, maps, angle table)"""
    for var, val in (("BIOEM_B200_OB", ob), ("BIOEM_B200_OG", og), ("BIOEM_B200_CACHED_PRODUCT", mode)):
        if val is None:
            monkeypatch.delenv(var, raising=False)
        else:
            monkeypatch.setenv(var, str(val))
    hi, parts, ctf, cfg = _case_inputs(spec)
    e = _engine_with(hi, parts, ctf=ctf, cfg=cfg)
    cap = e.run_capture()
    pm, pa = e.download()
    if mode is not None:
        assert e.cached_product() == int(mode)
    return hi, ctf, e, cap, pm, pa


def _model(e, hi, ctf, cap):
    """float64 windows, map rms and double logpro [O, C, M, D] of every captured value, from the GPU's own operands"""
    N, O, Cn, M = hi.N, e.O, e.C, e.M
    xs = likmodel.window(N, hi.cfg.maxDisplaceCenter, hi.cfg.GridSpaceCenter)
    refs, sR, ssR = zip(*(e.debug_particle(m) for m in range(M)))
    refs, sR, ssR = np.stack(refs), np.array(sR, np.float32), np.array(ssR, np.float32)
    ctfparam = hi.CtfParam if ctf is None else ctf[1]
    pri = [likmodel.prior(hi, ctfparam[c]) for c in range(Cn)]
    conv = np.empty((O, Cn) + refs.shape[1:], np.float32)
    lp = np.empty((O, Cn, M, cap.shape[-1] ** 2))
    lp_err = np.empty_like(lp)
    for o in range(O):
        for c in range(Cn):
            conv[o, c], sC, ssC = e.debug_convolved(o, c)
            lp[o, c], lp_err[o, c] = likmodel.logpro(cap[o, c].reshape(M, -1), sR[:, None], ssR[:, None], sC, ssC,
                                                     hi.cfg.Ntotpi, pri[c], with_err=True)
    win, rms = likmodel.corr_windows(conv, refs, N, xs)
    return win, rms, lp, lp_err


def _check(tag, e, hi, ctf, cap, pm, pa, inspect=()):
    """checks 1-4 of the module docstring; returns the measured worst ratios"""
    N, O, Cn, M = hi.N, e.O, e.C, e.M
    generic = not api.lib().bioem_b200_supported_size(N)
    # 1. coverage
    assert not np.isnan(cap).any(), (tag, np.argwhere(np.isnan(cap))[:8])
    # 2. values
    win, rms, lp, lp_err = _model(e, hi, ctf, cap)
    scale = EPS32 * np.log2(N * N) * np.maximum(rms * np.sqrt(N), np.abs(win).max(axis=(-1, -2)))
    ratio = (np.abs(cap - win).max(axis=(-1, -2)) / scale)
    worst = float(ratio.max())
    assert worst <= VALUE_K, (tag, worst, np.unravel_index(np.argmax(ratio), ratio.shape))
    # 3. inspection path: the same bits
    for o, c, m in ((0, 0, 0), (O - 1, Cn - 1, M - 1)) + tuple(inspect):
        np.testing.assert_array_equal(e.debug_correlation(o, c, m), cap[o, c, m], err_msg=f"{tag} {(o, c, m)}")
    # 4. epilogue
    meas = dict(value=worst, total=0.0, angle=0.0, narrow=0.0, share=[])
    maxd, G = hi.cfg.maxDisplaceCenter, hi.cfg.GridSpaceCenter
    for m in range(M):
        g = pm[m]
        assert np.isfinite(g["Total"]) and g["Total"] >= 1.0, (tag, m, g)
        a = 0.5 * (3.0 - hi.cfg.Ntotpi)
        ref = likmodel.fold(lp[:, :, m], kernel=False, lp_err=lp_err[:, :, m])
        ker = likmodel.fold(lp[:, :, m], kernel=True, a=a)
        want, eps = (ref, DOUBLE_RTOL) if generic else (ker, TOTAL_RTOL)
        rtol = eps + want["err"] / want["Total"]
        where = (tag, m, g, {k: want[k] for k in ("Total", "Constoadd", "orient", "conv", "lin")})
        assert g["Constoadd"] == want["Constoadd"], where
        assert (g["orient"], g["conv"]) == (want["orient"], want["conv"]), where
        assert (g["cent_x"], g["cent_y"]) == likmodel.centre(N, maxd, G, want["lin"]), where
        meas["share"].append(float(want["share"].min()))
        rel = abs(g["Total"] / want["Total"] - 1)
        assert rel <= rtol, where + (rel, rtol)
        meas["total"] = max(meas["total"], rel)
        if pa is not None:
            np.testing.assert_array_equal(pa[:, m]["ConstAngle"], want["ConstAngle"], err_msg=tag)
            arel = np.abs(pa[:, m]["forAngles"] / want["forAngles"] - 1)
            atol = eps + want["err_angles"] / want["forAngles"]
            assert np.all(arel <= atol), (tag, m, arel, atol)
            meas["angle"] = max(meas["angle"], float(arel.max()))
        # kernel against reference semantics: each term exp(lp_d) is taken as exp(lp_d + (float(lpmax) - lpmax)) instead
        # of exp(float(lp_d)); both shifts are at most half an ulp of logpro, so |log(ratio)| <= one ulp of max |logpro|
        ulp = float(np.spacing(np.float32(np.abs(lp[:, :, m]).max())))
        d = abs(np.log(ker["Total"] / ref["Total"]))
        assert d <= ulp, (tag, m, d, ulp)
        meas["narrow"] = max(meas["narrow"], d / float(np.spacing(np.float32(abs(want["Constoadd"])))))
    print(f"\n[likelihoods] {tag}: N={N} O={O} C={Cn} M={M} nw={cap.shape[-1]} {'direct-DFT' if generic else 'fused mode %d' % e.cached_product()}"
          f"  value/FFT-bound {meas['value']:.3f}  Total rel {meas['total']:.2e}  angles rel {meas['angle']:.2e}"
          f"  |log(Tref/Tkernel)|/ulp(Constoadd) {meas['narrow']:.3f}  smallest share {min(meas['share']):.1e}")
    return meas


def _case(name, **kw):
    return dict(case=name, **kw)


def _custom(N, maxd, G=1, n_orient=12, grid=None, **kw):
    """a toy32-like case of another edge / window; grid: CTF grid (default CFG1's 3 CTFs)"""
    sigma = N / 6.0
    c = Case(f"n{N}d{maxd}", N, 1.5, 60, 3, 576, n_orient, grid or CASES["toy32"].ctf, maxd, G, model_sigma=sigma,
             model_rmax=2.4 * sigma)
    return dict(case=c, **kw)


BOTH = (0, 1)  # real CTF tables: the complex and the cached-product mode of the fused kernel
# planted-signal cases: every edge class and window shape
PLANTED = {
    "n16": _custom(16, 3, modes=BOTH),
    "n18": _custom(18, 4, modes=BOTH),  # odd second radix
    "toy32": _case("toy32", modes=BOTH),
    "toy36g2": _case("toy36g2", modes=BOTH),  # grid 2, odd window (padding row)
    "toy32d0": _case("toy32d0", modes=BOTH),  # one displacement
    "toy32g2odd": _case("toy32g2odd", modes=BOTH),
    "toy32g3": _case("toy32g3", modes=BOTH),
    "n120d59": _custom(120, 59, n_orient=3, modes=BOTH),  # the middle radix output groups
    "cfg2_slice": _case("cfg2_slice", modes=BOTH),  # N <= 224 class, production window, 32 CTFs
    "cfg4_slice": _case("cfg4_slice", ctf=8, modes=BOTH),  # one CTA per SM
    "toy32psf": _case("toy32psf"),  # complex path only
    "toy33": _case("toy33"),  # direct-DFT path
    "toy35g2": _case("toy35g2"),
    "toy26": _case("toy26"),
}


def _planted_params():
    return [pytest.param(name, mode, id=name if mode is None else f"{name}-mode{mode}")
            for name, spec in PLANTED.items() for mode in spec.get("modes", (None,))]


@pytest.mark.gpu
@pytest.mark.parametrize("name,mode", _planted_params())
def test_every_captured_likelihood_matches_float64_model(monkeypatch, name, mode):
    _need_gpu()
    hi, ctf, e, cap, pm, pa = _capture(monkeypatch, PLANTED[name], mode=mode)
    try:
        _check(name, e, hi, ctf, cap, pm, pa)
    finally:
        e.close()


# CTF grid of the flat cases: DENSE_CTF's 256 CTFs with priors too wide to matter (with DENSE_CTF's own, CTFs far from
# the prior's centre carry e^-10 and less of Total, and a lost likelihood there would go unnoticed)
FLAT_CTF = dict(DENSE_CTF, SIGMA_PRIOR_B_CTF=1e4, SIGMA_PRIOR_DEFOCUS=1e4)

# pure-noise particles (flat posteriors) + one clean particle, WRITE_PROB_ANGLES on and off: the pending-likelihood ring
# of the fused kernel is flushed every 32 likelihoods and, with the angle table, at the end of every orientation --
# C = 1, 4, 5, 32, 33 put those flushes before, at and after the ends of orientations
FLAT = {f"flat32-C{c}-angles{a}": _custom(32, 4, n_orient=5, grid=FLAT_CTF, ctf=c, noise=3, angles=a,
                                          modes=(1,) if c == 1 else (None,))
        for c in (1, 4, 5, 32, 33) for a in (0, 1)}
FLAT["flat16-C5-angles1"] = _custom(16, 3, n_orient=7, grid=FLAT_CTF, ctf=5, noise=3, angles=1, modes=BOTH)
FLAT["flat33-C5-angles1"] = _custom(33, 4, n_orient=7, grid=FLAT_CTF, ctf=5, noise=3, angles=1)


@pytest.mark.gpu
@pytest.mark.parametrize("name,mode", [pytest.param(n, m, id=n if m is None else f"{n}-mode{m}")
                                       for n, s in FLAT.items() for m in s.get("modes", (None,))])
def test_flat_posteriors_every_likelihood_counts(monkeypatch, name, mode):
    _need_gpu()
    hi, ctf, e, cap, pm, pa = _capture(monkeypatch, FLAT[name], mode=mode)
    try:
        meas = _check(name, e, hi, ctf, cap, pm, pa)
        # the noise particles' posteriors are flat: every likelihood carries a part of Total far above the tolerance
        assert min(meas["share"][:-1]) > 1e-3 / (e.O * e.C), (name, meas["share"])
    finally:
        e.close()


@pytest.mark.gpu
def test_scratch_slots_are_reused_across_many_ctas(monkeypatch):
    """cached-product mode: each CTA takes a scratch map for its product projection * conj(particle) and frees it at
    exit.  1024 particles x 8 CTA groups = 8192 CTAs in one launch, far more than can be resident (one slot each)."""
    _need_gpu()
    spec = _custom(32, 4, n_orient=16, grid=FLAT_CTF, ctf=4, noise=1023)
    hi, ctf, e, cap, pm, pa = _capture(monkeypatch, spec, ob=16, og=2, mode=1)
    try:
        _check("slots", e, hi, ctf, cap, pm, pa, inspect=((15, 3, 1023), (7, 2, 511)))
    finally:
        e.close()


GEOMETRY = [(None, None), (1, 1), (5, 2), (7, 3)]  # O = 12: not a multiple of OB = 5 or 7; OB not a multiple of OG


@pytest.mark.gpu
@pytest.mark.parametrize("name,spec,mode", [
    ("flat32-C5", _custom(32, 4, grid=FLAT_CTF, ctf=5, noise=3, angles=1), 0),
    ("flat32-C5", _custom(32, 4, grid=FLAT_CTF, ctf=5, noise=3, angles=1), 1),
    ("toy36g2", _custom(36, 6, G=2, n_orient=12), 1),
    ("flat33-C5", _custom(33, 4, grid=FLAT_CTF, ctf=5, noise=3, angles=1), None),
], ids=["flat32-mode0", "flat32-mode1", "n36g2-mode1", "flat33-direct"])
def test_capture_does_not_depend_on_batch_or_group_geometry(monkeypatch, name, spec, mode):
    """Every likelihood is computed by one CTA on its own: the values cannot depend on which batch (OB orientations
    per launch) or CTA group (OG orientations per CTA) it falls in, nor on the tail groups and launches"""
    _need_gpu()
    first = None
    for ob, og in GEOMETRY:
        hi, ctf, e, cap, pm, pa = _capture(monkeypatch, spec, ob=ob, og=og, mode=mode)
        try:
            last_group = ((ob - 1, e.C // 2, e.M // 2),) if ob else ()
            _check(f"{name} OB={ob} OG={og}", e, hi, ctf, cap, pm, pa, inspect=last_group)
        finally:
            e.close()
        if first is None:
            first = (cap, pm)
        else:
            np.testing.assert_array_equal(cap, first[0])
            for k in ("Constoadd", "orient", "conv", "cent_x", "cent_y"):
                np.testing.assert_array_equal(pm[k], first[1][k])
            np.testing.assert_allclose(pm["Total"], first[1]["Total"], rtol=1e-12)

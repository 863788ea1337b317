"""Float64 model of the likelihood sums, shared by the tests (no GPU needed).

* correlation windows in double from the GPU's own operands (convolved map, particle spectrum), so that the rounding
  of stages 1 and 2 stays out of a comparison of stage 3;
* logpro with the library's arithmetic: firstele in FP32 in the kernel's operation order, including its one
  multiply-add, then a*log(firstele) + B in double;
* the two folds of logpro into a particle's record (bioem_algorithm.h:72-142):
    - reference semantics (the reference, and the library's direct-DFT path): logpro is narrowed to float at every
      displacement before exp;
    - kernel semantics (the fused kernel): only the maximum of each likelihood is narrowed (the record's Constoadd);
      inside a likelihood exp(logpro - its maximum) is summed unnarrowed.
  Both visit (orientation ascending, CTF ascending, displacement in enumeration order); the first maximum wins.
"""
from __future__ import annotations

import numpy as np

MIN_PROB = -999999.0  # initial Constoadd / ConstAngle (reference bioem.cpp:681-699)


def window(N: int, maxd: int, G: int) -> np.ndarray:
    """image rows (= columns) of the displacement window in doRefMapFFT's order (bioem_algorithm.h:156-197)"""
    return np.array(list(range(0, maxd + 1, G)) + list(range(N - maxd, N, G)))


def fma32(a, b, c):
    """float fma: the product of two floats is exact in double, one rounding to double, one to float"""
    return (a.astype(np.float64) * np.float64(b) + c.astype(np.float64)).astype(np.float32)


def prior(hi, ctfparam) -> float:
    """prior term of calc_logpro (bioem_algorithm.h:49-66) with the library's (and the reference's) arithmetic: in
    CTF mode products of floats are float products and the divisions run in double; PSF parameters are mapped to
    their Fourier-space counterparts in double.  hi: anything with the configuration as .cfg."""
    f32 = np.float32
    amp, pha, env = (f32(x) for x in ctfparam[:3])
    c = hi.cfg
    da = amp - f32(c.Priorampcent)
    amp_term = float(da * da) / 2. / float(f32(c.sigmaPrioramp)) / float(f32(c.sigmaPrioramp))
    if c.tousepsf:
        den = float(env * env + pha * pha)  # (a float expression there as well)
        envF = 4. * np.pi * np.pi * float(env) / den
        phaF = 4. * np.pi * np.pi * float(pha) / den
        return (envF * envF / 2. / float(f32(c.sigmaPriorbctf)) / float(f32(c.sigmaPriorbctf))
                - (phaF - float(f32(c.Priordefcent))) ** 2 / 2. / float(f32(c.sigmaPriordefo)) / float(f32(c.sigmaPriordefo))
                - amp_term)
    dp = pha - f32(c.Priordefcent)
    return (float(env * env) / 2. / float(f32(c.sigmaPriorbctf)) / float(f32(c.sigmaPriorbctf))
            - float(dp * dp) / 2. / float(f32(c.sigmaPriordefo)) / float(f32(c.sigmaPriordefo))
            - amp_term)


def firstele(v, sR, ssR, sC, ssC, Nt, fused: bool = True):
    """firstele (bioem_algorithm.h:29-36) of FP32 correlation values v in FP32, in source order, with the one
    multiply-add the library fuses (fused=False: without it, as the oracle, compiled with -ffp-contract=off; the
    reference's own build, -ffast-math, may contract it).  Returns it and the largest magnitude among its terms and
    itself."""
    f32 = np.float32
    v = np.asarray(v, dtype=np.float32)
    sC, ssC, sR, ssR = (np.asarray(x, dtype=np.float32) for x in (sC, ssC, sR, ssR))  # (broadcast against v)
    Nt = f32(Nt)
    t1, t2, t3, t4 = ssR * ssC - v * v, (f32(2.0) * sR * sC) * v, (ssR * sC) * sC, (sR * sR) * ssC
    fe = (fma32(t1, Nt, t2) if fused else Nt * t1 + t2) - t3 - t4
    assert fe.dtype == np.float32
    big = np.maximum(np.maximum(np.abs(Nt * t1), np.abs(t2)), np.maximum(np.maximum(np.abs(t3), np.abs(t4)), np.abs(fe)))
    return fe, big


def logpro(v, sR, ssR, sC, ssC, Nt, pr, fused: bool = True, with_err: bool = False):
    """Unnarrowed (double) logpro of FP32 correlation values v (bioem_algorithm.h:29-67): firstele as above,
    a*log(firstele) + B in double.  with_err: also a bound on how far another double evaluation of the same expression
    may lie (the two large terms cancel: a few ulps of a*log(firstele) and of B, the log's own few ulps times |a|)."""
    f32 = np.float32
    fe = firstele(v, sR, ssR, sC, ssC, Nt, fused)[0]
    sC, ssC, Nt = np.asarray(sC, dtype=np.float32), np.asarray(ssC, dtype=np.float32), f32(Nt)
    fl = ssC * Nt - sC * sC
    a = (3.0 - float(Nt)) * 0.5
    bterm = (float(Nt) * 0.5 - 2.0) * np.log(np.float64(Nt - f32(2.0)) * fl.astype(np.float64)) - np.asarray(pr, np.float64)
    lg = np.log(fe.astype(np.float64))
    if not with_err:
        return a * lg + bterm
    return a * lg + bterm, 4 * (abs(a) * np.spacing(np.abs(lg)) + np.spacing(np.abs(a * lg)) + np.spacing(np.abs(bterm)))


def corr_windows(conv, refs, N: int, xs) -> tuple[np.ndarray, np.ndarray]:
    """lCC / N^2 over the window in double: conv [..., N*(N/2+1), 2] and refs [M, N*(N/2+1), 2] in the reference's
    interleaved layout -> windows [..., M, nw, nw] and the rms of each whole map [..., M].  numpy's c2r keeps only
    the real part of the self-conjugate columns, as the library's inverse transforms do."""
    F = N * (N // 2 + 1)
    cz = np.asarray(conv, np.float64).reshape(-1, F, 2)
    rz = np.asarray(refs, np.float64)
    cz = cz[..., 0] + 1j * cz[..., 1]
    rz = np.conj(rz[..., 0] + 1j * rz[..., 1])
    xs = np.asarray(xs)
    win = np.empty((cz.shape[0], rz.shape[0], len(xs), len(xs)))
    rms = np.empty((cz.shape[0], rz.shape[0]))
    for k in range(cz.shape[0]):
        cc = np.fft.irfft2((cz[k][None, :] * rz).reshape(-1, N, N // 2 + 1), s=(N, N))
        win[k] = cc[:, xs[:, None], xs[None, :]]
        rms[k] = np.sqrt((cc ** 2).mean(axis=(1, 2)))
    lead = np.shape(conv)[:-2]
    return win.reshape(lead + win.shape[1:]), rms.reshape(lead + rms.shape[1:])


def fold(lp, kernel: bool, a: float | None = None, lp_err=None) -> dict:
    """One particle's record from its double logpro lp [O, C, D] (D = window in enumeration order).

    kernel=False: reference semantics; kernel=True: the fused kernel's (see the module docstring).  Returns Total,
    Constoadd, orient, conv, lin (first displacement of the maximum), the angle table forAngles / ConstAngle [O], each
    likelihood's share of Total [O, C] and error bounds of Total / forAngles beyond rounding ("err", "err_angles", absolute):
      kernel=True, a = (3 - N^2)/2 given: the kernel takes exp(a*log1p(t)), t = firstele/min - 1, as
        exp(a*(t - t^2/2 + t^3/3)); the bound is the sum over the terms of term * |a| * |log1p(t) - cubic(t)|;
      kernel=False, lp_err [O, C, D] given (how far another evaluation of lp may lie, in double): a term whose lp lies
        within lp_err of a float rounding boundary may narrow to the neighbouring float; the bound is the sum over
        those terms of term * (exp(ulp) - 1)."""
    lp = np.asarray(lp, dtype=np.float64)
    lpn = lp.astype(np.float32).astype(np.float64)
    lmax = lpn.max(-1)  # [O, C]: each likelihood's maximum narrowed (the same in both semantics)
    err = np.zeros_like(lp)
    if kernel:
        r = lp - lp.max(-1, keepdims=True)
        terms = np.exp(r)
        if a is not None:
            t = np.expm1(r / a)
            err = terms * abs(a) * np.abs(np.log1p(t) - t * (1.0 + t * (-0.5 + t / 3.0)))
    else:
        terms = np.exp(lpn - lmax[..., None])
        if lp_err is not None:
            ulp = np.spacing(np.abs(lpn.astype(np.float32))).astype(np.float64)
            near = 0.5 * ulp - np.abs(lp - lpn) <= lp_err
            err = np.where(near, terms * np.expm1(ulp), 0.0)
    L, E = terms.sum(-1), err.sum(-1)
    Const = float(lmax.max())
    assert Const > MIN_PROB
    o, c = divmod(int(np.argmax(lmax.ravel())), lmax.shape[1])  # argmax: the FIRST maximum
    lin = int(np.argmax(lpn[o, c]))
    Total = float((L * np.exp(lmax - Const)).sum())
    ConstAngle = lmax.max(1)
    forAngles = (L * np.exp(lmax - ConstAngle[:, None])).sum(1)
    return dict(Total=Total, Constoadd=Const, orient=o, conv=c, lin=lin, forAngles=forAngles, ConstAngle=ConstAngle,
                share=L * np.exp(lmax - Const) / Total,  # [O, C]: each likelihood's part of Total
                err=float((E * np.exp(lmax - Const)).sum()), err_angles=(E * np.exp(lmax - ConstAngle[:, None])).sum(1))


def centre(N: int, maxd: int, G: int, lin: int) -> tuple[int, int]:
    """(cent_x, cent_y) the reference reports for window entry lin: minus the displacement"""
    xs = window(N, maxd, G)
    d = [int(x) if x <= maxd else int(x) - N for x in xs[list(divmod(lin, len(xs)))]]
    return -d[0], -d[1]

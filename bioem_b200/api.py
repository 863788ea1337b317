"""ctypes mirror of include/bioem_b200.h — the host-side Python face of the C ABI.

Nothing here computes: every call goes to libbioem_b200.so (hand-written sm_100a
CUDA behind a C ABI).  If the library is missing, or there is no CUDA device,
calls fail loudly — there is no CPU fallback.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import build as _build

_LIB = None

ELECWAVEL_DEFAULT = 0.019866  # reference param.cpp:86


class BioemError(RuntimeError):
    pass


class Config(C.Structure):
    """bioem_b200_config (== fields of the reference's bioem_param_device + projection params)."""
    _fields_ = [("NumberPixels", C.c_int), ("maxDisplaceCenter", C.c_int),
                ("GridSpaceCenter", C.c_int), ("writeAngles", C.c_int), ("tousepsf", C.c_int),
                ("doquater", C.c_int), ("shiftX", C.c_int), ("shiftY", C.c_int),
                ("pixelSize", C.c_float), ("Ntotpi", C.c_float), ("volu", C.c_float),
                ("sigmaPriorbctf", C.c_float), ("sigmaPriordefo", C.c_float),
                ("Priordefcent", C.c_float), ("sigmaPrioramp", C.c_float),
                ("Priorampcent", C.c_float)]


PROB_MAP_DTYPE = np.dtype([("Total", "<f8"), ("Constoadd", "<f8"), ("cent_x", "<i4"),
                           ("cent_y", "<i4"), ("orient", "<i4"), ("conv", "<i4"),
                           ("norm", "<f4"), ("mu", "<f4")])
PROB_ANGLE_DTYPE = np.dtype([("forAngles", "<f8"), ("ConstAngle", "<f8")])
TOP_ANGLE_DTYPE = np.dtype([("orient", "<i4"), ("pad", "<i4"), ("forAngles", "<f8"), ("ConstAngle", "<f8")])
MODEL_POINT_DTYPE = np.dtype([("pos", "<f4", 3), ("quat4", "<f4"), ("radius", "<f4"),
                              ("density", "<f4")])
assert PROB_MAP_DTYPE.itemsize == 40 and PROB_ANGLE_DTYPE.itemsize == 16
assert MODEL_POINT_DTYPE.itemsize == 24

EXPORTS = [
    "bioem_b200_last_error", "bioem_b200_version", "bioem_b200_device_count",
    "bioem_b200_supported_size", "bioem_b200_create", "bioem_b200_destroy",
    "bioem_b200_upload_model", "bioem_b200_upload_orientations", "bioem_b200_upload_ctf",
    "bioem_b200_upload_ctf_real", "bioem_b200_upload_ctf_groups", "bioem_b200_set_particle_groups",
    "bioem_b200_upload_particles", "bioem_b200_upload_particles_mrc",
    "bioem_b200_upload_particles_fft",
    "bioem_b200_reset",
    "bioem_b200_run", "bioem_b200_synchronize", "bioem_b200_download", "bioem_b200_download_top_angles",
    "bioem_b200_partial_bytes", "bioem_b200_export_partial", "bioem_b200_import_partials",
    "bioem_b200_merge_host", "bioem_b200_merge_peers", "bioem_b200_merge_top_angles_peers",
    "bioem_b200_nccl_unique_id", "bioem_b200_nccl_init", "bioem_b200_nccl_attach", "bioem_b200_nccl_comm", "bioem_b200_merge_nccl",
    "bioem_b200_top_angles_nccl", "bioem_b200_set_kernel_timing", "bioem_b200_out_of_frame",
    "bioem_b200_exact_argmax_info", "bioem_b200_cached_product", "bioem_b200_stream", "bioem_b200_device_angles", "bioem_b200_stats",
    "bioem_b200_kernel_time", "bioem_b200_render_maps", "bioem_b200_debug_projection", "bioem_b200_debug_convolved",
    "bioem_b200_debug_correlation", "bioem_b200_debug_run_values", "bioem_b200_debug_particle",
    "bioem_b200_host_defocus_to_phase", "bioem_b200_host_ctf_table", "bioem_b200_host_psf_kernels",
    "bioem_b200_host_volu",
    "bioem_b200_host_model_prepare", "bioem_b200_host_normalise_map",
    "bioem_b200_host_final_logprob",
]


def lib_path() -> str:
    return _build.LIB


def lib():
    """Load libbioem_b200.so (building it with nvcc if the sources are newer)."""
    global _LIB
    if _LIB is not None:
        return _LIB
    path = os.environ.get("BIOEM_B200_LIB")  # an alternative build of the same library (experiments)
    if not path:
        path = _build.LIB
        if not os.path.exists(path) or (os.path.exists(_build.NVCC) and _build.needs_build()):
            path = _build.build()
    if not os.path.exists(path):
        raise BioemError(f"{path} is missing and cannot be built: the CUDA extension is required "
                         "(there is no CPU fallback)")
    L = C.CDLL(path)
    fp = C.POINTER(C.c_float)
    vp = C.c_void_p
    L.bioem_b200_last_error.restype = C.c_char_p
    L.bioem_b200_create.argtypes = [C.POINTER(Config), C.c_int, C.POINTER(vp)]
    L.bioem_b200_destroy.argtypes = [vp]
    L.bioem_b200_upload_model.argtypes = [vp, vp, C.c_int, C.c_float]
    L.bioem_b200_upload_orientations.argtypes = [vp, fp, C.c_int]
    L.bioem_b200_upload_ctf.argtypes = [vp, fp, fp, C.c_int]
    L.bioem_b200_upload_ctf_real.argtypes = [vp, fp, fp, C.c_int]
    L.bioem_b200_upload_ctf_groups.argtypes = [vp, fp, fp, fp, C.c_int, C.c_int]
    L.bioem_b200_set_particle_groups.argtypes = [vp, C.POINTER(C.c_int), C.c_int]
    L.bioem_b200_upload_particles.argtypes = [vp, fp, C.c_int]
    L.bioem_b200_upload_particles_mrc.argtypes = [vp, fp, C.c_int, C.c_int]
    L.bioem_b200_upload_particles_fft.argtypes = [vp, fp, fp, fp, C.c_int]
    L.bioem_b200_reset.argtypes = [vp]
    L.bioem_b200_run.argtypes = [vp, C.c_int, C.c_int]
    L.bioem_b200_synchronize.argtypes = [vp]
    L.bioem_b200_download.argtypes = [vp, vp, vp]
    L.bioem_b200_download_top_angles.argtypes = [vp, C.c_int, C.c_int, C.c_int, vp]
    L.bioem_b200_partial_bytes.argtypes = [vp]
    L.bioem_b200_partial_bytes.restype = C.c_size_t
    L.bioem_b200_export_partial.argtypes = [vp, vp]
    L.bioem_b200_import_partials.argtypes = [vp, vp, C.c_int]
    L.bioem_b200_merge_host.argtypes = [vp, C.c_int, C.c_int, vp]
    L.bioem_b200_merge_peers.argtypes = [C.POINTER(vp), C.c_int]
    L.bioem_b200_merge_top_angles_peers.argtypes = [C.POINTER(vp), C.POINTER(C.c_int), C.POINTER(C.c_int), C.c_int,
                                                    C.c_int, vp]
    L.bioem_b200_nccl_unique_id.argtypes = [vp]
    L.bioem_b200_nccl_init.argtypes = [vp, C.c_int, C.c_int, vp]
    L.bioem_b200_nccl_attach.argtypes = [vp, vp]
    L.bioem_b200_nccl_comm.argtypes = [vp]
    L.bioem_b200_nccl_comm.restype = vp
    L.bioem_b200_merge_nccl.argtypes = [vp]
    L.bioem_b200_top_angles_nccl.argtypes = [vp, C.c_int, C.c_int, C.c_int, vp]
    L.bioem_b200_set_kernel_timing.argtypes = [vp, C.c_int]
    L.bioem_b200_out_of_frame.argtypes = [vp, C.POINTER(C.c_int), C.POINTER(C.c_longlong)]
    L.bioem_b200_exact_argmax_info.argtypes = [vp, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]
    if hasattr(L, "bioem_b200_cached_product"):  # (absent from libraries built before the cached-product mode: A/B runs)
        L.bioem_b200_cached_product.argtypes = [vp]
    L.bioem_b200_stream.argtypes = [vp]
    L.bioem_b200_stream.restype = vp
    L.bioem_b200_device_angles.argtypes = [vp]
    L.bioem_b200_device_angles.restype = vp
    L.bioem_b200_stats.argtypes = [vp, C.POINTER(C.c_longlong), C.POINTER(C.c_longlong)]
    L.bioem_b200_kernel_time.argtypes = [vp, C.POINTER(C.c_double), C.POINTER(C.c_longlong)]
    L.bioem_b200_render_maps.argtypes = [vp, vp, C.c_int, fp]
    L.bioem_b200_debug_projection.argtypes = [vp, C.c_int, fp]
    L.bioem_b200_debug_convolved.argtypes = [vp, C.c_int, C.c_int, fp, fp, fp]
    L.bioem_b200_debug_correlation.argtypes = [vp, C.c_int, C.c_int, C.c_int, fp, C.POINTER(C.c_int)]
    L.bioem_b200_debug_run_values.argtypes = [vp, C.c_int, C.c_int, fp]
    L.bioem_b200_debug_particle.argtypes = [vp, C.c_int, fp, fp, fp]
    L.bioem_b200_host_defocus_to_phase.argtypes = [C.c_float, C.c_float, C.c_float, fp, fp, fp, fp]
    L.bioem_b200_host_defocus_to_phase.restype = None
    L.bioem_b200_host_ctf_table.argtypes = [C.c_int, C.c_float, C.c_int, C.c_float, C.c_float,
                                            C.c_int, C.c_float, C.c_float, C.c_int, C.c_float,
                                            C.c_float, C.c_int, fp, fp, fp]
    L.bioem_b200_host_psf_kernels.argtypes = [C.c_int, C.c_float, C.c_float, C.c_float, C.c_int,
                                              C.c_float, C.c_float, C.c_int, C.c_float, C.c_float,
                                              C.c_int, fp, fp, fp]
    L.bioem_b200_host_volu.argtypes = [C.c_float, C.c_int, C.c_float, C.c_int, C.c_int, C.c_float,
                                       C.c_float, C.c_float, C.c_float, C.c_float]
    L.bioem_b200_host_volu.restype = C.c_float
    L.bioem_b200_host_model_prepare.argtypes = [vp, C.c_int, C.c_int]
    L.bioem_b200_host_model_prepare.restype = C.c_float
    L.bioem_b200_host_normalise_map.argtypes = [fp, C.c_int]
    L.bioem_b200_host_normalise_map.restype = None
    L.bioem_b200_host_final_logprob.argtypes = [C.POINTER(Config), C.c_double, C.c_double]
    L.bioem_b200_host_final_logprob.restype = C.c_double
    _LIB = L
    return L


def _fp(a):
    return a.ctypes.data_as(C.POINTER(C.c_float)) if a is not None else None


def _chk(rc: int, what: str):
    if rc != 0:
        raise BioemError(f"{what} failed ({rc}): {lib().bioem_b200_last_error().decode()}")


class HostInputs:
    """One-off host-side preparation (the reference's readParameters / CalculateRefCTF /
    readModel tail), via the library's host entry points."""

    def __init__(self, n_pixels: int, pixel_size: float, max_disp: int, grid_space: int, ctf: dict,
                 model: np.ndarray, orientations: np.ndarray, write_angles: int = 0,
                 quaternions: bool = True, prior_mod: float = 1.0,
                 elecwavel: float = ELECWAVEL_DEFAULT, center_model: bool = True):
        L = lib()
        f32 = np.float32
        n = int(n_pixels)
        self.N = n
        self.F = n * (n // 2 + 1)
        sig_b = f32(ctf.get("SIGMA_PRIOR_B_CTF", 100.0))   # defaults: reference param.cpp:102-106
        sig_d = C.c_float(ctf.get("SIGMA_PRIOR_DEFOCUS", 2.0))
        cen_d = C.c_float(ctf.get("PRIOR_DEFOCUS_CENTER", 3.0))
        sig_a = f32(ctf.get("SIGMA_PRIOR_AMP_CTF", 0.5))
        cen_a = f32(ctf.get("PRIOR_AMP_CTF_CENTER", 0.0))
        self.use_psf = "PSF_PHASE" in ctf
        self.pixel_size = float(pixel_size)
        self.elecwavel = float(elecwavel)
        grids = np.zeros(3, dtype=np.float32)
        if not self.use_psf:
            d0, d1, nd = ctf["CTF_DEFOCUS"]
            b0, b1, nb = ctf["CTF_B_ENV"]
            a0, a1, na = ctf["CTF_AMPLITUDE"]
            p0, p1 = C.c_float(), C.c_float()
            L.bioem_b200_host_defocus_to_phase(f32(d0), f32(d1), f32(elecwavel), C.byref(p0), C.byref(p1),
                                               C.byref(cen_d), C.byref(sig_d))
            self.C = int(na) * int(nd) * int(nb)
            self.refCTF = np.zeros((self.C, self.F, 2), dtype=np.float32)
            self.CtfParam = np.zeros((self.C, 4), dtype=np.float32)
            c = L.bioem_b200_host_ctf_table(n, f32(pixel_size), 0, f32(a0), f32(a1), int(na), p0, p1, int(nd),
                                            f32(b0), f32(b1), int(nb), _fp(self.refCTF), _fp(self.CtfParam),
                                            _fp(grids))
            self.psf_kernels = None
        else:
            # USE_PSF (reference param.cpp:1466-1535): kernels in real space, transformed on the device
            p0, p1, nd = ctf["PSF_PHASE"]
            b0, b1, nb = ctf["PSF_ENVELOPE"]
            a0, a1, na = ctf["PSF_AMPLITUDE"]
            self.C = int(na) * int(nd) * int(nb)
            self.refCTF = None
            self.psf_kernels = np.zeros((self.C, n, n), dtype=np.float32)
            self.CtfParam = np.zeros((self.C, 4), dtype=np.float32)
            c = L.bioem_b200_host_psf_kernels(n, f32(pixel_size), f32(a0), f32(a1), int(na), f32(p0), f32(p1),
                                              int(nd), f32(b0), f32(b1), int(nb), _fp(self.psf_kernels),
                                              _fp(self.CtfParam), _fp(grids))
        if c != self.C:
            raise BioemError(f"CTF / PSF table: {c} kernels, expected {self.C}")
        self.angles = np.ascontiguousarray(orientations, dtype=np.float32)
        if self.angles.shape[1] == 3:
            self.angles = np.concatenate([self.angles, np.zeros((len(self.angles), 1), np.float32)], 1)
        self.O = self.angles.shape[0]
        voluang = f32(1.0 / float(f32(self.O)) * float(f32(prior_mod)))  # list: reference param.cpp:1131,1324
        volu = L.bioem_b200_host_volu(voluang, int(grid_space), f32(pixel_size), int(max_disp), int(na),
                                      grids[2], grids[1], sig_b, sig_d, sig_a)
        self.cfg = Config(n, int(max_disp), int(grid_space), int(write_angles), int(self.use_psf),
                          int(quaternions), 0, 0,
                          f32(pixel_size), f32(n * n), volu, sig_b, sig_d, cen_d, sig_a, cen_a)
        m = np.asarray(model, dtype=np.float32)
        self.points = np.zeros(m.shape[0], dtype=MODEL_POINT_DTYPE)
        self.points["pos"] = m[:, :3]
        self.points["radius"] = m[:, 3]
        self.points["density"] = m[:, 4]
        self.NormDen = L.bioem_b200_host_model_prepare(self.points.ctypes.data, len(self.points),
                                                       int(center_model))

    def ctf_groups(self, defocus_um, ctf: dict) -> tuple[np.ndarray, np.ndarray, np.ndarray]:
        """Per-micrograph CTF tables for upload_ctf_groups: for every defocus value d [micro-m] of defocus_um, the
        table of ctf's CTF_AMPLITUDE / CTF_B_ENV grids and a CTF_DEFOCUS grid of the same width and count centred on d,
        with the defocus prior centred on d.  Returns (refCTF [G, C, F, 2], CtfParam [G, C, 4], Priordefcent [G] in
        phase units)."""
        if self.use_psf:
            raise BioemError("ctf_groups: USE_PSF kernels are complex; grouped CTF tables must be real")
        L = lib()
        f32 = np.float32
        d0, d1, nd = ctf["CTF_DEFOCUS"]
        b0, b1, nb = ctf["CTF_B_ENV"]
        a0, a1, na = ctf["CTF_AMPLITUDE"]
        half = f32(0.5) * (f32(d1) - f32(d0))
        vals = np.asarray(defocus_um, dtype=np.float32).reshape(-1)
        G = len(vals)
        ref = np.zeros((G, self.C, self.F, 2), dtype=np.float32)
        par = np.zeros((G, self.C, 4), dtype=np.float32)
        cen = np.zeros(G, dtype=np.float32)
        grids = np.zeros(3, dtype=np.float32)
        for g, d in enumerate(vals):
            p0, p1, pc = C.c_float(), C.c_float(), C.c_float(d)
            L.bioem_b200_host_defocus_to_phase(f32(d - half), f32(d + half), f32(self.elecwavel), C.byref(p0),
                                               C.byref(p1), C.byref(pc), None)
            c = L.bioem_b200_host_ctf_table(self.N, f32(self.pixel_size), 0, f32(a0), f32(a1), int(na), p0, p1,
                                            int(nd), f32(b0), f32(b1), int(nb), _fp(ref[g]), _fp(par[g]), _fp(grids))
            if c != self.C:
                raise BioemError(f"ctf_groups: group {g}: {c} kernels, expected {self.C}")
            cen[g] = pc.value
        return ref, par, cen

    @staticmethod
    def normalise_particles(imgs: np.ndarray) -> np.ndarray:
        """What the reference's MRC reader does to every image (map.cpp:830-845)."""
        L = lib()
        out = np.ascontiguousarray(imgs, dtype=np.float32).copy()
        for k in range(out.shape[0]):
            L.bioem_b200_host_normalise_map(_fp(out[k]), out.shape[1])
        return out

    def final_logprob(self, total: float, const: float) -> float:
        return lib().bioem_b200_host_final_logprob(C.byref(self.cfg), float(total), float(const))


class Engine:
    """One handle = one GPU (bioem_b200_create .. destroy)."""

    def __init__(self, cfg: Config, device: int = 0):
        self._h = C.c_void_p()
        self.cfg = cfg
        self.O = self.C = self.M = 0
        _chk(lib().bioem_b200_create(C.byref(cfg), int(device), C.byref(self._h)), "bioem_b200_create")

    def close(self):
        if self._h:
            lib().bioem_b200_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- uploads
    def upload_model(self, points: np.ndarray, norm_den: float):
        assert points.dtype == MODEL_POINT_DTYPE
        _chk(lib().bioem_b200_upload_model(self._h, points.ctypes.data, len(points), np.float32(norm_den)),
             "upload_model")

    def upload_orientations(self, angles4: np.ndarray):
        a = np.ascontiguousarray(angles4, dtype=np.float32)
        assert a.ndim == 2 and a.shape[1] == 4
        self._keep_angles = a
        self.O = a.shape[0]
        _chk(lib().bioem_b200_upload_orientations(self._h, _fp(a), self.O), "upload_orientations")

    def upload_ctf(self, refCTF: np.ndarray, ctf_param4: np.ndarray):
        self.C = refCTF.shape[0]
        r = np.ascontiguousarray(refCTF, dtype=np.float32)
        p = np.ascontiguousarray(ctf_param4, dtype=np.float32)
        assert p.shape == (self.C, 4)
        _chk(lib().bioem_b200_upload_ctf(self._h, _fp(r), _fp(p), self.C), "upload_ctf")

    def upload_ctf_real(self, kernels: np.ndarray, ctf_param4: np.ndarray):
        self.C = kernels.shape[0]
        k = np.ascontiguousarray(kernels, dtype=np.float32)
        p = np.ascontiguousarray(ctf_param4, dtype=np.float32)
        assert p.shape == (self.C, 4)
        _chk(lib().bioem_b200_upload_ctf_real(self._h, _fp(k), _fp(p), self.C), "upload_ctf_real")

    def upload_ctf_groups(self, refCTF: np.ndarray, ctf_param4: np.ndarray, prior_defocus_center=None):
        """refCTF [G, C, F, 2] / ctf_param4 [G, C, 4]: G real CTF tables of C rows; prior_defocus_center [G] in phase
        units (None: the config's centre).  Particle m integrates over its group's rows (set_particle_groups); records
        name rows of the whole table, g*C + c.  run_capture then returns [O, C, M, nw, nw]."""
        r = np.ascontiguousarray(refCTF, dtype=np.float32)
        p = np.ascontiguousarray(ctf_param4, dtype=np.float32)
        G, Cg = int(r.shape[0]), int(r.shape[1])
        assert p.shape == (G, Cg, 4)
        cen = None if prior_defocus_center is None else np.ascontiguousarray(prior_defocus_center, dtype=np.float32)
        assert cen is None or cen.shape == (G,)
        _chk(lib().bioem_b200_upload_ctf_groups(self._h, _fp(r), _fp(p), _fp(cen), G, Cg), "upload_ctf_groups")
        self.C = Cg

    def set_particle_groups(self, group: np.ndarray):
        """group[M]: every particle's CTF group, in [0, G)."""
        g = np.ascontiguousarray(group, dtype=np.int32)
        _chk(lib().bioem_b200_set_particle_groups(self._h, g.ctypes.data_as(C.POINTER(C.c_int)), len(g)),
             "set_particle_groups")

    def upload_particles(self, maps: np.ndarray):
        m = np.ascontiguousarray(maps, dtype=np.float32)
        self.M = m.shape[0]
        _chk(lib().bioem_b200_upload_particles(self._h, _fp(m), self.M), "upload_particles")

    def upload_particles_mrc(self, raw: np.ndarray, normalise: bool = True):
        """raw: [M, nr, nc] images in MRC file order (before the reader's transposition)."""
        r = np.ascontiguousarray(raw, dtype=np.float32)
        self.M = r.shape[0]
        _chk(lib().bioem_b200_upload_particles_mrc(self._h, _fp(r), self.M, int(normalise)),
             "upload_particles_mrc")

    def upload_particles_fft(self, fft: np.ndarray, s: np.ndarray, ss: np.ndarray):
        f = np.ascontiguousarray(fft, dtype=np.float32)
        self.M = f.shape[0]
        _chk(lib().bioem_b200_upload_particles_fft(self._h, _fp(f), _fp(np.ascontiguousarray(s, np.float32)),
                                                   _fp(np.ascontiguousarray(ss, np.float32)), self.M),
             "upload_particles_fft")

    def upload_all(self, hi: HostInputs, particles: np.ndarray):
        self.upload_model(hi.points, hi.NormDen)
        self.upload_orientations(hi.angles)
        if hi.use_psf:
            self.upload_ctf_real(hi.psf_kernels, hi.CtfParam)
        else:
            self.upload_ctf(hi.refCTF, hi.CtfParam)
        self.upload_particles(particles)

    # ---- run
    def reset(self):
        _chk(lib().bioem_b200_reset(self._h), "reset")

    def run(self, o_begin: int = 0, o_end: int | None = None):
        _chk(lib().bioem_b200_run(self._h, int(o_begin), int(self.O if o_end is None else o_end)), "run")

    def synchronize(self):
        _chk(lib().bioem_b200_synchronize(self._h), "synchronize")

    def download(self, out_maps: np.ndarray | None = None, out_angles=None):
        """(maps[M], angle table [O, M] or None).  out_angles=False skips the O x M x 16-byte angle table
        (WRITE_PROB_ANGLES runs that only need the top-K rows, download_top_angles)."""
        pm = out_maps if out_maps is not None else np.zeros(self.M, dtype=PROB_MAP_DTYPE)
        pa = None if out_angles is False else out_angles
        if pa is None and out_angles is not False and self.cfg.writeAngles:
            pa = np.zeros((self.O, self.M), dtype=PROB_ANGLE_DTYPE)
        _chk(lib().bioem_b200_download(self._h, pm.ctypes.data, pa.ctypes.data if pa is not None else None),
             "download")
        return pm, pa

    def download_top_angles(self, k: int, o_begin: int = 0, o_end: int | None = None) -> np.ndarray:
        """[M, k] rows (orient, forAngles, ConstAngle): the k most probable orientations of every
        particle among [o_begin, o_end), most probable first (reference bioem.cpp:1254-1290)."""
        out = np.zeros((self.M, k), dtype=TOP_ANGLE_DTYPE)
        _chk(lib().bioem_b200_download_top_angles(self._h, int(o_begin), int(self.O if o_end is None else o_end),
                                                  int(k), out.ctypes.data), "download_top_angles")
        return out

    # ---- multi-GPU plumbing
    def partial_bytes(self) -> int:
        return int(lib().bioem_b200_partial_bytes(self._h))

    def export_partial(self, device_ptr: int):
        _chk(lib().bioem_b200_export_partial(self._h, C.c_void_p(device_ptr)), "export_partial")

    def import_partials(self, device_ptr: int, n_ranks: int):
        _chk(lib().bioem_b200_import_partials(self._h, C.c_void_p(device_ptr), int(n_ranks)), "import_partials")

    def nccl_init(self, n_ranks: int, rank: int, unique_id: bytes):
        """Build this handle's NCCL communicator from the 128-byte id rank 0 made with nccl_unique_id()
        (the launcher broadcasts it: plumbing)."""
        buf = C.create_string_buffer(bytes(unique_id), 128)
        _chk(lib().bioem_b200_nccl_init(self._h, int(n_ranks), int(rank), buf), "nccl_init")

    def nccl_comm(self) -> int:
        return int(lib().bioem_b200_nccl_comm(self._h) or 0)

    def nccl_attach(self, comm: int):
        """Use an existing ncclComm_t (e.g. another Engine's nccl_comm() on the same device); not owned."""
        _chk(lib().bioem_b200_nccl_attach(self._h, C.c_void_p(comm)), "nccl_attach")

    def merge_nccl(self):
        """One NCCL all-gather of the per-image partials + the fold in rank order, on the handle's stream."""
        _chk(lib().bioem_b200_merge_nccl(self._h), "merge_nccl")

    def top_angles_nccl(self, k: int, o_begin: int, o_end: int) -> np.ndarray:
        out = np.zeros((self.M, k), dtype=TOP_ANGLE_DTYPE)
        _chk(lib().bioem_b200_top_angles_nccl(self._h, int(o_begin), int(o_end), int(k), out.ctypes.data),
             "top_angles_nccl")
        return out

    def device_angles(self) -> int:
        return int(lib().bioem_b200_device_angles(self._h) or 0)

    # ---- stats
    def stats(self):
        a, b = C.c_longlong(), C.c_longlong()
        _chk(lib().bioem_b200_stats(self._h, C.byref(a), C.byref(b)), "stats")
        return a.value, b.value

    def set_kernel_timing(self, on: bool = True):
        _chk(lib().bioem_b200_set_kernel_timing(self._h, int(on)), "set_kernel_timing")

    def out_of_frame(self):
        """(per-orientation counts [O], total) of model points skipped because they left the frame."""
        per = np.zeros(self.O, dtype=np.int32)
        tot = C.c_longlong()
        _chk(lib().bioem_b200_out_of_frame(self._h, per.ctypes.data_as(C.POINTER(C.c_int)), C.byref(tot)),
             "out_of_frame")
        return per, tot.value

    def cached_product(self) -> int:
        """1: the fused kernel runs in cached-product mode (real CTF kernels), 0: complex conv spectra, -1: undecided."""
        return int(lib().bioem_b200_cached_product(self._h))

    def exact_argmax_info(self):
        """(re-evaluated, corrected, disagreed) of the exact arg-max pass of the last download()."""
        a, b, c = C.c_int(), C.c_int(), C.c_int()
        _chk(lib().bioem_b200_exact_argmax_info(self._h, C.byref(a), C.byref(b), C.byref(c)), "exact_argmax_info")
        return a.value, b.value, c.value

    def kernel_time(self):
        t, n = C.c_double(), C.c_longlong()
        _chk(lib().bioem_b200_kernel_time(self._h, C.byref(t), C.byref(n)), "kernel_time")
        return t.value, n.value

    # ---- calculated images
    def render_maps(self, records: np.ndarray) -> np.ndarray:
        """float32 [n, N, N]: the calculated image each record names (its orientation, CTF, displacement, norm and
        mu), in the layout of the particles given to upload_particles; records is a PROB_MAP_DTYPE array, e.g. the
        first result of download(), whose maps are then every particle's best fit."""
        r = np.ascontiguousarray(records)
        if r.dtype != PROB_MAP_DTYPE:
            raise TypeError(f"render_maps: records must be of PROB_MAP_DTYPE, not {r.dtype}")
        r = r.reshape(-1)
        n = self.cfg.NumberPixels
        out = np.zeros((len(r), n, n), dtype=np.float32)
        _chk(lib().bioem_b200_render_maps(self._h, r.ctypes.data, len(r), _fp(out)), "render_maps")
        return out

    # ---- inspection
    def debug_projection(self, o: int) -> np.ndarray:
        n = self.cfg.NumberPixels
        out = np.zeros((n, n), dtype=np.float32)
        _chk(lib().bioem_b200_debug_projection(self._h, int(o), _fp(out)), "debug_projection")
        return out

    def debug_convolved(self, o: int, c: int):
        n = self.cfg.NumberPixels
        out = np.zeros((n * (n // 2 + 1), 2), dtype=np.float32)
        s, ss = C.c_float(), C.c_float()
        _chk(lib().bioem_b200_debug_convolved(self._h, int(o), int(c), _fp(out), C.byref(s), C.byref(ss)),
             "debug_convolved")
        return out, s.value, ss.value

    def _window_edge(self) -> int:
        d, g = self.cfg.maxDisplaceCenter, self.cfg.GridSpaceCenter
        return d // g + 1 + (d + g - 1) // g  # Algo 1's window (bioem_algorithm.h:156-197), quirk Q3

    def debug_correlation(self, o: int, c: int, m: int) -> np.ndarray:
        nw = self._window_edge()
        out = np.zeros(nw * nw, dtype=np.float32)
        nv = C.c_int()
        _chk(lib().bioem_b200_debug_correlation(self._h, int(o), int(c), int(m), _fp(out), C.byref(nv)),
             "debug_correlation")
        return out.reshape(nw, nw)

    def run_capture(self, o_begin: int = 0, o_end: int | None = None) -> np.ndarray:
        """run(o_begin, o_end), returning every correlation window it computed: [o_end - o_begin, C, M, nw, nw]
        (each window as debug_correlation returns it)."""
        o_end = self.O if o_end is None else o_end
        nw = self._window_edge()
        out = np.zeros((max(0, o_end - o_begin), self.C, self.M, nw, nw), dtype=np.float32)
        _chk(lib().bioem_b200_debug_run_values(self._h, int(o_begin), int(o_end), _fp(out)), "debug_run_values")
        return out

    def debug_particle(self, m: int):
        n = self.cfg.NumberPixels
        out = np.zeros((n * (n // 2 + 1), 2), dtype=np.float32)
        s, ss = C.c_float(), C.c_float()
        _chk(lib().bioem_b200_debug_particle(self._h, int(m), _fp(out), C.byref(s), C.byref(ss)), "debug_particle")
        return out, s.value, ss.value


def merge_host(parts: np.ndarray) -> np.ndarray:
    """parts: [nRanks, M] of PROB_MAP_DTYPE -> merged [M] (lowest rank wins ties)."""
    p = np.ascontiguousarray(parts)
    out = np.zeros(p.shape[1], dtype=PROB_MAP_DTYPE)
    _chk(lib().bioem_b200_merge_host(p.ctypes.data, p.shape[0], p.shape[1], out.ctypes.data), "merge_host")
    return out


def nccl_unique_id() -> bytes:
    buf = C.create_string_buffer(128)
    _chk(lib().bioem_b200_nccl_unique_id(buf), "nccl_unique_id")
    return buf.raw


def merge_peers(engines) -> None:
    """Single process, one Engine per GPU (or several on one GPU): merged state lands in engines[0]."""
    arr = (C.c_void_p * len(engines))(*[e._h for e in engines])
    _chk(lib().bioem_b200_merge_peers(arr, len(engines)), "merge_peers")


def merge_top_angles_peers(engines, blocks, k: int) -> np.ndarray:
    arr = (C.c_void_p * len(engines))(*[e._h for e in engines])
    ob = (C.c_int * len(engines))(*[int(b[0]) for b in blocks])
    oe = (C.c_int * len(engines))(*[int(b[1]) for b in blocks])
    out = np.zeros((engines[0].M, k), dtype=TOP_ANGLE_DTYPE)
    _chk(lib().bioem_b200_merge_top_angles_peers(arr, ob, oe, len(engines), int(k), out.ctypes.data),
         "merge_top_angles_peers")
    return out


def inputs_for_case(cd) -> tuple[HostInputs, np.ndarray]:
    """HostInputs + particle array (as the reference's reader would hold it) for a cases.CaseData."""
    c = cd.case
    hi = HostInputs(c.n_pixels, c.pixel_size, c.max_disp, c.grid_space, c.ctf, cd.model, cd.quats,
                    write_angles=c.write_angles)
    parts = cd.particles
    if c.particle_format == "mrc":
        parts = HostInputs.normalise_particles(parts)
    return hi, np.ascontiguousarray(parts, dtype=np.float32)

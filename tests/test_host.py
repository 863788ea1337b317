"""CPU-only: the C-ABI library loads, exports every symbol include/bioem_b200.h declares, and
its host-side input preparation agrees bit for bit with the oracle's restatement of the
reference (no device compute is called here)."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from bioem_b200 import api
from bioem_b200.cases import CASES, build_case
from oracle import pyoracle

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))


def test_library_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "bioem_b200.h")).read()
    declared = set(re.findall(r"\b(bioem_b200_[a-z0-9_]+)\s*\(", hdr))
    declared -= {"bioem_b200_context"}
    L = api.lib()
    missing = [s for s in sorted(declared) if not hasattr(L, s)]
    assert not missing, missing
    assert declared == set(api.EXPORTS), declared ^ set(api.EXPORTS)
    assert L.bioem_b200_version() >= 100


def test_supported_sizes():
    L = api.lib()
    for n in (32, 36, 64, 100, 128, 200, 224, 240, 300, 360, 448, 512):
        assert L.bioem_b200_supported_size(n) == 1
    for n in (16, 18, 250, 486, 504):  # rule-generated splits
        assert L.bioem_b200_supported_size(n) == 1
    # no fused FFT kernel (odd, a prime factor above 7, no valid two-pass split, too large): these edges are accepted and
    # run on the direct-DFT path
    for n in (31, 102, 225, 490, 1024):
        assert L.bioem_b200_supported_size(n) == 0


def test_create_fails_loudly_without_device_or_with_bad_config():
    L = api.lib()
    cfg = api.Config(1, 0, 1, 0, 0, 1, 0, 0, 1.0, 1.0, 1.0, 1, 1, 1, 1, 0)
    h = C.c_void_p()
    assert L.bioem_b200_create(C.byref(cfg), 0, C.byref(h)) == 1  # no image
    assert b"NUMBER_PIXELS" in L.bioem_b200_last_error()
    # (an edge without a fused FFT kernel -- 102 = 2*3*17, 225 odd -- is NOT refused: it runs on the direct-DFT path)
    cfg = api.Config(64, 5, 0, 0, 0, 1, 0, 0, 1.0, 4096, 1.0, 1, 1, 1, 1, 0)
    assert L.bioem_b200_create(C.byref(cfg), 0, C.byref(h)) == 1  # grid spacing 0 (the reference divides by it)
    assert b"DISPLACE_CENTER" in L.bioem_b200_last_error()
    cfg = api.Config(64, 40, 1, 0, 0, 1, 0, 0, 1.0, 4096, 1.0, 1, 1, 1, 1, 0)
    assert L.bioem_b200_create(C.byref(cfg), 0, C.byref(h)) == 1  # window wider than the image
    # (a spacing that does not divide the maximum displacement is accepted: quirk Q3, Algo 1's window)
    if L.bioem_b200_device_count() == 0:
        cfg = api.Config(64, 4, 1, 0, 0, 1, 0, 0, 1.0, 4096, 1.0, 1, 1, 1, 1, 0)
        rc = L.bioem_b200_create(C.byref(cfg), 0, C.byref(h))
        assert rc == 2 and b"no CPU fallback" in L.bioem_b200_last_error()


@pytest.mark.parametrize("name", ["toy32", "toy36g2", "toy64", "cfg1", "cfg2_slice"])
def test_host_preparation_matches_oracle(name):
    cd = build_case(name)
    hi, parts = api.inputs_for_case(cd)
    P = pyoracle.Prepared(cd.case, cd.model, cd.quats, cd.particles)
    for f, _ in api.Config._fields_:
        a, b = getattr(hi.cfg, f), getattr(P.cfg, f)
        assert a == b, (f, a, b)
    assert hi.C == P.C and hi.O == P.O
    np.testing.assert_array_equal(hi.CtfParam[:, :3], P.CtfParam)
    np.testing.assert_array_equal(hi.refCTF, P.refCTF)
    assert hi.NormDen == P.NormDen
    np.testing.assert_array_equal(hi.points["pos"], P.pts[:, :3])
    np.testing.assert_array_equal(parts, P.maps)


def test_ctf_mirror_row_quirk_q1():
    """rows r <= N/2-2 use |k|=r, rows N/2-1 and N/2 use N/2, rows r > N/2 use N-1-r."""
    n = 16
    ref = np.zeros((1, n * (n // 2 + 1), 2), np.float32)
    par = np.zeros((1, 4), np.float32)
    g = np.zeros(3, np.float32)
    api.lib().bioem_b200_host_ctf_table(n, 1.5, 0, 0.1, 0.1, 1, 2.0, 2.0, 1, 50.0, 50.0, 1, api._fp(ref),
                                        api._fp(par), api._fp(g))
    t = ref[0, :, 0].reshape(n, n // 2 + 1)
    assert np.array_equal(t[n // 2 - 1], t[n // 2])
    for r in range(n // 2 + 1, n):
        assert np.array_equal(t[r], t[n - 1 - r])
    assert (ref[..., 1] == 0).all() and t[0, 0] == 1.0


def test_final_logprob_and_merge_host():
    cd = build_case("toy32")
    hi, _ = api.inputs_for_case(cd)
    P = pyoracle.Prepared(cd.case, cd.model, cd.quats, cd.particles)
    assert hi.final_logprob(3.5, -1234.5) == P.final_logprob(3.5, -1234.5)
    # split an oracle run into two orientation blocks and merge: equals the single run
    full = P.run()["prob"]
    a = P.run(0, 11)["prob"]
    b = P.run(11, P.O)["prob"]
    merged = api.merge_host(np.stack([a, b]))
    np.testing.assert_allclose(merged["Total"], full["Total"], rtol=1e-12)
    for k in ("Constoadd", "cent_x", "cent_y", "orient", "conv", "norm", "mu"):
        np.testing.assert_array_equal(merged[k], full[k])


# ---------------------------------------------------------------------------------------------
# bioEM_b200: the reference's command line / file formats on top of the C ABI (SURVEY §8 f1-f3).
# Without a GPU only the front end can run: BIOEM_B200_DUMP_INPUTS makes the binary write what it
# would upload and stop before any device work.
HOST_BIN = os.path.join(ROOT, "bioem_b200", "bin", "bioEM_b200")


def _build_host_bin():
    import subprocess
    api.lib()
    subprocess.check_call(["make", "-C", os.path.join(ROOT, "bioem_b200", "csrc", "host")],
                          stdout=subprocess.DEVNULL)
    return HOST_BIN


@pytest.mark.parametrize("name", ["toy32", "toy36g2", "toy64"])
def test_host_binary_reads_the_reference_formats(name, tmp_path):
    """Parameter file, fixed-width orientation list, text model, text / MRC particle stacks: the
    C++ front end must hand the library exactly the arrays the Python mirror builds (bit for bit;
    the mirror itself is pinned to the oracle in test_host_preparation_matches_oracle)."""
    import subprocess
    from bioem_b200.cases import reference_cli
    exe = _build_host_bin()
    cd = build_case(name, str(tmp_path))
    dump = tmp_path / "dump"
    dump.mkdir()
    r = subprocess.run([exe] + reference_cli(cd), cwd=tmp_path, capture_output=True, text=True,
                       env={**os.environ, "BIOEM_B200_DUMP_INPUTS": str(dump)})
    assert r.returncode == 0, r.stdout[-500:] + r.stderr[-500:]
    hi, parts = api.inputs_for_case(cd)
    pts = np.fromfile(dump / "points.bin", dtype=api.MODEL_POINT_DTYPE)
    assert pts.tobytes() == hi.points.tobytes()
    assert np.array_equal(np.fromfile(dump / "maps.bin", dtype=np.float32).reshape(parts.shape), parts)
    assert np.array_equal(np.fromfile(dump / "angles.bin", dtype=np.float32).reshape(-1, 4), hi.angles)
    assert np.array_equal(np.fromfile(dump / "ctfparam.bin", dtype=np.float32).reshape(-1, 4), hi.CtfParam)
    assert np.array_equal(np.fromfile(dump / "refctf.bin", dtype=np.float32).reshape(hi.refCTF.shape), hi.refCTF)
    meta = dict(ln.split() for ln in open(dump / "meta.txt"))
    assert np.float32(meta["volu"]) == np.float32(hi.cfg.volu)
    assert np.float32(meta["NormDen"]) == np.float32(hi.NormDen)
    assert int(meta["O"]) == hi.O and int(meta["C"]) == hi.C and int(meta["M"]) == parts.shape[0]


def test_host_binary_orientation_grids_and_errors(tmp_path):
    """Euler / quaternion grid generators (reference param.cpp:1009-1048,1141-1210) and the
    reference's fatal input errors (exit code 1)."""
    import subprocess
    from bioem_b200 import synth
    exe = _build_host_bin()
    cd = build_case("toy32", str(tmp_path))
    base = ["--Modelfile", cd.paths["model"], "--Particlesfile", cd.paths["particles"]]

    def run(param_text, extra=()):
        pf = tmp_path / "p.txt"
        pf.write_text(param_text)
        dump = tmp_path / "d"
        dump.mkdir(exist_ok=True)
        return subprocess.run([exe] + base + ["--Inputfile", str(pf)] + list(extra), cwd=tmp_path,
                              capture_output=True, text=True,
                              env={**os.environ, "BIOEM_B200_DUMP_INPUTS": str(dump)}), dump

    common = ("PIXEL_SIZE 1.5\nNUMBER_PIXELS 32\nDISPLACE_CENTER 4 1\nCTF_DEFOCUS 1.0 4.0 3\n"
              "CTF_B_ENV 2.0 300.0 1\nCTF_AMPLITUDE 0.1 0.1 1\n")
    # Euler grid: nAlpha * nBeta * nAlpha orientations, cell centres
    r, dump = run(common + "GRIDPOINTS_ALPHA 4\nGRIDPOINTS_BETA 3\n")
    assert r.returncode == 0, r.stderr
    ang = np.fromfile(dump / "angles.bin", dtype=np.float32).reshape(-1, 4)
    assert ang.shape[0] == 4 * 3 * 4
    ga = np.float32(2 * np.pi / 4)
    assert abs(ang[0, 0] - (-np.pi + ga / 2)) < 1e-6 and abs(ang[0, 1] - np.arccos(-1 + 1 / 3)) < 1e-6
    assert np.all(ang[:, 3] == 0)
    # quaternion grid: both signs of q4, unit norm
    r, dump = run(common + "USE_QUATERNIONS\nGRIDPOINTS_QUATERNION 3\n")
    assert r.returncode == 0, r.stderr
    q = np.fromfile(dump / "angles.bin", dtype=np.float32).reshape(-1, 4)
    assert q.shape[0] % 2 == 0 and q.shape[0] > 0
    np.testing.assert_allclose((q.astype(np.float64) ** 2).sum(1), 1.0, atol=1e-6)
    assert np.array_equal(q[0::2, :3], q[1::2, :3]) and np.array_equal(q[0::2, 3], -q[1::2, 3])
    # fatal errors of the reference
    r, _ = run(common.replace("PIXEL_SIZE 1.5\n", "") + "GRIDPOINTS_ALPHA 4\nGRIDPOINTS_BETA 3\n")
    assert r.returncode == 1 and "PIXEL_SIZE" in r.stderr
    r, _ = run(common)
    assert r.returncode == 1 and "GRIDPOINTS_ALPHA" in r.stderr
    r, _ = run(common.replace("CTF_DEFOCUS 1.0 4.0 3", "CTF_DEFOCUS 1.0 9.0 3") + "GRIDPOINTS_ALPHA 4\nGRIDPOINTS_BETA 3\n")
    assert r.returncode == 1 and "8micro-m" in r.stderr
    r = subprocess.run([exe, "--Modelfile", "x"], capture_output=True, text=True)
    assert r.returncode == 1
    r = subprocess.run([exe] + base + ["--Inputfile", "p.txt", "--ReadMultipleMRC"], cwd=tmp_path,
                       capture_output=True, text=True)
    assert r.returncode == 1 and "--ReadMRC" in r.stderr
    # PDB reader: CA atoms only, residue tables
    pdb = tmp_path / "m.pdb"
    pdb.write_text("ATOM      1  N   GLY A   1      11.104  13.207   2.100  1.00  0.00\n"
                   "ATOM      2  CA  GLY A   1      12.000  14.000   3.000  1.00  0.00\n"
                   "ATOM      3  CA  TRP A   2      -2.000   4.000  -6.000  1.00  0.00\n"
                   "HETATM    4  CA  XXX A   3       0.000   0.000   0.000  1.00  0.00\n")
    pf = tmp_path / "p.txt"
    pf.write_text(common + "GRIDPOINTS_ALPHA 4\nGRIDPOINTS_BETA 3\nNO_CENTEROFMASS\n")
    dump = tmp_path / "d"
    r = subprocess.run([exe, "--Modelfile", str(pdb), "--ReadPDB", "--Particlesfile", cd.paths["particles"],
                        "--Inputfile", str(pf)], cwd=tmp_path, capture_output=True, text=True,
                       env={**os.environ, "BIOEM_B200_DUMP_INPUTS": str(dump)})
    assert r.returncode == 0, r.stderr
    pts = np.fromfile(dump / "points.bin", dtype=api.MODEL_POINT_DTYPE)
    assert len(pts) == 2
    assert np.allclose(pts["pos"], [[12, 14, 3], [-2, 4, -6]])
    assert np.allclose(pts["radius"], [2.25, 3.4]) and np.allclose(pts["density"], [40, 108])


REF_BIN = os.path.join(ROOT, "oracle", "_ref", "bioEM_ref")


@pytest.mark.parametrize("name", ["toy32", "toy36g2"])
def test_dump_caches_are_interchangeable_with_the_reference(name, tmp_path):
    """--DumpModel / --DumpMaps / --LoadModelDump / --LoadMapDump (reference model.cpp:41-82,676-707,
    map.cpp:44-78): the binary caches have the reference's layout and meaning -- the model as read (before
    the centring, which is redone after loading), the particles as the reader leaves them -- so a cache
    written by the unmodified reference loads into bioEM_b200 and gives the arrays a direct read gives.
    Without the reference binary, the caches bioEM_b200 writes are the ones loaded back."""
    import subprocess
    from bioem_b200.cases import reference_cli
    exe = _build_host_bin()
    cd = build_case(name, str(tmp_path))
    cli = reference_cli(cd)
    ref_dir, our_dir, direct, loaded = (tmp_path / d for d in ("ref", "ours", "direct", "loaded"))
    for d in (ref_dir, our_dir, direct, loaded):
        d.mkdir()
    r = subprocess.run([exe] + cli + ["--DumpModel", "--DumpMaps", "--PrintCOORDREAD"], cwd=our_dir, capture_output=True, text=True,
                       env={**os.environ, "BIOEM_B200_DUMP_INPUTS": str(direct)})
    assert r.returncode == 0, r.stdout[-400:] + r.stderr[-400:]
    if os.path.exists(REF_BIN):
        r = subprocess.run([REF_BIN] + cli + ["--DumpModel", "--DumpMaps", "--PrintCOORDREAD"], cwd=ref_dir,
                           capture_output=True, text=True)
        assert r.returncode == 0, r.stdout[-400:] + r.stderr[-400:]
        _compare_caches_with_the_reference(cd, ref_dir, our_dir)
    else:
        ref_dir = our_dir
    # load the caches (the REFERENCE's when it is built): same arrays as the direct read (model centred after loading)
    r = subprocess.run([exe] + cli + ["--LoadModelDump", "--LoadMapDump"], cwd=ref_dir, capture_output=True, text=True,
                       env={**os.environ, "BIOEM_B200_DUMP_INPUTS": str(loaded)})
    assert r.returncode == 0, r.stdout[-400:] + r.stderr[-400:]
    p_direct = np.fromfile(direct / "points.bin", dtype=api.MODEL_POINT_DTYPE)
    p_loaded = np.fromfile(loaded / "points.bin", dtype=api.MODEL_POINT_DTYPE)
    np.testing.assert_allclose(p_loaded["pos"], p_direct["pos"], rtol=0, atol=2e-6)
    assert np.array_equal(p_loaded["radius"], p_direct["radius"]) and np.array_equal(p_loaded["density"], p_direct["density"])
    m_direct = np.fromfile(direct / "maps.bin", dtype=np.float32)
    m_loaded = np.fromfile(loaded / "maps.bin", dtype=np.float32)
    np.testing.assert_allclose(m_loaded, m_direct, rtol=0, atol=2.5e-7 * np.abs(m_direct).max())


def _compare_caches_with_the_reference(cd, ref_dir, our_dir):
    # COORDREAD (model.cpp:712-740): same lines, the centred coordinates to the last printed digit or one off
    la, lb = (open(d / "COORDREAD").read().split("\n") for d in (ref_dir, our_dir))
    assert len(la) == len(lb) and la[0] == lb[0]
    for x, y in zip(la[1:], lb[1:]):
        tx, ty = x.split(), y.split()
        assert len(tx) == len(ty) and tx[:2] == ty[:2]
        assert all(abs(float(u) - float(v)) <= 2e-6 * max(1.0, abs(float(u))) for u, v in zip(tx[2:], ty[2:])), (x, y)
    # model.dump: float NormDen, int n, n x 24-byte points
    a, b = (open(d / "model.dump", "rb").read() for d in (ref_dir, our_dir))
    assert len(a) == len(b) and a[4:8] == b[4:8]
    nd_ref, nd_our = np.frombuffer(a[:4], "<f4")[0], np.frombuffer(b[:4], "<f4")[0]
    assert abs(nd_ref - nd_our) <= 4e-7 * abs(nd_ref)  # the reference sums the densities per reader thread, -ffast-math
    pa, pb = (np.frombuffer(x[8:], "<f4").reshape(-1, 6) for x in (a, b))
    for col in (0, 1, 2, 4, 5):  # pos[3], radius, density (column 3 is the unused quat4 of the point struct)
        assert pa[:, col].tobytes() == pb[:, col].tobytes(), col
    # maps.dump: int nMaps, nMaps x N x N floats; MRC stacks are normalised by the reader, where the
    # reference's -ffast-math build rounds differently in the last place (quirk Q7)
    a, b = (open(d / "maps.dump", "rb").read() for d in (ref_dir, our_dir))
    assert len(a) == len(b) and a[:4] == b[:4]
    ma, mb = (np.frombuffer(x[4:], "<f4") for x in (a, b))
    if cd.case.particle_format == "text":
        assert ma.tobytes() == mb.tobytes()
    else:
        np.testing.assert_allclose(mb, ma, rtol=0, atol=2.5e-7 * np.abs(ma).max())


@pytest.mark.parametrize("tag,extra,ncol", [("euler", "GRIDPOINTS_ALPHA 4\nGRIDPOINTS_BETA 3\n", 3),
                                            ("quat2", "USE_QUATERNIONS\nGRIDPOINTS_QUATERNION 2\n", 4),
                                            ("quat3", "USE_QUATERNIONS\nGRIDPOINTS_QUATERNION 3\n", 4)])
def test_orientation_grids_match_the_reference_binary(tag, extra, ncol, tmp_path):
    """Euler / quaternion grid generators (param.cpp:1009-1048,1141-1210) against the unmodified reference:
    with WRITE_PROB_ANGLES = number of orientations its ANG_PROB lists every orientation of the grid (4
    decimals); the multiset of rows must be the grid bioEM_b200 hands to the library.  Without the reference binary,
    the Euler grid is checked against the reference's stored output for the same grid (tests/golden/toy32euler): every
    orientation it printed must be a point of the grid."""
    import collections
    import subprocess
    exe = _build_host_bin()
    cd = build_case("toy32", str(tmp_path))
    common = ("PIXEL_SIZE 1.5\nNUMBER_PIXELS 32\nDISPLACE_CENTER 4 1\nCTF_DEFOCUS 1.0 4.0 3\n"
              "CTF_B_ENV 2.0 300.0 1\nCTF_AMPLITUDE 0.1 0.1 1\n")
    base = ["--Modelfile", cd.paths["model"], "--Particlesfile", cd.paths["particles"], "--Inputfile", "p.txt"]
    hook = tmp_path / "hook"
    hook.mkdir()
    (tmp_path / "p.txt").write_text(common + extra)
    r = subprocess.run([exe] + base, cwd=tmp_path, capture_output=True, text=True,
                       env={**os.environ, "BIOEM_B200_DUMP_INPUTS": str(hook)})
    assert r.returncode == 0, r.stderr[-400:]
    ang = np.fromfile(hook / "angles.bin", dtype=np.float32).reshape(-1, 4).astype(np.float64)

    def norm(row):  # "-0.0000" and "0.0000" are the same angle
        return tuple(0.0 if abs(v) < 5e-5 else v for v in row)

    mine = [tuple(float(f"{v:.4f}") for v in a[:ncol]) for a in ang]
    if not os.path.exists(REF_BIN):
        if tag != "euler":
            pytest.skip("reference binary not built (oracle/_ref) and no stored reference output for this grid")
        from bioem_b200.cases import CASES
        from bioem_b200.outputs import parse_output_probabilities
        assert CASES["toy32euler"].euler_grid == (4, 3)
        gold = os.path.join(ROOT, "tests", "golden", "toy32euler")
        rows = [tuple(float(x) for x in ln.split()[1:4]) for ln in open(os.path.join(gold, "ANG_PROB")).read().split("\n")
                if "Separated:" in ln]
        rows += [tuple(a[:3]) for a in parse_output_probabilities(os.path.join(gold, "Output_Probabilities"), False)["angles"]]
        assert len(rows) >= 9 and len(mine) == 4 * 3 * 4
        grid = set(map(norm, mine))
        assert all(norm(r) in grid for r in rows), sorted(set(map(norm, rows)) - grid)
        return
    (tmp_path / "p.txt").write_text(common + extra + f"WRITE_PROB_ANGLES {len(ang)}\n")
    r = subprocess.run([REF_BIN] + base, cwd=tmp_path, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout[-400:] + r.stderr[-400:]
    rows = []
    for ln in open(tmp_path / "ANG_PROB").read().split("\n"):
        t = ln.split()
        if len(t) > 6 and t[0] == "0" and "Separated:" in t:
            rows.append(tuple(float(x) for x in t[1:1 + ncol]))
    assert len(rows) == len(mine)
    assert collections.Counter(map(norm, rows)) == collections.Counter(map(norm, mine))


def test_multiple_mrc_list_matches_the_reference_binary(tmp_path):
    """--ReadMRC --ReadMultipleMRC (map.cpp:196-243): a text file naming several MRC stacks; the particles must
    come out in the reference's order and normalisation (its maps.dump is the witness, when the reference binary is
    built), and as the single-stack reading of the same images leaves them."""
    import subprocess
    from bioem_b200 import synth
    exe = _build_host_bin()
    cd = build_case("toy36g2", str(tmp_path))
    imgs = cd.particles
    synth.write_particles_mrc(str(tmp_path / "a.mrc"), imgs[:3])
    synth.write_particles_mrc(str(tmp_path / "b.mrc"), imgs[3:])
    (tmp_path / "list.txt").write_text(f"{tmp_path / 'a.mrc'}\n{tmp_path / 'b.mrc'}\n")
    cli = ["--Modelfile", cd.paths["model"], "--Particlesfile", str(tmp_path / "list.txt"), "--Inputfile", cd.paths["param"],
           "--ReadOrientation", cd.paths["orient"], "--ReadMRC", "--ReadMultipleMRC", "--DumpMaps"]
    ref_dir, our_dir, hook = tmp_path / "ref", tmp_path / "ours", tmp_path / "hook"
    for d in (ref_dir, our_dir, hook):
        d.mkdir()
    r = subprocess.run([exe] + cli, cwd=our_dir, capture_output=True, text=True,
                       env={**os.environ, "BIOEM_B200_DUMP_INPUTS": str(hook)})
    assert r.returncode == 0, r.stdout[-400:] + r.stderr[-400:]
    b = open(our_dir / "maps.dump", "rb").read()
    assert np.frombuffer(b[:4], "<i4")[0] == len(imgs)
    if os.path.exists(REF_BIN):
        r = subprocess.run([REF_BIN] + cli, cwd=ref_dir, capture_output=True, text=True)
        assert r.returncode == 0, r.stdout[-400:] + r.stderr[-400:]
        a = open(ref_dir / "maps.dump", "rb").read()
        assert len(a) == len(b) and a[:4] == b[:4]
        ma, mb = (np.frombuffer(x[4:], "<f4") for x in (a, b))
        np.testing.assert_allclose(mb, ma, rtol=0, atol=2.5e-7 * np.abs(ma).max())  # -ffast-math rounding of the reference
    # and the single-stack reading of the same images gives the same particles
    single = tmp_path / "single"
    single.mkdir()
    from bioem_b200.cases import reference_cli
    r = subprocess.run([exe] + reference_cli(cd) + ["--DumpMaps"], cwd=single, capture_output=True, text=True,
                       env={**os.environ, "BIOEM_B200_DUMP_INPUTS": str(single)})
    assert r.returncode == 0
    assert open(single / "maps.dump", "rb").read() == b


def test_pdb_reader_matches_the_reference_binary(tmp_path):
    """--ReadPDB (model.cpp:85-329,738-844): C-alpha atoms only, residue name -> radius / number of electrons
    for all 20 residue types, fixed columns; the reference's model.dump is the witness when the reference binary is
    built.  Without it: one point per CA record, at the coordinates of its fixed columns."""
    import subprocess
    exe = _build_host_bin()
    cd = build_case("toy32", str(tmp_path))
    res = ["GLY", "ALA", "VAL", "LEU", "ILE", "MET", "PHE", "TRP", "PRO", "SER", "THR", "CYS", "TYR", "ASN", "GLN",
           "ASP", "GLU", "LYS", "ARG", "HIS"]
    rng = np.random.default_rng(5)
    lines, serial = [], 1
    for i, rn in enumerate(res):
        for atom in ("N", "CA", "C"):
            x, y, z = rng.uniform(-9.0, 9.0, size=3)
            lines.append(f"ATOM  {serial:5d}  {atom:<3s} {rn} A{i + 1:4d}    {x:8.3f}{y:8.3f}{z:8.3f}  1.00  0.00")
            serial += 1
    lines += ["TER", "END"]
    (tmp_path / "m.pdb").write_text("\n".join(lines) + "\n")
    cli = ["--Modelfile", str(tmp_path / "m.pdb"), "--ReadPDB", "--Particlesfile", cd.paths["particles"], "--Inputfile",
           cd.paths["param"], "--ReadOrientation", cd.paths["orient"], "--DumpModel"]
    ref_dir, our_dir, hook = tmp_path / "ref", tmp_path / "ours", tmp_path / "hook"
    for d in (ref_dir, our_dir, hook):
        d.mkdir()
    r = subprocess.run([exe] + cli, cwd=our_dir, capture_output=True, text=True,
                       env={**os.environ, "BIOEM_B200_DUMP_INPUTS": str(hook)})
    assert r.returncode == 0, r.stdout[-400:] + r.stderr[-400:]
    b = open(our_dir / "model.dump", "rb").read()
    assert np.frombuffer(b[4:8], "<i4")[0] == len(res)
    pb = np.frombuffer(b[8:], "<f4").reshape(-1, 6)
    ca = np.array([[float(ln[30:38]), float(ln[38:46]), float(ln[46:54])] for ln in lines if ln[12:16] == " CA "],
                  dtype=np.float32)
    assert np.array_equal(pb[:, :3], ca)
    if os.path.exists(REF_BIN):
        r = subprocess.run([REF_BIN] + cli, cwd=ref_dir, capture_output=True, text=True)
        assert r.returncode == 0, r.stdout[-400:] + r.stderr[-400:]
        _compare_model_dumps(open(ref_dir / "model.dump", "rb").read(), b)


def _compare_model_dumps(a, b):
    """model.dump of the reference (a) and of bioEM_b200 (b): same point count, NormDen to the reference's rounding, the
    same float bits of pos[3], radius and density (column 3 is the unused quat4 of the point struct)"""
    assert len(a) == len(b) and a[4:8] == b[4:8]
    assert abs(np.frombuffer(a[:4], "<f4")[0] - np.frombuffer(b[:4], "<f4")[0]) <= 4e-7 * np.frombuffer(a[:4], "<f4")[0]
    pa, pb = (np.frombuffer(x[8:], "<f4").reshape(-1, 6) for x in (a, b))
    for col in (0, 1, 2, 4, 5):
        assert pa[:, col].tobytes() == pb[:, col].tobytes(), col


def test_mrc_volume_model_reader_matches_the_reference_binary(tmp_path):
    """--ReadModelMRC (model.cpp:332-416, BASELINE configs[3]): one model point per voxel of a mode-2 volume at
    ((i - nx/2) px, (j - ny/2) px, (k - nz/2) px), radius 2 px, density = voxel; witness: the reference's model.dump
    when the reference binary is built, and always synth.volume_to_points, the restatement of the reader that the cfg4
    cases are built with (their oracle results are pinned to the reference's output in tests/golden/cfg4_voxel_slice)."""
    import struct
    import subprocess
    exe = _build_host_bin()
    cd = build_case("toy32", str(tmp_path))
    nx, ny, nz = 6, 5, 4
    vol = np.random.default_rng(2).uniform(0.0, 3.0, size=(nz, ny, nx)).astype("<f4")  # file order: x fastest
    hdr = bytearray(1024)
    struct.pack_into("<4i", hdr, 0, nx, ny, nz, 2)
    struct.pack_into("<3i", hdr, 28, nx, ny, nz)
    struct.pack_into("<3f", hdr, 40, float(nx), float(ny), float(nz))
    struct.pack_into("<3f", hdr, 52, 90.0, 90.0, 90.0)
    struct.pack_into("<3i", hdr, 64, 1, 2, 3)
    hdr[208:212] = b"MAP "
    (tmp_path / "model.mrc").write_bytes(bytes(hdr) + vol.tobytes())
    cli = ["--Modelfile", str(tmp_path / "model.mrc"), "--ReadModelMRC", "--Particlesfile", cd.paths["particles"],
           "--Inputfile", cd.paths["param"], "--ReadOrientation", cd.paths["orient"], "--DumpModel"]
    ref_dir, our_dir, hook = tmp_path / "ref", tmp_path / "ours", tmp_path / "hook"
    for d in (ref_dir, our_dir, hook):
        d.mkdir()
    r = subprocess.run([exe] + cli, cwd=our_dir, capture_output=True, text=True,
                       env={**os.environ, "BIOEM_B200_DUMP_INPUTS": str(hook)})
    assert r.returncode == 0, r.stdout[-400:] + r.stderr[-400:]
    b = open(our_dir / "model.dump", "rb").read()
    assert np.frombuffer(b[4:8], "<i4")[0] == nx * ny * nz
    pb = np.frombuffer(b[8:], "<f4").reshape(-1, 6)
    from bioem_b200 import synth
    want = synth.volume_to_points(vol.reshape(-1).reshape(nx, ny, nz), cd.case.pixel_size).astype(np.float32)
    for col, wcol in ((0, 0), (1, 1), (2, 2), (4, 3), (5, 4)):
        assert np.array_equal(pb[:, col], want[:, wcol]), col
    if os.path.exists(REF_BIN):
        r = subprocess.run([REF_BIN] + cli, cwd=ref_dir, capture_output=True, text=True)
        assert r.returncode == 0, r.stdout[-400:] + r.stderr[-400:]
        _compare_model_dumps(open(ref_dir / "model.dump", "rb").read(), b)

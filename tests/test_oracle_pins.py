"""Pin the oracle (oracle/*.c) against every golden vector the reference holds for this path
(SURVEY.md 8c) and against the reference's own CPU implementation NEP_CPU (oracle/_ref)."""
import numpy as np
import pytest

from conftest import GOLDEN, TOL, assert_close
from gpumd_b200.structures import nep_type_order, read_xyz, rocksalt_pbte


def _static(oracle):
    order = nep_type_order(GOLDEN / "nep_PbTe_static.txt")
    s = read_xyz(GOLDEN / "gpumd_static_model.xyz", order)
    gold = read_xyz(GOLDEN / "gpumd_static_dump.xyz", order)
    return s, gold, oracle.NepOracle(GOLDEN / "nep_PbTe_static.txt")


@pytest.mark.parametrize("precision", [32, 64])
def test_pbte_static_known_answer(oracle, precision):
    """examples/gpumd_static/dump.xyz: E, 9-component virial and per-atom forces of 250-atom PbTe
    written by the reference GPU code (triclinic, small-box path)."""
    s, gold, m = _static(oracle)
    r = m.compute(s["type"], s["h"], s["pbc"], s["pos"], precision=precision, lists=True)
    assert_close(r["pe"].sum(), gold["energy"], **TOL["energy"], what="energy")
    assert_close(r["force"], gold["forces"], **TOL["force"], what="force")
    v = r["virial"].sum(axis=1)  # GPUMD order xx yy zz xy xz yz yx zx zy -> row-major 3x3
    v33 = np.array([v[0], v[3], v[4], v[6], v[1], v[5], v[7], v[8], v[2]])
    assert_close(v33, gold["virial"], rtol=1e-4, atol=2e-4, what="virial")
    # examples/gpumd_static/neighbor.out: "radial(max=92,actual=72), angular(max=10,actual=8)"
    txt = (GOLDEN / "gpumd_static_neighbor.out").read_text()
    assert "actual=72" in txt and "actual=8" in txt
    assert r["NN_radial"].max() == 72 and r["NN_angular"].max() == 8


@pytest.mark.parametrize("precision", [32, 64])
def test_bazro3_golden_regression(oracle, precision):
    """tests_pytest/fixtures/golden/bulk_bazro3.npz (test_regression.py:35-44): energy, forces and
    ASE-convention stress of the 40-atom rattled BaZrO3 cell."""
    order = nep_type_order(GOLDEN / "nep_BaZrO3.txt")
    s = read_xyz(GOLDEN / "BaZrO3-nat40-rattled.xyz", order)
    g = np.load(GOLDEN / "bulk_bazro3.npz")
    r = oracle.NepOracle(GOLDEN / "nep_BaZrO3.txt").compute(
        s["type"], s["h"], s["pbc"], s["pos"], precision=precision)
    assert_close(r["pe"].sum(), g["energy"], **TOL["energy"], what="energy")
    assert_close(r["force"].T, g["forces"], rtol=1e-4, atol=2e-5, what="forces")
    vol = abs(np.linalg.det(s["h"].reshape(3, 3)))
    v = r["virial"].sum(axis=1)
    stress = -np.array([v[0], v[1], v[2], v[5], v[4], v[3]]) / vol  # Voigt xx yy zz yz xz xy
    assert_close(stress, g["stress"], rtol=1e-4, atol=1e-6, what="stress")


@pytest.mark.parametrize("model,structure", [
    ("nep_PbTe_static.txt", "static"), ("nep_BaZrO3.txt", "bazro3"), ("nep_PbTe.txt", "c1"),
    ("nep_synth_50types.txt", "synth50")])
def test_oracle_matches_reference_nep_cpu(oracle, model, structure):
    """FP64 restatement vs the reference's own NEP_CPU (tests/golden/refcpu_nep.npz: its energies,
    forces and virials with the inputs they were computed on; tests/golden/make_fixtures.py).
    Differences come only from NEP_CPU keeping the parameters in double while the GPU reference
    (and the restatement) round them to float on load."""
    d = np.load(GOLDEN / "refcpu_nep.npz")
    s = {k: d[f"{structure}_{k}"] for k in ("type", "h", "pbc", "pos")}
    ref = {k: d[f"{structure}_{k}"] for k in ("pe", "force", "virial")}
    r = oracle.NepOracle(GOLDEN / model).compute(s["type"], s["h"], s["pbc"], s["pos"], precision=64)
    n = s["type"].shape[0]
    assert abs(r["pe"].sum() - ref["pe"].sum()) / n < 1e-7
    assert_close(r["force"], ref["force"], rtol=1e-6, atol=5e-7, what="force")
    assert_close(r["virial"], ref["virial"], rtol=1e-5, atol=5e-6, what="virial")


@pytest.mark.parametrize("case,model", [("sp_pbte", "nep_PbTe.txt"), ("sp_unep", "nep_UNEP_v1.txt")])
def test_oracle_matches_reference_gpu_large_box(oracle, case, model):
    """tests/golden/refgpu_sp_*.npz: energy / per-atom forces / virial written by the UNMODIFIED
    reference gpumd (oracle/_ref/gpumd_ref, built from /root/reference with -arch=sm_100) on a B200,
    large-box path (find_neighbor_list_large_box ... find_force_ZBL), inputs from our generators
    (scripts/run_reference_gpumd.py).  This pins the FP32 restatement against the real GPU code."""
    d = np.load(GOLDEN / f"refgpu_{case}.npz")
    n = d["type"].shape[0]
    r = oracle.NepOracle(GOLDEN / model).compute(d["type"], d["h"], d["pbc"], d["pos"], precision=32)
    assert abs(r["pe"].sum() - float(d["energy"])) / n < 2e-7
    assert_close(r["force"], d["force"], rtol=1e-5, atol=1e-5, what="force")
    v = r["virial"].sum(axis=1)
    v33 = np.array([v[0], v[3], v[4], v[6], v[1], v[5], v[7], v[8], v[2]])
    assert_close(v33, d["virial"], rtol=1e-5, atol=5e-3, what="virial")


def test_lj_oracle_matches_reference_gpu(oracle):
    """LJ single point of the reference gpumd on B200 (10 976 Ar atoms): pins the LJ restatement,
    which has no golden vector in the reference's own tests."""
    d = np.load(GOLDEN / "refgpu_sp_lj.npz")
    n = d["type"].shape[0]
    r = oracle.lj_compute(np.array([[[1.032e-2, 3.405, 10.0]]]), d["type"], d["h"], d["pbc"], d["pos"])
    assert abs(r["pe"].sum() - float(d["energy"])) / n < 1e-9
    assert_close(r["force"], d["force"], rtol=1e-6, atol=5e-7, what="force")
    v = r["virial"].sum(axis=1)
    v33 = np.array([v[0], v[3], v[4], v[6], v[1], v[5], v[7], v[8], v[2]])
    assert_close(v33, d["virial"], rtol=1e-6, atol=1e-4, what="virial")


def test_tersoff_oracle_matches_reference_gpu(oracle):
    """Tersoff-1989 Si single point of the reference gpumd on B200 (8000 atoms, FP64 code): the
    restatement agrees to round-off."""
    d = np.load(GOLDEN / "refgpu_sp_si.npz")
    nt, para = oracle.tersoff_parameters(GOLDEN / "tersoff_Si_1989.txt")
    r = oracle.tersoff_compute(nt, para, d["type"], d["h"], d["pbc"], d["pos"])
    assert abs(r["pe"].sum() - float(d["energy"])) < 1e-9 * abs(float(d["energy"]))
    assert_close(r["force"], d["force"], rtol=1e-10, atol=1e-10, what="force")
    v = r["virial"].sum(axis=1)
    v33 = np.array([v[0], v[3], v[4], v[6], v[1], v[5], v[7], v[8], v[2]])
    assert_close(v33, d["virial"], rtol=1e-10, atol=1e-8, what="virial")


def test_eam_oracle_matches_reference_gpu(oracle):
    """Zhou-2004 Cu-Fe-Ni alloy single point of the reference gpumd on B200 (4000 atoms)."""
    d = np.load(GOLDEN / "refgpu_sp_eam.npz")
    n = d["type"].shape[0]
    model, nt, para = oracle.eam_parameters(GOLDEN / "eam_zhou_2004_CuFeNi.txt")
    r = oracle.eam_compute(model, nt, para, d["type"], d["h"], d["pbc"], d["pos"])
    assert abs(r["pe"].sum() - float(d["energy"])) / n < 1e-6
    assert_close(r["force"], d["force"], rtol=1e-5, atol=1e-5, what="force")


def test_oracle_f32_vs_f64(oracle):
    s = rocksalt_pbte(4, rattle=0.05, seed=1)
    m = oracle.NepOracle(GOLDEN / "nep_PbTe.txt")
    a = m.compute(s["type"], s["h"], s["pbc"], s["pos"], precision=32)
    b = m.compute(s["type"], s["h"], s["pbc"], s["pos"], precision=64)
    n = s["type"].shape[0]
    assert abs(a["pe"].sum() - b["pe"].sum()) / n < TOL["energy_per_atom"]
    assert_close(a["force"], b["force"], **TOL["force"], what="force")


def test_neighbor_oracle_bruteforce(oracle):
    """The cell-list candidate search must find exactly the FP32-membership sets an O(N^2) scan finds."""
    s = rocksalt_pbte(3, a=6.6, rattle=0.1, seed=11)  # 19.8 A box, rc 8 -> minimum image valid
    rc = 8.0
    NN, NL = oracle.neighbor_list(s["h"], s["pbc"], s["pos"], rc, mn=128)
    pos = s["pos"]
    L = np.float32(s["h"][0])
    n = pos.shape[1]
    for i in range(0, n, 7):
        d = (pos - pos[:, i:i + 1]).astype(np.float32)  # FP64 subtract, narrowed
        d = np.where(d < -L * np.float32(0.5), d + L, np.where(d > L * np.float32(0.5), d - L, d))
        x, y, z = d
        d2 = np.float32(1) * (y * y)
        # fma(z,z, fma(x,x, y*y)) evaluated exactly in float64 then rounded once per fma
        d2 = (x.astype(np.float64) * x + (y * y).astype(np.float64)).astype(np.float32)
        d2 = (z.astype(np.float64) * z + d2.astype(np.float64)).astype(np.float32)
        mine = np.nonzero((d2 < np.float32(rc * rc)) & (np.arange(n) != i))[0]
        assert np.array_equal(mine, NL[i, :NN[i]])


def test_lj_oracle_analytic(oracle):
    """LJ restatement vs the closed form for an fcc crystal (parity for LJ is otherwise unpinned)."""
    from gpumd_b200.structures import fcc
    s = fcc(5, 5.30)  # 26.5 A box; rc 10 -> thickness > 2 rc
    eps, sig, rc = 1.032e-2, 3.405, 10.0
    r = oracle.lj_compute(np.array([[[eps, sig, rc]]]), s["type"], s["h"], s["pbc"], s["pos"])
    pos = s["pos"]
    L = s["h"][0]
    d = pos - pos[:, :1]
    d -= L * np.round(d / L)
    dist = np.sqrt((d * d).sum(axis=0))
    dist = dist[(dist > 0) & (dist < rc)]
    u = 0.5 * np.sum(4 * eps * ((sig / dist) ** 12 - (sig / dist) ** 6))
    assert abs(r["pe"][0] - u) < 2e-6 * abs(u) + 1e-7
    assert np.abs(r["force"]).max() < 2e-5  # perfect lattice
    # virial trace = -1/2 sum r dU/dr
    w = -0.5 * np.sum(4 * eps * (-12 * (sig / dist) ** 12 + 6 * (sig / dist) ** 6))
    assert abs(r["virial"][:3, 0].sum() - w) < 1e-5 * abs(w)


def test_md_oracle_basics(oracle):
    rng = np.random.default_rng(0)
    n = 50
    mass = rng.uniform(1, 100, n)
    pos, vel, f = rng.normal(size=(3, n)), rng.normal(size=(3, n)), rng.normal(size=(3, n))
    p1, v1 = oracle.velocity_verlet(True, 0.1, mass, pos, vel, f)
    assert np.allclose(v1, vel + 0.05 * f / mass) and np.allclose(p1, pos + 0.1 * v1)
    p2, v2 = oracle.velocity_verlet(False, 0.1, mass, pos, vel, f)
    assert np.array_equal(p2, pos) and np.allclose(v2, v1)
    pe, vir = rng.normal(size=n), rng.normal(size=(9, n))
    t = oracle.find_thermo(n, 7.0, mass, pe, vel, vir)
    assert np.isclose(t[0], (mass * (vel ** 2).sum(0)).sum() / (3 * n * 8.617343e-5))
    assert np.isclose(t[1], pe.sum())
    assert np.isclose(t[5], (vir[3] + mass * vel[0] * vel[1]).sum() / 7.0)
    h = np.diag([10.0, 11.0, 12.0]).reshape(9)
    w = oracle.apply_pbc(h, [1, 1, 0], np.array([[-1.0, 10.5], [5.0, 12.0], [-3.0, 13.0]]))
    assert np.allclose(w, [[9.0, 0.5], [5.0, 1.0], [-3.0, 13.0]])


def test_bdp_random_stream_is_the_standard_librarys(oracle):
    """The reference's BDP thermostat draws from std::mt19937(12345678) through
    std::uniform_real_distribution<double>(0,1) (ensemble_bdp.cu:29-36, svr_utilities.cuh:29,54).  The
    restatement must produce the very same raw words and doubles as those library objects (built
    from <random> by oracle/Makefile with the compiler that builds the reference)."""
    R = oracle.stdrng()
    for seed in (12345678, 1, 4294967295):
        raw = np.zeros(2000, np.uint32)
        R.stdrng_raw(seed, raw.size, raw.ctypes.data)
        u = np.zeros(1000, np.float64)
        R.stdrng_uniform01(seed, u.size, u.ctypes.data)
        a = oracle.BdpOracle(seed)
        assert [a.raw() for _ in range(raw.size)] == raw.tolist()
        b = oracle.BdpOracle(seed)
        assert [b.rand01() for _ in range(u.size)] == u.tolist()  # bit-exact


def test_bdp_factor_statistics(oracle):
    """Known answer of the published algorithm: with tau -> 0 the resampled kinetic energy is a fresh
    Gamma(ndeg/2) draw, so <factor^2 * T_inst / T0> = 1 and its variance is 2/ndeg."""
    o = oracle.BdpOracle(7)
    n_atoms = 40
    x = np.array([o.factor(250.0, n_atoms, 300.0, 0.05) ** 2 * 250.0 / 300.0 for _ in range(4000)])
    assert abs(x.mean() - 1.0) < 4 * np.sqrt(2.0 / 120 / 4000)
    assert abs(x.var() - 2.0 / 120) < 0.15 * 2.0 / 120

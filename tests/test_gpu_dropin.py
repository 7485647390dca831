"""The drop-in proof: the reference `gpumd` itself, with libb200md plugged into its own plugin surface
(oracle/_ref/gpumd_b200, built by oracle/Makefile.gpumd_b200: reference objects + our adapter classes
compiled against the reference's force/potential.cuh and integrate/ensemble.cuh + the two call-site
hooks of INTEGRATION.md applied to a copy).  With GPUMD_B200 unset the binary IS the reference; with
GPUMD_B200=1 its Force / Integrate objects are libb200md's.  Same binary, same inputs, both ways."""
import os
import shutil
import subprocess

import numpy as np
import pytest

from conftest import GOLDEN, ROOT
from gpumd_b200.structures import init_velocities, nep_type_order, rocksalt_pbte, write_xyz

pytestmark = pytest.mark.gpu
EXE = ROOT / "oracle" / "_ref" / "gpumd_b200"


def read_thermo(path):
    return np.array([ln.split()[:18] for ln in open(path) if not ln.startswith("#")], dtype=np.float64)


def run(tmp, b200, timeout=900):
    for f in ("thermo.out", "neighbor.out"):
        (tmp / f).unlink(missing_ok=True)
    env = dict(os.environ)
    env.pop("GPUMD_B200", None)
    if b200:
        env["GPUMD_B200"] = "1"
    env["CUDA_VISIBLE_DEVICES"] = env.get("CUDA_VISIBLE_DEVICES", "0").split(",")[0]  # NEP, not NEP_MULTIGPU
    r = subprocess.run([str(EXE)], cwd=tmp, capture_output=True, text=True, timeout=timeout, env=env)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
    return r.stdout, read_thermo(tmp / "thermo.out")


@pytest.fixture(scope="module")
def exe():
    if not EXE.exists():
        pytest.skip("oracle/_ref/gpumd_b200 not built (build() with GPUMD_REFERENCE naming a GPUMD source tree)")
    return EXE


def test_reference_carbon_case_through_the_plugin(exe, tmp_path):
    """tests/gpumd/carbon of the reference (64 000 atoms, C_2022_NEP4, `velocity 300`, NVE, 100
    steps) executed by the reference binary with GPUMD_B200=1, against its checked-in thermo1.out."""
    d = np.load(GOLDEN / "carbon_model.npz")
    pos = d["pos"]
    with open(tmp_path / "model.xyz", "w") as f:
        f.write(f"{pos.shape[0]}\n{str(d['header'])}\n")
        for x, y, z in pos:
            f.write(f"C {x:.11f} {y:.11f} {z:.11f}\n")
    shutil.copyfile(GOLDEN / "nep_C_2022_NEP4.txt", tmp_path / "potential.txt")
    (tmp_path / "run.in").write_text(
        "potential potential.txt\nvelocity 300\ntime_step 1.0\nensemble nve\ndump_thermo 10\nrun 100\n")
    out, mine = run(tmp_path, b200=True)
    assert "Use the b200md NEP backend" in out and "Use the b200md integrator" in out
    ref = read_thermo(GOLDEN / "carbon_thermo1.out")
    n = pos.shape[0]
    assert mine.shape == ref.shape == (10, 18)
    e_mine, e_ref = mine[:, 1] + mine[:, 2], ref[:, 1] + ref[:, 2]
    # same bounds and reasoning as tests/test_gpu_host_exe.py (FP32 force-noise wander of ~1e-6 eV/atom)
    assert np.all(np.abs(e_mine - e_ref) / n < 4e-6)
    assert np.abs(e_mine - e_mine[0]).max() < 2.0 * np.abs(e_ref - e_ref[0]).max()
    assert np.all(np.abs(mine[:, 0] - ref[:, 0]) < 1.5)
    assert np.all(np.abs(mine[:, 2] - ref[:, 2]) / n < 3e-4)
    assert np.array_equal(mine[:, 9:], ref[:, 9:])
    # and against the SAME binary with the plugin off (= the reference, same rand() stream): the two
    # trajectories start identically and separate only through FP32 summation order
    out, theirs = run(tmp_path, b200=False)
    assert "b200md" not in out
    assert abs(mine[0, 0] - theirs[0, 0]) < 5e-3 and abs(mine[0, 2] - theirs[0, 2]) / n < 2e-7
    assert np.all(np.abs(mine[:, 0] - theirs[:, 0]) < 0.05)


@pytest.mark.parametrize("ensemble", ["nvt_ber 300 300 100", "nvt_nhc 300 300 100"])
def test_fix_and_move_groups_match_the_reference(exe, tmp_path, ensemble):
    """`fix` / `move` (integrate.cu:1362-1470, ensemble.cu:111-174): a PbTe slab with three groups along
    z -- bottom layer frozen, top layer dragged at a constant velocity, middle thermostatted -- through
    the plugin and through the reference's own classes in the same binary."""
    s = rocksalt_pbte(12, rattle=0.02, seed=1)  # 13 824 atoms
    n = s["type"].shape[0]
    z = s["pos"][2]
    L = s["h"][8]
    label = np.where(z < 0.15 * L, 0, np.where(z > 0.85 * L, 2, 1)).astype(np.int32)
    vel = init_velocities(s["mass"], 300.0, seed=42)
    write_xyz(tmp_path / "model0.xyz", s, nep_type_order(GOLDEN / "nep_PbTe.txt"), vel)
    lines = open(tmp_path / "model0.xyz").read().splitlines()
    lines[1] = lines[1].replace('pbc="T T T"', 'pbc="T T F"') + ":group:I:1"
    with open(tmp_path / "model.xyz", "w") as f:
        f.write(lines[0] + "\n" + lines[1] + "\n")
        for k, ln in enumerate(lines[2:]):
            f.write(f"{ln} {label[k]}\n")
    shutil.copyfile(GOLDEN / "nep_PbTe.txt", tmp_path / "potential.txt")
    (tmp_path / "run.in").write_text(
        f"potential potential.txt\nensemble {ensemble}\nfix 0\nmove 2 0.0005 0 0\ntime_step 1\n"
        "dump_thermo 10\nrun 100\n")
    _, mine = run(tmp_path, b200=True)
    _, theirs = run(tmp_path, b200=False)
    assert mine.shape == theirs.shape == (10, 18)
    for k in range(10):
        tol = 2e-5 * (1 + k)
        assert abs(mine[k, 0] - theirs[k, 0]) < tol * 3000, (k, mine[k, 0], theirs[k, 0])
        assert abs(mine[k, 2] - theirs[k, 2]) < tol * abs(theirs[k, 2])

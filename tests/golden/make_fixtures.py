"""Regenerate tests/golden/ from the read-only reference tree (run in the build container).

Everything copied here is DATA the reference's own tests/examples pin this path with
(SURVEY.md 8c): potential files, input structures and the checked-in known-answer outputs.
No reference source code is copied; the tests only ever read the committed copies.

    GPUMD_REFERENCE=<GPUMD source tree> python tests/golden/make_fixtures.py
"""
import os
import shutil
from pathlib import Path

import numpy as np

REF = Path(os.environ["GPUMD_REFERENCE"])
OUT = Path(__file__).resolve().parent

COPIES = {
    # PbTe 250-atom known-answer single point: examples/gpumd_static (E, virial, per-atom forces)
    "examples/gpumd_static/model.xyz": "gpumd_static_model.xyz",
    "examples/gpumd_static/dump.xyz": "gpumd_static_dump.xyz",
    "examples/gpumd_static/neighbor.out": "gpumd_static_neighbor.out",
    "examples/nep_train/nep.txt": "nep_PbTe_static.txt",
    # the PbTe model BASELINE.json's metric is quoted on
    "tests/gpumd/dump_observer/PbTe_species/PbTe.txt": "nep_PbTe.txt",
    # BaZrO3 40-atom golden regression (tests_pytest/test_regression.py:35-44)
    "tests_pytest/fixtures/models/nep_BaZrO3.txt": "nep_BaZrO3.txt",
    "tests_pytest/fixtures/structures/BaZrO3-nat40-rattled.xyz": "BaZrO3-nat40-rattled.xyz",
    # the other structure / model pairs of the reference's property tests (tests_pytest/conftest.py:
    # invariances, finite-difference forces): 3-type ZBL perovskite, 1-type carbon with 17/13 basis
    # functions and a 100-neuron layer, 2-type water with the 4-body term
    "tests_pytest/fixtures/models/nep_BaTiO3.txt": "nep_BaTiO3.txt",
    "tests_pytest/fixtures/structures/BaTiO3-nat40-rattled.xyz": "BaTiO3-nat40-rattled.xyz",
    "tests_pytest/fixtures/models/nep_C.txt": "nep_C_pytest.txt",
    "tests_pytest/fixtures/structures/C-nat16-rattled.xyz": "C-nat16-rattled.xyz",
    "tests_pytest/fixtures/models/nep_water.txt": "nep_water.txt",
    "tests_pytest/fixtures/structures/water-nat63-from-md.xyz": "water-nat63-from-md.xyz",
    # carbon 64 000-atom NVE trajectory golden (tests/gpumd/carbon): thermo + neighbour maxima
    "potentials/nep/C_2022_NEP4.txt": "nep_C_2022_NEP4.txt",
    "tests/gpumd/carbon/thermo1.out": "carbon_thermo1.out",
    "tests/gpumd/carbon/neighbor1.out": "carbon_neighbor1.out",
    "tests/gpumd/carbon/run.in": "carbon_run.in",
    # LJ argon parameters (config C2)
    "potentials/lj/Ar_10A.txt": "lj_Ar_10A.txt",
    "potentials/tersoff/Si_Tersoff_1989.txt": "tersoff_Si_1989.txt",
    # UNEP-v1 16-metal alloy model (config C4): 16 types, universal ZBL, 4- and 5-body terms
    "potentials/nep/Song-2024-UNEP-v1-AgAlAuCrCuMgMoNiPbPdPtTaTiVWZr.txt": "nep_UNEP_v1.txt",
}


# The other NEP models the reference ships under potentials/nep (tests/test_reference_models_cpu.py),
# xz-compressed.  NEP89 (89 species, 16 MB) is cut to the twelve metals that test draws from: their
# ANN blocks and the 12 x 12 block of both coefficient tables, so the slice gives the full model's
# energies for any structure made of these species.
SHIPPED_NEP = {
    "potentials/nep/Si_2022_NEP4_3body.txt": "nep_Si_2022_NEP4_3body.txt.xz",
    "potentials/nep/Si_2022_NEP4_4body.txt": "nep_Si_2022_NEP4_4body.txt.xz",
    "potentials/nep/Si_2022_NEP4_5body.txt": "nep_Si_2022_NEP4_5body.txt.xz",
    "potentials/nep/C_2024_NEP4.txt": "nep_C_2024_NEP4.txt.xz",
}
NEP89 = "potentials/nep/nep89_20250409/nep89_20250409.txt"
NEP89_SPECIES = ("Al", "Ti", "Fe", "Co", "Ni", "Cu", "Zr", "Mo", "Pd", "Ag", "Pt", "Au")


def nep_species_slice(text, species):
    """A NEP4 model file restricted to `species` (layout as NEP::NEP reads it, nep.cu:88-420: seven
    header lines, per-type ANN blocks w0[nneu][dim] b0[nneu] w1[nneu], the common bias, c_radial and
    c_angular indexed [(n*(K+1)+k)*Nt^2 + t1*Nt + t2], q_scaler[dim])."""
    lines = text.split("\n")
    head = lines[0].split()
    names, nt = head[2:], int(head[1])
    keep = sorted(names.index(x) for x in species)
    kw = {ln.split()[0]: ln.split()[1:] for ln in lines[1:7]}
    assert len(kw["cutoff"]) == 4, "only the global-cutoff layout"
    kw = {k: [int(v) for v in kw[k]] for k in ("n_max", "basis_size", "l_max", "ANN")}
    nr1, na1 = kw["n_max"][0] + 1, kw["n_max"][1] + 1
    kr1, ka1 = kw["basis_size"][0] + 1, kw["basis_size"][1] + 1
    lm = kw["l_max"]
    dim = nr1 + na1 * (lm[0] + (lm[1] > 0) + (lm[2] > 0))
    nneu = kw["ANN"][0]
    per = nneu * dim + 2 * nneu
    body = lines[7:]
    out = [f"{head[0]} {len(keep)} " + " ".join(names[k] for k in keep)] + lines[1:7]
    for k in keep:
        out += body[k * per:(k + 1) * per]
    out.append(body[nt * per])
    at = nt * per + 1
    for rows in (nr1 * kr1, na1 * ka1):
        for r in range(rows):
            out += [body[at + r * nt * nt + a * nt + b] for a in keep for b in keep]
        at += rows * nt * nt
    assert len(body) - at == dim + 1 and body[-1] == ""
    return "\n".join(out + body[at:])


def write_xz(path, text):
    import lzma
    path.write_bytes(lzma.compress(text.encode(), preset=9 | lzma.PRESET_EXTREME))
    print("wrote", path.name)


def nep_cpu_results():
    """refcpu_nep.npz: the reference's own NEP_CPU (FP64; oracle/_ref/libnep_cpu_ref.so, built by
    oracle/Makefile from $GPUMD_REFERENCE) on the inputs of tests/test_oracle_pins.py::
    test_oracle_matches_reference_nep_cpu, stored with those inputs."""
    import sys
    sys.path.insert(0, str(OUT.parents[1]))
    sys.path.insert(0, str(OUT.parent))
    from cases import NEP_CASES_SYNTH
    from gpumd_b200.structures import nep_type_order, read_xyz, rocksalt_pbte
    from oracle import oracle_py
    oracle_py.build()
    assert oracle_py.ref_available(), "oracle/_ref/libnep_cpu_ref.so not built (set GPUMD_REFERENCE)"
    cases = {
        "static": ("nep_PbTe_static.txt", lambda o: read_xyz(OUT / "gpumd_static_model.xyz", o)),
        "bazro3": ("nep_BaZrO3.txt", lambda o: read_xyz(OUT / "BaZrO3-nat40-rattled.xyz", o)),
        # config C1: 216-atom rocksalt PbTe, rattle 0.05 A, seed 1
        "c1": ("nep_PbTe.txt", lambda o: rocksalt_pbte(3, rattle=0.05, seed=1)),
        "synth50": ("nep_synth_50types.txt", lambda o: NEP_CASES_SYNTH["synth50"][1]()),
    }
    arrays = {}
    for name, (model, make) in cases.items():
        s = make(nep_type_order(OUT / model))
        r = oracle_py.RefNepCpu(OUT / model).compute(s["type"], s["h"], s["pos"])
        arrays.update({f"{name}_type": s["type"], f"{name}_h": s["h"], f"{name}_pbc": np.asarray(s["pbc"]),
                       f"{name}_pos": s["pos"], f"{name}_pe": r["pe"], f"{name}_force": r["force"],
                       f"{name}_virial": r["virial"]})
    np.savez_compressed(OUT / "refcpu_nep.npz", **arrays)
    print("wrote refcpu_nep.npz")


def main():
    for src, dst in COPIES.items():
        shutil.copyfile(REF / src, OUT / dst)
        print("copied", src, "->", dst)
    for src, dst in SHIPPED_NEP.items():
        write_xz(OUT / dst, (REF / src).read_text())
    write_xz(OUT / "nep_NEP89_12metals.txt.xz", nep_species_slice((REF / NEP89).read_text(), NEP89_SPECIES))
    nep_cpu_results()
    g = np.load(REF / "tests_pytest/fixtures/golden/bulk_bazro3.npz")
    np.savez(OUT / "bulk_bazro3.npz", **{k: g[k] for k in g})
    # The carbon model.xyz is 4 MB of text; keep it as compressed float64 arrays instead.
    lines = (REF / "tests/gpumd/carbon/model.xyz").read_text().splitlines()
    n = int(lines[0])
    pos = np.array([[float(v) for v in ln.split()[1:4]] for ln in lines[2 : 2 + n]])
    np.savez_compressed(OUT / "carbon_model.npz", header=np.array(lines[1]), pos=pos)
    print("wrote carbon_model.npz", pos.shape)


if __name__ == "__main__":
    main()

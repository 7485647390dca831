"""Every potential-energy NEP model the reference ships under potentials/nep (stored under tests/golden,
xz-compressed; tests/golden/make_fixtures.py): the model loader accepts it and the kernel bodies (host
build) reproduce the oracle on a small random structure.  NEP89 is stored as its slice to the twelve
metals the structure is drawn from, and run through the per-pair contraction of the radial descriptor,
the path its 89 species take."""
import lzma

import numpy as np
import pytest

from conftest import GOLDEN
from gpumd_b200.structures import diamond, fcc, nep_type_order
from test_kernel_bodies_cpu import check_nep

MODELS = {
    "Si_3body": ("nep_Si_2022_NEP4_3body.txt.xz", "diamond", 5.43),
    "Si_4body": ("nep_Si_2022_NEP4_4body.txt.xz", "diamond", 5.43),
    "Si_5body": ("nep_Si_2022_NEP4_5body.txt.xz", "diamond", 5.43),
    "C_2024": ("nep_C_2024_NEP4.txt.xz", "diamond", 3.57),
    "UNEP_v1": ("nep_UNEP_v1.txt", "alloy", 3.9),
    "NEP89": ("nep_NEP89_12metals.txt.xz", "alloy89", 3.9),
}


@pytest.mark.parametrize("name", list(MODELS))
def test_shipped_nep_models_match_oracle(oracle, emu, name, tmp_path, monkeypatch):
    fname, kind, a = MODELS[name]
    path = GOLDEN / fname
    if path.suffix == ".xz":
        path = tmp_path / path.stem
        path.write_bytes(lzma.decompress((GOLDEN / fname).read_bytes()))
    if kind == "alloy89":
        monkeypatch.setenv("B200MD_NEP_RADDIRECT", "1")
    order = nep_type_order(path)
    if kind == "diamond":
        s = diamond(3, a=a, rattle=0.05, seed=2, symbol="Si")
        s["symbols"] = order
    else:
        s = fcc(5, a, rattle=0.08, seed=4)
        rng = np.random.default_rng(4)
        if kind == "alloy89":  # a dozen of the 89 species, metals so that a = 3.9 A is not absurd
            pick = [order.index(x) for x in ("Al", "Ti", "Fe", "Co", "Ni", "Cu", "Zr", "Mo", "Pd", "Ag", "Pt", "Au")]
            s["type"] = rng.choice(pick, s["type"].shape[0]).astype(np.int32)
        else:
            s["type"] = rng.integers(0, len(order), s["type"].shape[0]).astype(np.int32)
        s["symbols"] = order
    n = s["type"].shape[0]
    check_nep(oracle, emu.nep(path, n), str(path), s, n)

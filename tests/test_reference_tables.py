"""The constant tables that define the reference's result are the reference's own bytes (VERDICT r1, item 1a):
the 512-point disk of ReSTIR PT's spatial search (IndirectLighting/ReSTIR_PT/SampleSet.hlsli:8-523), the 32-point set
of ReSTIR DI's spatial pass (DirectLighting/Emissive/Resampling.hlsli:352-386) and the directional-albedo volume
Assets/LUT/rho.dds. The committed assets are compared byte for byte with an extraction from the reference tree, frozen in
tests/golden/reference_tables.npz by `reference_outputs`, and their SHA-256 with the values recorded here at extraction time."""
import hashlib
import os
import sys
import numpy as np
import pytest

from tests.golden_pins import Golden, pin

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ASSETS = os.path.join(ROOT, "zetaray_b200", "assets")
SHA256 = {
    "disk512.bin": "5d1e6337be21687004bccc75cfe9d5a08af100ce450a624d3992fcf53b68c391",
    "disk32.bin": "5c157f153647d7b965b98535147cfbfc0477bf9ee35b8e806bda953d82371aa2",
    "rho_lut.bin": "e8bb63d6c42b97614f5288ff9fbc184240d76e19565a7aeea2dfaca2897f74f6",
}


@pytest.mark.parametrize("name", sorted(SHA256))
def test_asset_hash(name):
    assert hashlib.sha256(open(os.path.join(ASSETS, name), "rb").read()).hexdigest() == SHA256[name]


def reference_outputs():
    """The three tables as tools/extract_reference_tables.py reads them from the reference tree."""
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import extract_reference_tables as ert
    return {name: pin(arr) for name, arr in ert.tables().items()}


def test_assets_are_the_reference_bytes():
    ref = Golden("reference_tables.npz")
    for name in sorted(SHA256):
        ref.check(name, np.fromfile(os.path.join(ASSETS, name), dtype=np.uint8).reshape(-1, ref[name + ".rows"].shape[1]))


def test_table_shapes_and_ranges():
    d512 = np.fromfile(os.path.join(ASSETS, "disk512.bin"), dtype=np.float32).reshape(512, 2)
    assert (np.linalg.norm(d512, axis=1) <= 1.0 + 1e-3).all()          # unit disk
    assert (d512.astype(np.float16).astype(np.float32) == d512).all()    # binary16-representable
    d32 = np.fromfile(os.path.join(ASSETS, "disk32.bin"), dtype=np.float32).reshape(32, 2)
    assert (d32 >= 0).all() and (d32 <= 1).all()
    assert (d32.astype(np.float16).astype(np.float32) == d32).all()
    rho = np.fromfile(os.path.join(ASSETS, "rho_lut.bin"), dtype=np.uint16)
    assert rho.size == 64 * 32 * 16

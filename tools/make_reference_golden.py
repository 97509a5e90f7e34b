"""Freezes what the reference's own code returns for the inputs of the pinning tests into tests/golden/, so that those tests
run without the reference tree:

  reference_alias.npz   Kahan sum, alias table, RNG and Halton (oracle/_ref/libref_alias.so)   tests/test_alias_oracle.py
  reference_scene.npz   scene-data constructors and struct layouts (oracle/_ref/libref_scene.so) tests/test_scene_pinning.py
  reference_tables.npz  the constant tables of tools/extract_reference_tables.py                tests/test_reference_tables.py

Each test module's `reference_outputs` says what is frozen. Needs the reference tree and the libraries `make -C oracle ref`
builds from it; the product library must be built too (python -m zetaray_b200.build).

    python tools/make_reference_golden.py"""
import ctypes as C
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tests import golden_pins, orc  # noqa: E402
from tests import test_alias_oracle, test_reference_tables, test_scene_pinning  # noqa: E402


def main():
    reflib = orc.load_ref()
    scene_so = os.path.join(ROOT, "oracle", "_ref", "libref_scene.so")
    if reflib is None or not os.path.exists(scene_so):
        raise SystemExit("oracle/_ref is not built: run `make -C oracle ref` where the reference tree is present")
    golden_pins.save("reference_alias.npz", test_alias_oracle.reference_outputs(reflib))
    golden_pins.save("reference_scene.npz", test_scene_pinning.reference_outputs(C.CDLL(scene_so)))
    golden_pins.save("reference_tables.npz", test_reference_tables.reference_outputs())
    for name in ("reference_alias.npz", "reference_scene.npz", "reference_tables.npz"):
        path = os.path.join(golden_pins.GOLDEN, name)
        print("wrote %s (%d bytes)" % (path, os.path.getsize(path)))


if __name__ == "__main__":
    main()

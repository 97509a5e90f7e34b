"""Extracts the three constant tables that define the reference's result from the reference tree and writes them as the
product's data assets (zetaray_b200/assets/). They are inputs of the algorithm, not code: with other tables the neighbour
indices of both spatial passes and every dielectric-reflectance lookup differ from the reference by construction.

  disk512.bin  512 x float2  IndirectLighting/ReSTIR_PT/SampleSet.hlsli:8-523     (`k_samples`, half2 literals)
  disk32.bin    32 x float2  DirectLighting/Emissive/Resampling.hlsli:352-386      (`k_samples`, half2 literals)
  rho_lut.bin  64 x 32 x 16  Assets/LUT/rho.dds (DDS, L16 UNORM volume), read by Common/BSDF.hlsli:279-296

half2 literals are float32 literals narrowed to binary16 (round to nearest even); the .bin files hold them widened back to
float32, the form the kernels and the oracle consume. `--check` compares the committed assets with the reference tree
instead of writing (tests/test_reference_tables.py compares them with an extraction frozen in tests/golden/reference_tables.npz)."""
import os
import re
import struct
import sys
import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OUT = os.path.join(ROOT, "zetaray_b200", "assets")
REF = os.environ.get("ZR_REFERENCE", "/root/reference")
PASS = os.path.join(REF, "Source", "ZetaRenderPass")

HALF2 = re.compile(r"half2\(\s*([-+0-9.eE]+)\s*,\s*([-+0-9.eE]+)\s*\)")


def half2_table(path, begin_marker, count):
    """All half2(a, b) literals of the first `k_samples` initialiser after `begin_marker`."""
    text = open(path).read()
    at = text.index(begin_marker)
    body = text[text.index("{", at):text.index("};", at)]
    vals = HALF2.findall(body)
    if len(vals) != count:
        raise RuntimeError("%s: expected %d half2 literals, found %d" % (path, count, len(vals)))
    a = np.array(vals, dtype=np.float64).astype(np.float32)       # the literal's own type
    return a.astype(np.float16).astype(np.float32)                # half storage, float arithmetic in the shader


def rho_volume(path):
    raw = open(path, "rb").read()
    magic, size, flags, height, width, pitch, depth, mips = struct.unpack_from("<4sIIIIIII", raw, 0)
    pf_size, pf_flags, fourcc, bitcount, rmask = struct.unpack_from("<II4sII", raw, 76)
    if magic != b"DDS " or size != 124:
        raise RuntimeError("%s: not a DDS file" % path)
    if (width, height, depth) != (64, 32, 16) or bitcount != 16 or rmask != 0xffff or fourcc == b"DX10":
        raise RuntimeError("%s: expected a 64 x 32 x 16 L16 volume, got %dx%dx%d %d bit" % (path, width, height, depth, bitcount))
    data = np.frombuffer(raw, dtype="<u2", offset=128)
    if data.size != 64 * 32 * 16:
        raise RuntimeError("%s: unexpected payload size %d" % (path, data.size))
    return data.copy()


def tables():
    return {
        "disk512.bin": half2_table(os.path.join(PASS, "IndirectLighting", "ReSTIR_PT", "SampleSet.hlsli"), "k_samples[SAMPLE_SET_SIZE]", 512),
        "disk32.bin": half2_table(os.path.join(PASS, "DirectLighting", "Emissive", "Resampling.hlsli"), "k_samples[32]", 32),
        "rho_lut.bin": rho_volume(os.path.join(REF, "Assets", "LUT", "rho.dds")),
    }


def main():
    check = "--check" in sys.argv
    bad = 0
    for name, arr in tables().items():
        path = os.path.join(OUT, name)
        if check:
            same = os.path.exists(path) and open(path, "rb").read() == arr.tobytes()
            print("%-12s %s" % (name, "identical to the reference" if same else "DIFFERS"))
            bad += not same
        else:
            os.makedirs(OUT, exist_ok=True)
            arr.tofile(path)
            print("wrote %s (%d bytes)" % (path, arr.nbytes))
    sys.exit(1 if bad else 0)


if __name__ == "__main__":
    main()

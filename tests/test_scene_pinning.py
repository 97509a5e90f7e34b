"""The scene-ingest packers (zetaray_b200/scene.py: materials, emissive triangles, octahedral normals, instance transforms --
the flat-buffer formats on the caller's side of the drop-in boundary, SURVEY A.6 / A.8) are PINNED: bit-exact against the
reference's own constructors (ZetaCore/Core/Material.h, RayTracing/RtCommon.h, Math/OctahedralVector.h, Math/Vector.h,
Math/Color.h), compiled where they lie into oracle/_ref/libref_scene.so (oracle/ref_scene/build.sh).
What those constructors returned for the inputs below is frozen in tests/golden/reference_scene.npz by `reference_outputs`."""
import ctypes as C

import numpy as np
import pytest

from tests.golden_pins import Golden, pin
from zetaray_b200 import scene as zs

STRUCTS = (("MeshInstance", zs.MESH_INSTANCE), ("EmissiveTriangle", zs.EMISSIVE_TRI), ("Material", zs.MATERIAL))


def oct_half_rgb8_inputs():
    rng = np.random.default_rng(0)
    n = rng.normal(size=(30000, 3))
    n /= np.linalg.norm(n, axis=1, keepdims=True)
    n = n.astype(np.float32)
    n[:6] = [[1, 0, 0], [0, 1, 0], [0, 0, 1], [-1, 0, 0], [0, -1, 0], [0, 0, -1]]
    x = np.concatenate([(rng.normal(size=4000) * 10), [0.0, 1.0, 65504.0, 1e-5, 20.0, 0.3]]).astype(np.float32)
    c = rng.random((6000, 3)).astype(np.float32)
    c[:200] = (np.floor(c[:200] * 255) + 0.5) / 255          # values at / next to the .5 ties where the rounding rule shows
    c[200:206] = [[0, 0, 0], [1, 1, 1], [0.5, 0.5, 0.5], [0.3, 0.7, 0.1], [0.8, 0.8, 0.8], [1.0, 0.7759, 0.6167]]
    return n, x, c


def material_inputs():
    """(20 material parameters, double_sided, thin_walled) per case."""
    rng = np.random.default_rng(1)
    cases = []
    for k in range(1500):
        base = rng.random(4); met = rng.random(); rough = rng.random(); ior = 1.0 + 1.49 * rng.random(); tr = rng.random()
        em = rng.random(3) * (rng.random() < 0.5); es = rng.random() * 30; cw = rng.random(); cc = rng.random(3); cr = rng.random()
        cior = 1.0 + 1.49 * rng.random(); ss = rng.random(); td = rng.random() * 3
        if k < 8:       # the defaults and round numbers
            base = np.array([1, 1, 1, 1.0]); rough = [0.3, 0.5, 0.1, 0.0, 1.0, 0.7, 0.25, 0.85][k]; ior = 1.5; cior = 1.6; cc = np.array([0.8] * 3)
        ds, tw = bool(k & 1), bool(k & 2)
        p = np.array(list(base) + [met, rough, ior, tr] + list(em) + [es, cw] + list(cc) + [cr, cior, ss, td], dtype=np.float32)
        cases.append((p, ds, tw))
    return cases


def emissive_inputs():
    rng = np.random.default_rng(2)
    n = 4000
    v0 = rng.normal(size=(n, 3)) * 8
    v1 = v0 + rng.normal(size=(n, 3)) * rng.random((n, 1)) * 3
    v2 = v0 + rng.normal(size=(n, 3)) * rng.random((n, 1)) * 3
    # axis-aligned edges (octahedral fold lines) like the Cornell light quad
    v1[:50] = v0[:50] + np.eye(3)[rng.integers(0, 3, 50)] * 0.5
    v2[:50] = v0[:50] - np.eye(3)[rng.integers(0, 3, 50)] * 0.25
    uv = rng.random((3, n, 2))
    ids = rng.integers(0, 2**32, n, dtype=np.uint64).astype(np.uint32)
    V0, V1, V2 = (x.astype(np.float32) for x in (v0, v1, v2))
    return V0, V1, V2, uv, ids, int(zs.half_bits(20.0))


def instance_inputs():
    """(unit quaternion, scale) per case."""
    rng = np.random.default_rng(3)
    cases = []
    for k in range(2000):
        q = rng.normal(size=4); q /= np.linalg.norm(q)
        s = 0.05 + rng.random(3) * 4
        if k == 0:
            q = np.array([0, 0, 0, 1.0]); s = np.ones(3)
        cases.append((q, s))
    return cases


def reference_outputs(lib):
    """What the reference's constructors and struct layouts give for the inputs above (lib: oracle/_ref/libref_scene.so)."""
    lib.ref_oct32.restype = C.c_uint32
    lib.ref_half.restype = C.c_uint16
    lib.ref_rgb8.restype = C.c_uint32
    out = {}
    sz = (C.c_int * 4)()
    lib.ref_scene_sizes(sz)
    out["sizes"] = np.array(list(sz), dtype=np.int32)
    n, x, c = oct_half_rgb8_inputs()
    out["oct32"] = pin(np.array([lib.ref_oct32(C.c_float(a), C.c_float(b), C.c_float(d)) for a, b, d in n], dtype=np.uint32))
    out["half"] = pin(np.array([lib.ref_half(C.c_float(v)) for v in x], dtype=np.uint16))
    out["rgb8"] = pin(np.array([lib.ref_rgb8(C.c_float(v[0]), C.c_float(v[1]), C.c_float(v[2])) for v in c], dtype=np.uint32))
    cases = material_inputs()
    mats = np.zeros(len(cases), dtype=zs.MATERIAL)
    for k, (p, ds, tw) in enumerate(cases):
        lib.ref_material(p.ctypes.data_as(C.c_void_p), C.c_uint32(int(ds) | (int(tw) << 1)), mats[k:].ctypes.data_as(C.c_void_p))
    out["material"] = pin(mats)
    V0, V1, V2, uv, ids, strength = emissive_inputs()
    tris = np.zeros(len(V0), dtype=zs.EMISSIVE_TRI)
    for k in range(len(V0)):
        vv = np.concatenate([V0[k], V1[k], V2[k]]).astype(np.float32)
        uu = np.concatenate([uv[0][k], uv[1][k], uv[2][k]]).astype(np.float32)
        lib.ref_emissive_triangle(vv.ctypes.data_as(C.c_void_p), uu.ctypes.data_as(C.c_void_p), C.c_uint32(0x9dc6ff), C.c_uint32(zs.INVALID_ID),
                                  C.c_uint16(strength), C.c_uint32(int(ids[k])), 1, tris[k:].ctypes.data_as(C.c_void_p))
    tris["PackedA"] |= 1 << 24       # TriIDPatchedBit: set when the scene patches ID / world position (SceneCore.cpp:199-235); ours are stored patched
    out["emissive_triangle"] = pin(tris)
    cases = instance_inputs()
    rot = np.zeros((len(cases), 4), dtype=np.uint16); sc = np.zeros((len(cases), 3), dtype=np.uint16)
    for k, (q, s) in enumerate(cases):
        q32 = (q / np.linalg.norm(q)).astype(np.float32); s32 = s.astype(np.float32)
        lib.ref_instance_rotation_scale(q32.ctypes.data_as(C.c_void_p), s32.ctypes.data_as(C.c_void_p), rot[k].ctypes.data_as(C.c_void_p),
                                        sc[k].ctypes.data_as(C.c_void_p))
    out["instance_rotation"], out["instance_scale"] = pin(rot), pin(sc)
    from zetaray_b200 import _lib
    names = [f[0] for f in _lib.FrameConstants._fields_]
    out["frame_constants_size"] = np.array(lib.ref_frame_constants_offset(b""), dtype=np.int32)
    out["frame_constants_fields"] = np.array(names)
    out["frame_constants_offsets"] = np.array([lib.ref_frame_constants_offset(f.encode()) for f in names], dtype=np.int32)
    for strct, dt in STRUCTS:
        out[strct + "_fields"] = np.array(dt.names)
        out[strct + "_offsets"] = np.array([lib.ref_struct_offset(strct.encode(), f.encode()) for f in dt.names], dtype=np.int32)
    return out


@pytest.fixture(scope="module")
def ref():
    return Golden("reference_scene.npz")


def test_struct_sizes(ref):
    assert list(ref["sizes"]) == [zs.MATERIAL.itemsize, zs.MESH_INSTANCE.itemsize, zs.EMISSIVE_TRI.itemsize, zs.VERTEX.itemsize] == [32, 64, 48, 28]


def test_oct32_half_rgb8(ref):
    n, x, c = oct_half_rgb8_inputs()
    mine = zs.oct_encode_unorm16(n)
    ref.check("oct32", mine[:, 0].astype(np.uint32) | (mine[:, 1].astype(np.uint32) << 16))
    ref.check("half", np.array([int(zs.half_bits(v)) for v in x], dtype=np.uint16))
    ref.check("rgb8", np.array([zs.rgb8(v) for v in c], dtype=np.uint32))


def test_material_packing(ref):
    mine = [zs.make_material(base_color=tuple(p[0:4]), metallic=p[4], roughness=p[5], ior=p[6], transmission=p[7],
                             emissive_factor=tuple(p[8:11]), emissive_strength=p[11], coat_weight=p[12], coat_color=tuple(p[13:16]),
                             coat_roughness=p[16], coat_ior=p[17], double_sided=ds, thin_walled=tw, subsurface=p[18],
                             transmission_depth=p[19]) for p, ds, tw in material_inputs()]
    ref.check("material", np.frombuffer(b"".join(m.tobytes() for m in mine), dtype=zs.MATERIAL))


def test_emissive_triangle_packing(ref):
    V0, V1, V2, uv, ids, strength = emissive_inputs()
    ref.check("emissive_triangle", zs.emissive_triangles(V0, V1, V2, uv[0], uv[1], uv[2], 0x9dc6ff, strength, ids, True))


def test_instance_rotation_and_scale(ref):
    b = zs.SceneBuilder()
    insts = [b._instance(0, 0, 0, (0, 0, 0), tuple(q), tuple(s)) for q, s in instance_inputs()]
    ref.check("instance_rotation", np.array([inst["Rotation"] for inst in insts], dtype=np.uint16))
    ref.check("instance_scale", np.array([inst["Scale"] for inst in insts], dtype=np.uint16))


def test_frame_constants_layout_matches_the_reference_header(ref):
    """zr_frame_constants (include/zr_abi.h, mirrored by zetaray_b200._lib.FrameConstants) is cbFrameConstants field for field:
    every offset and the size, taken from the reference's own Common/FrameConstants.h compiled by g++."""
    from zetaray_b200 import _lib
    FC = _lib.FrameConstants
    assert int(ref["frame_constants_size"]) == C.sizeof(FC) == 544
    want = dict(zip(ref["frame_constants_fields"].tolist(), ref["frame_constants_offsets"].tolist()))
    names = [f[0] for f in FC._fields_]
    assert len(names) == 52
    for name in names:
        assert want.get(name, -1) >= 0, "the reference has no field " + name
        assert getattr(FC, name).offset == want[name], (name, getattr(FC, name).offset, want[name])


def test_scene_struct_field_offsets(ref):
    for strct, dt in STRUCTS:
        offsets = dict(zip(ref[strct + "_fields"].tolist(), ref[strct + "_offsets"].tolist()))
        for name in dt.names:
            want = offsets.get(name, -1)
            assert want >= 0, (strct, name)
            assert dt.fields[name][1] == want, (strct, name, dt.fields[name][1], want)

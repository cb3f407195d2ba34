"""Mesh ingestion (SURVEY section 8f, row N2): load_obj_with_mtl / load_mtl / load_stl of
ekzhang/rpt src/io.rs:83-149,202-360 through the C ABI, checked against pure-Python restatements of
the same functions on small synthetic files (CPU only: the parsers are host code)."""
import io
import math
import os
import struct
import zipfile

import numpy as np
import pytest

from rpt_b200 import api
from rpt_b200._capi import RptbError

MTL = """# two materials, one edited twice
newmtl red
Kd 0.8 0.1 0.1
Ns 96.078431
Ka 1 1 1
illum 2

newmtl glass
Kd 1 1 1
Ni 1.0
d 0.5
Ns 0

newmtl red
Ni 1.7
d 0.9
"""

OBJ = """# a strip cut into three material runs
mtllib ignored.mtl
v 0 0 0
v 1 0 0
v 1 1 0
v 0 1 0
vn 0 0 1
f 1 2 3
usemtl red
f 1//1 2//1 3//1 4//1
v 2 0 0
v 2 1 0
usemtl red
f -2 -1 3
usemtl glass
vt 0.5 0.5
f 2/1/1 5/1/1 6/1/1
usemtl red
f 2 5 6 3
"""


def mat_tuple(m):
    return (tuple(np.asarray(m.color, dtype=float)), m.index, m.roughness, m.metallic, m.emittance, bool(m.transparent))


def test_load_mtl_restatement_values():
    mats = api.load_mtl(io.BytesIO(MTL.encode()))
    assert set(mats) == {"red", "glass"}
    red, glass = mats["red"], mats["glass"]
    assert np.allclose(red.color, [0.8, 0.1, 0.1])
    assert red.roughness == math.sqrt(math.sqrt(2.0 / (96.078431 + 2.0)))
    assert red.index == 1.7 and not red.transparent          # second `newmtl red` kept editing it; d 0.9 >= 0.8
    assert glass.index == 1.0 + 1e-4 and glass.transparent   # Ni clamped, d 0.5 < 0.8
    assert glass.roughness == 1.0                            # Ns 0 -> (2/2)^(1/4)
    assert red.metallic == 0.0 and red.emittance == 0.0      # Material::default() fields survive


def test_obj_with_mtl_native_matches_restatement():
    objects = api.load_obj_with_mtl(io.BytesIO(OBJ.encode()), io.BytesIO(MTL.encode()), build=False)
    want = api.parse_obj_with_mtl(OBJ.split("\n"), api.load_mtl(io.BytesIO(MTL.encode())))
    # runs: default (1 tri) | red (2 + 1: the repeated `usemtl red` does not cut) | glass (1) | red (2)
    assert [len(o.shape.triangles) for o in objects] == [1, 3, 1, 2]
    assert len(objects) == len(want)
    for o, (m, tris) in zip(objects, want):
        assert mat_tuple(o.mat) == mat_tuple(m)
        assert np.array_equal(o.shape.triangles, tris)        # bit-exact: same strtod / float() values
    assert mat_tuple(objects[0].mat) == mat_tuple(api.Material.default())


def test_obj_with_mtl_errors():
    with pytest.raises(RptbError, match="Could not found `usemtl blue`"):
        api.load_obj_with_mtl(io.BytesIO(b"v 0 0 0\nusemtl blue\n"), io.BytesIO(MTL.encode()))
    with pytest.raises(RptbError, match="before properties were added"):
        api.load_obj_with_mtl(io.BytesIO(b"v 0 0 0\n"), io.BytesIO(b"Kd 1 1 1\n"))
    with pytest.raises(RptbError, match="Invalid vertex index"):
        api.load_obj_with_mtl(io.BytesIO(b"v 0 0 0\nf x 1 1\n"), io.BytesIO(b""))
    with pytest.raises(ValueError):
        api.load_mtl(io.BytesIO(b"Kd 1 1 1\n"))
    assert api.load_obj_with_mtl(io.BytesIO(b"v 0 0 0\n"), io.BytesIO(b"")) == []   # no faces: no objects


def stl_binary(facets, header=b"binary"):
    out = header.ljust(80, b" ") + struct.pack("<I", len(facets))
    for n, a, b, c in facets:
        out += struct.pack("<12f", *n, *a, *b, *c) + b"\x00\x00"
    return out


FACETS = [((0, 0, 1), (0, 0, 0), (1, 0, 0), (0, 1, 0)),
          ((0, 0, 0), (0.1, 0.2, 0.3), (1.5, -2.25, 3), (1e-3, 7, -8)),     # zero normal is kept as stored
          ((0, 2, 0), (1, 1, 1), (2, 1, 1), (1, 1, 2))]                      # and so is a non-unit one


def expected_stl(facets):
    rows = []
    for n, a, b, c in facets:
        f32 = lambda v: [float(np.float32(x)) for x in v]
        rows.append(f32(a) + f32(b) + f32(c) + f32(n) * 3)
    return np.array(rows)


def test_stl_binary():
    tris = api.parse_stl_native(stl_binary(FACETS))
    assert np.array_equal(tris, expected_stl(FACETS))
    # a binary file may start with "solid " (examples/cylinder.stl does): the size rule wins
    assert np.array_equal(api.parse_stl_native(stl_binary(FACETS, b"solid Cylinder_Big")), expected_stl(FACETS))
    assert api.parse_stl_native(stl_binary([])).shape == (0, 18)


def stl_ascii(facets, endsolid=True):
    s = "solid demo\n"
    for n, a, b, c in facets:
        s += "  facet normal %r %r %r\n    outer loop\n" % tuple(float(x) for x in n)
        for v in (a, b, c):
            s += "      vertex %r %r %r\n" % tuple(float(x) for x in v)
        s += "    endloop\n  endfacet\n"
    return (s + ("endsolid demo\n" if endsolid else "")).encode()


def test_stl_ascii():
    want = np.array([[*a, *b, *c, *n, *n, *n] for n, a, b, c in FACETS], dtype=np.float64)  # f64, not via f32
    assert np.array_equal(api.parse_stl_native(stl_ascii(FACETS, endsolid=False)), want)
    assert np.array_equal(api.parse_stl_native(stl_ascii(FACETS, endsolid=True)), want)     # documented deviation
    mesh = api.load_stl(io.BytesIO(stl_ascii(FACETS)))
    assert len(mesh) == 3 and mesh.nodes is not None


def test_stl_errors():
    with pytest.raises(RptbError, match="too short"):
        api.parse_stl_native(b"solid x\n")
    with pytest.raises(RptbError, match="could not determine format"):
        api.parse_stl_native(b"x" * 100)
    with pytest.raises(RptbError, match="expected `facet normal`"):
        api.parse_stl_native(b"solid demo\nfacet 0 0 1\n" + b" " * 20)
    with pytest.raises(RptbError, match="expected `vertex`"):
        api.parse_stl_native(b"solid demo\nfacet normal 0 0 1\nouter loop\nvertex 0 0 0\nvertexx 1 0 0\n")
    truncated = stl_binary(FACETS)[:-10]                       # size rule fails, header is not "solid "
    with pytest.raises(RptbError, match="could not determine format"):
        api.parse_stl_native(truncated)


GOLDEN = os.path.join(os.path.dirname(__file__), "golden")


def test_reference_assets_parse():
    """Inputs of rpt's examples/cylinder.rs and examples/lego.rs: cylinder.stl (364 binary facets), and the
    LEGO .obj/.mtl pair cut at every change of `usemtl`.  tests/golden keeps cylinder.stl whole; of lego.zip
    it keeps the .mtl whole and the first 7102 lines of the 21 MB .obj (up to the group `g 123_124`): four
    material runs, with many repeated `usemtl` of the running material that must not cut."""
    data = open(os.path.join(GOLDEN, "cylinder.stl"), "rb").read()
    tris = api.parse_stl_native(data)
    assert tris.shape == (364, 18) and np.isfinite(tris).all()
    assert np.array_equal(tris[:, 9:12], tris[:, 15:18])
    z = zipfile.ZipFile(os.path.join(GOLDEN, "lego_plane_head.zip"))
    obj = z.read("LEGO.Creator_Plane.obj")
    mtl = z.read("LEGO.Creator_Plane.mtl")
    objects = api.load_obj_with_mtl(io.BytesIO(obj), io.BytesIO(mtl), build=False)
    runs, last = 0, None
    open_faces = False
    for line in obj.split(b"\n"):
        tok = line.split()
        if not tok:
            continue
        if tok[0] == b"f":
            open_faces = True
        elif tok[0] == b"usemtl" and tok[1] != last:
            runs += open_faces
            open_faces, last = False, tok[1]
    runs += open_faces
    assert len(objects) == runs > 1
    assert [len(o.shape.triangles) for o in objects] == [2, 3696, 416, 64]
    names = api.load_mtl(io.BytesIO(mtl.decode("latin-1").encode()))
    have = {mat_tuple(m) for m in names.values()}
    assert all(mat_tuple(o.mat) in have for o in objects)
    assert sum(len(o.shape.triangles) for o in objects) == len(api.parse_obj_native(obj))

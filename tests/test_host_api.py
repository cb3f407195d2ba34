"""CPU tests of the host mirror of rpt's API (rpt_b200/api.py): builder semantics,
transform composition, camera construction, OBJ parsing, scene flattening."""
import io
import math

import numpy as np
import pytest

from rpt_b200 import api, scenes
from rpt_b200 import _capi as capi
from rpt_b200.distributed import tile_owner


def test_renderer_defaults_and_builder():
    r = api.Renderer(api.Scene(), api.Camera.default())
    assert (r._width, r._height, r._exposure_value, r._max_bounces, r._num_samples) == (800, 600, 0.0, 0, 1)
    assert r._filter.radius == 0  # src/renderer.rs:46-57
    r2 = r.width(10).height(20).max_bounces(3).num_samples(7).exposure_value(1.5).filter(api.Filter.Box(2))
    assert r2 is r and (r._width, r._height, r._max_bounces, r._num_samples) == (10, 20, 3, 7)
    p = r.params(5, first_sample=11, shard_index=1, shard_count=4)
    assert (p.width, p.height, p.iterations, p.max_bounces, p.first_sample, p.shard_index, p.shard_count) == \
        (10, 20, 5, 3, 11, 1, 4)


def test_camera_default_look_at_focus():
    c = api.Camera.default()
    np.testing.assert_array_equal(c.eye, [0, 0, 10])
    np.testing.assert_array_equal(c.direction, [0, 0, -1])
    assert c.fov == math.pi / 6 and c.aperture == 0 and c.focal_distance == 0
    c = api.Camera.look_at(api.vec3(-2.5, 4.0, 6.5), api.vec3(0, -0.25, 0), api.vec3(0, 1, 0), math.pi / 4)
    assert abs(np.linalg.norm(c.direction) - 1) < 1e-15 and abs(np.linalg.norm(c.up) - 1) < 1e-15
    assert abs(np.dot(c.direction, c.up)) < 1e-15  # up re-orthogonalised (src/camera.rs:45)
    c2 = c.focus(api.vec3(0, 0, 0), 0.1)
    assert c2 is c and c.aperture == 0.1
    np.testing.assert_allclose(c.focal_distance, np.dot(-c.eye, c.direction))


def test_transform_chaining_composes_left_to_right():
    """cube().scale(s).rotate_y(a).translate(t) == T * R * S (src/shape.rs:234-284)."""
    s, a, t = api.vec3(165, 330, 165), 2 * math.pi * (-253 / 360), api.vec3(368, 165, 351)
    tr = api.cube().scale(s).rotate_y(a).translate(t)
    assert isinstance(tr, api.Transformed) and isinstance(tr.shape, api.Cube)
    S = np.diag([165, 330, 165, 1.0])
    c, sn = math.cos(a), math.sin(a)
    R = np.array([[c, 0, sn, 0], [0, 1, 0, 0], [-sn, 0, c, 0], [0, 0, 0, 1.0]])
    T = np.eye(4)
    T[:3, 3] = t
    np.testing.assert_allclose(tr.matrix, T @ R @ S, atol=1e-12)
    # a point on the cube's top face centre goes to (368, 330, 351)
    np.testing.assert_allclose(tr.matrix @ np.array([0, 0.5, 0, 1.0]), [368, 330, 351, 1], atol=1e-9)
    # rotate about an arbitrary axis normalises the axis (glm::rotate)
    r1 = api.sphere().rotate(0.3, api.vec3(0, 2, 0)).matrix
    r2 = api.sphere().rotate_y(0.3).matrix
    np.testing.assert_allclose(r1, r2, atol=1e-15)


def test_materials_constructors():
    d = api.Material.diffuse(api.vec3(1, 1, 1))
    assert (d.index, d.roughness, d.metallic, d.emittance, d.transparent) == (1.5, 1.0, 0.0, 0.0, False)
    c = api.Material.clear(1.33, 0.01)
    assert c.transparent and c.index == 1.33 and (c.color == 1).all()
    m = api.Material.metallic_(api.vec3(1, 0, 0), 0.4)
    assert m.metallic == 1.0 and m.index == 1.5
    li = api.Material.light(api.vec3(1, 1, 1), 40.0)
    assert li.index == 1.0 and li.roughness == 1.0 and li.emittance == 40.0
    df = api.Material.default()
    np.testing.assert_allclose(df.color, api.hex_color(0xFF0000))
    assert df.roughness == 0.5


def test_parse_obj_fan_normals_negative_indices():
    obj = """
# comment
v 0 0 0
v 1 0 0
v 1 1 0
v 0 1 0
vn 0 0 1
vt 0.5 0.5
usemtl foo
f 1 2 3 4
f 1//1 2//1 3//1
f -4 -3 -2
"""
    tris = api.parse_obj(io.StringIO(obj))
    assert tris.shape == (4, 18)  # quad -> 2 (fan), + 2
    np.testing.assert_array_equal(tris[0, :9], [0, 0, 0, 1, 0, 0, 1, 1, 0])
    np.testing.assert_array_equal(tris[1, :9], [0, 0, 0, 1, 1, 0, 0, 1, 0])
    np.testing.assert_array_equal(tris[2, 9:], [0, 0, 1] * 3)  # explicit normals
    np.testing.assert_array_equal(tris[3, :9], tris[0, :9])  # negative indices
    np.testing.assert_allclose(tris[0, 9:12], [0, 0, 1])  # inferred normal


def test_teapot_asset_is_the_reference_mesh():
    t = scenes.teapot_triangles()
    assert t.shape == (2256, 18)  # SURVEY [probe]: teapot.obj has 2256 triangles
    assert np.isfinite(t).all()


def test_flatten_cornell():
    cfg = scenes.cornell_scene()
    flat = api.FlatScene(cfg.scene)
    d = flat.desc
    assert (d.nobjects, d.nlights, d.nmeshes) == (7, 1, 6)
    kinds = [flat.objects[i].kind for i in range(7)]
    assert kinds == [capi.SHAPE_MESH] * 5 + [capi.SHAPE_CUBE] * 2
    assert [flat.objects[i].has_transform for i in range(7)] == [0] * 5 + [1] * 2
    assert flat.lights[0].kind == capi.LIGHT_OBJECT and flat.lights[0].object.kind == capi.SHAPE_MESH
    lm = flat.materials[flat.lights[0].object.material]
    assert lm.emittance == 100.0
    assert flat.meshes[0].ntris == 2 and flat.meshes[0].nnodes == 1
    # column-major transform: translation in elements 12..14
    assert list(flat.objects[5].transform)[12:15] == [368.0, 165.0, 351.0]
    assert flat.host_bytes() > 0


def test_tile_owner_partition():
    for (w, h, n) in [(800, 800, 8), (37, 19, 3), (16, 8, 2), (1, 1, 4)]:
        own = tile_owner(w, h, n)
        assert own.shape == (h, w) and own.min() >= 0 and own.max() < n
        tiles_x = (w + 15) // 16
        assert own[0, 0] == 0
        if w > 16:
            assert own[0, 16] == 1 % n
        if h > 8:
            assert own[8, 0] == tiles_x % n
    own = tile_owner(1920, 1080, 8)
    frac = np.bincount(own.ravel(), minlength=8) / own.size
    assert np.abs(frac - 1 / 8).max() < 0.01  # interleaving balances the shards


def test_pegasus_proxy_is_the_reference_mesh_subdivided():
    """SURVEY 8(d): the dragon stand-in is examples/pegasus.zip (100 138 triangles) subdivided 1 -> 4 -> 2."""
    v, n, f = scenes.pegasus_indexed()
    assert v.shape == (50059, 3) and n.shape == (50059, 3) and f.shape == (100138, 3)
    t0 = scenes.pegasus_proxy(0)
    assert t0.shape == (100138, 18)
    assert abs(t0[:, [1, 4, 7]].min() * 3.4 + 1.0) < 1e-9  # rests on the plane y = -1 after scale 3.4
    ext = t0[:, 0:9].reshape(-1, 3).max(0) - t0[:, 0:9].reshape(-1, 3).min(0)
    assert abs(ext.max() - 0.7) < 1e-12  # the G3D dragon.obj's longest dimension
    t1v, t1n, t1f = scenes.subdivide4(*[a.copy() for a in (v, n, f)])
    assert t1f.shape == (4 * 100138, 3) and len(t1v) == 50059 + 150203  # one new vertex per edge: still an indexed, closed mesh
    ed = np.sort(np.concatenate([t1f[:, [0, 1]], t1f[:, [1, 2]], t1f[:, [2, 0]]]), axis=1)
    _, cnt = np.unique(ed[:, 0] * len(t1v) + ed[:, 1], return_counts=True)
    assert (cnt == 2).mean() > 0.9999  # pegasus.obj itself has 4 non-manifold edges
    # orientation and area survive: face normals of the children agree with the parent's
    p = v[f]
    pn = np.cross(p[:, 1] - p[:, 0], p[:, 2] - p[:, 0])
    c = t1v[t1f].reshape(-1, 4, 3, 3)
    cn = np.cross(c[:, :, 1] - c[:, :, 0], c[:, :, 2] - c[:, :, 0])
    assert ((cn * pn[:, None, :]).sum(2) > 0).mean() > 0.995
    t2 = scenes.subdivide2(t1v, t1n, t1f)
    assert t2.shape == (801104, 18) and np.isfinite(t2).all()
    a2 = 0.5 * np.linalg.norm(np.cross(t2[:, 3:6] - t2[:, 0:3], t2[:, 6:9] - t2[:, 0:3]), axis=1)
    a1 = 0.5 * np.linalg.norm(np.cross(c[:, :, 1] - c[:, :, 0], c[:, :, 2] - c[:, :, 0]), axis=2).reshape(-1)
    assert np.allclose(a2.reshape(-1, 2).sum(1), a1, rtol=1e-9, atol=1e-18)  # 1 -> 2 cuts, it does not move anything


def test_dragon_knot_is_closed_and_outward():
    tris = scenes.knot_proxy(120, 30)
    assert tris.shape == (120 * 30 * 2, 18)
    v1, v2, v3 = tris[:, 0:3], tris[:, 3:6], tris[:, 6:9]
    fn = np.cross(v2 - v1, v3 - v1)
    nn = tris[:, 9:12]
    assert ((fn * nn).sum(1) > 0).mean() > 0.999  # vertex normals agree with the winding
    # outward: signed volume positive
    vol = (v1 * np.cross(v2, v3)).sum(1).sum() / 6.0
    assert vol > 0
    assert abs(tris[:, [1, 4, 7]].min() * 3.4 + 1.0) < 1e-9  # rests on the plane y = -1 after scale 3.4


def test_native_obj_parser_matches_the_python_mirror():
    """rptb_parse_obj (C++, what load_obj uses) == parse_obj (Python mirror of src/io.rs:27-73)."""
    obj = "\n".join([
        "# comment", "v 0 0 0", "v 1 0 0", "v 1 1 0", "v 0 1 0", "v 0.5 0.5 1e0", "vn 0 0 1", "vn 0 1 0", "vt 0.5 0.5",
        "mtllib x.mtl", "usemtl foo", "f 1 2 3 4", "f 1//1 2//1 3//2", "f -5 -4 -3", "f 1/1/1 2/1/1 5/1/2", "f 1/1 2/1 3/1",
        "  f   2 3 5   ", "g group", "s off", ""])
    a = api.parse_obj(io.StringIO(obj))
    b = api.parse_obj_native(obj)
    assert a.shape == b.shape == (7, 18)
    np.testing.assert_array_equal(a, b)
    # the committed teapot triangles survive an OBJ round trip through the native parser bit for bit
    t = scenes.teapot_triangles()[:300]
    lines = []
    for i, tri in enumerate(t):
        lines += ["v %r %r %r" % tuple(float(x) for x in tri[3 * k:3 * k + 3]) for k in range(3)]
        lines += ["vn %r %r %r" % tuple(float(x) for x in tri[9 + 3 * k:12 + 3 * k]) for k in range(3)]
        lines.append("f %d//%d %d//%d %d//%d" % tuple(3 * i + 1 + k // 2 for k in range(6)))
    np.testing.assert_array_equal(api.parse_obj_native("\n".join(lines)), t)
    assert api.parse_obj_native("").shape == (0, 18)
    for bad in ("v 1 2", "f 1 2 3", "v 0 0 0\nv 1 0 0\nv 0 1 0\nf 1 2 9", "v 0 0 0\nf x y z"):
        with pytest.raises(capi.RptbError):
            api.parse_obj_native(bad)


def test_load_obj_builds_the_mesh(tmp_path):
    p = tmp_path / "quad.obj"
    p.write_text("v 0 0 0\nv 1 0 0\nv 1 1 0\nv 0 1 0\nf 1 2 3 4\n")
    m = api.load_obj(str(p))
    assert len(m) == 2 and len(m.nodes) == 1 and list(m.refs) == [0, 1]


def test_cpp_host_mirror_examples_compile_and_fail_loudly_without_a_gpu(tmp_path):
    """include/rpt.hpp is header-only over the C ABI: both examples build with plain g++ against the library.
    On a box without a GPU they must stop with the library's NO_DEVICE message (no CPU fallback); with one,
    the -m gpu tests compare their images with the Python host's."""
    import os
    import subprocess
    from rpt_b200 import _capi as capi

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    libdir = os.path.join(root, "rpt_b200", "lib")
    for name in ("sphere", "fractal_spheres"):
        exe = str(tmp_path / name)
        subprocess.check_call(["g++", "-std=c++17", "-O1", "-Wall", "-Werror", "-o", exe, os.path.join(root, "examples", name + ".cpp"),
                               "-L" + libdir, "-lrpt_b200", "-Wl,-rpath," + libdir])
        if capi.lib().rptb_device_count() <= 0:
            p = subprocess.run([exe, str(tmp_path / "out.ppm"), "small"], capture_output=True, text=True)
            assert p.returncode != 0 and "no CUDA device" in p.stderr


def test_flatten_kdtree_of_shapes_shares_meshes_and_keeps_child_order():
    tea = api.Mesh(scenes.teapot_triangles(), build=False)
    kids = [tea.scale(api.vec3(0.5, 0.5, 0.5)).translate(api.vec3(float(i), 0.0, 0.0)) for i in range(20)] + [api.sphere(), api.monomial_surface(2.0, 4.0)]
    scene = api.Scene()
    scene.add(api.Object(api.KdTree(kids).rotate_y(0.3)).material(api.Material.diffuse(api.hex_color(0x808080))))
    scene.add(api.Object(tea))
    flat = api.FlatScene(scene)
    assert flat.desc.nmeshes == 1 and flat.desc.ngroups == 1 and flat.desc.nobjects == 2
    g = flat.groups[0]
    assert g.nchildren == 22 and not g.nodes                       # the library builds the tree
    assert [g.children[i].kind for i in (0, 19, 20, 21)] == [3, 3, 0, 4]
    assert g.children[5].has_transform == 1 and g.children[5].transform[12] == 5.0 and g.children[5].transform[0] == 0.5
    assert g.children[20].has_transform == 0
    assert (g.children[21].monomial_height, g.children[21].monomial_exp) == (2.0, 4.0)
    assert flat.objects[0].kind == 5 and flat.objects[0].has_transform == 1 and flat.objects[0].mesh == 0
    assert flat.objects[1].kind == 3 and flat.objects[1].mesh == 0   # the same mesh record as the instances
    assert flat.host_bytes() > 22 * 184


def test_bench_arms_share_one_config_and_count_real_cores():
    """bench.py: the CPU arm's `config` is the GPU arm's (the driver compares them), the core count honours the cgroup
    quota, and the bytes model adds the BVH counters."""
    import importlib.util
    import os
    spec = importlib.util.spec_from_file_location("bench", os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    cfg = bench.workload("cornell")
    a, b = bench.config_dict(cfg, 1), bench.config_dict(bench.workload("cornell"), 1)
    assert a == b and a["spp_per_gpu"] == 512 and a["width"] == 800 and a["max_bounces"] == 6
    assert bench.config_dict(cfg, 8)["spp_total"] == 4096
    used, aff, quota = bench.host_cores()
    assert 1 <= used <= aff and (quota is None or used <= max(1, int(quota + 0.5)))
    st = {k: 0 for k in bench.KEYS}
    st.update(segments=10, bvh_node_visits=3, bvh_tri_tests=2, object_tests=4)
    assert bench.algorithmic_bytes(st, 5) == 64 * 4 + 64 * 3 + 52 * 2 + 32 * 10 + 12 * 5


@pytest.mark.parametrize("argv", [["--steps", "0"], ["--impl", "reference", "--dump-outputs", "out"]])
def test_bench_rejects_arguments_it_cannot_honour(argv):
    """No timed step would leave nothing to time or dump, and the reference arm keeps no image to dump."""
    import os
    import subprocess
    import sys
    bench = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "bench.py")
    p = subprocess.run([sys.executable, bench] + argv, capture_output=True, text=True)
    assert p.returncode == 2 and "error:" in p.stderr and p.stdout == ""

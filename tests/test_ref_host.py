"""The product's host pipeline against THE REFERENCE'S OWN HOST CODE.

oracle/ref_host_shim.cpp compiles P3/P4/P5 main.cpp and lib/hdrloader.cpp of the reference (GL/GLUT: no-op stand-ins that
capture uploads; glm: the subset main.cpp uses, oracle/ref_stubs/) and
  * runs the reference's main() -- its shipped scene -- up to glutMainLoop() and captures what it would upload to the GPU;
  * exposes readObj / buildBVH / buildBVHwithSAH / calculateHdrCache for other inputs.
The product (ezrt_b200/csrc/host_scene.cpp, SURVEY.md 8f rows) must produce the same BYTES.

What the reference computed is stored (tests/reference_golden.py): crc32s of its results on the inputs below, and samples of
its shipped data files where they are too large to keep (tests/golden/make_golden_reference.py regenerates both);
tests/golden/refhost.npz carries the reference-computed sampling cache of the synthetic environment and crc32s of
reference-built scenes."""
import os
import zlib

import numpy as np
import pytest

from ezrt_b200 import api, scenes
from tests import reference_golden as rg

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "refhost.npz")


def same_bytes(a, b):
    a = np.ascontiguousarray(a, np.float32); b = np.ascontiguousarray(b, np.float32)
    return a.shape == b.shape and a.tobytes() == b.tobytes()


def crc(a):
    return zlib.crc32(np.ascontiguousarray(a).tobytes())


def p5_main_meshes(directory):
    """P5/main.cpp:773-788 (the teapot is the stored patch of P5's teapot.obj): [(obj path, Material, trans16, smooth)]"""
    m1 = api.Material(roughness=0.5, specular=1.0, metallic=1.0, clearcoat=1.0, clearcoatGloss=0.0, baseColor=(1, 0.73, 0.25))
    m2 = api.Material(roughness=0.01, metallic=0.1, specular=1.0, clearcoat=1.0, clearcoatGloss=0.0, baseColor=(1, 1, 1))
    return [(rg.write_model(directory, "p5_teapot_patch"), m1, api.transform_matrix((0, 0, 0), (0, -0.5, 0), (0.75, 0.75, 0.75)), True),
            (rg.write_model(directory, "p5_quad"), m2, api.transform_matrix((0, 0, 0), (0, -0.5, 0), (13000.0, 0.01, 13000.0)), False)]


def p4_main_meshes(directory):
    """P4/main.cpp:689-743: one golden teapot (the stored patch of the teapot.obj P4 and P5 ship)"""
    m = api.Material(baseColor=(0.75, 0.7, 0.15), roughness=0.15, metallic=1.0, clearcoat=1.0, subsurface=1.0)
    return [(rg.write_model(directory, "p5_teapot_patch"), m, api.transform_matrix((0, 0, 0), (0, -0.4, 0), (1.75, 1.75, 1.75)), True)]


P3_DEFAULTS = dict(specular=0.0, roughness=0.0, sheenTint=0.0, clearcoatGloss=0.0)


def p3_main_meshes(directory):
    """P3/main.cpp:688-715 (Stanford bunny + floor + emissive sphere, the whole files P3 ships)"""
    d = P3_DEFAULTS
    return [(rg.write_model(directory, "p3_bunny"), api.Material(baseColor=(1, 1, 1), **d), api.transform_matrix((0, 0, 0), (0.3, -1.6, 0), (1.5, 1.5, 1.5)), True),
            (rg.write_model(directory, "p3_quad"), api.Material(baseColor=(0.725, 0.71, 0.68), **d),
             api.transform_matrix((0, 0, 0), (0, -1.4, 0), (18.83, 0.01, 18.83)), False),
            (rg.write_model(directory, "p3_sphere"), api.Material(baseColor=(1, 1, 1), emissive=(30, 20, 10), **d),
             api.transform_matrix((0, 0, 0), (0.0, 0.9, 0.0), (1, 1, 1)), False)]


def build(meshes, leaf_n, builder):
    tl = api.TriangleList()
    for path, m, t, s in meshes:
        tl.read_obj(path, m, t, s)
    return tl.build_bvh(leaf_n, builder)


def test_reference_main_uploads_are_reproduced_byte_for_byte(tmp_path):
    """P5's main(): its scene set-up (materials, transforms, readObj, buildBVHwithSAH with 8 triangles a leaf) on a patch of
    its teapot, HDRLoader and calculateHdrCache on scanlines of its chinese_garden_2k.hdr"""
    g = rg.load()
    meshes = p5_main_meshes(tmp_path)
    for builder in (api.BVH_SAH_LITERAL, api.BVH_SAH_FAST):
        tris, nodes = build(meshes, 8, builder)
        assert [crc(tris), crc(nodes)] == [int(c) for c in g["p5_main_scene_crc"]], "texture buffers, builder %d" % builder
    hdr = api.hdr_load(rg.hdr_rows_path(5))
    assert list(hdr.shape) == list(g["hdr_rows5_shape"]) and crc(hdr) == int(g["hdr_rows5_crc"])
    assert crc(api.hdr_cache(hdr)) == int(g["p5_cache_crc"]), "calculateHdrCache"


def test_reference_p4_main_uploads_are_reproduced_byte_for_byte(tmp_path):
    """P4/main.cpp:689-743: golden teapot (a patch of it), SAH tree, scanlines of its 4096x2048 map"""
    g = rg.load()
    tris, nodes = build(p4_main_meshes(tmp_path), 8, api.BVH_SAH_FAST)
    assert [crc(tris), crc(nodes)] == [int(c) for c in g["p4_main_scene_crc"]]
    hdr = api.hdr_load(rg.hdr_rows_path(4))
    assert list(hdr.shape) == list(g["hdr_rows4_shape"]) and crc(hdr) == int(g["hdr_rows4_crc"])


def test_reference_p3_main_uploads_equal_the_committed_p3_scene(tmp_path):
    """P3/main.cpp:688-715 (Stanford bunny + floor + emissive sphere).  Its main() opens ./HDR/sunset.hdr, which the
    reference does not ship: it was run in a directory whose HDR/sunset.hdr points at the map P3 does ship.
    tests/golden/p3_scene.npz (the scene the golden frames are rendered from) holds the same geometry and tree;
    only the Disney parameters differ, which P3's Material defaults to 0 (P3/main.cpp:28-43) and its shader never reads."""
    r = rg.load()
    r_tris_crc, r_nodes_crc, r_tris24_crc = (int(c) for c in r["p3_main_crc"])
    g = np.load(os.path.join(os.path.dirname(GOLDEN), "p3_scene.npz"))
    assert crc(np.ascontiguousarray(g["nodes"], np.float32)) == r_nodes_crc
    assert crc(np.ascontiguousarray(g["tris"][:, :24], np.float32)) == r_tris24_crc  # positions, normals, emissive, baseColor
    tris, nodes = build(p3_main_meshes(tmp_path), 8, api.BVH_SAH_LITERAL)
    assert [crc(tris), crc(nodes)] == [r_tris_crc, r_nodes_crc]
    hdr = api.hdr_load(rg.hdr_rows_path(3))
    assert list(hdr.shape) == list(r["hdr_rows3_shape"]) and crc(hdr) == int(r["hdr_rows3_crc"])


def _write(tmp_path, name, text):
    p = tmp_path / name
    p.write_text(text)
    return str(p)


def synthetic_meshes(tmp_path, leaf_n):
    """five meshes with random poses and materials (seeded by leaf_n): [(obj path, Material, trans16, smooth)] and the
    rotate / translate / scale of each transform"""
    blob = _write(tmp_path, "blob.obj", scenes.blob_obj(3, 11))
    sphere = _write(tmp_path, "sphere.obj", scenes.sphere_obj(2))
    box = _write(tmp_path, "box.obj", scenes.box_obj())
    rng = np.random.default_rng(leaf_n)
    meshes, poses = [], []
    for path, smooth in ((blob, True), (sphere, False), (box, False), (blob, False), (sphere, True)):
        rot, tr, sc = rng.uniform(-180, 180, 3), rng.uniform(-2, 2, 3), rng.uniform(0.2, 3, 3)
        mat = api.Material(baseColor=tuple(rng.uniform(0, 1, 3)), emissive=tuple(rng.uniform(0, 5, 3)), roughness=float(rng.uniform()),
                           metallic=float(rng.uniform()), sheen=float(rng.uniform()), clearcoat=float(rng.uniform()))
        meshes.append((path, mat, api.transform_matrix(tuple(rot), tuple(tr), tuple(sc)), smooth))
        poses.append((rot, tr, sc))
    return meshes, poses


@pytest.mark.parametrize("leaf_n", [1, 4, 8, 13])
def test_builders_equal_reference_functions_on_synthetic_meshes(tmp_path, leaf_n):
    g = rg.load()
    meshes, _ = synthetic_meshes(tmp_path, leaf_n)
    # same restatement of glm on both sides (see glm.hpp)
    assert [crc(t) for _, _, t, _ in meshes] == [int(c) for c in g["transforms_leaf%d" % leaf_n]]
    want = [int(c) for c in g["builders_leaf%d" % leaf_n]]  # tris, nodes of the SAH builder; tris, nodes of the median builder
    for sah, builders in ((True, (api.BVH_SAH_LITERAL, api.BVH_SAH_FAST)), (False, (api.BVH_MEDIAN,))):
        for b in builders:
            tris, nodes = build(meshes, leaf_n, b)
            assert [crc(tris), crc(nodes)] == (want[:2] if sah else want[2:]), (sah, b)


@pytest.mark.parametrize("w,h", [(128, 64), (64, 32), (96, 40), (16, 8)])
def test_hdr_cache_equals_reference_function(w, h):
    hdr = scenes.synth_hdr(w, h)
    assert crc(api.hdr_cache(hdr)) == int(rg.load()["hdr_cache_%dx%d" % (w, h)])


def test_golden_is_current():
    """refhost.npz's cache is what the reference's calculateHdrCache computed at the last regeneration of reference.npz"""
    g = np.load(GOLDEN)
    assert crc(np.ascontiguousarray(g["cache_128x64"], np.float32)) == int(rg.load()["hdr_cache_128x64"])


def test_hdr_cache_equals_reference_computed_golden():
    """runs everywhere: the cache the REFERENCE's calculateHdrCache computed for the synthetic environment"""
    g = np.load(GOLDEN)
    hdr = scenes.synth_hdr(128, 64)
    assert crc(hdr) == int(g["hdr_crc_128x64"])
    assert same_bytes(api.hdr_cache(hdr), g["cache_128x64"])


def test_synthetic_scenes_equal_reference_built_golden(bunny_scene, grid_scene):
    """runs everywhere: crc32 of the arrays the REFERENCE's readObj + buildBVHwithSAH built from the same OBJ text"""
    g = np.load(GOLDEN)
    for name, sc in (("bunny", bunny_scene), ("grid", grid_scene)):
        tris, nodes = sc[0], sc[1]
        assert (crc(tris), crc(nodes)) == (int(g[name + "_crc_tris"]), int(g[name + "_crc_nodes"])), name


FACE_FORM_MATERIAL = dict(baseColor=(0.3, 0.5, 0.7))
FACE_FORM_TRANSFORM = ((10, 20, 30), (0.1, -0.2, 0.3), (1.5, 0.5, 1.0))


def face_forms_obj(form):
    base = scenes.blob_obj(2, 5).splitlines()
    rng = np.random.default_rng(len(form))
    out = ["# a comment", "", "vt 0.5 0.5", "vn 0 1 0"]
    for ln in base:
        if ln.startswith("f "):
            ids = ln.split()[1:]
            if form == "v":
                tok = ids
            elif form == "v/vt":
                tok = ["%s/1" % i for i in ids]
            elif form == "v/vt/vn":
                tok = ["%s/1/1" % i for i in ids]
            else:
                tok = ["%s//1" % i for i in ids]
            out.append("f " + " ".join(tok) + ("  " if rng.uniform() < 0.2 else ""))
        else:
            out.append(ln)
    return "\n".join(out) + "\n"


@pytest.mark.parametrize("form", ["v", "v/vt", "v/vt/vn"])
def test_read_obj_face_forms_equal_reference(tmp_path, form):
    """the three `f` forms the reference's parser distinguishes by counting slashes (P5/main.cpp:306-333), among vt / vn /
    comment / blank lines and trailing spaces -- same triangles and tree as the reference's own parser.  (`v//vn` makes the
    reference read uninitialised indices -- it crashes there; the product reads the leading integer of every token, see
    test_read_obj_tolerates_the_form_the_reference_cannot_parse.)"""
    path = _write(tmp_path, "forms.obj", face_forms_obj(form))
    mat = api.Material(**FACE_FORM_MATERIAL)
    trans = api.transform_matrix(*FACE_FORM_TRANSFORM)
    want = [int(c) for c in rg.load()["face_form_" + form.replace("/", "_")]]  # tris, nodes flat; tris, nodes smooth
    for smooth in (False, True):
        tris, nodes = build([(path, mat, trans, smooth)], 8, api.BVH_SAH_FAST)
        assert [crc(tris), crc(nodes)] == want[2 * smooth:2 * smooth + 2], (form, smooth)


def test_read_obj_tolerates_the_form_the_reference_cannot_parse():
    plain = "v 0 0 0\nv 1 0 0\nv 0 1 0\nv 0 0 1\nf 1 2 3\nf 1 3 4\n"
    vn = "v 0 0 0\nv 1 0 0\nv 0 1 0\nv 0 0 1\nvn 0 0 1\nf 1//1 2//1 3//1\nf 1//1 3//1 4//1\n"
    out = []
    for text in (plain, vn):
        tl = api.TriangleList()
        tl.read_obj_text(text, api.Material(), api.transform_matrix(), False)
        out.append(tl.build_bvh(8, api.BVH_SAH_LITERAL))
    assert same_bytes(out[0][0], out[1][0]) and same_bytes(out[0][1], out[1][1])

"""CPU tests of the host scene pipeline (readObj / buildBVHwithSAH / encode / HDR / camera) and
of the oracle against the committed golden fixtures."""
import os
import zlib

import numpy as np
import pytest

from ezrt_b200 import api, scenes
from tests import reference_golden as rg

HERE = os.path.dirname(os.path.abspath(__file__))


def crc(a):
    return zlib.crc32(np.ascontiguousarray(a).tobytes())


@pytest.fixture(scope="module")
def golden_p3():
    return np.load(os.path.join(HERE, "golden", "p3_scene.npz"))


@pytest.fixture(scope="module")
def golden_synth():
    return np.load(os.path.join(HERE, "golden", "synth.npz"))


def check_bvh_invariants(tris, nodes, leaf_n=8):
    """SURVEY.md 4: every triangle in exactly one leaf, leaf n <= 8, children inside parent, node 0 dummy, root 1."""
    n_tris = tris.shape[0]
    assert list(nodes[0, [0, 1, 3]]) == [255, 128, 30]  # testNode, P5/main.cpp:830-835
    covered = np.zeros(n_tris, np.int32)
    seen = np.zeros(nodes.shape[0], np.int32)
    stack = [(1, 1)]
    depth_max = 0
    pos = tris[:, :9].reshape(n_tris, 3, 3)
    while stack:
        i, depth = stack.pop()
        seen[i] += 1
        depth_max = max(depth_max, depth)
        left, right, n, index = int(nodes[i, 0]), int(nodes[i, 1]), int(nodes[i, 3]), int(nodes[i, 4])
        AA, BB = nodes[i, 6:9], nodes[i, 9:12]
        if n > 0:
            assert n <= leaf_n and left == 0 and right == 0
            covered[index:index + n] += 1
            p = pos[index:index + n].reshape(-1, 3)
            assert (p.min(axis=0) == AA).all() and (p.max(axis=0) == BB).all()  # exact box of its triangles
        else:
            assert left > 0 and right > 0
            for c in (left, right):
                assert (nodes[c, 6:9] >= AA).all() and (nodes[c, 9:12] <= BB).all()
            assert left == i + 1  # pre-order push_back numbering
            stack.append((right, depth + 1))
            stack.append((left, depth + 1))
    assert (covered == 1).all()
    assert (seen[1:] == 1).all()
    return depth_max


def test_synthetic_scene_arrays_are_reproducible(golden_synth, bunny_scene, grid_scene):
    tris, nodes, eye, cam = bunny_scene
    assert [tris.shape[0], nodes.shape[0]] == list(golden_synth["bunny_shape"])
    assert crc(tris) == int(golden_synth["bunny_crc_tris"]) and crc(nodes) == int(golden_synth["bunny_crc_nodes"])
    tris, nodes, eye, cam = grid_scene
    assert crc(tris) == int(golden_synth["grid_crc_tris"]) and crc(nodes) == int(golden_synth["grid_crc_nodes"])


def test_bvh_invariants(bunny_scene, grid_scene):
    tris, nodes, _, _ = bunny_scene
    assert tris.shape[0] == 5120 + 12 + 320
    d = check_bvh_invariants(tris, nodes)
    assert 10 <= d <= 40
    assert 0.25 < nodes.shape[0] / tris.shape[0] < 0.45  # ~0.35 x triangles (SURVEY.md 4)
    tris, nodes, _, _ = grid_scene
    check_bvh_invariants(tris, nodes)


def test_fast_builder_equals_literal_builder():
    """EZRT_BVH_SAH_FAST must produce the tree buildBVHwithSAH as written (P5/main.cpp:458-589) produces."""
    for fn in (lambda b: scenes.s_bunny(b), lambda b: scenes.s_grid(2, 1, 1, b)):
        t0, n0, _, _ = fn(api.BVH_SAH_FAST)
        t1, n1, _, _ = fn(api.BVH_SAH_LITERAL)
        assert np.array_equal(t0, t1) and np.array_equal(n0, n1)


def test_std_sort_known_answer():
    """The reference's builders sort with order-only comparators (P5/main.cpp:403-413, :560-568): the order of equal keys is the
    C++ library's.  The goldens were made with libstdc++; the library reports whether this host's std::sort is the same."""
    assert api.host_sort_is_reference()


def test_sah_sentinel_quirk_falls_back_to_median_on_axis0():
    """cost >= INF=114514 disables SAH: split = (l+r)/2 on axis 0 (P5/main.cpp:20, :493-495, :569)."""
    tl = api.TriangleList()
    m = api.Material()
    # 64 huge triangles: every area*count exceeds 114514
    rng = np.random.default_rng(3)
    t = np.zeros((64, 36), np.float32)
    t[:, :9] = rng.uniform(-3000, 3000, (64, 9))
    t[:, 18:] = m.as_array()
    tl.append_encoded(t)
    tris, nodes = tl.build_bvh(8, api.BVH_SAH_LITERAL)
    root = nodes[1]
    left = nodes[int(root[0])]
    # median split: left child owns 32 triangles sorted by centroid x
    def count(i):
        nd = nodes[i]
        return int(nd[3]) if nd[3] > 0 else count(int(nd[0])) + count(int(nd[1]))
    assert count(int(root[0])) == 32 and count(int(root[1])) == 32
    cx = tris[:, [0, 3, 6]].astype(np.float64).sum(axis=1)
    assert cx[:32].max() <= cx[32:].min() + 1e-3


def test_median_builder_invariants(bunny_scene):
    tl = api.TriangleList()
    tl.append_encoded(bunny_scene[0])
    tris, nodes = tl.build_bvh(8, api.BVH_MEDIAN)
    check_bvh_invariants(tris, nodes)


def test_read_obj_forms_and_normalisation_quirk():
    """v, v/vt, v/vt/vn face forms (P5/main.cpp:321-333) and the maxy = max(maxx, y) quirk (:317-318)."""
    base = "v 0 0 0\nv 2 0 0\nv 0 4 0\n"
    outs = []
    for f in ("f 1 2 3\n", "f 1/1 2/2 3/3\n", "f 1/1/1 2/2/2 3/3/3\n"):
        tl = api.TriangleList()
        tl.read_obj_text(base + f, api.Material(), api.transform_matrix(), False)
        outs.append(tl.encode_triangles())
    assert np.array_equal(outs[0], outs[1]) and np.array_equal(outs[0], outs[2])
    # literal quirk: y-extent is measured against maxx/minx: maxy = max(maxx=2, 4) = 4, miny = min(minx=0, 4) = 0
    # -> maxaxis = 4, so the x = 2 vertex lands at 0.5
    assert outs[0][0, 3] == pytest.approx(0.5)
    n = outs[0][0, 9:12]
    assert np.allclose(n, [0, 0, 1])
    with pytest.raises(api.EzrtError):
        tl.read_obj_text("v 0 0 0\nf 1 2 3\n", api.Material(), api.transform_matrix(), False)


def test_transform_matrix_and_camera():
    m = api.transform_matrix((0, 90, 0), (1, 2, 3), (2, 2, 2)).reshape(4, 4).T  # row-major view
    p = m @ np.array([1, 0, 0, 1.0])
    assert np.allclose(p[:3], [1, 2, 3 - 2], atol=1e-6)  # +x rotates to -z under a 90 degree y-rotation
    eye, cam = api.camera_orbit(90.0, 10.0, 2.0)  # P5/main.cpp:796-798
    assert np.allclose(np.linalg.norm(eye), 2.0, atol=1e-6)
    C = cam.reshape(4, 4).T
    assert np.allclose(C[:3, 3], eye, atol=1e-5)  # inverse(lookAt) carries the eye in its last column
    fwd = C[:3, :3] @ np.array([0, 0, -1.0])
    assert np.allclose(fwd, -eye / 2.0, atol=1e-5)  # camera looks at the origin
    assert np.allclose(C[:3, :3] @ C[:3, :3].T, np.eye(3), atol=1e-5)


def test_p3_scene_rebuilds_to_golden_arrays(golden_p3):
    from tests.golden.make_golden import p3_scene
    for builder in (api.BVH_SAH_FAST, api.BVH_SAH_LITERAL):
        tris, nodes = p3_scene(builder)
        assert tris.shape == (5300, 36) and nodes.shape == (1868, 12)  # SURVEY.md 8d probe: 5300 / 1868
        assert crc(tris) == int(golden_p3["crc_tris"]) and crc(nodes) == int(golden_p3["crc_nodes"])
    check_bvh_invariants(golden_p3["tris"], golden_p3["nodes"])


def test_oracle_reproduces_golden_images(oracle, golden_p3, golden_synth, small_hdr):
    hdr, cache = small_hdr
    assert crc(hdr) == int(golden_synth["hdr_crc"]) and crc(cache) == int(golden_synth["cache_crc"])
    tris, nodes, eye, cam = golden_p3["tris"], golden_p3["nodes"], golden_p3["eye"], golden_p3["cam"]
    for mode, bounces in ((0, 3), (1, 4), (2, 2), (3, 2)):
        cfg = api.RenderConfig(width=48, height=32, spp=2, max_bounce=bounces, mode=mode, eye=tuple(eye), camera_rotate=tuple(cam),
                               env_color=(0.35, 0.45, 0.6))
        img, c = oracle.render(tris, nodes, cfg, hdr=hdr if mode == 3 else None, hdr_cache=cache if mode == 3 else None)
        assert img.tobytes() == golden_p3["img_mode%d" % mode].tobytes()
        assert [c["rays_primary"], c["rays_bounce"], c["rays_shadow"], c["n_node"], c["n_tri"], c["hits"]] == list(golden_p3["rays_mode%d" % mode])
        assert np.isfinite(img).all() and img.mean() > 0.05


def test_oracle_pruned_policy_is_result_invariant(oracle, golden_p3):
    tris, nodes, eye, cam = golden_p3["tris"], golden_p3["nodes"], golden_p3["eye"], golden_p3["cam"]
    cfg = api.RenderConfig(width=64, height=48, spp=2, max_bounce=3, mode=api.MODE_DISNEY_SOBOL_P5, eye=tuple(eye), camera_rotate=tuple(cam),
                           env_color=(0.3, 0.4, 0.5))
    a, ca = oracle.render(tris, nodes, cfg)
    cfg.traverse = api.TRAVERSE_REFERENCE
    b, cb = oracle.render(tris, nodes, cfg)
    assert a.tobytes() == b.tobytes()
    assert ca["rays"] == cb["rays"] and ca["n_node"] < cb["n_node"] and ca["n_tri"] <= cb["n_tri"]


def test_oracle_bvh_equals_brute_force(oracle, golden_p3):
    """hitBVH == hitArray over all triangles (P2/main.cpp:585-586) incl. the P2 demo ray (0,0,1)->(0.1,-0.1,-0.7)."""
    tris, nodes = golden_p3["tris"], golden_p3["nodes"]
    rng = np.random.default_rng(5)
    o = rng.uniform(-2, 2, (400, 3)).astype(np.float32)
    d = rng.normal(size=(400, 3))
    d = (d / np.linalg.norm(d, axis=1, keepdims=True)).astype(np.float32)
    o[0] = [0, 0, 1]
    d[0] = np.array([0.1, -0.1, -0.7]) / np.linalg.norm([0.1, -0.1, -0.7])
    for traverse in (0, 1):
        a = oracle.trace_rays(tris, nodes, o, d, traverse=traverse)
        b = oracle.trace_rays(tris, nodes, o, d, brute=True)
        assert np.array_equal(a["hit"], b["hit"]) and a["distance"].tobytes() == b["distance"].tobytes()
        # equal distances may come from different (coplanar) triangles only if the brute scan order differs; ties are rare
        assert (a["triangle"] == b["triangle"]).mean() > 0.99
    assert a["hit"][0] == 1


def test_multithreaded_oracle_equals_single_thread(oracle, bunny_scene):
    tris, nodes, eye, cam = bunny_scene
    cfg = api.RenderConfig(width=40, height=30, spp=2, max_bounce=2, mode=0, eye=tuple(eye), camera_rotate=tuple(cam))
    a, _ = oracle.render(tris, nodes, cfg, threads=1)
    b, _ = oracle.render(tris, nodes, cfg, threads=4)
    assert a.tobytes() == b.tobytes()


# ---------------------------------------------------------------- HDR loader + cache
def _write_hdr(path, rgbe, rle):
    """Write a Radiance .hdr: rgbe [h,w,4] uint8; rle selects the adaptive run-length scanline format."""
    h, w, _ = rgbe.shape
    with open(path, "wb") as f:
        f.write(b"#?RADIANCE\nFORMAT=32-bit_rle_rgbe\n\n")
        f.write(("-Y %d +X %d\n" % (h, w)).encode())
        for y in range(h):
            row = rgbe[y]
            if not rle:
                f.write(row.tobytes())
                continue
            f.write(bytes([2, 2, (w >> 8) & 0xFF, w & 0xFF]))
            for c in range(4):
                ch = row[:, c]
                i = 0
                while i < w:
                    run = 1
                    while i + run < w and run < 127 and ch[i + run] == ch[i]:
                        run += 1
                    if run >= 4:
                        f.write(bytes([128 + run, int(ch[i])]))
                        i += run
                    else:
                        j = i
                        lit = []
                        while j < w and len(lit) < 128:
                            r2 = 1
                            while j + r2 < w and r2 < 4 and ch[j + r2] == ch[j]:
                                r2 += 1
                            if r2 >= 4:
                                break
                            lit.append(int(ch[j]))
                            j += 1
                        f.write(bytes([len(lit)] + lit))
                        i = j


def write_rgbe_file(path, rle):
    """a 40x6 Radiance file with random texels and long runs (seeded); returns its rgbe [h,w,4]"""
    rng = np.random.default_rng(9)
    h, w = 6, 40
    rgbe = rng.integers(0, 256, (h, w, 4), dtype=np.uint8)
    rgbe[:, :, 3] = rng.integers(120, 136, (h, w))
    rgbe[2, 5:30, :] = rgbe[2, 5, :]  # long runs
    if not rle:
        rgbe[:, 0, 0] = 7  # make sure a flat scanline cannot be mistaken for the RLE marker (2,2,hi,lo)
    _write_hdr(path, rgbe, rle)
    return rgbe


@pytest.mark.parametrize("rle", [False, True])
def test_hdr_load_decodes_rgbe(tmp_path, rle):
    path = str(tmp_path / "t.hdr")
    rgbe = write_rgbe_file(path, rle)
    h, w = rgbe.shape[:2]
    cols = api.hdr_load(path)
    assert cols.shape == (h, w, 3)
    expect = rgbe[:, :, :3].astype(np.float64) / 256.0 * np.exp2(rgbe[:, :, 3:4].astype(np.float64) - 128.0)
    np.testing.assert_array_equal(cols, expect.astype(np.float32))  # row 0 = first scanline in the file
    # the unmodified reference decoder (HDRLoader::load, compiled by oracle/build_ref.py) decoded the same bytes
    assert crc(cols) == int(rg.load()["rgbe_rle%d" % rle])


def test_hdr_load_equals_reference_loader_on_shipped_map():
    """scanlines of the reference's chinese_garden_2k.hdr, as the reference's own HDRLoader::load decoded them"""
    g = rg.load()
    cols = api.hdr_load(rg.hdr_rows_path(5))
    assert list(cols.shape) == list(g["hdr_rows5_shape"]) and cols.shape[1] == 2048
    assert crc(cols) == int(g["hdr_rows5_crc"])


def test_hdr_cache_properties(small_hdr):
    """calculateHdrCache (P5/main.cpp:592-689): .b is the normalised luminance pdf, .rg are texel coordinates that
    concentrate on the bright lamps; xi_1 = i/height selects the column through the marginal cdf."""
    hdr, cache = small_hdr
    h, w, _ = hdr.shape
    lum = 0.2 * hdr[..., 0].astype(np.float64) + 0.7 * hdr[..., 1] + 0.1 * hdr[..., 2]
    np.testing.assert_allclose(cache[..., 2], lum / lum.sum(), rtol=2e-3)
    assert abs(cache[..., 2].astype(np.float64).sum() - 1.0) < 2e-3
    xs = np.rint(cache[..., 0] * w).astype(int)
    ys = np.rint(cache[..., 1] * h).astype(int)
    assert xs.min() >= 0 and xs.max() < w and ys.min() >= 0 and ys.max() <= h
    # the sample x only depends on the row index i (xi_1 = i/height), monotonically
    assert (xs == xs[:, :1]).all() and (np.diff(xs[:, 0]) >= 0).all()
    # importance: the mean luminance at sampled texels far exceeds the plain mean
    sampled = lum[np.clip(ys, 0, h - 1), xs]
    assert sampled.mean() > 5 * lum.mean()
    # literal re-statement in numpy (float32 accumulation order as the C++ loops)
    # (the luminance weights are double literals in the reference, P5/main.cpp:604: fp64 sum, rounded once)
    pdf = ((0.2 * hdr[..., 0].astype(np.float64) + 0.7 * hdr[..., 1].astype(np.float64)) + 0.1 * hdr[..., 2].astype(np.float64)).astype(np.float32)
    s = np.float32(0)
    for v in pdf.reshape(-1):
        s = np.float32(s + v)
    pdf = pdf / s
    np.testing.assert_array_equal(cache[..., 2], pdf)


# ---------------------------------------------------------------- hardened OBJ reader + scene files (8f row 4)
def test_hardened_obj_reader_triangulates_polygons_and_relative_indices():
    quad = "v 0 0 0\nv 1 0 0\nv 1 1 0\nv 0 1 0\nf 1 2 3 4\n"
    tl = api.TriangleList()
    tl.read_obj_text(quad, api.Material(), api.transform_matrix(), 0)
    assert len(tl) == 1  # reference behaviour: the polygon is cut to its first three vertices
    tl = api.TriangleList()
    tl.read_obj_text(quad, api.Material(), api.transform_matrix(), api.OBJ_HARDENED)
    t = tl.encode_triangles()
    assert t.shape[0] == 2 and np.allclose(t[1, :9], [0, 0, 0, 1, 1, 0, 0, 1, 0])  # fan (1,3,4)
    rel = "v 0 0 0\nv 1 0 0\nv 0 1 0\nf -3 -2 -1\n"
    tl2 = api.TriangleList()
    tl2.read_obj_text(rel, api.Material(), api.transform_matrix(), api.OBJ_HARDENED)
    tl3 = api.TriangleList()
    tl3.read_obj_text("v 0 0 0\nv 1 0 0\nv 0 1 0\nf 1 2 3\n", api.Material(), api.transform_matrix(), 0)
    assert np.array_equal(tl2.encode_triangles(), tl3.encode_triangles())
    with pytest.raises(api.EzrtError):
        tl3.read_obj_text(rel, api.Material(), api.transform_matrix(), 0)  # not hardened: negative index rejected


def test_scene_file_reproduces_programmatic_scene(tmp_path):
    (tmp_path / "blob.obj").write_text(scenes.blob_obj(2))
    (tmp_path / "box.obj").write_text(scenes.box_obj())
    (tmp_path / "scene.txt").write_text("""# P3-style scene
set baseColor 1 1 1
mesh blob.obj smooth rotate 0 0 0 translate 0.3 -0.65 0 scale 1.5 1.5 1.5
set baseColor 0.725 0.71 0.68
set roughness 0.3
mesh box.obj flat translate 0 -1.4 0 scale 18.83 0.01 18.83
reset
set emissive 30 20 10
mesh blob.obj flat translate 0 0.9 0
camera 90 10 2
hdr env.hdr
""")
    tl, cam, hdr = api.load_scene_file(tmp_path / "scene.txt")
    assert cam == (90.0, 10.0, 2.0) and hdr == str(tmp_path / "env.hdr")
    ref = api.TriangleList()
    ref.read_obj_text(scenes.blob_obj(2), api.Material(baseColor=(1, 1, 1)), api.transform_matrix((0, 0, 0), (0.3, -0.65, 0), (1.5, 1.5, 1.5)), 1)
    ref.read_obj_text(scenes.box_obj(), api.Material(baseColor=(0.725, 0.71, 0.68), roughness=0.3), api.transform_matrix((0, 0, 0), (0, -1.4, 0), (18.83, 0.01, 18.83)), 0)
    ref.read_obj_text(scenes.blob_obj(2), api.Material(emissive=(30, 20, 10)), api.transform_matrix((0, 0, 0), (0, 0.9, 0), (1, 1, 1)), 0)
    assert np.array_equal(tl.encode_triangles(), ref.encode_triangles())
    (tmp_path / "bad.txt").write_text("mesh nothere.obj smooth")
    with pytest.raises(api.EzrtError):
        api.load_scene_file(tmp_path / "bad.txt")


def test_accel_build_host_tree_is_well_formed(bunny_scene):
    """ezrt_accel_build(where = host): the binary SAH tree behind the device's acceleration structure (the GPU builder must
    reproduce it node for node, tests/test_gpu_accel_build.py): pre-order numbering, every triangle in exactly one leaf of
    <= leaf_n triangles, every node's box = the union of its triangles' boxes, children inside their parent."""
    tris = np.asarray(bunny_scene[0], np.float32).reshape(-1, 36)
    for leaf_n in (1, 4):
        links, boxes, order, ms = api.accel_build(tris, leaf_n, "host")
        n = len(tris)
        assert sorted(order.tolist()) == list(range(n))
        v = tris[order, :9].reshape(n, 3, 3)
        lo, hi = v.min(1), v.max(1)
        covered = np.zeros(n, np.int32)
        for i, (left, right, cnt, index) in enumerate(links):
            if cnt > 0:
                assert left == 0 and right == 0 and cnt <= leaf_n
                covered[index:index + cnt] += 1
                assert np.array_equal(boxes[i, :3], lo[index:index + cnt].min(0)) and np.array_equal(boxes[i, 3:], hi[index:index + cnt].max(0))
            else:
                assert left == i + 1 and right > left          # pre-order: the left sub-tree follows its parent
                for c in (left, right):
                    assert (boxes[c, :3] >= boxes[i, :3]).all() and (boxes[c, 3:] <= boxes[i, 3:]).all()
                assert np.array_equal(boxes[i, :3], np.minimum(boxes[left, :3], boxes[right, :3]))
                assert np.array_equal(boxes[i, 3:], np.maximum(boxes[left, 3:], boxes[right, 3:]))
        assert (covered == 1).all()

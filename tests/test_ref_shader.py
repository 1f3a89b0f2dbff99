"""The oracle against THE REFERENCE'S OWN SHADER SOURCE.

oracle/ref_shader/ transpiles P3/P4/P5 shaders/fshader.fsh of the reference to C++ and runs them per fragment on the CPU;
GLSL's built-ins -- which the GLSL specification leaves bit-unspecified -- are bound to include/ezrt_math.h.  Everything
else (statements, expression order, control flow, constants, the Sobol table, the RNG seeding) is the reference's text.

  * frames rendered that way are committed in tests/golden/refshader.npz and the hand-written oracle
    must reproduce them bit for bit (runs everywhere, GPU box included);
  * on more inputs, crc32s of the frames the transpiled shaders rendered are committed in tests/golden/reference.npz
    (tests/reference_golden.py) and the oracle's frames must have the same bits."""
import numpy as np
import pytest

from ezrt_b200 import api, scenes
from tests import reference_golden as rg
from tests import refshader_cases as cases


def same_bits(a, b):
    a = np.ascontiguousarray(a, np.float32); b = np.ascontiguousarray(b, np.float32)
    return a.shape == b.shape and bool(((a.view(np.uint32) == b.view(np.uint32)) | (np.isnan(a) & np.isnan(b))).all())


@pytest.mark.parametrize("name", cases.SCENES)
def test_oracle_reproduces_reference_shader_frames(oracle, name):
    g = cases.load()
    hdr, cache = cases.environment()
    tris, nodes, eye, cam = cases.scene(name)
    for case in cases.CASES:
        key, mode, mb, lin, first, spp = case
        want = g["%s_%s" % (name, key)]
        assert np.isfinite(want).all() and float(want.mean()) > 0.05, "golden frame is not a trivial image"
        for traverse in (api.TRAVERSE_REFERENCE, api.TRAVERSE_PRUNED):
            fb = g["%s_m3" % name].copy() if first else None
            got, _ = oracle.render(tris, nodes, cases.config(case, eye, cam, traverse=traverse), hdr=hdr, hdr_cache=cache, hdr_linear=lin,
                                   framebuffer=fb)
            assert same_bits(got, want), "%s %s traverse %d" % (name, key, traverse)


def test_golden_inputs_are_the_committed_ones():
    """refshader.npz was rendered from exactly these arrays (synth.npz pins their crc32)."""
    import os
    import zlib
    s = np.load(os.path.join(cases.GOLDEN, "synth.npz"))
    hdr, cache = cases.environment()
    crc = lambda a: zlib.crc32(np.ascontiguousarray(a).tobytes())
    assert crc(hdr) == int(s["hdr_crc"]) and crc(cache) == int(s["cache_crc"])
    tris, nodes, _, _ = cases.scene("bunny")
    assert crc(tris) == int(s["bunny_crc_tris"]) and crc(nodes) == int(s["bunny_crc_nodes"])
    tris, nodes, _, _ = cases.scene("grid")
    assert crc(tris) == int(s["grid_crc_tris"]) and crc(nodes) == int(s["grid_crc_nodes"])


def test_golden_frames_are_current():
    """the committed frames are what the transpiled shaders produced at the last regeneration of reference.npz"""
    g, r = cases.load(), rg.load()
    for case in cases.CASES[:4]:
        key = case[0]
        assert rg.bits_crc(g["bunny_" + key]) == int(r["shader_bunny_" + key]), key


def live_case(mode, bounces):
    """other image shape, camera, environment size, filter and bounce counts than the committed frames"""
    hdr = scenes.synth_hdr(64, 32)
    eye, cam = api.camera_orbit(37.0, 12.0, 5.5)
    cfg = api.RenderConfig(width=37, height=23, spp=4, max_bounce=bounces, mode=mode, eye=tuple(eye), camera_rotate=tuple(cam),
                           traverse=api.TRAVERSE_REFERENCE)
    return hdr, api.hdr_cache(hdr), cfg


@pytest.mark.parametrize("mode,bounces", [(0, 2), (0, 3), (1, 4), (1, 1), (2, 2), (2, 4), (3, 2), (3, 3)])
@pytest.mark.parametrize("linear", [False, True])
def test_oracle_equals_transpiled_shader_live(oracle, grid_scene, mode, bounces, linear):
    tris, nodes, _, _ = grid_scene
    hdr, cache, cfg = live_case(mode, bounces)
    got, _ = oracle.render(tris, nodes, cfg, hdr=hdr, hdr_cache=cache, hdr_linear=linear)
    assert float(got.mean()) > 0.01
    assert rg.bits_crc(got) == int(rg.load()["shader_live_m%d_b%d_lin%d" % (mode, bounces, linear)])


BOX_CASES = ((0, 3, False), (1, 4, False), (2, 3, True), (3, 3, True))


def box_scene():
    tl = api.TriangleList()
    tl.read_obj_text(scenes.box_obj(), api.Material(baseColor=(0.7, 0.6, 0.5), roughness=0.4, metallic=0.3), api.transform_matrix((0, 0, 0), (0, 0, 0), (3, 3, 3)), False)
    tl.read_obj_text(scenes.sphere_obj(2), api.Material(baseColor=(1, 1, 1), emissive=(9, 8, 7)), api.transform_matrix((0, 0, 0), (0, 0.6, 0), (0.5, 0.5, 0.5)), True)
    tris, nodes = tl.build_bvh(4, api.BVH_SAH_LITERAL)
    eye, cam = api.camera_orbit(20.0, -10.0, 1.2)
    return tris, nodes, lambda mode, mb: api.RenderConfig(width=32, height=24, spp=3, max_bounce=mb, mode=mode, eye=tuple(eye), camera_rotate=tuple(cam),
                                                          traverse=api.TRAVERSE_REFERENCE)


def test_oracle_equals_transpiled_shader_inside_a_box(oracle):
    """camera inside closed geometry (isInside hits, every path terminates on geometry or an emitter)"""
    tris, nodes, config = box_scene()
    hdr, cache = cases.environment()
    r = rg.load()
    for mode, mb, lin in BOX_CASES:
        got, _ = oracle.render(tris, nodes, config(mode, mb), hdr=hdr, hdr_cache=cache, hdr_linear=lin)
        assert rg.bits_crc(got) == int(r["shader_box_m%d" % mode]), mode


def _hdr_frame(seed=5, h=24, w=40, c=3):
    rng = np.random.default_rng(seed)
    fb = (rng.uniform(0, 1, (h, w, c)) ** 4 * 40.0).astype(np.float32)  # HDR range, many dark texels
    fb[0, 0, :3] = 0.0
    fb[0, 1, :3] = (1e-30, 1.0, 3e4)
    return fb


@pytest.mark.parametrize("channels", [3, 4])
def test_tonemap_equals_transpiled_pass3_shader(oracle, channels):
    """shaders/pass3.fsh (identical in parts 3, 4, 5): toneMapping(c, 1.5) then pow(c, 1/2.2)"""
    assert rg.bits_crc(oracle.tonemap(_hdr_frame(c=channels))) == int(rg.load()["pass3_c%d" % channels])


def test_tonemap_reproduces_reference_pass3_golden(oracle):
    """runs everywhere: pass3 output of the reference shader for a fixed frame, committed in refshader.npz"""
    g = cases.load()
    assert same_bits(oracle.tonemap(_hdr_frame()), g["pass3_out"])


SOUP_CASES = ((0, 3, False), (1, 3, False), (2, 2, True), (3, 2, True))


def soup_scene():
    from tests.test_gpu_parity import _soup
    tl = api.TriangleList()
    tl.append_encoded(_soup(3000, 4))
    tris, nodes = tl.build_bvh(8)
    eye, cam = api.camera_orbit(30.0, 20.0, 6.0)
    return tris, nodes, lambda mode, mb: api.RenderConfig(width=64, height=48, spp=2, max_bounce=mb, mode=mode, eye=tuple(eye), camera_rotate=tuple(cam),
                                                          traverse=api.TRAVERSE_REFERENCE)


def test_oracle_equals_transpiled_shader_on_degenerate_soup(oracle):
    """zero-area triangles (NaN normals), slivers, duplicated vertices, axis-aligned coordinates: the NaN / tie
    behaviour of the oracle is the shader's, statement by statement"""
    tris, nodes, config = soup_scene()
    hdr, cache = cases.environment()
    r = rg.load()
    for mode, mb, lin in SOUP_CASES:
        got, _ = oracle.render(tris, nodes, config(mode, mb), hdr=hdr, hdr_cache=cache, hdr_linear=lin)
        assert rg.bits_crc(got) == int(r["shader_soup_m%d" % mode]), mode


def p5_scene(directory):
    """the reference's own P5 set-up (tests/test_ref_host.py checks the product builds what its main() builds) on the
    stored patch of its teapot and scanlines of its map, with its own camera (P5/main.cpp:796-798) at a reduced size"""
    from tests.test_ref_host import p5_main_meshes
    tl = api.TriangleList()
    for path, m, t, s in p5_main_meshes(directory):
        tl.read_obj(path, m, t, s)
    tris, nodes = tl.build_bvh(8, api.BVH_SAH_LITERAL)
    hdr = api.hdr_load(rg.hdr_rows_path(5))
    eye, cam = api.camera_orbit(90.0, 10.0, 2.0)
    cfg = api.RenderConfig(width=64, height=64, spp=2, max_bounce=2, mode=api.MODE_DISNEY_IS_MIS_P5, eye=tuple(eye), camera_rotate=tuple(cam),
                           traverse=api.TRAVERSE_REFERENCE)
    return tris, nodes, hdr, api.hdr_cache(hdr), cfg


def test_oracle_equals_transpiled_shader_on_the_reference_p5_scene(oracle, tmp_path):
    """the reference's own P5 set-up, end to end: the scene, map and sampling cache its main() builds, rendered by its
    shader (transpiled); the oracle must agree bit for bit"""
    tris, nodes, hdr, cache, cfg = p5_scene(tmp_path)
    got, c = oracle.render(tris, nodes, cfg, hdr=hdr, hdr_cache=cache, hdr_linear=True)
    assert c["rays_shadow"] > 0 and float(got.mean()) > 0.01
    assert rg.bits_crc(got) == int(rg.load()["shader_p5_scene"])

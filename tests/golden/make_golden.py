#!/usr/bin/env python
"""Generate tests/golden/p3_scene.npz and synth.npz (the P3 meshes come from tests/golden/reference_models.npz).

  p3_scene.npz : the reference's own P3 scene (P3/main.cpp:688-701: Stanford bunny + quad floor + emissive
                 sphere, read with OUR readObj/buildBVHwithSAH restatement), encoded arrays (float16-free,
                 float32) + crc32s + camera, and the ORACLE's render of it in the four integrator modes at
                 48x32, 2 spp.  GPU tests re-render these arrays and must reproduce the images bit for bit;
                 CPU tests re-run the oracle and the literal BVH builder against them.
  synth.npz    : crc32 of the synthetic scenes' arrays + oracle images (platform-independent scene builders).
The reference holds no golden vectors (SURVEY.md 4); these files freeze OUR restatement against accidental drift.
The frames that pin it to the reference's own shader source are in refshader.npz (make_golden_refshader.py).
"""
import os
import sys
import tempfile
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from ezrt_b200 import api, scenes  # noqa: E402
from tests import oracle_binding as oracle  # noqa: E402
from tests import reference_golden as rg  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))


def crc(a):
    return zlib.crc32(np.ascontiguousarray(a).tobytes())


def p3_scene(builder=api.BVH_SAH_FAST):
    with tempfile.TemporaryDirectory() as d:
        tl = api.TriangleList()
        m = api.Material(baseColor=(1, 1, 1))
        tl.read_obj(rg.write_model(d, "p3_bunny"), m, api.transform_matrix((0, 0, 0), (0.3, -1.6, 0), (1.5, 1.5, 1.5)), True)
        m = api.Material(baseColor=(0.725, 0.71, 0.68))
        tl.read_obj(rg.write_model(d, "p3_quad"), m, api.transform_matrix((0, 0, 0), (0, -1.4, 0), (18.83, 0.01, 18.83)), False)
        m = api.Material(baseColor=(1, 1, 1), emissive=(30, 20, 10))
        tl.read_obj(rg.write_model(d, "p3_sphere"), m, api.transform_matrix((0, 0, 0), (0.0, 0.9, 0.0), (1, 1, 1)), False)
        return tl.build_bvh(8, builder)


def images(tris, nodes, eye, cam, hdr, cache, w=48, h=32, spp=2):
    out = {}
    for mode, bounces in ((0, 3), (1, 4), (2, 2), (3, 2)):
        cfg = api.RenderConfig(width=w, height=h, spp=spp, max_bounce=bounces, mode=mode, eye=tuple(eye), camera_rotate=tuple(cam),
                               env_color=(0.35, 0.45, 0.6))
        if mode == 3:
            img, c = oracle.render(tris, nodes, cfg, hdr=hdr, hdr_cache=cache, hdr_linear=True)
        else:
            img, c = oracle.render(tris, nodes, cfg)
        out["img_mode%d" % mode] = img
        out["rays_mode%d" % mode] = np.array([c["rays_primary"], c["rays_bounce"], c["rays_shadow"], c["n_node"], c["n_tri"], c["hits"]], np.int64)
    return out


def main():
    hdr = scenes.synth_hdr(128, 64)
    cache = api.hdr_cache(hdr)
    eye, cam = api.camera_orbit(0.0, 0.0, 4.0)
    tris, nodes = p3_scene()
    d = dict(tris=tris, nodes=nodes, eye=eye, cam=cam, crc_tris=np.uint32(crc(tris)), crc_nodes=np.uint32(crc(nodes)))
    d.update(images(tris, nodes, eye, cam, hdr, cache))
    np.savez_compressed(os.path.join(HERE, "p3_scene.npz"), **d)
    print("p3 scene", tris.shape, nodes.shape, hex(crc(tris)), hex(crc(nodes)))

    s = {}
    tris, nodes, eye, cam = scenes.s_bunny()
    s.update(bunny_crc_tris=np.uint32(crc(tris)), bunny_crc_nodes=np.uint32(crc(nodes)), bunny_shape=np.array([tris.shape[0], nodes.shape[0]]))
    s.update({"bunny_" + k: v for k, v in images(tris, nodes, eye, cam, hdr, cache).items()})
    tris, nodes, eye, cam = scenes.s_grid(3, 2, 2)
    s.update(grid_crc_tris=np.uint32(crc(tris)), grid_crc_nodes=np.uint32(crc(nodes)), grid_shape=np.array([tris.shape[0], nodes.shape[0]]))
    s.update({"grid_" + k: v for k, v in images(tris, nodes, eye, cam, hdr, cache, 40, 24, 2).items()})
    s.update(hdr_crc=np.uint32(crc(hdr)), cache_crc=np.uint32(crc(cache)))
    np.savez_compressed(os.path.join(HERE, "synth.npz"), **s)
    print("synthetic scenes done")


if __name__ == "__main__":
    main()

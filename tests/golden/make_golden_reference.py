#!/usr/bin/env python
"""Generate tests/golden/reference.npz, reference_models.npz and *_rows.hdr (see tests/reference_golden.py) from the
reference tree: its data files are sampled, and its own code -- compiled by oracle/build_ref.py into oracle/_ref/ --
computes the results the tests compare with.   python tests/golden/make_golden_reference.py"""
import ctypes as C
import os
import pathlib
import re
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from ezrt_b200 import api, build, scenes  # noqa: E402
from tests import reference_golden as rg  # noqa: E402
from tests import refhost_binding as refhost  # noqa: E402
from tests import refshader_binding as refshader  # noqa: E402
from tests import refshader_cases as cases  # noqa: E402
from tests import test_host_scene, test_ref_host, test_ref_shader  # noqa: E402

TEAPOT_FACES = (30000, 1536)   # first face and count of the stored teapot patch
HDR_SAMPLE_ROWS = {5: 6, 4: 6, 3: 2}   # scanlines kept of each map, evenly spread


def src(part, *rel):
    return os.path.join(refhost.source_dir(part), *rel)


def teapot_patch(path, first, count):
    """a block of consecutive faces of the OBJ file and the vertices they use (renumbered, in file order)"""
    lines = open(path, "rb").read().split(b"\n")
    verts = [ln for ln in lines if ln.startswith(b"v ")]
    faces = [ln for ln in lines if ln.startswith(b"f ")][first:first + count]
    used = sorted({int(tok.split(b"/")[0]) for f in faces for tok in f.split()[1:]})
    new = {old: i + 1 for i, old in enumerate(used)}
    out = [verts[i - 1] for i in used]
    for f in faces:
        toks = [b"/".join(b"%d" % new[int(tok.split(b"/")[0])] for _ in tok.split(b"/")) for tok in f.split()[1:]]
        out.append(b"f " + b" ".join(toks) + (b"\r" if f.endswith(b"\r") else b""))
    return b"\n".join(out) + b"\n"


def hdr_rows(path, n_rows):
    """a valid Radiance file made of `n_rows` evenly spread scanlines of `path`, each copied byte for byte"""
    data = open(path, "rb").read()
    head = data.index(b"\n\n") + 2
    res = data.index(b"\n", head) + 1
    _, h, _, w = data[head:res].split()
    h, w = int(h), int(w)
    spans, pos = [], res
    for _ in range(h):
        start = pos
        if data[pos] == 2 and data[pos + 1] == 2 and data[pos + 2] < 128:   # adaptive run-length scanline
            pos += 4
            for _ in range(4):
                n = 0
                while n < w:
                    cnt = data[pos]
                    n, pos = (n + cnt - 128, pos + 2) if cnt > 128 else (n + cnt, pos + 1 + cnt)
        else:
            pos += 4 * w
        spans.append((start, pos))
    rows = np.linspace(0, h - 1, n_rows + 2).round().astype(int)[1:-1]
    body = b"".join(data[spans[r][0]:spans[r][1]] for r in rows)
    return data[:head] + b"-Y %d +X %d\n" % (n_rows, w) + body, rows


def ref_hdr_load(path):
    lib = C.CDLL(build.build_reference_hdrloader())
    W, H, ptr = C.c_int(), C.c_int(), C.POINTER(C.c_float)()
    assert lib.ref_hdr_load(path.encode(), C.byref(W), C.byref(H), C.byref(ptr)) == 0
    out = np.ctypeslib.as_array(ptr, shape=(H.value, W.value, 3)).copy()
    lib.ref_hdr_free(ptr)
    return out


def ref_scene(meshes, leaf_n=8, sah=True, part=5):
    return refhost.build_scene([(p, m.as_array(), t, s) for p, m, t, s in meshes], leaf_n, sah, part)


def main():
    assert refhost.available() and refshader.available(), "needs the reference tree"
    crc, g = rg.crc, {}

    # ---- data fixtures sampled from the reference's shipped files
    models = {"p3_bunny": open(src(3, "models", "Stanford Bunny.obj"), "rb").read(), "p3_quad": open(src(3, "models", "quad.obj"), "rb").read(),
              "p3_sphere": open(src(3, "models", "sphere.obj"), "rb").read(), "p5_quad": open(src(5, "models", "quad.obj"), "rb").read(),
              "p5_teapot_patch": teapot_patch(src(5, "models", "teapot.obj"), *TEAPOT_FACES)}
    np.savez_compressed(rg.MODELS_NPZ, **{k: np.frombuffer(v, np.uint8) for k, v in models.items()})
    maps = {5: src(5, "HDR", "chinese_garden_2k.hdr"), 4: src(4, "HDR", "peppermint_powerplant_4k.hdr"), 3: src(3, "HDR", "circus_arena_4k.hdr")}
    for part, path in maps.items():
        data, rows = hdr_rows(path, HDR_SAMPLE_ROWS[part])
        with open(rg.hdr_rows_path(part), "wb") as f:
            f.write(data)
        ref = ref_hdr_load(rg.hdr_rows_path(part))
        assert np.array_equal(ref, api.hdr_load(path)[rows]), "sampled scanlines decode as in the whole map"
        g["hdr_rows%d_shape" % part] = np.array(ref.shape)
        g["hdr_rows%d_crc" % part] = np.uint32(crc(ref))

    with tempfile.TemporaryDirectory() as d:
        # ---- the reference's host code (tests/test_ref_host.py)
        g["p5_main_scene_crc"] = np.array([crc(a) for a in ref_scene(test_ref_host.p5_main_meshes(d))], np.uint32)
        g["p5_cache_crc"] = np.uint32(crc(refhost.hdr_cache(ref_hdr_load(rg.hdr_rows_path(5)))))
        g["p4_main_scene_crc"] = np.array([crc(a) for a in ref_scene(test_ref_host.p4_main_meshes(d), part=4)], np.uint32)
        run = os.path.join(d, "p3_main")   # P3's main() opens ./HDR/sunset.hdr, which P3 does not ship: give it the map it does ship
        os.makedirs(os.path.join(run, "HDR"))
        for sub in ("models", "shaders"):
            os.symlink(src(3, sub), os.path.join(run, sub))
        os.symlink(maps[3], os.path.join(run, "HDR", "sunset.hdr"))
        r_tris, r_nodes, _ = refhost.run_main(3, run)
        assert [crc(r_tris), crc(r_nodes)] == [crc(a) for a in ref_scene(test_ref_host.p3_main_meshes(d), part=3)]
        g["p3_main_crc"] = np.array([crc(r_tris), crc(r_nodes), crc(np.ascontiguousarray(r_tris[:, :24]))], np.uint32)
        for leaf_n in (1, 4, 8, 13):
            meshes, poses = test_ref_host.synthetic_meshes(pathlib.Path(d), leaf_n)
            g["transforms_leaf%d" % leaf_n] = np.array([crc(refhost.transform_matrix(*p)) for p in poses], np.uint32)
            g["builders_leaf%d" % leaf_n] = np.array([crc(a) for sah in (True, False) for a in ref_scene(meshes, leaf_n, sah)], np.uint32)
        for w, h in ((128, 64), (64, 32), (96, 40), (16, 8)):
            g["hdr_cache_%dx%d" % (w, h)] = np.uint32(crc(refhost.hdr_cache(scenes.synth_hdr(w, h))))
        for form in ("v", "v/vt", "v/vt/vn"):
            path = os.path.join(d, "forms.obj")
            with open(path, "w") as f:
                f.write(test_ref_host.face_forms_obj(form))
            m, t = api.Material(**test_ref_host.FACE_FORM_MATERIAL), api.transform_matrix(*test_ref_host.FACE_FORM_TRANSFORM)
            g["face_form_" + form.replace("/", "_")] = np.array([crc(a) for s in (False, True) for a in ref_scene([(path, m, t, s)])], np.uint32)
        for rle in (False, True):
            path = os.path.join(d, "t.hdr")
            test_host_scene.write_rgbe_file(path, rle)
            g["rgbe_rle%d" % rle] = np.uint32(crc(ref_hdr_load(path)))

        # ---- the reference's shaders, transpiled (tests/test_ref_shader.py)
        fsh = open(src(5, "shaders", "fshader.fsh")).read()
        m = re.search(r"const uint V\[8\*32\] = \{\s*([0-9u,\s]+)\};", fsh)
        g["sobol_V"] = np.array([int(x.strip().rstrip("u")) for x in m.group(1).split(",") if x.strip()], np.uint32)
        hdr, cache = cases.environment()
        tris, nodes, eye, cam = cases.scene("bunny")
        for case in cases.CASES[:4]:
            g["shader_bunny_" + case[0]] = np.uint32(rg.bits_crc(refshader.render(tris, nodes, cases.config(case, eye, cam), hdr, cache, hdr_linear=case[3])))
        tris, nodes, _, _ = cases.scene("grid")
        for mode, bounces in ((0, 2), (0, 3), (1, 4), (1, 1), (2, 2), (2, 4), (3, 2), (3, 3)):
            h2, c2, cfg = test_ref_shader.live_case(mode, bounces)
            for lin in (False, True):
                g["shader_live_m%d_b%d_lin%d" % (mode, bounces, lin)] = np.uint32(rg.bits_crc(refshader.render(tris, nodes, cfg, h2, c2, hdr_linear=lin)))
        for scene, key, modes in ((test_ref_shader.box_scene, "box", test_ref_shader.BOX_CASES), (test_ref_shader.soup_scene, "soup", test_ref_shader.SOUP_CASES)):
            tris, nodes, config = scene()
            for mode, mb, lin in modes:
                g["shader_%s_m%d" % (key, mode)] = np.uint32(rg.bits_crc(refshader.render(tris, nodes, config(mode, mb), hdr, cache, hdr_linear=lin)))
        for c in (3, 4):
            g["pass3_c%d" % c] = np.uint32(rg.bits_crc(refshader.pass3(test_ref_shader._hdr_frame(c=c))))
        tris, nodes, h5, c5, cfg = test_ref_shader.p5_scene(d)
        g["shader_p5_scene"] = np.uint32(rg.bits_crc(refshader.render(tris, nodes, cfg, h5, c5, hdr_linear=True)))

    np.savez_compressed(rg.REFERENCE_NPZ, **g)
    for f in [rg.MODELS_NPZ, rg.REFERENCE_NPZ] + [rg.hdr_rows_path(p) for p in maps]:
        print("%-60s %7d bytes" % (os.path.relpath(f, ROOT), os.path.getsize(f)))


if __name__ == "__main__":
    main()

"""ctypes binding of oracle/_ref/libezrt_refhost.so: the reference's OWN host code (P5 main.cpp and
lib/hdrloader.cpp), compiled from where it lies under /root/reference against the stand-in GL/GLUT/glm
headers of oracle/ref_stubs/ (oracle/ref_host_shim.cpp).  TEST INFRASTRUCTURE; exists only where
/root/reference does -- `available()` is False on the GPU box."""
import ctypes as C
import os

import numpy as np

from ezrt_b200 import build as _build

SOURCE_DIR = _build.REFERENCE_P5
_fp = C.POINTER(C.c_float)
_libs = {}


def source_dir(part):
    return os.path.join(_build.REFERENCE_ROOT, _build.REFERENCE_PARTS[part - 3], "source code")


def _load(part=5):
    if part not in _libs:
        so = _build.build_reference_host(part=part)
        if so is None or not os.path.exists(so):
            return None
        lib = C.CDLL(so)
        lib.refhost_upload_info.restype = C.c_longlong
        _libs[part] = lib
    return _libs[part]


def available():
    """the library AND the reference's data files (models/, HDR/) its tests read"""
    return os.path.isdir(source_dir(5)) and _load() is not None


def _f(a):
    return a.ctypes.data_as(_fp)


def transform_matrix(rotate, translate, scale):
    out = np.zeros(16, np.float32)
    r, t, s = (np.asarray(v, np.float32) for v in (rotate, translate, scale))
    _load().refhost_transform_matrix(_f(r), _f(t), _f(s), _f(out))
    return out


def build_scene(meshes, leaf_n=8, sah=True, part=5):
    """meshes: [(obj path, material18, trans16, smooth)] -> (tris [n,36], nodes [m,12]) as main() of tutorial `part` would upload them"""
    lib = _load(part)
    lib.refhost_reset()
    for path, material, trans, smooth in meshes:
        m = np.ascontiguousarray(material, np.float32); t = np.ascontiguousarray(trans, np.float32)
        assert m.size == 18 and t.size == 16
        lib.refhost_read_obj(os.fsencode(path), _f(m), _f(t), int(bool(smooth)))
    lib.refhost_build_bvh(int(leaf_n), int(bool(sah)))
    nt, nn = C.c_int(), C.c_int()
    lib.refhost_counts(C.byref(nt), C.byref(nn))
    tris = np.zeros((nt.value, 36), np.float32); nodes = np.zeros((nn.value, 12), np.float32)
    lib.refhost_encode(_f(tris), _f(nodes))
    return tris, nodes


def hdr_cache(hdr):
    hdr = np.ascontiguousarray(hdr, np.float32)
    out = np.zeros_like(hdr)
    _load().refhost_hdr_cache(_f(hdr), hdr.shape[1], hdr.shape[0], _f(out))
    return out


def run_main(part=5, cwd=None):
    """the reference's main() (of tutorial part 3, 4 or 5) up to glutMainLoop(), run in `cwd` (default: its own
    source directory -- it opens models/, HDR/ and shaders/ relative to the cwd).  Returns its uploads in call
    order: triangle texture buffer [n,36], BVH texture buffer [m,12], HDR map [h,w,3] and (part 5) the HDR sampling cache."""
    lib = _load(part)
    n = lib.refhost_run_main(os.fsencode(cwd or source_dir(part)))
    assert n == (4 if part == 5 else 3), n
    out = []
    for i in range(n):
        w, h, tg = C.c_int(), C.c_int(), C.c_uint()
        size = lib.refhost_upload_info(i, C.byref(w), C.byref(h), C.byref(tg))
        a = np.zeros(size // 4, np.float32)
        lib.refhost_upload_copy(i, a.ctypes.data_as(C.c_void_p))
        out.append(a.reshape(h.value, w.value, 3) if w.value else a)
    return [out[0].reshape(-1, 36), out[1].reshape(-1, 12)] + out[2:]

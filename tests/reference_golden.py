"""What the reference computed, stored so that the tests comparing with it run anywhere.

tests/golden/reference.npz holds crc32s (and a few small arrays) of results of the reference's own code -- its host code
(tests/refhost_binding.py), its transpiled shaders (tests/refshader_binding.py) and its HDR loader -- on fixed inputs.
The inputs are either generated from seeds or sampled from the reference's shipped data files:

  reference_models.npz   the text of P3's Stanford Bunny.obj, quad.obj and sphere.obj (whole files), P5's quad.obj, and
                         a connected patch of P5's teapot.obj (a block of its faces with the vertices they use)
  *_rows.hdr             a few scanlines, copied byte for byte, of the reference's environment maps

tests/golden/make_golden_reference.py regenerates all of it where the reference tree is present."""
import os
import zlib

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
REFERENCE_NPZ = os.path.join(GOLDEN, "reference.npz")
MODELS_NPZ = os.path.join(GOLDEN, "reference_models.npz")
# sampled environment maps: P5 chinese_garden_2k.hdr, P4 peppermint_powerplant_4k.hdr, P3 circus_arena_4k.hdr
HDR_ROWS = {5: "chinese_garden_rows.hdr", 4: "peppermint_powerplant_rows.hdr", 3: "circus_arena_rows.hdr"}


def crc(a):
    return zlib.crc32(np.ascontiguousarray(a).tobytes())


def bits_crc(a):
    """crc32 of a float32 array with every NaN made the same NaN (the bit comparisons treat all NaNs as equal)"""
    a = np.array(a, np.float32, copy=True, order="C")
    a[np.isnan(a)] = np.float32("nan")
    return crc(a)


def load():
    return np.load(REFERENCE_NPZ)


MODELS = ("p3_bunny", "p3_quad", "p3_sphere", "p5_quad", "p5_teapot_patch")


def write_model(directory, name):
    """writes the stored OBJ file `name` (one of MODELS) into `directory`, byte for byte; returns its path"""
    path = os.path.join(str(directory), name + ".obj")
    with open(path, "wb") as f:
        f.write(np.load(MODELS_NPZ)[name].tobytes())
    return path


def hdr_rows_path(part):
    return os.path.join(GOLDEN, HDR_ROWS[part])

"""Known-answer tests that pin the oracle (and the shared tables) to values derivable directly
from the reference's constants (SURVEY.md section 4) -- the only reference-provided pins there are."""
import os
import re
import struct
import zlib

import numpy as np

from tests import reference_golden as rg

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _table():
    text = open(os.path.join(ROOT, "include", "ezrt_sobol_table.inc")).read()
    return [int(x[:-1]) for x in re.findall(r"\d+u", text)]


def test_pi_literal_is_one_ulp_below_float_pi(oracle):
    # "#define PI 3.1415926", P5/fsh:27
    assert struct.pack("<f", oracle.pi()) == struct.pack("<I", 0x40490FDA)


def test_wang_hash_chain_from_seed_1(oracle):
    # P5/fsh:320-331
    h, r = oracle.wang_chain(1, 3)
    assert list(h) == [663891101, 1738326990, 801461103]
    np.testing.assert_allclose(r, [0.15457419, 0.40473580, 0.18660471], rtol=0, atol=1e-8)


def test_sobol_first_points_match_joe_kuo(oracle):
    # sobol(d, grayCode(i)), i = 0..7, dims 0..3 (P5/fsh:356-369; T5/tutorial.md:241-247)
    expect = {
        0: [0, .5, .75, .25, .375, .875, .625, .125],
        1: [0, .5, .25, .75, .375, .875, .125, .625],
        2: [0, .5, .25, .75, .625, .125, .875, .375],
        3: [0, .5, .25, .75, .875, .375, .625, .125],
    }
    for d, vals in expect.items():
        assert [oracle.sobol(d, i) for i in range(8)] == vals


def test_sobol_table_checksum_and_reference_literal():
    t = _table()
    assert len(t) == 256
    assert zlib.crc32(struct.pack("<256I", *t)) == 0xAB08B2B2
    # the literal `const uint V[8*32]` of P5's fshader.fsh, as tests/golden/make_golden_reference.py read it
    assert [int(v) for v in rg.load()["sobol_V"]] == t


def test_cranley_patterson_seed_and_wrap(oracle):
    # pseed = (px*1973 + py*9277 + 59*26699) | 1, two wang_hash draws, wrap into [0,1] (P5/fsh:378-396)
    assert 114514 // 1919 == 59
    px, py = 17, 5
    h, r = oracle.wang_chain((px * 1973 + py * 9277 + 59 * 26699) | 1, 2)
    x, y = oracle.cp_rotation(0.75, 0.5, px, py)
    ex = np.float32(0.75) + r[0]
    ey = np.float32(0.5) + r[1]
    ex = ex - np.float32(1) if ex > 1 else ex
    ey = ey - np.float32(1) if ey > 1 else ey
    assert (np.float32(x), np.float32(y)) == (ex, ey)
    assert 0.0 <= x <= 1.0 and 0.0 <= y <= 1.0


def test_math_functions_are_accurate(oracle):
    """ezrt_math.h defines sin/cos/log/exp/atan2/asin itself; they must still be those functions (<= 4 ulp-ish)."""
    rng = np.random.default_rng(0)
    x = rng.uniform(-13, 13, 20000).astype(np.float32)
    np.testing.assert_allclose(oracle.eval_math(0, x), np.sin(x.astype(np.float64)), atol=3e-7)
    np.testing.assert_allclose(oracle.eval_math(1, x), np.cos(x.astype(np.float64)), atol=3e-7)
    p = rng.uniform(1e-6, 50, 20000).astype(np.float32)
    np.testing.assert_allclose(oracle.eval_math(2, p), np.log(p.astype(np.float64)), rtol=5e-7, atol=2e-7)
    e = rng.uniform(-30, 30, 20000).astype(np.float32)
    np.testing.assert_allclose(oracle.eval_math(3, e), np.exp(e.astype(np.float64)), rtol=1e-6)
    a = rng.uniform(1e-6, 1, 20000).astype(np.float32); b = rng.uniform(0, 1, 20000).astype(np.float32)
    np.testing.assert_allclose(oracle.eval_math(4, a, b), np.power(a.astype(np.float64), b.astype(np.float64)), rtol=4e-6)
    y = rng.uniform(-2, 2, 20000).astype(np.float32); z = rng.uniform(-2, 2, 20000).astype(np.float32)
    np.testing.assert_allclose(oracle.eval_math(5, y, z), np.arctan2(y.astype(np.float64), z.astype(np.float64)), atol=5e-7)
    s = rng.uniform(-1, 1, 20000).astype(np.float32)
    np.testing.assert_allclose(oracle.eval_math(6, s), np.arcsin(s.astype(np.float64)), atol=5e-7)

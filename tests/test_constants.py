"""Device constants (tools/gen_curve_constants.py -> libecc_b200/csrc/curve_constants.inc) against the reference's
own curve parameters (read through ref_curve_info from src/curves/known/ec_params_*.h, stored under tests/golden/reference/)
and plain integers."""
import ctypes
import os
import re

import numpy as np
import pytest

from common import ALL_CURVES, CURVES, ORDER, PRIME, ROOT, ref_lib, reference_answer


def parse_inc():
    txt = open(os.path.join(ROOT, "libecc_b200", "csrc", "curve_constants.inc")).read()
    out = {}
    for m in re.finditer(r"struct (\w+) \{(.*?)\n\};", txt, re.S):
        name, body = m.group(1), m.group(2)
        vals = {}
        for a in re.finditer(r"ECC_CONST_ARRAY\((\w+), (\d+), ([^)]*)\)", body):
            words = [int(w.strip().rstrip("u"), 16) for w in a.group(3).split(",")]
            assert len(words) == int(a.group(2))
            vals[a.group(1)] = sum(w << (32 * i) for i, w in enumerate(words))
        m0 = re.search(r"M0 = (0x[0-9a-f]+)u", body)
        if m0:
            vals["M0"] = int(m0.group(1), 16)
        out[name] = vals
    return out


@reference_answer
def ref_curve_info(curve):
    """plen, qlen and the big-endian p, q, a, b, gx, gy of the reference's curve parameters."""
    plen, qlen = ctypes.c_uint32(), ctypes.c_uint32()
    bufs = [ctypes.create_string_buffer(66) for _ in range(6)]
    assert ref_lib().ref_curve_info(curve.encode(), ctypes.byref(plen), ctypes.byref(qlen), *bufs) == 0
    return (plen.value, qlen.value) + tuple(np.frombuffer(x.raw[: plen.value], np.uint8) for x in bufs)


@pytest.mark.parametrize("curve", list(ALL_CURVES))
def test_generated_constants(curve):
    inc = parse_inc()
    p, q = PRIME[curve], ORDER[curve]
    n = 2 * ((p.bit_length() + 63) // 64)  # two device words per reference limb
    R = 1 << (32 * n)
    for tag, mod in (("Fp_" + curve, p), ("Fq_" + curve, q)):
        f = inc[tag]
        assert f["P"] == mod
        assert f["ONE"] == R % mod and f["RR"] == R * R % mod and f["PM2"] == mod - 2
        assert (f["M0"] * mod + 1) % (1 << 32) == 0
    c = inc["Curve_" + curve]
    gx, gy = c["GX"], c["GY"]
    assert c["GX_MONT"] == gx * R % p and c["GY_MONT"] == gy * R % p
    b = c["B_MONT"] * pow(R, -1, p) % p
    a = c["A_MONT"] * pow(R, -1, p) % p
    assert (gy * gy - (gx ** 3 + a * gx + b)) % p == 0
    plen, qlen, *bufs = ref_curve_info(curve)
    rp, rq, ra, rb, rgx, rgy = [int.from_bytes(x.tobytes(), "big") for x in bufs]
    assert (rp, rq, rgx, rgy, rb, ra) == (p, q, gx, gy, b, a)
    assert (plen, qlen) == ALL_CURVES[curve][1:]

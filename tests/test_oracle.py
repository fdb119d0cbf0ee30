"""Pins the oracle port (oracle/ecc_oracle.c) against the reference's own known-answer vectors
(tests/golden/*.json, extracted by tests/golden/dump_golden.c from the reference's test headers) and against the
unmodified reference's results on seeded random inputs (tests/golden/reference/, see common.reference_answer)."""
import ctypes

import numpy as np
import pytest

from common import (hx_fit, ALL_CURVES, CURVES, HASHLEN, ORDER, edge_scalars, golden, hx, oracle_lib, oracle_sign, oracle_smul,
                    oracle_verify, random_scalars, ref_lib, ref_smul, reference_answer, _buf)


@pytest.mark.parametrize("curve", ["SECP256R1", "SECP384R1", "SECP521R1", "SECP224R1", "SECP192R1"])
def test_ecccdh_kat_fixed_and_variable_base(curve):
    vecs = [v for v in golden("ecccdh_kat.json") if v["curve"] == curve]
    assert len(vecs) == 25
    _, plen, qlen = ALL_CURVES[curve]
    d = np.stack([hx_fit(v["priv"], ALL_CURVES[v["curve"]][2]) for v in vecs])
    out, st = oracle_smul(curve, d)
    assert (st == 0).all()
    for v, o in zip(vecs, out):
        assert o.tobytes().hex() == v["our_pub"], v["name"]            # d*G, full affine point
    peers = np.stack([hx(v["peer_pub"]) for v in vecs])
    out, st = oracle_smul(curve, d, peers)
    assert (st == 0).all()
    for v, o in zip(vecs, out):
        assert o[:plen].tobytes().hex() == v["shared"], v["name"]      # x(d*Q)


def test_ecdsa_kat_verify_and_sign():
    vecs = golden("ecdsa_kat.json")
    assert {v["curve"] for v in vecs} >= {"SECP256R1", "SECP384R1", "FRP256V1", "BRAINPOOLP256R1"}
    for v in vecs:
        curve, hlen = v["curve"], HASHLEN[v["hash"]]
        assert v["ref_verdict"] == 0
        got = oracle_verify(curve, hx(v["sig"]), hx(v["pub"]), hx(v["digest"]), hlen)
        assert got[0] == 0, v["name"]
        # pubkey = priv * G
        out, st = oracle_smul(curve, hx_fit(v["priv"], ALL_CURVES[v["curve"]][2]))
        assert st[0] == 0 and out[0].tobytes().hex() == v["pub"], v["name"]
        if "nonce" in v:  # the reference's harness-injected nonce reproduces the expected signature
            sig, st = oracle_sign(curve, hx_fit(v["priv"], ALL_CURVES[v["curve"]][2]), hx_fit(v["nonce"], ALL_CURVES[v["curve"]][2]), hx(v["digest"]), hlen)
            assert st[0] == 0 and sig[0].tobytes().hex() == v["sig"], v["name"]


WYCHE_CURVES = ["SECP256R1", "SECP384R1", "BRAINPOOLP256R1", "BRAINPOOLP384R1", "SECP256K1", "SECP521R1", "BRAINPOOLP512R1",
                "SECP224R1"]


@pytest.mark.parametrize("curve", WYCHE_CURVES)
def test_wycheproof_ecdsa_matches_reference_verdicts(curve):
    _, plen, qlen = ALL_CURVES[curve]
    vecs = [v for v in golden("wycheproof_ecdsa.json.gz") if v["curve"] == curve]
    assert len(vecs) > 400
    by_h = {}
    for v in vecs:
        by_h.setdefault(v["hash"], []).append(v)
    checked = 0
    for h, vs in by_h.items():
        ok_len = [v for v in vs if len(v["sig"]) == 4 * qlen and len(v["pub"]) == 4 * plen]
        bad_len = [v for v in vs if v not in ok_len]
        for v in bad_len:  # the reference rejects a wrong siglen before any arithmetic (ecdsa_common.c:645)
            assert v["ref_verdict"] == -1
        if not ok_len:
            continue
        sig = np.stack([hx(v["sig"]) for v in ok_len])
        pub = np.stack([hx(v["pub"]) for v in ok_len])
        dg = np.stack([hx(v["digest"]) for v in ok_len])
        got = oracle_verify(curve, sig, pub, dg, HASHLEN[h])
        want = np.array([v["ref_verdict"] for v in ok_len], dtype=np.int8)
        assert (got == want).all(), [v["name"] for v, g, w in zip(ok_len, got, want) if g != w][:5]
        # and the Wycheproof labels themselves: valid -> accepted, invalid -> rejected
        for v, g in zip(ok_len, got):
            if v["expected"] == 1:
                assert g == 0
            if v["expected"] == -1:
                assert g == -1
        checked += len(ok_len)
    assert checked > 400


@pytest.mark.parametrize("curve", WYCHE_CURVES)
def test_wycheproof_ecdh_points(curve):
    _, plen, qlen = ALL_CURVES[curve]
    vecs = [v for v in golden("wycheproof_ecdh.json.gz") if v["curve"] == curve and len(v["priv"]) <= 2 * qlen]
    assert len(vecs) > 200
    d = np.stack([hx(v["priv"].rjust(2 * qlen, "0")) for v in vecs])
    q = np.stack([hx(v["peer_pub"]) for v in vecs])
    out, st = oracle_smul(curve, d, q)
    for v, o, s in zip(vecs, out, st):
        assert s == v["ref_status"], v["name"]
        assert o.tobytes().hex() == v["ref_point"], v["name"]
        if v["expected"] == 1:
            assert o[:plen].tobytes().hex() == v["shared"].rjust(2 * plen, "0")


@pytest.mark.parametrize("curve", list(ALL_CURVES))
def test_oracle_vs_compiled_reference_random_and_edges(curve):
    _, plen, qlen = ALL_CURVES[curve]
    sc = np.concatenate([random_scalars(curve, 24, tag=7, below_q=False), edge_scalars(curve)])
    o1, s1 = oracle_smul(curve, sc)
    o2, s2 = ref_smul(curve, sc)
    assert (s1 == s2).all() and (o1 == o2).all()
    # variable base on the finite results, plus two off-curve points
    good = s1 == 0
    pts = o1[good].copy()
    sc2 = random_scalars(curve, pts.shape[0], tag=8, below_q=False)
    sc2[: edge_scalars(curve).shape[0]] = edge_scalars(curve)[: pts.shape[0]][: sc2.shape[0]]
    pts[1, -1] ^= 1
    pts[2, :plen] = 0xFF  # x >= p
    o3, s3 = oracle_smul(curve, sc2, pts)
    o4, s4 = ref_smul(curve, sc2, pts)
    assert (s3 == s4).all() and (o3 == o4).all()
    assert s3[1] == -1 and s3[2] == -1


@reference_answer
def ref_smul_long_scalars(curve, sc):
    n, slen = sc.shape
    out, st = np.zeros((n, 2 * ALL_CURVES[curve][1]), np.uint8), np.zeros(n, np.int8)
    ref_lib().ref_prj_pt_mul_batch(curve.encode(), n, _buf(sc), slen, None, _buf(out), _buf(st), 4)
    return out, st


def test_oracle_scalars_longer_than_q_match_reference():
    curve = "SECP256R1"
    rng = np.random.default_rng(5)
    for slen in (40, 64, 72):
        sc = rng.integers(0, 256, size=(4, slen), dtype=np.uint8)
        out1 = np.zeros((4, 64), np.uint8); st1 = np.zeros(4, np.int8)
        oracle_lib().ora_prj_pt_mul_batch(curve.encode(), 4, _buf(sc), slen, None, _buf(out1), _buf(st1), 4)
        out2, st2 = ref_smul_long_scalars(curve, sc)
        assert (out1 == out2).all() and (st1 == st2).all()
        # (k mod q) * G through python ints
        for i in range(4):
            k = int.from_bytes(sc[i].tobytes(), "big") % ORDER[curve]
            o, s = oracle_smul(curve, np.frombuffer(k.to_bytes(32, "big"), dtype=np.uint8))
            assert (o[0] == out1[i]).all()


def test_reference_multiplication_count():
    """M_ref of SURVEY.md §8d: 513 complete additions x 17 products (+ the on-curve checks)."""
    lib = oracle_lib()
    for curve, adds in (("SECP256R1", 513), ("SECP384R1", 769)):
        sc = random_scalars(curve, 1, tag=3)
        oracle_smul(curve, sc, nthreads=1)
        cnt = lib.ora_last_mul_count()
        assert adds * 17 <= cnt <= adds * 17 + 40, cnt

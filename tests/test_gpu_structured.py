"""The reference's structured key / signature records through the C ABI (SURVEY.md §8f.2) against the UNMODIFIED
reference (ec_structured_*_export_to_buf / _import_from_buf, ec_verify through oracle/ref_shim.c; its answers are stored
under tests/golden/reference/)."""
import ctypes
import hashlib

import numpy as np
import pytest

import libecc_b200
from common import ALL_CURVES, ORDER, PRIME, oracle_smul, random_scalars, ref_lib, reference_answer, rng

pytestmark = pytest.mark.gpu

_engines = {}


def engine(curve):
    if curve not in _engines:
        _engines[curve] = libecc_b200.Engine(curve, comb_window=8)
    return _engines[curve]


def _p(a):
    return np.ascontiguousarray(a).ctypes.data_as(ctypes.c_void_p)


@reference_answer
def ref_keygen(curve, priv: bytes):
    ref = ref_lib()
    prec, pubrec = np.zeros(255, np.uint8), np.zeros(255, np.uint8)
    pl, ql = ctypes.c_uint32(), ctypes.c_uint32()
    rc = ref.ref_structured_keygen(curve.encode(), priv, len(priv), _p(prec), ctypes.byref(pl), _p(pubrec),
                                   ctypes.byref(ql))
    return rc, prec[: pl.value].copy(), pubrec[: ql.value].copy()


@reference_answer
def ref_pub_import(curve, rec):
    ref = ref_lib()
    plen = ALL_CURVES[curve][1]
    aff = np.zeros(2 * plen, np.uint8)
    inf = ctypes.c_int()
    rec = np.ascontiguousarray(rec)
    rc = ref.ref_structured_pub_import(curve.encode(), _p(rec), rec.size, _p(aff), ctypes.byref(inf))
    return rc, aff, inf.value


@reference_answer
def ref_verify(curve, hash_name, sig_rec, pub_rec, msg: bytes):
    ref = ref_lib()
    sig_rec, pub_rec = np.ascontiguousarray(sig_rec), np.ascontiguousarray(pub_rec)
    return ref.ref_structured_verify(curve.encode(), hash_name.encode(), _p(sig_rec), sig_rec.size, _p(pub_rec),
                                     pub_rec.size, msg, len(msg))


HASH = {"SHA256": hashlib.sha256, "SHA384": hashlib.sha384, "SHA512": hashlib.sha512}


@pytest.mark.parametrize("curve", list(ALL_CURVES))
def test_structured_records_against_reference(curve):
    cid, plen, qlen = ALL_CURVES[curve]
    q, p = ORDER[curve], PRIME[curve]
    eng = engine(curve)
    hname = "SHA256" if qlen <= 32 else ("SHA384" if qlen <= 48 else "SHA512")
    hlen = HASH[hname]().digest_size
    n = 40
    privs = [int.from_bytes(r.tobytes(), "big") for r in random_scalars(curve, n, tag=901)] + [1, q - 1]
    recs = [ref_keygen(curve, x.to_bytes(qlen, "big")) for x in privs]
    assert all(r[0] == 0 for r in recs)
    priv_len = recs[0][1].size - 3
    assert priv_len >= qlen and recs[0][2].size == 3 + 3 * plen
    priv_recs = np.stack([r[1] for r in recs])
    ref_pub_recs = np.stack([r[2] for r in recs])          # Z != 1: the reference blinds its scalar multiplication
    want_aff = np.stack([ref_pub_import(curve, r)[1] for r in ref_pub_recs])

    # --- key pairs from structured private keys: x*G on K1, structured public keys out
    bad = priv_recs.copy()
    extra = []
    for k, mut in enumerate(("type", "alg", "curve", "x=q", "x=0", "lead")):
        r = priv_recs[k].copy()
        if mut == "type": r[0] = 0
        elif mut == "alg": r[1] = 2
        elif mut == "curve": r[2] ^= 0x40
        elif mut == "x=q": r[3:] = np.frombuffer(q.to_bytes(priv_len, "big"), np.uint8)
        elif mut == "x=0": r[3:] = 0
        elif mut == "lead":
            if priv_len == qlen:
                continue
            r[3] = 1
        extra.append((mut, r))
    all_priv = np.concatenate([bad, np.stack([r for _, r in extra])])
    pub_recs, st = eng.structured_key_pair_batch(all_priv, priv_len)
    assert (st[: len(privs)] == 0).all()
    for i in range(len(privs)):
        rc, aff, inf = ref_pub_import(curve, pub_recs[i])   # the reference imports OUR record
        assert rc == 0 and not inf and (aff == want_aff[i]).all()
    for (mut, _), s_ in zip(extra, st[len(privs):]):
        assert s_ == (1 if mut == "x=0" else -1), mut

    # --- structured public keys in (projective, Z != 1), affine out; rejected records like the reference
    muts = []
    for k, mut in enumerate(("type", "alg", "curve", "offcurve", "x>=p", "infinity", "z=0 junk")):
        r = ref_pub_recs[k].copy()
        if mut == "type": r[0] = 1
        elif mut == "alg": r[1] = 14
        elif mut == "curve": r[2] = (r[2] % 20) + 1
        elif mut == "offcurve": r[3 + plen - 1] ^= 1
        elif mut == "x>=p": r[3: 3 + plen] = np.frombuffer(p.to_bytes(plen, "big"), np.uint8)
        elif mut == "infinity":
            r[3:] = 0; r[3 + 2 * plen - 1] = 1             # (0, 1, 0)
        elif mut == "z=0 junk":
            r[3 + 2 * plen:] = 0                            # (X, Y, 0) with X != 0: not on the curve
        muts.append((mut, r))
    recs_in = np.concatenate([ref_pub_recs, np.stack([r for _, r in muts])])
    aff, st = eng.structured_pub_key_import_batch(recs_in)
    assert (st[: len(privs)] == 0).all() and (aff[: len(privs)] == want_aff).all()
    for (mut, r), s_, a_ in zip(muts, st[len(privs):], aff[len(privs):]):
        rc, raff, inf = ref_pub_import(curve, r)
        assert s_ == (-1 if rc else (1 if inf else 0)), mut
        assert (a_ == raff).all(), mut
    # export -> reference import round trip
    out = eng.structured_pub_key_export_batch(want_aff)
    for i in range(0, len(privs), 7):
        rc, raff, inf = ref_pub_import(curve, out[i])
        assert rc == 0 and (raff == want_aff[i]).all()

    # --- sign on structured private keys; the reference verifies our signature records against ITS key records
    g = rng(902)
    msgs = [g.bytes(int(g.integers(1, 80))) for _ in privs]
    dg = np.stack([np.frombuffer(HASH[hname](m).digest(), np.uint8) for m in msgs])
    nonces = random_scalars(curve, len(privs), tag=903)
    sig_recs, st = eng.ecdsa_sign_structured_batch(priv_recs, priv_len, nonces, hname, dg, hlen)
    assert (st == 0).all() and sig_recs.shape[1] == 3 + 2 * qlen
    for i in range(len(privs)):
        assert ref_verify(curve, hname, sig_recs[i], ref_pub_recs[i], msgs[i]) == 0

    # --- verify on structured records, corrupted ones included: verdicts of the reference
    vs, vp, vd, vm = [], [], [], []
    for i in range(len(privs)):
        s_, p_, d_ = sig_recs[i].copy(), ref_pub_recs[i].copy(), dg[i].copy()
        kind = i % 8
        if kind == 1: s_[3 + qlen - 1] ^= 1                 # r
        elif kind == 2: s_[0] = 14                          # signature says DECDSA
        elif kind == 3: s_[1] ^= 1                          # other hash
        elif kind == 4: s_[2] = (s_[2] % 20) + 1            # other curve
        elif kind == 5: p_[3 + 2 * plen - 1] ^= 1           # key off the curve
        elif kind == 6: p_[1] = 14                          # key for another algorithm
        elif kind == 7: d_[0] ^= 0x80
        vs.append(s_); vp.append(p_); vd.append(d_); vm.append(msgs[i])
    got = eng.ecdsa_verify_structured_batch(np.stack(vs), np.stack(vp), hname, np.stack(vd), hlen)
    for i in range(len(privs)):
        if i % 8 == 7:
            want = -1                                       # digest of a different message
        else:
            want = ref_verify(curve, hname, vs[i], vp[i], vm[i])
        assert got[i] == want, (i, i % 8)
    assert (got[::8] == 0).all() and (got[1::8] == -1).all()

    # --- a public key record holding the point at infinity: imported by the reference, and then v*Y vanishes
    inf_rec = ref_pub_recs[0].copy()
    inf_rec[3:] = 0; inf_rec[3 + 2 * plen - 1] = 1
    m = b"forged under the infinity key"
    e_bytes = HASH[hname](m).digest()
    e = int.from_bytes(e_bytes[: min(hlen, qlen)], "big") >> max(0, 8 * min(hlen, qlen) - q.bit_length())
    s_val = 0x1234567
    u = e * pow(s_val, -1, q) % q
    pt, _ = oracle_smul(curve, np.frombuffer(u.to_bytes(qlen, "big"), np.uint8))
    r_val = int.from_bytes(pt[0, :plen].tobytes(), "big") % q
    forged = np.concatenate([sig_recs[0][:3], np.frombuffer(r_val.to_bytes(qlen, "big") + s_val.to_bytes(qlen, "big"),
                                                            np.uint8)])
    other = forged.copy(); other[3 + qlen - 1] ^= 1
    got = eng.ecdsa_verify_structured_batch(np.stack([forged, other]), np.stack([inf_rec, inf_rec]), hname,
                                            np.stack([np.frombuffer(e_bytes, np.uint8)] * 2), hlen)
    want = [ref_verify(curve, hname, forged, inf_rec, m), ref_verify(curve, hname, other, inf_rec, m)]
    assert list(got) == want

"""BIP0340 verification (SURVEY.md §8f.4; reference: src/sig/bip0340.c:383-577).

CPU: the oracle port against the reference's own BIP0340 known-answer vectors (tests/golden/bip0340_kat.json, from
src/tests/bip0340_test_vectors.h) and against the unmodified reference on signatures the reference made (its
signatures and verdicts are stored under tests/golden/reference/); the host build of the kernel's algorithm against
the oracle.  GPU (`-m gpu`): the C ABI against the oracle / the reference, corrupted signatures included."""
import hashlib

import numpy as np
import pytest

from common import ALL_CURVES, HASHLEN, ORDER, PRIME, golden, hostsim_lib, hx, oracle_lib, random_scalars, ref_lib, reference_answer, rng, _buf

HASH = {"SHA256": hashlib.sha256, "SHA384": hashlib.sha384, "SHA512": hashlib.sha512}
TAG = b"BIP0340/challenge"


def challenge(hash_name, r, px, msg):
    """H(H(tag) || H(tag) || r || x(Y) || m): _bip0340_hash (sig/bip0340.c:45-69) as _bip0340_verify_init feeds it."""
    ht = HASH[hash_name](TAG).digest()
    return np.frombuffer(HASH[hash_name](ht + ht + bytes(r) + bytes(px) + msg).digest(), np.uint8)


def oracle_bip_verify(curve, sigs, pubs, digests, hlen):
    _, plen, qlen = ALL_CURVES[curve]
    sg = np.ascontiguousarray(sigs, dtype=np.uint8).reshape(-1, plen + qlen)
    n = sg.shape[0]
    v = np.zeros(n, dtype=np.int8)
    assert oracle_lib().ora_bip0340_verify_digest_batch(curve.encode(), n, _buf(sg), _buf(np.ascontiguousarray(pubs)),
                                                        _buf(np.ascontiguousarray(digests)), hlen, _buf(v), 8) == 0
    return v


def pack(msgs):
    blob = np.frombuffer(b"".join(msgs) or b"\0", dtype=np.uint8).copy()
    off = np.zeros(len(msgs) + 1, dtype=np.uint64)
    off[1:] = np.cumsum([len(m) for m in msgs])
    return blob, off


@reference_answer
def ref_sign(curve, hash_name, privs, msgs):
    ref = ref_lib()
    _, plen, qlen = ALL_CURVES[curve]
    n = len(msgs)
    blob, off = pack(msgs)
    sigs = np.zeros((n, plen + qlen), np.uint8)
    pubs = np.zeros((n, 2 * plen), np.uint8)
    st = np.zeros(n, np.int8)
    assert ref.ref_bip0340_sign_batch(curve.encode(), hash_name.encode(), n, _buf(privs), _buf(blob), _buf(off),
                                      _buf(sigs), _buf(pubs), _buf(st), 8) == 0 and (st == 0).all()
    return sigs, pubs


@reference_answer
def ref_verify(curve, hash_name, sigs, pubs, msgs):
    ref = ref_lib()
    n = sigs.shape[0]
    blob, off = pack(msgs)
    v = np.zeros(n, np.int8)
    assert ref.ref_bip0340_verify_batch(curve.encode(), hash_name.encode(), n, _buf(sigs), _buf(pubs), _buf(blob),
                                        _buf(off), _buf(v), 8) == 0
    return v


@reference_answer
def ref_verify_batch_all(curve, hash_name, sigs, pubs, msgs, scratch):
    """ec_verify_batch(..., BIP0340, ...) of the reference, with or without a scratch pad: 0 / -1."""
    blob, off = pack(msgs)
    return ref_lib().ref_bip0340_verify_batch_all(curve.encode(), hash_name.encode(), sigs.shape[0], _buf(sigs),
                                                  _buf(pubs), _buf(blob), _buf(off), scratch)


def workload(curve, n, tag, hash_name="SHA256"):
    """n reference-made signatures, 1/4 corrupted (r, r >= p, s, s = q, key off the curve, key negated (same x: still
    valid — the scheme only sees x(Y)), other message); digests and the reference's own verdicts."""
    _, plen, qlen = ALL_CURVES[curve]
    p, q = PRIME[curve], ORDER[curve]
    g = rng(tag)
    privs = random_scalars(curve, n, tag=tag + 1)
    msgs = [g.bytes(int(g.integers(0, 70))) for _ in range(n)]
    sigs, pubs = ref_sign(curve, hash_name, privs, msgs)
    for j, i in enumerate(range(0, n, 4)):
        kind = j % 7
        if kind == 0: sigs[i, plen - 1] ^= 1                                                  # r
        elif kind == 1: sigs[i, :plen] = np.frombuffer(p.to_bytes(plen, "big"), np.uint8)     # r = p: not a field element
        elif kind == 2: sigs[i, -1] ^= 1                                                      # s
        elif kind == 3: sigs[i, plen:] = np.frombuffer(q.to_bytes(qlen, "big"), np.uint8)     # s = q
        elif kind == 4: pubs[i, plen - 1] ^= 1                                                # key off the curve
        elif kind == 5:                                                                       # key negated: -Y has the same x
            y = int.from_bytes(pubs[i, plen:].tobytes(), "big")
            pubs[i, plen:] = np.frombuffer(((p - y) % p).to_bytes(plen, "big"), np.uint8)
        else: msgs[i] = msgs[i] + b"!"                                                        # another message
    want = ref_verify(curve, hash_name, sigs, pubs, msgs)
    dg = np.stack([challenge(hash_name, sigs[i, :plen], pubs[i, :plen], msgs[i]) for i in range(n)])
    kinds = np.array([(j % 7) for j in range(len(range(0, n, 4)))])
    assert (want[::4][kinds != 5] == -1).all() and (want[::4][kinds == 5] == 0).all()
    assert (np.delete(want, np.s_[::4]) == 0).all()
    return sigs, pubs, dg, dg.shape[1], want


def test_oracle_against_reference_kats():
    vecs = golden("bip0340_kat.json")
    assert len(vecs) >= 4 and {v["curve"] for v in vecs} == {"SECP256K1"}
    for v in vecs:
        assert v["ref_verdict"] == 0
        plen = ALL_CURVES[v["curve"]][1]
        sig, pub, msg = hx(v["sig"]), hx(v["pub"]), bytes(hx(v["msg"]))
        dg = challenge(v["hash"], sig[:plen], pub[:plen], msg)
        assert dg.tobytes().hex() == v["digest_challenge"]          # the tagged hash as the reference computes it
        assert oracle_bip_verify(v["curve"], sig, pub, dg, len(dg))[0] == 0, v["name"]
        bad = sig.copy(); bad[-1] ^= 1
        assert oracle_bip_verify(v["curve"], bad, pub, dg, len(dg))[0] == -1


@pytest.mark.parametrize("curve,hash_name", [("SECP256K1", "SHA256"), ("SECP256R1", "SHA512"), ("FRP256V1", "SHA256"),
                                             ("SECP384R1", "SHA384"), ("SECP192R1", "SHA256")])
def test_oracle_and_host_algorithm_against_reference(curve, hash_name):
    sigs, pubs, dg, hlen, want = workload(curve, 28, 8100, hash_name)
    assert (oracle_bip_verify(curve, sigs, pubs, dg, hlen) == want).all()
    got = np.zeros(len(want), np.int8)
    assert hostsim_lib().hostsim_bip0340_verify_batch(ALL_CURVES[curve][0], 4, len(want), _buf(sigs), _buf(pubs), _buf(dg),
                                                      hlen, _buf(got)) == 0
    assert (got == want).all()


@pytest.mark.gpu
@pytest.mark.parametrize("curve", list(ALL_CURVES))
def test_gpu_bip0340_verify(curve):
    import libecc_b200
    _, plen, qlen = ALL_CURVES[curve]
    eng = libecc_b200.Engine(curve, comb_window=8)
    for tag, hname in ((8300, "SHA256"), (8400, "SHA512")):
        sigs, pubs, dg, hlen, want = workload(curve, 64, tag, hname)
        assert (oracle_bip_verify(curve, sigs, pubs, dg, hlen) == want).all()
        got = eng.bip0340_verify_batch(sigs, pubs, dg, hlen)
        assert (got == want).all(), (curve, hname)
    for v in golden("bip0340_kat.json"):
        if v["curve"] == curve:
            assert eng.bip0340_verify_batch(hx(v["sig"]), hx(v["pub"]), hx(v["digest_challenge"]), HASHLEN[v["hash"]])[0] == 0
    eng.close()


@pytest.mark.gpu
def test_gpu_bip0340_large_batch():
    """2^16 signatures through the chunked host pipeline: tiled reference-made signatures, every 4th corrupted."""
    import libecc_b200
    curve = "SECP256K1"
    sigs, pubs, dg, hlen, want = workload(curve, 256, 8500)
    reps = 1 << 8
    eng = libecc_b200.Engine(curve)
    got = eng.bip0340_verify_batch(np.tile(sigs, (reps, 1)), np.tile(pubs, (reps, 1)), np.tile(dg, (reps, 1)), hlen)
    assert (got == np.tile(want, reps)).all()
    eng.close()

"""ECFSDSA verification (SURVEY.md §8f.4; reference: src/sig/ecfsdsa.c:416-610).

CPU: the oracle port against the reference's own ECFSDSA known-answer vectors (tests/golden/ecfsdsa_kat.json) and
against the unmodified reference on signatures the reference made (its signatures and verdicts are stored under
tests/golden/reference/); the host build of the kernel's algorithm against the oracle.  GPU (`-m gpu`): the C ABI
against the oracle / the reference, corrupted signatures included."""
import ctypes
import hashlib

import numpy as np
import pytest

from common import ALL_CURVES, HASHLEN, ORDER, PRIME, golden, hostsim_lib, hx, oracle_lib, random_scalars, ref_lib, reference_answer, rng, _buf

HASH = {"SHA224": hashlib.sha224, "SHA256": hashlib.sha256, "SHA384": hashlib.sha384, "SHA512": hashlib.sha512}


def oracle_fs_verify(curve, sigs, pubs, digests, hlen):
    _, plen, qlen = ALL_CURVES[curve]
    sg = np.ascontiguousarray(sigs, dtype=np.uint8).reshape(-1, 2 * plen + qlen)
    n = sg.shape[0]
    v = np.zeros(n, dtype=np.int8)
    lib = oracle_lib()
    assert lib.ora_ecfsdsa_verify_digest_batch(curve.encode(), n, _buf(sg), _buf(np.ascontiguousarray(pubs)),
                                               _buf(np.ascontiguousarray(digests)), hlen, _buf(v), 8) == 0
    return v


def ref_sign(curve, hash_name, privs, msgs):
    """Signatures and public keys made by the unmodified reference (random nonces), and the packed messages."""
    n = len(msgs)
    blob = np.frombuffer(b"".join(msgs), dtype=np.uint8).copy()
    off = np.zeros(n + 1, dtype=np.uint64)
    off[1:] = np.cumsum([len(m) for m in msgs])
    return ref_sign_raw(curve, hash_name, privs, msgs) + (blob, off)


@reference_answer
def ref_sign_raw(curve, hash_name, privs, msgs):
    ref = ref_lib()
    _, plen, qlen = ALL_CURVES[curve]
    n = len(msgs)
    blob = np.frombuffer(b"".join(msgs), dtype=np.uint8).copy()
    off = np.zeros(n + 1, dtype=np.uint64)
    off[1:] = np.cumsum([len(m) for m in msgs])
    sigs = np.zeros((n, 2 * plen + qlen), np.uint8)
    pubs = np.zeros((n, 2 * plen), np.uint8)
    st = np.zeros(n, np.int8)
    assert ref.ref_ecfsdsa_sign_batch(curve.encode(), hash_name.encode(), n, _buf(privs), _buf(blob), _buf(off),
                                      _buf(sigs), _buf(pubs), _buf(st), 8) == 0 and (st == 0).all()
    return sigs, pubs


@reference_answer
def ref_verify(curve, hash_name, sigs, pubs, blob, off):
    ref = ref_lib()
    n = sigs.shape[0]
    v = np.zeros(n, np.int8)
    assert ref.ref_ecfsdsa_verify_batch(curve.encode(), hash_name.encode(), n, _buf(sigs), _buf(pubs), _buf(blob),
                                        _buf(off), _buf(v), 8) == 0
    return v


@reference_answer
def ref_verify_batch_all(curve, hash_name, sigs, pubs, blob, off):
    """ec_verify_batch(..., ECFSDSA, ...) of the reference without a scratch pad: 0 / -1."""
    return ref_lib().ref_ecfsdsa_verify_batch_all(curve.encode(), hash_name.encode(), sigs.shape[0], _buf(sigs), _buf(pubs),
                                                  _buf(blob), _buf(off), 0)


def workload(curve, n, tag, hash_name=None):
    """n reference-made signatures, 1/4 of them corrupted (r off the curve, r another point, s, s = 0, s = q, key,
    message); returns sigs, pubs, digests H(r || m), hlen and the reference's verdicts."""
    _, plen, qlen = ALL_CURVES[curve]
    q = ORDER[curve]
    hash_name = hash_name or ("SHA256" if qlen <= 32 else ("SHA384" if qlen <= 48 else "SHA512"))
    g = rng(tag)
    privs = random_scalars(curve, n, tag=tag + 1)
    msgs = [g.bytes(int(g.integers(0, 70))) for _ in range(n)]
    sigs, pubs, blob, off = ref_sign(curve, hash_name, privs, msgs)
    for j, i in enumerate(range(0, n, 4)):
        kind = j % 7
        if kind == 0: sigs[i, plen - 1] ^= 1                                  # r_x: off the curve
        elif kind == 1: sigs[i, :2 * plen] = sigs[(i + 1) % n, :2 * plen]     # r: a valid point, the wrong one
        elif kind == 2: sigs[i, -1] ^= 1                                      # s
        elif kind == 3: sigs[i, 2 * plen:] = 0                                # s = 0
        elif kind == 4: sigs[i, 2 * plen:] = np.frombuffer(q.to_bytes(qlen, "big"), np.uint8)
        elif kind == 5: pubs[i, 2 * plen - 1] ^= 1                            # key off the curve
        else: msgs[i] = msgs[i] + b"!"                                         # another message
    blob = np.frombuffer(b"".join(msgs), dtype=np.uint8).copy()
    off = np.zeros(n + 1, dtype=np.uint64)
    off[1:] = np.cumsum([len(m) for m in msgs])
    want = ref_verify(curve, hash_name, sigs, pubs, blob, off)
    dg = np.stack([np.frombuffer(HASH[hash_name](sigs[i, :2 * plen].tobytes() + msgs[i]).digest(), np.uint8)
                   for i in range(n)])
    assert (want[::4] == -1).all() and (np.delete(want, np.s_[::4]) == 0).all()
    return sigs, pubs, dg, dg.shape[1], want


def test_oracle_against_reference_kats():
    vecs = golden("ecfsdsa_kat.json")
    assert {v["curve"] for v in vecs} >= {"FRP256V1", "SECP256R1", "SECP384R1", "SECP521R1", "BRAINPOOLP256R1"}
    for v in vecs:
        assert v["ref_verdict"] == 0
        hl = HASHLEN[v["hash"]]
        assert oracle_fs_verify(v["curve"], hx(v["sig"]), hx(v["pub"]), hx(v["digest_rm"]), hl)[0] == 0, v["name"]
        bad = hx(v["sig"]).copy(); bad[-1] ^= 1
        assert oracle_fs_verify(v["curve"], bad, hx(v["pub"]), hx(v["digest_rm"]), hl)[0] == -1


@pytest.mark.parametrize("curve,hash_name", [("FRP256V1", "SHA256"), ("SECP256R1", "SHA512"), ("SECP384R1", "SHA384"),
                                             ("SECP521R1", "SHA512"), ("SECP224R1", "SHA256"), ("SECP256K1", "SHA256"),
                                             ("SECP192R1", "SHA512")])
def test_oracle_and_host_algorithm_against_reference(curve, hash_name):
    """Digests longer than the order (SHA-512 on P-256, SHA-256 on P-224) exercise the full-digest reduction."""
    sigs, pubs, dg, hlen, want = workload(curve, 24, 7100, hash_name)
    assert (oracle_fs_verify(curve, sigs, pubs, dg, hlen) == want).all()
    lib = hostsim_lib()
    got = np.zeros(len(want), np.int8)
    assert lib.hostsim_ecfsdsa_verify_batch(ALL_CURVES[curve][0], 4, len(want), _buf(sigs), _buf(pubs), _buf(dg), hlen,
                                            _buf(got)) == 0
    assert (got == want).all()


def test_reference_batch_entry_point_agrees_on_valid_batches():
    """ec_verify_batch(…, ECFSDSA, …) of the reference (no scratch pad) returns 0 for an all-valid batch and -1 once a
    signature is corrupted — the aggregate of the per-item verdicts this engine reports."""
    curve, hash_name = "FRP256V1", "SHA256"
    privs = random_scalars(curve, 6, tag=7201)
    msgs = [b"batch message %d" % i for i in range(6)]
    sigs, pubs, blob, off = ref_sign(curve, hash_name, privs, msgs)
    assert ref_verify_batch_all(curve, hash_name, sigs, pubs, blob, off) == 0
    sigs[2, -1] ^= 1
    assert ref_verify_batch_all(curve, hash_name, sigs, pubs, blob, off) == -1
    assert list(ref_verify(curve, hash_name, sigs, pubs, blob, off)) == [0, 0, -1, 0, 0, 0]


@pytest.mark.gpu
@pytest.mark.parametrize("curve", list(ALL_CURVES))
def test_gpu_ecfsdsa_verify(curve):
    import libecc_b200
    eng = libecc_b200.Engine(curve, comb_window=8)
    for tag, hname in ((7300, None), (7400, "SHA512")):
        sigs, pubs, dg, hlen, want = workload(curve, 64, tag, hname)
        assert (oracle_fs_verify(curve, sigs, pubs, dg, hlen) == want).all()
        got = eng.ecfsdsa_verify_batch(sigs, pubs, dg, hlen)
        assert (got == want).all(), (curve, hname)
    for v in golden("ecfsdsa_kat.json"):
        if v["curve"] == curve:
            assert eng.ecfsdsa_verify_batch(hx(v["sig"]), hx(v["pub"]), hx(v["digest_rm"]), HASHLEN[v["hash"]])[0] == 0
    eng.close()


@pytest.mark.gpu
def test_gpu_ecfsdsa_large_batch_properties():
    """2^16 signatures through the chunked host pipeline: tiled reference-made signatures, every 4th corrupted."""
    import libecc_b200
    curve = "FRP256V1"
    sigs, pubs, dg, hlen, want = workload(curve, 256, 7500)
    reps = 1 << 8
    eng = libecc_b200.Engine(curve)
    got = eng.ecfsdsa_verify_batch(np.tile(sigs, (reps, 1)), np.tile(pubs, (reps, 1)), np.tile(dg, (reps, 1)), hlen)
    assert (got == np.tile(want, reps)).all()
    eng.close()

"""The generic double-scalar multiplication W = a*G + b*Y (eccb200_double_smul_batch) and, on top of it, ECSDSA /
ECOSDSA verification as the reference defines it (src/sig/ecsdsa_common.c:425-609): s in ]0, q[, e = -(OS2I(r) mod q)
!= 0, W' = sG + eY, r' = H(W'x [|| W'y] || m) == r.  The EC part runs on the device; hashing the recomputed point stays
with the caller, as in the reference (src/hash).

CPU: the oracle's double-scalar multiplication + this wrapper against the unmodified reference's verdicts on signatures
the reference made (its signatures and verdicts are stored under tests/golden/reference/); the host build of the
kernel's algorithm against the oracle.  GPU (`-m gpu`): the C ABI."""
import hashlib

import numpy as np
import pytest

from common import ALL_CURVES, ORDER, PRIME, hostsim_lib, oracle_lib, oracle_smul, random_scalars, ref_lib, reference_answer, rng, _buf

HASH = {"SHA256": hashlib.sha256, "SHA384": hashlib.sha384, "SHA512": hashlib.sha512, "SHA224": hashlib.sha224}


def pack(msgs):
    blob = np.frombuffer(b"".join(msgs) or b"\0", dtype=np.uint8).copy()
    off = np.zeros(len(msgs) + 1, dtype=np.uint64)
    off[1:] = np.cumsum([len(m) for m in msgs])
    return blob, off


@reference_answer
def ref_siglen(curve, alg, hash_name):
    import ctypes
    sl = ctypes.c_uint32()
    assert ref_lib().ref_sig_len(curve.encode(), alg.encode(), hash_name.encode(), ctypes.byref(sl)) == 0
    return sl.value


@reference_answer
def ref_sign(curve, alg, hash_name, privs, msgs):
    _, plen, qlen = ALL_CURVES[curve]
    n = len(msgs)
    sl = ref_siglen(curve, alg, hash_name)
    blob, off = pack(msgs)
    sigs = np.zeros((n, sl), np.uint8)
    pubs = np.zeros((n, 2 * plen), np.uint8)
    st = np.zeros(n, np.int8)
    assert ref_lib().ref_sig_sign_batch(curve.encode(), alg.encode(), hash_name.encode(), n, _buf(privs), _buf(blob),
                                        _buf(off), _buf(sigs), _buf(pubs), _buf(st), 8) == 0 and (st == 0).all()
    return sigs, pubs


@reference_answer
def ref_verify(curve, alg, hash_name, sigs, pubs, msgs):
    n = sigs.shape[0]
    blob, off = pack(msgs)
    v = np.zeros(n, np.int8)
    assert ref_lib().ref_sig_verify_batch(curve.encode(), alg.encode(), hash_name.encode(), n, _buf(sigs), _buf(pubs),
                                          _buf(blob), _buf(off), _buf(v), 8) == 0
    return v


def oracle_double_smul(curve, ab, pubs):
    _, plen, qlen = ALL_CURVES[curve]
    ab = np.ascontiguousarray(ab, dtype=np.uint8).reshape(-1, 2 * qlen)
    n = ab.shape[0]
    out = np.zeros((n, 2 * plen), np.uint8)
    st = np.zeros(n, np.int8)
    assert oracle_lib().ora_double_smul_batch(curve.encode(), n, _buf(ab), _buf(np.ascontiguousarray(pubs)), _buf(out),
                                              _buf(st), 8) == 0
    return out, st


def ecsdsa_verify(curve, hash_name, optimized, sigs, pubs, msgs, double_smul):
    """The reference's __ecsdsa_verify_init / _finalize around a double-scalar multiplication back end."""
    _, plen, qlen = ALL_CURVES[curve]
    q = ORDER[curve]
    hl = HASH[hash_name]().digest_size
    n = sigs.shape[0]
    verdict = np.full(n, -1, np.int8)
    ab = np.zeros((n, 2 * qlen), np.uint8)
    live = np.zeros(n, bool)
    for i in range(n):
        r = int.from_bytes(sigs[i, :hl].tobytes(), "big")
        s = int.from_bytes(sigs[i, hl:].tobytes(), "big")
        if not (0 < s < q):                                    # 1. s in ]0, q[ (:474-478)
            continue
        e = (-r) % q                                           # 2. e = -r mod q (:486-488)
        if e == 0:                                             # 3. (:491-492)
            continue
        ab[i, :qlen] = np.frombuffer(s.to_bytes(qlen, "big"), np.uint8)
        ab[i, qlen:] = np.frombuffer(e.to_bytes(qlen, "big"), np.uint8)
        live[i] = True
    w, st = double_smul(ab, pubs)                              # 4. W' = sG + eY, unique representative (:495-498)
    for i in range(n):
        if not live[i] or st[i] != 0:
            continue
        pre = w[i, :plen].tobytes() if optimized else w[i].tobytes()
        rp = HASH[hash_name](pre + msgs[i]).digest()           # 5. r' = H(W'x [|| W'y] || m) (:500-520), 6. r == r'
        verdict[i] = 0 if rp == sigs[i, :hl].tobytes() else -1
    return verdict


def workload(curve, alg, hash_name, n, tag):
    _, plen, qlen = ALL_CURVES[curve]
    q = ORDER[curve]
    hl = HASH[hash_name]().digest_size
    g = rng(tag)
    privs = random_scalars(curve, n, tag=tag + 1)
    msgs = [g.bytes(int(g.integers(0, 70))) for _ in range(n)]
    sigs, pubs = ref_sign(curve, alg, hash_name, privs, msgs)
    assert sigs.shape[1] == hl + qlen
    for j, i in enumerate(range(0, n, 4)):
        kind = j % 6
        if kind == 0: sigs[i, 3] ^= 1                                                   # r
        elif kind == 1: sigs[i, -1] ^= 1                                                # s
        elif kind == 2: sigs[i, hl:] = 0                                                # s = 0
        elif kind == 3: sigs[i, hl:] = np.frombuffer(q.to_bytes(qlen, "big"), np.uint8)  # s = q
        elif kind == 4: pubs[i, plen - 1] ^= 1                                          # key off the curve
        else: msgs[i] = msgs[i] + b"!"                                                  # another message
    want = ref_verify(curve, alg, hash_name, sigs, pubs, msgs)
    assert (want[::4] == -1).all() and (np.delete(want, np.s_[::4]) == 0).all()
    return sigs, pubs, msgs, want


CASES = [("SECP256R1", "ECSDSA", "SHA256"), ("FRP256V1", "ECOSDSA", "SHA256"), ("SECP384R1", "ECSDSA", "SHA384"),
         ("BRAINPOOLP256R1", "ECOSDSA", "SHA512"), ("SECP521R1", "ECSDSA", "SHA512"), ("SECP224R1", "ECSDSA", "SHA224")]


@pytest.mark.parametrize("curve,alg,hash_name", CASES)
def test_oracle_and_host_algorithm_against_reference(curve, alg, hash_name):
    sigs, pubs, msgs, want = workload(curve, alg, hash_name, 24, 9100)
    got = ecsdsa_verify(curve, hash_name, alg == "ECOSDSA", sigs, pubs, msgs, lambda ab, pk: oracle_double_smul(curve, ab, pk))
    assert (got == want).all()

    def host(ab, pk):
        _, plen, _ = ALL_CURVES[curve]
        out = np.zeros((ab.shape[0], 2 * plen), np.uint8)
        st = np.zeros(ab.shape[0], np.int8)
        assert hostsim_lib().hostsim_double_smul_batch(ALL_CURVES[curve][0], 4, ab.shape[0], _buf(ab), _buf(pk), _buf(out),
                                                       _buf(st)) == 0
        return out, st
    assert (ecsdsa_verify(curve, hash_name, alg == "ECOSDSA", sigs, pubs, msgs, host) == want).all()


def test_double_smul_edge_cases_on_the_oracle_and_host_build():
    """a = 0, b = 0, both 0 (infinity), a*G = -b*Y (infinity), scalars >= q, key off the curve."""
    curve = "SECP256R1"
    cid, plen, qlen = ALL_CURVES[curve]
    q = ORDER[curve]
    G, _ = oracle_smul(curve, np.frombuffer((1).to_bytes(qlen, "big"), np.uint8).reshape(1, qlen))
    P5, _ = oracle_smul(curve, np.frombuffer((5).to_bytes(qlen, "big"), np.uint8).reshape(1, qlen))
    be = lambda v: np.frombuffer((v % (1 << (8 * qlen))).to_bytes(qlen, "big"), np.uint8)
    rows = [(7, 0, P5[0]), (0, 9, P5[0]), (0, 0, P5[0]), (5, q - 1, P5[0]), (q + 3, q + 4, P5[0]), ((1 << 256) - 1, 2, G[0]),
            (3, 4, G[0])]
    ab = np.stack([np.concatenate([be(a), be(b)]) for a, b, _ in rows])
    pk = np.stack([p for _, _, p in rows]).copy()
    bad = pk[-1].copy(); bad[plen - 1] ^= 1
    ab = np.concatenate([ab, ab[-1:]]); pk = np.concatenate([pk, bad[None]])
    out, st = oracle_double_smul(curve, ab, pk)
    assert list(st) == [0, 0, 1, 1, 0, 0, 0, -1]
    want7, _ = oracle_smul(curve, be(7).reshape(1, qlen))
    want45, _ = oracle_smul(curve, be(45).reshape(1, qlen))        # 0*G + 9*(5G)
    want23, _ = oracle_smul(curve, be(3 + 4 * 5).reshape(1, qlen))  # (q+3)G + (q+4)(5G)
    assert (out[0] == want7[0]).all() and (out[1] == want45[0]).all() and (out[4] == want23[0]).all()
    hout = np.zeros_like(out); hst = np.zeros_like(st)
    assert hostsim_lib().hostsim_double_smul_batch(cid, 5, len(st), _buf(ab), _buf(pk), _buf(hout), _buf(hst)) == 0
    assert (hst == st).all() and (hout == out).all()


@pytest.mark.gpu
@pytest.mark.parametrize("curve", list(ALL_CURVES))
def test_gpu_double_smul_against_oracle(curve):
    import libecc_b200
    cid, plen, qlen = ALL_CURVES[curve]
    q = ORDER[curve]
    n = 600
    g = rng(9300)
    ab = g.integers(0, 256, size=(n, 2 * qlen), dtype=np.uint8)
    top = (1 << (q.bit_length() - 8 * (qlen - 1))) - 1
    ab[:, 0] &= top; ab[:, qlen] &= top
    pts, _ = oracle_smul(curve, random_scalars(curve, n, tag=9301))
    ab[0, :qlen] = 0; ab[1, qlen:] = 0; ab[2] = 0                       # a = 0, b = 0, both
    ab[3, :qlen] = ab[3, qlen:]; pts[3] = oracle_smul(curve, np.frombuffer((q - 1).to_bytes(qlen, "big"), np.uint8).reshape(1, qlen))[0][0]
    pts[5, plen - 1] ^= 1                                               # key off the curve
    want, wst = oracle_double_smul(curve, ab, pts)
    assert wst[2] == 1 and wst[3] == 1 and wst[5] == -1                 # aG + a(q-1)G = infinity
    eng = libecc_b200.Engine(curve, comb_window=9)
    got, gst = eng.double_smul_batch(ab, pts)
    eng.close()
    assert (gst == wst).all() and (got == want).all()


@pytest.mark.gpu
@pytest.mark.parametrize("curve,alg,hash_name", CASES)
def test_gpu_ecsdsa_verify_against_reference(curve, alg, hash_name):
    import libecc_b200
    sigs, pubs, msgs, want = workload(curve, alg, hash_name, 96, 9400)
    eng = libecc_b200.Engine(curve, comb_window=10)
    got = ecsdsa_verify(curve, hash_name, alg == "ECOSDSA", sigs, pubs, msgs, eng.double_smul_batch)
    eng.close()
    assert (got == want).all()

"""ECFSDSA batch verification as ONE multi-scalar multiplication (SURVEY.md §8f.4; reference: _ecfsdsa_verify_batch
src/sig/ecfsdsa.c:814-1055 with the Bos-Coster heap src/sig/sig_algs.c:1052).

CPU: the coefficient generator against an independent ChaCha20, the signed-digit recoding against integers, and the
stages of the device algorithm (host build of msm_core.cuh) against the reference's own verify_batch entry point and its
per-item verdicts.  GPU (`-m gpu`): the C ABI against the same."""
import ctypes
import os

import numpy as np
import pytest

from common import ALL_CURVES, ORDER, hostsim_lib, ref_lib, reference_answer, rng, _buf
from test_ecfsdsa import workload

SEED = bytes(range(7, 39))


@reference_answer
def ref_batch_all(curve, hash_name, sigs, pubs, msgs):
    """The reference's ec_verify_batch(..., ECFSDSA, ...) on the same batch: 0 / -1."""
    ref = ref_lib()
    blob = np.frombuffer(b"".join(msgs), dtype=np.uint8).copy() if sum(map(len, msgs)) else np.zeros(1, np.uint8)
    off = np.zeros(len(msgs) + 1, dtype=np.uint64)
    off[1:] = np.cumsum([len(m) for m in msgs])
    return ref.ref_ecfsdsa_verify_batch_all(curve.encode(), hash_name.encode(), len(msgs), _buf(sigs), _buf(pubs),
                                            _buf(blob), _buf(off), 0)


def host_msm(curve, c, sigs, pubs, dg, hlen, seed=SEED):
    lib = hostsim_lib()
    ok = ctypes.c_int(-1)
    stats = (ctypes.c_ulonglong * 5)()
    sg = np.ascontiguousarray(sigs, dtype=np.uint8)
    n = sg.shape[0]
    assert lib.hostsim_ecfsdsa_msm(ALL_CURVES[curve][0], c, n, _buf(sg), _buf(np.ascontiguousarray(pubs)),
                                   _buf(np.ascontiguousarray(dg)), hlen, seed, ctypes.byref(ok), stats) == 0
    return ok.value, list(stats)


def test_coefficients_are_a_chacha20_stream():
    from cryptography.hazmat.primitives.ciphers import Cipher, algorithms
    lib = hostsim_lib()
    for i in (0, 1, 2, 12345, (1 << 32) - 1, 1 << 32, (7 << 32) + 9):
        out = (ctypes.c_uint32 * 8)()
        lib.hostsim_msm_coefficient(SEED, ctypes.c_uint64(i), out)
        nonce = (i & 0xFFFFFFFF).to_bytes(4, "little") + (i >> 32).to_bytes(4, "little") + b"MSM1" + bytes(4)
        ks = Cipher(algorithms.ChaCha20(SEED, nonce), mode=None).encryptor().update(bytes(32))
        assert bytes(out) == ks, i


@pytest.mark.parametrize("c", [2, 3, 5, 8, 13, 16])
def test_signed_digit_recoding(c):
    lib = hostsim_lib()
    g = rng(8800 + c)
    for bits, nwords in ((192, 6), (256, 8), (521, 17)):
        ks = [0, 1, (1 << bits) - 1, 1 << (bits - 1), (1 << (c - 1)), (1 << (c - 1)) + 1] + \
             [int.from_bytes(g.bytes((bits + 7) // 8), "big") >> ((-bits) % 8) for _ in range(40)]
        for k in ks:
            words = (ctypes.c_uint32 * nwords)(*[(k >> (32 * i)) & 0xFFFFFFFF for i in range(nwords)])
            digits = (ctypes.c_int * 600)()
            nwin = lib.hostsim_msm_digits(words, nwords, bits, c, digits)
            assert nwin == bits // c + 1
            ds = list(digits)[:nwin]
            assert all(abs(d) <= 1 << (c - 1) for d in ds)
            assert sum(d << (c * w) for w, d in enumerate(ds)) == k


@pytest.mark.parametrize("curve,hash_name,c", [("FRP256V1", "SHA256", 4), ("SECP256R1", "SHA512", 7),
                                               ("SECP384R1", "SHA384", 5), ("SECP521R1", "SHA512", 6),
                                               ("SECP224R1", "SHA256", 3), ("SECP192R1", "SHA512", 9)])
def test_host_algorithm_against_reference(curve, hash_name, c):
    sigs, pubs, dg, hlen, want = workload(curve, 28, 8900, hash_name)
    good = np.flatnonzero(want == 0)
    ok, stats = host_msm(curve, c, sigs[good], pubs[good], dg[good], hlen)
    assert ok == 1
    # every kind of corruption of test_ecfsdsa.workload sinks the batch, alone among valid signatures
    for bad in np.flatnonzero(want != 0):
        idx = np.concatenate([good[:5], [bad], good[5:9]])
        assert host_msm(curve, c, sigs[idx], pubs[idx], dg[idx], hlen)[0] == 0, (curve, int(bad))
    # a single signature, and an empty batch
    assert host_msm(curve, c, sigs[good[:1]], pubs[good[:1]], dg[good[:1]], hlen)[0] == 1
    assert host_msm(curve, c, sigs[:0], pubs[:0], dg[:0], hlen)[0] == 0
    # the same points many times over (one signature repeated; one key for all): buckets then hold equal points and the
    # accumulation takes its doubling branch
    rep = np.repeat(good[:3], 12)
    ok, stats = host_msm(curve, 2, sigs[rep], pubs[rep], dg[rep], hlen)
    assert ok == 1
    rep[7] = np.flatnonzero(want != 0)[2]
    assert host_msm(curve, 2, sigs[rep], pubs[rep], dg[rep], hlen)[0] == 0


def test_host_algorithm_and_reference_batch_entry_point():
    """ec_verify_batch(…, ECFSDSA, …) of the unmodified reference and the multi-scalar-multiplication form agree on
    valid and on corrupted batches (different random coefficients, same verdict)."""
    from test_ecfsdsa import ref_sign, HASH
    from common import random_scalars
    curve, hash_name = "FRP256V1", "SHA256"
    _, plen, qlen = ALL_CURVES[curve]
    n = 12
    privs = random_scalars(curve, n, tag=9001)
    msgs = [b"msm batch %d" % i for i in range(n)]
    sigs, pubs, blob, off = ref_sign(curve, hash_name, privs, msgs)
    dg = np.stack([np.frombuffer(HASH[hash_name](sigs[i, :2 * plen].tobytes() + msgs[i]).digest(), np.uint8)
                   for i in range(n)])
    assert ref_batch_all(curve, hash_name, sigs, pubs, msgs) == 0
    for seed in (SEED, bytes(32), os.urandom(32)):
        assert host_msm(curve, 6, sigs, pubs, dg, 32, seed)[0] == 1
    sigs[5, -1] ^= 1
    assert ref_batch_all(curve, hash_name, sigs, pubs, msgs) == -1
    assert host_msm(curve, 6, sigs, pubs, dg, 32)[0] == 0
    # s = 0 is not excluded by the batch function's range check (s < q only, sig/ecfsdsa.c:919-921): the verdict then
    # comes from the equation, in the reference and here alike
    sigs[5, -1] ^= 1
    sigs[3, 2 * plen:] = 0
    assert ref_batch_all(curve, hash_name, sigs, pubs, msgs) == -1
    assert host_msm(curve, 6, sigs, pubs, dg, 32)[0] == 0


def test_work_per_signature():
    """The count DESIGN.md quotes: field products per signature of the bucket method at the window the library picks
    for 2^20 signatures (c = 16) cannot be run on a CPU; at c = 8 and n = 256 the accumulation already shows the shape:
    one mixed addition per non-zero digit."""
    curve = "FRP256V1"
    sigs, pubs, dg, hlen, want = workload(curve, 64, 9100)
    good = np.flatnonzero(want == 0)
    rep = np.tile(good, 6)[:256]
    ok, (adds, buckets, nwin, muls, fullest) = host_msm(curve, 8, sigs[rep], pubs[rep], dg[rep], hlen)
    assert ok == 1 and nwin == 32 and buckets == 32 * 128
    n = len(rep)
    # W_i: 127-bit coefficients -> at most 16 non-zero digits; Y_i and G (folded to 255 bits): at most 32
    assert adds <= n * (16 + 32) + 32 and adds >= n * (16 + 32) * 0.97
    assert muls / n < 1500
    # no bucket collects a disproportionate share of the points (one thread adds up one bucket): mean load is
    # adds / buckets ~ 3; the top windows must not stand out
    assert fullest <= 20


# ------------------------------------------------------------------------------------------------------------- BIP0340


def host_msm_bip(curve, c, sigs, pubs, dg, hlen, seed=SEED):
    lib = hostsim_lib()
    ok = ctypes.c_int(-1)
    sg = np.ascontiguousarray(sigs, dtype=np.uint8)
    rc = lib.hostsim_bip0340_msm(ALL_CURVES[curve][0], c, sg.shape[0], _buf(sg), _buf(np.ascontiguousarray(pubs)),
                                 _buf(np.ascontiguousarray(dg)), hlen, seed, ctypes.byref(ok), None)
    return rc, ok.value


def test_square_root_of_the_lift():
    from common import PRIME
    lib = hostsim_lib()
    g = rng(9500)
    for curve in ("SECP256K1", "FRP256V1", "SECP384R1", "SECP521R1", "BRAINPOOLP512R1", "SECP192R1"):
        p = PRIME[curve]
        plen = ALL_CURVES[curve][1]
        assert p % 4 == 3
        for x in [0, 1, 4, p - 1] + [int.from_bytes(g.bytes(plen), "big") % p for _ in range(12)]:
            out = (ctypes.c_uint8 * plen)()
            rc = lib.hostsim_fp_sqrt(ALL_CURVES[curve][0], x.to_bytes(plen, "big"), out)
            is_square = x == 0 or pow(x, (p - 1) // 2, p) == 1
            assert rc == (1 if is_square else 0), (curve, x)
            if is_square:
                assert pow(int.from_bytes(bytes(out), "big"), 2, p) == x
    out = (ctypes.c_uint8 * 28)()
    assert lib.hostsim_fp_sqrt(ALL_CURVES["SECP224R1"][0], bytes(28), out) == -1      # p = 1 mod 4: not served


@pytest.mark.parametrize("curve,hash_name,c", [("SECP256K1", "SHA256", 5), ("FRP256V1", "SHA256", 4),
                                               ("SECP256R1", "SHA512", 8), ("SECP384R1", "SHA384", 6)])
def test_host_bip0340_algorithm_against_reference(curve, hash_name, c):
    import test_bip0340 as tb
    _, plen, qlen = ALL_CURVES[curve]
    sigs, pubs, dg, hlen, want = tb.workload(curve, 28, 9600, hash_name)
    good = np.flatnonzero(want == 0)            # includes the items whose key was negated: the scheme only sees x(Y)
    assert host_msm_bip(curve, c, sigs[good], pubs[good], dg[good], hlen) == (0, 1)
    for bad in np.flatnonzero(want != 0):
        idx = np.concatenate([good[:5], [bad], good[5:9]])
        assert host_msm_bip(curve, c, sigs[idx], pubs[idx], dg[idx], hlen) == (0, 0), (curve, int(bad))
    assert host_msm_bip(curve, c, sigs[good[:1]], pubs[good[:1]], dg[good[:1]], hlen) == (0, 1)
    rep = np.repeat(good[:3], 12)
    assert host_msm_bip(curve, 2, sigs[rep], pubs[rep], dg[rep], hlen) == (0, 1)
    # the reference's own batch entry point on the same valid batch, and with one corrupted signature
    privs = __import__("common").random_scalars(curve, 10, tag=9700)
    msgs = [b"bip batch %d" % i for i in range(10)]
    s2, p2 = tb.ref_sign(curve, hash_name, privs, msgs)
    d2 = np.stack([tb.challenge(hash_name, s2[i, :plen], p2[i, :plen], msgs[i]) for i in range(10)])
    for scratch in (0, 1):
        assert tb.ref_verify_batch_all(curve, hash_name, s2, p2, msgs, scratch) == 0
    assert host_msm_bip(curve, c, s2, p2, d2, d2.shape[1]) == (0, 1)
    s2[4, -1] ^= 1
    # NOTE: only the reference's scratch-pad-free form (_bip0340_verify_batch_no_memory: the same linear combination,
    # summed directly) is the anchor on corrupted batches.  Its Bos-Coster form (with a scratch pad) was observed here to
    # return 0 for a batch whose s_4 is corrupted - ec_verify_bos_coster (sig/sig_algs.c:1052) leaves its loop as soon as
    # the two largest scalars are equal and then multiplies by their difference, 0 - so it is deliberately not asserted.
    assert tb.ref_verify_batch_all(curve, hash_name, s2, p2, msgs, 0) == -1
    assert (tb.ref_verify(curve, hash_name, s2, p2, msgs) == [0, 0, 0, 0, -1, 0, 0, 0, 0, 0]).all()
    assert host_msm_bip(curve, c, s2, p2, d2, d2.shape[1]) == (0, 0)


def test_host_bip0340_msm_not_on_secp224r1():
    assert host_msm_bip("SECP224R1", 4, np.zeros((1, 56), np.uint8), np.zeros((1, 56), np.uint8),
                        np.zeros((1, 32), np.uint8), 32)[0] == -1


# ------------------------------------------------------------------------------------------------------------- GPU


@pytest.mark.gpu
@pytest.mark.parametrize("curve", list(ALL_CURVES))
def test_gpu_msm_against_reference(curve, monkeypatch):
    import libecc_b200
    eng = libecc_b200.Engine(curve, comb_window=8)
    sigs, pubs, dg, hlen, want = workload(curve, 96, 9200)
    good = np.flatnonzero(want == 0)
    for c in (None, 2, 5, 11, 16):
        if c is None:
            monkeypatch.delenv("ECCB200_MSM_WINDOW", raising=False)
        else:
            monkeypatch.setenv("ECCB200_MSM_WINDOW", str(c))
        assert eng.ecfsdsa_verify_msm_batch(sigs[good], pubs[good], dg[good], hlen, SEED) is True, (curve, c)
        assert eng.ecfsdsa_verify_msm_batch(sigs[good], pubs[good], dg[good], hlen) is True          # OS seed
        assert eng.ecfsdsa_verify_msm_batch(sigs, pubs, dg, hlen, SEED) is False
        for bad in np.flatnonzero(want != 0)[:7]:
            idx = np.concatenate([good[:9], [bad], good[9:30]])
            assert eng.ecfsdsa_verify_msm_batch(sigs[idx], pubs[idx], dg[idx], hlen, SEED) is False, (curve, c, int(bad))
        assert eng.ecfsdsa_verify_msm_batch(sigs[good[:1]], pubs[good[:1]], dg[good[:1]], hlen, SEED) is True
        rep = np.repeat(good[:4], 40)
        assert eng.ecfsdsa_verify_msm_batch(sigs[rep], pubs[rep], dg[rep], hlen, SEED) is True
    monkeypatch.delenv("ECCB200_MSM_WINDOW", raising=False)
    assert eng.ecfsdsa_verify_msm_batch(sigs[:0], pubs[:0], dg[:0], hlen, SEED) is False
    # the verdict is the conjunction of the per-item verdicts of the verification kernel
    per_item = eng.ecfsdsa_verify_batch(sigs, pubs, dg, hlen)
    assert (per_item == want).all()
    eng.close()


@pytest.mark.gpu
@pytest.mark.parametrize("log2n", [16, 20])
def test_gpu_msm_full_size_properties(log2n):
    """2^16 and 2^20 signatures (config 3's batch size): reference-made signatures tiled (equal points meet in the
    buckets), accepted as a whole; one flipped bit anywhere sinks the batch; host and device entry points agree."""
    import libecc_b200
    curve = "FRP256V1"
    sigs, pubs, dg, hlen, want = workload(curve, 512, 9300)
    good = np.flatnonzero(want == 0)
    n = 1 << log2n
    idx = np.resize(good, n)
    S, P, D = sigs[idx].copy(), pubs[idx].copy(), dg[idx].copy()
    eng = libecc_b200.Engine(curve, comb_window=8)
    assert eng.ecfsdsa_verify_msm_batch(S, P, D, hlen) is True
    g = rng(9400 + log2n)
    for kind in range(3):
        i = int(g.integers(0, n))
        arr = (S, P, D)[kind]
        arr[i, -1] ^= 1
        assert eng.ecfsdsa_verify_msm_batch(S, P, D, hlen) is False, (kind, i)
        arr[i, -1] ^= 1
    assert eng.ecfsdsa_verify_msm_batch(S, P, D, hlen, SEED) is True
    eng.close()


@pytest.mark.gpu
@pytest.mark.parametrize("curve", [c for c in ALL_CURVES])
def test_gpu_bip0340_msm_against_reference(curve, monkeypatch):
    import libecc_b200
    import test_bip0340 as tb
    eng = libecc_b200.Engine(curve, comb_window=8)
    sigs, pubs, dg, hlen, want = tb.workload(curve, 96, 9800)
    good = np.flatnonzero(want == 0)
    if curve == "SECP224R1":            # p = 1 mod 4: the lift of r is not served, the per-item kernel is
        with pytest.raises(libecc_b200.EccB200Error, match="3 mod 4"):
            eng.bip0340_verify_msm_batch(sigs[good], pubs[good], dg[good], hlen, SEED)
        assert (eng.bip0340_verify_batch(sigs, pubs, dg, hlen) == want).all()
        eng.close()
        return
    for c in (None, 3, 9, 16):
        if c is None:
            monkeypatch.delenv("ECCB200_MSM_WINDOW", raising=False)
        else:
            monkeypatch.setenv("ECCB200_MSM_WINDOW", str(c))
        assert eng.bip0340_verify_msm_batch(sigs[good], pubs[good], dg[good], hlen, SEED) is True, (curve, c)
        assert eng.bip0340_verify_msm_batch(sigs[good], pubs[good], dg[good], hlen) is True
        assert eng.bip0340_verify_msm_batch(sigs, pubs, dg, hlen, SEED) is False
        for bad in np.flatnonzero(want != 0)[:7]:
            idx = np.concatenate([good[:9], [bad], good[9:30]])
            assert eng.bip0340_verify_msm_batch(sigs[idx], pubs[idx], dg[idx], hlen, SEED) is False, (curve, c, int(bad))
        rep = np.repeat(good[:4], 40)
        assert eng.bip0340_verify_msm_batch(sigs[rep], pubs[rep], dg[rep], hlen, SEED) is True
    monkeypatch.delenv("ECCB200_MSM_WINDOW", raising=False)
    assert (eng.bip0340_verify_batch(sigs, pubs, dg, hlen) == want).all()
    # 2^16 tiled signatures: accepted as a whole; one flipped bit sinks the batch
    idx = np.resize(good, 1 << 16)
    S, P, D = sigs[idx].copy(), pubs[idx].copy(), dg[idx].copy()
    assert eng.bip0340_verify_msm_batch(S, P, D, hlen) is True
    S[31337, -1] ^= 1
    assert eng.bip0340_verify_msm_batch(S, P, D, hlen) is False
    eng.close()

"""Parity tests proper: the CUDA path, called through the C ABI (include/libecc_b200.h), against the golden
vectors and the oracle.  Bit-exact (integer/byte work): affine bytes, infinity flag, error code, verdicts."""
import numpy as np
import pytest

from common import (hx_fit, ALL_CURVES, CURVES, HASHLEN, ORDER, PRIME, edge_scalars, golden, hx, make_signatures, oracle_smul,
                    oracle_verify, random_scalars, rng)

pytestmark = pytest.mark.gpu

_engines = {}


def engine(curve, w=0):
    import libecc_b200
    key = (curve, w)
    if key not in _engines:
        _engines[key] = libecc_b200.Engine(curve, device=0, comb_window=w)
    return _engines[key]


def be(vals, nbytes):
    return np.frombuffer(b"".join(int(v).to_bytes(nbytes, "big") for v in vals), dtype=np.uint8).copy()


@pytest.mark.parametrize("curve", list(ALL_CURVES))
def test_fp_mul_monty_against_integers(curve):
    """fp_mul_monty unit test in the pattern of src/arithmetic_tests (NN_MUL_REDC1 / FP_MUL_MONTY)."""
    eng = engine(curve, 8)
    _, plen, _ = ALL_CURVES[curve]
    g = rng(31)
    for which, mod in ((0, PRIME[curve]), (1, ORDER[curve])):
        a = [int.from_bytes(g.bytes(plen + 8), "big") % mod for _ in range(4096)] + [0, 1, mod - 1, mod - 1]
        b = [int.from_bytes(g.bytes(plen + 8), "big") % mod for _ in range(4096)] + [mod - 1, 1, mod - 1, 0]
        out = eng.fp_mul_monty_batch(be(a, plen), be(b, plen), which)
        rinv = pow(1 << (64 * ((PRIME[curve].bit_length() + 63) // 64)), -1, mod)  # the reference's R
        got = [int.from_bytes(o.tobytes(), "big") for o in out]
        assert got == [x * y * rinv % mod for x, y in zip(a, b)]
        # FP_ADD / FP_SUB / FP_SQR_MONTY through their own unit kernel (the PTX add / sub / dedicated squaring)
        ints = lambda arr: [int.from_bytes(o.tobytes(), "big") for o in arr]
        assert ints(eng.fp_addsub_batch(be(a, plen), be(b, plen), 0, which)) == [(x + y) % mod for x, y in zip(a, b)]
        assert ints(eng.fp_addsub_batch(be(a, plen), be(b, plen), 1, which)) == [(x - y) % mod for x, y in zip(a, b)]
        assert ints(eng.fp_addsub_batch(be(a, plen), be(b, plen), 2, which)) == [x * x * rinv % mod for x in a]


@pytest.mark.parametrize("curve", ["SECP256R1", "SECP384R1", "SECP521R1", "SECP224R1", "SECP192R1"])
def test_ecccdh_kat(curve):
    """NIST ECC-CDH vectors (reference: src/tests/ecccdh_test_vectors.h:1501-2999)."""
    _, plen, _ = ALL_CURVES[curve]
    vecs = [v for v in golden("ecccdh_kat.json") if v["curve"] == curve]
    d = np.stack([hx_fit(v["priv"], ALL_CURVES[v["curve"]][2]) for v in vecs]); peers = np.stack([hx(v["peer_pub"]) for v in vecs])
    for w in (8, 0):
        out, st = engine(curve, w).prj_pt_mul_batch(d)
        assert (st == 0).all() and [o.tobytes().hex() for o in out] == [v["our_pub"] for v in vecs]
    out, st = engine(curve).prj_pt_mul_batch(d, peers)
    assert (st == 0).all() and [o[:plen].tobytes().hex() for o in out] == [v["shared"] for v in vecs]


@pytest.mark.parametrize("curve", list(ALL_CURVES))
@pytest.mark.parametrize("w", [5, 8, 13, 0])
def test_fixed_base_vs_oracle(curve, w):
    sc = np.concatenate([random_scalars(curve, 1024 if w else 4096, tag=41 + w, below_q=False), edge_scalars(curve)])
    want, wst = oracle_smul(curve, sc)
    out, st = engine(curve, w).prj_pt_mul_batch(sc)
    assert (st == wst).all()
    assert (out == want).all()


@pytest.mark.parametrize("curve,w", [("SECP256R1", 20), ("FRP256V1", 18), ("SECP384R1", 18), ("SECP256R1", 22)])
def test_fixed_base_wide_window_tables(curve, w):
    """Comb windows wider than 16 bits are built by merging a half-width table (k_table_merge): same results."""
    sc = np.concatenate([random_scalars(curve, 2048, tag=45 + w, below_q=False), edge_scalars(curve)])
    want, wst = oracle_smul(curve, sc)
    eng = engine(curve, w)
    assert eng.comb_window == w
    out, st = eng.prj_pt_mul_batch(sc)
    assert (st == wst).all() and (out == want).all()
    _engines.pop((curve, w)).close()   # give the table memory back


@pytest.mark.parametrize("curve", list(ALL_CURVES))
def test_variable_base_vs_oracle(curve):
    _, plen, qlen = ALL_CURVES[curve]
    base_sc = random_scalars(curve, 2048, tag=51)
    pts, st0 = oracle_smul(curve, base_sc)
    sc = random_scalars(curve, 2048, tag=52, below_q=False)
    es = edge_scalars(curve)
    sc[: es.shape[0]] = es
    pts[100, 7] ^= 0x04          # off the curve
    pts[101, :plen] = 0xFF       # x >= p
    pts[102, plen:] = 0xFF       # y >= p
    pts[103, :] = 0              # (0,0) is not on these curves
    want, wst = oracle_smul(curve, sc, pts)
    out, st = engine(curve).prj_pt_mul_batch(sc, pts)
    assert (st == wst).all() and (wst[100:104] == -1).all()
    assert (out == want).all()


WYCHE_CURVES = ["SECP256R1", "SECP384R1", "BRAINPOOLP256R1", "BRAINPOOLP384R1", "SECP256K1", "SECP521R1", "BRAINPOOLP512R1",
                "SECP224R1"]


@pytest.mark.parametrize("curve", WYCHE_CURVES)
def test_wycheproof_ecdh(curve):
    _, plen, qlen = ALL_CURVES[curve]
    vecs = [v for v in golden("wycheproof_ecdh.json.gz") if v["curve"] == curve and len(v["priv"]) <= 2 * qlen]
    d = np.stack([hx(v["priv"].rjust(2 * qlen, "0")) for v in vecs]); q = np.stack([hx(v["peer_pub"]) for v in vecs])
    out, st = engine(curve).prj_pt_mul_batch(d, q)
    assert [int(s) for s in st] == [v["ref_status"] for v in vecs]
    assert [o.tobytes().hex() for o in out] == [v["ref_point"] for v in vecs]


def test_ecdsa_kat():
    for v in golden("ecdsa_kat.json"):
        got = engine(v["curve"]).ecdsa_verify_batch(hx(v["sig"]), hx(v["pub"]), hx(v["digest"]), HASHLEN[v["hash"]])
        assert got[0] == 0 == v["ref_verdict"], v["name"]
        bad = hx(v["digest"]).copy(); bad[0] ^= 1
        assert engine(v["curve"]).ecdsa_verify_batch(hx(v["sig"]), hx(v["pub"]), bad, HASHLEN[v["hash"]])[0] == -1


@pytest.mark.parametrize("curve", WYCHE_CURVES)
def test_wycheproof_ecdsa_all(curve):
    """Every Wycheproof ECDSA vector the reference ships for the curve: verdict == the reference's own ec_verify."""
    _, plen, qlen = ALL_CURVES[curve]
    vecs = [v for v in golden("wycheproof_ecdsa.json.gz")
            if v["curve"] == curve and len(v["sig"]) == 4 * qlen and len(v["pub"]) == 4 * plen]
    assert len(vecs) > 400
    for h in sorted({v["hash"] for v in vecs}):
        vs = [v for v in vecs if v["hash"] == h]
        sig = np.stack([hx(v["sig"]) for v in vs]); pub = np.stack([hx(v["pub"]) for v in vs])
        dg = np.stack([hx(v["digest"]) for v in vs])
        got = engine(curve).ecdsa_verify_batch(sig, pub, dg, HASHLEN[h])
        want = np.array([v["ref_verdict"] for v in vs], dtype=np.int8)
        assert (got == want).all(), [v["name"] for v, g_, w_ in zip(vs, got, want) if g_ != w_][:5]


@pytest.mark.parametrize("curve,hlen,w", [("FRP256V1", 32, 0), ("SECP256R1", 32, 0), ("SECP384R1", 48, 0),
                                          ("SECP256R1", 64, 13), ("SECP384R1", 20, 8), ("FRP256V1", 32, 16),
                                          ("SECP256R1", 32, 18), ("BRAINPOOLP256R1", 32, 0),
                                          ("BRAINPOOLP384R1", 48, 13), ("SECP256K1", 32, 0)])
def test_ecdsa_synthetic_with_corruptions(curve, hlen, w):
    """Includes comb windows that straddle 32-bit words (13, 18, default 22) and ones that do not (8, 16)."""
    sigs, pubs, dg, expected = make_signatures(curve, 512, tag=hlen, hlen=hlen, corrupt_every=8)
    got = engine(curve, w).ecdsa_verify_batch(sigs, pubs, dg, hlen)
    assert (got == expected).all()
    assert (expected[::8] == -1).all() and (np.delete(expected, np.s_[::8]) == 0).all()


def test_device_pointer_api_and_ragged_sizes():
    import torch
    curve = "SECP256R1"
    eng = engine(curve)
    for n in (0, 1, 31, 129, 1000):
        sc = random_scalars(curve, max(n, 1), tag=60 + n)[:n]
        want, wst = oracle_smul(curve, sc) if n else (np.zeros((0, 64), np.uint8), np.zeros(0, np.int8))
        d_sc = torch.from_numpy(sc.copy()).cuda().reshape(-1)
        d_out = torch.zeros(n * 64, dtype=torch.uint8, device="cuda")
        d_st = torch.full((n,), 7, dtype=torch.int8, device="cuda")
        eng.prj_pt_mul_batch_dev(d_sc, None, d_out, d_st, torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        assert (d_st.cpu().numpy() == wst).all()
        assert (d_out.cpu().numpy().reshape(n, 64) == want).all()
        out, st = eng.prj_pt_mul_batch(sc)
        assert (out == want).all() and (st == wst).all()


def test_full_size_batch_properties_and_sample():
    """BASELINE.json config 2 at full size (2^20 scalars on G): the oracle cannot run 2^20 items in seconds, so
    (i) a seeded sample is compared bit-exactly with the oracle, (ii) size-independent properties are checked on the
    whole batch: k and q-k give the same x and y + y' = p (negation), all outputs are on the curve."""
    curve = "SECP256R1"
    n = 1 << 20
    p, q = PRIME[curve], ORDER[curve]
    sc = random_scalars(curve, n // 2, tag=70, below_q=False)
    sc[:, 0] &= 0x7F  # keep k < q so that q - k is in range
    ks = [int.from_bytes(r.tobytes(), "big") for r in sc[:4096]]
    neg = sc.copy()
    # q - k computed with numpy on 32-byte big-endian rows (vectorised borrow chain)
    qb = np.frombuffer(q.to_bytes(32, "big"), dtype=np.uint8).astype(np.int32)
    borrow = np.zeros(n // 2, dtype=np.int32)
    for j in range(31, -1, -1):
        dj = qb[j] - sc[:, j].astype(np.int32) - borrow
        borrow = (dj < 0).astype(np.int32)
        neg[:, j] = (dj + 256 * borrow).astype(np.uint8)
    assert int.from_bytes(neg[0].tobytes(), "big") == q - ks[0]
    allsc = np.concatenate([sc, neg])
    out, st = engine(curve).prj_pt_mul_batch(allsc)
    assert (st == 0).all()
    a, b = out[: n // 2], out[n // 2:]
    assert (a[:, :32] == b[:, :32]).all()                       # same x
    # y + y' == p : byte-wise big-endian addition with carry
    pb = np.frombuffer(p.to_bytes(32, "big"), dtype=np.uint8).astype(np.int32)
    carry = np.zeros(n // 2, dtype=np.int32)
    ok = np.ones(n // 2, dtype=bool)
    for j in range(31, -1, -1):
        s = a[:, 32 + j].astype(np.int32) + b[:, 32 + j].astype(np.int32) + carry
        ok &= (s & 0xFF) == pb[j]
        carry = s >> 8
    assert ok.all() and (carry == 0).all()
    idx = rng(71).choice(n, size=2048, replace=False)
    want, wst = oracle_smul(curve, allsc[idx])
    assert (out[idx] == want).all() and (st[idx] == wst).all()


@pytest.mark.parametrize("curve", list(ALL_CURVES))
def test_ecdsa_scalar_preparation_mod_q(curve):
    """u = e*s^-1, v = r*s^-1 mod q on the device (nn_modinv / nn_mod_mul on the order, ecdsa_common.c:781-791)
    against Python integers, including digests longer and shorter than the order."""
    _, plen, qlen = ALL_CURVES[curve]
    q = ORDER[curve]
    g = rng(81)
    for hlen in (20, qlen, 64):
        n = 500
        sig = g.integers(0, 256, size=(n, 2 * qlen), dtype=np.uint8)
        top = ((1 << (q.bit_length() - 8 * (qlen - 1))) - 1) >> 1
        sig[:, 0] &= top; sig[:, qlen] &= top            # r, s < q
        sig[0, qlen:] = 0; sig[0, -1] = 1                # s = 1
        sig[1, qlen:] = np.frombuffer((q - 1).to_bytes(qlen, "big"), dtype=np.uint8)
        dg = g.integers(0, 256, size=(n, hlen), dtype=np.uint8)
        dg[2] = 0xFF
        uv = engine(curve, 8).ecdsa_uv_batch(sig, dg, hlen)
        for i in range(n):
            r = int.from_bytes(sig[i, :qlen].tobytes(), "big"); s = int.from_bytes(sig[i, qlen:].tobytes(), "big")
            take = min(hlen, qlen)                       # leftmost min(8*hlen, bitlen(q)) bits (ecdsa_common.c:760-775)
            e = (int.from_bytes(dg[i, :take].tobytes(), "big") >> max(0, 8 * take - q.bit_length())) % q
            w = pow(s, -1, q)
            assert int.from_bytes(uv[i, :qlen].tobytes(), "big") == e * w % q
            assert int.from_bytes(uv[i, qlen:].tobytes(), "big") == r * w % q


def test_ecdsa_sign_batch_kat_and_oracle():
    """Row (f).1: batched ECDSA signing.  The reference's own KATs inject the nonce (ec_self_tests_core.h:34); with
    the same nonce the device must reproduce the expected signature bit for bit."""
    from common import oracle_sign
    for v in golden("ecdsa_kat.json"):
        if "nonce" not in v:
            continue
        sig, st = engine(v["curve"]).ecdsa_sign_batch(hx_fit(v["priv"], ALL_CURVES[v["curve"]][2]), hx_fit(v["nonce"], ALL_CURVES[v["curve"]][2]), hx(v["digest"]), HASHLEN[v["hash"]])
        assert st[0] == 0 and sig[0].tobytes().hex() == v["sig"], v["name"]
    for curve, hlen in (("SECP256R1", 32), ("FRP256V1", 32), ("SECP384R1", 48), ("SECP256R1", 64),
                        ("BRAINPOOLP256R1", 32), ("BRAINPOOLP384R1", 48), ("SECP256K1", 32)):
        _, plen, qlen = ALL_CURVES[curve]
        q = ORDER[curve]
        n = 3000
        d = random_scalars(curve, n, tag=91); k = random_scalars(curve, n, tag=92)
        dg = rng(93).integers(0, 256, size=(n, hlen), dtype=np.uint8)
        k[0] = 0                                                      # k = 0      -> -1
        k[1] = np.frombuffer(q.to_bytes(qlen, "big"), dtype=np.uint8)  # k = q      -> -1
        d[2] = 0                                                      # d = 0      -> -1
        d[3] = 0xFF                                                   # d >= q     -> -1
        want, wst = oracle_sign(curve, d, k, dg, hlen)
        sig, st = engine(curve).ecdsa_sign_batch(d, k, dg, hlen)
        assert (st == wst).all() and (wst[:4] == -1).all() and (wst[4:] == 0).all()
        assert (sig[4:] == want[4:]).all() and (sig[:4] == 0).all()
        pubs, pst = engine(curve).prj_pt_mul_batch(d[4:])             # key generation = fixed-base batch
        assert (engine(curve).ecdsa_verify_batch(sig[4:], pubs, dg[4:], hlen) == 0).all()


@pytest.mark.parametrize("curve", WYCHE_CURVES)
def test_ecccdh_derive_batch(curve):
    """Row (f).2: batched ecccdh_derive_secret — NIST KATs and every uncompressed Wycheproof ECDH vector."""
    _, plen, qlen = ALL_CURVES[curve]
    vecs = [v for v in golden("ecccdh_kat.json") if v["curve"] == curve]
    if vecs:  # the NIST ECC-CDH KATs exist for the NIST curves only
        sh, st = engine(curve).ecccdh_derive_batch(np.stack([hx_fit(v["priv"], ALL_CURVES[v["curve"]][2]) for v in vecs]),
                                                   np.stack([hx(v["peer_pub"]) for v in vecs]))
        assert (st == 0).all() and [s.tobytes().hex() for s in sh] == [v["shared"] for v in vecs]
    vecs = [v for v in golden("wycheproof_ecdh.json.gz") if v["curve"] == curve and len(v["priv"]) <= 2 * qlen]
    sh, st = engine(curve).ecccdh_derive_batch(np.stack([hx(v["priv"].rjust(2 * qlen, "0")) for v in vecs]),
                                               np.stack([hx(v["peer_pub"]) for v in vecs]))
    for v, s, t in zip(vecs, sh, st):
        if v["ref_status"] == 0:
            assert t == 0 and s.tobytes().hex() == v["ref_point"][: 2 * plen], v["name"]
        else:  # off-curve peer key (-1) or infinity result (1): ecccdh_derive_secret fails in both cases
            assert t == -1 and not s.any(), v["name"]


@pytest.mark.parametrize("curve", ["SECP256R1", "FRP256V1"])
def test_layout_experiment_kernels_agree(curve):
    """DESIGN.md §3: the lane-striped (__shfl_sync) multiplier computes the same products as the production one."""
    _, plen, _ = ALL_CURVES[curve]
    p = PRIME[curve]
    g = rng(97)
    n = 4096
    a = [int.from_bytes(g.bytes(plen + 8), "big") % p for _ in range(n)]
    b = [int.from_bytes(g.bytes(plen + 8), "big") % p for _ in range(n)]
    a[0], b[0] = p - 1, p - 1
    a[1], b[1] = 0, 5
    iters = 3
    o0, _ = engine(curve, 8).fp_mul_chain_bench(be(a, plen), be(b, plen), iters, striped=False)
    o1, _ = engine(curve, 8).fp_mul_chain_bench(be(a, plen), be(b, plen), iters, striped=True)
    rinv = pow(1 << (8 * plen), -1, p)
    want = [x * pow(y * rinv, iters, p) % p for x, y in zip(a, b)]
    assert [int.from_bytes(o.tobytes(), "big") for o in o0] == want
    assert (o0 == o1).all()


def test_full_size_ecdsa_verify_frp256v1():
    """BASELINE.json config 3 at full size: 2^20 FRP256V1 signatures under 2^20 distinct keys.  Keys and signatures
    come from the engine's own batch signer (cross-checked with the oracle on a sample); 1/16 are corrupted; the
    verdict vector must equal the by-construction expectation on the whole batch and the oracle on a sample."""
    import bench
    inp = bench.make_verify_inputs("FRP256V1", 1 << 20, rank=3)
    n = 1 << 20
    got = engine("FRP256V1").ecdsa_verify_batch(inp["sigs"], inp["pubkeys"], inp["digests_host"], inp["hlen"])
    assert (got == inp["expected"]).all()
    assert (got[::16] == -1).all() and int((got == 0).sum()) == n - (1 << 16)
    idx = rng(101).choice(n, size=1024, replace=False)
    want = oracle_verify("FRP256V1", inp["sigs"][idx], inp["pubkeys"][idx], bench.sha256_rows(inp["msgs"][idx]), inp["hlen"])
    assert (got[idx] == want).all()
    # the same batch as MESSAGES (what ec_verify takes): SHA-256 on the device, then the verification kernel
    off = np.arange(n + 1, dtype=np.uint64) * bench.MSG_LEN
    got_m = engine("FRP256V1").ecdsa_verify_msgs_batch_raw("SHA256", inp["sigs"], inp["pubkeys"], inp["msgs"], off)
    assert (got_m == inp["expected"]).all()


def test_full_size_secp384r1_fixed_base_properties():
    """BASELINE.json config 4 at full size (2^20 scalars on G, secp384r1): negation property on the whole batch and a
    seeded sample against the oracle."""
    curve = "SECP384R1"
    n = 1 << 20
    p, q = PRIME[curve], ORDER[curve]
    sc = random_scalars(curve, n // 2, tag=170, below_q=False)
    sc[:, 0] &= 0x7F
    qb = np.frombuffer(q.to_bytes(48, "big"), dtype=np.uint8).astype(np.int32)
    neg = sc.copy()
    borrow = np.zeros(n // 2, dtype=np.int32)
    for j in range(47, -1, -1):
        dj = qb[j] - sc[:, j].astype(np.int32) - borrow
        borrow = (dj < 0).astype(np.int32)
        neg[:, j] = (dj + 256 * borrow).astype(np.uint8)
    allsc = np.concatenate([sc, neg])
    out, st = engine(curve).prj_pt_mul_batch(allsc)
    assert (st == 0).all()
    a, b = out[: n // 2], out[n // 2:]
    assert (a[:, :48] == b[:, :48]).all()
    pb = np.frombuffer(p.to_bytes(48, "big"), dtype=np.uint8).astype(np.int32)
    carry = np.zeros(n // 2, dtype=np.int32)
    ok = np.ones(n // 2, dtype=bool)
    for j in range(47, -1, -1):
        s = a[:, 48 + j].astype(np.int32) + b[:, 48 + j].astype(np.int32) + carry
        ok &= (s & 0xFF) == pb[j]
        carry = s >> 8
    assert ok.all() and (carry == 0).all()
    idx = rng(171).choice(n, size=1024, replace=False)
    want, wst = oracle_smul(curve, allsc[idx])
    assert (out[idx] == want).all() and (st[idx] == wst).all()


def test_tma_staged_k1_variant_matches():
    """DESIGN.md §3 staging experiment: K1 with its scalars staged by cp.async.bulk (ECCB200_TMA_STAGING=1, read once
    per process, hence the subprocess) must give the same bytes, including for a ragged last CTA."""
    import subprocess
    import sys
    code = r"""
import sys, numpy as np
sys.path.insert(0, 'tests'); sys.path.insert(0, '.')
import libecc_b200
from common import random_scalars, edge_scalars, oracle_smul
import torch
for curve in ('SECP256R1', 'SECP384R1'):
    sc = np.concatenate([random_scalars(curve, 1000, tag=7, below_q=False), edge_scalars(curve)])
    want, wst = oracle_smul(curve, sc)
    eng = libecc_b200.Engine(curve, 0, 8)
    d_sc = torch.from_numpy(sc.copy()).cuda().reshape(-1)
    n = sc.shape[0]; rec = want.shape[1]
    d_out = torch.zeros(n * rec, dtype=torch.uint8, device='cuda'); d_st = torch.zeros(n, dtype=torch.int8, device='cuda')
    eng.prj_pt_mul_batch_dev(d_sc, None, d_out, d_st, 0)
    torch.cuda.synchronize()
    assert (d_out.cpu().numpy().reshape(n, rec) == want).all() and (d_st.cpu().numpy() == wst).all()
print('TMA-OK')
"""
    env = dict(**__import__("os").environ, ECCB200_TMA_STAGING="1")
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300, env=env,
                       cwd=__import__("common").ROOT)
    assert r.returncode == 0 and "TMA-OK" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]


def test_device_sha2_matches_hashlib_and_reference():
    """Row (f).3: SHA-256/384/512 on the device against hashlib and the reference's own src/hash (ref_hash)."""
    import hashlib
    from test_sha3 import ref_hash
    g = rng(111)
    lens = list(range(0, 150)) + [183, 184, 185, 239, 240, 247, 248, 255, 256, 257, 1000, 4097]
    msgs = [g.bytes(n) for n in lens]
    eng = engine("SECP256R1", 8)
    for name, fn in (("SHA256", hashlib.sha256), ("SHA384", hashlib.sha384), ("SHA512", hashlib.sha512)):
        out = eng.hash_batch(name, msgs)
        assert [o.tobytes() for o in out] == [fn(m).digest() for m in msgs], name
        for m in msgs[::17]:
            assert ref_hash(name, m).tobytes() == fn(m).digest()


def test_ecdsa_verify_msgs_batch():
    """ec_verify on raw messages (hash on the device, then K3): the reference's KATs that use SHA-2, and a seeded
    batch signed by the oracle over hashlib digests with a few corrupted messages."""
    import hashlib
    from common import oracle_sign
    fn = {"SHA256": hashlib.sha256, "SHA384": hashlib.sha384, "SHA512": hashlib.sha512, "SHA3_224": hashlib.sha3_224,
          "SHA3_256": hashlib.sha3_256, "SHA3_384": hashlib.sha3_384, "SHA3_512": hashlib.sha3_512}
    for v in golden("ecdsa_kat.json"):
        if v["hash"] not in fn:
            continue
        msg = bytes.fromhex(v["msg"])
        got = engine(v["curve"]).ecdsa_verify_msgs_batch(v["hash"], hx(v["sig"]), hx(v["pub"]), [msg])
        assert got[0] == 0, v["name"]
        assert engine(v["curve"]).ecdsa_verify_msgs_batch(v["hash"], hx(v["sig"]), hx(v["pub"]), [msg + b"x"])[0] == -1
    for curve, hname in (("FRP256V1", "SHA256"), ("SECP384R1", "SHA384"), ("SECP256R1", "SHA512")):
        n = 600
        g = rng(112)
        msgs = [g.bytes(int(g.integers(0, 200))) for _ in range(n)]
        dg = np.stack([np.frombuffer(fn[hname](m).digest(), dtype=np.uint8) for m in msgs])
        d = random_scalars(curve, n, tag=113); k = random_scalars(curve, n, tag=114)
        sigs, st = oracle_sign(curve, d, k, dg, dg.shape[1])
        assert (st == 0).all()
        pubs, _ = oracle_smul(curve, d)
        bad = list(range(0, n, 10))
        for i in bad:
            msgs[i] = msgs[i] + b"!"
        got = engine(curve).ecdsa_verify_msgs_batch(hname, sigs, pubs, msgs)
        want = np.zeros(n, dtype=np.int8); want[bad] = -1
        assert (got == want).all()
        if curve == "FRP256V1":
            # the same tuples tiled past one pipeline chunk (4 waves = 303 104 items): variable-length messages whose
            # offsets cross the chunk boundaries, empty messages included, and a ragged last chunk
            reps = 530
            blob = np.frombuffer(b"".join(msgs) * reps, dtype=np.uint8)
            lens = np.tile(np.array([len(m) for m in msgs], dtype=np.uint64), reps)
            off = np.zeros(n * reps + 1, dtype=np.uint64)
            off[1:] = np.cumsum(lens)
            big = engine(curve).ecdsa_verify_msgs_batch_raw(hname, np.tile(sigs, (reps, 1)), np.tile(pubs, (reps, 1)),
                                                            blob, off)
            assert big.shape[0] == n * reps and (big == np.tile(want, reps)).all()

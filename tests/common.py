"""Shared helpers for the test-suite: loaders for the checkers (oracle port, compiled reference, host build of
the device algorithms), the golden fixtures, and seeded input generators.

Only tests/, __graft_entry__.smoke() and bench.py's CPU legs may touch oracle/ (see oracle/ecc_oracle.h)."""
from __future__ import annotations

import ctypes
import gzip
import json
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
ORACLE_SO = os.path.join(ROOT, "oracle", "_ref", "libecc_oracle.so")
REF_SO = os.path.join(ROOT, "oracle", "_ref", "libecc_ref.so")
HOSTSIM_SO = os.path.join(ROOT, "tests", "hostsim", "_build", "libecc_hostsim.so")
SEED = 0x6C69626563632D31  # "libecc-1" (SURVEY.md §8d)

CURVES = {"SECP256R1": (4, 32, 32), "FRP256V1": (1, 32, 32), "SECP384R1": (5, 48, 48)}  # id, plen, qlen
# additional curves (SURVEY.md §8f.4): same kernels, generic-a / a = 0 doubling
EXTRA_CURVES = {"BRAINPOOLP256R1": (8, 32, 32), "BRAINPOOLP384R1": (12, 48, 48), "SECP256K1": (19, 32, 32),
                "SECP521R1": (6, 66, 66),
                "SM2P256V1": (17, 32, 32), "BRAINPOOLP512R1": (9, 64, 64), "SECP224R1": (3, 28, 28),
                "SECP192R1": (2, 24, 24)}  # 521-bit: byte lengths not a multiple of the word size
ALL_CURVES = dict(CURVES, **EXTRA_CURVES)
ORDER = {
    "SECP256R1": 0xffffffff00000000ffffffffffffffffbce6faada7179e84f3b9cac2fc632551,
    "FRP256V1": 0xf1fd178c0b3ad58f10126de8ce42435b53dc67e140d2bf941ffdd459c6d655e1,
    "SECP384R1": 0xffffffffffffffffffffffffffffffffffffffffffffffffc7634d81f4372ddf581a0db248b0a77aecec196accc52973,
    "BRAINPOOLP256R1": 0xa9fb57dba1eea9bc3e660a909d838d718c397aa3b561a6f7901e0e82974856a7,
    "BRAINPOOLP384R1": 0x8cb91e82a3386d280f5d6f7e50e641df152f7109ed5456b31f166e6cac0425a7cf3ab6af6b7fc3103b883202e9046565,
    "SECP256K1": 0xfffffffffffffffffffffffffffffffebaaedce6af48a03bbfd25e8cd0364141,
    "SECP521R1": 0x01fffffffffffffffffffffffffffffffffffffffffffffffffffffffffffffffffa51868783bf2f966b7fcc0148f709a5d03bb5c9b8899c47aebb6fb71e91386409,
    "SM2P256V1": 0xfffffffeffffffffffffffffffffffff7203df6b21c6052b53bbf40939d54123,
    "BRAINPOOLP512R1": 0xaadd9db8dbe9c48b3fd4e6ae33c9fc07cb308db3b3c9d20ed6639cca70330870553e5c414ca92619418661197fac10471db1d381085ddaddb58796829ca90069,
    "SECP224R1": 0xffffffffffffffffffffffffffff16a2e0b8f03e13dd29455c5c2a3d,
    "SECP192R1": 0xffffffffffffffffffffffff99def836146bc9b1b4d22831,
}
PRIME = {
    "SECP256R1": 0xffffffff00000001000000000000000000000000ffffffffffffffffffffffff,
    "FRP256V1": 0xf1fd178c0b3ad58f10126de8ce42435b3961adbcabc8ca6de8fcf353d86e9c03,
    "SECP384R1": 0xfffffffffffffffffffffffffffffffffffffffffffffffffffffffffffffffeffffffff0000000000000000ffffffff,
    "BRAINPOOLP256R1": 0xa9fb57dba1eea9bc3e660a909d838d726e3bf623d52620282013481d1f6e5377,
    "BRAINPOOLP384R1": 0x8cb91e82a3386d280f5d6f7e50e641df152f7109ed5456b412b1da197fb71123acd3a729901d1a71874700133107ec53,
    "SECP256K1": 0xfffffffffffffffffffffffffffffffffffffffffffffffffffffffefffffc2f,
    "SECP521R1": (1 << 521) - 1,
    "SM2P256V1": 0xfffffffeffffffffffffffffffffffffffffffff00000000ffffffffffffffff,
    "BRAINPOOLP512R1": 0xaadd9db8dbe9c48b3fd4e6ae33c9fc07cb308db3b3c9d20ed6639cca703308717d4d9b009bc66842aecda12ae6a380e62881ff2f2d82c68528aa6056583a48f3,
    "SECP224R1": 0xffffffffffffffffffffffffffffffff000000000000000000000001,
    "SECP192R1": 0xfffffffffffffffffffffffffffffffeffffffffffffffff,
}
HASHLEN = {"SHA224": 28, "SHA256": 32, "SHA384": 48, "SHA512": 64, "SHA3_224": 28, "SHA3_256": 32,
           "SHA3_384": 48, "SHA3_512": 64}

_cache = {}


def _build_oracle():
    if not os.path.exists(ORACLE_SO) or os.path.getmtime(ORACLE_SO) < os.path.getmtime(
            os.path.join(ROOT, "oracle", "ecc_oracle.c")):
        subprocess.run(["make", "-C", os.path.join(ROOT, "oracle"), "oracle"], check=True, capture_output=True)


def oracle_lib() -> ctypes.CDLL:
    if "oracle" not in _cache:
        _build_oracle()
        lib = ctypes.CDLL(ORACLE_SO)
        lib.ora_last_mul_count.restype = ctypes.c_uint64
        _cache["oracle"] = lib
    return _cache["oracle"]


def ref_lib():
    """The unmodified reference compiled by oracle/Makefile (`make -C oracle ref REF=<its sources>`).  Only the
    @reference_answer helpers call it, and only while their answers are being recorded."""
    if "ref" not in _cache:
        if not os.path.exists(REF_SO):
            raise RuntimeError(f"{REF_SO} is missing: build it with `make -C oracle ref REF=<reference sources>`")
        _cache["ref"] = ctypes.CDLL(REF_SO)
    return _cache["ref"]


# The reference's answers to the questions the tests ask it are stored under tests/golden/reference/ (one xz-compressed
# .npz per test module), keyed by the helper's name and a digest of its arguments, so that the comparisons run on any machine.
# RECORD_REFERENCE=1 asks the compiled reference instead and stores its answers (tests/golden/record_reference.sh).
REFERENCE_ANSWERS = os.path.join(GOLDEN, "reference")
RECORDING = os.environ.get("RECORD_REFERENCE") == "1"
_answers = {}


def _digest_args(h, a):
    if isinstance(a, np.ndarray):
        a = np.ascontiguousarray(a)
        h.update(b"A%s%r" % (a.dtype.str.encode(), a.shape))
        h.update(a.tobytes())
    elif isinstance(a, (bytes, bytearray)):
        h.update(b"B%d:" % len(a))
        h.update(bytes(a))
    elif isinstance(a, (list, tuple)):
        h.update(b"L%d:" % len(a))
        for x in a:
            _digest_args(h, x)
    elif a is None or isinstance(a, (str, int, np.integer)):
        h.update(b"S%r;" % (a if a is None or isinstance(a, str) else int(a),))
    else:
        raise TypeError(f"cannot key a reference answer on {type(a)}")


def _answer_file(module: str):
    if module not in _answers:
        import io
        import lzma
        path = os.path.join(REFERENCE_ANSWERS, module + ".npz.xz")
        stored = {}
        if os.path.exists(path):
            with lzma.open(path) as f, np.load(io.BytesIO(f.read())) as z:
                stored = {k: z[k] for k in z.files}
        _answers[module] = stored
    return _answers[module]


def _save_answers():
    import io
    import lzma
    os.makedirs(REFERENCE_ANSWERS, exist_ok=True)
    for module, stored in _answers.items():
        buf = io.BytesIO()
        np.savez(buf, **stored)    # one xz stream: the many small answers share their headers' compression
        with open(os.path.join(REFERENCE_ANSWERS, module + ".npz.xz"), "wb") as f:
            f.write(lzma.compress(buf.getvalue(), preset=9 | lzma.PRESET_EXTREME))


def reference_answer(fn):
    """Decorates a helper that asks the compiled reference something: its arguments are arrays, bytes, strings or ints,
    its result an array or an int, or a tuple of them.  The stored answer for the same arguments is returned; a question
    without a stored answer fails (its inputs changed: record the answers again)."""
    import functools
    import hashlib

    @functools.wraps(fn)
    def ask(*args):
        h = hashlib.sha256()
        _digest_args(h, args)
        key = f"{fn.__name__}-{h.hexdigest()[:24]}"
        stored = _answer_file(fn.__module__)
        if RECORDING:
            if "save" not in _cache:
                import atexit
                _cache["save"] = atexit.register(_save_answers)
            res = fn(*args)
            items = res if isinstance(res, tuple) else (res,)
            stored[key + ".n"] = np.array(len(items) if isinstance(res, tuple) else -1)
            for i, x in enumerate(items):
                stored[f"{key}.{i}"] = np.asarray(x)
        if key + ".n" not in stored:
            raise AssertionError(f"no stored answer of the reference to {fn.__module__}.{fn.__name__} for these "
                                 f"arguments: record them again (tests/golden/record_reference.sh)")
        n = int(stored[key + ".n"])
        items = [stored[f"{key}.{i}"] for i in range(max(n, 1))]
        items = [x.item() if x.ndim == 0 else x.copy() for x in items]
        return tuple(items) if n >= 0 else items[0]
    return ask


def hostsim_lib() -> ctypes.CDLL:
    if "hostsim" not in _cache:
        src = os.path.join(ROOT, "tests", "hostsim", "hostsim.cpp")
        deps = [src] + [os.path.join(ROOT, "libecc_b200", "csrc", f) for f in
                        ("fp.cuh", "ec.cuh", "msm_core.cuh", "curve_constants.inc", "sha3.cuh", "sha3_constants.inc")]
        if not os.path.exists(HOSTSIM_SO) or os.path.getmtime(HOSTSIM_SO) < max(os.path.getmtime(d) for d in deps):
            os.makedirs(os.path.dirname(HOSTSIM_SO), exist_ok=True)
            subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-x", "c++", src, "-o", HOSTSIM_SO],
                           check=True, capture_output=True)
        lib = ctypes.CDLL(HOSTSIM_SO)
        lib.hostsim_last_mul_count.restype = ctypes.c_ulonglong
        _cache["hostsim"] = lib
    return _cache["hostsim"]


STUB_SO = os.path.join(ROOT, "tests", "hostsim", "_build", "libecc_b200_stub.so")


def engine_stub_so() -> str:
    """Path of the TEST-ONLY stand-in for libecc_b200.so (tests/hostsim/engine_stub.cpp: the engine entry points the
    drop-in calls, served by the host build of the device algorithms), built on demand.  Preloaded in front of the
    C harness it lets the CPU suite run the drop-in's host logic against the unmodified reference."""
    src = os.path.join(ROOT, "tests", "hostsim", "engine_stub.cpp")
    deps = [src, os.path.join(ROOT, "tests", "hostsim", "hostsim.cpp")] + [
        os.path.join(ROOT, "libecc_b200", "csrc", f) for f in
        ("fp.cuh", "ec.cuh", "msm_core.cuh", "curve_constants.inc", "sha3.cuh", "sha3_constants.inc")]
    if not os.path.exists(STUB_SO) or os.path.getmtime(STUB_SO) < max(os.path.getmtime(d) for d in deps):
        os.makedirs(os.path.dirname(STUB_SO), exist_ok=True)
        subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-x", "c++", src, "-o", STUB_SO, "-lpthread"],
                       check=True, capture_output=True)
    return STUB_SO


def golden(name: str):
    path = os.path.join(GOLDEN, name)
    if path.endswith(".gz"):
        with gzip.open(path, "rt") as f:
            return json.load(f)
    with open(path) as f:
        return json.load(f)


def rng(tag: int = 0) -> np.random.Generator:
    return np.random.default_rng([SEED & 0xFFFFFFFF, SEED >> 32, tag])


def random_scalars(curve: str, n: int, tag: int = 0, below_q: bool = True) -> np.ndarray:
    """n big-endian qlen-byte scalars, uniform in [1, q-1] (rejection sampling) or raw bytes."""
    _, _, qlen = ALL_CURVES[curve]
    g = rng(tag)
    raw = g.integers(0, 256, size=(n, qlen), dtype=np.uint8)
    if below_q:
        q = ORDER[curve]
        top = (1 << (q.bit_length() - 8 * (qlen - 1))) - 1   # bitlen(q) is not a multiple of 8 for P-521
        raw[:, 0] &= top
        for i in range(n):
            while True:
                v = int.from_bytes(raw[i].tobytes(), "big")
                if 0 < v < q:
                    break
                raw[i] = g.integers(0, 256, size=qlen, dtype=np.uint8)
                raw[i, 0] &= top
    return raw


def edge_scalars(curve: str) -> np.ndarray:
    """The adversarial scalars of SURVEY.md §8a's edge table."""
    _, _, qlen = ALL_CURVES[curve]
    q = ORDER[curve]
    vals = [0, 1, 2, 3, q - 2, q - 1, q, q + 1, (1 << (8 * qlen)) - 1, 1 << (8 * qlen - 1), 0x10, 0x100, 1 << 16,
            (1 << 16) - 1, 1 << 64, q >> 1, (q >> 1) + 1]
    vals = [v % (1 << (8 * qlen)) for v in vals]
    return np.frombuffer(b"".join(v.to_bytes(qlen, "big") for v in vals), dtype=np.uint8).reshape(-1, qlen).copy()


def _buf(a):
    a = np.ascontiguousarray(a)
    return a.ctypes.data_as(ctypes.c_void_p)


def oracle_smul(curve: str, scalars: np.ndarray, points=None, nthreads: int = 8, lib=None):
    """(out[n,2plen], status[n]) from the oracle port (or the compiled reference with lib=ref_lib())."""
    _, plen, qlen = ALL_CURVES[curve]
    sc = np.ascontiguousarray(scalars, dtype=np.uint8).reshape(-1, qlen)
    n = sc.shape[0]
    out = np.zeros((n, 2 * plen), dtype=np.uint8)
    st = np.zeros(n, dtype=np.int8)
    pts = np.ascontiguousarray(points, dtype=np.uint8) if points is not None else None
    if lib is None:
        fn = oracle_lib().ora_prj_pt_mul_batch
    else:
        fn = lib.ref_prj_pt_mul_batch
    rc = fn(curve.encode(), n, _buf(sc), qlen, _buf(pts) if pts is not None else None, _buf(out), _buf(st), nthreads)
    assert rc == 0
    return out, st


@reference_answer
def ref_smul(curve: str, scalars: np.ndarray, points=None):
    """(out, status) of the compiled reference's prj_pt_mul for the same inputs as oracle_smul."""
    return oracle_smul(curve, scalars, points, lib=ref_lib())


def oracle_verify(curve: str, sigs, pubkeys, digests, hlen: int, nthreads: int = 8) -> np.ndarray:
    _, plen, qlen = ALL_CURVES[curve]
    sg = np.ascontiguousarray(sigs, dtype=np.uint8).reshape(-1, 2 * qlen)
    n = sg.shape[0]
    pk = np.ascontiguousarray(pubkeys, dtype=np.uint8).reshape(n, 2 * plen)
    dg = np.ascontiguousarray(digests, dtype=np.uint8).reshape(n, hlen)
    v = np.zeros(n, dtype=np.int8)
    rc = oracle_lib().ora_ecdsa_verify_digest_batch(curve.encode(), n, _buf(sg), _buf(pk), _buf(dg), hlen, _buf(v),
                                                    nthreads)
    assert rc == 0
    return v


def oracle_sign(curve: str, privkeys, nonces, digests, hlen: int, nthreads: int = 8):
    _, plen, qlen = ALL_CURVES[curve]
    d = np.ascontiguousarray(privkeys, dtype=np.uint8).reshape(-1, qlen)
    n = d.shape[0]
    k = np.ascontiguousarray(nonces, dtype=np.uint8).reshape(n, qlen)
    dg = np.ascontiguousarray(digests, dtype=np.uint8).reshape(n, hlen)
    sig = np.zeros((n, 2 * qlen), dtype=np.uint8)
    st = np.zeros(n, dtype=np.int8)
    rc = oracle_lib().ora_ecdsa_sign_digest_batch(curve.encode(), n, _buf(d), _buf(k), _buf(dg), hlen, _buf(sig),
                                                  _buf(st), nthreads)
    assert rc == 0
    return sig, st


def hx(s: str) -> np.ndarray:
    return np.frombuffer(bytes.fromhex(s), dtype=np.uint8)


def hx_fit(s: str, nbytes: int) -> np.ndarray:
    """Big-endian integer string resized to nbytes (the reference's vectors zero-pad some P-521 keys to 68 bytes;
    nn_init_from_buf, nn/nn.c:479, accepts any length)."""
    v = int(s, 16) if s else 0
    return np.frombuffer(v.to_bytes(nbytes, "big"), dtype=np.uint8)


def make_signatures(curve: str, n: int, tag: int = 0, hlen: int = 32, corrupt_every: int = 0):
    """Synthetic ECDSA workload (SURVEY.md §8d.3): n tuples (sig, pubkey, digest) with distinct random keys,
    produced with the oracle's deterministic signer; every `corrupt_every`-th tuple is corrupted in a way that
    rotates over {flip bit in r, in s, in digest, in key, r = 0, s >= q}.  Returns (sigs, pubs, digests, expected)
    where expected comes from the oracle's verifier."""
    _, plen, qlen = ALL_CURVES[curve]
    d = random_scalars(curve, n, tag=1000 + tag)
    k = random_scalars(curve, n, tag=2000 + tag)
    dg = rng(3000 + tag).integers(0, 256, size=(n, hlen), dtype=np.uint8)
    pubs, st = oracle_smul(curve, d)
    assert (st == 0).all()
    sigs, st = oracle_sign(curve, d, k, dg, hlen)
    assert (st == 0).all()
    if corrupt_every:
        q = ORDER[curve]
        for j, i in enumerate(range(0, n, corrupt_every)):
            kind = j % 6
            if kind == 0:
                sigs[i, qlen - 1] ^= 1
            elif kind == 1:
                sigs[i, 2 * qlen - 1] ^= 1
            elif kind == 2:
                dg[i, 0] ^= 0x80
            elif kind == 3:
                pubs[i, plen - 1] ^= 1  # almost surely off the curve
            elif kind == 4:
                sigs[i, :qlen] = 0
            else:
                sigs[i, qlen:] = np.frombuffer(q.to_bytes(qlen, "big"), dtype=np.uint8)
    expected = oracle_verify(curve, sigs, pubs, dg, hlen)
    return sigs, pubs, dg, expected

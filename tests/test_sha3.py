"""SHA-3 (libecc_b200/csrc/sha3.cuh, constants from tools/gen_sha3_constants.py): the host build of the device code
against hashlib on every length around the block boundaries, and the generated constants file being up to date.  The
GPU test runs the same messages through eccb200_hash_batch and the reference's own src/hash."""
import ctypes
import hashlib
import os
import sys

import numpy as np
import pytest

from common import ROOT, hostsim_lib, ref_lib, reference_answer, rng

FN = {28: hashlib.sha3_224, 32: hashlib.sha3_256, 48: hashlib.sha3_384, 64: hashlib.sha3_512}
NAMES = {28: "SHA3_224", 32: "SHA3_256", 48: "SHA3_384", 64: "SHA3_512"}


def messages():
    g = rng(4242)
    lens = list(range(0, 150)) + [199, 200, 201, 271, 272, 273, 287, 288, 289, 1000]
    return [g.bytes(n) for n in lens]


@reference_answer
def ref_hash(name, msg):
    """The digest of msg by the reference's own src/hash."""
    buf = ctypes.create_string_buffer(64)
    ol = ctypes.c_uint32()
    assert ref_lib().ref_hash(name.encode(), msg, len(msg), buf, ctypes.byref(ol)) == 0
    return np.frombuffer(buf.raw[: ol.value], np.uint8)


def test_host_build_matches_hashlib():
    lib = hostsim_lib()
    for ds, fn in FN.items():
        for m in messages():
            out = ctypes.create_string_buffer(ds)
            lib.hostsim_sha3(ds, m, ctypes.c_uint64(len(m)), out)
            assert out.raw == fn(m).digest(), (ds, len(m))


def test_constants_file_is_up_to_date():
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import gen_sha3_constants
    path = os.path.join(ROOT, "libecc_b200", "csrc", "sha3_constants.inc")
    before, st = open(path).read(), os.stat(path)
    gen_sha3_constants.main()
    assert open(path).read() == before
    os.utime(path, ns=(st.st_atime_ns, st.st_mtime_ns))   # same bytes: keep the timestamp (no needless rebuild)


@pytest.mark.gpu
def test_device_sha3_matches_hashlib_and_reference():
    import libecc_b200
    eng = libecc_b200.Engine("SECP256R1", comb_window=8)
    msgs = messages()
    for ds, fn in FN.items():
        out = eng.hash_batch(NAMES[ds], msgs)
        assert out.shape == (len(msgs), ds)
        for m, o in zip(msgs, out):
            assert o.tobytes() == fn(m).digest()
        for m, o in list(zip(msgs, out))[::9]:
            assert ref_hash(NAMES[ds], m).tobytes() == o.tobytes()
    eng.close()

"""Every evidence file the documents cite under profiles/ exists (a judge follows these paths), and every round-2 file
listed in profiles/README.md is there."""
import glob
import os
import re

import numpy as np

from common import ROOT, reference_answer


def _exists(name):
    path = os.path.join(ROOT, "profiles", name)
    return bool(glob.glob(path)) if "*" in name else os.path.exists(path)


def test_cited_profile_files_exist():
    missing = []
    for md in ("DESIGN.md", "INTEGRATION.md", "README.md", os.path.join("profiles", "README.md")):
        txt = open(os.path.join(ROOT, md)).read()
        names = {m.group(1).rstrip(".") for m in re.finditer(r"profiles/([A-Za-z0-9_.\-\*]+)", txt)}
        if md.endswith(os.path.join("profiles", "README.md")):
            names |= {m.group(1) for m in re.finditer(r"`(r0[12]_[A-Za-z0-9_.\-\*]+)`", txt)}
        missing += [(md, n) for n in sorted(names) if n != "README.md" and not _exists(n)]
    assert not missing, missing


def test_bench_reads_an_existing_traffic_file():
    import json
    t = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
    entries = t if isinstance(t, list) else t.get("entries", t)
    assert entries, "profiles/ncu_traffic.json is empty"


@reference_answer
def ref_source_lines(path):
    """Number of lines of `path` in the reference's sources (the directory REF names, as for oracle/Makefile), -1 when
    there is no such file."""
    full = os.path.join(os.environ["REF"], path)
    return np.int64(sum(1 for _ in open(full, errors="ignore")) if os.path.isfile(full) else -1)


def test_reference_citations_point_at_existing_lines():
    """`path:line` citations of the reference in the documents, headers and sources name files that exist in the
    reference and are long enough."""
    files = ["DESIGN.md", "INTEGRATION.md", "README.md", "include/libecc_b200.h", "include/libecc_b200_dropin.h",
             "oracle/ecc_oracle.c", "oracle/ref_shim.c", "tests/dropin/dropin_harness.c"]
    files += [os.path.join("libecc_b200", "csrc", f) for f in
              ("dropin.cpp", "ec.cuh", "kernels.cuh", "fp.cuh", "msm.cuh", "msm_core.cuh", "eccb200.cu", "wire.cuh")]
    pat = re.compile(r"((?:src/)?(?:sig|curves|fp|nn|hash|ecdh|tests|utils|words|wycheproof_tests)/[A-Za-z0-9_\-./]+\.[ch]):(\d+)")
    bad, total = [], 0
    for f in files:
        for m in pat.finditer(open(os.path.join(ROOT, f), errors="ignore").read()):
            path, line = m.group(1), int(m.group(2))
            lines = ref_source_lines(path if path.startswith("src/") else "src/" + path)
            total += 1
            if lines < 0:
                bad.append((f, path, "missing"))
            elif line > lines:
                bad.append((f, path, line))
    assert total > 200 and not bad, bad

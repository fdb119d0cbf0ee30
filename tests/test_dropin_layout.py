"""include/libecc_b200_dropin.h mirrors the reference's struct layout: compile a probe against OUR header and compare
every sizeof/offsetof with the same facts taken from the reference's own headers (oracle/ref_shim.c: ref_abi_facts,
stored under tests/golden/reference/).
Also checks the magic-word constants the drop-in writes."""
import ctypes
import os
import subprocess
import tempfile

import numpy as np

from common import ROOT, ref_lib, reference_answer

PROBE = r"""
#include <stddef.h>
#include <stdio.h>
#include "libecc_b200_dropin.h"
int main(void) {
  unsigned long long f[] = {
    sizeof(eccb200_nn), offsetof(eccb200_nn, magic), offsetof(eccb200_nn, wlen),
    sizeof(eccb200_fp), offsetof(eccb200_fp, ctx), offsetof(eccb200_fp, magic),
    sizeof(eccb200_prj_pt), offsetof(eccb200_prj_pt, Y), offsetof(eccb200_prj_pt, Z), offsetof(eccb200_prj_pt, crv),
    offsetof(eccb200_prj_pt, magic),
    sizeof(eccb200_fp_ctx), offsetof(eccb200_fp_ctx, p_bitlen), offsetof(eccb200_fp_ctx, mpinv),
    offsetof(eccb200_fp_ctx, r), offsetof(eccb200_fp_ctx, r_square), offsetof(eccb200_fp_ctx, magic),
    sizeof(eccb200_ec_shortw_crv), offsetof(eccb200_ec_shortw_crv, b), offsetof(eccb200_ec_shortw_crv, a_monty),
    offsetof(eccb200_ec_shortw_crv, order), offsetof(eccb200_ec_shortw_crv, magic),
  };
  for (unsigned i = 0; i < sizeof(f)/sizeof(f[0]); i++) printf("%llu\n", f[i]);
  printf("%llu\n%llu\n%llu\n%llu\n", (unsigned long long)sizeof(eccb200_ec_pub_key),
         (unsigned long long)offsetof(eccb200_ec_pub_key, params), (unsigned long long)offsetof(eccb200_ec_pub_key, y),
         (unsigned long long)offsetof(eccb200_ec_pub_key, magic));
  printf("%d\n", ECCB200_NN_MAX_WORD_LEN);
  return 0;
}
"""


@reference_answer
def ref_abi_facts():
    buf = (ctypes.c_uint64 * 64)()
    k = ref_lib().ref_abi_facts(buf, 64)
    return np.array(buf[:k], np.uint64)


def test_struct_layout_matches_reference():
    with tempfile.TemporaryDirectory() as td:
        src = os.path.join(td, "probe.c")
        open(src, "w").write(PROBE)
        exe = os.path.join(td, "probe")
        subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), src, "-o", exe], check=True)
        ours = [int(x) for x in subprocess.run([exe], check=True, capture_output=True, text=True).stdout.split()]
    facts = [int(x) for x in ref_abi_facts()]
    # ref_abi_facts order: nn(3) fp(3) prj_pt(5) fp_ctx(6) crv(5) ec_params(7) ec_pub_key(4) NN_MAX_WORD_LEN
    ref_struct = facts[:22]
    ref_pub = facts[29:33]
    ref_nwords = facts[33]
    assert ours[:22] == ref_struct
    assert ours[22:26] == ref_pub
    assert ours[26] == ref_nwords == 27

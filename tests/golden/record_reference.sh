#!/bin/bash
# Records the unmodified reference's answers to the questions the tests ask it (tests/golden/reference/*.npz.xz, read by
# common.reference_answer) by running the tests with RECORD_REFERENCE=1 against oracle/_ref/libecc_ref.so.  With REF
# set to the directory of the reference's sources, the library is built from them first (oracle/Makefile).  Extra
# arguments go to pytest (default: -m "not gpu"); the GPU tests' answers are recorded with `-m gpu` on a B200, the
# library built beforehand.  Answers recorded earlier are kept; delete tests/golden/reference/ to start afresh.  The
# .npz.xz files are committed.
set -euo pipefail
here="$(cd "$(dirname "$0")" && pwd)"
root="$(cd "$here/../.." && pwd)"
if [ -n "${REF:-}" ]; then
    make -C "$root/oracle" -j8 ref REF="$REF" >/dev/null
fi
cd "$root"
if [ $# -eq 0 ]; then set -- -m "not gpu"; fi
RECORD_REFERENCE=1 python -m pytest -q -p no:cacheprovider tests "$@"
ls -la "$here/reference"

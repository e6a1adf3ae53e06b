#!/bin/bash
# GPU tests against the bounds-checked library (make -C yagre_mcmc_b200/csrc checked): a failed YG_CHK aborts the
# kernel with a device assert, so the suite passing means no checked index left its array.
#   bash tools/run_checked_tests.sh > checked_tests.log 2>&1
set -u
export YAGRE_B200_LIB=$PWD/tools/_build/libyagre_b200_checked.so
python - <<'PY'
from yagre_mcmc_b200 import _lib
print("library under test:", _lib.LIB_PATH)
PY
python -m pytest tests -m gpu -q 2>&1 | tail -4

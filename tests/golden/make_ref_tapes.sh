#!/bin/sh
# Re-record the reference's results that the parity tests replay where the oracle cannot be built
# (tests/golden/ref/<module>.<test>.xz, see tests/refharness.py).  Needs the reference sources, so that
# oracle/_ref/libt4ref.so can be compiled (make -C oracle all REF=<reference checkout>); the tests marked gpu record
# only on a machine with a CUDA device.  Extra arguments go to pytest, e.g. -m "not gpu" or -m gpu.
set -e
cd "$(dirname "$0")/../.."
make -C oracle all
T4_REF_RECORD="$PWD/tests/golden/ref" python -m pytest tests -q -p no:cacheprovider "$@"

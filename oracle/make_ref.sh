#!/bin/bash
# oracle/make_ref.sh -- place the UNMODIFIED reference (pmgbergen/porepy, pure Python) under oracle/_ref so that it
# travels to the GPU box with the snapshot (oracle/_ref/ is git-ignored, not gpurun-ignored): `bench.py --impl
# reference` and `cpu_baseline` time pp.Mpfa.discretize + pp.Mpsa.discretize there (kind: "reference"), and the
# plugin model tests can run against the real DevicePlan on a B200.  Nothing is compiled: the reference's hot path
# is NumPy / SciPy / numba; its package directory is copied as it is.  Never commit the copy.
set -e
here="$(cd "$(dirname "$0")" && pwd)"
src=${1:-/root/reference/src/porepy}
[ -d "$src" ] || { echo "reference not present at $src (nothing to do on the GPU box)"; exit 0; }
rm -rf "$here/_ref"
mkdir -p "$here/_ref"
cp -r "$src" "$here/_ref/porepy"
find "$here/_ref" -name __pycache__ -type d -prune -exec rm -rf {} +
# the reference's own unit tests of the path, in the same layout (collected there by tools/run_reference_tests.py)
if [ -d "$(dirname "$(dirname "$src")")/tests/numerics/fv" ]; then
  mkdir -p "$here/_ref/tests/numerics"
  cp -r "$(dirname "$(dirname "$src")")/tests/numerics/fv" "$here/_ref/tests/numerics/fv"
  find "$here/_ref/tests" -name __pycache__ -type d -prune -exec rm -rf {} +
fi
du -sh "$here/_ref"

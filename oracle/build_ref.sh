#!/usr/bin/env bash
# TEST INFRASTRUCTURE — builds the UNMODIFIED reference (microsoft/maro) from /root/reference into oracle/_ref/.
#
# oracle/_ref/ is git-ignored (outputs only; nothing from the reference enters history) but travels to the GPU
# box, where `bench.py --impl reference` times the reference's own Env/VectorEnv on the host cores.
# The product (maro_b200/) never imports anything from here.
#
# Recipe (SURVEY.md §8c): copy to a scratch dir (the reference tree is read-only) -> scripts/code_gen.py ->
# two Cython-3 build-compat patches (no behaviour change) -> cython -> build_ext -i -> copy the built package.
#   patch 1: frame.pyx `self.__dict__` -> `object.__getattribute__(self, "__dict__")` (Cython>=3 rejects the former)
#   patch 2: raw_backend.pyx query result buffer format "f" -> "d" (Cython-3 buffer dtype check)
set -euo pipefail
HERE="$(cd "$(dirname "${BASH_SOURCE[0]}")" && pwd)"
REF="${MARO_REFERENCE_ROOT:-/root/reference}"
PY="${PYTHON:-python}"  # the interpreter whose Cython / setuptools build the package
OUT="$HERE/_ref"
if [ ! -d "$REF/maro" ]; then
  echo "build_ref: $REF not present (GPU box) - keeping prebuilt $OUT" >&2
  exit 0
fi
# import-time stubs for the networking packages maro.rl's distributed workers import (absent from this image; the
# single-process rollout / training path the tests drive never touches them)
write_rl_stubs() {
  mkdir -p "$OUT/_stubs/zmq/eventloop" "$OUT/_stubs/tornado"
  cat > "$OUT/_stubs/zmq/__init__.py" <<'PY'
class _Unavailable:
    def __init__(self, *a, **k): raise RuntimeError("zmq is not installed in this image (import-time stub)")
Context = Poller = _Unavailable
DEALER = ROUTER = PUSH = PULL = POLLIN = IDENTITY = LINGER = 0
PY
  cat > "$OUT/_stubs/zmq/asyncio.py" <<'PY'
from . import Context, Poller  # noqa: F401
PY
  : > "$OUT/_stubs/zmq/eventloop/__init__.py"
  cat > "$OUT/_stubs/zmq/eventloop/zmqstream.py" <<'PY'
from .. import _Unavailable as ZMQStream  # noqa: F401
PY
  : > "$OUT/_stubs/tornado/__init__.py"
  cat > "$OUT/_stubs/tornado/ioloop.py" <<'PY'
class IOLoop:
    def __init__(self, *a, **k): raise RuntimeError("tornado is not installed in this image (import-time stub)")
PY
}
# the reference's example scripts (unmodified; run by tests/test_gpu_shim.py on top of the maro_b200 import shim)
copy_examples() {
  mkdir -p "$OUT/examples"
  for d in hello_world/cim hello_world/citi_bike vector_env cim/rl citi_bike/greedy vm_scheduling/rule_based_algorithm; do
    [ -d "$REF/examples/$d" ] || continue
    mkdir -p "$OUT/examples/$d"
    cp -r "$REF/examples/$d/." "$OUT/examples/$d/"
  done
  [ -f "$REF/examples/__init__.py" ] && cp "$REF/examples/__init__.py" "$OUT/examples/" || true
  [ -f "$REF/examples/cim/__init__.py" ] && cp "$REF/examples/cim/__init__.py" "$OUT/examples/cim/" || true
}
# the package = python modules + built extension modules (if any) + topology/meta data files of $1/maro, into $OUT/maro
copy_package() {
  "$PY" - "$1" "$OUT" <<'PY'
import os, shutil, sys
src, dst = sys.argv[1], sys.argv[2]
keep = (".py", ".so", ".yml", ".yaml", ".json", ".csv", ".txt", ".toml", ".bin")
for root, _, files in os.walk(os.path.join(src, "maro")):
    for f in files:
        if f.endswith(keep):
            rel = os.path.relpath(os.path.join(root, f), src)
            os.makedirs(os.path.dirname(os.path.join(dst, rel)), exist_ok=True)
            shutil.copy2(os.path.join(root, f), os.path.join(dst, rel))
PY
}
# the example scripts first: the hello cases of tests/test_gpu_shim.py need only them, not the compiled package below
copy_examples
write_rl_stubs
if [ -f "$OUT/maro/backends/frame.cpython-312-x86_64-linux-gnu.so" ] && [ -z "${FORCE:-}" ]; then
  echo "build_ref: $OUT already built"; exit 0
fi
# then the Python sources on their own: maro.rl is pure Python and runs on the maro_b200 shim (the maro.rl cases of
# tests/test_gpu_shim.py) even where the Cython build below fails; the compiled package replaces them
rm -rf "$OUT/maro"
copy_package "$REF"
TMP="$(mktemp -d /tmp/maro_ref_build.XXXXXX)"
trap 'rm -rf "$TMP"' EXIT
cp -r "$REF/maro" "$REF/setup.py" "$REF/scripts" "$TMP/"
[ -f "$REF/README.md" ] && cp "$REF/README.md" "$TMP/" || true
cd "$TMP"
export SKIP_DEPLOYMENT=TRUE
"$PY" scripts/code_gen.py
"$PY" - <<'PY'
import re, io
p = "maro/backends/frame.pyx"
s = open(p).read()
n = s.count("self.__dict__")
s = s.replace("self.__dict__", 'object.__getattribute__(self, "__dict__")')
open(p, "w").write(s)
print("frame.pyx: patched", n, "__dict__ sites")
p = "maro/backends/raw_backend.pyx"
s = open(p).read()
n = s.count('format="f"')
s = s.replace('format="f"', 'format="d"')
open(p, "w").write(s)
print("raw_backend.pyx: patched", n, "buffer formats")
PY
"$PY" -m cython maro/backends/backend.pyx maro/backends/np_backend.pyx maro/backends/raw_backend.pyx maro/backends/frame.pyx \
  --cplus -3 -E NODES_MEMORY_LAYOUT=ONE_BLOCK -X embedsignature=True
"$PY" setup.py -q build_ext -i -j 8 2>&1 | tail -5
rm -rf "$OUT/maro"
copy_package "$TMP"
# import-time stubs for packages absent from this image (only touched by the citi_bike import chain)
mkdir -p "$OUT/_stubs/holidays" "$OUT/_stubs/geopy"
cat > "$OUT/_stubs/holidays/__init__.py" <<'PY'
class _NoHolidays:
    def __contains__(self, item):
        return False
def US(*a, **k):
    return _NoHolidays()
PY
cat > "$OUT/_stubs/geopy/__init__.py" <<'PY'
PY
cat > "$OUT/_stubs/geopy/distance.py" <<'PY'
import math
class _D:
    def __init__(self, km): self.km = km; self.kilometers = km; self.meters = km * 1000.0
def distance(a, b):
    (la1, lo1), (la2, lo2) = a, b
    p1, p2 = math.radians(la1), math.radians(la2)
    h = math.sin((p2 - p1) / 2) ** 2 + math.cos(p1) * math.cos(p2) * math.sin(math.radians(lo2 - lo1) / 2) ** 2
    return _D(2 * 6371.0088 * math.asin(math.sqrt(h)))
PY
echo "build_ref: built into $OUT"

#!/usr/bin/env bash
# Build DuckDB (CLI + unittest) with the UNMODIFIED reference extension `duckpgq` and the B200
# override `duckpgq_b200` statically linked, in that load order.  Needs the reference sources
# (/root/reference, build container only); the binaries land in duckdb_ext/build/ (git-ignored,
# travels to the GPU box with gpurun).  libduckpgq_b200.so must have been built first
# (python -c "import __graft_entry__ as g; g.build()").
set -euo pipefail
REF=${REF:-/root/reference}
HERE="$(cd "$(dirname "$0")" && pwd)"
OUT="$HERE/build"
# DuckDB's CMakeLists copies compile_commands.json into <build dir>/../../.cache/clangd, so the build dir sits
# two levels below a directory of this user's own (a build dir right under /tmp would aim that copy at /.cache).
BUILD=${BUILD:-${TMPDIR:-/tmp}/duckpgq_b200-$(id -u)/build/release}
JOBS=${JOBS:-$(nproc)}
if [ ! -d "$REF/duckdb/src" ]; then
  echo "reference sources not present at $REF - cannot build the DuckDB shim here" >&2; exit 0
fi
mkdir -p "$OUT" "$BUILD"
cmake -G Ninja -DEXTENSION_STATIC_BUILD=1 \
  -DDUCKDB_EXTENSION_CONFIGS="$HERE/extension_config.cmake" -DPGQ_REFERENCE_DIR="$REF" \
  -DCMAKE_CXX_STANDARD=17 -DOVERRIDE_GIT_DESCRIBE=v1.5.0-0-g86cc0b4b98 \
  -DUNITTEST_ROOT_DIRECTORY="$REF/" -DENABLE_UNITTEST_CPP_TESTS=FALSE \
  -DENABLE_EXTENSION_AUTOLOADING=0 -DENABLE_EXTENSION_AUTOINSTALL=0 \
  -DCMAKE_BUILD_TYPE=Release -S "$REF/duckdb" -B "$BUILD"
cmake --build "$BUILD" -j"$JOBS"
cp "$BUILD/duckdb" "$OUT/duckdb_b200"
cp "$BUILD/test/unittest" "$OUT/unittest_b200"
cp "$BUILD/src/libduckdb.so" "$OUT/libduckdb.so"  # unittest links it dynamically: tests run with LD_LIBRARY_PATH=$OUT
strip "$OUT/duckdb_b200" "$OUT/unittest_b200" || true
ls -la "$OUT"

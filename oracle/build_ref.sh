#!/usr/bin/env bash
# Build the UNMODIFIED reference (DuckDB + the duckpgq extension statically linked)
# out-of-tree from the read-only sources under /root/reference, and keep only the
# binaries under oracle/_ref/ (git-ignored; travels to the GPU box with gpurun).
#
# This is test/bench infrastructure: the product (duckpgq_extension_b200/) never
# links, loads or executes anything produced here.
#
# Recipe = SURVEY.md §8c (flags mirror extension-ci-tools/makefiles/duckdb_extension.Makefile:120,170-173).
# No reference SOURCES are copied into the repo; only the built binaries land in oracle/_ref/.
set -euo pipefail
REF=${REF:-/root/reference}
HERE="$(cd "$(dirname "$0")" && pwd)"
OUT="$HERE/_ref"
# DuckDB's CMakeLists copies compile_commands.json into <build dir>/../../.cache/clangd, so the build dir sits
# two levels below a directory of this user's own (a build dir right under /tmp would aim that copy at /.cache).
BUILD=${BUILD:-${TMPDIR:-/tmp}/duckpgq_ref-$(id -u)/build/release}
JOBS=${JOBS:-$(nproc)}

if [ -x "$OUT/duckdb" ] && [ -x "$OUT/unittest" ] && [ -z "${FORCE:-}" ]; then
  echo "oracle/_ref already built"; exit 0
fi
if [ ! -d "$REF/duckdb/src" ]; then
  echo "reference sources not present at $REF - nothing to build" >&2; exit 0
fi
mkdir -p "$OUT" "$BUILD"
cmake -G Ninja -DEXTENSION_STATIC_BUILD=1 \
  -DDUCKDB_EXTENSION_CONFIGS="$REF/extension_config.cmake" \
  -DCMAKE_CXX_STANDARD=17 -DOVERRIDE_GIT_DESCRIBE=v1.5.0-0-g86cc0b4b98 \
  -DUNITTEST_ROOT_DIRECTORY="$REF/" -DENABLE_UNITTEST_CPP_TESTS=FALSE \
  -DENABLE_EXTENSION_AUTOLOADING=0 -DENABLE_EXTENSION_AUTOINSTALL=0 \
  -DCMAKE_BUILD_TYPE=Release -S "$REF/duckdb" -B "$BUILD"
cmake --build "$BUILD" -j"$JOBS"
cp "$BUILD/duckdb" "$OUT/duckdb"
cp "$BUILD/test/unittest" "$OUT/unittest"
cp "$BUILD/src/libduckdb.so" "$OUT/libduckdb.so"  # unittest links it dynamically: tests run with LD_LIBRARY_PATH=$OUT
strip "$OUT/duckdb" "$OUT/unittest" || true
echo "built: $(ls -la "$OUT")"

#!/bin/bash
# Builds the UNMODIFIED reference (GrokImageCompression/Grok; source tree in GROK_SRC) with its own CMake build,
# following SURVEY.md 8c's recipe, into oracle/_ref/grok/ (git-ignored; like the rest of oracle/_ref it goes along
# with a built tree to the machine that runs the tests).
#   oracle/_ref/grok/bin/{libgrokj2k.so*, grk_compress, grk_decompress, grk_dump}   -- stock, loader-enabled
# The source tree is read where it lies (out-of-tree build); nothing is copied into the repo's history.
# -DGRK_BUILD_PLUGIN_LOADER is passed as a compiler definition (the CMake option of that name wants the
# private plugin submodule, CMakeLists.txt L225-230); the sources are unmodified.
set -e
HERE="$(cd "$(dirname "$0")" && pwd)"
SRC="${GROK_SRC:?the Grok source tree}"
BLD="${GROK_BUILD_DIR:-$HERE/_build/stock}"
OUT="${GROK_OUT_DIR:-$HERE/_ref/grok}"
[ -d "$SRC/src/lib/core" ] || { echo "no reference tree at $SRC"; exit 0; }
SHIM="$HERE/_build/fmt-shim"
mkdir -p "$SHIM/include" "$BLD" "$OUT/bin"
if [ ! -d "$SHIM/include/fmt" ]; then
  # spdlog v2 normally fetches fmt from the network; torch ships the fmt headers -> header-only shim
  cp -r "$(python3 -c 'import torch,os;print(os.path.dirname(torch.__file__))')/include/fmt" "$SHIM/include/"
  cat > "$SHIM/fmtConfig.cmake" <<'EOS'
if(NOT TARGET fmt::fmt)
  add_library(fmt::fmt INTERFACE IMPORTED)
  set_target_properties(fmt::fmt PROPERTIES
    INTERFACE_INCLUDE_DIRECTORIES "${CMAKE_CURRENT_LIST_DIR}/include"
    INTERFACE_COMPILE_DEFINITIONS "FMT_HEADER_ONLY=1")
endif()
set(fmt_FOUND TRUE)
EOS
fi
[ -f "$BLD/build.ninja" ] || cmake -S "$SRC" -B "$BLD" -G Ninja -DCMAKE_BUILD_TYPE=Release -DBUILD_TESTING=OFF \
      -DGRK_BUILD_CORE_SWIG_BINDINGS=OFF -DGRK_BUILD_JPEG=OFF -DSPDLOG_FMT_EXTERNAL=ON -Dfmt_DIR="$SHIM" \
      -DCMAKE_CXX_FLAGS=-DGRK_BUILD_PLUGIN_LOADER ${GROK_CMAKE_EXTRA} > "$BLD/cmake.log" 2>&1
ninja -C "$BLD" grk_compress grk_decompress grk_dump > "$BLD/ninja.log" 2>&1
# real files, no symlinks (the snapshot that travels to the GPU box may not keep them)
rm -f "$OUT"/bin/*
for f in libgrokj2k.so.1 libgrokj2kcodec.so.1 grk_compress grk_decompress grk_dump; do cp -L "$BLD/bin/$f" "$OUT/bin/$f"; done
# the reference-arm harness (baseline/grk_ref_bench.cpp): public API only (grok.h + the generated grk_config.h)
g++ -O2 -std=c++20 -shared -fPIC -o "$OUT/bin/libgrk_ref_bench.so" "$HERE/../baseline/grk_ref_bench.cpp" \
    -I"$SRC/src/lib/core" -I"$BLD/src/lib/core" -L"$OUT/bin" -l:libgrokj2k.so.1 -Wl,-rpath,'$ORIGIN'
ls -la "$OUT/bin"

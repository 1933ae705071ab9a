#!/bin/bash
# Builds the reference WITH baseline/patches/*.patch applied (the multi-tile plugin seam, SURVEY.md 8b) into
# oracle/_ref/grok_patched/bin/.  The patch is applied to a scratch copy of the source tree (GROK_SRC) under
# oracle/_build/; the tree itself is never written.  The unmodified build (oracle/build_grok.sh -> oracle/_ref/grok)
# stays the reference arm; this one is only the host that exercises the patched per-tile binding in tests.
set -e
HERE="$(cd "$(dirname "$0")" && pwd)"
SRC="${GROK_SRC:?the Grok source tree}"
PATCHES="$HERE/../baseline/patches"
[ -d "$SRC/src/lib/core" ] || { echo "no reference tree at $SRC"; exit 0; }
COPY="$HERE/_build/patched_src"
if [ ! -f "$COPY/.patched" ] || [ "$PATCHES/0001-multi-tile-plugin-encode-decode.patch" -nt "$COPY/.patched" ]; then
  rm -rf "$COPY"; mkdir -p "$HERE/_build"
  cp -r "$SRC" "$COPY"; rm -rf "$COPY/.git"; chmod -R u+w "$COPY"
  for p in "$PATCHES"/*.patch; do patch -s -p1 -d "$COPY" < "$p"; done
  touch "$COPY/.patched"
fi
GROK_SRC="$COPY" GROK_BUILD_DIR="$HERE/_build/patched" GROK_OUT_DIR="$HERE/_ref/grok_patched" bash "$HERE/build_grok.sh"

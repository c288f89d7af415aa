#!/bin/bash
# Three deliberately broken builds of the PNG decoder, each built in a temporary copy of the tree (the checkout is
# never touched), must fail the decoder's test files and leave the existing tests of the image-file code passing.
#   paeth     the Paeth predictor replaced by Up
#   midtoken  a match token ended after its length, so windows synchronise inside a token (before its distance)
#   overlap   a match byte pointing to p - d, and a source before the resolved segment not read from the final bytes
# Each is a compile-time switch of png_inflate.h / png_decode.cu, set through ATTWARP_NVCC_EXTRA; the copy keeps the
# tree's object cache and rebuilds png_decode.o only (the one object the switches change).
# Usage: profiles/png_decode_broken_builds.sh [out_dir]    (one summary line per build, pytest tails in out_dir)
set -u
ROOT=$(cd "$(dirname "$0")/.." && pwd)
OUT=${1:-$(mktemp -d)}
mkdir -p "$OUT"
OUT=$(cd "$OUT" && pwd)
for variant in paeth midtoken overlap; do
    TMP=$(mktemp -d)
    cp -r "$ROOT/." "$TMP/"
    rm -rf "$TMP/.git" "$TMP/attwarp_b200/csrc/build/png_decode.o"
    case $variant in
    paeth)    flag=-DAW_PNG_BROKEN_PAETH_AS_UP ;;
    midtoken) flag=-DAW_PNG_BROKEN_SYNC_MID_TOKEN ;;
    overlap)  flag=-DAW_PNG_BROKEN_OVERLAP ;;
    esac
    (cd "$TMP" && ATTWARP_NVCC_EXTRA=$flag python -m attwarp_b200.build > "$OUT/build_$variant.log" 2>&1) \
        || { echo "$variant: build failed"; exit 1; }
    (cd "$TMP" && python -m pytest -q -p no:cacheprovider tests/test_gpu_png_decode.py > "$OUT/new_$variant.log" 2>&1)
    new=$(tail -1 "$OUT/new_$variant.log")
    # the existing tests of the code next to the decoder: image files, the C ABI, PNG encode and JPEG decode
    (cd "$TMP" && python -m pytest -q -p no:cacheprovider tests/test_image_io.py tests/test_cabi_symbols.py \
        tests/test_png_host.py tests/test_gpu_png.py tests/test_gpu_jpeg.py tests/test_save_warped_image.py \
        > "$OUT/existing_$variant.log" 2>&1)
    old=$(tail -1 "$OUT/existing_$variant.log")
    echo "$variant | new files: $new | existing suite: $old"
    rm -rf "$TMP"
done

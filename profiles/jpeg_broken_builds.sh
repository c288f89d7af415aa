#!/bin/bash
# Three deliberately broken builds of the JPEG decoder, each built in a temporary copy of the tree (the checkout is
# never touched), must fail the decoder's test files and leave the existing tests of the image-file code passing.
#   upsample  fancy up-sampling replaced by sample replication
#   dcreset   the DC predictor not reset at RSTn (a prefix over the whole file instead of the interval)
#   syncpos   sub-sequence synchronisation accepted on the bit position alone
# Usage: profiles/jpeg_broken_builds.sh [out_dir]    (one summary line per build, pytest tails in out_dir)
set -u
ROOT=$(cd "$(dirname "$0")/.." && pwd)
OUT=${1:-$(mktemp -d)}
mkdir -p "$OUT"
OUT=$(cd "$OUT" && pwd)
for variant in upsample dcreset syncpos; do
    TMP=$(mktemp -d)
    cp -r "$ROOT/." "$TMP/"
    rm -rf "$TMP/.git"
    H="$TMP/attwarp_b200/csrc/jpeg_decode.h"
    K="$TMP/attwarp_b200/csrc/jpeg.cu"
    case $variant in
    upsample) sed -i 's/    switch (mode) {/    switch (mode == kFull ? (int)kFull : (int)kReplicate) {/' "$H"
              grep -q 'switch (mode == kFull' "$H" || { echo "$variant: patch did not apply"; exit 1; } ;;
    dcreset)  sed -i 's/ - (a > 0 ? (uint32_t)J.win\[a - 1\].cum_dc\[c\] : 0u)//' "$K"
              grep -q 'cum_dc\[c\] : 0u' "$K" && { echo "$variant: patch did not apply"; exit 1; } ;;
    syncpos)  sed -i 's/if (!fixed \&\& sx\[t - 1\] != entry) {/if (!fixed \&\& state_pos(sx[t - 1]) != state_pos(entry)) {/; s/while (!g.first \&\& ent != J.win\[w\].entry) {/while (!g.first \&\& state_pos(ent) != state_pos(J.win[w].entry)) {/' "$K"
              [ "$(grep -c 'state_pos(sx\[t - 1\]) != state_pos(entry)\|state_pos(ent) != state_pos(J.win' "$K")" = 2 ] || { echo "$variant: patch did not apply"; exit 1; } ;;
    esac
    (cd "$TMP" && python -m attwarp_b200.build > "$OUT/build_$variant.log" 2>&1) || { echo "$variant: build failed"; exit 1; }
    (cd "$TMP" && python -m pytest -q -p no:cacheprovider tests/test_jpeg_host.py tests/test_gpu_jpeg.py > "$OUT/new_$variant.log" 2>&1)
    new=$(tail -1 "$OUT/new_$variant.log")
    # the existing tests of the code next to the decoder: image files, the C ABI, PNG encode, save_warped_image
    (cd "$TMP" && python -m pytest -q -p no:cacheprovider tests/test_image_io.py tests/test_cabi_symbols.py \
        tests/test_png_host.py tests/test_gpu_png.py tests/test_save_warped_image.py tests/test_gpu_overlay.py \
        > "$OUT/existing_$variant.log" 2>&1)
    old=$(tail -1 "$OUT/existing_$variant.log")
    echo "$variant | new files: $new | existing suite: $old"
    rm -rf "$TMP"
done

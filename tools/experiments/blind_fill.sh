#!/bin/bash
# RECORD of an experiment (last of four variants of this script): the VOXCARVE_PATCH_BLOCKS / VOXCARVE_BLIND_BLOCKS /
# VOXCARVE_BLIND_LATE_PROBE switches it drove were removed again afterwards (results: profiles/r2B_fill_probes.txt).
# VOXCARVE_BLIND_FILL=0|1 was removed later as well: the blind fill + patch pass is the only fill of a fresh carve.
for c in C4 C5; do for mode in "1 1" "1 2" "1 4"; do set -- $mode
  echo "== $c blind=$1 patch_blocks_per_sm=$2"
  VOXCARVE_BLIND_FILL=$1 VOXCARVE_PATCH_BLOCKS=$2 python tools/profile_carve.py --config $c --reps 6 2>&1 | grep "carve ms\|executed" | sort | head -2
  VOXCARVE_BLIND_FILL=$1 VOXCARVE_PATCH_BLOCKS=$2 python tools/slab_timing.py --config $c --parts 1,8 --reps 5 2>&1 | grep "^N="
done; done

#!/bin/bash
# RECORD of an experiment: the VOXCARVE_FILL switch it drives was removed again afterwards (results: profiles/r2B_fill_probes.txt;
# DESIGN.md s.4 'The fill, measured').  VOXCARVE_COMPRESSIBLE still exists; VOXCARVE_BLIND_FILL=0, which later selected the
# fused flag-driven fill, was removed as well.
# carve time with the volumes in compressible / plain memory and the fill pass fused into / run before the per-voxel kernel
for c in C4 C5; do for comp in 1 0; do for fill in fused before; do
  echo "== $c compressible=$comp fill=$fill"
  VOXCARVE_COMPRESSIBLE=$comp VOXCARVE_FILL=$fill python tools/profile_carve.py --config $c --reps 6 2>&1 | grep "carve ms\|executed" | sort | head -2
  VOXCARVE_COMPRESSIBLE=$comp VOXCARVE_FILL=$fill python tools/slab_timing.py --config $c --parts 8 --reps 5 2>&1 | grep "^N="
done; done; done

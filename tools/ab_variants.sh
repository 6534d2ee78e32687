#!/bin/bash
# A/B of kernel build variants on the GPU box: tools/ab_variants.sh <tag> [ENV=VAL ...] [-- bench args...]
# libs = wave-fenics_b200/libwavefx*.so.  Prints one line per library: tag, library, ms per apply
# (median window), fraction of the HBM peak, shared memory per CTA.
tag=$1; shift
envs=()
while [ $# -gt 0 ] && [ "$1" != "--" ]; do envs+=("$1"); shift; done
[ "$1" = "--" ] && shift
for lib in wave-fenics_b200/libwavefx*.so; do
  [ -f "$lib" ] || continue
  out=$(env "${envs[@]}" WFX_LIB=$PWD/$lib python bench.py --no-rk4 --no-cpu-baseline --no-affine --windows 5 --steps 100 --sustain-s 0 "$@" 2>&1 | tail -1)
  echo "$tag ${envs[*]} $(basename $lib) $(echo "$out" | python -c "import json,sys; d=json.loads(sys.stdin.read()); print('%.4f ms  frac %.3f  min %.4f  %s  parity %.1e' % (d['ms_per_step'], d['roofline']['frac'], min(w / k for w, k in zip(d['windows_ms'], d['window_steps'])), d['config']['kernel'], d['parity']['rel_l2_vs_cell_kernel']))" 2>&1 | tail -1)"
done

# usage: bash tools/lin32_ab.sh [reps] [variant ...]
# A/B of k2_render_lin builds in one session: for each repetition and each workload, bench.py once per library,
# alternating.  "base" is variants/libhmrm_base.so (a build of the parent commit), "new" the in-tree libhmrm.so,
# any other name variants/libhmrm_<name>.so (python -c "import build; build.build_variant('c5', ['-DHMRM_LIN_CTAS=5'])"
# from heightmap-ray-marcher_b200/).  Prints the card, its power limit, one line per run, then compares the
# --dump-outputs frames of every variant with base's, on stdout (profiles/r09_lin32_ab.txt is such a run).
set -u
reps=${1:-3}; shift || true
variants=${*:-base new}
tmp=$(mktemp -d)
say() { echo "$@"; }
lib_of() { if [ "$1" = new ]; then echo heightmap-ray-marcher_b200/libhmrm.so; else echo heightmap-ray-marcher_b200/variants/libhmrm_$1.so; fi; }
say "$(nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv,noheader | head -1)"
say "variants: $variants"
fields='import json,sys; d=json.loads(sys.stdin.read().strip().splitlines()[-1]); r=d.get("roofline",{}); print("ms_per_step %.5f kernel_ms %.5f fetches_per_frame %.1f ref_steps_per_frame %.1f" % (d["ms_per_step"], r.get("kernel_ms", float("nan")), d["fetches_per_frame"], d["ref_steps_per_frame"]))'
for rep in $(seq 1 $reps); do
  for wl in flythrough4k ortho4k spherical1080 sample720 bands8k; do
    for v in $variants; do
      line=$(HMRM_LIBRARY=$PWD/$(lib_of $v) python bench.py --gpus 1 --workload $wl --no-cpu-baseline 2>$tmp/err | python -c "$fields" 2>&1) || line="FAILED: $(tail -2 $tmp/err)"
      say "rep $rep $wl $v $line"
    done
  done
done
# the frames: every variant's --dump-outputs against base's, byte for byte
for wl in flythrough4k ortho4k spherical1080 sample720 bands8k; do
  for v in $variants; do
    HMRM_LIBRARY=$PWD/$(lib_of $v) python bench.py --gpus 1 --workload $wl --no-cpu-baseline --steps 3 --warmup 1 \
      --dump-outputs $tmp/$wl.$v > /dev/null 2>$tmp/err || say "dump $wl $v FAILED: $(tail -2 $tmp/err)"
  done
  for v in $variants; do
    [ "$v" = base ] && continue
    same=$(python -c "
import numpy as np, sys, pathlib
a, b = pathlib.Path(sys.argv[1]), pathlib.Path(sys.argv[2])
fa = sorted(p.relative_to(a) for p in a.rglob('*.npy'))
ok = bool(fa) and fa == sorted(p.relative_to(b) for p in b.rglob('*.npy')) and all(
    np.load(a / f).tobytes() == np.load(b / f).tobytes() for f in fa)
print(('byte-equal' if ok else 'DIFFERENT') + ' (%d arrays)' % len(fa))" $tmp/$wl.base $tmp/$wl.$v 2>&1)
    say "dump $wl $v vs base: $same"
  done
done
rm -rf $tmp

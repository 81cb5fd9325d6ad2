# usage: bash tools/sweep_launch.sh "threads ctas" ...   — rebuilds libhmrm.so with each launch shape of k2_render_lin
for cfg in "$@"; do
  set -- $cfg
  echo "== threads=$1 ctas/SM=$2"
  HMRM_NVCC_EXTRA="-DHMRM_LIN_THREADS=$1 -DHMRM_LIN_CTAS=$2 -DHMRM_LIN_CTAS_LARGE=$2" python heightmap-ray-marcher_b200/build.py --force > /dev/null 2>&1 || echo build failed
  for wl in flythrough4k ortho4k spherical1080; do
    python tools/profile_frame.py --frames 6 --workload $wl | awk -v w=$wl 'NR>1 {s+=$4; n++} END {printf "   %-14s %.3f ms\n", w, s/n}'
  done
done

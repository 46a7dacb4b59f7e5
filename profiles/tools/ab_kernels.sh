# usage: VARIANTS="b200 a3" LAYOUT=pipeline [OUT=dir] bash profiles/tools/ab_kernels.sh
#   per variant library: un-profiled step time of the C4 workload (1M envs), then per-kernel ncu durations ($OUT/ab_<lib>.csv)
OUT=${OUT:-profile_out}
mkdir -p $OUT
LAYOUT=${LAYOUT:-pipeline}
for lib in ${VARIANTS:-b200}; do
  export DOCKAUV_LIB=$PWD/gym_dockauv_b200/_lib/libdockauv_$lib.so
  echo "== $lib"
  python profiles/tools/try_layout.py $LAYOUT 1048576 100 2>&1 | tail -1 | cut -c1-60
  ncu --metrics gpu__time_duration.sum --clock-control none -k "regex:dynamics_kernel|rays_finish|rays_thread|episode_end|step_warp|step_tpe" --launch-skip 400 -c 80 --csv --log-file $OUT/ab_$lib.csv python profiles/tools/run_scenario.py ObstaclesDocking3d $LAYOUT 3 125 > /dev/null 2>&1
  python profiles/tools/kernel_times.py $OUT/ab_$lib.csv
done

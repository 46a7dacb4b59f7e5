# full ncu capture of one steady-state step of the pipeline layout (C4, two halves x three launches): $OUT/prof_pipe_$TAG.ncu-rep
TAG=${TAG:-cur}
OUT=${OUT:-profile_out}
mkdir -p $OUT
python profiles/tools/run_scenario.py ObstaclesDocking3d pipeline 3 135 || exit 1
ncu --set full --clock-control none --import-source on -k "regex:dynamics_kernel|rays_finish|rays_thread|episode_end" --launch-skip 792 --launch-count 6 -f -o $OUT/prof_pipe_$TAG python profiles/tools/run_scenario.py ObstaclesDocking3d pipeline 3 135 > $OUT/prof_pipe_$TAG.log 2>&1

#!/bin/bash
# Tuning builds of the flagship kernel only (Panda, [MotionForceTask rank 6, JointTask]): tools/tune.sh name "flags" [name "flags" ...]
# -> sai_primitives_b200/_tune/lib_<name>.so  (bench with SAI_B200_OSC_LIB=...)
cd "$(dirname "$0")/../sai_primitives_b200/csrc"
mkdir -p ../_tune
while [ $# -ge 2 ]; do
  name=$1; flags=$2; shift 2
  # the report of the full-task kernels: flag words with CV_FULL (bit 0, csrc/osc_launch.h) set
  ( make -j4 --no-print-directory BUILD=../_tune/build_$name OUT=../_tune/lib_$name.so DOFS=7 \
      EXTRA="-DOSC_TUNE_DOF7_ONLY ${ONLY_R--DOSC_ONLY_R=6} $flags" > ../_tune/make_$name.log 2>&1 \
    && echo "built $name: $(grep -A2 'osc_cycle_kernelILi7ELi6ELb1ELj[0-9]*[13579]E' ../_tune/build_$name/ptxas_n7.log | grep -o 'Used [0-9]* registers\|[0-9]* bytes spill stores' | tr '\n' ' ')" \
    || { echo "FAILED $name"; tail -5 ../_tune/make_$name.log; } ) &
done
wait

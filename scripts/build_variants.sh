#!/bin/bash
# Build A/B variants of the library next to the default one:  scripts/build_variants.sh "bounds:-DEG_DEBUG_BOUNDS" "<name>:-D<switch>"
# -> eirgrid_b200/libeg_<name>.so each (picked up by scripts/gpu_ab.sh, which times every libeg_*.so on both weight tables and
# prints a hash of all outputs). Remove them with:  rm -f eirgrid_b200/libeg_*.so; rm -rf eirgrid_b200/build/libeg_*
set -e
cd "$(dirname "$0")/.."
for v in "$@"; do
  name=${v%%:*}; flags=${v#*:}
  EIRGRID_LIB_NAME=libeg_$name.so EIRGRID_NVCC_EXTRA="$flags" python -m eirgrid_b200.build --force | tail -1
  grep -h "eg_episode_kernelILb0ELi0ELi[12]" -A2 eirgrid_b200/build/libeg_$name/build.log | grep -o "Used [0-9]* registers\|[0-9]* bytes spill stores" | paste -sd' '
  for k in ILb0ELi0ELi1 ILb0ELi0ELi2; do
    cuobjdump -sass eirgrid_b200/libeg_$name.so | awk -v k=$k '/Function :/{f=index($0,k)>0;next} f && /^ +\/\*[0-9a-f]+\*\/ /{c++} END{printf "  %s: %d instructions = %.1f KB\n", k, c, c*16/1024}'
  done
done

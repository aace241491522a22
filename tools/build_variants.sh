# builds tools/bin/lib_<name>.so for each "name:flags" argument, e.g.  tools/build_variants.sh "s4:-DQV_CODE_SHIFT=4" "s5:-DQV_CODE_SHIFT=5"
set -e
cd "$(dirname "$0")/../qcnn_gpu_b200/csrc"
mkdir -p ../../tools/bin
NV="/usr/local/cuda/bin/nvcc -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 -Xcompiler -fPIC,-fvisibility=hidden"
for spec in "$@"; do
  name=${spec%%:*}; flags=${spec#*:}
  $NV $flags -c qv_fused.cu -o /tmp/qv_fused_$name.o
  $NV -shared -o ../../tools/bin/lib_$name.so qv_formats.o qv_api.o qv_strip.o qv_layered.o /tmp/qv_fused_$name.o -cudart static
  echo built lib_$name.so "($flags)"
done

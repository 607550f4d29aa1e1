#!/usr/bin/env bash
# Builds newtonnet_b200/lib/libnewtonnet_b200.so for sm_100a (cross-compiles without a GPU).
set -euo pipefail
here="$(cd "$(dirname "${BASH_SOURCE[0]}")" && pwd)"
out="$here/../lib"
mkdir -p "$out" "$here/obj"
NVCC="${NVCC:-/usr/local/cuda/bin/nvcc}"
FLAGS=(-gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -lineinfo -Xcompiler -fPIC -Xcompiler -fvisibility=hidden
       --expt-relaxed-constexpr -DNN_BUILD)
pids=()
for f in nbr gemm_simt gemm_tc gemm_ts gemm_chain gemm_tn_tc message_tc pair_ops eval train_ops p2p md_ops neb hessian; do
  if [ ! -f "$here/obj/$f.o" ] || [ "$here/$f.cu" -nt "$here/obj/$f.o" ] || [ "$here/common.cuh" -nt "$here/obj/$f.o" ] || [ "$here/tc_common.cuh" -nt "$here/obj/$f.o" ] \
     || [ "$here/../../include/newtonnet_b200.h" -nt "$here/obj/$f.o" ]; then
    "$NVCC" "${FLAGS[@]}" ${NN_PTXAS_V:+-Xptxas -v} -c "$here/$f.cu" -o "$here/obj/$f.o" &
    pids+=($!)
  fi
done
for p in "${pids[@]:-}"; do [ -n "$p" ] && wait "$p"; done
"$NVCC" -Wno-deprecated-gpu-targets -shared -o "$out/libnewtonnet_b200.so" "$here"/obj/{nbr,gemm_simt,gemm_tc,gemm_ts,gemm_chain,gemm_tn_tc,message_tc,pair_ops,eval,train_ops,p2p,md_ops,neb,hessian}.o -lcudart
echo "built $out/libnewtonnet_b200.so"

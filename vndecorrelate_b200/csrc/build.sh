#!/usr/bin/env bash
# Builds libvnd_b200.so for sm_100a in-tree (vndecorrelate_b200/_lib/).  -fmad=false: the reference
# rounds after every numpy ufunc, so no multiply-add may be contracted anywhere in this library.
set -euo pipefail
here="$(cd "$(dirname "${BASH_SOURCE[0]}")" && pwd)"
out="$here/../_lib"
mkdir -p "$out"
NVCC="${NVCC:-/usr/local/cuda/bin/nvcc}"
"$NVCC" -std=c++17 -O3 -lineinfo -fmad=false --threads 0 \
  -gencode arch=compute_100a,code=sm_100a \
  -Xcompiler -fPIC,-O2 -shared -diag-suppress 177 \
  ${VND_PTXAS_V:+-Xptxas -v} \
  -o "$out/libvnd_b200.so" \
  ${VND_EXTRA_DEFS:-} \
  "$here/vnd_abi.cu" "$here/vnd_fir.cu" "$here/vnd_fir_window.cu" "$here/vnd_fir_tmem.cu" "$here/vnd_fir_ring.cu" "$here/vnd_post.cu" "$here/vnd_objective.cu" "$here/vnd_dsp.cu" "$here/vnd_batch.cu"
echo "built $out/libvnd_b200.so"

#!/usr/bin/env bash
# Builds libsurprise_b200.so (sm_100a only) next to the Python package.  Called by __graft_entry__.build().
set -euo pipefail
HERE="$(cd "$(dirname "${BASH_SOURCE[0]}")" && pwd)"
OUT="$HERE/../libsurprise_b200.so"
NVCC=${NVCC:-/usr/local/cuda/bin/nvcc}
FLAGS="-gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 -Xcompiler -fPIC -Xcompiler -Wall -Xptxas -v ${SB2_EXTRA_NVCC_FLAGS:-}"
mkdir -p "$HERE/obj"
pids=()
for f in api sim sim_gemm sim_general segmented predict sgd coclustering top_n top_n_eval rank_metrics; do
  ( $NVCC $FLAGS -c "$HERE/$f.cu" -o "$HERE/obj/$f.o" > "$HERE/obj/$f.log" 2>&1 || { cat "$HERE/obj/$f.log"; exit 1; } ) &
  pids+=($!)
done
rc=0
for p in "${pids[@]}"; do wait "$p" || rc=1; done
[ $rc -eq 0 ] || { echo "build failed"; exit 1; }
$NVCC -gencode arch=compute_100a,code=sm_100a -shared -o "$OUT" "$HERE"/obj/{api,sim,sim_gemm,sim_general,segmented,predict,sgd,coclustering,top_n,top_n_eval,rank_metrics}.o -lcudart_static -ldl -lrt -lpthread
echo "built $OUT"

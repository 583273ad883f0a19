#!/usr/bin/env bash
# Builds libaoenv_b200.so in-tree for sm_100a (nvcc cross-compiles without a GPU).
set -euo pipefail
cd "$(dirname "$0")"
OUT=${OUT:-../libaoenv_b200.so}
SRCS="api.cu atm.cu step.cu vk.cu gemm.cu wfs.cu wfs_fused.cu wfs_geo.cu pyr.cu ctrl.cu dm.cu"
[ -f psf.cu ] && SRCS="$SRCS psf.cu"
[ -f gemm_tc.cu ] && SRCS="$SRCS gemm_tc.cu"
NVCC=${NVCC:-/usr/local/cuda/bin/nvcc}
TMP="$OUT.tmp.$$"
set +e
# one object per source, compiled in parallel (the sources are independent translation units), then one link
OBJ=$(mktemp -d)
FLAGS="-gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 -Xcompiler -fPIC,-O2,-Wall -Xptxas -v ${NVCC_EXTRA:-}"
pids=""
for f in $SRCS; do
  $NVCC $FLAGS -c -o "$OBJ/${f%.cu}.o" "$f" > "$OBJ/${f%.cu}.log" 2>&1 &
  pids="$pids $!"
done
rc=0
for p in $pids; do wait $p || rc=1; done
cat "$OBJ"/*.log > build.log
if [ $rc -eq 0 ]; then
  $NVCC -gencode arch=compute_100a,code=sm_100a --shared -o "$TMP" "$OBJ"/*.o >> build.log 2>&1 || rc=1
fi
rm -rf "$OBJ"
set -e
grep -E "error|warning|spill|Used" build.log || true
if [ $rc -ne 0 ] || [ ! -f "$TMP" ]; then
  rm -f "$TMP"
  echo "BUILD FAILED (nvcc exit $rc); $OUT left untouched" >&2
  exit 1
fi
mv -f "$TMP" "$OUT"
echo "built $OUT"

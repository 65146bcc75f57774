#!/usr/bin/env bash
# Builds libvo_b200.so (sm_100a only) next to the Python package.  nvcc cross-compiles without a GPU.
set -euo pipefail
here="$(cd "$(dirname "${BASH_SOURCE[0]}")" && pwd)"
out="${here}/../libvo_b200.so"
obj="${here}/build"
mkdir -p "${obj}"
NVCC="${NVCC:-/usr/local/cuda/bin/nvcc}"
COMMON=(-gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 -Xcompiler -fPIC -Xcompiler -fvisibility=hidden
        -Xptxas -v --expt-relaxed-constexpr)
# pnp / orb / sift: no implicit FMA contraction, so the device rounds like the host restatements the parity tests use
# (explicit fused operations, where OpenCV itself fuses, are spelled out with __fmaf_rn)
# VO_TC_EXTRA: extra nvcc flags for the tensor-core matcher, e.g. -DVO_TC_PERSIST_MAX_TILES=<n>
declare -A EXTRA=( [pnp]="-fmad=false" [orb]="-fmad=false" [sift]="-fmad=false" [match_f32_tc]="${VO_TC_EXTRA:-}" )
pids=()
for src in api match_finalize match_u8 match_f32_simt match_f32_tc geometry pnp sequence conv_tc r2d2_net orb sift; do
  (
    "${NVCC}" "${COMMON[@]}" ${EXTRA[$src]:-} -c "${here}/${src}.cu" -o "${obj}/${src}.o" > "${obj}/${src}.log" 2>&1 \
      || { cat "${obj}/${src}.log"; exit 1; }
  ) &
  pids+=($!)
done
fail=0
for p in "${pids[@]}"; do wait "$p" || fail=1; done
[ "$fail" = 0 ] || { echo "build failed"; exit 1; }
"${NVCC}" -gencode arch=compute_100a,code=sm_100a -shared -o "${out}" "${obj}"/*.o -cudart static -Xlinker --exclude-libs=ALL
echo "built ${out}"

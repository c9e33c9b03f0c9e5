#!/usr/bin/env bash
# Builds libgte_b200.so (sm_100a only) in-tree next to the Python package.
# Usage: csrc/build.sh [extra nvcc flags]
set -euo pipefail
here="$(cd "$(dirname "${BASH_SOURCE[0]}")" && pwd)"
root="$(cd "$here/../.." && pwd)"
out="$here/../libgte_b200.so"
bdir="$here/build"
NVCC="${NVCC:-/usr/local/cuda/bin/nvcc}"
srcs=("$here"/gte_*.cu)
mkdir -p "$bdir"
objs=()
pids=()
for s in "${srcs[@]}"; do
  o="$bdir/$(basename "${s%.cu}").o"
  objs+=("$o")
  if [[ ! -f "$o" || "$s" -nt "$o" || -n "$(find "$here" "$root/include" \( -name '*.cuh' -o -name '*.h' \) -newer "$o" -print -quit)" ]]; then
    "$NVCC" -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 \
      -Xcompiler -fPIC -I"$root/include" -I"$here" "$@" -c "$s" -o "$o" &
    pids+=($!)
  fi
done
fail=0
for p in "${pids[@]:-}"; do
  if [[ -n "$p" ]]; then wait "$p" || fail=1; fi
done
if [[ $fail -ne 0 ]]; then echo "build.sh: compilation failed" >&2; exit 1; fi
"$NVCC" -gencode arch=compute_100a,code=sm_100a -shared -Xcompiler -fPIC -o "$out" "${objs[@]}" -lcudart
echo "built $out"

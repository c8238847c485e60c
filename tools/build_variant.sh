#!/bin/bash
# Builds the current working tree into build/libaki_<name>.so from its own object directory, for same-box A/B runs
# through AKI_MMA_LIB (tools only).  usage: tools/build_variant.sh <name> [extra nvcc flags]
#   tools/build_variant.sh trace -DAKI_FWD_TRACE     clock64 stamps (tools/fwd_trace.py, tools/bwd_trace.py)
#   tools/build_variant.sh trap -DAKI_MBAR_TRAP      a stuck mbarrier wait traps after 4 s (tools/stress.py)
#   tools/build_variant.sh ko_red -DKO_RED           backward knockout (attn_bwd_sm100.cu): timing only, wrong results
set -e
name=${1:?usage: tools/build_variant.sh <name> [extra nvcc flags]}; shift
root=$(cd "$(dirname "$0")/.." && pwd)
rm -rf "$root/build/obj_$name"
make -C "$root/aki_b200/csrc" -j OBJ="$root/build/obj_$name" OUT="$root/build/libaki_$name.so" EXTRA="$*"
echo built "$root/build/libaki_$name.so"

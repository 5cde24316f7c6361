#!/bin/bash
# profiles/sass_linear_tc.txt: the tcgen05 / TMEM / bulk-copy instructions of the shipped library, per kernel
# (cuobjdump -sass of graph_marl_b200/lib/libgraphmarl_b200.so; see /opt/skills/guides/B200_PROFILING.md for the mnemonics)
set -e
cd "$(dirname "$0")/.."
LIB=graph_marl_b200/lib/libgraphmarl_b200.so
OUT=${1:-profiles/sass_linear_tc.txt}
{
  echo "# cuobjdump -sass $LIB  (sm_100a)  -- per-function counts of tensor-core / TMEM / bulk-copy SASS"
  echo "# UTCHMMA = tcgen05.mma (kind::f16: bf16 operands, fp32 accumulate in TMEM); .2CTA = cta_group::2"
  echo "# LDTM = tcgen05.ld (TMEM -> registers); UTCBAR = tcgen05.commit -> mbarrier; UBLKCP = cp.async.bulk (TMA bulk copy)"
  echo "# function | UTCHMMA | UTCHMMA.2CTA | LDTM | UTCBAR | UBLKCP | SYNCS (mbarrier)"
  cuobjdump -sass "$LIB" | awk '
    /Function :/ { if (fn != "") print fn " | " a " | " b " | " c " | " d " | " e " | " f; fn=$3; a=b=c=d=e=f=0 }
    /UTCHMMA/ { a++; if ($0 ~ /2CTA/) b++ }
    /LDTM/ { c++ } /UTCBAR/ { d++ } /UBLKCP/ { e++ } /SYNCS/ { f++ }
    END { if (fn != "") print fn " | " a " | " b " | " c " | " d " | " e " | " f }' | awk -F'|' '$2+$4+$6 > 0' | c++filt | cut -c1-220
  echo
  echo "# excerpt: the MMA issue loop of linear_tc_kernel<256,3,EPI_LSTM,4> (first 60 tensor-core / barrier lines)"
  cuobjdump -sass "$LIB" | awk '/Function : .*linear_tc_kernelILi256ELi3ELi1ELi4EE/ {p=1} p && /Function :/ && !/linear_tc_kernelILi256ELi3ELi1ELi4EE/ {p=0} p' \
    | grep -E "UTCHMMA|UTCBAR|LDTM|UBLKCP|SYNCS|UTCATOMSWS|UTCCP" | head -60
} > "$OUT"
wc -l "$OUT"

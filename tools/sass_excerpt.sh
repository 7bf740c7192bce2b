#!/bin/bash
# profiles/r2_sass_excerpt.txt: the SASS mnemonics that prove the Blackwell-native paths (B200_PROFILING.md: tcgen05.mma ->
# UTC*MMA, tcgen05.ld -> LDTM, cp.async.bulk -> UBLKCP, mma.sync f64 -> DMMA), counted per kernel of the built library,
# plus the first lines around the first UTCHMMA / UTCMMA of the two tcgen05 kernels.
set -e
cd "$(dirname "$0")/.."
LIB=w-ofdm-optimization_b200/libwofdm.so
OUT=profiles/r2_sass_excerpt.txt
cuobjdump -sass $LIB > /tmp/wofdm_sass.txt
{
echo "# cuobjdump -sass $LIB  ($(date -u +%F), nvcc $(nvcc --version | grep release | sed 's/.*release //'))"
echo "# whole library: $(grep -c UTCHMMA /tmp/wofdm_sass.txt) UTCHMMA (tcgen05.mma, kind::f16 in ber_tconv*_kernel and mask_gemm_f16, kind::tf32 in gemm_power_tf32), $(grep -c LDTM /tmp/wofdm_sass.txt) LDTM (tcgen05.ld), $(grep -c UBLKCP /tmp/wofdm_sass.txt) UBLKCP (cp.async.bulk), $(grep -c DMMA /tmp/wofdm_sass.txt) DMMA (mma.sync f64), $(grep -c 'FFMA2\|FADD2\|FMUL2' /tmp/wofdm_sass.txt) packed FP32 (FFMA2/FADD2/FMUL2), $(grep -c UTMALDG /tmp/wofdm_sass.txt) UTMALDG"
echo "# per kernel (only kernels that contain one of them):"
awk '/Function :/ {name=$3} /UTCHMMA|UTC[A-Z]*MMA|LDTM|UBLKCP|DMMA|UCGABAR|SYNCS/ {split($0,a," "); for(i in a) if (a[i] ~ /^(UTC[A-Z]*MMA|LDTM|UBLKCP[.A-Z0-9]*|DMMA[.A-Z0-9]*|UCGABAR_[A-Z]*|SYNCS[.A-Z0-9]*)/) {sub(/\..*/,"",a[i]); c[name" "a[i]]++}} END {for (k in c) print c[k], k}' /tmp/wofdm_sass.txt | sort -k2,2 -k3,3 | c++filt | awk '{n=$1; $1=""; printf "%6d %s\n", n, $0}'
for pat in 'ber_tconv2_kernelILi256ELi256ELi9ELi2ELb0ELi1ELi21ELb0' 'gemm_power_tf32' 'mask_gemm_f16'; do
  echo
  echo "# ---- $pat: the first tensor-core issue sequence"
  awk -v pat="$pat" '/Function :/ {on = index($0, pat) > 0} on' /tmp/wofdm_sass.txt | grep -n -m1 "UTC[A-Z]*MMA" | cut -d: -f1 | { read n; awk -v pat="$pat" '/Function :/ {on = index($0, pat) > 0} on' /tmp/wofdm_sass.txt | sed -n "$((n-12)),$((n+14))p" | sed 's#/\* 0x[0-9a-f]* \*/##'; }
  echo "# ---- $pat: a tcgen05.ld (LDTM) batch"
  awk -v pat="$pat" '/Function :/ {on = index($0, pat) > 0} on' /tmp/wofdm_sass.txt | grep -n -m1 "LDTM" | cut -d: -f1 | { read n; awk -v pat="$pat" '/Function :/ {on = index($0, pat) > 0} on' /tmp/wofdm_sass.txt | sed -n "$((n-2)),$((n+8))p" | sed 's#/\* 0x[0-9a-f]* \*/##'; }
done
} > $OUT
wc -l $OUT

#!/bin/bash
# Writes profiles/r02_sass_excerpts.md: the hot loops of the shipped kernels as SASS (cuobjdump of the objects that are
# linked into esp-audio-libs_b200/libesp_audio_b200.so), with mnemonic counts.  Run after `make -C esp-audio-libs_b200/csrc`.
set -e
HERE=$(cd "$(dirname "$0")/.." && pwd)
B=$HERE/esp-audio-libs_b200/csrc/build
OUT=$HERE/profiles/r02_sass_excerpts.md
sass() { cuobjdump -sass -fun "$2" "$B/$1" | grep -E '^\s+/\*[0-9a-f]{4}\*/' | sed -E 's#/\* 0x[0-9a-f]+ \*/##; s/[[:space:]]+$//'; }
count() { sass "$1" "$2" | grep -oE "$3" | sort | uniq -c | tr '\n' ';'; }
{
echo "# SASS excerpts of the shipped sm_100a kernels (round 2)"
echo
echo "Produced by \`tools/sass_excerpts.sh\` from the object files linked into \`libesp_audio_b200.so\` (nvcc 12.9, -O3,"
echo "\`-gencode arch=compute_100a,code=sm_100a\`).  Mnemonics to look for: \`FFMA2\` (packed FP32 pair FMA, Blackwell),"
echo "\`UBLKCP\` (TMA bulk copy, \`cp.async.bulk\`), \`SYNCS\` (mbarrier), \`LDGSTS\` (cp.async)."
echo
K='_ZN4espb20espb_resample_kernelILb0ELb0EEEvNS_14ResampleParamsE'
echo "## espb_resample_kernel<EXACT=false, TMCAP=false> (4 warps, 2 stages, 32-row chunks) — the dominant kernel (fast mode)"
echo; echo "Mnemonic counts: $(count resample_kernel.cu.o $K 'FFMA2|UBLKCP|SYNCS\.[A-Z.0-9]+|LDS\.128|FFMA |FMUL |FADD |ATOMS[A-Z.0-9]*')"
echo; echo "One 4-row group of the inner loop (32 FFMA2 + 5 LDS.128 per row; x as a scalar-broadcast operand):"; echo; echo '```'
sass resample_kernel.cu.o $K | awk '/FFMA2/{c++} c>=1 && c<=40' | head -60
echo '```'; echo; echo "Stage release and TMA refill (last-arriver protocol):"; echo; echo '```'
sass resample_kernel.cu.o $K | grep -n -E "ATOMS|UBLKCP|SYNCS" | head -20
echo '```'
K='_ZN4espb20espb_resample_kernelILb1ELb0EEEvNS_14ResampleParamsE'
echo; echo "## espb_resample_kernel<EXACT=true, false> — exact mode: no fused multiply-add in the accumulation"
echo; echo "Mnemonic counts: $(count resample_kernel.cu.o $K 'FFMA2|FFMA |FMUL |FADD |UBLKCP')"
echo; echo '```'; sass resample_kernel.cu.o $K | awk '/FMUL/{c++} c>=1 && c<=12' | head -28; echo '```'
K=$(cuobjdump -sass $B/resample_fs_kernel.cu.o | grep "Function :" | grep "ILi2ELi4ELb0E" | awk '{print $3}')
echo; echo "## espb_resample_fs_kernel<SV=2, B=4, EXACT=false> — few-series form (one stereo stream)"
echo; echo "Mnemonic counts: $(count resample_fs_kernel.cu.o $K 'FFMA2|UBLKCP|SYNCS\.[A-Z.0-9]+|LDS\.64|LDS |LDGSTS[A-Z.0-9]*')"
echo; echo "Per tap and output: two LDS (coefficients of phase and phase+1), one LDS.64 (x of both channels), two FFMA2:"; echo; echo '```'
sass resample_fs_kernel.cu.o $K | awk '/FFMA2/{c++} c>=1 && c<=10' | head -30
echo '```'
K=$(cuobjdump -sass $B/biquad_kernel.cu.o | grep "Function :" | grep "biquad_tm_kernelILi2ELb0E" | awk '{print $3}')
echo; echo "## espb_biquad_tm_kernel<NSEC=2, FIRST_ORDER=false> — un-fused Direct-Form-I recurrence, TMA loads and stores"
echo; echo "Mnemonic counts: $(count biquad_kernel.cu.o $K 'FFMA |FMUL |FADD |UBLKCP[A-Z.0-9]*|SYNCS\.[A-Z.0-9]+')"
K=_ZN4espb27espb_transpose_flags_kernelILi2ELb0ELb1EEEvPKflliiPfliiiPi
echo; echo "## Staging overlap: espb_transpose_flags_kernel<CH=2, PLANAR=false, POLICY=true> and the resampler's wait"
echo; echo "\`PREEXIT\` is \`griddepcontrol.launch_dependents\` (the resampler, launched with the programmatic-stream-serialization"
echo "attribute, may start as soon as every CTA of this grid has executed it); one tile = four evict-first 128-bit loads and four"
echo "128-bit stores per thread, then fence + one counting atomic per CTA:"; echo; echo '```'
sass resample_kernel.cu.o $K | grep -E "PREEXIT|LDG|STG|BAR\.SYNC|MEMBAR|ATOMG|EXIT" | head -20
echo '```'; echo; echo "The waiting side, once per CTA of espb_resample_kernel<false,false> (acquire load of the tile counter, back-off,"
echo "trap after ~4 s, then the generic-to-async proxy fence before the first TMA copy of xt):"; echo; echo '```'
sass resample_kernel.cu.o _ZN4espb20espb_resample_kernelILb0ELb0EEEvNS_14ResampleParamsE | grep -E "STRONG\.GPU|NANOSLEEP|BPT|FENCE\.VIEW\.ASYNC|UBLKCP" | head -8
echo '```'
K=_ZN4espb23espb_resample_ni_kernelILi4ELi2ELi32ELb0ELb0EEEvNS_14ResampleParamsE
echo; echo "## espb_resample_ni_kernel<4, 2, 32, EXACT=false, TMCAP=false> — non-interpolating form, 4 series x 16 outputs per warp"
echo; echo "Mnemonic counts: $(count resample_ni_kernel.cu.o $K 'FFMA2|UBLKCP|LDS\.128|FFMA ')"
} > "$OUT"
echo "wrote $OUT ($(wc -l < "$OUT") lines)"

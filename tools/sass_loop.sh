#!/bin/bash
# usage: tools/sass_loop.sh <mangled kernel name> [context lines]
# SASS around the first MUFU.RCP of a rotation kernel (the substep loop), then the instruction mix of one unrolled substep
# of a pair kernel: from the fifth to the seventh MUFU.RCP (two per substep), i.e. the third substep.  Moves are counted
# outside the cold branch around the out-of-line bounce call only.  CPS_B200_LIB: another build of the library.
SO=${CPS_B200_LIB:-$(dirname "$0")/../cartpolesimulation_b200/libcps_b200.so}
K=$1; N=${2:-40}
T=$(mktemp)
cuobjdump -sass -fun "$K" "$SO" 2>/dev/null | grep -E "^\s+/\*[0-9a-f]{4}\*/" | sed -E 's/\/\* 0x[0-9a-f]+ \*\/\s*$//' > "$T"
cuobjdump -res-usage "$SO" 2>/dev/null | grep -A1 "$K" | tail -1
L=$(grep -n "MUFU.RCP" "$T" | head -1 | cut -d: -f1)
sed -n "$((L-12)),$((L+N))p" "$T" | cut -c1-100
awk -v a=5 -v b=7 '
/MUFU.RCP/ { r++ }
r >= a && r < b {
    op = $2; if (op ~ /^@/) op = $3
    if ($0 ~ /@!?P[0-9] +BRA/) cold = 1
    if (op ~ /^(FFMA2|FMUL2|FADD2)/) {
        packed[op]++; p++
        split("", seen); n = 0; s = $0
        while (match(s, /R[0-9]+(\.reuse)?\.F32x2/)) {
            reg = substr(s, RSTART, RLENGTH); sub(/\..*/, "", reg)
            if (!(reg in seen)) { seen[reg] = 1; n++ }
            s = substr(s, RSTART + RLENGTH)
        }
        if (op == "FFMA2" && n == 3) three++
    }
    if (!cold && op ~ /MOV/) mov++
    if ($0 ~ /BSYNC/) cold = 0
    tot++
}
END {
    printf "one substep (MUFU.RCP %d..%d): %d instructions; packed FP32 %d (FFMA2 %d, FMUL2 %d, FADD2 %d), FFMA2 with three distinct pairs %d, hot-path moves %d\n",
           a, b, tot, p, packed["FFMA2"], packed["FMUL2"], packed["FADD2"], three, mov
}' "$T"
rm -f "$T"

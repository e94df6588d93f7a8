#!/bin/bash
# one full ncu capture of the K2 kernel of q: tools/ncu_k2.sh <q> <N> <tag> [out dir]   (report + logs into the out dir,
# default $TMPDIR/ncu_k2)
cd "$(dirname "$0")/.."
q=$1; N=$2; tag=$3; out=${4:-${TMPDIR:-/tmp}/ncu_k2}
mkdir -p "$out"
python tools/bench_k2.py $q $N > "$out/${tag}_plain.log" 2>&1 || exit 1
ncu --set full --clock-control none --import-source on -k regex:zsolve -s 1 -c 1 -f -o "$out/$tag" \
    python tools/bench_k2.py $q $N > "$out/${tag}_ncu.log" 2>&1
ls -la "$out/$tag.ncu-rep"

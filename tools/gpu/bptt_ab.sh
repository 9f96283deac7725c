#!/bin/bash
cd "$(dirname "$0")/../.." || exit 1
mkdir -p gpurun_out
O=gpurun_out/bptt_ab.log
: > $O
run() { echo "== $*" >> $O; timeout 300 env "$@" >> $O 2>&1; echo "rc=$?" >> $O; }
for B in ${BS:-96 128 256}; do
run AVVAD_BPTT_CHUNKS=1 python tools/micro/bptt_ab.py $B 317 --save /tmp/g$B.pt
run AVVAD_BPTT_CHUNKS=8 python tools/micro/bptt_ab.py $B 317 --cmp /tmp/g$B.pt
done
grep -v "^rc=0" $O

#!/bin/bash
# The drop-in's host pipeline (video-encoder_b200/host/*.c: caller's thread + staging-copy helpers, one thread per GPU, entropy workers, fifo)
# under ThreadSanitizer, CPU only: scripts/host_ceiling.c linked with the mock engine (tests/mock/mock_engine.c) in one TSan executable,
# (1) against the zero-latency engine (B2_MOCK_CANNED, made by scripts/host_ceiling.py) at 1080p on 2 pretend GPUs -- the high-rate paths --
# (2) against the oracle-backed engine at 160x96 on 3 pretend GPUs -- polling / wait paths -- and (3) with 4 slices per picture, in
# zero-delay mode (one GOP slot: the slice pool writes the slices of a picture at the same time) and with 2 GOP slots.
# usage: scripts/host_tsan.sh [workdir]
set -e
ROOT=$(cd "$(dirname "$0")/.." && pwd)
WORK=${1:-$(mktemp -d /tmp/b2_tsan_XXXX)}
B2_CEILING_CONTENT=static B2_CEILING_DIR=$WORK python "$ROOT/scripts/host_ceiling.py" 1920 1080 64 > /dev/null
gcc -O1 -g -fsanitize=thread -std=gnu99 -I"$ROOT/include" -I"$ROOT/video-encoder_b200/host" -o "$WORK/ceil_tsan" "$ROOT/scripts/host_ceiling.c" \
    "$ROOT/tests/mock/mock_engine.c" "$ROOT"/video-encoder_b200/host/*.c "$ROOT"/oracle/b2o_*.c -lm -lpthread
B2ENC_STATS=1 B2_MOCK_DEVICES=2 B2_MOCK_CANNED=$WORK/canned_1920x1080_static "$WORK/ceil_tsan" 1920 1080 600 2 6 2>&1 | grep -v "^b2enc stats" | tee "$WORK/tsan1.log"
B2_MOCK_DEVICES=3 "$WORK/ceil_tsan" 160 96 60 3 2 2>&1 | tee "$WORK/tsan2.log"
B2ENC_SLICES=4 B2_MOCK_DEVICES=1 "$WORK/ceil_tsan" 160 96 40 1 1 2>&1 | tee "$WORK/tsan3.log"
B2ENC_SLICES=4 B2_MOCK_DEVICES=2 "$WORK/ceil_tsan" 160 96 40 2 2 2>&1 | tee -a "$WORK/tsan3.log"
if grep -q "ThreadSanitizer" "$WORK/tsan1.log" "$WORK/tsan2.log" "$WORK/tsan3.log"; then echo "ThreadSanitizer reported findings"; exit 1; fi
echo "host pipeline: no ThreadSanitizer finding"

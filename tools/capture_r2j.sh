#!/usr/bin/env bash
set -u
T=${1:-r2j}
mkdir -p gpurun_out
step() { echo "== $1" >&2; }
step "decode probe: stats late (default) vs early"
python tools/probe_decode_tail.py 2>/dev/null | grep "^{" | sed 's/^{/{"stats": "late", /' | tee gpurun_out/${T}_decode_probe.jsonl
TWB200_LIB=$PWD/turbo-whisper-workspace_b200/variants/libtwb200_lnearly.so python tools/probe_decode_tail.py 2>/dev/null | grep "^{" | sed 's/^{/{"stats": "early", /' | tee -a gpurun_out/${T}_decode_probe.jsonl

#!/usr/bin/env bash
set -u
T=${1:-r2l}
mkdir -p gpurun_out
echo "== parity (engine + bench shapes)" >&2
timeout 900 python -m pytest tests/test_gpu_bench_shapes.py tests/test_gpu_engine.py tests/test_gpu_fullsize.py -m gpu -x -q > gpurun_out/${T}_tests.log 2>&1; tail -3 gpurun_out/${T}_tests.log
echo "== LN fold A/B" >&2
for rep in 1 2; do
  for mode in fold nofold; do
    if [ $mode = nofold ]; then export TWB200_NO_LN_FOLD=1; else unset TWB200_NO_LN_FOLD; fi
    python tools/probe_decode_tail.py 2>/dev/null | grep "^{" | sed "s/^{/{\"ln\": \"$mode\", /" | tee -a gpurun_out/${T}_decode_probe.jsonl
    timeout 600 python bench.py --steps 8 --warmup 3 --no-extras --no-cpu-baseline 2>/dev/null | python -c "
import json,sys
d=json.loads(sys.stdin.readline())
print(json.dumps({'ln':'$mode','value':round(d['value'],1),'e2e':round(d['e2e']['value'],1),'ms_per_step':round(d['ms_per_step'],1),'decode_alone_us':round(d['decode_step']['us'],1),'in_bench_us':round(d['decode_step']['in_bench_us'],1),'enc_ms':round(d['encoder']['ms'],2),'ok':d['output_check']['e2e_rows_equal_single_context']}))" | tee -a gpurun_out/${T}_bench_ab.jsonl
  done
done
unset TWB200_NO_LN_FOLD

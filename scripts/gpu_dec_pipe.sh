#!/bin/bash
# GPU runs of the MT3_DEC_PIPE study (decode.cuh dec_cluster_body).  Everything lands in $OUT (default: a directory under
# $TMPDIR or /tmp, so the tree stays untouched).
#   scripts/gpu_dec_pipe.sh study   the bit-identity tests, an in-process A/B of every bit combination (scripts/ab_prefetch.py:
#                                   same batch, tokens compared with the first setting), and the decode-step timeline at cache
#                                   position 512 with the pipeline off and on
#   scripts/gpu_dec_pipe.sh final   bench.py alternately with MT3_DEC_PIPE=0 and the default (3 each; the first pair also dumps
#                                   its tokens, which must be identical), smoke() and the whole -m gpu suite
set -u
OUT=${OUT:-${TMPDIR:-/tmp}/mt3_dec_pipe}
mkdir -p "$OUT"
echo "results in $OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.sm,clocks.max.sm --format=csv | tee $OUT/gpu.txt
if [ "${1:-study}" = "study" ]; then
  echo "== pytest tests/test_gpu_dec_pipeline.py"
  timeout 900 python -m pytest tests/test_gpu_dec_pipeline.py -q -m gpu 2>&1 | tail -15 | tee $OUT/pytest_dec_pipeline.log
  echo "== A/B"
  timeout 600 python scripts/ab_prefetch.py --reps 3 \
    --settings "pipe0:MT3_DEC_PIPE=0;pipe1:MT3_DEC_PIPE=1;pipe2:MT3_DEC_PIPE=2;pipe3:MT3_DEC_PIPE=3;pipe0b:MT3_DEC_PIPE=0;pipe3b:MT3_DEC_PIPE=3;pipe1b:MT3_DEC_PIPE=1;pipe2b:MT3_DEC_PIPE=2" \
    > $OUT/ab_dec_pipe.txt 2> $OUT/ab_dec_pipe.err; tail -10 $OUT/ab_dec_pipe.txt; tail -3 $OUT/ab_dec_pipe.err
  for p in 0 3; do
    echo "== decode-step timeline, MT3_DEC_PIPE=$p"
    MT3_DEC_PIPE=$p TRACE_POS=512 TRACE_ROWS=12 timeout 300 python scripts/trace_step.py > $OUT/trace_step_pipe$p.log 2>&1
    tail -13 $OUT/trace_step_pipe$p.log
  done
  exit 0
fi
for i in 1 2 3; do
  for p in 0 default; do
    dump=(); [ "$i" = 1 ] && dump=(--dump-outputs $OUT/dump_$p)
    if [ "$p" = 0 ]; then envs=(MT3_DEC_PIPE=0); else envs=(-u MT3_DEC_PIPE); fi
    timeout 600 env "${envs[@]}" python bench.py --gpus 1 --steps 5 --warmup 3 --no-cpu-baseline --no-alt-kv "${dump[@]}" \
      2> $OUT/bench_pipe${p}_$i.err | tail -1 > $OUT/bench_pipe${p}_$i.json
    python -c "import json,sys; d=json.load(open(sys.argv[1])); print('bench MT3_DEC_PIPE=%-8s run %s: ms_per_step %.2f  value %.1f  clocks %s' % (sys.argv[2], sys.argv[3], d['ms_per_step'], d['value'], d.get('clocks')))" \
      $OUT/bench_pipe${p}_$i.json $p $i || tail -5 $OUT/bench_pipe${p}_$i.err
  done
done
python -c "import numpy as np; a=np.load('$OUT/dump_0/tokens.npy'); b=np.load('$OUT/dump_default/tokens.npy'); print('dump tokens', a.shape, 'identical:', bool(np.array_equal(a, b)))"
echo "== smoke"; timeout 300 python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -3 | tee $OUT/smoke.log
echo "== pytest -m gpu"; timeout 1500 python -m pytest tests -q -m gpu 2>&1 | tail -8 | tee $OUT/pytest_gpu.log

#!/bin/bash
# usage: aireml.sh <output dir> [suite]
# AI-REML: the new GPU tests (the 2-rank fit also over gloo with both ranks on one GPU), smoke(), the 250K AI-REML vs L-BFGS-B measurement and a short bench; `aireml.sh <output dir> suite`: the 250K measurement and the whole -m gpu suite
OUT=$1; shift
mkdir -p "$OUT"
if [ "$1" = suite ]; then
  python -c "import __graft_entry__ as g; g.build()" > /dev/null 2>&1
  (timeout 300 python scripts/aireml_fit.py --out $OUT/aireml_fit.json > $OUT/aireml_fit.log 2>&1; echo "rc=$?" >> $OUT/aireml_fit.log)
  grep -a "card\|fit\|rc=" $OUT/aireml_fit.log | cut -c1-400
  (timeout 840 python -m pytest tests -m gpu -q > $OUT/aireml_gpu_suite.log 2>&1; echo "rc=$?" >> $OUT/aireml_gpu_suite.log)
  tail -5 $OUT/aireml_gpu_suite.log
  exit 0
fi
python -c "import __graft_entry__ as g; g.build()" > $OUT/aireml_build.log 2>&1 || { tail -20 $OUT/aireml_build.log; exit 1; }
(timeout 420 python -m pytest tests/test_gpu_aireml.py -m gpu -q -rs > $OUT/aireml_tests.log 2>&1; echo "rc=$?" >> $OUT/aireml_tests.log)
tail -4 $OUT/aireml_tests.log
(SLMM_TWO_RANK_BACKEND=gloo timeout 240 python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 \
   --master-port 29574 tests/nccl_two_rank_aireml.py > $OUT/aireml_two_rank_gloo.log 2>&1; echo "rc=$?" >> $OUT/aireml_two_rank_gloo.log)
grep -a "TWO_RANK_AIREML_OK\|rc=\|Error" $OUT/aireml_two_rank_gloo.log | tail -4
(timeout 420 python scripts/aireml_fit.py --out $OUT/aireml_fit.json > $OUT/aireml_fit.log 2>&1; echo "rc=$?" >> $OUT/aireml_fit.log)
grep -a "card\|fit:\|rc=" $OUT/aireml_fit.log
python -c "import __graft_entry__ as g; g.smoke()" > $OUT/aireml_smoke.log 2>&1; echo "smoke rc=$?"; tail -1 $OUT/aireml_smoke.log
(timeout 300 python bench.py --gpus 1 --steps 5 --warmup 3 --skip-fit --skip-he --skip-cpu > $OUT/aireml_bench.json 2> $OUT/aireml_bench.err; echo "bench rc=$?" >> $OUT/aireml_bench.err)
tail -1 $OUT/aireml_bench.err

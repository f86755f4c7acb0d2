#!/bin/bash
# VGG / AlexNet lowering, closing call: the VGG GPU tests with the measured band and the fp32-grade fc6 rule, the existing
# x3 / split whole-network tests, smoke(), and the VGG-16 bench line with the default tie policy.
OUT=$(realpath -m "${OUT:-vgg_out}")   # output directory (default ./vgg_out)
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > $OUT/card_final.txt 2>&1; cat $OUT/card_final.txt
python -c "import __graft_entry__ as g; g.build()" > $OUT/build_final.log 2>&1; echo "build rc=$?"
timeout 1500 python -m pytest tests/test_gpu_vgg.py tests/test_gpu_classifier.py -q -k "vgg or x3_mode or split_mode or Linear or raw_row or linear or whole_network or bench_config or dropin" -s > $OUT/pytest_vgg_final.log 2>&1; echo "pytest rc=$?"; grep -E "passed|failed|FAILED|\] |rel err" $OUT/pytest_vgg_final.log | tail -25
timeout 600 python -c "import __graft_entry__ as g; g.smoke()" > $OUT/smoke_final.log 2>&1; echo "smoke rc=$?"; tail -1 $OUT/smoke_final.log
timeout 900 python bench.py --gpus 1 --arch vgg16 --steps 5 --warmup 2 --no-cpu-baseline --no-gp > $OUT/bench_vgg16_default_final.log 2>&1; echo "bench vgg16 rc=$?"; tail -1 $OUT/bench_vgg16_default_final.log | cut -c1-300

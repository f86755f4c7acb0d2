#!/bin/bash
# VGG / AlexNet lowering: the whole VGG GPU test file after pinning the measured fp32-grade band.
OUT=$(realpath -m "${OUT:-vgg_out}")   # output directory (default ./vgg_out)
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit --format=csv > $OUT/card_pin.txt 2>&1; cat $OUT/card_pin.txt
python -c "import __graft_entry__ as g; g.build()" > $OUT/build_pin.log 2>&1; echo "build rc=$?"
timeout 1500 python -m pytest tests/test_gpu_vgg.py -q -s > $OUT/pytest_vgg_pin.log 2>&1; echo "pytest rc=$?"; grep -E "passed|failed|FAILED|\] " $OUT/pytest_vgg_pin.log | tail -30

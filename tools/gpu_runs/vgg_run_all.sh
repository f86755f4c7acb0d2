#!/bin/bash
# VGG / AlexNet lowering, one call: the kernel checks first (raw-row 3x3, Linear-as-conv), the flip studies the tie band
# rests on, the probe (bf16 error per network, mask synthesis into the 8-channel buffer, conv1_1, peak memory at
# tie_capacity=1024), the VGG-16 bench lines with and without the tie policy (+ per-layer profile), the whole GPU suite,
# smoke(), and ResNet-101 bench lines of this tree and of its parent (exported to build/parent_tree) alternated on one box.
OUT=$(realpath -m "${OUT:-vgg_out}")   # output directory (default ./vgg_out)
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > $OUT/card.txt 2>&1; cat $OUT/card.txt
python -c "import __graft_entry__ as g; g.build()" > $OUT/build.log 2>&1; echo "build rc=$?"
timeout 900 python -m pytest tests/test_gpu_vgg.py -q -x -k "raw_row or linear_as_conv" > $OUT/pytest_kernels.log 2>&1; echo "kernels rc=$?"; tail -3 $OUT/pytest_kernels.log
for a in vgg16 vgg16_bn; do
  timeout 900 python tools/r02_diag2.py 16384 $a > $OUT/flip_$a.log 2>&1; echo "flip $a rc=$?"
done
timeout 900 python tools/vgg_probe.py $OUT/vgg_probe.json > $OUT/vgg_probe.log 2>&1; echo "probe rc=$?"; tail -6 $OUT/vgg_probe.log
timeout 900 python bench.py --gpus 1 --arch vgg16 --steps 5 --warmup 2 --no-cpu-baseline --no-gp --refine-ties 0 --profile-json $OUT/vgg16_profile_mb384.json > $OUT/bench_vgg16_noties.log 2>&1; echo "bench vgg16 no ties rc=$?"; tail -1 $OUT/bench_vgg16_noties.log | cut -c1-300
timeout 900 python bench.py --gpus 1 --arch vgg16 --steps 5 --warmup 2 --no-cpu-baseline --no-gp > $OUT/bench_vgg16_default.log 2>&1; echo "bench vgg16 rc=$?"; tail -1 $OUT/bench_vgg16_default.log | cut -c1-300
timeout 2400 python -m pytest tests -q -m gpu > $OUT/pytest_gpu_all.log 2>&1; echo "pytest gpu rc=$?"; grep -E "passed|failed|FAILED|Error" $OUT/pytest_gpu_all.log | tail -12
timeout 600 python -c "import __graft_entry__ as g; g.smoke()" > $OUT/smoke.log 2>&1; echo "smoke rc=$?"; tail -2 $OUT/smoke.log
(cd build/parent_tree && python -c "from network_interpretation_imagenet_b200 import build; build.build()" > $OUT/build_parent.log 2>&1); echo "parent build rc=$?"
RB="bench.py --gpus 1 --steps 5 --warmup 3 --no-cpu-baseline --no-gp --no-library-bar"
for i in 1 2; do
  timeout 600 python $RB > $OUT/bench_resnet_new_$i.log 2>&1; echo "new $i rc=$?"
  (cd build/parent_tree && timeout 600 python $RB > $OUT/bench_resnet_parent_$i.log 2>&1); echo "parent $i rc=$?"
done
for f in $OUT/bench_resnet_*.log; do python -c "import json,sys;d=json.loads(open('$f').read().strip().splitlines()[-1]);print('$f',d['value'],d['e2e']['value'])"; done

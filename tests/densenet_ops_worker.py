"""Child process of test_preact_transform_matches_pack_pass_bitwise: runs the Cout 128 / 256 pre-activated 1x1 cases of
test_gpu_densenet_ops.py under whatever NIB_* environment it was started with (the engine reads NIB_TC_NO_XFORM once per
process) and saves {case id: (output, total launches, tcgen05 launches)} with torch.save to argv[1]."""
import os
import sys

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)
import test_gpu_densenet_ops as t  # noqa: E402

torch.save(t.preact_outputs_for_ab(), sys.argv[1])

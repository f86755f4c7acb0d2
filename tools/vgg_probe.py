"""VGG-16 / AlexNet measurements on the GPU that bench.py does not take: the bf16 row-wise logit error of every lowered
torchvision plain CNN against the torch fp32 CPU forward, the time of mask synthesis into the 8-channel haloed bf16
input buffer (against the 4-channel 128-bit path ResNet uses), the time and HBM rate of VGG-16's conv1_1 on the tcgen05
raw-row path, and the peak device allocation of the bench configuration with the tie policy at tie_capacity=1024.
Writes the JSON to the path given as the first argument (default ./vgg_probe.json)."""
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import network_interpretation_imagenet_b200 as nib  # noqa: E402
from network_interpretation_imagenet_b200 import synthetic  # noqa: E402
from network_interpretation_imagenet_b200.classifier import Classifier  # noqa: E402
from network_interpretation_imagenet_b200.masks import MaskSynth  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip()


def timed(fn, reps):
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else "vgg_probe.json"
    res = {"card": card()}
    x0 = synthetic.synthetic_image("imagenet")
    seg = synthetic.voronoi_labels(224, 224, 50)

    # bf16 logit error of each network (4 inputs: the image, a flipped / scaled copy, two random keep-masks)
    g = torch.Generator().manual_seed(3)
    xb = torch.from_numpy(x0)[None].repeat(4, 1, 1, 1)
    xb[1] = xb[1].flip(2) * 0.5
    xb[2:] = xb[2:] * (torch.rand(2, 1, 224, 224, generator=g) > 0.5).float()
    errs = {}
    for arch in ("vgg11", "vgg16", "vgg16_bn", "vgg19_bn", "alexnet"):
        m = synthetic.build_imagenet_model(arch)
        with torch.no_grad():
            want = m(xb).double()
        got = Classifier.from_torch(m, (224, 224), precision="bf16", max_batch=4).forward(xb.cuda()).cpu().double()
        errs[arch] = float(((got - want).abs() / want.abs().amax(1, keepdim=True)).max())
        print(arch, "bf16 row-wise err", errs[arch], flush=True)
    res["bf16_rowwise_logit_err"] = errs

    # mask synthesis: 384 keep-masks into the 8-channel, 1-pixel-halo buffer vs the 4-channel dense one
    synth = MaskSynth(x0, seg, S=50, device="cuda")
    sels = nib.draw_selections("subset_keep", 50, 384, seed=1)
    bits = torch.from_numpy(nib.selection_bits(sels, 50).view(np.int64)).cuda()
    o8 = torch.empty(384, 226, 226, 8, dtype=torch.bfloat16, device="cuda")
    o4 = torch.empty(384, 224, 224, 4, dtype=torch.bfloat16, device="cuda")
    ms8 = timed(lambda: synth.synth(bits, nib.KEEP_MUL, dtype=torch.bfloat16, layout="nhwc", c_stride=8, pad=1, out=o8), 20)
    ms4 = timed(lambda: synth.synth(bits, nib.KEEP_MUL, dtype=torch.bfloat16, layout="nhwc", c_stride=4, pad=0, out=o4), 20)
    res["mask_synth_384"] = {"c8_halo1_ms": ms8, "c8_halo1_write_GBps": o8.numel() * 2 / ms8 / 1e6,
                             "c4_dense_ms": ms4, "c4_dense_write_GBps": o4.numel() * 2 / ms4 / 1e6}
    print(res["mask_synth_384"], flush=True)
    del o8, o4

    # conv1_1 of VGG-16 at micro-batch 384 (profile of the lowered network, op 0), against HBM bytes
    m16 = synthetic.build_imagenet_model("vgg16")
    clf = Classifier.from_torch(m16, (224, 224), precision="bf16", max_batch=384)
    clf.forward_masked(synth, bits, nib.KEEP_MUL)
    profs = sorted((clf.profile(384) for _ in range(5)), key=lambda pr: pr[0][0])
    p0 = profs[2][0]
    byts = 384 * (226 * 226 * 8 + 224 * 224 * 64) * 2
    res["conv1_1_384"] = {"ms": p0[0], "kind": ["simt_conv", "tc_conv"][p0[1]], "gflop": p0[2] / 1e9,
                          "tflops": p0[2] / (p0[0] / 1e3) / 1e12, "bytes": byts, "GBps": byts / p0[0] / 1e6}
    print(res["conv1_1_384"], flush=True)
    del clf
    torch.cuda.synchronize()
    torch.cuda.empty_cache()

    # peak device memory of the bench configuration with the tie policy at tie_capacity=1024 (lowering + 2 steps)
    torch.cuda.reset_peak_memory_stats()
    free0, total = torch.cuda.mem_get_info()
    eng = nib.PerturbationEngine(m16, x0, seg, target=0, mode=nib.KEEP_MUL, precision="bf16", max_batch=384, S=50,
                                 streams=2, tie_capacity=1024)
    sels = nib.draw_selections("subset_keep", 50, 16384, seed=1)
    b16 = nib.selection_bits(sels, 50)
    eng._tie_state(eng.tie_window)           # the re-score lowering at its full capacity
    for _ in range(2):
        eng.score_masks(b16)
    torch.cuda.synchronize()
    free1, _ = torch.cuda.mem_get_info()
    res["bench_config_memory"] = {"tie_capacity": eng.tie_capacity, "tie_precision": eng.tie_precision,
                                  "band": eng.refine_ties, "device_used_GB": (total - free1) / 1e9,
                                  "used_before_GB": (total - free0) / 1e9, "torch_peak_GB": torch.cuda.max_memory_allocated() / 1e9,
                                  "tie_stats": eng.tie_stats()}
    print(res["bench_config_memory"], flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
    with open(out_path, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()

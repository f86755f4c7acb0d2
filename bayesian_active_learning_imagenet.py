"""Drop-in for the reference's bayesian_active_learning_imagenet.py.

    python bayesian_active_learning_imagenet.py -a resnet101 DIR [--eval_img_index I]

The reference runs Bayesian optimisation over `firstIndex`, the start of a 40 %-of-S superpixel window: the
objective `sample_loss(params, val_loader, model, criterion)` (:278-298) masks the image with that window, runs a
batch-1 forward and returns the softmax probability of the true class (:178-198) — after re-scanning the DataLoader
and re-running felzenszwalb on every evaluation (:126-150).  Here the image and label map stay on the device, one
evaluation is one mask-synthesis + forward + score launch sequence, and the GP / EI run in libnib.so.

After the search, `plot_summed_heatmap(val_img_index, bbox_threshold, gt_bbox)` (:312-377, called at :492 with
bbox_threshold = 180) sums the labels of the evaluated masks into a heat map, boxes its strongest region and reports the
IOU with the ground-truth box - heat map, 8-bit view and bounding box are device kernels here (localize.py).

`--masks` switches to the scaled-up form of BASELINE.json config 4: the GP input is the mask itself, n training
masks, `--rounds` acquisition rounds over m candidate masks scored by EI on the device.  `--acq-batch Q` (default 1)
evaluates Q masks per round: Kriging-believer picks on the device, scored in one batched forward (Q * `--rounds` masks in
all; `-b/--batch-size` stays the forward's micro-batch)."""
from __future__ import annotations

import argparse
import os
import time

import numpy as np
import torch
import torchvision.models as models

from BayesianOptimization import bayesian_optimisation, bayesian_optimisation_masks
from network_interpretation_imagenet_b200 import synthetic
from network_interpretation_imagenet_b200.engine import PerturbationEngine
from network_interpretation_imagenet_b200.masks import KEEP_MUL, draw_selections, selection_bits, window_at
from network_interpretation_imagenet_b200.pipeline import segment_image

model_names = sorted(name for name in models.__dict__
                     if name.islower() and not name.startswith("__") and callable(models.__dict__[name]))

parser = argparse.ArgumentParser(description="Bayesian active learning over superpixel masks (B200 engine)")
parser.add_argument("data", metavar="DIR", nargs="?", default=None)
parser.add_argument("--arch", "-a", metavar="ARCH", default="resnet18", choices=model_names)
parser.add_argument("-b", "--batch-size", default=256, type=int)
parser.add_argument("--eval_img_index", default=1600, type=int)
parser.add_argument("--synthetic", action="store_true")
parser.add_argument("--image", default=None)
parser.add_argument("--weights", default=None)
parser.add_argument("--target", default=None, type=int)
parser.add_argument("--precision", default="bf16", choices=["bf16", "fp32"])
parser.add_argument("--n_iters", default=10, type=int)
parser.add_argument("--n_pre_samples", default=3, type=int)
parser.add_argument("--masks", action="store_true", help="mask-space GP (BASELINE config 4)")
parser.add_argument("--n-train", default=8192, type=int)
parser.add_argument("--n-candidates", default=8192, type=int)
parser.add_argument("--rounds", default=20, type=int)
parser.add_argument("--acq-batch", default=1, type=int, help="masks acquired per round with --masks (Kriging believer)")
parser.add_argument("--mask-seed", default=0, type=int)
parser.add_argument("--gt-bbox", default=None, type=int, nargs=4, metavar=("X", "Y", "W", "H"),
                    help="ground-truth box of the image (the reference reads it from the ImageNet annotation, :454)")

_ENGINE = {}
_EVALS = {"bits": [], "labels": []}        # the masks this run evaluated and their 0/1 labels (the reference's ./masks PNGs)


def validate_nueral_network(val_loader, model, criterion, bo_iter, firstIndex):
    """Reference :116-221: target-class softmax probability of the image masked with the window at firstIndex."""
    eng = _ENGINE["engine"]
    sel = window_at(eng.synth.S, int(firstIndex))
    bits = selection_bits([sel], eng.synth.S)
    out = eng.score_masks(bits)
    label = int(out["correct"][0].item())                      # :199-213: 1 iff the masked image keeps its top-1
    _EVALS["bits"].append(bits[0])
    _EVALS["labels"].append(label)
    writer = _ENGINE.get("writer")
    if writer is not None:                                       # ./masks/mask_{bo_iter}_{label}.png, ./mask_on_img/... (:207-216)
        _, pm = eng.synth.synth(bits, eng.mode, return_pixel_masks=True)
        writer.submit("./masks", ["mask_{}_{}.png".format(bo_iter, label)], pm, scale=255)
        writer.submit("./mask_on_img", ["masked_imgs_{}_{}.png".format(bo_iter, label)], eng.synth.display_u8(bits, eng.mode))
    return float(out["target_prob"][0].item())


def sample_loss(params, val_loader, model, criterion):
    """Reference :278-298 (same signature; val_loader/criterion are unused, as the loss term is commented out there)."""
    firstIndex = int(params[0])
    print("firstIndex: ", firstIndex)
    return validate_nueral_network(val_loader, model, criterion, params[0], firstIndex)


def plot_summed_heatmap(val_img_index, bbox_threshold, gt_bbox):
    """Reference :312-377.  Heat map of the evaluated masks (sum of their 0/1 labels per pixel), its uint8 view, the box of
    the strongest region above `bbox_threshold` and the IOU with `gt_bbox` = [x, y, w, h].  The reference's
    generate_boundingbox returns [x, y, x, y] (utils.py:109); that quirk is reproduced, and the IOU of the real box is
    printed next to it."""
    import cv2
    from network_interpretation_imagenet_b200 import localize as loc
    eng = _ENGINE["engine"]
    bits = np.stack(_EVALS["bits"])
    labels = np.asarray(_EVALS["labels"], dtype=np.float32)
    print("%d samples, the correct prediction number: %d " % (len(labels), int(labels.sum())))
    heat = eng.synth.heatmap(bits, labels)
    IOU, pred_box, gray = loc.summed_heatmap_iou(heat, bbox_threshold, list(gt_bbox), quirk=True)
    IOU_box, real_box, _ = loc.summed_heatmap_iou(heat, bbox_threshold, list(gt_bbox), quirk=False)
    os.makedirs("heatmaps", exist_ok=True)
    cv2.imwrite("heatmaps/index_{}.png".format(val_img_index), cv2.applyColorMap(gray.cpu().numpy(), cv2.COLORMAP_JET))
    cv2.imwrite("heatmaps/gray_img_{}.png".format(val_img_index), gray.cpu().numpy())
    print('\033[91m' + "IOU: " + str(IOU) + '\033[0m')
    print("IOU with the real predicted box {}: {}".format(real_box, IOU_box))
    return IOU


def main():
    args = parser.parse_args()
    start_time = time.time()
    if args.weights:
        model = models.__dict__[args.arch](weights=None)
        model.load_state_dict(torch.load(args.weights, map_location="cpu"))
        model.eval()
    else:
        model = synthetic.build_imagenet_model(args.arch)
    if args.image:
        from generate_gp_training_data_imagenet import load_image
        image = load_image(args)
    else:
        image = synthetic.synthetic_image("imagenet")
    disp = image.transpose(1, 2, 0).copy()
    disp -= disp.min(); disp /= disp.max(); disp *= 255
    segments = segment_image(disp.astype(np.uint8), 50, 50)
    S = len(np.unique(segments))
    print("Felzenszwalb number of segments: {}".format(S))
    eng = PerturbationEngine(model, image, segments, target=0, mode=KEEP_MUL, precision=args.precision,
                             max_batch=args.batch_size, S=S)
    logits = eng.classifier.forward(torch.from_numpy(image)[None].cuda())
    eng.target = int(logits.argmax(1)[0]) if args.target is None else args.target
    _ENGINE["engine"] = eng
    if not args.masks:
        from network_interpretation_imagenet_b200.pipeline import AsyncPngWriter, reset_dir
        reset_dir("./masks")                                     # :469-474
        os.makedirs("./mask_on_img", exist_ok=True)
        _ENGINE["writer"] = AsyncPngWriter()
        firstIndex_upperbound = int(0.6 * S)                     # :467
        bounds = np.asarray([[0, firstIndex_upperbound]])
        xp, yp = bayesian_optimisation(n_iters=args.n_iters, sample_loss=sample_loss, val_loader=None, nn_model=model,
                                       criterion=None, bounds=bounds, n_pre_samples=args.n_pre_samples,
                                       random_search=False)      # :479-486
        print("xp", xp.ravel()); print("yp", yp)
        _ENGINE["writer"].close()
        bbox_threshold = 180                                     # :491
        gt = args.gt_bbox if args.gt_bbox is not None else [0, 0, image.shape[2], image.shape[1]]
        plot_summed_heatmap(args.eval_img_index, bbox_threshold, gt)
    else:
        sels = draw_selections("subset_keep", S, args.n_train + args.n_candidates, seed=args.mask_seed)
        bits = selection_bits(sels, S)
        train, cand = bits[:args.n_train], bits[args.n_train:]
        y = eng.score_masks(train)["target_prob"].cpu().numpy()
        Z, yy, hist = bayesian_optimisation_masks(args.rounds, lambda b: eng.score_masks(b)["target_prob"].cpu().numpy(),
                                                  train, y, cand, length_scale=3.0, batch_size=args.acq_batch)
        for h in hist:
            print(h)
    print("time duration is: ", time.time() - start_time)


if __name__ == "__main__":
    main()

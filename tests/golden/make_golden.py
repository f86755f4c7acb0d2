"""Generates tests/golden/*.npz by EXECUTING THE REFERENCE'S OWN CODE from a checkout of it.

Run once with that checkout (`python tests/golden/make_golden.py <reference checkout>`); the tests only ever read
the committed .npz files.  Nothing from the reference is copied into the repo: the hot
loops cannot be imported on Python 3.12 (`async=True` SyntaxError, argparse/downloads at import time), so the
loop-body statements are located in the reference files by content, dedented and exec'd in a namespace that
supplies the loop's free variables (`segments`, `org_img`, `input`, ...) — i.e. the fixtures are outputs of
the reference's statements, not of our restatement.  The located line numbers are stored in each fixture.

Fixtures
  masks_imagenet.npz   generate_gp_training_data_imagenet.py  selection draw + mask build + multiply
  masks_cifar.npz      generate_gp_training_data_cifar.py     a1 prep, draw, mask, min-max renormalise
  masks_mnist.npz      generate_gp_training_data_mnist.py     a1 prep, dummy randint + draw, mask, renormalise
  resnet56.npz         models/resnet.py createModel + shipped checkpoint -> logits of a seeded batch
  mnist_net.npz        generate_gp_training_data_mnist.py :72-105 class statements + shipped checkpoint -> 4-tuple
  utils.npz            utils.normalize_image / utils.generate_IOU executed on seeded inputs
  ei.npz               BayesianOptimization.expected_improvement on fixed (mu, sigma)
  gp_sklearn.npz       scikit-learn 1.9.0 GaussianProcessRegressor as built at BayesianOptimization.py:154-159
  localize.npz         generate_gp_training_data_imagenet.py get_pixel_sorted_mask_label / generate_new_mask / heat-map uint8
"""
from __future__ import annotations

import contextlib
import importlib.util
import io
import os
import random
import sys

import numpy as np
import torch

REF = None   # the reference checkout, from the command line
OUT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(OUT)))

from oracle import synthetic  # noqa: E402  (synthetic inputs only; no oracle arithmetic is used below)


def _load_ref_module(name, relpath):
    spec = importlib.util.spec_from_file_location(name, os.path.join(REF, relpath))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def _extract(relpath, start_marker, end_marker, after=None):
    """Source lines [first line containing start_marker .. first later line containing end_marker]."""
    lines = open(os.path.join(REF, relpath)).read().split("\n")
    i0 = 0
    if after is not None:
        i0 = next(i for i, l in enumerate(lines) if after in l)
    s = next(i for i in range(i0, len(lines)) if start_marker in lines[i])
    e = next(i for i in range(s, len(lines)) if end_marker in lines[i])
    ind = len(lines[s]) - len(lines[s].lstrip())
    body = []
    for l in lines[s:e + 1]:
        if len(l) - len(l.lstrip()) >= ind:
            body.append(l[ind:])
        else:  # blank / comment lines in the reference are indented inconsistently
            assert l.strip() == "" or l.strip().startswith("#"), l
            body.append(l.strip())
    return "\n".join(body), (s + 1, e + 1)


def _run(code, ns):
    with contextlib.redirect_stdout(io.StringIO()):
        exec(compile(code, "<reference>", "exec"), ns)
    return ns


class _FakeInput:
    """Stands in for the torch batch `input` of imagenet :240 (`input[0].numpy().copy()`)."""

    def __init__(self, arr):
        self._t = torch.from_numpy(arr)[None]

    def __getitem__(self, i):
        return self._t[i]


def make_masks_imagenet():
    rel = "generate_gp_training_data_imagenet.py"
    code, span = _extract(rel, "total_num_segments = len(np.unique(segments))", "masked_img = input[0].numpy().copy() * mask",
                          after="def validate(")
    g = torch.Generator().manual_seed(11)
    x = ((torch.rand(3, 24, 32, generator=g) - 0.45) / 0.25).numpy().astype(np.float32)
    segments = synthetic.voronoi_labels(24, 32, 13, seed=3)
    random.seed(2024)
    sels, masks, outs = [], [], []
    for _ in range(8):
        ns = dict(np=np, segments=segments, randint=random.randint, sample=random.sample,
                  img_show=np.zeros((24, 32, 3), np.uint8), input=_FakeInput(x))
        _run(code, ns)
        sels.append(np.array(ns["random_sampled_list"], dtype=np.int64))
        masks.append(ns["mask"].copy())
        outs.append(ns["masked_img"].copy())
    np.savez_compressed(os.path.join(OUT, "masks_imagenet.npz"), x=x, segments=segments, seed=2024,
                        sel=np.stack(sels), mask=np.stack(masks), out=np.stack(outs), ref_lines=np.array(span))


def _make_masks_remove(rel, kind, shape, S, seed, n_masks, prep_markers, loop_markers, after, fname):
    prep_code, span1 = _extract(rel, *prep_markers, after=after)
    loop_code, span2 = _extract(rel, *loop_markers, after=after)
    utils = _load_ref_module("ref_utils", "utils.py")
    g = torch.Generator().manual_seed(seed)
    C, H, W = shape
    raw = torch.rand(C, H, W, generator=g).numpy().astype(np.float32)
    if kind == "cifar":
        raw = (raw - 0.5) / 0.5
    org_img = raw.copy()
    ns = dict(np=np, org_img=org_img)
    _run(prep_code, ns)          # mutates org_img in place through the transpose view
    img_u8 = ns["img"]
    segments = synthetic.voronoi_labels(H, W, S, seed=5)
    random.seed(777)
    sels, masks, outs = [], [], []
    import cv2
    for _ in range(n_masks):
        ns = dict(np=np, random=random, randint=random.randint, sample=random.sample, segments=segments,
                  img=img_u8, org_img=org_img, normalize_image=utils.normalize_image, cv2=cv2)
        with np.errstate(all="ignore"):
            _run(loop_code, ns)
        sels.append(np.array(ns["random_sampled_list"], dtype=np.int64))
        masks.append(ns["mask"].copy())
        outs.append(ns["masked_img"].copy())
    np.savez_compressed(os.path.join(OUT, fname), raw=raw, org=org_img, img_u8=img_u8, segments=segments, seed=777,
                        sel=np.stack(sels), mask=np.stack(masks), out=np.stack(outs),
                        ref_lines=np.array(span1 + span2))


def make_masks_cifar():
    _make_masks_remove("generate_gp_training_data_cifar.py", "cifar", (3, 32, 32), 14, 21, 8,
                       ("img = org_img.transpose( 1, 2, 0 )", "img = img.astype(np.uint8)"),
                       ("random_sampled_list= random.sample(range(np.unique(segments)[0]", "masked_img = normalize_image(masked_img)"),
                       "def eval_superpixel(", "masks_cifar.npz")


def make_masks_mnist():
    _make_masks_remove("generate_gp_training_data_mnist.py", "mnist", (1, 28, 28), 9, 22, 8,
                       ("img = org_img.transpose( 1, 2, 0 )", "img = img.astype(np.uint8)"),
                       ("total_num_segments = len(np.unique(segments))", "masked_img = normalize_image(masked_img)"),
                       "def eval_superpixel(", "masks_mnist.npz")


def make_resnet56():
    sys.path.insert(0, REF)
    mod = _load_ref_module("ref_models_resnet", "models/resnet.py")
    with contextlib.redirect_stdout(io.StringIO()):
        model = mod.createModel(depth=56, data="cifar10", num_classes=10)
    ck = torch.load(os.path.join(REF, "saved_checkpoints/cifar10+-resnet-56/model_best.pth.tar"), map_location="cpu",
                    weights_only=False)
    dp = torch.nn.DataParallel(model)      # generate_gp_training_data_cifar.py:75,249-250
    dp.load_state_dict(ck["state_dict"])
    dp.eval()
    torch.manual_seed(0)
    x = torch.rand(4, 3, 32, 32)
    with torch.no_grad():
        y = dp.module(x)
    np.savez_compressed(os.path.join(OUT, "resnet56.npz"), x=x.numpy(), logits=y.numpy())


def make_mnist_net():
    """generate_gp_training_data_mnist.py cannot be imported (argparse + dataset download at import time, :44-69): its
    `conv` helper and `Classification_Net` class statements (:72-105) are exec'd as they stand, the shipped checkpoint is
    loaded the way the script does (:157-158, key 'model'), and the 4-tuple of a seeded batch is recorded."""
    rel = "generate_gp_training_data_mnist.py"
    code, span = _extract(rel, "def conv(", "return x0, x1, x2, pred0")
    ns = _run(code, {"nn": torch.nn, "torch": torch})
    model = ns["Classification_Net"]()
    ck = torch.load(os.path.join(REF, "saved_checkpoints/mnist/checkpoint.pth.tar"), map_location="cpu", weights_only=False)
    model.load_state_dict(ck["model"])
    model.eval()
    torch.manual_seed(0)
    x = torch.rand(4, 1, 28, 28)
    with torch.no_grad():
        x0, x1, x2, pred0 = model(x)
    np.savez_compressed(os.path.join(OUT, "mnist_net.npz"), x=x.numpy(), pred0=pred0.numpy(), x2=x2.numpy(),
                        x0_mean=x0.mean((2, 3)).numpy(), x1_mean=x1.mean((2, 3)).numpy(), ref_lines=np.array(span))


def make_utils():
    """utils.py imports cleanly: normalize_image and generate_IOU are executed as they stand.  generate_boundingbox unpacks
    three values from cv2.findContours (OpenCV 3) and raises under the container's OpenCV 4, so it is not pinned."""
    import tempfile
    mod = _load_ref_module("ref_utils", "utils.py")
    rng = np.random.RandomState(0)
    img_u8 = rng.randint(0, 256, size=(5, 7, 3)).astype(np.uint8)
    norm = mod.normalize_image(img_u8)
    boxes = rng.randint(0, 200, size=(16, 2, 2))
    A = np.concatenate([boxes[:, 0], boxes[:, 0] + rng.randint(1, 60, size=(16, 2))], 1)
    B = np.concatenate([boxes[:, 1], boxes[:, 1] + rng.randint(1, 60, size=(16, 2))], 1)
    canvas = np.zeros((300, 300, 3), np.uint8)
    with tempfile.TemporaryDirectory() as d, contextlib.redirect_stdout(io.StringIO()):
        iou = np.array([mod.generate_IOU(list(a), list(b), canvas, k, d) for k, (a, b) in enumerate(zip(A, B))])
    np.savez_compressed(os.path.join(OUT, "utils.npz"), img_u8=img_u8, norm=norm, boxA=A, boxB=B, iou=iou)


def make_ei():
    rel = "BayesianOptimization.py"
    code, span = _extract(rel, "def expected_improvement(", "return -1 * expected_improvement")
    from scipy.stats import norm

    class StubGP:
        def __init__(self, mu, sigma):
            self.mu, self.sigma = mu, sigma

        def predict(self, x, return_std=True):
            return self.mu, self.sigma

    rng = np.random.RandomState(5)
    mu = rng.randn(64)
    sigma = np.abs(rng.randn(64)) * 0.5
    sigma[3] = 0.0
    losses = rng.randn(9)
    ns = dict(np=np, norm=norm)
    _run(code, ns)
    with np.errstate(all="ignore"):
        neg_ei_max = ns["expected_improvement"](np.zeros((64, 1)), StubGP(mu, sigma), losses, greater_is_better=True, n_params=1)
        neg_ei_min = ns["expected_improvement"](np.zeros((64, 1)), StubGP(mu, sigma), losses, greater_is_better=False, n_params=1)
    np.savez_compressed(os.path.join(OUT, "ei.npz"), mu=mu, sigma=sigma, losses=losses, neg_ei_max=neg_ei_max,
                        neg_ei_min=neg_ei_min, ref_lines=np.array(span))


def make_gp_sklearn():
    import sklearn
    import sklearn.gaussian_process as gp

    rng = np.random.RandomState(0)
    S, n, m = 50, 96, 40
    X = np.zeros((n + m, S))
    for i in range(n + m):
        X[i, rng.choice(S - 1, 20, replace=False)] = 1.0
    w = rng.randn(S)
    y = 1.0 / (1.0 + np.exp(-(X @ w) * 0.3))
    Xt, yt, Xq = X[:n], y[:n], X[n:]
    # exactly BayesianOptimization.py:154-159 (+ a seed so the fixture is reproducible)
    model = gp.GaussianProcessRegressor(kernel=gp.kernels.RBF(), alpha=1e-5, n_restarts_optimizer=10, normalize_y=True,
                                        random_state=0)
    model.fit(Xt, yt)
    mu, std = model.predict(Xq, return_std=True)
    thetas = np.log(np.array([0.5, 1.0, 2.0, 4.0, 8.0]))
    lml = np.array([model.log_marginal_likelihood(np.array([t]), eval_gradient=True) for t in thetas], dtype=object)
    np.savez_compressed(os.path.join(OUT, "gp_sklearn.npz"), Xt=Xt, yt=yt, Xq=Xq, length_scale=model.kernel_.length_scale,
                        y_mean=model._y_train_mean, y_std=model._y_train_std, alpha_vec=model.alpha_, L=model.L_,
                        mu=mu, std=std, thetas=thetas, lml=np.array([v[0] for v in lml]),
                        lml_grad=np.array([v[1][0] for v in lml]), lml_opt=model.log_marginal_likelihood_value_,
                        sklearn_version=sklearn.__version__)
    # the reference's actual use: 1-D firstIndex inputs, n = 13 (BayesianOptimization.py:137-166)
    x1 = np.array([[3.], [17.], [25.], [8.], [12.], [29.], [1.], [21.], [14.], [6.], [27.], [10.], [19.]])
    y1 = np.sin(x1[:, 0] / 5.0) * 0.4 + 0.5
    m1 = gp.GaussianProcessRegressor(kernel=gp.kernels.RBF(), alpha=1e-5, n_restarts_optimizer=10, normalize_y=True,
                                     random_state=1).fit(x1, y1)
    xq1 = np.arange(0, 30, dtype=np.float64)[:, None]
    mu1, std1 = m1.predict(xq1, return_std=True)
    np.savez_compressed(os.path.join(OUT, "gp_sklearn_1d.npz"), x=x1, y=y1, xq=xq1, length_scale=m1.kernel_.length_scale,
                        mu=mu1, std=std1, lml_opt=m1.log_marginal_likelihood_value_)


def make_localize():
    """generate_gp_training_data_imagenet.py: the function definitions get_pixel_sorted_mask_label (:490-515) and
    generate_new_mask (:549-565) plus the min-max / uint8 statements of plot_summed_heatmap (:519-525), exec'd on a
    ./masks directory written in the reference's own format (mask_{i}_{label}.png, 0/255)."""
    import tempfile
    import cv2
    rel = "generate_gp_training_data_imagenet.py"
    defs1, span1 = _extract(rel, "def load_images_from_folder(folder):", "return img_filenames, labels")
    defs2, span2 = _extract(rel, "def get_pixel_sorted_mask_label():", "return dict_pixel")
    defs3, span3 = _extract(rel, "def generate_new_mask(dict_pixel, mask_threshold):", "return result_mask")
    norm, span4 = _extract(rel, "result_gray_img_show = result_gray_img.copy()",
                           "result_gray_img_show = np.array(result_gray_img_show, dtype = np.uint8)", after="def plot_summed_heatmap(")
    n = 24
    segments = synthetic.voronoi_labels(n, n, 13, seed=4)
    rng = random.Random(99)
    S, k = 13, int(0.4 * 13)
    sels, labels = [], []
    for _ in range(40):
        f = rng.randint(1, S - k)
        sels.append(list(range(f, f + k)))
        labels.append(rng.randint(0, 1))
    cwd = os.getcwd()
    with tempfile.TemporaryDirectory() as td:
        os.chdir(td)
        try:
            os.makedirs("masks")
            for i, (sel, lab) in enumerate(zip(sels, labels)):
                m = np.isin(segments, sel).astype(np.uint8) * 255
                cv2.imwrite("masks/mask_{}_{}.png".format(i, lab), m)
            ns = dict(np=np, os=os, cv2=cv2, n=n)
            _run(defs1 + "\n" + defs2 + "\n" + defs3, ns)
            with contextlib.redirect_stdout(io.StringIO()):
                dict_pixel = ns["get_pixel_sorted_mask_label"]()
            heat = np.full((n, n), -1.0)
            for (i, j), v in dict_pixel.items():
                heat[i, j] = v
            values = sorted(set(dict_pixel.values()))
            with contextlib.redirect_stdout(io.StringIO()):
                new_masks = np.stack([ns["generate_new_mask"](dict_pixel, t) for t in values])
            dense = np.where(heat >= 0, heat, 0.0)
            ns2 = dict(np=np, result_gray_img=dense.copy())
            _run(norm, ns2)
            gray = ns2["result_gray_img_show"]
        finally:
            os.chdir(cwd)
    np.savez_compressed(os.path.join(OUT, "localize.npz"), segments=segments, sels=np.array(sels, dtype=np.int64),
                        labels=np.array(labels, dtype=np.int64), heat=heat, values=np.array(values, dtype=np.float64),
                        new_masks=new_masks, gray=gray, ref_lines=np.array([span1, span2, span3, span4]))


if __name__ == "__main__":
    if len(sys.argv) != 2 or not os.path.isdir(sys.argv[1]):
        raise SystemExit("usage: python tests/golden/make_golden.py <checkout of LiliMeng/network_interpretation_imagenet>")
    REF = os.path.abspath(sys.argv[1])
    make_masks_imagenet()
    make_masks_cifar()
    make_masks_mnist()
    make_resnet56()
    make_mnist_net()
    make_utils()
    make_ei()
    make_gp_sklearn()
    make_localize()
    for f in sorted(os.listdir(OUT)):
        if f.endswith(".npz"):
            print(f, os.path.getsize(os.path.join(OUT, f)))

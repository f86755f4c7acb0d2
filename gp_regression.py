"""Drop-in for the reference's gp_regression.py: GP regression of the summed mask labels over pixel coordinates.

Same entry points and on-disk contract as the reference (file:line are the reference's):
  load_images_from_folder(folder)        :63-72    ./masks/mask_{i}_{label}.png, label parsed from the file name
  prepare_training_data()                :74-156   heat map H[p] = sum of labels of the masks whose pixel p is 255; train_x = the
                                                   covered pixel coordinates (i, j), train_y = H there
  GPRegressionModel(train_x, train_y, likelihood, grid_size=30)  :160-176  KISS-GP: RBF on a grid_size x grid_size interpolation
                                                   grid over [0, n]^2 + outputscale (grid_size=300 as the reference's
                                                   gp_superpixel_data_imagenet.py uses: the Kronecker solver, see below)
  train(...)                             :179-229  evaluates the marginal likelihood 20 times WITHOUT stepping the optimiser in the
                                                   branch it runs, then saves the (initial) parameters
  eval_superpixels(model, likelihood)    :232-281  posterior of `likelihood(model(x))` at all n x n pixels
  plot_result(predictions)               :284-372  heat maps (written to ./weighted_mask/ here instead of cv2.imshow / matplotlib)

What changed underneath: the O(N * n^2) Python dictionary loop is one HBM-bound kernel (`nib_heatmap_pixels`), and the GP is
solved exactly in its inducing-weight form on the device (network_interpretation_imagenet_b200/ski.py, csrc/ski.cu + gp.cu):
with dense G x G factors (G = grid_size^2) up to grid_size 100, and above that, where they no longer fit, matrix-free by
preconditioned conjugate gradients on the Kronecker structure of the grid kernel (csrc/ski_kron.cu).  The checkpoint
keeps grid_size, so eval_superpixels predicts on the grid the model was trained with.
gpytorch is not needed (and absent here): the checkpoint is a small dict of the model's hyper-parameters.
"""
from __future__ import annotations

import os

import cv2
import numpy as np
import torch

from network_interpretation_imagenet_b200.ski import GridGPRegression, heatmap_from_masks

dataset = 'IMAGENET'

# mode = 'Train'
mode = 'Eval'

if dataset == 'MNIST':
    n = 28
elif dataset == 'CIFAR':
    n = 32
elif dataset == 'IMAGENET':
    n = 224
else:
    raise Exception("This dataset Not implemented yet")

CHECKPOINT = './gp_saved_checkpoints/imagenet1000_gp_reg_checkpoint.pth.tar'


def load_images_from_folder(folder):
    img_filenames = []
    labels = []
    for filename in os.listdir(folder):
        label = filename.split('_')[2].split('.')[0]
        img_filenames.append(os.path.join(folder, filename))
        labels.append(label)
    return img_filenames, labels


def summed_label_heatmap(folder='./masks/'):
    """(H [n,n] fp32 CUDA, covered [n,n] bool CUDA): the reference's dict_pixel, built on the device in batches."""
    mask_filenames, labels = load_images_from_folder(folder)
    heat = torch.zeros(n, n, dtype=torch.float32, device="cuda")
    covered = torch.zeros(n, n, dtype=torch.float32, device="cuda")
    for i in range(0, len(mask_filenames), 2048):
        batch = np.stack([cv2.imread(f, 0) for f in mask_filenames[i:i + 2048]])
        lab = np.asarray([int(v) for v in labels[i:i + 2048]], dtype=np.float32)
        heat += heatmap_from_masks(batch, lab)
        covered += heatmap_from_masks(batch, np.ones_like(lab))
    return heat, covered > 0


def _to_u8(gray: np.ndarray) -> np.ndarray:
    g = gray.astype(np.float64).copy()
    g -= g.min()
    if g.max() > 0:
        g /= g.max()
    g *= 255
    return np.array(g, dtype=np.uint8)


def prepare_training_data():
    heat, covered = summed_label_heatmap('./masks/')
    idx = torch.nonzero(covered)                       # row-major (i, j) order, as the reference's nested loops
    train_x = idx.to(torch.float32)
    train_y = heat[covered]
    os.makedirs('./weighted_mask', exist_ok=True)
    cv2.imwrite('./weighted_mask/weighted_mask_heatmap.png', cv2.applyColorMap(_to_u8(heat.cpu().numpy()), cv2.COLORMAP_JET))
    print("train_x.shape: ", train_x.shape)
    print("train_y.shape: ", train_y.shape)
    return train_x, train_y


class GaussianLikelihood:
    """Stand-in for gpytorch.likelihoods.GaussianLikelihood: holds log_noise (initial value 0, as gpytorch's)."""

    def __init__(self):
        self.log_noise = 0.0

    def cuda(self):
        return self

    def train(self):
        return self

    def eval(self):
        return self


class GPRegressionModel:
    """KISS-GP regression with the reference's structure: near-zero constant mean, RBF base kernel on a grid_size x
    grid_size interpolation grid over [0, n]^2 (30 by default, as the reference's gp_regression.py; 300 as its
    gp_superpixel_data_imagenet.py), trainable log_outputscale (all initial values 0, as gpytorch's parameters)."""

    def __init__(self, train_x, train_y, likelihood, grid_size=30):
        self.train_x, self.train_y, self.likelihood = train_x, train_y, likelihood
        self.grid_size = grid_size
        self.log_lengthscale = 0.0
        self.log_outputscale = 0.0
        self.constant_mean = 0.0
        self._gp = None

    def cuda(self):
        return self

    def train(self):
        return self

    def eval(self):
        return self

    def state_dict(self):
        return {"log_lengthscale": self.log_lengthscale, "log_outputscale": self.log_outputscale,
                "constant_mean": self.constant_mean, "log_noise": self.likelihood.log_noise, "grid_size": self.grid_size}

    def load_state_dict(self, sd):
        self.log_lengthscale, self.log_outputscale = float(sd["log_lengthscale"]), float(sd["log_outputscale"])
        self.constant_mean, self.likelihood.log_noise = float(sd["constant_mean"]), float(sd["log_noise"])
        self.grid_size = int(sd.get("grid_size", self.grid_size))
        self._gp = None

    def fit(self):
        self._gp = GridGPRegression(self.grid_size, ((0.0, float(n)), (0.0, float(n))), np.exp(self.log_lengthscale),
                                    np.exp(self.log_outputscale), np.exp(self.likelihood.log_noise),
                                    self.constant_mean).fit(self.train_x, self.train_y)
        return self

    def predict(self, x, likelihood=True):
        if self._gp is None:
            self.fit()
        return self._gp.predict(x, return_var=True, likelihood=likelihood)


def train(train_x, train_y, model, optimizer=None, mll=None):
    # the reference computes the loss 20 times and never calls backward()/step() in this branch (:206-217): the parameters it
    # saves are the initial ones.  We fit once at those parameters and save them.
    model.fit()
    os.makedirs(os.path.dirname(CHECKPOINT), exist_ok=True)
    torch.save(model.state_dict(), CHECKPOINT)


def eval_superpixels(model, likelihood):
    if os.path.exists(CHECKPOINT):
        model.load_state_dict(torch.load(CHECKPOINT))
    model.eval()
    likelihood.eval()
    ii, jj = torch.meshgrid(torch.arange(n, dtype=torch.float32), torch.arange(n, dtype=torch.float32), indexing="ij")
    test_x = torch.stack([ii, jj], -1).reshape(-1, 2).cuda()
    print("test_x.shape")
    print(test_x.shape)
    mean, var = model.predict(test_x)          # all n*n pixels in one call (the reference loops over batches of 896)
    full_predictions = mean.cpu().numpy()
    print(full_predictions.shape)
    eval_superpixels.last_variance = var.cpu().numpy()
    return full_predictions


def plot_result(predictions):
    heat, _ = summed_label_heatmap('./masks')
    os.makedirs('./weighted_mask', exist_ok=True)
    cv2.imwrite('./weighted_mask/summed_label_training_heatmap.png',
                cv2.applyColorMap(_to_u8(heat.cpu().numpy()), cv2.COLORMAP_JET))
    org_test_gray_img = np.asarray(predictions).reshape(n, n)
    cv2.imwrite('./weighted_mask/predicted_mask_heatmap.png', cv2.applyColorMap(_to_u8(org_test_gray_img), cv2.COLORMAP_JET))
    var = getattr(eval_superpixels, "last_variance", None)
    if var is not None:
        cv2.imwrite('./weighted_mask/predicted_variance_heatmap.png', cv2.applyColorMap(_to_u8(var.reshape(n, n)), cv2.COLORMAP_JET))


def main():
    likelihood = GaussianLikelihood().cuda()
    train_x, train_y = prepare_training_data()
    model = GPRegressionModel(train_x, train_y, likelihood).cuda()
    if mode == 'Train':
        model.train()
        likelihood.train()
        train(train_x, train_y, model)
    elif mode == 'Eval':
        print("start to test the model")
        predictions = eval_superpixels(model, likelihood)
        plot_result(predictions)
    else:
        raise Exception("No such mode")


if __name__ == "__main__":
    main()

"""Drop-in for the reference's BayesianOptimization.py: same function names and signatures, with the Gaussian
process, its posterior and the Expected-Improvement acquisition computed by libnib.so on the B200.

  expected_improvement(x, gaussian_process, evaluated_loss, greater_is_better, n_params)   reference :16-54
  sample_next_hyperparameter(acquisition_func, gaussian_process, evaluated_loss, ...)      reference :57-96
  bayesian_optimisation(n_iters, sample_loss, val_loader, nn_model, criterion, bounds, ...) reference :99-192

Reference behaviours kept on purpose (SURVEY.md App. D): EI is returned negated; sigma == 0 yields NaN (the
reference's `== 0.0` line :52 is a comparison, not an assignment); the multi-start search starts from every
integer in [lo, hi) and ignores `n_restarts` (:84-90); duplicates are replaced by a random draw (:178-180).

`bayesian_optimisation_masks` is the scaled-up form BASELINE.json's config 4 names: the GP input is the mask
itself (selection bit-vector, Hamming-RBF kernel) and each round scores all m candidate masks on the device
(fit -> posterior on m candidates -> EI arg-max -> one new evaluation -> append), or with `batch_size` q > 1 q
Kriging-believer picks per round, scored in one batched forward."""
from __future__ import annotations

from random import randint

import numpy as np
from scipy.optimize import minimize

from network_interpretation_imagenet_b200 import gp as _gp
from network_interpretation_imagenet_b200.gp import GaussianProcessRegressor


def expected_improvement(x, gaussian_process, evaluated_loss, greater_is_better=False, n_params=1):
    """-EI at x (reference :16-54).  `gaussian_process` may be the engine's GP or any sklearn-like estimator."""
    if isinstance(gaussian_process, GaussianProcessRegressor):
        return _gp.expected_improvement(x, gaussian_process, evaluated_loss, greater_is_better, n_params)
    from scipy.stats import norm
    x_to_predict = np.asarray(x).reshape(-1, n_params)
    mu, sigma = gaussian_process.predict(x_to_predict, return_std=True)
    loss_optimum = np.max(evaluated_loss) if greater_is_better else np.min(evaluated_loss)
    scaling_factor = (-1) ** (not greater_is_better)
    with np.errstate(divide="ignore", invalid="ignore"):
        Z = scaling_factor * (mu - loss_optimum) / sigma
        ei = scaling_factor * (mu - loss_optimum) * norm.cdf(Z) + sigma * norm.pdf(Z)
    return -1 * ei


def sample_next_hyperparameter(acquisition_func, gaussian_process, evaluated_loss, greater_is_better=False,
                               bounds=(0, 10), n_restarts=25):
    """L-BFGS-B on the acquisition from every integer start in [bounds[0][0], bounds[0][1]) (reference :57-96)."""
    best_x = None
    best_acquisition_value = 1
    n_params = bounds.shape[0]
    for starting_point in range(bounds[0][0], bounds[0][1]):
        res = minimize(fun=acquisition_func, x0=[starting_point], bounds=bounds, method="L-BFGS-B",
                       args=(gaussian_process, evaluated_loss, greater_is_better, n_params))
        if res.fun < best_acquisition_value:
            best_acquisition_value = res.fun
            best_x = res.x
    return best_x


def bayesian_optimisation(n_iters, sample_loss, val_loader, nn_model, criterion, bounds, x0=None, n_pre_samples=5,
                          gp_params=None, random_search=False, alpha=1e-5, epsilon=1e-7):
    """Reference :99-192 with the GP on the device.  Returns (xp, yp)."""
    x_list, y_list = [], []
    n_params = bounds.shape[0]
    if x0 is None:
        for _ in range(n_pre_samples):
            params = [randint(bounds[0][0], bounds[0][1])]
            x_list.append(params)
            y_list.append(sample_loss(params, val_loader, nn_model, criterion))
    else:
        for params in x0:
            x_list.append(params)
            y_list.append(sample_loss(params, val_loader, nn_model, criterion))
    xp, yp = np.array(x_list), np.array(y_list)
    if gp_params is not None:
        model = GaussianProcessRegressor(**gp_params)
    else:   # kernel = RBF(), alpha, n_restarts_optimizer=10, normalize_y=True (reference :152-159)
        model = GaussianProcessRegressor(alpha=alpha, n_restarts_optimizer=10, normalize_y=True)
    for _ in range(n_iters):
        model.fit(xp.astype(np.float64), yp)
        if random_search:
            x_random = np.array([[randint(bounds[0][0], bounds[0][1])] for _ in range(int(random_search))], dtype=np.float64)
            ei = -1 * expected_improvement(x_random, model, yp, greater_is_better=True, n_params=n_params)
            next_sample = x_random[np.argmax(ei), :]
        else:
            next_sample = sample_next_hyperparameter(expected_improvement, model, yp, greater_is_better=True,
                                                     bounds=bounds, n_restarts=100)
        if next_sample is None or np.any(np.abs(next_sample - xp) <= epsilon):
            next_sample = [randint(bounds[0][0], bounds[0][1])]
        cv_score = sample_loss(next_sample, val_loader, nn_model, criterion)
        x_list.append(next_sample)
        y_list.append(cv_score)
        xp, yp = np.array(x_list), np.array(y_list)
    return xp, yp


def bayesian_optimisation_masks(n_iters, score_masks, train_bits, train_scores, candidate_bits, alpha=1e-5,
                                length_scale=None, n_restarts_optimizer=0, refit_every=0, random_state=0, batch_size=1):
    """Active learning over masks (BASELINE config 4: `n_iters` rounds on n training masks, m candidates).

    score_masks(bits[k, words]) -> np.ndarray[k] target-class probabilities, e.g.
    `lambda b: engine.score_masks(b)["target_prob"].cpu().numpy()` (PerturbationEngine.score_masks itself returns a dict
    of device tensors).
    Each round: GP fit on (train_bits, train_scores) -> posterior mean/std on every remaining candidate -> EI
    (greater_is_better, as reference :175) -> arg-max candidate is evaluated and appended.

    batch_size = q > 1 evaluates q masks per round: ActiveMaskGP.select_batch picks them by greedy Kriging believer on
    the device, one score_masks call scores them together, and set_batch_values enters the scores.  It needs the fixed
    length scale (`length_scale` given, refit_every = 0).  The history has one entry per evaluated mask."""
    import torch
    Z = np.ascontiguousarray(train_bits, dtype=np.uint64).copy()
    y = np.asarray(train_scores, dtype=np.float64).copy()
    cand = np.ascontiguousarray(candidate_bits, dtype=np.uint64)
    history = []
    q = int(batch_size)
    if q < 1:
        raise ValueError("batch_size must be >= 1")
    if q > 1:
        if length_scale is None or refit_every:
            raise ValueError("batch_size > 1 needs a fixed length_scale and refit_every=0: batch selection extends the "
                             "resident factor, which a length-scale search would rebuild")
        gp = _gp.ActiveMaskGP(cand, alpha=alpha, length_scale=length_scale, normalize_y=True,
                              capacity=n_iters * q).fit(Z, y)
        for it in range(n_iters):
            picks, ei = gp.select_batch(q, greater_is_better=True)
            if len(picks) == 0:   # every EI is NaN (all sigma == 0): one random candidate like reference :178-180
                alive = np.nonzero(gp.alive.cpu().numpy())[0]
                j = int(alive[np.random.RandomState(random_state + it).randint(len(alive))])
                s = float(np.asarray(score_masks(cand[j:j + 1]))[0])
                history.append({"round": it, "candidate": j, "ei": float("nan"), "score": s, "length_scale": length_scale})
                gp.append(j, s)
                continue
            scores = np.asarray(score_masks(cand[picks]), dtype=np.float64).reshape(-1)
            gp.set_batch_values(scores)
            for j, e, s in zip(picks, ei, scores):
                history.append({"round": it, "candidate": int(j), "ei": float(e), "score": float(s),
                                "length_scale": length_scale})
        return np.concatenate([Z, cand[[h["candidate"] for h in history]]], 0), np.asarray(gp.y_host), history
    if length_scale is not None and not refit_every:
        # fixed length scale: the Gram matrix of the points already seen never changes, so each round is a rank-one update
        # of the factor and of the posterior workspace (ActiveMaskGP) instead of an O(n^3 + m n^2) refit
        gp = _gp.ActiveMaskGP(cand, alpha=alpha, length_scale=length_scale, normalize_y=True, capacity=n_iters).fit(Z, y)
        for it in range(n_iters):
            mu, var, sd = gp.posterior()
            ei, arg = _gp.expected_improvement_device(mu, sd, float(np.max(gp.y_host)), True)
            j = int(arg.item())
            if j < 0:   # every EI is NaN (all sigma == 0): fall back to a random candidate like reference :178-180
                alive = np.nonzero(gp.alive.cpu().numpy())[0]
                j = int(alive[np.random.RandomState(random_state + it).randint(len(alive))])
            s = float(np.asarray(score_masks(cand[j:j + 1]))[0])
            history.append({"round": it, "candidate": j, "ei": float(ei[j].item()), "score": s, "length_scale": length_scale})
            gp.append(j, s)
        return np.concatenate([Z, cand[[h["candidate"] for h in history]]], 0), np.asarray(gp.y_host), history
    alive = np.ones(cand.shape[0], dtype=bool)
    ell = length_scale
    for it in range(n_iters):
        optimise = ell is None or (refit_every and it % refit_every == 0 and it > 0)
        gp = GaussianProcessRegressor(alpha=alpha, normalize_y=True, length_scale=ell or 1.0,
                                      optimizer="fmin_l_bfgs_b" if optimise else None,
                                      n_restarts_optimizer=n_restarts_optimizer, random_state=random_state)
        gp.fit(Z, y)
        ell = gp.length_scale_
        idx = np.nonzero(alive)[0]
        mu, var, sd = gp.predict_device(cand[idx])
        ei, arg = _gp.expected_improvement_device(mu, sd, float(y.max()), True)
        j = int(arg.item())
        if j < 0:   # every EI is NaN (all sigma == 0): fall back to a random candidate like reference :178-180
            j = int(np.random.RandomState(random_state + it).randint(len(idx)))
        pick = idx[j]
        alive[pick] = False
        s = float(np.asarray(score_masks(cand[pick:pick + 1]))[0])
        history.append({"round": it, "candidate": int(pick), "ei": float(ei[j].item()), "score": s, "length_scale": ell})
        Z = np.concatenate([Z, cand[pick:pick + 1]], 0)
        y = np.concatenate([y, [s]])
        del gp
    return Z, y, history

"""CPU: the Kriging-believer batch oracle (oracle/kriging_believer.py) against the dense GP it abbreviates."""
import numpy as np
import pytest

from oracle import gp as ogp
from oracle import masks as om
from oracle.kriging_believer import kriging_believer_batch


def _problem(n, m, S, seed):
    rng = np.random.RandomState(seed)
    sels, seen = [], set()
    while len(sels) < n + m:                        # distinct masks
        s = tuple(sorted(rng.choice(S - 1, size=max(1, int(0.4 * S)), replace=False)))
        if s not in seen:
            seen.add(s)
            sels.append(list(s))
    X = ogp.bits_to_matrix(om.selection_bits(sels, S), S)
    return X[:n], rng.rand(n), X[n:]


@pytest.mark.parametrize("gib", [True, False])
def test_fantasies_leave_the_mean_unchanged_and_give_the_oracle_variances(gib):
    """The premise: refitting with each pick's fantasy (its posterior mean) appended, y-normalisation frozen, leaves the
    mean at every candidate unchanged and yields exactly the variances the oracle selects with."""
    Xt, y, C = _problem(60, 80, 30, 1)
    ell, alpha, q = 3.0, 1e-5, 6
    kb = kriging_believer_batch(Xt, y, C, q, ell, alpha, greater_is_better=gib)
    assert len(kb["picks"]) == q and len(set(kb["picks"].tolist())) == q
    fit = ogp.gp_fit(Xt, y, ell, alpha)
    ybar, ystd = fit["y_mean"], fit["y_std"]
    for k in range(1, q + 1):
        P = kb["picks"][:k]
        yn = np.concatenate([(y - ybar) / ystd, (kb["mu"][P] - ybar) / ystd])
        f = ogp.gp_fit(np.vstack([Xt, C[P]]), yn, ell, alpha, normalize_y=False)
        mu_n, var_n, _ = ogp.gp_predict(f, C)
        np.testing.assert_allclose(ystd * mu_n + ybar, kb["mu"], rtol=0, atol=1e-10)
        np.testing.assert_allclose(var_n, kb["var"][k], rtol=0, atol=1e-10)


def test_single_pick_is_the_expected_improvement_argmax():
    Xt, y, C = _problem(50, 70, 30, 2)
    kb = kriging_believer_batch(Xt, y, C, 1, 3.0)
    mu, _, sd = ogp.gp_predict(ogp.gp_fit(Xt, y, 3.0), C)
    ei = -ogp.expected_improvement(mu, sd, y, greater_is_better=True)
    assert kb["picks"].tolist() == [int(np.argmax(ei))]
    np.testing.assert_allclose(kb["ei_at_pick"][0], ei.max(), rtol=1e-12)


@pytest.mark.parametrize("n,m,q", [(40, 60, 8), (130, 70, 20)])
def test_bordered_form_matches_refactoring_from_scratch(n, m, q):
    Xt, y, C = _problem(n, m, 40, n + m)
    a = kriging_believer_batch(Xt, y, C, q, 3.0)
    b = kriging_believer_batch(Xt, y, C, q, 3.0, bordered=True)
    assert a["picks"].tolist() == b["picks"].tolist()
    np.testing.assert_allclose(b["var"], a["var"], rtol=0, atol=1e-10)
    np.testing.assert_allclose(b["ei_at_pick"], a["ei_at_pick"], rtol=1e-9)


def test_used_candidates_are_never_picked_and_the_batch_stops_when_the_pool_is_empty():
    Xt, y, C = _problem(30, 5, 30, 3)
    kb = kriging_believer_batch(Xt, y, C, 9, 3.0)
    assert sorted(kb["picks"].tolist()) == list(range(5))


def test_follow_conditions_on_the_given_path():
    Xt, y, C = _problem(40, 50, 30, 4)
    own = kriging_believer_batch(Xt, y, C, 5, 3.0)
    path = [int(i) for i in np.argsort(own["mu"])[:5]]
    f = kriging_believer_batch(Xt, y, C, 5, 3.0, follow=path)
    assert f["picks"][0] == own["picks"][0]                      # the first step sees the same state
    ref = kriging_believer_batch(Xt, y, C, 5, 3.0, bordered=True, follow=path)
    np.testing.assert_allclose(f["var"], ref["var"], rtol=0, atol=1e-10)
    np.testing.assert_allclose(f["ei_at_pick"], [f["ei"][k][path[k]] for k in range(5)], rtol=0)

"""GPU: batch acquisition by greedy Kriging believer (ActiveMaskGP.select_batch / nib_gp_kb_select) against the dense
numpy oracle (oracle/kriging_believer.py), the from-scratch GP fits, the one-at-a-time rank-one path and the engine."""
import numpy as np
import pytest
import torch

from oracle import gp as ogp
from oracle import masks as om
from oracle.kriging_believer import kriging_believer_batch

pytestmark = pytest.mark.gpu

ELL = 3.0


def _distinct_masks(count, S, seed, size=None):
    rng = np.random.RandomState(seed)
    sels, seen = [], set()
    while len(sels) < count:                        # distinct masks (a duplicate makes K singular up to alpha)
        s = tuple(sorted(rng.choice(S - 1, size=size or max(1, int(0.4 * S)), replace=False)))
        if s not in seen:
            seen.add(s)
            sels.append(list(s))
    return om.selection_bits(sels, S), rng


@pytest.fixture
def problem():
    def make(n0, m, S, seed=None):
        Z, rng = _distinct_masks(n0 + m, S, n0 + m + S if seed is None else seed)
        return Z[:n0], rng.rand(n0), Z[n0:], rng
    return make


def _check_against_oracle(agp, picks, ei, Zt, y, cand, S, q, bordered=False, gib=True):
    """GPU picks == oracle picks up to EI ties (rel 1e-9), EI at the picks to 1e-8, fantasised variances to 1e-9."""
    kb = kriging_believer_batch(ogp.bits_to_matrix(Zt, S), y, ogp.bits_to_matrix(cand, S), q, ELL, bordered=bordered,
                                follow=picks, greater_is_better=gib)
    assert len(kb["picks"]) == len(picks)
    for k, j in enumerate(picks):
        top = np.nanmax(kb["ei"][k])
        assert j == kb["picks"][k] or abs(kb["ei"][k][j] - top) <= 1e-9 * abs(top), (k, j, kb["picks"][k])
    np.testing.assert_allclose(ei, kb["ei_at_pick"], rtol=1e-8, atol=0)
    var = (1.0 - agp.ssq).clamp(min=0.0).cpu().numpy()
    assert np.abs(var - kb["var"][-1]).max() <= 1e-9, np.abs(var - kb["var"][-1]).max()


@pytest.mark.parametrize("n0,m,q,S,gib", [(200, 300, 7, 50, True), (1000, 513, 64, 50, True), (256, 1024, 33, 100, True),
                                          (200, 300, 7, 50, False), (256, 1024, 33, 100, False)])
def test_batch_matches_the_oracle(nib, problem, n0, m, q, S, gib):
    Zt, y, cand, _ = problem(n0, m, S)
    agp = nib.ActiveMaskGP(cand, alpha=1e-5, length_scale=ELL, capacity=q).fit(Zt, y)
    picks, ei = agp.select_batch(q, greater_is_better=gib)
    assert len(picks) == q and len(set(picks.tolist())) == q and agp.n == n0 + q
    _check_against_oracle(agp, picks, ei, Zt, y, cand, S, q, gib=gib)
    alive = agp.alive.cpu().numpy()
    assert not alive[picks].any() and alive.sum() == m - q
    assert np.array_equal(agp.X_d[n0:n0 + q].cpu().numpy().view(np.uint64), cand[picks])


@pytest.mark.parametrize("n0,m,q,rounds", [(200, 300, 7, 3), (100, 257, 40, 2)])
def test_mean_is_unchanged_and_measured_values_equal_a_refit(nib, problem, n0, m, q, rounds):
    S = 50
    Zt, y, cand, rng = problem(n0, m, S)
    agp = nib.ActiveMaskGP(cand, alpha=1e-5, length_scale=ELL, capacity=q * rounds).fit(Zt, y)
    used, ys = [], []
    for _ in range(rounds):
        mu0, _, _ = agp.posterior()
        picks, _ = agp.select_batch(q)
        mu1, var1, sd1 = agp.posterior()
        assert torch.equal(mu0, mu1)                                   # the believer's fantasies leave the mean alone
        assert torch.isnan(sd1[torch.from_numpy(picks).cuda()]).all()
        yb = rng.rand(len(picks))
        agp.set_batch_values(yb)
        used += picks.tolist()
        ys += yb.tolist()
    assert len(set(used)) == len(used) == q * rounds
    mu, var, sd = (t.cpu().numpy() for t in agp.posterior())
    Zg, yg = np.concatenate([Zt, cand[used]], 0), np.concatenate([y, ys])
    assert agp.y_host == list(yg)
    mu0, var0, sd0 = ogp.gp_predict(ogp.gp_fit(ogp.bits_to_matrix(Zg, S), yg, ELL), ogp.bits_to_matrix(cand, S))
    live = np.ones(m, bool)
    live[used] = False
    assert np.isnan(sd[~live]).all() and not np.isnan(sd[live]).any()
    np.testing.assert_allclose(mu, mu0, rtol=1e-6, atol=1e-7)
    np.testing.assert_allclose(sd[live], sd0[live], rtol=1e-4, atol=1e-6)
    ref = nib.GaussianProcessRegressor(alpha=1e-5, length_scale=ELL, optimizer=None).fit(Zg, yg)
    mu1, var1, _ = (t.cpu().numpy() for t in ref.predict_device(cand))
    np.testing.assert_allclose(mu, mu1, rtol=1e-7, atol=1e-8)
    np.testing.assert_allclose(var, var1, rtol=1e-5, atol=1e-9)


def test_n8192_batch_of_32_matches_the_bordered_oracle(nib, problem):
    """BASELINE configs[3] size, n = m = 8192.  A from-scratch Cholesky per pick would take minutes on the host, so the
    oracle factors the training set once and borders it (tests/test_kb_oracle.py checks the two forms agree)."""
    n = m = 8192
    S, q = 50, 32
    Zt, y, cand, _ = problem(n, m, S, seed=8192)
    agp = nib.ActiveMaskGP(cand, alpha=1e-5, length_scale=ELL, capacity=q).fit(Zt, y)
    picks, ei = agp.select_batch(q)
    assert len(picks) == q
    _check_against_oracle(agp, picks, ei, Zt, y, cand, S, q, bordered=True)


def test_slice_count_falling_within_a_batch(nib, problem):
    """m = 1792, n = 9458, q = 16 on 148 SMs: the colreduce splits 9458 .. 9472 rows into 148 slices but 9473 into 146,
    so the partial-sum scratch must be sized for the largest count of the batch, not the last pick's."""
    n, m, q, S = 9458, 1792, 16, 50
    Zt, y, cand, _ = problem(n, m, S, seed=1792)
    agp = nib.ActiveMaskGP(cand, alpha=1e-5, length_scale=ELL, capacity=q).fit(Zt, y)
    picks, ei = agp.select_batch(q)
    assert len(picks) == q
    _check_against_oracle(agp, picks, ei, Zt, y, cand, S, q, bordered=True)


def test_batch_of_one_follows_the_sequential_loop(nib, problem):
    import BayesianOptimization as bo
    S = 50
    Zt, _, cand, rng = problem(150, 200, S, seed=3)
    w = rng.rand(S)
    score = lambda b: ogp.bits_to_matrix(np.asarray(b), S) @ w / 10.0
    y0 = score(Zt)
    _, ya, ha = bo.bayesian_optimisation_masks(8, score, Zt, y0, cand, length_scale=ELL)
    _, yb, hb = bo.bayesian_optimisation_masks(8, score, Zt, y0, cand, length_scale=ELL, batch_size=1)
    assert ha == hb and np.array_equal(ya, yb)
    seq = nib.ActiveMaskGP(cand, alpha=1e-5, length_scale=ELL, capacity=8).fit(Zt, y0)
    bat = nib.ActiveMaskGP(cand, alpha=1e-5, length_scale=ELL, capacity=8).fit(Zt, y0)
    for _ in range(8):
        mu, _, sd = seq.posterior()
        ei, arg = nib.expected_improvement_device(mu, sd, float(np.max(seq.y_host)), True)
        j = int(arg.item())
        seq.append(j, float(score(cand[j:j + 1])[0]))
        picks, eib = bat.select_batch(1)
        assert picks.tolist() == [j]
        np.testing.assert_allclose(eib[0], float(ei[j].item()), rtol=1e-9)
        bat.set_batch_values(score(cand[picks]))
    assert np.array_equal(bat.X_d[:158].cpu().numpy(), seq.X_d[:158].cpu().numpy())
    assert bat.y_host == seq.y_host


def test_selection_is_bitwise_reproducible(nib, problem):
    Zt, y, cand, _ = problem(500, 700, 50)
    q, n0 = 64, 500
    agp = nib.ActiveMaskGP(cand, alpha=1e-5, length_scale=ELL, capacity=q).fit(Zt, y)
    ssq0, alive0 = agp.ssq.clone(), agp.alive.clone()
    picks_a, ei_a = agp.select_batch(q)
    V_a, L_a = agp.V[n0:n0 + q].clone(), agp.L[n0:n0 + q, :n0 + q].clone()
    agp.ssq.copy_(ssq0)                                                # back to the state before the batch
    agp.alive.copy_(alive0)
    agp.n, agp._pending = n0, None
    picks_b, ei_b = agp.select_batch(q)
    assert np.array_equal(picks_a, picks_b) and np.array_equal(ei_a, ei_b)
    assert torch.equal(V_a, agp.V[n0:n0 + q]) and torch.equal(L_a, agp.L[n0:n0 + q, :n0 + q])


def test_capacity_is_enforced(nib, problem):
    Zt, y, cand, _ = problem(50, 80, 50)
    agp = nib.ActiveMaskGP(cand, alpha=1e-5, length_scale=ELL, capacity=5).fit(Zt, y)
    with pytest.raises(RuntimeError):
        agp.select_batch(6)
    picks, _ = agp.select_batch(5)
    with pytest.raises(RuntimeError):
        agp.select_batch(1)                                            # values of the last batch still outstanding
    agp.set_batch_values(np.zeros(len(picks)))
    with pytest.raises(RuntimeError):
        agp.select_batch(1)


def test_picking_a_duplicate_of_a_training_mask_without_jitter_raises_and_rolls_back(nib):
    """Training masks z0, z1 and candidates [far, dup(z1)], pairwise 40 bits apart so that every cross-kernel value is
    exactly 0 at l = 0.1: `far` is picked first, then `dup` (EI 0, the only one left) needs d^2 = 1 + 0 - 1 = 0."""
    Z = om.selection_bits([list(range(0, 20)), list(range(20, 40)), list(range(40, 60)), list(range(20, 40))], 64)
    agp = nib.ActiveMaskGP(Z[2:], alpha=0.0, length_scale=0.1, capacity=2).fit(Z[:2], np.array([0.9, 0.1]))
    mu0, var0, _ = agp.posterior()
    with pytest.raises(np.linalg.LinAlgError):
        agp.select_batch(2)
    mu1, var1, _ = agp.posterior()
    assert agp.n == 2 and bool(agp.alive.all()) and torch.equal(mu0, mu1) and torch.equal(var0, var1)
    picks, _ = agp.select_batch(1)
    assert picks.tolist() == [0]


def test_a_pool_smaller_than_the_batch_is_exhausted_once(nib, problem):
    Zt, y, cand, _ = problem(60, 5, 50)
    agp = nib.ActiveMaskGP(cand, alpha=1e-5, length_scale=ELL, capacity=9).fit(Zt, y)
    picks, ei = agp.select_batch(8)
    assert sorted(picks.tolist()) == list(range(5)) and len(ei) == 5 and agp.n == 65
    agp.set_batch_values(np.linspace(0.0, 1.0, 5))
    picks, ei = agp.select_batch(3)
    assert len(picks) == 0 and len(ei) == 0 and agp.n == 65


def test_bo_loop_batches_never_repeat_a_candidate(nib, problem):
    import BayesianOptimization as bo
    S = 50
    Zt, _, cand, rng = problem(120, 90, S, seed=11)
    w = rng.rand(S)
    score = lambda b: ogp.bits_to_matrix(np.asarray(b), S) @ w / 10.0
    Zg, yg, hist = bo.bayesian_optimisation_masks(4, score, Zt, score(Zt), cand, length_scale=ELL, batch_size=16)
    c = [h["candidate"] for h in hist]
    assert len(c) == 64 and len(set(c)) == 64
    assert [h["round"] for h in hist] == [r for r in range(4) for _ in range(16)]
    np.testing.assert_allclose([h["score"] for h in hist], score(cand[c]), rtol=0)
    assert np.array_equal(Zg[120:], cand[c]) and len(yg) == 120 + 64
    with pytest.raises(ValueError):
        bo.bayesian_optimisation_masks(2, score, Zt, score(Zt), cand, length_scale=None, batch_size=4)
    with pytest.raises(ValueError):
        bo.bayesian_optimisation_masks(2, score, Zt, score(Zt), cand, length_scale=ELL, refit_every=2, batch_size=4)


def test_engine_end_to_end_batches_of_16(nib):
    """ResNet-18 through PerturbationEngine, bf16 with the default tie policy: three rounds of 16 masks, each recorded
    score is the engine's score of that mask."""
    import BayesianOptimization as bo
    from network_interpretation_imagenet_b200 import synthetic
    x = synthetic.synthetic_image("imagenet")
    seg = synthetic.voronoi_labels(224, 224, 50)
    model = synthetic.build_imagenet_model("resnet18")
    eng = nib.PerturbationEngine(model, x, seg, 0, mode=nib.KEEP_MUL, precision="bf16", max_batch=64, S=50)
    assert eng.refine_ties is not None
    bits = nib.selection_bits(nib.draw_selections("subset_keep", 50, 600, seed=2), 50)
    Zt, cand = bits[:200], bits[200:]
    score = lambda b: eng.score_masks(b)["target_prob"].double().cpu().numpy()
    _, yg, hist = bo.bayesian_optimisation_masks(3, score, Zt, score(Zt), cand, length_scale=ELL, batch_size=16)
    c = [h["candidate"] for h in hist]
    assert len(c) == 48 and len(set(c)) == 48
    for h in hist:
        assert h["score"] == float(score(cand[[h["candidate"]]])[0]), h

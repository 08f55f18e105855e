"""CPU: the training-loss oracle (oracle/loss_oracle.py, SURVEY 8f rank 1 groundwork) -- certified optimal transport
and hand-checkable properties."""
import numpy as np

import loss_oracle as lo


def test_ot_emd_is_certified_optimal():
    """Primal feasible (uniform marginals), dual feasible (u_i + v_j <= c_ij) and zero duality gap: the value is THE
    optimum of the transport LP, which any exact solver (POT's network simplex included) returns."""
    rng = np.random.default_rng(0)
    for n, m in ((7, 50), (48, 50), (133, 50)):          # N_pocket range of the test sets (SURVEY 8d), K = 50 keypoints
        cost = lo.sq_dist_mat(rng.normal(0, 10, (n, 3)), rng.normal(0, 10, (m, 3)))
        val, plan, (u, v) = lo.ot_emd(cost)
        assert plan.min() >= -1e-12
        assert np.abs(plan.sum(1) - 1.0 / n).max() < 1e-12 and np.abs(plan.sum(0) - 1.0 / m).max() < 1e-12
        assert (u[:, None] + v[None, :] - cost).max() < 1e-8
        assert abs(u.sum() / n + v.sum() / m - val) < 1e-9 * max(1.0, val)
        assert (plan > 1e-14).sum() <= n + m - 1 + 1                 # a vertex of the transport polytope


def test_ot_emd_known_answers():
    # identical clouds, n == m: the identity matching costs 0
    x = np.random.default_rng(1).normal(size=(50, 3))
    assert lo.ot_emd(lo.sq_dist_mat(x, x))[0] < 1e-12
    # 2 x 2 by hand: costs [[0, 4], [4, 0]] -> 0; [[1, 2], [3, 1]] -> (1 + 1) / 2
    assert abs(lo.ot_emd(np.array([[0., 4.], [4., 0.]]))[0]) < 1e-12
    assert abs(lo.ot_emd(np.array([[1., 2.], [3., 1.]]))[0] - 1.0) < 1e-12
    # translation: every point moves by t -> cost |t|^2
    t = np.array([1.0, -2.0, 0.5])
    assert abs(lo.ot_emd(lo.sq_dist_mat(x, x + t))[0] - (t ** 2).sum()) < 1e-9


def test_intersection_loss_properties():
    rng = np.random.default_rng(2)
    lig, rec = rng.normal(0, 8, (60, 3)), rng.normal(0, 8, (75, 3))
    # far apart: G = -sigma log(1e-3) = 172.7 > surface_ct -> no penalty
    assert lo.body_intersection_loss(lig, rec + 500.0, 25.0, 10.0) == 0.0
    # overlapping bodies are penalised, symmetric in the two proteins
    a, b = lo.body_intersection_loss(lig, rec, 25.0, 10.0), lo.body_intersection_loss(rec, lig, 25.0, 10.0)
    assert a > 0 and abs(a - b) < 1e-12
    # G at a protein's own atom is below -sigma log(1e-3 + 1)
    assert (lo.G_fn(lig, lig, 25.0) <= -25.0 * np.log(1.0 + 1e-3) + 1e-12).all()


def test_batch_loss_assembly():
    rng = np.random.default_rng(3)
    B = 3
    mk = lambda n: [rng.normal(0, 10, (n, 3)) for _ in range(B)]
    pred, bound_l, bound_r = mk(40), mk(40), mk(55)
    kl, kr, pl_, pr_ = mk(50), mk(50), mk(20), mk(20)
    loss, parts = lo.batch_loss(pred, bound_l, bound_r, kl, kr, pl_, pr_)
    assert abs(loss - (parts['mse'] + 1.0 * parts['ot'] + 10.0 * parts['intersection'])) < 1e-9
    assert abs(parts['mse'] - np.mean([((p - q) ** 2).mean() for p, q in zip(pred, bound_l)])) < 1e-12

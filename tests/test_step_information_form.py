"""The gain of the product's IESKF step (information form, lv_ieskf.h) against the oracle's two 23x23 inverses.

The step solves (R P11^-1 + HTH) Z = [HTH | HTh] without pivoting and takes P11^-1 and T = P21 P11^-1 from
ieskf_prepare().  These cases stress that: a covariance streamed through many updates (correlated blocks), near-zero
extrinsic variances (P11 badly conditioned) and estimate_extrinsics off (HTH singular).  Host build, no GPU needed.
"""
import numpy as np
import pytest

import shim_binding as S


def _rows(rng, m, extrinsics):
    """m synthetic Jacobian rows of point-to-plane matches with lever arms up to 60 m, and their residuals"""
    n = rng.normal(size=(m, 3))
    n /= np.linalg.norm(n, axis=1, keepdims=True)
    p = rng.uniform(-60.0, 60.0, size=(m, 3))
    q = p + rng.uniform(-1.0, 1.0, size=(m, 3))
    H = np.zeros((m, 12))
    H[:, 0:3] = n
    H[:, 3:6] = np.cross(p, n)
    if extrinsics:
        H[:, 6:9] = np.cross(q, n)
        H[:, 9:12] = n
    h = rng.normal(scale=0.05, size=m)
    return H.T @ H, H.T @ h


def _state(O, rng):
    x0, _ = O.init_state()
    d = np.zeros(23)
    d[0:6] = rng.normal(scale=[0.05, 0.05, 0.05, 0.004, 0.004, 0.004])
    d[6:12] = rng.normal(scale=1e-3, size=6)
    d[21:23] = rng.normal(scale=1e-3, size=2)
    x_prop = x0
    x_cur = O.boxplus(x_prop, d)
    return x_prop, x_cur


def _streamed(O, prm, P, rng, n):
    """P after n exit-block updates at the propagated state"""
    x0, _ = O.init_state()
    for _ in range(n):
        HTH, HTh = _rows(rng, 2000, prm.estimate_extrinsics)
        dx, x_new, P_now, Kx, _ = O.update_step(x0, P, x0, prm, HTH, HTh)
        P = O.update_finish(x0, x_new, dx, P_now, Kx)
        P = 0.5 * (P + P.T) + 1e-6 * np.eye(23)     # the process noise a prediction would add
    return P


@pytest.mark.parametrize("case", ["P0", "streamed", "tiny_extrinsic_variance", "extrinsics_off"])
def test_step_matches_two_inverse_form(O, case):
    rng = np.random.default_rng(20261017)
    extr = case != "extrinsics_off"
    prm = O.make_params(estimate_extrinsics=extr)
    _, P = O.init_state()
    if case == "streamed":
        P = _streamed(O, prm, P, rng, 20)
    if case == "tiny_extrinsic_variance":
        P = P.copy()
        P[6:12, :] = 0.0
        P[:, 6:12] = 0.0
        P[np.arange(6, 12), np.arange(6, 12)] = 1e-9
    HTH, HTh = _rows(rng, 45000, extr)
    x_prop, x_cur = _state(O, rng)
    sp = S.make_params(prm)
    for it in range(prm.max_num_iters):     # the last one runs the exit block and returns P
        dx_o, x_o, P_now, Kx, _ = O.update_step(x_prop, P, x_cur, prm, HTH, HTh)
        st, dx_s, x_s, P_s, done = S.step(x_prop, P, x_cur, sp, HTH, HTh, 45000, it, 0)
        assert st == 0
        assert np.abs(dx_s - dx_o).max() < 1e-9, (case, it, np.abs(dx_s - dx_o).max())
        assert np.abs(x_s - x_o).max() < 1e-9, (case, it)
        assert done == (it == prm.max_num_iters - 1)
        if done:
            P_o = O.update_finish(x_prop, x_o, dx_o, P_now, Kx)
            assert np.abs(P_s - P_o).max() < 1e-8 * np.abs(P_o).max(), (case, np.abs(P_s - P_o).max())

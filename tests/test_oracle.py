"""The CPU oracle pinned against what can be pinned here (SURVEY.md 8c):

* its exact kNN and its Add_Points restatement against the reference's OWN ikd-Tree (its answers are stored
  under tests/golden/reference, see tests/reference_golden.py);
* its small dense algebra (LU inverse, symmetric 6x6 eigen, 5x3 least squares) against numpy/LAPACK;
* its IESKF step against an independent numpy statement of esekfom.hpp:1722-1733;
* manifold identities of the MTK restatement.
The reference ships no golden vectors for this path; Eigen's bit-level summation order is not
reproducible without Eigen ("parity unpinned" for that part, see oracle/lv_oracle.h).
"""
import numpy as np
import pytest

import reference_golden as RG


def _cloud(seed, m, span=20.0):
    rng = np.random.default_rng(seed)
    a = np.c_[rng.uniform(-span, span, m), rng.uniform(-span, span, m), rng.normal(0, 0.02, m)]
    b = np.c_[rng.uniform(-span, span, m // 4), np.full(m // 4, 5.0) + rng.normal(0, 0.02, m // 4),
              rng.uniform(0, 6, m // 4)]
    return np.vstack([a, b]).astype(np.float32)


def _knn_case():
    pts = _cloud(1, 20000)
    rng = np.random.default_rng(2)
    q = (pts[rng.integers(0, len(pts), 300)] + rng.normal(0, 0.1, (300, 3))).astype(np.float32)
    return pts, q


def _add_case():
    base = _cloud(3, 8000, span=6.0)
    rng = np.random.default_rng(4)
    new = (base[rng.integers(0, len(base), 3000)] + rng.normal(0, 0.05, (3000, 3))).astype(np.float32)
    new2 = (new[:1500] + np.float32([0.03, -0.02, 0.01])).astype(np.float32)
    return base, new, new2


def test_knn_backends_agree(O):
    pts, q = _knn_case()
    golden = RG.load()
    maps = {}
    for name, be in (("brute", O.KNN_BRUTE), ("kd", O.KNN_KDTREE)):
        maps[name] = O.Map(be)
        maps[name].build(pts)
    for i in range(len(q)):
        fb, ib, db, nb = maps["brute"].knn(q[i])
        fk, ik, dk, nk = maps["kd"].knn(q[i])
        assert fb == fk == 5
        assert (ib == ik).all() and (db == dk).all()
        assert (np.diff(db) >= 0).all()                       # ascending (ikd_Tree.cpp:452-459)
        # squared distance exactly as calc_dist evaluates it (ikd_Tree.cpp:1682-1687)
        d = q[i] - pts[ib]
        ref = (d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2]
        assert (ref.astype(np.float32) == db).all()
        # the reference ikd-Tree's answer
        assert golden["knn_found"][i] == 5 and (golden["knn_sqd"][i] == db).all() and (golden["knn_xyz"][i] == nb).all()


def test_knn_fewer_points_than_k(O):
    m = O.Map(O.KNN_KDTREE)
    m.build(np.float32([[0, 0, 0], [1, 0, 0], [0, 1, 0]]))
    found, idx, sqd, nn = m.knn(np.float32([0.1, 0.1, 0]))
    assert found == 3 and (idx[:3] == [0, 1, 2]).all() or found == 3


def test_map_add_matches_reference_ikdtree(O):
    """Add_Points with the 0.2 m voxel rule (ikd_Tree.cpp:478-573): oracle restatement vs the real thing."""
    golden = RG.load()
    base, new, new2 = _add_case()
    a = O.Map(O.KNN_KDTREE)
    a.build(base)
    a.add(new, downsample=True)
    sa = set(map(tuple, a.points().tolist()))
    # KD_TREE::size() counts lazily deleted nodes too (ikd_Tree.cpp size() = Root_Node->TreeSize), so
    # the CONTENT is compared through flatten (ikd_Tree.cpp:1626-1657), not through size()
    assert a.size() == len(sa) == golden["add_count"][0] and golden["add_tree_size"] >= len(sa)
    assert RG.set_digest(a.points()) == golden["add_digest"][0]
    # a second batch on top (touched voxels collapse to one point)
    a.add(new2, downsample=True)
    assert RG.set_digest(a.points()) == golden["add_digest"][1]
    # without downsampling everything is kept
    a.add(new2, downsample=False)
    assert len(a.points()) == golden["add_count"][1]


def test_dense_algebra_against_lapack(O):
    rng = np.random.default_rng(5)
    for n in (6, 12, 23):
        A = rng.normal(size=(n, n))
        A = A @ A.T + np.eye(n) * 0.5
        assert np.abs(O.inverse(A) - np.linalg.inv(A)).max() < 1e-9 * np.abs(np.linalg.inv(A)).max()
    B = rng.normal(size=(6, 6))
    B = B @ B.T
    ev, V = O.sym_eig6(B)
    assert np.abs(ev - np.linalg.eigvalsh(B)).max() < 1e-10 * np.abs(ev).max()
    assert np.abs(B @ V - V * ev).max() < 1e-10 * np.abs(ev).max()
    assert (np.diff(ev) >= 0).all()


def test_plane_fit_is_least_squares(O):
    """estimate_plane solves A n = -1 in the least-squares sense (Utils.cpp:32-57) and normalises."""
    rng = np.random.default_rng(6)
    for _ in range(200):
        n = rng.normal(size=3)
        n /= np.linalg.norm(n)
        d = rng.uniform(1.0, 30.0)
        basis = np.linalg.svd(n[None])[2][1:]
        pts = (-d * n + (rng.uniform(-0.3, 0.3, (5, 2)) @ basis) + rng.normal(0, 0.005, (5, 3))).astype(np.float32)
        abcd, ok = O.plane_fit(pts, 0.05)
        sol = np.linalg.lstsq(pts.astype(np.float64), -np.ones(5), rcond=None)[0]
        ref = np.r_[sol / np.linalg.norm(sol), 1.0 / np.linalg.norm(sol)]
        assert np.abs(abcd - ref).max() < 2e-3 * max(1.0, abs(ref[3]))     # fp32 QR vs fp64 SVD
        assert abs(np.linalg.norm(abcd[:3]) - 1) < 1e-5
        res = np.abs(pts @ abcd[:3] + abcd[3])
        assert ok == bool((res <= 0.05).all())
    # is_plane rejects (Utils.cpp:59-66)
    bad = np.float32([[0, 0, 1], [1, 0, 1], [0, 1, 1], [1, 1, 1.5], [0.5, 0.5, 0.4]])
    assert not O.plane_fit(bad, 0.05)[1]


def test_manifold_identities(O):
    rng = np.random.default_rng(7)
    x0, _ = O.init_state(I_Rotation_L=(1, 0, 0, 0, -1, 0, 0, 0, -1), I_Translation_L=(1.25, 0, 0))
    assert abs(np.linalg.norm(x0[23:26]) - 9.809) < 1e-12               # S2 length (use-ikfom.hpp:8)
    for _ in range(50):
        d = rng.normal(0, 0.05, 23)
        x = O.boxplus(x0, d)
        back = O.boxminus(x, x0)
        assert np.abs(back - d).max() < 1e-9                            # (x [+] d) [-] x = d
        assert abs(np.linalg.norm(x[3:7]) - 1) < 1e-12 and abs(np.linalg.norm(x[7:11]) - 1) < 1e-12
        assert abs(np.linalg.norm(x[23:26]) - 9.809) < 1e-9
    R = O.quat_to_rot(x[3:7])
    assert np.abs(R @ R.T - np.eye(3)).max() < 1e-12 and abs(np.linalg.det(R) - 1) < 1e-12
    assert np.abs(O.boxminus(x0, x0)).max() == 0


def test_ieskf_step_against_numpy_statement(O, lv, scene_xaloc):
    """dx_ = K_h + (K_x - I) J dx with the gains of esekfom.hpp:1722-1729, restated with numpy.linalg."""
    sc = scene_xaloc
    om = O.Map(O.KNN_KDTREE)
    om.build(sc.map)
    st, HTH, HTh, nm = om.measure_reduced(sc.x_prop, sc.oprm, sc.sweep)
    assert st == 0 and nm > 1000
    # first evaluation: x == x_prop, so dx = 0 and P_ = P_prop
    dx, x_new, P_now, Kx, conv = O.update_step(sc.x_prop, sc.P0, sc.x_prop, sc.oprm, HTH, HTh)
    R = sc.prm.LiDAR_noise
    T = np.linalg.inv(sc.P0 / R)
    T[:12, :12] += HTH
    Pinv = np.linalg.inv(T)
    assert np.abs(dx - Pinv[:, :12] @ HTh).max() < 1e-9
    assert np.abs(Kx - Pinv[:, :12] @ HTH).max() < 1e-7
    assert np.abs(P_now - sc.P0).max() < 1e-12      # J blocks are identity up to the S2 Nx*Mx product (1 ulp)
    assert np.abs(O.boxminus(x_new, sc.x_prop) - dx).max() < 1e-9       # non-degenerate scene: no masking
    # covariance of the exit block with dx_ small: P = (I - K_x H) P up to the J blocks
    P_out = O.update_finish(sc.x_prop, x_new, dx, P_now, Kx)
    approx = sc.P0 - Kx @ sc.P0[:12, :]
    assert np.abs(P_out - approx).max() < 5e-3 * np.abs(approx).max()
    assert np.abs(P_out - P_out.T).max() < 1e-6 * np.abs(P_out).max()


def test_oracle_update_converges_to_truth(O, scene_xaloc):
    sc = scene_xaloc
    om = O.Map(O.KNN_KDTREE)
    om.build(sc.map)
    st, x, P, logs = om.update_iterated(sc.x_prop, sc.P0, sc.oprm, sc.sweep)
    assert st == 0 and 2 <= len(logs) <= sc.prm.MAX_NUM_ITERS + 1           # esekfom.hpp:1634,1764
    e0 = np.abs(O.boxminus(sc.x_prop, sc.truth))[:6]
    e1 = np.abs(O.boxminus(x, sc.truth))[:6]
    assert e1[:3].max() < 0.2 * e0[:3].max() and e1[3:6].max() < 0.2 * e0[3:6].max()
    assert all(l["n_matches"] > 0.5 * len(sc.sweep) for l in logs)
    # empty map / too few matches
    empty = O.Map(O.KNN_KDTREE)
    assert empty.update_iterated(sc.x_prop, sc.P0, sc.oprm, sc.sweep)[0] == O.EMPTY_MAP
    assert om.update_iterated(sc.x_prop, sc.P0, sc.oprm, sc.sweep[:10])[0] == O.TOO_FEW_MATCHES


def test_oracle_openmp_team_matches_single_thread(O, scene_xaloc):
    """Mapper::match runs under OpenMP (Mapper.cpp:45-46); sums are order-insensitive to ~1e-12."""
    sc = scene_xaloc
    om = O.Map(O.KNN_KDTREE)
    om.build(sc.map)
    O.set_threads(1)
    _, H1, h1, n1 = om.measure_reduced(sc.x_prop, sc.oprm, sc.sweep)
    O.set_threads(3)
    _, H3, h3, n3 = om.measure_reduced(sc.x_prop, sc.oprm, sc.sweep)
    O.set_threads(1)
    assert n1 == n3 and np.abs(H1 - H3).max() <= 1e-12 * np.abs(H1).max()


def test_predict_restatement_properties(O, lv):
    """esekf::predict (esekfom.hpp:279-384): oracle vs the product's host implementation + invariants."""
    prm = lv.params_from_yaml(lv.CONFIG_DIR + "/xaloc.yaml")
    x0, P0 = lv.init_state_host(prm)
    xo, Po = O.init_state(initial_gravity=prm.initial_gravity[:], I_Rotation_L=prm.I_Rotation_L[:],
                          I_Translation_L=prm.I_Translation_L[:])
    assert np.abs(x0 - xo).max() == 0 and np.abs(P0 - Po).max() == 0       # Localizator.cpp:135-153
    rng = np.random.default_rng(8)
    x, P = x0.copy(), P0.copy()
    x[14:17] = [3.0, 0.2, -0.1]
    x[17:20] = [0.01, -0.02, 0.005]
    x[20:23] = [0.05, 0.02, -0.03]
    xa, Pa = x.copy(), P.copy()
    for _ in range(20):
        acc = np.array([0.3, -0.2, 9.7]) + rng.normal(0, 0.05, 3)
        gyr = np.array([0.01, -0.02, 0.3]) + rng.normal(0, 0.01, 3)
        x, P = lv.predict_host(prm, x, P, acc, gyr, 0.0025)
        xa, Pa = O.predict(xa, Pa, acc, gyr, 0.0025, prm.covariance_gyroscope, prm.covariance_acceleration,
                           prm.covariance_bias_gyroscope, prm.covariance_bias_acceleration)
    assert np.abs(x - xa).max() < 1e-12 and np.abs(P - Pa).max() < 1e-12 * np.abs(Pa).max()
    assert np.abs(P - P.T).max() < 1e-12 and np.linalg.eigvalsh(P).min() > 0
    assert abs(np.linalg.norm(x[3:7]) - 1) < 1e-12
    assert np.abs(x[7:14] - x0[7:14]).max() == 0 and np.abs(x[23:26] - x0[23:26]).max() == 0   # f = 0 there

"""GPU parity: the CUDA path (through the C ABI) against the CPU oracle on identical inputs.

Tolerances (SURVEY.md 8c): the fp32 stage (world point, neighbour ids/distances, plane, residual,
accept decision) must be BIT-EXACT; the fp64 rows of H are bit-exact; reduced sums HTH/HTh agree to
1e-12 relative (different summation order); per-evaluation dx_ to 1e-9 abs; final state 1e-9.
"""
import numpy as np
import pytest

import reference_golden as RG
from conftest import Scene

pytestmark = pytest.mark.gpu


def _oracle_map(O, scene, backend=None):
    om = O.Map(O.KNN_KDTREE if backend is None else backend)
    om.build(scene.map)
    return om


@pytest.mark.parametrize("name", ["scene_xaloc", "scene_kitti", "scene_ouster"])
def test_match_all_bit_exact(lv, O, name, request):
    sc = request.getfixturevalue(name)
    loc = lv.Localizer(sc.prm)
    loc.map_build(sc.map)
    got = loc.match_all(sc.x_prop, sc.sweep)
    ref = _oracle_map(O, sc).match_all(sc.x_prop, sc.oprm, sc.sweep)
    assert (got["g"] == ref["g"]).all()
    inside = np.isfinite(got["nn_sqd"][:, 4])
    # everything the gate can accept was searched exhaustively
    assert not ((ref["nn_sqd"][~inside, 4].astype(np.float64)) < sc.prm.MAX_DIST_PLANE ** 2).any()
    assert (got["nn_idx"][inside] == ref["nn_idx"][inside]).all()
    assert (got["nn_sqd"][inside] == ref["nn_sqd"][inside]).all()
    assert (got["valid"] == ref["valid"]).all()
    assert (got["plane"] == ref["plane"]).all()
    assert (got["dist"] == ref["dist"]).all()
    assert got["valid"].sum() > 0.8 * len(sc.sweep)
    loc.close()


def test_match_against_reference_ikdtree(lv, O, scene_xaloc):
    """neighbour distances/coordinates equal those of the reference's own ikd-Tree (stored as digests, see
    tests/reference_golden.py: the oracle reproduces them bit for bit and stands in for the reference below)"""
    sc = scene_xaloc
    golden = RG.load()
    RG.check_scene(golden, sc)
    ref = _oracle_map(O, sc).match_all(sc.x_prop, sc.oprm, sc.sweep)
    assert [RG.digest(ref[k]) for k in RG.MATCH_FIELDS] == golden["xaloc_match"].tolist()
    loc = lv.Localizer(sc.prm)
    loc.map_build(sc.map)
    got = loc.match_all(sc.x_prop, sc.sweep)
    inside = np.isfinite(got["nn_sqd"][:, 4])
    assert (got["nn_sqd"][inside] == ref["nn_sqd"][inside]).all()
    assert (got["valid"] == ref["valid"]).all()
    assert (got["plane"] == ref["plane"]).all()
    loc.close()


@pytest.mark.parametrize("name", ["scene_xaloc", "scene_kitti"])
def test_measure_rows_and_reduction(lv, O, name, request):
    sc = request.getfixturevalue(name)
    loc = lv.Localizer(sc.prm)
    loc.map_build(sc.map)
    om = _oracle_map(O, sc)
    st, hx, h = loc.measure(sc.x_prop, sc.sweep)
    st_o, hx_o, h_o = om.measure(sc.x_prop, sc.oprm, sc.sweep)
    assert st == st_o == 0 and hx.shape == hx_o.shape
    assert (hx == hx_o).all() and (h == h_o).all()          # h_share_model, row for row
    if not sc.prm.estimate_extrinsics:
        assert (hx[:, 6:] == 0).all()                       # Localizator.cpp:52
    st, HTH, HTh, nm = loc.measure_reduced(sc.x_prop, sc.sweep)
    st_o, HTH_o, HTh_o, nm_o = om.measure_reduced(sc.x_prop, sc.oprm, sc.sweep)
    assert nm == nm_o == hx.shape[0]
    assert np.abs(HTH - HTH_o).max() <= 1e-12 * np.abs(HTH_o).max()
    assert np.abs(HTh - HTh_o).max() <= 1e-12 * max(1.0, np.abs(HTh_o).max())
    assert np.abs(HTH - hx.T @ hx).max() <= 1e-11 * np.abs(HTH).max()
    loc.close()


@pytest.mark.parametrize("name", ["scene_xaloc", "scene_kitti", "scene_ouster"])
def test_correct_matches_oracle(lv, O, name, request):
    sc = request.getfixturevalue(name)
    loc = lv.Localizer(sc.prm)
    loc.map_build(sc.map)
    loc.set_state(sc.x_prop, sc.P0)
    st, x, P, logs = loc.correct(sc.sweep, time=1.5)
    st_o, x_o, P_o, logs_o = _oracle_map(O, sc).update_iterated(sc.x_prop, sc.P0, sc.oprm, sc.sweep)
    assert st == st_o == 0
    assert len(logs) == len(logs_o)
    for a, b in zip(logs, logs_o):
        assert a["n_matches"] == b["n_matches"]
        assert a["converged"] == b["converged"]
        assert np.abs(a["HTH"] - b["HTH"]).max() <= 1e-11 * np.abs(b["HTH"]).max()
        assert np.abs(a["dx"] - b["dx"]).max() < 1e-9
        assert np.abs(a["x_after"] - b["x_after"]).max() < 1e-9
    assert np.abs(x - x_o).max() < 1e-9
    assert np.abs(P - P_o).max() < 1e-8 * np.abs(P_o).max()
    x2, P2 = loc.get_state()
    assert (x2 == x).all() and (P2 == P).all()
    # the update pulls the pose towards the truth
    assert np.abs(O.boxminus(x, sc.truth))[:3].max() < 0.3 * np.abs(O.boxminus(sc.x_prop, sc.truth))[:3].max() + 2e-3
    loc.close()


def test_correct_device_resident_equals_host_call(lv, O, scene_xaloc):
    sc = scene_xaloc
    loc = lv.Localizer(sc.prm)
    loc.map_build(sc.map)
    loc.set_state(sc.x_prop, sc.P0)
    st, x, P, logs = loc.correct(sc.sweep)
    d = loc.upload(sc.sweep)
    loc.set_state(sc.x_prop, sc.P0)
    loc.correct_device(d, len(sc.sweep))
    st2, logs2 = loc.last_logs()
    x2, P2 = loc.get_state()
    assert (x2 == x).all() and (P2 == P).all() and len(logs2) == len(logs)   # deterministic
    loc.device_free(d)
    loc.close()


def test_edge_cases(lv, O, scene_xaloc):
    sc = scene_xaloc
    loc = lv.Localizer(sc.prm)
    # empty map: Localizator.cpp:24 / Mapper.cpp:42
    st, x, P, logs = loc.correct(sc.sweep)
    assert st == lv.EMPTY_MAP and logs == []
    assert loc.measure_reduced(sc.x_prop, sc.sweep)[0] == lv.EMPTY_MAP
    loc.map_build(sc.map)
    om = _oracle_map(O, sc)
    # ragged sizes (not multiples of the 128-point tile), single point
    for n in (1, 5, 127, 129, 1000):
        sub = sc.sweep[:n]
        st, HTH, HTh, nm = loc.measure_reduced(sc.x_prop, sub)
        st_o, HTH_o, HTh_o, nm_o = om.measure_reduced(sc.x_prop, sc.oprm, sub)
        assert nm == nm_o
        assert np.abs(HTH - HTH_o).max() <= 1e-12 * max(1e-30, np.abs(HTH_o).max())
    # fewer than 23 matches: LV_TOO_FEW_MATCHES (esekfom.hpp:1701-1709), state left at x_prop
    loc.set_state(sc.x_prop, sc.P0)
    st, x, P, logs = loc.correct(sc.sweep[:10])
    assert st == lv.TOO_FEW_MATCHES
    assert (x == sc.x_prop).all() and (P == sc.P0).all()
    # points with no map nearby: nothing accepted
    far = sc.sweep[:256] + np.float32([0, 0, 500.0])
    got = loc.match_all(sc.x_prop, far)
    assert got["valid"].sum() == 0 and (got["nn_idx"] == -1).all()
    # capacity
    big = np.zeros((sc.prm.max_points + 1, 3), np.float32)
    with pytest.raises(RuntimeError):
        loc.correct(big)
    loc.close()


def test_degenerate_planar_map(lv, O):
    """BASELINE cfg0 shape: purely planar map -> x, y, yaw unobservable; the degenerate branch
    (esekfom.hpp:1736-1744) must agree with the oracle's restatement of it."""
    sc = Scene(lv, O, "xaloc.yaml", seed=5, m=60000, rings=16, azimuths=256, max_map_points=1 << 18, max_points=1 << 15,
               degeneracy_threshold=2000.0)   # plane-fit noise alone lifts the x/y/yaw eigenvalues above 5
    ground = sc.map[sc.map[:, 2] < -1.6]
    sweep = sc.sweep[(sc.sweep @ np.array([0, 0, 1.0], np.float32)) > 0.5]   # xaloc LiDAR is mounted upside down
    loc = lv.Localizer(sc.prm)
    loc.map_build(ground)
    om = O.Map(O.KNN_KDTREE)
    om.build(ground)
    loc.set_state(sc.x_prop, sc.P0)
    st, x, P, logs = loc.correct(sweep)
    st_o, x_o, P_o, logs_o = om.update_iterated(sc.x_prop, sc.P0, sc.oprm, sweep)
    assert st == st_o == 0 and len(logs) == len(logs_o)
    assert any(l["degenerate"] for l in logs)
    for a, b in zip(logs, logs_o):
        assert a["n_matches"] == b["n_matches"]
        assert np.abs(a["dx"] - b["dx"]).max() < 1e-7
    assert np.abs(x - x_o).max() < 1e-7
    loc.close()


def test_map_build_roundtrip_and_add(lv, O, scene_xaloc):
    sc = scene_xaloc
    loc = lv.Localizer(sc.prm)
    loc.map_build(sc.map)
    assert loc.map_size() == len(sc.map)
    assert (loc.map_points() == sc.map).all()
    # Mapper::add with the 0.2 m voxel rule vs the oracle restatement (and the reference ikd-Tree)
    R = O.quat_to_rot(sc.truth[3:7]); RL = O.quat_to_rot(sc.truth[7:11])
    new = ((sc.sweep.astype(np.float64) @ RL.T + sc.truth[11:14]) @ R.T + sc.truth[0:3]).astype(np.float32)
    loc.map_add(new, downsample=True)
    got = loc.map_points()
    got_set = set(map(tuple, got.tolist()))
    assert len(got_set) == len(got)
    om = O.Map(O.KNN_KDTREE)
    om.build(sc.map)
    om.add(new, downsample=True)
    golden = RG.load()
    RG.check_scene(golden, sc)
    assert RG.set_digest(om.points()) == golden["xaloc_add"]         # the oracle holds what the reference ikd-Tree holds
    ref_set = set(map(tuple, om.points().tolist()))
    diff = len(got_set ^ ref_set)
    assert diff <= 1e-4 * len(ref_set), (diff, len(got_set), len(ref_set))
    # the rebuilt structure serves queries: parity after the add
    om = O.Map(O.KNN_KDTREE)
    om.build(got)
    g = loc.match_all(sc.x_prop, sc.sweep)
    r = om.match_all(sc.x_prop, sc.oprm, sc.sweep)
    assert (g["valid"] == r["valid"]).all() and (g["plane"] == r["plane"]).all()
    loc.close()


def test_tick_on_the_device_equals_the_host_path(lv, O, scene_xaloc):
    """main.cpp:84-105 without leaving the GPU: lv_correct + lv_map_add_last_sweep (the sweep is transformed by the update's own
    result on the device and merged under the 0.2 m rule) must leave exactly the map that the host path leaves
    (read the state back, transform in fp32 like State * RotTransl * point, lv_map_add)."""
    sc = scene_xaloc
    om = _oracle_map(O, sc)
    a, b = lv.Localizer(sc.prm), lv.Localizer(sc.prm)
    for loc in (a, b):
        loc.map_build(sc.map)
    x = sc.x_prop.copy()
    for k in range(2):
        for loc in (a, b):
            loc.set_state(x, sc.P0)
        st, xa, Pa, _ = a.correct(sc.sweep)
        st, xb, Pb, _ = b.correct(sc.sweep)
        assert (xa == xb).all()
        g = om.match_all(xa, sc.oprm, sc.sweep)["g"]              # fp32 world points of Mapper::match == main.cpp:101's
        a.map_add(g, downsample=True)
        b.map_add_last_sweep(downsample=True)
        a.map_status(); b.map_status()
        assert a.map_size() == b.map_size() > len(sc.map)
        assert sorted(map(tuple, a.map_points().tolist())) == sorted(map(tuple, b.map_points().tolist()))
        x = xa.copy()
        x[0] += 0.3                                                  # the next tick starts somewhere else
    # and the device variant with an explicit buffer
    d = b.upload(sc.sweep)
    b.map_add_sweep_device(d, len(sc.sweep), downsample=True)
    a.map_add(om.match_all(b.get_state()[0], sc.oprm, sc.sweep)["g"], downsample=True)
    assert sorted(map(tuple, a.map_points().tolist())) == sorted(map(tuple, b.map_points().tolist()))
    b.device_free(d)
    a.close(); b.close()


def test_propagate_on_the_device_equals_the_host_predict(lv, O, scene_xaloc):
    """esekf::predict (esekfom.hpp:279-384) for a run of IMU samples: one device launch (lv_propagate_device) against the host
    loop over lv_predict; then update -> propagate -> update with the state never leaving the GPU equals the host-driven
    sequence."""
    sc = scene_xaloc
    rng = np.random.default_rng(2)
    k = 37
    acc = np.array([0.2, -0.1, 9.8]) + rng.normal(0, 0.05, (k, 3))
    gyro = np.array([0.01, -0.02, 0.2]) + rng.normal(0, 0.01, (k, 3))
    dt = np.full(k, 0.0025) + rng.uniform(0, 1e-4, k)
    a, b = lv.Localizer(sc.prm), lv.Localizer(sc.prm)
    for loc in (a, b):
        loc.map_build(sc.map)
        loc.set_state(sc.x_prop, sc.P0)
    for i in range(k):
        a.predict(acc[i], gyro[i], dt[i])
    b.propagate_device(acc, gyro, dt)
    xa, Pa = a.get_state()
    xb, Pb = b.get_state()
    assert np.abs(xa - xb).max() < 1e-12 and np.abs(Pa - Pb).max() <= 1e-12 * np.abs(Pa).max()
    # a tick: correct, add the sweep, propagate, correct again
    for loc in (a, b):
        loc.set_state(sc.x_prop, sc.P0)
    sta, xa, Pa, la = a.correct(sc.sweep)
    for i in range(8):
        a.predict(acc[i], gyro[i], 1e-3)
    sta, xa, Pa, la = a.correct(sc.sweep)
    b.correct_device(b.upload(sc.sweep), len(sc.sweep))
    b.propagate_device(acc[:8], gyro[:8], np.full(8, 1e-3))
    stb, xb, Pb, lb = b.correct(sc.sweep)
    assert sta == stb == 0 and len(la) == len(lb)
    assert np.abs(xa - xb).max() < 1e-9 and np.abs(Pa - Pb).max() <= 1e-8 * np.abs(Pa).max()
    a.close(); b.close()

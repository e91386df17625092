"""Host build of the product's device headers (tests/cpu_shim) against the oracle — no GPU needed.

The kernels of liblimovelo_b200.so are thin wrappers around host+device headers
(limo-velo_b200/csrc/lv_voxel_search.h, lv_point_math.h, lv_ieskf.h).  tests/cpu_shim instantiates the
same code serially, so the arithmetic the GPU runs is checked here with the same bars as the GPU
parity tests: bit-exact fp32 stage, 1e-12 reductions, 1e-9 state.
"""
import numpy as np
import pytest

import reference_golden as RG
import shim_binding as S
from conftest import Scene


def _check_match(O, sc, cell):
    om = O.Map(O.KNN_KDTREE)
    om.build(sc.map)
    ref = om.match_all(sc.x_prop, sc.oprm, sc.sweep)
    sm = S.ShimMap(sc.map, cell, sc.prm.MAX_DIST_PLANE)
    got = sm.match_all(sc.x_prop, S.make_params(sc.oprm, cell), sc.sweep)
    assert (got["g"] == ref["g"]).all()
    inside = np.isfinite(got["nn_sqd"][:, 4])
    assert not (ref["nn_sqd"][~inside, 4].astype(np.float64) < sc.prm.MAX_DIST_PLANE ** 2).any()
    assert (got["nn_idx"][inside] == ref["nn_idx"][inside]).all()
    assert (got["nn_sqd"][inside] == ref["nn_sqd"][inside]).all()
    assert (got["valid"] == ref["valid"]).all()
    assert (got["plane"] == ref["plane"]).all() and (got["dist"] == ref["dist"]).all()
    st, hx, h = om.measure(sc.x_prop, sc.oprm, sc.sweep)
    rows = got["rows"][got["valid"] == 1]
    assert (rows[:, :12] == hx).all() and (rows[:, 12] == h).all()
    return got


@pytest.mark.parametrize("name", ["scene_xaloc", "scene_kitti", "scene_ouster"])
@pytest.mark.parametrize("cell", [0.5, 0.3, 1.0])
def test_search_fit_row_bit_exact(O, name, cell, request):
    """voxel pyramid search (1..4 levels depending on the edge), plane fit, Jacobian row"""
    got = _check_match(O, request.getfixturevalue(name), cell)
    assert got["valid"].mean() > 0.7


def test_sparse_and_far_queries(O, scene_xaloc):
    """queries level 0 cannot settle: shifted off the surfaces, beyond the search radius, huge coordinates"""
    sc = scene_xaloc
    om = O.Map(O.KNN_KDTREE)
    om.build(sc.map)
    sm = S.ShimMap(sc.map, 0.5, 2.0)
    prm = S.make_params(sc.oprm)
    for shift in ([0, 0, 0.7], [0, 0, 1.6], [0, 0, -1.9], [0.4, 0.4, 0.4], [0, 0, 40.0], [3e5, -2e5, 10.0]):
        q = sc.sweep[:3000] + np.float32(shift)
        ref = om.match_all(sc.x_prop, sc.oprm, q)
        got = sm.match_all(sc.x_prop, prm, q)
        inside = np.isfinite(got["nn_sqd"][:, 4])
        assert not (ref["nn_sqd"][~inside, 4].astype(np.float64) < 4.0).any()
        assert (got["nn_idx"][inside] == ref["nn_idx"][inside]).all()
        assert (got["nn_sqd"][inside] == ref["nn_sqd"][inside]).all()
        assert (got["valid"] == ref["valid"]).all() and (got["plane"] == ref["plane"]).all()


def test_tiny_and_clustered_maps(O, scene_xaloc):
    sc = scene_xaloc
    prm = S.make_params(sc.oprm)
    rng = np.random.default_rng(3)
    # fewer map points than neighbours, one voxel holding hundreds of points, duplicates
    cases = [sc.map[:3], sc.map[:7],
             (np.float32([5, 1, -1.8]) + rng.normal(0, 0.05, (600, 3))).astype(np.float32),
             np.repeat(sc.map[:50], 3, axis=0)]
    for mp in cases:
        om = O.Map(O.KNN_KDTREE)
        om.build(mp)
        sm = S.ShimMap(mp, 0.5, 2.0)
        q = (mp[rng.integers(0, len(mp), 200)] + rng.normal(0, 0.1, (200, 3))).astype(np.float32)
        x = sc.x0.copy()                       # identity pose: queries are given in the world frame
        x[7:11] = [0, 0, 0, 1]
        x[11:14] = 0
        ref = om.match_all(x, sc.oprm, q)
        got = sm.match_all(x, prm, q)
        inside = np.isfinite(got["nn_sqd"][:, 4])
        assert not (ref["nn_sqd"][~inside, 4].astype(np.float64) < 4.0).any()
        assert (got["nn_sqd"][inside] == ref["nn_sqd"][inside]).all()
        assert (got["valid"] == ref["valid"]).all() and (got["plane"] == ref["plane"]).all()


@pytest.mark.parametrize("name", ["scene_xaloc", "scene_kitti", "scene_ouster"])
def test_update_matches_oracle(O, name, request):
    sc = request.getfixturevalue(name)
    om = O.Map(O.KNN_KDTREE)
    om.build(sc.map)
    so, xo, Po, lo = om.update_iterated(sc.x_prop, sc.P0, sc.oprm, sc.sweep)
    sm = S.ShimMap(sc.map, 0.5, sc.prm.MAX_DIST_PLANE)
    ss, xs, Ps, ls = sm.update(sc.x_prop, sc.P0, S.make_params(sc.oprm), sc.sweep)
    assert so == ss == 0 and len(lo) == len(ls)
    for a, b in zip(lo, ls):
        assert a["n_matches"] == b["n_matches"] and a["converged"] == b["converged"]
        assert np.abs(a["HTH"] - b["HTH"]).max() <= 1e-12 * np.abs(a["HTH"]).max()
        assert np.abs(a["dx"] - b["dx"]).max() < 1e-9        # structured 12x12 gain solve vs two 23x23 inverses
        assert np.abs(a["x_after"] - b["x_after"]).max() < 1e-9
    assert np.abs(xo - xs).max() < 1e-9
    assert np.abs(Po - Ps).max() < 1e-8 * np.abs(Po).max()


def test_degenerate_and_too_few(O):
    """planar map (x, y, yaw unobservable) -> degenerate branch esekfom.hpp:1736-1744; Nm < 23 -> status 2"""
    import __graft_entry__ as G
    lv = G.load_package()
    sc = Scene(lv, O, "xaloc.yaml", seed=5, m=60000, rings=16, azimuths=256, degeneracy_threshold=2000.0)
    ground = sc.map[sc.map[:, 2] < -1.6]
    sweep = sc.sweep[sc.sweep[:, 2] > 0.5]
    om = O.Map(O.KNN_KDTREE)
    om.build(ground)
    sm = S.ShimMap(ground, 0.5, 2.0)
    so, xo, Po, lo = om.update_iterated(sc.x_prop, sc.P0, sc.oprm, sweep)
    ss, xs, Ps, ls = sm.update(sc.x_prop, sc.P0, S.make_params(sc.oprm), sweep)
    assert so == ss == 0 and all(l["degenerate"] for l in ls)
    for a, b in zip(lo, ls):
        assert a["n_matches"] == b["n_matches"] and np.abs(a["dx"] - b["dx"]).max() < 1e-8
    ss, xs, Ps, ls = sm.update(sc.x_prop, sc.P0, S.make_params(sc.oprm), sweep[:10])
    assert ss == 2 and (xs == sc.x_prop).all() and (Ps == sc.P0).all()


def test_manifold_and_plane_helpers_match_oracle(O):
    rng = np.random.default_rng(11)
    x0, _ = O.init_state(I_Rotation_L=(1, 0, 0, 0, -1, 0, 0, 0, -1), I_Translation_L=(1.25, 0, 0))
    for _ in range(100):
        d = rng.normal(0, 0.1, 23)
        xa, xb = O.boxplus(x0, d), S.boxplus(x0, d)
        assert np.abs(xa - xb).max() < 1e-14
        assert np.abs(O.boxminus(xa, x0) - S.boxminus(xb, x0)).max() < 1e-14
        pts = (rng.normal(0, 1, 3) + rng.normal(0, 0.2, (5, 3))).astype(np.float32)
        pa, oka = O.plane_fit(pts, 0.05)
        pb, okb = S.plane_fit(pts, 0.05)
        assert (pa == pb).all() and oka == okb
    # rank-deficient neighbour sets (collinear / repeated points) take the same path in both
    for pts in (np.float32([[0, 0, 1], [1, 0, 1], [2, 0, 1], [3, 0, 1], [4, 0, 1]]),
                np.float32([[1, 1, 1]] * 5), np.float32([[0, 0, 0], [1, 0, 0], [0, 1, 0], [1, 1, 0], [2, 2, 0]])):
        pa, oka = O.plane_fit(pts, 0.05)
        pb, okb = S.plane_fit(pts, 0.05)
        assert oka == okb and (np.isnan(pa) == np.isnan(pb)).all()
        assert (pa[~np.isnan(pa)] == pb[~np.isnan(pb)]).all()


@pytest.mark.parametrize("cell", [0.5, 0.3])
def test_neighbour_reuse_is_exact(O, scene_xaloc, cell):
    """query_reusable (lv_reuse_kernel): whenever it vouches for the neighbours found from an earlier iterate, a
    fresh exact search from the new iterate returns the same five points with bit-identical distances"""
    sc = scene_xaloc
    sm = S.ShimMap(sc.map, cell, sc.prm.MAX_DIST_PLANE)
    rates = []
    for pos, rot in ((0.0, 0.0), (2e-4, 1e-5), (3e-3, 1e-4), (2e-2, 5e-4), (8e-2, 5e-3), (0.5, 2e-2)):
        d = np.zeros(23)
        d[0:3] = [pos, -0.7 * pos, 0.4 * pos]
        d[3:6] = [rot, 0.5 * rot, -rot]
        x1 = O.boxplus(sc.x_prop, d)
        reused, same = sm.reuse_check(sc.x_prop, x1, sc.sweep, sc.prm.MAX_DIST_PLANE)
        assert same[reused].all(), (pos, rot, int((~same[reused]).sum()))
        rates.append(reused.mean())
    assert rates[0] > 0.8 and rates[1] > 0.7          # millimetre moves keep most answers
    assert rates[-1] < 0.2                             # half a metre keeps (almost) none
    assert all(a >= b - 0.02 for a, b in zip(rates, rates[1:]))
    # shifted off the surfaces: sparse buckets, upper-level answers, fewer than five neighbours
    for shift in ([0, 0, 0.7], [0, 0, 1.6], [0.4, 0.4, 0.4]):
        q = sc.sweep[:4000] + np.float32(shift)
        for mv in (1e-3, 2e-2):
            d = np.zeros(23)
            d[0:3] = mv
            reused, same = sm.reuse_check(sc.x_prop, O.boxplus(sc.x_prop, d), q, sc.prm.MAX_DIST_PLANE)
            assert same[reused].all()


def _world(sweep, x, O):
    R = O.quat_to_rot(x[3:7]); RL = O.quat_to_rot(x[7:11])
    return ((sweep.astype(np.float64) @ RL.T + x[11:14]) @ R.T + x[0:3]).astype(np.float32)


def _streamed_sweeps(sc, O):
    """three noisy copies of the sweep in world coordinates, 1.5 m apart along the road"""
    rng = np.random.default_rng(3)
    for k in range(3):
        x = sc.truth.copy()
        x[0:3] += [1.5 * k, 0.2 * k, 0.0]
        yield _world(sc.sweep, x, O) + rng.normal(0, 0.01, (len(sc.sweep), 3)).astype(np.float32)


@pytest.mark.parametrize("cell", [0.4, 0.2, 0.6])
def test_incremental_map_add_matches_reference_rule(O, scene_xaloc, cell):
    """Mapper::add = KD_TREE::Add_Points with the 0.2 m rule (ikd_Tree.cpp:478-573), three sweeps streamed into the map by
    the product's incremental update (map_point_key -> sort -> map_merge_run -> dilate -> halo): the content equals the
    oracle's (and the reference ikd-Tree's), the layout invariants hold, and searching the UPDATED map is still exact."""
    sc = scene_xaloc
    golden = RG.load()
    RG.check_scene(golden, sc)
    sm = S.ShimMap(sc.map, cell, 2.0)
    assert sm.size() == len(sc.map) and sm.check() == 0 and sm.error() == 0
    assert (sm.points() == sc.map).all()                            # Build keeps every point, insertion order
    om = O.Map(O.KNN_KDTREE)
    om.build(sc.map)
    for k, new in enumerate(_streamed_sweeps(sc, O)):
        sm.add(new, downsample=True)
        assert sm.check() == 0 and sm.error() == 0
        got = set(map(tuple, sm.points().tolist()))
        assert len(got) == sm.size()
        om.add(new, downsample=True)
        # the oracle holds exactly what the reference ikd-Tree holds after this sweep, so the bar below holds against both
        assert RG.set_digest(om.points()) == golden["xaloc_stream"][k], k
        ref = set(map(tuple, om.points().tolist()))
        assert len(got ^ ref) <= 1e-4 * len(ref), (k, len(got ^ ref), len(ref))     # voxel-face ulp cases
    # the updated map answers queries exactly like a kd-tree over the same points
    om = O.Map(O.KNN_KDTREE)
    om.build(sm.points())
    q = sc.sweep[::7]
    ref = om.match_all(sc.x_prop, sc.oprm, q)
    got = sm.match_all(sc.x_prop, S.make_params(sc.oprm, cell), q)
    inside = np.isfinite(got["nn_sqd"][:, 4])
    assert not (ref["nn_sqd"][~inside, 4].astype(np.float64) < 4.0).any()
    assert (got["nn_sqd"][inside] == ref["nn_sqd"][inside]).all()
    assert (got["valid"] == ref["valid"]).all() and (got["plane"] == ref["plane"]).all()


def test_incremental_map_without_downsampling_and_scattered_points(O):
    """Add_Points(..., downsample = false) appends; isolated random points (27 slots each) neither hang nor corrupt"""
    rng = np.random.default_rng(11)
    a = rng.uniform(-40, 40, (3000, 3)).astype(np.float32)          # every point alone in its voxel
    b = rng.uniform(-40, 40, (2000, 3)).astype(np.float32)
    sm = S.ShimMap(a, 0.4, 2.0)
    sm.add(b, downsample=False)
    assert sm.size() == 5000 and sm.check() == 0 and sm.error() == 0
    assert (sm.points() == np.concatenate([a, b])).all()
    om = O.Map(O.KNN_KDTREE)
    om.build(np.concatenate([a, b]))
    x = np.zeros(26); x[6] = 1; x[10] = 1; x[23] = 9.809
    prm = O.make_params()
    q = rng.uniform(-40, 40, (2000, 3)).astype(np.float32)
    ref = om.match_all(x, prm, q)
    got = sm.match_all(x, S.make_params(prm, 0.4), q)
    inside = np.isfinite(got["nn_sqd"][:, 4])
    assert not (ref["nn_sqd"][~inside, 4].astype(np.float64) < 4.0).any()
    assert (got["nn_sqd"][inside] == ref["nn_sqd"][inside]).all()


def test_block_cube_mask_matches_the_per_bit_test():
    """block_cube_mask (ring search: the occupancy mask of a 4x4x4 block clipped to the cube of wanted rings) against
    the per-voxel test it replaces, over every block offset and ring count the search can produce."""
    import ctypes as C
    L = S.lib()
    L.shim_block_cube_mask.restype = C.c_uint64
    L.shim_block_cube_mask.argtypes = [C.c_int] * 4
    for r in (1, 2, 3, 5, 8, 15):
        for cbx in range(-r - 5, r + 3):
            for cby in (-r - 4, -r - 3, -r, -1, 0, r - 3, r - 1, r, r + 1):
                for cbz in (-r - 4, -r - 2, -2, 0, r - 2, r, r + 1):
                    want = 0
                    for c in range(64):
                        dx, dy, dz = cbx + (c & 3), cby + ((c >> 2) & 3), cbz + (c >> 4)
                        if -r <= dx <= r and -r <= dy <= r and -r <= dz <= r:
                            want |= 1 << c
                    assert L.shim_block_cube_mask(cbx, cby, cbz, r) == want, (cbx, cby, cbz, r)

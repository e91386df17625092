"""The C-ABI library without a GPU: it loads, exports every symbol include/limovelo_b200.h declares,
refuses to compute without CUDA (no CPU fallback), and its host-side pieces (config reader, synthetic
reader, predict / init) behave like the reference's."""
import ctypes as C
import os
import re

import numpy as np
import pytest

import reference_golden as RG
from conftest import have_gpu


def test_library_exports_every_declared_symbol(lv):
    header = open(lv.HEADER_PATH).read()
    body = re.sub(r"/\*.*?\*/", "", header, flags=re.S)
    names = set(re.findall(r"\b(lv_[a-z0-9_]+)\s*\(", body))
    assert len(names) >= 35
    L = C.CDLL(lv.LIB_PATH)
    missing = [n for n in sorted(names) if not hasattr(L, n)]
    assert missing == []
    L.lv_version.restype = C.c_char_p
    assert b"limovelo_b200" in L.lv_version()


def test_synth_library_exports_every_declared_symbol_and_is_cuda_free(lv):
    """include/lv_synth.h <-> liblv_synth.so; the product library no longer carries the synthetic reader, and the
    synthetic reader does not pull in the CUDA runtime (bench.py's CPU reference arm loads only this one)"""
    header = open(os.path.join(os.path.dirname(lv.HEADER_PATH), "lv_synth.h")).read()
    body = re.sub(r"/\*.*?\*/", "", header, flags=re.S)
    names = set(re.findall(r"\b(lv_[a-z0-9_]+)\s*\(", body))
    assert len(names) >= 6
    S = C.CDLL(lv.SYNTH_LIB_PATH)
    assert [n for n in sorted(names) if not hasattr(S, n)] == []
    assert hasattr(S, "lv_params_from_yaml") and hasattr(S, "lv_default_params")
    L = C.CDLL(lv.LIB_PATH)
    assert not hasattr(L, "lv_synth_world_create")
    import subprocess
    needed = subprocess.run(["readelf", "-d", lv.SYNTH_LIB_PATH], capture_output=True, text=True).stdout
    assert "cudart" not in needed and "libcuda" not in needed


def test_struct_layouts_match_the_header(lv):
    assert C.sizeof(lv.IterLog) == 8 + 4 + 4 + 8 * (144 + 12 + 23 + 26)
    p = lv.default_params()
    assert p.MAX_NUM_ITERS == 3 and p.NUM_MATCH_POINTS == 5 and p.MAX_DIST_PLANE == 2.0
    assert abs(p.PLANES_THRESHOLD - 0.1) < 1e-7 and p.LiDAR_noise == 0.001 and p.degeneracy_threshold == 5.0
    assert list(p.LIMITS) == [0.001] * 23 and abs(p.map_downsample_size - 0.2) < 1e-7   # main.cpp:137-175


@pytest.mark.skipif(have_gpu(), reason="only meaningful without a CUDA device")
def test_no_cpu_fallback(lv):
    p = lv.default_params()
    with pytest.raises(RuntimeError, match="LV_ERR_CUDA"):
        lv.Localizer(p)


def test_argument_errors(lv):
    L = lv.lib()
    h = C.c_void_p()
    assert L.lv_create(None, C.byref(h)) == lv.ERR_ARG
    p = lv.default_params(NUM_MATCH_POINTS=7)
    assert L.lv_create(C.byref(p), C.byref(h)) == lv.ERR_ARG
    p = lv.default_params(MAX_NUM_ITERS=9)
    assert L.lv_create(C.byref(p), C.byref(h)) == lv.ERR_ARG
    assert L.lv_map_size(None) == 0 and L.lv_map_exists(None) == 0
    assert L.lv_params_from_yaml(b"/nonexistent.yaml", C.byref(p)) == lv.ERR_IO
    # the widened boundary (deskew, downsamplers, wire format): null handle / null buffers are argument errors, not crashes
    n_out = C.c_int64(7)
    assert L.lv_compensate(None, None, 0, None, None, None, C.c_int64(0), None) == lv.ERR_ARG
    assert L.lv_compensate_device(None, None, 0, None, None, None, C.c_int64(0), None) == lv.ERR_ARG
    assert L.lv_voxelgrid_downsample(None, None, C.c_int64(0), C.c_float(0.5), None, C.byref(n_out)) == lv.ERR_ARG
    assert L.lv_temporal_downsample(None, None, C.c_int64(0), 4, C.c_double(4.0), None, None, C.byref(n_out)) == lv.ERR_ARG
    assert L.lv_pointcloud2_to_points(0, None, None, C.c_int64(0), C.c_uint64(0), 0, 1, C.c_double(0.1), None, None, None, None) == lv.ERR_ARG
    lay = lv.CloudLayout(16, 0, 4, 8, 12, 12, 0)
    buf = (C.c_uint8 * 16)()
    xyz, t = (C.c_float * 3)(), (C.c_double * 1)()
    assert L.lv_pointcloud2_to_points(9, C.byref(lay), buf, C.c_int64(1), C.c_uint64(0), 0, 1, C.c_double(0.1), xyz, t, None, None) == lv.ERR_ARG
    assert L.lv_time_sort_indices(None, C.c_int64(0), None) == lv.ERR_ARG
    # inspection and tick entry points added in round 2
    assert L.lv_last_neighbours(None, C.c_int64(1), None) == lv.ERR_ARG
    assert L.lv_map_add_last_sweep(None, 1) == lv.ERR_ARG and L.lv_map_add_device(None, None, C.c_int64(0), 1) == lv.ERR_ARG


def test_yaml_reader_matches_pyyaml(lv):
    import yaml
    for name in ("xaloc.yaml", "kitti.yaml", "ouster.yaml"):
        path = os.path.join(lv.CONFIG_DIR, name)
        ref = yaml.safe_load(open(path))
        p = lv.params_from_yaml(path)
        assert p.MAX_NUM_ITERS == ref["MAX_NUM_ITERS"] and p.NUM_MATCH_POINTS == ref["NUM_MATCH_POINTS"]
        assert bool(p.estimate_extrinsics) == bool(ref["estimate_extrinsics"])
        assert p.MAX_DIST_PLANE == float(ref["MAX_DIST_PLANE"]) and p.LiDAR_noise == float(ref["LiDAR_noise"])
        assert abs(p.PLANES_THRESHOLD - float(ref["PLANES_THRESHOLD"])) < 1e-7
        assert p.degeneracy_threshold == float(ref["degeneracy_threshold"])
        assert np.allclose(list(p.initial_gravity), ref["initial_gravity"])
        assert np.allclose(list(p.I_Translation_L), ref["I_Translation_L"])
        assert np.allclose(list(p.I_Rotation_L), ref["I_Rotation_L"])
        assert p.covariance_gyroscope == float(ref["covariance_gyroscope"])
        assert p.covariance_bias_acceleration == float(ref["covariance_bias_acceleration"])


def test_yaml_reader_on_the_reference_configs(lv):
    """the full ROS config files of the reference (tests/golden/reference/config) parse to the same hot-path values as
    our subsets"""
    for name in ("xaloc.yaml", "kitti.yaml", "ouster.yaml"):
        a = lv.params_from_yaml(os.path.join(RG.CONFIG_DIR, name))
        b = lv.params_from_yaml(os.path.join(lv.CONFIG_DIR, name))
        for f in ("MAX_NUM_ITERS", "NUM_MATCH_POINTS", "estimate_extrinsics", "MAX_DIST_PLANE", "PLANES_THRESHOLD",
                  "LiDAR_noise", "degeneracy_threshold", "covariance_gyroscope", "covariance_acceleration",
                  "covariance_bias_gyroscope", "covariance_bias_acceleration"):
            assert getattr(a, f) == getattr(b, f), (name, f)
        assert list(a.I_Rotation_L) == list(b.I_Rotation_L) and list(a.I_Translation_L) == list(b.I_Translation_L)
        assert list(a.initial_gravity) == list(b.initial_gravity)


def test_synthetic_reader_is_seeded_and_sane(lv, O):
    prm = lv.params_from_yaml(os.path.join(lv.CONFIG_DIR, "xaloc.yaml"))
    w1, w2 = lv.SynthWorld(7, 30000), lv.SynthWorld(7, 30000)
    m1, m2 = w1.map(), w2.map()
    assert m1.shape == (30000, 3) and (m1 == m2).all()
    assert (lv.SynthWorld(8, 30000).map() != m1).any()
    assert m1[:, 2].min() < -1.7 and m1[:, 2].max() > 3.0           # ground and walls
    x = w1.pose(5.0, prm)
    s1 = w1.sweep(x, rings=16, azimuths=128, seed=3)
    s2 = w2.sweep(x, rings=16, azimuths=128, seed=3)
    assert s1.shape == (2048, 3) and (s1 == s2).all()
    r = np.linalg.norm(s1, axis=1)
    assert r.min() > 3.9 and r.max() < 125.0                        # min_dist 4 m (xaloc.yaml), 120 m + noise
    # the sweep lies on the map: nearly every point has a map point within 0.3 m
    om = O.Map(O.KNN_KDTREE)
    om.build(m1)
    Rw = O.quat_to_rot(x[3:7]); RL = O.quat_to_rot(x[7:11])
    g = ((s1.astype(np.float64) @ RL.T + x[11:14]) @ Rw.T + x[0:3]).astype(np.float32)
    d = np.array([np.sqrt(om.knn(p, 1)[2][0]) for p in g[:400]])
    assert np.median(d) < 0.15 and (d < 0.4).mean() > 0.95

"""What the reference's own ikd-Tree answered, stored under tests/golden/reference/ so that the tests which compare with it
run wherever the suite runs, not only where the LIMO-Velo sources are at hand.

The reference's answers are kept as the arrays themselves where they are small (kNN of test_oracle) and as SHA-256
digests where they are not (per-point match results and map contents of the scene_xaloc fixture, 100 k map points).  A
digest can only say "bit for bit the same", so a test checks that the oracle's own kd-tree reproduces the reference's
digest and then compares the product with the oracle exactly as it compared it with the reference.

Regenerate (needs oracle/_ref/libikdtree_ref.so, which oracle/Makefile builds from the LIMO-Velo sources):
    python tests/reference_golden.py
"""
import hashlib
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
DIR = os.path.join(HERE, "golden", "reference")
PATH = os.path.join(DIR, "ikdtree.npz")
CONFIG_DIR = os.path.join(DIR, "config")      # config/*.yaml of LIMO-Velo, unchanged
MATCH_FIELDS = ("nn_sqd", "valid", "plane")


def digest(*arrays):
    """SHA-256 over dtype, shape and bytes (C order) of each array"""
    h = hashlib.sha256()
    for a in arrays:
        a = np.ascontiguousarray(a)
        h.update(("%s%s" % (a.dtype.str, a.shape)).encode())
        h.update(a.tobytes())
    return h.hexdigest()


def set_digest(points):
    """digest of a point set as the tests compare it (a set of xyz tuples): rows sorted and deduplicated, -0.0 read as 0.0"""
    p = np.asarray(points, np.float32).reshape(-1, 3) + np.float32(0)
    return digest(np.unique(p, axis=0))


def load():
    return np.load(PATH)


def check_scene(ref, sc):
    """the scene_xaloc fixture still makes the inputs the stored answers were computed from"""
    assert digest(sc.map, sc.sweep, sc.x_prop) == ref["xaloc_inputs"], \
        "scene_xaloc changed: regenerate with python tests/reference_golden.py"


def main():
    sys.path.insert(0, os.path.dirname(HERE))
    sys.path.insert(0, HERE)
    import __graft_entry__ as G
    import test_cpu_shim
    import test_oracle
    from conftest import Scene
    lv, O = G.load_package(), G.load_oracle()
    if not O.ref_available():
        raise SystemExit("oracle/_ref/libikdtree_ref.so is not built (make -C oracle REFERENCE=<LIMO-Velo checkout>)")

    def ref_map(pts):
        m = O.Map(O.KNN_REF_IKDTREE)
        m.build(pts)
        return m

    out = {}
    # test_oracle.test_knn_backends_agree
    pts, q = test_oracle._knn_case()
    m = ref_map(pts)
    res = [m.knn(qi) for qi in q]
    out["knn_found"] = np.array([r[0] for r in res], np.int32)
    out["knn_sqd"] = np.stack([r[2] for r in res])
    out["knn_xyz"] = np.stack([r[3] for r in res])
    # test_oracle.test_map_add_matches_reference_ikdtree
    base, new, new2 = test_oracle._add_case()
    m = ref_map(base)
    m.add(new, downsample=True)
    out["add_tree_size"] = np.int64(m.size())                # KD_TREE::size(), lazily deleted nodes included
    counts, digests = [len(set(map(tuple, m.points().tolist())))], [set_digest(m.points())]
    m.add(new2, downsample=True)
    digests.append(set_digest(m.points()))
    m.add(new2, downsample=False)
    counts.append(len(m.points()))
    out["add_count"], out["add_digest"] = np.array(counts, np.int64), np.array(digests)
    # the scene_xaloc fixture (tests/conftest.py): test_gpu_parity and test_cpu_shim
    sc = Scene(lv, O, "xaloc.yaml", max_map_points=1 << 19, max_points=1 << 16)
    out["xaloc_inputs"] = np.array(digest(sc.map, sc.sweep, sc.x_prop))
    r = ref_map(sc.map).match_all(sc.x_prop, sc.oprm, sc.sweep)
    out["xaloc_match"] = np.array([digest(r[k]) for k in MATCH_FIELDS])
    m = ref_map(sc.map)
    m.add(test_cpu_shim._world(sc.sweep, sc.truth, O), downsample=True)
    out["xaloc_add"] = np.array(set_digest(m.points()))
    m = ref_map(sc.map)
    stream = []
    for new in test_cpu_shim._streamed_sweeps(sc, O):
        m.add(new, downsample=True)
        stream.append(set_digest(m.points()))
    out["xaloc_stream"] = np.array(stream)
    os.makedirs(DIR, exist_ok=True)
    np.savez_compressed(PATH, **out)
    print("wrote", PATH, os.path.getsize(PATH), "bytes")


if __name__ == "__main__":
    main()

"""What the reference computes on the fixtures of tests/golden, stored in tests/golden/reference_outputs.npz so that the oracle is held
against the reference's own code without the reference's sources.

The reference side was produced by small_gicp's own headers compiled against the Eigen API shim (oracle/ref_build ->
oracle/_ref/libsmallgicp_ref.so) and by its Registration<> on ParallelReductionOMP (tests/host_ref -> oracle/_ref/libsgb_host_ref.so).
Each `*_outputs(lib, ...)` below runs one comparison of tests/test_oracle_vs_reference.py on `lib` (None = the oracle); the tests run
it on the oracle and compare with the stored reference outputs.  Exact results (indices, structures, voxel-grid points) are stored as
SHA-256 digests of their bytes; floating-point results as values, of a fixed seeded sample of rows where the full array would be large.

Regenerate (needs oracle/_ref, i.e. a build with the reference's sources present):  python tests/reference_outputs.py
"""
import hashlib
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
for p in (ROOT, HERE):
    if p not in sys.path:
        sys.path.insert(0, p)

import oracle as O  # noqa: E402
from conftest import load_golden_xyz, noise_poses  # noqa: E402

PATH = os.path.join(HERE, "golden", "reference_outputs.npz")
LEAVES = [0.1, 0.25, 0.3, 1.0]
CASES = [(f, r) for f in (0, 1, 2) for r in (0, 1, 2)]
THREADS = [0, 2]
ALIGN_CASES = [(0, 0), (1, 0), (2, 0), (2, 1), (2, 2)]
OPTIMIZERS = [0, 1]
OFFSETS = (1, 7, 27)
SAMPLE_ROWS = 512  # rows of a large floating-point output kept at full precision
DROPIN_CASES = ((0, 1), (2, 0), (2, 1))  # (factor, optimizer) of test_host_ref_dropin::test_reference_arm_equals_oracle


def digest(a):
    """SHA-256 of dtype, shape and bytes: equal digests <=> np.array_equal for arrays of one dtype"""
    a = np.ascontiguousarray(a)
    h = hashlib.sha256(f"{a.dtype.str}{a.shape}".encode())
    h.update(a.tobytes())
    return h.hexdigest()


def sample_rows(n, tag):
    """a fixed sorted sample of min(n, SAMPLE_ROWS) row indices, seeded by the output's name"""
    if n <= SAMPLE_ROWS:
        return np.arange(n)
    seed = int.from_bytes(hashlib.sha256(tag.encode()).digest()[:4], "little")
    return np.sort(np.random.default_rng(seed).choice(n, SAMPLE_ROWS, replace=False))


def golden_clouds():
    T = np.loadtxt(os.path.join(HERE, "golden", "T_target_source.txt")).reshape(4, 4)
    return load_golden_xyz("target"), load_golden_xyz("source"), T


def prepare(lib, golden):
    """0.3 m voxel grid, k = 20 normals + covariances (1 thread), kd-trees: (target, target tree, source, source tree)"""
    tgt, src, _ = golden
    tc = O.Cloud(tgt, _lib=lib).voxelgrid_sampling(0.3)
    sc = O.Cloud(src, _lib=lib).voxelgrid_sampling(0.3)
    tt, st = O.KdTree(tc), O.KdTree(sc)
    tt.estimate(20, O.FEAT_NORMAL_COV, 1)
    st.estimate(20, O.FEAT_NORMAL_COV, 1)
    return tc, tt, sc, st


def voxelgrid_outputs(lib, golden, leaf):
    return {f"voxelgrid/{leaf}/{i}": digest(O.Cloud(xyz, _lib=lib).voxelgrid_sampling(leaf).points) for i, xyz in enumerate(golden[:2])}


def kdtree_outputs(prepared):
    """tree structure of the target and kNN of the source points in it.  Node payload: leaves (first, last) 8 bytes, inner nodes axis
    (4 bytes) + threshold (8 bytes at offset 8); padding bytes are unspecified and not compared."""
    tc, tt, sc, _ = prepared
    nodes, idx = tt.export()
    a = nodes.view(np.uint32).reshape(-1, 6)
    leaf = a[:, 4] == 0xFFFFFFFF  # left == INVALID_NODE
    out = {"kdtree/indices": digest(idx), "kdtree/children": digest(a[:, 4:]), "kdtree/leaf_range": digest(a[leaf, :2]),
           "kdtree/inner_axis": digest(a[~leaf, 0]), "kdtree/inner_threshold": digest(a[~leaf, 2:4])}
    for k in (1, 5, 20):
        for name, v in zip(("idx", "d2", "cnt"), tt.knn(sc.points, k)):
            out[f"kdtree/knn{k}/{name}"] = digest(v)
    return out


def features_outputs(prepared):
    tc = prepared[0]
    rows = sample_rows(len(tc), "features")
    return {"features/rows": rows, "features/normals": tc.normals[rows], "features/covs": tc.covs[rows]}


def linearize_outputs(lib, prepared, T_gt, factor, robust, threads):
    """linearize at identity, the ground truth and one noise pose; error at a pose nudged from each; the correspondences found"""
    tc, tt, sc, _ = prepared
    reg = O.Registration(factor=factor, robust=robust, robust_c=0.7, num_threads=threads, _lib=lib)
    key = f"linearize/{factor}/{robust}/{threads}"
    H, b, e, e2, corr = [], [], [], [], []
    for T in [np.eye(4), T_gt] + noise_poses()[1:2]:
        Hk, bk, ek = reg.linearize(tc, tt, sc, T)
        H.append(Hk), b.append(bk), e.append(ek)
        corr.append(digest(reg.correspondences(len(sc))))
        e2.append(reg.error(tc, sc, T @ O.se3_exp(np.array([0.01, -0.02, 0.005, 0.05, -0.03, 0.02]))))
    return {key + "/H": np.array(H), key + "/b": np.array(b), key + "/e": np.array(e), key + "/error": np.array(e2), key + "/corr": np.array(corr)}


def align_outputs(lib, prepared, factor, robust, opt):
    tc, tt, sc, _ = prepared
    reg = O.Registration(factor=factor, robust=robust, num_threads=0, _lib=lib)
    reg.set_optimizer(type=opt)
    rs = [reg.align(tc, tt, sc, Tn) for Tn in noise_poses()[:3]]
    key = f"align/{factor}/{robust}/{opt}"
    return {key + "/stats": np.array([[r.iterations, r.converged, r.num_inliers] for r in rs], dtype=np.int64), key + "/T": np.array([r.T_target_source for r in rs]),
            key + "/error": np.array([r.error for r in rs]), key + "/H": np.array([r.H for r in rs])}


def voxelmap_outputs(lib, prepared, offsets):
    """GaussianVoxelMap(1.0) of the target: its voxels, the nearest voxel of each source point, and a GICP align on it"""
    tc, _, sc, _ = prepared
    vm = O.GaussianVoxelMap(tc, 1.0, offsets)
    coords, means, covs, counts = vm.export()
    idx, d2, found = vm.nn(sc.points)
    rows = sample_rows(len(coords), "voxelmap/voxels")
    qrows = sample_rows(len(idx), f"voxelmap/{offsets}/queries")
    r = O.Registration(factor=O.FACTOR_GICP, num_threads=0, _lib=lib).align(vm, None, sc, np.eye(4))
    key = f"voxelmap/{offsets}"
    # the voxels do not depend on the search offsets: their sampled values are stored once (main() checks they agree)
    return {key + "/coords": digest(coords), key + "/counts": digest(counts), "voxelmap/rows": rows, "voxelmap/means": means[rows], "voxelmap/covs": covs[rows],
            key + "/nn_idx": digest(idx), key + "/nn_found": digest(found), key + "/query_rows": qrows, key + "/nn_d2": d2[qrows],
            key + "/nn_found_sample": found[qrows],
            key + "/align_stats": np.array([r.iterations, r.num_inliers], dtype=np.int64), key + "/align_T": r.T_target_source}


def algebra_inputs():
    rng = np.random.default_rng(1)
    out = []
    for _ in range(10):
        a = rng.normal(0, 0.5, 6)
        A = rng.normal(size=(6, 6))
        A = A @ A.T + 1e-3 * np.eye(6)
        out.append((a, A, rng.normal(size=6)))
    return out


def algebra_outputs(lib):
    import ctypes as C

    dp = C.POINTER(C.c_double)
    exp, solve = [], []
    for a, A, bvec in algebra_inputs():
        T = np.empty((4, 4))
        lib.orc_se3_exp(a.ctypes.data_as(dp), T.ctypes.data_as(dp))
        x = np.empty(6)
        lib.orc_ldlt_solve6(A.ctypes.data_as(dp), bvec.ctypes.data_as(dp), x.ctypes.data_as(dp))
        exp.append(T), solve.append(x)
    return {"algebra/se3_exp": np.array(exp), "algebra/ldlt_solve6": np.array(solve)}


def golden_prepared_clouds(golden):
    """the clouds of conftest.golden_prepared (0.3 m voxel grid, k = 20 normals + covariances, <= 4 threads)"""
    tgt, src, T = golden
    tc = O.Cloud(tgt).voxelgrid_sampling(0.3)
    sc = O.Cloud(src).voxelgrid_sampling(0.3)
    tt, st = O.KdTree(tc), O.KdTree(sc)
    nt = max(1, min(4, O.max_threads()))
    tt.estimate(20, O.FEAT_NORMAL_COV, nt)
    st.estimate(20, O.FEAT_NORMAL_COV, nt)
    return {"target": tc, "source": sc, "target_tree": tt, "source_tree": st, "T": T}


def dropin_outputs(align, omp, g):
    """the reference's Registration<> on its ParallelReductionOMP (tests/host_ref harness) for test_reference_arm_equals_oracle"""
    out = {}
    for factor, optimizer in DROPIN_CASES:
        rs = [align(omp, g["target"], g["source"], Tn, factor=factor, optimizer=optimizer) for Tn in noise_poses()[:2]]
        key = f"dropin_omp/{factor}/{optimizer}"
        out[key + "/T"] = np.array([r.T_target_source for r in rs])
        out[key + "/stats"] = np.array([[r.iterations, r.num_inliers] for r in rs], dtype=np.int64)
    return out


_LOADED = None


def load():
    global _LOADED
    if _LOADED is None:
        with np.load(PATH) as f:
            _LOADED = {k: f[k] for k in f.files}
    return _LOADED


def main():
    ref = O.reference_lib()
    if ref is None:
        raise SystemExit("oracle/_ref/libsmallgicp_ref.so is not built: it needs the reference's sources (oracle/ref_build/Makefile)")
    import test_host_ref_dropin as D

    golden = golden_clouds()
    prepared = prepare(ref, golden)
    out = {}
    for leaf in LEAVES:
        out.update(voxelgrid_outputs(ref, golden, leaf))
    out.update(kdtree_outputs(prepared))
    out.update(features_outputs(prepared))
    for factor, robust in CASES:
        for threads in THREADS:
            out.update(linearize_outputs(ref, prepared, golden[2], factor, robust, threads))
    for factor, robust in ALIGN_CASES:
        for opt in OPTIMIZERS:
            out.update(align_outputs(ref, prepared, factor, robust, opt))
    for offsets in OFFSETS:
        vm = voxelmap_outputs(ref, prepared, offsets)
        for k in ("voxelmap/rows", "voxelmap/means", "voxelmap/covs"):
            assert k not in out or np.array_equal(out[k], vm[k]), k
        out.update(vm)
    out.update(algebra_outputs(ref))
    out.update(dropin_outputs(D.align, D.OMP, golden_prepared_clouds(golden)))
    np.savez_compressed(PATH, **out)
    print(f"{PATH}: {len(out)} arrays, {os.path.getsize(PATH)} bytes")


if __name__ == "__main__":
    main()

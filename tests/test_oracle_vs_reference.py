"""Pins the oracle's restatement (oracle/sgicp_oracle.cpp) against the REFERENCE'S OWN CODE: the outputs of small_gicp's headers
compiled against the Eigen API shim (oracle/ref_build) on the fixtures of tests/golden, stored in tests/golden/reference_outputs.npz
by tests/reference_outputs.py.
Same inputs -> same outputs: bit-exact for integer / index / structure work (compared through SHA-256 digests of the exact bytes),
<= 1e-12 relative for floating point (the two differ only in summation order inside small fixed-size products); large floating-point
outputs are compared on a fixed seeded sample of their rows."""
import numpy as np
import pytest

import oracle as O
import reference_outputs as R


@pytest.fixture(scope="module")
def ref():
    return R.load()


@pytest.fixture(scope="module")
def prepared(golden):
    return R.prepare(None, golden)


def same_digests(out, ref):
    for k, v in out.items():
        assert np.array_equal(v, ref[k]), k


@pytest.mark.parametrize("leaf", R.LEAVES)
def test_voxelgrid_bit_exact(golden, ref, leaf):
    same_digests(R.voxelgrid_outputs(None, golden, leaf), ref)


def test_kdtree_structure_and_knn_bit_exact(prepared, ref):
    same_digests(R.kdtree_outputs(prepared), ref)


def test_features_match(prepared, ref):
    out = R.features_outputs(prepared)
    assert np.array_equal(out["features/rows"], ref["features/rows"])
    np.testing.assert_allclose(out["features/normals"], ref["features/normals"], rtol=0, atol=1e-12)
    np.testing.assert_allclose(out["features/covs"], ref["features/covs"], rtol=0, atol=1e-12)


@pytest.mark.parametrize("factor,robust", R.CASES)
@pytest.mark.parametrize("threads", R.THREADS)
def test_linearize_error_match(prepared, golden, ref, factor, robust, threads):
    out = R.linearize_outputs(None, prepared, golden[2], factor, robust, threads)
    key = f"linearize/{factor}/{robust}/{threads}"
    assert np.array_equal(out[key + "/corr"], ref[key + "/corr"])
    Ha, ba, ea, e1 = (out[key + s] for s in ("/H", "/b", "/e", "/error"))
    Hb, bb, eb, e2 = (ref[key + s] for s in ("/H", "/b", "/e", "/error"))
    for j in range(len(eb)):  # identity, ground truth, one noise pose
        assert np.linalg.norm(Ha[j] - Hb[j]) <= 1e-12 * np.linalg.norm(Hb[j])
        assert np.abs(ba[j] - bb[j]).max() <= 1e-11 * np.sqrt(2 * eb[j] * np.diag(Hb[j])).max()
        assert abs(ea[j] - eb[j]) <= 1e-12 * eb[j]
        assert abs(e1[j] - e2[j]) <= 1e-12 * e2[j]


@pytest.mark.parametrize("factor,robust", R.ALIGN_CASES)
@pytest.mark.parametrize("opt", R.OPTIMIZERS)
def test_align_match(prepared, ref, factor, robust, opt):
    out = R.align_outputs(None, prepared, factor, robust, opt)
    key = f"align/{factor}/{robust}/{opt}"
    assert np.array_equal(out[key + "/stats"], ref[key + "/stats"])  # iterations, converged, num_inliers
    Ta, ea, Ha = (out[key + s] for s in ("/T", "/error", "/H"))
    Tb, eb, Hb = (ref[key + s] for s in ("/T", "/error", "/H"))
    for j in range(len(eb)):  # the first three noise poses
        np.testing.assert_allclose(Ta[j], Tb[j], rtol=0, atol=1e-9)
        assert abs(ea[j] - eb[j]) <= 1e-9 * max(eb[j], 1e-12)
        assert np.linalg.norm(Ha[j] - Hb[j]) <= 1e-9 * np.linalg.norm(Hb[j])


def test_voxelmap_and_vgicp_match(prepared, ref):
    for offsets in R.OFFSETS:
        out = R.voxelmap_outputs(None, prepared, offsets)
        key = f"voxelmap/{offsets}"
        same_digests({k: out[k] for k in (key + "/coords", key + "/counts", key + "/nn_idx", key + "/nn_found", "voxelmap/rows", key + "/query_rows")}, ref)
        np.testing.assert_allclose(out["voxelmap/means"], ref["voxelmap/means"], rtol=0, atol=1e-12)
        np.testing.assert_allclose(out["voxelmap/covs"], ref["voxelmap/covs"], rtol=0, atol=1e-12)
        f = out[key + "/nn_found_sample"] == 1
        np.testing.assert_allclose(out[key + "/nn_d2"][f], ref[key + "/nn_d2"][f], rtol=1e-12)
        assert np.array_equal(out[key + "/align_stats"], ref[key + "/align_stats"])  # iterations, num_inliers
        np.testing.assert_allclose(out[key + "/align_T"], ref[key + "/align_T"], rtol=0, atol=1e-9)


def test_algebra_match(ref):
    for (a, A, bvec), T2, x2 in zip(R.algebra_inputs(), ref["algebra/se3_exp"], ref["algebra/ldlt_solve6"]):
        np.testing.assert_allclose(O.se3_exp(a), T2, rtol=0, atol=1e-15)
        np.testing.assert_allclose(O.ldlt_solve6(A, bvec), x2, rtol=1e-12, atol=1e-14)

"""The drop-in itself: the REFERENCE's own `Registration<Factor, Reduction, ...>` template (its headers, compiled in place by
tests/host_ref/Makefile) with `Reduction = ParallelReductionCUDA` from include/small_gicp/registration/reduction_cuda.hpp -- the
file INTEGRATION.md tells a maintainer to add -- against the same template on the reference's `ParallelReductionOMP`
(registration/registration.hpp:31-43, reduction.hpp:20-27,55-56, optimizer.hpp:24-63,83-149).

The harness (oracle/_ref/libsgb_host_ref.so) can only be built where the reference's sources are present; the tests that call it
skip elsewhere.  CPU (`-m "not gpu"`): the OMP arm's stored results equal the oracle, the CUDA arm refuses to run without a device
(no fallback), INTEGRATION.md shows the compiled file verbatim.  GPU (`-m gpu`): same RegistrationResult from both reductions -- pose within
1e-4 rad / 1e-3 m, same `iterations`, `num_inliers` +- 2 -- for every factor x robust kernel x optimizer, VGICP, a source edited in
place between two align() calls (no stale device mirror), and the generation-counted reuse of the mirror."""
import ctypes as C
import os

import numpy as np
import pytest

import oracle as O
from conftest import ROOT, noise_poses, pose_error

LIB = os.path.join(ROOT, "oracle", "_ref", "libsgb_host_ref.so")
_dp = C.POINTER(C.c_double)


def _lib():
    if not os.path.exists(LIB):
        pytest.skip("oracle/_ref/libsgb_host_ref.so not built (it compiles the reference's headers: `make -C tests/host_ref REF=<reference checkout>`)")
    L = C.CDLL(LIB)
    L.href_align.restype = C.c_int
    L.href_align.argtypes = [_dp, C.c_size_t, _dp, _dp, _dp, C.c_size_t, _dp, _dp, _dp, _dp]
    L.href_last_error.restype = C.c_char_p
    return L


class Result:
    def __init__(self, out):
        self.T_target_source = out[:16].reshape(4, 4).copy()
        self.iterations, self.converged, self.num_inliers, self.error = int(out[16]), bool(out[17]), int(out[18]), float(out[19])
        self.H, self.b = out[20:56].reshape(6, 6).copy(), out[56:62].copy()


def _d(a):
    return None if a is None else a.ctypes.data_as(_dp)


def align(backend, target, source, init_T=None, factor=2, robust=0, robust_c=1.0, rejector=1, max_dist_sq=1.0, optimizer=1, max_iterations=20, num_threads=4,
          vgicp=False, voxel_resolution=1.0, realign=0, sync_every_linearize=True, generation=0):
    L = _lib()
    f64 = lambda a: None if a is None else np.ascontiguousarray(a, dtype=np.float64)  # noqa: E731
    tp, tn, tc = f64(target.points), f64(target.normals), f64(target.covs)
    sp, sc = f64(source.points), f64(source.covs)
    args = np.array([backend, factor, robust, robust_c, rejector, max_dist_sq, optimizer, max_iterations, num_threads, int(vgicp), voxel_resolution, realign,
                     int(sync_every_linearize), generation], dtype=np.float64)
    T0 = np.ascontiguousarray(np.eye(4) if init_T is None else init_T, dtype=np.float64)
    out = np.zeros(62)
    rc = L.href_align(_d(args), len(tp), _d(tp), _d(tn), _d(tc), len(sp), _d(sp), _d(sc), _d(T0), _d(out))
    if rc != 0:
        raise RuntimeError(L.href_last_error().decode())
    return Result(out)


OMP, CUDA = 0, 1


def same_result(r, ref, tag):
    rot, trans = pose_error(ref.T_target_source, r.T_target_source)
    assert rot < 1e-4 and trans < 1e-3, (tag, rot, trans)  # BASELINE north_star bar
    assert r.converged == ref.converged and r.iterations == ref.iterations, (tag, r.iterations, ref.iterations)
    assert abs(r.num_inliers - ref.num_inliers) <= 2, (tag, r.num_inliers, ref.num_inliers)
    assert abs(r.error - ref.error) <= 1e-4 * max(ref.error, 1e-9), tag
    assert np.linalg.norm(r.H - ref.H) <= 1e-4 * np.linalg.norm(ref.H), tag


# ---------------------------------------------------------------- CPU
def test_reference_arm_equals_oracle(golden_prepared):
    """the harness' OMP arm IS the reference (its Registration<> on its ParallelReductionOMP): it must agree with the oracle.
    Its results are stored in tests/golden/reference_outputs.npz (tests/reference_outputs.py), so this runs without the harness."""
    import reference_outputs as R

    g, stored = golden_prepared, R.load()
    for factor, optimizer in R.DROPIN_CASES:
        reg = O.Registration(factor=factor, num_threads=0)
        reg.set_optimizer(type=optimizer)
        key = f"dropin_omp/{factor}/{optimizer}"
        for Tn, T_omp, (iterations, num_inliers) in zip(noise_poses()[:2], stored[key + "/T"], stored[key + "/stats"]):
            ref = reg.align(g["target"], g["target_tree"], g["source"], Tn)
            rot, trans = pose_error(ref.T_target_source, T_omp)
            assert rot < 1e-9 and trans < 1e-9 and iterations == ref.iterations and num_inliers == ref.num_inliers


def test_cuda_arm_has_no_fallback(golden_prepared):
    import torch

    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    g = golden_prepared
    with pytest.raises(RuntimeError, match="no CUDA device"):
        align(CUDA, g["target"], g["source"])


def test_integration_md_shows_the_compiled_header():
    """INTEGRATION.md must contain the binding that was actually compiled, line for line."""
    hdr = open(os.path.join(ROOT, "include", "small_gicp", "registration", "reduction_cuda.hpp")).read().strip()
    doc = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    assert hdr in doc


# ---------------------------------------------------------------- GPU
VARIANTS = [("ICP", 0, 0), ("PLANE_ICP", 1, 0), ("GICP", 2, 0), ("HUBER_GICP", 2, 1), ("CAUCHY_GICP", 2, 2), ("HUBER_ICP", 0, 1), ("CAUCHY_PLANE", 1, 2)]


@pytest.mark.gpu
@pytest.mark.parametrize("name,factor,robust", VARIANTS)
@pytest.mark.parametrize("optimizer", [0, 1])
def test_reference_registration_on_cuda_reduction(golden_prepared, name, factor, robust, optimizer):
    g = golden_prepared
    for j, Tn in enumerate(noise_poses()[:3]):
        kw = dict(factor=factor, robust=robust, robust_c=0.7, optimizer=optimizer)
        ref = align(OMP, g["target"], g["source"], Tn, **kw)
        r = align(CUDA, g["target"], g["source"], Tn, **kw)
        same_result(r, ref, (name, optimizer, j))
        rot, trans = pose_error(g["T"], r.T_target_source)
        assert rot < np.deg2rad(2.5) and trans < 0.2  # registration_test.cpp:139-151


@pytest.mark.gpu
def test_null_rejector_and_vgicp(golden_prepared):
    g = golden_prepared
    ref = align(OMP, g["target"], g["source"], rejector=0)
    r = align(CUDA, g["target"], g["source"], rejector=0)
    same_result(r, ref, "null-rejector")
    assert r.num_inliers == len(g["source"])
    for Tn in noise_poses()[:2]:
        ref = align(OMP, g["target"], g["source"], Tn, vgicp=True, voxel_resolution=1.0)
        r = align(CUDA, g["target"], g["source"], Tn, vgicp=True, voxel_resolution=1.0)
        same_result(r, ref, "vgicp")


@pytest.mark.gpu
@pytest.mark.parametrize("generation", [0, 7])
def test_source_edited_in_place_between_aligns(golden_prepared, generation):
    """An odometry loop re-uses its buffers: same address, same size, new content.  With generation 0 (default) every align()
    re-validates the mirror, so the second align() sees the shifted source -- exactly like the reference, which re-reads host memory.
    With a non-zero generation the caller vouches that the cloud is unchanged: the stale mirror is then the CALLER's contract,
    and the result equals the un-shifted alignment (this is what makes the difference observable)."""
    g = golden_prepared
    ref_shifted = align(OMP, g["target"], g["source"], realign=2)
    ref_plain = align(OMP, g["target"], g["source"])
    r = align(CUDA, g["target"], g["source"], realign=2, generation=generation)
    if generation == 0:
        same_result(r, ref_shifted, "re-uploaded")
        assert pose_error(ref_plain.T_target_source, r.T_target_source)[1] > 0.05  # and it IS a different problem
    else:
        same_result(r, ref_plain, "caller-vouched mirror")


@pytest.mark.gpu
def test_single_sync_mode(golden_prepared):
    """sync_every_linearize = false: correspondences are copied back only when sync_factors() is called -- with the STOCK optimizers
    (no 4-line change) num_inliers then reads 0, everything else is unchanged."""
    g = golden_prepared
    ref = align(CUDA, g["target"], g["source"])
    r = align(CUDA, g["target"], g["source"], sync_every_linearize=False)
    assert np.array_equal(r.T_target_source, ref.T_target_source) and r.iterations == ref.iterations and r.error == ref.error
    assert r.num_inliers == 0 and ref.num_inliers > 1000

#!/usr/bin/env python3
"""bench.py -- correspondence + linearisation + reduction throughput of the small_gicp hot path on B200.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--points P] [--no-extras] [--dump-outputs DIR]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 ... bench.py --gpus N ...

Headline workload (BASELINE.json configs[1]): synthetic room pair, P = 1,000,000 target points and 1,000,000 source points PER GPU,
GICP factor, DistanceRejector(1 m^2).  One "step" = one Reduction::linearize over the rank's source points at the next pose of a FIXED
pose schedule (+ for N > 1 the all-reduce of H|b|e, fused into the reduction kernel).  The schedule is the Gauss-Newton trajectory of
rank 0's own 1M x 1M pair from identity -- computed before the ranks are wired together, broadcast to all of them, hence the SAME
poses for every N -- and is walked like an align(): the identity-pose step searches UNSEEDED (sgb_drop_seeds), every later step is
seeded by its predecessor.  Metric: Mpoints/s per iteration = source points of all ranks / max-over-ranks device time of a step.

`value`        inputs resident in HBM, CUDA events on the launching stream, L2 flushed between steps.
`e2e`          the same step through the C-ABI with HOST (pinned) buffers: source upload (H2D) + linearize + H|b|e back, per step.
`roofline`     algorithmic bytes (GICP: 100 B / source point, SURVEY.md §8d) / kernel time vs the measured HBM copy peak.
`cpu_baseline` / --impl reference: the reference's own ParallelReductionOMP<GICPFactor> (oracle/_ref) on this box's host cores.
Extras on the same line (the other BASELINE configs on hardware; skipped with --no-extras):
`error_ms`     Reduction::error (LM inner loop) over the same 1M points per GPU.
`c1`           configs[0]: the bundled PLY pair, ICP, helper align() vs the 1-thread CPU pipeline; per-call latency (N = 1 only).
`c3`           configs[2]: 120k-ray LiDAR stream, per frame voxel grid / tree + grid / covariances / LM align (N = 1 only).
`c4`           configs[3]: 10M-point VGICP, LevenbergMarquardt, ONE source strong-sharded over the N GPUs.
`c5`           configs[4]: linearize over 100k .. 100M points (ONE cloud pair, source strong-sharded over the N GPUs).
`allreduce_check_rel`  N > 1: |fused sum - NCCL sum of the per-rank local sums| / |sum| (must be <= 1e-12).
`comm_wait_us` N > 1: time the finishing CTA waited for its peers per exchange: min over ranks = transport, max - min = skew.

--dump-outputs DIR writes what the last timed step returned -- H (6x6), b (6), e and, for our arm, the inlier count -- as float64
DIR/<name>.npy, so that two builds run with the same arguments (same seeded inputs) can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "correspondence+reduction Mpoints/sec per GICP iter"
UNIT = "Mpoints/s"
BYTES_PER_POINT = {"ICP": 36, "PLANE_ICP": 52, "GICP": 100, "VGICP": 116}  # SURVEY.md §8(d)
HBM_FALLBACK_GBS = 6650.0  # /opt/skills/guides/B200_PROFILING.md fallback


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--points", type=int, default=1_000_000)
    ap.add_argument("--covs", default="knn", choices=["knn", "analytic"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip c3 / c4 / c5 (profiler runs)")
    ap.add_argument("--c5-sizes", default="100000,1000000,10000000,100000000")
    ap.add_argument("--c4-points", type=int, default=10_000_000)
    ap.add_argument("--c3-frames", type=int, default=12)
    ap.add_argument("--leaf", type=int, default=0, help="max leaf size of the device kd-tree (0 = library default)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's H, b, e (and inlier count) as float64 DIR/<name>.npy")
    return ap.parse_args()


def dump_outputs(path, H, b, e, num_inliers=None):
    """--dump-outputs: the sums one linearize hands its caller, float64, one .npy per array"""
    os.makedirs(path, exist_ok=True)
    arrays = {"H": np.asarray(H).reshape(6, 6), "b": np.asarray(b).reshape(6), "e": np.asarray([e]).reshape(1)}
    if num_inliers is not None:
        arrays["num_inliers"] = np.asarray([num_inliers]).reshape(1)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), np.ascontiguousarray(a, dtype=np.float64))


def dist_env():
    return int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))


def hbm_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
    except Exception:
        return HBM_FALLBACK_GBS, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------------
# inputs
# ------------------------------------------------------------------------------------------------
def make_inputs(points, rank, covs_mode, estimator=None):
    """target (shared by all ranks) and this rank's source shard; covariances as 4x4 zero-padded doubles.
    covs_mode "knn": the reference recipe (k = 20 neighbours, eigenvalues -> (1e-3, 1, 1), normal_estimation.hpp:28-92)
    evaluated by `estimator(points4) -> covs` (our arm: the device estimator; reference arm: the oracle's)."""
    from small_gicp_b200 import synthetic as syn

    world = syn.make_world(points, 42)
    Tgt = syn.gt_transform()
    tgt, tn = syn.sample_cloud(world, points, 43, return_normals=True)
    src_w, sn_w = syn.sample_cloud(world, points, 44 + rank, return_normals=True)
    Ti = np.linalg.inv(Tgt)
    src = src_w @ Ti[:3, :3].T + Ti[:3, 3]
    sn = sn_w @ Ti[:3, :3].T
    tgt = tgt.astype(np.float32).astype(np.float64)
    src = src.astype(np.float32).astype(np.float64)
    tgt4 = np.concatenate([tgt, np.ones((len(tgt), 1))], axis=1)
    src4 = np.concatenate([src, np.ones((len(src), 1))], axis=1)
    if covs_mode == "knn" and estimator is not None:
        tcov, scov = estimator(tgt4), estimator(src4)
        desc = "k=20 nearest-neighbour covariances, eigenvalues regularised to (1e-3,1,1) (reference recipe)"
    else:
        tcov, scov = syn.plane_covariances(tn), syn.plane_covariances(sn)
        desc = "analytic plane covariances I-(1-1e-3)nn^T from the generator's face normals"
    return {"target": tgt4, "source": src4, "target_covs": tcov, "source_covs": scov, "T_gt": Tgt, "covs": desc}


def se3_exp(a):
    """util/lie.hpp:73-96 (host side of the optimizer; numpy)"""
    w, t = a[:3], a[3:]
    th2 = w @ w
    th = np.sqrt(th2)
    K = np.array([[0, -w[2], w[1]], [w[2], 0, -w[0]], [-w[1], w[0], 0]])
    T = np.eye(4)
    if th < 1e-10:
        R = np.eye(3) + K
        V = np.eye(3)
    else:
        R = np.eye(3) + np.sin(th) / th * K + (1 - np.cos(th)) / th2 * (K @ K)
        V = np.eye(3) + (1 - np.cos(th)) / th2 * K + (th - np.sin(th)) / (th2 * th) * (K @ K)
    T[:3, :3] = R
    T[:3, 3] = V @ t
    return T


def pose_error(T1, T2):
    """registration_test.cpp:139-151: angle of R1^T R2, norm of the translation of T1^-1 T2"""
    e = np.linalg.inv(T1) @ T2
    return float(np.arccos(np.clip((np.trace(e[:3, :3]) - 1) / 2, -1, 1))), float(np.linalg.norm(e[:3, 3]))


def gn_trajectory(linearize, max_iter=20, lam=1e-6):
    """GaussNewtonOptimizer::optimize (optimizer.hpp:24-63): returns the poses at which linearize was called."""
    T = np.eye(4)
    poses = []
    for _ in range(max_iter):
        poses.append(T.copy())
        H, b, e = linearize(T)
        d = np.linalg.solve(H + lam * np.eye(6), -b)
        T = T @ se3_exp(d)
        if np.linalg.norm(d[:3]) <= 0.1 * np.pi / 180 and np.linalg.norm(d[3:]) <= 1e-3:
            break
    return poses, T


def lm_align(linearize, error, max_iterations=20, max_inner=10, lam=1e-3, lam_factor=10.0):
    """LevenbergMarquardtOptimizer::optimize (optimizer.hpp:83-149) around linearize(T) -> (H, b, e) and error(T) -> e.
    Returns (T, outer iterations, converged, linearize calls, error calls)."""
    T = np.eye(4)
    converged, n_lin, n_err, last = False, 0, 0, 0
    for it in range(max_iterations):
        if converged:
            break
        last = it  # result.iterations = index of the last iteration that ran (optimizer.hpp:136)
        H, b, e = linearize(T)
        n_lin += 1
        success = False
        for _ in range(max_inner):
            d = np.linalg.solve(H + lam * np.eye(6), -b)
            T_new = T @ se3_exp(d)
            e_new = error(T_new)
            n_err += 1
            if e_new <= e:
                converged = bool(np.linalg.norm(d[:3]) <= 0.1 * np.pi / 180 and np.linalg.norm(d[3:]) <= 1e-3)
                T, e, success = T_new, e_new, True
                lam /= lam_factor
                break
            lam *= lam_factor
        if not success:
            break
    return T, last, converged, n_lin, n_err


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.path = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.out = open(self.path, "w")
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"], stdout=self.out, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def wait_first_sample(self, timeout_s):
        """block until nvidia-smi has written its first line (it needs ~0.1 s to start)"""
        t0 = time.perf_counter()
        while self.proc and time.perf_counter() - t0 < timeout_s:
            try:
                if os.path.getsize(self.path) > 0:
                    return True
            except OSError:
                pass
            time.sleep(0.02)
        return False

    def stop(self):
        res = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if not self.proc:
            return res
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.out.close()
        sm, smax, reasons = [], [], set()
        try:
            for line in open(self.path):
                f = [x.strip() for x in line.split(",")]
                if len(f) < 9:
                    continue
                try:
                    sm.append(float(f[1]))
                    smax.append(float(f[2]))
                except ValueError:
                    continue
                for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            res = {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(smax)), "reasons": sorted(reasons), "samples": len(sm)}
        return res


# ------------------------------------------------------------------------------------------------
# reference arm: the reference's own OpenMP reduction (oracle/_ref) on this box's host cores
# ------------------------------------------------------------------------------------------------
def cpu_kind():
    """("reference", lib) when oracle/_ref exists -- the reference's OWN headers compiled in place against the Eigen API shim
    (oracle/ref_build; built in the dev container, shipped as a .so) -- else ("port", None): the oracle's restatement."""
    import oracle as O

    ref = O.reference_lib()
    return ("reference", ref) if ref is not None else ("port", None)


CPU_NOTE = {
    "reference": "small_gicp's own headers (ParallelReductionOMP<GICPFactor>, schedule(guided,8)) compiled against an Eigen API shim: the reference's code, but without Eigen's SIMD kernels; -O3, no -march=native",
    "port": "oracle restatement of reduction_omp.hpp (schedule(guided,8)); not the reference binary, no Eigen SIMD; -O3, no -march=native",
}


def host_cpu_info():
    """what the CPU arm actually gets: logical CPUs, the affinity mask of this process and the cgroup CPU quota"""
    info = {"nproc": os.cpu_count()}
    try:
        info["affinity"] = len(os.sched_getaffinity(0))
    except Exception:
        info["affinity"] = None
    quota = None
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            quota = open(path).read().strip()
            break
        except Exception:
            continue
    info["cgroup_cpu_max"] = quota
    return info


def cpu_setup(inp, threads):
    import oracle as O

    kind, lib = cpu_kind()
    tc = O.Cloud(inp["target"], _lib=lib)
    sc = O.Cloud(inp["source"], _lib=lib)
    t0 = time.perf_counter()
    tt = O.KdTree(tc)
    build_s = time.perf_counter() - t0
    tc.set_features(None, inp["target_covs"])
    sc.set_features(None, inp["source_covs"])
    return O, tc, tt, sc, cpu_registration(threads), build_s


def cpu_registration(threads):
    import oracle as O

    return O.Registration(factor=O.FACTOR_GICP, rejector=O.REJECT_DISTANCE, max_dist_sq=1.0, num_threads=threads, _lib=cpu_kind()[1])


def thread_candidates():
    """torchrun exports OMP_NUM_THREADS=1 and torch pins OpenMP to the physical core count, so counts are passed explicitly (the
    reference's parallel regions carry a num_threads() clause, reduction_omp.hpp:36).  Candidates: 32 / 64 / 128 clipped to what the
    process may use, plus that limit itself."""
    try:
        limit = len(os.sched_getaffinity(0))
    except Exception:
        limit = os.cpu_count() or 1
    limit = max(1, limit)
    cand = {min(t, limit) for t in (32, 64, 128)} | {limit}
    try:  # a cgroup CPU quota below the CPU count (cpu.max "1600000 100000" = 16 CPUs): more threads than that only fight each other
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            cpus = max(1, int(round(int(q) / int(per))))
            cand |= {min(limit, cpus), min(limit, 2 * cpus)}
    except Exception:
        pass
    return sorted(cand, reverse=True)


def best_cpu_registration(inp, reps=3):
    """the fastest of the candidate thread counts, each timed over `reps` identity-pose linearizes after one warm-up"""
    trials, best = [], None
    O, tc, tt, sc, _, build_s = cpu_setup(inp, thread_candidates()[0])
    for threads in thread_candidates():
        reg = cpu_registration(threads)
        reg.linearize(tc, tt, sc, np.eye(4))
        t0 = time.perf_counter()
        for _ in range(reps):
            reg.linearize(tc, tt, sc, np.eye(4))
        dt = (time.perf_counter() - t0) / reps
        trials.append({"threads": threads, "ms": dt * 1e3})
        if best is None or dt < best[0]:
            best = (dt, threads, reg)
    return best[1], (O, tc, tt, sc, best[2], build_s), trials


def run_reference(args):
    rank, local_rank, world = dist_env()
    if rank != 0:
        return 0
    limit = thread_candidates()[0]
    os.environ["OMP_NUM_THREADS"] = str(limit)  # before libgomp is loaded (torchrun sets it to 1)
    import oracle as O

    def oracle_covs(p4):  # the reference arm prepares its inputs with the CPU oracle only (none of our kernels on this arm)
        c = O.Cloud(p4, _lib=cpu_kind()[1])
        t = O.KdTree(c)
        t.estimate(20, O.FEAT_COV, limit)
        return c.covs

    inp = make_inputs(args.points, 0, args.covs, oracle_covs)
    threads, (O, tc, tt, sc, reg, build_s), trials = best_cpu_registration(inp)
    poses, T_final = gn_trajectory(lambda T: reg.linearize(tc, tt, sc, T))
    for i in range(args.warmup):
        reg.linearize(tc, tt, sc, poses[i % len(poses)])
    t0 = time.perf_counter()
    for i in range(args.steps):
        last = reg.linearize(tc, tt, sc, poses[i % len(poses)])
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, *last)
    ms = dt / args.steps * 1e3
    value = args.points / (ms * 1e-3) / 1e6
    rot, trans = pose_error(inp["T_gt"], T_final)
    line = {
        "impl": "reference",
        "metric": METRIC,
        "value": value,
        "unit": UNIT,
        "n_gpus": args.gpus,
        "steps": args.steps,
        "warmup": args.warmup,
        "ms_per_step": ms,
        "higher_is_better": True,
        "scaling": "weak",
        "vs_baseline": None,
        "dtype": "f64",
        "data": "synthetic",
        "config": workload_config(args, inp),
        "cpu_baseline": {
            "value": value,
            "unit": UNIT,
            "cores": threads,
            "kind": cpu_kind()[0],
            "sample": f"{args.steps} x Reduction::linearize over all {args.points} source points at the poses of its own GaussNewton trajectory; " + CPU_NOTE[cpu_kind()[0]],
            "thread_trials": trials,
            "host": host_cpu_info(),
            "kdtree_build_s": build_s,
        },
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "final_pose_rowmajor": [float(x) for x in T_final.reshape(-1)],
        "pose_error_vs_gt": {"rot_rad": rot, "trans_m": trans, "gn_iterations": len(poses)},
    }
    print(json.dumps(line), flush=True)
    return 0


def workload_config(args, inp):
    """identical for both arms (the driver compares the dicts)"""
    return {
        "workload": f"BASELINE configs[1]: {args.points}-pt synthetic room pair per GPU, GICP factor, DistanceRejector(1.0), poses of a GaussNewton trajectory from identity (<=20 iters), one step = one linearize",
        "points_target": args.points,
        "points_source_per_gpu": args.points,
        "covariances": inp["covs"],
        "l2": "flushed between timed steps (256 MiB write)",
        "parallelism": f"source sharded over {args.gpus} GPU(s), target + search structure replicated, all-reduce of H|b|e (44 doubles) per step" if args.gpus > 1 else "single GPU",
    }


# ------------------------------------------------------------------------------------------------
# helpers of our arm
# ------------------------------------------------------------------------------------------------
class Bench:
    """per-process state shared by the legs of our arm"""

    def __init__(self, args):
        import torch

        import small_gicp_b200 as sg

        self.torch, self.sg, self.args = torch, sg, args
        self.rank, self.local_rank, self.world = dist_env()
        if self.world != args.gpus and self.world != 1:
            raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={self.world}")
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device; the hot path has no CPU fallback")
        torch.cuda.set_device(self.local_rank)
        self.use_dist = self.world > 1
        self.dist = None
        if self.use_dist:
            import torch.distributed as dist

            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local_rank))
            self.dist = dist
        self.dev = torch.device("cuda", self.local_rank)
        # one explicit (non-default) stream for everything: the contexts' kernels, torch's fills / events and NCCL all run on it,
        # so CUDA events recorded on it bracket exactly the work being timed
        self.stream = torch.cuda.Stream(device=self.dev)
        torch.cuda.set_stream(self.stream)
        assert self.stream.cuda_stream != 0
        self.flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=self.dev)
        self.out = torch.zeros(64, dtype=torch.float64, device=self.dev)
        self.fused_wanted = os.environ.get("SGB_FUSED_ALLREDUCE", "1") != "0"

    def context(self, connect=False):
        ctx = self.sg.Context(self.local_rank)
        ctx.set_stream(self.stream.cuda_stream)
        fused = False
        if connect and self.use_dist and self.fused_wanted:
            from small_gicp_b200.distributed import connect_fused

            fused = connect_fused(ctx)
        return ctx, fused

    def barrier(self):
        if self.use_dist:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, values):
        t = self.torch.tensor([float(v) for v in values], dtype=self.torch.float64, device=self.dev)
        if self.use_dist:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return [float(x) for x in t.cpu()]

    def event_ms(self, fn, reps, flush=True):
        """mean device time of fn() over reps calls (CUDA events on the launching stream, L2 flushed before each), max over ranks"""
        torch = self.torch
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
        self.barrier()
        for a, b in ev:
            if flush:
                self.flush.zero_()
            a.record(self.stream)
            fn()
            b.record(self.stream)
        self.barrier()
        return self.max_over_ranks([float(np.mean([a.elapsed_time(b) for a, b in ev]))])[0]


def shard(n, rank, world):
    from small_gicp_b200.distributed import shard_range

    return shard_range(n, rank, world)


# ------------------------------------------------------------------------------------------------
# extras: the other BASELINE configs on hardware
# ------------------------------------------------------------------------------------------------
def run_c5(B, sizes):
    """configs[4]: one cloud pair per size (density constant), target + search structure replicated, the source strong-sharded over
    the ranks (the pair's offset is synthetic.gt_transform_scaled: the same local misalignment at every size); one linearize at the
    iteration-0 pose (identity) and one at the converged pose (T_gt), GICP, everything device-resident:
    points generated on the GPU, kd-tree / block lists / k = 20 covariances built there."""
    from small_gicp_b200 import synthetic as syn

    sg, torch = B.sg, B.torch
    peak, _ = hbm_peak()
    rows = []
    for n in sizes:
        t0 = time.perf_counter()
        world_def = syn.make_world(n, 42)
        Tgt = syn.gt_transform_scaled(syn.world_side(n))
        ctx, fused = B.context(connect=True)
        try:
            tgt = syn.sample_cloud_torch(world_def, n, 43, B.dev)
            ctx.set_target(tgt)
            del tgt
            ctx.build_target_kdtree(0)
            ctx.estimate_target_features(20)
            src = syn.sample_cloud_torch(world_def, n, 44, B.dev, transform=np.linalg.inv(Tgt))
            lo, hi = shard(n, B.rank, B.world)
            if B.world > 1:  # spatially coherent shards (slabs along x): a rank only touches its part of the replicated target
                src = src[torch.argsort(src[:, 0])].contiguous()
            if B.world == 1:  # the whole source is this rank's: covariances estimated in place, nothing leaves the library
                ctx.set_source(src)
                ctx.estimate_source_features(20)
                del src
            else:  # covariances need the neighbours of the WHOLE source: estimate on the full cloud (scratch context), keep the shard
                tmp, _ = B.context()
                _, scov = tmp.estimate_features(src, 20, normals=False)
                tmp.close()
                ctx.set_source(src[lo:hi].contiguous(), scov[lo:hi].contiguous())
                del src, scov
            ctx.synchronize()
            torch.cuda.empty_cache()
            setup_s = time.perf_counter() - t0
            row = {"points": n, "points_per_gpu": hi - lo, "setup_s": setup_s}
            reps = 10 if n <= 10_000_000 else 5
            for fname, fkind in (("GICP", sg.FACTOR_GICP), ("ICP", sg.FACTOR_ICP)):  # SURVEY 8(d) C5: both factors
                for name, T in (("iteration0", np.eye(4)), ("converged", Tgt)):
                    def step():
                        ctx.drop_seeds()
                        ctx.linearize_device(T, B.out.data_ptr(), factor=fkind, rejector=sg.REJECT_DISTANCE, max_dist_sq=1.0)
                        if B.use_dist and not fused:
                            B.dist.all_reduce(B.out[:44])

                    for _ in range(2):
                        step()
                    ms = B.event_ms(step, reps)
                    gbs = BYTES_PER_POINT[fname] * (n / B.world) / (ms * 1e-3) / 1e9  # per GPU
                    res = {"ms": ms, "mpoints_per_s": n / (ms * 1e-3) / 1e6, "algorithmic_gbs_per_gpu": gbs, "roofline_frac": gbs / peak}
                    if fname == "GICP":
                        row[name] = res
                    else:
                        row.setdefault("icp", {})[name] = res
                if fname == "GICP":
                    h = B.out[:44].cpu().numpy()
                    row["inliers_converged"] = int(round(h[43]))
            rows.append(row)
        finally:
            B.barrier()
            ctx.close()
            torch.cuda.empty_cache()
    return {
        "what": "BASELINE configs[4]: linearize (GICP; `icp` = the same with the point-to-point factor, 36 algorithmic B / point; DistanceRejector(1.0)) over N target x N source points, density constant; ONE source strong-sharded over the GPUs (slabs along x), target + kd-tree + block lists replicated; clouds generated and prepared on the device (kd-tree, k=20 covariances); unseeded search; CUDA events, L2 flushed, max over ranks",
        "n_gpus": B.world,
        "rows": rows,
    }


def run_c4(B, n):
    """configs[3]: 10M-point VGICP (Gaussian voxel map target, leaf 1.0 m; registration_helper.cpp:125-137), default
    LevenbergMarquardt optimizer, ONE source strong-sharded over the ranks, H|b|e exchanged inside the kernel."""
    from small_gicp_b200 import synthetic as syn

    sg, torch = B.sg, B.torch
    peak, _ = hbm_peak()
    t0 = time.perf_counter()
    world_def = syn.make_world(n, 42)
    Tgt = syn.gt_transform_scaled(syn.world_side(n))
    ctx, fused = B.context(connect=True)
    tgt = syn.sample_cloud_torch(world_def, n, 43, B.dev)
    _, tcov = ctx.estimate_features(tgt, 20, normals=False)
    ctx.build_target_voxelmap(tgt, tcov, 1.0)
    n_vox = ctx.target_size
    del tgt, tcov
    src = syn.sample_cloud_torch(world_def, n, 44, B.dev, transform=np.linalg.inv(Tgt))
    if B.world > 1:  # spatially coherent shards (slabs along x)
        src = src[torch.argsort(src[:, 0])].contiguous()
    _, scov = ctx.estimate_features(src, 20, normals=False)
    lo, hi = shard(n, B.rank, B.world)
    ctx.set_source(src[lo:hi].contiguous(), scov[lo:hi].contiguous())
    del src, scov
    ctx.synchronize()
    torch.cuda.empty_cache()
    setup_s = time.perf_counter() - t0
    err = torch.zeros(8, dtype=torch.float64, device=B.dev)

    def lin(T):
        ctx.linearize_device(T, B.out.data_ptr(), factor=sg.FACTOR_GICP, rejector=sg.REJECT_DISTANCE, max_dist_sq=1.0)
        if B.use_dist and not fused:
            B.dist.all_reduce(B.out[:44])
        h = B.out[:44].cpu().numpy()
        return h[:36].reshape(6, 6), h[36:42], float(h[42])

    def error(T):
        ctx.error_device(T, err.data_ptr())
        if B.use_dist and not fused:
            B.dist.all_reduce(err[:1])
        return float(err[0].cpu())

    lm_align(lin, error)  # warm-up (allocations, lazy module loading)
    B.barrier()
    t0 = time.perf_counter()
    T, its, conv, n_lin, n_err = lm_align(lin, error)
    B.barrier()
    align_ms = B.max_over_ranks([(time.perf_counter() - t0) * 1e3])[0]
    inliers = int(round(float(B.out[43].cpu())))
    rot, trans = pose_error(Tgt, T)
    T_it0 = np.eye(4)
    lin_ms0 = B.event_ms(lambda: ctx.linearize_device(T_it0, B.out.data_ptr(), factor=sg.FACTOR_GICP, rejector=sg.REJECT_DISTANCE, max_dist_sq=1.0), 10)
    lin_ms1 = B.event_ms(lambda: ctx.linearize_device(T, B.out.data_ptr(), factor=sg.FACTOR_GICP, rejector=sg.REJECT_DISTANCE, max_dist_sq=1.0), 10)
    err_ms = B.event_ms(lambda: ctx.error_device(T, err.data_ptr()), 10)
    per_gpu = n / B.world
    res = {
        "what": "BASELINE configs[3]: VGICP = GICP factor on a GaussianVoxelMap(leaf 1.0 m) target built on the device from the 10M-point cloud (k=20 covariances), LevenbergMarquardt (optimizer.hpp:83-149) on the host, ONE source strong-sharded over the GPUs, voxel map replicated, H|b|e all-reduced inside the kernel; CUDA events, L2 flushed, max over ranks",
        "points": n,
        "points_per_gpu": hi - lo,
        "voxels": n_vox,
        "n_gpus": B.world,
        "setup_s": setup_s,
        "linearize_ms": {"iteration0": lin_ms0, "converged": lin_ms1},
        "linearize_mpoints_per_s": n / (lin_ms1 * 1e-3) / 1e6,
        "linearize_roofline_frac": BYTES_PER_POINT["VGICP"] * per_gpu / (lin_ms1 * 1e-3) / 1e9 / peak,
        "error_ms": err_ms,
        "error_roofline_frac": BYTES_PER_POINT["GICP"] * per_gpu / (err_ms * 1e-3) / 1e9 / peak,
        "lm": {"align_ms_wall": align_ms, "outer_iterations": its + 1, "linearize_calls": n_lin, "error_calls": n_err, "converged": conv, "inliers": inliers},
        "pose_error_vs_gt": {"rot_rad": rot, "trans_m": trans},
    }
    B.barrier()
    ctx.close()
    torch.cuda.empty_cache()
    # the same pipeline against the CPU oracle at a size it finishes in seconds (rank 0, single GPU run only)
    if B.world == 1:
        try:
            res["pose_vs_oracle_200k"] = c4_vs_oracle(B, 200_000)
        except Exception as e:  # the oracle is a checker: its absence must not take the bench line down
            res["pose_vs_oracle_200k"] = {"error": repr(e)}
    return res


def c4_vs_oracle(B, n):
    import oracle as O
    from small_gicp_b200.synthetic import make_pair

    sg = B.sg
    tgt, src, Tgt = make_pair(n)
    nt = max(1, O.max_threads())
    tc, sc = O.Cloud(tgt), O.Cloud(src)
    tt, st = O.KdTree(tc), O.KdTree(sc)
    tt.estimate(20, O.FEAT_COV, nt)
    st.estimate(20, O.FEAT_COV, nt)
    vm = O.GaussianVoxelMap(tc, 1.0)
    ref = O.Registration(factor=O.FACTOR_GICP, num_threads=nt).align(vm, None, sc, np.eye(4))
    ctx, _ = B.context()
    ctx.build_target_voxelmap(tc.points, tc.covs, 1.0)
    ctx.set_source(sc.points, sc.covs)
    T, its, conv, _, _ = lm_align(lambda T: ctx.linearize(T, factor=sg.FACTOR_GICP), ctx.error)
    ctx.close()
    rot, trans = pose_error(ref.T_target_source, T)
    return {"rot_rad": rot, "trans_m": trans, "iterations_gpu": its, "iterations_oracle": int(ref.iterations), "inputs": "identical (oracle-made k=20 covariances on both sides)"}


def run_c3(B, n_frames):
    """configs[2]: frame-to-frame GICP odometry over a 120k-ray LiDAR stream (benchmark_odom.hpp:49-82 +
    odometry_benchmark_small_gicp_tbb.cpp:22-48): per frame 0.25 m voxel grid -> kd-tree (+ grid front end) -> k = 20 covariances ->
    LM GICP against the previous frame from identity.  Frames arrive in HOST memory (as from a driver); everything after the upload
    stays on the device.  Wall clock per stage with a synchronisation after each (what a caller would see)."""
    from small_gicp_b200 import synthetic as syn

    sg, torch = B.sg, B.torch
    side = 400.0
    world_def = syn.make_world(16_000_000, 42)
    poses = [syn.lidar_pose(f, side) for f in range(n_frames)]
    # frames live in page-locked host buffers, as a capture pipeline would deliver them (a pageable 3.8 MB frame costs ~0.3 ms more to upload)
    frames_pin = [syn.lidar_frame_torch(world_def, poses[f], 45 + f, B.dev).cpu().pin_memory() for f in range(n_frames)]
    frames = [x.numpy() for x in frames_pin]
    torch.cuda.synchronize()
    ctx, _ = B.context()
    stages = {"voxelgrid_ms": [], "source_upload_tree_covariances_ms": [], "lm_align_ms": [], "handover_to_target_grid_ms": [], "total_ms": []}
    lm_stats, n_down, errs = [], [], []
    prev = None
    T_est, T_gt_acc = np.eye(4), np.eye(4)

    def clock():
        ctx.synchronize()
        return time.perf_counter()

    for f in range(n_frames):
        t0 = clock()
        pts = ctx.voxelgrid_sampling(frames[f], 0.25)
        t1 = clock()
        n_down.append(len(pts))
        ctx.set_source(pts)
        ctx.estimate_source_features(20)  # builds the frame's kd-tree on the device and keeps it
        t2 = clock()
        if prev is not None:
            T, its, conv, n_lin, n_err = lm_align(lambda T: ctx.linearize(T, factor=sg.FACTOR_GICP, rejector=sg.REJECT_DISTANCE, max_dist_sq=1.0), ctx.error)
            t3 = clock()
            lm_stats.append((its + 1, n_lin, n_err))
            gt = np.linalg.inv(poses[f - 1]) @ poses[f]
            errs.append(pose_error(gt, T))
            T_est, T_gt_acc = T_est @ T, T_gt_acc @ gt
        else:
            t3 = t2
        # this frame is the next target (odometry_benchmark_small_gicp_tbb.cpp:41-43): points, tree and covariances are taken over on the
        # device, only the grid front end is built on top
        ctx.adopt_source_as_target()
        t4 = clock()
        if prev is not None and f >= 2:  # frame 1 pays lazy module loading / first allocations
            stages["voxelgrid_ms"].append((t1 - t0) * 1e3)
            stages["source_upload_tree_covariances_ms"].append((t2 - t1) * 1e3)
            stages["lm_align_ms"].append((t3 - t2) * 1e3)
            stages["handover_to_target_grid_ms"].append((t4 - t3) * 1e3)
            stages["total_ms"].append((t4 - t0) * 1e3)
        prev = pts
    ctx.close()
    rot_acc, trans_acc = pose_error(T_gt_acc, T_est)
    res = {
        "what": "BASELINE configs[2]: synthetic 64-beam x 1875-azimuth LiDAR stream (120k rays / frame, sensor moving 1.0 m + 1 deg yaw per frame, range noise 0.02 m) in the 400 m room; per frame 0.25 m voxel grid, kd-tree, k=20 covariances, LevenbergMarquardt GICP vs the previous frame from identity, then the frame is handed over as the next target (sgb_target_adopt_source: tree and covariances reused as the reference's loop reuses them, grid front end built); input frames in page-locked host memory, wall clock per stage (synchronised), frames 2.. averaged",
        "frames": n_frames,
        "points_per_frame_raw": int(np.mean([len(x) for x in frames])),
        "points_per_frame_downsampled": int(np.mean(n_down)),
        "ms_per_frame": {k: float(np.mean(v)) for k, v in stages.items() if v},
        "frames_per_s": 1e3 / float(np.mean(stages["total_ms"])) if stages["total_ms"] else None,
        "lm_outer_iterations_mean": float(np.mean([x[0] for x in lm_stats])),
        "linearize_calls_mean": float(np.mean([x[1] for x in lm_stats])),
        "error_calls_mean": float(np.mean([x[2] for x in lm_stats])),
        "pose_error_vs_gt_per_frame": {"rot_rad_max": float(max(e[0] for e in errs)), "trans_m_max": float(max(e[1] for e in errs))},
        "pose_error_vs_gt_accumulated": {"rot_rad": rot_acc, "trans_m": trans_acc},
    }
    # the reference's per-frame cost on the host cores for three of the frames (same stages, the CPU oracle; bounded sample)
    try:
        import oracle as O

        best = None
        for nt in sorted({4, 16, min(64, thread_candidates()[0])}):  # the reference's odometry benchmark defaults to 4 threads; small frames do not scale far
            cpu_ms, prev_c = [], None
            for f in range(min(4, n_frames)):
                t0 = time.perf_counter()
                oc = O.Cloud(frames[f][:, :3]).voxelgrid_sampling(0.25)
                ot = O.KdTree(oc)
                ot.estimate(20, O.FEAT_COV, nt)
                if prev_c is not None:
                    O.Registration(factor=O.FACTOR_GICP, num_threads=nt).align(prev_c[0], prev_c[1], oc, np.eye(4))
                    cpu_ms.append((time.perf_counter() - t0) * 1e3)
                prev_c = (oc, ot)
            if best is None or np.mean(cpu_ms) < best[0]:
                best = (float(np.mean(cpu_ms)), nt, len(cpu_ms))
        res["cpu_ms_per_frame"] = {"value": best[0], "threads": best[1], "kind": "port", "sample": f"{best[2]} frames, best of 4 / 16 / 64 threads: voxel grid + kd-tree (serial builder, registration_helper.cpp:30) + k=20 covariances + LM GICP align, CPU oracle"}
    except Exception as e:
        res["cpu_ms_per_frame"] = {"error": repr(e)}
    return res


def run_c1(B):
    """configs[0]: the reference's bundled data/target.ply <-> data/source.ply (committed as tests/golden/*_xyz.f32), point-to-point ICP
    through the helper align() surface (registration_helper.cpp:58-115: 0.25 m voxel grid, k = 10 normals + covariances, kd-tree, LM,
    <= 20 iterations, 1 m): the C++ host mirror with every stage on the device, wall clock, next to the CPU oracle's restatement of the
    same pipeline on ONE thread (the configuration BASELINE.json names), and the per-call latency of sgb_linearize at that size."""
    import oracle as O
    from small_gicp_b200 import host_api

    sg = B.sg
    gold = os.path.join(ROOT, "tests", "golden")
    tgt = np.fromfile(os.path.join(gold, "target_xyz.f32"), dtype="<f4").reshape(-1, 3).astype(np.float64)
    src = np.fromfile(os.path.join(gold, "source_xyz.f32"), dtype="<f4").reshape(-1, 3).astype(np.float64)
    T_file = np.loadtxt(os.path.join(gold, "T_target_source.txt")).reshape(4, 4)
    for _ in range(2):
        r = host_api.helper_align(tgt, src, type=0)
    reps = 5
    t0 = time.perf_counter()
    for _ in range(reps):
        r = host_api.helper_align(tgt, src, type=0)
    gpu_ms = (time.perf_counter() - t0) * 1e3 / reps
    tp0 = time.perf_counter()
    tc, tt = O.preprocess_points(tgt, 0.25, 10, 1)
    sc, st = O.preprocess_points(src, 0.25, 10, 1)
    t1 = time.perf_counter()
    ref = O.Registration(factor=O.FACTOR_ICP, num_threads=1).align(tc, tt, sc, np.eye(4))
    t2 = time.perf_counter()
    cpu_pre_ms, cpu_total_ms = (t1 - tp0) * 1e3, (t2 - tp0) * 1e3
    rot, trans = pose_error(ref.T_target_source, r.T_target_source)
    rot_f, trans_f = pose_error(T_file, r.T_target_source)
    # per-call latency of the hot path at this size (host-returning sgb_linearize / sgb_error: launch + mapped result + one synchronisation)
    ctx, _ = B.context()
    ctx.set_target(tc.points)
    ctx.build_target_kdtree(0)
    ctx.set_source(sc.points)
    T = r.T_target_source
    for _ in range(20):
        ctx.linearize(T, factor=sg.FACTOR_ICP)
        ctx.error(T)
    n_calls = 200
    t0 = time.perf_counter()
    for _ in range(n_calls):
        ctx.linearize(T, factor=sg.FACTOR_ICP)
    lin_us = (time.perf_counter() - t0) * 1e6 / n_calls
    t0 = time.perf_counter()
    for _ in range(n_calls):
        ctx.error(T)
    err_us = (time.perf_counter() - t0) * 1e6 / n_calls
    reg1 = O.Registration(factor=O.FACTOR_ICP, num_threads=0)
    reg1.linearize(tc, tt, sc, T)
    t0 = time.perf_counter()
    for _ in range(20):
        reg1.linearize(tc, tt, sc, T)
    cpu_lin_us = (time.perf_counter() - t0) * 1e6 / 20
    ctx.close()
    return {
        "what": "BASELINE configs[0]: bundled target.ply <-> source.ply, point-to-point ICP, helper align() (0.25 m voxel grid, k=10 features, kd-tree, LM <= 20 iterations); GPU: C++ host mirror + device pipeline, wall clock per align() incl. both uploads; CPU: oracle restatement, 1 thread",
        "points": {"target_raw": len(tgt), "source_raw": len(src), "target": r.target_size, "source": r.source_size},
        "helper_align_ms": gpu_ms,
        "cpu_1thread_ms": {"preprocess": cpu_pre_ms, "align": (t2 - t1) * 1e3, "total": cpu_total_ms},
        "iterations": {"gpu": r.iterations, "cpu": int(ref.iterations)},
        "pose_vs_cpu": {"rot_rad": rot, "trans_m": trans},
        "pose_vs_T_target_source_txt": {"rot_rad": rot_f, "trans_m": trans_f},
        "sgb_linearize_call_us": lin_us,
        "sgb_error_call_us": err_us,
        "cpu_1thread_linearize_us": cpu_lin_us,
    }


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
def run_ours(args):
    B = Bench(args)
    torch, sg, dist = B.torch, B.sg, B.dist
    rank, world, dev, stream, out, flush = B.rank, B.world, B.dev, B.stream, B.out, B.flush
    use_dist = B.use_dist
    GICP = dict(factor=sg.FACTOR_GICP, rejector=sg.REJECT_DISTANCE, max_dist_sq=1.0)

    ctx, _ = B.context()
    inp = make_inputs(args.points, rank, args.covs, lambda p4: ctx.estimate_features(p4, 20, normals=False)[1])
    n_src = inp["source"].shape[0]
    ctx.set_target(inp["target"], None, inp["target_covs"])
    torch.cuda.synchronize()
    t_build = time.perf_counter()
    ctx.build_target_kdtree(args.leaf)  # device kd-tree + block lists of the grid front end
    ctx.synchronize()
    target_build_ms = (time.perf_counter() - t_build) * 1e3
    # pinned host copies of the step's inputs for the e2e leg
    src_pin = torch.from_numpy(inp["source"]).pin_memory()
    cov_pin = torch.from_numpy(inp["source_covs"]).pin_memory()
    ctx.set_source(src_pin.numpy(), cov_pin.numpy())

    # ---- the pose schedule: rank 0's OWN Gauss-Newton trajectory (local sums: the ranks are not wired together yet), the same for every N
    sched = torch.zeros(21 * 16, dtype=torch.float64, device=dev)
    if rank == 0:
        p0, _ = gn_trajectory(lambda T: ctx.linearize(T, **GICP))
        sched[0] = len(p0)
        sched[1 : 1 + 16 * len(p0)] = torch.from_numpy(np.stack(p0).reshape(-1)).to(dev)
    if use_dist:
        dist.broadcast(sched, src=0)
    hs = sched.cpu().numpy()
    poses = [hs[1 + 16 * k : 17 + 16 * k].reshape(4, 4).copy() for k in range(int(hs[0]))]

    fused = False
    if use_dist and B.fused_wanted:
        from small_gicp_b200.distributed import connect_fused

        fused = connect_fused(ctx)
    nccl = use_dist and not fused
    if use_dist:
        dist.barrier()  # the ranks prepared their shards at different speeds: enter the first collective linearize together

    def step_device(k):
        """step k of the schedule, walked like an align(): the identity pose searches unseeded, later poses are seeded by their predecessor"""
        if k % len(poses) == 0:
            ctx.drop_seeds()
        ctx.linearize_device(poses[k % len(poses)], out.data_ptr(), **GICP)
        if nccl:
            dist.all_reduce(out[:44])

    def linearize_host(T):
        ctx.linearize_device(T, out.data_ptr(), **GICP)
        if nccl:
            dist.all_reduce(out[:44])
        h = out[:44].cpu().numpy()
        return h[:36].reshape(6, 6), h[36:42], h[42]

    # the all-rank alignment (informational: where the whole job converges)
    ctx.drop_seeds()
    poses_all, T_final = gn_trajectory(linearize_host)
    rot_err, trans_err = pose_error(inp["T_gt"], T_final)

    barrier = B.barrier
    # ---- value: device-resident inputs, per-step CUDA events, L2 flushed between steps ----
    for i in range(max(args.warmup, len(poses))):
        flush.zero_()
        step_device(i)
    barrier()
    # Clocks: nvidia-smi needs ~0.1 s to start and samples every 0.1 s, the K timed steps take ~10 ms.  The sampler therefore runs
    # over the timed steps PLUS the same step repeated untimed before and after them (identical load, ~0.5 s each side), so that
    # the reported clocks / throttle reasons are those of the GPU under exactly this load.
    sampler = ClockSampler(B.local_rank)
    if rank == 0:
        sampler.start()
        sampler.wait_first_sample(1.5)
    barrier()  # rank 0 waited for the sampler: every rank enters the first collective step of the roll together
    roll_steps = int(min(2000, max(20, 2_000_000_000 // max(1, n_src))))  # the same count on every rank (the step holds a collective)
    roll_steps -= roll_steps % len(poses)
    if os.environ.get("SGB_BENCH_ROLL"):  # profiler runs: a short roll keeps the launch numbering simple (ncu -s / -c)
        roll_steps = max(len(poses), int(os.environ["SGB_BENCH_ROLL"]))

    def load_roll():
        for i in range(roll_steps):
            flush.zero_()
            step_device(i)
            if i % 64 == 63:
                stream.synchronize()  # keep the launch queue short
        barrier()

    load_roll()
    launches0 = ctx.kernel_launches
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    for i in range(args.steps):
        flush.zero_()
        if i % len(poses) == 0:
            ctx.drop_seeds()  # a host-side flag: nothing on the stream
        T = poses[i % len(poses)]
        ev[i][0].record(stream)
        kev[i][0].record(stream)
        ctx.linearize_device(T, out.data_ptr(), **GICP)
        kev[i][1].record(stream)
        if nccl:
            dist.all_reduce(out[:44])
        ev[i][1].record(stream)
    barrier()
    if args.dump_outputs and rank == 0:  # out holds the last timed step's H|b|e|inliers (all-reduced over the ranks)
        h = out[:44].cpu().numpy()
        dump_outputs(args.dump_outputs, h[:36], h[36:42], h[42], h[43])
    launches = ctx.kernel_launches - launches0
    step_ms = np.array([a.elapsed_time(b) for a, b in ev])
    kern_ms = np.array([a.elapsed_time(b) for a, b in kev])
    total_ms = float(step_ms.sum())
    # the same steps grouped by the pose of the schedule they ran at (misaligned first iterations walk the tree, converged ones settle in the grid)
    per_pose = [float(np.mean([kern_ms[i] for i in range(args.steps) if i % len(poses) == k])) if k < args.steps else 0.0 for k in range(len(poses))]
    per_pose_ms = B.max_over_ranks(per_pose)
    # ---- warm-L2 variant (what consecutive optimiser iterations actually see), informational ----
    barrier()
    w0, w1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    w0.record(stream)
    for i in range(args.steps):
        step_device(i)
    w1.record(stream)
    barrier()
    warm_ms = w0.elapsed_time(w1) / args.steps
    load_roll()
    clocks = sampler.stop() if rank == 0 else None
    if clocks is not None:
        clocks["window"] = f"the {args.steps} timed steps + {roll_steps} identical untimed steps before and after them"

    # ---- Reduction::error (LM inner loop): cached correspondences, no search ----
    err_buf = torch.zeros(8, dtype=torch.float64, device=dev)
    ctx.linearize_device(poses[-1], out.data_ptr(), **GICP)
    T_trial = poses[-1] @ se3_exp(np.array([1e-4, -2e-4, 1e-4, 1e-3, 2e-3, -1e-3]))

    def error_step():
        ctx.error_device(T_trial, err_buf.data_ptr())
        if nccl:
            dist.all_reduce(err_buf[:1])

    for _ in range(3):
        error_step()
    error_ms = B.event_ms(error_step, 20)

    # ---- N > 1: the fused exchange against NCCL on the per-rank LOCAL sums; how long the finishing CTAs waited for their peers ----
    allreduce_check, comm_wait = None, None
    if use_dist:
        local, _ = B.context()  # same target / source, not wired to the peers
        local.set_target(inp["target"], None, inp["target_covs"])
        local.build_target_kdtree(args.leaf)
        local.set_source(src_pin.numpy(), cov_pin.numpy())
        out2 = torch.zeros(64, dtype=torch.float64, device=dev)
        worst = 0.0
        for T in (poses[0], poses[-1]):
            ctx.drop_seeds()
            ctx.linearize_device(T, out.data_ptr(), **GICP)
            if nccl:
                dist.all_reduce(out[:44])
            local.linearize_device(T, out2.data_ptr(), **GICP)
            dist.all_reduce(out2[:44])
            a, b = out[:44].cpu().numpy(), out2[:44].cpu().numpy()
            worst = max(worst, float(np.linalg.norm(a[:36] - b[:36]) / np.linalg.norm(b[:36])), float(abs(a[42] - b[42]) / abs(b[42])), float(abs(a[43] - b[43])))
        local.close()
        allreduce_check = B.max_over_ranks([worst])[0]
        if fused:
            for i in range(64):  # fill the ring with steady-state exchanges
                step_device(i)
            barrier()
            ring, calls = ctx.comm_wait_ns()
            waits = torch.from_numpy(ring.astype(np.float64)).to(dev)
            lo_t, hi_t = waits.clone(), waits.clone()
            dist.all_reduce(lo_t, op=dist.ReduceOp.MIN)
            dist.all_reduce(hi_t, op=dist.ReduceOp.MAX)
            lo_h, hi_h = lo_t.cpu().numpy() * 1e-3, hi_t.cpu().numpy() * 1e-3
            comm_wait = {
                "transport_us": float(np.median(lo_h)),
                "skew_us": float(np.median(hi_h - lo_h)),
                "what": "per exchange: ns the finishing CTA of each rank spent between publishing its sums and seeing every peer's flag (%globaltimer); min over ranks = the rank that arrived last = bare mailbox transport over NVLink, max - min = how much earlier the first rank was ready (shard skew); medians over the last 64 exchanges",
                "status": ctx.comm_status(),
            }

    # ---- e2e: host buffers through the C-ABI, H2D of the step's inputs + H|b|e back inside the timed region ----
    def step_e2e(k):
        ctx.set_source(src_pin.numpy(), cov_pin.numpy())  # H2D 160 B / point (reference layout: Vector4d + Matrix4d), pipelined in the library
        if nccl:
            ctx.linearize_device(poses[k % len(poses)], out.data_ptr(), **GICP)
            dist.all_reduce(out[:44])
            return out[:44].cpu().numpy()
        return ctx.linearize(poses[k % len(poses)], **GICP)  # sgb_linearize: H|b|e land in mapped host memory, one stream synchronisation

    for i in range(2):
        step_e2e(i)
    barrier()
    e2e_steps = max(3, min(args.steps, 10))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record(stream)
    for i in range(e2e_steps):
        step_e2e(i)
    e1.record(stream)
    barrier()
    e2e_wall_ms = (time.perf_counter() - t0) * 1e3 / e2e_steps
    e2e_dev_ms = e0.elapsed_time(e1) / e2e_steps
    e2e_ms = max(e2e_wall_ms, e2e_dev_ms)

    # ---- informational: one whole align() through the host-facing calls -- source uploaded ONCE from pinned host memory, then every
    # Gauss-Newton iteration = pose in (128 B), linearize, H|b|e out (352 B) + host solve: what Registration<>::align does with the
    # ParallelReductionCUDA glue, whose device mirror of the source is reused by all iterations of an align() ----
    def align_e2e():
        ctx.set_source(src_pin.numpy(), cov_pin.numpy())
        p, _ = gn_trajectory(linearize_host)
        return len(p)

    align_e2e()
    barrier()
    t0 = time.perf_counter()
    align_reps, align_iters = 3, 0
    for _ in range(align_reps):
        align_iters += align_e2e()
    torch.cuda.synchronize()
    align_ms = (time.perf_counter() - t0) * 1e3 / align_reps
    align_iters //= align_reps

    # ---- max over ranks ----
    total_ms, kern_ms_mean, warm_ms, e2e_ms, align_ms = B.max_over_ranks([total_ms, float(kern_ms.mean()), warm_ms, e2e_ms, align_ms])
    total_points = n_src * world
    ms_per_step = total_ms / args.steps
    value = total_points / (ms_per_step * 1e-3) / 1e6

    cpu_baseline, pose_vs_ref = None, None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        # the SAME arrays (points and covariances) go to the CPU arm
        threads, (_, tc, tt, sc, reg, build_s), trials = best_cpu_registration(inp)
        reps = 0
        t0 = time.perf_counter()
        while reps < 3 or (time.perf_counter() - t0 < 10.0 and reps < len(poses)):
            H0, b0, e0c = reg.linearize(tc, tt, sc, poses[reps % len(poses)])
            reps += 1
        cpu_ms = (time.perf_counter() - t0) / reps * 1e3
        # parity of the sums at the last CPU pose, on the same inputs
        Hg, bg, eg = linearize_host(poses[(reps - 1) % len(poses)])
        cpu_baseline = {
            "value": args.points / (cpu_ms * 1e-3) / 1e6,
            "unit": UNIT,
            "cores": threads,
            "kind": cpu_kind()[0],
            "sample": f"{reps} x linearize over all {args.points} source points at the schedule's poses, SAME input arrays as the GPU arm; " + CPU_NOTE[cpu_kind()[0]],
            "thread_trials": trials,
            "host": host_cpu_info(),
            "ms_per_step": cpu_ms,
            "kdtree_build_s": build_s,
            "parity_rel_H": float(np.linalg.norm(Hg - H0) / np.linalg.norm(H0)),
            "parity_rel_e": float(abs(eg - e0c) / e0c),
        }
        # converged pose of the reference's own Gauss-Newton align on these inputs vs ours (north-star bar: 1e-4 rad / 1e-3 m)
        t0 = time.perf_counter()
        poses_ref, T_ref = gn_trajectory(lambda T: reg.linearize(tc, tt, sc, T))
        rot_r, trans_r = pose_error(T_ref, T_final)
        pose_vs_ref = {"rot_rad": rot_r, "trans_m": trans_r, "gn_iterations_reference": len(poses_ref), "gn_iterations_ours": len(poses_all), "reference_align_s": time.perf_counter() - t0,
                       "what": "converged SE(3) of GaussNewton from identity at the full 1M x 1M size: reference reduction on the host vs this backend, identical input arrays"}

    extras = {}
    if not args.no_extras:
        barrier()
        if fused:
            ctx.comm_disconnect()
        if world == 1:
            try:
                extras["c1"] = run_c1(B)
            except Exception as e:
                extras["c1"] = {"error": repr(e)}
        if world == 1 and args.c3_frames > 1:
            try:
                extras["c3"] = run_c3(B, args.c3_frames)
            except Exception as e:
                extras["c3"] = {"error": repr(e)}
        for key, fn in (("c4", lambda: run_c4(B, args.c4_points)), ("c5", lambda: run_c5(B, [int(x) for x in args.c5_sizes.split(",") if x]))):
            if key == "c4" and args.c4_points <= 0:
                continue
            try:
                extras[key] = fn()
            except Exception as e:  # every rank raises or none: the legs are collective
                extras[key] = {"error": repr(e)}

    if rank == 0:
        peak, peak_src = hbm_peak()
        alg_bytes = BYTES_PER_POINT["GICP"] * n_src
        achieved = alg_bytes / (kern_ms_mean * 1e-3) / 1e9
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "linearize_traffic.json")
        if os.path.exists(tpath):
            try:
                traffic = json.load(open(tpath)).get("dram_bytes_per_launch")
            except Exception:
                traffic = None
        line = {
            "metric": METRIC,
            "value": value,
            "unit": UNIT,
            "n_gpus": world,
            "steps": args.steps,
            "warmup": args.warmup,
            "ms_per_step": ms_per_step,
            "higher_is_better": True,
            "scaling": "weak",
            "vs_baseline": None,
            "dtype": "f32 search / f64 factor algebra + sums",
            "data": "synthetic",
            "config": workload_config(args, inp),
            "allreduce": "none (single GPU)" if not use_dist else "fused into factor_reduce_kernel: peer mailboxes over NVLink (sgb_comm_*)" if fused else "NCCL all_reduce of 44 doubles after the kernel",
            "clocks": clocks,
            "e2e": {
                "value": total_points / (e2e_ms * 1e-3) / 1e6,
                "unit": UNIT,
                "h2d_bytes_per_step": int(n_src * 160 + 128),
                "d2h_bytes_per_step": 44 * 8,
                "ms_per_step": e2e_ms,
                "what": "per step: sgb_source_set_points (pinned host Vector4d + Matrix4d layout; two-stream pipeline: covariance chunks converted while the next one is on the bus) + sgb_linearize (H|b|e written into mapped host memory)",
            },
            "gpu_launches": int(launches),
            "roofline": {
                "bound": "hbm",
                "kernel": "one sgb_linearize = sgb::grid_probe_blocks_kernel + packet_search_kernel (few pending queries: warp-per-query ring search, many: packet walk; picked on the device) + factor_reduce_kernel<2,0>: three launches, timed together",
                "achieved": achieved,
                "peak": peak,
                "peak_source": peak_src,
                "unit": "GB/s",
                "frac": achieved / peak,
                "traffic": traffic,
                "algorithmic_bytes_per_launch": alg_bytes,
                "kernel_ms": kern_ms_mean,
                "launches_per_step": launches / max(1, args.steps),
            },
            "cpu_baseline": cpu_baseline,
            "value_l2_warm": total_points / (warm_ms * 1e-3) / 1e6,
            "pose_schedule": {"poses": len(poses), "source": "Gauss-Newton trajectory of rank 0's own pair (local sums), identical for every N; identity pose unseeded, later poses seeded by their predecessor"},
            "per_pose_ms": per_pose_ms,
            "error_ms": {"value": error_ms, "mpoints_per_s": total_points / (error_ms * 1e-3) / 1e6, "roofline_frac": BYTES_PER_POINT["GICP"] * n_src / (error_ms * 1e-3) / 1e9 / peak,
                         "what": "Reduction::error (LM inner loop): cached correspondences, GICP precision frozen at the linearisation pose, + the all-reduce of 1 double; CUDA events, L2 flushed, max over ranks"},
            "e2e_align": {
                "value": total_points * align_iters / (align_ms * 1e-3) / 1e6,
                "unit": UNIT,
                "ms_per_align": align_ms,
                "gn_iterations": align_iters,
                "h2d_bytes_per_align": int(n_src * 160 + 128 * align_iters),
                "d2h_bytes_per_align": 44 * 8 * align_iters,
                "what": "informational: whole GaussNewton align() through the host-facing calls, wall clock -- source uploaded once (pinned host, reference layout), then per iteration pose in / linearize / H|b|e out / host 6x6 solve; Mpoints/s = points x iterations / time",
            },
            "setup": {"target_build_ms": target_build_ms, "what": "sgb_target_build_kdtree: device kd-tree construction + block lists + hash table, first call (includes allocations)"},
            "pose_error_vs_gt": {"rot_rad": rot_err, "trans_m": trans_err, "gn_iterations": len(poses_all)},
            "pose_error_vs_reference": pose_vs_ref,
            "allreduce_check_rel": allreduce_check,
            "comm_wait_us": comm_wait,
        }
        line.update(extras)
        print(json.dumps(line), flush=True)
    if use_dist:
        dist.barrier()  # nobody unmaps a mailbox a peer may still write to
    ctx.close()
    if use_dist:
        dist.destroy_process_group()
    return 0


def main():
    args = parse_args()
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())

#!/usr/bin/env python
"""bench.py — sliding-window FGO iterations/sec on BASELINE.json cfg 2 (W=20 keyframes, 100k surf pts/scan, 1M-point
local map, scan-to-map surf association + Ceres-semantics dogleg solve + marginalisation of the oldest keyframe), B200 vs
the CPU restatement.

One "step" = one complete optimizeSlidingWindowWithLandMark LiDAR pass (GLIO/src/Estimator.cpp:2046-2608):
  K0 grid build over the local map  ->  K1 association of all W scans  ->  minimizer iterations
  (K2 residual/Jacobian/normal-equation kernel + host factors incl. the previous window's marginalisation prior +
  Cholesky + dogleg) until Ceres' own convergence tests stop it  ->  K3 marginalisation of KF0 (device LiDAR blocks with
  the ambient quaternion columns + host factors -> Schur complement -> eigen-decomposition -> the next window's prior).
The problem has W+1 keyframes: window A = KF 0..W-1 is solved and marginalised once during set-up (its prior is what the
timed window consumes), every timed step is window B = KF 1..W.
metric value = minimizer iterations executed / time, whole job (association and marginalisation amortised into it).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
--dump-outputs DIR writes what the last timed step returned (see dump_outputs) as DIR/<name>.npy, so that two builds can be
compared output for output on identical, seeded inputs.
N>1 is launched by torchrun (one rank per GPU).  The window path does not shard (SURVEY 8e: 20 independent 6x6 blocks and
a 300x300 solve) -> "replicas only": every rank solves the same window; value is the sum over ranks.  The path that DOES
shard - the batch scan-to-multiscan solve, by keyframe, one NCCL all-reduce of the pose-block buffers per evaluation - is
measured in the `batch` object of the same line at every N (BASELINE cfg 3 / cfg 4), and the kNN + Jacobian microbench
(cfg 5) in the `microbench` object.
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True          # the benchmark writes nothing into the tree (it may be read-only)

CFG = dict(W=20, Q=100_000, M=1_000_000)
METRIC = "sliding-window FGO iterations/sec (20 KF, 100k surf pts/scan)"
WORKLOAD = ("cfg2: optimizeSlidingWindow, W=20, Q=100k/scan, M=1M, no selection, prior/IMU-like host factors (15 dims/KF), "
            "previous window's marginalisation prior consumed, KF0 marginalised")
SEED_OFFSET = 2


def xyzi(xyz, fill=0.0):
    """(n,3) float32 -> (n,8) float32 pcl::PointXYZI rows (GLIO/include/utils/common.h:87-89): x y z 1 | intensity pad pad pad."""
    out = np.full((len(xyz), 8), fill, np.float32)
    out[:, :3] = xyz
    out[:, 3] = 1.0
    return out


def build_problem():
    """W+1 keyframes (two overlapping windows), the cfg-2 map, and the host factor spec of the whole chain."""
    from glio_b200 import synth
    P = synth.window_problem(W=CFG["W"] + 1, Q=CFG["Q"], M=CFG["M"], seed=synth.SEED0 + SEED_OFFSET)
    rng = np.random.default_rng(1)
    T = P["poses_true"]; K = len(T)
    sw = np.concatenate([np.full(3, 20.0), np.full(3, 50.0), np.full(9, 5.0)])
    spec = dict(prior=(0, T[0, :3].copy(), T[0, 3:].copy(), np.zeros(9), sw), between=[])
    for i in range(K - 1):
        dq = synth.quat_mul(synth.quat_conj(T[i, 3:]), T[i + 1, 3:])
        dp = synth.quat_to_R(T[i, 3:]).T @ (T[i + 1, :3] - T[i, :3])
        spec["between"].append((i, i + 1, dp + rng.normal(0, 0.01, 3), dq, np.zeros(3), 0.1, sw * 0.5))
    return P, spec


def window_factors(spec, first, W):
    """Factors of the window KF first..first+W-1, renumbered from 0: the stand-in prior only when KF0 of the chain is in it."""
    prior = spec["prior"] if first == 0 else None
    between = [(i - first, j - first) + tuple(rest) for (i, j, *rest) in spec["between"] if first <= i and j < first + W]
    return prior, between


def dump_outputs(out_dir, match_counts, r, prior):
    """Writes what one window step returns to its caller as float64 arrays, out_dir/<name>.npy: the association's match count
    per keyframe, the solve's poses, speed-biases, accepted steps, per-iteration log and summary counters (not its timings),
    and the marginalisation prior handed to the next window.  Under 2 MB at cfg 2: the largest are the prior's two n x n
    matrices, n <= 15 W."""
    from glio_b200 import api
    out = dict(match_counts=match_counts, poses=r["poses"], speed_bias=r["speed_bias"], steps=r["steps"])
    for name, _ in api.Iteration._fields_:
        if name != "reserved":
            out["iteration_" + name] = [it[name] for it in r["iterations"]]
    s = r["summary"]
    for name in ("termination", "num_iterations", "num_successful_steps", "num_unsuccessful_steps", "num_evaluations",
                 "num_jacobian_evaluations", "num_linear_solves", "num_valid_steps", "initial_cost", "final_cost"):
        out["summary_" + name] = getattr(s, name)
    pa = prior.arrays()
    for name in ("lin_jac", "lin_res", "x0_pose", "x0_sb", "A_info", "b_info"):
        out["prior_" + name] = pa[name]
    os.makedirs(out_dir, exist_ok=True)
    for name, v in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(v, np.float64))


class ClockSampler:
    """SM clock / throttle reasons sampled DURING the timed region through NVML, from the timing thread itself at step
    boundaries (about five reads per run; one read stalls the launch queue for up to ~0.5 ms and is inside the timed region).  Polling from
    outside — an `nvidia-smi -lms` subprocess or a concurrent NVML thread — was measured to stall this workload's
    many short launches by milliseconds per step."""

    def __init__(self, dev_index):
        self.samples = []; self.reasons = set(); self.max_mhz = None; self.ok = False; self.cost_ms = 0.0
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nv = pynvml
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[dev_index]) if vis and all(v.strip().isdigit() for v in vis.split(",")) else dev_index
            self._h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM))
            nv = pynvml
            self._names = {"hw_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
                           "hw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
                           "sw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
                           "sw_power_cap": getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4)}
            self.ok = True
        except Exception:
            self.ok = False

    def sample(self):
        if not self.ok:
            return
        t0 = time.perf_counter()
        try:
            nv = self._nv
            self.samples.append(float(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM)))
            r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self._h)
            for k, bit in self._names.items():
                if r & bit:
                    self.reasons.add(k)
        except Exception:
            pass
        self.cost_ms += 1e3 * (time.perf_counter() - t0)

    def reset(self):
        self.samples = []; self.reasons = set(); self.cost_ms = 0.0

    def result(self):
        return dict(sm_mhz=float(np.median(self.samples)) if self.samples else None, sm_max_mhz=self.max_mhz,
                    reasons=sorted(self.reasons), samples=len(self.samples), sampling_cost_ms=round(self.cost_ms, 3),
                    how="NVML, read inside the timed region at step boundaries (three reads: first, middle, last step); sampling_cost_ms is the host time of those reads, which IS part of the timed region")


# ----------------------------------------------------------------------------------------------------------
# CPU arm: the oracle (port of the reference path) on host cores
# ----------------------------------------------------------------------------------------------------------
def cpu_window_pass(P, spec, first, prior, nthreads, q_sub=1, tree=None):
    """One full reference-style window pass on the CPU oracle: setInputCloud, association of the W scans, problem assembly,
    ceres::Solve, marginalisation.  Returns (iterations, seconds, detail, solve result, prior dict)."""
    from oracle import pyoracle as po
    from glio_b200 import synth
    W = CFG["W"]
    t0 = time.perf_counter()
    tree = tree if tree is not None else po.KdTree(P["map_xyz"])          # setInputCloud (Estimator.cpp:2056)
    t_tree = time.perf_counter() - t0
    ks = list(range(first, first + W))
    poses0 = P["poses_init"][ks]
    prob = po.WindowProblem(poses0, np.zeros((W, 9)), P["q_lb"], P["t_lb"], huber_delta=1.0)
    nres = 0
    for i, k in enumerate(ks):
        t2, q2 = synth.lidar_pose_in_world(poses0[i, :3], poses0[i, 3:])
        scan = P["scans"][k][::q_sub]
        o = po.assoc_scan_to_map(P["map_xyz"], scan, t2, q2, tree=tree, nthreads=nthreads)   # Estimator.cpp:2222
        v = o["status"] == po.GO_VALID
        prob.add_unary(np.full(int(v.sum()), i, np.int32), scan[v], o["nsd"][v], o["score"][v])
        nres += int(v.sum())
    t_assoc = time.perf_counter() - t0 - t_tree
    pr, between = window_factors(spec, first, W)
    if pr is not None:
        prob.add_prior(*pr)
    for b in between:
        prob.add_between(*b)
    prob.set_marg_prior(prior)
    r = prob.solve(po.solver_options(), mode=0, nthreads=nthreads)       # ceres::Solve (Estimator.cpp:2433)
    t_solve = time.perf_counter() - t0 - t_tree - t_assoc
    prob.reset_state(r["poses"], r["speed_bias"])
    m = prob.marginalize(eps=1e-8, mode=0)                               # Estimator.cpp:2462-2608
    dt = time.perf_counter() - t0
    iters = len(r["steps"])
    detail = dict(kdtree_s=round(t_tree, 3), assoc_s=round(t_assoc, 3), solve_s=round(t_solve, 3), marg_s=round(dt - t_tree - t_assoc - t_solve, 3), residuals=nres)
    newp = dict(W=W, lin_jac=m["lin_jac"], lin_res=m["lin_res"], x0_pose=m["x0_pose"], x0_sb=m["x0_sb"])
    return iters, dt, detail, r, newp


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU implementation of the path (the oracle port: Eigen/Ceres/PCL are absent
    from this image so oracle/_ref cannot be built — DESIGN.md) on all host threads."""
    if rank != 0:
        return
    from oracle import pyoracle as po
    cores = os.cpu_count() or 1
    P, spec = build_problem()
    q_sub = args.ref_subsample
    # set-up (untimed): window A -> the prior the timed window consumes
    _, _, _, _, priorA = cpu_window_pass(P, spec, 0, None, cores, q_sub)
    tot_it, tot_t, detail = 0, 0.0, None
    for s in range(args.warmup + args.steps):
        it, dt, detail, _, _ = cpu_window_pass(P, spec, 1, priorA, cores, q_sub)
        if s >= args.warmup:
            tot_it += it; tot_t += dt
    value = tot_it / tot_t
    line = dict(impl="reference", metric=METRIC, value=value, unit="iterations/s", n_gpus=args.gpus, steps=args.steps, warmup=args.warmup,
                ms_per_step=1e3 * tot_t / args.steps, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f64",
                data="synthetic", config=dict(workload=WORKLOAD, **CFG),
                cpu_baseline=dict(value=value, unit="iterations/s", cores=cores, kind="port",
                                  sample=f"full window pass per step (kd-tree build on the 1M map + association + solve + marginalisation) with every {q_sub}-th scan point; {detail}"),
                e2e=dict(value=value, unit="iterations/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0), gpu_launches=0)
    print(json.dumps(line))


# ----------------------------------------------------------------------------------------------------------
# batch (scan-to-multiscan) path: the one that shards by keyframe (BASELINE cfg 3 / cfg 4)
# ----------------------------------------------------------------------------------------------------------
def batch_run(torch, dist, local_rank, rank, world, K, Q, sr=6, solves=2, max_iter=100, check_against_single=False):
    """Keyframe-sharded optimizeBatchWithLandMark LiDAR part (Estimator.cpp:2739-3410): association of this rank's pairs,
    then the solve with one NCCL all-reduce of the pose-block buffers per evaluation.  Device-event times, max over ranks."""
    from glio_b200 import api, dist as gdist, synth
    cur, oth = gdist.batch_pairs(K, sr)
    own = gdist.owner_of(cur, K, world) == rank
    need = gdist.frames_needed(cur, oth, own)
    B = synth.batch_problem(K=K, Q=Q, search_range=sr, frames=need)
    ctx = api.Context(local_rank)
    hook = None
    if world > 1:
        hook = gdist.NcclHook(rank, world); hook.install(ctx)
    st = torch.cuda.ExternalStream(ctx.stream)

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
    dscans = {int(k): torch.from_numpy(B["scans"][k]).cuda() for k in need}
    for k in need:
        ctx.batch_set_frame(int(k), dscans[int(k)], B["poses_init"][k])
    ctx.batch_declare_pairs(cur, oth)
    ctx.batch_associate_pairs(cur[own], oth[own]); sync_all()                  # warm-up (allocations)
    for k in need:
        ctx.batch_set_pose(int(k), B["poses_init"][k])                          # invalidate the grids: the timed pass rebuilds them
    sync_all(); e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    e0.record(st); nm = ctx.batch_associate_pairs(cur[own], oth[own]); e1.record(st); sync_all()
    t_assoc = torch.tensor([e0.elapsed_time(e1)], device="cuda")
    nres = torch.tensor([float(nm.sum())], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t_assoc, op=dist.ReduceOp.MAX); dist.all_reduce(nres)
    hf = api.HostFactorSet(); T = B["poses_true"]; rng = np.random.default_rng(7)
    sw = np.concatenate([np.full(3, 10.0), np.full(3, 30.0), np.zeros(9)])
    hf.add_prior(0, T[0, :3], T[0, 3:], None, sw * 3)
    for i in range(K - 1):
        dq = synth.quat_mul(synth.quat_conj(T[i, 3:]), T[i + 1, 3:]); dp = synth.quat_to_R(T[i, 3:]).T @ (T[i + 1, :3] - T[i, :3])
        hf.add_between(i, i + 1, dp + rng.normal(0, 0.005, 3), dq, np.zeros(3), 0.1, sw)
    opt = api.batch_solver_options(max_num_iterations=max_iter)
    r = ctx.batch_solve(B["poses_init"], None, hf, opt)                         # warm-up
    sync_all(); e0.record(st); iters = 0
    for _ in range(solves):
        r = ctx.batch_solve(B["poses_init"], None, hf, opt); iters += len(r["steps"])
    e1.record(st); sync_all()
    t_solve = torch.tensor([e0.elapsed_time(e1)], device="cuda")
    if world > 1:
        dist.all_reduce(t_solve, op=dist.ReduceOp.MAX)
    ar_us = None
    if world > 1:                                                               # latency of the two block buffers alone
        Pn = len(cur); b1 = torch.zeros(K * 28, dtype=torch.float64, device="cuda"); b2 = torch.zeros(Pn * 36, dtype=torch.float64, device="cuda")
        for _ in range(5):
            dist.all_reduce(b1); dist.all_reduce(b2)
        torch.cuda.synchronize(); f0 = torch.cuda.Event(enable_timing=True); f1 = torch.cuda.Event(enable_timing=True)
        f0.record()
        for _ in range(30):
            dist.all_reduce(b1); dist.all_reduce(b2)
        f1.record(); torch.cuda.synchronize(); ar_us = f0.elapsed_time(f1) / 30 * 1e3
    s = r["summary"]
    out = dict(workload="optimizeBatch sms_fusion_level=1 scan-to-multiscan, keyframe-sharded", K=K, Q=Q, search_range=sr, n_gpus=world, pairs=int(len(cur)),
               queries=int(len(cur)) * Q, residuals=float(nres.item()), assoc_ms=float(t_assoc.item()), solve_ms=float(t_solve.item()) / solves,
               iterations=iters / solves, evaluations=int(s.num_evaluations), allreduce_us_per_eval=ar_us,
               linear_solver_ms=1e3 * s.linear_solver_seconds, eval_ms=1e3 * s.eval_seconds,
               final_cost=float(s.final_cost), initial_cost=float(s.initial_cost), termination=s.message.decode())
    if hook:
        ctx.set_allreduce(api.C.cast(None, api.ALLREDUCE_FN), None)
    final_poses = r["poses"].copy()
    ctx.close()
    if hook:
        hook.close()
    if check_against_single and world > 1:
        # the same problem on ONE GPU, no hook (rank 0 only; the others wait): the only place a multi-GPU product test can run
        # under the driver
        ok = True; detail = None
        if rank == 0:
            Bf = synth.batch_problem(K=K, Q=Q, search_range=sr)
            c1 = api.Context(local_rank)
            ds = [torch.from_numpy(Bf["scans"][k]).cuda() for k in range(K)]
            for k in range(K):
                c1.batch_set_frame(k, ds[k], Bf["poses_init"][k])
            nm1 = c1.batch_associate_pairs(cur, oth)
            r1 = c1.batch_solve(Bf["poses_init"], None, hf, opt)
            s1 = r1["summary"]
            dpos = float(np.max(np.abs(r1["poses"][:, :3] - final_poses[:, :3]))); dq = float(np.max(np.abs(r1["poses"][:, 3:] - final_poses[:, 3:])))
            detail = dict(single_gpu_final_cost=float(s1.final_cost), single_gpu_iterations=len(r1["steps"]), single_gpu_residuals=float(nm1.sum()),
                          max_pose_diff_m=dpos, max_quat_diff=dq)
            ok = (float(nm1.sum()) == out["residuals"] and len(r1["steps"]) == int(round(out["iterations"]))
                  and abs(s1.final_cost - out["final_cost"]) <= 1e-9 * abs(s1.final_cost) and dpos <= 1e-7 and dq <= 1e-9)
            c1.close()
        flag = torch.tensor([1.0 if ok else 0.0], device="cuda")
        dist.broadcast(flag, 0)
        out["equals_single_gpu"] = bool(flag.item() > 0.5)
        out["single_gpu_check"] = detail
        assert out["equals_single_gpu"], f"sharded batch solve differs from the single-GPU solve: {detail} vs {out}"
    return out


def microbench_run(torch, dist, local_rank, rank, world, peak, steps=10):
    """BASELINE cfg 5: K0 + K1 + K2 over a 1M-point map and 100k queries (sharded Q/N, map replicated), one pose."""
    from glio_b200 import api, synth
    M, Q = 1_000_000, 100_000
    P = synth.window_problem(W=1, Q=Q, M=M, seed=synth.SEED0 + 5)
    lo, hi = rank * Q // world, (rank + 1) * Q // world
    ctx = api.Context(local_rank)
    st = torch.cuda.ExternalStream(ctx.stream)
    dmap = torch.from_numpy(xyzi(P["map_xyz"])).cuda(); dscan = torch.from_numpy(xyzi(P["scans"][0][lo:hi])).cuda()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    blk = torch.zeros(28, dtype=torch.float64, device="cuda")
    pose = P["poses_init"][:1]

    def one_pass():
        ctx.set_map(dmap)
        ctx.window_set_scans([dscan]); nm = ctx.window_associate(pose)
        r = ctx.eval_unary(pose)
        if world > 1:
            blk.copy_(torch.from_numpy(np.concatenate([r["H"].reshape(-1)[:21], r["g"].reshape(-1), r["cost"]])), non_blocking=True)
            dist.all_reduce(blk)
        return int(nm[0])
    for _ in range(3):
        one_pass()
    ts = []
    for _ in range(steps):
        with torch.cuda.stream(st):
            flush.zero_()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record(st); n = one_pass(); e1.record(st); torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    t = torch.tensor([float(np.median(ts))], device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ctx.lib_profile(True)
    for _ in range(3):
        one_pass()
    ctx.synchronize(); prof = ctx.lib_profile_read(); ctx.lib_profile(False)
    ctx.close()
    byts = 12.0 * M + 172.0 * Q / world
    ms = float(t.item())
    kern = {k: round(v[0] / v[1], 4) for k, v in prof.items()}
    k1 = sum(v for k, v in kern.items() if k.startswith("k_knn") or k.startswith("k_plane"))
    return dict(workload="cfg5: kNN + point-to-plane Jacobian microbench, M=1M map, Q=100k queries (sharded Q/N, map replicated)", n_gpus=world,
                queries_per_gpu=hi - lo, pass_ms=ms, queries_per_s=Q / (ms * 1e-3), algorithmic_bytes_per_gpu=byts,
                achieved_GBps_per_gpu=byts / (ms * 1e-3) / 1e9, frac_of_measured_hbm=byts / (ms * 1e-3) / 1e9 / peak,
                kernel_ms_sum=round(sum(kern.values()), 4), knn_plus_fit_ms=round(k1, 4), kernels_ms=kern, matches_rank0=n,
                l2="256 MB flush before every pass", timing="CUDA events on the library stream, median, max over ranks")


# ----------------------------------------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------------------------------------
def share_of_cpus(cpus, n_share, idx, siblings=None):
    """The idx-th of n_share disjoint parts of `cpus`, whole physical cores at a time (siblings: cpu -> iterable of the hardware
    threads of its core).  Ranks whose GPUs hang off the same socket get disjoint cores, so one rank's worker thread can never
    wake onto a core where another rank's launching thread spins."""
    cpus = set(cpus)
    if n_share <= 1 or len(cpus) < 2 * n_share:
        return cpus
    cores, seen = [], set()
    for c in sorted(cpus):
        if c in seen:
            continue
        core = {c} | ({int(x) for x in siblings(c)} & cpus if siblings else set())
        seen |= core; cores.append(sorted(core))
    if len(cores) < n_share:
        return cpus
    lo, hi = idx * len(cores) // n_share, (idx + 1) * len(cores) // n_share
    return {c for core in cores[lo:hi] for c in core} or cpus


def _thread_siblings(cpu):
    with open(f"/sys/devices/system/cpu/cpu{cpu}/topology/thread_siblings_list") as f:
        out = []
        for part in f.read().strip().split(","):
            a, _, b = part.partition("-")
            out.extend(range(int(a), int(b or a) + 1))
        return out


def bind_to_gpu_numa_node(local_rank, n_local=1):
    """One process per GPU, pinned to CPUs NVML reports as local to that GPU: the step is a chain of short launches and host-side
    waits on pinned memory, and a rank that floats to the other socket pays a remote hop on every one of them.  Ranks that share
    a socket split its physical cores between them (share_of_cpus).  Returns the number of CPUs the process is bound to."""
    try:
        import pynvml
        pynvml.nvmlInit()
        nwords = (os.cpu_count() + 63) // 64
        vis = [v.strip() for v in os.environ.get("CUDA_VISIBLE_DEVICES", "").split(",") if v.strip()]

        def cpus_of(i):
            j = int(vis[i]) if i < len(vis) and vis[i].isdigit() else i          # NVML numbers the physical devices
            words = pynvml.nvmlDeviceGetCpuAffinity(pynvml.nvmlDeviceGetHandleByIndex(j), nwords)
            return frozenset(64 * k + b for k, w in enumerate(words) for b in range(64) if (w >> b) & 1)
        mine = cpus_of(local_rank)
        cpus = set(mine) & os.sched_getaffinity(0)
        if not cpus:
            return None
        try:
            peers = [i for i in range(max(n_local, 1)) if cpus_of(i) == mine]
            if local_rank in peers and len(peers) > 1:
                cpus = share_of_cpus(cpus, len(peers), peers.index(local_rank), _thread_siblings)
        except Exception:
            pass
        os.sched_setaffinity(0, cpus)
        return len(cpus)
    except Exception:
        pass
    return None


def run_glio(args, rank, world, local_rank):
    n_bound = bind_to_gpu_numa_node(local_rank, world)
    import torch
    from glio_b200 import api
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    P, spec = build_problem()                      # the SAME problem on every rank (replicas): per-rank work is identical
    W = CFG["W"]
    ctx = api.Context(local_rank)
    sb0 = np.zeros((W, 9))
    st = torch.cuda.ExternalStream(ctx.stream)
    posesA, posesB = P["poses_init"][:W], P["poses_init"][1:W + 1]
    # inputs in the reference's own layout (pcl::PointXYZI, 32 B per point): resident copies (value) and pinned host copies (e2e)
    map8 = xyzi(P["map_xyz"]); scans8 = [xyzi(s) for s in P["scans"]]
    dmap = torch.from_numpy(map8).cuda(); dscans = [torch.from_numpy(s).cuda() for s in scans8]
    pmap = torch.from_numpy(map8).pin_memory(); hmap = pmap.numpy()
    pnew = torch.from_numpy(scans8[W]).pin_memory(); hnew = pnew.numpy()          # the newest keyframe's scan (KF W)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")
    opts = api.default_solver_options()

    def factor_set(first, prior):
        hf = api.HostFactorSet()
        pr, between = window_factors(spec, first, W)
        if pr is not None:
            hf.add_prior(*pr)
        for b in between:
            hf.add_between(*b)
        hf.set_marg_prior(prior)
        return hf
    # ---- set-up: window A (KF 0..W-1), untimed -> the prior that every timed window consumes
    hfA = factor_set(0, None)
    ctx.set_map(dmap); ctx.window_set_scans(dscans[:W]); ctx.window_associate(posesA)
    rA = ctx.window_solve(posesA, sb0, hfA, opts, band=29)
    priorA = ctx.window_marginalize(rA["poses"], rA["speed_bias"], hfA)
    hfB = factor_set(1, priorA)
    band = max(29, hfB.marg_half_bandwidth())

    # The marginalisation's host half (Schur, decomposition, prior: ~0.15 ms) runs on the library's worker thread while the NEXT
    # step's map and association are on the GPU (glio_window_marginalize_async); the job is joined right before the solve that
    # would consume its prior, and the last one before the timed region ends: K steps contain K complete marginalisations.
    pipelined = not args.sync_marg

    class Done:                                      # a finished "job" for the synchronous variant
        def __init__(self, prior): self.prior = prior
        def wait(self): return self.prior

    def one_step(m, pending=None):
        ctx.set_map(m)
        nm = ctx.window_associate(posesB)
        if pending is not None:
            pending.wait()                           # the previous window's prior is complete before this solve starts
        r = ctx.window_solve(posesB, sb0, hfB, opts, band=band)
        job = ctx.window_marginalize_async(r["poses"], r["speed_bias"], hfB) if pipelined else Done(ctx.window_marginalize(r["poses"], r["speed_bias"], hfB))
        return len(r["steps"]), r, job, nm

    step_wall = {}

    def timed_run(nsteps, sampler=None):
        """Returns (iterations, device ms, wall s, what the last step returned: match counts, solve result, prior)."""
        iters = 0
        marks = {0, nsteps // 2, nsteps - 1}            # three NVML reads per run: a read stalls the launch queue for 0.5 - 4 ms depending on the box
        ctx.window_set_scans(dscans[1:W + 1])
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record(st)
        tick = [t0]
        job = None
        for si in range(nsteps):
            with torch.cuda.stream(st):
                flush.fill_(1)                      # L2 flush between steps (256 MB > 126 MB L2), inside the timed region
            it, r, job, nm = one_step(dmap, job)
            iters += it
            if sampler is not None and si in marks:
                sampler.sample()
            tick.append(time.perf_counter())
        prior = job.wait()                          # the last marginalisation completes inside the timed region
        e1.record(st)
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        ms = max(e0.elapsed_time(e1), 0.0)
        if dist is not None:
            dist.barrier()
        per = np.diff(np.array(tick)) * 1e3
        after = [per[i + 1] for i in sorted(marks) if sampler is not None and i + 1 < nsteps]
        step_wall.clear()
        step_wall.update(p50=round(float(np.median(per)), 4), mean=round(float(per.mean()), 4), max=round(float(per.max()), 4), argmax=int(per.argmax()), all=[round(float(v), 3) for v in per],
                         mean_of_steps_after_an_nvml_read=round(float(np.mean(after)), 4) if after else None)
        return iters, ms, wall, (nm, r, prior)

    # NVML is initialised and queried during the warm-up steps: the first query of a process can stall the GPU work queue for
    # tens of milliseconds on some boxes (measured: a fixed ~85 ms once per process), which must not land in the timed region.
    sampler = ClockSampler(local_rank) if rank == 0 else None
    ctx.window_set_scans(dscans[1:W + 1])
    for _ in range(max(args.warmup, 3)):                # warm-up steps are the timed step verbatim (flush included: the first launch
        with torch.cuda.stream(st):                    # of torch's fill kernel loads its module lazily, 5 - 20 ms once per process)
            flush.fill_(1)
        one_step(dmap)[2].wait()
        if sampler is not None:
            sampler.sample()
    if sampler is not None:
        sampler.reset()
    # (A) the reported value: K steps, inputs resident in HBM, no per-kernel instrumentation
    l0 = ctx.launch_count
    iters, ms, wall, last = timed_run(args.steps, sampler)
    launches = ctx.launch_count - l0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, *last)
    step_wall_value = dict(step_wall)
    clocks = sampler.result() if sampler else None
    # (B) the same K steps again with every kernel launch bracketed by CUDA events on the launching stream: the
    #     per-kernel durations the roofline uses (its step time is reported next to the value for transparency)
    ctx.lib_profile(True)
    ctx.knn_fallback_queries(reset=True)
    _, ms_prof, _, _ = timed_run(args.steps)
    prof = ctx.lib_profile_read()
    n_fallback = ctx.knn_fallback_queries()
    ctx.lib_profile(False)

    # (C) end to end through the C ABI with pinned HOST buffers in the reference's PointXYZI layout.  A sliding window gets ONE
    #     new keyframe per call: every step uploads the rebuilt local map (32 MB; it depends on the poses the previous solve
    #     produced, so its upload can only start when that solve has returned: it runs on the copy stream during the
    #     marginalisation of the previous window and the rest is waited for in line) and the newest keyframe's scan (3.2 MB, copy stream, handed over right
    #     after the association of the current window - the order a live system has: the next keyframe's cloud arrives while
    #     the current window is optimised); the other W-1 scans are resident, as they are after glio_window_slide.
    def timed_run_e2e(nsteps):
        iters = 0
        ctx.window_set_scans(dscans[1:W + 1])
        ctx.window_set_scan(W - 1, hnew)
        ctx.map_prefetch(hmap)                      # prologue upload of the first map (outside the timed region, like the first scan)
        if dist is not None:
            dist.barrier()
        ctx.synchronize(); torch.cuda.synchronize()
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record(st)
        job = None
        for si in range(nsteps):
            with torch.cuda.stream(st):
                flush.fill_(1)
            ctx.set_map(hmap)
            ctx.window_associate(posesB)
            ctx.window_set_scan(W - 1, hnew)        # next step's new keyframe: asynchronous, copy stream
            if job is not None:
                job.wait()
            r = ctx.window_solve(posesB, sb0, hfB, opts, band=band)
            ctx.map_prefetch(hmap)                  # the poses are final: the next window's rebuilt map starts its upload (copy stream)
            job = ctx.window_marginalize_async(r["poses"], r["speed_bias"], hfB) if pipelined else Done(ctx.window_marginalize(r["poses"], r["speed_bias"], hfB))
            iters += len(r["steps"])
        job.wait()
        ctx.synchronize()                           # both streams: the last uploads are inside the timed region too
        e1.record(st)
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        ms = max(e0.elapsed_time(e1), 0.0)
        if dist is not None:
            dist.barrier()
        return iters, ms, wall

    timed_run_e2e(2)
    iters_e, ms_e, wall_e = timed_run_e2e(args.steps)
    # wall-clock split of one resident step (every call ends synchronised, so these add up to the step)
    ctx.window_set_scans(dscans[1:W + 1])
    split = {}
    for _ in range(3):
        torch.cuda.synchronize(); tf = time.perf_counter()
        with torch.cuda.stream(st):
            flush.fill_(1)
        torch.cuda.synchronize()
        t0 = time.perf_counter(); ctx.set_map(dmap); t1 = time.perf_counter()
        ctx.window_associate(posesB); t2 = time.perf_counter(); rs = ctx.window_solve(posesB, sb0, hfB, opts, band=band); t3 = time.perf_counter()
        ctx.window_marginalize(rs["poses"], rs["speed_bias"], hfB); t4 = time.perf_counter()
        split = dict(l2_flush_ms=round(1e3 * (t0 - tf), 3), set_map_ms=round(1e3 * (t1 - t0), 3), associate_ms=round(1e3 * (t2 - t1), 3),
                     solve_ms=round(1e3 * (t3 - t2), 3), marginalize_ms=round(1e3 * (t4 - t3), 3))
    _, rlast, jlast, _ = one_step(dmap)
    plast = jlast.wait()

    tmax, tmax_e, it_sum, it_sum_e = ms, ms_e, iters, iters_e
    per_rank = [[ms / args.steps, ms_e / args.steps]]
    if dist is not None:
        t = torch.tensor([ms, ms_e], device="cuda"); dist.all_reduce(t, op=dist.ReduceOp.MAX); tmax, tmax_e = t.tolist()
        mine = torch.tensor([ms / args.steps, ms_e / args.steps], device="cuda"); allr = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(allr, mine); per_rank = [[round(float(v), 4) for v in a.tolist()] for a in allr]
        c = torch.tensor([iters, iters_e], device="cuda", dtype=torch.float64); dist.all_reduce(c); it_sum, it_sum_e = c.tolist()
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0)); peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if peaks else "fallback 6650 GB/s"
    residuals = int(sum(ctx.get_match_counts(W)))
    ctx.close()

    # ---- the paths that shard / the microbench, every rank takes part (collectives inside) ----
    batch = None; micro = None
    if not args.no_batch:
        try:
            batch = dict(strong_scaling_K400=batch_run(torch, dist, local_rank, rank, world, K=args.batch_k, Q=CFG["Q"], solves=2,
                                                       check_against_single=True))
            if world == 1 and not args.no_cfg4:          # BASELINE configs[2]: K = 200 keyframes on one GPU
                batch["cfg3_K200"] = batch_run(torch, dist, local_rank, rank, world, K=200, Q=CFG["Q"], solves=2)
            if world >= 8 and not args.no_cfg4:
                batch["cfg4_K2000"] = batch_run(torch, dist, local_rank, rank, world, K=2000, Q=CFG["Q"], solves=1, max_iter=20)
        except AssertionError:
            raise
        except Exception as e:                       # a failure here must not lose the headline line
            batch = dict(error=repr(e)[:300])
    if not args.no_microbench:
        try:
            micro = microbench_run(torch, dist, local_rank, rank, world, peak)
        except Exception as e:
            micro = dict(error=repr(e)[:300])
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return
    value = it_sum / (tmax * 1e-3)
    e2e = it_sum_e / (tmax_e * 1e-3)
    # roofline of the dominant kernel (K1 association): algorithmic bytes = 116*Qt + 12*M per launch (SURVEY 8d)
    Qt = CFG["W"] * CFG["Q"]
    kern = {}
    for name, (tot_ms, cnt) in prof.items():
        kern[name] = dict(ms_total=round(tot_ms, 4), launches=cnt, ms_avg=round(tot_ms / max(cnt, 1), 5))
    roof = None
    knn_names = ("k_knn_search", "k_knn_deferred", "k_knn_thread", "k_knn_box", "k_knn_tile", "k_knn_tile2", "k_knn_team", "k_knn_box_start", "k_knn_grow", "k_knn_box_far", "k_knn_far", "k_knn_box_cells")
    if any(k in prof for k in knn_names) and "k_plane_fit" in prof:
        # K1 is one association pass issued as two launches (exact 5-NN search, then the fp64 plane fit)
        used = [k for k in knn_names + ("k_plane_fit",) if k in prof and prof[k][1]]
        avg_ms = sum(prof[k][0] / prof[k][1] for k in used)
        alg = 116.0 * Qt + 12.0 * CFG["M"]
        ach = alg / (avg_ms * 1e-3) / 1e9
        # DRAM traffic of the same kernels from the committed ncu --set full captures (bytes per launch, cfg 2 sizes)
        traffic, traffic_src, issue = None, None, None
        try:
            tj = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
            if all(k in tj for k in used):
                traffic = float(sum(tj[k]["dram_bytes"] for k in used)); traffic_src = tj.get("_source")
                kb = tj.get("k_knn_box")
                if kb and "k_knn_box" in used:
                    issue = dict(kernel="k_knn_box", warp_instructions=kb["warp_inst"], issue_active_pct=kb["issue_active_pct"], active_threads_per_instruction=kb["threads_per_inst"],
                                 note="the association pass is bound by instruction issue, not HBM: see DESIGN.md section 4")
        except Exception:
            pass
        roof = dict(bound="hbm", kernel="K1 association pass = " + " + ".join(used) + " (exact 5-NN + plane fit + gates)",
                    achieved=round(ach, 2), peak=peak, unit="GB/s", frac=round(ach / peak, 5), traffic=traffic, algorithmic_bytes=alg,
                    avg_ms=round(avg_ms, 5), peak_source=peak_src, traffic_source=traffic_src, issue_bound_evidence=issue)
    if "k_eval_unary" in prof and prof["k_eval_unary"][1] > 0:
        avg_ms2 = prof["k_eval_unary"][0] / prof["k_eval_unary"][1]
        kern["k_eval_unary"]["achieved_GBps"] = round(32.0 * residuals / (avg_ms2 * 1e-3) / 1e9, 2)
        kern["k_eval_unary"]["frac_of_peak"] = round(kern["k_eval_unary"]["achieved_GBps"] / peak, 5)
        kern["k_eval_unary"]["residuals"] = residuals
    # CPU baseline (oracle port), 1 thread = the reference's own setting (options.num_threads = 1, Estimator.cpp:2426), and the
    # full-size parity check of the GPU arm against that very pass
    cpu = None; parity = None
    if not args.no_cpu_baseline and world == 1:
        from oracle import pyoracle as po
        q_sub = args.cpu_subsample
        cores = os.cpu_count() or 1
        tree = po.KdTree(P["map_xyz"])
        _, _, _, _, opriorA = cpu_window_pass(P, spec, 0, None, cores, q_sub, tree=tree)        # set-up for the timed pass (untimed, all threads)
        it_c, dt_c, det, ro, opriorB = cpu_window_pass(P, spec, 1, opriorA, 1, q_sub)
        cpu = dict(value=it_c / dt_c, unit="iterations/s", cores=1, kind="port",
                   sample=f"one full window pass (kd-tree build on the 1M map + association + solve + marginalisation) with every {q_sub}-th scan point; {det}")
        if q_sub == 1:
            a, b = rlast["steps"], ro["steps"]
            same_n = rlast["summary"].num_iterations == ro["summary"].num_iterations and len(a) == len(b)
            dt_max = max((float(np.max(np.abs(x.reshape(W, 15)[:, :3] - y.reshape(W, 15)[:, :3]))) for x, y in zip(a, b)), default=0.0)
            dr_max = max((float(np.max(2 * np.linalg.norm(x.reshape(W, 15)[:, 3:6] - y.reshape(W, 15)[:, 3:6], axis=1))) for x, y in zip(a, b)), default=0.0)
            dp = float(np.max(np.abs(rlast["poses"][:, :3] - ro["poses"][:, :3]))); dq = float(np.max(np.abs(rlast["poses"][:, 3:] - ro["poses"][:, 3:])))
            pa = plast.arrays()
            JtJ = opriorB["lin_jac"].T @ opriorB["lin_jac"]; Jtr = opriorB["lin_jac"].T @ opriorB["lin_res"]
            d_info = float(np.max(np.abs(pa["A_info"] - JtJ)) / np.abs(JtJ).max()); d_b = float(np.max(np.abs(pa["b_info"] - Jtr)) / np.abs(Jtr).max())
            ok = bool(same_n and dt_max <= 1e-6 and dr_max <= 1e-8 and dp <= 1e-6 and dq <= 1e-8 and d_info <= 1e-6 and d_b <= 1e-6)
            parity = dict(ok=ok, iterations_gpu=int(rlast["summary"].num_iterations), iterations_oracle=int(ro["summary"].num_iterations),
                          max_step_dt_m=dt_max, max_step_drot_rad=dr_max, final_pose_dt_m=dp, final_quat_diff=dq,
                          prior_JtJ_rel_diff=d_info, prior_Jtr_rel_diff=d_b,
                          bars="per-iteration tangent update <= 1e-6 m / 1e-8 rad, same iteration count, final poses, marginalisation prior J^T J / J^T r <= 1e-6 relative")
            assert ok, f"full-size parity against the oracle failed: {parity}"
    s = rlast["summary"]
    h2d = 32 * CFG["M"] + 32 * CFG["Q"] + 8 * 7 * W * (s.num_evaluations + 2)
    d2h = 8 * 28 * W * (s.num_evaluations + 1) + 4 * W + 8 * 7 * W
    line = dict(metric=METRIC, value=value, unit="iterations/s", n_gpus=world, steps=args.steps, warmup=max(args.warmup, 3),
                ms_per_step=tmax / args.steps, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f64", data="synthetic",
                config=dict(workload=WORKLOAD, **CFG, iterations_per_step=it_sum / args.steps / world, residuals=residuals,
                            parallelism="replicas only (window path does not shard; every rank solves the same window)" if world > 1 else "1 GPU",
                            point_layout="pcl::PointXYZI, 32 B per point (stride 8 floats), map and scans, resident and host legs",
                            l2="256 MB flush between steps inside the timed region; per-step working set > 126 MB L2; "
                               "K2 re-reads the 64 MB residual table every iteration as the real solve does",
                            host_wall_ms_per_step=1e3 * wall / args.steps, step_wall_ms=step_wall_value, per_rank_ms_per_step_value_e2e=per_rank, marginalisation=('pipelined: glio_window_marginalize_async, host half on the library worker thread under the next step\'s association, joined before the next solve; K steps contain K complete marginalisations' if pipelined else 'synchronous inside the step'), cpus_bound_to_gpu_numa_node=n_bound, ms_per_step_with_kernel_events=ms_prof / args.steps, knn_deferred_queries_per_step=n_fallback / args.steps, wall_split=split,
                            solve_split_ms=dict(total=round(1e3 * s.total_seconds, 3), evaluation=round(1e3 * s.eval_seconds, 3), band_cholesky=round(1e3 * s.linear_solver_seconds, 3)), kernels=kern),
                e2e=dict(value=e2e, unit="iterations/s", h2d_bytes_per_step=h2d, d2h_bytes_per_step=d2h, ms_per_step=tmax_e / args.steps,
                         how="pinned host buffers in the PointXYZI layout through the C ABI; per step: the rebuilt local map (32 MB; upload started when the previous solve has returned, overlapping that window's marginalisation, remainder in line) + the newest keyframe's scan (3.2 MB, copy stream, overlapping this window's solve; the other 19 scans are resident as after glio_window_slide) + per-iteration pose/result traffic; final poses and the prior stay on the host side"),
                gpu_launches=int(launches), clocks=clocks, roofline=roof, cpu_baseline=cpu, parity_fullsize=(parity["ok"] if parity else None), parity_detail=parity,
                batch=batch, microbench=micro)
    print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="glio", choices=["glio", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-batch", action="store_true", help="skip the keyframe-sharded batch object")
    ap.add_argument("--sync-marg", action="store_true", help="run the marginalisation synchronously inside the step instead of pipelining its host half under the next association")
    ap.add_argument("--no-cfg4", action="store_true", help="skip the BASELINE cfg 3 (K=200, 1 GPU) / cfg 4 (K=2000, 8 GPUs) batch runs")
    ap.add_argument("--no-microbench", action="store_true", help="skip the cfg 5 microbench object")
    ap.add_argument("--batch-k", type=int, default=400)
    ap.add_argument("--cpu-subsample", type=int, default=1, help="cpu_baseline leg: use every n-th scan point")
    ap.add_argument("--ref-subsample", type=int, default=1, help="--impl reference: use every n-th scan point")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step returned as DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "glio":
        ap.error("--dump-outputs is only supported with --impl glio")
    rank = int(os.environ.get("RANK", 0)); world = int(os.environ.get("WORLD_SIZE", 1)); local = int(os.environ.get("LOCAL_RANK", 0))
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_glio(args, rank, world, local)


if __name__ == "__main__":
    main()

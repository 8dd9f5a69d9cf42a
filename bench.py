#!/usr/bin/env python
"""bench.py -- LM iterations/sec on the batched SE3 pose graph of BASELINE.json, on N B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    (N>1: python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...)

HEADLINE (value / e2e / roofline / cpu_baseline / parity): BASELINE.json's scaling configuration C5 -- sphere-like SE3 pose graph,
2 500 poses, 4 949 edges + 1 prior (m = 29 700, n = 15 000), GLOBAL batch 4096 sharded over the N ranks (strong scaling: N=1 holds all
4096 problems, N=8 holds 512 each), LevenbergMarquardt(10 iterations, damping 1e-3, adaptive + ellipsoidal damping, tolerances 0)
with the block-sparse multifrontal Cholesky (BaspachoSparseSolver, layout "front") on SparseLinearization, fp64.
A "step" = one LM solve (10 iterations of linearize -> Gram -> damped factor -> substitutions -> retract -> error -> accept/reject) of
the whole 4096-problem batch; value = LM iterations per second of that batch.

BESIDE it, never mixed into `value` (key `dense_c2`): BASELINE.json's single-GPU configuration C2 -- 256 poses, batch 256 per GPU
(weak), LM + dense Cholesky -- with the dense DMMA factor's roofline and the GPU-library baseline (torch bmm + linalg.cholesky +
cholesky_solve: what the reference's DenseLinearization / CholeskyDenseSolver execute on the same GPU, dense_linearization.py:58-62,
dense_solver.py:38-64,159-161).

Prints ONE JSON line (rank 0).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

LM_ITERS = 10
LM_KW = dict(damping=1e-3, adaptive_damping=True, ellipsoidal_damping=True)
# ---- headline: C5 ----
C5_RINGS, C5_PER_RING = 50, 50
C5_GLOBAL_BATCH = int(os.environ.get("THB_BENCH_C5_BATCH", "4096"))
C5_LAYOUT = os.environ.get("THB_BENCH_C5_LAYOUT", "front")
METRIC = "LM iterations/sec on batched SE3 pose-graph (2500 poses, global batch 4096 over N GPUs, LM + block-sparse Cholesky, fp64)"
UNIT = "LM iterations/s of the 4096-problem batch (one iteration = one LM step of all 4096 pose graphs)"
WORKLOAD = ("C5: sphere-like SE3 pose graph (50 rings x 50 = 2 500 poses, 4 949 edges + 1 prior; m=29 700, n=15 000), global batch 4096 "
            "sharded over the ranks, LM(10 it, damping 1e-3, adaptive+ellipsoidal) + BaspachoSparseSolver(layout=front: multifrontal "
            "block-sparse Cholesky) on SparseLinearization, fp64")
# ---- beside it: C2 ----
C2_POSES, C2_BATCH = 256, 256
C2_WORKLOAD = ("C2: synthetic SE3 pose-graph (pose_graph_cube shape: 256 poses, loop_closure_ratio 0.2), batch=256 per GPU (weak), "
               "LM(10 it, adaptive+ellipsoidal damping) + CholeskyDenseSolver")
CPU_SAMPLE_ITEMS = 32
# --dump-outputs: the solution of a fixed, seeded sample of batch items (128 x 2 500 poses x 12 doubles = 31 MB; all 4096 would be 983 MB)
DUMP_ITEMS, DUMP_SEED = 128, 0
# sparse CPU arms: one process per batch item, as many items as the host has cores (bounded: 16..128) -- the reference's per-item loop on ALL cores
C5_CPU_ITEMS = int(os.environ.get("THB_BENCH_CPU_ITEMS", str(max(16, min(os.cpu_count() or 16, 128)))))


def _measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p)), "measured"
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0), "fallback"


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index=0):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return dict(sm_mhz=float(np.median(sm)) if sm else None, sm_max_mhz=max(mx) if mx else None, reasons=sorted(reasons),
                    samples=len(sm))


def _host_threads():
    """BLAS / OpenMP threads for the CPU arm: all host cores, asserted (torchrun exports OMP_NUM_THREADS=1)."""
    cores = os.cpu_count() or 1
    from threadpoolctl import threadpool_info, threadpool_limits   # hard requirement: a silent 1-thread CPU arm is a wrong baseline
    ctx = threadpool_limits(limits=cores)
    used = max([int(i.get("num_threads", 1)) for i in threadpool_info()] + [1])
    return ctx, cores, used


def oracle_spec(data, sl):
    """The pose-graph workload as a numpy problem description for the oracle port (CPU arms only)."""
    P, M = data["poses"][:, sl].numpy(), data["meas"][:, sl].numpy()
    spec = dict(dtype=np.dtype(np.float64), vars=[], costs=[])
    for i in range(P.shape[0]):
        spec["vars"].append(dict(kind="SE3", dof=6, value=P[i]))
    w = data["info"].numpy().reshape(1, 6)
    for e, (i, j) in enumerate(data["edges"]):
        spec["costs"].append(dict(kind="between", group="SE3", vars=(i, j), aux=M[e], weight=("diag", w)))
    spec["costs"].append(dict(kind="local", group="SE3", vars=(0,), aux=P[0], weight=("scale", np.full((1, 1), 1e-3))))
    return spec


def cpu_run(data, items, solver, iters=LM_ITERS):
    """Oracle port of the reference's CPU path on the first `items` batch items.  solver='dense': dense A, A^T A by BLAS, LAPACK
    Cholesky (DenseLinearization + CholeskyDenseSolver); solver='sparse': SparseLinearization + one sparse direct factorisation per batch
    item (the reference's CHOLMOD / BaSpaCho-CPU loop, scipy SuperLU standing in), items spread over a process pool of all host cores."""
    from oracle import nls
    spec = oracle_spec(data, slice(0, items))
    ctx, cores, used = _host_threads()
    with ctx:
        t0 = time.perf_counter()
        out = nls.optimize(spec, method="lm", max_iterations=iters, abs_err_tolerance=0, rel_err_tolerance=0, sample_trace=False,
                           solver=solver, n_jobs=min(cores, items) if solver == "sparse" else 1, **LM_KW)
        dt = time.perf_counter() - t0
    return dt, out, cores, (min(cores, items) if solver == "sparse" else used)


def dump_outputs(path, values, info, names):
    """--dump-outputs: what one LM solve of the timed path hands its caller, as float64 .npy files under `path`: per batch item the final
    error, the iteration counts, and the status code (NonlinearOptimizerStatus value: 1 converged, 2 max iterations, -1 failed); and the
    optimised poses ([items, poses, 3, 4]) of DUMP_ITEMS items drawn with DUMP_SEED (their indices in poses_sample_items.npy).  The inputs
    are seeded, so two builds run with the same arguments can be compared file by file."""
    import torch
    os.makedirs(path, exist_ok=True)
    B = info.last_err.shape[0]
    items = np.sort(np.random.default_rng(DUMP_SEED).choice(B, size=min(B, DUMP_ITEMS), replace=False))
    idx = torch.from_numpy(items).to(info.last_err.device)
    poses = torch.stack([values[n].index_select(0, idx) for n in names], 1)
    status = torch.tensor([s.value for s in info.status])
    arrays = dict(last_err=info.last_err, converged_iter=info.converged_iter, best_iter=info.best_iter, status=status, poses_sample=poses,
                  poses_sample_items=torch.from_numpy(items))
    for name, t in arrays.items():
        np.save(os.path.join(path, f"{name}.npy"), t.detach().to(torch.float64).cpu().numpy())


def make_c5_data(batch, seed, device="cpu"):
    from theseus_b200.datasets import pose_graph_sphere
    return pose_graph_sphere(C5_RINGS, C5_PER_RING, batch, seed=seed, device=device)


# ------------------------------------------------------------------------------------------------ --impl reference
def run_reference(args):
    """--impl reference: the reference's own CPU algorithm for the headline workload (numpy port in oracle/), all host cores, rank 0
    only.  Each of the --steps timed steps = the LM solve of a bounded sample (C5_CPU_ITEMS of the 4096 items); value = LM iterations/s
    of the 4096-batch assuming the reference's per-item loop scales linearly in the batch."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    sample = C5_CPU_ITEMS
    data = make_c5_data(sample, seed=0)
    cores = None
    for _ in range(min(args.warmup, 1)):
        cpu_run(data, sample, "sparse", iters=1)
    times = []
    for _ in range(args.steps):
        dt, _, cores, used = cpu_run(data, sample, "sparse")
        times.append(dt)
    t_sample = float(np.mean(times))
    t_full = t_sample * C5_GLOBAL_BATCH / sample
    value = LM_ITERS / t_full
    line = dict(impl="reference", metric=METRIC, value=value, unit=UNIT, n_gpus=args.gpus, steps=len(times), warmup=min(args.warmup, 1),
                ms_per_step=t_full * 1e3, higher_is_better=True, scaling="strong", vs_baseline=None, dtype="f64", data="synthetic",
                config=dict(workload=WORKLOAD, global_batch=C5_GLOBAL_BATCH,
                            note="CPU oracle port of the reference path (SparseLinearization + one sparse direct factorisation per item, SuperLU "
                                 f"standing in for CHOLMOD/BaSpaCho-CPU); {sample}-item sample timed ({t_sample:.2f} s per LM solve), scaled linearly "
                                 "to the 4096-item batch"),
                cpu_baseline=dict(value=value, unit=UNIT, cores=used, host_cores=cores, kind="port",
                                  sample=f"{sample} of {C5_GLOBAL_BATCH} batch items x {LM_ITERS} LM iterations per step, {len(times)} steps"),
                e2e=dict(value=value, unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=0), gpu_launches=0)
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------ ours
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None,
                    help="timed steps of every timed leg (default: 10; 3 with --impl reference, whose step is one CPU solve of "
                         "C5_CPU_ITEMS items, ~47 s on 128 cores)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-c2", action="store_true", help="skip the dense C2 leg reported beside the headline")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step returned to DIR/<name>.npy (with --gpus N > 1: "
                                                          "rank 0's shard only, so dumps are comparable between runs at the same N)")
    args = ap.parse_args()
    if args.steps is None:
        args.steps = 3 if args.impl == "reference" else 10
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference" and args.dump_outputs:
        ap.error("--dump-outputs writes the outputs of --impl ours")
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world != args.gpus:
        print(f"warning: WORLD_SIZE={world} != --gpus {args.gpus}", file=sys.stderr)
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    pg = None
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
        pg = dist.group.WORLD

    import theseus_b200 as th
    from theseus_b200 import _lib
    from theseus_b200.datasets import build_pose_graph_objective
    from theseus_b200.distributed import batch_shard
    lib = _lib.load()
    warmup = max(args.warmup, 3)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        """CUDA events on the launching stream, barrier + synchronize on both sides, max over ranks (ms)."""
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=device, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    # ================================================= headline: C5, strong scaling =================================================
    sl = batch_shard(C5_GLOBAL_BATCH, rank, world)
    B = sl.stop - sl.start
    data = make_c5_data(B, seed=1000 + rank, device=device)            # fabricated on the device, returned in HOST memory
    objective, poses = build_pose_graph_objective(th, data, device)
    opt = th.LevenbergMarquardt(objective, linear_solver_cls=th.BaspachoSparseSolver, linearization_cls=th.SparseLinearization,
                                max_iterations=LM_ITERS, step_size=1.0, abs_err_tolerance=0, rel_err_tolerance=0, process_group=pg,
                                linear_solver_kwargs=dict(layout=C5_LAYOUT), cuda_graph=os.environ.get("THB_BENCH_GRAPH", "0") == "1")
    layer = th.TheseusLayer(opt)
    names_pose = [p.name for p in poses]
    edge_names = [cf.measurement.name for cf in objective.cost_functions.values() if hasattr(cf, "measurement")]
    dev_inputs = {p.name: data["poses"][i].to(device) for i, p in enumerate(poses)}
    out = {}

    def step_resident():
        with torch.no_grad():
            out["values"], out["info"] = layer.forward(dev_inputs, optimizer_kwargs=LM_KW)

    for _ in range(warmup):
        step_resident()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    l0 = _lib.total_launches()
    prof_range = os.environ.get("THB_BENCH_PROFILE_RANGE", "0") == "1"   # ncu --profile-from-start off: the launch list of the timed steps only
    if prof_range:
        torch.cuda.profiler.start()
    ms_step = timed(step_resident, args.steps) / args.steps
    if prof_range:
        torch.cuda.profiler.stop()
    launches = int(_lib.total_launches() - l0)
    clocks = sampler.stop() if rank == 0 else None
    value = LM_ITERS * 1e3 / ms_step
    final_err = out["info"].last_err.clone()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, out["values"], out["info"], names_pose)

    # ---- e2e: pinned host inputs -> device, public API, solution + error back to pinned host memory, every step ----
    host_poses, host_meas = data["poses"].pin_memory(), data["meas"].pin_memory()
    dev_pose_buf = torch.empty_like(data["poses"], device=device)
    dev_meas_buf = torch.empty_like(data["meas"], device=device)
    host_out = torch.empty_like(data["poses"]).pin_memory()
    host_err = torch.empty(B, dtype=torch.float64).pin_memory()

    def step_e2e():
        dev_pose_buf.copy_(host_poses, non_blocking=True)
        dev_meas_buf.copy_(host_meas, non_blocking=True)
        inputs = {n: dev_pose_buf[i] for i, n in enumerate(names_pose)}
        inputs.update({n: dev_meas_buf[e] for e, n in enumerate(edge_names)})
        with torch.no_grad():
            values, info = layer.forward(inputs, optimizer_kwargs=LM_KW)
        torch.stack([values[n] for n in names_pose], 0, out=dev_pose_buf)
        host_out.copy_(dev_pose_buf, non_blocking=True)
        host_err.copy_(info.last_err, non_blocking=True)
        torch.cuda.current_stream().synchronize()

    e2e_steps = args.steps
    step_e2e()
    ms_e2e = timed(step_e2e, e2e_steps) / e2e_steps
    h2d = (host_poses.numel() + host_meas.numel()) * 8 * world       # whole job, per step
    d2h = (host_out.numel() + host_err.numel()) * 8 * world

    # ---- phase split + roofline of the dominant call: the numeric factorisation ----
    lin = opt.linear_solver.linearization
    solver = opt.linear_solver
    lam = torch.full((B,), 1e-3, dtype=torch.float64, device=device)
    ms_lin = timed(lin.linearize, 3) / 3
    ms_solve = timed(lambda: solver.solve(damping=lam, ellipsoidal_damping=True, damping_eps=1e-8), 3) / 3
    from theseus_b200.optimizer import convert_to_alpha_beta_damping_tensors
    A64, b64 = lin.A_val.contiguous(), lin.b.contiguous()
    alpha, beta = convert_to_alpha_beta_damping_tensors(lam, 1e-8, True, B, device, torch.float64)
    Atb = solver._numeric(A64, b64, alpha, beta)
    ms_numeric = timed(lambda: solver._numeric(A64, b64, alpha, beta), 3) / 3
    ms_subst = timed(lambda: solver._substitute(Atb), 3) / 3
    stats = {k: (float(v) if not isinstance(v, str) else v) for k, v in dict(solver.symbolic_stats).items()}
    flops_item = float(stats.get("flops", 0.0))
    nnz_l = float(stats.get("nnz_L", 0.0))
    # fp64 peak: MEASURED_PEAKS.json has no fp64 entry -> cuBLAS dgemm 8192^3 measured live, same method as the driver's bf16 peak
    am = torch.randn(8192, 8192, dtype=torch.float64, device=device)
    bm = torch.randn(8192, 8192, dtype=torch.float64, device=device)
    torch.matmul(am, bm)
    best = 1e30
    for _ in range(5):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        torch.matmul(am, bm)
        e1.record()
        torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1))
    peak_tf = 2 * 8192 ** 3 / (best * 1e-3) / 1e12
    del am, bm
    peaks, peaks_src = _measured_peaks()
    hbm = float(peaks.get("hbm_gbs", 6650.0))
    # algorithmic bytes of one numeric factorisation per item: AtA blocks read + L written (DESIGN.md 4); the substitutions read L twice
    ata_doubles = float(sum(int(a) * int(bb) for a, bb in zip(solver._gram_arrays["blk_rows"], solver._gram_arrays["blk_cols"])))
    bytes_factor = 8.0 * (ata_doubles + nnz_l) * B
    t_flops, t_bytes = flops_item * B / (peak_tf * 1e12), bytes_factor / (hbm * 1e9)
    achieved_tf = flops_item * B / (ms_numeric * 1e-3) / 1e12
    roofline = dict(bound="tensor", kernel=f"thb_front_factor_f64 + Gram: one numeric factorisation of {B} items (multifrontal: shared-memory front kernel "
                    "+ DMMA dense kernel in partial mode; kernel list: profiles/r02_*_launch_agg.txt)",
                    achieved=achieved_tf, peak=peak_tf, unit="TFLOP/s", frac=achieved_tf / peak_tf,
                    traffic=None, flops_per_item=flops_item, nnz_L=nnz_l, algorithmic_bytes=bytes_factor, ms_per_factorisation=ms_numeric,
                    hbm_frac_of_algorithmic_bytes=bytes_factor / (ms_numeric * 1e-3) / (hbm * 1e9),
                    binding_roofline_ms=max(t_flops, t_bytes) * 1e3, frac_of_binding_roofline=max(t_flops, t_bytes) * 1e3 / ms_numeric,
                    substitutions=dict(ms=ms_subst, algorithmic_bytes=16.0 * nnz_l * B, hbm_frac=16.0 * nnz_l * B / (ms_subst * 1e-3) / (hbm * 1e9)),
                    peak_source="fp64 cuBLAS dgemm 8192^3 measured live in this run (MEASURED_PEAKS.json carries no fp64 figure; "
                                f"its bf16/HBM entries [{peaks_src}]: {peaks.get('bf16_tflops')} TF/s, {hbm} GB/s)",
                    share_of_step=ms_numeric * LM_ITERS / ms_step,
                    # the largest single kernel of the factorisation, from the committed captures (NOT measured in this run): its traffic
                    # is the per-kernel dram figure the contract's `traffic` key asks for; the call above is ~100 launches of 6 kernels
                    dominant_kernel=dict(name="front_small_kernel<1024>", share_of_linear_solve=0.283,
                                         share_source="profiles/r02m_c5_B512_front_launch_agg.txt (ncu --metrics gpu__time_duration.sum, one solve, B=512)",
                                         ncu_launch="depth-6 launch of C5, B=512: 6 fronts (w 36-66, b 192-372) x 512 items, 26.3 MFLOP per item",
                                         duration_ms=1.47, achieved_tflops=9.2, dmma_pipe_pct=29.5, traffic=2.92e9,
                                         algorithmic_bytes=2.40e9, traffic_over_algorithmic=1.22,
                                         ncu_source="profiles/r02l_front_small_1024_ncu_full_details.txt, r02l_front_kernels_ncu_summary.txt"))

    # ---- bench-size parity: first-iteration delta and final error of the first items vs the CPU oracle's run on the same items.
    # Every rank runs the extra (untimed) solve so that the per-iteration collectives stay matched; rank 0 compares. ----
    parity, cpu = None, None
    k = min(C5_CPU_ITEMS, B)
    deltas = []

    def cb(optimizer, info, delta, it):
        if it == 0 and not deltas:
            deltas.append(delta[:k].cpu().numpy().copy())
    with torch.no_grad():
        _, info_p = layer.forward(dev_inputs, optimizer_kwargs=dict(LM_KW, end_iter_callback=cb))
    if rank == 0 and not args.no_cpu_baseline:
        dt, ora, cores, used = cpu_run(data, k, "sparse")
        rec = next((r for r in ora["trace"] if not ("reject" in r and bool(np.all(r["reject"])))), ora["trace"][0])   # first accepted attempt
        d_ref = rec["delta"]
        rel_delta = float(np.max(np.linalg.norm(deltas[0] - d_ref, axis=1) / np.linalg.norm(d_ref, axis=1)))
        e_ref = ora["err_history"][:, -1]
        rel_err = float(np.max(np.abs(info_p.last_err[:k].cpu().numpy() - e_ref) / np.abs(e_ref)))
        parity = dict(items=k, first_iteration_delta_rel=rel_delta, final_err_rel=rel_err, tolerance_delta=1e-5, tolerance_err=1e-5,
                      ok=bool(rel_delta <= 1e-5 and rel_err <= 1e-5),
                      against="CPU oracle (oracle/nls.py, sparse path) on the same first items of rank 0's shard")
        if world == 1:
            t_full = dt * C5_GLOBAL_BATCH / k
            cpu = dict(value=LM_ITERS / t_full, unit=UNIT, cores=used, host_cores=cores, kind="port",
                       sample=f"{k} of {C5_GLOBAL_BATCH} batch items x {LM_ITERS} LM iterations ({dt:.1f} s measured), scaled linearly in the batch; "
                              "SparseLinearization + per-item sparse direct factorisation (SuperLU standing in for CHOLMOD / BaSpaCho-CPU)",
                       final_err_mean_sample=float(e_ref.mean()))

    # ================================================= beside it: C2 dense =================================================
    c2 = None
    if not args.no_c2:
        try:
            c2 = dense_c2_leg(th, lib, _lib, device, rank, world, pg, timed, peak_tf, steps=args.steps, with_cpu=(rank == 0 and world == 1 and not args.no_cpu_baseline))
        except Exception as e:   # the leg is reported beside the headline: a failure there must not take the headline down
            c2 = dict(error=repr(e)[:300])

    if world > 1:
        dist.barrier()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    line = dict(
        metric=METRIC, value=value, unit=UNIT, n_gpus=world, steps=args.steps, warmup=warmup, ms_per_step=ms_step, higher_is_better=True,
        scaling="strong", vs_baseline=None, dtype="f64", data="synthetic",
        config=dict(workload=WORKLOAD, global_batch=C5_GLOBAL_BATCH, batch_per_gpu=B, num_poses=len(poses), num_edges=len(data["edges"]),
                    rows=int(lin.num_rows), cols=int(lin.num_cols), lm_iterations_per_step=LM_ITERS, problem_iterations_per_s=value * C5_GLOBAL_BATCH,
                    layout=solver.effective_layout, symbolic=stats,
                    l2="working set per iteration (factor panels + update-matrix arena, > 10 GB per rank) >> 126 MB L2, no flush needed",
                    parallelism=f"batch sharded over {world} GPU(s); per LM iteration one all-reduce of the reject / item counts (+ one of the "
                                "solve-failure flag), NCCL",
                    cuda_graph=bool(opt.cuda_graph)),
        clocks=clocks,
        e2e=dict(value=LM_ITERS * 1e3 / ms_e2e, unit=UNIT, ms_per_step=ms_e2e, steps=e2e_steps, h2d_bytes_per_step=h2d, d2h_bytes_per_step=d2h),
        gpu_launches=launches, roofline=roofline,
        phases_ms_per_iteration=dict(linearize=ms_lin, linear_solve=ms_solve, numeric_factorisation=ms_numeric, substitutions=ms_subst),
        cpu_baseline=cpu, parity=parity, final_err_mean=float(final_err.mean().item()), dense_c2=c2)
    print(json.dumps(line))
    if parity is not None and not parity["ok"]:
        print(f"PARITY FAILURE at bench size: {parity}", file=sys.stderr)
        sys.exit(3)
    if world > 1:
        dist.destroy_process_group()


def dense_c2_leg(th, lib, _lib, device, rank, world, pg, timed, peak_tf, steps, with_cpu):
    """Config C2 beside the headline (weak scaling, 256 problems per GPU): LM + CholeskyDenseSolver, the dense DMMA factor's roofline,
    the GPU-library baseline of the same linear solve, and (N=1) the CPU port on a 16-item sample."""
    import torch
    from theseus_b200.datasets import build_pose_graph_objective, pose_graph_synthetic_3d
    data = pose_graph_synthetic_3d(C2_POSES, C2_BATCH, translation_noise=0.05, rotation_noise=0.02, loop_closure_ratio=0.2, seed=rank)
    objective, poses = build_pose_graph_objective(th, data, device)
    opt = th.LevenbergMarquardt(objective, linear_solver_cls=th.CholeskyDenseSolver, max_iterations=LM_ITERS, step_size=1.0,
                                abs_err_tolerance=0, rel_err_tolerance=0, process_group=pg, cuda_graph=True)
    layer = th.TheseusLayer(opt)
    dev_inputs = {p.name: data["poses"][i].to(device) for i, p in enumerate(poses)}
    out = {}

    def step():
        with torch.no_grad():
            out["values"], out["info"] = layer.forward(dev_inputs, optimizer_kwargs=LM_KW)
    for _ in range(3):
        step()
    ms_step = timed(step, steps) / steps
    lin = opt.linear_solver.linearization
    lin.linearize()
    AtA = lin.AtA
    B, n = AtA.shape[0], AtA.shape[1]
    alpha = torch.full((B,), 1e-3, dtype=torch.float64, device=device)
    beta = torch.full((B,), 1e-8, dtype=torch.float64, device=device)
    infot = torch.empty(B, dtype=torch.int32, device=device)
    need = int(lib.thb_potrf_workspace_bytes(B, n))
    ws = torch.empty(need, dtype=torch.uint8, device=device)

    def factor():
        _lib.check(lib.thb_potrf_f64(_lib.ptr(AtA), _lib.ptr(alpha), _lib.ptr(beta), _lib.ptr(infot), B, n, _lib.ptr(ws), need, _lib.stream_ptr()), "potrf")
    for _ in range(3):
        factor()
    ms_factor = timed(factor, 10) / 10
    flops = B * (n ** 3) / 3.0
    achieved_tf = flops / (ms_factor * 1e-3) / 1e12
    res = dict(workload=C2_WORKLOAD, value=LM_ITERS * 1e3 / ms_step * world,
               unit="LM iterations/s (one iteration = one LM step of a 256-problem batch; summed over the GPUs: weak scaling)",
               ms_per_step=ms_step, steps=steps, batch_per_gpu=C2_BATCH, cols=int(n), final_err_mean=float(out["info"].last_err.mean().item()),
               roofline=dict(bound="tensor", kernel="chol_col_kernel (fp64 DMMA left-looking Cholesky, one launch = one batched factorisation of 256 matrices)",
                             achieved=achieved_tf, peak=peak_tf, unit="TFLOP/s", frac=achieved_tf / peak_tf, traffic=34.40e9,
                             traffic_note="dram bytes per launch from the round-1 ncu --set full capture (profiles/r01g_chol_col_ncu_full_details.txt)",
                             algorithmic_bytes=8.0 * B * n * n, ms_per_factorisation=ms_factor, share_of_step=ms_factor * LM_ITERS / ms_step))
    # ---- GPU-library baseline: what the reference's dense path executes on this GPU for one linear solve of the same system ----
    if rank == 0:
        try:
            S = lin.engine.structure
            m = int(S.num_rows)
            rows = torch.from_numpy(np.repeat(np.arange(m), np.diff(S.A_row_ptr))).to(device)
            cols = torch.from_numpy(np.asarray(S.A_col_ind)).to(device)
            A = torch.zeros(B, m, n, dtype=torch.float64, device=device)
            A[:, rows, cols] = lin._A_val
            bvec = lin.b

            def lib_solve():
                At = A.transpose(1, 2)
                AtA_l = At.bmm(A)                                          # dense_linearization.py:58-62
                Atb_l = At.bmm(bvec.unsqueeze(2))
                damp = 1e-3 * AtA_l.diagonal(dim1=1, dim2=2) + 1e-8        # dense_solver.py:38-64 (ellipsoidal)
                M = AtA_l + torch.diag_embed(damp)
                Lc = torch.linalg.cholesky(M)                              # dense_solver.py:159-161
                return torch.cholesky_solve(Atb_l, Lc).squeeze(2)
            x_lib = lib_solve()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(3):
                lib_solve()
            e1.record()
            torch.cuda.synchronize()
            ms_lib = e0.elapsed_time(e1) / 3
            x_ours = opt.linear_solver.solve(damping=alpha, ellipsoidal_damping=True, damping_eps=1e-8)
            e0.record()
            for _ in range(3):
                lin.linearize()
                opt.linear_solver.solve(damping=alpha, ellipsoidal_damping=True, damping_eps=1e-8)
            e1.record()
            torch.cuda.synchronize()
            ms_ours = e0.elapsed_time(e1) / 3
            rel = float(((x_ours - x_lib).norm(dim=1) / x_lib.norm(dim=1)).max().item())
            res["gpu_library_baseline"] = dict(what="torch (cuBLAS bmm of the dense A, cuSOLVER/MAGMA batched potrf, cholesky_solve) on the same inputs, "
                                               "one damped linear solve incl. A^T A (dense A already assembled, not timed)", ms_library=ms_lib,
                                               ms_ours_linearize_gram_factor_solve=ms_ours,
                                               note_ours="includes the Jacobian evaluation (linearize kernel), which the library figure does not", solution_rel_diff=rel)
            del A
        except Exception as e:
            res["gpu_library_baseline"] = dict(error=repr(e)[:300])
    if with_cpu:
        k = CPU_SAMPLE_ITEMS
        dt, ora, cores, used = cpu_run(data, k, "dense")
        t_full = dt * C2_BATCH / k
        rel_err = float(np.max(np.abs(out["info"].last_err[:k].cpu().numpy() - ora["err_history"][:, -1]) / np.abs(ora["err_history"][:, -1])))
        res["cpu_baseline"] = dict(value=LM_ITERS / t_full, cores=used, host_cores=cores, kind="port",
                                   sample=f"{k} of {C2_BATCH} items x {LM_ITERS} LM iterations ({dt:.1f} s), scaled linearly; dense A, BLAS A^T A, LAPACK potrf",
                                   final_err_rel_diff_vs_gpu_first_items=rel_err)
    return res


if __name__ == "__main__":
    main()

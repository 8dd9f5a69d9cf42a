"""Batched 2-D motion planning on the GPU: the planner objective of tests/golden/make_golden_motion_planning.py (motion_planning_problem: T steps, per step
Collision2D + GPMotionModel(GPCostWeight), boundary Differences; Point2 poses) over seeded synthetic 128 x 128 maps (random discs, SDF from
scipy.ndimage.distance_transform_edt), starts and goals in free space, straight-line initialisation, LevenbergMarquardt 10 iterations.

    python scratch/bench_motion_planning.py [--batch 512 4096] [--solvers dense front] [--steps 100] [--repeats 3]

Prints ONE JSON line: per (batch, solver) LM it/s and ms per iteration of the whole LM step; per batch the fused linearize time (CUDA
events over repeated thb_linearize_group launches, warm) against the same objective on the engine's torch route (subclasses whose schema()
returns no kind), bytes the linearize pass must move (from shapes) over its kernel time, the largest difference of the final trajectories
of the two routes (at the smallest batch), and the GPU's name and power limit.  Writes nothing."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
import theseus_b200 as th  # noqa: E402
import make_golden_motion_planning as G  # noqa: E402  (only the pure problem builders are used; the reference is imported under __main__ only)


def synthetic_inputs(B, T, seed=0, size=128, cell=10.0 / 128):
    from scipy import ndimage
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:size, 0:size] * cell - 5.0
    sdfs, starts, goals = [], [], []
    for _ in range(B):
        occ = np.zeros((size, size), bool)
        for _ in range(rng.integers(4, 9)):
            cx, cy, r = rng.uniform(-3.5, 3.5), rng.uniform(-3.5, 3.5), rng.uniform(0.4, 1.2)
            occ |= (xx - cx) ** 2 + (yy - cy) ** 2 < r * r
        sdf = (ndimage.distance_transform_edt(~occ) - ndimage.distance_transform_edt(occ)) * cell
        free = np.argwhere(sdf > 0.4)
        a, b = free[rng.integers(len(free))], free[rng.integers(len(free))]
        starts.append([a[1] * cell - 5.0, a[0] * cell - 5.0]); goals.append([b[1] * cell - 5.0, b[0] * cell - 5.0])
        sdfs.append(sdf)
    start, goal = np.array(starts), np.array(goals)
    return dict(sdf_data=np.stack(sdfs).astype(np.float64), sdf_origin=np.tile([[-5.0, -5.0]], (B, 1)), cell_size=np.full((B, 1), cell),
                start=start, goal=goal, start_se2=np.concatenate([start, np.ones((B, 1)), np.zeros((B, 1))], 1), steps=T,
                epsilon_dist=0.2, total_time=10.0, collision_weight=20.0)


class TorchCollision2D(th.eb.Collision2D):
    def schema(self):
        return None, super().schema()[1]


class TorchGPMotionModel(th.eb.GPMotionModel):
    def schema(self):
        return None, super().schema()[1]


def build(inputs, torch_route=False):
    saved = (th.eb.Collision2D, th.eb.GPMotionModel)
    if torch_route:
        th.eb.Collision2D, th.eb.GPMotionModel = TorchCollision2D, TorchGPMotionModel
    try:
        objective, poses, vels, _ = G.motion_planning_problem(th, torch, inputs, "point2", device="cuda")
    finally:
        th.eb.Collision2D, th.eb.GPMotionModel = saved
    init = {k: v.cuda() for k, v in G.motion_planning_straight_line(torch, inputs, "point2").items()}
    objective.update(init)
    return objective, poses, init


def event_time(fn, repeats):
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    fn()
    torch.cuda.synchronize()
    s.record()
    for _ in range(repeats):
        fn()
    e.record()
    torch.cuda.synchronize()
    return s.elapsed_time(e) / repeats


def linearize_bytes(eng, B):
    """Bytes the fused linearize pass must move, from shapes: A_val and b written once; per cost function its optimisation variables read
    once per item, a collision cost's four SDF samples (8 B each); broadcast auxiliaries (dt, Qc_inv, origin, cell, eps, weights) not counted."""
    byt = (eng.nnz + eng.m) * 8 * B
    for g in eng.groups:
        for f in g.cost_indices:
            cf = eng.costs[f]
            byt += sum(v.numel() for v in cf.optim_vars) * 8 * B
            if g.kind in (8, 9):
                byt += 4 * 8 * B
    return byt


def lm_run(objective, init, solver, repeats):
    skw = dict(linear_solver_cls=th.CholeskyDenseSolver) if solver == "dense" else dict(
        linear_solver_cls=th.BaspachoSparseSolver, linearization_cls=th.SparseLinearization, linear_solver_kwargs=dict(layout=solver))
    opt = th.LevenbergMarquardt(objective, max_iterations=10, step_size=1.0, abs_err_tolerance=0, rel_err_tolerance=0, **skw)
    lm = dict(damping=0.1, adaptive_damping=True)
    times = []
    for r in range(repeats + 1):                       # first run = warm-up (plans, buffers, module loads)
        objective.update({k: v.clone() for k, v in init.items()})
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        with torch.no_grad():
            opt.optimize(**lm)
        torch.cuda.synchronize()
        if r:
            times.append(time.perf_counter() - t0)
    return (min(times), float(np.median(times))) if times else (None, None)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, nargs="+", default=[512, 4096])
    ap.add_argument("--solvers", nargs="+", default=["dense", "front"])
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--repeats", type=int, default=3)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_motion_planning: needs a CUDA device")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    res = dict(workload=f"motion planning 2-D, Point2, T={a.steps}, LM 10 it, fp64", gpu=torch.cuda.get_device_name(), nvidia_smi=q, runs=[])
    for B in a.batch:
        inputs = synthetic_inputs(B, a.steps)
        objective, poses, init = build(inputs)
        eng = objective.engine()
        assert eng.generic == []
        row = dict(batch=B, costs=len(eng.costs), m=eng.m, n=eng.n, nnz=eng.nnz)
        lin_ms = event_time(lambda: eng.linearize_sparse(), 20)
        byt = linearize_bytes(eng, B)
        row.update(linearize_ms=lin_ms, linearize_bytes=byt, linearize_GBps=byt / (lin_ms * 1e-3) / 1e9)
        for solver in a.solvers:
            best, med = lm_run(objective, init, solver, a.repeats)
            row[solver] = dict(lm_it_per_s=10 / best, ms_per_iter=best / 10 * 1e3, ms_per_iter_median=med / 10 * 1e3,
                               solve_and_control_ms_per_iter=best / 10 * 1e3 - lin_ms)
        fused_final = None
        if B == min(a.batch):
            lm_run(objective, init, "dense", 0)
            fused_final = torch.stack([p.tensor for p in poses]).clone()
        tobj, tposes, tinit = build(inputs, torch_route=True)
        teng = tobj.engine()
        assert len(teng.generic) == 2 * a.steps
        row["torch_route_linearize_ms"] = event_time(lambda: teng.linearize_sparse(), 2)
        row["fused_speedup_linearize"] = row["torch_route_linearize_ms"] / lin_ms
        if fused_final is not None:
            lm_run(tobj, tinit, "dense", 0)
            row["max_abs_diff_final_traj_fused_vs_torch"] = float((torch.stack([p.tensor for p in tposes]) - fused_final).abs().max())
        res["runs"].append(row)
        del objective, tobj, eng, teng
        torch.cuda.empty_cache()
    print(json.dumps(res))


if __name__ == "__main__":
    main()

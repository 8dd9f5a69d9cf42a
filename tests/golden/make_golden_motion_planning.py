"""Generate tests/golden/motion_planning_kat.npz by running the REFERENCE ITSELF (facebookresearch/theseus v0.2.3): 2-D motion planning
(Collision2D, GPMotionModel + GPCostWeight, the planner objective of utils/examples/motion_planning/motion_planner.py).

Run in the build container only (the GPU box has no /root/reference):
    python tests/golden/make_golden_motion_planning.py
At test time only the pure problem builders below are loaded from this file (tests/mp_common.py, scratch/bench_motion_planning.py), so
generator, tests and benchmark build the same objective with either library; the reference is imported under __main__ only (through
make_golden._import_reference, which stubs lxml; nothing here imports theseus.utils.examples, so matplotlib is not needed)."""
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
REF = "/root/reference"

MP_DIR = REF + "/tutorials/data/motion_planning_2d"


def motion_planning_problem(th, torch, inputs, pose_type="point2", device="cpu", dtype=None, collision_w=None, cost_eps=None):
    """The objective of the reference's MotionPlannerObjective (utils/examples/motion_planning/motion_planner.py:58-280) for `T = steps`
    time steps: boundary Differences on pose_0 / vel_0 / pose_N / vel_N (weight 100; SE2: the goal cost on pose_N.xy is the planner's own
    user-defined _XYDifference), per step a Collision2D and a GPMotionModel (GPCostWeight(Qc_inv = I, dt)).  Builds with the reference
    (generator) and with theseus_b200 (tests).  Returns (objective, poses, vels, leaves)."""
    d = dtype or torch.float64
    T = int(inputs["steps"])
    P = th.SE2 if pose_type == "se2" else th.Point2
    dof = 3 if pose_type == "se2" else 2
    B = inputs["sdf_data"].shape[0]
    t = lambda k: torch.as_tensor(inputs[k]).to(d).clone()
    sdf_origin = th.Point2(tensor=t("sdf_origin"), name="sdf_origin")
    cell_size = th.Variable(t("cell_size").view(-1, 1), name="cell_size")
    sdf_data = th.Variable(t("sdf_data"), name="sdf_data")
    eps = th.Variable(cost_eps if cost_eps is not None else torch.tensor(float(inputs["epsilon_dist"]), dtype=d).view(1, 1), name="cost_eps")
    dt = th.Variable(torch.tensor(float(inputs["total_time"]) / T, dtype=d).view(1, 1), name="dt")
    gp_w = th.eb.GPCostWeight(torch.eye(dof, dtype=d), dt)
    cw = th.ScaleCostWeight(th.Variable(collision_w if collision_w is not None else torch.tensor(float(inputs["collision_weight"]), dtype=d).view(1, 1),
                                        name="collision_w"))
    bw = th.ScaleCostWeight(torch.tensor(100.0, dtype=d))
    start = t("start_se2") if pose_type == "se2" else t("start")
    poses = [P(tensor=start.clone(), name=f"pose_{i}") for i in range(T + 1)]
    vels = [th.Vector(tensor=torch.zeros(B, dof, dtype=d), name=f"vel_{i}") for i in range(T + 1)]
    objective = th.Objective(dtype=d)
    objective.add(th.Difference(poses[0], P(tensor=start.clone(), name="start"), bw, name="pose_0"))
    objective.add(th.Difference(vels[0], th.Vector(tensor=torch.zeros(1, dof, dtype=d), name="vel_0_target"), bw, name="vel_0"))
    goal = th.Point2(tensor=t("goal"), name="goal")
    if pose_type == "se2":
        objective.add(_xy_difference_cls(th, torch)(poses[-1], goal, bw, name="pose_N"))
    else:
        objective.add(th.Difference(poses[-1], goal, bw, name="pose_N"))
    objective.add(th.Difference(vels[-1], th.Vector(tensor=torch.zeros(1, dof, dtype=d), name="vel_N_target"), bw, name="vel_N"))
    for i in range(1, T + 1):
        objective.add(th.eb.Collision2D(poses[i], sdf_origin, sdf_data, cell_size, eps, cw, name=f"collision_{i}"))
        objective.add(th.eb.GPMotionModel(poses[i - 1], vels[i - 1], poses[i], vels[i], dt, gp_w, name=f"gp_{i}"))
    if str(device) != "cpu":
        objective.to(device)
    return objective, poses, vels, dict(collision_w=cw.scale, cost_eps=eps)


def _xy_difference_cls(th, torch):
    """The planner's goal cost on SE2 poses (motion_planner.py:17-55): e = pose.xy - goal, J = [R 0]; a user-defined cost function."""
    class XYDifference(th.CostFunction):
        def __init__(self, var, target, cost_weight, name=None):
            super().__init__(cost_weight, name=name)
            self.var, self.target = var, target
            self.register_optim_vars(["var"])
            self.register_aux_vars(["target"])

        def error(self):
            return self.var.tensor[:, :2] - self.target.tensor

        def jacobians(self):
            x = self.var.tensor
            c, s = x[:, 2], x[:, 3]
            z = torch.zeros_like(c)
            J = torch.stack([torch.stack([c, -s, z], 1), torch.stack([s, c, z], 1)], 1)
            return [J], self.error()

        def dim(self):
            return 2

        def _copy_impl(self, new_name=None):
            return XYDifference(self.var.copy(), self.target.copy(), self.weight.copy(), name=new_name)
    return XYDifference


def motion_planning_inputs(torch, T=100):
    """The two `tarpit` maps of the reference's tutorial data built like TrajectoryDataset (misc.py:84-115) without the map image:
    origin (-5, -5), cell size 10 / 128, the .npy SDF, the GPMP2 trajectory with rows 1 and 3 negated; start / goal = its end points;
    the planner's tutorial parameters (epsilon 0.2, total time 10, collision weight 20)."""
    sdf = np.stack([np.load(f"{MP_DIR}/im_sdf/tarpit/{i}_sdf.npy") for i in range(2)], 0).astype(np.float64)
    trajs = []
    for i in range(2):
        tr = np.load(f"{MP_DIR}/opt_trajs_gpmp2/tarpit/env_{i}_prob_0.npz")["th_opt"].T.astype(np.float64).copy()
        tr[1] *= -1.0
        tr[3] *= -1.0
        trajs.append(tr)
    expert = np.stack(trajs, 0)                                  # [2, 4, T+1]: x, y, vx, vy
    start, goal = expert[:, :2, 0], expert[:, :2, -1]
    theta = np.arctan2(goal[:, 1] - start[:, 1], goal[:, 0] - start[:, 0])
    return dict(sdf_data=sdf, sdf_origin=np.array([[-5.0, -5.0]] * 2), cell_size=np.full((2, 1), 10.0 / 128.0), expert=expert,
                start=start, goal=goal, start_se2=np.concatenate([start, np.cos(theta)[:, None], np.sin(theta)[:, None]], 1),
                steps=T, epsilon_dist=0.2, total_time=10.0, collision_weight=20.0)


def motion_planning_straight_line(torch, inputs, pose_type="point2"):
    """MotionPlanner.get_variable_values_from_straight_line (motion_planner.py:358-378): name -> tensor."""
    T = int(inputs["steps"])
    start = torch.as_tensor(inputs["start_se2" if pose_type == "se2" else "start"])
    goal = torch.as_tensor(inputs["goal"])
    dist = goal[:, :2] - start[:, :2]
    avg_vel, unit = dist / float(inputs["total_time"]), dist / T
    out = {}
    for i in range(T + 1):
        if pose_type == "se2":
            out[f"pose_{i}"] = torch.cat([start[:, :2] + unit * i, start[:, 2:]], 1)
            out[f"vel_{i}"] = torch.cat([avg_vel, torch.zeros_like(avg_vel[:, :1])], 1)
        else:
            out[f"pose_{i}"] = start + unit * i
            out[f"vel_{i}"] = avg_vel.clone()
    return out


MP_COST_CASES = [  # (name, pose kind, weight kind, batched aux) of the per-cost known answers
    ("col_p2_scale", "point2", "scale", False), ("col_p2_diag_b", "point2", "diag", True), ("col_se2_scale_b", "se2", "scale", True),
    ("col_se2_diag", "se2", "diag", False),
    ("di_p2_gp", "point2", "gp", False), ("di_p2_gp_b", "point2", "gp", True), ("di_p2_scale", "point2", "scale", False),
    ("di_se2_gp", "se2", "gp", False), ("di_se2_gp_b", "se2", "gp", True), ("di_se2_diag", "se2", "diag", True),
    ("di_v3_gp_b", "vector3", "gp", True), ("di_v3_scale", "vector3", "scale", False),
]


def motion_planning_cost_inputs(case, dtype_name, B=6, seed=3):
    """Deterministic inputs of one per-cost case: a 12 x 16 grid; collision points in bounds, out of bounds, exactly at eps and beyond
    eps (the SDF is linear in x so that d = eps is exact)."""
    name, pk, wk, batched = case
    rng = np.random.default_rng(seed + sum(map(ord, name)))
    dt_ = np.float64 if dtype_name == "f64" else np.float32
    out = {}
    if name.startswith("col"):
        rows, cols, cell = 12, 16, 0.25
        xx = np.arange(cols) * cell
        base = np.tile((xx - 1.0)[None, :], (rows, 1)) + 0.1 * np.sin(np.arange(rows))[:, None] * (np.arange(cols) > 8)[None, :]
        nb = B if batched else 1
        out["sdf_data"] = np.stack([base + 0.05 * k for k in range(nb)], 0)
        out["sdf_origin"] = np.tile([[0.5, -0.25]], (nb, 1))
        out["cell_size"] = np.full((nb, 1), cell)
        out["cost_eps"] = np.full((nb, 1), 0.5) + (0.1 * np.arange(nb)[:, None] if batched else 0.0)
        # point 0: d = eps exactly (linear region, row 0 .. 8); 1: out of bounds; 2: beyond eps; 3..: random in bounds
        eps0 = out["cost_eps"][0, 0]
        pts = [[0.5 + 1.0 + eps0 - 0.0, -0.25 + 0.5], [-1.0, 0.3], [0.5 + 1.9, 1.0]] + [
            [0.5 + rng.uniform(0, 3.7), -0.25 + rng.uniform(0, 2.7)] for _ in range(B - 3)]
        pts = np.array(pts)
        if pk == "se2":
            th_ = rng.uniform(-3, 3, B)
            out["pose"] = np.concatenate([pts, np.cos(th_)[:, None], np.sin(th_)[:, None]], 1)
        else:
            out["pose"] = pts
        out["w"] = (rng.uniform(0.5, 2.0, (B if batched else 1, 1)))
    else:
        dof = 3 if pk in ("se2", "vector3") else 2
        for nm in ("pose1", "pose2"):
            if pk == "se2":
                th_ = rng.uniform(-3, 3, B)
                out[nm] = np.concatenate([rng.standard_normal((B, 2)), np.cos(th_)[:, None], np.sin(th_)[:, None]], 1)
            else:
                out[nm] = rng.standard_normal((B, dof))
        out["vel1"], out["vel2"] = rng.standard_normal((B, dof)), rng.standard_normal((B, dof))
        out["dt"] = rng.uniform(0.05, 0.3, (B, 1)) if batched else np.array([[0.1]])
        if wk == "gp":
            nq = B if batched else 1
            A = rng.standard_normal((nq, dof, dof))
            out["Qc_inv"] = A @ np.transpose(A, (0, 2, 1)) + dof * np.eye(dof)[None]
            out["w_dt"] = rng.uniform(0.05, 0.3, (B, 1)) if batched else np.array([[0.2]])
        elif wk == "diag":
            out["w"] = rng.uniform(0.5, 2.0, (B if batched else 1, 2 * dof))
        else:
            out["w"] = rng.uniform(0.5, 2.0, (B if batched else 1, 1))
    return {k: v.astype(dt_) for k, v in out.items()}


def motion_planning_cost(th, torch, case, inp):
    """The cost function of one per-cost case over tensors `inp` (dict name -> tensor)."""
    name, pk, wk, batched = case
    if wk == "gp":
        W = th.eb.GPCostWeight(inp["Qc_inv"], th.Variable(inp["w_dt"], name="w_dt"))
    elif wk == "diag":
        W = th.DiagonalCostWeight(th.Variable(inp["w"], name="w"))
    else:
        W = th.ScaleCostWeight(th.Variable(inp["w"], name="w"))
    if name.startswith("col"):
        P = th.SE2 if pk == "se2" else th.Point2
        return th.eb.Collision2D(P(tensor=inp["pose"], name="pose"), th.Point2(tensor=inp["sdf_origin"], name="origin"),
                                 th.Variable(inp["sdf_data"], name="sdf"), th.Variable(inp["cell_size"], name="cell"),
                                 th.Variable(inp["cost_eps"], name="eps"), W, name="col")
    P = {"se2": th.SE2, "point2": th.Point2, "vector3": th.Vector}[pk]
    mk = lambda k: (P(tensor=inp[k], name=k) if pk != "vector3" else th.Vector(tensor=inp[k], name=k))
    cls = th.eb.GPMotionModel if wk == "gp" else th.eb.DoubleIntegrator
    return cls(mk("pose1"), th.Vector(tensor=inp["vel1"], name="vel1"), mk("pose2"), th.Vector(tensor=inp["vel2"], name="vel2"),
               th.Variable(inp["dt"], name="dt"), W, name="di")


def make_motion_planning(th):
    """tests/golden/motion_planning_kat.npz: inputs of the tutorial's tarpit problems, the straight-line initial values, the planner
    objective's SparseLinearization (A_val, b) for Point2 and SE2 poses, a dense-solver LM trace (100 steps, 10 iterations, damping 0.1,
    adaptive), gradients of an imitation loss w.r.t. the collision weight [B,1] and cost_eps (UNROLL 3 iterations, IMPLICIT), and the
    weighted errors / Jacobians of every new cost function case (MP_COST_CASES) in f64 and f32."""
    import torch
    inputs = motion_planning_inputs(torch)
    out = {"in_" + k: np.asarray(v) for k, v in inputs.items()}
    for pk in ("point2", "se2"):
        init = motion_planning_straight_line(torch, inputs, pk)
        out[f"init_{pk}"] = np.stack([init[f"pose_{i}"].numpy() for i in range(101)], 0)
        out[f"init_vel_{pk}"] = np.stack([init[f"vel_{i}"].numpy() for i in range(101)], 0)
        objective, poses, vels, _ = motion_planning_problem(th, torch, inputs, pk)
        objective.update(init)
        lin = th.SparseLinearization(objective)
        lin.linearize()
        out[f"A_val_{pk}"], out[f"b_{pk}"] = lin.A_val.numpy(), lin.b.numpy()
        out[f"A_col_ind_{pk}"], out[f"A_row_ptr_{pk}"] = np.asarray(lin.A_col_ind), np.asarray(lin.A_row_ptr)
        out[f"err0_{pk}"] = objective.error_metric().numpy()
        print(pk, "costs", len(objective.cost_functions), "dim", objective.dim(), "cols", lin.num_cols)
    # LM trace (Point2, dense)
    lm = dict(damping=0.1, adaptive_damping=True)
    objective, poses, vels, _ = motion_planning_problem(th, torch, inputs, "point2")
    objective.update(motion_planning_straight_line(torch, inputs, "point2"))
    opt = th.LevenbergMarquardt(objective, linear_solver_cls=th.CholeskyDenseSolver, max_iterations=10, step_size=1.0,
                                abs_err_tolerance=0, rel_err_tolerance=0)
    errs, deltas, lams = [], [], []

    def cb(optimizer, info, delta, it):
        errs.append(info.last_err.detach().numpy().copy()); deltas.append(delta.detach().numpy().copy())
        d = optimizer._damping
        lams.append(d.detach().numpy().copy() if torch.is_tensor(d) else np.full(delta.shape[0], d))
    with torch.no_grad():
        opt.optimize(end_iter_callback=cb, **lm)
    out["trace_err"], out["trace_delta"], out["trace_lam"] = np.stack(errs, 0), np.stack(deltas, 0), np.stack(lams, 0)
    out["final_poses"] = np.stack([p.tensor.numpy() for p in poses], 0)
    # imitation-loss gradients w.r.t. the collision weight [B,1] and cost_eps [B,1]
    expert = torch.as_tensor(inputs["expert"])
    for mode, iters in (("unroll", 3), ("implicit", 10)):
        cw = torch.full((2, 1), float(inputs["collision_weight"]), dtype=torch.float64, requires_grad=True)
        ce = torch.full((2, 1), float(inputs["epsilon_dist"]), dtype=torch.float64, requires_grad=True)
        objective, poses, vels, _ = motion_planning_problem(th, torch, inputs, "point2", collision_w=cw, cost_eps=ce)
        opt = th.LevenbergMarquardt(objective, linear_solver_cls=th.CholeskyDenseSolver, max_iterations=iters, step_size=1.0,
                                    abs_err_tolerance=0, rel_err_tolerance=0)
        sol, _ = th.TheseusLayer(opt).forward(motion_planning_straight_line(torch, inputs, "point2"),
                                              optimizer_kwargs=dict(lm, backward_mode=mode))
        P = torch.stack([sol[f"pose_{i}"] for i in range(101)], 2)
        loss = ((P - expert[:, :2]) ** 2).sum()
        loss.backward()
        out[f"grad_cw_{mode}"], out[f"grad_eps_{mode}"], out[f"loss_{mode}"] = cw.grad.numpy(), ce.grad.numpy(), loss.detach().numpy()
    # per-cost known answers
    for case in MP_COST_CASES:
        for dn, tdt in (("f64", torch.float64), ("f32", torch.float32)):
            inp = motion_planning_cost_inputs(case, dn)
            cf = motion_planning_cost(th, torch, case, {k: torch.from_numpy(v) for k, v in inp.items()})
            jacs, err = cf.weighted_jacobians_error()
            pre = f"cost_{case[0]}_{dn}_"
            out[pre + "err"] = err.detach().numpy()
            for i, J in enumerate(jacs):
                out[pre + f"J{i}"] = J.detach().numpy()
    np.savez_compressed(os.path.join(HERE, "motion_planning_kat.npz"), **out)
    print("motion_planning: trace err", out["trace_err"][:, 0], "grads", out["grad_cw_unroll"].ravel(), out["grad_eps_implicit"].ravel())


if __name__ == "__main__":
    import sys
    sys.path.insert(0, HERE)
    from make_golden import _import_reference
    make_motion_planning(_import_reference()[0])

"""Shared pieces of the 2-D motion-planning tests (tests/test_motion_planning.py on the CPU, tests/test_gpu_motion_planning.py on the
GPU): the problem builders of tests/golden/make_golden_motion_planning.py (the same code built the reference's objective for
motion_planning_kat.npz)
and the checks that run the fused kernels through the engine -- on the device, or on the host emulation of thb_costs.cu."""
import numpy as np
import torch

import theseus_b200 as th
from helpers import load


def _golden_module():
    """tests/golden/make_golden_motion_planning.py: pure problem builders only (the reference is imported under __main__ there)."""
    import importlib.util
    import os
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "make_golden_motion_planning.py")
    spec = importlib.util.spec_from_file_location("make_golden_motion_planning", path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod

LM = dict(damping=0.1, adaptive_damping=True)


def golden():
    return load("motion_planning_kat")


def inputs_of(g):
    keys = [k[3:] for k in g.files if k.startswith("in_")]
    return {k: (g["in_" + k].item() if g["in_" + k].ndim == 0 else g["in_" + k]) for k in keys}


def straight_line(g, pose_type, device):
    G = _golden_module()
    return {k: v.to(device) for k, v in G.motion_planning_straight_line(torch, inputs_of(g), pose_type).items()}


def planner(g, pose_type="point2", device="cuda", **kw):
    G = _golden_module()
    objective, poses, vels, leaves = G.motion_planning_problem(th, torch, inputs_of(g), pose_type, device=device, **kw)
    objective.update(straight_line(g, pose_type, device))
    return objective, poses, vels, leaves


def check_planner_linearization(g, pose_type, device):
    """A_val / b of the planner objective at the straight-line initialisation against the reference's SparseLinearization; the
    fused kernels carry every cost function except the SE2 planner's own _XYDifference goal cost."""
    objective, poses, vels, _ = planner(g, pose_type, device)
    lin = th.SparseLinearization(objective)
    lin.linearize()
    eng = objective.engine()
    names = [eng.costs[f].name for f in eng.generic]
    assert names == ([] if pose_type == "point2" else ["pose_N"])
    assert np.array_equal(np.asarray(lin.A_row_ptr.cpu() if torch.is_tensor(lin.A_row_ptr) else lin.A_row_ptr), g[f"A_row_ptr_{pose_type}"])
    assert np.array_equal(np.asarray(lin.A_col_ind.cpu() if torch.is_tensor(lin.A_col_ind) else lin.A_col_ind), g[f"A_col_ind_{pose_type}"])
    np.testing.assert_allclose(lin.A_val.cpu().numpy(), g[f"A_val_{pose_type}"], rtol=1e-10, atol=1e-10)
    np.testing.assert_allclose(lin.b.cpu().numpy(), g[f"b_{pose_type}"], rtol=1e-10, atol=1e-10)
    with torch.no_grad():
        np.testing.assert_allclose(objective.error_metric().cpu().numpy(), g[f"err0_{pose_type}"], rtol=1e-10)


def tolerances(dn, ref):
    """f64: 1e-10 relative; f32: 2e-4 relative plus 2e-5 of the largest entry (sums of products of entries of both signs cancel)."""
    if dn == "f64":
        return dict(rtol=1e-10, atol=1e-12)
    return dict(rtol=2e-4, atol=2e-5 * max(1.0, float(np.abs(ref).max())))


def cost_case_objective(case, dn, device):
    G = _golden_module()
    inp = {k: torch.from_numpy(v).to(device) for k, v in G.motion_planning_cost_inputs(case, dn).items()}
    cf = G.motion_planning_cost(th, torch, case, inp)
    objective = th.Objective(dtype=torch.float64 if dn == "f64" else torch.float32)
    objective.add(cf)
    if str(device) != "cpu":
        objective.to(device)
    return objective, cf


def check_cost_case_on_engine(g, case, dn, device):
    """Weighted error and Jacobians of one per-cost case through the engine's fused kernels (A_val / b of a one-cost objective whose
    columns are the cost's variables in order) and through the error pass, against the reference's values."""
    objective, cf = cost_case_objective(case, dn, device)
    eng = objective.engine()
    assert eng.generic == [] and len(eng.groups) == 1
    A, b = eng.linearize_sparse()
    B = objective.batch_size
    pre = f"cost_{case[0]}_{dn}_"
    Jref = np.concatenate([g[pre + f"J{i}"] for i in range(cf.num_optim_vars())], axis=2)
    np.testing.assert_allclose(A.cpu().numpy().reshape(B, cf.dim(), -1), Jref, **tolerances(dn, Jref))
    np.testing.assert_allclose(-b.cpu().numpy(), g[pre + "err"], **tolerances(dn, g[pre + "err"]))
    em, eref = eng.error_metric().cpu().numpy(), 0.5 * (g[pre + "err"].astype(np.float64) ** 2).sum(1)
    np.testing.assert_allclose(em, eref, rtol=1e-9 if dn == "f64" else 1e-3, atol=1e-12 if dn == "f64" else 1e-4 * max(1.0, eref.max()))


def lm_trace(objective, poses, **opt_kw):
    opt = th.LevenbergMarquardt(objective, max_iterations=10, step_size=1.0, abs_err_tolerance=0, rel_err_tolerance=0, **opt_kw)
    errs, deltas, lams = [], [], []

    def cb(optimizer, info, delta, it):
        errs.append(info.last_err.cpu().numpy().copy()); deltas.append(delta.cpu().numpy().copy())
        d = optimizer._damping
        lams.append(d.cpu().numpy().copy() if torch.is_tensor(d) else np.full(delta.shape[0], d))
    with torch.no_grad():
        info = opt.optimize(end_iter_callback=cb, **LM)
    return np.stack(errs, 0), np.stack(deltas, 0), np.stack(lams, 0), info


def decisive_per_item(err0, trace_err, tol=1e-7, floor=1.5):
    """Per batch item: the leading iterations whose accept / reject decision is numerically defined (helpers.decisive_iterations, per
    item): an accepted step reduced the error by more than `tol` relative, or a rejected step (error unchanged) was taken while the error
    was still above `floor` times the final one -- far from the rounding floor where the reference's decisions become arbitrary."""
    ks = []
    for i in range(trace_err.shape[1]):
        prev, k = err0[i], 0
        for it in range(trace_err.shape[0]):
            e = trace_err[it, i]
            red = (prev - e) / prev
            if not (red > tol or (red == 0 and e > floor * trace_err[-1, i])):
                break
            prev, k = e, k + 1
        ks.append(k)
    return ks


def check_lm_trace(g, errs, deltas, lams):
    """Error 1e-8 relative, delta 1e-5 norm-wise and lambda 1e-12 while the reference's decision is defined (decisive_per_item; the
    collision clamp makes the cost non-smooth); final error 1e-6."""
    ref = g["trace_err"]
    assert errs.shape == ref.shape
    ks = decisive_per_item(g["err0_point2"], ref)
    assert min(ks) >= 3, ks
    for i, k in enumerate(ks):
        np.testing.assert_allclose(errs[:k, i], ref[:k, i], rtol=1e-8)
        for it in range(k):
            dref = g["trace_delta"][it, i]
            assert np.linalg.norm(deltas[it, i] - dref) / np.linalg.norm(dref) < 1e-5, (i, it)
            np.testing.assert_allclose(lams[it, i], g["trace_lam"][it, i], rtol=1e-12)
    np.testing.assert_allclose(errs[-1], ref[-1], rtol=1e-6)

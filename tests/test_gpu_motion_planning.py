"""2-D motion planning on the GPU (th.eb.Collision2D, GPMotionModel + GPCostWeight on the fused kernels of thb_costs.cu): the
per-cost known answers through the C ABI, the planner objective's linearization and LM trace (dense, multifrontal and lane solvers)
against the reference (tests/golden/motion_planning_kat.npz: the tutorial's two tarpit maps, 100 steps), CUDA-graph replay and batch-size
independence bit for bit, and the imitation-loss gradients w.r.t. the collision weight and cost_eps in UNROLL and IMPLICIT mode."""
import numpy as np
import pytest
import torch

import theseus_b200 as th
import mp_common as M
from mp_common import _golden_module

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("dn", ["f64", "f32"])
@pytest.mark.parametrize("name", [c[0] for c in _golden_module().MP_COST_CASES])
def test_cost_known_answers_through_the_c_abi(name, dn):
    case = next(c for c in _golden_module().MP_COST_CASES if c[0] == name)
    M.check_cost_case_on_engine(M.golden(), case, dn, "cuda")


@pytest.mark.parametrize("pose_type", ["point2", "se2"])
def test_planner_linearization(pose_type):
    M.check_planner_linearization(M.golden(), pose_type, "cuda")


@pytest.mark.parametrize("solver", ["dense", "sparse_front", "sparse_lane"])
def test_planner_lm_trace(solver):
    g = M.golden()
    objective, poses, vels, _ = M.planner(g, "point2", "cuda")
    skw = dict(linear_solver_cls=th.CholeskyDenseSolver) if solver == "dense" else dict(
        linear_solver_cls=th.BaspachoSparseSolver, linearization_cls=th.SparseLinearization,
        linear_solver_kwargs=dict(layout=solver.split("_")[1]))
    errs, deltas, lams, info = M.lm_trace(objective, poses, **skw)
    assert objective.engine().generic == []
    M.check_lm_trace(g, errs, deltas, lams)
    if solver == "dense":
        final = np.stack([p.tensor.cpu().numpy() for p in poses], 0)
        np.testing.assert_allclose(final, g["final_poses"], rtol=1e-6, atol=1e-8)


@pytest.mark.parametrize("pose_type", ["point2", "se2"])
def test_cuda_graph_is_bitwise_identical_to_eager(pose_type):
    g = M.golden()
    res = {}
    for mode in (False, True):
        objective, poses, vels, _ = M.planner(g, pose_type, "cuda")
        opt = th.LevenbergMarquardt(objective, linear_solver_cls=th.CholeskyDenseSolver, max_iterations=6, step_size=1.0,
                                    abs_err_tolerance=0, rel_err_tolerance=0, cuda_graph=mode)
        layer = th.TheseusLayer(opt)
        with torch.no_grad():
            vals, info = layer.forward(M.straight_line(g, pose_type, "cuda"), optimizer_kwargs=dict(M.LM, track_err_history=True))
        res[mode] = (torch.stack([vals[p.name] for p in poses]).cpu().numpy(), info.err_history.numpy())
    for a, b in zip(res[False], res[True]):
        assert np.array_equal(a, b)


def test_item_results_do_not_depend_on_the_batch_size():
    """Item i of a 64-item batch (maps, starts and goals drawn per item) is bitwise the same item alone: the fused linearization, the
    error pass and the first LM step (delta) on the multifrontal solver.  (Later iterations are not compared: the LM loop's batch-global
    decisions -- an all-rejected batch retries the step, as in the reference -- make a lone item's path differ from its path in a batch.)"""
    g = M.golden()
    inp = M.inputs_of(g)
    gen = np.random.default_rng(4)
    B = 64
    pick = gen.integers(0, 2, B)
    big = dict(inp, sdf_data=inp["sdf_data"][pick], sdf_origin=inp["sdf_origin"][pick], cell_size=inp["cell_size"][pick],
               start=inp["start"][pick] + gen.normal(0, 0.05, (B, 2)), goal=inp["goal"][pick] + gen.normal(0, 0.05, (B, 2)),
               start_se2=inp["start_se2"][pick])
    G = _golden_module()

    def solve(inputs):
        objective, poses, vels, _ = G.motion_planning_problem(th, torch, inputs, "point2", device="cuda")
        objective.update({k: v.cuda() for k, v in G.motion_planning_straight_line(torch, inputs, "point2").items()})
        eng = objective.engine()
        A, b = eng.linearize_sparse()
        lin = (A.cpu().numpy().copy(), b.cpu().numpy().copy(), eng.error_metric().cpu().numpy().copy())
        opt = th.LevenbergMarquardt(objective, linear_solver_cls=th.BaspachoSparseSolver, linearization_cls=th.SparseLinearization,
                                    linear_solver_kwargs=dict(layout="front"), max_iterations=1, step_size=1.0,
                                    abs_err_tolerance=0, rel_err_tolerance=0)
        deltas = []
        with torch.no_grad():
            opt.optimize(end_iter_callback=lambda o, info, delta, it: deltas.append(delta.cpu().numpy().copy()), **M.LM)
        return lin, deltas[0]
    (A, b, e), delta = solve(big)
    for i in (0, 17, 63):
        (A1, b1, e1), t1 = solve({k: (v[i:i + 1] if isinstance(v, np.ndarray) and v.ndim >= 2 and v.shape[0] == B else v) for k, v in big.items()})
        assert np.array_equal(A[i:i + 1], A1) and np.array_equal(b[i:i + 1], b1) and np.array_equal(e[i:i + 1], e1), i
        assert np.array_equal(delta[i:i + 1], t1), i


@pytest.mark.parametrize("mode,iters", [("unroll", 3), ("implicit", 10)])
def test_imitation_loss_gradients(mode, iters):
    """d loss / d collision weight and d loss / d cost_eps of loss = |trajectory - expert|^2 against the reference (1e-6 relative)."""
    g = M.golden()
    inp = M.inputs_of(g)
    d = torch.float64
    cw = torch.full((2, 1), float(inp["collision_weight"]), dtype=d, device="cuda", requires_grad=True)
    ce = torch.full((2, 1), float(inp["epsilon_dist"]), dtype=d, device="cuda", requires_grad=True)
    objective, poses, vels, _ = _golden_module().motion_planning_problem(th, torch, inp, "point2", device="cuda", collision_w=cw, cost_eps=ce)
    opt = th.LevenbergMarquardt(objective, linear_solver_cls=th.CholeskyDenseSolver, max_iterations=iters, step_size=1.0,
                                abs_err_tolerance=0, rel_err_tolerance=0)
    sol, _ = th.TheseusLayer(opt).forward(M.straight_line(g, "point2", "cuda"), optimizer_kwargs=dict(M.LM, backward_mode=mode))
    P = torch.stack([sol[f"pose_{i}"] for i in range(101)], 2)
    loss = ((P - torch.from_numpy(inp["expert"][:, :2]).cuda()) ** 2).sum()
    loss.backward()
    np.testing.assert_allclose(loss.item(), g[f"loss_{mode}"], rtol=1e-6)
    np.testing.assert_allclose(cw.grad.cpu().numpy(), g[f"grad_cw_{mode}"], rtol=1e-6, atol=1e-9)
    np.testing.assert_allclose(ce.grad.cpu().numpy(), g[f"grad_eps_{mode}"], rtol=1e-6, atol=1e-9)

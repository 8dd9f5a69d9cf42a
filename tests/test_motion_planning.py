"""2-D motion planning on the CPU: the classes of th.eb (Collision2D, SignedDistanceField2D, DoubleIntegrator, GPMotionModel,
GPCostWeight) -- constructors and validation as in the reference, their torch restatements and the fused kernels (thb_costs.cu on the
host emulation, tests/simt/) against the reference's values (tests/golden/motion_planning_kat.npz, make_golden_motion_planning.py), and
the field offsets of thb_cost_group (include/thb200.h) against _lib.CostGroup."""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest
import torch

import theseus_b200 as th
from theseus_b200 import _lib
import mp_common as M
from mp_common import _golden_module
from test_simt_engine_emulation import _emulation_mode

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)


@pytest.fixture(scope="module")
def emu_lib():
    return _emulation_mode().load_emulated_lib()


@pytest.fixture
def emulated(monkeypatch, emu_lib):
    _emulation_mode().patch_host(monkeypatch.setattr, emu_lib)
    return emu_lib


def _case_ids():
    return [c[0] for c in _golden_module().MP_COST_CASES]


# ---------------------------------------------------------------------------------------------------------------- class API
def test_constructors_validate_like_the_reference():
    d = torch.float64
    sdf = torch.zeros(1, 4, 5, dtype=d)
    with pytest.raises(ValueError):
        th.eb.Collision2D(th.Vector(3, dtype=d), torch.zeros(1, 2, dtype=d), sdf, 0.1, 0.2, th.ScaleCostWeight(1.0))
    with pytest.raises(ValueError):
        th.eb.SignedDistanceField2D(torch.zeros(1, 2), 0.1, sdf_data=torch.zeros(4, 5))
    with pytest.raises(ValueError):
        th.eb.SignedDistanceField2D(torch.zeros(1, 2), 0.1)
    with pytest.raises(ValueError):
        th.eb.SignedDistanceField2D.convert_cell_size(1)
    eye = torch.eye(2, dtype=d)
    with pytest.raises(ValueError):
        th.eb.GPCostWeight(eye, 0.0)
    with pytest.raises(ValueError):
        th.eb.GPCostWeight(torch.zeros(2, 3, dtype=d), 0.1)
    with pytest.raises(ValueError):
        th.eb.GPCostWeight(-eye, 0.1)
    with pytest.raises(ValueError):
        th.eb.GPCostWeight(torch.zeros(1, 1, 2, 2, dtype=d), 0.1)
    p = lambda n: th.Point2(dtype=d, name=n)
    v = lambda n, k=2: th.Vector(k, dtype=d, name=n)
    with pytest.raises(ValueError):
        th.eb.GPMotionModel(p("a"), v("b"), p("c"), v("e"), 0.1, th.ScaleCostWeight(1.0))
    with pytest.raises(ValueError):
        th.eb.DoubleIntegrator(p("a"), v("b", 3), p("c"), v("e"), 0.1, th.ScaleCostWeight(1.0))


def test_schema_kinds_dims_and_copies():
    d = torch.float64
    sdf = torch.zeros(1, 4, 5, dtype=d)
    w = th.ScaleCostWeight(torch.tensor(1.0, dtype=d))
    c = th.eb.Collision2D(th.Point2(dtype=d), torch.zeros(1, 2, dtype=d), sdf, torch.tensor([[0.1]], dtype=d), torch.tensor(0.2, dtype=d), w)
    assert c.dim() == 1 and c.schema()[0] == 8 and len(c.schema()[1]) == 4
    assert th.eb.Collision2D(th.SE2(dtype=d), torch.zeros(1, 2, dtype=d), sdf, 0.1, 0.2, w).schema()[0] == 9
    gw = th.eb.GPCostWeight(torch.eye(3, dtype=d), torch.tensor(0.1, dtype=d))
    assert not gw.is_zero().any() and [x.shape for x in gw.aux_vars] == [(1, 3, 3), (1, 1)]
    dt = torch.tensor(0.1, dtype=d)
    gp = th.eb.GPMotionModel(th.SE2(dtype=d), th.Vector(3, dtype=d), th.SE2(dtype=d), th.Vector(3, dtype=d), dt, gw)
    assert gp.dim() == 6 and gp.schema()[0] == 11 and gp.schema()[1][1] is gw.dt
    v3 = th.eb.DoubleIntegrator(th.Vector(3, dtype=d), th.Vector(3, dtype=d), th.Vector(3, dtype=d), th.Vector(3, dtype=d), dt, w)
    assert v3.schema()[0] == 10 and len(v3.schema()[1]) == 1
    so2 = th.eb.DoubleIntegrator(th.SO2(dtype=d), th.Vector(1, dtype=d), th.SO2(dtype=d), th.Vector(1, dtype=d), dt, w)
    assert so2.schema()[0] is None                             # generic route on the same torch restatement
    robust = th.RobustCostFunction(c, th.HuberLoss, th.Variable(torch.zeros(1, 1, dtype=d)))
    assert robust.schema()[0] is None                          # no fused robust path for the new kinds
    for cf in (c, gp):
        cp = cf.copy()
        assert type(cp) is type(cf) and cp.optim_vars[0] is not cf.optim_vars[0]
    # set_aux_var_at keeps the SDF container on the new data
    new = th.Variable(torch.ones(1, 4, 5, dtype=d))
    c.set_aux_var_at(1, new)
    assert c.sdf.sdf_data is new


def test_signed_distance_matches_the_kernel_formula_and_the_reference_semantics():
    """Distance / gradient of SignedDistanceField2D.signed_distance: bilinear inside, 0 and zero gradient outside; the gradient is
    the derivative of the distance (finite differences)."""
    d = torch.float64
    gen = torch.Generator().manual_seed(0)
    data = torch.randn(2, 6, 7, generator=gen, dtype=d)
    sdf = th.eb.SignedDistanceField2D(torch.tensor([[0.0, 0.0], [1.0, -1.0]], dtype=d), torch.tensor([[0.5], [0.25]], dtype=d), sdf_data=data)
    pts = torch.tensor([[[0.3, 1.1, -0.1, 2.9], [0.2, 2.4, 0.5, 0.7]], [[1.2, 2.07, 0.9, 2.4], [-0.6, -0.3, 0.1, 0.2]]], dtype=d)
    dist, jac = sdf.signed_distance(pts)
    assert dist.shape == (2, 4) and jac.shape == (2, 4, 2)
    assert dist[0, 2] == 0 and (jac[0, 2] == 0).all() and dist[1, 2] == 0       # out of bounds (x < origin, x > far edge)
    h = 1e-6
    for k in range(2):
        dp = torch.zeros_like(pts); dp[:, k] = h
        fd = (sdf.signed_distance(pts + dp)[0] - sdf.signed_distance(pts - dp)[0]) / (2 * h)
        inside = dist != 0
        np.testing.assert_allclose(jac[..., k][inside].numpy(), fd[inside].numpy(), rtol=1e-6, atol=1e-8)
    occ = torch.zeros(1, 8, 8, dtype=d); occ[0, 3:5, 3:5] = 1.0
    from_map = th.eb.SignedDistanceField2D(torch.zeros(1, 2, dtype=d), torch.tensor([[0.5]], dtype=d), occupancy_map=occ)
    assert from_map.sdf_data.tensor[0, 3, 3] < 0 < from_map.sdf_data.tensor[0, 0, 0]


# ------------------------------------------------------------------------------------------------------ torch restatements
@pytest.mark.parametrize("dn", ["f64", "f32"])
@pytest.mark.parametrize("name", _case_ids())
def test_torch_restatements_against_the_reference(name, dn):
    G, g = _golden_module(), M.golden()
    case = next(c for c in G.MP_COST_CASES if c[0] == name)
    objective, cf = M.cost_case_objective(case, dn, "cpu")
    jacs, err = cf.weighted_jacobians_error()
    pre = f"cost_{name}_{dn}_"
    np.testing.assert_allclose(err.numpy(), g[pre + "err"], **M.tolerances(dn, g[pre + "err"]))
    for i, J in enumerate(jacs):
        np.testing.assert_allclose(J.numpy(), g[pre + f"J{i}"], **M.tolerances(dn, g[pre + f"J{i}"]))


def test_gp_weight_on_an_autodiff_cost_function():
    """A GPCostWeight on an AutoDiffCostFunction (the generic route) weights like the reference: U e, U J."""
    d = torch.float64
    gen = torch.Generator().manual_seed(1)
    x = th.Vector(tensor=torch.randn(3, 2, generator=gen, dtype=d), name="x")
    y = th.Vector(tensor=torch.randn(3, 2, generator=gen, dtype=d), name="y")
    w = th.eb.GPCostWeight(torch.tensor([[2.0, 0.3], [0.3, 1.0]], dtype=d), torch.tensor(0.2, dtype=d))
    cf = th.AutoDiffCostFunction([x], lambda optim_vars, aux_vars: torch.cat([optim_vars[0].tensor ** 2, aux_vars[0].tensor * optim_vars[0].tensor], 1),
                                 4, cost_weight=w, aux_vars=[y])
    jacs, err = cf.weighted_jacobians_error()
    U = w._compute_cost_weight()
    e0 = torch.cat([x.tensor ** 2, y.tensor * x.tensor], 1)
    J0 = torch.cat([torch.diag_embed(2 * x.tensor), torch.diag_embed(y.tensor)], 1)
    np.testing.assert_allclose(err.numpy(), (U @ e0.unsqueeze(2)).squeeze(2).numpy(), rtol=1e-13)
    np.testing.assert_allclose(jacs[0].numpy(), (U @ J0).numpy(), rtol=1e-13)
    assert torch.allclose(U.transpose(1, 2) @ U, torch.tensor([[12 / 0.008 * 2.0, 12 / 0.008 * 0.3, -6 / 0.04 * 2.0, -6 / 0.04 * 0.3],
                                                               [12 / 0.008 * 0.3, 12 / 0.008, -6 / 0.04 * 0.3, -6 / 0.04],
                                                               [-6 / 0.04 * 2.0, -6 / 0.04 * 0.3, 4 / 0.2 * 2.0, 4 / 0.2 * 0.3],
                                                               [-6 / 0.04 * 0.3, -6 / 0.04, 4 / 0.2 * 0.3, 4 / 0.2]], dtype=d))


def test_effector_contact_keeps_its_values_on_the_shared_lookup():
    """EffectorObjectContactPlanar now uses the lookup of SignedDistanceField2D: its error equals the SDF's distance minus the radius."""
    d = torch.float64
    gen = torch.Generator().manual_seed(2)
    data = torch.randn(1, 8, 8, generator=gen, dtype=d)
    obj = th.SE2(x_y_theta=torch.tensor([[0.1, -0.2, 0.3], [0.0, 0.1, -1.0]], dtype=d))
    eff = th.SE2(x_y_theta=torch.tensor([[0.4, 0.1, 0.0], [0.2, 0.5, 0.0]], dtype=d))
    origin, cell = torch.tensor([[-0.5, -0.5]], dtype=d), torch.tensor([[0.15]], dtype=d)
    cf = th.eb.EffectorObjectContactPlanar(obj, eff, origin, data, cell, torch.tensor(0.05, dtype=d), th.ScaleCostWeight(torch.tensor(1.0, dtype=d)))
    p = obj.transform_to(eff.xy()).tensor if hasattr(obj, "transform_to") else None
    sdf = th.eb.SignedDistanceField2D(origin, cell, sdf_data=data)
    dist, _ = sdf.signed_distance(p.unsqueeze(-1))
    np.testing.assert_allclose(cf.error().numpy(), (dist - 0.05).abs().numpy(), rtol=1e-14)


# ------------------------------------------------------------------------------------------------ kernels on the emulation
@pytest.mark.parametrize("dn", ["f64", "f32"])
@pytest.mark.parametrize("name", _case_ids())
def test_kernels_on_the_host_emulation_against_the_reference(emulated, name, dn):
    G, g = _golden_module(), M.golden()
    case = next(c for c in G.MP_COST_CASES if c[0] == name)
    M.check_cost_case_on_engine(g, case, dn, "cpu")


@pytest.mark.parametrize("pose_type", ["point2", "se2"])
def test_planner_linearization_on_the_host_emulation(emulated, pose_type):
    M.check_planner_linearization(M.golden(), pose_type, "cpu")


def test_planner_lm_trace_on_the_host_emulation(emulated):
    g = M.golden()
    objective, poses, vels, _ = M.planner(g, "point2", "cpu")
    errs, deltas, lams, info = M.lm_trace(objective, poses, linear_solver_cls=th.CholeskyDenseSolver)
    M.check_lm_trace(g, errs, deltas, lams)


# -------------------------------------------------------------------------------------------------------------- ABI
def test_cost_group_field_offsets_match_the_header():
    """thb_cost_group offsets from the C compiler (offsetof on include/thb200.h) == _lib.CostGroup's; test_abi.py checks prototypes only."""
    cc = shutil.which("cc") or shutil.which("gcc")
    if cc is None:
        pytest.skip("no C compiler")
    fields = [f for f, _ in _lib.CostGroup._fields_]
    src = "#include <stdio.h>\n#include <stddef.h>\n#include \"thb200.h\"\nint main(void){\n" + "".join(
        f'  printf("%s %zu\\n", "{f}", offsetof(thb_cost_group, {f}));\n' for f in fields) + '  printf("sizeof %zu\\n", sizeof(thb_cost_group));\n  return 0;\n}\n'
    import tempfile
    with tempfile.TemporaryDirectory() as tmp:
        c_file, exe = os.path.join(tmp, "off.c"), os.path.join(tmp, "off")
        with open(c_file, "w") as fh:
            fh.write(src)
        subprocess.run([cc, "-I", os.path.join(ROOT, "include"), c_file, "-o", exe], check=True)
        out = subprocess.run([exe], check=True, capture_output=True, text=True).stdout.split("\n")
    got = dict(line.split() for line in out if line)
    for f in fields:
        assert int(got[f]) == getattr(_lib.CostGroup, f).offset, f
    assert int(got["sizeof"]) == C.sizeof(_lib.CostGroup)

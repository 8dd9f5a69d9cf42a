"""`th.eb` namespace of the reference (theseus/embodied/__init__.py): Between / Local / Reprojection and the 2-D motion-planning costs
(Collision2D, DoubleIntegrator / GPMotionModel with GPCostWeight) have fused CUDA schemas; MovingFrameBetween and the tactile costs run
on the torch path (torch.func Jacobians + tangent-space projection, like an AutoDiffCostFunction)."""
from typing import List, Optional, Tuple, Union

import torch

from .core import (COST_COLLISION2D_POINT2, COST_COLLISION2D_SE2, COST_DOUBLE_INTEGRATOR_SE2, COST_DOUBLE_INTEGRATOR_VECTOR,  # noqa: F401
                   WEIGHT_GP, Between, CostFunction, CostWeight, Difference, Local, Reprojection)
from .geometry import SE2, LieGroup, Point2, Variable, Vector, as_variable


def _bilinear_sdf(data, ox, oy, cell, px, py):
    """Bilinear lookup of signed_distance_field.py:163-241: grid data [Bs, rows, cols], cell (r, c) at (ox, oy) + (c, r) * cell;
    floor / ceil indices clamped to the grid, the interpolation weights not; 0 outside [ox, ox + (cols-1) cell] x [oy, ...].
    px, py [B, ...] (the batch index of `data` is broadcast over the trailing dimensions); ox, oy, cell broadcast against them.
    Returns (dist, d dist / d px, d dist / d py) -- the gradient is 0 outside the grid, like the reference's."""
    nrows, ncols = data.shape[-2], data.shape[-1]
    oob = (px < ox) | (px > ox + (ncols - 1.0) * cell) | (py < oy) | (py > oy + (nrows - 1.0) * cell)
    col, row = (px - ox) / cell, (py - oy) / cell
    lr, lc = torch.floor(row), torch.floor(col)
    hr, hc = lr + 1.0, lc + 1.0
    lri, lci = lr.long().clamp(0, nrows - 1), lc.long().clamp(0, ncols - 1)
    hri, hci = hr.long().clamp(0, nrows - 1), hc.long().clamp(0, ncols - 1)
    bi = torch.arange(data.shape[0], device=data.device).view((-1,) + (1,) * (px.ndim - 1))
    g = lambda r, c: data[bi, r, c]
    s_ll, s_hl, s_lh, s_hh = g(lri, lci), g(hri, lci), g(lri, hci), g(hri, hci)
    dist = (hr - row) * (hc - col) * s_ll + (row - lr) * (hc - col) * s_hl + (hr - row) * (col - lc) * s_lh + (row - lr) * (col - lc) * s_hh
    dist = torch.where(oob, torch.zeros_like(dist), dist)    # sdf_boundary_value = 0 (signed_distance_field.py:26)
    jx = ((hr - row) * (s_lh - s_ll) + (row - lr) * (s_hh - s_hl)) / cell
    jy = ((hc - col) * (s_hl - s_ll) + (col - lc) * (s_hh - s_lh)) / cell
    zero = torch.zeros_like(jx)
    return dist, torch.where(oob, zero, jx), torch.where(oob, zero, jy)


class SignedDistanceField2D:
    """theseus/embodied/collision/signed_distance_field.py:16-246: a batch of 2-D signed distance grids sdf_data [Bs, rows, cols] with
    origin [Bo, 2] (cell (r, c) at origin + (c, r) * cell_size) and cell_size [Bc, 1]; bilinear interpolation, 0 outside the grid."""

    def __init__(self, origin: Union[Point2, torch.Tensor], cell_size: Union[float, torch.Tensor, Variable],
                 sdf_data: Optional[Union[torch.Tensor, Variable]] = None, occupancy_map: Optional[Union[torch.Tensor, Variable]] = None,
                 occupancy_threshold: float = 0.75, sdf_boundary_value: float = 0.0):
        if occupancy_map is not None:
            if sdf_data is not None:
                raise ValueError("Only one of sdf_data and occupancy_map should be provided.")
            sdf_data = self._compute_sdf_data_from_map(occupancy_map, SignedDistanceField2D.convert_cell_size(cell_size).tensor,
                                                       threshold=occupancy_threshold)
        elif sdf_data is None:
            raise ValueError("Either sdf_data or argument occupancy_map should be provided.")
        self.update_data(origin, sdf_data, cell_size)
        self._num_rows = sdf_data.shape[1]
        self._num_cols = sdf_data.shape[2]
        self.sdf_boundary_value = sdf_boundary_value

    def _compute_sdf_data_from_map(self, occupancy_map_batch, cell_size: torch.Tensor, threshold: float = 0.75) -> Variable:
        """signed_distance_field.py:54-100 (gpmp2's map -> SDF: Euclidean distance transforms of the map and of its complement)."""
        from scipy import ndimage
        if isinstance(occupancy_map_batch, Variable):
            occupancy_map_batch = occupancy_map_batch.tensor
        if cell_size.shape[0] != occupancy_map_batch.shape[0]:
            cell_size = cell_size.expand(occupancy_map_batch.shape[0], 1)
        if occupancy_map_batch.ndim != 3:
            raise ValueError("Argument occupancy_map to SignedDistanceField2D must be a batch of matrices.")
        out = []
        for i in range(occupancy_map_batch.shape[0]):
            occupancy_map = occupancy_map_batch[i]
            cur_map = (occupancy_map > threshold).int()
            if torch.max(cur_map) == 0:
                max_map_size = 2 * cell_size[i].item() * max(occupancy_map.size(0), occupancy_map.size(1))
                sdf = torch.ones(occupancy_map.shape, dtype=occupancy_map.dtype) * max_map_size
            else:
                map_dist = ndimage.distance_transform_edt((1 - cur_map).cpu().numpy())
                inv_map_dist = ndimage.distance_transform_edt(cur_map.cpu().numpy())
                sdf = torch.tensor(map_dist - inv_map_dist, dtype=occupancy_map.dtype) * cell_size[i].cpu()
            out.append(sdf)
        return Variable(torch.stack(out))

    @staticmethod
    def convert_origin(origin: Union[torch.Tensor, Point2]) -> Point2:
        if not isinstance(origin, (Point2, torch.Tensor)):
            raise ValueError("Argument origin to SignedDistanceField2D must be either a tensor or a Point2 variable.")
        if not isinstance(origin, Point2):
            try:
                return Point2(tensor=origin)
            except ValueError:
                raise ValueError("Argument origin to SignedDistanceField2D must be a batch of 2D tensors.")
        return origin

    @staticmethod
    def convert_cell_size(cell_size: Union[float, torch.Tensor, Variable]) -> Variable:
        if not isinstance(cell_size, Variable):
            if not isinstance(cell_size, torch.Tensor):
                if not isinstance(cell_size, float):
                    raise ValueError("Argument cell_size must be either a Variable, tensor, or float.")
                cell_size = torch.tensor(cell_size).view(-1, 1)
            return Variable(cell_size)
        if not (cell_size.ndim == 1 or (cell_size.ndim == 2 and cell_size.shape[1] == 1)):
            raise ValueError("Argument cell_size must be a batch of 0D or 1D tensors.")
        return cell_size

    @staticmethod
    def convert_sdf_data(sdf_data: Union[torch.Tensor, Variable]) -> Variable:
        sdf_data = as_variable(sdf_data)
        if sdf_data.ndim != 3:
            raise ValueError("Argument sdf_data to SignedDistanceField2D must be a batch of matrices.")
        return sdf_data

    def update_data(self, origin, sdf_data, cell_size):
        self.origin = SignedDistanceField2D.convert_origin(origin)
        self.cell_size = SignedDistanceField2D.convert_cell_size(cell_size)
        self.sdf_data = SignedDistanceField2D.convert_sdf_data(sdf_data)

    def convert_points_to_cell(self, points: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
        """points [B, 2, N] -> (row, col, out_of_bounds), each [B, N]."""
        origin = self.origin.tensor.unsqueeze(-1) if self.origin.ndim == 2 else self.origin.tensor
        cell_size = self.cell_size.tensor if self.cell_size.ndim == 2 else self.cell_size.tensor.unsqueeze(-1)
        px, py = points[:, 0], points[:, 1]
        oob = ((px < origin[:, 0]) | (px > origin[:, 0] + (self._num_cols - 1.0) * cell_size)
               | (py < origin[:, 1]) | (py > origin[:, 1] + (self._num_rows - 1.0) * cell_size))
        return (py - origin[:, 1]) / cell_size, (px - origin[:, 0]) / cell_size, oob

    def signed_distance(self, points: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
        """points [B, 2, N] -> (distances [B, N], Jacobians d dist / d point [B, N, 2])."""
        origin = self.origin.tensor
        cell = self.cell_size.tensor if self.cell_size.ndim == 2 else self.cell_size.tensor.unsqueeze(-1)
        data = self.sdf_data.tensor
        px, py = points[:, 0], points[:, 1]
        B = max(px.shape[0], data.shape[0])
        if data.shape[0] != B:
            data = data.expand(B, -1, -1)
        px, py = px.expand(B, -1), py.expand(B, -1)
        dist, jx, jy = _bilinear_sdf(data, origin[:, 0:1], origin[:, 1:2], cell, px, py)
        if self.sdf_boundary_value != 0.0:
            _, _, oob = self.convert_points_to_cell(points.expand(B, -1, -1))
            dist = torch.where(oob, torch.full_like(dist, self.sdf_boundary_value), dist)
        return dist, torch.stack([jx, jy], dim=2)

    def to(self, *args, **kwargs):
        self.cell_size.to(*args, **kwargs)
        self.origin.to(*args, **kwargs)
        self.sdf_data.to(*args, **kwargs)


class Collision2D(CostFunction):
    """theseus/embodied/collision/collision.py:17-110: e = max(cost_eps - sdf(pose.xy), 0), dim 1; J = -grad sdf (times the SE2.xy
    Jacobian [R 0] for SE2 poses), zero where sdf > cost_eps.  Fused kernels THB_COST_COLLISION2D_POINT2 / _SE2 (thb_costs.cu)."""

    def __init__(self, pose: Union[Point2, SE2], sdf_origin: Union[Point2, torch.Tensor], sdf_data: Union[torch.Tensor, Variable],
                 sdf_cell_size: Union[float, torch.Tensor, Variable], cost_eps: Union[float, Variable, torch.Tensor],
                 cost_weight: CostWeight, name: Optional[str] = None):
        if not isinstance(pose, (Point2, SE2)):
            raise ValueError("Collision2D only accepts Point2 or SE2 poses.")
        super().__init__(cost_weight, name=name)
        self.pose = pose
        self.sdf_origin = SignedDistanceField2D.convert_origin(sdf_origin)
        self.sdf_data = SignedDistanceField2D.convert_sdf_data(sdf_data)
        self.sdf_cell_size = SignedDistanceField2D.convert_cell_size(sdf_cell_size)
        self.cost_eps = as_variable(cost_eps)
        self.cost_eps.tensor = self.cost_eps.tensor.view(-1, 1)
        self.register_optim_vars(["pose"])
        self.register_aux_vars(["sdf_origin", "sdf_data", "sdf_cell_size", "cost_eps"])
        self.sdf = SignedDistanceField2D(self.sdf_origin, self.sdf_cell_size, self.sdf_data)

    def dim(self) -> int:
        return 1

    def _torch_error(self, optim_tensors, aux_tensors):
        x = optim_tensors[0]
        origin, data, cell, eps = aux_tensors
        dist, _, _ = _bilinear_sdf(data, origin[..., 0], origin[..., 1], cell.view(-1), x[..., 0], x[..., 1])
        return (eps.view(-1) - dist).clamp(min=0).unsqueeze(-1)    # clamp's gradient is kept at dist == eps, like the reference

    def schema(self):
        return (COST_COLLISION2D_SE2 if isinstance(self.pose, SE2) else COST_COLLISION2D_POINT2,
                [self.sdf_origin, self.sdf_data, self.sdf_cell_size, self.cost_eps])

    def _copy_impl(self, new_name: Optional[str] = None) -> "Collision2D":
        return Collision2D(self.pose.copy(), self.sdf_origin.copy(), self.sdf_data.copy(), self.sdf_cell_size.copy(),
                           self.cost_eps.copy(), self.weight.copy(), name=new_name)

    def set_aux_var_at(self, index: int, variable: Variable):
        """Keeps the SDF container on the new auxiliary variable (collision.py:104-107)."""
        super().set_aux_var_at(index, variable)
        self.sdf.update_data(self.sdf_origin, self.sdf_data, self.sdf_cell_size)


class DoubleIntegrator(CostFunction):
    """theseus/embodied/motionmodel/double_integrator.py:16-95: e = [pose1.local(pose2) - dt vel1 ; vel2 - vel1], dim 2 dof.
    Fused kernels for poses of Vector kind with dof 2 / 3 (THB_COST_DOUBLE_INTEGRATOR_VECTOR) and SE2 (_SE2); other poses take the
    generic route on the same torch restatement."""

    def __init__(self, pose1: LieGroup, vel1: Vector, pose2: LieGroup, vel2: Vector, dt: Union[float, torch.Tensor, Variable],
                 cost_weight: CostWeight, name: Optional[str] = None):
        super().__init__(cost_weight, name=name)
        dof = pose1.dof()
        if not (vel1.dof() == pose2.dof() == vel2.dof() == dof):
            raise ValueError("All variables for a DoubleIntegrator must have the same dimension.")
        self.dt = as_variable(dt)
        if self.dt.tensor.squeeze().ndim > 1:
            raise ValueError("dt data must be a 0-D or 1-D tensor with numel in {1, batch_size}.")
        self.dt.tensor = self.dt.tensor.view(-1, 1)
        self.pose1, self.vel1, self.pose2, self.vel2 = pose1, vel1, pose2, vel2
        self.register_optim_vars(["pose1", "vel1", "pose2", "vel2"])
        self.register_aux_vars(["dt"])

    def dim(self) -> int:
        return 2 * self.pose1.dof()

    def _torch_error(self, optim_tensors, aux_tensors):
        from . import lie_torch
        p1, v1, p2, v2 = optim_tensors
        dt = aux_tensors[0]
        local = lie_torch.local(self.pose1.KIND, p1, p2)
        return torch.cat([local - dt.view(-1, 1) * v1, v2 - v1], dim=-1)

    def schema(self):
        aux = [self.dt] + ([self.weight.dt] if getattr(self.weight, "WEIGHT_KIND", -1) == WEIGHT_GP else [])
        vels_ok = isinstance(self.vel1, Vector) and isinstance(self.vel2, Vector)
        same = type(self.pose1) is type(self.pose2)
        if vels_ok and same and isinstance(self.pose1, SE2):
            kind = COST_DOUBLE_INTEGRATOR_SE2
        elif vels_ok and same and isinstance(self.pose1, Vector) and self.pose1.dof() in (2, 3):
            kind = COST_DOUBLE_INTEGRATOR_VECTOR
        else:
            return None, aux                       # generic route
        if aux[1:] and self.weight.Qc_inv.tensor.shape[-1] != self.pose1.dof():
            return None, aux                       # (mismatched Qc_inv: the torch route raises the reference's shape error)
        return kind, aux

    def _copy_impl(self, new_name: Optional[str] = None) -> "DoubleIntegrator":
        return type(self)(self.pose1.copy(), self.vel1.copy(), self.pose2.copy(), self.vel2.copy(), self.dt.copy(), self.weight.copy(),
                          name=new_name)


class GPCostWeight(CostWeight):
    """theseus/embodied/motionmodel/double_integrator.py:98-175: the full-matrix weight of a constant-velocity Gaussian-process prior,
    U = chol(W^T)^T with W = [[12/dt^3, -6/dt^2], [-6/dt^2, 4/dt]] (x) Qc_inv; weighting is U e, U J_i.  Qc_inv [d, d] or [Bq, d, d],
    dt [Bw, 1].  On the DoubleIntegrator kinds the kernels form U in registers (THB_WEIGHT_GP); elsewhere the torch form below."""
    WEIGHT_KIND = WEIGHT_GP

    def __init__(self, Qc_inv: Union[Variable, torch.Tensor], dt: Union[float, Variable, torch.Tensor], name: Optional[str] = None):
        super().__init__(name=name)
        dt = as_variable(dt)
        if dt.tensor.squeeze().ndim > 1:
            raise ValueError("dt must be a 0-D or 1-D tensor.")
        self.dt = dt
        self.dt.tensor = self.dt.tensor.view(-1, 1)
        if not (self.dt.tensor > 0).all():
            raise ValueError("dt must be greater than 0.")
        Qc_inv = as_variable(Qc_inv)
        if Qc_inv.ndim not in [2, 3]:
            raise ValueError("Qc_inv must be a single matrix or a batch of matrices.")
        if not Qc_inv.shape[-2] == Qc_inv.shape[-1]:
            raise ValueError("Qc_inv must contain square matrices.")
        self.Qc_inv = Qc_inv
        self.Qc_inv.tensor = Qc_inv.tensor if Qc_inv.ndim == 3 else Qc_inv.tensor.unsqueeze(0)
        try:
            torch.linalg.cholesky(Qc_inv.tensor)
        except RuntimeError:
            raise ValueError("Qc_inv must be positive definite.")
        if self.dt.tensor.dtype != self.Qc_inv.tensor.dtype:
            self.dt.tensor = self.dt.tensor.to(self.Qc_inv.tensor.dtype)
        self.register_aux_vars(["Qc_inv", "dt"])

    @property
    def aux_vars(self) -> List[Variable]:
        return [self.Qc_inv, self.dt]

    def weight_tensor(self) -> Variable:
        return self.Qc_inv

    def is_zero(self) -> torch.Tensor:
        return torch.zeros(self.Qc_inv.shape[0]).bool()

    def _compute_cost_weight(self) -> torch.Tensor:
        Q = self.Qc_inv.tensor
        dof = Q.shape[-1]
        dt = self.dt.tensor.view(-1, 1, 1)
        q11, q12, q22 = 12.0 * dt.pow(-3.0) * Q, -6.0 * dt.pow(-2.0) * Q, 4.0 * dt.reciprocal() * Q
        W = torch.cat([torch.cat([q11, q12], dim=-1), torch.cat([q12, q22], dim=-1)], dim=-2)
        assert W.shape[-1] == 2 * dof
        return torch.linalg.cholesky(W.transpose(-2, -1)).transpose(-2, -1)

    def weight_error(self, error: torch.Tensor) -> torch.Tensor:
        return torch.matmul(self._compute_cost_weight(), error.unsqueeze(2)).squeeze(2)

    def weight_jacobians_and_error(self, jacobians, error):
        U = self._compute_cost_weight()
        return [torch.matmul(U, J) for J in jacobians], torch.matmul(U, error.unsqueeze(2)).squeeze(2)

    def copy(self, new_name: Optional[str] = None, keep_variable_names: bool = False) -> "GPCostWeight":
        return GPCostWeight(self.Qc_inv.copy(new_name=self.Qc_inv.name if keep_variable_names else None),
                            self.dt.copy(new_name=self.dt.name if keep_variable_names else None), name=new_name)


class GPMotionModel(DoubleIntegrator):
    """double_integrator.py:178-207: a DoubleIntegrator whose weight must be a GPCostWeight."""

    def __init__(self, pose1: LieGroup, vel1: Vector, pose2: LieGroup, vel2: Vector, dt: Union[float, Variable, torch.Tensor],
                 cost_weight: GPCostWeight, name: Optional[str] = None):
        if not isinstance(cost_weight, GPCostWeight):
            raise ValueError("GPMotionModel only accepts cost weights of type GPCostWeight. "
                             "For other weight types, consider using DoubleIntegrator instead.")
        dt = as_variable(dt)
        if dt.tensor.squeeze().ndim > 1:
            raise ValueError("dt must be a 0-D or 1-D tensor.")
        super().__init__(pose1, vel1, pose2, vel2, dt, cost_weight, name=name)


class MovingFrameBetween(CostFunction):
    """theseus/embodied/measurements/moving_frame_between.py:14-77:
        e = log(Z^-1 ((F1^-1 P1)^-1 (F2^-1 P2)))        optim vars: frame1, frame2, pose1, pose2 (SE2 or SE3); aux: measurement.
    No fused kernel (the engine's schemas hold at most two variables): torch path.  NOTE the reference's Jacobians are those of the
    group-valued D = (F1^-1 P1)^-1 (F2^-1 P2) in ITS tangent space (moving_frame_between.py:46-65 chains the `between` Jacobians and
    stops there) -- the d log factor of the final `measurement.local(D)` is not applied.  For drop-in parity the same quantity is
    computed here: Euclidean torch.func Jacobian of D, input side projected like every AutoDiff Jacobian, output side converted from a
    velocity dD to tangent coordinates vee(D^-1 dD)  (tests/test_torch_restatements.py compares with the reference's values)."""

    def __init__(self, frame1: LieGroup, frame2: LieGroup, pose1: LieGroup, pose2: LieGroup, measurement: LieGroup,
                 cost_weight: CostWeight, name: Optional[str] = None):
        if len(set(x.__class__.__name__ for x in (frame1, frame2, pose1, pose2, measurement))) > 1:
            raise ValueError("Inconsistent types between input variables.")
        super().__init__(cost_weight, name=name)
        self.frame1, self.frame2, self.pose1, self.pose2 = frame1, frame2, pose1, pose2
        self.register_optim_vars(["frame1", "frame2", "pose1", "pose2"])
        self.measurement = measurement
        self.register_aux_vars(["measurement"])

    def dim(self) -> int:
        return self.frame1.dof()

    def _torch_error(self, optim_tensors, aux_tensors):
        from . import lie_torch
        k = self.frame1.KIND
        f1, f2, p1, p2 = optim_tensors
        d = lie_torch.between(k, lie_torch.between(k, f1, p1), lie_torch.between(k, f2, p2))
        return lie_torch.local(k, aux_tensors[0], d)

    def _torch_frame_diff(self, optim_tensors):
        from . import lie_torch
        k = self.frame1.KIND
        f1, f2, p1, p2 = optim_tensors
        return lie_torch.between(k, lie_torch.between(k, f1, p1), lie_torch.between(k, f2, p2))

    def _generic_unweighted(self, optim_tensors, differentiable: bool = False):
        import torch
        from torch.func import jacrev, vmap
        from . import lie_torch
        k = self.frame1.KIND
        aux = self.measurement.tensor
        B = max([t.shape[0] for t in optim_tensors] + [aux.shape[0]])
        ex = lambda t: t if t.shape[0] == B else t.expand((B,) + tuple(t.shape[1:]))
        opt_t = tuple(ex(t) for t in optim_tensors)

        def one(o):
            return self._torch_frame_diff(tuple(x.unsqueeze(0) for x in o))[0]

        with torch.enable_grad():
            D = self._torch_frame_diff(opt_t)
            dD = vmap(jacrev(one))(opt_t)                      # per variable: [B, *group_shape(out), *group_shape(in)]
            err = lie_torch.local(k, ex(aux), D)
        gs = D.ndim - 1                                         # 1 for SE2 storage [4], 2 for SE3 storage [3,4]
        jacs = []
        for v, t, J in zip(self.optim_vars, opt_t, dD):
            Jin = type(v).project_tensor(t, J.reshape(B, -1, *t.shape[1:]))          # input side -> tangent: [B, prod(out), dof]
            Jin = Jin.reshape(B, *D.shape[1:], Jin.shape[-1])                         # [B, *out, dof]
            Jin = Jin.movedim(-1, 1)                                                  # [B, dof, *out] : one velocity dD per column
            jacs.append(lie_torch.velocity_to_tangent(k, D, Jin).transpose(1, 2))     # [B, dof_out, dof_in]
        if differentiable:
            return jacs, err
        return [j.detach() for j in jacs], err.detach()

    def schema(self):
        return None, []


class QuasiStaticPushingPlanar(CostFunction):
    """theseus/embodied/motionmodel/quasi_static_pushing_planar.py:19-297 (quasi-static pushing model of the tactile example, Zhou et
    al. 2017): object poses obj1, obj2 and end-effector poses eff1, eff2 (SE2) at consecutive times, aux c_square;
        e = D V - Vp,  V = [R2^T (t_o2 - t_o1), theta(o1^-1 o2)],  Vp = [R2^T (t_e2 - t_e1), 0],
        D = [[1, 0, -py], [0, 1, px], [-py, px, -c^2]],  (px, py) = R2^T (t_e2 - t_o2).
    Torch path (torch.func Jacobians + tangent-space projection = the reference's chained analytic Jacobians)."""

    def __init__(self, obj1, obj2, eff1, eff2, c_square, cost_weight: CostWeight, name: Optional[str] = None):
        from .geometry import Variable, as_variable
        super().__init__(cost_weight, name=name)
        self.obj1, self.obj2, self.eff1, self.eff2 = obj1, obj2, eff1, eff2
        self.register_optim_vars(["obj1", "obj2", "eff1", "eff2"])
        c_square = c_square if isinstance(c_square, Variable) else as_variable(c_square)
        if c_square.tensor.dtype != obj1.dtype:
            c_square.tensor = c_square.tensor.to(obj1.dtype)
        if c_square.tensor.squeeze().ndim > 1:
            raise ValueError("dt must be a 0-D or 1-D tensor.")
        c_square.tensor = c_square.tensor.view(-1, 1)
        self.c_square = c_square
        self.register_aux_vars(["c_square"])

    def dim(self) -> int:
        return 3

    def _torch_error(self, optim_tensors, aux_tensors):
        import torch
        o1, o2, e1, e2 = optim_tensors
        c2 = aux_tensors[0].view(-1)
        cos2, sin2 = o2[..., 2], o2[..., 3]

        def unrot(v):  # R2^T v
            return torch.stack((cos2 * v[..., 0] + sin2 * v[..., 1], -sin2 * v[..., 0] + cos2 * v[..., 1]), dim=-1)

        p = unrot(e2[..., :2] - o2[..., :2])
        v = unrot(o2[..., :2] - o1[..., :2])
        # theta of o1^-1 o2 (se2.py:318-339): cos = c1 c2 + s1 s2, sin = c1 s2 - s1 c2
        omega = torch.atan2(o1[..., 2] * sin2 - o1[..., 3] * cos2, o1[..., 2] * cos2 + o1[..., 3] * sin2)
        vp = unrot(e2[..., :2] - e1[..., :2])
        px, py = p[..., 0], p[..., 1]
        ex = v[..., 0] - py * omega - vp[..., 0]
        ey = v[..., 1] + px * omega - vp[..., 1]
        et = -py * v[..., 0] + px * v[..., 1] - c2 * omega
        return torch.stack((ex, ey, et), dim=-1)

    def schema(self):
        return None, []


class EffectorObjectContactPlanar(CostFunction):
    """theseus/embodied/collision/eff_obj_contact.py:21-126 (+ SignedDistanceField2D.signed_distance, collision/signed_distance_field.py:
    163-241): the end effector (a disc of radius eff_radius at eff.xy) touches the object whose signed distance field is given in the
    object frame:  e = | sdf(R_obj^T (t_eff - t_obj)) - eff_radius |,  dim 1.  sdf = bilinear interpolation of sdf_data [Bs, rows, cols]
    (cell (r,c) at origin + (c, r) * cell_size), 0 outside the grid.  Torch path; autograd of the bilinear form is exactly the
    reference's analytic gradient, the sign flip for dist < radius is d|.|."""

    def __init__(self, obj, eff, sdf_origin, sdf_data, sdf_cell_size, eff_radius, cost_weight: CostWeight, name: Optional[str] = None,
                 use_huber_loss: bool = False):
        import torch
        from .geometry import Point2, Variable, as_variable
        if use_huber_loss:
            raise NotImplementedError("Jacobians for huber loss are not yet implemented.")  # same as the reference (eff_obj_contact.py:49-52)
        super().__init__(cost_weight, name=name)
        self.obj, self.eff = obj, eff
        self.sdf_origin = sdf_origin if isinstance(sdf_origin, Point2) else Point2(tensor=sdf_origin)
        self.sdf_data = as_variable(sdf_data)
        if self.sdf_data.tensor.ndim != 3:
            raise ValueError("Argument sdf_data to SignedDistanceField2D must be a batch of matrices.")
        if isinstance(sdf_cell_size, Variable):
            self.sdf_cell_size = sdf_cell_size
        else:
            self.sdf_cell_size = Variable((sdf_cell_size if torch.is_tensor(sdf_cell_size) else torch.tensor(float(sdf_cell_size))).view(-1, 1))
        self.eff_radius = as_variable(eff_radius)
        if self.eff_radius.tensor.squeeze().ndim > 1:
            raise ValueError("eff_radius must be a 0-D or 1-D tensor.")
        self.eff_radius.tensor = self.eff_radius.tensor.view(-1, 1)
        for v in (self.sdf_cell_size, self.eff_radius, self.sdf_data):
            if v.tensor.dtype != obj.dtype:
                v.tensor = v.tensor.to(obj.dtype)
        self.register_optim_vars(["obj", "eff"])
        self.register_aux_vars(["sdf_origin", "sdf_data", "sdf_cell_size", "eff_radius"])

    def dim(self) -> int:
        return 1

    def _torch_error(self, optim_tensors, aux_tensors):
        o, e = optim_tensors
        origin, data, cell, radius = aux_tensors
        cell, radius = cell.view(-1), radius.view(-1)
        dx, dy = e[..., 0] - o[..., 0], e[..., 1] - o[..., 1]
        px = o[..., 2] * dx + o[..., 3] * dy       # eff position in the object frame (SE2.transform_to)
        py = -o[..., 3] * dx + o[..., 2] * dy
        dist, _, _ = _bilinear_sdf(data, origin[..., 0], origin[..., 1], cell, px, py)
        return (dist - radius).abs().unsqueeze(-1)

    def schema(self):
        return None, []

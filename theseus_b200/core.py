"""Objective / CostFunction / CostWeight: the host-side mirror of the reference plugin API for the hot path.

  CostWeight, ScaleCostWeight, DiagonalCostWeight   theseus/core/cost_weight.py:20-139
  CostFunction                                      theseus/core/cost_function.py:64-149
  Between                                           theseus/embodied/measurements/between.py:14-60
  Difference (Local)                                theseus/embodied/misc/local_cost_fn.py:15-70
  Objective                                         theseus/core/objective.py:42-960

What differs from the reference is *how* the objective is evaluated: instead of iterating over cost
functions in Python and re-batching them with torch.cat at every call (theseus/core/vectorizer.py), the
objective is compiled once into per-schema tables of device pointers and offsets (engine.py) and every
evaluation is O(#schemas) CUDA kernels from libthb200.
"""
import warnings
from enum import Enum
from collections import OrderedDict
from typing import Dict, List, Optional, Sequence, Union

import torch

from .geometry import LieGroup, Manifold, Point2, Point3, SE2, SE3, SO2, SO3, Variable, Vector, as_variable

# enum thb_cost_kind / thb_weight_kind (include/thb200.h)
COST_BETWEEN_SE3, COST_LOCAL_SE3, COST_BETWEEN_SO3, COST_LOCAL_SO3, COST_LOCAL_VECTOR, COST_REPROJECTION = 0, 1, 2, 3, 4, 5
COST_BETWEEN_SE2, COST_LOCAL_SE2 = 6, 7
COST_COLLISION2D_POINT2, COST_COLLISION2D_SE2, COST_DOUBLE_INTEGRATOR_VECTOR, COST_DOUBLE_INTEGRATOR_SE2 = 8, 9, 10, 11
WEIGHT_SCALE, WEIGHT_DIAGONAL, WEIGHT_GP = 0, 1, 2
# kinds whose kernels have no fused robust loss: a RobustCostFunction around them takes the generic route
_NO_FUSED_ROBUST = (COST_LOCAL_VECTOR, COST_COLLISION2D_POINT2, COST_COLLISION2D_SE2, COST_DOUBLE_INTEGRATOR_VECTOR, COST_DOUBLE_INTEGRATOR_SE2)


def _shallow_clone_with_copied_vars(obj, attr_names, new_name):
    """A copy of a cost function / cost weight that shares nothing mutable with the original: same class and plain attributes, every
    registered variable replaced by its copy (one copy per distinct variable object)."""
    import copy as _copy
    new = _copy.copy(obj)
    new.name = new_name
    for lst in ("_optim_vars_attr_names", "_aux_vars_attr_names"):
        if hasattr(obj, lst):
            setattr(new, lst, list(getattr(obj, lst)))
    memo = {}
    for a in attr_names:
        v = getattr(obj, a)
        if id(v) not in memo:
            memo[id(v)] = v.copy()
        setattr(new, a, memo[id(v)])
    return new


class CostWeight:
    """theseus/core/cost_weight.py:20-55.  A user-defined subclass (WEIGHT_KIND -1) registers its auxiliary variables and implements
    weight_error / weight_jacobians_and_error; cost functions carrying one take the engine's generic route."""
    WEIGHT_KIND = -1

    def __init__(self, name: Optional[str] = None):
        self.name = name or f"{self.__class__.__name__}__{id(self)}"
        self._aux_vars_attr_names: List[str] = []

    def register_aux_var(self, name: str):
        self._aux_vars_attr_names.append(name)

    def register_aux_vars(self, names: Sequence[str]):
        self._aux_vars_attr_names.extend(names)

    @property
    def aux_vars(self) -> List[Variable]:
        if self.WEIGHT_KIND >= 0:
            return [self.weight_tensor()]
        return [getattr(self, n) for n in getattr(self, "_aux_vars_attr_names", [])]

    def weight_tensor(self) -> Variable:
        raise NotImplementedError

    def num_aux_vars(self) -> int:
        return len(self.aux_vars)

    def aux_var_at(self, index: int) -> Variable:
        return self.aux_vars[index]

    def get_default_name(self) -> str:
        return f"{self.__class__.__name__}__{id(self)}"

    def copy(self, new_name: Optional[str] = None, keep_variable_names: bool = False) -> "CostWeight":
        """theseus_function.py:90-108 for a user-defined weight: _copy_impl if the subclass has one, else a shallow clone whose registered
        variables are copies."""
        new_name = new_name or f"{self.name}_copy"
        if hasattr(self, "_copy_impl"):
            new = self._copy_impl(new_name=new_name)
        else:
            new = _shallow_clone_with_copied_vars(self, list(getattr(self, "_aux_vars_attr_names", [])), new_name)
        if keep_variable_names:
            for o, n in zip(self.aux_vars, new.aux_vars):
                n.name = o.name
        return new

    def weight_error(self, error: torch.Tensor) -> torch.Tensor:
        """cost_weight.py:33-35."""
        return self.weight_jacobians_and_error([], error)[1]

    def weight_jacobians_and_error(self, jacobians, error):
        """cost_weight.py:37-43 (Scale: :81-90, Diagonal: :125-136): (w J_i, w e)."""
        if self.WEIGHT_KIND < 0:
            raise NotImplementedError
        w = self.weight_tensor().tensor
        w = w.view(-1, 1) if self.WEIGHT_KIND == WEIGHT_SCALE else w
        return [J * (w.unsqueeze(2) if w.ndim == 2 else w) for J in jacobians], error * w

    def to(self, *args, **kwargs):
        for v in self.aux_vars:
            v.to(*args, **kwargs)


class ScaleCostWeight(CostWeight):
    """theseus/core/cost_weight.py:60-93: tensor [Bw, 1]."""
    WEIGHT_KIND = WEIGHT_SCALE

    def __init__(self, scale: Union[float, torch.Tensor, Variable], name: Optional[str] = None):
        super().__init__(name=name)
        self.scale = as_variable(scale)
        if not self.scale.tensor.squeeze().ndim in [0, 1]:
            raise ValueError("ScaleCostWeight only accepts 0- or 1-dim (batched) tensors.")
        self.scale.tensor = self.scale.tensor.view(-1, 1)

    def weight_tensor(self) -> Variable:
        return self.scale

    def is_zero(self) -> torch.Tensor:
        return self.scale.tensor.squeeze(1) == 0

    def copy(self, new_name: Optional[str] = None, keep_variable_names: bool = False):
        return ScaleCostWeight(self.scale.copy(new_name=self.scale.name if keep_variable_names else None), name=new_name)


class DiagonalCostWeight(CostWeight):
    """theseus/core/cost_weight.py:98-139: tensor [Bw, dim]."""
    WEIGHT_KIND = WEIGHT_DIAGONAL

    def __init__(self, diagonal: Union[Sequence[float], torch.Tensor, Variable], name: Optional[str] = None):
        super().__init__(name=name)
        self.diagonal = as_variable(diagonal)
        if not self.diagonal.tensor.squeeze().ndim < 3:
            raise ValueError("DiagonalCostWeight only accepts tensors with ndim < 3.")
        if self.diagonal.tensor.ndim == 0:
            self.diagonal.tensor = self.diagonal.tensor.view(1, 1)
        if self.diagonal.tensor.ndim == 1:
            warnings.warn("1-D diagonal input is ambiguous. Dimension will be interpreted as dof dimension and not batch dimension.")
            self.diagonal.tensor = self.diagonal.tensor.view(1, -1)

    def weight_tensor(self) -> Variable:
        return self.diagonal

    def is_zero(self) -> torch.Tensor:
        return (self.diagonal.tensor == 0).min(dim=1)[0].bool()

    def copy(self, new_name: Optional[str] = None, keep_variable_names: bool = False):
        return DiagonalCostWeight(self.diagonal.copy(new_name=self.diagonal.name if keep_variable_names else None), name=new_name)


class masked_variables:
    """core/variable.py:134-148: inside the context every variable holds only the batch items selected by the boolean `mask`."""

    def __init__(self, vars: Sequence[Variable], mask: torch.Tensor) -> None:
        assert mask.dtype == torch.bool and mask.ndim == 1
        self._vars, self._mask = list(vars), mask
        self._original = [v.tensor for v in self._vars]

    def __enter__(self) -> None:
        for v in self._vars:
            assert v.tensor.shape[0] == self._mask.shape[0]
            v._tensor = v.tensor[self._mask]          # around the setter: a temporary view, no pointer table is invalidated

    def __exit__(self, exc_type, exc_value, traceback) -> None:
        for v, t in zip(self._vars, self._original):
            v._tensor = t


def masked_jacobians(cost_fn: "CostFunction", mask: torch.Tensor):
    """core/cost_function.py:37-55: jacobians() / error of `cost_fn` evaluated only for the batch items selected by `mask`; outputs keep
    the full batch shape, unselected items are zero."""
    cf_vars = list(cost_fn.optim_vars) + list(cost_fn.aux_vars)
    batch_size = max(v.tensor.shape[0] for v in cf_vars)
    ref = cf_vars[0].tensor
    jacobians = [ref.new_zeros(batch_size, cost_fn.dim(), v.dof()) for v in cost_fn.optim_vars]
    err = ref.new_zeros(batch_size, cost_fn.dim())
    with masked_variables(cf_vars, mask):
        mj, err[mask] = cost_fn.jacobians()
        for m, j in zip(mj, jacobians):
            j[mask] = m
    return jacobians, err


class CostFunction:
    """theseus/core/cost_function.py:64-149.  Subclasses with a CUDA schema set COST_KIND via schema()."""
    _ids = 0

    def __init__(self, cost_weight: CostWeight, name: Optional[str] = None):
        CostFunction._ids += 1
        self.name = name or f"{self.__class__.__name__}__{CostFunction._ids}"
        self.weight = cost_weight
        self._optim_vars_attr_names: List[str] = []
        self._aux_vars_attr_names: List[str] = []

    def register_optim_vars(self, names: Sequence[str]):
        self._optim_vars_attr_names.extend(names)

    def register_aux_vars(self, names: Sequence[str]):
        self._aux_vars_attr_names.extend(names)

    def register_optim_var(self, name: str):
        self.register_optim_vars([name])

    def register_aux_var(self, name: str):
        self.register_aux_vars([name])

    @property
    def optim_vars(self):
        return [getattr(self, n) for n in self._optim_vars_attr_names]

    @property
    def aux_vars(self):
        return [getattr(self, n) for n in self._aux_vars_attr_names]

    def optim_var_at(self, index: int) -> Manifold:
        return getattr(self, self._optim_vars_attr_names[index])

    def num_optim_vars(self) -> int:
        return len(self._optim_vars_attr_names)

    def aux_var_at(self, index: int) -> Variable:
        return getattr(self, self._aux_vars_attr_names[index])

    def num_aux_vars(self) -> int:
        return len(self._aux_vars_attr_names)

    def set_optim_var_at(self, index: int, variable: Manifold):
        """theseus_function.py:67-71."""
        setattr(self, self._optim_vars_attr_names[index], variable)

    def set_aux_var_at(self, index: int, variable: Variable):
        setattr(self, self._aux_vars_attr_names[index], variable)

    def register_vars(self, variables, is_optim_vars: bool = False):
        """theseus_function.py:52-58: registers variables that are attributes named after themselves."""
        for v in variables:
            if hasattr(self, v.name):
                raise RuntimeError(f"Variable name {v.name} is not allowed since it conflicts with an attribute of this function.")
            setattr(self, v.name, v)
            (self.register_optim_var if is_optim_vars else self.register_aux_var)(v.name)

    def get_default_name(self) -> str:
        return f"{self.__class__.__name__}__{CostFunction._ids}"

    def copy(self, new_name: Optional[str] = None, keep_variable_names: bool = False) -> "CostFunction":
        """theseus_function.py:90-108: a new cost function over COPIES of the variables and of the weight (a subclass's own
        _copy_impl(new_name=...) is used if it has one)."""
        new_name = new_name or f"{self.name}_copy"
        if hasattr(self, "_copy_impl"):
            new = self._copy_impl(new_name=new_name)
        else:
            new = _shallow_clone_with_copied_vars(self, self._optim_vars_attr_names + self._aux_vars_attr_names, new_name)
            new.weight = self.weight.copy(new_name=None, keep_variable_names=keep_variable_names)
            inner = getattr(self, "cost_function", None)          # robust wrappers share their inner function's variables and weight
            if isinstance(inner, CostFunction):
                new.cost_function = inner.copy(keep_variable_names=keep_variable_names)
                new.weight = new.cost_function.weight
        if keep_variable_names:
            for o, n in zip(self.optim_vars + self.aux_vars, new.optim_vars + new.aux_vars):
                n.name = o.name
        return new

    def dim(self) -> int:
        raise NotImplementedError

    def schema(self):
        """(cost kind enum, aux variables) for the CUDA linearize/error kernels; kind None = the engine's generic route.  A user-defined
        subclass written against the reference's plugin contract (error() + jacobians() + dim(), cost_function.py:64-105) takes the
        generic route with its own analytic Jacobians."""
        if self._user_defined("error") and self._user_defined("jacobians"):
            return None, list(self.aux_vars)
        raise NotImplementedError(
            f"{self.__class__.__name__} has no CUDA schema in libthb200 and does not define error() and jacobians(); "
            "built in: Between/Difference on SE3, SO3, SE2, SO2, Vector, Reprojection, the tactile costs, AutoDiffCostFunction")

    # ---- the reference's public cost-function interface (core/cost_function.py:64-149) ----
    def _user_defined(self, what: str) -> bool:
        return getattr(type(self), what) is not getattr(CostFunction, what)

    class _at:
        """The optimisation variables' tensors temporarily replaced (the engine evaluates user code at candidate values); the swap goes
        around the `tensor` setter so that no pointer table is invalidated."""

        def __init__(self, cf, tensors):
            self._vars, self._new = cf.optim_vars, list(tensors)

        def __enter__(self):
            self._old = [v._tensor for v in self._vars]
            for v, t in zip(self._vars, self._new):
                v._tensor = t

        def __exit__(self, *exc):
            for v, t in zip(self._vars, self._old):
                v._tensor = t
            return False

    def error(self) -> torch.Tensor:
        """Unweighted error [B, dim] at the variables' current tensors (cost_function.py:85-87).  Built-in cost functions: their torch
        restatement; user-defined subclasses override this."""
        return self._torch_error(tuple(v.tensor for v in self.optim_vars), tuple(v.tensor for v in self._torch_aux()))

    def jacobians(self):
        """([J_i [B, dim, dof_i]], error) unweighted (cost_function.py:99-105).  Built-in cost functions: torch.func Jacobians of the
        torch restatement projected to the tangent space (equal to the fused kernels' analytic blocks, tests/test_torch_restatements.py);
        user-defined subclasses override this."""
        return self._generic_unweighted([v.tensor for v in self.optim_vars], differentiable=torch.is_grad_enabled())

    def weighted_error(self) -> torch.Tensor:
        """cost_function.py:107-110."""
        return self.generic_error([v.tensor for v in self.optim_vars])

    def weighted_jacobians_error(self):
        """cost_function.py:112-122: (weighted Jacobians, weighted error)."""
        return self.generic_jacobians_error([v.tensor for v in self.optim_vars], differentiable=torch.is_grad_enabled())

    def to(self, *args, **kwargs):
        for v in self.optim_vars + self.aux_vars:
            v.to(*args, **kwargs)
        self.weight.to(*args, **kwargs)

    # ---- torch path: AutoDiffCostFunction always, the fused-kernel cost functions only on the autograd tape of the backward modes ----
    def _torch_error(self, optim_tensors: Sequence[torch.Tensor], aux_tensors: Sequence[torch.Tensor]) -> torch.Tensor:
        """Unweighted error [B, dim] from raw storage tensors with differentiable torch ops (lie_torch.py)."""
        raise NotImplementedError(f"{self.__class__.__name__} has no torch restatement: it cannot be put on the autograd tape")

    def _torch_aux(self) -> List[Variable]:
        return self.aux_vars

    def _weight(self, err: torch.Tensor, jacs):
        if self.weight.WEIGHT_KIND not in (WEIGHT_SCALE, WEIGHT_DIAGONAL):   # user-defined or full-matrix (GPCostWeight) CostWeight
            if jacs is None:
                return None, self.weight.weight_error(err)
            wj, we = self.weight.weight_jacobians_and_error(list(jacs), err)
            return list(wj), we
        w = self.weight.weight_tensor().tensor
        w = w.view(-1, 1) if self.weight.WEIGHT_KIND == WEIGHT_SCALE else w
        err = err * w
        if jacs is not None:
            jacs = [J * (w.unsqueeze(2) if w.ndim == 2 else w) for J in jacs]
        return jacs, err

    def generic_jacobians_error(self, optim_tensors: Sequence[torch.Tensor], differentiable: bool = False):
        """(weighted Jacobians [B,dim,dof_i], weighted error [B,dim]): _generic_unweighted + the cost weight.  differentiable=True keeps
        the graph to the aux variables / weights / variable values (backward modes)."""
        jacs, err = self._generic_unweighted(optim_tensors, differentiable)
        return self._weight(err, jacs)

    def _generic_unweighted(self, optim_tensors: Sequence[torch.Tensor], differentiable: bool = False):
        """(Jacobians [B,dim,dof_i], error [B,dim]), unweighted.  User-defined subclass: its own jacobians() evaluated at `optim_tensors`;
        otherwise vmap(jacrev(_torch_error)) + tangent-space projection (cost_function.py:318-393, v.project(jac, is_sparse=True))."""
        if self._user_defined("jacobians"):
            with CostFunction._at(self, optim_tensors):
                jacs, err = self.jacobians()
            jacs = list(jacs)
            if len(jacs) != self.num_optim_vars() or err.ndim != 2 or err.shape[1] != self.dim():
                raise ValueError(f"{self.name}: jacobians() must return one [B, {self.dim()}, dof] block per optimisation variable and an "
                                 f"error of shape [B, {self.dim()}]")
            if differentiable:
                return jacs, err
            return [j.detach() for j in jacs], err.detach()
        from torch.func import jacrev, vmap
        ovars = self.optim_vars
        aux = tuple(v.tensor for v in self._torch_aux())
        B = max([t.shape[0] for t in optim_tensors] + [t.shape[0] for t in aux])
        ex = lambda t: t if t.shape[0] == B else t.expand((B,) + tuple(t.shape[1:]))
        opt_t, aux_t = tuple(ex(t) for t in optim_tensors), tuple(ex(t) for t in aux)

        def one(o, a):
            return self._torch_error(tuple(x.unsqueeze(0) for x in o), tuple(x.unsqueeze(0) for x in a))[0]

        with torch.enable_grad():
            jacs = vmap(jacrev(one, argnums=0))(opt_t, aux_t)
            err = self._torch_error(opt_t, aux_t)
        jacs = [type(v).project_tensor(t, j) for v, t, j in zip(ovars, opt_t, jacs)]  # Euclidean -> tangent space (identity for Vector)
        if differentiable:
            return jacs, err
        return [j.detach() for j in jacs], err.detach()

    def generic_error(self, optim_tensors: Sequence[torch.Tensor]) -> torch.Tensor:
        """Weighted error [B, dim] at the given optimisation-variable tensors."""
        if self._user_defined("error"):
            with CostFunction._at(self, optim_tensors):
                err = self.error()
            return self._weight(err, None)[1]
        return self._weight(self._torch_error(tuple(optim_tensors), tuple(v.tensor for v in self._torch_aux())), None)[1]


class Between(CostFunction):
    """theseus/embodied/measurements/between.py:14-60: e = log(Z^-1 (X0^-1 X1))."""

    def __init__(self, v0: LieGroup, v1: LieGroup, measurement: LieGroup, cost_weight: CostWeight, name: Optional[str] = None):
        super().__init__(cost_weight, name=name)
        self.v0, self.v1 = v0, v1
        self.register_optim_vars(["v0", "v1"])
        self.measurement = measurement
        self.register_aux_vars(["measurement"])
        if not isinstance(v0, v1.__class__) or not isinstance(v0, measurement.__class__):
            raise ValueError("Inconsistent types between variables and measurement.")

    def dim(self) -> int:
        return self.v0.dof()

    def _torch_error(self, optim_tensors, aux_tensors):
        from . import lie_torch
        k = self.v0.KIND
        return lie_torch.local(k, aux_tensors[0], lie_torch.between(k, optim_tensors[0], optim_tensors[1]))  # between.py:34-37

    def schema(self):
        if isinstance(self.v0, SE3):
            return COST_BETWEEN_SE3, self.measurement
        if isinstance(self.v0, SO3):
            return COST_BETWEEN_SO3, self.measurement
        if isinstance(self.v0, SE2):
            return COST_BETWEEN_SE2, self.measurement
        if isinstance(self.v0, (SO2, Vector)):
            return None, [self.measurement]   # generic route: torch.func Jacobians of _torch_error (engine.py)
        return super().schema()


class Difference(CostFunction):
    """theseus/embodied/misc/local_cost_fn.py:15-70 (Local; `Difference` is the public alias): e = log(T^-1 X)."""

    def __init__(self, var: Manifold, target: Manifold, cost_weight: CostWeight, name: Optional[str] = None):
        super().__init__(cost_weight, name=name)
        if not isinstance(var, target.__class__):
            raise ValueError("Variable for the Local inconsistent with the given target.")
        if not var.dof() == target.dof():
            raise ValueError("Variable and target in the Local must have identical dof.")
        self.var, self.target = var, target
        self.register_optim_vars(["var"])
        self.register_aux_vars(["target"])

    def dim(self) -> int:
        return self.var.dof()

    def _torch_error(self, optim_tensors, aux_tensors):
        from . import lie_torch
        return lie_torch.local(self.var.KIND, aux_tensors[0], optim_tensors[0])  # local_cost_fn.py:40-43

    def schema(self):
        if isinstance(self.var, SE3):
            return COST_LOCAL_SE3, self.target
        if isinstance(self.var, SO3):
            return COST_LOCAL_SO3, self.target
        if isinstance(self.var, SE2):
            return COST_LOCAL_SE2, self.target
        if isinstance(self.var, SO2):
            return None, [self.target]        # generic route
        if isinstance(self.var, Vector):
            return COST_LOCAL_VECTOR, self.target
        return super().schema()


Local = Difference


class Reprojection(CostFunction):
    """theseus/embodied/measurements/reprojection.py:13-105: radial-distortion pinhole reprojection residual (dim 2).
    optim vars: camera_pose (SE3), world_point (Point3); aux: focal_length, image_feature_point, calib_k1, calib_k2."""

    def __init__(self, camera_pose: SE3, world_point: Point3, image_feature_point: Point2, focal_length: Vector,
                 calib_k1: Vector = None, calib_k2: Vector = None, weight: Optional[CostWeight] = None, name: Optional[str] = None):
        if weight is None:
            weight = ScaleCostWeight(torch.tensor(1.0).to(dtype=camera_pose.dtype))
        super().__init__(cost_weight=weight, name=name)
        self.camera_pose, self.world_point = camera_pose, world_point
        self.focal_length, self.image_feature_point = focal_length, image_feature_point
        batch_size = camera_pose.shape[0]
        self.calib_k1 = calib_k1 if calib_k1 is not None else Vector(
            tensor=torch.zeros((batch_size, 1), dtype=camera_pose.dtype, device=camera_pose.device), name=f"calib_k1__{self.name}")
        self.calib_k2 = calib_k2 if calib_k2 is not None else Vector(
            tensor=torch.zeros((batch_size, 1), dtype=camera_pose.dtype, device=camera_pose.device), name=f"calib_k2__{self.name}")
        self.register_optim_vars(["camera_pose", "world_point"])
        self.register_aux_vars(["focal_length", "image_feature_point", "calib_k1", "calib_k2"])

    def dim(self) -> int:
        return 2

    def _torch_error(self, optim_tensors, aux_tensors):
        X, p = optim_tensors
        f, z, k1, k2 = aux_tensors
        q = (X[..., :3] @ p[..., None])[..., 0] + X[..., 3]              # reprojection.py:54-66
        proj = -q[..., :2] / q[..., 2:3]
        n = (proj * proj).sum(dim=-1, keepdim=True)
        return proj * (f * (1.0 + n * (k1 + n * k2))) - z

    def schema(self):
        return COST_REPROJECTION, [self.focal_length, self.image_feature_point, self.calib_k1, self.calib_k2]


_LOSS_EPS = 1e-20


class RobustLoss:
    """theseus/core/robust_loss.py:13-30.  x = squared norm of the weighted error, radius = exp(log_radius).  Welsch and Huber are fused
    into the linearize / error kernels (ROBUST_KIND = the kernels' enum, thb_costs.cu); every loss also has its torch form below, used
    by the generic (torch.func) route and by the taped linearization of the backward modes."""
    ROBUST_KIND = 0
    FUSED = False   # True: thb_costs.cu has the formulas

    @classmethod
    def evaluate(cls, x: torch.Tensor, log_radius: torch.Tensor, *extra: torch.Tensor) -> torch.Tensor:
        return cls._evaluate_impl(x, log_radius.exp(), *extra)

    @classmethod
    def linearize(cls, x: torch.Tensor, log_radius: torch.Tensor, *extra: torch.Tensor) -> torch.Tensor:
        return cls._linearize_impl(x, log_radius.exp(), *extra)


class WelschLoss(RobustLoss):
    """robust_loss.py:33-41: rho(x) = r - r exp(-x/r)."""
    ROBUST_KIND = 1
    FUSED = True

    @staticmethod
    def _evaluate_impl(x, radius):
        return radius - radius * torch.exp(-x / (radius + _LOSS_EPS))

    @staticmethod
    def _linearize_impl(x, radius):
        return torch.exp(-x / (radius + _LOSS_EPS))


class HuberLoss(RobustLoss):
    """robust_loss.py:43-52: rho(x) = x below the radius, 2 sqrt(r x) - r above."""
    ROBUST_KIND = 2
    FUSED = True

    @staticmethod
    def _evaluate_impl(x, radius):
        return torch.where(x > radius, 2 * torch.sqrt(radius * torch.max(x, radius) + _LOSS_EPS) - radius, x)

    @staticmethod
    def _linearize_impl(x, radius):
        return torch.sqrt(radius / torch.max(x, radius) + _LOSS_EPS)


class HingeLoss(RobustLoss):
    """robust_loss.py:55-62: rho(x) = sqrt(x) - sqrt(r) above the radius, (numerically) zero below."""
    ROBUST_KIND = 3

    @staticmethod
    def _evaluate_impl(x, radius):
        return torch.where(x > radius, torch.sqrt(x) - torch.sqrt(radius), torch.full_like(x, _LOSS_EPS))

    @staticmethod
    def _linearize_impl(x, radius):
        return torch.where(x > radius, 1.0 / (2 * torch.sqrt(x) + _LOSS_EPS), torch.zeros_like(x))


class GNCRobustLoss(RobustLoss):
    """robust_loss.py:65-91: losses with a graduated-non-convexity control value mu (third argument)."""


class GemanMcClureLoss(GNCRobustLoss):
    """robust_loss.py:96-118: rho(x) = mu r x / (mu r + x); mu = 1: Geman-McClure, mu -> inf: quadratic."""
    ROBUST_KIND = 4

    @staticmethod
    def _evaluate_impl(x, radius, mu):
        return mu * radius * x / (mu * radius + x + _LOSS_EPS)

    @staticmethod
    def _linearize_impl(x, radius, mu):
        return (mu * radius) ** 2 / ((mu * radius + x) ** 2 + _LOSS_EPS)


class RobustCostFunction(CostFunction):
    """theseus/core/robust_cost_function.py:16-160: wraps a cost function; linearisation rescales J and e by
    sqrt(rho'(||w e||^2) + 1e-20), the error metric sees rho(||w e||^2).

    Welsch / Huber around a cost function with a CUDA schema are fused into that schema's kernels.  Everything else -- Hinge,
    Geman-McClure (GNCRobustCostFunction), flatten_dims=True, wrapped AutoDiff / Vector-difference costs -- takes the generic route of
    the engine (torch.func Jacobians of the wrapped cost, rescaled here in torch, scattered into the batched CSR)."""
    _EPS = 1e-20

    def __init__(self, cost_function: CostFunction, loss_cls, log_loss_radius: Variable, flatten_dims: bool = False,
                 name: Optional[str] = None):
        if not (isinstance(loss_cls, type) and issubclass(loss_cls, RobustLoss) and loss_cls.ROBUST_KIND > 0):
            raise NotImplementedError("loss_cls must be one of WelschLoss, HuberLoss, HingeLoss, GemanMcClureLoss")
        self.cost_function = cost_function
        super().__init__(cost_function.weight, name=name)
        for attr in cost_function._optim_vars_attr_names:
            setattr(self, attr, getattr(cost_function, attr))
            self._optim_vars_attr_names.append(attr)
        for attr in cost_function._aux_vars_attr_names:
            setattr(self, attr, getattr(cost_function, attr))
            self._aux_vars_attr_names.append(attr)
        self.log_loss_radius = log_loss_radius
        self._aux_vars_attr_names.append("log_loss_radius")
        self.loss = loss_cls()
        self.flatten_dims = bool(flatten_dims)
        self.robust_kind = loss_cls.ROBUST_KIND

    def dim(self) -> int:
        return self.cost_function.dim()

    def _loss_args(self):
        return (self.log_loss_radius.tensor,)

    def generic_jacobians_error(self, optim_tensors, differentiable: bool = False):
        """robust_cost_function.py:115-135: J, e of the wrapped cost rescaled by sqrt(rho'(||w e||^2) + eps)
        (flatten_dims: per error dimension, rho'((w e)_i^2))."""
        jacs, err = self.cost_function.generic_jacobians_error(optim_tensors, differentiable=differentiable)
        if self.flatten_dims:
            x = err ** 2
            sc = torch.sqrt(self.loss.linearize(x.reshape(-1, 1), *self._loss_args()) + self._EPS).reshape(err.shape)
        else:
            x = (err ** 2).sum(dim=1, keepdim=True)
            sc = torch.sqrt(self.loss.linearize(x, *self._loss_args()) + self._EPS)
        if not differentiable:
            sc = sc.detach()
        return [sc.unsqueeze(2) * J for J in jacs], sc * err

    def generic_error(self, optim_tensors) -> torch.Tensor:
        """robust_cost_function.py:87-109: an error whose squared norm is rho(||w e||^2): every entry sqrt(rho/dim + eps)
        (flatten_dims: entry i = sqrt(rho((w e)_i^2) + eps))."""
        err = self.cost_function.generic_error(optim_tensors)
        if self.flatten_dims:
            val = self.loss.evaluate((err ** 2).reshape(-1, 1), *self._loss_args()).reshape(err.shape)
            return torch.sqrt(val + self._EPS)
        val = self.loss.evaluate((err ** 2).sum(dim=1, keepdim=True), *self._loss_args())
        return torch.ones_like(err) * torch.sqrt(val / self.dim() + self._EPS)

    def schema(self):
        kind, aux = self.cost_function.schema()
        aux = list(aux) if isinstance(aux, (list, tuple)) else [aux]
        if kind is None or kind in _NO_FUSED_ROBUST or not type(self.loss).FUSED or self.flatten_dims:
            return None, aux   # generic route (engine: torch.func Jacobians through generic_jacobians_error / generic_error)
        return kind, (aux if len(aux) > 1 else aux[0])


class GNCRobustCostFunction(RobustCostFunction):
    """robust_cost_function.py:181-240: robust cost whose loss takes the graduated-non-convexity control value `gnc_control_val`
    (annealed by the caller between optimisations)."""

    def __init__(self, cost_function: CostFunction, loss_cls, log_loss_radius: Variable, gnc_control_val: Variable,
                 flatten_dims: bool = False, name: Optional[str] = None):
        if not (isinstance(loss_cls, type) and issubclass(loss_cls, GNCRobustLoss)):
            raise RuntimeError(f"{loss_cls} must be GNCRobustLoss type to initialize GNCRobustCostFunction.")
        super().__init__(cost_function, loss_cls, log_loss_radius, flatten_dims=flatten_dims, name=name)
        self.gnc_control_val = gnc_control_val
        self._aux_vars_attr_names.append("gnc_control_val")

    def _loss_args(self):
        return (self.log_loss_radius.tensor, self.gnc_control_val.tensor)


class AutogradMode(Enum):
    """theseus/core/cost_function.py:152-170.  Every mode is served by the vmap(jacrev) path here (the three modes of the reference give
    the same Jacobians; they differ in how torch computes them)."""
    DENSE = 0
    LOOP_BATCH = 1
    VMAP = 2

    @staticmethod
    def resolve(key) -> "AutogradMode":
        if isinstance(key, AutogradMode):
            return key
        if not isinstance(key, str):
            raise ValueError("Autograd mode must be of type th.AutogradMode or string.")
        try:
            return AutogradMode[key.upper()]
        except KeyError:
            raise ValueError(f"Unrecognized autograd mode {key}. Valid choices are dense, loop_batch, vmap.")


class AutoDiffCostFunction(CostFunction):
    """theseus/core/cost_function.py:203-420: user-defined error function, Jacobians by vmap(jacrev(err_fn)) -- kept as the
    reference's torch.func path (SURVEY.md a29); the results are scattered straight into the batched-CSR Jacobian.
    `err_fn(optim_vars, aux_vars) -> [B, dim]` receives tuples of Variable-like objects exposing `.tensor`.
    Lie-group optimisation variables: the user's err_fn works on the raw storage tensors (`.tensor`, e.g. SE3 [B,3,4]) with torch
    ops, the Euclidean Jacobians are projected onto the tangent space like `v.project(jac, is_sparse=True)` (cost_function.py:389-391)."""

    def __init__(self, optim_vars: Sequence[Manifold], err_fn, dim: int, cost_weight: Optional[CostWeight] = None,
                 aux_vars: Optional[Sequence[Variable]] = None, name: Optional[str] = None,
                 autograd_mode: Union[str, "AutogradMode"] = "vmap", **autograd_kwargs):
        if cost_weight is None:
            cost_weight = ScaleCostWeight(1.0)
        super().__init__(cost_weight, name=name)
        aux_vars = list(aux_vars or [])
        if len(optim_vars) < 1:
            raise ValueError("AutodiffCostFunction must receive at least one optimization variable.")
        for v in optim_vars:
            if not isinstance(v, Manifold):
                raise ValueError("AutoDiffCostFunction optimisation variables must be Manifold instances")
        for i, v in enumerate(optim_vars):          # the registered attributes are the only references (copy() / set_*_var_at replace them)
            setattr(self, f"_optim_var_{i}", v)
            self._optim_vars_attr_names.append(f"_optim_var_{i}")
        for i, v in enumerate(aux_vars):
            setattr(self, f"_aux_var_{i}", v)
            self._aux_vars_attr_names.append(f"_aux_var_{i}")
        self._err_fn = err_fn
        self._dim = dim
        self._autograd_mode = AutogradMode.resolve(autograd_mode)

    def dim(self) -> int:
        return self._dim

    class _T:  # minimal Variable-like holder handed to the user's err_fn
        def __init__(self, tensor):
            self.tensor = tensor

        def __getitem__(self, item):
            return self.tensor[item]

    def _torch_error(self, optim_tensors, aux_tensors):
        # err_fn sees variables of the registered classes (SE3, Vector, ...) holding the traced tensors, like the reference's
        # (cost_function.py:283-316): group methods called on them take the differentiable torch route (geometry_api.py)
        from .geometry_api import typed_view
        return self._err_fn(optim_vars=tuple(typed_view(v, t) for v, t in zip(self.optim_vars, optim_tensors)),
                            aux_vars=tuple(typed_view(v, t) for v, t in zip(self.aux_vars, aux_tensors)))

    def _torch_aux(self):
        return self.aux_vars

    def schema(self):
        return None, []


class Objective:
    """theseus/core/objective.py:42-960 (the subset the NLS loop uses)."""

    def __init__(self, dtype: Optional[torch.dtype] = None):
        self.optim_vars: "OrderedDict[str, Manifold]" = OrderedDict()
        self.aux_vars: "OrderedDict[str, Variable]" = OrderedDict()
        self.cost_functions: "OrderedDict[str, CostFunction]" = OrderedDict()
        self.dtype = dtype or torch.get_default_dtype()
        self.device = torch.device("cpu")
        self._batch_size: Optional[int] = None
        self._structure_version = 0
        self._engine = None

    # ---- construction ----
    def add(self, cost_function: CostFunction):
        """objective.py:210-300: registers the cost function and its variables (first-appearance order)."""
        if cost_function.name in self.cost_functions:
            raise ValueError(f"Two different cost function objects with the same name ({cost_function.name}) are not allowed in the same objective.")
        for v in cost_function.optim_vars + cost_function.aux_vars + cost_function.weight.aux_vars:
            if v.dtype != self.dtype:
                raise ValueError(f"Tried to add cost function with dtype {v.dtype} variable {v.name} to objective of dtype {self.dtype}.")
        self.cost_functions[cost_function.name] = cost_function
        for v in cost_function.optim_vars:
            if v.name in self.optim_vars and self.optim_vars[v.name] is not v:
                raise ValueError(f"Two different variable objects with the same name ({v.name}) are not allowed in the same objective.")
            self.optim_vars.setdefault(v.name, v)
        for v in cost_function.aux_vars + cost_function.weight.aux_vars:
            if v.name in self.aux_vars and self.aux_vars[v.name] is not v:
                raise ValueError(f"Two different variable objects with the same name ({v.name}) are not allowed in the same objective.")
            self.aux_vars.setdefault(v.name, v)
        self._structure_version += 1
        self._engine = None
        self._batch_size = None

    vectorized = False    # set by optimizer.Vectorize; the engine evaluates per schema group regardless (objective.py:916-960 by name)

    def disable_vectorization(self):
        self.vectorized = False

    def update_vectorization_if_needed(self):
        pass

    def copy(self) -> "Objective":
        """objective.py:643-700: copies of all cost functions, weights and variables with the same names and connectivity (a variable or
        weight shared by several cost functions is ONE object in the copy, too)."""
        new = Objective(dtype=self.dtype)
        weights = {}
        for cf in self.cost_functions.values():
            if id(cf.weight) not in weights:
                weights[id(cf.weight)] = cf.weight.copy(new_name=cf.weight.name, keep_variable_names=True)
        for cf in self.cost_functions.values():
            ncf = cf.copy(new_name=cf.name, keep_variable_names=True)
            ncf.weight = weights[id(cf.weight)]
            if isinstance(getattr(ncf, "cost_function", None), CostFunction):
                ncf.cost_function.weight = ncf.weight
            for target in [ncf] + ([ncf.cost_function] if isinstance(getattr(ncf, "cost_function", None), CostFunction) else []):
                for i, v in enumerate(target.optim_vars):
                    if v.name in new.optim_vars:
                        target.set_optim_var_at(i, new.optim_vars[v.name])
                for i, v in enumerate(target.aux_vars):
                    if v.name in new.aux_vars:
                        target.set_aux_var_at(i, new.aux_vars[v.name])
            new.add(ncf)
        new.device = self.device
        return new

    # ---- queries / removal (objective.py:302-470) ----
    def get_cost_function(self, name: str) -> CostFunction:
        return self.cost_functions.get(name, None)

    def has_cost_function(self, name: str) -> bool:
        return name in self.cost_functions

    def has_optim_var(self, name: str) -> bool:
        return name in self.optim_vars

    def has_aux_var(self, name: str) -> bool:
        return name in self.aux_vars

    def _cost_variables(self, cf: CostFunction):
        return cf.optim_vars, cf.aux_vars + cf.weight.aux_vars

    def get_functions_connected_to_optim_var(self, variable: Union[str, Manifold]) -> List[CostFunction]:
        name = variable if isinstance(variable, str) else variable.name
        if name not in self.optim_vars:
            raise ValueError(f"Optimization variable named {name} is not in the objective.")
        return [cf for cf in self.cost_functions.values() if any(v.name == name for v in cf.optim_vars)]

    def get_functions_connected_to_aux_var(self, aux_var: Union[str, Variable]) -> List[CostFunction]:
        name = aux_var if isinstance(aux_var, str) else aux_var.name
        if name not in self.aux_vars:
            raise ValueError(f"Aux variable named {name} is not in the objective.")
        return [cf for cf in self.cost_functions.values() if any(v.name == name for v in self._cost_variables(cf)[1])]

    def erase(self, name: str):
        """objective.py:395-416: removes the cost function and every variable no other cost function uses; the compiled engine
        (pointer tables, CSR structure, symbolic plans) is rebuilt at the next use."""
        if name not in self.cost_functions:
            warnings.warn("This cost function is not in the objective, nothing to be done.")
            return
        del self.cost_functions[name]
        used_o = set(v.name for cf in self.cost_functions.values() for v in cf.optim_vars)
        used_a = set(v.name for cf in self.cost_functions.values() for v in self._cost_variables(cf)[1])
        for k in [k for k in self.optim_vars if k not in used_o]:
            del self.optim_vars[k]
        for k in [k for k in self.aux_vars if k not in used_a]:
            del self.aux_vars[k]
        self._structure_version += 1
        self._engine = None
        self._batch_size = None

    def size(self) -> tuple:
        return len(self.cost_functions), len(self.optim_vars), len(self.aux_vars)

    def dim(self) -> int:
        return sum(cf.dim() for cf in self.cost_functions.values())

    def size_cost_functions(self) -> int:
        return len(self.cost_functions)

    def size_variables(self) -> int:
        return len(self.optim_vars)

    def size_aux_vars(self) -> int:
        return len(self.aux_vars)

    def get_optim_var(self, name: str) -> Manifold:
        return self.optim_vars[name]

    def get_aux_var(self, name: str) -> Variable:
        return self.aux_vars[name]

    def __iter__(self):
        return iter(self.cost_functions.values())

    @property
    def batch_size(self) -> int:
        if self._batch_size is None:
            self._resolve_batch_size()
        return self._batch_size

    def _resolve_batch_size(self):
        """objective.py:708-724."""
        sizes = set(v.tensor.shape[0] for v in self.optim_vars.values())
        sizes |= set(v.tensor.shape[0] for v in self.aux_vars.values())
        if len(sizes) == 1:
            self._batch_size = next(iter(sizes))
        elif len(sizes) == 2 and min(sizes) == 1:
            self._batch_size = max(sizes)
        else:
            raise ValueError("Provided tensors must be broadcastable.")

    def to(self, *args, **kwargs) -> "Objective":
        """objective.py:938-950."""
        for cf in self.cost_functions.values():
            cf.to(*args, **kwargs)
        device, dtype, *_ = torch._C._nn._parse_to(*args, **kwargs)
        if device is not None and device.type == "cuda" and device.index is None:
            device = torch.device("cuda", torch.cuda.current_device())  # tensors report cuda:<index>
        self.device = device or self.device
        self.dtype = dtype or self.dtype
        self._engine = None
        return self

    def update(self, input_tensors: Optional[Dict[str, torch.Tensor]] = None,
               batch_ignore_mask: Optional[torch.Tensor] = None, _update_vectorization: bool = True):
        """objective.py:729-811."""
        input_tensors = input_tensors or {}
        for var_name, tensor in input_tensors.items():
            if tensor.ndim < 2:
                raise ValueError(f"Input tensors must have a batch dimension and one ore more data dimensions, but tensor.ndim={tensor.ndim} for tensor with name {var_name}.")
            if tensor.device != self.device or tensor.dtype != self.dtype:
                raise ValueError(
                    f"Attempted to update variable {var_name} with a ({tensor.device},{tensor.dtype}) tensor, "
                    f"which is inconsistent with objective's expected ({self.device},{self.dtype}).")
            if var_name in self.optim_vars:
                self.optim_vars[var_name].update(tensor, batch_ignore_mask=batch_ignore_mask)
            elif var_name in self.aux_vars:
                self.aux_vars[var_name].update(tensor, batch_ignore_mask=batch_ignore_mask)
            else:
                warnings.warn(f"Attempted to update a tensor with name {var_name}, which is not associated to any variable in the objective.")
        self._resolve_batch_size()

    # ---- evaluation (CUDA) ----
    def engine(self, ordering=None):
        """The compiled form of this objective (engine.Engine).  `ordering`: variable names in column order (a Linearization passes its
        VariableOrdering); None keeps the order recorded by the last Linearization built on this objective (default: order of first
        appearance, variable_ordering.py:19-27).  A different order rebuilds the engine."""
        from .engine import Engine
        if ordering is not None:
            ordering = tuple(ordering)
            self._engine_ordering = None if list(ordering) == list(self.optim_vars.keys()) else ordering
        want = getattr(self, "_engine_ordering", None)
        if want is not None and set(want) != set(self.optim_vars.keys()):
            want = self._engine_ordering = None    # recorded for an earlier structure of this objective
        if (self._engine is None or self._engine.structure_version != self._structure_version
                or self._engine.custom_ordering != want):
            self._engine = Engine(self, want)
        return self._engine

    def error_metric(self, input_tensors: Optional[Dict[str, torch.Tensor]] = None, also_update: bool = False) -> torch.Tensor:
        """objective.py:615-641: 0.5 * sum((w e)^2) per batch item, shape [B]."""
        old = {}
        if input_tensors is not None:
            if not also_update:
                old = {n: self.optim_vars[n].tensor for n in self.optim_vars}
            self.update(input_tensors)
        err = self.engine().error_metric()
        if input_tensors is not None and not also_update:
            self.update(old)
        return err

    def error(self, input_tensors: Optional[Dict[str, torch.Tensor]] = None, also_update: bool = False) -> torch.Tensor:
        """objective.py:562-613: weighted error vector [B, m] (= -b of the linearization)."""
        old = {}
        if input_tensors is not None:
            if not also_update:
                old = {n: self.optim_vars[n].tensor for n in self.optim_vars}
            self.update(input_tensors)
        if any(isinstance(cf, RobustCostFunction) for cf in self.cost_functions.values()):
            # -b of the linearization is the sqrt(rho')-rescaled residual; the reference's error() concatenates weighted_error(), which for
            # a robust cost is sqrt(rho / dim + eps) per entry (robust_cost_function.py:87-109), so that error_metric == 0.5 * ||error()||^2
            err = torch.cat([cf.weighted_error() for cf in self.cost_functions.values()], dim=1)
        else:
            eng = self.engine()
            _, b = eng.linearize_sparse()   # (refreshes the engine's A_val / b buffers at the current variable values)
            err = -b
        if input_tensors is not None and not also_update:
            self.update(old)
        return err

    def retract_vars_sequence(self, delta: torch.Tensor, ordering, ignore_mask: Optional[torch.Tensor] = None,
                              force_update: bool = False):
        """objective.py:873-914: X_i <- X_i * exp(delta_i) for the variables in `ordering` (tmp containers)."""
        eng = self.engine()
        seq = list(ordering)
        names = [v.name for v in seq]
        if names != [v.name for v in eng.ordering]:
            # the engine's retraction kernel walks its own column order; a subset / another order of variables would be paired with the
            # wrong delta columns (the reference consumes delta sequentially over whatever sequence it is given, objective.py:857-871)
            raise NotImplementedError("retract_vars_sequence: `ordering` must list the objective's optimisation variables in the "
                                      f"linearization's column order ({len(eng.ordering)} variables), got {len(seq)}")
        eng.retract_into(delta, seq, 1.0, None if force_update else ignore_mask)

"""Engine: an Objective compiled into device-resident index tables + the kernel launches over them.

This replaces theseus/core/vectorizer.py (Vectorize): instead of torch.cat-ing the tensors of same-schema
cost functions at every evaluation, the objective structure is compiled ONCE into
  * per-schema cost groups (pointer tables to every cost function's variable / measurement / weight tensor),
  * the reference's batched-CSR layout of the Jacobian (structure.py),
  * Gram gather plans,
and every evaluation is O(#schemas) kernel launches from libthb200 on the current CUDA stream.

Optimisation variables are kept in two engine-owned pools (current / trial) so that device pointers stay
stable across LM iterations (no table rebuilds, CUDA-graph friendly); `Variable.tensor` of each
optimisation variable is a [B, ...] view into the pool.
"""
import ctypes as C
import os
from typing import List, Optional

import numpy as np
import torch

from . import _lib
from .geometry import Manifold, Variable
from .structure import build_gram_plan, build_structure


def _dev(arr: np.ndarray, device) -> torch.Tensor:
    return torch.from_numpy(np.ascontiguousarray(arr)).to(device)


def _batched_torch_route() -> bool:
    """Opt-in (THB_BATCHED_TORCH_ROUTE=1): evaluate the torch-route cost functions per group of equal signature (torch_route.py) instead of
    one by one.  CPU-verified against the per-cost loop (tests/test_torch_route.py); default off until it has run on a GPU."""
    return os.environ.get("THB_BATCHED_TORCH_ROUTE", "0") == "1"


# cost kinds with four optimisation variables (thb_cost_group.x2 / x3, bp of width 4) and the weight kinds each kernel takes
_FOUR_VAR_KINDS = (10, 11)             # THB_COST_DOUBLE_INTEGRATOR_VECTOR / _SE2
_COLLISION_KINDS = (8, 9)              # THB_COST_COLLISION2D_POINT2 / _SE2
_WEIGHT_SCALE, _WEIGHT_DIAGONAL, _WEIGHT_GP = 0, 1, 2


def _fused_weight(kind: int, weight_kind: int) -> bool:
    """True if the linearize / error kernels of `kind` apply cost weights of `weight_kind` (include/thb200.h, enum thb_weight_kind)."""
    if weight_kind in (_WEIGHT_SCALE, _WEIGHT_DIAGONAL):
        return True
    return weight_kind == _WEIGHT_GP and kind in _FOUR_VAR_KINDS


def _require_cuda_device(device):
    """The product has no CPU path: fail loudly.  (tests/test_simt_engine_emulation.py replaces this guard AND the library by a host
    emulation of the kernels to exercise the host code without a GPU; nothing in the package does.)"""
    if device.type != "cuda":
        raise RuntimeError(
            "theseus_b200: the objective must live on a CUDA device (call objective.to('cuda')); "
            "there is no CPU implementation of the linearize/solve/retract path in this package")


class _Group:
    """One cost-function schema: static placement arrays + (re)bindable pointer tables."""

    def __init__(self, kind, weight_kind, dim, cost_indices):
        self.kind, self.weight_kind, self.dim = kind, weight_kind, dim
        self.cost_indices = cost_indices
        self.K = len(cost_indices)
        self.static = {}
        self.bound = {}  # binding name -> (struct, keepalive tensors)


class Engine:
    def __init__(self, objective, ordering_names=None):
        self.objective = objective
        self.custom_ordering = None if ordering_names is None else tuple(ordering_names)   # None = default order (Objective.engine)
        self.structure_version = objective._structure_version
        self.device = torch.device(objective.device)
        _require_cuda_device(self.device)
        self.dtype = objective.dtype
        if self.dtype not in (torch.float64, torch.float32):
            raise ValueError(f"unsupported dtype {self.dtype}")
        self.sfx = "f64" if self.dtype == torch.float64 else "f32"
        self.lib = _lib.load()

        # ---- ordering (theseus/optimizer/variable_ordering.py:19-27: order of first appearance) ----
        self.ordering: List[Manifold] = (list(objective.optim_vars.values()) if ordering_names is None
                                         else [objective.optim_vars[n] for n in ordering_names])
        self.var_index = {v.name: i for i, v in enumerate(self.ordering)}
        for v in self.ordering:
            if int(getattr(v, "KIND", -1)) not in (0, 1, 2, 3, 4):
                raise NotImplementedError(
                    f"optimisation variable {v.name} ({type(v).__name__}): the retract / commit kernels are compiled for the variable kinds of "
                    "include/thb200.h (SE3, SO3, Vector / Point2 / Point3, SE2, SO2); a user-defined Manifold cannot be an optimisation variable")
        costs = list(objective.cost_functions.values())
        self.costs = costs
        cdesc = [(cf.dim(), [self.var_index[v.name] for v in cf.optim_vars]) for cf in costs]
        self.structure = build_structure([v.dof() for v in self.ordering], cdesc)
        S = self.structure
        self.n, self.m, self.nnz = S.num_cols, S.num_rows, S.nnz

        # ---- schema groups ----
        groups = {}
        self._aux_of = []
        self.generic = []  # cost functions without a CUDA schema (AutoDiffCostFunction): torch.func Jacobians, scattered into the CSR
        for f, cf in enumerate(costs):
            kind, aux = cf.schema()
            self._aux_of.append(list(aux) if isinstance(aux, (list, tuple)) else [aux])
            if kind is None or not _fused_weight(kind, cf.weight.WEIGHT_KIND):   # no fused kernel for this cost function / its CostWeight
                self.generic.append(f)
                continue
            grid = tuple(cf.sdf_data.tensor.shape[1:]) if kind in _COLLISION_KINDS else None   # the kernels take one grid shape per group
            key = (kind, cf.weight.WEIGHT_KIND, cf.dim(), int(getattr(cf, "robust_kind", 0)), grid)
            groups.setdefault(key, []).append(f)
        self.groups: List[_Group] = []
        dev = self.device
        for (kind, wkind, dim, robust, grid), idx in groups.items():
            g = _Group(kind, wkind, dim, idx)
            g.robust, g.grid = robust, grid
            ii = np.array(idx, dtype=np.int64)
            bp = np.zeros((g.K, 4 if kind in _FOUR_VAR_KINDS else 2), dtype=np.int32)
            for r, f in enumerate(idx):
                p = S.block_pointers[f]
                bp[r, : len(p)] = p
            g.static = dict(
                a_off=_dev(S.row_block_starts[ii], dev), a_stride=_dev(S.stride[ii].astype(np.int32), dev),
                bp=_dev(bp, dev), row0=_dev(S.cost_row0[ii].astype(np.int32), dev))
            self.groups.append(g)
        self.num_chunks = [int(self.lib.thb_error_num_chunks(g.K)) for g in self.groups]
        self.total_chunks = int(sum(self.num_chunks))

        # ---- variable table static parts ----
        self._vt_static = dict(
            kind=_dev(np.array([v.KIND for v in self.ordering], dtype=np.int32), dev),
            col=_dev(S.var_start_cols.astype(np.int32), dev),
            dof=_dev(S.var_dims.astype(np.int32), dev))

        self._B = None
        self._pool_cur = self._pool_tmp = None
        self.cur_views: List[torch.Tensor] = []
        self.tmp_views: List[torch.Tensor] = []
        self._bind_stamp = {"cur": -1, "tmp": -1}
        self._bind_sig = {}
        self._sig_vars = None
        self.table_version = 0
        self._vt = None
        self._gram_dense = None
        self._zero_filled = None  # (data_ptr, numel) of the AtA buffer whose off-pattern entries are known to be zero
        self._bufs = {}

    # ------------------------------------------------------------------ pools / bindings
    @property
    def batch_size(self) -> int:
        return self.objective.batch_size

    def _ensure_pools(self):
        B = self.batch_size
        if self._B == B and self._pool_cur is not None:
            return
        self._B = B
        sizes = [v.numel() for v in self.ordering]
        # every view starts on a 32-byte boundary (the kernels use 16-byte vector loads on SE3 elements; Point3 views
        # of odd length would otherwise push the following variable off alignment)
        lens = [B * s for s in sizes]
        padded = [(n + 3) // 4 * 4 for n in lens]
        offs = np.concatenate([[0], np.cumsum(padded)]).astype(np.int64)
        total = int(offs[-1])
        self._pool_cur = torch.empty(total, dtype=self.dtype, device=self.device)
        self._pool_tmp = torch.empty(total, dtype=self.dtype, device=self.device)
        self._view_offs, self._view_lens = offs, lens
        self.cur_views, self.tmp_views = [], []
        for i, v in enumerate(self.ordering):
            shp = (B,) + tuple(v.tensor.shape[1:])
            self.cur_views.append(self._pool_cur[offs[i]:offs[i] + lens[i]].view(shp))
            self.tmp_views.append(self._pool_tmp[offs[i]:offs[i] + lens[i]].view(shp))
        self._bufs = {}
        self._vt = None
        self._bind_stamp = {"cur": -1, "tmp": -1}
        self._bind_sig = {}

    def adopt_optim_vars(self):
        """Move every optimisation variable into the engine-owned pool (copying the current values) so that
        the optimiser can update them in place without touching caller-owned tensors."""
        self._ensure_pools()
        src, dst = [], []
        for v, view in zip(self.ordering, self.cur_views):
            t = v.tensor
            if t.data_ptr() == view.data_ptr() and t.shape == view.shape:
                continue
            if t.device != self.device or t.dtype != self.dtype:
                raise ValueError(f"variable {v.name} is on ({t.device},{t.dtype}), objective expects ({self.device},{self.dtype})")
            src.append(t.expand(view.shape) if t.shape[0] != view.shape[0] else t)
            dst.append(view)
        if src:
            torch._foreach_copy_(dst, src)
            for v, view in zip(self.ordering, self.cur_views):
                if v.tensor.data_ptr() != view.data_ptr():
                    v.tensor = view

    def solution_tensors(self):
        """name -> tensor of every optimisation variable, safe to hand to the caller: variables that live in the engine-owned pool (which
        the next optimize() overwrites in place) are returned as views of ONE clone of the pool -- the reference rebinds fresh tensors
        (Variable.update / torch.where, core/variable.py:42-72), so solutions it returned earlier never change."""
        out, snap = {}, None
        for i, v in enumerate(self.ordering):
            t = v.tensor
            if self._pool_cur is not None and i < len(getattr(self, "cur_views", ())) and t.data_ptr() == self.cur_views[i].data_ptr() and not t.requires_grad:
                if snap is None:
                    snap = self._pool_cur.clone()
                o = int(self._view_offs[i])
                t = snap[o:o + self._view_lens[i]].view(self.cur_views[i].shape)
            out[v.name] = t
        return out

    def _ptr_array(self, tensors) -> torch.Tensor:
        return _dev(np.fromiter((t.data_ptr() for t in tensors), dtype=np.int64, count=len(tensors)), self.device)

    def _bind(self, which: str):
        """(Re)build the pointer tables of every group for binding `which` ('cur' = objective variables,
        'tmp' = trial pool) if any variable tensor was rebound since the last build."""
        if self._bind_stamp[which] == Variable._global_updates:
            return
        # Some variable was rebound since the tables were built.  The common case inside a training / serving loop is that every
        # tensor still lives where it did (objective.update() + adopt_optim_vars() put the new VALUES into the same pool views and
        # the caller re-uses its input buffers): compare the device pointers before paying for the rebuild (~10 ms at C2: Python over
        # every cost function + pageable H2D copies of the pointer tables).
        sig = self._bind_signature(which)
        if sig is not None and sig == self._bind_sig.get(which):
            self._bind_stamp[which] = Variable._global_updates
            return
        B = self.batch_size
        if which == "tmp" or self._B is not None:
            self._ensure_pools()

        def optim_tensor(v):
            if which == "tmp":
                return self.tmp_views[self.var_index[v.name]]
            t = v.tensor
            if t.device != self.device:
                raise ValueError(f"variable {v.name} is on {t.device}, objective is on {self.device}")
            if not t.is_contiguous() or t.data_ptr() % 16 != 0:  # kernels use 16-byte vector loads
                t = t.clone(memory_format=torch.contiguous_format)
                v.tensor = t
            return t

        def aux_tensor(v):
            t = v.tensor
            if t.device != self.device or t.dtype != self.dtype:
                raise ValueError(f"variable {v.name} is on ({t.device},{t.dtype}), objective expects ({self.device},{self.dtype})")
            if not t.is_contiguous() or t.data_ptr() % 16 != 0:
                t = t.clone(memory_format=torch.contiguous_format)
                v.tensor = t
            return t

        def bstride(t):
            if t.shape[0] == B:
                return int(t[0].numel())
            if t.shape[0] == 1:
                return 0
            raise ValueError("Provided tensors must be broadcastable.")

        for g in self.groups:
            x0, x1, aux, w = [], [], [], []
            x2, x3 = [], []
            extra = [[], [], []]
            n_extra = len(self._aux_of[g.cost_indices[0]]) - 1
            bs = np.zeros((g.K, 4), dtype=np.int32)
            bs2 = np.zeros((g.K, 3), dtype=np.int32)
            bs3 = np.zeros((g.K, 2), dtype=np.int32)
            for r, f in enumerate(g.cost_indices):
                cf = self.costs[f]
                ov = cf.optim_vars
                t0 = optim_tensor(ov[0])
                t1 = optim_tensor(ov[1]) if len(ov) > 1 else t0
                auxs = [aux_tensor(a) for a in self._aux_of[f]]
                tw = aux_tensor(cf.weight.weight_tensor())
                x0.append(t0); x1.append(t1); aux.append(auxs[0]); w.append(tw)
                bs[r] = (bstride(t0), bstride(t1), bstride(auxs[0]), bstride(tw))
                if g.kind in _FOUR_VAR_KINDS:
                    t2, t3 = optim_tensor(ov[2]), optim_tensor(ov[3])
                    x2.append(t2); x3.append(t3)
                    bs3[r] = (bstride(t2), bstride(t3))
                if g.grid is not None and tuple(auxs[1].shape[1:]) != g.grid:
                    raise ValueError(f"{cf.name}: sdf_data changed shape from {g.grid} to {tuple(auxs[1].shape[1:])} after the objective was "
                                     "compiled; add the cost function again (or use maps of one shape)")
                for q in range(n_extra):
                    extra[q].append(auxs[1 + q])
                    bs2[r, q] = bstride(auxs[1 + q])
            keep = dict(x0=self._ptr_array(x0), x1=self._ptr_array(x1), aux=self._ptr_array(aux), w=self._ptr_array(w),
                        bstride=_dev(bs, self.device), tensors=(x0, x1, aux, w, extra, x2, x3))
            if x2:
                keep["x2"], keep["x3"], keep["bstride3"] = self._ptr_array(x2), self._ptr_array(x3), _dev(bs3, self.device)
            ex = [self._ptr_array(extra[q]) if n_extra > q else None for q in range(3)]
            keep["extra"] = ex
            keep["bstride2"] = _dev(bs2, self.device)
            lr_ptr = lr_bs = None
            if g.robust:
                lrs = [aux_tensor(self.costs[f].log_loss_radius) for f in g.cost_indices]
                lr_ptr = self._ptr_array(lrs)
                lr_bs = _dev(np.array([bstride(t) for t in lrs], dtype=np.int32), self.device)
                keep["lr"] = (lrs, lr_ptr, lr_bs)
            st = _lib.CostGroup(
                kind=g.kind, weight_kind=g.weight_kind, K=g.K, dim=g.dim,
                x0=keep["x0"].data_ptr(), x1=keep["x1"].data_ptr(), aux=keep["aux"].data_ptr(), w=keep["w"].data_ptr(),
                bstride=keep["bstride"].data_ptr(), a_off=g.static["a_off"].data_ptr(),
                a_stride=g.static["a_stride"].data_ptr(), bp=g.static["bp"].data_ptr(), row0=g.static["row0"].data_ptr(),
                aux2=ex[0].data_ptr() if ex[0] is not None else None, aux3=ex[1].data_ptr() if ex[1] is not None else None,
                aux4=ex[2].data_ptr() if ex[2] is not None else None, bstride2=keep["bstride2"].data_ptr(),
                robust_kind=g.robust, reserved0=0, log_radius=lr_ptr.data_ptr() if lr_ptr is not None else None,
                bstride_lr=lr_bs.data_ptr() if lr_bs is not None else None,
                x2=keep["x2"].data_ptr() if "x2" in keep else None, x3=keep["x3"].data_ptr() if "x3" in keep else None,
                bstride3=keep["bstride3"].data_ptr() if "bstride3" in keep else None,
                sdf_rows=g.grid[0] if g.grid is not None else 0, sdf_cols=g.grid[1] if g.grid is not None else 0)
            g.bound[which] = (st, keep)
        # NOTE: _bind may itself rebind non-contiguous tensors (bumping the counter); read it afterwards.
        self._bind_stamp[which] = Variable._global_updates
        self._bind_sig[which] = self._bind_signature(which)
        self.table_version += 1  # captured CUDA graphs hold the old tables' device pointers: optimizers re-capture on a change
        if which == "cur":
            self._vt = None

    def _bind_signature(self, which: str):
        """(data_ptr, batch) of every tensor the pointer tables of binding `which` refer to, or None if a tensor would need a
        contiguous/aligned copy (then the full rebuild handles it)."""
        if self._sig_vars is None:
            vs = []
            for g in self.groups:
                for f in g.cost_indices:
                    cf = self.costs[f]
                    vs.extend(self._aux_of[f])
                    vs.append(cf.weight.weight_tensor())
                    if g.robust:
                        vs.append(cf.log_loss_radius)
            vs.extend(self.ordering)
            seen, uniq = set(), []
            for v in vs:
                if id(v) not in seen:
                    seen.add(id(v)); uniq.append(v)
            self._sig_vars = uniq
        sig = [self._B if which == "tmp" else -1]
        for v in self._sig_vars:
            t = v.tensor
            p = t.data_ptr()
            if p % 16 != 0 or not t.is_contiguous():
                return None
            sig.append(p); sig.append(t.shape[0])
        return tuple(sig)

    def _var_table(self):
        """thb_var_table: x = current variables, out = trial pool."""
        self._ensure_pools()
        self._bind("cur")
        if self._vt is None:
            xs = [v.tensor for v in self.ordering]
            for v, t in zip(self.ordering, xs):
                if t.shape[0] != self._B:
                    raise ValueError(f"optimisation variable {v.name} has batch {t.shape[0]} != {self._B}; call adopt_optim_vars()")
            keep = dict(x=self._ptr_array(xs), out=self._ptr_array(self.tmp_views))
            st = _lib.VarTable(N=len(xs), x=keep["x"].data_ptr(), out=keep["out"].data_ptr(),
                               kind=self._vt_static["kind"].data_ptr(), col=self._vt_static["col"].data_ptr(),
                               dof=self._vt_static["dof"].data_ptr())
            self._vt = (st, keep)
        return self._vt[0]

    def buf(self, name, shape, dtype=None, zero=False):
        key = (name, tuple(shape), dtype or self.dtype)
        t = self._bufs.get(key)
        if t is None:
            t = (torch.zeros if zero else torch.empty)(shape, dtype=dtype or self.dtype, device=self.device)
            self._bufs[key] = t
        return t

    def buf_const(self, name, arr: np.ndarray):
        key = ("const", name)
        t = self._bufs.get(key)
        if t is None:
            t = _dev(arr, self.device)
            self._bufs[key] = t
        return t

    # ------------------------------------------------------------------ kernels
    def linearize_sparse(self, A_val: Optional[torch.Tensor] = None, b: Optional[torch.Tensor] = None):
        """A_val [B,nnz], b [B,m] in the layout of SparseLinearization (optimizer/sparse_linearization.py:102-140)."""
        self._bind("cur")
        B = self.batch_size
        if A_val is None:
            A_val = self.buf("A_val", (B, self.nnz))
        if b is None:
            b = self.buf("b", (B, self.m))
        fn = getattr(self.lib, f"thb_linearize_group_{self.sfx}")
        s = _lib.stream_ptr()
        for g in self.groups:
            _lib.check(fn(C.byref(g.bound["cur"][0]), B, _lib.ptr(A_val), self.nnz, _lib.ptr(b), self.m, s), "linearize_group")
        S = self.structure
        if self.generic and _batched_torch_route() and not self._user_costs(self.generic):
            self._route("generic").linearize(lambda v: self._expand(v.tensor), B, A_val, b, differentiable=False)
            return A_val, b
        for f in self.generic:
            cf = self.costs[f]
            jacs, err = cf.generic_jacobians_error([self._expand(v.tensor) for v in cf.optim_vars])
            d, st, off = int(S.cost_dims[f]), int(S.stride[f]), int(S.row_block_starts[f])
            blk = A_val[:, off:off + d * st].view(B, d, st)
            for kslot, J in enumerate(jacs):
                p0 = int(S.block_pointers[f][kslot])
                blk[:, :, p0:p0 + J.shape[2]] = J
            b[:, int(S.cost_row0[f]):int(S.cost_row0[f]) + d] = -err
        return A_val, b

    def linearize_sparse_differentiable(self):
        """(A_val, b) as autograd tensors: same layout, values from the cost functions' torch.func Jacobians without detaching, so
        gradients reach the auxiliary variables / cost weights / current variable values.  AutoDiffCostFunctions use the user's
        err_fn, the fused-kernel cost functions their torch restatement (core.CostFunction._torch_error)."""
        B, S = self.batch_size, self.structure
        A_val = torch.zeros(B, self.nnz, dtype=self.dtype, device=self.device)
        b = torch.zeros(B, self.m, dtype=self.dtype, device=self.device)
        if _batched_torch_route() and not self._user_costs(range(len(self.costs))):   # one vmap(jacrev) per group of stackable cost functions instead of one per cost function
            return self._route("all").linearize(lambda v: self._expand(v.tensor), B, A_val, b, differentiable=True)
        for f, cf in enumerate(self.costs):  # every cost function through its torch restatement (O(#costs) torch calls: taped steps only)
            jacs, err = cf.generic_jacobians_error([self._expand(v.tensor) for v in cf.optim_vars], differentiable=True)
            d, st, off = int(S.cost_dims[f]), int(S.stride[f]), int(S.row_block_starts[f])
            blk = A_val[:, off:off + d * st].view(B, d, st)
            for kslot, J in enumerate(jacs):
                p0 = int(S.block_pointers[f][kslot])
                blk[:, :, p0:p0 + J.shape[2]] = J
            b[:, int(S.cost_row0[f]):int(S.cost_row0[f]) + d] = -err
        return A_val, b

    def _user_costs(self, ids) -> bool:
        """True if any of these cost functions is a user-defined subclass (own error() / jacobians()): those run per cost function."""
        return any(self.costs[f]._user_defined("jacobians") or self.costs[f]._user_defined("error")
                   or self.costs[f].weight.WEIGHT_KIND not in (_WEIGHT_SCALE, _WEIGHT_DIAGONAL)
                   or getattr(getattr(self.costs[f], "cost_function", None), "_user_defined", lambda w: False)("jacobians") for f in ids)

    def _route(self, which: str):
        """torch_route.TorchRoute over the generic cost functions ("generic") or over all of them ("all", taped linearization)."""
        if not hasattr(self, "_routes"):
            self._routes = {}
        if which not in self._routes:
            from .torch_route import TorchRoute
            ids = list(self.generic) if which == "generic" else list(range(len(self.costs)))
            self._routes[which] = TorchRoute(self.costs, ids, self.structure)
        return self._routes[which]

    def _expand(self, t):
        B = self.batch_size
        return t if t.shape[0] == B else t.expand((B,) + tuple(t.shape[1:]))

    def error_metric(self, which: str = "cur", out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """0.5 * sum((w e)^2) per batch item (core/objective.py:615-641), deterministic two-stage reduction."""
        self._bind(which)
        B = self.batch_size
        partial = self.buf("err_partial", (max(self.total_chunks, 1), B))
        if out is None:
            out = torch.empty(B, dtype=self.dtype, device=self.device)
        fn = getattr(self.lib, f"thb_error_group_{self.sfx}")
        s = _lib.stream_ptr()
        row = 0
        for g, nc in zip(self.groups, self.num_chunks):
            _lib.check(fn(C.byref(g.bound[which][0]), B, _lib.ptr(partial[row:]), s), "error_group")
            row += nc
        _lib.check(getattr(self.lib, f"thb_error_reduce_{self.sfx}")(_lib.ptr(partial), self.total_chunks, B, _lib.ptr(out), s), "error_reduce")
        if self.generic and _batched_torch_route() and not self._user_costs(self.generic):
            of = (lambda v: self.tmp_views[self.var_index[v.name]]) if which == "tmp" else (lambda v: self._expand(v.tensor))
            out += self._route("generic").half_squared_error(of, B)
            return out
        for f in self.generic:
            cf = self.costs[f]
            ts = [self.tmp_views[self.var_index[v.name]] if which == "tmp" else self._expand(v.tensor) for v in cf.optim_vars]
            e = cf.generic_error(ts)
            out += (e * e).sum(dim=1) * 0.5
        return out

    def gram_plan_dense(self):
        if self._gram_dense is None:
            arrs = build_gram_plan(self.structure)
            dev = {k: _dev(v, self.device) for k, v in arrs.items() if isinstance(v, np.ndarray)}
            st = _lib.make_gram_plan(arrs, dev)
            self._gram_dense = (st, dev, arrs)   # arrs keeps the HOST segment table of the struct alive
        return self._gram_dense[0]

    def gram_dense(self, A_val, b, AtA, Atb, diag):
        """AtA [B,n,n] (block scatter over a zero background), Atb [B,n], diag(AtA) [B,n].

        The block pattern of AtA is fixed by the objective's structure and the Gram kernel overwrites every pattern
        block, so the 8*B*n^2-byte zero fill (4.8 GB, ~1.9 ms at C2) is paid once per buffer, not once per iteration.
        Nothing downstream writes AtA (the damping is fused into the factorisation's load)."""
        B = self.batch_size
        s = _lib.stream_ptr()
        if self.dense_jacobian(A_val):
            # every cost function touches every variable: A_val IS the row-major dense Jacobian [B, m, n] -> TMA + DMMA Gram kernel
            # (thb_gram_dense.cu); Atb / diag(AtA) from the column plan as usual
            _lib.check(self.lib.thb_gram_dense_f64(_lib.ptr(A_val), _lib.ptr(AtA), B, self.m, self.n, s), "gram_dense")
            self._zero_filled = None
            self.atb(A_val, b, Atb, diag)
            return
        plan = self.gram_plan_dense()
        key = (AtA.data_ptr(), AtA.numel())
        if self._zero_filled != key:
            _lib.check(self.lib.thb_fill_zero(_lib.ptr(AtA), AtA.numel() * AtA.element_size(), s), "fill_zero")
            self._zero_filled = key
        _lib.check(getattr(self.lib, f"thb_gram_{self.sfx}")(C.byref(plan), B, _lib.ptr(A_val), self.nnz, _lib.ptr(b), self.m, _lib.ptr(AtA),
                                                               self.n * self.n, _lib.ptr(Atb), _lib.ptr(diag), s), "gram")

    def dense_jacobian(self, A_val) -> bool:
        """True when the CSR pattern is full (nnz == m * n: A_val is the dense row-major Jacobian) and the dense Gram kernel applies
        (fp64, even n, enough work to fill tiles)."""
        return (self.nnz == self.m * self.n and A_val.dtype == torch.float64 and self.n % 2 == 0 and self.n >= 16 and self.m >= 64
                and A_val.is_contiguous() and A_val.data_ptr() % 16 == 0 and os.environ.get("THB_DENSE_GRAM", "1") != "0")

    def atb(self, A_val, b, Atb, diag=None):
        plan = self.gram_plan_dense()
        _lib.check(getattr(self.lib, f"thb_gram_{self.sfx}")(C.byref(plan), self.batch_size, _lib.ptr(A_val), self.nnz, _lib.ptr(b), self.m,
                                                               None, 0, _lib.ptr(Atb), _lib.ptr(diag), _lib.stream_ptr()), "atb")

    def retract_into(self, delta: torch.Tensor, out_vars, step: float, ignore_mask: Optional[torch.Tensor]):
        """tmp_i <- X_i * exp(step * delta_i), masked (core/objective.py:873-914)."""
        vt = self._var_table()
        for v, view in zip(out_vars, self.tmp_views):
            if v.tensor.data_ptr() != view.data_ptr():
                v.tensor = view  # trial containers are views of the trial pool
        B = self.batch_size
        delta = delta.contiguous()
        ig = None
        if ignore_mask is not None:
            ig = ignore_mask.to(torch.uint8) if ignore_mask.dtype != torch.uint8 else ignore_mask
        fn = getattr(self.lib, f"thb_retract_{self.sfx}")
        _lib.check(fn(C.byref(vt), B, _lib.ptr(delta), self.n, float(step), _lib.ptr(ig), _lib.stream_ptr()), "retract")
        self._keep = (delta, ig)

    def commit(self, keep_old_mask: Optional[torch.Tensor]):
        """X_i[b] <- tmp_i[b] where keep_old_mask[b] == 0 (objective.update(..., batch_ignore_mask), variable.py:65-69)."""
        vt = self._var_table()
        km = None
        if keep_old_mask is not None:
            km = keep_old_mask.to(torch.uint8) if keep_old_mask.dtype != torch.uint8 else keep_old_mask
        fn = getattr(self.lib, f"thb_commit_{self.sfx}")
        _lib.check(fn(C.byref(vt), self.batch_size, _lib.ptr(km), _lib.stream_ptr()), "commit")
        self._keep2 = km

// Fused cost-function kernels: residual + analytic Jacobians + weighting (linearize), residual-only
// error pass, retract, commit, LM control, and the stand-alone Lie kernels.
//
// One thread = one (cost function k, batch item b); b is the fast index so that the 96-byte SE3 chunks
// of consecutive batch items are read from consecutive addresses.  All Lie math lives in registers
// (thb_lie.cuh).  Kernels are HBM/latency bound (AI ~ 4 flop/B, SURVEY.md 8d): no tensor cores here
// by construction.
//
// Reference semantics: theseus/embodied/measurements/between.py:34-45, theseus/embodied/misc/local_cost_fn.py:40-61,
// theseus/core/cost_weight.py:81-90,125-136, theseus/optimizer/sparse_linearization.py:102-140.
#include "thb_common.cuh"
#include "thb_lie.cuh"

namespace thb {

constexpr int kErrCostsPerThread = 8;

template <typename T> struct GroupDev {
  int kind, weight_kind, K, dim;
  const T* const* x0;
  const T* const* x1;
  const T* const* aux;
  const T* const* w;
  const int32_t* bstride;
  const int64_t* a_off;
  const int32_t* a_stride;
  const int32_t* bp;
  const int32_t* row0;
  const T* const* aux2;
  const T* const* aux3;
  const T* const* aux4;
  const int32_t* bstride2;
  int robust_kind;
  const T* const* log_radius;
  const int32_t* bstride_lr;
  const T* const* x2;
  const T* const* x3;
  const int32_t* bstride3;
  int sdf_rows, sdf_cols;
};

template <typename T> static GroupDev<T> to_dev(const thb_cost_group* g) {
  GroupDev<T> d;
  d.kind = g->kind;
  d.weight_kind = g->weight_kind;
  d.K = g->K;
  d.dim = g->dim;
  d.x0 = reinterpret_cast<const T* const*>(g->x0);
  d.x1 = reinterpret_cast<const T* const*>(g->x1);
  d.aux = reinterpret_cast<const T* const*>(g->aux);
  d.w = reinterpret_cast<const T* const*>(g->w);
  d.bstride = g->bstride;
  d.a_off = g->a_off;
  d.a_stride = g->a_stride;
  d.bp = g->bp;
  d.row0 = g->row0;
  d.aux2 = reinterpret_cast<const T* const*>(g->aux2);
  d.aux3 = reinterpret_cast<const T* const*>(g->aux3);
  d.aux4 = reinterpret_cast<const T* const*>(g->aux4);
  d.bstride2 = g->bstride2;
  d.robust_kind = g->robust_kind;
  d.log_radius = reinterpret_cast<const T* const*>(g->log_radius);
  d.bstride_lr = g->bstride_lr;
  d.x2 = reinterpret_cast<const T* const*>(g->x2);
  d.x3 = reinterpret_cast<const T* const*>(g->x3);
  d.bstride3 = g->bstride3;
  d.sdf_rows = g->sdf_rows;
  d.sdf_cols = g->sdf_cols;
  return d;
}

// Robust wrapper (theseus/core/robust_cost_function.py:87-135; losses robust_loss.py:33-52; _EPS = _LOSS_EPS = 1e-20).
// x = squared norm of the weighted error.  linearize: rescale = sqrt(rho'(x) + eps) applied to J and e;
// evaluate: the error metric sees rho(x) (+ dim*eps) instead of x.
template <typename T> __device__ __forceinline__ T t_exp(T x);
template <> __device__ __forceinline__ float t_exp<float>(float x) { return expf(x); }
template <> __device__ __forceinline__ double t_exp<double>(double x) { return exp(x); }
template <typename T> __device__ __forceinline__ T robust_radius(const GroupDev<T>& g, int k, int64_t b) {
  return t_exp((g.log_radius[k] + (int64_t)g.bstride_lr[k] * b)[0]);
}
template <typename T> __device__ __forceinline__ T robust_rescale(const GroupDev<T>& g, int k, int64_t b, T x) {
  const T radius = robust_radius(g, k, b);
  T lin;
  if (g.robust_kind == THB_ROBUST_WELSCH) lin = t_exp(-x / (radius + T(1e-20)));
  else lin = t_sqrt(radius / (x > radius ? x : radius) + T(1e-20));
  return t_sqrt(lin + T(1e-20));
}
template <typename T> __device__ __forceinline__ T robust_value(const GroupDev<T>& g, int k, int64_t b, T x, int dim) {
  const T radius = robust_radius(g, k, b);
  T val;
  if (g.robust_kind == THB_ROBUST_WELSCH) val = radius - radius * t_exp(-x / (radius + T(1e-20)));
  else val = (x > radius) ? (T(2) * t_sqrt(radius * (x > radius ? x : radius) + T(1e-20)) - radius) : x;
  // the reference spreads rho over `dim` entries sqrt(rho/dim + eps); their squares sum to rho + dim*eps
  return val + T(dim) * T(1e-20);
}

template <typename T, int N> __device__ __forceinline__ void load_n(const T* p, T* r) {
#pragma unroll
  for (int i = 0; i < N; i++) r[i] = p[i];
}
// 12 scalars of an SE3 element; 16-byte vector loads when aligned (always true for [B,3,4] tensors)
__device__ __forceinline__ void load_se3(const double* p, double* r) {
  const double2* q = reinterpret_cast<const double2*>(p);
#pragma unroll
  for (int i = 0; i < 6; i++) {
    double2 v = q[i];
    r[2 * i] = v.x;
    r[2 * i + 1] = v.y;
  }
}
__device__ __forceinline__ void load_se3(const float* p, float* r) {
  const float4* q = reinterpret_cast<const float4*>(p);
#pragma unroll
  for (int i = 0; i < 3; i++) {
    float4 v = q[i];
    r[4 * i] = v.x;
    r[4 * i + 1] = v.y;
    r[4 * i + 2] = v.z;
    r[4 * i + 3] = v.w;
  }
}

// weights: returns true if all weights of this (k,b) are exactly zero (masked cost function,
// theseus/core/cost_function.py:37-55,107-122)
template <typename T, int DIM> __device__ __forceinline__ bool load_weight(const GroupDev<T>& g, int k, int64_t b, T* w) {
  const T* wp = g.w[k] + (int64_t)g.bstride[k * 4 + 3] * b;
  bool all_zero = true;
  if (g.weight_kind == THB_WEIGHT_SCALE) {
    const T s = wp[0];
#pragma unroll
    for (int r = 0; r < DIM; r++) w[r] = s;
    all_zero = (s == T(0));
  } else {
#pragma unroll
    for (int r = 0; r < DIM; r++) {
      w[r] = wp[r];
      all_zero = all_zero && (w[r] == T(0));
    }
  }
  return all_zero;
}

// ------------------------------------------------------------------------------------------------
// residual (+ Jacobians) of one SE3 cost function.  J0/J1 row-major 6x6, already weighted; e weighted.
template <typename T, bool WITH_J, bool BETWEEN>
__device__ __forceinline__ void se3_cost(const GroupDev<T>& g, int k, int64_t b, const T* w, T* e, T* J0, T* J1) {
  T X0[12], Z[12], D[12], E[12];
  load_se3(g.x0[k] + (int64_t)g.bstride[k * 4 + 0] * b, X0);
  load_se3(g.aux[k] + (int64_t)g.bstride[k * 4 + 2] * b, Z);
  if (BETWEEN) {
    T X1[12];
    load_se3(g.x1[k] + (int64_t)g.bstride[k * 4 + 1] * b, X1);
    se3_between(X0, X1, D);  // D = X0^-1 X1
    se3_between(Z, D, E);    // E = Z^-1 D
  } else {
    se3_between(Z, X0, E);   // E = T^-1 X
  }
  T Jl[36];
  se3_log_jlog<T, WITH_J>(E, e, Jl);
#pragma unroll
  for (int r = 0; r < 6; r++) e[r] *= w[r];
  if (WITH_J) {
    if (BETWEEN) {
      // J0 = -dlog @ Ad(D^-1)  (between.py:43); J1 = dlog
      T Di[12], Ad[36];
      se3_inverse(D, Di);
      se3_adjoint(Di, Ad);
#pragma unroll
      for (int r = 0; r < 6; r++) {
#pragma unroll
        for (int c = 0; c < 6; c++) {
          T s = T(0);
#pragma unroll
          for (int q = 0; q < 6; q++) s += Jl[r * 6 + q] * Ad[q * 6 + c];
          J0[r * 6 + c] = (-s) * w[r];
        }
      }
#pragma unroll
      for (int r = 0; r < 6; r++)
#pragma unroll
        for (int c = 0; c < 6; c++) J1[r * 6 + c] = Jl[r * 6 + c] * w[r];
    } else {
#pragma unroll
      for (int r = 0; r < 6; r++)
#pragma unroll
        for (int c = 0; c < 6; c++) J0[r * 6 + c] = Jl[r * 6 + c] * w[r];
    }
  }
}

template <typename T, bool WITH_J, bool BETWEEN>
__device__ __forceinline__ void so3_cost(const GroupDev<T>& g, int k, int64_t b, const T* w, T* e, T* J0, T* J1) {
  T X0[9], Z[9], D[9], E[9];
  load_n<T, 9>(g.x0[k] + (int64_t)g.bstride[k * 4 + 0] * b, X0);
  load_n<T, 9>(g.aux[k] + (int64_t)g.bstride[k * 4 + 2] * b, Z);
  if (BETWEEN) {
    T X1[9];
    load_n<T, 9>(g.x1[k] + (int64_t)g.bstride[k * 4 + 1] * b, X1);
    so3_between(X0, X1, D);
    so3_between(Z, D, E);
  } else {
    so3_between(Z, X0, E);
  }
  So3LogAux<T> a = so3_log<T, 3>(E, e);
  T Jl[9], bw[3];
  if (WITH_J) so3_jlog<T, 3>(e, a, Jl, bw);
  if (WITH_J) {
    if (BETWEEN) {
      // Ad(D^-1) = D^T
#pragma unroll
      for (int r = 0; r < 3; r++)
#pragma unroll
        for (int c = 0; c < 3; c++) {
          T s = Jl[r * 3 + 0] * D[c * 3 + 0] + Jl[r * 3 + 1] * D[c * 3 + 1] + Jl[r * 3 + 2] * D[c * 3 + 2];
          J0[r * 3 + c] = (-s) * w[r];
          J1[r * 3 + c] = Jl[r * 3 + c] * w[r];
        }
    } else {
#pragma unroll
      for (int i = 0; i < 9; i++) J0[i] = Jl[i] * w[i / 3];
    }
  }
#pragma unroll
  for (int r = 0; r < 3; r++) e[r] *= w[r];
}

template <typename T, bool WITH_J, bool BETWEEN>
__device__ __forceinline__ void se2_cost(const GroupDev<T>& g, int k, int64_t b, const T* w, T* e, T* J0, T* J1) {
  T X0[4], Z[4], D[4], E[4];
  load_n<T, 4>(g.x0[k] + (int64_t)g.bstride[k * 4 + 0] * b, X0);
  load_n<T, 4>(g.aux[k] + (int64_t)g.bstride[k * 4 + 2] * b, Z);
  if (BETWEEN) {
    T X1[4];
    load_n<T, 4>(g.x1[k] + (int64_t)g.bstride[k * 4 + 1] * b, X1);
    se2_between(X0, X1, D);
    se2_between(Z, D, E);
  } else {
    se2_between(Z, X0, E);
  }
  T Jl[9];
  se2_log_jlog<T, WITH_J>(E, e, Jl);
#pragma unroll
  for (int r = 0; r < 3; r++) e[r] *= w[r];
  if (WITH_J) {
    if (BETWEEN) {
      T Di[4], Ad[9];
      se2_inverse(D, Di);
      se2_adjoint(Di, Ad);
#pragma unroll
      for (int r = 0; r < 3; r++)
#pragma unroll
        for (int c = 0; c < 3; c++) {
          const T s = Jl[r * 3 + 0] * Ad[0 * 3 + c] + Jl[r * 3 + 1] * Ad[1 * 3 + c] + Jl[r * 3 + 2] * Ad[2 * 3 + c];
          J0[r * 3 + c] = (-s) * w[r];
          J1[r * 3 + c] = Jl[r * 3 + c] * w[r];
        }
    } else {
#pragma unroll
      for (int i = 0; i < 9; i++) J0[i] = Jl[i] * w[i / 3];
    }
  }
}

// ------------------------------------------------------------------------------------------------
template <typename T, int KIND>
__global__ void __launch_bounds__(128) linearize_kernel(GroupDev<T> g, int64_t B, T* __restrict__ A_val, int64_t nnz,
                                                        T* __restrict__ bvec, int64_t m) {
  extern __shared__ double lin_stage_raw[];
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const bool valid = t < (int64_t)g.K * B;     // (no early exit: every lane takes part in the warp-cooperative store below)
  const int k = valid ? (int)(t / B) : 0;
  const int64_t b = valid ? t - (int64_t)k * B : 0;
  constexpr int DIM = (KIND == THB_COST_BETWEEN_SE3 || KIND == THB_COST_LOCAL_SE3) ? 6 : 3;
  constexpr bool BETWEEN = (KIND == THB_COST_BETWEEN_SE3 || KIND == THB_COST_BETWEEN_SO3 || KIND == THB_COST_BETWEEN_SE2);
  constexpr bool IS_SE2 = (KIND == THB_COST_BETWEEN_SE2 || KIND == THB_COST_LOCAL_SE2);
  T w[DIM], e[DIM], J0[DIM * DIM], J1[DIM * DIM];
  const bool masked = load_weight<T, DIM>(g, k, b, w);
  if (masked) {
#pragma unroll
    for (int i = 0; i < DIM; i++) e[i] = T(0);
#pragma unroll
    for (int i = 0; i < DIM * DIM; i++) { J0[i] = T(0); J1[i] = T(0); }
  } else if (DIM == 6) {
    se3_cost<T, true, BETWEEN>(g, k, b, w, e, J0, J1);
  } else if (IS_SE2) {
    se2_cost<T, true, BETWEEN>(g, k, b, w, e, J0, J1);
  } else {
    so3_cost<T, true, BETWEEN>(g, k, b, w, e, J0, J1);
  }
  if (g.robust_kind != THB_ROBUST_NONE && !masked) {
    T x = T(0);
#pragma unroll
    for (int r = 0; r < DIM; r++) x += e[r] * e[r];
    const T sc = robust_rescale(g, k, b, x);
#pragma unroll
    for (int r = 0; r < DIM; r++) e[r] *= sc;
#pragma unroll
    for (int i = 0; i < DIM * DIM; i++) { J0[i] *= sc; if (BETWEEN) J1[i] *= sc; }
  }
  // A cost function's rows of A_val are ONE contiguous run of DIM * stride values per batch item (stride = its row length), but the
  // items of a warp lie nnz values apart: storing from the computing thread writes 8 bytes to 32 different sectors per instruction.
  // Stage the warp's 32 runs in shared memory and let the whole warp store each run with consecutive lanes (256-byte segments).
  T* Arow = A_val + b * nnz + g.a_off[k];
  const int stride = g.a_stride[k];
  constexpr int NVMAX = DIM * DIM * (BETWEEN ? 2 : 1);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  T* stage = reinterpret_cast<T*>(lin_stage_raw) + (size_t)warp * 32 * (NVMAX + 1);
  T* mine = stage + lane * (NVMAX + 1);
  const int nv = DIM * stride;                 // <= NVMAX by construction of the groups (stride = DIM or 2 DIM)
  const int bp0 = g.bp[k * 2 + 0];
#pragma unroll
  for (int r = 0; r < DIM; r++)
#pragma unroll
    for (int c = 0; c < DIM; c++) mine[r * stride + bp0 + c] = J0[r * DIM + c];
  if (BETWEEN) {
    const int bp1 = g.bp[k * 2 + 1];
#pragma unroll
    for (int r = 0; r < DIM; r++)
#pragma unroll
      for (int c = 0; c < DIM; c++) mine[r * stride + bp1 + c] = J1[r * DIM + c];
  }
  __syncwarp();
  const unsigned long long my_dst = valid ? reinterpret_cast<unsigned long long>(Arow) : 0ull;
  for (int i = 0; i < 32; i++) {
    const unsigned long long d = __shfl_sync(0xffffffffu, my_dst, i);
    const int nvi = __shfl_sync(0xffffffffu, nv, i);
    if (d != 0ull) {
      T* dst = reinterpret_cast<T*>(d);
      const T* src = stage + i * (NVMAX + 1);
      for (int v = lane; v < nvi; v += 32) dst[v] = src[v];
    }
  }
  if (valid) {
    T* brow = bvec + b * m + g.row0[k];
#pragma unroll
    for (int r = 0; r < DIM; r++) brow[r] = -e[r];
  }
}

// Reprojection (theseus/embodied/measurements/reprojection.py:54-94): q = R p + t, proj = -q_xy/q_z,
// e = proj * f (1 + n (k1 + n k2)) - z with n = |proj|^2.  Jacobians by the quotient rule on
// [R, -R hat(p) | R] (torchlie se3_impl.py:764-777), exactly as the reference composes them.
template <typename T, bool WITH_J>
__device__ __forceinline__ void reprojection_cost(const GroupDev<T>& g, int k, int64_t b, const T* w, T* e, T* Jc, T* Jp) {
  T X[12], p[3];
  load_se3(g.x0[k] + (int64_t)g.bstride[k * 4 + 0] * b, X);
  load_n<T, 3>(g.x1[k] + (int64_t)g.bstride[k * 4 + 1] * b, p);
  const T f = (g.aux[k] + (int64_t)g.bstride[k * 4 + 2] * b)[0];
  const T* z = g.aux2[k] + (int64_t)g.bstride2[k * 3 + 0] * b;
  const T k1 = (g.aux3[k] + (int64_t)g.bstride2[k * 3 + 1] * b)[0];
  const T k2 = (g.aux4[k] + (int64_t)g.bstride2[k * 3 + 2] * b)[0];
  T q[3];
#pragma unroll
  for (int i = 0; i < 3; i++) q[i] = X[i * 4 + 3] + (X[i * 4 + 0] * p[0] + X[i * 4 + 1] * p[1] + X[i * 4 + 2] * p[2]);
  const T pr0 = -q[0] / q[2], pr1 = -q[1] / q[2];
  const T n = pr0 * pr0 + pr1 * pr1;
  const T pf = f * (T(1) + n * (k1 + n * k2));
  e[0] = (pr0 * pf - z[0]) * w[0];
  e[1] = (pr1 * pf - z[1]) * w[1];
  if (WITH_J) {
    const T dpf = f * (k1 + T(2) * n * k2);
    // J (3 x 9) = [R | -R hat(p) | R]
    T J[3][9];
#pragma unroll
    for (int i = 0; i < 3; i++) {
      const T r0 = X[i * 4 + 0], r1 = X[i * 4 + 1], r2 = X[i * 4 + 2];
      J[i][0] = r0; J[i][1] = r1; J[i][2] = r2;
      // -(R hat(p)): hat(p) = [[0,-p2,p1],[p2,0,-p0],[-p1,p0,0]]
      J[i][3] = -(r1 * p[2] - r2 * p[1]);
      J[i][4] = -(-r0 * p[2] + r2 * p[0]);
      J[i][5] = -(r0 * p[1] - r1 * p[0]);
      J[i][6] = r0; J[i][7] = r1; J[i][8] = r2;
    }
#pragma unroll
    for (int c = 0; c < 9; c++) {
      const T jz = J[2][c] / q[2];
      const T pj0 = (q[0] * jz - J[0][c]) / q[2];   // (N D'/D - N') / D
      const T pj1 = (q[1] * jz - J[1][c]) / q[2];
      const T nj = T(2) * (pr0 * pj0 + pr1 * pj1);
      const T o0 = (pj0 * pf + (T(2) * pr0 * (pr0 * pj0 + pr1 * pj1)) * dpf) * w[0];
      const T o1 = (pj1 * pf + (T(2) * pr1 * (pr0 * pj0 + pr1 * pj1)) * dpf) * w[1];
      (void)nj;
      if (c < 6) { Jc[0 * 6 + c] = o0; Jc[1 * 6 + c] = o1; }
      else { Jp[0 * 3 + (c - 6)] = o0; Jp[1 * 3 + (c - 6)] = o1; }
    }
  }
}

template <typename T>
__global__ void __launch_bounds__(128) linearize_reprojection_kernel(GroupDev<T> g, int64_t B, T* __restrict__ A_val, int64_t nnz,
                                                                     T* __restrict__ bvec, int64_t m) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (int64_t)g.K * B) return;
  const int k = (int)(t / B);
  const int64_t b = t - (int64_t)k * B;
  T w[2], e[2], Jc[12], Jp[6];
  const bool masked = load_weight<T, 2>(g, k, b, w);
  if (masked) {
    e[0] = e[1] = T(0);
#pragma unroll
    for (int i = 0; i < 12; i++) Jc[i] = T(0);
#pragma unroll
    for (int i = 0; i < 6; i++) Jp[i] = T(0);
  } else {
    reprojection_cost<T, true>(g, k, b, w, e, Jc, Jp);
    if (g.robust_kind != THB_ROBUST_NONE) {
      const T sc = robust_rescale(g, k, b, e[0] * e[0] + e[1] * e[1]);
      e[0] *= sc;
      e[1] *= sc;
#pragma unroll
      for (int i = 0; i < 12; i++) Jc[i] *= sc;
#pragma unroll
      for (int i = 0; i < 6; i++) Jp[i] *= sc;
    }
  }
  T* Arow = A_val + b * nnz + g.a_off[k];
  const int stride = g.a_stride[k];
  const int bp0 = g.bp[k * 2 + 0], bp1 = g.bp[k * 2 + 1];
#pragma unroll
  for (int r = 0; r < 2; r++) {
#pragma unroll
    for (int c = 0; c < 6; c++) Arow[r * stride + bp0 + c] = Jc[r * 6 + c];
#pragma unroll
    for (int c = 0; c < 3; c++) Arow[r * stride + bp1 + c] = Jp[r * 3 + c];
  }
  T* brow = bvec + b * m + g.row0[k];
  brow[0] = -e[0];
  brow[1] = -e[1];
}

template <typename T>
__global__ void __launch_bounds__(128) error_reprojection_kernel(GroupDev<T> g, int64_t B, T* __restrict__ partial) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int nchunks = (g.K + kErrCostsPerThread - 1) / kErrCostsPerThread;
  if (t >= (int64_t)nchunks * B) return;
  const int c = (int)(t / B);
  const int64_t b = t - (int64_t)c * B;
  T acc = T(0);
  const int k1 = min(g.K, (c + 1) * kErrCostsPerThread);
  for (int k = c * kErrCostsPerThread; k < k1; k++) {
    T w[2], e[2];
    if (load_weight<T, 2>(g, k, b, w)) continue;
    reprojection_cost<T, false>(g, k, b, w, e, nullptr, nullptr);
    const T x = e[0] * e[0] + e[1] * e[1];
    acc += (g.robust_kind != THB_ROBUST_NONE) ? robust_value(g, k, b, x, 2) : x;
  }
  partial[(int64_t)c * B + b] = acc * T(0.5);
}

// Difference on Vector/Point: e = (x - target) * w ; J = I * w   (geometry/vector.py local/jacobians)
template <typename T>
__global__ void linearize_vector_kernel(GroupDev<T> g, int64_t B, T* __restrict__ A_val, int64_t nnz,
                                        T* __restrict__ bvec, int64_t m) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (int64_t)g.K * B) return;
  const int k = (int)(t / B);
  const int64_t b = t - (int64_t)k * B;
  const int d = g.dim;
  const T* x = g.x0[k] + (int64_t)g.bstride[k * 4 + 0] * b;
  const T* tg = g.aux[k] + (int64_t)g.bstride[k * 4 + 2] * b;
  const T* wp = g.w[k] + (int64_t)g.bstride[k * 4 + 3] * b;
  T* Arow = A_val + b * nnz + g.a_off[k];
  const int stride = g.a_stride[k];
  const int bp0 = g.bp[k * 2 + 0];
  T* brow = bvec + b * m + g.row0[k];
  for (int r = 0; r < d; r++) {
    const T w = (g.weight_kind == THB_WEIGHT_SCALE) ? wp[0] : wp[r];
    for (int c = 0; c < d; c++) Arow[r * stride + bp0 + c] = (r == c) ? w : T(0);
    brow[r] = -((x[r] - tg[r]) * w);
  }
}

template <typename T, int KIND>
__global__ void __launch_bounds__(128) error_kernel(GroupDev<T> g, int64_t B, T* __restrict__ partial) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int nchunks = (g.K + kErrCostsPerThread - 1) / kErrCostsPerThread;
  if (t >= (int64_t)nchunks * B) return;
  const int c = (int)(t / B);
  const int64_t b = t - (int64_t)c * B;
  constexpr int DIM = (KIND == THB_COST_BETWEEN_SE3 || KIND == THB_COST_LOCAL_SE3) ? 6 : 3;
  constexpr bool BETWEEN = (KIND == THB_COST_BETWEEN_SE3 || KIND == THB_COST_BETWEEN_SO3 || KIND == THB_COST_BETWEEN_SE2);
  constexpr bool IS_SE2 = (KIND == THB_COST_BETWEEN_SE2 || KIND == THB_COST_LOCAL_SE2);
  T acc = T(0);
  const int k1 = min(g.K, (c + 1) * kErrCostsPerThread);
  for (int k = c * kErrCostsPerThread; k < k1; k++) {
    T w[DIM], e[DIM];
    const bool masked = load_weight<T, DIM>(g, k, b, w);
    if (masked) continue;
    if (DIM == 6) se3_cost<T, false, BETWEEN>(g, k, b, w, e, nullptr, nullptr);
    else if (IS_SE2) se2_cost<T, false, BETWEEN>(g, k, b, w, e, nullptr, nullptr);
    else so3_cost<T, false, BETWEEN>(g, k, b, w, e, nullptr, nullptr);
    T x = T(0);
#pragma unroll
    for (int r = 0; r < DIM; r++) x += e[r] * e[r];
    acc += (g.robust_kind != THB_ROBUST_NONE) ? robust_value(g, k, b, x, DIM) : x;
  }
  partial[(int64_t)c * B + b] = acc * T(0.5);
}

template <typename T> __global__ void error_vector_kernel(GroupDev<T> g, int64_t B, T* __restrict__ partial) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int nchunks = (g.K + kErrCostsPerThread - 1) / kErrCostsPerThread;
  if (t >= (int64_t)nchunks * B) return;
  const int c = (int)(t / B);
  const int64_t b = t - (int64_t)c * B;
  T acc = T(0);
  const int k1 = min(g.K, (c + 1) * kErrCostsPerThread);
  for (int k = c * kErrCostsPerThread; k < k1; k++) {
    const T* x = g.x0[k] + (int64_t)g.bstride[k * 4 + 0] * b;
    const T* tg = g.aux[k] + (int64_t)g.bstride[k * 4 + 2] * b;
    const T* wp = g.w[k] + (int64_t)g.bstride[k * 4 + 3] * b;
    for (int r = 0; r < g.dim; r++) {
      const T w = (g.weight_kind == THB_WEIGHT_SCALE) ? wp[0] : wp[r];
      const T e = (x[r] - tg[r]) * w;
      acc += e * e;
    }
  }
  partial[(int64_t)c * B + b] = acc * T(0.5);
}

template <typename T> __global__ void error_reduce_kernel(const T* __restrict__ partial, int nchunks, int64_t B, T* __restrict__ err) {
  const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  T s = T(0);
  for (int c = 0; c < nchunks; c++) s += partial[(int64_t)c * B + b];
  err[b] = s;
}

// ------------------------------------------------------------------------------------------------
// 2-D motion planning (theseus/embodied/collision/collision.py, signed_distance_field.py:163-241,
// theseus/embodied/motionmodel/double_integrator.py:16-175).

// Collision2D: bilinear signed distance d of the pose's xy in the grid sdf_data [Bs, rows, cols] (cell (r, c) at
// origin + (c, r) * cell_size; floor / ceil indices clamped, weights not; 0 and zero gradient outside the grid),
// e = max(eps - d, 0) * w, J = -grad d (times [R 0] for SE2) * w, zeroed where d > eps.  DOF = 2 (Point2) or 3 (SE2).
template <typename T, bool IS_SE2, bool WITH_J>
__device__ __forceinline__ void collision2d_cost(const GroupDev<T>& g, int k, int64_t b, T w, T* e, T* J) {
  const T* x = g.x0[k] + (int64_t)g.bstride[k * 4 + 0] * b;
  const T* org = g.aux[k] + (int64_t)g.bstride[k * 4 + 2] * b;
  const T* data = g.aux2[k] + (int64_t)g.bstride2[k * 3 + 0] * b;
  const T cell = (g.aux3[k] + (int64_t)g.bstride2[k * 3 + 1] * b)[0];
  const T eps = (g.aux4[k] + (int64_t)g.bstride2[k * 3 + 2] * b)[0];
  const int rows = g.sdf_rows, cols = g.sdf_cols;
  const T px = x[0], py = x[1], ox = org[0], oy = org[1];
  const bool oob = (px < ox) || (px > ox + (T(cols) - T(1)) * cell) || (py < oy) || (py > oy + (T(rows) - T(1)) * cell);
  const T col = (px - ox) / cell, row = (py - oy) / cell;
  const T lr = floor(row), lc = floor(col);
  const T hr = lr + T(1), hc = lc + T(1);
  // float clamp first so that the integer conversion is defined for any input; the index clamp is the reference's
  auto idx = [](T v, int n) -> int64_t {
    const T vc = v < T(-1) ? T(-1) : (v > T(n) ? T(n) : v);
    const int64_t i = (int64_t)vc;
    return i < 0 ? 0 : (i > n - 1 ? n - 1 : i);
  };
  const int64_t lri = idx(lr, rows), hri = idx(hr, rows), lci = idx(lc, cols), hci = idx(hc, cols);
  const T s_ll = data[lri * cols + lci], s_hl = data[hri * cols + lci], s_lh = data[lri * cols + hci], s_hh = data[hri * cols + hci];
  const T hrd = hr - row, hcd = hc - col, lrd = row - lr, lcd = col - lc;
  T dist = hrd * hcd * s_ll + lrd * hcd * s_hl + hrd * lcd * s_lh + lrd * lcd * s_hh;
  if (oob) dist = T(0);
  const T err = eps - dist;
  e[0] = (err > T(0) ? err : T(0)) * w;
  if (WITH_J) {
    T gx = (hrd * (s_lh - s_ll) + lrd * (s_hh - s_hl)) / cell;
    T gy = (hcd * (s_hl - s_ll) + lcd * (s_hh - s_lh)) / cell;
    if (oob || dist > eps) { gx = T(0); gy = T(0); }
    if (IS_SE2) {  // d xy / d tangent = [R 0] (SE2.xy Jacobian)
      const T c = x[2], s = x[3];
      J[0] = -(gx * c + gy * s) * w;
      J[1] = -(-gx * s + gy * c) * w;
      J[2] = T(0) * w;
    } else {
      J[0] = -gx * w;
      J[1] = -gy * w;
    }
  }
}

template <typename T> __device__ __forceinline__ T weight_scalar(const GroupDev<T>& g, int k, int64_t b) {
  return (g.w[k] + (int64_t)g.bstride[k * 4 + 3] * b)[0];
}

template <typename T, bool IS_SE2>
__global__ void __launch_bounds__(128) linearize_collision2d_kernel(GroupDev<T> g, int64_t B, T* __restrict__ A_val, int64_t nnz,
                                                                    T* __restrict__ bvec, int64_t m) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (int64_t)g.K * B) return;
  const int k = (int)(t / B);
  const int64_t b = t - (int64_t)k * B;
  constexpr int DOF = IS_SE2 ? 3 : 2;
  const T w = weight_scalar(g, k, b);      // dim 1: scale and diagonal weights are one value
  T e[1], J[DOF];
  if (w == T(0)) {
    e[0] = T(0);
#pragma unroll
    for (int c = 0; c < DOF; c++) J[c] = T(0);
  } else {
    collision2d_cost<T, IS_SE2, true>(g, k, b, w, e, J);
  }
  T* Arow = A_val + b * nnz + g.a_off[k] + g.bp[k * 2 + 0];
#pragma unroll
  for (int c = 0; c < DOF; c++) Arow[c] = J[c];
  bvec[b * m + g.row0[k]] = -e[0];
}

template <typename T, bool IS_SE2>
__global__ void __launch_bounds__(128) error_collision2d_kernel(GroupDev<T> g, int64_t B, T* __restrict__ partial) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int nchunks = (g.K + kErrCostsPerThread - 1) / kErrCostsPerThread;
  if (t >= (int64_t)nchunks * B) return;
  const int c = (int)(t / B);
  const int64_t b = t - (int64_t)c * B;
  T acc = T(0);
  const int k1 = min(g.K, (c + 1) * kErrCostsPerThread);
  for (int k = c * kErrCostsPerThread; k < k1; k++) {
    const T w = weight_scalar(g, k, b);
    if (w == T(0)) continue;
    T e[1];
    collision2d_cost<T, IS_SE2, false>(g, k, b, w, e, nullptr);
    acc += e[0] * e[0];
  }
  partial[(int64_t)c * B + b] = acc * T(0.5);
}

// Weight of a DOUBLE_INTEGRATOR cost function as a (2D x 2D) matrix Wm applied from the left (e <- Wm e, J <- Wm J):
// scale / diagonal: diag(w); GP: U = (chol(M) (x) chol(Qc_inv^T))^T, U[(q,j),(p,i)] = Lm[p][q] Lq[i][j] (row (p,i) = p D + i).
// Returns true if the weight is all zero (masked cost function, like load_weight).
template <typename T, int D>
__device__ __forceinline__ bool integrator_weight(const GroupDev<T>& g, int k, int64_t b, T* Wm) {
  constexpr int N = 2 * D;
#pragma unroll
  for (int i = 0; i < N * N; i++) Wm[i] = T(0);
  const T* wp = g.w[k] + (int64_t)g.bstride[k * 4 + 3] * b;
  if (g.weight_kind == THB_WEIGHT_GP) {
    const T dt = (g.aux2[k] + (int64_t)g.bstride2[k * 3 + 0] * b)[0];
    const T idt = T(1) / dt;
    const T lm00 = t_sqrt(T(12) * idt * idt * idt);
    const T lm10 = (T(-6) * idt * idt) / lm00;
    const T lm11 = t_sqrt(T(4) * idt - lm10 * lm10);
    const T Lm[2][2] = {{lm00, T(0)}, {lm10, lm11}};
    T Lq[D][D];
#pragma unroll
    for (int j = 0; j < D; j++) {
      T s = wp[j * D + j];
#pragma unroll
      for (int q = 0; q < j; q++) s -= Lq[j][q] * Lq[j][q];
      const T ljj = t_sqrt(s);
      Lq[j][j] = ljj;
#pragma unroll
      for (int i = j + 1; i < D; i++) {
        T a = wp[j * D + i];          // (Qc_inv^T)[i][j]
#pragma unroll
        for (int q = 0; q < j; q++) a -= Lq[i][q] * Lq[j][q];
        Lq[i][j] = a / ljj;
      }
#pragma unroll
      for (int i = 0; i < j; i++) Lq[i][j] = T(0);
    }
#pragma unroll
    for (int p = 0; p < 2; p++)
#pragma unroll
      for (int q = 0; q < 2; q++)
#pragma unroll
        for (int i = 0; i < D; i++)
#pragma unroll
          for (int j = 0; j < D; j++) Wm[(q * D + j) * N + (p * D + i)] = Lm[p][q] * Lq[i][j];
    return false;
  }
  bool all_zero = true;
#pragma unroll
  for (int r = 0; r < N; r++) {
    const T v = (g.weight_kind == THB_WEIGHT_SCALE) ? wp[0] : wp[r];
    Wm[r * N + r] = v;
    all_zero = all_zero && (v == T(0));
  }
  return all_zero;
}

// Unweighted error [2D] and the pose Jacobians (top D x D blocks; the rest of the four blocks is constant) of
// e = [pose1.local(pose2) - dt vel1 ; vel2 - vel1].  SE2: local = log(pose1^-1 pose2), J1 = -dlog Ad(D^-1), J2 = dlog
// (= Between with an identity measurement); Vector: local = pose2 - pose1, J1 = -I, J2 = I.
template <typename T, int D, bool IS_SE2, bool WITH_J>
__device__ __forceinline__ T integrator_error(const GroupDev<T>& g, int k, int64_t b, T* e, T* Jp1, T* Jp2) {
  const T* p1 = g.x0[k] + (int64_t)g.bstride[k * 4 + 0] * b;
  const T* v1 = g.x1[k] + (int64_t)g.bstride[k * 4 + 1] * b;
  const T* p2 = g.x2[k] + (int64_t)g.bstride3[k * 2 + 0] * b;
  const T* v2 = g.x3[k] + (int64_t)g.bstride3[k * 2 + 1] * b;
  const T dt = (g.aux[k] + (int64_t)g.bstride[k * 4 + 2] * b)[0];
  T loc[D];
  if (IS_SE2) {
    T X0[4], X1[4], Dm[4], Jl[9];
    load_n<T, 4>(p1, X0);
    load_n<T, 4>(p2, X1);
    se2_between(X0, X1, Dm);
    se2_log_jlog<T, WITH_J>(Dm, loc, Jl);
    if (WITH_J) {
      T Di[4], Ad[9];
      se2_inverse(Dm, Di);
      se2_adjoint(Di, Ad);
#pragma unroll
      for (int r = 0; r < 3; r++)
#pragma unroll
        for (int c = 0; c < 3; c++) {
          Jp1[r * D + c] = -(Jl[r * 3 + 0] * Ad[0 * 3 + c] + Jl[r * 3 + 1] * Ad[1 * 3 + c] + Jl[r * 3 + 2] * Ad[2 * 3 + c]);
          Jp2[r * D + c] = Jl[r * 3 + c];
        }
    }
  } else {
#pragma unroll
    for (int i = 0; i < D; i++) loc[i] = p2[i] - p1[i];
    if (WITH_J) {
#pragma unroll
      for (int r = 0; r < D; r++)
#pragma unroll
        for (int c = 0; c < D; c++) {
          Jp1[r * D + c] = (r == c) ? T(-1) : T(0);
          Jp2[r * D + c] = (r == c) ? T(1) : T(0);
        }
    }
  }
#pragma unroll
  for (int i = 0; i < D; i++) {
    const T a = v1[i];
    e[i] = loc[i] - dt * a;
    e[D + i] = v2[i] - a;
  }
  return dt;
}

template <typename T, int D, bool IS_SE2>
__global__ void __launch_bounds__(128) linearize_integrator_kernel(GroupDev<T> g, int64_t B, T* __restrict__ A_val, int64_t nnz,
                                                                   T* __restrict__ bvec, int64_t m) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (int64_t)g.K * B) return;
  const int k = (int)(t / B);
  const int64_t b = t - (int64_t)k * B;
  constexpr int N = 2 * D;
  T Wm[N * N], e[N], Jp1[D * D], Jp2[D * D];
  const bool masked = integrator_weight<T, D>(g, k, b, Wm);
  const T dt = integrator_error<T, D, IS_SE2, true>(g, k, b, e, Jp1, Jp2);
  T* Arow = A_val + b * nnz + g.a_off[k];
  const int stride = g.a_stride[k];
  const int bp0 = g.bp[k * 4 + 0], bp1 = g.bp[k * 4 + 1], bp2 = g.bp[k * 4 + 2], bp3 = g.bp[k * 4 + 3];
  T* brow = bvec + b * m + g.row0[k];
  // unweighted blocks, column c of variable slot: pose1 [Jp1; 0], vel1 [-dt I; -I], pose2 [Jp2; 0], vel2 [0; I]
#pragma unroll
  for (int r = 0; r < N; r++) {
    T o0[D], o1[D], o2[D], o3[D];
    T we = T(0);
#pragma unroll
    for (int c = 0; c < D; c++) { o0[c] = T(0); o1[c] = T(0); o2[c] = T(0); o3[c] = T(0); }
#pragma unroll
    for (int q = 0; q < N; q++) {
      const T wq = Wm[r * N + q];
      we += wq * e[q];
      if (q < D) {
#pragma unroll
        for (int c = 0; c < D; c++) {
          o0[c] += wq * Jp1[q * D + c];
          o2[c] += wq * Jp2[q * D + c];
        }
        o1[q] += wq * (-dt);
      } else {
        o1[q - D] -= wq;
        o3[q - D] += wq;
      }
    }
    if (masked) {
      we = T(0);
#pragma unroll
      for (int c = 0; c < D; c++) { o0[c] = T(0); o1[c] = T(0); o2[c] = T(0); o3[c] = T(0); }
    }
#pragma unroll
    for (int c = 0; c < D; c++) {
      Arow[r * stride + bp0 + c] = o0[c];
      Arow[r * stride + bp1 + c] = o1[c];
      Arow[r * stride + bp2 + c] = o2[c];
      Arow[r * stride + bp3 + c] = o3[c];
    }
    brow[r] = -we;
  }
}

template <typename T, int D, bool IS_SE2>
__global__ void __launch_bounds__(128) error_integrator_kernel(GroupDev<T> g, int64_t B, T* __restrict__ partial) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int nchunks = (g.K + kErrCostsPerThread - 1) / kErrCostsPerThread;
  if (t >= (int64_t)nchunks * B) return;
  const int c = (int)(t / B);
  const int64_t b = t - (int64_t)c * B;
  constexpr int N = 2 * D;
  T acc = T(0);
  const int k1 = min(g.K, (c + 1) * kErrCostsPerThread);
  for (int k = c * kErrCostsPerThread; k < k1; k++) {
    T Wm[N * N], e[N];
    if (integrator_weight<T, D>(g, k, b, Wm)) continue;
    integrator_error<T, D, IS_SE2, false>(g, k, b, e, nullptr, nullptr);
#pragma unroll
    for (int r = 0; r < N; r++) {
      T we = T(0);
#pragma unroll
      for (int q = 0; q < N; q++) we += Wm[r * N + q] * e[q];
      acc += we * we;
    }
  }
  partial[(int64_t)c * B + b] = acc * T(0.5);
}

// ------------------------------------------------------------------------------------------------
template <typename T> struct VarDev {
  int N;
  const T* const* x;
  T* const* out;
  const int32_t* kind;
  const int32_t* col;
  const int32_t* dof;
};
template <typename T> static VarDev<T> to_dev(const thb_var_table* v) {
  VarDev<T> d;
  d.N = v->N;
  d.x = reinterpret_cast<const T* const*>(v->x);
  d.out = reinterpret_cast<T* const*>(v->out);
  d.kind = v->kind;
  d.col = v->col;
  d.dof = v->dof;
  return d;
}

template <typename T>
__global__ void __launch_bounds__(128) retract_kernel(VarDev<T> v, int64_t B, const T* __restrict__ delta, int64_t n, T step,
                                                      const uint8_t* __restrict__ ignore) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (int64_t)v.N * B) return;
  const int i = (int)(t / B);
  const int64_t b = t - (int64_t)i * B;
  const int kind = v.kind[i];
  const bool keep = ignore != nullptr && ignore[b] != 0;
  const T* d = delta + b * n + v.col[i];
  if (kind == THB_VAR_SE3) {
    const T* xp = v.x[i] + b * 12;
    T* op = v.out[i] + b * 12;
    T X[12], O[12];
    load_se3(xp, X);
    if (keep) {
#pragma unroll
      for (int q = 0; q < 12; q++) O[q] = X[q];
    } else {
      T xi[6], G[12];
#pragma unroll
      for (int q = 0; q < 6; q++) xi[q] = d[q] * step;
      se3_exp(xi, G);
      se3_compose(X, G, O);
    }
#pragma unroll
    for (int q = 0; q < 12; q++) op[q] = O[q];
  } else if (kind == THB_VAR_SO3) {
    const T* xp = v.x[i] + b * 9;
    T* op = v.out[i] + b * 9;
    T X[9], O[9];
    load_n<T, 9>(xp, X);
    if (keep) {
#pragma unroll
      for (int q = 0; q < 9; q++) O[q] = X[q];
    } else {
      T w[3], R[9];
#pragma unroll
      for (int q = 0; q < 3; q++) w[q] = d[q] * step;
      so3_exp<T, 3>(w, R);
      mat3_mul(X, R, O);
    }
#pragma unroll
    for (int q = 0; q < 9; q++) op[q] = O[q];
  } else if (kind == THB_VAR_SE2) {
    const T* xp = v.x[i] + b * 4;
    T* op = v.out[i] + b * 4;
    T X[4], O[4];
    load_n<T, 4>(xp, X);
    if (keep) {
#pragma unroll
      for (int q = 0; q < 4; q++) O[q] = X[q];
    } else {
      T xi[3], G[4];
#pragma unroll
      for (int q = 0; q < 3; q++) xi[q] = d[q] * step;
      se2_exp(xi, G);
      se2_compose(X, G, O);
    }
#pragma unroll
    for (int q = 0; q < 4; q++) op[q] = O[q];
  } else if (kind == THB_VAR_SO2) {  // storage [cos, sin], tangent theta: X * exp(theta) (geometry/so2.py:167-186 exp_map, :224-230 compose)
    const T* xp = v.x[i] + b * 2;
    T* op = v.out[i] + b * 2;
    const T c0 = xp[0], s0 = xp[1];
    if (keep) {
      op[0] = c0;
      op[1] = s0;
    } else {
      T s1, c1;
      t_sincos(d[0] * step, &s1, &c1);
      op[0] = c0 * c1 - s0 * s1;
      op[1] = s0 * c1 + c0 * s1;
    }
  } else {  // Vector / Point: x + delta
    const int dof = v.dof[i];
    const T* xp = v.x[i] + b * dof;
    T* op = v.out[i] + b * dof;
    for (int q = 0; q < dof; q++) op[q] = keep ? xp[q] : (xp[q] + d[q] * step);
  }
}

template <typename T>
__global__ void commit_kernel(VarDev<T> v, int64_t B, const uint8_t* __restrict__ keep_old) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (int64_t)v.N * B) return;
  const int i = (int)(t / B);
  const int64_t b = t - (int64_t)i * B;
  if (keep_old != nullptr && keep_old[b]) return;
  const int kind = v.kind[i];
  const int sz = (kind == THB_VAR_SE3) ? 12 : ((kind == THB_VAR_SO3) ? 9 : ((kind == THB_VAR_SE2) ? 4 : ((kind == THB_VAR_SO2) ? 2 : v.dof[i])));
  const T* src = v.out[i] + b * sz;
  T* dst = const_cast<T*>(v.x[i]) + b * sz;
  for (int q = 0; q < sz; q++) dst[q] = src[q];
}

// ------------------------------------------------------------------------------------------------
// LM control: one CTA per batch item reduces den over n columns (levenberg_marquardt.py:172-201); partial sums per thread, per warp
// (shuffles) and per CTA (warp order) -- a fixed order, so the accept decision is reproducible.  (One WARP per item left 512 warps to
// stream 3 x 61 MB at C5 B=512: 0.28 ms.)
constexpr int kLmCtrlThreads = 256;
template <typename T>
__global__ void __launch_bounds__(kLmCtrlThreads) lm_control_kernel(const T* __restrict__ delta, const T* __restrict__ Atb, const T* __restrict__ diag, int64_t B,
                                  int64_t n, T step, const T* __restrict__ err_prev, const T* __restrict__ err_new,
                                  T* __restrict__ lam, int ellipsoidal, T accept, T down, T up, uint8_t* __restrict__ reject,
                                  T* __restrict__ err_out, int32_t* __restrict__ stats) {
  __shared__ T part[kLmCtrlThreads / 32];
  const int tid = threadIdx.x, lane = tid & 31;
  const int64_t b = blockIdx.x;
  if (b >= B) return;
  const T l = lam[b];
  T acc = T(0);
#pragma unroll 4
  for (int64_t j = tid; j < n; j += kLmCtrlThreads) {
    const T d = delta[b * n + j] * step;
    const T le = ellipsoidal ? (l * diag[b * n + j]) : l;
    acc += d * (le * d + Atb[b * n + j]);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if (lane == 0) part[tid >> 5] = acc;
  __syncthreads();
  if (tid == 0) {
    T sum = T(0);
#pragma unroll
    for (int q = 0; q < kLmCtrlThreads / 32; q++) sum += part[q];
    const T den = sum / T(2);
    const T rho = (err_prev[b] - err_new[b]) / den;
    const bool rej = rho <= accept;  // NaN compares false -> accepted, like torch's `rho <= damping_accept`
    T nl = rej ? (l * up) : (l / down);
    nl = (nl < T(1e-7)) ? T(1e-7) : ((nl > T(1e7)) ? T(1e7) : nl);
    lam[b] = nl;
    reject[b] = rej ? 1 : 0;
    err_out[b] = rej ? err_prev[b] : err_new[b];
    if (rej) atomicAdd(&stats[0], 1);
  }
}

// ------------------------------------------------------------------------------------------------
// stand-alone Lie kernels
template <typename T> __global__ void k_se3_exp(const T* __restrict__ xi, T* __restrict__ G, int64_t N) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  T x[6], g[12];
  load_n<T, 6>(xi + i * 6, x);
  se3_exp(x, g);
#pragma unroll
  for (int q = 0; q < 12; q++) G[i * 12 + q] = g[q];
}
template <typename T> __global__ void k_se3_log(const T* __restrict__ G, T* __restrict__ xi, T* __restrict__ J, int64_t N) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  T g[12], x[6], jl[36];
  load_se3(G + i * 12, g);
  if (J != nullptr) {
    se3_log_jlog<T, true>(g, x, jl);
#pragma unroll
    for (int q = 0; q < 36; q++) J[i * 36 + q] = jl[q];
  } else {
    se3_log_jlog<T, false>(g, x, jl);
  }
#pragma unroll
  for (int q = 0; q < 6; q++) xi[i * 6 + q] = x[q];
}
template <typename T> __global__ void k_se3_adjoint(const T* __restrict__ G, T* __restrict__ A, int64_t N) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  T g[12], a[36];
  load_se3(G + i * 12, g);
  se3_adjoint(g, a);
#pragma unroll
  for (int q = 0; q < 36; q++) A[i * 36 + q] = a[q];
}
template <typename T> __global__ void k_se3_inverse(const T* __restrict__ G, T* __restrict__ O, int64_t N) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  T g[12], o[12];
  load_se3(G + i * 12, g);
  se3_inverse(g, o);
#pragma unroll
  for (int q = 0; q < 12; q++) O[i * 12 + q] = o[q];
}
template <typename T> __global__ void k_se3_compose(const T* __restrict__ G0, const T* __restrict__ G1, T* __restrict__ O, int64_t N) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  T a[12], b[12], o[12];
  load_se3(G0 + i * 12, a);
  load_se3(G1 + i * 12, b);
  se3_compose(a, b, o);
#pragma unroll
  for (int q = 0; q < 12; q++) O[i * 12 + q] = o[q];
}

// ------------------------------------------------------------------------------------------------
static inline unsigned grid_for(int64_t total, int threads) { return (unsigned)((total + threads - 1) / threads); }

// Argument checks of the motion-planning kinds: which tables must be present, which weights each kind takes.
static int check_collision2d(const thb_cost_group* g) {
  if (g->aux2 == nullptr || g->aux3 == nullptr || g->aux4 == nullptr || g->bstride2 == nullptr) return THB_ERR_BAD_ARG;
  if (g->sdf_rows < 1 || g->sdf_cols < 1 || g->dim != 1) return THB_ERR_BAD_ARG;
  if (g->weight_kind != THB_WEIGHT_SCALE && g->weight_kind != THB_WEIGHT_DIAGONAL) return THB_ERR_UNSUPPORTED;
  if (g->robust_kind != THB_ROBUST_NONE) return THB_ERR_UNSUPPORTED;
  return THB_OK;
}
static int check_integrator(const thb_cost_group* g) {
  if (g->x2 == nullptr || g->x3 == nullptr || g->bstride3 == nullptr) return THB_ERR_BAD_ARG;
  if (g->kind == THB_COST_DOUBLE_INTEGRATOR_SE2 ? g->dim != 6 : (g->dim != 4 && g->dim != 6)) return THB_ERR_BAD_ARG;
  if (g->weight_kind == THB_WEIGHT_GP) {
    if (g->aux2 == nullptr || g->bstride2 == nullptr) return THB_ERR_BAD_ARG;
  } else if (g->weight_kind != THB_WEIGHT_SCALE && g->weight_kind != THB_WEIGHT_DIAGONAL) {
    return THB_ERR_UNSUPPORTED;
  }
  if (g->robust_kind != THB_ROBUST_NONE) return THB_ERR_UNSUPPORTED;
  return THB_OK;
}

template <typename T>
static int linearize_group(const thb_cost_group* g, int64_t B, T* A_val, int64_t nnz, T* b, int64_t m, thb_stream_t s) {
  if (g == nullptr || g->K < 0 || B < 0) return THB_ERR_BAD_ARG;
  if (g->K == 0 || B == 0) return THB_OK;
  GroupDev<T> d = to_dev<T>(g);
  const int64_t total = (int64_t)g->K * B;
  const unsigned grid = grid_for(total, 128);
  cudaStream_t cs = thb_cs(s);
#define THB_LIN_LAUNCH(KIND, NV)                                                                                              \
  do {                                                                                                                      \
    const size_t smem_ = (size_t)4 * 32 * ((NV) + 1) * sizeof(T);                                                           \
    static bool attr_ = false;                                                                                              \
    if (!attr_ && smem_ > 48 * 1024) {                                                                                      \
      THB_CUDA(cudaFuncSetAttribute(linearize_kernel<T, KIND>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_));   \
      attr_ = true;                                                                                                         \
    }                                                                                                                       \
    linearize_kernel<T, KIND><<<grid, 128, smem_, cs>>>(d, B, A_val, nnz, b, m);                                            \
  } while (0)
  switch (g->kind) {
    case THB_COST_BETWEEN_SE3: THB_LIN_LAUNCH(THB_COST_BETWEEN_SE3, 72); break;
    case THB_COST_LOCAL_SE3: THB_LIN_LAUNCH(THB_COST_LOCAL_SE3, 36); break;
    case THB_COST_BETWEEN_SO3: THB_LIN_LAUNCH(THB_COST_BETWEEN_SO3, 18); break;
    case THB_COST_LOCAL_SO3: THB_LIN_LAUNCH(THB_COST_LOCAL_SO3, 9); break;
    case THB_COST_BETWEEN_SE2: THB_LIN_LAUNCH(THB_COST_BETWEEN_SE2, 18); break;
    case THB_COST_LOCAL_SE2: THB_LIN_LAUNCH(THB_COST_LOCAL_SE2, 9); break;
    case THB_COST_LOCAL_VECTOR: linearize_vector_kernel<T><<<grid, 128, 0, cs>>>(d, B, A_val, nnz, b, m); break;
    case THB_COST_REPROJECTION:
      if (g->aux2 == nullptr || g->aux3 == nullptr || g->aux4 == nullptr || g->bstride2 == nullptr) return THB_ERR_BAD_ARG;
      linearize_reprojection_kernel<T><<<grid, 128, 0, cs>>>(d, B, A_val, nnz, b, m);
      break;
    case THB_COST_COLLISION2D_POINT2:
    case THB_COST_COLLISION2D_SE2: {
      const int rc = check_collision2d(g);
      if (rc != THB_OK) return rc;
      if (g->kind == THB_COST_COLLISION2D_SE2) linearize_collision2d_kernel<T, true><<<grid, 128, 0, cs>>>(d, B, A_val, nnz, b, m);
      else linearize_collision2d_kernel<T, false><<<grid, 128, 0, cs>>>(d, B, A_val, nnz, b, m);
      break;
    }
    case THB_COST_DOUBLE_INTEGRATOR_VECTOR:
    case THB_COST_DOUBLE_INTEGRATOR_SE2: {
      const int rc = check_integrator(g);
      if (rc != THB_OK) return rc;
      if (g->kind == THB_COST_DOUBLE_INTEGRATOR_SE2) linearize_integrator_kernel<T, 3, true><<<grid, 128, 0, cs>>>(d, B, A_val, nnz, b, m);
      else if (g->dim == 4) linearize_integrator_kernel<T, 2, false><<<grid, 128, 0, cs>>>(d, B, A_val, nnz, b, m);
      else linearize_integrator_kernel<T, 3, false><<<grid, 128, 0, cs>>>(d, B, A_val, nnz, b, m);
      break;
    }
    default: return THB_ERR_UNSUPPORTED;
  }
  THB_CHECK_LAUNCH();
  return THB_OK;
}

template <typename T> static int error_group(const thb_cost_group* g, int64_t B, T* partial, thb_stream_t s) {
  if (g == nullptr || g->K < 0 || B < 0) return THB_ERR_BAD_ARG;
  if (g->K == 0 || B == 0) return THB_OK;
  GroupDev<T> d = to_dev<T>(g);
  const int nchunks = (g->K + kErrCostsPerThread - 1) / kErrCostsPerThread;
  const unsigned grid = grid_for((int64_t)nchunks * B, 128);
  cudaStream_t cs = thb_cs(s);
  switch (g->kind) {
    case THB_COST_BETWEEN_SE3: error_kernel<T, THB_COST_BETWEEN_SE3><<<grid, 128, 0, cs>>>(d, B, partial); break;
    case THB_COST_LOCAL_SE3: error_kernel<T, THB_COST_LOCAL_SE3><<<grid, 128, 0, cs>>>(d, B, partial); break;
    case THB_COST_BETWEEN_SO3: error_kernel<T, THB_COST_BETWEEN_SO3><<<grid, 128, 0, cs>>>(d, B, partial); break;
    case THB_COST_LOCAL_SO3: error_kernel<T, THB_COST_LOCAL_SO3><<<grid, 128, 0, cs>>>(d, B, partial); break;
    case THB_COST_BETWEEN_SE2: error_kernel<T, THB_COST_BETWEEN_SE2><<<grid, 128, 0, cs>>>(d, B, partial); break;
    case THB_COST_LOCAL_SE2: error_kernel<T, THB_COST_LOCAL_SE2><<<grid, 128, 0, cs>>>(d, B, partial); break;
    case THB_COST_LOCAL_VECTOR: error_vector_kernel<T><<<grid, 128, 0, cs>>>(d, B, partial); break;
    case THB_COST_REPROJECTION:
      if (g->aux2 == nullptr || g->aux3 == nullptr || g->aux4 == nullptr || g->bstride2 == nullptr) return THB_ERR_BAD_ARG;
      error_reprojection_kernel<T><<<grid, 128, 0, cs>>>(d, B, partial);
      break;
    case THB_COST_COLLISION2D_POINT2:
    case THB_COST_COLLISION2D_SE2: {
      const int rc = check_collision2d(g);
      if (rc != THB_OK) return rc;
      if (g->kind == THB_COST_COLLISION2D_SE2) error_collision2d_kernel<T, true><<<grid, 128, 0, cs>>>(d, B, partial);
      else error_collision2d_kernel<T, false><<<grid, 128, 0, cs>>>(d, B, partial);
      break;
    }
    case THB_COST_DOUBLE_INTEGRATOR_VECTOR:
    case THB_COST_DOUBLE_INTEGRATOR_SE2: {
      const int rc = check_integrator(g);
      if (rc != THB_OK) return rc;
      if (g->kind == THB_COST_DOUBLE_INTEGRATOR_SE2) error_integrator_kernel<T, 3, true><<<grid, 128, 0, cs>>>(d, B, partial);
      else if (g->dim == 4) error_integrator_kernel<T, 2, false><<<grid, 128, 0, cs>>>(d, B, partial);
      else error_integrator_kernel<T, 3, false><<<grid, 128, 0, cs>>>(d, B, partial);
      break;
    }
    default: return THB_ERR_UNSUPPORTED;
  }
  THB_CHECK_LAUNCH();
  return THB_OK;
}

template <typename T>
static int retract_impl(const thb_var_table* vt, int64_t B, const T* delta, int64_t n, T step, const uint8_t* ignore, thb_stream_t s) {
  if (vt == nullptr || vt->N < 0 || B < 0) return THB_ERR_BAD_ARG;
  if (vt->N == 0 || B == 0) return THB_OK;
  retract_kernel<T><<<grid_for((int64_t)vt->N * B, 128), 128, 0, thb_cs(s)>>>(to_dev<T>(vt), B, delta, n, step, ignore);
  THB_CHECK_LAUNCH();
  return THB_OK;
}
template <typename T> static int commit_impl(const thb_var_table* vt, int64_t B, const uint8_t* keep_old, thb_stream_t s) {
  if (vt == nullptr || vt->N < 0 || B < 0) return THB_ERR_BAD_ARG;
  if (vt->N == 0 || B == 0) return THB_OK;
  commit_kernel<T><<<grid_for((int64_t)vt->N * B, 128), 128, 0, thb_cs(s)>>>(to_dev<T>(vt), B, keep_old);
  THB_CHECK_LAUNCH();
  return THB_OK;
}

}  // namespace thb

// ================================================================================================
template <typename T>
static int lm_control_impl(const T* delta, const T* Atb, const T* diag, int64_t B, int64_t n, T step, const T* err_prev, const T* err_new,
                           T* lam, int32_t ellipsoidal, T damping_accept, T down_ratio, T up_ratio, uint8_t* reject, T* err_out,
                           int32_t* stats, thb_stream_t s) {
  if (B <= 0) return THB_OK;
  if (ellipsoidal && diag == nullptr) return THB_ERR_BAD_ARG;
  THB_CUDA(cudaMemsetAsync(stats, 0, sizeof(int32_t) * 4, thb_cs(s)));
  const int threads = thb::kLmCtrlThreads;
  const unsigned grid = (unsigned)B;
  thb::lm_control_kernel<T><<<grid, threads, 0, thb_cs(s)>>>(delta, Atb, diag, B, n, step, err_prev, err_new, lam, ellipsoidal,
                                                              damping_accept, down_ratio, up_ratio, reject, err_out, stats);
  THB_CHECK_LAUNCH();
  return THB_OK;
}

extern "C" {

int64_t thb_launch_counter_ = 0;
int64_t thb_launch_count(void) { return thb_launch_counter_; }
int thb_version(void) { return 100; }
int thb_compiled_arch(void) {
#ifdef THB_ARCH
  return THB_ARCH;
#else
  return 100;
#endif
}

int thb_linearize_group_f64(const thb_cost_group* g, int64_t B, double* A_val, int64_t nnz, double* b, int64_t m, thb_stream_t s) {
  return thb::linearize_group<double>(g, B, A_val, nnz, b, m, s);
}
int thb_linearize_group_f32(const thb_cost_group* g, int64_t B, float* A_val, int64_t nnz, float* b, int64_t m, thb_stream_t s) {
  return thb::linearize_group<float>(g, B, A_val, nnz, b, m, s);
}
int thb_error_num_chunks(int32_t K) { return (K + thb::kErrCostsPerThread - 1) / thb::kErrCostsPerThread; }
int thb_error_group_f64(const thb_cost_group* g, int64_t B, double* partial, thb_stream_t s) { return thb::error_group<double>(g, B, partial, s); }
int thb_error_group_f32(const thb_cost_group* g, int64_t B, float* partial, thb_stream_t s) { return thb::error_group<float>(g, B, partial, s); }
int thb_error_reduce_f64(const double* partial, int32_t nchunks, int64_t B, double* err, thb_stream_t s) {
  if (B <= 0) return THB_OK;
  thb::error_reduce_kernel<double><<<thb::grid_for(B, 128), 128, 0, thb_cs(s)>>>(partial, nchunks, B, err);
  THB_CHECK_LAUNCH();
  return THB_OK;
}
int thb_error_reduce_f32(const float* partial, int32_t nchunks, int64_t B, float* err, thb_stream_t s) {
  if (B <= 0) return THB_OK;
  thb::error_reduce_kernel<float><<<thb::grid_for(B, 128), 128, 0, thb_cs(s)>>>(partial, nchunks, B, err);
  THB_CHECK_LAUNCH();
  return THB_OK;
}
int thb_retract_f64(const thb_var_table* vt, int64_t B, const double* delta, int64_t n, double step, const uint8_t* ignore, thb_stream_t s) {
  return thb::retract_impl<double>(vt, B, delta, n, step, ignore, s);
}
int thb_retract_f32(const thb_var_table* vt, int64_t B, const float* delta, int64_t n, float step, const uint8_t* ignore, thb_stream_t s) {
  return thb::retract_impl<float>(vt, B, delta, n, step, ignore, s);
}
int thb_commit_f64(const thb_var_table* vt, int64_t B, const uint8_t* keep_old, thb_stream_t s) { return thb::commit_impl<double>(vt, B, keep_old, s); }
int thb_commit_f32(const thb_var_table* vt, int64_t B, const uint8_t* keep_old, thb_stream_t s) { return thb::commit_impl<float>(vt, B, keep_old, s); }

int thb_lm_control_f64(const double* delta, const double* Atb, const double* diag, int64_t B, int64_t n, double step,
                       const double* err_prev, const double* err_new, double* lam, int32_t ellipsoidal, double damping_accept,
                       double down_ratio, double up_ratio, uint8_t* reject, double* err_out, int32_t* stats, thb_stream_t s) {
  return lm_control_impl<double>(delta, Atb, diag, B, n, step, err_prev, err_new, lam, ellipsoidal, damping_accept, down_ratio, up_ratio,
                                 reject, err_out, stats, s);
}
int thb_lm_control_f32(const float* delta, const float* Atb, const float* diag, int64_t B, int64_t n, float step, const float* err_prev,
                       const float* err_new, float* lam, int32_t ellipsoidal, float damping_accept, float down_ratio, float up_ratio,
                       uint8_t* reject, float* err_out, int32_t* stats, thb_stream_t s) {
  return lm_control_impl<float>(delta, Atb, diag, B, n, step, err_prev, err_new, lam, ellipsoidal, damping_accept, down_ratio, up_ratio,
                                reject, err_out, stats, s);
}

int thb_fill_zero(void* ptr, int64_t bytes, thb_stream_t s) {
  THB_CUDA(cudaMemsetAsync(ptr, 0, (size_t)bytes, thb_cs(s)));
  return THB_OK;
}

#define THB_LIE_ENTRY(NAME, T, KERNEL, ...)                                                        \
  {                                                                                                \
    if (N <= 0) return THB_OK;                                                                     \
    KERNEL<T><<<thb::grid_for(N, 128), 128, 0, thb_cs(s)>>>(__VA_ARGS__);                          \
    THB_CHECK_LAUNCH();                                                                            \
    return THB_OK;                                                                                 \
  }
int thb_se3_exp_f64(const double* t, double* g, int64_t N, thb_stream_t s) THB_LIE_ENTRY(exp, double, thb::k_se3_exp, t, g, N)
int thb_se3_log_f64(const double* g, double* t, double* j, int64_t N, thb_stream_t s) THB_LIE_ENTRY(log, double, thb::k_se3_log, g, t, j, N)
int thb_se3_adjoint_f64(const double* g, double* a, int64_t N, thb_stream_t s) THB_LIE_ENTRY(adj, double, thb::k_se3_adjoint, g, a, N)
int thb_se3_inverse_f64(const double* g, double* o, int64_t N, thb_stream_t s) THB_LIE_ENTRY(inv, double, thb::k_se3_inverse, g, o, N)
int thb_se3_compose_f64(const double* a, const double* b, double* o, int64_t N, thb_stream_t s) THB_LIE_ENTRY(cmp, double, thb::k_se3_compose, a, b, o, N)
int thb_se3_exp_f32(const float* t, float* g, int64_t N, thb_stream_t s) THB_LIE_ENTRY(exp, float, thb::k_se3_exp, t, g, N)
int thb_se3_log_f32(const float* g, float* t, float* j, int64_t N, thb_stream_t s) THB_LIE_ENTRY(log, float, thb::k_se3_log, g, t, j, N)
int thb_se3_adjoint_f32(const float* g, float* a, int64_t N, thb_stream_t s) THB_LIE_ENTRY(adj, float, thb::k_se3_adjoint, g, a, N)
int thb_se3_inverse_f32(const float* g, float* o, int64_t N, thb_stream_t s) THB_LIE_ENTRY(inv, float, thb::k_se3_inverse, g, o, N)
int thb_se3_compose_f32(const float* a, const float* b, float* o, int64_t N, thb_stream_t s) THB_LIE_ENTRY(cmp, float, thb::k_se3_compose, a, b, o, N)

}  // extern "C"

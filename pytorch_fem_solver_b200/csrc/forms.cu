// Element-local integration: generic quadrature sum, fused named forms, weak residual fwd/bwd.
// Reference: basis/abstract_basis.py:65-112 applied to the forms of
// examples/example_weak.py:64-81 and tests/test_assembly.py:68-84.
#include "common.cuh"

namespace tfem {

// ---------------------------------------------------------------------------------------------
// (f * dx).sum(-3) for an arbitrary materialised integrand (abstract_basis.py:72,83,104).
// Thread (e, c): consecutive threads walk the trailing (contiguous) axis -> coalesced.
// ---------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256) quad_reduce_kernel(int64_t total, int n_q, int m,
                                                          const T* __restrict__ f, int64_t stride_e,
                                                          int64_t stride_q, const T* __restrict__ dx,
                                                          T* __restrict__ local) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int64_t e = i / m;
  const int c = (int)(i - e * m);
  const T* fe = f + e * stride_e + c;
  const T* dxe = dx + e * n_q;
  T acc = T(0);
  for (int q = 0; q < n_q; ++q) acc += __ldg(fe + q * stride_q) * __ldg(dxe + q);
  local[i] = acc;
}

constexpr int kStagedBlock = 128;  // elements per block of the kernels that stage their streams through shared memory

template <typename T>
struct FracLite {
  const T* jac;  // [n_mesh,3,2]
  const T* inv;  // [n_mesh,2,3]
  const T* det;  // [n_mesh]
  const T* t;    // [n_mesh,3]
};

// Gradients of the three P1 shape functions of an element: the planar ones, or on a fracture the tangential
// 3-D ones g_i J_f^+ (fracture_basis.py:20-22).  Planar rows have gr[i][2] = 0.
template <typename T, bool FRAC>
__device__ __forceinline__ void p1_gradients(const TriGeom<T>& g, const FracLite<T>& frac, int mesh, T gr[3][3]) {
  gr[0][0] = -g.i00 - g.i10; gr[0][1] = -g.i01 - g.i11; gr[0][2] = T(0);
  gr[1][0] = g.i00;          gr[1][1] = g.i01;          gr[1][2] = T(0);
  gr[2][0] = g.i10;          gr[2][1] = g.i11;          gr[2][2] = T(0);
  if constexpr (FRAC) {
    T jinv[2][3];
#pragma unroll
    for (int a = 0; a < 2; ++a)
#pragma unroll
      for (int c = 0; c < 3; ++c) jinv[a][c] = __ldg(frac.inv + 6 * mesh + 3 * a + c);
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      const T a0 = gr[i][0], a1 = gr[i][1];
#pragma unroll
      for (int c = 0; c < 3; ++c) gr[i][c] = a0 * jinv[0][c] + a1 * jinv[1][c];
    }
  }
}

// Local load vector b_i = sum_q w_q det f(x_q) phi_i(q) over the first n_q points of `quad`, term for term the loop of
// local_forms_kernel.  `sampled(q)` gives f at point q of a TFEM_SRC_SAMPLED source; analytic sources are evaluated
// at the mapped point (on a fracture at its first two 3-D coordinates).  local_forms_kernel keeps its own copy of the
// loop: calling this helper there reorders the instructions of its fracture instantiations.
template <typename T, bool FRAC, typename Sampled>
__device__ __forceinline__ void p1_load(const QuadT<T>& quad, int n_q, T x0, T y0, T x1, T y1, T x2, T y2, T det, const SourceT<T>& src,
                                        const FracLite<T>& frac, int mesh, Sampled sampled, T& b0, T& b1, T& b2) {
  b0 = T(0), b1 = T(0), b2 = T(0);
  if (src.kind == TFEM_SRC_NONE) return;
  for (int q = 0; q < n_q; ++q) {
    T f;
    if (src.kind == TFEM_SRC_SAMPLED) {
      f = sampled(q);
    } else {
      T px = quad.l0[q] * x0 + quad.l1[q] * x1 + quad.l2[q] * x2;
      T py = quad.l0[q] * y0 + quad.l1[q] * y1 + quad.l2[q] * y2;
      if constexpr (FRAC) {  // analytic sources see the first two 3-D coordinates
        const T X = __ldg(frac.jac + 6 * mesh + 0) * px + __ldg(frac.jac + 6 * mesh + 1) * py + __ldg(frac.t + 3 * mesh);
        const T Y = __ldg(frac.jac + 6 * mesh + 2) * px + __ldg(frac.jac + 6 * mesh + 3) * py + __ldg(frac.t + 3 * mesh + 1);
        px = X;
        py = Y;
      }
      f = source_eval(src, px, py);
    }
    const T wf = quad.w[q] * det * f;
    b0 += wf * quad.l0[q];
    b1 += wf * quad.l1[q];
    b2 += wf * quad.l2[q];
  }
}

// ---------------------------------------------------------------------------------------------
// Fused local forms, one thread per element.
//   local_mat[e,i,j] = alpha * (grad phi_i . grad phi_j) * sum_q dx_q + beta * det * mref[i][j]
//   local_vec[e,i]   = sum_q dx_q f(x_q) phi_i(q)
// For fractures the tangential 3-D gradients satisfy (g_i J_f^+)(g_j J_f^+)^T; the reference
// computes exactly that product (fracture_basis.py:20-22), restated here with the 3-vectors.
// ---------------------------------------------------------------------------------------------
template <typename T, bool FRAC>
__global__ void __launch_bounds__(256) local_forms_kernel(
    int n_el, int n_el_per_mesh, int n_vert_per_mesh, const T* __restrict__ coords,
    const int32_t* __restrict__ conn, const QuadT<T> quad, const FracLite<T> frac, T alpha, T beta,
    const SourceT<T> src, const T* __restrict__ f_q, T* __restrict__ local_mat,
    T* __restrict__ local_vec) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n_el) return;
  const int mesh = e / n_el_per_mesh;
  const int64_t voff = (int64_t)mesh * n_vert_per_mesh;
  const int v0 = __ldg(conn + 3 * (int64_t)e + 0);
  const int v1 = __ldg(conn + 3 * (int64_t)e + 1);
  const int v2 = __ldg(conn + 3 * (int64_t)e + 2);
  T x0, y0, x1, y1, x2, y2;
  load_xy(coords, voff + v0, x0, y0);
  load_xy(coords, voff + v1, x1, y1);
  load_xy(coords, voff + v2, x2, y2);
  const TriGeom<T> g = tri_geom(x0, y0, x1, y1, x2, y2);
  T detf = T(1);
  if constexpr (FRAC) detf = __ldg(frac.det + mesh);
  const T det = g.det * detf;

  if (local_mat) {
    T gr[3][3];
    p1_gradients<T, FRAC>(g, frac, mesh, gr);
    const T area = quad.wsum * det;  // sum_q dx_q
    T* out = local_mat + 9 * (int64_t)e;
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
      for (int j = 0; j < 3; ++j) {
        T dot = gr[i][0] * gr[j][0] + gr[i][1] * gr[j][1];
        if constexpr (FRAC) dot += gr[i][2] * gr[j][2];
        out[3 * i + j] = alpha * (dot * area) + beta * (quad.mref[3 * i + j] * det);
      }
  }

  if (local_vec) {
    T b0 = T(0), b1 = T(0), b2 = T(0);
    if (src.kind != TFEM_SRC_NONE) {
      for (int q = 0; q < quad.n_q; ++q) {
        T f;
        if (src.kind == TFEM_SRC_SAMPLED) {
          f = __ldg(f_q + (int64_t)e * quad.n_q + q);
        } else {
          T px = quad.l0[q] * x0 + quad.l1[q] * x1 + quad.l2[q] * x2;
          T py = quad.l0[q] * y0 + quad.l1[q] * y1 + quad.l2[q] * y2;
          if constexpr (FRAC) {  // analytic sources see the first two 3-D coordinates
            const T X = __ldg(frac.jac + 6 * mesh + 0) * px + __ldg(frac.jac + 6 * mesh + 1) * py + __ldg(frac.t + 3 * mesh);
            const T Y = __ldg(frac.jac + 6 * mesh + 2) * px + __ldg(frac.jac + 6 * mesh + 3) * py + __ldg(frac.t + 3 * mesh + 1);
            px = X;
            py = Y;
          }
          f = source_eval(src, px, py);
        }
        const T wf = quad.w[q] * det * f;
        b0 += wf * quad.l0[q];
        b1 += wf * quad.l1[q];
        b2 += wf * quad.l2[q];
      }
    }
    T* out = local_vec + 3 * (int64_t)e;
    out[0] = b0;
    out[1] = b1;
    out[2] = b2;
  }
}

// ---------------------------------------------------------------------------------------------
// Fused local forms with coefficient fields sampled at the quadrature points:
//   local_mat[e,i,j] = (grad phi_i . grad phi_j) det sum_q w_q alpha_q + det sum_q w_q beta_q phi_i(q) phi_j(q)
//   local_vec[e,i]   = as local_forms_kernel
// alpha_q / beta_q [n_el, NQ] (NULL: the constant alpha / beta) and f_q are NQ-strided per element; the rows of a
// block of kStagedBlock elements are staged through shared memory with coalesced loads, as in the residual kernel.
// ---------------------------------------------------------------------------------------------
template <typename T, bool FRAC, int NQ>
__global__ void __launch_bounds__(kStagedBlock) weighted_local_forms_kernel(
    int n_el, int n_el_per_mesh, int n_vert_per_mesh, const T* __restrict__ coords,
    const int32_t* __restrict__ conn, const QuadT<T> quad, const FracLite<T> frac, T alpha, T beta,
    const SourceT<T> src, const T* __restrict__ f_q, const T* __restrict__ alpha_q, const T* __restrict__ beta_q,
    T* __restrict__ local_mat, T* __restrict__ local_vec) {
  constexpr int ROWP = NQ | 1;  // odd stride: conflict-free rows
  __shared__ T s_a[kStagedBlock * ROWP];
  __shared__ T s_b[kStagedBlock * ROWP];
  __shared__ T s_f[kStagedBlock * ROWP];
  const int e0 = blockIdx.x * kStagedBlock;
  const int count = min(kStagedBlock, n_el - e0);
  const bool field_a = local_mat && alpha_q, field_b = local_mat && beta_q;
  const bool sampled = local_vec && src.kind == TFEM_SRC_SAMPLED;
  for (int i = threadIdx.x; i < count * NQ; i += kStagedBlock) {
    const int at = (i / NQ) * ROWP + i % NQ;
    const int64_t from = (int64_t)e0 * NQ + i;
    if (field_a) s_a[at] = __ldg(alpha_q + from);
    if (field_b) s_b[at] = __ldg(beta_q + from);
    if (sampled) s_f[at] = __ldg(f_q + from);
  }
  __syncthreads();
  const int e = e0 + threadIdx.x;
  if (e >= n_el) return;
  const int mesh = e / n_el_per_mesh;
  const int64_t voff = (int64_t)mesh * n_vert_per_mesh;
  const int v0 = __ldg(conn + 3 * (int64_t)e + 0);
  const int v1 = __ldg(conn + 3 * (int64_t)e + 1);
  const int v2 = __ldg(conn + 3 * (int64_t)e + 2);
  T x0, y0, x1, y1, x2, y2;
  load_xy(coords, voff + v0, x0, y0);
  load_xy(coords, voff + v1, x1, y1);
  load_xy(coords, voff + v2, x2, y2);
  const TriGeom<T> g = tri_geom(x0, y0, x1, y1, x2, y2);
  T detf = T(1);
  if constexpr (FRAC) detf = __ldg(frac.det + mesh);
  const T det = g.det * detf;
  const int row = threadIdx.x * ROWP;

  if (local_mat) {
    T gr[3][3];
    p1_gradients<T, FRAC>(g, frac, mesh, gr);
    T wa = T(0);
    T m[6] = {};  // sum_q w_q beta_q phi_i phi_j: 00 11 22 01 12 02
#pragma unroll
    for (int q = 0; q < NQ; ++q) {
      wa += quad.w[q] * (field_a ? s_a[row + q] : alpha);
      const T wb = quad.w[q] * (field_b ? s_b[row + q] : beta);
      const T l0 = quad.l0[q], l1 = quad.l1[q], l2 = quad.l2[q];
      m[0] += wb * (l0 * l0);
      m[1] += wb * (l1 * l1);
      m[2] += wb * (l2 * l2);
      m[3] += wb * (l0 * l1);
      m[4] += wb * (l1 * l2);
      m[5] += wb * (l0 * l2);
    }
    const T stiff = wa * det;
    const T mass[9] = {m[0], m[3], m[5], m[3], m[1], m[4], m[5], m[4], m[2]};
    T* out = local_mat + 9 * (int64_t)e;
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
      for (int j = 0; j < 3; ++j) {
        T dot = gr[i][0] * gr[j][0] + gr[i][1] * gr[j][1];
        if constexpr (FRAC) dot += gr[i][2] * gr[j][2];
        out[3 * i + j] = dot * stiff + mass[3 * i + j] * det;
      }
  }

  if (local_vec) {
    T b0, b1, b2;
    p1_load<T, FRAC>(quad, NQ, x0, y0, x1, y1, x2, y2, det, src, frac, mesh, [&](int q) { return s_f[row + q]; }, b0, b1, b2);
    T* out = local_vec + 3 * (int64_t)e;
    out[0] = b0;
    out[1] = b1;
    out[2] = b2;
  }
}

// ---------------------------------------------------------------------------------------------
// Weak residual, element part:  r_loc[e,i] = sum_q dx_q ( f_q phi_i(q) - grad phi_i . grad_u[e,q,:] )
// (examples/example_weak.py:64-75 integrated by abstract_basis.py:95-104).  grad_u is the big
// stream (n_q * d values per element) and is read exactly once.
// ---------------------------------------------------------------------------------------------
// The grad_u (and sampled f) rows of a block of 128 elements are copied to shared memory with fully
// coalesced loads (consecutive lanes, consecutive addresses) and read back row by row from a padded,
// bank-conflict-free layout: the per-element stride in global memory (144 B for the 6-point rule on a
// fracture) would otherwise make every warp load touch 32 different lines.
template <typename T, bool FRAC, int NQ>
__global__ void __launch_bounds__(kStagedBlock) weak_residual_local_kernel(
    int n_el, int n_el_per_mesh, int n_vert_per_mesh, const T* __restrict__ coords,
    const int32_t* __restrict__ conn, const QuadT<T> quad, const FracLite<T> frac,
    const SourceT<T> src, const T* __restrict__ f_q, const T* __restrict__ grad_u,
    T* __restrict__ local_vec) {
  constexpr int D = FRAC ? 3 : 2;
  constexpr int ROW = NQ * D, ROWP = ROW | 1;  // odd stride: conflict-free rows
  constexpr int FROWP = NQ | 1;
  __shared__ T s_gu[kStagedBlock * ROWP];
  __shared__ T s_f[kStagedBlock * FROWP];
  const int e0 = blockIdx.x * kStagedBlock;
  const int count = min(kStagedBlock, n_el - e0);
  {
    const T* g = grad_u + (int64_t)e0 * ROW;
    for (int i = threadIdx.x; i < count * ROW; i += kStagedBlock) s_gu[(i / ROW) * ROWP + i % ROW] = __ldg(g + i);
    if (src.kind == TFEM_SRC_SAMPLED) {
      const T* f = f_q + (int64_t)e0 * NQ;
      for (int i = threadIdx.x; i < count * NQ; i += kStagedBlock) s_f[(i / NQ) * FROWP + i % NQ] = __ldg(f + i);
    }
  }
  __syncthreads();
  const int e = e0 + threadIdx.x;
  if (e >= n_el) return;
  const int mesh = e / n_el_per_mesh;
  const int64_t voff = (int64_t)mesh * n_vert_per_mesh;
  const int v0 = __ldg(conn + 3 * (int64_t)e + 0);
  const int v1 = __ldg(conn + 3 * (int64_t)e + 1);
  const int v2 = __ldg(conn + 3 * (int64_t)e + 2);
  T x0, y0, x1, y1, x2, y2;
  load_xy(coords, voff + v0, x0, y0);
  load_xy(coords, voff + v1, x1, y1);
  load_xy(coords, voff + v2, x2, y2);
  const TriGeom<T> g = tri_geom(x0, y0, x1, y1, x2, y2);
  T gr[3][3];
  gr[0][0] = -g.i00 - g.i10; gr[0][1] = -g.i01 - g.i11; gr[0][2] = T(0);
  gr[1][0] = g.i00;          gr[1][1] = g.i01;          gr[1][2] = T(0);
  gr[2][0] = g.i10;          gr[2][1] = g.i11;          gr[2][2] = T(0);
  T detf = T(1);
  T jf[3][2] = {}, tf[3] = {};
  if constexpr (FRAC) {
    detf = __ldg(frac.det + mesh);
    T jinv[2][3];
#pragma unroll
    for (int a = 0; a < 2; ++a)
#pragma unroll
      for (int c = 0; c < 3; ++c) jinv[a][c] = __ldg(frac.inv + 6 * mesh + 3 * a + c);
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      const T a0 = gr[i][0], a1 = gr[i][1];
#pragma unroll
      for (int c = 0; c < 3; ++c) gr[i][c] = a0 * jinv[0][c] + a1 * jinv[1][c];
    }
    if (src.kind != TFEM_SRC_NONE && src.kind != TFEM_SRC_SAMPLED) {
#pragma unroll
      for (int r = 0; r < 3; ++r) {
        jf[r][0] = __ldg(frac.jac + 6 * mesh + 2 * r);
        jf[r][1] = __ldg(frac.jac + 6 * mesh + 2 * r + 1);
        tf[r] = __ldg(frac.t + 3 * mesh + r);
      }
    }
  }
  const T det = g.det * detf;
  T r0 = T(0), r1 = T(0), r2 = T(0);
  const T* gu = s_gu + threadIdx.x * ROWP;
#pragma unroll
  for (int q = 0; q < NQ; ++q) {
    T f = T(0);
    if (src.kind == TFEM_SRC_SAMPLED) {
      f = s_f[threadIdx.x * FROWP + q];
    } else if (src.kind != TFEM_SRC_NONE) {
      T px = quad.l0[q] * x0 + quad.l1[q] * x1 + quad.l2[q] * x2;
      T py = quad.l0[q] * y0 + quad.l1[q] * y1 + quad.l2[q] * y2;
      if constexpr (FRAC) {  // analytic sources see the first two 3-D coordinates
        const T X = jf[0][0] * px + jf[0][1] * py + tf[0];
        const T Y = jf[1][0] * px + jf[1][1] * py + tf[1];
        px = X;
        py = Y;
      }
      f = source_eval(src, px, py);
    }
    T u[3];
    u[0] = gu[q * D];
    u[1] = gu[q * D + 1];
    u[2] = D == 3 ? gu[q * D + (D - 1)] : T(0);
    const T dxq = quad.w[q] * det;
    T d0 = gr[0][0] * u[0] + gr[0][1] * u[1];
    T d1 = gr[1][0] * u[0] + gr[1][1] * u[1];
    T d2 = gr[2][0] * u[0] + gr[2][1] * u[1];
    if constexpr (FRAC) {
      d0 += gr[0][2] * u[2];
      d1 += gr[1][2] * u[2];
      d2 += gr[2][2] * u[2];
    }
    r0 += dxq * (f * quad.l0[q] - d0);
    r1 += dxq * (f * quad.l1[q] - d1);
    r2 += dxq * (f * quad.l2[q] - d2);
  }
  T* out = local_vec + 3 * (int64_t)e;
  out[0] = r0;
  out[1] = r1;
  out[2] = r2;
}

// ---------------------------------------------------------------------------------------------
// Weak residual of a BATCH OF SMALL MESHES whose DOFs are private to each mesh (PatchesBasis:
// 4 triangles around a centre vertex, 5 DOFs; examples/example_patches.py:102-113), in ONE launch:
// a group of G lanes takes one mesh, lane t integrates element t, and the (at most 8) DOF sums of
// the mesh are formed with warp shuffles in increasing element order -- the order of the reference's
// index_put_ -- and written straight to r[mesh, dof].  No per-element array, no scatter launch.
// ---------------------------------------------------------------------------------------------
template <typename T, int G>
__global__ void __launch_bounds__(256) batched_weak_residual_kernel(
    int n_mesh, int n_el_per_mesh, int n_vert_per_mesh, const T* __restrict__ coords,
    const int32_t* __restrict__ conn, const QuadT<T> quad, const SourceT<T> src,
    const T* __restrict__ f_q, const T* __restrict__ grad_u, T* __restrict__ r) {
  const int thread = blockIdx.x * blockDim.x + threadIdx.x;
  const int mesh = thread / G, t = thread % G;
  const bool active = mesh < n_mesh && t < n_el_per_mesh;
  int v0 = -1, v1 = -1, v2 = -1;
  T r0 = T(0), r1 = T(0), r2 = T(0);
  if (active) {
    const int64_t e = (int64_t)mesh * n_el_per_mesh + t;
    const int64_t voff = (int64_t)mesh * n_vert_per_mesh;
    v0 = __ldg(conn + 3 * e + 0);
    v1 = __ldg(conn + 3 * e + 1);
    v2 = __ldg(conn + 3 * e + 2);
    T x0, y0, x1, y1, x2, y2;
    load_xy(coords, voff + v0, x0, y0);
    load_xy(coords, voff + v1, x1, y1);
    load_xy(coords, voff + v2, x2, y2);
    const TriGeom<T> g = tri_geom(x0, y0, x1, y1, x2, y2);
    const T g00 = -g.i00 - g.i10, g01 = -g.i01 - g.i11;
    const T* gu = grad_u + e * quad.n_q * 2;
    for (int q = 0; q < quad.n_q; ++q) {
      T f = T(0);
      if (src.kind == TFEM_SRC_SAMPLED) {
        f = __ldg(f_q + e * quad.n_q + q);
      } else if (src.kind != TFEM_SRC_NONE) {
        const T px = quad.l0[q] * x0 + quad.l1[q] * x1 + quad.l2[q] * x2;
        const T py = quad.l0[q] * y0 + quad.l1[q] * y1 + quad.l2[q] * y2;
        f = source_eval(src, px, py);
      }
      const T ux = __ldg(gu + 2 * q), uy = __ldg(gu + 2 * q + 1);
      const T dxq = quad.w[q] * g.det;
      r0 += dxq * (f * quad.l0[q] - (g00 * ux + g01 * uy));
      r1 += dxq * (f * quad.l1[q] - (g.i00 * ux + g.i01 * uy));
      r2 += dxq * (f * quad.l2[q] - (g.i10 * ux + g.i11 * uy));
    }
  }
  const unsigned base = (threadIdx.x & 31u) - (unsigned)t;  // first lane of this group
  for (int v = 0; v < n_vert_per_mesh; ++v) {
    const T mine = (v0 == v ? r0 : T(0)) + (v1 == v ? r1 : T(0)) + (v2 == v ? r2 : T(0));
    T sum = __shfl_sync(0xffffffffu, mine, base);
    for (int k = 1; k < n_el_per_mesh; ++k) sum += __shfl_sync(0xffffffffu, mine, base + k);
    if (mesh < n_mesh && t == v % G) r[(int64_t)mesh * n_vert_per_mesh + v] = sum;
  }
}

template <typename T>
int batched_weak_residual(int64_t n_mesh, int n_el_per_mesh, int n_vert_per_mesh, const T* coords, const int32_t* conn,
                          int quad_order, const tfem_source* source, const T* f_q, const T* grad_u, T* r, void* stream) {
  if (n_mesh < 0 || n_el_per_mesh <= 0 || n_el_per_mesh > 8 || n_vert_per_mesh <= 0 || n_vert_per_mesh > 16) return TFEM_ERR_BAD_ARG;
  if (n_mesh == 0) return TFEM_OK;
  if (!coords || !conn || !grad_u || !r) return TFEM_ERR_BAD_ARG;
  if (n_mesh * 8 > kMaxIndex) return TFEM_ERR_TOO_LARGE;
  if (tri_n_q(quad_order) == 0) return TFEM_ERR_UNSUPPORTED;
  const SourceT<T> src = make_source<T>(source);
  if (src.kind < TFEM_SRC_NONE || src.kind > TFEM_SRC_SINSIN) return TFEM_ERR_BAD_ARG;
  if (src.kind == TFEM_SRC_SAMPLED && !f_q) return TFEM_ERR_BAD_ARG;
  const QuadT<T> quad = make_quad<T>(quad_order);
  auto s = static_cast<cudaStream_t>(stream);
  if (n_el_per_mesh <= 4)
    batched_weak_residual_kernel<T, 4><<<blocks_for(n_mesh * 4, 256), 256, 0, s>>>((int)n_mesh, n_el_per_mesh, n_vert_per_mesh, coords, conn, quad,
                                                                                  src, f_q, grad_u, r);
  else
    batched_weak_residual_kernel<T, 8><<<blocks_for(n_mesh * 8, 256), 256, 0, s>>>((int)n_mesh, n_el_per_mesh, n_vert_per_mesh, coords, conn, quad,
                                                                                  src, f_q, grad_u, r);
  return check_launch();
}

// grad_u_bar[e,q,:] = -dx[e,q] * sum_i grad phi_i[e,:] * r_bar[dof_conn[e,i]]
// Each thread lays its element's n_q * d values out in a padded shared-memory row; the block then writes
// the 128 rows with fully coalesced stores.
template <typename T, bool FRAC, int NQ>
__global__ void __launch_bounds__(kStagedBlock) weak_residual_bwd_kernel(
    int n_el, int n_el_per_mesh, int n_vert_per_mesh, const T* __restrict__ coords,
    const int32_t* __restrict__ conn, const int32_t* __restrict__ dof_conn, const QuadT<T> quad,
    const FracLite<T> frac, const T* __restrict__ r_bar, T* __restrict__ grad_u_bar) {
  constexpr int D = FRAC ? 3 : 2;
  constexpr int ROW = NQ * D, ROWP = ROW | 1;
  __shared__ T s_out[kStagedBlock * ROWP];
  const int e0 = blockIdx.x * kStagedBlock;
  const int count = min(kStagedBlock, n_el - e0);
  const int e = e0 + threadIdx.x;
  if (e < n_el) {
    const int mesh = e / n_el_per_mesh;
    const int64_t voff = (int64_t)mesh * n_vert_per_mesh;
    const int v0 = __ldg(conn + 3 * (int64_t)e + 0);
    const int v1 = __ldg(conn + 3 * (int64_t)e + 1);
    const int v2 = __ldg(conn + 3 * (int64_t)e + 2);
    T x0, y0, x1, y1, x2, y2;
    load_xy(coords, voff + v0, x0, y0);
    load_xy(coords, voff + v1, x1, y1);
    load_xy(coords, voff + v2, x2, y2);
    const TriGeom<T> g = tri_geom(x0, y0, x1, y1, x2, y2);
    const T rb0 = __ldg(r_bar + __ldg(dof_conn + 3 * (int64_t)e + 0));
    const T rb1 = __ldg(r_bar + __ldg(dof_conn + 3 * (int64_t)e + 1));
    const T rb2 = __ldg(r_bar + __ldg(dof_conn + 3 * (int64_t)e + 2));
    // s = sum_i r_bar_i grad phi_i (2-D), then mapped to 3-D with J_f^+ for fractures
    const T s0 = rb0 * (-g.i00 - g.i10) + rb1 * g.i00 + rb2 * g.i10;
    const T s1 = rb0 * (-g.i01 - g.i11) + rb1 * g.i01 + rb2 * g.i11;
    T sv[3] = {s0, s1, T(0)};
    T detf = T(1);
    if constexpr (FRAC) {
      detf = __ldg(frac.det + mesh);
#pragma unroll
      for (int c = 0; c < 3; ++c)
        sv[c] = s0 * __ldg(frac.inv + 6 * mesh + c) + s1 * __ldg(frac.inv + 6 * mesh + 3 + c);
    }
    const T det = g.det * detf;
    T* row = s_out + threadIdx.x * ROWP;
#pragma unroll
    for (int q = 0; q < NQ; ++q) {
      const T dxq = -(quad.w[q] * det);
#pragma unroll
      for (int c = 0; c < D; ++c) row[q * D + c] = dxq * sv[c];
    }
  }
  __syncthreads();
  T* out = grad_u_bar + (int64_t)e0 * ROW;
  for (int i = threadIdx.x; i < count * ROW; i += kStagedBlock) out[i] = s_out[(i / ROW) * ROWP + i % ROW];
}

// ---------------------------------------------------------------------------------------------
// H1 error functional of examples/example_weak.py:113-124 integrated by abstract_basis.py:65-72:
//   out[e] = sum_q dx_q ( (u_ex - u)^2 + |grad u_ex - grad u|^2 )   at the element's quadrature points.
// dx is recomputed from the coordinates (no weight tensor is read); the four fields are staged through
// shared memory with coalesced loads like the residual kernel's grad_u.
// ---------------------------------------------------------------------------------------------
template <typename T, int D, int NQ>
__global__ void __launch_bounds__(kStagedBlock) h1_error_kernel(int n_el, int n_el_per_mesh, int n_vert_per_mesh,
                                                       const T* __restrict__ coords, const int32_t* __restrict__ conn,
                                                       const QuadT<T> quad, const T* __restrict__ frac_det,
                                                       const T* __restrict__ u, const T* __restrict__ grad_u,
                                                       const T* __restrict__ u_ex, const T* __restrict__ grad_ex,
                                                       T* __restrict__ out) {
  constexpr int ROW = NQ * (D + 1), ROWP = ROW | 1;
  __shared__ T s_d[kStagedBlock * ROWP];  // per element: (u_ex - u)[NQ], (grad_ex - grad_u)[NQ * D]
  const int e0 = blockIdx.x * kStagedBlock;
  const int count = min(kStagedBlock, n_el - e0);
  for (int i = threadIdx.x; i < count * NQ; i += kStagedBlock)
    s_d[(i / NQ) * ROWP + i % NQ] = __ldg(u_ex + (int64_t)e0 * NQ + i) - __ldg(u + (int64_t)e0 * NQ + i);
  for (int i = threadIdx.x; i < count * NQ * D; i += kStagedBlock)
    s_d[(i / (NQ * D)) * ROWP + NQ + i % (NQ * D)] = __ldg(grad_ex + (int64_t)e0 * NQ * D + i) - __ldg(grad_u + (int64_t)e0 * NQ * D + i);
  __syncthreads();
  const int e = e0 + threadIdx.x;
  if (e >= n_el) return;
  const int mesh = e / n_el_per_mesh;
  const int64_t voff = (int64_t)mesh * n_vert_per_mesh;
  T x0, y0, x1, y1, x2, y2;
  load_xy(coords, voff + __ldg(conn + 3 * (int64_t)e + 0), x0, y0);
  load_xy(coords, voff + __ldg(conn + 3 * (int64_t)e + 1), x1, y1);
  load_xy(coords, voff + __ldg(conn + 3 * (int64_t)e + 2), x2, y2);
  T det = (x1 - x0) * (y2 - y0) - (x2 - x0) * (y1 - y0);
  if (frac_det) det *= __ldg(frac_det + mesh);
  const T* row = s_d + threadIdx.x * ROWP;
  T acc = T(0);
#pragma unroll
  for (int q = 0; q < NQ; ++q) {
    T sq = row[q] * row[q];
#pragma unroll
    for (int c = 0; c < D; ++c) sq += row[NQ + q * D + c] * row[NQ + q * D + c];
    acc += (quad.w[q] * det) * sq;
  }
  out[e] = acc;
}

template <typename T>
int h1_error(int64_t n_el, int64_t n_el_per_mesh, int64_t n_vert_per_mesh, const T* coords, const int32_t* conn, int quad_order,
             const T* frac_det, int d, const T* u, const T* grad_u, const T* u_ex, const T* grad_ex, T* out, void* stream) {
  if (n_el < 0 || n_el_per_mesh <= 0 || n_vert_per_mesh <= 0 || (d != 2 && d != 3)) return TFEM_ERR_BAD_ARG;
  if (n_el == 0) return TFEM_OK;
  if (!coords || !conn || !u || !grad_u || !u_ex || !grad_ex || !out) return TFEM_ERR_BAD_ARG;
  if (n_el > kMaxIndex / 24) return TFEM_ERR_TOO_LARGE;
  if (tri_n_q(quad_order) == 0) return TFEM_ERR_UNSUPPORTED;
  const QuadT<T> quad = make_quad<T>(quad_order);
  auto s = static_cast<cudaStream_t>(stream);
  const unsigned blocks = blocks_for(n_el, kStagedBlock);
#define TFEM_LAUNCH_H1(DD, Q)                                                                                                  \
  h1_error_kernel<T, DD, Q><<<blocks, kStagedBlock, 0, s>>>((int)n_el, (int)n_el_per_mesh, (int)n_vert_per_mesh, coords, conn, quad, frac_det, u, \
                                                   grad_u, u_ex, grad_ex, out)
  switch (quad.n_q) {
    case 1: if (d == 3) TFEM_LAUNCH_H1(3, 1); else TFEM_LAUNCH_H1(2, 1); break;
    case 3: if (d == 3) TFEM_LAUNCH_H1(3, 3); else TFEM_LAUNCH_H1(2, 3); break;
    case 4: if (d == 3) TFEM_LAUNCH_H1(3, 4); else TFEM_LAUNCH_H1(2, 4); break;
    default: if (d == 3) TFEM_LAUNCH_H1(3, 6); else TFEM_LAUNCH_H1(2, 6); break;
  }
#undef TFEM_LAUNCH_H1
  return check_launch();
}

template <typename T>
int quad_reduce(int64_t n_el, int n_q, int m, const T* integrand, int64_t stride_e, int64_t stride_q,
                const T* dx, T* local, void* stream) {
  if (n_el < 0 || n_q <= 0 || m <= 0 || stride_e < 0 || stride_q < 0) return TFEM_ERR_BAD_ARG;
  if (n_el == 0) return TFEM_OK;
  if (!integrand || !dx || !local) return TFEM_ERR_BAD_ARG;
  const int64_t total = n_el * m;
  const int threads = 256;
  if ((total + threads - 1) / threads > kMaxIndex) return TFEM_ERR_TOO_LARGE;
  quad_reduce_kernel<T><<<blocks_for(total, threads), threads, 0, static_cast<cudaStream_t>(stream)>>>(
      total, n_q, m, integrand, stride_e, stride_q, dx, local);
  return check_launch();
}

template <typename T>
int local_forms(int64_t n_el, int64_t n_el_per_mesh, int64_t n_vert_per_mesh, const T* coords,
                const int32_t* conn, int quad_order, const T* frac_jac, const T* frac_det,
                const T* frac_t, const T* frac_inv, const tfem_bilinear* form, const tfem_source* source,
                const T* f_q, T* local_mat, T* local_vec, void* stream) {
  if (n_el < 0 || n_el_per_mesh <= 0 || n_vert_per_mesh <= 0) return TFEM_ERR_BAD_ARG;
  if (n_el == 0) return TFEM_OK;
  if (!coords || !conn) return TFEM_ERR_BAD_ARG;
  if (local_mat && !form) return TFEM_ERR_BAD_ARG;
  if (n_el > kMaxIndex / 9) return TFEM_ERR_TOO_LARGE;
  if (tri_n_q(quad_order) == 0) return TFEM_ERR_UNSUPPORTED;
  const SourceT<T> src = make_source<T>(source);
  if (src.kind < TFEM_SRC_NONE || src.kind > TFEM_SRC_SINSIN) return TFEM_ERR_BAD_ARG;
  if (local_vec && src.kind == TFEM_SRC_SAMPLED && !f_q) return TFEM_ERR_BAD_ARG;
  const bool frac = frac_det != nullptr;
  if (frac && (!frac_inv || !frac_jac || !frac_t)) return TFEM_ERR_BAD_ARG;
  const QuadT<T> quad = make_quad<T>(quad_order);
  const FracLite<T> fl{frac_jac, frac_inv, frac_det, frac_t};
  const T alpha = form ? T(form->alpha) : T(0), beta = form ? T(form->beta) : T(0);
  const int threads = 256;
  auto s = static_cast<cudaStream_t>(stream);
  if (frac)
    local_forms_kernel<T, true><<<blocks_for(n_el, threads), threads, 0, s>>>(
        (int)n_el, (int)n_el_per_mesh, (int)n_vert_per_mesh, coords, conn, quad, fl, alpha, beta, src, f_q,
        local_mat, local_vec);
  else
    local_forms_kernel<T, false><<<blocks_for(n_el, threads), threads, 0, s>>>(
        (int)n_el, (int)n_el_per_mesh, (int)n_vert_per_mesh, coords, conn, quad, fl, alpha, beta, src, f_q,
        local_mat, local_vec);
  return check_launch();
}

template <typename T>
int weighted_local_forms(int64_t n_el, int64_t n_el_per_mesh, int64_t n_vert_per_mesh, const T* coords,
                         const int32_t* conn, int quad_order, const T* frac_jac, const T* frac_det, const T* frac_t,
                         const T* frac_inv, const tfem_bilinear* form, const tfem_source* source, const T* f_q,
                         const T* alpha_q, const T* beta_q, T* local_mat, T* local_vec, void* stream) {
  if (n_el < 0 || n_el_per_mesh <= 0 || n_vert_per_mesh <= 0) return TFEM_ERR_BAD_ARG;
  if (n_el == 0) return TFEM_OK;
  if (!coords || !conn) return TFEM_ERR_BAD_ARG;
  if (local_mat && !form && (!alpha_q || !beta_q)) return TFEM_ERR_BAD_ARG;
  if (n_el > kMaxIndex / 9) return TFEM_ERR_TOO_LARGE;
  if (tri_n_q(quad_order) == 0) return TFEM_ERR_UNSUPPORTED;
  const SourceT<T> src = make_source<T>(source);
  if (src.kind < TFEM_SRC_NONE || src.kind > TFEM_SRC_SINSIN) return TFEM_ERR_BAD_ARG;
  if (local_vec && src.kind == TFEM_SRC_SAMPLED && !f_q) return TFEM_ERR_BAD_ARG;
  const bool frac = frac_det != nullptr;
  if (frac && (!frac_inv || !frac_jac || !frac_t)) return TFEM_ERR_BAD_ARG;
  const QuadT<T> quad = make_quad<T>(quad_order);
  const FracLite<T> fl{frac_jac, frac_inv, frac_det, frac_t};
  const T alpha = form ? T(form->alpha) : T(0), beta = form ? T(form->beta) : T(0);
  auto s = static_cast<cudaStream_t>(stream);
  const unsigned blocks = blocks_for(n_el, kStagedBlock);
#define TFEM_LAUNCH_WEIGHTED(F, Q)                                                                                  \
  weighted_local_forms_kernel<T, F, Q><<<blocks, kStagedBlock, 0, s>>>((int)n_el, (int)n_el_per_mesh, (int)n_vert_per_mesh, \
                                                                      coords, conn, quad, fl, alpha, beta, src, f_q, alpha_q, \
                                                                      beta_q, local_mat, local_vec)
  switch (quad.n_q) {
    case 1: if (frac) TFEM_LAUNCH_WEIGHTED(true, 1); else TFEM_LAUNCH_WEIGHTED(false, 1); break;
    case 3: if (frac) TFEM_LAUNCH_WEIGHTED(true, 3); else TFEM_LAUNCH_WEIGHTED(false, 3); break;
    case 4: if (frac) TFEM_LAUNCH_WEIGHTED(true, 4); else TFEM_LAUNCH_WEIGHTED(false, 4); break;
    default: if (frac) TFEM_LAUNCH_WEIGHTED(true, 6); else TFEM_LAUNCH_WEIGHTED(false, 6); break;
  }
#undef TFEM_LAUNCH_WEIGHTED
  return check_launch();
}

template <typename T>
int weak_residual_local(int64_t n_el, int64_t n_el_per_mesh, int64_t n_vert_per_mesh, const T* coords,
                        const int32_t* conn, int quad_order, const T* frac_jac, const T* frac_inv,
                        const T* frac_det, const T* frac_t, const tfem_source* source, const T* f_q,
                        const T* grad_u, T* local_vec, void* stream) {
  if (n_el < 0 || n_el_per_mesh <= 0 || n_vert_per_mesh <= 0) return TFEM_ERR_BAD_ARG;
  if (n_el == 0) return TFEM_OK;
  if (!coords || !conn || !grad_u || !local_vec) return TFEM_ERR_BAD_ARG;
  if (n_el > kMaxIndex / 18) return TFEM_ERR_TOO_LARGE;
  if (tri_n_q(quad_order) == 0) return TFEM_ERR_UNSUPPORTED;
  const SourceT<T> src = make_source<T>(source);
  if (src.kind < TFEM_SRC_NONE || src.kind > TFEM_SRC_SINSIN) return TFEM_ERR_BAD_ARG;
  if (src.kind == TFEM_SRC_SAMPLED && !f_q) return TFEM_ERR_BAD_ARG;
  const bool frac = frac_inv != nullptr;
  if (frac && (!frac_det || !frac_jac || !frac_t)) return TFEM_ERR_BAD_ARG;
  const QuadT<T> quad = make_quad<T>(quad_order);
  const FracLite<T> fl{frac_jac, frac_inv, frac_det, frac_t};
  auto s = static_cast<cudaStream_t>(stream);
  const unsigned blocks = blocks_for(n_el, kStagedBlock);
#define TFEM_LAUNCH_FWD(F, Q)                                                                                   \
  weak_residual_local_kernel<T, F, Q><<<blocks, kStagedBlock, 0, s>>>((int)n_el, (int)n_el_per_mesh, (int)n_vert_per_mesh, coords, conn, quad, \
                                                             fl, src, f_q, grad_u, local_vec)
  switch (quad.n_q) {
    case 1: if (frac) TFEM_LAUNCH_FWD(true, 1); else TFEM_LAUNCH_FWD(false, 1); break;
    case 3: if (frac) TFEM_LAUNCH_FWD(true, 3); else TFEM_LAUNCH_FWD(false, 3); break;
    case 4: if (frac) TFEM_LAUNCH_FWD(true, 4); else TFEM_LAUNCH_FWD(false, 4); break;
    default: if (frac) TFEM_LAUNCH_FWD(true, 6); else TFEM_LAUNCH_FWD(false, 6); break;
  }
#undef TFEM_LAUNCH_FWD
  return check_launch();
}

template <typename T>
int weak_residual_bwd(int64_t n_el, int64_t n_el_per_mesh, int64_t n_vert_per_mesh, const T* coords,
                      const int32_t* conn, const int32_t* dof_conn, int quad_order, const T* frac_jac,
                      const T* frac_inv, const T* frac_det, const T* r_bar, T* grad_u_bar, void* stream) {
  (void)frac_jac;
  if (n_el < 0 || n_el_per_mesh <= 0 || n_vert_per_mesh <= 0) return TFEM_ERR_BAD_ARG;
  if (n_el == 0) return TFEM_OK;
  if (!coords || !conn || !dof_conn || !r_bar || !grad_u_bar) return TFEM_ERR_BAD_ARG;
  if (n_el > kMaxIndex / 18) return TFEM_ERR_TOO_LARGE;
  if (tri_n_q(quad_order) == 0) return TFEM_ERR_UNSUPPORTED;
  const bool frac = frac_inv != nullptr;
  if (frac && !frac_det) return TFEM_ERR_BAD_ARG;
  const QuadT<T> quad = make_quad<T>(quad_order);
  const FracLite<T> fl{nullptr, frac_inv, frac_det, nullptr};
  auto s = static_cast<cudaStream_t>(stream);
  const unsigned blocks = blocks_for(n_el, kStagedBlock);
#define TFEM_LAUNCH_BWD(F, Q)                                                                                 \
  weak_residual_bwd_kernel<T, F, Q><<<blocks, kStagedBlock, 0, s>>>((int)n_el, (int)n_el_per_mesh, (int)n_vert_per_mesh, coords, conn, dof_conn, \
                                                           quad, fl, r_bar, grad_u_bar)
  switch (quad.n_q) {
    case 1: if (frac) TFEM_LAUNCH_BWD(true, 1); else TFEM_LAUNCH_BWD(false, 1); break;
    case 3: if (frac) TFEM_LAUNCH_BWD(true, 3); else TFEM_LAUNCH_BWD(false, 3); break;
    case 4: if (frac) TFEM_LAUNCH_BWD(true, 4); else TFEM_LAUNCH_BWD(false, 4); break;
    default: if (frac) TFEM_LAUNCH_BWD(true, 6); else TFEM_LAUNCH_BWD(false, 6); break;
  }
#undef TFEM_LAUNCH_BWD
  return check_launch();
}

}  // namespace tfem

#define TFEM_FORMS_API(T, SUF)                                                                      \
  extern "C" int tfem_quad_reduce_##SUF(int64_t n_el, int n_q, int m, const T* integrand,           \
                                        int64_t stride_e, int64_t stride_q, const T* dx, T* local,  \
                                        void* stream) {                                             \
    return tfem::quad_reduce<T>(n_el, n_q, m, integrand, stride_e, stride_q, dx, local, stream);    \
  }                                                                                                 \
  extern "C" int tfem_tri_p1_local_forms_##SUF(                                                     \
      int64_t n_el, int64_t n_el_per_mesh, int64_t n_vert_per_mesh, const T* coords,                \
      const int32_t* conn, int quad_order, const T* frac_jac, const T* frac_inv, const T* frac_det, \
      const T* frac_t, const tfem_bilinear* host_form, const tfem_source* host_source,              \
      const T* f_q, T* local_mat, T* local_vec, void* stream) {                                     \
    return tfem::local_forms<T>(n_el, n_el_per_mesh, n_vert_per_mesh, coords, conn, quad_order,     \
                                frac_jac, frac_det, frac_t, frac_inv, host_form, host_source, f_q,  \
                                local_mat, local_vec, stream);                                      \
  }                                                                                                 \
  extern "C" int tfem_tri_p1_weighted_local_forms_##SUF(                                            \
      int64_t n_el, int64_t n_el_per_mesh, int64_t n_vert_per_mesh, const T* coords,                \
      const int32_t* conn, int quad_order, const T* frac_jac, const T* frac_inv, const T* frac_det, \
      const T* frac_t, const tfem_bilinear* host_form, const tfem_source* host_source,              \
      const T* f_q, const T* alpha_q, const T* beta_q, T* local_mat, T* local_vec, void* stream) {  \
    return tfem::weighted_local_forms<T>(n_el, n_el_per_mesh, n_vert_per_mesh, coords, conn,        \
                                         quad_order, frac_jac, frac_det, frac_t, frac_inv,          \
                                         host_form, host_source, f_q, alpha_q, beta_q, local_mat,   \
                                         local_vec, stream);                                        \
  }                                                                                                 \
  extern "C" int tfem_weak_residual_local_##SUF(                                                    \
      int64_t n_el, int64_t n_el_per_mesh, int64_t n_vert_per_mesh, const T* coords,                \
      const int32_t* conn, int quad_order, const T* frac_jac, const T* frac_inv, const T* frac_det, \
      const T* frac_t, const tfem_source* host_source, const T* f_q, const T* grad_u, T* local_vec, \
      void* stream) {                                                                               \
    return tfem::weak_residual_local<T>(n_el, n_el_per_mesh, n_vert_per_mesh, coords, conn,         \
                                        quad_order, frac_jac, frac_inv, frac_det, frac_t,           \
                                        host_source, f_q, grad_u, local_vec, stream);               \
  }                                                                                                 \
  extern "C" int tfem_weak_residual_bwd_##SUF(                                                      \
      int64_t n_el, int64_t n_el_per_mesh, int64_t n_vert_per_mesh, const T* coords,                \
      const int32_t* conn, const int32_t* dof_conn, int quad_order, const T* frac_jac,              \
      const T* frac_inv, const T* frac_det, const T* r_bar, T* grad_u_bar, void* stream) {          \
    return tfem::weak_residual_bwd<T>(n_el, n_el_per_mesh, n_vert_per_mesh, coords, conn, dof_conn, \
                                      quad_order, frac_jac, frac_inv, frac_det, r_bar, grad_u_bar,  \
                                      stream);                                                      \
  }

TFEM_FORMS_API(double, f64)
TFEM_FORMS_API(float, f32)

#define TFEM_BATCHED_API(T, SUF)                                                                                  \
  extern "C" int tfem_batched_weak_residual_##SUF(int64_t n_mesh, int n_el_per_mesh, int n_vert_per_mesh,         \
                                                  const T* coords, const int32_t* conn, int quad_order,           \
                                                  const tfem_source* host_source, const T* f_q, const T* grad_u,  \
                                                  T* r, void* stream) {                                           \
    return tfem::batched_weak_residual<T>(n_mesh, n_el_per_mesh, n_vert_per_mesh, coords, conn, quad_order,       \
                                          host_source, f_q, grad_u, r, stream);                                   \
  }
TFEM_BATCHED_API(double, f64)
TFEM_BATCHED_API(float, f32)

#define TFEM_H1_API(T, SUF)                                                                                          \
  extern "C" int tfem_h1_error_##SUF(int64_t n_el, int64_t n_el_per_mesh, int64_t n_vert_per_mesh, const T* coords,  \
                                     const int32_t* conn, int quad_order, const T* frac_det, int d, const T* u,      \
                                     const T* grad_u, const T* u_ex, const T* grad_ex, T* out, void* stream) {       \
    return tfem::h1_error<T>(n_el, n_el_per_mesh, n_vert_per_mesh, coords, conn, quad_order, frac_det, d, u, grad_u, \
                             u_ex, grad_ex, out, stream);                                                            \
  }
TFEM_H1_API(double, f64)
TFEM_H1_API(float, f32)

// CSR sparse matrix-vector product for the iterative solve on the assembled system
// (SURVEY.md 8(f).1: replaces the dense torch.linalg.solve of basis/abstract_basis.py:177-195 when
// the system is too large to densify).  HBM bound: 12 B per stored entry (value + column) plus the
// vectors; P1 rows hold ~7 entries, so 8 lanes share a row and a warp streams 4 consecutive rows,
// i.e. contiguous csr_val / col segments.
#include <limits>

#include "common.cuh"

namespace tfem {

// y[i] = keep[i] ? sum_k val[k] x[col[k]] : 0   (keep == nullptr: every row)
template <typename T, int LANES>
__global__ void __launch_bounds__(256) csr_spmv_kernel(int n_rows, const int32_t* __restrict__ crow,
                                                       const int32_t* __restrict__ col, const T* __restrict__ val,
                                                       const T* __restrict__ x, const uint8_t* __restrict__ keep,
                                                       T* __restrict__ y) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int row = (int)(t / LANES);
  const int lane = (int)(t % LANES);
  T acc = T(0);
  const bool live = row < n_rows && (keep == nullptr || keep[row] != 0);
  if (live) {
    const int begin = __ldg(crow + row), end = __ldg(crow + row + 1);
    for (int k = begin + lane; k < end; k += LANES) acc = fma(__ldg(val + k), __ldg(x + __ldg(col + k)), acc);
  }
#pragma unroll
  for (int offset = LANES / 2; offset > 0; offset >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, offset, LANES);
  if (lane == 0 && row < n_rows) y[row] = live ? acc : T(0);
}

template <typename T>
int csr_spmv(int64_t n_rows, const int32_t* crow, const int32_t* col, const T* val, const T* x, const uint8_t* keep,
             T* y, void* stream) {
  if (n_rows < 0) return TFEM_ERR_BAD_ARG;
  if (n_rows == 0) return TFEM_OK;
  if (!crow || !col || !val || !x || !y) return TFEM_ERR_BAD_ARG;
  if (n_rows > kMaxIndex / 8) return TFEM_ERR_TOO_LARGE;
  constexpr int kLanes = 8;
  csr_spmv_kernel<T, kLanes><<<blocks_for(n_rows * kLanes, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      (int)n_rows, crow, col, val, x, keep, y);
  return check_launch();
}

}  // namespace tfem

extern "C" int tfem_csr_spmv_f64(int64_t n_rows, const int32_t* crow, const int32_t* col, const double* val,
                                 const double* x, const uint8_t* keep, double* y, void* stream) {
  return tfem::csr_spmv<double>(n_rows, crow, col, val, x, keep, y, stream);
}

extern "C" int tfem_csr_spmv_f32(int64_t n_rows, const int32_t* crow, const int32_t* col, const float* val,
                                 const float* x, const uint8_t* keep, float* y, void* stream) {
  return tfem::csr_spmv<float>(n_rows, crow, col, val, x, keep, y, stream);
}

// ---------------------------------------------------------------------------------------------
// Fused conjugate-gradient iteration: three kernels, every dot product reduced in a fixed order
// (per-thread grid-stride partial -> warp shuffle tree -> per-block partial in global memory ->
// every block of the NEXT kernel sums the partials in the same order), so a solve is bitwise
// reproducible and nothing synchronises with the host.
//   K1  ap = M A p,  partial[b] = sum p.ap            (also moves rz_new -> rz for this iteration)
//   K2  alpha = rz / sum(partial);  x += alpha p;  r -= alpha ap;  z = r * inv_diag;  partial[b] = sum r.z
//   K3  rz_new = sum(partial);  p = z + (rz_new / rz) p
// scal[0] = rz of the current iteration, scal[1] = rz_new; each is written by one block in a kernel
// in which nobody reads it.
// ---------------------------------------------------------------------------------------------
namespace tfem {

constexpr int kCgThreads = 256;

template <typename T>
__device__ __forceinline__ T block_sum(T v, T* scratch) {
#pragma unroll
  for (int offset = 16; offset > 0; offset >>= 1) v += __shfl_xor_sync(0xffffffffu, v, offset);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  __syncthreads();  // scratch may still be read from a previous call
  if (lane == 0) scratch[warp] = v;
  __syncthreads();
  T total = T(0);
#pragma unroll
  for (int w = 0; w < kCgThreads / 32; ++w) total += scratch[w];
  return total;  // the same value in every thread
}

template <typename T>
__device__ __forceinline__ T sum_partials(const T* __restrict__ partial, int n, T* scratch) {
  T v = T(0);
  for (int i = threadIdx.x; i < n; i += kCgThreads) v += partial[i];
  return block_sum(v, scratch);
}

template <typename T, int LANES>
__global__ void __launch_bounds__(kCgThreads) cg_spmv_dot_kernel(int n_rows, const int32_t* __restrict__ crow,
                                                                const int32_t* __restrict__ col, const T* __restrict__ val,
                                                                const T* __restrict__ p, const uint8_t* __restrict__ keep,
                                                                T* __restrict__ ap, T* __restrict__ partial, T* scal) {
  __shared__ T scratch[kCgThreads / 32];
  if (blockIdx.x == 0 && threadIdx.x == 0) scal[0] = scal[1];
  const int lane = threadIdx.x % LANES;
  const int group = (blockIdx.x * kCgThreads + threadIdx.x) / LANES;
  const int n_groups = gridDim.x * kCgThreads / LANES;
  T dot = T(0);
  for (int base = 0; base < n_rows; base += n_groups) {  // uniform trip count: the shuffles below stay convergent
    const int row = base + group;
    const bool live = row < n_rows && (keep == nullptr || keep[row] != 0);
    T acc = T(0);
    if (live) {
      const int begin = __ldg(crow + row), end = __ldg(crow + row + 1);
      for (int k = begin + lane; k < end; k += LANES) acc = fma(__ldg(val + k), p[__ldg(col + k)], acc);
    }
#pragma unroll
    for (int offset = LANES / 2; offset > 0; offset >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, offset, LANES);
    if (lane == 0 && row < n_rows) {
      ap[row] = acc;
      dot = fma(p[row], acc, dot);
    }
  }
  const T total = block_sum(dot, scratch);
  if (threadIdx.x == 0) partial[blockIdx.x] = total;
}

template <typename T>
__global__ void __launch_bounds__(kCgThreads) cg_update_kernel(int n, const T* __restrict__ p, const T* __restrict__ ap,
                                                              const T* __restrict__ inv_diag, T* __restrict__ x, T* __restrict__ r,
                                                              T* __restrict__ z, const T* partial_in, int n_partial,
                                                              T* __restrict__ partial_out, const T* scal, T tiny) {
  __shared__ T scratch[kCgThreads / 32];
  const T pap = sum_partials(partial_in, n_partial, scratch);
  const T alpha = scal[0] / (pap > tiny ? pap : tiny);
  T dot = T(0);
  for (int i = blockIdx.x * kCgThreads + threadIdx.x; i < n; i += gridDim.x * kCgThreads) {
    const T pi = p[i], api = ap[i];
    x[i] = fma(alpha, pi, x[i]);
    const T ri = fma(-alpha, api, r[i]);
    r[i] = ri;
    const T zi = ri * inv_diag[i];
    z[i] = zi;
    dot = fma(ri, zi, dot);
  }
  const T total = block_sum(dot, scratch);
  if (threadIdx.x == 0) partial_out[blockIdx.x] = total;
}

template <typename T>
__global__ void __launch_bounds__(kCgThreads) cg_direction_kernel(int n, const T* __restrict__ z, T* __restrict__ p,
                                                                 const T* partial_in, int n_partial, T* scal, T tiny) {
  __shared__ T scratch[kCgThreads / 32];
  const T rz_new = sum_partials(partial_in, n_partial, scratch);
  const T rz = scal[0];
  const T beta = rz_new / (rz > tiny ? rz : tiny);
  if (blockIdx.x == 0 && threadIdx.x == 0) scal[1] = rz_new;
  for (int i = blockIdx.x * kCgThreads + threadIdx.x; i < n; i += gridDim.x * kCgThreads) p[i] = fma(beta, p[i], z[i]);
}

template <typename T>
int cg_iteration(int64_t n, const int32_t* crow, const int32_t* col, const T* val, const uint8_t* keep, const T* inv_diag,
                 T* x, T* r, T* z, T* p, T* ap, T* partial, int32_t n_partial, T* scal, void* stream) {
  if (n < 0 || n_partial <= 0) return TFEM_ERR_BAD_ARG;
  if (n == 0) return TFEM_OK;
  if (!crow || !col || !val || !inv_diag || !x || !r || !z || !p || !ap || !partial || !scal) return TFEM_ERR_BAD_ARG;
  if (n > kMaxIndex / 8) return TFEM_ERR_TOO_LARGE;
  auto s = static_cast<cudaStream_t>(stream);
  const T tiny = std::numeric_limits<T>::min();
  const unsigned grid = (unsigned)n_partial;  // one partial per block; the caller sizes it (SMs x 8)
  cg_spmv_dot_kernel<T, 8><<<grid, kCgThreads, 0, s>>>((int)n, crow, col, val, p, keep, ap, partial, scal);
  cg_update_kernel<T><<<grid, kCgThreads, 0, s>>>((int)n, p, ap, inv_diag, x, r, z, partial, n_partial, partial + n_partial, scal, tiny);
  cg_direction_kernel<T><<<grid, kCgThreads, 0, s>>>((int)n, z, p, partial + n_partial, n_partial, scal, tiny);
  return check_launch();
}

}  // namespace tfem

extern "C" int tfem_cg_iteration_f64(int64_t n, const int32_t* crow, const int32_t* col, const double* val,
                                     const uint8_t* keep, const double* inv_diag, double* x, double* r, double* z, double* p,
                                     double* ap, double* partial, int32_t n_partial, double* scal, void* stream) {
  return tfem::cg_iteration<double>(n, crow, col, val, keep, inv_diag, x, r, z, p, ap, partial, n_partial, scal, stream);
}

extern "C" int tfem_cg_iteration_f32(int64_t n, const int32_t* crow, const int32_t* col, const float* val,
                                     const uint8_t* keep, const float* inv_diag, float* x, float* r, float* z, float* p,
                                     float* ap, float* partial, int32_t n_partial, float* scal, void* stream) {
  return tfem::cg_iteration<float>(n, crow, col, val, keep, inv_diag, x, r, z, p, ap, partial, n_partial, scal, stream);
}

// ---------------------------------------------------------------------------------------------
// Smoothed-aggregation AMG V-cycle (set-up: sparse.amg) and the conjugate-gradient iteration preconditioned by it.
// One symmetric V-cycle, z = M r, from a zero initial guess on every level l (b = right-hand side of the level):
//   residual   x = w D^-1 b;  t = b - A x                 (one kernel: A x needs no stored x, x_j = w_j b_j)
//   restrict   b_c = R t
//   recurse    e_c = cycle(b_c)   (coarsest: e_c = A_c^-1 b_c, a dense matvec, one warp per row)
//   prolongate x += P e_c
//   smooth     y = x + w D^-1 (b - A x)                    (y: the level's result; t shares its buffer)
// Every launch is on the caller's stream and nothing allocates or synchronises: the cycle is graph capturable.
// Every sum is a fixed-order lane tree, so the cycle is bitwise reproducible.
// ---------------------------------------------------------------------------------------------
namespace tfem {

template <typename T, int LANES>
__global__ void __launch_bounds__(256) amg_residual_kernel(int n, const int32_t* __restrict__ crow, const int32_t* __restrict__ col,
                                                           const T* __restrict__ val, const T* __restrict__ wd, const T* __restrict__ b,
                                                           T* __restrict__ x, T* __restrict__ t) {
  const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int row = (int)(g / LANES);
  const int lane = (int)(g % LANES);
  T acc = T(0);
  if (row < n) {
    const int begin = __ldg(crow + row), end = __ldg(crow + row + 1);
    for (int k = begin + lane; k < end; k += LANES) {
      const int c = __ldg(col + k);
      acc = fma(__ldg(val + k), __ldg(wd + c) * __ldg(b + c), acc);
    }
  }
#pragma unroll
  for (int offset = LANES / 2; offset > 0; offset >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, offset, LANES);
  if (lane == 0 && row < n) {
    const T bi = b[row];
    x[row] = wd[row] * bi;
    t[row] = bi - acc;
  }
}

// x += P e
template <typename T, int LANES>
__global__ void __launch_bounds__(256) amg_prolong_kernel(int n, const int32_t* __restrict__ crow, const int32_t* __restrict__ col,
                                                          const T* __restrict__ val, const T* __restrict__ e, T* __restrict__ x) {
  const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int row = (int)(g / LANES);
  const int lane = (int)(g % LANES);
  T acc = T(0);
  if (row < n) {
    const int begin = __ldg(crow + row), end = __ldg(crow + row + 1);
    for (int k = begin + lane; k < end; k += LANES) acc = fma(__ldg(val + k), __ldg(e + __ldg(col + k)), acc);
  }
#pragma unroll
  for (int offset = LANES / 2; offset > 0; offset >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, offset, LANES);
  if (lane == 0 && row < n) x[row] += acc;
}

// y = x + w D^-1 (b - A x)
template <typename T, int LANES>
__global__ void __launch_bounds__(256) amg_smooth_kernel(int n, const int32_t* __restrict__ crow, const int32_t* __restrict__ col,
                                                         const T* __restrict__ val, const T* __restrict__ wd, const T* __restrict__ b,
                                                         const T* __restrict__ x, T* __restrict__ y) {
  const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int row = (int)(g / LANES);
  const int lane = (int)(g % LANES);
  T acc = T(0);
  if (row < n) {
    const int begin = __ldg(crow + row), end = __ldg(crow + row + 1);
    for (int k = begin + lane; k < end; k += LANES) acc = fma(__ldg(val + k), x[__ldg(col + k)], acc);
  }
#pragma unroll
  for (int offset = LANES / 2; offset > 0; offset >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, offset, LANES);
  if (lane == 0 && row < n) y[row] = fma(wd[row], b[row] - acc, x[row]);
}

// y = inv b, inv dense row-major [n, n]: one warp per row, lanes stride the columns, fixed shuffle tree
template <typename T>
__global__ void __launch_bounds__(256) amg_dense_kernel(int n, const T* __restrict__ inv, const T* __restrict__ b, T* __restrict__ y) {
  const int row = (int)(((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
  const int lane = threadIdx.x & 31;
  T acc = T(0);
  if (row < n)
    for (int j = lane; j < n; j += 32) acc = fma(__ldg(inv + (int64_t)row * n + j), __ldg(b + j), acc);
#pragma unroll
  for (int offset = 16; offset > 0; offset >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, offset);
  if (lane == 0 && row < n) y[row] = acc;
}

constexpr int kAmgLanes = 8;
constexpr int64_t kMaxCoarse = 32768;  // the dense coarsest inverse holds n_coarse^2 values

inline int check_levels(const tfem_amg_level* levels, int n_levels, const void* coarse_inv, int64_t n_coarse) {
  if (n_levels < 0 || n_coarse <= 0 || !coarse_inv || (n_levels > 0 && !levels)) return TFEM_ERR_BAD_ARG;
  if (n_coarse > kMaxCoarse) return TFEM_ERR_TOO_LARGE;
  for (int l = 0; l < n_levels; ++l) {
    const tfem_amg_level& v = levels[l];
    if (v.n <= 0 || v.n_coarse <= 0) return TFEM_ERR_BAD_ARG;
    if (v.n > kMaxIndex / kAmgLanes || v.n_coarse > kMaxIndex / kAmgLanes) return TFEM_ERR_TOO_LARGE;
    if (!v.a_crow || !v.a_col || !v.a_val || !v.p_crow || !v.p_col || !v.p_val || !v.r_crow || !v.r_col || !v.r_val || !v.wdinv ||
        !v.x || !v.rc || !v.ec)
      return TFEM_ERR_BAD_ARG;
    const int64_t next = l + 1 < n_levels ? levels[l + 1].n : n_coarse;
    if (v.n_coarse != next) return TFEM_ERR_BAD_ARG;
  }
  return TFEM_OK;
}

template <typename T>
void amg_vcycle_launch(const tfem_amg_level* levels, int n_levels, const T* coarse_inv, int64_t n_coarse, const T* r, T* z,
                       cudaStream_t s) {
  auto rhs = [&](int l) { return l == 0 ? r : static_cast<const T*>(levels[l - 1].rc); };
  auto out = [&](int l) { return l == 0 ? z : static_cast<T*>(levels[l - 1].ec); };
  for (int l = 0; l < n_levels; ++l) {
    const tfem_amg_level& v = levels[l];
    const unsigned grid = blocks_for(v.n * kAmgLanes, 256);
    amg_residual_kernel<T, kAmgLanes><<<grid, 256, 0, s>>>((int)v.n, v.a_crow, v.a_col, static_cast<const T*>(v.a_val),
                                                            static_cast<const T*>(v.wdinv), rhs(l), static_cast<T*>(v.x), out(l));
    csr_spmv_kernel<T, kAmgLanes><<<blocks_for(v.n_coarse * kAmgLanes, 256), 256, 0, s>>>(
        (int)v.n_coarse, v.r_crow, v.r_col, static_cast<const T*>(v.r_val), out(l), nullptr, static_cast<T*>(v.rc));
  }
  amg_dense_kernel<T><<<blocks_for(n_coarse * 32, 256), 256, 0, s>>>((int)n_coarse, coarse_inv, rhs(n_levels), out(n_levels));
  for (int l = n_levels - 1; l >= 0; --l) {
    const tfem_amg_level& v = levels[l];
    const unsigned grid = blocks_for(v.n * kAmgLanes, 256);
    amg_prolong_kernel<T, kAmgLanes><<<grid, 256, 0, s>>>((int)v.n, v.p_crow, v.p_col, static_cast<const T*>(v.p_val),
                                                           static_cast<const T*>(v.ec), static_cast<T*>(v.x));
    amg_smooth_kernel<T, kAmgLanes><<<grid, 256, 0, s>>>((int)v.n, v.a_crow, v.a_col, static_cast<const T*>(v.a_val),
                                                          static_cast<const T*>(v.wdinv), rhs(l), static_cast<const T*>(v.x), out(l));
  }
}

template <typename T>
int amg_vcycle(const tfem_amg_level* levels, int n_levels, const T* coarse_inv, int64_t n_coarse, const T* r, T* z, void* stream) {
  const int status = check_levels(levels, n_levels, coarse_inv, n_coarse);
  if (status != TFEM_OK) return status;
  if (!r || !z) return TFEM_ERR_BAD_ARG;
  amg_vcycle_launch<T>(levels, n_levels, coarse_inv, n_coarse, r, z, static_cast<cudaStream_t>(stream));
  return check_launch();
}

// alpha = rz / sum(partial);  x += alpha p;  r -= alpha ap   (z comes from the V-cycle)
template <typename T>
__global__ void __launch_bounds__(kCgThreads) pcg_update_kernel(int n, const T* __restrict__ p, const T* __restrict__ ap, T* __restrict__ x,
                                                               T* __restrict__ r, const T* partial_in, int n_partial, const T* scal, T tiny) {
  __shared__ T scratch[kCgThreads / 32];
  const T pap = sum_partials(partial_in, n_partial, scratch);
  const T alpha = scal[0] / (pap > tiny ? pap : tiny);
  for (int i = blockIdx.x * kCgThreads + threadIdx.x; i < n; i += gridDim.x * kCgThreads) {
    x[i] = fma(alpha, p[i], x[i]);
    r[i] = fma(-alpha, ap[i], r[i]);
  }
}

// partial[b] = sum over the block's grid-stride share of r.z
template <typename T>
__global__ void __launch_bounds__(kCgThreads) pcg_dot_kernel(int n, const T* __restrict__ r, const T* __restrict__ z,
                                                            T* __restrict__ partial_out) {
  __shared__ T scratch[kCgThreads / 32];
  T dot = T(0);
  for (int i = blockIdx.x * kCgThreads + threadIdx.x; i < n; i += gridDim.x * kCgThreads) dot = fma(r[i], z[i], dot);
  const T total = block_sum(dot, scratch);
  if (threadIdx.x == 0) partial_out[blockIdx.x] = total;
}

template <typename T>
int pcg_iteration(int64_t n, const int32_t* crow, const int32_t* col, const T* val, const uint8_t* keep, const tfem_amg_level* levels,
                  int n_levels, const T* coarse_inv, int64_t n_coarse, T* x, T* r, T* z, T* p, T* ap, T* partial, int32_t n_partial,
                  T* scal, void* stream) {
  if (n < 0 || n_partial <= 0) return TFEM_ERR_BAD_ARG;
  if (n == 0) return TFEM_OK;
  if (!crow || !col || !val || !x || !r || !z || !p || !ap || !partial || !scal) return TFEM_ERR_BAD_ARG;
  if (n > kMaxIndex / 8) return TFEM_ERR_TOO_LARGE;
  const int status = check_levels(levels, n_levels, coarse_inv, n_coarse);
  if (status != TFEM_OK) return status;
  if ((n_levels > 0 ? levels[0].n : n_coarse) != n) return TFEM_ERR_BAD_ARG;  // the hierarchy of another system
  auto s = static_cast<cudaStream_t>(stream);
  const T tiny = std::numeric_limits<T>::min();
  const unsigned grid = (unsigned)n_partial;
  cg_spmv_dot_kernel<T, 8><<<grid, kCgThreads, 0, s>>>((int)n, crow, col, val, p, keep, ap, partial, scal);
  pcg_update_kernel<T><<<grid, kCgThreads, 0, s>>>((int)n, p, ap, x, r, partial, n_partial, scal, tiny);
  amg_vcycle_launch<T>(levels, n_levels, coarse_inv, n_coarse, r, z, s);
  pcg_dot_kernel<T><<<grid, kCgThreads, 0, s>>>((int)n, r, z, partial + n_partial);
  cg_direction_kernel<T><<<grid, kCgThreads, 0, s>>>((int)n, z, p, partial + n_partial, n_partial, scal, tiny);
  return check_launch();
}

}  // namespace tfem

extern "C" int tfem_amg_vcycle_f64(const tfem_amg_level* levels, int32_t n_levels, const double* coarse_inv, int64_t n_coarse,
                                   const double* r, double* z, void* stream) {
  return tfem::amg_vcycle<double>(levels, n_levels, coarse_inv, n_coarse, r, z, stream);
}

extern "C" int tfem_amg_vcycle_f32(const tfem_amg_level* levels, int32_t n_levels, const float* coarse_inv, int64_t n_coarse,
                                   const float* r, float* z, void* stream) {
  return tfem::amg_vcycle<float>(levels, n_levels, coarse_inv, n_coarse, r, z, stream);
}

extern "C" int tfem_pcg_iteration_f64(int64_t n, const int32_t* crow, const int32_t* col, const double* val, const uint8_t* keep,
                                      const tfem_amg_level* levels, int32_t n_levels, const double* coarse_inv, int64_t n_coarse,
                                      double* x, double* r, double* z, double* p, double* ap, double* partial, int32_t n_partial,
                                      double* scal, void* stream) {
  return tfem::pcg_iteration<double>(n, crow, col, val, keep, levels, n_levels, coarse_inv, n_coarse, x, r, z, p, ap, partial, n_partial,
                                     scal, stream);
}

extern "C" int tfem_pcg_iteration_f32(int64_t n, const int32_t* crow, const int32_t* col, const float* val, const uint8_t* keep,
                                      const tfem_amg_level* levels, int32_t n_levels, const float* coarse_inv, int64_t n_coarse,
                                      float* x, float* r, float* z, float* p, float* ap, float* partial, int32_t n_partial,
                                      float* scal, void* stream) {
  return tfem::pcg_iteration<float>(n, crow, col, val, keep, levels, n_levels, coarse_inv, n_coarse, x, r, z, p, ap, partial, n_partial,
                                    scal, stream);
}

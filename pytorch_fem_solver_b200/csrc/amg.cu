// Set-up of the smoothed-aggregation AMG preconditioner (DESIGN.md 8(f).1): strength of connection and the
// parallel MIS(2) aggregation of Bell, Dalton and Olson (SIAM J. Sci. Comput. 34(4), 2012).  Integer and
// deterministic: every sweep reads one buffer and writes another, so the result does not depend on scheduling,
// and oracle/amg_oracle.py reproduces it bit for bit.  The only atomics are integer counters.
#include <cub/cub.cuh>

#include "common.cuh"

namespace tfem {

constexpr uint64_t kStateShift = 61;
constexpr uint64_t kStateOut = 0, kStateUndecided = 1, kStateIn = 2;
constexpr uint64_t kLowMask = (uint64_t(1) << kStateShift) - 1;

// murmur3 finaliser of i * 0x9E3779B1 + salt * 0x85EBCA77 + 0x165667B1 (mod 2^32); oracle/amg_oracle.py hash32
__device__ __forceinline__ uint32_t amg_hash32(uint32_t i, uint32_t salt) {
  uint32_t h = i * 0x9E3779B1u + salt * 0x85EBCA77u + 0x165667B1u;
  h ^= h >> 16;
  h *= 0x85EBCA6Bu;
  h ^= h >> 13;
  h *= 0xC2B2AE35u;
  h ^= h >> 16;
  return h;
}

template <typename T>
__global__ void __launch_bounds__(256) amg_diag_kernel(int n, const int32_t* __restrict__ crow, const int32_t* __restrict__ col,
                                                      const T* __restrict__ val, T* __restrict__ diag) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  T d = T(0);
  for (int k = crow[i]; k < crow[i + 1]; ++k)
    if (col[k] == i) d = val[k];
  diag[i] = d;
}

// strong[k] = 1 for the off-diagonal entries with |a_ij| >= theta sqrt(|a_ii a_jj|)
template <typename T>
__global__ void __launch_bounds__(256) amg_strength_kernel(int n, const int32_t* __restrict__ crow, const int32_t* __restrict__ col,
                                                          const T* __restrict__ val, const T* __restrict__ diag, T theta,
                                                          uint8_t* __restrict__ strong) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const T di = diag[i];
  for (int k = crow[i]; k < crow[i + 1]; ++k) {
    const int j = col[k];
    strong[k] = (j != i && fabs(val[k]) >= theta * sqrt(fabs(di * diag[j]))) ? 1 : 0;
  }
}

// key = state << 61 | (hash32(i, level) >> 3) << 32 | i; nodes without a strong connection start OUT
__global__ void __launch_bounds__(256) mis2_init_kernel(int n, const int32_t* __restrict__ crow, const uint8_t* __restrict__ strong,
                                                        uint32_t level, uint64_t* __restrict__ key) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  bool has = false;
  for (int k = crow[i]; k < crow[i + 1]; ++k) has |= strong[k] != 0;
  const uint64_t state = has ? kStateUndecided : kStateOut;
  key[i] = (state << kStateShift) | (uint64_t(amg_hash32((uint32_t)i, level) >> 3) << 32) | (uint32_t)i;
}

// out[i] = max(in[i], max over strong neighbours j of in[j])
__global__ void __launch_bounds__(256) mis2_sweep_kernel(int n, const int32_t* __restrict__ crow, const int32_t* __restrict__ col,
                                                         const uint8_t* __restrict__ strong, const uint64_t* __restrict__ in,
                                                         uint64_t* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint64_t m = in[i];
  for (int k = crow[i]; k < crow[i + 1]; ++k)
    if (strong[k]) {
      const uint64_t v = in[col[k]];
      m = v > m ? v : m;
    }
  out[i] = m;
}

// undecided i: its own key is the maximum within distance 2 -> IN; the maximum is an IN node -> OUT
__global__ void __launch_bounds__(256) mis2_update_kernel(int n, const uint64_t* __restrict__ t, uint64_t* __restrict__ key,
                                                          int32_t* __restrict__ n_undecided) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  int still = 0;
  if (i < n) {
    const uint64_t k = key[i];
    if ((k >> kStateShift) == kStateUndecided) {
      const uint64_t m = t[i];
      if (m == k) key[i] = (k & kLowMask) | (kStateIn << kStateShift);
      else if ((m >> kStateShift) == kStateIn) key[i] = k & kLowMask;
      else still = 1;
    }
  }
  const int count = __syncthreads_count(still);
  if (threadIdx.x == 0 && count) atomicAdd(n_undecided, count);  // integer count: order does not matter
}

__global__ void __launch_bounds__(256) root_flag_kernel(int n, const uint64_t* __restrict__ key, int32_t* __restrict__ flag) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) flag[i] = (key[i] >> kStateShift) == kStateIn ? 1 : 0;
  if (i == n) flag[n] = 0;
}

// Among the strong neighbours j of i with accept(j), the one of the largest key (-1 if none)
template <typename Accept>
__device__ __forceinline__ int best_neighbour(int i, const int32_t* __restrict__ crow, const int32_t* __restrict__ col,
                                              const uint8_t* __restrict__ strong, const uint64_t* __restrict__ key, Accept accept) {
  bool found = false;
  uint64_t best = 0;
  for (int k = crow[i]; k < crow[i + 1]; ++k) {
    if (!strong[k]) continue;
    const int j = col[k];
    if (!accept(j)) continue;
    const uint64_t v = key[j];
    if (!found || v > best) best = v, found = true;
  }
  return found ? (int)(best & 0xFFFFFFFFu) : -1;
}

// Phase 1: roots take their rank among the roots; a node with a strong root neighbour joins the root of the largest
// key; nodes without strong connections get -1; the rest (distance 2 from every root) -2
__global__ void __launch_bounds__(256) aggregate_phase1_kernel(int n, const int32_t* __restrict__ crow, const int32_t* __restrict__ col,
                                                               const uint8_t* __restrict__ strong, const uint64_t* __restrict__ key,
                                                               const int32_t* __restrict__ ids, int32_t* __restrict__ agg1) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  if ((key[i] >> kStateShift) == kStateIn) {
    agg1[i] = ids[i];
    return;
  }
  bool has = false;
  for (int k = crow[i]; k < crow[i + 1]; ++k) has |= strong[k] != 0;
  if (!has) {
    agg1[i] = -1;
    return;
  }
  const int j = best_neighbour(i, crow, col, strong, key, [&](int c) { return (key[c] >> kStateShift) == kStateIn; });
  agg1[i] = j >= 0 ? ids[j] : -2;
}

// Phase 2: the remaining nodes join the aggregate of their assigned strong neighbour of the largest key
__global__ void __launch_bounds__(256) aggregate_phase2_kernel(int n, const int32_t* __restrict__ crow, const int32_t* __restrict__ col,
                                                               const uint8_t* __restrict__ strong, const uint64_t* __restrict__ key,
                                                               const int32_t* __restrict__ agg1, int32_t* __restrict__ agg) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int a = agg1[i];
  if (a != -2) {
    agg[i] = a;
    return;
  }
  const int j = best_neighbour(i, crow, col, strong, key, [&](int c) { return agg1[c] >= 0; });
  agg[i] = j >= 0 ? agg1[j] : -1;
}

struct AggregateLayout {
  size_t flag, ids, agg1, cub_temp, cub_bytes, total;
};

inline size_t amg_align256(size_t v) { return (v + 255) & ~size_t(255); }

inline int aggregate_layout(int64_t n, AggregateLayout* out) {
  size_t scan = 0;
  if (cub::DeviceScan::ExclusiveSum(nullptr, scan, (const int32_t*)nullptr, (int32_t*)nullptr, (int)(n + 1)) != cudaSuccess)
    return TFEM_ERR_LAUNCH;
  size_t at = 0;
  out->flag = at;     at += amg_align256(4 * (size_t)(n + 1));
  out->ids = at;      at += amg_align256(4 * (size_t)(n + 1));
  out->agg1 = at;     at += amg_align256(4 * (size_t)n);
  out->cub_temp = at; at += amg_align256(scan);
  out->cub_bytes = scan;
  out->total = at;
  return TFEM_OK;
}

template <typename T>
int amg_strength(int64_t n, const int32_t* crow, const int32_t* col, const T* val, double theta, T* diag, uint8_t* strong,
                 void* stream) {
  if (n < 0 || !(theta >= 0.0)) return TFEM_ERR_BAD_ARG;
  if (n == 0) return TFEM_OK;
  if (!crow || !col || !val || !diag || !strong) return TFEM_ERR_BAD_ARG;
  if (n >= kMaxIndex) return TFEM_ERR_TOO_LARGE;
  auto s = static_cast<cudaStream_t>(stream);
  amg_diag_kernel<T><<<blocks_for(n, 256), 256, 0, s>>>((int)n, crow, col, val, diag);
  amg_strength_kernel<T><<<blocks_for(n, 256), 256, 0, s>>>((int)n, crow, col, val, diag, T(theta), strong);
  return check_launch();
}

}  // namespace tfem

extern "C" int tfem_amg_strength_f64(int64_t n, const int32_t* crow, const int32_t* col, const double* val, double theta, double* diag,
                                     uint8_t* strong, void* stream) {
  return tfem::amg_strength<double>(n, crow, col, val, theta, diag, strong, stream);
}

extern "C" int tfem_amg_strength_f32(int64_t n, const int32_t* crow, const int32_t* col, const float* val, double theta, float* diag,
                                     uint8_t* strong, void* stream) {
  return tfem::amg_strength<float>(n, crow, col, val, theta, diag, strong, stream);
}

extern "C" int tfem_amg_mis2_round(int64_t n, const int32_t* crow, const int32_t* col, const uint8_t* strong, int32_t level, int init,
                                   uint64_t* key, uint64_t* scratch, int32_t* n_undecided, void* stream) {
  using namespace tfem;
  if (n < 0 || level < 0) return TFEM_ERR_BAD_ARG;
  if (n == 0) return TFEM_OK;
  if (!crow || !col || !strong || !key || !scratch || !n_undecided) return TFEM_ERR_BAD_ARG;
  if (n >= kMaxIndex) return TFEM_ERR_TOO_LARGE;
  auto s = static_cast<cudaStream_t>(stream);
  const unsigned grid = blocks_for(n, 256);
  if (init) mis2_init_kernel<<<grid, 256, 0, s>>>((int)n, crow, strong, (uint32_t)level, key);
  if (cudaMemsetAsync(n_undecided, 0, sizeof(int32_t), s) != cudaSuccess) return TFEM_ERR_LAUNCH;
  mis2_sweep_kernel<<<grid, 256, 0, s>>>((int)n, crow, col, strong, key, scratch);
  mis2_sweep_kernel<<<grid, 256, 0, s>>>((int)n, crow, col, strong, scratch, scratch + n);
  mis2_update_kernel<<<grid, 256, 0, s>>>((int)n, scratch + n, key, n_undecided);
  return check_launch();
}

extern "C" int tfem_amg_aggregate_workspace(int64_t n, int64_t* bytes) {
  if (n < 0 || !bytes) return TFEM_ERR_BAD_ARG;
  if (n >= tfem::kMaxIndex) return TFEM_ERR_TOO_LARGE;
  tfem::AggregateLayout lay{};
  const int status = tfem::aggregate_layout(n > 0 ? n : 1, &lay);
  if (status != TFEM_OK) return status;
  *bytes = (int64_t)lay.total;
  return TFEM_OK;
}

extern "C" int tfem_amg_aggregate(int64_t n, const int32_t* crow, const int32_t* col, const uint8_t* strong, const uint64_t* key,
                                  void* workspace, int64_t workspace_bytes, int32_t* agg, int32_t* n_agg, void* stream) {
  using namespace tfem;
  if (n <= 0) return TFEM_ERR_BAD_ARG;
  if (!crow || !col || !strong || !key || !workspace || !agg || !n_agg) return TFEM_ERR_BAD_ARG;
  if (n >= kMaxIndex) return TFEM_ERR_TOO_LARGE;
  AggregateLayout lay{};
  int status = aggregate_layout(n, &lay);
  if (status != TFEM_OK) return status;
  if ((size_t)workspace_bytes < lay.total) return TFEM_ERR_BAD_ARG;
  auto s = static_cast<cudaStream_t>(stream);
  unsigned char* ws = static_cast<unsigned char*>(workspace);
  int32_t* flag = reinterpret_cast<int32_t*>(ws + lay.flag);
  int32_t* ids = reinterpret_cast<int32_t*>(ws + lay.ids);
  int32_t* agg1 = reinterpret_cast<int32_t*>(ws + lay.agg1);
  size_t cub_bytes = lay.cub_bytes;
  root_flag_kernel<<<blocks_for(n + 1, 256), 256, 0, s>>>((int)n, key, flag);
  // ids[i] = rank of root i among the roots (index order); ids[n] = number of roots
  if (cub::DeviceScan::ExclusiveSum(ws + lay.cub_temp, cub_bytes, flag, ids, (int)(n + 1), s) != cudaSuccess) return TFEM_ERR_LAUNCH;
  aggregate_phase1_kernel<<<blocks_for(n, 256), 256, 0, s>>>((int)n, crow, col, strong, key, ids, agg1);
  aggregate_phase2_kernel<<<blocks_for(n, 256), 256, 0, s>>>((int)n, crow, col, strong, key, agg1, agg);
  if (cudaMemcpyAsync(n_agg, ids + n, sizeof(int32_t), cudaMemcpyDeviceToDevice, s) != cudaSuccess) return TFEM_ERR_LAUNCH;
  return check_launch();
}

// ---------------------------------------------------------------------------------------------
// Numeric refresh of a hierarchy for new values on its pattern (sparse.AmgHierarchy.refresh): the diagonal, the
// smoother operator S = I - w D^-1 A, and a gather with fill (the finest masked operator from the input values, and
// R = P^T from P).  Each rounds like the torch expression of sparse.amg it replaces, so a refresh reproduces a build.
// ---------------------------------------------------------------------------------------------
namespace tfem {

__device__ __forceinline__ double amg_rcp_rn(double a) { return __drcp_rn(a); }
__device__ __forceinline__ float amg_rcp_rn(float a) { return __frcp_rn(a); }
__device__ __forceinline__ double amg_mul_rn(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ float amg_mul_rn(float a, float b) { return __fmul_rn(a, b); }

// wdinv[i] = (1 / a_ii) * omega (torch's `omega / diag` is reciprocal, then product); s[k] = delta_ij - wdinv[i] a_ij
template <typename T>
__global__ void __launch_bounds__(256) amg_smoother_kernel(int n, const int32_t* __restrict__ crow, const int32_t* __restrict__ col,
                                                          const T* __restrict__ val, const T* __restrict__ diag, T omega,
                                                          T* __restrict__ wdinv, T* __restrict__ s_val) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const T w = amg_mul_rn(amg_rcp_rn(diag[i]), omega);
  wdinv[i] = w;
  for (int k = crow[i]; k < crow[i + 1]; ++k) s_val[k] = T(col[k] == i ? 1 : 0) - amg_mul_rn(w, val[k]);
}

template <typename T>
__global__ void __launch_bounds__(256) gather_kernel(int n, const int32_t* __restrict__ src, const T* __restrict__ in, T fill,
                                                    T* __restrict__ out) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n) return;
  const int s = __ldg(src + k);
  out[k] = s >= 0 ? __ldg(in + s) : fill;
}

template <typename T>
int amg_diag(int64_t n, const int32_t* crow, const int32_t* col, const T* val, T* diag, void* stream) {
  if (n < 0) return TFEM_ERR_BAD_ARG;
  if (n == 0) return TFEM_OK;
  if (!crow || !col || !val || !diag) return TFEM_ERR_BAD_ARG;
  if (n >= kMaxIndex) return TFEM_ERR_TOO_LARGE;
  amg_diag_kernel<T><<<blocks_for(n, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>((int)n, crow, col, val, diag);
  return check_launch();
}

template <typename T>
int amg_smoother(int64_t n, const int32_t* crow, const int32_t* col, const T* val, const T* diag, double omega, T* wdinv, T* s_val,
                 void* stream) {
  if (n < 0 || !(omega == omega)) return TFEM_ERR_BAD_ARG;
  if (n == 0) return TFEM_OK;
  if (!crow || !col || !val || !diag || !wdinv || !s_val) return TFEM_ERR_BAD_ARG;
  if (n >= kMaxIndex) return TFEM_ERR_TOO_LARGE;
  amg_smoother_kernel<T><<<blocks_for(n, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>((int)n, crow, col, val, diag, T(omega),
                                                                                              wdinv, s_val);
  return check_launch();
}

template <typename T>
int gather(int64_t n, const int32_t* src, const T* in, double fill, T* out, void* stream) {
  if (n < 0) return TFEM_ERR_BAD_ARG;
  if (n == 0) return TFEM_OK;
  if (!src || !in || !out) return TFEM_ERR_BAD_ARG;
  if (n >= kMaxIndex) return TFEM_ERR_TOO_LARGE;
  gather_kernel<T><<<blocks_for(n, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>((int)n, src, in, T(fill), out);
  return check_launch();
}

}  // namespace tfem

extern "C" int tfem_amg_diag_f64(int64_t n, const int32_t* crow, const int32_t* col, const double* val, double* diag, void* stream) {
  return tfem::amg_diag<double>(n, crow, col, val, diag, stream);
}

extern "C" int tfem_amg_diag_f32(int64_t n, const int32_t* crow, const int32_t* col, const float* val, float* diag, void* stream) {
  return tfem::amg_diag<float>(n, crow, col, val, diag, stream);
}

extern "C" int tfem_amg_smoother_f64(int64_t n, const int32_t* crow, const int32_t* col, const double* val, const double* diag,
                                     double omega, double* wdinv, double* s_val, void* stream) {
  return tfem::amg_smoother<double>(n, crow, col, val, diag, omega, wdinv, s_val, stream);
}

extern "C" int tfem_amg_smoother_f32(int64_t n, const int32_t* crow, const int32_t* col, const float* val, const float* diag,
                                     double omega, float* wdinv, float* s_val, void* stream) {
  return tfem::amg_smoother<float>(n, crow, col, val, diag, omega, wdinv, s_val, stream);
}

extern "C" int tfem_gather_f64(int64_t n, const int32_t* src, const double* in, double fill, double* out, void* stream) {
  return tfem::gather<double>(n, src, in, fill, out, stream);
}

extern "C" int tfem_gather_f32(int64_t n, const int32_t* src, const float* in, double fill, float* out, void* stream) {
  return tfem::gather<float>(n, src, in, fill, out, stream);
}

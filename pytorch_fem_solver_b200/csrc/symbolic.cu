// One-time integer set-up of the sparse system (SURVEY 8(a) row a10, 8(b) tfem_csr_symbolic): the sorted-unique CSR
// pattern of the COO index maps of basis/basis.py:64-85 and the stable COO -> CSR permutations the deterministic
// scatter kernels walk, entirely on the device: CUB radix sort of the 64-bit (row, col) keys (only the bits a key can
// have are sorted), run-length encoding, prefix sums and binary searches.  Replaces the torch program
// sort / unique_consecutive / cumsum / bincount of csr.build_pattern (kept there for CPU tensors and as the oracle of
// the bit-exactness test).
#include <cub/cub.cuh>

#include "common.cuh"

namespace tfem {

__global__ void iota_kernel(int32_t* out, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = (int32_t)i;
}

// col[i] = key[i] % n_dof for the nnz unique keys; seg[nnz] = total (closes the exclusive scan of the run lengths)
__global__ void split_keys_kernel(const int64_t* __restrict__ keys, const int64_t* __restrict__ nnz_ptr, int64_t n_dof, int64_t total,
                                  int32_t* __restrict__ col, int32_t* __restrict__ seg) {
  const int64_t nnz = *nnz_ptr;
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < nnz) col[i] = (int32_t)(keys[i] % n_dof);
  if (i == nnz) seg[nnz] = (int32_t)total;
}

// out[r] = number of sorted values < r * scale   (r = 0 .. n_dof): row pointers by binary search
template <typename K>
__global__ void lower_bound_kernel(const K* __restrict__ sorted, const int64_t* __restrict__ n_ptr, int64_t n_fixed, int64_t n_dof, int64_t scale,
                                   int32_t* __restrict__ out) {
  const int64_t n = n_ptr ? *n_ptr : n_fixed;
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r > n_dof) return;
  const int64_t target = r * scale;
  int64_t lo = 0, hi = n;
  while (lo < hi) {
    const int64_t mid = (lo + hi) >> 1;
    if ((int64_t)sorted[mid] < target) lo = mid + 1;
    else hi = mid;
  }
  out[r] = (int32_t)lo;
}

inline int bits_for(int64_t v) {  // bits needed to represent values < v
  int b = 1;
  while (b < 63 && (int64_t(1) << b) < v) ++b;
  return b;
}

struct SymbolicLayout {
  size_t keys_in, keys_sorted, vals_in, counts, form_in, form_sorted, lvals_in, cub_temp, cub_bytes, total;
};

inline size_t align256(size_t v) { return (v + 255) & ~size_t(255); }

inline int symbolic_layout(int64_t n_el, int64_t n_dof, SymbolicLayout* out) {
  const int64_t n9 = 9 * n_el, n3 = 3 * n_el;
  size_t sort_pairs = 0, sort_lin = 0, rle = 0, scan = 0;
  if (cub::DeviceRadixSort::SortPairs(nullptr, sort_pairs, (const int64_t*)nullptr, (int64_t*)nullptr, (const int32_t*)nullptr, (int32_t*)nullptr,
                                      (int)n9) != cudaSuccess)
    return TFEM_ERR_LAUNCH;
  if (cub::DeviceRadixSort::SortPairs(nullptr, sort_lin, (const int32_t*)nullptr, (int32_t*)nullptr, (const int32_t*)nullptr, (int32_t*)nullptr,
                                      (int)n3) != cudaSuccess)
    return TFEM_ERR_LAUNCH;
  if (cub::DeviceRunLengthEncode::Encode(nullptr, rle, (const int64_t*)nullptr, (int64_t*)nullptr, (int32_t*)nullptr, (int64_t*)nullptr, (int)n9) !=
      cudaSuccess)
    return TFEM_ERR_LAUNCH;
  if (cub::DeviceScan::ExclusiveSum(nullptr, scan, (const int32_t*)nullptr, (int32_t*)nullptr, (int)(n9 + 1)) != cudaSuccess) return TFEM_ERR_LAUNCH;
  size_t cub_bytes = sort_pairs;
  cub_bytes = sort_lin > cub_bytes ? sort_lin : cub_bytes;
  cub_bytes = rle > cub_bytes ? rle : cub_bytes;
  cub_bytes = scan > cub_bytes ? scan : cub_bytes;
  size_t at = 0;
  out->keys_in = at;     at += align256(8 * (size_t)n9);
  out->keys_sorted = at; at += align256(8 * (size_t)n9);
  out->vals_in = at;     at += align256(4 * (size_t)n9);
  out->counts = at;      at += align256(4 * (size_t)(n9 + 1));
  out->form_in = at;     at += align256(4 * (size_t)n3);
  out->form_sorted = at; at += align256(4 * (size_t)n3);
  out->lvals_in = at;    at += align256(4 * (size_t)n3);
  out->cub_temp = at;    at += align256(cub_bytes);
  out->cub_bytes = cub_bytes;
  out->total = at;
  (void)n_dof;
  return TFEM_OK;
}

}  // namespace tfem

extern "C" int tfem_coo_keys(int64_t n_el, const int32_t* dof_conn, int64_t n_dof, int64_t* keys, void* stream);

extern "C" int tfem_csr_symbolic_workspace(int64_t n_el, int64_t n_dof, int64_t* bytes) {
  if (n_el < 0 || n_dof < 0 || !bytes) return TFEM_ERR_BAD_ARG;
  if (9 * n_el > tfem::kMaxIndex) return TFEM_ERR_TOO_LARGE;
  tfem::SymbolicLayout lay{};
  const int status = tfem::symbolic_layout(n_el > 0 ? n_el : 1, n_dof, &lay);
  if (status != TFEM_OK) return status;
  *bytes = (int64_t)lay.total;
  return TFEM_OK;
}

extern "C" int tfem_csr_symbolic(int64_t n_el, const int32_t* dof_conn, int64_t n_dof, void* workspace, int64_t workspace_bytes, int32_t* crow,
                                 int32_t* col, int32_t* seg, int32_t* perm, int32_t* lin_seg, int32_t* lin_perm, int64_t* keys, int64_t* nnz,
                                 void* stream) {
  using namespace tfem;
  if (n_el <= 0 || n_dof <= 0) return TFEM_ERR_BAD_ARG;
  if (!dof_conn || !workspace || !crow || !col || !seg || !perm || !lin_seg || !lin_perm || !keys || !nnz) return TFEM_ERR_BAD_ARG;
  if (9 * n_el > kMaxIndex || n_dof > kMaxIndex) return TFEM_ERR_TOO_LARGE;
  SymbolicLayout lay{};
  int status = symbolic_layout(n_el, n_dof, &lay);
  if (status != TFEM_OK) return status;
  if ((size_t)workspace_bytes < lay.total) return TFEM_ERR_BAD_ARG;
  auto s = static_cast<cudaStream_t>(stream);
  unsigned char* ws = static_cast<unsigned char*>(workspace);
  int64_t* keys_in = reinterpret_cast<int64_t*>(ws + lay.keys_in);
  int64_t* keys_sorted = reinterpret_cast<int64_t*>(ws + lay.keys_sorted);
  int32_t* vals_in = reinterpret_cast<int32_t*>(ws + lay.vals_in);
  int32_t* counts = reinterpret_cast<int32_t*>(ws + lay.counts);
  int32_t* form_sorted = reinterpret_cast<int32_t*>(ws + lay.form_sorted);
  int32_t* lvals_in = reinterpret_cast<int32_t*>(ws + lay.lvals_in);
  void* cub_temp = ws + lay.cub_temp;
  size_t cub_bytes = lay.cub_bytes;
  const int64_t n9 = 9 * n_el, n3 = 3 * n_el;

  // ---- bilinear form: keys, stable sort with the entry index as payload, unique keys and their run lengths --------
  status = tfem_coo_keys(n_el, dof_conn, n_dof, keys_in, stream);
  if (status != TFEM_OK) return status;
  iota_kernel<<<blocks_for(n9, 256), 256, 0, s>>>(vals_in, n9);
  const int key_bits = bits_for(n_dof) * 2 < 63 ? bits_for(n_dof * n_dof) : 63;
  if (cub::DeviceRadixSort::SortPairs(cub_temp, cub_bytes, keys_in, keys_sorted, vals_in, perm, (int)n9, 0, key_bits, s) != cudaSuccess)
    return TFEM_ERR_LAUNCH;
  if (cudaMemsetAsync(counts, 0, 4 * (size_t)(n9 + 1), s) != cudaSuccess) return TFEM_ERR_LAUNCH;
  cub_bytes = lay.cub_bytes;
  if (cub::DeviceRunLengthEncode::Encode(cub_temp, cub_bytes, keys_sorted, keys, counts, nnz, (int)n9, s) != cudaSuccess) return TFEM_ERR_LAUNCH;
  cub_bytes = lay.cub_bytes;
  // seg[i] = first COO entry of unique key i (i < nnz); the run lengths behind nnz are zero, split_keys closes seg[nnz]
  if (cub::DeviceScan::ExclusiveSum(cub_temp, cub_bytes, counts, seg, (int)(n9 + 1), s) != cudaSuccess) return TFEM_ERR_LAUNCH;
  split_keys_kernel<<<blocks_for(n9 + 1, 256), 256, 0, s>>>(keys, nnz, n_dof, n9, col, seg);
  lower_bound_kernel<int64_t><<<blocks_for(n_dof + 1, 256), 256, 0, s>>>(keys, nnz, 0, n_dof, n_dof, crow);

  // ---- linear form: the 3 n_el (element, local vertex) entries sorted by DOF --------------------------------------
  iota_kernel<<<blocks_for(n3, 256), 256, 0, s>>>(lvals_in, n3);
  cub_bytes = lay.cub_bytes;
  if (cub::DeviceRadixSort::SortPairs(cub_temp, cub_bytes, dof_conn, form_sorted, lvals_in, lin_perm, (int)n3, 0, bits_for(n_dof), s) != cudaSuccess)
    return TFEM_ERR_LAUNCH;
  lower_bound_kernel<int32_t><<<blocks_for(n_dof + 1, 256), 256, 0, s>>>(form_sorted, nullptr, n3, n_dof, 1, lin_seg);
  return check_launch();
}

// ---------------------------------------------------------------------------------------------
// Deterministic expand-sort-reduce SpGEMM C = op(A) B (AMG set-up: P = S T, A P, R = P^T, R (A P)).
// Every product a_ik b_kj is written with its 64-bit key row * n_cols_c + col; a stable radix sort of the keys
// (only the bits a key can have) with the product index as payload, run-length encoding and a prefix sum give
// the CSR pattern, and tfem_scatter_bilinear sums each run left to right -- in product order, so C is bitwise
// reproducible with no float atomics.  op(A) = A^T takes the products of A entry (i, k) with row i of B, keyed
// (k, j); B == NULL stands for the identity (the transpose is then the same program on swapped keys).
// ---------------------------------------------------------------------------------------------
extern "C" int tfem_scatter_bilinear_f64(int64_t nnz, const int32_t* seg, const int32_t* perm, const double* local, double* csr_val,
                                         void* stream);
extern "C" int tfem_scatter_bilinear_f32(int64_t nnz, const int32_t* seg, const int32_t* perm, const float* local, float* csr_val,
                                         void* stream);

namespace tfem {

inline int scatter_bilinear(int64_t n, const int32_t* seg, const int32_t* perm, const double* v, double* out, void* s) {
  return tfem_scatter_bilinear_f64(n, seg, perm, v, out, s);
}
inline int scatter_bilinear(int64_t n, const int32_t* seg, const int32_t* perm, const float* v, float* out, void* s) {
  return tfem_scatter_bilinear_f32(n, seg, perm, v, out, s);
}

// products of row i of op(A): sum over its entries of the length of the B row they meet (1 without B)
__global__ void spgemm_count_kernel(int n_rows_a, const int32_t* __restrict__ a_crow, const int32_t* __restrict__ a_col, int transpose,
                                    const int32_t* __restrict__ b_crow, int32_t* __restrict__ counts) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i > n_rows_a) return;
  if (i == n_rows_a) {
    counts[i] = 0;
    return;
  }
  const int begin = a_crow[i], end = a_crow[i + 1];
  int c = end - begin;
  if (b_crow != nullptr) {
    if (transpose) {
      c *= b_crow[i + 1] - b_crow[i];
    } else {
      c = 0;
      for (int k = begin; k < end; ++k) c += b_crow[a_col[k] + 1] - b_crow[a_col[k]];
    }
  }
  counts[i] = c;
}

template <typename T>
__global__ void spgemm_expand_kernel(int n_rows_a, const int32_t* __restrict__ a_crow, const int32_t* __restrict__ a_col,
                                     const T* __restrict__ a_val, int transpose, const int32_t* __restrict__ b_crow,
                                     const int32_t* __restrict__ b_col, const T* __restrict__ b_val, int64_t n_cols_c,
                                     const int32_t* __restrict__ offset, int64_t capacity, int64_t* __restrict__ keys,
                                     int32_t* __restrict__ index, T* __restrict__ prod) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_rows_a) return;
  int64_t at = offset[i];
  for (int k = a_crow[i]; k < a_crow[i + 1]; ++k) {
    const int j = a_col[k];
    const T a = a_val[k];
    const int64_t row = transpose ? j : i;
    if (b_crow == nullptr) {
      if (at < capacity) {
        keys[at] = row * n_cols_c + (transpose ? i : j);
        index[at] = (int32_t)at;
        prod[at] = a;
      }
      ++at;
      continue;
    }
    const int brow = transpose ? i : j;
    for (int q = b_crow[brow]; q < b_crow[brow + 1]; ++q, ++at) {
      if (at >= capacity) continue;
      keys[at] = row * n_cols_c + b_col[q];
      index[at] = (int32_t)at;
      prod[at] = a * b_val[q];
    }
  }
}

struct SpgemmLayout {
  size_t counts, offset, keys_in, keys_sorted, index, perm, prod, runs, seg, unique, cub_temp, cub_bytes, total;
};

inline int spgemm_layout(int64_t n_rows_a, int64_t n_products, SpgemmLayout* out) {
  size_t sort = 0, rle = 0, scan_rows = 0, scan_runs = 0;
  if (cub::DeviceRadixSort::SortPairs(nullptr, sort, (const int64_t*)nullptr, (int64_t*)nullptr, (const int32_t*)nullptr, (int32_t*)nullptr,
                                      (int)n_products) != cudaSuccess)
    return TFEM_ERR_LAUNCH;
  if (cub::DeviceRunLengthEncode::Encode(nullptr, rle, (const int64_t*)nullptr, (int64_t*)nullptr, (int32_t*)nullptr, (int64_t*)nullptr,
                                         (int)n_products) != cudaSuccess)
    return TFEM_ERR_LAUNCH;
  if (cub::DeviceScan::ExclusiveSum(nullptr, scan_rows, (const int32_t*)nullptr, (int32_t*)nullptr, (int)(n_rows_a + 1)) != cudaSuccess)
    return TFEM_ERR_LAUNCH;
  if (cub::DeviceScan::ExclusiveSum(nullptr, scan_runs, (const int32_t*)nullptr, (int32_t*)nullptr, (int)(n_products + 1)) != cudaSuccess)
    return TFEM_ERR_LAUNCH;
  size_t cub_bytes = sort;
  cub_bytes = rle > cub_bytes ? rle : cub_bytes;
  cub_bytes = scan_rows > cub_bytes ? scan_rows : cub_bytes;
  cub_bytes = scan_runs > cub_bytes ? scan_runs : cub_bytes;
  const size_t np = (size_t)n_products;
  size_t at = 0;
  out->counts = at;      at += align256(4 * (size_t)(n_rows_a + 1));
  out->offset = at;      at += align256(4 * (size_t)(n_rows_a + 1));
  out->keys_in = at;     at += align256(8 * np);
  out->keys_sorted = at; at += align256(8 * np);
  out->index = at;       at += align256(4 * np);
  out->perm = at;        at += align256(4 * np);
  out->prod = at;        at += align256(8 * np);  // sized for fp64 products
  out->runs = at;        at += align256(4 * (np + 1));
  out->seg = at;         at += align256(4 * (np + 1));
  out->unique = at;      at += align256(8 * np);
  out->cub_temp = at;    at += align256(cub_bytes);
  out->cub_bytes = cub_bytes;
  out->total = at;
  return TFEM_OK;
}

template <typename T>
int csr_spgemm(int64_t n_rows_a, const int32_t* a_crow, const int32_t* a_col, const T* a_val, int transpose, const int32_t* b_crow,
               const int32_t* b_col, const T* b_val, int64_t n_rows_c, int64_t n_cols_c, int64_t n_products, void* workspace,
               int64_t workspace_bytes, int32_t* c_crow, int32_t* c_col, T* c_val, int64_t* c_nnz, void* stream) {
  if (n_rows_a < 0 || n_rows_c < 0 || n_cols_c <= 0 || n_products < 0 || (transpose != 0 && transpose != 1)) return TFEM_ERR_BAD_ARG;
  if (!a_crow || !workspace || !c_crow || !c_nnz) return TFEM_ERR_BAD_ARG;
  if ((n_products > 0 || n_rows_a > 0) && (!a_col || !a_val)) return TFEM_ERR_BAD_ARG;
  if (b_crow != nullptr && (!b_col || !b_val)) return TFEM_ERR_BAD_ARG;
  if (n_products > 0 && (!c_col || !c_val)) return TFEM_ERR_BAD_ARG;
  if (n_rows_a >= kMaxIndex || n_rows_c >= kMaxIndex || n_cols_c >= kMaxIndex || n_products >= kMaxIndex) return TFEM_ERR_TOO_LARGE;
  SpgemmLayout lay{};
  int status = spgemm_layout(n_rows_a, n_products > 0 ? n_products : 1, &lay);
  if (status != TFEM_OK) return status;
  if ((size_t)workspace_bytes < lay.total) return TFEM_ERR_BAD_ARG;
  auto s = static_cast<cudaStream_t>(stream);
  if (n_products == 0) {
    if (cudaMemsetAsync(c_crow, 0, 4 * (size_t)(n_rows_c + 1), s) != cudaSuccess) return TFEM_ERR_LAUNCH;
    if (cudaMemsetAsync(c_nnz, 0, sizeof(int64_t), s) != cudaSuccess) return TFEM_ERR_LAUNCH;
    return check_launch();
  }
  unsigned char* ws = static_cast<unsigned char*>(workspace);
  int32_t* counts = reinterpret_cast<int32_t*>(ws + lay.counts);
  int32_t* offset = reinterpret_cast<int32_t*>(ws + lay.offset);
  int64_t* keys_in = reinterpret_cast<int64_t*>(ws + lay.keys_in);
  int64_t* keys_sorted = reinterpret_cast<int64_t*>(ws + lay.keys_sorted);
  int32_t* index = reinterpret_cast<int32_t*>(ws + lay.index);
  int32_t* perm = reinterpret_cast<int32_t*>(ws + lay.perm);
  T* prod = reinterpret_cast<T*>(ws + lay.prod);
  int32_t* runs = reinterpret_cast<int32_t*>(ws + lay.runs);
  int32_t* seg = reinterpret_cast<int32_t*>(ws + lay.seg);
  int64_t* unique = reinterpret_cast<int64_t*>(ws + lay.unique);
  void* cub_temp = ws + lay.cub_temp;
  size_t cub_bytes = lay.cub_bytes;

  spgemm_count_kernel<<<blocks_for(n_rows_a + 1, 256), 256, 0, s>>>((int)n_rows_a, a_crow, a_col, transpose, b_crow, counts);
  if (cub::DeviceScan::ExclusiveSum(cub_temp, cub_bytes, counts, offset, (int)(n_rows_a + 1), s) != cudaSuccess) return TFEM_ERR_LAUNCH;
  spgemm_expand_kernel<T><<<blocks_for(n_rows_a, 256), 256, 0, s>>>((int)n_rows_a, a_crow, a_col, a_val, transpose, b_crow, b_col, b_val,
                                                                     n_cols_c, offset, n_products, keys_in, index, prod);
  cub_bytes = lay.cub_bytes;
  if (cub::DeviceRadixSort::SortPairs(cub_temp, cub_bytes, keys_in, keys_sorted, index, perm, (int)n_products, 0,
                                      bits_for(n_rows_c * n_cols_c), s) != cudaSuccess)
    return TFEM_ERR_LAUNCH;
  if (cudaMemsetAsync(runs, 0, 4 * (size_t)(n_products + 1), s) != cudaSuccess) return TFEM_ERR_LAUNCH;
  cub_bytes = lay.cub_bytes;
  if (cub::DeviceRunLengthEncode::Encode(cub_temp, cub_bytes, keys_sorted, unique, runs, c_nnz, (int)n_products, s) != cudaSuccess)
    return TFEM_ERR_LAUNCH;
  cub_bytes = lay.cub_bytes;
  // seg[p] = first sorted product of entry p; entries past nnz have empty runs and sum to zero
  if (cub::DeviceScan::ExclusiveSum(cub_temp, cub_bytes, runs, seg, (int)(n_products + 1), s) != cudaSuccess) return TFEM_ERR_LAUNCH;
  status = scatter_bilinear(n_products, seg, perm, prod, c_val, stream);
  if (status != TFEM_OK) return status;
  split_keys_kernel<<<blocks_for(n_products + 1, 256), 256, 0, s>>>(unique, c_nnz, n_cols_c, n_products, c_col, seg);
  lower_bound_kernel<int64_t><<<blocks_for(n_rows_c + 1, 256), 256, 0, s>>>(unique, c_nnz, 0, n_rows_c, n_cols_c, c_crow);
  return check_launch();
}

}  // namespace tfem

extern "C" int tfem_csr_spgemm_workspace(int64_t n_rows_a, int64_t n_products, int64_t* bytes) {
  if (n_rows_a < 0 || n_products < 0 || !bytes) return TFEM_ERR_BAD_ARG;
  if (n_rows_a >= tfem::kMaxIndex || n_products >= tfem::kMaxIndex) return TFEM_ERR_TOO_LARGE;
  tfem::SpgemmLayout lay{};
  const int status = tfem::spgemm_layout(n_rows_a, n_products > 0 ? n_products : 1, &lay);
  if (status != TFEM_OK) return status;
  *bytes = (int64_t)lay.total;
  return TFEM_OK;
}

extern "C" int tfem_csr_spgemm_f64(int64_t n_rows_a, const int32_t* a_crow, const int32_t* a_col, const double* a_val, int transpose,
                                   const int32_t* b_crow, const int32_t* b_col, const double* b_val, int64_t n_rows_c, int64_t n_cols_c,
                                   int64_t n_products, void* workspace, int64_t workspace_bytes, int32_t* c_crow, int32_t* c_col,
                                   double* c_val, int64_t* c_nnz, void* stream) {
  return tfem::csr_spgemm<double>(n_rows_a, a_crow, a_col, a_val, transpose, b_crow, b_col, b_val, n_rows_c, n_cols_c, n_products, workspace,
                                  workspace_bytes, c_crow, c_col, c_val, c_nnz, stream);
}

extern "C" int tfem_csr_spgemm_f32(int64_t n_rows_a, const int32_t* a_crow, const int32_t* a_col, const float* a_val, int transpose,
                                   const int32_t* b_crow, const int32_t* b_col, const float* b_val, int64_t n_rows_c, int64_t n_cols_c,
                                   int64_t n_products, void* workspace, int64_t workspace_bytes, int32_t* c_crow, int32_t* c_col,
                                   float* c_val, int64_t* c_nnz, void* stream) {
  return tfem::csr_spgemm<float>(n_rows_a, a_crow, a_col, a_val, transpose, b_crow, b_col, b_val, n_rows_c, n_cols_c, n_products, workspace,
                                 workspace_bytes, c_crow, c_col, c_val, c_nnz, stream);
}

// ---------------------------------------------------------------------------------------------
// Numeric-only SpGEMM: the values of C = A B on a known pattern (c_crow, c_col sorted within rows, as
// tfem_csr_spgemm returns it), for a refresh of the AMG hierarchy with new values (sparse.AmgHierarchy.refresh).
// Bitwise equal to tfem_csr_spgemm's c_val: each entry is +0 plus its products added left to right in expansion
// order (A-row entries in stored order, then B-row entries in stored order) -- the order the stable sort gives the
// segmented sum -- and each product is rounded on its own (__dmul_rn / __fmul_rn: no contraction into an FMA).
// One warp per C row.  The warp takes the products of one A entry 32 at a time; each lane forms one product and finds
// its C slot by binary search; then every lane walks the staged products in order and adds those of the slots it
// owns (slot = lane + 32 t) to registers.  Rows longer than 32 * kNumericSlots run in several passes over the same
// products.  No sort, no workspace, no float atomics; products whose column C's row lacks are dropped and counted.
// ---------------------------------------------------------------------------------------------
namespace tfem {

constexpr int kNumericSlots = 4;  // C slots per lane and pass: rows up to 128 entries in one pass

__device__ __forceinline__ double mul_rn(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ float mul_rn(float a, float b) { return __fmul_rn(a, b); }

template <typename T>
__global__ void __launch_bounds__(256) spgemm_numeric_kernel(int n_rows, const int32_t* __restrict__ a_crow, const int32_t* __restrict__ a_col,
                                                             const T* __restrict__ a_val, const int32_t* __restrict__ b_crow,
                                                             const int32_t* __restrict__ b_col, const T* __restrict__ b_val,
                                                             const int32_t* __restrict__ c_crow, const int32_t* __restrict__ c_col,
                                                             T* __restrict__ c_val, int32_t* __restrict__ n_missing) {
  const int row = (int)(((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= n_rows) return;  // warp-uniform
  const int c_begin = __ldg(c_crow + row), c_len = __ldg(c_crow + row + 1) - c_begin;
  const int a_begin = __ldg(a_crow + row), a_end = __ldg(a_crow + row + 1);
  const int32_t* cc = c_col + c_begin;
  int missing = 0;
  for (int chunk = 0; chunk == 0 || chunk < c_len; chunk += 32 * kNumericSlots) {
    T acc[kNumericSlots];
#pragma unroll
    for (int t = 0; t < kNumericSlots; ++t) acc[t] = T(0);
    for (int k = a_begin; k < a_end; ++k) {
      const int j = __ldg(a_col + k);
      const T a = __ldg(a_val + k);
      const int b_begin = __ldg(b_crow + j), b_end = __ldg(b_crow + j + 1);
      for (int base = b_begin; base < b_end; base += 32) {
        const int q = base + lane;
        int slot = -1;
        T prod = T(0);
        if (q < b_end) {
          prod = mul_rn(a, __ldg(b_val + q));
          const int c = __ldg(b_col + q);
          int lo = 0, hi = c_len;
          while (lo < hi) {
            const int mid = (lo + hi) >> 1;
            if (__ldg(cc + mid) < c) lo = mid + 1;
            else hi = mid;
          }
          if (lo < c_len && __ldg(cc + lo) == c) slot = lo - chunk;
          else if (chunk == 0) ++missing;
        }
        const int staged = min(32, b_end - base);
        for (int s = 0; s < staged; ++s) {
          const int sl = __shfl_sync(0xffffffffu, slot, s);
          const T p = __shfl_sync(0xffffffffu, prod, s);
#pragma unroll
          for (int t = 0; t < kNumericSlots; ++t)
            if (sl == lane + 32 * t) acc[t] += p;
        }
      }
    }
#pragma unroll
    for (int t = 0; t < kNumericSlots; ++t) {
      const int sl = chunk + lane + 32 * t;
      if (sl < c_len) c_val[c_begin + sl] = acc[t];
    }
  }
  missing = __reduce_add_sync(0xffffffffu, missing);
  if (lane == 0 && missing) atomicAdd(n_missing, missing);  // integer count: order does not matter
}

template <typename T>
int csr_spgemm_numeric(int64_t n_rows, const int32_t* a_crow, const int32_t* a_col, const T* a_val, const int32_t* b_crow,
                       const int32_t* b_col, const T* b_val, const int32_t* c_crow, const int32_t* c_col, T* c_val, int32_t* n_missing,
                       void* stream) {
  if (n_rows < 0) return TFEM_ERR_BAD_ARG;
  if (n_rows == 0) return TFEM_OK;
  if (!a_crow || !a_col || !a_val || !b_crow || !b_col || !b_val || !c_crow || !c_col || !c_val || !n_missing) return TFEM_ERR_BAD_ARG;
  if (n_rows > kMaxIndex / 32) return TFEM_ERR_TOO_LARGE;
  spgemm_numeric_kernel<T><<<blocks_for(n_rows * 32, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      (int)n_rows, a_crow, a_col, a_val, b_crow, b_col, b_val, c_crow, c_col, c_val, n_missing);
  return check_launch();
}

}  // namespace tfem

extern "C" int tfem_csr_spgemm_numeric_f64(int64_t n_rows, const int32_t* a_crow, const int32_t* a_col, const double* a_val,
                                           const int32_t* b_crow, const int32_t* b_col, const double* b_val, const int32_t* c_crow,
                                           const int32_t* c_col, double* c_val, int32_t* n_missing, void* stream) {
  return tfem::csr_spgemm_numeric<double>(n_rows, a_crow, a_col, a_val, b_crow, b_col, b_val, c_crow, c_col, c_val, n_missing, stream);
}

extern "C" int tfem_csr_spgemm_numeric_f32(int64_t n_rows, const int32_t* a_crow, const int32_t* a_col, const float* a_val,
                                           const int32_t* b_crow, const int32_t* b_col, const float* b_val, const int32_t* c_crow,
                                           const int32_t* c_col, float* c_val, int32_t* n_missing, void* stream) {
  return tfem::csr_spgemm_numeric<float>(n_rows, a_crow, a_col, a_val, b_crow, b_col, b_val, c_crow, c_col, c_val, n_missing, stream);
}

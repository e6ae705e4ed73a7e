/*
 * tfem_b200.h -- C ABI of the B200-native element-assembly hot path of torch_fem.
 *
 * The reference (Nicolas-Zamorano/pytorch_fem_solver, package `torch_fem`) is pure
 * Python/PyTorch and has no FFI of its own; the boundary is its Python object API
 * (SURVEY.md section 8(b)).  Every entry point below replaces the tensor program of
 * the reference method it cites (paths relative to the reference's `torch_fem/`).
 * The Python package binds these symbols with ctypes and registers them as
 * `torch.library` custom ops (pytorch_fem_solver_b200/ops.py); INTEGRATION.md shows
 * the binding a maintainer of the reference would add.
 *
 * Conventions
 *   - plain C: device pointers, sizes, scalars; no torch / C++ types.
 *   - every `T*` is a DEVICE pointer unless the name says `host`; T is double for the
 *     `_f64` symbols and float for `_f32` (same argument lists; declared by macro).
 *   - indices are int32_t; element/vertex counts are int64_t.
 *   - the last argument is a `cudaStream_t` passed as `void*`; calls only enqueue work:
 *     they never allocate, free, synchronise or throw, and are re-entrant.
 *   - return value: TFEM_OK (0) or a negative tfem_status.
 *   - batched meshes (MeshesTri / Patches / FracturesTri) are passed flattened:
 *     element e belongs to mesh  m = e / n_el_per_mesh  and its geometry vertex ids are
 *     conn[e][k] + m * n_vert_per_mesh.  A single mesh has n_el_per_mesh == n_el.
 *   - fracture maps are optional (NULL for planar meshes): frac_jac [n_mesh,3,2],
 *     frac_inv [n_mesh,2,3], frac_det [n_mesh], frac_t [n_mesh,3].  With maps the
 *     spatial dimension d of points / gradients is 3, otherwise 2.
 *   - any OUTPUT pointer may be NULL, in which case that output is skipped.
 */
#ifndef TFEM_B200_H
#define TFEM_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum tfem_status {
  TFEM_OK = 0,
  TFEM_ERR_BAD_ARG = -1,      /* NULL required pointer, negative size, unknown enum */
  TFEM_ERR_UNSUPPORTED = -2,  /* e.g. quadrature order outside the reference's tables */
  TFEM_ERR_LAUNCH = -3,       /* cudaGetLastError() != cudaSuccess after enqueue */
  TFEM_ERR_TOO_LARGE = -4     /* a count does not fit the 32-bit index type */
} tfem_status;

/* Source term f evaluated inside the kernels at the mapped quadrature points.
 * Covers the load used by every reference test/example
 * (tests/test_assembly.py:75-84, examples/example_weak.py:59-75). */
typedef enum tfem_source_kind {
  TFEM_SRC_NONE = 0,     /* f == 0 */
  TFEM_SRC_SAMPLED = 1,  /* f given at the quadrature points: f_q[n_el, n_q]       */
  TFEM_SRC_CONST = 2,    /* f == p[0]                                               */
  TFEM_SRC_SINSIN = 3    /* f == p[0] * sin(p[1]*x) * sin(p[2]*y)                   */
} tfem_source_kind;

typedef struct tfem_source {
  int32_t kind;
  double p[4];
} tfem_source;

/* Which bilinear form the fused kernels integrate: alpha * grad u . grad v + beta * u v
 * (examples/example_weak.py:78-81, tests/test_assembly.py:68-73). */
typedef struct tfem_bilinear {
  double alpha; /* stiffness coefficient */
  double beta;  /* mass coefficient      */
} tfem_bilinear;

/* Tile plan (format v2) of the fused assembly kernel (all pointers DEVICE memory, built once per mesh by
 * pytorch_fem_solver_b200/tileplan.py; see DESIGN.md "tile plan").
 * A tile owns a set of CSR rows; its elements are all elements touching those rows.  The index data of
 * a tile are split into a TEMPLATE -- the tile-local structure, which depends on the mesh topology
 * around the tile only and is shared by all congruent tiles (every interior tile of a lattice-numbered
 * mesh) -- and a small per-tile INSTANCE.  Blobs are 32-bit words, 16 B aligned and whole 16 B units so
 * that one TMA bulk copy fetches each; every section is padded to a multiple of 4 words; 16-bit
 * sections are packed little-endian.
 *
 *   instance blob (one per tile)
 *     header[4]        n_vert, n_segs, n_rows, base_vertex (tile-local index of a vertex near the middle
 *                      of the tile: the source's sin/cos are evaluated once there and rotated to the
 *                      centroid of every tile element)
 *     vert[n_vert]     u32  row of `coords` of each tile-local vertex
 *     seg_start[n_segs] u32 csr_val offset of the first entry of each segment: a run of consecutive CSR
 *                      rows cut into pieces of at most 32 entries (one warp pass each)
 *     row_id[n_rows]   u32  global row (DOF) of each owned row, ascending
 *     elem_id[n_elem]  u32  (only with has_elem_ids) global id of each tile element, in the order of elem[]
 *   template, part TB (integration phase)
 *     header[8]        n_vert, n_elem, n_rows, n_segs, n_chunks, n_heavy, n_heavy_contrib, 0
 *     elem[n_elem]     u32  tile-local connectivity  v0 | v1<<10 | v2<<20
 *   template, part TC (reduction phase)
 *     pair[n_segs][32]     u32  one word per lane of each segment: lane l of segment s owns
 *                               csr_val[seg_start[s] + l].  lo 16 bits = first, hi 16 bits = second
 *                               contribution, each a CODE = byte offset (fp64) of a local value in the
 *                               CTA's local table, in increasing element id (the summation order of the
 *                               reference's index_put_/coalesce); code 0 = "no contribution" (a zero);
 *                               0xFFFFFFFF = lane without an entry, or entry summed elsewhere (row_diag or
 *                               the heavy list).  The table has R = max_elem + 2 rows (row 0 = zeros,
 *                               row 1 + p = the tile element at position p of elem[], last row = scratch):
 *                                 48 * row + 16 * k      diagonal term of local vertex k   (K00 K11 K22)
 *                                 48 * row + 16 * k + 8  load term of local vertex k
 *                                 od_base[m] + 8 * row   off-diagonal term m = 0, 1, 2     (K01 K12 K20)
 *                               (elem[] lists a tile's elements in ascending id, or even positions first
 *                               and odd positions second: whichever gives fewer shared-memory bank
 *                               conflicts; od_base likewise -- see tileplan._choose_layout)
 *     row_chunk[n_chunks][8] u16  chunk j < n_rows belongs to owned row j: 7 codes of the diagonal terms
 *                               of the elements around the row's vertex (ascending element id), padded
 *                               with 0; the load term sits 8 bytes further; the 8th value is the index of
 *                               the row's next chunk (rows with more than 7 elements), 0 = none
 *     row_diag[n_rows]     u16  entry code (segment * 32 + lane) of the row's diagonal when the row's
 *                               thread sums it (same element list as the load entry), else 0xFFFF
 *     heavy_seg[n_heavy+1] u16  offsets into heavy_contrib[] of the other entries with more than two
 *                               contributions (non-manifold edges, degenerate elements)
 *     heavy_contrib[n_heavy_contrib] u16  their codes
 *     heavy_pos[n_heavy]   u16  their entry codes (segment * 32 + lane)
 *   A CTA keeps ONE template resident in shared memory; TB is refetched after the integration phase of
 *   the previous tile and TC after its reduction phase, only when the template changes.               */
typedef struct tfem_tile_plan {
  int64_t n_tiles;           /* tiles this call processes (length of tile_list) */
  const int32_t* tile_list;  /* [n_tiles] ids of those tiles, in processing order (congruent tiles adjacent); lets one
                                plan be run in parts (interface tiles first, interior tiles while the exchange runs).
                                The first n_progress_tiles are dealt round-robin over the CTAs, the rest in contiguous
                                blocks (one per CTA), so that a CTA rarely changes template */
  const int32_t* tile_desc;  /* [all tiles][4]: instance word offset, instance words, template id, 0 */
  const int32_t* inst_blob;
  const int32_t* tpl_desc;   /* [templates][4]: TB word offset, TB words, TC word offset, TC words */
  const int32_t* tpl_blob;
  int32_t max_vert, max_elem, max_inst_words, max_tb_words, max_tc_words; /* per-tile maxima (shared-memory sizing) */
  int32_t has_elem_ids;     /* instances end with elem_id[n_elem]: the global id of every tile element in elem[] order
                               (needed by tfem_tri_p1_assemble_csr_ex with a sampled source or fracture metrics) */
  int32_t table_bytes;      /* size of the CTA's local table in fp64 bytes (the fp32 kernels use half) */
  int32_t od_base[3];       /* byte offsets of the off-diagonal arrays K01, K12, K20 inside the table (see below) */
  int32_t consumer_threads; /* kernel selector: 0 = library default (the role-specialised kernel, 12 integration +
                               12 reduction warps, one CTA per SM; plans too large for its shared memory run on the
                               classic kernel); 384 = classic kernel, 384 compute threads, two CTAs per SM;
                               100 * NB + NC = role-specialised kernel with NB + NC warps (1212 is built) */
  int32_t reserve_ctas;     /* CTA slots of the persistent grid left free so that kernels on other streams
                               (interface pack / signal / add) can run beside it; 0 = use every slot.  Counted in
                               slots of the classic kernel (two per SM): the role-specialised kernel leaves
                               (reserve_ctas + 1) / 2 SMs free */
  int32_t n_progress_tiles; /* the first n_progress_tiles tiles of the call (in tile_list order) report on
                               `progress` when they are finished: every reduction warp adds 1 after its stores
                               (release), so the counter grows by n_progress_tiles * 12 per call (12 = reduction
                               warps of both built kernels; in general NC, or consumer_threads / 32 for the
                               classic kernel); 0 = nobody reports */
  uint32_t* progress;       /* device counter, never reset by the library (callers wait for a growing target
                               with tfem_iface_pack_after); NULL = nobody reports */
} tfem_tile_plan;

int tfem_abi_version(void);
const char* tfem_status_string(int status);
/* Bind the calling thread to a device before enqueuing (the library links the static
 * CUDA runtime; the Python wrapper calls this with the tensors' device index). */
int tfem_set_device(int device);
/* Number of SMs of the current device (grid sizing of persistent kernels; 148 on B200). */
int tfem_sm_count(void);

/* One smoothed level of an AMG hierarchy (pytorch_fem_solver_b200/sparse.py `amg`; DESIGN.md 8(f).1), all pointers
 * DEVICE memory in the precision of the call (T = double for _f64, float for _f32).  Level l holds its operator
 * A [n x n], the prolongator P [n x n_coarse] and restriction R = P^T [n_coarse x n] as CSR (int32 crow / col),
 * wdinv [n] = omega / a_ii, and work vectors x [n] (the level's smoothed iterate), rc [n_coarse] (restricted
 * residual = right-hand side of level l + 1) and ec [n_coarse] (its correction = result of level l + 1).
 * n_coarse equals the n of the next level, or of the dense coarsest operator after the last level. */
typedef struct tfem_amg_level {
  int64_t n;
  int64_t n_coarse;
  const int32_t* a_crow;
  const int32_t* a_col;
  const void* a_val;
  const int32_t* p_crow;
  const int32_t* p_col;
  const void* p_val;
  const int32_t* r_crow;
  const int32_t* r_col;
  const void* r_val;
  const void* wdinv;
  void* x;
  void* rc;
  void* ec;
} tfem_amg_level;

#define TFEM_DECLARE(T, SUF)                                                                        \
  /* a1-a9: AbstractBasis._compute_integral_values (basis/abstract_basis.py:42-63) with          \
   * Basis._compute_jacobian_map/_integration_points/_integral_weights (basis/basis.py:87-96),   \
   * ElementTri.compute_det_and_inv_map/shape functions (element/element_tri.py:28-41,132-145), \
   * the gather of mesh/abstract_mesh.py:257-262 / mesh/meshes_tri.py:33-41, and the fracture   \
   * post-scaling of basis/fracture_basis.py:20-26,189-207.                                     \
   * inv_jac [n_el,2,d], v_grad [n_el,3,d], x_q [n_el,n_q,d], dx [n_el,n_q]. */                 \
  int tfem_tri_p1_geometry_##SUF(int64_t n_el, int64_t n_el_per_mesh, int64_t n_vert_per_mesh,     \
                                 const T* coords, const int32_t* conn, int quad_order,             \
                                 const T* frac_jac, const T* frac_inv, const T* frac_det,          \
                                 const T* frac_t, T* inv_jac, T* v_grad, T* x_q, T* dx,            \
                                 void* stream);                                                    \
  /* Edge variant: basis/interior_edges_basis.py:63-72, interior_edges_fracture_basis.py:65-86,  \
   * element/element_line.py:45-73.  edge_coords [n_edge,2,2] (2-D end points).                 \
   * inv_jac [n_edge], v_grad [n_edge,2], x_q [n_edge,n_q,d], dx [n_edge,n_q]. */               \
  int tfem_edge_p1_geometry_##SUF(int64_t n_edge, int64_t n_edge_per_mesh, const T* edge_coords,   \
                                  int quad_order, const T* frac_jac, const T* frac_det,            \
                                  const T* frac_t, T* inv_jac, T* v_grad, T* x_q, T* dx,           \
                                  void* stream);                                                   \
  /* `(f * dx).sum(-3)` of basis/abstract_basis.py:72,83,104 for an arbitrary user integrand:    \
   * local[e,c] = sum_q dx[e,q] * f[e*stride_e + q*stride_q + c], c < m (strides in elements;    \
   * a stride of 0 broadcasts, as the reference's broadcasting does). */                         \
  int tfem_quad_reduce_##SUF(int64_t n_el, int n_q, int m, const T* integrand, int64_t stride_e,    \
                             int64_t stride_q, const T* dx, T* local, void* stream);                \
  /* The local-to-global scatter of basis/abstract_basis.py:87-91,106-110, as a deterministic    \
   * segmented reduction instead of index_put_(accumulate=True):                                 \
   * out[p] = sum_{s in [seg[p], seg[p+1])} values[perm[s]], summed in increasing s.              \
   * With (seg, perm) = stable sort of `bilinear_form_idx` this yields the CSR value array,       \
   * with the sort of `linear_form_idx` the global vector. */                                     \
  int tfem_scatter_bilinear_##SUF(int64_t nnz, const int32_t* seg, const int32_t* perm,            \
                                  const T* local, T* csr_val, void* stream);                       \
  int tfem_scatter_linear_##SUF(int64_t n_dof, const int32_t* seg, const int32_t* perm,            \
                                const T* local, T* vec, void* stream);                             \
  /* Fused local forms (never materialising v, v_grad, x_q, dx):                                 \
   * local_mat[e,i,j] = sum_q dx (alpha grad phi_i . grad phi_j + beta phi_i phi_j)   [n_el,3,3]   \
   * local_vec[e,i]   = sum_q dx f(x_q) phi_i                                        [n_el,3]     \
   * Forms: examples/example_weak.py:78-81, tests/test_assembly.py:68-84. */                      \
  int tfem_tri_p1_local_forms_##SUF(int64_t n_el, int64_t n_el_per_mesh, int64_t n_vert_per_mesh,  \
                                    const T* coords, const int32_t* conn, int quad_order,          \
                                    const T* frac_jac, const T* frac_inv, const T* frac_det,       \
                                    const T* frac_t, const tfem_bilinear* host_form,               \
                                    const tfem_source* host_source,                                \
                                    const T* f_q, T* local_mat, T* local_vec, void* stream);       \
  /* The same local forms with coefficient fields sampled at the quadrature points:               \
   * local_mat[e,i,j] = (grad phi_i . grad phi_j) det sum_q w_q alpha_q[e,q]                      \
   *                  + det sum_q w_q beta_q[e,q] phi_i(q) phi_j(q)                  [n_el,3,3]   \
   * (on a fracture: tangential 3-D gradients, det includes det J_f); local_vec exactly as        \
   * tfem_tri_p1_local_forms writes it.  alpha_q, beta_q [n_el,n_q]; a NULL field takes the       \
   * matching constant of host_form (which may then be NULL only if both fields are given). */    \
  int tfem_tri_p1_weighted_local_forms_##SUF(int64_t n_el, int64_t n_el_per_mesh,                  \
                                             int64_t n_vert_per_mesh, const T* coords,             \
                                             const int32_t* conn, int quad_order,                  \
                                             const T* frac_jac, const T* frac_inv,                 \
                                             const T* frac_det, const T* frac_t,                   \
                                             const tfem_bilinear* host_form,                       \
                                             const tfem_source* host_source, const T* f_q,         \
                                             const T* alpha_q, const T* beta_q, T* local_mat,      \
                                             T* local_vec, void* stream);                          \
  /* Fused assembly to CSR + load vector in ONE pass over row tiles (BASELINE config 2):          \
   * csr_val[p] = sum over elements of alpha K_loc + beta M_loc, load[r] = sum of local loads,    \
   * each summed in increasing element order (deterministic, no atomics).  The tile plan is      \
   * built once from the connectivity by pytorch_fem_solver_b200/csr.py. */                      \
  int tfem_tri_p1_assemble_csr_##SUF(const tfem_tile_plan* host_plan, const T* coords,             \
                                     int quad_order, const tfem_bilinear* host_form,               \
                                     const tfem_source* host_source, T* csr_val, T* load,          \
                                     void* stream);                                                \
  /* The same launch for sources given AT THE QUADRATURE POINTS and for fracture networks:        \
   * f_q [n_el, n_q] (host_source->kind == TFEM_SRC_SAMPLED; what `Load(callable)` of every       \
   * reference call site reduces to, tests/test_assembly.py:79-84,                                \
   * examples/example_fractures_fem.py:102-116) is read per tile element through the plan's       \
   * elem_id section; frac_metric [n_mesh, 4] = (a00, a01, a11, det J_f) with                     \
   * a = J_f^+ J_f^+^T turns the planar forms into the tangential ones of                         \
   * basis/fracture_basis.py:20-26,189-197 (element e lies on fracture e / n_el_per_mesh).        \
   * Both NULL: identical to tfem_tri_p1_assemble_csr. */                                         \
  int tfem_tri_p1_assemble_csr_ex_##SUF(const tfem_tile_plan* host_plan, const T* coords,          \
                                        int quad_order, const tfem_bilinear* host_form,            \
                                        const tfem_source* host_source, const T* f_q,              \
                                        int64_t n_el_per_mesh, const T* frac_metric, T* csr_val,   \
                                        T* load, void* stream);                                    \
  /* Weak residual r_i = sum_q dx (f phi_i - grad phi_i . grad u) of                              \
   * examples/example_weak.py:64-75 / example_patches.py:102-113 /                               \
   * example_fracture_vpinns.py:104-113 integrated by basis/abstract_basis.py:95-112:            \
   * per-element part local_vec [n_el,3]; grad_u [n_el,n_q,d]. */                                 \
  int tfem_weak_residual_local_##SUF(int64_t n_el, int64_t n_el_per_mesh, int64_t n_vert_per_mesh, \
                                     const T* coords, const int32_t* conn, int quad_order,         \
                                     const T* frac_jac, const T* frac_inv, const T* frac_det,      \
                                     const T* frac_t, const tfem_source* host_source,              \
                                     const T* f_q, const T* grad_u, T* local_vec, void* stream);   \
  /* The same residual summed straight to the DOF vector r [n_dof] in ONE launch of the tiled      \
   * kernel (no per-element tensor, no scatter pass; rows sum their elements in increasing         \
   * element order): f_q [n_el,n_q] or NULL (f = 0), grad_u [n_el,n_q,d]; on a fracture network    \
   * frac_inv [n_mesh,2,3] = J_f^+ and frac_metric [n_mesh,4] as in assemble_csr_ex (d = 3), both  \
   * NULL on planar meshes (d = 2).  The plan must carry element ids (has_elem_ids). */            \
  int tfem_weak_residual_tiled_##SUF(const tfem_tile_plan* host_plan, const T* coords,             \
                                     int quad_order, const T* f_q, const T* grad_u,                \
                                     int64_t n_el_per_mesh, const T* frac_inv,                     \
                                     const T* frac_metric, T* r, void* stream);                    \
  /* Adjoint of the above w.r.t. grad_u (what autograd derives from index_put_/sum/matmul):       \
   * grad_u_bar[e,q,:] = -dx[e,q] * sum_i grad phi_i[e,:] * r_bar[dof_conn[e,i]]. */              \
  int tfem_weak_residual_bwd_##SUF(int64_t n_el, int64_t n_el_per_mesh, int64_t n_vert_per_mesh,   \
                                   const T* coords, const int32_t* conn, const int32_t* dof_conn,  \
                                   int quad_order, const T* frac_jac, const T* frac_inv,           \
                                   const T* frac_det, const T* r_bar, T* grad_u_bar,               \
                                   void* stream);                                                  \
  /* The same residual for a BATCH OF SMALL MESHES whose DOFs are private to each mesh           \
   * (PatchesBasis, basis/patches_basis.py:44-105; examples/example_patches.py:102-113), summed   \
   * to r [n_mesh, n_vert_per_mesh] in ONE launch: a lane group per mesh, a lane per element,     \
   * DOF sums by warp shuffles in increasing element order.  n_el_per_mesh <= 8,                  \
   * n_vert_per_mesh <= 16, planar (d = 2); grad_u [n_mesh * n_el_per_mesh, n_q, 2].  Its adjoint \
   * is tfem_weak_residual_bwd with dof_conn[e][k] = mesh * n_vert_per_mesh + conn[e][k]. */      \
  int tfem_batched_weak_residual_##SUF(int64_t n_mesh, int n_el_per_mesh, int n_vert_per_mesh,     \
                                       const T* coords, const int32_t* conn, int quad_order,       \
                                       const tfem_source* host_source, const T* f_q,               \
                                       const T* grad_u, T* r, void* stream);                       \
  /* H1 error functional of examples/example_weak.py:113-124 integrated by                       \
   * basis/abstract_basis.py:65-72, fused (no integrand, no dx tensor):                          \
   * out[e] = sum_q dx_q ((u_ex - u)^2 + |grad u_ex - grad u|^2); fields sampled at the           \
   * quadrature points: u, u_ex [n_el,n_q]; grad_u, grad_ex [n_el,n_q,d]; frac_det [n_mesh] or   \
   * NULL (planar). */                                                                           \
  int tfem_h1_error_##SUF(int64_t n_el, int64_t n_el_per_mesh, int64_t n_vert_per_mesh,            \
                          const T* coords, const int32_t* conn, int quad_order, const T* frac_det, \
                          int d, const T* u, const T* grad_u, const T* u_ex, const T* grad_ex,     \
                          T* out, void* stream);                                                   \
  /* Basis.interpolate(self, u) (basis/basis.py:105-112,149-159; fracture_basis.py:214-223):     \
   * val[e,q] = sum_i u[dof_conn[e,i]] phi_i(q),  grad[e,:] = sum_i u[...] grad phi_i[e,:]. */    \
  int tfem_interp_cells_##SUF(int64_t n_el, const int32_t* dof_conn, const T* v_grad, int d,       \
                              int quad_order, const T* u, T* val, T* grad, void* stream);          \
  /* Basis.interpolate(InteriorEdgesBasis, u) (basis/basis.py:114-159;                            \
   * fracture_basis.py:225-257; element/abstract_element.py:18-26): both cells of every          \
   * interior edge evaluated at the edge quadrature points.  edge_cells [n_edge,2] are cell ids   \
   * local to the mesh of the edge, conn [n_el,3] the ids used to index `u`,                      \
   * first_vertex [n_el,d], inv_jac [n_el,2,d], x_q [n_edge,n_q,d].                              \
   * val [n_edge,2,n_q], grad [n_edge,2,d]. */                                                    \
  int tfem_interp_edges_##SUF(int64_t n_edge, int64_t n_edge_per_mesh, int64_t n_el_per_mesh,      \
                              const int32_t* edge_cells, const int32_t* conn,                      \
                              const T* first_vertex, const T* inv_jac, int d, const T* x_q,        \
                              int n_q, const T* u, T* val, T* grad, void* stream);                 \
  /* Adjoints of the two interpolations w.r.t. the nodal vector (what autograd derives from the   \
   * gather + multiply + sum of basis/basis.py:149-159 when the nodal values come from a network,\
   * examples/example_jump.py:58,75-87).  They produce the per-element / per-(edge, side) part     \
   * local[., i] = sum_q val_bar[., q] phi_i(q) + sum_c grad_bar[., c] grad phi_i[c];              \
   * the deterministic scatter (tfem_scatter_linear) then sums it into u_bar.                     \
   * val_bar / grad_bar may be NULL (treated as zero). */                                         \
  int tfem_interp_cells_bwd_##SUF(int64_t n_el, const T* v_grad, int d, int quad_order,            \
                                  const T* val_bar, const T* grad_bar, T* local, void* stream);    \
  int tfem_interp_edges_bwd_##SUF(int64_t n_edge, int64_t n_edge_per_mesh, int64_t n_el_per_mesh,  \
                                  const int32_t* edge_cells, const T* first_vertex,                \
                                  const T* inv_jac, int d, const T* x_q, int n_q,                  \
                                  const T* val_bar, const T* grad_bar, T* local, void* stream);    \
  /* Jump estimator eta_E = sum_q dx h_E (grad u+ . n - grad u- . n)^2                            \
   * (examples/example_jump.py:75-87 integrated by basis/abstract_basis.py:65-72).              \
   * grad_edges [n_edge,2,d] from tfem_interp_edges, normals [n_edge,d], h_e [n_edge],           \
   * dx [n_edge,n_q]. */                                                                         \
  int tfem_edge_jump_##SUF(int64_t n_edge, int d, int n_q, const T* grad_edges, const T* normals,  \
                           const T* h_e, const T* dx, T* eta, void* stream);                       \
  /* Multi-GPU interface exchange (SURVEY.md 8(e)): gather interface entries into a             \
   * contiguous send buffer, and add a received buffer into the owner's entries                  \
   * (idx entries are unique, so no atomics). */                                                 \
  int tfem_iface_pack_##SUF(int64_t n, const int32_t* idx, const T* src, T* buf, void* stream);    \
  /* The same gather, started early: every block first waits (bounded spin, then trap) until the   \
   * device counter `progress` has reached `target` (wrap-safe), i.e. until the tiles holding the  \
   * interface rows of a tfem_tri_p1_assemble_csr call running beside it are complete.  `buf`      \
   * may be peer memory (NVLink). */                                                             \
  int tfem_iface_pack_after_##SUF(int64_t n, const int32_t* idx, const T* src, T* buf,             \
                                  const uint32_t* progress, uint32_t target, void* stream);        \
  int tfem_iface_unpack_add_##SUF(int64_t n, const int32_t* idx, const T* buf, T* dst,             \
                                  void* stream);                                                   \
  /* SURVEY.md 8(f).1 -- y = A x on the assembled CSR system, the operator of the iterative       \
   * solve that replaces the dense torch.linalg.solve of basis/abstract_basis.py:177-195 when   \
   * the matrix cannot be densified.  keep [n_rows] (0/1 bytes) or NULL: rows with keep == 0     \
   * (Dirichlet rows of AbstractBasis.reduce, abstract_basis.py:114-117) give y = 0. */          \
  int tfem_csr_spmv_##SUF(int64_t n_rows, const int32_t* crow, const int32_t* col, const T* val,   \
                          const T* x, const uint8_t* keep, T* y, void* stream);                    \
  /* One Jacobi-preconditioned conjugate-gradient iteration on (M A M) x = M b, M = diag(keep),   \
   * as three launches with the dot products reduced in a fixed order (bitwise reproducible).    \
   * State vectors x, r, z, p, ap [n]; inv_diag [n]; partial [2 * n_partial] scratch (n_partial  \
   * = number of thread blocks used, e.g. 8 per SM); scal [2]: before the FIRST call set          \
   * scal[1] = r.z (scal[0] is overwritten); after a call scal[1] holds the new r.z. */           \
  int tfem_cg_iteration_##SUF(int64_t n, const int32_t* crow, const int32_t* col, const T* val,    \
                              const uint8_t* keep, const T* inv_diag, T* x, T* r, T* z, T* p,      \
                              T* ap, T* partial, int32_t n_partial, T* scal, void* stream);      \
  /* The same iteration preconditioned by smoothed-aggregation AMG instead of Jacobi: SpMV + p.Ap   \
   * (the kernel of tfem_cg_iteration), x += alpha p and r -= alpha ap, z = M_AMG r (one V-cycle,   \
   * as tfem_amg_vcycle), partials of r.z, the new direction.  Same state and scal contract as      \
   * tfem_cg_iteration; levels / n_levels / coarse_inv / n_coarse as in tfem_amg_vcycle, and the    \
   * finest level (or the coarse operator when n_levels == 0) must have n rows. */                  \
  int tfem_pcg_iteration_##SUF(int64_t n, const int32_t* crow, const int32_t* col, const T* val,   \
                               const uint8_t* keep, const tfem_amg_level* host_levels,             \
                               int32_t n_levels, const T* coarse_inv, int64_t n_coarse, T* x,      \
                               T* r, T* z, T* p, T* ap, T* partial, int32_t n_partial, T* scal,    \
                               void* stream);                                                      \
  /* One symmetric AMG V-cycle z = M_AMG r from a zero initial guess: on every level x = w D^-1 b,  \
   * b_c = R (b - A x), recursion, x += P e_c, y = x + w D^-1 (b - A x); the coarsest system is     \
   * solved by the dense inverse coarse_inv [n_coarse, n_coarse] (row-major, 1 <= n_coarse <=       \
   * 32768), one warp per row.  host_levels: HOST array of n_levels >= 0 levels, finest first (the   \
   * pointers inside are device memory; their work vectors are overwritten).  r, z [levels[0].n].   \
   * Fixed-order sums, no allocation, no synchronisation: bitwise reproducible and graph-capturable. \
   * TFEM_ERR_BAD_ARG for a NULL pointer or sizes that do not chain (levels[l].n_coarse ==           \
   * levels[l+1].n, last == n_coarse). */                                                          \
  int tfem_amg_vcycle_##SUF(const tfem_amg_level* host_levels, int32_t n_levels,                   \
                            const T* coarse_inv, int64_t n_coarse, const T* r, T* z,              \
                            void* stream);                                                         \
  /* AMG set-up, strength of connection: diag [n] = a_ii (0 when the row stores none) and, per       \
   * stored entry, strong [nnz] = 1 when j != i and |a_ij| >= theta sqrt(|a_ii a_jj|), else 0.       \
   * theta >= 0. */                                                                                \
  int tfem_amg_strength_##SUF(int64_t n, const int32_t* crow, const int32_t* col, const T* val,    \
                              double theta, T* diag, uint8_t* strong, void* stream);              \
  /* Deterministic SpGEMM C = op(A) B by expansion, stable radix sort of the 64-bit (row, col) keys, \
   * run-length encoding and in-order segmented sums (bitwise reproducible, no float atomics).       \
   * A [n_rows_a x .] CSR; transpose = 1 takes op(A) = A^T; b_crow == NULL stands for B = I (so      \
   * transpose = 1 with no B is the transpose of A).  n_rows_c / n_cols_c: shape of C.  n_products  \
   * must be the exact number of products: sum over the entries (i, k) of A of the length of row k   \
   * of B (row i with transpose; 1 without B).  Outputs sized for the worst case: c_crow            \
   * [n_rows_c + 1], c_col / c_val [n_products] (the first *c_nnz valid), c_nnz DEVICE int64.       \
   * workspace: at least tfem_csr_spgemm_workspace(n_rows_a, n_products) bytes. */                  \
  int tfem_csr_spgemm_##SUF(int64_t n_rows_a, const int32_t* a_crow, const int32_t* a_col,         \
                            const T* a_val, int transpose, const int32_t* b_crow,                 \
                            const int32_t* b_col, const T* b_val, int64_t n_rows_c,               \
                            int64_t n_cols_c, int64_t n_products, void* workspace,                \
                            int64_t workspace_bytes, int32_t* c_crow, int32_t* c_col, T* c_val,   \
                            int64_t* c_nnz, void* stream);                                         \
  /* Numeric-only SpGEMM: c_val of C = A B on a known pattern c_crow [n_rows + 1] / c_col (sorted   \
   * within rows, as tfem_csr_spgemm returns it).  A [n_rows x .] and B CSR.  For the pattern        \
   * tfem_csr_spgemm returned for the same A and B, c_val equals its c_val bit for bit: each entry   \
   * is +0 plus its products, each rounded on its own, added in expansion order (A-row entries in   \
   * stored order, then B-row entries in stored order).  A product whose column C's row lacks is     \
   * dropped and counted in *n_missing (DEVICE int32, zeroed by the caller; integer atomics only).  \
   * One warp per row; no workspace, no synchronisation: graph-capturable. */                       \
  int tfem_csr_spgemm_numeric_##SUF(int64_t n_rows, const int32_t* a_crow, const int32_t* a_col,  \
                                    const T* a_val, const int32_t* b_crow, const int32_t* b_col,  \
                                    const T* b_val, const int32_t* c_crow, const int32_t* c_col,  \
                                    T* c_val, int32_t* n_missing, void* stream);                  \
  /* AMG refresh, diagonal: diag [n] = a_ii (0 when the row stores none), the diag of             \
   * tfem_amg_strength without the strength pattern. */                                            \
  int tfem_amg_diag_##SUF(int64_t n, const int32_t* crow, const int32_t* col, const T* val,        \
                          T* diag, void* stream);                                                  \
  /* AMG refresh, smoother operator S = I - omega D^-1 A on A's pattern: wdinv [n] =               \
   * (1 / diag_i) * omega and s_val [nnz] = delta_ij - wdinv_i * a_ij, each operation rounded on its \
   * own (the rounding of sparse.amg's torch expressions).  omega must not be NaN. */               \
  int tfem_amg_smoother_##SUF(int64_t n, const int32_t* crow, const int32_t* col, const T* val,    \
                              const T* diag, double omega, T* wdinv, T* s_val, void* stream);     \
  /* Gather with fill: out [n] [k] = src[k] >= 0 ? in[src[k]] : fill (src int32). */                \
  int tfem_gather_##SUF(int64_t n, const int32_t* src, const T* in, double fill, T* out,           \
                        void* stream);                                                             \
  /* SURVEY.md 8(f).3 -- fused MLP-at-quadrature-points producer: N(x) and dN/dx of the body of the\
   * reference's FeedForwardNeuralNetwork (model/neural_network.py:50-100: Linear(d,w) act         \
   * {Linear(w,w) act} x n_square Linear(w,1)) by forward-mode differentiation in one pass over    \
   * the points: no autograd graph, no per-layer activation tensors.  params: W0 [w][d] | b0 [w] | \
   * {Wk [w][w] | bk [w]} x n_square | w_out [w] | b_out [1] (torch.nn.Linear layout);             \
   * act 0 = tanh, 1 = ReLU; d = 1..3, w <= 32.  x [n_pts,d] -> value [n_pts], grad [n_pts,d]. */  \
  int tfem_mlp_value_grad_##SUF(int64_t n_pts, int d, int width, int n_square, int act,            \
                                const T* params, const T* x, T* value, T* grad, void* stream);     \
  /* Its adjoint with respect to the parameters (what loss.backward() needs; the double backward   \
   * of neural_network.py:85-100 with create_graph=True): params_bar [n_params] from value_bar     \
   * [n_pts] and grad_bar [n_pts,d].  partial: scratch of n_partial * n_params values (n_partial = \
   * thread blocks used, e.g. one per SM); the blocks' sums are added in block order               \
   * (reproducible).  n_square <= 7. */                                                            \
  int tfem_mlp_value_grad_bwd_##SUF(int64_t n_pts, int d, int width, int n_square, int act,        \
                                    const T* params, const T* x, const T* value_bar,               \
                                    const T* grad_bar, T* partial, int n_partial, T* params_bar,   \
                                    void* stream);

TFEM_DECLARE(double, f64)
TFEM_DECLARE(float, f32)

/* Symbolic phase helper (integer, one-time): COO keys of basis/basis.py:72-75,
 * key[9e+3i+j] = dof_conn[e][j] * n_dof + dof_conn[e][i]   (row-major (row, col)). */
int tfem_coo_keys(int64_t n_el, const int32_t* dof_conn, int64_t n_dof, int64_t* keys, void* stream);

/* The whole symbolic phase of the sparse system on the device (SURVEY 8(b) tfem_csr_symbolic): the sorted-unique CSR
 * pattern of bilinear_form_idx (basis/basis.py:72-77) and the stable COO -> CSR permutations the deterministic scatter
 * kernels walk -- CUB radix sort of the (row, col) keys, run-length encoding, prefix sums, binary searches.
 *   dof_conn [n_el,3] int32, DOFs 0 .. n_dof-1.  Outputs, sized for the worst case (the caller slices by *nnz):
 *   crow [n_dof+1], col [9 n_el] (first nnz valid), seg [9 n_el + 1] (first nnz + 1 valid: COO entries perm[seg[p] ..
 *   seg[p+1]) sum to CSR entry p, in increasing COO index), perm [9 n_el], lin_seg [n_dof+1] / lin_perm [3 n_el] (the same
 *   for linear_form_idx), keys [9 n_el] (the nnz sorted unique keys row * n_dof + col), nnz (DEVICE int64).
 * workspace: device scratch of at least tfem_csr_symbolic_workspace() bytes (the library never allocates). */
int tfem_csr_symbolic_workspace(int64_t n_el, int64_t n_dof, int64_t* bytes);
int tfem_csr_symbolic(int64_t n_el, const int32_t* dof_conn, int64_t n_dof, void* workspace, int64_t workspace_bytes,
                      int32_t* crow, int32_t* col, int32_t* seg, int32_t* perm, int32_t* lin_seg, int32_t* lin_perm,
                      int64_t* keys, int64_t* nnz, void* stream);

/* AMG set-up, aggregation by parallel MIS(2) (Bell, Dalton, Olson 2012) on the strength graph (strong [nnz] from
 * tfem_amg_strength).  key [n] (uint64) = state << 61 | (hash32(i, level) >> 3) << 32 | i, state 0 = out,
 * 1 = undecided, 2 = in (a root); nodes without a strong connection start out.
 * tfem_amg_mis2_round: one round (init != 0 first writes the initial keys): two sweeps t = max(t, max over strong
 *   neighbours) from key into scratch [2n] (each sweep reads one buffer and writes the other), then an undecided node
 *   whose own key is the maximum becomes in and one whose maximum is an in node becomes out.  *n_undecided (DEVICE
 *   int32) = nodes still undecided; the caller repeats rounds until it reads 0 (each round decides at least one).
 * tfem_amg_aggregate: after the last round, agg [n] (int32) = rank of the node's root among the roots for every root
 *   and for each node with a strong root neighbour (the one of the largest key), else the aggregate of its strong
 *   neighbour of the largest key among those so assigned, -1 for nodes without a strong connection; *n_agg (DEVICE
 *   int32) = number of roots.  workspace: at least tfem_amg_aggregate_workspace() bytes. */
int tfem_amg_mis2_round(int64_t n, const int32_t* crow, const int32_t* col, const uint8_t* strong, int32_t level, int init,
                        uint64_t* key, uint64_t* scratch, int32_t* n_undecided, void* stream);
int tfem_amg_aggregate_workspace(int64_t n, int64_t* bytes);
int tfem_amg_aggregate(int64_t n, const int32_t* crow, const int32_t* col, const uint8_t* strong, const uint64_t* key,
                       void* workspace, int64_t workspace_bytes, int32_t* agg, int32_t* n_agg, void* stream);
int tfem_csr_spgemm_workspace(int64_t n_rows_a, int64_t n_products, int64_t* bytes);

/* SURVEY 8(f).2 -- edge topology on the device, replacing AbstractMesh._compute_interior_and_boundary_edges /
 * _compute_cells_4_edges (mesh/abstract_mesh.py:104-255, mesh/meshes_tri.py:54-123).
 * tfem_half_edges: every cell edge of n_mesh stacked meshes (conn [n_mesh * n_cells, 3], mesh-local vertex ids;
 *   local_pairs: HOST array of the 3 local vertex pairs, e.g. {0,1, 1,2, 0,2}) as the key
 *   mesh * n_vert^2 + min(v) * n_vert + max(v), stably sorted with its cell (index within the mesh) as payload:
 *   he_sorted / cell_sorted [3 n_mesh n_cells]; unique_keys / counts (same capacity, the first *n_unique valid;
 *   counts = incidence, 1 = boundary edge); n_unique: DEVICE int64.  workspace >= tfem_half_edges_workspace() bytes.
 * tfem_edge_cells: the n_sides (1 or 2) cells adjacent to each edge of edge_vertices [n_mesh * n_edges, 2], in increasing
 *   cell id; *status (DEVICE int32, zeroed by the caller) collects 1 = an edge belongs to no cell, 2 = a two-sided edge
 *   has a single adjacent cell.
 * tfem_interior_edge_geometry: end points x [.,2,2], length [.], unit normal [.,2] of each interior edge, the normal
 *   pointing from the first listed cell's centroid towards the second's (abstract_mesh.py:143-162). */
int tfem_half_edges_workspace(int64_t n_mesh, int64_t n_cells, int64_t* bytes);
int tfem_half_edges(int64_t n_mesh, int64_t n_cells, int64_t n_vert, const int32_t* conn, const int32_t* local_pairs,
                    void* workspace, int64_t workspace_bytes, int64_t* he_sorted, int32_t* cell_sorted, int64_t* unique_keys,
                    int32_t* counts, int64_t* n_unique, void* stream);
int tfem_edge_cells(int64_t n_mesh, int64_t n_edges, int64_t n_vert, const int32_t* edge_vertices, int n_sides,
                    const int64_t* he_sorted, const int32_t* cell_sorted, int64_t n_half, int32_t* cells, int32_t* status,
                    void* stream);
int tfem_interior_edge_geometry_f64(int64_t n_mesh, int64_t n_edges, int64_t n_vert, int64_t n_cells, const double* coords,
                                    const int32_t* conn, const int32_t* edge_vertices, const int32_t* edge_cells, double* x,
                                    double* length, double* normal, void* stream);
int tfem_interior_edge_geometry_f32(int64_t n_mesh, int64_t n_edges, int64_t n_vert, int64_t n_cells, const float* coords,
                                    const int32_t* conn, const int32_t* edge_vertices, const int32_t* edge_cells, float* x,
                                    float* length, float* normal, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* TFEM_B200_H */

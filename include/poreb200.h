/* poreb200.h -- C ABI of libporeb200.so: B200 (sm_100a) MPFA / MPSA / Biot
 * interaction-region assembly and CSR SpMV behind PorePy's discretization API.
 *
 * Plain pointers and sizes only; no torch / numpy types.  The Python host side
 * (porepy_b200/_lib.py) binds these with ctypes.  Every entry point names the
 * reference interface (pmgbergen/porepy v1.11.0) it replaces.
 *
 * Ownership: the caller owns every host buffer passed in or out.  The library
 * owns the device memory inside a plan handle.  Handles are not thread-safe;
 * use one host thread (one process under torchrun) per GPU.
 *
 * Return codes (all functions returning int):
 *   PB_OK 0
 *   PB_EINVAL 1     invalid argument
 *   PB_ESINGULAR 2  singular local system; the node id is in pb_last_error_node()
 *                   -> Python raises ValueError("Error in inversion of local linear
 *                   systems"), parity with numerics/linalg/matrix_operations.py:1487-1490
 *   PB_ECELLTYPE 3  a cell vertex does not have exactly nd faces of the cell meeting
 *                   in it (pyramids ...) -> AssertionError, parity with
 *                   numerics/fv/_fvutils.py:735 and mpsa.py:1569
 *   PB_ECUDA 4      CUDA runtime error (text in pb_last_error())
 *   PB_ENOTIMPL 5   feature of the reference not covered by this build
 */
#ifndef POREB200_H
#define POREB200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PB_OK 0
#define PB_EINVAL 1
#define PB_ESINGULAR 2
#define PB_ECELLTYPE 3
#define PB_ECUDA 4
#define PB_ENOTIMPL 5

/* boundary-condition codes per face (scalar) / per component and face (vector) */
#define PB_BC_INTERIOR 0
#define PB_BC_DIR 1
#define PB_BC_NEU 2
#define PB_BC_ROB 3

/* sparsity patterns shared by the output matrices (scalar "base" patterns) */
#define PB_PAT_FACE_CELL 0  /* nf x nc : flux, bound_pressure_cell; x nd columns: vector_source;
                               nd x nd blocks: stress, bound_displacement_cell; ...          */
#define PB_PAT_FACE_BFACE 1 /* nf x nf : bound_flux, bound_pressure_face, bound_stress, ...   */
#define PB_PAT_CELL_CELL 2  /* nc x nc : mpsa_consistency, displacement_divergence (x nd)     */
#define PB_PAT_CELL_BFACE 3 /* nc x nf : boundary_displacement_divergence (x nd)              */

typedef struct pb_plan pb_plan; /* opaque */
struct pb_csr;                  /* opaque device CSR matrix, see "CSR SpMV" below */

/* ---- library state ------------------------------------------------------------------ */
const char *pb_last_error(void);
int64_t pb_last_error_node(void);
/* number of CUDA devices visible, or -1 (no driver / no device).  Never falls back to CPU. */
int pb_device_count(void);
/* device allocations that missed the pooled blocks: {cudaMalloc calls, seconds, cudaFree calls, seconds} since load */
void pb_alloc_stats(double *out4);
/* cudaSetDevice for this process (one process per GPU). */
int pb_set_device(int device);
/* kernels launched by this library since load (bench.py's gpu_launches evidence). */
int64_t pb_launch_count(void);

/* Return the device blocks cached by the library's size-keyed pool (see csrc/plan.hpp: DevPool) to the driver. */
void pb_device_pool_trim(void);

/* FP64 peak of this device, measured by a dependency-free register loop: kind 0 = DMMA (mma.sync.m8n8k4.f64, the
 * pipe of the block Gauss-Jordan), kind 1 = scalar DFMA.  TFLOP/s, best of 5 launches (roofline denominator). */
int pb_fp64_peak(int kind, double *tflops);

/* Page-locked host buffers for the CSR value arrays the *_download calls fill (full PCIe rate;
 * pageable NumPy buffers go through the driver's staging copies).  The caller frees them. */
int pb_host_alloc(uint64_t bytes, void **out);
void pb_host_free(void *p);

/* ---- plan: sub-cell topology + output patterns --------------------------------------- */
/* Replaces _fvutils.SubcellTopology.__init__ (numerics/fv/_fvutils.py:51-172), the
 * sub-face pairing (:163-172, pair_over_subfaces :183-216), cell_node_blocks /
 * sub_cell_index of scalar_tensor_vector_prod (:697-762), Mpfa._block_diagonal_structure
 * (numerics/fv/mpfa.py:1357-1412) and the implicit sparsity patterns of the scipy SpGEMM
 * chains (mpfa.py:1080-1147, mpsa.py:735-781, biot.py:776-866).
 *   nd: grid dimension (2 or 3).  cell_faces: nf x nc CSC with +-1 data (pp.Grid.cell_faces),
 *   face_nodes: nn x nf CSC (pp.Grid.face_nodes).  Row indices need not be sorted. */
int pb_plan_create(int nd, int64_t nc, int64_t nf, int64_t nn,
                   const int32_t *cf_indptr, const int32_t *cf_indices, const int8_t *cf_data,
                   const int32_t *fn_indptr, const int32_t *fn_indices,
                   pb_plan **out);
void pb_plan_destroy(pb_plan *p);

/* sizes: sub-cells, unique sub-faces, sub-half-faces, largest local system (sub-faces at a node) */
int pb_plan_sizes(const pb_plan *p, int64_t *num_subcells, int64_t *num_subfaces,
                  int64_t *num_subhalffaces, int32_t *max_subfaces_per_node,
                  int32_t *max_subcells_per_node);
/* The node classes the last build made (kind 0: MPFA, at plan creation; kind 1: MPSA / Biot, at pb_mpsa_upload):
 * *count = number of classes; for the first min(count, cap) classes, the solver configuration, whether the matrix
 * lives in the global-memory workspace, and the number of nodes.  Host only: no kernel runs. */
int pb_plan_node_classes(const pb_plan *p, int kind, int cap, int32_t *cfg, uint8_t *a_global, int64_t *nodes,
                         int *count);
/* Shards: cell e of this plan is cell cells[e] of a larger (global) grid of n_source_cells cells.  The cell tensors of
 * the following pb_mpfa_upload / pb_mpsa_upload (permeability, stiffness, coupling tensors) are then the GLOBAL arrays
 * ((3,3,n_source), (9,9,n_source)) and are restricted on the device; NULL removes the map. */
int pb_plan_set_cell_map(pb_plan *p, const int64_t *cells, int64_t n_source_cells);
/* Restrict the assembly to the interaction regions of the flagged nodes (mask: nn bytes, NULL = all nodes).
 * Used by the multi-GPU path: a shard assembles the regions of its OWN nodes only; the outer nodes of its halo
 * layer are incomplete there and their rows are discarded anyway (reference: the overlap removal of
 * numerics/fv/mpfa.py:301-304).  Rows of faces with an inactive node are incomplete. */
int pb_plan_set_active_nodes(pb_plan *p, const uint8_t *mask);
/* base pattern `which` (PB_PAT_*): nrows and nnz; then copy indptr (nrows+1) / indices (nnz). */
int pb_plan_pattern_size(const pb_plan *p, int which, int64_t *nrows, int64_t *nnz);
int pb_plan_pattern_get(const pb_plan *p, int which, int32_t *indptr, int32_t *indices);

/* Block expansion of base pattern `which` into br x bc blocks (row r*br+i, column c*bc+j), built
 * on the device and copied to the caller's buffers: indptr (nrows*br+1), indices (br*bc*nnz).
 * The value of block entry (i,j) of base entry q of base row r lives at
 * br*bc*indptr[r] + i*bc*len_r + (q-indptr[r])*bc + j -- the layout the kernels scatter into.
 * PB_ENOTIMPL when br*bc*nnz does not fit int32. */
int pb_plan_pattern_expanded(pb_plan *p, int which, int br, int bc, int32_t *indptr, int32_t *indices);

/* Geometry the path reads from pp.Grid (grids/grid.py:32): nodes (3 x nn), face_normals /
 * face_centers (3 x nf), cell_centers (3 x nc) row-major as numpy stores them; face_areas (nf),
 * cell_volumes (nc).  Copied to the device inside the plan. */
int pb_plan_set_geometry(pb_plan *p, const double *nodes, const double *face_normals,
                         const double *face_centers, const double *face_areas,
                         const double *cell_centers, const double *cell_volumes);

/* ---- MPFA ----------------------------------------------------------------------------- */
/* Replaces Mpfa._flux_discretization (numerics/fv/mpfa.py:592-1156) incl. _create_bound_rhs
 * (:1414-1578), _discretize_vector_source (:1158-1307), reconstruct_presssure (:1628-1690),
 * _fvutils.scalar_tensor_vector_prod / compute_dist_face_cell / ExcludeBoundaries and
 * matrix_operations.invert_diagonal_blocks (numerics/linalg/matrix_operations.py:1175).
 *   perm:  SecondOrderTensor.values, (3,3,nc) row-major (params/tensor.py:157)
 *   bc:    nf codes PB_BC_* (internal/fracture faces already mapped to PB_BC_NEU, mpfa.py:1452)
 *   robin_weight: nf doubles (may be NULL when no Robin face)
 *   eta:   continuity point parameter (mpfa_eta)
 * Outputs: CSR `data` arrays on the base patterns; NULL = not wanted.
 *   flux, bound_pressure_cell: nnz(FACE_CELL);  vector_source, bound_pressure_vector_source:
 *   nd*nnz(FACE_CELL) (entry p expands to p*nd+j);  bound_flux, bound_pressure_face:
 *   nnz(FACE_BFACE). */
int pb_mpfa_upload(pb_plan *p, const double *perm, const uint8_t *bc, const double *robin_weight,
                   double eta);
/* device-resident assembly of the uploaded problem; want_* select outputs. ms = device time. */
int pb_mpfa_assemble(pb_plan *p, int want_flux_terms, int want_trace_terms,
                     int want_vector_source, float *ms);
int pb_mpfa_download(pb_plan *p, double *flux, double *bound_flux, double *bound_pressure_cell,
                     double *bound_pressure_face, double *vector_source,
                     double *bound_pressure_vector_source);

/* ---- device-resident results ----------------------------------------------------------------------------
 * The value array of one output matrix can be MOVED out of the plan as a pb_values handle: the matrix then
 * stays in HBM until the caller asks for it (the Python layer stores scipy-compatible matrices whose data /
 * indices are downloaded on first touch), and the plan allocates a fresh array at its next assemble.  Keys: */
#define PB_OUT_FLUX 0
#define PB_OUT_BOUND_FLUX 1
#define PB_OUT_BOUND_PRESSURE_CELL 2
#define PB_OUT_BOUND_PRESSURE_FACE 3
#define PB_OUT_VECTOR_SOURCE 4
#define PB_OUT_BOUND_PRESSURE_VECTOR_SOURCE 5
#define PB_OUT_STRESS 6
#define PB_OUT_BOUND_STRESS 7
#define PB_OUT_BOUND_DISPLACEMENT_CELL 8
#define PB_OUT_BOUND_DISPLACEMENT_FACE 9
/* Biot, coupling tensor q: PB_OUT_BIOT + 5*q + {0 displacement_divergence, 1 boundary_displacement_divergence,
 * 2 scalar_gradient, 3 mpsa_consistency, 4 bound_displacement_pressure} */
#define PB_OUT_BIOT 10
typedef struct pb_values pb_values; /* opaque: device array of doubles */
int pb_plan_take_output(pb_plan *p, int key, pb_values **out);
int64_t pb_values_size(const pb_values *v);
int pb_values_download(pb_values *v, double *host); /* D2H of all values (page-locked host buffer: full PCIe rate) */
int pb_values_checksum(pb_values *v, double *sum, double *sum_of_squares); /* device reduction, 16-byte read */
void pb_values_destroy(pb_values *v);

/* One output matrix as a device CSR handle (block-expanded pattern + a copy of the values): operand of the
 * device-side AD chain below.  which / br / bc as in pb_plan_pattern_expanded. */
int pb_plan_output_csr(pb_plan *p, const pb_values *v, int which, int br, int bc, struct pb_csr **out);

/* Device-side system of the flow problem, replacing the host scipy products of
 * FVElliptic.assemble_matrix_rhs (numerics/fv/fv_elliptic.py:67-112):
 *   A = div @ flux  on the CELL_CELL pattern, kept in HBM as a device CSR handle, no D2H of the matrices;
 *   b = -div @ (bound_flux @ bc_values) [- div @ (vector_source @ v)]   (host vectors in/out).
 * The discretization matrices are given by their value handles (NULL = the plan's last assembled arrays). */
int pb_mpfa_system(pb_plan *p, const pb_values *flux, struct pb_csr **out);
int pb_mpfa_rhs(pb_plan *p, const pb_values *bound_flux, const pb_values *vector_source_discr,
                const double *bc_values, const double *vector_source, double *rhs);
/* Same for mechanics (Mpsa.assemble_matrix_rhs, numerics/fv/mpsa.py:486-529): A = div_nd @ stress
 * (nd x nd blocks on the CELL_CELL pattern, row c*nd+i, column k*nd+j) as a device CSR and
 * b = -div_nd @ (bound_stress @ bc_values) + source  (bc_values: nf*nd face-major, source: nc*nd). */
int pb_mpsa_system(pb_plan *p, const pb_values *stress, struct pb_csr **out);
int pb_mpsa_rhs(pb_plan *p, const pb_values *bound_stress, const double *bc_values, const double *source,
                double *rhs);

/* ---- MPSA / Biot ------------------------------------------------------------------------ */
/* Replaces Mpsa._stress_discretization (numerics/fv/mpsa.py:531-781),
 * _create_inverse_gradient_matrix (:784-930), _tensor_vector_prod (:1520-1675),
 * _eliminate_ncasym (:1932-2000), _create_bound_rhs (:984-1185), _reconstruct_displacement
 * (:1187-1275) and, with n_alpha > 0, Biot._local_discretization (numerics/fv/biot.py:714-878).
 *   stiffness: FourthOrderTensor.values (9,9,nc) row-major (params/tensor.py:348)
 *   bc:        (nd, nf) codes PB_BC_* row-major (BoundaryConditionVectorial.is_dir/is_neu/is_rob)
 *   robin_weight: (nd,nd,nf) row-major or NULL
 *   alpha:     n_alpha coupling tensors, each (3,3,nc) row-major (scalar_vector_mappings)
 * Outputs: data arrays; block expansion of the base patterns, row f*nd+i, column c*nd+j:
 *   stress, bound_displacement_cell: nd*nd*nnz(FACE_CELL); bound_stress,
 *   bound_displacement_face: nd*nd*nnz(FACE_BFACE); per coupling tensor:
 *   displacement_divergence nd*nnz(CELL_CELL), boundary_displacement_divergence
 *   nd*nnz(CELL_BFACE), scalar_gradient / bound_displacement_pressure nd*nnz(FACE_CELL),
 *   mpsa_consistency nnz(CELL_CELL). */
int pb_mpsa_upload(pb_plan *p, const double *stiffness, const uint8_t *bc,
                   const double *robin_weight, double eta, int n_alpha, const double *alpha);
/* Boundary conditions in a rotated basis (BoundaryConditionVectorial.basis, params/bc.py; applied to the
 * boundary equations by ExcludeBoundaries, numerics/fv/_fvutils.py:765-945): basis (nd,nd,nf) row-major,
 * NULL = identity.  Call after pb_mpsa_upload (which resets it to the identity). */
int pb_mpsa_set_basis(pb_plan *p, const double *basis);
int pb_mpsa_assemble(pb_plan *p, float *ms);
int pb_mpsa_download(pb_plan *p, double *stress, double *bound_stress,
                     double *bound_displacement_cell, double *bound_displacement_face);
int pb_biot_download(pb_plan *p, int which_alpha, double *displacement_divergence,
                     double *boundary_displacement_divergence, double *scalar_gradient,
                     double *mpsa_consistency, double *bound_displacement_pressure);

/* ---- CSR SpMV ---------------------------------------------------------------------------- */
/* Replaces the scipy `M @ val` of AdArray.__rmatmul__ (numerics/ad/forward_mode.py:565-595)
 * and the residual chain of EquationSystem.assemble(evaluate_jacobian=False)
 * (numerics/ad/equation_system.py:1579-1713).  y = A x (+ beta*y).  */
typedef struct pb_csr pb_csr; /* opaque: device-resident CSR matrix */

/* ---- two-point flux approximation and first-order upwinding (one thread per face) ----------------
 * A pb_facegrid is the face-indexed device view of a grid of ANY dimension (1-D lines and 2-D planes
 * embedded in 3-D included): the face -> cell table built from cell_faces (nf x nc CSC, +-1 data) and
 * face_normals / face_centers (3 x nf), cell_centers (3 x nc), row-major.  No interaction-region plan.
 * Replaces Tpfa.discretize (numerics/fv/tpfa.py:40-280), incl. the 1-D delegation of MPFA / MPSA
 * (mpfa.py:690-712, mpsa.py:666-697), and Upwind.discretize (numerics/fv/upwind.py:150-300).
 * bc_bits (nf): bits 0-1 = PB_BC_* effective code, bit 2 = raw is_dir, bit 3 = raw is_neu.
 * pb_tpfa: fc_indptr = row pointer of cell_faces in CSR-by-face form with ascending columns; value
 * arrays in that pattern (flux, bound_pressure_cell: nnz; vector sources: nnz*vdim, entry-major) and
 * the two diagonals (nf).  pb_upwind: upstream cell per face (-1 = face removed from the matrix) and the
 * diagonals of the Neumann / Dirichlet-inflow boundary matrices.  Host pointers; outputs may be NULL
 * for pb_tpfa. */
typedef struct pb_facegrid pb_facegrid; /* opaque */
int pb_facegrid_create(int64_t nc, int64_t nf, const int32_t *cf_indptr, const int32_t *cf_indices,
                       const int8_t *cf_data, const double *face_normals, const double *face_centers,
                       const double *cell_centers, pb_facegrid **out);
void pb_facegrid_destroy(pb_facegrid *g);
int pb_tpfa(pb_facegrid *g, const double *permeability, const uint8_t *bc_bits, const int32_t *fc_indptr,
            int vdim, double *flux, double *bound_pressure_cell, double *vector_source,
            double *bound_pressure_vector_source, double *bound_flux_diag,
            double *bound_pressure_face_diag);
/* Differentiable TPFA (csrc/tpfa_diff.cuh; reference numerics/fv/tpfa.py:281-760 DifferentiableTpfa and the AD
 * expression of models/constitutive_laws.py:1544-1583): k = 9 * nc doubles, the 3 x 3 tensor of cell c at k[9c..9c+8]
 * row-major; fc_indptr as for pb_tpfa (half-faces numbered by face, then by cell).  Outputs: half-face
 * transmissibilities t_hf (nhf), face transmissibilities T (nf), dT/dk (nhf * 9: the 9 derivatives with respect to the
 * tensor of the half-face's cell).  Host pointers. */
int pb_tpfa_diff(pb_facegrid *g, const double *k, const int32_t *fc_indptr, double *t_hf, double *T, double *dT_dk);
int pb_upwind(pb_facegrid *g, const double *darcy_flux, const uint8_t *bc_bits, int32_t *upstream_cell,
              double *neumann_diag, double *dirichlet_diag);

/* Interface upwinding (UpwindCoupling.discretize, numerics/fv/upwind.py:427-528): per mortar cell the sign of the
 * interface flux and the masks "upstream is the higher-dimensional side" / "... the lower-dimensional side".
 * Host pointers, n doubles each. */
int pb_upwind_coupling(int64_t n, const double *interface_flux, double *sign, double *from_primary,
                       double *from_secondary);

/* ---- Grid.compute_geometry for 3-D grids (csrc/geometry.cu; reference grids/grid.py:362-381, 572-778) ---------
 * Face normals (area weighted) / centres / areas and cell centres / volumes of a grid of general polyhedral cells
 * from its topology and nodes: each face is fanned into triangles around the mean of its nodes, each cell into
 * tetrahedra around the mean of its faces' centres.  Host arrays in the reference's layouts: CSC of cell_faces
 * (nf x nc, row indices ascending inside a column, data +-1), CSC of face_nodes (nn x nf, the nodes of a face in loop
 * order), nodes (3, nn) row-major; outputs (3, nf), (3, nf), (nf), (3, nc), (nc).  kernel_ms (may be NULL) = device
 * time of the two kernels.  PB_EINVAL ("Some tetrahedra have negative volume", grid.py:754; cell in
 * pb_last_error_node()) for inverted cells. */
int pb_compute_geometry_3d(int64_t nc, int64_t nf, int64_t nn, const int32_t *cf_indptr, const int32_t *cf_indices,
                           const int8_t *cf_data, const int32_t *fn_indptr, const int32_t *fn_indices,
                           const double *nodes, double *face_normals, double *face_centers, double *face_areas,
                           double *cell_centers, double *cell_volumes, float *kernel_ms);

/* ---- sharding of ONE grid across ranks (csrc/shard.cu; host code) ---------------------------------------------
 * This rank's share of a grid from the GLOBAL topology: replaces the reference's memory-splitting chain
 * _fvutils.subproblems (numerics/fv/_fvutils.py:414-539) -> partition.extract_subgrid (grids/partition.py:540-640)
 * for this path.  cf_* / fn_*: CSC arrays of cell_faces (nf x nc, data +-1) and face_nodes (nn x nf); part: rank of
 * each cell.  Shard cells = every cell with a face holding a node of an own cell (one halo layer), OWN CELLS FIRST
 * (ascending), then the halo; faces / nodes ascending.  pb_shard_sizes: {cells, faces, nodes, own cells, nnz of the
 * local cell_faces, nnz of the local face_nodes}.  pb_shard_fill: local->global maps, per local face the flags
 * "row kept by this rank" / "cut face of the overlap" / "one cell inside the shard", per local node "interaction
 * region assembled by this rank", and the local CSC arrays (any output may be NULL). */
typedef struct pb_shard pb_shard; /* opaque */
int pb_shard_create(int64_t nc, int64_t nf, int64_t nn, const int32_t *cf_indptr, const int32_t *cf_indices,
                    const double *cf_data, const int32_t *fn_indptr, const int32_t *fn_indices,
                    const int64_t *part, int64_t rank, pb_shard **out);
int pb_shard_sizes(const pb_shard *s, int64_t *sizes6);
int pb_shard_fill(const pb_shard *s, int64_t *cells, int64_t *faces, int64_t *nodes, uint8_t *own_face,
                  uint8_t *cut_face, uint8_t *single_face, uint8_t *own_node, int32_t *cf_indptr,
                  int32_t *cf_indices, double *cf_data, int32_t *fn_indptr, int32_t *fn_indices);
void pb_shard_destroy(pb_shard *s);
/* dst[r, j] = src[r, idx[j]]: the (3, n) geometry arrays of a sub-grid (row-major host arrays) */
int pb_gather_columns(const double *src, int64_t nrows, int64_t ncols, const int64_t *idx, int64_t n, double *dst);

/* device-resident CSR matrix */
int pb_csr_create(int64_t nrows, int64_t ncols, int64_t nnz, const int32_t *indptr,
                  const int32_t *indices, const double *data, pb_csr **out);
void pb_csr_destroy(pb_csr *a);
/* Keep the first nrows rows (a row-partitioned system: the rows of a rank's own cells come first). */
int pb_csr_truncate_rows(pb_csr *a, int64_t nrows);
/* lanes per row the SpMV of this matrix runs with (autotuned at creation; POREB200_SPMV_TPR overrides) */
int pb_csr_lanes_per_row(const pb_csr *a);
/* diagonal (min(nrows, ncols) doubles, host) -- the Jacobi preconditioner of the Krylov solve */
int pb_csr_diagonal(pb_csr *a, double *diag);
/* ---- device-side sparse algebra of the AD Jacobian chain (csrc/sparse_ops.cu) ---------------------------------
 * M @ jac (AdArray.__rmatmul__, numerics/ad/forward_mode.py:565-595), diag(v) @ jac (:613-616), jac + jac,
 * the block concatenation of MergedOperator.parse (numerics/ad/ad_utils.py:597-664) and the vstack of
 * EquationSystem.assemble (numerics/ad/equation_system.py:1695-1713), on matrices that stay in HBM.
 * All results are new handles with sorted rows.  d_dev: DEVICE vector. */
int pb_csr_spgemm(const pb_csr *a, const pb_csr *b, pb_csr **out);                      /* C = A @ B */
int pb_csr_axpby(double alpha, const pb_csr *a, double beta, const pb_csr *b, pb_csr **out); /* C = alpha A + beta B */
int pb_csr_scale_dev(const pb_csr *a, const double *d_dev, int by_cols, pb_csr **out);  /* diag(d) A  |  A diag(d) */
/* nbr x nbc grid of blocks, row-major, NULL = zero block; row_sizes (nbr) / col_sizes (nbc) */
int pb_csr_bmat(int nbr, int nbc, const pb_csr *const *blocks, const int64_t *row_sizes, const int64_t *col_sizes,
                pb_csr **out);
/* sum and sum of squares of the stored values (device reduction) */
int pb_csr_checksum(pb_csr *a, double *sum, double *sum_of_squares);
/* copy a device-resident matrix back (indptr nrows+1, indices nnz, data nnz); sizes via pb_csr_shape */
int pb_csr_shape(const pb_csr *a, int64_t *nrows, int64_t *ncols, int64_t *nnz);
int pb_csr_download(pb_csr *a, int32_t *indptr, int32_t *indices, double *data);
/* host vectors in/out (H2D + kernel + D2H) */
int pb_csr_spmv(pb_csr *a, const double *x, double *y);
/* device pointers (e.g. torch tensors' data_ptr()); stream = cudaStream_t as integer (0 = default) */
int pb_csr_spmv_dev(pb_csr *a, const double *x_dev, double *y_dev, uint64_t stream);
/* y = A x on device pointers with the Krylov dot products in the epilogue: *d1 += (w1, y), *d2 += (w2, y)
 * (w2 NULL: (y, y)); d1 / d2 are device addresses or NULL. */
int pb_csr_spmv_dots_dev(pb_csr *a, const double *x_dev, double *y_dev, const double *w1_dev, double *d1_dev,
                         const double *w2_dev, double *d2_dev, uint64_t stream);

/* ---- fused vector kernels of the Jacobi-BiCGStab (csrc/krylov.cu; SURVEY 8f rank 1, replaces the direct solve of
 * models/solution_strategy.py:830-884).  All pointers are DEVICE pointers; `scal` is the 14-double scalar buffer
 * described in krylov.cu (every scalar of the recurrence stays on the device; the caller all-reduces slices of it
 * between the kernels under torch.distributed and polls it every few iterations); cur = iteration parity. */
int pb_kry_init(int64_t n, const double *b, double *x, double *r, double *rhat, double *p, double *v, double *scal,
                double tol, uint64_t stream);
int pb_kry_seed(double *scal, uint64_t stream);
/* minv / bs: the preconditioner M^-1 -- bs = 1: inverse diagonal (n doubles, Jacobi); bs = 2, 3: inverted bs x bs
 * diagonal blocks, row-major (n/bs blocks; block Jacobi over the displacement components of a cell); NULL: none */
int pb_kry_p(int64_t n, const double *r, double *p, const double *v, const double *minv, double *ph, double *scal,
             int cur, int bs, uint64_t stream);
int pb_kry_s(int64_t n, const double *r, const double *v, const double *minv, double *s, double *sh, double *scal,
             int cur, int bs, uint64_t stream);
/* inverses of the first nblocks bs x bs diagonal blocks of a device CSR, to a DEVICE array (nblocks*bs*bs doubles) */
int pb_csr_block_diag_inv_dev(const pb_csr *a, int bs, int64_t nblocks, double *out_dev, uint64_t stream);
int pb_kry_xr(int64_t n, double *x, const double *ph, const double *sh, const double *s, const double *t, double *r,
              const double *rhat, double *scal, int cur, int carry /* 1 on exactly one rank */, uint64_t stream);

/* ---- local-block inverse preconditioner (csrc/local_blocks.cu).  A layout partitions rows and columns of a square
 * matrix into nblocks blocks: block b pairs rows[blk_ptr[b] .. blk_ptr[b+1]) with cols[same range], s_b <= 32.
 * inv_ptr: prefix sums of s_b^2 (nblocks + 1); order: the block ids grouped by team size (s_b <= 4, 8, 16, 32), with the
 * HOST array class_ptr[5] delimiting the four groups.  All other pointers are DEVICE pointers.
 * Factorisation: inv[inv_ptr[b] ..] = A[rows_b, cols_b]^-1, row-major, by Gauss-Jordan with partial pivoting (FP64).
 * A non-finite entry, a pivot that is not finite or <= 1e-14 max|B_b|, or a non-finite inverse returns PB_ESINGULAR
 * naming the first failing block (err_dev: one device word of scratch; the call synchronises the stream once to read it).
 * Application: z[cols_b] = B_b^-1 r[rows_b] for every block, one launch per team size; skip: NULL or a device double,
 * when it is non-zero the call does nothing (the sticky DONE flag of the GMRES loop). */
int pb_csr_local_block_inv_dev(const pb_csr *a, int64_t nblocks, const int64_t *blk_ptr, const int32_t *rows,
                               const int32_t *cols, const int64_t *inv_ptr, const int32_t *order,
                               const int64_t *class_ptr, double *inv, uint64_t *err_dev, uint64_t stream);
int pb_local_block_apply_dev(int64_t nblocks, const int64_t *blk_ptr, const int32_t *rows, const int32_t *cols,
                             const int64_t *inv_ptr, const int32_t *order, const int64_t *class_ptr, const double *inv,
                             const double *r, double *z, const double *skip, uint64_t stream);

/* ---- vector kernels of the restarted right-preconditioned GMRES(m) with CGS2 (csrc/gmres.cu).  V: n x (m+1) basis,
 * column-major; H: (m+1) x m Hessenberg matrix, column-major; hb: 2 (m+1) + 2 doubles (two Gram-Schmidt passes and
 * their ||w||^2); scal: the 8-double scalar buffer described in gmres.cu.  All pointers are DEVICE pointers. */
int pb_gm_dots(int64_t n, const double *V, int ncols, const double *w, double *h, const double *scal, uint64_t stream);
int pb_gm_orth(int64_t n, const double *V, int ncols, const double *h, double *w, double *ww, const double *scal,
               uint64_t stream);
int pb_gm_givens(int j, int m, double *H, double *hb, double *cs, double *sn, double *g, double *scal, uint64_t stream);
int pb_gm_scale(int64_t n, double *v, const double *scal, uint64_t stream);
int pb_gm_residual(int64_t n, const double *b, double *r, double *scal, int with_bb, uint64_t stream);
int pb_gm_start(int m, double tol, double *hb, double *g, double *scal, uint64_t stream);
int pb_gm_ysolve(int m, const double *H, const double *g, double *y, const double *scal, uint64_t stream);
int pb_gm_combine(int64_t n, const double *V, int m, const double *y, double *t, const double *scal, int accumulate,
                  uint64_t stream);
int pb_gm_axpy(int64_t n, const double *z, double *x, uint64_t stream);

/* time `reps` device SpMVs with CUDA events on the launching stream; returns mean ms */
int pb_csr_spmv_bench(pb_csr *a, int reps, float *mean_ms);

/* ---- diagnostics of the interaction-region solvers (solver_check.cu) ----
 * Solver configuration cfg (0..7, the class table of plan.hpp): threads per team and the largest system order and
 * augmented width it takes (INT_MAX for the catch-all configuration 6). */
int pb_solver_limits(int cfg, int *team, int *max_n, int *max_w);
/* Solve nsys dense systems with configuration cfg, one team per system, exactly as the assembly kernels run it
 * (launch geometry, shared-memory layout, row stride (n + nrhs) | 1, rowidx starting as the identity; a_global != 0:
 * the matrix lives in a global-memory workspace).  Host arrays: A (nsys, n, n + nrhs) row-major, the augmented
 * [M | B]; X (nsys, n, nrhs) receives M^-1 B (NaN where the solver refused the system); ok (nsys) 1 / 0.
 * PB_EINVAL before any launch when the system does not fit the configuration or its shared memory. */
int pb_local_solve_batch(int cfg, int a_global, int64_t nsys, int n, int nrhs, const double *A, double *X,
                         int32_t *ok);

#ifdef __cplusplus
}
#endif
#endif /* POREB200_H */

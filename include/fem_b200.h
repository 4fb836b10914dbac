/*
 * fem_b200.h - C ABI of the B200-native FEM elasto-plasticity hot path.
 *
 * The reference (MartinBeseda/FEM-ElastoPlasticity) is pure Python and has no FFI;
 * these entry points are what a ctypes binding of its pythonFEM.py hot path binds
 * (INTEGRATION.md shows the stub).  Each symbol cites the reference statement it
 * replaces (paths relative to the reference root).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name starts with h_ (host);
 *   - all arrays are FP64 / int32 / uint8, structure-of-arrays, C-contiguous:
 *       elem[n_p][n_e] (0-based), coord[2][n_n], E[3][n_int], S[4][n_int], DS[9][n_int],
 *       Ep[4][n_int]; nodal vectors are DOF-interleaved: u[2*node + comp]
 *       (== U.reshape(-1, order='F') of the reference's (2, n_n) arrays);
 *   - integration point g = e*n_q + q; DS[k] is entry (k%3, k/3) of the 3x3 tangent;
 *   - K is CSR (int32 row_ptr/col_idx, sorted columns) over the STRUCTURAL pattern of
 *     B^T D B (2x2 node blocks); values arrays are aligned with fem_plan_pattern();
 *   - functions return fem_status; fem_last_error_string() describes the last failure
 *     on the calling thread.  Nothing throws across the ABI.  There is no CPU fallback.
 *   - `stream` is a cudaStream_t (NULL = legacy default stream).  Kernels are
 *     asynchronous on it; only functions that return host scalars synchronise.
 */
#ifndef FEM_B200_H
#define FEM_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct fem_plan fem_plan; /* opaque: CSR pattern, incidence lists, geometry, workspaces */
typedef void* fem_stream;         /* cudaStream_t */

typedef enum fem_status {
  FEM_OK = 0,
  FEM_ERR_INVALID_ARG = 1,
  FEM_ERR_CUDA = 2,
  FEM_ERR_NONFINITE_JACOBIAN = 3, /* degenerate element: det == 0 or non-finite (reference lets inf/nan propagate) */
  FEM_ERR_PCG_BREAKDOWN = 4,      /* p'Ap <= 0 or non-finite */
  FEM_ERR_PCG_MAXIT = 5,          /* not converged in maxit iterations (x holds the last iterate) */
  FEM_ERR_UNSUPPORTED = 6,        /* element type / node valence outside the compiled kernels */
  FEM_ERR_NO_DEVICE = 7
} fem_status;

const char* fem_last_error_string(void);
int fem_version(void);
/* sm_count, compute capability and free/total HBM bytes of the current device */
int fem_device_info(int* sm_count, int* cc_major, int* cc_minor, int64_t* free_bytes, int64_t* total_bytes);

/* ---- plan: mesh topology -> structural CSR pattern + geometry (once per mesh) -----------------
 * Replaces the geometry/B/D part of get_elastic_stiffness_matrix
 * (Plasticity2D_DP/pythonFEM.py:500-592 == tsx-tunnel/pythonFEM.py:441-533 == Elasticity2D/pythonFEM.py:375-467)
 * and the implicit pattern construction of scipy's coo_tocsr/csr_matmat (:570,592,595).
 * h_dhatp1/h_dhatp2 are (n_p, n_q) row-major, h_wf is (n_q,): the outputs of
 * get_local_basis_volume / get_quadrature_volume, accepted unchanged.
 * Supported (n_p, n_q): (3,1) P1, (6,7) P2, (4,4) Q1, (8,9) Q2.                                  */
int fem_plan_create(int64_t n_n, int64_t n_e, int n_p, int n_q, const int32_t* elem, const double* coord,
                    const double* h_dhatp1, const double* h_dhatp2, const double* h_wf, fem_stream stream,
                    fem_plan** out);
int fem_plan_destroy(fem_plan* plan);
/* n_n, n_e, n_int, n_dof, nnz, max node degree (neighbours incl. self) */
int fem_plan_sizes(const fem_plan* plan, int64_t* n_n, int64_t* n_e, int64_t* n_int, int64_t* n_dof, int64_t* nnz,
                   int* max_degree);
/* structural CSR pattern (device pointers owned by the plan; row_ptr has n_dof+1 entries) */
int fem_plan_pattern(const fem_plan* plan, const int32_t** row_ptr, const int32_t** col_idx, int64_t* nnz);
/* node-block form of the same pattern used by the SpMV: nbr_ptr[n_n+1], nbr_idx[nnz/4] */
int fem_plan_blocks(const fem_plan* plan, const int32_t** nbr_ptr, const int32_t** nbr_idx, int64_t* n_blocks);
/* dphi1, dphi2 (n_p, n_int) and weight (n_int,) = |det J| * wf  (:545-546, :585); owned by the plan.
 * These are exactly the stored values of the reference's sparse B (:549-571).                    */
int fem_plan_geometry(const fem_plan* plan, const double** dphi1, const double** dphi2, const double** weight);
/* whether the TMA-staged assembly kernel applies to this mesh (P1, degree <= 8, most 32-node slices touching at most two
 * runs of consecutive elements) and the width (elements) of its TMA boxes */
int fem_plan_stage_info(const fem_plan* plan, int* stage_ok, int* stage_cap);
/* bytes of device memory held by the plan */
int64_t fem_plan_bytes(const fem_plan* plan);

/* vd[k][g] = (2*Dev[k]*G + Vol[k]*K) * weight[g], k < 9: the stored values of the reference's sparse D
 * (Plasticity2D_DP/pythonFEM.py:579-592), for callers that need D_elast itself.                   */
int fem_elastic_dmat(const fem_plan* plan, const double* shear, const double* bulk, double* vd, fem_stream stream);

/* ---- assembly ---------------------------------------------------------------------------------
 * K_elast = B^T D B, D = weight*(2G*Dev + K*Vol)          (Plasticity2D_DP/pythonFEM.py:579-595)
 * Values are accumulated per CSR entry in ascending (element, quadrature point, strain row) order,
 * i.e. the order of scipy's csr_matmat, without FMA contraction: bit-identical to the reference. */
int fem_assemble_elastic(const fem_plan* plan, const double* shear, const double* bulk, double* K_vals,
                         fem_stream stream);
/* K_tangent, direct form: sum_g B_g^T (w_g * DS_g) B_g     (Plasticity2D_DP/pythonFEM.py:1047-1050,
 * tsx-tunnel/pythonFEM.py:1773-1777; equal to the reference within rounding, one pass, K written once) */
int fem_assemble_tangent(const fem_plan* plan, const double* DS, double* K_vals, fem_stream stream);
/* K_tangent in the reference's own operation order: K_elast + B^T (D_p - D_elast) B  (:1050);
 * bit-identical to the reference; reads K_elast_vals and shear/bulk in addition.                 */
int fem_assemble_tangent_ref(const fem_plan* plan, const double* DS, const double* shear, const double* bulk,
                             const double* K_elast_vals, double* K_vals, fem_stream stream);
/* Fused Newton-iteration assembly: K_tangent (direct form) and F = B^T (w*S[0:3]) in one pass.   */
int fem_assemble_tangent_force(const fem_plan* plan, const double* DS, const double* S, double* K_vals, double* F,
                               fem_stream stream);

/* E = reshape(B @ U(:), (3, n_int), 'F')                    (Plasticity2D_DP/pythonFEM.py:1043,1095) */
int fem_strain(const fem_plan* plan, const double* u, double* E, fem_stream stream);
/* F = B^T vec(w * S[0:3])  (S has leading dimension n_int)  (Plasticity2D_DP/pythonFEM.py:1058) */
int fem_internal_force(const fem_plan* plan, const double* S, double* F, fem_stream stream);

/* ---- Drucker-Prager return map + consistent tangent -------------------------------------------
 * construct_constitutive_problem (Plasticity2D_DP/pythonFEM.py:604-757; tsx-tunnel/pythonFEM.py:990-1157).
 * h_e0: host 4-vector added to the strain (tsx signature) or NULL.  Ep_prev may be NULL (treated as 0).
 * apply != 0: Ep_prev is updated IN PLACE (the reference aliases ep = ep_prev, :750-755) and, if Ep_out is
 * non-NULL and != Ep_prev, also copied there; apply == 0: Ep_out (if non-NULL) is zero-filled (:749).
 * ind_p: uint8 flags CRIT1 > 0.  lambda (nullable): plastic multipliers, smooth branch as the reference
 * (:710); apex entries hold the intended (eta*p_tr - c)/denom_a (the reference's outer-product expression
 * at :714 makes its lambda_final None; not under parity).  counts (nullable): device int64[2] =
 * {n_smooth, n_apex}, ADDED to (zero it first) - the numbers the reference logs at :730.          */
int fem_dp_return_map(int64_t n_int, const double* E, const double* h_e0, double* Ep_prev, const double* shear,
                      const double* bulk, const double* eta, const double* c, int apply, double* S, double* DS,
                      uint8_t* ind_p, double* lambda, double* Ep_out, int64_t* counts, fem_stream stream);

/* ---- CSR SpMV + PCG (replaces the dense solve, Plasticity2D_DP/pythonFEM.py:1062-1066, and serves
 * the energy-norm criterion, :1072-1075) ----------------------------------------------------------
 * y = mask .* (K x); free_mask (uint8[n_dof], nullable = all free).  If dot != NULL, x'y over the
 * masked rows is ADDED to *dot (device double).                                                   */
int fem_spmv(const fem_plan* plan, const double* K_vals, const double* x, double* y, const uint8_t* free_mask,
             double* dot, fem_stream stream);
/* minv[i] = free_mask[i] ? 1/K[i,i] : 0   (Jacobi preconditioner with the Dirichlet rows removed) */
int fem_jacobi_setup(const fem_plan* plan, const double* K_vals, const uint8_t* free_mask, double* minv,
                     fem_stream stream);
/* PCG building blocks (device-resident scalars; used directly by the multi-GPU driver, which inserts
 * the halo exchange and the NCCL all-reduces between them).  scal is a device double[8]:
 * scal[0]=rz (even iterations), scal[1]=r'r, scal[2]=rz (odd iterations), scal[3]=p'Kp, scal[4]=|b|^2.
 * The sums are order-deterministic (block sums added in a fixed order by the last block to finish, not atomically): the
 * same inputs give the same bits.  The library keeps one 196 KB partial-sum buffer per distinct scal pointer (created by
 * the first call, which must not be inside a stream capture) and one per plan for the SpMV's x'y: run at most one
 * solve per scal array, and one dot-product SpMV per plan, at a time. */
int fem_pcg_init(int64_t n, const double* rhs, const double* Kx0, const uint8_t* free_mask, const double* minv,
                 double* r, double* p, double* scal, fem_stream stream);
int fem_pcg_spmv_dot(const fem_plan* plan, const double* K_vals, const double* p, double* q,
                     const uint8_t* free_mask, double* scal, int iter, fem_stream stream);
int fem_pcg_update_xr(int64_t n, const double* p, const double* q, const double* minv, double* x, double* r,
                      double* scal, int iter, fem_stream stream);
int fem_pcg_update_p(int64_t n, const double* r, const double* minv, double* p, double* scal, int iter,
                     fem_stream stream);
/* Multi-GPU variants over NVLink peer memory (one process per GPU; dst0/dst1 are the neighbours' ghost rows of the same
 * vector, mapped into this process by CUDA IPC / symmetric memory; NULL = no neighbour on that side).
 * fem_halo_push: dst0[0:n0] = v[src0:src0+n0], dst1[0:n1] = v[src1:src1+n1] (peer stores).
 * fem_pcg_update_p_push: fem_pcg_update_p restricted to the owned DOF range [own_lo, own_hi) and fused with that push of the
 * freshly computed p - the interface rows leave for the neighbours from the kernel that produces them instead of through
 * a separate send/recv.  Ghost rows of p are never written locally (their owners push them).                  */
int fem_halo_push(const double* v, int64_t src0, int64_t n0, double* dst0, int64_t src1, int64_t n1, double* dst1,
                  fem_stream stream);
int fem_pcg_update_p_push(int64_t own_lo, int64_t own_hi, const double* r, const double* minv, double* p, double* scal, int iter,
                          int64_t src0, int64_t n0, double* dst0, int64_t src1, int64_t n1, double* dst1, fem_stream stream);
/* Fused multi-GPU PCG iteration (csrc/peer_pcg.cu): the three exchanges of an iteration (ghost rows of p, p'q, {r'z, r'r})
 * leave from the kernel that produces them as NVLink peer stores (scalars as self-validating 16-byte lines, interface rows
 * followed by a release flag) and are awaited (bounded spin on local memory) by the kernel that consumes them.  No collective call and no host round trip inside an iteration, so the three
 * launches are CUDA-graph capturable; all ranks sum the partials in rank order and get bit-identical alpha and beta.
 * comm: this rank's communication block, fem_ppcg_words() 8-byte words of symmetric (peer-mapped) memory, zero-filled once
 *   at allocation; peers[r] = rank r's block as mapped into this process (host array of `world` device pointers, <= 16).
 * fem_ppcg_begin: call after fem_pcg_init and the all-reduce of scal[0:5]; loads {r'z, r'r} = scal[0:2] (local stores).
 *   The ghost rows of the initial p must be in place (fem_halo_push + a barrier across ranks) before the first iteration.
 * One iteration = fem_ppcg_spmv_dot, fem_ppcg_update_xr, fem_ppcg_update_p, the same number on every rank.
 * fem_ppcg_update_p: [own_lo, own_hi) = owned DOF range; p[src_up : src_up+n_up] is also stored to dst_up (the upper
 *   neighbour's ghost row, NULL if none), likewise *_lo.  Words FEM_PPCG_WORD_OUT, +1 of comm then hold the global r'z and
 *   r'r (doubles) and word FEM_PPCG_WORD_ERR is non-zero if a wait timed out (10 s, tuning key "peer_timeout_ms"; the results are
 *   then invalid).                         */
#define FEM_PPCG_WORDS 176     /* 8-byte words of a communication block */
#define FEM_PPCG_WORD_ERR 167  /* non-zero: a wait timed out */
#define FEM_PPCG_WORD_OUT 172  /* two doubles: global r'z, r'r after the last finished iteration */
int fem_ppcg_words(void);
int fem_ppcg_begin(void* comm, const double* scal, int world, fem_stream stream);
int fem_ppcg_spmv_dot(const fem_plan* plan, const double* K_vals, const double* p, double* q, const uint8_t* free_mask,
                      void* comm, const void* const* peers, int rank, int world, fem_stream stream);
int fem_ppcg_update_xr(const fem_plan* plan, const double* p, const double* q, const double* minv, double* x, double* r,
                       void* comm, const void* const* peers, int rank, int world, fem_stream stream);
int fem_ppcg_update_p(const fem_plan* plan, int64_t own_lo, int64_t own_hi, const double* r, const double* minv, double* p,
                      int64_t src_up, int64_t n_up, double* dst_up, int64_t src_lo, int64_t n_lo, double* dst_lo,
                      void* comm, const void* const* peers, int rank, int world, fem_stream stream);
/* Single-GPU Jacobi-PCG on K[Q,Q] x[Q] = rhs[Q], x[~Q] left untouched at 0.  work: 4*n_dof doubles.
 * Stops when |r| <= rtol*|rhs| (checked every check_every iterations).  Synchronises.            */
int fem_pcg(const fem_plan* plan, const double* K_vals, const double* rhs, const uint8_t* free_mask, double rtol,
            int maxit, int check_every, double* x, double* work, int* h_iters, double* h_relres, fem_stream stream);

/* ---- two-level additive preconditioner M^-1 = D^-1 + P A_c^-1 P^T (csrc/twolevel.cu) ---------------------------------
 * P: bilinear interpolation from a coarse grid of ncx x ncy cells of size hx x hy with origin (x0, y0) laid over the mesh's
 * bounding box to the fine nodes (coord = the (2, n_n) coordinates), Dirichlet rows zeroed; n_c = 2 (ncx+1)(ncy+1).
 * fem_coarse_galerkin: Ac[n_c][n_c] = P_row^T K P_col (zero-filled by the call, accumulated with FP64 atomics; once per matrix);
 *   P_row keeps the DOFs of row_mask, P_col those of col_mask (NULL = row_mask).  One GPU: both the free DOFs.  Strip-partitioned:
 *   row_mask = free AND owned, col_mask = free (ghost columns included), and the ranks' matrices are summed.
 * fem_dense_gemv: y = A x, dense row-major (applies the inverted coarse operator); if dot != NULL, *dot += x'y.
 * r'z is never formed by a pass of its own: r'z = r'D^-1 r + r'(P z_c) and r'(P z_c) = (P^T r)'z_c = rc'zc, so
 * fem_tl_init: r = mask (rhs - Kx0) (Kx0 nullable), rc = P^T r, scal[1] = r'r, scal[4] = |rhs|^2, scal[0] = r'D^-1 r
 *   (scal and rc zeroed first);
 * fem_tl_update_xr: x += alpha p, r -= alpha q, scal[1] += r'r, scal[rz_new] += r'D^-1 r, rc = P^T r (alpha from scal as in
 *   fem_pcg_update_xr); the coarse GEMV then adds rc'zc to the same slot through its `dot` argument;
 * fem_tl_apply: z = minv r + P zc;  mode 0: scal[slot] += r'z (checks);  mode 1: p = z;  mode 2: p = z + beta p.
 * Together with fem_pcg_spmv_dot these are the steps of the preconditioned CG; the host sequences them.                  */
int fem_coarse_galerkin(const fem_plan* plan, const double* K_vals, const uint8_t* row_mask, const uint8_t* col_mask,
                        const double* coord, double x0, double y0, double hx, double hy, int ncx, int ncy, double* Ac,
                        fem_stream stream);
int fem_dense_gemv(int n, const double* A, const double* x, double* y, double* dot, fem_stream stream);
int fem_tl_init(int64_t n_n, const double* rhs, const double* Kx0, const uint8_t* free_mask, const double* minv, const double* coord,
                double x0, double y0, double hx, double hy, int ncx, int ncy, double* r, double* rc, double* scal, fem_stream stream);
int fem_tl_update_xr(int64_t n_n, const double* p, const double* q, const double* minv, const double* coord, double x0, double y0,
                     double hx, double hy, int ncx, int ncy, double* x, double* r, double* rc, double* scal, int iter, fem_stream stream);
int fem_tl_apply(int64_t n_n, int mode, const double* r, const double* minv, const uint8_t* free_mask, const double* coord, double x0,
                 double y0, double hx, double hy, int ncx, int ncy, const double* zc, double* p, double* scal, int slot, int iter,
                 fem_stream stream);

/* ---- geometric multigrid V-cycle preconditioner (csrc/mg.cu) -------------------------------------------------------------
 * For meshes whose nodes lie on a uniform lattice (the uniform P1/Q1 meshes of the footing problem and of configs 1/4/5).
 * Level 0 is the mesh itself (the CSR matrix of the plan); level l >= 1 is a grid of bilinear (Q1) cells of 2^l lattice
 * steps, stored as a 9-point stencil of 2x2 blocks, S[(4*slot + 2*i + j) * n + node], slot = 3*(dy+1) + (dx+1); the
 * operators are Galerkin products A_{l+1} = P^T A_l P with P = bilinear interpolation, Dirichlet DOFs masked on level 0.
 * Smoother: Chebyshev polynomial of `degree` in D^-1 A (D = the nodes' 2x2 diagonal blocks), the same before and after the coarse correction,
 * so the V-cycle is a symmetric positive definite preconditioner for the CG of the Newton step
 * (replaces the dense LU of Plasticity2D_DP/pythonFEM.py:1062-1066; any SPD preconditioner gives the same solution).
 * Every transfer is a gather (no atomics): results are bit-reproducible run to run.
 * Strip partition: a level holds the owned node rows [own_lo, own_hi) plus one ghost row on each side that exists; row 0
 * of the local arrays is global row g0.  Ghost rows are refreshed by fem_mg_exchange descriptors: peer stores over NVLink
 * followed by a release flag, and an acquire wait for the neighbours' flags, in ONE small kernel (no library call, CUDA
 * graph capturable).  On one GPU every exchange is empty.  The host (mg.py) computes the layouts and owns all buffers.   */
#define FEM_MG_MAX_LEVELS 16
#define FEM_MG_MAX_DEGREE 8
#define FEM_MG_MAX_PEERS 16
typedef struct fem_mg_exchange {
  int32_t n_send, n_wait;
  int64_t src_off[FEM_MG_MAX_PEERS]; /* first node (double2) of the rows sent */
  int64_t count[FEM_MG_MAX_PEERS];   /* nodes sent */
  double* dst[FEM_MG_MAX_PEERS];     /* destination in the peer's copy of the same vector (peer-mapped address) */
  uint64_t* dst_flag[FEM_MG_MAX_PEERS];        /* flag word in the peer's communication block raised by this send */
  const uint64_t* wait_flag[FEM_MG_MAX_PEERS]; /* flag words in this rank's block the sources raise */
  uint64_t* seq;                     /* this rank: [0] sequence number of the exchange, [1] block ticket */
} fem_mg_exchange;
typedef struct fem_mg_level {
  int32_t nxn, nrows, g0, own_lo, own_hi, nrows_global; /* nodes per row, local rows, global index of local row 0, owned local rows */
  int32_t res_lo, res_hi;                               /* local rows of b this rank computes by restriction (= owned rows on a
                                                           distributed level; its share of the rows on the first replicated level) */
  const double* S;                                      /* [36][nxn*nrows] */
  const float* S32;                                     /* optional FP32 copy of S streamed by the smoother / residual (NULL: use S) */
  const double* dinv;                                   /* [4*nxn*nrows]: inverse 2x2 diagonal blocks, plane A[node] = (i00, i01), plane B = (i01, i11) */
  double *b, *xa, *xb, *d, *r;                          /* work vectors, [2*nxn*nrows] */
  double c1[FEM_MG_MAX_DEGREE], c2[FEM_MG_MAX_DEGREE];  /* Chebyshev recurrence d = c1 d + c2 D^-1 r */
  fem_mg_exchange ex_xa, ex_xb, ex_r, ex_b;             /* ex_b: gather of b to every rank (first replicated level) */
} fem_mg_level;
typedef struct fem_mg_desc {
  int32_t n_levels, degree;          /* structured levels (>= 1); the last one is solved with the dense inverse */
  int32_t LX, lat_rows, g0, nrows_global; /* level 0: lattice nodes per row, local lattice rows, global index of local row 0 */
  const int32_t* lat;                /* [lat_rows][LX] lattice point -> node (-1: none) */
  const int32_t* node_lat;           /* [n_n] node -> lattice point iy_local*LX + ix */
  int64_t own_node_lo, own_node_hi;  /* nodes of the owned lattice rows (a contiguous id range); ghost nodes are never written */
  const uint8_t* mask;               /* unknowns of this rank on level 0 (free AND owned) */
  const double* dinv;                /* level 0: masked inverse 2x2 diagonal blocks of the CURRENT matrix (fem_mg_block_jacobi), [2*n_dof] in two planes */
  double *xa, *xb, *d, *r;           /* level 0 work vectors [n_dof] */
  double c1[FEM_MG_MAX_DEGREE], c2[FEM_MG_MAX_DEGREE];
  fem_mg_exchange ex_xa, ex_xb, ex_r;
  fem_mg_level lev[FEM_MG_MAX_LEVELS]; /* lev[l-1] = level l */
  const double* coarse_inv;          /* dense inverse of the last level, [n_c][n_c], n_c = 2*nxn*nrows of that level */
  const float* K32;                  /* optional FP32 copy of K_vals (fem_mg_to_f32): streamed by the level-0 smoother and residual
                                        instead of the FP64 values (half the bytes; sums stay FP64); NULL = use K_vals */
  uint64_t* err;                     /* sticky word: a wait timed out (NULL on one GPU) */
  const float* lat32;                /* optional level-0 stencil (fem_mg_to_f32_lattice): node id == lattice point, 7-point pattern;
                                        [16][lat32_stride] planes 4*slot + 2*i + j, slots self, E, N, diagonal (upper half of the
                                        symmetric matrix).  Read by the V-cycle's level-0 smoother and residual instead of K32
                                        (NULL: block-CSR path) */
  int64_t lat32_stride;              /* plane stride (>= n_n, multiple of 32) */
  int32_t lat32_nw;                  /* diagonal slot: 1 = north-west (the lower partner is south-east), 0 = north-east */
  int32_t lat32_pad;
} fem_mg_desc;
int fem_mg_sizeof(int which); /* sizeof fem_mg_exchange (0), fem_mg_level (1), fem_mg_desc (2): checked by the binding */
/* set-up steps (once per mesh / per matrix the hierarchy is built from) */
int fem_mg_lattice(int64_t n_n, const double* coord, double x0, double y0, double hx, double hy, int LX, int lat_rows, int g0,
                   int32_t* lat, int32_t* node_lat, int32_t* err, fem_stream stream);
int fem_mg_galerkin_fine(const fem_plan* plan, const double* K_vals, const uint8_t* row_mask, const uint8_t* col_mask,
                         const int32_t* lat, int lat_rows, const int32_t* node_lat, int LX, int g0, int nxn, int nrows, int g0c,
                         double* S, int32_t* err, fem_stream stream); /* gather per level-1 node, no atomics: reproducible */
int fem_mg_galerkin_stencil(int nxf, int nrows_f, int g0f, int nrows_global_f, const double* Sf, int nxc, int nrows_c, int g0c,
                            int row_lo, int row_hi, double* Sc, fem_stream stream);
int fem_mg_level_finalize(int64_t n, double* S, double thresh, double* dinv, fem_stream stream);
/* dinv[2*n_dof]: inverse of every node's 2x2 diagonal block (block-Jacobi smoother), rows/columns of masked DOFs zero */
int fem_mg_block_jacobi(const fem_plan* plan, const double* K_vals, const uint8_t* mask, double* dinv, fem_stream stream);
int fem_mg_stencil_apply(int nxn, int nrows, int row_lo, int row_hi, const double* S, const double* x, double* y, fem_stream stream);
int fem_mg_stencil_to_dense(int nxn, int nrows, const double* S, double* A, fem_stream stream);
/* z = V(r): one V-cycle on the current matrix K_vals (level 0) and the stored coarse operators; if dot != NULL, *dot += r'z
 * over this rank's unknowns.  r must be zero on masked DOFs.                                         */
int fem_mg_vcycle(const fem_plan* plan, const fem_mg_desc* desc, const double* K_vals, const double* r, double* z, double* dot,
                  fem_stream stream);
/* vals[0:n] (n <= 8, device) <- sum over all ranks, through peer memory (no library call, CUDA-graph capturable).
 * comm: this rank's communication block; peers[r]: rank r's block as mapped here; lines_word: first of FEM_PEER_ALLREDUCE_WORDS
 * 8-byte words reserved for the lines; seq_word: sequence counter; err_word: sticky time-out word (all zero-filled once).   */
#define FEM_PEER_ALLREDUCE_WORDS 512
int fem_peer_allreduce(double* vals, int n, void* comm, const void* const* peers, int64_t lines_word, int64_t seq_word, int64_t err_word,
                       int rank, int world, fem_stream stream);
/* one level-0 step of the V-cycle on its own (benchmarks / tests): mode 1: out = mask .* (b - K x); mode 2 (Chebyshev step):
 * d = c1 d + c2 D^-1 (b - K x), out = x + d, *dot += b'out (dot nullable); d, D^-1, mask and the optional FP32 matrix from desc */
int fem_mg_fine_step(const fem_plan* plan, const fem_mg_desc* desc, int mode, const double* K_vals, const double* b, const double* x,
                     double* out, double c1, double c2, double* dot, fem_stream stream);
int fem_mg_to_f32(int64_t n, const double* src, float* dst, fem_stream stream); /* n % 4 == 0 (nnz of the 2x2-block pattern) */
/* level-0 stencil on the lattice.  _check (set-up, once per mesh): err |= 1 node id != lattice point, 2 a neighbour outside
 * the 3x3 window, 4 a north-east/south-west edge, 8 a north-west/south-east edge (the stencil needs err in {0, 4, 8}).
 * _to_f32_lattice (per matrix): one pass over K_vals writes the FP32 block-CSR copy k32 (== fem_mg_to_f32) and the planes of
 * fem_mg_desc.lat32.  _fine_step_lattice: fem_mg_fine_step on desc->lat32 (benchmarks, tests).                       */
int fem_mg_lattice_check(const fem_plan* plan, const int32_t* node_lat, int LX, int32_t* err, fem_stream stream);
int fem_mg_to_f32_lattice(const fem_plan* plan, const double* K_vals, float* k32, float* planes, int64_t stride, int LX, int nw,
                          fem_stream stream);
int fem_mg_fine_step_lattice(const fem_plan* plan, const fem_mg_desc* desc, int mode, const double* b, const double* x, double* out,
                             double c1, double c2, double* dot, fem_stream stream);
int fem_mg_exchange_run(const fem_mg_exchange* ex, double* v, uint64_t* err, fem_stream stream);
/* CG steps around the V-cycle (scal as in fem_pcg_*: [0]/[2] r'z by iteration parity, [1] r'r, [3] p'Kp, [4] |b|^2):
 * init: r = mask .* rhs, x = 0, scal zeroed, [1] = [4] = |r|^2;  update_xr: x += alpha p, r -= alpha q, [1] += r'r;
 * update_p: p = z + beta p (iter < 0: p = z), [3] = 0.                                               */
int fem_mg_pcg_init(int64_t n, const double* rhs, const uint8_t* mask, double* r, double* x, double* scal, fem_stream stream);
int fem_mg_pcg_update_xr(int64_t n, const double* p, const double* q, double* x, double* r, double* scal, int iter, fem_stream stream);
int fem_mg_pcg_update_p(int64_t n, const double* z, double* p, double* scal, int iter, fem_stream stream);

/* energy products for the Newton stopping criterion: out[i] = v_i' K v_i, i < 3 (device double[3], overwritten) */
int fem_energy_norms(const fem_plan* plan, const double* K_vals, const double* v0, const double* v1, const double* v2,
                     double* work, double* out, fem_stream stream);

/* out = a*x + b*y (n doubles; out may alias x or y): the vector updates of the Newton / load-stepping glue
 * (U_new = U_it + dU, :1069; U_it = d_zeta*(U-U_old)/d_zeta_old + U, :1120)                        */
int fem_vec_axpby(int64_t n, double a, const double* x, double b, const double* y, double* out, fem_stream stream);
/* transform(): integration-point values -> nodal weighted averages, q_node[n] = sum_g w_g q_g / sum_g w_g over the
 * points of the elements around node n (Plasticity2D_DP/pythonFEM.py:760-816)                      */
int fem_transform(const fem_plan* plan, const double* q_int, double* q_node, fem_stream stream);

/* Load vectors of the linear-elastic demo (Elasticity2D/pythonFEM.py:246-364).
 * fem_vector_volume: out[c*n_n + n] = sum_g hatp[la, q] * (weight[g] * f_int[c*n_int + g]) over the integration points of the
 *   elements around node n in ascending g - SciPy's summation order of the reference's COO triplets (:281-290), bit-identical.
 *   h_hatp: HOST (n_p, n_q) row-major basis values (get_local_basis_volume).  out is (2, n_n) like the reference's f_V.
 * fem_segment_sum_ordered: out[s] = sequential sum of vals[seg_ptr[s] : seg_ptr[s+1]] (one thread per segment): the ordered
 *   duplicate summation for contributions stably sorted by node (surface tractions, :327-362).                          */
int fem_vector_volume(const fem_plan* plan, const double* f_int, const double* h_hatp, double* out, fem_stream stream);
int fem_segment_sum_ordered(int64_t n_seg, const int64_t* seg_ptr, const double* vals, double* out, fem_stream stream);

/* P1 -> P2 midpoint enrichment (create_midpoints_P2, tsx-tunnel/pythonFEM.py:1508-1626) without the reference's O(n_e^2)
 * search: edge occurrences o = 3*element + edge (edges V2-V3, V3-V1, V1-V2) go into a device hash table keyed by the vertex
 * pair; a midpoint's index is the number of edges whose first occurrence precedes its own (prefix sum) - the reference's
 * visiting order, bit-identical numbering and coordinates.  Two calls because the output sizes are results:
 * fem_midpoints_p2_count: elem [3][n_e] int32 (0-based, DEVICE, must stay alive until _fill) -> opaque handle, n_mid, n_bnd
 *   (boundary edges) and status (bit 0: an edge is shared by more than two triangles; bit 1: two triangles traverse a shared
 *   edge in the same direction, for which the reference's neighbour-slot rule is undefined).  Synchronises the stream.
 * fem_midpoints_p2_fill: coord [2][n_n] -> coord_mid [2][n_mid] = (x_from + x_to) / 2 of the first occurrence;
 *   elem_mid [3][n_e] midpoint index of every element edge (the reference's elem_ed; elem_ext rows 3..5 = elem_mid + n_n);
 *   edge_el [2][n_mid] the elements of the first and (if shared, else 0) the second occurrence (:1536, :1544);
 *   surf [3][n_bnd] = (to vertex, from vertex, n_n + midpoint) per boundary edge in midpoint order (:1556, :1586, :1616).
 * fem_midpoints_p2_destroy frees the handle (after synchronising the stream).                                          */
int fem_midpoints_p2_count(int64_t n_n, int64_t n_e, const int32_t* elem, void** handle, int64_t* n_mid, int64_t* n_bnd,
                           int* status, fem_stream stream);
int fem_midpoints_p2_fill(void* handle, const double* coord, double* coord_mid, int32_t* elem_mid, int32_t* edge_el,
                          int32_t* surf, fem_stream stream);
int fem_midpoints_p2_destroy(void* handle, fem_stream stream);

/* launch-shape knobs for benchmarking ("return_map_variant", "assemble_variant", "assemble_warps", "spmv_group", "spmv_blocks_per_sm",
 * "spmv_staged", "peer_timeout_ms", "strain_variant", "assemble_canon", "mg_stencil_sym", "mg_fine_lattice" (2: the V-cycle's
 * level 0 reads the block-CSR copy even when the descriptor carries the lattice stencil));
 * value 0 restores the default.  Results never depend on them.                                     */
int fem_set_tuning(const char* key, int value);

#ifdef __cplusplus
}
#endif
#endif /* FEM_B200_H */

// Shared definitions for the sm_100a FEM kernels.  Compiled with -fmad=false: the assembly,
// strain and force kernels reproduce scipy's accumulation order bit-for-bit, so the compiler
// must not contract a*b+c.  Kernels that do not need that (SpMV, PCG) call fma() explicitly.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "../../include/fem_b200.h"

#define FEM_MAX_NP 8
#define FEM_MAX_NQ 9
#define FEM_WARP 32
#define FEM_INVALID_KEY 0xFFFFFFFFu
#define FEM_SLICE_COUNTERS 64  // dynamic-scheduler counters per plan (dscratch[8 .. 8 + FEM_SLICE_COUNTERS))
#define FEM_SPMV_TILE 256      // nodes (row pairs) per SpMV tile
#define FEM_SPMV_THREADS (2 * FEM_SPMV_TILE)  // CTA size of the tiled SpMV kernels: 4 lanes per node, 2 nodes in flight per lane group
#define FEM_SPMV_MAXSEG 4      // contiguous column ranges per tile
#define FEM_SPMV_CAP 1024      // staged x entries (nodes) per tile: 16 KB of shared memory per buffer
#define FEM_SPMV_DESC 12       // int32 words per tile descriptor
#define FEM_STAGE_MAXBOXW 96   // widest TMA box (elements); longer runs are split
// 2-D tensor map over `rows` SoA rows of n_int doubles (row stride n_int), box = rows x boxw
int fem_encode_rows_map(CUtensorMap* out, const double* base, int64_t n_int, int rows, int boxw);

void fem_set_error(const char* fmt, ...);

struct FemTuning {
  int return_map_variant;  // 0 auto, 1 scalar/256, 2 double2/128, 3 double2/256
  int assemble_warps;      // warps per block of the assembly kernel (0 = 4)
  int spmv_group;          // lanes per node in the SpMV (0 = by degree)
  int spmv_blocks_per_sm;  // 0 = 32
  int assemble_variant;    // 0 auto, 1 shared-memory accumulators (A), 2 register accumulators (B), 7 one-shot TMA (C), 6 persistent TMA (D), 8 persistent TMA with shared-memory accumulators (E)
  int spmv_unroll;         // nodes per lane group in flight (0 = default)
  int spmv_staged;         // 0 auto (every operand streamed through shared memory when the tiles fit, else as 2), 1 gather x from global memory (round-1 kernel), 2 x staged, matrix through registers
  int peer_timeout_ms;     // bound of the in-kernel waits of the fused multi-GPU PCG (0 = 10 000 ms)
  int assemble_canon;      // 0 auto (straight-line path for slices of the reference's regular triangulation), 2 off
  int strain_variant;      // 0/1 stored gradients (default), 2 P1 gradients recomputed from the coordinates (slower: L2 gathers)
  int mg_stencil_sym;      // 0 auto: coarse-level stencil sweeps read the lower half of the (symmetric) stencil as transposes of the neighbours' upper half; 2 = read all 36 planes
  int mg_fine_lattice;     // 0 auto: the V-cycle's level-0 smoother and residual read the lattice stencil when the descriptor carries one; 2 = the block-CSR copy
  int peer_nowait;         // DIAGNOSTIC ONLY: fused multi-GPU PCG kernels skip their waits (wrong results; isolates the wait time)
};
extern FemTuning g_fem_tuning;

#define FEM_CUDA_CHECK(expr)                                                                     \
  do {                                                                                           \
    cudaError_t _e = (expr);                                                                     \
    if (_e != cudaSuccess) {                                                                     \
      fem_set_error("%s failed at %s:%d: %s", #expr, __FILE__, __LINE__, cudaGetErrorString(_e)); \
      return FEM_ERR_CUDA;                                                                       \
    }                                                                                            \
  } while (0)

#define FEM_REQUIRE(cond, msg)                                    \
  do {                                                            \
    if (!(cond)) {                                                \
      fem_set_error("invalid argument: %s (%s)", msg, #cond);     \
      return FEM_ERR_INVALID_ARG;                                 \
    }                                                             \
  } while (0)

// Reference-element tables, passed by value as a kernel parameter (<= 1.3 KB).
struct FemRefElem {
  double dhat1[FEM_MAX_NP * FEM_MAX_NQ];  // (n_p, n_q) row-major
  double dhat2[FEM_MAX_NP * FEM_MAX_NQ];
  double wf[FEM_MAX_NQ];
};

struct fem_plan {
  int64_t n_n, n_e, n_int, n_dof, nnz, n_blocks;
  int n_p, n_q, max_degree, max_inc, sm_count;
  int meta_words;  // uint32 words of (la, pos[]) metadata per incidence
  FemRefElem ref;
  // mesh (device copies owned by the plan)
  int32_t* elem;  // [n_p][n_e]
  // node-block pattern and its CSR expansion
  int32_t* nbr_ptr;  // [n_n+1]
  int32_t* nbr_idx;  // [n_blocks], sorted per node, contains the node itself
  int32_t* row_ptr;  // [n_dof+1]
  int32_t* col_idx;  // [nnz]
  // node -> element incidences in sliced-ELL(32) layout, ascending element order per node
  int64_t n_slices;
  int64_t sell_entries;
  int32_t* inc_cnt;     // [n_n]
  int64_t* slice_ptr;   // [n_slices+1] entry offsets
  uint32_t* inc_key;    // [sell_entries]  (element << 3) | local node, FEM_INVALID_KEY = padding
  uint32_t* inc_meta;   // [meta_words][sell_entries]  byte-packed: word0 = la | pos0<<8 | pos1<<16 | pos2<<24, ...
  // geometry
  double* dphi1;   // [n_p][n_int]
  double* dphi2;   // [n_p][n_int]
  double* weight;  // [n_int]
  double2* coord2;  // [n_n] node coordinates (x, y) interleaved: one 16-byte gather per node (P1 strain kernel)
  // scratch
  double* dscratch;  // small device scratch: 8 doubles (PCG scalars) + FEM_SLICE_COUNTERS 8-byte counters
  double* red_partials;  // [3][FEM_RED_MAXB] block sums + ticket counter of the order-deterministic dot products of this plan's SpMV
  unsigned* red_ticket;
  // TMA staging data of the P1 assembly kernel (valid when stage_ok): per 32-node slice the touched elements as
  // <= FEM_STAGE_RMAX runs of consecutive ids (16-byte aligned), and per incidence its position in the staged buffer
  int stage_ok, stage_boxw;
  int64_t stage_fallback_slices;
  int64_t stage_canon_slices;  // slices of the reference's regular triangulation (straight-line path of the assembly)
  int32_t* stage_box;    // [n_slices][3]: number of boxes, start element of box 0, of box 1 (TMA path when <= 2 boxes)
  uint32_t* inc_stage;   // [sell_entries]: li | la<<9 | slot0<<11 | slot1<<15 | slot2<<19 | valid<<31, li = box*boxw + offset
  double* geom;          // one allocation [1 + 2*n_p][n_int]: weight, dphi1 rows, dphi2 rows (one TMA box brings all rows)
  double* geom_rec;      // [n_int][geom_rs] records (weight, dphi1[n_p], dphi2[n_p], padding to a multiple of 4 doubles) for the
                         // direct-load assembly kernels (P2 / Q1 / Q2, unstructured P1): a point's geometry in 2-5 whole sectors instead
                         // of 1 + 2 n_p sectors of the row arrays; nullptr when the TMA-staged P1 kernel serves the mesh
  int geom_rs;
  CUtensorMap geom_map;
  // x-staging plan of the SpMV (spmv.cuh): per tile of FEM_SPMV_TILE consecutive nodes the referenced columns as
  // <= FEM_SPMV_MAXSEG contiguous node ranges (brought into shared memory by bulk async copies), and per 2x2 block the
  // position of its column inside that staged buffer
  int64_t n_tiles;
  int32_t* tile_seg;   // [n_tiles][FEM_SPMV_DESC]: nseg (0 = gather from global), total nodes, (start, len) per segment, [10] first block, [11] blocks
  uint16_t* nbr_loc;   // [n_blocks]
  int64_t spmv_fallback_tiles;
  int tile_max_blocks;  // most 2x2 blocks in one tile (the streaming SpMV needs them to fit a shared-memory stage)
  int64_t bytes;
};

// ---- the regular triangulation of the reference's mesh generator (get_nodes_1, Plasticity2D_DP/pythonFEM.py:73-122) -------
// incidence k = 0..5 (ascending element id): local index of the node, and slots of the element's nodes 0, 1, 2 packed 4 bits each
//   k:      0        1        2        3        4        5
//   la:     1        2        2        1        0        0
//   slots: {0,3,2}  {0,1,3}  {1,4,3}  {2,3,5}  {3,6,5}  {3,4,6}
__host__ __device__ constexpr int canon_la(int k) { return (0x001221 >> (4 * k)) & 15; }
__host__ __device__ constexpr int canon_slot(int k, int lb) {
  return ((k == 0 ? 0x230 : k == 1 ? 0x310 : k == 2 ? 0x341 : k == 3 ? 0x532 : k == 4 ? 0x563 : 0x643) >> (4 * lb)) & 15;
}
constexpr uint32_t CANON_MASK = 0x807FFE00u;  // valid bit, la, the three slots (everything but the staged position)
__host__ __device__ constexpr uint32_t canon_word(int k) {
  return 0x80000000u | ((uint32_t)canon_la(k) << 9) | ((uint32_t)canon_slot(k, 0) << 11) | ((uint32_t)canon_slot(k, 1) << 15) |
         ((uint32_t)canon_slot(k, 2) << 19);
}
static_assert(canon_word(0) == 0x80118200u && canon_word(1) == 0x80188400u && canon_word(2) == 0x801a0c00u && canon_word(3) == 0x80299200u &&
                  canon_word(4) == 0x802b1800u && canon_word(5) == 0x80321800u, "canonical incidence words (oracle mesh)");


static inline int fem_div_up(int64_t a, int64_t b) { return (int)((a + b - 1) / b); }

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Block-wide sum (blockDim.x multiple of 32, <= 1024); result valid in thread 0.
__device__ __forceinline__ double block_sum(double v, double* smem /* >= 32 doubles */) {
  v = warp_sum(v);
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  if (lane == 0) smem[w] = v;
  __syncthreads();
  const int nw = (blockDim.x + 31) >> 5;
  v = (threadIdx.x < nw) ? smem[threadIdx.x] : 0.0;
  if (w == 0) v = warp_sum(v);
  __syncthreads();
  return v;
}

// Order-deterministic grid-wide sums.  Every block stores its sums (block_sum: a fixed tree) into its own slot of a buffer;
// the block that draws the last ticket adds the slots in a fixed order (lane-strided, then the butterfly) and adds the
// totals to their destinations - one addition by one thread, so `+=` onto a slot another kernel has zeroed keeps its
// meaning and the result does not depend on the order in which the blocks finish (atomicAdd of the block sums did).
// Grids larger than the buffer, or a missing buffer, fall back to atomics.  One buffer serves kernels that are ordered
// on a stream (the ticket counter wraps back to zero in every launch).
#define FEM_RED_MAXB 8192
struct FemRedBuf {
  double* partials;  // [3][FEM_RED_MAXB]
  unsigned* ticket;
};
template <int N>
__device__ __forceinline__ void ordered_accumulate(const double (&v)[N], double* const (&dst)[N], const FemRedBuf rb) {
  static_assert(N <= 3, "partial buffer holds three sums per block");
  if (gridDim.x > FEM_RED_MAXB || rb.partials == nullptr) {
    if (threadIdx.x == 0) {
#pragma unroll
      for (int i = 0; i < N; ++i) atomicAdd(dst[i], v[i]);
    }
    return;
  }
  __shared__ int s_last;
  if (threadIdx.x == 0) {
#pragma unroll
    for (int i = 0; i < N; ++i) rb.partials[i * FEM_RED_MAXB + blockIdx.x] = v[i];
    __threadfence();
    s_last = atomicInc(rb.ticket, gridDim.x - 1) == gridDim.x - 1;
  }
  __syncthreads();
  if (s_last && threadIdx.x < 32) {
    __threadfence();
#pragma unroll
    for (int i = 0; i < N; ++i) {
      double t = 0.0;
      for (unsigned b = threadIdx.x; b < gridDim.x; b += 32) t += __ldcg(rb.partials + i * FEM_RED_MAXB + b);
      t = warp_sum(t);
      if (threadIdx.x == 0) *dst[i] += t;
    }
  }
}
FemRedBuf fem_red_buffer_for(const void* key, cudaStream_t st);  // solver.cu: buffer registered for a scalar array (created on first use)

// streaming (read-once) loads/stores: keep them out of L1 so that L1 serves the gathers
__device__ __forceinline__ double ld_stream(const double* p) { return __ldcs(p); }
__device__ __forceinline__ double2 ld_stream2(const double2* p) { return __ldcs(p); }
__device__ __forceinline__ void st_stream(double* p, double v) { __stcs(p, v); }
__device__ __forceinline__ void st_stream2(double2* p, double2 v) { __stcs(p, v); }

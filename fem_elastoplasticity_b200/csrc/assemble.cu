// K3/K4/K6: stiffness assembly, strain and internal force.
//
// Assembly is a deterministic GATHER, not a scatter: one thread owns one node (two CSR rows), walks
// the node's incident elements in ascending element order (sliced-ELL incidence list, coalesced) and
// accumulates every entry of its two rows in exactly the order scipy's csr_matmat uses for
// K = B^T D B (Plasticity2D_DP/pythonFEM.py:595): ascending (element, quadrature point, strain row).
// No atomics, no zero-fill pass, every K value is written exactly once; with -fmad=false the values
// are bit-identical to the reference.  The 2*deg*2 row accumulators live in warp-private shared
// memory laid out [entry][lane] (conflict-free), and are written out as contiguous CSR row pairs.
#include <atomic>

#include "common.cuh"

struct AsmArgs {
  int64_t n_n, n_e, n_int, n_slices, sell_entries;
  const int32_t* nbr_ptr;
  const int64_t* slice_ptr;
  const uint32_t* inc_key;
  const uint32_t* inc_meta;
  const double* dphi1;
  const double* dphi2;
  const double* weight;
  const double* geom_rec;  // [n_int][geom_rs] geometry records (plan: direct-load kernels) or nullptr
  int geom_rs;
  // mode inputs
  const double* shear;  // MODE 0, 2
  const double* bulk;   // MODE 0, 2
  const double* DS;     // MODE 1, 2   [9][n_int]
  const double* Kel;    // MODE 2
  const double* S;      // FORCE       [>=3][n_int]
  double* K_vals;
  double* F;
  // TMA-staged variant
  const int32_t* stage_box;
  const uint32_t* inc_stage;
  int boxw;
  unsigned long long* slice_counter;  // dynamic tile scheduler of the persistent kernels (zeroed before launch)
  int acc_rows;         // 4 * max_degree
  int canon;            // 1: slices of the reference's regular triangulation take the straight-line path of variant D
  double dev2[9];       // 2*Dev (column-major) formed as numpy forms it (:579-582)
  double vol[9];
};

__device__ __forceinline__ bool g_canon_enabled(const AsmArgs& A) { return A.canon != 0; }

constexpr int ACC_LD = 33;  // padded leading dimension: bank = (entry + lane) mod 16 for doubles

enum { MODE_ELASTIC = 0, MODE_TANGENT = 1, MODE_TANGENT_REF = 2, MODE_FORCE_ONLY = 3 };

// Per (element, quadrature point) data and the terms both assembly kernels derive from it.
template <int NP, int MODE, bool FORCE>
struct PointData {
  double w, d1[NP], d2[NP];
  double raw[MODE == MODE_ELASTIC ? 2 : (MODE == MODE_TANGENT ? 9 : (MODE == MODE_TANGENT_REF ? 11 : 1))];
  double s[FORCE ? 3 : 1];
};

template <int NP, int MODE, bool FORCE>
__device__ __forceinline__ void load_point_geom(const AsmArgs& A, int64_t g, PointData<NP, MODE, FORCE>& P);

template <int NP, int MODE, bool FORCE>
__device__ __forceinline__ void load_point(const AsmArgs& A, int64_t g, PointData<NP, MODE, FORCE>& P) {
  const int64_t n_int = A.n_int;
  load_point_geom<NP, MODE, FORCE>(A, g, P);
  if (MODE == MODE_ELASTIC) {
    P.raw[0] = A.shear[g];
    P.raw[1] = A.bulk[g];
  } else if (MODE == MODE_TANGENT || MODE == MODE_TANGENT_REF) {
#pragma unroll
    for (int k = 0; k < 9; ++k) P.raw[k] = A.DS[(int64_t)k * n_int + g];
    if (MODE == MODE_TANGENT_REF) {
      P.raw[9] = A.shear[g];
      P.raw[10] = A.bulk[g];
    }
  }
  if (FORCE) {
    P.s[0] = A.S[g];
    P.s[1] = A.S[n_int + g];
    P.s[2] = A.S[2 * n_int + g];
  }
}

// The direct-load kernels (variants A and B) were bound by L2 sector traffic on elements with several quadrature points
// (ncu, P2: 835 M sectors per launch, L1 hit rate 3 %): a lane read the 1 + 2 NP + 9 values of a point from as many
// different rows of the [row][n_int] arrays, one 32-byte sector each for 8 useful bytes, and by the time the next point of
// the same element wanted the neighbouring 8 bytes the sector had left L1.  Two changes, same values and same arithmetic:
//   * the geometry of a point comes from a record [weight, dphi1[NP], dphi2[NP], padding] of the plan (geom_rec), read with
//     256-bit loads: (1 + 2 NP) / 4 whole sectors instead of 1 + 2 NP partial ones;
//   * the material / tangent-operator / stress rows of QC consecutive points of the element are loaded row by row before the
//     points are processed, so that the loads of one row hit the sector its first load brought in.
template <int NP>
__device__ __forceinline__ void load_geom_record(const AsmArgs& A, int64_t g, double& w, double (&d1)[NP], double (&d2)[NP]) {
  constexpr int NV = 1 + 2 * NP, RS = (NV + 3) & ~3;
  double v[RS];
  const double* rec = A.geom_rec + g * RS;
#pragma unroll
  for (int k = 0; k < RS; k += 4)
    asm volatile("ld.global.nc.v4.f64 {%0, %1, %2, %3}, [%4];" : "=d"(v[k]), "=d"(v[k + 1]), "=d"(v[k + 2]), "=d"(v[k + 3]) : "l"(rec + k));
  w = v[0];
#pragma unroll
  for (int p = 0; p < NP; ++p) {
    d1[p] = v[1 + p];
    d2[p] = v[1 + NP + p];
  }
}

// rows of QC consecutive points g0 .. g0 + QC - 1 (only the first `n` exist), row by row
template <int NP, int MODE, bool FORCE, int QC>
__device__ __forceinline__ void load_rows_chunk(const AsmArgs& A, int64_t g0, int n, PointData<NP, MODE, FORCE> (&P)[QC]) {
  const int64_t n_int = A.n_int;
  if (MODE == MODE_ELASTIC || MODE == MODE_TANGENT_REF) {
    constexpr int o = MODE == MODE_TANGENT_REF ? 9 : 0;
#pragma unroll
    for (int q = 0; q < QC; ++q) if (q < n) P[q].raw[o] = A.shear[g0 + q];
#pragma unroll
    for (int q = 0; q < QC; ++q) if (q < n) P[q].raw[MODE == MODE_FORCE_ONLY ? 0 : o + 1] = A.bulk[g0 + q];
  }
  if (MODE == MODE_TANGENT || MODE == MODE_TANGENT_REF) {
#pragma unroll
    for (int k = 0; k < 9; ++k)
#pragma unroll
      for (int q = 0; q < QC; ++q) if (q < n) P[q].raw[MODE == MODE_TANGENT || MODE == MODE_TANGENT_REF ? k : 0] = A.DS[(int64_t)k * n_int + g0 + q];
  }
  if (FORCE) {
#pragma unroll
    for (int k = 0; k < 3; ++k)
#pragma unroll
      for (int q = 0; q < QC; ++q) if (q < n) P[q].s[FORCE ? k : 0] = A.S[(int64_t)k * n_int + g0 + q];
  }
}

// geometry of one point: record (plan) when there is one, else the row arrays
template <int NP, int MODE, bool FORCE>
__device__ __forceinline__ void load_point_geom(const AsmArgs& A, int64_t g, PointData<NP, MODE, FORCE>& P) {
  if (A.geom_rec) {
    load_geom_record<NP>(A, g, P.w, P.d1, P.d2);
  } else {
    const int64_t n_int = A.n_int;
    P.w = A.weight[g];
#pragma unroll
    for (int p = 0; p < NP; ++p) {
      P.d1[p] = A.dphi1[(int64_t)p * n_int + g];
      P.d2[p] = A.dphi2[(int64_t)p * n_int + g];
    }
  }
}

// t = (B^T D)[dof, 3g + c] for the two DOFs of local node `la`, and the internal-force update.
template <int NP, int MODE, bool FORCE>
__device__ __forceinline__ void point_terms(const AsmArgs& A, const PointData<NP, MODE, FORCE>& P, int la, double (&tx)[3],
                                            double (&ty)[3], double& f0, double& f1) {
  const double w = P.w;
  double d1a = P.d1[0], d2a = P.d2[0];
#pragma unroll
  for (int p = 1; p < NP; ++p)
    if (p == la) {
      d1a = P.d1[p];
      d2a = P.d2[p];
    }
  if (FORCE) {  // F = B^T (w*s), csc_matvec order: strain rows 3g, 3g+1, 3g+2   (:1058)
    const double ws0 = w * P.s[0], ws1 = w * P.s[1], ws2 = w * P.s[2];
    f0 = (f0 + d1a * ws0) + d2a * ws2;
    f1 = (f1 + d2a * ws1) + d1a * ws2;
  }
  if (MODE == MODE_FORCE_ONLY) return;
  double D[9];  // D[r + 3c]
  if (MODE == MODE_ELASTIC) {            // vd = (2*dev*G + vol*K) * (1*w)        (:582,591)
#pragma unroll
    for (int k = 0; k < 9; ++k) D[k] = (A.dev2[k] * P.raw[0] + A.vol[k] * P.raw[1]) * w;
  } else if (MODE == MODE_TANGENT) {     // vD = w * ds                            (:1047)
#pragma unroll
    for (int k = 0; k < 9; ++k) D[k] = w * P.raw[k];
  } else {                               // D_p - D_elast                          (:1050)
#pragma unroll
    for (int k = 0; k < 9; ++k) D[k] = w * P.raw[k] - (A.dev2[k] * P.raw[MODE == MODE_TANGENT_REF ? 9 : 0] + A.vol[k] * P.raw[MODE == MODE_TANGENT_REF ? 10 : 0]) * w;
  }
  // B columns of node la: x-dof (d1,0,d2), y-dof (0,d2,d1)
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    tx[c] = d1a * D[3 * c] + d2a * D[2 + 3 * c];
    ty[c] = d2a * D[1 + 3 * c] + d1a * D[2 + 3 * c];
  }
}

// ---- variant A: accumulators in warp-private shared memory (any node degree) ---------------------
template <int NP, int NQ, int MODE, bool FORCE>
__global__ void __launch_bounds__(128) assemble_rows_kernel(const AsmArgs A) {
  extern __shared__ double smem[];
  constexpr int MW = (NP + 1 + 3) / 4;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t slice = (int64_t)blockIdx.x * (blockDim.x >> 5) + warp;
  if (slice >= A.n_slices) return;  // warp-uniform; only warp-level synchronisation below
  double* acc = smem + (size_t)warp * A.acc_rows * ACC_LD;
  const int64_t a = slice * 32 + lane;
  int deg = 0, base = 0;
  if (a < A.n_n) {
    const int nb = A.nbr_ptr[a];
    deg = A.nbr_ptr[a + 1] - nb;
    base = 4 * nb;
  }
  if (MODE != MODE_FORCE_ONLY)
    for (int k = 0; k < 4 * deg; ++k) acc[k * ACC_LD + lane] = 0.0;
  const int64_t sbase = A.slice_ptr[slice];
  const int width = (int)((A.slice_ptr[slice + 1] - sbase) >> 5);
  double f0 = 0.0, f1 = 0.0;
  for (int i = 0; i < width; ++i) {
    const int64_t at = sbase + (int64_t)i * 32 + lane;
    const uint32_t key = __ldcs(A.inc_key + at);
    if (key == FEM_INVALID_KEY) continue;
    const int64_t e = key >> 3;
    const int la = key & 7;
    uint32_t meta[MW];
#pragma unroll
    for (int w = 0; w < MW; ++w) meta[w] = __ldcs(A.inc_meta + (int64_t)w * A.sell_entries + at);
    // The 4*NP entries this incidence contributes to are distinct (distinct nodes of one element): they are taken out of
    // shared memory once, accumulated over the element's NQ quadrature points in registers - same order: ascending
    // (quadrature point, strain row) within the element - and put back, instead of a read-modify-write per point
    // (48 shared-memory accesses per point for P2, which bounded the kernel).
    double a4[NP][4];
    if (MODE != MODE_FORCE_ONLY) {
#pragma unroll
      for (int lb = 0; lb < NP; ++lb) {
        const int byte = lb + 1;
        const int slot = (meta[byte >> 2] >> (8 * (byte & 3))) & 0xFF;
        const double* r0 = acc + (2 * slot) * ACC_LD + lane;
        const double* r1 = acc + (2 * deg + 2 * slot) * ACC_LD + lane;
        a4[lb][0] = r0[0]; a4[lb][1] = r0[ACC_LD]; a4[lb][2] = r1[0]; a4[lb][3] = r1[ACC_LD];
      }
    }
    constexpr int QC = NQ >= 4 ? 4 : NQ;  // points whose rows are loaded together (load_rows_chunk)
#pragma unroll 1
    for (int q0 = 0; q0 < NQ; q0 += QC) {
      PointData<NP, MODE, FORCE> pc[QC];
      load_rows_chunk<NP, MODE, FORCE, QC>(A, e * NQ + q0, NQ - q0, pc);
#pragma unroll
      for (int qq = 0; qq < QC; ++qq) {
        if (q0 + qq >= NQ) break;
        double tx[3], ty[3];
        PointData<NP, MODE, FORCE>& pd = pc[qq];
        load_point_geom<NP, MODE, FORCE>(A, e * NQ + q0 + qq, pd);
        point_terms<NP, MODE, FORCE>(A, pd, la, tx, ty, f0, f1);
        if (MODE == MODE_FORCE_ONLY) continue;
#pragma unroll
        for (int lb = 0; lb < NP; ++lb) {
          const double b1 = pd.d1[lb], b2 = pd.d2[lb];
          a4[lb][0] = (a4[lb][0] + tx[0] * b1) + tx[2] * b2;  // K[2a  , 2b  ]
          a4[lb][1] = (a4[lb][1] + tx[1] * b2) + tx[2] * b1;  // K[2a  , 2b+1]
          a4[lb][2] = (a4[lb][2] + ty[0] * b1) + ty[2] * b2;  // K[2a+1, 2b  ]
          a4[lb][3] = (a4[lb][3] + ty[1] * b2) + ty[2] * b1;  // K[2a+1, 2b+1]
        }
      }
    }
    if (MODE != MODE_FORCE_ONLY) {
#pragma unroll
      for (int lb = 0; lb < NP; ++lb) {
        const int byte = lb + 1;
        const int slot = (meta[byte >> 2] >> (8 * (byte & 3))) & 0xFF;
        double* r0 = acc + (2 * slot) * ACC_LD + lane;
        double* r1 = acc + (2 * deg + 2 * slot) * ACC_LD + lane;
        r0[0] = a4[lb][0]; r0[ACC_LD] = a4[lb][1]; r1[0] = a4[lb][2]; r1[ACC_LD] = a4[lb][3];
      }
    }
  }
  if (FORCE && a < A.n_n) reinterpret_cast<double2*>(A.F)[a] = make_double2(f0, f1);
  if (MODE == MODE_FORCE_ONLY) return;
  __syncwarp();
  // write-out: the two rows of node t are 4*deg_t contiguous CSR values starting at base_t
  for (int t = 0; t < 32; ++t) {
    const int n4 = 4 * __shfl_sync(0xffffffffu, deg, t);
    const int bt = __shfl_sync(0xffffffffu, base, t);
    for (int l = lane; l < n4; l += 32) {
      double v = acc[l * ACC_LD + t];
      if (MODE == MODE_TANGENT_REF) v = A.Kel[bt + l] + v;  // csr_plus_csr: K_elast + correction
      __stcs(A.K_vals + bt + l, v);
    }
  }
}

// ---- variant B: accumulators in registers (node degree <= MAXDEG) ---------------------------------
// The slot a contribution goes to is data (position of the neighbour in the node's sorted list), so the
// 4*MAXDEG accumulators are addressed through a `switch`: every case touches compile-time register names.
// On structured meshes all lanes of a warp take the same case (same local topology) so the branch is
// warp-uniform; on irregular meshes the cases serialise but stay correct.  No shared memory: the whole
// 228 KB stay L1, which is what serves the re-reads of an element's DS/dphi by its three nodes.
template <int NP, int NQ, int MODE, bool FORCE, int MAXDEG>
__global__ void __launch_bounds__(128) assemble_rows_reg_kernel(const AsmArgs A) {
  constexpr int MW = (NP + 1 + 3) / 4;
  const int64_t a = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t slice = a >> 5;
  if (slice >= A.n_slices) return;
  const int lane = threadIdx.x & 31;
  int deg = 0;
  int64_t base = 0;
  if (a < A.n_n) {
    const int nb = A.nbr_ptr[a];
    deg = A.nbr_ptr[a + 1] - nb;
    base = 4 * (int64_t)nb;
  }
  double acc[MAXDEG][4];
#pragma unroll
  for (int j = 0; j < MAXDEG; ++j) acc[j][0] = acc[j][1] = acc[j][2] = acc[j][3] = 0.0;
  const int64_t sbase = A.slice_ptr[slice];
  const int width = (int)((A.slice_ptr[slice + 1] - sbase) >> 5);
  double f0 = 0.0, f1 = 0.0;
  // The incidence keys/metadata of a whole chunk are fetched up front (one memory latency instead of one per incidence).
  // Double-buffering the element data as well was measured slower: register pressure costs more occupancy than it hides.
  constexpr int CH = 8;
  using PD = PointData<NP, MODE, FORCE>;
  for (int c0 = 0; c0 < width; c0 += CH) {
    uint32_t keys[CH], metas[CH][MW];
#pragma unroll
    for (int i = 0; i < CH; ++i) {
      keys[i] = FEM_INVALID_KEY;
      if (c0 + i < width) {
        const int64_t at = sbase + (int64_t)(c0 + i) * 32 + lane;
        keys[i] = __ldcs(A.inc_key + at);
#pragma unroll
        for (int w = 0; w < MW; ++w) metas[i][w] = __ldcs(A.inc_meta + (int64_t)w * A.sell_entries + at);
      }
    }
    PD cur;
    const int n_it = (width - c0) < CH ? (width - c0) : CH;
#pragma unroll 1
    for (int i = 0; i < n_it; ++i) {  // rolled: keys[0] is the current incidence (register queue)
      const uint32_t key = keys[0];
      const bool valid = key != FEM_INVALID_KEY;
      const int64_t e = key >> 3;
      const int la = key & 7;
      uint32_t meta[MW];
#pragma unroll
      for (int w = 0; w < MW; ++w) meta[w] = metas[0][w];
#pragma unroll 1
      for (int q = 0; q < NQ; ++q) {
        if (valid) load_point<NP, MODE, FORCE>(A, e * NQ + q, cur);
        if (valid) {
          double tx[3], ty[3];
          point_terms<NP, MODE, FORCE>(A, cur, la, tx, ty, f0, f1);
#pragma unroll
          for (int lb = 0; lb < NP; ++lb) {
            const int byte = lb + 1;
            const int slot = (meta[byte >> 2] >> (8 * (byte & 3))) & 0xFF;
            const double b1 = cur.d1[lb], b2 = cur.d2[lb];
            const double p00 = tx[0] * b1, p01 = tx[2] * b2, p10 = tx[1] * b2, p11 = tx[2] * b1;
            const double p20 = ty[0] * b1, p21 = ty[2] * b2, p30 = ty[1] * b2, p31 = ty[2] * b1;
#define FEM_UPD(J)                               \
  case J:                                        \
    if (J < MAXDEG) {                            \
      acc[J < MAXDEG ? J : 0][0] = (acc[J < MAXDEG ? J : 0][0] + p00) + p01; \
      acc[J < MAXDEG ? J : 0][1] = (acc[J < MAXDEG ? J : 0][1] + p10) + p11; \
      acc[J < MAXDEG ? J : 0][2] = (acc[J < MAXDEG ? J : 0][2] + p20) + p21; \
      acc[J < MAXDEG ? J : 0][3] = (acc[J < MAXDEG ? J : 0][3] + p30) + p31; \
    }                                            \
    break;
            switch (slot) {
              FEM_UPD(0) FEM_UPD(1) FEM_UPD(2) FEM_UPD(3) FEM_UPD(4) FEM_UPD(5) FEM_UPD(6) FEM_UPD(7)
              FEM_UPD(8) FEM_UPD(9) FEM_UPD(10) FEM_UPD(11) FEM_UPD(12) FEM_UPD(13) FEM_UPD(14) FEM_UPD(15)
              default: break;
            }
#undef FEM_UPD
          }
        }
      }
#pragma unroll
      for (int k = 0; k + 1 < CH; ++k) {  // shift the key queue
        keys[k] = keys[k + 1];
#pragma unroll
        for (int w = 0; w < MW; ++w) metas[k][w] = metas[k + 1][w];
      }
    }
  }
  if (a >= A.n_n) return;
  if (FORCE) reinterpret_cast<double2*>(A.F)[a] = make_double2(f0, f1);
  double2* row0 = reinterpret_cast<double2*>(A.K_vals + base);
  double2* row1 = row0 + deg;
#pragma unroll
  for (int j = 0; j < MAXDEG; ++j)
    if (j < deg) {
      double2 v0 = make_double2(acc[j][0], acc[j][1]), v1 = make_double2(acc[j][2], acc[j][3]);
      if (MODE == MODE_TANGENT_REF) {  // csr_plus_csr: K_elast + correction
        const double2 k0 = reinterpret_cast<const double2*>(A.Kel + base)[j];
        const double2 k1 = reinterpret_cast<const double2*>(A.Kel + base)[deg + j];
        v0.x = k0.x + v0.x; v0.y = k0.y + v0.y; v1.x = k1.x + v1.x; v1.y = k1.y + v1.y;
      }
      __stcs(row0 + j, v0);
      __stcs(row1 + j, v1);
    }
}

// ---- TMA staging of the P1 kernel (variant D; node degree <= 8) -------------------------------------
// The elements touched by the 32 nodes of a slice form (on structured meshes) two runs of consecutive ids, each covered
// by one fixed-width box (plan: stage_box).  One lane brings the boxes into warp-private shared memory with 2-D TMA
// tensor copies (cp.async.bulk.tensor.2d completing on an mbarrier): one copy per tensor and box - all 7 geometry rows,
// all 9 DS rows, the 3 S rows - so 3 copies per box instead of 19 row copies (a 1-D bulk-copy version was TMA
// issue-rate bound, ~50 cycles per copy per SM).  Each element is fetched once per slice, fully coalesced, with ~20 KB
// in flight per warp regardless of occupancy; the accumulation then runs out of shared memory with exactly the
// arithmetic of variants A/B.  Slices that need more than two boxes take direct loads.
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

struct alignas(64) StageMaps {
  CUtensorMap geom;  // [7][n_int]  weight, dphi1[3], dphi2[3]
  CUtensorMap t0;    // MODE_ELASTIC: shear [1][n_int]; else DS [9][n_int]
  CUtensorMap t1;    // MODE_ELASTIC: bulk;  MODE_TANGENT_REF: shear
  CUtensorMap t2;    // MODE_TANGENT_REF: bulk
  CUtensorMap s;     // FORCE: S rows 0..2 [3][n_int]
};

__host__ __device__ constexpr int pad128(int bytes) { return (bytes + 127) & ~127; }

template <int MODE, bool FORCE>
struct StageLayout {
  static constexpr int NRAW = MODE == MODE_ELASTIC ? 2 : (MODE == MODE_TANGENT ? 9 : 11);
  // byte sizes of one box of each tensor, as a function of the box width
  __host__ __device__ static constexpr int geom_b(int w) { return pad128(7 * w * 8); }
  __host__ __device__ static constexpr int t0_b(int w) { return pad128((MODE == MODE_ELASTIC ? 1 : 9) * w * 8); }
  __host__ __device__ static constexpr int t1_b(int w) { return (MODE == MODE_ELASTIC || MODE == MODE_TANGENT_REF) ? pad128(w * 8) : 0; }
  __host__ __device__ static constexpr int t2_b(int w) { return MODE == MODE_TANGENT_REF ? pad128(w * 8) : 0; }
  __host__ __device__ static constexpr int s_b(int w) { return FORCE ? pad128(3 * w * 8) : 0; }
  __host__ __device__ static constexpr int box_b(int w) { return geom_b(w) + t0_b(w) + t1_b(w) + t2_b(w) + s_b(w); }
  __host__ __device__ static constexpr int warp_b(int w) { return 2 * box_b(w) + 128; }  // + mbarrier
};

__device__ __forceinline__ void tma_box_2d(uint32_t dst, const CUtensorMap* map, int c0, uint32_t bar) {
  asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(dst),
               "l"(map), "r"(c0), "r"(0), "r"(bar)
               : "memory");
}

#ifndef FEM_ASM_CHUNK
#define FEM_ASM_CHUNK 2  // consecutive slices per claim of the dynamic scheduler of variant D (measured: 1: see NC, 2: 0.922 ms, 4: 0.942, 8: 0.992, 16: 1.176)
#endif
#ifndef FEM_ASM_NC
#define FEM_ASM_NC 1     // interleaved claim counters of variant D (1, 2, 4: no difference once claims come in chunks of two)
#endif
#ifndef FEM_ASM_UNROLL
#define FEM_ASM_UNROLL 2  // incidence steps per rotation of the register queue in variant D (1, 2, 4 or 8)
#endif
// ---- variant D: persistent, software-pipelined TMA staging ------------------------------------------------------
// Each warp walks many slices and keeps the TMA engine one half-slice ahead: box 0 of slice s+1 is requested as soon as
// the incidences living in box 0 of slice s are consumed, box 1 of s+1 after box 1 of s.  The dependent chain (box table
// -> TMA -> compute -> store) of a slice is thereby overlapped with the computation of the previous one without any extra
// shared memory.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok = 0;
  do {
    asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
                 : "=r"(ok)
                 : "r"(bar), "r"(parity)
                 : "memory");
  } while (!ok);
}

template <int MODE, bool FORCE>
__device__ __forceinline__ void issue_box(const StageMaps& M, unsigned char* bb, int bw, int start, uint32_t bar) {
  using L = StageLayout<MODE, FORCE>;
  const uint32_t bytes = (uint32_t)((7 + L::NRAW + (FORCE ? 3 : 0)) * bw * 8);
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
  tma_box_2d(smem_u32(bb), &M.geom, start, bar);
  bb += L::geom_b(bw);
  tma_box_2d(smem_u32(bb), &M.t0, start, bar);
  bb += L::t0_b(bw);
  if (MODE == MODE_ELASTIC || MODE == MODE_TANGENT_REF) {
    tma_box_2d(smem_u32(bb), &M.t1, start, bar);
    bb += L::t1_b(bw);
  }
  if (MODE == MODE_TANGENT_REF) {
    tma_box_2d(smem_u32(bb), &M.t2, start, bar);
    bb += L::t2_b(bw);
  }
  if (FORCE) tma_box_2d(smem_u32(bb), &M.s, start, bar);
}

// ---- fast path of variant D for the reference's regular triangulation --------------------------------------------------
// On the uniform P1 meshes of the reference's generator (get_nodes_1, Plasticity2D_DP/pythonFEM.py:73-122: cells split along
// V2-V4, two triangles per cell, node id = ix + iy (nx + 1)) every interior node meets the same six elements in the same
// roles: its local index in each element and the positions of the element's three nodes in its sorted neighbour list are
// CONSTANTS (derived with the oracle's mesh; common.cuh).  A slice whose 32 incidence lists all carry exactly that pattern -
// flagged by the plan (build_stage: a warp vote on the incidence words); ~97 % of the slices of config 4 - is processed
// by straight-line code on lane 0's incidence words (the others' staged positions are two elements further per lane): no queue,
// no validity tests, no selects on the local node, and the accumulators addressed statically instead of through a
// `switch` on the slot.  Same incidences in the same order with the same arithmetic: bit-identical to the generic path
// (test_assembly_variants_agree_bitwise), which every other slice and every other mesh still takes.
template <int MODE, bool FORCE, int K, int MAXDEG>
__device__ __forceinline__ void canon_incidence(const AsmArgs& A, const unsigned char* box, const int o, const int bw, double (&acc)[MAXDEG][4],
                                                double& f0, double& f1) {
  using L = StageLayout<MODE, FORCE>;
  static_assert(MAXDEG >= 7, "the canonical node has seven neighbours");
  PointData<3, MODE, FORCE> pd;
  const double* g = reinterpret_cast<const double*>(box) + o;
  pd.w = g[0];
#pragma unroll
  for (int p = 0; p < 3; ++p) {
    pd.d1[p] = g[(1 + p) * bw];
    pd.d2[p] = g[(4 + p) * bw];
  }
  const unsigned char* bb = box + L::geom_b(bw);
  const double* t0 = reinterpret_cast<const double*>(bb) + o;
  if (MODE == MODE_ELASTIC) {
    pd.raw[0] = t0[0];
    pd.raw[1] = (reinterpret_cast<const double*>(bb + L::t0_b(bw)) + o)[0];
  } else {
#pragma unroll
    for (int k = 0; k < 9; ++k) pd.raw[k] = t0[k * bw];
    if (MODE == MODE_TANGENT_REF) {
      pd.raw[MODE == MODE_TANGENT_REF ? 9 : 0] = (reinterpret_cast<const double*>(bb + L::t0_b(bw)) + o)[0];
      pd.raw[MODE == MODE_TANGENT_REF ? 10 : 0] = (reinterpret_cast<const double*>(bb + L::t0_b(bw) + L::t1_b(bw)) + o)[0];
    }
  }
  if (FORCE) {
    const double* sp = reinterpret_cast<const double*>(bb + L::t0_b(bw) + L::t1_b(bw) + L::t2_b(bw)) + o;
#pragma unroll
    for (int k = 0; k < 3; ++k) pd.s[k] = sp[k * bw];
  }
  double tx[3], ty[3];
  point_terms<3, MODE, FORCE>(A, pd, canon_la(K), tx, ty, f0, f1);
#pragma unroll
  for (int lb = 0; lb < 3; ++lb) {
    const int slot = canon_slot(K, lb);  // compile-time after unrolling
    const double b1 = pd.d1[lb], b2 = pd.d2[lb];
    const double p00 = tx[0] * b1, p01 = tx[2] * b2, p10 = tx[1] * b2, p11 = tx[2] * b1;
    const double p20 = ty[0] * b1, p21 = ty[2] * b2, p30 = ty[1] * b2, p31 = ty[2] * b1;
    acc[slot][0] = (acc[slot][0] + p00) + p01;
    acc[slot][1] = (acc[slot][1] + p10) + p11;
    acc[slot][2] = (acc[slot][2] + p20) + p21;
    acc[slot][3] = (acc[slot][3] + p30) + p31;
  }
}

template <int MODE, bool FORCE, int MAXDEG, int BW>
__global__ void __launch_bounds__(352) assemble_rows_tmap_kernel(const AsmArgs A, const __grid_constant__ StageMaps M) {
  constexpr int NP = 3;
  using L = StageLayout<MODE, FORCE>;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int bw = BW ? BW : A.boxw;  // BW = 66 (uniform P1 meshes) folds every shared-memory offset into an immediate
  unsigned char* wbase = smem_raw + (size_t)warp * L::warp_b(bw);
  unsigned char* box0 = wbase;
  unsigned char* box1 = wbase + L::box_b(bw);
  uint64_t* mbar = reinterpret_cast<uint64_t*>(wbase + 2 * L::box_b(bw));  // [0] box 0, [1] box 1
  const uint32_t bar0 = smem_u32(mbar), bar1 = smem_u32(mbar + 1);
  if (lane == 0) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar0), "r"(1));
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar1), "r"(1));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncwarp();
  const int64_t n_slices = A.n_slices;
  // Dynamic tile scheduler: slices are claimed in ascending order from a global counter, so the set of slices in flight
  // is a window that slides smoothly through the mesh.  (A static warp + k*n_warps assignment advances in lock-step
  // rounds: the two node rows that share a row of elements then fetch it at the same instant and both miss in L2 -
  // measured 1.5x DRAM reads.)  The claim for slice s+2 is made while slice s is being computed.
  // The counter is claimed in CHUNKS of consecutive slices: one atomic per slice on a single address is a serial resource
  // (250 000 claims in 1 ms = the kernel's run time; the broadcast of the claimed value was 25 % of all stall samples,
  // profiles/r2w).  A warp owns two chunks at any time; the atomic for the chunk after the current one is issued when the
  // current chunk starts and its value is only read (shuffled from lane 0) one whole chunk later.
  // The chunks are dealt from FEM_ASM_NC interleaved counters (counter j hands out the chunks c = NC k + j to the CTAs with
  // blockIdx % NC == j): the counters advance at the same pace, so the set of slices in flight is still a window sliding
  // through the mesh, at 1/NC of the atomic rate per address.
  constexpr int CHUNK = FEM_ASM_CHUNK, NC = FEM_ASM_NC;
  unsigned long long pending = 0;  // lane 0: chunk index returned by the atomic in flight
  const int cj = (int)(blockIdx.x % NC);
  auto request = [&]() {
    if (lane == 0) pending = atomicAdd(A.slice_counter + cj, 1ULL) * NC + cj;
  };
  auto collect = [&]() -> int64_t { return (int64_t)__shfl_sync(0xffffffffu, pending, 0) * CHUNK; };
  request();
  int64_t cbase = collect();
  request();
  int cpos = 0;
  auto claim = [&]() -> int64_t {  // next slice of this warp's sequence
    if (cpos == CHUNK) {
      cbase = collect();
      request();
      cpos = 0;
    }
    return cbase + cpos++;
  };
  int64_t slice = claim();
  int64_t slice1 = claim();  // the slice after the current one
  uint32_t ph0 = 0, ph1 = 0;
  constexpr int CH = 8;  // plan guarantees <= 8 incidences per node when stage_ok
  // Per-slice bookkeeping, fetched one slice ahead (two for the SELL offsets the incidence words depend on):
  //   box table {nb, st0, st1}, node degree/base, SELL offset + width, incidence words.
  struct Book { int nb, cn, st0, st1, deg, width; int64_t base, sbase; };
  auto load_box = [&](int64_t s, Book& k) {
    k.nb = 0; k.cn = 0; k.st0 = 0; k.st1 = 0;
    if (s < n_slices) {
      const int raw = A.stage_box[s * 3];  // boxes | canonical flag << 8
      k.nb = raw & 0xFF; k.cn = (raw >> 8) & 1; k.st0 = A.stage_box[s * 3 + 1]; k.st1 = A.stage_box[s * 3 + 2];
    }
  };
  auto load_node = [&](int64_t s, Book& k) {
    k.deg = 0; k.base = 0;
    const int64_t a = s * 32 + lane;
    if (s < n_slices && a < A.n_n) {
      const int nbp = A.nbr_ptr[a];
      k.deg = A.nbr_ptr[a + 1] - nbp;
      k.base = 4 * (int64_t)nbp;
    }
  };
  auto load_sell = [&](int64_t s, Book& k) {
    k.sbase = 0; k.width = 0;
    if (s < n_slices) { k.sbase = A.slice_ptr[s]; k.width = (int)((A.slice_ptr[s + 1] - k.sbase) >> 5); }
  };
  Book cur, nxt;
  uint32_t words[CH], nwords[CH];
  // incidence words of a slice: canonical slices (flag from the plan) read lane 0's words - one sector per word instead of
  // four - and derive the staged positions (two elements further per lane)
  auto load_words = [&](const Book& k, uint32_t (&w)[CH]) {
    const bool cn = k.cn != 0 && A.canon != 0;
#pragma unroll
    for (int i = 0; i < CH; ++i) {
      w[i] = (i < k.width) ? __ldcs(A.inc_stage + k.sbase + (int64_t)i * 32 + (cn ? 0 : lane)) : 0u;
      if (cn && i < 6) w[i] += 2u * (uint32_t)lane;
    }
  };
  load_box(slice, cur); load_node(slice, cur); load_sell(slice, cur);
  load_sell(slice1, nxt);
  load_words(cur, words);
  if (slice < n_slices && lane == 0 && cur.nb >= 1 && cur.nb <= 2) {
    issue_box<MODE, FORCE>(M, box0, bw, cur.st0, bar0);
    if (cur.nb == 2) issue_box<MODE, FORCE>(M, box1, bw, cur.st1, bar1);
  }
  while (slice < n_slices) {
    const int64_t next = slice1;
    const int64_t slice2 = claim();
    // requests for the next slice (and the SELL offsets of the one after) fly during this slice's computation
    load_box(next, nxt);
    load_node(next, nxt);
    load_words(nxt, nwords);
    Book nn;
    load_sell(slice2, nn);
    const int nb = cur.nb;
    const bool staged = nb >= 1 && nb <= 2;
    const int64_t a = slice * 32 + lane;
    double acc[MAXDEG][4];
#pragma unroll
    for (int j = 0; j < MAXDEG; ++j) acc[j][0] = acc[j][1] = acc[j][2] = acc[j][3] = 0.0;
    double f0 = 0.0, f1 = 0.0;
        const bool canon = MAXDEG >= 7 && nb == 2 && cur.cn != 0 && g_canon_enabled(A);  // flag set by build_stage (plan.cu)
    if (canon) {
      mbar_wait(bar0, ph0);
      ph0 ^= 1;
      canon_incidence<MODE, FORCE, 0, MAXDEG>(A, box0, (int)(words[0] & 0x1FF), bw, acc, f0, f1);
      canon_incidence<MODE, FORCE, 1, MAXDEG>(A, box0, (int)(words[1] & 0x1FF), bw, acc, f0, f1);
      canon_incidence<MODE, FORCE, 2, MAXDEG>(A, box0, (int)(words[2] & 0x1FF), bw, acc, f0, f1);
      __syncwarp();
      if (lane == 0 && nxt.nb >= 1 && nxt.nb <= 2) issue_box<MODE, FORCE>(M, box0, bw, nxt.st0, bar0);
      mbar_wait(bar1, ph1);
      ph1 ^= 1;
      canon_incidence<MODE, FORCE, 3, MAXDEG>(A, box1, (int)(words[3] & 0x1FF) - bw, bw, acc, f0, f1);
      canon_incidence<MODE, FORCE, 4, MAXDEG>(A, box1, (int)(words[4] & 0x1FF) - bw, bw, acc, f0, f1);
      canon_incidence<MODE, FORCE, 5, MAXDEG>(A, box1, (int)(words[5] & 0x1FF) - bw, bw, acc, f0, f1);
      __syncwarp();
      if (lane == 0 && nxt.nb == 2) issue_box<MODE, FORCE>(M, box1, bw, nxt.st1, bar1);
    } else
#pragma unroll 1
    for (int pass = 0; pass < 2; ++pass) {
      // pass 0: incidences whose element lives in box 0 (or every incidence on the direct-load path); pass 1: box 1.
      // A node's incidences are ascending in element id and box 0 precedes box 1, so the accumulation order is kept.
      if (staged) {
        if (pass == 0) { mbar_wait(bar0, ph0); ph0 ^= 1; }
        else if (nb == 2) { mbar_wait(bar1, ph1); ph1 ^= 1; }
      }
      if (pass == 0 || (staged && nb == 2)) {
        // The incidence words live in registers; a runtime loop can only address them by rotating the queue (16 register
        // moves per step in SASS: 20 % of the kernel's instructions, all on the serial path - profiles/r2c_D).  UN steps
        // are unrolled with static indices and the queue is rotated by UN at once: back in place after CH steps.
        // Measured (16M elements, tangent + force): UN = 1: 1.118 ms, 2: 1.109, 4: 1.143, 8: 1.300 (4 400 SASS instructions:
        // instruction-cache misses) - the moves are not what the kernel waits for.  Fused multiply-adds in the one-pass
        // tangent (-34 FP64 instructions per incidence, not bit-exact): 1.099 vs 1.107 ms, not kept.
        constexpr int UN = FEM_ASM_UNROLL;
        static_assert(CH % UN == 0, "unroll factor");
#pragma unroll 1
        for (int i0 = 0; i0 < CH; i0 += UN) {
#pragma unroll
        for (int k0 = 0; k0 < UN; ++k0) {
          const int i = i0 + k0;
          const uint32_t word = words[k0];
          if (!(word & 0x80000000u)) continue;
          const int li = word & 0x1FF;
          if (staged && ((li >= bw) != (pass == 1))) continue;
          const int la = (word >> 9) & 3;
          PointData<NP, MODE, FORCE> pd;
          if (staged) {
            const int o = li - pass * bw;
            const unsigned char* bb = pass ? box1 : box0;
            const double* g = reinterpret_cast<const double*>(bb) + o;
            pd.w = g[0];
#pragma unroll
            for (int p = 0; p < NP; ++p) {
              pd.d1[p] = g[(1 + p) * bw];
              pd.d2[p] = g[(4 + p) * bw];
            }
            bb += L::geom_b(bw);
            const double* t0 = reinterpret_cast<const double*>(bb) + o;
            if (MODE == MODE_ELASTIC) {
              pd.raw[0] = t0[0];
              pd.raw[1] = (reinterpret_cast<const double*>(bb + L::t0_b(bw)) + o)[0];
            } else {
#pragma unroll
              for (int k = 0; k < 9; ++k) pd.raw[k] = t0[k * bw];
              if (MODE == MODE_TANGENT_REF) {
                pd.raw[MODE == MODE_TANGENT_REF ? 9 : 0] = (reinterpret_cast<const double*>(bb + L::t0_b(bw)) + o)[0];
                pd.raw[MODE == MODE_TANGENT_REF ? 10 : 0] = (reinterpret_cast<const double*>(bb + L::t0_b(bw) + L::t1_b(bw)) + o)[0];
              }
            }
            if (FORCE) {
              const double* sp = reinterpret_cast<const double*>(bb + L::t0_b(bw) + L::t1_b(bw) + L::t2_b(bw)) + o;
#pragma unroll
              for (int k = 0; k < 3; ++k) pd.s[k] = sp[k * bw];
            }
          } else {  // direct loads (slices with more than two boxes); i-th entry of the queue is incidence i
            const uint32_t key = A.inc_key[cur.sbase + (int64_t)i * 32 + lane];
            load_point<NP, MODE, FORCE>(A, (int64_t)(key >> 3), pd);
          }
          double tx[3], ty[3];
          point_terms<NP, MODE, FORCE>(A, pd, la, tx, ty, f0, f1);
#pragma unroll
          for (int lb = 0; lb < NP; ++lb) {
            const int slot = (word >> (11 + 4 * lb)) & 15;
            const double b1 = pd.d1[lb], b2 = pd.d2[lb];
            const double p00 = tx[0] * b1, p01 = tx[2] * b2, p10 = tx[1] * b2, p11 = tx[2] * b1;
            const double p20 = ty[0] * b1, p21 = ty[2] * b2, p30 = ty[1] * b2, p31 = ty[2] * b1;
#define FEM_UPD(J)                               \
  case J:                                        \
    if (J < MAXDEG) {                            \
      acc[J < MAXDEG ? J : 0][0] = (acc[J < MAXDEG ? J : 0][0] + p00) + p01; \
      acc[J < MAXDEG ? J : 0][1] = (acc[J < MAXDEG ? J : 0][1] + p10) + p11; \
      acc[J < MAXDEG ? J : 0][2] = (acc[J < MAXDEG ? J : 0][2] + p20) + p21; \
      acc[J < MAXDEG ? J : 0][3] = (acc[J < MAXDEG ? J : 0][3] + p30) + p31; \
    }                                            \
    break;
            switch (slot) {
              FEM_UPD(0) FEM_UPD(1) FEM_UPD(2) FEM_UPD(3) FEM_UPD(4) FEM_UPD(5) FEM_UPD(6) FEM_UPD(7)
              default: break;
            }
#undef FEM_UPD
          }
        }
        if (UN < CH) {  // rotate by UN
          uint32_t head[UN];
#pragma unroll
          for (int k = 0; k < UN; ++k) head[k] = words[k];
#pragma unroll
          for (int k = 0; k + UN < CH; ++k) words[k] = words[k + UN];
#pragma unroll
          for (int k = 0; k < UN; ++k) words[CH - UN + k] = head[k];
        }
        }
      }
      __syncwarp();  // every lane is done reading this pass's box: it may be overwritten by the next slice's copy
      if (lane == 0 && nxt.nb >= 1 && nxt.nb <= 2) {
        if (pass == 0) issue_box<MODE, FORCE>(M, box0, bw, nxt.st0, bar0);
        else if (nxt.nb == 2) issue_box<MODE, FORCE>(M, box1, bw, nxt.st1, bar1);
      }
    }
    if (MAXDEG >= 7 && canon && A.canon == 1 && __all_sync(0xffffffffu, cur.deg == 7)) {
      // Canonical slice: every node has 7 neighbours, so a lane's two rows are 28 consecutive doubles = seven whole 32-byte
      // sectors (K_vals 32-byte aligned: checked at launch).  Seven 256-bit stores (STG.256) write each sector once; the
      // 16-byte stores of the generic path below write every sector in two halves from two instructions.
      if (FORCE) reinterpret_cast<double2*>(A.F)[a] = make_double2(f0, f1);
      double* dst = A.K_vals + cur.base;
#pragma unroll
      for (int k = 0; k < 7; ++k) {
        // doubles 4k .. 4k+3 of [row 2a: acc[j][0], acc[j][1], j = 0..6 | row 2a+1: acc[j][2], acc[j][3]]
        double v[4];
#pragma unroll
        for (int t = 0; t < 4; ++t) {
          const int i = 4 * k + t;
          v[t] = i < 14 ? acc[(i >> 1) < MAXDEG ? (i >> 1) : 0][i & 1] : acc[((i - 14) >> 1) < MAXDEG ? ((i - 14) >> 1) : 0][2 + ((i - 14) & 1)];
        }
        if (MODE == MODE_TANGENT_REF) {  // csr_plus_csr: K_elast + correction; K_elast streamed as whole sectors too
          double k0, k1, k2, k3;
          asm volatile("ld.global.nc.L1::no_allocate.v4.f64 {%0, %1, %2, %3}, [%4];" : "=d"(k0), "=d"(k1), "=d"(k2), "=d"(k3) : "l"(A.Kel + cur.base + 4 * k));
          v[0] = k0 + v[0]; v[1] = k1 + v[1]; v[2] = k2 + v[2]; v[3] = k3 + v[3];
        }
        asm volatile("st.global.cs.v4.f64 [%0], {%1, %2, %3, %4};" ::"l"(dst + 4 * k), "d"(v[0]), "d"(v[1]), "d"(v[2]), "d"(v[3]) : "memory");
      }
    } else if (a < A.n_n) {
      const int deg = cur.deg;
      if (FORCE) reinterpret_cast<double2*>(A.F)[a] = make_double2(f0, f1);
      double2* row0 = reinterpret_cast<double2*>(A.K_vals + cur.base);
      double2* row1 = row0 + deg;
#pragma unroll
      for (int j = 0; j < MAXDEG; ++j)
        if (j < deg) {
          double2 v0 = make_double2(acc[j][0], acc[j][1]), v1 = make_double2(acc[j][2], acc[j][3]);
          if (MODE == MODE_TANGENT_REF) {  // csr_plus_csr: K_elast + correction
            const double2 k0 = reinterpret_cast<const double2*>(A.Kel + cur.base)[j];
            const double2 k1 = reinterpret_cast<const double2*>(A.Kel + cur.base)[deg + j];
            v0.x = k0.x + v0.x; v0.y = k0.y + v0.y; v1.x = k1.x + v1.x; v1.y = k1.y + v1.y;
          }
          __stcs(row0 + j, v0);
          __stcs(row1 + j, v1);
        }
    }
    slice = next;
    slice1 = slice2;
    cur.nb = nxt.nb; cur.cn = nxt.cn; cur.st0 = nxt.st0; cur.st1 = nxt.st1; cur.deg = nxt.deg; cur.base = nxt.base;
    cur.sbase = nxt.sbase; cur.width = nxt.width;
    nxt.sbase = nn.sbase; nxt.width = nn.width;
#pragma unroll
    for (int i = 0; i < CH; ++i) words[i] = nwords[i];
  }
}

template <int MODE, bool FORCE>
static int launch_assemble_tma(const fem_plan* P, AsmArgs& A, cudaStream_t st) {
  using L = StageLayout<MODE, FORCE>;
  const int bw = P->stage_boxw;
  A.stage_box = P->stage_box;
  A.inc_stage = P->inc_stage;
  A.boxw = bw;
  if (A.canon == 1 && ((reinterpret_cast<uintptr_t>(A.K_vals) | reinterpret_cast<uintptr_t>(A.Kel)) & 31u) != 0) A.canon = 2;  // 256-bit accesses need whole sectors
  auto mis = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) != 0; };
  if ((A.DS && mis(A.DS)) || (A.shear && mis(A.shear)) || (A.bulk && mis(A.bulk)) || (FORCE && mis(A.S))) return -1;  // TMA needs 16-byte aligned rows
  StageMaps M;
  memset(&M, 0, sizeof(M));
  M.geom = P->geom_map;
  int rc = FEM_OK;
  if (MODE == MODE_ELASTIC) {
    if ((rc = fem_encode_rows_map(&M.t0, A.shear, P->n_int, 1, bw)) != FEM_OK) return rc;
    if ((rc = fem_encode_rows_map(&M.t1, A.bulk, P->n_int, 1, bw)) != FEM_OK) return rc;
  } else {
    if ((rc = fem_encode_rows_map(&M.t0, A.DS, P->n_int, 9, bw)) != FEM_OK) return rc;
    if (MODE == MODE_TANGENT_REF) {
      if ((rc = fem_encode_rows_map(&M.t1, A.shear, P->n_int, 1, bw)) != FEM_OK) return rc;
      if ((rc = fem_encode_rows_map(&M.t2, A.bulk, P->n_int, 1, bw)) != FEM_OK) return rc;
    }
  }
  if (FORCE && (rc = fem_encode_rows_map(&M.s, A.S, P->n_int, 3, bw)) != FEM_OK) return rc;
  auto kern = (bw == 66) ? assemble_rows_tmap_kernel<MODE, FORCE, 8, 66> : assemble_rows_tmap_kernel<MODE, FORCE, 8, 0>;
  const size_t per_warp = L::warp_b(bw);
  // warps per CTA that packs the most warps into the 227 KB of an SM (1 KB per CTA is reserved)
  int warps = 4, best = 0;
  for (int w = 4; w <= 11; ++w) {
    const size_t sm = (size_t)w * per_warp;
    const int per = (int)((227 * 1024) / (sm + 1024));
    if (per * w >= best) { best = per * w; warps = w; }
  }
  const size_t smem = (size_t)warps * per_warp;
  if (smem > 227 * 1024) return -1;
  FEM_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int per_sm = 0;
  FEM_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, warps * 32, smem));
  if (per_sm < 1) return -1;
  int64_t blocks = (int64_t)per_sm * P->sm_count;
  const int64_t need = fem_div_up(P->n_slices, warps);
  if (blocks > need) blocks = need;
  // one of FEM_SLICE_COUNTERS counters of this plan, round-robin per launch (atomic: host threads may launch concurrently),
  // so up to FEM_SLICE_COUNTERS launches of one plan may be in flight on different streams without sharing a counter
  // (the kernel spreads its claims over FEM_ASM_NC interleaved counters: a group of FEM_ASM_NC consecutive ones)
  static std::atomic<unsigned> launch_no{0};
  static_assert(FEM_SLICE_COUNTERS % FEM_ASM_NC == 0, "counter groups");
  A.slice_counter = reinterpret_cast<unsigned long long*>(P->dscratch + 8) + FEM_ASM_NC * (launch_no.fetch_add(1u) % (FEM_SLICE_COUNTERS / FEM_ASM_NC));
  FEM_CUDA_CHECK(cudaMemsetAsync(A.slice_counter, 0, FEM_ASM_NC * sizeof(unsigned long long), st));
  kern<<<(unsigned)blocks, warps * 32, smem, st>>>(A, M);
  FEM_CUDA_CHECK(cudaGetLastError());
  return FEM_OK;
}

// host-formed constants, exactly as numpy does at Plasticity2D_DP/pythonFEM.py:579-582
static void elastic_coeffs(double* dev2, double* vol) {
  const double iota[3] = {1.0, 1.0, 0.0};
  const double diag[3] = {1.0, 1.0, 0.5};
  for (int c = 0; c < 3; ++c)
    for (int r = 0; r < 3; ++r) {
      const volatile double v = iota[r] * iota[c];
      const volatile double third = v / 3.0;
      const volatile double dev = (r == c ? diag[r] : 0.0) - third;
      dev2[r + 3 * c] = 2.0 * dev;
      vol[r + 3 * c] = v;
    }
}

struct DmatCoef { double dev2[9], vol[9]; };
__global__ void elastic_dmat_kernel(int64_t n_int, DmatCoef k, const double* __restrict__ shear, const double* __restrict__ bulk,
                                    const double* __restrict__ weight, double* __restrict__ vd) {
  for (int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; g < n_int; g += (int64_t)gridDim.x * blockDim.x) {
    const double G = shear[g], Kb = bulk[g], w = weight[g];
#pragma unroll
    for (int q = 0; q < 9; ++q) vd[(int64_t)q * n_int + g] = (k.dev2[q] * G + k.vol[q] * Kb) * w;
  }
}

extern "C" int fem_elastic_dmat(const fem_plan* P, const double* shear, const double* bulk, double* vd, fem_stream stream) {
  FEM_REQUIRE(P && shear && bulk && vd, "null pointer");
  DmatCoef k;
  elastic_coeffs(k.dev2, k.vol);
  int64_t b = (P->n_int + 255) / 256;
  if (b > (int64_t)P->sm_count * 64) b = (int64_t)P->sm_count * 64;
  elastic_dmat_kernel<<<(unsigned)b, 256, 0, (cudaStream_t)stream>>>(P->n_int, k, shear, bulk, P->weight, vd);
  FEM_CUDA_CHECK(cudaGetLastError());
  return FEM_OK;
}

template <int MODE, bool FORCE>
static int launch_assemble(const fem_plan* P, AsmArgs& A, cudaStream_t st) {
  // variant B (register accumulators) for P1/Q1 meshes of bounded valence; variant A (shared memory) otherwise
  const int variant = g_fem_tuning.assemble_variant;
  // measured defaults (tools/tune.py, tools/ab_assemble.py, 16M elements): persistent pipelined TMA kernel; the reference-order
  // tangent (reads K_elast in its write-out) takes it where the straight-line path with 256-bit accesses covers most slices
  // (1.14 ms against 1.51 ms of the register kernel), else the register kernel
  const bool ref_tma = MODE != MODE_TANGENT_REF || (2 * P->stage_canon_slices >= P->n_slices && g_fem_tuning.assemble_canon != 2);
  if (MODE != MODE_FORCE_ONLY && P->stage_ok && ((variant == 0 && ref_tma) || variant == 6)) {
    const int rc = launch_assemble_tma<MODE == MODE_FORCE_ONLY ? MODE_TANGENT : MODE, FORCE>(P, A, st);
    if (rc >= 0) return rc;  // -1: inputs not 16-byte aligned / too much shared memory -> register kernel
  }
  if (MODE != MODE_FORCE_ONLY && variant != 1) {
    const unsigned blocks = (unsigned)fem_div_up(P->n_slices * 32, 128);
    bool done = true;
    if (P->n_p == 3 && P->n_q == 1 && P->max_degree <= 8) assemble_rows_reg_kernel<3, 1, MODE, FORCE, 8><<<blocks, 128, 0, st>>>(A);
    else if (P->n_p == 3 && P->n_q == 1 && P->max_degree <= 12) assemble_rows_reg_kernel<3, 1, MODE, FORCE, 12><<<blocks, 128, 0, st>>>(A);
    else if (P->n_p == 4 && P->n_q == 4 && P->max_degree <= 12) assemble_rows_reg_kernel<4, 4, MODE, FORCE, 12><<<blocks, 128, 0, st>>>(A);
    else done = false;
    if (done) {
      FEM_CUDA_CHECK(cudaGetLastError());
      return FEM_OK;
    }
  }
  const int warps = 4;
  int acc_rows = (MODE == MODE_FORCE_ONLY) ? 0 : 4 * P->max_degree;
  A.acc_rows = acc_rows;
  size_t smem = (size_t)warps * acc_rows * ACC_LD * sizeof(double);
  int threads = warps * 32;
  if (smem > 200 * 1024) {  // very high valence: one warp per block
    threads = 32;
    smem = (size_t)acc_rows * ACC_LD * sizeof(double);
    if (smem > 227 * 1024) {
      fem_set_error("node degree %d needs %zu B of shared memory", P->max_degree, smem);
      return FEM_ERR_UNSUPPORTED;
    }
  }
  const unsigned blocks = (unsigned)fem_div_up(P->n_slices, threads / 32);
#define LAUNCH(NP, NQ)                                                                                          \
  do {                                                                                                          \
    auto kern = assemble_rows_kernel<NP, NQ, MODE, FORCE>;                                                      \
    if (smem > 48 * 1024) FEM_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
    kern<<<blocks, threads, smem, st>>>(A);                                                                     \
  } while (0)
  if (P->n_p == 3 && P->n_q == 1) LAUNCH(3, 1);
  else if (P->n_p == 6 && P->n_q == 7) LAUNCH(6, 7);
  else if (P->n_p == 4 && P->n_q == 4) LAUNCH(4, 4);
  else if (P->n_p == 8 && P->n_q == 9) LAUNCH(8, 9);
  else {
    fem_set_error("unsupported element n_p=%d n_q=%d", P->n_p, P->n_q);
    return FEM_ERR_UNSUPPORTED;
  }
#undef LAUNCH
  FEM_CUDA_CHECK(cudaGetLastError());
  return FEM_OK;
}

static void fill_args(const fem_plan* P, AsmArgs& A) {
  memset(&A, 0, sizeof(A));
  A.n_n = P->n_n; A.n_e = P->n_e; A.n_int = P->n_int; A.n_slices = P->n_slices; A.sell_entries = P->sell_entries;
  A.nbr_ptr = P->nbr_ptr; A.slice_ptr = P->slice_ptr; A.inc_key = P->inc_key; A.inc_meta = P->inc_meta;
  A.dphi1 = P->dphi1; A.dphi2 = P->dphi2; A.weight = P->weight;
  A.geom_rec = P->geom_rec; A.geom_rs = P->geom_rs;
  elastic_coeffs(A.dev2, A.vol);
  // tuning key assemble_canon: 0 auto = regular-triangulation fast path with 256-bit row stores (launch_assemble_tma drops to
  // the 16-byte stores of the generic path when K is not 32-byte aligned), 2 = fast path off
  A.canon = g_fem_tuning.assemble_canon == 2 ? 0 : 1;
}

extern "C" int fem_assemble_elastic(const fem_plan* P, const double* shear, const double* bulk, double* K_vals,
                                    fem_stream stream) {
  FEM_REQUIRE(P && shear && bulk && K_vals, "null pointer");
  FEM_REQUIRE((reinterpret_cast<uintptr_t>(K_vals) & 15u) == 0, "K_vals must be 16-byte aligned");
  AsmArgs A;
  fill_args(P, A);
  A.shear = shear; A.bulk = bulk; A.K_vals = K_vals;
  return launch_assemble<MODE_ELASTIC, false>(P, A, (cudaStream_t)stream);
}

extern "C" int fem_assemble_tangent(const fem_plan* P, const double* DS, double* K_vals, fem_stream stream) {
  FEM_REQUIRE(P && DS && K_vals, "null pointer");
  FEM_REQUIRE((reinterpret_cast<uintptr_t>(K_vals) & 15u) == 0, "K_vals must be 16-byte aligned");
  AsmArgs A;
  fill_args(P, A);
  A.DS = DS; A.K_vals = K_vals;
  return launch_assemble<MODE_TANGENT, false>(P, A, (cudaStream_t)stream);
}

extern "C" int fem_assemble_tangent_ref(const fem_plan* P, const double* DS, const double* shear, const double* bulk,
                                        const double* K_elast_vals, double* K_vals, fem_stream stream) {
  FEM_REQUIRE(P && DS && shear && bulk && K_elast_vals && K_vals, "null pointer");
  FEM_REQUIRE(((reinterpret_cast<uintptr_t>(K_vals) | reinterpret_cast<uintptr_t>(K_elast_vals)) & 15u) == 0, "K_vals and K_elast_vals must be 16-byte aligned");
  AsmArgs A;
  fill_args(P, A);
  A.DS = DS; A.shear = shear; A.bulk = bulk; A.Kel = K_elast_vals; A.K_vals = K_vals;
  return launch_assemble<MODE_TANGENT_REF, false>(P, A, (cudaStream_t)stream);
}

extern "C" int fem_assemble_tangent_force(const fem_plan* P, const double* DS, const double* S, double* K_vals, double* F,
                                          fem_stream stream) {
  FEM_REQUIRE(P && DS && S && K_vals && F, "null pointer");
  FEM_REQUIRE(((reinterpret_cast<uintptr_t>(F) | reinterpret_cast<uintptr_t>(K_vals)) & 15u) == 0, "F and K_vals must be 16-byte aligned");
  AsmArgs A;
  fill_args(P, A);
  A.DS = DS; A.S = S; A.K_vals = K_vals; A.F = F;
  return launch_assemble<MODE_TANGENT, true>(P, A, (cudaStream_t)stream);
}

extern "C" int fem_internal_force(const fem_plan* P, const double* S, double* F, fem_stream stream) {
  FEM_REQUIRE(P && S && F, "null pointer");
  FEM_REQUIRE((reinterpret_cast<uintptr_t>(F) & 15u) == 0, "F must be 16-byte aligned");
  AsmArgs A;
  fill_args(P, A);
  A.S = S; A.F = F;
  return launch_assemble<MODE_FORCE_ONLY, true>(P, A, (cudaStream_t)stream);
}

// ------------------------------------------------------------------------------------------------
// K4 strain: E = B u, one thread per integration point.  csr_matvec adds the stored entries of a row
// in ascending column order, i.e. ascending node id, x-dof before y-dof (:1043).
// ------------------------------------------------------------------------------------------------
template <int NP, int NQ>
__global__ void __launch_bounds__(256) strain_kernel(int64_t n_e, const int32_t* __restrict__ elem,
                                                     const double* __restrict__ dphi1, const double* __restrict__ dphi2,
                                                     const double* __restrict__ u, double* __restrict__ E) {
  const int64_t n_int = n_e * NQ;
  for (int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; g < n_int; g += (int64_t)gridDim.x * blockDim.x) {
    const int64_t e = g / NQ;
    int32_t nd[NP];
    int pp[NP];
#pragma unroll
    for (int p = 0; p < NP; ++p) {
      nd[p] = elem[(int64_t)p * n_e + e];
      pp[p] = p;
    }
#pragma unroll
    for (int i = 1; i < NP; ++i)  // insertion sort by node id (fully unrolled -> registers)
#pragma unroll
      for (int j = i; j > 0; --j)
        if (nd[j - 1] > nd[j]) {
          const int32_t tn = nd[j]; nd[j] = nd[j - 1]; nd[j - 1] = tn;
          const int tp = pp[j]; pp[j] = pp[j - 1]; pp[j - 1] = tp;
        }
    double e0 = 0.0, e1 = 0.0, e2 = 0.0;
#pragma unroll
    for (int s = 0; s < NP; ++s) {
      const double2 uv = reinterpret_cast<const double2*>(u)[nd[s]];
      const double a1 = dphi1[(int64_t)pp[s] * n_int + g], a2 = dphi2[(int64_t)pp[s] * n_int + g];
      e0 = e0 + a1 * uv.x;
      e1 = e1 + a2 * uv.y;
      e2 = (e2 + a2 * uv.x) + a1 * uv.y;
    }
    __stcs(E + g, e0);
    __stcs(E + n_int + g, e1);
    __stcs(E + 2 * n_int + g, e2);
  }
}

extern "C" int fem_strain(const fem_plan* P, const double* u, double* E, fem_stream stream) {
  FEM_REQUIRE(P && u && E, "null pointer");
  FEM_REQUIRE((reinterpret_cast<uintptr_t>(u) & 15u) == 0, "u must be 16-byte aligned");
  const int threads = 256;
  int64_t b = (P->n_int + threads - 1) / threads;
  if (b > (int64_t)P->sm_count * 2048) b = (int64_t)P->sm_count * 2048;
  const unsigned blocks = (unsigned)b;
  cudaStream_t st = (cudaStream_t)stream;
#define STRAIN(NP, NQ) strain_kernel<NP, NQ><<<blocks, threads, 0, st>>>(P->n_e, P->elem, P->dphi1, P->dphi2, u, E)
  if (P->n_p == 3 && P->n_q == 1) STRAIN(3, 1);
  else if (P->n_p == 6 && P->n_q == 7) STRAIN(6, 7);
  else if (P->n_p == 4 && P->n_q == 4) STRAIN(4, 4);
  else if (P->n_p == 8 && P->n_q == 9) STRAIN(8, 9);
  else {
    fem_set_error("unsupported element n_p=%d n_q=%d", P->n_p, P->n_q);
    return FEM_ERR_UNSUPPORTED;
  }
#undef STRAIN
  FEM_CUDA_CHECK(cudaGetLastError());
  return FEM_OK;
}

// transform(): one thread per node walks its incidence list (Plasticity2D_DP/pythonFEM.py:760-816)
__global__ void transform_kernel(int64_t n_n, int64_t n_slices, int n_q, const int64_t* __restrict__ slice_ptr,
                                 const uint32_t* __restrict__ inc_key, const double* __restrict__ weight,
                                 const double* __restrict__ q_int, double* __restrict__ q_node) {
  const int64_t a = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t slice = a >> 5;
  if (slice >= n_slices) return;
  const int lane = (int)(a & 31);
  const int64_t sbase = slice_ptr[slice];
  const int width = (int)((slice_ptr[slice + 1] - sbase) >> 5);
  double num = 0.0, den = 0.0;
  for (int i = 0; i < width; ++i) {
    const uint32_t key = inc_key[sbase + (int64_t)i * 32 + lane];
    if (key == FEM_INVALID_KEY) continue;
    const int64_t e = key >> 3;
    for (int q = 0; q < n_q; ++q) {
      const double w = weight[e * n_q + q];
      num = num + w * q_int[e * n_q + q];
      den = den + w;
    }
  }
  if (a < n_n) q_node[a] = num / den;
}

extern "C" int fem_transform(const fem_plan* P, const double* q_int, double* q_node, fem_stream stream) {
  FEM_REQUIRE(P && q_int && q_node, "null pointer");
  const int threads = 128;
  transform_kernel<<<(unsigned)fem_div_up(P->n_slices * 32, threads), threads, 0, (cudaStream_t)stream>>>(
      P->n_n, P->n_slices, P->n_q, P->slice_ptr, P->inc_key, P->weight, q_int, q_node);
  FEM_CUDA_CHECK(cudaGetLastError());
  return FEM_OK;
}

// ---- load vectors of the linear-elastic demo (Elasticity2D/pythonFEM.py:246-364) ---------------------------------------
// Volume forces: f_V[c, n] = sum over the integration points g = e*n_q + q of the elements around node n (ascending g) of
// hatp[la, q] * (weight[g] * f[c, g]) - the order in which SciPy sums the reference's COO triplets (:281-290), so the
// result is bit-identical.  Same walk of the node's incidence list as transform_kernel; no atomics.
struct HatTable { double h[FEM_MAX_NP * FEM_MAX_NQ]; };  // (n_p, n_q) row-major
__global__ void vector_volume_kernel(int64_t n_n, int64_t n_slices, int n_q, int64_t n_int, const int64_t* __restrict__ slice_ptr,
                                     const uint32_t* __restrict__ inc_key, const double* __restrict__ weight, const HatTable hat,
                                     const double* __restrict__ f_int, double* __restrict__ out) {
  const int64_t a = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t slice = a >> 5;
  if (slice >= n_slices) return;
  const int lane = (int)(a & 31);
  const int64_t sbase = slice_ptr[slice];
  const int width = (int)((slice_ptr[slice + 1] - sbase) >> 5);
  double f0 = 0.0, f1 = 0.0;
  for (int i = 0; i < width; ++i) {
    const uint32_t key = inc_key[sbase + (int64_t)i * 32 + lane];
    if (key == FEM_INVALID_KEY) continue;
    const int64_t e = key >> 3;
    const int la = (int)(key & 7u);
    for (int q = 0; q < n_q; ++q) {
      const int64_t g = e * n_q + q;
      const double w = weight[g], hp = hat.h[la * n_q + q];
      f0 = f0 + hp * (w * f_int[g]);
      f1 = f1 + hp * (w * f_int[n_int + g]);
    }
  }
  if (a < n_n) {
    out[a] = f0;
    out[n_n + a] = f1;
  }
}

extern "C" int fem_vector_volume(const fem_plan* P, const double* f_int, const double* h_hatp, double* out, fem_stream stream) {
  FEM_REQUIRE(P && f_int && h_hatp && out, "null pointer");
  HatTable hat;
  memset(&hat, 0, sizeof(hat));
  for (int i = 0; i < P->n_p * P->n_q; ++i) hat.h[i] = h_hatp[i];
  const int threads = 128;
  vector_volume_kernel<<<(unsigned)fem_div_up(P->n_slices * 32, threads), threads, 0, (cudaStream_t)stream>>>(
      P->n_n, P->n_slices, P->n_q, P->n_int, P->slice_ptr, P->inc_key, P->weight, hat, f_int, out);
  FEM_CUDA_CHECK(cudaGetLastError());
  return FEM_OK;
}

// out[s] = ((0 + v[ptr[s]]) + v[ptr[s]+1]) + ... : the sequential sum of every segment, one thread per segment.  With the
// contributions stably sorted by target node this is SciPy's duplicate summation of COO triplets in input order
// (surface tractions, :327-362: the boundary mesh has no incidence lists in the plan).
__global__ void segment_sum_ordered_kernel(int64_t n_seg, const int64_t* __restrict__ ptr, const double* __restrict__ v, double* __restrict__ out) {
  for (int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; s < n_seg; s += (int64_t)gridDim.x * blockDim.x) {
    double acc = 0.0;
    for (int64_t i = ptr[s]; i < ptr[s + 1]; ++i) acc = acc + v[i];
    out[s] = acc;
  }
}

extern "C" int fem_segment_sum_ordered(int64_t n_seg, const int64_t* seg_ptr, const double* vals, double* out, fem_stream stream) {
  FEM_REQUIRE(seg_ptr && out && n_seg >= 0, "null pointer");
  if (n_seg == 0) return FEM_OK;
  segment_sum_ordered_kernel<<<(unsigned)fem_div_up(n_seg, 256), 256, 0, (cudaStream_t)stream>>>(n_seg, seg_ptr, vals, out);
  FEM_CUDA_CHECK(cudaGetLastError());
  return FEM_OK;
}

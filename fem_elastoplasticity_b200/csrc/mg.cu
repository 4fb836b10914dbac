// Geometric multigrid V-cycle preconditioner for the masked CG of the Newton step (include/fem_b200.h, "geometric
// multigrid").  The reference solves K_tangent[Q,Q] dU = -F[Q] with a dense LU (Plasticity2D_DP/pythonFEM.py:1062-1066);
// point-Jacobi CG needs 57 500 iterations on the 16M-element footing mesh and the two-level method 1 900; a V-cycle with
// Chebyshev-Jacobi smoothing needs ~30-50, independent of the mesh size.
//
// Level 0 = the mesh (block-CSR matrix of the plan, SpMV of spmv.cuh with the smoother's vector updates fused into its
// epilogue: one pass over the matrix per Chebyshev step).  Levels >= 1 = lattices of bilinear cells, 9-point stencils of
// 2x2 blocks in structure-of-arrays planes (coalesced: one thread per node).  Restriction and prolongation are gathers
// through the lattice (no atomics, bit-reproducible).  Everything is HBM-bound FP64 streaming; no tensor cores.
#include "common.cuh"
#include "spmv.cuh"
#include "spmv_stream.cuh"
#include "peer.cuh"

struct fem_peer_table {
  void* p[FEM_MG_MAX_PEERS];
};

namespace {

struct Geom {  // local part of one structured level
  int nxn, nrows, g0, nrows_global;
  int64_t n;
};
static Geom geom_of(const fem_mg_level& L) { return Geom{L.nxn, L.nrows, L.g0, L.nrows_global, (int64_t)L.nxn * L.nrows}; }

__device__ __forceinline__ double w1(int o) { return o ? 0.5 : 1.0; }

// ---- lattice of level 0 ----------------------------------------------------------------------------------------------
__global__ void mg_lattice_kernel(int64_t n_n, const double* __restrict__ coord, double x0, double y0, double ihx, double ihy, int LX,
                                  int lat_rows, int g0, int32_t* lat, int32_t* __restrict__ node_lat, int32_t* err) {
  for (int64_t a = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; a < n_n; a += (int64_t)gridDim.x * blockDim.x) {
    const double fx = (coord[a] - x0) * ihx, fy = (coord[n_n + a] - y0) * ihy;
    const long long ix = llrint(fx), iy = llrint(fy) - g0;
    if (fabs(fx - (double)ix) > 1e-6 || fabs(fy - (double)(iy + g0)) > 1e-6 || ix < 0 || ix >= LX || iy < 0 || iy >= lat_rows) {
      atomicOr(err, 1);  // node off the lattice
      node_lat[a] = 0;
      continue;
    }
    const int32_t li = (int32_t)(iy * LX + ix);
    node_lat[a] = li;
    if (atomicCAS(lat + li, -1, (int32_t)a) != -1) atomicOr(err, 2);  // two nodes on one lattice point
  }
}

// parents of lattice point (ix, jg) on the next level: ids along x, global rows along y, weights
__device__ __forceinline__ void parents(int ix, int jg, int (&I)[2], int (&J)[2], double (&wx)[2], double (&wy)[2]) {
  I[0] = ix >> 1;
  I[1] = I[0] + (ix & 1);
  wx[0] = (ix & 1) ? 0.5 : 1.0;
  wx[1] = (ix & 1) ? 0.5 : 0.0;
  J[0] = jg >> 1;
  J[1] = J[0] + (jg & 1);
  wy[0] = (jg & 1) ? 0.5 : 1.0;
  wy[1] = (jg & 1) ? 0.5 : 0.0;
}

// ---- A_1 = P^T K P from the block-CSR matrix: one thread per level-1 node gathers its nine 2x2 blocks from the matrix rows of
// the <= 9 fine nodes it interpolates to (weights 1, 1/2, 1/4), rows in row_mask x columns in col_mask, in a fixed order: no
// atomics, so the hierarchy - and with it every multigrid solve - is reproducible bit for bit (a scatter with FP64 atomics
// was not).  A fine row is read by up to four coarse nodes; set-up only. ----
__global__ void __launch_bounds__(128) mg_galerkin_fine_kernel(const int32_t* __restrict__ nbr_ptr, const int32_t* __restrict__ nbr_idx,
                                                               const double* __restrict__ vals, const uint8_t* __restrict__ rmask,
                                                               const uint8_t* __restrict__ cmask, const int32_t* __restrict__ lat, int lat_rows,
                                                               const int32_t* __restrict__ node_lat, int LX, int g0, Geom c, double* __restrict__ S,
                                                               int32_t* err) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= c.n) return;
  const int I = (int)(t % c.nxn), Jg = (int)(t / c.nxn) + c.g0;
  double acc[9][4];
#pragma unroll
  for (int s = 0; s < 9; ++s) acc[s][0] = acc[s][1] = acc[s][2] = acc[s][3] = 0.0;
  for (int oy = -1; oy <= 1; ++oy)
    for (int ox = -1; ox <= 1; ++ox) {
      const int ix = 2 * I + ox, jl = 2 * Jg + oy - g0;  // fine lattice point: column, local row
      if (ix < 0 || ix >= LX || jl < 0 || jl >= lat_rows) continue;
      const int a = lat[(int64_t)jl * LX + ix];
      if (a < 0) continue;
      const double mi0 = rmask ? (double)(rmask[2 * (int64_t)a] != 0) : 1.0, mi1 = rmask ? (double)(rmask[2 * (int64_t)a + 1] != 0) : 1.0;
      if (mi0 == 0.0 && mi1 == 0.0) continue;
      const double wa = (ox ? 0.5 : 1.0) * (oy ? 0.5 : 1.0);
      const int p0 = nbr_ptr[a], deg = nbr_ptr[a + 1] - p0;
      const double* row0 = vals + 4 * (int64_t)p0;
      const double* row1 = row0 + 2 * deg;
      for (int j = 0; j < deg; ++j) {
        const int b = nbr_idx[p0 + j];
        const int lb = node_lat[b];
        int Ib[2], Jb[2];
        double wxb[2], wyb[2];
        parents(lb % LX, lb / LX + g0, Ib, Jb, wxb, wyb);
        const double mj0 = cmask ? (double)(cmask[2 * (int64_t)b] != 0) : 1.0, mj1 = cmask ? (double)(cmask[2 * (int64_t)b + 1] != 0) : 1.0;
        const double k[4] = {row0[2 * j] * mi0 * mj0, row0[2 * j + 1] * mi0 * mj1, row1[2 * j] * mi1 * mj0, row1[2 * j + 1] * mi1 * mj1};
        if (k[0] == 0.0 && k[1] == 0.0 && k[2] == 0.0 && k[3] == 0.0) continue;
        for (int yb = 0; yb < 2; ++yb)
          for (int xb = 0; xb < 2; ++xb) {
            const double w = wa * wxb[xb] * wyb[yb];
            if (w == 0.0) continue;
            const int dx = Ib[xb] - I, dy = Jb[yb] - Jg;
            if (dx < -1 || dx > 1 || dy < -1 || dy > 1) { atomicOr(err, 8); continue; }  // mesh edge longer than one lattice step
            const int s = (dy + 1) * 3 + dx + 1;
#pragma unroll
            for (int q = 0; q < 4; ++q) acc[s][q] += w * k[q];
          }
      }
    }
  for (int s = 0; s < 9; ++s)
#pragma unroll
    for (int q = 0; q < 4; ++q) S[(int64_t)(4 * s + q) * c.n + t] = acc[s][q];
}

// ---- A_{l+1} = P^T A_l P between structured levels: one thread per coarse node gathers its 9 blocks (fully unrolled: the
// interpolation weights and the target slot of every (fine point, fine neighbour) pair are compile-time constants) ----
__global__ void __launch_bounds__(128) mg_galerkin_stencil_kernel(Geom f, const double* __restrict__ Sf, Geom c, int row_lo, int row_hi,
                                                                  double* __restrict__ Sc) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (int64_t)(row_hi - row_lo) * c.nxn) return;
  const int I = (int)(t % c.nxn), J = row_lo + (int)(t / c.nxn);
  const int Jg = J + c.g0;
  double acc[9][4];
#pragma unroll
  for (int s = 0; s < 9; ++s)
#pragma unroll
    for (int q = 0; q < 4; ++q) acc[s][q] = 0.0;
#pragma unroll
  for (int db = -1; db <= 1; ++db)
#pragma unroll
    for (int da = -1; da <= 1; ++da) {
      const int fi = 2 * I + da, fjg = 2 * Jg + db, fj = fjg - f.g0;
      const bool va = fi >= 0 && fi < f.nxn && fjg >= 0 && fjg < f.nrows_global && fj >= 0 && fj < f.nrows;
      if (!va) continue;
      const int64_t fn = fi + (int64_t)fj * f.nxn;
      const double wa = w1(da) * w1(db);
#pragma unroll
      for (int ey = -1; ey <= 1; ++ey)
#pragma unroll
        for (int ex = -1; ex <= 1; ++ex) {
          const int s = (ey + 1) * 3 + ex + 1;
          double k[4];
#pragma unroll
          for (int q = 0; q < 4; ++q) k[q] = wa * Sf[(int64_t)(4 * s + q) * f.n + fn];
#pragma unroll
          for (int DY = -1; DY <= 1; ++DY)
#pragma unroll
            for (int DX = -1; DX <= 1; ++DX) {
              const int ox = da + ex - 2 * DX, oy = db + ey - 2 * DY;  // neighbour relative to coarse node I + D, in fine steps
              if (ox < -1 || ox > 1 || oy < -1 || oy > 1) continue;
              const double wb = w1(ox) * w1(oy);
#pragma unroll
              for (int q = 0; q < 4; ++q) acc[(DY + 1) * 3 + DX + 1][q] = fma(wb, k[q], acc[(DY + 1) * 3 + DX + 1][q]);
            }
        }
    }
  const int64_t cn = I + (int64_t)J * c.nxn;
#pragma unroll
  for (int s = 0; s < 9; ++s)
#pragma unroll
    for (int q = 0; q < 4; ++q) Sc[(int64_t)(4 * s + q) * c.n + cn] = acc[s][q];
}

// The smoother's D is the 2x2 diagonal block of a node (both displacement components): block Jacobi.  On this
// near-incompressible operator (nu = 0.48) it needs ~17 % fewer CG iterations than point Jacobi at the same cost per
// sweep.  Inverse of the symmetric block [k00 k01; k01 k11]; a component that is not an unknown (masked / dead) is
// decoupled and gets a zero row and column.  Stored as two planes of double2: A[node] = (i00, i01), B[node] = (i01, i11).
__device__ __forceinline__ void block_inverse(double k00, double k01, double k11, bool f0, bool f1, double2& ia, double2& ib) {
  ia = make_double2(0.0, 0.0);
  ib = make_double2(0.0, 0.0);
  if (f0 && f1) {
    const double det = k00 * k11 - k01 * k01;
    if (det > 0.0 && k00 > 0.0) {
      ia = make_double2(k11 / det, -k01 / det);
      ib = make_double2(-k01 / det, k00 / det);
      return;
    }
  }
  if (f0 && k00 != 0.0) ia.x = 1.0 / k00;
  if (f1 && k11 != 0.0) ib.y = 1.0 / k11;
}

// coarse DOFs without free fine support get a unit diagonal; dinv = inverse of the node's 2x2 diagonal block
__global__ void mg_level_finalize_kernel(int64_t n, double* S, double thresh, double2* __restrict__ dinv) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    double d0 = S[(int64_t)16 * n + i], d1 = S[(int64_t)19 * n + i];
    double off = 0.5 * (S[(int64_t)17 * n + i] + S[(int64_t)18 * n + i]);
    if (!(d0 > thresh)) {
      d0 = 1.0;
      off = 0.0;
      S[(int64_t)16 * n + i] = 1.0;
    }
    if (!(d1 > thresh)) {
      d1 = 1.0;
      off = 0.0;
      S[(int64_t)19 * n + i] = 1.0;
    }
    double2 ia, ib;
    block_inverse(d0, off, d1, true, true, ia, ib);
    dinv[i] = ia;
    dinv[n + i] = ib;
  }
}

// level 0: inverse 2x2 diagonal blocks of the block-CSR matrix, masked
__global__ void mg_block_jacobi_kernel(int64_t n_n, const int32_t* __restrict__ nbr_ptr, const int32_t* __restrict__ nbr_idx,
                                       const double* __restrict__ vals, const uint8_t* __restrict__ mask, double2* __restrict__ dinv) {
  for (int64_t a = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; a < n_n; a += (int64_t)gridDim.x * blockDim.x) {
    const int p0 = nbr_ptr[a], deg = nbr_ptr[a + 1] - p0;
    double k00 = 0.0, k01 = 0.0, k10 = 0.0, k11 = 0.0;
    for (int j = 0; j < deg; ++j)
      if (nbr_idx[p0 + j] == a) {
        k00 = vals[4 * (int64_t)p0 + 2 * j];
        k01 = vals[4 * (int64_t)p0 + 2 * j + 1];
        k10 = vals[4 * (int64_t)p0 + 2 * deg + 2 * j];
        k11 = vals[4 * (int64_t)p0 + 2 * deg + 2 * j + 1];
        break;
      }
    const bool f0 = mask ? mask[2 * a] != 0 : true, f1 = mask ? mask[2 * a + 1] != 0 : true;
    double2 ia, ib;
    block_inverse(k00, 0.5 * (k01 + k10), k11, f0, f1, ia, ib);
    dinv[a] = ia;
    dinv[n_n + a] = ib;
  }
}

__global__ void mg_stencil_to_dense_kernel(Geom g, const double* __restrict__ S, double* __restrict__ A) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= g.n * 9) return;
  const int64_t node = t / 9;
  const int s = (int)(t % 9);
  const int i = (int)(node % g.nxn), j = (int)(node / g.nxn);
  const int ii = i + s % 3 - 1, jj = j + s / 3 - 1;
  if (ii < 0 || ii >= g.nxn || jj < 0 || jj >= g.nrows) return;
  const int64_t nb = ii + (int64_t)jj * g.nxn, nc = 2 * g.n;
#pragma unroll
  for (int q = 0; q < 4; ++q) A[(2 * node + (q >> 1)) * nc + 2 * nb + (q & 1)] = S[(int64_t)(4 * s + q) * g.n + node];
}

// ---- smoother / residual on a structured level ------------------------------------------------------------------------
enum { MG_APPLY = 0, MG_RESID = 1, MG_CHEB = 2, MG_FIRST = 3 };

// SYM: the level operators are symmetric (Galerkin products of a symmetric matrix), so the block towards the neighbour in
// direction -k is the transpose of that neighbour's block in direction +k.  The sweep then streams only the upper half of
// the stencil from HBM - the self block (3 planes: its two off-diagonal entries are equal) and the directions E, NW, N, NE
// (16 planes): 19 planes = 76 B per node with the FP32 copy instead of 36 planes = 144 B - and takes W, SW, S, SE from the
// planes of the west neighbour (same warp: L1) and of the row below (read by the CTAs just before: L2).
template <int MODE, class ST, bool SYM>
__global__ void __launch_bounds__(256) mg_stencil_kernel(Geom g, int row_lo, int row_hi, const ST* __restrict__ S, const double2* x,
                                                         const double2* __restrict__ b, const double2* __restrict__ dinv, double2* d,
                                                         double2* out, double c1, double c2) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (int64_t)(row_hi - row_lo) * g.nxn) return;
  const int64_t node = (int64_t)row_lo * g.nxn + t;
  if (MODE == MG_FIRST) {  // x = 0: d = c2 D^-1 b, x = d
    const double2 bi = b[node], da = dinv[node], db = dinv[g.n + node];
    const double2 dn = make_double2(c2 * (da.x * bi.x + da.y * bi.y), c2 * (db.x * bi.x + db.y * bi.y));
    d[node] = dn;
    out[node] = dn;
    return;
  }
  const int i = (int)(node % g.nxn), j = (int)(node / g.nxn);
  double y0 = 0.0, y1 = 0.0;
#pragma unroll
  for (int s = 0; s < 9; ++s) {
    const int dx = s % 3 - 1, dy = s / 3 - 1;
    const bool v = (i + dx >= 0) && (i + dx < g.nxn) && (j + dy >= 0) && (j + dy < g.nrows);
    const double2 xv = v ? x[node + dy * g.nxn + dx] : make_double2(0.0, 0.0);
    if (SYM && s < 4) {  // block (node -> node + off) = transpose of the block (node + off -> node) stored with the neighbour
      const ST* sp = S + (int64_t)(4 * (8 - s)) * g.n + (v ? node + dy * g.nxn + dx : node);
      y0 = fma((double)__ldg(sp), xv.x, y0);
      y0 = fma((double)__ldg(sp + 2 * g.n), xv.y, y0);
      y1 = fma((double)__ldg(sp + g.n), xv.x, y1);
      y1 = fma((double)__ldg(sp + 3 * g.n), xv.y, y1);
    } else if (SYM) {    // own upper half: ordinary cached loads - the neighbours read these planes again
      const ST* sp = S + (int64_t)(4 * s) * g.n + node;
      const double s01 = (double)__ldg(sp + g.n);
      y0 = fma((double)__ldg(sp), xv.x, y0);
      y0 = fma(s01, xv.y, y0);
      y1 = fma(s == 4 ? s01 : (double)__ldg(sp + 2 * g.n), xv.x, y1);
      y1 = fma((double)__ldg(sp + 3 * g.n), xv.y, y1);
    } else {
      const ST* sp = S + (int64_t)(4 * s) * g.n + node;
      y0 = fma((double)__ldcs(sp), xv.x, y0);
      y0 = fma((double)__ldcs(sp + g.n), xv.y, y0);
      y1 = fma((double)__ldcs(sp + 2 * g.n), xv.x, y1);
      y1 = fma((double)__ldcs(sp + 3 * g.n), xv.y, y1);
    }
  }
  if (MODE == MG_APPLY) {
    out[node] = make_double2(y0, y1);
    return;
  }
  const double2 bi = b[node];
  const double r0 = bi.x - y0, r1 = bi.y - y1;
  if (MODE == MG_RESID) {
    out[node] = make_double2(r0, r1);
    return;
  }
  const double2 da = dinv[node], db = dinv[g.n + node];
  double2 dn = make_double2(c2 * (da.x * r0 + da.y * r1), c2 * (db.x * r0 + db.y * r1));
  if (c1 != 0.0) {
    const double2 dd = d[node];
    dn.x = fma(c1, dd.x, dn.x);
    dn.y = fma(c1, dd.y, dn.y);
  }
  d[node] = dn;
  const double2 xi = x[node];
  out[node] = make_double2(xi.x + dn.x, xi.y + dn.y);
}

// ---- level 0: the same steps fused into the epilogue of the block-CSR SpMV --------------------------------------------
template <int MODE>
struct MgFineEpilogue {
  const double2* __restrict__ b;
  const double2* __restrict__ dinv;
  double2* d;
  const double2* x;
  double2* out;
  const uint8_t* __restrict__ mask;
  double c1, c2;
  bool want_dot;
  int64_t own_lo, own_hi;  // ghost nodes are never written: their owners store them (fem_mg_exchange)
  int group;               // lanes per node (>= 4)
  int64_t n_n;             // plane stride of dinv
  // operands of the update, one per lane of the node's group, requested together with the matrix values
  __device__ __forceinline__ double2 prefetch(const int64_t a, const int sub) const {
    if (a >= own_lo && a < own_hi) {
      if (sub == 0) return b[a];
      if (MODE != MG_RESID) {
        if (sub == 1) return dinv[a];
        if (sub == 2 && c1 != 0.0) return d[a];
        if (sub == 3) return x[a];
      }
    }
    return make_double2(0.0, 0.0);
  }
  __device__ __forceinline__ void operator()(const int64_t a, const bool lead, const double acc0, const double acc1, double& dot, const double2 pf) const {
    const int base = (threadIdx.x & 31) & ~(group - 1);
    double2 di = make_double2(0.0, 0.0), dd = di, xi = di;
    if (MODE != MG_RESID) {  // executed by every lane of the warp: the lead lane collects its neighbours' operands
      di.x = __shfl_sync(0xffffffffu, pf.x, base + 1);
      di.y = __shfl_sync(0xffffffffu, pf.y, base + 1);
      dd.x = __shfl_sync(0xffffffffu, pf.x, base + 2);
      dd.y = __shfl_sync(0xffffffffu, pf.y, base + 2);
      xi.x = __shfl_sync(0xffffffffu, pf.x, base + 3);
      xi.y = __shfl_sync(0xffffffffu, pf.y, base + 3);
    }
    if (!lead || a < own_lo || a >= own_hi) return;
    const double2 bi = pf;
    double r0 = bi.x - acc0, r1 = bi.y - acc1;
    if (MODE == MG_RESID) {
      if (mask) {
        const uchar2 mk = reinterpret_cast<const uchar2*>(mask)[a];
        if (!mk.x) r0 = 0.0;
        if (!mk.y) r1 = 0.0;
      }
      out[a] = make_double2(r0, r1);
      return;
    }
    // D^-1 has zero rows and columns on masked DOFs: d and x stay zero there
    const double2 db = dinv[n_n + a];
    double2 dn = make_double2(c2 * (di.x * r0 + di.y * r1), c2 * (db.x * r0 + db.y * r1));
    dn.x = fma(c1, dd.x, dn.x);  // dd == 0 when c1 == 0 (first step of a sweep)
    dn.y = fma(c1, dd.y, dn.y);
    d[a] = dn;
    const double2 xo = make_double2(xi.x + dn.x, xi.y + dn.y);
    out[a] = xo;
    if (want_dot) dot = fma(bi.x, xo.x, fma(bi.y, xo.y, dot));
  }
};

template <int GROUP, int MODE, class VT>
__global__ void __launch_bounds__(FEM_SPMV_THREADS) mg_fine_tiles_kernel(int64_t n_n, int64_t n_tiles, const int32_t* __restrict__ nbr_ptr,
                                                                         const int32_t* __restrict__ nbr_idx, const uint16_t* __restrict__ nbr_loc,
                                                                         const int32_t* __restrict__ tile_seg, const VT* __restrict__ vals,
                                                                         const double* x, const MgFineEpilogue<MODE> epi, double* dot_out, const FemRedBuf rb) {
  __shared__ double red[32];
  __shared__ SpmvTileSmem sm;
  double dot = spmv_tiles_epi<GROUP, false, MgFineEpilogue<MODE>, VT>(n_n, n_tiles, nbr_ptr, nbr_idx, nbr_loc, tile_seg, vals, x, epi, sm);
  if (dot_out) {
    const double v[1] = {block_sum(dot, red)};
    double* const dst[1] = {dot_out};
    ordered_accumulate<1>(v, dst, rb);
  }
}

template <int GROUP, int MODE, class VT>
__global__ void __launch_bounds__(256) mg_fine_rows_kernel(int64_t n_n, const int32_t* __restrict__ nbr_ptr, const int32_t* __restrict__ nbr_idx,
                                                           const VT* __restrict__ vals, const double* __restrict__ x,
                                                           const MgFineEpilogue<MODE> epi, double* dot_out, const FemRedBuf rb) {
  __shared__ double red[32];
  double dot = spmv_rows_epi<GROUP, 2, MgFineEpilogue<MODE>, VT>(n_n, nbr_ptr, nbr_idx, vals, x, epi);
  if (dot_out) {
    const double v[1] = {block_sum(dot, red)};
    double* const dst[1] = {dot_out};
    ordered_accumulate<1>(v, dst, rb);
  }
}

// the same steps for the streaming SpMV (spmv_stream.cuh): b, D^-1, d, x of the tile's nodes arrive in shared memory with
// the matrix values; the lead lane of a node only computes and stores
template <int MODE>
struct MgStreamEpilogue {
  static constexpr int N_IN = MODE == MG_RESID ? 1 : 5;
  const double2* b;
  const double2* dinv;  // two planes of n_n double2: rows of the inverse 2x2 diagonal blocks
  double2* d;
  const double2* x;
  double2* out;
  const uint8_t* mask;
  double c1, c2;
  bool want_dot;
  int64_t own_lo, own_hi, n_n;
  __device__ __forceinline__ const double2* in(int k) const {
    return k == 0 ? b : (k == 1 ? dinv : (k == 2 ? dinv + n_n : (k == 3 ? d : x)));
  }
  __device__ __forceinline__ const uint8_t* mask_ptr() const { return MODE == MG_RESID ? mask : nullptr; }
  __device__ __forceinline__ void operator()(const int64_t a, const double acc0, const double acc1, const double2 (&s)[N_IN], const uchar2 mk,
                                             double& dot) const {
    if (a < own_lo || a >= own_hi) return;
    const double2 bi = s[0];
    double r0 = bi.x - acc0, r1 = bi.y - acc1;
    if (MODE == MG_RESID) {
      if (!mk.x) r0 = 0.0;
      if (!mk.y) r1 = 0.0;
      out[a] = make_double2(r0, r1);
      return;
    }
    const double2 da = s[N_IN > 1 ? 1 : 0], db = s[N_IN > 2 ? 2 : 0], dd = s[N_IN > 3 ? 3 : 0], xi = s[N_IN > 4 ? 4 : 0];
    double2 dn = make_double2(c2 * (da.x * r0 + da.y * r1), c2 * (db.x * r0 + db.y * r1));  // zero rows/columns on masked DOFs
    if (c1 != 0.0) {
      dn.x = fma(c1, dd.x, dn.x);
      dn.y = fma(c1, dd.y, dn.y);
    }
    d[a] = dn;
    const double2 xo = make_double2(xi.x + dn.x, xi.y + dn.y);
    out[a] = xo;
    if (want_dot) dot = fma(bi.x, xo.x, fma(bi.y, xo.y, dot));
  }
};

template <int GROUP, int MODE, class VT>
__global__ void __launch_bounds__(FEM_STREAM_THREADS, 1) mg_fine_stream_kernel(const SpmvStreamArgs A, const VT* __restrict__ vals, const double* x,
                                                                           const MgStreamEpilogue<MODE> epi, double* dot_out, const FemRedBuf rb) {
  extern __shared__ __align__(128) unsigned char stream_smem[];
  __shared__ double red[32];
  double dot = spmv_stream<GROUP, false, VT>(A, vals, x, epi, stream_smem);
  if (dot_out) {
    const double v[1] = {block_sum(dot, red)};
    double* const dst[1] = {dot_out};
    ordered_accumulate<1>(v, dst, rb);
  }
}

__global__ void __launch_bounds__(256) mg_fine_first_kernel(int64_t lo, int64_t hi, int64_t n_n, const double2* __restrict__ b,
                                                            const double2* __restrict__ dinv, double2* __restrict__ d, double2* __restrict__ out,
                                                            double c2) {
  for (int64_t i = lo + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < hi; i += (int64_t)gridDim.x * blockDim.x) {
    const double2 bi = b[i], da = dinv[i], db = dinv[n_n + i];
    const double2 dn = make_double2(c2 * (da.x * bi.x + da.y * bi.y), c2 * (db.x * bi.x + db.y * bi.y));
    d[i] = dn;
    out[i] = dn;
  }
}

// ---- transfers --------------------------------------------------------------------------------------------------------
// b_c = P^T r: coarse node (I, J) gathers the 3x3 fine points around lattice point (2I, 2J).  LAT: the fine level is level
// 0 (points -> nodes through the lattice map); otherwise the fine vector is indexed by the lattice itself.
template <bool LAT>
__global__ void __launch_bounds__(256) mg_restrict_kernel(Geom c, int row_lo, int row_hi, int nxf, int nrows_f, int g0f, int nrows_global_f,
                                                          const int32_t* __restrict__ lat, const double2* __restrict__ r, double2* __restrict__ bc) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (int64_t)(row_hi - row_lo) * c.nxn) return;
  const int I = (int)(t % c.nxn), J = row_lo + (int)(t / c.nxn), Jg = J + c.g0;
  double a0 = 0.0, a1 = 0.0;
#pragma unroll
  for (int db = -1; db <= 1; ++db) {
    const int fjg = 2 * Jg + db, fj = fjg - g0f;
    if (fjg < 0 || fjg >= nrows_global_f || fj < 0 || fj >= nrows_f) continue;
#pragma unroll
    for (int da = -1; da <= 1; ++da) {
      const int fi = 2 * I + da;
      if (fi < 0 || fi >= nxf) continue;
      int64_t fn = fi + (int64_t)fj * nxf;
      if (LAT) {
        fn = lat[fn];
        if (fn < 0) continue;
      }
      const double w = w1(da) * w1(db);
      const double2 v = r[fn];
      a0 = fma(w, v.x, a0);
      a1 = fma(w, v.y, a1);
    }
  }
  bc[I + (int64_t)J * c.nxn] = make_double2(a0, a1);
}

__device__ __forceinline__ double2 prolong_point(const Geom& c, int ix, int jg, const double2* xc) {
  int I[2], J[2];
  double wx[2], wy[2];
  parents(ix, jg, I, J, wx, wy);
  double2 z = make_double2(0.0, 0.0);
#pragma unroll
  for (int yy = 0; yy < 2; ++yy)
#pragma unroll
    for (int xx = 0; xx < 2; ++xx) {
      const double w = wx[xx] * wy[yy];
      if (w == 0.0) continue;
      const int jl = J[yy] - c.g0;
      if (jl < 0 || jl >= c.nrows || I[xx] >= c.nxn) continue;
      const double2 v = xc[I[xx] + (int64_t)jl * c.nxn];
      z.x = fma(w, v.x, z.x);
      z.y = fma(w, v.y, z.y);
    }
  return z;
}

// x_f += P x_c on the owned rows of a structured level
__global__ void __launch_bounds__(256) mg_prolong_kernel(Geom f, int row_lo, int row_hi, Geom c, const double2* xc, double2* __restrict__ xf) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (int64_t)(row_hi - row_lo) * f.nxn) return;
  const int64_t node = (int64_t)row_lo * f.nxn + t;
  const int i = (int)(node % f.nxn), j = (int)(node / f.nxn);
  const double2 z = prolong_point(c, i, j + f.g0, xc);
  double2 v = xf[node];
  v.x += z.x;
  v.y += z.y;
  xf[node] = v;
}

// level 0: every node of the mesh, masked (Dirichlet DOFs and rows of other ranks receive nothing)
__global__ void __launch_bounds__(256) mg_prolong_fine_kernel(int64_t n_n, const int32_t* __restrict__ node_lat, int LX, int g0,
                                                              const uint8_t* __restrict__ mask, Geom c, const double2* xc, double2* __restrict__ xf) {
  for (int64_t a = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; a < n_n; a += (int64_t)gridDim.x * blockDim.x) {
    uchar2 mk = make_uchar2(1, 1);
    if (mask) mk = reinterpret_cast<const uchar2*>(mask)[a];
    if (!mk.x && !mk.y) continue;
    const int la = node_lat[a];
    const double2 z = prolong_point(c, la % LX, la / LX + g0, xc);
    double2 v = xf[a];
    if (mk.x) v.x += z.x;
    if (mk.y) v.y += z.y;
    xf[a] = v;
  }
}

// ---- ghost rows over NVLink peer memory: push, release flags, wait for the neighbours' flags - one kernel -------------
__global__ void __launch_bounds__(256) mg_exchange_kernel(const fem_mg_exchange ex, const double2* __restrict__ v, uint64_t* err, uint64_t timeout_ns) {
  __shared__ int sh_last;
  int64_t total = 0;
  for (int k = 0; k < ex.n_send; ++k) total += ex.count[k];
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
    int64_t o = t;
    int k = 0;
    while (o >= ex.count[k]) o -= ex.count[k++];
    reinterpret_cast<double2*>(ex.dst[k])[o] = v[ex.src_off[k] + o];
  }
  __threadfence_system();
  if (arrive_last(ex.seq + 1, gridDim.x, &sh_last)) {
    const uint64_t seq = ex.seq[0] + 1;
    if (threadIdx.x < ex.n_send) st_release_sys(ex.dst_flag[threadIdx.x], seq);
    if (threadIdx.x >= 32 && threadIdx.x < 32 + ex.n_wait) wait_flag(ex.wait_flag[threadIdx.x - 32], seq, err, 0, timeout_ns);
    __syncthreads();
    if (threadIdx.x == 0) {
      ex.seq[0] = seq;
      *reinterpret_cast<unsigned*>(ex.seq + 1) = 0u;
    }
  }
}

// ---- sum of a few scalars over all ranks through peer memory (the CG's dot products): every rank stores its values as
// self-validating 16-byte lines into every rank's block, polls its own block for all ranks' lines and adds them in rank
// order (bit-identical result everywhere).  Lines are double-buffered by the parity of the sequence number: a rank can
// only be one all-reduce ahead of any other, since finishing one needs everybody's lines of that one. ----
__global__ void __launch_bounds__(256) peer_allreduce_kernel(double* vals, int n, uint64_t* local, const fem_peer_table peers, int64_t lines_off,
                                                             int64_t seq_off, int64_t err_off, int rank, int world, uint64_t timeout_ns) {
  __shared__ double sh[FEM_MG_MAX_PEERS][8];
  const uint32_t seq = (uint32_t)local[seq_off] + 1u;
  const int par = (int)(seq & 1u), t = threadIdx.x;
  if (t < world * n) {
    const int r = t / n, i = t % n;
    uint64_t* dst = reinterpret_cast<uint64_t*>(peers.p[r]) + lines_off + (int64_t)(((par * FEM_MG_MAX_PEERS + rank) * 8 + i) * 2);
    line_store(dst, vals[i], seq);
  }
  if (t < world * n) {
    const int r = t / n, i = t % n;
    sh[r][i] = line_wait(local + lines_off + (int64_t)(((par * FEM_MG_MAX_PEERS + r) * 8 + i) * 2), seq, local + err_off, 0, timeout_ns);
  }
  __syncthreads();
  if (t < n) {
    double acc = 0.0;
    for (int r = 0; r < world; ++r) acc += sh[r][t];
    vals[t] = acc;
  }
  if (t == 0) local[seq_off] = seq;
}

// ---- CG steps around the V-cycle --------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) mg_pcg_init_kernel(int64_t n, const double* __restrict__ rhs, const uint8_t* __restrict__ mask,
                                                          double* __restrict__ r, double* __restrict__ x, double* scal, const FemRedBuf rb) {
  __shared__ double red[32];
  double rr = 0.0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const double ri = (mask ? mask[i] != 0 : true) ? rhs[i] : 0.0;
    r[i] = ri;
    x[i] = 0.0;
    rr = fma(ri, ri, rr);
  }
  rr = block_sum(rr, red);
  const double v[2] = {rr, rr};
  double* const dst[2] = {scal + 1, scal + 4};
  ordered_accumulate<2>(v, dst, rb);
}

__global__ void __launch_bounds__(256) mg_pcg_update_xr_kernel(int64_t n2, const double2* __restrict__ p, const double2* __restrict__ q,
                                                               double2* __restrict__ x, double2* __restrict__ r, double* scal, int it, const FemRedBuf rb) {
  __shared__ double red[32];
  const double rz_old = scal[(it & 1) ? 2 : 0], pq = scal[3];
  const double alpha = (pq != 0.0) ? rz_old / pq : 0.0;
  double rr = 0.0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n2; i += (int64_t)gridDim.x * blockDim.x) {
    const double2 pi = p[i], qi = __ldcs(q + i);
    double2 xi = x[i], ri = r[i];
    xi.x = fma(alpha, pi.x, xi.x);
    xi.y = fma(alpha, pi.y, xi.y);
    ri.x = fma(-alpha, qi.x, ri.x);
    ri.y = fma(-alpha, qi.y, ri.y);
    x[i] = xi;
    r[i] = ri;
    rr = fma(ri.x, ri.x, fma(ri.y, ri.y, rr));
  }
  const double v[1] = {block_sum(rr, red)};
  double* const dst[1] = {scal + 1};
  ordered_accumulate<1>(v, dst, rb);
}

__global__ void __launch_bounds__(256) mg_pcg_update_p_kernel(int64_t n2, const double2* __restrict__ z, double2* __restrict__ p, double* scal, int it) {
  double beta = 0.0;
  if (it >= 0) {
    const double rz_old = scal[(it & 1) ? 2 : 0], rz_new = scal[(it & 1) ? 0 : 2];
    beta = (rz_old != 0.0) ? rz_new / rz_old : 0.0;
  }
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n2; i += (int64_t)gridDim.x * blockDim.x) {
    const double2 zi = z[i];
    double2 pi = make_double2(0.0, 0.0);
    if (it >= 0) pi = p[i];
    pi.x = fma(beta, pi.x, zi.x);
    pi.y = fma(beta, pi.y, zi.y);
    p[i] = pi;
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) scal[3] = 0.0;
}

__global__ void __launch_bounds__(256) mg_dense_gemv_kernel(int n, const double* __restrict__ A, const double* __restrict__ x, double* __restrict__ y) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= n) return;
  const double* row = A + (int64_t)warp * n;
  double acc = 0.0;
  for (int j = lane; j < n; j += 32) acc = fma(row[j], x[j], acc);
  acc = warp_sum(acc);
  if (lane == 0) y[warp] = acc;
}

unsigned grid_for(int64_t items, int threads = 256) { return (unsigned)((items + threads - 1) / threads < 1 ? 1 : (items + threads - 1) / threads); }
unsigned vgrid(int64_t items, int sms) {
  int64_t b = (items + 255) / 256;
  const int64_t cap = (int64_t)(sms > 0 ? sms : 148) * 8;
  if (b > cap) b = cap;
  return (unsigned)(b < 1 ? 1 : b);
}

int run_exchange(const fem_mg_exchange& ex, const double* v, uint64_t* err, cudaStream_t st) {
  if (ex.n_send == 0 && ex.n_wait == 0) return FEM_OK;
  FEM_REQUIRE(ex.seq != nullptr && err != nullptr && ex.n_send <= FEM_MG_MAX_PEERS && ex.n_wait <= FEM_MG_MAX_PEERS, "exchange descriptor");
  int64_t total = 0;
  for (int k = 0; k < ex.n_send; ++k) total += ex.count[k];
  unsigned blocks = grid_for(total);
  if (blocks > 64) blocks = 64;
  const uint64_t timeout_ns = (uint64_t)(g_fem_tuning.peer_timeout_ms > 0 ? g_fem_tuning.peer_timeout_ms : 10000) * 1000000ull;
  mg_exchange_kernel<<<blocks, 256, 0, st>>>(ex, reinterpret_cast<const double2*>(v), err, timeout_ns);
  FEM_CUDA_CHECK(cudaGetLastError());
  return FEM_OK;
}

template <int MODE>
int launch_stencil(const fem_mg_level& L, const double* x, double* out, double c1, double c2, cudaStream_t st) {
  const Geom g = geom_of(L);
  const int64_t items = (int64_t)(L.own_hi - L.own_lo) * L.nxn;
  if (items <= 0) return FEM_OK;
  const bool sym = g_fem_tuning.mg_stencil_sym != 2 && MODE != MG_FIRST;
#define MG_STENCIL(ST, SYMM, SPTR)                                                                                              \
  mg_stencil_kernel<MODE, ST, SYMM><<<grid_for(items), 256, 0, st>>>(g, L.own_lo, L.own_hi, SPTR, reinterpret_cast<const double2*>(x), \
                                                                     reinterpret_cast<const double2*>(L.b), reinterpret_cast<const double2*>(L.dinv), \
                                                                     reinterpret_cast<double2*>(L.d), reinterpret_cast<double2*>(out), c1, c2)
  if (L.S32 && MODE != MG_FIRST) {
    if (sym) MG_STENCIL(float, true, L.S32);
    else MG_STENCIL(float, false, L.S32);
  } else {
    if (sym) MG_STENCIL(double, true, L.S);
    else MG_STENCIL(double, false, L.S);
  }
#undef MG_STENCIL
  FEM_CUDA_CHECK(cudaGetLastError());
  return FEM_OK;
}

template <int MODE, class VT>
int launch_fine_vt(const fem_plan* P, const fem_mg_desc* D, const VT* K, const double* b, const double* x, double* out, double c1, double c2,
                   double* dot, cudaStream_t st) {
  MgFineEpilogue<MODE> epi{reinterpret_cast<const double2*>(b), reinterpret_cast<const double2*>(D->dinv), reinterpret_cast<double2*>(D->d),
                           reinterpret_cast<const double2*>(x), reinterpret_cast<double2*>(out), D->mask, c1, c2, dot != nullptr,
                           D->own_node_lo, D->own_node_hi, 0, P->n_n};
  const SpmvShape sh = spmv_shape(P);
  epi.group = sh.group;
  const FemRedBuf rb{P->red_partials, P->red_ticket};  // order-deterministic r'z of the last post-smoothing step
  const bool aligned = ((reinterpret_cast<uintptr_t>(b) | reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(out) |
                         reinterpret_cast<uintptr_t>(D->dinv) | reinterpret_cast<uintptr_t>(D->d) | reinterpret_cast<uintptr_t>(D->mask)) & 15u) == 0;
  // default: every operand streamed through shared memory by a producer warp (FP32 values: three stages, 0.352 ms per
  // Chebyshev step at 16M elements against 0.569 ms of the register-fed kernel below)
  if (g_fem_tuning.spmv_staged == 0 && spmv_can_stream(P) && aligned) {
    const SpmvStreamArgs A{P->n_n, P->n_tiles, P->nbr_ptr, P->nbr_idx, P->nbr_loc, P->tile_seg};
    const MgStreamEpilogue<MODE> se{reinterpret_cast<const double2*>(b), reinterpret_cast<const double2*>(D->dinv), reinterpret_cast<double2*>(D->d),
                                    reinterpret_cast<const double2*>(x), reinterpret_cast<double2*>(out), D->mask, c1, c2, dot != nullptr,
                                    D->own_node_lo, D->own_node_hi, P->n_n};
    constexpr int smem = SpmvStreamSmem<VT>::TOTAL;
    const unsigned sb = spmv_stream_blocks(P);
#define MGS(G)                                                                                                              \
  do {                                                                                                                      \
    static bool attr_set = false;                                                                                           \
    if (!attr_set) {                                                                                                        \
      FEM_CUDA_CHECK(cudaFuncSetAttribute(mg_fine_stream_kernel<G, MODE, VT>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem)); \
      attr_set = true;                                                                                                      \
    }                                                                                                                       \
    mg_fine_stream_kernel<G, MODE, VT><<<sb, FEM_STREAM_THREADS, smem, st>>>(A, K, x, se, dot, rb);                           \
  } while (0)
    if (sh.group == 4) MGS(4);
    else if (sh.group == 8) MGS(8);
    else MGS(16);
#undef MGS
    FEM_CUDA_CHECK(cudaGetLastError());
    return FEM_OK;
  }
  if (spmv_use_tiles(P)) {
    const unsigned tb = spmv_tile_blocks(P);
#define MGT(G) mg_fine_tiles_kernel<G, MODE, VT><<<tb, FEM_SPMV_THREADS, 0, st>>>(P->n_n, P->n_tiles, P->nbr_ptr, P->nbr_idx, P->nbr_loc, P->tile_seg, K, x, epi, dot, rb)
    if (sh.group == 4) MGT(4);
    else if (sh.group == 8) MGT(8);
    else MGT(16);
#undef MGT
  } else {
#define MGR(G) mg_fine_rows_kernel<G, MODE, VT><<<sh.blocks, 256, 0, st>>>(P->n_n, P->nbr_ptr, P->nbr_idx, K, x, epi, dot, rb)
    if (sh.group == 4) MGR(4);
    else if (sh.group == 8) MGR(8);
    else MGR(16);
#undef MGR
  }
  FEM_CUDA_CHECK(cudaGetLastError());
  return FEM_OK;
}

// level-0 step on the FP32 copy of the matrix when the descriptor carries one (smoother and residual of the V-cycle only)
template <int MODE>
int launch_fine(const fem_plan* P, const fem_mg_desc* D, const double* K, const double* b, const double* x, double* out, double c1, double c2,
                double* dot, cudaStream_t st) {
  if (D->K32) return launch_fine_vt<MODE, float>(P, D, D->K32, b, x, out, c1, c2, dot, st);
  return launch_fine_vt<MODE, double>(P, D, K, b, x, out, c1, c2, dot, st);
}

__global__ void __launch_bounds__(256) mg_to_f32_kernel(int64_t n4, const double4* __restrict__ src, float4* __restrict__ dst) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
    const double2 a = __ldcs(reinterpret_cast<const double2*>(src + i)), b = __ldcs(reinterpret_cast<const double2*>(src + i) + 1);
    __stcs(dst + i, make_float4((float)a.x, (float)a.y, (float)b.x, (float)b.y));
  }
}

// ---- level 0 on the lattice: the smoother and the residual as a symmetric FP32 stencil ---------------------------------
// When node id == lattice point (iy * LX + ix) and the triangulation has one diagonal orientation, every node couples to
// E, W, N, S and one diagonal pair (NE + SW or NW + SE): a 7-point stencil of 2x2 blocks.  The matrix is symmetric, so
// only the upper half is stored - the self block and the blocks towards E, N and the upper diagonal neighbour, 16 planes
// of FP32 = 64 B per node and no index bytes (the block-CSR copy: 112 B of values + 14 B of block positions + the row
// pointers).  The blocks towards W, S and the lower diagonal neighbour are the transposes of those neighbours' E, N and
// diagonal blocks.
enum { LAT_SELF = 0, LAT_E = 1, LAT_N = 2, LAT_D = 3 };

__global__ void __launch_bounds__(256) mg_lattice_check_kernel(int64_t n_n, const int32_t* __restrict__ nbr_ptr, const int32_t* __restrict__ nbr_idx,
                                                               const int32_t* __restrict__ node_lat, int LX, int32_t* err) {
  for (int64_t a = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; a < n_n; a += (int64_t)gridDim.x * blockDim.x) {
    int e = node_lat[a] != (int32_t)a ? 1 : 0;
    const int64_t ia = a % LX, ja = a / LX;
    for (int p = nbr_ptr[a]; p < nbr_ptr[a + 1]; ++p) {
      const int64_t b = nbr_idx[p];
      const int64_t dx = b % LX - ia, dy = b / LX - ja;
      if (dx < -1 || dx > 1 || dy < -1 || dy > 1) e |= 2;
      else if (dx * dy == 1) e |= 4;
      else if (dx * dy == -1) e |= 8;
    }
    if (e) atomicOr(err, e);
  }
}

// one thread per node: its block-CSR row of FP64 values -> the FP32 copy of the row (the layout fem_mg_to_f32 writes) and
// its four upper-half blocks -> the planes (zero where the neighbour does not exist).  Plain FP32 rounding of the same values.
__global__ void __launch_bounds__(256) mg_to_f32_lattice_kernel(int64_t n_n, const int32_t* __restrict__ nbr_ptr, const int32_t* __restrict__ nbr_idx,
                                                                const double* __restrict__ vals, float* __restrict__ k32, float* __restrict__ planes,
                                                                int64_t stride, int LX, int64_t diag_off) {
  for (int64_t a = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; a < n_n; a += (int64_t)gridDim.x * blockDim.x) {
    const int p0 = nbr_ptr[a], deg = nbr_ptr[a + 1] - p0;
    const double2* r0 = reinterpret_cast<const double2*>(vals + 4 * (int64_t)p0);
    const double2* r1 = r0 + deg;
    float2* o0 = reinterpret_cast<float2*>(k32 + 4 * (int64_t)p0);
    float2* o1 = o0 + deg;
    float s[16];
#pragma unroll
    for (int q = 0; q < 16; ++q) s[q] = 0.0f;
    for (int j = 0; j < deg; ++j) {
      const double2 u = __ldcs(r0 + j), v = __ldcs(r1 + j);
      const float2 fu = make_float2((float)u.x, (float)u.y), fv = make_float2((float)v.x, (float)v.y);
      o0[j] = fu;
      o1[j] = fv;
      const int64_t off = (int64_t)nbr_idx[p0 + j] - a;
      const int slot = off == 0 ? LAT_SELF : (off == 1 ? LAT_E : (off == LX ? LAT_N : (off == diag_off ? LAT_D : -1)));
#pragma unroll
      for (int sl = 0; sl < 4; ++sl)
        if (slot == sl) {
          s[4 * sl + 0] = fu.x;
          s[4 * sl + 1] = fu.y;
          s[4 * sl + 2] = fv.x;
          s[4 * sl + 3] = fv.y;
        }
    }
#pragma unroll
    for (int q = 0; q < 16; ++q) __stcs(planes + q * stride + a, s[q]);
  }
}

// One step of the V-cycle's level 0 on the planes, one thread per owned node, nodes in order (the grid walks the lattice
// row by row): the self block is read once (streaming loads), the E, N and diagonal blocks with cached loads - the E block
// of node a - 1 comes from the neighbouring lane, the N and diagonal blocks of the row below were read by the blocks just
// before (L2).  Epilogue: MgStreamEpilogue, the formulas of the block-CSR path (b, D^-1, d, x; Dirichlet mask of the residual).
template <int MODE, bool NW>
__global__ void __launch_bounds__(256) mg_fine_lattice_kernel(const float* __restrict__ S, int64_t stride, int LX, int lat_rows, const double* x,
                                                              const MgStreamEpilogue<MODE> epi, double* dot_out, const FemRedBuf rb) {
  __shared__ double red[32];
  const double2* xv = reinterpret_cast<const double2*>(x);
  const int lane = threadIdx.x & 31;
  double dot = 0.0;
  // warp-uniform loop: every lane takes part in the shuffle of the E blocks
  for (int64_t base = epi.own_lo + (int64_t)blockIdx.x * blockDim.x + (threadIdx.x & ~31); base < epi.own_hi; base += (int64_t)gridDim.x * blockDim.x) {
    const int64_t a = base + lane;
    const bool act = a < epi.own_hi;
    const int64_t ac = act ? a : epi.own_lo;
    const int i = (int)(ac % LX), j = (int)(ac / LX);
    const bool hw = i > 0, he = i < LX - 1, hs = j > 0, hn = j < lat_rows - 1;
    const bool hdu = NW ? (hn && hw) : (hn && he), hdl = NW ? (hs && he) : (hs && hw);
    const int64_t up_d = NW ? ac + LX - 1 : ac + LX + 1, lo_d = NW ? ac - LX + 1 : ac - LX - 1;
    float k[4], e[4], nn[4], dd[4], w[4], sb[4], db[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      k[q] = __ldcs(S + (4 * LAT_SELF + q) * stride + ac);
      e[q] = __ldg(S + (4 * LAT_E + q) * stride + ac);
      nn[q] = __ldg(S + (4 * LAT_N + q) * stride + ac);
      dd[q] = __ldg(S + (4 * LAT_D + q) * stride + ac);
    }
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      w[q] = __shfl_up_sync(0xffffffffu, e[q], 1);
      if (lane == 0) w[q] = hw ? __ldg(S + (4 * LAT_E + q) * stride + ac - 1) : 0.0f;
      if (!hw) w[q] = 0.0f;
      sb[q] = hs ? __ldg(S + (4 * LAT_N + q) * stride + ac - LX) : 0.0f;
      db[q] = hdl ? __ldg(S + (4 * LAT_D + q) * stride + lo_d) : 0.0f;
    }
    const double2 z2 = make_double2(0.0, 0.0);
    const double2 x0 = xv[ac], xe = he ? xv[ac + 1] : z2, xw = hw ? xv[ac - 1] : z2, xn = hn ? xv[ac + LX] : z2, xs = hs ? xv[ac - LX] : z2;
    const double2 xdu = hdu ? xv[up_d] : z2, xdl = hdl ? xv[lo_d] : z2;
    // upper blocks as stored (row i of the block times x of the neighbour), lower blocks transposed
    double y0 = (double)k[0] * x0.x;
    y0 = fma((double)k[1], x0.y, y0);
    double y1 = (double)k[2] * x0.x;
    y1 = fma((double)k[3], x0.y, y1);
#define LAT_UP(B, X)                        \
  y0 = fma((double)B[0], X.x, y0);          \
  y0 = fma((double)B[1], X.y, y0);          \
  y1 = fma((double)B[2], X.x, y1);          \
  y1 = fma((double)B[3], X.y, y1);
#define LAT_LO(B, X)                        \
  y0 = fma((double)B[0], X.x, y0);          \
  y0 = fma((double)B[2], X.y, y0);          \
  y1 = fma((double)B[1], X.x, y1);          \
  y1 = fma((double)B[3], X.y, y1);
    LAT_UP(e, xe)
    LAT_UP(nn, xn)
    LAT_UP(dd, xdu)
    LAT_LO(w, xw)
    LAT_LO(sb, xs)
    LAT_LO(db, xdl)
#undef LAT_UP
#undef LAT_LO
    if (act) {
      double2 sv[MgStreamEpilogue<MODE>::N_IN];
      uchar2 mk = make_uchar2(1, 1);
      sv[0] = epi.b[a];
      if constexpr (MODE == MG_RESID) {
        if (epi.mask) mk = reinterpret_cast<const uchar2*>(epi.mask)[a];
      } else {
        sv[1] = epi.dinv[a];
        sv[2] = epi.dinv[epi.n_n + a];
        sv[3] = epi.c1 != 0.0 ? epi.d[a] : z2;  // d is not read when c1 == 0 (first step of a sweep)
        sv[4] = x0;
      }
      epi(a, y0, y1, sv, mk, dot);
    }
  }
  if (dot_out) {
    const double v[1] = {block_sum(dot, red)};
    double* const dst[1] = {dot_out};
    ordered_accumulate<1>(v, dst, rb);
  }
}

template <int MODE>
int launch_fine_lattice(const fem_plan* P, const fem_mg_desc* D, const double* b, const double* x, double* out, double c1, double c2, double* dot,
                        cudaStream_t st) {
  const MgStreamEpilogue<MODE> se{reinterpret_cast<const double2*>(b), reinterpret_cast<const double2*>(D->dinv), reinterpret_cast<double2*>(D->d),
                                  reinterpret_cast<const double2*>(x), reinterpret_cast<double2*>(out), D->mask, c1, c2, dot != nullptr,
                                  D->own_node_lo, D->own_node_hi, P->n_n};
  const FemRedBuf rb{P->red_partials, P->red_ticket};
  const unsigned blocks = vgrid(D->own_node_hi - D->own_node_lo, P->sm_count);  // <= 8 per SM: the ordered dot's slots
  if (D->lat32_nw) mg_fine_lattice_kernel<MODE, true><<<blocks, 256, 0, st>>>(D->lat32, D->lat32_stride, D->LX, D->lat_rows, x, se, dot, rb);
  else mg_fine_lattice_kernel<MODE, false><<<blocks, 256, 0, st>>>(D->lat32, D->lat32_stride, D->LX, D->lat_rows, x, se, dot, rb);
  FEM_CUDA_CHECK(cudaGetLastError());
  return FEM_OK;
}

// the V-cycle's level-0 smoother and residual: the lattice stencil when the descriptor carries one, else the block-CSR copy
template <int MODE>
int launch_vcycle_fine(const fem_plan* P, const fem_mg_desc* D, const double* K, const double* b, const double* x, double* out, double c1, double c2,
                       double* dot, cudaStream_t st) {
  if (D->lat32 && g_fem_tuning.mg_fine_lattice != 2) return launch_fine_lattice<MODE>(P, D, b, x, out, c1, c2, dot, st);
  return launch_fine<MODE>(P, D, K, b, x, out, c1, c2, dot, st);
}

#define MG_TRY(expr)             \
  do {                           \
    const int _rc = (expr);      \
    if (_rc != FEM_OK) return _rc; \
  } while (0)

// levels l >= 1 (index li = l - 1 into desc->lev); the solution of level l ends in *x_out (one of its xa/xb)
int vcycle_level(const fem_mg_desc* D, int li, const double** x_out, cudaStream_t st) {
  const fem_mg_level& L = D->lev[li];
  const int k = D->degree;
  if (li == D->n_levels - 1) {  // dense inverse (replicated: every rank holds the whole level)
    const int nc = 2 * L.nxn * L.nrows;
    mg_dense_gemv_kernel<<<grid_for((int64_t)nc * 32), 256, 0, st>>>(nc, D->coarse_inv, L.b, L.xa);
    FEM_CUDA_CHECK(cudaGetLastError());
    *x_out = L.xa;
    return FEM_OK;
  }
  double *cur = L.xa, *oth = L.xb;
  const fem_mg_exchange *ecur = &L.ex_xa, *eoth = &L.ex_xb;
  auto swap = [&]() { double* t = cur; cur = oth; oth = t; const fem_mg_exchange* e = ecur; ecur = eoth; eoth = e; };
  MG_TRY(launch_stencil<MG_FIRST>(L, nullptr, cur, 0.0, L.c2[0], st));
  for (int s = 1; s < k; ++s) {
    MG_TRY(run_exchange(*ecur, cur, D->err, st));
    MG_TRY(launch_stencil<MG_CHEB>(L, cur, oth, L.c1[s], L.c2[s], st));
    swap();
  }
  MG_TRY(run_exchange(*ecur, cur, D->err, st));
  MG_TRY(launch_stencil<MG_RESID>(L, cur, L.r, 0.0, 0.0, st));
  MG_TRY(run_exchange(L.ex_r, L.r, D->err, st));
  const fem_mg_level& C = D->lev[li + 1];
  {
    const Geom c = geom_of(C);
    const int64_t items = (int64_t)(C.res_hi - C.res_lo) * C.nxn;
    if (items > 0) {
      mg_restrict_kernel<false><<<grid_for(items), 256, 0, st>>>(c, C.res_lo, C.res_hi, L.nxn, L.nrows, L.g0, L.nrows_global, nullptr,
                                                                 reinterpret_cast<const double2*>(L.r), reinterpret_cast<double2*>(C.b));
      FEM_CUDA_CHECK(cudaGetLastError());
    }
    MG_TRY(run_exchange(C.ex_b, C.b, D->err, st));
  }
  const double* xc = nullptr;
  MG_TRY(vcycle_level(D, li + 1, &xc, st));
  MG_TRY(run_exchange(xc == C.xa ? C.ex_xa : C.ex_xb, xc, D->err, st));
  {
    const int64_t items = (int64_t)(L.own_hi - L.own_lo) * L.nxn;
    if (items > 0) {
      mg_prolong_kernel<<<grid_for(items), 256, 0, st>>>(geom_of(L), L.own_lo, L.own_hi, geom_of(C), reinterpret_cast<const double2*>(xc),
                                                         reinterpret_cast<double2*>(cur));
      FEM_CUDA_CHECK(cudaGetLastError());
    }
  }
  for (int s = 0; s < k; ++s) {
    MG_TRY(run_exchange(*ecur, cur, D->err, st));
    MG_TRY(launch_stencil<MG_CHEB>(L, cur, oth, s == 0 ? 0.0 : L.c1[s], L.c2[s], st));
    swap();
  }
  *x_out = cur;
  return FEM_OK;
}

}  // namespace

extern "C" int fem_mg_sizeof(int which) {
  return which == 0 ? (int)sizeof(fem_mg_exchange) : (which == 1 ? (int)sizeof(fem_mg_level) : (int)sizeof(fem_mg_desc));
}

extern "C" int fem_mg_lattice(int64_t n_n, const double* coord, double x0, double y0, double hx, double hy, int LX, int lat_rows, int g0,
                              int32_t* lat, int32_t* node_lat, int32_t* err, fem_stream stream) {
  FEM_REQUIRE(coord && lat && node_lat && err && n_n > 0 && hx > 0.0 && hy > 0.0 && LX > 0 && lat_rows > 0, "lattice arguments");
  FEM_REQUIRE((int64_t)LX * lat_rows < 2147483647LL, "lattice too large for 32-bit point ids");
  cudaStream_t st = (cudaStream_t)stream;
  FEM_CUDA_CHECK(cudaMemsetAsync(lat, 0xFF, sizeof(int32_t) * (size_t)LX * lat_rows, st));
  mg_lattice_kernel<<<grid_for(n_n), 256, 0, st>>>(n_n, coord, x0, y0, 1.0 / hx, 1.0 / hy, LX, lat_rows, g0, lat, node_lat, err);
  FEM_CUDA_CHECK(cudaGetLastError());
  return FEM_OK;
}

extern "C" int fem_mg_galerkin_fine(const fem_plan* P, const double* K_vals, const uint8_t* row_mask, const uint8_t* col_mask,
                                    const int32_t* lat, int lat_rows, const int32_t* node_lat, int LX, int g0, int nxn, int nrows, int g0c,
                                    double* S, int32_t* err, fem_stream stream) {
  FEM_REQUIRE(P && K_vals && lat && node_lat && S && err && LX > 0 && lat_rows > 0 && nxn > 0 && nrows > 0, "null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  const Geom c{nxn, nrows, g0c, 0, (int64_t)nxn * nrows};
  mg_galerkin_fine_kernel<<<grid_for(c.n, 128), 128, 0, st>>>(P->nbr_ptr, P->nbr_idx, K_vals, row_mask, col_mask ? col_mask : row_mask, lat, lat_rows,
                                                              node_lat, LX, g0, c, S, err);
  FEM_CUDA_CHECK(cudaGetLastError());
  return FEM_OK;
}

extern "C" int fem_mg_galerkin_stencil(int nxf, int nrows_f, int g0f, int nrows_global_f, const double* Sf, int nxc, int nrows_c, int g0c,
                                       int row_lo, int row_hi, double* Sc, fem_stream stream) {
  FEM_REQUIRE(Sf && Sc && nxf > 0 && nrows_f > 0 && nxc > 0 && nrows_c > 0 && row_lo >= 0 && row_hi <= nrows_c, "null pointer or bad rows");
  const Geom f{nxf, nrows_f, g0f, nrows_global_f, (int64_t)nxf * nrows_f}, c{nxc, nrows_c, g0c, 0, (int64_t)nxc * nrows_c};
  const int64_t items = (int64_t)(row_hi - row_lo) * nxc;
  if (items <= 0) return FEM_OK;
  mg_galerkin_stencil_kernel<<<grid_for(items, 128), 128, 0, (cudaStream_t)stream>>>(f, Sf, c, row_lo, row_hi, Sc);
  FEM_CUDA_CHECK(cudaGetLastError());
  return FEM_OK;
}

extern "C" int fem_mg_block_jacobi(const fem_plan* P, const double* K_vals, const uint8_t* mask, double* dinv, fem_stream stream) {
  FEM_REQUIRE(P && K_vals && dinv, "null pointer");
  mg_block_jacobi_kernel<<<grid_for(P->n_n), 256, 0, (cudaStream_t)stream>>>(P->n_n, P->nbr_ptr, P->nbr_idx, K_vals, mask,
                                                                             reinterpret_cast<double2*>(dinv));
  FEM_CUDA_CHECK(cudaGetLastError());
  return FEM_OK;
}

extern "C" int fem_mg_level_finalize(int64_t n, double* S, double thresh, double* dinv, fem_stream stream) {
  FEM_REQUIRE(S && dinv && n > 0, "null pointer");
  mg_level_finalize_kernel<<<grid_for(n), 256, 0, (cudaStream_t)stream>>>(n, S, thresh, reinterpret_cast<double2*>(dinv));
  FEM_CUDA_CHECK(cudaGetLastError());
  return FEM_OK;
}

extern "C" int fem_mg_stencil_apply(int nxn, int nrows, int row_lo, int row_hi, const double* S, const double* x, double* y, fem_stream stream) {
  FEM_REQUIRE(S && x && y && nxn > 0 && nrows > 0 && row_lo >= 0 && row_hi <= nrows, "null pointer or bad rows");
  const Geom g{nxn, nrows, 0, nrows, (int64_t)nxn * nrows};
  const int64_t items = (int64_t)(row_hi - row_lo) * nxn;
  if (items <= 0) return FEM_OK;
  mg_stencil_kernel<MG_APPLY, double, false><<<grid_for(items), 256, 0, (cudaStream_t)stream>>>(g, row_lo, row_hi, S, reinterpret_cast<const double2*>(x), nullptr,
                                                                                 nullptr, nullptr, reinterpret_cast<double2*>(y), 0.0, 0.0);
  FEM_CUDA_CHECK(cudaGetLastError());
  return FEM_OK;
}

extern "C" int fem_mg_stencil_to_dense(int nxn, int nrows, const double* S, double* A, fem_stream stream) {
  FEM_REQUIRE(S && A && nxn > 0 && nrows > 0, "null pointer");
  const Geom g{nxn, nrows, 0, nrows, (int64_t)nxn * nrows};
  cudaStream_t st = (cudaStream_t)stream;
  FEM_CUDA_CHECK(cudaMemsetAsync(A, 0, sizeof(double) * 4 * (size_t)g.n * g.n, st));
  mg_stencil_to_dense_kernel<<<grid_for(g.n * 9), 256, 0, st>>>(g, S, A);
  FEM_CUDA_CHECK(cudaGetLastError());
  return FEM_OK;
}

extern "C" int fem_mg_to_f32(int64_t n, const double* src, float* dst, fem_stream stream) {
  FEM_REQUIRE(src && dst && n > 0 && n % 4 == 0, "null pointer or length not a multiple of 4");
  FEM_REQUIRE((reinterpret_cast<uintptr_t>(src) & 15u) == 0 && (reinterpret_cast<uintptr_t>(dst) & 15u) == 0, "16-byte alignment");
  mg_to_f32_kernel<<<vgrid(n / 4, 0) * 4, 256, 0, (cudaStream_t)stream>>>(n / 4, reinterpret_cast<const double4*>(src), reinterpret_cast<float4*>(dst));
  FEM_CUDA_CHECK(cudaGetLastError());
  return FEM_OK;
}

extern "C" int fem_mg_lattice_check(const fem_plan* P, const int32_t* node_lat, int LX, int32_t* err, fem_stream stream) {
  FEM_REQUIRE(P && node_lat && err && LX > 0, "null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  mg_lattice_check_kernel<<<vgrid(P->n_n, P->sm_count), 256, 0, st>>>(P->n_n, P->nbr_ptr, P->nbr_idx, node_lat, LX, err);
  FEM_CUDA_CHECK(cudaGetLastError());
  return FEM_OK;
}

extern "C" int fem_mg_to_f32_lattice(const fem_plan* P, const double* K_vals, float* k32, float* planes, int64_t stride, int LX, int nw,
                                     fem_stream stream) {
  FEM_REQUIRE(P && K_vals && k32 && planes && stride >= P->n_n && LX > 0, "null pointer or plane stride");
  FEM_REQUIRE(((reinterpret_cast<uintptr_t>(K_vals) | reinterpret_cast<uintptr_t>(k32)) & 15u) == 0, "16-byte alignment");
  cudaStream_t st = (cudaStream_t)stream;
  mg_to_f32_lattice_kernel<<<vgrid(P->n_n, P->sm_count), 256, 0, st>>>(P->n_n, P->nbr_ptr, P->nbr_idx, K_vals, k32, planes, stride, LX,
                                                                      nw ? (int64_t)LX - 1 : (int64_t)LX + 1);
  FEM_CUDA_CHECK(cudaGetLastError());
  return FEM_OK;
}

extern "C" int fem_mg_exchange_run(const fem_mg_exchange* ex, double* v, uint64_t* err, fem_stream stream) {
  FEM_REQUIRE(ex && v, "null pointer");
  return run_exchange(*ex, v, err, (cudaStream_t)stream);
}

extern "C" int fem_peer_allreduce(double* vals, int n, void* comm, const void* const* peers, int64_t lines_word, int64_t seq_word,
                                  int64_t err_word, int rank, int world, fem_stream stream) {
  FEM_REQUIRE(vals && comm && peers && n >= 1 && n <= 8 && world >= 1 && world <= FEM_MG_MAX_PEERS && rank >= 0 && rank < world, "arguments");
  fem_peer_table tab;
  for (int r = 0; r < FEM_MG_MAX_PEERS; ++r) tab.p[r] = r < world ? const_cast<void*>(peers[r]) : nullptr;
  tab.p[rank] = comm;
  const uint64_t timeout_ns = (uint64_t)(g_fem_tuning.peer_timeout_ms > 0 ? g_fem_tuning.peer_timeout_ms : 10000) * 1000000ull;
  peer_allreduce_kernel<<<1, 256, 0, (cudaStream_t)stream>>>(vals, n, reinterpret_cast<uint64_t*>(comm), tab, lines_word, seq_word, err_word, rank, world,
                                                            timeout_ns);
  FEM_CUDA_CHECK(cudaGetLastError());
  return FEM_OK;
}

extern "C" int fem_mg_vcycle(const fem_plan* P, const fem_mg_desc* D, const double* K_vals, const double* r, double* z, double* dot,
                             fem_stream stream) {
  FEM_REQUIRE(P && D && K_vals && r && z, "null pointer");
  FEM_REQUIRE(D->n_levels >= 1 && D->n_levels <= FEM_MG_MAX_LEVELS && D->degree >= 1 && D->degree <= FEM_MG_MAX_DEGREE, "levels / degree");
  FEM_REQUIRE(D->lat && D->node_lat && D->dinv && D->xa && D->xb && D->d && D->r && D->coarse_inv, "descriptor");
  FEM_REQUIRE(D->own_node_lo >= 0 && D->own_node_hi <= P->n_n && D->own_node_lo < D->own_node_hi, "owned node range");
  cudaStream_t st = (cudaStream_t)stream;
  const int k = D->degree;
  const int64_t n2 = P->n_n;
  // pre-smoothing from x = 0
  double *cur = D->xa, *oth = D->xb;
  const fem_mg_exchange *ecur = &D->ex_xa, *eoth = &D->ex_xb;
  auto swap = [&]() { double* t = cur; cur = oth; oth = t; const fem_mg_exchange* e = ecur; ecur = eoth; eoth = e; };
  mg_fine_first_kernel<<<vgrid(n2, P->sm_count), 256, 0, st>>>(D->own_node_lo, D->own_node_hi, n2, reinterpret_cast<const double2*>(r), reinterpret_cast<const double2*>(D->dinv),
                                                              reinterpret_cast<double2*>(D->d), reinterpret_cast<double2*>(cur), D->c2[0]);
  FEM_CUDA_CHECK(cudaGetLastError());
  for (int s = 1; s < k; ++s) {
    MG_TRY(run_exchange(*ecur, cur, D->err, st));
    MG_TRY(launch_vcycle_fine<MG_CHEB>(P, D, K_vals, r, cur, oth, D->c1[s], D->c2[s], nullptr, st));
    swap();
  }
  MG_TRY(run_exchange(*ecur, cur, D->err, st));
  MG_TRY(launch_vcycle_fine<MG_RESID>(P, D, K_vals, r, cur, D->r, 0.0, 0.0, nullptr, st));
  MG_TRY(run_exchange(D->ex_r, D->r, D->err, st));
  const fem_mg_level& C = D->lev[0];
  {
    const Geom c = geom_of(C);
    const int64_t items = (int64_t)(C.res_hi - C.res_lo) * C.nxn;
    if (items > 0) {
      mg_restrict_kernel<true><<<grid_for(items), 256, 0, st>>>(c, C.res_lo, C.res_hi, D->LX, D->lat_rows, D->g0, D->nrows_global, D->lat,
                                                                reinterpret_cast<const double2*>(D->r), reinterpret_cast<double2*>(C.b));
      FEM_CUDA_CHECK(cudaGetLastError());
    }
    MG_TRY(run_exchange(C.ex_b, C.b, D->err, st));
  }
  const double* xc = nullptr;
  MG_TRY(vcycle_level(D, 0, &xc, st));
  MG_TRY(run_exchange(xc == C.xa ? C.ex_xa : C.ex_xb, xc, D->err, st));
  mg_prolong_fine_kernel<<<vgrid(n2, P->sm_count), 256, 0, st>>>(n2, D->node_lat, D->LX, D->g0, D->mask, geom_of(C), reinterpret_cast<const double2*>(xc),
                                                                reinterpret_cast<double2*>(cur));
  FEM_CUDA_CHECK(cudaGetLastError());
  for (int s = 0; s < k; ++s) {
    const bool last = s == k - 1;
    MG_TRY(run_exchange(*ecur, cur, D->err, st));
    MG_TRY(launch_vcycle_fine<MG_CHEB>(P, D, K_vals, r, cur, last ? z : oth, s == 0 ? 0.0 : D->c1[s], D->c2[s], last ? dot : nullptr, st));
    swap();
  }
  return FEM_OK;
}

// One level-0 step on its own (benchmarks, tests): mode 1: out = mask .* (b - K x); mode 2: d = c1 d + c2 D^-1 (b - K x),
// out = x + d, *dot += b'out if dot != NULL.  K_vals is used unless the descriptor carries an FP32 copy.
extern "C" int fem_mg_fine_step(const fem_plan* P, const fem_mg_desc* D, int mode, const double* K_vals, const double* b, const double* x,
                                double* out, double c1, double c2, double* dot, fem_stream stream) {
  FEM_REQUIRE(P && D && K_vals && b && x && out && (mode == MG_RESID || mode == MG_CHEB) && out != x, "arguments");
  cudaStream_t st = (cudaStream_t)stream;
  if (mode == MG_RESID) return launch_fine<MG_RESID>(P, D, K_vals, b, x, out, 0.0, 0.0, nullptr, st);
  return launch_fine<MG_CHEB>(P, D, K_vals, b, x, out, c1, c2, dot, st);
}

extern "C" int fem_mg_fine_step_lattice(const fem_plan* P, const fem_mg_desc* D, int mode, const double* b, const double* x, double* out,
                                        double c1, double c2, double* dot, fem_stream stream) {
  FEM_REQUIRE(P && D && D->lat32 && b && x && out && (mode == MG_RESID || mode == MG_CHEB) && out != x, "arguments");
  cudaStream_t st = (cudaStream_t)stream;
  if (mode == MG_RESID) return launch_fine_lattice<MG_RESID>(P, D, b, x, out, 0.0, 0.0, nullptr, st);
  return launch_fine_lattice<MG_CHEB>(P, D, b, x, out, c1, c2, dot, st);
}

extern "C" int fem_mg_pcg_init(int64_t n, const double* rhs, const uint8_t* mask, double* r, double* x, double* scal, fem_stream stream) {
  FEM_REQUIRE(rhs && r && x && scal && n > 0, "null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  FEM_CUDA_CHECK(cudaMemsetAsync(scal, 0, 8 * sizeof(double), st));
  mg_pcg_init_kernel<<<vgrid(n, 0), 256, 0, st>>>(n, rhs, mask, r, x, scal, fem_red_buffer_for(scal, st));
  FEM_CUDA_CHECK(cudaGetLastError());
  return FEM_OK;
}

extern "C" int fem_mg_pcg_update_xr(int64_t n, const double* p, const double* q, double* x, double* r, double* scal, int iter, fem_stream stream) {
  FEM_REQUIRE(p && q && x && r && scal && n > 0 && n % 2 == 0, "null pointer or odd n");
  mg_pcg_update_xr_kernel<<<vgrid(n / 2, 0), 256, 0, (cudaStream_t)stream>>>(n / 2, reinterpret_cast<const double2*>(p), reinterpret_cast<const double2*>(q),
                                                                            reinterpret_cast<double2*>(x), reinterpret_cast<double2*>(r), scal, iter,
                                                                            fem_red_buffer_for(scal, (cudaStream_t)stream));
  FEM_CUDA_CHECK(cudaGetLastError());
  return FEM_OK;
}

extern "C" int fem_mg_pcg_update_p(int64_t n, const double* z, double* p, double* scal, int iter, fem_stream stream) {
  FEM_REQUIRE(z && p && scal && n > 0 && n % 2 == 0, "null pointer or odd n");
  mg_pcg_update_p_kernel<<<vgrid(n / 2, 0), 256, 0, (cudaStream_t)stream>>>(n / 2, reinterpret_cast<const double2*>(z), reinterpret_cast<double2*>(p), scal, iter);
  FEM_CUDA_CHECK(cudaGetLastError());
  return FEM_OK;
}

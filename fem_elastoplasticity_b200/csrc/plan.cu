// K1 + K2: mesh topology -> structural CSR pattern, node->element incidence lists and geometry.
// Runs once per mesh.  Replaces what scipy's coo_tocsr / csr_matmat build implicitly inside
// get_elastic_stiffness_matrix (Plasticity2D_DP/pythonFEM.py:570,592,595) and the Jacobian part
// (:506-546,585).  Everything is deterministic: per-node lists are sorted, no result depends on
// the order in which atomics land.
#include <stdarg.h>

#include <vector>

#include "common.cuh"

static thread_local char g_err[512] = "no error";
void fem_set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
extern "C" const char* fem_last_error_string(void) { return g_err; }
extern "C" int fem_version(void) { return 100; }

FemTuning g_fem_tuning = {};
extern "C" int fem_set_tuning(const char* key, int value) {
  FEM_REQUIRE(key != nullptr, "key");
  if (!strcmp(key, "spmv_group")) g_fem_tuning.spmv_group = value;
  else if (!strcmp(key, "spmv_blocks_per_sm")) g_fem_tuning.spmv_blocks_per_sm = value;
  else if (!strcmp(key, "assemble_variant")) {
    FEM_REQUIRE(value == 0 || value == 1 || value == 2 || value == 6, "assemble_variant is 0, 1, 2 or 6");
    g_fem_tuning.assemble_variant = value;
  } else if (!strcmp(key, "spmv_unroll")) g_fem_tuning.spmv_unroll = value;
  else if (!strcmp(key, "spmv_staged")) g_fem_tuning.spmv_staged = value;
  else if (!strcmp(key, "peer_timeout_ms")) g_fem_tuning.peer_timeout_ms = value;
  else if (!strcmp(key, "peer_nowait")) g_fem_tuning.peer_nowait = value;
  else if (!strcmp(key, "assemble_canon")) {
    FEM_REQUIRE(value == 0 || value == 2, "assemble_canon is 0 or 2");
    g_fem_tuning.assemble_canon = value;
  } else if (!strcmp(key, "mg_stencil_sym")) g_fem_tuning.mg_stencil_sym = value;
  else if (!strcmp(key, "mg_fine_lattice")) g_fem_tuning.mg_fine_lattice = value;
  else {
    fem_set_error("unknown tuning key %s", key);
    return FEM_ERR_INVALID_ARG;
  }
  return FEM_OK;
}

extern "C" int fem_device_info(int* sm_count, int* cc_major, int* cc_minor, int64_t* free_bytes, int64_t* total_bytes) {
  int dev = 0, n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0) {
    fem_set_error("no CUDA device visible");
    return FEM_ERR_NO_DEVICE;
  }
  FEM_CUDA_CHECK(cudaGetDevice(&dev));
  if (sm_count) FEM_CUDA_CHECK(cudaDeviceGetAttribute(sm_count, cudaDevAttrMultiProcessorCount, dev));
  if (cc_major) FEM_CUDA_CHECK(cudaDeviceGetAttribute(cc_major, cudaDevAttrComputeCapabilityMajor, dev));
  if (cc_minor) FEM_CUDA_CHECK(cudaDeviceGetAttribute(cc_minor, cudaDevAttrComputeCapabilityMinor, dev));
  size_t f = 0, t = 0;
  FEM_CUDA_CHECK(cudaMemGetInfo(&f, &t));
  if (free_bytes) *free_bytes = (int64_t)f;
  if (total_bytes) *total_bytes = (int64_t)t;
  return FEM_OK;
}

// ------------------------------------------------------------------------------------------------
// exclusive scan (int32), three-phase, warp-shuffle based: out[i] = sum_{j<i} in[j], out[n] = total
// ------------------------------------------------------------------------------------------------
constexpr int SCAN_THREADS = 256;
constexpr int SCAN_ITEMS = 8;
constexpr int SCAN_TILE = SCAN_THREADS * SCAN_ITEMS;

__global__ void scan_tile_sums(const int32_t* __restrict__ in, int64_t n, int32_t* __restrict__ tile_sums) {
  __shared__ int32_t ws[SCAN_THREADS / 32];
  const int64_t base = (int64_t)blockIdx.x * SCAN_TILE + (int64_t)threadIdx.x * SCAN_ITEMS;
  int32_t s = 0;
#pragma unroll
  for (int k = 0; k < SCAN_ITEMS; ++k)
    if (base + k < n) s += in[base + k];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if ((threadIdx.x & 31) == 0) ws[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    int32_t t = 0;
    for (int w = 0; w < SCAN_THREADS / 32; ++w) t += ws[w];
    tile_sums[blockIdx.x] = t;
  }
}

__global__ void scan_tiles(const int32_t* __restrict__ in, int64_t n, const int32_t* __restrict__ tile_offsets,
                           int32_t* __restrict__ out) {
  __shared__ int32_t ws[SCAN_THREADS / 32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t base = (int64_t)blockIdx.x * SCAN_TILE + (int64_t)threadIdx.x * SCAN_ITEMS;
  int32_t v[SCAN_ITEMS], s = 0;
#pragma unroll
  for (int k = 0; k < SCAN_ITEMS; ++k) {
    v[k] = (base + k < n) ? in[base + k] : 0;
    s += v[k];
  }
  int32_t inc = s;  // inclusive warp scan of the per-thread sums
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int32_t t = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc += t;
  }
  if (lane == 31) ws[warp] = inc;
  __syncthreads();
  int32_t woff = 0;
  for (int w = 0; w < warp; ++w) woff += ws[w];
  int32_t run = tile_offsets[blockIdx.x] + woff + (inc - s);
#pragma unroll
  for (int k = 0; k < SCAN_ITEMS; ++k) {
    if (base + k < n) out[base + k] = run;
    run += v[k];
  }
  if (base <= n && n < base + SCAN_ITEMS) {  // the thread whose item range contains index n writes the total
    int32_t tot = tile_offsets[blockIdx.x] + woff + (inc - s);
    for (int k = 0; base + k < n; ++k) tot += v[k];
    out[n] = tot;
  }
}

// out has n+1 entries.  Recursive on the tile sums.
static int exclusive_scan_i32(const int32_t* in, int32_t* out, int64_t n, cudaStream_t st) {
  if (n == 0) {
    FEM_CUDA_CHECK(cudaMemsetAsync(out, 0, sizeof(int32_t), st));
    return FEM_OK;
  }
  const int64_t tiles = (n + 1 + SCAN_TILE - 1) / SCAN_TILE;  // +1: the total slot needs an owning thread
  int32_t *sums = nullptr, *offs = nullptr;
  FEM_CUDA_CHECK(cudaMalloc(&sums, sizeof(int32_t) * tiles));
  FEM_CUDA_CHECK(cudaMalloc(&offs, sizeof(int32_t) * (tiles + 1)));
  scan_tile_sums<<<(unsigned)tiles, SCAN_THREADS, 0, st>>>(in, n, sums);
  int rc = FEM_OK;
  if (tiles == 1) {
    FEM_CUDA_CHECK(cudaMemsetAsync(offs, 0, sizeof(int32_t), st));
  } else {
    rc = exclusive_scan_i32(sums, offs, tiles, st);
  }
  if (rc == FEM_OK) scan_tiles<<<(unsigned)tiles, SCAN_THREADS, 0, st>>>(in, n, offs, out);
  cudaError_t e = cudaGetLastError();
  cudaStreamSynchronize(st);
  cudaFree(sums);
  cudaFree(offs);
  if (rc != FEM_OK) return rc;
  FEM_CUDA_CHECK(e);
  return FEM_OK;
}
int fem_exclusive_scan_i32(const int32_t* in, int32_t* out, int64_t n, cudaStream_t st) {  // midpoints.cu
  return exclusive_scan_i32(in, out, n, st);
}

// ------------------------------------------------------------------------------------------------
// incidence lists
// ------------------------------------------------------------------------------------------------
__global__ void count_incidences(const int32_t* __restrict__ elem, int64_t total, int64_t n_n, int32_t* cnt, int* bad) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int32_t node = elem[i];
    if (node < 0 || node >= n_n) {
      atomicAdd(bad, 1);
      continue;
    }
    atomicAdd(&cnt[node], 1);
  }
}

__global__ void fill_incidences(const int32_t* __restrict__ elem, int64_t n_e, int n_p, const int32_t* __restrict__ inc_ptr,
                                int32_t* fill, uint32_t* keys) {
  const int64_t total = n_e * n_p;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int p = (int)(i / n_e);
    const int64_t e = i - (int64_t)p * n_e;
    const int32_t node = elem[i];
    const int32_t slot = atomicAdd(&fill[node], 1);
    keys[inc_ptr[node] + slot] = ((uint32_t)e << 3) | (uint32_t)p;
  }
}

// insertion sort of each node's keys: ascending element (then local index) -> deterministic lists
__global__ void sort_incidences(int64_t n_n, const int32_t* __restrict__ inc_ptr, uint32_t* keys, int* max_inc) {
  int my_max = 0;
  for (int64_t a = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; a < n_n; a += (int64_t)gridDim.x * blockDim.x) {
    const int32_t b = inc_ptr[a], e = inc_ptr[a + 1];
    for (int32_t i = b + 1; i < e; ++i) {
      const uint32_t k = keys[i];
      int32_t j = i - 1;
      while (j >= b && keys[j] > k) {
        keys[j + 1] = keys[j];
        --j;
      }
      keys[j + 1] = k;
    }
    my_max = max(my_max, e - b);
  }
  atomicMax(max_inc, my_max);
}

// Unique neighbours of node a = union of the nodes of its incident elements.  Pass 0 counts, pass 1
// writes them (then sorts).  A candidate is "new" when no earlier candidate of the same node equals it.
template <bool WRITE>
__global__ void node_neighbours(int64_t n_n, int64_t n_e, int n_p, const int32_t* __restrict__ elem,
                                const int32_t* __restrict__ inc_ptr, const uint32_t* __restrict__ keys, int32_t* deg,
                                const int32_t* __restrict__ nbr_ptr, int32_t* nbr_idx, int* max_deg) {
  int my_max = 0;
  for (int64_t a = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; a < n_n; a += (int64_t)gridDim.x * blockDim.x) {
    const int32_t b = inc_ptr[a], e = inc_ptr[a + 1];
    int32_t n_unique = 0;
    const int32_t out0 = WRITE ? nbr_ptr[a] : 0;
    for (int32_t i = b; i < e; ++i) {
      const int64_t el = keys[i] >> 3;
      for (int p = 0; p < n_p; ++p) {
        const int32_t cand = elem[(int64_t)p * n_e + el];
        bool seen = false;
        for (int32_t i2 = b; i2 <= i && !seen; ++i2) {
          const int64_t el2 = keys[i2] >> 3;
          const int pmax = (i2 == i) ? p : n_p;
          for (int p2 = 0; p2 < pmax; ++p2)
            if (elem[(int64_t)p2 * n_e + el2] == cand) {
              seen = true;
              break;
            }
        }
        if (!seen) {
          if (WRITE) {  // insert keeping the list sorted
            int32_t j = out0 + n_unique - 1;
            while (j >= out0 && nbr_idx[j] > cand) {
              nbr_idx[j + 1] = nbr_idx[j];
              --j;
            }
            nbr_idx[j + 1] = cand;
          }
          ++n_unique;
        }
      }
    }
    // a node that belongs to no element keeps empty rows, as in the reference's B^T D B
    if (!WRITE) deg[a] = n_unique;
    my_max = max(my_max, n_unique);
  }
  if (!WRITE) atomicMax(max_deg, my_max);
}

__global__ void slice_widths(int64_t n_n, int64_t n_slices, const int32_t* __restrict__ inc_ptr, int32_t* width32,
                             int32_t* inc_cnt) {
  const int64_t gw = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (gw >= n_slices) return;
  const int64_t a = gw * 32 + lane;
  int c = 0;
  if (a < n_n) {
    c = inc_ptr[a + 1] - inc_ptr[a];
    inc_cnt[a] = c;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) c = max(c, __shfl_xor_sync(0xffffffffu, c, o));
  if (lane == 0) width32[gw] = c * 32;
}

__global__ void widen_i32_to_i64(const int32_t* __restrict__ in, int64_t n, int64_t* __restrict__ out) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) out[i] = in[i];
}

// SELL-32 fill: entry (slice, i, lane) holds incidence i of node slice*32+lane, plus the positions of the
// element's nodes inside that node's (sorted) neighbour list.
__global__ void fill_sell(int64_t n_n, int64_t n_e, int n_p, int meta_words, int64_t sell_entries,
                          const int32_t* __restrict__ elem, const int32_t* __restrict__ inc_ptr,
                          const uint32_t* __restrict__ keys, const int32_t* __restrict__ nbr_ptr,
                          const int32_t* __restrict__ nbr_idx, const int64_t* __restrict__ slice_ptr, uint32_t* inc_key,
                          uint32_t* inc_meta) {
  for (int64_t a = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; a < n_n; a += (int64_t)gridDim.x * blockDim.x) {
    const int64_t sbase = slice_ptr[a >> 5];
    const int lane = (int)(a & 31);
    const int32_t b = inc_ptr[a], e = inc_ptr[a + 1];
    const int32_t nb = nbr_ptr[a], deg = nbr_ptr[a + 1] - nb;
    for (int32_t i = b; i < e; ++i) {
      const uint32_t key = keys[i];
      const int64_t el = key >> 3;
      const int64_t dst = sbase + (int64_t)(i - b) * 32 + lane;
      inc_key[dst] = key;
      uint32_t words[3] = {key & 7u, 0u, 0u};
      for (int p = 0; p < n_p; ++p) {
        const int32_t node = elem[(int64_t)p * n_e + el];
        int lo = 0, hi = deg - 1, pos = 0;
        while (lo <= hi) {  // binary search in the sorted neighbour list
          const int mid = (lo + hi) >> 1;
          const int32_t v = nbr_idx[nb + mid];
          if (v == node) {
            pos = mid;
            break;
          }
          if (v < node) lo = mid + 1; else hi = mid - 1;
        }
        const int byte = p + 1;  // byte 0 of word 0 is the local index
        words[byte >> 2] |= (uint32_t)pos << (8 * (byte & 3));
      }
      for (int w = 0; w < meta_words; ++w) inc_meta[(int64_t)w * sell_entries + dst] = words[w];
    }
  }
}

__global__ void expand_csr(int64_t n_n, const int32_t* __restrict__ nbr_ptr, const int32_t* __restrict__ nbr_idx,
                           int32_t* row_ptr, int32_t* col_idx) {
  for (int64_t a = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; a < n_n; a += (int64_t)gridDim.x * blockDim.x) {
    const int32_t nb = nbr_ptr[a], deg = nbr_ptr[a + 1] - nb;
    const int32_t base = 4 * nb;
    row_ptr[2 * a] = base;
    row_ptr[2 * a + 1] = base + 2 * deg;
    if (a == n_n - 1) row_ptr[2 * n_n] = base + 4 * deg;
    for (int j = 0; j < deg; ++j) {
      const int32_t m = nbr_idx[nb + j];
      col_idx[base + 2 * j] = 2 * m;
      col_idx[base + 2 * j + 1] = 2 * m + 1;
      col_idx[base + 2 * deg + 2 * j] = 2 * m;
      col_idx[base + 2 * deg + 2 * j + 1] = 2 * m + 1;
    }
  }
}

// ------------------------------------------------------------------------------------------------
// K1 geometry: one thread per integration point (Plasticity2D_DP/pythonFEM.py:517-546, :585)
// ------------------------------------------------------------------------------------------------
template <int NP, int NQ>
__global__ void __launch_bounds__(256) geometry_kernel(int64_t n_e, int64_t n_n, FemRefElem ref,
                                                       const int32_t* __restrict__ elem, const double* __restrict__ coord,
                                                       double* __restrict__ dphi1, double* __restrict__ dphi2,
                                                       double* __restrict__ weight, int* bad) {
  const int64_t n_int = n_e * NQ;
  for (int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; g < n_int; g += (int64_t)gridDim.x * blockDim.x) {
    const int64_t e = g / NQ;
    const int q = (int)(g - e * NQ);
    double j11 = 0.0, j12 = 0.0, j21 = 0.0, j22 = 0.0;
#pragma unroll
    for (int p = 0; p < NP; ++p) {  // python sum(): 0 + t0 + t1 + ...   (:530-533)
      const int32_t n = elem[(int64_t)p * n_e + e];
      const double x = coord[n], y = coord[n_n + n];
      const double h1 = ref.dhat1[p * NQ + q], h2 = ref.dhat2[p * NQ + q];
      j11 = j11 + x * h1;
      j12 = j12 + y * h1;
      j21 = j21 + x * h2;
      j22 = j22 + y * h2;
    }
    const double det = j11 * j22 - j12 * j21;                                          // :536
    const double i11 = j22 / det, i12 = -j12 / det, i21 = -j21 / det, i22 = j11 / det;  // :539-542
#pragma unroll
    for (int p = 0; p < NP; ++p) {                                                     // :545-546
      const double h1 = ref.dhat1[p * NQ + q], h2 = ref.dhat2[p * NQ + q];
      dphi1[(int64_t)p * n_int + g] = i11 * h1 + i12 * h2;
      dphi2[(int64_t)p * n_int + g] = i21 * h1 + i22 * h2;
    }
    weight[g] = fabs(det) * ref.wf[q];                                                  // :585
    if (!(fabs(det) > 0.0) || isinf(det)) atomicAdd(bad, 1);
  }
}


// ------------------------------------------------------------------------------------------------
// Staging plan for the TMA assembly kernel (P1, node degree <= 8).  The elements touched by the 32 nodes of a slice
// form a few runs of consecutive ids; each run is covered by fixed-width boxes so that one 2-D TMA box copy brings
// all SoA rows of a tensor (7 geometry rows, 9 DS rows, 3 S rows) for a run.  Pass A (boxw == 0) measures the longest
// run; pass B assigns boxes and the per-incidence position li = box*boxw + offset.  Slices needing more than two
// boxes (row ends of a structured mesh, irregular meshes) are processed by the kernel's direct-load path.
// Every lane of the warp builds the same run list redundantly (no divergence).
// ------------------------------------------------------------------------------------------------
__global__ void build_stage(int64_t n_n, int64_t n_slices, int64_t n_int, int boxw, const int64_t* __restrict__ slice_ptr,
                            const uint32_t* __restrict__ inc_key, const uint32_t* __restrict__ inc_meta,
                            int32_t* __restrict__ stage_box, uint32_t* __restrict__ inc_stage, int* flags) {
  // flags: [0] slices that cannot be described (too many incidences/runs), [1] longest run, [2] slices with > 2 boxes
  constexpr int RT = 8, W = 8;
  const int64_t slice = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (slice >= n_slices) return;
  const int64_t sbase = slice_ptr[slice];
  const int width = (int)((slice_ptr[slice + 1] - sbase) >> 5);
  int32_t* out = stage_box + slice * 3;
  if (width > W) {
    if (lane == 0) { atomicAdd(flags, 1); out[0] = 99; }
    return;
  }
  uint32_t keys[W];
#pragma unroll
  for (int i = 0; i < W; ++i) keys[i] = (i < width) ? inc_key[sbase + (int64_t)i * 32 + lane] : FEM_INVALID_KEY;
  int rs[RT], re[RT];  // [start, end) sorted by start
  int nr = 0;
  bool bad = false;
#pragma unroll
  for (int i = 0; i < W; ++i) {
    if (i >= width) break;
    for (int t = 0; t < 32; ++t) {
      const uint32_t k = __shfl_sync(0xffffffffu, keys[i], t);
      if (k == FEM_INVALID_KEY) continue;
      const int x = (int)(k >> 3);
      bool done = false;
      for (int r = 0; r < nr; ++r)
        if (x >= rs[r] - 2 && x <= re[r] + 1) {  // inside, adjacent, or one element away (the gap is staged too)
          if (x < rs[r]) rs[r] = x;
          else if (x >= re[r]) re[r] = x + 1;
          done = true;
          break;
        }
      if (!done) {
        if (nr == RT) { bad = true; continue; }
        int pos = nr;
        while (pos > 0 && rs[pos - 1] > x) { rs[pos] = rs[pos - 1]; re[pos] = re[pos - 1]; --pos; }
        rs[pos] = x; re[pos] = x + 1;
        ++nr;
      }
    }
  }
  // align to 16 bytes (even element ids) and merge runs that touch or overlap
  for (int r = 0; r < nr; ++r) { rs[r] &= ~1; re[r] = (re[r] + 1) & ~1; if (re[r] > n_int) re[r] = (int)n_int; }
  int m = 0;
  for (int r = 0; r < nr; ++r) {
    if (m > 0 && rs[r] <= re[m - 1] + 2) { if (re[r] > re[m - 1]) re[m - 1] = re[r]; }
    else { rs[m] = rs[r]; re[m] = re[r]; ++m; }
  }
  nr = m;
  if (bad) {
    if (lane == 0) { atomicAdd(flags, 1); out[0] = 99; }
    return;
  }
  if (boxw == 0) {  // pass A: longest run
    int longest = 0;
    for (int r = 0; r < nr; ++r) longest = max(longest, re[r] - rs[r]);
    if (lane == 0) atomicMax(flags + 1, longest);
    return;
  }
  int nb = 0;
  for (int r = 0; r < nr; ++r) nb += (re[r] - rs[r] + boxw - 1) / boxw;
  if (lane == 0) {
    out[0] = nb;
    if (nb > 2) atomicAdd(flags + 2, 1);
    int b = 0;
    for (int r = 0; r < nr && b < 2; ++r)
      for (int st = rs[r]; st < re[r] && b < 2; st += boxw) out[1 + b++] = st;
  }
  // canonical slice (common.cuh): all 32 lists carry the interior-node pattern of the regular triangulation, incidences 0-2 in
  // box 0 and 3-5 in box 1, staged positions advancing by two elements per lane: the assembly then needs lane 0's words only
  bool canon_ok = nb == 2 && width >= 6 && slice * 32 + lane < n_n;
#pragma unroll
  for (int i = 0; i < W; ++i) {
    if (i >= width) break;
    const int64_t at = sbase + (int64_t)i * 32 + lane;
    uint32_t word = 0;
    if (keys[i] != FEM_INVALID_KEY) {
      const int x = (int)(keys[i] >> 3);
      int b0 = 0, li = 0;
      for (int r = 0; r < nr; ++r) {
        if (x >= rs[r] && x < re[r]) li = (b0 + (x - rs[r]) / boxw) * boxw + (x - rs[r]) % boxw;
        b0 += (re[r] - rs[r] + boxw - 1) / boxw;
      }
      if (nb > 2) li = 0;
      const uint32_t meta = inc_meta[at];  // la | pos0<<8 | pos1<<16 | pos2<<24
      word = (uint32_t)li | ((meta & 3u) << 9) | (((meta >> 8) & 15u) << 11) | (((meta >> 16) & 15u) << 15) |
             (((meta >> 24) & 15u) << 19) | 0x80000000u;
    }
    inc_stage[at] = word;
    const int li0 = __shfl_sync(0xffffffffu, (int)(word & 0x1FF), 0);
    if (i < 6) canon_ok = canon_ok && (word & CANON_MASK) == canon_word(i) && (((int)(word & 0x1FF) >= boxw) == (i >= 3)) &&
                          (int)(word & 0x1FF) == li0 + 2 * lane;
    else canon_ok = canon_ok && word == 0u;
  }
  if (__all_sync(0xffffffffu, canon_ok) && lane == 0) { out[0] = nb | 0x100; atomicAdd(flags + 3, 1); }
}


// ------------------------------------------------------------------------------------------------
// x-staging plan of the SpMV.  One CTA per tile of FEM_SPMV_TILE consecutive nodes: the columns (neighbour nodes) its
// rows reference are marked in a shared-memory bitmap over [cmin, cmin + WIN); one thread merges the set bits into
// contiguous ranges (gaps < GAP nodes are bridged); when they fit FEM_SPMV_MAXSEG ranges / FEM_SPMV_CAP nodes, every
// block gets the position of its column inside the concatenated ranges (nbr_loc), else the tile gathers from global memory.
// On a structured P1 mesh a tile sees three ranges of 130 nodes (the node rows below, at and above it).
//
// Bank phases.  The kernels gather x from the concatenated ranges with 16-byte shared-memory loads, eight lanes (two
// nodes x four blocks) per wavefront: two entries whose positions agree mod 8 cost a replay, and whether the entries of
// different ranges collide depends only on the ranges' relative positions mod 8 (ncu on the streaming kernel: every x gather
// took 8 wavefronts instead of 4, a third of the kernel's shared-memory wavefronts, profiles/r2zz).  So every range after
// the first is extended backwards by 0-7 nodes (a few more bytes copied), chosen greedily range by range to minimise the
// collisions of the streaming kernel's access pattern (spmv_stream.cuh: the nodes n and n ^ 2 of an aligned group of
// eight share a wavefront; blocks 0-3 and 4-7 of a row are separate loads), counted over the tile's own rows.
// ------------------------------------------------------------------------------------------------
constexpr int SPMV_WIN = 1 << 16;  // nodes covered by the bitmap
constexpr int SPMV_GAP = 32;
__global__ void __launch_bounds__(FEM_SPMV_TILE) build_spmv_tiles(int64_t n_n, const int32_t* __restrict__ nbr_ptr,
                                                                 const int32_t* __restrict__ nbr_idx, int32_t* __restrict__ tile_seg,
                                                                 uint16_t* __restrict__ nbr_loc, int* n_fallback) {
  __shared__ uint32_t bits[SPMV_WIN / 32];
  __shared__ int s_min, s_max, s_nseg, s_start[FEM_SPMV_MAXSEG], s_len[FEM_SPMV_MAXSEG], s_off[FEM_SPMV_MAXSEG];
  __shared__ int s_total, s_ok, s_shift[FEM_SPMV_MAXSEG], s_cost[8];
  const int64_t tile = blockIdx.x;
  const int64_t a = tile * FEM_SPMV_TILE + threadIdx.x;
  int p0 = 0, deg = 0;
  if (a < n_n) { p0 = nbr_ptr[a]; deg = nbr_ptr[a + 1] - p0; }
  if (threadIdx.x == 0) { s_min = INT32_MAX; s_max = -1; s_nseg = 0; }
  for (int w = threadIdx.x; w < SPMV_WIN / 32; w += blockDim.x) bits[w] = 0u;
  __syncthreads();
  int cmin = INT32_MAX, cmax = -1;
  for (int j = 0; j < deg; ++j) { const int c = nbr_idx[p0 + j]; cmin = min(cmin, c); cmax = max(cmax, c); }
  if (deg > 0) { atomicMin(&s_min, cmin); atomicMax(&s_max, cmax); }
  __syncthreads();
  const int lo = s_min, hi = s_max;
  const bool window_ok = hi >= lo && (hi - lo) < SPMV_WIN;
  if (window_ok) {
    for (int j = 0; j < deg; ++j) { const int c = nbr_idx[p0 + j] - lo; atomicOr(&bits[c >> 5], 1u << (c & 31)); }
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    int nseg = 0, total = 0;
    if (window_ok) {
      int run_start = -1, last = -1;
      const int nwords = ((hi - lo) >> 5) + 1;
      for (int w = 0; w < nwords && nseg <= FEM_SPMV_MAXSEG; ++w) {
        uint32_t m = bits[w];
        while (m) {
          const int b = (w << 5) + __ffs(m) - 1;
          m &= m - 1;
          if (run_start < 0) { run_start = b; }
          else if (b - last > SPMV_GAP) {  // close the run
            if (nseg < FEM_SPMV_MAXSEG) { s_start[nseg] = lo + run_start; s_len[nseg] = last - run_start + 1; s_off[nseg] = total; }
            total += last - run_start + 1;
            ++nseg;
            run_start = b;
          }
          last = b;
        }
      }
      if (run_start >= 0) {
        if (nseg < FEM_SPMV_MAXSEG) { s_start[nseg] = lo + run_start; s_len[nseg] = last - run_start + 1; s_off[nseg] = total; }
        total += last - run_start + 1;
        ++nseg;
      }
    }
    const bool ok = window_ok && nseg >= 1 && nseg <= FEM_SPMV_MAXSEG && total <= FEM_SPMV_CAP;
    s_nseg = ok ? nseg : 0;
    s_total = total;
    s_ok = ok;
    for (int k = 0; k < FEM_SPMV_MAXSEG; ++k) s_shift[k] = 0;
    if (!ok && hi >= lo) atomicAdd(n_fallback, 1);
  }
  __syncthreads();
  // ---- bank phases: shift of range k (mod 8), greedy over the ranges; thread t with bit 1 clear owns the node pair (t, t ^ 2)
  {
    const int nsg = s_nseg;
    int eloc[16], eseg[16], ne = 0;  // raw position and range of the pair's blocks 0-7 (entry e: node e / 8, block e % 8)
    const bool owner = (threadIdx.x & 2) == 0;
    if (nsg > 1 && owner) {
      for (int h = 0; h < 2; ++h) {
        const int64_t an = tile * FEM_SPMV_TILE + (threadIdx.x ^ (h ? 2 : 0));
        int q0 = 0, dg = 0;
        if (an < n_n) { q0 = nbr_ptr[an]; dg = nbr_ptr[an + 1] - q0; }
        for (int j = 0; j < 8; ++j) {
          eloc[8 * h + j] = -1;
          eseg[8 * h + j] = 0;
          if (j < dg) {
            const int c = nbr_idx[q0 + j];
            for (int k = 0; k < nsg; ++k)
              if (c >= s_start[k] && c < s_start[k] + s_len[k]) { eloc[8 * h + j] = s_off[k] + (c - s_start[k]); eseg[8 * h + j] = k; }
          }
        }
      }
      ne = 16;
    }
    for (int k = 1; k < nsg; ++k) {
      if (threadIdx.x < 8) s_cost[threadIdx.x] = 0;
      __syncthreads();
      if (ne) {
        for (int cand = 0; cand < 8; ++cand) {
          int cost = 0;
          for (int b = 0; b < 2; ++b) {  // one wavefront: blocks 4b .. 4b+3 of both nodes
            int unit[8], pos[8], m = 0;
            for (int h = 0; h < 2; ++h)
              for (int j = 4 * b; j < 4 * b + 4; ++j) {
                const int e = 8 * h + j;
                if (eloc[e] < 0 || eseg[e] > k) continue;
                const int l = eloc[e] + (eseg[e] == k ? cand : s_shift[eseg[e]]);
                bool dup = false;
                for (int t = 0; t < m; ++t) dup = dup || pos[t] == l;
                if (!dup) { pos[m] = l; unit[m] = l & 7; ++m; }
              }
            int worst = 1;
            for (int t = 0; t < m; ++t) {
              int mult = 0;
              for (int r = 0; r < m; ++r) mult += unit[r] == unit[t];
              worst = max(worst, mult);
            }
            cost += worst - 1;
          }
          if (cost) atomicAdd(&s_cost[cand], cost);
        }
      }
      __syncthreads();
      if (threadIdx.x == 0) {
        int best = 0;
        for (int cand = 1; cand < 8; ++cand)
          if (s_cost[cand] < s_cost[best]) best = cand;
        s_shift[k] = best;
      }
      __syncthreads();
    }
  }
  if (threadIdx.x == 0) {
    const int nseg = s_nseg;
    bool ok = s_ok != 0;
    // shift (mod 8) of range k relative to its raw position = sum of the backward extensions of ranges 1 .. k
    int ext[FEM_SPMV_MAXSEG] = {0, 0, 0, 0}, total = s_total;
    if (ok && nseg > 1) {
      int prev = 0, extra = 0;
      for (int k = 1; k < nseg; ++k) {
        ext[k] = (s_shift[k] - prev) & 7;
        prev = s_shift[k];
        extra += ext[k];
      }
      bool fits = total + extra <= FEM_SPMV_CAP;
      for (int k = 1; k < nseg; ++k) fits = fits && s_start[k] - ext[k] >= s_start[k - 1] + s_len[k - 1];
      if (!fits)
        for (int k = 0; k < FEM_SPMV_MAXSEG; ++k) ext[k] = 0;
      int off = 0;
      for (int k = 0; k < nseg; ++k) {
        s_start[k] -= ext[k];
        s_len[k] += ext[k];
        s_off[k] = off;
        off += s_len[k];
      }
      total = off;
    }
    int32_t* d = tile_seg + tile * FEM_SPMV_DESC;
    d[0] = ok ? nseg : 0;
    d[1] = ok ? total : 0;
    for (int k = 0; k < FEM_SPMV_MAXSEG; ++k) {
      d[2 + 2 * k] = (ok && k < nseg) ? s_start[k] : 0;
      d[3 + 2 * k] = (ok && k < nseg) ? s_len[k] : 0;
    }
    // block range of the tile (its matrix values and positions are contiguous): streamed as one copy each (spmv_stream.cuh)
    const int64_t a0 = tile * FEM_SPMV_TILE, a1 = (a0 + FEM_SPMV_TILE < n_n) ? a0 + FEM_SPMV_TILE : n_n;
    d[10] = nbr_ptr[a0];
    d[11] = nbr_ptr[a1] - nbr_ptr[a0];
    atomicMax(n_fallback + 1, d[11]);
  }
  __syncthreads();
  const int nseg = s_nseg;
  for (int j = 0; j < deg; ++j) {
    uint16_t loc = 0;
    if (nseg > 0) {
      const int c = nbr_idx[p0 + j];
      for (int k = 0; k < nseg; ++k)
        if (c >= s_start[k] && c < s_start[k] + s_len[k]) loc = (uint16_t)(s_off[k] + (c - s_start[k]));
    }
    nbr_loc[p0 + j] = loc;
  }
}

typedef CUresult (*fem_encode_tiled_fn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                        const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                        CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

int fem_encode_rows_map(CUtensorMap* out, const double* base, int64_t n_int, int rows, int boxw) {
  static fem_encode_tiled_fn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess || !p) {
      fem_set_error("cuTensorMapEncodeTiled is not available from the driver");
      return FEM_ERR_CUDA;
    }
    fn = (fem_encode_tiled_fn)p;
  }
  const cuuint64_t gdim[2] = {(cuuint64_t)n_int, (cuuint64_t)rows};
  const cuuint64_t gstride[1] = {(cuuint64_t)n_int * sizeof(double)};
  const cuuint32_t box[2] = {(cuuint32_t)boxw, (cuuint32_t)rows};
  const cuuint32_t estr[2] = {1, 1};
  const CUresult r = fn(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, const_cast<double*>(base), gdim, gstride, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    fem_set_error("cuTensorMapEncodeTiled failed with CUresult %d (rows=%d boxw=%d)", (int)r, rows, boxw);
    return FEM_ERR_CUDA;
  }
  return FEM_OK;
}

// ------------------------------------------------------------------------------------------------
template <typename T>
static int dmalloc(fem_plan* p, T** ptr, int64_t count) {
  const size_t bytes = sizeof(T) * (size_t)(count > 0 ? count : 1);
  FEM_CUDA_CHECK(cudaMalloc((void**)ptr, bytes));
  p->bytes += (int64_t)bytes;
  return FEM_OK;
}
#define FEM_TRY(x)                \
  do {                            \
    int _rc = (x);                \
    if (_rc != FEM_OK) return _rc; \
  } while (0)

// geometry records of the direct-load assembly kernels (common.cuh: geom_rec): one thread per (point, record entry)
__global__ void build_geom_records(int64_t n_int, int n_p, int rs, const double* __restrict__ geom, double* __restrict__ rec) {
  const int64_t total = n_int * rs;
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
    const int64_t g = t / rs;
    const int k = (int)(t - g * rs);
    rec[t] = k < 1 + 2 * n_p ? geom[(int64_t)k * n_int + g] : 0.0;
  }
}

static int launch_geometry(fem_plan* P, const double* coord, int* d_bad, cudaStream_t st) {
  const int threads = 256;
  const unsigned blocks = (unsigned)fem_div_up(P->n_int, threads);
#define GEO(NP, NQ) \
  geometry_kernel<NP, NQ><<<blocks, threads, 0, st>>>(P->n_e, P->n_n, P->ref, P->elem, coord, P->dphi1, P->dphi2, P->weight, d_bad)
  if (P->n_p == 3 && P->n_q == 1) GEO(3, 1);
  else if (P->n_p == 6 && P->n_q == 7) GEO(6, 7);
  else if (P->n_p == 4 && P->n_q == 4) GEO(4, 4);
  else if (P->n_p == 8 && P->n_q == 9) GEO(8, 9);
  else {
    fem_set_error("unsupported element: n_p=%d n_q=%d (compiled: P1 3/1, P2 6/7, Q1 4/4, Q2 8/9)", P->n_p, P->n_q);
    return FEM_ERR_UNSUPPORTED;
  }
#undef GEO
  FEM_CUDA_CHECK(cudaGetLastError());
  return FEM_OK;
}

static int build_plan(fem_plan* P, const int32_t* elem, const double* coord, cudaStream_t st) {
  const int64_t n_n = P->n_n, n_e = P->n_e;
  const int n_p = P->n_p;
  const int threads = 256;
  auto grid = [&](int64_t n) { int64_t b = (n + threads - 1) / threads; if (b > 65535 * 16) b = 65535 * 16; if (b < 1) b = 1; return (unsigned)b; };

  FEM_TRY(dmalloc(P, &P->elem, n_p * n_e));
  FEM_CUDA_CHECK(cudaMemcpyAsync(P->elem, elem, sizeof(int32_t) * n_p * n_e, cudaMemcpyDeviceToDevice, st));

  int32_t *cnt = nullptr, *inc_ptr = nullptr, *deg = nullptr, *width32 = nullptr, *width_ptr = nullptr;
  uint32_t* keys = nullptr;
  int* flags = nullptr;  // [0] bad node ids, [1] max_inc, [2] max_deg, [3] bad det
  FEM_CUDA_CHECK(cudaMalloc(&flags, 4 * sizeof(int)));
  FEM_CUDA_CHECK(cudaMemsetAsync(flags, 0, 4 * sizeof(int), st));
  FEM_CUDA_CHECK(cudaMalloc(&cnt, sizeof(int32_t) * (n_n + 1)));
  FEM_CUDA_CHECK(cudaMalloc(&inc_ptr, sizeof(int32_t) * (n_n + 1)));
  FEM_CUDA_CHECK(cudaMalloc(&keys, sizeof(uint32_t) * n_p * n_e));
  FEM_CUDA_CHECK(cudaMemsetAsync(cnt, 0, sizeof(int32_t) * (n_n + 1), st));
  int rc = FEM_OK;
  int h_flags[4] = {0, 0, 0, 0};
  do {
    count_incidences<<<grid(n_p * n_e), threads, 0, st>>>(P->elem, n_p * n_e, n_n, cnt, flags);
    if ((rc = exclusive_scan_i32(cnt, inc_ptr, n_n, st)) != FEM_OK) break;
    cudaMemcpy(h_flags, flags, sizeof(h_flags), cudaMemcpyDeviceToHost);
    if (h_flags[0]) {
      fem_set_error("elements reference %d node ids outside [0, n_n)", h_flags[0]);
      rc = FEM_ERR_INVALID_ARG;
      break;
    }
    cudaMemsetAsync(cnt, 0, sizeof(int32_t) * (n_n + 1), st);
    fill_incidences<<<grid(n_p * n_e), threads, 0, st>>>(P->elem, n_e, n_p, inc_ptr, cnt, keys);
    sort_incidences<<<grid(n_n), threads, 0, st>>>(n_n, inc_ptr, keys, flags + 1);
    // neighbour lists
    if (cudaMalloc(&deg, sizeof(int32_t) * (n_n + 1)) != cudaSuccess) { rc = FEM_ERR_CUDA; fem_set_error("cudaMalloc deg"); break; }
    cudaMemsetAsync(deg, 0, sizeof(int32_t) * (n_n + 1), st);
    node_neighbours<false><<<grid(n_n), threads, 0, st>>>(n_n, n_e, n_p, P->elem, inc_ptr, keys, deg, nullptr, nullptr, flags + 2);
    if ((rc = dmalloc(P, &P->nbr_ptr, n_n + 1)) != FEM_OK) break;
    if ((rc = exclusive_scan_i32(deg, P->nbr_ptr, n_n, st)) != FEM_OK) break;
    int32_t n_blocks = 0;
    cudaMemcpy(&n_blocks, P->nbr_ptr + n_n, sizeof(int32_t), cudaMemcpyDeviceToHost);
    cudaMemcpy(h_flags, flags, sizeof(h_flags), cudaMemcpyDeviceToHost);
    P->n_blocks = n_blocks;
    P->nnz = 4 * (int64_t)n_blocks;
    P->max_inc = h_flags[1];
    P->max_degree = h_flags[2];
    if (P->nnz >= (int64_t)INT32_MAX) {
      fem_set_error("nnz=%lld does not fit int32 CSR indices; partition the mesh", (long long)P->nnz);
      rc = FEM_ERR_UNSUPPORTED;
      break;
    }
    if (P->max_degree > 255) {
      fem_set_error("node degree %d > 255 unsupported", P->max_degree);
      rc = FEM_ERR_UNSUPPORTED;
      break;
    }
    if ((rc = dmalloc(P, &P->nbr_idx, n_blocks)) != FEM_OK) break;
    node_neighbours<true><<<grid(n_n), threads, 0, st>>>(n_n, n_e, n_p, P->elem, inc_ptr, keys, nullptr, P->nbr_ptr, P->nbr_idx, nullptr);
    // CSR expansion
    if ((rc = dmalloc(P, &P->row_ptr, P->n_dof + 1)) != FEM_OK) break;
    if ((rc = dmalloc(P, &P->col_idx, P->nnz)) != FEM_OK) break;
    expand_csr<<<grid(n_n), threads, 0, st>>>(n_n, P->nbr_ptr, P->nbr_idx, P->row_ptr, P->col_idx);
    // x-staging plan of the SpMV
    P->n_tiles = (n_n + FEM_SPMV_TILE - 1) / FEM_SPMV_TILE;
    if ((rc = dmalloc(P, &P->tile_seg, P->n_tiles * FEM_SPMV_DESC)) != FEM_OK) break;
    if ((rc = dmalloc(P, &P->nbr_loc, n_blocks + 16)) != FEM_OK) break;  // + slack: the streamed copies are rounded to 16 bytes
    {
      int* nfb = nullptr;  // [0] tiles whose x ranges do not fit, [1] most blocks in one tile
      if (cudaMalloc(&nfb, 2 * sizeof(int)) != cudaSuccess) { rc = FEM_ERR_CUDA; fem_set_error("cudaMalloc nfb"); break; }
      cudaMemsetAsync(nfb, 0, 2 * sizeof(int), st);
      cudaMemsetAsync(P->nbr_loc + n_blocks, 0, 16 * sizeof(uint16_t), st);
      build_spmv_tiles<<<(unsigned)P->n_tiles, FEM_SPMV_TILE, 0, st>>>(n_n, P->nbr_ptr, P->nbr_idx, P->tile_seg, P->nbr_loc, nfb);
      int h_nfb[2] = {0, 0};
      cudaMemcpy(h_nfb, nfb, sizeof(h_nfb), cudaMemcpyDeviceToHost);
      cudaFree(nfb);
      P->spmv_fallback_tiles = h_nfb[0];
      P->tile_max_blocks = h_nfb[1];
    }
    // SELL-32 incidence storage
    P->n_slices = (n_n + 31) / 32;
    if (cudaMalloc(&width32, sizeof(int32_t) * (P->n_slices + 1)) != cudaSuccess ||
        cudaMalloc(&width_ptr, sizeof(int32_t) * (P->n_slices + 1)) != cudaSuccess) { rc = FEM_ERR_CUDA; fem_set_error("cudaMalloc widths"); break; }
    if ((rc = dmalloc(P, &P->inc_cnt, n_n)) != FEM_OK) break;
    slice_widths<<<(unsigned)((P->n_slices * 32 + threads - 1) / threads), threads, 0, st>>>(n_n, P->n_slices, inc_ptr, width32, P->inc_cnt);
    if ((rc = exclusive_scan_i32(width32, width_ptr, P->n_slices, st)) != FEM_OK) break;
    int32_t entries = 0;
    cudaMemcpy(&entries, width_ptr + P->n_slices, sizeof(int32_t), cudaMemcpyDeviceToHost);
    P->sell_entries = entries;
    if ((rc = dmalloc(P, &P->slice_ptr, P->n_slices + 1)) != FEM_OK) break;
    widen_i32_to_i64<<<grid(P->n_slices + 1), threads, 0, st>>>(width_ptr, P->n_slices + 1, P->slice_ptr);
    if ((rc = dmalloc(P, &P->inc_key, P->sell_entries)) != FEM_OK) break;
    if ((rc = dmalloc(P, &P->inc_meta, P->sell_entries * P->meta_words)) != FEM_OK) break;
    cudaMemsetAsync(P->inc_key, 0xFF, sizeof(uint32_t) * (size_t)(P->sell_entries > 0 ? P->sell_entries : 1), st);
    cudaMemsetAsync(P->inc_meta, 0, sizeof(uint32_t) * (size_t)(P->sell_entries * P->meta_words > 0 ? P->sell_entries * P->meta_words : 1), st);
    fill_sell<<<grid(n_n), threads, 0, st>>>(n_n, n_e, n_p, P->meta_words, P->sell_entries, P->elem, inc_ptr, keys, P->nbr_ptr,
                                             P->nbr_idx, P->slice_ptr, P->inc_key, P->inc_meta);
    // geometry
    if ((rc = dmalloc(P, &P->geom, (int64_t)(1 + 2 * n_p) * P->n_int)) != FEM_OK) break;
    P->weight = P->geom;
    P->dphi1 = P->geom + P->n_int;
    P->dphi2 = P->geom + (int64_t)(1 + n_p) * P->n_int;
    if ((rc = dmalloc(P, &P->dscratch, 8 + FEM_SLICE_COUNTERS)) != FEM_OK) break;
    if ((rc = dmalloc(P, &P->red_partials, 3 * FEM_RED_MAXB + 8)) != FEM_OK) break;
    P->red_ticket = reinterpret_cast<unsigned*>(P->red_partials + 3 * FEM_RED_MAXB);
    cudaMemsetAsync(P->red_ticket, 0, 8 * sizeof(double), st);
    if ((rc = launch_geometry(P, coord, flags + 3, st)) != FEM_OK) break;
    // TMA staging plan (P1 meshes of bounded valence whose slices touch few runs of consecutive elements)
    P->stage_ok = 0;
    if (n_p == 3 && P->n_q == 1 && P->max_degree <= 8 && P->max_inc <= 8 && (P->n_int % 2) == 0 && P->n_int >= 64) {
      int* sflags = nullptr;
      if (cudaMalloc(&sflags, 4 * sizeof(int)) != cudaSuccess) { rc = FEM_ERR_CUDA; fem_set_error("cudaMalloc sflags"); break; }
      cudaMemsetAsync(sflags, 0, 4 * sizeof(int), st);
      if ((rc = dmalloc(P, &P->stage_box, P->n_slices * 3)) != FEM_OK) break;
      if ((rc = dmalloc(P, &P->inc_stage, P->sell_entries)) != FEM_OK) break;
      const unsigned sblocks = (unsigned)((P->n_slices * 32 + threads - 1) / threads);
      build_stage<<<sblocks, threads, 0, st>>>(n_n, P->n_slices, P->n_int, 0, P->slice_ptr, P->inc_key, P->inc_meta, P->stage_box,
                                               P->inc_stage, sflags);
      int hs[4] = {1, 0, 0, 0};
      cudaStreamSynchronize(st);
      cudaMemcpy(hs, sflags, sizeof(hs), cudaMemcpyDeviceToHost);
      if (hs[0] == 0 && hs[1] > 0) {
        int boxw = (hs[1] + 1) & ~1;
        if (boxw > FEM_STAGE_MAXBOXW) boxw = FEM_STAGE_MAXBOXW;
        if (boxw < 16) boxw = 16;
        cudaMemsetAsync(sflags, 0, 4 * sizeof(int), st);
        build_stage<<<sblocks, threads, 0, st>>>(n_n, P->n_slices, P->n_int, boxw, P->slice_ptr, P->inc_key, P->inc_meta, P->stage_box,
                                                 P->inc_stage, sflags);
        cudaStreamSynchronize(st);
        cudaMemcpy(hs, sflags, sizeof(hs), cudaMemcpyDeviceToHost);
        P->stage_boxw = boxw;
        P->stage_fallback_slices = hs[2];
        P->stage_canon_slices = hs[3];
        // worth it only when most slices take the TMA path
        if (hs[0] == 0 && (int64_t)hs[2] * 8 <= P->n_slices &&
            fem_encode_rows_map(&P->geom_map, P->geom, P->n_int, 7, boxw) == FEM_OK)
          P->stage_ok = 1;
      }
      cudaFree(sflags);
    }
    P->geom_rec = nullptr;
    P->geom_rs = (1 + 2 * n_p + 3) & ~3;
    if (!P->stage_ok) {  // the direct-load assembly kernels serve this mesh
      if ((rc = dmalloc(P, &P->geom_rec, P->n_int * P->geom_rs)) != FEM_OK) break;
      build_geom_records<<<grid(P->n_int * P->geom_rs), threads, 0, st>>>(P->n_int, n_p, P->geom_rs, P->geom, P->geom_rec);
    }
    cudaError_t e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) { fem_set_error("plan build failed: %s", cudaGetErrorString(e)); rc = FEM_ERR_CUDA; break; }
    cudaMemcpy(h_flags, flags, sizeof(h_flags), cudaMemcpyDeviceToHost);
    if (h_flags[3]) {
      fem_set_error("%d integration points have a zero or non-finite Jacobian determinant", h_flags[3]);
      rc = FEM_ERR_NONFINITE_JACOBIAN;
      break;
    }
  } while (0);
  cudaFree(cnt);
  cudaFree(inc_ptr);
  cudaFree(keys);
  cudaFree(deg);
  cudaFree(width32);
  cudaFree(width_ptr);
  cudaFree(flags);
  if (rc == FEM_OK) {
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { fem_set_error("plan build failed: %s", cudaGetErrorString(e)); rc = FEM_ERR_CUDA; }
  }
  return rc;
}

extern "C" int fem_plan_create(int64_t n_n, int64_t n_e, int n_p, int n_q, const int32_t* elem, const double* coord,
                               const double* h_dhatp1, const double* h_dhatp2, const double* h_wf, fem_stream stream,
                               fem_plan** out) {
  FEM_REQUIRE(out != nullptr, "out");
  *out = nullptr;
  FEM_REQUIRE(n_n > 0 && n_e > 0, "empty mesh");
  FEM_REQUIRE(n_p >= 1 && n_p <= FEM_MAX_NP && n_q >= 1 && n_q <= FEM_MAX_NQ, "n_p/n_q out of range");
  FEM_REQUIRE(elem && coord && h_dhatp1 && h_dhatp2 && h_wf, "null pointer");
  FEM_REQUIRE(n_e < ((int64_t)1 << 28) && n_n < ((int64_t)1 << 30), "mesh too large for one plan; partition it");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    fem_set_error("no CUDA device visible: this library has no CPU fallback");
    return FEM_ERR_NO_DEVICE;
  }
  fem_plan* P = new fem_plan();
  memset(P, 0, sizeof(*P));
  P->n_n = n_n; P->n_e = n_e; P->n_p = n_p; P->n_q = n_q;
  P->n_int = n_e * n_q;
  P->n_dof = 2 * n_n;
  P->meta_words = (n_p + 1 + 3) / 4;
  for (int i = 0; i < n_p * n_q; ++i) { P->ref.dhat1[i] = h_dhatp1[i]; P->ref.dhat2[i] = h_dhatp2[i]; }
  for (int i = 0; i < n_q; ++i) P->ref.wf[i] = h_wf[i];
  int dev = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&P->sm_count, cudaDevAttrMultiProcessorCount, dev);
  const int rc = build_plan(P, elem, coord, (cudaStream_t)stream);
  if (rc != FEM_OK) {
    fem_plan_destroy(P);
    return rc;
  }
  *out = P;
  return FEM_OK;
}

extern "C" int fem_plan_destroy(fem_plan* P) {
  if (!P) return FEM_OK;
  cudaFree(P->stage_box); cudaFree(P->inc_stage); cudaFree(P->tile_seg); cudaFree(P->nbr_loc);
  cudaFree(P->elem); cudaFree(P->nbr_ptr); cudaFree(P->nbr_idx); cudaFree(P->row_ptr); cudaFree(P->col_idx);
  cudaFree(P->inc_cnt); cudaFree(P->slice_ptr); cudaFree(P->inc_key); cudaFree(P->inc_meta);
  cudaFree(P->geom); cudaFree(P->dscratch); cudaFree(P->geom_rec); cudaFree(P->red_partials);
  delete P;
  return FEM_OK;
}

extern "C" int fem_plan_sizes(const fem_plan* P, int64_t* n_n, int64_t* n_e, int64_t* n_int, int64_t* n_dof, int64_t* nnz,
                              int* max_degree) {
  FEM_REQUIRE(P, "plan");
  if (n_n) *n_n = P->n_n;
  if (n_e) *n_e = P->n_e;
  if (n_int) *n_int = P->n_int;
  if (n_dof) *n_dof = P->n_dof;
  if (nnz) *nnz = P->nnz;
  if (max_degree) *max_degree = P->max_degree;
  return FEM_OK;
}
extern "C" int fem_plan_pattern(const fem_plan* P, const int32_t** row_ptr, const int32_t** col_idx, int64_t* nnz) {
  FEM_REQUIRE(P, "plan");
  if (row_ptr) *row_ptr = P->row_ptr;
  if (col_idx) *col_idx = P->col_idx;
  if (nnz) *nnz = P->nnz;
  return FEM_OK;
}
extern "C" int fem_plan_blocks(const fem_plan* P, const int32_t** nbr_ptr, const int32_t** nbr_idx, int64_t* n_blocks) {
  FEM_REQUIRE(P, "plan");
  if (nbr_ptr) *nbr_ptr = P->nbr_ptr;
  if (nbr_idx) *nbr_idx = P->nbr_idx;
  if (n_blocks) *n_blocks = P->n_blocks;
  return FEM_OK;
}
extern "C" int fem_plan_geometry(const fem_plan* P, const double** dphi1, const double** dphi2, const double** weight) {
  FEM_REQUIRE(P, "plan");
  if (dphi1) *dphi1 = P->dphi1;
  if (dphi2) *dphi2 = P->dphi2;
  if (weight) *weight = P->weight;
  return FEM_OK;
}
extern "C" int fem_plan_stage_info(const fem_plan* P, int* stage_ok, int* stage_cap) {
  FEM_REQUIRE(P, "plan");
  if (stage_ok) *stage_ok = P->stage_ok;
  if (stage_cap) *stage_cap = P->stage_boxw;
  return FEM_OK;
}
extern "C" int64_t fem_plan_bytes(const fem_plan* P) { return P ? P->bytes : 0; }

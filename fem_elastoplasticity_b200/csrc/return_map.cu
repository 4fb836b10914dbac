// K5: Drucker-Prager return mapping + consistent tangent, one thread per Gauss point.
// Follows construct_constitutive_problem (Plasticity2D_DP/pythonFEM.py:604-757,
// tsx-tunnel/pythonFEM.py:990-1157) operation by operation; compiled with -fmad=false.
// Pure streaming: 193 B/point (+40 B when the plastic strain / multiplier are written).
#include <math.h>

#include "common.cuh"

struct DpConst {
  double dev_d;   // 1 - 1/3        (dev[0][0])                 :653
  double dev_o;   // 0 - 1/3        (dev[0][1])
  double sqrt2;   // sqrt(2)
  double two_sqrt2;
  double e0[4];   // tsx initial strain (zeros when absent)     tsx :1052
};

struct DpPoint {
  double s[4], ds[9], ep[4], lam;
  int flag;  // 0 elastic, 1 smooth, 2 apex
};

__device__ __forceinline__ void dp_point(const DpConst& k, double e0, double e1, double e2, double p0, double p1,
                                         double p2, double p3, double G, double K, double eta, double c, DpPoint& o) {
  // trial strain E_tr = (e, 0) + e0 - ep_prev                                    :663-668
  const double t0 = (e0 + k.e0[0]) - p0, t1 = (e1 + k.e0[1]) - p1, t2 = (e2 + k.e0[2]) - p2, t3 = (0.0 + k.e0[3]) - p3;
  // dev_E = dev @ E_tr, vol @ E_tr                                                :670-673
  const double d0 = k.dev_d * t0 + k.dev_o * t1 + k.dev_o * t3;
  const double d1 = k.dev_o * t0 + k.dev_d * t1 + k.dev_o * t3;
  const double d2 = 0.5 * t2;
  const double d3 = k.dev_o * t0 + k.dev_o * t1 + k.dev_d * t3;
  const double tr = t0 + t1 + t3;
  const double G2 = 2.0 * G;
  const double st0 = G2 * d0 + K * tr, st1 = G2 * d1 + K * tr, st2 = G2 * d2, st3 = G2 * d3 + K * tr;
  double sq = t0 * d0 + t1 * d1 + t2 * d2 + t3 * d3;                               // :676
  sq = sq > 0.0 ? sq : 0.0;
  const double norm = sqrt(sq);
  const double rho = 2.0 * (G * norm);                                             // :679
  const double ptr = K * tr;                                                       // :682
  const double den_a = K * (eta * eta);                                            // :687-690
  const double den_s = G + den_a;
  const double crit1 = (rho / k.sqrt2 + eta * ptr) - c;
  const double crit2 = (eta * ptr - (den_a * rho) / (G * k.sqrt2)) - c;
  // elastic prediction DS = 2*Dev*G + Vol*K                                       :703
  const double a = (2.0 * k.dev_d) * G + K, b = (2.0 * k.dev_o) * G + K;
  const double dev3[9] = {k.dev_d, k.dev_o, 0.0, k.dev_o, k.dev_d, 0.0, 0.0, 0.0, 0.5};
  o.ds[0] = a; o.ds[1] = b; o.ds[2] = 0.0; o.ds[3] = b; o.ds[4] = a; o.ds[5] = 0.0; o.ds[6] = 0.0; o.ds[7] = 0.0;
  o.ds[8] = G;
  o.s[0] = st0; o.s[1] = st1; o.s[2] = st2; o.s[3] = st3;
  o.ep[0] = p0; o.ep[1] = p1; o.ep[2] = p2; o.ep[3] = p3;
  o.lam = 0.0;
  o.flag = 0;
  if (crit1 > 0.0) {
    if (crit2 <= 0.0) {  // return to the smooth portion                            :710-727
      o.flag = 1;
      const double lam = crit1 / den_s;
      const double n0 = d0 / norm, n1 = d1 / norm, n2 = d2 / norm, n3 = d3 / norm;
      const double sg = k.sqrt2 * G, ke = K * eta;
      const double m0 = sg * n0 + ke, m1 = sg * n1 + ke, m2 = sg * n2, m3 = sg * n3 + ke;
      o.s[0] = st0 - lam * m0; o.s[1] = st1 - lam * m1; o.s[2] = st2 - lam * m2; o.s[3] = st3 - lam * m3;
      const double coef = ((k.two_sqrt2 * (G * G)) * lam) / rho;
      const double nv[3] = {n0, n1, n2}, mv[3] = {m0, m1, m2};
#pragma unroll
      for (int q = 0; q < 9; ++q) {
        const int r = q % 3, cc = q / 3;
        o.ds[q] = (o.ds[q] - coef * (dev3[q] - nv[r] * nv[cc])) - (mv[r] * mv[cc]) / den_s;
      }
      o.lam = lam;
      // plastic strain increment                                                  :752
      const double e3 = eta / 3.0;
      o.ep[0] = p0 + lam * (n0 / k.sqrt2 + e3);
      o.ep[1] = p1 + lam * (n1 / k.sqrt2 + e3);
      o.ep[2] = p2 + (2.0 * lam) * (n2 / k.sqrt2);
      o.ep[3] = p3 + lam * (n3 / k.sqrt2 + e3);
    } else {  // return to the apex                                                 :721,728,755
      o.flag = 2;
      const double sa = c / eta;
      o.s[0] = sa; o.s[1] = sa; o.s[2] = 0.0; o.s[3] = sa;
#pragma unroll
      for (int q = 0; q < 9; ++q) o.ds[q] = 0.0;
      o.lam = (eta * ptr - c) / den_a;
      const double sh = c / ((3.0 * K) * eta);
      o.ep[0] = t0 - sh; o.ep[1] = t1 - sh; o.ep[2] = t2; o.ep[3] = t3 - sh;     // E4 is already E_tr (SURVEY B-2)
    }
  }
}

// One thread per Gauss point, 128 threads, 6 blocks per SM: measured best at 16M points (tools/tune.py) against two points
// per thread (double2 loads and stores) and other block shapes.
__global__ void __launch_bounds__(128, 6) dp_return_map_kernel(
    int64_t n_int, DpConst k, const double* __restrict__ E, double* Ep_prev,
    const double* __restrict__ shear, const double* __restrict__ bulk, const double* __restrict__ eta,
    const double* __restrict__ c, int apply, double* __restrict__ S, double* __restrict__ DS,
    uint8_t* __restrict__ ind_p, double* __restrict__ lambda, double* Ep_out, unsigned long long* counts) {
  __shared__ unsigned int s_cnt[2];
  if (threadIdx.x < 2) s_cnt[threadIdx.x] = 0;
  __syncthreads();
  unsigned int my_s = 0, my_a = 0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_int; i += (int64_t)gridDim.x * blockDim.x) {
    auto ldv = [&](const double* base, int row) { return __ldcs(base + row * n_int + i); };
    const double e0 = ldv(E, 0), e1 = ldv(E, 1), e2 = ldv(E, 2);
    const double g = ldv(shear, 0), kb = ldv(bulk, 0), et = ldv(eta, 0), cc = ldv(c, 0);
    double p0 = 0.0, p1 = 0.0, p2 = 0.0, p3 = 0.0;
    if (Ep_prev) {
      p0 = ldv(Ep_prev, 0); p1 = ldv(Ep_prev, 1); p2 = ldv(Ep_prev, 2); p3 = ldv(Ep_prev, 3);
    }
    DpPoint o;
    dp_point(k, e0, e1, e2, p0, p1, p2, p3, g, kb, et, cc, o);
    my_s += (o.flag == 1);
    my_a += (o.flag == 2);
    auto stv = [&](double* base, int row, double v) { __stcs(base + row * n_int + i, v); };
#pragma unroll
    for (int q = 0; q < 4; ++q) stv(S, q, o.s[q]);
#pragma unroll
    for (int q = 0; q < 9; ++q) stv(DS, q, o.ds[q]);
    ind_p[i] = o.flag != 0;
    if (lambda) stv(lambda, 0, o.lam);
    if (apply) {
      if (Ep_prev && o.flag != 0) {  // in-place history update (ep aliases ep_prev, :751)
#pragma unroll
        for (int q = 0; q < 4; ++q) Ep_prev[q * n_int + i] = o.ep[q];
      }
      if (Ep_out && Ep_out != Ep_prev) {
#pragma unroll
        for (int q = 0; q < 4; ++q) stv(Ep_out, q, o.ep[q]);
      }
    } else if (Ep_out) {
#pragma unroll
      for (int q = 0; q < 4; ++q) stv(Ep_out, q, 0.0);
    }
  }
  if (counts) {
    my_s = __reduce_add_sync(0xffffffffu, my_s);
    my_a = __reduce_add_sync(0xffffffffu, my_a);
    if ((threadIdx.x & 31) == 0) {
      if (my_s) atomicAdd(&s_cnt[0], my_s);
      if (my_a) atomicAdd(&s_cnt[1], my_a);
    }
    __syncthreads();
    if (threadIdx.x < 2 && s_cnt[threadIdx.x]) atomicAdd(&counts[threadIdx.x], (unsigned long long)s_cnt[threadIdx.x]);
  }
}

extern "C" int fem_dp_return_map(int64_t n_int, const double* E, const double* h_e0, double* Ep_prev,
                                 const double* shear, const double* bulk, const double* eta, const double* c, int apply,
                                 double* S, double* DS, uint8_t* ind_p, double* lambda, double* Ep_out, int64_t* counts,
                                 fem_stream stream) {
  FEM_REQUIRE(n_int >= 0, "n_int");
  if (n_int == 0) return FEM_OK;
  FEM_REQUIRE(E && shear && bulk && eta && c && S && DS && ind_p, "null device pointer");
  DpConst k;
  // the constants are formed exactly as numpy forms them (Plasticity2D_DP/pythonFEM.py:651-653, :689)
  const volatile double third = 1.0 / 3.0;
  k.dev_d = 1.0 - third;
  k.dev_o = 0.0 - third;
  k.sqrt2 = sqrt(2.0);
  k.two_sqrt2 = 2.0 * k.sqrt2;
  for (int i = 0; i < 4; ++i) k.e0[i] = h_e0 ? h_e0[i] : 0.0;
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const int64_t cap = (int64_t)sms * 8 * 64;  // grid-stride beyond that
  int64_t blocks = (n_int + 127) / 128;
  if (blocks > cap) blocks = cap;
  dp_return_map_kernel<<<(unsigned)blocks, 128, 0, (cudaStream_t)stream>>>(n_int, k, E, Ep_prev, shear, bulk, eta, c, apply, S, DS, ind_p,
                                                                           lambda, Ep_out, reinterpret_cast<unsigned long long*>(counts));
  FEM_CUDA_CHECK(cudaGetLastError());
  return FEM_OK;
}

// Host side of the CWT / ssq_cwt plan: buffers, twiddle tables, chunking over
// (signal, scale) rows and kernel dispatch.  Included once per dtype
// (cwt_f32.cu, cwt_f64.cu) so the two sets of kernels compile in parallel.
#pragma once
#include "host_common.h"
#include "cwt_kernels.cuh"
#include "cwt_fast.cuh"
#include "cwt_grid.cuh"
#include "cwt_sblk.cuh"
#include "cwt_generic.cuh"
#include <cstdlib>
#include <cstring>
#include <algorithm>

namespace ssqb {

template <typename T>
static std::vector<cx<T>> make_roots(long long count, long long step, long long n) {
  // exp(+2 pi i (m*step) / n), m < count, evaluated in float64
  std::vector<cx<T>> v((size_t)count);
  for (long long m = 0; m < count; ++m) {
    long long k = (m * step) % n;
    // octant-exact angles keep cos/sin symmetric
    double ang = 2.0 * M_PI * (double)k / (double)n;
    v[(size_t)m] = mkc<T>((T)cos(ang), (T)sin(ang));
  }
  return v;
}


template <typename T, int LOG_M, int MODE>
static int launch_pass1_t(const CwtArgs<T>& A, int narr, cudaStream_t st) {
  constexpr int M = 1 << LOG_M;
  constexpr int R1 = Tile<T>::ELEMS / M;
  size_t smem = ((size_t)M * (R1 + 1) + M) * sizeof(cx<T>);
  auto kern = cwt_pass1_kernel<T, LOG_M, MODE>;
  SSQB_CUDA(set_smem_limit(kern, smem));
  long long ncol1 = (long long)A.nrows << A.logF;
  dim3 grid((unsigned)((ncol1 + R1 - 1) / R1), (unsigned)narr);
  kern<<<grid, Tile<T>::NT, smem, st>>>(A);
  SSQB_LAUNCH_CHECK();
  return 0;
}

template <typename T, int MODE>
static int launch_pass1(const CwtArgs<T>& A, int narr, cudaStream_t st) {
  switch (A.logI2) {
#define SSQB_P1(L) case L: return launch_pass1_t<T, L, MODE>(A, narr, st);
    SSQB_P1(1) SSQB_P1(2) SSQB_P1(3) SSQB_P1(4) SSQB_P1(5) SSQB_P1(6)
    SSQB_P1(7) SSQB_P1(8) SSQB_P1(9) SSQB_P1(10) SSQB_P1(11) SSQB_P1(12)
#undef SSQB_P1
    default: break;
  }
  return set_error(SSQB_E_UNSUPP, "unsupported pass-1 length 2^%d", A.logI2);
}

template <typename T, int LOG_F, int NARR, int EPI>
static int launch_pass2_t(const CwtArgs<T>& A, int write_dWx, cudaStream_t st) {
  constexpr int F = 1 << LOG_F;
  constexpr int R2 = Tile<T>::ELEMS / F;
  size_t smem = ((size_t)NARR * Tile<T>::ELEMS + F) * sizeof(cx<T>);
  auto kern = cwt_pass2_kernel<T, LOG_F, NARR, EPI>;
  SSQB_CUDA(set_smem_limit(kern, smem));
  long long ncols = (long long)A.nrows << A.logI2;
  dim3 grid((unsigned)((ncols + R2 - 1) / R2));
  kern<<<grid, Tile<T>::NT, smem, st>>>(A, write_dWx);
  SSQB_LAUNCH_CHECK();
  return 0;
}

template <typename T, int NARR, int EPI>
static int launch_pass2(const CwtArgs<T>& A, int write_dWx, cudaStream_t st) {
  switch (A.logF) {
#define SSQB_P2(L) case L: return launch_pass2_t<T, L, NARR, EPI>(A, write_dWx, st);
    SSQB_P2(1) SSQB_P2(2) SSQB_P2(3) SSQB_P2(4) SSQB_P2(5) SSQB_P2(6)
    SSQB_P2(7) SSQB_P2(8) SSQB_P2(9)
#undef SSQB_P2
    default: return set_error(SSQB_E_UNSUPP, "unsupported pass-2 length 2^%d", A.logF);
  }
}

// cwt_rows_kernel: every row tile is 2^ROWS_LOGE points -- direct rows, block rows and pass 2 of
// the two-pass rows (R2 = 8 lanes at F = 512).  One butterfly per thread in float32, two in
// float64 (1024-thread CTAs need <= 64 registers).
static constexpr int ROWS_LOGE = 12;

template <typename T, int LOG_F, int NARR, int GEN, int QMAX>
static int launch_rows(const FastArgs<T>& P, unsigned grid_y, cudaStream_t st) {
  constexpr int LOGE = ROWS_LOGE, BPT = sizeof(T) == 4 ? 1 : 2;
  constexpr int ELEMS = 1 << LOGE;
  constexpr int NT = ELEMS / (8 * BPT);
  constexpr int F = 1 << LOG_F;
  const CwtArgs<T>& A = P.A;
  size_t smem = (size_t)512 * sizeof(cx<T>);
  if (LOG_F > 3) smem += (size_t)NARR * RowsTile<T, LOGE, LOG_F>::SARR * sizeof(cx<T>);
  if (GEN == GEN_DIRECT) smem += (size_t)QMAX * F * 4 * sizeof(T);
  auto kern = cwt_rows_kernel<T, LOGE, LOG_F, NARR, GEN, QMAX, false, BPT>;
  if constexpr (NARR == 2)
    if (P.ssq) kern = cwt_rows_kernel<T, LOGE, LOG_F, 2, GEN, QMAX, true, BPT>;
  SSQB_CUDA(set_smem_limit(kern, smem));
  long long nF = (long long)A.n_up >> LOG_F;         // output phases per row
  dim3 grid((unsigned)(nF / (ELEMS / F)), grid_y);
  kern<<<grid, NT, smem, st>>>(P);
  SSQB_LAUNCH_CHECK();
  return 0;
}

// direct classes: 0: band <= 8 bins (F=8), 1: <= 64 (F=64), 2..5: <= 512*{1,2,4,8} (F=512);
// float64 has no class 5 (its band staging + tiles fit 227 KB only up to Q = 4)
template <typename T, int NARR>
static int launch_direct_q(const FastArgs<T>& P, int qclass, unsigned gy, cudaStream_t st) {
  switch (qclass) {
    case 0: return launch_rows<T, 3, NARR, GEN_DIRECT, 1>(P, gy, st);
    case 1: return launch_rows<T, 6, NARR, GEN_DIRECT, 1>(P, gy, st);
    case 2: return launch_rows<T, 9, NARR, GEN_DIRECT, 1>(P, gy, st);
    case 3: return launch_rows<T, 9, NARR, GEN_DIRECT, 2>(P, gy, st);
    case 4: return launch_rows<T, 9, NARR, GEN_DIRECT, 4>(P, gy, st);
    case 5:
      if constexpr (sizeof(T) == 4) return launch_rows<T, 9, NARR, GEN_DIRECT, 8>(P, gy, st);
      break;
    default: break;
  }
  return set_error(SSQB_E_UNSUPP, "no direct row class %d", qclass);
}

template <typename T>
static int launch_direct(const FastArgs<T>& P, int qclass, int narr, long long B, cudaStream_t st) {
  const unsigned gy = (unsigned)(B * P.n_rows);
  return narr == 2 ? launch_direct_q<T, 2>(P, qclass, gy, st) : launch_direct_q<T, 1>(P, qclass, gy, st);
}

// pass 2 of the two-pass route through the same row kernel; the scratch written by
// pass 1 is tiled [col / R2][512][R2] with R2 = 2^P.scratch_logR2 = this kernel's lanes
template <typename T>
static int launch_rows_scratch(const FastArgs<T>& P, int narr, cudaStream_t st) {
  const unsigned gy = (unsigned)P.A.nrows;
  return narr == 2 ? launch_rows<T, 9, 2, GEN_SCRATCH, 1>(P, gy, st)
                   : launch_rows<T, 9, 1, GEN_SCRATCH, 1>(P, gy, st);
}

// pass 1 of the two-pass rows in tiles of Tile<T>::ELEMS points; gridDim.z = nz picks the
// first array of a CTA (NARR = 1, nz = 2: W and dW in CTAs of their own)
template <typename T, int LOG_M, int NARR>
static int launch_pass1f_t(const FastArgs<T>& P, cudaStream_t st, int nz = 1) {
  constexpr int LOGE1 = Tile<T>::ELEMS == 8192 ? 13 : 12;
  constexpr int NT = Tile<T>::NT;
  constexpr int M = 1 << LOG_M;
  constexpr int R1 = (1 << LOGE1) / M;
  static_assert(R1 >= 1, "tile smaller than the transform");
  size_t smem = ((size_t)NARR * M * (R1 + 1) + M) * sizeof(cx<T>);
  auto kern = cwt_pass1f_kernel<T, LOG_M, NARR, LOGE1, NT>;
  SSQB_CUDA(set_smem_limit(kern, smem));
  dim3 grid((unsigned)(512 / R1), (unsigned)P.A.nrows, (unsigned)nz);
  kern<<<grid, NT, smem, st>>>(P);
  SSQB_LAUNCH_CHECK();
  return 0;
}

// long pass-1 transforms (I2 = 1024 .. 4096): one array per CTA when two do not fit the
// 227 KB of shared memory
template <typename T, int LOG_M>
static int launch_pass1f_long(const FastArgs<T>& P, int narr, cudaStream_t st) {
  constexpr int M = 1 << LOG_M;
  constexpr int R1 = Tile<T>::ELEMS / M;
  constexpr size_t two = ((size_t)2 * M * (R1 + 1) + M) * sizeof(cx<T>);
  if (narr == 2 && two <= (size_t)227 * 1024)
    return launch_pass1f_t<T, LOG_M, 2>(P, st, 1);
  return launch_pass1f_t<T, LOG_M, 1>(P, st, narr);
}

template <typename T>
static int launch_pass1v(const FastArgs<T>& P, cudaStream_t st) {
  constexpr int R1 = 8;
  using V4 = typename V4T<T>::type;
  size_t smem = (size_t)512 * R1 * sizeof(V4) + 512 * sizeof(cx<T>);
  auto kern = cwt_pass1v_kernel<T, R1>;
  SSQB_CUDA(set_smem_limit(kern, smem));
  kern<<<dim3(512 / R1, (unsigned)P.A.nrows), 64 * R1, smem, st>>>(P);
  SSQB_LAUNCH_CHECK();
  return 0;
}

// returns -100 when this geometry has no fast pass 1 (caller uses the generic kernel)
template <typename T>
static int launch_pass1f(const FastArgs<T>& P, int narr, cudaStream_t st) {
  switch (P.A.logI2) {
#define SSQB_P1F(L) case L: return narr == 2 ? launch_pass1f_t<T, L, 2>(P, st) \
                                             : launch_pass1f_t<T, L, 1>(P, st);
    SSQB_P1F(4) SSQB_P1F(5) SSQB_P1F(6) SSQB_P1F(7) SSQB_P1F(8)
#undef SSQB_P1F
    // 512-point transforms of W and dW: both arrays as one 16-byte element
    case 9: return narr == 2 ? launch_pass1v<T>(P, st) : launch_pass1f_t<T, 9, 1>(P, st);
    case 10: return launch_pass1f_long<T, 10>(P, narr, st);
    case 11: return launch_pass1f_long<T, 11>(P, narr, st);
    case 12: return launch_pass1f_long<T, 12>(P, narr, st);
    default: return -100;
  }
}


// ---- short-block rows (cwt_sblk.cuh) ----------------------------------------------------
template <typename T>
static int launch_sblk_fwd(const SblkArgs<T>& S, cudaStream_t st) {
  constexpr int LP = SblkGeom<T>::LOG_P;
  size_t smem = ((size_t)1 << LP) * sizeof(cx<T>);
  auto kern = sblk_fwd_kernel<T, LP>;
  SSQB_CUDA(set_smem_limit(kern, smem));
  kern<<<dim3((unsigned)S.nblk, (unsigned)S.B), (1 << LP) / 8, smem, st>>>(S);
  SSQB_LAUNCH_CHECK();
  return 0;
}
template <typename T, int NARR, bool SSQ>
static int launch_sblk_rows_t(const SblkArgs<T>& S, cudaStream_t st) {
  constexpr int LP = SblkGeom<T>::LOG_P;
  using V4 = typename V4T<T>::type;
  size_t smem = ((size_t)1 << LP) * (sizeof(V4) + sizeof(cx<T>));
  auto kern = sblk_rows_kernel<T, LP, NARR, SSQ>;
  SSQB_CUDA(set_smem_limit(kern, smem));
  // persistent grid: as many CTAs as the current device holds at once
  int dev = 0, sms = 0, per = 0;
  SSQB_CUDA(cudaGetDevice(&dev));
  SSQB_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  SSQB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per, kern, (1 << LP) / 8, smem));
  const long long ctas = (long long)sms * (per < 1 ? 1 : per);
  long long items = S.B * (long long)S.n_rows * S.nblk;
  unsigned g = (unsigned)(items < ctas ? items : ctas);
  if (g < 1) return 0;
  kern<<<g, (1 << LP) / 8, smem, st>>>(S);
  SSQB_LAUNCH_CHECK();
  return 0;
}
template <typename T>
static int launch_sblk_rows(const SblkArgs<T>& S, int narr, bool ssq, cudaStream_t st) {
  if (narr == 2 && ssq) return launch_sblk_rows_t<T, 2, true>(S, st);
  if (narr == 2) return launch_sblk_rows_t<T, 2, false>(S, st);
  return launch_sblk_rows_t<T, 1, false>(S, st);
}

// ---- gridded narrow-band rows (cwt_grid.cuh) ------------------------------------------
// phi_hat(nu) = int phi(s) e^{-2 pi i nu s} ds of the exponential-of-semicircle kernel,
// Gauss-Legendre in theta after s = (K/2) sin(theta) (the integrand becomes smooth)
static void gauss_legendre(int n, std::vector<double>& x, std::vector<double>& w) {
  x.assign((size_t)n, 0.0); w.assign((size_t)n, 0.0);
  for (int i = 0; i < (n + 1) / 2; ++i) {
    double z = cos(M_PI * (i + 0.75) / (n + 0.5)), pp = 1.0;
    for (int it = 0; it < 100; ++it) {
      double p1 = 1.0, p2 = 0.0;
      for (int j = 0; j < n; ++j) { double p3 = p2; p2 = p1; p1 = ((2.0 * j + 1.0) * z * p2 - j * p3) / (j + 1.0); }
      pp = n * (z * p1 - p2) / (z * z - 1.0);
      double z1 = z; z = z1 - p1 / pp;
      if (fabs(z - z1) < 1e-15) break;
    }
    x[(size_t)i] = -z; x[(size_t)(n - 1 - i)] = z;
    w[(size_t)i] = w[(size_t)(n - 1 - i)] = 2.0 / ((1.0 - z * z) * pp * pp);
  }
}
static inline double grid_phi(double s, int K, double beta) {
  double z = 1.0 - (2.0 * s / K) * (2.0 * s / K);
  return z > 0.0 ? exp(beta * (sqrt(z) - 1.0)) : 0.0;
}
static double grid_phi_hat(double nu, int K, double beta, const std::vector<double>& gx,
                           const std::vector<double>& gw) {
  double acc = 0.0;
  for (size_t q = 0; q < gx.size(); ++q) {
    double th = 0.5 * M_PI * gx[q], ct = cos(th), sn = sin(th);
    acc += gw[q] * exp(beta * (ct - 1.0)) * cos(2.0 * M_PI * nu * 0.5 * K * sn) * ct;
  }
  return acc * 0.5 * M_PI * 0.5 * K;
}

template <typename T, int LOG_M>
static int launch_grid_dec_t(const GridArgs<T>& G, const GridRow* rows, int n_cls, cudaStream_t st) {
  using Geo = DecGeom<LOG_M>;
  size_t smem = ((size_t)2 * Geo::M * Geo::R + Geo::M) * sizeof(cx<T>);
  if (smem > (size_t)227 * 1024) return set_error(SSQB_E_UNSUPP, "coarse grid 2^%d too long", LOG_M);
  auto kern = grid_dec_ifft_kernel<T, LOG_M>;
  SSQB_CUDA(set_smem_limit(kern, smem));
  long long pairs = (long long)n_cls * G.B;
  dim3 grid((unsigned)((pairs + Geo::R - 1) / Geo::R));
  kern<<<grid, Geo::NT, smem, st>>>(G, rows, n_cls);
  SSQB_LAUNCH_CHECK();
  return 0;
}
template <typename T, int LOG_M>
static int launch_grid_dec_single(const GridArgs<T>& G, const GridRow* rows, int n_cls, cudaStream_t st) {
  size_t smem = ((size_t)1 << LOG_M) * sizeof(cx<T>);
  auto kern = grid_dec_single_kernel<T, LOG_M>;
  SSQB_CUDA(set_smem_limit(kern, smem));
  kern<<<dim3((unsigned)(n_cls * G.B), 2), 1024, smem, st>>>(G, rows, n_cls);
  SSQB_LAUNCH_CHECK();
  return 0;
}

template <typename T, int LOG_MB>
static int launch_grid_dec_split(const GridArgs<T>& G, int logR, const GridRow* rows, int n_cls,
                                 cudaStream_t st) {
  size_t smem = ((size_t)1 << LOG_MB) * sizeof(cx<T>);
  auto kern = grid_dec_split_kernel<T, LOG_MB>;
  SSQB_CUDA(set_smem_limit(kern, smem));
  kern<<<dim3((unsigned)(((long long)n_cls * G.B) << logR), 2), 1024, smem, st>>>(G, rows, n_cls, logR);
  SSQB_LAUNCH_CHECK();
  return 0;
}

template <typename T>
static int launch_grid_dec(const GridArgs<T>& G, int logM, const GridRow* rows, int n_cls,
                           cudaStream_t st) {
  constexpr int BASE = (sizeof(T) == 4) ? 14 : 13;
  if (logM > BASE) return launch_grid_dec_split<T, BASE>(G, logM - BASE, rows, n_cls, st);
  // one CTA per transform of 2^BASE points (it fills an SM's shared memory)
  if (logM == BASE) return launch_grid_dec_single<T, BASE>(G, rows, n_cls, st);
  switch (logM) {
#define SSQB_GD(L) case L: return launch_grid_dec_t<T, L>(G, rows, n_cls, st);
    SSQB_GD(6) SSQB_GD(7) SSQB_GD(8) SSQB_GD(9) SSQB_GD(10) SSQB_GD(11) SSQB_GD(12)
#undef SSQB_GD
    case 13:
      if constexpr (sizeof(T) == 4) return launch_grid_dec_t<T, 13>(G, rows, n_cls, st);
      break;
    default: break;
  }
  return set_error(SSQB_E_UNSUPP, "no coarse-grid transform of 2^%d points", logM);
}

template <typename T>
static int launch_grid_dec_small(const GridArgs<T>& G, const DecSmallPlan& P, cudaStream_t st) {
  size_t smem = ((size_t)2 * 2048 + 2048) * sizeof(cx<T>);
  auto kern = grid_dec_ifft_small_kernel<T>;
  SSQB_CUDA(set_smem_limit(kern, smem));
  if (P.cta_start[6] <= 0) return 0;
  kern<<<dim3((unsigned)P.cta_start[6]), 256, smem, st>>>(G, P);
  SSQB_LAUNCH_CHECK();
  return 0;
}

template <typename T> struct GridTaps;            // kernel width K
template <> struct GridTaps<float>  { static constexpr int K = 8; };
template <> struct GridTaps<double> { static constexpr int K = 14; };

// outputs per thread of the interpolation kernel: K * interp_ppk.  ssq in float32: 16 (measured,
// B = 64, groups of 8: PPK = 4: 17.78 ms / step, 8: 16.74, 16: 16.49 -- a CTA's fixed cost (TMA
// window, modulation table, kernel values) is amortised over more outputs); ssq in float64: 4
// (C5: 22.80 -> 21.89 ms / 2 signals against 2)
template <typename T> constexpr int interp_ppk(bool ssq) {
  return sizeof(T) == 4 ? (ssq ? 16 : 4) : (ssq ? 4 : 2);
}

template <typename T, int NARR, bool SSQ>
static int launch_grid_interp_t(const GridArgs<T>& G, unsigned max_tiles, cudaStream_t st) {
  constexpr int K = GridTaps<T>::K, PPK = interp_ppk<T>(SSQ), PP = K * PPK;
  using V4 = typename V4T<T>::type;
  // coarse samples per CTA = (256 / min(U, 256)) * PP; U >= 16
  size_t smem = (size_t)(16 * PP + K - 1) * sizeof(V4) + (size_t)16 * PP * sizeof(cx<T>);
  auto kern = grid_interp_kernel<T, K, PPK, NARR, SSQ>;
  SSQB_CUDA(set_smem_limit(kern, smem));
  dim3 grid(max_tiles, (unsigned)(G.B * G.n_rows));
  kern<<<grid, 256, smem, st>>>(G);
  SSQB_LAUNCH_CHECK();
  return 0;
}
template <typename T>
static int launch_grid_interp(const GridArgs<T>& G, int narr, unsigned max_tiles, cudaStream_t st) {
  if (narr == 2 && G.ssq) return launch_grid_interp_t<T, 2, true>(G, max_tiles, st);
  if (narr == 2) return launch_grid_interp_t<T, 2, false>(G, max_tiles, st);
  return launch_grid_interp_t<T, 1, false>(G, max_tiles, st);
}


template <typename T>
struct CwtPlan : public CwtPlanBase {
  ssqb_cwt_desc d;
  int logn = 0, logF = 0, logI2 = 0, log_lo = 0;
  DevBuf<T> scales_d, out_mul_d;
  DevBuf<long long> band_lo_d, band_len_d;
  DevBuf<double> cst_d;
  DevBuf<cx<T>> tw1_d, tw2_d, tw_lo_d, tw_hi_d, xh_d, G_d;
  // host-buffer staging (exec_host)
  DevBuf<T> x_stage;
  DevBuf<cx<T>> Wx_stage, dWx_stage, Tx_stage;
  ReassignGrid grid;
  bool have_grid = false;
  // scratch of the two-pass route.  The path is issue-bound, not HBM-bound, so a
  // scratch larger than L2 (fewer, fuller launches) beats an L2-resident one.
  static constexpr size_t SCRATCH_BYTES = (size_t)512 << 20;
  // route switches, read from the environment once per plan (init): a route that is off leaves
  // its rows to the next one, which is how tests reach the direct, block and two-pass rows at
  // shapes where the default routes claim every row
  struct Routes {
    bool fast, grid, sblk, block;     // SSQB_NO_FAST / _NO_GRID / _NO_SBLK / _NO_BLOCK = 1: off
    int grid_max_logm;                // SSQB_GRID_MAX_LOGM: longest coarse grid (0: no cap)
  } routes{};
  // fast path (n_up >= 2^13, device-evaluated wavelets): band tables + row classes
  bool fast = false;
  DevBuf<long long> tab_off_d;
  DevBuf<T> tab_p_d, tab_pd_d;
  static constexpr int NCLS = 6;          // band <= 8, 64, 512, 1024, 2048, 4096 bins
  DevBuf<RowInfo> qrows_d[NCLS];
  int n_qrows[NCLS] = {0, 0, 0, 0, 0, 0};
  std::vector<int> big_scales;          // scale indices that need the two-pass route
  std::vector<int> big_scales_all;      // same, before rows moved to the block route
  DevBuf<int> bigmap_d;                 // (b*na + a) list for the current batch size
  long long bigmap_B = -1;
  // overlap-save block route (float32, compactly supported wavelets): class c uses
  // blocks of P = 2^logP samples with a halo of h2 samples on each side
  static constexpr int BLK_NCLS = 5;
  struct BlockClass {
    int logP = 13, h2 = 0, hop = 0, nblk = 0, log_lo = 7;
    DevBuf<RowInfo> rows[4];                  // Q <= 1, 2, 4, 8 on the block grid
    int n_rows[4] = {0, 0, 0, 0};
    DevBuf<long long> row_n1;                 // [B*nblk] per-block left pad for the loader
    long long row_n1_B = -1;
    DevBuf<cx<T>> Xb;                         // [B*nblk][P] block spectra / P
    DevBuf<long long> lo_d, len_d, off_d;     // per-scale band on the block grid
    DevBuf<T> p_d, pd_d;                      // psih / psih*xi/dt tables on that band
    DevBuf<cx<T>> tw1_d, twlo_d, twhi_d;      // roots for pass length P/512 and for P
    bool used() const { return n_rows[0] + n_rows[1] + n_rows[2] + n_rows[3] > 0; }
  };
  BlockClass blk[BLK_NCLS];
  bool have_blocks = false;
  // short-block rows (cwt_sblk.cuh): blocks of 2^SBLK_LOGP samples inside one CTA.
  // class 0: halo 256, class 1: halo 512 (float32 only), class 2: halo 256 on the analytic
  // part of the signal (rows cut at Nyquist)
  static constexpr int SBLK_LOGP = SblkGeom<T>::LOG_P;
  static constexpr int SBLK_NCLS = 3;
  struct SblkClass {
    int h2 = 0, hop = 0, nblk = 0;
    bool analytic = false;
    std::vector<SblkRow> rows;
    DevBuf<SblkRow> rows_d;
    DevBuf<cx<T>> Xs;                         // [B][nblk][P] block spectra / P
    DevBuf<T> p_d, pd_d;                      // [rows][P]
    bool used() const { return !rows.empty(); }
  };
  SblkClass sblk[SBLK_NCLS];
  bool have_sblk = false, have_cut = false;
  DevBuf<cx<T>> rootsP_d, twsP_d, xa_d, Gxa_d;
  DevBuf<T> ctab_d;
  DevBuf<long long> xa_lo_d, xa_len_d;
  // taper of the cut rows: erfc((xi - 3 pi / 2) / sigma) / 2, time kernel within +-taper_half
  static constexpr double SBLK_SIGMA = (sizeof(T) == 4) ? 0.374 : 0.262;
  static constexpr int SBLK_TAPER_HALF = (sizeof(T) == 4) ? 23 : 46;
  // gridded rows (cwt_grid.cuh): band of L bins -> coarse grid M = 2^logM >= 2(L+2), M <= n/32
  static constexpr int GRID_MIN_LOGM = 6;
  static constexpr int GRID_BASE_LOGM = (sizeof(T) == 4) ? 14 : 13;  // longest single-CTA transform
  static constexpr int GRID_MAX_LOGM = GRID_BASE_LOGM + 4;           // beyond it: R = 2..16 CTAs per transform
  std::vector<GridRow> grid_rows;              // sorted by logM
  int grid_cls_first[20], grid_cls_n[20];      // per logM: first row / count in grid_rows
  DevBuf<GridRow> grid_rows_d;
  DevBuf<T> gtab_p_d, gtab_pd_d, gcomp_d, htab_d;
  DevBuf<cx<T>> rootsM_d, rootsMh_d;
  DevBuf<typename V4T<T>::type> V_d;
  long long grid_v_total = 0;
  int grid_log_umax = 0;
  bool have_grid_rows = false;
  DevBuf<cx<T>> Gb_d;                         // scratch of the block forward FFTs (side stream)
  // side stream: the memset of Tx (pure HBM writes) overlaps the forward FFT and
  // pass 1 (which never touch Tx); joined before the first reassigning kernel
  cudaStream_t side = nullptr;
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  // worker lanes: the row kernels of one call are independent of each other (disjoint
  // rows, commutative atomics); spreading them over a few streams lets the partial last
  // wave of one launch be filled by the next (12 launches, ~9 % of a step in tails)
  static constexpr int NLANES = 3;
  cudaStream_t lanes[NLANES] = {nullptr, nullptr, nullptr};
  cudaEvent_t ev_lane_fork = nullptr, ev_lane_done[NLANES] = {nullptr, nullptr, nullptr};
  ~CwtPlan() {
    for (int i = 0; i < NLANES; ++i) {
      if (ev_lane_done[i]) cudaEventDestroy(ev_lane_done[i]);
      if (lanes[i]) cudaStreamDestroy(lanes[i]);
    }
    if (ev_lane_fork) cudaEventDestroy(ev_lane_fork);
    if (ev_fork) cudaEventDestroy(ev_fork);
    if (ev_join) cudaEventDestroy(ev_join);
    if (side) cudaStreamDestroy(side);
    for (int i = 0; i < 2; ++i) {
      if (ev_comp[i]) cudaEventDestroy(ev_comp[i]);
      if (ev_d2h[i]) cudaEventDestroy(ev_d2h[i]);
    }
    if (copy_st) cudaStreamDestroy(copy_st);
    if (ev_done) cudaEventDestroy(ev_done);
    for (int i = 0; i < 2; ++i) if (ev_sa[i]) cudaEventDestroy(ev_sa[i]);
  }
  // optional per-kernel timing (bench.py roofline): CUDA events on the launch stream
  bool profiling = false;
  std::vector<cudaEvent_t> ev;          // pairs (start, stop)
  std::vector<int> ev_kind;             // see SSQB_PROFILE_KINDS in ssq_b200.h
  std::vector<long long> ev_rows;

  int prof_begin(int kind, long long rows, cudaStream_t st) {
    if (!profiling) return 0;
    cudaEvent_t a, b;
    SSQB_CUDA(cudaEventCreate(&a)); SSQB_CUDA(cudaEventCreate(&b));
    ev.push_back(a); ev.push_back(b); ev_kind.push_back(kind); ev_rows.push_back(rows);
    SSQB_CUDA(cudaEventRecord(a, st));
    return 0;
  }
  int prof_end(cudaStream_t st) {
    if (!profiling) return 0;
    SSQB_CUDA(cudaEventRecord(ev.back(), st));
    return 0;
  }
  int set_profiling(int on) override {
    for (auto e : ev) cudaEventDestroy(e);
    ev.clear(); ev_kind.clear(); ev_rows.clear();
    profiling = on != 0;
    return 0;
  }
  int get_profile(double* ms, long long* launches, long long* rows) override {
    for (int k = 0; k < SSQB_PROFILE_KINDS; ++k) { ms[k] = 0; launches[k] = 0; rows[k] = 0; }
    for (size_t i = 0; i < ev_kind.size(); ++i) {
      float t = 0;
      SSQB_CUDA(cudaEventSynchronize(ev[2 * i + 1]));
      SSQB_CUDA(cudaEventElapsedTime(&t, ev[2 * i], ev[2 * i + 1]));
      ms[ev_kind[i]] += t; launches[ev_kind[i]] += 1; rows[ev_kind[i]] += ev_rows[i];
    }
    return 0;
  }

  int init(const ssqb_cwt_desc* desc) {
    d = *desc;
    logn = ilog2_exact(d.n_up);
    if (logn < 2 || logn > 21)
      return set_error(SSQB_E_UNSUPP, "n_up=%lld must be a power of two in [4, 2^21]",
                       (long long)d.n_up);
    if (d.N < 1 || d.n1 < 0 || d.n1 + d.N > d.n_up)
      return set_error(SSQB_E_ARG, "bad padding geometry N=%lld n1=%lld n_up=%lld",
                       (long long)d.N, (long long)d.n1, (long long)d.n_up);
    if (d.na < 1) return set_error(SSQB_E_ARG, "na must be >= 1");
    if (d.wavelet < 0 || d.wavelet > 2) return set_error(SSQB_E_ARG, "bad wavelet kind");
    if (d.wavelet == SSQB_WAV_TABLE && !d.psih_table_dev)
      return set_error(SSQB_E_ARG, "SSQB_WAV_TABLE needs psih_table_dev");
    if (logn >= 13) {
      logF = 9;                      // fast path geometry: F = 512, I2 = n/512 >= 16
    } else {
      logF = (logn + 1) / 2;
    }
    logI2 = logn - logF;
    if (logI2 < 1) { logI2 = 1; logF = logn - 1; }
    log_lo = (logn + 1) / 2;
    auto env = [](const char* name) { const char* e = getenv(name); return e ? atoi(e) : 0; };
    routes = Routes{!env("SSQB_NO_FAST"), !env("SSQB_NO_GRID"), !env("SSQB_NO_SBLK"),
                    !env("SSQB_NO_BLOCK"), env("SSQB_GRID_MAX_LOGM")};
    std::vector<T> sc((size_t)d.na);
    std::vector<long long> lo((size_t)d.na), len((size_t)d.na);
    for (int a = 0; a < d.na; ++a) {
      sc[a] = (T)d.scales_host[a];
      lo[a] = d.band_lo_host ? (long long)d.band_lo_host[a] : 0;
      len[a] = d.band_len_host ? (long long)d.band_len_host[a] : (long long)d.n_up;
      if (len[a] < 0 || len[a] > d.n_up) return set_error(SSQB_E_ARG, "bad band_len[%d]", a);
    }
    SSQB_CUDA(scales_d.upload(sc));
    SSQB_CUDA(band_lo_d.upload(lo));
    SSQB_CUDA(band_len_d.upload(len));
    long long n = d.n_up, F = 1ll << logF, I2 = 1ll << logI2;
    SSQB_CUDA(tw1_d.upload(make_roots<T>(I2, 1, I2)));
    SSQB_CUDA(tw2_d.upload(make_roots<T>(F, 1, F)));
    SSQB_CUDA(tw_lo_d.upload(make_roots<T>(1ll << log_lo, 1, n)));
    SSQB_CUDA(tw_hi_d.upload(make_roots<T>(n >> log_lo, 1ll << log_lo, n)));
    SSQB_CUDA(cudaStreamCreateWithFlags(&side, cudaStreamNonBlocking));
    SSQB_CUDA(cudaEventCreateWithFlags(&ev_fork, cudaEventDisableTiming));
    SSQB_CUDA(cudaEventCreateWithFlags(&ev_join, cudaEventDisableTiming));
    SSQB_CUDA(cudaEventCreateWithFlags(&ev_lane_fork, cudaEventDisableTiming));
    for (int i = 0; i < NLANES; ++i) {
      SSQB_CUDA(cudaStreamCreateWithFlags(&lanes[i], cudaStreamNonBlocking));
      SSQB_CUDA(cudaEventCreateWithFlags(&ev_lane_done[i], cudaEventDisableTiming));
    }
    return init_fast(lo, len);
  }

  int init_fast(const std::vector<long long>& lo, const std::vector<long long>& len) {
    fast = false; have_blocks = false;
    if (!routes.fast) return 0;
    if (logF != 9 || logI2 < 4 || d.wavelet == SSQB_WAV_TABLE) return 0;
    // float64 staging (32 B per band bin) + 128 KB of tiles must fit 227 KB: Q <= 4
    constexpr int qmax_direct = (sizeof(T) == 4) ? 8 : 4;
    const bool use_blocks = d.tsupport_host != nullptr && routes.block;
    // short blocks: the signal must be a few blocks long, and every halo must stay inside the
    // padding the reference adds (the block loader extends the signal by the padding rule)
    bool use_sblk = use_blocks && routes.sblk;
    if (logn < SBLK_LOGP + 2 || d.n1 < 512 || d.n_up - d.n1 - d.N < 512) use_sblk = false;
    for (int c = 0; c < SBLK_NCLS; ++c) sblk[c].rows.clear();
    have_sblk = false; have_cut = false;

    // ---- route every scale: block class / direct class / two-pass --------------------
    // block length 2^logP with a halo of h2 samples each side; the two long classes only
    // exist for n_up >= 2^19 / 2^20 (very long signals), where they spare rows the two-pass route
    const int logPs[BLK_NCLS] = {13, 13, 16, 18, 19};
    const int h2s[BLK_NCLS] = {256, 1024, 8192, 32768, 131072};
    std::vector<long long> off((size_t)d.na);
    long long total = 0, lmax = 1;
    std::vector<int> cls[NCLS];
    std::vector<RowInfo> blists[BLK_NCLS][4];
    std::vector<long long> blo[BLK_NCLS], blen[BLK_NCLS], boff[BLK_NCLS];
    long long btotal[BLK_NCLS] = {0, 0, 0, 0, 0};
    for (int c = 0; c < BLK_NCLS; ++c) {
      blo[c].assign((size_t)d.na, 0); blen[c].assign((size_t)d.na, 0); boff[c].assign((size_t)d.na, 0);
    }
    big_scales.clear(); big_scales_all.clear();
    std::vector<char> is_grid((size_t)d.na, 0);
    { int rc = init_grid(lo, len, is_grid); if (rc) return rc; }
    for (int a = 0; a < d.na; ++a) {
      off[a] = total; total += len[a];
      if (len[a] > lmax) lmax = len[a];
      if (is_grid[(size_t)a]) continue;              // decimate + interpolate route
      const long long q = (len[a] + 511) / 512;
      bool routed = false;
      if (use_sblk && q >= 2 && len[a] < d.n_up) {
        const long long S = d.tsupport_host[a];
        int sc = -1;
        if (S > 0 && S <= 512) sc = 0;
        else if (S > 512 && S <= 1024 && sizeof(T) == 4) sc = 1;
        else if (S < 0 && d.wavelet != SSQB_WAV_TABLE && lo[a] >= 0 &&
                 lo[a] + len[a] - 1 == d.n_up / 2 && (-S) + 2 * SBLK_TAPER_HALF <= 512) sc = 2;
        if (sc >= 0) {
          SblkRow r; r.a = a; r.cut = (sc == 2) ? 1 : 0;
          r.tab_off = (long long)sblk[sc].rows.size() << SBLK_LOGP;
          sblk[sc].rows.push_back(r);
          routed = true;
        }
      }
      if (!routed && use_blocks && q >= 2 && len[a] < d.n_up) {
        const long long S = d.tsupport_host[a];
        for (int c = 0; c < BLK_NCLS && !routed; ++c) {
          if (!(S > 0 && S <= 2 * h2s[c]) || logn <= logPs[c]) continue;
          const long long Pn = 1ll << logPs[c], ratio = d.n_up >> logPs[c];
          // signed band on the block grid (one-bin margin each side)
          long long slo = lo[a], shi = lo[a] + len[a] - 1;
          if (slo > d.n_up / 2) { slo -= d.n_up; shi -= d.n_up; }
          long long bl = (slo >= 0 ? slo / ratio : -((-slo + ratio - 1) / ratio)) - 1;
          long long bh = (shi >= 0 ? (shi + ratio - 1) / ratio : -((-shi) / ratio)) + 1;
          if (bl < -(Pn / 2 - 1)) bl = -(Pn / 2 - 1);
          if (bh > Pn / 2) bh = Pn / 2;
          const long long bn = bh - bl + 1, qb = (bn + 511) / 512;
          // worth it when the row is two-pass today, or when the block band needs
          // fewer terms than the whole-signal band
          // (block rows run the direct kernel: at most qmax_direct terms)
          if (bn <= 0 || qb > qmax_direct || !(q > qmax_direct || qb < q)) continue;
          blo[c][a] = bl; blen[c][a] = bn; boff[c][a] = btotal[c]; btotal[c] += bn;
          RowInfo ri; ri.a = a; ri.lo = (int)(bl & (Pn - 1)); ri.len = (int)bn; ri.pad = 0;
          ri.tab_off = boff[c][a]; ri.pad2 = 0;
          blists[c][qb <= 1 ? 0 : qb <= 2 ? 1 : qb <= 4 ? 2 : 3].push_back(ri);
          routed = true;
        }
      }
      if (routed) { big_scales_all.push_back(a); continue; }   // two-pass when blocks are off
      if (q > qmax_direct) { big_scales.push_back(a); big_scales_all.push_back(a); continue; }
      int c = q <= 1 ? 2 : q <= 2 ? 3 : q <= 4 ? 4 : 5;
      if (len[a] <= 8) c = 0; else if (len[a] <= 64) c = 1;
      cls[c].push_back(a);
    }
    SSQB_CUDA(tab_off_d.upload(off));
    SSQB_CUDA(tab_p_d.ensure((size_t)(total > 0 ? total : 1)));
    SSQB_CUDA(tab_pd_d.ensure((size_t)(total > 0 ? total : 1)));
    for (int c = 0; c < NCLS; ++c) {
      n_qrows[c] = (int)cls[c].size();
      if (!n_qrows[c]) continue;
      std::vector<RowInfo> ri(cls[c].size());
      for (size_t k = 0; k < cls[c].size(); ++k) {
        int a = cls[c][k];
        ri[k].a = a; ri[k].lo = (int)(lo[a] & (d.n_up - 1)); ri[k].len = (int)len[a];
        ri[k].pad = 0; ri[k].tab_off = off[a]; ri[k].pad2 = 0;
      }
      SSQB_CUDA(qrows_d[c].upload(ri));
    }
    CwtArgs<T> A; base_args(A);
    unsigned gx = (unsigned)((lmax + 255) / 256); if (gx > 1024) gx = 1024;
    psih_band_kernel<T><<<dim3(gx, (unsigned)d.na), 256>>>(A, tab_off_d.p, tab_p_d.p, tab_pd_d.p);
    SSQB_LAUNCH_CHECK();
    // ---- block classes: tables on the block grids ---------------------------------------
    for (int c = 0; c < BLK_NCLS; ++c) {
      BlockClass& K = blk[c];
      for (int k = 0; k < 4; ++k) K.n_rows[k] = (int)blists[c][k].size();
      if (!K.used()) continue;
      have_blocks = true;
      K.logP = logPs[c]; K.h2 = h2s[c]; K.hop = (1 << K.logP) - 2 * K.h2;
      K.nblk = (int)((d.N + K.hop - 1) / K.hop);
      K.log_lo = (K.logP + 1) / 2;
      for (int k = 0; k < 4; ++k)
        if (K.n_rows[k]) SSQB_CUDA(K.rows[k].upload(blists[c][k]));
      const long long Pn = 1ll << K.logP;
      SSQB_CUDA(K.lo_d.upload(blo[c])); SSQB_CUDA(K.len_d.upload(blen[c]));
      SSQB_CUDA(K.off_d.upload(boff[c]));
      SSQB_CUDA(K.p_d.ensure((size_t)btotal[c])); SSQB_CUDA(K.pd_d.ensure((size_t)btotal[c]));
      SSQB_CUDA(K.tw1_d.upload(make_roots<T>(Pn >> 9, 1, Pn >> 9)));
      SSQB_CUDA(K.twlo_d.upload(make_roots<T>(1ll << K.log_lo, 1, Pn)));
      SSQB_CUDA(K.twhi_d.upload(make_roots<T>(Pn >> K.log_lo, 1ll << K.log_lo, Pn)));
      CwtArgs<T> Ab; block_args(Ab, K);
      psih_band_kernel<T><<<dim3(64, (unsigned)d.na), 256>>>(Ab, K.off_d.p, K.p_d.p, K.pd_d.p);
      SSQB_LAUNCH_CHECK();
    }
    { int rc = init_sblk(); if (rc) return rc; }
    SSQB_CUDA(cudaDeviceSynchronize());
    fast = true;
    bigmap_B = -1;
    return 0;
  }

  // tables of the short-block classes (rows were chosen by init_fast)
  int init_sblk() {
    constexpr long long Pn = 1ll << SBLK_LOGP;
    static const int h2s[SBLK_NCLS] = {256, 512, 256};
    for (int c = 0; c < SBLK_NCLS; ++c) {
      SblkClass& K = sblk[c];
      if (!K.used()) continue;
      have_sblk = true; have_blocks = true;
      K.h2 = h2s[c]; K.hop = (int)Pn - 2 * K.h2; K.analytic = (c == 2);
      K.nblk = (int)((d.N + K.hop - 1) / K.hop);
      if (K.analytic) have_cut = true;
      SSQB_CUDA(K.rows_d.upload(K.rows));
      SSQB_CUDA(K.p_d.ensure(K.rows.size() * (size_t)Pn));
      SSQB_CUDA(K.pd_d.ensure(K.rows.size() * (size_t)Pn));
    }
    if (!have_sblk) return 0;
    SSQB_CUDA(rootsP_d.upload(make_roots<T>(Pn, 1, Pn)));
    {
      // per-stage twiddles of sblk_rows_kernel: stage Ns (radix r) at Ns - 8, [q - 1][k]
      std::vector<cx<T>> tws((size_t)Pn, mkc<T>((T)1, (T)0));
      auto fill = [&](long long Ns, int r) {
        const long long tstep = Pn / (Ns * r);
        for (int q = 1; q < r; ++q)
          for (long long k = 0; k < Ns; ++k) {
            const double ang = 2.0 * M_PI * (double)((k * q * tstep) % Pn) / (double)Pn;
            tws[(size_t)(Ns - 8 + (q - 1) * Ns + k)] = mkc<T>((T)cos(ang), (T)sin(ang));
          }
      };
      long long Ns = 8;
      for (; Ns * 8 <= Pn; Ns *= 8) fill(Ns, 8);
      if (Ns * 4 == Pn) fill(Ns, 4);
      SSQB_CUDA(twsP_d.upload(tws));
    }
    for (int c = 0; c < SBLK_NCLS; ++c) {
      SblkClass& K = sblk[c];
      if (!K.used()) continue;
      SblkArgs<T> S; memset(&S, 0, sizeof(S));
      base_args(S.A);
      S.rows = K.rows_d.p; S.n_rows = (int)K.rows.size(); S.sigma = (T)SBLK_SIGMA;
      sblk_tab_kernel<T, SBLK_LOGP><<<dim3((unsigned)(Pn / 256), (unsigned)K.rows.size()), 256>>>(
          S, K.p_d.p, K.pd_d.p);
      SSQB_LAUNCH_CHECK();
    }
    if (have_cut) {
      // c[k] of the analytic part: 1 below Nyquist, 1/2 at Nyquist, 0 above
      std::vector<T> ct((size_t)d.n_up, (T)0);
      for (long long k = 0; k < d.n_up / 2; ++k) ct[(size_t)k] = (T)1;
      ct[(size_t)(d.n_up / 2)] = (T)0.5;
      SSQB_CUDA(ctab_d.upload(ct));
      std::vector<long long> l0(1, 0), l1(1, d.n_up / 2 + 1);
      SSQB_CUDA(xa_lo_d.upload(l0)); SSQB_CUDA(xa_len_d.upload(l1));
    }
    return 0;
  }

  void sblk_args(SblkArgs<T>& S, const SblkClass& K, long long B) {
    memset(&S, 0, sizeof(S));
    base_args(S.A);
    S.rows = K.rows_d.p; S.n_rows = (int)K.rows.size(); S.B = B;
    S.Xs = K.Xs.p; S.Xs_out = K.Xs.p; S.tab_p = K.p_d.p; S.tab_pd = K.pd_d.p;
    S.rootsP = rootsP_d.p; S.twsP = twsP_d.p; S.nblk = K.nblk; S.hop = K.hop; S.h2 = K.h2;
    S.sigma = (T)SBLK_SIGMA;
  }
  // spectra of the blocks of class K: from x (padding rule applied on the fly) or from xa
  int sblk_forward(SblkClass& K, const T* x, long long B, cudaStream_t s) {
    SSQB_CUDA(K.Xs.ensure((size_t)B * (size_t)K.nblk << SBLK_LOGP));
    SblkArgs<T> S; sblk_args(S, K, B);
    S.x = x; S.xa = K.analytic ? xa_d.p : nullptr;
    return launch_sblk_fwd<T>(S, s);
  }
  // xa = ifft(xh * c): the part of the padded signal the Nyquist-cut rows see
  // (its own scratch: it runs on a worker lane next to the two-pass rows)
  int analytic(long long B, cudaStream_t st) {
    SSQB_CUDA(xa_d.ensure((size_t)B * (size_t)d.n_up));
    long long chunk = rows_per_chunk(1, B);
    SSQB_CUDA(Gxa_d.ensure((size_t)arr_stride(chunk)));
    for (long long b0 = 0; b0 < B; b0 += chunk) {
      long long nb = (B - b0 < chunk) ? (B - b0) : chunk;
      CwtArgs<T> A; base_args(A);
      A.na = 1; A.row0 = (int)b0; A.nrows = (int)nb;
      A.wavelet = WAV_TABLE; A.psih_table = ctab_d.p;
      A.band_lo = xa_lo_d.p; A.band_len = xa_len_d.p;
      A.xh = xh_d.p; A.G = Gxa_d.p; A.G_arr_stride = arr_stride(nb);
      A.Wx = xa_d.p; A.dWx = nullptr; A.Tx = nullptr;
      A.Nout = d.n_up; A.out_off = 0; A.out_mul = nullptr;
      int rc = prof_begin(0, nb, st); if (rc) return rc;
      rc = launch_pass1<T, MODE_CWT>(A, 1, st); if (rc) return rc;
      rc = launch_pass2<T, 1, EPI_CWT>(A, 0, st); if (rc) return rc;
      rc = prof_end(st); if (rc) return rc;
    }
    return 0;
  }


  // rows whose band fits a coarse grid of M <= min(2^GRID_MAX_LOGM, n/32) points with
  // oversampling >= 2 take the gridded route (cwt_grid.cuh)
  int init_grid(const std::vector<long long>& lo, const std::vector<long long>& len,
                std::vector<char>& is_grid) {
    have_grid_rows = false; grid_rows.clear(); grid_v_total = 0;
    for (int l = 0; l < 20; ++l) { grid_cls_first[l] = 0; grid_cls_n[l] = 0; }
    if (!routes.grid || logn < 13) return 0;
    int max_logm = GRID_MAX_LOGM;
    if (max_logm > logn - 4) max_logm = logn - 4;          // U = n/M >= 16
    const int v = routes.grid_max_logm;
    if (v >= GRID_MIN_LOGM && v < max_logm) max_logm = v;
    std::vector<GridRow> rows;
    for (int a = 0; a < d.na; ++a) {
      const long long L = len[a];
      if (L < 1 || L >= d.n_up / 4) continue;
      int lm = GRID_MIN_LOGM;
      while ((1ll << lm) < 2 * (L + 2)) ++lm;
      if (lm > max_logm) continue;
      GridRow r{}; r.a = a; r.logM = lm; r.len = (int)L;
      r.lo = (int)(lo[a] & (d.n_up - 1));
      r.c = (int)((lo[a] + (L >> 1)) & (d.n_up - 1));
      r.tab_off = 0; r.v_off = 0;
      rows.push_back(r);
      is_grid[(size_t)a] = 1;
    }
    if (rows.empty()) return 0;
    std::stable_sort(rows.begin(), rows.end(),
                     [](const GridRow& x, const GridRow& y) { return x.logM < y.logM; });
    long long ttot = 0, vtot = 0;
    for (size_t k = 0; k < rows.size(); ++k) {
      GridRow& r = rows[k];
      if (grid_cls_n[r.logM] == 0) grid_cls_first[r.logM] = (int)k;
      ++grid_cls_n[r.logM];
      r.tab_off = ttot; ttot += r.len;
      r.v_off = vtot; vtot += 1ll << r.logM;
    }
    grid_rows = rows; grid_v_total = vtot;
    SSQB_CUDA(grid_rows_d.upload(rows));
    { int rc = init_grid_tables(); if (rc) return rc; }
    SSQB_CUDA(gtab_p_d.ensure((size_t)ttot));
    SSQB_CUDA(gtab_pd_d.ensure((size_t)ttot));
    CwtArgs<T> A; base_args(A);
    psih_grid_kernel<T><<<dim3(16, (unsigned)rows.size()), 256>>>(A, grid_rows_d.p, gcomp_d.p,
                                                                 gtab_p_d.p, gtab_pd_d.p);
    SSQB_LAUNCH_CHECK();
    have_grid_rows = true;
    return 0;
  }


  // kernel tables of the gridded / block routes, float64 on the host: 1/phi_hat per coarse
  // length, phi per fine phase, roots of unity
  bool grid_tables_ready = false;
  int init_grid_tables() {
    if (grid_tables_ready) return 0;
    constexpr int K = GridTaps<T>::K;
    const double beta = 2.30 * K;
    std::vector<double> gx, gw; gauss_legendre(96, gx, gw);
    const int top = GRID_MAX_LOGM < logn - 4 ? GRID_MAX_LOGM : logn - 4;
    std::vector<T> comp((size_t)(1ll << (top + 1)), (T)0);
    for (int lm = GRID_MIN_LOGM; lm <= top; ++lm) {
      const long long M = 1ll << lm;
      for (long long m = -M / 2; m < M / 2; ++m) {
        // only |m| <= M/4 + 1 is ever used; beyond it phi_hat is tiny
        double v = (llabs(m) <= M / 4 + 2) ? 1.0 / grid_phi_hat((double)m / (double)M, K, beta, gx, gw) : 0.0;
        comp[(size_t)((M - 64) + M / 2 + m)] = (T)v;
      }
    }
    SSQB_CUDA(gcomp_d.upload(comp));
    grid_log_umax = logn - GRID_MIN_LOGM;
    const long long UMAX = 1ll << grid_log_umax;
    std::vector<T> ht((size_t)UMAX * K);
    for (long long u = 0; u < UMAX; ++u)
      for (int k = 0; k < K; ++k)
        ht[(size_t)u * K + k] = (T)grid_phi((double)u / (double)UMAX - (double)k + 0.5 * K - 1.0, K, beta);
    SSQB_CUDA(htab_d.upload(ht));
    SSQB_CUDA(rootsM_d.upload(make_roots<T>(1ll << GRID_BASE_LOGM, 1, 1ll << GRID_BASE_LOGM)));
    SSQB_CUDA(rootsMh_d.upload(make_roots<T>(1ll << (GRID_BASE_LOGM - 1), 1, 1ll << (GRID_BASE_LOGM - 1))));
    grid_tables_ready = true;
    return 0;
  }

  // forward FFTs of the overlap-save blocks of class K (side stream)
  int block_forward(BlockClass& K, const T* x, long long B, cudaStream_t s) {
    const long long vrows = B * K.nblk, Pn = 1ll << K.logP;
    if (K.row_n1_B != B) {
      std::vector<long long> rn((size_t)vrows);
      for (long long b = 0; b < B; ++b)
        for (int k = 0; k < K.nblk; ++k)
          rn[(size_t)(b * K.nblk + k)] = (long long)K.h2 - (long long)k * K.hop;
      SSQB_CUDA(K.row_n1.upload(rn));
      K.row_n1_B = B;
    }
    SSQB_CUDA(K.Xb.ensure((size_t)vrows * (size_t)Pn));
    CwtArgs<T> A; block_args(A, K);
    A.na = 1; A.row0 = 0; A.nrows = (int)vrows;
    A.x = x; A.row_n1 = K.row_n1.p; A.x_row_div = K.nblk;
    A.xh_out = K.Xb.p; A.G = Gb_d.p; A.G_arr_stride = vrows * Pn;
    int rc = launch_pass1<T, MODE_X>(A, 1, s); if (rc) return rc;
    return launch_pass2<T, 1, EPI_FWD>(A, 0, s);
  }

  // gridded rows: stage (A) needs xh only; stage (B) also the zeroed Tx (when ssq)
  void grid_args(GridArgs<T>& G, long long B, cx<T>* Wx, cx<T>* dWx, cx<T>* Tx, bool ssq,
                 const T* out_mul, bool rpadded, long long Nout) {
    memset(&G, 0, sizeof(G));
    base_args(G.A);
    G.A.xh = xh_d.p; G.A.Wx = Wx; G.A.dWx = dWx; G.A.Tx = Tx;
    G.A.Nout = Nout; G.A.out_off = rpadded ? 0 : d.n1; G.A.out_mul = out_mul;
    G.rows = grid_rows_d.p; G.n_rows = (int)grid_rows.size(); G.B = B;
    G.V = V_d.p; G.v_total = grid_v_total;
    G.gtab_p = gtab_p_d.p; G.gtab_pd = gtab_pd_d.p;
    G.rootsM = rootsM_d.p; G.rootsMh = rootsMh_d.p; G.log_mmax = GRID_BASE_LOGM;
    G.htab = htab_d.p; G.log_umax = grid_log_umax;
    G.write_dWx = dWx ? 1 : 0; G.ssq = ssq ? 1 : 0;
    G.t0 = rpadded ? 0 : (int)d.n1; G.tcount = (int)Nout;
  }
  // coarse-grid inverse FFTs: the two long classes (2^13, 2^12 points: a few CTAs each) and the
  // merged launch of all shorter ones go to three streams so that their latencies overlap
  cudaEvent_t ev_sa[2] = {nullptr, nullptr};
  int grid_stage_a(const GridArgs<T>& G, long long B, cudaStream_t st, cudaStream_t s1,
                   cudaStream_t s2) {
    int rc = prof_begin(3, B * (long long)grid_rows.size(), st); if (rc) return rc;
    cudaStream_t order[3] = {st, s1, s2};
    int slot = 0;
    bool used[3] = {false, false, false};
    for (int lm = GRID_MAX_LOGM; lm >= 12; --lm) {             // long transforms first
      if (!grid_cls_n[lm]) continue;
      rc = launch_grid_dec<T>(G, lm, grid_rows_d.p + grid_cls_first[lm], grid_cls_n[lm], order[slot]);
      if (rc) return rc;
      used[slot] = true; slot = (slot + 1) % 3;
    }
    {
      DecSmallPlan P; int acc = 0;
      for (int c = 0; c < 6; ++c) {
        const int lm = 6 + c, R = 2048 >> lm;
        P.cta_start[c] = acc; P.row_first[c] = grid_cls_first[lm]; P.n_cls[c] = grid_cls_n[lm];
        acc += (int)(((long long)grid_cls_n[lm] * B + R - 1) / R);
      }
      P.cta_start[6] = acc;
      rc = launch_grid_dec_small<T>(G, P, order[slot]); if (rc) return rc;
      used[slot] = true;
    }
    for (int i = 1; i < 3; ++i)
      if (used[i] && order[i] != st) {
        if (!ev_sa[i - 1]) SSQB_CUDA(cudaEventCreateWithFlags(&ev_sa[i - 1], cudaEventDisableTiming));
        SSQB_CUDA(cudaEventRecord(ev_sa[i - 1], order[i]));
        SSQB_CUDA(cudaStreamWaitEvent(st, ev_sa[i - 1], 0));
      }
    return prof_end(st);
  }
  int grid_stage_b(const GridArgs<T>& G, long long B, int narr, cudaStream_t st) {
    const int PP = GridTaps<T>::K * interp_ppk<T>(G.ssq != 0);
    unsigned max_tiles = 1;                               // tiles of the widest row class
    for (int lm = GRID_MIN_LOGM; lm <= GRID_MAX_LOGM; ++lm) {
      if (!grid_cls_n[lm]) continue;
      const int logU = logn - lm, logUT = logU < 8 ? logU : 8;
      const long long n_ut = 1ll << (logU - logUT), ptile = (256ll >> logUT) * PP;
      const long long p_first = (long long)G.t0 >> logU, p_last = ((long long)G.t0 + G.tcount - 1) >> logU;
      const long long n_pt = (p_last - p_first + ptile) / ptile;
      if ((unsigned)(n_ut * n_pt) > max_tiles) max_tiles = (unsigned)(n_ut * n_pt);
    }
    int rc = prof_begin(4, B * (long long)grid_rows.size(), st); if (rc) return rc;
    rc = launch_grid_interp<T>(G, narr, max_tiles, st); if (rc) return rc;
    return prof_end(st);
  }

  // CwtArgs describing ONE block of class K as a length-P signal transform
  void block_args(CwtArgs<T>& A, const BlockClass& K) {
    base_args(A);
    A.n_up = 1ll << K.logP; A.logn = K.logP; A.logF = 9; A.logI2 = K.logP - 9;
    A.n1 = 0;
    A.band_lo = K.lo_d.p; A.band_len = K.len_d.p;
    A.tw1 = K.tw1_d.p; A.tw_lo = K.twlo_d.p; A.tw_hi = K.twhi_d.p;
    A.log_lo = K.log_lo;
  }

  void base_args(CwtArgs<T>& A) {
    memset(&A, 0, sizeof(A));
    A.N = d.N; A.n_up = d.n_up; A.n1 = d.n1;
    A.logn = logn; A.logF = logF; A.logI2 = logI2;
    A.padtype = d.padtype; A.na = d.na;
    A.scales = scales_d.p; A.band_lo = band_lo_d.p; A.band_len = band_len_d.p;
    A.psih_table = (const T*)d.psih_table_dev;
    A.wavelet = d.wavelet;
    if (d.wavelet == SSQB_WAV_MORLET) {
      // constants cast to dtype exactly as wavelets.py:510-516
      double mu = d.wparams[0];
      double cs = pow(1 + exp(-mu * mu) - 2 * exp(-0.75 * mu * mu), -0.5);
      double ks = exp(-0.5 * mu * mu);
      A.wp[0] = (T)mu; A.wp[1] = (T)ks; A.wp[2] = (T)-0.5;
      A.wp[3] = (T)(sqrt(2.0) * cs * pow(M_PI, 0.25));
    } else if (d.wavelet == SSQB_WAV_GMW_L1) {
      // _gmw.py:191-198: gamma, beta, wc, wcl cast to dtype; k0 = -beta*wcl + wc**gamma
      double gam = d.wparams[0], bet = d.wparams[1];
      double wc = exp((1.0 / gam) * (log(bet) - log(gam)));
      T gT = (T)gam, bT = (T)bet, wcT = (T)wc, wclT = (T)log(wc);
      T wcg = (T)pow((double)wcT, (double)gT);         // wc**gamma rounded to dtype
      A.wp[0] = gT; A.wp[1] = bT; A.wp[2] = (T)(-(bT * wclT)) + wcg;
    }
    A.dt = (T)d.dt;
    A.tw1 = tw1_d.p; A.tw2 = tw2_d.p; A.tw_lo = tw_lo_d.p; A.tw_hi = tw_hi_d.p;
    A.log_lo = log_lo;
    A.cst = cst_d.p;
    if (have_grid) A.grid = grid;
    A.zero_next = zero_next_; A.zero_off = zero_off_;
  }

  int set_reassign(const ssqb_reassign_desc* r) override {
    int rc = fill_grid(r, d.na, &grid);
    if (rc) return rc;
    std::vector<double> c(r->cst_host, r->cst_host + d.na);
    SSQB_CUDA(cst_d.upload(c));
    have_grid = true;
    return 0;
  }

  // rows of G that fit the scratch budget
  long long rows_per_chunk(int narr, long long total_rows) {
    size_t per_row = (size_t)narr * (size_t)d.n_up * sizeof(cx<T>);
    long long r = (long long)(SCRATCH_BYTES / per_row);
    if (r < 1) r = 1;
    if (r > total_rows) r = total_rows;
    return r;
  }
  cudaError_t ensure_scratch(int narr, long long rows) {
    long long E = fast ? (1ll << ROWS_LOGE) : (long long)Tile<T>::ELEMS;
    long long R2 = E >> logF;
    long long ncols = rows << logI2;
    long long tiles = (ncols + R2 - 1) / R2;
    return G_d.ensure((size_t)narr * (size_t)tiles * (size_t)E);
  }
  long long arr_stride(long long rows) {
    long long E = fast ? (1ll << ROWS_LOGE) : (long long)Tile<T>::ELEMS;
    long long R2 = E >> logF;
    long long ncols = rows << logI2;
    return ((ncols + R2 - 1) / R2) * E;
  }

  int forward(const T* x, long long B, cx<T>* xh, cudaStream_t st) {
    long long chunk = rows_per_chunk(1, B);
    SSQB_CUDA(ensure_scratch(1, chunk));
    for (long long b0 = 0; b0 < B; b0 += chunk) {
      long long nb = (B - b0 < chunk) ? (B - b0) : chunk;
      CwtArgs<T> A; base_args(A);
      A.na = 1; A.row0 = (int)b0; A.nrows = (int)nb;
      A.x = x; A.xh_out = xh; A.G = G_d.p; A.G_arr_stride = arr_stride(nb);
      int rc = prof_begin(0, nb, st); if (rc) return rc;
      rc = launch_pass1<T, MODE_X>(A, 1, st); if (rc) return rc;
      rc = launch_pass2<T, 1, EPI_FWD>(A, 0, st); if (rc) return rc;
      rc = prof_end(st); if (rc) return rc;
    }
    return 0;
  }

  // Calls on one plan share its scratch, tables and worker streams, so consecutive calls are
  // ordered on the device whatever streams they arrive on: each call first waits for the
  // completion event of the previous one (a no-op when both use the same stream).  If a call
  // fails half-way, the side / lane streams are still joined into the caller's stream.
  cudaEvent_t ev_done = nullptr;
  bool ev_done_valid = false;
  long long maps_B = -1;                   // batch size the per-batch row maps were built for
  // zero-ahead state of the group being launched (see CwtArgs::zero_next)
  int zero_next_ = 0;
  long long zero_off_ = 0;
  bool zero_self_ = true;

  // Signals per group of a batched ssq call.  The zero fill of Tx is pure HBM writes while the row
  // kernels are issue-bound, but as a kernel of its own it runs before them; in groups, the row
  // kernels of group g zero the Tx of group g+1 alongside their Wx stores (same threads, same
  // addresses + a constant), and only group 0 is zeroed by zero_fill_kernel.  The group size
  // divides B (the per-batch row maps are built once): SSQB_GROUP=<signals>, 0 = no grouping.
  long long group_size(long long B, bool ssq, bool rpadded) const {
    if (!ssq || rpadded || B < 2) return B;
    long long env = -1;
    if (const char* e = getenv("SSQB_GROUP")) env = atoll(e);       // read per call (tests toggle it)
    if (env == 0) return B;
    long long target, smin = 1;
    if (env > 0) target = env;
    else {
      // measured on B200 (GMW, 300 scales, N = 160 000): B = 64: one group 21.0 ms, groups of
      // 16 / 8 / 4 / 2: 19.3 / 19.0 / 19.1 / 20.3 ms; B = 8: 2.72 ms, groups of 4 / 2 / 1: 2.57 / 2.62 / 3.00
      target = (B >= 32) ? 8 : B / 2;
      // a group must stream enough output to amortise its own launches and tails (>= 128 MB of Tx)
      const double plane = (double)d.na * (double)d.N * (double)sizeof(cx<T>);
      smin = (long long)ceil(128.0 * 1048576.0 / plane);
      if (target < smin) target = smin;
    }
    if (target >= B) return B;
    long long S = target;
    while (S > 1 && B % S) --S;
    if (S < smin) return B;
    return S;
  }

  int exec(const void* xv, long long B, void* Wxv, void* dWxv, void* Txv, bool ssq,
           const double* out_mul_host, bool rpadded, cudaStream_t st) override {
    if (!ev_done) SSQB_CUDA(cudaEventCreateWithFlags(&ev_done, cudaEventDisableTiming));
    if (ev_done_valid) SSQB_CUDA(cudaStreamWaitEvent(st, ev_done, 0));
    const long long S = (B >= 1) ? group_size(B, ssq, rpadded) : B;
    if (maps_B != S) {
      // the row maps are re-uploaded with blocking copies when the batch size changes:
      // nothing of an earlier call may still be reading them
      if (maps_B >= 0) SSQB_CUDA(cudaDeviceSynchronize());
      maps_B = S;
    }
    int rc = 0;
    if (S >= B || S < 1) {
      zero_next_ = 0; zero_off_ = 0; zero_self_ = true;
      rc = exec_body(xv, B, Wxv, dWxv, Txv, ssq, out_mul_host, rpadded, st);
    } else {
      const size_t plane = (size_t)d.na * (size_t)d.N;            // ssq: outputs are unpadded
      for (long long b0 = 0; b0 < B && rc == 0; b0 += S) {
        zero_self_ = (b0 == 0);
        zero_next_ = (b0 + S < B) ? (int)S : 0;
        zero_off_ = (long long)((size_t)S * plane);
        rc = exec_body((const T*)xv + (size_t)b0 * (size_t)d.N, S,
                       (cx<T>*)Wxv + (size_t)b0 * plane,
                       dWxv ? (cx<T>*)dWxv + (size_t)b0 * plane : nullptr,
                       (cx<T>*)Txv + (size_t)b0 * plane, ssq, out_mul_host, rpadded, st);
      }
      zero_next_ = 0; zero_off_ = 0; zero_self_ = true;
    }
    if (rc != 0) {                          // error path: leave no stream dangling
      cudaGetLastError();
      cudaEvent_t e;
      if (cudaEventCreateWithFlags(&e, cudaEventDisableTiming) == cudaSuccess) {
        cudaStream_t others[1 + NLANES] = {side, lanes[0], lanes[1], lanes[2]};
        for (cudaStream_t o : others)
          if (o) { cudaEventRecord(e, o); cudaStreamWaitEvent(st, e, 0); }
        cudaEventDestroy(e);
      }
    }
    cudaEventRecord(ev_done, st);
    ev_done_valid = true;
    return rc;
  }

  int exec_body(const void* xv, long long B, void* Wxv, void* dWxv, void* Txv, bool ssq,
                const double* out_mul_host, bool rpadded, cudaStream_t st) {
    if (B < 1) return set_error(SSQB_E_ARG, "B must be >= 1");
    if (!xv || !Wxv) return set_error(SSQB_E_ARG, "null x / Wx");
    if (ssq && (!Txv || !have_grid))
      return set_error(SSQB_E_ARG, "ssq needs Tx and ssqb_cwt_plan_set_reassign()");
    if (ssq && rpadded) return set_error(SSQB_E_ARG, "ssq works on the unpadded part");
    const T* x = (const T*)xv;
    cx<T>* Wx = (cx<T>*)Wxv; cx<T>* dWx = (cx<T>*)dWxv; cx<T>* Tx = (cx<T>*)Txv;
    long long total_rows = B * d.na;
    if (total_rows > 0x7fffffffll) return set_error(SSQB_E_UNSUPP, "too many rows");
    long long Nout = rpadded ? d.n_up : d.N;
    const bool use_blocks = fast && have_blocks && !rpadded;
    bool need_join = false;
    int rc = 0;
    if (ssq || use_blocks) {
      // side stream: zero Tx and transform the overlap-save blocks, concurrently with
      // everything on the main stream that needs neither (forward FFT, pass 1)
      SSQB_CUDA(cudaEventRecord(ev_fork, st));
      SSQB_CUDA(cudaStreamWaitEvent(side, ev_fork, 0));
      if (ssq && zero_self_) {                // later groups were zeroed by the previous group's kernels
        const size_t bytes = (size_t)total_rows * (size_t)Nout * sizeof(cx<T>);   // multiple of 8
        const size_t n16 = bytes / 16;
        int dev = 0, sms = 0;                  // at most 16 CTAs per SM of the current device
        SSQB_CUDA(cudaGetDevice(&dev));
        SSQB_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
        size_t nb = (n16 + 255) / 256; if (nb > (size_t)sms * 16) nb = (size_t)sms * 16; if (nb < 1) nb = 1;
        zero_fill_kernel<<<(unsigned)nb, 256, 0, side>>>(reinterpret_cast<uint4*>(Tx), n16,
                                                        reinterpret_cast<unsigned char*>(Tx) + n16 * 16,
                                                        (int)(bytes - n16 * 16));
        SSQB_LAUNCH_CHECK();
      }
      if (use_blocks) {
        long long gmax = 0;
        for (int c = 0; c < BLK_NCLS; ++c)
          if (blk[c].used() && B * blk[c].nblk * (1ll << blk[c].logP) > gmax)
            gmax = B * blk[c].nblk * (1ll << blk[c].logP);
        SSQB_CUDA(Gb_d.ensure((size_t)gmax + 8192));        // + one pass-2 tile (odd block counts)
        for (int c = 0; c < BLK_NCLS; ++c) {
          BlockClass& K = blk[c];
          if (!K.used()) continue;
          rc = block_forward(K, x, B, side); if (rc) return rc;
        }
        for (int c = 0; c < SBLK_NCLS; ++c)
          if (sblk[c].used() && !sblk[c].analytic) { rc = sblk_forward(sblk[c], x, B, side); if (rc) return rc; }
      }
      SSQB_CUDA(cudaEventRecord(ev_join, side));
      need_join = true;
    }
    SSQB_CUDA(xh_d.ensure((size_t)B * (size_t)d.n_up));

    const T* out_mul = nullptr;
    if (out_mul_host) {
      std::vector<T> m((size_t)d.na);
      for (int a = 0; a < d.na; ++a) m[a] = (T)out_mul_host[a];
      SSQB_CUDA(out_mul_d.ensure((size_t)d.na));
      SSQB_CUDA(cudaMemcpyAsync(out_mul_d.p, m.data(), m.size() * sizeof(T),
                                cudaMemcpyHostToDevice, st));
      SSQB_CUDA(cudaStreamSynchronize(st));   // `m` is a local
      out_mul = out_mul_d.p;
    }
    int narr = (ssq || dWx) ? 2 : 1;

    // ---- streams of this call: 0 = the caller's stream, 1.. = worker lanes ---------------
    // Every row kernel is independent of the others; what a kernel needs is
    //   * the spectrum xh (forward FFT, main stream)         -> direct and two-pass rows
    //   * the block spectra + zeroed Tx (side stream, ev_join) -> block rows / any ssq row
    // so block rows can run under the forward FFT and pass 1, which leave most SMs idle.
    const bool lanes_on = !profiling && fast;
    const bool side_used = need_join;
    bool lane_used[NLANES] = {false, false, false};
    bool got_join[NLANES + 1] = {false, false, false, false};
    bool got_fwd[NLANES + 1] = {true, false, false, false};
    double load[NLANES + 1] = {0, 0, 0, 0};
    // need_join: the work reads the block spectra or writes Tx (zeroed on the side stream)
    auto acquire = [&](int k, bool need_xh, bool need_join = true) -> cudaStream_t {
      cudaStream_t s = (k == 0) ? st : lanes[k - 1];
      if (k > 0) lane_used[k - 1] = true;
      if (need_join && side_used && !got_join[k]) { cudaStreamWaitEvent(s, ev_join, 0); got_join[k] = true; }
      if ((need_xh || !side_used) && !got_fwd[k]) {
        cudaStreamWaitEvent(s, ev_lane_fork, 0); got_fwd[k] = true;
      }
      return s;
    };
    auto least_loaded = [&](int first) -> int {
      int k = first;
      for (int i = first + 1; i <= (lanes_on ? NLANES : 0); ++i) if (load[i] < load[k]) k = i;
      return k;
    };
    struct Job { double w; FastArgs<T> P; int cls; long long gb; long long rows; int sblk_cls; };
    auto run_jobs = [&](std::vector<Job>& jobs, bool need_xh, int first) -> int {
      std::sort(jobs.begin(), jobs.end(), [](const Job& a, const Job& b) { return a.w > b.w; });
      for (const Job& J : jobs) {
        const int k = lanes_on ? least_loaded(first) : 0;
        load[k] += J.w;
        cudaStream_t ls = acquire(k, need_xh);
        int r2 = 0;
        if (J.sblk_cls >= 0 && sblk[J.sblk_cls].analytic) {     // xa and its block spectra, same lane
          r2 = analytic(B, ls); if (r2) return r2;
          r2 = sblk_forward(sblk[J.sblk_cls], x, B, ls); if (r2) return r2;
        }
        r2 = prof_begin(2, J.rows, ls); if (r2) return r2;
        if (J.sblk_cls >= 0) {
          SblkArgs<T> S; sblk_args(S, sblk[J.sblk_cls], B);
          S.A.Wx = Wx; S.A.dWx = dWx; S.A.Tx = Tx; S.A.Nout = Nout; S.A.out_mul = out_mul;
          S.write_dWx = dWx ? 1 : 0;
          r2 = launch_sblk_rows<T>(S, narr, ssq, ls);
        } else {
          r2 = launch_direct<T>(J.P, J.cls, narr, J.gb, ls);
        }
        if (r2) return r2;
        r2 = prof_end(ls); if (r2) return r2;
      }
      return 0;
    };
    static const double qw[4] = {1.0, 1.25, 1.6, 2.2};

    // (c) compact-wavelet rows: overlap-save blocks, single pass each.  With lanes they
    // are queued first (they do not wait for the forward FFT of the whole signal).
    std::vector<Job> bjobs;
    if (use_blocks) {
      for (int c = 0; c < BLK_NCLS; ++c) {
        BlockClass& K = blk[c];
        if (!K.used()) continue;
        const long long vrows = B * K.nblk;
        const double frac = (double)K.nblk * (double)(1ll << K.logP) / (double)d.n_up;
        for (int k = 0; k < 4; ++k) {
          if (!K.n_rows[k]) continue;
          Job J; memset(&J.P, 0, sizeof(J.P));
          block_args(J.P.A, K);
          J.P.A.xh = K.Xb.p; J.P.A.Wx = Wx; J.P.A.dWx = dWx; J.P.A.Tx = Tx;
          J.P.A.Nout = Nout; J.P.A.out_off = 0; J.P.A.out_mul = out_mul;
          J.P.rowinfo = K.rows[k].p; J.P.n_rows = K.n_rows[k];
          J.P.tab_off = K.off_d.p; J.P.tab_p = K.p_d.p; J.P.tab_pd = K.pd_d.p;
          J.P.write_dWx = dWx ? 1 : 0; J.P.ssq = ssq ? 1 : 0;
          J.P.blk_n = K.nblk; J.P.blk_hop = K.hop; J.P.blk_h2 = K.h2;
          J.cls = 2 + k; J.gb = vrows; J.rows = B * K.n_rows[k];
          J.w = (double)J.rows * frac * qw[k]; J.sblk_cls = -1;
          bjobs.push_back(J);
        }
      }
      for (int c = 0; c < SBLK_NCLS; ++c) {
        if (!sblk[c].used() || sblk[c].analytic) continue;
        Job J; memset(&J.P, 0, sizeof(J.P));
        J.cls = 0; J.gb = 0; J.rows = B * (long long)sblk[c].rows.size();
        J.w = (double)J.rows * 0.8; J.sblk_cls = c;
        bjobs.push_back(J);
      }
    }
    if (lanes_on && !bjobs.empty()) {
      rc = run_jobs(bjobs, false, 1); if (rc) return rc;       // lanes only: st does the FFT
      bjobs.clear();
    }

    rc = forward(x, B, xh_d.p, st); if (rc) return rc;
    const bool use_cut = use_blocks && have_cut && sblk[2].used();
    if (lanes_on) SSQB_CUDA(cudaEventRecord(ev_lane_fork, st));

    const int* rowmap = nullptr;
    long long two_pass_rows = total_rows;
    if (fast) {
      const std::vector<int>& bs = use_blocks ? big_scales : big_scales_all;
      two_pass_rows = B * (long long)bs.size();
      if (two_pass_rows > 0) {
        const long long mkey = B * 2 + (use_blocks ? 1 : 0);
        if (bigmap_B != mkey) {
          std::vector<int> mp((size_t)two_pass_rows);
          size_t k = 0;
          for (long long b = 0; b < B; ++b)
            for (int a : bs) mp[k++] = (int)(b * d.na + a);
          SSQB_CUDA(bigmap_d.upload(mp));
          bigmap_B = mkey;
        }
        rowmap = bigmap_d.p;
      }
    }
    // (g) gridded narrow-band rows first on the caller's stream: the coarse-grid transforms
    // need only xh; the interpolation kernel (the largest launch of a step) starts as soon
    // as Tx is zeroed
    if (fast && have_grid_rows) {
      SSQB_CUDA(V_d.ensure((size_t)B * (size_t)grid_v_total));
      GridArgs<T> G; grid_args(G, B, Wx, dWx, Tx, ssq, out_mul, rpadded, Nout);
      cudaStream_t s1 = st, s2 = st;
      if (lanes_on) { s1 = acquire(2, true, false); s2 = acquire(3, true, false); }
      rc = grid_stage_a(G, B, st, s1, s2); if (rc) return rc;
      acquire(0, true);
      rc = grid_stage_b(G, B, narr, st); if (rc) return rc;
      load[0] += 0.45 * (double)B * (double)grid_rows.size();
    }
    // (a) wide-band rows: two passes through the scratch, on a worker lane
    if (two_pass_rows > 0) {
      cudaStream_t ts = st;
      int tk = 0;
      if (lanes_on) { tk = least_loaded(1); load[tk] += 3.0 * (double)two_pass_rows; ts = acquire(tk, true, false); }
      long long chunk = rows_per_chunk(narr, two_pass_rows);
      SSQB_CUDA(ensure_scratch(narr, chunk));
      for (long long r0 = 0; r0 < two_pass_rows; r0 += chunk) {
        long long nr = (two_pass_rows - r0 < chunk) ? (two_pass_rows - r0) : chunk;
        CwtArgs<T> A; base_args(A);
        A.row0 = (int)r0; A.nrows = (int)nr; A.rowmap = rowmap;
        A.xh = xh_d.p; A.G = G_d.p; A.G_arr_stride = arr_stride(nr);
        A.Wx = Wx; A.dWx = dWx; A.Tx = Tx;
        A.Nout = Nout; A.out_off = rpadded ? 0 : d.n1;
        A.out_mul = out_mul;
        FastArgs<T> P; memset(&P, 0, sizeof(P));
        P.A = A; P.rowinfo = nullptr; P.n_rows = 0;
        P.tab_off = tab_off_d.p; P.tab_p = tab_p_d.p; P.tab_pd = tab_pd_d.p;
        P.write_dWx = dWx ? 1 : 0; P.ssq = ssq ? 1 : 0;
        P.scratch_logR2 = ROWS_LOGE - 9;
        rc = prof_begin(1, nr, ts); if (rc) return rc;
        rc = fast ? launch_pass1f<T>(P, narr, ts) : -100;
        if (rc == -100) rc = launch_pass1<T, MODE_CWT>(A, narr, ts);
        if (rc) return rc;
        rc = prof_end(ts); if (rc) return rc;
        acquire(tk, true);                                 // pass 2 writes Tx: wait for the zero fill
        rc = prof_begin(2, nr, ts); if (rc) return rc;
        if (fast)           rc = launch_rows_scratch<T>(P, narr, ts);
        else if (ssq)       rc = launch_pass2<T, 2, EPI_SSQ>(A, dWx ? 1 : 0, ts);
        else if (narr == 2) rc = launch_pass2<T, 2, EPI_CWT>(A, 1, ts);
        else                rc = launch_pass2<T, 1, EPI_CWT>(A, 0, ts);
        if (rc) return rc;
        rc = prof_end(ts); if (rc) return rc;
      }
      if (ts == st) load[0] += 8.0 * (double)B + 3.0 * (double)two_pass_rows;
    }
    acquire(0, true);

    // (b) narrow-band rows: single-pass direct kernel, one launch per class
    std::vector<Job> jobs;
    if (fast) {
      static const double cw[NCLS] = {0.65, 0.85, 1.0, 1.25, 1.6, 2.2};
      for (int c = 0; c < NCLS; ++c) {
        if (!n_qrows[c]) continue;
        Job J; memset(&J.P, 0, sizeof(J.P));
        base_args(J.P.A);
        J.P.A.xh = xh_d.p; J.P.A.Wx = Wx; J.P.A.dWx = dWx; J.P.A.Tx = Tx;
        J.P.A.Nout = Nout; J.P.A.out_off = rpadded ? 0 : d.n1; J.P.A.out_mul = out_mul;
        J.P.rowinfo = qrows_d[c].p; J.P.n_rows = n_qrows[c];
        J.P.tab_off = tab_off_d.p; J.P.tab_p = tab_p_d.p; J.P.tab_pd = tab_pd_d.p;
        J.P.write_dWx = dWx ? 1 : 0; J.P.ssq = ssq ? 1 : 0; J.P.scratch_logR2 = 0;
        J.cls = c; J.gb = B; J.rows = B * n_qrows[c];
        J.w = (double)J.rows * cw[c]; J.sblk_cls = -1;
        jobs.push_back(J);
      }
      if (use_cut) {
        Job J; memset(&J.P, 0, sizeof(J.P));
        J.cls = 0; J.gb = 0; J.rows = B * (long long)sblk[2].rows.size();
        J.w = (double)J.rows * 0.9; J.sblk_cls = 2;
        jobs.push_back(J);
      }
    }
    for (const Job& J : bjobs) jobs.push_back(J);        // lanes off: blocks run here
    rc = run_jobs(jobs, true, 0); if (rc) return rc;
    if (lanes_on)
      for (int i = 0; i < NLANES; ++i)
        if (lane_used[i]) {
          SSQB_CUDA(cudaEventRecord(ev_lane_done[i], lanes[i]));
          SSQB_CUDA(cudaStreamWaitEvent(st, ev_lane_done[i], 0));
        }
    return 0;
  }

  // Host buffers in, host buffers out (pinned memory recommended).  The batch is cut into
  // chunks of two signals that ping-pong between two device staging slots:
  // chunk c is transformed on the caller's stream while the copy stream still drains the
  // outputs of chunk c-1 over PCIe, so the device holds two chunks of outputs, not the batch.
  cudaStream_t copy_st = nullptr;
  cudaEvent_t ev_comp[2] = {nullptr, nullptr}, ev_d2h[2] = {nullptr, nullptr};
  int exec_host(const void* x, long long B, void* Wx, void* dWx, void* Tx, bool ssq,
                const double* out_mul_host, bool rpadded, cudaStream_t st) override {
    if (B < 1) return set_error(SSQB_E_ARG, "B must be >= 1");
    const long long CH = B < 2 ? B : 2;
    const long long Nout = rpadded ? d.n_up : d.N;
    const size_t nx = (size_t)CH * (size_t)d.N, nout = (size_t)CH * d.na * (size_t)Nout;
    SSQB_CUDA(x_stage.ensure(2 * nx));
    SSQB_CUDA(Wx_stage.ensure(2 * nout));
    if (dWx) SSQB_CUDA(dWx_stage.ensure(2 * nout));
    if (ssq) SSQB_CUDA(Tx_stage.ensure(2 * nout));
    if (!copy_st) {
      SSQB_CUDA(cudaStreamCreateWithFlags(&copy_st, cudaStreamNonBlocking));
      for (int i = 0; i < 2; ++i) {
        SSQB_CUDA(cudaEventCreateWithFlags(&ev_comp[i], cudaEventDisableTiming));
        SSQB_CUDA(cudaEventCreateWithFlags(&ev_d2h[i], cudaEventDisableTiming));
      }
    }
    const T* xh_ = (const T*)x;
    cx<T>* Wh = (cx<T>*)Wx; cx<T>* dWh = (cx<T>*)dWx; cx<T>* Th = (cx<T>*)Tx;
    int rc = 0, c = 0;
    bool slot_busy[2] = {false, false};
    for (long long b0 = 0; b0 < B; b0 += CH, ++c) {
      const int sl = c & 1;
      const long long nb = (B - b0 < CH) ? (B - b0) : CH;
      const size_t cx_ = (size_t)nb * (size_t)d.N, co = (size_t)nb * d.na * (size_t)Nout;
      if (slot_busy[sl]) SSQB_CUDA(cudaStreamWaitEvent(st, ev_d2h[sl], 0));   // slot drained
      T* xs = x_stage.p + sl * nx;
      cx<T>* Ws = Wx_stage.p + sl * nout;
      cx<T>* dWs = dWx ? dWx_stage.p + sl * nout : nullptr;
      cx<T>* Ts = ssq ? Tx_stage.p + sl * nout : nullptr;
      SSQB_CUDA(cudaMemcpyAsync(xs, xh_ + (size_t)b0 * (size_t)d.N, cx_ * sizeof(T),
                                cudaMemcpyHostToDevice, st));
      rc = exec(xs, nb, Ws, dWs, Ts, ssq, out_mul_host, rpadded, st);
      if (rc) break;
      SSQB_CUDA(cudaEventRecord(ev_comp[sl], st));
      SSQB_CUDA(cudaStreamWaitEvent(copy_st, ev_comp[sl], 0));
      const size_t ho = (size_t)b0 * d.na * (size_t)Nout;
      SSQB_CUDA(cudaMemcpyAsync(Wh + ho, Ws, co * sizeof(cx<T>), cudaMemcpyDeviceToHost, copy_st));
      if (dWx) SSQB_CUDA(cudaMemcpyAsync(dWh + ho, dWs, co * sizeof(cx<T>), cudaMemcpyDeviceToHost, copy_st));
      if (ssq) SSQB_CUDA(cudaMemcpyAsync(Th + ho, Ts, co * sizeof(cx<T>), cudaMemcpyDeviceToHost, copy_st));
      SSQB_CUDA(cudaEventRecord(ev_d2h[sl], copy_st));
      slot_busy[sl] = true;
    }
    // the call returns with the results in the host buffers
    cudaError_t e1 = cudaStreamSynchronize(copy_st), e2 = cudaStreamSynchronize(st);
    if (rc) return rc;
    SSQB_CUDA(e1); SSQB_CUDA(e2);
    return 0;
  }

  int debug_xh(const void* x, long long B, void* xh, cudaStream_t st) override {
    return forward((const T*)x, B, (cx<T>*)xh, st);
  }
  CwtAdjoint<T> adj;
  int backward(const void* gWx, const void* gdWx, long long B, const double* out_mul_host,
               bool rpadded, void* gx, cudaStream_t st) override {
    CwtArgs<T> A; base_args(A);
    return adj.run(d, A, (const cx<T>*)gWx, (const cx<T>*)gdWx, B, out_mul_host, rpadded, (T*)gx, st);
  }
};

template <typename T>
static CwtPlanBase* make_cwt_plan(const ssqb_cwt_desc* d, int* err) {
  if (d->n_up > 0 && (d->n_up & (d->n_up - 1))) {     // not a power of two: generic-length FFT
    GenericCwtPlan<T>* g = new GenericCwtPlan<T>();
    *err = g->init(d);
    if (*err) { delete g; return nullptr; }
    return g;
  }
  CwtPlan<T>* p = new CwtPlan<T>();
  *err = p->init(d);
  if (*err) { delete p; return nullptr; }
  return p;
}

}  // namespace ssqb

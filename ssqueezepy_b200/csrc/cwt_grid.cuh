// Gridded evaluation of narrow-band CWT rows: decimate, then interpolate.
//
// A scale whose wavelet spectrum occupies L << n bins (ssqueezepy/wavelets.py:62-95,
// `Psih` row) yields a row  W[t] = sum_i Z[i] e^{2 pi i i t / n}  (ssqueezepy/_cwt.py:167-177)
// that is band-limited to L/n of the sampling rate: the n-point inverse FFT the reference
// runs is almost entirely interpolation.  With c the band centre and m = i - c:
//
//   W[t] = e^{2 pi i c t / n} * E(t),     E(t) = sum_m Z[c+m] e^{2 pi i m t / n}
//
// E is evaluated by the standard "type 2" gridding scheme on a coarse grid of M >= 2L points
// (U = n / M fine samples per coarse sample):
//   (A) V[p] = sum_m (Z[c+m] / phi_hat(m/M)) e^{2 pi i m p / M}      one M-point inverse FFT
//   (B) E(t) = sum_k phi(t/U - q_k) V[q_k],  q_k = floor(t/U) - K/2 + 1 + k,  k < K
// phi(s) = exp(beta (sqrt(1 - (2s/K)^2) - 1)) on |s| < K/2 ("exponential of semicircle"),
// beta = 2.30 K.  The aliasing error is ~1e-8 of the row for K = 8 (float32: below the
// rounding noise of the transform) and 2.5e-14 for K = 14 (float64); measured against
// the reference in tests/test_gpu_shapes.py.  Stage (A) costs M log M per row (< 1 % of
// the work); stage (B) is K packed FMAs per output point per array, reads V from L2 and
// writes every output exactly once -- no padded samples are ever computed.
//
// Kernels:
//   psih_grid_kernel       per plan: band tables pre-divided by phi_hat (the reference's
//                          `Wavelet.Psih` cache, wavelets.py:135-160)
//   grid_dec_ifft_kernel   stage (A): CTA = R rows x M points, both arrays (W, dW)
//   grid_interp_kernel     stage (B) + epilogue: unpad, store Wx[, dWx], phase transform,
//                          bin index (algos.py:912-924), red.global.add into Tx
#pragma once
#include "cwt_fast.cuh"

namespace ssqb {

struct GridRow {               // one gridded row (host-built)
  int a;                       // scale index
  int logM;                    // coarse length M = 2^logM
  int c;                       // band centre bin (mod n)
  int lo;                      // first band bin (mod n)
  int len;                     // band length L
  int pad;
  long long tab_off;           // offset of the band in gtab_p / gtab_pd
  long long v_off;             // offset of this row's V (V4 elements) within one signal
};

// ---- 1-D bulk asynchronous copy (TMA unit, `cp.async.bulk`; SASS: UBLKCP) + mbarrier -------------
__device__ __forceinline__ unsigned smem_u32(const void* p) {
  return (unsigned)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(unsigned long long* bar, unsigned count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(smem_u32(bar)), "r"(count) : "memory");
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long* bar, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, unsigned bytes,
                                         unsigned long long* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               :: "r"(smem_u32(dst_smem)), "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, unsigned parity) {
  asm volatile(
      "{\n .reg .pred p;\n WAIT_%=:\n"
      " mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      " @p bra DONE_%=;\n bra WAIT_%=;\n DONE_%=:\n}"
      :: "r"(smem_u32(bar)), "r"(parity) : "memory");
}

template <typename T>
struct GridArgs {
  CwtArgs<T> A;
  const GridRow* rows;
  int n_rows;                  // rows per signal in `rows`
  long long B;                 // signals
  typename V4T<T>::type* V;    // [B][v_total]  (W.re, W.im, dW.re, dW.im) on the coarse grids
  long long v_total;
  const T* gtab_p;             // psih / phi_hat on the band
  const T* gtab_pd;            // psih * xi / dt / phi_hat
  const cx<T>* rootsM;         // exp(2 pi i m / MMAX), m < MMAX
  const cx<T>* rootsMh;        // exp(2 pi i m / (MMAX/2)), m < MMAX/2 (split transforms of MMAX points)
  int log_mmax;
  const T* htab;               // [UMAX][K] phi(u/UMAX - k + K/2 - 1)
  int log_umax;
  int write_dWx, ssq;
  int t0, tcount;              // padded time indices wanted: [t0, t0 + tcount)
};

// ---- per-plan tables ------------------------------------------------------------------
// comp holds 1/phi_hat(m/M) for every class logM = 6..: entries (m + M/2) at offset M - 64
template <typename T>
__global__ void __launch_bounds__(256)
psih_grid_kernel(const CwtArgs<T> A, const GridRow* __restrict__ rows, const T* __restrict__ comp,
                 T* __restrict__ tab_p, T* __restrict__ tab_pd) {
  const GridRow ri = rows[blockIdx.y];
  const int M = 1 << ri.logM;
  const T sc = A.scales[ri.a];
  const T* cm = comp + (M - 64) + M / 2;
  for (int m = blockIdx.x * blockDim.x + threadIdx.x; m < ri.len; m += gridDim.x * blockDim.x) {
    long long i = ((long long)ri.lo + m) & (A.n_up - 1);
    int ms = m - (ri.len >> 1);                      // i - c, signed
    T p = psih_eval<T>(A, ri.a, i, sc) * cm[ms];
    tab_p[ri.tab_off + m] = p;
    tab_pd[ri.tab_off + m] = p * (xi_of<T>(i, A.n_up) / A.dt);
  }
}

// ---- stage (A): coarse-grid inverse FFTs -----------------------------------------------
template <int LOG_M> struct DecGeom {
  static constexpr int M = 1 << LOG_M;
  static constexpr int ELEMS = (LOG_M <= 11) ? 2048 : M;
  static constexpr int R = ELEMS / M;                // rows per CTA
  static constexpr int NT = ELEMS / 8;
};

template <typename T, int LOG_M>
__device__ __forceinline__ void grid_dec_body(const GridArgs<T>& G, const GridRow* __restrict__ rows,
                                              int n_cls, int cta) {
  using Geo = DecGeom<LOG_M>;
  constexpr int M = Geo::M, R = Geo::R, NT = Geo::NT;
  using V4 = typename V4T<T>::type;
  const CwtArgs<T>& A = G.A;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  cx<T>* s = reinterpret_cast<cx<T>*>(smem_raw);     // [2][M][R]
  cx<T>* tw = s + 2 * M * R;                         // [M]
  __shared__ GridRow rinfo[R];
  __shared__ int rsig[R];
  const int tid = threadIdx.x;
  const unsigned nmask = (unsigned)(A.n_up - 1);
  const long long total = (long long)n_cls * G.B;    // (signal, row) pairs of this class
  const long long pair0 = (long long)cta * R;
  if (tid < R) {
    const long long pr = pair0 + tid;
    int b = -1;
    if (pr < total) {
      b = (int)(pr / n_cls);
      rinfo[tid] = rows[pr - (long long)b * n_cls];
    }
    rsig[tid] = b;
  }
  for (int m = tid; m < M; m += NT) tw[m] = G.rootsM[(size_t)m << (G.log_mmax - LOG_M)];
  __syncthreads();
  // element e of lane r holds band bin m = (e + L/2) mod M  (e = (i - c) mod M), zero outside
  for (int idx = tid; idx < M * R; idx += NT) {
    const int e = idx & (M - 1), r = idx >> LOG_M;
    cx<T> zw = mkc<T>((T)0, (T)0), zd = zw;
    const int b = rsig[r];
    if (b >= 0) {
      const int L = rinfo[r].len;
      const int m = (e + (L >> 1)) & (M - 1);
      if (m < L) {
        const cx<T> xv = __ldg(&A.xh[(long long)b * A.n_up + ((unsigned)(rinfo[r].lo + m) & nmask)]);
        zw = cscale<T>(xv, __ldg(&G.gtab_p[rinfo[r].tab_off + m]));      // Psih * xh      (_cwt.py:169)
        zd = cscale<T>(xv, __ldg(&G.gtab_pd[rinfo[r].tab_off + m]));     // ... * xi / dt  (_cwt.py:175)
      }
    }
    s[e * R + r] = zw;
    s[M * R + e * R + r] = zd;
  }
  __syncthreads();
  stockham_from_n<T, LOG_M, R, NT, R, 1, 2>(s, tw);
  for (int idx = tid; idx < M * R; idx += NT) {
    const int p = idx & (M - 1), r = idx >> LOG_M;
    const int b = rsig[r];
    if (b < 0) continue;
    const cx<T> w = s[p * R + r], d = s[M * R + p * R + r];
    V4 o; o.x = w.x; o.y = w.y; o.z = -d.y; o.w = d.x;         // dW carries the 1j of 1j*xi/dt
    G.V[(long long)b * G.v_total + rinfo[r].v_off + p] = o;
  }
}

template <typename T, int LOG_M>
__global__ void __launch_bounds__(DecGeom<LOG_M>::NT)
grid_dec_ifft_kernel(const GridArgs<T> G, const GridRow* __restrict__ rows, int n_cls) {
  grid_dec_body<T, LOG_M>(G, rows, n_cls, blockIdx.x);
}

// the longest coarse grid (2^14 points in float32, 2^13 in float64): one array (W or dW) per CTA
// -- two would not fit shared memory --, roots read from the global table (= exactly M entries)
template <typename T, int LOG_M>
__global__ void __launch_bounds__(1024)
grid_dec_single_kernel(const GridArgs<T> G, const GridRow* __restrict__ rows, int n_cls) {
  constexpr int M = 1 << LOG_M, NT = 1024;
  const CwtArgs<T>& A = G.A;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  cx<T>* s = reinterpret_cast<cx<T>*>(smem_raw);     // [M]
  const int tid = threadIdx.x;
  const int arr = blockIdx.y;                         // 0: W, 1: dW
  const unsigned nmask = (unsigned)(A.n_up - 1);
  const long long pr = blockIdx.x;
  const int b = (int)(pr / n_cls);
  const GridRow ri = rows[pr - (long long)b * n_cls];
  const cx<T>* __restrict__ xh = A.xh + (long long)b * A.n_up;
  const T* __restrict__ tp = (arr == 0 ? G.gtab_p : G.gtab_pd) + ri.tab_off;
  const int L = ri.len;
  for (int e = tid; e < M; e += NT) {
    const int m = (e + (L >> 1)) & (M - 1);
    cx<T> z = mkc<T>((T)0, (T)0);
    if (m < L) z = cscale<T>(__ldg(&xh[(unsigned)(ri.lo + m) & nmask]), __ldg(&tp[m]));
    s[e] = z;
  }
  __syncthreads();
  stockham_from_n<T, LOG_M, 1, NT, 1, 1, 1>(s, G.rootsM);
  T* __restrict__ Vr = reinterpret_cast<T*>(G.V + (long long)b * G.v_total + ri.v_off);
  for (int p = tid; p < M; p += NT) {
    const cx<T> v = s[p];
    if (arr == 0) { Vr[4 * p] = v.x; Vr[4 * p + 1] = v.y; }
    else          { Vr[4 * p + 2] = -v.y; Vr[4 * p + 3] = v.x; }     // dW carries the 1j of 1j*xi/dt
  }
}

// coarse grids longer than one CTA's shared memory, M = R * Mb (R = 2 .. 16): the first
// decimation-in-frequency stage is done while the band is read,
//   y_c[j] = w_M^(c j) sum_q z[j + q Mb] w_R^(c q),   V[R k + c] = iFFT_Mb(y_c)[k],
// so CTA c of the R that share a (row, array) works on its own Mb points and nothing is
// exchanged between CTAs.  z is the band (zero elsewhere): at most R/2 + 1 of the R terms exist.
template <typename T, int LOG_MB>
__global__ void __launch_bounds__(1024)
grid_dec_split_kernel(const GridArgs<T> G, const GridRow* __restrict__ rows, int n_cls, int logR) {
  constexpr int Mb = 1 << LOG_MB, NT = 1024;
  const CwtArgs<T>& A = G.A;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  cx<T>* s = reinterpret_cast<cx<T>*>(smem_raw);     // [Mb]
  __shared__ cx<T> wR[16];
  const int tid = threadIdx.x;
  const int arr = blockIdx.y;                         // 0: W, 1: dW
  const int R = 1 << logR, c = (int)(blockIdx.x & (unsigned)(R - 1));
  const long long pr = (long long)(blockIdx.x >> logR);
  const int b = (int)(pr / n_cls);
  const GridRow ri = rows[pr - (long long)b * n_cls];
  const int logM = LOG_MB + logR, logU = A.logn - logM;
  const unsigned Mm = (1u << logM) - 1u, nmask = (unsigned)(A.n_up - 1);
  const cx<T>* __restrict__ xh = A.xh + (long long)b * A.n_up;
  const T* __restrict__ tp = (arr == 0 ? G.gtab_p : G.gtab_pd) + ri.tab_off;
  const int L = ri.len;
  if (tid < R)
    wR[tid] = twiddle_n<T>(A.tw_lo, A.tw_hi, A.log_lo, (unsigned long long)tid << (A.logn - logR));
  __syncthreads();
  for (int j = tid; j < Mb; j += NT) {
    cx<T> acc = mkc<T>((T)0, (T)0);
    for (int q = 0; q < R; ++q) {
      const unsigned m = ((unsigned)(j + (q << LOG_MB)) + (unsigned)(L >> 1)) & Mm;
      if (m < (unsigned)L) {
        const cx<T> z = cscale<T>(__ldg(&xh[((unsigned)ri.lo + m) & nmask]), __ldg(&tp[m]));
        acc = cadd<T>(acc, cmul<T>(z, wR[(c * q) & (R - 1)]));
      }
    }
    const unsigned long long ph = ((unsigned long long)(unsigned)c * (unsigned)j) & Mm;
    s[j] = cmul<T>(acc, twiddle_n<T>(A.tw_lo, A.tw_hi, A.log_lo, ph << logU));
  }
  __syncthreads();
  stockham_from_n<T, LOG_MB, 1, NT, 1, 1, 1>(s, LOG_MB == G.log_mmax ? G.rootsM : G.rootsMh);
  T* __restrict__ Vr = reinterpret_cast<T*>(G.V + (long long)b * G.v_total + ri.v_off);
  for (int p = tid; p < Mb; p += NT) {
    const cx<T> v = s[p];
    const size_t o = 4 * (((size_t)p << logR) + (size_t)c);
    if (arr == 0) { Vr[o] = v.x; Vr[o + 1] = v.y; }
    else          { Vr[o + 2] = -v.y; Vr[o + 3] = v.x; }
  }
}

// all coarse lengths up to 2^11 in one launch (256 threads): CTA -> (class, tile) by prefix table
struct DecSmallPlan {
  int cta_start[7];            // classes 2^6 .. 2^11, exclusive prefix; [6] = total
  int row_first[6], n_cls[6];
};
template <typename T>
__global__ void __launch_bounds__(256)
grid_dec_ifft_small_kernel(const GridArgs<T> G, const DecSmallPlan P) {
  const int cta = blockIdx.x;
  int c = 0;
#pragma unroll
  for (int k = 1; k < 6; ++k) if (cta >= P.cta_start[k]) c = k;
  const GridRow* rows = G.rows + P.row_first[c];
  const int loc = cta - P.cta_start[c], n = P.n_cls[c];
  switch (c) {
    case 0: grid_dec_body<T, 6>(G, rows, n, loc); break;
    case 1: grid_dec_body<T, 7>(G, rows, n, loc); break;
    case 2: grid_dec_body<T, 8>(G, rows, n, loc); break;
    case 3: grid_dec_body<T, 9>(G, rows, n, loc); break;
    case 4: grid_dec_body<T, 10>(G, rows, n, loc); break;
    default: grid_dec_body<T, 11>(G, rows, n, loc); break;
  }
}

// ---- stage (B): interpolation + fused epilogue --------------------------------------------
// CTA of 256 threads = UT consecutive fine phases u (UT = min(U, 256)) x PG = 256/UT groups of
// PP = K*PPK consecutive coarse samples p.  A thread keeps its phase: the K kernel values
// phi(u/U - .) live in registers, the K-sample window slides one coarse sample per output
// (one 16-byte shared-memory load per output for both arrays), and the 32 lanes of a warp
// write 32 consecutive time samples (256 contiguous bytes of Wx).
template <typename T, int K, int PPK> struct InterpGeom {
  static constexpr int PP = K * PPK;
  static constexpr int NT = 256;
};

template <typename T, int K, int PPK, int NARR, bool SSQ>
__global__ void __launch_bounds__(256, (sizeof(T) == 4) ? 3 : 1)
grid_interp_kernel(const GridArgs<T> G) {
  constexpr int PP = K * PPK;
  constexpr int NT = 256;
  using V4 = typename V4T<T>::type;
  const CwtArgs<T>& A = G.A;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int tid = threadIdx.x;
  const int y = blockIdx.y;
  const int b = y / G.n_rows;
  const GridRow ri = G.rows[y - b * G.n_rows];
  const int logM = ri.logM, logU = A.logn - logM;
  const int logUT = logU < 8 ? logU : 8;
  const int UT = 1 << logUT, PG = NT >> logUT;
  const int PTILE = PG * PP;                          // coarse samples per CTA
  const int n_ut = 1 << (logU - logUT);
  const int p_first = G.t0 >> logU;
  const int p_last = (G.t0 + G.tcount - 1) >> logU;
  const int n_pt = (p_last - p_first + PTILE) / PTILE;
  const int tile = blockIdx.x;
  if (tile >= n_ut * n_pt) return;
  const int ut = tile % n_ut, pt = tile / n_ut;
  const int p_cta = p_first + pt * PTILE;             // first coarse sample of this CTA
  V4* Vs = reinterpret_cast<V4*>(smem_raw);           // [PTILE + K - 1]
  cx<T>* As = reinterpret_cast<cx<T>*>(Vs + (PTILE + K - 1));   // [PTILE] e^{2 pi i c p / M}
  const unsigned Mm = (1u << logM) - 1u;
  __shared__ __align__(8) unsigned long long vbar;
  {
    const V4* __restrict__ Vr = G.V + (long long)b * G.v_total + ri.v_off;
    // the CTA's window of the coarse sequence: one bulk copy by the TMA unit when it does not wrap
    // around the (periodic) sequence, signalled on an mbarrier; element-wise otherwise
    const int w0 = p_cta - (K / 2 - 1), nw = PTILE + K - 1;
    const bool bulk = (w0 >= 0) && (w0 + nw <= (1 << logM));
    if (bulk) {
      if (tid == 0) mbar_init(&vbar, 1);
      __syncthreads();
      if (tid == 0) {
        mbar_expect_tx(&vbar, (unsigned)(nw * sizeof(V4)));
        bulk_g2s(Vs, Vr + w0, (unsigned)(nw * sizeof(V4)), &vbar);
      }
    } else {
      for (int w = tid; w < nw; w += NT) Vs[w] = Vr[(unsigned)(w0 + w) & Mm];
    }
    for (int w = tid; w < PTILE; w += NT) {
      const unsigned long long ph = ((unsigned long long)(unsigned)ri.c * (unsigned)(p_cta + w)) & Mm;
      As[w] = twiddle_n<T>(A.tw_lo, A.tw_hi, A.log_lo, ph << logU);
    }
  }
  const int ul = tid & (UT - 1), pg = tid >> logUT;
  const int u = ut * UT + ul;
  T h[K];
  {
    const T* __restrict__ hp = G.htab + ((size_t)u << (G.log_umax - logU)) * K;
#pragma unroll
    for (int k = 0; k < K; ++k) h[k] = __ldg(&hp[k]);
  }
  const cx<T> Bu = twiddle_n<T>(A.tw_lo, A.tw_hi, A.log_lo,
                                ((unsigned long long)(unsigned)ri.c * (unsigned)u) & (unsigned long long)(A.n_up - 1));
  const int wl0 = pg * PP;                            // this thread's window base in Vs / As
  int np = p_last + 1 - (p_cta + wl0);                // coarse samples left for this thread
  if (np > PP) np = PP;

  const int a = ri.a;
  const long long row = (long long)b * A.na + a;
  const int Nout = (int)A.Nout;
  cx<T>* __restrict__ Wrow = A.Wx + row * Nout;
  cx<T>* __restrict__ dWrow = A.dWx ? A.dWx + row * Nout : nullptr;
  cx<T>* __restrict__ Tb = A.Tx ? A.Tx + (long long)b * A.na * Nout : nullptr;
  cx<T>* __restrict__ Zrow = (SSQ && b < A.zero_next) ? A.Tx + row * Nout + A.zero_off : nullptr;   // zero-ahead
  // epilogue constants
  const T mlt = (!SSQ && A.out_mul != nullptr) ? A.out_mul[a] : (T)1;
  double cwide = 0; T cre = 0, g2lo = 0, g2hi = 0; bool fast_ok = false; unsigned rowbytes = 0;
  if (SSQ) {
    cwide = A.cst[a]; cre = (T)cwide;
    const T g2 = (T)(A.grid.gamma * A.grid.gamma);
    const T g2tol = g2 * (T)(sizeof(T) == 4 ? 1e-5 : 1e-13);
    g2lo = g2 - g2tol;
    g2hi = fmax(g2 + g2tol, (T)1e-30);
    fast_ok = (A.grid.kind <= 1) && (A.grid.ftol < 0.25f);
    rowbytes = (unsigned)Nout * (unsigned)sizeof(cx<T>);
  }
  {
    const int w0 = p_cta - (K / 2 - 1);
    if ((w0 >= 0) && (w0 + PTILE + K - 1 <= (1 << logM))) mbar_wait(&vbar, 0);   // window has landed
  }
  __syncthreads();
  if (np <= 0) return;

  const int tbase = ((p_cta + wl0) << logU) + u;      // padded time index of output i = 0
  const int tlo = G.t0, thi = G.t0 + G.tcount;
  const int joff = (int)A.out_off;

  auto emit = [&](int i, cx<T> aw, cx<T> ad) {
    const int t = tbase + (i << logU);
    if (i < np && t >= tlo && t < thi) {
      const cx<T> tw = cmul<T>(As[wl0 + i], Bu);
      const cx<T> W = cmul<T>(aw, tw);
      const int jo = t - joff;
      if (!SSQ) {
        Wrow[jo] = cscale<T>(W, mlt);
        if (NARR == 2 && G.write_dWx) dWrow[jo] = cscale<T>(cmul<T>(ad, tw), mlt);
      } else {
        const cx<T> dW = cmul<T>(ad, tw);
        Wrow[jo] = W;
        if (G.write_dWx) dWrow[jo] = dW;
        if (Zrow) Zrow[jo] = mkc<T>((T)0, (T)0);
        ssq_point<T>(W, dW, Tb + jo, rowbytes, cre, cwide, g2lo, g2hi, fast_ok, A.grid);
      }
    }
  };

  // register-resident sliding window
  V4 win[K];
#pragma unroll
  for (int k = 0; k < K - 1; ++k) win[k] = Vs[wl0 + k];
#pragma unroll 1
  for (int g = 0; g < PPK; ++g) {
    if (g * K >= np) break;
#pragma unroll
    for (int kk = 0; kk < K; ++kk) {
      const int i = g * K + kk;
      win[(kk + K - 1) % K] = Vs[wl0 + i + K - 1];
      cx<T> aw = cscale<T>(mkc<T>(win[kk % K].x, win[kk % K].y), h[0]);
      cx<T> ad = mkc<T>((T)0, (T)0);
      if (NARR == 2) ad = cscale<T>(mkc<T>(win[kk % K].z, win[kk % K].w), h[0]);
#pragma unroll
      for (int k = 1; k < K; ++k) {
        const V4 v = win[(kk + k) % K];
        aw = caxpy<T>(mkc<T>(v.x, v.y), h[k], aw);
        if (NARR == 2) ad = caxpy<T>(mkc<T>(v.z, v.w), h[k], ad);
      }
      emit(i, aw, ad);
    }
  }
}


}  // namespace ssqb

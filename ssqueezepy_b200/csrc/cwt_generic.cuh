// CWT / ssq_cwt at transform lengths that are not powers of two (`padtype=None` on any N):
// host side of the generic-length FFT (gfft.cuh) and a plan with the same interface as the
// power-of-two plan.  The transform is materialised like the reference's
// (ssqueezepy/_cwt.py:167-177): xh = fft(x); per scale Psih * xh -> ifft, * 1j xi / dt -> ifft;
// synchrosqueezing then runs the deterministic column-owner operator on (Wx, dWx)
// (algos.py:912-924), so Tx is bit-identical to the reference's for identical transforms.
#pragma once
#include "host_common.h"
#include "cwt_kernels.cuh"
#include "gfft.cuh"
#include <memory>

namespace ssqb {

constexpr long long GFFT_SMEM_MAX = 4096;

template <typename T>
struct Gfft {
  long long n = 0;
  int kind = -1;                               // 0 shared memory, 1 two passes, 2 Bluestein
  GfftStages S{}, S1{}, S2{};
  long long n1 = 0, n2 = 0, M = 0;
  std::unique_ptr<Gfft<T>> sub;
  DevBuf<cx<T>> Y, a0, a1, bh[2];
  bool bh_ready[2] = {false, false};

  static bool factor(long long n, GfftStages& S) {
    if (n < 1 || n > GFFT_SMEM_MAX) return false;
    S.n = (int)n; S.nst = 0;
    long long m = n;
    auto push = [&](int r) { if (S.nst < GFFT_MAX_STAGES) S.radix[S.nst++] = r; };
    while (m % 8 == 0) { push(8); m /= 8; }
    while (m % 4 == 0) { push(4); m /= 4; }
    for (int p = 2; p <= 31; ++p) while (m % p == 0) { push(p); m /= p; }
    if (n == 1) { push(1); }
    return m == 1 && S.nst < GFFT_MAX_STAGES;
  }

  int init(long long n_) {
    n = n_;
    if (factor(n, S)) { kind = 0; return 0; }
    // balanced split n = n1 * n2 with both factors transformable in shared memory
    long long best = 0;
    for (long long dv = 2; dv * dv <= n; ++dv) {
      if (n % dv) continue;
      GfftStages t1, t2;
      if (n / dv <= GFFT_SMEM_MAX && factor(dv, t1) && factor(n / dv, t2)) best = dv;
    }
    if (best) {
      kind = 1; n1 = best; n2 = n / best;
      factor(n1, S1); factor(n2, S2);
      return 0;
    }
    kind = 2;
    M = 1; while (M < 2 * n - 1) M <<= 1;
    if (M > GFFT_SMEM_MAX * GFFT_SMEM_MAX)
      return set_error(SSQB_E_UNSUPP, "transform length %lld too long for the generic FFT", n);
    sub.reset(new Gfft<T>());
    return sub->init(M);
  }

  static int launch(const GfftStages& S, const cx<T>* in, cx<T>* out, GfftView vin, GfftView vout,
                    long long count, long long inner_n, int sign, long long tw_n, T scale,
                    cudaStream_t st) {
    GfftArgs<T> A;
    A.S = S; A.in = in; A.out = out; A.vin = vin; A.vout = vout; A.count = count;
    A.inner_n = inner_n; A.sign = sign; A.tw_n = tw_n; A.scale = scale;
    int R = (int)(2048 / S.n); if (R < 1) R = 1; if (R > 16) R = 16;
    A.R = R;
    size_t smem = ((size_t)2 * S.n * R + S.n) * sizeof(cx<T>);
    auto kern = gfft_smem_kernel<T>;
    SSQB_CUDA(set_smem_limit(kern, smem));
    kern<<<(unsigned)((count + R - 1) / R), 256, smem, st>>>(A);
    SSQB_LAUNCH_CHECK();
    return 0;
  }

  // out[b][k] = scale * sum_j in[b][j] e^{sign 2 pi i j k / n};  in != out, both [batch][n]
  int exec(const cx<T>* in, cx<T>* out, long long batch, int sign, T scale, cudaStream_t st) {
    if (kind == 0)
      return launch(S, in, out, GfftView{n, 0, 1}, GfftView{n, 0, 1}, batch, 1, sign, 0, scale, st);
    if (kind == 1) {
      SSQB_CUDA(Y.ensure((size_t)batch * (size_t)n));
      // columns: transform (b, i2) over i1 (stride n2) -> Y[b][t1 n2 + i2] * w_n^(i2 t1)
      int rc = launch(S1, in, Y.p, GfftView{n, 1, n2}, GfftView{n, 1, n2}, batch * n2, n2, sign, n,
                      (T)1, st);
      if (rc) return rc;
      // rows: transform (b, t1) over i2 (contiguous) -> out[b][t1 + n1 t2]
      return launch(S2, Y.p, out, GfftView{n, n2, 1}, GfftView{n, 1, n1}, batch * n1, n1, sign, 0,
                    scale, st);
    }
    // Bluestein, in chunks that keep the two convolution buffers below ~256 MB each
    const int si = sign > 0 ? 1 : 0;
    if (!bh_ready[si]) {
      SSQB_CUDA(a0.ensure((size_t)M)); SSQB_CUDA(bh[si].ensure((size_t)M));
      gfft_chirp_kernel_kernel<T><<<(unsigned)((M + 255) / 256), 256, 0, st>>>(a0.p, n, M, sign);
      SSQB_LAUNCH_CHECK();
      int rc = sub->exec(a0.p, bh[si].p, 1, -1, (T)1, st); if (rc) return rc;
      bh_ready[si] = true;
    }
    long long cb = ((256ll << 20) / (long long)sizeof(cx<T>)) / M; if (cb < 1) cb = 1;
    if (cb > batch) cb = batch;
    SSQB_CUDA(a0.ensure((size_t)cb * (size_t)M)); SSQB_CUDA(a1.ensure((size_t)cb * (size_t)M));
    for (long long b0 = 0; b0 < batch; b0 += cb) {
      const long long nb = batch - b0 < cb ? batch - b0 : cb;
      const unsigned gM = (unsigned)((nb * M + 255) / 256), gn = (unsigned)((nb * n + 255) / 256);
      gfft_chirp_in_kernel<T><<<gM, 256, 0, st>>>(in + b0 * n, a0.p, n, M, nb, sign);
      SSQB_LAUNCH_CHECK();
      int rc = sub->exec(a0.p, a1.p, nb, -1, (T)1, st); if (rc) return rc;
      gfft_mul_kernel<T><<<gM, 256, 0, st>>>(a1.p, bh[si].p, M, nb);
      SSQB_LAUNCH_CHECK();
      rc = sub->exec(a1.p, a0.p, nb, +1, (T)1, st); if (rc) return rc;
      gfft_chirp_out_kernel<T><<<gn, 256, 0, st>>>(a0.p, out + b0 * n, n, M, nb, sign,
                                                   (T)((double)scale / (double)M));
      SSQB_LAUNCH_CHECK();
    }
    return 0;
  }
};

// ---- element-wise kernels of the generic CWT plan -------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256)
gen_pad_kernel(const T* __restrict__ x, cx<T>* __restrict__ xp, long long N, long long n, long long n1,
               int padtype, long long B) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= B * n) return;
  const long long b = idx / n, t = idx - b * n;
  const long long src = pad_src_index(t, n1, N, padtype);
  xp[idx] = mkc<T>(src >= 0 ? x[b * N + src] : (T)0, (T)0);
}
// Z[arr][r][i] = psih(a_r, i) * xh[b_r][i] (* 1j xi_i / dt for arr = 1); rows r = r0 .. r0 + nr
template <typename T>
__global__ void __launch_bounds__(256)
gen_mul_kernel(const CwtArgs<T> A, cx<T>* __restrict__ ZW, cx<T>* __restrict__ ZD, long long r0,
               long long nr) {
  const long long n = A.n_up;
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= nr * n) return;
  const long long rl = idx / n, i = idx - rl * n;
  const long long row = r0 + rl;
  const int b = (int)(row / A.na), a = (int)(row - (long long)b * A.na);
  T p;
  if (A.wavelet == WAV_TABLE) p = A.psih_table[(long long)a * n + i];
  else {
    p = psih_eval<T>(A, a, i, A.scales[a]);
    if ((n & 1) && i == n / 2) p = p * (T)2;              // no Nyquist bin for odd n (wavelets.py:86-95)
  }
  const cx<T> z = cscale<T>(A.xh[(long long)b * n + i], p);               // Psih * xh   (_cwt.py:169)
  ZW[idx] = z;
  if (ZD) ZD[idx] = cmuli<T>(cscale<T>(z, xi_of<T>(i, n) / A.dt));          // *= 1j*xi/dt (_cwt.py:175)
}
template <typename T>
__global__ void __launch_bounds__(256)
gen_unpad_kernel(const cx<T>* __restrict__ src, cx<T>* __restrict__ dst, long long n, long long off,
                 long long Nout, long long nr, long long r0, const T* __restrict__ out_mul, int na) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= nr * Nout) return;
  const long long rl = idx / Nout, j = idx - rl * Nout;
  const T m = out_mul ? out_mul[(r0 + rl) % na] : (T)1;
  dst[(r0 + rl) * Nout + j] = cscale<T>(src[rl * n + off + j], m);
}

// =============================================================================================
// Adjoint of the CWT (backward pass of `cwt` for torch.autograd; the reference's GPU mode is
// differentiable because it is written in torch ops, ssqueezepy/_cwt.py:19,
// examples/reconstruction.py:38-70).  With P = padding, F = DFT, D_a = diag(psih_a [* 1j xi/dt]),
// U = unpadding:   Wx_a = U F^-1 D_a F P x   =>   grad_x = Re( P^T F^-1 sum_a D_a^H F U^T G_a ).
// Built on the generic-length FFT (any n_up); not a tuned path.
// =============================================================================================

// Z[r][t] = mul_a * G[row][t - off] inside [off, off + Nout), 0 elsewhere; rows r0 .. r0 + nr
template <typename T>
__global__ void __launch_bounds__(256)
adj_pad_kernel(const cx<T>* __restrict__ G, cx<T>* __restrict__ Z, long long n, long long off,
               long long Nout, long long r0, long long nr, const T* __restrict__ out_mul, int na) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= nr * n) return;
  const long long rl = idx / n, t = idx - rl * n;
  cx<T> v = mkc<T>((T)0, (T)0);
  if (t >= off && t < off + Nout) {
    const T m = out_mul ? out_mul[(r0 + rl) % na] : (T)1;
    v = cscale<T>(G[(r0 + rl) * Nout + (t - off)], m);
  }
  Z[idx] = v;
}
// acc[i] += sum_rows conj(D_a[i]) * Zh[r][i]; the chunk's rows belong to ONE signal (scales a0 ..)
template <typename T>
__global__ void __launch_bounds__(256)
adj_accum_kernel(const CwtArgs<T> A, const cx<T>* __restrict__ Zh, cx<T>* __restrict__ acc,
                 int a0, int nr, int deriv) {
  const long long n = A.n_up;
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  cx<T> s = acc[i];
  const T xi = xi_of<T>(i, n) / A.dt;
  for (int r = 0; r < nr; ++r) {
    const int a = a0 + r;
    T p;
    if (A.wavelet == WAV_TABLE) p = A.psih_table[(long long)a * n + i];
    else {
      p = psih_eval<T>(A, a, i, A.scales[a]);
      if ((n & 1) && i == n / 2) p = p * (T)2;
    }
    cx<T> z = cscale<T>(Zh[(long long)r * n + i], p);
    if (deriv) z = mkc<T>(z.y * xi, -z.x * xi);                 // conj(1j * xi / dt) = -1j xi / dt
    s = cadd<T>(s, z);
  }
  acc[i] = s;
}
template <typename T>
__global__ void __launch_bounds__(256)
adj_unpad_kernel(const cx<T>* __restrict__ g, T* __restrict__ gx, long long N, long long n, long long n1,
                 int padtype, long long B) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= B * n) return;
  const long long b = idx / n, t = idx - b * n;
  const long long src = pad_src_index(t, n1, N, padtype);
  if (src >= 0) atomicAdd(&gx[b * N + src], g[idx].x);
}

template <typename T>
struct CwtAdjoint {
  Gfft<T> fft; bool ready = false;
  DevBuf<cx<T>> Z, Zh, acc, gp;
  DevBuf<T> mul_d;
  // gW / gdW [B][na][Nout] (either may be null), gx [B][N] (overwritten)
  int run(const ssqb_cwt_desc& d, CwtArgs<T> A, const cx<T>* gW, const cx<T>* gdW, long long B,
          const double* out_mul_host, bool rpadded, T* gx, cudaStream_t st) {
    const long long n = d.n_up, Nout = rpadded ? n : d.N, off = rpadded ? 0 : d.n1;
    if (!ready) { int rc = fft.init(n); if (rc) return rc; ready = true; }
    const T* out_mul = nullptr;
    if (out_mul_host) {
      std::vector<T> m((size_t)d.na);
      for (int a = 0; a < d.na; ++a) m[a] = (T)out_mul_host[a];
      SSQB_CUDA(cudaStreamSynchronize(st));
      SSQB_CUDA(mul_d.upload(m));
      out_mul = mul_d.p;
    }
    long long chunk = ((64ll << 20) / (long long)sizeof(cx<T>)) / n; if (chunk < 1) chunk = 1;
    if (chunk > d.na) chunk = d.na;
    SSQB_CUDA(Z.ensure((size_t)chunk * (size_t)n)); SSQB_CUDA(Zh.ensure((size_t)chunk * (size_t)n));
    SSQB_CUDA(acc.ensure((size_t)B * (size_t)n)); SSQB_CUDA(gp.ensure((size_t)B * (size_t)n));
    SSQB_CUDA(cudaMemsetAsync(acc.p, 0, (size_t)B * (size_t)n * sizeof(cx<T>), st));
    SSQB_CUDA(cudaMemsetAsync(gx, 0, (size_t)B * (size_t)d.N * sizeof(T), st));
    for (long long b = 0; b < B; ++b)
      for (int pass = 0; pass < 2; ++pass) {
        const cx<T>* G = pass == 0 ? gW : gdW;
        if (!G) continue;
        for (int a0 = 0; a0 < d.na; a0 += (int)chunk) {
          const int nr = d.na - a0 < chunk ? d.na - a0 : (int)chunk;
          const long long r0 = b * d.na + a0;
          adj_pad_kernel<T><<<(unsigned)(((long long)nr * n + 255) / 256), 256, 0, st>>>(G, Z.p, n, off, Nout, r0, nr, out_mul, d.na);
          SSQB_LAUNCH_CHECK();
          int rc = fft.exec(Z.p, Zh.p, nr, -1, (T)1, st); if (rc) return rc;
          adj_accum_kernel<T><<<(unsigned)((n + 255) / 256), 256, 0, st>>>(A, Zh.p, acc.p + b * n, a0, nr, pass);
          SSQB_LAUNCH_CHECK();
        }
      }
    int rc = fft.exec(acc.p, gp.p, B, +1, (T)(1.0 / (double)n), st); if (rc) return rc;
    adj_unpad_kernel<T><<<(unsigned)((B * n + 255) / 256), 256, 0, st>>>(gp.p, gx, d.N, n, d.n1, d.padtype, B);
    SSQB_LAUNCH_CHECK();
    return 0;
  }
};


template <typename T>
struct GenericCwtPlan : public CwtPlanBase {
  ssqb_cwt_desc d;
  Gfft<T> fft;
  DevBuf<T> scales_d, out_mul_d;
  DevBuf<double> cst_d;
  DevBuf<cx<T>> xp_d, xh_d, ZW, ZD, OW, OD, dW_tmp;
  ssqb_reassign_desc rd{}; std::vector<double> rd_cst; bool have_grid = false;
  int init(const ssqb_cwt_desc* desc) {
    d = *desc;
    if (d.N < 1 || d.n1 < 0 || d.n1 + d.N > d.n_up) return set_error(SSQB_E_ARG, "bad padding geometry");
    if (d.na < 1) return set_error(SSQB_E_ARG, "na must be >= 1");
    if (d.wavelet == SSQB_WAV_TABLE && !d.psih_table_dev)
      return set_error(SSQB_E_ARG, "SSQB_WAV_TABLE needs psih_table_dev");
    std::vector<T> sc((size_t)d.na);
    for (int a = 0; a < d.na; ++a) sc[a] = (T)d.scales_host[a];
    SSQB_CUDA(scales_d.upload(sc));
    return fft.init(d.n_up);
  }
  void args(CwtArgs<T>& A) {
    memset(&A, 0, sizeof(A));
    A.N = d.N; A.n_up = d.n_up; A.n1 = d.n1; A.padtype = d.padtype; A.na = d.na;
    A.scales = scales_d.p; A.psih_table = (const T*)d.psih_table_dev; A.wavelet = d.wavelet;
    if (d.wavelet == SSQB_WAV_MORLET) {
      double mu = d.wparams[0];
      double cs = pow(1 + exp(-mu * mu) - 2 * exp(-0.75 * mu * mu), -0.5);
      A.wp[0] = (T)mu; A.wp[1] = (T)exp(-0.5 * mu * mu); A.wp[2] = (T)-0.5;
      A.wp[3] = (T)(sqrt(2.0) * cs * pow(M_PI, 0.25));
    } else if (d.wavelet == SSQB_WAV_GMW_L1) {
      double gam = d.wparams[0], bet = d.wparams[1];
      double wc = exp((1.0 / gam) * (log(bet) - log(gam)));
      T gT = (T)gam, bT = (T)bet, wcT = (T)wc, wclT = (T)log(wc);
      T wcg = (T)pow((double)wcT, (double)gT);
      A.wp[0] = gT; A.wp[1] = bT; A.wp[2] = (T)(-(bT * wclT)) + wcg;
    }
    A.dt = (T)d.dt;
  }
  int set_reassign(const ssqb_reassign_desc* r) override {
    rd = *r;
    rd_cst.assign(r->cst_host, r->cst_host + d.na);
    rd.cst_host = rd_cst.data();
    have_grid = true;
    return 0;
  }
  int exec(const void* xv, long long B, void* Wxv, void* dWxv, void* Txv, bool ssq,
           const double* out_mul_host, bool rpadded, cudaStream_t st) override {
    if (B < 1 || !xv || !Wxv) return set_error(SSQB_E_ARG, "bad arguments");
    if (ssq && (!Txv || !have_grid)) return set_error(SSQB_E_ARG, "ssq needs Tx and a reassignment grid");
    if (ssq && rpadded) return set_error(SSQB_E_ARG, "ssq works on the unpadded part");
    const long long n = d.n_up, Nout = rpadded ? n : d.N, off = rpadded ? 0 : d.n1;
    const long long rows = B * d.na;
    cx<T>* Wx = (cx<T>*)Wxv; cx<T>* dWx = (cx<T>*)dWxv;
    if (ssq && !dWx) { SSQB_CUDA(dW_tmp.ensure((size_t)rows * (size_t)Nout)); dWx = dW_tmp.p; }
    const T* out_mul = nullptr;
    if (out_mul_host) {
      std::vector<T> m((size_t)d.na);
      for (int a = 0; a < d.na; ++a) m[a] = (T)out_mul_host[a];
      SSQB_CUDA(cudaStreamSynchronize(st));
      SSQB_CUDA(out_mul_d.upload(m));
      out_mul = out_mul_d.p;
    }
    // forward transform of the (padded) signal, scaled by 1/n (the 1/n of ifft)
    SSQB_CUDA(xp_d.ensure((size_t)B * (size_t)n)); SSQB_CUDA(xh_d.ensure((size_t)B * (size_t)n));
    gen_pad_kernel<T><<<(unsigned)((B * n + 255) / 256), 256, 0, st>>>((const T*)xv, xp_d.p, d.N, n,
                                                                       d.n1, d.padtype, B);
    SSQB_LAUNCH_CHECK();
    int rc = fft.exec(xp_d.p, xh_d.p, B, -1, (T)(1.0 / (double)n), st); if (rc) return rc;
    CwtArgs<T> A; args(A); A.xh = xh_d.p;
    // rows in chunks of <= 64 MB per buffer
    long long chunk = ((64ll << 20) / (long long)sizeof(cx<T>)) / n; if (chunk < 1) chunk = 1;
    if (chunk > rows) chunk = rows;
    const bool deriv = dWx != nullptr;
    SSQB_CUDA(ZW.ensure((size_t)chunk * (size_t)n)); SSQB_CUDA(OW.ensure((size_t)chunk * (size_t)n));
    if (deriv) { SSQB_CUDA(ZD.ensure((size_t)chunk * (size_t)n)); SSQB_CUDA(OD.ensure((size_t)chunk * (size_t)n)); }
    for (long long r0 = 0; r0 < rows; r0 += chunk) {
      const long long nr = rows - r0 < chunk ? rows - r0 : chunk;
      gen_mul_kernel<T><<<(unsigned)((nr * n + 255) / 256), 256, 0, st>>>(A, ZW.p, deriv ? ZD.p : nullptr, r0, nr);
      SSQB_LAUNCH_CHECK();
      rc = fft.exec(ZW.p, OW.p, nr, +1, (T)1, st); if (rc) return rc;
      gen_unpad_kernel<T><<<(unsigned)((nr * Nout + 255) / 256), 256, 0, st>>>(OW.p, Wx, n, off, Nout, nr, r0, out_mul, d.na);
      SSQB_LAUNCH_CHECK();
      if (deriv) {
        rc = fft.exec(ZD.p, OD.p, nr, +1, (T)1, st); if (rc) return rc;
        gen_unpad_kernel<T><<<(unsigned)((nr * Nout + 255) / 256), 256, 0, st>>>(OD.p, dWx, n, off, Nout, nr, r0, out_mul, d.na);
        SSQB_LAUNCH_CHECK();
      }
    }
    if (ssq)
      return run_ssqueeze(sizeof(T) == 4 ? SSQB_F32 : SSQB_F64, Wx, dWx, Txv, B, d.na, Nout, &rd, nullptr, st);
    return 0;
  }
  int exec_host(const void* x, long long B, void* Wx, void* dWx, void* Tx, bool ssq,
                const double* out_mul_host, bool rpadded, cudaStream_t st) override {
    const long long Nout = rpadded ? d.n_up : d.N;
    const size_t nx = (size_t)B * (size_t)d.N, nout = (size_t)B * d.na * (size_t)Nout;
    DevBuf<T> xs; DevBuf<cx<T>> Ws, dWs, Ts;
    SSQB_CUDA(xs.ensure(nx)); SSQB_CUDA(Ws.ensure(nout));
    if (dWx) SSQB_CUDA(dWs.ensure(nout));
    if (ssq) SSQB_CUDA(Ts.ensure(nout));
    SSQB_CUDA(cudaMemcpyAsync(xs.p, x, nx * sizeof(T), cudaMemcpyHostToDevice, st));
    int rc = exec(xs.p, B, Ws.p, dWx ? dWs.p : nullptr, ssq ? Ts.p : nullptr, ssq, out_mul_host, rpadded, st);
    if (rc == 0) {
      SSQB_CUDA(cudaMemcpyAsync(Wx, Ws.p, nout * sizeof(cx<T>), cudaMemcpyDeviceToHost, st));
      if (dWx) SSQB_CUDA(cudaMemcpyAsync(dWx, dWs.p, nout * sizeof(cx<T>), cudaMemcpyDeviceToHost, st));
      if (ssq) SSQB_CUDA(cudaMemcpyAsync(Tx, Ts.p, nout * sizeof(cx<T>), cudaMemcpyDeviceToHost, st));
    }
    cudaError_t e = cudaStreamSynchronize(st);
    if (rc) return rc;
    SSQB_CUDA(e);
    return 0;
  }
  int debug_xh(const void* x, long long B, void* xh, cudaStream_t st) override {
    const long long n = d.n_up;
    SSQB_CUDA(xp_d.ensure((size_t)B * (size_t)n));
    gen_pad_kernel<T><<<(unsigned)((B * n + 255) / 256), 256, 0, st>>>((const T*)x, xp_d.p, d.N, n,
                                                                       d.n1, d.padtype, B);
    SSQB_LAUNCH_CHECK();
    return fft.exec(xp_d.p, (cx<T>*)xh, B, -1, (T)(1.0 / (double)n), st);
  }
  CwtAdjoint<T> adj;
  int backward(const void* gWx, const void* gdWx, long long B, const double* out_mul_host,
               bool rpadded, void* gx, cudaStream_t st) override {
    CwtArgs<T> A; args(A);
    return adj.run(d, A, (const cx<T>*)gWx, (const cx<T>*)gdWx, B, out_mul_host, rpadded, (T*)gx, st);
  }
  int set_profiling(int) override { return 0; }
  int get_profile(double* ms, long long* launches, long long* rows) override {
    for (int k = 0; k < SSQB_PROFILE_KINDS; ++k) { ms[k] = 0; launches[k] = 0; rows[k] = 0; }
    return 0;
  }
};

}  // namespace ssqb

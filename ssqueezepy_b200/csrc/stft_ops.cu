// Host dispatch of the STFT / ssq_stft kernels.
#include "host_common.h"
#include "stft_kernels.cuh"
#include "cwt_generic.cuh"      // Gfft<T>: generic-length FFT
#include <map>
#include <memory>
#include <vector>
#include <mutex>

namespace ssqb {

// Device copies of host table blobs, keyed by content and device (LRU of 16, a few KB
// each).  Entries are only ever read by kernels, so sharing them across streams is safe;
// an evicted blob is freed with cudaFree, which waits for the kernels that may still use it.
struct TableBlob { int dev; std::vector<unsigned char> bytes; unsigned char* ptr; unsigned long long tick; };
static std::mutex g_blob_mu;
static std::vector<TableBlob> g_blobs;
static unsigned long long g_blob_tick = 0;

static int table_blob(const std::vector<unsigned char>& h, cudaStream_t st, unsigned char** out) {
  int dev = 0;
  SSQB_CUDA(cudaGetDevice(&dev));
  std::lock_guard<std::mutex> lk(g_blob_mu);
  for (auto& e : g_blobs)
    if (e.dev == dev && e.bytes == h) { e.tick = ++g_blob_tick; *out = e.ptr; return 0; }
  unsigned char* p = nullptr;
  SSQB_CUDA(cudaMalloc((void**)&p, h.size() + 64));
  SSQB_CUDA(cudaMemcpyAsync(p, h.data(), h.size(), cudaMemcpyHostToDevice, st));
  SSQB_CUDA(cudaStreamSynchronize(st));                      // other streams may use it next
  if (g_blobs.size() >= 16) {
    size_t victim = 0;
    for (size_t i = 1; i < g_blobs.size(); ++i) if (g_blobs[i].tick < g_blobs[victim].tick) victim = i;
    cudaFree(g_blobs[victim].ptr);
    g_blobs.erase(g_blobs.begin() + (long)victim);
  }
  g_blobs.push_back(TableBlob{dev, h, p, ++g_blob_tick});
  *out = p;
  return 0;
}

template <typename T, bool SSQ>
static int launch_stft_pow2(const StftArgs<T>& A, int logm, cudaStream_t st) {
  long long total = (long long)A.B * A.n_hops;
  switch (logm) {
#define SSQB_S(L)                                                                         \
    case L: {                                                                             \
      constexpr int M = 1 << L; constexpr int R = Tile<T>::ELEMS / M;                     \
      size_t smem = ((size_t)M * (R + 1) + M) * sizeof(cx<T>);                            \
      auto kern = stft_pow2_kernel<T, L, SSQ>;                                            \
      SSQB_CUDA(set_smem_limit(kern, smem));                                              \
      kern<<<(unsigned)((total + R - 1) / R), Tile<T>::NT, smem, st>>>(A);                \
      SSQB_LAUNCH_CHECK();                                                                \
      return 0; }
    SSQB_S(1) SSQB_S(2) SSQB_S(3) SSQB_S(4) SSQB_S(5) SSQB_S(6) SSQB_S(7) SSQB_S(8)
    SSQB_S(9) SSQB_S(10) SSQB_S(11) SSQB_S(12)
#undef SSQB_S
    default: return -1;
  }
}

// n_fft that is not a power of two (e.g. 598 = 2 * 13 * 23, the reference's own benchmark
// size): frames -> batched mixed-radix / Bluestein FFT -> Hermitian split + epilogue, in
// chunks of frames that keep the two frame buffers below ~128 MB each.
template <typename T> struct StftGeneric {
  Gfft<T> fft; DevBuf<cx<T>> c, C;
};
static std::mutex g_gen_mu;
template <typename T> static std::map<std::pair<int, int>, std::unique_ptr<StftGeneric<T>>>& gen_cache() {
  static std::map<std::pair<int, int>, std::unique_ptr<StftGeneric<T>>> m; return m;
}
template <typename T, bool SSQ>
static int launch_stft_generic(const StftArgs<T>& A, cudaStream_t st) {
  int dev = 0; SSQB_CUDA(cudaGetDevice(&dev));
  std::lock_guard<std::mutex> lk(g_gen_mu);            // one caller at a time per process
  auto& slot = gen_cache<T>()[{dev, A.n_fft}];
  if (!slot) {
    slot.reset(new StftGeneric<T>());
    int rc = slot->fft.init(A.n_fft);
    if (rc) { slot.reset(); return rc; }
  }
  StftGeneric<T>& G = *slot;
  const long long total = (long long)A.B * A.n_hops, M = A.n_fft, nrows = M / 2 + 1;
  long long chunk = ((128ll << 20) / (long long)sizeof(cx<T>)) / M; if (chunk < 1) chunk = 1;
  if (chunk > total) chunk = total;
  SSQB_CUDA(G.c.ensure((size_t)chunk * (size_t)M)); SSQB_CUDA(G.C.ensure((size_t)chunk * (size_t)M));
  for (long long f0 = 0; f0 < total; f0 += chunk) {
    const long long nf = total - f0 < chunk ? total - f0 : chunk;
    stft_frames_kernel<T><<<(unsigned)((nf * M + 255) / 256), 256, 0, st>>>(A, G.c.p, f0, nf);
    SSQB_LAUNCH_CHECK();
    int rc = G.fft.exec(G.c.p, G.C.p, nf, -1, (T)1, st); if (rc) return rc;
    stft_emit_kernel<T, SSQ><<<(unsigned)((nf * nrows + 255) / 256), 256, 0, st>>>(A, G.C.p, f0, nf);
    SSQB_LAUNCH_CHECK();
  }
  SSQB_CUDA(cudaStreamSynchronize(st));                // buffers are shared by later callers
  return 0;
}

template <typename T>
static int stft_t(const ssqb_stft_desc* d, const ssqb_reassign_desc* r, const void* x,
                  long long B, void* Sx, void* Tx, void* dSx, bool ssq, cudaStream_t st) {
  const int M = d->n_fft, nrows = M / 2 + 1;
  StftArgs<T> A;
  memset(&A, 0, sizeof(A));
  A.N = d->N; A.n_fft = M; A.hop = d->hop; A.n1 = d->n1; A.padtype = d->padtype;
  A.modulated = d->modulated; A.B = (int)B;
  A.n_hops = (d->N - 1) / d->hop + 1;
  A.x = (const T*)x; A.Sx = (cx<T>*)Sx; A.dSx = (cx<T>*)dSx; A.Tx = (cx<T>*)Tx;
  A.write_dSx = dSx ? 1 : 0;
  const T* win = (const T*)d->win_host; const T* dwin = (const T*)d->dwin_host;
  // kappa = power of two that balances ||win|| and ||dwin||
  double nw = 0, nd = 0;
  for (int l = 0; l < M; ++l) { nw += (double)win[l] * win[l]; nd += (double)dwin[l] * dwin[l]; }
  double kap = 1.0;
  if (nd > 0 && nw > 0) kap = exp2(rint(0.5 * log2(nw / nd)));
  if (!(kap > 1e-30 && kap < 1e30)) kap = 1.0;
  A.kappa = (T)kap; A.inv_kappa = (T)(1.0 / kap);
  // device copies of the small tables: built on the host, cached on the device by content
  // (a streaming caller repeats the same window / grid thousands of times; without the
  // cache every call pays an allocation, a copy and a stream synchronisation)
  size_t tb = sizeof(T) * (size_t)(2 * M + nrows) + sizeof(cx<T>) * (size_t)M + sizeof(double) * nrows;
  std::vector<unsigned char> h(tb);
  size_t off = 0;
  auto put = [&](const void* src, size_t bytes) { memcpy(h.data() + off, src, bytes); size_t o = off; off += bytes; return o; };
  // n_fft-th roots: computed once per (length, dtype), not on every call
  static std::mutex tw_mu;
  static std::map<int, std::vector<cx<T>>> tw_cache;
  std::vector<cx<T>>* twp;
  {
    std::lock_guard<std::mutex> lk(tw_mu);
    auto it = tw_cache.find(M);
    if (it == tw_cache.end()) {
      std::vector<cx<T>> v((size_t)M);
      for (int m = 0; m < M; ++m) {
        double ang = 2.0 * M_PI * (double)m / (double)M;
        v[m] = mkc<T>((T)cos(ang), (T)sin(ang));
      }
      it = tw_cache.emplace(M, std::move(v)).first;
    }
    twp = &it->second;                       // map nodes are stable
  }
  const std::vector<cx<T>>& tw = *twp;
  std::vector<double> cst((size_t)nrows, 0.0);
  if (ssq) for (int i = 0; i < nrows; ++i) cst[i] = r->cst_host[i];
  size_t o_tw = put(tw.data(), sizeof(cx<T>) * M);          // 16-byte aligned first
  size_t o_cst = put(cst.data(), sizeof(double) * nrows);
  size_t o_win = put(win, sizeof(T) * M);
  size_t o_dwin = put(dwin, sizeof(T) * M);
  size_t o_sfs = put(d->Sfs_host, sizeof(T) * nrows);
  unsigned char* blob = nullptr;
  int rcb = table_blob(h, st, &blob); if (rcb) return rcb;
  A.tw = (const cx<T>*)(blob + o_tw); A.cst = (const double*)(blob + o_cst);
  A.win = (const T*)(blob + o_win); A.dwin = (const T*)(blob + o_dwin);
  A.Sfs = (const T*)(blob + o_sfs);
  if (ssq) {
    int rc = fill_grid(r, nrows, &A.grid); if (rc) return rc;
    A.grid.kind = 3;
    SSQB_CUDA(cudaMemsetAsync(Tx, 0, (size_t)B * nrows * (size_t)A.n_hops * sizeof(cx<T>), st));
  }
  int logm = ilog2_exact(M);
  int rc;
  if (logm >= 1 && logm <= 12 && (Tile<T>::ELEMS >> logm) >= 1)
    rc = ssq ? launch_stft_pow2<T, true>(A, logm, st) : launch_stft_pow2<T, false>(A, logm, st);
  else
    rc = ssq ? launch_stft_generic<T, true>(A, st) : launch_stft_generic<T, false>(A, st);
  return rc;
}

int run_stft(const ssqb_stft_desc* d, const ssqb_reassign_desc* r, const void* x, long long B,
             void* Sx, void* Tx, void* dSx, bool ssq, cudaStream_t st) {
  if (!d || !x || !Sx) return set_error(SSQB_E_ARG, "null pointer");
  if (!d->win_host || !d->dwin_host || !d->Sfs_host) return set_error(SSQB_E_ARG, "null table");
  if (ssq && (!r || !r->cst_host || !Tx)) return set_error(SSQB_E_ARG, "ssq needs Tx + reassign");
  if (d->N < 1 || d->n_fft < 2 || d->hop < 1 || B < 1) return set_error(SSQB_E_ARG, "bad shape");
  return d->dtype == SSQB_F32 ? stft_t<float>(d, r, x, B, Sx, Tx, dSx, ssq, st)
                              : stft_t<double>(d, r, x, B, Sx, Tx, dSx, ssq, st);
}

}  // namespace ssqb

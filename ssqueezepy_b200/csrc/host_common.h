// Host-side helpers shared by the translation units of libssq_b200.so.
#pragma once
#include <cuda_runtime.h>
#include <atomic>
#include <cstdio>
#include <cstdarg>
#include <map>
#include <mutex>
#include <string>
#include <vector>
#include <cmath>
#include "../../include/ssq_b200.h"

namespace ssqb {

extern thread_local std::string g_last_error;
extern std::atomic<long long> g_launch_count;

inline int set_error(int code, const char* fmt, ...) {
  char buf[512];
  va_list ap; va_start(ap, fmt); vsnprintf(buf, sizeof(buf), fmt, ap); va_end(ap);
  g_last_error = buf;
  return code;
}

#define SSQB_CUDA(expr)                                                          \
  do {                                                                           \
    cudaError_t _e = (expr);                                                     \
    if (_e != cudaSuccess)                                                       \
      return ::ssqb::set_error((int)_e, "%s failed: %s (%s:%d)", #expr,          \
                               cudaGetErrorString(_e), __FILE__, __LINE__);      \
  } while (0)

#define SSQB_LAUNCH_CHECK()                                                      \
  do {                                                                           \
    ::ssqb::g_launch_count.fetch_add(1, std::memory_order_relaxed);              \
    cudaError_t _e = cudaGetLastError();                                         \
    if (_e != cudaSuccess)                                                       \
      return ::ssqb::set_error((int)_e, "kernel launch failed: %s (%s:%d)",      \
                               cudaGetErrorString(_e), __FILE__, __LINE__);      \
  } while (0)

// Raises the dynamic shared-memory limit of a kernel on the current device to `bytes`, unless an
// earlier launch there set at least that much.  The attribute belongs to the device, so a process
// that launches on a second GPU sets it again there.
template <typename... Args>
inline cudaError_t set_smem_limit(void (*kern)(Args...), size_t bytes) {
  static std::mutex mu;
  static std::map<std::pair<const void*, int>, size_t> done;    // (kernel, device) -> bytes set
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  std::lock_guard<std::mutex> lk(mu);
  size_t& have = done[{reinterpret_cast<const void*>(kern), dev}];
  if (bytes <= have) return cudaSuccess;
  e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
  if (e == cudaSuccess) have = bytes;
  return e;
}

inline int ilog2_exact(long long v) {     // -1 if not a power of two
  if (v <= 0 || (v & (v - 1))) return -1;
  int l = 0; while ((1ll << l) < v) ++l; return l;
}

// owning device buffer that only ever grows
template <typename T>
struct DevBuf {
  T* p = nullptr; size_t n = 0;
  ~DevBuf() { if (p) cudaFree(p); }
  cudaError_t ensure(size_t count) {
    if (count <= n) return cudaSuccess;
    if (p) cudaFree(p);
    p = nullptr; n = 0;
    cudaError_t e = cudaMalloc((void**)&p, count * sizeof(T));
    if (e == cudaSuccess) n = count;
    return e;
  }
  cudaError_t upload(const std::vector<T>& h) {
    cudaError_t e = ensure(h.size() ? h.size() : 1);
    if (e != cudaSuccess) return e;
    return cudaMemcpy(p, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice);
  }
};

// dtype-erased interface of the CWT plan (implemented per dtype in cwt_impl.cuh)
struct CwtPlanBase {
  virtual ~CwtPlanBase() {}
  virtual int set_reassign(const ssqb_reassign_desc* r) = 0;
  virtual int exec(const void* x, long long B, void* Wx, void* dWx, void* Tx, bool ssq,
                   const double* out_mul_host, bool rpadded, cudaStream_t st) = 0;
  virtual int exec_host(const void* x, long long B, void* Wx, void* dWx, void* Tx, bool ssq,
                        const double* out_mul_host, bool rpadded, cudaStream_t st) = 0;
  virtual int debug_xh(const void* x, long long B, void* xh, cudaStream_t st) = 0;
  // adjoint of cwt: gWx / gdWx [B][na][Nout] complex (either may be null) -> gx [B][N] real
  virtual int backward(const void* gWx, const void* gdWx, long long B, const double* out_mul_host,
                       bool rpadded, void* gx, cudaStream_t st) = 0;
  virtual int set_profiling(int on) = 0;
  virtual int get_profile(double* ms, long long* launches, long long* rows) = 0;
};
CwtPlanBase* make_cwt_plan_f32(const ssqb_cwt_desc* d, int* err);
CwtPlanBase* make_cwt_plan_f64(const ssqb_cwt_desc* d, int* err);

// fills the float32 fast-path helpers of a device-side grid from the descriptor
struct ReassignGrid;
int fill_grid(const ssqb_reassign_desc* r, int n_rows, ReassignGrid* g);

// dtype-dispatched stand-alone operators (reassign_ops.cu / stft_ops.cu)
int run_ssqueeze(int dtype, const void* Wx, const void* dWx, void* Tx, long long B, int na,
                 long long N, const ssqb_reassign_desc* r, const void* Sfs, cudaStream_t st);
int run_indexed_sum(int dtype, const void* Wx, const void* w, void* Tx, long long B, int na,
                    long long N, const ssqb_reassign_desc* r, cudaStream_t st);
int run_phase(int dtype, bool stft, const void* Wx, const void* dWx, const void* Sfs, void* out,
              long long total, long long ncols, int nrows, double gamma, cudaStream_t st);
int run_stft(const ssqb_stft_desc* d, const ssqb_reassign_desc* r, const void* x, long long B,
             void* Sx, void* Tx, void* dSx, bool ssq, cudaStream_t st);
// inverse_ops.cu
int run_colsum_real(int dtype, int wide, const void* M, long long B, int na, long long N,
                    const double* div_host, double scale, int has_scale, void* out,
                    cudaStream_t st);
int run_invert_components(int dtype, const void* M, int na, long long N, const int* cc,
                          const int* cw, int K, double scale, double* out, cudaStream_t st);
int run_istft(const ssqb_istft_desc* d, const void* Sx, long long B, void* x, cudaStream_t st);
// ridge_ops.cu
int run_extract_ridges(int dtype, const void* Tf, long long B, int na, long long N, const double* ls_host,
                       const double* scales_host, double penalty, double eps, int n_ridges, int bw,
                       long long* idx_out, void* f_out, void* e_out, cudaStream_t st);

}  // namespace ssqb

// api.cu — C ABI of libb2l.so (see include/b2l.h): contexts, memory, plans and the launch logic for
// the forward (stft / spectrogram / melspectrogram / mfcc) and inverse (istft) kernels.
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <atomic>
#include <map>
#include <string>
#include <thread>
#include <vector>

#include "../../include/b2l.h"
#include "aux_kernels.cuh"
#include "common.cuh"
#include "czt_kernel.cuh"
#include "mr_kernel.cuh"
#include "feat_kernels.cuh"
#include "internal.h"
#include <complex>

using namespace b2l;

// ------------------------------------------------------------------ errors
static thread_local std::string g_last_error;

static int fail(int code, const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_last_error = buf;
  return code;
}

#define CUDA_TRY(expr)                                                                        \
  do {                                                                                        \
    cudaError_t _e = (expr);                                                                  \
    if (_e != cudaSuccess) {                                                                  \
      cudaGetLastError();                                                                     \
      return fail(_e == cudaErrorMemoryAllocation ? B2L_ERR_OOM : B2L_ERR_CUDA, "%s: %s (%s:%d)", #expr, \
                  cudaGetErrorString(_e), __FILE__, __LINE__);                                \
    }                                                                                         \
  } while (0)

// ------------------------------------------------------------------ NCCL (loaded on demand)
// Only the handful of entry points needed for the batch split / join; resolved from libnccl.so.2 with
// dlopen so that single-GPU use has no NCCL dependency.
typedef struct ncclComm* ncclComm_t;
typedef struct { char internal[128]; } ncclUniqueId;
typedef int ncclResult_t;
enum { ncclChar = 0 };
struct NcclApi {
  void* handle = nullptr;
  ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  ncclResult_t (*Broadcast)(const void*, void*, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*Send)(const void*, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*Recv)(void*, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*GroupStart)() = nullptr;
  ncclResult_t (*GroupEnd)() = nullptr;
  ncclResult_t (*AllReduce)(const void*, void*, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
  const char* (*GetErrorString)(ncclResult_t) = nullptr;
};
static NcclApi g_nccl;

static int nccl_load() {
  if (g_nccl.handle) return B2L_OK;
  const char* names[] = {"libnccl.so.2", "libnccl.so"};
  void* h = nullptr;
  for (const char* n : names) {
    h = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
    if (h) break;
  }
  if (!h) return fail(B2L_ERR_NCCL, "cannot dlopen libnccl.so.2: %s", dlerror());
#define SYM(field, name)                                                       \
  *(void**)(&g_nccl.field) = dlsym(h, name);                                   \
  if (!g_nccl.field) return fail(B2L_ERR_NCCL, "libnccl is missing %s", name);
  SYM(GetUniqueId, "ncclGetUniqueId")
  SYM(CommInitRank, "ncclCommInitRank")
  SYM(CommDestroy, "ncclCommDestroy")
  SYM(Broadcast, "ncclBroadcast")
  SYM(Send, "ncclSend")
  SYM(Recv, "ncclRecv")
  SYM(GroupStart, "ncclGroupStart")
  SYM(GroupEnd, "ncclGroupEnd")
  SYM(AllReduce, "ncclAllReduce")
  SYM(GetErrorString, "ncclGetErrorString")
#undef SYM
  g_nccl.handle = h;
  return B2L_OK;
}
#define NCCL_TRY(expr)                                                                            \
  do {                                                                                            \
    ncclResult_t _r = (expr);                                                                     \
    if (_r != 0) return fail(B2L_ERR_NCCL, "%s: %s", #expr, g_nccl.GetErrorString ? g_nccl.GetErrorString(_r) : "?"); \
  } while (0)

// ------------------------------------------------------------------ objects
struct b2l_ctx {
  int device = 0;
  int sm_count = 0;
  size_t smem_optin = 0;
  cudaStream_t stream = nullptr;
  uint64_t launches = 0;
  ncclComm_t comm = nullptr;
  int rank = 0, world = 1;
  unsigned int* d_clip_max = nullptr;   // scratch for per-clip maxima
  int* d_status = nullptr;              // bit 0: a non-finite input sample was seen since the last reset
  float* d_scratch = nullptr;           // grow-only scratch (chirp-z istft frames)
  size_t scratch_bytes = 0;
  std::map<unsigned long long, int> launch_cache;   // (kernel variant, smem) -> blocks/SM, attribute already set
  size_t clip_max_cap = 0;
  // pinned staging ring for uploads from pageable host memory (staged_h2d)
  std::vector<void*> stage_bufs;
  std::vector<cudaEvent_t> stage_evs;
};

struct b2l_event {
  cudaEvent_t ev;
  int device;
};

struct b2l_plan {
  b2l_ctx* ctx = nullptr;
  int n_fft = 0, hop = 0, center = 0, pad_mode = 0, log2m = 0;
  float* d_win_fwd = nullptr;   // window * 1/2
  float* d_win_inv = nullptr;   // window * 1/n_fft
  float2* d_tw = nullptr;
  float2* d_twn = nullptr;
  int tw_count = 0;
  // mel: band-sparse rows (bins [lo, lo+len) of each mel row); d_mel_w / d_band feed mel_project, the
  // fused kernel uses a MelRow table built per tile geometry (H rows per warp step), cached here
  int n_mels = 0, mel_w_count = 0;
  float* d_mel_w = nullptr;
  MelBand* d_band = nullptr;
  float* d_mel_wT = nullptr;     // n_mels <= 16: dense transposed weights [bin][16] (dense_project_kernel)
  std::vector<MelBand> h_band;
  std::vector<float> h_mel_w;
  struct RowTable { MelRow* d_rows = nullptr; float* d_w = nullptr; unsigned short* d_order = nullptr; int n_rows = 0, w_count = 0, list_len = 0; };
  mutable std::map<int, RowTable> row_tables;
  int power_mode = 2;
  float power = 2.0f;
  // chirp-z path for n_fft that is not a power of two (czt_kernel.cuh): transform size P = 2^log2p
  int czt = 0, log2p = 0;
  float2* d_czt_wb = nullptr;   // [n_fft] window * b
  float2* d_czt_bk = nullptr;   // [1 + n_fft/2] b
  float2* d_czt_hf = nullptr;   // [P] FFT_P(h)/P followed by the engine's inter-pass twiddles
  float2* d_czt_bfull = nullptr;   // [n_fft] b (inverse)
  float2* d_czt_wbi = nullptr;     // [n_fft] conj(b) * window / n_fft (inverse)
  // mixed-radix forward path for even n_fft whose half is 5-smooth (mr_kernel.cuh); the inverse stays chirp-z
  int mr = 0, mr_n_pass = 0, mr_tw_count = 0;
  int mr_radix[kMrMaxPass] = {0}, mr_tw_off[kMrMaxPass] = {0};
  float* d_mr_win = nullptr;       // [n_fft] window * 1/2
  float* d_mr_win_inv = nullptr;   // [n_fft] window / n_fft (inverse)
  float2* d_mr_tw = nullptr;       // pass twiddles
  float2* d_mr_twn = nullptr;      // [n_fft/4 + 1] exp(-2 pi i k / n_fft)
  // mfcc
  int n_mfcc = 0;
  float* d_dct = nullptr;
  float amin = 1e-10f, ref_value = 1.0f, top_db = 80.0f;
};

struct DeviceGuard {
  int prev = -1;
  explicit DeviceGuard(int dev) {
    cudaGetDevice(&prev);
    if (prev != dev) cudaSetDevice(dev);
    else prev = -1;
  }
  ~DeviceGuard() {
    if (prev >= 0) cudaSetDevice(prev);
  }
};

static size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// ------------------------------------------------------------------ glue for the other translation units
cudaStream_t b2l_internal_stream(b2l_ctx* c) { return c->stream; }
int b2l_internal_device(b2l_ctx* c) { return c->device; }
int* b2l_internal_status(b2l_ctx* c) { return c->d_status; }
size_t b2l_internal_smem_optin(b2l_ctx* c) { return c->smem_optin; }
int b2l_internal_sm_count(b2l_ctx* c) { return c->sm_count; }
void b2l_internal_count_launches(b2l_ctx* c, int n) { c->launches += n; }
int b2l_internal_fail(int code, const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_last_error = buf;
  return code;
}

// ------------------------------------------------------------------ library / device
extern "C" int b2l_version(void) { return B2L_VERSION; }
extern "C" const char* b2l_last_error(void) { return g_last_error.c_str(); }

extern "C" int b2l_device_count(int* count) {
  if (!count) return fail(B2L_ERR_INVALID, "count is NULL");
  CUDA_TRY(cudaGetDeviceCount(count));
  return B2L_OK;
}

extern "C" int b2l_ctx_create(int device, b2l_ctx** out) {
  if (!out) return fail(B2L_ERR_INVALID, "ctx out pointer is NULL");
  int n = 0;
  CUDA_TRY(cudaGetDeviceCount(&n));
  if (device < 0 || device >= n) return fail(B2L_ERR_INVALID, "device %d out of range (have %d)", device, n);
  cudaDeviceProp prop;
  CUDA_TRY(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10)
    return fail(B2L_ERR_UNSUPPORTED, "device %d is sm_%d%d; libb2l is built for sm_100a only (no fallback path)",
                device, prop.major, prop.minor);
  DeviceGuard g(device);
  b2l_ctx* c = new b2l_ctx();
  c->device = device;
  c->sm_count = prop.multiProcessorCount;
  c->smem_optin = prop.sharedMemPerBlockOptin;
  cudaError_t e = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = cudaMalloc((void**)&c->d_status, 256);
  if (e == cudaSuccess) e = cudaMemset(c->d_status, 0, 256);
  if (e != cudaSuccess) {
    if (c->stream) cudaStreamDestroy(c->stream);
    delete c;
    return fail(B2L_ERR_CUDA, "context setup: %s", cudaGetErrorString(e));
  }
  *out = c;
  return B2L_OK;
}

extern "C" int b2l_ctx_destroy(b2l_ctx* c) {
  if (!c) return B2L_OK;
  DeviceGuard g(c->device);
  if (c->comm && g_nccl.CommDestroy) g_nccl.CommDestroy(c->comm);
  if (c->d_clip_max) cudaFree(c->d_clip_max);
  if (c->d_status) cudaFree(c->d_status);
  if (c->d_scratch) cudaFree(c->d_scratch);
  if (c->stream) cudaStreamSynchronize(c->stream);
  for (void* b : c->stage_bufs) cudaFreeHost(b);
  for (cudaEvent_t e : c->stage_evs) cudaEventDestroy(e);
  if (c->stream) cudaStreamDestroy(c->stream);
  delete c;
  return B2L_OK;
}

extern "C" int b2l_ctx_sync(b2l_ctx* c) {
  if (!c) return fail(B2L_ERR_INVALID, "ctx is NULL");
  DeviceGuard g(c->device);
  CUDA_TRY(cudaStreamSynchronize(c->stream));
  return B2L_OK;
}
extern "C" int b2l_ctx_device(const b2l_ctx* c, int* device) {
  if (!c || !device) return fail(B2L_ERR_INVALID, "NULL argument");
  *device = c->device;
  return B2L_OK;
}
extern "C" int b2l_ctx_sm_count(const b2l_ctx* c, int* sms) {
  if (!c || !sms) return fail(B2L_ERR_INVALID, "NULL argument");
  *sms = c->sm_count;
  return B2L_OK;
}
extern "C" int b2l_ctx_launch_count(const b2l_ctx* c, uint64_t* launches) {
  if (!c || !launches) return fail(B2L_ERR_INVALID, "NULL argument");
  *launches = c->launches;
  return B2L_OK;
}

// ------------------------------------------------------------------ device-side input validation
extern "C" int b2l_status_reset(b2l_ctx* c) {
  if (!c) return fail(B2L_ERR_INVALID, "ctx is NULL");
  DeviceGuard g(c->device);
  CUDA_TRY(cudaMemsetAsync(c->d_status, 0, sizeof(int), c->stream));
  return B2L_OK;
}
extern "C" int b2l_status_read(b2l_ctx* c, int* status) {
  if (!c || !status) return fail(B2L_ERR_INVALID, "NULL argument");
  DeviceGuard g(c->device);
  CUDA_TRY(cudaMemcpyAsync(status, c->d_status, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
  CUDA_TRY(cudaStreamSynchronize(c->stream));
  return B2L_OK;
}
extern "C" int b2l_scan_finite(b2l_ctx* c, const float* d_y, int64_t n_clips, int64_t n, int64_t y_stride,
                               int64_t begin) {
  if (!c || !d_y) return fail(B2L_ERR_INVALID, "NULL argument");
  if (n_clips <= 0 || begin >= n) return B2L_OK;
  if (n > 0x7fffffffLL) return fail(B2L_ERR_UNSUPPORTED, "scan_finite: clips longer than 2^31-1 samples");
  DeviceGuard g(c->device);
  long long bx = ((n - begin) + 1023) / 1024;
  if (bx > 64) bx = 64;
  dim3 grid((unsigned)bx, (unsigned)(n_clips > 65535 ? 65535 : n_clips));
  finite_scan_kernel<<<grid, 256, 0, c->stream>>>(d_y, y_stride, (int)n, (int)(begin < 0 ? 0 : begin), n_clips,
                                                  c->d_status);
  CUDA_TRY(cudaGetLastError());
  c->launches++;
  return B2L_OK;
}

// ------------------------------------------------------------------ memory
extern "C" int b2l_alloc(b2l_ctx* c, size_t bytes, void** d_ptr) {
  if (!c || !d_ptr) return fail(B2L_ERR_INVALID, "NULL argument");
  DeviceGuard g(c->device);
  *d_ptr = nullptr;
  if (bytes == 0) bytes = 16;
  CUDA_TRY(cudaMalloc(d_ptr, bytes));
  return B2L_OK;
}
extern "C" int b2l_free(b2l_ctx* c, void* d_ptr) {
  if (!c) return fail(B2L_ERR_INVALID, "ctx is NULL");
  if (!d_ptr) return B2L_OK;
  DeviceGuard g(c->device);
  CUDA_TRY(cudaStreamSynchronize(c->stream));
  CUDA_TRY(cudaFree(d_ptr));
  return B2L_OK;
}
extern "C" int b2l_memset(b2l_ctx* c, void* d_ptr, int value, size_t bytes) {
  if (!c) return fail(B2L_ERR_INVALID, "ctx is NULL");
  DeviceGuard g(c->device);
  CUDA_TRY(cudaMemsetAsync(d_ptr, value, bytes, c->stream));
  return B2L_OK;
}
// Upload from PAGEABLE host memory (what a drop-in caller's ndarray is): cudaMemcpyAsync would stage it through
// the driver's single bounce buffer on the calling thread (10-20 GB/s).  Instead `nthreads` host threads copy
// 4 MB pieces into a ring of pinned buffers (two per thread) and enqueue the DMA of each piece on the context's
// stream as soon as it is staged, so the host-side copies run in parallel and overlap the PCIe transfer.
// Piece order on the stream is arbitrary (the pieces are disjoint); work enqueued after the call returns is
// ordered behind all of them.
static const size_t kStagePiece = 4u << 20;
static int staged_h2d(b2l_ctx* c, char* d_dst, const char* h_src, size_t bytes, int nthreads) {
  const size_t want = 2 * (size_t)nthreads;
  while (c->stage_bufs.size() < want) {
    void* b = nullptr;
    CUDA_TRY(cudaHostAlloc(&b, kStagePiece, cudaHostAllocPortable));
    c->stage_bufs.push_back(b);
    cudaEvent_t e;
    CUDA_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    c->stage_evs.push_back(e);
  }
  std::atomic<size_t> next(0);
  std::atomic<int> err(0);
  auto worker = [&](int w) {
    cudaSetDevice(c->device);
    for (int k = 0;; ++k) {
      const size_t off = next.fetch_add(1) * kStagePiece;
      if (off >= bytes || err.load()) break;
      const size_t len = std::min(kStagePiece, bytes - off);
      const int b = 2 * w + (k & 1);
      cudaError_t e = cudaEventSynchronize(c->stage_evs[b]);   // the DMA that last used this buffer is done
      if (e == cudaSuccess) {
        memcpy(c->stage_bufs[b], h_src + off, len);
        e = cudaMemcpyAsync(d_dst + off, c->stage_bufs[b], len, cudaMemcpyHostToDevice, c->stream);
      }
      if (e == cudaSuccess) e = cudaEventRecord(c->stage_evs[b], c->stream);
      if (e != cudaSuccess) err.store((int)e);
    }
  };
  std::vector<std::thread> pool;
  for (int w = 1; w < nthreads; ++w) pool.emplace_back(worker, w);
  worker(0);
  for (auto& t : pool) t.join();
  if (err.load()) {
    cudaGetLastError();
    return fail(B2L_ERR_CUDA, "staged upload: %s", cudaGetErrorString((cudaError_t)err.load()));
  }
  return B2L_OK;
}

extern "C" int b2l_h2d(b2l_ctx* c, void* d_dst, const void* h_src, size_t bytes) {
  if (!c) return fail(B2L_ERR_INVALID, "ctx is NULL");
  DeviceGuard g(c->device);
  if (bytes >= (16u << 20)) {
    static int threads = -1;   // B2L_H2D_THREADS: staging threads for pageable sources (0 = plain cudaMemcpyAsync)
    if (threads < 0) {
      const char* e = getenv("B2L_H2D_THREADS");
      threads = e && *e ? atoi(e) : 6;
      if (threads > 32) threads = 32;
    }
    cudaPointerAttributes attr;
    if (threads > 0 && cudaPointerGetAttributes(&attr, h_src) == cudaSuccess && attr.type == cudaMemoryTypeUnregistered)
      return staged_h2d(c, (char*)d_dst, (const char*)h_src, bytes, threads);
    cudaGetLastError();
  }
  CUDA_TRY(cudaMemcpyAsync(d_dst, h_src, bytes, cudaMemcpyHostToDevice, c->stream));
  return B2L_OK;
}
extern "C" int b2l_d2h(b2l_ctx* c, void* h_dst, const void* d_src, size_t bytes) {
  if (!c) return fail(B2L_ERR_INVALID, "ctx is NULL");
  DeviceGuard g(c->device);
  CUDA_TRY(cudaMemcpyAsync(h_dst, d_src, bytes, cudaMemcpyDeviceToHost, c->stream));
  return B2L_OK;
}
extern "C" int b2l_d2d(b2l_ctx* c, void* d_dst, const void* d_src, size_t bytes) {
  if (!c) return fail(B2L_ERR_INVALID, "ctx is NULL");
  DeviceGuard g(c->device);
  CUDA_TRY(cudaMemcpyAsync(d_dst, d_src, bytes, cudaMemcpyDeviceToDevice, c->stream));
  return B2L_OK;
}
extern "C" int b2l_copy2d(b2l_ctx* c, void* d_dst, size_t dst_pitch, const void* d_src, size_t src_pitch,
                          size_t width_bytes, size_t rows) {
  if (!c || !d_dst || !d_src) return fail(B2L_ERR_INVALID, "NULL argument");
  if (width_bytes == 0 || rows == 0) return B2L_OK;
  if (dst_pitch < width_bytes || src_pitch < width_bytes) return fail(B2L_ERR_INVALID, "pitch smaller than the row width");
  DeviceGuard g(c->device);
  CUDA_TRY(cudaMemcpy2DAsync(d_dst, dst_pitch, d_src, src_pitch, width_bytes, rows, cudaMemcpyDeviceToDevice, c->stream));
  return B2L_OK;
}
extern "C" int b2l_host_alloc(size_t bytes, void** h_ptr) {
  if (!h_ptr) return fail(B2L_ERR_INVALID, "NULL argument");
  if (bytes == 0) bytes = 16;
  CUDA_TRY(cudaHostAlloc(h_ptr, bytes, cudaHostAllocPortable));
  return B2L_OK;
}
extern "C" int b2l_host_free(void* h_ptr) {
  if (!h_ptr) return B2L_OK;
  CUDA_TRY(cudaFreeHost(h_ptr));
  return B2L_OK;
}
extern "C" int b2l_mem_info(b2l_ctx* c, size_t* free_bytes, size_t* total_bytes) {
  if (!c || !free_bytes || !total_bytes) return fail(B2L_ERR_INVALID, "NULL argument");
  DeviceGuard g(c->device);
  CUDA_TRY(cudaMemGetInfo(free_bytes, total_bytes));
  return B2L_OK;
}

// ------------------------------------------------------------------ events
extern "C" int b2l_event_create(b2l_ctx* c, b2l_event** ev) {
  if (!c || !ev) return fail(B2L_ERR_INVALID, "NULL argument");
  DeviceGuard g(c->device);
  b2l_event* e = new b2l_event();
  e->device = c->device;
  cudaError_t r = cudaEventCreate(&e->ev);
  if (r != cudaSuccess) {
    delete e;
    return fail(B2L_ERR_CUDA, "cudaEventCreate: %s", cudaGetErrorString(r));
  }
  *ev = e;
  return B2L_OK;
}
extern "C" int b2l_event_record(b2l_ctx* c, b2l_event* ev) {
  if (!c || !ev) return fail(B2L_ERR_INVALID, "NULL argument");
  DeviceGuard g(c->device);
  CUDA_TRY(cudaEventRecord(ev->ev, c->stream));
  return B2L_OK;
}
extern "C" int b2l_event_elapsed_ms(b2l_event* start, b2l_event* stop, float* ms) {
  if (!start || !stop || !ms) return fail(B2L_ERR_INVALID, "NULL argument");
  DeviceGuard g(stop->device);
  CUDA_TRY(cudaEventSynchronize(stop->ev));
  CUDA_TRY(cudaEventElapsedTime(ms, start->ev, stop->ev));
  return B2L_OK;
}
extern "C" int b2l_event_destroy(b2l_event* ev) {
  if (!ev) return B2L_OK;
  DeviceGuard g(ev->device);
  cudaEventDestroy(ev->ev);
  delete ev;
  return B2L_OK;
}

// ------------------------------------------------------------------ plans
static int ilog2_exact(int x) {
  int l = 0;
  while ((1 << l) < x) ++l;
  return (1 << l) == x ? l : -1;
}

template <class T>
static int upload(b2l_ctx* c, const std::vector<T>& h, T** d) {
  *d = nullptr;
  size_t bytes = h.size() * sizeof(T);
  CUDA_TRY(cudaMalloc((void**)d, bytes ? bytes : 16));
  if (bytes) CUDA_TRY(cudaMemcpy(*d, h.data(), bytes, cudaMemcpyHostToDevice));
  return B2L_OK;
}

// inter-pass twiddles of the register FFT for a complex size 2^log2m (FftCfg::tw_offset layout)
static std::vector<float2> engine_twiddles(const HostFftCfg& cfg) {
  const double two_pi = 6.283185307179586476925286766559;
  std::vector<float2> tw((size_t)cfg.tw_count());
  for (int s = 1; s < cfg.npass; ++s) {
    const int R = cfg.radix(s), pl = cfg.sublen(s), off = cfg.tw_offset(s);
    for (int r = 1; r < R; ++r)
      for (int k = 0; k < pl; ++k) {
        // exp(-2*pi*i * r*k / (p*R)); reduce the integer phase first to keep the argument small
        long long num = ((long long)r * k) % ((long long)pl * R);
        double ang = -two_pi * (double)num / (double)((long long)pl * R);
        tw[(size_t)off + (size_t)(r - 1) * pl + k] = make_float2((float)cos(ang), (float)sin(ang));
      }
  }
  return tw;
}

// in-place radix-2 FFT in double precision (host, plan construction only)
static void host_fft(std::vector<std::complex<double>>& x) {
  const size_t n = x.size();
  for (size_t i = 1, j = 0; i < n; ++i) {
    size_t bit = n >> 1;
    for (; j & bit; bit >>= 1) j ^= bit;
    j ^= bit;
    if (i < j) std::swap(x[i], x[j]);
  }
  const double pi = 3.14159265358979323846264338327950288;
  for (size_t len = 2; len <= n; len <<= 1) {
    for (size_t i = 0; i < n; i += len)
      for (size_t k = 0; k < len / 2; ++k) {
        const double ang = -2.0 * pi * (double)k / (double)len;
        const std::complex<double> w(cos(ang), sin(ang));
        const std::complex<double> u = x[i + k], v = x[i + k + len / 2] * w;
        x[i + k] = u + v;
        x[i + k + len / 2] = u - v;
      }
  }
}

extern "C" int b2l_plan_destroy(b2l_plan* p) {
  if (!p) return B2L_OK;
  DeviceGuard g(p->ctx->device);
  cudaStreamSynchronize(p->ctx->stream);
  cudaFree(p->d_win_fwd);
  cudaFree(p->d_win_inv);
  cudaFree(p->d_tw);
  cudaFree(p->d_twn);
  cudaFree(p->d_mel_w);
  cudaFree(p->d_mel_wT);
  cudaFree(p->d_czt_wb);
  cudaFree(p->d_czt_bk);
  cudaFree(p->d_czt_hf);
  cudaFree(p->d_czt_bfull);
  cudaFree(p->d_czt_wbi);
  cudaFree(p->d_mr_win);
  cudaFree(p->d_mr_win_inv);
  cudaFree(p->d_mr_tw);
  cudaFree(p->d_mr_twn);
  cudaFree(p->d_band);
  for (auto& kv : p->row_tables) {
    cudaFree(kv.second.d_rows);
    cudaFree(kv.second.d_w);
    cudaFree(kv.second.d_order);
  }
  cudaFree(p->d_dct);
  delete p;
  return B2L_OK;
}

// Radix schedule of the mixed-radix kernel for n_fft = 2 M: M = 5^c 3^b 2^a as c fives, b threes, then eights and a
// four / two.  False when n_fft is odd, M has another prime factor, or the schedule / buffers would not fit.
static bool mr_factor(int n_fft, std::vector<int>& radices) {
  radices.clear();
  if (n_fft < 12 || (n_fft & 1) || n_fft > 4096) return false;
  int m = n_fft / 2;
  while (m % 5 == 0) { radices.push_back(5); m /= 5; }
  while (m % 3 == 0) { radices.push_back(3); m /= 3; }
  while (m % 8 == 0) { radices.push_back(8); m /= 8; }
  if (m % 4 == 0) { radices.push_back(4); m /= 4; }
  if (m % 2 == 0) { radices.push_back(2); m /= 2; }
  return m == 1 && (int)radices.size() <= kMrMaxPass && !radices.empty();
}

extern "C" int b2l_plan_create(b2l_ctx* c, const b2l_plan_desc* d, b2l_plan** out) {
  if (!c || !d || !out) return fail(B2L_ERR_INVALID, "NULL argument");
  if (d->n_fft < 1) return fail(B2L_ERR_INVALID, "n_fft=%d must be positive", d->n_fft);
  if (d->hop_length < 1) return fail(B2L_ERR_INVALID, "hop_length=%d must be a positive integer", d->hop_length);
  int l2n = ilog2_exact(d->n_fft);
  int czt_log2p = 0;
  if (l2n < 0) {
    // not a power of two: Bluestein with P = next power of two >= 2*n_fft - 1 (czt_kernel.cuh)
    while ((1 << czt_log2p) < 2 * d->n_fft - 1) ++czt_log2p;
    if (czt_log2p < 5) czt_log2p = 5;
    std::vector<int> probe;
    if (d->n_fft < 3 || (czt_log2p > 12 && !mr_factor(d->n_fft, probe)))
      return fail(B2L_ERR_UNSUPPORTED,
                  "n_fft=%d: non-power-of-two sizes are supported from 3 to 2047, and even sizes up to 4096 whose half "
                  "has no prime factor above 5 (no CPU fallback)", d->n_fft);
  } else if (l2n - 1 < kMinLog2M || l2n - 1 > kMaxLog2M) {
    return fail(B2L_ERR_UNSUPPORTED,
                "n_fft=%d: the sm_100a kernels are built for powers of two from %d to %d (no CPU fallback)",
                d->n_fft, 2 << kMinLog2M, 2 << kMaxLog2M);
  }
  if (!d->h_window) return fail(B2L_ERR_INVALID, "window is NULL");
  if (d->pad_mode < 0 || d->pad_mode > B2L_PAD_EMPTY) return fail(B2L_ERR_INVALID, "bad pad_mode %d", d->pad_mode);
  if (d->n_mels < 0 || d->n_mfcc < 0) return fail(B2L_ERR_INVALID, "negative n_mels / n_mfcc");
  if (d->n_mels > 0 && !d->h_mel_basis) return fail(B2L_ERR_INVALID, "mel basis is NULL");
  if (d->n_mfcc > 0 && (!d->h_dct_basis || d->n_mels == 0))
    return fail(B2L_ERR_INVALID, "mfcc stage needs a mel stage and a DCT basis");
  if (d->n_mfcc > 0 && !(d->amin > 0.0f)) return fail(B2L_ERR_INVALID, "amin must be strictly positive");

  DeviceGuard g(c->device);
  b2l_plan* p = new b2l_plan();
  p->ctx = c;
  p->n_fft = d->n_fft;
  p->hop = d->hop_length;
  p->center = d->center ? 1 : 0;
  p->pad_mode = d->pad_mode;
  p->log2m = l2n - 1;
  p->power = d->power;
  p->power_mode = d->power == 2.0f ? 2 : (d->power == 1.0f ? 1 : 0);
  p->amin = d->amin;
  p->ref_value = d->ref_value;
  p->top_db = d->top_db;
  const int N = d->n_fft, M = N / 2;
  int rc = B2L_OK;
  if (l2n < 0) {
    // ---- chirp-z tables (double precision on the host)
    p->czt = 1;
    p->log2p = czt_log2p;
    p->log2m = -1;
    const int L = N, P = 1 << czt_log2p;
    const double pi = 3.14159265358979323846264338327950288;
    if (czt_log2p > 12) p->log2p = 0;   // beyond the chirp-z range: the mixed-radix kernels alone serve this size
    if (czt_log2p <= 12) {
    std::vector<std::complex<double>> b(L);
    for (int n = 0; n < L; ++n) {
      const long long q = ((long long)n * n) % (2LL * L);          // n^2 mod 2L keeps the phase exact
      const double ang = -pi * (double)q / (double)L;
      b[n] = std::complex<double>(cos(ang), sin(ang));
    }
    std::vector<float2> wb(L), bk(L / 2 + 1);
    for (int n = 0; n < L; ++n) {
      const std::complex<double> z = d->h_window[n] * b[n];
      wb[n] = make_float2((float)z.real(), (float)z.imag());
    }
    for (int k = 0; k <= L / 2; ++k) bk[k] = make_float2((float)b[k].real(), (float)b[k].imag());
    std::vector<std::complex<double>> h(P, std::complex<double>(0.0, 0.0));
    h[0] = std::conj(b[0]);
    for (int m = 1; m < L; ++m) h[m] = h[P - m] = std::conj(b[m]);
    host_fft(h);
    HostFftCfg ccfg(czt_log2p);
    std::vector<float2> hf((size_t)P);
    for (int i = 0; i < P; ++i) hf[i] = make_float2((float)(h[i].real() / P), (float)(h[i].imag() / P));
    std::vector<float2> tw = engine_twiddles(ccfg);
    hf.insert(hf.end(), tw.begin(), tw.end());
    std::vector<float2> bfull(L), wbi(L);
    for (int n = 0; n < L; ++n) {
      bfull[n] = make_float2((float)b[n].real(), (float)b[n].imag());
      const std::complex<double> z = std::conj(b[n]) * (d->h_window[n] / (double)L);
      wbi[n] = make_float2((float)z.real(), (float)z.imag());
    }
    if ((rc = upload(c, wb, &p->d_czt_wb)) || (rc = upload(c, bk, &p->d_czt_bk)) || (rc = upload(c, hf, &p->d_czt_hf)) ||
        (rc = upload(c, bfull, &p->d_czt_bfull)) || (rc = upload(c, wbi, &p->d_czt_wbi)))
      goto bad;
    }
    // ---- mixed-radix tables when n_fft = 2 M with M = 2^a 3^b 5^c (odd radices first, see mr_kernel.cuh)
    {
      std::vector<int> radices;
      if (mr_factor(N, radices)) {
        p->mr = 1;
        p->mr_n_pass = (int)radices.size();
        std::vector<float2> tw;
        int sub = 1;
        for (int s = 0; s < p->mr_n_pass; ++s) {
          const int R = radices[s];
          p->mr_radix[s] = R;
          p->mr_tw_off[s] = (int)tw.size();
          if (sub > 1)
            for (int r = 1; r < R; ++r)
              for (int k = 0; k < sub; ++k) {
                const long long num = ((long long)r * k) % ((long long)sub * R);
                const double ang = -2.0 * pi * (double)num / (double)((long long)sub * R);
                tw.push_back(make_float2((float)cos(ang), (float)sin(ang)));
              }
          sub *= R;
        }
        if (tw.empty()) tw.push_back(make_float2(1.0f, 0.0f));
        p->mr_tw_count = (int)tw.size();
        std::vector<float> wf(N), wi(N);
        for (int i = 0; i < N; ++i) {
          wf[i] = (float)(d->h_window[i] * 0.5);
          wi[i] = (float)(d->h_window[i] / (double)N);
        }
        std::vector<float2> twn((size_t)M / 2 + 1);
        for (int k = 0; k <= M / 2; ++k) {
          const double ang = -2.0 * pi * (double)k / (double)N;
          twn[k] = make_float2((float)cos(ang), (float)sin(ang));
        }
        if ((rc = upload(c, wf, &p->d_mr_win)) || (rc = upload(c, wi, &p->d_mr_win_inv)) || (rc = upload(c, tw, &p->d_mr_tw)) ||
            (rc = upload(c, twn, &p->d_mr_twn)))
          goto bad;
      }
    }
  } else {
    HostFftCfg cfg(p->log2m);
    {
      std::vector<float> wf(N), wi(N);
      for (int i = 0; i < N; ++i) {
        wf[i] = (float)(d->h_window[i] * 0.5);
        wi[i] = (float)(d->h_window[i] / (double)N);
      }
      if ((rc = upload(c, wf, &p->d_win_fwd)) || (rc = upload(c, wi, &p->d_win_inv))) goto bad;
    }
    {
      const double two_pi = 6.283185307179586476925286766559;
      std::vector<float2> tw = engine_twiddles(cfg);
      p->tw_count = cfg.tw_count();
      std::vector<float2> twn((size_t)M / 2 + 1);
      for (int k = 0; k <= M / 2; ++k) {
        double ang = -two_pi * (double)k / (double)N;
        twn[k] = make_float2((float)cos(ang), (float)sin(ang));
      }
      if ((rc = upload(c, tw, &p->d_tw)) || (rc = upload(c, twn, &p->d_twn))) goto bad;
    }
  }
  if (d->n_mels > 0) {
    const int F = M + 1;
    std::vector<MelBand> bands(d->n_mels);
    std::vector<float> w;
    for (int m = 0; m < d->n_mels; ++m) {
      const float* row = d->h_mel_basis + (size_t)m * F;
      int lo = -1, hi = -1;
      for (int k = 0; k < F; ++k)
        if (row[k] != 0.0f) {
          if (lo < 0) lo = k;
          hi = k;
        }
      MelBand b;
      b.off = (int)w.size();
      b.pad = 0;
      if (lo < 0) {
        b.lo = 0;
        b.len = 0;
      } else {
        b.lo = lo;
        b.len = hi - lo + 1;
        w.insert(w.end(), row + lo, row + hi + 1);
      }
      bands[m] = b;
    }
    p->n_mels = d->n_mels;
    p->mel_w_count = (int)w.size();
    p->h_band = bands;
    p->h_mel_w = w;
    if ((rc = upload(c, w, &p->d_mel_w)) || (rc = upload(c, bands, &p->d_band))) goto bad;
    if (d->n_mels <= 16) {
      std::vector<float> wT((size_t)F * 16, 0.0f);
      for (int m = 0; m < d->n_mels; ++m)
        for (int k = 0; k < F; ++k) wT[(size_t)k * 16 + m] = d->h_mel_basis[(size_t)m * F + k];
      if ((rc = upload(c, wT, &p->d_mel_wT))) goto bad;
    }
  }
  if (d->n_mfcc > 0) {
    // transposed and zero padded to 8-coefficient groups: dctT[m][8*KG] (dct_clamp4_kernel)
    const int KP = (d->n_mfcc + 7) / 8 * 8;
    std::vector<float> dct((size_t)d->n_mels * KP, 0.0f);
    for (int k = 0; k < d->n_mfcc; ++k)
      for (int m = 0; m < d->n_mels; ++m) dct[(size_t)m * KP + k] = d->h_dct_basis[(size_t)k * d->n_mels + m];
    p->n_mfcc = d->n_mfcc;
    if ((rc = upload(c, dct, &p->d_dct))) goto bad;
  }
  *out = p;
  return B2L_OK;
bad:
  b2l_plan_destroy(p);
  return rc;
}

static long long plan_frames(const b2l_plan* p, long long n) {
  long long padded = n + (p->center ? 2LL * (p->n_fft / 2) : 0);
  if (padded < p->n_fft) return 0;
  return 1 + (padded - p->n_fft) / p->hop;
}

extern "C" int b2l_plan_n_frames(const b2l_plan* p, int64_t n, int64_t* n_frames) {
  if (!p || !n_frames) return fail(B2L_ERR_INVALID, "NULL argument");
  *n_frames = plan_frames(p, n);
  return B2L_OK;
}

// ------------------------------------------------------------------ forward launches
typedef cudaError_t (*fwd_op_fn)(int, int, int, const FwdArgs*, int, size_t, cudaStream_t, int*);
typedef cudaError_t (*inv_op_fn)(int, int, const InvArgs*, int, size_t, cudaStream_t, int*);
static fwd_op_fn fwd_table(int log2m) {
  switch (log2m) {
    case 2: return fwd_op_2; case 3: return fwd_op_3; case 4: return fwd_op_4; case 5: return fwd_op_5;
    case 6: return fwd_op_6; case 7: return fwd_op_7; case 8: return fwd_op_8; case 9: return fwd_op_9;
    case 10: return fwd_op_10; case 11: return fwd_op_11; case 12: return fwd_op_12;
  }
  return nullptr;
}
static inv_op_fn inv_table(int log2m) {
  switch (log2m) {
    case 2: return inv_op_2; case 3: return inv_op_3; case 4: return inv_op_4; case 5: return inv_op_5;
    case 6: return inv_op_6; case 7: return inv_op_7; case 8: return inv_op_8; case 9: return inv_op_9;
    case 10: return inv_op_10; case 11: return inv_op_11; case 12: return inv_op_12;
  }
  return nullptr;
}

static int ensure_clip_max(b2l_ctx* c, size_t n_clips) {
  if (c->clip_max_cap < n_clips) {
    if (c->d_clip_max) {
      CUDA_TRY(cudaStreamSynchronize(c->stream));
      CUDA_TRY(cudaFree(c->d_clip_max));
      c->d_clip_max = nullptr;
      c->clip_max_cap = 0;
    }
    size_t cap = n_clips < 1024 ? 1024 : n_clips;
    CUDA_TRY(cudaMalloc((void**)&c->d_clip_max, cap * sizeof(unsigned int)));
    c->clip_max_cap = cap;
  }
  return B2L_OK;
}

// MelRow table for warps that process H mel rows at a time (see MelRow / MelLayout in common.cuh), plus the
// work-item lists of the `hw` warps of a half: items dealt round-robin in row order, which keeps neighbouring
// rows (whose bands overlap in shared memory) on warps that run at the same time.
static int get_row_table(b2l_ctx* c, const b2l_plan* p, int H, int hw, const b2l_plan::RowTable** out) {
  const int key = H * 64 + hw;
  auto it = p->row_tables.find(key);
  if (it != p->row_tables.end()) {
    *out = &it->second;
    return B2L_OK;
  }
  const int rsm = H < 4 ? 4 : H, G = rsm / 4;   // row starts: lo_j == 4*(j mod G) (mod rsm)
  const int n_rows = (p->n_mels + H - 1) / H * H;
  const int n_items = n_rows / H;
  std::vector<MelRow> rows(n_rows);
  std::vector<float> w;
  for (int item = 0; item < n_items; ++item) {
    std::vector<int> start(H), lenp(H);
    int quads = 0;
    for (int j = 0; j < H; ++j) {
      const int m = item * H + j;
      if (m < p->n_mels && p->h_band[m].len > 0) {
        const MelBand& b = p->h_band[m];
        const int want = 4 * (j % G);
        int st = b.lo - ((((b.lo - want) % rsm) + rsm) % rsm);   // largest bin <= lo congruent to `want` mod rsm
        if (st < 0) st = b.lo - (b.lo % 4);                       // lowest rows: keep the 16-byte alignment only
        start[j] = st;
        lenp[j] = b.lo + b.len - st;
      } else {
        start[j] = 4 * (j % G);
        lenp[j] = 0;
      }
      quads = std::max(quads, (lenp[j] + 3) / 4);
    }
    for (int j = 0; j < H; ++j) {
      const int m = item * H + j;
      MelRow r;
      r.lo = (unsigned short)start[j];
      r.quads = (unsigned short)quads;
      r.off = (unsigned int)w.size();
      size_t base = w.size();
      w.resize(base + (size_t)4 * quads, 0.0f);
      if (lenp[j] > 0) {
        const MelBand& b = p->h_band[m];
        for (int i = 0; i < b.len; ++i) w[base + (b.lo - start[j]) + i] = p->h_mel_w[b.off + i];
      }
      rows[m] = r;
    }
  }
  std::vector<std::vector<int>> lists(hw);
  for (int i = 0; i < n_items; ++i) lists[i % hw].push_back(i);
  size_t list_len = 0;
  for (auto& l : lists) list_len = std::max(list_len, l.size());
  std::vector<unsigned short> order(list_len * hw, (unsigned short)0xffff);
  for (int wv = 0; wv < hw; ++wv)
    for (size_t k = 0; k < lists[wv].size(); ++k) order[k * hw + wv] = (unsigned short)lists[wv][k];
  if (order.empty()) order.push_back(0xffff);
  b2l_plan::RowTable t;
  t.n_rows = n_rows;
  t.w_count = (int)w.size();
  t.list_len = (int)list_len;
  int rc;
  if ((rc = upload(c, rows, &t.d_rows)) || (rc = upload(c, w, &t.d_w)) || (rc = upload(c, order, &t.d_order))) return rc;
  auto ins = p->row_tables.emplace(key, t);
  *out = &ins.first->second;
  return B2L_OK;
}

// Kernel variants tried in order (first that fits shared memory wins): 116 = 16 warps as two independent
// 8-warp halves, 16 / 8 = plain CTAs.  B2L_FWD_VARIANT forces one (A/B measurements).
#ifndef B2L_TMEM_DEFAULT
#define B2L_TMEM_DEFAULT true
#endif
static int fwd_variants(const HostFftCfg& cfg, int out[6]) {
  int n = 0;
  const char* force = getenv("B2L_FWD_VARIANT");
  if (force && *force) {
    out[n++] = atoi(force);
    return n;
  }
  // + 1000: window / twiddle tables in Tensor Memory (B2L_TMEM=0 keeps them in shared memory)
  const char* tm_env = getenv("B2L_TMEM");
  const bool tm = tm_env && *tm_env ? atoi(tm_env) != 0 : B2L_TMEM_DEFAULT;
  if (cfg.log2m >= 9 && cfg.log2m <= 11) {
    if (tm) out[n++] = 1116;
    out[n++] = 116;
  }
  if (tm && cfg.log2m == 12) out[n++] = 1016;
  int nws[2];
  const int k = cfg.nw_options(nws);
  for (int i = 0; i < k; ++i) out[n++] = nws[i];
  return n;
}

struct StatsCall { StatsParams sp; const float* d_freq; };

static int run_forward(b2l_ctx* c, const b2l_plan* p, int mode, int log_mode, const float* d_y, int64_t n_clips,
                       int64_t n, int64_t y_stride, float2* out_c, float* out_r, const StatsCall* stats = nullptr) {
  if (!c || !p) return fail(B2L_ERR_INVALID, "NULL ctx / plan");
  if (p->ctx != c) return fail(B2L_ERR_INVALID, "plan belongs to another context");
  if (n_clips < 0 || n < 0 || y_stride < n) return fail(B2L_ERR_INVALID, "bad clip geometry");
  if (n > 0x7fffffffLL) return fail(B2L_ERR_UNSUPPORTED, "clips longer than 2^31-1 samples are not supported");
  const long long T = plan_frames(p, n);
  if (T <= 0)
    return fail(B2L_ERR_INVALID, "n_fft=%d is too large for input signal of length=%lld", p->n_fft, (long long)n);
  if (n_clips == 0) return B2L_OK;
  if (!d_y || (mode == MODE_STFT ? (void*)out_c : (void*)out_r) == nullptr)
    return fail(B2L_ERR_INVALID, "NULL device pointer");
  if (mode == MODE_MEL && p->n_mels == 0) return fail(B2L_ERR_INVALID, "plan has no mel stage");
  DeviceGuard g(c->device);

  HostFftCfg cfg(p->log2m);
  const int N = p->n_fft, M = N / 2;
  fwd_op_fn op = fwd_table(p->log2m);
  int variants[6];
  const int n_opt = fwd_variants(cfg, variants);
  FwdArgs a;
  memset(&a, 0, sizeof(a));
  int variant = 0, ft = 0, halves = 1;
  size_t smem = 0;
  const b2l_plan::RowTable* rt = nullptr;
  for (int i = 0; i < n_opt && !variant; ++i) {
    const int v = variants[i];
    const bool tmem = v >= 1000;
    const int nh = (v % 1000) == 116 ? 2 : 1;
    const int nw = nh > 1 ? 16 : v % 1000;
    if (nw * 32 % (cfg.tpf * nh) != 0) continue;
    const int f = nw * 32 / nh / cfg.tpf;
    if (f < 1 || f > 32) continue;
    const long long span = (long long)(f - 1) * p->hop + N;
    if (span > 0x3fffffff) continue;
    const b2l_plan::RowTable* t = nullptr;
    if (mode == MODE_MEL) {
      int rc = get_row_table(c, p, mel_rows_per_warp(f), nw / nh, &t);
      if (rc) return rc;
    }
    size_t off = 0;
    a.off_win = (int)off; if (!tmem) off = align_up(off + (size_t)N * 4, 16);       // TMEM variants keep these
    a.off_tw = (int)off; if (!tmem) off = align_up(off + (size_t)cfg.tw_count() * 8, 16);   // tables off shared memory
    a.off_bar = (int)off; off = align_up(off + 64, 16);   // "tile landed" mbarrier per half, TMEM base address, one more mbarrier per half (initialised only)
    if (t) {
      a.off_melw = (int)off; off = align_up(off + (size_t)t->w_count * 4, 16);
      a.off_melband = (int)off; off = align_up(off + (size_t)t->n_rows * sizeof(MelRow), 16);
      a.off_melorder = (int)off; off = align_up(off + (size_t)std::max(1, t->list_len) * (nw / nh) * 2, 16);
    }
    if (mode == MODE_STATS) {   // bin frequencies take the place of the mel weights
      a.off_melw = (int)off; off = align_up(off + (size_t)(M + 1) * 4, 16);
    }
    a.off_in = (int)(off = align_up(off, 128));
    a.in_stride = (int)align_up((size_t)span * 4, 128);
    off += (size_t)a.in_stride * nh;
    a.off_xbuf = (int)(off = align_up(off, 128));
    size_t xbytes = (size_t)f * cfg.xbuf_f2() * 8;
    if (mode == MODE_MEL || mode == MODE_STATS) {
      // the power row of a frame lives in the (padded) exchange region of its group: MelLayout (common.cuh);
      // slack after the last row: a short row of a work item may read up to one band length past bin M + 3
      // (only possible when 2 * GS < 2 * M + 8, i.e. M < 128)
      xbytes = (size_t)f * mel_group_stride(M, f) * 8 + (M < 128 ? (size_t)(M + 16) * 4 : 0);
    }
    a.xbuf_stride = (int)align_up(xbytes, 128);
    off += (size_t)a.xbuf_stride * nh;
    if (off > c->smem_optin) continue;
    variant = v;
    ft = f;
    halves = nh;
    smem = off;
    rt = t;
    a.in_floats = (int)span;
  }
  if (!variant)
    return fail(B2L_ERR_UNSUPPORTED, "hop_length=%d with n_fft=%d needs more shared memory than one SM has", p->hop,
                p->n_fft);

  a.y = d_y;
  a.clip_stride = y_stride;
  a.n = (int)n;
  a.n_clips = (int)n_clips;
  a.n_fft = N;
  a.hop = p->hop;
  a.pad = p->center ? N / 2 : 0;
  a.pad_mode = p->pad_mode;
  a.n_frames = (int)T;
  a.tiles_per_clip = (int)((T + ft - 1) / ft);
  a.total_tiles = (long long)a.tiles_per_clip * n_clips;
  a.tma_ok = (((uintptr_t)d_y & 15) == 0) && (y_stride % 4 == 0) && (a.in_floats % 4 == 0);
  a.window = p->d_win_fwd;
  a.tw = p->d_tw;
  a.twn = p->d_twn;
  a.out_c = out_c;
  a.out_r = out_r;
  a.power_mode = p->power_mode;
  a.power = p->power;
  a.n_mels = p->n_mels;
  if (mode == MODE_STATS) {
    if (!stats || !stats->d_freq) return fail(B2L_ERR_INVALID, "NULL frequency table");
    a.power_mode = 1;          // the statistics are defined on the magnitude |X|
    a.power = 1.0f;
    a.stats = stats->sp;
    a.mel_w = stats->d_freq;
    a.mel_w_count = M + 1;
  }
  if (rt) {
    a.mel_w_count = rt->w_count;
    a.mel_w = rt->d_w;
    a.mel_rows = rt->d_rows;
    a.n_mel_rows = rt->n_rows;
    a.mel_order = rt->d_order;
    a.mel_list_len = rt->list_len;
  }
  a.log_mode = log_mode ? 1 : 0;
  a.out_tiled = log_mode == 2 ? 1 : 0;   // b2l_mfcc: log-mel goes to the tiled scratch
  a.amin = p->amin;
  a.db_sub = 10.0f * log10f(fmaxf(p->amin, fabsf(p->ref_value)));
  a.clip_max = c->d_clip_max;
  a.status = c->d_status;

  // cudaFuncSetAttribute + the occupancy query cost tens of microseconds: raise the kernel's dynamic
  // shared-memory limit to the device maximum once per kernel, cache blocks/SM per (kernel, smem)
  const unsigned long long kkey = ((unsigned long long)p->log2m << 56) | ((unsigned long long)variant << 44) |
                                  ((unsigned long long)mode << 40);
  if (c->launch_cache.find(kkey) == c->launch_cache.end()) {
    CUDA_TRY(op(OP_SET_SMEM, variant, mode, &a, 0, c->smem_optin, c->stream, nullptr));
    c->launch_cache[kkey] = 1;
  }
  int occ = 0;
  auto hit = c->launch_cache.find(kkey | (unsigned long long)smem);
  if (hit != c->launch_cache.end()) {
    occ = hit->second;
  } else {
    CUDA_TRY(op(OP_OCCUPANCY, variant, mode, &a, 0, smem, c->stream, &occ));
    c->launch_cache[kkey | (unsigned long long)smem] = occ;
  }
  if (occ < 1) return fail(B2L_ERR_CUDA, "forward kernel does not fit on an SM (smem %zu)", smem);
  long long grid = (long long)c->sm_count * occ;
  const long long ctas_needed = (a.total_tiles + halves - 1) / halves;
  if (grid > ctas_needed) grid = ctas_needed;
  CUDA_TRY(op(OP_LAUNCH, variant, mode, &a, (int)grid, smem, c->stream, nullptr));
  c->launches++;
  return B2L_OK;
}

// ------------------------------------------------------------------ chirp-z launch (n_fft not a power of two)
typedef cudaError_t (*czt_op_fn)(int, const CztArgs*, int, size_t, cudaStream_t, int*);
static czt_op_fn czt_table(int log2p) {
  switch (log2p) {
    case 5: return czt_op_5; case 6: return czt_op_6; case 7: return czt_op_7; case 8: return czt_op_8;
    case 9: return czt_op_9; case 10: return czt_op_10; case 11: return czt_op_11; case 12: return czt_op_12;
  }
  return nullptr;
}

typedef cudaError_t (*czt_inv_op_fn)(int, const CztInvArgs*, int, size_t, cudaStream_t, int*);
static czt_inv_op_fn czt_inv_table(int log2p) {
  switch (log2p) {
    case 5: return czt_inv_op_5; case 6: return czt_inv_op_6; case 7: return czt_inv_op_7; case 8: return czt_inv_op_8;
    case 9: return czt_inv_op_9; case 10: return czt_inv_op_10; case 11: return czt_inv_op_11; case 12: return czt_inv_op_12;
  }
  return nullptr;
}

static int run_czt(b2l_ctx* c, const b2l_plan* p, int mode, const float* d_y, int64_t n_clips, int64_t n,
                   int64_t y_stride, float2* out_c, float* out_r) {
  if (p->ctx != c) return fail(B2L_ERR_INVALID, "plan belongs to another context");
  if (n_clips < 0 || n < 0 || y_stride < n) return fail(B2L_ERR_INVALID, "bad clip geometry");
  if (n > 0x7fffffffLL) return fail(B2L_ERR_UNSUPPORTED, "clips longer than 2^31-1 samples are not supported");
  const long long T = plan_frames(p, n);
  if (T <= 0)
    return fail(B2L_ERR_INVALID, "n_fft=%d is too large for input signal of length=%lld", p->n_fft, (long long)n);
  if (n_clips == 0) return B2L_OK;
  if (!d_y || (mode == 0 ? (void*)out_c : (void*)out_r) == nullptr) return fail(B2L_ERR_INVALID, "NULL device pointer");
  DeviceGuard g(c->device);
  HostFftCfg cfg(p->log2p);
  const int nw = cfg.czt_nw();
  const int G = nw * 32 / cfg.tpf;
  CztArgs a;
  memset(&a, 0, sizeof(a));
  a.y = d_y;
  a.clip_stride = y_stride;
  a.n = (int)n;
  a.n_clips = (int)n_clips;
  a.L = p->n_fft;
  a.hop = p->hop;
  a.pad = p->center ? p->n_fft / 2 : 0;
  a.pad_mode = p->pad_mode;
  a.n_frames = (int)T;
  a.n_bins = 1 + p->n_fft / 2;
  a.wb = p->d_czt_wb;
  a.bk = p->d_czt_bk;
  a.hf = p->d_czt_hf;
  a.out_c = out_c;
  a.out_r = out_r;
  a.mode = mode;
  a.power_mode = p->power_mode;
  a.power = p->power;
  a.status = c->d_status;
  const size_t smem = (size_t)((cfg.tw_count() + 15) & ~15) * 8 + (size_t)G * cfg.xbuf_f2() * 8 +
                      ((size_t)(1 << p->log2p) + (size_t)((p->n_fft + 1) & ~1) + (size_t)a.n_bins) * 8;   // + the three tables
  czt_op_fn op = czt_table(p->log2p);
  const unsigned long long kkey = (1ULL << 63) | ((unsigned long long)p->log2p << 40);
  int occ = 0;
  auto hit = c->launch_cache.find(kkey);
  if (hit != c->launch_cache.end()) {
    occ = hit->second;
  } else {
    // the table part of the shared memory depends on n_fft, not only on P: allow the device maximum once and
    // size the grid for the largest case (the kernels run one block per SM anyway)
    CUDA_TRY(op(OP_SET_SMEM, &a, 0, c->smem_optin, c->stream, nullptr));
    CUDA_TRY(op(OP_OCCUPANCY, &a, 0, c->smem_optin / 2 + 1, c->stream, &occ));
    c->launch_cache[kkey] = occ;
  }
  if (smem > c->smem_optin) return fail(B2L_ERR_UNSUPPORTED, "n_fft=%d needs more shared memory than one SM has", p->n_fft);
  if (occ < 1) return fail(B2L_ERR_CUDA, "chirp-z kernel does not fit on an SM (smem %zu)", smem);
  const long long steps = ((long long)n_clips * ((T + 1) / 2) + G - 1) / G;   // frames go in pairs inside a clip
  long long grid = (long long)c->sm_count * occ;
  if (grid > steps) grid = steps;
  CUDA_TRY(op(OP_LAUNCH, &a, (int)grid, smem, c->stream, nullptr));
  c->launches++;
  return B2L_OK;
}

// ------------------------------------------------------------------ mixed-radix launch (even n_fft, 5-smooth half)
// mode 0: complex STFT, 1: |X|^power, 2: mel (log_mode 1: dB values + per-clip maximum for mfcc)
// frames per warp of mr_kernel: 2 (16 lanes each) for short frames, else 1; B2L_MR_LANES = 16 / 32 forces one (A/B)
static int mr_frames_per_warp(int M) {
  int lanes = M <= 512 ? 16 : 32;
  const char* e = getenv("B2L_MR_LANES");
  if (e && *e && (atoi(e) == 16 || atoi(e) == 32)) lanes = atoi(e);
  return 32 / lanes;
}
static bool mr_enabled(const b2l_plan* p) {
  if (p->log2p == 0) return true;   // no chirp-z tables for this size
  const char* e = getenv("B2L_MR");
  return !(e && *e) || atoi(e) != 0;
}
static int run_mr(b2l_ctx* c, const b2l_plan* p, int mode, int log_mode, const float* d_y, int64_t n_clips, int64_t n,
                  int64_t y_stride, float2* out_c, float* out_r) {
  if (p->ctx != c) return fail(B2L_ERR_INVALID, "plan belongs to another context");
  if (n_clips < 0 || n < 0 || y_stride < n) return fail(B2L_ERR_INVALID, "bad clip geometry");
  if (n > 0x7fffffffLL) return fail(B2L_ERR_UNSUPPORTED, "clips longer than 2^31-1 samples are not supported");
  const long long T = plan_frames(p, n);
  if (T <= 0)
    return fail(B2L_ERR_INVALID, "n_fft=%d is too large for input signal of length=%lld", p->n_fft, (long long)n);
  if (n_clips == 0) return B2L_OK;
  if (!d_y || (mode == 0 ? (void*)out_c : (void*)out_r) == nullptr) return fail(B2L_ERR_INVALID, "NULL device pointer");
  if (mode == 2 && p->n_mels == 0) return fail(B2L_ERR_INVALID, "plan has no mel stage");
  if (n_clips > 0x7fffffffLL || T > 0x7fffffffLL) return fail(B2L_ERR_UNSUPPORTED, "batch too large");
  DeviceGuard g(c->device);
  MrArgs a;
  memset(&a, 0, sizeof(a));
  a.y = d_y;
  a.clip_stride = y_stride;
  a.n = (int)n;
  a.n_clips = (int)n_clips;
  a.L = p->n_fft;
  a.M = p->n_fft / 2;
  a.hop = p->hop;
  a.pad = p->center ? p->n_fft / 2 : 0;
  a.pad_mode = p->pad_mode;
  a.n_frames = (int)T;
  a.n_bins = 1 + p->n_fft / 2;
  a.n_pass = p->mr_n_pass;
  for (int s = 0; s < p->mr_n_pass; ++s) {
    a.radix[s] = p->mr_radix[s];
    a.tw_off[s] = p->mr_tw_off[s];
  }
  a.tw_count = p->mr_tw_count;
  a.win = p->d_mr_win;
  a.tw = p->d_mr_tw;
  a.twn = p->d_mr_twn;
  a.out_c = out_c;
  a.out_r = out_r;
  a.mode = mode;
  a.power_mode = p->power_mode;
  a.power = p->power;
  a.status = c->d_status;
  if (mode == 2) {
    a.band = p->d_band;
    a.mel_w = p->d_mel_w;
    a.n_mels = p->n_mels;
    a.mel_w_count = p->mel_w_count;
    a.log_mode = log_mode ? 1 : 0;
    a.amin = p->amin;
    a.db_sub = 10.0f * log10f(fmaxf(p->amin, fabsf(p->ref_value)));
    a.clip_max = c->d_clip_max;
  }
  const size_t tables = mr_table_bytes(a.L, a.tw_count, a.n_mels, a.mel_w_count);
  const size_t per_warp = (size_t)2 * a.M * sizeof(float2) * (size_t)mr_frames_per_warp(a.M);
  // two resident blocks per SM when they fit: at most half of the SM's shared memory each
  const size_t budget = (c->smem_optin + 1024) / 2 - 1024;
  int nw = 16;
  while (nw > 1 && tables + nw * per_warp > budget) --nw;
  if (tables + nw * per_warp > c->smem_optin)
    return fail(B2L_ERR_UNSUPPORTED, "n_fft=%d needs more shared memory than one SM has", p->n_fft);
  const size_t smem = tables + nw * per_warp;
  // lanes per frame: short frames ride two to a warp (their butterfly rounds fill 16 lanes better than 32)
  const int fpw = mr_frames_per_warp(a.M);
  const int lanes = 32 / fpw;
  auto kern = lanes == 16 ? (mode == 0 ? mr_kernel<0, 16> : (mode == 1 ? mr_kernel<1, 16> : mr_kernel<2, 16>))
                          : (mode == 0 ? mr_kernel<0, 32> : (mode == 1 ? mr_kernel<1, 32> : mr_kernel<2, 32>));
  const unsigned long long kkey = (1ULL << 62) | (unsigned long long)(mode + 8 * fpw);
  if (c->launch_cache.find(kkey) == c->launch_cache.end()) {
    CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)c->smem_optin));
    c->launch_cache[kkey] = 1;
  }
  int occ = 0;
  CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, nw * 32, smem));
  if (occ < 1) return fail(B2L_ERR_CUDA, "mixed-radix kernel does not fit on an SM (smem %zu)", smem);
  const long long total = (long long)n_clips * T;
  long long grid = (long long)c->sm_count * occ;
  const long long need = (total + (long long)nw * fpw - 1) / ((long long)nw * fpw);
  if (grid > need) grid = need;
  kern<<<(int)grid, nw * 32, smem, c->stream>>>(a);
  CUDA_TRY(cudaGetLastError());
  c->launches++;
  return B2L_OK;
}

extern "C" int b2l_stft(b2l_ctx* c, const b2l_plan* p, const float* d_y, int64_t n_clips, int64_t n, int64_t y_stride,
                        void* d_D) {
  if (c && p && p->czt)
    return p->mr && mr_enabled(p) ? run_mr(c, p, 0, 0, d_y, n_clips, n, y_stride, (float2*)d_D, nullptr)
                                 : run_czt(c, p, 0, d_y, n_clips, n, y_stride, (float2*)d_D, nullptr);
  return run_forward(c, p, MODE_STFT, 0, d_y, n_clips, n, y_stride, (float2*)d_D, nullptr);
}
extern "C" int b2l_spectrogram(b2l_ctx* c, const b2l_plan* p, const float* d_y, int64_t n_clips, int64_t n,
                               int64_t y_stride, float* d_S) {
  if (c && p && p->czt)
    return p->mr && mr_enabled(p) ? run_mr(c, p, 1, 0, d_y, n_clips, n, y_stride, nullptr, d_S)
                                 : run_czt(c, p, 1, d_y, n_clips, n, y_stride, nullptr, d_S);
  return run_forward(c, p, MODE_SPEC, 0, d_y, n_clips, n, y_stride, nullptr, d_S);
}
// ------------------------------------------------------------------ frame-wise spectral statistics / framings
static int check_stats_desc(const b2l_stats_desc* d, StatsParams* sp) {
  if (!d) return fail(B2L_ERR_INVALID, "NULL stats descriptor");
  if (!(d->roll_percent > 0.0f && d->roll_percent < 1.0f))
    return fail(B2L_ERR_INVALID, "roll_percent must lie in the range (0, 1)");
  if (!(d->flat_amin > 0.0f)) return fail(B2L_ERR_INVALID, "amin must be strictly positive");
  if (!(d->bw_p > 0.0f)) return fail(B2L_ERR_INVALID, "p must be strictly positive");
  if (d->frame_length < 1) return fail(B2L_ERR_INVALID, "frame_length must be positive");
  sp->roll_percent = d->roll_percent;
  sp->flat_amin = d->flat_amin;
  sp->flat_power = d->flat_power;
  sp->bw_p = d->bw_p;
  sp->bw_norm = d->bw_norm ? 1 : 0;
  sp->frame_length = d->frame_length;
  sp->want = d->want ? (d->want & ((1 << N_STATS) - 1)) : (1 << N_STATS) - 1;
  return B2L_OK;
}

extern "C" int b2l_spectral_stats_from_spec(b2l_ctx* c, const b2l_stats_desc* d, const float* d_S, int64_t n_clips,
                                            int64_t n_frames, int32_t n_bins, const float* d_freq, float* d_out) {
  if (!c || !d_S || !d_freq || !d_out) return fail(B2L_ERR_INVALID, "NULL argument");
  StatsCall sc;
  int rc = check_stats_desc(d, &sc.sp);
  if (rc) return rc;
  if (n_bins < 2) return fail(B2L_ERR_INVALID, "a spectrum needs at least two bins");
  if (n_clips <= 0 || n_frames <= 0) return B2L_OK;
  if (n_frames > 0x7fffffffLL) return fail(B2L_ERR_UNSUPPORTED, "too many frames");
  DeviceGuard g(c->device);
  const int Fp = (n_bins + 3) & ~3;
  int nw = 8;
  while (nw > 1 && (size_t)(nw + 1) * Fp * 4 > c->smem_optin) nw >>= 1;
  const size_t smem = (size_t)(nw + 1) * Fp * 4;
  if (smem > c->smem_optin) return fail(B2L_ERR_UNSUPPORTED, "n_bins=%d rows do not fit in shared memory", n_bins);
  CUDA_TRY(cudaFuncSetAttribute(stats_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)c->smem_optin));
  const long long rows = (long long)n_clips * n_frames;
  long long grid = (rows + nw - 1) / nw;
  const long long cap = (long long)c->sm_count * 8;
  if (grid > cap) grid = cap;
  stats_kernel<<<(int)grid, nw * 32, smem, c->stream>>>(d_S, rows, (int)n_frames, n_bins, d_freq, sc.sp, d_out,
                                                        c->d_status);
  CUDA_TRY(cudaGetLastError());
  c->launches++;
  return B2L_OK;
}

extern "C" int b2l_spectral_stats(b2l_ctx* c, const b2l_plan* p, const b2l_stats_desc* d, const float* d_y,
                                  int64_t n_clips, int64_t n, int64_t y_stride, const float* d_freq, float* d_out) {
  if (!c || !p) return fail(B2L_ERR_INVALID, "NULL ctx / plan");
  if (p->czt)
    return fail(B2L_ERR_UNSUPPORTED,
                "n_fft=%d: compose b2l_spectrogram + b2l_spectral_stats_from_spec for non-power-of-two sizes", p->n_fft);
  StatsCall sc;
  int rc = check_stats_desc(d, &sc.sp);
  if (rc) return rc;
  sc.d_freq = d_freq;
  return run_forward(c, p, MODE_STATS, 0, d_y, n_clips, n, y_stride, nullptr, d_out, &sc);
}

extern "C" int b2l_frame_feature(b2l_ctx* c, int32_t what, const float* d_y, int64_t n_clips, int64_t n,
                                 int64_t y_stride, int32_t frame_length, int32_t hop_length, int32_t center,
                                 int32_t pad_mode, float threshold, int32_t zero_pos, int32_t pad_first, float out_scale,
                                 float* d_out) {
  if (!c) return fail(B2L_ERR_INVALID, "NULL ctx");
  if (what != B2L_FRAME_RMS && what != B2L_FRAME_ZERO_CROSSINGS) return fail(B2L_ERR_INVALID, "bad feature id %d", what);
  if (frame_length < 1) return fail(B2L_ERR_INVALID, "frame_length=%d must be positive", frame_length);
  if (hop_length < 1) return fail(B2L_ERR_INVALID, "hop_length=%d must be a positive integer", hop_length);
  if (pad_mode < 0 || pad_mode > B2L_PAD_EMPTY) return fail(B2L_ERR_INVALID, "bad pad_mode %d", pad_mode);
  if (n_clips < 0 || n < 0 || y_stride < n) return fail(B2L_ERR_INVALID, "bad clip geometry");
  if (n > 0x7fffffffLL) return fail(B2L_ERR_UNSUPPORTED, "clips longer than 2^31-1 samples are not supported");
  const int pad = center ? frame_length / 2 : 0;
  const long long padded = n + 2LL * pad;
  if (padded < frame_length)
    return fail(B2L_ERR_INVALID, "Input is too short (n=%lld) for frame_length=%d", (long long)padded, frame_length);
  const long long T = 1 + (padded - frame_length) / hop_length;
  if (n_clips == 0) return B2L_OK;
  if (!d_y || !d_out) return fail(B2L_ERR_INVALID, "NULL device pointer");
  if (T > 0x7fffffffLL) return fail(B2L_ERR_UNSUPPORTED, "too many frames");
  DeviceGuard g(c->device);
  // frame_length a multiple of hop_length: block form, every sample read once (feat_kernels.cuh)
  {
    const char* env = getenv("B2L_TD_BLOCK");
    const long long tiles = (T + TD_FRAMES - 1) / TD_FRAMES;
    if (!(env && *env && atoi(env) == 0) && frame_length % hop_length == 0 && frame_length / hop_length <= 64 &&
        n_clips <= 65535 && tiles <= 0x7fffffffLL) {
      const int R = frame_length / hop_length;
      const size_t smem = (size_t)(TD_FRAMES + R - 1) * 8;
      frame_td_block_kernel<<<dim3((unsigned)tiles, (unsigned)n_clips), 256, smem, c->stream>>>(
          d_y, y_stride, (int)n, frame_length, hop_length, pad, pad_mode, (int)T, what, threshold, zero_pos, pad_first,
          out_scale, d_out, c->d_status);
      CUDA_TRY(cudaGetLastError());
      c->launches++;
      return B2L_OK;
    }
  }
  const long long rows = (long long)n_clips * T;
  long long grid = (rows + 7) / 8;
  const long long cap = (long long)c->sm_count * 8;
  if (grid > cap) grid = cap;
  frame_td_kernel<<<(int)grid, 256, 0, c->stream>>>(d_y, y_stride, (int)n, n_clips, frame_length, hop_length, pad,
                                                    pad_mode, (int)T, what, threshold, zero_pos, pad_first, out_scale,
                                                    d_out,                                                    c->d_status);
  CUDA_TRY(cudaGetLastError());
  c->launches++;
  return B2L_OK;
}

extern "C" int b2l_melspectrogram(b2l_ctx* c, const b2l_plan* p, const float* d_y, int64_t n_clips, int64_t n,
                                  int64_t y_stride, float* d_mel) {
  if (c && p && p->czt && p->mr) return run_mr(c, p, 2, 0, d_y, n_clips, n, y_stride, nullptr, d_mel);
  if (p && p->czt)
    return fail(B2L_ERR_UNSUPPORTED, "n_fft=%d: compose b2l_spectrogram + b2l_mel_project for non-power-of-two sizes",
                p->n_fft);
  return run_forward(c, p, MODE_MEL, 0, d_y, n_clips, n, y_stride, nullptr, d_mel);
}

static int launch_dct(b2l_ctx* c, const b2l_plan* p, const float* d_L, int64_t n_clips, int64_t T, int clamp,
                      float* d_out, int tiled = 0) {
  const int KG = (p->n_mfcc + 7) / 8;
  if (KG > 16) return fail(B2L_ERR_UNSUPPORTED, "n_mfcc=%d > 128 is not supported", p->n_mfcc);
  // dct_clamp4_kernel: the DCT table [n_mels][8*KG] and one tile of DCT4_TILE frames in shared memory
  const size_t smem = (size_t)p->n_mels * (8 * KG + DCT4_TILE) * 4;
  if (smem > c->smem_optin) {
    // too many input rows for the shared-memory tile (e.g. mfcc(S=...) of a 1025-bin spectrogram): generic kernel
    if (tiled) return fail(B2L_ERR_UNSUPPORTED, "n_mels=%d is too large for the fused mfcc path", p->n_mels);
    if (n_clips > 65535) return fail(B2L_ERR_UNSUPPORTED, "dct: more than 65535 leading indices");
    dct_generic_kernel<<<dim3((unsigned)((T + 127) / 128), (unsigned)n_clips), 128, 0, c->stream>>>(
        d_L, p->d_dct, clamp ? c->d_clip_max : nullptr, clamp ? p->top_db : -1.0f, p->n_mels, p->n_mfcc, 8 * KG, (int)T,
        d_out);
    CUDA_TRY(cudaGetLastError());
    c->launches++;
    return B2L_OK;
  }
  // two warp sets over the mel rows when the partial sums fit in the tile buffer
  const int ks = KG <= 10 && p->n_mels >= 8 * KG ? 2 : 1;   // 640 threads at most; 32*KG*32 partial sums <= 2*n_mels*64 tile words
  auto kern = ks == 2 ? dct_clamp4_kernel<2> : dct_clamp4_kernel<1>;
  const int threads = KG * 32 * ks;
  CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int tiles = (int)((T + DCT4_TILE - 1) / DCT4_TILE);
  const long long total = (long long)tiles * n_clips;
  int occ = 0;
  CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, threads, smem));
  if (occ < 1) return fail(B2L_ERR_CUDA, "DCT kernel does not fit on an SM");
  long long grid = (long long)c->sm_count * occ;
  if (grid > total) grid = total;
  kern<<<(int)grid, threads, smem, c->stream>>>(d_L, p->d_dct, clamp ? c->d_clip_max : nullptr,
                                                clamp ? p->top_db : -1.0f, p->n_mels, p->n_mfcc, (int)T, tiles, total,
                                                tiled, d_out);
  CUDA_TRY(cudaGetLastError());
  c->launches++;
  return B2L_OK;
}

extern "C" int b2l_mfcc(b2l_ctx* c, const b2l_plan* p, const float* d_y, int64_t n_clips, int64_t n, int64_t y_stride,
                        float* d_mfcc, float* d_logmel) {
  if (!c || !p) return fail(B2L_ERR_INVALID, "NULL ctx / plan");
  if (p->n_mfcc == 0) return fail(B2L_ERR_INVALID, "plan has no mfcc stage");
  if (p->czt && !p->mr)
    return fail(B2L_ERR_UNSUPPORTED, "n_fft=%d: compose spectrogram, mel_project, power_to_db and dct_project for "
                "non-power-of-two sizes", p->n_fft);
  if (n_clips <= 0) return n_clips == 0 ? B2L_OK : fail(B2L_ERR_INVALID, "negative n_clips");
  DeviceGuard g(c->device);
  const long long T = plan_frames(p, n);
  if (T <= 0) return fail(B2L_ERR_INVALID, "n_fft=%d is too large for input signal of length=%lld", p->n_fft, (long long)n);
  int rc = ensure_clip_max(c, (size_t)n_clips);
  if (rc) return rc;
  CUDA_TRY(cudaMemsetAsync(c->d_clip_max, 0, (size_t)n_clips * sizeof(unsigned int), c->stream));
  float* scratch = d_logmel;
  // the log-mel scratch is tiled: [clip][ceil(T/64)][n_mels][64] (see dct_clamp4_kernel)
  if (!scratch) CUDA_TRY(cudaMalloc((void**)&scratch, (size_t)n_clips * p->n_mels * ((T + 63) / 64 * 64) * sizeof(float)));
  // mixed-radix frames (mr_kernel): the dB rows go to the scratch in the plain [clip][mel][frame] layout
  const int tiled = p->czt ? 0 : 1;
  rc = p->czt ? run_mr(c, p, 2, 1, d_y, n_clips, n, y_stride, nullptr, scratch)
              : run_forward(c, p, MODE_MEL, 2, d_y, n_clips, n, y_stride, nullptr, scratch);
  if (rc == B2L_OK) rc = launch_dct(c, p, scratch, n_clips, T, 1, d_mfcc, tiled);
  if (!d_logmel) {
    cudaStreamSynchronize(c->stream);
    cudaFree(scratch);
  }
  return rc;
}

// ------------------------------------------------------------------ inverse launch
extern "C" int b2l_istft(b2l_ctx* c, const b2l_plan* p, const void* d_D, int64_t n_clips, int64_t n_frames_stored,
                         int64_t n_frames_used, const float* d_inv_wss, int64_t out_len, float* d_y,
                         int64_t y_stride) {
  if (!c || !p) return fail(B2L_ERR_INVALID, "NULL ctx / plan");
  if (p->ctx != c) return fail(B2L_ERR_INVALID, "plan belongs to another context");
  if (n_clips < 0 || n_frames_used < 1 || n_frames_used > n_frames_stored || out_len < 0 || y_stride < out_len)
    return fail(B2L_ERR_INVALID, "bad istft geometry");
  if (n_clips == 0 || out_len == 0) return B2L_OK;
  if (!d_D || !d_inv_wss || !d_y) return fail(B2L_ERR_INVALID, "NULL device pointer");
  if (p->czt) {
    // chirp-z inverse frames into scratch, then a gather overlap-add (czt_kernel.cuh)
    if (out_len > 0x7fffffffLL || n_clips > 65535) return fail(B2L_ERR_UNSUPPORTED, "istft batch too large");
    DeviceGuard g(c->device);
    const int L = p->n_fft;
    const size_t need = (size_t)n_clips * (size_t)n_frames_used * L * sizeof(float);
    if (c->scratch_bytes < need) {
      CUDA_TRY(cudaStreamSynchronize(c->stream));
      if (c->d_scratch) CUDA_TRY(cudaFree(c->d_scratch));
      c->d_scratch = nullptr;
      c->scratch_bytes = 0;
      CUDA_TRY(cudaMalloc((void**)&c->d_scratch, need));
      c->scratch_bytes = need;
    }
    if (p->mr && mr_enabled(p)) {
      // mixed-radix inverse frames (mr_inv_kernel) into the scratch array, then the same overlap-add
      MrInvArgs ma;
      memset(&ma, 0, sizeof(ma));
      ma.D = (const float2*)d_D;
      ma.d_clip_stride = (long long)n_frames_stored * (L / 2 + 1);
      ma.n_clips = (int)n_clips;
      ma.n_frames = (int)n_frames_used;
      ma.L = L;
      ma.M = L / 2;
      ma.n_bins = L / 2 + 1;
      ma.n_pass = p->mr_n_pass;
      for (int s = 0; s < p->mr_n_pass; ++s) {
        ma.radix[s] = p->mr_radix[s];
        ma.tw_off[s] = p->mr_tw_off[s];
      }
      ma.tw_count = p->mr_tw_count;
      ma.win = p->d_mr_win_inv;
      ma.tw = p->d_mr_tw;
      ma.twn = p->d_mr_twn;
      ma.ytmp = c->d_scratch;
      const size_t tables = mr_table_bytes(L, ma.tw_count, 0, 0);
      const size_t per_warp = (size_t)2 * ma.M * sizeof(float2);
      const size_t budget = (c->smem_optin + 1024) / 2 - 1024;
      int nw = 16;
      while (nw > 1 && tables + nw * per_warp > budget) --nw;
      if (tables + nw * per_warp > c->smem_optin)
        return fail(B2L_ERR_UNSUPPORTED, "n_fft=%d needs more shared memory than one SM has", L);
      const size_t smem = tables + nw * per_warp;
      const unsigned long long kkey = (1ULL << 62) | 7ULL;
      if (c->launch_cache.find(kkey) == c->launch_cache.end()) {
        CUDA_TRY(cudaFuncSetAttribute(mr_inv_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)c->smem_optin));
        c->launch_cache[kkey] = 1;
      }
      int occ = 0;
      CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, mr_inv_kernel, nw * 32, smem));
      if (occ < 1) return fail(B2L_ERR_CUDA, "mixed-radix inverse kernel does not fit on an SM (smem %zu)", smem);
      const long long total = (long long)n_clips * n_frames_used;
      long long grid = (long long)c->sm_count * occ;
      const long long need_blocks = (total + nw - 1) / nw;
      if (grid > need_blocks) grid = need_blocks;
      mr_inv_kernel<<<(int)grid, nw * 32, smem, c->stream>>>(ma);
      CUDA_TRY(cudaGetLastError());
      c->launches++;
    } else {
    HostFftCfg cfg(p->log2p);
    const int nw = cfg.czt_nw();
    const int G = nw * 32 / cfg.tpf;
    CztInvArgs a;
    memset(&a, 0, sizeof(a));
    a.D = (const float2*)d_D;
    a.d_clip_stride = (long long)n_frames_stored * (L / 2 + 1);
    a.n_clips = (int)n_clips;
    a.n_frames = (int)n_frames_used;
    a.L = L;
    a.n_bins = L / 2 + 1;
    a.bfull = p->d_czt_bfull;
    a.wbi = p->d_czt_wbi;
    a.hf = p->d_czt_hf;
    a.ytmp = c->d_scratch;
    const size_t smem = (size_t)((cfg.tw_count() + 15) & ~15) * 8 + (size_t)G * cfg.xbuf_f2() * 8 +
                        ((size_t)(1 << p->log2p) + (size_t)((L + 1) & ~1)) * 8;   // + FFT_P(h)/P and window * chirp
    if (smem > c->smem_optin) return fail(B2L_ERR_UNSUPPORTED, "n_fft=%d needs more shared memory than one SM has", L);
    czt_inv_op_fn op = czt_inv_table(p->log2p);
    const unsigned long long kkey = (3ULL << 62) | ((unsigned long long)p->log2p << 40);
    int occ = 0;
    auto hit = c->launch_cache.find(kkey);
    if (hit != c->launch_cache.end()) {
      occ = hit->second;
    } else {
      CUDA_TRY(op(OP_SET_SMEM, &a, 0, c->smem_optin, c->stream, nullptr));
      CUDA_TRY(op(OP_OCCUPANCY, &a, 0, c->smem_optin / 2 + 1, c->stream, &occ));
      c->launch_cache[kkey] = occ;
    }
    if (occ < 1) return fail(B2L_ERR_CUDA, "chirp-z inverse kernel does not fit on an SM");
    const long long steps = ((long long)n_clips * ((n_frames_used + 1) / 2) + G - 1) / G;   // frames go in pairs inside a clip
    long long grid = (long long)c->sm_count * occ;
    if (grid > steps) grid = steps;
    CUDA_TRY(op(OP_LAUNCH, &a, (int)grid, smem, c->stream, nullptr));
    c->launches++;
    }
    long long bx = (out_len + 255) / 256;
    const long long cap = (8LL * c->sm_count + n_clips - 1) / n_clips;
    if (bx > cap) bx = cap;
    if (bx < 1) bx = 1;
    dim3 og((unsigned)bx, (unsigned)n_clips);
    ola_kernel<<<og, 256, 0, c->stream>>>(c->d_scratch, (int)n_frames_used, L, p->hop, p->center ? L / 2 : 0, (int)out_len,
                                          y_stride, d_inv_wss, d_y);
    CUDA_TRY(cudaGetLastError());
    c->launches++;
    return B2L_OK;
  }
  if (out_len > 0x7fffffffLL || n_frames_stored > 0x7fffffffLL)
    return fail(B2L_ERR_UNSUPPORTED, "istft output longer than 2^31-1 samples is not supported");
  DeviceGuard g(c->device);
  HostFftCfg cfg(p->log2m);
  const int N = p->n_fft, M = N / 2;
  inv_op_fn op = inv_table(p->log2m);
  int variants[3];
  int n_opt = 0;
  {
    const char* force = getenv("B2L_INV_VARIANT");
    if (force && *force) {
      variants[n_opt++] = atoi(force);
    } else {
      if (cfg.log2m >= 9 && cfg.log2m <= 11) variants[n_opt++] = 116;
      int nws[2];
      const int k = cfg.nw_options(nws);
      for (int i = 0; i < k; ++i) variants[n_opt++] = nws[i];
    }
  }
  InvArgs a;
  memset(&a, 0, sizeof(a));
  // hop = n_fft / 4 or / 2, one or more whole warps per frame: autonomous frame groups with the overlap-add
  // state in Tensor Memory (inv2_kernel.cuh); B2L_INV2=0 keeps the gather kernel
  {
    const char* e2 = getenv("B2L_INV2");
    const bool want2 = !(e2 && *e2 && atoi(e2) == 0) && !(getenv("B2L_INV_VARIANT") && *getenv("B2L_INV_VARIANT"));
    const int R = p->hop > 0 && N % p->hop == 0 ? N / p->hop : 0;
    if (want2 && cfg.log2m >= 10 && cfg.log2m <= 12 && (R == 4 || R == 2)) {
      const int NG = 16 * 32 / cfg.tpf;
      size_t off = 0;
      a.off_acc = (int)off; off = align_up(off + 16, 128);            // TMEM base address
      a.off_xbuf = (int)off; off += (size_t)NG * cfg.xbuf_f2() * 8;
      if (off <= c->smem_optin) {
        a.D = (const float2*)d_D;
        a.d_clip_stride = (long long)n_frames_stored * (M + 1);
        a.n_clips = (int)n_clips;
        a.n_frames = (int)n_frames_used;
        a.n_fft = N;
        a.hop = p->hop;
        a.start = p->center ? N / 2 : 0;
        a.out_len = (int)out_len;
        a.y_clip_stride = y_stride;
        a.y = d_y;
        a.window = p->d_win_inv;
        a.inv_wss = d_inv_wss;
        a.tw = p->d_tw;
        a.twn = p->d_twn;
        a.vec4 = (y_stride % 2 == 0) && (((uintptr_t)d_y & 7) == 0) && (((uintptr_t)d_inv_wss & 7) == 0);   // 8-byte stores
        const long long total_frames = (long long)n_clips * n_frames_used;
        const long long groups = (long long)c->sm_count * NG;
        long long fps = (total_frames + groups - 1) / groups;
        if (fps < 8) fps = 8;                                          // replayed frames stay a bounded fraction
        a.frames_per_slot = (int)fps;
        {
          const char* ea = getenv("B2L_INV2_AHEAD");           // spectrum rows prefetched to L2 ahead of the transform
          a.acc_floats = ea && *ea ? std::max(1, std::min(4, atoi(ea))) : 1;
        }
        const long long runs = (total_frames + fps - 1) / fps;
        const long long grid = (runs + NG - 1) / NG;
        const int v2 = 2000 + R;
        CUDA_TRY(op(OP_SET_SMEM, v2, &a, 0, off, c->stream, nullptr));
        CUDA_TRY(op(OP_LAUNCH, v2, &a, (int)grid, off, c->stream, nullptr));
        c->launches++;
        return B2L_OK;
      }
    }
  }
  int variant = 0, G = 0, halves = 1;
  size_t smem = 0;
  const int clen = N > p->hop ? N - p->hop : 0;
  for (int i = 0; i < n_opt && !variant; ++i) {
    const int v = variants[i];
    const bool dual = v == 116;
    const int nw = dual ? 16 : v;
    const int nh = dual ? 2 : 1;
    if (nw * 32 % (cfg.tpf * nh) != 0) continue;
    const int gg = nw * 32 / nh / cfg.tpf;
    if (gg < 1) continue;
    size_t off = 0;
    a.off_win = (int)off; off = align_up(off + (size_t)N * 4, 16);
    a.off_tw = (int)off; off = align_up(off + (size_t)cfg.tw_count() * 8, 16);
    a.off_acc = (int)off;
    a.acc_stride = (int)align_up((size_t)2 * clen * 4, 16);
    off += (size_t)a.acc_stride * nh;
    a.off_xbuf = (int)(off = align_up(off, 128));
    a.xbuf_stride = (int)align_up((size_t)gg * cfg.xbuf_f2() * 8, 128);
    off += (size_t)a.xbuf_stride * nh;
    if (off > c->smem_optin) continue;
    variant = v;
    G = gg;
    halves = nh;
    smem = off;
  }
  if (!variant) return fail(B2L_ERR_UNSUPPORTED, "istft configuration does not fit in shared memory");
  a.acc_floats = 2 * clen;
  a.D = (const float2*)d_D;
  a.d_clip_stride = (long long)n_frames_stored * (M + 1);
  a.n_clips = (int)n_clips;
  a.n_frames = (int)n_frames_used;
  a.n_fft = N;
  a.hop = p->hop;
  a.start = p->center ? N / 2 : 0;
  a.out_len = (int)out_len;
  a.y_clip_stride = y_stride;
  a.y = d_y;
  a.window = p->d_win_inv;
  a.inv_wss = d_inv_wss;
  a.tw = p->d_tw;
  a.twn = p->d_twn;
  a.vec4 = (p->hop % 4 == 0) && (clen % 4 == 0) && (a.start % 4 == 0) && (y_stride % 4 == 0) &&
           (cfg.xbuf_f2() % 2 == 0) &&   // frame buffers 16-byte aligned inside the exchange area
           (((uintptr_t)d_y & 15) == 0) && (((uintptr_t)d_inv_wss & 15) == 0);
  // one slot of consecutive (clip, frame) pairs per resident half-CTA (1 CTA per SM): equal work everywhere,
  // no partial last wave; slots are whole rounds of G frames, and at least 4 rounds long so that the halo
  // frames recomputed at the start of a slot stay a small fraction
  const long long total_frames = (long long)n_clips * n_frames_used;
  long long fps = (total_frames + (long long)c->sm_count * halves - 1) / ((long long)c->sm_count * halves);
  if (fps < 4LL * G) fps = 4LL * G;
  fps = (fps + G - 1) / G * G;
  if (fps > 0x7fffffffLL) return fail(B2L_ERR_UNSUPPORTED, "istft batch too large");
  a.frames_per_slot = (int)fps;
  const long long items = (total_frames + fps - 1) / fps;
  const long long grid = (items + halves - 1) / halves;
  CUDA_TRY(op(OP_SET_SMEM, variant, &a, 0, smem, c->stream, nullptr));
  CUDA_TRY(op(OP_LAUNCH, variant, &a, (int)grid, smem, c->stream, nullptr));
  c->launches++;
  return B2L_OK;
}

// ------------------------------------------------------------------ S= pieces
extern "C" int b2l_mel_project(b2l_ctx* c, const b2l_plan* p, const float* d_S, int64_t n_clips, int64_t n_frames,
                               float* d_mel) {
  if (!c || !p || !d_S || !d_mel) return fail(B2L_ERR_INVALID, "NULL argument");
  if (p->n_mels == 0) return fail(B2L_ERR_INVALID, "plan has no mel stage");
  if (n_clips <= 0 || n_frames <= 0) return B2L_OK;
  DeviceGuard g(c->device);
  const int F = p->n_fft / 2 + 1;
  {
    // a few rows whose bands cover most of the spectrum (chroma): dense_project_kernel (B2L_DENSE_PROJECT=0: off)
    const char* e = getenv("B2L_DENSE_PROJECT");
    const size_t dsmem = ((((size_t)F * 33 + 3) & ~(size_t)3) + (size_t)F * 16 + 8 * 16 * 32) * 4;
    if (p->d_mel_wT && (long long)p->mel_w_count * 4 >= (long long)p->n_mels * F && dsmem <= c->smem_optin &&
        !(e && *e && atoi(e) == 0)) {
      const int r4 = (p->n_mels + 3) / 4;
      auto kern = r4 == 1 ? dense_project_kernel<1> : r4 == 2 ? dense_project_kernel<2> : r4 == 3 ? dense_project_kernel<3> : dense_project_kernel<4>;
      CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dsmem));
      const int tiles_d = (int)((n_frames + 31) / 32);
      const long long total = (long long)tiles_d * n_clips;
      long long grid_d = c->sm_count;
      if (grid_d > total) grid_d = total;
      kern<<<(int)grid_d, 256, dsmem, c->stream>>>(d_S, p->d_mel_wT, p->n_mels, F, (int)n_frames, tiles_d, total, d_mel);
      CUDA_TRY(cudaGetLastError());
      c->launches++;
      return B2L_OK;
    }
  }
  size_t smem = (size_t)F * 33 * 4;
  if (smem > c->smem_optin) return fail(B2L_ERR_UNSUPPORTED, "n_fft too large for mel_project");
  CUDA_TRY(cudaFuncSetAttribute(mel_project_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int tiles = (int)((n_frames + 31) / 32);
  const long long grid = (long long)tiles * n_clips;
  if (grid > 0x7fffffffLL) return fail(B2L_ERR_UNSUPPORTED, "too many tiles");
  mel_project_kernel<<<(int)grid, 256, smem, c->stream>>>(d_S, p->d_mel_w, p->d_band, p->n_mels, F, (int)n_frames,
                                                          tiles, d_mel);
  CUDA_TRY(cudaGetLastError());
  c->launches++;
  return B2L_OK;
}

// ------------------------------------------------------------------ polyphase resampling
extern "C" int b2l_resample_poly(b2l_ctx* c, const float* d_x, int64_t n_clips, int64_t n_in, int64_t x_stride,
                                 const float* d_h, int32_t n_h, int32_t up, int32_t down, int64_t n_pre_remove,
                                 int64_t n_keep, int64_t n_total, float out_scale, float* d_out) {
  if (!c || !d_x || !d_h || !d_out) return fail(B2L_ERR_INVALID, "NULL argument");
  if (up < 1 || down < 1 || n_h < 1 || n_pre_remove < 0 || n_keep < 0 || n_total < n_keep || x_stride < n_in)
    return fail(B2L_ERR_INVALID, "bad resampling geometry");
  if (n_clips <= 0 || n_total <= 0) return B2L_OK;
  if (n_in > 0x7fffffffLL || n_total > 0x7fffffffLL) return fail(B2L_ERR_UNSUPPORTED, "signals longer than 2^31-1 samples");
  DeviceGuard g(c->device);
  const long long total = (long long)n_clips * n_total;
  long long grid = (total + 255) / 256;
  const long long cap = (long long)c->sm_count * 32;
  if (grid > cap) grid = cap;
  resample_poly_kernel<<<(int)grid, 256, 0, c->stream>>>(d_x, x_stride, (int)n_in, d_h, n_h, up, down, n_pre_remove,
                                                          (int)n_keep, (int)n_total, n_clips, out_scale, d_out);
  CUDA_TRY(cudaGetLastError());
  c->launches++;
  return B2L_OK;
}

extern "C" int b2l_power_to_db(b2l_ctx* c, const float* d_in, int64_t n_clips, int64_t per_clip, float amin,
                               float ref_value, float top_db, float* d_out) {
  if (!c || !d_in || !d_out) return fail(B2L_ERR_INVALID, "NULL argument");
  if (!(amin > 0.0f)) return fail(B2L_ERR_INVALID, "amin must be strictly positive");
  if (n_clips <= 0 || per_clip <= 0) return B2L_OK;
  DeviceGuard g(c->device);
  int rc = ensure_clip_max(c, (size_t)n_clips);
  if (rc) return rc;
  CUDA_TRY(cudaMemsetAsync(c->d_clip_max, 0, (size_t)n_clips * sizeof(unsigned int), c->stream));
  const float db_sub = 10.0f * log10f(fmaxf(amin, fabsf(ref_value)));
  // the clip index rides in grid.y (at most 65535): larger batches go in slices, like the kernels they accompany
  for (int64_t c0 = 0; c0 < n_clips; c0 += 65535) {
    const int64_t m = std::min<int64_t>(65535, n_clips - c0);
    long long bx = (per_clip + 256LL * 8 - 1) / (256LL * 8);
    long long cap = (4LL * c->sm_count + m - 1) / m;
    if (bx > cap) bx = cap;
    if (bx < 1) bx = 1;
    dim3 grid((unsigned)bx, (unsigned)m);
    db_kernel<<<grid, 256, 0, c->stream>>>(d_in + c0 * per_clip, per_clip, amin, db_sub, c->d_clip_max + c0, d_out + c0 * per_clip);
    CUDA_TRY(cudaGetLastError());
    c->launches++;
    if (top_db >= 0.0f) {
      db_clamp_kernel<<<grid, 256, 0, c->stream>>>(d_out + c0 * per_clip, per_clip, c->d_clip_max + c0, top_db);
      CUDA_TRY(cudaGetLastError());
      c->launches++;
    }
  }
  return B2L_OK;
}

extern "C" int b2l_onset_from_spec(b2l_ctx* c, const b2l_onset_desc* d, const float* d_S, int64_t n_clips,
                                   int64_t n_rows, int64_t n_frames, float* d_out) {
  if (!c || !d || !d_S || !d_out) return fail(B2L_ERR_INVALID, "NULL argument");
  if (d->lag < 1) return fail(B2L_ERR_INVALID, "lag=%d must be a positive integer", d->lag);
  if (d->max_size < 1) return fail(B2L_ERR_INVALID, "max_size=%d must be a positive integer", d->max_size);
  if (d->pad_width < 0) return fail(B2L_ERR_INVALID, "negative pad_width");
  if (d->n_channels < 0 || d->n_channels > 32) return fail(B2L_ERR_UNSUPPORTED, "at most 32 onset channels");
  if (n_clips <= 0 || n_rows <= 0 || n_frames <= 0) return B2L_OK;
  if (n_clips > 65535 || n_rows > 0x7fffffffLL || n_frames > 0x7fffffffLL)
    return fail(B2L_ERR_UNSUPPORTED, "onset: batch too large");
  OnsetArgs a;
  memset(&a, 0, sizeof(a));
  for (int i = 0; i <= d->n_channels; ++i) {
    a.bounds[i] = d->bounds[i];
    if (a.bounds[i] < 0 || a.bounds[i] > n_rows || (i > 0 && a.bounds[i] < a.bounds[i - 1]))
      return fail(B2L_ERR_INVALID, "channel boundaries must be non-decreasing row indices");
  }
  a.n_ch = d->n_channels;
  a.lag = d->lag;
  a.max_size = d->max_size;
  a.pad_width = d->pad_width;
  a.n_rows = (int)n_rows;
  a.T = (int)n_frames;
  DeviceGuard g(c->device);
  dim3 grid((unsigned)((n_frames + 127) / 128), (unsigned)n_clips);
  onset_kernel<<<grid, 128, 0, c->stream>>>(d_S, a, d_out);
  CUDA_TRY(cudaGetLastError());
  c->launches++;
  if (d->detrend) {
    const long long rows = (long long)n_clips * (a.n_ch > 0 ? a.n_ch : a.n_rows);
    detrend_kernel<<<(unsigned)((rows + 127) / 128), 128, 0, c->stream>>>(d_out, rows, a.T);
    CUDA_TRY(cudaGetLastError());
    c->launches++;
  }
  return B2L_OK;
}

extern "C" int b2l_pcen(b2l_ctx* c, const b2l_pcen_desc* d, const float* d_S, int64_t n_clips, int64_t n_rows,
                        int64_t n_frames, const float* d_zi, float* d_zf, float* d_scratch, float* d_out) {
  if (!c || !d || !d_S || !d_out) return fail(B2L_ERR_INVALID, "NULL argument");
  if (d->power < 0.0f) return fail(B2L_ERR_INVALID, "power=%g must be nonnegative", d->power);
  if (d->gain < 0.0f) return fail(B2L_ERR_INVALID, "gain=%g must be non-negative", d->gain);
  if (d->bias < 0.0f) return fail(B2L_ERR_INVALID, "bias=%g must be non-negative", d->bias);
  if (!(d->eps > 0.0f)) return fail(B2L_ERR_INVALID, "eps=%g must be strictly positive", d->eps);
  if (!(d->b >= 0.0f && d->b <= 1.0f)) return fail(B2L_ERR_INVALID, "b=%g must be between 0 and 1", d->b);
  if (d->max_size < 1) return fail(B2L_ERR_INVALID, "max_size=%d must be a positive integer", d->max_size);
  if (n_clips <= 0 || n_rows <= 0 || n_frames <= 0) return B2L_OK;
  if (n_frames > 0x7fffffffLL || n_rows > 65535 || n_clips > 65535) return fail(B2L_ERR_UNSUPPORTED, "pcen: batch too large");
  DeviceGuard g(c->device);
  const float* ref = d_S;
  if (d->max_size > 1) {
    if (!d_scratch) return fail(B2L_ERR_INVALID, "max_size > 1 needs a scratch buffer of the size of S");
    dim3 grid((unsigned)((n_frames + 127) / 128), (unsigned)n_rows, (unsigned)n_clips);
    maxfilter_rows_kernel<<<grid, 128, 0, c->stream>>>(d_S, (int)n_rows, (int)n_frames, d->max_size, d_scratch);
    CUDA_TRY(cudaGetLastError());
    c->launches++;
    ref = d_scratch;
  }
  PcenArgs a;
  a.gain = d->gain;
  a.bias = d->bias;
  a.power = d->power;
  a.eps = d->eps;
  a.b = d->b;
  a.mode = d->power == 0.0f ? 0 : (d->bias == 0.0f ? 1 : 2);
  const long long rows = (long long)n_clips * n_rows;
  const long long blocks = (rows + 127) / 128;
  pcen_kernel<<<(unsigned)blocks, 128, 0, c->stream>>>(d_S, ref, rows, (int)n_frames, a, d_zi, d_zf, d_out);
  CUDA_TRY(cudaGetLastError());
  c->launches++;
  return B2L_OK;
}

extern "C" int b2l_spectral_contrast(b2l_ctx* c, const b2l_contrast_desc* d, const float* d_S, int64_t n_clips,
                                     int64_t n_frames, int32_t n_bins, float* d_peak, float* d_valley) {
  if (!c || !d || !d_S || !d_peak || !d_valley) return fail(B2L_ERR_INVALID, "NULL argument");
  if (d->n_bands < 1 || d->n_bands > 16) return fail(B2L_ERR_UNSUPPORTED, "1 to 16 bands (n_bands + 1) are supported");
  if (n_clips <= 0 || n_frames <= 0) return B2L_OK;
  ContrastArgs a;
  memset(&a, 0, sizeof(a));
  a.n_bands = d->n_bands;
  int max_count = 1;
  for (int b = 0; b < d->n_bands; ++b) {
    if (d->lo[b] < 0 || d->count[b] < 0 || d->lo[b] + d->count[b] > n_bins || d->k[b] < 1)
      return fail(B2L_ERR_INVALID, "band %d: bad bin range / tail length", b);
    a.lo[b] = d->lo[b];
    a.count[b] = d->count[b];
    a.k[b] = d->k[b];
    max_count = std::max(max_count, d->count[b]);
  }
  int cap = 32;   // at least one entry per lane: the short-tail path parks 32 sorted runs in the scratch
  while (cap < max_count) cap <<= 1;
  DeviceGuard g(c->device);
  const size_t per_warp = ((size_t)((n_bins + 3) & ~3) + cap) * 4;
  int nw = 8;
  while (nw > 1 && per_warp * nw > c->smem_optin) nw >>= 1;
  const size_t smem = per_warp * nw;
  if (smem > c->smem_optin) return fail(B2L_ERR_UNSUPPORTED, "n_bins=%d rows do not fit in shared memory", n_bins);
  CUDA_TRY(cudaFuncSetAttribute(contrast_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)c->smem_optin));
  const long long rows = (long long)n_clips * n_frames;
  long long grid = (rows + nw - 1) / nw;
  const long long lim = (long long)c->sm_count * 8;
  if (grid > lim) grid = lim;
  contrast_kernel<<<(int)grid, nw * 32, smem, c->stream>>>(d_S, rows, (int)n_frames, n_bins, cap, a, d_peak, d_valley);
  CUDA_TRY(cudaGetLastError());
  c->launches++;
  return B2L_OK;
}

extern "C" int b2l_sub(b2l_ctx* c, const float* d_x, const float* d_y, int64_t n, float* d_out) {
  if (!c || !d_x || !d_y || !d_out) return fail(B2L_ERR_INVALID, "NULL argument");
  if (n <= 0) return B2L_OK;
  DeviceGuard g(c->device);
  long long grid = (n + 256LL * 8 - 1) / (256LL * 8);
  if (grid > 8LL * c->sm_count) grid = 8LL * c->sm_count;
  sub_kernel<<<(int)grid, 256, 0, c->stream>>>(d_x, d_y, n, d_out);
  CUDA_TRY(cudaGetLastError());
  c->launches++;
  return B2L_OK;
}

extern "C" int b2l_pip_pass(b2l_ctx* c, const b2l_pip_desc* d, const float* d_S, int64_t n_rows, int32_t n_bins,
                            const double* h_edges, uint64_t* h_hist) {
  if (!c || !d || !d_S || !h_hist) return fail(B2L_ERR_INVALID, "NULL argument");
  if (d->mode < 0 || d->mode > 3) return fail(B2L_ERR_INVALID, "bad pass mode %d", d->mode);
  if (d->mode == 3 && (!h_edges || d->n_res_bins < 1 || d->n_res_bins > 2048))
    return fail(B2L_ERR_INVALID, "residual histogram needs 1..2048 bins and their edges");
  if (d->k_lo < 0 || d->k_hi > n_bins) return fail(B2L_ERR_INVALID, "bad bin range");
  const int n_hist = d->mode == 3 ? d->n_res_bins : (d->mode == 2 ? 1024 : 2048);
  for (int i = 0; i < n_hist; ++i) h_hist[i] = 0;
  if (n_rows <= 0 || d->k_hi <= d->k_lo) return B2L_OK;
  DeviceGuard g(c->device);
  const size_t need = 2048 * sizeof(unsigned long long) + 2049 * sizeof(double);
  if (c->scratch_bytes < need) {
    if (c->d_scratch) {
      CUDA_TRY(cudaStreamSynchronize(c->stream));
      CUDA_TRY(cudaFree(c->d_scratch));
      c->d_scratch = nullptr;
      c->scratch_bytes = 0;
    }
    CUDA_TRY(cudaMalloc((void**)&c->d_scratch, need));
    c->scratch_bytes = need;
  }
  unsigned long long* d_hist = reinterpret_cast<unsigned long long*>(c->d_scratch);
  double* d_edges = reinterpret_cast<double*>(d_hist + 2048);
  CUDA_TRY(cudaMemsetAsync(d_hist, 0, 2048 * sizeof(unsigned long long), c->stream));
  if (d->mode == 3)
    CUDA_TRY(cudaMemcpyAsync(d_edges, h_edges, (size_t)(d->n_res_bins + 1) * sizeof(double), cudaMemcpyHostToDevice, c->stream));
  PipArgs a;
  a.k_lo = d->k_lo;
  a.k_hi = d->k_hi;
  a.threshold = d->threshold;
  a.ref_abs = d->ref_abs;
  a.hz_per_bin = d->hz_per_bin;
  a.mode = d->mode;
  a.prefix = d->prefix;
  a.mag_threshold = d->mag_threshold;
  a.bins_per_octave = d->bins_per_octave;
  a.n_res_bins = d->n_res_bins;
  const size_t per_warp = (size_t)((n_bins + 3) & ~3) * 4;
  int nw = 8;
  while (nw > 1 && per_warp * nw + 8192 + 1024 > c->smem_optin) nw >>= 1;
  const size_t smem = per_warp * nw;
  if (smem + 8192 + 1024 > c->smem_optin) return fail(B2L_ERR_UNSUPPORTED, "n_bins=%d rows do not fit in shared memory", n_bins);
  CUDA_TRY(cudaFuncSetAttribute(pip_pass_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(c->smem_optin - 8192 - 1024)));
  long long grid = (n_rows + nw - 1) / nw;
  const long long lim = (long long)c->sm_count * 4;
  if (grid > lim) grid = lim;
  pip_pass_kernel<<<(int)grid, nw * 32, smem, c->stream>>>(d_S, n_rows, n_bins, a, d_edges, d_hist);
  CUDA_TRY(cudaGetLastError());
  c->launches++;
  CUDA_TRY(cudaMemcpyAsync(h_hist, d_hist, (size_t)n_hist * sizeof(unsigned long long), cudaMemcpyDeviceToHost, c->stream));
  CUDA_TRY(cudaStreamSynchronize(c->stream));
  return B2L_OK;
}

extern "C" int b2l_normalize_rows(b2l_ctx* c, const float* d_in, int64_t n_clips, int64_t n_rows, int64_t n_frames,
                                  int32_t norm_kind, float norm_p, float* d_out) {
  if (!c || !d_in || !d_out) return fail(B2L_ERR_INVALID, "NULL argument");
  if (norm_kind < 0 || norm_kind > 3) return fail(B2L_ERR_INVALID, "bad norm kind %d", norm_kind);
  if (norm_kind == 3 && !(norm_p > 0.0f)) return fail(B2L_ERR_INVALID, "Unsupported norm: %g", norm_p);
  if (n_clips <= 0 || n_rows <= 0 || n_frames <= 0) return B2L_OK;
  if (n_clips > 65535 || n_rows > 0x7fffffffLL || n_frames > 0x7fffffffLL) return fail(B2L_ERR_UNSUPPORTED, "normalize: batch too large");
  DeviceGuard g(c->device);
  dim3 grid((unsigned)((n_frames + 127) / 128), (unsigned)n_clips);
  normalize_rows_kernel<<<grid, 128, 0, c->stream>>>(d_in, (int)n_rows, (int)n_frames, norm_kind, norm_p, d_out);
  CUDA_TRY(cudaGetLastError());
  c->launches++;
  return B2L_OK;
}

extern "C" int b2l_cabs(b2l_ctx* c, const void* d_complex, int64_t n, float* d_out) {
  if (!c || !d_complex || !d_out) return fail(B2L_ERR_INVALID, "NULL argument");
  if (n <= 0) return B2L_OK;
  DeviceGuard g(c->device);
  long long grid = (n + 256LL * 8 - 1) / (256LL * 8);
  if (grid > 8LL * c->sm_count) grid = 8LL * c->sm_count;
  cabs_kernel<<<(int)grid, 256, 0, c->stream>>>((const float2*)d_complex, n, d_out);
  CUDA_TRY(cudaGetLastError());
  c->launches++;
  return B2L_OK;
}

extern "C" int b2l_hpss(b2l_ctx* c, const b2l_hpss_desc* d, const float* d_mag, const void* d_S_complex,
                        int64_t n_clips, int64_t n_frames, int64_t n_bins, void* d_out_harm, void* d_out_perc) {
  if (!c || !d || !d_mag || !d_out_harm || !d_out_perc) return fail(B2L_ERR_INVALID, "NULL argument");
  if (d->win_harm < 1 || d->win_perc < 1) return fail(B2L_ERR_INVALID, "kernel sizes must be positive");
  if (d->win_harm > 64 || d->win_perc > 64) return fail(B2L_ERR_UNSUPPORTED, "median filters longer than 64 are not supported");
  if (d->margin_harm < 1.0f || d->margin_perc < 1.0f)
    return fail(B2L_ERR_INVALID, "Margins must be >= 1.0. A typical range is between 1 and 10.");
  if (!(d->power > 0.0f)) return fail(B2L_ERR_INVALID, "power must be strictly positive");
  if (n_clips <= 0 || n_frames <= 0 || n_bins <= 0) return B2L_OK;
  if (n_frames > 65535 || n_clips > 65535 || n_bins > 0x7fffffffLL) return fail(B2L_ERR_UNSUPPORTED, "hpss: batch too large");
  HpssArgs a;
  a.T = (int)n_frames;
  a.F = (int)n_bins;
  a.win_h = d->win_harm;
  a.win_p = d->win_perc;
  a.margin_h = d->margin_harm;
  a.margin_p = d->margin_perc;
  a.power = d->power;
  a.split_zeros = (d->margin_harm == 1.0f && d->margin_perc == 1.0f) ? 1 : 0;
  a.mode = d->mask_only ? 1 : 0;
  DeviceGuard g(c->device);
  const int w = std::max(d->win_harm, d->win_perc);
  dim3 grid((unsigned)((n_bins + 127) / 128), (unsigned)n_frames, (unsigned)n_clips);
  const float2* sc = d->mask_only ? nullptr : (const float2*)d_S_complex;
  if (w <= 8) hpss_kernel<8><<<grid, 128, 0, c->stream>>>(d_mag, sc, a, (float*)d_out_harm, (float*)d_out_perc);
  else if (w <= 16) hpss_kernel<16><<<grid, 128, 0, c->stream>>>(d_mag, sc, a, (float*)d_out_harm, (float*)d_out_perc);
  else if (w <= 32) hpss_kernel<32><<<grid, 128, 0, c->stream>>>(d_mag, sc, a, (float*)d_out_harm, (float*)d_out_perc);
  else hpss_kernel<64><<<grid, 128, 0, c->stream>>>(d_mag, sc, a, (float*)d_out_harm, (float*)d_out_perc);
  CUDA_TRY(cudaGetLastError());
  c->launches++;
  return B2L_OK;
}

extern "C" int b2l_reassign(b2l_ctx* c, const b2l_reassign_desc* d, const void* d_Sh, const void* d_Sdh,
                            const void* d_Sth, int64_t n_clips, int64_t n_frames, int64_t n_bins,
                            const float* d_bin_freqs, const float* d_frame_times, float* d_freqs, float* d_times,
                            float* d_mags) {
  if (!c || !d || !d_Sh || !d_bin_freqs || !d_frame_times || !d_freqs || !d_times || !d_mags)
    return fail(B2L_ERR_INVALID, "NULL argument");
  if ((d->reassign_frequencies && !d_Sdh) || (d->reassign_times && !d_Sth))
    return fail(B2L_ERR_INVALID, "missing derivative / time-weighted STFT");
  if (n_clips <= 0 || n_frames <= 0 || n_bins <= 0) return B2L_OK;
  if (n_frames > 0x7fffffffLL || n_bins > 0x7fffffffLL) return fail(B2L_ERR_UNSUPPORTED, "reassign: too large");
  ReassignArgs a;
  a.T = (int)n_frames;
  a.F = (int)n_bins;
  a.freq_scale = (float)(0.5 * (double)d->sr / 3.14159265358979323846);
  a.inv_sr = (float)(1.0 / (double)d->sr);
  a.mag_threshold = d->mag_threshold;
  a.max_freq = (float)(0.5 * (double)d->sr);
  a.max_time = d->max_time;
  a.do_freq = d->reassign_frequencies ? 1 : 0;
  a.do_time = d->reassign_times ? 1 : 0;
  a.apply_threshold = d->apply_threshold ? 1 : 0;
  a.fill_nan = d->fill_nan ? 1 : 0;
  a.clip = d->clip ? 1 : 0;
  DeviceGuard g(c->device);
  const long long n = (long long)n_clips * n_frames * n_bins;
  long long grid = (n + 256LL * 4 - 1) / (256LL * 4);
  if (grid > 16LL * c->sm_count) grid = 16LL * c->sm_count;
  reassign_kernel<<<(int)grid, 256, 0, c->stream>>>((const float2*)d_Sh, (const float2*)d_Sdh, (const float2*)d_Sth,
                                                    d_bin_freqs, d_frame_times, a, n, d_freqs, d_times, d_mags);
  CUDA_TRY(cudaGetLastError());
  c->launches++;
  return B2L_OK;
}

extern "C" int b2l_phase_vocoder(b2l_ctx* c, const void* d_D, int64_t n_clips, int64_t n_frames, int64_t n_bins,
                                 int64_t n_out, const int32_t* d_i0, const int32_t* d_i1, const int32_t* d_lo,
                                 const double* d_dx, void* d_out) {
  if (!c || !d_D || !d_i0 || !d_i1 || !d_lo || !d_dx || !d_out) return fail(B2L_ERR_INVALID, "NULL argument");
  if (n_clips <= 0 || n_bins <= 0 || n_out <= 0) return B2L_OK;
  if (n_frames < 2) return fail(B2L_ERR_UNSUPPORTED, "phase_vocoder needs at least two input frames");
  if (n_frames > 0x7fffffffLL || n_bins > 0x7fffffffLL || n_out > 0x7fffffffLL)
    return fail(B2L_ERR_UNSUPPORTED, "phase_vocoder: too large");
  DeviceGuard g(c->device);
  const long long threads = (long long)n_clips * n_bins;
  phase_vocoder_kernel<<<(unsigned)((threads + 127) / 128), 128, 0, c->stream>>>(
      (const float2*)d_D, (int)n_frames, (int)n_bins, n_clips, (int)n_out, d_i0, d_i1, d_lo, d_dx, (float2*)d_out);
  CUDA_TRY(cudaGetLastError());
  c->launches++;
  return B2L_OK;
}

extern "C" int b2l_unary(b2l_ctx* c, int32_t op, const float* d_in, int64_t n, float param, float* d_out) {
  if (!c || !d_in || !d_out) return fail(B2L_ERR_INVALID, "NULL argument");
  if (op < 0 || op > B2L_UNARY_DB_TO_AMPLITUDE) return fail(B2L_ERR_INVALID, "bad unary op %d", op);
  if (n <= 0) return B2L_OK;
  DeviceGuard g(c->device);
  long long grid = (n + 256LL * 8 - 1) / (256LL * 8);
  if (grid > 8LL * c->sm_count) grid = 8LL * c->sm_count;
  unary_kernel<<<(int)grid, 256, 0, c->stream>>>(d_in, n, op, param, d_out);
  CUDA_TRY(cudaGetLastError());
  c->launches++;
  return B2L_OK;
}

extern "C" int b2l_dct_project(b2l_ctx* c, const b2l_plan* p, const float* d_S, int64_t n_clips, int64_t n_frames,
                               float* d_mfcc) {
  if (!c || !p || !d_S || !d_mfcc) return fail(B2L_ERR_INVALID, "NULL argument");
  if (p->n_mfcc == 0) return fail(B2L_ERR_INVALID, "plan has no mfcc stage");
  if (n_clips <= 0 || n_frames <= 0) return B2L_OK;
  DeviceGuard g(c->device);
  return launch_dct(c, p, d_S, n_clips, n_frames, 0, d_mfcc);
}

extern "C" int b2l_gl_update(b2l_ctx* c, const void* d_rebuilt, const void* d_tprev, const float* d_S, float scale,
                             float eps, void* d_angles, int64_t n) {
  if (!c || !d_rebuilt || !d_S || !d_angles) return fail(B2L_ERR_INVALID, "NULL argument");
  if (n <= 0) return B2L_OK;
  DeviceGuard g(c->device);
  long long blocks = (n + 255) / 256;
  const long long cap = 8LL * c->sm_count;
  if (blocks > cap) blocks = cap;
  gl_update_kernel<<<(int)blocks, 256, 0, c->stream>>>((const float2*)d_rebuilt, (const float2*)d_tprev, d_S, scale, eps,
                                                     (float2*)d_angles, n);
  CUDA_TRY(cudaGetLastError());
  c->launches++;
  return B2L_OK;
}

extern "C" int b2l_transpose(b2l_ctx* c, const void* d_in, int64_t n_clips, int64_t rows, int64_t cols,
                             int32_t elem_bytes, void* d_out) {
  if (!c || !d_in || !d_out) return fail(B2L_ERR_INVALID, "NULL argument");
  if (n_clips <= 0 || rows <= 0 || cols <= 0) return B2L_OK;
  if (elem_bytes != 4 && elem_bytes != 8) return fail(B2L_ERR_INVALID, "elem_bytes must be 4 or 8");
  DeviceGuard g(c->device);
  dim3 block(32, 8);
  for (int64_t c0 = 0; c0 < n_clips; c0 += 65535) {   // the clip index rides in grid.z: larger batches go in slices
    const int64_t m = std::min<int64_t>(65535, n_clips - c0);
    dim3 grid((unsigned)((cols + 31) / 32), (unsigned)((rows + 31) / 32), (unsigned)m);
    const size_t off = (size_t)c0 * (size_t)rows * (size_t)cols;
    if (elem_bytes == 4)
      transpose_kernel<float><<<grid, block, 0, c->stream>>>((const float*)d_in + off, (int)rows, (int)cols, (float*)d_out + off);
    else
      transpose_kernel<float2><<<grid, block, 0, c->stream>>>((const float2*)d_in + off, (int)rows, (int)cols, (float2*)d_out + off);
    CUDA_TRY(cudaGetLastError());
    c->launches++;
  }
  return B2L_OK;
}

// ------------------------------------------------------------------ multi-GPU split / join
extern "C" int b2l_comm_unique_id(void* id128) {
  if (!id128) return fail(B2L_ERR_INVALID, "NULL argument");
  int rc = nccl_load();
  if (rc) return rc;
  ncclUniqueId id;
  NCCL_TRY(g_nccl.GetUniqueId(&id));
  memcpy(id128, &id, sizeof(id));
  return B2L_OK;
}
extern "C" int b2l_comm_init(b2l_ctx* c, const void* id128, int rank, int world) {
  if (!c || !id128) return fail(B2L_ERR_INVALID, "NULL argument");
  if (world < 1 || rank < 0 || rank >= world) return fail(B2L_ERR_INVALID, "bad rank %d / world %d", rank, world);
  int rc = nccl_load();
  if (rc) return rc;
  DeviceGuard g(c->device);
  ncclUniqueId id;
  memcpy(&id, id128, sizeof(id));
  NCCL_TRY(g_nccl.CommInitRank(&c->comm, world, id, rank));
  c->rank = rank;
  c->world = world;
  return B2L_OK;
}
extern "C" int b2l_comm_destroy(b2l_ctx* c) {
  if (!c || !c->comm) return B2L_OK;
  DeviceGuard g(c->device);
  cudaStreamSynchronize(c->stream);
  NCCL_TRY(g_nccl.CommDestroy(c->comm));
  c->comm = nullptr;
  c->world = 1;
  c->rank = 0;
  return B2L_OK;
}
extern "C" int b2l_comm_broadcast(b2l_ctx* c, void* d_buf, size_t bytes, int root) {
  if (!c || !c->comm) return fail(B2L_ERR_INVALID, "communicator not initialised");
  DeviceGuard g(c->device);
  NCCL_TRY(g_nccl.Broadcast(d_buf, d_buf, bytes, ncclChar, root, c->comm, c->stream));
  return B2L_OK;
}
extern "C" int b2l_comm_scatter(b2l_ctx* c, const void* d_full, void* d_shard, size_t shard_bytes, int root) {
  if (!c || !c->comm) return fail(B2L_ERR_INVALID, "communicator not initialised");
  DeviceGuard g(c->device);
  NCCL_TRY(g_nccl.GroupStart());
  if (c->rank == root)
    for (int r = 0; r < c->world; ++r)
      NCCL_TRY(g_nccl.Send((const char*)d_full + (size_t)r * shard_bytes, shard_bytes, ncclChar, r, c->comm, c->stream));
  NCCL_TRY(g_nccl.Recv(d_shard, shard_bytes, ncclChar, root, c->comm, c->stream));
  NCCL_TRY(g_nccl.GroupEnd());
  return B2L_OK;
}
extern "C" int b2l_comm_gather(b2l_ctx* c, const void* d_shard, void* d_full, size_t shard_bytes, int root) {
  if (!c || !c->comm) return fail(B2L_ERR_INVALID, "communicator not initialised");
  DeviceGuard g(c->device);
  NCCL_TRY(g_nccl.GroupStart());
  if (c->rank == root)
    for (int r = 0; r < c->world; ++r)
      NCCL_TRY(g_nccl.Recv((char*)d_full + (size_t)r * shard_bytes, shard_bytes, ncclChar, r, c->comm, c->stream));
  NCCL_TRY(g_nccl.Send(d_shard, shard_bytes, ncclChar, root, c->comm, c->stream));
  NCCL_TRY(g_nccl.GroupEnd());
  return B2L_OK;
}
extern "C" int b2l_comm_barrier(b2l_ctx* c) {
  if (!c || !c->comm) return fail(B2L_ERR_INVALID, "communicator not initialised");
  DeviceGuard g(c->device);
  int rc = ensure_clip_max(c, 1);
  if (rc) return rc;
  NCCL_TRY(g_nccl.AllReduce(c->d_clip_max, c->d_clip_max, 1, ncclChar, 0 /* ncclSum */, c->comm, c->stream));
  CUDA_TRY(cudaStreamSynchronize(c->stream));
  return B2L_OK;
}

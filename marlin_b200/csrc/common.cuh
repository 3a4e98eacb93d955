// Shared host-side plumbing for the CUDA translation units: error handling, the device
// context (one device, one stream, one stream-ordered memory pool) and typed device buffers.
#pragma once
#include <cuda_runtime.h>

#include <cstdarg>
#include <cstdio>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../include/b2m.h"

namespace b2m {

struct Error : std::runtime_error {
  int code;
  Error(int c, const std::string& m) : std::runtime_error(m), code(c) {}
};

inline std::string fmt(const char* f, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, f);
  vsnprintf(buf, sizeof(buf), f, ap);
  va_end(ap);
  return buf;
}

#define B2M_CUDA(expr)                                                                      \
  do {                                                                                      \
    cudaError_t e__ = (expr);                                                               \
    if (e__ != cudaSuccess)                                                                 \
      throw ::b2m::Error(B2M_ERR_CUDA, ::b2m::fmt("%s:%d: %s -> %s", __FILE__, __LINE__, #expr, \
                                                  cudaGetErrorString(e__)));                \
  } while (0)

#define B2M_CHECK_LAUNCH() B2M_CUDA(cudaGetLastError())

#define B2M_REQUIRE(cond, code, ...)                                   \
  do {                                                                 \
    if (!(cond)) throw ::b2m::Error((code), ::b2m::fmt(__VA_ARGS__));  \
  } while (0)

struct Ctx {
  int device = 0;
  int sm_count = 148;
  cudaStream_t stream = nullptr;  // the stream every helper launches on (see StreamSwap)
  cudaStream_t side = nullptr;    // second stream: sort of the next MSM while the current one accumulates
  cudaStream_t lane1 = nullptr;   // third stream: Msm::run_batch's second bucket-pass lane (`stream` is the first)
  cudaMemPool_t pool = nullptr;
  // multi-GPU MSM sharding (comm.cuh): rank / world of this process and its ncclComm_t
  int rank = 0, world = 1;
  void* comm = nullptr;
  // kernel-launch counter (bench.py reports it as gpu_launches)
  unsigned long long launches = 0;
  // optional per-kernel timing (CUDA events on `stream`) for the roofline line of bench.py
  struct Span {
    std::string name;
    double units;
    cudaEvent_t a, b;
  };
  bool profiling = false;
  std::vector<Span> spans;
  size_t span_begin(const char* name, double units) {
    if (!profiling) return (size_t)-1;
    Span s{name, units, nullptr, nullptr};
    cudaEventCreate(&s.a);
    cudaEventCreate(&s.b);
    cudaEventRecord(s.a, stream);
    spans.push_back(s);
    return spans.size() - 1;
  }
  void span_end(size_t id) {
    if (id != (size_t)-1) cudaEventRecord(spans[id].b, stream);
  }
  // {"name": {"launches": n, "ms": total, "units": total}, ...}; clears the log
  std::string span_report() {
    cudaStreamSynchronize(stream);
    struct Acc { double ms = 0, units = 0; long n = 0; };
    std::vector<std::pair<std::string, Acc>> acc;
    for (auto& s : spans) {
      float ms = 0;
      cudaEventElapsedTime(&ms, s.a, s.b);
      cudaEventDestroy(s.a);
      cudaEventDestroy(s.b);
      size_t k = 0;
      for (; k < acc.size(); k++)
        if (acc[k].first == s.name) break;
      if (k == acc.size()) acc.push_back({s.name, Acc()});
      acc[k].second.ms += ms; acc[k].second.units += s.units; acc[k].second.n++;
    }
    spans.clear();
    std::string out = "{";
    for (size_t k = 0; k < acc.size(); k++)
      out += fmt("%s\"%s\": {\"launches\": %ld, \"ms\": %.4f, \"units\": %.0f}", k ? ", " : "", acc[k].first.c_str(), acc[k].second.n,
                 acc[k].second.ms, acc[k].second.units);
    return out + "}";
  }

  explicit Ctx(int dev) : device(dev) {
    B2M_CUDA(cudaSetDevice(dev));
    cudaDeviceProp prop;
    B2M_CUDA(cudaGetDeviceProperties(&prop, dev));
    B2M_REQUIRE(prop.major >= 10, B2M_ERR_CUDA, "device %d is sm_%d%d; this library is built for sm_100a only",
                dev, prop.major, prop.minor);
    sm_count = prop.multiProcessorCount;
    B2M_CUDA(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
    B2M_CUDA(cudaStreamCreateWithFlags(&side, cudaStreamNonBlocking));
    B2M_CUDA(cudaStreamCreateWithFlags(&lane1, cudaStreamNonBlocking));
    B2M_CUDA(cudaDeviceGetDefaultMemPool(&pool, dev));
    unsigned long long thr = ~0ull;  // keep freed blocks cached in the pool
    B2M_CUDA(cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr));
  }
  ~Ctx() {
    if (lane1) cudaStreamDestroy(lane1);
    if (side) cudaStreamDestroy(side);
    if (stream) cudaStreamDestroy(stream);
  }
  void use() const { cudaSetDevice(device); }
  void sync() { B2M_CUDA(cudaStreamSynchronize(stream)); }
  void* alloc_bytes(size_t n) {
    void* p = nullptr;
    if (n == 0) n = 16;
    B2M_CUDA(cudaMallocAsync(&p, n, stream));
    return p;
  }
  void free_bytes(void* p) {
    if (p) cudaFreeAsync(p, stream);
  }
};

// Issue a scope's work on another stream: every helper (DBuf, scans, spans) follows ctx.stream.
struct StreamSwap {
  Ctx& c;
  cudaStream_t saved;
  StreamSwap(Ctx& ctx, cudaStream_t s) : c(ctx), saved(ctx.stream) { c.stream = s; }
  ~StreamSwap() { c.stream = saved; }
};

// RAII device array bound to a context's stream-ordered pool.
template <class T>
struct DBuf {
  Ctx* ctx = nullptr;
  T* p = nullptr;
  size_t n = 0;
  DBuf() = default;
  DBuf(Ctx& c, size_t count) : ctx(&c), n(count) { p = static_cast<T*>(c.alloc_bytes(count * sizeof(T))); }
  DBuf(const DBuf&) = delete;
  DBuf& operator=(const DBuf&) = delete;
  DBuf(DBuf&& o) noexcept : ctx(o.ctx), p(o.p), n(o.n) { o.p = nullptr; o.n = 0; }
  DBuf& operator=(DBuf&& o) noexcept {
    if (this != &o) {
      release();
      ctx = o.ctx; p = o.p; n = o.n;
      o.p = nullptr; o.n = 0;
    }
    return *this;
  }
  ~DBuf() { release(); }
  void release() {
    if (p && ctx) ctx->free_bytes(p);
    p = nullptr; n = 0;
  }
  void zero() { B2M_CUDA(cudaMemsetAsync(p, 0, n * sizeof(T), ctx->stream)); }
  void upload(const T* h, size_t count) { B2M_CUDA(cudaMemcpyAsync(p, h, count * sizeof(T), cudaMemcpyHostToDevice, ctx->stream)); }
  void download(T* h, size_t count) const {
    B2M_CUDA(cudaMemcpyAsync(h, p, count * sizeof(T), cudaMemcpyDeviceToHost, ctx->stream));
    B2M_CUDA(cudaStreamSynchronize(ctx->stream));
  }
};

inline unsigned div_up(size_t a, size_t b) { return (unsigned)((a + b - 1) / b); }

}  // namespace b2m

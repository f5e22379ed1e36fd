// Host-side plumbing of the library: handle, device / pinned arenas, per-kernel
// CUDA-event timers.  No algorithmic work happens here.
#pragma once
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdio.h>
#include <string.h>

#include <string>
#include <vector>

#include "common.cuh"

namespace bk {

struct CudaError {
  cudaError_t e;
  const char* what;
  int line;
};
#define BK_CUDA(x)                                              \
  do {                                                          \
    cudaError_t _e = (x);                                       \
    if (_e != cudaSuccess) throw bk::CudaError{_e, #x, __LINE__}; \
  } while (0)

struct ApiError {
  int code;
  std::string msg;
};
[[noreturn]] inline void fail(int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  throw ApiError{code, buf};
}

// Bump allocator over a few large chunks.  reset() keeps one chunk as large as
// everything the previous call needed, so steady-state calls never cudaMalloc.
template <bool PINNED_HOST>
class Arena {
 public:
  ~Arena() { release(); }
  void* alloc(size_t bytes) {
    bytes = (bytes + 255) & ~size_t(255);
    if (bytes == 0) bytes = 256;
    if (chunks_.empty() || used_ + bytes > chunks_.back().size) {
      size_t want = bytes > grow_ ? bytes : grow_;
      Chunk c{nullptr, want};
      if (PINNED_HOST) BK_CUDA(cudaMallocHost(&c.p, want));
      else BK_CUDA(cudaMalloc(&c.p, want));
      chunks_.push_back(c);
      used_ = 0;
      grow_ = want * 2;
    }
    void* r = (char*)chunks_.back().p + used_;
    used_ += bytes;
    total_ += bytes;
    return r;
  }
  template <typename T> T* get(size_t n) { return (T*)alloc(n * sizeof(T)); }
  void reset() {
    if (chunks_.size() > 1) {
      size_t sum = 0;
      for (auto& c : chunks_) sum += c.size;
      release();
      Chunk c{nullptr, sum};
      if (PINNED_HOST) BK_CUDA(cudaMallocHost(&c.p, sum));
      else BK_CUDA(cudaMalloc(&c.p, sum));
      chunks_.push_back(c);
    }
    used_ = 0;
    total_ = 0;
    ++resets_;
  }
  size_t resets() const { return resets_; }   // changes whenever earlier allocations may be reused
  void release() {
    for (auto& c : chunks_) {
      if (PINNED_HOST) cudaFreeHost(c.p);
      else cudaFree(c.p);
    }
    chunks_.clear();
    used_ = 0;
  }
  size_t total() const { return total_; }

 private:
  struct Chunk { void* p; size_t size; };
  std::vector<Chunk> chunks_;
  size_t used_ = 0, total_ = 0, grow_ = size_t(64) << 20, resets_ = 0;
};

enum KernelFamily : int {
  KF_NW_BATCH = 0, KF_EMIT, KF_SORT_COUNT, KF_SORT_SCAN, KF_SORT_SCATTER, KF_RUN_SELECT, KF_RUN_SCATTER, KF_SCAN,
  KF_GROUP, KF_INDEX, KF_PREP, KF_ASSEMBLE, KF_AUX_SORT, KF_REGION_KMERS, KF_COUNT_
};
static const char* const kKernelFamilyNames =
    "nw_batch;kmer_emit;sort_count;sort_scan;sort_scatter;run_select;run_scatter;scan;group_reads;index;prep;assemble;aux_sort;region_kmers";

struct KernelTimers {
  bool enabled = false;
  struct Rec { int fam; cudaEvent_t a, b; };
  std::vector<Rec> recs;
  std::vector<cudaEvent_t> pool;
  double ms[KF_COUNT_] = {0};
  int64_t launches[KF_COUNT_] = {0};
  cudaEvent_t get() {
    if (!pool.empty()) { cudaEvent_t e = pool.back(); pool.pop_back(); return e; }
    cudaEvent_t e;
    BK_CUDA(cudaEventCreate(&e));
    return e;
  }
  void collect() {
    for (auto& r : recs) {
      float t = 0;
      BK_CUDA(cudaEventSynchronize(r.b));
      BK_CUDA(cudaEventElapsedTime(&t, r.a, r.b));
      ms[r.fam] += t;
      pool.push_back(r.a);
      pool.push_back(r.b);
    }
    recs.clear();
  }
  void reset() {
    collect();
    for (int i = 0; i < KF_COUNT_; ++i) { ms[i] = 0; launches[i] = 0; }
  }
  ~KernelTimers() {
    for (auto& r : recs) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); }
    for (auto e : pool) cudaEventDestroy(e);
  }
};

// scope guard: times everything launched on `st` between construction and destruction
struct TimedLaunch {
  KernelTimers& t;
  cudaStream_t st;
  int fam;
  int n;
  cudaEvent_t a{}, b{};
  TimedLaunch(KernelTimers& t_, cudaStream_t st_, int fam_, int n_launches = 1) : t(t_), st(st_), fam(fam_), n(n_launches) {
    t.launches[fam] += n;
    if (t.enabled) { a = t.get(); b = t.get(); cudaEventRecord(a, st); }
  }
  ~TimedLaunch() {
    if (t.enabled) { cudaEventRecord(b, st); t.recs.push_back({fam, a, b}); }
  }
};

}  // namespace bk

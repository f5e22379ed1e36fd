// Common definitions for the breakmer_b200 device library (sm_100a).
//
// Execution-model shim: the per-region assembler (assemble.cuh) is written as
// warp-SPMD code -- every lane of a warp runs the same control flow, data
// parallel loops stride by `bk::lane()`.  The same source can be compiled by a
// host compiler with BK_SIM defined, where a "warp" is one lane; that build
// exists ONLY for tests/sim (logic debugging without a GPU).  It is never part
// of the shipped library and is not reachable from the product API.
#pragma once
#include <stdint.h>

#ifdef BK_SIM
#include <string.h>
#define BK_DEV inline
#define BK_HD inline
namespace bk {
constexpr int WARP = 1;
inline int lane() { return 0; }
inline void syncwarp() {}
inline unsigned ballot(bool p) { return p ? 1u : 0u; }
template <typename T> inline T shfl(T v, int) { return v; }
inline int popc(unsigned x) { return __builtin_popcount(x); }
inline int ffs(unsigned x) { return __builtin_ffs((int)x); }
inline int atomic_add(int* p, int v) { int o = *p; *p = o + v; return o; }
inline unsigned long long atomic_add(unsigned long long* p, unsigned long long v) { unsigned long long o = *p; *p = o + v; return o; }
inline void threadfence() {}
inline int atomic_cas(int* p, int cmp, int val) { int o = *p; if (o == cmp) *p = val; return o; }
inline unsigned atomic_max(unsigned* p, unsigned v) { unsigned o = *p; if (v > o) *p = v; return o; }
}  // namespace bk
#elif defined(BK_SIMT)
// tests/sim only: the kernels on a host SIMT emulator (tests/sim/simt_host.h, fibers + barriers at the warp and block
// collectives; tests/sim/cuda_runtime.h stands in for the runtime).  Like BK_SIM this build is a test tool; it is
// never part of the shipped library.
#include "cuda_runtime.h"
#define BK_DEV inline
#define BK_HD inline
#define BK_DYN_SMEM(T, name) T* name = reinterpret_cast<T*>(simt::dyn_smem())
namespace bk {
constexpr int WARP = 32;
inline int lane() { return simt::lane_id(); }
inline void syncwarp() { __syncwarp(); }
inline unsigned ballot(bool p) { return __ballot_sync(0xffffffffu, p); }
template <typename T> inline T shfl(T v, int src) { return __shfl_sync(0xffffffffu, v, src); }
inline int popc(unsigned x) { return __builtin_popcount(x); }
inline int ffs(unsigned x) { return __builtin_ffs((int)x); }
inline int atomic_add(int* p, int v) { return atomicAdd(p, v); }                    // (the emulator's, simt_host.h)
inline unsigned long long atomic_add(unsigned long long* p, unsigned long long v) { return atomicAdd(p, v); }
inline void threadfence() {}
inline int atomic_cas(int* p, int cmp, int val) { return atomicCAS(p, cmp, val); }
inline unsigned atomic_max(unsigned* p, unsigned v) { return atomicMax(p, v); }
}  // namespace bk
#else
#include <cuda_runtime.h>
#define BK_DEV __device__ __forceinline__
#define BK_HD __host__ __device__ __forceinline__
// the dynamic shared memory of a kernel (a macro so that the host emulator of tests/sim can supply it)
#define BK_DYN_SMEM(T, name) extern __shared__ __align__(16) T name[]
namespace bk {
constexpr int WARP = 32;
BK_DEV int lane() { return threadIdx.x & 31; }
BK_DEV void syncwarp() { __syncwarp(); }
BK_DEV unsigned ballot(bool p) { return __ballot_sync(0xffffffffu, p); }
template <typename T> BK_DEV T shfl(T v, int src) { return __shfl_sync(0xffffffffu, v, src); }
BK_DEV int popc(unsigned x) { return __popc(x); }
BK_DEV int ffs(unsigned x) { return __ffs((int)x); }
BK_DEV int atomic_add(int* p, int v) { return atomicAdd(p, v); }
BK_DEV unsigned long long atomic_add(unsigned long long* p, unsigned long long v) { return atomicAdd(p, v); }
BK_DEV void threadfence() { __threadfence(); }
BK_DEV int atomic_cas(int* p, int cmp, int val) { return atomicCAS(p, cmp, val); }
BK_DEV unsigned atomic_max(unsigned* p, unsigned v) { return atomicMax(p, v); }
}  // namespace bk
#endif

namespace bk {

// 2-bit base code, 4 = anything that is not ACGT (jellyfish skips the window;
// lower case is folded, oracle/kmers_py.py K1)
BK_HD int base_code(uint8_t c) {
  switch (c) {
    case 'A': case 'a': return 0;
    case 'C': case 'c': return 1;
    case 'G': case 'g': return 2;
    case 'T': case 't': return 3;
    default: return 4;
  }
}

// strict variant used for matching a k-mer inside a read/contig string: the
// reference uses str.find / re.search, which are case sensitive, and sample-only
// mers are upper case, so only upper-case ACGT can ever match
BK_HD int base_code_strict(uint8_t c) {
  switch (c) {
    case 'A': return 0;
    case 'C': return 1;
    case 'G': return 2;
    case 'T': return 3;
    default: return 4;
  }
}

constexpr uint64_t KEY_INVALID = ~0ull;

// per-region status written by device code: ST_OK (BK_OK in include/breakmer_b200.h), or the RR_* reason below the
// region stopped for, which bk_batch_wait reports as BK_ERR_CAPACITY
constexpr int ST_OK = 0;

// per-region report (AsmParams::region_report): fields and reason codes, the BK_RR_* values of include/breakmer_b200.h
enum {
  RR_REASON = 0, RR_PASS, RR_FIRST_REASON, RR_SEEDS, RR_FIND_READS, RR_CHECK_ALIGN, RR_GROWN, RR_REJ_SUPPORT,
  RR_REJ_LENGTH, RR_FIELDS
};
enum { RR_OK = 0, RR_READ_TOO_LONG, RR_CONTIG_TOO_LONG, RR_KMER_LIST_FULL, RR_TOO_MANY_CONTIGS, RR_OUTPUT_ARENA };
enum { RR_PASS_NONE = 0, RR_PASS_BATCHED, RR_PASS_LONG };
// why a grown contig failed the acceptance test (AsmParams::keep_rejected, bk_rejected_contigs): the BK_REJ_* values;
// RR_REJ_SUPPORT - REJ_SUPPORT + reason is its report counter
enum { REJ_NONE = 0, REJ_SUPPORT, REJ_LENGTH };
static_assert(RR_REJ_LENGTH == RR_REJ_SUPPORT + REJ_LENGTH - REJ_SUPPORT, "report counters follow the rejection reasons");

// hard limits of the packed DP cell (nw.cuh): 14-bit signed score field
constexpr int NW_MAX_LEN = 4095;

}  // namespace bk

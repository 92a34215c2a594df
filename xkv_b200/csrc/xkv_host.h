// xkv_b200 — host-side plumbing shared by the C-ABI translation units.
#pragma once

#include <cuda.h>
#include <cuda_runtime.h>

#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstring>

#include "../../include/xkv_b200.h"

namespace xkv {

// thread-local error text returned by xkv_last_error()
char* error_buffer();
int set_error(const char* fmt, ...);
extern std::atomic<long long> g_launch_count;

// Device predicate of the calling thread's next batched launches (normalise, batched slab reduction, Cholesky,
// rdiag update): matrix b is skipped when flags[b] == 0.  nullptr (the default) = unconditional.
const int*& launch_predicate();

// Launch priority of the calling thread's next GEMM launches: true = the lowest CTA-level priority whatever the stream's.
// The factorisation driver sets it around the projection A = X V, the last kernel of a chain (thousands of CTAs, nothing
// waits for its first results): the SMs that free up go to the latency-bound kernels of the other chains first
// (measured on the bench step: 39.4 -> 38.3 ms; the same hint on the Gram, the FIRST kernel of a chain, costs 0.7 ms).
bool& gemm_low_priority();
struct GemmLowPriorityScope {
  GemmLowPriorityScope() { gemm_low_priority() = true; }
  ~GemmLowPriorityScope() { gemm_low_priority() = false; }
};

inline cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }

// One-time per-DEVICE set-up (cudaFuncSetAttribute and occupancy queries apply to the current device only; a
// process that drives several GPUs must configure each).  Usage: static PerDevice<bool> done; if (!done()) {...}
constexpr int kMaxDevices = 64;
inline int current_device() {
  int d = 0;
  if (cudaGetDevice(&d) != cudaSuccess) d = 0;
  return d < 0 ? 0 : (d >= kMaxDevices ? kMaxDevices - 1 : d);
}
template <class T>
struct PerDevice {
  T v[kMaxDevices];
  PerDevice() {
    for (int i = 0; i < kMaxDevices; ++i) v[i] = T();
  }
  T& operator()() { return v[current_device()]; }
};
// SM count of the current device (cached per device)
int device_sm_count();

#define XKV_CHECK_CUDA(expr)                                                                        \
  do {                                                                                              \
    cudaError_t _e = (expr);                                                                        \
    if (_e != cudaSuccess)                                                                          \
      return ::xkv::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
  } while (0)

#define XKV_REQUIRE(cond, ...)                    \
  do {                                            \
    if (!(cond)) return ::xkv::set_error(__VA_ARGS__); \
  } while (0)

// after a kernel launch: count it and surface launch-configuration errors immediately
#define XKV_LAUNCHED()                 \
  do {                                 \
    ::xkv::g_launch_count.fetch_add(1); \
    XKV_CHECK_CUDA(cudaGetLastError()); \
  } while (0)

// Encode a 2-D bf16 tensor map (row-major [outer][ld], `inner` valid elements per row) with
// 128-byte swizzle. Returns 0 on success.
int encode_tmap_2d_bf16(CUtensorMap* map, const void* base, uint64_t inner, uint64_t outer, uint64_t ld_elems,
                        uint32_t box_inner, uint32_t box_outer);

}  // namespace xkv

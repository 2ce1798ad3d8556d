// Shared helpers for librgbmp (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>
#include "../../include/rgbmp.h"

namespace rgbmp {

// per-thread error text (the only thread-local in the library; it carries no op state)
inline char* err_buf() {
  static thread_local char buf[512] = {0};
  return buf;
}
inline int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(err_buf(), 512, fmt, ap);
  va_end(ap);
  return code;
}
inline int cuda_fail(cudaError_t e, const char* what) {
  snprintf(err_buf(), 512, "%s: %s", what, cudaGetErrorString(e));
  return (int)e;
}

#define RGBMP_CUDA(call)                                         \
  do {                                                           \
    cudaError_t _e = (call);                                     \
    if (_e != cudaSuccess) return ::rgbmp::cuda_fail(_e, #call); \
  } while (0)

#define RGBMP_LAUNCH_CHECK(name)                                      \
  do {                                                                \
    cudaError_t _e = cudaGetLastError();                              \
    if (_e != cudaSuccess) return ::rgbmp::cuda_fail(_e, name);       \
  } while (0)

struct DeviceGuard {
  int prev = -1;
  bool ok = true;
  explicit DeviceGuard(int dev) {
    if (cudaGetDevice(&prev) != cudaSuccess) { ok = false; return; }
    if (prev != dev && cudaSetDevice(dev) != cudaSuccess) ok = false;
    cur = dev;
  }
  ~DeviceGuard() {
    if (prev >= 0 && prev != cur) cudaSetDevice(prev);
  }
  int cur = -1;
};

constexpr int kSMs = 148;  // B200: 2 dies x 74 SMs

inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }
inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }
// fp32 rows read as float4: 16-byte aligned base, ld a multiple of 4
inline bool al16(const void* p, int64_t ld) { return (((uintptr_t)p) & 15) == 0 && (ld % 4) == 0; }

// carve aligned regions out of a caller workspace
struct Carver {
  char* base;
  size_t off = 0, cap;
  Carver(void* p, size_t c) : base((char*)p), cap(c) {}
  template <typename T>
  T* take(size_t n) {
    off = align_up(off, 256);
    T* r = (T*)(base + off);
    off += n * sizeof(T);
    return r;
  }
  bool ok() const { return off <= cap; }
};

}  // namespace rgbmp

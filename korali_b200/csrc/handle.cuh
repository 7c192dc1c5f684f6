// handle.cuh — the parts of a solver handle that do not depend on the solver (host code only): error reporting, tracked
// allocations, device selection, the pinned mirror of the device scalars, the <prefix>run loop and the get_array / set_array copies.
// Each solver's handle struct derives from Handle<H, S> and keeps its own fields; the four C ABIs (kcma_, kdea_, kmocma_, ktmcmc_)
// implement their entry points with these pieces.
#pragma once
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <string>
#include <type_traits>
#include <vector>

namespace kc {

// Device and pinned host allocations, freed together when their owner goes out of scope.
struct Allocations {
  std::vector<void*> dev, host;
  Allocations() = default;
  Allocations(const Allocations&) = delete;
  Allocations& operator=(const Allocations&) = delete;
  ~Allocations() {
    for (void* p : dev) cudaFree(p);
    for (void* p : host) cudaFreeHost(p);
  }
};

// count elements of T (at least one), zero-filled; a frees them
template <class T>
cudaError_t alloc(Allocations& a, T** p, size_t count) {
  const size_t bytes = sizeof(T) * (count ? count : 1);
  cudaError_t e = cudaMalloc((void**)p, bytes);
  if (e != cudaSuccess) return e;
  a.dev.push_back(*p);
  return cudaMemset(*p, 0, bytes);
}
template <class T>
cudaError_t alloc_host(Allocations& a, T** p, size_t count) {
  const size_t bytes = sizeof(T) * (count ? count : 1);
  cudaError_t e = cudaMallocHost((void**)p, bytes);
  if (e != cudaSuccess) return e;
  a.host.push_back(*p);
  memset(*p, 0, bytes);
  return cudaSuccess;
}

// H: the solver's handle struct; S: its block of device scalars (dSc), mirrored in pinned host memory (hSc).
template <class H, class S>
struct Handle {
  int device = 0;
  cudaStream_t stream = 0;
  uint64_t gen = 1, launches = 0;
  std::string err, reason;
  S* dSc = nullptr;
  S* hSc = nullptr;
  bool scalars_fresh = false;   // hSc holds what dSc holds (CMA-ES and DEA skip a pull while it is set)
  Allocations mem;
  // <prefix>last_error(NULL): the last failure of <prefix>create, or of a call with a NULL handle. One buffer per ABI.
  inline static char create_err[1024] = "";
  ~Handle() { cudaSetDevice(device); }   // mem frees its buffers after this
};

template <class H>
int vfail(H* h, const char* fmt, va_list ap) {
  if (h) {
    char buf[1024];
    vsnprintf(buf, sizeof(buf), fmt, ap);
    h->err = buf;
  } else {
    vsnprintf(H::create_err, sizeof(H::create_err), fmt, ap);
  }
  return 1;
}

// Records the message on the handle, or in the ABI's create-error buffer when h is NULL; returns 1.
template <class H>
int fail(H* h, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vfail(h, fmt, ap);
  va_end(ap);
  return 1;
}

// A failure of <prefix>create after the handle exists: reports like fail(NULL, ...) and destroys the half-built handle.
template <class H>
int create_fail(H*& h, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vfail((H*)nullptr, fmt, ap);
  va_end(ap);
  delete h;
  h = nullptr;
  return 1;
}

#define CUDA_OK(h, call)                                                                                                      \
  do {                                                                                                                        \
    cudaError_t e_ = (call);                                                                                                  \
    if (e_ != cudaSuccess) return kc::fail(h, "CUDA error %s at %s:%d (%s)", cudaGetErrorString(e_), __FILE__, __LINE__, #call); \
  } while (0)
#define CREATE_OK(h, call)                                                                                                    \
  do {                                                                                                                        \
    cudaError_t e_ = (call);                                                                                                  \
    if (e_ != cudaSuccess)                                                                                                    \
      return kc::create_fail(h, "CUDA error %s at %s:%d (%s)", cudaGetErrorString(e_), __FILE__, __LINE__, #call);             \
  } while (0)

// Fails when no CUDA device is visible or the index is out of range; otherwise makes the device current.
template <class H>
int open_device(int device) {
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) {
    cudaGetLastError();
    return fail<H>(nullptr, "libkcma needs a CUDA device (sm_100a); none is visible. There is no CPU fallback.");
  }
  if (device < 0 || device >= ndev) return fail<H>(nullptr, "invalid CUDA device %d", device);
  CUDA_OK((H*)nullptr, cudaSetDevice(device));
  return 0;
}

// The device scalars into the pinned mirror (pull) and back (push), on the handle's stream.
template <class H>
int pull(H* h) {
  CUDA_OK(h, cudaMemcpyAsync(h->hSc, h->dSc, sizeof(*h->hSc), cudaMemcpyDeviceToHost, h->stream));
  CUDA_OK(h, cudaStreamSynchronize(h->stream));
  h->scalars_fresh = true;
  return 0;
}
template <class H>
int pull_cached(H* h) { return h->scalars_fresh ? 0 : pull(h); }
template <class H>
int push(H* h) {
  CUDA_OK(h, cudaMemcpyAsync(h->dSc, h->hSc, sizeof(*h->hSc), cudaMemcpyHostToDevice, h->stream));
  CUDA_OK(h, cudaStreamSynchronize(h->stream));
  return 0;
}

// <prefix>run: generations until max_generations or a termination criterion; *done = the generations run, on every return.
template <class H>
int run(H* h, uint64_t max_generations, uint64_t* done, int (*check_termination)(H*, int*, const char**), int (*run_generation)(H*)) {
  int rc = h ? 0 : fail(h, "null solver handle"), fin = 0;
  uint64_t n = 0;
  while (!rc && n < max_generations) {
    rc = check_termination(h, &fin, nullptr);
    if (rc || fin) break;
    rc = run_generation(h);
    if (!rc) n++;
  }
  if (done) *done = n;
  return rc;
}

// A rows x cols array with leading dimension ld (in elements), on the device or in host memory (host arrays are dense).
enum class Elem { f64, i32, u32, u64 };
struct Array {
  void* p = nullptr;
  size_t rows = 0, cols = 0, ld = 0;
  Elem type = Elem::f64;
  bool host = false;
};
inline Array dense(void* p, size_t n, Elem type = Elem::f64) { return Array{p, 1, n, n, type, false}; }
inline Array pitched(void* p, size_t rows, size_t cols, size_t ld) { return Array{p, rows, cols, ld, Elem::f64, false}; }

// get_array: *count = the element count; with out == NULL nothing else. Otherwise the elements in row order, converted to Out.
// too_small is the solver's message for cap < count; it receives (key, cap, count).
template <class H, class Out>
int copy_out(H* h, const char* key, const Array& a, Out* out, size_t cap, size_t* count, const char* too_small) {
  const size_t n = a.rows * a.cols;
  if (count) *count = n;
  if (!out) return 0;
  if (cap < n) return fail(h, too_small, key, cap, n);
  if (n == 0) return 0;
  const size_t es = a.type == Elem::f64 || a.type == Elem::u64 ? 8 : 4;
  const bool direct = std::is_same<Out, double>::value && a.type == Elem::f64;
  std::vector<char> tmp(direct ? 0 : n * es);
  void* dst = direct ? (void*)out : (void*)tmp.data();
  if (a.host) {
    memcpy(dst, a.p, n * es);
  } else {
    CUDA_OK(h, cudaMemcpy2DAsync(dst, es * a.cols, a.p, es * a.ld, es * a.cols, a.rows, cudaMemcpyDeviceToHost, h->stream));
    CUDA_OK(h, cudaStreamSynchronize(h->stream));
  }
  if (direct) return 0;
  for (size_t i = 0; i < n; i++) {
    switch (a.type) {
      case Elem::f64: out[i] = (Out)((const double*)dst)[i]; break;
      case Elem::i32: out[i] = (Out)((const int32_t*)dst)[i]; break;
      case Elem::u32: out[i] = (Out)((const uint32_t*)dst)[i]; break;
      case Elem::u64: out[i] = (Out)((const uint64_t*)dst)[i]; break;
    }
  }
  return 0;
}

// set_array: exactly rows x cols doubles into a device array.
template <class H>
int copy_in(H* h, const char* key, const Array& a, const double* in, size_t count) {
  if (count != a.rows * a.cols) return fail(h, "size mismatch for '%s' (%zu != %zu)", key, count, a.rows * a.cols);
  CUDA_OK(h, cudaMemcpy2DAsync(a.p, sizeof(double) * a.ld, in, sizeof(double) * a.cols, sizeof(double) * a.cols, a.rows,
                               cudaMemcpyHostToDevice, h->stream));
  CUDA_OK(h, cudaStreamSynchronize(h->stream));
  return 0;
}

// A double on the handle, read by get_scalar and, when writable, written by set_scalar.
template <class H>
struct HostScalar {
  using Member = double H::*;
  const char* key;
  Member member;
  bool writable;
};
template <class H, size_t K>
double* host_scalar(H* h, const HostScalar<H> (&list)[K], const char* key, bool write) {
  for (const HostScalar<H>& s : list)
    if (!strcmp(key, s.key) && (s.writable || !write)) return &(h->*s.member);
  return nullptr;
}

}  // namespace kc

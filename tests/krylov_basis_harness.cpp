// extern "C" entry points over the FP32-basis launchers of the GMRES loop (hymls_b200/csrc/kernels.hpp), so that
// tests/test_gpu_krylov_basis.py can call them directly on device memory owned by torch and compare them with the
// FP64 launchers of tests/kernel_harness.cpp.
//
// Every wrapper calls one hymls:: launcher on the given stream, synchronises the stream and returns 0, the
// hymls::Error code the launcher threw, or HYMLS_B200_ERR_CUDA when the CUDA runtime reports an error.
#include <cuda_runtime.h>

#include <cstdint>
#include <exception>

#include "kernels.hpp"

namespace {

template <class F>
int run(void* stream, F&& launch) {
  try {
    launch(static_cast<cudaStream_t>(stream));
  } catch (const hymls::Error& e) {
    return e.code;
  } catch (const std::exception&) {
    return HYMLS_B200_ERR_ARG;
  }
  if (cudaStreamSynchronize(static_cast<cudaStream_t>(stream)) != cudaSuccess) return HYMLS_B200_ERR_CUDA;
  if (cudaGetLastError() != cudaSuccess) return HYMLS_B200_ERR_CUDA;
  return 0;
}

}  // namespace

extern "C" {

int kbh_multi_dot(const float* V, int64_t ldv, int k, const double* w, int64_t n, double* partial, double* h,
                  int accumulate, void* stream, int64_t* launches) {
  return run(stream, [&](cudaStream_t s) { hymls::multiDot(V, ldv, k, w, n, partial, h, accumulate, s, launches); });
}

int kbh_multi_axpy(const float* V, int64_t ldv, int k, const double* h, double* w, int64_t n, double sign, void* stream,
                   int64_t* launches) {
  return run(stream, [&](cudaStream_t s) { hymls::multiAxpy(V, ldv, k, h, w, n, sign, s, launches); });
}

int kbh_scale_narrow(const double* x, const double* nrm2, float* y, double* wide, int64_t n, void* stream,
                     int64_t* launches) {
  return run(stream, [&](cudaStream_t s) { hymls::scaleByInvNormNarrow(x, nrm2, y, wide, n, s, launches); });
}

}  // extern "C"

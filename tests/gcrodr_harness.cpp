// extern "C" entry points over the restart-phase launchers of GCRO-DR (hymls_b200/csrc/kernels.hpp: blockDot,
// combine), so that tests/test_gpu_gcrodr.py can call them directly on device memory owned by torch.
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

int64_t gh_block_dot_partial() { return (int64_t)hymls::blockDotPartial(); }

int gh_block_dot(const double* X, int64_t ldx, int nx, const double* Y, int64_t ldy, int ny, int64_t n,
                 double* partial, double* H, int64_t ldh, void* stream, int64_t* launches) {
  return run(stream, [&](cudaStream_t s) { hymls::blockDot(X, ldx, nx, Y, ldy, ny, n, partial, H, ldh, s, launches); });
}

int gh_combine(const double* X, int64_t ldx, int nx, const double* coef, int64_t ldc, double* Y, int64_t ldy, int ny,
               int64_t n, int accumulate, void* stream, int64_t* launches) {
  return run(stream,
             [&](cudaStream_t s) { hymls::combine(X, ldx, nx, coef, ldc, Y, ldy, ny, n, accumulate, s, launches); });
}

}  // extern "C"

// extern "C" entry points over the launchers of the bordered owner-distributed path (hymls_b200/csrc/kernels.hpp), so
// that tests/test_gpu_bordered_dist.py can call each kernel directly on device memory owned by torch.
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

int bdh_border_spmv_rows(const int64_t* ptr, const int* col, const double* val, const double* x, const double* V,
                         const double* W, int64_t ld, int m, const double* sv, const int* rows, int64_t nrows,
                         double* y, double* partial, double* dots, void* stream, int64_t* launches) {
  return run(stream, [&](cudaStream_t s) {
    hymls::borderSpmvRows(ptr, col, val, x, V, W, ld, m, sv, rows, nrows, y, partial, dots, s, launches);
  });
}

int bdh_multi_dot_rows(const double* V, int64_t ldv, int k, const double* w, int64_t n, double* partial, double* h,
                       const int* widx, const int* rows, void* stream, int64_t* launches) {
  return run(stream,
             [&](cudaStream_t s) { hymls::multiDot(V, ldv, k, w, n, partial, h, 0, s, launches, widx, rows); });
}

int bdh_border_correct_list(double* X, const int* idx, const double* Q, int64_t ld, int m, const double* S, int64_t n,
                            const int* list, void* stream, int64_t* launches) {
  return run(stream, [&](cudaStream_t s) { hymls::borderCorrect(X, idx, Q, ld, m, S, n, s, launches, list); });
}

int bdh_multi_dot_blocks() { return hymls::multiDotBlocks(); }

}  // extern "C"

// extern "C" entry points over the FP32-storage paths of the GEMV launchers and over narrowToFloat
// (hymls_b200/csrc/kernels.hpp), so that tests/test_gpu_single_inverse.py can call them directly on device memory
// owned by torch and compare them with the FP64 launchers of tests/kernel_harness.cpp.
//
// Every wrapper calls one hymls:: launcher on the given stream, synchronises the stream and returns 0, the
// hymls::Error code the launcher threw, or HYMLS_B200_ERR_CUDA when the CUDA runtime reports an error.  GemvArgs
// fields are passed flat, in the order of kernel_harness.cpp, with the matrices as floats (GemvArgs::A32).
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

hymls::GemvArgs gemvArgs32(const int* itemMat, const int* itemRow0, const int* n, const int* np,
                           const int64_t* matOff, const int64_t* vecOff, const int64_t* outOff, const int* nrows,
                           const int* ncols, const float* A32, const double* xin, const int* gather,
                           const double* xsub, const double* xprev, double* out, const int* scatter, int mode,
                           int rowsPerWarp) {
  hymls::GemvArgs a{};
  a.itemMat = itemMat;
  a.itemRow0 = itemRow0;
  a.n = n;
  a.np = np;
  a.matOff = matOff;
  a.vecOff = vecOff;
  a.outOff = outOff;
  a.nrows = nrows;
  a.ncols = ncols;
  a.A32 = A32;
  a.xin = xin;
  a.gather = gather;
  a.xsub = xsub;
  a.xprev = xprev;
  a.out = out;
  a.scatter = scatter;
  a.mode = mode;
  a.rowsPerWarp = rowsPerWarp;
  return a;
}

}  // namespace

#define SIH_GEMV_PARAMS                                                                                        \
  const int *itemMat, const int *itemRow0, const int *n, const int *np, const int64_t *matOff,                 \
      const int64_t *vecOff, const int64_t *outOff, const int *nrows, const int *ncols, const float *A32,      \
      const double *xin, const int *gather, const double *xsub, const double *xprev, double *out,              \
      const int *scatter, int mode, int rowsPerWarp
#define SIH_GEMV_ARGS                                                                                           \
  gemvArgs32(itemMat, itemRow0, n, np, matOff, vecOff, outOff, nrows, ncols, A32, xin, gather, xsub, xprev, out, \
             scatter, mode, rowsPerWarp)

extern "C" {

int sih_batched_gemv(SIH_GEMV_PARAMS, int numItems, int npMax, void* stream, int64_t* launches) {
  return run(stream, [&](cudaStream_t s) { hymls::batchedGemv(SIH_GEMV_ARGS, numItems, npMax, s, launches); });
}

// *accepted: the launcher's return value (false: nv vectors of npMax entries do not fit shared memory)
int sih_batched_gemv_multi(SIH_GEMV_PARAMS, int numItems, int npMax, int nv, int64_t ldIn, int64_t ldSub,
                           int64_t ldOut, int* accepted, void* stream, int64_t* launches) {
  return run(stream, [&](cudaStream_t s) {
    *accepted = hymls::batchedGemvMulti(SIH_GEMV_ARGS, numItems, npMax, nv, ldIn, ldSub, ldOut, s, launches);
  });
}

// the transposed GEMV of Compute: must refuse a narrowed store
int sih_batched_gemv_t(SIH_GEMV_PARAMS, int count, int npMax, void* stream, int64_t* launches) {
  return run(stream, [&](cudaStream_t s) { hymls::batchedGemvT(SIH_GEMV_ARGS, count, npMax, s, launches); });
}

int sih_narrow_to_float(const double* src, float* dst, int64_t n, int* overflow, void* stream, int64_t* launches) {
  return run(stream, [&](cudaStream_t s) { hymls::narrowToFloat(src, dst, n, overflow, s, launches); });
}

}  // extern "C"

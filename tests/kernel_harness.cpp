// extern "C" entry points over the launchers of libhymls_b200.so (hymls_b200/csrc/kernels.hpp), so that
// tests/test_gpu_kernels.py can call each CUDA kernel directly on device memory owned by torch.
//
// Every wrapper only marshals arguments: it calls one hymls:: launcher on the given stream, synchronises the
// stream and returns 0, the hymls::Error code the launcher threw, or HYMLS_B200_ERR_CUDA when the CUDA runtime
// reports an error.  `launches` is the launcher's kernel-launch counter (incremented, never reset here).
// GemvArgs fields are passed flat, in the order of the struct; a null pointer leaves the field unset.
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

hymls::GemvArgs gemvArgs(const int* itemMat, const int* itemRow0, const int* n, const int* np, const int64_t* matOff,
                         const int64_t* vecOff, const int64_t* outOff, const int* nrows, const int* ncols,
                         const double* A, const double* xin, const int* gather, const double* xsub,
                         const double* xprev, double* out, const int* scatter, int mode, int rowsPerWarp) {
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
  a.A = A;
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

#define KH_GEMV_PARAMS                                                                                         \
  const int *itemMat, const int *itemRow0, const int *n, const int *np, const int64_t *matOff,                 \
      const int64_t *vecOff, const int64_t *outOff, const int *nrows, const int *ncols, const double *A,       \
      const double *xin, const int *gather, const double *xsub, const double *xprev, double *out,              \
      const int *scatter, int mode, int rowsPerWarp
#define KH_GEMV_ARGS \
  gemvArgs(itemMat, itemRow0, n, np, matOff, vecOff, outOff, nrows, ncols, A, xin, gather, xsub, xprev, out, scatter, \
           mode, rowsPerWarp)

extern "C" {

int kh_invert_batched(double* W, double* F, const int64_t* off, const int* n, const int* np, int count, int npMax,
                      int* piv, int* perm, int* swap, int* info, void* stream, int64_t* launches) {
  return run(stream, [&](cudaStream_t s) {
    hymls::invertBatched(W, F, off, n, np, count, npMax, piv, perm, swap, info, s, launches);
  });
}

int kh_refine_inverse_batched(double* A, double* F, double* R, const int64_t* off, const int* n, const int* np,
                              int count, int npMax, void* stream, int64_t* launches) {
  return run(stream, [&](cudaStream_t s) {
    hymls::refineInverseBatched(A, F, R, off, n, np, count, npMax, s, launches);
  });
}

int kh_refine_inverse_sparse(const double* val, const int64_t* src, const int64_t* dst, const int64_t* listPtr,
                             int64_t dstBase, double* T, double* F, double* R, const int64_t* off, const int* n,
                             const int* np, int count, int npMax, void* stream, int64_t* launches) {
  return run(stream, [&](cudaStream_t s) {
    hymls::refineInverseSparse(val, src, dst, listPtr, dstBase, T, F, R, off, n, np, count, npMax, s, launches);
  });
}

int kh_dense_gemm(const double* A, int lda, const double* B, int ldb, double* C, int ldc, int M, int N, int K,
                  double alpha, double beta, void* stream, int64_t* launches) {
  return run(stream, [&](cudaStream_t s) {
    hymls::denseGemm(A, lda, B, ldb, C, ldc, M, N, K, alpha, beta, s, launches);
  });
}

int kh_batched_gemv(KH_GEMV_PARAMS, int numItems, int npMax, void* stream, int64_t* launches) {
  return run(stream, [&](cudaStream_t s) { hymls::batchedGemv(KH_GEMV_ARGS, numItems, npMax, s, launches); });
}

// *accepted: the launcher's return value (false: nv vectors of npMax entries do not fit shared memory)
int kh_batched_gemv_multi(KH_GEMV_PARAMS, int numItems, int npMax, int nv, int64_t ldIn, int64_t ldSub, int64_t ldOut,
                          int* accepted, void* stream, int64_t* launches) {
  return run(stream, [&](cudaStream_t s) {
    *accepted = hymls::batchedGemvMulti(KH_GEMV_ARGS, numItems, npMax, nv, ldIn, ldSub, ldOut, s, launches);
  });
}

// *accepted: the launcher's return value (false: npMax is above the warp-per-matrix kernel's limit)
int kh_small_gemv(KH_GEMV_PARAMS, const int* matList, int numMats, int npMax, int* accepted, void* stream,
                  int64_t* launches) {
  return run(stream, [&](cudaStream_t s) {
    *accepted = hymls::smallGemv(KH_GEMV_ARGS, matList, numMats, npMax, s, launches);
  });
}

int kh_cta_gemv(KH_GEMV_PARAMS, const int* matList, int numMats, int npMax, void* stream, int64_t* launches) {
  return run(stream, [&](cudaStream_t s) { hymls::ctaGemv(KH_GEMV_ARGS, matList, numMats, npMax, s, launches); });
}

int kh_gemv_rows_per_item() { return hymls::gemvRowsPerItem(); }

int kh_multi_dot(const double* V, int64_t ldv, int k, const double* w, int64_t n, double* partial, double* h,
                 int accumulate, const int* widx, void* stream, int64_t* launches) {
  return run(stream, [&](cudaStream_t s) {
    hymls::multiDot(V, ldv, k, w, n, partial, h, accumulate, s, launches, widx);
  });
}

int kh_multi_dot_blocks() { return hymls::multiDotBlocks(); }

int kh_multi_axpy(const double* V, int64_t ldv, int k, const double* h, double* w, int64_t n, double sign,
                  void* stream, int64_t* launches) {
  return run(stream, [&](cudaStream_t s) { hymls::multiAxpy(V, ldv, k, h, w, n, sign, s, launches); });
}

int kh_spmv(const int64_t* ptr, const int* col, const double* val, const double* x, double* y, int64_t n,
            double alpha, const double* b, const int* bidx, double beta, void* stream, int64_t* launches) {
  return run(stream, [&](cudaStream_t s) { hymls::spmv(ptr, col, val, x, y, n, alpha, b, bidx, beta, s, launches); });
}

int kh_householder(const int* uniqStart, int nuniq, const double* w, const double* in, double* out, double* vsumOut,
                   const double* vsumIn, double* X, const int* sepRow, void* stream, int64_t* launches) {
  return run(stream, [&](cudaStream_t s) {
    hymls::householder(uniqStart, nuniq, w, in, out, vsumOut, vsumIn, X, sepRow, s, launches);
  });
}

}  // extern "C"

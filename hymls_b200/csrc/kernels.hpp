// Host-callable launchers of the CUDA kernels (definitions in gj.cu, schur.cu, apply.cu).
#pragma once
#include <cuda_runtime.h>

#include <cstdint>
#include <vector>

#include "device.cuh"

namespace hymls {

// ---- gj.cu: batched dense inversion, W (workspace, destroyed) -> F (inverse), same offsets ----
void invertBatched(double* W, double* F, const int64_t* dOff, const int* dN, const int* dNp, int count, int npMax,
                   int* dPiv, int* dPerm, int* dSwap, int* dInfo, cudaStream_t s, int64_t* launches);

// One Newton-Schulz step X <- X + X (I - A X) on the inverses F of a batch (same offsets for A, F and the
// scratch R; A holds the ORIGINAL matrices and is destroyed).  Restores O(cond(A) eps) accuracy after the
// Gauss-Jordan inversion (whose forward error grows with cond(U)).
void refineInverseBatched(double* A, double* F, double* R, const int64_t* dOff, const int* dN, const int* dNp, int count,
                          int npMax, cudaStream_t s, int64_t* launches);

// the same step with the residual R = I - A X formed from the SPARSE original (dense-fill list src/dst of its entries,
// range listPtr[m]..listPtr[m+1] per matrix, dst relative to dstBase): one GEMM instead of two.  T: scratch (layout of R)
void refineInverseSparse(const double* val, const int64_t* src, const int64_t* dst, const int64_t* listPtr,
                         int64_t dstBase, double* T, double* F, double* R, const int64_t* dOff, const int* dN,
                         const int* dNp, int count, int npMax, cudaStream_t s, int64_t* launches);
// C (M x N) = alpha A (M x K) B (K x N) + beta C, row major, FP64 tensor cores; even dimensions / leading dimensions
void denseGemm(const double* A, int lda, const double* B, int ldb, double* C, int ldc, int M, int N, int K, double alpha,
               double beta, cudaStream_t s, int64_t* launches);

// ---- schur.cu ----
struct SchurArgs {
  // per local separator row R (row i of subdomain sd: R = sdRowPtr[sd] + i)
  const int* rowSd;
  const int* rowInst;      // group instance (global index) the row belongs to
  const int* rowLinkPos;   // position of the row inside its linked set
  const int* sdSep;        // separator position of the row
  const int64_t* sdRowPtr;
  const int *sdM, *sdN, *sdNp;
  const int64_t* a11Off;
  const double* Ainv;
  const double* val;       // values of this level's matrix
  const int64_t *s21Ptr, *s12Ptr, *s22Ptr;
  const int *s21Col, *s12Row, *s22Col;
  const int64_t *s21Src, *s12Src, *s22Src;
  // group instances
  const int64_t* sdInstPtr;
  const int *instLoc, *instLen, *instUniq, *instLink;
  // linked sets per subdomain
  const int64_t* sdLinkPtr;  // nsd+1
  const int* lnkSd;
  const int* lnkSize;
  const int64_t* lnkOff;     // offset of the S_LL block in wsSLL (chunk relative)
  // unique groups
  const int* uniqStart;      // nuniq+1 (separator positions)
  const int *uniqBlk, *uniqBlkOff;
  const double* wd;          // reflector used for the matrix transform (0 where the dense variant is the identity)
  const double* usign;
  // outputs
  const int64_t* redPtr;
  const int* redCol;
  double* redVal;
  const int* blkNp;
  const int64_t* blkOff;
  double* blkW;
  // workspace (per chunk)
  const int64_t* wsOffC;     // per subdomain: offset of its m x G arrays C and SV
  // dense path of the coarser levels (many entries per A21 row): D = A21(sd) A11(sd)^-1 by a DMMA GEMM
  const int64_t* wsOffD;     // per subdomain: offset of its m x np arrays A21d and D (chunk relative)
  double* A21d;              // densified A21(sd), m x np row major
  double* D;                 // nullptr: rows of A21 A11^-1 are accumulated sparsely inside k_schur_rows
  const int64_t *wsOffA, *wsOffS;  // per subdomain: offsets of A12d (np x mp) and SkD (m x mp), mp = roundup8(m)
  double* A12d;              // densified A12(sd)
  double* SkD;               // -D A12d = the dense -A21 A11^-1 A12 of the subdomain (nullptr: sparse product)
  double *wsC, *wsSV, *wsSLL;
  int dLen;                  // doubles reserved for the A21*Ainv row in shared memory
  int* info;
};
// rows of Sk for the local separator rows [R0, R1) (or rowList[R0..R1)) into the per-subdomain workspaces
void schurRows(const SchurArgs& a, int64_t R0, int64_t R1, int pass, size_t rowSmem, cudaStream_t s,
               int64_t* launches, const int64_t* rowList = nullptr);
// transformed V-sum x V-sum entries and separator-block entries of the subdomains [sd0, sd1) / linked sets
// [lk0, lk1) (or of the lists).  pass 1 stores; pass 2 adds WITHOUT atomics: the caller launches one colour of
// subdomains (no shared separator group) at a time, which fixes the order of every sum (reproducible Compute)
void schurScatter(const SchurArgs& a, int pass, int sd0, int sd1, int64_t lk0, int64_t lk1, size_t blkSmem,
                  cudaStream_t s, int64_t* launches, const int* sdList = nullptr, const int64_t* lkList = nullptr);
// D = A21(sd) * A11(sd)^-1 for the subdomains [sd0, sd1) (or sdList[sd0..sd1)) whose local rows are [R0, R1)
// (or rowList[R0..R1)); dLen = doubles of the chunk's A21d / D arrays
void schurGemm(const SchurArgs& a, int sd0, int sd1, int64_t R0, int64_t R1, int64_t dLen, int64_t aLen, int maxM,
               int maxNp, cudaStream_t s, int64_t* launches, const int* sdList = nullptr,
               const int64_t* rowList = nullptr);
// dense -A21 A11^-1 A12 added into denseS; the rows of one call belong to subdomains of one colour
void schurDense(const SchurArgs& a, int64_t R0, int64_t R1, double* denseS, int64_t ldS, size_t rowSmem,
                cudaStream_t s, int64_t* launches, const int64_t* rowList = nullptr);
void dropByValue(double* val, const int64_t* ptr, const int* col, double* diagScratch, int n, double tol,
                 cudaStream_t s, int64_t* launches);

// ---- apply.cu ----
struct GemvArgs {
  const int* itemMat;
  const int* itemRow0;
  const int *n, *np;
  const int64_t* matOff;   // offset of each matrix in A
  const int64_t* vecOff;   // offset of each matrix' segment in the packed vectors
  const int64_t* outOff;   // optional: offset of each matrix' segment in `out` (default: vecOff)
  const int* nrows;        // optional: only rows [0, nrows[mat]) are computed (default: all n)
  const int* ncols;        // optional: x is zero beyond its first ncols[mat] entries, the rows are read that far only
  const double* A;
  const float* A32;        // optional: the matrices stored in FP32 (narrowToFloat); when set, A is not read
  const double* xin;
  const int* gather;
  const double* xsub;      // optional: x_sd[q] = xin[...] - xsub[p]
  const double* xprev;
  double* out;
  const int* scatter;
  int mode;
  int rowsPerWarp;         // 0: default (4 rows per warp = 32-row slabs); otherwise the slab is 8 * rowsPerWarp rows
};
void batchedGemv(const GemvArgs& a, int numItems, int npMax, cudaStream_t s, int64_t* launches);
// nv = 2..4 vectors in one pass over the matrices (vector v of xin / xsub / out at v * ldIn / ldSub / ldOut; mode 0);
// false: does not fit shared memory, the caller loops over the columns
bool batchedGemvMulti(const GemvArgs& a, int numItems, int npMax, int nv, int64_t ldIn, int64_t ldSub, int64_t ldOut,
                      cudaStream_t s, int64_t* launches);
// many small matrices (np <= 256): one warp per matrix of matList[0..numMats) (nullptr: all); false = too large
// medium matrices (np <= 512 here): one CTA per matrix of matList
void ctaGemv(const GemvArgs& a, const int* matList, int numMats, int npMax, cudaStream_t s, int64_t* launches);
bool smallGemv(const GemvArgs& a, const int* matList, int numMats, int npMax, cudaStream_t s, int64_t* launches);
int gemvRowsPerItem();
// dst[i] = (float)src[i] (round to nearest even) for i in [0, n); *overflow = 1 where a finite entry becomes infinite
void narrowToFloat(const double* src, float* dst, int64_t n, int* overflow, cudaStream_t s, int64_t* launches);
void spmv(const int64_t* ptr, const int* col, const double* val, const double* x, double* y, int64_t n, double alpha,
          const double* b, const int* bidx, double beta, cudaStream_t s, int64_t* launches);
// indexing.cu: index arrays built on the device from the pattern
void buildRowPos(const int* intRow, int64_t nI, const int* sepRow, int64_t nS, int* rowPos, cudaStream_t s,
                 int64_t* launches);
void buildPosMat(const int* n, const int64_t* vecOff, int count, int64_t nI, int* posMat, cudaStream_t s,
                 int64_t* launches);
int64_t buildA11List(const int64_t* rowptr, const int* colidx, const int* intRow, const int* rowPos,
                     const int* posMat, const int* posSd, int64_t nI, const int* np, const int64_t* matOff,
                     const int64_t* vecOff, int count, DevBuf<int64_t>& src, DevBuf<int64_t>& dst,
                     DevBuf<int64_t>& listPtrDev, std::vector<int64_t>& listPtr, DeviceArena* scratch, cudaStream_t s,
                     int64_t* launches);
struct SplitOut {
  DevBuf<int64_t>* p12; DevBuf<int>* c12; DevBuf<int64_t>* src12;
  DevBuf<int64_t>* p21; DevBuf<int>* c21; DevBuf<int64_t>* src21;
  DevBuf<int64_t>* p22; DevBuf<int>* c22; DevBuf<int64_t>* src22;
  DevBuf<int64_t>* t12Ptr; DevBuf<int>* t12Col; DevBuf<int64_t>* t12Idx;
  int64_t nnz12 = 0, nnz21 = 0, nnz22 = 0;
};
void buildSplit(const int64_t* rowptr, const int* colidx, const int* intRow, const int* sepRow, const int* rowPos,
                const int* posMat, bool ownedOnly, bool want22, int64_t nI, int64_t nS, SplitOut& o,
                DeviceArena* scratch, cudaStream_t s, int64_t* launches);
struct LocalOut {
  DevBuf<int64_t>* s21Ptr; DevBuf<int>* s21Col; DevBuf<int64_t>* s21Src;
  DevBuf<int64_t>* s22Ptr; DevBuf<int>* s22Col; DevBuf<int64_t>* s22Src;
  DevBuf<int64_t>* s12Ptr; DevBuf<int>* s12Row; DevBuf<int64_t>* s12Src;
  int64_t nnz21 = 0, nnz22 = 0, nnz12 = 0;
};
void buildLocalPieces(const int64_t* rowptr, const int* colidx, const int* sepRow, const int* rowPos, const int* rowSd,
                      const int* sdSep, const int64_t* intPtr, const int* uniqStart, int nuniq, int64_t nS,
                      const int64_t* occPtr, const int* occSd, const int* occLoc, const int64_t* t12Ptr,
                      const int* t12Col, const int64_t* t12Idx, const int64_t* src12, int64_t totalRows, LocalOut& o,
                      DeviceArena* scratch, cudaStream_t s, int64_t* launches);
void gatherValues(const double* src, const int64_t* idx, double* dst, int64_t n, cudaStream_t s, int64_t* launches);
void scatterValues(const double* src, const int64_t* srcIdx, const int64_t* dstIdx, int64_t dstBase, double* dst,
                   int64_t n, cudaStream_t s, int64_t* launches);
void householder(const int* uniqStart, int nuniq, const double* w, const double* in, double* out, double* vsumOut,
                 const double* vsumIn, double* X, const int* sepRow, cudaStream_t s, int64_t* launches);
// h[i] (+)= V_i' w over the rows r in [0, n), or r = rows[0..n) with a row list; widx: w[widx[r]].  Deterministic
// (fixed reduction order, no atomics).
void multiDot(const double* V, int64_t ldv, int k, const double* w, int64_t n, double* partial, double* h,
              int accumulate, cudaStream_t s, int64_t* launches, const int* widx = nullptr, const int* rows = nullptr);
// the same over an FP32 basis (entries widened to double, FP64 products and sums), plain form
void multiDot(const float* V, int64_t ldv, int k, const double* w, int64_t n, double* partial, double* h,
              int accumulate, cudaStream_t s, int64_t* launches);
int multiDotBlocks();

void multiAxpy(const double* V, int64_t ldv, int k, const double* h, double* w, int64_t n, double sign,
               cudaStream_t s, int64_t* launches);
void multiAxpy(const float* V, int64_t ldv, int k, const double* h, double* w, int64_t n, double sign,
               cudaStream_t s, int64_t* launches);
// restart phase of GCRO-DR (deterministic, each X read once per 128 of its vectors and 32 of Y):
// H[j * ldh + i] = X_i' Y_j over rows [0, n), i < nx, j < ny; partial: blockDotPartial() doubles
void blockDot(const double* X, int64_t ldx, int nx, const double* Y, int64_t ldy, int ny, int64_t n, double* partial,
              double* H, int64_t ldh, cudaStream_t s, int64_t* launches);
size_t blockDotPartial();
// Y_j (+)= sum_{i < nx} X_i coef[j * ldc + i] for j < ny, rows [0, n) (coef on the device, column major)
void combine(const double* X, int64_t ldx, int nx, const double* coef, int64_t ldc, double* Y, int64_t ldy, int ny,
             int64_t n, int accumulate, cudaStream_t s, int64_t* launches);
void axpby(double a, const double* x, double b, double* y, int64_t n, cudaStream_t s, int64_t* launches);
void scaleByInvNorm(const double* x, const double* nrm2, double* y, int64_t n, cudaStream_t s, int64_t* launches);
// y = (float)(x * (1 / sqrt(*nrm2))) (FP64 product, round to nearest even); wide (nullptr: not written) = (double)y
void scaleByInvNormNarrow(const double* x, const double* nrm2, float* y, double* wide, int64_t n, cudaStream_t s,
                          int64_t* launches);
void setValue(double* x, int64_t idx, double v, cudaStream_t s, int64_t* launches);
void csrToDense(const int64_t* ptr, const int* col, const double* val, double* D, int n, int np, cudaStream_t s,
                int64_t* launches);
void putDirichlet(double* D, int n, int np, int fix, cudaStream_t s, int64_t* launches);
void gatherAdd(const double* b, const int* idx, const double* t, double* y, int64_t n, cudaStream_t s,
               int64_t* launches);
void scatterVec(const double* x, const int* idx, double* y, int64_t n, cudaStream_t s, int64_t* launches);
// y[idx[i]] = x[i] for idx[i] >= 0
void scatterVecMasked(const double* x, const int* idx, double* y, int64_t n, cudaStream_t s, int64_t* launches);

// ---- owner-computes multi-GPU path (apply.cu; used by dist.cu) ----
void spmvRows(const int64_t* ptr, const int* col, const double* val, const double* x, double* y, const int* rows,
              int64_t nrows, double alpha, const double* b, const int* bidx, double beta, int compact, cudaStream_t s,
              int64_t* launches);
void householderList(const int* uniqStart, const int* list, int nlist, const double* w, const double* in, double* out,
                     double* vsumOut, const double* vsumIn, double* X, const int* sepRow, cudaStream_t s,
                     int64_t* launches);
void packIdx(const double* x, const int* idx, double* out, int64_t n, cudaStream_t s, int64_t* launches);
void haloAdd(double* z, const int* node, const int64_t* ptr, const int64_t* src, const double* buf, int64_t n,
             cudaStream_t s, int64_t* launches);
void gatherAddList(const double* b, const int* bidx, const double* t, double* y, const int* list, int64_t n,
                   cudaStream_t s, int64_t* launches);

// ---- coarse.cu ----
void putDirichletCsr(double* val, const int64_t* ptr, const int* col, int row, cudaStream_t s, int64_t* launches);

// ---- bordered variant (apply.cu) ----
// out = Ainv^T x on an FP64 store (Compute only; refuses A32)
void batchedGemvT(const GemvArgs& a, int count, int npMax, cudaStream_t s, int64_t* launches);
// y = alpha A^T x through a host-built transposed index into A's values (deterministic: no atomics)
void spmvIndexed(const int64_t* ptr, const int* col, const int64_t* idx, const double* val, const double* x, double* y,
                 int64_t n, double alpha, cudaStream_t s, int64_t* launches);
void zeroAt(double* x, const int* idx, int64_t n, cudaStream_t s, int64_t* launches);
// X[idx[p]] -= sum_j Q[j*ld + p] S[j] for p in [0, n), or p = list[0..n) with a position list
void borderCorrect(double* X, const int* idx, const double* Q, int64_t ld, int m, const double* S, int64_t n,
                   cudaStream_t s, int64_t* launches, const int* list = nullptr);
void denseBorder(double* D, int n, int np, const double* V, const double* W, int64_t ld, const double* C, int m,
                 cudaStream_t s, int64_t* launches);

void borderRows(const double* dots, const double* C, const double* sv, int m, int i0, int i1, double* out,
                cudaStream_t s, int64_t* launches);
// owned rows r = rows[i] of [K V; W' C] in one pass: y[i] = (K x)[r] + (V sv)[r], dots[j] = sum_i W[j*ld + r] x[r]
// (this rank's partial sums, deterministic; partial: m * multiDotBlocks() doubles)
void borderSpmvRows(const int64_t* ptr, const int* col, const double* val, const double* x, const double* V,
                    const double* W, int64_t ld, int m, const double* sv, const int* rows, int64_t nrows, double* y,
                    double* partial, double* dots, cudaStream_t s, int64_t* launches);

}  // namespace hymls

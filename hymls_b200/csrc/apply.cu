// Kernels of Preconditioner::ApplyInverse (src/HYMLS_Preconditioner.cpp:930-1070),
// SchurPreconditioner::ApplyInverse / ApplyOT / ApplyBlockDiagonal / UpdateVsumRhs
// (src/HYMLS_SchurPreconditioner.cpp:1010-1093,1236-1265,1311-1346,1435-1459),
// MatrixBlock::Apply / ApplyInverse (src/HYMLS_MatrixBlock.cpp:294-385) and the vector kernels of the
// Krylov loop (Belos inside src/HYMLS_BaseSolver.cpp:347-356).  All of them are HBM-bandwidth bound.
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdint>

#include "device.cuh"
#include "kernels.hpp"

namespace hymls {

// ---------------------------------------------------------------------------------------------
// Batched dense mat-vec with the explicit inverses:  y_sd = Ainv_sd * x_sd  for every subdomain.
// The dominant kernel of ApplyInverse: streams 8 n_sd^2 bytes per subdomain exactly once.
// Work item = (matrix, slab of GEMV_ROWS rows); one warp per row, lanes stride the row with 16-byte
// loads, x_sd staged in shared memory.
//   x_sd[q] = xin[gather ? gather[p] : p] (- xsub[p]),  p = vecOff[mat] + q
//   rows [0, nrows[mat]) only when nrows is given (the first solve of ApplyInverse needs a leading block)
//   mode 0:  out[scatter ? scatter[p] : p] = acc
//   mode 1:  out[scatter ? scatter[p] : p] = xprev[p] - acc   (second A11 solve of ApplyInverse: fused update + export)
// (Tried in round 2 and dropped: two rows per warp at a time -- 8 loads in flight per lane, x read once for both rows --
//  needs 78 registers, 3 CTAs per SM instead of 4, and ran the full pass at 5.6 TB/s instead of 6.1 TB/s.)
// ---------------------------------------------------------------------------------------------
static constexpr int GEMV_ROWS = 32;   // rows per CTA
static constexpr int GEMV_T = 256;     // 8 warps, 4 rows each

__global__ void __launch_bounds__(GEMV_T)
k_batched_gemv(GemvArgs a) {
  const int item = blockIdx.x;
  const int mat = a.itemMat[item];
  const int r0 = a.itemRow0[item];
  const int n = a.n[mat], np = a.np[mat];
  const int nr = a.nrows ? a.nrows[mat] : n;
  const int64_t v0 = a.vecOff[mat];  // offset of this matrix' segment in the packed vectors
  const double* __restrict__ A = a.A + a.matOff[mat];
  extern __shared__ double sx[];
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  // columns read: all (padded) np, or the leading ncols[mat] rounded up to a 16-byte pair
  const int nc = a.ncols ? min(np, (a.ncols[mat] + 1) & ~1) : np;
  for (int q = tid; q < nc; q += GEMV_T) {
    double v = 0.0;
    if (q < n) {
      v = a.gather ? a.xin[a.gather[v0 + q]] : a.xin[v0 + q];
      if (a.xsub) v -= a.xsub[v0 + q];
    }
    sx[q] = v;
  }
  __syncthreads();
  // rows per warp: 4 (a 32-row slab per CTA) unless the work list was built with thinner slabs (a.rowsPerWarp:
  // single large matrices such as the coarse inverse need more CTAs than n / 32 to fill 148 SMs)
  const int rpw = a.rowsPerWarp > 0 ? a.rowsPerWarp : GEMV_ROWS / (GEMV_T / 32);
  for (int rr = 0; rr < rpw; ++rr) {
    const int r = r0 + wid * rpw + rr;
    if (r >= nr) break;
    const double2* __restrict__ row = reinterpret_cast<const double2*>(A + (int64_t)r * np);
    const double2* __restrict__ x2 = reinterpret_cast<const double2*>(sx);
    double acc0 = 0.0, acc1 = 0.0;
    const int n2 = nc >> 1;
    int q = lane;
    for (; q + 96 < n2; q += 128) {  // 4 independent 16-byte loads in flight per lane
      double2 m0 = __ldg(row + q), m1 = __ldg(row + q + 32), m2 = __ldg(row + q + 64), m3 = __ldg(row + q + 96);
      double2 b0 = x2[q], b1 = x2[q + 32], b2 = x2[q + 64], b3 = x2[q + 96];
      acc0 += m0.x * b0.x + m1.x * b1.x + m2.x * b2.x + m3.x * b3.x;
      acc1 += m0.y * b0.y + m1.y * b1.y + m2.y * b2.y + m3.y * b3.y;
    }
    for (; q < n2; q += 32) {
      double2 m0 = __ldg(row + q);
      double2 b0 = x2[q];
      acc0 += m0.x * b0.x;
      acc1 += m0.y * b0.y;
    }
    double acc = acc0 + acc1;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (lane == 0) {
      const double v = (a.mode == 0) ? acc : a.xprev[v0 + r] - acc;
      const int64_t o = (a.outOff ? a.outOff[mat] : v0) + r;
      a.out[a.scatter ? a.scatter[o] : o] = v;
    }
  }
}

void batchedGemv(const GemvArgs& a, int numItems, int npMax, cudaStream_t s, int64_t* launches) {
  if (numItems == 0) return;
  static PerDeviceLimit limit;
  size_t smem = (size_t)npMax * sizeof(double);
  if (smem > 227 * 1024) throw Error(HYMLS_B200_ERR_UNSUPPORTED, "dense block too large for the GEMV kernel");
  if (limit.raise(smem))
    HY_CUDA(cudaFuncSetAttribute(k_batched_gemv, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  k_batched_gemv<<<numItems, GEMV_T, smem, s>>>(a);
  ++*launches;
}
int gemvRowsPerItem() { return GEMV_ROWS; }

// ---------------------------------------------------------------------------------------------
// Small matrices (the separator blocks: 8 .. a few hundred rows, ~10^5 of them at 128^3): one WARP per matrix, grid-stride,
// x in per-warp shared memory, min(32, np/2) lanes per row and several rows per pass for the tiny ones.
// k_batched_gemv spends a 256-thread CTA per 32-row slab, which for these blocks is CTA-launch bound (ncu: 0.73 ms
// for 0.83 GB = 14 % of the DRAM throughput, profiles/r02_ncu_gemv_traffic.json).  mode 0 only.
// ---------------------------------------------------------------------------------------------
static constexpr int SMALL_NP_MAX = 2048;  // 8 warps x 2048 doubles = 128 KB of shared memory at most
__global__ void __launch_bounds__(256)
k_small_gemv(GemvArgs a, const int* __restrict__ matList, int numMats, int npMax) {
  extern __shared__ double sxAll[];  // 8 x npMax
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  double* sx = sxAll + wid * npMax;
  for (int idx = blockIdx.x * 8 + wid; idx < numMats; idx += gridDim.x * 8) {
    const int mat = matList ? matList[idx] : idx;
    const int n = a.n[mat], np = a.np[mat];
    const int64_t v0 = a.vecOff[mat];
    const double* __restrict__ A = a.A + a.matOff[mat];
    for (int q = lane; q < np; q += 32) sx[q] = q < n ? (a.gather ? a.xin[a.gather[v0 + q]] : a.xin[v0 + q]) : 0.0;
    __syncwarp();
    const int L = np >= 64 ? 32 : (np >= 32 ? 16 : (np >= 16 ? 8 : 4));  // lanes per row (np is a multiple of 8)
    const int rowsPerPass = 32 / L, sub = lane % L, rsel = lane / L;
    if (np <= 64) {
      // at most two 16-byte loads per lane and row: issue the loads of FOUR passes before the first use, otherwise the
      // warp waits one DRAM latency per pass (ncu r02: 0.55 ms for 0.84 GB with one pass in flight)
      const int q0 = 2 * sub, q1 = q0 + 2 * L;
      const bool two = q1 < np;
      const double x00 = sx[q0], x01 = sx[q0 + 1], x10 = two ? sx[q1] : 0.0, x11 = two ? sx[q1 + 1] : 0.0;
      for (int r0 = 0; r0 < n; r0 += 4 * rowsPerPass) {
        double2 m0[4], m1[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int r = r0 + u * rowsPerPass + rsel;
          const double* __restrict__ row = A + (int64_t)r * np;
          m0[u] = r < n ? __ldg(reinterpret_cast<const double2*>(row + q0)) : make_double2(0.0, 0.0);
          m1[u] = (r < n && two) ? __ldg(reinterpret_cast<const double2*>(row + q1)) : make_double2(0.0, 0.0);
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int r = r0 + u * rowsPerPass + rsel;
          double acc = m0[u].x * x00 + m0[u].y * x01;
          acc += m1[u].x * x10 + m1[u].y * x11;
          for (int o = L >> 1; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
          if (sub == 0 && r < n) {
            const int64_t o = (a.outOff ? a.outOff[mat] : v0) + r;
            a.out[a.scatter ? a.scatter[o] : o] = acc;
          }
        }
      }
    } else {
      for (int r0 = 0; r0 < n; r0 += rowsPerPass) {
        const int r = r0 + rsel;
        double acc = 0.0;
        if (r < n) {
          const double* __restrict__ row = A + (int64_t)r * np;
          for (int q = 2 * sub; q < np; q += 2 * L) {
            const double2 m = __ldg(reinterpret_cast<const double2*>(row + q));
            acc += m.x * sx[q] + m.y * sx[q + 1];
          }
        }
        for (int o = L >> 1; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
        if (sub == 0 && r < n) {
          const int64_t o = (a.outOff ? a.outOff[mat] : v0) + r;
          a.out[a.scatter ? a.scatter[o] : o] = acc;
        }
      }
    }
    __syncwarp();
  }
}
// Medium matrices (64 < np <= 512, e.g. the face blocks: a few hundred rows): one CTA per MATRIX, grid-stride; the 8
// warps share x in shared memory and take the rows round-robin.  The slab kernel would spend one CTA (launch, x staging,
// barrier) per 32 rows = per ~70 KB of such a block.
__global__ void __launch_bounds__(256)
k_cta_gemv(GemvArgs a, const int* __restrict__ matList, int numMats) {
  extern __shared__ double sx[];
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  for (int idx = blockIdx.x; idx < numMats; idx += gridDim.x) {
    const int mat = matList[idx];
    const int n = a.n[mat], np = a.np[mat];
    const int64_t v0 = a.vecOff[mat];
    const double* __restrict__ A = a.A + a.matOff[mat];
    for (int q = tid; q < np; q += 256) sx[q] = q < n ? (a.gather ? a.xin[a.gather[v0 + q]] : a.xin[v0 + q]) : 0.0;
    __syncthreads();
    const double2* __restrict__ x2 = reinterpret_cast<const double2*>(sx);
    const int n2 = np >> 1;
    for (int r = wid; r < n; r += 8) {
      const double2* __restrict__ row = reinterpret_cast<const double2*>(A + (int64_t)r * np);
      double acc0 = 0.0, acc1 = 0.0;
      int q = lane;
      for (; q + 32 < n2; q += 64) {
        const double2 m0 = __ldg(row + q), m1 = __ldg(row + q + 32);
        const double2 b0 = x2[q], b1 = x2[q + 32];
        acc0 += m0.x * b0.x + m0.y * b0.y;
        acc1 += m1.x * b1.x + m1.y * b1.y;
      }
      if (q < n2) {
        const double2 m0 = __ldg(row + q);
        const double2 b0 = x2[q];
        acc0 += m0.x * b0.x + m0.y * b0.y;
      }
      double acc = acc0 + acc1;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
      if (lane == 0) {
        const int64_t o = (a.outOff ? a.outOff[mat] : v0) + r;
        a.out[a.scatter ? a.scatter[o] : o] = acc;
      }
    }
    __syncthreads();
  }
}
void ctaGemv(const GemvArgs& a, const int* matList, int numMats, int npMax, cudaStream_t s, int64_t* launches) {
  if (numMats == 0) return;
  const size_t smem = (size_t)npMax * sizeof(double);
  k_cta_gemv<<<std::min(numMats, 148 * 8), 256, smem, s>>>(a, matList, numMats);
  ++*launches;
}

bool smallGemv(const GemvArgs& a, const int* matList, int numMats, int npMax, cudaStream_t s, int64_t* launches) {
  if (npMax > SMALL_NP_MAX) return false;
  if (numMats == 0) return true;
  const size_t smem = (size_t)8 * npMax * sizeof(double);
  static PerDeviceLimit limit;
  if (limit.raise(smem))
    HY_CUDA(cudaFuncSetAttribute(k_small_gemv, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  // resident CTAs per SM follow from the shared memory; a few waves of warps keep the load balanced
  const int perSm = std::max(1, std::min(8, (int)((200 * 1024) / std::max<size_t>(smem, 1))));
  const int blocks = std::min((numMats + 7) / 8, 148 * perSm);
  k_small_gemv<<<blocks, 256, smem, s>>>(a, matList, numMats, npMax);
  ++*launches;
  return true;
}

// ---------------------------------------------------------------------------------------------
// The same kernel for NV right-hand sides at once (Epetra_MultiVector with several columns: the reference resizes
// its subdomain solvers to the number of columns, src/HYMLS_MatrixBlock.cpp:335-344): every row of A11^-1 is loaded
// ONCE and multiplied with NV vectors staged in shared memory, so k columns cost one pass over the inverses instead
// of k.  Vector v of xin / xsub / out starts at v * ldIn / ldSub / ldOut.  mode 0 only.
// ---------------------------------------------------------------------------------------------
template <int NV>
__global__ void __launch_bounds__(GEMV_T)
k_batched_gemv_multi(GemvArgs a, int64_t ldIn, int64_t ldSub, int64_t ldOut) {
  const int item = blockIdx.x;
  const int mat = a.itemMat[item];
  const int r0 = a.itemRow0[item];
  const int n = a.n[mat], np = a.np[mat];
  const int nr = a.nrows ? a.nrows[mat] : n;
  const int64_t v0 = a.vecOff[mat];
  const double* __restrict__ A = a.A + a.matOff[mat];
  extern __shared__ double sx[];  // NV x np
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  for (int q = tid; q < np; q += GEMV_T) {
    const int64_t src = q < n ? (a.gather ? (int64_t)a.gather[v0 + q] : v0 + q) : 0;
#pragma unroll
    for (int v = 0; v < NV; ++v) {
      double x = 0.0;
      if (q < n) {
        x = a.xin[v * ldIn + src];
        if (a.xsub) x -= a.xsub[v * ldSub + v0 + q];
      }
      sx[v * np + q] = x;
    }
  }
  __syncthreads();
#pragma unroll
  for (int rr = 0; rr < GEMV_ROWS / (GEMV_T / 32); ++rr) {
    const int r = r0 + wid * (GEMV_ROWS / (GEMV_T / 32)) + rr;
    if (r >= nr) break;
    const double2* __restrict__ row = reinterpret_cast<const double2*>(A + (int64_t)r * np);
    double acc[NV];
#pragma unroll
    for (int v = 0; v < NV; ++v) acc[v] = 0.0;
    const int n2 = np >> 1;
    int q = lane;
    for (; q + 32 < n2; q += 64) {  // two independent 16-byte loads in flight per lane
      const double2 m0 = __ldg(row + q), m1 = __ldg(row + q + 32);
#pragma unroll
      for (int v = 0; v < NV; ++v) {
        const double2 b0 = reinterpret_cast<const double2*>(sx + v * np)[q];
        const double2 b1 = reinterpret_cast<const double2*>(sx + v * np)[q + 32];
        acc[v] += m0.x * b0.x + m0.y * b0.y + m1.x * b1.x + m1.y * b1.y;
      }
    }
    for (; q < n2; q += 32) {
      const double2 m0 = __ldg(row + q);
#pragma unroll
      for (int v = 0; v < NV; ++v) {
        const double2 b0 = reinterpret_cast<const double2*>(sx + v * np)[q];
        acc[v] += m0.x * b0.x + m0.y * b0.y;
      }
    }
#pragma unroll
    for (int v = 0; v < NV; ++v) {
      double t = acc[v];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
      acc[v] = t;
    }
    if (lane == 0) {
      const int64_t o = (a.outOff ? a.outOff[mat] : v0) + r;
      const int64_t dst = a.scatter ? (int64_t)a.scatter[o] : o;
#pragma unroll
      for (int v = 0; v < NV; ++v) a.out[v * ldOut + dst] = acc[v];
    }
  }
}

// nv in 2..4; returns false when the kernel cannot hold nv vectors of npMax entries in shared memory
bool batchedGemvMulti(const GemvArgs& a, int numItems, int npMax, int nv, int64_t ldIn, int64_t ldSub, int64_t ldOut,
                      cudaStream_t s, int64_t* launches) {
  if (numItems == 0) return true;
  const size_t smem = (size_t)npMax * nv * sizeof(double);
  if (smem > 200 * 1024 || nv < 2 || nv > 4) return false;
  static PerDeviceLimit lim2, lim3, lim4;
  if (nv == 2) {
    if (lim2.raise(smem)) HY_CUDA(cudaFuncSetAttribute(k_batched_gemv_multi<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k_batched_gemv_multi<2><<<numItems, GEMV_T, smem, s>>>(a, ldIn, ldSub, ldOut);
  } else if (nv == 3) {
    if (lim3.raise(smem)) HY_CUDA(cudaFuncSetAttribute(k_batched_gemv_multi<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k_batched_gemv_multi<3><<<numItems, GEMV_T, smem, s>>>(a, ldIn, ldSub, ldOut);
  } else {
    if (lim4.raise(smem)) HY_CUDA(cudaFuncSetAttribute(k_batched_gemv_multi<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k_batched_gemv_multi<4><<<numItems, GEMV_T, smem, s>>>(a, ldIn, ldSub, ldOut);
  }
  ++*launches;
  return true;
}

// ---------------------------------------------------------------------------------------------
// CSR SpMV variants (thread per row; rows have 1..~10 entries on level 0)
//   y[r] = alpha * (b ? b[bidx ? bidx[r] : r] : 0) + beta * sum_e val[e] x[col[e]]
// ---------------------------------------------------------------------------------------------
__global__ void k_spmv(const int64_t* __restrict__ ptr, const int* __restrict__ col, const double* __restrict__ val,
                       const double* __restrict__ x, double* __restrict__ y, int64_t n, double alpha,
                       const double* __restrict__ b, const int* __restrict__ bidx, double beta) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n) return;
  double s = 0.0;
  for (int64_t e = ptr[r]; e < ptr[r + 1]; ++e) s += val[e] * x[col[e]];
  double base = 0.0;
  if (b) base = alpha * b[bidx ? bidx[r] : r];
  y[r] = base + beta * s;
}
void spmv(const int64_t* ptr, const int* col, const double* val, const double* x, double* y, int64_t n, double alpha,
          const double* b, const int* bidx, double beta, cudaStream_t s, int64_t* launches) {
  if (n == 0) return;
  k_spmv<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(ptr, col, val, x, y, n, alpha, b, bidx, beta);
  ++*launches;
}

__global__ void k_gather_values(const double* __restrict__ src, const int64_t* __restrict__ idx,
                                double* __restrict__ dst, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[i] = src[idx[i]];
}
void gatherValues(const double* src, const int64_t* idx, double* dst, int64_t n, cudaStream_t s, int64_t* launches) {
  if (n == 0) return;
  k_gather_values<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(src, idx, dst, n);
  ++*launches;
}
// dst[dstIdx[i] - dstBase] = src[srcIdx[i]]   (dense fill of the A11 blocks of one chunk)
__global__ void k_scatter_values(const double* __restrict__ src, const int64_t* __restrict__ srcIdx,
                                 const int64_t* __restrict__ dstIdx, int64_t dstBase, double* __restrict__ dst,
                                 int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[dstIdx[i] - dstBase] = src[srcIdx[i]];
}
void scatterValues(const double* src, const int64_t* srcIdx, const int64_t* dstIdx, int64_t dstBase, double* dst,
                   int64_t n, cudaStream_t s, int64_t* launches) {
  if (n == 0) return;
  k_scatter_values<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(src, srcIdx, dstIdx, dstBase, dst, n);
  ++*launches;
}

// ---------------------------------------------------------------------------------------------
// Householder transforms on the separator vector, one warp per separator group (ApplyOT):
//   forward :  z = H rhs ;  vsumRhs[u] = z[first]                      (steps (1) and UpdateVsumRhs)
//   backward:  y[first] = vsumSol[u];  x2 = H y;  X[sepRow[p]] = x2[p]  (:1078-1081 + export :1052)
// H = 2 w w' - I with w = 0 for groups whose reflector is degenerate (sparse variant: H = -I).
// ---------------------------------------------------------------------------------------------
__global__ void k_householder(const int* __restrict__ uniqStart, int nuniq, const double* __restrict__ w,
                              const double* __restrict__ in, double* __restrict__ out, double* __restrict__ vsumOut,
                              const double* __restrict__ vsumIn, double* __restrict__ X, const int* __restrict__ sepRow) {
  const int u = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (u >= nuniq) return;
  const int lane = threadIdx.x & 31;
  const int a = uniqStart[u], z = uniqStart[u + 1];
  double t = 0.0;
  for (int p = a + lane; p < z; p += 32) {
    double v = (vsumIn && p == a) ? vsumIn[u] : in[p];
    t += w[p] * v;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
  for (int p = a + lane; p < z; p += 32) {
    double v = (vsumIn && p == a) ? vsumIn[u] : in[p];
    double r = 2.0 * w[p] * t - v;
    out[p] = r;
    if (vsumOut && p == a) vsumOut[u] = r;
    if (X) X[sepRow[p]] = r;
  }
}
void householder(const int* uniqStart, int nuniq, const double* w, const double* in, double* out, double* vsumOut,
                 const double* vsumIn, double* X, const int* sepRow, cudaStream_t s, int64_t* launches) {
  if (nuniq == 0) return;
  const int wpb = 8;
  k_householder<<<(nuniq + wpb - 1) / wpb, wpb * 32, 0, s>>>(uniqStart, nuniq, w, in, out, vsumOut, vsumIn, X, sepRow);
  ++*launches;
}

// ---------------------------------------------------------------------------------------------
// small vector kernels of the Krylov loop
// ---------------------------------------------------------------------------------------------
// partial[i * nblk + b] = sum over rows of block b of V_i[r] * w[r],  i = 0..k-1; r runs over [0, n) or, with a row
// list, over rows[0..n).
// The basis vectors are taken DOT_G at a time: one read of w[r] feeds DOT_G products with independent loads
// in flight, and the block reduction is paid once per group instead of once per vector.
static constexpr int DOT_G = 8;
__global__ void __launch_bounds__(256)
k_multi_dot(const double* __restrict__ V, int64_t ldv, int k, const double* __restrict__ w, int64_t n,
            double* __restrict__ partial, const int* __restrict__ widx, const int* __restrict__ rows) {
  __shared__ double red[DOT_G][8];
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int i0 = 0; i0 < k; i0 += DOT_G) {
    const int ng = min(DOT_G, k - i0);
    const double* __restrict__ v0 = V + (int64_t)i0 * ldv;
    double acc[DOT_G];
#pragma unroll
    for (int g = 0; g < DOT_G; ++g) acc[g] = 0.0;
    if (ng == DOT_G) {
      for (int64_t i = (int64_t)blockIdx.x * blockDim.x + tid; i < n; i += stride) {
        const int64_t r = rows ? (int64_t)rows[i] : i;
        const double wv = widx ? w[widx[r]] : w[r];
#pragma unroll
        for (int g = 0; g < DOT_G; ++g) acc[g] += v0[(int64_t)g * ldv + r] * wv;
      }
    } else {
      for (int64_t i = (int64_t)blockIdx.x * blockDim.x + tid; i < n; i += stride) {
        const int64_t r = rows ? (int64_t)rows[i] : i;
        const double wv = widx ? w[widx[r]] : w[r];
#pragma unroll
        for (int g = 0; g < DOT_G; ++g)
          if (g < ng) acc[g] += v0[(int64_t)g * ldv + r] * wv;
      }
    }
#pragma unroll
    for (int g = 0; g < DOT_G; ++g) {
      double s = acc[g];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
      if (lane == 0) red[g][wid] = s;
    }
    __syncthreads();
    if (tid < DOT_G * 8) {
      const int g = tid >> 3, j = tid & 7;
      double s = red[g][j];
#pragma unroll
      for (int o = 4; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o, 8);
      if (j == 0 && g < ng) partial[(int64_t)(i0 + g) * gridDim.x + blockIdx.x] = s;
    }
    __syncthreads();
  }
}
// h[i] (+)= sum_b partial[i*nblk+b]   (fixed order: deterministic)
__global__ void k_reduce_partials(const double* __restrict__ partial, int nblk, int k, double* __restrict__ h,
                                  int accumulate) {
  const int i = blockIdx.x;
  if (i >= k) return;
  __shared__ double red[32];
  double s = 0.0;
  for (int b = threadIdx.x; b < nblk; b += blockDim.x) s += partial[(int64_t)i * nblk + b];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if (lane == 0) red[wid] = s;
  __syncthreads();
  if (wid == 0) {
    s = lane < (blockDim.x >> 5) ? red[lane] : 0.0;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) h[i] = accumulate ? h[i] + s : s;
  }
}
static const int DOT_BLOCKS = 592;  // 4 x 148 SMs
void multiDot(const double* V, int64_t ldv, int k, const double* w, int64_t n, double* partial, double* h,
              int accumulate, cudaStream_t s, int64_t* launches, const int* widx, const int* rows) {
  if (k == 0) return;
  k_multi_dot<<<DOT_BLOCKS, 256, 0, s>>>(V, ldv, k, w, n, partial, widx, rows);
  k_reduce_partials<<<k, 256, 0, s>>>(partial, DOT_BLOCKS, k, h, accumulate);
  *launches += 2;
}
int multiDotBlocks() { return DOT_BLOCKS; }

// w += sign * sum_i h[i] V_i : coefficients in shared memory; a thread owns two adjacent rows (16-byte loads,
// eight of them in flight) when the basis is 16-byte aligned, one row otherwise
template <bool PAIR>
__global__ void __launch_bounds__(256)
k_multi_axpy(const double* __restrict__ V, int64_t ldv, int k, const double* __restrict__ h,
             double* __restrict__ w, int64_t n, double sign) {
  extern __shared__ double sh[];
  for (int i = threadIdx.x; i < k; i += blockDim.x) sh[i] = h[i];
  __syncthreads();
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  if (PAIR) {
    const int64_t n2 = n >> 1;
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n2; r += stride) {
      const double2* __restrict__ v = reinterpret_cast<const double2*>(V) + r;
      const int64_t ld2 = ldv >> 1;
      double2 s0 = make_double2(0.0, 0.0), s1 = s0, s2 = s0, s3 = s0;
      int i = 0;
      for (; i + 8 <= k; i += 8) {
        const double2 a0 = v[(int64_t)i * ld2], a1 = v[(int64_t)(i + 1) * ld2], a2 = v[(int64_t)(i + 2) * ld2],
                      a3 = v[(int64_t)(i + 3) * ld2], a4 = v[(int64_t)(i + 4) * ld2], a5 = v[(int64_t)(i + 5) * ld2],
                      a6 = v[(int64_t)(i + 6) * ld2], a7 = v[(int64_t)(i + 7) * ld2];
        s0.x += sh[i] * a0.x + sh[i + 4] * a4.x;
        s0.y += sh[i] * a0.y + sh[i + 4] * a4.y;
        s1.x += sh[i + 1] * a1.x + sh[i + 5] * a5.x;
        s1.y += sh[i + 1] * a1.y + sh[i + 5] * a5.y;
        s2.x += sh[i + 2] * a2.x + sh[i + 6] * a6.x;
        s2.y += sh[i + 2] * a2.y + sh[i + 6] * a6.y;
        s3.x += sh[i + 3] * a3.x + sh[i + 7] * a7.x;
        s3.y += sh[i + 3] * a3.y + sh[i + 7] * a7.y;
      }
      for (; i < k; ++i) {
        const double2 a0 = v[(int64_t)i * ld2];
        s0.x += sh[i] * a0.x;
        s0.y += sh[i] * a0.y;
      }
      double2* wp = reinterpret_cast<double2*>(w) + r;
      double2 wv = *wp;
      wv.x += sign * ((s0.x + s1.x) + (s2.x + s3.x));
      wv.y += sign * ((s0.y + s1.y) + (s2.y + s3.y));
      *wp = wv;
    }
    if ((n & 1) && blockIdx.x == 0 && threadIdx.x == 0) {  // odd tail row
      const int64_t r = n - 1;
      double s = 0.0;
      for (int i = 0; i < k; ++i) s += sh[i] * V[(int64_t)i * ldv + r];
      w[r] += sign * s;
    }
  } else {
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n; r += stride) {
      const double* __restrict__ v = V + r;
      double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
      int i = 0;
      for (; i + 8 <= k; i += 8) {
        const double a0 = v[(int64_t)i * ldv], a1 = v[(int64_t)(i + 1) * ldv], a2 = v[(int64_t)(i + 2) * ldv],
                     a3 = v[(int64_t)(i + 3) * ldv], a4 = v[(int64_t)(i + 4) * ldv], a5 = v[(int64_t)(i + 5) * ldv],
                     a6 = v[(int64_t)(i + 6) * ldv], a7 = v[(int64_t)(i + 7) * ldv];
        s0 += sh[i] * a0 + sh[i + 4] * a4;
        s1 += sh[i + 1] * a1 + sh[i + 5] * a5;
        s2 += sh[i + 2] * a2 + sh[i + 6] * a6;
        s3 += sh[i + 3] * a3 + sh[i + 7] * a7;
      }
      for (; i < k; ++i) s0 += sh[i] * v[(int64_t)i * ldv];
      w[r] += sign * ((s0 + s1) + (s2 + s3));
    }
  }
}
void multiAxpy(const double* V, int64_t ldv, int k, const double* h, double* w, int64_t n, double sign,
               cudaStream_t s, int64_t* launches) {
  if (k == 0 || n == 0) return;
  if ((size_t)k * sizeof(double) > 48 * 1024)
    throw Error(HYMLS_B200_ERR_UNSUPPORTED, "more than 6144 Krylov vectors in one orthogonalisation");
  const bool pair = !(ldv & 1) && !(reinterpret_cast<uintptr_t>(V) & 15) && !(reinterpret_cast<uintptr_t>(w) & 15);
  if (pair) k_multi_axpy<true><<<DOT_BLOCKS, 256, (size_t)k * sizeof(double), s>>>(V, ldv, k, h, w, n, sign);
  else k_multi_axpy<false><<<DOT_BLOCKS, 256, (size_t)k * sizeof(double), s>>>(V, ldv, k, h, w, n, sign);
  ++*launches;
}
// y = a*x + b*y   (b == 0 : y = a*x, no read of y)
__global__ void k_axpby(double a, const double* __restrict__ x, double b, double* __restrict__ y, int64_t n) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n; r += stride)
    y[r] = (b == 0.0) ? a * x[r] : a * x[r] + b * y[r];
}
void axpby(double a, const double* x, double b, double* y, int64_t n, cudaStream_t s, int64_t* launches) {
  if (n == 0) return;
  k_axpby<<<DOT_BLOCKS, 256, 0, s>>>(a, x, b, y, n);
  ++*launches;
}
// y = x * (1 / *dnorm)  with the norm on the device (avoids a host round trip)
__global__ void k_scale_by_inv(const double* __restrict__ x, const double* __restrict__ nrm2, double* __restrict__ y,
                               int64_t n) {
  const double inv = 1.0 / sqrt(*nrm2);
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n; r += stride) y[r] = x[r] * inv;
}
void scaleByInvNorm(const double* x, const double* nrm2, double* y, int64_t n, cudaStream_t s, int64_t* launches) {
  if (n == 0) return;
  k_scale_by_inv<<<DOT_BLOCKS, 256, 0, s>>>(x, nrm2, y, n);
  ++*launches;
}
// y[i] = b[idx[i]] + t[i]
__global__ void k_gather_add(const double* __restrict__ b, const int* __restrict__ idx, const double* __restrict__ t,
                             double* __restrict__ y, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) y[i] = b[idx[i]] + t[i];
}
void gatherAdd(const double* b, const int* idx, const double* t, double* y, int64_t n, cudaStream_t s,
               int64_t* launches) {
  if (n == 0) return;
  k_gather_add<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(b, idx, t, y, n);
  ++*launches;
}
__global__ void k_set_value(double* x, int64_t idx, double v) { x[idx] = v; }
void setValue(double* x, int64_t idx, double v, cudaStream_t s, int64_t* launches) {
  k_set_value<<<1, 1, 0, s>>>(x, idx, v);
  ++*launches;
}
// dense fill of the coarse matrix from CSR (+ FullDiag semantics) and Dirichlet rows/cols (PutDirichlet)
__global__ void k_csr_to_dense(const int64_t* __restrict__ ptr, const int* __restrict__ col,
                               const double* __restrict__ val, double* __restrict__ D, int n, int np) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n) return;
  for (int64_t e = ptr[r]; e < ptr[r + 1]; ++e) D[(int64_t)r * np + col[e]] = val[e];
}
__global__ void k_put_dirichlet(double* __restrict__ D, int n, int np, int fix) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  D[(int64_t)fix * np + i] = (i == fix) ? 1.0 : 0.0;
  if (i != fix) D[(int64_t)i * np + fix] = 0.0;
}
void csrToDense(const int64_t* ptr, const int* col, const double* val, double* D, int n, int np, cudaStream_t s,
                int64_t* launches) {
  if (n == 0) return;
  k_csr_to_dense<<<(n + 255) / 256, 256, 0, s>>>(ptr, col, val, D, n, np);
  ++*launches;
}
void putDirichlet(double* D, int n, int np, int fix, cudaStream_t s, int64_t* launches) {
  k_put_dirichlet<<<(n + 255) / 256, 256, 0, s>>>(D, n, np, fix);
  ++*launches;
}
// y[idx[i]] = x[i]  /  y[i] = x[idx[i]]
__global__ void k_scatter_vec(const double* __restrict__ x, const int* __restrict__ idx, double* __restrict__ y,
                              int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) y[idx[i]] = x[i];
}
__global__ void k_scatter_vec_masked(const double* __restrict__ x, const int* __restrict__ idx,
                                     double* __restrict__ y, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n && idx[i] >= 0) y[idx[i]] = x[i];
}
void scatterVecMasked(const double* x, const int* idx, double* y, int64_t n, cudaStream_t s, int64_t* launches) {
  if (n == 0) return;
  k_scatter_vec_masked<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(x, idx, y, n);
  ++*launches;
}
void scatterVec(const double* x, const int* idx, double* y, int64_t n, cudaStream_t s, int64_t* launches) {
  if (n == 0) return;
  k_scatter_vec<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(x, idx, y, n);
  ++*launches;
}

// ---------------------------------------------------------------------------------------------
// Row-list / group-list variants for the owner-computes multi-GPU path (dist.cu): a rank touches only the
// rows it owns (plus its halo), addressed through index lists into the global-length work vectors.
// ---------------------------------------------------------------------------------------------
// r = rows[i]:  y[compact ? i : r] = alpha * b[bidx ? bidx[r] : r] + beta * sum_e val[e] x[col[e]]
__global__ void k_spmv_rows(const int64_t* __restrict__ ptr, const int* __restrict__ col, const double* __restrict__ val,
                            const double* __restrict__ x, double* __restrict__ y, const int* __restrict__ rows,
                            int64_t nrows, double alpha, const double* __restrict__ b, const int* __restrict__ bidx,
                            double beta, int compact) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nrows) return;
  const int r = rows[i];
  double s = 0.0;
  for (int64_t e = ptr[r]; e < ptr[r + 1]; ++e) s += val[e] * x[col[e]];
  double base = 0.0;
  if (b) base = alpha * b[bidx ? bidx[r] : r];
  y[compact ? i : (int64_t)r] = base + beta * s;
}
void spmvRows(const int64_t* ptr, const int* col, const double* val, const double* x, double* y, const int* rows,
              int64_t nrows, double alpha, const double* b, const int* bidx, double beta, int compact, cudaStream_t s,
              int64_t* launches) {
  if (nrows == 0) return;
  k_spmv_rows<<<(unsigned)((nrows + 255) / 256), 256, 0, s>>>(ptr, col, val, x, y, rows, nrows, alpha, b, bidx, beta,
                                                               compact);
  ++*launches;
}
// k_householder over a list of unique groups
__global__ void k_householder_list(const int* __restrict__ uniqStart, const int* __restrict__ list, int nlist,
                                   const double* __restrict__ w, const double* __restrict__ in, double* __restrict__ out,
                                   double* __restrict__ vsumOut, const double* __restrict__ vsumIn,
                                   double* __restrict__ X, const int* __restrict__ sepRow) {
  const int idx = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (idx >= nlist) return;
  const int u = list[idx];
  const int lane = threadIdx.x & 31;
  const int a = uniqStart[u], z = uniqStart[u + 1];
  double t = 0.0;
  for (int p = a + lane; p < z; p += 32) {
    double v = (vsumIn && p == a) ? vsumIn[u] : in[p];
    t += w[p] * v;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
  for (int p = a + lane; p < z; p += 32) {
    double v = (vsumIn && p == a) ? vsumIn[u] : in[p];
    double r = 2.0 * w[p] * t - v;
    out[p] = r;
    if (vsumOut && p == a) vsumOut[u] = r;
    if (X) X[sepRow[p]] = r;
  }
}
void householderList(const int* uniqStart, const int* list, int nlist, const double* w, const double* in, double* out,
                     double* vsumOut, const double* vsumIn, double* X, const int* sepRow, cudaStream_t s,
                     int64_t* launches) {
  if (nlist == 0) return;
  const int wpb = 8;
  k_householder_list<<<(nlist + wpb - 1) / wpb, wpb * 32, 0, s>>>(uniqStart, list, nlist, w, in, out, vsumOut, vsumIn,
                                                                  X, sepRow);
  ++*launches;
}
// out[i] = x[idx[i]]  (halo pack, compact gather)
__global__ void k_pack_idx(const double* __restrict__ x, const int* __restrict__ idx, double* __restrict__ out,
                           int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = x[idx[i]];
}
void packIdx(const double* x, const int* idx, double* out, int64_t n, cudaStream_t s, int64_t* launches) {
  if (n == 0) return;
  k_pack_idx<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(x, idx, out, n);
  ++*launches;
}
// z[node[i]] = (base ? base[bidx[node[i]]] : 0) + z[node[i]] + sum_{e in [ptr[i], ptr[i+1])} buf[src[e]]: the partial
// sums received from the neighbouring ranks are added in a fixed order (by rank), one thread per node
__global__ void k_halo_add(double* __restrict__ z, const int* __restrict__ node, const int64_t* __restrict__ ptr,
                           const int64_t* __restrict__ src, const double* __restrict__ buf, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  double t = z[node[i]];
  for (int64_t e = ptr[i]; e < ptr[i + 1]; ++e) t += buf[src[e]];
  z[node[i]] = t;
}
void haloAdd(double* z, const int* node, const int64_t* ptr, const int64_t* src, const double* buf, int64_t n,
             cudaStream_t s, int64_t* launches) {
  if (n == 0) return;
  k_halo_add<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(z, node, ptr, src, buf, n);
  ++*launches;
}
// y[p] = b[bidx[p]] + t[p] for p = list[i]
__global__ void k_gather_add_list(const double* __restrict__ b, const int* __restrict__ bidx,
                                  const double* __restrict__ t, double* __restrict__ y, const int* __restrict__ list,
                                  int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int p = list[i];
  y[p] = b[bidx[p]] + t[p];
}
void gatherAddList(const double* b, const int* bidx, const double* t, double* y, const int* list, int64_t n,
                   cudaStream_t s, int64_t* launches) {
  if (n == 0) return;
  k_gather_add_list<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(b, bidx, t, y, list, n);
  ++*launches;
}

// ---------------------------------------------------------------------------------------------
// Kernels of the bordered variant (Preconditioner::ComputeBorder src/HYMLS_Preconditioner.cpp:519-588,
// SchurPreconditioner::ComputeBorder src/HYMLS_SchurPreconditioner.cpp:631-664, CoarseSolver's
// AugmentedMatrix src/HYMLS_CoarseSolver.cpp:200-224).  Borders have m <= a few columns and these run
// once per Compute, so they are plain coalesced kernels.
// ---------------------------------------------------------------------------------------------
// y_sd = Ainv_sd^T x_sd (the transposed subdomain solve of ComputeBorder :564-566): thread per column,
// rows streamed (coalesced across the columns of the row-major inverse)
__global__ void __launch_bounds__(256)
k_batched_gemv_t(GemvArgs a, int tilesPerMat) {
  const int mat = blockIdx.x / tilesPerMat;
  const int j = (blockIdx.x % tilesPerMat) * 256 + threadIdx.x;
  const int n = a.n[mat], np = a.np[mat];
  if ((blockIdx.x % tilesPerMat) * 256 >= n) return;
  const int64_t v0 = a.vecOff[mat];
  const double* __restrict__ A = a.A + a.matOff[mat];
  __shared__ double sx[256];
  double acc = 0.0;
  for (int i0 = 0; i0 < n; i0 += 256) {
    const int i = i0 + threadIdx.x;
    __syncthreads();
    sx[threadIdx.x] = i < n ? (a.gather ? a.xin[a.gather[v0 + i]] : a.xin[v0 + i]) : 0.0;
    __syncthreads();
    const int lim = min(256, n - i0);
    if (j < n)
      for (int q = 0; q < lim; ++q) acc += sx[q] * A[(int64_t)(i0 + q) * np + j];
  }
  if (j < n) a.out[v0 + j] = acc;
}
void batchedGemvT(const GemvArgs& a, int count, int npMax, cudaStream_t s, int64_t* launches) {
  if (count == 0 || npMax == 0) return;
  const int tiles = (npMax + 255) / 256;
  k_batched_gemv_t<<<(unsigned)(count * tiles), 256, 0, s>>>(a, tiles);
  ++*launches;
}
// y[r] = alpha * sum_e val[idx[e]] * x[col[e]]: SpMV with a transposed index (ptr/col/idx built on the host from
// the CSR pattern) over the values of the untransposed matrix -- A12' w of ComputeBorder without atomics
__global__ void k_spmv_indexed(const int64_t* __restrict__ ptr, const int* __restrict__ col,
                               const int64_t* __restrict__ idx, const double* __restrict__ val,
                               const double* __restrict__ x, double* __restrict__ y, int64_t n, double alpha) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n) return;
  double s = 0.0;
  for (int64_t e = ptr[r]; e < ptr[r + 1]; ++e) s += val[idx[e]] * x[col[e]];
  y[r] = alpha * s;
}
void spmvIndexed(const int64_t* ptr, const int* col, const int64_t* idx, const double* val, const double* x, double* y,
                 int64_t n, double alpha, cudaStream_t s, int64_t* launches) {
  if (n == 0) return;
  k_spmv_indexed<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(ptr, col, idx, val, x, y, n, alpha);
  ++*launches;
}
__global__ void k_zero_at(double* __restrict__ x, const int* __restrict__ idx, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) x[idx[i]] = 0.0;
}
void zeroAt(double* x, const int* idx, int64_t n, cudaStream_t s, int64_t* launches) {
  if (n == 0) return;
  k_zero_at<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(x, idx, n);
  ++*launches;
}
// X[idx[p]] -= sum_j Q[j*ld + p] * S[j]    (x1 -= Q1 S of the bordered ApplyInverse, Preconditioner.cpp:1036-1041)
// for p in [0, n) or, with a position list, p = list[0..n)
__global__ void k_border_correct(double* __restrict__ X, const int* __restrict__ idx, const double* __restrict__ Q,
                                 int64_t ld, int m, const double* __restrict__ S, int64_t n,
                                 const int* __restrict__ list) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int64_t p = list ? (int64_t)list[i] : i;
  double t = 0.0;
  for (int j = 0; j < m; ++j) t += Q[(int64_t)j * ld + p] * S[j];
  X[idx[p]] -= t;
}
void borderCorrect(double* X, const int* idx, const double* Q, int64_t ld, int m, const double* S, int64_t n,
                   cudaStream_t s, int64_t* launches, const int* list) {
  if (n == 0 || m == 0) return;
  k_border_correct<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(X, idx, Q, ld, m, S, n, list);
  ++*launches;
}
// augmented dense matrix [D V; W' C]: D is n x n inside an np x np row-major array, V, W are n x m
// (column major, leading dimension ld), C is m x m column major
__global__ void k_dense_border(double* __restrict__ D, int n, int np, const double* __restrict__ V,
                               const double* __restrict__ W, int64_t ld, const double* __restrict__ C, int m) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r < n) {
    for (int j = 0; j < m; ++j) {
      D[(int64_t)r * np + n + j] = V[(int64_t)j * ld + r];
      D[(int64_t)(n + j) * np + r] = W[(int64_t)j * ld + r];
    }
  } else if (r < n + m) {
    const int i = r - n;
    for (int j = 0; j < m; ++j) D[(int64_t)(n + i) * np + n + j] = C[i + (int64_t)j * m];
  }
}
void denseBorder(double* D, int n, int np, const double* V, const double* W, int64_t ld, const double* C, int m,
                 cudaStream_t s, int64_t* launches) {
  if (m == 0) return;
  k_dense_border<<<(n + m + 255) / 256, 256, 0, s>>>(D, n, np, V, W, ld, C, m);
  ++*launches;
}

// Rows r = rows[i] of the bordered operator [K V; W' C] on the owner distribution, one pass over the owned rows:
//   y[i] = sum_e val[e] x[col[e]] + sum_j V[j*ld + r] sv[j]
//   partial[j * gridDim.x + b] = sum over the rows of block b of W[j*ld + r] x[r]    (reduced like multiDot)
// x is a global-length vector valid at the owned rows and their matrix halo, sv the border part of the argument.
static constexpr int BORDER_G = 8;  // border columns per sweep of the dot part (m > 8 re-reads x)
__global__ void __launch_bounds__(256)
k_border_spmv_rows(const int64_t* __restrict__ ptr, const int* __restrict__ col, const double* __restrict__ val,
                   const double* __restrict__ x, const double* __restrict__ V, const double* __restrict__ W, int64_t ld,
                   int m, const double* __restrict__ sv, const int* __restrict__ rows, int64_t nrows,
                   double* __restrict__ y, double* __restrict__ partial) {
  __shared__ double red[BORDER_G][8];
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int j0 = 0; j0 < m; j0 += BORDER_G) {
    const int ng = min(BORDER_G, m - j0);
    double acc[BORDER_G];
#pragma unroll
    for (int g = 0; g < BORDER_G; ++g) acc[g] = 0.0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + tid; i < nrows; i += stride) {
      const int64_t r = rows[i];
      const double xr = x[r];
      if (j0 == 0) {
        double s = 0.0;
        for (int64_t e = ptr[r]; e < ptr[r + 1]; ++e) s += val[e] * x[col[e]];
        double t = 0.0;
        for (int j = 0; j < m; ++j) t += V[(int64_t)j * ld + r] * sv[j];
        y[i] = s + t;
      }
#pragma unroll
      for (int g = 0; g < BORDER_G; ++g)
        if (g < ng) acc[g] += W[(int64_t)(j0 + g) * ld + r] * xr;
    }
#pragma unroll
    for (int g = 0; g < BORDER_G; ++g) {
      double s = acc[g];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
      if (lane == 0) red[g][wid] = s;
    }
    __syncthreads();
    if (tid < BORDER_G * 8) {
      const int g = tid >> 3, j = tid & 7;
      double s = red[g][j];
#pragma unroll
      for (int o = 4; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o, 8);
      if (j == 0 && g < ng) partial[(int64_t)(j0 + g) * gridDim.x + blockIdx.x] = s;
    }
    __syncthreads();
  }
}
void borderSpmvRows(const int64_t* ptr, const int* col, const double* val, const double* x, const double* V,
                    const double* W, int64_t ld, int m, const double* sv, const int* rows, int64_t nrows, double* y,
                    double* partial, double* dots, cudaStream_t s, int64_t* launches) {
  if (m == 0) return;
  k_border_spmv_rows<<<DOT_BLOCKS, 256, 0, s>>>(ptr, col, val, x, V, W, ld, m, sv, rows, nrows, y, partial);
  k_reduce_partials<<<m, 256, 0, s>>>(partial, DOT_BLOCKS, m, dots, 0);
  *launches += 2;
}

// out[i - i0] = dots[i] + sum_j C[i + j*m] sv[j]  (border rows of BorderedOperator::Apply)
__global__ void k_border_rows(const double* __restrict__ dots, const double* __restrict__ C,
                              const double* __restrict__ sv, int m, int i0, int i1, double* __restrict__ out) {
  const int i = i0 + threadIdx.x;
  if (i >= i1) return;
  double t = dots[i];
  for (int j = 0; j < m; ++j) t += C[i + (int64_t)j * m] * sv[j];
  out[i - i0] = t;
}
void borderRows(const double* dots, const double* C, const double* sv, int m, int i0, int i1, double* out,
                cudaStream_t s, int64_t* launches) {
  if (i1 <= i0) return;
  k_border_rows<<<1, 32 * ((i1 - i0 + 31) / 32), 0, s>>>(dots, C, sv, m, i0, i1, out);
  ++*launches;
}

}  // namespace hymls

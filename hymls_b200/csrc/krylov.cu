// Krylov driver (BaseSolver::ApplyInverse -> Belos BlockGmresSolMgr / BlockCGSolMgr, block size 1).
//
// One GMRES(m) / CG serves both vector layouts of the library; KrylovLayout carries the operations in which they
// differ:
//   * replicated: every rank holds whole vectors of length n (+ border).  One GPU, and several ranks without the
//     owner path (HYMLS_B200_DIST=0, Number of Levels = 0).
//   * owner: a rank holds the rows it owns (DistPlan, dist.cu), packed, followed by the border entries, which every
//     rank keeps (bitwise equal); useDist() selects it.
// Independently of the layout, the caller's b, x0 and x live on one of the VecEnds distributions; load and store
// convert between the two at the ends of the solve, so the loop itself does not depend on the caller.
#include <algorithm>
#include <chrono>
#include <cmath>
#include <functional>
#include <random>

#include "dense_eig.hpp"
#include "engine.hpp"

namespace hymls {

// Solution-side vectors are what the driver keeps x, b, r, z in: `len` entries on this rank, `ld` allocated.  Every
// rank stores rows [row0, row0 + rows) of them in the GMRES basis, with stride rowLd; the first dotRows of those
// rows enter this rank's partial sums of the inner products (rows stored on several ranks are counted on one).
struct KrylovLayout {
  int64_t len = 0, ld = 0;
  int64_t rows = 0, rowLd = 0, row0 = 0, dotRows = 0;
  std::function<void(const double* in, double* out)> A, M;  // operator, preconditioner on solution-side vectors
  std::function<void(const double* u, const double* v, double* d)> dot;  // *d = u'v on the device
  // the Arnoldi step w = A M^-1 v, M^-1 A v or A v on basis rows; it may use kZ_ and kW_, which the driver leaves
  // free during a GMRES cycle
  std::function<void(const double* v, double* w)> step;
  std::function<const double*(const double* u)> expand;  // basis rows -> solution-side vector
  // b or x0 of the caller, followed by the border entries T (nullptr: zeros)
  std::function<void(const double* src, const double* T, double* dst, cudaMemcpyKind kind)> load;
  std::function<void(std::vector<double>& full)> keepOwn;  // a host vector of length n (+ border) -> this rank's part
  // x to the caller, and its border entries to S (nullptr: discarded)
  std::function<void(const double* src, double* dst, double* S, cudaMemcpyKind kind)> store;
};

// Replicated vectors; the GMRES basis is row-sharded over the ranks: rank r keeps rows [r*chunk, (r+1)*chunk) of every
// basis vector, so its Gram-Schmidt dots are local partial sums + one all-reduce of (k+1) doubles (the reference's
// SumAll).  The preconditioner wants its argument replicated, so v_k is all-gathered before each ApplyInverse.
// Distributed ends: one all-gather of the owned rows builds the full b (with one rank the owned rows are all rows),
// and each rank picks its rows out of x.
KrylovLayout Engine::replicatedLayout(bool left, bool right, VecEnds ends) {
  // With a border set the bordered system [K V; W' C] [x; s] = [b; T] is solved on vectors of length n + m
  // (HYMLS::BorderedSolver::ApplyInverse, src/HYMLS_BorderedSolver.cpp:159-219), preconditioned by the
  // bordered ApplyInverse.  ("Use Bordering" = true without a border is the plain solve with a warning there.)
  const int bm = borderM_;
  const int64_t nK = n_, n = n_ + bm;
  cudaStream_t s = stream_;
  const int P = comm_.active() ? comm_.size() : 1;
  const int64_t chunk = (n + P - 1) / P;
  const int64_t r0 = std::min<int64_t>(n, (int64_t)(comm_.active() ? comm_.rank() : 0) * chunk);
  const int64_t r1 = std::min<int64_t>(n, r0 + chunk);
  const int64_t nloc = r1 - r0;
  double *gath = nullptr, *wloc = nullptr;
  if (P > 1) {
    kS1_.alloc((size_t)P * chunk);  // all-gather target (padded)
    kS2_.alloc((size_t)chunk);      // local rows scratch
    HY_CUDA(cudaMemsetAsync(kS2_.p, 0, (size_t)chunk * sizeof(double), s));
    gath = kS1_.p;
    wloc = kS2_.p;
  }
  KrylovLayout L;
  L.len = L.ld = n;
  L.rows = L.dotRows = nloc;
  L.rowLd = chunk;
  L.row0 = r0;
  auto A = [=](const double* in, double* out) { operatorRows(in, out, 0, n); };
  auto M = [=](const double* in, double* out) {
    applyDevice(in, out, bm ? in + nK : nullptr, bm ? out + nK : nullptr);
  };
  auto expand = [=](const double* loc) -> const double* {
    if (P == 1) return loc;
    comm_.allGather(loc, gath, (size_t)chunk, s);
    return gath;
  };
  L.A = A;
  L.M = M;
  L.dot = [=](const double* u, const double* v, double* d) {
    multiDot(u, n, 1, v, n, kPartial_.p, d, 0, s, &launches_);
  };
  L.step = [=](const double* v, double* w) {
    const double* vfull = expand(v);
    if (right) {
      M(vfull, kZ_.p);
      operatorRows(kZ_.p, w, r0, r1);
    } else if (left) {
      if (P == 1) {
        A(vfull, kZ_.p);
      } else {
        operatorRows(vfull, wloc, r0, r1);
        comm_.allGather(wloc, gath, (size_t)chunk, s);
        HY_CUDA(cudaMemcpyAsync(kZ_.p, gath, n * sizeof(double), cudaMemcpyDeviceToDevice, s));
      }
      M(kZ_.p, kW_.p);
      HY_CUDA(cudaMemcpyAsync(w, kW_.p + r0, nloc * sizeof(double), cudaMemcpyDeviceToDevice, s));
    } else {
      operatorRows(vfull, w, r0, r1);
    }
  };
  L.expand = expand;
  DistPlan* D = P > 1 ? &levels_[0]->dist : nullptr;
  RowMapPlan* R = &rowMap_;
  const int64_t nOwn = D ? D->nOwn : nK;
  if (ends == VecEnds::Owned && D) bufG_.alloc(nOwn);
  L.load = [=](const double* src, const double* T, double* dst, cudaMemcpyKind kind) {
    if (ends == VecEnds::Replicated || (ends == VecEnds::Owned && !D)) {
      HY_CUDA(cudaMemcpyAsync(dst, src, nK * sizeof(double), kind, s));
    } else {
      if (ends == VecEnds::Owned) {
        HY_CUDA(cudaMemcpyAsync(bufG_.p, src, nOwn * sizeof(double), kind, s));
        scatterVec(bufG_.p, D->ownRows.p, dst, nOwn, s, &launches_);
      } else {
        if (R->nLocal) HY_CUDA(cudaMemcpyAsync(R->stage.p, src, R->nLocal * sizeof(double), kind, s));
        haloExchange(R->toOwner, R->stage.p, dst, true);
      }
      if (D) gatherOwned(dst, dst);
    }
    if (!bm) return;
    if (T) HY_CUDA(cudaMemcpyAsync(dst + nK, T, bm * sizeof(double), kind, s));
    else HY_CUDA(cudaMemsetAsync(dst + nK, 0, bm * sizeof(double), s));
  };
  L.keepOwn = [](std::vector<double>&) {};
  L.store = [=](const double* src, double* dst, double* S, cudaMemcpyKind kind) {
    if (ends == VecEnds::Replicated || (ends == VecEnds::Owned && !D)) {
      HY_CUDA(cudaMemcpyAsync(dst, src, nK * sizeof(double), kind, s));
    } else if (ends == VecEnds::Owned) {
      packIdx(src, D->ownRows.p, bufG_.p, nOwn, s, &launches_);
      HY_CUDA(cudaMemcpyAsync(dst, bufG_.p, nOwn * sizeof(double), kind, s));
    } else {
      double* cX = R->stage.p + std::max<int64_t>(R->nLocal, 1);
      haloExchange(R->fromOwner, src, cX, true);
      if (R->nLocal) HY_CUDA(cudaMemcpyAsync(dst, cX, R->nLocal * sizeof(double), kind, s));
    }
    if (bm && S) HY_CUDA(cudaMemcpyAsync(S, src + nK, bm * sizeof(double), kind, s));
  };
  return L;
}

// Packed owned rows, then the m border entries (bordered system [K V; W' C], replicated: only rank 0 counts them in
// the inner products); the basis lives in the same rows, so the loop contains no full-vector collective.  The
// operator and the preconditioner work on global-length vectors with the owned entries valid: kS1_ (argument) and
// kS2_ (result); the border adds one all-reduce of m doubles to the operator.
//
// Ends: owned rows are copied straight into / out of the packed rows (no collective of length n); the caller's map
// takes one grouped exchange each way (RowMapPlan, boundary.cu); replicated ends copy all n rows in and all-gather x.
KrylovLayout Engine::ownerLayout(bool left, bool right, VecEnds ends) {
  Level* L0 = levels_[0].get();
  DistPlan* D = &L0->dist;
  buildMatrixHalo();
  cudaStream_t s = stream_;
  const int bm = borderM_;
  const int64_t n = n_, nOwn = D->nOwn, ld = (D->maxOwn + bm + 7) & ~(int64_t)7;
  kS1_.alloc(n);
  kS2_.alloc(n);
  double* gIn = kS1_.p;
  double* gOut = kS2_.p;
  KrylovLayout L;
  L.len = L.rows = nOwn + bm;
  L.dotRows = nOwn + (comm_.rank() == 0 ? bm : 0);
  L.ld = L.rowLd = ld;
  L.row0 = 0;
  const int64_t dotRows = L.dotRows;
  auto toGlobal = [=](const double* c, double* full) { scatterVec(c, D->ownRows.p, full, nOwn, s, &launches_); };
  // outC = [K V; W' C] [full; sv] on the owned rows + the border rows; the halo of `full` is filled in place
  auto Aglobal = [=](double* full, const double* sv, double* outC) {
    haloExchange(D->mat, full, full, true);
    if (!bm) {
      spmvRows(L0->rowptr.p, L0->colidx.p, L0->val.p, full, outC, D->ownRows.p, nOwn, 0.0, nullptr, nullptr, 1.0, 1, s,
               &launches_);
      return;
    }
    borderSpmvRows(L0->rowptr.p, L0->colidx.p, L0->val.p, full, L0->bV.p, L0->bW.p, n, bm, sv, D->ownRows.p, nOwn,
                   outC, bPartial_.p, bDots_.p, s, &launches_);
    comm_.allReduceSum(bDots_.p, (size_t)bm, s);
    borderRows(bDots_.p, bC0_.p, sv, bm, 0, bm, outC + nOwn, s, &launches_);
  };
  auto Mglobal = [=](const double* inC, double* outFull) {  // with a border: S -> bS_
    toGlobal(inC, gIn);
    applyLevel0Dist(gIn, outFull, bm ? inC + nOwn : nullptr);
    stats_.num_apply_inverse++;
  };
  auto A = [=](const double* inC, double* outC) {
    toGlobal(inC, gIn);
    Aglobal(gIn, inC + nOwn, outC);
  };
  auto M = [=](const double* inC, double* outC) {
    Mglobal(inC, gOut);
    packIdx(gOut, D->ownRows.p, outC, nOwn, s, &launches_);
    if (bm) HY_CUDA(cudaMemcpyAsync(outC + nOwn, bS_.p, bm * sizeof(double), cudaMemcpyDeviceToDevice, s));
  };
  L.A = A;
  L.M = M;
  L.dot = [=](const double* u, const double* v, double* d) {
    multiDot(u, ld, 1, v, dotRows, kPartial_.p, d, 0, s, &launches_);
    comm_.allReduceSum(d, 1, s);
  };
  L.step = [=](const double* v, double* w) {
    if (right) {  // the global result of M^-1 goes straight into the operator
      Mglobal(v, gOut);
      Aglobal(gOut, bS_.p, w);
    } else if (left) {
      A(v, kW_.p);
      M(kW_.p, w);
    } else {
      A(v, w);
    }
  };
  L.expand = [](const double* u) { return u; };
  RowMapPlan* R = &rowMap_;
  L.load = [=](const double* src, const double* T, double* dst, cudaMemcpyKind kind) {
    if (ends == VecEnds::Owned) {
      HY_CUDA(cudaMemcpyAsync(dst, src, nOwn * sizeof(double), kind, s));
    } else {
      if (ends == VecEnds::Replicated) {
        HY_CUDA(cudaMemcpyAsync(gOut, src, n * sizeof(double), kind, s));
      } else {
        if (R->nLocal) HY_CUDA(cudaMemcpyAsync(R->stage.p, src, R->nLocal * sizeof(double), kind, s));
        haloExchange(R->toOwner, R->stage.p, gOut, true);
      }
      packIdx(gOut, D->ownRows.p, dst, nOwn, s, &launches_);
    }
    if (!bm) return;
    if (T) HY_CUDA(cudaMemcpyAsync(dst + nOwn, T, bm * sizeof(double), kind, s));
    else HY_CUDA(cudaMemsetAsync(dst + nOwn, 0, bm * sizeof(double), s));
  };
  L.keepOwn = [=](std::vector<double>& full) {  // n + m host numbers -> owned rows + border entries
    std::vector<double> own(nOwn + bm);
    for (int64_t i = 0; i < nOwn; ++i) own[i] = full[D->hOwnRows[i]];
    for (int j = 0; j < bm; ++j) own[nOwn + j] = full[n + j];
    full.swap(own);
  };
  L.store = [=](const double* src, double* dst, double* S, cudaMemcpyKind kind) {
    if (ends == VecEnds::Owned) {
      HY_CUDA(cudaMemcpyAsync(dst, src, nOwn * sizeof(double), kind, s));
    } else if (ends == VecEnds::Replicated) {  // like the single-GPU entry point
      toGlobal(src, gIn);
      gatherOwned(gIn, gOut);
      HY_CUDA(cudaMemcpyAsync(dst, gOut, n * sizeof(double), kind, s));
    } else {
      double* cX = R->stage.p + std::max<int64_t>(R->nLocal, 1);
      toGlobal(src, gIn);
      haloExchange(R->fromOwner, gIn, cX, true);
      if (R->nLocal) HY_CUDA(cudaMemcpyAsync(dst, cX, R->nLocal * sizeof(double), kind, s));
    }
    if (bm && S) HY_CUDA(cudaMemcpyAsync(S, src + nOwn, bm * sizeof(double), kind, s));
  };
  return L;
}

// ---- GCRO-DR (Parks, de Sturler, Mackey, Johnson, Maiti, SIAM J. Sci. Comput. 28(5), 2006, Algorithm 2) ----
// The recycled space: U in kRec_ (block recU_), C = A^ U with C' C = I in the recDim_ slots before the Arnoldi vectors,
// A^ = L.step.  Inside a cycle U enters scaled, Utilde = U D with D = diag(1 / ||u_i||) (recD_), so the first kc
// columns of Ghat are D.  The small matrices are formed on every rank from all-reduced partial sums and handled by the
// host routines of dense_eig.cpp, so every rank makes the same choices.

// upper triangular inverse of R (n x n, column major)
static std::vector<double> upperInverse(const std::vector<double>& R, int n) {
  std::vector<double> X((size_t)n * n, 0.0);
  for (int j = 0; j < n; ++j) {
    X[(size_t)j * n + j] = 1.0 / R[(size_t)j * n + j];
    for (int i = j - 1; i >= 0; --i) {
      double t = 0.0;
      for (int l = i + 1; l <= j; ++l) t += R[(size_t)l * n + i] * X[(size_t)j * n + l];
      X[(size_t)j * n + i] = -t / R[(size_t)i * n + i];
    }
  }
  return X;
}

// H = X' Y (nx x ny, column major) over this layout's rows, all-reduced, on the host
std::vector<double> Engine::crossProducts(const KrylovLayout& L, const double* X, int nx, const double* Y, int ny) {
  cudaStream_t s = stream_;
  blockDot(X, L.rowLd, nx, Y, L.rowLd, ny, L.dotRows, kPartialB_.p, kSmall_.p, nx, s, &launches_);
  comm_.allReduceSum(kSmall_.p, (size_t)nx * ny, s);
  std::vector<double> h((size_t)nx * ny);
  HY_CUDA(cudaMemcpyAsync(h.data(), kSmall_.p, h.size() * sizeof(double), cudaMemcpyDeviceToHost, s));
  HY_CUDA(cudaStreamSynchronize(s));
  return h;
}

void Engine::recycleNorms(const KrylovLayout& L, int K1) {
  cudaStream_t s = stream_;
  const double* U = kRec_.p + (size_t)recU_ * K1 * L.rowLd;
  for (int i = 0; i < recDim_; ++i) {  // ||u_i||^2 into kSmall_[i]
    const double* u = U + (size_t)i * L.rowLd;
    multiDot(u, L.rowLd, 1, u, L.dotRows, kPartial_.p, kSmall_.p + i, 0, s, &launches_);
  }
  comm_.allReduceSum(kSmall_.p, (size_t)recDim_, s);
  std::vector<double> g(recDim_);
  HY_CUDA(cudaMemcpyAsync(g.data(), kSmall_.p, recDim_ * sizeof(double), cudaMemcpyDeviceToHost, s));
  HY_CUDA(cudaStreamSynchronize(s));
  recD_.assign(recDim_, 0.0);
  for (int i = 0; i < recDim_; ++i) recD_[i] = 1.0 / std::sqrt(g[i]);
}

// C = A^ U after a Compute, then the thin QR C = Q R by two Cholesky-QR passes: C <- Q, U <- U R^-1.  Returns the
// number of recycled columns kept (0: C was numerically rank deficient and the space is dropped).
int Engine::rebuildRecycled(const KrylovLayout& L, int K1) {
  cudaStream_t s = stream_;
  const int kc = recDim_;
  const int64_t ldV = L.rowLd;
  double* Cb = kV_.p + (size_t)(K1 - kc) * ldV;
  for (int i = 0; i < kc; ++i) L.step(kRec_.p + ((size_t)recU_ * K1 + i) * ldV, Cb + (size_t)i * ldV);
  for (int pass = 0; pass < 2; ++pass) {
    std::vector<double> g = crossProducts(L, Cb, kc, Cb, kc);
    if (hy_cholesky(kc, g.data())) {
      recDim_ = 0;
      return 0;
    }
    std::vector<double> R((size_t)kc * kc);  // R = L'
    for (int j = 0; j < kc; ++j)
      for (int i = 0; i < kc; ++i) R[(size_t)j * kc + i] = g[(size_t)i * kc + j];
    const std::vector<double> Ri = upperInverse(R, kc);
    HY_CUDA(cudaMemcpyAsync(kSmall_.p, Ri.data(), Ri.size() * sizeof(double), cudaMemcpyHostToDevice, s));
    double* U = kRec_.p + (size_t)recU_ * K1 * ldV;
    double* scratch = kRec_.p + (size_t)(1 - recU_) * K1 * ldV;
    combine(Cb, ldV, kc, kSmall_.p, kc, scratch, ldV, kc, L.rows, 0, s, &launches_);
    HY_CUDA(cudaMemcpyAsync(Cb, scratch, (size_t)kc * ldV * sizeof(double), cudaMemcpyDeviceToDevice, s));
    combine(U, ldV, kc, kSmall_.p, kc, scratch, ldV, kc, L.rows, 0, s, &launches_);
    recU_ = 1 - recU_;
    HY_CUDA(cudaStreamSynchronize(s));  // Ri is pageable host memory
  }
  recEpoch_ = opEpoch_;
  recycleNorms(L, K1);
  return kc;
}

// x += [M^-1] U C' r (r: the residual the Krylov space is built on, b - A x or M^-1 (b - A x))
void Engine::recycleProject(const KrylovLayout& L, int K1, int kc, const double* r, bool right) {
  cudaStream_t s = stream_;
  const int64_t ldV = L.rowLd;
  const double* Cb = kV_.p + (size_t)(K1 - kc) * ldV;
  multiDot(Cb, ldV, kc, r + L.row0, L.dotRows, kPartial_.p, kH_.p, 0, s, &launches_);
  comm_.allReduceSum(kH_.p, (size_t)kc, s);
  HY_CUDA(cudaMemsetAsync(kZ_.p, 0, ldV * sizeof(double), s));  // r may live in kZ_: read above, in stream order
  multiAxpy(kRec_.p + (size_t)recU_ * K1 * ldV, ldV, kc, kH_.p, kZ_.p, L.rows, 1.0, s, &launches_);
  HY_CUDA(cudaStreamSynchronize(s));
  const double* upd = L.expand(kZ_.p);
  if (right) {
    L.M(upd, kW_.p);
    upd = kW_.p;
  }
  axpby(1.0, upd, 1.0, kX_.p, L.len, s, &launches_);
}

// start of a cycle with kc recycled columns: v0 = (I - C C') r / beta', g = [C' r; beta' e1], the first kc columns
// of the Hessenberg matrix D (no rotations).  false: beta' = 0, r lies in range(C).
bool Engine::cycleStart(const KrylovLayout& L, double* base, int kc, const double* r, double* g, double* H, double* cs,
                        double* sn, int m) {
  cudaStream_t s = stream_;
  const int64_t ldV = L.rowLd;
  double* Vb = base + (size_t)kc * ldV;
  double* dc = kH_.p;
  double* dN = kH_.p + 2 * m + 2;
  multiDot(base, ldV, kc, r + L.row0, L.dotRows, kPartial_.p, dc, 0, s, &launches_);
  comm_.allReduceSum(dc, (size_t)kc, s);
  axpby(1.0, r + L.row0, 0.0, Vb, L.rows, s, &launches_);
  multiAxpy(base, ldV, kc, dc, Vb, L.rows, -1.0, s, &launches_);
  multiDot(Vb, ldV, 1, Vb, L.dotRows, kPartial_.p, dN, 0, s, &launches_);
  comm_.allReduceSum(dN, 1, s);
  std::vector<double> h(2 * m + 3);
  HY_CUDA(cudaMemcpyAsync(h.data(), kH_.p, (2 * m + 3) * sizeof(double), cudaMemcpyDeviceToHost, s));
  HY_CUDA(cudaStreamSynchronize(s));
  const double bp = std::sqrt(h[2 * m + 2]);
  for (int i = 0; i < kc; ++i) {
    g[i] = h[i];
    for (int j = 0; j < kc; ++j) H[(size_t)i * m + j] = i == j ? recD_[i] : 0.0;
    cs[i] = 1.0;
    sn[i] = 0.0;
  }
  g[kc] = bp;
  if (!(bp > 0.0)) return false;
  scaleByInvNorm(Vb, dN, Vb, L.rows, s, &launches_);
  return true;
}

// end of a cycle of kDone columns (kc recycled + the Arnoldi steps): the harmonic Ritz vectors of
// Ghat' Ghat z = theta Ghat' (What' Vhat) z for the recK smallest |theta| give Ytilde = Vhat P, Ghat P = Q R,
// C = What Q, U = Ytilde R^-1.  What = [C | v_0 .. v_p] (base, kDone + 1 vectors), Vhat = [Utilde | v_0 .. v_(p-1)].
// Returns the new number of recycled columns; 0 when the Cholesky factorisation fails or Ghat P is rank deficient:
// then no space is kept, and the next cycle is a plain GMRES cycle.
int Engine::recycleUpdate(const KrylovLayout& L, int K1, int recK, double* base, int kc, int kDone,
                          const std::vector<double>& G, int m) {
  cudaStream_t s = stream_;
  const int64_t ldV = L.rowLd;
  const int mt = kDone, R1 = kDone + 1, pD = kDone - kc;
  std::vector<double> Gh((size_t)R1 * mt, 0.0), WV((size_t)R1 * mt, 0.0);
  for (int j = 0; j < kc; ++j) Gh[(size_t)j * R1 + j] = recD_[j];
  for (int j = kc; j < mt; ++j) {
    for (int i = 0; i <= j + 1; ++i) Gh[(size_t)j * R1 + i] = G[(size_t)i * m + j];
    WV[(size_t)j * R1 + j] = 1.0;
  }
  if (kc) {  // What' Utilde: [C' U; V' U] D
    const std::vector<double> wu = crossProducts(L, base, R1, kRec_.p + (size_t)recU_ * K1 * ldV, kc);
    for (int j = 0; j < kc; ++j)
      for (int i = 0; i < R1; ++i) WV[(size_t)j * R1 + i] = wu[(size_t)j * R1 + i] * recD_[j];
  }
  std::vector<double> A((size_t)mt * mt), B((size_t)mt * mt);
  for (int j = 0; j < mt; ++j)
    for (int i = 0; i < mt; ++i) {
      double a = 0.0, b = 0.0;
      for (int l = 0; l < R1; ++l) {
        a += Gh[(size_t)i * R1 + l] * Gh[(size_t)j * R1 + l];
        b += Gh[(size_t)i * R1 + l] * WV[(size_t)j * R1 + l];
      }
      A[(size_t)j * mt + i] = a;
      B[(size_t)j * mt + i] = b;
    }
  const int kMax = std::min(K1, m - 1);  // at least one Arnoldi step per cycle
  std::vector<double> P((size_t)mt * kMax);
  int kn = 0;
  auto drop = [&]() {
    recDim_ = 0;
    return 0;
  };
  if (hy_harmonic_ritz(mt, A.data(), B.data(), recK, kMax, P.data(), &kn) || kn == 0) return drop();
  std::vector<double> GP((size_t)R1 * kn, 0.0), Q((size_t)R1 * kn), R((size_t)kn * kn);
  for (int c = 0; c < kn; ++c)
    for (int l = 0; l < mt; ++l) {
      const double p = P[(size_t)c * mt + l];
      if (p != 0.0)
        for (int i = 0; i < R1; ++i) GP[(size_t)c * R1 + i] += Gh[(size_t)l * R1 + i] * p;
    }
  if (hy_qr(R1, kn, GP.data(), Q.data(), R.data(), 1e-12)) return drop();
  const std::vector<double> Ri = upperInverse(R, kn);
  // coefficients: [D P_u R^-1 (kc x kn) | P_v R^-1 (pD x kn) | Q (R1 x kn)], each column major
  std::vector<double> coef((size_t)(mt + R1) * kn, 0.0);
  double* cu = coef.data();
  double* cv = cu + (size_t)kc * kn;
  double* cq = cv + (size_t)pD * kn;
  for (int c = 0; c < kn; ++c)
    for (int l = 0; l < mt; ++l) {
      double t = 0.0;
      for (int q = 0; q <= c; ++q) t += P[(size_t)q * mt + l] * Ri[(size_t)c * kn + q];
      if (l < kc) cu[(size_t)c * kc + l] = recD_[l] * t;
      else cv[(size_t)c * pD + (l - kc)] = t;
    }
  std::copy(Q.begin(), Q.end(), cq);
  HY_CUDA(cudaMemcpyAsync(kSmall_.p, coef.data(), coef.size() * sizeof(double), cudaMemcpyHostToDevice, s));
  double* U = kRec_.p + (size_t)recU_ * K1 * ldV;
  double* Un = kRec_.p + (size_t)(1 - recU_) * K1 * ldV;
  const double* dcu = kSmall_.p;
  const double* dcv = dcu + (size_t)kc * kn;
  const double* dcq = dcv + (size_t)pD * kn;
  if (kc) combine(U, ldV, kc, dcu, kc, Un, ldV, kn, L.rows, 0, s, &launches_);
  combine(base + (size_t)kc * ldV, ldV, pD, dcv, pD, Un, ldV, kn, L.rows, kc ? 1 : 0, s, &launches_);
  combine(base, ldV, R1, dcq, R1, U, ldV, kn, L.rows, 0, s, &launches_);  // C into the old U block
  HY_CUDA(cudaMemcpyAsync(kV_.p + (size_t)(K1 - kn) * ldV, U, (size_t)kn * ldV * sizeof(double),
                          cudaMemcpyDeviceToDevice, s));
  HY_CUDA(cudaStreamSynchronize(s));  // coef is pageable host memory
  recU_ = 1 - recU_;
  recDim_ = kn;
  recEpoch_ = opEpoch_;
  recycleNorms(L, K1);
  return kn;
}

void Engine::solve(const double* b, const double* T, double* x, double* S, VecEnds ends, int where, uint64_t seed,
                   hymls_b200_solve_info* info, double* hist, int histCap) {
  needDevice();
  needComm();
  if (!computed_) throw Error(HYMLS_B200_ERR_STATE, "The preconditioner has not yet been computed.");
  if (ends != VecEnds::Replicated) {
    const char* what = ends == VecEnds::Owned ? "solve_dist" : "solve_map";
    if (!b || !x) throw Error(HYMLS_B200_ERR_ARG, std::string(what) + ": b_local and x_local are required");
    if (ends == VecEnds::RowMap && !rowMap_.ready)
      throw Error(HYMLS_B200_ERR_STATE, "solve_map: call hymls_b200_set_row_map first");
    if (comm_.size() > 1 && !levels_[0]->dist.ready)
      throw Error(HYMLS_B200_ERR_STATE, std::string(what) + ": no distributed plan (Number of Levels = 0?)");
  }
  ParameterList& sol = params_.sublist("Solver");
  ParameterList& it = sol.sublist("Iterative Solver");
  if (sol.get("Use Deflation", false))
    throw Error(HYMLS_B200_ERR_UNSUPPORTED, "deflated solvers are not implemented");
  const std::string method = sol.get("Krylov Method", "GMRES");
  const std::string side = sol.get("Left or Right Preconditioning", "Right");
  const std::string startVec = sol.get("Initial Vector", "Random");
  const int maxIters = it.get("Maximum Iterations", 1000);
  const double tol = it.get("Convergence Tolerance", 1e-8);
  const int numBlocks = it.get("Num Blocks", 300);
  const int maxRestarts = it.get("Maximum Restarts", 20);
  const bool explicitTest = it.get("Explicit Residual Test", false);
  const std::string impScaling = it.get("Implicit Residual Scaling", "Norm of Preconditioned Initial Residual");
  const std::string expScaling = it.get("Explicit Residual Scaling", "Norm of Initial Residual");
  if (method != "GMRES" && method != "CG" && method != "GCRODR")
    throw Error(HYMLS_B200_ERR_ARG, "Krylov Method '" + method + "' not supported (GMRES, CG, GCRODR)");
  const bool gcrodr = method == "GCRODR";
  const bool gmres = method == "GMRES" || gcrodr;  // GCRO-DR runs the GMRES cycle with the recycled space in front
  const bool single = gmres && singleBasis_;  // FP32 basis slots 1..m (readParameters refuses Single with CG)
  if (borderM_ && !gmres) throw Error(HYMLS_B200_ERR_UNSUPPORTED, "bordered solves use GMRES");
  const int m = std::max(1, std::min(numBlocks, maxIters));
  // GCRO-DR: k recycled columns (k + 1 when a complex pair straddles k); only a GCRODR solve reads (and writes back)
  // the parameter
  const int recK = gcrodr ? it.get("Num Recycled Blocks", 5) : 0;
  if (gcrodr && (recK < 1 || recK >= m))
    throw Error(HYMLS_B200_ERR_ARG, "Num Recycled Blocks must be at least 1 and less than min(Num Blocks, Maximum "
                                    "Iterations) = " + std::to_string(m));
  const int K1 = gcrodr ? recK + 1 : 0;  // slots of C in front of the Arnoldi vectors
  const bool left = side == "Left", right = side == "Right";
  const KrylovLayout L = useDist() ? ownerLayout(left, right, ends) : replicatedLayout(left, right, ends);
  const int64_t n = L.len;
  cudaStream_t s = stream_;

  kX_.alloc(L.ld);
  kB_.alloc(L.ld);
  kR_.alloc(L.ld);
  kW_.alloc(L.ld);
  kZ_.alloc(L.ld);
  kH_.alloc(2 * m + 8);
  kPartial_.alloc((size_t)(m + 2) * multiDotBlocks());
  // the Krylov basis is workspace like the vectors above (grow-only, reused by later solves): a 40 GB cudaMalloc
  // does not belong into the event-timed iteration.  Each basis precision releases the storage of the other, so
  // switching a handle's mode frees that memory.
  if (!gcrodr) {  // the recycled space of an earlier GCRODR list is gone (SetParameters dropped it): free its storage
    kRec_.release();
    kSmall_.release();
    kPartialB_.release();
    recDim_ = 0;
  }
  if (single) {
    if (kV_.cap > (size_t)L.rowLd) kV_.release();
    kV_.alloc(L.rowLd);
    kVf_.alloc((size_t)m * L.rowLd);
    kGs_.alloc(2 * (size_t)L.rowLd);
  } else if (gmres) {
    kVf_.release();
    kGs_.release();
    const size_t need = (size_t)(K1 + m + 1) * L.rowLd;
    if (gcrodr) {  // a recycled space survives only on the same rows
      if (recDim_ && (recRows_ != L.rows || recLd_ != L.rowLd || recRow0_ != L.row0 || recBorder_ != borderM_ ||
                      recM_ != m || recCap_ != K1 || kV_.cap < need || kRec_.cap < 2 * (size_t)K1 * L.rowLd))
        recDim_ = 0;
      kRec_.alloc(2 * (size_t)K1 * L.rowLd);
      kSmall_.alloc(3 * (size_t)(m + 2) * K1);
      kPartialB_.alloc(blockDotPartial());
      recRows_ = L.rows;
      recLd_ = L.rowLd;
      recRow0_ = L.row0;
      recBorder_ = borderM_;
      recM_ = m;
      recCap_ = K1;
      if (!recDim_) HY_CUDA(cudaMemsetAsync(kRec_.p, 0, kRec_.bytes(), stream_));
    }
    kV_.alloc(need);
  } else {
    kQ_.alloc(L.ld);
  }
  const auto kind = where == HYMLS_B200_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
  L.load(b, T, kB_.p, kind);
  if (startVec == "Random") {
    // MatrixUtils::Random (src/HYMLS_MatrixUtils.cpp:961-1007): uniform in (-1,1); the reference's
    // Epetra_Util LCG stream is replaced by a documented 64-bit Mersenne Twister with `seed`.
    std::vector<double> h(n_ + borderM_);
    std::mt19937_64 rng(seed);
    for (auto& v : h) v = (double)(rng() >> 11) * (1.0 / 9007199254740992.0) * 2.0 - 1.0;
    L.keepOwn(h);
    HY_CUDA(cudaMemcpyAsync(kX_.p, h.data(), n * sizeof(double), cudaMemcpyHostToDevice, s));
    HY_CUDA(cudaStreamSynchronize(s));
  } else if (startVec == "Zero") {
    HY_CUDA(cudaMemsetAsync(kX_.p, 0, L.ld * sizeof(double), s));
  } else {
    L.load(x, nullptr, kX_.p, kind);
  }
  // the ranks start the timed region together (a late rank would otherwise bill its delay to the others' first
  // collective)
  comm_.allReduceSum(kH_.p, 1, s);
  HY_CUDA(cudaStreamSynchronize(s));
  HY_CUDA(cudaEventRecord(ev0_, s));
  auto dot = [&](const double* u, const double* v) {
    double* d = kH_.p + 2 * m + 4;
    L.dot(u, v, d);
    double h;
    HY_CUDA(cudaMemcpyAsync(&h, d, sizeof(double), cudaMemcpyDeviceToHost, s));
    HY_CUDA(cudaStreamSynchronize(s));
    return h;
  };
  auto residual = [&]() {  // r = b - A x ; returns ||r||
    L.A(kX_.p, kR_.p);
    axpby(1.0, kB_.p, -1.0, kR_.p, n, s, &launches_);
    return std::sqrt(dot(kR_.p, kR_.p));
  };
  std::vector<double> history;
  int iters = 0;
  bool converged = false;
  double lastRel = 0;
  const double bnorm = std::sqrt(dot(kB_.p, kB_.p));

  if (!gmres) {
    // r = b - A x ; z = M r ; p = z
    double* p = kW_.p;
    double* q = kQ_.p;  // A p
    const double r0 = residual();
    history.push_back(1.0);
    if (r0 == 0) {
      converged = true;
    } else {
      L.M(kR_.p, kZ_.p);
      axpby(1.0, kZ_.p, 0.0, p, n, s, &launches_);
      double rz = dot(kR_.p, kZ_.p);
      while (iters < maxIters) {
        L.A(p, q);
        const double alpha = rz / dot(p, q);
        axpby(alpha, p, 1.0, kX_.p, n, s, &launches_);
        axpby(-alpha, q, 1.0, kR_.p, n, s, &launches_);
        ++iters;
        lastRel = std::sqrt(dot(kR_.p, kR_.p)) / r0;
        history.push_back(lastRel);
        if (lastRel <= tol) {
          converged = true;
          break;
        }
        L.M(kR_.p, kZ_.p);
        const double rzNew = dot(kR_.p, kZ_.p);
        axpby(1.0, kZ_.p, rzNew / rz, p, n, s, &launches_);
        rz = rzNew;
      }
    }
  } else {
    const int64_t ldV = L.rowLd, nloc = L.rows, nDot = L.dotRows;
    // GCRO-DR keeps C in the K1 slots in front of the Arnoldi vectors Vb; GMRES has K1 = 0
    double* Vb = kV_.p + (size_t)K1 * ldV;
    if (gcrodr && recDim_) HY_CUDA(cudaMemsetAsync(Vb, 0, (size_t)(m + 1) * ldV * sizeof(double), s));
    else HY_CUDA(cudaMemsetAsync(kV_.p, 0, kV_.bytes(), s));
    if (single) {
      HY_CUDA(cudaMemsetAsync(kVf_.p, 0, kVf_.bytes(), s));
      HY_CUDA(cudaMemsetAsync(kGs_.p, 0, kGs_.bytes(), s));
    }
    // Single: v0 stays FP64 in kV_ (rounding it would leave beta 2^-24 of r0 that no cycle can remove); slot j of
    // 1..m is FP32 at Vf + (j-1) ldV.  The Arnoldi step reads v0 or the widened slot vin, bitwise the vector that the
    // update of x uses; w is an FP64 work vector, orthogonalised in FP64 against v0 and the widened slots.
    const double* v0 = kV_.p;
    float* Vf = kVf_.p;
    double* wS = single ? kGs_.p : nullptr;
    double* vin = single ? kGs_.p + ldV : nullptr;
    std::vector<double> H((size_t)(m + 1) * m, 0.0), cs(m), sn(m), g(m + 1), hbuf(2 * m + 8);
    double* dH1 = kH_.p;              // first Gram-Schmidt pass  (m+1)
    double* dH2 = kH_.p + (m + 1);    // second pass              (m+1)
    double* dNrm = kH_.p + 2 * m + 2; // ||w||^2
    // GCRO-DR after a Compute: C = A^ U again (k operator applications, not iterations)
    if (gcrodr && recDim_ && recEpoch_ != opEpoch_) rebuildRecycled(L, K1);
    const double r0norm = residual();
    double* r = kR_.p;
    if (left) {
      L.M(kR_.p, kZ_.p);
      r = kZ_.p;
    }
    const double pr0norm = left ? std::sqrt(dot(r, r)) : r0norm;
    auto scaleOf = [&](const std::string& k) {
      double v = 1.0;
      if (k == "Norm of RHS") v = bnorm;
      else if (k == "Norm of Initial Residual") v = r0norm;
      else if (k == "Norm of Preconditioned Initial Residual") v = pr0norm;
      else if (k == "None") v = 1.0;
      else throw Error(HYMLS_B200_ERR_ARG, "unknown residual scaling '" + k + "'");
      return v == 0.0 ? 1.0 : v;
    };
    const double impScale = scaleOf(impScaling), expScale = scaleOf(expScaling);
    double beta = pr0norm;
    double trueRes = r0norm;
    // GCRO-DR state of this solve: kc recycled columns in use, C at Cb (the kc slots before Vb), U at Ub
    int kc = 0;
    std::vector<double> G;  // Ghat before the Givens rotations ((m+1) x m, row stride m)
    if (gcrodr) {
      G.assign((size_t)(m + 1) * m, 0.0);
      kc = recDim_;
      if (kc) {  // x += [M^-1] U C' r, then the residual of the new x (history[0] stays that of the initial guess)
        history.push_back(beta / impScale);
        recycleProject(L, K1, kc, r, right);
        trueRes = residual();
        r = kR_.p;
        beta = trueRes;
        if (left) {
          L.M(kR_.p, kZ_.p);
          r = kZ_.p;
          beta = std::sqrt(dot(r, r));
        }
      }
    }
    // HYMLS_B200_VERBOSE_SOLVE: wall time of the phases of every 50th Arnoldi step on stderr (synchronises the stream)
    static const bool verboseSolve = getenv("HYMLS_B200_VERBOSE_SOLVE") != nullptr;
    for (int restart = 0; restart <= maxRestarts; ++restart) {
      if (restart == 0 && history.empty()) history.push_back(beta / impScale);
      lastRel = beta / impScale;
      if (beta == 0.0 || (lastRel <= tol && !explicitTest)) {  // a zero residual cannot be normalised
        converged = true;
        break;
      }
      std::fill(g.begin(), g.end(), 0.0);
      // basis of the cycle: [C | v_0 v_1 ...] from `base`; column k >= kc of the Hessenberg matrix belongs to v_(k-kc)
      double* base = Vb - (size_t)kc * ldV;
      bool empty = false;
      if (kc) {  // v0 = (I - C C') r / beta', g = [C' r; beta' e1]; the first kc columns of Ghat are D (triangular)
        empty = !cycleStart(L, base, kc, r, g.data(), H.data(), cs.data(), sn.data(), m);
        if (empty) recycleProject(L, K1, kc, r, right);  // r lies in range(C): the projection solves
      } else {
        axpby(1.0 / beta, r + L.row0, 0.0, Vb, nloc, s, &launches_);  // v0 = r / beta (this rank's rows)
        g[0] = beta;
      }
      int kDone = kc;
      for (int k = kc; k < m && iters < maxIters && !empty; ++k) {
        const double* vk = !single ? base + (size_t)k * ldV : k == 0 ? v0 : vin;
        double* w = single ? wS : base + (size_t)(k + 1) * ldV;
        const bool lapIt = verboseSolve && comm_.rank() == 0 && (k % 50) == 20;
        auto tl = std::chrono::steady_clock::now();
        auto lap = [&](const char* what) {
          if (!lapIt) return;
          cudaStreamSynchronize(s);
          auto t1 = std::chrono::steady_clock::now();
          fprintf(stderr, "[hymls_b200 solve] it %d %-28s %8.3f ms\n", k, what,
                  std::chrono::duration<double, std::milli>(t1 - tl).count());
          tl = t1;
        };
        if (lapIt) {
          cudaStreamSynchronize(s);
          tl = std::chrono::steady_clock::now();
        }
        L.step(vk, w);
        lap("operator step");
        // two passes of classical Gram-Schmidt (Belos ICGS/DGKS), fused multi-dot + multi-axpy
        for (double* dh : {dH1, dH2}) {
          if (single) {  // h[0] against v0, h[1..k] against the FP32 slots 1..k
            multiDot(v0, ldV, 1, w, nDot, kPartial_.p, dh, 0, s, &launches_);
            multiDot(Vf, ldV, k, w, nDot, kPartial_.p, dh + 1, 0, s, &launches_);
          } else {
            multiDot(base, ldV, k + 1, w, nDot, kPartial_.p, dh, 0, s, &launches_);
          }
          comm_.allReduceSum(dh, (size_t)(k + 1), s);
          if (single) {
            multiAxpy(v0, ldV, 1, dh, w, nloc, -1.0, s, &launches_);
            multiAxpy(Vf, ldV, k, dh + 1, w, nloc, -1.0, s, &launches_);
          } else {
            multiAxpy(base, ldV, k + 1, dh, w, nloc, -1.0, s, &launches_);
          }
        }
        multiDot(w, ldV, 1, w, nDot, kPartial_.p, dNrm, 0, s, &launches_);
        comm_.allReduceSum(dNrm, 1, s);
        if (single) scaleByInvNormNarrow(w, dNrm, Vf + (size_t)k * ldV, vin, nloc, s, &launches_);
        else scaleByInvNorm(w, dNrm, w, nloc, s, &launches_);
        lap("CGS2 (4 sweeps, 3 allreduces)");
        HY_CUDA(cudaMemcpyAsync(hbuf.data(), kH_.p, (2 * m + 3) * sizeof(double), cudaMemcpyDeviceToHost, s));
        HY_CUDA(cudaStreamSynchronize(s));
        lap("Hessenberg column to host");
        for (int i = 0; i <= k; ++i) H[(size_t)i * m + k] = hbuf[i] + hbuf[m + 1 + i];
        const double hn = std::sqrt(hbuf[2 * m + 2]);
        // happy breakdown: w is (numerically) in the span of the basis.  scaleByInvNorm has produced Inf/NaN in
        // v_{k+1}, which is never used: the cycle ends after this column (Belos stops likewise)
        double colNorm = 0.0;
        for (int i = 0; i <= k; ++i) colNorm = std::hypot(colNorm, hbuf[i] + hbuf[m + 1 + i]);
        const bool breakdown = !(hn > 1e-300) || hn <= 1e-15 * colNorm;
        H[(size_t)(k + 1) * m + k] = breakdown ? 0.0 : hn;
        if (gcrodr) {  // the unrotated column for the harmonic Ritz problem; a breakdown leaves no finite v_(k+1)
          for (int i = 0; i <= k + 1; ++i) G[(size_t)i * m + k] = H[(size_t)i * m + k];
          if (breakdown) HY_CUDA(cudaMemsetAsync(w, 0, ldV * sizeof(double), s));
        }
        for (int i = kc; i < k; ++i) {
          const double t = cs[i] * H[(size_t)i * m + k] + sn[i] * H[(size_t)(i + 1) * m + k];
          H[(size_t)(i + 1) * m + k] = -sn[i] * H[(size_t)i * m + k] + cs[i] * H[(size_t)(i + 1) * m + k];
          H[(size_t)i * m + k] = t;
        }
        const double d = std::hypot(H[(size_t)k * m + k], H[(size_t)(k + 1) * m + k]);
        cs[k] = H[(size_t)k * m + k] / d;
        sn[k] = H[(size_t)(k + 1) * m + k] / d;
        H[(size_t)k * m + k] = d;
        H[(size_t)(k + 1) * m + k] = 0.0;
        g[k + 1] = -sn[k] * g[k];
        g[k] = cs[k] * g[k];
        ++iters;
        kDone = k + 1;
        lastRel = std::fabs(g[k + 1]) / impScale;
        history.push_back(lastRel);
        if (lastRel <= tol || breakdown) break;
      }
      if (kDone > kc) {
        // y = triu(H)^-1 g ; x += [M^-1] V y
        std::vector<double> y(kDone);
        for (int i = kDone - 1; i >= 0; --i) {
          double t = g[i];
          for (int j = i + 1; j < kDone; ++j) t -= H[(size_t)i * m + j] * y[j];
          y[i] = t / H[(size_t)i * m + i];
        }
        HY_CUDA(cudaMemcpyAsync(dH1, y.data(), kDone * sizeof(double), cudaMemcpyHostToDevice, s));
        HY_CUDA(cudaMemsetAsync(kZ_.p, 0, ldV * sizeof(double), s));
        if (single) {
          multiAxpy(v0, ldV, 1, dH1, kZ_.p, nloc, 1.0, s, &launches_);
          multiAxpy(Vf, ldV, kDone - 1, dH1 + 1, kZ_.p, nloc, 1.0, s, &launches_);
        } else {
          multiAxpy(Vb, ldV, kDone - kc, dH1 + kc, kZ_.p, nloc, 1.0, s, &launches_);
          if (kc) {  // + Utilde y_u = U (D y_u)
            std::vector<double> yu(kc);
            for (int i = 0; i < kc; ++i) yu[i] = y[i] * recD_[i];
            HY_CUDA(cudaMemcpyAsync(dH2, yu.data(), kc * sizeof(double), cudaMemcpyHostToDevice, s));
            multiAxpy(kRec_.p + (size_t)recU_ * K1 * ldV, ldV, kc, dH2, kZ_.p, nloc, 1.0, s, &launches_);
          }
        }
        HY_CUDA(cudaStreamSynchronize(s));
        const double* upd = L.expand(kZ_.p);
        if (right) {
          L.M(upd, kW_.p);
          upd = kW_.p;
        }
        axpby(1.0, upd, 1.0, kX_.p, n, s, &launches_);
      }
      // GCRO-DR: the harmonic Ritz vectors of this cycle become the recycled space of the next cycle and solve
      if (gcrodr && kDone > kc && kDone > recK) kc = recycleUpdate(L, K1, recK, base, kc, kDone, G, m);
      trueRes = residual();
      r = kR_.p;
      beta = trueRes;
      if (left) {
        L.M(kR_.p, kZ_.p);
        r = kZ_.p;
        beta = std::sqrt(dot(r, r));
      }
      // Single: the recurrence residual does not include the rounding of the basis, so the cycle counts as converged
      // only when the residual recomputed in FP64 meets tol in the implicit criterion's own scaling as well
      const bool fp64Met = !single || (left ? beta : trueRes) / impScale <= tol;
      if (history.back() <= tol && fp64Met) {
        if (!explicitTest || trueRes / expScale <= tol) {
          converged = true;
          break;
        }
      }
      if (iters >= maxIters) break;
    }
  }
  HY_CUDA(cudaEventRecord(ev1_, s));
  HY_CUDA(cudaStreamSynchronize(s));
  float ms = 0;
  HY_CUDA(cudaEventElapsedTime(&ms, ev0_, ev1_));
  const double res = residual();  // explicit residual of [K V; W' C] [x; s] = [b; T]
  L.store(kX_.p, x, S, where == HYMLS_B200_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost);
  HY_CUDA(cudaStreamSynchronize(s));
  if (info) {
    info->iterations = iters;
    info->converged = converged ? 1 : 0;
    info->rel_residual = lastRel;
    info->explicit_rel_residual = bnorm > 0 ? res / bnorm : res;
    info->solve_seconds = ms * 1e-3;
    info->history_len = (int)history.size();
  }
  if (hist)
    for (int i = 0; i < (int)history.size() && i < histCap; ++i) hist[i] = history[i];
}

}  // namespace hymls

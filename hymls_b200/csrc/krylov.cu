// Krylov driver (BaseSolver::ApplyInverse -> Belos BlockGmresSolMgr / BlockCGSolMgr, block size 1).
//
// One GMRES(m) / CG serves both vector layouts of the library; KrylovLayout carries the operations in which they
// differ:
//   * replicated: every rank holds whole vectors of length n (+ border).  One GPU, and several ranks without the
//     owner path (HYMLS_B200_DIST=0, Number of Levels = 0).
//   * owner: a rank holds the rows it owns (DistPlan, dist.cu), packed, followed by the border entries, which every
//     rank keeps (bitwise equal); useDist() selects it.
#include <algorithm>
#include <chrono>
#include <cmath>
#include <functional>
#include <random>

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
  std::function<void(const double* src, double* dst, cudaMemcpyKind kind)> load;   // b or x0 of the caller
  std::function<void(std::vector<double>& full)> keepOwn;  // a host vector of length n (+ border) -> this rank's part
  std::function<void(const double* src, double* dst, cudaMemcpyKind kind)> store;  // x to the caller (replicated)
};

// Replicated vectors; the GMRES basis is row-sharded over the ranks: rank r keeps rows [r*chunk, (r+1)*chunk) of every
// basis vector, so its Gram-Schmidt dots are local partial sums + one all-reduce of (k+1) doubles (the reference's
// SumAll).  The preconditioner wants its argument replicated, so v_k is all-gathered before each ApplyInverse.
KrylovLayout Engine::replicatedLayout(bool left, bool right) {
  // With a border set the bordered system [K V; W' C] [x; s] = [b; 0] is solved on vectors of length n + m
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
  L.load = [=](const double* src, double* dst, cudaMemcpyKind kind) {
    HY_CUDA(cudaMemcpyAsync(dst, src, nK * sizeof(double), kind, s));
    if (bm) HY_CUDA(cudaMemsetAsync(dst + nK, 0, bm * sizeof(double), s));
  };
  L.keepOwn = [](std::vector<double>&) {};
  L.store = [=](const double* src, double* dst, cudaMemcpyKind kind) {
    HY_CUDA(cudaMemcpyAsync(dst, src, nK * sizeof(double), kind, s));
  };
  return L;
}

// Packed owned rows, then the m border entries (bordered system [K V; W' C], replicated: only rank 0 counts them in
// the inner products); the basis lives in the same rows, so the loop contains no full-vector collective.  The
// operator and the preconditioner work on global-length vectors with the owned entries valid: kS1_ (argument) and
// kS2_ (result); the border adds one all-reduce of m doubles to the operator.
KrylovLayout Engine::ownerLayout(bool left, bool right) {
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
  L.load = [=](const double* src, double* dst, cudaMemcpyKind kind) {
    HY_CUDA(cudaMemcpyAsync(gOut, src, n * sizeof(double), kind, s));
    packIdx(gOut, D->ownRows.p, dst, nOwn, s, &launches_);
    if (bm) HY_CUDA(cudaMemsetAsync(dst + nOwn, 0, bm * sizeof(double), s));
  };
  L.keepOwn = [=](std::vector<double>& full) {  // n + m host numbers -> owned rows + border entries
    std::vector<double> own(nOwn + bm);
    for (int64_t i = 0; i < nOwn; ++i) own[i] = full[D->hOwnRows[i]];
    for (int j = 0; j < bm; ++j) own[nOwn + j] = full[n + j];
    full.swap(own);
  };
  L.store = [=](const double* src, double* dst, cudaMemcpyKind kind) {  // replicated, like the single-GPU entry point
    toGlobal(src, gIn);
    gatherOwned(gIn, gOut);
    HY_CUDA(cudaMemcpyAsync(dst, gOut, n * sizeof(double), kind, s));
  };
  return L;
}

void Engine::solve(const double* b, double* x, int where, uint64_t seed, hymls_b200_solve_info* info, double* hist,
                   int histCap) {
  needDevice();
  needComm();
  if (!computed_) throw Error(HYMLS_B200_ERR_STATE, "The preconditioner has not yet been computed.");
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
  if (method != "GMRES" && method != "CG")
    throw Error(HYMLS_B200_ERR_ARG, "Krylov Method '" + method + "' not supported (GMRES, CG)");
  const bool gmres = method == "GMRES";
  if (borderM_ && !gmres) throw Error(HYMLS_B200_ERR_UNSUPPORTED, "bordered solves use GMRES");
  const int m = std::max(1, std::min(numBlocks, maxIters));
  const bool left = side == "Left", right = side == "Right";
  const KrylovLayout L = useDist() ? ownerLayout(left, right) : replicatedLayout(left, right);
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
  // does not belong into the event-timed iteration
  if (gmres) kV_.alloc((size_t)(m + 1) * L.rowLd);
  else kQ_.alloc(L.ld);
  const auto kind = where == HYMLS_B200_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
  L.load(b, kB_.p, kind);
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
    L.load(x, kX_.p, kind);
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
    HY_CUDA(cudaMemsetAsync(kV_.p, 0, (size_t)(m + 1) * ldV * sizeof(double), s));
    std::vector<double> H((size_t)(m + 1) * m, 0.0), cs(m), sn(m), g(m + 1), hbuf(2 * m + 8);
    double* dH1 = kH_.p;              // first Gram-Schmidt pass  (m+1)
    double* dH2 = kH_.p + (m + 1);    // second pass              (m+1)
    double* dNrm = kH_.p + 2 * m + 2; // ||w||^2
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
    // HYMLS_B200_VERBOSE_SOLVE: wall time of the phases of every 50th Arnoldi step on stderr (synchronises the stream)
    static const bool verboseSolve = getenv("HYMLS_B200_VERBOSE_SOLVE") != nullptr;
    for (int restart = 0; restart <= maxRestarts; ++restart) {
      if (restart == 0) history.push_back(beta / impScale);
      lastRel = beta / impScale;
      if (beta == 0.0 || (lastRel <= tol && !explicitTest)) {  // a zero residual cannot be normalised
        converged = true;
        break;
      }
      axpby(1.0 / beta, r + L.row0, 0.0, kV_.p, nloc, s, &launches_);  // v0 = r / beta (this rank's rows)
      std::fill(g.begin(), g.end(), 0.0);
      g[0] = beta;
      int kDone = 0;
      for (int k = 0; k < m && iters < maxIters; ++k) {
        double* vk = kV_.p + (size_t)k * ldV;
        double* w = kV_.p + (size_t)(k + 1) * ldV;
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
        multiDot(kV_.p, ldV, k + 1, w, nDot, kPartial_.p, dH1, 0, s, &launches_);
        comm_.allReduceSum(dH1, (size_t)(k + 1), s);
        multiAxpy(kV_.p, ldV, k + 1, dH1, w, nloc, -1.0, s, &launches_);
        multiDot(kV_.p, ldV, k + 1, w, nDot, kPartial_.p, dH2, 0, s, &launches_);
        comm_.allReduceSum(dH2, (size_t)(k + 1), s);
        multiAxpy(kV_.p, ldV, k + 1, dH2, w, nloc, -1.0, s, &launches_);
        multiDot(w, ldV, 1, w, nDot, kPartial_.p, dNrm, 0, s, &launches_);
        comm_.allReduceSum(dNrm, 1, s);
        scaleByInvNorm(w, dNrm, w, nloc, s, &launches_);
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
        for (int i = 0; i < k; ++i) {
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
      if (kDone > 0) {
        // y = triu(H)^-1 g ; x += [M^-1] V y
        std::vector<double> y(kDone);
        for (int i = kDone - 1; i >= 0; --i) {
          double t = g[i];
          for (int j = i + 1; j < kDone; ++j) t -= H[(size_t)i * m + j] * y[j];
          y[i] = t / H[(size_t)i * m + i];
        }
        HY_CUDA(cudaMemcpyAsync(dH1, y.data(), kDone * sizeof(double), cudaMemcpyHostToDevice, s));
        HY_CUDA(cudaMemsetAsync(kZ_.p, 0, ldV * sizeof(double), s));
        multiAxpy(kV_.p, ldV, kDone, dH1, kZ_.p, nloc, 1.0, s, &launches_);
        HY_CUDA(cudaStreamSynchronize(s));
        const double* upd = L.expand(kZ_.p);
        if (right) {
          L.M(upd, kW_.p);
          upd = kW_.p;
        }
        axpby(1.0, upd, 1.0, kX_.p, n, s, &launches_);
      }
      trueRes = residual();
      r = kR_.p;
      beta = trueRes;
      if (left) {
        L.M(kR_.p, kZ_.p);
        r = kZ_.p;
        beta = std::sqrt(dot(r, r));
      }
      if (history.back() <= tol) {
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
  const double res = residual();  // explicit residual
  L.store(kX_.p, x, where == HYMLS_B200_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost);
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

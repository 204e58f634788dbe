// Owner-computes multi-GPU path of level 0 (one process per GPU, NCCL over NVLink / NVSwitch).
//
// The reference distributes subdomains over MPI ranks (BasePartitioner::CreatePIDMap) and moves only what
// Epetra's Import/Export move: the off-rank columns of A21 x1 / A12 x2 (MatrixBlock::Apply,
// src/HYMLS_MatrixBlock.cpp:294-308), the V-sums to the next level (src/HYMLS_SchurPreconditioner.cpp:1076-1078)
// and the Krylov dot products (SumAll).  Here:
//   * a rank owns the interiors of its subdomains and the separator groups whose owner subdomain is its own
//     (HierarchicalMap: the first subdomain listing a group owns it, src/HYMLS_HierarchicalMap.cpp:261-271);
//   * rhs2 = b2 - A21 x1: every rank multiplies with the columns of its interiors; partial sums at separators
//     owned by a neighbour go to the owner with one grouped ncclSend/ncclRecv ("rev" halo) and are added there
//     in rank order (deterministic);
//   * Householder transform and separator-block solves run on the owned groups only; the V-sums (a vector of
//     nuniq doubles, 0.76 MB at 128^3) are summed to every rank for the next level, which stays replicated in /
//     replicated out because its vectors are 100x smaller;
//   * x2 of the owned separators goes to the ranks whose subdomains touch them ("fwd" halo) for A12 x2;
//   * the result is distributed by row owner.  The Krylov basis lives in this distribution, the operator apply
//     exchanges the matrix halo ("mat"), so the GMRES loop contains no full-vector collective at all.
// Vectors keep GLOBAL length and indexing (only owned + halo entries are touched), so every index array of the
// single-GPU path stays valid; kernels get row / group lists.
#include <algorithm>
#include <chrono>

#include "engine.hpp"
#include "hostpar.hpp"

namespace hymls {

bool Engine::useDist() const {
  static const bool off = getenv("HYMLS_B200_DIST") && atoi(getenv("HYMLS_B200_DIST")) == 0;
  return !off && comm_.active() && comm_.size() > 1 && !levels_.empty() && levels_[0]->sharded && !levels_[0]->exact;
}

static void uploadHalo(Halo& h, const std::vector<std::vector<int>>& send, const std::vector<std::vector<int>>& recv,
                       cudaStream_t s, bool device = true) {
  const int P = (int)send.size();
  h.peers.clear();
  h.sendPtr.assign(1, 0);
  h.recvPtr.assign(1, 0);
  std::vector<int> si, ri;
  for (int q = 0; q < P; ++q) {
    if (send[q].empty() && recv[q].empty()) continue;
    h.peers.push_back(q);
    si.insert(si.end(), send[q].begin(), send[q].end());
    ri.insert(ri.end(), recv[q].begin(), recv[q].end());
    h.sendPtr.push_back((int64_t)si.size());
    h.recvPtr.push_back((int64_t)ri.size());
  }
  if (!device) return;
  h.sendIdx.upload(si, s);
  h.recvIdx.upload(ri, s);
  h.sendBuf.alloc(std::max<size_t>(si.size(), 1));
  h.recvBuf.alloc(std::max<size_t>(ri.size(), 1));
}

static void sortUnique(std::vector<int>& v) {
  std::sort(v.begin(), v.end());
  v.erase(std::unique(v.begin(), v.end()), v.end());
}

void Engine::buildDistPlan(Level& L) {
  const LevelSym& S = L.sym;
  DistPlan& D = L.dist;
  cudaStream_t s = stream_;
  const int P = comm_.size(), me = comm_.rank();
  // owner of every separator position
  std::vector<int> sepOwner(S.nS, 0), uniqRank(S.nuniq, 0);
  std::vector<int> ownUniq, ownSepPos;
  for (int u = 0; u < S.nuniq; ++u) {
    uniqRank[u] = L.sdRank[S.H.uniqOwnerSd[u]];
    for (int64_t p = S.H.uniqPtr[u]; p < S.H.uniqPtr[u + 1]; ++p) sepOwner[p] = uniqRank[u];
    if (uniqRank[u] == me) {
      ownUniq.push_back(u);
      for (int64_t p = S.H.uniqPtr[u]; p < S.H.uniqPtr[u + 1]; ++p) ownSepPos.push_back((int)p);
    }
  }
  // separators touched by the subdomains of every rank: mine give the row list of the A21 product and the ghosts,
  // the others tell which of my separators they will send partial sums for
  std::vector<std::vector<int>> sendRev(P), recvRev(P);
  std::vector<int> rows21;
  for (int sd = 0; sd < S.nsd; ++sd) {
    const int q = L.sdRank[sd];
    for (int64_t R = S.sdRowPtr[sd]; R < S.sdRowPtr[sd + 1]; ++R) {
      const int p = S.sdSep[R];
      if (q == me) {
        rows21.push_back(p);
        if (sepOwner[p] != me) sendRev[sepOwner[p]].push_back(p);
      } else if (sepOwner[p] == me) {
        recvRev[q].push_back(p);
      }
    }
  }
  sortUnique(rows21);
  for (int q = 0; q < P; ++q) {
    sortUnique(sendRev[q]);
    sortUnique(recvRev[q]);
  }
  const bool dev = deviceOk_;  // without a device only the host side of the plan exists (owned_rows, tests)
  uploadHalo(D.rev, sendRev, recvRev, s, dev);
  uploadHalo(D.fwd, recvRev, sendRev, s, dev);  // the same lists, opposite direction
  // deterministic accumulation of the received partial sums: per owned node its sources in rank order
  {
    std::vector<std::pair<int, int64_t>> ent;  // (node, index in rev.recvBuf)
    int64_t off = 0;
    for (int q = 0; q < P; ++q) {
      for (size_t i = 0; i < recvRev[q].size(); ++i) ent.emplace_back(recvRev[q][i], off + (int64_t)i);
      off += (int64_t)recvRev[q].size();
    }
    std::stable_sort(ent.begin(), ent.end(),
                     [](const std::pair<int, int64_t>& a, const std::pair<int, int64_t>& b) { return a.first < b.first; });
    std::vector<int> node;
    std::vector<int64_t> ptr(1, 0), src;
    for (size_t i = 0; i < ent.size(); ++i) {
      if (node.empty() || node.back() != ent[i].first) {
        if (!node.empty()) ptr.push_back((int64_t)src.size());
        node.push_back(ent[i].first);
      }
      src.push_back(ent[i].second);
    }
    if (!node.empty()) ptr.push_back((int64_t)src.size());
    D.nAdd = (int64_t)node.size();
    if (dev) {
      D.addNode.upload(node, s);
      D.addPtr.upload(ptr, s);
      D.addSrc.upload(src, s);
    }
  }
  std::vector<int> rows12;
  for (int sd : L.ownSd)
    for (int64_t p = S.H.intPtr[sd]; p < S.H.intPtr[sd + 1]; ++p) rows12.push_back((int)p);
  // row ownership in matrix numbering
  D.rowOwner.assign(S.n, 0);
  for (int sd = 0; sd < S.nsd; ++sd)
    for (int64_t p = S.H.intPtr[sd]; p < S.H.intPtr[sd + 1]; ++p) D.rowOwner[S.intRow[p]] = L.sdRank[sd];
  for (int64_t p = 0; p < S.nS; ++p) D.rowOwner[S.sepRow[p]] = sepOwner[p];
  std::vector<int64_t> cnt(P, 0);
  for (int64_t r = 0; r < S.n; ++r) cnt[D.rowOwner[r]]++;
  D.maxOwn = *std::max_element(cnt.begin(), cnt.end());
  D.nOwn = cnt[me];
  std::vector<int> allRows((size_t)P * D.maxOwn, -1);
  std::vector<int64_t> fill(P, 0);
  D.hOwnRows.clear();
  for (int64_t r = 0; r < S.n; ++r) {
    const int q = D.rowOwner[r];
    allRows[(size_t)q * D.maxOwn + fill[q]++] = (int)r;
    if (q == me) D.hOwnRows.push_back((int)r);
  }
  D.nRows21 = (int64_t)rows21.size();
  D.nRows12 = (int64_t)rows12.size();
  D.nOwnUniq = (int64_t)ownUniq.size();
  D.nOwnSep = (int64_t)ownSepPos.size();
  if (dev) {
    D.rows21.upload(rows21, s);
    D.rows12.upload(rows12, s);
    D.ownUniq.upload(ownUniq, s);
    D.ownSepPos.upload(ownSepPos, s);
    D.ownRows.upload(D.hOwnRows, s);
    D.allRows.upload(allRows, s);
    D.gath.alloc((size_t)P * D.maxOwn);
    HY_CUDA(cudaStreamSynchronize(s));
  }
  D.ready = true;
  D.matReady = false;
  buildMatrixHalo();
}

// columns of my rows owned elsewhere (receive) and my rows that appear as columns of other ranks' rows (send).
// Part of Initialize (threaded over the rows): a rank that built this inside the first solve would make the others
// wait in their first collective.
void Engine::buildMatrixHalo() {
  Level& L = *levels_[0];
  DistPlan& D = L.dist;
  if (D.matReady) return;
  const int P = comm_.size(), me = comm_.rank();
  const int T = 64;
  std::vector<std::vector<std::vector<int>>> sendT(T, std::vector<std::vector<int>>(P)),
      recvT(T, std::vector<std::vector<int>>(P));
  parallelFor(n_, [&](int64_t r0, int64_t r1, int t) {
    auto& snd = sendT[t & (T - 1)];
    auto& rcv = recvT[t & (T - 1)];
    for (int64_t r = r0; r < r1; ++r) {
      const int q = D.rowOwner[r];
      for (int64_t e = hRowptr_[r]; e < hRowptr_[r + 1]; ++e) {
        const int c = hColidx_[e];
        const int qc = D.rowOwner[c];
        if (q == qc) continue;
        if (q == me) rcv[qc].push_back(c);
        else if (qc == me) snd[q].push_back(c);
      }
    }
  });
  std::vector<std::vector<int>> send(P), recv(P);
  for (int t = 0; t < T; ++t)
    for (int q = 0; q < P; ++q) {
      send[q].insert(send[q].end(), sendT[t][q].begin(), sendT[t][q].end());
      recv[q].insert(recv[q].end(), recvT[t][q].begin(), recvT[t][q].end());
    }
  for (int q = 0; q < P; ++q) {
    sortUnique(send[q]);
    sortUnique(recv[q]);
  }
  uploadHalo(D.mat, send, recv, stream_, deviceOk_);
  if (deviceOk_) HY_CUDA(cudaStreamSynchronize(stream_));
  D.matReady = true;
}

// src[sendIdx] -> peers; received values land in dst[recvIdx] (scatter) or stay in h.recvBuf (for haloAdd)
void Engine::haloExchange(Halo& h, const double* src, double* dst, bool scatter) {
  cudaStream_t s = stream_;
  packIdx(src, h.sendIdx.p, h.sendBuf.p, h.sendPtr.back(), s, &launches_);
  comm_.neighbourExchange(h.peers, h.sendBuf.p, h.sendPtr, h.recvBuf.p, h.recvPtr, s);
  if (scatter) scatterVec(h.recvBuf.p, h.recvIdx.p, dst, h.recvPtr.back(), s, &launches_);
}

// Level-0 ApplyInverse on distributed vectors: B and X have global length; B is read and X written at the rows this
// rank owns (Preconditioner::ApplyInverse, src/HYMLS_Preconditioner.cpp:930-1070).  With a border, T (replicated,
// nullptr: 0) enters the border right-hand sides and S lands in bS_, bitwise equal on every rank.  The border terms
// read owned positions only: the other entries of B and Y are stale on this rank.
void Engine::applyLevel0Dist(const double* B, double* X, const double* T) {
  Level& L = *levels_[0];
  const LevelSym& S = L.sym;
  DistPlan& D = L.dist;
  cudaStream_t s = stream_;
  static const bool verboseApply = getenv("HYMLS_B200_VERBOSE_APPLY") != nullptr;
  const bool lap = verboseApply && comm_.rank() == 0 && (stats_.num_apply_inverse % 16) == 5;
  auto t0 = std::chrono::steady_clock::now();
  auto mark = [&](const char* what) {
    if (!lap) return;
    cudaStreamSynchronize(s);
    auto t1 = std::chrono::steady_clock::now();
    fprintf(stderr, "[hymls_b200 apply dist] %-36s %8.3f ms\n", what,
            std::chrono::duration<double, std::milli>(t1 - t0).count());
    t0 = t1;
  };
  if (lap) cudaStreamSynchronize(s);
  t0 = std::chrono::steady_clock::now();
  // x1 = leading rows of A11 \ b1 on the owned subdomains
  GemvArgs g = L.a11.args();
  g.xin = B;
  g.gather = L.intRow.p;
  g.out = L.x1.p;
  g.mode = 0;
  g.itemMat = L.a11.itemMatLead.p;
  g.itemRow0 = L.a11.itemRow0Lead.p;
  g.nrows = L.a11.rowLimit.p;
  const bool timeIt = timeA11_;
  if (timeIt) HY_CUDA(cudaEventRecord(evA_, s));
  batchedGemv(g, L.a11.numItemsLead, L.a11.npMax, s, &launches_);
  if (timeIt) {
    HY_CUDA(cudaEventRecord(evB_, s));
    HY_CUDA(cudaEventSynchronize(evB_));
    float ms = 0;
    HY_CUDA(cudaEventElapsedTime(&ms, evA_, evB_));
    a11LeadMs_ += ms;
  }
  const bool split = splitActive(L, 0);  // see Engine::applyLevel
  if (split) {
    HY_CUDA(cudaEventRecord(evFork_, s));
    HY_CUDA(cudaStreamWaitEvent(side_, evFork_, 0));
    GemvArgs t = g;
    t.itemMat = L.a11.itemMatTrail.p;
    t.itemRow0 = L.a11.itemRow0Trail.p;
    t.nrows = nullptr;
    batchedGemv(t, L.a11.numItemsTrail, L.a11.npMax, side_, &launches_);
    HY_CUDA(cudaEventRecord(evJoin_, side_));
  }
  mark("A11 gemv 1 (leading rows)");
  const int bm = borderM_;
  if (bm) {  // q = T - W1' b1 over the owned interiors (applyLevel)
    multiDot(L.W1t.p, S.nI, bm, B, D.nRows12, bPartial_.p, L.bQ.p, 0, s, &launches_, L.intRow.p, D.rows12.p);
    comm_.allReduceSum(L.bQ.p, (size_t)bm, s);
    axpby(T ? 1.0 : 0.0, T ? T : L.bQ.p, -1.0, L.bQ.p, bm, s, &launches_);
  }
  // Z = -A21[:, owned interiors] x1 at the separators my subdomains touch; ghost parts go to their owners
  spmvRows(L.p21.p, L.c21.p, L.v21.p, L.x1.p, L.Z.p, D.rows21.p, D.nRows21, 0.0, nullptr, nullptr, -1.0, 0, s,
           &launches_);
  haloExchange(D.rev, L.Z.p, nullptr, false);
  haloAdd(L.Z.p, D.addNode.p, D.addPtr.p, D.addSrc.p, D.rev.recvBuf.p, D.nAdd, s, &launches_);
  gatherAddList(B, L.sepRow.p, L.Z.p, L.rhsS.p, D.ownSepPos.p, D.nOwnSep, s, &launches_);
  mark("A21 spmv + halo (partial sums)");
  // Householder on the owned groups; V-sum right-hand side summed to every rank (zeros elsewhere: exact)
  HY_CUDA(cudaMemsetAsync(L.vsRhs.p, 0, (size_t)S.nuniq * sizeof(double), s));
  householderList(L.uniqStart.p, D.ownUniq.p, (int)D.nOwnUniq, L.what.p, L.rhsS.p, L.Z.p, L.vsRhs.p, nullptr, nullptr,
                  nullptr, s, &launches_);
  comm_.allReduceSum(L.vsRhs.p, (size_t)S.nuniq, s);
  blockSolves(L, L.Z.p, L.Y.p);
  if (bm) {  // Tc = q - sW' Y over the owned separators (sW is zero at the V-sums)
    multiDot(L.sW.p, S.nS, bm, L.Y.p, D.nOwnSep, bPartial_.p, L.bT.p, 0, s, &launches_, nullptr, D.ownSepPos.p);
    comm_.allReduceSum(L.bT.p, (size_t)bm, s);
    axpby(1.0, L.bQ.p, -1.0, L.bT.p, bm, s, &launches_);
  }
  mark("householder + blocks + vsum allreduce");
  if (levels_.size() > 1) {
    applyLevel(1, L.vsRhs.p, L.vsSol.p, bm ? L.bT.p : nullptr);
  } else {
    // the coarse solve is replicated: rank 0's result becomes the common one (see applyLevel)
    if (bm) coarseSolveBordered(L.vsRhs.p, L.bT.p, L.vsSol.p, S.nuniq);
    else coarseSolve(L.vsRhs.p, L.vsSol.p, S.nuniq);
    comm_.broadcast(L.vsSol.p, (size_t)S.nuniq, 0, s);
    if (bm) comm_.broadcast(bS_.p, (size_t)bm, 0, s);
  }
  mark("next level / coarse");
  householderList(L.uniqStart.p, D.ownUniq.p, (int)D.nOwnUniq, L.what.p, L.Y.p, L.Y.p, nullptr, L.vsSol.p, X,
                  L.sepRow.p, s, &launches_);
  haloExchange(D.fwd, L.Y.p, L.Y.p, true);
  mark("householder back + halo (x2)");
  spmvRows(L.p12.p, L.c12.p, L.v12.p, L.Y.p, L.y1.p, D.rows12.p, D.nRows12, 0.0, nullptr, nullptr, 1.0, 0, s,
           &launches_);
  g = L.a11.args();
  g.xin = B;
  g.gather = L.intRow.p;
  g.xsub = L.y1.p;
  g.out = X;
  g.scatter = L.intRow.p;
  g.mode = 0;
  if (split) {  // X[interior] = x1 - A11^-1[:, :nb] y1
    HY_CUDA(cudaStreamWaitEvent(s, evJoin_, 0));
    g.xin = L.y1.p;
    g.gather = nullptr;
    g.xsub = nullptr;
    g.xprev = L.x1.p;
    g.ncols = L.a11.rowLimit.p;
    g.mode = 1;
  }
  if (timeIt) HY_CUDA(cudaEventRecord(evA_, s));
  batchedGemv(g, L.a11.numItems, L.a11.npMax, s, &launches_);
  if (timeIt) {
    HY_CUDA(cudaEventRecord(evB_, s));
    HY_CUDA(cudaEventSynchronize(evB_));
    float ms = 0;
    HY_CUDA(cudaEventElapsedTime(&ms, evA_, evB_));
    a11Ms_ += ms;
    a11Launches_++;
  }
  // x1 -= Q1 S on the owned interiors
  if (bm) borderCorrect(X, L.intRow.p, L.Q1.p, S.nI, bm, bS_.p, D.nRows12, s, &launches_, D.rows12.p);
  mark("A12 spmv + A11 gemv 2");
}

// owned entries of a global-length vector -> the full vector on every rank (replicated output of the plain API)
void Engine::gatherOwned(const double* Xowned, double* Xfull) {
  DistPlan& D = levels_[0]->dist;
  cudaStream_t s = stream_;
  const int P = comm_.size();
  double* mine = D.gath.p + (int64_t)comm_.rank() * D.maxOwn;
  packIdx(Xowned, D.ownRows.p, mine, D.nOwn, s, &launches_);
  comm_.allGather(mine, D.gath.p, (size_t)D.maxOwn, s);
  scatterVecMasked(D.gath.p, D.allRows.p, Xfull, (int64_t)P * D.maxOwn, s, &launches_);
}

int64_t Engine::ownedRows(int64_t* rows, int64_t cap) {
  if (!initialized_) throw Error(HYMLS_B200_ERR_STATE, "not initialized");
  if (comm_.size() <= 1) {
    if (rows && cap >= n_)
      for (int64_t r = 0; r < n_; ++r) rows[r] = r;
    return n_;
  }
  DistPlan& D = levels_[0]->dist;
  if (!D.ready) throw Error(HYMLS_B200_ERR_STATE, "owned_rows: no distributed plan (Number of Levels = 0 is single-GPU only)");
  if (rows && cap >= D.nOwn)
    for (int64_t i = 0; i < D.nOwn; ++i) rows[i] = D.hOwnRows[i];
  return D.nOwn;
}

}  // namespace hymls

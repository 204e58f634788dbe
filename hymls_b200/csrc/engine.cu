#include "engine.hpp"

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstring>
#include <functional>
#include <random>
#include <thread>

#include "hostpar.hpp"

namespace hymls {

thread_local double g_devBytes = 0;
thread_local DeviceArena* g_arena = nullptr;

static const double SMALL_ENTRY = 1e-14;  // HYMLS_SMALL_ENTRY

// ---------------------------------------------------------------------------------------------
// parameter validation (Preconditioner::getValidParameters, src/HYMLS_Preconditioner.cpp:135-276)
// ---------------------------------------------------------------------------------------------
static bool startsWith(const std::string& s, const char* p) { return s.rfind(p, 0) == 0; }
static void validatePreconditionerList(const ParameterList& prec) {
  static const char* valid[] = {
      "Apply Dropping", "Apply Orthogonal Transformation", "B-Grid Transform", "Coarsening Factor",
      "Coarsening Factor (x)", "Coarsening Factor (y)", "Coarsening Factor (z)", "Dense Solvers on Level",
      "Eliminate Retained Nodes Together", "Eliminate Velocities Together", "Fix Pressure Level",
      "Number of Levels", "Partitioner", "Preconditioner Variant", "Separator Length", "Separator Length (x)",
      "Separator Length (y)", "Separator Length (z)", "Subdivide Separators", "Subdivide based on variable",
      "Subdomain Solver Num Threads", "Subdomain Solver Type", "Visualize Solver",
      // extension of this implementation (DESIGN.md, "Deviations")
      "Eliminate Tube Pressures With Velocities", "Refine Inverses"};
  for (const std::string& name : prec.parameterNames()) {
    bool ok = startsWith(name, "Fix GID ") || startsWith(name, "Retain Nodes");
    for (const char* v : valid) ok = ok || name == v;
    if (!ok)
      throw Error(HYMLS_B200_ERR_ARG, "Error, the parameter {name=\"" + name +
                                          "\"} in the parameter (sub)list \"Preconditioner\" was not found in the "
                                          "list of valid parameters");
  }
  for (const std::string& name : prec.sublistNames())
    if (name != "Sparse Solver" && name != "Dense Solver" && name != "Coarse Solver" && name != "Direct Solver")
      throw Error(HYMLS_B200_ERR_ARG, "unknown sublist \"" + name + "\" in \"Preconditioner\"");
}

Engine::Engine(const std::string& xml) {
  params_ = ParameterList::fromXml(xml);
  int ndev = 0;
  deviceOk_ = (cudaGetDeviceCount(&ndev) == cudaSuccess && ndev > 0);
  if (!deviceOk_) cudaGetLastError();
  readParameters();
  if (deviceOk_) {
    HY_CUDA(cudaGetDevice(&device_));
    HY_CUDA(cudaEventCreate(&ev0_));
    HY_CUDA(cudaEventCreate(&ev1_));
    HY_CUDA(cudaEventCreate(&evA_));
    HY_CUDA(cudaEventCreate(&evB_));
    if (const char* e = getenv("HYMLS_B200_SPLIT_SOLVE")) splitSolve_ = atoi(e) != 0;
    int lo = 0, hi = 0;
    HY_CUDA(cudaDeviceGetStreamPriorityRange(&lo, &hi));  // lo = least priority
    HY_CUDA(cudaStreamCreateWithPriority(&side_, cudaStreamNonBlocking, lo));
    HY_CUDA(cudaEventCreateWithFlags(&evFork_, cudaEventDisableTiming));
    HY_CUDA(cudaEventCreateWithFlags(&evJoin_, cudaEventDisableTiming));
  }
}

// validates the list and reads what the engine itself needs (setParameterList / validateParameters,
// src/HYMLS_Preconditioner.cpp:45-130); everything else is read where it is used
void Engine::readParameters() {
  ParameterList& prec = params_.sublist("Preconditioner");
  validatePreconditionerList(prec);
  maxLevel_ = prec.get("Number of Levels", 1);
  // extension: one Newton-Schulz step on every explicit inverse (DESIGN.md, parity section); default on
  refine_ = prec.get("Refine Inverses", true);
  if (const char* e = getenv("HYMLS_B200_REFINE")) refine_ = atoi(e) != 0;
  std::string method = prec.get("Partitioner", "Cartesian");
  if (method != "Cartesian" && method != "Skew Cartesian")
    throw Error(HYMLS_B200_ERR_ARG, "Partitioner '" + method + "': Up to now we only support Cartesian partitioning");
  std::string variant = prec.get("Preconditioner Variant", "Block Diagonal");
  bool dropping = prec.get("Apply Dropping", true);
  bool ot = prec.get("Apply Orthogonal Transformation", dropping);
  if (variant != "Block Diagonal" || !dropping || !ot)
    throw Error(HYMLS_B200_ERR_UNSUPPORTED,
                "only 'Block Diagonal' with dropping and orthogonal transformation is implemented");
}

// Preconditioner::SetParameters (src/HYMLS_Preconditioner.cpp:87-114): a new list; Initialize() has to follow
void Engine::setParameters(const std::string& xml) {
  ParameterList fresh = ParameterList::fromXml(xml);
  ParameterList old = params_;
  params_ = fresh;
  try {
    readParameters();
  } catch (...) {
    params_ = old;
    readParameters();
    throw;
  }
  initialized_ = false;
  computed_ = false;
}

void Engine::commInit(const void* id128, int rank, int nranks) {
  needDevice();
  if (nranks < 1 || rank < 0 || rank >= nranks) throw Error(HYMLS_B200_ERR_ARG, "comm_init: bad rank");
  if (nranks > 1) comm_.init(id128, rank, nranks); else comm_.setRankOnly(0, 1);
  if (comm_.active()) {
    // NCCL connects its channels lazily, per protocol, at the first collective that needs them (hundreds of ms
    // on 8 ranks): do that here, as part of communicator setup, with one tiny and one large call of every
    // collective the library uses, instead of inside the first Compute / ApplyInverse
    DevBuf<double> warm;
    const size_t big = (size_t)1 << 20;
    warm.alloc(big * (size_t)nranks);
    HY_CUDA(cudaMemsetAsync(warm.p, 0, warm.bytes(), stream_));
    for (size_t cnt : {(size_t)1, big}) {
      comm_.allReduceSum(warm.p, cnt, stream_);
      comm_.broadcast(warm.p, cnt, 0, stream_);
      comm_.allGather(warm.p + (size_t)rank * cnt, warm.p, cnt, stream_);
    }
    HY_CUDA(cudaStreamSynchronize(stream_));
  }
  initialized_ = false;
  computed_ = false;
}
void Engine::setRankOnly(int rank, int nranks) {
  if (nranks < 1 || rank < 0 || rank >= nranks) throw Error(HYMLS_B200_ERR_ARG, "set_rank: bad rank");
  comm_.setRankOnly(rank, nranks);
  initialized_ = false;
  computed_ = false;
}

void Engine::needDevice() const {
  if (!deviceOk_)
    throw Error(HYMLS_B200_ERR_CUDA, "hymls_b200 needs a CUDA device for this call: there is no CPU fallback");
}

Engine::~Engine() {
  if (ev0_) cudaEventDestroy(ev0_);
  if (ev1_) cudaEventDestroy(ev1_);
  if (evA_) cudaEventDestroy(evA_);
  if (evB_) cudaEventDestroy(evB_);
  if (evFork_) cudaEventDestroy(evFork_);
  if (evJoin_) cudaEventDestroy(evJoin_);
  if (side_) cudaStreamDestroy(side_);
  destroyPipeEvents();
  if (pipeStart_) cudaEventDestroy(pipeStart_);
  if (pipeCopy_) cudaStreamDestroy(pipeCopy_);
}

void Engine::setMatrix(int64_t n, const int64_t* rowptr, const int32_t* colidx, const double* values, int where) {
  if (n <= 0 || !rowptr || !colidx) throw Error(HYMLS_B200_ERR_ARG, "set_matrix_csr: bad arguments");
  if (where == HYMLS_B200_DEVICE || values) needDevice();  // values live on the device only
  std::vector<int64_t> rp(n + 1);
  if (where == HYMLS_B200_DEVICE) {
    HY_CUDA(cudaMemcpy(rp.data(), rowptr, (n + 1) * sizeof(int64_t), cudaMemcpyDeviceToHost));
  } else {
    std::memcpy(rp.data(), rowptr, (n + 1) * sizeof(int64_t));
  }
  const int64_t nnz = rp[n];
  bool samePattern = haveMatrix_ && n == n_ && hRowptr_ == rp;
  std::vector<int> ci;
  {  // the column indices are compared on both paths: equal row lengths do not make an equal pattern
    ci.resize(nnz);
    if (where == HYMLS_B200_DEVICE) {
      HY_CUDA(cudaMemcpy(ci.data(), colidx, nnz * sizeof(int), cudaMemcpyDeviceToHost));
    } else {
      std::memcpy(ci.data(), colidx, nnz * sizeof(int));
    }
    samePattern = samePattern && ci == hColidx_;
  }
  if (!samePattern) {
    n_ = n;
    hRowptr_.swap(rp);
    hColidx_.swap(ci);
    levels_.clear();
    initialized_ = false;
    haveMatrix_ = true;
    levels_.emplace_back(new Level());
    if (deviceOk_) {
      Level& L0 = *levels_[0];
      L0.rowptr.upload(hRowptr_, stream_);
      L0.colidx.upload(hColidx_, stream_);
      L0.val.alloc(nnz);
    }
  }
  computed_ = false;
  if (!values) return;  // pattern only: enough for Initialize (index maps) without a device
  Level& L0 = *levels_[0];
  HY_CUDA(cudaMemcpyAsync(L0.val.p, values, nnz * sizeof(double),
                          where == HYMLS_B200_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, stream_));
  HY_CUDA(cudaStreamSynchronize(stream_));
  computed_ = false;
}

void Engine::setTestVector(const double* tv) {
  if (!haveMatrix_) throw Error(HYMLS_B200_ERR_STATE, "set the matrix before the test vector");
  if (tv) hTestVector_.assign(tv, tv + n_); else hTestVector_.clear();
  initialized_ = false;
  computed_ = false;
}

// ---------------------------------------------------------------------------------------------
void BatchedInverse::setup(const std::vector<int>& n_, const std::vector<int>& np_,
                           const std::vector<int64_t>& matOff_, const std::vector<int64_t>& vecOff_,
                           cudaStream_t s, const std::vector<char>* applyMask, const std::vector<int>* leadRows) {
  hN = n_;
  hNp = np_;
  hMatOff = matOff_;
  hVecOff = vecOff_;
  count = (int)n_.size();
  npMax = 0;
  std::vector<int> im, ir, ml, mid;
  midNpMax = 0;
  const int rows = rowsPerWarp > 0 ? 8 * rowsPerWarp : gemvRowsPerItem();
  for (int m = 0; m < count; ++m) {
    npMax = std::max(npMax, np_[m]);
    if (applyMask && !(*applyMask)[m]) continue;
    if (smallSplit > 0 && np_[m] <= smallSplit) {  // tiny matrix: handled by the warp-per-matrix kernel
      if (n_[m] > 0) ml.push_back(m);
      continue;
    }
    if (midSplit > 0 && np_[m] <= midSplit) {      // medium matrix: one CTA per matrix
      mid.push_back(m);
      midNpMax = std::max(midNpMax, np_[m]);
      continue;
    }
    for (int r0 = 0; r0 < n_[m]; r0 += rows) {
      im.push_back(m);
      ir.push_back(r0);
    }
  }
  hItemPtr.assign(1, 0);  // first item of every matrix (exact when no matrix is masked or split off, see uses)
  {
    size_t i = 0;
    for (int m = 0; m < count; ++m) {
      while (i < im.size() && im[i] == m) ++i;
      hItemPtr.push_back((int)i);
    }
  }
  numItems = (int)im.size();
  numMats = (int)ml.size();
  matList.upload(ml, s);
  numMid = (int)mid.size();
  midList.upload(mid, s);
  numItemsLead = 0;
  if (leadRows) {
    std::vector<int> lm, lr;
    for (int m = 0; m < count; ++m)
      for (int r0 = 0; r0 < (*leadRows)[m]; r0 += rows) {
        lm.push_back(m);
        lr.push_back(r0);
      }
    numItemsLead = (int)lm.size();
    hItemPtrLead.assign(1, 0);
    {
      size_t i = 0;
      for (int m = 0; m < count; ++m) {
        while (i < lm.size() && lm[i] == m) ++i;
        hItemPtrLead.push_back((int)i);
      }
    }
    rowLimit.upload(*leadRows, s);
    itemMatLead.upload(lm, s);
    itemRow0Lead.upload(lr, s);
    std::vector<int> tm, tr;
    for (int m = 0; m < count; ++m)
      for (int r0 = (*leadRows)[m]; r0 < n_[m]; r0 += rows) {
        tm.push_back(m);
        tr.push_back(r0);
      }
    numItemsTrail = (int)tm.size();
    itemMatTrail.upload(tm, s);
    itemRow0Trail.upload(tr, s);
  }
  n.upload(hN, s);
  np.upload(hNp, s);
  matOff.upload(hMatOff, s);
  vecOff.upload(hVecOff, s);
  itemMat.upload(im, s);
  itemRow0.upload(ir, s);
  F.alloc((size_t)(count ? matOff_[count] : 0));
  HY_CUDA(cudaStreamSynchronize(s));
}
GemvArgs BatchedInverse::args() const {
  GemvArgs a{};
  a.itemMat = itemMat.p;
  a.itemRow0 = itemRow0.p;
  a.n = n.p;
  a.np = np.p;
  a.matOff = matOff.p;
  a.vecOff = vecOff.p;
  a.A = F.p;
  a.rowsPerWarp = rowsPerWarp;
  return a;
}

// ---------------------------------------------------------------------------------------------
// Initialize: symbolic phase of every level (host) + upload of the index arrays
// ---------------------------------------------------------------------------------------------
void Engine::initialize() {
  if (!haveMatrix_) throw Error(HYMLS_B200_ERR_STATE, "Initialize: no matrix set");
  auto t0 = std::chrono::steady_clock::now();
  ParameterList levelParams = params_.deepCopy();
  levels_.resize(1);
  // the symbolic phase is threaded on the host; ranks of one node share its cores
  if (!getenv("HYMLS_B200_HOST_THREADS")) {
    const unsigned hw = std::thread::hardware_concurrency();
    setHostThreads((int)std::max(1u, std::min(16u, (hw ? hw : 1u) / (unsigned)std::max(1, comm_.size()))));
  }
  const int nlev = std::max(maxLevel_, 1);
  std::vector<int> gid2row;
  for (int l = 0; l < nlev; ++l) {
    if (l > 0) levels_.emplace_back(new Level());
    Level& L = *levels_[l];
    L.sym = LevelSym();  // a re-Initialize starts from scratch
    coarseBT_.planned = coarseBT_.active = false;
    LevelSym& S = L.sym;
    S.level = l;
    L.exact = (maxLevel_ == 0);
    std::unique_ptr<CartesianPartitioner> partPtr(makePartitioner(levelParams, l));
    CartesianPartitioner& part = *partPtr;
    if (l == 0) {
      // write the defaults back like the reference does (Fix GID 1, ...) so later queries see them
      params_.sublist("Preconditioner") = levelParams.sublist("Preconditioner").deepCopy();
      params_.sublist("Problem") = levelParams.sublist("Problem").deepCopy();
      if (part.numGlobalNodes() != n_)
        throw Error(HYMLS_B200_ERR_ARG, "matrix has " + std::to_string(n_) + " rows but nx*ny*nz*dof = " +
                                            std::to_string(part.numGlobalNodes()));
      S.n = n_;
      S.rowGid.resize(n_);
      for (int64_t i = 0; i < n_; ++i) S.rowGid[i] = i;
      S.rowptr = hRowptr_.data();
      S.colidx = hColidx_.data();
      S.nnz = (int64_t)hColidx_.size();
      S.testVector = hTestVector_;
      gid2row.assign(n_, -1);
    } else {
      const LevelSym& P = levels_[l - 1]->sym;
      S.n = P.nuniq;
      S.rowGid.resize(S.n);
      for (int u = 0; u < P.nuniq; ++u) S.rowGid[u] = P.H.sepGid[P.H.uniqPtr[u]];
      S.rowptr = P.redPtr.data();
      S.colidx = P.redCol.data();
      S.nnz = (int64_t)P.redCol.size();
      S.testVector = P.nextTestVector;
      std::fill(gid2row.begin(), gid2row.end(), -1);
    }
    for (int64_t r = 0; r < S.n; ++r) gid2row[S.rowGid[r]] = (int)r;
    auto tp0 = std::chrono::steady_clock::now();
    part.partition();
    auto tp1 = std::chrono::steady_clock::now();
    buildLevelSym(S, part, gid2row);
    if (getenv("HYMLS_B200_VERBOSE"))
      fprintf(stderr, "[hymls_b200] level %d initialize: partition %.3f s, symbolic %.3f s\n", l,
              std::chrono::duration<double>(tp1 - tp0).count(),
              std::chrono::duration<double>(std::chrono::steady_clock::now() - tp1).count());
    // ownership: every level is sharded by the reference's subdomain -> rank map of that level
    // (BasePartitioner::CreatePIDMap); with fewer subdomains than ranks some ranks own nothing there
    L.ownSd.clear();
    // Level 0 runs the owner-computes halo scheme (dist.cu).  The coarser levels are 100x smaller and latency bound:
    // their subdomain solves (1 GB of inverses at 128^3) stay distributed, but everything on the separators
    // (Householder, block solves, the next level / coarse solve) is REPLICATED -- bitwise identical on every rank --
    // so that a coarse level costs two small collectives (separator right-hand side, interior result) instead of
    // four (measured at 128^3 on 8 GPUs: 0.41 ms with four collectives, 0.60 ms fully replicated).
    // HYMLS_B200_SHARD_LEVELS=k: only the first k levels are distributed at all.
    static const int shardLevels = getenv("HYMLS_B200_SHARD_LEVELS") ? atoi(getenv("HYMLS_B200_SHARD_LEVELS")) : 1 << 20;
    L.sharded = comm_.size() > 1 && l < shardLevels;
    L.repSep = L.sharded && l >= 1;
    if (L.sharded) {
      if (maxLevel_ == 0) throw Error(HYMLS_B200_ERR_UNSUPPORTED, "Number of Levels = 0 is single-GPU only");
      ParameterList pp = levelParams.deepCopy();
      std::unique_ptr<CartesianPartitioner> pidPartPtr(makePartitioner(pp, l, comm_.size(), comm_.rank()));
      CartesianPartitioner& pidPart = *pidPartPtr;
      pidPart.partition();
      const std::vector<int>& pm = pidPart.pidMap();
      L.sdRank.assign(S.nsd, 0);
      for (int sd = 0; sd < S.nsd; ++sd) {
        L.sdRank[sd] = pm[part.globalSubdomain(sd)];
        if (L.sdRank[sd] == comm_.rank()) L.ownSd.push_back(sd);
      }
    } else {
      for (int sd = 0; sd < S.nsd; ++sd) L.ownSd.push_back(sd);
    }
    // parameters of the next level (SetNextLevelParameters; sx *= cx)
    part.setNextLevelParameters(levelParams);
    L.dist.ready = false;
    if (!deviceOk_) S.ignoredInteriorCouplings = countInteriorCouplings(S);
  }
  // The inversion workspace of Compute is allocated now (its size follows from the symbolic phase alone): the device
  // side of Initialize below uses it as scratch
  if (deviceOk_) {
    auto tw0 = std::chrono::steady_clock::now();
    work_.alloc(inversionWorkspace());
    if (getenv("HYMLS_B200_VERBOSE"))
      fprintf(stderr, "[hymls_b200] initialize: inversion workspace (%.2f GB) %.3f s\n", work_.bytes() / 1e9,
              std::chrono::duration<double>(std::chrono::steady_clock::now() - tw0).count());
  }
  for (int l = 0; l < nlev; ++l) {
    Level& L = *levels_[l];
    auto tu0 = std::chrono::steady_clock::now();
    if (L.sharded && l == 0 && !L.exact) buildDistPlan(L);  // host lists always, device copies with a device
    auto tu1 = std::chrono::steady_clock::now();
    if (deviceOk_) uploadLevel(L);
    if (getenv("HYMLS_B200_VERBOSE"))
      fprintf(stderr, "[hymls_b200] level %d initialize: distributed plan %.3f s, device index arrays %.3f s\n", l,
              std::chrono::duration<double>(tu1 - tu0).count(),
              std::chrono::duration<double>(std::chrono::steady_clock::now() - tu1).count());
  }
  planHostPipeline();
  if (deviceOk_) {
    auto tr0 = std::chrono::steady_clock::now();
    reserveComputeScratch();
    HY_CUDA(cudaStreamSynchronize(stream_));
    if (getenv("HYMLS_B200_VERBOSE"))
      fprintf(stderr, "[hymls_b200] initialize: scratch reservation %.3f s\n",
              std::chrono::duration<double>(std::chrono::steady_clock::now() - tr0).count());
  }
  initialized_ = true;
  computed_ = false;
  stats_.num_initialize++;
  stats_.time_initialize += std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
}

template <typename T>
static std::vector<int> toInt(const std::vector<T>& v) {
  return std::vector<int>(v.begin(), v.end());
}

void Engine::uploadLevel(Level& L) {
  LevelSym& S = L.sym;
  cudaStream_t s = stream_;
  ArenaScope arenaScope(&L.arena);
  // scratch of the device-side index construction: one or two slabs, released together at the end
  DeviceArena scratch((size_t)512 << 20, ~(size_t)0 >> 1);
  scratch.adopt(work_.p, work_.bytes());  // the Compute workspace is idle now: no extra cudaMalloc / cudaFree
  const bool lapOn = getenv("HYMLS_B200_VERBOSE_SYM") != nullptr;
  auto lapT = std::chrono::steady_clock::now();
  auto lap = [&](const char* what) {
    if (!lapOn) return;
    cudaStreamSynchronize(s);
    auto t1 = std::chrono::steady_clock::now();
    fprintf(stderr, "[hymls_b200 upload] %-40s %.3f s\n", what, std::chrono::duration<double>(t1 - lapT).count());
    lapT = t1;
  };
  if (S.level > 0) {
    const LevelSym& P = levels_[S.level - 1]->sym;
    L.rowptr.upload(P.redPtr, s);
    L.colidx.upload(P.redCol, s);
    L.val.alloc(P.redCol.size());
  }
  L.intRow.upload(S.intRow, s);
  L.sepRow.upload(S.sepRow, s);
  // A11: compact storage of the owned subdomains
  const int nown = (int)L.ownSd.size();
  std::vector<char> isOwn(S.nsd, 0);
  std::vector<int> on(nown), onp(nown), onb(nown);
  std::vector<int64_t> ovec(nown), a11OffG(S.nsd, -1);
  L.ownOff.assign(nown + 1, 0);
  for (int k = 0; k < nown; ++k) {
    const int sd = L.ownSd[k];
    isOwn[sd] = 1;
    on[k] = S.sdN[sd];
    onp[k] = S.sdNp[sd];
    onb[k] = S.sdNb[sd];
    ovec[k] = S.H.intPtr[sd];
    a11OffG[sd] = L.ownOff[k];
    L.ownOff[k + 1] = L.ownOff[k] + (int64_t)onp[k] * onp[k];
  }
  lap("row lists");
  L.a11.setup(on, onp, L.ownOff, ovec, s, nullptr, &onb);
  lap("A11 batched-inverse setup");
  L.sdNG.upload(S.sdN, s);
  L.sdNpG.upload(S.sdNp, s);
  L.a11OffG.upload(a11OffG, s);
  L.intPtrG.upload(S.H.intPtr, s);
  // Index arrays derived from the pattern are built on the device (indexing.cu): row -> position map, the dense-fill
  // scatter list of the owned subdomains (destinations in compact numbering), the A12 / A21 / A22 split with the
  // transposed index of A12 (A21 restricted to the columns of owned interiors when sharded: partial products are
  // summed over the ranks)
  L.rowPos.alloc(S.n);
  buildRowPos(L.intRow.p, S.nI, L.sepRow.p, S.nS, L.rowPos.p, s, &launches_);
  L.posMat.alloc(S.nI);
  buildPosMat(L.a11.n.p, L.a11.vecOff.p, nown, S.nI, L.posMat.p, s, &launches_);
  {
    DevBuf<int> posSdBuf;  // interior position -> subdomain; equals posMat when every subdomain is owned
    const int* posSd = L.posMat.p;
    if (nown != S.nsd) {
      ArenaScope tmpScope(&scratch);
      posSdBuf.alloc(S.nI);
      buildPosMat(L.sdNG.p, L.intPtrG.p, S.nsd, S.nI, posSdBuf.p, s, &launches_);
      posSd = posSdBuf.p;
    }
    S.ignoredInteriorCouplings =
        buildA11List(L.rowptr.p, L.colidx.p, L.intRow.p, L.rowPos.p, L.posMat.p, posSd, S.nI, L.a11.np.p,
                     L.a11.matOff.p, L.a11.vecOff.p, nown, L.a11Src, L.a11Dst, L.a11ListPtrDev, L.a11ListPtr, &scratch, s,
                     &launches_);
  }
  lap("A11 scatter list");
  {
    SplitOut so{&L.p12, &L.c12, &L.src12, &L.p21, &L.c21, &L.src21, &L.p22, &L.c22, &L.src22, &L.t12Ptr, &L.t12Col, &L.t12Idx};
    buildSplit(L.rowptr.p, L.colidx.p, L.intRow.p, L.sepRow.p, L.rowPos.p, L.posMat.p, L.sharded, L.exact, S.nI, S.nS,
               so, &scratch, s, &launches_);
    L.nnz12 = so.nnz12;
    L.nnz21 = so.nnz21;
    L.nnz22 = so.nnz22;
    L.v12.alloc(L.nnz12);
    L.v21.alloc(L.nnz21);
  }
  if (L.sharded) {
    // interior results: every rank packs its owned segments, the packs are all-gathered
    const int P = comm_.size();
    std::vector<int64_t> cnt(P, 0);
    for (int sd = 0; sd < S.nsd; ++sd) cnt[L.sdRank[sd]] += S.sdN[sd];
    L.maxOwnI = *std::max_element(cnt.begin(), cnt.end());
    std::vector<int> packedRow((size_t)P * L.maxOwnI, -1);
    std::vector<int64_t> fill(P, 0), outOff(nown);
    int k = 0;
    for (int sd = 0; sd < S.nsd; ++sd) {
      const int q = L.sdRank[sd];
      const int64_t base = (int64_t)q * L.maxOwnI + fill[q];
      for (int i = 0; i < S.sdN[sd]; ++i) packedRow[base + i] = S.intRow[S.H.intPtr[sd] + i];
      if (q == comm_.rank()) outOff[k++] = base;
      fill[q] += S.sdN[sd];
    }
    L.packedRow.upload(packedRow, s);
    L.gatherOutOff.upload(outOff, s);
    L.xI.alloc((size_t)P * L.maxOwnI);
  }
  lap("A12 / A21 / A22");
  // Schur assembly data
  const int64_t totalRows = S.sdRowPtr[S.nsd];
  std::vector<int> rowSd(totalRows), rowInst(totalRows), rowLinkPos(totalRows);
  std::vector<int64_t> sdLinkPtr(S.nsd + 1, 0);
  std::vector<int> lnkSd, lnkSize;
  int maxM = 0, maxG = 0, maxN = 0;
  size_t maxBlkSmem = 0;
  for (int sd = 0; sd < S.nsd; ++sd) {
    const int64_t ia = S.sdInstPtr[sd], iz = S.sdInstPtr[sd + 1];
    const int nl = S.sdNumLink[sd];
    std::vector<int> lsz(nl, 0), lcnt(nl, 0);
    for (int64_t g = ia; g < iz; ++g) {
      const int l = S.instLink[g];
      for (int q = 0; q < S.instLen[g]; ++q) {
        const int64_t R = S.sdRowPtr[sd] + S.instLoc[g] + q;
        rowSd[R] = sd;
        rowInst[R] = (int)g;
        rowLinkPos[R] = lsz[l] + q;
      }
      lsz[l] += S.instLen[g];
      lcnt[l]++;
    }
    for (int l = 0; l < nl; ++l) {
      lnkSd.push_back(sd);
      lnkSize.push_back(lsz[l]);
      maxBlkSmem = std::max(maxBlkSmem, (size_t)(2 * (size_t)lsz[l] * lcnt[l] + (size_t)lcnt[l] * lcnt[l]) * 8);
    }
    sdLinkPtr[sd + 1] = (int64_t)lnkSd.size();
    maxM = std::max(maxM, S.sdM[sd]);
    maxG = std::max(maxG, (int)(iz - ia));
    maxN = std::max(maxN, S.sdNp[sd]);
  }
  L.dLen = maxN;
  L.rowSmem = (size_t)(maxN + maxM) * sizeof(double);
  L.blkSmem = maxBlkSmem;
  // per-subdomain local pieces of A21 / A22 / A12 for the Schur assembly, built on the device
  L.rowSd.upload(rowSd, s);
  L.sdSep.upload(S.sdSep, s);
  L.uniqStart.upload(toInt(S.H.uniqPtr), s);
  {
    // occurrences of every unique group: (subdomain, local offset of the group in that subdomain)
    std::vector<int64_t> occPtr(S.nuniq + 1, 0);
    const int64_t ninst = S.sdInstPtr[S.nsd];
    for (int64_t g = 0; g < ninst; ++g) occPtr[S.instUniq[g] + 1]++;
    for (int u = 0; u < S.nuniq; ++u) occPtr[u + 1] += occPtr[u];
    std::vector<int> occSd(ninst), occLoc(ninst);
    std::vector<int64_t> f(occPtr.begin(), occPtr.end() - 1);
    for (int sd = 0; sd < S.nsd; ++sd)
      for (int64_t g = S.sdInstPtr[sd]; g < S.sdInstPtr[sd + 1]; ++g) {
        const int64_t o = f[S.instUniq[g]]++;
        occSd[o] = sd;
        occLoc[o] = S.instLoc[g];
      }
    DevBuf<int64_t> dOccPtr;
    DevBuf<int> dOccSd, dOccLoc;
    {
      ArenaScope tmpScope(&scratch);
      dOccPtr.upload(occPtr, s);
      dOccSd.upload(occSd, s);
      dOccLoc.upload(occLoc, s);
    }
    LocalOut lo{&L.s21Ptr, &L.s21Col, &L.s21Src, &L.s22Ptr, &L.s22Col, &L.s22Src, &L.s12Ptr, &L.s12Row, &L.s12Src};
    buildLocalPieces(L.rowptr.p, L.colidx.p, L.sepRow.p, L.rowPos.p, L.rowSd.p, L.sdSep.p, L.intPtrG.p, L.uniqStart.p,
                     S.nuniq, S.nS, dOccPtr.p, dOccSd.p, dOccLoc.p, L.t12Ptr.p, L.t12Col.p, L.t12Idx.p, L.src12.p,
                     totalRows, lo, &scratch, s, &launches_);
    L.nnzS21 = lo.nnz21;
  }
  lap("row -> instance lists, local pieces");
  // chunks of subdomains whose workspace (C, SV: m*G each; S_LL: sum lsz^2) fits the budget
  const int64_t budget = (int64_t)96 << 20;  // doubles per array (768 MB)
  std::vector<int64_t> wsOffC(S.nsd, 0), wsOffD(S.nsd, 0), wsOffA(S.nsd, 0), wsOffS(S.nsd, 0), lnkOff(lnkSd.size(), 0);
  L.chunks.clear();
  L.chunkDLen.clear();
  L.chunkALen.clear();
  L.wsCLen = L.wsSLLLen = L.wsDLen = L.wsALen = L.wsSLen = 0;
  {
    int sd0 = 0;
    int64_t cUsed = 0, lUsed = 0, dUsed = 0, aUsed = 0, sUsed = 0;
    for (int sd = 0; sd < S.nsd; ++sd) {
      const int64_t G = S.sdInstPtr[sd + 1] - S.sdInstPtr[sd];
      const int64_t needC = (int64_t)S.sdM[sd] * G;
      int64_t needL = 0;
      for (int64_t lk = sdLinkPtr[sd]; lk < sdLinkPtr[sd + 1]; ++lk) needL += (int64_t)lnkSize[lk] * lnkSize[lk];
      if (sd > sd0 && (cUsed + needC > budget || lUsed + needL > budget)) {
        L.chunks.push_back({sd0, sd, S.sdRowPtr[sd0], S.sdRowPtr[sd], sdLinkPtr[sd0], sdLinkPtr[sd]});
        L.chunkDLen.push_back(dUsed);
        L.chunkALen.push_back(aUsed);
        sd0 = sd;
        cUsed = lUsed = dUsed = aUsed = sUsed = 0;
      }
      wsOffC[sd] = cUsed;
      wsOffD[sd] = dUsed;  // m x np arrays of the dense Schur path (A21d, D)
      wsOffA[sd] = aUsed;  // np x mp (A12d)
      wsOffS[sd] = sUsed;  // m x mp (SkD)
      {
        const int64_t mp = (S.sdM[sd] + 7) & ~7;
        dUsed += (int64_t)S.sdM[sd] * S.sdNp[sd];
        aUsed += (int64_t)S.sdNp[sd] * mp;
        sUsed += (int64_t)S.sdM[sd] * mp;
      }
      L.wsDLen = std::max(L.wsDLen, dUsed);
      L.wsALen = std::max(L.wsALen, aUsed);
      L.wsSLen = std::max(L.wsSLen, sUsed);
      cUsed += needC;
      for (int64_t lk = sdLinkPtr[sd]; lk < sdLinkPtr[sd + 1]; ++lk) {
        lnkOff[lk] = lUsed;
        lUsed += (int64_t)lnkSize[lk] * lnkSize[lk];
      }
      L.wsCLen = std::max(L.wsCLen, cUsed);
      L.wsSLLLen = std::max(L.wsSLLLen, lUsed);
    }
    if (S.nsd > sd0) {
      L.chunks.push_back({sd0, S.nsd, S.sdRowPtr[sd0], S.sdRowPtr[S.nsd], sdLinkPtr[sd0], sdLinkPtr[S.nsd]});
      L.chunkDLen.push_back(dUsed);
      L.chunkALen.push_back(aUsed);
    }
  }
  // Dense path for the rows of A21 A11^-1 (schurGemm): on the coarser levels a separator row couples to ~100
  // interior nodes, and streaming that many rows of A11^-1 per separator row costs more than one DMMA GEMM
  // per subdomain.  Level 0 (a few entries per row) keeps the sparse accumulation.
  {
    const double avgNnz = totalRows ? (double)L.nnzS21 / (double)totalRows : 0.0;
    // Measured at 128^3 (level 1: 200 subdomains, n ~ 700, m ~ 830, ~100 entries per A21 row): sparse path 113 ms,
    // dense D = A21 A11^-1 only 123 ms (the sparse product with A12 dominates), both products as GEMMs 25 ms.
    // HYMLS_B200_SCHUR_GEMM overrides: 0 = sparse everywhere, 1 = dense on every level that fits, 2 = first GEMM only.
    const bool fits = std::max(L.wsDLen, std::max(L.wsALen, L.wsSLen)) <= ((int64_t)1 << 28);
    // (sharded runs keep the sparse path by default: the owned-list variant of the dense path has not been run
    // on several GPUs yet; HYMLS_B200_SCHUR_GEMM=1 enables it there too)
    L.schurGemm = (S.level > 0 && avgNnz >= 16.0 && fits && !L.sharded) ? 1 : 0;
    if (const char* e = getenv("HYMLS_B200_SCHUR_GEMM")) L.schurGemm = fits ? atoi(e) : 0;
    L.maxM = maxM;
    L.maxNp = maxN;
  }
  if (L.sharded) {
    std::vector<int64_t> rows, links;
    const size_t nch = L.chunks.size();
    L.chunkOwnSd.assign(nch + 1, 0);
    L.chunkOwnRow.assign(nch + 1, 0);
    L.chunkOwnLink.assign(nch + 1, 0);
    size_t k = 0;
    for (size_t c = 0; c < nch; ++c) {
      while (k < L.ownSd.size() && L.ownSd[k] < L.chunks[c].sd1) {
        const int sd = L.ownSd[k];
        for (int64_t R = S.sdRowPtr[sd]; R < S.sdRowPtr[sd + 1]; ++R) rows.push_back(R);
        for (int64_t lk = sdLinkPtr[sd]; lk < sdLinkPtr[sd + 1]; ++lk) links.push_back(lk);
        ++k;
      }
      L.chunkOwnSd[c + 1] = (int64_t)k;
      L.chunkOwnRow[c + 1] = (int64_t)rows.size();
      L.chunkOwnLink[c + 1] = (int64_t)links.size();
    }
    L.ownSdList.upload(L.ownSd, s);
    L.ownRowList.upload(rows, s);
    L.ownLinkList.upload(links, s);
  }
  lap("chunks");
  {
    // Colouring of the subdomains for the pass-2 assembly: greedy, in subdomain order, on the conflict graph
    // "share a separator group".  One colour is one launch, so contributions to an entry arrive in colour order.
    std::vector<std::vector<int>> uniqSds(S.nuniq);
    for (int sd = 0; sd < S.nsd; ++sd)
      for (int64_t g = S.sdInstPtr[sd]; g < S.sdInstPtr[sd + 1]; ++g) uniqSds[S.instUniq[g]].push_back(sd);
    std::vector<int> color(S.nsd, -1);
    std::vector<char> used;
    L.ncolors = 0;
    for (int sd = 0; sd < S.nsd; ++sd) {
      used.assign(L.ncolors + 1, 0);
      for (int64_t g = S.sdInstPtr[sd]; g < S.sdInstPtr[sd + 1]; ++g)
        for (int other : uniqSds[S.instUniq[g]])
          if (color[other] >= 0) used[color[other]] = 1;
      int c = 0;
      while (used[c]) ++c;
      color[sd] = c;
      L.ncolors = std::max(L.ncolors, c + 1);
    }
    const size_t nch = L.chunks.size();
    std::vector<char> isOwnSd(S.nsd, 0);
    for (int sd : L.ownSd) isOwnSd[sd] = 1;
    std::vector<int> colSd;
    std::vector<int64_t> colLk, colRow;
    L.colSdPtr.assign(1, 0);
    L.colLkPtr.assign(1, 0);
    L.colRowPtr.assign(1, 0);
    for (size_t c = 0; c < nch; ++c)
      for (int k = 0; k < L.ncolors; ++k) {
        for (int sd = L.chunks[c].sd0; sd < L.chunks[c].sd1; ++sd) {
          if (color[sd] != k || !isOwnSd[sd]) continue;
          colSd.push_back(sd);
          for (int64_t lk = sdLinkPtr[sd]; lk < sdLinkPtr[sd + 1]; ++lk) colLk.push_back(lk);
          if (L.exact)
            for (int64_t R = S.sdRowPtr[sd]; R < S.sdRowPtr[sd + 1]; ++R) colRow.push_back(R);
        }
        L.colSdPtr.push_back((int64_t)colSd.size());
        L.colLkPtr.push_back((int64_t)colLk.size());
        L.colRowPtr.push_back((int64_t)colRow.size());
      }
    L.colSd.upload(colSd, s);
    L.colLk.upload(colLk, s);
    L.colRow.upload(colRow, s);
  }
  lap("colouring");
  L.rowInst.upload(rowInst, s);
  L.rowLinkPos.upload(rowLinkPos, s);
  L.sdM.upload(S.sdM, s);
  L.sdRowPtr.upload(S.sdRowPtr, s);
  L.sdInstPtr.upload(S.sdInstPtr, s);
  L.instLoc.upload(S.instLoc, s);
  L.instLen.upload(S.instLen, s);
  L.instUniq.upload(S.instUniq, s);
  L.instLink.upload(S.instLink, s);
  L.sdLinkPtr.upload(sdLinkPtr, s);
  L.lnkSd.upload(lnkSd, s);
  L.lnkSize.upload(lnkSize, s);
  L.lnkOff.upload(lnkOff, s);
  L.wsOffC.upload(wsOffC, s);
  L.wsOffD.upload(wsOffD, s);
  L.wsOffA.upload(wsOffA, s);
  L.wsOffS.upload(wsOffS, s);
  L.uniqBlk.upload(S.uniqBlk, s);
  L.uniqBlkOff.upload(S.uniqBlkOff, s);
  L.what.upload(S.what, s);
  std::vector<double> wd(S.what);
  for (int u = 0; u < S.nuniq; ++u)
    if (S.usign[u] < 0)
      for (int64_t p = S.H.uniqPtr[u]; p < S.H.uniqPtr[u + 1]; ++p) wd[p] = 0.0;
  L.wd.upload(wd, s);
  L.usign.upload(S.usign, s);
  L.redPtr.upload(S.redPtr, s);
  L.redCol.upload(S.redCol, s);
  lap("Schur index uploads");
  // separator blocks
  std::vector<int64_t> blkVecOff(S.blkRowPtr.begin(), S.blkRowPtr.end() - 1);
  if (L.sharded && !L.repSep) {
    // every rank holds (and inverts) all separator blocks, but applies only the ones whose owner
    // subdomain it owns; the block results are summed over the ranks in ApplyInverse
    std::vector<char> mask(S.nblk, 0);
    for (int b = 0; b < S.nblk; ++b) mask[b] = isOwn[S.blkOwnerSd[b]];
    L.blk.smallSplit = 64;
    L.blk.midSplit = 512;
    L.blk.setup(S.blkN, S.blkNp, S.blkOff, blkVecOff, s, &mask);
  } else {
    L.blk.smallSplit = 64;
    L.blk.midSplit = 512;
    L.blk.setup(S.blkN, S.blkNp, S.blkOff, blkVecOff, s);
  }
  L.blkRows.upload(S.blkRows, s);
  lap("separator-block setup");
  // work vectors
  L.x1.alloc(S.nI);
  L.y1.alloc(S.nI);
  L.rhsS.alloc(S.nS);
  L.Z.alloc(S.nS);
  L.Y.alloc(S.nS);
  L.vsRhs.alloc(S.nuniq);
  L.vsSol.alloc(S.nuniq);
  // x1 keeps zeros outside the owned subdomains and Y finite values in the V-sum rows: the border dot
  // products of the bordered ApplyInverse run over the whole vectors
  if (L.x1.n) HY_CUDA(cudaMemsetAsync(L.x1.p, 0, L.x1.bytes(), s));
  if (L.Y.n) HY_CUDA(cudaMemsetAsync(L.Y.p, 0, L.Y.bytes(), s));
  HY_CUDA(cudaStreamSynchronize(s));
  lap("work vectors");
}

// ---------------------------------------------------------------------------------------------
// Compute
// ---------------------------------------------------------------------------------------------
// Collective when sharded: every rank learns whether ANY rank met a zero pivot, so that all of them leave
// Compute with the same error instead of one rank throwing while the others wait in the next collective.
void Engine::checkInfo(const std::string& what) {
  cudaStream_t s = stream_;
  int h = 0;
  HY_CUDA(cudaMemcpyAsync(&h, info_.p, sizeof(int), cudaMemcpyDeviceToHost, s));
  HY_CUDA(cudaStreamSynchronize(s));
  bool elsewhere = false;
  if (comm_.active()) {
    flag_.alloc(1);
    double f = h != 0 ? 1.0 : 0.0;
    HY_CUDA(cudaMemcpyAsync(flag_.p, &f, sizeof(double), cudaMemcpyHostToDevice, s));
    comm_.allReduceSum(flag_.p, 1, s);
    HY_CUDA(cudaMemcpyAsync(&f, flag_.p, sizeof(double), cudaMemcpyDeviceToHost, s));
    HY_CUDA(cudaStreamSynchronize(s));
    elsewhere = (f != 0.0 && h == 0);
  }
  if (h != 0 || elsewhere)
    throw Error(HYMLS_B200_ERR_NUMERIC,
                what + ": zero pivot (" + (elsewhere ? std::string("on another rank") : "matrix " + std::to_string(h - 1)) +
                    " is exactly singular). For 3D Stokes-C on the Cartesian partitioner the reference's pressure "
                    "'tube' blocks are identically zero; see 'Eliminate Tube Pressures With Velocities' in DESIGN.md");
}

void Engine::needComm() const {
  if (comm_.size() > 1 && !comm_.active())
    throw Error(HYMLS_B200_ERR_STATE,
                "this handle was given a rank of a multi-rank run (hymls_b200_set_rank) but no communicator: "
                "call hymls_b200_comm_init before Compute / ApplyInverse / solve");
}

void Engine::compute() {
  needDevice();
  needComm();
  computed_ = false;  // a Compute that throws must not leave half-updated factors marked usable
  if (!initialized_) initialize();  // "I'll do it for you", Preconditioner.cpp:403-409
  HY_CUDA(cudaEventRecord(ev0_, stream_));
  info_.alloc(1);
  HY_CUDA(cudaMemsetAsync(info_.p, 0, sizeof(int), stream_));
  stats_.flops_compute = 0;
  for (int l = 0; l < (int)levels_.size(); ++l) computeLevel(l);
  HY_CUDA(cudaEventRecord(ev1_, stream_));
  HY_CUDA(cudaStreamSynchronize(stream_));
  float ms = 0;
  HY_CUDA(cudaEventElapsedTime(&ms, ev0_, ev1_));
  stats_.time_compute += ms * 1e-3;
  stats_.num_compute++;
  // the scratch of Compute (about 6 GB at the 128^3 workload) is kept for the next Compute: NOX recomputes the
  // preconditioner every Newton step, and cudaFree / cudaMalloc of buffers this size stall for 100s of ms
  computed_ = true;
}

// inverts the matrices [m0, m1) of `B` whose dense input has been assembled in W (chunk-relative offsets).
// `refill` (optional) writes the original matrices into W again after the inversion: with it and the scratch
// R (same size as W) every inverse gets one Newton-Schulz step against its original matrix (gj.cu)
static void invertRange(BatchedInverse& B, int m0, int m1, double* W, DevBuf<int>& piv, DevBuf<int>& perm,
                        DevBuf<int64_t>& relOff, int* info, cudaStream_t s, int64_t* launches,
                        const std::function<void()>& refill = nullptr, double* R = nullptr) {
  const int cnt = m1 - m0;
  if (cnt <= 0) return;
  int npMax = 0;
  std::vector<int64_t> rel(cnt);
  for (int m = m0; m < m1; ++m) {
    npMax = std::max(npMax, B.hNp[m]);
    rel[m - m0] = B.hMatOff[m] - B.hMatOff[m0];
  }
  if (npMax == 0) return;
  relOff.upload(rel, s);
  piv.alloc((size_t)cnt * (npMax + 128));  // pivots + the composed interchange lists (2 x 64 per matrix)
  perm.alloc((size_t)cnt * npMax);
  invertBatched(W, B.F.p + B.hMatOff[m0], relOff.p, B.n.p + m0, B.np.p + m0, cnt, npMax, piv.p, perm.p,
                piv.p + (size_t)cnt * npMax, info, s, launches);
  if (refill && R) {
    refill();
    refineInverseBatched(W, B.F.p + B.hMatOff[m0], R, relOff.p, B.n.p + m0, B.np.p + m0, cnt, npMax, s, launches);
  }
  HY_CUDA(cudaStreamSynchronize(s));  // relOff is reused by the next chunk
}

// the same for an arbitrary subset `list` of the matrices of `B` (absolute offsets; W, F, the copy of the
// originals A0 and the scratch R share the layout)
static void invertSubset(BatchedInverse& B, const std::vector<int>& list, size_t lo, size_t hi, double* Wbase,
                         DevBuf<int>& piv, DevBuf<int>& perm, DevBuf<int64_t>& offBuf, DevBuf<int>& nBuf,
                         DevBuf<int>& npBuf, int* info, cudaStream_t s, int64_t* launches, double* A0 = nullptr,
                         double* R = nullptr) {
  const int cnt = (int)(hi - lo);
  if (cnt <= 0) return;
  int npMax = 0;
  std::vector<int64_t> off(cnt);
  std::vector<int> n(cnt), np(cnt);
  for (int k = 0; k < cnt; ++k) {
    const int m = list[lo + k];
    off[k] = B.hMatOff[m];
    n[k] = B.hN[m];
    np[k] = B.hNp[m];
    npMax = std::max(npMax, np[k]);
  }
  if (npMax == 0) return;
  offBuf.upload(off, s);
  nBuf.upload(n, s);
  npBuf.upload(np, s);
  piv.alloc((size_t)cnt * (npMax + 128));
  perm.alloc((size_t)cnt * npMax);
  invertBatched(Wbase, B.F.p, offBuf.p, nBuf.p, npBuf.p, cnt, npMax, piv.p, perm.p, piv.p + (size_t)cnt * npMax, info,
                s, launches);
  if (A0 && R) refineInverseBatched(A0, B.F.p, R, offBuf.p, nBuf.p, npBuf.p, cnt, npMax, s, launches);
  HY_CUDA(cudaStreamSynchronize(s));  // the host vectors and offBuf are reused by the next chunk
}

struct PhaseTimer {
  cudaStream_t s;
  bool on;
  int level;
  std::chrono::steady_clock::time_point t0;
  PhaseTimer(cudaStream_t st, int lvl) : s(st), on(getenv("HYMLS_B200_VERBOSE") != nullptr), level(lvl) {
    if (on) { cudaStreamSynchronize(s); t0 = std::chrono::steady_clock::now(); }
  }
  void lap(const char* what) {
    if (!on) return;
    cudaStreamSynchronize(s);
    auto t1 = std::chrono::steady_clock::now();
    fprintf(stderr, "[hymls_b200] level %d %-28s %9.3f ms\n", level, what,
            std::chrono::duration<double, std::milli>(t1 - t0).count());
    t0 = t1;
  }
};

// chunks [k0, k1) of owned subdomains whose dense input fits the inversion workspace (4 GB)
std::vector<std::pair<int, int>> Engine::a11Chunks(const Level& L) const {
  std::vector<std::pair<int, int>> out;
  const int nown = (int)L.ownSd.size();
  const int64_t budget = (int64_t)1 << 29;  // doubles
  int k0 = 0;
  while (k0 < nown) {
    int k1 = k0;
    int64_t used = 0;
    while (k1 < nown && k1 - k0 < 16384) {
      const int64_t need = L.ownOff[k1 + 1] - L.ownOff[k1];
      if (k1 > k0 && used + need > budget) break;
      used += need;
      ++k1;
    }
    out.emplace_back(k0, k1);
    k0 = k1;
  }
  return out;
}

// doubles of the inversion workspace: the largest chunk of dense subdomain matrices over the levels, or the dense
// coarse matrix.  Needs the symbolic phase only.
size_t Engine::inversionWorkspace() const {
  size_t work = 0;
  const int64_t budget = (int64_t)1 << 29;  // as in a11Chunks
  for (auto& lp : levels_) {
    const Level& L = *lp;
    const LevelSym& S = L.sym;
    int64_t used = 0;
    int cnt = 0;
    for (int sd : L.ownSd) {
      const int64_t need = (int64_t)S.sdNp[sd] * S.sdNp[sd];
      if (cnt > 0 && (used + need > budget || cnt >= 16384)) {
        used = 0;
        cnt = 0;
      }
      used += need;
      ++cnt;
      work = std::max(work, (size_t)used);
    }
  }
  const LevelSym& T = levels_.back()->sym;
  const int64_t nc = ((levels_.back()->exact ? T.nS : (int64_t)T.nuniq) + 8 + 7) & ~(int64_t)7;
  return std::max(work, (size_t)(nc * nc));
}

// Allocates the scratch of Compute once, at the end of Initialize, so that the first Compute does not pay
// for cudaMalloc of multi-GB buffers (the buffers only grow afterwards).  All of it comes from ONE allocation:
// cudaMalloc / cudaFree cost 10-100 ms a call next to a 17 GB resident factor store.
void Engine::reserveComputeScratch() {
  size_t work = 0, piv = 0, perm = 0, blkW = 0, wsC = 0, wsSLL = 0, red = 0, dD = 0, dA = 0, dS = 0;
  auto batch = [&](int cnt, int npMax) {
    piv = std::max(piv, (size_t)cnt * (npMax + 128));
    perm = std::max(perm, (size_t)cnt * npMax);
  };
  for (auto& lp : levels_) {
    const Level& L = *lp;
    const LevelSym& S = L.sym;
    for (const auto& ch : a11Chunks(L)) {
      work = std::max(work, (size_t)(L.ownOff[ch.second] - L.ownOff[ch.first]));
      int npMax = 0;
      for (int k = ch.first; k < ch.second; ++k) npMax = std::max(npMax, L.a11.hNp[k]);
      batch(ch.second - ch.first, npMax);
    }
    if (!L.exact) {
      blkW = std::max(blkW, (size_t)S.blkOff[S.nblk]);
      red = std::max(red, S.redCol.size());
      wsC = std::max(wsC, (size_t)L.wsCLen);
      wsSLL = std::max(wsSLL, (size_t)L.wsSLLLen);
      if (L.schurGemm) dD = std::max(dD, (size_t)L.wsDLen);
      if (L.schurGemm == 1) {
        dA = std::max(dA, (size_t)L.wsALen);
        dS = std::max(dS, (size_t)L.wsSLen);
      }
      int npMax = 0;
      for (int b = 0; b < S.nblk; ++b) npMax = std::max(npMax, S.blkNp[b]);
      batch(std::min(S.nblk, 16384), npMax);
    }
  }
  // coarse solver: V-sums of the last level (or all separators when Number of Levels = 0), room for a border
  const LevelSym& T = levels_.back()->sym;
  const int64_t nc = ((levels_.back()->exact ? T.nS : (int64_t)T.nuniq) + 8 + 7) & ~(int64_t)7;
  work = std::max(work, (size_t)(nc * nc));
  batch(1, (int)nc);
  work_.alloc(work);  // (already there: sized by inversionWorkspace() before the uploads)
  const bool multi = comm_.size() > 1;
  struct Want { std::function<bool()> fits; std::function<void()> release, alloc; size_t bytes; };
  std::vector<Want> wants;
  auto want = [&](auto& buf, size_t cnt) {
    if (cnt == 0) return;
    auto* b = &buf;
    wants.push_back({[b, cnt] { return b->p && cnt <= b->cap; }, [b] { b->release(); }, [b, cnt] { b->alloc(cnt); },
                     (cnt * sizeof(*b->p) + 255) & ~(size_t)255});
  };
  if (refine_) {
    want(work2_, work);
    want(blkA_, std::max(blkW, (size_t)(nc * nc)));
    want(blkR_, blkW);
  }
  want(piv_, piv);
  want(perm_, perm);
  want(blkW_, blkW);
  want(wsC_, wsC);
  want(wsSV_, wsC);
  want(wsSLL_, wsSLL);
  want(a21d_, dD);  // dense Schur path (coarser levels)
  want(dmat_, dD);
  want(a12d_, dA);
  want(skd_, dS);
  if (multi) {
    want(red2_, red);
    want(blk2_, blkW);
  }
  bool allFit = true;
  size_t total = 0;
  for (const Want& w : wants) {
    allFit = allFit && w.fits();
    total += w.bytes;
  }
  if (!allFit) {  // (re-Initialize with larger needs: everything moves to a new block)
    for (const Want& w : wants) w.release();
    computeArena_.reset(new DeviceArena(total + 4096, ~(size_t)0 >> 1));
    ArenaScope scope(computeArena_.get());
    for (const Want& w : wants) w.alloc();
  } else {
    for (const Want& w : wants) w.alloc();  // sets the sizes in use
  }
}

void Engine::computeLevel(int l) {
  Level& L = *levels_[l];
  LevelSym& S = L.sym;
  cudaStream_t s = stream_;
  PhaseTimer pt(s, l);
  // (1) off-diagonal blocks: value gathers (MatrixBlock::Compute)
  gatherValues(L.val.p, L.src12.p, L.v12.p, L.nnz12, s, &launches_);
  gatherValues(L.val.p, L.src21.p, L.v21.p, (int64_t)L.v21.n, s, &launches_);
  // (2) A11 blocks: dense fill + batched inversion, in chunks of (owned) subdomains (ComputeSubdomainSolvers)
  {
    DevBuf<int64_t>& relOff = relOff_;
    for (const auto& ch : a11Chunks(L)) {
      const int k0 = ch.first, k1 = ch.second;
      const int64_t used = L.ownOff[k1] - L.ownOff[k0];
      work_.alloc((size_t)used);
      HY_CUDA(cudaMemsetAsync(work_.p, 0, used * sizeof(double), s));
      const int64_t e0 = L.a11ListPtr[k0], e1 = L.a11ListPtr[k1];
      scatterValues(L.val.p, L.a11Src.p + e0, L.a11Dst.p + e0, L.ownOff[k0], work_.p, e1 - e0, s, &launches_);
      pt.lap("  chunk fill");
      auto fillChunk = [&]() {
        HY_CUDA(cudaMemsetAsync(work_.p, 0, used * sizeof(double), s));
        scatterValues(L.val.p, L.a11Src.p + e0, L.a11Dst.p + e0, L.ownOff[k0], work_.p, e1 - e0, s, &launches_);
      };
      if (refine_) work2_.alloc((size_t)used);
      // Newton-Schulz step: with a sparse original (level 0: ~8 entries per row) the residual I - A X comes from
      // the dense-fill list directly (one GEMM per inverse instead of two); denser levels use two GEMMs
      const double avgNnz = S.nI ? (double)L.a11ListPtr.back() / (double)S.nI : 0.0;
      const bool sparseResidual = refine_ && avgNnz * 8.0 < (double)L.a11.npMax;
      invertRange(L.a11, k0, k1, work_.p, piv_, perm_, relOff, info_.p, s, &launches_,
                  (refine_ && !sparseResidual) ? std::function<void()>(fillChunk) : nullptr,
                  (refine_ && !sparseResidual) ? work2_.p : nullptr);
      if (sparseResidual) {
        int npMax = 0;
        for (int k = k0; k < k1; ++k) npMax = std::max(npMax, L.a11.hNp[k]);
        refineInverseSparse(L.val.p, L.a11Src.p, L.a11Dst.p, L.a11ListPtrDev.p + k0, L.ownOff[k0], work_.p,
                            L.a11.F.p + L.ownOff[k0], work2_.p, relOff.p, L.a11.n.p + k0, L.a11.np.p + k0, k1 - k0, npMax,
                            s, &launches_);
        HY_CUDA(cudaStreamSynchronize(s));
      }
      pt.lap("  chunk inversion");
      for (int k = k0; k < k1; ++k) stats_.flops_compute += 2.0 * std::pow((double)L.a11.hN[k], 3);
    }
    checkInfo("subdomain solver (A11) of level " + std::to_string(l));
  }
  pt.lap("A11 fill + inversion");
  if (borderM_ > 0) {
    computeBorder(l);
    pt.lap("border");
  }
  // (3) Schur complement
  SchurArgs a{};
  a.rowSd = L.rowSd.p;
  a.rowInst = L.rowInst.p;
  a.rowLinkPos = L.rowLinkPos.p;
  a.sdSep = L.sdSep.p;
  a.sdRowPtr = L.sdRowPtr.p;
  a.sdM = L.sdM.p;
  a.sdN = L.sdNG.p;
  a.sdNp = L.sdNpG.p;
  a.a11Off = L.a11OffG.p;
  a.Ainv = L.a11.F.p;
  a.val = L.val.p;
  a.s21Ptr = L.s21Ptr.p;
  a.s12Ptr = L.s12Ptr.p;
  a.s22Ptr = L.s22Ptr.p;
  a.s21Col = L.s21Col.p;
  a.s12Row = L.s12Row.p;
  a.s22Col = L.s22Col.p;
  a.s21Src = L.s21Src.p;
  a.s12Src = L.s12Src.p;
  a.s22Src = L.s22Src.p;
  a.sdInstPtr = L.sdInstPtr.p;
  a.instLoc = L.instLoc.p;
  a.instLen = L.instLen.p;
  a.instUniq = L.instUniq.p;
  a.instLink = L.instLink.p;
  a.sdLinkPtr = L.sdLinkPtr.p;
  a.lnkSd = L.lnkSd.p;
  a.lnkSize = L.lnkSize.p;
  a.lnkOff = L.lnkOff.p;
  a.uniqStart = L.uniqStart.p;
  a.uniqBlk = L.uniqBlk.p;
  a.uniqBlkOff = L.uniqBlkOff.p;
  a.wd = L.wd.p;
  a.usign = L.usign.p;
  a.redPtr = L.redPtr.p;
  a.redCol = L.redCol.p;
  a.blkNp = L.blk.np.p;
  a.blkOff = L.blk.matOff.p;
  a.wsOffC = L.wsOffC.p;
  a.dLen = L.dLen;
  a.info = info_.p;

  if (L.exact) {
    // Number of Levels = 0: S = A22 - sum_sd A21 A11^-1 A12, dense, solved directly
    // (Preconditioner::Compute :485-500 -> CoarseSolver)
    const int nS = (int)S.nS;
    const int bm = borderM_;
    const int np = (nS + bm + 7) & ~7;
    work_.alloc((size_t)np * np);
    HY_CUDA(cudaMemsetAsync(work_.p, 0, (size_t)np * np * sizeof(double), s));
    // A22 part: gather the values of the A22 block into a temporary and densify
    DevBuf<double> v22;
    v22.alloc(L.nnz22);
    gatherValues(L.val.p, L.src22.p, v22.p, L.nnz22, s, &launches_);
    csrToDense(L.p22.p, L.c22.p, v22.p, work_.p, nS, np, s, &launches_);
    for (size_t q = 0; q + 1 < L.colRowPtr.size(); ++q)  // one colour of subdomains per launch: plain adds
      schurDense(a, L.colRowPtr[q], L.colRowPtr[q + 1], work_.p, np, L.rowSmem, s, &launches_, L.colRow.p);
    coarseFix_.clear();
    ParameterList& prec = params_.sublist("Preconditioner");
    for (int pos = 1; prec.isParameter("Fix GID " + std::to_string(pos)); ++pos) {
      gidx g = prec.get("Fix GID " + std::to_string(pos), -1);
      int row = -1;
      for (int64_t p = 0; p < S.nS; ++p)
        if (S.H.sepGid[p] == g) row = (int)p;
      if (row < 0) throw Error(HYMLS_B200_ERR_ARG, "fix GID: " + std::to_string(g) + " not in matrix row map");
      coarseFix_.push_back(row);
      putDirichlet(work_.p, nS, np, row, s, &launches_);
    }
    // with a border the Schur complement's border (sV, sW, sC of ComputeBorder) augments the dense matrix
    augmentAndInvertCoarse(nS, np, bm ? L.sV.p : nullptr, bm ? L.sW.p : nullptr, bm ? &L.hC : nullptr,
                           "exact Schur complement");
    v22.release();
    return;
  }

  // transformed + dropped Schur complement: reduced matrix on the V-sums (next level) and separator blocks
  Level* next = (l + 1 < (int)levels_.size()) ? levels_[l + 1].get() : nullptr;
  double* redVal;
  if (next) {
    redVal = next->val.p;
  } else {
    L.redValLast.alloc(S.redCol.size());
    redVal = L.redValLast.p;
  }
  HY_CUDA(cudaMemsetAsync(redVal, 0, S.redCol.size() * sizeof(double), s));
  DevBuf<double>& blkW = blkW_;
  blkW.alloc((size_t)S.blkOff[S.nblk]);
  HY_CUDA(cudaMemsetAsync(blkW.p, 0, blkW.bytes(), s));
  wsC_.alloc((size_t)L.wsCLen);
  wsSV_.alloc((size_t)L.wsCLen);
  wsSLL_.alloc((size_t)L.wsSLLLen);
  a.redVal = redVal;
  a.blkW = blkW.p;
  a.wsC = wsC_.p;
  a.wsSV = wsSV_.p;
  a.wsSLL = wsSLL_.p;
  a.wsOffD = L.wsOffD.p;
  a.wsOffA = L.wsOffA.p;
  a.wsOffS = L.wsOffS.p;
  a.A21d = a.D = a.A12d = a.SkD = nullptr;
  if (L.schurGemm) {
    a21d_.alloc((size_t)L.wsDLen);
    dmat_.alloc((size_t)L.wsDLen);
    if (L.schurGemm == 1) {
      a12d_.alloc((size_t)L.wsALen);
      skd_.alloc((size_t)L.wsSLen);
    }
  }
  auto denseRows = [&](SchurArgs& aa, size_t c, bool owned) {  // D = A21 A11^-1 of one chunk, before its pass 2
    if (!L.schurGemm) return;
    aa.A21d = a21d_.p;
    aa.D = dmat_.p;
    if (L.schurGemm == 1) {
      aa.A12d = a12d_.p;
      aa.SkD = skd_.p;
    }
    const Level::Chunk& ch = L.chunks[c];
    if (!owned)
      schurGemm(aa, ch.sd0, ch.sd1, ch.R0, ch.R1, L.chunkDLen[c], L.chunkALen[c], L.maxM, L.maxNp, s, &launches_);
    else
      schurGemm(aa, (int)L.chunkOwnSd[c], (int)L.chunkOwnSd[c + 1], L.chunkOwnRow[c], L.chunkOwnRow[c + 1],
                L.chunkDLen[c], L.chunkALen[c], L.maxM, L.maxNp, s, &launches_, L.ownSdList.p, L.ownRowList.p);
  };
  // pass 2 of one chunk: rows of -A21 A11^-1 A12 for the (owned) subdomains into the per-subdomain workspaces,
  // then the transformed entries colour by colour (plain adds, fixed order: bitwise reproducible)
  auto pass2 = [&](SchurArgs& aa, size_t c) {
    const Level::Chunk& ch = L.chunks[c];
    if (!L.sharded) {
      denseRows(aa, c, false);
      schurRows(aa, ch.R0, ch.R1, 2, L.rowSmem, s, &launches_);
    } else {
      denseRows(aa, c, true);
      schurRows(aa, L.chunkOwnRow[c], L.chunkOwnRow[c + 1], 2, L.rowSmem, s, &launches_, L.ownRowList.p);
    }
    for (int k = 0; k < L.ncolors; ++k) {
      const size_t q = c * (size_t)L.ncolors + k;
      schurScatter(aa, 2, (int)L.colSdPtr[q], (int)L.colSdPtr[q + 1], L.colLkPtr[q], L.colLkPtr[q + 1], L.blkSmem, s,
                   &launches_, L.colSd.p, L.colLk.p);
    }
  };
  auto pass1 = [&](SchurArgs& aa, size_t c) {  // A22 part: every subdomain sharing an entry stores the same value
    const Level::Chunk& ch = L.chunks[c];
    schurRows(aa, ch.R0, ch.R1, 1, L.rowSmem, s, &launches_);
    schurScatter(aa, 1, ch.sd0, ch.sd1, ch.lk0, ch.lk1, L.blkSmem, s, &launches_);
  };
  if (!L.sharded) {
    for (size_t c = 0; c < L.chunks.size(); ++c) pass1(a, c);
    for (size_t c = 0; c < L.chunks.size(); ++c) pass2(a, c);
  } else {
    // pass 1 (A22 part, no A11 needed) for every subdomain on every rank; pass 2 (-A21 A11^-1 A12) for the
    // owned subdomains into zeroed buffers that are summed over the ranks (FECrsMatrix::GlobalAssemble)
    for (size_t c = 0; c < L.chunks.size(); ++c) pass1(a, c);
    DevBuf<double>&red2 = red2_, &blk2 = blk2_;
    red2.alloc(S.redCol.size());
    blk2.alloc((size_t)S.blkOff[S.nblk]);
    HY_CUDA(cudaMemsetAsync(red2.p, 0, red2.bytes(), s));
    HY_CUDA(cudaMemsetAsync(blk2.p, 0, blk2.bytes(), s));
    SchurArgs a2 = a;
    a2.redVal = red2.p;
    a2.blkW = blk2.p;
    for (size_t c = 0; c < L.chunks.size(); ++c) pass2(a2, c);
    HY_CUDA(cudaStreamSynchronize(s));  // surface kernel faults here rather than inside NCCL
    comm_.allReduceSum(red2.p, red2.n, s);
    comm_.allReduceSum(blk2.p, blk2.n, s);
    axpby(1.0, red2.p, 1.0, redVal, (int64_t)red2.n, s, &launches_);
    axpby(1.0, blk2.p, 1.0, blkW.p, (int64_t)blk2.n, s, &launches_);
    HY_CUDA(cudaStreamSynchronize(s));
  }
  pt.lap("Schur assembly (2 passes)");
  {
    int h = 0;
    HY_CUDA(cudaMemcpyAsync(&h, info_.p, sizeof(int), cudaMemcpyDeviceToHost, s));
    HY_CUDA(cudaStreamSynchronize(s));
    if (h == -7) throw Error(HYMLS_B200_ERR_UNSUPPORTED, "more than 32 groups in one linked separator set");
  }
  // separator blocks (SchurPreconditioner::Compute :284-291)
  {
    DevBuf<int64_t>& relOff = relOff_;
    if (refine_) {  // the assembled blocks are needed again for the Newton-Schulz step
      blkA_.alloc(blkW.n);
      blkR_.alloc(blkW.n);
      HY_CUDA(cudaMemcpyAsync(blkA_.p, blkW.p, blkW.bytes(), cudaMemcpyDeviceToDevice, s));
    }
    if (!L.sharded || L.repSep) {
      int b0 = 0;
      while (b0 < S.nblk) {
        int b1 = std::min(S.nblk, b0 + 16384);
        const int64_t o0 = S.blkOff[b0], len = S.blkOff[b1] - o0;
        auto refill = [&]() {
          HY_CUDA(cudaMemcpyAsync(blkW.p + o0, blkA_.p + o0, len * sizeof(double), cudaMemcpyDeviceToDevice, s));
        };
        invertRange(L.blk, b0, b1, blkW.p + o0, piv_, perm_, relOff, info_.p, s, &launches_,
                    refine_ ? std::function<void()>(refill) : nullptr, refine_ ? blkR_.p + o0 : nullptr);
        b0 = b1;
      }
    } else {
      // a rank applies only the blocks whose owner subdomain it owns (uploadLevel): it inverts only those
      std::vector<int> mine;
      for (int b = 0; b < S.nblk; ++b)
        if (L.sdRank[S.blkOwnerSd[b]] == comm_.rank()) mine.push_back(b);
      for (size_t lo = 0; lo < mine.size(); lo += 16384)
        invertSubset(L.blk, mine, lo, std::min(mine.size(), lo + 16384), blkW.p, piv_, perm_, relOff, subsetN_,
                     subsetNp_, info_.p, s, &launches_, refine_ ? blkA_.p : nullptr, refine_ ? blkR_.p : nullptr);
    }
    for (int b = 0; b < S.nblk; ++b) stats_.flops_compute += 2.0 * std::pow((double)S.blkN[b], 3);
    checkInfo("separator block of level " + std::to_string(l));
  }
  pt.lap("separator block inversion");
  // reduced Schur complement: drop (RelDropDiag, ComputeNextLevel :548), then next level or coarse solver
  diagScratch_.alloc(S.nuniq);
  dropByValue(redVal, L.redPtr.p, L.redCol.p, diagScratch_.p, S.nuniq, SMALL_ENTRY, s, &launches_);
  if (!next) {
    std::vector<gidx> rowGid(S.nuniq);
    for (int u = 0; u < S.nuniq; ++u) rowGid[u] = S.H.sepGid[S.H.uniqPtr[u]];
    if (borderM_ > 0)
      computeCoarse(L.redPtr.p, L.redCol.p, redVal, S.nuniq, rowGid, S.redPtr, S.redCol, L.cV.p, L.cW.p, &L.hC);
    else
      computeCoarse(L.redPtr.p, L.redCol.p, redVal, S.nuniq, rowGid, S.redPtr, S.redCol);
  }
  pt.lap("drop + coarse solver");
  HY_CUDA(cudaStreamSynchronize(s));
}

// CoarseSolver::Compute (src/HYMLS_CoarseSolver.cpp:131-248): drop (RelFullDiag), Dirichlet rows for the
// "Fix GID k" entries, dense inverse.
// largest coarse system that is inverted densely; beyond it the block-tridiagonal factorization of coarse.cu
static int coarseDenseMax() {
  if (const char* e = getenv("HYMLS_B200_COARSE_DENSE_MAX")) return atoi(e);
  return 8192;
}

void Engine::computeCoarse(const int64_t* ptr, const int* col, double* val, int n, const std::vector<gidx>& rowGid,
                           const std::vector<int64_t>& hPtr, const std::vector<int>& hCol, const double* bV,
                           const double* bW, const std::vector<double>* bC) {
  cudaStream_t s = stream_;
  const int bm = bV ? borderM_ : 0;
  const int np = (n + bm + 7) & ~7;
  coarseBT_.active = false;
  if (n == 0) {
    std::vector<int> z(1, 0);
    std::vector<int64_t> off{0, 0}, voff(1, 0);
    coarse_.setup(z, z, off, voff, s);
    coarseN_ = coarseM_ = 0;
    return;
  }
  diagScratch_.alloc(n);
  dropByValue(val, ptr, col, diagScratch_.p, n, SMALL_ENTRY, s, &launches_);
  coarseFix_.clear();
  ParameterList& prec = params_.sublist("Preconditioner");
  for (int pos = 1; prec.isParameter("Fix GID " + std::to_string(pos)); ++pos) {
    gidx g = prec.get("Fix GID " + std::to_string(pos), -1);
    int row = -1;
    for (int r = 0; r < n; ++r)
      if (rowGid[r] == g) row = r;
    if (row < 0) throw Error(HYMLS_B200_ERR_ARG, "fix GID: " + std::to_string(g) + " not in matrix row map");
    coarseFix_.push_back(row);
  }
  if (n + bm > coarseDenseMax()) {
    // sparse route: block-tridiagonal factorization on BFS level sets (coarse.cu)
    if (bm)
      throw Error(HYMLS_B200_ERR_UNSUPPORTED,
                  "a bordered coarse system with more than " + std::to_string(coarseDenseMax()) +
                      " rows is not supported: use one more level");
    for (int row : coarseFix_) putDirichletCsr(val, ptr, col, row, s, &launches_);
    if (!coarseBT_.planned) planCoarseBT(hPtr, hCol, n);
    factorCoarseBT(ptr, col, val);
    coarseN_ = n;
    coarseM_ = 0;
    return;
  }
  work_.alloc((size_t)np * np);
  HY_CUDA(cudaMemsetAsync(work_.p, 0, (size_t)np * np * sizeof(double), s));
  csrToDense(ptr, col, val, work_.p, n, np, s, &launches_);
  for (int row : coarseFix_) putDirichlet(work_.p, n, np, row, s, &launches_);
  augmentAndInvertCoarse(n, np, bV, bW, bC, "coarse solver");
}

// CoarseSolver::ApplyInverse (src/HYMLS_CoarseSolver.cpp:268-323) without a border
void Engine::coarseSolve(double* rhs, double* sol, int n) {
  cudaStream_t s = stream_;
  for (int row : coarseFix_)
    if (row > 0) setValue(rhs, row, 0.0, s, &launches_);  // sic: 'lid > 0'
  if (coarseBT_.active) {
    solveCoarseBT(rhs, sol);
    return;
  }
  GemvArgs c = coarse_.args();
  c.xin = rhs;
  c.out = sol;
  c.mode = 0;
  batchedGemv(c, coarse_.numItems, coarse_.npMax, s, &launches_);
  (void)n;
}

// work_ holds the n x n coarse matrix (leading dimension np >= n + m): append the border
// (AugmentedMatrix [S V; W' C], src/HYMLS_CoarseSolver.cpp:200-224) and invert
void Engine::augmentAndInvertCoarse(int n, int np, const double* bV, const double* bW, const std::vector<double>* bC,
                                    const char* what) {
  cudaStream_t s = stream_;
  const int bm = bV ? borderM_ : 0;
  if (bm) {
    bC_.upload(*bC, s);
    denseBorder(work_.p, n, np, bV, bW, n, bC_.p, bm, s, &launches_);
  }
  std::vector<int> cn(1, n + bm), cnp(1, np);
  std::vector<int64_t> off{0, (int64_t)np * np}, voff(1, 0);
  coarse_.rowsPerWarp = (n + bm) < 32 * 148 * 4 ? 1 : 0;  // one matrix: 8-row slabs give 4x the CTAs
  coarse_.setup(cn, cnp, off, voff, s);
  coarseN_ = n;
  coarseM_ = bm;
  coarseRhs_.alloc(n + bm);
  coarseSol_.alloc(n + bm);
  DevBuf<int64_t>& relOff = relOff_;
  const size_t clen = (size_t)np * np;
  if (refine_) {
    blkA_.alloc(clen);
    work2_.alloc(clen);
    HY_CUDA(cudaMemcpyAsync(blkA_.p, work_.p, clen * sizeof(double), cudaMemcpyDeviceToDevice, s));
  }
  auto refill = [&]() {
    HY_CUDA(cudaMemcpyAsync(work_.p, blkA_.p, clen * sizeof(double), cudaMemcpyDeviceToDevice, s));
  };
  invertRange(coarse_, 0, 1, work_.p, piv_, perm_, relOff, info_.p, s, &launches_,
              refine_ ? std::function<void()>(refill) : nullptr, refine_ ? work2_.p : nullptr);
  checkInfo(what);
  stats_.flops_compute += 2.0 * std::pow((double)(n + bm), 3);
}

// ---------------------------------------------------------------------------------------------
// Border (Preconditioner::SetBorder / ComputeBorder, src/HYMLS_Preconditioner.cpp:844-918, 519-588;
// SchurPreconditioner::ComputeBorder, src/HYMLS_SchurPreconditioner.cpp:631-664)
// ---------------------------------------------------------------------------------------------
void Engine::setBorder(const double* V, const double* W, const double* C, int m) {
  if (!haveMatrix_) throw Error(HYMLS_B200_ERR_STATE, "set the matrix before the border");
  if (!V || m <= 0) {  // removes the border
    borderM_ = 0;
    hV_.clear();
    hW_.clear();
    hC_.clear();
  } else {
    borderM_ = m;
    hV_.assign(V, V + (size_t)n_ * m);
    if (W) hW_.assign(W, W + (size_t)n_ * m); else hW_ = hV_;
    if (C) hC_.assign(C, C + (size_t)m * m); else hC_.assign((size_t)m * m, 0.0);
  }
  computed_ = false;  // "Compute() needs to be called after SetBorder" (:874-875)
}

void Engine::computeBorder(int l) {
  Level& L = *levels_[l];
  const LevelSym& S = L.sym;
  cudaStream_t s = stream_;
  const int bm = borderM_;
  const int64_t n = S.n, nI = S.nI, nS = S.nS;
  if (l == 0) {
    L.bV.upload(hV_, s);
    L.bW.upload(hW_, s);
    bC0_.upload(hC_, s);
    L.hC = hC_;
  }
  L.Q1.alloc((size_t)nI * bm);
  L.W1t.alloc((size_t)nI * bm);
  L.sV.alloc((size_t)nS * bm);
  L.sW.alloc((size_t)nS * bm);
  L.bQ.alloc(bm);
  L.bT.alloc(bm);
  bS_.alloc(bm);
  bTin_.alloc(bm);
  bPartial_.alloc((size_t)(bm + 2) * multiDotBlocks());
  bDots_.alloc((size_t)bm * bm + bm);
  if (L.Q1.n) HY_CUDA(cudaMemsetAsync(L.Q1.p, 0, L.Q1.bytes(), s));
  for (int j = 0; j < bm; ++j) {
    const double* Vj = L.bV.p + (int64_t)j * n;
    const double* Wj = L.bW.p + (int64_t)j * n;
    double* Q1j = L.Q1.p + (int64_t)j * nI;
    double* sVj = L.sV.p + (int64_t)j * nS;
    double* sWj = L.sW.p + (int64_t)j * nS;
    // Q1 = A11 \ V1  (owned subdomains; the other ranks' parts are added below)
    GemvArgs g = L.a11.args();
    g.xin = Vj;
    g.gather = L.intRow.p;
    g.out = Q1j;
    g.mode = 0;
    batchedGemv(g, L.a11.numItems, L.a11.npMax, s, &launches_);
    // sV = V2 - A21 Q1
    if (!L.sharded) {
      spmv(L.p21.p, L.c21.p, L.v21.p, Q1j, sVj, nS, 1.0, Vj, L.sepRow.p, -1.0, s, &launches_);
    } else {
      spmv(L.p21.p, L.c21.p, L.v21.p, Q1j, L.Z.p, nS, 0.0, nullptr, nullptr, -1.0, s, &launches_);
      comm_.allReduceSum(L.Z.p, (size_t)nS, s);
      gatherAdd(Vj, L.sepRow.p, L.Z.p, sVj, nS, s, &launches_);
    }
    // W1t = A11' \ W1 (transposed subdomain solves, :564-566) ;  sW = W2 - A12' W1t
    double* w1t = L.W1t.p + (int64_t)j * nI;
    if (nI) HY_CUDA(cudaMemsetAsync(w1t, 0, (size_t)nI * sizeof(double), s));
    GemvArgs gt = L.a11.args();
    gt.xin = Wj;
    gt.gather = L.intRow.p;
    gt.out = w1t;
    batchedGemvT(gt, L.a11.count, L.a11.npMax, s, &launches_);
    spmvIndexed(L.t12Ptr.p, L.t12Col.p, L.t12Idx.p, L.v12.p, w1t, L.Z.p, nS, -1.0, s, &launches_);
    if (L.sharded) comm_.allReduceSum(L.Z.p, (size_t)nS, s);
    gatherAdd(Wj, L.sepRow.p, L.Z.p, sWj, nS, s, &launches_);
  }
  // sC = C - W1' Q1 (Q1 still holds the owned subdomains only: partial sums over the ranks); entry (i, j) is
  // W_i[interior] . Q1_j, with W gathered on the fly
  for (int j = 0; j < bm; ++j)
    for (int i = 0; i < bm; ++i)
      multiDot(L.Q1.p + (int64_t)j * nI, nI, 1, L.bW.p + (int64_t)i * n, nI, bPartial_.p,
               bDots_.p + (size_t)j * bm + i, 0, s, &launches_, L.intRow.p);
  if (nI == 0) HY_CUDA(cudaMemsetAsync(bDots_.p, 0, bDots_.bytes(), s));
  if (L.sharded) {
    comm_.allReduceSum(bDots_.p, (size_t)bm * bm, s);
    comm_.allReduceSum(L.Q1.p, L.Q1.n, s);
  }
  std::vector<double> dots((size_t)bm * bm), sC(L.hC);
  HY_CUDA(cudaMemcpyAsync(dots.data(), bDots_.p, dots.size() * sizeof(double), cudaMemcpyDeviceToHost, s));
  HY_CUDA(cudaStreamSynchronize(s));
  for (int j = 0; j < bm; ++j)
    for (int i = 0; i < bm; ++i) sC[i + (size_t)j * bm] -= dots[(size_t)j * bm + i];
  if (L.exact) {  // the dense Schur complement takes (sV, sW, sC) as they are
    L.hC = sC;
    return;
  }
  // borders of the transformed Schur complement: H sV, H sW; their V-sum rows are the next level's border
  Level* next = (l + 1 < (int)levels_.size()) ? levels_[l + 1].get() : nullptr;
  DevBuf<double>& nV = next ? next->bV : L.cV;
  DevBuf<double>& nW = next ? next->bW : L.cW;
  nV.alloc((size_t)S.nuniq * bm);
  nW.alloc((size_t)S.nuniq * bm);
  for (int j = 0; j < bm; ++j) {
    double* sVj = L.sV.p + (int64_t)j * nS;
    double* sWj = L.sW.p + (int64_t)j * nS;
    householder(L.uniqStart.p, S.nuniq, L.what.p, sVj, sVj, nV.p + (int64_t)j * S.nuniq, nullptr, nullptr, nullptr, s,
                &launches_);
    householder(L.uniqStart.p, S.nuniq, L.what.p, sWj, sWj, nW.p + (int64_t)j * S.nuniq, nullptr, nullptr, nullptr, s,
                &launches_);
    zeroAt(sWj, L.uniqStart.p, S.nuniq, s, &launches_);  // "note zeros in X2" (SchurPreconditioner.cpp:1585)
  }
  if (next) next->hC = sC; else L.hC = sC;  // last level: hC is what the coarse solver gets
  HY_CUDA(cudaStreamSynchronize(s));
}

// ---------------------------------------------------------------------------------------------
// ApplyInverse
// ---------------------------------------------------------------------------------------------
struct ApplyTimer {
  cudaStream_t s;
  bool on;
  int level;
  std::chrono::steady_clock::time_point t0;
  ApplyTimer(cudaStream_t st, int lvl, bool enable) : s(st), on(enable), level(lvl) {
    if (on) { cudaStreamSynchronize(s); t0 = std::chrono::steady_clock::now(); }
  }
  void lap(const char* what) {
    if (!on) return;
    cudaStreamSynchronize(s);
    auto t1 = std::chrono::steady_clock::now();
    fprintf(stderr, "[hymls_b200 apply] level %d %-34s %8.3f ms\n", level, what,
            std::chrono::duration<double, std::milli>(t1 - t0).count());
    t0 = t1;
  }
};

// [sol; S] = coarse^-1 [rhs; T]  (CoarseSolver::ApplyInverse with a border, src/HYMLS_CoarseSolver.cpp:454-564:
// no zeroing of the fixed rows in the augmented solve); S goes to bS_
void Engine::coarseSolveBordered(const double* rhs, const double* T, double* sol, int n) {
  cudaStream_t s = stream_;
  const int bm = coarseM_;
  HY_CUDA(cudaMemcpyAsync(coarseRhs_.p, rhs, (size_t)n * sizeof(double), cudaMemcpyDeviceToDevice, s));
  HY_CUDA(cudaMemcpyAsync(coarseRhs_.p + n, T, (size_t)bm * sizeof(double), cudaMemcpyDeviceToDevice, s));
  GemvArgs c = coarse_.args();
  c.xin = coarseRhs_.p;
  c.out = coarseSol_.p;
  c.mode = 0;
  batchedGemv(c, coarse_.numItems, coarse_.npMax, s, &launches_);
  HY_CUDA(cudaMemcpyAsync(sol, coarseSol_.p, (size_t)n * sizeof(double), cudaMemcpyDeviceToDevice, s));
  HY_CUDA(cudaMemcpyAsync(bS_.p, coarseSol_.p + n, (size_t)bm * sizeof(double), cudaMemcpyDeviceToDevice, s));
}

// separator-block solves Y[blkRows] = blockinv * Z[blkRows] (ApplyBlockDiagonal, src/HYMLS_SchurPreconditioner.cpp:1311-1346)
void Engine::blockSolves(Level& L, const double* Z, double* Y) {
  GemvArgs b = L.blk.args();
  b.xin = Z;
  b.gather = L.blkRows.p;
  b.out = Y;
  b.scatter = L.blkRows.p;
  b.mode = 0;
  // blocks of up to 64 rows (edges, pressure tubes, ragged faces) go one per warp, blocks of up to 512 rows (faces)
  // one per CTA; only larger ones (coarser levels) use the CTA-per-32-row-slab kernel
  smallGemv(b, L.blk.matList.p, L.blk.numMats, std::min(L.blk.npMax, L.blk.smallSplit), stream_, &launches_);
  ctaGemv(b, L.blk.midList.p, L.blk.numMid, L.blk.midNpMax, stream_, &launches_);
  batchedGemv(b, L.blk.numItems, L.blk.npMax, stream_, &launches_);
}

void Engine::applyLevel(int l, const double* B, double* X, const double* T) {
  Level& L = *levels_[l];
  const LevelSym& S = L.sym;
  cudaStream_t s = stream_;
  static const bool verboseApply = getenv("HYMLS_B200_VERBOSE_APPLY") != nullptr;
  ApplyTimer at(s, l, verboseApply && comm_.rank() == 0 && (stats_.num_apply_inverse % 16) == 5);
  // x1 = A11 \ b1 (b1 gathered from B on the fly).  x1 is only used in A21 x1, so only the leading rows of every
  // A11^-1 -- the interior nodes that separator rows couple to (LevelSym::sdNb) -- are computed and streamed;
  // the interior part of the result comes from ONE full solve at the end, x1 = A11 \ (b1 - A12 x2).
  GemvArgs g = L.a11.args();
  g.xin = B;
  g.gather = L.intRow.p;
  g.out = L.x1.p;
  g.scatter = nullptr;
  g.mode = 0;
  g.itemMat = L.a11.itemMatLead.p;
  g.itemRow0 = L.a11.itemRow0Lead.p;
  g.nrows = L.a11.rowLimit.p;
  const bool timeIt = timeA11_ && l == 0;
  // host-buffer call with the copies overlapped (applyHostPiped): b arrives in chunks on the copy stream
  const bool piped = l == 0 && pipeHostX_ != nullptr && !timeIt;
  if (timeIt) HY_CUDA(cudaEventRecord(evA_, s));
  if (piped) {
    const HostPipePlan& P = pipePlan_;
    for (int c = 0; c < P.K; ++c) {
      HY_CUDA(cudaStreamWaitEvent(s, pipeIn_[c], 0));  // rows [0, inRows[c+1]) of b are on the device
      GemvArgs gc = g;
      gc.itemMat += P.leadItem[c];
      gc.itemRow0 += P.leadItem[c];
      batchedGemv(gc, P.leadItem[c + 1] - P.leadItem[c], L.a11.npMax, s, &launches_);
    }
  } else {
    batchedGemv(g, L.a11.numItemsLead, L.a11.npMax, s, &launches_);
  }
  if (timeIt) {
    HY_CUDA(cudaEventRecord(evB_, s));
    HY_CUDA(cudaEventSynchronize(evB_));
    float ms = 0;
    HY_CUDA(cudaEventElapsedTime(&ms, evA_, evB_));
    a11LeadMs_ += ms;
  }
  // Split second solve (level 0):  x1 = A11^-1 b1 - A11^-1[:, :nb] (A12 x2)[:nb].  The leading rows of A11^-1 b1 are
  // in x1 already; the remaining rows [nb, n) are computed NOW on the low-priority side stream, concurrently with
  // the latency-bound separator phase below, and the pass that has to wait for x2 reads the leading nb columns only
  // (A12 x2 is zero outside the leading interior nodes, symbolic.cpp).  Same bytes as one full pass, (n - nb) n of
  // them off the critical path.
  const bool split = splitActive(L, l);
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
  at.lap("A11 gemv 1 (leading rows)");
  const int bm = borderM_;
  if (bm) {
    // q = T - W1' (A11 \ b1) = T - (A11' \ W1)' b1 (Preconditioner.cpp:1006-1013); W1t is zero outside the
    // owned subdomains
    multiDot(L.W1t.p, S.nI, bm, B, S.nI, bPartial_.p, L.bQ.p, 0, s, &launches_, L.intRow.p);
    if (S.nI == 0) HY_CUDA(cudaMemsetAsync(L.bQ.p, 0, bm * sizeof(double), s));
    if (L.sharded) comm_.allReduceSum(L.bQ.p, (size_t)bm, s);
    axpby(T ? 1.0 : 0.0, T ? T : L.bQ.p, -1.0, L.bQ.p, bm, s, &launches_);
  }
  // schurRhs = b2 - A21 x1
  if (!L.sharded) {
    spmv(L.p21.p, L.c21.p, L.v21.p, L.x1.p, L.rhsS.p, S.nS, 1.0, B, L.sepRow.p, -1.0, s, &launches_);
  } else {
    // each rank multiplies with the columns of its own interiors; the partial products are summed
    // (the separator-halo exchange of the reference's Epetra_CrsMatrix::Apply / Import)
    spmv(L.p21.p, L.c21.p, L.v21.p, L.x1.p, L.Z.p, S.nS, 0.0, nullptr, nullptr, -1.0, s, &launches_);
    comm_.allReduceSum(L.Z.p, (size_t)S.nS, s);
    gatherAdd(B, L.sepRow.p, L.Z.p, L.rhsS.p, S.nS, s, &launches_);
  }
  at.lap("A21 spmv (+allreduce)");
  double* x2 = L.Y.p;
  if (L.exact) {
    // direct solve with the dense Schur complement (CoarseSolver::ApplyInverse :268-323)
    if (bm) {
      coarseSolveBordered(L.rhsS.p, L.bQ.p, x2, (int)S.nS);
    } else {
      for (int row : coarseFix_)
        if (row > 0) setValue(L.rhsS.p, row, 0.0, s, &launches_);  // sic: 'lid > 0'
      GemvArgs c = coarse_.args();
      c.xin = L.rhsS.p;
      c.out = x2;
      c.mode = 0;
      batchedGemv(c, coarse_.numItems, coarse_.npMax, s, &launches_);
    }
    scatterVec(x2, L.sepRow.p, X, S.nS, s, &launches_);
  } else {
    // B' = H rhs ; V-sum part goes to the next level (ApplyOT + UpdateVsumRhs)
    householder(L.uniqStart.p, S.nuniq, L.what.p, L.rhsS.p, L.Z.p, L.vsRhs.p, nullptr, nullptr, nullptr, s,
                &launches_);
    // non-V-sums: block diagonal solves (ApplyBlockDiagonal)
    const bool sumSep = L.sharded && !L.repSep;  // separator work distributed: results summed over the ranks
    if (sumSep) HY_CUDA(cudaMemsetAsync(L.Y.p, 0, (size_t)S.nS * sizeof(double), s));
    blockSolves(L, L.Z.p, L.Y.p);
    if (sumSep) comm_.allReduceSum(L.Y.p, (size_t)S.nS, s);  // owned block rows from every rank
    at.lap("householder + separator blocks");
    if (bm) {
      // Tc = q - bW' Y with zeros in the V-sum rows (SchurPreconditioner.cpp:1585-1590)
      multiDot(L.sW.p, S.nS, bm, L.Y.p, S.nS, bPartial_.p, L.bT.p, 0, s, &launches_);
      axpby(1.0, L.bQ.p, -1.0, L.bT.p, bm, s, &launches_);
    }
    // V-sums: next level or coarse solver
    if (l + 1 < (int)levels_.size()) {
      applyLevel(l + 1, L.vsRhs.p, L.vsSol.p, bm ? L.bT.p : nullptr);
    } else if (bm) {
      coarseSolveBordered(L.vsRhs.p, L.bT.p, L.vsSol.p, S.nuniq);
      if (sumSep) {
        comm_.broadcast(L.vsSol.p, (size_t)S.nuniq, 0, s);
        comm_.broadcast(bS_.p, (size_t)bm, 0, s);
      }
    } else {
      coarseSolve(L.vsRhs.p, L.vsSol.p, S.nuniq);
      // the coarse solve is replicated; rank 0's copy becomes the common one so that every rank
      // continues with bit-identical data (replicas may differ in the last bit, which a Krylov method
      // mixing per-rank partial results would amplify)
      if (sumSep) comm_.broadcast(L.vsSol.p, (size_t)S.nuniq, 0, s);
    }
    at.lap("next level / coarse");
    // x2 = H [Y(non-V-sum); vsumSol], exported to X
    householder(L.uniqStart.p, S.nuniq, L.what.p, L.Y.p, L.Y.p, nullptr, L.vsSol.p, X, L.sepRow.p, s, &launches_);
  }
  at.lap("householder back (+bcast)");
  // y1 = A12 x2 ;  X[interior] = A11 \ (b1 - y1)
  spmv(L.p12.p, L.c12.p, L.v12.p, x2, L.y1.p, S.nI, 0.0, nullptr, nullptr, 1.0, s, &launches_);
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
  if (L.sharded) {  // owned interiors packed per rank, all-gathered, then exported
    g.out = L.xI.p;
    g.outOff = L.gatherOutOff.p;
    g.scatter = nullptr;
  }
  if (timeIt) HY_CUDA(cudaEventRecord(evA_, s));
  if (piped && !L.sharded && !split) {
    // the separator rows of X are final already (Householder above); after chunk c so are the interior rows below
    // the first row of the later chunks: they leave on the copy stream while the next chunk runs
    const HostPipePlan& P = pipePlan_;
    for (int c = 0; c < P.K; ++c) {
      GemvArgs gc = g;
      gc.itemMat += P.fullItem[c];
      gc.itemRow0 += P.fullItem[c];
      batchedGemv(gc, P.fullItem[c + 1] - P.fullItem[c], L.a11.npMax, s, &launches_);
      HY_CUDA(cudaEventRecord(pipeOut_[c], s));
      HY_CUDA(cudaStreamWaitEvent(pipeCopy_, pipeOut_[c], 0));
      const int64_t r0 = P.outRows[c], r1 = P.outRows[c + 1];
      if (r1 > r0)
        HY_CUDA(cudaMemcpyAsync(pipeHostX_ + r0, X + r0, (size_t)(r1 - r0) * sizeof(double), cudaMemcpyDeviceToHost,
                                pipeCopy_));
    }
  } else {
    batchedGemv(g, L.a11.numItems, L.a11.npMax, s, &launches_);
  }
  if (timeIt) {
    HY_CUDA(cudaEventRecord(evB_, s));
    HY_CUDA(cudaEventSynchronize(evB_));
    float ms = 0;
    HY_CUDA(cudaEventElapsedTime(&ms, evA_, evB_));
    a11Ms_ += ms;
    a11Launches_++;
  }
  at.lap("A12 spmv + A11 gemv 2");
  if (L.sharded) {
    comm_.allGather(L.xI.p + (int64_t)comm_.rank() * L.maxOwnI, L.xI.p, (size_t)L.maxOwnI, s);
    scatterVecMasked(L.xI.p, L.packedRow.p, X, (int64_t)comm_.size() * L.maxOwnI, s, &launches_);
  }
  // x1 -= Q1 S (Preconditioner.cpp:1036-1041), on the exported interior rows
  if (bm) borderCorrect(X, L.intRow.p, L.Q1.p, S.nI, bm, bS_.p, S.nI, s, &launches_);
  at.lap("interior allreduce + export");
}

// ApplyInverse on nv = 2..4 columns at once (single rank, no border, transformed levels): the two passes over the
// level-0 subdomain inverses -- 85 % of the time -- are shared by the columns; the small separator-side work in
// between runs column by column.  Returns false when the configuration is not covered (the caller loops instead).
bool Engine::applyDeviceMulti(const double* dB, int64_t ldb, double* dX, int64_t ldx, int nv) {
  Level& L = *levels_[0];
  const LevelSym& S = L.sym;
  cudaStream_t s = stream_;
  if (nv < 2 || nv > 4 || L.sharded || L.exact || borderM_ > 0) return false;
  if ((size_t)L.a11.npMax * nv * sizeof(double) > 200 * 1024) return false;
  x1m_.alloc((size_t)S.nI * nv);
  y1m_.alloc((size_t)S.nI * nv);
  GemvArgs g = L.a11.args();
  g.xin = dB;
  g.gather = L.intRow.p;
  g.out = x1m_.p;
  g.mode = 0;
  g.itemMat = L.a11.itemMatLead.p;
  g.itemRow0 = L.a11.itemRow0Lead.p;
  g.nrows = L.a11.rowLimit.p;
  if (!batchedGemvMulti(g, L.a11.numItemsLead, L.a11.npMax, nv, ldb, 0, S.nI, s, &launches_)) return false;
  for (int v = 0; v < nv; ++v) {
    const double* B = dB + (int64_t)v * ldb;
    double* X = dX + (int64_t)v * ldx;
    spmv(L.p21.p, L.c21.p, L.v21.p, x1m_.p + (int64_t)v * S.nI, L.rhsS.p, S.nS, 1.0, B, L.sepRow.p, -1.0, s, &launches_);
    householder(L.uniqStart.p, S.nuniq, L.what.p, L.rhsS.p, L.Z.p, L.vsRhs.p, nullptr, nullptr, nullptr, s, &launches_);
    blockSolves(L, L.Z.p, L.Y.p);
    if (levels_.size() > 1) applyLevel(1, L.vsRhs.p, L.vsSol.p, nullptr);
    else coarseSolve(L.vsRhs.p, L.vsSol.p, S.nuniq);
    householder(L.uniqStart.p, S.nuniq, L.what.p, L.Y.p, L.Y.p, nullptr, L.vsSol.p, X, L.sepRow.p, s, &launches_);
    spmv(L.p12.p, L.c12.p, L.v12.p, L.Y.p, y1m_.p + (int64_t)v * S.nI, S.nI, 0.0, nullptr, nullptr, 1.0, s, &launches_);
  }
  g = L.a11.args();
  g.xin = dB;
  g.gather = L.intRow.p;
  g.xsub = y1m_.p;
  g.out = dX;
  g.scatter = L.intRow.p;
  g.mode = 0;
  batchedGemvMulti(g, L.a11.numItems, L.a11.npMax, nv, ldb, S.nI, ldx, s, &launches_);
  stats_.num_apply_inverse += nv;
  return true;
}

void Engine::applyDevice(const double* dB, double* dX, const double* dT, double* dS) {
  if (useDist()) {
    // replicated argument / result around the owner-computes path: every rank applies to its own rows, the
    // owned parts of the result are all-gathered (S is replicated already)
    bufD_.alloc(n_);
    applyLevel0Dist(dB, bufD_.p, dT);
    gatherOwned(bufD_.p, dX);
  } else {
    applyLevel(0, dB, dX, dT);
  }
  if (dS && borderM_)
    HY_CUDA(cudaMemcpyAsync(dS, bS_.p, borderM_ * sizeof(double), cudaMemcpyDeviceToDevice, stream_));
  stats_.num_apply_inverse++;
}

// BorderedOperator::ApplyInverse(X, T, Y, S) of the preconditioner (src/HYMLS_Preconditioner.cpp:930-1070)
void Engine::applyInverseBordered(const double* B, int64_t ldb, const double* T, double* X, int64_t ldx, double* Sout,
                                  int nvec, int where) {
  needDevice();
  needComm();
  if (!computed_) throw Error(HYMLS_B200_ERR_STATE, "The preconditioner has not yet been computed.");
  if (!B || !X || nvec < 0 || ldb < n_ || ldx < n_) throw Error(HYMLS_B200_ERR_ARG, "apply_inverse: bad arguments");
  const int bm = borderM_;
  if (bm == 0) {  // no border: S = 0 (:985-995 falls through to the plain path)
    applyInverse(B, ldb, X, ldx, nvec, where);
    return;
  }
  if (!T || !Sout) throw Error(HYMLS_B200_ERR_ARG, "apply_inverse_bordered: T and S are required");
  for (int k = 0; k < nvec; ++k) {
    const double* b = B + k * ldb;
    double* x = X + k * ldx;
    if (where == HYMLS_B200_DEVICE) {
      applyDevice(b, x, T + (size_t)k * bm, Sout + (size_t)k * bm);
    } else {
      bufB_.alloc(n_);
      bufX_.alloc(n_);
      HY_CUDA(cudaMemcpyAsync(bufB_.p, b, n_ * sizeof(double), cudaMemcpyHostToDevice, stream_));
      HY_CUDA(cudaMemcpyAsync(bTin_.p, T + (size_t)k * bm, bm * sizeof(double), cudaMemcpyHostToDevice, stream_));
      applyDevice(bufB_.p, bufX_.p, bTin_.p, nullptr);
      HY_CUDA(cudaMemcpyAsync(x, bufX_.p, n_ * sizeof(double), cudaMemcpyDeviceToHost, stream_));
      HY_CUDA(cudaMemcpyAsync(Sout + (size_t)k * bm, bS_.p, bm * sizeof(double), cudaMemcpyDeviceToHost, stream_));
      HY_CUDA(cudaStreamSynchronize(stream_));
    }
  }
}

void Engine::applyInverse(const double* B, int64_t ldb, double* X, int64_t ldx, int nvec, int where) {
  needDevice();
  needComm();
  if (!computed_) throw Error(HYMLS_B200_ERR_STATE, "The preconditioner has not yet been computed.");
  if (!B || !X || nvec < 0 || ldb < n_ || ldx < n_) throw Error(HYMLS_B200_ERR_ARG, "apply_inverse: bad arguments");
  const bool multiOk = comm_.size() <= 1 && borderM_ == 0 && !levels_[0]->exact;
  int k = 0;
  while (k < nvec) {
    // up to 4 columns share the passes over the subdomain inverses
    const int nv = multiOk ? std::min(4, nvec - k) : 1;
    const double* b = B + (int64_t)k * ldb;
    double* x = X + (int64_t)k * ldx;
    bool done = false;
    if (where == HYMLS_B200_DEVICE) {
      if (nv > 1) done = applyDeviceMulti(b, ldb, x, ldx, nv);
      if (!done) applyDevice(b, x);
    } else if (nv == 1 && hostPipeUsable(b, x)) {
      applyHostPiped(b, x);  // copies overlapped with the two passes over the level-0 inverses
    } else {
      bufB_.alloc((size_t)n_ * nv);
      bufX_.alloc((size_t)n_ * nv);
      for (int v = 0; v < nv; ++v)
        HY_CUDA(cudaMemcpyAsync(bufB_.p + (int64_t)v * n_, b + (int64_t)v * ldb, n_ * sizeof(double),
                                cudaMemcpyHostToDevice, stream_));
      if (nv > 1) done = applyDeviceMulti(bufB_.p, n_, bufX_.p, n_, nv);
      if (!done) applyDevice(bufB_.p, bufX_.p);
      const int got = done ? nv : 1;
      for (int v = 0; v < got; ++v)
        HY_CUDA(cudaMemcpyAsync(x + (int64_t)v * ldx, bufX_.p + (int64_t)v * n_, n_ * sizeof(double),
                                cudaMemcpyDeviceToHost, stream_));
      HY_CUDA(cudaStreamSynchronize(stream_));
    }
    k += done ? nv : 1;
  }
}

// ---------------------------------------------------------------------------------------------
// Host-buffer ApplyInverse with the copies overlapped (one GPU, pinned buffers)
// ---------------------------------------------------------------------------------------------
void Engine::destroyPipeEvents() {
  for (cudaEvent_t e : pipeIn_) cudaEventDestroy(e);
  for (cudaEvent_t e : pipeOut_) cudaEventDestroy(e);
  pipeIn_.clear();
  pipeOut_.clear();
}

// Part of Initialize: the chunk schedule follows from the orderings alone (host work: also done without a device, so
// that the CPU tests see it).  HYMLS_B200_HOST_PIPELINE=0 switches the pipeline off, .._CHUNKS sets K, .._TAPER=0
// makes the chunks equal, .._MIN_ROWS is the smallest problem it is used for (default 2^20 rows: at 64^3 the copies
// are 0.15 ms each and nothing is gained).  Defaults from profiles/r02_host_pipeline_variants_1gpu.log (128^3, one
// B200, serial copies 13.7 ms): 6 tapered chunks 11.87 ms, 8 tapered 11.95, 8 equal 12.10, 12 tapered 12.02,
// 16 equal 12.35 -- every chunk boundary costs about 30 us of kernel tails and event waits.
void Engine::planHostPipeline() {
  pipePlan_ = HostPipePlan();
  pipeState_ = 0;
  pipeHostX_ = nullptr;
  destroyPipeEvents();
  const char* e = getenv("HYMLS_B200_HOST_PIPELINE");
  pipeEnabled_ = e ? atoi(e) != 0 : true;  // (read again at every host-buffer call: the switch works at run time)
  e = getenv("HYMLS_B200_HOST_PIPELINE_CHUNKS");
  const int K = e ? atoi(e) : 6;
  e = getenv("HYMLS_B200_HOST_PIPELINE_MIN_ROWS");
  const int64_t minRows = e ? atoll(e) : ((int64_t)1 << 20);
  if (comm_.size() > 1 || levels_.empty() || levels_[0]->exact || n_ < minRows || K < 2 || K > 64) return;
  const Level& L = *levels_[0];
  const LevelSym& S = L.sym;
  if ((int)L.ownSd.size() != S.nsd) return;
  const std::vector<int64_t> vecOff(S.H.intPtr.begin(), S.H.intPtr.begin() + S.nsd);
  const int rows = gemvRowsPerItem();
  e = getenv("HYMLS_B200_HOST_PIPELINE_TAPER");
  const bool taper = e ? atoi(e) != 0 : true;
  HostPipePlan P = planHostPipe(S.sdN, S.sdNb, vecOff, S.intRow, S.n, rows, K, taper);
  if (P.K < 2 || !checkHostPipe(P, S.sdN, S.sdNb, vecOff, S.intRow, S.n, rows)) return;
  if (deviceOk_) {
    // the work lists on the device must be cut exactly where the plan says
    const BatchedInverse& a = L.a11;
    if ((int)a.hItemPtr.size() != S.nsd + 1 || (int)a.hItemPtrLead.size() != S.nsd + 1) return;
    for (int c = 0; c <= P.K; ++c)
      if (a.hItemPtr[P.matStart[c]] != P.fullItem[c] || a.hItemPtrLead[P.matStart[c]] != P.leadItem[c]) return;
    if (a.numItems != P.fullItem[P.K] || a.numItemsLead != P.leadItem[P.K]) return;
    if (!pipeCopy_) HY_CUDA(cudaStreamCreateWithFlags(&pipeCopy_, cudaStreamNonBlocking));
    if (!pipeStart_) HY_CUDA(cudaEventCreateWithFlags(&pipeStart_, cudaEventDisableTiming));
    pipeIn_.assign(P.K, nullptr);
    pipeOut_.assign(P.K, nullptr);
    for (int c = 0; c < P.K; ++c) {
      HY_CUDA(cudaEventCreateWithFlags(&pipeIn_[c], cudaEventDisableTiming));
      HY_CUDA(cudaEventCreateWithFlags(&pipeOut_[c], cudaEventDisableTiming));
    }
  }
  pipePlan_ = P;
}

bool Engine::hostPipeUsable(const double* b, const double* x) {
  if (const char* e = getenv("HYMLS_B200_HOST_PIPELINE")) pipeEnabled_ = atoi(e) != 0;
  if (!pipeEnabled_ || pipeState_ < 0 || pipePlan_.K < 2 || !pipeCopy_ || (int)pipeIn_.size() != pipePlan_.K) return false;
  if (comm_.size() > 1 || borderM_ > 0 || levels_.empty() || levels_[0]->exact || levels_[0]->sharded || splitSolve_ ||
      timeA11_)
    return false;
  if (b < x + n_ && x < b + n_) return false;  // in-place call: the self-check of the first call needs b intact
  // pageable memory gains nothing (its copies are staged synchronously): pinned / registered buffers only
  cudaPointerAttributes ab{}, ax{};
  if (cudaPointerGetAttributes(&ab, b) != cudaSuccess || cudaPointerGetAttributes(&ax, x) != cudaSuccess) {
    cudaGetLastError();
    return false;
  }
  return ab.type == cudaMemoryTypeHost && ax.type == cudaMemoryTypeHost;
}

void Engine::applyHostPiped(const double* b, double* x) {
  cudaStream_t s = stream_;
  const size_t bytes = (size_t)n_ * sizeof(double);
  bufB_.alloc(n_);
  bufX_.alloc(n_);
  auto piped = [&]() {
    const HostPipePlan& P = pipePlan_;
    HY_CUDA(cudaEventRecord(pipeStart_, s));  // the staging buffers may still be in use by earlier work on s
    HY_CUDA(cudaStreamWaitEvent(pipeCopy_, pipeStart_, 0));
    for (int c = 0; c < P.K; ++c) {
      const int64_t r0 = P.inRows[c], r1 = P.inRows[c + 1];
      if (r1 > r0)
        HY_CUDA(cudaMemcpyAsync(bufB_.p + r0, b + r0, (size_t)(r1 - r0) * sizeof(double), cudaMemcpyHostToDevice,
                                pipeCopy_));
      HY_CUDA(cudaEventRecord(pipeIn_[c], pipeCopy_));
    }
    pipeHostX_ = x;
    try {
      applyDevice(bufB_.p, bufX_.p);  // applyLevel(0) waits for / hands over the chunks
    } catch (...) {
      pipeHostX_ = nullptr;
      cudaStreamSynchronize(pipeCopy_);
      cudaStreamSynchronize(s);
      throw;
    }
    pipeHostX_ = nullptr;
    HY_CUDA(cudaStreamSynchronize(pipeCopy_));
    HY_CUDA(cudaStreamSynchronize(s));
  };
  if (pipeState_ == 1) {
    piped();
    return;
  }
  // first use: the serial path gives the expected result; the pipelined call then starts from poisoned buffers and
  // has to reproduce it bit for bit (same kernels on the same data, only cut into chunks)
  const int callsBefore = stats_.num_apply_inverse;
  HY_CUDA(cudaMemcpyAsync(bufB_.p, b, bytes, cudaMemcpyHostToDevice, s));
  applyDevice(bufB_.p, bufX_.p);
  HY_CUDA(cudaMemcpyAsync(x, bufX_.p, bytes, cudaMemcpyDeviceToHost, s));
  HY_CUDA(cudaStreamSynchronize(s));
  std::vector<double> expect(x, x + n_);
  HY_CUDA(cudaMemsetAsync(bufB_.p, 0xff, bytes, s));
  HY_CUDA(cudaMemsetAsync(bufX_.p, 0xff, bytes, s));
  memset(x, 0xff, bytes);
  bool same = false;
  std::string why = "results differ";
  try {
    piped();
    same = memcmp(x, expect.data(), bytes) == 0;
  } catch (const Error& err) {
    why = err.what();
  }
  stats_.num_apply_inverse = callsBefore + 1;  // one call of the user
  if (same) {
    pipeState_ = 1;
  } else {
    pipeState_ = -1;
    memcpy(x, expect.data(), bytes);
    fprintf(stderr, "[hymls_b200] host-buffer pipeline failed its self-check (%s): serial copies from now on\n",
            why.c_str());
  }
}

void Engine::localRows(int64_t* r0, int64_t* r1) const {
  if (comm_.size() > 1)
    throw Error(HYMLS_B200_ERR_STATE,
                "local_rows: with several ranks the rows are distributed by owner, not in contiguous blocks: use "
                "hymls_b200_owned_rows");
  *r0 = 0;
  *r1 = n_;
}

// Distributed-vector ApplyInverse: Bloc / Xloc hold the rows hymls_b200_owned_rows lists (ascending), i.e. the
// distribution the subdomain -> rank map of the reference induces.  With T and S (replicated m-vectors, on the same
// side as Bloc) it is the bordered ApplyInverse; without them and a border set, T = 0 and S is discarded.
void Engine::applyInverseDist(const double* Bloc, double* Xloc, int where, const double* T, double* S) {
  needDevice();
  needComm();
  if (!computed_) throw Error(HYMLS_B200_ERR_STATE, "The preconditioner has not yet been computed.");
  const int bm = T ? borderM_ : 0;  // no border set: m = 0, S has no entries and is not written
  if (comm_.size() <= 1) {
    if (bm) applyInverseBordered(Bloc, n_, T, Xloc, n_, S, 1, where);
    else applyInverse(Bloc, n_, Xloc, n_, 1, where);
    return;
  }
  DistPlan& D = levels_[0]->dist;
  if (!D.ready) throw Error(HYMLS_B200_ERR_STATE, "apply_inverse_dist: no distributed plan (Number of Levels = 0?)");
  cudaStream_t s = stream_;
  const int64_t ld = (D.maxOwn + 7) & ~(int64_t)7;
  bufB_.alloc(n_);
  bufX_.alloc(n_);
  bufG_.alloc(2 * ld);
  double* cB = bufG_.p;
  double* cX = bufG_.p + ld;
  const auto in = where == HYMLS_B200_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
  const auto out = where == HYMLS_B200_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost;
  HY_CUDA(cudaMemcpyAsync(cB, Bloc, D.nOwn * sizeof(double), in, s));
  scatterVec(cB, D.ownRows.p, bufB_.p, D.nOwn, s, &launches_);
  if (bm) HY_CUDA(cudaMemcpyAsync(bTin_.p, T, bm * sizeof(double), in, s));
  applyOwned(bufB_.p, bufX_.p, bm ? bTin_.p : nullptr);
  packIdx(bufX_.p, D.ownRows.p, cX, D.nOwn, s, &launches_);
  HY_CUDA(cudaMemcpyAsync(Xloc, cX, D.nOwn * sizeof(double), out, s));
  if (bm) HY_CUDA(cudaMemcpyAsync(S, bS_.p, bm * sizeof(double), out, s));
  if (where == HYMLS_B200_HOST) HY_CUDA(cudaStreamSynchronize(s));
}

void Engine::applyOwned(const double* Bglobal, double* Xglobal, const double* dT) {
  if (comm_.size() <= 1) {
    applyDevice(Bglobal, Xglobal, dT, nullptr);  // (S stays in bS_)
    return;
  }
  if (useDist()) {
    applyLevel0Dist(Bglobal, Xglobal, dT);
  } else {  // fallback path (HYMLS_B200_DIST=0, Number of Levels = 0) works on replicated vectors
    bufD_.alloc(n_);
    gatherOwned(Bglobal, bufD_.p);
    applyLevel(0, bufD_.p, Xglobal, dT);
  }
  stats_.num_apply_inverse++;
}

void Engine::applyMatrix(const double* x, double* y, int where) {
  needDevice();
  if (!haveMatrix_) throw Error(HYMLS_B200_ERR_STATE, "no matrix set");
  Level& L0 = *levels_[0];
  if (where == HYMLS_B200_DEVICE) {
    spmv(L0.rowptr.p, L0.colidx.p, L0.val.p, x, y, n_, 0.0, nullptr, nullptr, 1.0, stream_, &launches_);
  } else {
    bufB_.alloc(n_);
    bufX_.alloc(n_);
    HY_CUDA(cudaMemcpyAsync(bufB_.p, x, n_ * sizeof(double), cudaMemcpyHostToDevice, stream_));
    spmv(L0.rowptr.p, L0.colidx.p, L0.val.p, bufB_.p, bufX_.p, n_, 0.0, nullptr, nullptr, 1.0, stream_, &launches_);
    HY_CUDA(cudaMemcpyAsync(y, bufX_.p, n_ * sizeof(double), cudaMemcpyDeviceToHost, stream_));
    HY_CUDA(cudaStreamSynchronize(stream_));
  }
}

void Engine::timeApply(int reps, double* msApply, double* msA11) {
  needDevice();
  needComm();
  if (!computed_) throw Error(HYMLS_B200_ERR_STATE, "The preconditioner has not yet been computed.");
  bufB_.alloc(n_);
  bufX_.alloc(n_);
  std::vector<double> h(n_);
  std::mt19937_64 rng(7);
  for (auto& v : h) v = (double)(rng() >> 11) * (1.0 / 9007199254740992.0) * 2.0 - 1.0;
  HY_CUDA(cudaMemcpyAsync(bufB_.p, h.data(), n_ * sizeof(double), cudaMemcpyHostToDevice, stream_));
  // sharded: the distributed-vector apply (what the Krylov loop calls), every rank on the rows it owns
  const bool dist = useDist();
  auto applyOnce = [&]() {
    if (dist) {
      applyLevel0Dist(bufB_.p, bufX_.p);
      stats_.num_apply_inverse++;
    } else {
      applyDevice(bufB_.p, bufX_.p);
    }
  };
  for (int i = 0; i < 3; ++i) applyOnce();
  HY_CUDA(cudaStreamSynchronize(stream_));
  HY_CUDA(cudaEventRecord(ev0_, stream_));
  for (int i = 0; i < reps; ++i) applyOnce();
  HY_CUDA(cudaEventRecord(ev1_, stream_));
  HY_CUDA(cudaStreamSynchronize(stream_));
  float ms = 0;
  HY_CUDA(cudaEventElapsedTime(&ms, ev0_, ev1_));
  if (msApply) *msApply = ms / reps;
  // second loop with per-launch events around the A11 kernel (serialises the stream: not used for msApply)
  timeA11_ = true;
  a11Ms_ = 0;
  a11LeadMs_ = 0;
  a11Launches_ = 0;
  for (int i = 0; i < reps; ++i) applyOnce();
  HY_CUDA(cudaStreamSynchronize(stream_));
  timeA11_ = false;
  if (msA11) *msA11 = a11Launches_ ? a11Ms_ / a11Launches_ : 0.0;
  stats_.ms_a11_lead = a11Launches_ ? a11LeadMs_ / a11Launches_ : 0.0;
}

void Engine::operatorRows(const double* full, double* out, int64_t r0, int64_t r1) {
  Level& L0 = *levels_[0];
  cudaStream_t s = stream_;
  const int64_t a0 = std::min(r0, n_), a1 = std::min(r1, n_);
  spmv(L0.rowptr.p + a0, L0.colidx.p, L0.val.p, full, out, a1 - a0, 0.0, nullptr, nullptr, 1.0, s, &launches_);
  const int bm = borderM_;
  if (!bm) return;
  // BorderedOperator::Apply (src/HYMLS_BorderedOperator.cpp:99-140): Y = K X + V S ; T = W' X + C S
  multiAxpy(L0.bV.p + a0, n_, bm, full + n_, out, a1 - a0, 1.0, s, &launches_);
  if (r1 > n_) {
    multiDot(L0.bW.p, n_, bm, full, n_, bPartial_.p, bDots_.p, 0, s, &launches_);
    const int i0 = (int)(std::max(r0, n_) - n_), i1 = (int)(r1 - n_);
    borderRows(bDots_.p, bC0_.p, full + n_, bm, i0, i1, out + (n_ + i0 - r0), s, &launches_);
  }
}

// test hook: copies a device array to the host (doubles). Returns its length.
int64_t Engine::debugCopy(int level, const std::string& name, double* out, int64_t cap) {
  if (name.rfind("pipe_", 0) == 0) {  // schedule of the pipelined host-buffer ApplyInverse (host data, no device needed)
    const HostPipePlan& P = pipePlan_;
    std::vector<double> v;
    if (name == "pipe_matstart") v.assign(P.matStart.begin(), P.matStart.end());
    else if (name == "pipe_leaditem") v.assign(P.leadItem.begin(), P.leadItem.end());
    else if (name == "pipe_fullitem") v.assign(P.fullItem.begin(), P.fullItem.end());
    else if (name == "pipe_inrows") v.assign(P.inRows.begin(), P.inRows.end());
    else if (name == "pipe_outrows") v.assign(P.outRows.begin(), P.outRows.end());
    else throw Error(HYMLS_B200_ERR_ARG, "debug_copy: unknown array '" + name + "'");
    if (out && cap >= (int64_t)v.size()) std::copy(v.begin(), v.end(), out);
    return (int64_t)v.size();
  }
  needDevice();
  Level& L = *levels_.at(level);
  const double* p = nullptr;
  int64_t n = 0;
  if (name == "a11inv") { p = L.a11.F.p; n = (int64_t)L.a11.F.n; }
  else if (name == "blkinv") { p = L.blk.F.p; n = (int64_t)L.blk.F.n; }
  else if (name == "coarseinv") { p = coarse_.F.p; n = (int64_t)coarse_.F.n; }
  else if (name == "redval") {
    if (level + 1 < (int)levels_.size()) { p = levels_[level + 1]->val.p; n = (int64_t)levels_[level + 1]->val.n; }
    else { p = L.redValLast.p; n = (int64_t)L.redValLast.n; }
  }
  else if (name == "v12") { p = L.v12.p; n = (int64_t)L.v12.n; }
  else if (name == "v21") { p = L.v21.p; n = (int64_t)L.v21.n; }
  else if (name == "what") { p = L.what.p; n = (int64_t)L.what.n; }
  else if (name == "redptr" || name == "redcol" || name == "a11off" || name == "blkoff" || name == "blkrows" ||
           name == "introw" || name == "seprow") {
    const LevelSym& S = L.sym;
    std::vector<double> v;
    if (name == "redptr") v.assign(S.redPtr.begin(), S.redPtr.end());
    else if (name == "redcol") v.assign(S.redCol.begin(), S.redCol.end());
    else if (name == "a11off") v.assign(S.a11Off.begin(), S.a11Off.end());
    else if (name == "blkoff") v.assign(S.blkOff.begin(), S.blkOff.end());
    else if (name == "introw") v.assign(S.intRow.begin(), S.intRow.end());
    else if (name == "seprow") v.assign(S.sepRow.begin(), S.sepRow.end());
    else v.assign(S.blkRows.begin(), S.blkRows.end());
    if (out && cap >= (int64_t)v.size()) std::copy(v.begin(), v.end(), out);
    return (int64_t)v.size();
  }
  else throw Error(HYMLS_B200_ERR_ARG, "debug_copy: unknown array '" + name + "'");
  if (out && cap >= n && n > 0) {
    HY_CUDA(cudaMemcpyAsync(out, p, n * sizeof(double), cudaMemcpyDeviceToHost, stream_));
    HY_CUDA(cudaStreamSynchronize(stream_));
  }
  return n;
}

void Engine::getStats(hymls_b200_stats* st) {
  *st = stats_;
  st->kernel_launches = launches_;
  if (!levels_.empty() && initialized_) {
    const LevelSym& S = levels_[0]->sym;
    st->n = S.n;
    st->num_interior = S.nI;
    st->num_separator = S.nS;
    st->num_vsum = S.nuniq;
    st->num_subdomains = S.nsd;
    st->num_blocks = S.nblk;
    st->sum_nsd_sq = S.sumNsq;
    st->sum_nsd_nb = S.sumNNb;
    st->interior_couplings = 0;
    for (auto& lp : levels_) st->interior_couplings += lp->sym.ignoredInteriorCouplings;
    {
      double own = 0, ownLead = 0;
      for (int sd : levels_[0]->ownSd) {
        own += (double)S.sdN[sd] * S.sdN[sd];
        ownLead += (double)S.sdN[sd] * S.sdNb[sd];
      }
      st->a11_split = splitActive(*levels_[0], 0) ? 1 : 0;
      st->host_pipeline_chunks = pipePlan_.K;
      st->host_pipeline_state = pipeEnabled_ ? pipeState_ : -2;
      st->bytes_a11_full_pass = 8.0 * (st->a11_split ? ownLead : own);  // this rank's share when sharded
      st->bytes_a11_level0 = 8.0 * (own + ownLead);
    }
    // SURVEY 8(d): algorithmic bytes of one ApplyInverse, summed over the levels; the A11 term is
    // 8 (sum n^2 + sum n nb) since the first solve needs only the leading nb rows of every inverse
    double bytes = 0;
    for (auto& lp : levels_) {
      const LevelSym& T = lp->sym;
      double sb = 0;
      for (int b = 0; b < T.nblk; ++b) sb += 8.0 * (double)T.blkN[b] * T.blkN[b];
      bytes += 8.0 * (T.sumNsq + T.sumNNb) + 12.0 * (double)(lp->nnz12 + lp->nnz21) +
               4.0 * (double)(T.nI + T.nS + 2) + sb + 2.0 * 12.0 * (double)T.nS * 2.0 + 8.0 * (10.0 * T.nI + 14.0 * T.nS);
    }
    if (coarseBT_.active) {
      for (int b = 0; b < coarseBT_.m; ++b) bytes += 2.0 * 8.0 * (double)coarseBT_.inv.hN[b] * coarseBT_.inv.hN[b];
    } else {
      bytes += 8.0 * (double)coarseN_ * coarseN_;
    }
    st->bytes_apply = bytes;
  }
  st->collective_calls = comm_.calls();
  st->collective_bytes = comm_.bytes();
}

}  // namespace hymls

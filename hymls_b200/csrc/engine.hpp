// Device-side engine: numeric Compute / ApplyInverse of all levels and the Krylov driver.
#pragma once
#include <memory>
#include <string>
#include <vector>

#include "comm.hpp"
#include "device.cuh"
#include "kernels.hpp"
#include "symbolic.hpp"

namespace hymls {

struct BatchedInverse {  // a set of dense inverses + the GEMV work list over them
  DevBuf<double> F;
  DevBuf<int> n, np, itemMat, itemRow0;
  DevBuf<int64_t> matOff, vecOff;
  std::vector<int> hN, hNp;
  std::vector<int64_t> hMatOff, hVecOff;
  int count = 0, numItems = 0, npMax = 0;
  int smallSplit = 0;   // > 0: matrices with np <= smallSplit get no slab items but are listed in matList
  DevBuf<int> matList;  // (flagged) matrices of at most smallSplit rows, for the warp-per-matrix kernel
  int numMats = 0;
  int midSplit = 0;     // > 0: matrices with smallSplit < np <= midSplit are listed in midList (CTA-per-matrix kernel)
  DevBuf<int> midList;
  int numMid = 0, midNpMax = 0;
  // second work list over the leading `leadRows[m]` rows of every matrix (first solve of ApplyInverse)
  DevBuf<int> rowLimit, itemMatLead, itemRow0Lead;
  int numItemsLead = 0;
  std::vector<int> hItemPtr, hItemPtrLead;  // count+1: first work item of every matrix in itemMat / itemMatLead
  // third work list: the remaining rows [leadRows[m], n) (computed off the critical path, see Engine::applyLevel)
  DevBuf<int> itemMatTrail, itemRow0Trail;
  int numItemsTrail = 0;
  // `applyMask` (optional, one flag per matrix): GEMV work items are created for flagged matrices only
  int rowsPerWarp = 0;  // thinner GEMV slabs (see GemvArgs::rowsPerWarp); set before setup()
  void setup(const std::vector<int>& n_, const std::vector<int>& np_, const std::vector<int64_t>& matOff_,
             const std::vector<int64_t>& vecOff_, cudaStream_t s, const std::vector<char>* applyMask = nullptr,
             const std::vector<int>* leadRows = nullptr);
  GemvArgs args() const;
};

// one sparse neighbour exchange (grouped ncclSend / ncclRecv): positions to pack per peer, positions to unpack
struct Halo {
  std::vector<int> peers;                 // ranks exchanged with, ascending
  std::vector<int64_t> sendPtr, recvPtr;  // peers+1: ranges of the packed buffers
  DevBuf<int> sendIdx, recvIdx;
  DevBuf<double> sendBuf, recvBuf;
};

// Owner-computes plan of a sharded level 0 (dist.cu): every rank works on the interiors of its subdomains and on
// the separator groups it owns; only separator values on the interfaces between ranks are exchanged.
struct DistPlan {
  bool ready = false, matReady = false;
  Halo rev;   // partial sums of A21 x1 at the ghost separators -> their owners
  Halo fwd;   // x2 of owned separators -> the ranks whose subdomains touch them
  Halo mat;   // columns of the owned matrix rows that other ranks own (operator apply of the Krylov loop)
  DevBuf<int> addNode;                    // owned separators receiving partial sums, with their sources in
  DevBuf<int64_t> addPtr, addSrc;         // rev.recvBuf in rank order (deterministic sum)
  int64_t nAdd = 0;
  DevBuf<int> rows21, rows12, ownUniq, ownSepPos, ownRows, allRows;
  int64_t nRows21 = 0, nRows12 = 0, nOwnUniq = 0, nOwnSep = 0, nOwn = 0, maxOwn = 0;
  std::vector<int> hOwnRows;              // matrix rows this rank owns, ascending
  std::vector<int> rowOwner;              // owner rank of every matrix row
  DevBuf<double> gath;                    // nranks * maxOwn: all-gather target for replicated output
};

struct Level {
  DeviceArena arena;  // owns the index arrays uploaded by Initialize (declared first: destroyed last)
  LevelSym sym;
  DistPlan dist;
  bool exact = false;  // Number of Levels == 0: dense Schur complement instead of transform + drop
  // matrix of this level
  DevBuf<int64_t> rowptr;
  DevBuf<int> colidx;
  DevBuf<double> val;
  // orderings
  DevBuf<int> intRow, sepRow;
  DevBuf<int> rowPos;  // per row: interior position (>= 0) or -(separator position) - 1
  DevBuf<int> posMat;  // per interior position: owned matrix (index into a11) or -1
  DevBuf<int64_t> intPtrG;  // per (global) subdomain: first interior position, nsd+1
  int64_t nnz12 = 0, nnz21 = 0, nnz22 = 0, nnzS21 = 0;  // entries of the device-built index arrays
  // A11: inverses of the subdomains this rank owns (all of them on one GPU), compact storage
  BatchedInverse a11;
  std::vector<int> ownSd;           // owned subdomains, ascending
  std::vector<int> sdRank;          // owner rank of every subdomain (sharded levels)
  std::vector<int64_t> ownOff;      // compact offsets (doubles) of the owned matrices, ownSd.size()+1
  DevBuf<int> sdNG, sdNpG;          // per (global) subdomain: n, np
  DevBuf<int64_t> a11OffG;          // per (global) subdomain: compact offset (undefined if not owned)
  DevBuf<int64_t> a11Src, a11Dst;
  std::vector<int64_t> a11ListPtr;  // per owned sd: range of the scatter list
  DevBuf<int64_t> a11ListPtrDev;
  bool sharded = false;
  bool repSep = false;              // sharded coarser level: subdomain solves distributed, separator side replicated
  DevBuf<int> ownSdList;            // device copies of the owned lists for the pass-2 Schur kernels
  DevBuf<int64_t> ownRowList, ownLinkList;
  std::vector<int64_t> chunkOwnSd, chunkOwnRow, chunkOwnLink;  // per chunk: ranges in the lists (nchunks+1)
  // Deterministic pass-2 assembly: (owned) subdomains coloured so that two subdomains of one colour share no
  // separator group; per (chunk, colour) lists of subdomains / linked sets (/ local rows, exact path only)
  int ncolors = 0;
  DevBuf<int> colSd;
  DevBuf<int64_t> colLk, colRow;
  std::vector<int64_t> colSdPtr, colLkPtr, colRowPtr;  // nchunks * ncolors + 1
  DevBuf<double> xI;                // per-rank packed interior results, all-gathered (nranks * maxOwnI)
  DevBuf<int64_t> gatherOutOff;     // per owned matrix: position of its segment in xI
  DevBuf<int> packedRow;            // matrix row of every xI entry (-1: padding)
  int64_t maxOwnI = 0;
  // off-diagonal blocks
  DevBuf<int64_t> p12, p21, src12, src21, p22, src22;
  DevBuf<int> c12, c21, c22;
  DevBuf<double> v12, v21;
  // Schur assembly index data
  DevBuf<int> rowSd, rowInst, rowLinkPos, sdSep, sdM;
  DevBuf<int64_t> sdRowPtr, s21Ptr, s12Ptr, s22Ptr, s21Src, s12Src, s22Src;
  DevBuf<int> s21Col, s12Row, s22Col;
  DevBuf<int64_t> sdInstPtr, sdLinkPtr, lnkOff, wsOffC, wsOffD, wsOffA, wsOffS;
  DevBuf<int> instLoc, instLen, instUniq, instLink, lnkSd, lnkSize;
  DevBuf<int> uniqStart, uniqBlk, uniqBlkOff;
  DevBuf<double> what, wd, usign;
  DevBuf<int64_t> redPtr;
  DevBuf<int> redCol;
  // chunking of the assembly workspace
  struct Chunk { int sd0, sd1; int64_t R0, R1, lk0, lk1; };
  std::vector<Chunk> chunks;
  int64_t wsCLen = 0, wsSLLLen = 0, wsDLen = 0, wsALen = 0, wsSLen = 0;
  std::vector<int64_t> chunkDLen, chunkALen;   // per chunk: doubles of the m x np arrays of the dense Schur path
  int schurGemm = 0;                // dense (DMMA GEMM) Schur rows: 0 off, 1 both products, 2 only A21 A11^-1
  int maxM = 0, maxNp = 0;
  size_t rowSmem = 0, blkSmem = 0;
  int dLen = 0;
  // separator blocks
  BatchedInverse blk;
  DevBuf<int> blkRows;
  // work vectors
  DevBuf<double> x1, y1, rhsS, Z, Y, vsRhs, vsSol;
  DevBuf<double> redValLast;  // reduced Schur values when this is the last level (kept for inspection)
  // bordered variant (BorderedOperator): V, W of this level in its row numbering (n_l x m), Q1 = A11^-1 V1,
  // W1t = A11^-T W1, the transformed separator border sW (V-sum positions zeroed), the border handed to the coarse
  // solver (cV, cW) and the border right-hand sides q (after the interior elimination) / Tc (next level's T)
  DevBuf<double> bV, bW, Q1, W1t, sV, sW, cV, cW, bQ, bT;
  DevBuf<int64_t> t12Ptr, t12Idx;  // transposed index of A12 (rows = separator positions), built at the first
  DevBuf<int> t12Col;              // ComputeBorder: A12' w without atomics
  std::vector<double> hC;     // C of this level (m x m, column major)
};

// the caller's distribution of vectors <-> the owner distribution (boundary.cu)
struct RowMapPlan {
  bool ready = false;
  int64_t nLocal = 0;
  Halo toOwner, fromOwner;
  DevBuf<double> stage;
};
// assembly map of a distributed matrix input (boundary.cu)
struct DistMatrixCache {
  bool ready = false;
  std::vector<int64_t> signature, ptr, slot;
  std::vector<int> col;
};

// block-tridiagonal coarse factorization on BFS level sets (coarse.cu)
struct KrylovLayout;  // the vector layout of one Krylov solve (krylov.cu)

struct CoarseBT {
  bool planned = false, active = false;
  int n = 0, m = 0;
  std::vector<int> lvlPtr, perm, itemPtr;
  std::vector<int64_t> dListPtr;
  BatchedInverse inv;                    // F_i = inv(D_i')
  DevBuf<int> dPerm, loCol, upCol;
  DevBuf<int64_t> dSrc, dDst, loPtr, upPtr, loSrc, upSrc;
  DevBuf<double> loVal, upVal, y, t, r, xp;
};

class Engine {
 public:
  explicit Engine(const std::string& xml);
  ~Engine();
  void setStream(cudaStream_t s) { stream_ = s; }
  void commInit(const void* id128, int rank, int nranks);
  void setRankOnly(int rank, int nranks);
  const std::vector<int>& ownedSubdomains(int level) const { return levels_.at(level)->ownSd; }
  void setMatrix(int64_t n, const int64_t* rowptr, const int32_t* colidx, const double* values, int where);
  void setMatrixDist(int64_t nGlobal, int64_t nLocal, const int64_t* rowGids, const int64_t* rowptr,
                     const int64_t* colGids, const double* values);
  void setRowMap(int64_t nLocal, const int64_t* rowGids);
  void applyInverseMap(const double* B, int64_t ldb, double* X, int64_t ldx, int nvec, int where,
                       const double* T = nullptr, double* S = nullptr);
  void setTestVectorDist(int64_t nLocal, const int64_t* gids, const double* tv);
  void setBorderDist(int64_t nLocal, const int64_t* gids, const double* V, const double* W, const double* C, int m);
  void setParameters(const std::string& xml);
  void setTestVector(const double* tv);
  void initialize();
  void compute();
  void applyInverse(const double* B, int64_t ldb, double* X, int64_t ldx, int nvec, int where);
  void setBorder(const double* V, const double* W, const double* C, int m);
  void applyInverseBordered(const double* B, int64_t ldb, const double* T, double* X, int64_t ldx, double* S, int nvec,
                            int where);
  int borderSize() const { return borderM_; }
  int device() const { return device_; }  // CUDA device the handle is bound to (-1: none)
  void applyMatrix(const double* x, double* y, int where);
  void localRows(int64_t* r0, int64_t* r1) const;
  void applyInverseDist(const double* Bloc, double* Xloc, int where, const double* T = nullptr, double* S = nullptr);
  int64_t ownedRows(int64_t* rows, int64_t cap);
  void solve(const double* b, double* x, int where, uint64_t seed, hymls_b200_solve_info* info, double* hist,
             int histCap);
  void timeApply(int reps, double* msApply, double* msA11);
  void getStats(hymls_b200_stats* st);
  int64_t debugCopy(int level, const std::string& name, double* out, int64_t cap);

  int numLevels() const { return (int)levels_.size(); }
  const LevelSym& sym(int l) const { return levels_.at(l)->sym; }
  ParameterList& params() { return params_; }
  bool initialized() const { return initialized_; }

 private:
  void applyLevel(int l, const double* B, double* X, const double* T = nullptr);  // device pointers
  void blockSolves(Level& L, const double* Z, double* Y);
  void computeLevel(int l);
  void computeBorder(int l);
  std::vector<std::pair<int, int>> a11Chunks(const Level& L) const;
  void reserveComputeScratch();
  size_t inversionWorkspace() const;
  void checkInfo(const std::string& what);
  void computeCoarse(const int64_t* ptr, const int* col, double* val, int n, const std::vector<gidx>& rowGid,
                     const std::vector<int64_t>& hPtr, const std::vector<int>& hCol, const double* bV = nullptr,
                     const double* bW = nullptr, const std::vector<double>* bC = nullptr);
  void coarseSolve(double* rhs, double* sol, int n);  // unbordered coarse solve (zeroes the fixed rows of rhs)
  void planCoarseBT(const std::vector<int64_t>& ptr, const std::vector<int>& col, int n);
  void factorCoarseBT(const int64_t* ptr, const int* col, const double* val);
  void solveCoarseBT(const double* rhs, double* sol);
  CoarseBT coarseBT_;
  void augmentAndInvertCoarse(int n, int np, const double* bV, const double* bW, const std::vector<double>* bC,
                              const char* what);
  void coarseSolveBordered(const double* rhs, const double* T, double* sol, int n);
  void uploadLevel(Level& L);
  void readParameters();
  // global-length vectors with the owned rows valid in, the same out (one rank: the whole vector)
  void applyOwned(const double* Bglobal, double* Xglobal, const double* dT = nullptr);
  RowMapPlan rowMap_;
  DistMatrixCache distMat_;
  // owner-computes multi-GPU path (dist.cu)
  bool useDist() const;
  void buildDistPlan(Level& L);
  void buildMatrixHalo();
  void haloExchange(Halo& h, const double* src, double* dst, bool scatter);
  void applyLevel0Dist(const double* B, double* X, const double* T = nullptr);  // with a border: S -> bS_
  void gatherOwned(const double* Xowned, double* Xfull);
  // Krylov solves on replicated vectors and on the owner distribution (krylov.cu)
  KrylovLayout replicatedLayout(bool left, bool right);
  KrylovLayout ownerLayout(bool left, bool right);
  void applyDevice(const double* dB, double* dX, const double* dT = nullptr, double* dS = nullptr);
  bool applyDeviceMulti(const double* dB, int64_t ldb, double* dX, int64_t ldx, int nv);
  DevBuf<double> x1m_, y1m_;  // interior work vectors of the multi-column apply
  // rows [r0, r1) of the (bordered) operator [K V; W' C] applied to the replicated vector `full`
  void operatorRows(const double* full, double* out, int64_t r0, int64_t r1);

  ParameterList params_;
  Comm comm_;
  cudaStream_t stream_ = 0;
  int maxLevel_ = 1;
  int64_t n_ = 0;
  std::vector<int64_t> hRowptr_;
  std::vector<int> hColidx_;
  std::vector<double> hTestVector_;
  bool haveMatrix_ = false, initialized_ = false, computed_ = false, deviceOk_ = false;
  int device_ = -1;
  void needDevice() const;
  void needComm() const;
  std::vector<std::unique_ptr<Level>> levels_;
  // coarse solver (dense inverse)
  BatchedInverse coarse_;
  std::vector<int> coarseFix_;  // rows with a Dirichlet condition
  int coarseN_ = 0, coarseM_ = 0;
  DevBuf<double> coarseRhs_, coarseSol_;
  // border (SetBorder): host copies of V, W (n x m, column major) and C (m x m)
  int borderM_ = 0;
  std::vector<double> hV_, hW_, hC_;
  DevBuf<double> bS_, bTin_, bPartial_, bDots_, bC_, bC0_;
  // scratch
  std::unique_ptr<DeviceArena> computeArena_;  // one block for the scratch of Compute (declared before its users)
  DevBuf<double> work_;      // inversion workspace
  DevBuf<double> work2_, blkA_, blkR_;  // Newton-Schulz refinement: residuals, copies of the dense originals
  bool refine_ = true;
  DevBuf<int> piv_, perm_, info_, subsetN_, subsetNp_;
  DevBuf<double> wsC_, wsSV_, wsSLL_, diagScratch_, blkW_, red2_, blk2_, a21d_, dmat_, a12d_, skd_;
  DevBuf<int64_t> relOff_;
  DevBuf<double> flag_;
  DevBuf<double> bufB_, bufX_;  // staging for host vectors
  DevBuf<double> bufG_;          // compact staging of the distributed-vector entry point
  DevBuf<double> bufD_;          // global-length scratch of the owner-computes path
  // Krylov workspace
  DevBuf<double> kV_, kW_, kZ_, kH_, kPartial_, kX_, kB_, kR_, kQ_;
  DevBuf<double> kS1_, kS2_;  // scratch of the vector layouts
  int kCap_ = 0;
  // statistics
  hymls_b200_stats stats_{};
  int64_t launches_ = 0;
  cudaEvent_t ev0_ = nullptr, ev1_ = nullptr, evA_ = nullptr, evB_ = nullptr;
  // split second subdomain solve (applyLevel): low-priority side stream + fork / join events
  cudaStream_t side_ = nullptr;
  cudaEvent_t evFork_ = nullptr, evJoin_ = nullptr;
  bool splitSolve_ = false;  // HYMLS_B200_SPLIT_SOLVE=1 enables (measured slower on 1 GPU, see DESIGN.md)
  bool splitActive(const Level& L, int l) const { return splitSolve_ && l == 0 && !L.exact && side_ != nullptr; }
  // Host-buffer ApplyInverse on one GPU (pinned buffers): the H2D copy of b runs beside the leading-rows pass over the
  // level-0 inverses, the D2H copy of x beside the full pass (HostPipePlan, symbolic.hpp).  The first pipelined call
  // is checked bitwise against the serial path and the pipeline is switched off for the handle if they differ.
  HostPipePlan pipePlan_;        // K == 0: none (several ranks, exact level 0, small problem)
  bool pipeEnabled_ = true;      // HYMLS_B200_HOST_PIPELINE=0 switches it off
  int pipeState_ = 0;            // 0: not used yet, 1: verified and in use, -1: self-check failed, serial path from now on
  cudaStream_t pipeCopy_ = nullptr;
  cudaEvent_t pipeStart_ = nullptr;
  std::vector<cudaEvent_t> pipeIn_, pipeOut_;
  double* pipeHostX_ = nullptr;  // host destination of the pipelined call in flight (nullptr: none)
  void planHostPipeline();
  void destroyPipeEvents();
  bool hostPipeUsable(const double* b, const double* x);
  void applyHostPiped(const double* b, double* x);
  bool timeA11_ = false;
  double a11Ms_ = 0, a11LeadMs_ = 0;
  int a11Launches_ = 0;
};

}  // namespace hymls

#include "comm.hpp"

#include <dlfcn.h>

#include <cstdlib>
#include <string>

#include "../../include/hymls_b200.h"
#include "params.hpp"

namespace hymls {

namespace {
typedef struct { char internal[128]; } NcclUniqueId;
typedef int (*GetUniqueIdFn)(NcclUniqueId*);
typedef int (*CommInitRankFn)(void**, int, NcclUniqueId, int);
typedef int (*AllReduceFn)(const void*, void*, size_t, int, int, void*, cudaStream_t);
typedef int (*CommDestroyFn)(void*);
typedef int (*AllGatherFn)(const void*, void*, size_t, int, void*, cudaStream_t);
typedef int (*BroadcastFn)(const void*, void*, size_t, int, int, void*, cudaStream_t);
typedef const char* (*GetErrorStringFn)(int);
typedef int (*SendFn)(const void*, size_t, int, int, void*, cudaStream_t);
typedef int (*RecvFn)(void*, size_t, int, int, void*, cudaStream_t);
typedef int (*GroupFn)(void);

struct Api {
  void* lib = nullptr;
  GetUniqueIdFn getUniqueId = nullptr;
  CommInitRankFn commInitRank = nullptr;
  AllReduceFn allReduce = nullptr;
  CommDestroyFn commDestroy = nullptr;
  BroadcastFn broadcast = nullptr;
  AllGatherFn allGather = nullptr;
  GetErrorStringFn errorString = nullptr;
  SendFn send = nullptr;
  RecvFn recv = nullptr;
  GroupFn groupStart = nullptr, groupEnd = nullptr;
};

Api& api() {
  static Api a;
  if (a.lib) return a;
  const char* names[] = {"libnccl.so.2", "libnccl.so"};
  for (const char* n : names) {
    a.lib = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
    if (a.lib) break;
  }
  if (!a.lib) throw Error(HYMLS_B200_ERR_CUDA, std::string("cannot load NCCL (libnccl.so.2): ") + dlerror());
  a.getUniqueId = (GetUniqueIdFn)dlsym(a.lib, "ncclGetUniqueId");
  a.commInitRank = (CommInitRankFn)dlsym(a.lib, "ncclCommInitRank");
  a.allReduce = (AllReduceFn)dlsym(a.lib, "ncclAllReduce");
  a.commDestroy = (CommDestroyFn)dlsym(a.lib, "ncclCommDestroy");
  a.broadcast = (BroadcastFn)dlsym(a.lib, "ncclBroadcast");
  a.allGather = (AllGatherFn)dlsym(a.lib, "ncclAllGather");
  a.errorString = (GetErrorStringFn)dlsym(a.lib, "ncclGetErrorString");
  a.send = (SendFn)dlsym(a.lib, "ncclSend");
  a.recv = (RecvFn)dlsym(a.lib, "ncclRecv");
  a.groupStart = (GroupFn)dlsym(a.lib, "ncclGroupStart");
  a.groupEnd = (GroupFn)dlsym(a.lib, "ncclGroupEnd");
  if (!a.getUniqueId || !a.commInitRank || !a.allReduce || !a.commDestroy || !a.broadcast || !a.allGather ||
      !a.send || !a.recv || !a.groupStart || !a.groupEnd)
    throw Error(HYMLS_B200_ERR_CUDA, "NCCL library lacks the expected symbols");
  return a;
}

void check(int rc, const char* what) {
  if (rc != 0) {
    Api& a = api();
    throw Error(HYMLS_B200_ERR_CUDA,
                std::string("NCCL error in ") + what + ": " + (a.errorString ? a.errorString(rc) : "?"));
  }
}
}  // namespace

Comm::~Comm() {
  if (comm_) api().commDestroy(comm_);
}

void Comm::uniqueId(void* id128) { check(api().getUniqueId((NcclUniqueId*)id128), "ncclGetUniqueId"); }

void Comm::init(const void* id128, int rank, int nranks) {
  NcclUniqueId id = *(const NcclUniqueId*)id128;
  check(api().commInitRank(&comm_, nranks, id, rank), "ncclCommInitRank");
  rank_ = rank;
  nranks_ = nranks;
  // NCCL builds its rings and the peer-to-peer connections lazily, on the first collective / the first send to a
  // peer (measured: ~1 s inside the first GMRES solve on 8 GPUs, whose operator halo met 7 new peers).  Creating the
  // communicator is the place for that: one collective of each kind and one message between every pair.
  if (nranks > 1 && !getenv("HYMLS_B200_NO_COMM_WARMUP")) {
    // (1 MB per pair rather than 8 bytes: NCCL connects the channels an operation needs, larger messages use more)
    const size_t msg = (size_t)1 << 17;
    const size_t total = 2 + (size_t)nranks + 2 * (size_t)nranks * msg;
    double* buf = nullptr;
    if (cudaMalloc((void**)&buf, sizeof(double) * total) != cudaSuccess)
      throw Error(HYMLS_B200_ERR_CUDA, "cudaMalloc failed in the communicator warm-up");
    cudaMemset(buf, 0, sizeof(double) * total);
    const int ncclDouble = 8, ncclSum = 0;
    cudaStream_t s = 0;
    double* sendBase = buf + 2 + nranks;
    double* recvBase = sendBase + (size_t)nranks * msg;
    check(api().allReduce(sendBase, sendBase, msg, ncclDouble, ncclSum, comm_, s), "ncclAllReduce (warm-up)");
    check(api().broadcast(buf, buf, 1, ncclDouble, 0, comm_, s), "ncclBroadcast (warm-up)");
    check(api().allGather(buf + 1, buf + 2, 1, ncclDouble, comm_, s), "ncclAllGather (warm-up)");
    check(api().groupStart(), "ncclGroupStart (warm-up)");
    for (int q = 0; q < nranks; ++q) {
      if (q == rank) continue;
      check(api().send(sendBase + (size_t)q * msg, msg, ncclDouble, q, comm_, s), "ncclSend (warm-up)");
      check(api().recv(recvBase + (size_t)q * msg, msg, ncclDouble, q, comm_, s), "ncclRecv (warm-up)");
    }
    check(api().groupEnd(), "ncclGroupEnd (warm-up)");
    cudaStreamSynchronize(s);
    cudaFree(buf);
  }
}

void Comm::allReduceSum(double* buf, size_t count, cudaStream_t s) const {
  if (!comm_ || count == 0) return;
  const int ncclDouble = 8, ncclSum = 0;  // ncclFloat64, ncclSum (nccl.h enums, stable across 2.x)
  static const bool syncEach = getenv("HYMLS_B200_SYNC_NCCL") != nullptr;
  if (syncEach) cudaStreamSynchronize(s);
  tally(count);
  check(api().allReduce(buf, buf, count, ncclDouble, ncclSum, comm_, s), "ncclAllReduce");
  if (syncEach) cudaStreamSynchronize(s);
}

}  // namespace hymls

namespace hymls {
void Comm::allGather(const double* send, double* recv, size_t count, cudaStream_t s) const {
  if (!comm_ || count == 0) return;
  const int ncclDouble = 8;
  tally(count);
  check(api().allGather(send, recv, count, ncclDouble, comm_, s), "ncclAllGather");
}
void Comm::broadcast(double* buf, size_t count, int root, cudaStream_t s) const {
  if (!comm_ || count == 0) return;
  const int ncclDouble = 8;
  tally(count);
  check(api().broadcast(buf, buf, count, ncclDouble, root, comm_, s), "ncclBroadcast");
}
}  // namespace hymls

namespace hymls {
// One grouped neighbour exchange (the halo Import/Export of Epetra_CrsMatrix::Apply): for every peer k the range
// [sendPtr[k], sendPtr[k+1]) of sendBuf goes to peers[k] and [recvPtr[k], recvPtr[k+1]) of recvBuf comes from it.
void Comm::neighbourExchange(const std::vector<int>& peers, const double* sendBuf, const std::vector<int64_t>& sendPtr,
                             double* recvBuf, const std::vector<int64_t>& recvPtr, cudaStream_t s) const {
  if (peers.empty()) return;
  // the part a rank "sends to itself" is a device copy (also the whole exchange of a single-rank run)
  bool others = false;
  for (size_t k = 0; k < peers.size(); ++k) {
    if (peers[k] != rank_) { others = true; continue; }
    const size_t ns = (size_t)(sendPtr[k + 1] - sendPtr[k]);
    if (ns) cudaMemcpyAsync(recvBuf + recvPtr[k], sendBuf + sendPtr[k], ns * sizeof(double), cudaMemcpyDeviceToDevice, s);
  }
  if (!comm_ || !others) return;
  const int ncclDouble = 8;
  size_t moved = 0;
  for (size_t k = 0; k < peers.size(); ++k)
    if (peers[k] != rank_) moved += (size_t)(sendPtr[k + 1] - sendPtr[k] + recvPtr[k + 1] - recvPtr[k]);
  tally(moved);
  Api& a = api();
  check(a.groupStart(), "ncclGroupStart");
  for (size_t k = 0; k < peers.size(); ++k) {
    if (peers[k] == rank_) continue;
    const size_t ns = (size_t)(sendPtr[k + 1] - sendPtr[k]), nr = (size_t)(recvPtr[k + 1] - recvPtr[k]);
    if (ns) check(a.send(sendBuf + sendPtr[k], ns, ncclDouble, peers[k], comm_, s), "ncclSend");
    if (nr) check(a.recv(recvBuf + recvPtr[k], nr, ncclDouble, peers[k], comm_, s), "ncclRecv");
  }
  check(a.groupEnd(), "ncclGroupEnd");
}
}  // namespace hymls

// Thin NCCL shim: the library is dlopen'ed on first use so that single-GPU use and the CPU-side tests
// need no NCCL at all, and so that a process that already loaded torch's bundled NCCL shares it.
// Replaces the Epetra/MPI collectives of the reference on this path (SumAll / Import / Export,
// SURVEY 5 "Distributed communication backend").
#pragma once
#include <cuda_runtime.h>

#include <cstddef>
#include <cstdint>
#include <vector>

namespace hymls {

class Comm {
 public:
  Comm() {}
  ~Comm();
  static void uniqueId(void* id128);                       // ncclGetUniqueId (128 bytes)
  void init(const void* id128, int rank, int nranks);      // ncclCommInitRank (collective)
  void setRankOnly(int rank, int nranks) { rank_ = rank; nranks_ = nranks; }  // host logic without NCCL
  int rank() const { return rank_; }
  int size() const { return nranks_; }
  bool active() const { return comm_ != nullptr; }
  void allReduceSum(double* buf, size_t count, cudaStream_t s) const;  // in place
  void broadcast(double* buf, size_t count, int root, cudaStream_t s) const;  // in place
  // recv[rank * count + i] = send_rank[i]; recv may alias send at offset rank*count
  void allGather(const double* send, double* recv, size_t count, cudaStream_t s) const;
  // grouped ncclSend / ncclRecv with a set of neighbour ranks (halo exchange)
  void neighbourExchange(const std::vector<int>& peers, const double* sendBuf, const std::vector<int64_t>& sendPtr,
                         double* recvBuf, const std::vector<int64_t>& recvPtr, cudaStream_t s) const;
  // this rank's collective calls and their payload bytes since init (all-reduce / broadcast / all-gather: the count
  // of one rank; neighbour exchange: sent + received to / from other ranks).  The warm-up of init is not counted.
  int64_t calls() const { return calls_; }
  int64_t bytes() const { return bytes_; }

 private:
  void* comm_ = nullptr;
  int rank_ = 0, nranks_ = 1;
  mutable int64_t calls_ = 0, bytes_ = 0;
  void tally(size_t doubles) const { calls_++; bytes_ += (int64_t)(doubles * sizeof(double)); }
};

}  // namespace hymls

// C ABI (include/hymls_b200.h) -> Engine.  No exception crosses the boundary.
#include <cstring>
#include <memory>
#include <string>

#include "../../include/hymls_b200.h"
#include "engine.hpp"

using namespace hymls;

struct hymls_b200 {
  Engine* eng;
};

static thread_local std::string g_lastError;

#define HY_TRY try {
#define HY_CATCH                                   \
  }                                                \
  catch (const hymls::Error& e) {                  \
    g_lastError = e.what();                        \
    return e.code;                                 \
  }                                                \
  catch (const std::exception& e) {                \
    g_lastError = e.what();                        \
    return HYMLS_B200_ERR_ARG;                     \
  }                                                \
  catch (...) {                                    \
    g_lastError = "unknown exception";             \
    return HYMLS_B200_ERR_ARG;                     \
  }

extern "C" {

const char* hymls_b200_last_error(void) { return g_lastError.c_str(); }

const char* hymls_b200_version(void) {
  static std::string v;
  v = "hymls_b200 0.1 (sm_100a)";
  int dev = 0;
  cudaDeviceProp p;
  if (cudaGetDevice(&dev) != cudaSuccess || cudaGetDeviceProperties(&p, dev) != cudaSuccess) return nullptr;
  v += std::string(" on ") + p.name;
  return v.c_str();
}

int hymls_b200_create(const char* xml, hymls_b200_t** out) {
  HY_TRY
  if (!xml || !out) throw Error(HYMLS_B200_ERR_ARG, "create: null argument");
  *out = nullptr;
  Engine* e = new Engine(xml);
  *out = new hymls_b200{e};
  return 0;
  HY_CATCH
}

void hymls_b200_destroy(hymls_b200_t* h) {
  if (!h) return;
  delete h->eng;
  delete h;
}

int hymls_b200_set_stream(hymls_b200_t* h, void* s) {
  HY_TRY
  h->eng->setStream((cudaStream_t)s);
  return 0;
  HY_CATCH
}

int hymls_b200_comm_get_unique_id(void* id128) {
  HY_TRY
  if (!id128) throw Error(HYMLS_B200_ERR_ARG, "null id");
  Comm::uniqueId(id128);
  return 0;
  HY_CATCH
}

int hymls_b200_comm_init(hymls_b200_t* h, const void* id128, int rank, int nranks) {
  HY_TRY
  h->eng->commInit(id128, rank, nranks);
  return 0;
  HY_CATCH
}

int hymls_b200_set_rank(hymls_b200_t* h, int rank, int nranks) {
  HY_TRY
  h->eng->setRankOnly(rank, nranks);
  return 0;
  HY_CATCH
}

int hymls_b200_get_owned_subdomains(hymls_b200_t* h, int level, int32_t* sd, int cap) {
  HY_TRY
  if (!h->eng->initialized()) throw Error(HYMLS_B200_ERR_STATE, "not initialized");
  const std::vector<int>& v = h->eng->ownedSubdomains(level);
  if (sd && !v.empty() && cap >= (int)v.size()) std::memcpy(sd, v.data(), v.size() * sizeof(int));
  return (int)v.size();
  HY_CATCH
}

int hymls_b200_set_matrix_csr(hymls_b200_t* h, int64_t n, const int64_t* rowptr, const int32_t* colidx,
                              const double* values, int where) {
  HY_TRY
  h->eng->setMatrix(n, rowptr, colidx, values, where);
  return 0;
  HY_CATCH
}

int hymls_b200_set_matrix_csr_dist(hymls_b200_t* h, int64_t n_global, int64_t n_local, const int64_t* row_gids,
                                   const int64_t* rowptr, const int64_t* col_gids, const double* values) {
  HY_TRY
  h->eng->setMatrixDist(n_global, n_local, row_gids, rowptr, col_gids, values);
  return 0;
  HY_CATCH
}

int hymls_b200_set_parameters(hymls_b200_t* h, const char* xml) {
  HY_TRY
  if (!xml) throw Error(HYMLS_B200_ERR_ARG, "set_parameters: null argument");
  h->eng->setParameters(xml);
  return 0;
  HY_CATCH
}

int hymls_b200_set_row_map(hymls_b200_t* h, int64_t n_local, const int64_t* row_gids) {
  HY_TRY
  h->eng->setRowMap(n_local, row_gids);
  return 0;
  HY_CATCH
}

int hymls_b200_apply_inverse_map(hymls_b200_t* h, const double* B, int64_t ldb, double* X, int64_t ldx, int nvec,
                                 int where) {
  HY_TRY
  h->eng->applyInverseMap(B, ldb, X, ldx, nvec, where);
  return 0;
  HY_CATCH
}

int hymls_b200_apply_inverse_bordered_map(hymls_b200_t* h, const double* B, int64_t ldb, const double* T, double* X,
                                          int64_t ldx, double* S, int nvec, int where) {
  HY_TRY
  if (!T || !S) throw Error(HYMLS_B200_ERR_ARG, "apply_inverse_bordered_map: T and S are required");
  h->eng->applyInverseMap(B, ldb, X, ldx, nvec, where, T, S);
  return 0;
  HY_CATCH
}

int hymls_b200_set_testvector_dist(hymls_b200_t* h, int64_t n_local, const int64_t* row_gids, const double* tv) {
  HY_TRY
  h->eng->setTestVectorDist(n_local, row_gids, tv);
  return 0;
  HY_CATCH
}

int hymls_b200_set_border_dist(hymls_b200_t* h, int64_t n_local, const int64_t* row_gids, const double* V,
                               const double* W, const double* C, int m) {
  HY_TRY
  h->eng->setBorderDist(n_local, row_gids, V, W, C, m);
  return 0;
  HY_CATCH
}

int hymls_b200_set_testvector(hymls_b200_t* h, const double* tv) {
  HY_TRY
  h->eng->setTestVector(tv);
  return 0;
  HY_CATCH
}

int hymls_b200_initialize(hymls_b200_t* h) {
  HY_TRY
  h->eng->initialize();
  return 0;
  HY_CATCH
}

int hymls_b200_compute(hymls_b200_t* h) {
  HY_TRY
  h->eng->compute();
  return 0;
  HY_CATCH
}

int hymls_b200_apply_inverse(hymls_b200_t* h, const double* B, int64_t ldb, double* X, int64_t ldx, int nvec,
                             int where) {
  HY_TRY
  h->eng->applyInverse(B, ldb, X, ldx, nvec, where);
  return 0;
  HY_CATCH
}

int hymls_b200_local_rows(hymls_b200_t* h, int64_t* r0, int64_t* r1) {
  HY_TRY
  if (!r0 || !r1) throw Error(HYMLS_B200_ERR_ARG, "null argument");
  h->eng->localRows(r0, r1);
  return 0;
  HY_CATCH
}

int64_t hymls_b200_owned_rows(hymls_b200_t* h, int64_t* rows, int64_t cap) {
  HY_TRY
  return h->eng->ownedRows(rows, cap);
  HY_CATCH
}

int hymls_b200_apply_inverse_dist(hymls_b200_t* h, const double* Bl, double* Xl, int where) {
  HY_TRY
  h->eng->applyInverseDist(Bl, Xl, where);
  return 0;
  HY_CATCH
}

int hymls_b200_apply_inverse_bordered_dist(hymls_b200_t* h, const double* Bl, const double* T, double* Xl, double* S,
                                           int where) {
  HY_TRY
  if (!T || !S) throw Error(HYMLS_B200_ERR_ARG, "apply_inverse_bordered_dist: T and S are required");
  h->eng->applyInverseDist(Bl, Xl, where, T, S);
  return 0;
  HY_CATCH
}

int hymls_b200_border_size(hymls_b200_t* h) { return h->eng->borderSize(); }

int hymls_b200_get_device(hymls_b200_t* h) {
  HY_TRY
  if (h->eng->device() < 0) throw Error(HYMLS_B200_ERR_CUDA, "no CUDA device");
  return h->eng->device();
  HY_CATCH
}

int hymls_b200_set_border(hymls_b200_t* h, const double* V, const double* W, const double* C, int m) {
  HY_TRY
  h->eng->setBorder(V, W, C, m);
  return 0;
  HY_CATCH
}
int hymls_b200_apply_inverse_bordered(hymls_b200_t* h, const double* B, int64_t ldb, const double* T, double* X,
                                      int64_t ldx, double* S, int nvec, int where) {
  HY_TRY
  h->eng->applyInverseBordered(B, ldb, T, X, ldx, S, nvec, where);
  return 0;
  HY_CATCH
}

int hymls_b200_apply_matrix(hymls_b200_t* h, const double* x, double* y, int where) {
  HY_TRY
  h->eng->applyMatrix(x, y, where);
  return 0;
  HY_CATCH
}

int hymls_b200_solve(hymls_b200_t* h, const double* b, double* x, int where, uint64_t seed,
                     hymls_b200_solve_info* info, double* hist, int cap) {
  HY_TRY
  h->eng->solve(b, nullptr, x, nullptr, VecEnds::Replicated, where, seed, info, hist, cap);
  return 0;
  HY_CATCH
}

int hymls_b200_solve_dist(hymls_b200_t* h, const double* b_local, const double* T, double* x_local, double* S,
                          int where, uint64_t seed, hymls_b200_solve_info* info, double* hist, int cap) {
  HY_TRY
  h->eng->solve(b_local, T, x_local, S, VecEnds::Owned, where, seed, info, hist, cap);
  return 0;
  HY_CATCH
}

int hymls_b200_solve_map(hymls_b200_t* h, const double* b_local, const double* T, double* x_local, double* S,
                         int where, uint64_t seed, hymls_b200_solve_info* info, double* hist, int cap) {
  HY_TRY
  h->eng->solve(b_local, T, x_local, S, VecEnds::RowMap, where, seed, info, hist, cap);
  return 0;
  HY_CATCH
}

int hymls_b200_set_tolerance(hymls_b200_t* h, double tol) {
  HY_TRY
  if (!(tol > 0)) throw Error(HYMLS_B200_ERR_ARG, "set_tolerance: tolerance must be positive");
  h->eng->params().sublist("Solver").sublist("Iterative Solver").set("Convergence Tolerance", tol);
  return 0;
  HY_CATCH
}

int64_t hymls_b200_get_parameters_xml(hymls_b200_t* h, char* buf, int64_t cap) {
  HY_TRY
  const std::string xml = h->eng->params().toXml("Trilinos HYMLS");
  if (buf && cap > (int64_t)xml.size()) std::memcpy(buf, xml.c_str(), xml.size() + 1);
  return (int64_t)xml.size();
  HY_CATCH
}

int hymls_b200_num_levels(hymls_b200_t* h) { return h->eng->initialized() ? h->eng->numLevels() : 0; }

int hymls_b200_num_subdomains(hymls_b200_t* h, int level) {
  HY_TRY
  if (!h->eng->initialized()) throw Error(HYMLS_B200_ERR_STATE, "not initialized");
  return h->eng->sym(level).nsd;
  HY_CATCH
}

int64_t hymls_b200_get_interior(hymls_b200_t* h, int level, int sd, int64_t* gids, int64_t cap) {
  HY_TRY
  if (!h->eng->initialized()) throw Error(HYMLS_B200_ERR_STATE, "not initialized");
  const HierarchicalMap& H = h->eng->sym(level).H;
  if (sd < 0 || sd >= H.nsd) throw Error(HYMLS_B200_ERR_ARG, "subdomain index out of range");
  int64_t a = H.intPtr[sd], z = H.intPtr[sd + 1];
  if (gids && z > a && cap >= z - a) std::memcpy(gids, H.intGid.data() + a, (z - a) * sizeof(int64_t));
  return z - a;
  HY_CATCH
}

int hymls_b200_get_groups(hymls_b200_t* h, int level, int sd, int64_t* ptr, int32_t* types, int64_t* gids,
                          int64_t cap, int64_t* totalLen) {
  HY_TRY
  if (!h->eng->initialized()) throw Error(HYMLS_B200_ERR_STATE, "not initialized");
  const HierarchicalMap& H = h->eng->sym(level).H;
  if (sd < 0 || sd >= H.nsd) throw Error(HYMLS_B200_ERR_ARG, "subdomain index out of range");
  int64_t ga = H.sdGrpPtr[sd], gz = H.sdGrpPtr[sd + 1];
  int64_t a = H.grpPtr[ga], z = H.grpPtr[gz];
  if (totalLen) *totalLen = z - a;
  if (ptr && types && gids && cap >= z - a) {
    for (int64_t g = ga; g <= gz; ++g) ptr[g - ga] = H.grpPtr[g] - a;
    for (int64_t g = ga; g < gz; ++g) types[g - ga] = H.grpType[g];
    if (z > a) std::memcpy(gids, H.grpGid.data() + a, (z - a) * sizeof(int64_t));
  }
  return (int)(gz - ga);
  HY_CATCH
}

int64_t hymls_b200_get_map(hymls_b200_t* h, int level, int which, int64_t* gids, int64_t cap) {
  HY_TRY
  if (!h->eng->initialized()) throw Error(HYMLS_B200_ERR_STATE, "not initialized");
  const LevelSym& S = h->eng->sym(level);
  const std::vector<gidx>* v = nullptr;
  std::vector<gidx> vsum;
  switch (which) {
    case HYMLS_B200_MAP_OVERLAPPING: v = &S.H.overlappingGid; break;
    case HYMLS_B200_MAP_INTERIOR: v = &S.H.intGid; break;
    case HYMLS_B200_MAP_SEPARATOR: v = &S.H.sepGid; break;
    case HYMLS_B200_MAP_VSUM:
      for (int u = 0; u < S.nuniq; ++u) vsum.push_back(S.H.sepGid[S.H.uniqPtr[u]]);
      v = &vsum;
      break;
    default: throw Error(HYMLS_B200_ERR_ARG, "unknown map");
  }
  if (gids && !v->empty() && cap >= (int64_t)v->size()) std::memcpy(gids, v->data(), v->size() * sizeof(int64_t));
  return (int64_t)v->size();
  HY_CATCH
}

int hymls_b200_pid_map(const char* xml, int nprocs, int32_t* pid, int cap) {
  HY_TRY
  ParameterList p = ParameterList::fromXml(xml);
  std::unique_ptr<CartesianPartitioner> part(makePartitioner(p, 0, nprocs, 0));
  part->partition();
  const std::vector<int>& m = part->pidMap();
  if (pid && !m.empty() && cap >= (int)m.size()) std::memcpy(pid, m.data(), m.size() * sizeof(int));
  return (int)m.size();
  HY_CATCH
}

int hymls_b200_get_stats(hymls_b200_t* h, hymls_b200_stats* st) {
  HY_TRY
  h->eng->getStats(st);
  return 0;
  HY_CATCH
}

int64_t hymls_b200_debug_copy(hymls_b200_t* h, int level, const char* name, double* out, int64_t cap) {
  HY_TRY
  return h->eng->debugCopy(level, name, out, cap);
  HY_CATCH
}

int hymls_b200_time_apply(hymls_b200_t* h, int reps, double* msApply, double* msA11) {
  HY_TRY
  h->eng->timeApply(reps, msApply, msA11);
  return 0;
  HY_CATCH
}

}  // extern "C"

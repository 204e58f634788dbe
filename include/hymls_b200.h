/*
 * hymls_b200 -- C ABI of the B200-native HYMLS preconditioner hot path.
 *
 * Drop-in boundary for HYMLS::Preconditioner (reference: src/HYMLS_Preconditioner.hpp:56-254)
 * and for the Krylov driver HYMLS::Solver/BaseSolver (src/HYMLS_Solver.hpp, src/HYMLS_BaseSolver.cpp:309-359).
 * Plain pointers and sizes only; every function returns 0 on success and a negative code on
 * failure (hymls_b200_last_error() gives the message) -- the reference's convention
 * (`int` return, 0 = OK, src/HYMLS_Macros.hpp:147-158), with no exception crossing the boundary.
 *
 * A handle is not thread safe (same as the reference object): one call at a time per handle.
 * All compute runs on the CUDA device that is current when hymls_b200_create() is called, on the
 * stream set with hymls_b200_set_stream() (default: the legacy default stream).
 * There is no CPU fallback: every entry point that computes (set values on the device, Compute,
 * ApplyInverse, solve, ...) fails with HYMLS_B200_ERR_CUDA when no device is usable.  Only the integer
 * host work of Initialize (partitioning, index maps) runs without a device, so that the maps can be
 * compared with the reference anywhere.
 */
#ifndef HYMLS_B200_H
#define HYMLS_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct hymls_b200 hymls_b200_t;

enum {
  HYMLS_B200_OK = 0,
  HYMLS_B200_ERR_ARG = -1,      /* bad argument / bad parameter list (Tools::Error in the reference) */
  HYMLS_B200_ERR_STATE = -2,    /* call order: ApplyInverse before Compute (Preconditioner.cpp:936-939) */
  HYMLS_B200_ERR_CUDA = -3,     /* CUDA failure or no device */
  HYMLS_B200_ERR_NUMERIC = -4,  /* singular block met during Compute */
  HYMLS_B200_ERR_UNSUPPORTED = -99 /* same code the reference returns for unimplemented paths */
};

/* where a vector/matrix argument lives */
enum { HYMLS_B200_HOST = 0, HYMLS_B200_DEVICE = 1 };

/* CUDA device the handle is bound to (the current device at hymls_b200_create); HYMLS_B200_ERR_CUDA without one. */
int hymls_b200_get_device(hymls_b200_t* h);

/* Message of the last failure on this thread ("" if none). */
const char* hymls_b200_last_error(void);

/* Library version string and the device it is bound to (NULL if no CUDA device). */
const char* hymls_b200_version(void);

/*
 * Constructor -- HYMLS::Preconditioner::Preconditioner(K, params, testVector, myLevel=0)
 * (src/HYMLS_Preconditioner.hpp:80-84).  `xml` is a Teuchos XML parameter list (the text, not a
 * file name) with the sublists "Problem" and "Preconditioner" (and optionally "Solver"), exactly as
 * in the reference's testSuite XML files; unknown entries in "Preconditioner" are rejected like
 * validateParameters does (src/HYMLS_Preconditioner.cpp:126-130) unless they are listed in
 * DESIGN.md as extensions.
 */
int hymls_b200_create(const char* xml, hymls_b200_t** out);
void hymls_b200_destroy(hymls_b200_t* h);

/* CUDA stream (cudaStream_t passed as void*) used for every launch of this handle. */
int hymls_b200_set_stream(hymls_b200_t* h, void* cuda_stream);

/*
 * Multi-GPU: one process per GPU, one handle per process.  Level-0 subdomains are sharded by the
 * reference's subdomain -> rank map (BasePartitioner::CreatePIDMap, src/HYMLS_BasePartitioner.cpp:361-586);
 * the exchanges of the reference's Epetra Import/Export/SumAll become NCCL all-reduces on the handle's
 * stream.  Rank 0 creates the id (128 bytes, ncclUniqueId) and ships it to the others (e.g. with
 * torch.distributed); comm_init is collective and must precede Initialize().  After it, set_matrix,
 * Initialize, Compute, ApplyInverse and solve are collective calls with replicated arguments.
 * hymls_b200_set_rank only records (rank, nranks) for the host-side ownership logic (no NCCL, no GPU).
 */
int hymls_b200_comm_get_unique_id(void* id128);
int hymls_b200_comm_init(hymls_b200_t* h, const void* id128, int rank, int nranks);
int hymls_b200_set_rank(hymls_b200_t* h, int rank, int nranks);
/* local subdomain ids (level numbering of hymls_b200_get_interior) owned by this rank; returns the count */
int hymls_b200_get_owned_subdomains(hymls_b200_t* h, int level, int32_t* sd, int cap);

/*
 * Matrix K as CSR with 0-based indices, rows in global (GID) order: row i <-> GID i
 * (Epetra_CrsMatrix::ExtractMyRowView on a linear map).  `where` says whether the three arrays are
 * host or device pointers.  The pattern is fixed by the first call; later calls with the same
 * pattern only replace values (SetMatrix + Compute recompute path, Preconditioner.hpp:244-254).
 */
int hymls_b200_set_matrix_csr(hymls_b200_t* h, int64_t n, const int64_t* rowptr, const int32_t* colidx,
                              const double* values, int where);

/*
 * Distributed matrix input (one MPI rank per GPU): every rank passes the rows it holds -- n_local rows with global
 * ids row_gids (any distribution that tiles [0, n_global)), CSR with GLOBAL column ids, host pointers -- exactly what
 * Epetra_CrsMatrix::ExtractMyRowView + RowMap().MyGlobalElements() + ColMap().GID() give.  Collective.  Replaces
 * the import of the matrix to the partitioner's map (src/HYMLS_Preconditioner.cpp:420-431): rows are gathered over
 * NCCL (the symbolic phase is replicated on every rank).  Same pattern again: only values move.  values == NULL:
 * pattern only.  With one rank it is hymls_b200_set_matrix_csr up to the row permutation.
 */
int hymls_b200_set_matrix_csr_dist(hymls_b200_t* h, int64_t n_global, int64_t n_local, const int64_t* row_gids,
                                   const int64_t* rowptr, const int64_t* col_gids, const double* values);

/* Preconditioner::SetParameters (src/HYMLS_Preconditioner.cpp:87-114): replaces the parameter list (XML text as in
 * hymls_b200_create); Initialize() has to follow.  An invalid list is rejected and the old one kept. */
int hymls_b200_set_parameters(hymls_b200_t* h, const char* xml);

/* Test vector (length n, host); NULL = ones (Preconditioner::CreateTestVector, .cpp:780-790). */
int hymls_b200_set_testvector(hymls_b200_t* h, const double* tv);

/* Preconditioner::Initialize / Compute (src/HYMLS_Preconditioner.cpp:279-394, 400-517). */
int hymls_b200_initialize(hymls_b200_t* h);
int hymls_b200_compute(hymls_b200_t* h);

/*
 * Preconditioner::ApplyInverse(B, X) (src/HYMLS_Preconditioner.cpp:594-605, 930-1070).
 * B, X: nvec columns of length n, column stride ldb / ldx (Epetra_MultiVector::Values()/Stride()).
 */
int hymls_b200_apply_inverse(hymls_b200_t* h, const double* B, int64_t ldb, double* X, int64_t ldx,
                             int nvec, int where);

/*
 * Distributed-vector variant for multi-GPU use (the reference's vectors are distributed Epetra_MultiVectors on the
 * map its partitioner induces, src/HYMLS_Preconditioner.cpp:978-979, 1050-1052).  A rank owns the rows of the
 * interiors of its subdomains (BasePartitioner::CreatePIDMap) and of the separator groups whose owner subdomain is
 * its own; hymls_b200_owned_rows lists them (ascending GIDs; returns the count, rows may be NULL to query it).
 * hymls_b200_apply_inverse_dist takes / returns exactly those rows, in that order.  Nothing but separator values on
 * the interfaces between ranks, the V-sums and (in hymls_b200_solve) dot products cross NVLink.
 * With one rank: all rows, the same as hymls_b200_apply_inverse.
 * hymls_b200_local_rows (contiguous row blocks) is kept for one rank only and fails with several.
 */
int64_t hymls_b200_owned_rows(hymls_b200_t* h, int64_t* rows, int64_t cap);
int hymls_b200_local_rows(hymls_b200_t* h, int64_t* r0, int64_t* r1);
int hymls_b200_apply_inverse_dist(hymls_b200_t* h, const double* B_local, double* X_local, int where);
/*
 * Bordered form on the same rows: [X; S] = [K V; W' C]^-1 [B; T] with B_local / X_local the rows of
 * hymls_b200_owned_rows and T, S replicated m-vectors (S comes out bitwise equal on every rank); `where` applies to
 * all four buffers.  Only separator values on the interfaces, the V-sums and a few m-vectors cross NVLink.  With one
 * rank it is hymls_b200_apply_inverse_bordered.  hymls_b200_apply_inverse_dist with a border set means T = 0 with S
 * discarded, as for hymls_b200_apply_inverse.  Without a border set m = 0: X is the plain ApplyInverse and S, which
 * has no entries, is not written (as for hymls_b200_apply_inverse_bordered).
 */
int hymls_b200_apply_inverse_bordered_dist(hymls_b200_t* h, const double* B_local, const double* T, double* X_local,
                                           double* S, int where);

/*
 * Vectors in the CALLER's distribution (Epetra_Operator::ApplyInverse on the matrix' row map, any map):
 * hymls_b200_set_row_map declares the rows this rank holds, in its local order (collective, after Initialize);
 * hymls_b200_apply_inverse_map then takes B_local / X_local (n_local x nvec, column major, leading dimensions
 * ldb / ldx) in that order.  Values travel to the rows' owners and back with one grouped ncclSend/ncclRecv each
 * way; when the caller's map is the owner map (hymls_b200_owned_rows) this is a local permutation.
 */
int hymls_b200_set_row_map(hymls_b200_t* h, int64_t n_local, const int64_t* row_gids);
int hymls_b200_apply_inverse_map(hymls_b200_t* h, const double* B_local, int64_t ldb, double* X_local, int64_t ldx,
                                 int nvec, int where);
/* BorderedOperator::ApplyInverse(X, T, Y, S) on the caller's map; T and S (m x nvec, column major) are replicated */
int hymls_b200_apply_inverse_bordered_map(hymls_b200_t* h, const double* B_local, int64_t ldb, const double* T,
                                          double* X_local, int64_t ldx, double* S, int nvec, int where);
/* distributed forms of hymls_b200_set_testvector / hymls_b200_set_border: this rank's entries (rows row_gids, V and
 * W with leading dimension n_local); collective */
int hymls_b200_set_testvector_dist(hymls_b200_t* h, int64_t n_local, const int64_t* row_gids, const double* tv);
int hymls_b200_set_border_dist(hymls_b200_t* h, int64_t n_local, const int64_t* row_gids, const double* V,
                               const double* W, const double* C, int m);

/*
 * BorderedOperator interface (src/HYMLS_Preconditioner.cpp:844-918): V, W are n x m (column major,
 * host), C is m x m; W == NULL means W = V, C == NULL means 0.  V == NULL removes the border.
 * Compute() must be called afterwards.
 */
int hymls_b200_set_border(hymls_b200_t* h, const double* V, const double* W, const double* C, int m);
/* m of the border set by hymls_b200_set_border / hymls_b200_set_border_dist (0: none) */
int hymls_b200_border_size(hymls_b200_t* h);
/* [X;S] = [K V; W' C]^-1 [B;T]  (Preconditioner.cpp:930-1070); T, S are m x nvec column major. */
int hymls_b200_apply_inverse_bordered(hymls_b200_t* h, const double* B, int64_t ldb, const double* T,
                                      double* X, int64_t ldx, double* S, int nvec, int where);

/* y = K x with the matrix held by the handle (Epetra_CrsMatrix::Apply). */
int hymls_b200_apply_matrix(hymls_b200_t* h, const double* x, double* y, int where);

/*
 * Krylov driver -- HYMLS::Solver(K, P, params)::ApplyInverse(b, x) (src/HYMLS_BaseSolver.cpp:309-359).
 * Uses the "Solver" sublist of the XML given at creation (Krylov Method GMRES|CG, Left or Right
 * Preconditioning, Initial Vector Zero|Random|Previous, "Iterative Solver": Maximum Iterations,
 * Num Blocks, Maximum Restarts, Convergence Tolerance, Explicit Residual Test, *Residual Scaling).
 * x holds the initial guess when Initial Vector = Previous and receives the solution.
 * If a border is set the bordered system is solved (HYMLS::BorderedSolver) with right-hand side [b;0], on several
 * ranks on the owner distribution like the unbordered system (the m border entries are replicated on every rank).
 * resid_history (may be NULL) receives up to history_cap relative implicit residuals, iteration 0 first.
 */
typedef struct {
  int iterations;
  int converged;
  double rel_residual;        /* last implicit relative residual */
  double explicit_rel_residual; /* ||b - K x|| / ||b|| evaluated at the end */
  double solve_seconds;       /* device time of the whole solve (CUDA events) */
  int history_len;
} hymls_b200_solve_info;
int hymls_b200_solve(hymls_b200_t* h, const double* b, double* x, int where, uint64_t random_seed,
                     hymls_b200_solve_info* info, double* resid_history, int history_cap);

/* BaseSolver::SetTolerance (src/HYMLS_BaseSolver.cpp, used by NOX_Epetra_LinearSystem_Hymls.cpp:330-334 to
   override "Convergence Tolerance" per solve). */
int hymls_b200_set_tolerance(hymls_b200_t* h, double tol);

/* The parameter list as it stands -- with the defaults the partitioner / preconditioner / solver wrote back
   (e.g. "Fix GID 1", "Degrees of Freedom"), like the reference's "Store Final Parameter List" (src/main.cpp:492-509) --
   as Teuchos XML.  Returns the length (without the terminating 0); writes only if cap > length. */
int64_t hymls_b200_get_parameters_xml(hymls_b200_t* h, char* buf, int64_t cap);

/* ---- index maps, for bit-exact comparison with the reference (HierarchicalMap) ---- */
int hymls_b200_num_levels(hymls_b200_t* h);
int hymls_b200_num_subdomains(hymls_b200_t* h, int level);
/* interior group of subdomain sd: GIDs ascending (HierarchicalMap::GetInteriorGroup). cap<len -> len returned, nothing written */
int64_t hymls_b200_get_interior(hymls_b200_t* h, int level, int sd, int64_t* gids, int64_t cap);
/* separator groups of sd in reference order: ptr has ngroups+1 entries, types ngroups; returns ngroups.
   Call with NULL pointers to query sizes: *total_len receives the number of GIDs. */
int hymls_b200_get_groups(hymls_b200_t* h, int level, int sd, int64_t* ptr, int32_t* types,
                          int64_t* gids, int64_t cap, int64_t* total_len);
/* overlapping (row) map, separator map and V-sum map of a level (GIDs); returns length */
int64_t hymls_b200_get_map(hymls_b200_t* h, int level, int which, int64_t* gids, int64_t cap);
enum { HYMLS_B200_MAP_OVERLAPPING = 0, HYMLS_B200_MAP_INTERIOR = 1, HYMLS_B200_MAP_SEPARATOR = 2,
       HYMLS_B200_MAP_VSUM = 3 };
/* subdomain -> rank map of BasePartitioner::CreatePIDMap for `nprocs` ranks (level 0), length = #subdomains */
int hymls_b200_pid_map(const char* xml, int nprocs, int32_t* pid, int cap);

/* ---- statistics (Ifpack-style counters, src/HYMLS_Preconditioner.cpp:612-717) ---- */
typedef struct {
  int num_initialize, num_compute, num_apply_inverse;
  double time_initialize, time_compute, time_apply_inverse; /* seconds (host wall for init, CUDA events else) */
  int64_t n, num_interior, num_separator, num_vsum;          /* level 0 */
  int64_t num_subdomains, num_blocks;
  double sum_nsd_sq;            /* sum over subdomains of n_sd^2 (level 0), the roofline figure of SURVEY 8(d) */
  double bytes_apply;           /* algorithmic bytes of one ApplyInverse (all levels), SURVEY 8(d) formula */
  double flops_compute;         /* algorithmic flops of Compute (inversions: 2 n^3) */
  double bytes_a11_level0;      /* this rank's level-0 A11^-1 bytes streamed by one ApplyInverse:
                                   8 * sum (n_sd^2 + n_sd * nb_sd), full second solve + leading rows of the first */
  int64_t kernel_launches;      /* launches issued by this handle so far */
  double device_bytes;          /* device memory held */
  double sum_nsd_nb;            /* sum n_sd * nb_sd (level 0): nb_sd = interior nodes that separator rows couple to;
                                   the first subdomain solve of ApplyInverse needs only these rows of A11^-1 */
  double bytes_a11_full_pass;   /* this rank's 8 * sum n_sd^2: one full pass over its level-0 inverses */
  double ms_a11_lead;           /* set by hymls_b200_time_apply: CUDA-event time of the leading-rows pass */
  int64_t interior_couplings;   /* matrix entries between interiors of DIFFERENT subdomains, all levels: must be 0
                                   for a correct domain decomposition (Tester::isDDcorrect, src/HYMLS_Tester.cpp:253-455);
                                   such entries would be ignored by the subdomain solvers */
  int64_t a11_split;            /* 1: the second level-0 subdomain solve is split (HYMLS_B200_SPLIT_SOLVE=1, off by default): rows [nb, n) of A11^-1 b1
                                   run on a low-priority stream beside the separator phase, and the pass on the critical
                                   path reads only the leading nb COLUMNS (x1 = A11^-1 b1 - A11^-1[:, :nb] (A12 x2)); the
                                   bytes per ApplyInverse are unchanged.  bytes_a11_full_pass / ms_a11_kernel_per_launch
                                   then describe that leading-columns pass (8 * sum n_sd nb_sd bytes).  0: one full pass */
  int64_t host_pipeline_chunks; /* ApplyInverse with HOST buffers on one GPU: number of chunks in which the copy of b is
                                   overlapped with the leading-rows pass and the copy of x with the full pass over the
                                   level-0 inverses (0: no schedule -- several ranks, Number of Levels = 0, or fewer rows
                                   than HYMLS_B200_HOST_PIPELINE_MIN_ROWS, default 2^20).  Used for pinned buffers only */
  int64_t host_pipeline_state;  /* 0: not used yet, 1: in use (its first call reproduced the serial path bit for bit),
                                   -1: that check failed, serial copies are used, -2: switched off (HYMLS_B200_HOST_PIPELINE=0) */
  int64_t collective_calls;     /* NCCL calls of this rank since comm_init (all-reduce, broadcast, all-gather, one per grouped
                                   neighbour exchange); 0 on one rank */
  int64_t collective_bytes;     /* their payload on this rank: 8 * count of every all-reduce / broadcast / all-gather (one
                                   rank's part), plus the bytes sent and received by the neighbour exchanges */
} hymls_b200_stats;
int hymls_b200_get_stats(hymls_b200_t* h, hymls_b200_stats* st);

/* Timed loop helpers used by bench.py: run ApplyInverse `reps` times on device-resident vectors and
   return the average CUDA-event time per call of (a) the whole call, (b) the dominant kernel
   (batched A11^-1 apply, the full pass of the second subdomain solve; the shorter leading-rows pass of the
   first solve is reported in hymls_b200_stats.ms_a11_lead). */
int hymls_b200_time_apply(hymls_b200_t* h, int reps, double* ms_per_apply, double* ms_a11_kernel_per_launch);

/* Test hook: copies a named device array of a level ("a11inv", "blkinv", "coarseinv", "redval", "v12",
   "v21", "what") or host index array ("a11off", "blkoff", "blkrows", "redptr", "redcol", "introw", "seprow":
   the matrix row of every interior / separator position) to the host as doubles; returns its length
   (call with out == NULL to query). */
int64_t hymls_b200_debug_copy(hymls_b200_t* h, int level, const char* name, double* out, int64_t cap);

#ifdef __cplusplus
}
#endif
#endif

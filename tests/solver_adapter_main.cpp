// Drives include/HYMLS_B200_Solver.hpp the way hymls_main / NOX drive HYMLS::Solver, on a serial stand-in
// Epetra_CrsMatrix whose row map is NOT in GID order (tests/shim/).  Usage:
//   solver_adapter_main <matrix.bin> <levels> <tv.bin> <out.bin>
// matrix.bin / tv.bin as written by tests/test_adapter_shim.py (2D Stokes-C).  Solves two right-hand sides through
// B200Solver::ApplyInverse, then sets the constant-pressure border and solves [K V; V' 0] [x; s] = [b; t] through the
// bordered ApplyInverse.  Every solve is repeated with hymls_b200_solve_map on the same handle and must agree bitwise.
// Writes, in GID order: X (2 columns), the bordered x, B (2 columns), then s, the iteration counts of the second
// column's solve and of the bordered solve, and the bordered solve's explicit relative residual.
// exit code 0: ok, 3: the library refused because there is no CUDA device (expected on a CPU-only host)
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <numeric>
#include "HYMLS_B200_Solver.hpp"

static bool same(const double* a, const double* b, int n) { return std::memcmp(a, b, sizeof(double) * n) == 0; }

int main(int argc, char** argv) {
  if (argc < 5) return 2;
  const int levels = atoi(argv[2]);
  std::ifstream in(argv[1], std::ios::binary);
  int n = 0, nnz = 0, nx = 0;
  in.read((char*)&n, 4); in.read((char*)&nnz, 4); in.read((char*)&nx, 4);
  std::vector<int> ptr(n + 1), col(nnz);
  std::vector<double> val(nnz);
  in.read((char*)ptr.data(), 4 * (n + 1)); in.read((char*)col.data(), 4 * nnz); in.read((char*)val.data(), 8 * nnz);
  std::vector<long long> perm(n), ident(n);
  std::iota(ident.begin(), ident.end(), 0LL);
  for (int i = 0; i < n; ++i) perm[i] = ((long long)i * 7 + 3) % n;  // 7 is coprime with the test sizes
  std::vector<int> pptr(n + 1, 0), pcol;
  std::vector<double> pval;
  for (int i = 0; i < n; ++i) {
    const int g = (int)perm[i];
    for (int e = ptr[g]; e < ptr[g + 1]; ++e) { pcol.push_back(col[e]); pval.push_back(val[e]); }
    pptr[i + 1] = (int)pcol.size();
  }
  Epetra_SerialComm comm;
  Epetra_Map rowMap(n, n, perm.data(), 0, comm), colMap(n, n, ident.data(), 0, comm);
  Teuchos::RCP<const Epetra_RowMatrix> K(new Epetra_CrsMatrix(rowMap, colMap, pptr, pcol, pval));
  Teuchos::RCP<Teuchos::ParameterList> params(new Teuchos::ParameterList("HYMLS"));
  params->sublist("Problem").set("Equations", "Stokes-C").set("Dimension", 2).set("nx", nx).set("ny", nx).set("nz", 1);
  params->sublist("Preconditioner").set("Separator Length", 4).set("Number of Levels", levels);
  Teuchos::ParameterList& sol = params->sublist("Solver");
  sol.set("Krylov Method", "GMRES").set("Left or Right Preconditioning", "Right").set("Initial Vector", "Random");
  sol.sublist("Iterative Solver").set("Maximum Iterations", 300).set("Num Blocks", 300).set("Maximum Restarts", 1)
      .set("Convergence Tolerance", 1e-8);
  Teuchos::RCP<Epetra_Vector> tv(new Epetra_Vector(rowMap));
  {
    std::ifstream tin(argv[3], std::ios::binary);
    std::vector<double> t(n);
    tin.read((char*)t.data(), 8 * n);
    for (int i = 0; i < n; ++i) (*tv)[0][i] = t[perm[i]];
  }
  try {
    Teuchos::RCP<HYMLS::B200Preconditioner> P(new HYMLS::B200Preconditioner(K, params, tv));
    if (P->Initialize() != 0 || P->Compute() != 0) {
      fprintf(stderr, "Initialize / Compute: %s\n", hymls_b200_last_error());
      return strstr(hymls_b200_last_error(), "needs a CUDA device") ? 3 : 1;
    }
    HYMLS::B200Solver S(P);
    Epetra_Operator& op = S;  // used through the Epetra_Operator interface, like NOX does
    Epetra_MultiVector B(rowMap, 2), X(rowMap, 2);
    for (int i = 0; i < n; ++i) {
      B[0][i] = std::sin(0.37 * (double)perm[i]);
      B[1][i] = 1.0 / (1.0 + (double)perm[i]);
    }
    std::vector<int> its;
    if (op.ApplyInverse(B, X) != 0) return 1;
    its.push_back(S.getNumIter());
    hymls_b200_solve_info info;
    std::vector<double> x(n);
    for (int j = 0; j < 2; ++j) {  // the last column's solve is the one getNumIter reports
      if (hymls_b200_solve_map(P->Handle(), B[j], nullptr, x.data(), nullptr, HYMLS_B200_HOST, 43, &info, nullptr, 0))
        return 1;
      if (!same(x.data(), X[j], n)) { fprintf(stderr, "column %d differs from solve_map\n", j); return 1; }
    }
    if (info.iterations != its[0]) return 1;

    // BorderedSolver: constant-pressure border (dof 3, pressure = GID % 3 == 2), t = 0.5
    Teuchos::RCP<Epetra_MultiVector> V(new Epetra_MultiVector(rowMap, 1));
    int np = 0;
    for (int i = 0; i < n; ++i) np += perm[i] % 3 == 2;
    for (int i = 0; i < n; ++i) (*V)[0][i] = perm[i] % 3 == 2 ? 1.0 / std::sqrt((double)np) : 0.0;
    if (S.SetBorder(V) != 0 || P->Compute() != 0) { fprintf(stderr, "border: %s\n", hymls_b200_last_error()); return 1; }
    Epetra_SerialDenseMatrix T(1, 1), Sb(1, 1);
    T(0, 0) = 0.5;
    Epetra_MultiVector B1(rowMap, 1), Xb(rowMap, 1);
    std::copy(B[0], B[0] + n, B1[0]);
    S.ApplyInverse(B1, T, Xb, Sb);
    its.push_back(S.getNumIter());
    double t = 0.5, s = 0.0;
    if (hymls_b200_solve_map(P->Handle(), B[0], &t, x.data(), &s, HYMLS_B200_HOST, 43, &info, nullptr, 0)) return 1;
    if (!same(x.data(), Xb[0], n) || !same(&s, &Sb(0, 0), 1) || info.iterations != its[1]) {
      fprintf(stderr, "bordered solve differs from solve_map\n");
      return 1;
    }
    std::vector<double> out((size_t)5 * n + 4);
    for (int i = 0; i < n; ++i) {
      out[perm[i]] = X[0][i];
      out[(size_t)n + perm[i]] = X[1][i];
      out[(size_t)2 * n + perm[i]] = Xb[0][i];
      out[(size_t)3 * n + perm[i]] = B[0][i];
      out[(size_t)4 * n + perm[i]] = B[1][i];
    }
    out[(size_t)5 * n] = Sb(0, 0);
    out[(size_t)5 * n + 1] = its[0];
    out[(size_t)5 * n + 2] = its[1];
    out[(size_t)5 * n + 3] = S.LastSolveInfo().explicit_rel_residual;
    std::ofstream of(argv[4], std::ios::binary);
    of.write((const char*)out.data(), 8 * out.size());
    printf("solver adapter ok: %s, %d and %d iterations\n", S.Label(), its[0], its[1]);
    return 0;
  } catch (const std::exception& e) {
    fprintf(stderr, "exception: %s\n", e.what());
    return strstr(e.what(), "needs a CUDA device") ? 3 : 1;
  }
}

// HYMLS::B200Solver -- Trilinos-side stand-in for HYMLS::Solver / HYMLS::BorderedSolver (src/HYMLS_Solver.hpp,
// src/HYMLS_BorderedSolver.cpp:100-219): the Krylov solve runs on the GPU through hymls_b200_solve_map (include/
// hymls_b200.h) on Epetra vectors of the matrix' row map, one column at a time.  Built on a B200Preconditioner, whose
// handle it shares; the "Solver" sublist of that preconditioner's parameter list configures it.  NOX
// (NOX_Epetra_LinearSystem_Hymls) and hymls_main take it where they take HYMLS::Solver.
//
// Errors go through Tools::Error, like the reference's HYMLS_CHECK_ZERO around its solves.  Apply (the matrix) is not
// offered: the reference's callers use the matrix itself for that.
#ifndef HYMLS_B200_SOLVER_HPP
#define HYMLS_B200_SOLVER_HPP

#include <cstdint>
#include <vector>

#include "HYMLS_B200_Preconditioner.hpp"

namespace HYMLS {

class B200Solver : public Epetra_Operator, public BorderedOperator {
 public:
  // HYMLS::Solver(K, P, params): P is initialized and computed before the first ApplyInverse.  `seed` feeds Initial
  // Vector = Random (the same stream as hymls_b200_solve for any row map).
  explicit B200Solver(Teuchos::RCP<B200Preconditioner> prec, uint64_t seed = 43) : prec_(prec), seed_(seed) {}

  // BaseSolver::SetTolerance: "Convergence Tolerance" of the following solves
  int SetTolerance(double tol) {
    Check(hymls_b200_set_tolerance(prec_->Handle(), tol));
    return 0;
  }
  int getNumIter() const { return info_.iterations; }
  const hymls_b200_solve_info& LastSolveInfo() const { return info_; }  // of the last column solved

  // Solver::ApplyInverse(B, X): X holds the initial guesses for Initial Vector = Previous.  With a border set on the
  // preconditioner this is the bordered solve with T = 0 and s discarded.
  int ApplyInverse(const Epetra_MultiVector& B, Epetra_MultiVector& X) const {
    for (int j = 0; j < B.NumVectors(); ++j)
      Check(hymls_b200_solve_map(prec_->Handle(), B[j], nullptr, X[j], nullptr, HYMLS_B200_HOST, seed_, &info_,
                                 nullptr, 0));
    return 0;
  }

  // BorderedSolver::ApplyInverse(B, T, X, S): [K V; W' C] [X; S] = [B; T]
  int ApplyInverse(const Epetra_MultiVector& B, const Epetra_SerialDenseMatrix& T, Epetra_MultiVector& X,
                   Epetra_SerialDenseMatrix& S) const {
    const int m = hymls_b200_border_size(prec_->Handle());
    if (T.M() != m || T.N() != B.NumVectors() || S.M() != m || S.N() != B.NumVectors())
      Tools::Error("B200Solver::ApplyInverse: T and S must be m x (number of columns of B)", __FILE__, __LINE__);
    std::vector<double> t(m), s(m);
    for (int j = 0; j < B.NumVectors(); ++j) {
      for (int i = 0; i < m; ++i) t[i] = T(i, j);
      Check(hymls_b200_solve_map(prec_->Handle(), B[j], t.data(), X[j], s.data(), HYMLS_B200_HOST, seed_, &info_,
                                 nullptr, 0));
      for (int i = 0; i < m; ++i) S(i, j) = s[i];
    }
    return 0;
  }

  // BorderedSolver::SetBorder: the border lives in the preconditioner; Compute() of the preconditioner must follow
  int SetBorder(Teuchos::RCP<const Epetra_MultiVector> V, Teuchos::RCP<const Epetra_MultiVector> W = Teuchos::null,
                Teuchos::RCP<const Epetra_SerialDenseMatrix> C = Teuchos::null) {
    return prec_->SetBorder(V, W, C);
  }

  int Apply(const Epetra_MultiVector&, Epetra_MultiVector&) const { return -1; }
  int Apply(const Epetra_MultiVector&, const Epetra_SerialDenseMatrix&, Epetra_MultiVector&,
            Epetra_SerialDenseMatrix&) const { return -1; }
  int SetUseTranspose(bool) { return -1; }
  bool UseTranspose() const { return false; }
  bool HasNormInf() const { return false; }
  double NormInf() const { return -1.0; }
  const char* Label() const { return "HYMLS::B200Solver"; }
  const Epetra_Comm& Comm() const { return prec_->Comm(); }
  const Epetra_Map& OperatorDomainMap() const { return prec_->OperatorDomainMap(); }
  const Epetra_Map& OperatorRangeMap() const { return prec_->OperatorRangeMap(); }

 private:
  void Check(int e) const {
    if (e) Tools::Error(hymls_b200_last_error(), __FILE__, __LINE__);
  }
  Teuchos::RCP<B200Preconditioner> prec_;
  uint64_t seed_;
  mutable hymls_b200_solve_info info_{};
};

}  // namespace HYMLS
#endif

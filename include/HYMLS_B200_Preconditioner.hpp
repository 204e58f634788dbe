// HYMLS::B200Preconditioner -- Trilinos-side adapter: the reference's HYMLS::Preconditioner interface
// (Ifpack_Preconditioner + BorderedOperator, src/HYMLS_Preconditioner.hpp:56-254) implemented by calls into
// libhymls_b200.so (include/hymls_b200.h).  HYMLS::Solver / Belos (src/HYMLS_BaseSolver.cpp:119-139),
// HYMLS::BorderedSolver (src/HYMLS_BorderedSolver.cpp:100-219), hymls_main (src/main.cpp:330-372) and
// NOX_Epetra_LinearSystem_Hymls (src/NOX_Epetra_LinearSystem_Hymls.cpp:177-220) take it unchanged as `precPtr`.
//
// Needs the Trilinos headers (Epetra, Ifpack, Teuchos) and two headers of the reference tree; inside the reference
// tree it is added to src/ and linked with -lhymls_b200.  This repository has no Trilinos: tests/shim/ holds
// minimal stand-ins for exactly the declarations used here, and tests/test_adapter_shim.py compiles this header
// against them, links it with the library and runs it (construction, SetParameters, Initialize, Compute,
// ApplyInverse on a serial Epetra_CrsMatrix stand-in).
// Matrix and vectors may live on ANY Epetra map: rows go through hymls_b200_set_matrix_csr_dist (rows of this rank
// with their GIDs), vectors through hymls_b200_set_row_map / hymls_b200_apply_inverse_map (the matrix' row map).
// One MPI rank per GPU: call CommInit() on every rank before Initialize() (rank 0 creates the NCCL id with
// hymls_b200_comm_get_unique_id and broadcasts it with MPI_Bcast).
#ifndef HYMLS_B200_PRECONDITIONER_HPP
#define HYMLS_B200_PRECONDITIONER_HPP

#include <algorithm>
#include <cstdint>
#include <sstream>
#include <string>
#include <vector>

#include "Epetra_CrsMatrix.h"
#include "Epetra_MultiVector.h"
#include "Epetra_SerialDenseMatrix.h"
#include "Ifpack_Preconditioner.h"
#include "Teuchos_ParameterList.hpp"
#include "Teuchos_RCP.hpp"
#include "Teuchos_XMLParameterListCoreHelpers.hpp"

#include "HYMLS_BorderedOperator.hpp"
#include "HYMLS_Tools.hpp"
#include "hymls_b200.h"

namespace HYMLS {

class B200Preconditioner : public Ifpack_Preconditioner, public BorderedOperator {
 public:
  // HYMLS::Preconditioner(K, params, testVector), src/HYMLS_Preconditioner.hpp:80-84
  B200Preconditioner(Teuchos::RCP<const Epetra_RowMatrix> K, Teuchos::RCP<Teuchos::ParameterList> params,
                     Teuchos::RCP<Epetra_Vector> testVector = Teuchos::null)
      : K_(Teuchos::rcp_dynamic_cast<const Epetra_CrsMatrix>(K, true)), params_(params) {
    commPending_ = K_->Comm().NumProc() > 1;
    std::ostringstream xml;  // the list the reference's XML files are parsed into
    Teuchos::writeParameterListToXmlOStream(*params, xml);
    Check(hymls_b200_create(xml.str().c_str(), &h_));
    Check(PushMatrix());
    testVector_ = testVector;
    PushTestVector();
  }
  virtual ~B200Preconditioner() { hymls_b200_destroy(h_); }

  // one process per GPU: id128 from hymls_b200_comm_get_unique_id on rank 0, shipped with MPI_Bcast
  int CommInit(const void* id128, int rank, int nranks) {
    int e = hymls_b200_comm_init(h_, id128, rank, nranks);
    if (e == 0) {
      commPending_ = false;
      e = PushMatrix();  // the rows of the other ranks can be gathered now
    }
    return e;
  }

  // SetMatrix + Initialize reuses the ordering when the pattern is unchanged (:250-254)
  int SetMatrix(Teuchos::RCP<const Epetra_CrsMatrix> K) {
    K_ = K;
    computed_ = false;
    return PushMatrix();
  }
  int SetMatrix(Teuchos::RCP<const Epetra_RowMatrix> K) {
    return SetMatrix(Teuchos::rcp_dynamic_cast<const Epetra_CrsMatrix>(K, true));
  }
  // Preconditioner::SetParameters (src/HYMLS_Preconditioner.cpp:87-114): a new list; Initialize() has to follow
  int SetParameters(Teuchos::ParameterList& list) {
    params_->setParameters(list);
    std::ostringstream xml;
    Teuchos::writeParameterListToXmlOStream(*params_, xml);
    initialized_ = computed_ = false;
    return hymls_b200_set_parameters(h_, xml.str().c_str());
  }
  int Initialize() {
    if (commPending_) return -1;  // several MPI ranks but CommInit() has not been called
    PushTestVector();             // (collective with several ranks: the communicator exists by now)
    int e = hymls_b200_initialize(h_);
    if (e == 0) e = hymls_b200_set_row_map(h_, (int64_t)gids_.size(), gids_.data());  // vectors live on the row map
    initialized_ = (e == 0);
    return e;
  }
  int Compute() {
    int e = hymls_b200_compute(h_);
    computed_ = (e == 0);
    return e;
  }
  bool IsInitialized() const { return initialized_; }
  bool IsComputed() const { return computed_; }

  // Epetra_Operator
  int ApplyInverse(const Epetra_MultiVector& B, Epetra_MultiVector& X) const {
    return hymls_b200_apply_inverse_map(h_, B.Values(), B.Stride(), X.Values(), X.Stride(), B.NumVectors(),
                                        HYMLS_B200_HOST);
  }
  int Apply(const Epetra_MultiVector&, Epetra_MultiVector&) const { return -1; }  // as the reference (:122-123)
  int SetUseTranspose(bool) { return -1; }                                        // (:162-166)
  bool UseTranspose() const { return false; }
  bool HasNormInf() const { return false; }
  double NormInf() const { return -1.0; }
  const char* Label() const { return "HYMLS::B200Preconditioner"; }
  const Epetra_Comm& Comm() const { return K_->Comm(); }
  const Epetra_Map& OperatorDomainMap() const { return K_->OperatorDomainMap(); }
  const Epetra_Map& OperatorRangeMap() const { return K_->OperatorRangeMap(); }
  const Epetra_RowMatrix& Matrix() const { return *K_; }

  // BorderedOperator (src/HYMLS_Preconditioner.cpp:844-918, 930-1070); Compute() must follow SetBorder
  int SetBorder(Teuchos::RCP<const Epetra_MultiVector> V, Teuchos::RCP<const Epetra_MultiVector> W = Teuchos::null,
                Teuchos::RCP<const Epetra_SerialDenseMatrix> C = Teuchos::null) {
    computed_ = false;
    if (V == Teuchos::null) return hymls_b200_set_border(h_, nullptr, nullptr, nullptr, 0);
    const int m = V->NumVectors(), n = V->MyLength();
    std::vector<double> v((size_t)n * m), w, c;
    for (int j = 0; j < m; ++j) std::copy((*V)[j], (*V)[j] + n, v.begin() + (size_t)j * n);
    if (W != Teuchos::null) {
      w.resize((size_t)n * m);
      for (int j = 0; j < m; ++j) std::copy((*W)[j], (*W)[j] + n, w.begin() + (size_t)j * n);
    }
    if (C != Teuchos::null) {
      c.resize((size_t)m * m);
      for (int j = 0; j < m; ++j)
        for (int i = 0; i < m; ++i) c[i + (size_t)j * m] = (*C)(i, j);
    }
    return hymls_b200_set_border_dist(h_, (int64_t)gids_.size(), gids_.data(), v.data(), w.empty() ? nullptr : w.data(),
                                      c.empty() ? nullptr : c.data(), m);
  }
  // [Y; S] = [K V; W' C] \ [X; T]
  int ApplyInverse(const Epetra_MultiVector& X, const Epetra_SerialDenseMatrix& T, Epetra_MultiVector& Y,
                   Epetra_SerialDenseMatrix& S) const {
    std::vector<double> t((size_t)T.M() * T.N()), s(t.size());
    for (int j = 0; j < T.N(); ++j)
      for (int i = 0; i < T.M(); ++i) t[i + (size_t)j * T.M()] = T(i, j);
    int e = hymls_b200_apply_inverse_bordered_map(h_, X.Values(), X.Stride(), t.data(), Y.Values(), Y.Stride(),
                                                  s.data(), X.NumVectors(), HYMLS_B200_HOST);
    for (int j = 0; j < S.N(); ++j)
      for (int i = 0; i < S.M(); ++i) S(i, j) = s[i + (size_t)j * S.M()];
    return e;
  }
  int Apply(const Epetra_MultiVector&, const Epetra_SerialDenseMatrix&, Epetra_MultiVector&,
            Epetra_SerialDenseMatrix&) const { return -1; }

  // Ifpack counters (src/HYMLS_Preconditioner.cpp:612-717)
  int NumInitialize() const { return Stats().num_initialize; }
  int NumCompute() const { return Stats().num_compute; }
  int NumApplyInverse() const { return Stats().num_apply_inverse; }
  double InitializeTime() const { return Stats().time_initialize; }
  double ComputeTime() const { return Stats().time_compute; }
  double ApplyInverseTime() const { return Stats().time_apply_inverse; }
  double InitializeFlops() const { return 0.0; }
  double ComputeFlops() const { return Stats().flops_compute; }
  double ApplyInverseFlops() const { return 0.0; }
  double Condest(const Ifpack_CondestType = Ifpack_Cheap, const int = 1550, const double = 1e-9,
                 Epetra_RowMatrix* = 0) { return -1.0; }
  double Condest() const { return -1.0; }
  std::ostream& Print(std::ostream& os) const { return os << Label() << " (" << hymls_b200_version() << ")\n"; }

  // HYMLS::Solver-side helpers when the device Krylov solve replaces the Belos loop (see HYMLS_B200_Solver.hpp)
  int SetTolerance(double tol) { return hymls_b200_set_tolerance(h_, tol); }  // BaseSolver::SetTolerance
  std::string FinalParameterListXml() const {                                  // "Store Final Parameter List"
    std::string s((size_t)hymls_b200_get_parameters_xml(h_, nullptr, 0) + 1, '\0');
    hymls_b200_get_parameters_xml(h_, &s[0], (int64_t)s.size());
    s.resize(s.size() - 1);
    return s;
  }
  hymls_b200_t* Handle() const { return h_; }

 private:
  // rows of this rank with their global ids: Epetra_CrsMatrix::ExtractMyRowView + RowMap().GID64 + GCID64
  int PushMatrix() {
    const int n = K_->NumMyRows();
    gids_.resize(n);
    for (int i = 0; i < n; ++i) gids_[i] = (int64_t)K_->RowMap().GID64(i);
    if (K_->Comm().NumProc() > 1 && commPending_) return 0;  // gathered in CommInit()
    std::vector<int64_t> ptr(n + 1, 0), col;
    std::vector<double> val;
    col.reserve(K_->NumMyNonzeros());
    val.reserve(K_->NumMyNonzeros());
    for (int i = 0; i < n; ++i) {
      int len;
      double* v;
      int* c;
      K_->ExtractMyRowView(i, len, v, c);
      for (int k = 0; k < len; ++k) {
        col.push_back((int64_t)K_->GCID64(c[k]));
        val.push_back(v[k]);
      }
      ptr[i + 1] = (int64_t)col.size();
    }
    return hymls_b200_set_matrix_csr_dist(h_, (int64_t)K_->NumGlobalRows64(), n, gids_.data(), ptr.data(), col.data(),
                                          val.data());
  }
  void PushTestVector() {
    if (testVector_ == Teuchos::null || testVectorPushed_) return;
    if (K_->Comm().NumProc() > 1 && commPending_) return;
    Check(hymls_b200_set_testvector_dist(h_, (int64_t)gids_.size(), gids_.data(), testVector_->Values()));
    testVectorPushed_ = true;
  }
  hymls_b200_stats Stats() const {
    hymls_b200_stats st;
    hymls_b200_get_stats(h_, &st);
    return st;
  }
  void Check(int e) const {
    if (e) Tools::Error(hymls_b200_last_error(), __FILE__, __LINE__);
  }
  hymls_b200_t* h_ = nullptr;
  Teuchos::RCP<const Epetra_CrsMatrix> K_;
  Teuchos::RCP<Teuchos::ParameterList> params_;
  Teuchos::RCP<Epetra_Vector> testVector_;
  std::vector<int64_t> gids_;  // global ids of the rows of this rank (the matrix' row map)
  bool initialized_ = false, computed_ = false, testVectorPushed_ = false;
  bool commPending_ = false;   // several MPI ranks: the matrix is gathered once the NCCL communicator exists
};

}  // namespace HYMLS
#endif

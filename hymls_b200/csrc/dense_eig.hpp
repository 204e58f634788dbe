// Small dense linear algebra on the host for the GCRO-DR restart (dense_eig.cpp): plain C++, single-threaded and
// deterministic, so every rank that feeds the same (all-reduced) entries gets bitwise the same results.  All matrices
// are column major.
#pragma once

extern "C" {
// Real nonsymmetric eigenproblem A v = lambda v (n x n): Householder reduction to Hessenberg form, Francis double-shift
// QR, eigenvectors by back-substitution.  wr / wi: eigenvalues; a complex pair sits in two consecutive entries with
// wi > 0 first, and its columns j, j + 1 of V hold the real and imaginary part of the eigenvector of wr + i wi.
// Returns 0, or 1 when the QR iteration did not converge.
int hy_eig(int n, const double* A, double* wr, double* wi, double* V);
// In-place Cholesky A = L L' (lower triangle); 1 when a pivot is not above n eps max_i A_ii (numerically singular).
int hy_cholesky(int n, double* A);
// Householder QR A = Q R of an m x n matrix (m >= n), diagonal of R >= 0.  Returns 1 when R is rank deficient:
// |R_jj| <= rankTol max_i |R_ii| for some j.
int hy_qr(int m, int n, const double* A, double* Q, double* R, double rankTol);
// Harmonic Ritz vectors of GCRO-DR: the generalized problem A z = theta B z (n x n, A symmetric positive definite) is
// reduced to the standard problem L^-1 B L^-T w = mu w (mu = 1/theta, A = L L', z = L^-T w), and the k vectors of
// the smallest |theta| are returned in P (n x kOut).  A complex pair is kept whole as its real and imaginary parts,
// so kOut is k or k + 1; when k + 1 exceeds kMax the straddling pair is left out (kOut = k - 1).  Returns 0, 1 when
// the Cholesky factorisation fails, 2 when the eigen-solver does not converge.
int hy_harmonic_ritz(int n, const double* A, const double* B, int k, int kMax, double* P, int* kOut);
}

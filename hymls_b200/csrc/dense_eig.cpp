// Host dense eigensolver and QR for the GCRO-DR restart (see dense_eig.hpp).  The nonsymmetric eigensolver follows
// the published EISPACK routines orthes / hqr2 (in the form of the public-domain JAMA EigenvalueDecomposition):
// Householder reduction to upper Hessenberg form with the transformations accumulated, Francis double-shift QR to
// real Schur form, and eigenvectors by back-substitution followed by the back-transformation.
#include "dense_eig.hpp"

#include <algorithm>
#include <cmath>
#include <vector>

namespace {

struct Mat {  // column major n x n
  int n;
  std::vector<double> a;
  explicit Mat(int n_) : n(n_), a((size_t)n_ * n_, 0.0) {}
  double& operator()(int i, int j) { return a[(size_t)j * n + i]; }
};

void cdiv(double xr, double xi, double yr, double yi, double& cr, double& ci) {
  double r, d;
  if (std::fabs(yr) > std::fabs(yi)) {
    r = yi / yr;
    d = yr + r * yi;
    cr = (xr + r * xi) / d;
    ci = (xi - r * xr) / d;
  } else {
    r = yr / yi;
    d = yi + r * yr;
    cr = (r * xr + xi) / d;
    ci = (r * xi - xr) / d;
  }
}

// Householder reduction to Hessenberg form; V accumulates the transformations
void orthes(Mat& H, Mat& V) {
  const int n = H.n, low = 0, high = n - 1;
  std::vector<double> ort(n, 0.0);
  for (int m = low + 1; m <= high - 1; ++m) {
    double scale = 0.0;
    for (int i = m; i <= high; ++i) scale += std::fabs(H(i, m - 1));
    if (scale == 0.0) continue;
    double h = 0.0;
    for (int i = high; i >= m; --i) {
      ort[i] = H(i, m - 1) / scale;
      h += ort[i] * ort[i];
    }
    double g = std::sqrt(h);
    if (ort[m] > 0) g = -g;
    h -= ort[m] * g;
    ort[m] -= g;
    for (int j = m; j < n; ++j) {
      double f = 0.0;
      for (int i = high; i >= m; --i) f += ort[i] * H(i, j);
      f /= h;
      for (int i = m; i <= high; ++i) H(i, j) -= f * ort[i];
    }
    for (int i = 0; i <= high; ++i) {
      double f = 0.0;
      for (int j = high; j >= m; --j) f += ort[j] * H(i, j);
      f /= h;
      for (int j = m; j <= high; ++j) H(i, j) -= f * ort[j];
    }
    ort[m] *= scale;
    H(m, m - 1) = scale * g;
  }
  for (int i = 0; i < n; ++i)
    for (int j = 0; j < n; ++j) V(i, j) = i == j ? 1.0 : 0.0;
  for (int m = high - 1; m >= low + 1; --m) {
    if (H(m, m - 1) == 0.0) continue;
    for (int i = m + 1; i <= high; ++i) ort[i] = H(i, m - 1);
    for (int j = m; j <= high; ++j) {
      double g = 0.0;
      for (int i = m; i <= high; ++i) g += ort[i] * V(i, j);
      g = (g / ort[m]) / H(m, m - 1);  // double division avoids possible underflow
      for (int i = m; i <= high; ++i) V(i, j) += g * ort[i];
    }
  }
}

// real Schur form by Francis double-shift QR, then the eigenvectors; false when the iteration does not converge
bool hqr2(Mat& H, Mat& V, std::vector<double>& d, std::vector<double>& e) {
  const int nn = H.n, low = 0, high = nn - 1;
  int n = nn - 1;
  const double eps = std::ldexp(1.0, -52);
  double exshift = 0.0, p = 0, q = 0, r = 0, s = 0, z = 0, t, w, x, y;
  double norm = 0.0;
  for (int i = 0; i < nn; ++i)
    for (int j = std::max(i - 1, 0); j < nn; ++j) norm += std::fabs(H(i, j));
  int iter = 0, total = 0;
  while (n >= low) {
    int l = n;
    while (l > low) {
      s = std::fabs(H(l - 1, l - 1)) + std::fabs(H(l, l));
      if (s == 0.0) s = norm;
      if (H(l, l - 1) == 0.0 || std::fabs(H(l, l - 1)) < eps * s) break;
      --l;
    }
    if (l == n) {  // one root
      H(n, n) += exshift;
      d[n] = H(n, n);
      e[n] = 0.0;
      --n;
      iter = 0;
    } else if (l == n - 1) {  // two roots
      w = H(n, n - 1) * H(n - 1, n);
      p = (H(n - 1, n - 1) - H(n, n)) / 2.0;
      q = p * p + w;
      z = std::sqrt(std::fabs(q));
      H(n, n) += exshift;
      H(n - 1, n - 1) += exshift;
      x = H(n, n);
      if (q >= 0) {  // real pair
        z = p >= 0 ? p + z : p - z;
        d[n - 1] = x + z;
        d[n] = d[n - 1];
        if (z != 0.0) d[n] = x - w / z;
        e[n - 1] = 0.0;
        e[n] = 0.0;
        x = H(n, n - 1);
        s = std::fabs(x) + std::fabs(z);
        p = x / s;
        q = z / s;
        r = std::sqrt(p * p + q * q);
        p /= r;
        q /= r;
        for (int j = n - 1; j < nn; ++j) {
          z = H(n - 1, j);
          H(n - 1, j) = q * z + p * H(n, j);
          H(n, j) = q * H(n, j) - p * z;
        }
        for (int i = 0; i <= n; ++i) {
          z = H(i, n - 1);
          H(i, n - 1) = q * z + p * H(i, n);
          H(i, n) = q * H(i, n) - p * z;
        }
        for (int i = low; i <= high; ++i) {
          z = V(i, n - 1);
          V(i, n - 1) = q * z + p * V(i, n);
          V(i, n) = q * V(i, n) - p * z;
        }
      } else {  // complex pair
        d[n - 1] = x + p;
        d[n] = x + p;
        e[n - 1] = z;
        e[n] = -z;
      }
      n -= 2;
      iter = 0;
    } else {  // no convergence yet
      if (++total > 60 * nn) return false;
      x = H(n, n);
      y = 0.0;
      w = 0.0;
      if (l < n) {
        y = H(n - 1, n - 1);
        w = H(n, n - 1) * H(n - 1, n);
      }
      if (iter == 10) {  // Wilkinson's ad hoc shift
        exshift += x;
        for (int i = low; i <= n; ++i) H(i, i) -= x;
        s = std::fabs(H(n, n - 1)) + std::fabs(H(n - 1, n - 2));
        x = y = 0.75 * s;
        w = -0.4375 * s * s;
      }
      if (iter == 30) {  // MATLAB's ad hoc shift
        s = (y - x) / 2.0;
        s = s * s + w;
        if (s > 0) {
          s = std::sqrt(s);
          if (y < x) s = -s;
          s = x - w / ((y - x) / 2.0 + s);
          for (int i = low; i <= n; ++i) H(i, i) -= s;
          exshift += s;
          x = y = w = 0.964;
        }
      }
      ++iter;
      // two consecutive small sub-diagonal elements
      int m = n - 2;
      while (m >= l) {
        z = H(m, m);
        r = x - z;
        s = y - z;
        p = (r * s - w) / H(m + 1, m) + H(m, m + 1);
        q = H(m + 1, m + 1) - z - r - s;
        r = H(m + 2, m + 1);
        s = std::fabs(p) + std::fabs(q) + std::fabs(r);
        p /= s;
        q /= s;
        r /= s;
        if (m == l) break;
        if (std::fabs(H(m, m - 1)) * (std::fabs(q) + std::fabs(r)) <
            eps * (std::fabs(p) * (std::fabs(H(m - 1, m - 1)) + std::fabs(z) + std::fabs(H(m + 1, m + 1)))))
          break;
        --m;
      }
      for (int i = m + 2; i <= n; ++i) {
        H(i, i - 2) = 0.0;
        if (i > m + 2) H(i, i - 3) = 0.0;
      }
      // double QR step on rows l..n and columns m..n
      for (int k = m; k <= n - 1; ++k) {
        const bool notlast = k != n - 1;
        if (k != m) {
          p = H(k, k - 1);
          q = H(k + 1, k - 1);
          r = notlast ? H(k + 2, k - 1) : 0.0;
          x = std::fabs(p) + std::fabs(q) + std::fabs(r);
          if (x == 0.0) continue;
          p /= x;
          q /= x;
          r /= x;
        }
        s = std::sqrt(p * p + q * q + r * r);
        if (p < 0) s = -s;
        if (s != 0) {
          if (k != m) H(k, k - 1) = -s * x;
          else if (l != m) H(k, k - 1) = -H(k, k - 1);
          p += s;
          x = p / s;
          y = q / s;
          z = r / s;
          q /= p;
          r /= p;
          for (int j = k; j < nn; ++j) {
            p = H(k, j) + q * H(k + 1, j);
            if (notlast) {
              p += r * H(k + 2, j);
              H(k + 2, j) -= p * z;
            }
            H(k, j) -= p * x;
            H(k + 1, j) -= p * y;
          }
          for (int i = 0; i <= std::min(n, k + 3); ++i) {
            p = x * H(i, k) + y * H(i, k + 1);
            if (notlast) {
              p += z * H(i, k + 2);
              H(i, k + 2) -= p * r;
            }
            H(i, k) -= p;
            H(i, k + 1) -= p * q;
          }
          for (int i = low; i <= high; ++i) {
            p = x * V(i, k) + y * V(i, k + 1);
            if (notlast) {
              p += z * V(i, k + 2);
              V(i, k + 2) -= p * r;
            }
            V(i, k) -= p;
            V(i, k + 1) -= p * q;
          }
        }
      }
    }
  }
  if (norm == 0.0) return true;
  // back-substitution: eigenvectors of the quasi-triangular form
  for (n = nn - 1; n >= 0; --n) {
    p = d[n];
    q = e[n];
    if (q == 0) {  // real vector
      int l = n;
      H(n, n) = 1.0;
      for (int i = n - 1; i >= 0; --i) {
        w = H(i, i) - p;
        r = 0.0;
        for (int j = l; j <= n; ++j) r += H(i, j) * H(j, n);
        if (e[i] < 0.0) {
          z = w;
          s = r;
        } else {
          l = i;
          if (e[i] == 0.0) {
            H(i, n) = w != 0.0 ? -r / w : -r / (eps * norm);
          } else {
            x = H(i, i + 1);
            y = H(i + 1, i);
            q = (d[i] - p) * (d[i] - p) + e[i] * e[i];
            t = (x * s - z * r) / q;
            H(i, n) = t;
            H(i + 1, n) = std::fabs(x) > std::fabs(z) ? (-r - w * t) / x : (-s - y * t) / z;
          }
          t = std::fabs(H(i, n));  // overflow control
          if ((eps * t) * t > 1)
            for (int j = i; j <= n; ++j) H(j, n) /= t;
        }
      }
    } else if (q < 0) {  // complex vector (the pair's second entry)
      int l = n - 1;
      if (std::fabs(H(n, n - 1)) > std::fabs(H(n - 1, n))) {
        H(n - 1, n - 1) = q / H(n, n - 1);
        H(n - 1, n) = -(H(n, n) - p) / H(n, n - 1);
      } else {
        cdiv(0.0, -H(n - 1, n), H(n - 1, n - 1) - p, q, H(n - 1, n - 1), H(n - 1, n));
      }
      H(n, n - 1) = 0.0;
      H(n, n) = 1.0;
      for (int i = n - 2; i >= 0; --i) {
        double ra = 0.0, sa = 0.0, vr, vi;
        for (int j = l; j <= n; ++j) {
          ra += H(i, j) * H(j, n - 1);
          sa += H(i, j) * H(j, n);
        }
        w = H(i, i) - p;
        if (e[i] < 0.0) {
          z = w;
          r = ra;
          s = sa;
        } else {
          l = i;
          if (e[i] == 0) {
            cdiv(-ra, -sa, w, q, H(i, n - 1), H(i, n));
          } else {
            x = H(i, i + 1);
            y = H(i + 1, i);
            vr = (d[i] - p) * (d[i] - p) + e[i] * e[i] - q * q;
            vi = (d[i] - p) * 2.0 * q;
            if (vr == 0.0 && vi == 0.0)
              vr = eps * norm * (std::fabs(w) + std::fabs(q) + std::fabs(x) + std::fabs(y) + std::fabs(z));
            cdiv(x * r - z * ra + q * sa, x * s - z * sa - q * ra, vr, vi, H(i, n - 1), H(i, n));
            if (std::fabs(x) > std::fabs(z) + std::fabs(q)) {
              H(i + 1, n - 1) = (-ra - w * H(i, n - 1) + q * H(i, n)) / x;
              H(i + 1, n) = (-sa - w * H(i, n) - q * H(i, n - 1)) / x;
            } else {
              cdiv(-r - y * H(i, n - 1), -s - y * H(i, n), z, q, H(i + 1, n - 1), H(i + 1, n));
            }
          }
          t = std::max(std::fabs(H(i, n - 1)), std::fabs(H(i, n)));  // overflow control
          if ((eps * t) * t > 1)
            for (int j = i; j <= n; ++j) {
              H(j, n - 1) /= t;
              H(j, n) /= t;
            }
        }
      }
    }
  }
  // back-transformation to the eigenvectors of the original matrix
  std::vector<double> col(nn);
  for (int j = nn - 1; j >= low; --j) {
    for (int i = low; i <= high; ++i) {
      double zz = 0.0;
      for (int k = low; k <= std::min(j, high); ++k) zz += V(i, k) * H(k, j);
      col[i] = zz;
    }
    for (int i = low; i <= high; ++i) V(i, j) = col[i];
  }
  return true;
}

}  // namespace

extern "C" {

int hy_eig(int n, const double* A, double* wr, double* wi, double* V) {
  if (n <= 0) return 0;
  Mat H(n), Q(n);
  std::copy(A, A + (size_t)n * n, H.a.begin());
  orthes(H, Q);
  std::vector<double> d(n, 0.0), e(n, 0.0);
  if (!hqr2(H, Q, d, e)) return 1;
  std::copy(d.begin(), d.end(), wr);
  std::copy(e.begin(), e.end(), wi);
  std::copy(Q.a.begin(), Q.a.end(), V);
  return 0;
}

int hy_cholesky(int n, double* A) {
  double dmax = 0.0;
  for (int i = 0; i < n; ++i) dmax = std::max(dmax, std::fabs(A[(size_t)i * n + i]));
  const double floor = n * std::ldexp(1.0, -52) * dmax;
  for (int j = 0; j < n; ++j) {
    double s = A[(size_t)j * n + j];
    for (int k = 0; k < j; ++k) s -= A[(size_t)k * n + j] * A[(size_t)k * n + j];
    if (!(s > floor)) return 1;
    const double ljj = std::sqrt(s);
    A[(size_t)j * n + j] = ljj;
    for (int i = j + 1; i < n; ++i) {
      double t = A[(size_t)j * n + i];
      for (int k = 0; k < j; ++k) t -= A[(size_t)k * n + i] * A[(size_t)k * n + j];
      A[(size_t)j * n + i] = t / ljj;
    }
    for (int i = 0; i < j; ++i) A[(size_t)j * n + i] = 0.0;  // upper triangle cleared
  }
  return 0;
}

int hy_qr(int m, int n, const double* A, double* Q, double* R, double rankTol) {
  std::vector<double> W(A, A + (size_t)m * n), vs((size_t)m * n, 0.0), beta(n, 0.0);
  for (int j = 0; j < n; ++j) {
    double* a = &W[(size_t)j * m];
    double nrm = 0.0;
    for (int i = j; i < m; ++i) nrm = std::hypot(nrm, a[i]);
    double* v = &vs[(size_t)j * m];
    if (nrm == 0.0) continue;
    const double alpha = a[j] > 0 ? -nrm : nrm;
    for (int i = j; i < m; ++i) v[i] = a[i];
    v[j] -= alpha;
    double vv = 0.0;
    for (int i = j; i < m; ++i) vv += v[i] * v[i];
    beta[j] = vv > 0 ? 2.0 / vv : 0.0;
    for (int c = j; c < n; ++c) {  // W <- (I - beta v v') W
      double* wc = &W[(size_t)c * m];
      double t = 0.0;
      for (int i = j; i < m; ++i) t += v[i] * wc[i];
      t *= beta[j];
      for (int i = j; i < m; ++i) wc[i] -= t * v[i];
    }
  }
  // Q = H_0 ... H_{n-1} [I; 0]
  for (int c = 0; c < n; ++c) {
    double* q = &Q[(size_t)c * m];
    for (int i = 0; i < m; ++i) q[i] = i == c ? 1.0 : 0.0;
    for (int j = n - 1; j >= 0; --j) {
      const double* v = &vs[(size_t)j * m];
      double t = 0.0;
      for (int i = j; i < m; ++i) t += v[i] * q[i];
      t *= beta[j];
      for (int i = j; i < m; ++i) q[i] -= t * v[i];
    }
  }
  for (int c = 0; c < n; ++c)
    for (int i = 0; i < n; ++i) R[(size_t)c * n + i] = i <= c ? W[(size_t)c * m + i] : 0.0;
  double rmax = 0.0;
  for (int j = 0; j < n; ++j) {  // positive diagonal: flip row j of R and column j of Q
    if (R[(size_t)j * n + j] < 0) {
      for (int c = j; c < n; ++c) R[(size_t)c * n + j] = -R[(size_t)c * n + j];
      for (int i = 0; i < m; ++i) Q[(size_t)j * m + i] = -Q[(size_t)j * m + i];
    }
    rmax = std::max(rmax, R[(size_t)j * n + j]);
  }
  for (int j = 0; j < n; ++j)
    if (!(R[(size_t)j * n + j] > rankTol * rmax)) return 1;
  return 0;
}

int hy_harmonic_ritz(int n, const double* A, const double* B, int k, int kMax, double* P, int* kOut) {
  *kOut = 0;
  if (n <= 0 || k <= 0) return 0;
  k = std::min(k, n);
  std::vector<double> L(A, A + (size_t)n * n);
  if (hy_cholesky(n, L.data())) return 1;
  auto Lat = [&](int i, int j) { return L[(size_t)j * n + i]; };
  // X = L^-1 B (columns), then S' = L^-1 X'  ->  S = L^-1 B L^-T
  std::vector<double> X(B, B + (size_t)n * n), S((size_t)n * n);
  for (int c = 0; c < n; ++c) {
    double* x = &X[(size_t)c * n];
    for (int i = 0; i < n; ++i) {
      double t = x[i];
      for (int j = 0; j < i; ++j) t -= Lat(i, j) * x[j];
      x[i] = t / Lat(i, i);
    }
  }
  for (int r = 0; r < n; ++r) {  // row r of X -> solve -> row r of S
    std::vector<double> y(n);
    for (int i = 0; i < n; ++i) {
      double t = X[(size_t)i * n + r];
      for (int j = 0; j < i; ++j) t -= Lat(i, j) * y[j];
      y[i] = t / Lat(i, i);
    }
    for (int i = 0; i < n; ++i) S[(size_t)i * n + r] = y[i];
  }
  std::vector<double> wr(n), wi(n), W((size_t)n * n);
  if (hy_eig(n, S.data(), wr.data(), wi.data(), W.data())) return 2;
  // largest |mu| = smallest |theta|; ties keep the eigen-solver's order
  std::vector<int> order(n);
  for (int i = 0; i < n; ++i) order[i] = i;
  std::vector<double> mod(n);
  for (int i = 0; i < n; ++i) mod[i] = std::hypot(wr[i], wi[i]);
  std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return mod[a] > mod[b]; });
  auto partner = [&](int i) { return wi[i] > 0 ? i + 1 : wi[i] < 0 ? i - 1 : i; };
  std::vector<char> chosen(n, 0);
  for (int q = 0; q < k; ++q) chosen[order[q]] = 1;
  int count = k;
  for (int q = 0; q < k; ++q) {
    const int i = order[q], j = partner(i);
    if (!chosen[j]) {
      chosen[j] = 1;
      ++count;
      if (count > kMax) {  // the pair straddles k and does not fit: leave it out
        chosen[i] = chosen[j] = 0;
        count -= 2;
      }
    }
  }
  // columns in the selection order: a real vector, or the real and imaginary part of a pair (wi > 0 column first)
  int col = 0;
  std::vector<char> done(n, 0);
  for (int q = 0; q < n; ++q) {
    const int i = order[q];
    if (!chosen[i] || done[i]) continue;
    const int j0 = wi[i] < 0 ? i - 1 : i;
    const int ncol = wi[i] != 0 ? 2 : 1;
    for (int c = 0; c < ncol; ++c) {
      const double* w = &W[(size_t)(j0 + c) * n];
      double* z = &P[(size_t)col * n];
      for (int r = n - 1; r >= 0; --r) {  // z = L^-T w
        double t = w[r];
        for (int s = r + 1; s < n; ++s) t -= Lat(s, r) * z[s];
        z[r] = t / Lat(r, r);
      }
      ++col;
    }
    done[i] = done[partner(i)] = 1;
  }
  *kOut = col;
  return 0;
}

}  // extern "C"

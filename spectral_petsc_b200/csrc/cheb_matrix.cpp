#include "cheb_matrix.h"

#include <cmath>

namespace sb200 {

static std::vector<long double> cgl_diff_matrix_ld(int P) {
  const int n = P - 1;
  std::vector<long double> D((size_t)P * P, 0.0L);
  if (n < 1) return D;
  const long double pi = 3.14159265358979323846264338327950288L;
  auto cbar = [n](int i) { return (i == 0 || i == n) ? 2.0L : 1.0L; };
  for (int i = 0; i <= n; i++) {
    for (int j = 0; j <= n; j++) {
      long double v;
      if (i != j) {
        // x_i - x_j = cos(a) - cos(b) = -2 sin((a+b)/2) sin((a-b)/2)
        long double sp = sinl(pi * (long double)(i + j) / (2.0L * n));
        long double sm = sinl(pi * (long double)(i - j) / (2.0L * n));
        long double dx = -2.0L * sp * sm;
        long double sgn = ((i + j) & 1) ? -1.0L : 1.0L;
        v = (cbar(i) / cbar(j)) * sgn / dx;
      } else if (i == 0) {
        v = (2.0L * n * n + 1.0L) / 6.0L;
      } else if (i == n) {
        v = -(2.0L * n * n + 1.0L) / 6.0L;
      } else if (2 * i == n) {
        v = 0.0L;  // x_i = 0 at the middle node of an odd P; cosl(pi * i / n) would leave about 1e-20 here
      } else {
        long double s = sinl(pi * (long double)i / n);
        long double c = cosl(pi * (long double)i / n);
        v = -c / (2.0L * s * s);
      }
      D[(size_t)i * P + j] = v;
    }
  }
  return D;
}

std::vector<double> cgl_diff_matrix(int P) {
  std::vector<long double> L = cgl_diff_matrix_ld(P);
  std::vector<double> D(L.size());
  for (size_t k = 0; k < L.size(); k++) D[k] = (double)L[k];
  return D;
}

void cgl_even_odd(int P, std::vector<double>& Ae, std::vector<double>& Bo) {
  const int n = P - 1, h = P / 2;
  std::vector<long double> L = cgl_diff_matrix_ld(P);
  Ae.assign((size_t)h * h, 0.0);
  Bo.assign((size_t)h * h, 0.0);
  for (int i = 0; i < h; i++)
    for (int j = 0; j < h; j++) {
      const long double p = L[(size_t)i * P + j], q = L[(size_t)i * P + (n - j)];
      Ae[(size_t)i * h + j] = (double)(0.5L * (p + q));
      Bo[(size_t)i * h + j] = (double)(0.5L * (p - q));
    }
}

// Any P >= 2: hh = ceil(P/2) pair rows (pair j couples nodes j and n-j; for odd P the last pair is the middle node
// with itself), zero padded to HP x HP.  With s_j = u_j + u_{n-j}, d_j = u_j - u_{n-j} formed for EVERY pair the same way, the
// self-paired middle node gives s = 2 u_c, d = 0, so its column of Ae carries D[i][c]/2 (an exact scaling) and its column of Bo
// is zero; the middle ROW has a = 0 identically (D[c][n-j] = -D[c][j]) and is set to zero, its value is b alone.
void cgl_even_odd_padded(int P, int HP, std::vector<double>& Ae, std::vector<double>& Bo) {
  const int n = P - 1, hh = (P + 1) / 2;
  std::vector<long double> L = cgl_diff_matrix_ld(P);
  Ae.assign((size_t)HP * HP, 0.0);
  Bo.assign((size_t)HP * HP, 0.0);
  for (int i = 0; i < hh; i++)
    for (int j = 0; j < hh; j++) {
      const long double p = L[(size_t)i * P + j], q = L[(size_t)i * P + (n - j)];
      const bool midcol = (j == n - j), midrow = (i == n - i);
      long double a = 0.5L * (p + q), b = 0.5L * (p - q);
      if (midcol) { a = 0.5L * p; b = 0.0L; }
      if (midrow) a = 0.0L;
      Ae[(size_t)i * HP + j] = (double)a;
      Bo[(size_t)i * HP + j] = (double)b;
    }
}

}  // namespace sb200

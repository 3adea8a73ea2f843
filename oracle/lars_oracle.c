/*
 * lars_oracle.c -- plain-C (double) restatement of the ONMF step's CPU algorithm.
 *
 * TEST INFRASTRUCTURE ONLY: loaded through ctypes by tests/ (the checker at sizes where the numpy
 * restatement in oracle/onmf_oracle.py is too slow) and by bench.py's cpu_baseline leg.  Never linked
 * or called by the product package.
 *
 * Follows, function by function:
 *   oracle_lars_positive  sklearn/linear_model/_least_angle.py:415-917 (_lars_path_solver: Gram mode,
 *                         method='lasso', positive=True, return_path=False) as reached from the
 *                         reference's src/ontf.py:79-86 via sklearn/decomposition/_dict_learning.py:118-135
 *                         (alpha/n_features scaling) and LassoLars._fit (:1136-1153, one path per sample)
 *   oracle_sparse_code    the per-sample loop + gram/cov products (_dict_learning.py:422,426)
 *   oracle_update_dict    reference src/ontf.py:91-115
 *   oracle_aggregate      reference src/ontf.py:141-148
 * Validated against scikit-learn 1.9.0 and the reference's golden fixtures by tests/test_oracle.py.
 */
#include <float.h>
#include <math.h>
#include <stdlib.h>
#include <string.h>

#define TINY32 1.1754943508222875e-38
#define EPS32 1.1920928955078125e-07
#define EPS64 2.220446049250313e-16

static double min_pos_init(void) { return DBL_MAX; }

/* Cholesky factor L (row-major, leading dim ld) of the active Gram block. */
static double chol_append(double* L, int ld, int s, const double* G, int k, const int* act, int j) {
  double* row = L + (size_t)s * ld;
  double v = 0.0;
  for (int i = 0; i < s; ++i) {
    double t = G[(size_t)j * k + act[i]];
    const double* Li = L + (size_t)i * ld;
    for (int q = 0; q < i; ++q) t -= Li[q] * row[q];
    row[i] = t / Li[i];
    v += row[i] * row[i];
  }
  double piv = sqrt(fabs(G[(size_t)j * k + j] - v));
  if (piv < EPS64) piv = EPS64;
  row[s] = piv;
  return piv;
}

static void chol_solve_ones(const double* L, int ld, int s, double* x) {
  for (int i = 0; i < s; ++i) {
    double t = 1.0;
    const double* Li = L + (size_t)i * ld;
    for (int q = 0; q < i; ++q) t -= Li[q] * x[q];
    x[i] = t / Li[i];
  }
  for (int i = s - 1; i >= 0; --i) {
    double t = x[i];
    for (int q = i + 1; q < s; ++q) t -= L[(size_t)q * ld + i] * x[q];
    x[i] = t / L[(size_t)i * ld + i];
  }
}

static void chol_delete(double* L, int ld, int s, int out) {
  for (int i = out; i < s - 1; ++i) memcpy(L + (size_t)i * ld, L + (size_t)(i + 1) * ld, sizeof(double) * (i + 2));
  for (int i = out; i < s - 1; ++i) {
    double a = L[(size_t)i * ld + i], b = L[(size_t)i * ld + i + 1];
    double r = hypot(a, b), c = 1.0, sn = 0.0;
    if (r != 0.0) { c = a / r; sn = b / r; }
    L[(size_t)i * ld + i] = r;
    L[(size_t)i * ld + i + 1] = 0.0;
    for (int q = i + 1; q < s - 1; ++q) {
      double x = L[(size_t)q * ld + i], y = L[(size_t)q * ld + i + 1];
      L[(size_t)q * ld + i] = c * x + sn * y;
      L[(size_t)q * ld + i + 1] = c * y - sn * x;
    }
  }
}

/* relative gap of the two smallest of a, b (a <= b) */
static double rel_gap(double a, double b) { return (b - a) / (fabs(b) > 0.0 ? fabs(b) : 1.0); }

/* One column.  G (k x k), c (k) -> coef (k).  Returns status bits (1 degenerate, 2 alpha-increase, 4 max_iter);
 * info[0]=n_iter, info[1]=max_active, info[2]=drops if info != NULL.  min_gap (if not NULL): min_gap[0] = the smallest
 * relative gap, over the knots, between the joining covariance and the runner-up, and between the shortest drop step and
 * the join / full step or the next drop -- a near-tie, where rounding may change the path; min_gap[1] = the smallest
 * pivot^2 / G_jj of an accepted join (a nearly dependent atom: whether it passes the 1e-7 pivot rule is up to rounding
 * when this is small).  work: caller scratch of
 * (k+1)*(k+1) + 6*k doubles and 2*k ints. */
int oracle_lars_positive(const double* G, const double* c, int k, int d, double reg, int max_iter, double* coef,
                         int* info, double* work, int* iwork, double* min_gap) {
  const int ld = k + 1;
  double* L = work;
  double* cov = L + (size_t)ld * ld;
  double* prev = cov + k;
  double* w = prev + k;
  double* corr = w + k;
  double* cur = corr + k;
  int* act = iwork;        /* ordered like the factor */
  int* inact = iwork + k;  /* ordered like sklearn's shortened Cov (tie-breaking) */
  int n_act = 0, n_in = k, n_iter = 0, drop = 0, status = 0, max_act = 0, drops = 0;
  double a_cur = 0.0, a_prev = 0.0;
  const double amin = reg / d;
  double gap = INFINITY, minsig = INFINITY;
  memcpy(cov, c, sizeof(double) * k);
  for (int i = 0; i < k; ++i) { cur[i] = 0.0; prev[i] = 0.0; inact[i] = i; }
  for (;;) {
    int pos = -1;
    double C = 0.0;
    if (n_in > 0) {
      pos = 0;
      C = cov[inact[0]];
      for (int i = 1; i < n_in; ++i)
        if (cov[inact[i]] > C) { C = cov[inact[i]]; pos = i; }
      if (!drop && C / d > amin + EPS32)
        for (int i = 0; i < n_in; ++i)
          if (i != pos) { double g = rel_gap(cov[inact[i]], C); if (g < gap) gap = g; }
    }
    a_cur = C / d;
    if (a_cur <= amin + EPS32) {
      if (fabs(a_cur - amin) > EPS32 && n_iter > 0) {
        double ss = (a_prev - amin) / (a_prev - a_cur);
        for (int i = 0; i < k; ++i) cur[i] = prev[i] + ss * (cur[i] - prev[i]);
      }
      break;
    }
    if (n_iter >= max_iter || n_act >= k) {
      if (n_iter >= max_iter) status |= 4;
      break;
    }
    if (!drop) {
      int t = inact[pos]; inact[pos] = inact[0]; inact[0] = t;
      int j = inact[0];
      double piv = chol_append(L, ld, n_act, G, k, act, j);
      if (piv < 1e-7) {
        cov[j] = 0.0;
        t = inact[pos]; inact[pos] = inact[0]; inact[0] = t;
        status |= 1;
        continue;
      }
      if (piv * piv / G[(size_t)j * k + j] < minsig) minsig = piv * piv / G[(size_t)j * k + j];
      memmove(inact, inact + 1, sizeof(int) * (n_in - 1));
      --n_in;
      act[n_act++] = j;
      if (n_act > max_act) max_act = n_act;
    }
    if (n_iter > 0 && a_prev < a_cur) { status |= 2; break; }
    chol_solve_ones(L, ld, n_act, w);
    double sw = 0.0;
    for (int i = 0; i < n_act; ++i) sw += w[i];
    const double AA = 1.0 / sqrt(sw);
    for (int i = 0; i < n_act; ++i) w[i] *= AA;
    double g1 = min_pos_init();
    for (int i = 0; i < n_in; ++i) {
      const double* Gi = G + (size_t)inact[i] * k;
      double a = 0.0;
      for (int q = 0; q < n_act; ++q) a += Gi[act[q]] * w[q];
      a = rint(a * 1e15) / 1e15; /* np.around(decimals=15) */
      corr[i] = a;
      double v = (C - cov[inact[i]]) / (AA - a + TINY32);
      if (v > 0.0 && v < g1) g1 = v;
    }
    double gamma = C / AA;
    if (g1 < gamma) gamma = g1;
    double zpos = min_pos_init(), z2 = min_pos_init();
    int zi = -1;
    for (int q = 0; q < n_act; ++q) {
      double z = -cur[act[q]] / (w[q] + TINY32);
      if (z > 0.0 && z < zpos) { z2 = zpos; zpos = z; zi = q; } else if (z > 0.0 && z < z2) z2 = z;
    }
    /* a drop against the join / full step, or against a second drop, decides the knot and drop counts */
    if (zpos < min_pos_init()) {
      double g = zpos < gamma ? rel_gap(zpos, gamma) : rel_gap(gamma, zpos);
      if (z2 < min_pos_init() && rel_gap(zpos, z2) < g) g = rel_gap(zpos, z2);
      if (g < gap) gap = g;
    }
    drop = 0;
    if (zpos < gamma) { gamma = zpos; drop = 1; }
    ++n_iter;
    a_prev = a_cur;
    memcpy(prev, cur, sizeof(double) * k);
    memset(cur, 0, sizeof(double) * k);
    for (int q = 0; q < n_act; ++q) cur[act[q]] = prev[act[q]] + gamma * w[q];
    for (int i = 0; i < n_in; ++i) cov[inact[i]] -= gamma * corr[i];
    if (drop) {
      ++drops;
      chol_delete(L, ld, n_act, zi);
      int jd = act[zi];
      memmove(act + zi, act + zi + 1, sizeof(int) * (n_act - zi - 1));
      --n_act;
      double t = c[jd];
      const double* Gj = G + (size_t)jd * k;
      for (int i = 0; i < k; ++i) t -= Gj[i] * cur[i];
      cov[jd] = t;
      memmove(inact + 1, inact, sizeof(int) * n_in);
      inact[0] = jd;
      ++n_in;
    }
  }
  memcpy(coef, cur, sizeof(double) * k);
  if (info) { info[0] = n_iter; info[1] = max_act; info[2] = drops; }
  if (min_gap) { min_gap[0] = gap; min_gap[1] = minsig; }
  return status;
}

/* X (d x n) row-major, W (d x k) row-major -> H (k x n) row-major.  Returns the OR of the status bits. */
int oracle_sparse_code(const double* X, const double* W, int d, int n, int k, double reg, int max_iter, double* H) {
  double* G = (double*)malloc(sizeof(double) * k * k);
  double* cv = (double*)malloc(sizeof(double) * k);
  double* h = (double*)malloc(sizeof(double) * k);
  double* work = (double*)malloc(sizeof(double) * ((size_t)(k + 1) * (k + 1) + 6 * k));
  int* iwork = (int*)malloc(sizeof(int) * 2 * k);
  int status = 0;
  for (int a = 0; a < k; ++a)
    for (int b = 0; b < k; ++b) {
      double s = 0.0;
      for (int f = 0; f < d; ++f) s += W[(size_t)f * k + a] * W[(size_t)f * k + b];
      G[(size_t)a * k + b] = s;
    }
  for (int j = 0; j < n; ++j) {
    for (int a = 0; a < k; ++a) {
      double s = 0.0;
      for (int f = 0; f < d; ++f) s += W[(size_t)f * k + a] * X[(size_t)f * n + j];
      cv[a] = s;
    }
    status |= oracle_lars_positive(G, cv, k, d, reg, max_iter, h, NULL, work, iwork, NULL);
    for (int a = 0; a < k; ++a) H[(size_t)a * n + j] = h[a];
  }
  free(G); free(cv); free(h); free(work); free(iwork);
  return status;
}

/* W (d x k), A (k x k), B (k x d), all row-major; W updated in place. */
void oracle_update_dict(double* W, const double* A, const double* B, int d, int k) {
  double* col = (double*)malloc(sizeof(double) * d);
  for (int j = 0; j < k; ++j) {
    const double c = 1.0 / (A[(size_t)j * k + j] + 1.0);
    double nrm = 0.0;
    for (int f = 0; f < d; ++f) {
      double dot = 0.0;
      for (int q = 0; q < k; ++q) dot += W[(size_t)f * k + q] * A[(size_t)q * k + j];
      double v = W[(size_t)f * k + j] - c * (dot - B[(size_t)j * d + f]);
      if (v < 0.0) v = 0.0;
      col[f] = v;
      nrm += v * v;
    }
    nrm = sqrt(nrm);
    const double sc = 1.0 / (nrm > 1.0 ? nrm : 1.0);
    for (int f = 0; f < d; ++f) W[(size_t)f * k + j] = sc * col[f];
  }
  free(col);
}

/* A = (1-w) A + w H H^T ; B = (1-w) B + w H X^T ; H (k x n), X (d x n) row-major. */
void oracle_aggregate(double* A, double* B, const double* H, const double* X, int d, int n, int k, double w) {
  for (int a = 0; a < k; ++a) {
    for (int b = 0; b < k; ++b) {
      double s = 0.0;
      for (int j = 0; j < n; ++j) s += H[(size_t)a * n + j] * H[(size_t)b * n + j];
      A[(size_t)a * k + b] = (1.0 - w) * A[(size_t)a * k + b] + w * s;
    }
    for (int f = 0; f < d; ++f) {
      double s = 0.0;
      for (int j = 0; j < n; ++j) s += H[(size_t)a * n + j] * X[(size_t)f * n + j];
      B[(size_t)a * d + f] = (1.0 - w) * B[(size_t)a * d + f] + w * s;
    }
  }
}

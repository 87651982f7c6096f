// downstream.cu -- the frozen-embedding evaluation: 10-fold scoring of exported embeddings.
//
// Replaces (reference file:line):
//   TopKRanker(LogisticRegression(C=1000)) per fold     gcc/tasks/node_classification.py:54-90
//   SVC(C=100000), gamma='scale', one-vs-one, libsvm    gcc/tasks/graph_classification.py:46-66
//   argsort of e2 . e1[q] for every shared key          gcc/tasks/similarity_search.py:40-70
// The reference runs sklearn on the host, one fold and one binary problem after the other.  Here one
// launch solves every (fold, class) or (fold, class pair) problem, one CTA each; the host passes a fold
// id per row.  Every quantity that decides a prediction is fp64, like sklearn and libsvm.
#include <math.h>

#include "common.cuh"

namespace gccb {

#define DS_THREADS 256
#define DS_TAU 1e-12   // libsvm's TAU: floor of a non-positive quadratic coefficient
// a / b without the slow-path subroutine of IEEE division (its call forces spills in the solver loops):
// reciprocal estimate, two Newton steps and a residual correction -- correctly rounded for the normal-range
// operands met here
__device__ __forceinline__ double ddiv(double a, double b) {
#ifdef GCCB_EMU
  return a / b;
#else
  double r;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(b));
  double e = fma(-b, r, 1.0);
  r = fma(r, e, r);
  e = fma(-b, r, 1.0);
  r = fma(r, e, r);
  const double q = a * r;
  return fma(fma(-b, q, a), r, q);
#endif
}

__device__ __forceinline__ double block_sum_dbl(double v, double* red) {
  v = warp_sum_d(v);
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = blockDim.x >> 5;
  __syncthreads();
  if (lane == 0) red[w] = v;
  __syncthreads();
  double s = 0.0;
  for (int i = 0; i < nw; ++i) s += red[i];   // fixed order: every thread gets the same bits
  return s;
}

__device__ __forceinline__ double block_max_dbl(double v, double* red) {
  for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = blockDim.x >> 5;
  __syncthreads();
  if (lane == 0) red[w] = v;
  __syncthreads();
  double s = red[0];
  for (int i = 1; i < nw; ++i) s = fmax(s, red[i]);
  return s;
}

// (value, index) arg-reduction over the block: the larger value wins (sign = +1) or the smaller
// (sign = -1); a tie goes to the larger index, which is what libsvm's `>=` / `<=` scans select.
__device__ __forceinline__ void block_arg_dbl(double& v, int& idx, double sign, double* redv, int* redi) {
  for (int o = 16; o > 0; o >>= 1) {
    double ov = __shfl_xor_sync(0xffffffffu, v, o);
    int oi = __shfl_xor_sync(0xffffffffu, idx, o);
    if (sign * ov > sign * v || (ov == v && oi > idx)) { v = ov; idx = oi; }
  }
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = blockDim.x >> 5;
  __syncthreads();
  if (lane == 0) { redv[w] = v; redi[w] = idx; }
  __syncthreads();
  v = redv[0];
  idx = redi[0];
  for (int i = 1; i < nw; ++i)
    if (sign * redv[i] > sign * v || (redv[i] == v && redi[i] > idx)) { v = redv[i]; idx = redi[i]; }
}

// ---------------------------------------------------------------------------------------------------
// a. one-vs-rest L2 logistic regression, Newton with backtracking.  Problem (fold f, class c):
//    min_w,b  1/2 |w|^2 + C sum_{i: fold_i != f} log(1 + exp(-s_i (w.x_i + b))),  s_i = +1 iff label_i == c.
//    The intercept is not penalised (sklearn's lbfgs).  Hessian X~^T D X~ + diag(1..1, 0) in the workspace
//    (257^2 doubles at d = 256 do not fit in shared memory), Cholesky and both triangular solves in the CTA.

__device__ __forceinline__ double sigmoid_d(double z) {
  if (z >= 0.0) return ddiv(1.0, 1.0 + exp(-z));
  const double e = exp(z);
  return ddiv(e, 1.0 + e);
}
// log(1 + exp(-m)) without overflow
__device__ __forceinline__ double log1pexp_neg(double m) {
  return m > 0.0 ? log1p(exp(-m)) : -m + log1p(exp(m));
}
__device__ __forceinline__ double xt(const float* X, int d, int i, int j) {   // [x_i, 1]
  return j < d ? (double)X[(size_t)i * d + j] : 1.0;
}

__host__ __device__ inline size_t lr_problem_doubles(int n, int d) {
  const size_t m = (size_t)d + 1;
  return m * m + 4 * (size_t)n + 2 * m;
}

__global__ void __launch_bounds__(DS_THREADS, 1)
logreg_newton_kernel(const float* __restrict__ X, const int32_t* __restrict__ label,
                     const int32_t* __restrict__ fold, int n, int d, int n_classes, double Creg, int max_iter,
                     double tol, double* __restrict__ W, int32_t* __restrict__ status, double* __restrict__ ws) {
  const int prob = blockIdx.x, f = prob / n_classes, c = prob % n_classes;
  const int m = d + 1, tid = threadIdx.x, nt = blockDim.x;
  double* H = ws + (size_t)prob * lr_problem_doubles(n, d);
  double* Dw = H + (size_t)m * m;   // C s (1 - s) of the training rows, 0 for test rows
  double* r = Dw + n;               // C (s - y)
  double* z = r + n;                // margins w.x~
  double* u = z + n;                // step . x~
  double* dl = u + n;               // Newton step
  double* g = dl + m;               // gradient
  double* w = W + (size_t)prob * m;
  __shared__ double red[32];
  __shared__ double xa[32][16], xb[32][16], dd[32];

  double np_ = 0.0, nt_ = 0.0;
  for (int i = tid; i < n; i += nt)
    if (fold[i] != f) { nt_ += 1.0; np_ += label[i] == c; }
  const double npos = block_sum_dbl(np_, red), ntrain = block_sum_dbl(nt_, red);
  for (int j = tid; j < m; j += nt) w[j] = 0.0;
  for (int i = tid; i < n; i += nt) z[i] = 0.0;
  if (npos == 0.0 || npos == ntrain) {   // sklearn's _ConstantPredictor: probability 0 or 1 everywhere
    if (tid == 0) status[prob] = npos == 0.0 ? 3 : 4;
    return;
  }
  double F = 0.0;
  for (int i = tid; i < n; i += nt)
    if (fold[i] != f) F += log1pexp_neg(0.0);
  F = Creg * block_sum_dbl(F, red);
  int st = 1;
  for (int it = 0; it < max_iter; ++it) {
    for (int i = tid; i < n; i += nt) {
      if (fold[i] != f) {
        const double s = sigmoid_d(z[i]);
        Dw[i] = Creg * s * (1.0 - s);
        r[i] = Creg * (s - (label[i] == c ? 1.0 : 0.0));
      } else {
        Dw[i] = 0.0;
        r[i] = 0.0;
      }
    }
    __syncthreads();
    for (int j = tid; j < m; j += nt) {              // gradient: w + sum_i r_i x~_i (rows coalesced over j)
      double acc = 0.0;
      for (int i = 0; i < n; ++i) acc += r[i] * xt(X, d, i, j);
      g[j] = (j < d ? w[j] : 0.0) + acc;
    }
    // Hessian, lower triangle, 16 x 16 tiles over 32-row chunks
    const int nb = (m + 15) / 16, ty = tid >> 4, tx = tid & 15;
    for (int ti = 0; ti < nb; ++ti)
      for (int tj = 0; tj <= ti; ++tj) {
        double acc = 0.0;
        for (int i0 = 0; i0 < n; i0 += 32) {
          for (int e = tid; e < 32 * 16; e += nt) {
            const int rr = e >> 4, cc = e & 15, i = i0 + rr;
            const int ja = ti * 16 + cc, jb = tj * 16 + cc;
            xa[rr][cc] = (i < n && ja < m) ? xt(X, d, i, ja) : 0.0;
            xb[rr][cc] = (i < n && jb < m) ? xt(X, d, i, jb) : 0.0;
          }
          if (tid < 32) dd[tid] = i0 + tid < n ? Dw[i0 + tid] : 0.0;
          __syncthreads();
          for (int rr = 0; rr < 32; ++rr) acc += dd[rr] * xa[rr][ty] * xb[rr][tx];
          __syncthreads();
        }
        const int a = ti * 16 + ty, b = tj * 16 + tx;
        if (a < m && b < m && b <= a) H[(size_t)a * m + b] = acc + ((a == b && a < d) ? 1.0 : 0.0);
      }
    __syncthreads();
    // Cholesky H = L L^T in place (lower triangle)
    for (int k = 0; k < m; ++k) {
      if (tid == 0) {
        double v = H[(size_t)k * m + k];
        if (!(v > 1e-300)) v = 1e-300;   // a fully saturated intercept column: keep the factor finite
        H[(size_t)k * m + k] = sqrt(v);
      }
      __syncthreads();
      const double piv = H[(size_t)k * m + k];
      for (int a = k + 1 + tid; a < m; a += nt) H[(size_t)a * m + k] = ddiv(H[(size_t)a * m + k], piv);
      __syncthreads();
      const int R = m - k - 1;
      for (int e = tid; e < R * R; e += nt) {
        const int a = k + 1 + e / R, b = k + 1 + e % R;
        if (b <= a) H[(size_t)a * m + b] -= H[(size_t)a * m + k] * H[(size_t)b * m + k];
      }
      __syncthreads();
    }
    // L y = -g, then L^T dl = y
    for (int j = tid; j < m; j += nt) dl[j] = -g[j];
    __syncthreads();
    for (int k = 0; k < m; ++k) {
      if (tid == 0) dl[k] = ddiv(dl[k], H[(size_t)k * m + k]);
      __syncthreads();
      const double yk = dl[k];
      for (int a = k + 1 + tid; a < m; a += nt) dl[a] -= H[(size_t)a * m + k] * yk;
      __syncthreads();
    }
    for (int k = m - 1; k >= 0; --k) {
      if (tid == 0) dl[k] = ddiv(dl[k], H[(size_t)k * m + k]);
      __syncthreads();
      const double xk = dl[k];
      for (int a = tid; a < k; a += nt) dl[a] -= H[(size_t)k * m + a] * xk;
      __syncthreads();
    }
    double part = 0.0;
    for (int j = tid; j < m; j += nt) part -= g[j] * dl[j];
    const double lam2 = block_sum_dbl(part, red);    // Newton decrement squared: g^T H^-1 g
    // u_i = dl . x~_i, one warp per row
    {
      const int lane = tid & 31, wp = tid >> 5, nw = nt >> 5;
      for (int i = wp; i < n; i += nw) {
        double acc = 0.0;
        for (int j = lane; j < m; j += 32) acc += dl[j] * xt(X, d, i, j);
        acc = warp_sum_d(acc);
        if (lane == 0) u[i] = acc;
      }
    }
    __syncthreads();
    if (lam2 * 0.5 <= tol * fmax(1.0, F)) {          // converged: the last (tiny) full Newton step is taken
      for (int j = tid; j < m; j += nt) w[j] += dl[j];
      for (int i = tid; i < n; i += nt) z[i] += u[i];
      st = 0;
      break;
    }
    double t = 1.0, Ft = 0.0;
    bool ok = false;
    for (int ls = 0; ls < 60; ++ls) {
      double loss = 0.0, reg = 0.0;
      for (int i = tid; i < n; i += nt)
        if (fold[i] != f) {
          const double s = label[i] == c ? 1.0 : -1.0;
          loss += log1pexp_neg(s * (z[i] + t * u[i]));
        }
      for (int j = tid; j < d; j += nt) {
        const double wj = w[j] + t * dl[j];
        reg += wj * wj;
      }
      Ft = Creg * block_sum_dbl(loss, red) + 0.5 * block_sum_dbl(reg, red);
      if (Ft <= F - 0.25 * t * lam2) { ok = true; break; }
      t *= 0.5;
    }
    if (!ok) { st = 2; break; }                      // no decrease left at fp64 resolution
    for (int j = tid; j < m; j += nt) w[j] += t * dl[j];
    for (int i = tid; i < n; i += nt) z[i] += t * u[i];
    F = Ft;
    __syncthreads();
  }
  if (tid == 0) status[prob] = st;
}

// per-row class probabilities of the row's own fold model and the top-1 class (ties -> highest index)
__global__ void __launch_bounds__(DS_THREADS)
logreg_predict_kernel(const float* __restrict__ X, const int32_t* __restrict__ fold, int n, int d, int n_classes,
                      const double* __restrict__ W, const int32_t* __restrict__ status, double* __restrict__ prob,
                      int32_t* __restrict__ pred) {
  const int lane = threadIdx.x & 31;
  const int i = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (i >= n) return;
  const int f = fold[i], m = d + 1;
  double best = -1.0;
  int bc = 0;
  for (int c = 0; c < n_classes; ++c) {
    const int pb = f * n_classes + c;
    const double* w = W + (size_t)pb * m;
    double acc = 0.0;
    for (int j = lane; j < d; j += 32) acc += (double)X[(size_t)i * d + j] * w[j];
    acc = warp_sum_d(acc);
    const int s = status[pb];
    const double p = s == 3 ? 0.0 : s == 4 ? 1.0 : sigmoid_d(acc + w[d]);
    if (p >= best) { best = p; bc = c; }
    if (lane == 0 && prob) prob[(size_t)i * n_classes + c] = p;
  }
  if (lane == 0) pred[i] = bc;
}

// ---------------------------------------------------------------------------------------------------
// b. RBF-kernel C-SVC, one-vs-one, libsvm's SMO (Fan, Chen & Lin 2005 working-set selection), no shrinking.
//    Squared distances |x_i|^2 + |x_j|^2 - 2 x_i.x_j are computed once in fp64 and stored as fp32 (libsvm
//    caches kernel values as float); problem (fold f, pair (ci < cj)) reads them with its own gamma.

__global__ void __launch_bounds__(DS_THREADS)
sqdist_kernel(const float* __restrict__ X, int n, int d, float* __restrict__ D2) {
  __shared__ double ta[16][17], tb[16][17];
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const int i = blockIdx.y * 16 + ty, j = blockIdx.x * 16 + tx;
  double dot = 0.0, sa = 0.0, sb = 0.0;
  for (int k0 = 0; k0 < d; k0 += 16) {
    const int ia = blockIdx.y * 16 + ty, ib = blockIdx.x * 16 + ty;
    ta[ty][tx] = (ia < n && k0 + tx < d) ? (double)X[(size_t)ia * d + k0 + tx] : 0.0;
    tb[ty][tx] = (ib < n && k0 + tx < d) ? (double)X[(size_t)ib * d + k0 + tx] : 0.0;
    __syncthreads();
    for (int k = 0; k < 16; ++k) {
      dot += ta[ty][k] * tb[tx][k];
      sa += ta[ty][k] * ta[ty][k];
      sb += tb[tx][k] * tb[tx][k];
    }
    __syncthreads();
  }
  if (i < n && j < n) D2[(size_t)i * n + j] = i == j ? 0.f : (float)(sa + sb - 2.0 * dot);
}

// gamma = 1 / (d * var(X_train)) per fold (sklearn gamma='scale'; two-pass variance like numpy)
__global__ void __launch_bounds__(DS_THREADS)
svc_gamma_kernel(const float* __restrict__ X, const int32_t* __restrict__ fold, int n, int d,
                 double* __restrict__ gamma) {
  __shared__ double red[32];
  const int f = blockIdx.x;
  double s = 0.0, cnt = 0.0;
  for (int i = 0; i < n; ++i) {
    if (fold[i] == f) continue;
    for (int j = threadIdx.x; j < d; j += blockDim.x) s += (double)X[(size_t)i * d + j];
    cnt += 1.0;
  }
  const double total = cnt * d;
  const double mean = block_sum_dbl(s, red) / total;
  double q = 0.0;
  for (int i = 0; i < n; ++i) {
    if (fold[i] == f) continue;
    for (int j = threadIdx.x; j < d; j += blockDim.x) {
      const double v = (double)X[(size_t)i * d + j] - mean;
      q += v * v;
    }
  }
  const double var = block_sum_dbl(q, red) / total;
  if (threadIdx.x == 0) gamma[f] = var != 0.0 ? 1.0 / (d * var) : 1.0;
}

struct SvcWs {
  int32_t* idx;
  int32_t* y;
  double* alpha;
  double* G;
  float* Qi;
};
// per problem: alpha, G (double), idx, y (int32), Qi (float); the stride is rounded up to 256 bytes so that
// every problem's doubles stay 8-byte aligned for odd n
__host__ __device__ inline size_t svc_problem_bytes(int64_t n) { return ((size_t)n * 28 + 255) & ~(size_t)255; }
__device__ __forceinline__ SvcWs svc_ws(void* base, int n, int prob) {
  char* p = (char*)base + (size_t)prob * svc_problem_bytes(n);
  SvcWs w;
  w.alpha = (double*)p;
  w.G = w.alpha + n;
  w.idx = (int32_t*)(w.G + n);
  w.y = w.idx + n;
  w.Qi = (float*)(w.y + n);
  return w;
}

__device__ __forceinline__ int2 pair_of(int pr, int k) {
  int a = 0;
  while (pr >= k - 1 - a) { pr -= k - 1 - a; ++a; }
  return make_int2(a, a + 1 + pr);
}

__global__ void __launch_bounds__(DS_THREADS, 1)
svc_smo_kernel(const float* __restrict__ D2, const int32_t* __restrict__ label, const int32_t* __restrict__ fold,
               int n, int n_classes, double Cc, double eps, long long max_iter, const double* __restrict__ gamma,
               double* __restrict__ coef, double* __restrict__ rho, double* __restrict__ obj,
               int32_t* __restrict__ status, void* __restrict__ wsbase) {
  const int n_pairs = n_classes * (n_classes - 1) / 2;
  const int prob = blockIdx.x, f = prob / n_pairs, pr = prob % n_pairs;
  const int tid = threadIdx.x, nt = blockDim.x;
  const int2 cc_ = pair_of(pr, n_classes);
  const int ci = cc_.x, cj = cc_.y;
  SvcWs W = svc_ws(wsbase, n, prob);
  const double gam = gamma[f];
  __shared__ int scan[33];
  __shared__ double redv[32];
  __shared__ int redi[32];
  __shared__ double sh_da[2];

  // problem rows: class ci (+1) then class cj (-1), each in dataset order (libsvm groups by class)
  int l = 0;
  for (int pass = 0; pass < 2; ++pass) {
    const int cls = pass ? cj : ci;
    for (int base = 0; base < n; base += nt) {
      const int i = base + tid;
      const int p = (i < n && fold[i] != f && label[i] == cls) ? 1 : 0;
      int tot;
      const int off = block_scan_excl(p, scan, &tot);
      if (p) { W.idx[l + off] = i; W.y[l + off] = pass ? -1 : 1; }
      l += tot;
    }
  }
  for (int p = tid; p < l; p += nt) { W.alpha[p] = 0.0; W.G[p] = -1.0; }
  for (int i = tid; i < n; i += nt) coef[(size_t)prob * n + i] = 0.0;
  __syncthreads();

  // i-selection: max over I_up of -y G  (ties -> last)
  double gmax = -INFINITY;
  int gi = -1;
  for (int p = tid; p < l; p += nt) {
    const double v = W.y[p] > 0 ? -W.G[p] : W.G[p];   // alpha = 0: only y = +1 rows are in I_up
    if (W.y[p] > 0 && v >= gmax) { gmax = v; gi = p; }
  }
  block_arg_dbl(gmax, gi, 1.0, redv, redi);
  int st = 1;
  long long it = 0;
  for (; it < max_iter; ++it) {
    if (gi < 0) { st = 0; break; }
    const int i = gi, yi = W.y[i];
    const size_t rowi = (size_t)W.idx[i] * n;
    double gmax2 = -INFINITY, omin = INFINITY;
    int jm = -1;
    for (int p = tid; p < l; p += nt) {
      const int yp = W.y[p];
      const float q = (float)(yi * yp * exp(-gam * (double)D2[rowi + W.idx[p]]));
      W.Qi[p] = q;
      const double a = W.alpha[p], Gp = W.G[p];
      if (yp > 0) {
        if (!(a <= 0.0)) {
          const double gd = gmax + Gp;
          if (Gp >= gmax2) gmax2 = Gp;
          if (gd > 0.0) {
            double qc = 2.0 - 2.0 * yi * (double)q;
            const double od = -ddiv(gd * gd, qc > 0.0 ? qc : DS_TAU);
            if (od <= omin) { omin = od; jm = p; }
          }
        }
      } else {
        if (!(a >= Cc)) {
          const double gd = gmax - Gp;
          if (-Gp >= gmax2) gmax2 = -Gp;
          if (gd > 0.0) {
            double qc = 2.0 + 2.0 * yi * (double)q;
            const double od = -ddiv(gd * gd, qc > 0.0 ? qc : DS_TAU);
            if (od <= omin) { omin = od; jm = p; }
          }
        }
      }
    }
    gmax2 = block_max_dbl(gmax2, redv);
    block_arg_dbl(omin, jm, -1.0, redv, redi);
    if (gmax + gmax2 < eps || jm < 0) { st = 0; break; }
    const int j = jm;
    if (tid == 0) {
      const double Qij = (double)W.Qi[j];
      const double oai = W.alpha[i], oaj = W.alpha[j];
      double ai = oai, aj = oaj;
      const double Gi = W.G[i], Gj = W.G[j];
      if (W.y[i] != W.y[j]) {
        double qc = 2.0 + 2.0 * Qij;
        if (qc <= 0.0) qc = DS_TAU;
        const double delta = ddiv(-Gi - Gj, qc), diff = ai - aj;
        ai += delta;
        aj += delta;
        if (diff > 0.0) { if (aj < 0.0) { aj = 0.0; ai = diff; } }
        else { if (ai < 0.0) { ai = 0.0; aj = -diff; } }
        if (diff > 0.0) { if (ai > Cc) { ai = Cc; aj = Cc - diff; } }   // C_i - C_j = 0
        else { if (aj > Cc) { aj = Cc; ai = Cc + diff; } }
      } else {
        double qc = 2.0 - 2.0 * Qij;
        if (qc <= 0.0) qc = DS_TAU;
        const double delta = ddiv(Gi - Gj, qc), sum = ai + aj;
        ai -= delta;
        aj += delta;
        if (sum > Cc) { if (ai > Cc) { ai = Cc; aj = sum - Cc; } }
        else { if (aj < 0.0) { aj = 0.0; ai = sum; } }
        if (sum > Cc) { if (aj > Cc) { aj = Cc; ai = sum - Cc; } }
        else { if (ai < 0.0) { ai = 0.0; aj = sum; } }
      }
      W.alpha[i] = ai;
      W.alpha[j] = aj;
      sh_da[0] = ai - oai;
      sh_da[1] = aj - oaj;
    }
    __syncthreads();
    const double dai = sh_da[0], daj = sh_da[1];
    const int yj = W.y[j];
    const size_t rowj = (size_t)W.idx[j] * n;
    gmax = -INFINITY;
    gi = -1;
    for (int p = tid; p < l; p += nt) {
      const int yp = W.y[p];
      const float qj = (float)(yj * yp * exp(-gam * (double)D2[rowj + W.idx[p]]));
      const double Gp = W.G[p] + (double)W.Qi[p] * dai + (double)qj * daj;
      W.G[p] = Gp;
      const double a = W.alpha[p];
      if (yp > 0) { if (!(a >= Cc) && -Gp >= gmax) { gmax = -Gp; gi = p; } }
      else { if (!(a <= 0.0) && Gp >= gmax) { gmax = Gp; gi = p; } }
    }
    block_arg_dbl(gmax, gi, 1.0, redv, redi);
  }
  // rho (libsvm calculate_rho) and the dual objective 1/2 sum alpha (G - 1)
  double ub = INFINITY, lb = -INFINITY, sfree = 0.0, nfree = 0.0, ov = 0.0;
  for (int p = tid; p < l; p += nt) {
    const double a = W.alpha[p], yG = W.y[p] * W.G[p];
    const bool up = a >= Cc, lo = a <= 0.0;
    if (up) { if (W.y[p] < 0) ub = fmin(ub, yG); else lb = fmax(lb, yG); }
    else if (lo) { if (W.y[p] > 0) ub = fmin(ub, yG); else lb = fmax(lb, yG); }
    else { nfree += 1.0; sfree += yG; }
    ov += a * (W.G[p] - 1.0);
    coef[(size_t)prob * n + W.idx[p]] = W.y[p] * a;
  }
  nfree = block_sum_dbl(nfree, redv);
  sfree = block_sum_dbl(sfree, redv);
  ov = block_sum_dbl(ov, redv);
  lb = block_max_dbl(lb, redv);
  ub = -block_max_dbl(-ub, redv);
  if (tid == 0) {
    rho[prob] = nfree > 0.0 ? ddiv(sfree, nfree) : 0.5 * (ub + lb);
    obj[prob] = 0.5 * ov;
    status[prob] = st;
  }
}

// libsvm vote over the pairs of the row's own fold: f > 0 votes for ci; ties -> the lowest class
__global__ void __launch_bounds__(DS_THREADS)
svc_predict_kernel(const float* __restrict__ D2, const int32_t* __restrict__ fold, int n, int n_classes,
                   const double* __restrict__ gamma, const double* __restrict__ coef, const double* __restrict__ rho,
                   double* __restrict__ dec, int32_t* __restrict__ pred) {
  __shared__ double red[32];
  __shared__ int votes[64];
  const int row = blockIdx.x, f = fold[row];
  const int n_pairs = n_classes * (n_classes - 1) / 2;
  const double gam = gamma[f];
  if (threadIdx.x < 64) votes[threadIdx.x] = 0;
  for (int pr = 0; pr < n_pairs; ++pr) {
    const int prob = f * n_pairs + pr;
    const double* cf = coef + (size_t)prob * n;
    double s = 0.0;
    for (int k = threadIdx.x; k < n; k += blockDim.x) {
      const double a = cf[k];
      if (a != 0.0) s += a * exp(-gam * (double)D2[(size_t)row * n + k]);
    }
    s = block_sum_dbl(s, red) - rho[prob];
    if (threadIdx.x == 0) {
      const int2 cc_ = pair_of(pr, n_classes);
      const int ci = cc_.x, cj = cc_.y;
      if (dec) dec[(size_t)row * n_pairs + pr] = s;
      ++votes[s > 0.0 ? ci : cj];
    }
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    int b = 0;
    for (int c = 1; c < n_classes; ++c)
      if (votes[c] > votes[b]) b = c;
    pred[row] = b;
  }
}

// ---------------------------------------------------------------------------------------------------
// c. similarity-search rank: rows normalised in fp64, rank[q] = #{c : e1[q].e2[c] > e1[q].e2[q]} over the
//    m shared keys.  Every score is the same sequential fma chain over k, so the true match never
//    outranks itself.

__global__ void __launch_bounds__(DS_THREADS)
sim_normalize_kernel(const float* __restrict__ E1, const float* __restrict__ E2, int d,
                     const int32_t* __restrict__ idx1, const int32_t* __restrict__ idx2, int m,
                     double* __restrict__ A, double* __restrict__ B) {
  const int lane = threadIdx.x & 31;
  const int r = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (r >= 2 * m) return;
  const int side = r >= m, q = side ? r - m : r;
  const float* src = side ? E2 + (size_t)idx2[q] * d : E1 + (size_t)idx1[q] * d;
  double* dst = (side ? B : A) + (size_t)q * d;
  double s = 0.0;
  for (int j = lane; j < d; j += 32) s += (double)src[j] * (double)src[j];
  const double nrm = sqrt(warp_sum_d(s));
  for (int j = lane; j < d; j += 32) dst[j] = (double)src[j] / nrm;
}

__global__ void __launch_bounds__(DS_THREADS)
sim_true_kernel(const double* __restrict__ A, const double* __restrict__ B, int m, int d, double* __restrict__ tr) {
  const int q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= m) return;
  double acc = 0.0;
  for (int k = 0; k < d; ++k) acc = fma(A[(size_t)q * d + k], B[(size_t)q * d + k], acc);
  tr[q] = acc;
}

// 64 queries x 64 candidates per CTA, 4 x 4 per thread, d in chunks of 16
__global__ void __launch_bounds__(DS_THREADS)
sim_rank_kernel(const double* __restrict__ A, const double* __restrict__ B, int m, int d,
                const double* __restrict__ tr, int32_t* __restrict__ rank) {
  __shared__ double sa[64][17], sb[64][17];
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const int q0 = blockIdx.y * 64, c0 = blockIdx.x * 64;
  double acc[4][4];
  for (int a = 0; a < 4; ++a)
    for (int b = 0; b < 4; ++b) acc[a][b] = 0.0;
  for (int k0 = 0; k0 < d; k0 += 16) {
    for (int e = threadIdx.x; e < 64 * 16; e += blockDim.x) {
      const int rr = e >> 4, kk = e & 15;
      sa[rr][kk] = (q0 + rr < m && k0 + kk < d) ? A[(size_t)(q0 + rr) * d + k0 + kk] : 0.0;
      sb[rr][kk] = (c0 + rr < m && k0 + kk < d) ? B[(size_t)(c0 + rr) * d + k0 + kk] : 0.0;
    }
    __syncthreads();
    const int kend = min(16, d - k0);
    for (int kk = 0; kk < kend; ++kk)
      for (int a = 0; a < 4; ++a)
        for (int b = 0; b < 4; ++b) acc[a][b] = fma(sa[ty + 16 * a][kk], sb[tx + 16 * b][kk], acc[a][b]);
    __syncthreads();
  }
  for (int a = 0; a < 4; ++a) {
    const int q = q0 + ty + 16 * a;
    if (q >= m) continue;
    const double t = tr[q];
    int cnt = 0;
    for (int b = 0; b < 4; ++b) cnt += (c0 + tx + 16 * b < m) && acc[a][b] > t;
    if (cnt) atomicAdd(&rank[q], cnt);
  }
}

}  // namespace gccb

using namespace gccb;

static size_t align256(size_t b) { return (b + 255) & ~(size_t)255; }

extern "C" size_t gccb_logreg_ovr_workspace(int32_t n, int32_t d, int32_t n_classes, int32_t n_folds) {
  if (n <= 0 || d <= 0 || n_classes <= 0 || n_folds <= 0) return 0;
  return align256((size_t)n_folds * n_classes * lr_problem_doubles(n, d) * sizeof(double));
}

extern "C" int gccb_logreg_ovr(const float* X, const int32_t* label, const int32_t* fold, int32_t n, int32_t d,
                               int32_t n_classes, int32_t n_folds, double C, int32_t max_iter, double tol,
                               double* weights, double* prob, int32_t* pred, int32_t* status, void* workspace,
                               size_t workspace_bytes, gccb_stream_t stream) {
  if (!X || !label || !fold || !weights || !pred || !status || !workspace || n <= 0 || d <= 0 ||
      n_classes <= 0 || n_folds <= 0 || !(C > 0.0) || max_iter <= 0) {
    set_last_error("gccb_logreg_ovr: bad argument");
    return GCCB_ERR_BADARG;
  }
  if (workspace_bytes < gccb_logreg_ovr_workspace(n, d, n_classes, n_folds)) {
    set_last_error("gccb_logreg_ovr: workspace too small");
    return GCCB_ERR_CAPACITY;
  }
  GCCB_LAUNCH(logreg_newton_kernel, n_folds * n_classes, DS_THREADS, 0, stream, X, label, fold, (int)n, (int)d,
              (int)n_classes, C, (int)max_iter, tol, weights, status, (double*)workspace);
  const int rows_per = DS_THREADS / 32;
  GCCB_LAUNCH(logreg_predict_kernel, (n + rows_per - 1) / rows_per, DS_THREADS, 0, stream, X, fold, (int)n, (int)d,
              (int)n_classes, (const double*)weights, (const int32_t*)status, prob, pred);
  return check_launch("gccb_logreg_ovr");
}

extern "C" size_t gccb_svc_ovo_workspace(int32_t n, int32_t n_classes, int32_t n_folds) {
  if (n <= 0 || n_classes < 2 || n_folds <= 0) return 0;
  const size_t P = (size_t)n_folds * (n_classes * (n_classes - 1) / 2);
  return align256((size_t)n * n * sizeof(float)) + align256(P * svc_problem_bytes(n));
}

extern "C" int gccb_svc_ovo(const float* X, const int32_t* label, const int32_t* fold, int32_t n, int32_t d,
                            int32_t n_classes, int32_t n_folds, double C, double eps, int64_t max_iter,
                            double* gamma, double* coef, double* rho, double* obj, double* dec, int32_t* pred,
                            int32_t* status, void* workspace, size_t workspace_bytes, gccb_stream_t stream) {
  if (!X || !label || !fold || !gamma || !coef || !rho || !obj || !pred || !status || !workspace || n <= 0 ||
      d <= 0 || n_classes < 2 || n_classes > 64 || n_folds <= 0 || !(C > 0.0) || !(eps > 0.0) || max_iter <= 0) {
    set_last_error("gccb_svc_ovo: bad argument");
    return GCCB_ERR_BADARG;
  }
  if (workspace_bytes < gccb_svc_ovo_workspace(n, n_classes, n_folds)) {
    set_last_error("gccb_svc_ovo: workspace too small");
    return GCCB_ERR_CAPACITY;
  }
  float* D2 = (float*)workspace;
  void* per = (char*)workspace + align256((size_t)n * n * sizeof(float));
  const int P = n_folds * (n_classes * (n_classes - 1) / 2);
  const dim3 tiles((n + 15) / 16, (n + 15) / 16);
  GCCB_LAUNCH(sqdist_kernel, tiles, DS_THREADS, 0, stream, X, (int)n, (int)d, D2);
  GCCB_LAUNCH(svc_gamma_kernel, n_folds, DS_THREADS, 0, stream, X, fold, (int)n, (int)d, gamma);
  GCCB_LAUNCH(svc_smo_kernel, P, DS_THREADS, 0, stream, (const float*)D2, label, fold, (int)n, (int)n_classes, C, eps,
              (long long)max_iter, (const double*)gamma, coef, rho, obj, status, per);
  GCCB_LAUNCH(svc_predict_kernel, n, DS_THREADS, 0, stream, (const float*)D2, fold, (int)n, (int)n_classes,
              (const double*)gamma, (const double*)coef, (const double*)rho, dec, pred);
  return check_launch("gccb_svc_ovo");
}

extern "C" size_t gccb_sim_rank_workspace(int32_t m, int32_t d) {
  if (m <= 0 || d <= 0) return 0;
  return align256((size_t)2 * m * d * sizeof(double)) + align256((size_t)m * sizeof(double));
}

extern "C" int gccb_sim_rank(const float* E1, const float* E2, int32_t d, const int32_t* idx1, const int32_t* idx2,
                             int32_t m, int32_t* rank, void* workspace, size_t workspace_bytes,
                             gccb_stream_t stream) {
  if (!E1 || !E2 || !idx1 || !idx2 || !rank || !workspace || d <= 0 || m <= 0) {
    set_last_error("gccb_sim_rank: bad argument");
    return GCCB_ERR_BADARG;
  }
  if (workspace_bytes < gccb_sim_rank_workspace(m, d)) {
    set_last_error("gccb_sim_rank: workspace too small");
    return GCCB_ERR_CAPACITY;
  }
  double* A = (double*)workspace;
  double* B = A + (size_t)m * d;
  double* tr = (double*)((char*)workspace + align256((size_t)2 * m * d * sizeof(double)));
  cudaMemsetAsync(rank, 0, (size_t)m * sizeof(int32_t), (cudaStream_t)stream);
  const int rows_per = DS_THREADS / 32;
  GCCB_LAUNCH(sim_normalize_kernel, (2 * m + rows_per - 1) / rows_per, DS_THREADS, 0, stream, E1, E2, (int)d, idx1,
              idx2, (int)m, A, B);
  GCCB_LAUNCH(sim_true_kernel, (m + DS_THREADS - 1) / DS_THREADS, DS_THREADS, 0, stream, (const double*)A,
              (const double*)B, (int)m, (int)d, tr);
  const dim3 tiles((m + 63) / 64, (m + 63) / 64);
  GCCB_LAUNCH(sim_rank_kernel, tiles, DS_THREADS, 0, stream, (const double*)A, (const double*)B, (int)m, (int)d,
              (const double*)tr, rank);
  return check_launch("gccb_sim_rank");
}

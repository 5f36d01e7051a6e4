// RANSAC homography estimation for batches of matched point sets: the cv2.findHomography(src, dst, cv2.RANSAC, t) call
// of eval_homography.py (the homography AUC) and eval_matches.py (the inlier count), on the device.
//
// The algorithm is the one oracle/ransac_oracle.py restates in numpy, and the results equal it bit for bit: every
// floating-point operation is an explicit round-to-nearest intrinsic in the restatement's order, every sum over points
// is 256 strided partials combined by a halving tree, and counts are integers.
//
//   k_ransac             one CTA per pair, persistent over waves of 256 hypotheses.  Each thread draws the sample of
//                        one hypothesis (counter-based splitmix64, so hypotheses are independent) and solves its DLT;
//                        each warp then scores its 32 hypotheses in turn with all lanes over the points.  After a wave
//                        one thread replays cv2's acceptance and stopping rule over the wave in hypothesis order, so
//                        hypotheses past the current iteration bound are discarded and the result does not depend on
//                        the wave size.
//   k_homography_refine  one CTA per pair: the inliers of the model, compacted in order with a block scan; the DLT refit
//                        and 10 Levenberg-Marquardt steps on them; the mask of the refined model.  Repeated (at most
//                        three rounds) while the refined model's inlier set grows.
#include <float.h>

#include <cmath>

#include "common.cuh"

namespace gims {
namespace {

constexpr int kThreads = 256;            // = the wave size = the number of strided partials of every sum
constexpr int kMaxAttempts = 1000;
constexpr int kMaxRetries = 64;
constexpr int kLmIters = 10;
constexpr int kRefitRounds = 3;
constexpr int kNormTerms = 44;           // 36 upper-triangle entries of AtA, then 8 of Atb
constexpr int kLmTerms = 45;             // 36 of JtJ, 8 of Jtr, the cost
constexpr double kPivotEps = 1e-12;

__device__ __forceinline__ double dm(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double da(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double ds(double a, double b) { return __dsub_rn(a, b); }
__device__ __forceinline__ double dd(double a, double b) { return __ddiv_rn(a, b); }

__device__ __forceinline__ uint64_t splitmix64(uint64_t x) {
  uint64_t z = x + 0x9E3779B97F4A7C15ull;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}

// cv2 HomographyEstimatorCallback::computeError in fp32 with h = (float)H[0..7]
__device__ __forceinline__ bool is_inlier(const float* h, float2 s, float2 d, float thr2) {
  const float ww = __fdiv_rn(1.0f, __fadd_rn(__fadd_rn(__fmul_rn(h[6], s.x), __fmul_rn(h[7], s.y)), 1.0f));
  const float dx = __fsub_rn(__fmul_rn(__fadd_rn(__fadd_rn(__fmul_rn(h[0], s.x), __fmul_rn(h[1], s.y)), h[2]), ww), d.x);
  const float dy = __fsub_rn(__fmul_rn(__fadd_rn(__fadd_rn(__fmul_rn(h[3], s.x), __fmul_rn(h[4], s.y)), h[5]), ww), d.y);
  return __fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)) <= thr2;
}

// element a of the two DLT rows of a normalised point (X, Y) -> (u, v), h33 = 1
__device__ __forceinline__ double dlt_r1(int a, double X, double Y, double uX, double uY) {
  return a == 0 ? X : a == 1 ? Y : a == 2 ? 1.0 : a < 6 ? 0.0 : a == 6 ? -uX : -uY;
}
__device__ __forceinline__ double dlt_r2(int a, double X, double Y, double vX, double vY) {
  return a < 3 ? 0.0 : a == 3 ? X : a == 4 ? Y : a == 5 ? 1.0 : a == 6 ? -vX : -vY;
}

// the 44 normal-equation terms of one point, t[q] for q in the fixed order
__device__ __forceinline__ void dlt_terms(double X, double Y, double u, double v, double* t) {
  const double uX = dm(u, X), uY = dm(u, Y), vX = dm(v, X), vY = dm(v, Y);
  int q = 0;
#pragma unroll
  for (int a = 0; a < 8; ++a)
#pragma unroll
    for (int c = a; c < 8; ++c)
      t[q++] = da(dm(dlt_r1(a, X, Y, uX, uY), dlt_r1(c, X, Y, uX, uY)), dm(dlt_r2(a, X, Y, vX, vY), dlt_r2(c, X, Y, vX, vY)));
#pragma unroll
  for (int a = 0; a < 8; ++a) t[36 + a] = da(dm(dlt_r1(a, X, Y, uX, uY), u), dm(dlt_r2(a, X, Y, vX, vY), v));
}

// Gaussian elimination with partial pivoting (first maximal |pivot|); a pivot <= 1e-12 max|diag| fails
__device__ bool solve8(double (*A)[8], double* b, double* x) {
  double dmax = 0.0;
  for (int i = 0; i < 8; ++i) { const double d = fabs(A[i][i]); if (d > dmax) dmax = d; }
  const double thr = dm(kPivotEps, dmax);
  for (int k = 0; k < 8; ++k) {
    int r = k;
    double best = fabs(A[k][k]);
    for (int i = k + 1; i < 8; ++i) { const double v = fabs(A[i][k]); if (v > best) { r = i; best = v; } }
    if (!(best > thr)) return false;
    if (r != k) {
      for (int j = 0; j < 8; ++j) { const double t = A[k][j]; A[k][j] = A[r][j]; A[r][j] = t; }
      const double t = b[k]; b[k] = b[r]; b[r] = t;
    }
    for (int i = k + 1; i < 8; ++i) {
      const double f = dd(A[i][k], A[k][k]);
      for (int j = k + 1; j < 8; ++j) A[i][j] = ds(A[i][j], dm(f, A[k][j]));
      b[i] = ds(b[i], dm(f, b[k]));
    }
  }
  for (int i = 7; i >= 0; --i) {
    double s = b[i];
    for (int j = i + 1; j < 8; ++j) s = ds(s, dm(A[i][j], x[j]));
    x[i] = dd(s, A[i][i]);
  }
  return true;
}

__device__ __forceinline__ void mat3(const double* a, const double* b, double* c) {
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j)
      c[3 * i + j] = da(da(dm(a[3 * i], b[j]), dm(a[3 * i + 1], b[3 + j])), dm(a[3 * i + 2], b[6 + j]));
}

struct Norm { double cxs, cys, cxd, cyd, sxs, sys, sxd, syd; };

// scales n / sum|x - c| from the four absolute-deviation sums; false if one is below DBL_EPSILON
__device__ __forceinline__ bool norm_scales(Norm& nm, double n, const double* sa) {
  for (int k = 0; k < 4; ++k)
    if (fabs(sa[k]) < DBL_EPSILON) return false;
  nm.sxs = dd(n, sa[0]); nm.sys = dd(n, sa[1]); nm.sxd = dd(n, sa[2]); nm.syd = dd(n, sa[3]);
  return true;
}

__device__ __forceinline__ void normalise(const Norm& nm, float2 s, float2 d, double& X, double& Y, double& u, double& v) {
  X = dm(ds((double)s.x, nm.cxs), nm.sxs);
  Y = dm(ds((double)s.y, nm.cys), nm.sys);
  u = dm(ds((double)d.x, nm.cxd), nm.sxd);
  v = dm(ds((double)d.y, nm.cyd), nm.syd);
}

// the normal equations' sums S[44] -> H (H[8] = 1); false on a failed or non-finite solve
__device__ bool dlt_finish(const Norm& nm, const double* S, double* H) {
  double A[8][8], b[8], h[8];
  int q = 0;
  for (int a = 0; a < 8; ++a)
    for (int c = a; c < 8; ++c) { A[a][c] = S[q]; A[c][a] = S[q]; ++q; }
  for (int a = 0; a < 8; ++a) b[a] = S[36 + a];
  if (!solve8(A, b, h)) return false;
  const double hn[9] = {h[0], h[1], h[2], h[3], h[4], h[5], h[6], h[7], 1.0};
  const double inv_dst[9] = {dd(1.0, nm.sxd), 0.0, nm.cxd, 0.0, dd(1.0, nm.syd), nm.cyd, 0.0, 0.0, 1.0};
  const double nrm_src[9] = {nm.sxs, 0.0, -dm(nm.cxs, nm.sxs), 0.0, nm.sys, -dm(nm.cys, nm.sys), 0.0, 0.0, 1.0};
  double t1[9], T[9];
  mat3(inv_dst, hn, t1);
  mat3(t1, nrm_src, T);
  bool ok = true;
  for (int j = 0; j < 9; ++j) { H[j] = dd(T[j], T[8]); ok &= isfinite(H[j]); }
  return ok;
}

// the fixed-order sum of four points: partials p = 0..3 hold 0 + t_p, the tree adds (t0 + t2) + (t1 + t3)
__device__ __forceinline__ double sum4(double t0, double t1, double t2, double t3) {
  return da(da(da(0.0, t0), da(0.0, t2)), da(da(0.0, t1), da(0.0, t3)));
}

// DLT of four correspondences, in one thread
__device__ bool dlt4(const float2* s, const float2* d, double* H) {
  Norm nm;
  nm.cxs = dd(sum4(s[0].x, s[1].x, s[2].x, s[3].x), 4.0);
  nm.cys = dd(sum4(s[0].y, s[1].y, s[2].y, s[3].y), 4.0);
  nm.cxd = dd(sum4(d[0].x, d[1].x, d[2].x, d[3].x), 4.0);
  nm.cyd = dd(sum4(d[0].y, d[1].y, d[2].y, d[3].y), 4.0);
  double sa[4];
  sa[0] = sum4(fabs(ds(s[0].x, nm.cxs)), fabs(ds(s[1].x, nm.cxs)), fabs(ds(s[2].x, nm.cxs)), fabs(ds(s[3].x, nm.cxs)));
  sa[1] = sum4(fabs(ds(s[0].y, nm.cys)), fabs(ds(s[1].y, nm.cys)), fabs(ds(s[2].y, nm.cys)), fabs(ds(s[3].y, nm.cys)));
  sa[2] = sum4(fabs(ds(d[0].x, nm.cxd)), fabs(ds(d[1].x, nm.cxd)), fabs(ds(d[2].x, nm.cxd)), fabs(ds(d[3].x, nm.cxd)));
  sa[3] = sum4(fabs(ds(d[0].y, nm.cyd)), fabs(ds(d[1].y, nm.cyd)), fabs(ds(d[2].y, nm.cyd)), fabs(ds(d[3].y, nm.cyd)));
  if (!norm_scales(nm, 4.0, sa)) return false;
  double S[kNormTerms], t[4][kNormTerms];
  for (int i = 0; i < 4; ++i) {
    double X, Y, u, v;
    normalise(nm, s[i], d[i], X, Y, u, v);
    dlt_terms(X, Y, u, v, t[i]);
  }
  for (int q = 0; q < kNormTerms; ++q) S[q] = sum4(t[0][q], t[1][q], t[2][q], t[3][q]);
  return dlt_finish(nm, S, H);
}

// cv2's haveCollinearPoints test for the triple (a, b, c), c as the last point: fp32 differences, fp64 rest
__device__ __forceinline__ bool collinear(const float2* p, int a, int b, int c) {
  const double dx1 = __fsub_rn(p[b].x, p[c].x), dy1 = __fsub_rn(p[b].y, p[c].y);
  const double dx2 = __fsub_rn(p[a].x, p[c].x), dy2 = __fsub_rn(p[a].y, p[c].y);
  const double lhs = fabs(ds(dm(dx2, dy1), dm(dy2, dx1)));
  const double rhs = dm((double)FLT_EPSILON, da(da(da(fabs(dx1), fabs(dy1)), fabs(dx2)), fabs(dy2)));
  return lhs <= rhs;
}

__device__ __forceinline__ double det3(const float2* p, int i0, int i1, int i2) {
  const double x0 = p[i0].x, x1 = p[i1].x, x2 = p[i2].x, y0 = p[i0].y, y1 = p[i1].y, y2 = p[i2].y;
  return da(ds(dm(x0, ds(y1, y2)), dm(y0, ds(x1, x2))), ds(dm(x1, y2), dm(x2, y1)));
}

// cv2 HomographyEstimatorCallback::checkSubset, with every triple tested for collinearity
__device__ bool subset_ok(const float2* s, const float2* d) {
  const int tri[4][3] = {{0, 1, 2}, {0, 1, 3}, {0, 2, 3}, {1, 2, 3}};
  for (int k = 0; k < 4; ++k)
    if (collinear(s, tri[k][0], tri[k][1], tri[k][2]) || collinear(d, tri[k][0], tri[k][1], tri[k][2])) return false;
  const int tt[4][3] = {{0, 1, 2}, {1, 2, 3}, {0, 2, 3}, {0, 1, 3}};
  int neg = 0;
  for (int k = 0; k < 4; ++k)
    neg += dm(det3(s, tt[k][0], tt[k][1], tt[k][2]), det3(d, tt[k][0], tt[k][1], tt[k][2])) < 0.0;
  return neg == 0 || neg == 4;
}

// the sample of hypothesis `hyp`: false if no attempt passes
__device__ bool draw_sample(uint64_t base, long long hyp, int m, const float2* src, const float2* dst, float2* s, float2* d) {
  const uint64_t mm = (uint64_t)m;
  for (int a = 0; a < kMaxAttempts; ++a) {
    const uint64_t att = (uint64_t)hyp * kMaxAttempts + (uint64_t)a;
    uint64_t idx[4];
    bool drew = true;
    for (int k = 0; k < 4 && drew; ++k) {
      drew = false;
      for (int r = 0; r < kMaxRetries; ++r) {
        const uint64_t cand = splitmix64(base + ((att * 4 + (uint64_t)k) * kMaxRetries + (uint64_t)r)) % mm;
        bool fresh = true;
        for (int j = 0; j < k; ++j) fresh &= cand != idx[j];
        if (fresh) { idx[k] = cand; drew = true; break; }
      }
    }
    if (!drew) continue;
    for (int k = 0; k < 4; ++k) { s[k] = src[idx[k]]; d[k] = dst[idx[k]]; }
    if (subset_ok(s, d)) return true;
  }
  return false;
}

// N(g): the least k >= 1 with q^k <= 1 - confidence, q = 1 - (g/m)^4, q^k by sequential products, capped at K
__device__ int iter_bound(int g, int m, double confidence, int max_iters) {
  const double w = dd((double)g, (double)m);
  const double q = ds(1.0, dm(dm(dm(w, w), w), w));
  const double lim = ds(1.0, confidence);
  int k = 1;
  double prod = q;
  while (!(prod <= lim) && k < max_iters) { prod = dm(prod, q); ++k; }
  return k;
}

__device__ __forceinline__ bool pair_range(const int* offsets, int p, int cap, int& lo, int& m) {
  lo = offsets[p];
  const int hi = offsets[p + 1];
  m = hi - lo;
  return lo >= 0 && hi >= lo && hi <= cap;
}

__global__ void __launch_bounds__(kThreads) k_ransac(const float2* __restrict__ src, const float2* __restrict__ dst,
                                                     const int* __restrict__ offsets, int cap, float thr2, int max_iters,
                                                     double confidence, uint64_t seed, double* __restrict__ best_h,
                                                     int* __restrict__ best_n, int* __restrict__ iters) {
  __shared__ float s_hf[kThreads][8];
  __shared__ double s_h[kThreads][9];
  __shared__ int s_cnt[kThreads];
  __shared__ unsigned char s_state[kThreads];     // 0: not drawn, 1: drawn, solve failed, 3: drawn and solved
  __shared__ int s_niters, s_best, s_i, s_stop;
  const int p = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  int lo, m;
  double* bh = best_h + (size_t)p * 9;
  if (!pair_range(offsets, p, cap, lo, m) || m < 4) {
    if (tid < 9) bh[tid] = 0.0;
    if (tid == 0) { best_n[p] = 0; iters[p] = 0; }
    return;
  }
  const float2* ps = src + lo;
  const float2* pd = dst + lo;
  if (m == 4) {                                   // cv2: H = DLT(all four), no sampling, no refinement
    if (tid == 0) {
      double H[9];
      const bool ok = dlt4(ps, pd, H);
      for (int j = 0; j < 9; ++j) bh[j] = ok ? H[j] : 0.0;
      best_n[p] = ok ? 4 : 0;
      iters[p] = 0;
    }
    return;
  }
  if (tid == 0) { s_niters = max_iters; s_best = 0; s_i = 0; s_stop = 0; }
  if (tid < 9) bh[tid] = 0.0;
  const uint64_t base = splitmix64(seed);
  for (;;) {
    __syncthreads();
    const int i0 = s_i, niters = s_niters;
    if (s_stop || i0 >= niters) break;
    const int hyp = i0 + tid;
    unsigned char state = 0;
    if (hyp < niters) {
      float2 s[4], d[4];
      if (draw_sample(base, hyp, m, ps, pd, s, d)) {
        double H[9];
        state = dlt4(s, d, H) ? 3 : 1;
        if (state == 3) {
          for (int j = 0; j < 9; ++j) s_h[tid][j] = H[j];
          for (int j = 0; j < 8; ++j) s_hf[tid][j] = (float)H[j];
        }
      }
    }
    s_state[tid] = state;
    s_cnt[tid] = 0;
    __syncthreads();
    for (int j = 0; j < 32; ++j) {
      const int t = warp * 32 + j;
      if (s_state[t] != 3) continue;               // warp-uniform
      float h[8];
#pragma unroll
      for (int k = 0; k < 8; ++k) h[k] = s_hf[t][k];
      int c = 0;
      for (int i = lane; i < m; i += 32) c += is_inlier(h, ps[i], pd[i], thr2);
      c = __reduce_add_sync(0xffffffffu, c);
      if (lane == 0) s_cnt[t] = c;
    }
    __syncthreads();
    if (tid == 0) {                                // cv2's acceptance and stopping rule, in hypothesis order
      for (int t = 0; t < kThreads; ++t) {
        const int h = i0 + t;
        if (h >= s_niters) break;
        if (s_state[t] == 0) { s_stop = 1; break; }
        s_i = h + 1;
        const int c = s_cnt[t];
        if (c > max(s_best, 3)) {
          s_best = c;
          for (int j = 0; j < 9; ++j) bh[j] = s_h[t][j];
          s_niters = min(s_niters, iter_bound(c, m, confidence, max_iters));
        }
      }
    }
  }
  if (tid == 0) {
    best_n[p] = s_best;
    iters[p] = s_i;
    if (s_best == 0)
      for (int j = 0; j < 9; ++j) bh[j] = 0.0;
  }
}

// red[V][256]: every thread has added its strided partials in column tid; afterwards red[v][0] holds the sum
__device__ void block_tree(double* red, int V) {
  for (int s = kThreads / 2; s; s >>= 1) {
    __syncthreads();
    for (int idx = threadIdx.x; idx < V * s; idx += kThreads) {
      const int v = idx / s, q = idx - v * s;
      red[v * kThreads + q] = da(red[v * kThreads + q], red[v * kThreads + q + s]);
    }
  }
  __syncthreads();
}

__device__ __forceinline__ void clear(double* red, int V) {
  for (int v = 0; v < V; ++v) red[v * kThreads + threadIdx.x] = 0.0;
}

// residuals and Jacobian rows of cv2 HomographyRefineCallback::compute at h (fp64)
__device__ __forceinline__ void lm_point(const double* h, float2 s, float2 d, double& ex, double& ey, double* jx, double* jy) {
  const double X = s.x, Y = s.y;
  const double den = da(da(dm(h[6], X), dm(h[7], Y)), 1.0);
  const double ww = fabs(den) > DBL_EPSILON ? dd(1.0, den) : 0.0;
  const double xi = dm(da(da(dm(h[0], X), dm(h[1], Y)), h[2]), ww);
  const double yi = dm(da(da(dm(h[3], X), dm(h[4], Y)), h[5]), ww);
  ex = ds(xi, (double)d.x);
  ey = ds(yi, (double)d.y);
  const double Xw = dm(X, ww), Yw = dm(Y, ww);
  jx[0] = Xw; jx[1] = Yw; jx[2] = ww; jx[3] = 0.0; jx[4] = 0.0; jx[5] = 0.0; jx[6] = -dm(Xw, xi); jx[7] = -dm(Yw, xi);
  jy[0] = 0.0; jy[1] = 0.0; jy[2] = 0.0; jy[3] = Xw; jy[4] = Yw; jy[5] = ww; jy[6] = -dm(Xw, yi); jy[7] = -dm(Yw, yi);
}

// cost (and with `normal`, JtJ and Jtr) over the n compacted points at h; red[] ends with the sums in column 0
__device__ void lm_pass(const double* h, const float2* ps, const float2* pd, const int* idx, int n, bool normal, double* red) {
  const int V = normal ? kLmTerms : 1;
  clear(red, V);
  for (int k = threadIdx.x; k < n; k += kThreads) {
    const int i = idx[k];
    double ex, ey, jx[8], jy[8];
    lm_point(h, ps[i], pd[i], ex, ey, jx, jy);
    const double cost = da(dm(ex, ex), dm(ey, ey));
    if (!normal) { red[threadIdx.x] = da(red[threadIdx.x], cost); continue; }
    int q = 0;
#pragma unroll
    for (int a = 0; a < 8; ++a)
#pragma unroll
      for (int c = a; c < 8; ++c, ++q)
        red[q * kThreads + threadIdx.x] = da(red[q * kThreads + threadIdx.x], da(dm(jx[a], jx[c]), dm(jy[a], jy[c])));
#pragma unroll
    for (int a = 0; a < 8; ++a)
      red[(36 + a) * kThreads + threadIdx.x] = da(red[(36 + a) * kThreads + threadIdx.x], da(dm(jx[a], ex), dm(jy[a], ey)));
    red[44 * kThreads + threadIdx.x] = da(red[44 * kThreads + threadIdx.x], cost);
  }
  block_tree(red, V);
}

__global__ void __launch_bounds__(kThreads) k_homography_refine(const float2* __restrict__ src, const float2* __restrict__ dst,
                                                                const int* __restrict__ offsets, int cap, float thr2,
                                                                const double* __restrict__ best_h, const int* __restrict__ best_n,
                                                                const int* __restrict__ iters, int* __restrict__ idx_ws,
                                                                double* __restrict__ H_out, unsigned char* __restrict__ mask_out,
                                                                int* __restrict__ n_inliers, int* __restrict__ n_iters) {
  extern __shared__ double red[];                 // [kLmTerms][kThreads]
  __shared__ double s_H[9], s_h[8], s_hn[8], s_A[36], s_g[8], s_cost, s_lam;
  __shared__ float s_hf[8];
  __shared__ int s_wcnt[kThreads / 32], s_count, s_flag;
  const int p = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  int lo, m;
  const bool in_range = pair_range(offsets, p, cap, lo, m);
  const int best = in_range ? best_n[p] : 0;
  if (tid == 0 && n_iters) n_iters[p] = iters[p];
  if (!in_range || best == 0 || m < 4) {
    if (tid < 9) H_out[(size_t)p * 9 + tid] = 0.0;
    if (tid == 0) n_inliers[p] = 0;
    if (in_range)
      for (int i = tid; i < m; i += kThreads) mask_out[lo + i] = 0;
    return;
  }
  if (m == 4) {
    if (tid < 9) H_out[(size_t)p * 9 + tid] = best_h[(size_t)p * 9 + tid];
    if (tid == 0) n_inliers[p] = 4;
    if (tid < 4) mask_out[lo + tid] = 1;
    return;
  }
  const float2* ps = src + lo;
  const float2* pd = dst + lo;
  int* idx = idx_ws + lo;
  if (tid < 9) s_H[tid] = best_h[(size_t)p * 9 + tid];
  for (int round = 0; round < kRefitRounds; ++round) {
    __syncthreads();
    if (tid < 8) s_hf[tid] = (float)s_H[tid];
    __syncthreads();
    // the inliers of the current model, compacted in index order
    int n = 0;
    for (int b = 0; b < m; b += kThreads) {
      const int i = b + tid;
      const bool in = i < m && is_inlier(s_hf, ps[i], pd[i], thr2);
      const unsigned bal = __ballot_sync(0xffffffffu, in);
      if (lane == 0) s_wcnt[warp] = __popc(bal);
      __syncthreads();
      int off = 0, tot = 0;
      for (int w = 0; w < kThreads / 32; ++w) { off += w < warp ? s_wcnt[w] : 0; tot += s_wcnt[w]; }
      if (in) idx[n + off + __popc(bal & ((1u << lane) - 1u))] = i;
      n += tot;
      __syncthreads();
    }
    // DLT refit on them: centroids, absolute deviations, normal equations
    const double nd = (double)n;
    Norm nm;
    clear(red, 4);
    for (int k = tid; k < n; k += kThreads) {
      const float2 s = ps[idx[k]], d = pd[idx[k]];
      red[0 * kThreads + tid] = da(red[0 * kThreads + tid], (double)s.x);
      red[1 * kThreads + tid] = da(red[1 * kThreads + tid], (double)s.y);
      red[2 * kThreads + tid] = da(red[2 * kThreads + tid], (double)d.x);
      red[3 * kThreads + tid] = da(red[3 * kThreads + tid], (double)d.y);
    }
    block_tree(red, 4);
    nm.cxs = dd(red[0], nd); nm.cys = dd(red[kThreads], nd); nm.cxd = dd(red[2 * kThreads], nd); nm.cyd = dd(red[3 * kThreads], nd);
    __syncthreads();
    clear(red, 4);
    for (int k = tid; k < n; k += kThreads) {
      const float2 s = ps[idx[k]], d = pd[idx[k]];
      red[0 * kThreads + tid] = da(red[0 * kThreads + tid], fabs(ds((double)s.x, nm.cxs)));
      red[1 * kThreads + tid] = da(red[1 * kThreads + tid], fabs(ds((double)s.y, nm.cys)));
      red[2 * kThreads + tid] = da(red[2 * kThreads + tid], fabs(ds((double)d.x, nm.cxd)));
      red[3 * kThreads + tid] = da(red[3 * kThreads + tid], fabs(ds((double)d.y, nm.cyd)));
    }
    block_tree(red, 4);
    const double sa[4] = {red[0], red[kThreads], red[2 * kThreads], red[3 * kThreads]};
    const bool norm_ok = norm_scales(nm, nd, sa);
    __syncthreads();
    if (norm_ok) {
      clear(red, kNormTerms);
      for (int k = tid; k < n; k += kThreads) {
        double X, Y, u, v, t[kNormTerms];
        normalise(nm, ps[idx[k]], pd[idx[k]], X, Y, u, v);
        dlt_terms(X, Y, u, v, t);
        for (int q = 0; q < kNormTerms; ++q) red[q * kThreads + tid] = da(red[q * kThreads + tid], t[q]);
      }
      block_tree(red, kNormTerms);
    }
    if (tid == 0) {
      double S[kNormTerms], H0[9];
      for (int q = 0; q < kNormTerms; ++q) S[q] = red[q * kThreads];
      const bool ok = norm_ok && dlt_finish(nm, S, H0);
      for (int j = 0; j < 8; ++j) s_h[j] = ok ? H0[j] : s_H[j];       // fall back to the current model
      s_lam = 1e-3;
    }
    __syncthreads();
    // Levenberg-Marquardt on the 8 parameters, h33 = 1
    lm_pass(s_h, ps, pd, idx, n, true, red);
    if (tid == 0) {
      for (int q = 0; q < 36; ++q) s_A[q] = red[q * kThreads];
      for (int a = 0; a < 8; ++a) s_g[a] = red[(36 + a) * kThreads];
      s_cost = red[44 * kThreads];
    }
    for (int it = 0; it < kLmIters; ++it) {
      __syncthreads();
      if (tid == 0) {
        double A[8][8], b[8], dlt[8];
        int q = 0;
        for (int a = 0; a < 8; ++a)
          for (int c = a; c < 8; ++c, ++q) { A[a][c] = s_A[q]; A[c][a] = s_A[q]; }
        for (int a = 0; a < 8; ++a) { A[a][a] = da(A[a][a], dm(s_lam, A[a][a])); b[a] = -s_g[a]; }
        s_flag = solve8(A, b, dlt);
        if (s_flag)
          for (int a = 0; a < 8; ++a) s_hn[a] = da(s_h[a], dlt[a]);
        else
          s_lam = dm(s_lam, 10.0);
      }
      __syncthreads();
      if (!s_flag) continue;
      lm_pass(s_hn, ps, pd, idx, n, false, red);
      const bool accept = red[0] < s_cost;
      __syncthreads();
      if (tid == 0) s_lam = accept ? dd(s_lam, 10.0) : dm(s_lam, 10.0);
      if (!accept) continue;
      if (tid < 8) s_h[tid] = s_hn[tid];
      __syncthreads();
      lm_pass(s_h, ps, pd, idx, n, true, red);
      if (tid == 0) {
        for (int q = 0; q < 36; ++q) s_A[q] = red[q * kThreads];
        for (int a = 0; a < 8; ++a) s_g[a] = red[(36 + a) * kThreads];
        s_cost = red[44 * kThreads];
      }
    }
    __syncthreads();
    // the inliers of the refined model; another round while they grow
    if (tid < 8) { s_H[tid] = s_h[tid]; s_hf[tid] = (float)s_h[tid]; }
    if (tid == 8) s_H[8] = 1.0;
    if (tid == 0) s_count = 0;
    __syncthreads();
    int c = 0;
    for (int i = tid; i < m; i += kThreads) c += is_inlier(s_hf, ps[i], pd[i], thr2);
    c = __reduce_add_sync(0xffffffffu, c);
    if (lane == 0) atomicAdd(&s_count, c);
    __syncthreads();
    if (s_count <= n) break;
  }
  __syncthreads();
  for (int i = tid; i < m; i += kThreads) mask_out[lo + i] = is_inlier(s_hf, ps[i], pd[i], thr2);
  if (tid < 9) H_out[(size_t)p * 9 + tid] = s_H[tid];
  if (tid == 0) n_inliers[p] = s_count;
}

size_t head_bytes(int n_pairs) {
  const size_t P = (size_t)(n_pairs > 0 ? n_pairs : 0);
  return align_up(P * 9 * sizeof(double), 256) + 2 * align_up(P * sizeof(int), 256);
}

}  // namespace
}  // namespace gims

using namespace gims;

extern "C" size_t gims_homography_workspace_bytes(int n_pairs, int total_points) {
  const size_t T = (size_t)(total_points > 0 ? total_points : 0);
  return head_bytes(n_pairs) + align_up(T * sizeof(int), 256) + 256;
}

extern "C" int gims_find_homographies(const float* src, const float* dst, const int* offsets_dev, int n_pairs, double thresh,
                                      int max_iters, double confidence, unsigned long long seed, void* workspace,
                                      size_t workspace_bytes, double* H_out, unsigned char* mask_out, int* n_inliers,
                                      int* n_iters, void* stream) {
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (n_pairs < 0) { set_error("gims_find_homographies: n_pairs %d < 0", n_pairs); return GIMS_ERR_ARG; }
  if (n_pairs == 0) return GIMS_OK;
  if (!src || !dst || !offsets_dev || !workspace || !H_out || !mask_out || !n_inliers) {
    set_error("gims_find_homographies: null argument"); return GIMS_ERR_ARG;
  }
  if (!(thresh > 0.0) || !std::isfinite(thresh) || !(confidence > 0.0 && confidence < 1.0) || max_iters < 1) {
    set_error("gims_find_homographies: bad parameters (thresh %g, confidence %g, max_iters %d)", thresh, confidence, max_iters);
    return GIMS_ERR_ARG;
  }
  if (workspace_bytes < gims_homography_workspace_bytes(n_pairs, 0)) {
    set_error("gims_find_homographies: workspace too small"); return GIMS_ERR_WORKSPACE;
  }
  Arena a(workspace, workspace_bytes);
  double* best_h = a.take<double>((size_t)n_pairs * 9);
  int* best_n = a.take<int>(n_pairs);
  int* iters = a.take<int>(n_pairs);
  a.off = align_up(a.off, 256);
  int* idx = reinterpret_cast<int*>(a.base + a.off);
  // points past the index buffer belong to no pair: such a pair reports "not found" and writes no mask
  const size_t room = (workspace_bytes - a.off) / sizeof(int);
  const int cap = room > 0x7fffffff ? 0x7fffffff : (int)room;
  const float thr2 = (float)(thresh * thresh);
  const float2* s2 = reinterpret_cast<const float2*>(src);
  const float2* d2 = reinterpret_cast<const float2*>(dst);
  k_ransac<<<n_pairs, kThreads, 0, st>>>(s2, d2, offsets_dev, cap, thr2, max_iters, confidence, (uint64_t)seed, best_h,
                                         best_n, iters);
  GIMS_LAUNCH_OK();
  const int smem = kLmTerms * kThreads * (int)sizeof(double);
  GIMS_CUDA_OK(cudaFuncSetAttribute(k_homography_refine, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  k_homography_refine<<<n_pairs, kThreads, smem, st>>>(s2, d2, offsets_dev, cap, thr2, best_h, best_n, iters, idx, H_out,
                                                       mask_out, n_inliers, n_iters);
  GIMS_LAUNCH_OK();
  return GIMS_OK;
}

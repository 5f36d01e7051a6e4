// SIFT keypoint detection on the device: OpenCV 4.x SIFT::detect with frontend.SIFT_CONFIG (3 layers per octave,
// contrastThreshold 0.001, edgeThreshold 80, sigma 1.6, the image doubled first), in the float32 order of operations that
// oracle/cv_sift_oracle.py fixes.  Every step below follows that restatement operation for operation (explicit _rn
// intrinsics where contraction into a fused multiply-add would change a result, fused ones where the restatement fuses),
// so the keypoint records are bit-identical to it; the restatement itself agrees with cv2 within a tolerance
// (tests/test_sift_cpu.py), as cv2's own SIMD and scalar paths agree with each other.
//
// Steps:
//   1. grey (BGR2GRAY fixed point) and the x2 bilinear upsample, in one kernel;
//   2. per octave six float32 Gaussian levels (separable symmetric blur, BORDER_REFLECT_101: a row pass into the
//      workspace, then a column pass that also writes the difference to the previous level, the DoG);
//   3. one launch scans every octave's DoG layers 1..3 for extrema and compacts them (atomic counter: the candidate order
//      varies run to run, the sort of step 5 removes that);
//   4. a warp per candidate: lane 0 runs the sub-pixel refinement (adjustLocalExtrema), the warp builds the orientation
//      histogram — each bin summed in window order by one lane, no float atomics — and lane 0 emits one keypoint per peak;
//   5. a rank sort (each record counts the records ordered before it: ~7 k records at 800 x 600), duplicates removed in
//      one CTA, then either all records or the max_keypoints strongest (a second rank pass by response), halved back to
//      input coordinates.
#include <cfloat>
#include <climits>
#include <cmath>

#include "common.cuh"

namespace gims {
namespace {

constexpr int kLayers = 3;
constexpr int kPerOctave = kLayers + 3;  // Gaussian levels per octave
constexpr int kDogPerOctave = kLayers + 2;
constexpr int kBorder = 5;               // SIFT_IMG_BORDER
constexpr int kMaxSteps = 5;             // SIFT_MAX_INTERP_STEPS
constexpr int kBins = 36;
constexpr int kMaxOctaves = 32;
constexpr int kMaxTaps = 64;             // widest kernel: 27 taps (sigma 3.09)
constexpr int kThreads = 256;
constexpr int kWarpsPerBlock = 8;
constexpr int kSortTile = 256;
constexpr int kFinishThreads = 1024;
constexpr double kSigma = 1.6;

struct Kernel1D {
  int r;                                 // radius: n = 2 r + 1 taps
  float k[kMaxTaps / 2 + 1];             // k[j] = tap at distance j from the centre
};

struct Octaves {
  int n;
  int h[kMaxOctaves], w[kMaxOctaves];
  long long gauss[kMaxOctaves];          // float offset of level 0; level i at gauss + i * h * w
  long long dog[kMaxOctaves];            // float offset of DoG layer 0
};

struct Candidate { int o, layer, r, c; };
struct Record { float x, y, size, angle, response; int octave; };

struct Consts {                          // constants of cv::hal::exp32f and cv::fastAtan2, computed on the host
  float exp_tab[64];
  float a1, a2, a3, a4, prescale, postscale, minval, maxval;
  float p1, p3, p5, p7, atan_eps;
};

// getGaussianKernel(cvRound(8 sigma + 1) | 1, sigma, CV_32F): the bit-exact double kernel rounded to float
int float_kernel(double sigma, Kernel1D* out) {
  const int n = (int)std::nearbyint(sigma * 8 + 1) | 1;
  const int n2 = n / 2;
  if (n2 > kMaxTaps / 2) return -1;
  double vals[kMaxTaps];
  double sum = 0.0;
  for (int i = 0, x = 1 - n; i < n2; ++i, x += 2) {
    vals[i] = std::exp((double)(x * x) * (-0.125 / (sigma * sigma)));
    sum += vals[i];
  }
  const double mul = 1.0 / (2 * sum + 1.0);
  out->r = n2;
  for (int i = 0; i < n2; ++i) out->k[n2 - i] = (float)(vals[i] * mul);
  out->k[0] = (float)mul;
  return n;
}

__device__ __forceinline__ int reflect101(int i, int n) {
  if ((unsigned)i < (unsigned)n) return i;
  if (n == 1) return 0;
  const int p = 2 * (n - 1);
  i %= p;
  if (i < 0) i += p;
  return i >= n ? p - i : i;
}

__device__ __forceinline__ int bgr_grey(const unsigned char* p, int cn) {
  return cn == 3 ? (p[0] * 3735 + p[1] * 19235 + p[2] * 9798 + (1 << 14)) >> 15 : p[0];
}

// 1. grey + x2 upsample: d[2k] = 0.25 s[k - 1] + 0.75 s[k], d[2k + 1] = 0.75 s[k] + 0.25 s[k + 1] per axis (exact)
__global__ void __launch_bounds__(kThreads) k_sift_upsample(const unsigned char* __restrict__ img, int h, int w, int cn,
                                                            float* __restrict__ dst) {
  const int dw = 2 * w;
  const long long total = 4LL * h * w;
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
    const int y = (int)(e / dw), x = (int)(e % dw);
    const int xb = x >> 1, xa = min(max((x & 1) ? xb + 1 : xb - 1, 0), w - 1);
    const int yb = y >> 1, ya = min(max((y & 1) ? yb + 1 : yb - 1, 0), h - 1);
    auto row = [&](int yy) {
      const unsigned char* s = img + (size_t)yy * w * cn;
      return __fadd_rn(__fmul_rn(0.25f, (float)bgr_grey(s + xa * cn, cn)), __fmul_rn(0.75f, (float)bgr_grey(s + xb * cn, cn)));
    };
    dst[e] = __fadd_rn(__fmul_rn(0.25f, row(ya)), __fmul_rn(0.75f, row(yb)));
  }
}

// octave seed: every second pixel of level 3 of the octave before
__global__ void __launch_bounds__(kThreads) k_sift_seed(const float* __restrict__ src, int sw, float* __restrict__ dst, int h,
                                                        int w) {
  const long long total = (long long)h * w;
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
    const int y = (int)(e / w), x = (int)(e % w);
    dst[e] = src[(size_t)(2 * y) * sw + 2 * x];
  }
}

// row pass: k[0] s[x] + sum_j k[j] (s[x - j] + s[x + j]), j = 1..r in order
__global__ void __launch_bounds__(kThreads) k_sift_blur_rows(const float* __restrict__ src, float* __restrict__ dst, int h,
                                                             int w, const Kernel1D kr) {
  const long long total = (long long)h * w;
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
    const int y = (int)(e / w), x = (int)(e % w);
    const float* s = src + (size_t)y * w;
    float acc = __fmul_rn(kr.k[0], s[x]);
    if (x >= kr.r && x + kr.r < w) {
      for (int j = 1; j <= kr.r; ++j) acc = __fadd_rn(acc, __fmul_rn(kr.k[j], __fadd_rn(s[x - j], s[x + j])));
    } else {
      for (int j = 1; j <= kr.r; ++j)
        acc = __fadd_rn(acc, __fmul_rn(kr.k[j], __fadd_rn(s[reflect101(x - j, w)], s[reflect101(x + j, w)])));
    }
    dst[e] = acc;
  }
}

// column pass, the same sum down a column; `prev` (may be null) is the level below: dog = result - prev
__global__ void __launch_bounds__(kThreads) k_sift_blur_cols(const float* __restrict__ src, float* __restrict__ dst,
                                                             const float* __restrict__ prev, float* __restrict__ dog, int h,
                                                             int w, const Kernel1D kr) {
  const long long total = (long long)h * w;
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
    const int y = (int)(e / w), x = (int)(e % w);
    const float* s = src + x;
    float acc = __fmul_rn(kr.k[0], s[(size_t)y * w]);
    if (y >= kr.r && y + kr.r < h) {
      for (int j = 1; j <= kr.r; ++j)
        acc = __fadd_rn(acc, __fmul_rn(kr.k[j], __fadd_rn(s[(size_t)(y - j) * w], s[(size_t)(y + j) * w])));
    } else {
      for (int j = 1; j <= kr.r; ++j)
        acc = __fadd_rn(acc, __fmul_rn(kr.k[j], __fadd_rn(s[(size_t)reflect101(y - j, h) * w],
                                                          s[(size_t)reflect101(y + j, h) * w])));
    }
    dst[e] = acc;
    if (dog) dog[e] = __fsub_rn(acc, prev[e]);
  }
}

// 3. extrema of DoG layers 1..3 of every octave, at least kBorder px from the border
__global__ void __launch_bounds__(kThreads) k_sift_extrema(const float* __restrict__ ws, const Octaves oc,
                                                           Candidate* __restrict__ cand, int cand_cap, int* __restrict__ n_cand) {
  long long total = 0;
  for (int o = 0; o < oc.n; ++o) total += 3LL * oc.h[o] * oc.w[o];
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
    long long q = e;
    int o = 0;
    while (q >= 3LL * oc.h[o] * oc.w[o]) { q -= 3LL * oc.h[o] * oc.w[o]; ++o; }
    const int h = oc.h[o], w = oc.w[o];
    const long long plane = (long long)h * w;
    const int layer = 1 + (int)(q / plane);
    const int r = (int)((q % plane) / w), c = (int)(q % w);
    if (r < kBorder || r >= h - kBorder || c < kBorder || c >= w - kBorder) continue;
    const float* cur = ws + oc.dog[o] + layer * plane + (size_t)r * w + c;
    const float v = *cur;
    if (!(v > 0.f || v < 0.f)) continue;
    bool mx = v > 0.f, mn = v < 0.f;
    for (int dl = -1; dl <= 1; ++dl)
      for (int dr = -1; dr <= 1; ++dr)
        for (int dc = -1; dc <= 1; ++dc) {
          if (dl == 0 && dr == 0 && dc == 0) continue;
          const float nb = cur[dl * plane + dr * w + dc];
          mx = mx && v >= nb;
          mn = mn && v <= nb;
        }
    if (mx || mn) {
      const int slot = atomicAdd(n_cand, 1);
      if (slot < cand_cap) cand[slot] = {o, layer, r, c};
    }
  }
}

// hal::LU32f on the 3 x 3 system A x = b (partial pivoting, eps = 10 FLT_EPSILON); x = 0 when a pivot is below eps
__device__ void lu_solve3(float A[3][3], float b[3]) {
  const float eps = FLT_EPSILON * 10.f;
  for (int i = 0; i < 3; ++i) {
    int k = i;
    for (int j = i + 1; j < 3; ++j)
      if (fabsf(A[j][i]) > fabsf(A[k][i])) k = j;
    if (fabsf(A[k][i]) < eps) { b[0] = b[1] = b[2] = 0.f; return; }
    if (k != i) {
      for (int j = 0; j < 3; ++j) { const float t = A[i][j]; A[i][j] = A[k][j]; A[k][j] = t; }
      const float t = b[i]; b[i] = b[k]; b[k] = t;
    }
    const float d = __fdiv_rn(-1.f, A[i][i]);
    for (int j = i + 1; j < 3; ++j) {
      const float alpha = __fmul_rn(A[j][i], d);
      for (int kk = i + 1; kk < 3; ++kk) A[j][kk] = __fadd_rn(A[j][kk], __fmul_rn(alpha, A[i][kk]));
      b[j] = __fadd_rn(b[j], __fmul_rn(alpha, b[i]));
    }
  }
  for (int i = 2; i >= 0; --i) {
    float s = b[i];
    for (int kk = i + 1; kk < 3; ++kk) s = __fsub_rn(s, __fmul_rn(A[i][kk], b[kk]));
    b[i] = __fdiv_rn(s, A[i][i]);
  }
}

struct Derivs { float v, g[3], dxx, dyy, dss, dxy, dxs, dys; };

__device__ __forceinline__ Derivs derivs(const float* img, const float* prev, const float* next, int w) {
  const float img_scale = 1.f / 255.f, deriv_scale = img_scale * 0.5f, cross_scale = img_scale * 0.25f;
  Derivs d;
  d.v = img[0];
  d.g[0] = __fmul_rn(__fsub_rn(img[1], img[-1]), deriv_scale);
  d.g[1] = __fmul_rn(__fsub_rn(img[w], img[-w]), deriv_scale);
  d.g[2] = __fmul_rn(__fsub_rn(next[0], prev[0]), deriv_scale);
  const float v2 = __fmul_rn(d.v, 2.f);
  d.dxx = __fmul_rn(__fsub_rn(__fadd_rn(img[1], img[-1]), v2), img_scale);
  d.dyy = __fmul_rn(__fsub_rn(__fadd_rn(img[w], img[-w]), v2), img_scale);
  d.dss = __fmul_rn(__fsub_rn(__fadd_rn(next[0], prev[0]), v2), img_scale);
  d.dxy = __fmul_rn(__fadd_rn(__fsub_rn(__fsub_rn(img[w + 1], img[w - 1]), img[-w + 1]), img[-w - 1]), cross_scale);
  d.dxs = __fmul_rn(__fadd_rn(__fsub_rn(__fsub_rn(next[1], next[-1]), prev[1]), prev[-1]), cross_scale);
  d.dys = __fmul_rn(__fadd_rn(__fsub_rn(__fsub_rn(next[w], next[-w]), prev[w]), prev[-w]), cross_scale);
  return d;
}

__device__ __forceinline__ float exp32f(float x, const Consts& k) {
  x = __fmul_rn(fminf(fmaxf(x, k.minval), k.maxval), k.prescale);
  const int xi = __float2int_rn(x);
  const float xf = __fmul_rn(__fsub_rn(x, (float)xi), k.postscale);
  const int e = min(max((xi >> 6) + 127, 0), 255);
  const float yf = __fmul_rn(k.exp_tab[xi & 63], __int_as_float(e << 23));
  float z = __fadd_rn(xf, k.a1);
  z = __fadd_rn(__fmul_rn(z, xf), k.a2);
  z = __fadd_rn(__fmul_rn(z, xf), k.a3);
  z = __fadd_rn(__fmul_rn(z, xf), k.a4);
  return __fmul_rn(z, yf);
}

__device__ __forceinline__ float fast_atan2(float y, float x, const Consts& k) {
  const float ax = fabsf(x), ay = fabsf(y);
  const float c = __fdiv_rn(fminf(ax, ay), __fadd_rn(fmaxf(ax, ay), k.atan_eps));
  const float cc = __fmul_rn(c, c);
  float a = __fmul_rn(__fmaf_rn(__fmaf_rn(__fmaf_rn(cc, k.p7, k.p5), cc, k.p3), cc, k.p1), c);
  if (!(ax >= ay)) a = __fsub_rn(90.f, a);
  if (x < 0.f) a = __fsub_rn(180.f, a);
  if (y < 0.f) a = __fsub_rn(360.f, a);
  return a;
}

// 4. a warp per candidate: refinement (lane 0), orientation histogram (the warp), peaks (lane 0)
__global__ void __launch_bounds__(kWarpsPerBlock * 32) k_sift_keypoints(
    const float* __restrict__ ws, const Octaves oc, const Candidate* __restrict__ cand, const int* __restrict__ n_cand,
    int cand_cap, const Consts kc, Record* __restrict__ rec, int rec_cap, int* __restrict__ n_rec,
    unsigned* __restrict__ status) {
  __shared__ float hist_s[kWarpsPerBlock][kBins];
  __shared__ float smooth_s[kWarpsPerBlock][kBins];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int nc = *n_cand;
  if (blockIdx.x == 0 && threadIdx.x == 0 && nc > cand_cap) atomicOr(status, GIMS_STATUS_KEYPOINT_OVERFLOW);
  const int n = min(nc, cand_cap);
  for (int ci = blockIdx.x * kWarpsPerBlock + wib; ci < n; ci += gridDim.x * kWarpsPerBlock) {
    Candidate cd = cand[ci];
    const int o = cd.o, h = oc.h[o], w = oc.w[o];
    const long long plane = (long long)h * w;
    int ok = 0;
    float xc = 0.f, xr = 0.f, xi = 0.f, contr = 0.f;
    if (lane == 0) {
      int layer = cd.layer, r = cd.r, c = cd.c, step = 0;
      const float big = (float)(INT_MAX / 3);
      for (; step < kMaxSteps; ++step) {
        const float* img = ws + oc.dog[o] + layer * plane + (size_t)r * w + c;
        const Derivs d = derivs(img, img - plane, img + plane, w);
        float A[3][3] = {{d.dxx, d.dxy, d.dxs}, {d.dxy, d.dyy, d.dys}, {d.dxs, d.dys, d.dss}};
        float X[3] = {d.g[0], d.g[1], d.g[2]};
        lu_solve3(A, X);
        xi = -X[2]; xr = -X[1]; xc = -X[0];
        if (fabsf(xi) < 0.5f && fabsf(xr) < 0.5f && fabsf(xc) < 0.5f) break;
        if (!(fabsf(xi) <= big && fabsf(xr) <= big && fabsf(xc) <= big)) { step = kMaxSteps + 1; break; }
        c += __float2int_rn(xc);
        r += __float2int_rn(xr);
        layer += __float2int_rn(xi);
        if (layer < 1 || layer > kLayers || c < kBorder || c >= w - kBorder || r < kBorder || r >= h - kBorder) {
          step = kMaxSteps + 1;
          break;
        }
      }
      if (step < kMaxSteps) {
        const float* img = ws + oc.dog[o] + layer * plane + (size_t)r * w + c;
        const Derivs d = derivs(img, img - plane, img + plane, w);
        float t = __fmul_rn(d.g[0], xc);
        t = __fadd_rn(t, __fmul_rn(d.g[1], xr));
        t = __fadd_rn(t, __fmul_rn(d.g[2], xi));
        contr = __fadd_rn(__fmul_rn(d.v, 1.f / 255.f), __fmul_rn(t, 0.5f));
        const float tr = __fadd_rn(d.dxx, d.dyy);
        const float det = __fsub_rn(__fmul_rn(d.dxx, d.dyy), __fmul_rn(d.dxy, d.dxy));
        ok = !(__fmul_rn(fabsf(contr), (float)kLayers) < 0.001f) &&
             !(det <= 0.f || __fmul_rn(__fmul_rn(tr, tr), 80.f) >= __fmul_rn(6561.f, det));
      }
      cd.layer = layer; cd.r = r; cd.c = c;
    }
    ok = __shfl_sync(0xffffffffu, ok, 0);
    if (!ok) continue;
    cd.layer = __shfl_sync(0xffffffffu, cd.layer, 0);
    cd.r = __shfl_sync(0xffffffffu, cd.r, 0);
    cd.c = __shfl_sync(0xffffffffu, cd.c, 0);
    xc = __shfl_sync(0xffffffffu, xc, 0);
    xr = __shfl_sync(0xffffffffu, xr, 0);
    xi = __shfl_sync(0xffffffffu, xi, 0);
    contr = __shfl_sync(0xffffffffu, contr, 0);
    const float s = (float)(1 << o);
    const float p = (float)exp2((double)__fdiv_rn(__fadd_rn((float)cd.layer, xi), (float)kLayers));
    const float size = __fmul_rn(__fmul_rn(__fmul_rn((float)kSigma, p), s), 2.f);
    // orientation histogram on Gaussian level (o, layer)
    const float scl = __fdiv_rn(__fmul_rn(size, 0.5f), s);
    const int R = __float2int_rn(__fmul_rn(4.5f, scl));
    const float sw = __fmul_rn(1.5f, scl);
    const float escale = __fdiv_rn(-1.f, __fmul_rn(__fmul_rn(2.f, sw), sw));
    const float* L = ws + oc.gauss[o] + cd.layer * plane;
    const int side = 2 * R + 1, npix = side * side;
    float h0 = 0.f, h1 = 0.f;                          // bins lane and lane + 32
    for (int base = 0; base < npix; base += 32) {
      const int k = base + lane;
      int bin = -1;
      float val = 0.f;
      if (k < npix) {
        const int di = k / side - R, dj = k % side - R;
        const int y = cd.r + di, x = cd.c + dj;
        if (y > 0 && y < h - 1 && x > 0 && x < w - 1) {
          const float* q = L + (size_t)y * w + x;
          const float dx = __fsub_rn(q[1], q[-1]);
          const float dy = __fsub_rn(q[-w], q[w]);
          const float wt = exp32f(__fmul_rn((float)(di * di + dj * dj), escale), kc);
          const float ori = fast_atan2(dy, dx, kc);
          const float mag = __fsqrt_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)));
          bin = __float2int_rn(__fmul_rn((float)kBins / 360.f, ori));
          if (bin >= kBins) bin -= kBins;
          if (bin < 0) bin += kBins;
          val = __fmul_rn(wt, mag);
        }
      }
      for (int t = 0; t < 32; ++t) {                   // window order within the chunk
        const int b = __shfl_sync(0xffffffffu, bin, t);
        const float v = __shfl_sync(0xffffffffu, val, t);
        if (b == lane) h0 = __fadd_rn(h0, v);
        if (b == lane + 32) h1 = __fadd_rn(h1, v);
      }
    }
    hist_s[wib][lane] = h0;
    if (lane + 32 < kBins) hist_s[wib][lane + 32] = h1;
    __syncwarp();
    if (lane == 0) {
      const float* t = hist_s[wib];
      float* hs = smooth_s[wib];
      for (int i = 0; i < kBins; ++i) {
        const float a = __fadd_rn(t[(i + kBins - 2) % kBins], t[(i + 2) % kBins]);
        const float b = __fadd_rn(t[(i + kBins - 1) % kBins], t[(i + 1) % kBins]);
        const float m6 = __fmul_rn(t[i], 6.f / 16.f);
        hs[i] = i < 32 ? __fmaf_rn(a, 1.f / 16.f, __fmaf_rn(b, 4.f / 16.f, m6))
                       : __fadd_rn(__fadd_rn(__fmul_rn(a, 1.f / 16.f), __fmul_rn(b, 4.f / 16.f)), m6);
      }
      float omax = hs[0];
      for (int i = 1; i < kBins; ++i) omax = fmaxf(omax, hs[i]);
      const float thr = __fmul_rn(omax, 0.8f);
      const float x = __fmul_rn(__fadd_rn((float)cd.c, xc), s);
      const float y = __fmul_rn(__fadd_rn((float)cd.r, xr), s);
      const int octv = o + (cd.layer << 8) + (__double2int_rn(((double)xi + 0.5) * 255.0) << 16);
      for (int j = 0; j < kBins; ++j) {
        const int l = j > 0 ? j - 1 : kBins - 1, r2 = j < kBins - 1 ? j + 1 : 0;
        const float a = hs[l], b = hs[r2], m = hs[j];
        if (m > a && m > b && m >= thr) {
          float bn = __fadd_rn((float)j, __fdiv_rn(__fmul_rn(0.5f, __fsub_rn(a, b)), __fadd_rn(__fsub_rn(a, __fmul_rn(2.f, m)), b)));
          bn = bn < 0.f ? __fadd_rn((float)kBins, bn) : (bn >= (float)kBins ? __fsub_rn(bn, (float)kBins) : bn);
          float ang = __fsub_rn(360.f, __fmul_rn(360.f / kBins, bn));
          if (fabsf(__fsub_rn(ang, 360.f)) < FLT_EPSILON) ang = 0.f;
          const int slot = atomicAdd(n_rec, 1);
          if (slot < rec_cap) rec[slot] = {x, y, size, ang, fabsf(contr), octv};
        }
      }
    }
    __syncwarp();
  }
}

// KeyPoint_LessThan of OpenCV's removeDuplicatedSorted: x, y ascending, size descending, angle ascending, response
// descending, octave descending
__device__ __forceinline__ bool kp_less(const Record& a, const Record& b) {
  if (a.x != b.x) return a.x < b.x;
  if (a.y != b.y) return a.y < b.y;
  if (a.size != b.size) return a.size > b.size;
  if (a.angle != b.angle) return a.angle < b.angle;
  if (a.response != b.response) return a.response > b.response;
  return a.octave > b.octave;
}

// 5a. sorted[rank(i)] = rec[i], rank = records ordered before i (ties by index: such records are identical)
__global__ void __launch_bounds__(kSortTile) k_sift_sort(const Record* __restrict__ rec, const int* __restrict__ n_rec,
                                                        int rec_cap, Record* __restrict__ sorted) {
  __shared__ Record tile[kSortTile];
  const int n = min(*n_rec, rec_cap);
  const int i = blockIdx.x * kSortTile + threadIdx.x;
  if (blockIdx.x * kSortTile >= n) return;
  Record me = {};
  if (i < n) me = rec[i];
  int rank = 0;
  for (int t0 = 0; t0 < n; t0 += kSortTile) {
    __syncthreads();
    if (t0 + (int)threadIdx.x < n) tile[threadIdx.x] = rec[t0 + threadIdx.x];
    __syncthreads();
    const int m = min(kSortTile, n - t0);
    if (i < n)
      for (int j = 0; j < m; ++j) {
        const Record& o = tile[j];
        rank += kp_less(o, me) || (!kp_less(me, o) && t0 + j < i);
      }
  }
  if (i < n) sorted[rank] = me;
}

// 5b. one CTA: drop records equal to the one before in (pt, size, angle), compact in order
__global__ void __launch_bounds__(kFinishThreads) k_sift_dedupe(const Record* __restrict__ sorted, const int* __restrict__ n_rec,
                                                               int rec_cap, Record* __restrict__ uniq, int* __restrict__ n_uniq,
                                                               unsigned* __restrict__ status) {
  __shared__ int warp_sums[kFinishThreads / 32];
  __shared__ int carry;
  const int nr = *n_rec;
  const bool overflow = nr > rec_cap || (*status & GIMS_STATUS_KEYPOINT_OVERFLOW);
  if (threadIdx.x == 0) {
    carry = 0;
    if (nr > rec_cap) atomicOr(status, GIMS_STATUS_KEYPOINT_OVERFLOW);
  }
  const int n = overflow ? 0 : nr;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  for (int b0 = 0; b0 < n; b0 += kFinishThreads) {
    __syncthreads();
    const int i = b0 + threadIdx.x;
    int keep = 0;
    Record me = {};
    if (i < n) {
      me = sorted[i];
      keep = 1;
      if (i > 0) {
        const Record& p = sorted[i - 1];
        keep = !(p.x == me.x && p.y == me.y && p.size == me.size && p.angle == me.angle);
      }
    }
    int incl = keep;
    for (int d = 1; d < 32; d <<= 1) {
      const int v = __shfl_up_sync(0xffffffffu, incl, d);
      if (lane >= d) incl += v;
    }
    if (lane == 31) warp_sums[wid] = incl;
    __syncthreads();
    if (wid == 0) {
      int v = warp_sums[lane];
      for (int d = 1; d < 32; d <<= 1) {
        const int u = __shfl_up_sync(0xffffffffu, v, d);
        if (lane >= d) v += u;
      }
      warp_sums[lane] = v;                              // inclusive over warps
    }
    __syncthreads();
    const int before = carry + (wid > 0 ? warp_sums[wid - 1] : 0) + incl - keep;
    if (keep) uniq[before] = me;
    __syncthreads();
    if (threadIdx.x == kFinishThreads - 1) carry += warp_sums[kFinishThreads / 32 - 1];
  }
  __syncthreads();
  if (threadIdx.x == 0) *n_uniq = carry;
}

// 5c. the output records, halved back to input coordinates (octave byte - 1); with 0 < max_kp < n the max_kp strongest,
// ranked by response descending, ties by position
__global__ void __launch_bounds__(kSortTile) k_sift_output(const Record* __restrict__ uniq, const int* __restrict__ n_uniq,
                                                          int max_kp, float* __restrict__ pt, float* __restrict__ size,
                                                          float* __restrict__ angle, float* __restrict__ response,
                                                          int* __restrict__ octave, int* __restrict__ n_kp) {
  __shared__ float tile[kSortTile];
  const int n = *n_uniq;
  const bool topk = max_kp > 0 && n > max_kp;
  const int n_out = topk ? max_kp : n;
  if (blockIdx.x == 0 && threadIdx.x == 0) *n_kp = n_out;
  const int i = blockIdx.x * kSortTile + threadIdx.x;
  if (blockIdx.x * kSortTile >= n) return;
  Record me = {};
  if (i < n) me = uniq[i];
  int rank = i;
  if (topk) {
    rank = 0;
    for (int t0 = 0; t0 < n; t0 += kSortTile) {
      __syncthreads();
      if (t0 + (int)threadIdx.x < n) tile[threadIdx.x] = uniq[t0 + threadIdx.x].response;
      __syncthreads();
      const int m = min(kSortTile, n - t0);
      if (i < n)
        for (int j = 0; j < m; ++j) rank += tile[j] > me.response || (tile[j] == me.response && t0 + j < i);
    }
  }
  if (i < n && rank < n_out) {
    pt[2 * rank] = __fmul_rn(me.x, 0.5f);
    pt[2 * rank + 1] = __fmul_rn(me.y, 0.5f);
    size[rank] = __fmul_rn(me.size, 0.5f);
    angle[rank] = me.angle;
    response[rank] = me.response;
    octave[rank] = (me.octave & ~255) | ((me.octave - 1) & 255);
  }
}

int grid_for(long long elems, int threads) {
  long long b = (elems + threads - 1) / threads;
  return (int)(b < 1 ? 1 : (b > (1 << 16) ? (1 << 16) : b));
}

// octave table and workspace layout: the upsample and row-pass buffers, then per octave 6 Gaussian + 5 DoG levels
struct Layout {
  Octaves oc;
  long long up, tmp, floats;             // float offsets / total floats
};

int sift_layout(int h, int w, Layout* L) {
  int n_levels = 0;
  GIMS_TRY(gims_pyramid_layout(h, w, 1, &n_levels, nullptr, nullptr, nullptr));
  const int n_oct = n_levels / kPerOctave;
  if (n_oct > kMaxOctaves) { set_error("gims_sift_detect: %d octaves", n_oct); return GIMS_ERR_ARG; }
  *L = {};
  L->oc.n = n_oct;
  const long long base = 4LL * h * w;
  L->up = 0;
  L->tmp = base;
  long long off = 2 * base;
  for (int o = 0; o < n_oct; ++o) {
    L->oc.h[o] = (2 * h) >> o;
    L->oc.w[o] = (2 * w) >> o;
    const long long plane = (long long)L->oc.h[o] * L->oc.w[o];
    L->oc.gauss[o] = off;
    off += kPerOctave * plane;
    L->oc.dog[o] = off;
    off += kDogPerOctave * plane;
  }
  L->floats = off;
  return GIMS_OK;
}

size_t sift_bytes(const Layout& L, int kp_cap, size_t* cand_off, size_t* rec_off, size_t* sorted_off, size_t* uniq_off,
                  size_t* count_off) {
  size_t off = align_up((size_t)L.floats * sizeof(float), 256);
  *cand_off = off;
  off = align_up(off + (size_t)2 * kp_cap * sizeof(Candidate), 256);
  *rec_off = off;
  off = align_up(off + (size_t)kp_cap * sizeof(Record), 256);
  *sorted_off = off;
  off = align_up(off + (size_t)kp_cap * sizeof(Record), 256);
  *uniq_off = off;
  off = align_up(off + (size_t)kp_cap * sizeof(Record), 256);
  *count_off = off;
  return off + 4 * sizeof(int);
}

Consts make_consts() {
  Consts k;
  const double a0 = .9670371139572337719125840413672004409288e-2;
  for (int j = 0; j < 64; ++j) k.exp_tab[j] = (float)(std::pow(2.0, j / 64.0) * a0);
  k.a4 = (float)(1.000000000000002438532970795181890933776 / a0);
  k.a3 = (float)(.6931471805521448196800669615864773144641 / a0);
  k.a2 = (float)(.2402265109513301490103372422686535526573 / a0);
  k.a1 = (float)(.5550339366753125211915322047004666939128e-1 / a0);
  const double log2e64 = 1.4426950408889634073599246810019 * 64;
  k.prescale = (float)log2e64;
  k.postscale = (float)(1.0 / 64);
  k.minval = (float)(-3000.0 * 64 / log2e64);
  k.maxval = (float)(3000.0 * 64 / log2e64);
  const float r2d = (float)(180 / 3.14159265358979323846);
  k.p1 = 0.9997878412794807f * r2d;
  k.p3 = -0.3258083974640975f * r2d;
  k.p5 = 0.1555786518463281f * r2d;
  k.p7 = -0.04432655554792128f * r2d;
  k.atan_eps = (float)DBL_EPSILON;
  return k;
}

}  // namespace
}  // namespace gims

using namespace gims;

extern "C" size_t gims_sift_workspace_bytes(int h, int w, int channels, int kp_cap) {
  if (h < 1 || w < 1 || (channels != 1 && channels != 3) || kp_cap < 1) return 0;
  Layout L;
  if (sift_layout(h, w, &L) != GIMS_OK) return 0;
  size_t a, b, c, d, e;
  return sift_bytes(L, kp_cap, &a, &b, &c, &d, &e);
}

extern "C" int gims_sift_detect(const unsigned char* image, int h, int w, int channels, int max_keypoints, int kp_cap,
                                void* workspace, size_t workspace_bytes, float* pt, float* size, float* angle,
                                float* response, int* octave, int* n_kp_dev, unsigned* status_dev, void* stream) {
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (!image || !workspace || !pt || !size || !angle || !response || !octave || !n_kp_dev || !status_dev) {
    set_error("gims_sift_detect: null argument");
    return GIMS_ERR_ARG;
  }
  if (h < 1 || w < 1 || (channels != 1 && channels != 3) || kp_cap < 1 || kp_cap > (1 << 26)) {
    set_error("gims_sift_detect: bad arguments (%d x %d x %d, kp_cap %d)", h, w, channels, kp_cap);
    return GIMS_ERR_ARG;
  }
  Layout L;
  GIMS_TRY(sift_layout(h, w, &L));
  size_t cand_off, rec_off, sorted_off, uniq_off, count_off;
  const size_t need = sift_bytes(L, kp_cap, &cand_off, &rec_off, &sorted_off, &uniq_off, &count_off);
  if (workspace_bytes < need) {
    set_error("gims_sift_detect: workspace of %zu bytes, %zu needed", workspace_bytes, need);
    return GIMS_ERR_ARG;
  }
  char* base = static_cast<char*>(workspace);
  float* ws = reinterpret_cast<float*>(base);
  Candidate* cand = reinterpret_cast<Candidate*>(base + cand_off);
  Record* rec = reinterpret_cast<Record*>(base + rec_off);
  Record* sorted = reinterpret_cast<Record*>(base + sorted_off);
  Record* uniq = reinterpret_cast<Record*>(base + uniq_off);
  int* counts = reinterpret_cast<int*>(base + count_off);   // candidates, raw records, unique records
  GIMS_CUDA_OK(cudaMemsetAsync(counts, 0, 4 * sizeof(int), st));
  GIMS_CUDA_OK(cudaMemsetAsync(n_kp_dev, 0, sizeof(int), st));
  if (L.oc.n == 0) return GIMS_OK;

  Kernel1D init_k, oct_k[kPerOctave];
  const float s16 = 1.6f;
  const double init_sigma = (double)sqrtf(fmaxf(s16 * s16 - 0.5f * 0.5f * 4.f, 0.01f));
  if (float_kernel(init_sigma, &init_k) < 0) { set_error("gims_sift_detect: kernel too wide"); return GIMS_ERR_ARG; }
  const double kstep = std::pow(2.0, 1.0 / kLayers);
  for (int i = 1; i < kPerOctave; ++i) {
    const double prev = std::pow(kstep, (double)(i - 1)) * kSigma, total = prev * kstep;
    if (float_kernel(std::sqrt(total * total - prev * prev), &oct_k[i]) < 0) {
      set_error("gims_sift_detect: kernel too wide");
      return GIMS_ERR_ARG;
    }
  }
  const Octaves& oc = L.oc;
  float* up = ws + L.up;
  float* tmp = ws + L.tmp;
  {
    const long long e = 4LL * h * w;
    k_sift_upsample<<<grid_for(e, kThreads), kThreads, 0, st>>>(image, h, w, channels, up);
    GIMS_LAUNCH_OK();
    k_sift_blur_rows<<<grid_for(e, kThreads), kThreads, 0, st>>>(up, tmp, 2 * h, 2 * w, init_k);
    GIMS_LAUNCH_OK();
    k_sift_blur_cols<<<grid_for(e, kThreads), kThreads, 0, st>>>(tmp, ws + oc.gauss[0], nullptr, nullptr, 2 * h, 2 * w,
                                                                 init_k);
    GIMS_LAUNCH_OK();
  }
  for (int o = 0; o < oc.n; ++o) {
    const int oh = oc.h[o], ow = oc.w[o];
    const long long plane = (long long)oh * ow;
    float* g = ws + oc.gauss[o];
    float* d = ws + oc.dog[o];
    if (o > 0) {
      k_sift_seed<<<grid_for(plane, kThreads), kThreads, 0, st>>>(ws + oc.gauss[o - 1] + kLayers * (long long)oc.h[o - 1] * oc.w[o - 1],
                                                                  oc.w[o - 1], g, oh, ow);
      GIMS_LAUNCH_OK();
    }
    for (int i = 1; i < kPerOctave; ++i) {
      k_sift_blur_rows<<<grid_for(plane, kThreads), kThreads, 0, st>>>(g + (i - 1) * plane, tmp, oh, ow, oct_k[i]);
      GIMS_LAUNCH_OK();
      k_sift_blur_cols<<<grid_for(plane, kThreads), kThreads, 0, st>>>(tmp, g + i * plane, g + (i - 1) * plane,
                                                                       d + (i - 1) * plane, oh, ow, oct_k[i]);
      GIMS_LAUNCH_OK();
    }
  }
  long long scan = 0;
  for (int o = 0; o < oc.n; ++o) scan += 3LL * oc.h[o] * oc.w[o];
  const int cand_cap = 2 * kp_cap;
  k_sift_extrema<<<grid_for(scan, kThreads), kThreads, 0, st>>>(ws, oc, cand, cand_cap, counts + 0);
  GIMS_LAUNCH_OK();
  const Consts kc = make_consts();
  const int kp_blocks = (int)std::min<long long>((cand_cap + kWarpsPerBlock - 1) / kWarpsPerBlock, 148 * 16);
  k_sift_keypoints<<<kp_blocks, kWarpsPerBlock * 32, 0, st>>>(ws, oc, cand, counts + 0, cand_cap, kc, rec, kp_cap,
                                                              counts + 1, status_dev);
  GIMS_LAUNCH_OK();
  const int rec_blocks = (kp_cap + kSortTile - 1) / kSortTile;
  k_sift_sort<<<rec_blocks, kSortTile, 0, st>>>(rec, counts + 1, kp_cap, sorted);
  GIMS_LAUNCH_OK();
  k_sift_dedupe<<<1, kFinishThreads, 0, st>>>(sorted, counts + 1, kp_cap, uniq, counts + 2, status_dev);
  GIMS_LAUNCH_OK();
  k_sift_output<<<rec_blocks, kSortTile, 0, st>>>(uniq, counts + 2, max_keypoints, pt, size, angle, response, octave,
                                                  n_kp_dev);
  GIMS_LAUNCH_OK();
  return GIMS_OK;
}

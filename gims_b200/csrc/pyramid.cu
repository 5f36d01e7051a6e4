// The 8-bit Gaussian scale space of OpenCV's SIFT on the device (frontend.gaussian_pyramid, utils/library.py:234-293):
// the image doubled with cv2.resize(INTER_LINEAR_EXACT), then per octave LAYERS + 3 = 6 levels, level i the
// cv2.GaussianBlur of level i - 1 with the incremental sigma, each next octave seeded by cv2.resize(INTER_NEAREST, 0.5) of
// level LAYERS of the previous one.  Every step is OpenCV's fixed-point integer arithmetic, so the levels are reproduced
// byte for byte (oracle/cv_pyramid_oracle.py restates it in numpy and is checked against cv2, tests/test_pyramid_cpu.py):
//   * blur kernel (getGaussianKernelBitExact + fixed point with error diffusion): n = cvRound(6 sigma + 1) | 1 taps,
//     exp(-x^2 / (2 sigma^2)) normalised in double, the left half quantised to 8 fraction bits with the rounding error
//     carried to the next tap, mirrored, centre = 256 - 2 * (sum of the left half);
//   * row pass r = sum k_j src (uint16, 1/256 units), column pass c = sum k_j r (2^-16 units), output (c + 2^15) >> 16;
//   * BORDER_REFLECT_101 repeated as often as needed (small octaves have levels narrower than the kernel radius);
//   * x2 upsample: weights 64 / 192 per axis, source index clamped, rounded as the blur;
//   * octave seed: dst[y][x] = src[2y][2x], size rint(n / 2) with ties to even (301 -> 150).
// Layout: 1 or 3 interleaved channels, every level at a 256-byte aligned offset of one buffer (the level table that
// gims_extract_patches reads).
//
// Launches: the large octaves run one grid-wide launch per step (upsample, seed, blur row pass, blur column pass); the
// row pass keeps its uint16 result in the caller's workspace.  Once an octave's levels hold at most kTailElems bytes x channels, ONE
// CTA builds every remaining octave, its row pass in shared memory and __syncthreads between the steps: the levels there
// are too small to fill the GPU, and launching each one would cost more than computing it.
#include <cmath>

#include "common.cuh"

namespace gims {
namespace {

constexpr int kPerOctave = 6;            // nOctaveLayers + 3
constexpr int kSeedLayer = 3;            // nOctaveLayers
constexpr int kFirstOctave = -1;
constexpr int kMaxTaps = 32;             // the pyramid's widest kernel has 21 taps (sigma 3.09)
constexpr int kDebugMaxTaps = 127;       // gims_debug_gaussian_kernel
constexpr int kLevelAlign = 256;
constexpr int kTailElems = 12288;        // uint16 row buffer of the single-CTA tail: 24 KB of shared memory
constexpr int kTailThreads = 1024;
constexpr int kThreads = 256;

struct Taps {
  int n;                                 // odd
  int k[kMaxTaps];
};
struct PyrTaps {
  Taps t[kPerOctave];                    // t[0] unused (level 0 of an octave is not blurred)
};

// getGaussianKernelBitExact + getGaussianKernelFixedPoint_ED (imgproc/src/smooth.dispatch.cpp) for 8-bit images
int gaussian_taps(double sigma, int* taps, int max_taps) {
  int n = (int)std::lrint(sigma * 3 * 2 + 1) | 1;
  if (n > max_taps || n < 1) return -1;
  const int n2 = n / 2;
  double vals[kDebugMaxTaps];
  const double scale2x = -0.125 / (sigma * sigma);
  double sum = 0.0;
  for (int i = 0, x = 1 - n; i < n2; ++i, x += 2) {
    vals[i] = std::exp((double)(x * x) * scale2x);
    sum += vals[i];
  }
  sum *= 2.0;
  sum += 1.0;
  const double mul = 1.0 / sum;
  double err = 0.0;
  long long tot = 0;
  for (int i = 0; i < n2; ++i) {
    const double adj = vals[i] * mul * 256.0 + err;
    const long long v = std::llrint(adj);           // cvRound: ties to even
    err = adj - (double)v;
    taps[i] = taps[n - 1 - i] = (int)v;
    tot += v;
  }
  taps[n2] = (int)(256 - 2 * tot);
  return n;
}

// the incremental sigmas as frontend.gaussian_pyramid computes them with numpy float32 scalars: k = float32(2^(1/3)),
// prev = k^(i-1) * 1.6, total = prev * k and total^2 - prev^2 all in float32, then the square root in double
void pyramid_sigmas(double* sig) {
  const float k = (float)std::pow(2.0, 1.0 / 3);
  sig[0] = 1.6;
  for (int i = 1; i < kPerOctave; ++i) {
    const float prev = powf(k, (float)(i - 1)) * 1.6f;
    const float total = prev * k;
    const float tt = total * total, pp = prev * prev;
    sig[i] = std::sqrt((double)(tt - pp));
  }
}

inline int seed_size(int n) {          // cvRound(n * 0.5)
  const int m = n >> 1;
  return (n & 1) ? m + (m & 1) : m;
}

struct Level { int h, w; long long off; };

// level table; returns the number of levels (0 if the image is too small for one octave)
int pyramid_levels(int h, int w, int channels, Level* out, int max_levels, long long* total_bytes) {
  const int bh = 2 * h, bw = 2 * w;
  const double v = (double)logf((float)(bh < bw ? bh : bw)) / std::log(2.0) - 2;
  int n_oct = (int)std::nearbyint(v) - kFirstOctave;
  if (n_oct < 0) n_oct = 0;
  const int n = n_oct * kPerOctave;
  long long off = 0;
  int ch = bh, cw = bw;
  for (int l = 0; l < n; ++l) {
    const int o = l / kPerOctave, i = l % kPerOctave;
    if (i == 0 && o > 0) { ch = seed_size(ch); cw = seed_size(cw); }
    if (l < max_levels) out[l] = {ch, cw, off};
    off += ((long long)ch * cw * channels + kLevelAlign - 1) / kLevelAlign * kLevelAlign;
  }
  *total_bytes = off;
  return n;
}

constexpr int kMaxLevels = 64 * kPerOctave;

__device__ __forceinline__ int reflect101(int i, int n) {
  if ((unsigned)i < (unsigned)n) return i;
  if (n == 1) return 0;
  const int p = 2 * (n - 1);
  i %= p;
  if (i < 0) i += p;
  return i >= n ? p - i : i;
}

// ---- the steps, each over elements [first, total) with stride `step`, so that a grid or a single CTA can run them ----

// x2 upsample (INTER_LINEAR_EXACT); elements of the destination (2h x 2w x cn)
template <int CN>
__device__ __forceinline__ void upsample_step(const unsigned char* src, int h, int w, unsigned char* dst, long long first,
                                              long long step) {
  const int dw = 2 * w;
  const long long total = (long long)2 * h * dw * CN;
  for (long long e = first; e < total; e += step) {
    const int c = (int)(e % CN);
    const long long p = e / CN;
    const int y = (int)(p / dw), x = (int)(p % dw);
    // destination i reads 0.25 * s[a] + 0.75 * s[b], b = i / 2, a = b - 1 (i even) or b + 1 (i odd), clamped
    const int xb = x >> 1, xa = min(max((x & 1) ? xb + 1 : xb - 1, 0), w - 1);
    const int yb = y >> 1, ya = min(max((y & 1) ? yb + 1 : yb - 1, 0), h - 1);
    const unsigned char* ra = src + (size_t)ya * w * CN;
    const unsigned char* rb = src + (size_t)yb * w * CN;
    const int row_a = 64 * ra[xa * CN + c] + 192 * ra[xb * CN + c];
    const int row_b = 64 * rb[xa * CN + c] + 192 * rb[xb * CN + c];
    dst[e] = (unsigned char)((64 * row_a + 192 * row_b + (1 << 15)) >> 16);
  }
}

// octave seed (INTER_NEAREST, fx = fy = 0.5)
template <int CN>
__device__ __forceinline__ void seed_step(const unsigned char* src, int sw, unsigned char* dst, int h, int w, long long first,
                                          long long step) {
  const long long total = (long long)h * w * CN;
  for (long long e = first; e < total; e += step) {
    const int c = (int)(e % CN);
    const long long p = e / CN;
    const int y = (int)(p / w), x = (int)(p % w);
    dst[e] = src[((size_t)(2 * y) * sw + 2 * x) * CN + c];
  }
}

// blur row pass: r[y][x][c] = sum_j k_j src[y][reflect(x + j - R)][c]
template <int CN>
__device__ __forceinline__ void row_step(const unsigned char* src, unsigned short* rbuf, int h, int w, const Taps& t,
                                         long long first, long long step) {
  const int r = t.n >> 1;
  const int wc = w * CN;
  const long long total = (long long)h * wc;
  for (long long e = first; e < total; e += step) {
    const int y = (int)(e / wc), xc = (int)(e % wc);
    const int x = xc / CN, c = xc % CN;
    const unsigned char* row = src + (size_t)y * wc;
    int acc = 0;
    if (x >= r && x + r < w) {
      const unsigned char* s = row + xc - r * CN;
      for (int j = 0; j < t.n; ++j) acc += t.k[j] * s[j * CN];
    } else {
      for (int j = 0; j < t.n; ++j) acc += t.k[j] * row[reflect101(x + j - r, w) * CN + c];
    }
    rbuf[e] = (unsigned short)acc;
  }
}

// blur column pass: dst = (sum_j k_j r[reflect(y + j - R)] + 2^15) >> 16
__device__ __forceinline__ void col_step(const unsigned short* rbuf, unsigned char* dst, int h, int wc, const Taps& t,
                                         long long first, long long step) {
  const int r = t.n >> 1;
  const long long total = (long long)h * wc;
  for (long long e = first; e < total; e += step) {
    const int y = (int)(e / wc), xc = (int)(e % wc);
    int acc = 0;
    if (y >= r && y + r < h) {
      const unsigned short* s = rbuf + (size_t)(y - r) * wc + xc;
      for (int j = 0; j < t.n; ++j) acc += t.k[j] * (int)s[(size_t)j * wc];
    } else {
      for (int j = 0; j < t.n; ++j) acc += t.k[j] * (int)rbuf[(size_t)reflect101(y + j - r, h) * wc + xc];
    }
    dst[e] = (unsigned char)((acc + (1 << 15)) >> 16);
  }
}

__device__ __forceinline__ long long grid_first() { return (long long)blockIdx.x * blockDim.x + threadIdx.x; }
__device__ __forceinline__ long long grid_step() { return (long long)gridDim.x * blockDim.x; }

template <int CN>
__global__ void __launch_bounds__(kThreads) k_pyr_upsample(const unsigned char* __restrict__ src, int h, int w,
                                                           unsigned char* __restrict__ dst) {
  upsample_step<CN>(src, h, w, dst, grid_first(), grid_step());
}

template <int CN>
__global__ void __launch_bounds__(kThreads) k_pyr_seed(const unsigned char* __restrict__ src, int sw,
                                                       unsigned char* __restrict__ dst, int h, int w) {
  seed_step<CN>(src, sw, dst, h, w, grid_first(), grid_step());
}

template <int CN>
__global__ void __launch_bounds__(kThreads) k_pyr_blur_rows(const unsigned char* __restrict__ src,
                                                            unsigned short* __restrict__ rbuf, int h, int w, Taps t) {
  row_step<CN>(src, rbuf, h, w, t, grid_first(), grid_step());
}

__global__ void __launch_bounds__(kThreads) k_pyr_blur_cols(const unsigned short* __restrict__ rbuf,
                                                            unsigned char* __restrict__ dst, int h, int wc, Taps t) {
  col_step(rbuf, dst, h, wc, t, grid_first(), grid_step());
}

struct TailLevels {                     // 3.6 KB: passed as a kernel argument (sm_70+ takes up to 32 KB of them)
  int first_octave, n_octaves;
  int h[64], w[64];                      // per octave (every level of an octave has the same size)
  long long off[64 * kPerOctave];        // byte offset of each level
};

// every octave from first_octave on, in one CTA: the seed of each octave from level 3 of the one before (written by this
// CTA or, for the first tail octave, by the grid launches before it), then the five blurs.  Plain (coherent) global
// loads: the CTA reads what it wrote before the last __syncthreads.
template <int CN>
__global__ void __launch_bounds__(kTailThreads) k_pyr_tail(unsigned char* base, const TailLevels tl, const PyrTaps taps) {
  __shared__ unsigned short rbuf[kTailElems];
  const long long first = threadIdx.x, step = blockDim.x;
  for (int o = tl.first_octave; o < tl.n_octaves; ++o) {
    const int h = tl.h[o], w = tl.w[o];
    const long long* off = tl.off + (size_t)o * kPerOctave;
    seed_step<CN>(base + tl.off[(size_t)(o - 1) * kPerOctave + kSeedLayer], tl.w[o - 1], base + off[0], h, w, first, step);
    __syncthreads();
    for (int i = 1; i < kPerOctave; ++i) {
      row_step<CN>(base + off[i - 1], rbuf, h, w, taps.t[i], first, step);
      __syncthreads();
      col_step(rbuf, base + off[i], h, w * CN, taps.t[i], first, step);
      __syncthreads();
    }
  }
}

int grid_for(long long elems) {
  long long b = (elems + kThreads - 1) / kThreads;
  return (int)(b < 1 ? 1 : (b > (1 << 20) ? (1 << 20) : b));
}

template <int CN>
int launch_pyramid(const unsigned char* image, int h, int w, const Level* lv, int n_levels, unsigned char* out,
                   unsigned short* rbuf, cudaStream_t st) {
  PyrTaps taps = {};
  double sig[kPerOctave];
  pyramid_sigmas(sig);
  for (int i = 1; i < kPerOctave; ++i) {
    taps.t[i].n = gaussian_taps(sig[i], taps.t[i].k, kMaxTaps);
    if (taps.t[i].n < 0) { set_error("gims_gaussian_pyramid: kernel of sigma %g too wide", sig[i]); return GIMS_ERR_ARG; }
  }
  const int n_oct = n_levels / kPerOctave;
  int tail = n_oct;
  for (int o = 1; o < n_oct; ++o)
    if ((long long)lv[o * kPerOctave].h * lv[o * kPerOctave].w * CN <= kTailElems) { tail = o; break; }
  for (int o = 0; o < tail; ++o) {
    const Level& l0 = lv[o * kPerOctave];
    const long long elems = (long long)l0.h * l0.w * CN;
    if (o == 0) {
      k_pyr_upsample<CN><<<grid_for(elems), kThreads, 0, st>>>(image, h, w, out + l0.off);
    } else {
      const Level& s = lv[(o - 1) * kPerOctave + kSeedLayer];
      k_pyr_seed<CN><<<grid_for(elems), kThreads, 0, st>>>(out + s.off, s.w, out + l0.off, l0.h, l0.w);
    }
    GIMS_LAUNCH_OK();
    for (int i = 1; i < kPerOctave; ++i) {
      const Level& a = lv[o * kPerOctave + i - 1];
      const Level& b = lv[o * kPerOctave + i];
      k_pyr_blur_rows<CN><<<grid_for(elems), kThreads, 0, st>>>(out + a.off, rbuf, a.h, a.w, taps.t[i]);
      GIMS_LAUNCH_OK();
      k_pyr_blur_cols<<<grid_for(elems), kThreads, 0, st>>>(rbuf, out + b.off, b.h, b.w * CN, taps.t[i]);
      GIMS_LAUNCH_OK();
    }
  }
  if (tail < n_oct) {
    TailLevels tl = {};
    tl.first_octave = tail;
    tl.n_octaves = n_oct;
    for (int o = 0; o < n_oct; ++o) { tl.h[o] = lv[o * kPerOctave].h; tl.w[o] = lv[o * kPerOctave].w; }
    for (int l = 0; l < n_levels; ++l) tl.off[l] = lv[l].off;
    k_pyr_tail<CN><<<1, kTailThreads, 0, st>>>(out, tl, taps);
    GIMS_LAUNCH_OK();
  }
  return GIMS_OK;
}

}  // namespace
}  // namespace gims

using namespace gims;

extern "C" int gims_pyramid_layout(int h, int w, int channels, int* n_levels, int64_t* offset_host, int* height_host,
                                   int* width_host) {
  if (!n_levels || h < 1 || w < 1 || (channels != 1 && channels != 3)) {
    set_error("gims_pyramid_layout: bad arguments (%d x %d x %d)", h, w, channels);
    return GIMS_ERR_ARG;
  }
  if (h > (1 << 14) || w > (1 << 14)) {
    set_error("gims_pyramid_layout: image %d x %d larger than 16384 x 16384", h, w);
    return GIMS_ERR_ARG;
  }
  Level lv[kMaxLevels];
  long long total = 0;
  const int n = pyramid_levels(h, w, channels, lv, kMaxLevels, &total);
  *n_levels = n;
  for (int l = 0; l < n; ++l) {
    if (offset_host) offset_host[l] = lv[l].off;
    if (height_host) height_host[l] = lv[l].h;
    if (width_host) width_host[l] = lv[l].w;
  }
  return GIMS_OK;
}

extern "C" size_t gims_pyramid_workspace_bytes(int h, int w, int channels) {
  if (h < 1 || w < 1 || (channels != 1 && channels != 3)) return 0;
  return (size_t)4 * h * w * channels * sizeof(unsigned short);     // the row pass of level 0
}

extern "C" int gims_gaussian_pyramid(const unsigned char* image, int h, int w, int channels, unsigned char* levels_out,
                                     void* workspace, size_t workspace_bytes, void* stream) {
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (!image || !levels_out || !workspace) {
    set_error("gims_gaussian_pyramid: null argument");
    return GIMS_ERR_ARG;
  }
  int n = 0;
  GIMS_TRY(gims_pyramid_layout(h, w, channels, &n, nullptr, nullptr, nullptr));
  if (workspace_bytes < gims_pyramid_workspace_bytes(h, w, channels)) {
    set_error("gims_gaussian_pyramid: workspace of %zu bytes, %zu needed", workspace_bytes,
              gims_pyramid_workspace_bytes(h, w, channels));
    return GIMS_ERR_ARG;
  }
  if (n == 0) return GIMS_OK;
  Level lv[kMaxLevels];
  long long total = 0;
  pyramid_levels(h, w, channels, lv, kMaxLevels, &total);
  unsigned short* rbuf = static_cast<unsigned short*>(workspace);
  return channels == 3 ? launch_pyramid<3>(image, h, w, lv, n, levels_out, rbuf, st)
                       : launch_pyramid<1>(image, h, w, lv, n, levels_out, rbuf, st);
}

// test hook: the 8-bit fixed-point taps cv2.GaussianBlur uses for `sigma`
extern "C" int gims_debug_gaussian_kernel(double sigma, int* taps_host, int* n_host) {
  if (!taps_host || !n_host || !(sigma > 0)) { set_error("gims_debug_gaussian_kernel: bad argument"); return GIMS_ERR_ARG; }
  const int n = gaussian_taps(sigma, taps_host, kDebugMaxTaps);
  if (n < 0) { set_error("gims_debug_gaussian_kernel: sigma %g needs more than %d taps", sigma, kDebugMaxTaps); return GIMS_ERR_ARG; }
  *n_host = n;
  return GIMS_OK;
}

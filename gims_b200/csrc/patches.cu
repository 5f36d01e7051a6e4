// Oriented keypoint patches on the device (SURVEY.md §8f row 2): replaces the per-keypoint loop of `ComputePatches`
// (utils/library.py:84-110: cv2.warpAffine(level, M, (64, 64), INTER_CUBIC, BORDER_CONSTANT) for every keypoint) and the
// 64 -> 32 px INTER_AREA resize + /255 of utils/common.py:882-884.  The Gaussian pyramid it reads is built by
// pyramid.cu, or by OpenCV on the host and uploaded (the loop this kernel replaces is 200-500 ms per image).
//
// The patch must be what OpenCV produces, bit for bit — the descriptors and therefore the matches depend on it — so the
// kernel follows OpenCV's 8-bit fixed-point warp exactly (imgproc/src/imgwarp.cpp, WarpAffineInvoker + remapBicubic):
//   * the caller passes the INVERSE map M (dst -> src) in double, inverted the way cv::warpAffine does it;
//   * source coordinates in 1/1024 pixel: X = (round(M0 x 1024) + round((M1 y + M2) 1024) + 16) >> 5, i.e. 1/32-pixel
//     positions; integer part -> 4 x 4 taps starting one pixel up-left, fractional part -> one of 32 x 32 weight sets;
//   * weights: separable cubic (A = -0.75) in float, products rounded to int16 at scale 2^15, the largest (or smallest) of
//     the four central taps adjusted so that every set sums to exactly 2^15 (initInterTab2D);
//   * pixel = saturate_u8((sum of taps x weights + 2^14) >> 15), taps outside the image contribute 0 (BORDER_CONSTANT).
// A numpy restatement of the same steps was checked against cv2.warpAffine first (147 456 pixels identical); the GPU test
// compares whole patch sets with the host path (tests/test_gpu_frontend.py).
// INTER_AREA from 64 to 32 px on the float image is the mean of 2 x 2 blocks — exact in fp32 for 8-bit inputs — then / 255.
#include <cmath>
#include <mutex>
#include <vector>

#include "common.cuh"

namespace gims {
namespace {

constexpr int kInterBits = 5, kTab = 32, kCoefBits = 15, kCoefScale = 1 << kCoefBits;
constexpr int kAbBits = 10, kAbScale = 1 << kAbBits;
constexpr int kPatchSrc = 64, kPatchDst = 32;

void cubic_coeffs(float x, float* c) {             // interpolateCubic, float arithmetic in this order
  const float A = -0.75f;
  c[0] = ((A * (x + 1) - 5 * A) * (x + 1) + 8 * A) * (x + 1) - 4 * A;
  c[1] = ((A + 2) * x - (A + 3)) * x * x + 1;
  c[2] = ((A + 2) * (1 - x) - (A + 3)) * (1 - x) * (1 - x) + 1;
  c[3] = 1.f - c[0] - c[1] - c[2];
}

// [32 fy][32 fx][4 ky][4 kx] int16 weights (initInterTab2D with fixed-point output)
void build_bicubic_tab(std::vector<short>& tab) {
  float t1[kTab][4];
  const float scale = 1.f / kTab;
  for (int i = 0; i < kTab; ++i) cubic_coeffs(i * scale, t1[i]);
  tab.assign((size_t)kTab * kTab * 16, 0);
  for (int i = 0; i < kTab; ++i)
    for (int j = 0; j < kTab; ++j) {
      short* it = &tab[((size_t)i * kTab + j) * 16];
      int isum = 0;
      for (int k1 = 0; k1 < 4; ++k1) {
        const float vy = t1[i][k1];
        for (int k2 = 0; k2 < 4; ++k2) {
          const float v = vy * t1[j][k2];
          long r = lrintf(v * kCoefScale);          // saturate_cast<short>(float): round half to even, then clamp
          r = r < -32768 ? -32768 : (r > 32767 ? 32767 : r);
          it[k1 * 4 + k2] = (short)r;
          isum += (int)r;
        }
      }
      if (isum != kCoefScale) {
        const int diff = isum - kCoefScale;
        int Mk1 = 2, Mk2 = 2, mk1 = 2, mk2 = 2;
        for (int k1 = 2; k1 < 4; ++k1)
          for (int k2 = 2; k2 < 4; ++k2) {
            if (it[k1 * 4 + k2] < it[mk1 * 4 + mk2]) { mk1 = k1; mk2 = k2; }
            else if (it[k1 * 4 + k2] > it[Mk1 * 4 + Mk2]) { Mk1 = k1; Mk2 = k2; }
          }
        if (diff < 0) it[Mk1 * 4 + Mk2] = (short)(it[Mk1 * 4 + Mk2] - diff);
        else          it[mk1 * 4 + mk2] = (short)(it[mk1 * 4 + mk2] - diff);
      }
    }
}

struct TabDev { int dev; short* ptr; };
std::mutex g_tab_mu;
std::vector<TabDev> g_tabs;

int bicubic_tab_dev(const short** out, cudaStream_t st) {
  int dev = 0;
  GIMS_CUDA_OK(cudaGetDevice(&dev));
  std::lock_guard<std::mutex> lk(g_tab_mu);
  for (const TabDev& t : g_tabs)
    if (t.dev == dev) { *out = t.ptr; return GIMS_OK; }
  std::vector<short> host;
  build_bicubic_tab(host);
  short* p = nullptr;
  GIMS_CUDA_OK(cudaMalloc(&p, host.size() * sizeof(short)));
  GIMS_CUDA_OK(cudaMemcpyAsync(p, host.data(), host.size() * sizeof(short), cudaMemcpyHostToDevice, st));
  GIMS_CUDA_OK(cudaStreamSynchronize(st));             // `host` goes out of scope; once per device and process
  g_tabs.push_back({dev, p});
  *out = p;
  return GIMS_OK;
}

struct LevelTable {            // pyramid levels inside one device buffer
  const unsigned char* base;
  const long long* offset;     // [n_levels] byte offset of level l
  const int* height;           // [n_levels]
  const int* width;            // [n_levels]
};

// One CTA per keypoint, 256 threads; thread t computes output pixels t, t + 256, ... of the 32 x 32 patch, each the mean of
// a 2 x 2 block of warped 64 x 64 pixels, every channel.
template <int CN>
__global__ void __launch_bounds__(256) k_extract_patches(LevelTable lv, const int* __restrict__ kp_level,
                                                         const double* __restrict__ kp_m, int n_kp,
                                                         const short* __restrict__ tab, float* __restrict__ out) {
  const int k = blockIdx.x;
  if (k >= n_kp) return;
  const int level = kp_level[k];
  const unsigned char* src = lv.base + lv.offset[level];
  const int h = lv.height[level], w = lv.width[level];
  const double m0 = kp_m[6 * k + 0], m1 = kp_m[6 * k + 1], m2 = kp_m[6 * k + 2];
  const double m3 = kp_m[6 * k + 3], m4 = kp_m[6 * k + 4], m5 = kp_m[6 * k + 5];
  const int round_delta = kAbScale / kTab / 2;
  for (int o = threadIdx.x; o < kPatchDst * kPatchDst; o += blockDim.x) {
    const int oy = o / kPatchDst, ox = o % kPatchDst;
    int sum[CN];
#pragma unroll
    for (int c = 0; c < CN; ++c) sum[c] = 0;
#pragma unroll
    for (int dy = 0; dy < 2; ++dy) {
      const int y = 2 * oy + dy;
      const int X0 = __double2int_rn(__dmul_rn(__dadd_rn(__dmul_rn(m1, (double)y), m2), (double)kAbScale)) + round_delta;
      const int Y0 = __double2int_rn(__dmul_rn(__dadd_rn(__dmul_rn(m4, (double)y), m5), (double)kAbScale)) + round_delta;
#pragma unroll
      for (int dx = 0; dx < 2; ++dx) {
        const int x = 2 * ox + dx;
        const int adelta = __double2int_rn(__dmul_rn(__dmul_rn(m0, (double)x), (double)kAbScale));
        const int bdelta = __double2int_rn(__dmul_rn(__dmul_rn(m3, (double)x), (double)kAbScale));
        const int X = (X0 + adelta) >> (kAbBits - kInterBits), Y = (Y0 + bdelta) >> (kAbBits - kInterBits);
        // (OpenCV stores the integer parts as int16: patches never come near +-32768 pixels)
        const int sx = (X >> kInterBits) - 1, sy = (Y >> kInterBits) - 1;
        const short* wt = tab + (((Y & (kTab - 1)) * kTab + (X & (kTab - 1))) << 4);
        int acc[CN];
#pragma unroll
        for (int c = 0; c < CN; ++c) acc[c] = 0;
#pragma unroll
        for (int k1 = 0; k1 < 4; ++k1) {
          const int yy = sy + k1;
          if (yy < 0 || yy >= h) continue;
          const unsigned char* row = src + (size_t)yy * w * CN;
#pragma unroll
          for (int k2 = 0; k2 < 4; ++k2) {
            const int xx = sx + k2;
            if (xx < 0 || xx >= w) continue;
            const int wgt = wt[k1 * 4 + k2];
#pragma unroll
            for (int c = 0; c < CN; ++c) acc[c] += (int)row[(size_t)xx * CN + c] * wgt;
          }
        }
#pragma unroll
        for (int c = 0; c < CN; ++c) {
          int v = (acc[c] + (1 << (kCoefBits - 1))) >> kCoefBits;
          v = v < 0 ? 0 : (v > 255 ? 255 : v);
          sum[c] += v;
        }
      }
    }
#pragma unroll
    for (int c = 0; c < CN; ++c)
      out[((size_t)k * kPatchDst * kPatchDst + o) * CN + c] = __fdiv_rn(__fmul_rn((float)sum[c], 0.25f), 255.0f);
  }
}

}  // namespace
}  // namespace gims

using namespace gims;

extern "C" int gims_extract_patches(const unsigned char* levels, const long long* level_offset_dev, const int* level_height_dev,
                                    const int* level_width_dev, int n_levels, int channels, const int* kp_level_dev,
                                    const double* kp_inverse_map_dev, int n_kp, float* patches_out, void* stream) {
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (!levels || !level_offset_dev || !level_height_dev || !level_width_dev || !kp_level_dev || !kp_inverse_map_dev || !patches_out) {
    set_error("gims_extract_patches: null argument");
    return GIMS_ERR_ARG;
  }
  if (n_levels < 1 || n_kp < 0 || (channels != 1 && channels != 3)) {
    set_error("gims_extract_patches: bad sizes (levels %d, keypoints %d, channels %d)", n_levels, n_kp, channels);
    return GIMS_ERR_ARG;
  }
  if (n_kp == 0) return GIMS_OK;
  const short* tab = nullptr;
  GIMS_TRY(bicubic_tab_dev(&tab, st));
  LevelTable lv = {levels, level_offset_dev, level_height_dev, level_width_dev};
  if (channels == 3) k_extract_patches<3><<<n_kp, 256, 0, st>>>(lv, kp_level_dev, kp_inverse_map_dev, n_kp, tab, patches_out);
  else               k_extract_patches<1><<<n_kp, 256, 0, st>>>(lv, kp_level_dev, kp_inverse_map_dev, n_kp, tab, patches_out);
  GIMS_LAUNCH_OK();
  count_launch();
  return GIMS_OK;
}

// test hook: the 32 x 32 x 16 int16 weight table as built on the host (tests/test_frontend_cpu.py compares it with a numpy
// restatement that is itself checked against cv2.warpAffine)
extern "C" int gims_debug_bicubic_table(short* out_host) {
  if (!out_host) { set_error("gims_debug_bicubic_table: null argument"); return GIMS_ERR_ARG; }
  std::vector<short> t;
  build_bicubic_tab(t);
  for (size_t i = 0; i < t.size(); ++i) out_host[i] = t[i];
  return GIMS_OK;
}


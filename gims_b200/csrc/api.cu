// C-ABI entry points of libgims_b200.so (declared in include/gims_b200.h): model handle, per-stage
// forwards and the whole-pair forward that chains them (GMatcher.forward, models/gmatcher.py:219-307).
#include <stdarg.h>
#include <string.h>

#include <atomic>
#include <mutex>
#include <new>
#include <vector>

#include "common.cuh"

namespace gims {

static thread_local char g_err[512] = "";
static std::atomic<long long> g_launches{0};

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
void count_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }

// ---- profiler ---------------------------------------------------------------------------------
static std::mutex g_prof_mu;
static int g_prof_class = GIMS_PROF_NONE;
static int g_prof_max = 0;
static std::vector<cudaEvent_t> g_prof_ev;   // pairs (start, stop)

ProfScope::ProfScope(int kernel_class, cudaStream_t s) : slot(-1), st(s) {
  if (g_prof_class != kernel_class) return;
  std::lock_guard<std::mutex> lk(g_prof_mu);
  if (g_prof_class != kernel_class || (int)g_prof_ev.size() / 2 >= g_prof_max) return;
  cudaEvent_t a, b;
  if (cudaEventCreate(&a) != cudaSuccess) return;
  if (cudaEventCreate(&b) != cudaSuccess) { cudaEventDestroy(a); return; }
  slot = (int)g_prof_ev.size();
  g_prof_ev.push_back(a);
  g_prof_ev.push_back(b);
  cudaEventRecord(a, st);
}
ProfScope::~ProfScope() {
  if (slot < 0) return;
  std::lock_guard<std::mutex> lk(g_prof_mu);
  if (slot + 1 < (int)g_prof_ev.size()) cudaEventRecord(g_prof_ev[slot + 1], st);
}

// ---- cooperative-kernel chain -------------------------------------------------------------------
static std::mutex g_coop_mu;
static cudaEvent_t g_coop_ev[64][2];
static bool g_coop_has[64][2];
static unsigned g_coop_next[64];

static std::mutex g_coop_launch_mu;
void coop_chain_lock() { g_coop_launch_mu.lock(); }
void coop_chain_unlock() { g_coop_launch_mu.unlock(); }

int coop_chain_pick_lane() {
  static const int lanes = [] { const char* e = getenv("GIMS_COOP_LANES"); int v = e ? atoi(e) : 2; return v == 1 ? 1 : 2; }();
  if (lanes == 1) return 0;          // (tuning knob: at most one half-GPU cooperative kernel at a time)
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev >= 64) return 0;
  std::lock_guard<std::mutex> lk(g_coop_mu);
  return (int)(g_coop_next[dev]++ & 1u);
}
int coop_chain_wait(cudaStream_t st, int lane) {
  int dev = 0;
  GIMS_CUDA_OK(cudaGetDevice(&dev));
  if (dev >= 64) return GIMS_OK;
  std::lock_guard<std::mutex> lk(g_coop_mu);
  for (int l = 0; l < 2; ++l)
    if ((lane < 0 || lane == l) && g_coop_has[dev][l]) GIMS_CUDA_OK(cudaStreamWaitEvent(st, g_coop_ev[dev][l], 0));
  return GIMS_OK;
}
int coop_chain_record(cudaStream_t st, int lane) {
  int dev = 0;
  GIMS_CUDA_OK(cudaGetDevice(&dev));
  if (dev >= 64) return GIMS_OK;
  std::lock_guard<std::mutex> lk(g_coop_mu);
  for (int l = 0; l < 2; ++l) {
    if (lane >= 0 && lane != l) continue;
    if (!g_coop_has[dev][l]) {
      GIMS_CUDA_OK(cudaEventCreateWithFlags(&g_coop_ev[dev][l], cudaEventDisableTiming));
      g_coop_has[dev][l] = true;
    }
    GIMS_CUDA_OK(cudaEventRecord(g_coop_ev[dev][l], st));
  }
  return GIMS_OK;
}

}  // namespace gims

extern "C" int gims_profile_begin(int kernel_class, int max_launches) {
  std::lock_guard<std::mutex> lk(gims::g_prof_mu);
  for (cudaEvent_t e : gims::g_prof_ev) cudaEventDestroy(e);
  gims::g_prof_ev.clear();
  gims::g_prof_class = kernel_class;
  gims::g_prof_max = max_launches;
  return GIMS_OK;
}

extern "C" int gims_profile_end(double* total_ms, int* launches) {
  std::lock_guard<std::mutex> lk(gims::g_prof_mu);
  gims::g_prof_class = GIMS_PROF_NONE;
  double tot = 0.0;
  int n = 0;
  for (size_t i = 0; i + 1 < gims::g_prof_ev.size(); i += 2) {
    float ms = 0.f;
    if (cudaEventSynchronize(gims::g_prof_ev[i + 1]) == cudaSuccess &&
        cudaEventElapsedTime(&ms, gims::g_prof_ev[i], gims::g_prof_ev[i + 1]) == cudaSuccess) {
      tot += ms;
      ++n;
    }
  }
  for (cudaEvent_t e : gims::g_prof_ev) cudaEventDestroy(e);
  gims::g_prof_ev.clear();
  if (total_ms) *total_ms = tot;
  if (launches) *launches = n;
  return GIMS_OK;
}

using namespace gims;

// Packed weight blobs, in the order gims_b200/packing.py emits them.
struct Wt {                    // one weight matrix [N][K]: fp32 + its tensor-core planes
  const float* w;
  const float* hi;             // tf32(W)
  const float* lo;             // W - tf32(W)
  const void* h16;             // fp16(W * 2^e)
  const void* l16;             // fp16(W * 2^e - h16)
  const float* sinv;           // 2^-e
  WPlanes planes() const { WPlanes p; p.hi32 = hi; p.lo32 = lo; p.h16 = h16; p.l16 = l16; p.sinv = sinv; return p; }
};

struct gims_model {
  gims_config cfg;
  const float* bin_score;
  Wt kenc_w[GIMS_MAX_KENC];
  const float* kenc_b[GIMS_MAX_KENC];
  Wt sage_w[3];                // L0: [256][256] rows 0..127 fc_neigh, 128..255 fc_self
                               // L1: [128][256] cols 0..127 fc_self, 128..255 fc_neigh;  L2: [256][256] likewise
  const float* sage_b[3];
  Wt wqkv[GIMS_MAX_LAYERS];    // [768][256]  Q|K|V rows, head-major
  const float* bqkv[GIMS_MAX_LAYERS];
  Wt w1[GIMS_MAX_LAYERS];      // [512][512]  BN folded, `merge` composed in: input = [x | attention output]
  const float* b1[GIMS_MAX_LAYERS];
  Wt w2[GIMS_MAX_LAYERS];      // [256][512]
  const float* b2[GIMS_MAX_LAYERS];
  Wt wfinal;
  const float* bfinal;
};

static std::atomic<int> g_gemm_mode{GIMS_GEMM_TC_F16};
// projection GEMM operands: fp16 hi + lo in the f16 / bf16 modes (GIMS_GEMM_F16_PROJ=0 keeps them on 3xTF32)
static int gemm_prec(int mode) {
  static const int on = [] { const char* e = getenv("GIMS_GEMM_F16_PROJ"); return e ? atoi(e) : 1; }();
  return (on && (mode == GIMS_GEMM_TC_F16 || mode == GIMS_GEMM_BF16)) ? 1 : 0;
}

extern "C" int gims_version(void) { return 100; }
extern "C" const char* gims_last_error(void) { return g_err; }
extern "C" long long gims_launch_count(void) { return g_launches.load(); }

extern "C" int gims_set_gemm_mode(int mode) {
  if (mode < GIMS_GEMM_SIMT || mode > GIMS_GEMM_BF16) { set_error("gims_set_gemm_mode: bad mode %d", mode); return GIMS_ERR_ARG; }
  g_gemm_mode.store(mode);
  return GIMS_OK;
}
extern "C" int gims_get_gemm_mode(void) { return g_gemm_mode.load(); }

extern "C" int gims_packed_blob_count(const gims_config* c) {
  if (!c) return -1;
  // every weight matrix contributes 6 blobs (W, tf32 hi / lo, fp16 hi / lo, 2^-e), every bias 1
  return 1 + 7 * c->kenc_num + 7 * 3 + 21 * c->num_layers + 7;
}

extern "C" int gims_model_create(const gims_config* c, const float* packed, const int64_t* off, int n_off,
                                 gims_model** out) {
  if (!c || !packed || !off || !out) { set_error("gims_model_create: null argument"); return GIMS_ERR_ARG; }
  if (c->descriptor_dim != kD) { set_error("gims_model_create: descriptor_dim %d unsupported (built for 256)", c->descriptor_dim); return GIMS_ERR_ARG; }
  if (c->num_layers < 0 || c->num_layers > GIMS_MAX_LAYERS || c->kenc_num < 2 || c->kenc_num > GIMS_MAX_KENC) {
    set_error("gims_model_create: bad layer counts"); return GIMS_ERR_ARG;
  }
  if (c->kenc_dims[0] != 2 || c->kenc_dims[c->kenc_num] != kD) { set_error("gims_model_create: kenc must map 2 -> 256"); return GIMS_ERR_ARG; }
  for (int i = 1; i < c->kenc_num; ++i)
    if (c->kenc_dims[i] % 16) { set_error("gims_model_create: kenc width %d not a multiple of 16", c->kenc_dims[i]); return GIMS_ERR_ARG; }
  if (n_off != gims_packed_blob_count(c)) { set_error("gims_model_create: expected %d blobs, got %d", gims_packed_blob_count(c), n_off); return GIMS_ERR_ARG; }
  gims_model* m = new (std::nothrow) gims_model;
  if (!m) { set_error("gims_model_create: out of host memory"); return GIMS_ERR_ARG; }
  m->cfg = *c;
  int k = 0;
  auto next = [&]() { return packed + off[k++]; };
  auto next_w = [&]() { Wt w; w.w = next(); w.hi = next(); w.lo = next(); w.h16 = next(); w.l16 = next(); w.sinv = next(); return w; };
  m->bin_score = next();
  for (int i = 0; i < c->kenc_num; ++i) { m->kenc_w[i] = next_w(); m->kenc_b[i] = next(); }
  for (int i = 0; i < 3; ++i) { m->sage_w[i] = next_w(); m->sage_b[i] = next(); }
  for (int l = 0; l < c->num_layers; ++l) {
    m->wqkv[l] = next_w(); m->bqkv[l] = next();
    m->w1[l] = next_w(); m->b1[l] = next(); m->w2[l] = next_w(); m->b2[l] = next();
  }
  m->wfinal = next_w(); m->bfinal = next();
  *out = m;
  return GIMS_OK;
}

extern "C" void gims_model_destroy(gims_model* m) { delete m; }

// Y = epi(A W^T + bias): tcgen05 kernel when the shape allows and the mode asks for it (fp16 hi+lo operands in the f16 / bf16
// modes, 3xTF32 otherwise), else fp32 SIMT.
static int gemm(const float* A0, int lda0, int K0, const float* A1, int lda1, int K1, const Wt& W, const float* bias,
                const float* R, int ldr, float* Y, int ldy, int N, int relu, Segs s, int mode, cudaStream_t st,
                unsigned* status = nullptr) {
  GemmArgs g;
  g.A0 = A0; g.lda0 = lda0; g.K0 = K0; g.A1 = A1; g.lda1 = lda1; g.K1 = K1; g.W = W.w; g.bias = bias;
  g.R = R; g.ldr = ldr; g.Y = Y; g.ldy = ldy; g.N = N; g.relu = relu; g.segs = s; g.status = status;
  bool tc_ok = W.hi && W.lo && K0 % 32 == 0 && K1 % 32 == 0 && N % 32 == 0 && lda0 % 4 == 0 && (K1 == 0 || lda1 % 4 == 0);
  if (mode != GIMS_GEMM_SIMT && tc_ok) return launch_gemm_tc(g, W.planes(), gemm_prec(mode), st);
  return launch_gemm(g, st);
}

// a-9 ------------------------------------------------------------------------------------------
static int sage_fwd(const gims_model* m, const float* feat, const int* indptr, const int* indices, int n_max,
                    const int* n_dev, float* out, float* scratch, int mode, cudaStream_t st) {
  if (!m || n_max < 1) { set_error("gims_sage_forward: bad arguments"); return GIMS_ERR_ARG; }
  const int H = kD / 2;
  float* y0 = scratch;                          // [n][256]  = feat @ [Wn0; Ws0]^T
  float* h1 = y0 + (size_t)n_max * kD;          // [n][128]
  float* agg = h1 + (size_t)n_max * H;          // [n][128]
  float* h2 = agg + (size_t)n_max * H;          // [n][128]   (total 2.5 * n * 256 floats)
  Segs s = one_seg(n_max, n_dev);
  // layer 0 (256 -> 128, fc_neigh before aggregation)
  GIMS_TRY(gemm(feat, kD, kD, nullptr, 0, 0, m->sage_w[0], nullptr, nullptr, 0, y0, kD, kD, 0, s, mode, st));
  GIMS_TRY(launch_sage_aggregate(y0, kD, H, indptr, indices, n_max, n_dev, y0 + H, kD, m->sage_b[0], 1, h1, H, st));
  // layer 1 (128 -> 128, aggregate then fc_neigh)
  GIMS_TRY(launch_sage_aggregate(h1, H, H, indptr, indices, n_max, n_dev, nullptr, 0, nullptr, 0, agg, H, st));
  GIMS_TRY(gemm(h1, H, H, agg, H, H, m->sage_w[1], m->sage_b[1], nullptr, 0, h2, H, H, 1, s, mode, st));
  // layer 2 (128 -> 256)
  GIMS_TRY(launch_sage_aggregate(h2, H, H, indptr, indices, n_max, n_dev, nullptr, 0, nullptr, 0, agg, H, st));
  GIMS_TRY(gemm(h2, H, H, agg, H, H, m->sage_w[2], m->sage_b[2], nullptr, 0, out, kD, kD, 0, s, mode, st));
  return GIMS_OK;
}
extern "C" int gims_sage_forward(const gims_model* m, const float* feat, const int* indptr, const int* indices,
                                 int n_max, const int* n_dev, float* out, float* scratch, void* stream) {
  return sage_fwd(m, feat, indptr, indices, n_max, n_dev, out, scratch, g_gemm_mode.load(), static_cast<cudaStream_t>(stream));
}

// a-8 + a-10 -----------------------------------------------------------------------------------
static int kenc_fwd(const gims_model* m, const float* kpts, int n_max, const int* n_dev, float img_w, float img_h,
                    const float* add, float* desc, float* scratch, int mode, cudaStream_t st) {
  if (!m || n_max < 1) { set_error("gims_kenc_forward: bad arguments"); return GIMS_ERR_ARG; }
  const gims_config& c = m->cfg;
  float* buf[2] = {scratch, scratch + (size_t)n_max * kD};
  Segs s = one_seg(n_max, n_dev);
  GIMS_TRY(launch_kenc_first(kpts, n_max, n_dev, img_w, img_h, m->kenc_w[0].w, m->kenc_b[0], c.kenc_dims[1], buf[0], st));
  int cur = 0;
  for (int i = 1; i < c.kenc_num; ++i) {
    int cin = c.kenc_dims[i], cout = c.kenc_dims[i + 1];
    bool last = (i == c.kenc_num - 1);
    float* y = last ? desc : buf[cur ^ 1];
    GIMS_TRY(gemm(buf[cur], cin, cin, nullptr, 0, 0, m->kenc_w[i], m->kenc_b[i], last ? add : nullptr, kD, y,
                              last ? kD : cout, cout, last ? 0 : 1, s, mode, st));
    cur ^= 1;
  }
  return GIMS_OK;
}
extern "C" int gims_kenc_forward(const gims_model* m, const float* kpts, int n_max, const int* n_dev, float img_w,
                                 float img_h, const float* add, float* desc, float* scratch, void* stream) {
  return kenc_fwd(m, kpts, n_max, n_dev, img_w, img_h, add, desc, scratch, g_gemm_mode.load(), static_cast<cudaStream_t>(stream));
}

// a-11 + a-12 ----------------------------------------------------------------------------------
// qkv (or its planes: 6 * rows * 256 floats + padding of the transposed V rows) | att | msg | hid
static size_t attn_scratch_floats(size_t rows, int nseg) {
  return rows * (6 * kD + kD + kD + 2 * kD) + (size_t)nseg * 128 * kD;
}
extern "C" size_t gims_attn_scratch_floats(int rows) { return attn_scratch_floats((size_t)rows, 2); }

// One AttentionalPropagation layer for every segment of `s` (2 per pair, pair-major: segment i ^ 1 is the other image)
static int attn_layer(const gims_model* m, int layer, float* desc, const Segs& s, float* scratch, unsigned* status_dev,
                      int mode, cudaStream_t st) {
  if (!m || layer < 0 || layer >= m->cfg.num_layers) { set_error("gims_attn_layer_forward: bad layer %d", layer); return GIMS_ERR_ARG; }
  if (s.nseg < 2 || (s.nseg & 1)) { set_error("gims_attn_layer_forward: segments must come in pairs"); return GIMS_ERR_ARG; }
  const size_t rows = (size_t)segs_rows(s);
  float* qkv = scratch;                    // [rows][768]  (SIMT)  |  Qp, Kp, Vt planes (tensor cores)
  float* att = qkv + rows * 6 * kD + (size_t)s.nseg * 128 * kD;   // [rows][256]
  float* msg = att + rows * kD;            // [rows][256]
  float* hid = msg + rows * kD;            // [rows][512]
  const int cross = m->cfg.layer_is_cross[layer];
  if (mode != GIMS_GEMM_SIMT) {
    QkvPlanes pl;
    pl.qp = qkv; pl.kp = pl.qp + 2 * rows * kD; pl.vt = static_cast<float*>(pl.kp) + 2 * rows * kD;
    pl.ldv = attn_vt_layout(s, pl.vbase);  // <= rows + 63 * nseg
    for (int i = s.nseg; i < kMaxSegs; ++i) pl.vbase[i] = 0;
    pl.fmt = mode == GIMS_GEMM_TC_F16 ? 0 : (mode == GIMS_GEMM_BF16 ? 1 : -1);
    pl.planes = mode == GIMS_GEMM_BF16 ? 1 : 2;
    pl.status = status_dev;
    GemmArgs g;
    g.A0 = desc; g.lda0 = kD; g.K0 = kD; g.A1 = nullptr; g.lda1 = 0; g.K1 = 0; g.W = m->wqkv[layer].w;
    g.bias = m->bqkv[layer]; g.R = nullptr; g.ldr = 0; g.Y = nullptr; g.ldy = 0; g.N = 3 * kD; g.relu = 0; g.segs = s;
    g.status = status_dev;
    GIMS_TRY(launch_gemm_tc(g, m->wqkv[layer].planes(), gemm_prec(mode), st, &pl));
    if (pl.fmt >= 0) GIMS_TRY(launch_attention_f16(pl, att, s, cross, st));
    else             GIMS_TRY(launch_attention_tc(pl, att, s, cross, st));
  } else {
    GIMS_TRY(gemm(desc, kD, kD, nullptr, 0, 0, m->wqkv[layer], m->bqkv[layer], nullptr, 0, qkv, 3 * kD, 3 * kD, 0, s, mode, st));
    GIMS_TRY(launch_attention(qkv, att, s, cross, st));
  }
  (void)msg;   // the merge conv is composed into W1 at pack time
  GIMS_TRY(gemm(desc, kD, kD, att, kD, kD, m->w1[layer], m->b1[layer], nullptr, 0, hid, 2 * kD, 2 * kD, 1, s, mode, st, status_dev));
  GIMS_TRY(gemm(hid, 2 * kD, 2 * kD, nullptr, 0, 0, m->w2[layer], m->b2[layer], desc, kD, desc, kD, kD, 0, s, mode, st, status_dev));
  return GIMS_OK;
}
extern "C" int gims_attn_layer_forward(const gims_model* m, int layer, float* desc, int n0_max, int n1_max,
                                       const int* n_dev, float* scratch, unsigned* status_dev, void* stream) {
  return attn_layer(m, layer, desc, two_segs(n0_max, n1_max, n_dev), scratch, status_dev, g_gemm_mode.load(),
                    static_cast<cudaStream_t>(stream));
}

// a-13 -----------------------------------------------------------------------------------------
static int final_proj(const gims_model* m, const float* desc, const Segs& s, float* mdesc, int mode, cudaStream_t st,
                      unsigned* status = nullptr) {
  return gemm(desc, kD, kD, nullptr, 0, 0, m->wfinal, m->bfinal, nullptr, 0, mdesc, kD, kD, 0, s, mode, st, status);
}
static int score_matrix(const gims_model* m, const float* mdesc, int n0_max, int n1_max, const int* n_dev, float* couplings,
                        float* scratch, int mode, cudaStream_t st, unsigned* status = nullptr) {
  if (mode != GIMS_GEMM_SIMT && scratch) {
    // the bf16 variant (BASELINE configs[4]: "bf16 score GEMM") runs the score matrix on ONE bf16 plane per operand
    const int prec = mode == GIMS_GEMM_BF16 ? 2 : gemm_prec(mode);
    GIMS_TRY(launch_score_gemm_tc(mdesc, n0_max, n1_max, n_dev, scratch, couplings, prec, status, st));
    GIMS_TRY(launch_score_border(n0_max, n1_max, n_dev, m->bin_score, couplings, st));
  } else {
    GIMS_TRY(launch_score_gemm(mdesc, n0_max, n1_max, n_dev, m->bin_score, couplings, st));
  }
  return GIMS_OK;
}
static int final_scores(const gims_model* m, const float* desc, int n0_max, int n1_max, const int* n_dev, float* mdesc,
                        float* couplings, float* scratch, int mode, cudaStream_t st) {
  if (!m) { set_error("gims_final_scores: null model"); return GIMS_ERR_ARG; }
  GIMS_TRY(final_proj(m, desc, two_segs(n0_max, n1_max, n_dev), mdesc, mode, st));
  return score_matrix(m, mdesc, n0_max, n1_max, n_dev, couplings, scratch, mode, st);
}
extern "C" int gims_final_scores(const gims_model* m, const float* desc, int n0_max, int n1_max, const int* n_dev,
                                 float* mdesc, float* couplings, float* scratch, void* stream) {
  return final_scores(m, desc, n0_max, n1_max, n_dev, mdesc, couplings, scratch, g_gemm_mode.load(), static_cast<cudaStream_t>(stream));
}

// test / bring-up entry points ----------------------------------------------------------------
extern "C" int gims_linear(const float* A0, int lda0, int K0, const float* A1, int lda1, int K1, const float* W,
                           const float* W_hi, const float* W_lo, const void* W_h16, const void* W_l16, const float* W_sinv,
                           const float* bias, const float* R, int ldr, float* Y,
                           int ldy, int N, int relu, int rows_max, const int* rows_dev, int mode, unsigned* status_dev,
                           void* stream) {
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  GemmArgs g;
  g.A0 = A0; g.lda0 = lda0; g.K0 = K0; g.A1 = A1; g.lda1 = lda1; g.K1 = K1; g.W = W; g.bias = bias;
  g.R = R; g.ldr = ldr; g.Y = Y; g.ldy = ldy; g.N = N; g.relu = relu; g.segs = one_seg(rows_max, rows_dev); g.status = status_dev;
  if (mode != GIMS_GEMM_SIMT) {
    if (!W_hi || !W_lo) { set_error("gims_linear: tensor-core mode needs W_hi / W_lo"); return GIMS_ERR_ARG; }
    WPlanes p; p.hi32 = W_hi; p.lo32 = W_lo; p.h16 = W_h16; p.l16 = W_l16; p.sinv = W_sinv;
    const int prec = (mode == GIMS_GEMM_TC_F16 || mode == GIMS_GEMM_BF16) ? 1 : 0;
    if (prec && (!W_h16 || !W_l16 || !W_sinv)) { set_error("gims_linear: fp16 mode needs W_h16 / W_l16 / W_sinv"); return GIMS_ERR_ARG; }
    return launch_gemm_tc(g, p, prec, st);
  }
  return launch_gemm(g, st);
}

extern "C" int gims_debug_attention_trace(long long* dev_buf) { return set_attention_trace(dev_buf); }
extern "C" int gims_debug_gemm_trace(long long* dev_buf) { return set_gemm_trace(dev_buf); }

extern "C" int gims_split_tf32(const float* x, float* hi, float* lo, size_t n, void* stream) {
  if (n % 4) { set_error("gims_split_tf32: n must be a multiple of 4"); return GIMS_ERR_ARG; }
  return launch_split_planes(x, hi, lo, n, static_cast<cudaStream_t>(stream));
}

namespace {
__global__ void k_or_status(const unsigned* __restrict__ src, unsigned* __restrict__ dst, unsigned mask) {
  const unsigned v = *src & mask;
  if (v) atomicOr(dst, v);
}
int launch_or_status(const unsigned* src, unsigned* dst, unsigned mask, cudaStream_t st) {
  k_or_status<<<1, 1, 0, st>>>(src, dst, mask);
  GIMS_LAUNCH_OK();
  return GIMS_OK;
}
}  // namespace

// whole pairs ----------------------------------------------------------------------------------
// A batch of up to GIMS_MAX_BATCH pairs goes through the dense stages TOGETHER: the rows of all images are stacked in one
// activation buffer (image 0 of pair 0, image 1 of pair 0, image 0 of pair 1, ...), so that each projection GEMM and each
// attention layer is ONE launch over all of them (2 P row segments).  The graph stages, the score matrix and the Sinkhorn
// kernel run per pair on the same stream and share one scratch area each.
namespace {
struct BatchWs {
  void* agc[2];     size_t agc_bytes;          // one per image: the two graph chains of a pair run on two streams
  float* sage_out;  // [rows][256]
  float* desc;      // [rows][256]
  float* mdesc;     // [rows][256]
  float* scratch;   // attention scratch (also SAGE / kenc / score-plane scratch)
  float* couplings;
  void* sink;       size_t sink_bytes;
};
size_t carve_batch(BatchWs& w, void* base, size_t cap, int n_pairs, const int* n0, const int* n1, int edge_cap) {
  Arena a(base, cap);
  size_t rows = 0, coup = 0, sink = 0;
  int nmax = 0;
  for (int p = 0; p < n_pairs; ++p) {
    rows += (size_t)n0[p] + n1[p];
    nmax = n0[p] > nmax ? n0[p] : nmax; nmax = n1[p] > nmax ? n1[p] : nmax;
    size_t c = (size_t)(n0[p] + 1) * coup_ld(n1[p]);
    coup = c > coup ? c : coup;
    size_t sb = gims_sinkhorn_workspace_bytes(n0[p], n1[p]);
    sink = sb > sink ? sb : sink;
  }
  w.agc_bytes = gims_agc_workspace_bytes(nmax, edge_cap);
  w.agc[0] = a.take<char>(w.agc_bytes);
  w.agc[1] = a.take<char>(w.agc_bytes);
  w.sage_out = a.take<float>(rows * kD);
  w.desc = a.take<float>(rows * kD);
  w.mdesc = a.take<float>(rows * kD);
  w.scratch = a.take<float>(attn_scratch_floats(rows, 2 * n_pairs));
  w.couplings = a.take<float>(coup);
  w.sink_bytes = sink;
  w.sink = a.take<char>(sink);
  return align_up(a.off, 256);
}
// Image 0 and image 1 of a pair are independent until the first attention layer: graph construction, GraphSAGE and the
// keypoint encoder of image 1 run on a side stream forked from the caller's stream and joined before the layers (about
// 60 small, strictly serial launches per image — alone on one stream they are a third of a single caller's latency).
// One side stream + two events per caller stream, created on first use (GIMS_FORK_IMAGES=0: everything on one stream).
struct SideStream { cudaStream_t s; cudaEvent_t fork, join; };
static std::mutex g_side_mu;
static std::vector<std::pair<std::pair<int, cudaStream_t>, SideStream>> g_side;
bool fork_images() {
  static const bool on = [] { const char* e = getenv("GIMS_FORK_IMAGES"); return !(e && e[0] == '0'); }();
  return on;
}
int side_stream_for(cudaStream_t main, SideStream& out) {
  int dev = 0;
  GIMS_CUDA_OK(cudaGetDevice(&dev));
  std::lock_guard<std::mutex> lk(g_side_mu);
  for (auto& e : g_side)
    if (e.first.first == dev && e.first.second == main) { out = e.second; return GIMS_OK; }
  if (g_side.size() >= 64) { out = {main, nullptr, nullptr}; return GIMS_OK; }   // a caller that keeps making streams: no fork
  SideStream n;
  GIMS_CUDA_OK(cudaStreamCreateWithFlags(&n.s, cudaStreamNonBlocking));
  GIMS_CUDA_OK(cudaEventCreateWithFlags(&n.fork, cudaEventDisableTiming));
  GIMS_CUDA_OK(cudaEventCreateWithFlags(&n.join, cudaEventDisableTiming));
  g_side.push_back({{dev, main}, n});
  out = n;
  return GIMS_OK;
}

__global__ void k_copy_rows(const float* __restrict__ src, float* __restrict__ dst, size_t n4) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n4) reinterpret_cast<float4*>(dst)[i] = reinterpret_cast<const float4*>(src)[i];
}
int copy_rows(const float* src, float* dst, size_t floats, cudaStream_t st) {
  k_copy_rows<<<(unsigned)((floats / 4 + 255) / 256), 256, 0, st>>>(src, dst, floats / 4);
  GIMS_LAUNCH_OK();
  return GIMS_OK;
}

int validate_pair(const gims_pair_inputs* in, const gims_pair_outputs* o) {
  const int n0 = in->n[0], n1 = in->n[1];
  // validate everything BEFORE the first launch: a late error would leave half a forward enqueued
  if (n0 < 2 || n1 < 2 || n0 > GIMS_MAX_KPTS || n1 > GIMS_MAX_KPTS) {
    set_error("gims_forward_pair: keypoint counts (%d, %d) outside [2, %d]", n0, n1, GIMS_MAX_KPTS);
    return GIMS_ERR_ARG;
  }
  if (in->edge_cap < 1) { set_error("gims_forward_pair: edge_cap %d", in->edge_cap); return GIMS_ERR_ARG; }
  if (!o->n_kept_dev || !o->n_edges_dev || !o->n_comp_dev || !o->thr_dev || !o->mdesc || !o->u || !o->v || !o->status_dev) {
    set_error("gims_forward_pair: null output pointer");
    return GIMS_ERR_ARG;
  }
  for (int s = 0; s < 2; ++s) {
    if (!in->kpts[s] || !in->desc[s] || !in->scores[s] || !o->kept_idx[s] || !o->csr_indptr[s] || !o->csr_indices[s] ||
        !o->kpts[s] || !o->feat[s] || !o->scores[s] || !o->matches[s] || !o->mscores[s] || !o->indices[s]) {
      set_error("gims_forward_pair: null pointer for image %d", s);
      return GIMS_ERR_ARG;
    }
    long long len = (long long)in->n[s] * (in->n[s] - 1) / 2;
    if (in->k_rank[s] < 0 || in->k_rank[s] >= len) {
      set_error("gims_forward_pair: k_rank[%d]=%lld outside [0, %lld)", s, in->k_rank[s], len);
      return GIMS_ERR_ARG;
    }
  }
  return GIMS_OK;
}
}  // namespace

extern "C" size_t gims_batch_workspace_bytes(int n_pairs, const int* n0_host, const int* n1_host, int edge_cap) {
  if (n_pairs < 1 || n_pairs > GIMS_MAX_BATCH || !n0_host || !n1_host) return 0;
  BatchWs w;
  return carve_batch(w, nullptr, 0, n_pairs, n0_host, n1_host, edge_cap);
}

extern "C" size_t gims_pair_workspace_bytes(const gims_model* m, int n0, int n1, int edge_cap) {
  (void)m;
  return gims_batch_workspace_bytes(1, &n0, &n1, edge_cap);
}

extern "C" int gims_forward_pairs(const gims_model* m, int n_pairs, const gims_pair_inputs* in, const gims_pair_outputs* out,
                                  void* workspace, size_t workspace_bytes, void* stream) {
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (!m || !in || !out || !workspace) { set_error("gims_forward_pairs: null argument"); return GIMS_ERR_ARG; }
  if (n_pairs < 1 || n_pairs > GIMS_MAX_BATCH) { set_error("gims_forward_pairs: n_pairs %d outside [1, %d]", n_pairs, GIMS_MAX_BATCH); return GIMS_ERR_ARG; }
  int n0[GIMS_MAX_BATCH], n1[GIMS_MAX_BATCH], edge_cap = 0;
  const int mode = in[0].gemm_mode > 0 ? in[0].gemm_mode - 1 : g_gemm_mode.load();
  if (mode < GIMS_GEMM_SIMT || mode > GIMS_GEMM_BF16) { set_error("gims_forward_pairs: gemm_mode %d", in[0].gemm_mode); return GIMS_ERR_ARG; }
  for (int p = 0; p < n_pairs; ++p) {
    GIMS_TRY(validate_pair(in + p, out + p));
    if (in[p].gemm_mode != in[0].gemm_mode) { set_error("gims_forward_pairs: the pairs of a batch must share gemm_mode"); return GIMS_ERR_ARG; }
    n0[p] = in[p].n[0]; n1[p] = in[p].n[1];
    edge_cap = in[p].edge_cap > edge_cap ? in[p].edge_cap : edge_cap;
  }
  BatchWs w;
  size_t need = carve_batch(w, workspace, workspace_bytes, n_pairs, n0, n1, edge_cap);
  if (need > workspace_bytes) { set_error("gims_forward_pairs: workspace %zu < %zu", workspace_bytes, need); return GIMS_ERR_WORKSPACE; }
  // the stacked row segments: 2 p = image 0 of pair p, 2 p + 1 = image 1
  Segs segs = {};
  segs.nseg = 2 * n_pairs;
  int row = 0;
  for (int p = 0; p < n_pairs; ++p)
    for (int s = 0; s < 2; ++s) {
      segs.base[2 * p + s] = row;
      segs.nmax[2 * p + s] = in[p].n[s];
      segs.n_ptr[2 * p + s] = out[p].n_kept_dev + s;
      row += in[p].n[s];
    }
  const size_t rows = (size_t)row;
  // a-1 .. a-7: graphs + pruning (gmatcher.py:233-252), then a-9, a-8, a-10: desc = SAGE(feat) + kenc(normalize(kpts))
  // (gmatcher.py:265-271), image by image into the stacked buffer
  for (int p = 0; p < n_pairs; ++p) GIMS_CUDA_OK(cudaMemsetAsync(out[p].status_dev, 0, sizeof(unsigned), st));
  SideStream side = {st, nullptr, nullptr};
  bool forked = fork_images();
  if (forked) {
    GIMS_TRY(side_stream_for(st, side));
    forked = side.fork != nullptr;
  }
  if (forked) {
    GIMS_CUDA_OK(cudaEventRecord(side.fork, st));
    GIMS_CUDA_OK(cudaStreamWaitEvent(side.s, side.fork, 0));
  }
  // each image's chain has its own graph workspace and its own half of the scratch area (2.5 n x 256 floats are needed,
  // half the attention scratch is 5 (n0 + n1) x 256)
  float* scratch_img[2] = {w.scratch, w.scratch + (attn_scratch_floats(rows, 2 * n_pairs) / 2 / 64) * 64};
  for (int p = 0; p < n_pairs; ++p) {
    const gims_pair_inputs* ip = in + p;
    const gims_pair_outputs* o = out + p;
    for (int s = 0; s < 2; ++s) {
      cudaStream_t ss = s ? side.s : st;
      GIMS_TRY(gims_agc_build(ip->kpts[s], ip->desc[s], ip->desc_channel_major, ip->scores[s], ip->n[s], ip->radius,
                              ip->k_rank[s], ip->min_size, w.agc[s], w.agc_bytes, o->kept_idx[s], o->n_kept_dev + s,
                              o->csr_indptr[s], o->csr_indices[s], ip->edge_cap, o->n_edges_dev + s, o->kpts[s], o->feat[s],
                              o->scores[s], o->thr_dev + s, o->n_comp_dev + s, o->status_dev, ss));
      const size_t base = (size_t)segs.base[2 * p + s];
      GIMS_TRY(sage_fwd(m, o->feat[s], o->csr_indptr[s], o->csr_indices[s], ip->n[s], o->n_kept_dev + s,
                        w.sage_out + base * kD, scratch_img[s], mode, ss));
      GIMS_TRY(kenc_fwd(m, o->kpts[s], ip->n[s], o->n_kept_dev + s, ip->img_w[s], ip->img_h[s],
                        w.sage_out + base * kD, w.desc + base * kD, scratch_img[s], mode, ss));
    }
  }
  if (forked) {
    GIMS_CUDA_OK(cudaEventRecord(side.join, side.s));
    GIMS_CUDA_OK(cudaStreamWaitEvent(st, side.join, 0));
  }
  for (int p = 0; p < n_pairs; ++p) {
    if (!out[p].desc_in) continue;
    const size_t base = (size_t)segs.base[2 * p], cnt = (size_t)in[p].n[0] + in[p].n[1];
    GIMS_TRY(copy_rows(w.desc + base * kD, out[p].desc_in, cnt * kD, st));
  }
  // a-11, a-12: attention stack (gmatcher.py:272) — one launch per stage and layer for the whole batch.  The fp16-range
  // flag of the batch is raised in pair 0's status word and copied to the others below.
  for (int l = 0; l < m->cfg.num_layers; ++l)
    GIMS_TRY(attn_layer(m, l, w.desc, segs, w.scratch, out[0].status_dev, mode, st));
  // a-13: final_proj for every row at once
  GIMS_TRY(final_proj(m, w.desc, segs, w.mdesc, mode, st, out[0].status_dev));
  (void)rows;
  for (int p = 0; p < n_pairs; ++p) {
    const gims_pair_inputs* ip = in + p;
    const gims_pair_outputs* o = out + p;
    const size_t base = (size_t)segs.base[2 * p], cnt = (size_t)ip->n[0] + ip->n[1];
    if (o->desc_gnn) GIMS_TRY(copy_rows(w.desc + base * kD, o->desc_gnn, cnt * kD, st));
    GIMS_TRY(copy_rows(w.mdesc + base * kD, o->mdesc, cnt * kD, st));
    if (p > 0) GIMS_TRY(launch_or_status(out[0].status_dev, o->status_dev, GIMS_STATUS_FP16_RANGE, st));
    // a-13 .. a-15 per pair
    float* coup = o->couplings ? o->couplings : w.couplings;
    GIMS_TRY(score_matrix(m, w.mdesc + base * kD, ip->n[0], ip->n[1], o->n_kept_dev, coup, w.scratch, mode, st, o->status_dev));
    GIMS_TRY(gims_sinkhorn_match(coup, coup_ld(ip->n[1]), ip->n[0], ip->n[1], o->n_kept_dev, m->cfg.sinkhorn_iterations,
                                 m->cfg.match_threshold, w.sink, w.sink_bytes, o->u, o->v, o->indices[0], o->indices[1],
                                 o->matches[0], o->matches[1], o->mscores[0], o->mscores[1], o->status_dev, stream));
  }
  return GIMS_OK;
}

extern "C" int gims_forward_pair(const gims_model* m, const gims_pair_inputs* in, const gims_pair_outputs* o,
                                 void* workspace, size_t workspace_bytes, void* stream) {
  return gims_forward_pairs(m, 1, in, o, workspace, workspace_bytes, stream);
}

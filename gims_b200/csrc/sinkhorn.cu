// Fused log-domain Sinkhorn + mutual-nearest-neighbour match extraction (SURVEY.md §8 a-14, a-15).
//
// Replaces log_optimal_transport / log_sinkhorn_iterations (models/gmatcher.py:41-69) and the match
// extraction of GMatcher.forward (gmatcher.py:284-294).
//
// Persistent cooperative kernels, one CTA per SM; CTA b owns a contiguous slab of rows of the couplings
// matrix Z0 ((N+1) x (M+1), dustbin row/column included).  Three kernels share the final pass:
//
//   k_sinkhorn_reg      SCALED-KERNEL iteration, slab in REGISTERS (<= 16 rows per CTA, <= 2051 columns:
//                       up to 2048 keypoints per image).  Z0 is read from HBM once.
//   k_sinkhorn_stream   SCALED-KERNEL iteration for every larger problem: the scaled matrix E is written to a
//                       scratch buffer once and streamed (L2 at 4096 keypoints, HBM at 8192) ONCE per
//                       iteration — the row sums and the column partials of a row chunk come from the same
//                       registers.
//   k_sinkhorn_exact    log-sum-exp iteration in the log domain (any input).  Runs only when a scaled-kernel
//                       launch reports that its sums left the fp32 range (never seen on real score matrices),
//                       or when the caller's buffer cannot be read with 128-bit loads.
//
// Scaled-kernel iteration.  With rmax_r = max_j z_rj and cmax_j = max_r (z_rj - rmax_r) the matrix
//   E_rj = exp(z_rj - rmax_r - cmax_j)  lies in [0, 1] and has a 1 in every row and every column, whatever the
// offset between the scores and the dustbin score is (trained weights: scores ~ 90, bin_score 1).  Writing
// u_r = -rmax_r + log a_r, v_j = -cmax_j + log b_j the Sinkhorn updates become
//   row pass   sr_r = sum_j E_rj w_j            w_j = b_j / exp(vref)
//   col pass   cs_j = sum_r E_rj e_r            e_r = a_r / exp(Rref)
// i.e. two FMAs per matrix element and iteration instead of two exp: no transcendental in the inner loops.
// All CTAs share the references, so per-CTA column partials add up directly: `red.global.add.v4.f32` into
// rotating column-sum buffers, ONE grid-wide arrive/wait on a counter per iteration, then every CTA computes
// v_j and w_j for all columns itself.  Every sum is checked to be a normal fp32 number; if one is not (potentials
// more than ~e^80 apart), the launch raises a flag and the exact kernel redoes the problem.
//
// The last pass evaluates the reference's expression ((Z0 + u) + v) - norm element-wise and takes
// row / column max + first argmax; a tiny follow-up kernel applies the mutual / threshold rule.
#include <math_constants.h>

#include "common.cuh"

namespace gims {

namespace {

constexpr int kThreads = 512;
constexpr int kWarps = kThreads / 32;
constexpr int kMaxGrid = 256;
constexpr int kRMax = 16;            // rows per CTA handled by the register-resident kernel
constexpr int kRowChunks = 17;       // float4 chunks per lane of the exact kernel's register row pass (<= 2176 columns)
constexpr float kLog2e = 1.4426950408889634f;
// Bound of every poll in clock64 cycles (~2 s at 1.9 GHz): far beyond any legitimate wait, also under ncu replay, MPS
// time-slicing or a debugger; on expiry the launch poisons its outputs and raises GIMS_STATUS_SINKHORN_TIMEOUT.
constexpr long long kPollTimeoutClk = 4000000000LL;
constexpr int kWays = 2;             // copies of the column-sum buffer (CTA b adds into copy b % kWays): the red.adds of
                                     // 148 CTAs on one 128-byte line serialize in L2, four copies cut that chain by four

typedef unsigned long long u64;

// words of the `err` block (zeroed before every launch chain)
constexpr int kErrTimeout = 0;       // a poll expired
constexpr int kErrPath = 1;          // GIMS_STATUS_SINKHORN_FAST / _EXACT: which kernel produced the results
constexpr int kErrRedo = 2;          // the scaled-kernel launch left the fp32 range: the exact kernel must run
constexpr int kErrCounter = 32;      // grid-wide arrival counter of the scaled-kernel kernels

struct SinkArgs {
  const float* Z; int ld;          // couplings, row pitch in floats
  int n0_max, n1_max;
  const int* n_dev;
  int iters;
  float* u; float* v;              // outputs: final potentials
  float2* part;                    // [grid][ldp]  (m, s): per-CTA column partials; last pass: (best value, row index bits)
  float* vg;                       // [ldp + 4]    v_j exchange buffer (exact kernel)
  unsigned* pflag;                 // [grid]       iteration number of the partials CTA g has published
  unsigned* vflag;                 // [grid]       iteration number of the v_j CTA g has published
  float* colsum;                   // [3][kWays][cs_ld] scaled-kernel: column sums accumulated with red.add, 3 rotating buffers
  unsigned* cmkey;                 // [cs_ld]      scaled-kernel: ~bits of the column maxima of z - rowmax (atomicMax, 0 = unset)
  float* E;                        // [(n0_max+1)][ld] streaming kernel: the scaled matrix (scratch)
  int ldp;
  unsigned* err;                   // kErr* words
  int* idx0; int* idx1; float* max0; float* max1;
  int rpc_max;                     // ceil((n0_max+1)/grid): capacity of the per-CTA u buffer
  int slab_rows;                   // rows of the smem slab (0 = stream from global)
  int slab_ld;                     // padded row length of the slab (multiple of 4)
  int only_if_redo;                // exact kernel: return at once unless err[kErrRedo] is set
  int ring, rb;                    // streaming kernel: stages of the ring, rows per stage
};

__device__ __forceinline__ unsigned ld_acquire_u32(const unsigned* p) {
  unsigned v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
// Publish: every thread of the CTA has written its data with plain stores; one fence + one flag store makes them
// visible (the block barrier orders the other threads' stores before thread 0's fence — cumulativity).
__device__ __forceinline__ void publish_flag(unsigned* flag, unsigned epoch) {
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    asm volatile("st.relaxed.gpu.global.u32 [%0], %1;" ::"l"(flag), "r"(epoch) : "memory");
  }
}
// Warp 0 waits until flags[0..n) have all reached `epoch`, then the whole CTA proceeds (data is then read with
// ld.global.cg, which cannot hit a stale L1 line).  Bounded like every other wait in this file.
__device__ __forceinline__ void wait_flags(const unsigned* flags, int n, unsigned epoch, unsigned* err) {
  if (threadIdx.x < 32) {
    const int lane = threadIdx.x;
    long long t0 = clock64();
    unsigned spins = 0;
    while (true) {
      bool ok = true;
      for (int g = lane; g < n; g += 32) ok = ok && (ld_acquire_u32(&flags[g]) >= epoch);
      if (__all_sync(0xffffffffu, ok)) break;
      if ((++spins & 63u) == 0) {
        bool bail = *(volatile unsigned*)err != 0u;
        if (clock64() - t0 > kPollTimeoutClk) { atomicExch(err, 1u); bail = true; }
        if (__any_sync(0xffffffffu, bail)) break;
      }
    }
  }
  __syncthreads();
}

// Grid-wide arrive + wait on one monotonically increasing counter (every CTA is co-resident: cooperative launch).
// Measured on B200 (tools/micro/hop_latency.cu): 2.5 k cycles per hop, about half of a per-CTA flag scheme.
__device__ __forceinline__ void grid_hop(unsigned* counter, unsigned target, unsigned* err) {
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    atomicAdd(counter, 1u);
    long long t0 = clock64();
    unsigned spins = 0;
    while (ld_acquire_u32(counter) < target) {
      if ((++spins & 255u) == 0) {
        if (*(volatile unsigned*)err) break;
        if (clock64() - t0 > kPollTimeoutClk) { atomicExch(err, 1u); break; }
      }
    }
  }
  __syncthreads();
}

__device__ __forceinline__ float warp_max(float x) {
#pragma unroll
  for (int o = 16; o; o >>= 1) x = fmaxf(x, __shfl_xor_sync(0xffffffffu, x, o));
  return x;
}
__device__ __forceinline__ float warp_sum(float x) {
#pragma unroll
  for (int o = 16; o; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
  return x;
}
// 2^x for x <= 0: one MUFU (results below 2^-126 flush to zero, which is what a log-sum-exp term wants)
__device__ __forceinline__ float ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// (m, s) <- combine of two (max, sum-of-exp) partials
__device__ __forceinline__ void lse_merge(float& m, float& s, float pm, float ps) {
  float mn = fmaxf(m, pm);
  s = s * ex2((m - mn) * kLog2e) + ps * ex2((pm - mn) * kLog2e);
  m = mn;
}
// a scaled-kernel sum is usable iff it is a normal, comfortably representable positive number
__device__ __forceinline__ bool sum_ok(float s) { return s > 1e-35f && s < 1e35f; }
// column maxima of (z - rowmax) <= 0 travel as ~bits: for non-positive floats a larger value has a smaller bit pattern,
// so max(value) = max(~bits), and the zero-initialised word means "nothing yet" (decodes to NaN, never read for a
// column that has a row)
__device__ __forceinline__ unsigned cm_key(float x) { return ~__float_as_uint(fminf(x, 0.f)); }
__device__ __forceinline__ float cm_val(unsigned k) { return __uint_as_float(~k); }

// Optional timeline (profiling): CTA 0 / thread 0 stores clock64() at 6 points of each of the first 16 iterations.
__device__ long long* g_sink_trace = nullptr;
#define SINK_TRACE(slot)                                                        \
  do {                                                                          \
    if (trace && it < 16) trace[it * 8 + (slot)] = clock64();                   \
    if (gtrace && it == 5) {                                                    \
      unsigned long long gt_;                                                   \
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt_));                   \
      gtrace[128 + blockIdx.x * 8 + (slot)] = (long long)gt_;                   \
    }                                                                           \
  } while (0)

// Everything the three kernels derive from the arguments in the same way.
struct SinkGeom {
  int n0, n1, R, C, G, b, rpc, r_begin, r_end, nrows, Ga, cpc, c_begin, c_end;
  float norm, log_mu_last, log_nu_last;
};
__device__ __forceinline__ SinkGeom sink_geom(const SinkArgs& a) {
  SinkGeom g;
  g.n0 = a.n_dev ? min(a.n_dev[0], a.n0_max) : a.n0_max;
  g.n1 = a.n_dev ? min(a.n_dev[1], a.n1_max) : a.n1_max;
  g.R = g.n0 + 1; g.C = g.n1 + 1;
  g.G = gridDim.x; g.b = blockIdx.x;
  // marginals exactly as gmatcher.py:62-64 computes them in fp32
  const float ms = (float)g.n0, ns = (float)g.n1;
  g.norm = -logf(ms + ns);
  g.log_mu_last = logf(ns) + g.norm;
  g.log_nu_last = logf(ms) + g.norm;
  g.rpc = (g.R + g.G - 1) / g.G;                   // rows per CTA
  g.r_begin = min(g.b * g.rpc, g.R);
  g.r_end = min(g.r_begin + g.rpc, g.R);
  g.nrows = g.r_end - g.r_begin;
  g.Ga = (g.R + g.rpc - 1) / g.rpc;                // CTAs that own at least one row
  g.cpc = (g.C + g.G - 1) / g.G;                   // columns per CTA in the combine steps
  g.c_begin = min(g.b * g.cpc, g.C);
  g.c_end = min(g.c_begin + g.cpc, g.C);
  return g;
}

// ---- final pass: Z = ((Z0 + u) + v) - norm, row / column max + first argmax (gmatcher.py:284-285) -------------
// u_s: this CTA's final u; v_s: the final v of every column (true potentials); Z0 is re-read from global memory.
__device__ __forceinline__ void sink_final_pass(const SinkArgs& a, const SinkGeom& g, const float* u_s, const float* v_s,
                                                float (*red_m)[17], float (*red_s)[17], unsigned epoch) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const float* zbase = a.Z + (size_t)g.r_begin * a.ld;
  const int n0 = g.n0, n1 = g.n1;
  const float norm = g.norm;
  for (int r = warp; r < g.nrows; r += kWarps) {
    int gr = g.r_begin + r;
    float ur = (a.iters > 0) ? u_s[r] : 0.f;
    if (lane == 0) a.u[gr] = ur;
    if (gr >= n0) continue;
    const float* z = zbase + (size_t)r * a.ld;
    float best = -CUDART_INF_F;
    int bj = 0x7fffffff;
#pragma unroll 4
    for (int j = lane; j < n1; j += 32) {
      float t = ((z[j] + ur) + v_s[j]) - norm;
      if (t > best) { best = t; bj = j; }
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) {
      float ob = __shfl_xor_sync(0xffffffffu, best, o);
      int oj = __shfl_xor_sync(0xffffffffu, bj, o);
      if (ob > best || (ob == best && oj < bj)) { best = ob; bj = oj; }
    }
    if (lane == 0) { a.idx0[gr] = bj; a.max0[gr] = best; }
  }
  if (g.b < g.Ga) {
    int live = min(g.r_end, n0) - g.r_begin;       // rows of mine that are real keypoints (may be <= 0)
    for (int j = tid; j < n1; j += kThreads) {
      float best = -CUDART_INF_F;
      int bi = 0x7ffffffe;
      float vj = v_s[j];
      for (int r = 0; r < live; ++r) {
        float ur = (a.iters > 0) ? u_s[r] : 0.f;
        float t = ((zbase[(size_t)r * a.ld + j] + ur) + vj) - norm;
        if (t > best) { best = t; bi = g.r_begin + r; }
      }
      a.part[(size_t)g.b * a.ldp + j] = make_float2(best, __int_as_float(bi));
    }
  }
  publish_flag(&a.pflag[g.b], epoch);
  wait_flags(a.pflag, g.Ga, epoch, a.err);
  for (int jc = g.c_begin; jc < g.c_end; jc += 16) {
    const int jj = tid & 15, gs = tid >> 4, j = jc + jj;
    float best = -CUDART_INF_F;
    int bi = 0x7fffffff;
    if (j < g.c_end && j < n1) {
      const int cnt = (g.Ga - gs + 31) >> 5;
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        if (k < cnt) {
          const float2 w = __ldcg(&a.part[(size_t)(gs + 32 * k) * a.ldp + j]);
          const float pv = w.x;
          const int pi = __float_as_int(w.y);
          if (pv > best || (pv == best && pi < bi)) { best = pv; bi = pi; }
        }
      }
    }
    red_m[gs][jj] = best; red_s[gs][jj] = __int_as_float(bi);
    __syncthreads();
    const int jw = jc + warp;
    if (jw < g.c_end && jw < n1) {
      float bb = red_m[lane][warp];
      int ii = __float_as_int(red_s[lane][warp]);
#pragma unroll
      for (int o = 16; o; o >>= 1) {
        float ob = __shfl_xor_sync(0xffffffffu, bb, o);
        int oi = __shfl_xor_sync(0xffffffffu, ii, o);
        if (ob > bb || (ob == bb && oi < ii)) { bb = ob; ii = oi; }
      }
      if (lane == 0) { a.idx1[jw] = ii; a.max1[jw] = bb; }
    }
    __syncthreads();
  }
}

// ---- the per-column update shared by the scaled-kernel kernels --------------------------------------------------
// From the gathered column sums: v~_j = log_nu_j - (Rref + log cs_j) (potential of the column-scaled problem),
// w_j = exp(v~_j - v0).  During the iterations v_s holds v~; the LAST iteration stores the true potential
// v_j = v~_j - cmax_j (what the final pass and the caller need).  finish() returns false if a sum left the safe range.
struct ColUpdate {
  const SinkArgs& a; const SinkGeom& g;
  const float* cs; size_t cs_ld; float Rref, v0; bool last;
  float* v_s; float* w_s;
  __device__ __forceinline__ float4 load(int g4) const {
    float4 c4 = __ldcg(reinterpret_cast<const float4*>(cs) + g4);
#pragma unroll
    for (int w = 1; w < kWays; ++w) {
      const float4 cw = __ldcg(reinterpret_cast<const float4*>(cs + (size_t)w * cs_ld) + g4);
      c4.x += cw.x; c4.y += cw.y; c4.z += cw.z; c4.w += cw.w;
    }
    return c4;
  }
  __device__ __forceinline__ bool finish(int g4, const float4 c4, float4& wn4) const {
    const float cc[4] = {c4.x, c4.y, c4.z, c4.w};
    float wn[4];
    bool ok = true;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int j = 4 * g4 + q;
      wn[q] = 0.f;
      if (j < g.C) {
        ok = ok && sum_ok(cc[q]);
        const float lnu = (j == g.n1) ? g.log_nu_last : g.norm;
        const float vj = lnu - (Rref + logf(cc[q]));
        wn[q] = ex2((vj - v0) * kLog2e);
        w_s[j] = wn[q];
        if (last) {
          const float vt = vj - cm_val(__ldcg(&a.cmkey[j]));
          v_s[j] = vt;
          if (j >= g.c_begin && j < g.c_end) a.v[j] = vt;
        } else {
          v_s[j] = vj;
        }
      }
    }
    wn4 = make_float4(wn[0], wn[1], wn[2], wn[3]);
    return ok;
  }
};

// =====================================================================================================================
// Scaled-kernel iteration, slab on chip: thread t owns the float4 column group t of every slab row together with the
// group's weights.  The first kRMax (16) rows live in REGISTERS, up to kRSmem (16) more in shared memory, so neither pass
// touches global memory: the row pass is 4 FMAs per row + a block reduction of the row sums, the column pass 4 FMAs per
// row whose result is already this CTA's complete partial for those columns.  The (<= 3) columns past the last full
// group, among them the dustbin column, sit in a small shared array.
//
// Why up to 32 rows per CTA: the iteration is bound by the exchange (148 CTAs x 513 red.v4 into L2, then every CTA reading
// every column sum back), whose cost grows with the number of CTAs, not by the arithmetic.  With twice the rows on HALF
// the SMs an iteration takes about as long (profiles/), and the other half of the GPU runs other pairs' kernels
// meanwhile — this kernel allocates a whole SM's register file, nothing shares an SM with it.
// =====================================================================================================================
constexpr int kRSmem = 16;
__global__ void __launch_bounds__(kThreads, 1) k_sinkhorn_reg(SinkArgs a) {
  extern __shared__ __align__(16) float smem[];
  __shared__ float red_m[32][17], red_s[32][17];
  __shared__ float left[kRMax + kRSmem][4];
  const SinkGeom g = sink_geom(a);
  const int n0 = g.n0, C = g.C, G = g.G, b = g.b, nrows = g.nrows, r_begin = g.r_begin, Ga = g.Ga;
  const int c_begin = g.c_begin, c_end = g.c_end;
  const float norm = g.norm, log_mu_last = g.log_mu_last;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int nreg = min(nrows, kRMax), nsm = nrows - nreg;      // rows in registers / in shared memory

  const int vlen = (a.n1_max + 1 + 3) & ~3;
  const int rlen = (a.rpc_max + 3) & ~3;
  float* v_s = smem;                                // [vlen]  v~_j (true v_j after the last iteration)
  float* w_s = v_s + vlen;                          // [vlen]  exp(v~_j - vref), pads 0
  float* u_s = w_s + vlen;                          // [rlen]  u_r
  float* rmax_s = u_s + rlen;                       // [rlen]  row maxima of my slab
  float* e_s = rmax_s + rlen;                       // [rlen]  column-pass weight of row r
  float* slab = e_s + rlen;                         // [min(rpc, 16)][slab_ld]: staging of the register rows, then rows 16..
  const int C4 = (C + 3) & ~3;                      // slab rows are padded up to a multiple of 4
  const int n4 = C4 >> 2;
  const int Gf = C >> 2;                            // full groups: one per thread (host guarantees Gf <= kThreads)
  const size_t cs_ld = ((size_t)a.ldp + 3) & ~(size_t)3;
  unsigned* counter = a.err + kErrCounter;
  unsigned target = 0;
  const bool own = tid < Gf;
  float4 ereg[kRMax];

  // ---- load the slab (raw scores), row maxima, column maxima of z - rowmax over ALL rows (one grid-wide exchange) ----
  // two rounds through the same staging area: rows [0, nreg) end up in registers, rows [nreg, nrows) stay
  for (int round = 0; round < 2; ++round) {
    const int r0 = round ? nreg : 0, cnt = round ? nsm : nreg;
    if (round) __syncthreads();                     // round 0's readers are done with the staging area
    for (int r = warp; r < cnt; r += kWarps) {
      const float* src = a.Z + (size_t)(r_begin + r0 + r) * a.ld;
      float* dst = slab + (size_t)r * a.slab_ld;
      float mx = -CUDART_INF_F;
      for (int j = lane; j < C4; j += 32) {
        float z = (j < C) ? src[j] : -CUDART_INF_F;
        dst[j] = z;
        mx = fmaxf(mx, z);
      }
      mx = warp_max(mx);
      if (lane == 0) rmax_s[r0 + r] = mx;
    }
    __syncthreads();
    if (b < Ga && cnt > 0) {
      for (int j = tid; j < C; j += kThreads) {
        float m = -CUDART_INF_F;
        for (int r = 0; r < cnt; ++r) m = fmaxf(m, slab[(size_t)r * a.slab_ld + j] - rmax_s[r0 + r]);
        atomicMax(&a.cmkey[j], cm_key(m));
      }
    }
    if (tid < 4 * cnt) {
      const int r = tid >> 2, q = tid & 3, j = 4 * Gf + q;
      left[r0 + r][q] = (j < C) ? slab[(size_t)r * a.slab_ld + j] : -CUDART_INF_F;
    }
    if (round == 0) {
#pragma unroll
      for (int r = 0; r < kRMax; ++r)
        ereg[r] = (own && r < nreg) ? *reinterpret_cast<const float4*>(slab + (size_t)r * a.slab_ld + 4 * tid)
                                    : make_float4(0.f, 0.f, 0.f, 0.f);
    }
  }
  target += (unsigned)G;
  grid_hop(counter, target, a.err);
  // v = 0 at the start, i.e. v~_j = cmax_j (<= 0) and, with vref = 0, w_j = exp(cmax_j)
  for (int j = tid; j < vlen; j += kThreads) {
    const float cm = (j < C) ? cm_val(__ldcg(&a.cmkey[j])) : 0.f;
    v_s[j] = cm;
    w_s[j] = (j < C) ? ex2(cm * kLog2e) : 0.f;
  }
  __syncthreads();
  // slab <- E = exp(z - rowmax - cmax), pads 0: in the registers, in shared memory, in the left-over array
  {
    const float4 cm4 = own ? *reinterpret_cast<const float4*>(v_s + 4 * tid) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int r = 0; r < kRMax; ++r) {
      if (own && r < nreg) {
        const float rm = rmax_s[r];
        ereg[r].x = ex2(((ereg[r].x - rm) - cm4.x) * kLog2e); ereg[r].y = ex2(((ereg[r].y - rm) - cm4.y) * kLog2e);
        ereg[r].z = ex2(((ereg[r].z - rm) - cm4.z) * kLog2e); ereg[r].w = ex2(((ereg[r].w - rm) - cm4.w) * kLog2e);
      }
    }
  }
  for (int r = warp; r < nsm; r += kWarps) {
    float* row = slab + (size_t)r * a.slab_ld;
    const float rm = rmax_s[kRMax + r];
    for (int j = lane; j < C4; j += 32) row[j] = (j < C) ? ex2(((row[j] - rm) - v_s[j]) * kLog2e) : 0.f;
  }
  if (tid < 4 * (kRMax + kRSmem)) {
    const int r = tid >> 2, q = tid & 3, j = 4 * Gf + q;
    left[r][q] = (r < nrows && j < C) ? ex2(((left[r][q] - rmax_s[r]) - v_s[j]) * kLog2e) : 0.f;
  }
  if (b == 0 && tid == 0) a.err[kErrPath] = GIMS_STATUS_SINKHORN_FAST;
  __syncthreads();

  // the trace pointer is read once: a load of the global per stamp would sit on every iteration's critical path
  long long* const gtrace = (tid == 0) ? g_sink_trace : nullptr;
  long long* trace = (b == 0) ? gtrace : nullptr;

  const float4* slab4 = reinterpret_cast<const float4*>(slab) + tid;     // my column group of shared-memory row r: [r * ld4]
  const int ld4 = a.slab_ld >> 2;
  float4 wreg = own ? *reinterpret_cast<const float4*>(w_s + 4 * tid) : make_float4(0.f, 0.f, 0.f, 0.f);
  float vref = 0.f;                               // reference the current w_s was scaled with
  float v0_prev = v_s[0];                         // v~_0 after the previous iteration
  bool bad = false;
  for (int it = 0; it < a.iters; ++it) {
    SINK_TRACE(0);
    float* cs = a.colsum + (size_t)(it % 3) * kWays * cs_ld;   // [kWays][cs_ld]
    float* my = cs + (size_t)(b % kWays) * cs_ld;
    const float Rref = norm - vref;
    // 16 sums over 32 lanes with 16 shuffles (a butterfly that halves the number of live values per step) instead
    // of 16 x 5: shuffles issue at one warp instruction per clock per SM and were the longest part of this pass
    static_assert(kRMax == 16 && kRSmem == 16, "the butterfly below is written for 16 row sums");
#pragma unroll
    for (int half = 0; half < 2; ++half) {
      if (half == 1 && nsm == 0) break;
      float part[kRMax];
      if (half == 0) {
#pragma unroll
        for (int r = 0; r < kRMax; ++r)
          part[r] = fmaf(ereg[r].x, wreg.x, ereg[r].y * wreg.y) + fmaf(ereg[r].z, wreg.z, ereg[r].w * wreg.w);
      } else {
#pragma unroll
        for (int r = 0; r < kRSmem; ++r) {
          const float4 e = (own && r < nsm) ? slab4[(size_t)r * ld4] : make_float4(0.f, 0.f, 0.f, 0.f);
          part[r] = fmaf(e.x, wreg.x, e.y * wreg.y) + fmaf(e.z, wreg.z, e.w * wreg.w);
        }
      }
#pragma unroll
      for (int h = 8, bit = 16; h >= 1; h >>= 1, bit >>= 1) {
        const bool up = (lane & bit) != 0;
#pragma unroll
        for (int i = 0; i < h; ++i) {
          const float send = up ? part[i] : part[i + h];
          const float keep = up ? part[i + h] : part[i];
          part[i] = keep + __shfl_xor_sync(0xffffffffu, send, bit);
        }
      }
      part[0] += __shfl_xor_sync(0xffffffffu, part[0], 1);
      if ((lane & 1) == 0) red_m[half * kWarps + warp][lane >> 1] = part[0];      // lane 2r holds the warp's sum of row r
    }
    __syncthreads();
    SINK_TRACE(7);
    if (tid < nrows) {                              // thread r finishes row r
      float sr = 0.f;
      const int hb = (tid >> 4) * kWarps, rr = tid & 15;
#pragma unroll
      for (int w = 0; w < kWarps; ++w) sr += red_m[hb + w][rr];
      for (int j = 4 * Gf; j < C; ++j) sr = fmaf(left[tid][j - 4 * Gf], w_s[j], sr);
      bad = bad || !sum_ok(sr);
      const float lmu = (r_begin + tid == n0) ? log_mu_last : norm;
      const float lse_rel = vref + logf(sr);               // LSE_j(z + v) - rowmax
      e_s[tid] = ex2(((lmu - lse_rel) - Rref) * kLog2e);    // exp(u_r + rowmax_r - Rref)
      u_s[tid] = lmu - (rmax_s[tid] + lse_rel);
    }
    __syncthreads();
    SINK_TRACE(1);
    if (b < Ga) {
      if (own) {
        float4 sm = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int r = 0; r < kRMax; ++r) {
          const float er = (r < nreg) ? e_s[r] : 0.f;
          sm.x = fmaf(ereg[r].x, er, sm.x); sm.y = fmaf(ereg[r].y, er, sm.y);
          sm.z = fmaf(ereg[r].z, er, sm.z); sm.w = fmaf(ereg[r].w, er, sm.w);
        }
        if (nsm > 0) {
#pragma unroll
          for (int r = 0; r < kRSmem; ++r) {
            if (r < nsm) {
              const float er = e_s[kRMax + r];
              const float4 e = slab4[(size_t)r * ld4];
              sm.x = fmaf(e.x, er, sm.x); sm.y = fmaf(e.y, er, sm.y);
              sm.z = fmaf(e.z, er, sm.z); sm.w = fmaf(e.w, er, sm.w);
            }
          }
        }
        // (packed FFMA2 for these passes and a 16-lanes-per-row finish were tried: both slower on B200)
        SINK_TRACE(6);
        asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(my + 4 * tid), "f"(sm.x), "f"(sm.y),
                     "f"(sm.z), "f"(sm.w)
                     : "memory");
      }
      const int jl = 4 * Gf + warp;                 // the (at most 3) left-over columns: lane = row
      if (jl < C) {
        const float xx = (lane < nrows) ? left[lane][warp] * e_s[lane] : 0.f;
        const float ss = warp_sum(xx);
        if (lane == 0) atomicAdd(my + jl, ss);
      }
    }
    SINK_TRACE(2);
    target += (unsigned)G;
    grid_hop(counter, target, a.err);
    SINK_TRACE(3);
    {                                               // recycle the buffer that was read one iteration ago
      float* old = a.colsum + (size_t)((it + 2) % 3) * kWays * cs_ld;
      for (int w = 0; w < kWays; ++w)
        for (int j = c_begin + tid; j < c_end; j += kThreads) old[(size_t)w * cs_ld + j] = 0.f;
    }
    // Reference of the new weights: v~_0 of the PREVIOUS iteration — every thread already has it, and any reference
    // inside the (bounded) range of v~ works.  (Deriving it from this iteration's colsum[0] made every warp of the
    // grid load the same address right after the hop: 2400 serialized requests on one L2 sector per iteration.)
    const float v0 = v0_prev;
    ColUpdate cu{a, g, cs, cs_ld, Rref, v0, it == a.iters - 1, v_s, w_s};
    // n4 <= kThreads + 1 here: a thread has its own group and at most one more (the left-over columns); both loads
    // are issued before either is used — one L2 round trip, not two, on the thread every other thread waits for
    const int g4b = tid + kThreads;
    float4 ca = make_float4(1.f, 1.f, 1.f, 1.f), cb = ca, wa, wb;
    if (tid < n4) ca = cu.load(tid);
    if (g4b < n4) cb = cu.load(g4b);
    if (tid < n4) { bad = !cu.finish(tid, ca, wa) || bad; wreg = wa; }
    if (g4b < n4) bad = !cu.finish(g4b, cb, wb) || bad;
    SINK_TRACE(4);
    vref = v0;
    __syncthreads();
    v0_prev = v_s[0];
    SINK_TRACE(5);
  }
  if (bad) atomicOr(&a.err[kErrRedo], 1u);
  if (a.iters == 0) {                               // degenerate call: potentials stay 0
    __syncthreads();
    for (int j = tid; j < C; j += kThreads) v_s[j] = 0.f;
    for (int j = c_begin + tid; j < c_end; j += kThreads) a.v[j] = 0.f;
    __syncthreads();
  }
  sink_final_pass(a, g, u_s, v_s, red_m, red_s, (unsigned)(a.iters + 1));
}

// =====================================================================================================================
// Scaled-kernel iteration, streamed: for problems whose slab does not fit the chip.  The prologue writes
// E = exp(z - rowmax - cmax) to a scratch matrix (3 reads of Z0 + 1 write, about 2.5 iterations' worth); each
// iteration then reads E ONCE.  Rows arrive through a ring of shared-memory stages filled by bulk asynchronous copies
// (cp.async.bulk, one row per stage, completion on an mbarrier): thread 0 refills a stage right after the block
// barrier that follows its last reader, so `ring` rows (100+ KB per SM) are always in flight — with one row of register
// prefetch the kernel reached only half of the HBM copy bandwidth (32 KB per SM per memory latency).  The ring runs
// ahead across iterations (E does not change), i.e. the next iteration's first rows load during the grid-wide exchange.
// Thread t owns the float4 column groups t, t + 512, ... (KG of them) of every row: it copies them from the stage into
// registers, the row sum is reduced across the CTA (one __syncthreads per row, partials double-buffered by row parity,
// every warp finishes the sum itself), and the same registers then update the thread's column partials.  After the last
// row the partials go out with red.global.add, then hop and gather exactly like the on-chip kernel.
// HBM-bound at 8192 keypoints (268 MB per iteration), L2-bound at 4096 (67 MB).
// =====================================================================================================================
__device__ __forceinline__ void sink_bulk_row(float* dst_smem, const float* src, unsigned bytes, unsigned long long* bar) {
  const unsigned d = (unsigned)__cvta_generic_to_shared(dst_smem), m = (unsigned)__cvta_generic_to_shared(bar);
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(m), "r"(bytes) : "memory");
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(d), "l"(src),
               "r"(bytes), "r"(m)
               : "memory");
}
__device__ __forceinline__ void sink_bar_wait(unsigned long long* bar, unsigned parity, unsigned* err) {
  const unsigned m = (unsigned)__cvta_generic_to_shared(bar);
  unsigned ok = 0, spins = 0;
  while (true) {
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                 : "=r"(ok) : "r"(m), "r"(parity) : "memory");
    if (ok) break;
    if ((++spins & 1023u) == 0 && *(volatile unsigned*)err) break;       // another CTA timed out: give up as well
    if (spins > 4000000u) { atomicExch(err, 1u); break; }
  }
}
constexpr int kMaxRing = 8;
// KG float4 groups per thread and row; RC rows per step (their latency chains — two warp reductions, a barrier, logf —
// overlap); HOLD: the rows of a step stay in registers between the row pass and the column pass (KG * RC float4), otherwise
// the column pass reads them from the stage again and the stages are released one barrier later.
template <int KG, int RC, bool HOLD>
__global__ void __launch_bounds__(kThreads, 1) k_sinkhorn_stream(SinkArgs a) {
  extern __shared__ __align__(16) float smem[];
  __shared__ float red_m[32][17], red_s[32][17];
  __shared__ float rsum_s[2][kWarps][RC];
  __shared__ __align__(8) unsigned long long full_bar[kMaxRing];
  const SinkGeom g = sink_geom(a);
  const int n0 = g.n0, C = g.C, G = g.G, b = g.b, nrows = g.nrows, r_begin = g.r_begin, Ga = g.Ga;
  const int c_begin = g.c_begin, c_end = g.c_end;
  const float norm = g.norm, log_mu_last = g.log_mu_last;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

  const int vlen = (a.n1_max + 1 + 3) & ~3;
  const int rlen = (a.rpc_max + 3) & ~3;
  float* v_s = smem;                                // [vlen]
  float* w_s = v_s + vlen;                          // [vlen]
  float* u_s = w_s + vlen;                          // [rlen]
  float* rmax_s = u_s + rlen;                       // [rlen]
  float* ring_s = rmax_s + rlen;                    // [a.ring][slab_ld]: the stages (16-byte aligned: vlen, rlen % 4 == 0)
  const int C4 = (C + 3) & ~3;
  const int n4 = C4 >> 2;                           // float4 groups per row (host guarantees n4 <= KG * kThreads)
  const size_t cs_ld = ((size_t)a.ldp + 3) & ~(size_t)3;
  unsigned* counter = a.err + kErrCounter;
  unsigned target = 0;
  const float* zrows = a.Z + (size_t)r_begin * a.ld;
  float* erows = a.E + (size_t)r_begin * a.ld;
  const float4 ninf4 = make_float4(-CUDART_INF_F, -CUDART_INF_F, -CUDART_INF_F, -CUDART_INF_F);

  // z of group g4 of row r with the pad columns (j >= C) masked to -inf
  auto load_z = [&](int r, int g4) {
    float4 z = __ldcg(reinterpret_cast<const float4*>(zrows + (size_t)r * a.ld) + g4);
    const int j = 4 * g4;
    if (j + 1 >= C) z.y = -CUDART_INF_F;
    if (j + 2 >= C) z.z = -CUDART_INF_F;
    if (j + 3 >= C) z.w = -CUDART_INF_F;
    return z;
  };
  // ---- prologue 1: row maxima (warp per row) ----------------------------------------------------------------------
  for (int r = warp; r < nrows; r += kWarps) {
    float mx = -CUDART_INF_F;
    for (int g4 = lane; g4 < n4; g4 += 32) {
      const float4 z = load_z(r, g4);
      mx = fmaxf(mx, fmaxf(fmaxf(z.x, z.y), fmaxf(z.z, z.w)));
    }
    mx = warp_max(mx);
    if (lane == 0) rmax_s[r] = mx;
  }
  for (int j = tid; j < vlen; j += kThreads) { v_s[j] = 0.f; w_s[j] = 0.f; }
  __syncthreads();
  // ---- prologue 2: column maxima of z - rowmax over my rows -> global max ---------------------------------------------
  if (b < Ga) {
#pragma unroll
    for (int k = 0; k < KG; ++k) {
      const int g4 = tid + k * kThreads;
      if (g4 >= n4) continue;
      float4 m = ninf4;
      for (int r = 0; r < nrows; ++r) {
        const float4 z = load_z(r, g4);
        const float rm = rmax_s[r];
        m.x = fmaxf(m.x, z.x - rm); m.y = fmaxf(m.y, z.y - rm); m.z = fmaxf(m.z, z.z - rm); m.w = fmaxf(m.w, z.w - rm);
      }
      const int j = 4 * g4;
      atomicMax(&a.cmkey[j], cm_key(m.x));
      if (j + 1 < C) atomicMax(&a.cmkey[j + 1], cm_key(m.y));
      if (j + 2 < C) atomicMax(&a.cmkey[j + 2], cm_key(m.z));
      if (j + 3 < C) atomicMax(&a.cmkey[j + 3], cm_key(m.w));
    }
  }
  target += (unsigned)G;
  grid_hop(counter, target, a.err);
  // ---- prologue 3: E = exp(z - rowmax - cmax) -> scratch; start weights w_j = exp(cmax_j) (v = 0) ----------------------
#pragma unroll
  for (int k = 0; k < KG; ++k) {
    const int g4 = tid + k * kThreads;
    if (g4 >= n4) continue;
    const int j = 4 * g4;
    float4 cm;
    cm.x = cm_val(__ldcg(&a.cmkey[j]));
    cm.y = (j + 1 < C) ? cm_val(__ldcg(&a.cmkey[j + 1])) : 0.f;
    cm.z = (j + 2 < C) ? cm_val(__ldcg(&a.cmkey[j + 2])) : 0.f;
    cm.w = (j + 3 < C) ? cm_val(__ldcg(&a.cmkey[j + 3])) : 0.f;
    for (int r = 0; r < nrows; ++r) {
      const float4 z = load_z(r, g4);               // pads are -inf -> E = 0
      const float rm = rmax_s[r];
      float4 e;
      e.x = ex2(((z.x - rm) - cm.x) * kLog2e); e.y = ex2(((z.y - rm) - cm.y) * kLog2e);
      e.z = ex2(((z.z - rm) - cm.z) * kLog2e); e.w = ex2(((z.w - rm) - cm.w) * kLog2e);
      *reinterpret_cast<float4*>(erows + (size_t)r * a.ld + j) = e;   // read back by this same thread only
    }
    const float cmv[4] = {cm.x, cm.y, cm.z, cm.w};
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      if (j + q < C) { v_s[j + q] = cmv[q]; w_s[j + q] = ex2(cmv[q] * kLog2e); }
    }
  }
  if (b == 0 && tid == 0) a.err[kErrPath] = GIMS_STATUS_SINKHORN_FAST;
  // E was written with ordinary stores and is read back by the bulk-copy engine (async proxy)
  __threadfence();
  asm volatile("fence.proxy.async;" ::: "memory");
  if (tid == 0) {
    for (int s = 0; s < kMaxRing; ++s) {
      const unsigned m = (unsigned)__cvta_generic_to_shared(&full_bar[s]);
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(m) : "memory");
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();

  long long* const gtrace = (tid == 0) ? g_sink_trace : nullptr;
  long long* trace = (b == 0) ? gtrace : nullptr;
  // ---- the ring: a stage holds a BLOCK of a.rb consecutive rows (contiguous in E: its pitch a.ld equals the stage's row
  // pitch a.slab_ld, the host checks it), fetched by ONE bulk copy.  Measured: an SM's bulk copies complete one after the
  // other, each taking ~1.0 k clk + bytes / 50 — row-sized copies (12 .. 33 KB) gave 9 .. 20 B/clk per SM whatever the
  // number of stages in flight; ~64 KB blocks give ~28 B/clk, above an SM's share of the HBM bandwidth.
  // Global block number gb = it * nblocks + block lives in stage gb % ring.
  const int ring = a.ring, RB = a.rb;
  const int nblocks = (nrows + RB - 1) / RB;
  const int total_blocks = a.iters * nblocks;           // (host: < 2^31)
  const size_t stage_floats = (size_t)RB * a.slab_ld;
  auto issue_block = [&](int gb, int s) {              // thread 0 only
    if (gb >= total_blocks) return;
    const int r0 = (gb % nblocks) * RB;
    const int cnt = min(RB, nrows - r0);
    sink_bulk_row(ring_s + (size_t)s * stage_floats, erows + (size_t)r0 * a.ld, (unsigned)cnt * (unsigned)a.ld * 4u, &full_bar[s]);
  };
  if (tid == 0 && nrows > 0)
    for (int s = 0; s < ring; ++s) issue_block(s, s);
  int gb = 0, stage = 0;
  unsigned phase = 0;
  float vref = 0.f;
  float v0_prev = v_s[0];
  bool bad = false;
  for (int it = 0; it < a.iters; ++it) {
    SINK_TRACE(0);
    float* cs = a.colsum + (size_t)(it % 3) * kWays * cs_ld;
    float* my = cs + (size_t)(b % kWays) * cs_ld;
    const float Rref = norm - vref;
    float4 cacc[KG];
#pragma unroll
    for (int k = 0; k < KG; ++k) cacc[k] = make_float4(0.f, 0.f, 0.f, 0.f);
    // the weights of my column groups are fixed for the iteration: in registers where they fit next to the rows and
    // the column partials, otherwise re-read from shared memory with every row
    constexpr bool kCacheW = HOLD && KG * (RC + 2) <= 24;
    float4 w4[kCacheW ? KG : 1];
    if (kCacheW) {
#pragma unroll
      for (int k = 0; k < KG; ++k) {
        const int g4 = tid + k * kThreads;
        w4[k] = (g4 < n4) ? *reinterpret_cast<const float4*>(w_s + 4 * g4) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
    }
    const float4 zero4 = make_float4(0.f, 0.f, 0.f, 0.f);
    int step = 0;
    for (int blk = 0; blk < nblocks; ++blk, ++gb) {
      const int rows_blk = min(RB, nrows - blk * RB);
      sink_bar_wait(&full_bar[stage], phase, a.err);
      const float* blk_s = ring_s + (size_t)stage * stage_floats;
      for (int rb0 = 0; rb0 < rows_blk; rb0 += RC, ++step) {
        const int par = step & 1;
        const int r0 = blk * RB + rb0;
        const int nr = min(RC, rows_blk - rb0);           // live rows of this step (uniform)
        const bool last_step = rb0 + RC >= rows_blk;      // of this block: its stage can be refilled afterwards
        const float4* row4[RC];
#pragma unroll
        for (int rr = 0; rr < RC; ++rr) row4[rr] = reinterpret_cast<const float4*>(blk_s + (size_t)(rb0 + rr) * a.slab_ld);
        float4 cur[HOLD ? RC : 1][HOLD ? KG : 1];
        float p[RC];
#pragma unroll
        for (int rr = 0; rr < RC; ++rr) p[rr] = 0.f;
#pragma unroll
        for (int k = 0; k < KG; ++k) {
          const int g4 = tid + k * kThreads;
          const float4 wk = kCacheW ? w4[kCacheW ? k : 0] : ((g4 < n4) ? *reinterpret_cast<const float4*>(w_s + 4 * g4) : zero4);
#pragma unroll
          for (int rr = 0; rr < RC; ++rr) {
            const float4 e = (rr < nr && g4 < n4) ? row4[rr][g4] : zero4;
            if (HOLD) cur[HOLD ? rr : 0][HOLD ? k : 0] = e;
            p[rr] += fmaf(e.x, wk.x, e.y * wk.y) + fmaf(e.z, wk.z, e.w * wk.w);
          }
        }
#pragma unroll
        for (int o = 16; o; o >>= 1) {
#pragma unroll
          for (int rr = 0; rr < RC; ++rr) p[rr] += __shfl_xor_sync(0xffffffffu, p[rr], o);
        }
        if (lane < RC) {
          float mine = p[0];
#pragma unroll
          for (int rr = 1; rr < RC; ++rr) mine = (lane == rr) ? p[rr] : mine;
          rsum_s[par][warp][lane] = mine;
        }
        __syncthreads();                               // the row sums are published (HOLD: and the rows are in registers)
        if (HOLD && last_step && tid == 0) issue_block(gb + ring, stage);
        float er[RC];
        {
          float sr[RC];
#pragma unroll
          for (int rr = 0; rr < RC; ++rr) sr[rr] = (lane < kWarps) ? rsum_s[par][lane][rr] : 0.f;
#pragma unroll
          for (int o = 8; o; o >>= 1) {                 // 16 partials: every warp finishes the rows itself
#pragma unroll
            for (int rr = 0; rr < RC; ++rr) sr[rr] += __shfl_xor_sync(0xffffffffu, sr[rr], o);
          }
#pragma unroll
          for (int rr = 0; rr < RC; ++rr) {
            sr[rr] = __shfl_sync(0xffffffffu, sr[rr], 0);
            er[rr] = 0.f;
            if (rr < nr) {
              const int r = r0 + rr;
              bad = bad || !sum_ok(sr[rr]);
              const float lmu = (r_begin + r == n0) ? log_mu_last : norm;
              const float lse_rel = vref + logf(sr[rr]);
              er[rr] = ex2(((lmu - lse_rel) - Rref) * kLog2e);
              if (tid == 0) u_s[r] = lmu - (rmax_s[r] + lse_rel);
            }
          }
        }
#pragma unroll
        for (int k = 0; k < KG; ++k) {
          const int g4 = tid + k * kThreads;
#pragma unroll
          for (int rr = 0; rr < RC; ++rr) {
            const float4 e = HOLD ? cur[HOLD ? rr : 0][HOLD ? k : 0] : ((rr < nr && g4 < n4) ? row4[rr][g4] : zero4);
            cacc[k].x = fmaf(e.x, er[rr], cacc[k].x); cacc[k].y = fmaf(e.y, er[rr], cacc[k].y);
            cacc[k].z = fmaf(e.z, er[rr], cacc[k].z); cacc[k].w = fmaf(e.w, er[rr], cacc[k].w);
          }
        }
        if (!HOLD && last_step) {
          __syncthreads();                             // everybody has read the block for the second time
          if (tid == 0) issue_block(gb + ring, stage);
        }
      }
      if (++stage == ring) { stage = 0; phase ^= 1u; }
    }
    SINK_TRACE(1);
    if (b < Ga) {
#pragma unroll
      for (int k = 0; k < KG; ++k) {
        const int g4 = tid + k * kThreads;
        if (g4 < n4)
          asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(my + 4 * g4), "f"(cacc[k].x), "f"(cacc[k].y),
                       "f"(cacc[k].z), "f"(cacc[k].w)
                       : "memory");
      }
    }
    SINK_TRACE(2);
    target += (unsigned)G;
    grid_hop(counter, target, a.err);
    SINK_TRACE(3);
    {                                               // recycle the buffer that was read one iteration ago
      float* old = a.colsum + (size_t)((it + 2) % 3) * kWays * cs_ld;
      for (int w = 0; w < kWays; ++w)
        for (int j = c_begin + tid; j < c_end; j += kThreads) old[(size_t)w * cs_ld + j] = 0.f;
    }
    const float v0 = v0_prev;
    ColUpdate cu{a, g, cs, cs_ld, Rref, v0, it == a.iters - 1, v_s, w_s};
    float4 cl[KG], wn;
#pragma unroll
    for (int k = 0; k < KG; ++k) {
      const int g4 = tid + k * kThreads;
      cl[k] = (g4 < n4) ? cu.load(g4) : make_float4(1.f, 1.f, 1.f, 1.f);
    }
#pragma unroll
    for (int k = 0; k < KG; ++k) {
      const int g4 = tid + k * kThreads;
      if (g4 < n4) bad = !cu.finish(g4, cl[k], wn) || bad;
    }
    SINK_TRACE(4);
    vref = v0;
    __syncthreads();
    v0_prev = v_s[0];
    SINK_TRACE(5);
  }
  if (bad) atomicOr(&a.err[kErrRedo], 1u);
  if (a.iters == 0) {
    __syncthreads();
    for (int j = tid; j < C; j += kThreads) v_s[j] = 0.f;
    for (int j = c_begin + tid; j < c_end; j += kThreads) a.v[j] = 0.f;
    __syncthreads();
  }
  sink_final_pass(a, g, u_s, v_s, red_m, red_s, (unsigned)(a.iters + 1));
}

// =====================================================================================================================
// Exact iteration (log-sum-exp per element): (max, sum) partials per CTA and column, combined by the CTA that owns the
// column and broadcast back through L2; flags instead of a grid barrier.  Fallback only.
// =====================================================================================================================
__global__ void __launch_bounds__(kThreads, 1) k_sinkhorn_exact(SinkArgs a) {
  extern __shared__ __align__(16) float smem[];
  __shared__ float red_m[32][17], red_s[32][17];
  if (a.only_if_redo && ld_acquire_u32(&a.err[kErrRedo]) == 0u) return;    // the scaled-kernel launch succeeded
  const SinkGeom g = sink_geom(a);
  const int n0 = g.n0, n1 = g.n1, C = g.C, G = g.G, b = g.b, nrows = g.nrows, r_begin = g.r_begin, Ga = g.Ga;
  const int c_begin = g.c_begin, c_end = g.c_end;
  const float norm = g.norm, log_mu_last = g.log_mu_last, log_nu_last = g.log_nu_last;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

  const int vlen = (a.n1_max + 1 + 3) & ~3;
  const int rlen = (a.rpc_max + 3) & ~3;
  float* v_s = smem;                                // [vlen], entries >= C stay 0
  float* u_s = v_s + vlen;                          // [rlen]  u_r
  float* slab = u_s + rlen;
  const bool resident = a.slab_rows > 0 && nrows <= a.slab_rows && C <= a.slab_ld;
  const int zs = resident ? a.slab_ld : a.ld;       // row stride used by the passes
  const float* zbase = resident ? slab : a.Z + (size_t)r_begin * a.ld;
  const int C4 = resident ? ((C + 3) & ~3) : C;     // resident rows are padded with -inf up to a multiple of 4

  if (resident) {
    for (int r = warp; r < nrows; r += kWarps) {
      const float* src = a.Z + (size_t)(r_begin + r) * a.ld;
      float* dst = slab + (size_t)r * a.slab_ld;
      for (int j = lane; j < C4; j += 32) dst[j] = (j < C) ? src[j] : -CUDART_INF_F;
    }
  }
  for (int j = tid; j < vlen; j += kThreads) v_s[j] = 0.f;
  if (a.iters == 0) for (int j = c_begin + tid; j < c_end; j += kThreads) a.v[j] = 0.f;
  if (b == 0 && tid == 0) a.err[kErrPath] = GIMS_STATUS_SINKHORN_EXACT;
  __syncthreads();

  long long* const gtrace = (tid == 0) ? g_sink_trace : nullptr;
  long long* trace = (b == 0) ? gtrace : nullptr;
  const bool reg_rows = resident && (C4 >> 2) <= kRowChunks * 32;   // a row's (z + v) fits the lanes' registers
  const bool reg_cols = resident && nrows <= kRMax;
  // epochs continue after those a preceding scaled-kernel launch has used for its final pass
  const unsigned ep0 = a.only_if_redo ? (unsigned)(a.iters + 1) : 0u;
  for (int it = 0; it < a.iters; ++it) {
    SINK_TRACE(0);
    // ---- row pass -------------------------------------------------------------------------
    if (reg_rows) {
      const int n4 = C4 >> 2;
      for (int r = warp; r < nrows; r += kWarps) {
        const float4* z4 = reinterpret_cast<const float4*>(slab + (size_t)r * a.slab_ld);
        const float4* v4 = reinterpret_cast<const float4*>(v_s);
        float4 x[kRowChunks];
        float m = -CUDART_INF_F;
#pragma unroll
        for (int k = 0; k < kRowChunks; ++k) {
          const int i = lane + 32 * k;
          if (i < n4) {
            const float4 zz = z4[i], vv = v4[i];
            x[k] = make_float4(zz.x + vv.x, zz.y + vv.y, zz.z + vv.z, zz.w + vv.w);
            m = fmaxf(m, fmaxf(fmaxf(x[k].x, x[k].y), fmaxf(x[k].z, x[k].w)));
          } else {
            x[k] = make_float4(-CUDART_INF_F, -CUDART_INF_F, -CUDART_INF_F, -CUDART_INF_F);
          }
        }
        m = warp_max(m);
        float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
#pragma unroll
        for (int k = 0; k < kRowChunks; ++k) {
          s0 += ex2((x[k].x - m) * kLog2e); s1 += ex2((x[k].y - m) * kLog2e);
          s2 += ex2((x[k].z - m) * kLog2e); s3 += ex2((x[k].w - m) * kLog2e);
        }
        const float s = warp_sum((s0 + s1) + (s2 + s3));
        if (lane == 0) {
          float lmu = (r_begin + r == n0) ? log_mu_last : norm;
          u_s[r] = lmu - (m + logf(s));
        }
      }
    } else {
      for (int r = warp; r < nrows; r += kWarps) {
        const float* z = zbase + (size_t)r * zs;
        float m = -CUDART_INF_F, s = 0.f;
#pragma unroll 4
        for (int j = lane; j < C; j += 32) m = fmaxf(m, z[j] + v_s[j]);
        m = warp_max(m);
#pragma unroll 4
        for (int j = lane; j < C; j += 32) s += ex2((z[j] + v_s[j] - m) * kLog2e);
        s = warp_sum(s);
        if (lane == 0) {
          float lmu = (r_begin + r == n0) ? log_mu_last : norm;
          u_s[r] = lmu - (m + logf(s));
        }
      }
    }
    __syncthreads();
    SINK_TRACE(1);
    // ---- column pass: per-CTA partial LSE ------------------------------------------------------------------
    const unsigned epoch = ep0 + (unsigned)(it + 1);
    if (b < Ga) {
      if (reg_cols) {
        const int Gf = C >> 2;                               // groups of 4 columns, one 128-bit LDS per row
        for (int gq = tid; gq < Gf; gq += kThreads) {
          float4 x[kRMax];
          float4 m = make_float4(-CUDART_INF_F, -CUDART_INF_F, -CUDART_INF_F, -CUDART_INF_F);
#pragma unroll
          for (int r = 0; r < kRMax; ++r) {
            if (r < nrows) {
              const float4 zz = *reinterpret_cast<const float4*>(slab + (size_t)r * a.slab_ld + 4 * gq);
              const float ur = u_s[r];
              x[r] = make_float4(zz.x + ur, zz.y + ur, zz.z + ur, zz.w + ur);
              m.x = fmaxf(m.x, x[r].x); m.y = fmaxf(m.y, x[r].y); m.z = fmaxf(m.z, x[r].z); m.w = fmaxf(m.w, x[r].w);
            } else {
              x[r] = make_float4(-CUDART_INF_F, -CUDART_INF_F, -CUDART_INF_F, -CUDART_INF_F);
            }
          }
          float4 sm = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
          for (int r = 0; r < kRMax; ++r) {
            sm.x += ex2((x[r].x - m.x) * kLog2e); sm.y += ex2((x[r].y - m.y) * kLog2e);
            sm.z += ex2((x[r].z - m.z) * kLog2e); sm.w += ex2((x[r].w - m.w) * kLog2e);
          }
          float2* dst = &a.part[(size_t)b * a.ldp + 4 * gq];
          dst[0] = make_float2(m.x, sm.x); dst[1] = make_float2(m.y, sm.y);
          dst[2] = make_float2(m.z, sm.z); dst[3] = make_float2(m.w, sm.w);
        }
        // the (at most 3) columns left over — among them the dustbin column — are reduced across the lanes of a warp
        const int jl = 4 * Gf + warp;
        if (jl < C) {
          const float xx = (lane < nrows) ? slab[(size_t)lane * a.slab_ld + jl] + u_s[lane] : -CUDART_INF_F;
          const float mm = warp_max(xx);
          const float ss = warp_sum(ex2((xx - mm) * kLog2e));
          if (lane == 0) a.part[(size_t)b * a.ldp + jl] = make_float2(mm, ss);
        }
      } else {
        for (int j = tid; j < C; j += kThreads) {
          float m = -CUDART_INF_F;
          for (int r = 0; r < nrows; ++r) m = fmaxf(m, zbase[(size_t)r * zs + j] + u_s[r]);
          float s = 0.f;
          for (int r = 0; r < nrows; ++r) s += ex2((zbase[(size_t)r * zs + j] + u_s[r] - m) * kLog2e);
          a.part[(size_t)b * a.ldp + j] = make_float2(m, s);
        }
      }
    }
    publish_flag(&a.pflag[b], epoch);
    SINK_TRACE(2);
    // ---- combine the partials of my column range -> v_j ------------------------------------------------
    wait_flags(a.pflag, Ga, epoch, a.err);
    for (int jc = c_begin; jc < c_end; jc += 16) {
      const int jj = tid & 15, gs = tid >> 4, j = jc + jj;
      float m = -CUDART_INF_F, s = 0.f;
      if (j < c_end) {
        float2 w[8];                                   // grid <= 256 -> at most 8 producers per (column, slot)
        const int cnt = (Ga - gs + 31) >> 5;
#pragma unroll
        for (int k = 0; k < 8; ++k)
          if (k < cnt) w[k] = __ldcg(&a.part[(size_t)(gs + 32 * k) * a.ldp + j]);
#pragma unroll
        for (int k = 0; k < 8; ++k)
          if (k < cnt) lse_merge(m, s, w[k].x, w[k].y);
      }
      red_m[gs][jj] = m; red_s[gs][jj] = s;
      __syncthreads();
      SINK_TRACE(3);
      const int jw = jc + warp;                      // warp w finishes column jc + w
      if (jw < c_end) {
        float mm = red_m[lane][warp], ss = red_s[lane][warp];
        float M = warp_max(mm);
        ss = (ss > 0.f) ? ss * ex2((mm - M) * kLog2e) : 0.f;
        ss = warp_sum(ss);
        if (lane == 0) {
          float lnu = (jw == n1) ? log_nu_last : norm;
          float vj = lnu - (M + logf(ss));
          a.vg[jw] = vj;
          if (it == a.iters - 1) a.v[jw] = vj;
        }
      }
      __syncthreads();
    }
    publish_flag(&a.vflag[b], epoch);
    SINK_TRACE(4);
    // ---- gather the new v ----------------------------------------------------------------------------------
    wait_flags(a.vflag, G, epoch, a.err);
    for (int j = tid; j < C; j += kThreads) v_s[j] = __ldcg(&a.vg[j]);
    __syncthreads();
    SINK_TRACE(5);
  }
  sink_final_pass(a, g, u_s, v_s, red_m, red_s, ep0 + (unsigned)(a.iters + 1));
}

// gmatcher.py:286-294
__global__ void k_match_finalize(int n0_max, int n1_max, const int* __restrict__ n_dev, const int* __restrict__ idx0,
                                 const int* __restrict__ idx1, const float* __restrict__ max0, float thr,
                                 int64_t* __restrict__ matches0, int64_t* __restrict__ matches1,
                                 float* __restrict__ ms0, float* __restrict__ ms1, const unsigned* __restrict__ err,
                                 unsigned* __restrict__ status) {
  int n0 = n_dev ? min(n_dev[0], n0_max) : n0_max;
  int n1 = n_dev ? min(n_dev[1], n1_max) : n1_max;
  int t = blockIdx.x * blockDim.x + threadIdx.x;
  // err[0]: a poll timed out; err[1]: which iteration produced the results (GIMS_STATUS_SINKHORN_FAST / _EXACT)
  if (t == 0 && status) atomicOr(status, (err[kErrTimeout] ? GIMS_STATUS_SINKHORN_TIMEOUT : 0u) | err[kErrPath]);
  if (err[kErrTimeout]) {                         // a poll timed out inside the kernel: fail loudly, not silently
    if (t < n0) { ms0[t] = CUDART_NAN_F; matches0[t] = -2; }
    if (t < n1) { ms1[t] = CUDART_NAN_F; matches1[t] = -2; }
    return;
  }
  if (t < n0) {
    int j = idx0[t];
    bool mutual = (unsigned)j < (unsigned)n1 && idx1[j] == t;      // (an argmax over NaNs leaves the index unset)
    float s = mutual ? expf(max0[t]) : 0.f;
    ms0[t] = s;
    matches0[t] = (mutual && s > thr) ? (int64_t)j : (int64_t)-1;
  }
  if (t < n1) {
    int i = idx1[t];
    bool mutual = (unsigned)i < (unsigned)n0 && idx0[i] == t;
    float s = mutual ? expf(max0[i]) : 0.f;      // mutual1 implies mutual0[i]
    ms1[t] = s;
    matches1[t] = (mutual && s > thr) ? (int64_t)i : (int64_t)-1;
  }
}

// =====================================================================================================================
// Wide iteration: problems whose potentials do not fit shared memory (plan() below rejects them; on a B200 about 56 k
// columns and more).  The reference's log-sum-exp iteration in the log domain, streamed from global memory with ordinary,
// non-cooperative launches — three per iteration:
//   k_wide_rows      u_r = log_mu_r - LSE_j (z_rj + v_j): a CTA per kWideRows rows, v read through L1 / L2;
//   k_wide_cols      per (row block, column): the (max, sum) partial of LSE_r (z_rj + u_r) over the block's rows;
//   k_wide_combine   v_j = log_nu_j - LSE over the kWideBlocks partials of column j, merged in row-block order.
// No float atomics and no grid-wide waits: the results do not change from run to run and nothing can time out.  At
// 65536 x 65536 the matrix (17.2 GB) is read twice per iteration, so the iteration is bound by HBM; the exponentials
// (one ex2 per element plus one per chunk of four) hide behind the loads.  The final pass (the same three kernels,
// FINAL = true) evaluates ((Z0 + u) + v) - norm like the shared-memory kernels and feeds k_match_finalize.
// Element offsets are 64-bit throughout: (n0 + 1) * ld exceeds 2^31 from 46341 keypoints on.
// =====================================================================================================================
constexpr int kWideThreads = 256;
constexpr int kWideRows = 8;                  // rows per CTA of the row pass
constexpr int kWideChunk = 4;                 // columns per thread and step of the row pass (strided by kWideThreads)
constexpr int kWideColsPerThread = 4;         // columns per thread of the column pass (strided by kWideThreads)
constexpr int kWideRowStep = 8;               // rows per step of the column pass
constexpr int kWideBlocks = kMaxGrid;         // row blocks of the column pass: the partial buffer is the kernels' `part`

struct WideDims {
  int n0, n1;                                 // live counts
  float norm, log_mu_last, log_nu_last;
};
__device__ __forceinline__ WideDims wide_dims(int n0_max, int n1_max, const int* n_dev) {
  WideDims d;
  d.n0 = n_dev ? min(n_dev[0], n0_max) : n0_max;
  d.n1 = n_dev ? min(n_dev[1], n1_max) : n1_max;
  const float ms = (float)d.n0, ns = (float)d.n1;          // as sink_geom (gmatcher.py:62-64)
  d.norm = -logf(ms + ns);
  d.log_mu_last = logf(ns) + d.norm;
  d.log_nu_last = logf(ms) + d.norm;
  return d;
}
// rows per block of the column pass over `rows` rows, and the number of blocks that own at least one
__device__ __forceinline__ int wide_rows_per_block(int rows) { return max(1, (rows + kWideBlocks - 1) / kWideBlocks); }

// (m, s) <- LSE-combine with (pm, ps); empty partials are (-inf, 0) and leave the other side as it is
__device__ __forceinline__ void lse_merge_safe(float& m, float& s, float pm, float ps) {
  const float mn = fmaxf(m, pm);
  if (mn == -CUDART_INF_F) return;
  s = s * ex2((m - mn) * kLog2e) + ps * ex2((pm - mn) * kLog2e);
  m = mn;
}
// online LSE over a chunk of N values (-inf = masked): one rescale per chunk, one ex2 per value
template <int N>
__device__ __forceinline__ void lse_chunk(float& m, float& s, const float* x) {
  float cm = x[0];
#pragma unroll
  for (int k = 1; k < N; ++k) cm = fmaxf(cm, x[k]);
  const float mn = fmaxf(m, cm);
  if (mn == -CUDART_INF_F) return;
  float acc = s * ex2((m - mn) * kLog2e);
#pragma unroll
  for (int k = 0; k < N; ++k) acc += ex2((x[k] - mn) * kLog2e);
  s = acc;
  m = mn;
}
__device__ __forceinline__ bool argmax_better(float b, int j, float best, int bj) { return b > best || (b == best && j < bj); }

// Row pass.  FINAL = false: u_r for the live rows r <= n0 (dustbin row included) from the current v.
// FINAL = true: row max + first argmax of ((z + u_r) + v_j) - norm over the keypoint columns, rows < n0.
template <bool FINAL>
__global__ void __launch_bounds__(kWideThreads) k_wide_rows(const float* __restrict__ Z, size_t ld, int n0_max, int n1_max,
                                                            const int* __restrict__ n_dev, const float* __restrict__ v,
                                                            float* __restrict__ u, int* __restrict__ idx0,
                                                            float* __restrict__ max0) {
  __shared__ float red_a[kWideThreads / 32][kWideRows];
  __shared__ float red_b[kWideThreads / 32][kWideRows];
  const WideDims d = wide_dims(n0_max, n1_max, n_dev);
  const int rows = FINAL ? d.n0 : d.n0 + 1, cols = FINAL ? d.n1 : d.n1 + 1;
  const int r0 = blockIdx.x * kWideRows;
  if (r0 >= rows) return;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  float a[kWideRows], b[kWideRows], ur[kWideRows];        // (max, sum) or (best value, best column as int bits)
#pragma unroll
  for (int rr = 0; rr < kWideRows; ++rr) {
    a[rr] = -CUDART_INF_F;
    b[rr] = FINAL ? __int_as_float(0x7fffffff) : 0.f;
    ur[rr] = (FINAL && r0 + rr < rows) ? u[r0 + rr] : 0.f;
  }
  const float* zr = Z + (size_t)r0 * ld;
  for (int j0 = 0; j0 < cols; j0 += kWideChunk * kWideThreads) {
    float vj[kWideChunk], x[kWideRows][kWideChunk];
#pragma unroll
    for (int q = 0; q < kWideChunk; ++q) {
      const int j = j0 + tid + q * kWideThreads;
      vj[q] = (j < cols) ? v[j] : 0.f;
#pragma unroll
      for (int rr = 0; rr < kWideRows; ++rr)
        x[rr][q] = (j < cols && r0 + rr < rows) ? __ldcs(zr + (size_t)rr * ld + j) : -CUDART_INF_F;
    }
#pragma unroll
    for (int rr = 0; rr < kWideRows; ++rr) {
      if (FINAL) {
#pragma unroll
        for (int q = 0; q < kWideChunk; ++q) {                // columns ascending: strict > keeps the first maximum
          const float t = ((x[rr][q] + ur[rr]) + vj[q]) - d.norm;
          if (t > a[rr]) { a[rr] = t; b[rr] = __int_as_float(j0 + tid + q * kWideThreads); }
        }
      } else {
#pragma unroll
        for (int q = 0; q < kWideChunk; ++q) x[rr][q] += vj[q];
        lse_chunk<kWideChunk>(a[rr], b[rr], x[rr]);
      }
    }
  }
#pragma unroll
  for (int rr = 0; rr < kWideRows; ++rr) {
#pragma unroll
    for (int o = 16; o; o >>= 1) {
      const float pa = __shfl_xor_sync(0xffffffffu, a[rr], o), pb = __shfl_xor_sync(0xffffffffu, b[rr], o);
      if (FINAL) {
        if (argmax_better(pa, __float_as_int(pb), a[rr], __float_as_int(b[rr]))) { a[rr] = pa; b[rr] = pb; }
      } else {
        lse_merge_safe(a[rr], b[rr], pa, pb);
      }
    }
    if (lane == 0) { red_a[warp][rr] = a[rr]; red_b[warp][rr] = b[rr]; }
  }
  __syncthreads();
  if (tid < kWideRows && r0 + tid < rows) {
    const int r = r0 + tid;
    float m = red_a[0][tid], s = red_b[0][tid];
    for (int w = 1; w < kWideThreads / 32; ++w) {             // warps in order
      if (FINAL) {
        if (argmax_better(red_a[w][tid], __float_as_int(red_b[w][tid]), m, __float_as_int(s))) { m = red_a[w][tid]; s = red_b[w][tid]; }
      } else {
        lse_merge_safe(m, s, red_a[w][tid], red_b[w][tid]);
      }
    }
    if (FINAL) {
      idx0[r] = __float_as_int(s);
      max0[r] = m;
    } else {
      const float lmu = (r == d.n0) ? d.log_mu_last : d.norm;
      u[r] = lmu - (m + logf(s));
    }
  }
}

// Column pass: CTA (x, y) covers columns [x * 1024, +1024) and row block y.  FINAL = false: (max, sum) of z_rj + u_r over
// the block's live rows (dustbin row included).  FINAL = true: (best value, first row) of ((z + u_r) + v_j) - norm over
// the block's keypoint rows, keypoint columns only.
template <bool FINAL>
__global__ void __launch_bounds__(kWideThreads) k_wide_cols(const float* __restrict__ Z, size_t ld, int n0_max, int n1_max,
                                                            const int* __restrict__ n_dev, const float* __restrict__ u,
                                                            const float* __restrict__ v, float2* __restrict__ part,
                                                            size_t ldp) {
  const WideDims d = wide_dims(n0_max, n1_max, n_dev);
  const int rows = FINAL ? d.n0 : d.n0 + 1, cols = FINAL ? d.n1 : d.n1 + 1;
  const int rpb = wide_rows_per_block(rows);
  const int rb = blockIdx.y * rpb, re = min(rb + rpb, rows);
  const int c0 = blockIdx.x * (kWideColsPerThread * kWideThreads) + threadIdx.x;
  if (rb >= re || blockIdx.x * (kWideColsPerThread * kWideThreads) >= cols) return;
  float a[kWideColsPerThread], b[kWideColsPerThread], vj[kWideColsPerThread];
#pragma unroll
  for (int q = 0; q < kWideColsPerThread; ++q) {
    const int j = c0 + q * kWideThreads;
    a[q] = -CUDART_INF_F;
    b[q] = FINAL ? __int_as_float(0x7fffffff) : 0.f;
    vj[q] = (FINAL && j < cols) ? v[j] : 0.f;
  }
  for (int r0 = rb; r0 < re; r0 += kWideRowStep) {
    float x[kWideColsPerThread][kWideRowStep], urs[kWideRowStep];
#pragma unroll
    for (int rr = 0; rr < kWideRowStep; ++rr) urs[rr] = (r0 + rr < re) ? u[r0 + rr] : 0.f;
#pragma unroll
    for (int q = 0; q < kWideColsPerThread; ++q) {
      const int j = c0 + q * kWideThreads;
#pragma unroll
      for (int rr = 0; rr < kWideRowStep; ++rr)
        x[q][rr] = (j < cols && r0 + rr < re) ? __ldcs(Z + (size_t)(r0 + rr) * ld + j) : -CUDART_INF_F;
    }
#pragma unroll
    for (int q = 0; q < kWideColsPerThread; ++q) {
      if (FINAL) {
#pragma unroll
        for (int rr = 0; rr < kWideRowStep; ++rr) {           // rows ascending: strict > keeps the first maximum
          const float t = ((x[q][rr] + urs[rr]) + vj[q]) - d.norm;
          if (t > a[q]) { a[q] = t; b[q] = __int_as_float(r0 + rr); }
        }
      } else {
#pragma unroll
        for (int rr = 0; rr < kWideRowStep; ++rr) x[q][rr] += urs[rr];
        lse_chunk<kWideRowStep>(a[q], b[q], x[q]);
      }
    }
  }
#pragma unroll
  for (int q = 0; q < kWideColsPerThread; ++q) {
    const int j = c0 + q * kWideThreads;
    if (j < cols) part[(size_t)blockIdx.y * ldp + j] = make_float2(a[q], b[q]);
  }
}

// Fixed-order combine of the row-block partials of each column.  FINAL = false: v_j (into v_it, and into v_out after the
// last iteration).  FINAL = true: column max + first argmax, and the path bit for k_match_finalize.
template <bool FINAL>
__global__ void __launch_bounds__(kWideThreads) k_wide_combine(int n0_max, int n1_max, const int* __restrict__ n_dev,
                                                               const float2* __restrict__ part, size_t ldp,
                                                               float* __restrict__ v_it, float* __restrict__ v_out,
                                                               int* __restrict__ idx1, float* __restrict__ max1,
                                                               unsigned* __restrict__ err) {
  const WideDims d = wide_dims(n0_max, n1_max, n_dev);
  const int rows = FINAL ? d.n0 : d.n0 + 1, cols = FINAL ? d.n1 : d.n1 + 1;
  const int rpb = wide_rows_per_block(rows);
  const int nb = (rows + rpb - 1) / rpb;
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (FINAL && j == 0) err[kErrPath] = GIMS_STATUS_SINKHORN_WIDE;
  if (j >= cols) return;
  float m = -CUDART_INF_F, s = FINAL ? __int_as_float(0x7fffffff) : 0.f;
  for (int k = 0; k < nb; ++k) {                              // row blocks in order
    const float2 p = part[(size_t)k * ldp + j];
    if (FINAL) {
      if (argmax_better(p.x, __float_as_int(p.y), m, __float_as_int(s))) { m = p.x; s = p.y; }
    } else {
      lse_merge_safe(m, s, p.x, p.y);
    }
  }
  if (FINAL) {
    idx1[j] = __float_as_int(s);
    max1[j] = m;
  } else {
    const float lnu = (j == d.n1) ? d.log_nu_last : d.norm;
    const float vj = lnu - (m + logf(s));
    v_it[j] = vj;
    if (v_out) v_out[j] = vj;
  }
}

// iters == 0: the potentials stay 0 (live entries only, as the other kernels leave the rest untouched)
__global__ void k_wide_zero(int n0_max, int n1_max, const int* __restrict__ n_dev, float* __restrict__ u,
                            float* __restrict__ v) {
  const WideDims d = wide_dims(n0_max, n1_max, n_dev);
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t <= d.n0) u[t] = 0.f;
  if (t <= d.n1) v[t] = 0.f;
}

int launch_wide(const float* Z, int ld, int n0_max, int n1_max, const int* n_dev, int iters, float* u, float* v,
                float* v_it, float2* part, int* idx0, int* idx1, float* max0, float* max1, unsigned* err, cudaStream_t st) {
  const size_t ldz = (size_t)ld, ldp = (size_t)n1_max + 1;
  const unsigned row_grid = (unsigned)cdiv(n0_max + 1, kWideRows);
  const dim3 col_grid((unsigned)cdiv(n1_max + 1, kWideColsPerThread * kWideThreads), kWideBlocks);
  const unsigned comb_grid = (unsigned)cdiv(n1_max + 1, kWideThreads);
  GIMS_CUDA_OK(cudaMemsetAsync(v_it, 0, ldp * sizeof(float), st));
  if (iters == 0) {
    k_wide_zero<<<cdiv((n0_max > n1_max ? n0_max : n1_max) + 1, 256), 256, 0, st>>>(n0_max, n1_max, n_dev, u, v);
    GIMS_LAUNCH_OK();
  }
  for (int it = 0; it < iters; ++it) {
    k_wide_rows<false><<<row_grid, kWideThreads, 0, st>>>(Z, ldz, n0_max, n1_max, n_dev, v_it, u, nullptr, nullptr);
    GIMS_LAUNCH_OK();
    k_wide_cols<false><<<col_grid, kWideThreads, 0, st>>>(Z, ldz, n0_max, n1_max, n_dev, u, nullptr, part, ldp);
    GIMS_LAUNCH_OK();
    k_wide_combine<false><<<comb_grid, kWideThreads, 0, st>>>(n0_max, n1_max, n_dev, part, ldp, v_it,
                                                              it == iters - 1 ? v : nullptr, nullptr, nullptr, nullptr);
    GIMS_LAUNCH_OK();
  }
  k_wide_rows<true><<<row_grid, kWideThreads, 0, st>>>(Z, ldz, n0_max, n1_max, n_dev, v_it, u, idx0, max0);
  GIMS_LAUNCH_OK();
  k_wide_cols<true><<<col_grid, kWideThreads, 0, st>>>(Z, ldz, n0_max, n1_max, n_dev, u, v_it, part, ldp);
  GIMS_LAUNCH_OK();
  k_wide_combine<true><<<comb_grid, kWideThreads, 0, st>>>(n0_max, n1_max, n_dev, part, ldp, nullptr, nullptr, idx1, max1,
                                                           err);
  GIMS_LAUNCH_OK();
  return GIMS_OK;
}

// Which kernel serves a problem of at most (n0_max + 1) x (n1_max + 1) on a grid of G CTAs — decided on the host from
// the capacities, so that workspace sizing and launch agree.
enum SinkKind { kSinkReg = 0, kSinkStream = 1, kSinkExact = 2 };
struct SinkPlan {
  SinkKind kind;
  int kg, rc, rb;      // streaming kernel: float4 groups per thread and row; stages of the ring; rows per stage
  int rpc, slab_ld, slab_rows;
  size_t dyn_smem;     // of the chosen scaled-kernel kernel
  size_t dyn_exact;    // of the exact kernel
  int exact_slab_rows;
};
bool plan(SinkPlan& p, int n0_max, int n1_max, int G, int smem_optin, bool vec_ok, int iters) {
  const int R = n0_max + 1, C = n1_max + 1;
  p.rpc = (R + G - 1) / G;
  p.slab_ld = (C + 3) & ~3;
  const size_t vlen = (size_t)p.slab_ld, rlen = (size_t)((p.rpc + 3) & ~3);
  const size_t budget = (size_t)smem_optin - 6144;     // static smem (reduction arrays) + margin
  const size_t slab_bytes = (size_t)p.rpc * p.slab_ld * sizeof(float);
  // exact kernel: v | u | slab (if it fits)
  const size_t fixed_exact = (vlen + rlen) * sizeof(float);
  p.exact_slab_rows = (fixed_exact + slab_bytes <= budget) ? p.rpc : 0;
  p.dyn_exact = fixed_exact + (p.exact_slab_rows ? slab_bytes : 0);
  if (p.dyn_exact > budget) return false;
  p.kind = kSinkExact; p.kg = 0; p.rc = 0; p.slab_rows = 0; p.dyn_smem = 0;
  if (iters <= 0) return true;
  // on-chip kernel: v, w | u, rmax, e | staging / shared-memory rows (16 rows in registers + up to 16 in shared memory)
  const size_t fixed_reg = (2 * vlen + 3 * rlen) * sizeof(float);
  const size_t stage_bytes = (size_t)(p.rpc < kRMax ? p.rpc : kRMax) * p.slab_ld * sizeof(float);
  if (p.rpc <= kRMax + kRSmem && (C >> 2) <= kThreads && fixed_reg + stage_bytes <= budget) {
    p.kind = kSinkReg; p.slab_rows = p.rpc; p.dyn_smem = fixed_reg + stage_bytes;
    return true;
  }
  if (!vec_ok) return true;
  const int n4 = p.slab_ld >> 2;
  const int kg = (n4 + kThreads - 1) / kThreads;
  const size_t fixed_stream = (2 * vlen + 2 * rlen) * sizeof(float);
  const size_t row_bytes = (size_t)p.slab_ld * sizeof(float);
  // (more than ~14 k columns leave no room for two stages next to v and w: those problems run the exact kernel)
  if (kg <= 9 && fixed_stream + 2 * row_bytes <= budget) {
    p.kind = kSinkStream;
    p.kg = kg <= 3 ? 3 : (kg <= 5 ? 5 : 9);
    // stages of about 64 KB (see the kernel: bulk copies complete one at a time), at least two stages
    const size_t avail = budget - fixed_stream;
    size_t rb = (66 * 1024) / row_bytes;
    if (rb < 2) rb = 2;
    while (rb > 1 && 2 * rb * row_bytes > avail) --rb;
    size_t ring = avail / (rb * row_bytes);
    if (ring > 4) ring = 4;
    p.rc = (int)ring; p.rb = (int)rb;
    p.dyn_smem = fixed_stream + ring * rb * row_bytes;
  }
  return true;
}

struct SinkWs {
  // zeroed before every launch (tags)
  unsigned* err;
  unsigned* pflag;
  unsigned* vflag;
  float* colsum;
  unsigned* cmkey;
  size_t zero_bytes;
  float2* part;
  float* vg;
  float* max0;
  float* max1;
  float* E;
};

size_t carve(SinkWs& w, void* base, size_t cap, int n0_max, int n1_max, int grid, bool with_e) {
  Arena a(base, cap);
  size_t ldp = (size_t)n1_max + 1;
  size_t cs_ld = (ldp + 3) & ~(size_t)3;
  w.err = a.take<unsigned>(64);
  w.pflag = a.take<unsigned>(kMaxGrid);
  w.vflag = a.take<unsigned>(kMaxGrid);
  w.colsum = a.take<float>(3 * kWays * cs_ld);
  w.cmkey = a.take<unsigned>(cs_ld);
  w.zero_bytes = align_up(a.off, 256);
  w.part = a.take<float2>((size_t)grid * ldp);
  w.vg = a.take<float>(ldp + 4);
  w.max0 = a.take<float>(n0_max + 1);
  w.max1 = a.take<float>(n1_max + 1);
  w.E = with_e ? a.take<float>((size_t)(n0_max + 1) * cs_ld) : nullptr;
  return align_up(a.off, 256);
}

// Capacities above which the scaled matrix may need the scratch buffer (the register kernel needs none).  The grid of
// the launch is not known to the workspace query, so it assumes the streaming kernel whenever the register kernel
// cannot be guaranteed on a part with >= 128 SMs.  The widest streaming instantiation holds 9 float4 groups per thread
// (plan()): wider problems never stream, and E ((n0_max + 1) x ld floats, 17.2 GB at 65536 x 65536) is not reserved.
bool may_stream(int n0_max, int n1_max) {
  if ((((size_t)n1_max + 1 + 3) >> 2) > (size_t)9 * kThreads) return false;
  return n0_max + 1 > (kRMax + kRSmem) * 64 || ((n1_max + 1) >> 2) > kThreads;
}

// Grid of a problem.  The on-chip kernel runs on HALF the SMs whenever its slab then still fits (<= 32 rows per CTA):
// an iteration is bound by the grid-wide exchange, which gets cheaper with fewer CTAs about as fast as the arithmetic
// gets longer, and the other half of the GPU stays free for other streams (GIMS_SINKHORN_GRID=full: all SMs, for A/B
// measurements).  Everything else uses every SM.
struct SinkGrid { int G; bool half; };
SinkGrid choose_grid(int n0_max, int n1_max, int sms, int smem_optin, int iters) {
  static const bool force_full = [] { const char* e = getenv("GIMS_SINKHORN_GRID"); return e && e[0] == 'f'; }();
  const int full = sms < kMaxGrid ? sms : kMaxGrid;
  const int half = full / 2;
  SinkPlan p;
  if (!force_full && half >= 32 && plan(p, n0_max, n1_max, half, smem_optin, false, iters) && p.kind == kSinkReg)
    return {half, true};
  return {full, false};
}

template <int KG, int RC, bool HOLD>
int launch_stream(SinkArgs& a, int G, size_t dyn, int budget, cudaStream_t st) {
  GIMS_CUDA_OK(cudaFuncSetAttribute(k_sinkhorn_stream<KG, RC, HOLD>, cudaFuncAttributeMaxDynamicSharedMemorySize, budget));
  void* params[] = {&a};
  GIMS_CUDA_OK(cudaLaunchCooperativeKernel((const void*)k_sinkhorn_stream<KG, RC, HOLD>, dim3(G), dim3(kThreads), params, dyn, st));
  return GIMS_OK;
}

}  // namespace

}  // namespace gims

using namespace gims;

extern "C" int gims_debug_sinkhorn_trace(long long* dev_buf) {
  GIMS_CUDA_OK(cudaMemcpyToSymbol(g_sink_trace, &dev_buf, sizeof(dev_buf)));
  return GIMS_OK;
}

extern "C" int gims_couplings_ld(int n1_max) { return coup_ld(n1_max); }

// (kMaxGrid rows of partials: the largest grid of the cooperative kernels and the row blocks of the wide path)
extern "C" size_t gims_sinkhorn_workspace_bytes(int n0_max, int n1_max) {
  SinkWs w;
  return carve(w, nullptr, 0, n0_max, n1_max, kMaxGrid, may_stream(n0_max, n1_max));
}

// largest n1_max (image-1 keypoints) whose potentials fit the scaled-kernel kernels' budget for n0_max <= GIMS_MAX_KPTS,
// capped at the widest streaming instantiation; the exact kernel serves wider problems while its potentials fit shared
// memory, the wide path the rest (plan())
extern "C" int gims_sinkhorn_max_columns(void) {
  int dev = 0, sms = 0, smem_optin = 0;
  if (cudaGetDevice(&dev) != cudaSuccess ||
      cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess ||
      cudaDeviceGetAttribute(&smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev) != cudaSuccess || sms < 1)
    return 0;
  int G = sms < kMaxGrid ? sms : kMaxGrid;
  long long budget = (long long)smem_optin - 6144;
  long long rlen = ((GIMS_MAX_KPTS + 1 + G - 1) / G + 3) & ~3;
  long long c = (budget / 4 - 3 * rlen) / 2 - 4;         // 2 * round4(C) + 3 * rlen floats <= budget
  long long cap = 9LL * kThreads * 4 - 4;                // widest streaming-kernel instantiation
  if (c > cap) c = cap;
  return (int)(c < 2 ? 0 : c - 1);
}

extern "C" int gims_sinkhorn_match(const float* couplings, int ld, int n0_max, int n1_max, const int* n_dev, int iters,
                                   float match_threshold, void* workspace, size_t workspace_bytes, float* u, float* v,
                                   int* indices0, int* indices1, int64_t* matches0, int64_t* matches1, float* mscores0,
                                   float* mscores1, unsigned* status_dev, void* stream) {
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (!couplings || !workspace || !u || !v || !indices0 || !indices1 || !matches0 || !matches1 || !mscores0 || !mscores1) {
    set_error("gims_sinkhorn_match: null pointer argument");
    return GIMS_ERR_ARG;
  }
  if (n0_max < 1 || n1_max < 1 || iters < 0 || ld < n1_max + 1) { set_error("gims_sinkhorn_match: bad sizes"); return GIMS_ERR_ARG; }
  int dev = 0, sms = 0, smem_optin = 0;
  GIMS_CUDA_OK(cudaGetDevice(&dev));
  GIMS_CUDA_OK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  GIMS_CUDA_OK(cudaDeviceGetAttribute(&smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
  const SinkGrid grid = choose_grid(n0_max, n1_max, sms, smem_optin, iters);
  const int G = grid.G;
  const bool with_e = may_stream(n0_max, n1_max);
  // 128-bit loads of whole rows need a 16-byte aligned base and pitch (gims_couplings_ld gives such a pitch); the scratch
  // matrix E uses the caller's pitch
  const bool vec_ok = with_e && (ld % 4 == 0) && (reinterpret_cast<uintptr_t>(couplings) % 16 == 0) &&
                      (size_t)ld == (((size_t)n1_max + 1 + 3) & ~(size_t)3);
  SinkPlan p;
  // potentials wider than the shared memory of the cooperative kernels: the wide path
  const bool wide = !plan(p, n0_max, n1_max, G, smem_optin, vec_ok, iters);
  SinkWs w;
  size_t need = carve(w, workspace, workspace_bytes, n0_max, n1_max, wide ? kMaxGrid : G, with_e);
  if (need > workspace_bytes) { set_error("gims_sinkhorn_match: workspace %zu < %zu", workspace_bytes, need); return GIMS_ERR_WORKSPACE; }
  if (wide) {
    GIMS_CUDA_OK(cudaMemsetAsync(w.err, 0, w.zero_bytes, st));
    {
      ProfScope prof(GIMS_PROF_SINKHORN, st);
      GIMS_TRY(launch_wide(couplings, ld, n0_max, n1_max, n_dev, iters, u, v, w.vg, w.part, indices0, indices1, w.max0,
                           w.max1, w.err, st));
    }
    const int m = n0_max > n1_max ? n0_max : n1_max;
    k_match_finalize<<<cdiv(m, 256), 256, 0, st>>>(n0_max, n1_max, n_dev, indices0, indices1, w.max0, match_threshold,
                                                   matches0, matches1, mscores0, mscores1, w.err, status_dev);
    GIMS_LAUNCH_OK();
    return GIMS_OK;
  }
  const int budget = smem_optin - 6144;
  SinkArgs a;
  a.Z = couplings; a.ld = ld; a.n0_max = n0_max; a.n1_max = n1_max; a.n_dev = n_dev; a.iters = iters;
  a.u = u; a.v = v; a.part = w.part; a.vg = w.vg; a.pflag = w.pflag; a.vflag = w.vflag; a.colsum = w.colsum;
  a.cmkey = w.cmkey; a.E = w.E; a.ldp = n1_max + 1; a.err = w.err;
  a.idx0 = indices0; a.idx1 = indices1; a.max0 = w.max0; a.max1 = w.max1;
  a.rpc_max = p.rpc; a.slab_ld = p.slab_ld; a.slab_rows = p.slab_rows; a.only_if_redo = 0; a.ring = 0; a.rb = 0;
  // the attribute is per function, not per launch: always the full budget, so that concurrent callers with different
  // problem sizes cannot lower it under one another's launch (found by test_concurrent_callers_match_sequential)
  GIMS_CUDA_OK(cudaFuncSetAttribute(k_sinkhorn_reg, cudaFuncAttributeMaxDynamicSharedMemorySize, budget));
  GIMS_CUDA_OK(cudaFuncSetAttribute(k_sinkhorn_exact, cudaFuncAttributeMaxDynamicSharedMemorySize, budget));
  GIMS_CUDA_OK(cudaMemsetAsync(w.err, 0, w.zero_bytes, st));    // clears err and every flag / tag word (contiguous)
  void* params[] = {&a};
  {
    CoopChainScope chain(st, grid.half);
    GIMS_TRY(chain.rc);
    ProfScope prof(GIMS_PROF_SINKHORN, st);
    if (p.kind == kSinkReg) {
      GIMS_CUDA_OK(cudaLaunchCooperativeKernel((const void*)k_sinkhorn_reg, dim3(G), dim3(kThreads), params, p.dyn_smem, st));
      count_launch();
    } else if (p.kind == kSinkStream) {
      a.ring = p.rc; a.rb = p.rb;
      int rc = p.kg == 3 ? launch_stream<3, 2, true>(a, G, p.dyn_smem, budget, st)
             : p.kg == 5 ? launch_stream<5, 2, true>(a, G, p.dyn_smem, budget, st)
                         : launch_stream<9, 2, false>(a, G, p.dyn_smem, budget, st);
      GIMS_TRY(rc);
      count_launch();
    }
    // the exact kernel: the whole job if no scaled-kernel kernel applies, otherwise a no-op unless that launch
    // reported sums outside the fp32 range
    a.only_if_redo = (p.kind != kSinkExact) ? 1 : 0;
    a.slab_rows = p.exact_slab_rows;
    GIMS_CUDA_OK(cudaLaunchCooperativeKernel((const void*)k_sinkhorn_exact, dim3(G), dim3(kThreads), params, p.dyn_exact, st));
    count_launch();
  }
  int m = n0_max > n1_max ? n0_max : n1_max;
  k_match_finalize<<<cdiv(m, 256), 256, 0, st>>>(n0_max, n1_max, n_dev, indices0, indices1, w.max0, match_threshold,
                                                 matches0, matches1, mscores0, mscores1, w.err, status_dev);
  GIMS_LAUNCH_OK();
  return GIMS_OK;
}

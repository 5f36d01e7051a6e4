// Adaptive graph construction on the GPU (SURVEY.md §8 a-1 .. a-7).
//
// Replaces /root/reference/models/agc.py:682-709 `build_optimize_graph_with_cosine_similarity`
// (cosine matrix 382-391, percentile threshold 367-380, radius+similarity graph 413-449,
// connect_isolated_nodes 476-495, remove_small_components 497-516, fast_connect_components 518-565,
// relabel + dgl.from_networkx 699-708) and the repack of models/gmatcher.py:244-252.
//
// Numeric contract C1..C8 (oracle/gims_oracle.py header): fp64-accumulated cosine rounded to fp32,
// exact k-th order statistic, inclusive fp64 radius test, lowest-index tie-breaks, CSR rows ascending.
// Everything stays on the device; data-dependent counts (N', E, #components) are device scalars.
#include <float.h>

#include "common.cuh"

namespace gims {

namespace {

constexpr int kSelBins = 2048;

struct SelState {
  unsigned prefix;
  unsigned pad;
  unsigned long long rank;
};

struct AgcWs {
  // zero-initialised block (one memset)
  unsigned* hist;          // [kSelBins]
  int* extra_cnt;          // [n]
  int* comp_size;          // [n]
  double* csum;            // [n][2] centroid sums
  int* iso_count;          // [1]
  int* comp_edge_valid;    // [n]
  int* scalars;            // [8]: 0 = n_base_edges
  size_t zero_bytes;
  char* zero_base;
  // plain scratch
  SelState* sel;
  float* xhat;             // [n][256]
  float* feat;             // [n][256] node-major input descriptors
  float* S;                // [n][n]
  int* deg_base;           // [n]
  int* indptr_base;        // [n+1]
  int* idx_base;           // [edge_cap]
  int* nn_iso;             // [n]
  int* iso_u;              // [n]
  int* iso_v;              // [n]
  int* parent;             // [n]
  int* new_id;             // [n]
  int* comp_of_root;       // [n]
  int* comp_root;          // [n]
  float* cent;             // [n][2]
  int* comp_nn;            // [n]
  int* comp_eu;            // [n]
  int* comp_ev;            // [n]
  int* fdeg;               // [n]
};

size_t carve(AgcWs& w, void* base, size_t cap, int n, int edge_cap) {
  Arena a(base, cap);
  w.zero_base = a.take<char>(0);
  w.hist = a.take<unsigned>(kSelBins);
  w.extra_cnt = a.take<int>(n);
  w.comp_size = a.take<int>(n);
  w.csum = a.take<double>(2 * (size_t)n);
  w.iso_count = a.take<int>(1);
  w.comp_edge_valid = a.take<int>(n);
  w.scalars = a.take<int>(8);
  size_t zend = align_up(a.off, 256);
  w.zero_bytes = zend - (size_t)(w.zero_base - (char*)base);
  w.sel = a.take<SelState>(1);
  w.xhat = a.take<float>((size_t)n * kD);
  w.feat = a.take<float>((size_t)n * kD);
  w.S = a.take<float>((size_t)n * n);
  w.deg_base = a.take<int>(n);
  w.indptr_base = a.take<int>(n + 1);
  w.idx_base = a.take<int>(edge_cap);
  w.nn_iso = a.take<int>(n);
  w.iso_u = a.take<int>(n);
  w.iso_v = a.take<int>(n);
  w.parent = a.take<int>(n);
  w.new_id = a.take<int>(n);
  w.comp_of_root = a.take<int>(n);
  w.comp_root = a.take<int>(n);
  w.cent = a.take<float>(2 * (size_t)n);
  w.comp_nn = a.take<int>(n);
  w.comp_eu = a.take<int>(n);
  w.comp_ev = a.take<int>(n);
  w.fdeg = a.take<int>(n);
  return align_up(a.off, 256);
}

// ---------------------------------------------------------------------------------------------
// a-1  descriptors: (D,N) -> (N,D), C1 row normalisation
// ---------------------------------------------------------------------------------------------
__global__ void k_transpose_dn(const float* __restrict__ src, int n, float* __restrict__ dst) {
  __shared__ float tile[32][33];
  int n0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  for (int r = threadIdx.y; r < 32; r += blockDim.y) {
    int c = c0 + r, i = n0 + threadIdx.x;
    tile[r][threadIdx.x] = (i < n) ? src[(size_t)c * n + i] : 0.f;
  }
  __syncthreads();
  for (int r = threadIdx.y; r < 32; r += blockDim.y) {
    int i = n0 + r, c = c0 + threadIdx.x;
    if (i < n) dst[(size_t)i * kD + c] = tile[threadIdx.x][r];
  }
}

__global__ void k_normalize_rows(const float* __restrict__ feat, int n, float* __restrict__ xhat) {
  int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  int lane = threadIdx.x & 31;
  if (row >= n) return;
  const float4* p = reinterpret_cast<const float4*>(feat + (size_t)row * kD);
  float4 a = p[lane], b = p[lane + 32];
  double s = (double)a.x * a.x + (double)a.y * a.y + (double)a.z * a.z + (double)a.w * a.w +
             (double)b.x * b.x + (double)b.y * b.y + (double)b.z * b.z + (double)b.w * b.w;
#pragma unroll
  for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  float nrm = (float)sqrt(s);
  float den = fmaxf(nrm, 1e-12f);
  float4 oa = make_float4(a.x / den, a.y / den, a.z / den, a.w / den);
  float4 ob = make_float4(b.x / den, b.y / den, b.z / den, b.w / den);
  float4* q = reinterpret_cast<float4*>(xhat + (size_t)row * kD);
  q[lane] = oa;
  q[lane + 32] = ob;
}

// ---------------------------------------------------------------------------------------------
// a-1  C2: S = fl32(Xhat Xhat^T accumulated in fp64), upper-triangular 64x64 tiles mirrored
// ---------------------------------------------------------------------------------------------
constexpr int kCT = 128;  // tile edge
constexpr int kCK = 16;   // k-slab
constexpr int kCLd = kCT + 4;   // row pitch of the k-major slabs in doubles: 132 = 4 (mod 16) makes the fragment loads
                                // (4 k values x 8 rows per half-warp) conflict-free

// D (8x8) += A (8x4, row) * B (4x8, col) in fp64 on the tensor core (DMMA).  Lane l holds A[l>>2][l&3], B[l&3][l>>2] and
// D[l>>2][2*(l&3) .. +1].
__device__ __forceinline__ void dmma_8x8x4(double& d0, double& d1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0, %1}, {%2}, {%3}, {%0, %1};"
               : "+d"(d0), "+d"(d1)
               : "d"(a), "d"(b));
}

// One CTA = one 128 x 128 tile of the upper triangle, 8 warps, warp w owns rows 32 (w & 3) .. +32 and columns
// 64 (w >> 2) .. +64 as 4 x 8 DMMA tiles (64 fp64 accumulators per thread).  Per k-step of 4: 12 fragment loads for 32 DMMAs
// — the scalar version (8 x 8 DFMA per thread, 16 loads per 64 DFMA) issued 8 x as many instructions for the same FMAs and
// ran at 47 % of the fp64 pipe with its two warps per scheduler (ncu: no eligible warp 60 % of the cycles).
__global__ void __launch_bounds__(256) k_cosine_fp64(const float* __restrict__ xhat, int n, float* __restrict__ S) {
  int bi = blockIdx.y, bj = blockIdx.x;
  if (bj < bi) return;
  __shared__ double As[kCK][kCLd];
  __shared__ double Bs[kCK][kCLd];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int wr = 32 * (warp & 3), wc = 64 * (warp >> 2);      // this warp's corner inside the tile
  const int fr = lane >> 2, fk = lane & 3;                    // fragment row / column index, k index
  double acc[4][8][2];
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int b = 0; b < 8; ++b) acc[a][b][0] = acc[a][b][1] = 0.0;
  const int i0 = bi * kCT, j0 = bj * kCT;
  // loader mapping: 256 threads load 128 rows x 16 k per operand: two float4 each (rows tid/4 and tid/4 + 64, k4 = tid%4)
  const int lr = tid >> 2, lk = (tid & 3) * 4;
  float4 va[2], vb[2];
  auto fetch = [&](int k0) {
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      va[h] = make_float4(0.f, 0.f, 0.f, 0.f); vb[h] = va[h];
      int r = lr + 64 * h;
      if (i0 + r < n) va[h] = *reinterpret_cast<const float4*>(xhat + (size_t)(i0 + r) * kD + k0 + lk);
      if (j0 + r < n) vb[h] = *reinterpret_cast<const float4*>(xhat + (size_t)(j0 + r) * kD + k0 + lk);
    }
  };
  fetch(0);
  for (int k0 = 0; k0 < kD; k0 += kCK) {
    __syncthreads();
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      int r = lr + 64 * h;
      As[lk + 0][r] = va[h].x; As[lk + 1][r] = va[h].y; As[lk + 2][r] = va[h].z; As[lk + 3][r] = va[h].w;
      Bs[lk + 0][r] = vb[h].x; Bs[lk + 1][r] = vb[h].y; Bs[lk + 2][r] = vb[h].z; Bs[lk + 3][r] = vb[h].w;
    }
    __syncthreads();
    if (k0 + kCK < kD) fetch(k0 + kCK);      // the next slab's global loads fly during this slab's MMAs
#pragma unroll
    for (int kk = 0; kk < kCK; kk += 4) {    // k ascending
      double a[4], b[8];
#pragma unroll
      for (int q = 0; q < 4; ++q) a[q] = As[kk + fk][wr + 8 * q + fr];
#pragma unroll
      for (int q = 0; q < 8; ++q) b[q] = Bs[kk + fk][wc + 8 * q + fr];
#pragma unroll
      for (int q = 0; q < 4; ++q)
#pragma unroll
        for (int r = 0; r < 8; ++r) dmma_8x8x4(acc[q][r][0], acc[q][r][1], a[q], b[r]);
    }
  }
  // lane l holds rows fr, column pairs 2 fk, 2 fk + 1 of every 8 x 8 tile: 8-byte stores, the mirror image as scalars
#pragma unroll
  for (int q = 0; q < 4; ++q)
#pragma unroll
    for (int r = 0; r < 8; ++r) {
      const int i = i0 + wr + 8 * q + fr, j = j0 + wc + 8 * r + 2 * fk;
      if (i >= n) continue;
      const float v0 = (float)acc[q][r][0], v1 = (float)acc[q][r][1];
      if (j < n) { S[(size_t)i * n + j] = v0; if (bi != bj) S[(size_t)j * n + i] = v0; }
      if (j + 1 < n) { S[(size_t)i * n + j + 1] = v1; if (bi != bj) S[(size_t)(j + 1) * n + i] = v1; }
    }
}

// ---------------------------------------------------------------------------------------------
// a-1  C3: exact k-th smallest of the strict upper triangle — 3-pass radix select (11+11+10 bits)
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned f2key(float f) {
  unsigned u = __float_as_uint(f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float key2f(unsigned k) {
  unsigned u = (k & 0x80000000u) ? (k & 0x7fffffffu) : ~k;
  return __uint_as_float(u);
}

__global__ void k_sel_init(SelState* st, unsigned long long rank) {
  st->prefix = 0; st->pad = 0; st->rank = rank;
}

__global__ void __launch_bounds__(256) k_sel_hist(const float* __restrict__ S, int n, int pass,
                                                  const SelState* __restrict__ st, unsigned* __restrict__ hist) {
  __shared__ unsigned sh[kSelBins];
  for (int b = threadIdx.x; b < kSelBins; b += blockDim.x) sh[b] = 0;
  __syncthreads();
  unsigned prefix = st->prefix;
  for (int i = blockIdx.x; i < n - 1; i += gridDim.x) {
    const float* row = S + (size_t)i * n;
    for (int j = i + 1 + threadIdx.x; j < n; j += blockDim.x) {
      unsigned key = f2key(row[j]);
      if (pass == 0) {
        atomicAdd(&sh[key >> 21], 1u);
      } else if (pass == 1) {
        if ((key >> 21) == prefix) atomicAdd(&sh[(key >> 10) & 0x7ffu], 1u);
      } else {
        if ((key >> 10) == prefix) atomicAdd(&sh[key & 0x3ffu], 1u);
      }
    }
  }
  __syncthreads();
  for (int b = threadIdx.x; b < kSelBins; b += blockDim.x)
    if (sh[b]) atomicAdd(&hist[b], sh[b]);
}

// one block of 1024 threads, 2 bins per thread
__global__ void __launch_bounds__(1024) k_sel_scan(SelState* st, unsigned* hist, int pass, float* thr_out) {
  __shared__ unsigned long long warp_tot[32];
  int t = threadIdx.x;
  unsigned c0 = hist[2 * t], c1 = hist[2 * t + 1];
  unsigned long long mine = (unsigned long long)c0 + c1;
  unsigned long long incl = mine;
  int lane = t & 31, wid = t >> 5;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    unsigned long long v = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += v;
  }
  if (lane == 31) warp_tot[wid] = incl;
  __syncthreads();
  if (wid == 0) {
    unsigned long long v = warp_tot[lane];
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      unsigned long long x = __shfl_up_sync(0xffffffffu, v, o);
      if (lane >= o) v += x;
    }
    warp_tot[lane] = v;   // inclusive over warps
  }
  __syncthreads();
  unsigned long long excl = incl - mine + (wid ? warp_tot[wid - 1] : 0ull);
  unsigned long long rank = st->rank;
  unsigned prefix = st->prefix;
  __syncthreads();
  hist[2 * t] = 0; hist[2 * t + 1] = 0;   // ready for the next pass
  if (rank >= excl && rank < excl + mine) {
    unsigned digit; unsigned long long before;
    if (rank < excl + c0) { digit = 2 * t; before = excl; } else { digit = 2 * t + 1; before = excl + c0; }
    unsigned np = (pass == 2) ? ((prefix << 10) | digit) : ((prefix << 11) | digit);
    st->prefix = np;
    st->rank = rank - before;
    if (pass == 2) *thr_out = key2f(np);
  }
}

// ---------------------------------------------------------------------------------------------
// a-2  base graph: radius (C4) AND similarity >= thr, warp per row, ascending neighbours
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ double sqdist64(float2 a, float2 b) {
  double dx = (double)a.x - (double)b.x, dy = (double)a.y - (double)b.y;
  return __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy));
}

// One warp per row i; the keypoints of the candidate columns are staged through shared memory in chunks of 2048 — with
// kpts[j] read from L2 inside the ballot loop every iteration paid a dependent global round trip (23 us per pass).
constexpr int kEdgeChunk = 2048;

template <bool FILL>
__global__ void __launch_bounds__(256) k_base_edges(const float2* __restrict__ kpts, const float* __restrict__ S, int n,
                                                    double r2, const float* __restrict__ thr_p, int* __restrict__ deg,
                                                    const int* __restrict__ indptr, int* __restrict__ idx, int edge_cap,
                                                    unsigned* status) {
  __shared__ float2 kp_s[kEdgeChunk];
  const int i = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  const bool live = i < n;
  const float thr = *thr_p;
  const float2 pi = live ? kpts[i] : make_float2(0.f, 0.f);
  const float* srow = S + (size_t)(live ? i : 0) * n;
  int cnt = 0;
  const int base = (FILL && live) ? indptr[i] : 0;
  for (int c0 = 0; c0 < n; c0 += kEdgeChunk) {
    const int cn = min(kEdgeChunk, n - c0);
    __syncthreads();
    for (int j = threadIdx.x; j < cn; j += blockDim.x) kp_s[j] = kpts[c0 + j];
    __syncthreads();
    if (!live) continue;
    for (int j0 = 0; j0 < cn; j0 += 32) {
      const int jl = j0 + lane, j = c0 + jl;
      bool p = false;
      if (jl < cn && j != i) {
        if (sqdist64(pi, kp_s[jl]) <= r2) p = srow[j] >= thr;
      }
      const unsigned m = __ballot_sync(0xffffffffu, p);
      if (FILL && p) {
        const int pos = base + cnt + __popc(m & ((1u << lane) - 1u));
        if (pos < edge_cap) idx[pos] = j; else atomicOr(status, GIMS_STATUS_EDGE_OVERFLOW);
      }
      cnt += __popc(m);
    }
  }
  if (!FILL && live && lane == 0) deg[i] = cnt;
}

// exclusive scan of `in[0..n)` into out[0..n], out[n] = total; n = n_dev ? *n_dev : n_max. One block.
__global__ void __launch_bounds__(1024) k_excl_scan(const int* __restrict__ in, int* __restrict__ out, int n_max,
                                                    const int* __restrict__ n_dev, int* total_out) {
  __shared__ int warp_tot[32];
  __shared__ int carry_s;
  int n = n_dev ? min(*n_dev, n_max) : n_max;
  int t = threadIdx.x, lane = t & 31, wid = t >> 5;
  if (t == 0) carry_s = 0;
  __syncthreads();
  for (int b0 = 0; b0 < n; b0 += 1024) {
    int i = b0 + t;
    int v = (i < n) ? in[i] : 0;
    int incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      int x = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += x;
    }
    if (lane == 31) warp_tot[wid] = incl;
    __syncthreads();
    if (wid == 0) {
      int w = warp_tot[lane];
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        int x = __shfl_up_sync(0xffffffffu, w, o);
        if (lane >= o) w += x;
      }
      warp_tot[lane] = w;
    }
    __syncthreads();
    int carry = carry_s;
    int excl = carry + incl - v + (wid ? warp_tot[wid - 1] : 0);
    if (i < n) out[i] = excl;
    __syncthreads();
    if (t == 1023) carry_s = carry + warp_tot[31];
    __syncthreads();
  }
  if (t == 0) {
    out[n] = carry_s;
    if (total_out) *total_out = carry_s;
  }
}

// ---------------------------------------------------------------------------------------------
// a-3  connect_isolated_nodes (agc.py:476-495): nearest neighbour of degree-0 nodes (C5), then the
//      sequential "degree at that moment" rule resolved in ascending node order.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_iso_nn(const float2* __restrict__ kpts, int n, const int* __restrict__ deg,
                                                const int* __restrict__ n_base_edges, int* __restrict__ nn) {
  int i = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  int lane = threadIdx.x & 31;
  if (i >= n) return;
  if (*n_base_edges == 0 || deg[i] != 0) return;
  float2 pi = kpts[i];
  double best = DBL_MAX;
  int bj = 0x7fffffff;
  for (int j = lane; j < n; j += 32) {
    if (j == i) continue;
    double d = sqdist64(pi, kpts[j]);
    if (d < best) { best = d; bj = j; }   // ascending j per lane: strict < keeps the lowest index
  }
#pragma unroll
  for (int o = 16; o; o >>= 1) {
    double od = __shfl_xor_sync(0xffffffffu, best, o);
    int oj = __shfl_xor_sync(0xffffffffu, bj, o);
    if (od < best || (od == best && oj < bj)) { best = od; bj = oj; }
  }
  if (lane == 0) nn[i] = bj;
}

// One block.  Pass 1: ordered compaction of the isolated nodes; pass 2 (warp 0): sequential rule.
__global__ void __launch_bounds__(1024) k_iso_resolve(int n, const int* __restrict__ deg, const int* __restrict__ n_base_edges,
                                                      const int* __restrict__ nn, int* __restrict__ iso_u, int* __restrict__ iso_v,
                                                      int* __restrict__ iso_count, int* __restrict__ extra_cnt) {
  __shared__ unsigned hit[GIMS_MAX_KPTS / 32];   // one bit per node (8 KB at 65536 nodes)
  __shared__ int warp_tot[32];
  __shared__ int carry_s;
  if (*n_base_edges == 0) return;   // agc.py:487: graphs without edges are returned untouched
  int t = threadIdx.x, lane = t & 31, wid = t >> 5;
  for (int i = t; i < (n + 31) / 32; i += 1024) hit[i] = 0u;
  if (t == 0) carry_s = 0;
  __syncthreads();
  // compaction: iso_u[k] = k-th isolated node (ascending), iso_v[k] = its nearest neighbour (tentative)
  for (int b0 = 0; b0 < n; b0 += 1024) {
    int i = b0 + t;
    bool p = (i < n) && deg[i] == 0;
    unsigned m = __ballot_sync(0xffffffffu, p);
    if (lane == 0) warp_tot[wid] = __popc(m);
    __syncthreads();
    int before = carry_s;
    for (int w = 0; w < wid; ++w) before += warp_tot[w];
    if (p) {
      int k = before + __popc(m & ((1u << lane) - 1u));
      iso_u[k] = i;
      iso_v[k] = nn[i];
    }
    __syncthreads();
    if (t == 0) {
      int tot = 0;
      for (int w = 0; w < 32; ++w) tot += warp_tot[w];
      carry_s += tot;
    }
    __syncthreads();
  }
  int cnt = carry_s;
  if (wid != 0) return;
  // sequential resolution, 32 candidates per step; survivors are re-packed in place
  int out = 0;
  for (int k0 = 0; k0 < cnt; k0 += 32) {
    int k = k0 + lane;
    int u = (k < cnt) ? iso_u[k] : -1;
    int v = (k < cnt) ? iso_v[k] : -1;
    __syncwarp();
    unsigned active = 0;
    int m = min(32, cnt - k0);
    for (int s = 0; s < m; ++s) {
      int su = __shfl_sync(0xffffffffu, u, s);
      int sv = __shfl_sync(0xffffffffu, v, s);
      const unsigned h = (hit[su >> 5] >> (su & 31)) & 1u;   // all lanes read the same word
      if (!h) {
        active |= 1u << s;
        if (lane == 0) { hit[sv >> 5] |= 1u << (sv & 31); hit[su >> 5] |= 1u << (su & 31); }
      }
      __syncwarp();
    }
    bool mine = (active >> lane) & 1u;
    int pos = out + __popc(active & ((1u << lane) - 1u));
    if (mine) {
      iso_u[pos] = u;                       // pos <= k: in-place compaction is safe (reads done above)
      iso_v[pos] = v;
      atomicAdd(&extra_cnt[u], 1);
      atomicAdd(&extra_cnt[v], 1);
    }
    out += __popc(active);
    __syncwarp();
  }
  if (lane == 0) *iso_count = out;
}

// ---------------------------------------------------------------------------------------------
// a-4  connected components: lock-free union-find, smaller root wins (root == smallest member id)
// ---------------------------------------------------------------------------------------------
// The whole component search in ONE CTA with the parent array in SHARED memory: a find is a chain of dependent loads, and
// through L2 (volatile, ~500 clk per hop) the grid-wide version took 40-86 us for 15 k edges however the unions were
// distributed; in shared memory a hop is ~30 clk.  Init, base-graph unions, isolated-node unions and the final labelling
// are one launch instead of four.  Parents are `int` up to 16384 nodes (64 KB) and `unsigned short` above: every node id
// is below GIMS_MAX_KPTS = 65536, so 16 bits hold it and 65536 nodes take 128 KB (16-bit atomicCAS exists since sm_70).
//   init: every node points at its smallest neighbour if that is smaller than itself (CSR rows are ascending, so it is the
//   first entry) — pointers only ever go to strictly smaller ids along real edges, a forest with the same components;
//   union: lock-free, smaller root wins (root == smallest member id whatever the order of the unions), so the labels do
//   not depend on the parent type or on the order of the unions.
constexpr int kCcIntMaxNodes = 16384;
static_assert(GIMS_MAX_KPTS <= 65536, "16-bit union-find parents need node ids below 65536");
template <typename P>
__device__ __forceinline__ int ufs_find(volatile P* p, int x) {
  int cur = x, par = p[cur];
  while (par != cur) {
    const int gp = p[par];
    if (gp != par) p[cur] = (P)gp;   // path halving; only ever rewires non-roots to an ancestor
    cur = par;
    par = gp;
  }
  return cur;
}
template <typename P>
__device__ __forceinline__ void ufs_union(P* parent, int a, int b) {
  while (true) {
    a = ufs_find<P>(parent, a);
    b = ufs_find<P>(parent, b);
    if (a == b) return;
    if (a > b) { const int t = a; a = b; b = t; }
    if ((int)atomicCAS(&parent[b], (P)b, (P)a) == b) return;
  }
}
template <typename P>
__global__ void __launch_bounds__(1024) k_cc_components(int* __restrict__ parent_out, int n, const int* __restrict__ indptr,
                                                        const int* __restrict__ idx, int edge_cap, const int* __restrict__ iso_u,
                                                        const int* __restrict__ iso_v, const int* __restrict__ iso_count) {
  extern __shared__ __align__(16) unsigned char sp_raw[];
  P* sp = reinterpret_cast<P*>(sp_raw);
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const int e0 = indptr[i];
    sp[i] = (P)((e0 < indptr[i + 1] && e0 < edge_cap) ? min(i, idx[e0]) : i);
  }
  __syncthreads();
  // a thread per node (each undirected edge once, from its smaller end): with ~7 edges per node a warp per node leaves
  // nine lanes in ten idle, and the unions of a node are short now that a hop costs a shared-memory access
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const int e0 = indptr[i], e1 = min(indptr[i + 1], edge_cap);
    for (int e = e0; e < e1; ++e) {
      const int j = idx[e];
      if (j > i) ufs_union<P>(sp, i, j);
    }
  }
  const int n_iso = *iso_count;
  for (int k = threadIdx.x; k < n_iso; k += blockDim.x) ufs_union<P>(sp, iso_u[k], iso_v[k]);
  __syncthreads();
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    int r = i;
    while ((int)sp[r] != r) r = sp[r];
    parent_out[i] = r;
  }
}

// The attribute belongs to the function, not to one launch: it is always the most the instantiation can need, so that
// concurrent callers with different node counts cannot lower it under one another's launch.
template <typename P>
int launch_cc_components(const AgcWs& w, int n, int edge_cap, cudaStream_t st) {
  constexpr int kMaxSmem = (sizeof(P) == sizeof(int) ? kCcIntMaxNodes : GIMS_MAX_KPTS) * (int)sizeof(P);
  const size_t smem = (size_t)n * sizeof(P);
  GIMS_CUDA_OK(cudaFuncSetAttribute(k_cc_components<P>, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxSmem));
  k_cc_components<P><<<1, 1024, smem, st>>>(w.parent, n, w.indptr_base, w.idx_base, edge_cap, w.iso_u, w.iso_v, w.iso_count);
  GIMS_LAUNCH_OK();
  return GIMS_OK;
}

__global__ void k_cc_count(const int* __restrict__ label, int n, int* comp_size) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) atomicAdd(&comp_size[label[i]], 1);
}

// a-4 keep mask + ordered compaction (kept ids ascending, agc.py:677) + component numbering in
// ascending-root order (networkx connected_components order).  One block.
__global__ void __launch_bounds__(1024) k_keep_compact(int n, const int* __restrict__ label, const int* __restrict__ comp_size,
                                                       int min_size, int* __restrict__ new_id, int* __restrict__ kept_idx,
                                                       int* __restrict__ comp_of_root, int* __restrict__ comp_root,
                                                       int* n_kept_out, int* n_comp_out) {
  __shared__ int wk[32], wc[32];
  __shared__ int carry_k, carry_c;
  int t = threadIdx.x, lane = t & 31, wid = t >> 5;
  if (t == 0) { carry_k = 0; carry_c = 0; }
  __syncthreads();
  for (int b0 = 0; b0 < n; b0 += 1024) {
    int i = b0 + t;
    bool keep = false, root = false;
    if (i < n) {
      int r = label[i];
      keep = comp_size[r] >= min_size;
      root = keep && (r == i);
    }
    unsigned mk = __ballot_sync(0xffffffffu, keep), mc = __ballot_sync(0xffffffffu, root);
    if (lane == 0) { wk[wid] = __popc(mk); wc[wid] = __popc(mc); }
    __syncthreads();
    int bk = carry_k, bc = carry_c;
    for (int w = 0; w < wid; ++w) { bk += wk[w]; bc += wc[w]; }
    unsigned lt = (1u << lane) - 1u;
    if (i < n) {
      if (keep) {
        int id = bk + __popc(mk & lt);
        new_id[i] = id;
        kept_idx[id] = i;
      } else {
        new_id[i] = -1;
      }
      if (root) {
        int c = bc + __popc(mc & lt);
        comp_of_root[i] = c;
        comp_root[c] = i;
      }
    }
    __syncthreads();
    if (t == 0) {
      int a = 0, b = 0;
      for (int w = 0; w < 32; ++w) { a += wk[w]; b += wc[w]; }
      carry_k += a; carry_c += b;
    }
    __syncthreads();
  }
  if (t == 0) { *n_kept_out = carry_k; *n_comp_out = carry_c; }
}

// ---------------------------------------------------------------------------------------------
// a-5  fast_connect_components (agc.py:518-565), one round
// ---------------------------------------------------------------------------------------------
__global__ void k_centroid_acc(const float2* __restrict__ kpts, int n, const int* __restrict__ label,
                               const int* __restrict__ new_id, const int* __restrict__ comp_of_root,
                               const int* __restrict__ n_comp, double* __restrict__ csum) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n || *n_comp <= 1 || new_id[i] < 0) return;
  int c = comp_of_root[label[i]];
  float2 p = kpts[i];
  atomicAdd(&csum[2 * c], (double)p.x);
  atomicAdd(&csum[2 * c + 1], (double)p.y);
}

__global__ void k_centroid_fin(const double* __restrict__ csum, const int* __restrict__ comp_root,
                               const int* __restrict__ comp_size, const int* __restrict__ n_comp, float* __restrict__ cent) {
  int c = blockIdx.x * blockDim.x + threadIdx.x;
  int nc = *n_comp;
  if (nc <= 1 || c >= nc) return;
  double cnt = (double)comp_size[comp_root[c]];
  cent[2 * c] = (float)(csum[2 * c] / cnt);          // C6
  cent[2 * c + 1] = (float)(csum[2 * c + 1] / cnt);
}

__global__ void __launch_bounds__(256) k_comp_nn(const float2* __restrict__ cent, const int* __restrict__ n_comp, int* __restrict__ cnn) {
  int c = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  int lane = threadIdx.x & 31;
  int nc = *n_comp;
  if (nc <= 1 || c >= nc) return;
  float2 pc = cent[c];
  double best = DBL_MAX;
  int bj = 0x7fffffff;
  for (int j = lane; j < nc; j += 32) {
    if (j == c) continue;
    double d = sqdist64(pc, cent[j]);
    if (d < best) { best = d; bj = j; }
  }
#pragma unroll
  for (int o = 16; o; o >>= 1) {
    double od = __shfl_xor_sync(0xffffffffu, best, o);
    int oj = __shfl_xor_sync(0xffffffffu, bj, o);
    if (od < best || (od == best && oj < bj)) { best = od; bj = oj; }
  }
  if (lane == 0) cnn[c] = bj;
}

constexpr int kPairChunk = 2048;

// block per component c: closest pair (u in c, v in nn(c)) by (d2, v, u) — C7.
// The smaller of the two components is staged in shared memory, the threads scan the larger one.
__global__ void __launch_bounds__(256) k_comp_pair(const float2* __restrict__ kpts, int n, const int* __restrict__ label,
                                                   const int* __restrict__ new_id, const int* __restrict__ comp_of_root,
                                                   const int* __restrict__ comp_root, const int* __restrict__ comp_size,
                                                   const int* __restrict__ n_comp, const int* __restrict__ cnn,
                                                   int* __restrict__ eu, int* __restrict__ ev, int* __restrict__ evalid,
                                                   int* __restrict__ extra_cnt) {
  __shared__ int mem_id[kPairChunk];
  __shared__ float2 mem_p[kPairChunk];
  __shared__ int mem_cnt;
  __shared__ double rd[256];
  __shared__ int rv[256], ru[256];
  int nc = *n_comp;
  if (nc <= 1) return;
  for (int c = blockIdx.x; c < nc; c += gridDim.x) {
    int j = cnn[c];
    if (j < c && cnn[j] == c) continue;      // (j,c) was connected when j was visited (agc.py:550-552)
    const bool c_small = comp_size[comp_root[c]] <= comp_size[comp_root[j]];
    const int cs = c_small ? c : j;          // staged in shared memory
    const int cl = c_small ? j : c;          // scanned by the threads
    double best = DBL_MAX;
    int bv = 0x7fffffff, bu = 0x7fffffff;
    for (int s0 = 0; s0 < n; s0 += kPairChunk) {
      __syncthreads();
      if (threadIdx.x == 0) mem_cnt = 0;
      __syncthreads();
      for (int i = s0 + threadIdx.x; i < min(n, s0 + kPairChunk); i += blockDim.x) {
        if (new_id[i] >= 0 && comp_of_root[label[i]] == cs) {
          int k = atomicAdd(&mem_cnt, 1);
          mem_id[k] = i;
          mem_p[k] = kpts[i];
        }
      }
      __syncthreads();
      int mc = mem_cnt;
      if (mc == 0) continue;
      for (int x = threadIdx.x; x < n; x += blockDim.x) {
        if (new_id[x] < 0 || comp_of_root[label[x]] != cl) continue;
        float2 px = kpts[x];
        for (int k = 0; k < mc; ++k) {
          double d = sqdist64(px, mem_p[k]);
          int u = c_small ? mem_id[k] : x;   // u in component c, v in component j
          int v = c_small ? x : mem_id[k];
          if (d < best || (d == best && (v < bv || (v == bv && u < bu)))) { best = d; bv = v; bu = u; }
        }
      }
    }
    rd[threadIdx.x] = best; rv[threadIdx.x] = bv; ru[threadIdx.x] = bu;
    __syncthreads();
    for (int o = 128; o; o >>= 1) {
      if (threadIdx.x < o) {
        double od = rd[threadIdx.x + o]; int ov = rv[threadIdx.x + o], ou = ru[threadIdx.x + o];
        double md = rd[threadIdx.x]; int mv = rv[threadIdx.x], mu = ru[threadIdx.x];
        if (od < md || (od == md && (ov < mv || (ov == mv && ou < mu)))) {
          rd[threadIdx.x] = od; rv[threadIdx.x] = ov; ru[threadIdx.x] = ou;
        }
      }
      __syncthreads();
    }
    if (threadIdx.x == 0 && rv[0] != 0x7fffffff) {
      eu[c] = ru[0]; ev[c] = rv[0]; evalid[c] = 1;
      atomicAdd(&extra_cnt[ru[0]], 1);
      atomicAdd(&extra_cnt[rv[0]], 1);
    }
    __syncthreads();
  }
}

// ---------------------------------------------------------------------------------------------
// a-6 / a-7  final CSR over kept nodes (C8) and the repack of point/feat/score
// ---------------------------------------------------------------------------------------------
__global__ void k_final_deg(int n, const int* __restrict__ new_id, const int* __restrict__ deg_base,
                            const int* __restrict__ extra_cnt, int* __restrict__ fdeg) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  int id = new_id[i];
  if (id >= 0) fdeg[id] = deg_base[i] + extra_cnt[i];
}

__global__ void __launch_bounds__(256) k_final_fill(int n, const int* __restrict__ new_id, const int* __restrict__ indptr_base,
                                                    const int* __restrict__ idx_base, const int* __restrict__ iso_u,
                                                    const int* __restrict__ iso_v, const int* __restrict__ iso_count,
                                                    const int* __restrict__ eu, const int* __restrict__ ev,
                                                    const int* __restrict__ evalid, const int* __restrict__ n_comp,
                                                    const int* __restrict__ extra_cnt, const int* __restrict__ indptr,
                                                    int* __restrict__ indices, int edge_cap, unsigned* status) {
  int i = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  int lane = threadIdx.x & 31;
  if (i >= n) return;
  int id = new_id[i];
  if (id < 0) return;
  int row = indptr[id];
  int b0 = indptr_base[i], nb = indptr_base[i + 1] - b0;
  int total = nb + extra_cnt[i];
  // the base CSR itself may have overflowed (entries past edge_cap were never written): never read or write past
  // either capacity; the status bit makes the host retry with a larger edge_cap
  if (row + total > edge_cap || b0 + nb > edge_cap) {
    if (lane == 0) atomicOr(status, GIMS_STATUS_EDGE_OVERFLOW);
    return;
  }
  for (int e = lane; e < nb; e += 32) indices[row + e] = new_id[idx_base[b0 + e]];
  int nx = extra_cnt[i];
  if (nx == 0) return;
  int pos = nb;
  int ic = *iso_count;
  for (int k0 = 0; k0 < ic; k0 += 32) {
    int k = k0 + lane;
    int other = -1;
    if (k < ic) {
      int u = iso_u[k], v = iso_v[k];
      if (u == i) other = v; else if (v == i) other = u;
    }
    unsigned m = __ballot_sync(0xffffffffu, other >= 0);
    if (other >= 0) indices[row + pos + __popc(m & ((1u << lane) - 1u))] = new_id[other];
    pos += __popc(m);
  }
  int nc = *n_comp;
  if (nc > 1) {
    for (int k0 = 0; k0 < nc; k0 += 32) {
      int k = k0 + lane;
      int other = -1;
      if (k < nc && evalid[k]) {
        int u = eu[k], v = ev[k];
        if (u == i) other = v; else if (v == i) other = u;
      }
      unsigned m = __ballot_sync(0xffffffffu, other >= 0);
      if (other >= 0) indices[row + pos + __popc(m & ((1u << lane) - 1u))] = new_id[other];
      pos += __popc(m);
    }
  }
  __syncwarp();
  if (lane == 0) {                       // insertion of the few extra neighbours into the ascending base part
    for (int e = nb; e < total; ++e) {
      int val = indices[row + e];
      int p = e - 1;
      while (p >= 0 && indices[row + p] > val) { indices[row + p + 1] = indices[row + p]; --p; }
      indices[row + p + 1] = val;
    }
  }
}

__global__ void __launch_bounds__(256) k_gather_kept(int n, const int* __restrict__ kept_idx, const int* __restrict__ n_kept,
                                                     const float2* __restrict__ kpts, const float* __restrict__ feat,
                                                     const float* __restrict__ scores, float2* __restrict__ kpts_out,
                                                     float* __restrict__ feat_out, float* __restrict__ scores_out) {
  int id = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  int lane = threadIdx.x & 31;
  if (id >= *n_kept) return;
  int i = kept_idx[id];
  const float4* s = reinterpret_cast<const float4*>(feat + (size_t)i * kD);
  float4* d = reinterpret_cast<float4*>(feat_out + (size_t)id * kD);
  d[lane] = s[lane];
  d[lane + 32] = s[lane + 32];
  if (lane == 0) {
    kpts_out[id] = kpts[i];
    scores_out[id] = scores[i];
  }
}

// Edge-capacity overflow: the CSR is incomplete (rows past the capacity were never written) while indptr / E hold the
// uncapped totals.  Report an EMPTY graph (N' = 0, E = 0) so that no later kernel — they all size themselves from
// N' in device memory — walks the unwritten part of `indices`; the status bit tells the host to retry.
__global__ void k_overflow_guard(const unsigned* __restrict__ status, int* n_kept, int* n_edges, int* n_comp, int* indptr) {
  if (*status & GIMS_STATUS_EDGE_OVERFLOW) { *n_kept = 0; *n_edges = 0; *n_comp = 0; indptr[0] = 0; }
}

}  // namespace

}  // namespace gims

using namespace gims;

extern "C" size_t gims_agc_workspace_bytes(int n, int edge_cap) {
  AgcWs w;
  return carve(w, nullptr, 0, n, edge_cap);
}

extern "C" int gims_agc_build(const float* kpts, const float* desc, int desc_channel_major, const float* scores, int n,
                              double radius, long long k_rank, int min_size, void* workspace, size_t workspace_bytes,
                              int* kept_idx, int* n_kept_dev, int* indptr, int* indices, int edge_cap, int* n_edges_dev,
                              float* kpts_out, float* feat_out, float* scores_out, float* thr_out, int* n_comp_dev,
                              unsigned* status_dev, void* stream) {
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (n < 2 || n > GIMS_MAX_KPTS) { set_error("gims_agc_build: n=%d outside [2, %d]", n, GIMS_MAX_KPTS); return GIMS_ERR_ARG; }
  if (edge_cap < 1 || k_rank < 0 || k_rank >= (long long)n * (n - 1) / 2) {
    set_error("gims_agc_build: bad edge_cap %d / k_rank %lld (need 0 <= k_rank < n(n-1)/2)", edge_cap, k_rank);
    return GIMS_ERR_ARG;
  }
  if (!kpts || !desc || !scores || !workspace || !kept_idx || !n_kept_dev || !indptr || !indices || !n_edges_dev ||
      !kpts_out || !feat_out || !scores_out || !thr_out || !n_comp_dev || !status_dev) {
    set_error("gims_agc_build: null pointer argument");
    return GIMS_ERR_ARG;
  }
  AgcWs w;
  size_t need = carve(w, workspace, workspace_bytes, n, edge_cap);
  if (need > workspace_bytes) { set_error("gims_agc_build: workspace %zu < %zu", workspace_bytes, need); return GIMS_ERR_WORKSPACE; }
  const float2* kp = reinterpret_cast<const float2*>(kpts);
  int* n_base_edges = w.scalars;
  GIMS_CUDA_OK(cudaMemsetAsync(w.zero_base, 0, w.zero_bytes, st));

  // a-1
  const float* feat = desc;
  if (desc_channel_major) {
    k_transpose_dn<<<dim3(cdiv(n, 32), kD / 32), dim3(32, 8), 0, st>>>(desc, n, w.feat);
    GIMS_LAUNCH_OK();
    feat = w.feat;
  }
  k_normalize_rows<<<cdiv(n, 8), 256, 0, st>>>(feat, n, w.xhat);
  GIMS_LAUNCH_OK();
  int T = cdiv(n, kCT);
  {
    ProfScope prof(GIMS_PROF_COSINE, st);
    k_cosine_fp64<<<dim3(T, T), 256, 0, st>>>(w.xhat, n, w.S);
  }
  GIMS_LAUNCH_OK();
  k_sel_init<<<1, 1, 0, st>>>(w.sel, (unsigned long long)k_rank);
  GIMS_LAUNCH_OK();
  for (int pass = 0; pass < 3; ++pass) {
    k_sel_hist<<<min(n - 1, 148 * 8), 256, 0, st>>>(w.S, n, pass, w.sel, w.hist);
    GIMS_LAUNCH_OK();
    k_sel_scan<<<1, 1024, 0, st>>>(w.sel, w.hist, pass, thr_out);
    GIMS_LAUNCH_OK();
  }
  // a-2
  double r2 = radius * radius;
  k_base_edges<false><<<cdiv(n, 8), 256, 0, st>>>(kp, w.S, n, r2, thr_out, w.deg_base, nullptr, nullptr, edge_cap, status_dev);
  GIMS_LAUNCH_OK();
  k_excl_scan<<<1, 1024, 0, st>>>(w.deg_base, w.indptr_base, n, nullptr, n_base_edges);
  GIMS_LAUNCH_OK();
  k_base_edges<true><<<cdiv(n, 8), 256, 0, st>>>(kp, w.S, n, r2, thr_out, nullptr, w.indptr_base, w.idx_base, edge_cap, status_dev);
  GIMS_LAUNCH_OK();
  // a-3
  k_iso_nn<<<cdiv(n, 8), 256, 0, st>>>(kp, n, w.deg_base, n_base_edges, w.nn_iso);
  GIMS_LAUNCH_OK();
  k_iso_resolve<<<1, 1024, 0, st>>>(n, w.deg_base, n_base_edges, w.nn_iso, w.iso_u, w.iso_v, w.iso_count, w.extra_cnt);
  GIMS_LAUNCH_OK();
  // a-4
  GIMS_TRY(n <= kCcIntMaxNodes ? launch_cc_components<int>(w, n, edge_cap, st)
                                : launch_cc_components<unsigned short>(w, n, edge_cap, st));
  k_cc_count<<<cdiv(n, 256), 256, 0, st>>>(w.parent, n, w.comp_size);
  GIMS_LAUNCH_OK();
  k_keep_compact<<<1, 1024, 0, st>>>(n, w.parent, w.comp_size, min_size, w.new_id, kept_idx, w.comp_of_root, w.comp_root,
                                     n_kept_dev, n_comp_dev);
  GIMS_LAUNCH_OK();
  // a-5
  k_centroid_acc<<<cdiv(n, 256), 256, 0, st>>>(kp, n, w.parent, w.new_id, w.comp_of_root, n_comp_dev, w.csum);
  GIMS_LAUNCH_OK();
  k_centroid_fin<<<cdiv(n, 256), 256, 0, st>>>(w.csum, w.comp_root, w.comp_size, n_comp_dev, w.cent);
  GIMS_LAUNCH_OK();
  k_comp_nn<<<cdiv(n, 8), 256, 0, st>>>(reinterpret_cast<const float2*>(w.cent), n_comp_dev, w.comp_nn);
  GIMS_LAUNCH_OK();
  k_comp_pair<<<min(n, 296), 256, 0, st>>>(kp, n, w.parent, w.new_id, w.comp_of_root, w.comp_root, w.comp_size, n_comp_dev,
                                           w.comp_nn, w.comp_eu,
                                           w.comp_ev, w.comp_edge_valid, w.extra_cnt);
  GIMS_LAUNCH_OK();
  // a-6
  k_final_deg<<<cdiv(n, 256), 256, 0, st>>>(n, w.new_id, w.deg_base, w.extra_cnt, w.fdeg);
  GIMS_LAUNCH_OK();
  k_excl_scan<<<1, 1024, 0, st>>>(w.fdeg, indptr, n, n_kept_dev, n_edges_dev);
  GIMS_LAUNCH_OK();
  k_final_fill<<<cdiv(n, 8), 256, 0, st>>>(n, w.new_id, w.indptr_base, w.idx_base, w.iso_u, w.iso_v, w.iso_count, w.comp_eu,
                                           w.comp_ev, w.comp_edge_valid, n_comp_dev, w.extra_cnt, indptr, indices, edge_cap,
                                           status_dev);
  GIMS_LAUNCH_OK();
  // a-7
  k_gather_kept<<<cdiv(n, 8), 256, 0, st>>>(n, kept_idx, n_kept_dev, kp, feat, scores,
                                            reinterpret_cast<float2*>(kpts_out), feat_out, scores_out);
  GIMS_LAUNCH_OK();
  k_overflow_guard<<<1, 1, 0, st>>>(status_dev, n_kept_dev, n_edges_dev, n_comp_dev, indptr);
  GIMS_LAUNCH_OK();
  return GIMS_OK;
}

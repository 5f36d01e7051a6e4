// Microbenchmark: the one-CTA union-find of gims_agc_build (k_cc_components, csrc/agc.cu) with 32-bit and with 16-bit
// parents in shared memory, on random geometric graphs (~7 neighbours per node, a few isolated-node unions), alternated
// launch by launch; both must give the same labels.  Decides up to which size the 32-bit kernel stays.
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -I include tools/micro/cc_parent_width.cu -o tools/micro/cc_parent_width
#include <cstdio>
#include <cstdlib>
#include <cstdarg>
#include <random>
#include <vector>

#include "../../gims_b200/csrc/agc.cu"

namespace gims {   // the library's host helpers this translation unit needs, as no-ops
void set_error(const char*, ...) {}
void count_launch(int) {}
ProfScope::ProfScope(int, cudaStream_t s) : slot(-1), st(s) {}
ProfScope::~ProfScope() {}
}  // namespace gims

static double time_one(bool wide16, const gims::AgcWs& w, int n, int cap, cudaStream_t st, int reps) {
  cudaEvent_t a, b;
  cudaEventCreate(&a); cudaEventCreate(&b);
  cudaEventRecord(a, st);
  for (int i = 0; i < reps; ++i) {
    if (wide16) gims::launch_cc_components<unsigned short>(w, n, cap, st);
    else gims::launch_cc_components<int>(w, n, cap, st);
  }
  cudaEventRecord(b, st);
  cudaEventSynchronize(b);
  float ms = 0.f;
  cudaEventElapsedTime(&ms, a, b);
  return 1e3 * ms / reps;
}

int main(int argc, char** argv) {
  const int sizes[] = {2048, 8192, 16384};
  cudaStream_t st;
  cudaStreamCreate(&st);
  for (int n : sizes) {
    std::mt19937 rng(n);
    std::uniform_real_distribution<float> U(0.f, 1.f);
    std::vector<float> x(n), y(n);
    for (int i = 0; i < n; ++i) { x[i] = U(rng); y[i] = U(rng); }
    const float r2 = 7.f / (3.14159f * n);
    std::vector<int> indptr(n + 1, 0), idx;
    for (int i = 0; i < n; ++i) {
      for (int j = 0; j < n; ++j)
        if (j != i && (x[i] - x[j]) * (x[i] - x[j]) + (y[i] - y[j]) * (y[i] - y[j]) <= r2) idx.push_back(j);
      indptr[i + 1] = (int)idx.size();
    }
    std::vector<int> iu, iv;
    for (int i = 0; i < n; ++i)
      if (indptr[i] == indptr[i + 1]) { iu.push_back(i); iv.push_back((i * 7919 + 13) % n); }
    const int cap = (int)idx.size() + 1, n_iso = (int)iu.size();
    gims::AgcWs w{};
    int *d_indptr, *d_idx, *d_iu, *d_iv, *d_cnt, *d_parent;
    cudaMalloc(&d_indptr, (n + 1) * 4); cudaMalloc(&d_idx, cap * 4); cudaMalloc(&d_iu, (n_iso + 1) * 4);
    cudaMalloc(&d_iv, (n_iso + 1) * 4); cudaMalloc(&d_cnt, 4); cudaMalloc(&d_parent, n * 4);
    cudaMemcpy(d_indptr, indptr.data(), (n + 1) * 4, cudaMemcpyHostToDevice);
    cudaMemcpy(d_idx, idx.data(), idx.size() * 4, cudaMemcpyHostToDevice);
    if (n_iso) {
      cudaMemcpy(d_iu, iu.data(), n_iso * 4, cudaMemcpyHostToDevice);
      cudaMemcpy(d_iv, iv.data(), n_iso * 4, cudaMemcpyHostToDevice);
    }
    cudaMemcpy(d_cnt, &n_iso, 4, cudaMemcpyHostToDevice);
    w.parent = d_parent; w.indptr_base = d_indptr; w.idx_base = d_idx; w.iso_u = d_iu; w.iso_v = d_iv; w.iso_count = d_cnt;
    std::vector<int> l32(n), l16(n);
    gims::launch_cc_components<int>(w, n, cap, st);
    cudaMemcpyAsync(l32.data(), d_parent, n * 4, cudaMemcpyDeviceToHost, st);
    gims::launch_cc_components<unsigned short>(w, n, cap, st);
    cudaMemcpyAsync(l16.data(), d_parent, n * 4, cudaMemcpyDeviceToHost, st);
    cudaStreamSynchronize(st);
    const bool same = l32 == l16;
    double t32 = 0, t16 = 0;
    const int rounds = 10, reps = 50;
    for (int k = 0; k < rounds; ++k) {
      t32 += time_one(false, w, n, cap, st, reps);
      t16 += time_one(true, w, n, cap, st, reps);
    }
    printf("{\"nodes\": %d, \"edges\": %d, \"iso_unions\": %d, \"us_int32\": %.2f, \"us_uint16\": %.2f, \"same_labels\": %s, "
           "\"error\": \"%s\"}\n",
           n, (int)idx.size(), n_iso, t32 / rounds, t16 / rounds, same ? "true" : "false",
           cudaGetErrorString(cudaGetLastError()));
    cudaFree(d_indptr); cudaFree(d_idx); cudaFree(d_iu); cudaFree(d_iv); cudaFree(d_cnt); cudaFree(d_parent);
  }
  cudaStreamDestroy(st);
  return 0;
}

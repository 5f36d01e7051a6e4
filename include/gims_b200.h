/*
 * gims_b200.h — C ABI of the B200-native GIMS matcher forward path (libgims_b200.so).
 *
 * The reference (songxf1024/GIMS) has no native/FFI interface: its boundary for this path is the
 * Python call `Matching(config)(data)` -> `GMatcher.forward` (models/matching.py:15-30,
 * models/gmatcher.py:219-307).  The entry points below are what a binding for that call needs;
 * each one names the reference code it replaces.  `gims_b200/gmatcher.py` is the ctypes host side
 * that mirrors the reference's Python interface on top of this ABI; INTEGRATION.md shows the stub a
 * maintainer of the reference would add.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless its name ends in `_host`;
 *   - `stream` is a `cudaStream_t` passed as `void*`; all work is enqueued on it, nothing
 *     synchronises unless stated;
 *   - scratch memory comes from caller-provided workspaces sized by the matching `*_workspace_bytes()`
 *     query; a `gims_model` only stores pointers/config (host heap).  The library itself owns, per
 *     process and device, only: the 32 KB cubic-weight table of gims_extract_patches (one cudaMalloc on
 *     first use), one side stream + two events per caller stream (gims_forward_pairs forks the two
 *     images' graph chains; at most 64 caller streams, further ones run unforked), the two events
 *     that order cooperative kernels of different streams, the default arithmetic mode
 *     (gims_set_gemm_mode) and the optional profiler / trace hooks.  All of it is mutex-protected;
 *   - functions return 0 on success, a negative `GIMS_ERR_*` otherwise; `gims_last_error()` gives the
 *     thread-local message;
 *   - features are node-major fp32 rows `[n][256]`; graphs are int32 CSR; counts that depend on the
 *     data (kept keypoints N', edges E) live in device memory (`*_dev` int pointers) so the whole
 *     forward is enqueued without a host round trip.  (Stream capture of a whole forward is NOT supported: the
 *     cooperative Sinkhorn kernels of different streams are ordered through process-wide events, and the two images'
 *     graph chains fork onto a library-owned side stream.)
 */
#ifndef GIMS_B200_H
#define GIMS_B200_H

#include <stddef.h>
#include <stdint.h>

#if defined(__GNUC__)
#define GIMS_API __attribute__((visibility("default")))
#else
#define GIMS_API
#endif

#ifdef __cplusplus
extern "C" {
#endif

#define GIMS_OK              0
#define GIMS_ERR_ARG        -1   /* bad argument / unsupported configuration */
#define GIMS_ERR_CUDA       -2   /* CUDA runtime error (message has the CUDA string) */
#define GIMS_ERR_WORKSPACE  -3   /* workspace too small */
#define GIMS_ERR_OVERFLOW   -4   /* a data-dependent capacity (edge list) was exceeded */

#define GIMS_DESC_DIM      256   /* descriptor_dim the kernels are built for (gmatcher.py:167) */
#define GIMS_NUM_HEADS       4   /* hard-coded in the reference too (gmatcher.py:131) */
#define GIMS_MAX_LAYERS     64
#define GIMS_MAX_KENC        8
#define GIMS_MAX_BATCH       4   /* pairs per gims_forward_pairs call */
#define GIMS_MAX_KPTS    65536   /* per image.  Memory does not bound it (the AGC cosine matrix is n^2 fp32 = 16 GiB, the
                                    couplings (n+1) x ld fp32 = 17.2 GB at this size); the index arithmetic does: element
                                    offsets into those matrices are 64-bit, the AGC rank select counts the n(n-1)/2 < 2^31
                                    pairs in 32 bits, and every node id is below 65536, so the component
                                    search keeps its union-find parents as 16-bit words in shared memory (128 KB) */

/* status word written by the kernels into `gims_pair_outputs.status_dev` / the `status_dev` arguments.
 * Error bits (the host side raises on them): */
#define GIMS_STATUS_EDGE_OVERFLOW     1u   /* edge_cap exceeded: the graph is reported EMPTY (N' = 0), retry larger */
#define GIMS_STATUS_SINKHORN_TIMEOUT  2u   /* a bounded poll inside k_sinkhorn expired: outputs are poisoned (NaN / -2) */
#define GIMS_STATUS_FP16_RANGE        4u   /* GIMS_GEMM_TC_F16: a tensor-core operand reached 32768 — rerun with GIMS_GEMM_TC */
#define GIMS_STATUS_KEYPOINT_OVERFLOW 8u   /* gims_sift_detect: kp_cap exceeded, no keypoints reported — retry larger */
#define GIMS_STATUS_ERROR_MASK        0xffu
/* Information bits: which Sinkhorn iteration the launch ran */
#define GIMS_STATUS_SINKHORN_FAST   0x100u /* exp-free scaled-kernel iteration */
#define GIMS_STATUS_SINKHORN_EXACT  0x200u /* log-sum-exp iteration (fallback) */
#define GIMS_STATUS_SINKHORN_WIDE   0x400u /* log-sum-exp iteration streamed from global memory: problems whose potentials
                                              do not fit the shared memory of the kernels above */

typedef struct gims_model gims_model;

/* Mirror of GMatcher.default_config (gmatcher.py:166-176) — the fields the forward path reads. */
typedef struct {
  int   descriptor_dim;                    /* must be 256 */
  int   num_layers;                        /* len(transformer_layers), 18 */
  int   layer_is_cross[GIMS_MAX_LAYERS];   /* 0 = 'self', 1 = 'cross' (gmatcher.py:136-140) */
  int   kenc_num;                          /* number of Conv1d in kenc: len(keypoint_encoder)+1 */
  int   kenc_dims[GIMS_MAX_KENC + 1];      /* [2, 32, 64, 128, 256, 256] */
  int   sinkhorn_iterations;               /* 100 */
  float match_threshold;                   /* 0.2 */
} gims_config;

/* ---- library ---------------------------------------------------------------------------- */
GIMS_API int         gims_version(void);
GIMS_API const char* gims_last_error(void);
/* number of kernels this library has launched in the calling process (for bench `gpu_launches`) */
GIMS_API long long   gims_launch_count(void);

/* Arithmetic of the dense contractions.  Process-wide default (gims_set_gemm_mode), or per call
 * (gims_pair_inputs.gemm_mode):
 *   GIMS_GEMM_SIMT    fp32 FMA CUDA-core kernels (bit-for-bit fp32 products; used to validate the others)
 *   GIMS_GEMM_TC      tcgen05/TMEM/TMA tensor-core kernels, 3xTF32 error-compensated fp32 everywhere
 *   GIMS_GEMM_TC_F16  (default) every tensor-core operand as fp16 hi + lo planes instead of tf32 hi + lo: the same error class
 *                     (|x - hi - lo| <= max(2^-22 |x|, 2^-25)) at twice the tensor-pipe rate.  fp16 overflows at
 *                     65504: a value >= 32768 raises GIMS_STATUS_FP16_RANGE and the caller reruns with GIMS_GEMM_TC.
 *   GIMS_GEMM_BF16    the "bf16 variant": attention operands in bf16 (8-bit mantissa, one MMA per product), projections
 *                     as GIMS_GEMM_TC_F16.  NOT fp32 parity — reported separately (BASELINE.json north_star). */
#define GIMS_GEMM_SIMT   0
#define GIMS_GEMM_TC     1
#define GIMS_GEMM_TC_F16 2
#define GIMS_GEMM_BF16   3
GIMS_API int gims_set_gemm_mode(int mode);
GIMS_API int gims_get_gemm_mode(void);

/* Bring-up / test entry points for the GEMM kernels: Y[r][o] = act(sum_k A(r,k) W[o][k] + bias[o] + R[r][o]),
 * A = [A0 | A1] along K (K0 + K1), W [N][K0+K1]; W_hi/W_lo = tf32 planes (GIMS_GEMM_TC); W_h16/W_l16 = fp16 planes of
 * W * 2^e and W_sinv -> 2^-e (GIMS_GEMM_TC_F16; K0, K1 multiples of 64, otherwise the tf32 kernel runs). */
GIMS_API int gims_linear(const float* A0, int lda0, int K0, const float* A1, int lda1, int K1, const float* W,
                const float* W_hi, const float* W_lo, const void* W_h16, const void* W_l16, const float* W_sinv,
                const float* bias, const float* R, int ldr, float* Y, int ldy,
                int N, int relu, int rows_max, const int* rows_dev, int mode, unsigned* status_dev, void* stream);
GIMS_API int gims_split_tf32(const float* x, float* hi, float* lo, size_t n, void* stream);
/* Profiling aid: CTA (0,0,0) of every following attention launch stores clock64() stamps of its pipeline
 * (8 int64 per 64-key tile, see attention_tc.cu) into dev_buf; pass NULL to switch the trace off. */
GIMS_API int gims_debug_attention_trace(long long* dev_buf);
/* Same for the tensor-core GEMM: CTA (0,0) of every following launch stores 64 int64 stamps (tools/gemm_trace.py). */
GIMS_API int gims_debug_gemm_trace(long long* dev_buf);
/* Same for k_sinkhorn: CTA 0 stores 6 stamps (8 int64 slots) for each of its first 16 iterations. */
GIMS_API int gims_debug_sinkhorn_trace(long long* dev_buf);

/* ---- profiling hooks (bench.py roofline): CUDA-event timing of ONE kernel class, recorded on the
 * stream each launch goes to.  begin() arms it for at most max_launches launches; end() waits for
 * the recorded events and returns the summed device time and the number of launches timed. */
#define GIMS_PROF_NONE        0
#define GIMS_PROF_GEMM        1   /* projection / MLP GEMMs */
#define GIMS_PROF_ATTENTION   2   /* flash attention */
#define GIMS_PROF_SINKHORN    3   /* fused Sinkhorn + argmax kernel */
#define GIMS_PROF_SCORE       4   /* descriptor score GEMM */
#define GIMS_PROF_COSINE      5   /* AGC cosine-similarity matrix */
#define GIMS_PROF_SAGE_GATHER 6   /* SAGE mean aggregation */
GIMS_API int gims_profile_begin(int kernel_class, int max_launches);
GIMS_API int gims_profile_end(double* total_ms_host, int* launches_host);

/* ---- model: replaces GMatcher.__init__ / load_state_dict (gmatcher.py:177-217) ------------
 * `packed` is ONE device buffer of fp32 weights already packed by the host side
 * (gims_b200/packing.py: BatchNorm folded, attention heads de-interleaved, K|V|Q stacked);
 * `offsets_host[i]` is the float offset of blob i in the order documented in packing.py /
 * DESIGN.md §"Packed weights".  The model keeps the pointer; the caller keeps the buffer alive. */
GIMS_API int  gims_model_create(const gims_config* cfg_host, const float* packed, const int64_t* offsets_host,
                       int n_offsets, gims_model** out_host);
GIMS_API void gims_model_destroy(gims_model* m);
GIMS_API int  gims_packed_blob_count(const gims_config* cfg_host);

/* Weight packing for integrators that do not run Python (the Python host uses gims_b200/packing.py, the specification of
 * the layout; both produce the same buffer).  HOST function, no GPU involved: `tensors` is the reference
 * GMatcher.state_dict() (models/gmatcher.py:177-217) as fp32 host arrays under the reference's own key names
 * ("kenc.encoder.0.weight", "gnn.layers.3.attn.proj.1.bias", "gnn_encoder.layers.0.fc_neigh.weight", "bin_score", ...;
 * Conv1d weights as (out, in[, 1]) row-major; num_batches_tracked and input_proj.* are ignored).  Writes the packed
 * buffer (gims_pack_weights_floats(cfg) floats) and the blob offsets (gims_packed_blob_count(cfg) entries); copy the
 * buffer to the device and hand both to gims_model_create. */
typedef struct gims_named_tensor {
  const char*  name;
  const float* data;
  int64_t      numel;
} gims_named_tensor;
GIMS_API size_t gims_pack_weights_floats(const gims_config* cfg_host);
GIMS_API int    gims_pack_weights(const gims_config* cfg_host, const gims_named_tensor* tensors, int n_tensors,
                         float* packed_host, size_t capacity_floats, int64_t* offsets_host, int n_offsets);

/* ---- a-1..a-7: adaptive graph construction for ONE image ----------------------------------
 * replaces models/agc.py:682-709 build_optimize_graph_with_cosine_similarity (+ 367-391, 413-449,
 * 476-565, 660-678) and the repack of gmatcher.py:244-252.
 *   kpts      [n][2]   pixel xy
 *   desc      descriptors, channel-major [256][n] if desc_channel_major else node-major [n][256]
 *   scores    [n]
 *   k_rank    = min(int(L*percentile/100), L-1), L = n(n-1)/2   (agc.py:377-378; host computes it
 *               with the reference's own float arithmetic)
 * outputs (capacity n unless noted):
 *   kept_idx  [n]      original ids of surviving keypoints, ascending (agc.py:677)
 *   n_kept_dev         N'
 *   indptr    [n+1], indices [edge_cap]  relabelled CSR, neighbours ascending; n_edges_dev = E
 *   kpts_out [n][2], feat_out [n][256], scores_out [n]   = ndata point/feat/score (agc.py:705-707)
 *   thr_out            the cosine threshold (agc.py:439-440)
 *   n_comp_dev         number of components after pruning (the value agc.py:540 prints)
 *   status_dev         GIMS_STATUS_* bits are OR-ed in.  On GIMS_STATUS_EDGE_OVERFLOW the CSR is incomplete and the
 *                      graph is reported empty (*n_kept_dev = *n_edges_dev = 0), so nothing downstream reads it.
 * edge_cap = capacity of `indices` in ints (directed edges). */
GIMS_API size_t gims_agc_workspace_bytes(int n, int edge_cap);
GIMS_API int gims_agc_build(const float* kpts, const float* desc, int desc_channel_major, const float* scores, int n,
                   double radius, long long k_rank, int min_size,
                   void* workspace, size_t workspace_bytes,
                   int* kept_idx, int* n_kept_dev, int* indptr, int* indices, int edge_cap, int* n_edges_dev,
                   float* kpts_out, float* feat_out, float* scores_out, float* thr_out, int* n_comp_dev,
                   unsigned* status_dev, void* stream);

/* ---- a-9: GraphSAGE encoder (gmatcher.py:145-162, 268-269; dgl SAGEConv 'mean') ------------
 * feat [n_max][256] -> out [n_max][256]; rows >= *n_dev are untouched.  scratch: 3*n_max*256 floats. */
GIMS_API int gims_sage_forward(const gims_model* m, const float* feat, const int* indptr, const int* indices,
                      int n_max, const int* n_dev, float* out, float* scratch, void* stream);

/* ---- a-8 + a-10: normalize_keypoints + KeypointEncoder (gmatcher.py:26-33, 87-97, 265-271) --
 * desc[i] = add[i] + kenc(normalize(kpts[i]))  (add = SAGE output, gmatcher.py:270-271; may be NULL).
 * img_w / img_h are `width`/`height` as gmatcher.py:28 unpacks them from image.shape.
 * scratch: 2*n_max*256 floats. */
GIMS_API int gims_kenc_forward(const gims_model* m, const float* kpts, int n_max, const int* n_dev, float img_w, float img_h,
                      const float* add, float* desc, float* scratch, void* stream);

/* ---- a-11 + a-12: one AttentionalPropagation layer for BOTH images (gmatcher.py:99-143) -----
 * desc holds image 0 in rows [0,n0_max) and image 1 in rows [n0_max, n0_max+n1_max); n_dev[2] are the
 * live row counts.  Updates desc in place: desc += MLP(cat[desc, MHA(desc, src, src)]).
 * scratch: gims_attn_scratch_floats(n0_max + n1_max) floats. */
GIMS_API size_t gims_attn_scratch_floats(int rows);
GIMS_API int gims_attn_layer_forward(const gims_model* m, int layer, float* desc, int n0_max, int n1_max, const int* n_dev,
                            float* scratch, unsigned* status_dev /* may be NULL */, void* stream);

/* ---- a-13: final_proj + score matrix (gmatcher.py:273-275) ----------------------------------
 * mdesc [rows][256] = final_proj(desc); couplings (n0_max+1) x ld, ld = gims_couplings_ld(n1_max) (n1_max+1 rounded up
 * to a multiple of 4, so that every row starts 16-byte aligned):
 *   Z0[i][j] = <mdesc0_i, mdesc1_j>/16 for i<N0', j<N1'; bin_score on row N0' and column N1'
 *   (the torch.cat of gmatcher.py:59-60).  scratch: 2*(n0_max+n1_max)*256 floats (tf32 planes of mdesc for the
 *   tensor-core score GEMM) or NULL (CUDA-core score GEMM). */
GIMS_API int gims_couplings_ld(int n1_max);
GIMS_API int gims_final_scores(const gims_model* m, const float* desc, int n0_max, int n1_max, const int* n_dev,
                      float* mdesc, float* couplings, float* scratch, void* stream);

/* ---- a-14 + a-15: log-domain Sinkhorn + mutual-NN matches (gmatcher.py:41-69, 284-294) ------
 * couplings as written by gims_final_scores, row pitch `ld` floats (>= n1_max+1; the fast kernels for more than 2048
 * keypoints need ld == gims_couplings_ld(n1_max) and a 16-byte aligned base, anything else runs the exact kernel).
 * Outputs (capacities n0_max / n1_max):
 *   u [n0_max+1], v [n1_max+1]  final potentials (log_sinkhorn_iterations' u, v)
 *   indices0/1 int32  pre-threshold row/column argmax (gmatcher.py:284-285)
 *   matches0/1 int64 (-1 = unmatched), mscores0/1 fp32 (gmatcher.py:286-294)
 *   status_dev (may be NULL): GIMS_STATUS_SINKHORN_* bits are OR-ed in
 * workspace: gims_sinkhorn_workspace_bytes(n0_max, n1_max).
 * gims_sinkhorn_max_columns() is a column count up to which the scaled-kernel kernels are built for every n0_max <=
 * GIMS_MAX_KPTS: capped at the widest streaming instantiation, 18427 on a B200.  It is not where the WIDE path starts:
 * the EXACT kernel serves wider problems as long as its potentials fit shared memory (about 56 k columns on a B200).
 * Problems wider than that run the WIDE path: three non-cooperative launches per iteration (a row pass, per-row-block
 * column partials, a fixed-order combine of those partials), no float atomics and no grid-wide waits, deterministic run
 * to run (GIMS_STATUS_SINKHORN_WIDE says it ran). */
GIMS_API int gims_sinkhorn_max_columns(void);
GIMS_API size_t gims_sinkhorn_workspace_bytes(int n0_max, int n1_max);
GIMS_API int gims_sinkhorn_match(const float* couplings, int ld, int n0_max, int n1_max, const int* n_dev, int iters,
                        float match_threshold, void* workspace, size_t workspace_bytes,
                        float* u, float* v, int* indices0, int* indices1,
                        int64_t* matches0, int64_t* matches1, float* mscores0, float* mscores1,
                        unsigned* status_dev, void* stream);

/* ---- front end: oriented keypoint patches on the device (SURVEY.md §8f row 2) ------------------
 * replaces the per-keypoint loop of ComputePatches (utils/library.py:84-110: cv2.warpAffine INTER_CUBIC / BORDER_CONSTANT
 * into 64 x 64) and the INTER_AREA resize to 32 x 32 + /255 of utils/common.py:882-884; bit-identical to OpenCV's 8-bit
 * fixed-point warp.  The Gaussian pyramid (utils/library.py:234-293) is gims_gaussian_pyramid's output (below) or built by
 * the caller (OpenCV) and uploaded:
 *   levels           uint8, every level H x W x channels (channels 1 or 3), concatenated; level l starts at byte
 *                    level_offset_dev[l] and is level_height_dev[l] x level_width_dev[l]
 *   kp_level_dev     [n_kp] pyramid level of each keypoint ((octave - firstOctave) * (nOctaveLayers + 3) + layer)
 *   kp_inverse_map_dev [n_kp][6] double: the dst -> src affine map, i.e. the 2 x 3 matrix the reference passes to
 *                    cv2.warpAffine, inverted as cv::warpAffine inverts it
 *   patches_out      [n_kp][32][32][channels] fp32 in [0, 1] */
GIMS_API int gims_extract_patches(const unsigned char* levels, const long long* level_offset_dev, const int* level_height_dev,
                         const int* level_width_dev, int n_levels, int channels, const int* kp_level_dev,
                         const double* kp_inverse_map_dev, int n_kp, float* patches_out, void* stream);

/* test hook: the 32 x 32 x 16 int16 bicubic weight table of gims_extract_patches, as built on the host */
GIMS_API int gims_debug_bicubic_table(short* out_host);

/* ---- front end: the Gaussian pyramid the patches are cut from, on the device ---------------------------------------
 * replaces frontend.gaussian_pyramid (utils/library.py:234-293: cv2.resize x2 INTER_LINEAR_EXACT, per octave five
 * cv2.GaussianBlur with the incremental SIFT sigmas, each next octave seeded by INTER_NEAREST x0.5 of level 3); byte for
 * byte what OpenCV's 8-bit fixed-point arithmetic gives.  `image` is h x w x channels uint8 (channels 1 or 3, interleaved).
 * gims_pyramid_layout (host only) gives the level count, nOctaves * 6 with
 * nOctaves = round_half_even(log(float32(min(2h, 2w))) / log(2) - 2) + 1, and, for each level, its byte offset inside the
 * level buffer and its size: the level table gims_extract_patches takes.  The three arrays may be null (call once to get
 * the count); each one that is not null must hold n_levels entries.  The buffer holds
 * offset_host[n - 1] + height_host[n - 1] * width_host[n - 1] * channels bytes.
 * gims_gaussian_pyramid writes every level into `levels_out` in that layout; the workspace holds the uint16 row pass. */
GIMS_API int gims_pyramid_layout(int h, int w, int channels, int* n_levels, int64_t* offset_host, int* height_host,
                        int* width_host);
GIMS_API size_t gims_pyramid_workspace_bytes(int h, int w, int channels);
GIMS_API int gims_gaussian_pyramid(const unsigned char* image, int h, int w, int channels, unsigned char* levels_out,
                          void* workspace, size_t workspace_bytes, void* stream);

/* test hook: the 8-bit fixed-point taps (sum 256) cv2.GaussianBlur uses for `sigma`; taps_host holds at least 127 ints */
GIMS_API int gims_debug_gaussian_kernel(double sigma, int* taps_host, int* n_host);

/* ---- front end: SIFT keypoint detection on the device --------------------------------------------------------------
 * OpenCV 4.x SIFT::detect with frontend.SIFT_CONFIG (3 layers, contrastThreshold 0.001, edgeThreshold 80, sigma 1.6,
 * the image doubled first) on the float32 scale space of the grey image, in the float32 order of operations that
 * oracle/cv_sift_oracle.py fixes: the records equal that restatement bit for bit and agree with cv2 within a tolerance
 * (cv2 does not reproduce itself bit for bit).  The octave count is gims_pyramid_layout's, so the keypoints index the
 * patch pyramid.  `image` is h x w x channels uint8 (channels 1 or 3, BGR), on the device.
 * Outputs (kp_cap entries each, on the device): pt [kp_cap][2] float xy in input pixels, size, angle (degrees), response
 * float, octave int32 packed as cv2.KeyPoint.octave; *n_kp_dev the number written.  The order is cv2's (sorted by x, y,
 * -size, angle, -response, -octave, duplicates of (pt, size, angle) removed); with max_keypoints > 0 and more keypoints
 * than that, the max_keypoints strongest by response, strongest first, ties in that sorted order.
 * kp_cap bounds the keypoints before duplicates are removed; the scale-space extrema are bounded by 2 * kp_cap.  When
 * either bound is exceeded GIMS_STATUS_KEYPOINT_OVERFLOW is OR-ed into *status_dev and *n_kp_dev is 0: retry with a
 * larger kp_cap.  Enqueue-only on `stream`; the workspace holds gims_sift_workspace_bytes(h, w, channels, kp_cap). */
GIMS_API size_t gims_sift_workspace_bytes(int h, int w, int channels, int kp_cap);
GIMS_API int gims_sift_detect(const unsigned char* image, int h, int w, int channels, int max_keypoints, int kp_cap,
                     void* workspace, size_t workspace_bytes, float* pt, float* size, float* angle, float* response,
                     int* octave, int* n_kp_dev, unsigned* status_dev, void* stream);

/* ---- caller-side result consumption on the device (SURVEY.md §8f row 3) --------------------
 * gims_gt_matches replaces utils/preprocess_utils.py:98-132 torch_find_matches (called at eval_homography.py:205):
 *   kpts0 [n0][2], kpts1 [n1][2] pixel xy (fp32, device); homography_dev: 9 fp32, row-major, maps image 0 -> image 1.
 *   n_iters rounds of mutual nearest neighbours among the still unmatched points, accepted below dist_thresh pixels.
 *   gt0 [n0] = index in image 1 of the ground-truth partner or -1; gt1 [n1] likewise; round0 [n0] = the round (0-based) in
 *   which point i was matched, -1 if never (the reference returns the pairs ordered by round, then by image-1 index).
 * gims_match_counts replaces eval_homography.py:224-228: counts_dev[3] = { true positives, predicted matches, missed
 *   ground-truth matches } over the first *n_dev (or n0_max) rows; precision = c0 / c1, recall = c0 / (c0 + c2). */
GIMS_API size_t gims_gt_workspace_bytes(int n0, int n1);
GIMS_API int gims_gt_matches(const float* kpts0, int n0, const float* kpts1, int n1, const float* homography_dev,
                    float dist_thresh, int n_iters, void* workspace, size_t workspace_bytes, int* gt0, int* gt1,
                    int* round0, void* stream);
GIMS_API int gims_match_counts(const int64_t* matches0, const int* gt0, int n0_max, const int* n_dev /* may be NULL */,
                      int* counts_dev, void* stream);

/* ---- RANSAC homographies of a batch of matched point sets ---------------------------------------------------------
 * gims_find_homographies replaces cv2.findHomography(mkpts0, mkpts1, cv2.RANSAC, thresh) of eval_homography.py:180-235
 * (the homography behind the AUC) and eval_matches.py (the inlier count), for n_pairs pairs in one call.  The algorithm is the
 * deterministic restatement oracle/ransac_oracle.py fixes (cv2's RANSAC + DLT + Levenberg-Marquardt refinement, with a
 * counter-based sampler and Gaussian-elimination solves); the results equal it bit for bit, and a pair gives the same
 * result alone and in any batch.
 *   src, dst: [total][2] fp32 pixel xy on the device; pair p owns rows [offsets_dev[p], offsets_dev[p+1]) (device int32
 *   [n_pairs + 1], non-decreasing, from 0).  thresh: reprojection threshold in pixels (> 0); max_iters >= 1 hypotheses;
 *   0 < confidence < 1; seed: the sampler's key.
 *   H_out [n_pairs][9] fp64 row-major with H[8] = 1; mask_out [total] uint8, 1 for the inliers of H; n_inliers [n_pairs];
 *   n_iters [n_pairs] the number of hypotheses run (may be NULL).  "Not found" (fewer than 4 points, a degenerate set,
 *   or no hypothesis with more than 3 inliers) is n_inliers = 0, H = 0 and a zero mask.  Pairs with 4 points get the
 *   DLT of the four and an all-ones mask, as in cv2.
 *   Enqueue-only on `stream`; the workspace holds gims_homography_workspace_bytes(n_pairs, offsets_dev[n_pairs]). */
GIMS_API size_t gims_homography_workspace_bytes(int n_pairs, int total_points);
GIMS_API int gims_find_homographies(const float* src, const float* dst, const int* offsets_dev, int n_pairs, double thresh,
                           int max_iters, double confidence, unsigned long long seed, void* workspace,
                           size_t workspace_bytes, double* H_out, unsigned char* mask_out, int* n_inliers, int* n_iters,
                           void* stream);

/* ---- whole pair: replaces GMatcher.forward (gmatcher.py:219-307), test mode ----------------- */
typedef struct {
  const float* kpts[2];          /* [n][2] */
  const float* desc[2];          /* [256][n] channel-major (reference layout) or [n][256] */
  const float* scores[2];        /* [n] */
  int   n[2];                    /* input keypoint counts */
  int   desc_channel_major;
  float img_w[2], img_h[2];      /* as unpacked by gmatcher.py:28 from image{0,1}.shape */
  double radius;                 /* data.get('radius', 25) */
  long long k_rank[2];           /* see gims_agc_build */
  int   min_size;                /* data.get('min_size', 8) */
  int   edge_cap;                /* per-image capacity of csr_indices */
  int   gemm_mode;               /* 0 = the library default (gims_set_gemm_mode), else GIMS_GEMM_* + 1 */
} gims_pair_inputs;

typedef struct {
  int*     n_kept_dev;           /* [2]  N0', N1' */
  int*     kept_idx[2];          /* [n]  kept_kpts{0,1}_indices */
  int*     csr_indptr[2];        /* [n+1] */
  int*     csr_indices[2];       /* [edge_cap] */
  int*     n_edges_dev;          /* [2] */
  int*     n_comp_dev;           /* [2] */
  float*   thr_dev;              /* [2] */
  float*   kpts[2];              /* [n][2]    data['keypoints*'] after pruning */
  float*   feat[2];              /* [n][256]  data['descriptors*'] after pruning (node-major) */
  float*   scores[2];            /* [n] */
  float*   mdesc;                /* [(n0+n1)][256], image 1 at row n0 */
  int64_t* matches[2];           /* [n] */
  float*   mscores[2];           /* [n] */
  int*     indices[2];           /* [n]  pre-threshold argmax */
  float*   u;                    /* [n0+1] */
  float*   v;                    /* [n1+1] */
  float*   couplings;            /* optional (may be NULL -> internal): (n0+1) x gims_couplings_ld(n1) */
  float*   desc_gnn;             /* optional: [(n0+n1)][256] descriptors after the attention stack */
  float*   desc_in;              /* optional: [(n0+n1)][256] SAGE + kenc (input of the attention stack) */
  unsigned* status_dev;          /* [1] GIMS_STATUS_* bits */
} gims_pair_outputs;

GIMS_API size_t gims_pair_workspace_bytes(const gims_model* m, int n0, int n1, int edge_cap);
GIMS_API int gims_forward_pair(const gims_model* m, const gims_pair_inputs* in_host, const gims_pair_outputs* out_host,
                      void* workspace, size_t workspace_bytes, void* stream);

/* ---- a batch of pairs: same results as n_pairs calls of gims_forward_pair, but the rows of all images are stacked and
 * every projection GEMM / attention layer is ONE launch for the whole batch (fewer, fuller launches).  `in_host` /
 * `out_host` are arrays of n_pairs (<= GIMS_MAX_BATCH) descriptors; the pairs may have different sizes but must share
 * gemm_mode.  `out_host[p].mdesc` holds image 1 at row in_host[p].n[0], as for a single pair.
 * workspace: gims_batch_workspace_bytes(n_pairs, n0[], n1[], max edge_cap). */
GIMS_API size_t gims_batch_workspace_bytes(int n_pairs, const int* n0_host, const int* n1_host, int edge_cap);
GIMS_API int gims_forward_pairs(const gims_model* m, int n_pairs, const gims_pair_inputs* in_host,
                       const gims_pair_outputs* out_host, void* workspace, size_t workspace_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* GIMS_B200_H */

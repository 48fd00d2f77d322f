/*
 * neddf_b200 -- C ABI of the B200-native NeDDF volumetric-rendering hot path.
 *
 * This is the drop-in boundary: plain pointers and sizes, no torch types.  The reference
 * (ueda0319/neddf @ f71838ea) is pure Python/PyTorch and has no FFI of its own, so every
 * entry point below names the reference *function* it replaces (file:line relative to the
 * reference root).  The Python host classes in neddf_b200/ (NeRFRender, NeDDF) bind
 * these with ctypes; INTEGRATION.md shows the binding a reference maintainer would add.
 *
 * Conventions
 *   - every pointer named d_* is a DEVICE pointer (fp32 unless stated), row-major,
 *     contiguous; h_* is a HOST pointer.
 *   - `stream` is a cudaStream_t passed as void* (NULL = default stream).  Calls only
 *     enqueue work; they never synchronise and never allocate caller-visible memory.
 *   - return value: 0 on success, a negative NEDDF_E_* code on failure;
 *     neddf_last_error() returns a thread-local message for the last failure.
 *   - "edges": the reference samples S+1 edge distances per ray; the last one only closes
 *     the last interval (base_neural_render.py:145-151).
 */
#ifndef NEDDF_B200_H
#define NEDDF_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NEDDF_ABI_VERSION 2

#define NEDDF_OK 0
#define NEDDF_E_INVALID (-1)     /* bad argument / unsupported configuration */
#define NEDDF_E_CUDA (-2)        /* CUDA runtime error (message has the detail) */
#define NEDDF_E_UNSUPPORTED (-3) /* valid reference config this build does not cover */

/* activation ids (neddf/network/neddf.py:95-118) */
#define NEDDF_ACT_TANHEXP 0
#define NEDDF_ACT_RELU 1
#define NEDDF_ACT_LEAKYRELU 2

/* sampling types (neddf/render/nerf_render.py:141-146) */
#define NEDDF_SAMPLING_POINT 0
#define NEDDF_SAMPLING_CONE 1

/* uv dtypes accepted by neddf_make_rays (nerf_trainer.py:100-106 uses int16, render_image int64) */
#define NEDDF_UV_I64 0
#define NEDDF_UV_I32 1
#define NEDDF_UV_I16 2
#define NEDDF_UV_F32 3

/* field engines */
#define NEDDF_ENGINE_AUTO 0  /* TC when the configuration allows, else TC2, else fp32 */
#define NEDDF_ENGINE_FP32 1  /* CUDA-core fp32 FMA megakernel (bit-faithful fp32 arithmetic) */
#define NEDDF_ENGINE_TC 2    /* tcgen05 megakernel, 3-product fp16-split operands, fp32 accumulate; one CTA per SM */
#define NEDDF_ENGINE_TC2 3   /* same arithmetic, CTA pairs (tcgen05 cta_group::2): half the weight stream per sample */

/* output-selection flags for neddf_field_forward* */
#define NEDDF_OUT_FULL 0      /* everything NeDDF.forward returns, incl. fields_penalty */
#define NEDDF_OUT_EVAL 1      /* penalty not required: colour-trunk Jacobian rows may be skipped */

#define NEDDF_MAX_SKIPS 8
#define NEDDF_N_PENALTY 6

/* Constructor arguments of NeDDF (neddf/network/neddf.py:52-66). */
typedef struct neddf_field_config {
  int32_t embed_pos_rank;          /* 10 */
  int32_t embed_dir_rank;          /* 4  */
  int32_t ddf_layer_count;         /* 8  -> 7 hidden layers + heads */
  int32_t ddf_layer_width;         /* 256 (only 256 is built) */
  int32_t col_layer_count;         /* 4  -> 3 hidden layers + head */
  int32_t col_layer_width;         /* 256 */
  int32_t activation_type;         /* NEDDF_ACT_* for hidden layers */
  int32_t density_activation_type; /* NEDDF_ACT_* for the density output */
  float d_near;
  int32_t n_skips;
  int32_t skips[NEDDF_MAX_SKIPS];
  /* weights in the reference's insertion order (neddf.py:259-300):
   * constraints_aux_grad, constraints_dDdt, range_distance, range_aux_grad, range_color,
   * constraints_color; a key absent from the reference dict is passed as 1.0 */
  float penalty_weight[NEDDF_N_PENALTY];
} neddf_field_config_t;

/* Warm-up scalars, NeDDF.set_iter (neddf/network/neddf.py:311-326). */
typedef struct neddf_field_state {
  float aux_grad_scale;
  float distance_range_max;
  float lowpass_alpha;
  /* penalty weights as the reference reads them: from the module's dict on EVERY forward
   * (neddf.py:296-299), same order as neddf_field_config_t.penalty_weight */
  float penalty_weight[NEDDF_N_PENALTY];
} neddf_field_state_t;

typedef struct neddf_field neddf_field_t; /* opaque: config + packed device weights */

int32_t neddf_abi_version(void);
const char* neddf_last_error(void);

/* Number of linear layers of a configuration and their [in,out] shapes, in the order
 * layers_ddf.0.., layers_col.0.., layer_ddf_out, layer_aux_out, layer_col_out
 * (neddf/network/neddf.py:129-145).  shapes_out receives 2*n int32 (may be NULL). */
int32_t neddf_field_layer_shapes(const neddf_field_config_t* cfg, int32_t* shapes_out, int32_t max_layers);

/* NeDDF.__init__ (neddf.py:52-160): validates the configuration, allocates packed-weight
 * storage on the current device.  A handle also owns per-launch scratch of its kernels (status word, the parked
 * rows of the batched colour trunk, head partial sums of the pair kernel): launches on ONE handle must be
 * stream-ordered with respect to each other (the reference's module is not re-entrant either); different
 * handles - e.g. the coarse and the fine network - are independent. */
int32_t neddf_field_create(const neddf_field_config_t* cfg, neddf_field_t** out);
int32_t neddf_field_destroy(neddf_field_t* f);

/* Which engine a NEDDF_ENGINE_* request resolves to for this field (AUTO -> TC when the
 * tensor-core megakernel covers the configuration, else FP32). */
int32_t neddf_field_resolve_engine(const neddf_field_t* f, int32_t engine);

/* Read and clear the field's device status word (synchronises `stream`): bit 2 (value 4) = the
 * tensor-core engine met an activation outside fp16 range (|x| > 65504); results of that call are
 * invalid and the caller should use NEDDF_ENGINE_FP32 for this network. */
int32_t neddf_field_status(const neddf_field_t* f, int32_t* h_status_out, void* stream);

/* Profiling aid for the tensor-core engine: when d_buf != NULL, CTA 0 of every following launch
 * writes 4 SM-clock stamps per (tile, step) into d_buf[capacity] (int64): MMA phase start, MMA
 * issue done, epilogue start, epilogue done.  Pass NULL to switch it off. */
int32_t neddf_field_set_timeline(neddf_field_t* f, int64_t* d_buf, int32_t capacity);

/* The reference's training objective in one launch (loss/base_loss.py:45-85, color_loss.py:41-55,
 * mask_bce_loss.py:41-59, fields_constraint_loss.py:40-54; summed as nerf_trainer.py:118-121):
 *   d_weights[6] = weight, weight_coarse of ColorLoss, MaskBCELoss, FieldsConstraintLoss (0 = term off)
 *   d_terms[6]   = the six weighted terms (device); g_* = gradients of their SUM w.r.t. the render outputs
 * Any input / gradient pointer may be NULL when its weight is 0. */
int32_t neddf_render_loss(const float* d_color, const float* d_color_coarse, const float* d_trans,
                          const float* d_trans_coarse, const float* d_penalty, const float* d_penalty_coarse,
                          const float* d_target_color, const float* d_target_mask, int64_t n_rays,
                          const float* d_weights, float* d_terms, float* g_color, float* g_color_coarse,
                          float* g_trans, float* g_trans_coarse, float* g_penalty, float* g_penalty_coarse,
                          void* stream);

/* torch.optim.Adam step of n_tensors parameter tensors in one launch (nerf_trainer.py:38-42, 129); with a
 * field handle the tensors must be (weight, bias) of every layer in reference order and the kernel-layout
 * weights are re-packed on the same stream (what neddf_field_set_weights does after every optimiser step). */
int32_t neddf_field_adam_step(neddf_field_t* f, float* const* d_params, const float* const* d_grads,
                              float* const* d_exp_avg, float* const* d_exp_avg_sq, const int64_t* h_numel,
                              int32_t n_tensors, float lr, float beta1, float beta2, float eps, float weight_decay,
                              int64_t step, void* stream);

/* Weight gradients of LinearGradFunction.backward (nn_module/with_grad/linear.py:72-80) as a tensor-core
 * split-K GEMM with fp16 hi/lo operands split on the fly (3 products, fp32 accumulation, deterministic):
 *     out[m, n] = sum_r A[r, a_col0 + m] * B[r, n],   m < ka <= 128,  n < n_cols <= 256
 * A: [rows, lda] fp32 (layer inputs X, or the head gradients), B: [rows, ldb] fp32 with 256 columns (the
 * pre-activation gradients G, or the last hidden activations).  d_workspace: neddf_wgrad_workspace_bytes(). */
int64_t neddf_wgrad_workspace_bytes(void);
int32_t neddf_wgrad(const float* d_a, int64_t lda, int32_t a_col0, int32_t ka, const float* d_b, int64_t ldb,
                    int64_t rows, float* d_out, int64_t ld_out, int32_t n_cols, float* d_workspace, void* stream);
/* Bias gradients (linear.py:80): out[c] = sum over samples of G[sample][0][c] (value rows of [n,4,256]). */
int32_t neddf_colsum_value_rows(const float* d_g, int64_t n_samples, int64_t sample_stride, float* d_out,
                                float* d_workspace, void* stream);

/* Early ray termination (BASELINE.json configs[4]; opt-in, not in the reference whose compositing visits every
 * sample, base_neural_render.py:148-172).  The field on ONE depth segment: samples [edge0, edge0+seg_len) of the
 * rays listed in d_ray_index[0 .. *d_n_active) (both NULL = all n_rays rays); density / colour are scattered to
 * [ray, edge] of the full [n_rays, n_edges] arrays, which the caller zero-fills: a sample that is never
 * evaluated has density 0 and contributes nothing to neddf_composite.  *d_n_active is read on the device. */
int32_t neddf_field_forward_rays_segment(const neddf_field_t* f, const neddf_field_state_t* st,
                                         const float* d_ray_dir, const float* d_ray_orig, const float* d_dists,
                                         int64_t n_rays, int32_t n_edges, int32_t sampling_type, float ray_radius,
                                         int32_t edge0, int32_t seg_len, const int32_t* d_ray_index,
                                         const int32_t* d_n_active, float* d_density, float* d_color,
                                         int32_t engine, void* stream);

/* After a segment: d_transmittance[ray] *= prod_j (1 - o_j + 1e-7) over the segment's intervals (the factors of
 * base_neural_render.py:148-160), and the rays with transmittance > eps are written to d_idx_out / *d_n_out
 * (order without meaning).  d_executed (optional, uint64) accumulates rays_in * seg_len = MLP evaluations
 * actually executed.  d_idx_in / d_n_in NULL = all rays. */
int32_t neddf_terminate_rays(const float* d_dists, const float* d_density, int64_t n_rays, int32_t n_edges,
                             int32_t edge0, int32_t seg_len, const int32_t* d_idx_in, const int32_t* d_n_in,
                             float* d_transmittance, float eps, int32_t* d_idx_out, int32_t* d_n_out,
                             uint64_t* d_executed, void* stream);

/* Debugging aid for the tensor-core pair engine: when d_buf != NULL, cluster 0 of every following
 * launch copies, at (its first tile, hidden step `step`), per CTA the AUX operand buffer (hi parts,
 * 6144 words) and both accumulator halves (2 x 128 lanes x 128 columns fp32) into
 * d_buf[2][6144 + 32768].  Pass NULL to switch it off. */
int32_t neddf_field_set_debug_dump(neddf_field_t* f, float* d_buf, int32_t step);

/* Re-pack the module's parameters into kernel layout.  d_weights[i] is the i-th layer's
 * weight, fp32 [in,out] row-major exactly as LinearGradLayer stores it
 * (nn_module/with_grad/linear.py:111-116); d_biases[i] its bias [out].  Must be called
 * after load_state_dict / every optimiser step (weights are read when the call is enqueued
 * on `stream`). */
int32_t neddf_field_set_weights(neddf_field_t* f, const float* const* d_weights,
                                const float* const* d_biases, int32_t n_layers, void* stream);

/* Camera.create_rays (neddf/camera/camera.py:155-187, pinhole_calib.py:51-74).
 * h_R[9] row-major, h_T[3], h_calib = {fx, fy, cx, cy}. */
int32_t neddf_make_rays(const void* d_uv, int32_t uv_dtype, int64_t n_rays, const float* h_R,
                        const float* h_T, const float* h_calib, float* d_ray_dir,
                        float* d_ray_orig, void* stream);

/* Pixel grid of render_image (neddf/render/nerf_render.py:220-230) fused with create_rays for
 * the row-major pixel range [first, first+n_rays) of a (width/ds) x (height/ds) image. */
int32_t neddf_make_image_rays(int32_t width, int32_t height, int32_t downsampling, int64_t first,
                              int64_t n_rays, const float* h_R, const float* h_T,
                              const float* h_calib, float* d_ray_dir, float* d_ray_orig,
                              void* stream);

/* Stratified coarse edges: linspace(near,far,n_edges)[j] + u[b,j]*(far-near)/(n_edges-1)
 * (neddf/render/nerf_render.py:131-139). d_u, d_dists: [n_rays, n_edges]. */
int32_t neddf_coarse_dists(const float* d_u, int64_t n_rays, int32_t n_edges, float dist_near,
                           float dist_far, float* d_dists, void* stream);

/* Ray.get_sampling_points / get_sampling_cones (neddf/ray/ray.py:88-194): materialises the
 * Sampling tensors pos/dir/var [n_rays, n_edges, 3]. */
int32_t neddf_make_samples(const float* d_ray_dir, const float* d_ray_orig, const float* d_dists,
                           int64_t n_rays, int32_t n_edges, int32_t sampling_type,
                           float ray_radius, float* d_pos, float* d_dir, float* d_var,
                           void* stream);

/* NeDDF.forward (neddf/network/neddf.py:162-309) on n samples given as Sampling tensors
 * pos/dir/var [n,3].  Outputs: distance[n], density[n], color[n,3], penalty[n], aux_grad[n];
 * any output pointer may be NULL.  `flags` is NEDDF_OUT_*; `engine` NEDDF_ENGINE_*. */
int32_t neddf_field_forward(const neddf_field_t* f, const neddf_field_state_t* st,
                            const float* d_pos, const float* d_dir, const float* d_var, int64_t n,
                            float* d_distance, float* d_density, float* d_color,
                            float* d_penalty, float* d_aux_grad, int32_t flags, int32_t engine,
                            void* stream);

/* Same network, with get_sampling_points/cones fused into the prologue: samples are
 * described by rays + edge distances, nothing of size [n,3] touches HBM. */
int32_t neddf_field_forward_rays(const neddf_field_t* f, const neddf_field_state_t* st,
                                 const float* d_ray_dir, const float* d_ray_orig,
                                 const float* d_dists, int64_t n_rays, int32_t n_edges,
                                 int32_t sampling_type, float ray_radius, float* d_distance,
                                 float* d_density, float* d_color, float* d_penalty,
                                 float* d_aux_grad, int32_t flags, int32_t engine, void* stream);

/* Training forward of NeDDF.forward on rays + edge distances (tensor-core engine when available): like
 * neddf_field_forward_rays with NEDDF_OUT_FULL, and additionally keeps the pre-activations of every
 * hidden layer in d_save_pre [n_hidden][n][4][256] (n = n_rays*n_edges; value row incl. bias, then the
 * three Jacobian rows) for neddf_field_backward. */
int32_t neddf_field_forward_train(const neddf_field_t* f, const neddf_field_state_t* st,
                                  const float* d_ray_dir, const float* d_ray_orig, const float* d_dists,
                                  int64_t n_rays, int32_t n_edges, int32_t sampling_type, float ray_radius,
                                  float* d_density, float* d_color, float* d_penalty, float* d_save_pre,
                                  int32_t engine, void* stream);

/* Backward of NeDDF.forward (the reference's hand-written backward passes, nn_module/with_grad
 * linear.py:49-84, tanh_exp.py:57-88, softplus.py:55-89, sigmoid.py:49-83, and autograd through
 * neddf.py:220-300).  Inputs: the forward's geometry, d_save_pre, and the upstream gradients of
 * density[n], color[n,3], fields_penalty[n] (g_penalty may be NULL).  The kernel does all sample-local
 * work and the data-gradient GEMMs; it writes what the weight-gradient GEMMs  gW_l = X_l^T G_l  need:
 *   d_post [n_hidden][n][4][256]  post-activations (h part of the next layer's / the heads' input)
 *   d_gpre [n_hidden][n][4][256]  gradient w.r.t. each layer's pre-activations (bias grad = sum of row 0)
 *   d_ghead_da [n][4][2], d_ghead_col [n][4][4]  gradients w.r.t. the head outputs (value + Jacobian rows)
 *   d_xes [n][4][6*embed_pos]     scaled position embedding (input of layer 0 and of skip layers)
 *   d_xcol [n][4][6*(embed_pos+embed_dir)+3]   [E0 | D | normal] (input part of the first colour layer) */
int32_t neddf_field_backward(const neddf_field_t* f, const neddf_field_state_t* st, const float* d_ray_dir,
                             const float* d_ray_orig, const float* d_dists, int64_t n_rays, int32_t n_edges,
                             int32_t sampling_type, float ray_radius, const float* d_save_pre,
                             const float* g_density, const float* g_color, const float* g_penalty, float* d_post,
                             float* d_gpre, float* d_ghead_da, float* d_ghead_col, float* d_xes, float* d_xcol,
                             void* stream);

/* The same training forward / backward on Sampling tensors pos/dir/var [n,3] (NeDDF.forward(sampling)
 * under autograd).  The forward also returns distance and aux_grad; their gradients are not
 * propagated (the reference's losses never consume them). */
int32_t neddf_field_forward_train_samples(const neddf_field_t* f, const neddf_field_state_t* st,
                                          const float* d_pos, const float* d_dir, const float* d_var, int64_t n,
                                          float* d_distance, float* d_density, float* d_color, float* d_penalty,
                                          float* d_aux_grad, float* d_save_pre, int32_t engine, void* stream);
int32_t neddf_field_backward_samples(const neddf_field_t* f, const neddf_field_state_t* st, const float* d_pos,
                                     const float* d_dir, const float* d_var, int64_t n, const float* d_save_pre,
                                     const float* g_density, const float* g_color, const float* g_penalty,
                                     float* d_post, float* d_gpre, float* d_ghead_da, float* d_ghead_col,
                                     float* d_xes, float* d_xcol, void* stream);

/* BaseNeuralRender.integrate_volume_render (neddf/render/base_neural_render.py:117-172) plus
 * the penalty integration of render_rays (nerf_render.py:153-159).
 * in : dists[n_rays,n_edges], density[n_rays,n_edges], color[n_rays,n_edges,3],
 *      penalty[n_rays,n_edges] (NULL to skip)
 * out: weight[n_rays,n_edges-1], depth[n_rays], color_out[n_rays,3], transmittance[n_rays],
 *      penalty_out[n_rays] (NULL to skip).  d_status (int32, may be NULL) gets bit0 set if a
 *      NaN weight is produced (the reference asserts, base_neural_render.py:155). */
int32_t neddf_composite(const float* d_dists, const float* d_density, const float* d_color,
                        const float* d_penalty, int64_t n_rays, int32_t n_edges, float max_dist,
                        float* d_weight, float* d_depth, float* d_color_out,
                        float* d_transmittance, float* d_penalty_out, int32_t* d_status,
                        void* stream);

/* Backward of neddf_composite (what autograd derives through base_neural_render.py:148-172 and
 * nerf_render.py:153-159 in the reference).  Upstream gradients g_* of weight[n_rays,n_edges-1],
 * depth[n_rays], color_out[n_rays,3], transmittance[n_rays], penalty_out[n_rays] (any may be NULL =
 * zero) -> gradients of density[n_rays,n_edges], color[n_rays,n_edges,3], penalty[n_rays,n_edges]
 * (any may be NULL).  Edge distances carry no gradient (the reference samples them under no_grad). */
int32_t neddf_composite_backward(const float* d_dists, const float* d_density, const float* d_color,
                                 int64_t n_rays, int32_t n_edges, float max_dist, const float* g_weight,
                                 const float* g_depth, const float* g_color, const float* g_transmittance,
                                 const float* g_penalty, float* d_grad_density, float* d_grad_color,
                                 float* d_grad_penalty, void* stream);

/* BaseNeuralRender.sample_pdf (base_neural_render.py:27-115).
 * in : dists[n_rays,n_edges], weights[n_rays,n_edges-1] (IN/OUT: negative and NaN entries are
 *      zeroed in place exactly as the reference does to its argument, :52-55), u[n_rays,n_new]
 * cat_coarse != 0 (what render_rays uses): out dists_fine[n_rays, n_edges+n_new] = sort(new | coarse edges);
 * cat_coarse == 0: neighbour-max smoothing of the biased weights (:61-68), out dists_fine[n_rays, n_new].
 * out: dists_fine sorted; optional ids[n_rays,n_new] (int64,
 *      searchsorted right=True) and cdf[n_rays,n_edges].  The batch-wide NaN fallback
 *      (base_neural_render.py:105-114) is applied on device, per launch like the reference:
 *      d_status (optional) points to TWO int32 - [0] persistent flags (bit1 = "pdf sampling failed"
 *      happened since the host last cleared it), [1] scratch holding this launch's decision. */
int32_t neddf_sample_pdf(const float* d_dists, float* d_weights, const float* d_u,
                         int64_t n_rays, int32_t n_edges, int32_t n_new, int32_t cat_coarse,
                         float* d_dists_fine, int64_t* d_ids, float* d_cdf, int32_t* d_status, void* stream);

/* The inverse-CDF step alone on a caller-supplied cdf (base_neural_render.py:77-98); used to
 * check sample indices bit-exactly against torch.searchsorted. */
int32_t neddf_invert_cdf(const float* d_dists, const float* d_cdf, const float* d_u,
                         int64_t n_rays, int32_t n_edges, int32_t n_new, float* d_samples,
                         int64_t* d_ids, void* stream);

/* How many kernels this library has launched since load (bench.py "gpu_launches"). */
int64_t neddf_launch_count(void);

/* Self-test of the tcgen05 GEMM building block: C[M,N] = A[M,K] * B[N,K]^T with fp16-split
 * operands; returns 0 and fills d_c.  Used by tests to pin the UMMA descriptor layouts. */
int32_t neddf_tc_selftest(const float* d_a, const float* d_b, int32_t m, int32_t n, int32_t k,
                          float* d_c, void* stream);

/* Self-test of the "A operand in tensor memory" MMA form (weights written to TMEM with
 * tcgen05.st, activations MN-major in shared memory): C[128,128] = A[128,k] B[128,k]^T, averaged
 * over `reps` repeated accumulations; d_cycles[0] (optional) = SM cycles for reps*k/16*3 MMAs. */
int32_t neddf_tc_selftest_ts(const float* d_a, const float* d_b, int32_t k, float* d_c, int64_t* d_cycles,
                             int32_t reps, void* stream);

/* tcgen05 issue-rate microbenchmark (profiling aid): reps x 16 MMAs 128 x n x 16 on resident
 * shared-memory operands; a_mn / b_mn = 1 for MN-major operands, swizzle 0 (none) or 2 (128B).
 * d_cycles[0] = SM cycles to issue, d_cycles[1] = cycles until the last MMA completed. */
int32_t neddf_tc_mma_bench(int32_t a_mn, int32_t b_mn, int32_t swizzle, int32_t n, int32_t reps,
                           int64_t* d_cycles, void* stream);

/* Self-test of the CTA-pair MMA (tcgen05.mma.cta_group::2, cluster of two CTAs on one TPC):
 * C[256,n] = A[256,k] B[n,k]^T with A written to tensor memory by each CTA (rows 128r..128r+127) and
 * B MN-major in shared memory (CTA r holds rows (n/2)r..(n/2)(r+1)-1); averaged over `reps`
 * accumulations; d_cycles[0] (optional) = SM cycles for reps*k/16*3 MMAs.  Pins the operand split,
 * the multicast commit and the accumulator layout the pair kernel (field_tc2.cu) relies on. */
int32_t neddf_tc_pair_selftest(const float* d_a, const float* d_b, int32_t n, int32_t k, float* d_c,
                               int64_t* d_cycles, int32_t reps, void* stream);

/* Distributed-shared-memory store rate (profiling aid): every CTA of n_clusters CTA pairs writes
 * `bytes` x reps with 16-byte st.shared::cluster (mode 0 = own shared memory, 1 = both CTAs into the
 * peer, 2 = rank 0 into rank 1 only, 3 = like 1 with 512-byte blocks permuted).  d_cycles[cta]. */
int32_t neddf_dsmem_bench(int32_t mode, int32_t reps, int32_t bytes, int32_t n_clusters, int64_t* d_cycles,
                          void* stream);

/* tcgen05.cp layout probe (profiling / bring-up aid): one 128x256b shared-memory -> tensor-memory copy of
 * the 16-bit pattern value[i] = i with descriptor strides (lbo, sbo); d_out[128 lanes][8 columns]. */
int32_t neddf_tc_cp_probe(int32_t lbo, int32_t sbo, uint32_t* d_out, void* stream);

/* ------------------------------------------------------------------------------------------------
 * NeRF field variant (SURVEY 8(f) item 3; neddf/network/nerf.py).  Forward, fp32 CUDA-core kernel
 * (csrc/nerf.cu + csrc/nerf_train_kernel.cuh): the same renderer entry points (coarse_dists, composite, sample_pdf) serve it.
 * ------------------------------------------------------------------------------------------------ */
typedef struct neddf_nerf_config {
  int32_t embed_pos_rank;          /* nerf.py:36 (6 * rank <= 64) */
  int32_t embed_dir_rank;          /* nerf.py:37 (6 * rank <= 32) */
  int32_t layer_count;             /* nerf.py:38, 2..12 */
  int32_t layer_width;             /* nerf.py:39, must be 256 */
  int32_t activation_type;         /* NEDDF_ACT_* (nerf.py:40) */
  int32_t density_activation_type; /* NEDDF_ACT_* (nerf.py:41) */
  int32_t n_skips;                 /* nerf.py:42: ids of the layers AFTER which [h | embed_pos] is concatenated */
  int32_t skips[8];
} neddf_nerf_config_t;

typedef struct neddf_nerf neddf_nerf_t; /* opaque: config + packed device weights */

/* Number of linear layers and their [in,out] shapes in state_dict order layers.0 .. layers.{L-1}, outL_density,
 * outL_color.0, outL_color.2 (nerf.py:86-103).  shapes_out receives 2*n int32 (may be NULL). */
int32_t neddf_nerf_layer_shapes(const neddf_nerf_config_t* cfg, int32_t* shapes_out, int32_t max_layers);

/* NeRF.__init__ (nerf.py:34-105).  NEDDF_E_UNSUPPORTED for widths other than 256 or a skip after the last layer. */
int32_t neddf_nerf_create(const neddf_nerf_config_t* cfg, neddf_nerf_t** out);
void neddf_nerf_destroy(neddf_nerf_t* h);

/* Re-pack the weights: d_w[i] / d_b[i] are device pointers to torch nn.Linear tensors ([out,in] row-major and [out])
 * in the order of neddf_nerf_layer_shapes; n_layers = layer_count + 3.  Call after every change of the parameters. */
int32_t neddf_nerf_set_weights(neddf_nerf_t* h, const float* const* d_w, const float* const* d_b, int32_t n_layers,
                               void* stream);

/* NeRF.forward (nerf.py:107-165) on n samples given explicitly (Sampling.sample_pos / sample_dir / sample_var, each
 * [n,3]).  lowpass = host array [embed_pos_rank] of PositionalEncoding.get_lowpass_scale(lowpass_alpha)
 * (positional_encoding.py:67-89).  Outputs density [n], color [n,3] (raw, the renderer applies the range limits). */
int32_t neddf_nerf_forward(const neddf_nerf_t* h, const float* lowpass, const float* d_pos, const float* d_dir,
                           const float* d_var, int64_t n, float* d_density, float* d_color, void* stream);

/* Same with the sample geometry fused (Ray.get_sampling_points / get_sampling_cones, ray.py:88-194): rays [n_rays,3],
 * dists [n_rays, n_edges]; outputs [n_rays, n_edges] and [n_rays, n_edges, 3]. */
int32_t neddf_nerf_forward_rays(const neddf_nerf_t* h, const float* lowpass, const float* d_ray_dir, const float* d_ray_orig,
                                const float* d_dists, int64_t n_rays, int32_t n_edges, int32_t sampling_type,
                                float ray_radius, float* d_density, float* d_color, void* stream);

/* ------------------------------------------------------------------------------------------------
 * NeuS field variant (SURVEY 8(f) item 3; neddf/network/neus.py).  Forward only, fp32 CUDA-core kernel
 * (csrc/neus_simt.cu + csrc/neus_kernel.cuh + csrc/simt_mlp.cuh); the normal d sdf / d position, which the reference takes with
 * torch.autograd.grad (neus.py:133-142), is carried forward through the SDF trunk as three Jacobian rows.
 * ------------------------------------------------------------------------------------------------ */
typedef struct neddf_neus_config {
  int32_t embed_pos_rank;   /* neus.py:31 (6 * rank <= 64) */
  int32_t embed_dir_rank;   /* neus.py:32 (6 + 6 * rank <= 32) */
  int32_t sdf_layer_count;  /* neus.py:33, 1..12 */
  int32_t sdf_layer_width;  /* neus.py:34, must be 256 */
  int32_t col_layer_count;  /* neus.py:35, 1..12 (+ the 3-channel output layer) */
  int32_t col_layer_width;  /* neus.py:36, must be 256 */
  int32_t activation_type;  /* NEDDF_ACT_RELU | NEDDF_ACT_TANHEXP (neus.py:70-75) */
  int32_t n_skips;          /* neus.py:39: ids of the SDF layers AFTER which [h | embed_pos] is concatenated */
  int32_t skips[8];
} neddf_neus_config_t;

typedef struct neddf_neus neddf_neus_t; /* opaque: config + packed device weights */

/* Number of linear layers and their [in,out] shapes in state_dict order layers_sdf.0 .. layers_sdf.{Ls-1},
 * layers_col.0 .. layers_col.{Lc} (neus.py:83-98).  shapes_out receives 2*n int32 (may be NULL). */
int32_t neddf_neus_layer_shapes(const neddf_neus_config_t* cfg, int32_t* shapes_out, int32_t max_layers);

/* NeuS.__init__ (neus.py:29-99).  NEDDF_E_UNSUPPORTED for widths other than 256, activations other than
 * ReLU / tanhExp or a skip after the last SDF layer. */
int32_t neddf_neus_create(const neddf_neus_config_t* cfg, neddf_neus_t** out);
void neddf_neus_destroy(neddf_neus_t* h);

/* Re-pack the weights: d_w[i] / d_b[i] are device pointers to torch nn.Linear tensors ([out,in] row-major and [out])
 * in the order of neddf_neus_layer_shapes (n_layers = sdf_layer_count + col_layer_count + 1); d_variance = the
 * scalar `variance` parameter (neus.py:99).  Call after every change of the parameters. */
int32_t neddf_neus_set_weights(neddf_neus_t* h, const float* const* d_w, const float* const* d_b, int32_t n_layers,
                               const float* d_variance, void* stream);

/* NeuS.forward (neus.py:101-162) on n samples given explicitly (Sampling.sample_pos / sample_dir, each [n,3]; the
 * reference ignores the sample variance too).  Outputs sdf [n], density [n], color [n,3]; d_normal (may be NULL)
 * receives the gradient d sdf / d position [n,3] that feeds the colour trunk. */
int32_t neddf_neus_forward(const neddf_neus_t* h, const float* d_pos, const float* d_dir, int64_t n, float* d_sdf,
                           float* d_density, float* d_color, float* d_normal, void* stream);

/* Same with the sample geometry fused (Ray.get_sampling_points / get_sampling_cones, ray.py:88-194): rays [n_rays,3],
 * dists [n_rays, n_edges]; outputs [n_rays, n_edges] (x3 for color / normal). */
int32_t neddf_neus_forward_rays(const neddf_neus_t* h, const float* d_ray_dir, const float* d_ray_orig, const float* d_dists,
                                int64_t n_rays, int32_t n_edges, int32_t sampling_type, float ray_radius, float* d_sdf,
                                float* d_density, float* d_color, float* d_normal, void* stream);

/* ------------------------------------------------------------------------------------------------
 * NeRF field variant, training backward (the autograd graph of nerf.py:107-165 with respect to the parameters that
 * nerf_trainer.py:38-42 hands to Adam).  fp32 CUDA-core kernel (csrc/nerf.cu + csrc/nerf_train_kernel.cuh, the forward's tile
 * program): one launch recomputes the forward per 64-sample tile, walks back through the network and leaves the operands of the
 * weight-gradient GEMMs in global memory; the gradients themselves are neddf_wgrad / neddf_colsum_value_rows calls on
 * those buffers (what neddf_b200/nerf.py does).  STATUS: validated by the host emulation of its tile program only
 * (tests/test_nerf_train_emul.py); opt-in in the Python layer until it has been run on hardware.
 * ------------------------------------------------------------------------------------------------ */
typedef struct neddf_nerf_train neddf_nerf_train_t; /* opaque: config + forward and transposed weight packs */

int32_t neddf_nerf_train_create(const neddf_nerf_config_t* cfg, neddf_nerf_train_t** out);
void neddf_nerf_train_destroy(neddf_nerf_train_t* h);
/* Same arguments as neddf_nerf_set_weights. */
int32_t neddf_nerf_train_set_weights(neddf_nerf_train_t* h, const float* const* d_w, const float* const* d_b, int32_t n_layers,
                                     void* stream);

/* Backward of NeRF.forward on n explicit samples.  Upstream gradients d_g_density [n], d_g_color [n,3].  Outputs, all
 * fp32 row-major with the sample as the row: d_x [layer_count][n][256] hidden activations h_l, d_g [layer_count][n][256]
 * gradients of the hidden pre-activations, d_e [n][6 embed_pos_rank] / d_d [n][6 embed_dir_rank] the embeddings,
 * d_c1 / d_gc1 [n][256] activations / pre-activation gradients of outL_color.0 (columns >= 128 zero), d_gzd [n] gradient
 * of the density pre-activation.  Then, with in_0 = E, in_l = [h_{l-1} | E if l-1 in skips]:
 *   d layers.l.weight^T = in_l^T G_l, d layers.l.bias = colsum G_l, d outL_density.weight = GZD^T h_{L-1},
 *   d outL_color.0.weight^T = [h_{L-1} | D]^T GC1, d outL_color.2.weight = g_color^T C1. */
int32_t neddf_nerf_train_backward(const neddf_nerf_train_t* h, const float* lowpass, const float* d_pos, const float* d_dir,
                                  const float* d_var, int64_t n, const float* d_g_density, const float* d_g_color, float* d_x,
                                  float* d_g, float* d_e, float* d_d, float* d_c1, float* d_gc1, float* d_gzd, void* stream);
/* Same with the sample geometry fused (rays [n_rays,3], dists [n_rays, n_edges]; n = n_rays * n_edges). */
int32_t neddf_nerf_train_backward_rays(const neddf_nerf_train_t* h, const float* lowpass, const float* d_ray_dir,
                                       const float* d_ray_orig, const float* d_dists, int64_t n_rays, int32_t n_edges,
                                       int32_t sampling_type, float ray_radius, const float* d_g_density, const float* d_g_color,
                                       float* d_x, float* d_g, float* d_e, float* d_d, float* d_c1, float* d_gc1, float* d_gzd,
                                       void* stream);

#ifdef __cplusplus
}
#endif
#endif /* NEDDF_B200_H */

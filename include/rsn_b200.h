/* rsn_b200 -- C-ABI of the B200-native (sm_100a) per-ray rendering hot path of
 * 236088/reflect-sampling-nerf.
 *
 * The reference is pure Python on un-vendored nerfstudio and has NO native interface of its own
 * (SURVEY.md 2.3); each entry point below names the reference call site(s) whose eager-PyTorch work it
 * replaces (paths relative to /root/reference/reflect_sampling_nerf/).  INTEGRATION.md shows the ctypes
 * binding a maintainer of the reference adds.
 *
 * Conventions (SURVEY.md 8b):
 *   - every pointer is a DEVICE pointer to caller-owned memory (torch-allocated in the shipped host
 *     code); the library never allocates, frees or synchronises; work is enqueued on `stream`;
 *   - shapes are int64_t, tensors are dense row-major unless a stride argument says otherwise;
 *   - return value: 0 = ok, < 0 = bad argument, > 0 = cudaError_t; rsn_last_error() returns the
 *     thread-local message of the last failing call;
 *   - every data-path entry point is re-entrant (no mutable global state: no __constant__ parameters, no
 *     environment reads; the only process-wide state is an idempotent per-device cache of the SM count and of
 *     "max dynamic shared memory already opted in"), enqueues on `stream` only and is CUDA-graph capturable;
 *   - `n_rays_dev` (where present, may be NULL): a DEVICE int32 holding the number of valid rays; the launch is sized
 *     for the host-side capacity `n_rays` and processes min(*n_rays_dev, n_rays) rays.  This is how the bounce passes
 *     run without the host ever reading the number of masked rays (reflect_sampling_nerf_model.py:229,267-289 syncs);
 *   - built with -arch=sm_100a only.  Alternative kernel forms and timing ablations (RSN_* environment switches) and
 *     the tcgen05 probes exist only in the test build librsn_b200_dbg.so (include/rsn_b200_test.h).
 */
#ifndef RSN_B200_H
#define RSN_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct CUstream_st* rsn_stream_t; /* == cudaStream_t */

/* ---- housekeeping ------------------------------------------------------------------------------ */
int rsn_version(void);               /* 200 = 0.2.0 */
const char* rsn_last_error(void);
int rsn_device_ok(void);             /* 0 iff the current device is sm_100 */

/* ---- K1: spaced ray sampling ---------------------------------------------------------------------
 * Replaces UniformSampler / ReciprocalSampler.generate_ray_samples:
 *   reflect_sampling_nerf_model.py:109,111,148,292 ; reflect_sampling_nerf_components.py:14-36.
 * lin_bins [S+1] = torch.linspace(0,1,S+1); t_rand [N, t_rand_cols] stratification noise or NULL (eval);
 * spacing_kind 0 = uniform, 1 = reciprocal with s(x) = x / (1/tan + x) (the model uses tan = 0.25; ignored for kind 0).
 * Writes spacing and Euclidean bins [N,S+1].
 * Bit-exact with the oracle. */
int rsn_sample_spaced(const float* nears, const float* fars, const float* lin_bins, const float* t_rand,
                      int64_t t_rand_cols, int spacing_kind, float tan, float* spacing_bins, float* euclid_bins,
                      int64_t n_rays, int64_t n_samples, const int* n_rays_dev, rsn_stream_t stream);

/* ---- K2: PDF (importance) resampling -------------------------------------------------------------
 * Replaces PDFSampler(include_original=False).generate_ray_samples:
 *   reflect_sampling_nerf_model.py:110,112,182,317.
 * weights [N,S] (row stride given), spacing_bins_in [N,S+1], u_base [S'+1] (eval: already centred),
 * rand [N,S'+1] or NULL.  Writes new spacing / Euclidean bins [N,S'+1] and, if inds_out != NULL, the
 * searchsorted(side="right") indices (int64) for the bit-exact index test. */
int rsn_pdf_resample(const float* weights, int64_t weights_row_stride, const float* spacing_bins_in,
                     const float* nears, const float* fars, const float* u_base, const float* rand,
                     int spacing_kind, float tan, float histogram_padding, float* spacing_bins_out,
                     float* euclid_bins_out, int64_t* inds_out, int64_t n_rays, int64_t n_in_samples,
                     int64_t n_out_samples, const int* n_rays_dev, rsn_stream_t stream);

/* ---- K8: alpha compositing ------------------------------------------------------------------------
 * Replaces RaySamples.get_weights + Accumulation / RGB / Depth(median) / Normals / Semantic renderers:
 *   reflect_sampling_nerf_model.py:154-156,176,188-190,210,215-226,296,311,322,337,341.
 * sigma [N,S]; starts/ends point at element [0] of the per-ray start / end arrays with a common row
 * stride (pass bins and bins+1 with stride S+1 to composite straight from a bins array);
 * feat [N,S,C] per-sample channels, C in {0,1,3,4,8,16}.  Outputs: weights [N,S], accumulation [N],
 * depth_median [N], feat_out [N,C] = sum_s w*feat (background blending is the caller's per-ray op). */
int rsn_composite_fwd(const float* sigma, const float* starts, const float* ends, int64_t bin_row_stride,
                      const float* feat, int64_t n_channels, float* weights, float* accumulation,
                      float* depth_median, float* feat_out, int64_t n_rays, int64_t n_samples,
                      const int* n_rays_dev, rsn_stream_t stream);
/* Backward of the above w.r.t. sigma and feat.  grad_weights [N,S], grad_accumulation [N],
 * grad_feat_out [N,C] may each be NULL (= zero).  grad_feat may be NULL (not needed). */
int rsn_composite_bwd(const float* sigma, const float* starts, const float* ends, int64_t bin_row_stride,
                      const float* feat, int64_t n_channels, const float* grad_weights,
                      const float* grad_accumulation, const float* grad_feat_out, float* grad_sigma,
                      float* grad_feat, int64_t n_rays, int64_t n_samples, const int* n_rays_dev,
                      rsn_stream_t stream);

/* 16-channel form (the model's feature row).  Optional riders on the same pass over the samples:
 *  - normals [N,S,3] != NULL: the two per-sample normal losses of reflect_sampling_nerf_model.py:403-407, per ray
 *    pred_normal_loss = sum_s w_s |normals_s - feat_s[9:12]|^2 and orientation_loss = sum_s w_s max(0, feat_s[13])^2
 *    with w the (detached) compositing weights; the backward adds their gradients into grad_feat columns 9-11 and 13;
 *  - rgb_blend [N,3] != NULL: renderer_rgb's white-background blend and the clip after it (model.py:176-177,210-211),
 *    clip(feat_out[:, 0:3] + (1 - accumulation), 0, 1); its backward (grad_rgb_blend) needs the forward's feat_out and
 *    accumulation to rebuild the clip mask.
 * Backward: grad_* per-ray inputs may be NULL (= 0); grad_sigma == NULL skips the density gradient (the bounce passes
 * detach the weights, model.py:297,323). */
int rsn_composite16_fwd(const float* sigma, const float* starts, const float* ends, int64_t bin_row_stride,
                        const float* feat, const float* normals, float* weights, float* accumulation,
                        float* depth_median, float* feat_out, float* pred_normal_loss, float* orientation_loss,
                        float* rgb_blend, int64_t n_rays, int64_t n_samples, const int* n_rays_dev,
                        rsn_stream_t stream);
int rsn_composite16_bwd(const float* sigma, const float* starts, const float* ends, int64_t bin_row_stride,
                        const float* feat, const float* normals, const float* grad_weights,
                        const float* grad_accumulation, const float* grad_feat_out,
                        const float* grad_pred_normal_loss, const float* grad_orientation_loss,
                        const float* grad_rgb_blend, const float* feat_out, const float* accumulation,
                        float* grad_sigma, float* grad_feat, int64_t n_rays, int64_t n_samples, const int* n_rays_dev,
                        rsn_stream_t stream);

/* The upstream renderers' call forms take WEIGHTS (reflect_sampling_nerf_model.py:117-124,155-156,215-226; SURVEY.md
 * App. A.6): accumulation [N] = sum w, feat_out [N,C] = sum w feat (C <= 16; NULL/0 = none), depth_median [N] (needs
 * starts/ends as above; NULL = none).  API form behind components.*Renderer; the model uses rsn_composite16_fwd. */
int rsn_render_weights(const float* weights, const float* feat, int64_t n_channels, const float* starts,
                       const float* ends, int64_t bin_row_stride, float* accumulation, float* feat_out,
                       float* depth_median, int64_t n_rays, int64_t n_samples, rsn_stream_t stream);

/* ---- K3+K4+K5+K7: fused field forward --------------------------------------------------------------
 * Replaces, for one pass over the samples of a ray batch (mode 0), field.get_blob -> contract ->
 * get_density -> get_pred_normals / get_roughness / get_diff / get_tint -> IntegratedSHEncoding -> get_mid:
 *   reflect_sampling_nerf_field.py:90-186,203-207 ; reflect_sampling_nerf_components.py:52-140 ;
 *   call sites reflect_sampling_nerf_model.py:151-175,185-209,293-310,319-336
 * and, in mode 1, field.get_inf_color (reflect_sampling_nerf_field.py:190-201; model.py:290) with
 * dirs = w_r [N,3], area = sqradius [N], n_samples = 1 (origins/bins ignored).
 * wblob: bf16 weight blob of rsn_field_blob_bytes() bytes and bias: fp32 [rsn_field_bias_count()], both
 * produced by rsn_pack_field.  origins/dirs [N,3], area [N] (pixel_area), bins [N,S+1] Euclidean bin edges.
 * Outputs: sigma [N*S] (softplus density) and
 * feat [N*S,16]: 0-2 rgb = diff + tint*mid (mode 1: mid) | 3-5 diff | 6-8 tint | 9-11 pred_normal |
 * 12 sigmoid(roughness) | 13 n.d | 14 raw density | 15 softplus(roughness).
 * bf16 tensor-core MLP (tcgen05), fp32 encodings/heads. */
int rsn_field_forward(const void* wblob, const float* bias, int mode, const float* origins, const float* dirs,
                      const float* area, const float* bins, int64_t n_rays, int64_t n_samples, float* sigma,
                      float* feat, const int* n_rays_dev, rsn_stream_t stream);
/* Training form of rsn_field_forward: additionally writes the activation stash (rsn_field_stash_bytes(N*S)
 * bytes: per 128-point tile 41 bf16 block slots = IPE, the 8 hidden activations, bottleneck (unused), IDE, mid hidden,
 * followed by the ReLU bit masks; the encodings as swizzled shared-memory images, the activations as chunk-major images,
 * csrc/field_layout.cuh) that the normals / backward / wgrad kernels read, and aux [N*S,8] = mid rgb (3), raw normal head (3), raw roughness head, 1 spare.
 * (stash == NULL with aux != NULL: inference that also returns the raw mid colour.) */
int rsn_field_forward_train(const void* wblob, const float* bias, int mode, const float* origins,
                            const float* dirs, const float* area, const float* bins, int64_t n_rays,
                            int64_t n_samples, float* sigma, float* feat, void* stash, float* aux,
                            const int* n_rays_dev, rsn_stream_t stream);
int64_t rsn_field_stash_bytes(int64_t n_points);
/* The same network on caller-supplied Gaussians -- the reference's method-by-method Field API
 * (get_density(mean, cov) -> heads -> get_mid(directions, roughness, embedding), reflect_sampling_nerf_field.py:122-186):
 * mean [P,3], cov [P,3,3] (only the diagonal is read, as NeRFEncoding does), dirs [P,3] per point (IDE input and n.d),
 * rho_override [P] or NULL (NULL: softplus(roughness head), what the model feeds).  Outputs as rsn_field_forward;
 * aux [P,8] or NULL. */
int rsn_field_forward_points(const void* wblob, const float* bias, const float* mean, const float* cov,
                             const float* dirs, const float* rho_override, int64_t n_points, float* sigma, float* feat,
                             float* aux, rsn_stream_t stream);
/* field.get_blob (field.py:90-96; conical frustum -> Gaussian, SURVEY.md App. A.1): mean [N*S,3], FULL cov [N*S,3,3];
 * field.contract (field.py:98-119): contracted mean and J cov J with the diagonal ReLU.  API / test forms of the fused
 * kernel's prologue (the model never materialises them). */
int rsn_frustum_gaussians(const float* origins, const float* dirs, const float* pixel_area, const float* bins,
                          int64_t n_rays, int64_t n_samples, float* mean, float* cov, rsn_stream_t stream);
int rsn_contract(const float* mean, const float* cov, float* mean_out, float* cov_out, int64_t n_points,
                 rsn_stream_t stream);
/* Stand-alone encoders (component API + direct parity tests of the fused kernel's device functions):
 * NeRFEncoding(3, 16, 0, 16, include_input=True).forward(x, covs) (reflect_sampling_nerf_model.py:98-100; App. A.4):
 * x [P,3], cov [P,3,3] or NULL -> out99 [P,99];  IntegratedSHEncoding.forward (reflect_sampling_nerf_components.py:52-140):
 * dirs [P,3], roughness [P] -> out34 [P,34]. */
int rsn_ipe_encode(const float* x, const float* cov, float* out99, int64_t n_points, rsn_stream_t stream);
int rsn_ide_encode(const float* dirs, const float* roughness, float* out34, int64_t n_points, rsn_stream_t stream);

/* ---- K6: density-gradient normals -------------------------------------------------------------------
 * Replaces Field.get_normals = -normalize(d raw_density / d contracted mean) (autograd.grad through the
 * density head, the 8 base layers and the IPE with the covariance held constant):
 *   reflect_sampling_nerf_field.py:125-127,134-135,146-147 ; reflect_sampling_nerf_model.py:159-160,194-195.
 * wblob_t: transposed bf16 weight blob (rsn_field_blob_t_bytes()), wd_bf16: the density head row as 256 bf16,
 * x_stash: the stash of the forward pass.  Output normals [N*S,3]. */
int rsn_field_normals(const void* wblob_t, const void* wd_bf16, const void* x_stash, int64_t n_rays,
                      int64_t n_samples, float* normals, rsn_stream_t stream);
int64_t rsn_field_blob_t_bytes(void);

/* ---- K5 backward, dgrad chain -----------------------------------------------------------------------
 * Replaces the autograd backward of reflect_sampling_nerf_field.py:122-186 (mode 0) / 190-201 (mode 1) for one
 * pass: from g_sigma [N*S] = dL/d sigma and g_feat [N*S,16] = dL/d feat (forward layout; columns 14,15 are
 * ignored; g_sigma may be NULL = zero) to the pre-activation gradient of every Linear, written to dy_stash
 * (rsn_field_dy_stash_bytes; chunk-major bf16 block images, csrc/field_layout.cuh) for rsn_field_wgrad.  feat / aux are the forward outputs.  If g_area != NULL the chain continues through layer 0
 * and the IPE damping and writes dL/d pixel_area (mode 0) or dL/d sqradius (mode 1) of every POINT [N*S]
 * (the caller sums over the samples of a ray): the roughness -> cone width path of
 * reflect_sampling_nerf_model.py:272,286,290. */
int rsn_field_backward(const void* wblob_t, const void* x_stash, int mode, const float* origins, const float* dirs,
                       const float* area, const float* bins, int64_t n_rays, int64_t n_samples,
                       const float* g_sigma, const float* g_feat, const float* feat, const float* aux,
                       void* dy_stash, float* g_area, const int* n_rays_dev, rsn_stream_t stream);
int64_t rsn_field_dy_stash_bytes(int64_t n_points);

/* ---- K5 backward, wgrad -----------------------------------------------------------------------------
 * dW = dY^T X and db = sum dY of every Linear of the field over all points of a pass, ACCUMULATED into grad_blob,
 * whose regions rsn_field_wgrad_layout describes (HOST pointers: offsets[2j] = dW offset, offsets[2j+1] = db offset
 * or -1, shapes[2j], shapes[2j+1] = rows, cols; returns the job count).  workspace (rsn_field_wgrad_workspace_bytes,
 * 16-byte aligned, no initial contents) holds the per-CTA partial sums, added into grad_blob in a fixed order: the
 * same inputs give the same gradient every run.  One workspace per launch in flight.
 * n_rays_dev != NULL: the pass covers min(*n_rays_dev * points_per_ray, n_points) points. */
int rsn_field_wgrad(const void* x_stash, const void* dy_stash, int64_t n_points, float* grad_blob, void* workspace,
                    const int* n_rays_dev, int64_t points_per_ray, rsn_stream_t stream);
int64_t rsn_field_wgrad_workspace_bytes(void);
int rsn_field_wgrad_layout(int64_t* host_offsets, int64_t* host_shapes, int64_t* total_floats);

/* Completes the gradient blob once per step, after the last rsn_field_wgrad (and after the all-reduce): the bottleneck
 * layer is linear in h7 and feeds only the mid layer, so the kernels stash neither its activations nor their gradients;
 * with G = dY_mid^T h7 (rows 64-191 of job 10's region) this fills dW/db of field_output_bottleneck (job 9's region) =
 * Wmb^T G, Wmb^T db_mid and job 12's region = the bottleneck columns of d mlp_mid.layers.0.weight = G Wb^T + db_mid bb^T
 * (and db_mid).
 * w_bott [256][256], b_bott [256], w_mid [128][290]: the fp32 parameters (field.py:54-86), device pointers. */
int rsn_field_wgrad_finish(float* grad_blob, const float* w_bott, const float* b_bott, const float* w_mid,
                           rsn_stream_t stream);
/* Gradient blob -> flat fp32 gradient vector laid out parameter after parameter in rsn_pack_field order
 * (rsn_field_flat_layout: HOST array of 32 float offsets, returns the vector length, 617,742).  One launch. */
int rsn_unpack_grads(const float* grad_blob, float* flat_grads, rsn_stream_t stream);
int64_t rsn_field_flat_layout(int64_t* host_offsets32);

int64_t rsn_field_blob_bytes(void);
/* Packs the 32 fp32 parameter tensors of the field (HOST array of DEVICE pointers, order documented in
 * csrc/pack.cu: base weights 0-7, base biases 8-15, bottleneck, mid, rgb, density, normals, roughness, diff,
 * tint -- weight then bias each; names of reflect_sampling_nerf_field.py:54-86) into the forward blob, the
 * transposed blob, the bias vector and the bf16 density row.  Derived state: call after every optimizer step. */
int rsn_pack_field(const float* const* params, void* wblob, void* wblob_t, float* bias, void* wd_bf16,
                   rsn_stream_t stream);
int64_t rsn_field_bias_count(void);
/* The 16 IPE frequencies 2**linspace(0,16,16) the kernels use (HOST pointer; for the table test). */
int rsn_ipe_freqs(float* host_out16);

/* ---- fused optimizer step (SURVEY.md 8 f2) -------------------------------------------------------------
 * Replaces torch.optim.RAdam(lr 1e-3, eps 1e-15) + ExponentialDecay(lr_final 1e-4, max_steps 50000) as configured at
 * reflect_sampling_nerf_config.py:50-53, for the 32 parameters above in ONE launch: params32 = HOST array of DEVICE
 * pointers (rsn_pack_field order), flat_grad = rsn_unpack_grads output (scaled by grad_scale = 1 / world_size for data
 * parallel averaging), exp_avg / exp_avg_sq = flat fp32 state, step_dev = DEVICE int64 steps taken so far (incremented
 * by the launch: the step number never visits the host), counter_dev = DEVICE uint32 zeroed once, lr_out_dev = DEVICE
 * float receiving the learning rate used or NULL.  lr_final <= 0 = constant lr.  Follows torch's foreach RAdam
 * arithmetic (1e-6 parity over 100 steps).  Call rsn_pack_field afterwards. */
int rsn_radam_step(float* const* params32, const float* flat_grad, float* exp_avg, float* exp_avg_sq,
                   long long* step_dev, unsigned int* counter_dev, float* lr_out_dev, double lr_init, double lr_final,
                   long long max_steps, double beta1, double beta2, double eps, float grad_scale, rsn_stream_t stream);

/* ---- losses (SURVEY.md 8 a19) ---------------------------------------------------------------------------
 * Replaces ReflectSamplingNeRFModel.get_loss_dict (reflect_sampling_nerf_model.py:395-429): out9[0..7] = the eight
 * scaled terms in the reference's dict order (loss_mid_coarse, loss_mid_fine, loss_reflect_mid_coarse,
 * loss_reflect_mid_fine, predicted_normal_loss_coarse, predicted_normal_loss_fine, orientation_loss_coarse,
 * orientation_loss_fine), out9[8] = their sum.  Predictions and image [N,3]; pnl_* / ol_* [N] = per-ray sums of
 * rsn_composite16_fwd (NULL = term is 0); coef8 = DEVICE coefficients; workspace = rsn_loss_workspace_bytes() bytes,
 * zeroed once by the caller.  Backward: grad_terms8 [8] and / or grad_total [1] (DEVICE, either may be NULL). */
int64_t rsn_loss_workspace_bytes(void);
int rsn_loss_fwd(const float* mid_rgb_coarse, const float* mid_rgb_fine, const float* mid_reflect_coarse,
                 const float* mid_reflect_fine, const float* image, const float* pnl_coarse, const float* pnl_fine,
                 const float* ol_coarse, const float* ol_fine, const float* coef8, float* out9, void* workspace,
                 int64_t n_rays, rsn_stream_t stream);
int rsn_loss_bwd(const float* mid_rgb_coarse, const float* mid_rgb_fine, const float* mid_reflect_coarse,
                 const float* mid_reflect_fine, const float* image, const float* coef8, const float* grad_terms8,
                 const float* grad_total, float* g_mid_rgb_coarse, float* g_mid_rgb_fine, float* g_mid_reflect_coarse,
                 float* g_mid_reflect_fine, float* g_pnl_coarse, float* g_pnl_fine, float* g_ol_coarse, float* g_ol_fine,
                 int64_t n_rays, rsn_stream_t stream);

/* ---- K9: reflection set-up, device-side compaction, reflected bundle, composition of the bounce ------------
 * rsn_reflect_setup replaces reflect_sampling_nerf_model.py:215-229,267-271: from the composited feature row of the fine
 * pass comp16 [N,16] (rsn_field_forward feature layout), accumulation [N], median depth [N] and the rays, per ray:
 * diff [N,3] (white-blended), tint [N,3], normal [N,3] (safe-normalised), n_dot_d [N], mask [N] (uint8:
 * accumulation > 1e-2 and n.d < 0), bounce origins o + depth d and directions normalize(d - 2 (n.d) n).  clamp01 =
 * eval mode (RGBRenderer clamps).
 * rsn_reflect_compact replaces the boolean-mask indexing `x[mask, :]` (model.py:267-289, a host sync each): idx [N]
 * (int64; the first *count entries = ascending indices of the masked rays), inv [N] (int32; rank of ray r among the
 * masked rays, or -1), count [1] (int32) -- all on the device.
 * rsn_reflect_bundle_fwd gathers the reflected RayBundle of the masked rays (model.py:267-289): origins / dirs [cap,3],
 * sqradius = 2 |n.d| roughness^2 (model.py:272; roughness = comp16[:, 12]) and pixel_area = pi sqradius [cap];
 * rsn_reflect_bundle_bwd is its gradient w.r.t. the roughness as a full grad_comp16 [N,16] (zero but column 12).
 * rsn_reflect_compose_* replace model.py:240-241,311-313,337-339: out[r] = 1 - acc_fine[r] for rays that do not bounce,
 * else clip(diff[r] + tint[r] * (comp[j,:3] + bg[j] (1 - acc_r[j])), 0, 1), j = inv[r]; depth_out [N] (optional) =
 * depth_r[j] or 0: the padded outputs["depth_reflect_fine"].  Backward: grad_comp16 [cap,16] (rows < count written in
 * full), grad_bg [cap,3], grad_acc_fine [N]. */
int rsn_reflect_setup(const float* comp16, const float* acc, const float* depth, const float* origins, const float* dirs,
                      int clamp01, float* diff, float* tint, float* normal, float* n_dot_d, uint8_t* mask,
                      float* bounce_origins, float* bounce_dirs, int64_t n_rays, rsn_stream_t stream);
int rsn_reflect_compact(const uint8_t* mask, int64_t* idx, int32_t* inv, int32_t* count, int64_t n_rays,
                        rsn_stream_t stream);
int rsn_reflect_bundle_fwd(const int64_t* idx, const int32_t* count, const float* bounce_origins_all,
                           const float* bounce_dirs_all, const float* n_dot_d, const float* comp16, float* origins,
                           float* dirs, float* sqradius, float* pixel_area, int64_t n_rays, rsn_stream_t stream);
int rsn_reflect_bundle_bwd(const int32_t* inv, const float* n_dot_d, const float* comp16, const float* grad_sqradius,
                           const float* grad_pixel_area, float* grad_comp16, int64_t n_rays, rsn_stream_t stream);
int rsn_reflect_compose_fwd(const float* acc_fine, const float* diff, const float* tint, const int32_t* inv,
                            const float* comp, int64_t comp_ld, const float* bg, const float* acc_r, int clamp_inner,
                            float* out, const float* depth_r, float* depth_out, int64_t n_rays, rsn_stream_t stream);
int rsn_reflect_compose_bwd(const float* grad_out, const float* diff, const float* tint, const int32_t* inv,
                            const float* comp, int64_t comp_ld, const float* bg, const float* acc_r, float* grad_comp16,
                            float* grad_bg, float* grad_acc_fine, int64_t n_rays, rsn_stream_t stream);

/* ---- pixel sampling + ray generation + target gather (SURVEY.md 8 f1) ------------------------------------
 * Replaces reflect_sampling_nerf_datamanager.py:49-58 (PixelSampler.sample_method -> RayGenerator ->
 * Cameras.generate_rays, perspective, no distortion; Blender alpha blend onto white).  c2w [V,3,4], intrinsics [V,4] =
 * fx, fy, cx, cy; exactly one of rand3 [N,3] (uniform [0,1): (cam, y, x) = floor(rand * (V, H, W))) or pixels_in [N,3]
 * (int64 cam, y, x); images [V,H,W,C] uint8 (C = 3 or 4) or NULL.  Outputs origins / dirs [N,3], pixel_area [N],
 * pixels_out [N,3] (int64) or NULL, target_rgb [N,3] (when images).  Bit-exact with oracle/cameras.py. */
int rsn_raygen(const float* c2w, const float* intrinsics, const float* rand3, const int64_t* pixels_in,
               const uint8_t* images, int64_t n_channels, int64_t n_views, int64_t height, int64_t width, float* origins,
               float* dirs, float* pixel_area, int64_t* pixels_out, float* target_rgb, int64_t n_rays,
               rsn_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* RSN_B200_H */

/* b200gs -- training-step kernels around the rasterizer (SURVEY.md section 8(f), rows 1 and 3).
 *
 * These are the callers on either side of the rasterizer hot path inside one SDP-GS training iteration
 * (train.py:93-231).  Same C-ABI rules as b200gs.h: plain device pointers, caller-owned memory, explicit stream,
 * nothing allocated, 0 / negative B200GS_E_* return codes.
 *
 * What each entry point replaces in the reference:
 *   b200gs_photometric_loss   <- Ll1 = l1_loss_mask(image, gt); loss = (1-l)*Ll1 + l*(1 - ssim(image, gt))
 *                                train.py:98-100, utils/loss_utils.py:119-163 (11x11 Gaussian window, sigma 1.5,
 *                                zero padding, C1 = 0.01^2, C2 = 0.03^2, mean over 3*H*W) -- value AND dL/dimage
 *   b200gs_depth_pearson_loss <- depth_loss = min(1 - pearson(depth_mono, depth), 1 - pearson(1/(200 - depth_mono), depth))
 *                                train.py:115-131 (torchmetrics pearson_corrcoef) -- value AND dL/ddepth
 *   b200gs_param_step         <- the activations of scene/gaussian_model.py:44-57, 145-160 (exp / sigmoid / normalize)
 *                                with their backward, torch.optim.Adam(eps=1e-15) over the parameter groups of
 *                                scene/gaussian_model.py:228-267 (one fused launch instead of ~7 x 10 kernels),
 *                                and add_densification_stats + max_radii2D (train.py:218-221, gaussian_model.py:610-612)
 */
#ifndef B200GS_TRAIN_H_
#define B200GS_TRAIN_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* Hyper-parameters that change from step to step live in DEVICE memory, so a captured CUDA graph can be replayed:
 * the caller writes the block once, b200gs_hparams_advance() moves it to the next iteration on the device. */
typedef struct b200gs_hparams {
	float step;            /* Adam step count t (1-based) of THIS update */
	float lr_xyz, lr_f_dc, lr_f_rest, lr_opacity, lr_scaling, lr_rotation, lr_feature;
	float beta1, beta2, eps;
	float lambda_dssim;    /* train.py:100 */
	float depth_weight;    /* train.py:131 */
	float pad[3];
} b200gs_hparams_t;       /* 64 bytes */

/* Raw (pre-activation) parameters, their Adam moments and the gradients w.r.t. the ACTIVATED values the rasterizer
 * consumed.  All device f32, contiguous.  NULL feature pointers = no language-feature group. */
typedef struct b200gs_param_state {
	int32_t P;
	float* xyz;         float* m_xyz;      float* v_xyz;      const float* g_xyz;       /* [P,3]              identity */
	float* shs;         float* m_shs;      float* v_shs;      const float* g_shs;       /* [P,16,3]  f_dc = [:,0], f_rest = [:,1:] */
	float* opacity;     float* m_opacity;  float* v_opacity;  const float* g_opacity;   /* [P,1]  raw; g is dL/d sigmoid(raw) */
	float* scaling;     float* m_scaling;  float* v_scaling;  const float* g_scaling;   /* [P,3]  raw; g is dL/d exp(raw)     */
	float* rotation;    float* m_rotation; float* v_rotation; const float* g_rotation;  /* [P,4]  raw; g is dL/d normalize(raw) */
	float* feature;     float* m_feature;  float* v_feature;  const float* g_feature;   /* [P,3]              identity */
	/* activated copies rewritten after the update (what the next forward reads) */
	float* opacity_act;  /* [P,1] sigmoid */
	float* scaling_act;  /* [P,3] exp */
	float* rotation_act; /* [P,4] normalize */
	/* densification statistics (may be NULL to skip) */
	const float* g_means2D;      /* [P,3] viewspace gradient of this step */
	const int32_t* radii;        /* [P]   of this step's view */
	float* xyz_gradient_accum;   /* [P,1] += ||g_means2D[:, :2]|| where radii > 0 */
	float* denom;                /* [P,1] += 1 where radii > 0 */
	int32_t* max_radii2D;        /* [P]   = max(., radii) where radii > 0 */
} b200gs_param_state_t;

/* One fused launch: chain rule through the activations, Adam update, re-activation, densification statistics.
 * `update` == 0 only refreshes the activated copies from the raw parameters (no gradient needed); 2 = densification
 * statistics only (train.py:218-231 on a densify iteration: the parameters were just re-created, optimizer.step() is a no-op).
 * Add B200GS_STEP_AFTER_FOREIGN (4) when the previous operation in the stream is NOT one of this library's kernels (an NCCL
 * all-reduce, a copy, a torch kernel): the launch then uses full stream ordering instead of a programmatic dependent launch. */
#define B200GS_STEP_AFTER_FOREIGN 4
/* sizeof(b200gs_param_state_t), sizeof(b200gs_hparams_t): checked by bindings at load time */
void b200gs_train_abi_sizes(int64_t* out2);

int b200gs_param_step(const b200gs_param_state_t* s, const b200gs_hparams_t* hp_device, int32_t update, void* stream);

/* End of an iteration: step += 1 and lr_xyz = the exponential position schedule of utils/general_utils.py:
 * get_expon_lr_func(lr_init, lr_final, lr_delay_steps = 0, lr_delay_mult, max_steps) (scene/gaussian_model.py:276-285)
 * evaluated at the iteration just finished -- the reference calls update_learning_rate(iteration) after
 * optimizer.step() (train.py:230-233), so Adam step t runs at the rate of iteration t-1 -- on the device, so that
 * a captured step never waits for the host. */
int b200gs_hparams_advance(b200gs_hparams_t* hp_device, float lr_init, float lr_final, float lr_delay_mult,
                           float max_steps, void* stream);

/* loss_out (device f64[4]): [0] = (1-l)*L1 + l*(1-SSIM) (assigned: the depth losses add to it afterwards), [1] L1, [2] SSIM
 * (both means), written by the last block.
 * scratch: device f32[3*3*H*W] (the three derivative maps).  dL_dimage: device f32[3,H,W], fully written.
 * accum: device f64[b200gs_loss_accum_doubles()], must be zero on entry (the kernel leaves it zero on exit); partial
 * sums are spread over 64 lines so that the per-block atomics do not serialise in L2. */
int b200gs_photometric_loss(const float* image, const float* gt, int32_t width, int32_t height,
                            const b200gs_hparams_t* hp_device, float* scratch, double* accum, double* loss_out,
                            float* dL_dimage, void* stream);
size_t b200gs_photometric_scratch_bytes(int32_t width, int32_t height);
size_t b200gs_loss_accum_doubles(void);

/* loss_out[3] = depth_weight * depth_loss is ADDED to loss_out[0]; dL_ddepth: device f32[H*W], fully written.
 * accum: its own device f64[b200gs_loss_accum_doubles()], zero on entry, left zero on exit (the last few words carry
 * the gradient coefficients from the reduction kernel to the gradient kernel). */
int b200gs_depth_pearson_loss(const float* depth, const float* depth_mono, int32_t n,
                              const b200gs_hparams_t* hp_device, double* accum, double* loss_out,
                              float* dL_ddepth, void* stream);

/* The pseudo-view form of the same loss (train.py:138-153: a second render from an unobserved pose, supervised by a
 * monocular depth estimate): loss_out[3] = w * (1 - pearson(depth, depth_ref)) is ADDED to loss_out[0], with
 * w = *weight_device (loss_scale * depth_pseudo_weight, its own device word so that the ramp of train.py:150 needs no
 * re-capture) or hp->depth_weight when weight_device is NULL; single_branch != 0 selects the single correlation
 * (pass depth_ref = -midas), 0 the min over (depth_ref, 1 / (200 - depth_ref)) of the training views. */
int b200gs_depth_pearson_loss_pseudo(const float* depth, const float* depth_ref, int32_t n, const b200gs_hparams_t* hp_device,
                                     const float* weight_device, int32_t single_branch, double* accum, double* loss_out,
                                     float* dL_ddepth, void* stream);

/* Exact 3 nearest neighbours of every point (self excluded): what the proximity densification of SDP-GS reads from
 * its simple_knn fork (`dist, nearest_indices = distCUDA2(xyz)`, scene/gaussian_model.py:513-516; the extension is not
 * vendored under /root/reference, SURVEY.md F5).  mean_dist2[i] = mean of the three squared distances (simple_knn's
 * definition), indices[i] = the neighbours in order of increasing distance (ties: lower index first).
 * Tiled brute force, O(P^2 / 1024) shared-memory passes: the faster choice for small clouds, and the reference that
 * b200gs_knn3_tree is tested against.  Points with a non-finite coordinate are nobody's neighbour; a point with fewer than
 * three finite neighbours within squared distance 3e38 gets index -1 and distance 3e38 in the missing places. */
int b200gs_knn3(int32_t P, const float* xyz, float* mean_dist2, int32_t* indices, void* stream);

/* Bytes of device scratch b200gs_knn3_tree needs for P points (0 when P is out of range). */
size_t b200gs_knn3_scratch_bytes(int32_t P);
/* Same outputs, bit for bit, as b200gs_knn3 on every input; O(P log P) work (Morton-ordered implicit box hierarchy,
 * knn.cu); no host synchronisation, so the call can be captured in a CUDA graph.
 * 4 <= P < 2^30 (the onesweep look-back counters); scratch needs no initialisation.  B200GS_E_ARG, with nothing launched,
 * when P is out of range, a pointer is NULL or scratch_bytes < b200gs_knn3_scratch_bytes(P). */
int b200gs_knn3_tree(int32_t P, const float* xyz, float* mean_dist2, int32_t* indices,
                     void* scratch, size_t scratch_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* B200GS_TRAIN_H_ */

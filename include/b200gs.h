/* b200gs -- Blackwell-native (sm_100a) differentiable Gaussian-splatting rasterizer.
 *
 * C-ABI drop-in boundary for the rasterizer hot path of dengyangyan/SDP-GS.  Plain
 * pointers and sizes only; no torch / C++ types.  Every pointer marked "device" is a
 * CUDA device pointer owned by the caller; the library never allocates device memory.
 * All work is enqueued on the `stream` argument (a cudaStream_t passed as void*).
 *
 * What each entry point replaces in the reference ("DGR" = submodules/diff-gaussian-rasterization):
 *   b200gs_forward*      <- CudaRasterizer::Rasterizer::forward   DGR/cuda_rasterizer/rasterizer.h:31-53,
 *                           bound by RasterizeGaussiansCUDA        DGR/rasterize_points.cu:35-115 (pybind: DGR/ext.cpp:16)
 *   b200gs_backward      <- CudaRasterizer::Rasterizer::backward  DGR/cuda_rasterizer/rasterizer.h:55-84,
 *                           bound by RasterizeGaussiansBackwardCUDA DGR/rasterize_points.cu:117-196 (DGR/ext.cpp:17)
 *   b200gs_backward_camera  the same, plus gradients w.r.t. viewmatrix / projmatrix / campos (no reference counterpart)
 *   b200gs_mark_visible  <- CudaRasterizer::Rasterizer::markVisible DGR/cuda_rasterizer/rasterizer.h:24-29,
 *                           bound by markVisible                   DGR/rasterize_points.cu:198-217 (DGR/ext.cpp:18)
 *   b200gs_*_bytes       <- CudaRasterizer::required<T>()          DGR/cuda_rasterizer/rasterizer_impl.h:66-72
 *                           (the three growable byte workspaces, rasterize_points.cu:70-77)
 *   b200gs_view_t        <- GaussianRasterizationSettings          DGR/diff_gaussian_rasterization/__init__.py:157-169
 *                           plus SDP-GS's include_feature/confidence, gaussian_renderer/__init__.py:228-243
 *
 * Conventions kept from the reference: viewmatrix/projmatrix are the row-major storage of
 * the TRANSPOSED matrices (element (r,c) at m[4c+r], scene/cameras.py:78-80); a NULL pointer
 * means "input absent" exactly as an empty tensor does there (forward.cu:205,241); colours
 * are CHW; radii are int32; means2D gradients are in NDC units (x 0.5W, 0.5H).
 *
 * Return value: 0 on success, negative B200GS_E_* otherwise; b200gs_last_error() describes it.
 */
#ifndef B200GS_H_
#define B200GS_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200GS_VERSION 100

#define B200GS_OK 0
#define B200GS_E_ARG (-1)       /* bad argument (shape, missing required input, workspace too small) */
#define B200GS_E_CUDA (-2)      /* a CUDA call or kernel failed (checked after every stage when debug!=0) */
#define B200GS_E_OVERFLOW (-3)  /* num_rendered exceeded the binning capacity (only reported by *_status) */

/* Per-view constants. */
typedef struct b200gs_view {
	int32_t width, height;
	float tan_fovx, tan_fovy;
	float scale_modifier;
	int32_t sh_degree;       /* active SH degree D (0..3) */
	int32_t sh_coeffs;       /* M = coefficients per channel in `shs` (0 when shs == NULL) */
	int32_t prefiltered;     /* reference semantics: a culled Gaussian is then a fatal error (auxiliary.h:156-160) */
	int32_t debug;           /* !=0: synchronize + check after every stage (auxiliary.h:166-173) */
	int32_t extended;        /* 0: vanilla (color, radii); 1: SDP-GS (color, depth, alpha, feature, radii) */
	const float* background; /* device f32[3] */
	const float* viewmatrix; /* device f32[16] */
	const float* projmatrix; /* device f32[16] */
	const float* campos;     /* device f32[3] */
} b200gs_view_t;

/* Per-Gaussian inputs (device, contiguous f32).  Exactly one of shs / colors_precomp, and exactly
 * one of (scales, rotations) / cov3D_precomp, as GaussianRasterizer.forward enforces
 * (DGR/diff_gaussian_rasterization/__init__.py:191-195). */
typedef struct b200gs_gaussians {
	int32_t P;
	const float* means3D;        /* [P,3] */
	const float* shs;            /* [P,M,3] or NULL */
	const float* colors_precomp; /* [P,3]   or NULL */
	const float* opacities;      /* [P,1] */
	const float* scales;         /* [P,3]   or NULL */
	const float* rotations;      /* [P,4]   or NULL (unit quaternions r,x,y,z; NOT re-normalised, forward.cu:127) */
	const float* cov3D_precomp;  /* [P,6]   or NULL */
	/* SDP-GS extensions (used only when view.extended != 0) */
	const float* language_feature_precomp; /* [P,3] or NULL */
	const float* shs_language;             /* [P,3] degree-0 SH of the feature head, or NULL; feature =
	                                          normalize(C0*shs_language) as gaussian_renderer/__init__.py:283-287 */
	const float* confidence;               /* [P,1] or NULL (== all ones); multiplies opacity, no gradient */
	/* Optional (NULL: all P rows are Gaussians).  Device word holding the number of live rows: rows >= *live_count are
	 * treated as culled (radius 0, no instances, zero gradients).  For capacity-sized parameter buffers whose Gaussian count
	 * changes on the device (densify / prune, scene/gaussian_model.py:400-608) while P, the launch geometry and any CUDA
	 * graph that captured this call stay fixed. */
	const uint32_t* live_count;
} b200gs_gaussians_t;

typedef struct b200gs_outputs {
	float* color;   /* device f32[3,H,W] */
	float* depth;   /* device f32[1,H,W]  (extended only) */
	float* alpha;   /* device f32[1,H,W]  (extended only) */
	float* feature; /* device f32[3,H,W]  (extended only) */
	int32_t* radii; /* device i32[P] */
} b200gs_outputs_t;

/* The three opaque byte workspaces saved between forward and backward, as in the reference
 * (geomBuffer, binningBuffer, imgBuffer).  Sizes from the *_bytes functions below; 256-B aligned. */
typedef struct b200gs_workspace {
	void* geom;
	size_t geom_bytes;
	void* binning;
	size_t binning_bytes;
	void* image;
	size_t image_bytes;
	/* persistent != 0: the caller keeps these workspaces (and b200gs_grads_t.scratch) alive across calls, initialised them
	 * once with b200gs_workspace_init, and lets nothing else write to them.  The kernels then leave every counter,
	 * histogram and look-back word they consumed zeroed for the next call (and the backward re-zeroes the scratch rows it
	 * read), so no call issues a memset -- the steady state of a training loop (CUDA-graph sessions).  A persistent image
	 * workspace also carries, per tile, what its blend units cost in the previous call; the next call launches the units
	 * heaviest first by that measure (scheduling only: results do not depend on it).  0: fresh or foreign memory; every call
	 * zeroes what it needs first (the eager autograd path, which allocates per call) and orders the units by list length. */
	int32_t persistent;
	int32_t reserved_;
} b200gs_workspace_t;

/* Cotangents of the outputs (device, CHW).  NULL == zero. */
typedef struct b200gs_grad_outputs {
	const float* dL_dcolor;   /* [3,H,W] */
	const float* dL_ddepth;   /* [1,H,W] */
	const float* dL_dalpha;   /* [1,H,W] */
	const float* dL_dfeature; /* [3,H,W] */
} b200gs_grad_outputs_t;

/* Gradients w.r.t. the inputs (device).  Every non-NULL buffer is fully written (zeros for
 * Gaussians with radii == 0), so the caller may pass uninitialised memory -- this replaces the
 * nine torch::zeros fills of rasterize_points.cu:151-159.  `scratch` is P*64 bytes of device
 * memory the blend backward accumulates into (contents on return are unspecified). */
typedef struct b200gs_grads {
	float* dL_dmeans3D;       /* [P,3] */
	float* dL_dmeans2D;       /* [P,3] (x,y used; NDC units) */
	float* dL_dshs;           /* [P,M,3] or NULL */
	float* dL_dcolors;        /* [P,3]   or NULL (for colors_precomp) */
	float* dL_dopacities;     /* [P,1] */
	float* dL_dscales;        /* [P,3]   or NULL */
	float* dL_drotations;     /* [P,4]   or NULL */
	float* dL_dcov3D;         /* [P,6]   or NULL (for cov3D_precomp) */
	float* dL_dfeatures;      /* [P,3]   or NULL (language_feature_precomp) */
	float* dL_dshs_language;  /* [P,3]   or NULL */
	void* scratch;            /* P*64 bytes; with ws->persistent: all zeros on entry, all zeros again on return */
	/* Image-parallel training (include/b200gs_collective.h): when scatter_bases != NULL the six parameter-gradient arrays
	 * (means3D, shs [M = 16], opacities, scales, rotations, features / shs_language) are NOT written to the pointers above
	 * but pushed, 128-Gaussian tile by tile, over NVLink into the staging buffer of the rank that owns the tile
	 * (rank o owns Gaussians [o * shard_rows, (o+1) * shard_rows), shard_rows % 128 == 0): the reduce-scatter half of the
	 * gradient exchange rides inside the preprocess-backward kernel.  scatter_bases: DEVICE array [world] of peer-mapped
	 * staging base pointers (b200gs_gather_reduce_f32 describes the layout).  dL_dmeans2D stays local. */
	void* const* scatter_bases;
	int64_t scatter_shard_rows;
	int32_t scatter_rank, scatter_world;
	/* accumulate != 0: the six parameter-gradient arrays receive (their current contents + this view's gradient) instead of
	 * being overwritten -- several views per optimizer step (image-parallel training with more views than ranks).  With
	 * scatter_bases set, the sum of the local arrays and this view's gradient is what gets pushed (the local arrays
	 * themselves are left alone): accumulate locally for all but the rank's last view, push on the last one.
	 * 8-byte padding keeps the struct size a multiple of 8. */
	int32_t accumulate;
	int32_t reserved_;
} b200gs_grads_t;

int b200gs_version(void);
const char* b200gs_last_error(void);

size_t b200gs_geom_bytes(int32_t P);
size_t b200gs_image_bytes(int32_t width, int32_t height);
size_t b200gs_binning_bytes(int64_t capacity, int32_t width, int32_t height); /* capacity = max number of (Gaussian,tile)
                                                  instances, < 2^30; the image size enters through the per-block survivor bitmap */
size_t b200gs_scratch_bytes(int32_t P);

/* One-time initialisation of persistent workspaces (see b200gs_workspace_t.persistent): zeroes the geom workspace's
 * counter region, the image workspace (no cost history yet) and, when `scratch` != NULL, the P*64-byte backward scratch. */
int b200gs_workspace_init(const b200gs_workspace_t* ws, int32_t P, void* scratch, void* stream);

/* Stage 1 of the forward: preprocess, depth ordering, instance count.  Needs ws->geom and
 * ws->image.  Writes out->radii.  If `num_rendered_host` != NULL the instance count is copied to
 * it and the stream is synchronized before returning -- the reference's one blocking D2H
 * (rasterizer_impl.cu:281), used to size the binning workspace exactly.  With NULL nothing
 * synchronizes and the count stays on the device. */
int b200gs_forward_preprocess(const b200gs_view_t* view, const b200gs_gaussians_t* g, const b200gs_outputs_t* out,
                              const b200gs_workspace_t* ws, void* stream, int64_t* num_rendered_host);

/* Stage 2: duplicate-with-keys, tile sort, tile ranges, blend.  ws->binning must hold
 * b200gs_binning_bytes(capacity, width, height) bytes.  If the device-side instance count exceeds `capacity`
 * the overflow flag is raised (see b200gs_forward_status) and the surplus instances are dropped. */
int b200gs_forward_render(const b200gs_view_t* view, const b200gs_gaussians_t* g, const b200gs_outputs_t* out,
                          const b200gs_workspace_t* ws, int64_t capacity, void* stream);

/* Stage 1 + stage 2 with no host synchronization (capacity supplied by the caller). */
int b200gs_forward(const b200gs_view_t* view, const b200gs_gaussians_t* g, const b200gs_outputs_t* out,
                   const b200gs_workspace_t* ws, int64_t capacity, void* stream);

/* Synchronizes `stream`, then reports the instance count and whether it overflowed `capacity`. */
int b200gs_forward_status(const b200gs_workspace_t* ws, void* stream, int64_t* num_rendered, int32_t* overflow);

int b200gs_backward(const b200gs_view_t* view, const b200gs_gaussians_t* g, const int32_t* radii,
                    const b200gs_workspace_t* ws, int64_t capacity, const b200gs_grad_outputs_t* gout,
                    const b200gs_grads_t* grads, void* stream);

/* Gradients w.r.t. the camera of one view (device), for pose refinement.  Indexed like b200gs_view_t's arrays, so
 * dL_dviewmatrix[4c+r] is the gradient of element (r,c).  Entries the rasterizer never reads are written as exact zeros:
 * row 3 of the view matrix (3, 7, 11, 15), row 2 of the projection (2, 6, 10, 14), and campos without shs.  The 35
 * floats are assigned on every call, whatever b200gs_grads_t.accumulate says (camera gradients are per view), and are
 * bitwise reproducible for the same inputs.  The intrinsics (tan_fov, hence focal) get no gradient. */
typedef struct b200gs_camera_grads {
	float* dL_dviewmatrix;  /* device f32[16], indexed like b200gs_view_t.viewmatrix; row 3 written 0 */
	float* dL_dprojmatrix;  /* device f32[16], indexed like projmatrix; row 2 written 0 */
	float* dL_dcampos;      /* device f32[3]; 0 without shs */
	void* scratch;          /* b200gs_camera_scratch_bytes(P) bytes; no initialisation, contents on return unspecified */
} b200gs_camera_grads_t;

size_t b200gs_camera_scratch_bytes(int32_t P);

/* b200gs_backward plus, when `cam` != NULL, the camera gradients (one more kernel launch).  b200gs_backward is this call
 * with cam == NULL.  With cam: every pointer in it is required, and grads->scatter_bases must be NULL (camera gradients
 * are not combined with the image-parallel gradient scatter); either violation returns B200GS_E_ARG. */
int b200gs_backward_camera(const b200gs_view_t* view, const b200gs_gaussians_t* g, const int32_t* radii,
                           const b200gs_workspace_t* ws, int64_t capacity, const b200gs_grad_outputs_t* gout,
                           const b200gs_grads_t* grads, const b200gs_camera_grads_t* cam, void* stream);

/* sizeof(b200gs_camera_grads_t); b200gs_abi_sizes reports the six structs before it. */
int64_t b200gs_camera_grads_abi_size(void);

/* present: device u8[P] (bool). */
int b200gs_mark_visible(int32_t P, const float* means3D, const float* viewmatrix, const float* projmatrix,
                        uint8_t* present, void* stream);

/* ---- inspection (tests / parity tooling; not needed by a caller) ---- */
/* Byte offsets of the decodable arrays inside each workspace.
 * geom   : [0] header, [1] depths f32[P], [2] rect u16[P][4] (x0,y0,x1,y1), [3] record f32[P][16],
 *          [4] clamped u8[P] (bit c = colour channel c clamped), [5] order u32[P] (Gaussian ids by
 *          (depth bits, id)), [6] sorted depth keys u32[P] (0xFFFFFFFF for culled Gaussians)
 * image  : [0] final_T f32[N], [1] n_contrib u32[N], [2] ranges u32[tiles][2]
 * binning: [0] point_list u32[L] (sorted), [1] tile ids u32[L] (sorted)   -- valid after forward_render */
void b200gs_geom_layout(int32_t P, int64_t* offsets7);
void b200gs_image_layout(int32_t width, int32_t height, int64_t* offsets3);
void b200gs_binning_layout(int32_t width, int32_t height, int64_t capacity, int64_t* offsets2);
/* Materialise the reference's 64-bit sort keys (tile<<32 | depth bits) in sorted order: keys_out u64[L]. */
int b200gs_debug_sorted_keys(const b200gs_view_t* view, int32_t P, const b200gs_workspace_t* ws, int64_t capacity,
                             uint64_t* keys_out, int64_t L, void* stream);
/* Number of kernel launches issued by this library since load (bench.py's gpu_launches). */
int64_t b200gs_launch_count(void);
/* Optional per-stage timing with CUDA events on the launch stream (bench.py's roofline numbers).
 * Stages: 0 memsets, 1 preprocess fwd, 2 depth sort, 3 offsets scan, 4 duplicate-with-keys, 5 tile sort,
 * 6 tile ranges, 7 blend fwd, 8 blend bwd, 9 preprocess bwd (with the camera-gradient reduction when asked for).
 * profile_read synchronizes the pending events and
 * returns accumulated milliseconds / call counts per stage (arrays of 10). */
#define B200GS_NUM_STAGES 10
void b200gs_profile_enable(int32_t on);
int b200gs_profile_read(double* ms_out10, int64_t* n_out10, int32_t reset);
/* sizeof() of the six structs above, in declaration order (lets a foreign-language binding check its layout). */
void b200gs_abi_sizes(int64_t* out6);

#ifdef __cplusplus
}
#endif
#endif /* B200GS_H_ */

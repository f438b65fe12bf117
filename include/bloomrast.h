/*
 * bloomrast.h — C-ABI of the B200-native differentiable Gaussian rasterizer.
 *
 * This is the drop-in boundary for BloomScene's `submodules/depth-diff-gaussian-rasterization`.
 * Every entry point replaces one member of the reference's C++ static API
 * `CudaRasterizer::Rasterizer` (reference: cuda_rasterizer/rasterizer.h:24-105), which the
 * reference's torch binding (rasterize_points.cu:35-288, ext.cpp:15-20) calls with raw device
 * pointers.  Plain C: device pointers and sizes only, no torch / C++ types, no exceptions.
 *
 * Conventions (same as the reference unless stated):
 *   - all arrays are fp32 / int32 device memory, densely packed, row-major as PyTorch lays them out;
 *   - `viewmatrix` / `projmatrix` are 16 floats whose memory is the transpose of the maths matrix
 *     (row-vector convention, reference scene/cameras.py:59-62);
 *   - a NULL pointer means "optional input absent" — the reference relies on empty tensors having
 *     data_ptr()==nullptr (forward.cu:205,241; backward.cu:390,394; rasterizer_impl.cu:322,453,481);
 *   - every function is asynchronous on `stream` except where noted, re-entrant, and never owns
 *     memory: buffers come from the caller through `brs_alloc_fn`;
 *   - return value: BRS_OK (0) or a negative brs_status; brs_error_string() names it.
 */
#ifndef BLOOMRAST_H_
#define BLOOMRAST_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BRS_VERSION 200 /* 0.2.0: optimistic and deferred forward, see brs_forward_ex */

typedef struct CUstream_st* brs_stream; /* == cudaStream_t */

typedef enum brs_status {
	BRS_OK = 0,
	BRS_ERR_INVALID_ARG = -1, /* NULL where required, negative size, both/neither of an either-or pair */
	BRS_ERR_ALLOC = -2,       /* allocator callback returned NULL */
	BRS_ERR_CUDA = -3,        /* a CUDA call failed; see brs_last_cuda_error() */
	BRS_ERR_UNSUPPORTED = -4, /* e.g. sh_degree > 3, more than 2^30 tile instances */
	BRS_ERR_STATE = -5        /* forward state handed to backward does not match the sizes given */
} brs_status;

/* Which caller-owned buffer an allocation request is for.  GEOM / BINNING / IMAGE are the three
 * byte buffers the reference keeps on the autograd context (rasterize_points.cu:74-79, "geomBuffer",
 * "binningBuffer", "imgBuffer"); SCRATCH is temporary and may be released when the call returns
 * (stream-ordered). */
typedef enum brs_buffer {
	BRS_BUF_GEOM = 0,
	BRS_BUF_BINNING = 1,
	BRS_BUF_IMAGE = 2,
	BRS_BUF_SCRATCH = 3
} brs_buffer;

/* Replaces the reference's three std::function<char*(size_t)> resize callbacks
 * (rasterizer.h:34-36, rasterize_points.cu:27-33).  Must return device memory of at least `bytes`
 * bytes aligned to 256 bytes, usable on the stream of the call, or NULL on failure. */
typedef void* (*brs_alloc_fn)(void* ctx, int which /* brs_buffer */, size_t bytes);

/* Per-call camera / configuration: the fields of GaussianRasterizationSettings
 * (depth_diff_gaussian_rasterization/__init__.py:158-170). */
typedef struct brs_view {
	int image_width;
	int image_height;
	float tanfovx;
	float tanfovy;
	float scale_modifier;
	int sh_degree;           /* active degree D, 0..3 */
	int sh_coeffs;           /* M = coefficients stored per Gaussian (shs is [P, M, 3]); 0 without SH */
	int prefiltered;         /* reference traps on the device if a culled point is seen with this set */
	int debug;               /* synchronise + check after every stage (reference CHECK_CUDA) */
	const float* bg;         /* [3]  device */
	const float* viewmatrix; /* [16] device */
	const float* projmatrix; /* [16] device */
	const float* campos;     /* [3]  device */
} brs_view;

/* Gaussian attributes, device pointers (reference rasterizer.h:37-52). Exactly one of
 * shs / colors_precomp and exactly one of (scales, rotations) / cov3D_precomp is non-NULL. */
typedef struct brs_gaussians {
	int P;
	const float* means3D;        /* [P,3] */
	const float* opacities;      /* [P]   */
	const float* shs;            /* [P,M,3] or NULL */
	const float* colors_precomp; /* [P,3]   or NULL */
	const float* scales;         /* [P,3]   or NULL */
	const float* rotations;      /* [P,4]   or NULL (not normalised in-kernel, forward.cu:127) */
	const float* cov3D_precomp;  /* [P,6]   or NULL */
} brs_gaussians;

/* What forward leaves behind for backward (the reference's geom/binning/img chunks + num_rendered). */
typedef struct brs_fwd_state {
	void* geom;
	size_t geom_bytes;
	void* binning;
	size_t binning_bytes;
	void* image;
	size_t image_bytes;
	int num_rendered; /* R = number of (tile, Gaussian) instances; -1 after a DEFERRED forward (it stayed on the device) */
} brs_fwd_state;

/* Gradient outputs (reference rasterize_points.cu:154-162).  Every pointer that is non-NULL is
 * fully written by brs_backward (zeros for Gaussians that were not rendered) — the caller does
 * NOT need to zero-fill.  dL_dconic is internal in the reference and is not exposed. */
typedef struct brs_grads {
	float* dL_dmeans2D;   /* [P,3], z = 0   */
	float* dL_dcolors;    /* [P,3]          */
	float* dL_dopacity;   /* [P,1]          */
	float* dL_dmeans3D;   /* [P,3]          */
	float* dL_dcov3D;     /* [P,6]          */
	float* dL_dsh;        /* [P,M,3] or NULL when M == 0 */
	float* dL_dscales;    /* [P,3]          */
	float* dL_drotations; /* [P,4]          */
	/* 0 (reference behaviour): every element of every tensor above is written, zeros for culled
	 * Gaussians (the reference zero-fills first: rasterize_points.cu:154-162).
	 * 1 (extension for multi-view steps): the gradients of the inputs that were given — means3D,
	 * opacity, sh | colors_precomp, scales + rotations | cov3D_precomp — are ADDED to what the
	 * buffers hold, for visible Gaussians only; tensors of absent inputs may be NULL and are not
	 * touched; dL_dmeans2D (a per-view statistic) is still overwritten. */
	int accumulate;
	/* 0 (reference behaviour): the depth image carries no gradient, dL_dout_depth is ignored — the
	 * reference has every depth line of its backward commented out (backward.cu:443-554).
	 * 1 (extension, SURVEY.md 8f N3): dL_dout_depth [1,H,W] is back-propagated through the depth the
	 * forward actually outputs — D / acc with D = sum T alpha z, acc = 1e-6 + sum T alpha, zero where
	 * acc <= 0.5 (forward.cu:464-468) — into opacity, means2D, conic and the view-space depth z of every
	 * Gaussian, i.e. into means3D, scales / rotations | cov3D_precomp and opacities.  `out_depth` must
	 * then be the [1,H,W] depth image brs_forward wrote for this state. */
	int depth_gradient;
	const float* out_depth;
} brs_grads;

/* --- entry points ------------------------------------------------------------------------- */

/* Replaces CudaRasterizer::Rasterizer::forward (rasterizer.h:32-57, rasterizer_impl.cu:198-339).
 * Writes out_color [3,H,W] (planar), out_depth [1,H,W], radii [P]; all three are fully written.
 * P == 0 writes zeros and returns R = 0 (reference skips the kernels: rasterize_points.cu:82).
 * Performs at most ONE host wait (for R) like the reference (rasterizer_impl.cu:282); see
 * brs_fwd_options for when it happens.  Same as brs_forward_ex with opt == NULL. */
int brs_forward(const brs_view* view, const brs_gaussians* g,
                float* out_color, float* out_depth, int* radii,
                brs_alloc_fn alloc, void* alloc_ctx,
                brs_fwd_state* state, brs_stream stream);

/* Extension: how the forward learns its instance counts.  The reference copies num_rendered to the host
 * with a blocking cudaMemcpy between its scan and its sort (rasterizer_impl.cu:282) and sizes the
 * binning buffer from it.  Here every kernel after preprocess reads the counts from the device and takes
 * only CAPACITIES from the host, so the host does not have to know them before it launches:
 *   BRS_FWD_AUTO     (default) the first forward of a (device, P, W, H) shape runs EXACT; later ones size
 *                    their buffers from the high-water marks of that shape (+25 %), enqueue everything
 *                    through the blend, and only then wait for the header that left the device right
 *                    after preprocess — the GPU never drains.  If a capacity was too small (the header's
 *                    overflow word) the binning and the blend are run again with the exact sizes.
 *   BRS_FWD_EXACT    wait for the counts right after preprocess, then size exactly (reference behaviour).
 *   BRS_FWD_DEFERRED no host wait at all: capacities from this struct (0 = the high-water marks); the
 *                    8-word header {R, R1, ~min depth key, max depth key, V, overflow, key bits, 0} (overflow: bit 0
 *                    R, bit 1 R1, bit 2 depth-key bits, bit 3 V exceeded its capacity) is copied
 *                    asynchronously to `report` (pinned host memory).  state->num_rendered is -1.  The caller
 *                    inspects report[5] after it has synchronised with the stream for its own reasons — e.g.
 *                    once per batch of views — and repeats the overflowed forwards in EXACT mode.  A deferred
 *                    forward (and the backward of its state) can be captured in a CUDA graph.
 * Results are bit-identical in all three modes. */
enum { BRS_FWD_AUTO = 0, BRS_FWD_EXACT = 1, BRS_FWD_DEFERRED = 2 };
typedef struct brs_fwd_options {
	int mode;
	int R_cap;        /* DEFERRED: capacity of the binning buffer in tile instances (0: high-water mark) */
	int R1_cap;       /* DEFERRED: capacity in supertile instances (0: high-water mark) */
	int depth_bits;   /* DEFERRED: significant depth-key bits to sort on (0: high-water mark) */
	uint32_t* report; /* DEFERRED: 8 words of pinned host memory (may be NULL when overflow_accum is given) */
	/* DEFERRED, optional: DEVICE word into which the overflow bits of this forward are OR-ed.  A caller that
	 * replays a captured forward many times (CUDA graph) zeroes it once, reads it once per batch. */
	uint32_t* overflow_accum;
} brs_fwd_options;
int brs_forward_ex(const brs_view* view, const brs_gaussians* g,
                   float* out_color, float* out_depth, int* radii,
                   brs_alloc_fn alloc, void* alloc_ctx,
                   brs_fwd_state* state, const brs_fwd_options* opt, brs_stream stream);
/* Extension (SURVEY.md 8f N1): forward-only render of n_views views of ONE set of Gaussians as one pipeline — the
 * batched form of the loops the reference's callers run one blocking view at a time (bloomscene.py:191-204,
 * gaussian_renderer/__init__.py:211-291).  The views' preprocess launches write into one instance space
 * (instance v * P + i, tile rectangle shifted down by v * grid_y rows), then ONE depth sort, ONE emission /
 * coarse sort / fine binning and ONE blend launch serve all views: per-tile order is (depth bits, Gaussian id)
 * exactly as in n_views separate forwards, so every output is bit-identical to them.
 * All views share image size, sh_degree / sh_coeffs and debug; the background of views[0] is used; tanfov,
 * matrices, campos, scale_modifier and prefiltered are per view.  out_color [n,3,H,W], out_depth [n,1,H,W],
 * radii [n,P].  Nothing is kept for a backward.  *num_rendered (optional) = the instances of all views together
 * (-1 after a DEFERRED forward).  opt as in brs_forward_ex (NULL = BRS_FWD_AUTO: at most one host wait per STACK).
 * Limits: n_views * P < 2^31, n_views * ceil(H / 16) < 65536. */
int brs_forward_views(const brs_view* views, int n_views, const brs_gaussians* g,
                      float* out_color, float* out_depth, int* radii,
                      brs_alloc_fn alloc, void* alloc_ctx, long long* num_rendered,
                      const brs_fwd_options* opt, brs_stream stream);
/* Extension: brs_forward_views where every view renders its OWN Gaussians (BloomScene's render loop, whose anchor
 * culling and neural-Gaussian generation give each frame its own rows, bloomscene.py:174-219).  g holds the views'
 * rows concatenated: view v owns rows [off_v, off_v + view_P[v]), off_v = view_P[0] + ... + view_P[v - 1], and
 * g->P must equal the sum of view_P.  radii [g->P] in the same row order.  Each view's outputs are bit-identical to
 * a brs_forward_ex of its own rows; a view with view_P[v] == 0 gets zeros without background, as that forward
 * does.  view_P == NULL: every view sees all g->P rows (= brs_forward_views).  A negative entry or a sum other than
 * g->P returns BRS_ERR_INVALID_ARG, a sum of 2^31 or more BRS_ERR_UNSUPPORTED, before any CUDA call.
 * Limit: n_views * ceil(H / 16) < 65536. */
int brs_forward_views_ex(const brs_view* views, int n_views, const brs_gaussians* g, const int* view_P,
                         float* out_color, float* out_depth, int* radii,
                         brs_alloc_fn alloc, void* alloc_ctx, long long* num_rendered,
                         const brs_fwd_options* opt, brs_stream stream);
/* Feeds the counts of a DEFERRED forward's report back into the high-water marks of its shape. */
void brs_note_counts(int P, int image_width, int image_height, const uint32_t* report);
/* High-water marks of a shape on the current device: returns 1 and fills out[3] = {R, R1, depth-key bits} if a
 * forward of that shape has been seen, else 0. */
int brs_get_marks(int P, int image_width, int image_height, uint32_t* out);
/* Per calling thread: out[0] = EXACT forwards, out[1] = optimistic ones, out[2] = of those, re-run because a
 * capacity overflowed, out[3] = DEFERRED ones. */
void brs_forward_stats(long long* out, int reset);
/* Forgets all high-water marks (the next forward of every shape runs EXACT again). */
void brs_reset_marks(void);

/* Replaces CudaRasterizer::Rasterizer::backward (rasterizer.h:78-105, rasterizer_impl.cu:403-504).
 * dL_dout_depth is accepted and, unless grads->depth_gradient is set, ignored: the reference plumbs it
 * but every use is commented out (backward.cu:443-554), so depth carries no gradient by default.
 * No host synchronisation. */
int brs_backward(const brs_view* view, const brs_gaussians* g, const int* radii,
                 const brs_fwd_state* state,
                 const float* dL_dout_color, const float* dL_dout_depth,
                 const brs_grads* grads,
                 brs_alloc_fn alloc, void* alloc_ctx, brs_stream stream);

/* Extension: densification statistics of one view, added by the backward itself.  The reference's callers read
 * means2D.grad[:, :2] and radii > 0 after every view and add the gradient norm and a count into per-Gaussian
 * accumulators (Scaffold-GS training_statis, scene/gaussian_model.py:742-759; 3DGS add_densification_stats).
 * With `stats`, for every Gaussian i with radii[i] > 0 and slot s = index ? index[i] : i:
 *   grad_norm[s] += sqrtf(gx*gx + gy*gy)   (gx, gy: the fp32 values written to dL_dmeans2D[i, 0:2])
 *   count[s]     += 1                       (also when that gradient is zero)
 * Slots outside [0, rows) are skipped (-1 = "no slot").  The additions are float reductions, so views running on
 * different streams may add into the same accumulators at the same time; works in every brs_grads mode, after a
 * DEFERRED forward and inside a CUDA graph.  The index type is that of brs_visible_filter_compact's `indices`. */
typedef struct brs_densify_stats {
	float* grad_norm;       /* [rows] */
	float* count;           /* [rows] */
	const long long* index; /* [P] slot of Gaussian i, or NULL = identity (then rows >= P is required) */
	int rows;
} brs_densify_stats;
/* brs_backward plus optional densification statistics; stats == NULL is exactly brs_backward.  Returns
 * BRS_ERR_INVALID_ARG, before any CUDA call, when grad_norm or count is NULL, rows < 0, or index is NULL and
 * rows < P. */
int brs_backward_ex(const brs_view* view, const brs_gaussians* g, const int* radii,
                    const brs_fwd_state* state,
                    const float* dL_dout_color, const float* dL_dout_depth,
                    const brs_grads* grads, const brs_densify_stats* stats,
                    brs_alloc_fn alloc, void* alloc_ctx, brs_stream stream);

/* Replaces CudaRasterizer::Rasterizer::visible_filter (rasterizer.h:59-76, rasterizer_impl.cu:342-398):
 * radii only.  `scales_stride` is the row stride of `scales` in floats (3 when dense); BloomScene
 * passes a [:, :3] view of a [P,6] tensor (gaussian_renderer/__init__.py:344).  No allocations. */
int brs_visible_filter(const brs_view* view, int P, const float* means3D,
                       const float* scales, int scales_stride, const float* rotations,
                       const float* cov3D_precomp, int* radii, brs_stream stream);

/* Extension (SURVEY.md 8f N2): the same filter fused with the compaction BloomScene performs next — it turns the
 * radii into visible_mask = radii > 0 and boolean-indexes every per-anchor tensor with it
 * (gaussian_renderer/__init__.py:294-349, :39-60).  Also writes `indices` (int64 [P] capacity): the ascending
 * indices of the Gaussians with radii > 0, and their number into the device scalar `count`, in the same kernel.
 * `scratch` = brs_filter_scratch_bytes(P) bytes. */
size_t brs_filter_scratch_bytes(int P);
int brs_visible_filter_compact(const brs_view* view, int P, const float* means3D,
                               const float* scales, int scales_stride, const float* rotations,
                               const float* cov3D_precomp, int* radii, long long* indices, uint32_t* count,
                               void* scratch, brs_stream stream);

/* Replaces CudaRasterizer::Rasterizer::markVisible (rasterizer.h:24-30, rasterizer_impl.cu:141-153):
 * present[i] = (view-space z of mean i) > 0.2. */
int brs_mark_visible(int P, const float* means3D, const float* viewmatrix, const float* projmatrix,
                     uint8_t* present, brs_stream stream);

/* Buffer sizes: pure functions of the sizes (the reference re-derives its layout in backward the
 * same way: rasterizer_impl.h:66-72 `required<T>`). */
size_t brs_geom_bytes(int P);
size_t brs_binning_bytes(int num_rendered);
size_t brs_image_bytes(int image_width, int image_height);
size_t brs_forward_scratch_bytes(int P, int num_rendered, int image_width, int image_height);
size_t brs_backward_scratch_bytes(int P);

/* Stable LSD radix sort of (u32 key, u32 value) pairs on key bits [begin_bit, end_bit) — the
 * hand-written onesweep-style sort that replaces cub::DeviceRadixSort::SortPairs
 * (rasterizer_impl.cu:304-309).  If vals_in is NULL the values are 0..n-1.  `scratch` must hold
 * brs_sort_scratch_bytes(n) bytes; sorted output lands in keys_out / vals_out. */
size_t brs_sort_scratch_bytes(int n);
int brs_sort_pairs_u32(const uint32_t* keys_in, const uint32_t* vals_in,
                       uint32_t* keys_out, uint32_t* vals_out, int n,
                       int begin_bit, int end_bit, void* scratch, brs_stream stream);

/* Layout of the private state, for stage-level parity tests (offsets in bytes from the start of
 * each buffer; strides in bytes). */
typedef struct brs_layout {
	/* geom */
	size_t geom_records;   /* float4[3*P]: {x,y,tau,0} {conic a,b,c,opacity} {r,g,b,depth} */
	size_t geom_depth_key; /* u32[P]: float bits of view-space depth, 0xFFFFFFFF when culled */
	size_t geom_rect;      /* u32[2*P]: (x0 | x1<<16), (y0 | y1<<16) tile rectangle */
	size_t geom_order;     /* u32[P]: Gaussian ids sorted by (depth, id) */
	/* binning */
	size_t binning_point_list; /* u32[R]: Gaussian ids sorted by (tile, depth, id) */
	/* image */
	size_t image_ranges;    /* uint2[ceil(W/16)*ceil(H/16)] */
	size_t image_final_T;   /* f32[W*H] */
	size_t image_n_contrib; /* u32[W*H] */
} brs_layout;
int brs_state_layout(int P, int num_rendered, int image_width, int image_height, brs_layout* out);

const char* brs_error_string(int status);
/* cudaError_t of the last failing CUDA call on this thread (0 if none), and its name. */
int brs_last_cuda_error(void);
const char* brs_last_cuda_error_string(void);
int brs_version(void);
/* Number of kernels this library launched (process-wide, all threads) since the last reset. */
long long brs_launch_count(int reset);

/* --- the steps either side of the rasterizer (extensions, SURVEY.md 8f N4; opt-in) ------------------- */

/* Fused photometric loss of the training step: loss = (1 - lambda) * mean|x - y| + lambda * (1 - mean SSIM(x, y)),
 * replacing the torch-op chains of reference utils/loss.py:83-84 (l1_loss) and :91-135 (ssim: 11 x 11 Gaussian
 * window, sigma 1.5, zero padding, C1 = 0.01^2, C2 = 0.03^2) as used in bloomscene.py:284-287.
 * Forward: x, y are [C,H,W]; writes the three derivative maps the backward needs into dmaps [3,C,H,W] and one
 * (sum of SSIM, sum of |x - y|) pair per 16 x 16 block into partial [brs_l1_ssim_blocks()][2]; the caller sums
 * them (deterministic) and forms the loss.  Backward: dL_dx [C,H,W] = *dL_dloss * d loss / d x. */
size_t brs_l1_ssim_blocks(int C, int H, int W);
int brs_l1_ssim_forward(const float* x, const float* y, int C, int H, int W, float* dmaps, float* partial, brs_stream stream);
int brs_l1_ssim_backward(const float* x, const float* y, const float* dmaps, int C, int H, int W,
                         const float* dL_dloss, float lambda_dssim, float* dL_dx, brs_stream stream);

/* Fused epilogue of the neural-Gaussian generation, replacing the mask / concat / boolean-index / split /
 * post-process chain of reference gaussian_renderer/__init__.py:168-203: for every (anchor n, offset k) row with
 * neural_opacity > 0, in row order,
 *   xyz = anchor[n] + offsets[n,k] * grid_scaling[n,:3]      scaling = grid_scaling[n,3:] * sigmoid(scale_rot[:3])
 *   rot = normalize(scale_rot[3:7])                          colour, opacity copied
 * written to the first *count rows of the output arrays (capacity N*K rows each); index[n*K+k] = output row or -1.
 * `scratch` = brs_neural_scratch_bytes(N) bytes.  K <= 32.  Backward: all six input gradients, fully written. */
typedef struct brs_neural_inputs {
	int N, K;
	const float* anchor;         /* [N,3]   */
	const float* grid_scaling;   /* [N,6]   */
	const float* offsets;        /* [N*K,3] */
	const float* neural_opacity; /* [N*K]   */
	const float* color;          /* [N*K,3] */
	const float* scale_rot;      /* [N*K,7] */
} brs_neural_inputs;
typedef struct brs_neural_outputs {
	float* xyz;      /* [N*K,3] */
	float* color;    /* [N*K,3] */
	float* opacity;  /* [N*K]   */
	float* scaling;  /* [N*K,3] */
	float* rot;      /* [N*K,4] */
	int* index;      /* [N*K]   */
	uint32_t* count; /* device scalar */
} brs_neural_outputs;
typedef struct brs_neural_grads {
	const float* d_xyz;      /* [M,3] upstream */
	const float* d_color;    /* [M,3] */
	const float* d_opacity;  /* [M]   */
	const float* d_scaling;  /* [M,3] */
	const float* d_rot;      /* [M,4] */
	float* d_anchor;         /* [N,3] outputs */
	float* d_grid_scaling;   /* [N,6] */
	float* d_offsets;        /* [N*K,3] */
	float* d_neural_opacity; /* [N*K] */
	float* d_color_in;       /* [N*K,3] */
	float* d_scale_rot;      /* [N*K,7] */
} brs_neural_grads;
size_t brs_neural_scratch_bytes(int N);
int brs_neural_gaussians_forward(const brs_neural_inputs* in, const brs_neural_outputs* out, void* scratch, brs_stream stream);
int brs_neural_gaussians_backward(const brs_neural_inputs* in, const int* index, const brs_neural_grads* g, brs_stream stream);

/* --- measurement hooks (bench / profiling only; off by default) ---------------------------- */

/* Stage ids for brs_stage_times(). */
enum {
	BRS_STAGE_PREPROCESS = 0,
	BRS_STAGE_DEPTH_SORT = 1,
	BRS_STAGE_COARSE_EMIT = 2, /* scan + emission of (supertile, Gaussian) instances in depth order */
	BRS_STAGE_COARSE_SORT = 3, /* stable radix pass(es) on the supertile id */
	BRS_STAGE_FINE_BIN = 4,    /* per-tile count / scan / scatter -> point_list, tile ranges */
	BRS_STAGE_BLEND_FWD = 5,
	BRS_STAGE_BLEND_BWD = 6,
	BRS_STAGE_PREPROCESS_BWD = 7,
	BRS_NUM_STAGES = 8
};
/* When enabled, every stage is bracketed by CUDA events on the call's stream (per thread). */
void brs_stage_timing(int enable);
/* When enabled (process-wide), the launches of every stage sit inside an NVTX range named "brs:<stage>", for
 * nsys timelines and `ncu --nvtx --nvtx-include`.  enable: 1 / 0 to set, -1 to query; returns the previous setting.
 * Also switched on by the environment variable BRS_NVTX=1 at the first forward. */
int brs_stage_nvtx(int enable);

/* Scheduling option (no reference counterpart).  When the caller's stream has a higher priority than
 * the device's lowest, brs_forward / brs_backward launch their blend kernels on an internal
 * lowest-priority companion stream fenced by events on both sides, so that other views' small
 * preprocess / sort / binning kernels (on other high-priority streams) are dispatched ahead of a
 * blend grid's remaining blocks.  Stream order as seen by the caller is unchanged.  enable: 1 / 0 to
 * set, -1 to query; returns the previous setting (default 1).  No effect on default-priority streams. */
int brs_blend_companion_stream(int enable);
/* Synchronises the recorded events; adds the accumulated milliseconds per stage into ms[BRS_NUM_STAGES]
 * and the number of timed launches per stage into calls[BRS_NUM_STAGES] (either may be NULL),
 * then clears the accumulators. */
int brs_stage_times(float* ms, int* calls);

/* Counts (pixel, instance) pairs of a finished forward under the REFERENCE's per-pixel semantics
 * (forward.cu:409-452): out[0] = E pairs evaluated until each pixel's own stop, out[1] = C pairs
 * that contribute, out[2] = E_b = sum of n_contrib (pairs the backward replays).  `out` is 3 x u64
 * device memory.  Used for the roofline's algorithmic flop count (SURVEY.md 8d). */
int brs_count_pairs(const brs_view* view, const brs_fwd_state* state, int P, unsigned long long* out,
                    brs_stream stream);

/* FP32 FMA micro-benchmark: returns the achieved TFLOP/s of a dependent-FFMA kernel filling the
 * GPU (the denominator for the blend kernels' roofline); synchronous. */
double brs_probe_fp32_tflops(brs_stream stream);

#ifdef __cplusplus
}
#endif
#endif /* BLOOMRAST_H_ */

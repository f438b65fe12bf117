// Per-Gaussian forward preprocessing for sm_100a.
//
//   preprocess_kernel      <- reference preprocessCUDA        (cuda_rasterizer/forward.cu:155-256)
//   filter_kernel          <- reference filter_preprocessCUDA (forward.cu:260-335)
//   check_frustum_kernel   <- reference checkFrustum          (rasterizer_impl.cu:54-66)
//
// What differs from the reference (layout / scheduling only — the arithmetic keeps its shapes):
//   * one packed 48-byte blend record per Gaussian {x,y,tau,0 | conic a,b,c,opacity | r,g,b,depth}
//     instead of five separate arrays, so the blend kernels gather three aligned float4s;
//   * SH coefficients of the *visible* Gaussians of a block are staged through shared memory with
//     coalesced 128-bit streaming loads (row pitch 13 float4 -> conflict-free per-thread reads);
//   * cov3D and the `clamped` flags are not stored: the backward recomputes them bit-identically;
//   * the per-Gaussian tile rectangle is stored packed (8 B) and the grid-wide instance count R is
//     accumulated here with one integer atomic per block, so the host can read R while the depth
//     sort is already running;
//   * tau: a conservative bound on q = d^T conic d beyond which this Gaussian's alpha cannot reach
//     1/255 (used by the blend kernels for warp-level culling; see cull_tau()).
#include "common.cuh"
#include "gaussian_math.cuh"
#include "kernels.h"

namespace brs {

// ---- geometry shared by preprocess / filter ---------------------------------------------------

// reference forward.cu:74-113
__device__ __forceinline__ float3 compute_cov2d(const float3& mean, float focal_x, float focal_y, float tan_fovx,
                                                float tan_fovy, const float* cov3D, const float* viewmatrix)
{
	float3 t = transform_point_4x3(mean, viewmatrix);

	const float limx = 1.3f * tan_fovx;
	const float limy = 1.3f * tan_fovy;
	const float txtz = t.x / t.z;
	const float tytz = t.y / t.z;
	t.x = min(limx, max(-limx, txtz)) * t.z;
	t.y = min(limy, max(-limy, tytz)) * t.z;

	mat3 J = make_mat3(focal_x / t.z, 0.0f, -(focal_x * t.x) / (t.z * t.z), 0.0f, focal_y / t.z,
	                   -(focal_y * t.y) / (t.z * t.z), 0, 0, 0);

	mat3 W = make_mat3(viewmatrix[0], viewmatrix[4], viewmatrix[8], viewmatrix[1], viewmatrix[5], viewmatrix[9],
	                   viewmatrix[2], viewmatrix[6], viewmatrix[10]);

	mat3 T = mul(W, J);

	mat3 Vrk = make_mat3(cov3D[0], cov3D[1], cov3D[2], cov3D[1], cov3D[3], cov3D[4], cov3D[2], cov3D[4], cov3D[5]);

	mat3 cov = mul(mul(transpose(T), transpose(Vrk)), T);

	cov.c[0].x += 0.3f;
	cov.c[1].y += 0.3f;
	return {float(cov.c[0].x), float(cov.c[0].y), float(cov.c[1].y)};
}

struct Geometry {
	float depth;     // p_view.z
	float2 xy;       // pixel-space centre
	float3 cov;      // 2D covariance (a, b, c) after the +0.3 dilation
	float3 conic;    // inverse
	int radius;      // ceil(3 sqrt(lambda_max))
	uint2 rect_min, rect_max;
};

// The per-Gaussian inputs of the geometry half, fetched up front so that all loads of a thread are in
// flight together (fetched where the reference reads them, behind the frustum test, each group would
// expose its own DRAM latency).
struct GeomInputs {
	float3 mean;
	float cov3D[6];
};
__device__ __forceinline__ GeomInputs load_geom_inputs(const float* means3D, const float* scales, int scales_stride,
                                                       const float* rotations, const float* cov3D_precomp, int idx,
                                                       float scale_modifier)
{
	GeomInputs in;
	const float* mp = means3D + 3 * (size_t)idx;
	in.mean = {__ldg(mp), __ldg(mp + 1), __ldg(mp + 2)};
	if (cov3D_precomp != nullptr) {
#pragma unroll
		for (int i = 0; i < 6; i++)
			in.cov3D[i] = __ldg(cov3D_precomp + 6 * (size_t)idx + i);
	} else {
		const float* sp = scales + (size_t)idx * scales_stride;
		v3 s = make_v3(__ldg(sp), __ldg(sp + 1), __ldg(sp + 2));
		const float* rp = rotations + 4 * (size_t)idx;
		float4 q = make_float4(__ldg(rp), __ldg(rp + 1), __ldg(rp + 2), __ldg(rp + 3));
		compute_cov3d(s, scale_modifier, q, in.cov3D); // reference forward.cu:118-152 (after its frustum test; no side effects)
	}
	return in;
}

// Everything of preprocessCUDA up to the tile rectangle (forward.cu:186-237). Returns false when
// the reference would `return` early (culled / degenerate / zero-area rectangle).
__device__ __forceinline__ bool compute_geometry(const GeomInputs& in, const float* view, const float* proj, int W,
                                                 int H, float tan_fovx, float tan_fovy, float focal_x, float focal_y,
                                                 uint32_t grid_x, uint32_t grid_y, bool prefiltered, Geometry& g)
{
	const float3 p_orig = in.mean;
	const float* cov3D = in.cov3D;
	// in_frustum (auxiliary.h:139-164): only the view-space z test is live.
	float3 p_view = transform_point_4x3(p_orig, view);
	if (p_view.z <= 0.2f) {
		if (prefiltered) {
			printf("Point is filtered although prefiltered is set. This shouldn't happen!");
			__trap();
		}
		return false;
	}

	float4 p_hom = transform_point_4x4(p_orig, proj);
	float p_w = 1.0f / (p_hom.w + 0.0000001f);
	float3 p_proj = {p_hom.x * p_w, p_hom.y * p_w, p_hom.z * p_w};

	float3 cov = compute_cov2d(p_orig, focal_x, focal_y, tan_fovx, tan_fovy, cov3D, view);

	float det = (cov.x * cov.z - cov.y * cov.y);
	if (det == 0.0f)
		return false;
	float det_inv = 1.f / det;
	g.conic = {cov.z * det_inv, -cov.y * det_inv, cov.x * det_inv};

	float mid = 0.5f * (cov.x + cov.z);
	float lambda1 = mid + sqrt(max(0.1f, mid * mid - det));
	float lambda2 = mid - sqrt(max(0.1f, mid * mid - det));
	float my_radius = ceil(3.f * sqrt(max(lambda1, lambda2)));
	float2 point_image = {ndc2pix(p_proj.x, W), ndc2pix(p_proj.y, H)};
	uint2 rect_min, rect_max;
	get_rect(point_image, my_radius, rect_min, rect_max, grid_x, grid_y);
	if ((rect_max.x - rect_min.x) * (rect_max.y - rect_min.y) == 0)
		return false;
	// A finite covariance always gives my_radius >= 1 (lambda1 >= mid + sqrt(0.1)).  A NaN covariance gives
	// (int)NaN = 0 with a one-tile rect: the reference then counts an instance in tiles_touched that
	// duplicateWithKeys never writes (`if (radii[idx] > 0)`, rasterizer_impl.cu:89) and sorts an uninitialised
	// key slot.  Treat it as culled, which is what `radii == 0` tells every caller anyway.
	if ((int)my_radius <= 0)
		return false;

	g.depth = p_view.z;
	g.xy = point_image;
	g.cov = cov;
	g.radius = (int)my_radius; // reference: radii[idx] = my_radius (float -> int)
	g.rect_min = rect_min;
	g.rect_max = rect_max;
	return true;
}

// Conservative threshold for the blend kernels' warp-level culling (block_may_contribute(), common.cuh).
// The reference blend keeps a (pixel, Gaussian) pair only if alpha = min(0.99, o*exp(power)) >= 1/255
// with power = -0.5 (a dx^2 + c dy^2) - b dx dy evaluated in fp32 (forward.cu:416-429), i.e. only if
// q(d) = d^T Q d <= tau := 2 ln(255 o) up to fp32 evaluation noise.  A warp skips a Gaussian when the
// minimum of q over its pixel block exceeds the value returned here: tau inflated by a bound on the
// fp32 evaluation error of q (the reference's evaluation at the pixel AND the culling test's own at the
// block's closest point) over every offset this Gaussian can meet (|d| <= radius + tile), plus an
// absolute and a relative margin.  Computed from the SAME fp32 conic the blend uses.
// +inf (never cull) where no bound can be given, -inf (always cull) where opacity < 1/255 (alpha <= o).
__device__ __forceinline__ float cull_tau(const float3 conic, float opacity, int radius)
{
	const float inf = __int_as_float(0x7f800000);
	if (opacity < 1.0f / 255.0f)
		return -inf;
	if (!(opacity <= 3.0e38f)) // NaN / inf opacity: let the blend decide
		return inf;
	const float a = conic.x, b = conic.y, c = conic.z;
	const float det = a * c - b * b;
	if (!(det > 0.0f) || !(a > 0.0f) || !(c > 0.0f))
		return inf;
	const float dmax = (float)radius + (float)(TILE_X + 1);
	const float eval_err = 8.0f * 5.9604644775390625e-08f * (fabsf(a) + fabsf(c) + 2.0f * fabsf(b)) * dmax * dmax;
	// logf is good to a few ulp (~1e-6 absolute on a value of at most 11.1), far inside the 2e-4 margin
	float tau = 2.0f * logf(255.0f * opacity);
	tau = (tau + 4.0f * eval_err + 2e-4f) * (1.0f + 2e-5f);
	if (!(tau < 1e30f))
		return inf;
	return tau;
}

// ---- K1 -----------------------------------------------------------------------------------------

constexpr int PRE_THREADS = 128;

__device__ __forceinline__ void stage_camera(float* s_cam, const float* view, const float* proj, const float* campos)
{
	const int t = threadIdx.x;
	if (t < 16)
		s_cam[t] = __ldg(view + t);
	else if (t < 32)
		s_cam[t] = __ldg(proj + t - 16);
	else if (t < 35 && campos != nullptr)
		s_cam[t] = __ldg(campos + t - 32);
}

// VEC: rows are 16 coefficient triples (48 floats = 12 float4 = 192 bytes) and `shs` is 16-byte aligned.  Every
//   pair of rows is fetched with one bulk asynchronous copy (cp.async.bulk -> SASS UBLKCP, 384 bytes) into a
//   shared-memory tile whose pair pitch makes the lanes' LDS.128 reads conflict-free (sh_row_slot, common.cuh);
//   the bytes are collected by one mbarrier per warp, so there is no block barrier between the geometry, load and evaluation phases and no
//   SH data passes through registers on its way in.
// EAGER: the rows of ALL 32 Gaussians of the warp are requested at the very start, together with the
//   geometry inputs, so that a thread exposes one DRAM round trip instead of two; otherwise only the rows of
//   the visible Gaussians are requested, after the geometry phase.  The host picks EAGER when the last views
//   of this shape had most Gaussians visible (the rows of culled Gaussians are wasted traffic).
template <bool VEC, bool EAGER>
__device__ __forceinline__ void preprocess_body(const PreprocessArgs& a, const PreprocessViewTable::Slot& v, uint32_t row_offset)
{
	extern __shared__ float4 s_dyn[]; // SH staging (only when a.shs != nullptr)
	__shared__ float s_cam[36];
	__shared__ uint32_t s_tiles[5][PRE_THREADS / 32];
	__shared__ uint64_t s_bar[PRE_THREADS / 32];

	const int block_first = blockIdx.x * PRE_THREADS;
	const int idx = block_first + threadIdx.x;
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	const int P = (int)v.count;
	const bool in_range = idx < P;
	const bool bulk = VEC && a.shs != nullptr;

	if (bulk) {
		if (lane == 0)
			mbar_init(&s_bar[warp], 1);
		__syncwarp();
		if (EAGER) {
			// even lanes fetch their own row and their neighbour's (one 384-byte copy; 192 at the end of the array)
			const uint32_t rows = (uint32_t)max(0, min(32, P - (block_first + 32 * warp)));
			if (in_range && !(lane & 1))
				bulk_copy_g2s(s_dyn + sh_row_slot(threadIdx.x), a.shs + (size_t)idx * 48, idx + 1 < P ? 384u : 192u, &s_bar[warp]);
			if (lane == 0)
				mbar_arrive_expect_tx(&s_bar[warp], 192u * rows);
		}
	}
	// all per-Gaussian geometry inputs and the opacity are requested before anything is computed
	GeomInputs in;
	float opacity = 0.f;
	if (in_range) {
		in = load_geom_inputs(a.means3D, a.scales, 3, a.rotations, a.cov3D_precomp, idx, v.scale_modifier);
		opacity = __ldg(a.opacities + idx);
	}
	stage_camera(s_cam, v.viewmatrix, v.projmatrix, v.campos);
	__syncthreads();
	const float* view = s_cam;
	const float* proj = s_cam + 16;

	Geometry g;
	bool visible = false;
	float3 p_orig = {0.f, 0.f, 0.f};
	if (in_range) {
		p_orig = in.mean;
		visible = compute_geometry(in, view, proj, a.W, a.H, v.tan_fovx, v.tan_fovy, v.focal_x, v.focal_y, a.grid_x,
		                           a.grid_y, v.prefiltered != 0, g);
	}

	const uint32_t vis_mask = __ballot_sync(0xffffffffu, visible);
	uint32_t tiles = 0u, cells = 0u; // tile / supertile instances of this Gaussian
	if (visible) {
		g.rect_min.y += row_offset; // the view's place in a stack of views (0 for a single view)
		g.rect_max.y += row_offset;
		tiles = (g.rect_max.y - g.rect_min.y) * (g.rect_max.x - g.rect_min.x);
		cells = ((((g.rect_max.x - 1) >> ST_SHIFT) + 1) - (g.rect_min.x >> ST_SHIFT)) *
		        ((((g.rect_max.y - 1) >> ST_SHIFT) + 1) - (g.rect_min.y >> ST_SHIFT));
	}

	// ---- colour ----
	float3 rgb = {0.f, 0.f, 0.f};
	if (a.shs != nullptr) {
		// every warp stages the rows of ITS 32 Gaussians (no block barrier: warps of a block overlap
		// their geometry, load and evaluation phases)
		const int row_f = 3 * a.M; // floats per Gaussian
		const int warp_first = block_first + 32 * warp;
		if (VEC) {
			if (!EAGER) {
				// a pair of rows is fetched (by its even lane) when either of its Gaussians is visible
				const uint32_t pair_mask = (vis_mask | (vis_mask >> 1)) & 0x55555555u;
				const uint32_t short_pair = (in_range && !(lane & 1) && idx + 1 >= P && ((pair_mask >> lane) & 1u)) ? 1u : 0u;
				if (in_range && ((pair_mask >> lane) & 1u))
					bulk_copy_g2s(s_dyn + sh_row_slot(threadIdx.x), a.shs + (size_t)idx * 48, short_pair ? 192u : 384u, &s_bar[warp]);
				const uint32_t shorts = __popc(__ballot_sync(0xffffffffu, short_pair != 0u));
				if (lane == 0)
					mbar_arrive_expect_tx(&s_bar[warp], 384u * (uint32_t)__popc(pair_mask) - 192u * shorts);
			}
			if (vis_mask != 0u || EAGER)
				mbar_wait(&s_bar[warp], 0u);
		} else {
			const int pitch = row_f | 1; // odd pitch: conflict-free scalar reads
			float* s_sh = reinterpret_cast<float*>(s_dyn) + 32 * warp * pitch;
			const float* src = a.shs + (size_t)warp_first * row_f;
			const int total = 32 * row_f;
			for (int f = lane; f < total; f += 32) {
				const int row = f / row_f, col = f - row * row_f;
				if ((vis_mask >> row) & 1u)
					s_sh[row * pitch + col] = __ldg(src + f);
			}
			__syncwarp();
		}
		if (visible) {
			const v3 pos = make_v3(p_orig.x, p_orig.y, p_orig.z);
			const v3 cam = make_v3(s_cam[32], s_cam[33], s_cam[34]);
			v3 res;
			if (VEC) {
				// coefficients are read from the staged row where they are used (conflict-free LDS.128)
				res = eval_sh(a.D, pos, cam, ShRowView{s_dyn + sh_row_slot(threadIdx.x)});
			} else {
				res = eval_sh(a.D, pos, cam, reinterpret_cast<const float*>(s_dyn) + threadIdx.x * (row_f | 1));
			}
			// glm::max(result, 0.0f)  (forward.cu:67-70); the `clamped` flags are recomputed in backward.
			rgb = {(res.x < 0.0f) ? 0.0f : res.x, (res.y < 0.0f) ? 0.0f : res.y, (res.z < 0.0f) ? 0.0f : res.z};
		}
	} else if (visible) {
		const float* cp = a.colors_precomp + 3 * (size_t)idx;
		rgb = {__ldg(cp), __ldg(cp + 1), __ldg(cp + 2)};
	}

	// ---- outputs ----
	if (idx < P) {
		if (visible) {
			const float tau = cull_tau(g.conic, opacity, g.radius);
			float4* rec = a.records + 3 * (size_t)idx;
			rec[0] = make_float4(g.xy.x, g.xy.y, tau, 0.f);
			rec[1] = make_float4(g.conic.x, g.conic.y, g.conic.z, opacity);
			rec[2] = make_float4(rgb.x, rgb.y, rgb.z, g.depth);
			a.radii[idx] = g.radius;
			a.depth_key[idx] = __float_as_uint(g.depth);
			a.rect[idx] = make_uint2(g.rect_min.x | (g.rect_max.x << 16), g.rect_min.y | (g.rect_max.y << 16));
		} else {
			a.radii[idx] = 0;
			a.depth_key[idx] = DEPTH_KEY_CULLED;
			a.rect[idx] = make_uint2(0u, 0u);
		}
	}

	// ---- grid-wide instance counts R, R1 and the range of the visible depth keys (integers ->
	// deterministic).  The range lets the depth sort skip the key bits all visible Gaussians share.
	uint32_t inv_min = visible ? ~__float_as_uint(g.depth) : 0u; // max of ~key == ~min key
	uint32_t key_max = visible ? __float_as_uint(g.depth) : 0u;
#pragma unroll
	for (int o = 16; o > 0; o >>= 1) {
		tiles += __shfl_xor_sync(0xffffffffu, tiles, o);
		cells += __shfl_xor_sync(0xffffffffu, cells, o);
		inv_min = max(inv_min, __shfl_xor_sync(0xffffffffu, inv_min, o));
		key_max = max(key_max, __shfl_xor_sync(0xffffffffu, key_max, o));
	}
	if (lane == 0) {
		s_tiles[0][warp] = tiles;
		s_tiles[1][warp] = cells;
		s_tiles[2][warp] = inv_min;
		s_tiles[3][warp] = key_max;
		s_tiles[4][warp] = (uint32_t)__popc(vis_mask);
	}
	__syncthreads();
	if (threadIdx.x < 2 || threadIdx.x == 4) {
		uint32_t sum = 0;
#pragma unroll
		for (int w = 0; w < PRE_THREADS / 32; w++)
			sum += s_tiles[threadIdx.x][w];
		if (sum)
			atomicAdd(a.total_tiles + threadIdx.x, sum);
	} else if (threadIdx.x < 4) {
		uint32_t m = 0;
#pragma unroll
		for (int w = 0; w < PRE_THREADS / 32; w++)
			m = max(m, s_tiles[threadIdx.x][w]);
		if (m)
			atomicMax(a.total_tiles + threadIdx.x, m);
	}
}

// Offsets an optional input (nullptr = absent, which preprocess_body tests) to the view's first row.
__device__ __forceinline__ const float* view_rows(const float* p, size_t floats) { return p != nullptr ? p + floats : p; }

// One view, or a stack of views in ONE launch (brs_forward_views[_ex]): blockIdx.y picks the view; its camera, its
// place in the stack (tile row offset), its input rows and its slice of the instance-indexed outputs come from the
// view table in parameter space.  When the views share one Gaussian set, its inputs are read once per view, the
// later views' reads hitting L2.  A single view runs the same kernel with a one-entry table, so a stacked forward
// and per-view forwards execute the same instructions (two separately compiled copies of the SH evaluation
// differed in the last bit).  The grid has ceil(max count / PRE_THREADS) blocks in x: blocks past their view's
// count leave before they touch anything (shared memory, barriers, the header atomics).
template <bool VEC, bool EAGER>
__global__ void __launch_bounds__(PRE_THREADS) preprocess_kernel(PreprocessArgs a, PreprocessViewTable t)
{
	const PreprocessViewTable::Slot v = t.v[blockIdx.y];
	if (blockIdx.x * PRE_THREADS >= v.count)
		return;
	const size_t row = v.row, first = v.inst;
	a.means3D += 3 * row;
	a.scales = view_rows(a.scales, 3 * row);
	a.rotations = view_rows(a.rotations, 4 * row);
	a.opacities += row;
	a.shs = view_rows(a.shs, (size_t)(3 * a.M) * row);
	a.cov3D_precomp = view_rows(a.cov3D_precomp, 6 * row);
	a.colors_precomp = view_rows(a.colors_precomp, 3 * row);
	a.radii += first;
	a.records += 3 * first;
	a.depth_key += first;
	a.rect += first;
	const uint32_t row_offset = (t.first_view + blockIdx.y) * a.grid_y;
	preprocess_body<VEC, EAGER>(a, v, row_offset);
}

// ---- K10 ----------------------------------------------------------------------------------------

__global__ void __launch_bounds__(256) filter_kernel(FilterArgs a)
{
	__shared__ float s_cam[36];
	stage_camera(s_cam, a.viewmatrix, a.projmatrix, nullptr);
	__syncthreads();
	const int idx = blockIdx.x * blockDim.x + threadIdx.x;
	if (idx >= a.P)
		return;
	const GeomInputs in = load_geom_inputs(a.means3D, a.scales, a.scales_stride, a.rotations, a.cov3D_precomp, idx, a.scale_modifier);
	Geometry g;
	bool visible = compute_geometry(in, s_cam, s_cam + 16, a.W, a.H, a.tan_fovx, a.tan_fovy, a.focal_x, a.focal_y, a.grid_x,
	                                a.grid_y, a.prefiltered != 0, g);
	a.radii[idx] = visible ? g.radius : 0;
}

// K10 fused with the compaction its caller does next (SURVEY.md 8f N2): BloomScene turns the radii into
// visible_mask = radii > 0 and boolean-indexes anchors, features, offsets, scalings with it
// (gaussian_renderer/__init__.py:294-349, :39-60) - one torch nonzero (and one host synchronisation) per
// indexed tensor.  This kernel also writes the ascending list of visible indices and their count, so the caller
// gathers with index_select after a single read of the count.  Order-preserving compaction: block scan +
// decoupled look-back over blocks (tickets handed out in order).
__global__ void __launch_bounds__(256) filter_compact_kernel(FilterArgs a)
{
	__shared__ float s_cam[36];
	__shared__ uint32_t s_warp[8];
	__shared__ uint32_t s_bcast[2];
	constexpr uint32_t F_LOCAL = 1u << 30, F_INCL = 2u << 30, F_MASK = 3u << 30;
	const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
	if (tid == 0)
		s_bcast[0] = atomicAdd(a.ticket, 1u);
	stage_camera(s_cam, a.viewmatrix, a.projmatrix, nullptr);
	__syncthreads();
	const uint32_t blk = s_bcast[0];
	const int idx = (int)(blk * 256 + tid);
	bool visible = false;
	if (idx < a.P) {
		const GeomInputs in = load_geom_inputs(a.means3D, a.scales, a.scales_stride, a.rotations, a.cov3D_precomp, idx, a.scale_modifier);
		Geometry g;
		visible = compute_geometry(in, s_cam, s_cam + 16, a.W, a.H, a.tan_fovx, a.tan_fovy, a.focal_x, a.focal_y, a.grid_x,
		                           a.grid_y, a.prefiltered != 0, g);
		a.radii[idx] = visible ? g.radius : 0;
	}
	const uint32_t vmask = __ballot_sync(0xffffffffu, visible);
	if (lane == 0)
		s_warp[warp] = __popc(vmask);
	__syncthreads();
	uint32_t warp_off = 0, block_total = 0;
#pragma unroll
	for (int w = 0; w < 8; w++) {
		if ((uint32_t)w < warp)
			warp_off += s_warp[w];
		block_total += s_warp[w];
	}
	if (warp == 0) {
		if (lane == 0) {
			const uint32_t v = (blk == 0 ? F_INCL : F_LOCAL) | block_total;
			asm volatile("st.relaxed.gpu.global.u32 [%0], %1;" ::"l"(a.status + blk), "r"(v) : "memory");
		}
		uint32_t excl = 0;
		int p = (int)blk - 1;
		while (p >= 0) {
			const int q = p - (int)lane;
			uint32_t v = F_INCL;
			if (q >= 0)
				asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(a.status + q) : "memory");
			const uint32_t f = v & F_MASK;
			const uint32_t not_ready = __ballot_sync(0xffffffffu, f == 0);
			const uint32_t inclusive = __ballot_sync(0xffffffffu, f == F_INCL);
			const int first_nr = not_ready ? __ffs(not_ready) - 1 : 32;
			const int first_in = inclusive ? __ffs(inclusive) - 1 : 32;
			const int take = (first_in < first_nr) ? first_in + 1 : first_nr;
			uint32_t c = ((int)lane < take) ? (v & ~F_MASK) : 0u;
#pragma unroll
			for (int o = 16; o > 0; o >>= 1)
				c += __shfl_xor_sync(0xffffffffu, c, o);
			excl += c;
			if (first_in < first_nr)
				break;
			p -= first_nr;
		}
		if (lane == 0) {
			if (blk > 0) {
				const uint32_t v = F_INCL | (excl + block_total);
				asm volatile("st.relaxed.gpu.global.u32 [%0], %1;" ::"l"(a.status + blk), "r"(v) : "memory");
			}
			s_bcast[1] = excl;
			if (blk == gridDim.x - 1)
				*a.count = excl + block_total;
		}
	}
	__syncthreads();
	if (visible)
		a.indices[s_bcast[1] + warp_off + __popc(vmask & lanemask_lt())] = (long long)idx;
}

// ---- K11 ----------------------------------------------------------------------------------------

__global__ void __launch_bounds__(256)
    check_frustum_kernel(int P, const float* means3D, const float* viewmatrix, uint8_t* present)
{
	__shared__ float s_view[16];
	if (threadIdx.x < 16)
		s_view[threadIdx.x] = __ldg(viewmatrix + threadIdx.x);
	__syncthreads();
	const int idx = blockIdx.x * blockDim.x + threadIdx.x;
	if (idx >= P)
		return;
	const float* mp = means3D + 3 * (size_t)idx;
	float3 p_orig = {__ldg(mp), __ldg(mp + 1), __ldg(mp + 2)};
	float3 p_view = transform_point_4x3(p_orig, s_view);
	present[idx] = (p_view.z <= 0.2f) ? 0 : 1;
}

// ---- launchers ----------------------------------------------------------------------------------

// The grid is sized by the largest view of the launch (not a flat grid over all rows with a per-block search of
// the table): the block -> (view, row) map stays blockIdx.y / blockIdx.x * PRE_THREADS as for a single view, at
// the price of blocks that exit at once in the shorter views of a ragged stack.
cudaError_t launch_preprocess(const PreprocessArgs& a, const PreprocessViewTable& t, int n_views, cudaStream_t stream)
{
	if (n_views <= 0)
		return cudaSuccess;
	if (n_views > PreprocessViewTable::MAX_VIEWS)
		return cudaErrorInvalidValue;
	uint32_t max_count = 0;
	for (int k = 0; k < n_views; k++)
		max_count = t.v[k].count > max_count ? t.v[k].count : max_count;
	if (max_count == 0)
		return cudaSuccess;
	const dim3 grid((max_count + PRE_THREADS - 1) / PRE_THREADS, n_views, 1);
	size_t smem = 0;
	bool vec = false;
	if (a.shs != nullptr) {
		vec = (a.M == 16) && ((reinterpret_cast<uintptr_t>(a.shs) & 15u) == 0);
		smem = vec ? (size_t)(PRE_THREADS / 2) * SH_PAIR_PITCH * sizeof(float4) : (size_t)PRE_THREADS * ((3 * a.M) | 1) * sizeof(float);
	}
	if (vec && a.eager_sh)
		preprocess_kernel<true, true><<<grid, PRE_THREADS, smem, stream>>>(a, t);
	else if (vec)
		preprocess_kernel<true, false><<<grid, PRE_THREADS, smem, stream>>>(a, t);
	else
		preprocess_kernel<false, false><<<grid, PRE_THREADS, smem, stream>>>(a, t);
	count_launch();
	return cudaGetLastError();
}

cudaError_t launch_filter(const FilterArgs& a, cudaStream_t stream)
{
	if (a.P <= 0)
		return cudaSuccess;
	if (a.indices != nullptr)
		filter_compact_kernel<<<(a.P + 255) / 256, 256, 0, stream>>>(a);
	else
		filter_kernel<<<(a.P + 255) / 256, 256, 0, stream>>>(a);
	count_launch();
	return cudaGetLastError();
}

cudaError_t launch_check_frustum(int P, const float* means3D, const float* viewmatrix, uint8_t* present,
                                 cudaStream_t stream)
{
	if (P <= 0)
		return cudaSuccess;
	check_frustum_kernel<<<(P + 255) / 256, 256, 0, stream>>>(P, means3D, viewmatrix, present);
	count_launch();
	return cudaGetLastError();
}

} // namespace brs

// Backward of the per-Gaussian preprocessing for sm_100a: ONE kernel for the reference's two
//   computeCov2DCUDA (cuda_rasterizer/backward.cu:144-274)  and
//   preprocessCUDA   (backward.cu:346-396) with computeColorFromSH (20-139) / computeCov3D (278-341).
//
// Fusing them removes the dL_dcov3D / dL_dmeans round trip through HBM, and this kernel also
//   * consumes the blend-backward accumulator (48 B per Gaussian) and applies the per-Gaussian
//     constants (0.5*W, 0.5*H, -0.5) that the reference multiplies into every pair;
//   * writes EVERY element of every gradient tensor (zeros for Gaussians with radii <= 0), so the
//     caller needs no zero-fill: the reference zero-fills (108 + 12 M) bytes per Gaussian first
//     (rasterize_points.cu:154-162);
//   * or, in ACCUMULATE mode (brs_grads.accumulate, used by the view-sharded step), adds the parameter
//     gradients of the visible Gaussians straight into the caller's gradient bucket with float
//     reductions (red.global.add, 16-byte vectors for the SH rows), which replaces one fresh
//     (44 + 12 M)-byte-per-Gaussian tensor set plus a read-modify-write pass over the bucket per view
//     by a single reduction of the visible rows — and is safe when views on different streams add
//     into the same bucket concurrently;
//   * recomputes the 3D covariance and the SH colour sign (`clamped`, with the forward's own function)
//     instead of reading stored copies;
//   * fetches SH rows with one bulk asynchronous copy per Gaussian (cp.async.bulk + mbarrier) and writes
//     dL_dsh rows through shared memory in 48-byte chunks, consecutive lanes to consecutive addresses.
// The per-Gaussian maths is NOT the reference's statement sequence: it is derived from the forward model
// in matrix form (preprocess_bwd_math.h: dL/dC2 = -conic G conic, dL/dSigma = T^T H T, dL/dT = 2 H T Sigma
// with Sigma T shared between the forward recompute and the gradient, K = 2 G Rq diag(s^2) for the
// quaternion, SH coefficients contracted with dL_dRGB before the basis gradients are applied) and checked
// against finite differences on the CPU (tests/test_bwd_math.py) and against the reference on the GPU.
#include "common.cuh"
#include "gaussian_math.cuh"
#include "kernels.h"
#include "preprocess_bwd_math.h"

namespace brs {

namespace {

constexpr int PB_THREADS = 128;

// 16-byte vector reduction (sm_90+): four float adds in one L2 atomic, no return value.
__device__ __forceinline__ void red_add_v4(float* addr, float x, float y, float z, float w)
{
	asm volatile("red.relaxed.gpu.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(addr), "f"(x), "f"(y), "f"(z), "f"(w)
	             : "memory");
}
constexpr int FACT_PITCH = 19; // 16 basis values + dL_dRGB, odd pitch -> conflict-free

// VEC / EAGER: as in the forward preprocess (preprocess.cu) - SH rows arrive by one bulk asynchronous copy per
// lane, either for the whole warp at the very start (EAGER) or for the rendered Gaussians once `radii` is known.
// STATS: also add the densification statistics of this view (brs_densify_stats).  A template parameter, not a
// runtime branch, so that the instantiations without it compile to the code they had before the option existed.
template <bool VEC, bool EAGER, bool STATS>
__global__ void __launch_bounds__(PB_THREADS, 6) preprocess_backward_kernel(PreprocessBwdArgs a)
{
	using namespace bwdmath;
	extern __shared__ float4 s_dyn[]; // SH rows in | basis rows out
	__shared__ float s_cam[36];
	__shared__ uint64_t s_bar[PB_THREADS / 32];

	const int block_first = blockIdx.x * PB_THREADS;
	const int idx = block_first + threadIdx.x;
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	const bool in_range = idx < a.P;
	const bool bulk = VEC && a.shs != nullptr;

	if (bulk) {
		if (lane == 0)
			mbar_init(&s_bar[warp], 1);
		__syncwarp();
		if (EAGER) {
			// even lanes fetch their own row and their neighbour's (one 384-byte copy; 192 at the end of the array)
			const uint32_t rows = (uint32_t)max(0, min(32, a.P - (block_first + 32 * warp)));
			if (in_range && !(lane & 1))
				bulk_copy_g2s(s_dyn + sh_row_slot(threadIdx.x), a.shs + (size_t)idx * 48, idx + 1 < a.P ? 384u : 192u, &s_bar[warp]);
			if (lane == 0)
				mbar_arrive_expect_tx(&s_bar[warp], 192u * rows);
		}
	}
	// every per-Gaussian input is requested before anything is computed (one exposed round trip, not four)
	int radius = 0;
	float4 a0 = make_float4(0.f, 0.f, 0.f, 0.f), a1 = a0, a2 = a0;
	V3 mean = {0.f, 0.f, 0.f}, scale = {0.f, 0.f, 0.f};
	float4 rot = a0;
	float cov_in[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
	if (in_range) {
		radius = __ldg(a.radii + idx);
		const float4* ap = reinterpret_cast<const float4*>(a.accum + (size_t)idx * ACCUM_STRIDE);
		a0 = __ldg(ap);
		a1 = __ldg(ap + 1);
		a2 = __ldg(ap + 2);
		const float* mp = a.means3D + 3 * (size_t)idx;
		mean = vec3(__ldg(mp), __ldg(mp + 1), __ldg(mp + 2));
		if (a.cov3D_precomp != nullptr) {
#pragma unroll
			for (int i = 0; i < 6; i++)
				cov_in[i] = __ldg(a.cov3D_precomp + 6 * (size_t)idx + i);
		} else {
			const float* sp = a.scales + 3 * (size_t)idx;
			scale = vec3(__ldg(sp), __ldg(sp + 1), __ldg(sp + 2));
			const float* rp = a.rotations + 4 * (size_t)idx;
			rot = make_float4(__ldg(rp), __ldg(rp + 1), __ldg(rp + 2), __ldg(rp + 3));
		}
	}
	{
		const int t = threadIdx.x;
		if (t < 16)
			s_cam[t] = __ldg(a.viewmatrix + t);
		else if (t < 32)
			s_cam[t] = __ldg(a.projmatrix + t - 16);
		else if (t < 35 && a.campos != nullptr) // only the SH chain reads it; colors_precomp callers may pass none
			s_cam[t] = __ldg(a.campos + t - 32);
	}
	__syncthreads(); // camera block
	const float* view = s_cam;
	const float* proj = s_cam + 16;

	const bool visible = in_range && radius > 0;
	const uint32_t vis_mask = __ballot_sync(0xffffffffu, visible);
	const int row_f = 3 * a.M;
	const int warp_first = block_first + 32 * warp;
	if (a.shs != nullptr) {
		if (VEC) {
			if (!EAGER) {
				// a pair of rows is fetched (by its even lane) when either of its Gaussians was rendered
				const uint32_t pair_mask = (vis_mask | (vis_mask >> 1)) & 0x55555555u;
				const uint32_t short_pair = (in_range && !(lane & 1) && idx + 1 >= a.P && ((pair_mask >> lane) & 1u)) ? 1u : 0u;
				if (in_range && ((pair_mask >> lane) & 1u))
					bulk_copy_g2s(s_dyn + sh_row_slot(threadIdx.x), a.shs + (size_t)idx * 48, short_pair ? 192u : 384u, &s_bar[warp]);
				const uint32_t shorts = __popc(__ballot_sync(0xffffffffu, short_pair != 0u));
				if (lane == 0)
					mbar_arrive_expect_tx(&s_bar[warp], 384u * (uint32_t)__popc(pair_mask) - 192u * shorts);
			}
		} else {
			const int pitch = row_f | 1;
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
	}

	// basis values + dL_dRGB of this Gaussian go straight to their own shared-memory row (not through
	// registers); rows of Gaussians that do not run the SH chain must read as zero
	float* const s_fact = reinterpret_cast<float*>(s_dyn) + a.fact_offset;
	float* const fact = s_fact + threadIdx.x * FACT_PITCH;
	const bool sh_rows = a.dL_dsh != nullptr && a.M > 0;
	if (sh_rows && !(visible && a.shs != nullptr)) {
#pragma unroll
		for (int k = 0; k < FACT_PITCH; k++)
			fact[k] = 0.f;
	}

	float o_m2x = 0.f, o_m2y = 0.f, o_opacity = 0.f;
	V3 o_color = {0.f, 0.f, 0.f}, o_mean = {0.f, 0.f, 0.f}, o_scale = {0.f, 0.f, 0.f};
	float4 o_rot = make_float4(0.f, 0.f, 0.f, 0.f);
	Sym3 dSigma = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};

	if (visible) {
		// the blend backward leaves sums over (pixel, Gaussian) pairs; the per-Gaussian constants the reference
		// multiplies into every pair (backward.cu:473-474,574-580) are applied here, once
		o_m2x = a0.x * (0.5f * a.W);
		o_m2y = a0.y * (0.5f * a.H);
		const float gx = -0.5f * a0.z, gy = -0.5f * a0.w, gz = -0.5f * a1.x;
		o_opacity = a1.y;
		o_color = vec3(a1.z, a1.w, a2.x);

		Sym3 Sigma;
		Rot R = {};
		V3 s = {0.f, 0.f, 0.f};
		if (a.cov3D_precomp != nullptr) {
			Sigma = Sym3{cov_in[0], cov_in[1], cov_in[2], cov_in[3], cov_in[4], cov_in[5]};
		} else {
			R = rotation(rot.x, rot.y, rot.z, rot.w);
			s = vec3(a.scale_modifier * scale.x, a.scale_modifier * scale.y, a.scale_modifier * scale.z);
			Sigma = covariance(R, s);
		}
		const ProjectionGrad pg = projection_backward(view, mean, Sigma, a.focal_x, a.focal_y, a.tan_fovx, a.tan_fovy, gx, gy, gz);
		dSigma = pg.dSigma;
		const V3 px = pixel_backward(proj, mean, o_m2x, o_m2y);
		o_mean = vec3(pg.dmean.x + px.x, pg.dmean.y + px.y, pg.dmean.z + px.z);
		if (a.depth_gradient) {
			// opt-in depth gradient: z = p_view.z = view[2] x + view[6] y + view[10] z + view[14] (forward.cu:186)
			const float dz = a2.y;
			o_mean.x += view[2] * dz;
			o_mean.y += view[6] * dz;
			o_mean.z += view[10] * dz;
		}
		if (a.scales != nullptr) {
			const ShapeGrad sg = shape_backward(R, s, rot.x, rot.y, rot.z, rot.w, dSigma);
			o_scale = sg.dscale;
			o_rot = make_float4(sg.dr, sg.dx, sg.dy, sg.dz);
		}

		if (a.shs != nullptr) {
			if (VEC)
				mbar_wait(&s_bar[warp], 0u);
			const v3 pos = make_v3(mean.x, mean.y, mean.z);
			const v3 cam = make_v3(s_cam[32], s_cam[33], s_cam[34]);
			const V3 vdir = vec3(mean.x - cam.x, mean.y - cam.y, mean.z - cam.z);
			const float inv_len = 1.0f / sqrtf(dot(vdir, vdir));
			const V3 dir = vec3(vdir.x * inv_len, vdir.y * inv_len, vdir.z * inv_len);
			// the colour's sign decides whether its gradient passes (`clamped`, forward.cu:67-70): evaluated
			// with the forward's own function so that both directions take the same decision
			V3 g_rgb;
			float q[16];
			if (VEC) {
				const ShRowView c{s_dyn + sh_row_slot(threadIdx.x)};
				const v3 rgb = eval_sh(a.D, pos, cam, c);
				g_rgb = vec3(rgb.x < 0 ? 0.f : o_color.x, rgb.y < 0 ? 0.f : o_color.y, rgb.z < 0 ? 0.f : o_color.z);
#pragma unroll
				for (int k = 0; k < 16; k++)
					q[k] = c[3 * k] * g_rgb.x + c[3 * k + 1] * g_rgb.y + c[3 * k + 2] * g_rgb.z;
			} else {
				const float* sh = reinterpret_cast<const float*>(s_dyn) + threadIdx.x * (row_f | 1);
				const v3 rgb = eval_sh(a.D, pos, cam, sh);
				g_rgb = vec3(rgb.x < 0 ? 0.f : o_color.x, rgb.y < 0 ? 0.f : o_color.y, rgb.z < 0 ? 0.f : o_color.z);
#pragma unroll
				for (int k = 0; k < 16; k++)
					q[k] = (k < a.M) ? sh[3 * k] * g_rgb.x + sh[3 * k + 1] * g_rgb.y + sh[3 * k + 2] * g_rgb.z : 0.f;
			}
			const V3 g_dir = sh_direction_gradient(a.D, dir.x, dir.y, dir.z, q);
			const V3 g_pos = normalize_backward(dir, inv_len, g_dir);
			o_mean.x += g_pos.x;
			o_mean.y += g_pos.y;
			o_mean.z += g_pos.z;
			if (sh_rows) {
				sh_basis(a.D, dir.x, dir.y, dir.z, fact);
				fact[16] = g_rgb.x;
				fact[17] = g_rgb.y;
				fact[18] = g_rgb.z;
			}
		}
	}
	if (VEC && EAGER && a.shs != nullptr && !visible)
		mbar_wait(&s_bar[warp], 0u); // the copies into this CTA's shared memory must have landed before it exits

	// ---- per-Gaussian outputs ----
	// plain mode: every row of every tensor is written (zeros for culled Gaussians);
	// accumulate mode: parameter gradients of VISIBLE Gaussians are added to what the buffers hold,
	// other rows are left alone; dL_dmeans2D is a per-view statistic and is always overwritten.
	if (in_range) {
		float* p;
		p = a.dL_dmeans2D + 3 * (size_t)idx;
		p[0] = o_m2x; p[1] = o_m2y; p[2] = 0.f;
		if (STATS && visible) {
			// reference scene/gaussian_model.py:756-759: norm of the per-view means2D gradient and one count per
			// rendered Gaussian (also when that gradient is zero).  Float reductions: views on other streams add
			// into the same accumulators concurrently.
			const long long slot = a.stats_index != nullptr ? __ldg(a.stats_index + idx) : (long long)idx;
			if (slot >= 0 && slot < a.stats_rows) {
				atomicAdd(a.stats_grad_norm + slot, sqrtf(o_m2x * o_m2x + o_m2y * o_m2y));
				atomicAdd(a.stats_count + slot, 1.0f);
			}
		}
		if (!a.accumulate) {
			p = a.dL_dcolors + 3 * (size_t)idx;
			p[0] = o_color.x; p[1] = o_color.y; p[2] = o_color.z;
			a.dL_dopacity[idx] = o_opacity;
			p = a.dL_dmeans3D + 3 * (size_t)idx;
			p[0] = o_mean.x; p[1] = o_mean.y; p[2] = o_mean.z;
			// reference layout of dL_dcov3D: the six unique entries, off-diagonal ones counted twice
			p = a.dL_dcov3D + 6 * (size_t)idx;
			p[0] = dSigma.xx; p[1] = 2.f * dSigma.xy; p[2] = 2.f * dSigma.xz;
			p[3] = dSigma.yy; p[4] = 2.f * dSigma.yz; p[5] = dSigma.zz;
			p = a.dL_dscales + 3 * (size_t)idx;
			p[0] = o_scale.x; p[1] = o_scale.y; p[2] = o_scale.z;
			p = a.dL_drotations + 4 * (size_t)idx;
			p[0] = o_rot.x; p[1] = o_rot.y; p[2] = o_rot.z; p[3] = o_rot.w;
		} else if (visible) {
			// float atomics (RED, no return value): several views may be adding into the same bucket from
			// different streams at the same time.  A NULL sink is a parameter the caller froze.
			if (a.dL_dmeans3D != nullptr) {
				float* p3 = a.dL_dmeans3D + 3 * (size_t)idx;
				atomicAdd(p3 + 0, o_mean.x);
				atomicAdd(p3 + 1, o_mean.y);
				atomicAdd(p3 + 2, o_mean.z);
			}
			if (a.dL_dopacity != nullptr)
				atomicAdd(a.dL_dopacity + idx, o_opacity);
			if (a.scales != nullptr) {
				if (a.dL_dscales != nullptr) {
					float* ps = a.dL_dscales + 3 * (size_t)idx;
					atomicAdd(ps + 0, o_scale.x);
					atomicAdd(ps + 1, o_scale.y);
					atomicAdd(ps + 2, o_scale.z);
				}
				if (a.dL_drotations != nullptr) {
					float* pr = a.dL_drotations + 4 * (size_t)idx;
					if ((reinterpret_cast<uintptr_t>(a.dL_drotations) & 15u) == 0) {
						red_add_v4(pr, o_rot.x, o_rot.y, o_rot.z, o_rot.w);
					} else { // a bucket slice that is not 16-byte aligned (odd P)
						atomicAdd(pr + 0, o_rot.x);
						atomicAdd(pr + 1, o_rot.y);
						atomicAdd(pr + 2, o_rot.z);
						atomicAdd(pr + 3, o_rot.w);
					}
				}
			} else if (a.dL_dcov3D != nullptr) {
				p = a.dL_dcov3D + 6 * (size_t)idx;
				atomicAdd(p + 0, dSigma.xx);
				atomicAdd(p + 1, 2.f * dSigma.xy);
				atomicAdd(p + 2, 2.f * dSigma.xz);
				atomicAdd(p + 3, dSigma.yy);
				atomicAdd(p + 4, 2.f * dSigma.yz);
				atomicAdd(p + 5, dSigma.zz);
			}
			if (a.shs == nullptr && a.dL_dcolors != nullptr) {
				p = a.dL_dcolors + 3 * (size_t)idx;
				atomicAdd(p + 0, o_color.x);
				atomicAdd(p + 1, o_color.y);
				atomicAdd(p + 2, o_color.z);
			}
		}
	}

	// ---- dL_dsh rows: dL_dsh[k][c] = basis_k * dL_dRGB[c], written through shared memory ----
	if (sh_rows) {
		__syncwarp(); // the 32 rows of this warp in s_fact are complete
		const int rows = min(32, a.P - warp_first);
		const float* wfact = s_fact + 32 * warp * FACT_PITCH;
		if (VEC) {
			// a row is 16 coefficients x 3 channels = four 48-byte chunks of 4 coefficients each; lane l takes
			// chunks l, l + 32, l + 64, l + 96 of the warp's 128: consecutive lanes write consecutive 48 bytes
			float4* dst = reinterpret_cast<float4*>(a.dL_dsh) + (size_t)warp_first * 12;
#pragma unroll
			for (int k = 0; k < 4; k++) {
				const int chunk = lane + 32 * k;
				const int row = chunk >> 2, c4 = (chunk & 3) * 4;
				if (row < rows && (!a.accumulate || ((vis_mask >> row) & 1u))) {
					const float* fr = wfact + row * FACT_PITCH;
					const float r = fr[16], g = fr[17], b = fr[18];
					const float b0 = fr[c4], b1 = fr[c4 + 1], b2 = fr[c4 + 2], b3 = fr[c4 + 3];
					float4* o = dst + 3 * chunk;
					if (a.accumulate) {
						red_add_v4(reinterpret_cast<float*>(o), b0 * r, b0 * g, b0 * b, b1 * r);
						red_add_v4(reinterpret_cast<float*>(o + 1), b1 * g, b1 * b, b2 * r, b2 * g);
						red_add_v4(reinterpret_cast<float*>(o + 2), b2 * b, b3 * r, b3 * g, b3 * b);
					} else {
						o[0] = make_float4(b0 * r, b0 * g, b0 * b, b1 * r);
						o[1] = make_float4(b1 * g, b1 * b, b2 * r, b2 * g);
						o[2] = make_float4(b2 * b, b3 * r, b3 * g, b3 * b);
					}
				}
			}
		} else {
			float* dst = a.dL_dsh + (size_t)warp_first * row_f;
			const int total = rows * row_f;
			for (int f = lane; f < total; f += 32) {
				const int row = f / row_f, e = f - row * row_f;
				const float* fr = wfact + row * FACT_PITCH;
				const float val = fr[e / 3] * fr[16 + (e % 3)];
				if (!a.accumulate)
					dst[f] = val;
				else if ((vis_mask >> row) & 1u)
					atomicAdd(dst + f, val);
			}
		}
	}
}

template <bool VEC, bool EAGER>
void launch_as(const PreprocessBwdArgs& args, int blocks, size_t smem, cudaStream_t stream)
{
	if (args.stats_grad_norm != nullptr)
		preprocess_backward_kernel<VEC, EAGER, true><<<blocks, PB_THREADS, smem, stream>>>(args);
	else
		preprocess_backward_kernel<VEC, EAGER, false><<<blocks, PB_THREADS, smem, stream>>>(args);
}

} // namespace

cudaError_t launch_preprocess_backward(const PreprocessBwdArgs& a, cudaStream_t stream)
{
	if (a.P <= 0)
		return cudaSuccess;
	const int blocks = (a.P + PB_THREADS - 1) / PB_THREADS;
	// dynamic shared memory: [SH rows in | basis-factor rows out]
	size_t in = 0;
	bool vec = false;
	if (a.shs != nullptr) {
		vec = (a.M == 16) && ((reinterpret_cast<uintptr_t>(a.shs) & 15u) == 0) &&
		      ((reinterpret_cast<uintptr_t>(a.dL_dsh) & 15u) == 0);
		in = vec ? align_up((size_t)(PB_THREADS / 2) * SH_PAIR_PITCH * sizeof(float4), 16) : align_up((size_t)PB_THREADS * ((3 * a.M) | 1) * sizeof(float), 16);
	}
	PreprocessBwdArgs args = a;
	args.fact_offset = (int)(in / sizeof(float));
	const size_t smem = in + (size_t)PB_THREADS * FACT_PITCH * sizeof(float);
	if (vec && a.eager_sh)
		launch_as<true, true>(args, blocks, smem, stream);
	else if (vec)
		launch_as<true, false>(args, blocks, smem, stream);
	else
		launch_as<false, false>(args, blocks, smem, stream);
	count_launch();
	return cudaGetLastError();
}

} // namespace brs

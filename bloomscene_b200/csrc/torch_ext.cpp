// Thin PyTorch binding over the C-ABI in include/bloomrast.h.  Compiled by g++ only (no CUDA code
// here); every compute call goes through libbloomrast.so.
//
// Mirrors the reference's binding: module functions, argument order and return tuples of
// ext.cpp:15-20 / rasterize_points.cu:35-288, so the reference's Python wrapper
// (depth_diff_gaussian_rasterization/__init__.py) works unchanged on top of it:
//   rasterize_gaussians(19 args)            -> (R, color, depth, radii, geomBuffer, binningBuffer, imgBuffer)
//   rasterize_gaussians_backward(22 args)   -> (dL_dmeans2D, dL_dcolors, dL_dopacity, dL_dmeans3D,
//                                               dL_dcov3D, dL_dsh, dL_dscales, dL_drotations)
//   rasterize_aussians_filter(13 args)      -> radii            (the reference's own spelling)
//   mark_visible(means3D, view, proj)       -> bool[P]
// Differences: work is issued on torch's CURRENT stream (the reference uses the legacy default
// stream), gradient tensors are torch::empty (the kernels write every element), and C-ABI status
// codes become exceptions here, never inside the library.
#include <c10/cuda/CUDAGuard.h>
#include <c10/cuda/CUDAStream.h>
#include <torch/extension.h>

#include <string>
#include <tuple>
#include <vector>

#include "../../include/bloomrast.h"

namespace {

struct AllocCtx {
	torch::TensorOptions byte_opts;
	torch::Tensor geom, binning, image;
	std::vector<torch::Tensor> scratch;
};

void* alloc_cb(void* vctx, int which, size_t bytes)
{
	auto* ctx = static_cast<AllocCtx*>(vctx);
	try {
		torch::Tensor t = torch::empty({(int64_t)bytes}, ctx->byte_opts);
		void* p = t.data_ptr();
		switch (which) {
		case BRS_BUF_GEOM: ctx->geom = t; break;
		case BRS_BUF_BINNING: ctx->binning = t; break;
		case BRS_BUF_IMAGE: ctx->image = t; break;
		default: ctx->scratch.push_back(t); break;
		}
		return p;
	} catch (...) {
		return nullptr; // no exceptions across the C ABI
	}
}

void check_status(int st, const char* what)
{
	if (st == BRS_OK)
		return;
	std::string msg = std::string(what) + ": " + brs_error_string(st);
	if (st == BRS_ERR_CUDA)
		msg += std::string(" [") + brs_last_cuda_error_string() + "]";
	TORCH_CHECK(false, msg);
}

// Absent optionals arrive as empty (CPU) tensors: reference Python passes torch.Tensor([])
// (depth_diff_gaussian_rasterization/__init__.py:198-208) and relies on data_ptr()==nullptr.
const float* opt_ptr(const torch::Tensor& t, torch::Tensor& keep, const char* name)
{
	if (!t.defined() || t.numel() == 0)
		return nullptr;
	TORCH_CHECK(t.is_cuda(), name, " must be a CUDA tensor");
	TORCH_CHECK(t.scalar_type() == torch::kFloat32, name, " must be float32");
	keep = t.contiguous();
	return keep.data_ptr<float>();
}

const float* req_ptr(const torch::Tensor& t, torch::Tensor& keep, const char* name)
{
	TORCH_CHECK(t.defined() && t.is_cuda(), name, " must be a CUDA tensor");
	TORCH_CHECK(t.scalar_type() == torch::kFloat32, name, " must be float32");
	keep = t.contiguous();
	return keep.data_ptr<float>();
}

brs_stream current_stream() { return reinterpret_cast<brs_stream>(c10::cuda::getCurrentCUDAStream().stream()); }

} // namespace

using ForwardTuple = std::tuple<int, torch::Tensor, torch::Tensor, torch::Tensor, torch::Tensor, torch::Tensor, torch::Tensor>;

// Extension of the reference binding: the same 19 arguments plus brs_fwd_options (include/bloomrast.h).
// `report`: pinned CPU int32[8] that a DEFERRED forward fills asynchronously.
ForwardTuple RasterizeGaussiansExCUDA(const torch::Tensor& background, const torch::Tensor& means3D, const torch::Tensor& colors,
                                      const torch::Tensor& opacity, const torch::Tensor& scales, const torch::Tensor& rotations,
                                      const float scale_modifier, const torch::Tensor& cov3D_precomp,
                                      const torch::Tensor& viewmatrix, const torch::Tensor& projmatrix, const float tan_fovx,
                                      const float tan_fovy, const int image_height, const int image_width,
                                      const torch::Tensor& sh, const int degree, const torch::Tensor& campos,
                                      const bool prefiltered, const bool debug, const int mode, const int R_cap,
                                      const int R1_cap, const int depth_bits, const c10::optional<torch::Tensor>& report,
                                      const c10::optional<torch::Tensor>& overflow_accum)
{
	if (means3D.ndimension() != 2 || means3D.size(1) != 3) {
		AT_ERROR("means3D must have dimensions (num_points, 3)");
	}
	TORCH_CHECK(means3D.is_cuda(), "means3D must be a CUDA tensor");
	c10::cuda::CUDAGuard guard(means3D.device());

	const int P = means3D.size(0);
	const int H = image_height;
	const int W = image_width;

	auto float_opts = means3D.options().dtype(torch::kFloat32);
	auto int_opts = means3D.options().dtype(torch::kInt32);
	torch::Tensor out_color = torch::empty({3, H, W}, float_opts);
	torch::Tensor out_depth = torch::empty({1, H, W}, float_opts);
	torch::Tensor radii = torch::empty({P}, int_opts);

	AllocCtx ctx;
	ctx.byte_opts = torch::TensorOptions(torch::kByte).device(means3D.device());
	ctx.geom = torch::empty({0}, ctx.byte_opts);
	ctx.binning = torch::empty({0}, ctx.byte_opts);
	ctx.image = torch::empty({0}, ctx.byte_opts);

	torch::Tensor k[11];
	brs_view view{};
	view.image_width = W;
	view.image_height = H;
	view.tanfovx = tan_fovx;
	view.tanfovy = tan_fovy;
	view.scale_modifier = scale_modifier;
	view.sh_degree = degree;
	view.prefiltered = prefiltered;
	view.debug = debug;
	view.bg = req_ptr(background, k[0], "bg");
	view.viewmatrix = req_ptr(viewmatrix, k[1], "viewmatrix");
	view.projmatrix = req_ptr(projmatrix, k[2], "projmatrix");
	view.campos = opt_ptr(campos, k[3], "campos");

	brs_gaussians g{};
	g.P = P;
	g.means3D = req_ptr(means3D, k[4], "means3D");
	g.opacities = P ? req_ptr(opacity, k[5], "opacities") : nullptr;
	g.shs = opt_ptr(sh, k[6], "shs");
	g.colors_precomp = opt_ptr(colors, k[7], "colors_precomp");
	g.scales = opt_ptr(scales, k[8], "scales");
	g.rotations = opt_ptr(rotations, k[9], "rotations");
	g.cov3D_precomp = opt_ptr(cov3D_precomp, k[10], "cov3D_precomp");
	view.sh_coeffs = (g.shs != nullptr) ? (int)sh.size(1) : 0; // rasterize_points.cu:84-88

	brs_fwd_options opt{};
	opt.mode = mode;
	opt.R_cap = R_cap;
	opt.R1_cap = R1_cap;
	opt.depth_bits = depth_bits;
	if (report.has_value() && report->defined()) {
		TORCH_CHECK(report->is_cpu() && report->is_pinned() && report->scalar_type() == torch::kInt32 && report->numel() >= 8 &&
		                report->is_contiguous(),
		            "report must be a pinned contiguous CPU int32 tensor of at least 8 elements");
		opt.report = reinterpret_cast<uint32_t*>(report->data_ptr<int>());
	}
	if (overflow_accum.has_value() && overflow_accum->defined()) {
		TORCH_CHECK(overflow_accum->is_cuda() && overflow_accum->scalar_type() == torch::kInt32 && overflow_accum->numel() >= 1,
		            "overflow_accum must be a CUDA int32 tensor");
		opt.overflow_accum = reinterpret_cast<uint32_t*>(overflow_accum->data_ptr<int>());
	}
	brs_fwd_state state{};
	int st = brs_forward_ex(&view, &g, out_color.data_ptr<float>(), out_depth.data_ptr<float>(),
	                        P ? radii.data_ptr<int>() : nullptr, alloc_cb, &ctx, &state, &opt, current_stream());
	check_status(st, "rasterize_gaussians");
	return std::make_tuple(state.num_rendered, out_color, out_depth, radii, ctx.geom, ctx.binning, ctx.image);
}

// reference binding (rasterize_points.h:18-40): 19 arguments
ForwardTuple RasterizeGaussiansCUDA(const torch::Tensor& background, const torch::Tensor& means3D, const torch::Tensor& colors,
                                    const torch::Tensor& opacity, const torch::Tensor& scales, const torch::Tensor& rotations,
                                    const float scale_modifier, const torch::Tensor& cov3D_precomp,
                                    const torch::Tensor& viewmatrix, const torch::Tensor& projmatrix, const float tan_fovx,
                                    const float tan_fovy, const int image_height, const int image_width,
                                    const torch::Tensor& sh, const int degree, const torch::Tensor& campos,
                                    const bool prefiltered, const bool debug)
{
	return RasterizeGaussiansExCUDA(background, means3D, colors, opacity, scales, rotations, scale_modifier, cov3D_precomp,
	                                viewmatrix, projmatrix, tan_fovx, tan_fovy, image_height, image_width, sh, degree, campos,
	                                prefiltered, debug, BRS_FWD_AUTO, 0, 0, 0, c10::nullopt, c10::nullopt);
}

// Extension (brs_forward_views): n views of the same Gaussians as ONE pipeline, forward only.
// viewmatrices / projmatrices [n,4,4], camposes [n,3], tan_fovx / tan_fovy one value per view (or one for all).
// Returns (instances of all views, color [n,3,H,W], depth [n,1,H,W], radii [n,P]).
std::tuple<int64_t, torch::Tensor, torch::Tensor, torch::Tensor>
RasterizeGaussiansViewsCUDA(const torch::Tensor& background, const torch::Tensor& means3D, const torch::Tensor& colors,
                            const torch::Tensor& opacity, const torch::Tensor& scales, const torch::Tensor& rotations,
                            const float scale_modifier, const torch::Tensor& cov3D_precomp, const torch::Tensor& viewmatrices,
                            const torch::Tensor& projmatrices, const std::vector<double>& tan_fovx,
                            const std::vector<double>& tan_fovy, const int image_height, const int image_width,
                            const torch::Tensor& sh, const int degree, const torch::Tensor& camposes, const bool prefiltered,
                            const bool debug, const int mode, const c10::optional<torch::Tensor>& color_out,
                            const c10::optional<torch::Tensor>& depth_out)
{
	TORCH_CHECK(means3D.ndimension() == 2 && means3D.size(1) == 3, "means3D must have dimensions (num_points, 3)");
	TORCH_CHECK(means3D.is_cuda(), "means3D must be a CUDA tensor");
	TORCH_CHECK(viewmatrices.ndimension() == 3 && viewmatrices.size(1) == 4 && viewmatrices.size(2) == 4,
	            "viewmatrices must have dimensions (views, 4, 4)");
	const int n = (int)viewmatrices.size(0);
	TORCH_CHECK(n >= 1, "at least one view");
	TORCH_CHECK(projmatrices.sizes() == viewmatrices.sizes(), "projmatrices must have dimensions (views, 4, 4)");
	TORCH_CHECK((tan_fovx.size() == 1 || (int)tan_fovx.size() == n) && (tan_fovy.size() == 1 || (int)tan_fovy.size() == n),
	            "tan_fovx / tan_fovy: one value, or one per view");
	c10::cuda::CUDAGuard guard(means3D.device());

	const int P = means3D.size(0), H = image_height, W = image_width;
	auto float_opts = means3D.options().dtype(torch::kFloat32);
	// the caller may hand in (a slice of) its own output stacks: written in place, no copy afterwards
	auto take = [&](const c10::optional<torch::Tensor>& t, int64_t ch, const char* name) {
		if (!t.has_value() || !t->defined())
			return torch::empty({n, ch, H, W}, float_opts);
		TORCH_CHECK(t->is_cuda() && t->device() == means3D.device() && t->scalar_type() == torch::kFloat32 && t->is_contiguous() &&
		                t->numel() == (int64_t)n * ch * H * W,
		            name, " must be a contiguous float32 CUDA tensor of views x ", ch, " x H x W elements");
		return *t;
	};
	torch::Tensor out_color = take(color_out, 3, "color_out");
	torch::Tensor out_depth = take(depth_out, 1, "depth_out");
	torch::Tensor radii = torch::empty({n, P}, means3D.options().dtype(torch::kInt32));

	AllocCtx ctx;
	ctx.byte_opts = torch::TensorOptions(torch::kByte).device(means3D.device());

	torch::Tensor k[11];
	const float* bg = req_ptr(background, k[0], "bg");
	const float* vm = req_ptr(viewmatrices, k[1], "viewmatrices");
	const float* pm = req_ptr(projmatrices, k[2], "projmatrices");
	const float* cp = opt_ptr(camposes, k[3], "camposes");
	TORCH_CHECK(cp == nullptr || (camposes.numel() == 3 * (int64_t)n), "camposes must have dimensions (views, 3)");

	brs_gaussians g{};
	g.P = P;
	g.means3D = req_ptr(means3D, k[4], "means3D");
	g.opacities = P ? req_ptr(opacity, k[5], "opacities") : nullptr;
	g.shs = opt_ptr(sh, k[6], "shs");
	g.colors_precomp = opt_ptr(colors, k[7], "colors_precomp");
	g.scales = opt_ptr(scales, k[8], "scales");
	g.rotations = opt_ptr(rotations, k[9], "rotations");
	g.cov3D_precomp = opt_ptr(cov3D_precomp, k[10], "cov3D_precomp");

	std::vector<brs_view> views((size_t)n);
	for (int v = 0; v < n; v++) {
		brs_view& view = views[(size_t)v];
		view = brs_view{};
		view.image_width = W;
		view.image_height = H;
		view.tanfovx = (float)tan_fovx[tan_fovx.size() == 1 ? 0 : (size_t)v];
		view.tanfovy = (float)tan_fovy[tan_fovy.size() == 1 ? 0 : (size_t)v];
		view.scale_modifier = scale_modifier;
		view.sh_degree = degree;
		view.sh_coeffs = (g.shs != nullptr) ? (int)sh.size(1) : 0;
		view.prefiltered = prefiltered;
		view.debug = debug;
		view.bg = bg;
		view.viewmatrix = vm + 16 * (size_t)v;
		view.projmatrix = pm + 16 * (size_t)v;
		view.campos = cp ? cp + 3 * (size_t)v : nullptr;
	}
	brs_fwd_options opt{};
	opt.mode = mode;
	long long R = 0;
	int st = brs_forward_views(views.data(), n, &g, out_color.data_ptr<float>(), out_depth.data_ptr<float>(),
	                           P ? radii.data_ptr<int>() : nullptr, alloc_cb, &ctx, &R, &opt, current_stream());
	check_status(st, "rasterize_gaussians_views");
	return std::make_tuple((int64_t)R, out_color, out_depth, radii);
}

namespace {

// Shared body of the two backward bindings: tensors -> C structs -> brs_backward with `grads`.
void run_backward(const torch::Tensor& background, const torch::Tensor& means3D, const torch::Tensor& radii,
                  const torch::Tensor& colors, const torch::Tensor& scales, const torch::Tensor& rotations,
                  const float scale_modifier, const torch::Tensor& cov3D_precomp, const torch::Tensor& viewmatrix,
                  const torch::Tensor& projmatrix, const float tan_fovx, const float tan_fovy,
                  const torch::Tensor& dL_dout_color, const torch::Tensor& dL_dout_depth, const torch::Tensor& sh,
                  const int degree, const torch::Tensor& campos, const torch::Tensor& geomBuffer, const int R,
                  const torch::Tensor& binningBuffer, const torch::Tensor& imageBuffer, const bool debug, const int M,
                  const brs_grads& grads_in, const brs_densify_stats* stats, const char* what,
                  const c10::optional<torch::Tensor>& out_depth = c10::nullopt)
{
	brs_grads grads = grads_in;
	torch::Tensor out_depth_c;
	if (out_depth.has_value() && out_depth->defined() && out_depth->numel() != 0) {
		// opt-in depth gradient (brs_grads.depth_gradient): needs the forward's depth image and dL_dout_depth
		TORCH_CHECK(out_depth->is_cuda() && out_depth->scalar_type() == torch::kFloat32, "out_depth must be CUDA float32");
		TORCH_CHECK(dL_dout_depth.defined() && dL_dout_depth.numel() == out_depth->numel(),
		            "depth gradient: dL_dout_depth must have the shape of out_depth");
		out_depth_c = out_depth->contiguous();
		grads.out_depth = out_depth_c.data_ptr<float>();
		grads.depth_gradient = 1;
	}
	const int P = means3D.size(0);
	const int H = dL_dout_color.size(1);
	const int W = dL_dout_color.size(2);
	AllocCtx ctx;
	ctx.byte_opts = torch::TensorOptions(torch::kByte).device(means3D.device());

	torch::Tensor k[13];
	brs_view view{};
	view.image_width = W;
	view.image_height = H;
	view.tanfovx = tan_fovx;
	view.tanfovy = tan_fovy;
	view.scale_modifier = scale_modifier;
	view.sh_degree = degree;
	view.sh_coeffs = M;
	view.prefiltered = 0;
	view.debug = debug;
	view.bg = req_ptr(background, k[0], "bg");
	view.viewmatrix = req_ptr(viewmatrix, k[1], "viewmatrix");
	view.projmatrix = req_ptr(projmatrix, k[2], "projmatrix");
	view.campos = opt_ptr(campos, k[3], "campos");

	brs_gaussians g{};
	g.P = P;
	g.means3D = req_ptr(means3D, k[4], "means3D");
	g.opacities = g.means3D; // not read by backward (opacity lives in the forward records); non-NULL for validation
	g.shs = opt_ptr(sh, k[6], "shs");
	g.colors_precomp = opt_ptr(colors, k[7], "colors_precomp");
	g.scales = opt_ptr(scales, k[8], "scales");
	g.rotations = opt_ptr(rotations, k[9], "rotations");
	g.cov3D_precomp = opt_ptr(cov3D_precomp, k[10], "cov3D_precomp");

	TORCH_CHECK(radii.is_cuda() && radii.scalar_type() == torch::kInt32, "radii must be a CUDA int32 tensor");
	torch::Tensor radii_c = radii.contiguous();
	const float* dcol = req_ptr(dL_dout_color, k[11], "dL_dout_color");
	const float* ddepth = opt_ptr(dL_dout_depth, k[12], "dL_dout_depth");

	torch::Tensor geom_c = geomBuffer.contiguous(), bin_c = binningBuffer.contiguous(), img_c = imageBuffer.contiguous();
	brs_fwd_state state{};
	state.geom = geom_c.data_ptr();
	state.geom_bytes = (size_t)geom_c.numel();
	state.binning = bin_c.numel() ? bin_c.data_ptr() : nullptr;
	state.binning_bytes = (size_t)bin_c.numel();
	state.image = img_c.data_ptr();
	state.image_bytes = (size_t)img_c.numel();
	state.num_rendered = R;

	int st = brs_backward_ex(&view, &g, radii_c.data_ptr<int>(), &state, dcol, ddepth, &grads, stats, alloc_cb, &ctx,
	                         current_stream());
	check_status(st, what);
}

int sh_coeffs_of(const torch::Tensor& sh)
{
	return (sh.numel() != 0 && sh.size(0) != 0) ? (int)sh.size(1) : 0;
}

// Gradient sink of the accumulate binding: absent (undefined / empty) -> NULL, else a contiguous CUDA
// float32 tensor of exactly `numel` elements that is updated in place.
float* sink_ptr(const c10::optional<torch::Tensor>& t, int64_t numel, const char* name)
{
	if (!t.has_value() || !t->defined() || t->numel() == 0)
		return nullptr;
	TORCH_CHECK(t->is_cuda() && t->scalar_type() == torch::kFloat32 && t->is_contiguous(), name,
	            " sink must be a contiguous CUDA float32 tensor");
	TORCH_CHECK(t->numel() == numel, name, " sink has the wrong number of elements");
	return t->data_ptr<float>();
}


// Densification statistics of the backward bindings (brs_densify_stats): absent (all three None) -> nullptr.
// grad_norm / count are caller-owned accumulators of any shape with the same number of elements (e.g. [rows, 1]),
// updated in place; index, if given, maps each of the P Gaussians to its accumulator row.
const brs_densify_stats* stats_of(const c10::optional<torch::Tensor>& grad_norm, const c10::optional<torch::Tensor>& count,
                                  const c10::optional<torch::Tensor>& index, const torch::Tensor& means3D,
                                  brs_densify_stats& out)
{
	auto given = [](const c10::optional<torch::Tensor>& t) { return t.has_value() && t->defined(); };
	if (!given(grad_norm) && !given(count) && !given(index))
		return nullptr;
	TORCH_CHECK(given(grad_norm) && given(count), "densification statistics need both stats_grad_norm and stats_count");
	for (const torch::Tensor* t : {&*grad_norm, &*count})
		TORCH_CHECK(t->is_cuda() && t->device() == means3D.device() && t->scalar_type() == torch::kFloat32 && t->is_contiguous(),
		            "stats_grad_norm / stats_count must be contiguous float32 tensors on the device of means3D");
	TORCH_CHECK(grad_norm->numel() == count->numel(), "stats_grad_norm and stats_count must have the same number of elements");
	TORCH_CHECK(grad_norm->numel() <= INT32_MAX, "densification statistics: more than 2^31 - 1 rows");
	out = brs_densify_stats{};
	out.grad_norm = grad_norm->data_ptr<float>();
	out.count = count->data_ptr<float>();
	out.rows = (int)grad_norm->numel();
	if (given(index)) {
		TORCH_CHECK(index->is_cuda() && index->device() == means3D.device() && index->scalar_type() == torch::kInt64 &&
		                index->is_contiguous(),
		            "stats_index must be a contiguous int64 tensor on the device of means3D");
		TORCH_CHECK(index->numel() == means3D.size(0), "stats_index must have one entry per Gaussian");
		out.index = reinterpret_cast<const long long*>(index->data_ptr<int64_t>());
	} else {
		TORCH_CHECK(out.rows >= means3D.size(0), "densification statistics without stats_index need at least P rows");
	}
	return &out;
}

} // namespace

std::tuple<torch::Tensor, torch::Tensor, torch::Tensor, torch::Tensor, torch::Tensor, torch::Tensor, torch::Tensor,
           torch::Tensor>
RasterizeGaussiansBackwardImpl(const c10::optional<torch::Tensor>& out_depth, const torch::Tensor& background,
                               const torch::Tensor& means3D,
                               const torch::Tensor& radii, const torch::Tensor& colors, const torch::Tensor& scales,
                               const torch::Tensor& rotations, const float scale_modifier,
                               const torch::Tensor& cov3D_precomp, const torch::Tensor& viewmatrix,
                               const torch::Tensor& projmatrix, const float tan_fovx, const float tan_fovy,
                               const torch::Tensor& dL_dout_color, const torch::Tensor& dL_dout_depth,
                               const torch::Tensor& sh, const int degree, const torch::Tensor& campos,
                               const torch::Tensor& geomBuffer, const int R, const torch::Tensor& binningBuffer,
                               const torch::Tensor& imageBuffer, const bool debug,
                               const c10::optional<torch::Tensor>& stats_grad_norm,
                               const c10::optional<torch::Tensor>& stats_count,
                               const c10::optional<torch::Tensor>& stats_index)
{
	TORCH_CHECK(means3D.is_cuda(), "means3D must be a CUDA tensor");
	c10::cuda::CUDAGuard guard(means3D.device());
	const int P = means3D.size(0);
	const int M = sh_coeffs_of(sh);
	brs_densify_stats stats_buf;
	const brs_densify_stats* stats = stats_of(stats_grad_norm, stats_count, stats_index, means3D, stats_buf);

	auto opts = means3D.options().dtype(torch::kFloat32);
	torch::Tensor dL_dmeans3D = torch::empty({P, 3}, opts);
	torch::Tensor dL_dmeans2D = torch::empty({P, 3}, opts);
	torch::Tensor dL_dcolors = torch::empty({P, 3}, opts);
	torch::Tensor dL_dopacity = torch::empty({P, 1}, opts);
	torch::Tensor dL_dcov3D = torch::empty({P, 6}, opts);
	torch::Tensor dL_dsh = torch::empty({P, M, 3}, opts);
	torch::Tensor dL_dscales = torch::empty({P, 3}, opts);
	torch::Tensor dL_drotations = torch::empty({P, 4}, opts);

	if (P != 0) {
		brs_grads grads{};
		grads.dL_dmeans2D = dL_dmeans2D.data_ptr<float>();
		grads.dL_dcolors = dL_dcolors.data_ptr<float>();
		grads.dL_dopacity = dL_dopacity.data_ptr<float>();
		grads.dL_dmeans3D = dL_dmeans3D.data_ptr<float>();
		grads.dL_dcov3D = dL_dcov3D.data_ptr<float>();
		grads.dL_dsh = M > 0 ? dL_dsh.data_ptr<float>() : nullptr;
		grads.dL_dscales = dL_dscales.data_ptr<float>();
		grads.dL_drotations = dL_drotations.data_ptr<float>();
		grads.accumulate = 0;
		run_backward(background, means3D, radii, colors, scales, rotations, scale_modifier, cov3D_precomp, viewmatrix,
		             projmatrix, tan_fovx, tan_fovy, dL_dout_color, dL_dout_depth, sh, degree, campos, geomBuffer, R,
		             binningBuffer, imageBuffer, debug, M, grads, stats, "rasterize_gaussians_backward", out_depth);
	}

	return std::make_tuple(dL_dmeans2D, dL_dcolors, dL_dopacity, dL_dmeans3D, dL_dcov3D, dL_dsh, dL_dscales,
	                       dL_drotations);
}

using GradTuple = std::tuple<torch::Tensor, torch::Tensor, torch::Tensor, torch::Tensor, torch::Tensor, torch::Tensor,
                             torch::Tensor, torch::Tensor>;

// reference binding (rasterize_points.h:42-66): 22 arguments, depth carries no gradient
GradTuple RasterizeGaussiansBackwardCUDA(
    const torch::Tensor& background, const torch::Tensor& means3D, const torch::Tensor& radii, const torch::Tensor& colors,
    const torch::Tensor& scales, const torch::Tensor& rotations, const float scale_modifier,
    const torch::Tensor& cov3D_precomp, const torch::Tensor& viewmatrix, const torch::Tensor& projmatrix,
    const float tan_fovx, const float tan_fovy, const torch::Tensor& dL_dout_color, const torch::Tensor& dL_dout_depth,
    const torch::Tensor& sh, const int degree, const torch::Tensor& campos, const torch::Tensor& geomBuffer, const int R,
    const torch::Tensor& binningBuffer, const torch::Tensor& imageBuffer, const bool debug,
    const c10::optional<torch::Tensor>& stats_grad_norm, const c10::optional<torch::Tensor>& stats_count,
    const c10::optional<torch::Tensor>& stats_index)
{
	return RasterizeGaussiansBackwardImpl(c10::nullopt, background, means3D, radii, colors, scales, rotations,
	                                      scale_modifier, cov3D_precomp, viewmatrix, projmatrix, tan_fovx, tan_fovy,
	                                      dL_dout_color, dL_dout_depth, sh, degree, campos, geomBuffer, R, binningBuffer,
	                                      imageBuffer, debug, stats_grad_norm, stats_count, stats_index);
}

// Extension (SURVEY.md 8f N3, opt-in): the same 22 arguments plus the forward's depth image; dL_dout_depth
// is then back-propagated (brs_grads.depth_gradient).
GradTuple RasterizeGaussiansBackwardDepthCUDA(
    const torch::Tensor& background, const torch::Tensor& means3D, const torch::Tensor& radii, const torch::Tensor& colors,
    const torch::Tensor& scales, const torch::Tensor& rotations, const float scale_modifier,
    const torch::Tensor& cov3D_precomp, const torch::Tensor& viewmatrix, const torch::Tensor& projmatrix,
    const float tan_fovx, const float tan_fovy, const torch::Tensor& dL_dout_color, const torch::Tensor& dL_dout_depth,
    const torch::Tensor& sh, const int degree, const torch::Tensor& campos, const torch::Tensor& geomBuffer, const int R,
    const torch::Tensor& binningBuffer, const torch::Tensor& imageBuffer, const bool debug, const torch::Tensor& out_depth,
    const c10::optional<torch::Tensor>& stats_grad_norm, const c10::optional<torch::Tensor>& stats_count,
    const c10::optional<torch::Tensor>& stats_index)
{
	return RasterizeGaussiansBackwardImpl(out_depth, background, means3D, radii, colors, scales, rotations, scale_modifier,
	                                      cov3D_precomp, viewmatrix, projmatrix, tan_fovx, tan_fovy, dL_dout_color,
	                                      dL_dout_depth, sh, degree, campos, geomBuffer, R, binningBuffer, imageBuffer,
	                                      debug, stats_grad_norm, stats_count, stats_index);
}

// Extension (no reference counterpart): the same backward, but the parameter gradients are ADDED in
// place to caller-owned sinks (brs_grads.accumulate) instead of being returned as fresh tensors; only
// the per-view dL_dmeans2D is returned.  Used by the view-sharded step, whose sinks are slices of
// the flat allreduce bucket.
torch::Tensor RasterizeGaussiansBackwardAccumulateCUDA(
    const torch::Tensor& background, const torch::Tensor& means3D, const torch::Tensor& radii, const torch::Tensor& colors,
    const torch::Tensor& scales, const torch::Tensor& rotations, const float scale_modifier,
    const torch::Tensor& cov3D_precomp, const torch::Tensor& viewmatrix, const torch::Tensor& projmatrix,
    const float tan_fovx, const float tan_fovy, const torch::Tensor& dL_dout_color, const torch::Tensor& dL_dout_depth,
    const torch::Tensor& sh, const int degree, const torch::Tensor& campos, const torch::Tensor& geomBuffer, const int R,
    const torch::Tensor& binningBuffer, const torch::Tensor& imageBuffer, const bool debug,
    const c10::optional<torch::Tensor>& sink_means3D, const c10::optional<torch::Tensor>& sink_colors,
    const c10::optional<torch::Tensor>& sink_opacity, const c10::optional<torch::Tensor>& sink_cov3D,
    const c10::optional<torch::Tensor>& sink_sh, const c10::optional<torch::Tensor>& sink_scales,
    const c10::optional<torch::Tensor>& sink_rotations, const c10::optional<torch::Tensor>& out_depth,
    const c10::optional<torch::Tensor>& stats_grad_norm, const c10::optional<torch::Tensor>& stats_count,
    const c10::optional<torch::Tensor>& stats_index)
{
	TORCH_CHECK(means3D.is_cuda(), "means3D must be a CUDA tensor");
	c10::cuda::CUDAGuard guard(means3D.device());
	const int64_t P = means3D.size(0);
	const int M = sh_coeffs_of(sh);
	brs_densify_stats stats_buf;
	const brs_densify_stats* stats = stats_of(stats_grad_norm, stats_count, stats_index, means3D, stats_buf);
	torch::Tensor dL_dmeans2D = torch::empty({P, 3}, means3D.options().dtype(torch::kFloat32));
	if (P != 0) {
		brs_grads grads{};
		grads.dL_dmeans2D = dL_dmeans2D.data_ptr<float>();
		grads.dL_dmeans3D = sink_ptr(sink_means3D, P * 3, "means3D");
		grads.dL_dopacity = sink_ptr(sink_opacity, P, "opacity");
		grads.dL_dcolors = sink_ptr(sink_colors, P * 3, "colors_precomp");
		grads.dL_dcov3D = sink_ptr(sink_cov3D, P * 6, "cov3D_precomp");
		grads.dL_dsh = sink_ptr(sink_sh, P * M * 3, "shs");
		grads.dL_dscales = sink_ptr(sink_scales, P * 3, "scales");
		grads.dL_drotations = sink_ptr(sink_rotations, P * 4, "rotations");
		grads.accumulate = 1;
		run_backward(background, means3D, radii, colors, scales, rotations, scale_modifier, cov3D_precomp, viewmatrix,
		             projmatrix, tan_fovx, tan_fovy, dL_dout_color, dL_dout_depth, sh, degree, campos, geomBuffer, R,
		             binningBuffer, imageBuffer, debug, M, grads, stats, "rasterize_gaussians_backward_accumulate", out_depth);
	}
	return dL_dmeans2D;
}

torch::Tensor markVisible(torch::Tensor& means3D, torch::Tensor& viewmatrix, torch::Tensor& projmatrix)
{
	TORCH_CHECK(means3D.is_cuda(), "means3D must be a CUDA tensor");
	c10::cuda::CUDAGuard guard(means3D.device());
	const int P = means3D.size(0);
	torch::Tensor present = torch::empty({P}, means3D.options().dtype(at::kBool));
	if (P != 0) {
		torch::Tensor k[3];
		int st = brs_mark_visible(P, req_ptr(means3D, k[0], "means3D"), req_ptr(viewmatrix, k[1], "viewmatrix"),
		                          req_ptr(projmatrix, k[2], "projmatrix"),
		                          reinterpret_cast<uint8_t*>(present.data_ptr<bool>()), current_stream());
		check_status(st, "mark_visible");
	}
	return present;
}

namespace {
// radii, and with `compact` also (indices int64 [P] capacity, count int32 [1]) of the Gaussians with radii > 0
std::tuple<torch::Tensor, torch::Tensor, torch::Tensor> filter_impl(const torch::Tensor& means3D, const torch::Tensor& scales,
                                                                    const torch::Tensor& rotations, const float scale_modifier,
                                                                    const torch::Tensor& cov3D_precomp,
                                                                    const torch::Tensor& viewmatrix, const torch::Tensor& projmatrix,
                                                                    const float tan_fovx, const float tan_fovy,
                                                                    const int image_height, const int image_width,
                                                                    const bool prefiltered, const bool debug, const bool compact)
{
	if (means3D.ndimension() != 2 || means3D.size(1) != 3) {
		AT_ERROR("means3D must have dimensions (num_points, 3)");
	}
	TORCH_CHECK(means3D.is_cuda(), "means3D must be a CUDA tensor");
	c10::cuda::CUDAGuard guard(means3D.device());
	const int P = means3D.size(0);
	torch::Tensor radii = torch::empty({P}, means3D.options().dtype(torch::kInt32));
	torch::Tensor indices, count;
	if (compact) {
		indices = torch::empty({P}, means3D.options().dtype(torch::kInt64));
		count = torch::zeros({1}, means3D.options().dtype(torch::kInt32));
	}
	if (P != 0) {
		torch::Tensor k[6];
		brs_view view{};
		view.image_width = image_width;
		view.image_height = image_height;
		view.tanfovx = tan_fovx;
		view.tanfovy = tan_fovy;
		view.scale_modifier = scale_modifier;
		view.prefiltered = prefiltered;
		view.debug = debug;
		view.viewmatrix = req_ptr(viewmatrix, k[0], "viewmatrix");
		view.projmatrix = req_ptr(projmatrix, k[1], "projmatrix");

		// BloomScene passes scales as a [:, :3] view of a [P,6] tensor (gaussian_renderer/__init__.py:344):
		// read it in place through its row stride instead of materialising a copy.
		const float* scales_ptr = nullptr;
		int scales_stride = 3;
		if (scales.defined() && scales.numel() != 0) {
			TORCH_CHECK(scales.is_cuda() && scales.scalar_type() == torch::kFloat32, "scales must be CUDA float32");
			if (scales.dim() == 2 && scales.stride(1) == 1 && scales.stride(0) >= 3) {
				scales_ptr = scales.data_ptr<float>();
				scales_stride = (int)scales.stride(0);
			} else {
				k[2] = scales.contiguous();
				scales_ptr = k[2].data_ptr<float>();
			}
		}
		int st;
		if (compact) {
			torch::Tensor scratch = torch::empty({(int64_t)brs_filter_scratch_bytes(P)}, means3D.options().dtype(torch::kByte));
			st = brs_visible_filter_compact(&view, P, req_ptr(means3D, k[3], "means3D"), scales_ptr, scales_stride,
			                                opt_ptr(rotations, k[4], "rotations"), opt_ptr(cov3D_precomp, k[5], "cov3D_precomp"),
			                                radii.data_ptr<int>(), reinterpret_cast<long long*>(indices.data_ptr<int64_t>()),
			                                reinterpret_cast<uint32_t*>(count.data_ptr<int>()), scratch.data_ptr(), current_stream());
		} else {
			st = brs_visible_filter(&view, P, req_ptr(means3D, k[3], "means3D"), scales_ptr, scales_stride,
			                        opt_ptr(rotations, k[4], "rotations"), opt_ptr(cov3D_precomp, k[5], "cov3D_precomp"),
			                        radii.data_ptr<int>(), current_stream());
		}
		check_status(st, "rasterize_aussians_filter");
	}
	return std::make_tuple(radii, indices, count);
}
} // namespace

torch::Tensor RasterizeGaussiansfilterCUDA(const torch::Tensor& means3D, const torch::Tensor& scales,
                                           const torch::Tensor& rotations, const float scale_modifier,
                                           const torch::Tensor& cov3D_precomp, const torch::Tensor& viewmatrix,
                                           const torch::Tensor& projmatrix, const float tan_fovx, const float tan_fovy,
                                           const int image_height, const int image_width, const bool prefiltered,
                                           const bool debug)
{
	return std::get<0>(filter_impl(means3D, scales, rotations, scale_modifier, cov3D_precomp, viewmatrix, projmatrix, tan_fovx,
	                               tan_fovy, image_height, image_width, prefiltered, debug, false));
}

// Extension (SURVEY.md 8f N2): (radii, indices int64 [P] of which the first count[0] are valid, count int32 [1])
std::tuple<torch::Tensor, torch::Tensor, torch::Tensor> RasterizeGaussiansfilterCompactCUDA(
    const torch::Tensor& means3D, const torch::Tensor& scales, const torch::Tensor& rotations, const float scale_modifier,
    const torch::Tensor& cov3D_precomp, const torch::Tensor& viewmatrix, const torch::Tensor& projmatrix, const float tan_fovx,
    const float tan_fovy, const int image_height, const int image_width, const bool prefiltered, const bool debug)
{
	return filter_impl(means3D, scales, rotations, scale_modifier, cov3D_precomp, viewmatrix, projmatrix, tan_fovx, tan_fovy,
	                   image_height, image_width, prefiltered, debug, true);
}

// ---- the steps either side of the rasterizer (SURVEY.md 8f N4) -----------------------------------------

namespace {
const float* f32_cuda(const torch::Tensor& t, torch::Tensor& keep, const char* name)
{
	TORCH_CHECK(t.defined() && t.is_cuda() && t.scalar_type() == torch::kFloat32, name, " must be a CUDA float32 tensor");
	keep = t.contiguous();
	return keep.data_ptr<float>();
}
} // namespace

// (dmaps [3,C,H,W], partial [blocks,2]) of loss = (1 - l) mean|x - y| + l (1 - mean SSIM(x, y))
std::tuple<torch::Tensor, torch::Tensor> L1SsimForward(const torch::Tensor& x, const torch::Tensor& y)
{
	TORCH_CHECK(x.dim() == 3 && x.sizes() == y.sizes(), "l1_ssim: image and target must both be [C,H,W]");
	c10::cuda::CUDAGuard guard(x.device());
	torch::Tensor k[2];
	const float* xp = f32_cuda(x, k[0], "image");
	const float* yp = f32_cuda(y, k[1], "target");
	const int C = x.size(0), H = x.size(1), W = x.size(2);
	torch::Tensor dmaps = torch::empty({3, C, H, W}, x.options());
	torch::Tensor partial = torch::empty({(int64_t)brs_l1_ssim_blocks(C, H, W), 2}, x.options());
	check_status(brs_l1_ssim_forward(xp, yp, C, H, W, dmaps.data_ptr<float>(), partial.data_ptr<float>(), current_stream()),
	             "l1_ssim_forward");
	return std::make_tuple(dmaps, partial);
}

torch::Tensor L1SsimBackward(const torch::Tensor& x, const torch::Tensor& y, const torch::Tensor& dmaps,
                             const torch::Tensor& dL_dloss, double lambda_dssim)
{
	c10::cuda::CUDAGuard guard(x.device());
	torch::Tensor k[4];
	const float* xp = f32_cuda(x, k[0], "image");
	const float* yp = f32_cuda(y, k[1], "target");
	const float* dp = f32_cuda(dmaps, k[2], "dmaps");
	const float* up = f32_cuda(dL_dloss, k[3], "dL_dloss");
	TORCH_CHECK(dL_dloss.numel() == 1, "dL_dloss must be a scalar");
	const int C = x.size(0), H = x.size(1), W = x.size(2);
	torch::Tensor dx = torch::empty({C, H, W}, x.options());
	check_status(brs_l1_ssim_backward(xp, yp, dp, C, H, W, up, (float)lambda_dssim, dx.data_ptr<float>(), current_stream()),
	             "l1_ssim_backward");
	return dx;
}

// (xyz, color, opacity, scaling, rot, index, count) with capacity N*K rows; count is a device int32 scalar
std::vector<torch::Tensor> NeuralGaussiansForward(const torch::Tensor& anchor, const torch::Tensor& grid_scaling,
                                                  const torch::Tensor& offsets, const torch::Tensor& neural_opacity,
                                                  const torch::Tensor& color, const torch::Tensor& scale_rot)
{
	c10::cuda::CUDAGuard guard(anchor.device());
	const int64_t N = anchor.size(0);
	TORCH_CHECK(anchor.dim() == 2 && anchor.size(1) == 3 && grid_scaling.dim() == 2 && grid_scaling.size(0) == N && grid_scaling.size(1) == 6,
	            "neural_gaussians: anchor [N,3], grid_scaling [N,6]");
	const int64_t NK = neural_opacity.numel();
	TORCH_CHECK(N == 0 ? NK == 0 : NK % N == 0, "neural_gaussians: neural_opacity must hold N*K values");
	const int64_t K = N ? NK / N : 0;
	TORCH_CHECK(offsets.numel() == NK * 3 && color.numel() == NK * 3 && scale_rot.numel() == NK * 7,
	            "neural_gaussians: offsets [N*K,3], color [N*K,3], scale_rot [N*K,7]");
	torch::Tensor k[6];
	brs_neural_inputs in{};
	in.N = (int)N;
	in.K = (int)K;
	in.anchor = f32_cuda(anchor, k[0], "anchor");
	in.grid_scaling = f32_cuda(grid_scaling, k[1], "grid_scaling");
	in.offsets = f32_cuda(offsets, k[2], "offsets");
	in.neural_opacity = f32_cuda(neural_opacity, k[3], "neural_opacity");
	in.color = f32_cuda(color, k[4], "color");
	in.scale_rot = f32_cuda(scale_rot, k[5], "scale_rot");
	auto fo = anchor.options().dtype(torch::kFloat32);
	auto io = anchor.options().dtype(torch::kInt32);
	torch::Tensor xyz = torch::empty({NK, 3}, fo), col = torch::empty({NK, 3}, fo), op = torch::empty({NK, 1}, fo),
	              sc = torch::empty({NK, 3}, fo), rot = torch::empty({NK, 4}, fo), index = torch::empty({NK}, io),
	              count = torch::empty({1}, io);
	torch::Tensor scratch = torch::empty({(int64_t)brs_neural_scratch_bytes((int)N)}, anchor.options().dtype(torch::kByte));
	brs_neural_outputs out{};
	out.xyz = xyz.data_ptr<float>();
	out.color = col.data_ptr<float>();
	out.opacity = op.data_ptr<float>();
	out.scaling = sc.data_ptr<float>();
	out.rot = rot.data_ptr<float>();
	out.index = index.data_ptr<int>();
	out.count = reinterpret_cast<uint32_t*>(count.data_ptr<int>());
	check_status(brs_neural_gaussians_forward(&in, &out, scratch.data_ptr(), current_stream()), "neural_gaussians_forward");
	return {xyz, col, op, sc, rot, index, count};
}

std::vector<torch::Tensor> NeuralGaussiansBackward(const torch::Tensor& grid_scaling, const torch::Tensor& offsets,
                                                   const torch::Tensor& scale_rot, const torch::Tensor& index,
                                                   const torch::Tensor& d_xyz, const torch::Tensor& d_color,
                                                   const torch::Tensor& d_opacity, const torch::Tensor& d_scaling,
                                                   const torch::Tensor& d_rot)
{
	c10::cuda::CUDAGuard guard(grid_scaling.device());
	const int64_t N = grid_scaling.size(0), NK = index.numel();
	const int64_t K = N ? NK / N : 0;
	torch::Tensor k[8];
	brs_neural_inputs in{};
	in.N = (int)N;
	in.K = (int)K;
	in.grid_scaling = f32_cuda(grid_scaling, k[0], "grid_scaling");
	in.offsets = f32_cuda(offsets, k[1], "offsets");
	in.scale_rot = f32_cuda(scale_rot, k[2], "scale_rot");
	TORCH_CHECK(index.is_cuda() && index.scalar_type() == torch::kInt32 && index.is_contiguous(), "index: contiguous CUDA int32");
	const int64_t M = d_xyz.size(0);
	TORCH_CHECK(d_xyz.numel() == M * 3 && d_color.numel() == M * 3 && d_opacity.numel() == M && d_scaling.numel() == M * 3 &&
	                d_rot.numel() == M * 4,
	            "neural_gaussians_backward: upstream gradients must all have M rows");
	auto fo = grid_scaling.options().dtype(torch::kFloat32);
	torch::Tensor d_anchor = torch::empty({N, 3}, fo), d_gs = torch::empty({N, 6}, fo), d_off = torch::empty({NK, 3}, fo),
	              d_nop = torch::empty({NK, 1}, fo), d_col = torch::empty({NK, 3}, fo), d_sr = torch::empty({NK, 7}, fo);
	brs_neural_grads g{};
	if (M > 0) {
		g.d_xyz = f32_cuda(d_xyz, k[3], "d_xyz");
		g.d_color = f32_cuda(d_color, k[4], "d_color");
		g.d_opacity = f32_cuda(d_opacity, k[5], "d_opacity");
		g.d_scaling = f32_cuda(d_scaling, k[6], "d_scaling");
		g.d_rot = f32_cuda(d_rot, k[7], "d_rot");
	}
	g.d_anchor = d_anchor.data_ptr<float>();
	g.d_grid_scaling = d_gs.data_ptr<float>();
	g.d_offsets = d_off.data_ptr<float>();
	g.d_neural_opacity = d_nop.data_ptr<float>();
	g.d_color_in = d_col.data_ptr<float>();
	g.d_scale_rot = d_sr.data_ptr<float>();
	check_status(brs_neural_gaussians_backward(&in, index.data_ptr<int>(), &g, current_stream()), "neural_gaussians_backward");
	return {d_anchor, d_gs, d_off, d_nop, d_col, d_sr};
}

// ---- extras used by tests / bench (not part of the reference surface) ----------------------------

std::tuple<torch::Tensor, torch::Tensor> SortPairs(const torch::Tensor& keys, const c10::optional<torch::Tensor>& vals,
                                                   int begin_bit, int end_bit)
{
	TORCH_CHECK(keys.is_cuda() && keys.scalar_type() == torch::kInt32 && keys.dim() == 1, "keys: 1-D CUDA int32");
	c10::cuda::CUDAGuard guard(keys.device());
	const int n = keys.numel();
	torch::Tensor kin = keys.contiguous();
	torch::Tensor vin;
	const uint32_t* vptr = nullptr;
	if (vals.has_value() && vals->defined()) {
		TORCH_CHECK(vals->is_cuda() && vals->scalar_type() == torch::kInt32 && vals->numel() == n, "vals: CUDA int32 [n]");
		vin = vals->contiguous();
		vptr = reinterpret_cast<const uint32_t*>(vin.data_ptr<int>());
	}
	torch::Tensor kout = torch::empty_like(kin), vout = torch::empty_like(kin);
	torch::Tensor scratch =
	    torch::empty({(int64_t)brs_sort_scratch_bytes(n)}, torch::TensorOptions(torch::kByte).device(keys.device()));
	int st = brs_sort_pairs_u32(reinterpret_cast<const uint32_t*>(kin.data_ptr<int>()), vptr,
	                            reinterpret_cast<uint32_t*>(kout.data_ptr<int>()),
	                            reinterpret_cast<uint32_t*>(vout.data_ptr<int>()), n, begin_bit, end_bit,
	                            scratch.data_ptr(), current_stream());
	check_status(st, "sort_pairs");
	return std::make_tuple(kout, vout);
}

pybind11::dict StateLayout(int P, int R, int W, int H)
{
	brs_layout l{};
	check_status(brs_state_layout(P, R, W, H, &l), "state_layout");
	pybind11::dict d;
	d["geom_records"] = l.geom_records;
	d["geom_depth_key"] = l.geom_depth_key;
	d["geom_rect"] = l.geom_rect;
	d["geom_order"] = l.geom_order;
	d["binning_point_list"] = l.binning_point_list;
	d["image_ranges"] = l.image_ranges;
	d["image_final_T"] = l.image_final_T;
	d["image_n_contrib"] = l.image_n_contrib;
	return d;
}

// (E, C, E_b) pair counts of a finished forward, reference semantics (measurement only).
std::tuple<int64_t, int64_t, int64_t> CountPairs(const torch::Tensor& geom, const torch::Tensor& binning,
                                                 const torch::Tensor& image, int P, int R, int W, int H)
{
	c10::cuda::CUDAGuard guard(geom.device());
	brs_view view{};
	view.image_width = W;
	view.image_height = H;
	brs_fwd_state state{};
	state.geom = geom.data_ptr();
	state.geom_bytes = (size_t)geom.numel();
	state.binning = binning.numel() ? binning.data_ptr() : nullptr;
	state.binning_bytes = (size_t)binning.numel();
	state.image = image.data_ptr();
	state.image_bytes = (size_t)image.numel();
	state.num_rendered = R;
	torch::Tensor out = torch::zeros({3}, torch::TensorOptions(torch::kInt64).device(geom.device()));
	check_status(brs_count_pairs(&view, &state, P, reinterpret_cast<unsigned long long*>(out.data_ptr<int64_t>()),
	                             current_stream()),
	             "count_pairs");
	torch::Tensor h = out.cpu();
	return std::make_tuple(h[0].item<int64_t>(), h[1].item<int64_t>(), h[2].item<int64_t>());
}

pybind11::dict StageTimes()
{
	float ms[BRS_NUM_STAGES] = {0};
	int calls[BRS_NUM_STAGES] = {0};
	check_status(brs_stage_times(ms, calls), "stage_times");
	static const char* names[BRS_NUM_STAGES] = {"preprocess", "depth_sort", "coarse_emit", "coarse_sort", "fine_bin",
	                                            "blend_fwd", "blend_bwd", "preprocess_bwd"};
	pybind11::dict d;
	for (int i = 0; i < BRS_NUM_STAGES; i++)
		d[names[i]] = pybind11::make_tuple(ms[i], calls[i]);
	return d;
}

PYBIND11_MODULE(TORCH_EXTENSION_NAME, m)
{
	m.def("l1_ssim_forward", &L1SsimForward);
	m.def("l1_ssim_backward", &L1SsimBackward);
	m.def("neural_gaussians_forward", &NeuralGaussiansForward);
	m.def("neural_gaussians_backward", &NeuralGaussiansBackward);
	m.def("count_pairs", &CountPairs);
	m.def("stage_timing", [](bool enable) { brs_stage_timing(enable ? 1 : 0); });
	m.def("stage_times", &StageTimes);
	m.def("stage_nvtx", [](int enable) { return brs_stage_nvtx(enable); }, pybind11::arg("enable") = -1);
	m.def("probe_fp32_tflops", []() { return brs_probe_fp32_tflops(current_stream()); });
	// the forward blocks once on the device (instance count); it touches no Python object, so it runs
	// without the GIL and several host threads can drive one CUDA stream each (render_views)
	m.def("rasterize_gaussians", &RasterizeGaussiansCUDA, pybind11::call_guard<pybind11::gil_scoped_release>());
	m.def("rasterize_gaussians_views", &RasterizeGaussiansViewsCUDA, pybind11::arg("bg"), pybind11::arg("means3D"),
	      pybind11::arg("colors"), pybind11::arg("opacity"), pybind11::arg("scales"), pybind11::arg("rotations"),
	      pybind11::arg("scale_modifier"), pybind11::arg("cov3D_precomp"), pybind11::arg("viewmatrices"),
	      pybind11::arg("projmatrices"), pybind11::arg("tan_fovx"), pybind11::arg("tan_fovy"), pybind11::arg("image_height"),
	      pybind11::arg("image_width"), pybind11::arg("sh"), pybind11::arg("degree"), pybind11::arg("camposes"),
	      pybind11::arg("prefiltered"), pybind11::arg("debug"), pybind11::arg("mode") = (int)BRS_FWD_AUTO,
	      pybind11::arg("color_out") = c10::nullopt, pybind11::arg("depth_out") = c10::nullopt);
	m.def("rasterize_gaussians_ex", &RasterizeGaussiansExCUDA, pybind11::arg("bg"), pybind11::arg("means3D"), pybind11::arg("colors"),
	      pybind11::arg("opacity"), pybind11::arg("scales"), pybind11::arg("rotations"), pybind11::arg("scale_modifier"),
	      pybind11::arg("cov3D_precomp"), pybind11::arg("viewmatrix"), pybind11::arg("projmatrix"), pybind11::arg("tan_fovx"),
	      pybind11::arg("tan_fovy"), pybind11::arg("image_height"), pybind11::arg("image_width"), pybind11::arg("sh"),
	      pybind11::arg("degree"), pybind11::arg("campos"), pybind11::arg("prefiltered"), pybind11::arg("debug"),
	      pybind11::arg("mode"), pybind11::arg("R_cap") = 0, pybind11::arg("R1_cap") = 0, pybind11::arg("depth_bits") = 0,
	      pybind11::arg("report") = pybind11::none(), pybind11::arg("overflow_accum") = pybind11::none(),
	      pybind11::call_guard<pybind11::gil_scoped_release>());
	m.def("note_counts", [](int P, int W, int H, const torch::Tensor& report) {
		TORCH_CHECK(report.is_cpu() && report.scalar_type() == torch::kInt32 && report.numel() >= 8 && report.is_contiguous());
		brs_note_counts(P, W, H, reinterpret_cast<const uint32_t*>(report.data_ptr<int>()));
	});
	m.def("reset_marks", []() { brs_reset_marks(); });
	m.def("has_marks", [](int P, int W, int H) { return brs_get_marks(P, W, H, nullptr) != 0; });
	m.def("forward_stats", [](bool reset) {
		long long v[4];
		brs_forward_stats(v, reset ? 1 : 0);
		pybind11::dict d;
		d["exact"] = v[0];
		d["optimistic"] = v[1];
		d["overflow_reruns"] = v[2];
		d["deferred"] = v[3];
		return d;
	}, pybind11::arg("reset") = false);
	m.attr("FWD_AUTO") = (int)BRS_FWD_AUTO;
	m.attr("FWD_EXACT") = (int)BRS_FWD_EXACT;
	m.attr("FWD_DEFERRED") = (int)BRS_FWD_DEFERRED;
	// the reference's 22 backward arguments (positional, as it calls them), then each binding's own extras; the
	// densification statistics (brs_densify_stats) are trailing keywords that default to None
	using pybind11::arg;
#define BRS_BWD_ARGS                                                                                                       \
	arg("bg"), arg("means3D"), arg("radii"), arg("colors"), arg("scales"), arg("rotations"), arg("scale_modifier"),        \
	    arg("cov3D_precomp"), arg("viewmatrix"), arg("projmatrix"), arg("tan_fovx"), arg("tan_fovy"), arg("dL_dout_color"), \
	    arg("dL_dout_depth"), arg("sh"), arg("degree"), arg("campos"), arg("geomBuffer"), arg("R"), arg("binningBuffer"),  \
	    arg("imageBuffer"), arg("debug")
#define BRS_STATS_ARGS \
	arg("stats_grad_norm") = pybind11::none(), arg("stats_count") = pybind11::none(), arg("stats_index") = pybind11::none()
	m.def("rasterize_gaussians_backward", &RasterizeGaussiansBackwardCUDA, BRS_BWD_ARGS, BRS_STATS_ARGS,
	      pybind11::call_guard<pybind11::gil_scoped_release>());
	m.def("rasterize_gaussians_backward_accumulate", &RasterizeGaussiansBackwardAccumulateCUDA, BRS_BWD_ARGS,
	      arg("sink_means3D"), arg("sink_colors"), arg("sink_opacity"), arg("sink_cov3D"), arg("sink_sh"), arg("sink_scales"),
	      arg("sink_rotations"), arg("out_depth"), BRS_STATS_ARGS, pybind11::call_guard<pybind11::gil_scoped_release>());
	m.def("rasterize_gaussians_backward_depth", &RasterizeGaussiansBackwardDepthCUDA, BRS_BWD_ARGS, arg("out_depth"),
	      BRS_STATS_ARGS, pybind11::call_guard<pybind11::gil_scoped_release>());
#undef BRS_STATS_ARGS
#undef BRS_BWD_ARGS
	m.attr("HAS_DENSIFY_STATS") = true;
	m.def("rasterize_aussians_filter", &RasterizeGaussiansfilterCUDA);
	m.def("rasterize_gaussians_filter_compact", &RasterizeGaussiansfilterCompactCUDA);
	m.def("mark_visible", &markVisible);
	m.def("sort_pairs", &SortPairs, pybind11::arg("keys"), pybind11::arg("vals") = pybind11::none(),
	      pybind11::arg("begin_bit") = 0, pybind11::arg("end_bit") = 32);
	m.def("state_layout", &StateLayout);
	m.def("launch_count", [](bool reset) { return brs_launch_count(reset ? 1 : 0); }, pybind11::arg("reset") = false);
	m.def("version", []() { return brs_version(); });
	m.def("blend_companion_stream", [](int enable) { return brs_blend_companion_stream(enable); }, pybind11::arg("enable") = -1);
}

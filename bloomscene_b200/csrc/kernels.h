// Internal launcher interface between api.cu and the kernel translation units.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

namespace brs {

void count_launch();

// ---- preprocess.cu ------------------------------------------------------------------------------
struct PreprocessArgs {
	int P, D, M;
	const float* means3D;
	const float* scales;
	float scale_modifier;
	const float* rotations;
	const float* opacities;
	const float* shs;
	const float* cov3D_precomp;
	const float* colors_precomp;
	const float* viewmatrix;
	const float* projmatrix;
	const float* campos;
	int W, H;
	float tan_fovx, tan_fovy, focal_x, focal_y;
	uint32_t grid_x, grid_y;
	int prefiltered;
	int eager_sh;         // request every Gaussian's SH row up front (most are visible) instead of the visible ones' later
	uint32_t row_offset;  // tile rows added to the rectangle: this view's place in a stack of views (brs_forward_views), else 0
	// outputs
	int* radii;
	float4* records;      // [3P]
	uint32_t* depth_key;  // [P]
	uint2* rect;          // [P]
	uint32_t* total_tiles; // [5], pre-zeroed: R = tile instances, R1 = supertile instances, max(~depth bits),
	                       // max(depth bits) over visible, V = number of visible Gaussians
};
cudaError_t launch_preprocess(const PreprocessArgs& a, cudaStream_t stream);
// Up to MAX_VIEWS views of a stack in one launch: the per-view fields of PreprocessArgs come from the table,
// view k of the launch is view first_view + k of the stack (row offset, output slices).
struct PreprocessViewTable {
	static constexpr int MAX_VIEWS = 16;
	struct Slot {
		const float* viewmatrix;
		const float* projmatrix;
		const float* campos;
		float tan_fovx, tan_fovy, focal_x, focal_y, scale_modifier;
		int prefiltered;
	} v[MAX_VIEWS];
	uint32_t first_view;
};
cudaError_t launch_preprocess_stack(const PreprocessArgs& a, const PreprocessViewTable& t, int n_views, cudaStream_t stream);

struct FilterArgs {
	int P;
	const float* means3D;
	const float* scales;
	int scales_stride;
	float scale_modifier;
	const float* rotations;
	const float* cov3D_precomp;
	const float* viewmatrix;
	const float* projmatrix;
	int W, H;
	float tan_fovx, tan_fovy, focal_x, focal_y;
	uint32_t grid_x, grid_y;
	int prefiltered;
	int* radii;
	// compaction (optional: all four or none): ascending indices of the Gaussians with radii > 0 and their count
	long long* indices; // [P]
	uint32_t* count;    // device scalar
	uint32_t* ticket;   // pre-zeroed
	uint32_t* status;   // [ceil(P / 256)], pre-zeroed
};
cudaError_t launch_filter(const FilterArgs& a, cudaStream_t stream);
cudaError_t launch_check_frustum(int P, const float* means3D, const float* viewmatrix, uint8_t* present,
                                 cudaStream_t stream);

// ---- binning.cu ---------------------------------------------------------------------------------
// Words of the geometry header (device memory, zeroed before preprocess).  preprocess accumulates
// 0..4; the depth sort's histogram kernel writes 5..6.
enum HeaderWord : int {
	HDR_R = 0,          // tile instances (reference num_rendered)
	HDR_R1 = 1,         // supertile instances
	HDR_KEY_INVMIN = 2, // max over visible Gaussians of ~depth bits (= ~min)
	HDR_KEY_MAX = 3,    // max depth bits over visible Gaussians
	HDR_V = 4,          // visible Gaussians
	HDR_OVERFLOW = 5,   // bit 0: R > R_cap, bit 1: R1 > R1_cap, bit 2: depth keys need more bits than planned, bit 3: V > V_cap
	HDR_KEY_BITS = 6,   // significant bits of (max key - bias)
	HDR_WORDS = 8
};
enum DepthCtl : int { DCTL_TICKET = 0 /* one per pass */, DCTL_WORDS = 16 };
enum InstCtl : int { ICTL_EMIT_TICKET = 0, ICTL_EMIT_DONE = 1, ICTL_N_INSTANCES = 2, ICTL_FINE_DONE = 3, ICTL_COARSE_TICKET = 4 /* one per pass */, ICTL_WORDS = 16 };

// Scratch of the depth sort: a zeroed part (tickets, digit histograms, look-back status words) and
// a plain part (ping-pong pairs).
struct DepthScratch {
	uint32_t* ctl;    // [DCTL_WORDS]
	uint32_t* hist;   // [4][256]
	uint32_t* status; // [tiles][256] of the first pass, then [passes - 1][tiles_rest][256]
	uint32_t* keys[2];
	uint32_t* vals[2];
	uint32_t tiles;      // tiles of the first pass (over P keys)
	uint32_t tiles_rest; // tiles of the later passes (over at most V_cap keys)
};
size_t depth_zero_bytes(size_t P, size_t V_cap, int passes);
size_t depth_plain_bytes(size_t P);
DepthScratch carve_depth_scratch(void* zeroed, void* plain, size_t P, size_t V_cap, int passes);

// Scratch of the instance levels (emission, coarse sort, fine binning), sized by the CAPACITY R1_cap.
struct InstScratch {
	uint32_t* ctl;           // [ICTL_WORDS]
	uint32_t* cell_count;    // [ns]
	uint32_t* emit_status;   // [emit blocks]
	uint32_t* coarse_status; // [coarse passes][tiles][256]
	uint32_t* cell_keys;     // [R1_cap]
	uint32_t* cell_ids;      // [R1_cap]
	uint32_t* tmp_keys;      // [R1_cap] (two coarse passes only)
	uint32_t* tmp_ids;
	uint32_t* coarse_list;   // [R1_cap] ids in (supertile, depth, id) order
	uint2* coarse_ranges;    // [ns]
	uint32_t* slice_base;    // [ns + 1]
	uint32_t* tile_count;    // [tiles]
	uint32_t* tile_start;    // [tiles]
	uint32_t* table;         // [max slices][64]
	uint32_t coarse_tiles;
	int coarse_passes;
};
size_t inst_zero_bytes(size_t P, size_t R1_cap, uint32_t grid_x, uint32_t grid_y);
size_t inst_plain_bytes(size_t P, size_t R1_cap, uint32_t grid_x, uint32_t grid_y);
InstScratch carve_inst_scratch(void* zeroed, void* plain, size_t P, size_t R1_cap, uint32_t grid_x, uint32_t grid_y);

// One forward's binning: capacities from the host, counts from the header on the device.
struct BinPlan {
	uint32_t P, R1_cap, R_cap;
	uint32_t V_cap;            // capacity of the visible Gaussians: sizes the depth sort's passes after the first
	uint32_t grid_x, grid_y, ns_x, ns;
	int depth_passes;          // 8-bit digits of (depth key - bias) that are sorted on
	uint32_t* hdr;             // geometry header
	uint32_t* overflow_accum;  // optional device word that collects the overflow bits of many forwards (atomicOr)
	const uint32_t* depth_key; // [P]
	const uint2* rect;         // [P]
	uint32_t* order;           // [P]: the V visible ids in (depth bits, id) order
	uint32_t* point_list;      // [R_cap]
	uint2* ranges;             // [tiles]
	DepthScratch d;
	InstScratch i;
};
// Histogram of all digits + first pass (needs no host knowledge), then the remaining passes.
cudaError_t launch_depth_sort_begin(const BinPlan& pl, int planned_passes, cudaStream_t stream);
cudaError_t launch_depth_sort_rest(const BinPlan& pl, cudaStream_t stream);
cudaError_t launch_emit(const BinPlan& pl, cudaStream_t stream);
cudaError_t launch_coarse_sort(const BinPlan& pl, cudaStream_t stream);
cudaError_t launch_fine_binning(const BinPlan& pl, cudaStream_t stream);

// Stand-alone stable LSD radix sort of (u32,u32) pairs on key bits [begin_bit, end_bit) with the same
// kernels (one histogram kernel + one onesweep kernel per 8-bit digit).  vals_in == nullptr -> iota.
// The result is written to keys_out/vals_out; the inputs are not modified.
size_t sort_scratch_bytes(size_t n);
cudaError_t sort_pairs(const uint32_t* keys_in, const uint32_t* vals_in, uint32_t* keys_out, uint32_t* vals_out,
                       size_t n, int begin_bit, int end_bit, void* scratch, cudaStream_t stream);

// ---- blend_fwd.cu -------------------------------------------------------------------------------
struct BlendFwdArgs {
	float exp_c_scale, exp_c_252; // constants of expf_exact (common.cuh), filled by the launcher
	const uint2* ranges;
	const uint32_t* point_list;
	const float4* records;
	const float* bg;
	int W, H;
	uint32_t grid_x, grid_y;
	int views;     // > 1: `ranges` holds views * grid_y tile rows (a stack of views, brs_forward_views); outputs are [views][...]
	float* final_T;      // nullptr: not kept (forward-only)
	uint32_t* n_contrib; // nullptr: not kept
	float* out_color;
	float* out_depth;
};
cudaError_t launch_blend_forward(const BlendFwdArgs& a, cudaStream_t stream);

// ---- blend_bwd.cu -------------------------------------------------------------------------------
struct BlendBwdArgs {
	float exp_c_scale, exp_c_252; // constants of expf_exact (common.cuh), filled by the launcher
	const uint2* ranges;
	const uint32_t* point_list;
	const float4* records;
	const float* bg;
	int W, H;
	uint32_t grid_x, grid_y;
	const float* final_T;
	const uint32_t* n_contrib;
	const float* dL_dpixels; // [3,H,W]
	const float* dL_ddepth;  // [H,W]; with out_depth: opt-in depth gradient (brs_grads.depth_gradient), else nullptr
	const float* out_depth;  // [H,W] the forward's depth output
	float* accum;            // [P][12] fp32, pre-zeroed: {dmean2D.x, .y, dconic.x, .y, .w, dopacity, dcol r,g,b, dz, pad x2}
};
cudaError_t launch_blend_backward(const BlendBwdArgs& a, cudaStream_t stream);

// ---- preprocess_bwd.cu --------------------------------------------------------------------------
struct PreprocessBwdArgs {
	int P, D, M;
	const float* means3D;
	const int* radii;
	const float* shs;
	const float* scales;
	const float* rotations;
	float scale_modifier;
	const float* cov3D_precomp;
	const float* viewmatrix;
	const float* projmatrix;
	const float* campos;
	int W, H;
	float tan_fovx, tan_fovy, focal_x, focal_y;
	const float* accum; // [P][12] from the blend backward
	int accumulate;     // 0: every output element is written; 1: see brs_grads.accumulate
	int depth_gradient; // 1: accum slot 9 holds dL_dz (view-space depth) and feeds dL_dmeans3D
	int eager_sh;       // request every Gaussian's SH row up front (most were rendered) instead of the rendered ones' later
	int fact_offset;    // (set by the launcher) float offset of the basis-factor rows in dynamic shared memory
	// outputs
	float* dL_dmeans2D;   // [P,3]
	float* dL_dcolors;    // [P,3]
	float* dL_dopacity;   // [P]
	float* dL_dmeans3D;   // [P,3]
	float* dL_dcov3D;     // [P,6]
	float* dL_dsh;        // [P,M,3] or nullptr
	float* dL_dscales;    // [P,3]
	float* dL_drotations; // [P,4]
	// optional densification statistics (brs_densify_stats); stats_grad_norm == nullptr: off
	float* stats_grad_norm;       // [stats_rows] += |dL_dmeans2D[i, 0:2]| for radii[i] > 0
	float* stats_count;           // [stats_rows] += 1 for the same Gaussians
	const long long* stats_index; // [P] slot of Gaussian i (outside [0, stats_rows): skipped), or nullptr = identity
	int stats_rows;
};
cudaError_t launch_preprocess_backward(const PreprocessBwdArgs& a, cudaStream_t stream);

// ---- loss.cu: fused L1 + SSIM loss (SURVEY.md 8f N4) ------------------------------------------------
size_t l1_ssim_blocks(int C, int H, int W); // number of (SSIM sum, L1 sum) pairs the forward writes
cudaError_t launch_l1_ssim_forward(const float* x, const float* y, int C, int H, int W, float* dmaps /* [3][C][H][W] */,
                                   float* partial /* [blocks][2] */, cudaStream_t stream);
cudaError_t launch_l1_ssim_backward(const float* x, const float* y, const float* dmaps, int C, int H, int W,
                                    const float* dL_dloss /* device scalar */, float lambda_dssim, float* dL_dx,
                                    cudaStream_t stream);

// ---- neural.cu: fused epilogue of the neural-Gaussian generation (SURVEY.md 8f N4) ---------------------
struct NeuralFwdArgs {
	int N, K;                    // anchors, offsets per anchor (K <= 32)
	const float* anchor;         // [N,3]
	const float* grid_scaling;   // [N,6]
	const float* offsets;        // [N*K,3]
	const float* neural_opacity; // [N*K]
	const float* color;          // [N*K,3]
	const float* scale_rot;      // [N*K,7]
	// outputs, capacity N*K rows; rows [0, *count) are valid
	float* xyz;         // [.,3]
	float* out_color;   // [.,3]
	float* out_opacity; // [.]
	float* scaling;     // [.,3]
	float* rot;         // [.,4]
	int* index;         // [N*K]: output row of every input row, -1 where neural_opacity <= 0
	uint32_t* count;    // device scalar: number of surviving rows
	uint32_t* ticket;   // (set by the launcher)
	uint32_t* status;   // (set by the launcher)
};
struct NeuralBwdArgs {
	int N, K;
	const float* grid_scaling;
	const float* offsets;
	const float* scale_rot;
	const int* index;
	const float* d_xyz;     // [M,3]
	const float* d_color;   // [M,3]
	const float* d_opacity; // [M]
	const float* d_scaling; // [M,3]
	const float* d_rot;     // [M,4]
	float* d_anchor;         // [N,3]
	float* d_grid_scaling;   // [N,6]
	float* d_offsets;        // [N*K,3]
	float* d_neural_opacity; // [N*K]
	float* d_color_in;       // [N*K,3]
	float* d_scale_rot;      // [N*K,7]
};
size_t neural_scratch_bytes(int N);
cudaError_t launch_neural_forward(const NeuralFwdArgs& a, void* scratch, cudaStream_t stream);
cudaError_t launch_neural_backward(const NeuralBwdArgs& a, cudaStream_t stream);

// ---- measure.cu (bench / profiling only) ----------------------------------------------------------
cudaError_t launch_count_pairs(const BlendFwdArgs& a, unsigned long long* out, cudaStream_t stream);
double probe_fp32_tflops(cudaStream_t stream);

constexpr int ACCUM_STRIDE = 12; // floats per Gaussian in the blend-backward accumulator

} // namespace brs

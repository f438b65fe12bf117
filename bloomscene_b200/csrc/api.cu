// C-ABI of libbloomrast (see include/bloomrast.h): stage orchestration, private state layout,
// error handling.  Replaces the reference driver CudaRasterizer::Rasterizer::{forward, backward,
// visible_filter, markVisible} (cuda_rasterizer/rasterizer_impl.cu:141-504) and its chunk
// sub-allocator (rasterizer_impl.h:21-73, rasterizer_impl.cu:155-194).
//
// Stage order of brs_forward (all on the caller's stream):
//   memset(header) -> preprocess -> [async copy of R, R1 and the depth-key range to pinned host + event]
//   -> depth sort pass 1 (low 8 key bits of P keys; needs none of them, so the GPU stays busy while the
//      host waits for the event) -> host: wait, allocate binning/scratch, choose the remaining digit
//      widths from the key range -> depth sort passes 2..k -> coarse binning (scan + emit of supertile
//      instances, one radix pass on the supertile id) -> fine binning (count, scan, scatter:
//      point_list and tile ranges) -> blend.
// brs_backward: memset(accumulator) -> blend backward -> fused preprocess backward (plain or
// accumulate mode, see brs_grads).  No host sync.
#include <cuda_runtime.h>
#include <nvtx3/nvToolsExt.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <atomic>
#include <map>
#include <mutex>
#include <utility>
#include <vector>

#include "common.cuh"
#include "kernels.h"

namespace brs {

namespace {

std::atomic<long long> g_launches{0}; // process-wide: autograd runs the backward on its own thread
thread_local long long t_fwd_stats[4] = {0, 0, 0, 0}; // exact, optimistic, overflow re-runs, deferred
thread_local int t_last_cuda_error = 0;

struct HostSlot { // per thread: pinned word for the R readback + its event
	int device = -1;
	uint32_t* pinned = nullptr;
	cudaEvent_t event = nullptr;
	~HostSlot() // host threads come and go (one per lane of a view batch): give the pinned word and the event back
	{
		if (pinned != nullptr)
			cudaFreeHost(pinned);
		if (event != nullptr)
			cudaEventDestroy(event);
	}
};
thread_local HostSlot t_slot;

cudaError_t ensure_slot()
{
	int dev = 0;
	cudaError_t e = cudaGetDevice(&dev);
	if (e != cudaSuccess)
		return e;
	if (t_slot.pinned != nullptr && t_slot.device == dev)
		return cudaSuccess;
	if (t_slot.pinned != nullptr) {
		cudaFreeHost(t_slot.pinned);
		cudaEventDestroy(t_slot.event);
		t_slot.pinned = nullptr;
		t_slot.event = nullptr;
		t_slot.device = -1;
	}
	e = cudaHostAlloc(reinterpret_cast<void**>(&t_slot.pinned), 64, cudaHostAllocDefault);
	if (e != cudaSuccess)
		return e;
	e = cudaEventCreateWithFlags(&t_slot.event, cudaEventDisableTiming);
	if (e != cudaSuccess)
		return e;
	t_slot.device = dev;
	return cudaSuccess;
}

// Optional per-stage CUDA-event timing (brs_stage_timing / brs_stage_times).
struct StageTimer {
	bool enabled = false;
	struct Pending { int stage; cudaEvent_t a, b; };
	std::vector<Pending> pending;
	std::vector<cudaEvent_t> pool;
	~StageTimer()
	{
		for (auto& p : pending) {
			cudaEventDestroy(p.a);
			cudaEventDestroy(p.b);
		}
		for (cudaEvent_t e : pool)
			cudaEventDestroy(e);
	}
	cudaEvent_t get()
	{
		if (!pool.empty()) {
			cudaEvent_t e = pool.back();
			pool.pop_back();
			return e;
		}
		cudaEvent_t e = nullptr;
		cudaEventCreate(&e);
		return e;
	}
};
thread_local StageTimer t_timer;

int g_nvtx_enabled = 0;
const char* const kStageNames[BRS_NUM_STAGES] = {"brs:preprocess", "brs:depth_sort", "brs:coarse_emit", "brs:coarse_sort",
                                                 "brs:fine_bin", "brs:blend_fwd", "brs:blend_bwd", "brs:preprocess_bwd"};

struct StageScope {
	int stage;
	cudaStream_t stream;
	cudaEvent_t a = nullptr;
	bool nvtx = false;
	StageScope(int stage_, cudaStream_t s) : stage(stage_), stream(s)
	{
		if (g_nvtx_enabled && stage >= 0 && stage < BRS_NUM_STAGES) {
			nvtxRangePushA(kStageNames[stage]); // host-side range around the stage's launches (nsys / ncu --nvtx)
			nvtx = true;
		}
		if (t_timer.enabled) {
			a = t_timer.get();
			cudaEventRecord(a, stream);
		}
	}
	~StageScope()
	{
		if (nvtx)
			nvtxRangePop();
		if (a != nullptr) {
			cudaEvent_t b = t_timer.get();
			cudaEventRecord(b, stream);
			t_timer.pending.push_back({stage, a, b});
		}
	}
};

// Companion stream for the blend kernels.  The blend kernels are large, issue-bound grids; everything
// else on the path is small or bandwidth-bound.  When the caller runs several views on several streams
// (view-sharded step), a blend grid monopolises the block scheduler and the other views' small kernels
// wait for its tail.  If the caller's stream has a HIGHER priority than the device's lowest, the blend
// kernels are therefore launched on a lowest-priority companion stream, fenced by events on both
// sides: stream order as the caller sees it is unchanged, but pending blocks of the (higher-priority)
// preprocess / sort / binning kernels of other views are dispatched ahead of the blend's remaining
// blocks and run underneath it.  Callers on default-priority streams get no companion.
struct Companion {
	cudaStream_t stream = nullptr;
	cudaEvent_t before = nullptr, after = nullptr;
};
std::mutex g_companion_mutex;
std::map<std::pair<int, cudaStream_t>, Companion> g_companions;
int g_companion_enabled = 1;

// Returns false when the blend should simply run on `stream`; otherwise `out` is a copy of the entry
// (handles only: the table may be rebuilt by another thread at any time).
bool companion_for(cudaStream_t stream, Companion& out)
{
	if (!g_companion_enabled || t_timer.enabled || stream == nullptr)
		return false;
	int least = 0, greatest = 0, prio = 0, dev = 0;
	if (cudaDeviceGetStreamPriorityRange(&least, &greatest) != cudaSuccess || least == greatest)
		return false;
	if (cudaStreamGetPriority(stream, &prio) != cudaSuccess || prio >= least) // numerically lower = higher priority
		return false;
	if (cudaGetDevice(&dev) != cudaSuccess)
		return false;
	std::lock_guard<std::mutex> lock(g_companion_mutex);
	if (g_companions.size() >= 64 && g_companions.find(std::make_pair(dev, stream)) == g_companions.end()) {
		// callers that keep creating streams would grow the table without bound: drop it and start over
		// (destroying a stream / event with work in flight is legal, the driver releases it afterwards)
		for (auto& kv : g_companions) {
			cudaStreamDestroy(kv.second.stream);
			cudaEventDestroy(kv.second.before);
			cudaEventDestroy(kv.second.after);
		}
		g_companions.clear();
	}
	Companion& c = g_companions[std::make_pair(dev, stream)];
	if (c.stream == nullptr) {
		if (cudaStreamCreateWithPriority(&c.stream, cudaStreamNonBlocking, least) != cudaSuccess ||
		    cudaEventCreateWithFlags(&c.before, cudaEventDisableTiming) != cudaSuccess ||
		    cudaEventCreateWithFlags(&c.after, cudaEventDisableTiming) != cudaSuccess) {
			c = Companion{};
			return false;
		}
	}
	out = c;
	return true;
}

inline int fail_cuda(cudaError_t e)
{
	t_last_cuda_error = (int)e;
	return BRS_ERR_CUDA;
}

#define BRS_CUDA(expr)                                                                                                 \
	do {                                                                                                               \
		cudaError_t _e = (expr);                                                                                       \
		if (_e != cudaSuccess)                                                                                         \
			return fail_cuda(_e);                                                                                      \
	} while (0)

// reference CHECK_CUDA (auxiliary.h:166-173): only when debug, synchronise and surface errors
#define BRS_STAGE(stage_id, expr, debug, stream)                                                                       \
	do {                                                                                                               \
		StageScope _scope(stage_id, stream);                                                                           \
		BRS_CUDA(expr);                                                                                                \
		if (debug)                                                                                                     \
			BRS_CUDA(cudaStreamSynchronize(stream));                                                                   \
	} while (0)

constexpr size_t HEADER_BYTES = 256;

struct GeomLayout {
	size_t header, records, depth_key, rect, order, total;
};
GeomLayout geom_layout(size_t P)
{
	GeomLayout l{};
	size_t off = 0;
	l.header = off;
	off += HEADER_BYTES;
	l.records = off;
	off += align_up(sizeof(float4) * 3 * P, 256);
	l.depth_key = off;
	off += align_up(sizeof(uint32_t) * P, 256);
	l.rect = off;
	off += align_up(sizeof(uint2) * P, 256);
	l.order = off;
	off += align_up(sizeof(uint32_t) * P, 256);
	l.total = off;
	return l;
}

struct ImageLayout {
	size_t ranges, final_T, n_contrib, total;
};
ImageLayout image_layout(int W, int H, bool pixel_state = true)
{
	ImageLayout l{};
	const size_t gx = (W + TILE_X - 1) / TILE_X, gy = (H + TILE_Y - 1) / TILE_Y;
	const size_t npix = (size_t)W * H;
	size_t off = 0;
	l.ranges = off;
	off += align_up(sizeof(uint2) * gx * gy, 256);
	l.final_T = off;
	off += pixel_state ? align_up(sizeof(float) * npix, 256) : 0;
	l.n_contrib = off;
	off += pixel_state ? align_up(sizeof(uint32_t) * npix, 256) : 0;
	l.total = off < 256 ? 256 : off;
	return l;
}

size_t binning_bytes(size_t R) { return align_up(sizeof(uint32_t) * (R ? R : 1), 256); }

int validate_view(const brs_view* v, bool need_campos_bg)
{
	if (v == nullptr || v->viewmatrix == nullptr || v->projmatrix == nullptr)
		return BRS_ERR_INVALID_ARG;
	if (v->image_width < 0 || v->image_height < 0)
		return BRS_ERR_INVALID_ARG;
	if (v->image_width >= 65536 * TILE_X || v->image_height >= 65536 * TILE_Y)
		return BRS_ERR_UNSUPPORTED; // tile coordinates are packed into 16 bits
	if (need_campos_bg && v->bg == nullptr)
		return BRS_ERR_INVALID_ARG;
	return BRS_OK;
}

int validate_gaussians(const brs_view* v, const brs_gaussians* g)
{
	if (g == nullptr || g->P < 0)
		return BRS_ERR_INVALID_ARG;
	if (g->P == 0)
		return BRS_OK;
	if (g->means3D == nullptr || g->opacities == nullptr)
		return BRS_ERR_INVALID_ARG;
	// reference Python wrapper raises for both / neither (depth_diff_gaussian_rasterization/__init__.py:192-196)
	if ((g->shs == nullptr) == (g->colors_precomp == nullptr))
		return BRS_ERR_INVALID_ARG;
	const bool has_sr = g->scales != nullptr && g->rotations != nullptr;
	if (has_sr == (g->cov3D_precomp != nullptr))
		return BRS_ERR_INVALID_ARG;
	if (!has_sr && (g->scales != nullptr || g->rotations != nullptr))
		return BRS_ERR_INVALID_ARG;
	if (g->shs != nullptr) {
		if (v->sh_degree < 0 || v->sh_degree > 3)
			return BRS_ERR_UNSUPPORTED;
		if (v->sh_coeffs < (v->sh_degree + 1) * (v->sh_degree + 1) || v->sh_coeffs > 16)
			return BRS_ERR_INVALID_ARG;
		if (v->campos == nullptr)
			return BRS_ERR_INVALID_ARG;
	}
	return BRS_OK;
}

} // namespace

void count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }

} // namespace brs

using namespace brs;

extern "C" {

int brs_version(void) { return BRS_VERSION; }

long long brs_launch_count(int reset)
{
	const long long v = reset ? g_launches.exchange(0) : g_launches.load();
	return v;
}

int brs_last_cuda_error(void) { return t_last_cuda_error; }
const char* brs_last_cuda_error_string(void) { return cudaGetErrorString((cudaError_t)t_last_cuda_error); }

const char* brs_error_string(int status)
{
	switch (status) {
	case BRS_OK: return "ok";
	case BRS_ERR_INVALID_ARG: return "invalid argument";
	case BRS_ERR_ALLOC: return "allocator callback returned NULL";
	case BRS_ERR_CUDA: return "CUDA error (see brs_last_cuda_error_string)";
	case BRS_ERR_UNSUPPORTED: return "unsupported configuration";
	case BRS_ERR_STATE: return "forward state does not match the given sizes";
	default: return "unknown status";
	}
}

size_t brs_geom_bytes(int P) { return geom_layout(P < 0 ? 0 : (size_t)P).total; }
size_t brs_binning_bytes(int R) { return binning_bytes(R < 0 ? 0 : (size_t)R); }
size_t brs_image_bytes(int W, int H) { return image_layout(W, H).total; }
size_t brs_sort_scratch_bytes(int n) { return sort_scratch_bytes(n < 0 ? 0 : (size_t)n); }

// Scratch of one forward with the given capacities: [zeroed: depth sort | instance levels][plain: both].
static size_t forward_scratch_bytes(size_t P, size_t V_cap, size_t R1_cap, uint32_t grid_x, uint32_t grid_y, int depth_passes)
{
	return depth_zero_bytes(P, V_cap, depth_passes) + inst_zero_bytes(P, R1_cap, grid_x, grid_y) + depth_plain_bytes(P) +
	       inst_plain_bytes(P, R1_cap, grid_x, grid_y);
}
size_t brs_forward_scratch_bytes(int P, int R, int W, int H)
{
	const uint32_t gx = W > 0 ? (W + TILE_X - 1) / TILE_X : 0, gy = H > 0 ? (H + TILE_Y - 1) / TILE_Y : 0;
	// R1 (supertile instances) never exceeds R (tile instances)
	return forward_scratch_bytes(P < 0 ? 0 : P, P < 0 ? 0 : P, R < 0 ? 0 : R, gx, gy, 4);
}
size_t brs_backward_scratch_bytes(int P) { return align_up(sizeof(float) * ACCUM_STRIDE * (P < 0 ? 0 : (size_t)P), 256); }

int brs_state_layout(int P, int R, int W, int H, brs_layout* out)
{
	if (out == nullptr || P < 0 || R < 0 || W < 0 || H < 0)
		return BRS_ERR_INVALID_ARG;
	const GeomLayout g = geom_layout(P);
	const ImageLayout im = image_layout(W, H);
	out->geom_records = g.records;
	out->geom_depth_key = g.depth_key;
	out->geom_rect = g.rect;
	out->geom_order = g.order;
	out->binning_point_list = 0;
	out->image_ranges = im.ranges;
	out->image_final_T = im.final_T;
	out->image_n_contrib = im.n_contrib;
	return BRS_OK;
}

void brs_stage_timing(int enable) { t_timer.enabled = enable != 0; }

int brs_stage_nvtx(int enable)
{
	const int old = g_nvtx_enabled;
	if (enable >= 0)
		g_nvtx_enabled = enable != 0;
	return old;
}

int brs_blend_companion_stream(int enable)
{
	const int old = g_companion_enabled;
	if (enable >= 0)
		g_companion_enabled = enable != 0;
	return old;
}

int brs_stage_times(float* ms, int* calls)
{
	for (auto& p : t_timer.pending) {
		BRS_CUDA(cudaEventSynchronize(p.b));
		float t = 0.f;
		BRS_CUDA(cudaEventElapsedTime(&t, p.a, p.b));
		if (p.stage >= 0 && p.stage < BRS_NUM_STAGES) {
			if (ms)
				ms[p.stage] += t;
			if (calls)
				calls[p.stage] += 1;
		}
		t_timer.pool.push_back(p.a);
		t_timer.pool.push_back(p.b);
	}
	t_timer.pending.clear();
	return BRS_OK;
}

double brs_probe_fp32_tflops(brs_stream stream) { return probe_fp32_tflops(stream); }

int brs_count_pairs(const brs_view* view, const brs_fwd_state* state, int P, unsigned long long* out, brs_stream stream)
{
	if (view == nullptr || state == nullptr || out == nullptr || P < 0)
		return BRS_ERR_INVALID_ARG;
	const int W = view->image_width, H = view->image_height;
	const GeomLayout gl = geom_layout(P);
	const ImageLayout il = image_layout(W, H);
	if (P == 0 || state->geom == nullptr || state->image == nullptr) {
		BRS_CUDA(cudaMemsetAsync(out, 0, 3 * sizeof(unsigned long long), stream));
		return BRS_OK;
	}
	const char* geom = static_cast<const char*>(state->geom);
	char* image = static_cast<char*>(state->image);
	BlendFwdArgs ba{};
	ba.ranges = reinterpret_cast<const uint2*>(image + il.ranges);
	ba.point_list = reinterpret_cast<const uint32_t*>(state->binning);
	ba.records = reinterpret_cast<const float4*>(geom + gl.records);
	ba.W = W;
	ba.H = H;
	ba.grid_x = (W + TILE_X - 1) / TILE_X;
	ba.grid_y = (H + TILE_Y - 1) / TILE_Y;
	ba.n_contrib = reinterpret_cast<uint32_t*>(image + il.n_contrib);
	BRS_CUDA(launch_count_pairs(ba, out, stream));
	return BRS_OK;
}

int brs_sort_pairs_u32(const uint32_t* keys_in, const uint32_t* vals_in, uint32_t* keys_out, uint32_t* vals_out, int n,
                       int begin_bit, int end_bit, void* scratch, brs_stream stream)
{
	if (n < 0 || begin_bit < 0 || end_bit > 32 || begin_bit > end_bit)
		return BRS_ERR_INVALID_ARG;
	if (n == 0)
		return BRS_OK;
	if (n > (1 << 30))
		return BRS_ERR_UNSUPPORTED;
	if (keys_in == nullptr || keys_out == nullptr || vals_out == nullptr || scratch == nullptr)
		return BRS_ERR_INVALID_ARG;
	BRS_CUDA(sort_pairs(keys_in, vals_in, keys_out, vals_out, (size_t)n, begin_bit, end_bit, scratch, stream));
	return BRS_OK;
}

} // extern "C"

namespace {

// High-water marks of the instance counts per (device, P, W, H): what sizes an optimistic forward.
struct Marks {
	uint32_t R = 0, R1 = 0, key_bits = 0, V = 0;
};
struct MarksKey {
	int dev, P, W, H;
	bool operator<(const MarksKey& o) const
	{
		return dev != o.dev ? dev < o.dev : (P != o.P ? P < o.P : (W != o.W ? W < o.W : H < o.H));
	}
};
std::mutex g_marks_mutex;
std::map<MarksKey, Marks> g_marks;

bool lookup_marks(const MarksKey& k, Marks& out)
{
	std::lock_guard<std::mutex> lock(g_marks_mutex);
	auto it = g_marks.find(k);
	if (it == g_marks.end())
		return false;
	out = it->second;
	return true;
}
void raise_marks(const MarksKey& k, uint32_t R, uint32_t R1, uint32_t key_bits, uint32_t V)
{
	std::lock_guard<std::mutex> lock(g_marks_mutex);
	if (g_marks.size() >= 256 && g_marks.find(k) == g_marks.end())
		g_marks.clear();
	Marks& m = g_marks[k];
	m.R = R > m.R ? R : m.R;
	m.R1 = R1 > m.R1 ? R1 : m.R1;
	m.key_bits = key_bits > m.key_bits ? key_bits : m.key_bits;
	m.V = V > m.V ? V : m.V;
}

struct Caps {
	uint32_t R_cap, R1_cap;
	uint32_t V_cap = 0xffffffffu; // visible Gaussians (all of them unless known better)
	int depth_passes;
};
int passes_for_bits(uint32_t key_bits)
{
	int p = ((int)key_bits + 7) / 8;
	return p < 2 ? 2 : (p > 4 ? 4 : p); // >= 2: see launch_depth_sort_begin
}
Caps caps_from_marks(const Marks& m)
{
	Caps c;
	c.R_cap = m.R + m.R / 4 + 4096;
	c.R1_cap = m.R1 + m.R1 / 4 + 4096;
	c.V_cap = m.V + m.V / 4 + 4096;
	c.depth_passes = passes_for_bits(m.key_bits + 1);
	return c;
}

struct ForwardCtx {
	const brs_view* view; // n_views of them
	int n_views;          // > 1: a stack of views rendered as one pipeline (brs_forward_views[_ex])
	const int* view_P;    // Gaussians of each view (brs_forward_views_ex), or nullptr: every view sees all of them
	size_t P_inst;        // instances (view, Gaussian) of the pipeline: the sum of view_P, else n_views * P
	int W, H;
	uint32_t grid_x, grid_y; // tiles of ONE view; the stack has n_views * grid_y tile rows
	bool debug;
	brs_alloc_fn alloc;
	void* alloc_ctx;
	brs_fwd_state* state;
	cudaStream_t stream;
	char* geom;
	char* image;
	GeomLayout gl;
	ImageLayout il;
	float* out_color;
	float* out_depth;
};

// Everything after preprocess, sized by `caps`: depth sort -> emission -> coarse sort -> fine binning ->
// blend.  No host wait in here.  If `report` is given, the header (counts + overflow word) is copied to
// it right after the depth sort's histogram kernel has judged the capacities.
int enqueue_binning_and_blend(const ForwardCtx& c, const Caps& caps, uint32_t* report, cudaEvent_t report_event,
                              uint32_t* overflow_accum = nullptr)
{
	cudaStream_t stream = c.stream;
	const bool debug = c.debug;
	uint32_t* hdr = reinterpret_cast<uint32_t*>(c.geom + c.gl.header);
	char* binning = static_cast<char*>(c.alloc(c.alloc_ctx, BRS_BUF_BINNING, binning_bytes(caps.R_cap)));
	if (binning == nullptr)
		return BRS_ERR_ALLOC;
	c.state->binning = binning;
	c.state->binning_bytes = binning_bytes(caps.R_cap);

	const size_t P_inst = c.P_inst;
	const uint32_t rows = c.grid_y * (uint32_t)c.n_views;   // tile rows of the stack of views
	BinPlan pl{};
	pl.P = (uint32_t)P_inst;
	pl.R1_cap = caps.R1_cap;
	pl.R_cap = caps.R_cap;
	pl.V_cap = caps.V_cap < P_inst ? caps.V_cap : (uint32_t)P_inst;
	pl.grid_x = c.grid_x;
	pl.grid_y = rows;
	pl.ns_x = supertiles(c.grid_x);
	pl.ns = pl.ns_x * supertiles(rows);
	pl.depth_passes = caps.depth_passes;
	pl.hdr = hdr;
	pl.depth_key = reinterpret_cast<const uint32_t*>(c.geom + c.gl.depth_key);
	pl.rect = reinterpret_cast<const uint2*>(c.geom + c.gl.rect);
	pl.order = reinterpret_cast<uint32_t*>(c.geom + c.gl.order);
	pl.point_list = reinterpret_cast<uint32_t*>(binning);
	pl.ranges = reinterpret_cast<uint2*>(c.image + c.il.ranges);
	pl.overflow_accum = overflow_accum;

	const bool have_grid = c.grid_x * rows > 0;
	if (have_grid) {
		const size_t dz = depth_zero_bytes(P_inst, caps.V_cap, caps.depth_passes), iz = inst_zero_bytes(P_inst, caps.R1_cap, c.grid_x, rows);
		const size_t dp = depth_plain_bytes(P_inst);
		char* scratch = static_cast<char*>(
		    c.alloc(c.alloc_ctx, BRS_BUF_SCRATCH, forward_scratch_bytes(P_inst, caps.V_cap, caps.R1_cap, c.grid_x, rows, caps.depth_passes)));
		if (scratch == nullptr)
			return BRS_ERR_ALLOC;
		BRS_CUDA(cudaMemsetAsync(scratch, 0, dz + iz, stream)); // tickets, histograms, look-back status words
		pl.d = carve_depth_scratch(scratch, scratch + dz + iz, P_inst, caps.V_cap, caps.depth_passes);
		pl.i = carve_inst_scratch(scratch + dz, scratch + dz + iz + dp, P_inst, caps.R1_cap, c.grid_x, rows);

		BRS_STAGE(BRS_STAGE_DEPTH_SORT, launch_depth_sort_begin(pl, caps.depth_passes, stream), debug, stream);
		if (report != nullptr) {
			BRS_CUDA(cudaMemcpyAsync(report, hdr, HDR_WORDS * sizeof(uint32_t), cudaMemcpyDeviceToHost, stream));
			if (report_event != nullptr)
				BRS_CUDA(cudaEventRecord(report_event, stream));
		}
		BRS_STAGE(BRS_STAGE_DEPTH_SORT, launch_depth_sort_rest(pl, stream), debug, stream);
		BRS_STAGE(BRS_STAGE_COARSE_EMIT, launch_emit(pl, stream), debug, stream);
		BRS_STAGE(BRS_STAGE_COARSE_SORT, launch_coarse_sort(pl, stream), debug, stream);
		// also writes the (0,0) ranges of empty tiles (reference: cudaMemset, rasterizer_impl.cu:311)
		BRS_STAGE(BRS_STAGE_FINE_BIN, launch_fine_binning(pl, stream), debug, stream);
	} else if (report != nullptr) {
		BRS_CUDA(cudaMemcpyAsync(report, hdr, HDR_WORDS * sizeof(uint32_t), cudaMemcpyDeviceToHost, stream));
		if (report_event != nullptr)
			BRS_CUDA(cudaEventRecord(report_event, stream));
	}

	BlendFwdArgs ba{};
	ba.ranges = pl.ranges;
	ba.point_list = pl.point_list;
	ba.records = reinterpret_cast<const float4*>(c.geom + c.gl.records);
	ba.bg = c.view->bg;
	ba.W = c.W;
	ba.H = c.H;
	ba.grid_x = c.grid_x;
	ba.grid_y = c.grid_y;
	ba.views = c.n_views;
	// a stack of views is forward-only: the per-pixel state the backward needs is not kept
	ba.final_T = c.n_views > 1 ? nullptr : reinterpret_cast<float*>(c.image + c.il.final_T);
	ba.n_contrib = c.n_views > 1 ? nullptr : reinterpret_cast<uint32_t*>(c.image + c.il.n_contrib);
	ba.out_color = c.out_color;
	ba.out_depth = c.out_depth;
	Companion comp;
	if (!debug && companion_for(stream, comp)) {
		BRS_CUDA(cudaEventRecord(comp.before, stream));
		BRS_CUDA(cudaStreamWaitEvent(comp.stream, comp.before, 0));
		BRS_CUDA(launch_blend_forward(ba, comp.stream));
		BRS_CUDA(cudaEventRecord(comp.after, comp.stream));
		BRS_CUDA(cudaStreamWaitEvent(stream, comp.after, 0));
	} else {
		BRS_STAGE(BRS_STAGE_BLEND_FWD, launch_blend_forward(ba, stream), debug, stream);
	}
	if (c.view_P != nullptr) {
		// a view without Gaussians comes out as the reference's P == 0 forward does: zeros, no background
		const size_t npix = (size_t)c.W * c.H;
		for (int v = 0; v < c.n_views; v++) {
			if (c.view_P[v] == 0 && npix > 0) {
				BRS_CUDA(cudaMemsetAsync(c.out_color + (size_t)v * NUM_CHANNELS * npix, 0, sizeof(float) * NUM_CHANNELS * npix, stream));
				BRS_CUDA(cudaMemsetAsync(c.out_depth + (size_t)v * npix, 0, sizeof(float) * npix, stream));
			}
		}
	}
	return BRS_OK;
}

// One forward over a stack of n_views views (n_views == 1: brs_forward_ex).  The views' preprocess launches write
// into ONE instance space — with view_P == nullptr instance v * P + i is Gaussian i seen from view v, else view v
// owns rows and instances [off_v, off_v + view_P[v]) — each instance's tile rectangle shifted down by v * grid_y
// rows, so that everything behind it (depth sort, emission, coarse sort, fine binning, blend) runs once over all
// views.
int forward_impl(const brs_view* views, int n_views, const brs_gaussians* g, const int* view_P, float* out_color,
                 float* out_depth, int* radii, brs_alloc_fn alloc, void* alloc_ctx, brs_fwd_state* state,
                 const brs_fwd_options* opt, cudaStream_t stream)
{
	const brs_view* view = views;
	if (views == nullptr || n_views < 1 || n_views > 65535)
		return BRS_ERR_INVALID_ARG;
	int st = BRS_OK;
	for (int v = 0; v < n_views && st == BRS_OK; v++) {
		st = validate_view(views + v, true);
		if (st == BRS_OK)
			st = validate_gaussians(views + v, g);
		// one image size, one SH layout and one debug flag for the whole stack; the background of views[0] is used
		if (st == BRS_OK && (views[v].image_width != view->image_width || views[v].image_height != view->image_height ||
		                     views[v].sh_degree != view->sh_degree || views[v].sh_coeffs != view->sh_coeffs ||
		                     views[v].debug != view->debug))
			st = BRS_ERR_INVALID_ARG;
	}
	if (st != BRS_OK)
		return st;
	if (view_P != nullptr) {
		long long sum = 0;
		for (int v = 0; v < n_views; v++) {
			if (view_P[v] < 0)
				return BRS_ERR_INVALID_ARG;
			sum += view_P[v];
		}
		if (sum > (1ll << 31) - 1)
			return BRS_ERR_UNSUPPORTED; // instance ids are 32-bit
		if (sum != g->P)
			return BRS_ERR_INVALID_ARG;
	}
	if (alloc == nullptr || state == nullptr)
		return BRS_ERR_INVALID_ARG;
	static const bool nvtx_env = [] {
		const char* e = getenv("BRS_NVTX");
		if (e != nullptr && e[0] == '1')
			g_nvtx_enabled = 1;
		return true;
	}();
	(void)nvtx_env;
	const int mode = opt ? opt->mode : BRS_FWD_AUTO;
	if (mode != BRS_FWD_AUTO && mode != BRS_FWD_EXACT && mode != BRS_FWD_DEFERRED)
		return BRS_ERR_INVALID_ARG;
	if (mode == BRS_FWD_DEFERRED && opt->report == nullptr && opt->overflow_accum == nullptr)
		return BRS_ERR_INVALID_ARG;
	const int W = view->image_width, H = view->image_height, P = g->P;
	const size_t npix = (size_t)W * H * n_views;
	const size_t P_inst = view_P != nullptr ? (size_t)P : (size_t)P * n_views;
	if (P_inst > (1ull << 31) - 1 || (size_t)((H + TILE_Y - 1) / TILE_Y) * n_views >= 65536)
		return BRS_ERR_UNSUPPORTED; // instance ids are 32-bit, tile rows of the stack are packed into 16 bits
	if ((npix > 0 && (out_color == nullptr || out_depth == nullptr)) || (P > 0 && radii == nullptr))
		return BRS_ERR_INVALID_ARG;
	const bool debug = view->debug != 0;

	memset(state, 0, sizeof(*state));

	if (P == 0) {
		// reference rasterize_points.cu:68-82: outputs are zero-filled and no kernel runs (so the
		// background is NOT composited when there are no Gaussians at all).
		if (npix > 0) {
			BRS_CUDA(cudaMemsetAsync(out_color, 0, sizeof(float) * NUM_CHANNELS * npix, stream));
			BRS_CUDA(cudaMemsetAsync(out_depth, 0, sizeof(float) * npix, stream));
		}
		if (mode == BRS_FWD_DEFERRED && opt->report != nullptr)
			memset(opt->report, 0, HDR_WORDS * sizeof(uint32_t));
		return BRS_OK;
	}

	ForwardCtx c{};
	c.view = view;
	c.n_views = n_views;
	c.view_P = view_P;
	c.P_inst = P_inst;
	c.W = W;
	c.H = H;
	c.grid_x = (W + TILE_X - 1) / TILE_X;
	c.grid_y = (H + TILE_Y - 1) / TILE_Y;
	c.debug = debug;
	c.alloc = alloc;
	c.alloc_ctx = alloc_ctx;
	c.state = state;
	c.stream = stream;
	c.gl = geom_layout(P_inst);
	c.il = n_views > 1 ? image_layout(W, (int)(c.grid_y * n_views * TILE_Y), false) : image_layout(W, H);
	c.out_color = out_color;
	c.out_depth = out_depth;

	c.geom = static_cast<char*>(alloc(alloc_ctx, BRS_BUF_GEOM, c.gl.total));
	c.image = static_cast<char*>(alloc(alloc_ctx, BRS_BUF_IMAGE, c.il.total));
	if (c.geom == nullptr || c.image == nullptr)
		return BRS_ERR_ALLOC;
	state->geom = c.geom;
	state->geom_bytes = c.gl.total;
	state->image = c.image;
	state->image_bytes = c.il.total;

	uint32_t* hdr = reinterpret_cast<uint32_t*>(c.geom + c.gl.header);
	BRS_CUDA(cudaMemsetAsync(hdr, 0, HEADER_BYTES, stream));

	PreprocessArgs pa{};
	pa.D = view->sh_degree;
	pa.M = g->shs ? view->sh_coeffs : 0;
	pa.means3D = g->means3D;
	pa.scales = g->scales;
	pa.rotations = g->rotations;
	pa.opacities = g->opacities;
	pa.shs = g->shs;
	pa.cov3D_precomp = g->cov3D_precomp;
	pa.colors_precomp = g->colors_precomp;
	pa.W = W;
	pa.H = H;
	pa.grid_x = c.grid_x;
	pa.grid_y = c.grid_y;
	pa.total_tiles = hdr;
	int dev = 0;
	BRS_CUDA(cudaGetDevice(&dev));
	const MarksKey key{dev, (int)P_inst, W, H * n_views};
	Marks marks;
	const bool have_marks = lookup_marks(key, marks);
	// SH rows: requested for all Gaussians up front when most of them were visible in the last views of this shape
	pa.eager_sh = (have_marks && 2ull * marks.V > (unsigned long long)P_inst) ? 1 : 0;
	pa.radii = radii;
	pa.records = reinterpret_cast<float4*>(c.geom + c.gl.records);
	pa.depth_key = reinterpret_cast<uint32_t*>(c.geom + c.gl.depth_key);
	pa.rect = reinterpret_cast<uint2*>(c.geom + c.gl.rect);
	// one launch per MAX_VIEWS views: blockIdx.y picks the view, its outputs go to instances [v * P, (v + 1) * P), or
	// with view_P to [off_v, off_v + view_P[v]), where off_v is also its first input row.  A single view is the
	// table {(0, 0, P)}.
	size_t off = 0;
	for (int v0 = 0; v0 < n_views; v0 += PreprocessViewTable::MAX_VIEWS) {
		const int nv = n_views - v0 < PreprocessViewTable::MAX_VIEWS ? n_views - v0 : PreprocessViewTable::MAX_VIEWS;
		PreprocessViewTable t{};
		t.first_view = (uint32_t)v0;
		for (int k = 0; k < nv; k++) {
			const brs_view* vw = views + v0 + k;
			PreprocessViewTable::Slot& sl = t.v[k];
			sl.viewmatrix = vw->viewmatrix;
			sl.projmatrix = vw->projmatrix;
			sl.campos = vw->campos;
			sl.tan_fovx = vw->tanfovx;
			sl.tan_fovy = vw->tanfovy;
			sl.focal_y = H / (2.0f * vw->tanfovy); // rasterizer_impl.cu:223-224
			sl.focal_x = W / (2.0f * vw->tanfovx);
			sl.scale_modifier = vw->scale_modifier;
			sl.prefiltered = vw->prefiltered;
			sl.count = (uint32_t)(view_P != nullptr ? view_P[v0 + k] : P);
			sl.row = view_P != nullptr ? (uint32_t)off : 0u;
			sl.inst = (uint32_t)off;
			off += sl.count;
		}
		BRS_STAGE(BRS_STAGE_PREPROCESS, launch_preprocess(pa, t, nv, stream), debug, stream);
	}

	// ---- deferred: the caller's capacities (or the high-water marks), no host wait at all ----
	if (mode == BRS_FWD_DEFERRED) {
		Caps caps = caps_from_marks(marks); // zero marks -> the 4096-instance floor
		if (!have_marks)
			caps.V_cap = 0xffffffffu; // the caller's capacities speak for R and R1 only
		if (opt->R_cap > 0)
			caps.R_cap = (uint32_t)opt->R_cap;
		if (opt->R1_cap > 0)
			caps.R1_cap = (uint32_t)opt->R1_cap;
		if (opt->depth_bits > 0)
			caps.depth_passes = passes_for_bits((uint32_t)opt->depth_bits);
		if (caps.R_cap > (1u << 30) || caps.R1_cap > (1u << 30))
			return BRS_ERR_UNSUPPORTED;
		state->num_rendered = -1; // on the device; the caller reads it from `report` once the stream has passed it
		t_fwd_stats[3]++;
		return enqueue_binning_and_blend(c, caps, opt->report, nullptr, opt->overflow_accum);
	}

	BRS_CUDA(ensure_slot());
	Caps caps{};
	bool counts_known = false;
	if (mode == BRS_FWD_AUTO && have_marks) {
		// ---- optimistic: everything is enqueued with capacities from the high-water marks; the host then
		// waits for the header, which left the device right after preprocess + one histogram kernel, while
		// the GPU still has the sort, the binning and the blend queued behind it ----
		caps = caps_from_marks(marks);
		t_fwd_stats[1]++;
		st = enqueue_binning_and_blend(c, caps, t_slot.pinned, t_slot.event);
		if (st != BRS_OK)
			return st;
		BRS_CUDA(cudaEventSynchronize(t_slot.event));
		counts_known = true;
		if (t_slot.pinned[HDR_OVERFLOW] == 0) {
			state->num_rendered = (int)t_slot.pinned[HDR_R];
			raise_marks(key, t_slot.pinned[HDR_R], t_slot.pinned[HDR_R1], t_slot.pinned[HDR_KEY_BITS], t_slot.pinned[HDR_V]);
			return BRS_OK;
		}
		// a capacity was too small: what was enqueued is memory-safe but wrong; run it again with the exact sizes
		t_fwd_stats[2]++;
	} else {
		t_fwd_stats[0]++;
		// ---- exact: wait for the counts right after preprocess (the reference's one host wait,
		// rasterizer_impl.cu:282), then size everything exactly ----
		BRS_CUDA(cudaMemcpyAsync(t_slot.pinned, hdr, HDR_WORDS * sizeof(uint32_t), cudaMemcpyDeviceToHost, stream));
		BRS_CUDA(cudaEventRecord(t_slot.event, stream));
		BRS_CUDA(cudaEventSynchronize(t_slot.event));
	}
	const uint32_t R = t_slot.pinned[HDR_R], R1 = t_slot.pinned[HDR_R1], V = t_slot.pinned[HDR_V];
	if (R > (1u << 30))
		return BRS_ERR_UNSUPPORTED;
	uint32_t key_bits = 8;
	if (counts_known) {
		key_bits = t_slot.pinned[HDR_KEY_BITS];
	} else if (V > 0) {
		const uint32_t key_min = ~t_slot.pinned[HDR_KEY_INVMIN], key_max = t_slot.pinned[HDR_KEY_MAX];
		const uint32_t span = key_max - (key_min & ~0xFFu);
		while (key_bits < 32 && (span >> key_bits) != 0u)
			key_bits++;
	}
	caps.R_cap = R;
	caps.R1_cap = R1;
	caps.V_cap = V;
	caps.depth_passes = passes_for_bits(key_bits);
	state->num_rendered = (int)R;
	raise_marks(key, R, R1, key_bits, V);
	return enqueue_binning_and_blend(c, caps, nullptr, nullptr);
}

} // namespace

extern "C" {

int brs_forward(const brs_view* view, const brs_gaussians* g, float* out_color, float* out_depth, int* radii,
                brs_alloc_fn alloc, void* alloc_ctx, brs_fwd_state* state, brs_stream stream)
{
	return brs_forward_ex(view, g, out_color, out_depth, radii, alloc, alloc_ctx, state, nullptr, stream);
}

int brs_forward_ex(const brs_view* view, const brs_gaussians* g, float* out_color, float* out_depth, int* radii,
                   brs_alloc_fn alloc, void* alloc_ctx, brs_fwd_state* state, const brs_fwd_options* opt, brs_stream stream)
{
	return forward_impl(view, 1, g, nullptr, out_color, out_depth, radii, alloc, alloc_ctx, state, opt, stream);
}

int brs_forward_views(const brs_view* views, int n_views, const brs_gaussians* g, float* out_color, float* out_depth,
                      int* radii, brs_alloc_fn alloc, void* alloc_ctx, long long* num_rendered, const brs_fwd_options* opt,
                      brs_stream stream)
{
	return brs_forward_views_ex(views, n_views, g, nullptr, out_color, out_depth, radii, alloc, alloc_ctx, num_rendered, opt,
	                            stream);
}

int brs_forward_views_ex(const brs_view* views, int n_views, const brs_gaussians* g, const int* view_P, float* out_color,
                         float* out_depth, int* radii, brs_alloc_fn alloc, void* alloc_ctx, long long* num_rendered,
                         const brs_fwd_options* opt, brs_stream stream)
{
	brs_fwd_state st{};
	const int rc = forward_impl(views, n_views, g, view_P, out_color, out_depth, radii, alloc, alloc_ctx, &st, opt, stream);
	if (num_rendered != nullptr)
		*num_rendered = st.num_rendered;
	return rc;
}

void brs_forward_stats(long long* out, int reset)
{
	for (int i = 0; i < 4; i++) {
		if (out)
			out[i] = t_fwd_stats[i];
		if (reset)
			t_fwd_stats[i] = 0;
	}
}

int brs_get_marks(int P, int image_width, int image_height, uint32_t* out)
{
	int dev = 0;
	Marks m;
	if (cudaGetDevice(&dev) != cudaSuccess || !lookup_marks(MarksKey{dev, P, image_width, image_height}, m))
		return 0;
	if (out != nullptr) {
		out[0] = m.R;
		out[1] = m.R1;
		out[2] = m.key_bits;
	}
	return 1;
}

void brs_reset_marks(void)
{
	std::lock_guard<std::mutex> lock(g_marks_mutex);
	g_marks.clear();
}

void brs_note_counts(int P, int image_width, int image_height, const uint32_t* report)
{
	int dev = 0;
	if (report == nullptr || cudaGetDevice(&dev) != cudaSuccess)
		return;
	raise_marks(MarksKey{dev, P, image_width, image_height}, report[HDR_R], report[HDR_R1], report[HDR_KEY_BITS], report[HDR_V]);
}

int brs_backward(const brs_view* view, const brs_gaussians* g, const int* radii, const brs_fwd_state* state,
                 const float* dL_dout_color, const float* dL_dout_depth, const brs_grads* grads, brs_alloc_fn alloc,
                 void* alloc_ctx, brs_stream stream)
{
	return brs_backward_ex(view, g, radii, state, dL_dout_color, dL_dout_depth, grads, nullptr, alloc, alloc_ctx, stream);
}

int brs_backward_ex(const brs_view* view, const brs_gaussians* g, const int* radii, const brs_fwd_state* state,
                    const float* dL_dout_color, const float* dL_dout_depth, const brs_grads* grads,
                    const brs_densify_stats* stats, brs_alloc_fn alloc, void* alloc_ctx, brs_stream stream)
{
	// reference: dL_dout_depth is plumbed and never used (backward.cu:443-554); it is read only when
	// the caller opts in with brs_grads.depth_gradient
	int st = validate_view(view, true);
	if (st != BRS_OK)
		return st;
	st = validate_gaussians(view, g);
	if (st != BRS_OK)
		return st;
	if (grads == nullptr || state == nullptr || alloc == nullptr)
		return BRS_ERR_INVALID_ARG;
	if (stats != nullptr && (stats->grad_norm == nullptr || stats->count == nullptr || stats->rows < 0 ||
	                         (stats->index == nullptr && stats->rows < g->P)))
		return BRS_ERR_INVALID_ARG;
	const int P = g->P;
	if (P == 0)
		return BRS_OK;
	const int W = view->image_width, H = view->image_height;
	const int M = g->shs ? view->sh_coeffs : 0;
	const bool acc = grads->accumulate != 0;
	const bool has_sr = g->scales != nullptr;
	// plain mode needs every tensor; in accumulate mode every parameter sink is optional (a NULL sink
	// = a frozen parameter whose gradient the caller does not want) and only dL_dmeans2D is required
	if (radii == nullptr || grads->dL_dmeans2D == nullptr)
		return BRS_ERR_INVALID_ARG;
	if (!acc && (grads->dL_dopacity == nullptr || grads->dL_dmeans3D == nullptr || (M > 0 && grads->dL_dsh == nullptr) ||
	             grads->dL_dcolors == nullptr || grads->dL_dcov3D == nullptr || grads->dL_dscales == nullptr ||
	             grads->dL_drotations == nullptr))
		return BRS_ERR_INVALID_ARG;
	const GeomLayout gl = geom_layout(P);
	const ImageLayout il = image_layout(W, H);
	const int R = state->num_rendered;
	// R == -1: a deferred forward, whose instance count never reached the host (brs_fwd_options)
	if (state->geom == nullptr || state->image == nullptr || state->geom_bytes < gl.total ||
	    state->image_bytes < il.total || R < -1 || (R > 0 && (state->binning == nullptr || state->binning_bytes < binning_bytes(R))) ||
	    (R == -1 && state->binning == nullptr))
		return BRS_ERR_STATE;
	if ((size_t)W * H > 0 && dL_dout_color == nullptr)
		return BRS_ERR_INVALID_ARG;
	const bool depth_grad = grads->depth_gradient != 0;
	if (depth_grad && (size_t)W * H > 0 && (dL_dout_depth == nullptr || grads->out_depth == nullptr))
		return BRS_ERR_INVALID_ARG;
	const bool debug = view->debug != 0;
	const uint32_t grid_x = (W + TILE_X - 1) / TILE_X, grid_y = (H + TILE_Y - 1) / TILE_Y;

	const char* geom = static_cast<const char*>(state->geom);
	const char* image = static_cast<const char*>(state->image);

	float* accum = static_cast<float*>(alloc(alloc_ctx, BRS_BUF_SCRATCH, brs_backward_scratch_bytes(P)));
	if (accum == nullptr)
		return BRS_ERR_ALLOC;
	BRS_CUDA(cudaMemsetAsync(accum, 0, sizeof(float) * ACCUM_STRIDE * (size_t)P, stream));

	if (R != 0 && grid_x * grid_y > 0) {
		BlendBwdArgs bb{};
		bb.ranges = reinterpret_cast<const uint2*>(image + il.ranges);
		bb.point_list = reinterpret_cast<const uint32_t*>(state->binning);
		bb.records = reinterpret_cast<const float4*>(geom + gl.records);
		bb.bg = view->bg;
		bb.W = W;
		bb.H = H;
		bb.grid_x = grid_x;
		bb.grid_y = grid_y;
		bb.final_T = reinterpret_cast<const float*>(image + il.final_T);
		bb.n_contrib = reinterpret_cast<const uint32_t*>(image + il.n_contrib);
		bb.dL_dpixels = dL_dout_color;
		bb.dL_ddepth = depth_grad ? dL_dout_depth : nullptr;
		bb.out_depth = depth_grad ? grads->out_depth : nullptr;
		bb.accum = accum;
		Companion comp;
		if (!debug && companion_for(stream, comp)) {
			BRS_CUDA(cudaEventRecord(comp.before, stream));
			BRS_CUDA(cudaStreamWaitEvent(comp.stream, comp.before, 0));
			BRS_CUDA(launch_blend_backward(bb, comp.stream));
			BRS_CUDA(cudaEventRecord(comp.after, comp.stream));
			BRS_CUDA(cudaStreamWaitEvent(stream, comp.after, 0));
		} else {
			BRS_STAGE(BRS_STAGE_BLEND_BWD, launch_blend_backward(bb, stream), debug, stream);
		}
	}

	PreprocessBwdArgs pb{};
	pb.P = P;
	pb.D = view->sh_degree;
	pb.M = M;
	pb.means3D = g->means3D;
	pb.radii = radii;
	pb.shs = g->shs;
	pb.scales = g->scales;
	pb.rotations = g->rotations;
	pb.scale_modifier = view->scale_modifier;
	pb.cov3D_precomp = g->cov3D_precomp;
	pb.viewmatrix = view->viewmatrix;
	pb.projmatrix = view->projmatrix;
	pb.campos = view->campos;
	pb.W = W;
	pb.H = H;
	pb.tan_fovx = view->tanfovx;
	pb.tan_fovy = view->tanfovy;
	pb.focal_y = H / (2.0f * view->tanfovy);
	pb.focal_x = W / (2.0f * view->tanfovx);
	pb.accum = accum;
	pb.accumulate = acc ? 1 : 0;
	pb.depth_gradient = depth_grad ? 1 : 0;
	{
		int dev = 0;
		Marks marks;
		pb.eager_sh = (cudaGetDevice(&dev) == cudaSuccess && lookup_marks(MarksKey{dev, P, W, H}, marks) &&
		               2ull * marks.V > (unsigned long long)P)
		                  ? 1
		                  : 0;
	}
	pb.dL_dmeans2D = grads->dL_dmeans2D;
	pb.dL_dcolors = grads->dL_dcolors;
	pb.dL_dopacity = grads->dL_dopacity;
	pb.dL_dmeans3D = grads->dL_dmeans3D;
	pb.dL_dcov3D = grads->dL_dcov3D;
	pb.dL_dsh = M > 0 ? grads->dL_dsh : nullptr;
	pb.dL_dscales = grads->dL_dscales;
	pb.dL_drotations = grads->dL_drotations;
	if (stats != nullptr) {
		pb.stats_grad_norm = stats->grad_norm;
		pb.stats_count = stats->count;
		pb.stats_index = stats->index;
		pb.stats_rows = stats->rows;
	}
	// (measured: moving this kernel to the companion stream as well is slightly slower)
	BRS_STAGE(BRS_STAGE_PREPROCESS_BWD, launch_preprocess_backward(pb, stream), debug, stream);
	return BRS_OK;
}

size_t brs_l1_ssim_blocks(int C, int H, int W) { return (C > 0 && H > 0 && W > 0) ? l1_ssim_blocks(C, H, W) : 0; }

int brs_l1_ssim_forward(const float* x, const float* y, int C, int H, int W, float* dmaps, float* partial, brs_stream stream)
{
	if (C < 0 || H < 0 || W < 0)
		return BRS_ERR_INVALID_ARG;
	if ((size_t)C * H * W == 0)
		return BRS_OK;
	if (x == nullptr || y == nullptr || dmaps == nullptr || partial == nullptr)
		return BRS_ERR_INVALID_ARG;
	BRS_CUDA(launch_l1_ssim_forward(x, y, C, H, W, dmaps, partial, stream));
	return BRS_OK;
}

int brs_l1_ssim_backward(const float* x, const float* y, const float* dmaps, int C, int H, int W, const float* dL_dloss,
                         float lambda_dssim, float* dL_dx, brs_stream stream)
{
	if (C < 0 || H < 0 || W < 0)
		return BRS_ERR_INVALID_ARG;
	if ((size_t)C * H * W == 0)
		return BRS_OK;
	if (x == nullptr || y == nullptr || dmaps == nullptr || dL_dloss == nullptr || dL_dx == nullptr)
		return BRS_ERR_INVALID_ARG;
	BRS_CUDA(launch_l1_ssim_backward(x, y, dmaps, C, H, W, dL_dloss, lambda_dssim, dL_dx, stream));
	return BRS_OK;
}

size_t brs_neural_scratch_bytes(int N) { return neural_scratch_bytes(N < 0 ? 0 : N); }

int brs_neural_gaussians_forward(const brs_neural_inputs* in, const brs_neural_outputs* out, void* scratch, brs_stream stream)
{
	if (in == nullptr || out == nullptr || in->N < 0 || in->K < 0 || out->count == nullptr || scratch == nullptr)
		return BRS_ERR_INVALID_ARG;
	if (in->K > 32)
		return BRS_ERR_UNSUPPORTED;
	const bool empty = (size_t)in->N * in->K == 0;
	if (!empty && (in->anchor == nullptr || in->grid_scaling == nullptr || in->offsets == nullptr || in->neural_opacity == nullptr ||
	               in->color == nullptr || in->scale_rot == nullptr || out->xyz == nullptr || out->color == nullptr ||
	               out->opacity == nullptr || out->scaling == nullptr || out->rot == nullptr || out->index == nullptr))
		return BRS_ERR_INVALID_ARG;
	NeuralFwdArgs a{};
	a.N = empty ? 0 : in->N;
	a.K = in->K;
	a.anchor = in->anchor;
	a.grid_scaling = in->grid_scaling;
	a.offsets = in->offsets;
	a.neural_opacity = in->neural_opacity;
	a.color = in->color;
	a.scale_rot = in->scale_rot;
	a.xyz = out->xyz;
	a.out_color = out->color;
	a.out_opacity = out->opacity;
	a.scaling = out->scaling;
	a.rot = out->rot;
	a.index = out->index;
	a.count = out->count;
	BRS_CUDA(launch_neural_forward(a, scratch, stream));
	return BRS_OK;
}

int brs_neural_gaussians_backward(const brs_neural_inputs* in, const int* index, const brs_neural_grads* g, brs_stream stream)
{
	if (in == nullptr || g == nullptr || in->N < 0 || in->K < 0)
		return BRS_ERR_INVALID_ARG;
	if (in->K > 32)
		return BRS_ERR_UNSUPPORTED;
	if ((size_t)in->N * in->K == 0)
		return BRS_OK;
	if (index == nullptr || in->grid_scaling == nullptr || in->offsets == nullptr || in->scale_rot == nullptr ||
	    g->d_anchor == nullptr || g->d_grid_scaling == nullptr || g->d_offsets == nullptr || g->d_neural_opacity == nullptr ||
	    g->d_color_in == nullptr || g->d_scale_rot == nullptr)
		return BRS_ERR_INVALID_ARG;
	NeuralBwdArgs a{};
	a.N = in->N;
	a.K = in->K;
	a.grid_scaling = in->grid_scaling;
	a.offsets = in->offsets;
	a.scale_rot = in->scale_rot;
	a.index = index;
	a.d_xyz = g->d_xyz;
	a.d_color = g->d_color;
	a.d_opacity = g->d_opacity;
	a.d_scaling = g->d_scaling;
	a.d_rot = g->d_rot;
	a.d_anchor = g->d_anchor;
	a.d_grid_scaling = g->d_grid_scaling;
	a.d_offsets = g->d_offsets;
	a.d_neural_opacity = g->d_neural_opacity;
	a.d_color_in = g->d_color_in;
	a.d_scale_rot = g->d_scale_rot;
	BRS_CUDA(launch_neural_backward(a, stream));
	return BRS_OK;
}

static int visible_filter_impl(const brs_view* view, int P, const float* means3D, const float* scales, int scales_stride,
                               const float* rotations, const float* cov3D_precomp, int* radii, long long* indices,
                               uint32_t* count, void* scratch, brs_stream stream)
{
	int st = validate_view(view, false);
	if (st != BRS_OK)
		return st;
	if (P < 0)
		return BRS_ERR_INVALID_ARG;
	if (P == 0) {
		if (count != nullptr)
			BRS_CUDA(cudaMemsetAsync(count, 0, sizeof(uint32_t), stream));
		return BRS_OK;
	}
	const bool has_sr = scales != nullptr && rotations != nullptr;
	if (means3D == nullptr || radii == nullptr || has_sr == (cov3D_precomp != nullptr) || (has_sr && scales_stride < 3))
		return BRS_ERR_INVALID_ARG;
	const int W = view->image_width, H = view->image_height;
	FilterArgs fa{};
	fa.P = P;
	fa.means3D = means3D;
	fa.scales = scales;
	fa.scales_stride = scales_stride;
	fa.scale_modifier = view->scale_modifier;
	fa.rotations = rotations;
	fa.cov3D_precomp = cov3D_precomp;
	fa.viewmatrix = view->viewmatrix;
	fa.projmatrix = view->projmatrix;
	fa.W = W;
	fa.H = H;
	fa.tan_fovx = view->tanfovx;
	fa.tan_fovy = view->tanfovy;
	fa.focal_y = H / (2.0f * view->tanfovy);
	fa.focal_x = W / (2.0f * view->tanfovx);
	fa.grid_x = (W + TILE_X - 1) / TILE_X;
	fa.grid_y = (H + TILE_Y - 1) / TILE_Y;
	fa.prefiltered = view->prefiltered;
	fa.radii = radii;
	if (indices != nullptr) {
		BRS_CUDA(cudaMemsetAsync(scratch, 0, brs_filter_scratch_bytes(P), stream));
		fa.indices = indices;
		fa.count = count;
		fa.ticket = static_cast<uint32_t*>(scratch);
		fa.status = fa.ticket + 64;
	}
	BRS_STAGE(BRS_STAGE_PREPROCESS, launch_filter(fa, stream), view->debug != 0, stream);
	return BRS_OK;
}

size_t brs_filter_scratch_bytes(int P) { return align_up(256 + sizeof(uint32_t) * (size_t)((P < 0 ? 0 : P) / 256 + 1), 256); }

int brs_visible_filter(const brs_view* view, int P, const float* means3D, const float* scales, int scales_stride,
                       const float* rotations, const float* cov3D_precomp, int* radii, brs_stream stream)
{
	return visible_filter_impl(view, P, means3D, scales, scales_stride, rotations, cov3D_precomp, radii, nullptr, nullptr, nullptr,
	                           stream);
}

int brs_visible_filter_compact(const brs_view* view, int P, const float* means3D, const float* scales, int scales_stride,
                               const float* rotations, const float* cov3D_precomp, int* radii, long long* indices,
                               uint32_t* count, void* scratch, brs_stream stream)
{
	if (indices == nullptr || count == nullptr || scratch == nullptr)
		return BRS_ERR_INVALID_ARG;
	return visible_filter_impl(view, P, means3D, scales, scales_stride, rotations, cov3D_precomp, radii, indices, count, scratch,
	                           stream);
}

int brs_mark_visible(int P, const float* means3D, const float* viewmatrix, const float* projmatrix, uint8_t* present,
                     brs_stream stream)
{
	(void)projmatrix; // reference in_frustum computes p_proj but only tests view-space z (auxiliary.h:154)
	if (P < 0)
		return BRS_ERR_INVALID_ARG;
	if (P == 0)
		return BRS_OK;
	if (means3D == nullptr || viewmatrix == nullptr || present == nullptr)
		return BRS_ERR_INVALID_ARG;
	BRS_CUDA(launch_check_frustum(P, means3D, viewmatrix, present, stream));
	return BRS_OK;
}

} // extern "C"

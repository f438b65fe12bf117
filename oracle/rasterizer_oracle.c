/*
 * rasterizer_oracle.c — CPU restatement of BloomScene's depth-diff-gaussian-rasterization.
 *
 * TEST INFRASTRUCTURE ONLY.  This file is the oracle, not the product: only tests/,
 * __graft_entry__.smoke() and bench.py's cpu_baseline / reference legs may build, load or call it.
 * The product path (bloomscene_b200/, libbloomrast.so) never does and has no CPU fallback.
 *
 * Parity status: the reference ships no tests, golden vectors or CPU implementation for this path
 * ("parity unpinned" by the reference itself).  This restatement is pinned instead against
 * outputs of the reference's OWN CUDA code (oracle/_ref, built from /root/reference) captured on a
 * B200: tests/golden/ (npz files) + tests/golden/make_golden.py.  Integer outputs agree except for rare
 * +-1 cases at ceil()/tile-edge boundaries, because the GPU build fuses multiply-adds (nvcc
 * -fmad=true) and uses its own expf, which plain C cannot reproduce bit for bit; floats agree to
 * ~1e-6.  The CUDA-vs-CUDA comparison on the GPU box is what defines bit-exactness.
 *
 * Every function cites the reference lines it follows (paths relative to
 * /root/reference/submodules/depth-diff-gaussian-rasterization/).  Plain C99 + optional OpenMP.
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#ifdef _OPENMP
#include <omp.h>
#endif

#define BLOCK_X 16 /* cuda_rasterizer/config.h:16-17 */
#define BLOCK_Y 16
#define NCH 3 /* config.h:15 */

/* cuda_rasterizer/auxiliary.h:22-39 */
static const float SH_C0 = 0.28209479177387814f;
static const float SH_C1 = 0.4886025119029199f;
static const float SH_C2[] = {1.0925484305920792f, -1.0925484305920792f, 0.31539156525252005f, -1.0925484305920792f,
                              0.5462742152960396f};
static const float SH_C3[] = {-0.5900435899266435f, 2.890611442640554f, -0.4570457994644658f, 0.3731763325901154f,
                              -0.4570457994644658f, 1.445305721320277f,  -0.5900435899266435f};

typedef struct { float x, y, z; } v3;
typedef struct { float m[3][3]; } m3; /* m[col][row], like glm::mat3 */

static v3 V3(float x, float y, float z) { v3 r = {x, y, z}; return r; }
static v3 v3_add(v3 a, v3 b) { return V3(a.x + b.x, a.y + b.y, a.z + b.z); }
static v3 v3_sub(v3 a, v3 b) { return V3(a.x - b.x, a.y - b.y, a.z - b.z); }
static v3 v3_scale(float s, v3 a) { return V3(s * a.x, s * a.y, s * a.z); }
static float v3_dot(v3 a, v3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }

/* glm mat3 * mat3: R[c][r] = A[0][r]*B[c][0] + A[1][r]*B[c][1] + A[2][r]*B[c][2] */
static m3 m3_mul(m3 a, m3 b)
{
	m3 r;
	for (int c = 0; c < 3; c++)
		for (int k = 0; k < 3; k++)
			r.m[c][k] = a.m[0][k] * b.m[c][0] + a.m[1][k] * b.m[c][1] + a.m[2][k] * b.m[c][2];
	return r;
}
static m3 m3_transpose(m3 a)
{
	m3 r;
	for (int c = 0; c < 3; c++)
		for (int k = 0; k < 3; k++)
			r.m[c][k] = a.m[k][c];
	return r;
}
static m3 m3_cols(float x0, float y0, float z0, float x1, float y1, float z1, float x2, float y2, float z2)
{
	m3 r = {{{x0, y0, z0}, {x1, y1, z1}, {x2, y2, z2}}};
	return r;
}

/* auxiliary.h:41-44 — double arithmetic (the literals are doubles) */
static float ndc2Pix(float v, int S) { return (float)(((v + 1.0) * S - 1.0) * 0.5); }

static int imin(int a, int b) { return a < b ? a : b; }
static int imax(int a, int b) { return a > b ? a : b; }

/* auxiliary.h:46-56 */
static void getRect(float px, float py, int max_radius, int gx, int gy, int* x0, int* y0, int* x1, int* y1)
{
	*x0 = imin(gx, imax(0, (int)((px - max_radius) / BLOCK_X)));
	*y0 = imin(gy, imax(0, (int)((py - max_radius) / BLOCK_Y)));
	*x1 = imin(gx, imax(0, (int)((px + max_radius + BLOCK_X - 1) / BLOCK_X)));
	*y1 = imin(gy, imax(0, (int)((py + max_radius + BLOCK_Y - 1) / BLOCK_Y)));
}

/* auxiliary.h:58-77 */
static v3 transformPoint4x3(v3 p, const float* m)
{
	return V3(m[0] * p.x + m[4] * p.y + m[8] * p.z + m[12], m[1] * p.x + m[5] * p.y + m[9] * p.z + m[13],
	          m[2] * p.x + m[6] * p.y + m[10] * p.z + m[14]);
}
static void transformPoint4x4(v3 p, const float* m, float out[4])
{
	out[0] = m[0] * p.x + m[4] * p.y + m[8] * p.z + m[12];
	out[1] = m[1] * p.x + m[5] * p.y + m[9] * p.z + m[13];
	out[2] = m[2] * p.x + m[6] * p.y + m[10] * p.z + m[14];
	out[3] = m[3] * p.x + m[7] * p.y + m[11] * p.z + m[15];
}
/* auxiliary.h:89-97 */
static v3 transformVec4x3Transpose(v3 p, const float* m)
{
	return V3(m[0] * p.x + m[1] * p.y + m[2] * p.z, m[4] * p.x + m[5] * p.y + m[6] * p.z,
	          m[8] * p.x + m[9] * p.y + m[10] * p.z);
}
/* auxiliary.h:107-117 */
static v3 dnormvdv(v3 v, v3 dv)
{
	float sum2 = v.x * v.x + v.y * v.y + v.z * v.z;
	float invsum32 = 1.0f / sqrtf(sum2 * sum2 * sum2);
	v3 r;
	r.x = ((+sum2 - v.x * v.x) * dv.x - v.y * v.x * dv.y - v.z * v.x * dv.z) * invsum32;
	r.y = (-v.x * v.y * dv.x + (sum2 - v.y * v.y) * dv.y - v.z * v.y * dv.z) * invsum32;
	r.z = (-v.x * v.z * dv.x - v.y * v.z * dv.y + (sum2 - v.z * v.z) * dv.z) * invsum32;
	return r;
}

/* ---- context ---------------------------------------------------------------------------------- */

typedef struct orc_ctx {
	int P, W, H, D, M, R, gx, gy;
	float tanfovx, tanfovy, focal_x, focal_y, scale_modifier;
	float bg[3], view[16], proj[16], campos[3];
	/* inputs (borrowed) */
	const float *means3D, *opacities, *shs, *colors_precomp, *scales, *rotations, *cov3D_precomp;
	/* geometry state (rasterizer_impl.h:29-45) */
	float* depths;
	uint8_t* clamped;
	int* radii;
	float* means2D;
	float* cov3D;
	float* conic_opacity;
	float* rgb;
	uint32_t* tiles_touched;
	uint32_t* point_offsets;
	/* binning state (rasterizer_impl.h:55-64) */
	uint64_t *keys_unsorted, *keys;
	uint32_t *values_unsorted, *values;
	/* image state (rasterizer_impl.h:47-53) */
	uint32_t* ranges; /* [tiles][2] */
	float* final_T;
	uint32_t* n_contrib;
	float *acc_final, *D_final; /* per pixel: the forward's accumulated weight and un-normalised depth (opt-in depth gradient) */
	long long pairs_evaluated, pairs_contributing; /* E and C of SURVEY.md §8(d) */
} orc_ctx;

orc_ctx* orc_create(void) { return (orc_ctx*)calloc(1, sizeof(orc_ctx)); }

static void free_state(orc_ctx* c)
{
	free(c->depths); free(c->clamped); free(c->radii); free(c->means2D); free(c->cov3D); free(c->conic_opacity);
	free(c->rgb); free(c->tiles_touched); free(c->point_offsets); free(c->keys_unsorted); free(c->keys);
	free(c->values_unsorted); free(c->values); free(c->ranges); free(c->final_T); free(c->n_contrib); free(c->acc_final); free(c->D_final);
	c->depths = NULL; c->clamped = NULL; c->radii = NULL; c->means2D = NULL; c->cov3D = NULL; c->conic_opacity = NULL;
	c->rgb = NULL; c->tiles_touched = NULL; c->point_offsets = NULL; c->keys_unsorted = NULL; c->keys = NULL;
	c->values_unsorted = NULL; c->values = NULL; c->ranges = NULL; c->final_T = NULL; c->n_contrib = NULL; c->acc_final = NULL; c->D_final = NULL;
}

void orc_destroy(orc_ctx* c)
{
	if (!c) return;
	free_state(c);
	free(c);
}

void orc_set_threads(int n)
{
#ifdef _OPENMP
	if (n > 0) omp_set_num_threads(n);
#else
	(void)n;
#endif
}
int orc_max_threads(void)
{
#ifdef _OPENMP
	return omp_get_max_threads();
#else
	return 1;
#endif
}

/* state getters for ctypes */
int orc_num_rendered(const orc_ctx* c) { return c->R; }
long long orc_pairs_evaluated(const orc_ctx* c) { return c->pairs_evaluated; }
long long orc_pairs_contributing(const orc_ctx* c) { return c->pairs_contributing; }
const float* orc_depths(const orc_ctx* c) { return c->depths; }
const float* orc_means2D(const orc_ctx* c) { return c->means2D; }
const float* orc_cov3D(const orc_ctx* c) { return c->cov3D; }
const float* orc_conic_opacity(const orc_ctx* c) { return c->conic_opacity; }
const float* orc_rgb(const orc_ctx* c) { return c->rgb; }
const uint8_t* orc_clamped(const orc_ctx* c) { return c->clamped; }
const uint32_t* orc_tiles_touched(const orc_ctx* c) { return c->tiles_touched; }
const uint32_t* orc_point_offsets(const orc_ctx* c) { return c->point_offsets; }
const uint64_t* orc_keys_unsorted(const orc_ctx* c) { return c->keys_unsorted; }
const uint64_t* orc_keys(const orc_ctx* c) { return c->keys; }
const uint32_t* orc_point_list(const orc_ctx* c) { return c->values; }
const uint32_t* orc_ranges(const orc_ctx* c) { return c->ranges; }
const float* orc_final_T(const orc_ctx* c) { return c->final_T; }
const uint32_t* orc_n_contrib(const orc_ctx* c) { return c->n_contrib; }

/* ---- forward pieces --------------------------------------------------------------------------- */

/* forward.cu:118-152 (no quaternion normalisation, :127) */
static void computeCov3D(v3 scale, float mod, const float* rot, float* cov3D)
{
	m3 S = m3_cols(1, 0, 0, 0, 1, 0, 0, 0, 1);
	S.m[0][0] = mod * scale.x;
	S.m[1][1] = mod * scale.y;
	S.m[2][2] = mod * scale.z;
	float r = rot[0], x = rot[1], y = rot[2], z = rot[3];
	m3 R = m3_cols(1.f - 2.f * (y * y + z * z), 2.f * (x * y - r * z), 2.f * (x * z + r * y),
	               2.f * (x * y + r * z), 1.f - 2.f * (x * x + z * z), 2.f * (y * z - r * x),
	               2.f * (x * z - r * y), 2.f * (y * z + r * x), 1.f - 2.f * (x * x + y * y));
	m3 M = m3_mul(S, R);
	m3 Sigma = m3_mul(m3_transpose(M), M);
	cov3D[0] = Sigma.m[0][0];
	cov3D[1] = Sigma.m[0][1];
	cov3D[2] = Sigma.m[0][2];
	cov3D[3] = Sigma.m[1][1];
	cov3D[4] = Sigma.m[1][2];
	cov3D[5] = Sigma.m[2][2];
}

/* shared by forward.cu:74-113 and backward.cu:164-194: t (clamped), J, W, T, Vrk, cov2D */
typedef struct { v3 t; float txtz, tytz, limx, limy; m3 J, Wm, T, Vrk, cov; } cov2d_parts;
static void cov2d_common(v3 mean, float fx, float fy, float tan_fovx, float tan_fovy, const float* cov3D,
                         const float* view, cov2d_parts* o)
{
	v3 t = transformPoint4x3(mean, view);
	o->limx = 1.3f * tan_fovx;
	o->limy = 1.3f * tan_fovy;
	o->txtz = t.x / t.z;
	o->tytz = t.y / t.z;
	t.x = fminf(o->limx, fmaxf(-o->limx, o->txtz)) * t.z;
	t.y = fminf(o->limy, fmaxf(-o->limy, o->tytz)) * t.z;
	o->t = t;
	o->J = m3_cols(fx / t.z, 0.0f, -(fx * t.x) / (t.z * t.z), 0.0f, fy / t.z, -(fy * t.y) / (t.z * t.z), 0, 0, 0);
	o->Wm = m3_cols(view[0], view[4], view[8], view[1], view[5], view[9], view[2], view[6], view[10]);
	o->T = m3_mul(o->Wm, o->J);
	o->Vrk = m3_cols(cov3D[0], cov3D[1], cov3D[2], cov3D[1], cov3D[3], cov3D[4], cov3D[2], cov3D[4], cov3D[5]);
	o->cov = m3_mul(m3_mul(m3_transpose(o->T), m3_transpose(o->Vrk)), o->T);
}

/* forward.cu:20-71 */
static v3 computeColorFromSH_fwd(int deg, int M, v3 pos, v3 campos, const float* shs_row, uint8_t* clamped)
{
	(void)M;
	v3 dir = v3_sub(pos, campos);
	float len = sqrtf(v3_dot(dir, dir));
	dir = V3(dir.x / len, dir.y / len, dir.z / len);
#define SH(k) V3(shs_row[3 * (k)], shs_row[3 * (k) + 1], shs_row[3 * (k) + 2])
	v3 result = v3_scale(SH_C0, SH(0));
	if (deg > 0) {
		float x = dir.x, y = dir.y, z = dir.z;
		result = v3_sub(v3_add(v3_sub(result, v3_scale(SH_C1 * y, SH(1))), v3_scale(SH_C1 * z, SH(2))),
		                v3_scale(SH_C1 * x, SH(3)));
		if (deg > 1) {
			float xx = x * x, yy = y * y, zz = z * z, xy = x * y, yz = y * z, xz = x * z;
			result = v3_add(result, v3_scale(SH_C2[0] * xy, SH(4)));
			result = v3_add(result, v3_scale(SH_C2[1] * yz, SH(5)));
			result = v3_add(result, v3_scale(SH_C2[2] * (2.0f * zz - xx - yy), SH(6)));
			result = v3_add(result, v3_scale(SH_C2[3] * xz, SH(7)));
			result = v3_add(result, v3_scale(SH_C2[4] * (xx - yy), SH(8)));
			if (deg > 2) {
				result = v3_add(result, v3_scale(SH_C3[0] * y * (3.0f * xx - yy), SH(9)));
				result = v3_add(result, v3_scale(SH_C3[1] * xy * z, SH(10)));
				result = v3_add(result, v3_scale(SH_C3[2] * y * (4.0f * zz - xx - yy), SH(11)));
				result = v3_add(result, v3_scale(SH_C3[3] * z * (2.0f * zz - 3.0f * xx - 3.0f * yy), SH(12)));
				result = v3_add(result, v3_scale(SH_C3[4] * x * (4.0f * zz - xx - yy), SH(13)));
				result = v3_add(result, v3_scale(SH_C3[5] * z * (xx - yy), SH(14)));
				result = v3_add(result, v3_scale(SH_C3[6] * x * (xx - 3.0f * yy), SH(15)));
			}
		}
	}
#undef SH
	result.x += 0.5f;
	result.y += 0.5f;
	result.z += 0.5f;
	clamped[0] = result.x < 0;
	clamped[1] = result.y < 0;
	clamped[2] = result.z < 0;
	return V3(fmaxf(result.x, 0.0f), fmaxf(result.y, 0.0f), fmaxf(result.z, 0.0f));
}

/* Geometry part of preprocessCUDA (forward.cu:186-237); returns 0 where the reference returns early.
 * Also used for filter_preprocessCUDA (forward.cu:260-335). */
static int preprocess_geometry(const orc_ctx* c, int idx, const float* scales, int scales_stride, float* cov3D_out,
                               float* depth, float* px, float* py, float conic[3], int* radius, int rect[4])
{
	v3 p = V3(c->means3D[3 * idx], c->means3D[3 * idx + 1], c->means3D[3 * idx + 2]);
	v3 p_view = transformPoint4x3(p, c->view); /* in_frustum, auxiliary.h:139-164 */
	if (p_view.z <= 0.2f) return 0;
	float hom[4];
	transformPoint4x4(p, c->proj, hom);
	float p_w = 1.0f / (hom[3] + 0.0000001f);
	float projx = hom[0] * p_w, projy = hom[1] * p_w;

	float cov3D[6];
	if (c->cov3D_precomp) {
		memcpy(cov3D, c->cov3D_precomp + 6 * (size_t)idx, sizeof(cov3D));
	} else {
		const float* s = scales + (size_t)idx * scales_stride;
		computeCov3D(V3(s[0], s[1], s[2]), c->scale_modifier, c->rotations + 4 * (size_t)idx, cov3D);
	}
	if (cov3D_out) memcpy(cov3D_out, cov3D, sizeof(cov3D));

	cov2d_parts cp;
	cov2d_common(p, c->focal_x, c->focal_y, c->tanfovx, c->tanfovy, cov3D, c->view, &cp);
	float cx = cp.cov.m[0][0] + 0.3f, cy = cp.cov.m[0][1], cz = cp.cov.m[1][1] + 0.3f;

	float det = (cx * cz - cy * cy);
	if (det == 0.0f) return 0;
	float det_inv = 1.f / det;
	conic[0] = cz * det_inv;
	conic[1] = -cy * det_inv;
	conic[2] = cx * det_inv;

	float mid = 0.5f * (cx + cz);
	float lambda1 = mid + sqrtf(fmaxf(0.1f, mid * mid - det));
	float lambda2 = mid - sqrtf(fmaxf(0.1f, mid * mid - det));
	float my_radius = ceilf(3.f * sqrtf(fmaxf(lambda1, lambda2)));
	*px = ndc2Pix(projx, c->W);
	*py = ndc2Pix(projy, c->H);
	getRect(*px, *py, (int)my_radius, c->gx, c->gy, &rect[0], &rect[1], &rect[2], &rect[3]);
	if ((rect[2] - rect[0]) * (rect[3] - rect[1]) == 0) return 0;
	*depth = p_view.z;
	*radius = (int)my_radius;
	return 1;
}

/* rasterizer_impl.cu:35-50 */
static uint32_t getHigherMsb(uint32_t n)
{
	uint32_t msb = sizeof(n) * 4;
	uint32_t step = msb;
	while (step > 1) {
		step /= 2;
		if (n >> msb) msb += step;
		else msb -= step;
	}
	if (n >> msb) msb++;
	return msb;
}

/* Stable LSD radix sort on key bits [0, nbits) — what cub::DeviceRadixSort::SortPairs
 * (rasterizer_impl.cu:304-309) guarantees: ascending, stable. */
static void radix_sort_pairs(uint64_t* keys, uint32_t* vals, uint64_t* keys_tmp, uint32_t* vals_tmp, size_t n, int nbits)
{
	const int RB = 11;
	const size_t NB = (size_t)1 << RB;
	size_t* count = (size_t*)malloc(sizeof(size_t) * NB);
	uint64_t *ks = keys, *kd = keys_tmp;
	uint32_t *vs = vals, *vd = vals_tmp;
	int swapped = 0;
	for (int shift = 0; shift < nbits; shift += RB) {
		memset(count, 0, sizeof(size_t) * NB);
		for (size_t i = 0; i < n; i++) count[(ks[i] >> shift) & (NB - 1)]++;
		size_t run = 0;
		for (size_t b = 0; b < NB; b++) { size_t cnt = count[b]; count[b] = run; run += cnt; }
		for (size_t i = 0; i < n; i++) {
			size_t d = count[(ks[i] >> shift) & (NB - 1)]++;
			kd[d] = ks[i];
			vd[d] = vs[i];
		}
		uint64_t* tk = ks; ks = kd; kd = tk;
		uint32_t* tv = vs; vs = vd; vd = tv;
		swapped ^= 1;
	}
	if (swapped) {
		memcpy(keys, ks, sizeof(uint64_t) * n);
		memcpy(vals, vs, sizeof(uint32_t) * n);
	}
	free(count);
}

/* renderCUDA forward for one pixel (forward.cu:341-471): same loop, tests and accumulation order. */
static void render_pixel(const orc_ctx* c, int px, int py, uint32_t start, uint32_t end, const float* features,
                         float* out_color, float* out_depth, long long* evaluated, long long* contributing)
{
	const int W = c->W, H = c->H;
	const uint32_t pix_id = (uint32_t)W * py + px;
	const float pixfx = (float)px, pixfy = (float)py;
	float T = 1.0f;
	uint32_t contributor = 0, last_contributor = 0;
	float C[NCH] = {0, 0, 0};
	float D = 0, acc = 0.000001f;
	long long ev = 0, co = 0;
	for (uint32_t k = start; k < end; k++) {
		contributor++;
		ev++;
		const uint32_t id = c->values[k];
		const float dx = c->means2D[2 * id] - pixfx, dy = c->means2D[2 * id + 1] - pixfy;
		const float* con_o = c->conic_opacity + 4 * (size_t)id;
		const float power = -0.5f * (con_o[0] * dx * dx + con_o[2] * dy * dy) - con_o[1] * dx * dy;
		if (power > 0.0f) continue;
		const float alpha = fminf(0.99f, con_o[3] * expf(power));
		if (alpha < 1.0f / 255.0f) continue;
		const float test_T = T * (1 - alpha);
		if (test_T < 0.0001f) break; /* done = true: the thread stops evaluating (forward.cu:409,431-435) */
		for (int ch = 0; ch < NCH; ch++) C[ch] += features[id * NCH + ch] * alpha * T;
		D += c->depths[id] * alpha * T;
		acc += alpha * T;
		T = test_T;
		last_contributor = contributor;
		co++;
	}
	c->final_T[pix_id] = T;
	c->n_contrib[pix_id] = last_contributor;
	c->acc_final[pix_id] = acc;
	c->D_final[pix_id] = D;
	for (int ch = 0; ch < NCH; ch++) out_color[(size_t)ch * H * W + pix_id] = C[ch] + T * c->bg[ch];
	out_depth[pix_id] = (acc > 0.5f) ? D / acc : 0.0f; /* forward.cu:464-468 */
	*evaluated += ev;
	*contributing += co;
}

typedef struct orc_inputs {
	int P, D, M, W, H;
	float tanfovx, tanfovy, scale_modifier;
	const float *bg, *viewmatrix, *projmatrix, *campos;
	const float *means3D, *opacities, *shs, *colors_precomp, *scales, *rotations, *cov3D_precomp;
} orc_inputs;

static void bind_inputs(orc_ctx* c, const orc_inputs* in)
{
	c->P = in->P; c->D = in->D; c->M = in->M; c->W = in->W; c->H = in->H;
	c->tanfovx = in->tanfovx; c->tanfovy = in->tanfovy; c->scale_modifier = in->scale_modifier;
	c->focal_y = in->H / (2.0f * in->tanfovy); /* rasterizer_impl.cu:223-224 */
	c->focal_x = in->W / (2.0f * in->tanfovx);
	c->gx = (in->W + BLOCK_X - 1) / BLOCK_X;
	c->gy = (in->H + BLOCK_Y - 1) / BLOCK_Y;
	if (in->bg) memcpy(c->bg, in->bg, sizeof(c->bg));
	memcpy(c->view, in->viewmatrix, sizeof(c->view));
	memcpy(c->proj, in->projmatrix, sizeof(c->proj));
	if (in->campos) memcpy(c->campos, in->campos, sizeof(c->campos));
	c->means3D = in->means3D; c->opacities = in->opacities; c->shs = in->shs; c->colors_precomp = in->colors_precomp;
	c->scales = in->scales; c->rotations = in->rotations; c->cov3D_precomp = in->cov3D_precomp;
}

/* Rasterizer::forward (rasterizer_impl.cu:198-339). out_color [3,H,W], out_depth [H,W], radii [P]. */
int orc_forward(orc_ctx* c, const orc_inputs* in, float* out_color, float* out_depth, int* radii_out)
{
	free_state(c);
	bind_inputs(c, in);
	const int P = c->P, W = c->W, H = c->H;
	const size_t npix = (size_t)W * H;
	c->R = 0;
	c->pairs_evaluated = c->pairs_contributing = 0;
	memset(out_color, 0, sizeof(float) * NCH * npix); /* rasterize_points.cu:68-70 */
	memset(out_depth, 0, sizeof(float) * npix);
	if (P == 0) return 0; /* rasterize_points.cu:82 */

	c->depths = (float*)calloc(P, sizeof(float));
	c->clamped = (uint8_t*)calloc((size_t)3 * P, 1);
	c->radii = (int*)calloc(P, sizeof(int));
	c->means2D = (float*)calloc((size_t)2 * P, sizeof(float));
	c->cov3D = (float*)calloc((size_t)6 * P, sizeof(float));
	c->conic_opacity = (float*)calloc((size_t)4 * P, sizeof(float));
	c->rgb = (float*)calloc((size_t)3 * P, sizeof(float));
	c->tiles_touched = (uint32_t*)calloc(P, sizeof(uint32_t));
	c->point_offsets = (uint32_t*)calloc(P, sizeof(uint32_t));

	/* preprocessCUDA (forward.cu:155-256) */
#pragma omp parallel for schedule(static)
	for (int idx = 0; idx < P; idx++) {
		float depth, px, py, conic[3];
		int radius, rect[4];
		if (!preprocess_geometry(c, idx, c->scales, 3, c->cov3D + 6 * (size_t)idx, &depth, &px, &py, conic, &radius, rect))
			continue;
		if (c->colors_precomp == NULL) {
			v3 p = V3(c->means3D[3 * idx], c->means3D[3 * idx + 1], c->means3D[3 * idx + 2]);
			v3 col = computeColorFromSH_fwd(c->D, c->M, p, V3(c->campos[0], c->campos[1], c->campos[2]),
			                                c->shs + (size_t)idx * c->M * 3, c->clamped + 3 * (size_t)idx);
			c->rgb[3 * idx] = col.x;
			c->rgb[3 * idx + 1] = col.y;
			c->rgb[3 * idx + 2] = col.z;
		}
		c->depths[idx] = depth;
		c->radii[idx] = radius;
		c->means2D[2 * idx] = px;
		c->means2D[2 * idx + 1] = py;
		c->conic_opacity[4 * idx] = conic[0];
		c->conic_opacity[4 * idx + 1] = conic[1];
		c->conic_opacity[4 * idx + 2] = conic[2];
		c->conic_opacity[4 * idx + 3] = c->opacities[idx];
		c->tiles_touched[idx] = (uint32_t)((rect[3] - rect[1]) * (rect[2] - rect[0]));
	}
	if (radii_out) memcpy(radii_out, c->radii, sizeof(int) * P);

	/* InclusiveSum (rasterizer_impl.cu:278) */
	uint32_t run = 0;
	for (int i = 0; i < P; i++) { run += c->tiles_touched[i]; c->point_offsets[i] = run; }
	const uint32_t R = run;
	c->R = (int)R;

	c->keys_unsorted = (uint64_t*)malloc(sizeof(uint64_t) * (R ? R : 1));
	c->keys = (uint64_t*)malloc(sizeof(uint64_t) * (R ? R : 1));
	c->values_unsorted = (uint32_t*)malloc(sizeof(uint32_t) * (R ? R : 1));
	c->values = (uint32_t*)malloc(sizeof(uint32_t) * (R ? R : 1));

	/* duplicateWithKeys (rasterizer_impl.cu:70-111) */
#pragma omp parallel for schedule(dynamic, 1024)
	for (int idx = 0; idx < P; idx++) {
		if (c->radii[idx] > 0) {
			uint32_t off = (idx == 0) ? 0 : c->point_offsets[idx - 1];
			int rect[4];
			getRect(c->means2D[2 * idx], c->means2D[2 * idx + 1], c->radii[idx], c->gx, c->gy, &rect[0], &rect[1], &rect[2], &rect[3]);
			uint32_t dbits;
			memcpy(&dbits, &c->depths[idx], 4);
			for (int y = rect[1]; y < rect[3]; y++)
				for (int x = rect[0]; x < rect[2]; x++) {
					uint64_t key = (uint64_t)(y * c->gx + x);
					key <<= 32;
					key |= dbits;
					c->keys_unsorted[off] = key;
					c->values_unsorted[off] = (uint32_t)idx;
					off++;
				}
		}
	}

	/* SortPairs on bits [0, 32 + getHigherMsb(#tiles)) (rasterizer_impl.cu:301-309) */
	memcpy(c->keys, c->keys_unsorted, sizeof(uint64_t) * R);
	memcpy(c->values, c->values_unsorted, sizeof(uint32_t) * R);
	{
		uint64_t* kt = (uint64_t*)malloc(sizeof(uint64_t) * (R ? R : 1));
		uint32_t* vt = (uint32_t*)malloc(sizeof(uint32_t) * (R ? R : 1));
		radix_sort_pairs(c->keys, c->values, kt, vt, R, 32 + (int)getHigherMsb((uint32_t)(c->gx * c->gy)));
		free(kt);
		free(vt);
	}

	/* identifyTileRanges after memset (rasterizer_impl.cu:311-319,116-138) */
	const size_t ntiles = (size_t)c->gx * c->gy;
	c->ranges = (uint32_t*)calloc(2 * (ntiles ? ntiles : 1), sizeof(uint32_t));
	for (uint32_t i = 0; i < R; i++) {
		uint32_t cur = (uint32_t)(c->keys[i] >> 32);
		if (i == 0) c->ranges[2 * cur] = 0;
		else {
			uint32_t prev = (uint32_t)(c->keys[i - 1] >> 32);
			if (cur != prev) { c->ranges[2 * prev + 1] = i; c->ranges[2 * cur] = i; }
		}
		if (i == R - 1) c->ranges[2 * cur + 1] = R;
	}

	/* renderCUDA (forward.cu:341-471) */
	c->final_T = (float*)calloc(npix ? npix : 1, sizeof(float));
	c->n_contrib = (uint32_t*)calloc(npix ? npix : 1, sizeof(uint32_t));
	c->acc_final = (float*)calloc(npix ? npix : 1, sizeof(float));
	c->D_final = (float*)calloc(npix ? npix : 1, sizeof(float));
	const float* features = c->colors_precomp ? c->colors_precomp : c->rgb; /* rasterizer_impl.cu:322 */
	long long ev_total = 0, co_total = 0;
#pragma omp parallel for schedule(dynamic, 1) reduction(+ : ev_total, co_total)
	for (int tile = 0; tile < (int)ntiles; tile++) {
		const int tx = tile % c->gx, ty = tile / c->gx;
		const uint32_t start = c->ranges[2 * tile], end = c->ranges[2 * tile + 1];
		long long ev = 0, co = 0;
		for (int ly = 0; ly < BLOCK_Y; ly++)
			for (int lx = 0; lx < BLOCK_X; lx++) {
				const int px = tx * BLOCK_X + lx, py = ty * BLOCK_Y + ly;
				if (px < W && py < H) render_pixel(c, px, py, start, end, features, out_color, out_depth, &ev, &co);
			}
		ev_total += ev;
		co_total += co;
	}
	c->pairs_evaluated = ev_total;
	c->pairs_contributing = co_total;
	return (int)R;
}

/* Rasterizer::visible_filter (rasterizer_impl.cu:342-398, forward.cu:260-335) */
int orc_visible_filter(const orc_inputs* in, int scales_stride, int* radii)
{
	orc_ctx* c = orc_create();
	bind_inputs(c, in);
#pragma omp parallel for schedule(static)
	for (int idx = 0; idx < c->P; idx++) {
		float depth, px, py, conic[3];
		int radius, rect[4];
		radii[idx] = preprocess_geometry(c, idx, c->scales, scales_stride, NULL, &depth, &px, &py, conic, &radius, rect) ? radius : 0;
	}
	orc_destroy(c);
	return 0;
}

/* Rasterizer::markVisible (rasterizer_impl.cu:141-153,54-66) */
int orc_mark_visible(int P, const float* means3D, const float* viewmatrix, uint8_t* present)
{
	for (int idx = 0; idx < P; idx++) {
		v3 p = V3(means3D[3 * idx], means3D[3 * idx + 1], means3D[3 * idx + 2]);
		present[idx] = transformPoint4x3(p, viewmatrix).z <= 0.2f ? 0 : 1;
	}
	return 0;
}

/* ---- backward ---------------------------------------------------------------------------------- */

/* Diagnostic (tests only): with orc_set_f64_sums(1) the per-Gaussian sums of the blend backward — the same fp32
 * per-pixel terms — are accumulated in DOUBLE and rounded to float once, before the per-Gaussian stage consumes them.
 * This separates summation error (the reference adds up to W*H float terms into one float with atomicAdd,
 * backward.cu:556-575) from arithmetic differences when two implementations disagree on a gradient.  Default off. */
static int g_f64_sums = 0;
void orc_set_f64_sums(int enable) { g_f64_sums = enable != 0; }
typedef struct sum64 { /* shadows of the float accumulators, NULL when the diagnostic is off */
	double *mean2D, *conic, *opacity, *colors, *z;
} sum64;
static void acc_add(float* f, double* d, size_t i, float v)
{
	if (d) {
#pragma omp atomic
		d[i] += (double)v;
	} else {
#pragma omp atomic
		f[i] += v;
	}
}

/* renderCUDA backward for one pixel (backward.cu:399-586). dL_dconic is [P][4] (x, y, -, w). */
/* With dL_ddepths != NULL (EXTENSION, default off: the reference has every depth line commented out,
 * backward.cu:443-554) the depth image also carries gradient.  The forward's depth is D/acc with
 * D = sum T alpha z, acc = 1e-6 + sum T alpha, gated by acc > 0.5 (forward.cu:464-468), so D and acc
 * enter the recurrence as two more blended channels (per-Gaussian values z and 1, no background term)
 * with pixel gradients gD = g/acc and gA = -g D/acc^2, exactly like the dead code treats its depth
 * channel (accum_depth_rec / last_depth), and z collects dL_dz = sum alpha T gD. */
static void render_pixel_backward(const orc_ctx* c, int px, int py, uint32_t start, uint32_t end, const float* colors,
                                  const float* dL_dpixels, const float* dL_ddepths, float* dL_dmean2D, float* dL_dconic,
                                  float* dL_dopacity, float* dL_dcolors, float* dL_dz, const sum64* s64)
{
	const int W = c->W, H = c->H;
	const uint32_t pix_id = (uint32_t)W * py + px;
	const float pixfx = (float)px, pixfy = (float)py;
	const float T_final = c->final_T[pix_id];
	float T = T_final;
	uint32_t contributor = end - start;
	const uint32_t last_contributor = c->n_contrib[pix_id];
	float accum_rec[NCH] = {0, 0, 0}, dL_dpixel[NCH], last_color[NCH] = {0, 0, 0};
	for (int i = 0; i < NCH; i++) dL_dpixel[i] = dL_dpixels[(size_t)i * H * W + pix_id];
	float last_alpha = 0;
	float gD = 0, gA = 0, accum_depth_rec = 0, last_depth = 0, accum_one_rec = 0, last_one = 0;
	if (dL_ddepths) {
		const float acc = c->acc_final[pix_id];
		if (acc > 0.5f) {
			gD = dL_ddepths[pix_id] / acc;
			gA = -dL_ddepths[pix_id] * c->D_final[pix_id] / (acc * acc);
		}
	}
	const float ddelx_dx = (float)(0.5 * W), ddely_dy = (float)(0.5 * H); /* backward.cu:473-474 (double) */

	for (uint32_t k = end; k-- > start;) {
		contributor--;
		if (contributor >= last_contributor) continue;
		const uint32_t id = c->values[k];
		const float dx = c->means2D[2 * id] - pixfx, dy = c->means2D[2 * id + 1] - pixfy;
		const float* con_o = c->conic_opacity + 4 * (size_t)id;
		const float power = -0.5f * (con_o[0] * dx * dx + con_o[2] * dy * dy) - con_o[1] * dx * dy;
		if (power > 0.0f) continue;
		const float G = expf(power);
		const float alpha = fminf(0.99f, con_o[3] * G);
		if (alpha < 1.0f / 255.0f) continue;

		T = T / (1.f - alpha);
		const float dchannel_dcolor = alpha * T;
		float dL_dalpha = 0.0f;
		for (int ch = 0; ch < NCH; ch++) {
			const float col = colors[id * NCH + ch];
			accum_rec[ch] = last_alpha * last_color[ch] + (1.f - last_alpha) * accum_rec[ch];
			last_color[ch] = col;
			const float dL_dchannel = dL_dpixel[ch];
			dL_dalpha += (col - accum_rec[ch]) * dL_dchannel;
			acc_add(dL_dcolors, s64->colors, (size_t)id * NCH + ch, dchannel_dcolor * dL_dchannel);
		}
		if (dL_ddepths) {
			const float c_d = c->depths[id];
			accum_depth_rec = last_alpha * last_depth + (1.f - last_alpha) * accum_depth_rec;
			last_depth = c_d;
			dL_dalpha += (c_d - accum_depth_rec) * gD;
			accum_one_rec = last_alpha * last_one + (1.f - last_alpha) * accum_one_rec;
			last_one = 1.f;
			dL_dalpha += (1.f - accum_one_rec) * gA;
			acc_add(dL_dz, s64->z, id, dchannel_dcolor * gD);
		}
		dL_dalpha *= T;
		last_alpha = alpha;
		float bg_dot_dpixel = 0;
		for (int i = 0; i < NCH; i++) bg_dot_dpixel += c->bg[i] * dL_dpixel[i];
		dL_dalpha += (-T_final / (1.f - alpha)) * bg_dot_dpixel;

		const float dL_dG = con_o[3] * dL_dalpha;
		const float gdx = G * dx, gdy = G * dy;
		const float dG_ddelx = -gdx * con_o[0] - gdy * con_o[1];
		const float dG_ddely = -gdy * con_o[2] - gdx * con_o[1];
		acc_add(dL_dmean2D, s64->mean2D, 3 * (size_t)id, dL_dG * dG_ddelx * ddelx_dx);
		acc_add(dL_dmean2D, s64->mean2D, 3 * (size_t)id + 1, dL_dG * dG_ddely * ddely_dy);
		acc_add(dL_dconic, s64->conic, 4 * (size_t)id, -0.5f * gdx * dx * dL_dG);
		acc_add(dL_dconic, s64->conic, 4 * (size_t)id + 1, -0.5f * gdx * dy * dL_dG);
		acc_add(dL_dconic, s64->conic, 4 * (size_t)id + 3, -0.5f * gdy * dy * dL_dG);
		acc_add(dL_dopacity, s64->opacity, id, G * dL_dalpha);
	}
}

typedef struct orc_grads {
	float *dL_dmeans2D, *dL_dcolors, *dL_dopacity, *dL_dmeans3D, *dL_dcov3D, *dL_dsh, *dL_dscales, *dL_drotations;
} orc_grads;

/* computeCov2DCUDA (backward.cu:144-274) */
static void cov2d_backward(const orc_ctx* c, int idx, const float* cov3D, const float* dL_dconics, float* dL_dmeans,
                           float* dL_dcov)
{
	v3 mean = V3(c->means3D[3 * idx], c->means3D[3 * idx + 1], c->means3D[3 * idx + 2]);
	float dcx = dL_dconics[4 * idx], dcy = dL_dconics[4 * idx + 1], dcz = dL_dconics[4 * idx + 3];
	cov2d_parts p;
	cov2d_common(mean, c->focal_x, c->focal_y, c->tanfovx, c->tanfovy, cov3D, c->view, &p);
	const float x_grad_mul = (p.txtz < -p.limx || p.txtz > p.limx) ? 0 : 1;
	const float y_grad_mul = (p.tytz < -p.limy || p.tytz > p.limy) ? 0 : 1;
	const float h_x = c->focal_x, h_y = c->focal_y;
	float a = p.cov.m[0][0] + 0.3f, b = p.cov.m[0][1], cc = p.cov.m[1][1] + 0.3f;
	float denom = a * cc - b * b;
	float dL_da = 0, dL_db = 0, dL_dc = 0;
	float denom2inv = 1.0f / ((denom * denom) + 0.0000001f);
#define T_(i, j) p.T.m[i][j]
#define V_(i, j) p.Vrk.m[i][j]
#define W_(i, j) p.Wm.m[i][j]
	if (denom2inv != 0) {
		dL_da = denom2inv * (-cc * cc * dcx + 2 * b * cc * dcy + (denom - a * cc) * dcz);
		dL_dc = denom2inv * (-a * a * dcz + 2 * a * b * dcy + (denom - a * cc) * dcx);
		dL_db = denom2inv * 2 * (b * cc * dcx - (denom + 2 * b * b) * dcy + a * b * dcz);
		dL_dcov[6 * idx + 0] = (T_(0, 0) * T_(0, 0) * dL_da + T_(0, 0) * T_(1, 0) * dL_db + T_(1, 0) * T_(1, 0) * dL_dc);
		dL_dcov[6 * idx + 3] = (T_(0, 1) * T_(0, 1) * dL_da + T_(0, 1) * T_(1, 1) * dL_db + T_(1, 1) * T_(1, 1) * dL_dc);
		dL_dcov[6 * idx + 5] = (T_(0, 2) * T_(0, 2) * dL_da + T_(0, 2) * T_(1, 2) * dL_db + T_(1, 2) * T_(1, 2) * dL_dc);
		dL_dcov[6 * idx + 1] = 2 * T_(0, 0) * T_(0, 1) * dL_da + (T_(0, 0) * T_(1, 1) + T_(0, 1) * T_(1, 0)) * dL_db + 2 * T_(1, 0) * T_(1, 1) * dL_dc;
		dL_dcov[6 * idx + 2] = 2 * T_(0, 0) * T_(0, 2) * dL_da + (T_(0, 0) * T_(1, 2) + T_(0, 2) * T_(1, 0)) * dL_db + 2 * T_(1, 0) * T_(1, 2) * dL_dc;
		dL_dcov[6 * idx + 4] = 2 * T_(0, 2) * T_(0, 1) * dL_da + (T_(0, 1) * T_(1, 2) + T_(0, 2) * T_(1, 1)) * dL_db + 2 * T_(1, 1) * T_(1, 2) * dL_dc;
	} else {
		for (int i = 0; i < 6; i++) dL_dcov[6 * idx + i] = 0;
	}
	float dL_dT00 = 2 * (T_(0, 0) * V_(0, 0) + T_(0, 1) * V_(0, 1) + T_(0, 2) * V_(0, 2)) * dL_da + (T_(1, 0) * V_(0, 0) + T_(1, 1) * V_(0, 1) + T_(1, 2) * V_(0, 2)) * dL_db;
	float dL_dT01 = 2 * (T_(0, 0) * V_(1, 0) + T_(0, 1) * V_(1, 1) + T_(0, 2) * V_(1, 2)) * dL_da + (T_(1, 0) * V_(1, 0) + T_(1, 1) * V_(1, 1) + T_(1, 2) * V_(1, 2)) * dL_db;
	float dL_dT02 = 2 * (T_(0, 0) * V_(2, 0) + T_(0, 1) * V_(2, 1) + T_(0, 2) * V_(2, 2)) * dL_da + (T_(1, 0) * V_(2, 0) + T_(1, 1) * V_(2, 1) + T_(1, 2) * V_(2, 2)) * dL_db;
	float dL_dT10 = 2 * (T_(1, 0) * V_(0, 0) + T_(1, 1) * V_(0, 1) + T_(1, 2) * V_(0, 2)) * dL_dc + (T_(0, 0) * V_(0, 0) + T_(0, 1) * V_(0, 1) + T_(0, 2) * V_(0, 2)) * dL_db;
	float dL_dT11 = 2 * (T_(1, 0) * V_(1, 0) + T_(1, 1) * V_(1, 1) + T_(1, 2) * V_(1, 2)) * dL_dc + (T_(0, 0) * V_(1, 0) + T_(0, 1) * V_(1, 1) + T_(0, 2) * V_(1, 2)) * dL_db;
	float dL_dT12 = 2 * (T_(1, 0) * V_(2, 0) + T_(1, 1) * V_(2, 1) + T_(1, 2) * V_(2, 2)) * dL_dc + (T_(0, 0) * V_(2, 0) + T_(0, 1) * V_(2, 1) + T_(0, 2) * V_(2, 2)) * dL_db;
	float dL_dJ00 = W_(0, 0) * dL_dT00 + W_(0, 1) * dL_dT01 + W_(0, 2) * dL_dT02;
	float dL_dJ02 = W_(2, 0) * dL_dT00 + W_(2, 1) * dL_dT01 + W_(2, 2) * dL_dT02;
	float dL_dJ11 = W_(1, 0) * dL_dT10 + W_(1, 1) * dL_dT11 + W_(1, 2) * dL_dT12;
	float dL_dJ12 = W_(2, 0) * dL_dT10 + W_(2, 1) * dL_dT11 + W_(2, 2) * dL_dT12;
#undef T_
#undef V_
#undef W_
	float tz = 1.f / p.t.z, tz2 = tz * tz, tz3 = tz2 * tz;
	float dL_dtx = x_grad_mul * -h_x * tz2 * dL_dJ02;
	float dL_dty = y_grad_mul * -h_y * tz2 * dL_dJ12;
	float dL_dtz = -h_x * tz2 * dL_dJ00 - h_y * tz2 * dL_dJ11 + (2 * h_x * p.t.x) * tz3 * dL_dJ02 + (2 * h_y * p.t.y) * tz3 * dL_dJ12;
	v3 dm = transformVec4x3Transpose(V3(dL_dtx, dL_dty, dL_dtz), c->view);
	dL_dmeans[3 * idx] = dm.x; /* overwrite (backward.cu:273) */
	dL_dmeans[3 * idx + 1] = dm.y;
	dL_dmeans[3 * idx + 2] = dm.z;
}

/* computeColorFromSH backward (backward.cu:20-139) */
static void sh_backward(const orc_ctx* c, int idx, const float* dL_dcolor, float* dL_dmeans, float* dL_dshs)
{
	const int deg = c->D, M = c->M;
	v3 pos = V3(c->means3D[3 * idx], c->means3D[3 * idx + 1], c->means3D[3 * idx + 2]);
	v3 dir_orig = v3_sub(pos, V3(c->campos[0], c->campos[1], c->campos[2]));
	float len = sqrtf(v3_dot(dir_orig, dir_orig));
	v3 dir = V3(dir_orig.x / len, dir_orig.y / len, dir_orig.z / len);
	const float* shs_row = c->shs + (size_t)idx * M * 3;
#define SH(k) V3(shs_row[3 * (k)], shs_row[3 * (k) + 1], shs_row[3 * (k) + 2])
	v3 dL_dRGB = V3(dL_dcolor[3 * idx], dL_dcolor[3 * idx + 1], dL_dcolor[3 * idx + 2]);
	dL_dRGB.x *= c->clamped[3 * idx + 0] ? 0 : 1;
	dL_dRGB.y *= c->clamped[3 * idx + 1] ? 0 : 1;
	dL_dRGB.z *= c->clamped[3 * idx + 2] ? 0 : 1;
	v3 dRGBdx = V3(0, 0, 0), dRGBdy = V3(0, 0, 0), dRGBdz = V3(0, 0, 0);
	float x = dir.x, y = dir.y, z = dir.z;
	float* dL_dsh = dL_dshs + (size_t)idx * M * 3;
#define SET(k, f) do { v3 _g = v3_scale((f), dL_dRGB); dL_dsh[3 * (k)] = _g.x; dL_dsh[3 * (k) + 1] = _g.y; dL_dsh[3 * (k) + 2] = _g.z; } while (0)
	SET(0, SH_C0);
	if (deg > 0) {
		SET(1, -SH_C1 * y);
		SET(2, SH_C1 * z);
		SET(3, -SH_C1 * x);
		dRGBdx = v3_scale(-SH_C1, SH(3));
		dRGBdy = v3_scale(-SH_C1, SH(1));
		dRGBdz = v3_scale(SH_C1, SH(2));
		if (deg > 1) {
			float xx = x * x, yy = y * y, zz = z * z, xy = x * y, yz = y * z, xz = x * z;
			SET(4, SH_C2[0] * xy);
			SET(5, SH_C2[1] * yz);
			SET(6, SH_C2[2] * (2.f * zz - xx - yy));
			SET(7, SH_C2[3] * xz);
			SET(8, SH_C2[4] * (xx - yy));
			dRGBdx = v3_add(dRGBdx, v3_add(v3_add(v3_add(v3_scale(SH_C2[0] * y, SH(4)), v3_scale(SH_C2[2] * 2.f * -x, SH(6))), v3_scale(SH_C2[3] * z, SH(7))), v3_scale(SH_C2[4] * 2.f * x, SH(8))));
			dRGBdy = v3_add(dRGBdy, v3_add(v3_add(v3_add(v3_scale(SH_C2[0] * x, SH(4)), v3_scale(SH_C2[1] * z, SH(5))), v3_scale(SH_C2[2] * 2.f * -y, SH(6))), v3_scale(SH_C2[4] * 2.f * -y, SH(8))));
			dRGBdz = v3_add(dRGBdz, v3_add(v3_add(v3_scale(SH_C2[1] * y, SH(5)), v3_scale(SH_C2[2] * 2.f * 2.f * z, SH(6))), v3_scale(SH_C2[3] * x, SH(7))));
			if (deg > 2) {
				SET(9, SH_C3[0] * y * (3.f * xx - yy));
				SET(10, SH_C3[1] * xy * z);
				SET(11, SH_C3[2] * y * (4.f * zz - xx - yy));
				SET(12, SH_C3[3] * z * (2.f * zz - 3.f * xx - 3.f * yy));
				SET(13, SH_C3[4] * x * (4.f * zz - xx - yy));
				SET(14, SH_C3[5] * z * (xx - yy));
				SET(15, SH_C3[6] * x * (xx - 3.f * yy));
				v3 ax = V3(0, 0, 0), ay = V3(0, 0, 0), az = V3(0, 0, 0);
				ax = v3_add(ax, v3_scale(SH_C3[0] * 3.f * 2.f * xy, SH(9)));
				ax = v3_add(ax, v3_scale(SH_C3[1] * yz, SH(10)));
				ax = v3_add(ax, v3_scale(SH_C3[2] * -2.f * xy, SH(11)));
				ax = v3_add(ax, v3_scale(SH_C3[3] * -3.f * 2.f * xz, SH(12)));
				ax = v3_add(ax, v3_scale(SH_C3[4] * (-3.f * xx + 4.f * zz - yy), SH(13)));
				ax = v3_add(ax, v3_scale(SH_C3[5] * 2.f * xz, SH(14)));
				ax = v3_add(ax, v3_scale(SH_C3[6] * 3.f * (xx - yy), SH(15)));
				ay = v3_add(ay, v3_scale(SH_C3[0] * 3.f * (xx - yy), SH(9)));
				ay = v3_add(ay, v3_scale(SH_C3[1] * xz, SH(10)));
				ay = v3_add(ay, v3_scale(SH_C3[2] * (-3.f * yy + 4.f * zz - xx), SH(11)));
				ay = v3_add(ay, v3_scale(SH_C3[3] * -3.f * 2.f * yz, SH(12)));
				ay = v3_add(ay, v3_scale(SH_C3[4] * -2.f * xy, SH(13)));
				ay = v3_add(ay, v3_scale(SH_C3[5] * -2.f * yz, SH(14)));
				ay = v3_add(ay, v3_scale(SH_C3[6] * -3.f * 2.f * xy, SH(15)));
				az = v3_add(az, v3_scale(SH_C3[1] * xy, SH(10)));
				az = v3_add(az, v3_scale(SH_C3[2] * 4.f * 2.f * yz, SH(11)));
				az = v3_add(az, v3_scale(SH_C3[3] * 3.f * (2.f * zz - xx - yy), SH(12)));
				az = v3_add(az, v3_scale(SH_C3[4] * 4.f * 2.f * xz, SH(13)));
				az = v3_add(az, v3_scale(SH_C3[5] * (xx - yy), SH(14)));
				dRGBdx = v3_add(dRGBdx, ax);
				dRGBdy = v3_add(dRGBdy, ay);
				dRGBdz = v3_add(dRGBdz, az);
			}
		}
	}
#undef SET
#undef SH
	v3 dL_ddir = V3(v3_dot(dRGBdx, dL_dRGB), v3_dot(dRGBdy, dL_dRGB), v3_dot(dRGBdz, dL_dRGB));
	v3 dm = dnormvdv(dir_orig, dL_ddir);
	dL_dmeans[3 * idx] += dm.x;
	dL_dmeans[3 * idx + 1] += dm.y;
	dL_dmeans[3 * idx + 2] += dm.z;
}

/* computeCov3D backward (backward.cu:278-341) */
static void cov3d_backward(const orc_ctx* c, int idx, const float* dL_dcov3Ds, float* dL_dscales, float* dL_drots)
{
	const float* rot = c->rotations + 4 * (size_t)idx;
	const float* sc = c->scales + 3 * (size_t)idx;
	float r = rot[0], x = rot[1], y = rot[2], z = rot[3];
	m3 R = m3_cols(1.f - 2.f * (y * y + z * z), 2.f * (x * y - r * z), 2.f * (x * z + r * y),
	               2.f * (x * y + r * z), 1.f - 2.f * (x * x + z * z), 2.f * (y * z - r * x),
	               2.f * (x * z - r * y), 2.f * (y * z + r * x), 1.f - 2.f * (x * x + y * y));
	m3 S = m3_cols(1, 0, 0, 0, 1, 0, 0, 0, 1);
	v3 s = v3_scale(c->scale_modifier, V3(sc[0], sc[1], sc[2]));
	S.m[0][0] = s.x;
	S.m[1][1] = s.y;
	S.m[2][2] = s.z;
	m3 M = m3_mul(S, R);
	const float* d = dL_dcov3Ds + 6 * (size_t)idx;
	m3 dL_dSigma = m3_cols(d[0], 0.5f * d[1], 0.5f * d[2], 0.5f * d[1], d[3], 0.5f * d[4], 0.5f * d[2], 0.5f * d[4], d[5]);
	m3 M2 = M;
	for (int a = 0; a < 3; a++)
		for (int b = 0; b < 3; b++) M2.m[a][b] = M.m[a][b] * 2.0f;
	m3 dL_dM = m3_mul(M2, dL_dSigma);
	m3 Rt = m3_transpose(R);
	m3 dL_dMt = m3_transpose(dL_dM);
	float* ds = dL_dscales + 3 * (size_t)idx;
	ds[0] = Rt.m[0][0] * dL_dMt.m[0][0] + Rt.m[0][1] * dL_dMt.m[0][1] + Rt.m[0][2] * dL_dMt.m[0][2];
	ds[1] = Rt.m[1][0] * dL_dMt.m[1][0] + Rt.m[1][1] * dL_dMt.m[1][1] + Rt.m[1][2] * dL_dMt.m[1][2];
	ds[2] = Rt.m[2][0] * dL_dMt.m[2][0] + Rt.m[2][1] * dL_dMt.m[2][1] + Rt.m[2][2] * dL_dMt.m[2][2];
	for (int k = 0; k < 3; k++) { dL_dMt.m[0][k] *= s.x; dL_dMt.m[1][k] *= s.y; dL_dMt.m[2][k] *= s.z; }
#define MT(a, b) dL_dMt.m[a][b]
	float* dq = dL_drots + 4 * (size_t)idx;
	dq[0] = 2 * z * (MT(0, 1) - MT(1, 0)) + 2 * y * (MT(2, 0) - MT(0, 2)) + 2 * x * (MT(1, 2) - MT(2, 1));
	dq[1] = 2 * y * (MT(1, 0) + MT(0, 1)) + 2 * z * (MT(2, 0) + MT(0, 2)) + 2 * r * (MT(1, 2) - MT(2, 1)) - 4 * x * (MT(2, 2) + MT(1, 1));
	dq[2] = 2 * x * (MT(1, 0) + MT(0, 1)) + 2 * r * (MT(2, 0) - MT(0, 2)) + 2 * z * (MT(1, 2) + MT(2, 1)) - 4 * y * (MT(2, 2) + MT(0, 0));
	dq[3] = 2 * r * (MT(0, 1) - MT(1, 0)) + 2 * x * (MT(2, 0) + MT(0, 2)) + 2 * y * (MT(1, 2) + MT(2, 1)) - 4 * z * (MT(1, 1) + MT(0, 0));
#undef MT
}

/* preprocessCUDA backward for every rendered Gaussian (rasterizer_impl.cu:476-503, backward.cu:144-396) from the
 * per-Gaussian sums of the blend backward: dL_dmeans2D [P,3], dL_dconic [P,4] (x, y, -, w), dL_dcolors [P,3] and
 * dL_dz [P] (NULL: no depth term).  Writes the rows with radii > 0 of g->dL_dmeans3D, dL_dcov3D, dL_dsh, dL_dscales
 * and dL_drotations and leaves the other rows alone.  Call after orc_forward on the same ctx. */
int orc_preprocess_backward(const orc_ctx* c, const float* dL_dmeans2D, const float* dL_dconic, const float* dL_dcolors,
                            const float* dL_dz, const orc_grads* g)
{
	const int P = c->P;
	const float* cov3D_all = c->cov3D_precomp ? c->cov3D_precomp : c->cov3D; /* rasterizer_impl.cu:481 */
#pragma omp parallel for schedule(static)
	for (int idx = 0; idx < P; idx++) {
		if (!(c->radii[idx] > 0)) continue;
		cov2d_backward(c, idx, cov3D_all + 6 * (size_t)idx, dL_dconic, g->dL_dmeans3D, g->dL_dcov3D);
		/* preprocessCUDA backward (backward.cu:346-396) */
		v3 m = V3(c->means3D[3 * idx], c->means3D[3 * idx + 1], c->means3D[3 * idx + 2]);
		const float* proj = c->proj;
		float hom[4];
		transformPoint4x4(m, proj, hom);
		float m_w = 1.0f / (hom[3] + 0.0000001f);
		float mul1 = (proj[0] * m.x + proj[4] * m.y + proj[8] * m.z + proj[12]) * m_w * m_w;
		float mul2 = (proj[1] * m.x + proj[5] * m.y + proj[9] * m.z + proj[13]) * m_w * m_w;
		const float d2x = dL_dmeans2D[3 * idx], d2y = dL_dmeans2D[3 * idx + 1];
		g->dL_dmeans3D[3 * idx] += (proj[0] * m_w - proj[3] * mul1) * d2x + (proj[1] * m_w - proj[3] * mul2) * d2y;
		g->dL_dmeans3D[3 * idx + 1] += (proj[4] * m_w - proj[7] * mul1) * d2x + (proj[5] * m_w - proj[7] * mul2) * d2y;
		g->dL_dmeans3D[3 * idx + 2] += (proj[8] * m_w - proj[11] * mul1) * d2x + (proj[9] * m_w - proj[11] * mul2) * d2y;
		if (dL_dz) { /* z = p_view.z = view[2] x + view[6] y + view[10] z + view[14] (forward.cu:186,250) */
			g->dL_dmeans3D[3 * idx] += c->view[2] * dL_dz[idx];
			g->dL_dmeans3D[3 * idx + 1] += c->view[6] * dL_dz[idx];
			g->dL_dmeans3D[3 * idx + 2] += c->view[10] * dL_dz[idx];
		}
		if (c->shs) sh_backward(c, idx, dL_dcolors, g->dL_dmeans3D, g->dL_dsh);
		if (c->scales) cov3d_backward(c, idx, g->dL_dcov3D, g->dL_dscales, g->dL_drotations);
	}
	return 0;
}

/* Rasterizer::backward (rasterizer_impl.cu:403-504) after orc_forward on the same ctx.
 * All gradient arrays are zero-filled here like rasterize_points.cu:154-162. dL_dout_depth is unused. */
int orc_backward_ex(orc_ctx* c, const float* dL_dpixels, const float* dL_ddepths, const orc_grads* g);
int orc_backward(orc_ctx* c, const float* dL_dpixels, const orc_grads* g) { return orc_backward_ex(c, dL_dpixels, NULL, g); }

/* dL_ddepths == NULL: the reference's behaviour (depth carries no gradient).  Non-NULL: the opt-in
 * depth-gradient extension described at render_pixel_backward. */
int orc_backward_ex(orc_ctx* c, const float* dL_dpixels, const float* dL_ddepths, const orc_grads* g)
{
	const int P = c->P, M = c->M, W = c->W, H = c->H;
	memset(g->dL_dmeans2D, 0, sizeof(float) * 3 * (size_t)P);
	memset(g->dL_dcolors, 0, sizeof(float) * 3 * (size_t)P);
	memset(g->dL_dopacity, 0, sizeof(float) * (size_t)P);
	memset(g->dL_dmeans3D, 0, sizeof(float) * 3 * (size_t)P);
	memset(g->dL_dcov3D, 0, sizeof(float) * 6 * (size_t)P);
	if (M > 0 && g->dL_dsh) memset(g->dL_dsh, 0, sizeof(float) * 3 * (size_t)P * M);
	memset(g->dL_dscales, 0, sizeof(float) * 3 * (size_t)P);
	memset(g->dL_drotations, 0, sizeof(float) * 4 * (size_t)P);
	if (P == 0) return 0;
	float* dL_dconic = (float*)calloc((size_t)4 * P, sizeof(float));
	float* dL_dz = (float*)calloc((size_t)P, sizeof(float));
	const float* colors = c->colors_precomp ? c->colors_precomp : c->rgb; /* rasterizer_impl.cu:453 */
	const int ntiles = c->gx * c->gy;
	sum64 s64 = {NULL, NULL, NULL, NULL, NULL};
	if (g_f64_sums) {
		s64.mean2D = (double*)calloc((size_t)3 * P, sizeof(double));
		s64.conic = (double*)calloc((size_t)4 * P, sizeof(double));
		s64.opacity = (double*)calloc((size_t)P, sizeof(double));
		s64.colors = (double*)calloc((size_t)3 * P, sizeof(double));
		s64.z = (double*)calloc((size_t)P, sizeof(double));
	}
#pragma omp parallel for schedule(dynamic, 1)
	for (int tile = 0; tile < ntiles; tile++) {
		const int tx = tile % c->gx, ty = tile / c->gx;
		const uint32_t start = c->ranges[2 * tile], end = c->ranges[2 * tile + 1];
		if (end <= start) continue;
		for (int ly = 0; ly < BLOCK_Y; ly++)
			for (int lx = 0; lx < BLOCK_X; lx++) {
				const int px = tx * BLOCK_X + lx, py = ty * BLOCK_Y + ly;
				if (px < W && py < H)
					render_pixel_backward(c, px, py, start, end, colors, dL_dpixels, dL_ddepths, g->dL_dmeans2D, dL_dconic,
					                      g->dL_dopacity, g->dL_dcolors, dL_dz, &s64);
			}
	}
	if (g_f64_sums) { /* round the double sums once */
		for (size_t i = 0; i < (size_t)3 * P; i++) g->dL_dmeans2D[i] = (float)s64.mean2D[i];
		for (size_t i = 0; i < (size_t)4 * P; i++) dL_dconic[i] = (float)s64.conic[i];
		for (size_t i = 0; i < (size_t)P; i++) g->dL_dopacity[i] = (float)s64.opacity[i];
		for (size_t i = 0; i < (size_t)3 * P; i++) g->dL_dcolors[i] = (float)s64.colors[i];
		for (size_t i = 0; i < (size_t)P; i++) dL_dz[i] = (float)s64.z[i];
		free(s64.mean2D); free(s64.conic); free(s64.opacity); free(s64.colors); free(s64.z);
	}
	orc_preprocess_backward(c, g->dL_dmeans2D, dL_dconic, g->dL_dcolors, dL_ddepths ? dL_dz : NULL, g);
	free(dL_dconic);
	free(dL_dz);
	return 0;
}

/*
 * blend_f64.c — double-precision referee for the blend kernels (tests only; built with gcc by tests/blend_f64.py).
 *
 * Input: the per-Gaussian records the library blends (means2D, conic + opacity, colour, depth, all fp32), the
 * depth-sorted `point_list` and the per-tile `ranges`.  Everything after the list is recomputed in double from
 * those fp32 values, with the reference's rules (renderCUDA, forward.cu:341-471 / backward.cu:399-586):
 *   - no culling: every pair of a tile's list is evaluated;
 *   - power > 0 skips; alpha = min(0.99f, o G); alpha < 1/255 skips;
 *   - a record that would take T below 1e-4 is not blended and the pixel stops;
 *   - acc = 1e-6 + sum T alpha; depth = D / acc when acc > 0.5.
 * The thresholds are the fp32 constants the kernels compare against (1.0f/255.0f, 0.99f, 0.0001f, 0.000001f).
 *
 * Per-Gaussian outputs are the ten accumulator slots of blend_bwd.cu, before the per-Gaussian constants of the
 * preprocess backward (preprocess_bwd.cu:163-167): 0-1 mean2D x, y (before 0.5 W, 0.5 H), 2-4 conic a, b, c
 * (before -0.5), 5 opacity, 6-8 colour, 9 dL/dz (depth gradient).  The documented quirk is kept: the alpha
 * derivative ignores the 0.99 clamp (blend_bwd.cu:27; reference backward.cu:547-551 uses G * dL_dalpha).
 * With every pair's T taken from the forward in double, no division back to front is needed here.
 *
 * Threshold decisions.  A CPU cannot reproduce ex2.approx bit for bit, so each of the two tests has a guard band
 * from an fp32 error model; a pair inside it is "undecided":
 *   - alpha >= 1/255 (and power > 0): q = a dx^2 + 2 b dx dy + c dy^2 is evaluated in fp32 with an absolute error
 *     of at most Eq = 8 eps (|a| dx^2 + |c| dy^2 + 2 |b| |dx dy|) — the model cull_tau() (preprocess.cu:157) uses —
 *     so power carries 0.5 Eq, and exp (<= 2 ulp) and the product with o add 4 eps relative:
 *     alpha's relative error is da = 0.5 Eq + 4 eps;
 *   - T (1 - alpha) < 1e-4: T's relative error grows along the list (rT below), plus alpha's contribution
 *     alpha da / (1 - alpha) and 2 eps for this step's subtraction and product.
 * Undecided pairs of a pixel are resolved from the implementation's own per-pixel outputs (impl_T / impl_n): of
 * the at most 2^3 assignments, the one whose n_contrib equals the implementation's and whose T lies within the
 * forward bound is kept.  A pixel with more than 3 undecided pairs, or with two matching assignments that blend
 * different records, is excluded; so is every Gaussian that may contribute to it.
 *
 * Error model of T (used by every tolerance): each blended record multiplies T by (1 - alpha) in fp32, which adds
 * 2 eps of relative error (the subtraction and the product), and alpha's own error da adds alpha da / (1 - alpha)
 * (none when alpha is clamped to 0.99, which both sides represent exactly).  rho = sum of these, in units of eps,
 * is at least 2 n_contrib: a bound linear in n_contrib, widened where alpha's error is amplified.
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#define EPS 5.9604644775390625e-08 /* 2^-24 */
#define NSLOT 10
#define MAX_UNDECIDED 3

enum { MUT_NONE = 0, MUT_DROP_PAIR, MUT_DROP_BLOCK, MUT_ROW_SHIFT, MUT_DOUBLE_RECORD, MUT_DROP_PARTIAL_GROUP, MUT_SKIP_FIRST_LIVE };
enum { PIX_DECIDED = 0, PIX_RESOLVED = 1, PIX_EXCLUDED = 2, PIX_MISMATCH = 3 };

typedef struct bf_in {
	int P, W, H;
	const float *means2D;       /* [P,2] */
	const float *conic_opacity; /* [P,4] */
	const float *colors;        /* [P,3] */
	const float *depths;        /* [P] */
	const uint32_t *point_list; /* [R] */
	const uint32_t *ranges;     /* [tiles,2] */
	const float *bg;            /* [3] */
	const float *dL_dpix;       /* [3,H,W] */
	const float *dL_ddepth;     /* [H,W] or NULL: the depth gradient is off */
	const float *impl_T;        /* [H,W] implementation's final T, or NULL */
	const uint32_t *impl_n;     /* [H,W] implementation's n_contrib, or NULL */
	int mutation, mut_a, mut_b; /* reference-side mutations, for the tests that prove the bounds catch bugs */
} bf_in;

typedef struct bf_out {
	double *T, *color, *depth, *acc; /* [H,W], [3,H,W], [H,W], [H,W] */
	uint32_t *n_contrib;             /* [H,W] */
	double *rho;                     /* [H,W] T's relative error bound, in units of eps */
	double *color_mag, *depth_mag;   /* [3,H,W], [H,W]: sums of |terms| */
	double *da_max;                  /* [H,W] largest relative error bound of a blended alpha, in units of eps */
	int32_t *pix_state;              /* [H,W] PIX_* */
	double *g, *m;                   /* [P,10] exact sums and magnitude sums */
	int32_t *L;                      /* [P] deepest list position (0-based, within the tile) it contributes at, -1 none */
	double *rho_max;                 /* [P] largest rho of the pixels it contributes to */
	double *da_g;                    /* [P] largest relative error bound of its alphas, in units of eps */
	int32_t *blocks;                 /* [P] number of 8x8 pixel blocks it contributes in */
	uint8_t *excluded;               /* [P] */
	long long stats[4];              /* pairs evaluated, pairs contributing, undecided pairs seen, pixels excluded */
} bf_out;

typedef struct contrib {
	int32_t pos; /* list position within the tile */
	double alpha, G, T; /* T before this record */
	double da;          /* alpha's relative error bound */
} contrib;

typedef struct path {
	int n_und;      /* undecided pairs met on this path (> MAX_UNDECIDED: overflow) */
	int ncon;       /* blended records */
	uint32_t last;  /* n_contrib: 1 + list position of the last blended record */
	double T, rT;
} path;

static const float F_ALPHA_MIN = 1.0f / 255.0f, F_ALPHA_MAX = 0.99f, F_T_MIN = 0.0001f, F_ACC0 = 0.000001f;

typedef struct pair_eval {
	double dx, dy, power, G, raw, alpha, da;
	int pass; /* 1 pass, 0 skip, -1 undecided */
} pair_eval;

static void eval_pair(const bf_in* in, uint32_t id, double px, double py, pair_eval* e)
{
	const float* co = in->conic_opacity + 4 * (size_t)id;
	const double a = co[0], b = co[1], c = co[2], o = co[3];
	e->dx = (double)in->means2D[2 * id] - px;
	e->dy = (double)in->means2D[2 * id + 1] - py;
	const double dx = e->dx, dy = e->dy;
	e->power = -0.5 * (a * dx * dx + c * dy * dy) - b * dx * dy;
	const double Ep = 0.5 * 8.0 * EPS * (fabs(a) * dx * dx + fabs(c) * dy * dy + 2.0 * fabs(b) * fabs(dx * dy));
	e->G = exp(e->power);
	const double raw = o * e->G;
	e->raw = raw;
	e->da = Ep + 4.0 * EPS;
	e->alpha = raw < (double)F_ALPHA_MAX ? raw : (double)F_ALPHA_MAX;
	if (raw >= (double)F_ALPHA_MAX * (1.0 + e->da))
		e->da = 0.0; /* clamped on both sides: 0.99f exactly */
	int p_pos; /* power > 0 */
	if (e->power > Ep)
		p_pos = 1;
	else if (e->power < -Ep || Ep == 0.0)
		p_pos = 0;
	else
		p_pos = -1;
	const double thr = (double)F_ALPHA_MIN, band = (Ep + 4.0 * EPS) * (raw > thr ? raw : thr);
	int a_ok;
	if (raw - thr > band)
		a_ok = 1;
	else if (thr - raw > band)
		a_ok = 0;
	else
		a_ok = -1;
	if (!(o == o)) /* non-finite opacity: the constructed and random scenes have none */
		a_ok = -1;
	if (p_pos == 1 || a_ok == 0)
		e->pass = 0;
	else if (p_pos == 0 && a_ok == 1)
		e->pass = 1;
	else
		e->pass = -1;
}

/* y coordinate at which a pixel is evaluated: the true row, or (MUT_ROW_SHIFT) rows 4..7 of each 8x8 block shifted,
 * as if a lane's second pixel were taken at y + 4 + shift. */
static double eval_y(const bf_in* in, int py)
{
	if (in->mutation == MUT_ROW_SHIFT && (py & 7) >= 4)
		return (double)(py + in->mut_a);
	return (double)py;
}

/* One pixel's forward.  assign >= 0: the k-th undecided decision on the path takes bit k of assign (1 = the pair
 * passes the alpha test / the record saturates the pixel); assign < 0: undecided pairs take the double-precision
 * decision.  Contributors go to `out` (may be NULL). */
static void pixel_path(const bf_in* in, int px, int py, uint32_t start, uint32_t end, int assign, contrib* out, path* r,
                       long long* evaluated)
{
	double T = 1.0, rT = 0.0;
	int und = 0, ncon = 0;
	uint32_t last = 0;
	const double fx = (double)px, fy = eval_y(in, py);
	for (uint32_t k = start; k < end; k++) {
		const uint32_t id = in->point_list[k];
		pair_eval e;
		eval_pair(in, id, fx, fy, &e);
		if (evaluated)
			(*evaluated)++;
		int pass = e.pass;
		if (pass < 0) {
			pass = assign >= 0 ? (assign >> und) & 1 : (e.power <= 0.0 && e.raw >= (double)F_ALPHA_MIN);
			und++;
		}
		if (!pass)
			continue;
		const double om = 1.0 - e.alpha, test = T * om, thr = (double)F_T_MIN;
		const double step = 2.0 * EPS + (om > 0 ? e.alpha * e.da / om : 0.0);
		const double band = (rT + step) * thr;
		int sat;
		if (thr - test > band)
			sat = 1;
		else if (test - thr > band)
			sat = 0;
		else {
			sat = assign >= 0 ? (assign >> und) & 1 : (test < thr);
			und++;
		}
		if (sat)
			break;
		if (out) {
			out[ncon].pos = (int32_t)(k - start);
			out[ncon].alpha = e.alpha;
			out[ncon].G = e.G;
			out[ncon].T = T;
			out[ncon].da = e.da;
		}
		ncon++;
		T = test;
		rT += step;
		last = k - start + 1;
	}
	r->n_und = und;
	r->ncon = ncon;
	r->last = last;
	r->T = T;
	r->rT = rT;
}

/* Forward tolerance factor: rho (in eps) bounds T's relative error; colour and depth add at most one more rounding
 * per term (alpha * colour, the fma into the sum), which the factor 2 covers: tol = 2 eps (1 + rho) |terms|. */
#define KAPPA_F 2.0

static int same_path(const contrib* a, int na, const contrib* b, int nb)
{
	if (na != nb)
		return 0;
	for (int i = 0; i < na; i++)
		if (a[i].pos != b[i].pos)
			return 0;
	return 1;
}

/* The forward of one pixel with its undecided pairs resolved; returns the PIX_* state. */
static int resolve_pixel(const bf_in* in, int px, int py, uint32_t start, uint32_t end, contrib* buf, contrib* tmp,
                         path* r, long long* stats)
{
	pixel_path(in, px, py, start, end, -1, buf, r, &stats[0]);
	if (r->n_und == 0)
		return PIX_DECIDED;
	stats[2] += r->n_und;
	const size_t pix = (size_t)in->W * py + px;
	if (in->impl_T == NULL || in->impl_n == NULL || r->n_und > MAX_UNDECIDED)
		return PIX_EXCLUDED;
	const double Ti = in->impl_T[pix];
	const uint32_t ni = in->impl_n[pix];
	int found = 0, ambiguous = 0;
	path best = *r;
	for (int a = 0; a < (1 << MAX_UNDECIDED); a++) {
		path q;
		contrib* dst = found ? tmp : buf;
		pixel_path(in, px, py, start, end, a, dst, &q, NULL);
		if (q.n_und > MAX_UNDECIDED || q.last != ni || fabs(q.T - Ti) > KAPPA_F * (EPS + q.rT) * q.T)
			continue;
		if (!found) {
			found = 1;
			best = q;
		} else if (!same_path(buf, best.ncon, tmp, q.ncon)) {
			ambiguous = 1;
		}
	}
	if (!found) { /* no assignment reproduces the implementation: keep the double-precision path, the checks fail */
		pixel_path(in, px, py, start, end, -1, buf, r, NULL);
		return PIX_MISMATCH;
	}
	*r = best;
	return ambiguous ? PIX_EXCLUDED : PIX_RESOLVED;
}

static int block_of(int W, int px, int py) { return (py >> 3) * ((W + 7) >> 3) + (px >> 3); }

int bf64_run(const bf_in* in, bf_out* out)
{
	const int W = in->W, H = in->H, P = in->P;
	const int gx = (W + 15) / 16, gy = (H + 15) / 16;
	memset(out->g, 0, sizeof(double) * NSLOT * (size_t)P);
	memset(out->m, 0, sizeof(double) * NSLOT * (size_t)P);
	memset(out->blocks, 0, sizeof(int32_t) * (size_t)P);
	memset(out->excluded, 0, (size_t)P);
	memset(out->stats, 0, sizeof(out->stats));
	for (int i = 0; i < P; i++) {
		out->L[i] = -1;
		out->rho_max[i] = 0.0;
		out->da_g[i] = 0.0;
	}
	uint32_t maxlen = 0;
	for (int t = 0; t < gx * gy; t++) {
		const uint32_t len = in->ranges[2 * t + 1] - in->ranges[2 * t];
		if (in->ranges[2 * t + 1] > in->ranges[2 * t] && len > maxlen)
			maxlen = len;
	}
	const size_t cap = (size_t)maxlen + 1;
	contrib* buf = (contrib*)malloc(sizeof(contrib) * 256 * cap);
	contrib* tmp = (contrib*)malloc(sizeof(contrib) * cap);
	path* paths = (path*)malloc(sizeof(path) * 256);
	int32_t* lastblk = (int32_t*)malloc(sizeof(int32_t) * (size_t)(P > 0 ? P : 1));
	uint8_t* used = (uint8_t*)malloc(cap);
	uint8_t* drop = (uint8_t*)malloc(cap);
	int* stage_pos = (int*)malloc(sizeof(int) * cap);
	if (!buf || !tmp || !paths || !lastblk || !used || !drop || !stage_pos) {
		free(buf); free(tmp); free(paths); free(lastblk); free(used); free(drop); free(stage_pos);
		return -1;
	}
	for (int i = 0; i < P; i++)
		lastblk[i] = -1;
	const size_t plane = (size_t)W * H;
	const int depth_on = in->dL_ddepth != NULL;

	for (int ty = 0; ty < gy; ty++)
		for (int tx = 0; tx < gx; tx++) {
			const int t = ty * gx + tx;
			uint32_t start = in->ranges[2 * t], end = in->ranges[2 * t + 1];
			if (end < start)
				end = start;
			const uint32_t len = end - start;
			uint32_t tile_max = 0;
			/* ---- forward of the tile's pixels ---- */
			for (int l = 0; l < 256; l++) {
				const int px = tx * 16 + (l & 15), py = ty * 16 + (l >> 4);
				if (px >= W || py >= H)
					continue;
				const size_t pix = (size_t)W * py + px;
				contrib* c = buf + (size_t)l * cap;
				path* r = &paths[l];
				int st = resolve_pixel(in, px, py, start, end, c, tmp, r, out->stats);
				double C[3] = {0, 0, 0}, Cm[3] = {0, 0, 0}, D = 0, Dm = 0, acc = (double)F_ACC0, da_max = 0;
				for (int i = 0; i < r->ncon; i++) {
					if (c[i].da > da_max)
						da_max = c[i].da;
					const uint32_t id = in->point_list[start + c[i].pos];
					const double wgt = c[i].alpha * c[i].T;
					for (int ch = 0; ch < 3; ch++) {
						C[ch] += in->colors[3 * (size_t)id + ch] * wgt;
						Cm[ch] += fabs((double)in->colors[3 * (size_t)id + ch]) * wgt;
					}
					D += in->depths[id] * wgt;
					Dm += fabs((double)in->depths[id]) * wgt;
					acc += wgt;
				}
				out->stats[1] += r->ncon;
				const double rho = r->rT / EPS;
				for (int ch = 0; ch < 3; ch++) {
					out->color[ch * plane + pix] = C[ch] + r->T * in->bg[ch];
					out->color_mag[ch * plane + pix] = Cm[ch] + r->T * fabs((double)in->bg[ch]);
				}
				/* the depth gate acc > 0.5 is a threshold decision too: acc carries the relative error of T */
				const int gate_undecided = fabs(acc - 0.5) <= KAPPA_F * (EPS + r->rT + da_max) * acc;
				const double depth = acc > 0.5 ? D / acc : 0.0;
				out->depth[pix] = depth;
				out->depth_mag[pix] = gate_undecided ? INFINITY : (acc > 0.5 ? (Dm + fabs(depth) * acc) / acc : 0.0);
				if (gate_undecided && depth_on && st != PIX_MISMATCH)
					st = PIX_EXCLUDED;
				out->T[pix] = r->T;
				out->acc[pix] = acc;
				out->n_contrib[pix] = r->last;
				out->rho[pix] = rho;
				out->da_max[pix] = da_max / EPS;
				out->pix_state[pix] = st;
				if (st == PIX_EXCLUDED) {
					out->stats[3]++;
					for (uint32_t k = start; k < end; k++) { /* every Gaussian that may contribute to it */
						pair_eval e;
						eval_pair(in, in->point_list[k], (double)px, eval_y(in, py), &e);
						if (e.pass != 0)
							out->excluded[in->point_list[k]] = 1;
					}
				}
				if (r->last > tile_max)
					tile_max = r->last;
			}
			/* ---- backward, one 8x8 block at a time (the kernels' warp blocks) ---- */
			const uint32_t n_tile = len < tile_max ? len : tile_max;
			for (int wb = 0; wb < 4; wb++) {
				const int bx = tx * 16 + (wb & 1) * 8, by = ty * 16 + (wb >> 1) * 8;
				if (bx >= W || by >= H)
					continue;
				const int blk = block_of(W, bx, by);
				uint32_t warp_max = 0;
				memset(used, 0, cap);
				memset(drop, 0, cap);
				for (int l = 0; l < 64; l++) {
					const int px = bx + (l & 7), py = by + (l >> 3);
					if (px >= W || py >= H)
						continue;
					const int tl = (py - ty * 16) * 16 + (px - tx * 16);
					const path* r = &paths[tl];
					if (r->last > warp_max)
						warp_max = r->last;
					for (int i = 0; i < r->ncon; i++)
						used[buf[(size_t)tl * cap + i].pos] = 1;
				}
				const int here = in->mut_a < 0 || in->mut_a == blk;
				if (in->mutation == MUT_DROP_PARTIAL_GROUP && here) {
					/* blend_bwd.cu: batches of 128 list positions walked back to front from the tile's
					 * min(len, max n_contrib); a batch's records that some pixel of the block blends are staged
					 * 8 at a time, and the remainder (the partial group) is dropped */
					int staged = 0; /* records of the current batch staged so far */
					for (int p = (int)n_tile - 1; p >= 0; p--) {
						if (p < (int)warp_max && used[p])
							stage_pos[staged++] = p;
						if (p == 0 || ((int)n_tile - 1 - p) % 128 == 127) { /* end of a batch */
							for (int k = staged - staged % 8; k < staged; k++)
								drop[stage_pos[k]] = 1;
							staged = 0;
						}
					}
				}
				if (in->mutation == MUT_SKIP_FIRST_LIVE && here && warp_max > 0)
					drop[warp_max - 1] = 2; /* the deepest live record of the block: skipped by the whole warp */

				for (int l = 0; l < 64; l++) {
					const int px = bx + (l & 7), py = by + (l >> 3);
					if (px >= W || py >= H)
						continue;
					const size_t pix = (size_t)W * py + px;
					if (out->pix_state[pix] == PIX_EXCLUDED)
						continue;
					const int tl = (py - ty * 16) * 16 + (px - tx * 16);
					const path* r = &paths[tl];
					const contrib* c = buf + (size_t)tl * cap;
					const double fx = (double)px, fy = eval_y(in, py), Tf = r->T, rho = r->rT / EPS;
					double dp[3], bgd = 0.0, bgdm = 0.0;
					for (int ch = 0; ch < 3; ch++) {
						dp[ch] = in->dL_dpix[ch * plane + pix];
						bgd += in->bg[ch] * dp[ch];
						bgdm += fabs(in->bg[ch] * dp[ch]);
					}
					double gD = 0.0, gA = 0.0;
					const double acc = out->acc[pix];
					if (depth_on && acc > 0.5) {
						gD = in->dL_ddepth[pix] / acc;
						gA = -in->dL_ddepth[pix] * out->depth[pix] / acc;
					}
					double beta = 0.0, betam = 0.0, la = 0.0, lcd = 0.0, lcdm = 0.0;
					for (int i = r->ncon - 1; i >= 0; i--) {
						const int pos = c[i].pos;
						const uint32_t id = in->point_list[start + pos];
						if (drop[pos] == 2)
							continue; /* skipped record: no recurrence step, no contribution */
						const float* co = in->conic_opacity + 4 * (size_t)id;
						const double a = co[0], b = co[1], cc = co[2], o = co[3];
						const double dx = (double)in->means2D[2 * id] - fx, dy = (double)in->means2D[2 * id + 1] - fy;
						const double al = c[i].alpha, G = c[i].G, T = c[i].T;
						beta = la * lcd + (1.0 - la) * beta;
						betam = la * lcdm + (1.0 - la) * betam;
						double cd = 0.0, cdm = 0.0;
						for (int ch = 0; ch < 3; ch++) {
							cd += in->colors[3 * (size_t)id + ch] * dp[ch];
							cdm += fabs(in->colors[3 * (size_t)id + ch] * dp[ch]);
						}
						if (depth_on) {
							cd += in->depths[id] * gD + gA;
							cdm += fabs(in->depths[id] * gD) + fabs(gA);
						}
						la = al;
						lcd = cd;
						lcdm = cdm;
						int mult = 1;
						if (drop[pos] == 1)
							mult = 0;
						if (in->mutation == MUT_DROP_PAIR && (size_t)in->mut_a == pix && (uint32_t)in->mut_b == id)
							mult = 0;
						if (in->mutation == MUT_DROP_BLOCK && in->mut_a == blk && (uint32_t)in->mut_b == id)
							mult = 0;
						if (in->mutation == MUT_DOUBLE_RECORD && in->mut_a == blk && (uint32_t)in->mut_b == id)
							mult = 2;
						const double dLda = (cd - beta) * T - Tf * bgd / (1.0 - al);
						const double dLdam = (cdm + betam) * T + Tf * bgdm / (1.0 - al);
						const double w = G * dLda, wm = G * dLdam, u = al * T;
						double v[NSLOT], vm[NSLOT];
						v[0] = -o * w * (a * dx + b * dy);
						vm[0] = fabs(o) * wm * (fabs(a * dx) + fabs(b * dy));
						v[1] = -o * w * (cc * dy + b * dx);
						vm[1] = fabs(o) * wm * (fabs(cc * dy) + fabs(b * dx));
						v[2] = o * w * dx * dx;
						vm[2] = fabs(o) * wm * dx * dx;
						v[3] = o * w * dx * dy;
						vm[3] = fabs(o) * wm * fabs(dx * dy);
						v[4] = o * w * dy * dy;
						vm[4] = fabs(o) * wm * dy * dy;
						v[5] = w;
						vm[5] = wm;
						for (int ch = 0; ch < 3; ch++) {
							v[6 + ch] = u * dp[ch];
							vm[6 + ch] = u * fabs(dp[ch]);
						}
						v[9] = depth_on ? u * gD : 0.0;
						vm[9] = depth_on ? u * fabs(gD) : 0.0;
						for (int s = 0; s < NSLOT; s++) {
							out->g[NSLOT * (size_t)id + s] += mult * v[s];
							out->m[NSLOT * (size_t)id + s] += vm[s];
						}
						if (pos > out->L[id])
							out->L[id] = pos;
						if (rho > out->rho_max[id])
							out->rho_max[id] = rho;
						if (c[i].da / EPS > out->da_g[id])
							out->da_g[id] = c[i].da / EPS;
						if (lastblk[id] != blk) {
							lastblk[id] = blk;
							out->blocks[id]++;
						}
					}
				}
			}
		}
	free(buf); free(tmp); free(paths); free(lastblk); free(used); free(drop); free(stage_pos);
	return 0;
}

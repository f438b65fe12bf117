// Double-precision referee of the preprocess backward (bloomscene_b200/csrc/preprocess_bwd.cu), Gaussian by Gaussian.
//
// Input: exactly the fp32 values the kernel sees — the Gaussians, the camera, radii and the blend accumulator
// [P, 12] (slots 0-1 means2D sums, 2-4 conic sums, 5 opacity, 6-8 colour, 9 depth) — with the kernel's per-Gaussian
// constants applied the kernel's way: dL_dmeans2D = slot * (0.5f W), dL_dconic = -0.5f * slot.
// Output, for every Gaussian with radii > 0: dL_dmeans3D, dL_dcov3D (reference layout, off-diagonals doubled),
// dL_dscales, dL_drotations and dL_dsh [M, 3], each with an error bound.
//
// The statements are the reference's, in the order oracle/rasterizer_oracle.c restates them (cov2d_common,
// cov2d_backward, the means2D block of orc_backward_ex, sh_backward, cov3d_backward; computeColorFromSH_fwd for the
// colour clamp).  They are NOT the kernel's derivation (preprocess_bwd_math.h), which this file must not share.
// Reference quirks kept: 1e-7 added to det^2; x/y_grad_mul, the clamped u ignoring its t_z dependence;
// 1 / (hw + 1e-7); the unnormalised quaternion; dL/dscale with respect to mod * scale; the colour clamp passing
// the gradient when rgb >= 0; the optional depth term view[2, 6, 10] * slot 9.
//
// The statements are written once, as a template over the scalar type:
//   double  the value;
//   Err     (double value, absolute bound): first-order running error of an fp32 evaluation of these statements,
//           u = 2^-24 per operation — add e = ea + eb + u|v|; mul |a|eb + |b|ea + u|v|;
//           div (ea + |v|eb)/|b| + u|v|, valid only while eb < |b|/2 (otherwise the Gaussian is excluded);
//           sqrt ea/(2|v|) + u|v|;
//   float   an fp32 evaluation, which the CPU tests use to show that the bound holds.
// Threshold decisions (|t_x/t_z| against 1.3 tan fov on both axes, each colour channel against 0 before the clamp)
// inside their value's error band are resolved by trying both branches.  pbwd_check passes a Gaussian when every
// element of one branch assignment satisfies |got - ref| <= K e + u |ref|.
#include <cmath>
#include <cstdint>
#include <cstring>

namespace {

constexpr double U = 1.0 / 16777216.0; // 2^-24

struct Err {
	double v, e;
	Err() : v(0), e(0) {}
	Err(double x) : v(x), e(0) {}
	Err(double x, double err) : v(x), e(err) {}
};
thread_local bool t_div_invalid = false;
inline Err operator+(Err a, Err b) { const double v = a.v + b.v; return Err(v, a.e + b.e + U * std::fabs(v)); }
inline Err operator-(Err a, Err b) { const double v = a.v - b.v; return Err(v, a.e + b.e + U * std::fabs(v)); }
inline Err operator-(Err a) { return Err(-a.v, a.e); }
inline Err operator*(Err a, Err b)
{
	const double v = a.v * b.v;
	return Err(v, std::fabs(a.v) * b.e + std::fabs(b.v) * a.e + U * std::fabs(v));
}
inline Err operator/(Err a, Err b)
{
	if (!(b.e < 0.5 * std::fabs(b.v)))
		t_div_invalid = true;
	const double v = a.v / b.v;
	return Err(v, (a.e + std::fabs(v) * b.e) / std::fabs(b.v) + U * std::fabs(v));
}
inline Err& operator+=(Err& a, Err b) { return a = a + b; }
inline Err& operator*=(Err& a, Err b) { return a = a * b; }
inline Err sqrt_(Err a)
{
	const double v = std::sqrt(a.v);
	return Err(v, a.e / (2 * v) + U * v);
}
inline double sqrt_(double a) { return std::sqrt(a); }
inline float sqrt_(float a) { return sqrtf(a); }
inline double val(Err a) { return a.v; }
inline double val(double a) { return a; }
inline double val(float a) { return a; }
inline double err(Err a) { return a.e; }
inline double err(double) { return 0; }
inline double err(float) { return 0; }

// cuda_rasterizer/auxiliary.h:22-39 (float constants, as the reference and the kernel use them)
const float SH_C0 = 0.28209479177387814f;
const float SH_C1 = 0.4886025119029199f;
const float SH_C2[] = {1.0925484305920792f, -1.0925484305920792f, 0.31539156525252005f, -1.0925484305920792f,
                       0.5462742152960396f};
const float SH_C3[] = {-0.5900435899266435f, 2.890611442640554f, -0.4570457994644658f, 0.3731763325901154f,
                       -0.4570457994644658f, 1.445305721320277f, -0.5900435899266435f};

template <class T> struct v3 { T x, y, z; };
template <class T> struct m3 { T m[3][3]; }; // m[col][row], like glm::mat3

template <class T> v3<T> V3(T x, T y, T z) { return v3<T>{x, y, z}; }
template <class T> v3<T> add(v3<T> a, v3<T> b) { return V3<T>(a.x + b.x, a.y + b.y, a.z + b.z); }
template <class T> v3<T> sub(v3<T> a, v3<T> b) { return V3<T>(a.x - b.x, a.y - b.y, a.z - b.z); }
template <class T> v3<T> scale(T s, v3<T> a) { return V3<T>(s * a.x, s * a.y, s * a.z); }
template <class T> T dot(v3<T> a, v3<T> b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
template <class T> m3<T> mul(const m3<T>& a, const m3<T>& b)
{
	m3<T> r;
	for (int c = 0; c < 3; c++)
		for (int k = 0; k < 3; k++)
			r.m[c][k] = a.m[0][k] * b.m[c][0] + a.m[1][k] * b.m[c][1] + a.m[2][k] * b.m[c][2];
	return r;
}
template <class T> m3<T> transpose(const m3<T>& a)
{
	m3<T> r;
	for (int c = 0; c < 3; c++)
		for (int k = 0; k < 3; k++)
			r.m[c][k] = a.m[k][c];
	return r;
}
template <class T> m3<T> cols(T x0, T y0, T z0, T x1, T y1, T z1, T x2, T y2, T z2)
{
	m3<T> r;
	r.m[0][0] = x0; r.m[0][1] = y0; r.m[0][2] = z0;
	r.m[1][0] = x1; r.m[1][1] = y1; r.m[1][2] = z1;
	r.m[2][0] = x2; r.m[2][1] = y2; r.m[2][2] = z2;
	return r;
}

} // namespace

extern "C" {

typedef struct pbwd_scene {
	int P, D, M, W, H, depth_gradient;
	float tanfovx, tanfovy, scale_modifier;
	const float *view, *proj, *campos;
	const float *means3D, *scales, *rotations, *cov3D_precomp, *shs; // shs NULL: precomputed colours
	const int* radii;
	const float* accum;      // [P, 12]
	const float* color_hint; // [P, 3] the forward's clamped colours (0 exactly where clamped), or NULL
} pbwd_scene;

} // extern "C"

namespace {

constexpr int NFIXED = 16; // mean 3 | cov 6 | scale 3 | rot 4 | sh 3 M
inline int nout(const pbwd_scene* s) { return NFIXED + (s->shs ? 3 * s->M : 0); }

// Branch assignment of the threshold decisions: -1 = the value's own, 0 = free / passes, 1 = clamped.
struct Branches {
	int x = -1, y = -1, c[3] = {-1, -1, -1};
};
// Which decisions lay inside their error band (only meaningful for Err).
struct Ambiguity {
	bool x = false, y = false, c[3] = {false, false, false};
};

template <class T>
void gaussian(const pbwd_scene* s, int idx, const Branches& br, T* out, Ambiguity* amb)
{
	const float* vw = s->view;
	const float* pj = s->proj;
	const float* acc = s->accum + 12 * (size_t)idx;
	const T fx = T(s->W / (2.0f * s->tanfovx)); // api.cu: focal lengths in fp32
	const T fy = T(s->H / (2.0f * s->tanfovy));
	const T d2x = T(acc[0]) * T(0.5f * s->W), d2y = T(acc[1]) * T(0.5f * s->H);
	const T dcx = T(-0.5f * acc[2]), dcy = T(-0.5f * acc[3]), dcz = T(-0.5f * acc[4]);
	const v3<T> mean = V3<T>(T(s->means3D[3 * idx]), T(s->means3D[3 * idx + 1]), T(s->means3D[3 * idx + 2]));
	for (int i = 0; i < nout(s); i++)
		out[i] = T(0.f);
	T* o_mean = out;
	T* o_cov = out + 3;
	T* o_scale = out + 9;
	T* o_rot = out + 12;
	T* o_sh = out + 16;

	// ---- 3D covariance (forward.cu:118-152 / computeCov3D) ----
	T cov3D[6];
	m3<T> R, M;
	v3<T> sv = V3<T>(T(0.f), T(0.f), T(0.f));
	T qr = T(0.f), qx = qr, qy = qr, qz = qr;
	if (s->cov3D_precomp) {
		for (int i = 0; i < 6; i++)
			cov3D[i] = T(s->cov3D_precomp[6 * (size_t)idx + i]);
	} else {
		const float* rot = s->rotations + 4 * (size_t)idx;
		const float* sc = s->scales + 3 * (size_t)idx;
		qr = T(rot[0]), qx = T(rot[1]), qy = T(rot[2]), qz = T(rot[3]);
		const T one = T(1.f), two = T(2.f);
		R = cols<T>(one - two * (qy * qy + qz * qz), two * (qx * qy - qr * qz), two * (qx * qz + qr * qy),
		            two * (qx * qy + qr * qz), one - two * (qx * qx + qz * qz), two * (qy * qz - qr * qx),
		            two * (qx * qz - qr * qy), two * (qy * qz + qr * qx), one - two * (qx * qx + qy * qy));
		const T mod = T(s->scale_modifier);
		sv = V3<T>(mod * T(sc[0]), mod * T(sc[1]), mod * T(sc[2]));
		m3<T> S = cols<T>(sv.x, T(0.f), T(0.f), T(0.f), sv.y, T(0.f), T(0.f), T(0.f), sv.z);
		M = mul(S, R);
		const m3<T> Sigma = mul(transpose(M), M);
		cov3D[0] = Sigma.m[0][0];
		cov3D[1] = Sigma.m[0][1];
		cov3D[2] = Sigma.m[0][2];
		cov3D[3] = Sigma.m[1][1];
		cov3D[4] = Sigma.m[1][2];
		cov3D[5] = Sigma.m[2][2];
	}

	// ---- cov2d_common + cov2d_backward (backward.cu:144-274) ----
	v3<T> t = V3<T>(T(vw[0]) * mean.x + T(vw[4]) * mean.y + T(vw[8]) * mean.z + T(vw[12]),
	                T(vw[1]) * mean.x + T(vw[5]) * mean.y + T(vw[9]) * mean.z + T(vw[13]),
	                T(vw[2]) * mean.x + T(vw[6]) * mean.y + T(vw[10]) * mean.z + T(vw[14]));
	const T limx = T(1.3f) * T(s->tanfovx), limy = T(1.3f) * T(s->tanfovy);
	const T txtz = t.x / t.z, tytz = t.y / t.z;
	// a clamp decision: outside = |t/t_z| > lim; inside the band of |t/t_z| - lim it may go either way
	auto decide = [](T r, T lim, int forced, bool* ambiguous) {
		const double band = err(r) + err(lim);
		*ambiguous = std::fabs(std::fabs(val(r)) - val(lim)) <= band;
		return forced >= 0 ? forced == 1 : (val(r) < -val(lim) || val(r) > val(lim));
	};
	const bool out_x = decide(txtz, limx, br.x, &amb->x), out_y = decide(tytz, limy, br.y, &amb->y);
	t.x = (out_x ? (val(txtz) < 0 ? -limx : limx) : txtz) * t.z;
	t.y = (out_y ? (val(tytz) < 0 ? -limy : limy) : tytz) * t.z;
	const T zero = T(0.f);
	const m3<T> J = cols<T>(fx / t.z, zero, -(fx * t.x) / (t.z * t.z), zero, fy / t.z, -(fy * t.y) / (t.z * t.z), zero, zero, zero);
	const m3<T> Wm = cols<T>(T(vw[0]), T(vw[4]), T(vw[8]), T(vw[1]), T(vw[5]), T(vw[9]), T(vw[2]), T(vw[6]), T(vw[10]));
	const m3<T> Tm = mul(Wm, J);
	const m3<T> Vrk = cols<T>(cov3D[0], cov3D[1], cov3D[2], cov3D[1], cov3D[3], cov3D[4], cov3D[2], cov3D[4], cov3D[5]);
	const m3<T> cov = mul(mul(transpose(Tm), transpose(Vrk)), Tm);

	const T x_grad_mul = out_x ? T(0.f) : T(1.f), y_grad_mul = out_y ? T(0.f) : T(1.f);
	const T a = cov.m[0][0] + T(0.3f), b = cov.m[0][1], cc = cov.m[1][1] + T(0.3f);
	const T denom = a * cc - b * b;
	const T two = T(2.f);
	const T denom2inv = T(1.0f) / ((denom * denom) + T(0.0000001f));
	const T dL_da = denom2inv * (-cc * cc * dcx + two * b * cc * dcy + (denom - a * cc) * dcz);
	const T dL_dc = denom2inv * (-a * a * dcz + two * a * b * dcy + (denom - a * cc) * dcx);
	const T dL_db = denom2inv * two * (b * cc * dcx - (denom + two * b * b) * dcy + a * b * dcz);
#define T_(i, j) Tm.m[i][j]
#define V_(i, j) Vrk.m[i][j]
#define W_(i, j) Wm.m[i][j]
	o_cov[0] = (T_(0, 0) * T_(0, 0) * dL_da + T_(0, 0) * T_(1, 0) * dL_db + T_(1, 0) * T_(1, 0) * dL_dc);
	o_cov[3] = (T_(0, 1) * T_(0, 1) * dL_da + T_(0, 1) * T_(1, 1) * dL_db + T_(1, 1) * T_(1, 1) * dL_dc);
	o_cov[5] = (T_(0, 2) * T_(0, 2) * dL_da + T_(0, 2) * T_(1, 2) * dL_db + T_(1, 2) * T_(1, 2) * dL_dc);
	o_cov[1] = two * T_(0, 0) * T_(0, 1) * dL_da + (T_(0, 0) * T_(1, 1) + T_(0, 1) * T_(1, 0)) * dL_db + two * T_(1, 0) * T_(1, 1) * dL_dc;
	o_cov[2] = two * T_(0, 0) * T_(0, 2) * dL_da + (T_(0, 0) * T_(1, 2) + T_(0, 2) * T_(1, 0)) * dL_db + two * T_(1, 0) * T_(1, 2) * dL_dc;
	o_cov[4] = two * T_(0, 2) * T_(0, 1) * dL_da + (T_(0, 1) * T_(1, 2) + T_(0, 2) * T_(1, 1)) * dL_db + two * T_(1, 1) * T_(1, 2) * dL_dc;
	const T dL_dT00 = two * (T_(0, 0) * V_(0, 0) + T_(0, 1) * V_(0, 1) + T_(0, 2) * V_(0, 2)) * dL_da + (T_(1, 0) * V_(0, 0) + T_(1, 1) * V_(0, 1) + T_(1, 2) * V_(0, 2)) * dL_db;
	const T dL_dT01 = two * (T_(0, 0) * V_(1, 0) + T_(0, 1) * V_(1, 1) + T_(0, 2) * V_(1, 2)) * dL_da + (T_(1, 0) * V_(1, 0) + T_(1, 1) * V_(1, 1) + T_(1, 2) * V_(1, 2)) * dL_db;
	const T dL_dT02 = two * (T_(0, 0) * V_(2, 0) + T_(0, 1) * V_(2, 1) + T_(0, 2) * V_(2, 2)) * dL_da + (T_(1, 0) * V_(2, 0) + T_(1, 1) * V_(2, 1) + T_(1, 2) * V_(2, 2)) * dL_db;
	const T dL_dT10 = two * (T_(1, 0) * V_(0, 0) + T_(1, 1) * V_(0, 1) + T_(1, 2) * V_(0, 2)) * dL_dc + (T_(0, 0) * V_(0, 0) + T_(0, 1) * V_(0, 1) + T_(0, 2) * V_(0, 2)) * dL_db;
	const T dL_dT11 = two * (T_(1, 0) * V_(1, 0) + T_(1, 1) * V_(1, 1) + T_(1, 2) * V_(1, 2)) * dL_dc + (T_(0, 0) * V_(1, 0) + T_(0, 1) * V_(1, 1) + T_(0, 2) * V_(1, 2)) * dL_db;
	const T dL_dT12 = two * (T_(1, 0) * V_(2, 0) + T_(1, 1) * V_(2, 1) + T_(1, 2) * V_(2, 2)) * dL_dc + (T_(0, 0) * V_(2, 0) + T_(0, 1) * V_(2, 1) + T_(0, 2) * V_(2, 2)) * dL_db;
	const T dL_dJ00 = W_(0, 0) * dL_dT00 + W_(0, 1) * dL_dT01 + W_(0, 2) * dL_dT02;
	const T dL_dJ02 = W_(2, 0) * dL_dT00 + W_(2, 1) * dL_dT01 + W_(2, 2) * dL_dT02;
	const T dL_dJ11 = W_(1, 0) * dL_dT10 + W_(1, 1) * dL_dT11 + W_(1, 2) * dL_dT12;
	const T dL_dJ12 = W_(2, 0) * dL_dT10 + W_(2, 1) * dL_dT11 + W_(2, 2) * dL_dT12;
#undef T_
#undef V_
#undef W_
	const T tz = T(1.f) / t.z, tz2 = tz * tz, tz3 = tz2 * tz;
	const T dL_dtx = x_grad_mul * -fx * tz2 * dL_dJ02;
	const T dL_dty = y_grad_mul * -fy * tz2 * dL_dJ12;
	const T dL_dtz = -fx * tz2 * dL_dJ00 - fy * tz2 * dL_dJ11 + (two * fx * t.x) * tz3 * dL_dJ02 + (two * fy * t.y) * tz3 * dL_dJ12;
	o_mean[0] = T(vw[0]) * dL_dtx + T(vw[1]) * dL_dty + T(vw[2]) * dL_dtz;
	o_mean[1] = T(vw[4]) * dL_dtx + T(vw[5]) * dL_dty + T(vw[6]) * dL_dtz;
	o_mean[2] = T(vw[8]) * dL_dtx + T(vw[9]) * dL_dty + T(vw[10]) * dL_dtz;

	// ---- means2D block of orc_backward_ex (backward.cu:346-396) ----
	{
		const T hw = T(pj[3]) * mean.x + T(pj[7]) * mean.y + T(pj[11]) * mean.z + T(pj[15]);
		const T m_w = T(1.0f) / (hw + T(0.0000001f));
		const T mul1 = (T(pj[0]) * mean.x + T(pj[4]) * mean.y + T(pj[8]) * mean.z + T(pj[12])) * m_w * m_w;
		const T mul2 = (T(pj[1]) * mean.x + T(pj[5]) * mean.y + T(pj[9]) * mean.z + T(pj[13])) * m_w * m_w;
		o_mean[0] += (T(pj[0]) * m_w - T(pj[3]) * mul1) * d2x + (T(pj[1]) * m_w - T(pj[3]) * mul2) * d2y;
		o_mean[1] += (T(pj[4]) * m_w - T(pj[7]) * mul1) * d2x + (T(pj[5]) * m_w - T(pj[7]) * mul2) * d2y;
		o_mean[2] += (T(pj[8]) * m_w - T(pj[11]) * mul1) * d2x + (T(pj[9]) * m_w - T(pj[11]) * mul2) * d2y;
		if (s->depth_gradient) {
			const T dz = T(acc[9]);
			o_mean[0] += T(vw[2]) * dz;
			o_mean[1] += T(vw[6]) * dz;
			o_mean[2] += T(vw[10]) * dz;
		}
	}

	// ---- sh_backward (backward.cu:20-139), clamp decision from computeColorFromSH_fwd (forward.cu:20-71) ----
	if (s->shs) {
		const int deg = s->D, Mc = s->M;
		const float* row = s->shs + (size_t)idx * Mc * 3;
		auto SH = [&](int k) { return V3<T>(T(row[3 * k]), T(row[3 * k + 1]), T(row[3 * k + 2])); };
		const v3<T> dir_orig = sub(mean, V3<T>(T(s->campos[0]), T(s->campos[1]), T(s->campos[2])));
		const T len = sqrt_(dot(dir_orig, dir_orig));
		const v3<T> dir = V3<T>(dir_orig.x / len, dir_orig.y / len, dir_orig.z / len);
		const T x = dir.x, y = dir.y, z = dir.z;
		// forward colour (the statements of computeColorFromSH_fwd) for the sign decision
		v3<T> rgb = scale(T(SH_C0), SH(0));
		if (deg > 0) {
			rgb = sub(add(sub(rgb, scale(T(SH_C1) * y, SH(1))), scale(T(SH_C1) * z, SH(2))), scale(T(SH_C1) * x, SH(3)));
			if (deg > 1) {
				const T xx = x * x, yy = y * y, zz = z * z, xy = x * y, yz = y * z, xz = x * z;
				rgb = add(rgb, scale(T(SH_C2[0]) * xy, SH(4)));
				rgb = add(rgb, scale(T(SH_C2[1]) * yz, SH(5)));
				rgb = add(rgb, scale(T(SH_C2[2]) * (T(2.0f) * zz - xx - yy), SH(6)));
				rgb = add(rgb, scale(T(SH_C2[3]) * xz, SH(7)));
				rgb = add(rgb, scale(T(SH_C2[4]) * (xx - yy), SH(8)));
				if (deg > 2) {
					rgb = add(rgb, scale(T(SH_C3[0]) * y * (T(3.0f) * xx - yy), SH(9)));
					rgb = add(rgb, scale(T(SH_C3[1]) * xy * z, SH(10)));
					rgb = add(rgb, scale(T(SH_C3[2]) * y * (T(4.0f) * zz - xx - yy), SH(11)));
					rgb = add(rgb, scale(T(SH_C3[3]) * z * (T(2.0f) * zz - T(3.0f) * xx - T(3.0f) * yy), SH(12)));
					rgb = add(rgb, scale(T(SH_C3[4]) * x * (T(4.0f) * zz - xx - yy), SH(13)));
					rgb = add(rgb, scale(T(SH_C3[5]) * z * (xx - yy), SH(14)));
					rgb = add(rgb, scale(T(SH_C3[6]) * x * (xx - T(3.0f) * yy), SH(15)));
				}
			}
		}
		const T ch[3] = {rgb.x + T(0.5f), rgb.y + T(0.5f), rgb.z + T(0.5f)};
		T up[3];
		for (int c = 0; c < 3; c++) {
			amb->c[c] = std::fabs(val(ch[c])) <= err(ch[c]);
			const bool clamped = br.c[c] >= 0 ? br.c[c] == 1 : val(ch[c]) < 0;
			up[c] = clamped ? T(0.f) : T(acc[6 + c]);
		}
		const v3<T> dL_dRGB = V3<T>(up[0], up[1], up[2]);
		v3<T> dRGBdx = V3<T>(zero, zero, zero), dRGBdy = dRGBdx, dRGBdz = dRGBdx;
		auto SET = [&](int k, T f) {
			const v3<T> g = scale(f, dL_dRGB);
			o_sh[3 * k] = g.x;
			o_sh[3 * k + 1] = g.y;
			o_sh[3 * k + 2] = g.z;
		};
		SET(0, T(SH_C0));
		if (deg > 0) {
			SET(1, T(-SH_C1) * y);
			SET(2, T(SH_C1) * z);
			SET(3, T(-SH_C1) * x);
			dRGBdx = scale(T(-SH_C1), SH(3));
			dRGBdy = scale(T(-SH_C1), SH(1));
			dRGBdz = scale(T(SH_C1), SH(2));
			if (deg > 1) {
				const T xx = x * x, yy = y * y, zz = z * z, xy = x * y, yz = y * z, xz = x * z;
				SET(4, T(SH_C2[0]) * xy);
				SET(5, T(SH_C2[1]) * yz);
				SET(6, T(SH_C2[2]) * (T(2.f) * zz - xx - yy));
				SET(7, T(SH_C2[3]) * xz);
				SET(8, T(SH_C2[4]) * (xx - yy));
				dRGBdx = add(dRGBdx, add(add(add(scale(T(SH_C2[0]) * y, SH(4)), scale(T(SH_C2[2]) * T(2.f) * -x, SH(6))), scale(T(SH_C2[3]) * z, SH(7))), scale(T(SH_C2[4]) * T(2.f) * x, SH(8))));
				dRGBdy = add(dRGBdy, add(add(add(scale(T(SH_C2[0]) * x, SH(4)), scale(T(SH_C2[1]) * z, SH(5))), scale(T(SH_C2[2]) * T(2.f) * -y, SH(6))), scale(T(SH_C2[4]) * T(2.f) * -y, SH(8))));
				dRGBdz = add(dRGBdz, add(add(scale(T(SH_C2[1]) * y, SH(5)), scale(T(SH_C2[2]) * T(2.f) * T(2.f) * z, SH(6))), scale(T(SH_C2[3]) * x, SH(7))));
				if (deg > 2) {
					SET(9, T(SH_C3[0]) * y * (T(3.f) * xx - yy));
					SET(10, T(SH_C3[1]) * xy * z);
					SET(11, T(SH_C3[2]) * y * (T(4.f) * zz - xx - yy));
					SET(12, T(SH_C3[3]) * z * (T(2.f) * zz - T(3.f) * xx - T(3.f) * yy));
					SET(13, T(SH_C3[4]) * x * (T(4.f) * zz - xx - yy));
					SET(14, T(SH_C3[5]) * z * (xx - yy));
					SET(15, T(SH_C3[6]) * x * (xx - T(3.f) * yy));
					v3<T> ax = V3<T>(zero, zero, zero), ay = ax, az = ax;
					ax = add(ax, scale(T(SH_C3[0]) * T(3.f) * T(2.f) * xy, SH(9)));
					ax = add(ax, scale(T(SH_C3[1]) * yz, SH(10)));
					ax = add(ax, scale(T(SH_C3[2]) * T(-2.f) * xy, SH(11)));
					ax = add(ax, scale(T(SH_C3[3]) * T(-3.f) * T(2.f) * xz, SH(12)));
					ax = add(ax, scale(T(SH_C3[4]) * (T(-3.f) * xx + T(4.f) * zz - yy), SH(13)));
					ax = add(ax, scale(T(SH_C3[5]) * T(2.f) * xz, SH(14)));
					ax = add(ax, scale(T(SH_C3[6]) * T(3.f) * (xx - yy), SH(15)));
					ay = add(ay, scale(T(SH_C3[0]) * T(3.f) * (xx - yy), SH(9)));
					ay = add(ay, scale(T(SH_C3[1]) * xz, SH(10)));
					ay = add(ay, scale(T(SH_C3[2]) * (T(-3.f) * yy + T(4.f) * zz - xx), SH(11)));
					ay = add(ay, scale(T(SH_C3[3]) * T(-3.f) * T(2.f) * yz, SH(12)));
					ay = add(ay, scale(T(SH_C3[4]) * T(-2.f) * xy, SH(13)));
					ay = add(ay, scale(T(SH_C3[5]) * T(-2.f) * yz, SH(14)));
					ay = add(ay, scale(T(SH_C3[6]) * T(-3.f) * T(2.f) * xy, SH(15)));
					az = add(az, scale(T(SH_C3[1]) * xy, SH(10)));
					az = add(az, scale(T(SH_C3[2]) * T(4.f) * T(2.f) * yz, SH(11)));
					az = add(az, scale(T(SH_C3[3]) * T(3.f) * (T(2.f) * zz - xx - yy), SH(12)));
					az = add(az, scale(T(SH_C3[4]) * T(4.f) * T(2.f) * xz, SH(13)));
					az = add(az, scale(T(SH_C3[5]) * (xx - yy), SH(14)));
					dRGBdx = add(dRGBdx, ax);
					dRGBdy = add(dRGBdy, ay);
					dRGBdz = add(dRGBdz, az);
				}
			}
		}
		const v3<T> dv = V3<T>(dot(dRGBdx, dL_dRGB), dot(dRGBdy, dL_dRGB), dot(dRGBdz, dL_dRGB));
		// dnormvdv (auxiliary.h:107-117)
		const v3<T> v = dir_orig;
		const T sum2 = v.x * v.x + v.y * v.y + v.z * v.z;
		const T invsum32 = T(1.0f) / sqrt_(sum2 * sum2 * sum2);
		o_mean[0] += ((sum2 - v.x * v.x) * dv.x - v.y * v.x * dv.y - v.z * v.x * dv.z) * invsum32;
		o_mean[1] += (-v.x * v.y * dv.x + (sum2 - v.y * v.y) * dv.y - v.z * v.y * dv.z) * invsum32;
		o_mean[2] += (-v.x * v.z * dv.x - v.y * v.z * dv.y + (sum2 - v.z * v.z) * dv.z) * invsum32;
	}

	// ---- cov3d_backward (backward.cu:278-341) ----
	if (!s->cov3D_precomp) {
		const T* d = o_cov;
		const T h = T(0.5f);
		const m3<T> dL_dSigma = cols<T>(d[0], h * d[1], h * d[2], h * d[1], d[3], h * d[4], h * d[2], h * d[4], d[5]);
		m3<T> M2 = M;
		for (int i = 0; i < 3; i++)
			for (int j = 0; j < 3; j++)
				M2.m[i][j] = M.m[i][j] * T(2.0f);
		const m3<T> dL_dM = mul(M2, dL_dSigma);
		const m3<T> Rt = transpose(R);
		m3<T> dMt = transpose(dL_dM);
		o_scale[0] = Rt.m[0][0] * dMt.m[0][0] + Rt.m[0][1] * dMt.m[0][1] + Rt.m[0][2] * dMt.m[0][2];
		o_scale[1] = Rt.m[1][0] * dMt.m[1][0] + Rt.m[1][1] * dMt.m[1][1] + Rt.m[1][2] * dMt.m[1][2];
		o_scale[2] = Rt.m[2][0] * dMt.m[2][0] + Rt.m[2][1] * dMt.m[2][1] + Rt.m[2][2] * dMt.m[2][2];
		for (int k = 0; k < 3; k++) {
			dMt.m[0][k] *= sv.x;
			dMt.m[1][k] *= sv.y;
			dMt.m[2][k] *= sv.z;
		}
#define MT(i, j) dMt.m[i][j]
		const T four = T(4.f);
		o_rot[0] = two * qz * (MT(0, 1) - MT(1, 0)) + two * qy * (MT(2, 0) - MT(0, 2)) + two * qx * (MT(1, 2) - MT(2, 1));
		o_rot[1] = two * qy * (MT(1, 0) + MT(0, 1)) + two * qz * (MT(2, 0) + MT(0, 2)) + two * qr * (MT(1, 2) - MT(2, 1)) - four * qx * (MT(2, 2) + MT(1, 1));
		o_rot[2] = two * qx * (MT(1, 0) + MT(0, 1)) + two * qr * (MT(2, 0) - MT(0, 2)) + two * qz * (MT(1, 2) + MT(2, 1)) - four * qy * (MT(2, 2) + MT(0, 0));
		o_rot[3] = two * qr * (MT(0, 1) - MT(1, 0)) + two * qx * (MT(2, 0) + MT(0, 2)) + two * qy * (MT(1, 2) + MT(2, 1)) - four * qz * (MT(1, 1) + MT(0, 0));
#undef MT
	}
}

// The colour decision of channel c, restricted by the forward's own colour where the value is inside its band:
// a colour > 0 means the gradient passed; exactly 0 means clamped or rgb == 0 exactly, so both stay possible.
void colour_options(const pbwd_scene* s, int idx, int c, bool ambiguous, int* opts, int* n)
{
	*n = 0;
	if (!ambiguous) {
		opts[(*n)++] = -1;
		return;
	}
	if (s->color_hint && s->color_hint[3 * (size_t)idx + c] > 0.f) {
		opts[(*n)++] = 0;
		return;
	}
	opts[(*n)++] = 0;
	opts[(*n)++] = 1;
}

} // namespace

extern "C" {

int pbwd_nout(const pbwd_scene* s) { return nout(s); }

// kind 0: double values; 1: float values; 2: values and bounds (Err).  Default branches (each decision from the
// evaluating type's own value).  flags[i]: bit 0 invisible, bit 1 excluded by the division rule, bit 2 a decision
// inside its band (Err only).
void pbwd_eval(const pbwd_scene* s, int kind, double* val_out, double* err_out, int* flags)
{
	const int n = nout(s);
	for (int i = 0; i < s->P; i++) {
		double* vo = val_out + (size_t)i * n;
		flags[i] = 0;
		if (!(s->radii[i] > 0)) {
			flags[i] = 1;
			for (int k = 0; k < n; k++) {
				vo[k] = 0;
				if (err_out) err_out[(size_t)i * n + k] = 0;
			}
			continue;
		}
		Ambiguity amb;
		Branches br;
		if (kind == 0) {
			double o[NFIXED + 48];
			gaussian<double>(s, i, br, o, &amb);
			for (int k = 0; k < n; k++) vo[k] = o[k];
		} else if (kind == 1) {
			float o[NFIXED + 48];
			gaussian<float>(s, i, br, o, &amb);
			for (int k = 0; k < n; k++) vo[k] = o[k];
		} else {
			Err o[NFIXED + 48];
			t_div_invalid = false;
			gaussian<Err>(s, i, br, o, &amb);
			for (int k = 0; k < n; k++) {
				vo[k] = o[k].v;
				err_out[(size_t)i * n + k] = o[k].e;
			}
			if (t_div_invalid) flags[i] |= 2;
			if (amb.x || amb.y || amb.c[0] || amb.c[1] || amb.c[2]) flags[i] |= 4;
		}
	}
}

// got [P, nout] (float).  For every visible Gaussian: ratio[i] = the smallest, over the branch assignments its
// ambiguous decisions allow, of max_k |got - ref| / (K e + u |ref| + slack) (0/0 counts as 0, a NaN as infinity);
// slack [P, nout] or NULL: an error the comparison itself adds (a difference of two rounded sums);
// elem[i] the element of that maximum.  status[i]: 0 checked, 1 resolved (more than one branch assignment was
// possible), 2 excluded (division rule), 3 invisible (not checked here).
void pbwd_check(const pbwd_scene* s, const float* got, const double* slack, double K, double* ratio, int* elem,
                int* status)
{
	const int n = nout(s);
	for (int i = 0; i < s->P; i++) {
		ratio[i] = 0;
		elem[i] = -1;
		if (!(s->radii[i] > 0)) {
			status[i] = 3;
			continue;
		}
		Ambiguity amb;
		Err o[NFIXED + 48];
		t_div_invalid = false;
		gaussian<Err>(s, i, Branches{}, o, &amb);
		if (t_div_invalid) {
			status[i] = 2;
			continue;
		}
		int xo[2] = {-1, -1}, yo[2] = {-1, -1}, co[3][2], nx = 1, ny = 1, nc[3];
		if (amb.x) { xo[0] = 0; xo[1] = 1; nx = 2; }
		if (amb.y) { yo[0] = 0; yo[1] = 1; ny = 2; }
		for (int c = 0; c < 3; c++) colour_options(s, i, c, s->shs && amb.c[c], co[c], &nc[c]);
		const int combos = nx * ny * nc[0] * nc[1] * nc[2];
		status[i] = combos > 1 ? 1 : 0;
		const float* g = got + (size_t)i * n;
		const double* sl = slack ? slack + (size_t)i * n : nullptr;
		double best = INFINITY;
		int best_k = -1;
		for (int ix = 0; ix < nx; ix++)
			for (int iy = 0; iy < ny; iy++)
				for (int i0 = 0; i0 < nc[0]; i0++)
					for (int i1 = 0; i1 < nc[1]; i1++)
						for (int i2 = 0; i2 < nc[2]; i2++) {
							Branches br;
							br.x = xo[ix];
							br.y = yo[iy];
							br.c[0] = co[0][i0];
							br.c[1] = co[1][i1];
							br.c[2] = co[2][i2];
							Ambiguity unused;
							if (combos > 1) gaussian<Err>(s, i, br, o, &unused);
							double worst = 0;
							int wk = -1;
							for (int k = 0; k < n; k++) {
								const double d = std::fabs((double)g[k] - o[k].v);
								const double tol = K * o[k].e + U * std::fabs(o[k].v) + (sl ? sl[k] : 0.0);
								double r = d == 0 ? 0 : (tol > 0 ? d / tol : INFINITY);
								if (std::isnan(r)) r = INFINITY;
								if (wk < 0 || r > worst) { worst = r; wk = k; }
							}
							if (worst < best) { best = worst; best_k = wk; }
						}
		ratio[i] = best;
		elem[i] = best_k;
	}
}

} // extern "C"

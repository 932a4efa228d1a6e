/*
 * spp_oracle.c -- TEST INFRASTRUCTURE ONLY. CPU restatement (plain C, scalar, single thread) of the
 * reference's algorithm for the NLS hot path. It is the checker of tests/ and of __graft_entry__.smoke(), and
 * the "port" CPU baseline of bench.py; it is never linked into or called by the product (libspp_b200.so).
 *
 * PARITY PINNED: validated against the unmodified reference compiled from /root/reference (oracle/_ref, built
 * by oracle/build_ref.sh) through the golden vectors in tests/golden/*.npz (tests/test_oracle_cpu.py):
 * chi2 to 1e-12, lambda / eta at the forward-difference noise floor, Schur increments to 1e-11, LM traces.
 *
 * Every function cites the reference code it follows (paths relative to the SLAM++ tree):
 *   3D  = include/slam/3DSolverBase.h        BA   = include/slam/BASolverBase.h
 *   BAT = include/slam/BA_Types.h            BIN  = include/slam/BaseTypes_Binary.h
 *   LM  = include/slam/NonlinearSolver_Lambda_LM.h
 *   SCH = include/slam/LinearSolver_Schur.h  SCC  = src/slam/LinearSolver_Schur.cpp
 *   LB  = include/slam/NonlinearSolver_Lambda_Base.h
 * Where the reference calls Eigen (quaternion product, _transformVector, toRotationMatrix, 3x3 inverse,
 * LLT<Upper>) the published Eigen algorithm is written out.
 */
#define _GNU_SOURCE
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#ifndef M_PI
#define M_PI 3.14159265358979323846
#endif

#define SPO_API __attribute__((visibility("default")))

typedef struct { double w, x, y, z; } quat_t;

/* ---- SE(3) helpers ------------------------------------------------------------------------------ */

static void quat_normalize(quat_t *q)
{
	double n = sqrt(q->x * q->x + q->y * q->y + q->z * q->z + q->w * q->w);
	q->x /= n; q->y /= n; q->z /= n; q->w /= n;
}

/* C3DJacobians::f_AxisAngle_to_Quat, 3D:476-519 */
static void axis_angle_to_quat(const double *a, quat_t *q)
{
	double f_angle = sqrt(a[0] * a[0] + a[1] * a[1] + a[2] * a[2]);
	if(f_angle < 1e-12) {
		q->w = cos(f_angle * .5);
		q->x = a[0] * .5; q->y = a[1] * .5; q->z = a[2] * .5;
		quat_normalize(q);
	} else {
		double f_half_angle = f_angle * .5;
		double c = cos(f_half_angle);
		double f_q = sin(f_half_angle) / f_angle;
		if(c < 0) {
			c = -c;
			f_q = -f_q;
		}
		q->w = c;
		q->x = a[0] * f_q; q->y = a[1] * f_q; q->z = a[2] * f_q;
		if(c > 1 - 1e-6)
			quat_normalize(q);
	}
}

/* C3DJacobians::f_Quat_to_AxisAngle, 3D:556-649 (the compiled-in "norm and atan and atan2" branch) */
static void quat_to_axis_angle(const quat_t *q, double *a)
{
	const double f_w = q->w;
	const double f_abs_w = fabs(f_w), f_norm = sqrt(q->x * q->x + q->y * q->y + q->z * q->z);
	const double f_abs_half = (f_abs_w > 1e-3)? atan(f_norm / f_abs_w) : atan2(f_norm, f_abs_w);
	const double f_half = copysign(f_abs_half, f_w);
	if(f_norm < 1e-12) {
		a[0] = q->x * 2.0; a[1] = q->y * 2.0; a[2] = q->z * 2.0;
	} else {
		double f_s = f_half * 2 / f_norm;
		a[0] = q->x * f_s; a[1] = q->y * f_s; a[2] = q->z * f_s;
	}
}

/* Eigen quaternion product */
static quat_t quat_mul(const quat_t *a, const quat_t *b)
{
	quat_t r;
	r.w = a->w * b->w - a->x * b->x - a->y * b->y - a->z * b->z;
	r.x = a->w * b->x + a->x * b->w + a->y * b->z - a->z * b->y;
	r.y = a->w * b->y + a->y * b->w + a->z * b->x - a->x * b->z;
	r.z = a->w * b->z + a->z * b->w + a->x * b->y - a->y * b->x;
	return r;
}

/* Eigen QuaternionBase::_transformVector */
static void quat_rotate(const quat_t *q, const double *v, double *r)
{
	double ux = q->y * v[2] - q->z * v[1], uy = q->z * v[0] - q->x * v[2], uz = q->x * v[1] - q->y * v[0];
	ux += ux; uy += uy; uz += uz;
	r[0] = v[0] + q->w * ux + (q->y * uz - q->z * uy);
	r[1] = v[1] + q->w * uy + (q->z * ux - q->x * uz);
	r[2] = v[2] + q->w * uz + (q->x * uy - q->y * ux);
}

/* Eigen QuaternionBase::toRotationMatrix, row-major */
static void quat_to_rotmat(const quat_t *q, double *R)
{
	const double tx = 2 * q->x, ty = 2 * q->y, tz = 2 * q->z;
	const double twx = tx * q->w, twy = ty * q->w, twz = tz * q->w;
	const double txx = tx * q->x, txy = ty * q->x, txz = tz * q->x;
	const double tyy = ty * q->y, tyz = tz * q->y, tzz = tz * q->z;
	R[0] = 1 - (tyy + tzz); R[1] = txy - twz; R[2] = txz + twy;
	R[3] = txy + twz; R[4] = 1 - (txx + tzz); R[5] = tyz - twx;
	R[6] = txz - twy; R[7] = tyz + twx; R[8] = 1 - (txx + tyy);
}

/* C3DJacobians::Relative_to_Absolute, 3D:806-849 */
static void relative_to_absolute(const double *v1, const double *v2, double *dest)
{
	quat_t q1, q2, q;
	double r[3], t[6];
	axis_angle_to_quat(v1 + 3, &q1);
	axis_angle_to_quat(v2 + 3, &q2);
	quat_rotate(&q1, v2, r);
	t[0] = v1[0] + r[0]; t[1] = v1[1] + r[1]; t[2] = v1[2] + r[2];
	q = quat_mul(&q1, &q2);
	quat_to_axis_angle(&q, t + 3);
	memcpy(dest, t, sizeof(t));
}

/* CBAJacobians::Project_P2C (value), BA:260-327 */
static void project_p2c(const double *cam, const double *intr, const double *X, double *uv)
{
	double fx = intr[0], fy = intr[1], cx = intr[2], cy = intr[3];
	double k = intr[4] / (.5 * (fx + fy));
	quat_t q;
	double R[9];
	axis_angle_to_quat(cam + 3, &q); /* t_AxisAngle_to_RotMatrix, 3D:292-299 */
	quat_to_rotmat(&q, R);
	double x0 = R[0] * X[0] + R[1] * X[1] + R[2] * X[2] + cam[0];
	double x1 = R[3] * X[0] + R[4] * X[1] + R[5] * X[2] + cam[1];
	double x2 = R[6] * X[0] + R[7] * X[1] + R[8] * X[2] + cam[2];
	double u0 = fx * x0 + cx * x2, u1 = fy * x1 + cy * x2;
	u0 /= x2; u1 /= x2;
	double dx = u0 - cx, dy = u1 - cy;
	double r = sqrt(dx * dx + dy * dy);
	double f_s = 1 + r * r * k;
	uv[0] = cx + f_s * dx;
	uv[1] = cy + f_s * dy;
}

/* CBAJacobians::Project_P2C (with Jacobians), BA:559-619: forward differences, delta = 1e-9.
 * H1: 2x6 row-major, H2: 2x3 row-major */
static void project_p2c_jacobians(const double *cam, const double *intr, const double *X, double *uv,
	double *H1, double *H2)
{
	const double delta = 1e-9;
	const double scalar = 1.0 / (delta);
	double d1[2];
	project_p2c(cam, intr, X, uv);
	for(int j = 0; j < 6; ++ j) {
		double eps[6] = {0, 0, 0, 0, 0, 0}, p_delta[6];
		eps[j] = delta;
		relative_to_absolute(cam, eps, p_delta);
		project_p2c(p_delta, intr, X, d1);
		H1[j] = (d1[0] - uv[0]) * scalar;
		H1[6 + j] = (d1[1] - uv[1]) * scalar;
	}
	for(int j = 0; j < 3; ++ j) {
		double Xd[3] = {X[0], X[1], X[2]}; /* Relative_to_Absolute_XYZ, BA:167-175 */
		Xd[j] += delta;
		project_p2c(cam, intr, Xd, d1);
		H2[j] = (d1[0] - uv[0]) * scalar;
		H2[3 + j] = (d1[1] - uv[1]) * scalar;
	}
}

/* ---- graph bookkeeping ---------------------------------------------------------------------------- */

typedef struct {
	size_t nv, C, P, O;
	const uint8_t *vtype;
	uint32_t *local;   /* vertex id -> camera / point index */
	double *cam;       /* C x 6 (state) */
	double *intr;      /* C x 5 */
	double *pt;        /* P x 3 */
	const uint64_t *obs_pt, *obs_cam;
	const double *z, *info;
} ba_t;

static int ba_init(ba_t *g, size_t nv, const uint8_t *vtype, const double *cams11, const double *pts, size_t no,
	const uint64_t *obs_pt, const uint64_t *obs_cam, const double *z, const double *info)
{
	memset(g, 0, sizeof(*g));
	g->nv = nv; g->vtype = vtype; g->O = no; g->obs_pt = obs_pt; g->obs_cam = obs_cam; g->z = z; g->info = info;
	g->local = (uint32_t*)malloc((nv + 1) * sizeof(uint32_t));
	for(size_t v = 0; v < nv; ++ v)
		g->local[v] = (uint32_t)((vtype[v] == 0)? g->C ++ : g->P ++);
	g->cam = (double*)malloc((g->C + 1) * 6 * sizeof(double));
	g->intr = (double*)malloc((g->C + 1) * 5 * sizeof(double));
	g->pt = (double*)malloc((g->P + 1) * 3 * sizeof(double));
	for(size_t c = 0; c < g->C; ++ c) {
		memcpy(g->cam + c * 6, cams11 + c * 11, 6 * sizeof(double));
		memcpy(g->intr + c * 5, cams11 + c * 11 + 6, 5 * sizeof(double));
	}
	memcpy(g->pt, pts, g->P * 3 * sizeof(double));
	for(size_t e = 0; e < no; ++ e) {
		if(obs_pt[e] >= nv || obs_cam[e] >= nv || vtype[obs_pt[e]] != 1 || vtype[obs_cam[e]] != 0)
			return -1;
	}
	return 0;
}

static void ba_free(ba_t *g)
{
	free(g->local); free(g->cam); free(g->intr); free(g->pt);
}

/* CEdgeP2C3D::f_Chi_Squared_Error summed serially in edge order, BAT:511-531, NonlinearSolver_Base.h:278-297 */
static double ba_chi2(const ba_t *g)
{
	double f_chi2 = 0;
	for(size_t e = 0; e < g->O; ++ e) {
		const double *cam = g->cam + (size_t)g->local[g->obs_cam[e]] * 6;
		const double *intr = g->intr + (size_t)g->local[g->obs_cam[e]] * 5;
		const double *X = g->pt + (size_t)g->local[g->obs_pt[e]] * 3;
		const double *S = g->info + e * 4;
		double uv[2];
		project_p2c(cam, intr, X, uv);
		double eu = uv[0] - g->z[e * 2], ev = uv[1] - g->z[e * 2 + 1];
		f_chi2 += (eu * S[0] + ev * S[2]) * eu + (eu * S[1] + ev * S[3]) * ev;
	}
	return f_chi2;
}

/* Refresh_Lambda: per-edge Calculate_Hessians_v2 (BIN:759-848) + the reduction plan (LB:152-197, 563-607): every
 * destination block is the sum of its per-edge sources in edge insertion order; the unary factor UF^T UF = I of
 * vertex 0 (FlatSystem.h:432-473, LB:1903-1923) is one more source of that vertex's diagonal block.
 * U: C x 36 (col-major 6x6), V: P x 9, W: O x 18 (col-major 6x3 = J_cam^T Sigma^-1 J_pt, edge order),
 * gc: C x 6, gp: P x 3. Returns the largest per-edge diagonal entry (LM:162-166, BIN:1200-1224). */
static double ba_linearise(const ba_t *g, double *U, double *V, double *W, double *gc, double *gp)
{
	double f_max_diag = 0;
	memset(U, 0, g->C * 36 * sizeof(double));
	memset(V, 0, g->P * 9 * sizeof(double));
	memset(gc, 0, g->C * 6 * sizeof(double));
	memset(gp, 0, g->P * 3 * sizeof(double));
	if(g->nv) {
		if(g->vtype[0] == 0) { for(int i = 0; i < 6; ++ i) U[i * 7] += 1.0; }
		else { for(int i = 0; i < 3; ++ i) V[i * 4] += 1.0; }
	}
	for(size_t e = 0; e < g->O; ++ e) {
		const size_t c = g->local[g->obs_cam[e]], p = g->local[g->obs_pt[e]];
		const double *S = g->info + e * 4;
		double uv[2], J0[12], J1[6], r[2];
		project_p2c_jacobians(g->cam + c * 6, g->intr + c * 5, g->pt + p * 3, uv, J0, J1);
		r[0] = g->z[e * 2] - uv[0]; /* BAT:503 */
		r[1] = g->z[e * 2 + 1] - uv[1];
		double T[12]; /* t_H0_sigma_inv = J0^T Sigma^-1 (6x2), BIN:774; T[j*2 + k] */
		for(int j = 0; j < 6; ++ j) {
			T[j * 2] = J0[j] * S[0] + J0[6 + j] * S[2];
			T[j * 2 + 1] = J0[j] * S[1] + J0[6 + j] * S[3];
		}
		double *We = W + e * 18; /* off-diagonal block, BIN:805 */
		for(int cc = 0; cc < 3; ++ cc)
			for(int j = 0; j < 6; ++ j)
				We[cc * 6 + j] = T[j * 2] * J1[cc] + T[j * 2 + 1] * J1[3 + cc];
		/* vertex 0 diagonal source = selfadjointView<Upper>(T J0), BIN:813; rhs = T r, BIN:823 */
		for(int cc = 0; cc < 6; ++ cc) {
			for(int rr = 0; rr <= cc; ++ rr) {
				double v = T[rr * 2] * J0[cc] + T[rr * 2 + 1] * J0[6 + cc];
				U[c * 36 + cc * 6 + rr] += v;
				if(rr != cc)
					U[c * 36 + rr * 6 + cc] += v;
				else if(v > f_max_diag)
					f_max_diag = v;
			}
		}
		for(int j = 0; j < 6; ++ j)
			gc[c * 6 + j] += T[j * 2] * r[0] + T[j * 2 + 1] * r[1];
		/* vertex 1 diagonal source = selfadjointView<Upper>(J1^T Sigma^-1 J1), BIN:831; rhs = J1^T (Sigma^-1 r), BIN:845 */
		double A[6];
		for(int j = 0; j < 3; ++ j) {
			A[j * 2] = J1[j] * S[0] + J1[3 + j] * S[2];
			A[j * 2 + 1] = J1[j] * S[1] + J1[3 + j] * S[3];
		}
		for(int cc = 0; cc < 3; ++ cc) {
			for(int rr = 0; rr <= cc; ++ rr) {
				double v = A[rr * 2] * J1[cc] + A[rr * 2 + 1] * J1[3 + cc];
				V[p * 9 + cc * 3 + rr] += v;
				if(rr != cc)
					V[p * 9 + rr * 3 + cc] += v;
				else if(v > f_max_diag)
					f_max_diag = v;
			}
		}
		double s0 = S[0] * r[0] + S[1] * r[1], s1 = S[2] * r[0] + S[3] * r[1];
		for(int j = 0; j < 3; ++ j)
			gp[p * 3 + j] += J1[j] * s0 + J1[3 + j] * s1;
	}
	return f_max_diag;
}

/* ---- dense Cholesky: Eigen::LLT<MatrixXd, Upper> + solve, SCC:2314-2333 ------------------------------- */

/* A: n x n column-major, upper triangle read and overwritten by R (A = R^T R). Returns 0, or k + 1 when pivot k
 * is not positive (Eigen's llt_inplace returns the index of the failing column; the reference returns false). */
static int dense_llt_upper(size_t n, double *A)
{
	for(size_t j = 0; j < n; ++ j) {
		double d = A[j * n + j];
		for(size_t k = 0; k < j; ++ k)
			d -= A[j * n + k] * A[j * n + k];
		if(!(d > 0))
			return (int)j + 1;
		d = sqrt(d);
		A[j * n + j] = d;
		for(size_t c = j + 1; c < n; ++ c) {
			double s = A[c * n + j];
			for(size_t k = 0; k < j; ++ k)
				s -= A[j * n + k] * A[c * n + k];
			A[c * n + j] = s / d;
		}
	}
	return 0;
}

static void dense_llt_solve(size_t n, const double *R, double *b)
{
	for(size_t i = 0; i < n; ++ i) { /* R^T y = b */
		double s = b[i];
		for(size_t k = 0; k < i; ++ k)
			s -= R[i * n + k] * b[k];
		b[i] = s / R[i * n + i];
	}
	for(size_t i = n; i -- > 0;) { /* R x = y */
		double s = b[i];
		for(size_t k = i + 1; k < n; ++ k)
			s -= R[k * n + i] * b[k];
		b[i] = s / R[i * n + i];
	}
}

/* ---- Schur complement solve, SCH:1623-1935 ---------------------------------------------------------------- */

/* Eigen fixed-size 3x3 inverse (cofactors / determinant), BlockMatrixBase.h:1256-1270; column-major in and out */
static void inverse3(const double *m, double *inv)
{
	double m00 = m[0], m10 = m[1], m20 = m[2], m01 = m[3], m11 = m[4], m21 = m[5], m02 = m[6], m12 = m[7], m22 = m[8];
	double c00 = m11 * m22 - m12 * m21, c10 = m21 * m02 - m22 * m01, c20 = m01 * m12 - m02 * m11;
	double det = c00 * m00 + c10 * m10 + c20 * m20;
	double id = 1.0 / det;
	inv[0] = c00 * id; inv[3] = c10 * id; inv[6] = c20 * id;
	inv[1] = (m12 * m20 - m10 * m22) * id; inv[4] = (m22 * m00 - m20 * m02) * id; inv[7] = (m02 * m10 - m00 * m12) * id;
	inv[2] = (m10 * m21 - m11 * m20) * id; inv[5] = (m20 * m01 - m21 * m00) * id; inv[8] = (m00 * m11 - m01 * m10) * id;
}

/* Solves (lambda + alpha I) dx = eta for lambda = [U W; W^T V] in the guided Schur ordering (cameras first, points
 * after, id order kept: SCC:771-838). obs_c / obs_p: camera / point index per observation, edge order.
 * Stages follow SCH:1687-1886: C^-1 (SCH:1720-1735), Y = U_offdiag C^-1 (SCH:1743-1745), S = A - Y V accumulated
 * per destination block in ascending landmark order (SCH:1757-1767, BlockMatrixFBS.h:395-448), reduced rhs
 * (SCH:1829-1830), dense LLT (SCH:1842), back-substitution (SCH:1867-1881).
 * S_out (n x n col-major, upper valid) and rhs_out (n) are optional. Returns 0, 1 = not positive definite. */
static int schur_solve(size_t C, size_t P, size_t O, const uint32_t *obs_c, const uint32_t *obs_p, const double *U,
	const double *V, const double *W, const double *gc, const double *gp, double alpha, double *dxc, double *dxp,
	double *S_out, double *rhs_out)
{
	const size_t n = 6 * C;
	double *Cinv = (double*)malloc((P + 1) * 9 * sizeof(double));
	double *Y = (double*)malloc((O + 1) * 18 * sizeof(double));
	double *S = (double*)calloc(n * n + 1, sizeof(double));
	double *b = (double*)malloc((n + 1) * sizeof(double));
	/* observations of every landmark, in edge order */
	uint32_t *ptr = (uint32_t*)calloc(P + 2, sizeof(uint32_t)), *lst = (uint32_t*)malloc((O + 1) * sizeof(uint32_t));
	for(size_t e = 0; e < O; ++ e) ++ ptr[obs_p[e] + 1];
	for(size_t p = 0; p < P; ++ p) ptr[p + 1] += ptr[p];
	{
		uint32_t *fill = (uint32_t*)malloc((P + 1) * sizeof(uint32_t));
		memcpy(fill, ptr, P * sizeof(uint32_t));
		for(size_t e = 0; e < O; ++ e) lst[fill[obs_p[e]] ++] = (uint32_t)e;
		free(fill);
	}
	for(size_t p = 0; p < P; ++ p) {
		double m[9];
		memcpy(m, V + p * 9, sizeof(m));
		m[0] += alpha; m[4] += alpha; m[8] += alpha; /* Apply_Damping, LM:228-239 */
		inverse3(m, Cinv + p * 9);
	}
	for(size_t e = 0; e < O; ++ e) {
		const double *w = W + e * 18, *ci = Cinv + (size_t)obs_p[e] * 9;
		double *y = Y + e * 18;
		for(int cc = 0; cc < 3; ++ cc)
			for(int r = 0; r < 6; ++ r)
				y[cc * 6 + r] = w[r] * ci[cc * 3] + w[6 + r] * ci[cc * 3 + 1] + w[12 + r] * ci[cc * 3 + 2];
	}
	for(size_t c = 0; c < C; ++ c) {
		for(int cc = 0; cc < 6; ++ cc)
			for(int r = 0; r < 6; ++ r)
				S[(c * 6 + cc) * n + c * 6 + r] = U[c * 36 + cc * 6 + r] + ((r == cc)? alpha : 0.0);
		for(int r = 0; r < 6; ++ r)
			b[c * 6 + r] = gc[c * 6 + r];
	}
	for(size_t p = 0; p < P; ++ p) { /* ascending landmark order */
		for(uint32_t ia = ptr[p]; ia < ptr[p + 1]; ++ ia) {
			const uint32_t ea = lst[ia], ca = obs_c[ea];
			const double *y = Y + (size_t)ea * 18;
			for(int r = 0; r < 6; ++ r)
				b[ca * 6 + r] -= y[r] * gp[p * 3] + y[6 + r] * gp[p * 3 + 1] + y[12 + r] * gp[p * 3 + 2];
			for(uint32_t ib = ptr[p]; ib < ptr[p + 1]; ++ ib) {
				const uint32_t eb = lst[ib], cb = obs_c[eb];
				if(!(ca < cb || ea == eb))
					continue; /* upper triangle only */
				const double *w = W + (size_t)eb * 18;
				for(int cc = 0; cc < 6; ++ cc)
					for(int r = 0; r < 6; ++ r)
						S[((size_t)cb * 6 + cc) * n + (size_t)ca * 6 + r] -=
							y[r] * w[cc] + y[6 + r] * w[6 + cc] + y[12 + r] * w[12 + cc];
			}
		}
	}
	if(S_out) memcpy(S_out, S, n * n * sizeof(double));
	if(rhs_out) memcpy(rhs_out, b, n * sizeof(double));
	int rc = dense_llt_upper(n, S);
	if(!rc) {
		dense_llt_solve(n, S, b);
		memcpy(dxc, b, n * sizeof(double));
		for(size_t p = 0; p < P; ++ p) {
			double l[3] = {gp[p * 3], gp[p * 3 + 1], gp[p * 3 + 2]};
			for(uint32_t ia = ptr[p]; ia < ptr[p + 1]; ++ ia) {
				const uint32_t e = lst[ia];
				const double *w = W + (size_t)e * 18, *d = dxc + (size_t)obs_c[e] * 6;
				for(int k = 0; k < 3; ++ k)
					for(int r = 0; r < 6; ++ r)
						l[k] -= w[k * 6 + r] * d[r];
			}
			const double *ci = Cinv + p * 9;
			for(int r = 0; r < 3; ++ r)
				dxp[p * 3 + r] = ci[r] * l[0] + ci[3 + r] * l[1] + ci[6 + r] * l[2];
		}
	}
	free(Cinv); free(Y); free(S); free(b); free(ptr); free(lst);
	return rc? 1 : 0;
}

/* ---- exported entry points (ctypes) -------------------------------------------------------------------- */

SPO_API int spo_ba_chi2(size_t nv, const uint8_t *vtype, const double *cams11, const double *pts, size_t no,
	const uint64_t *obs_pt, const uint64_t *obs_cam, const double *z, const double *info, double *p_chi2)
{
	ba_t g;
	if(ba_init(&g, nv, vtype, cams11, pts, no, obs_pt, obs_cam, z, info)) { ba_free(&g); return -1; }
	*p_chi2 = ba_chi2(&g);
	ba_free(&g);
	return 0;
}

/* U: C x 36, V: P x 9, W: O x 18 (edge order), gc: C x 6, gp: P x 3 */
SPO_API int spo_ba_linearise(size_t nv, const uint8_t *vtype, const double *cams11, const double *pts, size_t no,
	const uint64_t *obs_pt, const uint64_t *obs_cam, const double *z, const double *info,
	double *U, double *V, double *W, double *gc, double *gp, double *p_max_diag)
{
	ba_t g;
	if(ba_init(&g, nv, vtype, cams11, pts, no, obs_pt, obs_cam, z, info)) { ba_free(&g); return -1; }
	*p_max_diag = ba_linearise(&g, U, V, W, gc, gp);
	ba_free(&g);
	return 0;
}

SPO_API int spo_schur_solve(size_t C, size_t P, size_t O, const uint32_t *obs_c, const uint32_t *obs_p, const double *U,
	const double *V, const double *W, const double *gc, const double *gp, double alpha, double *dxc, double *dxp,
	double *S_out, double *rhs_out)
{
	return schur_solve(C, P, O, obs_c, obs_p, U, V, W, gc, gp, alpha, dxc, dxp, S_out, rhs_out);
}

SPO_API int spo_dense_llt_solve(size_t n, double *A, double *b)
{
	int rc = dense_llt_upper(n, A);
	if(rc) return 1;
	dense_llt_solve(n, A, b);
	return 0;
}

/* pose (+) dx, exported for unit tests of the SE(3) composition */
SPO_API void spo_relative_to_absolute(const double *v1, const double *v2, double *dest)
{
	relative_to_absolute(v1, v2, dest);
}

/* Optional replacement of the linear solve inside spo_ba_optimize: the reference's linear-solver slot, so that a
 * solver under test (the GPU library through its C ABI) can run inside the reference's LM loop. Receives the
 * linearisation (U, V, W, gc, gp as spo_ba_linearise returns them) and the damping; writes dxc, dxp; nonzero = failed. */
typedef int (*spo_ba_solver_t)(size_t C, size_t P, size_t O, const double *U, const double *V, const double *W,
	const double *gc, const double *gp, double alpha, double *dxc, double *dxp);
static spo_ba_solver_t g_ba_solver = 0;
SPO_API void spo_set_ba_linear_solver(spo_ba_solver_t f) { g_ba_solver = f; }

/* CNonlinearSolver_Lambda_LM::Optimize, LM:796-1116, batch use. trace: 6 doubles per solve
 * (alpha before, chi2 last, chi2 new, dx.(alpha dx + eta), accepted, alpha after), at most max_trace solves.
 * cam_out: C x 6, pts_out: P x 3. scalars: [0] chi2 initial, [1] chi2 final, [2] alpha initial, [3] n solves,
 * [4] status (1 = factorisation failed). */
SPO_API int spo_ba_optimize(size_t nv, const uint8_t *vtype, const double *cams11, const double *pts, size_t no,
	const uint64_t *obs_pt, const uint64_t *obs_cam, const double *z, const double *info,
	size_t n_max_iteration_num, double f_min_dx_norm, double *cam_out, double *pts_out, double *trace, size_t max_trace,
	double *scalars)
{
	ba_t g;
	if(ba_init(&g, nv, vtype, cams11, pts, no, obs_pt, obs_cam, z, info)) { ba_free(&g); return -1; }
	const size_t C = g.C, P = g.P, O = g.O;
	double *U = (double*)malloc((C + 1) * 36 * 8), *V = (double*)malloc((P + 1) * 9 * 8), *W = (double*)malloc((O + 1) * 18 * 8);
	double *gc = (double*)malloc((C + 1) * 6 * 8), *gp = (double*)malloc((P + 1) * 3 * 8);
	double *dxc = (double*)malloc((C + 1) * 6 * 8), *dxp = (double*)malloc((P + 1) * 3 * 8);
	double *cam_saved = (double*)malloc((C + 1) * 6 * 8), *pt_saved = (double*)malloc((P + 1) * 3 * 8);
	uint32_t *oc = (uint32_t*)malloc((O + 1) * 4), *op = (uint32_t*)malloc((O + 1) * 4);
	for(size_t e = 0; e < O; ++ e) { oc[e] = g.local[obs_cam[e]]; op[e] = g.local[obs_pt[e]]; }
	size_t n_solves = 0;
	int status = 0;
	double f_alpha = 0, f_last_error = 0;
	memset(scalars, 0, 5 * sizeof(double));
	if(O) {
		double f_max_diag = ba_linearise(&g, U, V, W, gc, gp); /* Refresh_Lambda, LM:828-831 */
		f_alpha = f_max_diag * 1e-3; /* f_InitialDamping, LM:151-199 */
		double f_nu = 2.0;
		scalars[2] = f_alpha;
		f_last_error = ba_chi2(&g); /* LM:899 */
		scalars[0] = f_last_error;
		int b_dirty = 0, fail = 10;
		for(size_t it = 0; it < n_max_iteration_num; ++ it) {
			if(it && b_dirty) /* LM:942-949; after a rejected step only the damping changes */
				ba_linearise(&g, U, V, W, gc, gp);
			b_dirty = 0;
			int rc = (g_ba_solver)? g_ba_solver(C, P, O, U, V, W, gc, gp, f_alpha, dxc, dxp) :
				schur_solve(C, P, O, oc, op, U, V, W, gc, gp, f_alpha, dxc, dxp, 0, 0); /* LM:967, 1512-1568 */
			double *t = (n_solves < max_trace)? trace + n_solves * 6 : 0;
			++ n_solves;
			if(t) { t[0] = f_alpha; t[1] = f_last_error; t[2] = t[3] = t[4] = 0; t[5] = f_alpha; }
			if(rc) { status = 1; break; } /* LM:972-974 */
			double f_norm2 = 0, f_den = 0;
			for(size_t v = 0; v < nv; ++ v) { /* vertex order, as Eigen's dot over the full vector */
				const size_t d = (vtype[v] == 0)? 6 : 3;
				const double *dx = (vtype[v] == 0)? dxc + (size_t)g.local[v] * 6 : dxp + (size_t)g.local[v] * 3;
				const double *et = (vtype[v] == 0)? gc + (size_t)g.local[v] * 6 : gp + (size_t)g.local[v] * 3;
				for(size_t i = 0; i < d; ++ i) {
					f_norm2 += dx[i] * dx[i];
					f_den += dx[i] * (f_alpha * dx[i] + et[i]);
				}
			}
			if(sqrt(f_norm2) <= f_min_dx_norm) /* LM:1054 */
				break;
			memcpy(cam_saved, g.cam, C * 6 * 8); /* Save_State, LM:1062 */
			memcpy(pt_saved, g.pt, P * 3 * 8);
			for(size_t c = 0; c < C; ++ c) /* CVertexCam::Operator_Plus, BAT:107-110 */
				relative_to_absolute(g.cam + c * 6, dxc + c * 6, g.cam + c * 6);
			for(size_t i = 0; i < P * 3; ++ i) /* CVertexXYZ::Operator_Plus, BAT:384-388 */
				g.pt[i] += dxp[i];
			double f_error = ba_chi2(&g); /* LM:1078 */
			double rho = (f_last_error - f_error) / f_den; /* Aftermath, LM:204-223 */
			if(t) { t[2] = f_error; t[3] = f_den; }
			if(rho > 0) {
				double f = 1.0 - pow((2 * rho - 1), 3);
				f_alpha *= (f > 1 / 3.0)? f : 1 / 3.0;
				f_nu = 2;
				f_last_error = f_error;
				b_dirty = 1;
				if(t) t[4] = 1;
			} else {
				f_alpha *= f_nu;
				f_nu *= 2;
				memcpy(g.cam, cam_saved, C * 6 * 8); /* Load_State, LM:1096-1106 */
				memcpy(g.pt, pt_saved, P * 3 * 8);
				if(fail > 0) {
					-- fail;
					++ n_max_iteration_num;
				}
			}
			if(t) t[5] = f_alpha;
		}
	}
	scalars[1] = f_last_error;
	scalars[3] = (double)n_solves;
	scalars[4] = status;
	memcpy(cam_out, g.cam, C * 6 * 8);
	memcpy(pts_out, g.pt, P * 3 * 8);
	free(U); free(V); free(W); free(gc); free(gp); free(dxc); free(dxp); free(cam_saved); free(pt_saved); free(oc); free(op);
	ba_free(&g);
	return 0;
}

/* ---- SE(2) pose graphs (SURVEY 8(a) rows a4, a15) --------------------------------------------------------------
 *   2D  = include/slam/2DSolverBase.h      SE2 = include/slam/SE2_Types.h     GN = include/slam/NonlinearSolver_Lambda.h
 *   UB  = include/slam/LinearSolver_UberBlock.h */

/* C2DJacobians::f_ClampAngle_2Pi / f_ClampAngularError_2Pi, 2D:44-95 */
static double clamp_angle_2pi(double a)
{
	return isfinite(a)? fmod(a, M_PI * 2) : 0.0;
}

static double clamp_angular_error_2pi(double e)
{
	e = clamp_angle_2pi(e);
	double a = e, b = e - 2 * M_PI, c = e + 2 * M_PI;
	double m = (fabs(a) < fabs(b))? a : b;
	return (fabs(m) < fabs(c))? m : c;
}

/* C2DJacobians::Absolute_to_Relative with Jacobians, 2D:373-430 (row-major 3x3) */
static void se2_absolute_to_relative(const double *v1, const double *v2, double *d, double *J1, double *J2)
{
	double p1e = v1[0], p1n = v1[1], p1a = v1[2], p2e = v2[0], p2n = v2[1], p2a = v2[2];
	double de = p2e - p1e, dn = p2n - p1n, da = p2a - p1a;
	double o = -p1a, co = cos(o), so = sin(o);
	d[0] = co * de - so * dn;
	d[1] = so * de + co * dn;
	d[2] = clamp_angle_2pi(da);
	if(J1) {
		double cp1a = cos(p1a), sp1a = sin(p1a);
		J1[0] = -cp1a; J1[1] = -sp1a; J1[2] = sp1a * (p1e - p2e) - cp1a * (p1n - p2n);
		J1[3] = sp1a; J1[4] = -cp1a; J1[5] = cp1a * (p1e - p2e) + sp1a * (p1n - p2n);
		J1[6] = 0; J1[7] = 0; J1[8] = -1;
		J2[0] = cp1a; J2[1] = sp1a; J2[2] = 0;
		J2[3] = -sp1a; J2[4] = cp1a; J2[5] = 0;
		J2[6] = 0; J2[7] = 0; J2[8] = 1;
	}
}

/* CEdgePose2D::Calculate_Jacobians_Expectation_Error, SE2:308-319 */
static void se2_edge(const double *states, uint64_t a, uint64_t b, const double *z, double *J0, double *J1, double *r)
{
	double d[3];
	se2_absolute_to_relative(states + a * 3, states + b * 3, d, J0, J1);
	r[0] = z[0] - d[0];
	r[1] = z[1] - d[1];
	r[2] = clamp_angular_error_2pi(z[2] - d[2]);
}

/* f_Chi_Squared_Error_Denorm: serial sum over the edges, SE2:325-335 */
SPO_API int spo_se2_chi2(size_t N, const double *states, size_t E, const uint64_t *from, const uint64_t *to, const double *z,
	const double *info, double *chi2)
{
	(void)N;
	double s = 0;
	for(size_t e = 0; e < E; ++ e) {
		double r[3];
		se2_edge(states, from[e], to[e], z + e * 3, 0, 0, r);
		const double *W = info + e * 9;
		for(int i = 0; i < 3; ++ i)
			s += r[i] * (W[i * 3] * r[0] + W[i * 3 + 1] * r[1] + W[i * 3 + 2] * r[2]);
	}
	*chi2 = s;
	return 0;
}

/* Refresh_Lambda for a pose graph into a DENSE n x n lambda (column-major, full symmetric) and eta: per edge the
 * blocks of Calculate_Hessians_v2 (BIN:759-848: vertex blocks mirrored from the upper triangle, off-diagonal block
 * J0^T W J1 at (min id, max id), transposed if id0 > id1), summed in edge order, the unary factor I on vertex 0 last
 * (LB:1903-1923) */
SPO_API int spo_se2_linearise_dense(size_t N, const double *states, size_t E, const uint64_t *from, const uint64_t *to,
	const double *z, const double *info, double *lambda, double *eta)
{
	const size_t n = N * 3;
	memset(lambda, 0, n * n * sizeof(double));
	memset(eta, 0, n * sizeof(double));
	for(size_t e = 0; e < E; ++ e) {
		double J0[9], J1[9], r[3], T[9], WJ1[9], Wr[3];
		se2_edge(states, from[e], to[e], z + e * 3, J0, J1, r);
		const double *W = info + e * 9;
		for(int i = 0; i < 3; ++ i)
			for(int j = 0; j < 3; ++ j)
				T[i * 3 + j] = J0[0 * 3 + i] * W[0 * 3 + j] + J0[1 * 3 + i] * W[1 * 3 + j] + J0[2 * 3 + i] * W[2 * 3 + j];
		for(int i = 0; i < 3; ++ i) {
			for(int j = 0; j < 3; ++ j)
				WJ1[i * 3 + j] = W[i * 3 + 0] * J1[0 * 3 + j] + W[i * 3 + 1] * J1[1 * 3 + j] + W[i * 3 + 2] * J1[2 * 3 + j];
			Wr[i] = W[i * 3 + 0] * r[0] + W[i * 3 + 1] * r[1] + W[i * 3 + 2] * r[2];
		}
		const size_t a = from[e] * 3, b = to[e] * 3;
		for(int c = 0; c < 3; ++ c) {
			for(int rr = 0; rr < 3; ++ rr) {
				int p = (rr <= c)? rr : c, q = (rr <= c)? c : rr;
				double h00 = T[p * 3 + 0] * J0[0 * 3 + q] + T[p * 3 + 1] * J0[1 * 3 + q] + T[p * 3 + 2] * J0[2 * 3 + q];
				double h11 = J1[0 * 3 + p] * WJ1[0 * 3 + q] + J1[1 * 3 + p] * WJ1[1 * 3 + q] + J1[2 * 3 + p] * WJ1[2 * 3 + q];
				double h01 = T[rr * 3 + 0] * J1[0 * 3 + c] + T[rr * 3 + 1] * J1[1 * 3 + c] + T[rr * 3 + 2] * J1[2 * 3 + c];
				lambda[(a + c) * n + a + rr] += h00;
				lambda[(b + c) * n + b + rr] += h11;
				lambda[(b + c) * n + a + rr] += h01; /* block (v0, v1) */
				lambda[(a + rr) * n + b + c] += h01; /* and its mirror */
			}
		}
		for(int i = 0; i < 3; ++ i) {
			eta[a + i] += T[i * 3 + 0] * r[0] + T[i * 3 + 1] * r[1] + T[i * 3 + 2] * r[2];
			eta[b + i] += J1[0 * 3 + i] * Wr[0] + J1[1 * 3 + i] * Wr[1] + J1[2 * 3 + i] * Wr[2];
		}
	}
	if(N)
		for(int i = 0; i < 3; ++ i)
			lambda[i * n + i] += 1.0;
	return 0;
}

/* Optional replacement of the linear solve inside spo_se2_optimize / spo_se3_optimize (the reference's linear-solver
 * slot): solves lambda (n x n, dense, symmetric) dx = eta in place of eta; nonzero = failed. */
typedef int (*spo_pose_solver_t)(size_t n, const double *lambda, double *eta);
static spo_pose_solver_t g_pose_solver = 0;
SPO_API void spo_set_pose_linear_solver(spo_pose_solver_t f) { g_pose_solver = f; }

static int pose_solve(size_t n, double *lambda, double *eta)
{
	if(g_pose_solver)
		return g_pose_solver(n, lambda, eta);
	if(dense_llt_upper(n, lambda))
		return 1;
	dense_llt_solve(n, lambda, eta);
	return 0;
}

/* CNonlinearSolver_Lambda::Optimize (GN:476-667) with a dense LLT standing in for the block-sparse one (the
 * Cholesky factor is unique: CLinearSolver_UberBlock, UB:312-426, yields the same increment up to rounding).
 * out[0] = chi2 before, out[1] = chi2 after, out[2] = number of solves; dx_norms[k] per solve. */
SPO_API int spo_se2_optimize(size_t N, double *states, size_t E, const uint64_t *from, const uint64_t *to, const double *z,
	const double *info, size_t max_iter, double min_dx, double *out, double *dx_norms)
{
	const size_t n = N * 3;
	double *lambda = (double*)malloc(n * n * sizeof(double)), *eta = (double*)malloc(n * sizeof(double));
	if(!lambda || !eta) return -1;
	spo_se2_chi2(N, states, E, from, to, z, info, &out[0]);
	size_t n_solves = 0;
	int rc = 0;
	for(size_t it = 0; it < max_iter; ++ it) {
		spo_se2_linearise_dense(N, states, E, from, to, z, info, lambda, eta);
		if(pose_solve(n, lambda, eta)) { rc = 1; ++ n_solves; break; }
		double s = 0;
		for(size_t i = 0; i < n; ++ i) s += eta[i] * eta[i];
		dx_norms[n_solves ++] = sqrt(s);
		if(sqrt(s) <= min_dx)
			break;
		for(size_t v = 0; v < N; ++ v) { /* CVertexPose2D::Operator_Plus, SE2:70-74 */
			states[v * 3] += eta[v * 3];
			states[v * 3 + 1] += eta[v * 3 + 1];
			states[v * 3 + 2] = clamp_angle_2pi(states[v * 3 + 2] + eta[v * 3 + 2]);
		}
	}
	spo_se2_chi2(N, states, E, from, to, z, info, &out[1]);
	out[2] = (double)n_solves;
	free(lambda); free(eta);
	return rc;
}

/* ---- SE(3) pose graphs (SURVEY 8(a) row a3) ----------------------------------------------------------------------
 *   3D  = include/slam/3DSolverBase.h    SE3 = include/slam/SE3_Types.h    ROB = include/slam/RobustUtils.h,
 *   include/geometry/RobustLoss.h        BIN = include/slam/BaseTypes_Binary.h */

/* C3DJacobians::Absolute_to_Relative (value), 3D:892-946 */
static void absolute_to_relative(const double *v1, const double *v2, double *dest)
{
	quat_t q1, q2, q1i, q;
	double d[3], t[6];
	axis_angle_to_quat(v1 + 3, &q1);
	axis_angle_to_quat(v2 + 3, &q2);
	q1i.w = q1.w; q1i.x = -q1.x; q1i.y = -q1.y; q1i.z = -q1.z;
	d[0] = v2[0] - v1[0]; d[1] = v2[1] - v1[1]; d[2] = v2[2] - v1[2];
	quat_rotate(&q1i, d, t);
	q = quat_mul(&q1i, &q2);
	quat_to_axis_angle(&q, t + 3);
	memcpy(dest, t, sizeof(t));
}

/* CEdgePose3D::Calculate_Jacobians_Expectation_Error, SE3:265-288: expectation + forward-difference Jacobians
 * (delta = 1e-9, 3D:1043-1059, 1332-1370), error = [t_meas - t_exp, axis-angle of q_meas * conj(q_exp)].
 * J0, J1 row-major 6 x 6 (may be NULL). */
static void se3_edge(const double *states, uint64_t a, uint64_t b, const double *z, double *J0, double *J1, double *r)
{
	const double *v0 = states + a * 6, *v1 = states + b * 6;
	double d[6];
	absolute_to_relative(v0, v1, d);
	if(J0) {
		const double delta = 1e-9, scalar = 1.0 / delta;
		for(int j = 0; j < 6; ++ j) {
			double eps[6] = {0, 0, 0, 0, 0, 0}, p[6], d1[6];
			eps[j] = delta;
			relative_to_absolute(v0, eps, p);
			absolute_to_relative(p, v1, d1);
			for(int i = 0; i < 6; ++ i) J0[i * 6 + j] = (d1[i] - d[i]) * scalar;
			relative_to_absolute(v1, eps, p);
			absolute_to_relative(v0, p, d1);
			for(int i = 0; i < 6; ++ i) J1[i * 6 + j] = (d1[i] - d[i]) * scalar;
		}
	}
	quat_t pq, dq, dqc, e;
	r[0] = z[0] - d[0]; r[1] = z[1] - d[1]; r[2] = z[2] - d[2];
	axis_angle_to_quat(z + 3, &pq);
	axis_angle_to_quat(d + 3, &dq);
	dqc.w = dq.w; dqc.x = -dq.x; dqc.y = -dq.y; dqc.z = -dq.z;
	e = quat_mul(&pq, &dqc);
	quat_to_axis_angle(&e, r + 3);
}

/* CRobustify_ErrorNorm_Default<CCTFraction<30, 100>, CHuberLossd>::f_RobustWeight, SE3:128-129, ROB:412-438, Huber weight
 * with the default parameter 1.345 (RobustLoss.h:63,100-104) */
static double se3_robust_weight(const double *r)
{
	double s = 0;
	for(int i = 0; i < 6; ++ i) s += r[i] * r[i];
	double e = sqrt(s) / (30.0 / 100.0);
	return (e <= 1.345)? 1.0 : 1.345 / e;
}

/* f_Chi_Squared_Error_Denorm: serial sum of the UNWEIGHTED r^T Sigma^-1 r, SE3:318-327 */
SPO_API int spo_se3_chi2(size_t N, const double *states, size_t E, const uint64_t *from, const uint64_t *to, const double *z,
	const double *info, double *chi2)
{
	(void)N;
	double s = 0;
	for(size_t e = 0; e < E; ++ e) {
		double r[6];
		se3_edge(states, from[e], to[e], z + e * 6, 0, 0, r);
		const double *W = info + e * 36;
		for(int i = 0; i < 6; ++ i) {
			double t = 0;
			for(int k = 0; k < 6; ++ k) t += W[i * 6 + k] * r[k];
			s += r[i] * t;
		}
	}
	*chi2 = s;
	return 0;
}

/* Refresh_Lambda into a dense lambda (column-major, full symmetric) and eta. Calculate_Hessians_v2 for a ROBUST edge
 * (BIN:759-848): T = J0^T Sigma^-1 w; H01 = T J1; H00 = sym_U(T J0); H11 = sym_U(J1^T Sigma^-1 J1 w);
 * g0 = T r w (the weight enters twice, as in the reference, BIN:820-821); g1 = J1^T (Sigma^-1 r) w. */
SPO_API int spo_se3_linearise_dense(size_t N, const double *states, size_t E, const uint64_t *from, const uint64_t *to,
	const double *z, const double *info, double *lambda, double *eta)
{
	const size_t n = N * 6;
	memset(lambda, 0, n * n * sizeof(double));
	memset(eta, 0, n * sizeof(double));
	for(size_t e = 0; e < E; ++ e) {
		double J0[36], J1[36], r[6], T[36], WJ1[36], Wr[6];
		se3_edge(states, from[e], to[e], z + e * 6, J0, J1, r);
		const double w = se3_robust_weight(r);
		const double *W = info + e * 36;
		for(int i = 0; i < 6; ++ i)
			for(int j = 0; j < 6; ++ j) {
				double t = 0;
				for(int k = 0; k < 6; ++ k) t += J0[k * 6 + i] * W[k * 6 + j];
				T[i * 6 + j] = t * w;
			}
		for(int i = 0; i < 6; ++ i) {
			for(int j = 0; j < 6; ++ j) {
				double t = 0;
				for(int k = 0; k < 6; ++ k) t += W[i * 6 + k] * J1[k * 6 + j];
				WJ1[i * 6 + j] = t;
			}
			double t = 0;
			for(int k = 0; k < 6; ++ k) t += W[i * 6 + k] * r[k];
			Wr[i] = t;
		}
		const size_t a = from[e] * 6, b = to[e] * 6;
		for(int c = 0; c < 6; ++ c) {
			for(int rr = 0; rr < 6; ++ rr) {
				int p = (rr <= c)? rr : c, q = (rr <= c)? c : rr;
				double h00 = 0, h11 = 0, h01 = 0;
				for(int k = 0; k < 6; ++ k) {
					h00 += T[p * 6 + k] * J0[k * 6 + q];
					h11 += J1[k * 6 + p] * WJ1[k * 6 + q];
					h01 += T[rr * 6 + k] * J1[k * 6 + c];
				}
				h11 *= w;
				lambda[(a + c) * n + a + rr] += h00;
				lambda[(b + c) * n + b + rr] += h11;
				lambda[(b + c) * n + a + rr] += h01;
				lambda[(a + rr) * n + b + c] += h01;
			}
		}
		for(int i = 0; i < 6; ++ i) {
			double g0 = 0, g1 = 0;
			for(int k = 0; k < 6; ++ k) {
				g0 += T[i * 6 + k] * r[k];
				g1 += J1[k * 6 + i] * Wr[k];
			}
			eta[a + i] += g0 * w;
			eta[b + i] += g1 * w;
		}
	}
	if(N)
		for(int i = 0; i < 6; ++ i)
			lambda[i * n + i] += 1.0;
	return 0;
}

/* CNonlinearSolver_Lambda::Optimize (GN:476-667) on an SE(3) graph; CVertexPose3D::Operator_Plus = Relative_to_Absolute
 * (SE3:45-48). Dense LLT stands in for the block-sparse factorisation, as in spo_se2_optimize. */
SPO_API int spo_se3_optimize(size_t N, double *states, size_t E, const uint64_t *from, const uint64_t *to, const double *z,
	const double *info, size_t max_iter, double min_dx, double *out, double *dx_norms)
{
	const size_t n = N * 6;
	double *lambda = (double*)malloc(n * n * sizeof(double)), *eta = (double*)malloc(n * sizeof(double));
	if(!lambda || !eta) return -1;
	spo_se3_chi2(N, states, E, from, to, z, info, &out[0]);
	size_t n_solves = 0;
	int rc = 0;
	for(size_t it = 0; it < max_iter; ++ it) {
		spo_se3_linearise_dense(N, states, E, from, to, z, info, lambda, eta);
		if(pose_solve(n, lambda, eta)) { rc = 1; ++ n_solves; break; }
		double s = 0;
		for(size_t i = 0; i < n; ++ i) s += eta[i] * eta[i];
		dx_norms[n_solves ++] = sqrt(s);
		if(sqrt(s) <= min_dx)
			break;
		for(size_t v = 0; v < N; ++ v)
			relative_to_absolute(states + v * 6, eta + v * 6, states + v * 6);
	}
	spo_se3_chi2(N, states, E, from, to, z, info, &out[1]);
	out[2] = (double)n_solves;
	free(lambda); free(eta);
	return rc;
}

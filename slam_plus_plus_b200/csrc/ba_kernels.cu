// ba_kernels.cu -- stage 1 of the hot path on the device: per-edge linearisation of the BA edges and
// deterministic accumulation into the block Hessian / gradient, plus chi2 and the vertex update.
//
// Reference functions replaced (SURVEY 8(a) rows a1, a2, a5, a7, a17, a18):
//   CEdgeP2C3D::Calculate_Jacobians_Expectation_Error   include/slam/BA_Types.h:494-505
//   CBAJacobians::Project_P2C (value / FD Jacobians)    include/slam/BASolverBase.h:260-327, 559-619
//   CBaseEdgeImpl::Calculate_Hessians_v2                include/slam/BaseTypes_Binary.h:759-848
//   CMatrixReductionPlan / CVectorReductionPlan         include/slam/NonlinearSolver_Lambda_Base.h:152-197, 563-607
//   CEdgeP2C3D::f_Chi_Squared_Error                     include/slam/BA_Types.h:511-531
//   CVertexCam / CVertexXYZ::Operator_Plus              include/slam/BA_Types.h:107-110, 384-388
//
// Design: the reference materialises 72 doubles per edge and reduces them by destination. Here nothing
// per-edge is materialised except W (the camera x point block that the Schur complement needs anyway):
//   * k_cam_prepare: the six forward-difference perturbations of a camera pose do not depend on the
//     observation, so [R|t] of the base pose and of the six perturbed poses are formed once per camera
//     (7 x 12 doubles) -- every observation then costs ten cheap projections instead of ten pose
//     compositions with sin/cos/atan.
//   * k_linearise_cams: one CTA per camera, camera [R|t]s staged in shared memory, observations gathered
//     through the camera's list; writes W and the landmark share (V_e, g_e) of every observation through shared
//     memory, accumulates U_c and g_c in registers and reduces them with a fixed-shape tree (no atomics,
//     bit-reproducible).
//   * k_sum_point_records: a warp stages the contiguous records of 32 landmarks in shared memory, and the lane of each
//     landmark adds its track's records in insertion order into V_p and g_p -- the reference's reduction plan's order.
//
// Robust losses (spp_ba_set_robust_loss): k_linearise_cams, k_chi2_partial and k_obs_errors take the loss as a template
// parameter and share robust_loss(). The SPP_LOSS_NONE instantiations are the plain kernels (the loss code is compiled
// out); under a loss the weight of an observation is computed on the fly from its residual, so no per-observation array
// is added to the LM path.

#include "spp_ctx.h"
#include <stdlib.h>
#include "ba_geometry.cuh"

namespace spp {

#define FD_DELTA 1e-9
#define FD_SCALAR (1.0 / FD_DELTA)

// ---------------------------------------------------------------------------------------------------

// thread per (camera, j): j = 0 base pose, j = 1..6 pose (+) delta e_{j-1}
__global__ void k_cam_prepare(size_t C, const double *__restrict__ cam_state, const double *__restrict__ cam_intr,
	double *__restrict__ camRt, double *__restrict__ camK, int n_variants)
{
	size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
	if(i >= C * n_variants)
		return;
	size_t c = i / n_variants;
	int j = int(i % n_variants);
	double pose[6];
	#pragma unroll
	for(int k = 0; k < 6; ++ k)
		pose[k] = cam_state[c * 6 + k];
	if(j > 0) {
		double eps[6] = {0, 0, 0, 0, 0, 0};
		eps[j - 1] = FD_DELTA;
		double dest[6];
		relative_to_absolute(pose, eps, dest);
		#pragma unroll
		for(int k = 0; k < 6; ++ k)
			pose[k] = dest[k];
	}
	double Rt[12];
	pose_to_Rt(pose, Rt);
	#pragma unroll
	for(int k = 0; k < 12; ++ k)
		camRt[(c * 7 + j) * 12 + k] = Rt[k];
	if(j == 0) {
		double fx = cam_intr[c * 5 + 0], fy = cam_intr[c * 5 + 1];
		camK[c * 5 + 0] = fx;
		camK[c * 5 + 1] = fy;
		camK[c * 5 + 2] = cam_intr[c * 5 + 2];
		camK[c * 5 + 3] = cam_intr[c * 5 + 3];
		camK[c * 5 + 4] = cam_intr[c * 5 + 4] / (.5 * (fx + fy));
	}
}

// analytic derivative of the projection wrt the camera-frame point x; returns d(u,v)/dx (2x3, row-major)
__device__ __forceinline__ void project_with_dx(const double *Rt, double fx, double fy, double cx, double cy, double k,
	double X, double Y, double Z, double &u, double &v, double *x_cam, double *D)
{
	double x0 = Rt[0] * X + Rt[1] * Y + Rt[2] * Z + Rt[9];
	double x1 = Rt[3] * X + Rt[4] * Y + Rt[5] * Z + Rt[10];
	double x2 = Rt[6] * X + Rt[7] * Y + Rt[8] * Z + Rt[11];
	x_cam[0] = x0; x_cam[1] = x1; x_cam[2] = x2;
	double iz = 1.0 / x2;
	double dx = fx * x0 * iz, dy = fy * x1 * iz; // offsets from the principal point
	double r2 = dx * dx + dy * dy;
	double s = 1 + r2 * k;
	u = cx + s * dx;
	v = cy + s * dy;
	// d(dx,dy)/dx_cam
	double a00 = fx * iz, a02 = -dx * iz, a11 = fy * iz, a12 = -dy * iz;
	// d(u,v)/d(dx,dy) = s I + 2 k [dx;dy][dx dy]
	double m00 = s + 2 * k * dx * dx, m01 = 2 * k * dx * dy, m11 = s + 2 * k * dy * dy;
	D[0] = m00 * a00; D[1] = m01 * a11; D[2] = m00 * a02 + m01 * a12;
	D[3] = m01 * a00; D[4] = m11 * a11; D[5] = m01 * a02 + m11 * a12;
}

// Jacobians of one observation. Jc: 2x6 row-major, Jp: 2x3 row-major, r = z - h
__device__ __forceinline__ void observation_jacobians(int jac_mode, const double *sRt /* 7x12 */, const double *K,
	double X, double Y, double Z, double zu, double zv, double *Jc, double *Jp, double &ru, double &rv,
	bool want_Jc, bool want_Jp)
{
	const double fx = K[0], fy = K[1], cx = K[2], cy = K[3], k = K[4];
	if(jac_mode == SPP_JAC_FD_REFERENCE) {
		double u0, v0;
		project_Rt(sRt, fx, fy, cx, cy, k, X, Y, Z, u0, v0);
		ru = zu - u0; rv = zv - v0;
		if(want_Jc) {
			#pragma unroll
			for(int j = 0; j < 6; ++ j) {
				double u, v;
				project_Rt(sRt + 12 * (j + 1), fx, fy, cx, cy, k, X, Y, Z, u, v);
				Jc[j] = (u - u0) * FD_SCALAR;
				Jc[6 + j] = (v - v0) * FD_SCALAR;
			}
		}
		if(want_Jp) {
			double u, v;
			project_Rt(sRt, fx, fy, cx, cy, k, X + FD_DELTA, Y, Z, u, v);
			Jp[0] = (u - u0) * FD_SCALAR; Jp[3] = (v - v0) * FD_SCALAR;
			project_Rt(sRt, fx, fy, cx, cy, k, X, Y + FD_DELTA, Z, u, v);
			Jp[1] = (u - u0) * FD_SCALAR; Jp[4] = (v - v0) * FD_SCALAR;
			project_Rt(sRt, fx, fy, cx, cy, k, X, Y, Z + FD_DELTA, u, v);
			Jp[2] = (u - u0) * FD_SCALAR; Jp[5] = (v - v0) * FD_SCALAR;
		}
	} else {
		double u0, v0, xc[3], D[6];
		project_with_dx(sRt, fx, fy, cx, cy, k, X, Y, Z, u0, v0, xc, D);
		ru = zu - u0; rv = zv - v0;
		// pose (+) eps: t' = t + R eps_t, R' = R exp(eps_r)  =>  dx_cam/deps_t = R, dx_cam/deps_r = -R [X]_x
		const double *R = sRt;
		if(want_Jp) {
			#pragma unroll
			for(int r = 0; r < 2; ++ r) {
				#pragma unroll
				for(int c = 0; c < 3; ++ c)
					Jp[r * 3 + c] = D[r * 3 + 0] * R[0 + c] + D[r * 3 + 1] * R[3 + c] + D[r * 3 + 2] * R[6 + c];
			}
		}
		if(want_Jc) {
			double DR[6];
			#pragma unroll
			for(int r = 0; r < 2; ++ r) {
				#pragma unroll
				for(int c = 0; c < 3; ++ c)
					DR[r * 3 + c] = D[r * 3 + 0] * R[0 + c] + D[r * 3 + 1] * R[3 + c] + D[r * 3 + 2] * R[6 + c];
			}
			#pragma unroll
			for(int r = 0; r < 2; ++ r) {
				Jc[r * 6 + 0] = DR[r * 3 + 0];
				Jc[r * 6 + 1] = DR[r * 3 + 1];
				Jc[r * 6 + 2] = DR[r * 3 + 2];
				// -DR [X]_x with [X]_x = [0 -Z Y; Z 0 -X; -Y X 0]
				Jc[r * 6 + 3] = DR[r * 3 + 2] * Y - DR[r * 3 + 1] * Z;
				Jc[r * 6 + 4] = DR[r * 3 + 0] * Z - DR[r * 3 + 2] * X;
				Jc[r * 6 + 5] = DR[r * 3 + 1] * X - DR[r * 3 + 0] * Y;
			}
		}
	}
}

// squared Mahalanobis error s2 = e^T Sigma^-1 e (the expression and operation order of the chi2 kernel: with e = -r the
// same bits)
__device__ __forceinline__ double obs_sq_error(double eu, double ev, double2 i01, double2 i23)
{
	return (eu * i01.x + ev * i23.x) * eu + (eu * i01.y + ev * i23.y) * ev;
}

// cost rho(s2) and IRLS weight w = rho'(s2) of one observation under the loss LOSS with scale k (spp_b200.h; the
// reference's robust kernels: RobustUtils.h:368-586). Below the Huber threshold rho = s2 and w = 1 exactly.
template <int LOSS>
__device__ __forceinline__ double robust_loss(double s2, double k, double &w)
{
	if(LOSS == SPP_LOSS_HUBER) {
		if(s2 <= k * k) {
			w = 1.0;
			return s2;
		}
		const double s = sqrt(s2);
		w = k / s;
		return 2 * k * s - k * k;
	} else if(LOSS == SPP_LOSS_CAUCHY) {
		const double q = s2 / (k * k);
		w = 1.0 / (1.0 + q);
		return k * k * log1p(q);
	}
	w = 1.0;
	return s2;
}

__device__ __forceinline__ double warp_sum(double v)
{
	#pragma unroll
	for(int o = 16; o > 0; o >>= 1)
		v += __shfl_down_sync(0xffffffffu, v, o);
	return v;
}

__device__ __forceinline__ double warp_max(double v)
{
	#pragma unroll
	for(int o = 16; o > 0; o >>= 1)
		v = fmax(v, __shfl_down_sync(0xffffffffu, v, o));
	return v;
}

#define CAM_THREADS 256
#define CAM_MIN_CTAS 2   // 128 registers: two CTAs per SM (the per-thread accumulators of U_c, g_c are gone, see below)
#define GR_LD 68         // row length of the Gram operands in shared memory (64 + 4: fragment loads at most 2-way conflicted)

__device__ __forceinline__ void dmma884(double &d0, double &d1, double a, double b)
{
	asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
		: "+d"(d0), "+d"(d1) : "d"(a), "d"(b));
}

// W = T Jp (6x3, column-major) and the landmark's share of the observation, V_e = upper(Jp^T Sigma^-1 Jp) and
// g_e = Jp^T (Sigma^-1 r) (record of 10 doubles, the last one padding): the Jacobian is at hand here, so the landmark
// kernel only has to add these records up along its track (same expressions and the same summation order as the
// landmark kernel that recomputed Jp: bit-identical V, gp)
__device__ __forceinline__ void observation_outputs(const double *T0, const double *T1, const double *Jp, double2 i01,
	double2 i23, double ru, double rv, double *Wo, double *rec, double &dmax)
{
	#pragma unroll
	for(int cc = 0; cc < 3; ++ cc) {
		double w[6];
		#pragma unroll
		for(int j = 0; j < 6; ++ j)
			w[j] = T0[j] * Jp[cc] + T1[j] * Jp[3 + cc];
		*reinterpret_cast<double2*>(Wo + cc * 6 + 0) = make_double2(w[0], w[1]);
		*reinterpret_cast<double2*>(Wo + cc * 6 + 2) = make_double2(w[2], w[3]);
		*reinterpret_cast<double2*>(Wo + cc * 6 + 4) = make_double2(w[4], w[5]);
	}
	double A0[3], A1[3];
	#pragma unroll
	for(int j = 0; j < 3; ++ j) {
		A0[j] = Jp[j] * i01.x + Jp[3 + j] * i23.x;
		A1[j] = Jp[j] * i01.y + Jp[3 + j] * i23.y;
	}
	const double e00 = A0[0] * Jp[0] + A1[0] * Jp[3], e01 = A0[0] * Jp[1] + A1[0] * Jp[4], e02 = A0[0] * Jp[2] + A1[0] * Jp[5];
	const double e11 = A0[1] * Jp[1] + A1[1] * Jp[4], e12 = A0[1] * Jp[2] + A1[1] * Jp[5], e22 = A0[2] * Jp[2] + A1[2] * Jp[5];
	const double s0 = i01.x * ru + i01.y * rv, s1 = i23.x * ru + i23.y * rv;
	*reinterpret_cast<double2*>(rec + 0) = make_double2(e00, e01);
	*reinterpret_cast<double2*>(rec + 2) = make_double2(e02, e11);
	*reinterpret_cast<double2*>(rec + 4) = make_double2(e12, e22);
	*reinterpret_cast<double2*>(rec + 6) = make_double2(Jp[0] * s0 + Jp[3] * s1, Jp[1] * s0 + Jp[4] * s1);
	*reinterpret_cast<double2*>(rec + 8) = make_double2(Jp[2] * s0 + Jp[5] * s1, 0.0);
	dmax = fmax(dmax, fmax(e00, fmax(e11, e22)));
}

static const size_t CAM_SMEM = (size_t)(CAM_THREADS / 32) * 2 * 8 * GR_LD * sizeof(double);

// one CTA per camera. JAC: Jacobian mode as a compile-time constant (the other branch does not cost registers).
// U_c = sum_e T_e Jc_e and g_c = sum_e T_e r_e (T_e = Jc_e^T Sigma_e^-1, 6 x 2) are ONE small GEMM per warp: the 32
// observations of a warp trip put T (6 x 64: two columns per observation) and [Jc | r] (64 x 7) into shared memory and
// sixteen mma.sync.m8n8k4.f64 add [U | g] (6 x 7 of the 8 x 8 tile) to two accumulator registers per lane -- instead of
// 27 accumulators (54 registers) per thread and 27 FMAs per observation. With that the kernel fits 128 registers and
// two CTAs share an SM (it was latency bound at 254 registers, 8 warps per SM, 12 % of the warp slots active:
// profiles/r1k_full.csv). The expressions of the products are the reference's (U_e = T Jc, g = T r,
// BaseTypes_Binary.h:813-843); the summation order is fixed (k ascending inside the warp, then the warps in order), so
// the result is bit-reproducible.
// After the products the warp's tile is free: W and the landmark records of its 32 observations are staged there and
// stored as consecutive 16-byte pieces (Venice shape: 519 -> 352 us; DESIGN.md §4), and the indices of the next trip are
// fetched one trip ahead (352 -> 348 us).
// (Measured alternatives of round 1: ten lanes per observation -- one projection per lane, the Hessian algebra spread
// over the lanes through shared memory -- 0.97 ms against 0.81 ms.)
// LOSS: robust loss as a compile-time constant; under a loss the observation's information matrix is scaled by its weight
// before any other use, so U_c, g_c, W, the landmark record and the damping maximum are those of the weighted problem.
template <int JAC, int LOSS>
__global__ void __launch_bounds__(CAM_THREADS, CAM_MIN_CTAS) k_linearise_cams(int, const uint32_t *__restrict__ cam_ptr,
	const uint32_t *__restrict__ cam_obs, const uint32_t *__restrict__ obs_pt, const double *__restrict__ pts,
	const double *__restrict__ z, const double *__restrict__ info, const double *__restrict__ camRt,
	const double *__restrict__ camK, double *__restrict__ W, double *__restrict__ U, double *__restrict__ gc,
	unsigned long long *__restrict__ maxdiag, long uf_cam, double *__restrict__ PtRec, double loss_k)
{
	extern __shared__ __align__(16) double gram[]; // per warp: T [8][GR_LD], then [Jc | r] [8][GR_LD]
	__shared__ double sRt[7 * 12];
	__shared__ double sK[5];
	__shared__ double sred[CAM_THREADS / 32][65];
	const unsigned c = blockIdx.x;
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	const int g = lane >> 2, t = lane & 3;
	double *sT = gram + (size_t)warp * (2 * 8 * GR_LD), *sJ = sT + 8 * GR_LD;
	for(int i = threadIdx.x; i < 7 * 12; i += CAM_THREADS)
		sRt[i] = camRt[(size_t)c * 84 + i];
	if(threadIdx.x < 5)
		sK[threadIdx.x] = camK[(size_t)c * 5 + threadIdx.x];
	__syncthreads();

	double acc0 = 0, acc1 = 0, dmax = 0; // [U | g](g, 2 t), (g, 2 t + 1)
	const unsigned beg = cam_ptr[c], end = cam_ptr[c + 1];
	unsigned o_nx = 0, p_nx = 0;
	if(beg + threadIdx.x < end) {
		o_nx = cam_obs[beg + threadIdx.x];
		p_nx = obs_pt[o_nx];
	}
	for(unsigned base = beg; base < end; base += CAM_THREADS) {
		const unsigned idx = base + threadIdx.x;
		double2 *pT = reinterpret_cast<double2*>(sT + 2 * lane), *pJ = reinterpret_cast<double2*>(sJ + 2 * lane);
		double T0[6], T1[6], Jp[6], ru, rv;
		double2 i01, i23;
		const unsigned o = o_nx, p = p_nx;
		if(idx + CAM_THREADS < end) // next trip's indices: its dependent chain becomes one memory round trip
			o_nx = cam_obs[idx + CAM_THREADS];
		if(idx < end) {
			const double X = pts[(size_t)p * 3], Y = pts[(size_t)p * 3 + 1], Z = pts[(size_t)p * 3 + 2];
			const double2 zz = *reinterpret_cast<const double2*>(z + (size_t)o * 2);
			i01 = *reinterpret_cast<const double2*>(info + (size_t)o * 4);
			i23 = *reinterpret_cast<const double2*>(info + (size_t)o * 4 + 2);
			if(idx + CAM_THREADS < end)
				p_nx = obs_pt[o_nx];
			double Jc[12];
			observation_jacobians(JAC, sRt, sK, X, Y, Z, zz.x, zz.y, Jc, Jp, ru, rv, true, true);
			if(LOSS != SPP_LOSS_NONE) { // Sigma^-1 <- w Sigma^-1
				double w;
				robust_loss<LOSS>(obs_sq_error(ru, rv, i01, i23), loss_k, w);
				i01.x *= w; i01.y *= w;
				i23.x *= w; i23.y *= w;
			}
			// T = Jc^T Sigma^-1 (6x2): T(j,0) = Jc(0,j) s00 + Jc(1,j) s10 ; T(j,1) = Jc(0,j) s01 + Jc(1,j) s11
			#pragma unroll
			for(int j = 0; j < 6; ++ j) {
				T0[j] = Jc[j] * i01.x + Jc[6 + j] * i23.x;
				T1[j] = Jc[j] * i01.y + Jc[6 + j] * i23.y;
			}
			// the Gram operands of this observation: columns 2 lane, 2 lane + 1
			#pragma unroll
			for(int j = 0; j < 6; ++ j) {
				pT[j * (GR_LD / 2)] = make_double2(T0[j], T1[j]);
				pJ[j * (GR_LD / 2)] = make_double2(Jc[j], Jc[6 + j]);
				dmax = fmax(dmax, T0[j] * Jc[j] + T1[j] * Jc[6 + j]); // the diagonal of U_e (initial damping, LM.h:162-166)
			}
			pJ[6 * (GR_LD / 2)] = make_double2(ru, rv);
		} else {
			#pragma unroll
			for(int j = 0; j < 6; ++ j) {
				pT[j * (GR_LD / 2)] = make_double2(0.0, 0.0);
				pJ[j * (GR_LD / 2)] = make_double2(0.0, 0.0);
			}
			pJ[6 * (GR_LD / 2)] = make_double2(0.0, 0.0);
		}
		__syncwarp();
		// [U | g] += T [Jc | r]: A(m, k) = T(m, k), B(k, n) = [Jc | r](k, n), k = 0 .. 63; rows 6, 7 of A and column 7 of B
		// are zero (the tile holds other data between the products)
		#pragma unroll 4
		for(int k4 = 0; k4 < 64; k4 += 4)
			dmma884(acc0, acc1, (g < 6)? sT[g * GR_LD + k4 + t] : 0.0, (g < 7)? sJ[g * GR_LD + k4 + t] : 0.0);
		__syncwarp();
		// W and the landmark record of the warp's 32 observations go through the tile: consecutive lanes then store
		// consecutive 16-byte pieces of one observation's block instead of 32 scattered pieces per instruction
		double *sW = sT, *sR = sT + 32 * 18;
		if(idx < end)
			observation_outputs(T0, T1, Jp, i01, i23, ru, rv, sW + lane * 18, sR + lane * 10, dmax);
		__syncwarp();
		const unsigned n_valid = (end - base > (unsigned)warp * 32)? end - base - (unsigned)warp * 32 : 0;
		#pragma unroll
		for(int k = 0; k < 9; ++ k) { // 32 x 9 pieces of W
			const unsigned q = k * 32 + lane, ob = q / 9;
			const unsigned oq = __shfl_sync(0xffffffffu, o, ob);
			if(ob < n_valid)
				reinterpret_cast<double2*>(W + (size_t)oq * 18)[q - ob * 9] = reinterpret_cast<const double2*>(sW)[q];
		}
		#pragma unroll
		for(int k = 0; k < 5; ++ k) { // 32 x 5 pieces of the landmark records
			const unsigned q = k * 32 + lane, ob = q / 5;
			const unsigned oq = __shfl_sync(0xffffffffu, o, ob);
			if(ob < n_valid)
				reinterpret_cast<double2*>(PtRec + (size_t)oq * 10)[q - ob * 5] = reinterpret_cast<const double2*>(sR)[q];
		}
		__syncwarp();
	}

	// fixed-shape reduction: the 8 warp tiles in order
	sred[warp][g * 8 + 2 * t] = acc0;
	sred[warp][g * 8 + 2 * t + 1] = acc1;
	dmax = warp_max(dmax);
	if(lane == 0) sred[warp][64] = dmax;
	__syncthreads();
	if(threadIdx.x < 65) {
		double v = sred[0][threadIdx.x];
		if(threadIdx.x < 64) {
			for(int w = 1; w < CAM_THREADS / 32; ++ w)
				v += sred[w][threadIdx.x];
		} else {
			for(int w = 1; w < CAM_THREADS / 32; ++ w)
				v = fmax(v, sred[w][threadIdx.x]);
		}
		sred[0][threadIdx.x] = v;
	}
	__syncthreads();
	if(threadIdx.x < 36) {
		int cc = threadIdx.x / 6, rr = threadIdx.x % 6;
		int a = (rr <= cc)? rr : cc, b = (rr <= cc)? cc : rr; // selfadjointView<Upper>
		double v = sred[0][a * 8 + b];
		if(rr == cc && (long)c == uf_cam)
			v += 1.0; // unary factor on vertex 0 (FlatSystem.h:432-473)
		U[(size_t)c * 36 + threadIdx.x] = v;
	} else if(threadIdx.x < 42)
		gc[(size_t)c * 6 + threadIdx.x - 36] = sred[0][(threadIdx.x - 36) * 8 + 6];
	else if(threadIdx.x == 42 && maxdiag)
		atomicMax(maxdiag, (unsigned long long)__double_as_longlong(sred[0][64]));
}

// warp per 32 consecutive landmarks: V_p, g_p = sum of the per-observation records written by k_linearise_cams. The
// records of the warp's 32 tracks are one contiguous range; the warp stages it chunk by chunk in shared memory with
// coalesced 16-byte loads, and the owning lane adds its landmark's records in edge insertion order (the reference's
// summation order, NonlinearSolver_Lambda_Base.h:152-197, 563-607). V and g_p leave through shared memory as the
// warp's contiguous 32 x 9 and 32 x 3 ranges.
#define SR_WARPS 4
#define SR_CHUNK 64 // records per chunk: 320 double2, ten loads per lane in flight

__global__ void __launch_bounds__(SR_WARPS * 32) k_sum_point_records(size_t P, const uint32_t *__restrict__ pt_ptr,
	const double *__restrict__ PtRec, double *__restrict__ V, double *__restrict__ gp, long uf_pt)
{
	__shared__ double2 sRec[SR_WARPS][SR_CHUNK * 5];
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	const size_t p0 = (blockIdx.x * (size_t)SR_WARPS + warp) * 32;
	if(p0 >= P) return;
	const unsigned np = (unsigned)((P - p0 < 32)? P - p0 : 32);
	const unsigned wbeg = pt_ptr[p0], wend = pt_ptr[p0 + np];
	const unsigned beg = ((unsigned)lane < np)? pt_ptr[p0 + lane] : wend, end = ((unsigned)lane < np)? pt_ptr[p0 + lane + 1] : wend;
	double2 *s = sRec[warp];
	const double2 *src = reinterpret_cast<const double2*>(PtRec);
	double v00 = 0, v01 = 0, v02 = 0, v11 = 0, v12 = 0, v22 = 0, g0 = 0, g1 = 0, g2 = 0;
	for(unsigned b = wbeg; b < wend; b += SR_CHUNK) {
		const unsigned n5 = ((wend - b < SR_CHUNK)? wend - b : SR_CHUNK) * 5;
		#pragma unroll
		for(unsigned k = 0; k < SR_CHUNK * 5 / 32; ++ k) {
			const unsigned i = k * 32 + lane;
			if(i < n5)
				s[i] = src[(size_t)b * 5 + i];
		}
		__syncwarp();
		const unsigned lo = (beg > b)? beg : b, hi = (end < b + SR_CHUNK)? end : b + SR_CHUNK;
		for(unsigned o = lo; o < hi; ++ o) {
			const double2 *rec = s + (o - b) * 5;
			const double2 ra = rec[0], rb = rec[1], rc = rec[2], rd = rec[3], re = rec[4];
			v00 += ra.x; v01 += ra.y; v02 += rb.x; v11 += rb.y; v12 += rc.x; v22 += rc.y;
			g0 += rd.x; g1 += rd.y; g2 += re.x;
		}
		__syncwarp();
	}
	if(p0 + lane == (size_t)uf_pt) {
		v00 += 1.0; v11 += 1.0; v22 += 1.0;
	}
	double *sv = reinterpret_cast<double*>(s), *sg = sv + 32 * 9;
	if((unsigned)lane < np) {
		double *Vp = sv + lane * 9;
		Vp[0] = v00; Vp[1] = v01; Vp[2] = v02;
		Vp[3] = v01; Vp[4] = v11; Vp[5] = v12;
		Vp[6] = v02; Vp[7] = v12; Vp[8] = v22;
		sg[lane * 3] = g0; sg[lane * 3 + 1] = g1; sg[lane * 3 + 2] = g2;
	}
	__syncwarp();
	for(unsigned i = lane; i < np * 9; i += 32)
		V[p0 * 9 + i] = sv[i];
	for(unsigned i = lane; i < np * 3; i += 32)
		gp[p0 * 3 + i] = sg[i];
}

// chi2 (under a loss: sum rho(s2)): thread per observation, block partials, then a fixed-order final pass
#define RED_THREADS 256

template <int LOSS>
__global__ void __launch_bounds__(RED_THREADS) k_chi2_partial(size_t O, const uint32_t *__restrict__ obs_cam,
	const uint32_t *__restrict__ obs_pt, const double *__restrict__ pts, const double *__restrict__ z,
	const double *__restrict__ info, const double *__restrict__ camRt, const double *__restrict__ camK,
	double *__restrict__ partial, double loss_k)
{
	__shared__ double sred[RED_THREADS / 32];
	double acc = 0;
	for(size_t o = blockIdx.x * (size_t)RED_THREADS + threadIdx.x; o < O; o += (size_t)gridDim.x * RED_THREADS) {
		const unsigned c = obs_cam[o], p = obs_pt[o];
		const double *Rt = camRt + (size_t)c * 84;
		const double *K = camK + (size_t)c * 5;
		double u, v;
		project_Rt(Rt, K[0], K[1], K[2], K[3], K[4], pts[(size_t)p * 3], pts[(size_t)p * 3 + 1], pts[(size_t)p * 3 + 2], u, v);
		const double2 zz = *reinterpret_cast<const double2*>(z + o * 2);
		const double2 i01 = *reinterpret_cast<const double2*>(info + o * 4);
		const double2 i23 = *reinterpret_cast<const double2*>(info + o * 4 + 2);
		double eu = u - zz.x, ev = v - zz.y;
		// (e^T Sigma^-1) . e
		double w;
		acc += robust_loss<LOSS>(obs_sq_error(eu, ev, i01, i23), loss_k, w);
	}
	acc = warp_sum(acc);
	if((threadIdx.x & 31) == 0) sred[threadIdx.x >> 5] = acc;
	__syncthreads();
	if(threadIdx.x == 0) {
		double v = sred[0];
		for(int w = 1; w < RED_THREADS / 32; ++ w) v += sred[w];
		partial[blockIdx.x] = v;
	}
}

// s2 and w of every observation at the current states, written in edge insertion order (spp_ba_get_observation_errors).
// The residual comes from observation_jacobians in the Jacobian mode JAC (FD: project_Rt of the base pose, analytic:
// project_with_dx), as in k_linearise_cams, so w is bit for bit the weight of the linearisation.
template <int JAC, int LOSS>
__global__ void __launch_bounds__(RED_THREADS) k_obs_errors(size_t O, const uint32_t *__restrict__ obs_cam,
	const uint32_t *__restrict__ obs_pt, const uint32_t *__restrict__ obs_orig, const double *__restrict__ pts,
	const double *__restrict__ z, const double *__restrict__ info, const double *__restrict__ camRt,
	const double *__restrict__ camK, double loss_k, double *__restrict__ sq_err, double *__restrict__ weight)
{
	const size_t o = blockIdx.x * (size_t)RED_THREADS + threadIdx.x;
	if(o >= O)
		return;
	const unsigned c = obs_cam[o], p = obs_pt[o];
	const double2 zz = *reinterpret_cast<const double2*>(z + o * 2);
	const double2 i01 = *reinterpret_cast<const double2*>(info + o * 4);
	const double2 i23 = *reinterpret_cast<const double2*>(info + o * 4 + 2);
	double Jc[12], Jp[6], ru, rv;
	observation_jacobians(JAC, camRt + (size_t)c * 84, camK + (size_t)c * 5, pts[(size_t)p * 3], pts[(size_t)p * 3 + 1],
		pts[(size_t)p * 3 + 2], zz.x, zz.y, Jc, Jp, ru, rv, false, false);
	const double s2 = obs_sq_error(ru, rv, i01, i23);
	double w;
	robust_loss<LOSS>(s2, loss_k, w);
	const size_t e = obs_orig[o];
	sq_err[e] = s2;
	weight[e] = w;
}

// out[k] = sum_i partial[k * stride + i], i < n ; single block, fixed order
__global__ void __launch_bounds__(RED_THREADS) k_final_sum(const double *__restrict__ partial, size_t n, size_t stride,
	double *__restrict__ out)
{
	__shared__ double sred[RED_THREADS / 32];
	const double *src = partial + blockIdx.x * stride;
	double acc = 0;
	for(size_t i = threadIdx.x; i < n; i += RED_THREADS)
		acc += src[i];
	acc = warp_sum(acc);
	if((threadIdx.x & 31) == 0) sred[threadIdx.x >> 5] = acc;
	__syncthreads();
	if(threadIdx.x == 0) {
		double v = sred[0];
		for(int w = 1; w < RED_THREADS / 32; ++ w) v += sred[w];
		out[blockIdx.x] = v;
	}
}

// partial[0*G + b] = sum dx.dx ; partial[1*G + b] = sum dx.(alpha dx + eta) over this block's slice
__global__ void __launch_bounds__(RED_THREADS) k_step_dots(size_t n, const double *__restrict__ dx,
	const double *__restrict__ eta, double alpha, double w_norm, double *__restrict__ partial, size_t G, int accumulate)
{
	__shared__ double sred[2][RED_THREADS / 32];
	double a0 = 0, a1 = 0;
	for(size_t i = blockIdx.x * (size_t)RED_THREADS + threadIdx.x; i < n; i += (size_t)gridDim.x * RED_THREADS) {
		double d = dx[i];
		a0 += w_norm * d * d;
		a1 += d * (alpha * d + eta[i]);
	}
	a0 = warp_sum(a0); a1 = warp_sum(a1);
	if((threadIdx.x & 31) == 0) { sred[0][threadIdx.x >> 5] = a0; sred[1][threadIdx.x >> 5] = a1; }
	__syncthreads();
	if(threadIdx.x == 0) {
		double v0 = sred[0][0], v1 = sred[1][0];
		for(int w = 1; w < RED_THREADS / 32; ++ w) { v0 += sred[0][w]; v1 += sred[1][w]; }
		if(accumulate) { v0 += partial[blockIdx.x]; v1 += partial[G + blockIdx.x]; }
		partial[blockIdx.x] = v0;
		partial[G + blockIdx.x] = v1;
	}
}

// x <- x (+) dx : cameras through the SE(3) composition, points additively
__global__ void k_update_cams(size_t C, double *__restrict__ cam_state, const double *__restrict__ dxc)
{
	size_t c = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
	if(c >= C) return;
	double v1[6], v2[6], d[6];
	#pragma unroll
	for(int k = 0; k < 6; ++ k) { v1[k] = cam_state[c * 6 + k]; v2[k] = dxc[c * 6 + k]; }
	relative_to_absolute(v1, v2, d);
	#pragma unroll
	for(int k = 0; k < 6; ++ k) cam_state[c * 6 + k] = d[k];
}

__global__ void k_axpy(size_t n, double *__restrict__ x, const double *__restrict__ dx)
{
	size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
	if(i < n) x[i] += dx[i];
}

// ---------------------------------------------------------------------------------------------------
// launch wrappers

#define LAUNCH_CHECK(ctx) do { ++ (ctx)->n_launches; SPP_CUDA(cudaGetLastError()); } while(0)

void ba_prepare_cameras(spp_ctx *ctx, bool b_with_perturbations)
{
	BAProblem &ba = ctx->ba;
	SchurSystem &s = ctx->sys;
	if(!s.C) return;
	// the base pose only (chi2) still uses the 7-slot layout
	int nv = b_with_perturbations? 7 : 1;
	size_t n = s.C * nv;
	k_cam_prepare<<<n_blocks(n, 128), 128, 0, ctx->stream>>>(s.C, ba.cam_state.p(), ba.cam_intr.p(),
		ba.camRt.p(), ba.camK.p(), nv);
	LAUNCH_CHECK(ctx);
}

template <int JAC, int LOSS>
static void launch_linearise_cams(spp_ctx *ctx, unsigned long long *p_max)
{
	BAProblem &ba = ctx->ba;
	SchurSystem &s = ctx->sys;
	k_linearise_cams<JAC, LOSS><<<(unsigned)s.C, CAM_THREADS, CAM_SMEM, ctx->stream>>>(ba.jac_mode, s.cam_ptr.p(),
		s.cam_obs.p(), s.obs_pt.p(), ba.pts.p(), ba.z.p(), ba.info.p(), ba.camRt.p(), ba.camK.p(), s.W.p(), s.U.p(), s.gc.p(),
		p_max, ba.uf_is_cam? ba.uf_index : -1, ba.pt_rec.p(), ba.loss_scale);
}

template <int JAC>
static void launch_linearise_cams_loss(spp_ctx *ctx, unsigned long long *p_max)
{
	switch(ctx->ba.loss_kind) {
	case SPP_LOSS_HUBER: launch_linearise_cams<JAC, SPP_LOSS_HUBER>(ctx, p_max); break;
	case SPP_LOSS_CAUCHY: launch_linearise_cams<JAC, SPP_LOSS_CAUCHY>(ctx, p_max); break;
	default: launch_linearise_cams<JAC, SPP_LOSS_NONE>(ctx, p_max); break;
	}
}

template <int JAC>
static void set_linearise_cams_smem()
{
	SPP_CUDA(cudaFuncSetAttribute(k_linearise_cams<JAC, SPP_LOSS_NONE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CAM_SMEM));
	SPP_CUDA(cudaFuncSetAttribute(k_linearise_cams<JAC, SPP_LOSS_HUBER>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CAM_SMEM));
	SPP_CUDA(cudaFuncSetAttribute(k_linearise_cams<JAC, SPP_LOSS_CAUCHY>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CAM_SMEM));
}

void ba_linearise(spp_ctx *ctx, bool b_want_maxdiag)
{
	BAProblem &ba = ctx->ba;
	SchurSystem &s = ctx->sys;
	ba_prepare_cameras(ctx, ba.jac_mode == SPP_JAC_FD_REFERENCE);
	unsigned long long *p_max = 0;
	if(b_want_maxdiag) {
		ba.maxdiag.resize(1);
		ba.maxdiag.zero(ctx->stream);
		p_max = ba.maxdiag.p();
	}
	ba.pt_rec.resize(s.O * 10);
	if(s.C) {
		static bool attr_done[64] = {false};
		if(ctx->device >= 0 && ctx->device < 64 && !attr_done[ctx->device]) {
			set_linearise_cams_smem<SPP_JAC_FD_REFERENCE>();
			set_linearise_cams_smem<SPP_JAC_ANALYTIC>();
			attr_done[ctx->device] = true;
		}
		if(ba.jac_mode == SPP_JAC_FD_REFERENCE)
			launch_linearise_cams_loss<SPP_JAC_FD_REFERENCE>(ctx, p_max);
		else
			launch_linearise_cams_loss<SPP_JAC_ANALYTIC>(ctx, p_max);
		LAUNCH_CHECK(ctx);
	}
	if(s.P) {
		k_sum_point_records<<<n_blocks(s.P, SR_WARPS * 32), SR_WARPS * 32, 0, ctx->stream>>>(s.P, s.pt_ptr.p(), ba.pt_rec.p(), s.V.p(), s.gp.p(),
			ba.uf_is_cam? -1 : ba.uf_index);
		LAUNCH_CHECK(ctx);
	}
	ba.linearised = true;
}

// leaves the (local) chi2 in d_out[0]
void ba_chi2_device(spp_ctx *ctx, double *d_out)
{
	BAProblem &ba = ctx->ba;
	SchurSystem &s = ctx->sys;
	ba_prepare_cameras(ctx, false);
	const unsigned G = 148 * 4;
	ba.partial.resize(4 * 1024);
#define LAUNCH_CHI2(LOSS) k_chi2_partial<LOSS><<<G, RED_THREADS, 0, ctx->stream>>>(s.O, s.obs_cam.p(), s.obs_pt.p(), ba.pts.p(), \
		ba.z.p(), ba.info.p(), ba.camRt.p(), ba.camK.p(), ba.partial.p(), ba.loss_scale)
	switch(ba.loss_kind) {
	case SPP_LOSS_HUBER: LAUNCH_CHI2(SPP_LOSS_HUBER); break;
	case SPP_LOSS_CAUCHY: LAUNCH_CHI2(SPP_LOSS_CAUCHY); break;
	default: LAUNCH_CHI2(SPP_LOSS_NONE); break;
	}
#undef LAUNCH_CHI2
	LAUNCH_CHECK(ctx);
	k_final_sum<<<1, RED_THREADS, 0, ctx->stream>>>(ba.partial.p(), G, 0, d_out);
	LAUNCH_CHECK(ctx);
}

template <int JAC>
static void launch_obs_errors(spp_ctx *ctx, double *d_sq_err, double *d_weight)
{
	BAProblem &ba = ctx->ba;
	SchurSystem &s = ctx->sys;
#define LAUNCH_ERR(LOSS) k_obs_errors<JAC, LOSS><<<n_blocks(s.O, RED_THREADS), RED_THREADS, 0, ctx->stream>>>(s.O, s.obs_cam.p(), \
		s.obs_pt.p(), ba.d_obs_orig.p(), ba.pts.p(), ba.z.p(), ba.info.p(), ba.camRt.p(), ba.camK.p(), ba.loss_scale, d_sq_err, d_weight)
	switch(ba.loss_kind) {
	case SPP_LOSS_HUBER: LAUNCH_ERR(SPP_LOSS_HUBER); break;
	case SPP_LOSS_CAUCHY: LAUNCH_ERR(SPP_LOSS_CAUCHY); break;
	default: LAUNCH_ERR(SPP_LOSS_NONE); break;
	}
#undef LAUNCH_ERR
}

// d_sq_err[O], d_weight[O]: s2 and w of every observation at the current states, in edge insertion order
void ba_obs_errors_device(spp_ctx *ctx, double *d_sq_err, double *d_weight)
{
	BAProblem &ba = ctx->ba;
	SchurSystem &s = ctx->sys;
	if(!s.O)
		return;
	ba_prepare_cameras(ctx, false); // the base pose: all the residual needs in either Jacobian mode
	if(ba.jac_mode == SPP_JAC_FD_REFERENCE)
		launch_obs_errors<SPP_JAC_FD_REFERENCE>(ctx, d_sq_err, d_weight);
	else
		launch_obs_errors<SPP_JAC_ANALYTIC>(ctx, d_sq_err, d_weight);
	LAUNCH_CHECK(ctx);
}

// d_out[0] = |dx|^2, d_out[1] = dx . (alpha dx + eta) over cameras and points
void ba_step_dots_device(spp_ctx *ctx, double alpha, double *d_out)
{
	BAProblem &ba = ctx->ba;
	SchurSystem &s = ctx->sys;
	const unsigned G = 148 * 2;
	ba.partial.resize(4 * 1024);
	// multi-GPU: the camera increments are replicated while eta_c is a per-rank partial sum: every rank adds
	// dx_c . eta_c(partial), only rank 0 adds |dx_c|^2 and alpha |dx_c|^2; landmarks are disjoint
	const bool first = ctx->rank == 0;
	k_step_dots<<<G, RED_THREADS, 0, ctx->stream>>>(s.C * 6, s.dxc.p(), s.gc.p(), first? alpha : 0.0, first? 1.0 : 0.0,
		ba.partial.p(), G, 0);
	LAUNCH_CHECK(ctx);
	k_step_dots<<<G, RED_THREADS, 0, ctx->stream>>>(s.P * 3, s.dxp.p(), s.gp.p(), alpha, 1.0, ba.partial.p(), G, 1);
	LAUNCH_CHECK(ctx);
	k_final_sum<<<2, RED_THREADS, 0, ctx->stream>>>(ba.partial.p(), G, G, d_out);
	LAUNCH_CHECK(ctx);
}

void ba_apply_update(spp_ctx *ctx)
{
	BAProblem &ba = ctx->ba;
	SchurSystem &s = ctx->sys;
	if(s.C) {
		k_update_cams<<<n_blocks(s.C, 128), 128, 0, ctx->stream>>>(s.C, ba.cam_state.p(), s.dxc.p());
		LAUNCH_CHECK(ctx);
	}
	if(s.P) {
		k_axpy<<<n_blocks(s.P * 3, 256), 256, 0, ctx->stream>>>(s.P * 3, ba.pts.p(), s.dxp.p());
		LAUNCH_CHECK(ctx);
	}
}

} // namespace spp

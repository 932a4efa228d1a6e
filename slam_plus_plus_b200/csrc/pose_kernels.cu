// pose_kernels.cu -- stage 1 of the hot path for pose graphs: per-edge linearisation of the SE(2) pose-pose edges,
// deterministic accumulation into the block Hessian / gradient, chi2 and the vertex update; plus the Gauss-Newton
// control flow of CNonlinearSolver_Lambda::Optimize.
//
// Reference functions replaced (SURVEY 8(a) rows a4, a2, a5, a17, a18 for pose graphs):
//   CEdgePose2D::Calculate_Jacobians_Expectation_Error   include/slam/SE2_Types.h:308-319
//   C2DJacobians::Absolute_to_Relative (analytic J)      include/slam/2DSolverBase.h:373-430, angle clamps :44-95
//   CBaseEdgeImpl::Calculate_Hessians_v2                 include/slam/BaseTypes_Binary.h:759-848
//   CMatrixReductionPlan / CVectorReductionPlan          include/slam/NonlinearSolver_Lambda_Base.h:152-197, 563-607
//   unary factor on vertex 0                             include/slam/NonlinearSolver_Lambda_Base.h:1903-1923
//   CEdgePose2D::f_Chi_Squared_Error                     include/slam/SE2_Types.h:325-335
//   CVertexPose2D::Operator_Plus                         include/slam/SE2_Types.h:70-74
//   CNonlinearSolver_Lambda::Optimize                    include/slam/NonlinearSolver_Lambda.h:476-667
//
// Like the reference, every edge first writes its own contributions (J0^T W J0, J0^T W J1, J1^T W J1, J0^T W r,
// J1^T W r) and every destination block then sums its sources in edge insertion order: no atomics, bit-reproducible,
// duplicate edges between the same pair of poses simply give a longer source list. lambda is produced directly in
// the reference's layout (upper block-triangular, vertex order, column-major blocks), which is also what the
// block-sparse Cholesky (sparse_chol.cu) consumes.

#include "spp_ctx.h"
#include "ba_geometry.cuh"
#include <math.h>
#include <algorithm>
#include <map>

namespace spp {

void sparse_chol_symbolic(spp_ctx *ctx, int owner, size_t n, size_t B, const uint64_t *col_ptr, const uint64_t *row_idx,
	const uint64_t *p_order_in);
int sparse_chol_solve_device(spp_ctx *ctx, const double *d_A, const double *d_rhs, double *d_x);

#define LAUNCH_CHECK(ctx) do { ++ (ctx)->n_launches; SPP_CUDA(cudaGetLastError()); } while(0)

// 2DSolverBase.h:44-95
__device__ __forceinline__ double clamp_angle_2pi(double a)
{
	return isfinite(a)? fmod(a, M_PI * 2) : 0.0;
}

__device__ __forceinline__ double min_abs_3(double a, double b, double c)
{
	const double m = (fabs(a) < fabs(b))? a : b;
	return (fabs(m) < fabs(c))? m : c;
}

__device__ __forceinline__ double clamp_angular_error_2pi(double e)
{
	e = clamp_angle_2pi(e);
	return min_abs_3(e, e - 2 * M_PI, e + 2 * M_PI);
}

// 2DSolverBase.h:373-430: expectation of the relative pose and its Jacobians (row-major 3 x 3)
__device__ __forceinline__ void se2_absolute_to_relative(const double *v1, const double *v2, double *d, double *J1, double *J2)
{
	const double p1e = v1[0], p1n = v1[1], p1a = v1[2], p2e = v2[0], p2n = v2[1], p2a = v2[2];
	const double de = p2e - p1e, dn = p2n - p1n, da = p2a - p1a;
	const double o = -p1a;
	const double co = cos(o), so = sin(o);
	d[0] = co * de - so * dn;
	d[1] = so * de + co * dn;
	d[2] = clamp_angle_2pi(da);
	if(J1) {
		const double cp1a = cos(p1a), sp1a = sin(p1a);
		J1[0] = -cp1a; J1[1] = -sp1a; J1[2] = sp1a * (p1e - p2e) - cp1a * (p1n - p2n);
		J1[3] = sp1a;  J1[4] = -cp1a; J1[5] = cp1a * (p1e - p2e) + sp1a * (p1n - p2n);
		J1[6] = 0;     J1[7] = 0;     J1[8] = -1;
		J2[0] = cp1a;  J2[1] = sp1a;  J2[2] = 0;
		J2[3] = -sp1a; J2[4] = cp1a;  J2[5] = 0;
		J2[6] = 0;     J2[7] = 0;     J2[8] = 1;
	}
}

// per-edge record: H00 (9), H01 (9), H11 (9), g0 (3), g1 (3); blocks column-major
#define SE2_REC 33

__global__ void k_se2_edges(size_t E, const double *__restrict__ states, const uint32_t *__restrict__ e_from,
	const uint32_t *__restrict__ e_to, const double *__restrict__ z, const double *__restrict__ info, double *__restrict__ rec)
{
	size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
	if(e >= E) return;
	const double *v0 = states + (size_t)e_from[e] * 3, *v1 = states + (size_t)e_to[e] * 3;
	double d[3], J0[9], J1[9], r[3];
	se2_absolute_to_relative(v0, v1, d, J0, J1);
	r[0] = z[e * 3] - d[0];
	r[1] = z[e * 3 + 1] - d[1];
	r[2] = clamp_angular_error_2pi(z[e * 3 + 2] - d[2]);
	const double *W = info + e * 9; // row-major (symmetric)
	// T = J0^T W (3 x 3), row-major: T(i, j) = sum_k J0(k, i) W(k, j)
	double T[9], WJ1[9], Wr[3];
	#pragma unroll
	for(int i = 0; i < 3; ++ i)
		#pragma unroll
		for(int j = 0; j < 3; ++ j)
			T[i * 3 + j] = J0[0 * 3 + i] * W[0 * 3 + j] + J0[1 * 3 + i] * W[1 * 3 + j] + J0[2 * 3 + i] * W[2 * 3 + j];
	#pragma unroll
	for(int i = 0; i < 3; ++ i) {
		#pragma unroll
		for(int j = 0; j < 3; ++ j)
			WJ1[i * 3 + j] = W[i * 3 + 0] * J1[0 * 3 + j] + W[i * 3 + 1] * J1[1 * 3 + j] + W[i * 3 + 2] * J1[2 * 3 + j];
		Wr[i] = W[i * 3 + 0] * r[0] + W[i * 3 + 1] * r[1] + W[i * 3 + 2] * r[2];
	}
	double *out = rec + e * SE2_REC;
	#pragma unroll
	for(int c = 0; c < 3; ++ c) {
		#pragma unroll
		for(int rr = 0; rr < 3; ++ rr) {
			// the reference mirrors the upper triangle of the vertex blocks (selfadjointView<Upper>)
			const int a = (rr <= c)? rr : c, b = (rr <= c)? c : rr;
			out[c * 3 + rr] = T[a * 3 + 0] * J0[0 * 3 + b] + T[a * 3 + 1] * J0[1 * 3 + b] + T[a * 3 + 2] * J0[2 * 3 + b];
			out[9 + c * 3 + rr] = T[rr * 3 + 0] * J1[0 * 3 + c] + T[rr * 3 + 1] * J1[1 * 3 + c] + T[rr * 3 + 2] * J1[2 * 3 + c];
			out[18 + c * 3 + rr] = J1[0 * 3 + a] * WJ1[0 * 3 + b] + J1[1 * 3 + a] * WJ1[1 * 3 + b] + J1[2 * 3 + a] * WJ1[2 * 3 + b];
		}
	}
	#pragma unroll
	for(int i = 0; i < 3; ++ i) {
		out[27 + i] = T[i * 3 + 0] * r[0] + T[i * 3 + 1] * r[1] + T[i * 3 + 2] * r[2];
		out[30 + i] = J1[0 * 3 + i] * Wr[0] + J1[1 * 3 + i] * Wr[1] + J1[2 * 3 + i] * Wr[2];
	}
}

// ---- SE(3) (SURVEY 8(a) row a3) --------------------------------------------------------------------------------------
//   CEdgePose3D::Calculate_Jacobians_Expectation_Error   include/slam/SE3_Types.h:265-288
//   C3DJacobians::Absolute_to_Relative, forward differences, delta = 1e-9: 13 Absolute_to_Relative and 12
//   Relative_to_Absolute evaluations per edge            include/slam/3DSolverBase.h:892-946, 1043-1059, 1332-1370
//   Huber weight, CRobustify_ErrorNorm_Default<30/100>   include/slam/SE3_Types.h:128-129, RobustUtils.h:412-438,
//                                                        include/geometry/RobustLoss.h:63,100-104
//   robust Calculate_Hessians_v2                         include/slam/BaseTypes_Binary.h:759-848 (the weight enters the
//                                                        gradient of vertex 0 twice and that of vertex 1 once, :820-843)
//   CVertexPose3D::Operator_Plus = Relative_to_Absolute  include/slam/SE3_Types.h:45-48

// error of an SE(3) edge given the expectation d
__device__ __forceinline__ void se3_error(const double *z, const double *d, double *r)
{
	r[0] = z[0] - d[0]; r[1] = z[1] - d[1]; r[2] = z[2] - d[2];
	Quat pq, dq;
	axis_angle_to_quat(z[3], z[4], z[5], pq);
	axis_angle_to_quat(d[3], d[4], d[5], dq);
	const Quat e = quat_mul(pq, quat_conj(dq));
	quat_to_axis_angle(e, r[3], r[4], r[5]);
}

__device__ __forceinline__ double se3_robust_weight(const double *r)
{
	double s = 0;
	#pragma unroll
	for(int i = 0; i < 6; ++ i) s += r[i] * r[i];
	const double e = sqrt(s) / (30.0 / 100.0);
	return (e <= 1.345)? 1.0 : 1.345 / e;
}

// per-edge record: H00 (36), H01 (36), H11 (36), g0 (6), g1 (6); blocks column-major
#define SE3_REC 120
#define SE3_EDGES_PER_CTA 8

// 16 lanes per edge: lane 0 evaluates the expectation, lanes 1..6 / 7..12 the perturbed expectations for the columns of
// J0 / J1 (the 25 pose compositions of an edge run side by side instead of one after the other); the 6 x 6 products are
// then spread over the 16 lanes through shared memory.
__global__ void __launch_bounds__(SE3_EDGES_PER_CTA * 16) k_se3_edges(size_t E, const double *__restrict__ states,
	const uint32_t *__restrict__ e_from, const uint32_t *__restrict__ e_to, const double *__restrict__ z,
	const double *__restrict__ info, double *__restrict__ rec)
{
	__shared__ double sD[SE3_EDGES_PER_CTA][13][6]; // expectation and the 12 perturbed expectations
	__shared__ double sJ[SE3_EDGES_PER_CTA][2][36]; // J0, J1 row-major
	__shared__ double sT[SE3_EDGES_PER_CTA][2][36]; // T = J0^T W w, WJ1 = W J1
	__shared__ double sR[SE3_EDGES_PER_CTA][16];    // r (6), W r (6), w
	const int sub = threadIdx.x & 15, le = threadIdx.x >> 4;
	const size_t e = blockIdx.x * (size_t)SE3_EDGES_PER_CTA + le;
	const bool live = e < E;
	const size_t ee = live? e : 0;
	const double *v0 = states + (size_t)e_from[ee] * 6, *v1 = states + (size_t)e_to[ee] * 6;
	if(sub < 13) {
		double a[6], b[6], eps[6] = {0, 0, 0, 0, 0, 0}, d[6];
		#pragma unroll
		for(int i = 0; i < 6; ++ i) { a[i] = v0[i]; b[i] = v1[i]; }
		if(sub >= 1 && sub <= 6) {
			eps[sub - 1] = 1e-9;
			relative_to_absolute(a, eps, a);
		} else if(sub >= 7) {
			eps[sub - 7] = 1e-9;
			relative_to_absolute(b, eps, b);
		}
		absolute_to_relative(a, b, d);
		#pragma unroll
		for(int i = 0; i < 6; ++ i) sD[le][sub][i] = d[i];
	}
	__syncthreads();
	// Jacobians: J(i, j) = (d_j(i) - d(i)) * (1 / delta); 72 entries over 16 lanes
	const double scalar = 1.0 / 1e-9;
	for(int k = sub; k < 72; k += 16) {
		const int m = k / 36, q = k - m * 36, i = q / 6, j = q - i * 6;
		sJ[le][m][i * 6 + j] = (sD[le][1 + m * 6 + j][i] - sD[le][0][i]) * scalar;
	}
	if(sub == 0) {
		double r[6];
		se3_error(z + ee * 6, sD[le][0], r);
		#pragma unroll
		for(int i = 0; i < 6; ++ i) sR[le][i] = r[i];
		sR[le][12] = se3_robust_weight(r);
	}
	__syncthreads();
	const double *W = info + ee * 36; // row-major
	const double w = sR[le][12];
	const double *J0 = sJ[le][0], *J1 = sJ[le][1];
	for(int k = sub; k < 72; k += 16) {
		const int m = k / 36, q = k - m * 36, i = q / 6, j = q - i * 6;
		double t = 0;
		if(m == 0) { // T(i, j) = (sum_k J0(k, i) W(k, j)) * w
			#pragma unroll
			for(int c = 0; c < 6; ++ c) t += J0[c * 6 + i] * W[c * 6 + j];
			t *= w;
		} else {     // WJ1(i, j) = sum_k W(i, k) J1(k, j)
			#pragma unroll
			for(int c = 0; c < 6; ++ c) t += W[i * 6 + c] * J1[c * 6 + j];
		}
		sT[le][m][q] = t;
	}
	if(sub < 6) {
		double t = 0;
		#pragma unroll
		for(int c = 0; c < 6; ++ c) t += W[sub * 6 + c] * sR[le][c];
		sR[le][6 + sub] = t;
	}
	__syncthreads();
	if(!live) return;
	const double *T = sT[le][0], *WJ1 = sT[le][1];
	double *out = rec + e * SE3_REC;
	for(int k = sub; k < 120; k += 16) {
		double v = 0;
		if(k < 108) {
			const int part = k / 36, q = k - part * 36, c = q / 6, rr = q - c * 6; // column-major block element (rr, c)
			const int a = (rr <= c)? rr : c, b = (rr <= c)? c : rr; // vertex blocks are mirrored from the upper triangle
			if(part == 0) {
				#pragma unroll
				for(int i = 0; i < 6; ++ i) v += T[a * 6 + i] * J0[i * 6 + b];
			} else if(part == 1) {
				#pragma unroll
				for(int i = 0; i < 6; ++ i) v += T[rr * 6 + i] * J1[i * 6 + c];
			} else {
				#pragma unroll
				for(int i = 0; i < 6; ++ i) v += J1[i * 6 + a] * WJ1[i * 6 + b];
				v *= w;
			}
		} else if(k < 114) {
			const int i = k - 108;
			#pragma unroll
			for(int c = 0; c < 6; ++ c) v += T[i * 6 + c] * sR[le][c];
			v *= w;
		} else {
			const int i = k - 114;
			#pragma unroll
			for(int c = 0; c < 6; ++ c) v += J1[c * 6 + i] * sR[le][6 + c];
			v *= w;
		}
		out[k] = v;
	}
}

__global__ void k_se3_chi2(size_t E, const double *__restrict__ states, const uint32_t *__restrict__ e_from,
	const uint32_t *__restrict__ e_to, const double *__restrict__ z, const double *__restrict__ info, double *__restrict__ out)
{
	size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
	if(e >= E) return;
	double d[6], r[6];
	absolute_to_relative(states + (size_t)e_from[e] * 6, states + (size_t)e_to[e] * 6, d);
	se3_error(z + e * 6, d, r);
	const double *W = info + e * 36;
	double s = 0;
	#pragma unroll
	for(int i = 0; i < 6; ++ i) {
		double t = 0;
		#pragma unroll
		for(int k = 0; k < 6; ++ k) t += W[i * 6 + k] * r[k];
		s += r[i] * t;
	}
	out[e] = s; // unweighted, as the reference's f_Chi_Squared_Error (SE3_Types.h:318-327)
}

__global__ void k_se3_update(size_t N, double *__restrict__ states, const double *__restrict__ dx)
{
	size_t v = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
	if(v >= N) return;
	double a[6], d[6];
	#pragma unroll
	for(int i = 0; i < 6; ++ i) { a[i] = states[v * 6 + i]; d[i] = dx[v * 6 + i]; }
	relative_to_absolute(a, d, a);
	#pragma unroll
	for(int i = 0; i < 6; ++ i) states[v * 6 + i] = a[i];
}

// thread per scalar of lambda / eta: sum of the sources in edge insertion order.
// source code: edge * 4 + part; part 0: H00, 1: H01 as is, 2: H01 transposed, 3: H11 (blocks); 0: g0, 1: g1 (vectors)
template <int B, int REC>
__global__ void k_pose_reduce(size_t n_blocks, size_t n_vertices, const uint64_t *__restrict__ blk_src_ptr,
	const uint64_t *__restrict__ blk_src, const uint64_t *__restrict__ vec_src_ptr, const uint64_t *__restrict__ vec_src,
	const double *__restrict__ rec, long uf_block, double *__restrict__ vals, double *__restrict__ eta)
{
	constexpr int BB = B * B;
	size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
	if(i < n_blocks * BB) {
		const size_t b = i / BB;
		const int k = int(i % BB), r = k % B, c = k / B;
		double s = 0;
		for(uint64_t q = blk_src_ptr[b]; q < blk_src_ptr[b + 1]; ++ q) {
			const uint64_t code = blk_src[q];
			const double *p = rec + (code >> 2) * REC;
			const int part = int(code & 3);
			s += (part == 0)? p[k] : ((part == 1)? p[BB + k] : ((part == 2)? p[BB + c + B * r] : p[2 * BB + k]));
		}
		if((long)b == uf_block && r == c)
			s += 1.0; // UF^T UF = I on the first vertex, added after the edges (Lambda_Base.h:1903-1923)
		vals[i] = s;
		return;
	}
	i -= n_blocks * BB;
	if(i < n_vertices * B) {
		const size_t v = i / B;
		const int k = int(i % B);
		double s = 0;
		for(uint64_t q = vec_src_ptr[v]; q < vec_src_ptr[v + 1]; ++ q) {
			const uint64_t code = vec_src[q];
			s += rec[(code >> 2) * REC + 3 * BB + (code & 3) * B + k];
		}
		eta[i] = s;
	}
}

// chi2 per edge, then a fixed-order tree (deterministic); the reference sums serially in edge order
__global__ void k_se2_chi2(size_t E, const double *__restrict__ states, const uint32_t *__restrict__ e_from,
	const uint32_t *__restrict__ e_to, const double *__restrict__ z, const double *__restrict__ info, double *__restrict__ out)
{
	size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
	if(e >= E) return;
	double d[3], r[3];
	se2_absolute_to_relative(states + (size_t)e_from[e] * 3, states + (size_t)e_to[e] * 3, d, 0, 0);
	r[0] = z[e * 3] - d[0];
	r[1] = z[e * 3 + 1] - d[1];
	r[2] = clamp_angular_error_2pi(z[e * 3 + 2] - d[2]);
	const double *W = info + e * 9;
	double s = 0;
	#pragma unroll
	for(int i = 0; i < 3; ++ i)
		s += r[i] * (W[i * 3] * r[0] + W[i * 3 + 1] * r[1] + W[i * 3 + 2] * r[2]);
	out[e] = s;
}

// one CTA: out[0] = sum of in[0 .. n) in a fixed order (thread-strided partial sums, then a tree); out[1] likewise
// for in2 if given
__global__ void __launch_bounds__(1024) k_sum_fixed(size_t n, const double *__restrict__ in, size_t n2, const double *__restrict__ in2,
	double *__restrict__ out)
{
	__shared__ double sh[1024];
	for(int pass = 0; pass < 2; ++ pass) {
		const double *p = pass? in2 : in;
		const size_t m = pass? n2 : n;
		if(!p) break;
		double s = 0;
		for(size_t i = threadIdx.x; i < m; i += 1024)
			s += p[i];
		sh[threadIdx.x] = s;
		__syncthreads();
		for(int w = 512; w > 0; w >>= 1) {
			if((int)threadIdx.x < w) sh[threadIdx.x] += sh[threadIdx.x + w];
			__syncthreads();
		}
		if(threadIdx.x == 0) out[pass] = sh[0];
		__syncthreads();
	}
}

__global__ void k_square(size_t n, const double *__restrict__ x, double *__restrict__ out)
{
	size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
	if(i < n) out[i] = x[i] * x[i];
}

// CVertexPose2D::Operator_Plus: x += dx, angle clamped
__global__ void k_se2_update(size_t N, double *__restrict__ states, const double *__restrict__ dx)
{
	size_t v = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
	if(v >= N) return;
	states[v * 3] += dx[v * 3];
	states[v * 3 + 1] += dx[v * 3 + 1];
	states[v * 3 + 2] = clamp_angle_2pi(states[v * 3 + 2] + dx[v * 3 + 2]);
}

// ---------------------------------------------------------------------------------------------------

// builds the structure of lambda (upper block CSC in vertex order) and the source lists; uploads the graph
void pose_set_graph(spp_ctx *ctx, int dim, size_t N, const double *p_states, size_t E, const uint64_t *p_from,
	const uint64_t *p_to, const double *p_z, const double *p_info)
{
	PoseProblem &pp = ctx->pose;
	pp.valid = false;
	if(dim != 3 && dim != 6)
		throw invalid_error("pose graphs: dim must be 3 (SE(2)) or 6 (SE(3))");
	if(N >= 0x7fffffffu || E >= 0x3fffffffu)
		throw invalid_error("pose graph too large for 32-bit indices");
	pp.dim = dim; pp.N = N; pp.E = E;
	const size_t B = dim;
	std::vector<uint32_t> ef(E), et(E);
	std::vector<std::map<uint32_t, uint32_t> > cols(N); // column -> (row -> block slot within the column)
	for(size_t v = 0; v < N; ++ v)
		cols[v][(uint32_t)v] = 0;
	for(size_t e = 0; e < E; ++ e) {
		if(p_from[e] >= N || p_to[e] >= N || p_from[e] == p_to[e])
			throw invalid_error("pose graph: edge references a vertex out of range (or a vertex with itself)");
		ef[e] = (uint32_t)p_from[e];
		et[e] = (uint32_t)p_to[e];
		cols[std::max(ef[e], et[e])][std::min(ef[e], et[e])] = 0;
	}
	// CSC, rows ascending (the diagonal block is the last of its column, as in the reference's lambda)
	pp.h_col_ptr.assign(N + 1, 0);
	pp.h_row_idx.clear();
	for(size_t c = 0; c < N; ++ c) {
		for(std::map<uint32_t, uint32_t>::iterator it = cols[c].begin(); it != cols[c].end(); ++ it) {
			it->second = (uint32_t)pp.h_row_idx.size();
			pp.h_row_idx.push_back(it->first);
		}
		pp.h_col_ptr[c + 1] = pp.h_row_idx.size();
	}
	const size_t nb = pp.h_row_idx.size();
	pp.n_blocks = nb;
	// source lists in edge insertion order
	std::vector<std::vector<uint64_t> > bsrc(nb), vsrc(N);
	for(size_t e = 0; e < E; ++ e) {
		const uint32_t a = ef[e], b = et[e];
		bsrc[cols[a][a]].push_back(e * 4 + 0);
		bsrc[cols[b][b]].push_back(e * 4 + 3);
		// H01 = J0^T W J1 is the block (vertex0, vertex1); stored transposed when id0 > id1 (BaseTypes_Binary.h:783-806)
		if(a < b) bsrc[cols[b][a]].push_back(e * 4 + 1);
		else bsrc[cols[a][b]].push_back(e * 4 + 2);
		vsrc[a].push_back(e * 4 + 0);
		vsrc[b].push_back(e * 4 + 1);
	}
	std::vector<uint64_t> bptr(nb + 1, 0), vptr(N + 1, 0), bflat, vflat;
	for(size_t b = 0; b < nb; ++ b) {
		bflat.insert(bflat.end(), bsrc[b].begin(), bsrc[b].end());
		bptr[b + 1] = bflat.size();
	}
	for(size_t v = 0; v < N; ++ v) {
		vflat.insert(vflat.end(), vsrc[v].begin(), vsrc[v].end());
		vptr[v + 1] = vflat.size();
	}
	pp.uf_block = N? (long)cols[0][0] : -1;
	cudaStream_t st = ctx->stream;
	pp.states.upload(p_states, N * B, st);
	pp.states0.upload(p_states, N * B, st);
	pp.e_from.upload(ef, st);
	pp.e_to.upload(et, st);
	pp.z.upload(p_z, E * B, st);
	pp.info.upload(p_info, E * B * B, st);
	pp.blk_src_ptr.upload(bptr, st);
	pp.blk_src.upload(bflat, st);
	pp.vec_src_ptr.upload(vptr, st);
	pp.vec_src.upload(vflat, st);
	pp.rec.resize(E * (dim == 3? SE2_REC : SE3_REC));
	pp.vals.resize(nb * B * B);
	pp.eta.resize(N * B);
	pp.dx.resize(N * B);
	pp.scratch.resize(std::max(E, N * B) + 16);
	SPP_CUDA(cudaStreamSynchronize(st));
	pp.symbolic_done = false;
	pp.linearised = false;
	pp.valid = true;
}

void pose_linearise(spp_ctx *ctx)
{
	PoseProblem &pp = ctx->pose;
	cudaStream_t st = ctx->stream;
	if(pp.dim == 6) {
		if(pp.E) {
			k_se3_edges<<<n_blocks(pp.E, SE3_EDGES_PER_CTA), SE3_EDGES_PER_CTA * 16, 0, st>>>(pp.E, pp.states.p(), pp.e_from.p(),
				pp.e_to.p(), pp.z.p(), pp.info.p(), pp.rec.p());
			LAUNCH_CHECK(ctx);
		}
		const size_t total = pp.n_blocks * 36 + pp.N * 6;
		k_pose_reduce<6, SE3_REC><<<n_blocks(total, 256), 256, 0, st>>>(pp.n_blocks, pp.N, pp.blk_src_ptr.p(), pp.blk_src.p(),
			pp.vec_src_ptr.p(), pp.vec_src.p(), pp.rec.p(), pp.uf_block, pp.vals.p(), pp.eta.p());
		LAUNCH_CHECK(ctx);
		pp.linearised = true;
		return;
	}
	if(pp.E) {
		k_se2_edges<<<n_blocks(pp.E, 128), 128, 0, st>>>(pp.E, pp.states.p(), pp.e_from.p(), pp.e_to.p(), pp.z.p(), pp.info.p(), pp.rec.p());
		LAUNCH_CHECK(ctx);
	}
	const size_t total = pp.n_blocks * 9 + pp.N * 3;
	k_pose_reduce<3, SE2_REC><<<n_blocks(total, 256), 256, 0, st>>>(pp.n_blocks, pp.N, pp.blk_src_ptr.p(), pp.blk_src.p(),
		pp.vec_src_ptr.p(), pp.vec_src.p(), pp.rec.p(), pp.uf_block, pp.vals.p(), pp.eta.p());
	LAUNCH_CHECK(ctx);
	pp.linearised = true;
}

double pose_chi2(spp_ctx *ctx)
{
	PoseProblem &pp = ctx->pose;
	cudaStream_t st = ctx->stream;
	if(!pp.E)
		return 0;
	if(pp.dim == 6)
		k_se3_chi2<<<n_blocks(pp.E, 64), 64, 0, st>>>(pp.E, pp.states.p(), pp.e_from.p(), pp.e_to.p(), pp.z.p(), pp.info.p(), pp.scratch.p());
	else
		k_se2_chi2<<<n_blocks(pp.E, 128), 128, 0, st>>>(pp.E, pp.states.p(), pp.e_from.p(), pp.e_to.p(), pp.z.p(), pp.info.p(), pp.scratch.p());
	LAUNCH_CHECK(ctx);
	k_sum_fixed<<<1, 1024, 0, st>>>(pp.E, pp.scratch.p(), 0, 0, pp.scratch.p() + pp.E);
	LAUNCH_CHECK(ctx);
	ctx->h_scalars.resize(16);
	SPP_CUDA(cudaMemcpyAsync(ctx->h_scalars.p(), pp.scratch.p() + pp.E, 8, cudaMemcpyDeviceToHost, st));
	SPP_CUDA(cudaStreamSynchronize(st));
	return ctx->h_scalars[0];
}

static double pose_dx_norm(spp_ctx *ctx)
{
	PoseProblem &pp = ctx->pose;
	cudaStream_t st = ctx->stream;
	const size_t n = pp.N * pp.dim;
	k_square<<<n_blocks(n, 256), 256, 0, st>>>(n, pp.dx.p(), pp.scratch.p());
	LAUNCH_CHECK(ctx);
	k_sum_fixed<<<1, 1024, 0, st>>>(n, pp.scratch.p(), 0, 0, pp.scratch.p() + n);
	LAUNCH_CHECK(ctx);
	ctx->h_scalars.resize(16);
	SPP_CUDA(cudaMemcpyAsync(ctx->h_scalars.p(), pp.scratch.p() + n, 8, cudaMemcpyDeviceToHost, st));
	SPP_CUDA(cudaStreamSynchronize(st));
	return sqrt(ctx->h_scalars[0]);
}

// one linear solve on the current linearisation: dx = lambda^-1 eta through the block-sparse Cholesky
int pose_solve(spp_ctx *ctx)
{
	PoseProblem &pp = ctx->pose;
	// FinalBlockStructure: once per structure (Lambda.h:607-612), and again after spp_chol_symbolic has put the slot's
	// analysis in the shared SparseChol
	if(!pp.symbolic_done || ctx->schol.owner != SC_OWNER_POSE) {
		sparse_chol_symbolic(ctx, SC_OWNER_POSE, pp.N, pp.dim, pp.h_col_ptr.data(), pp.h_row_idx.data(),
			pp.h_order_in.size() == pp.N? pp.h_order_in.data() : 0);
		pp.symbolic_done = true;
	}
	return sparse_chol_solve_device(ctx, pp.vals.p(), pp.eta.p(), pp.dx.p());
}

// CNonlinearSolver_Lambda::Optimize, Lambda.h:476-667 (batch use)
int pose_optimize(spp_ctx *ctx, size_t n_max_iteration_num, double f_min_dx_norm, spp_report_t *rep)
{
	PoseProblem &pp = ctx->pose;
	memset(rep, 0, sizeof(*rep));
	if(!pp.E)
		return SPP_OK; // "the system contains no edges at all: nothing to optimize"
	cudaStream_t st = ctx->stream;
	cudaEvent_t t0 = ctx->ev[2], t1 = ctx->ev[3], a = ctx->ev[0], b = ctx->ev[1];
	float ms;
	SPP_CUDA(cudaEventRecord(t0, st));
	rep->chi2_initial = rep->chi2_final = pose_chi2(ctx);
	bool b_dirty = true;
	for(size_t it = 0; it < n_max_iteration_num; ++ it) {
		if(b_dirty) {
			cudaEventRecord(a, st);
			pose_linearise(ctx);
			cudaEventRecord(b, st);
			cudaEventSynchronize(b);
			cudaEventElapsedTime(&ms, a, b);
			rep->ms_linearise += ms;
			b_dirty = false;
		}
		cudaEventRecord(a, st);
		int rc = pose_solve(ctx);
		cudaEventRecord(b, st);
		cudaEventSynchronize(b);
		cudaEventElapsedTime(&ms, a, b);
		rep->ms_factor += ms;
		const int k = rep->n_iterations ++;
		if(rc != SPP_OK) {
			rep->status = rc;
			break; // "Cholesky failed"
		}
		const double f_norm = pose_dx_norm(ctx);
		rep->last_dx_norm = f_norm;
		if(k < SPP_MAX_TRACE)
			rep->trace_dx_norm[k] = f_norm;
		if(f_norm <= f_min_dx_norm)
			break;
		cudaEventRecord(a, st);
		if(pp.dim == 6)
			k_se3_update<<<n_blocks(pp.N, 64), 64, 0, st>>>(pp.N, pp.states.p(), pp.dx.p());
		else
			k_se2_update<<<n_blocks(pp.N, 128), 128, 0, st>>>(pp.N, pp.states.p(), pp.dx.p()); // PushValuesInGraphSystem
		LAUNCH_CHECK(ctx);
		cudaEventRecord(b, st);
		cudaEventSynchronize(b);
		cudaEventElapsedTime(&ms, a, b);
		rep->ms_update += ms;
		b_dirty = true;
		++ rep->n_accepted;
		if(k < SPP_MAX_TRACE)
			rep->trace_accepted[k] = 1;
	}
	pp.linearised = !b_dirty;
	cudaEventRecord(a, st);
	rep->chi2_final = pose_chi2(ctx);
	cudaEventRecord(b, st);
	cudaEventSynchronize(b);
	cudaEventElapsedTime(&ms, a, b);
	rep->ms_chi2 += ms;
	SPP_CUDA(cudaEventRecord(t1, st));
	SPP_CUDA(cudaEventSynchronize(t1));
	cudaEventElapsedTime(&ms, t0, t1);
	rep->ms_total = ms;
	return SPP_OK;
}

} // namespace spp

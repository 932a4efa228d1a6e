// marginals.cu -- block diagonal of the covariance (Lambda + alpha I)^-1 recovered from the Schur-complemented system
// (SURVEY 8(f) rank 4).
//
// Reference replaced: CSchurComplement_Marginals::Schur_Marginals, include/slam/BAMarginals.h:579-760, as it is
// called at the end of CNonlinearSolver_Lambda_LM::Optimize() (NonlinearSolver_Lambda_LM.h:1118-1350, marginals policy
// mpart_Diagonal): with Lambda = [A U; U^T D], S = A - U D^-1 U^T = R^T R,
//     camera blocks    Sigma_cc = (S^-1)_cc                                              (BAMarginals.h:735-742)
//     landmark blocks  Sigma_pp = D_p^-1 + (R^-T U D^-1)_p^T (R^-T U D^-1)_p             (BAMarginals.h:671-699)
//                               = D_p^-1 + sum_{a,b in track(p)} Y_a^T (S^-1)_{c(a) c(b)} Y_b,   Y_o = W_o D_p^-1.
// The reference solves with R^T one camera at a time and keeps the sparse result; here S is dense (the dense-RCS
// path, 6C <= 16384), so S^-1 is formed once on the FP64 tensor pipe (dense_chol_inverse_device: panel factorisation of
// [S | I], then Z^T Z) and every landmark gathers the k x k camera blocks of its track from it.

#include "spp_ctx.h"
#include <vector>

namespace spp {

size_t dense_chol_ld(size_t n);
void schur_form_reduced_system(spp_ctx *ctx, double alpha, double alpha_diag, bool sparse_rcs);
int dense_chol_inverse_device(spp_ctx *ctx, double *A, size_t n);

#define LAUNCH_CHECK(ctx) do { ++ (ctx)->n_launches; SPP_CUDA(cudaGetLastError()); } while(0)

// element (r, c) of the symmetric matrix whose upper tiles hold MINUS the inverse
__device__ __forceinline__ double minus_inv_at(const double *__restrict__ Ni, size_t ld, unsigned r, unsigned c)
{
	return (r <= c)? Ni[(size_t)c * ld + r] : Ni[(size_t)r * ld + c];
}

// (-S^-1)_ab of the dense path: the upper tiles of minus the inverse, ld x ld
struct DenseMinusInverse {
	const double *Ni;
	size_t ld;
	struct Block {
		const double *Ni;
		size_t ld;
		unsigned r0, c0;
		__device__ __forceinline__ double operator()(int i, int j) const { return minus_inv_at(Ni, ld, r0 + i, c0 + j); }
	};
	__device__ __forceinline__ Block block(unsigned ca, unsigned cb) const { Block b = {Ni, ld, ca * 6, cb * 6}; return b; }
};

// (-S^-1)_ab after the selected inversion (selinv.cu): block (min(a, b), max(a, b)) of S is found by a binary search in
// its column of the upper block CSC; d_asm_dst gives where the factorisation assembled it in the panels, and so where
// Z holds it now (bit 63: stored transposed). A diagonal block is read through its upper triangle.
struct PanelInverse {
	const double *L;
	const uint64_t *csc_ptr, *dst;
	const uint32_t *csc_row, *csc_blk, *ld;
	struct Block {
		const double *P;
		size_t ld;
		int mode; // 0: as stored, 1: transposed, 2: symmetric
		__device__ __forceinline__ double operator()(int i, int j) const
		{
			const bool tr = mode == 1 || (mode == 2 && i > j);
			return -(tr? P[(size_t)i * ld + j] : P[(size_t)j * ld + i]);
		}
	};
	__device__ __forceinline__ Block block(unsigned ca, unsigned cb) const
	{
		const unsigned lo = min(ca, cb), hi = max(ca, cb);
		uint64_t a = csc_ptr[hi], b = csc_ptr[hi + 1]; // the last entry with row <= lo: the block (it is in the pattern)
		while(b - a > 1) {
			const uint64_t m = (a + b) >> 1;
			if(csc_row[m] <= lo) a = m; else b = m;
		}
		const uint32_t k = csc_blk[a];
		const uint64_t d = dst[k];
		Block r;
		r.P = L + (d & ~((uint64_t)1 << 63));
		r.ld = ld[k];
		r.mode = (ca == cb)? 2 : ((((d >> 63) != 0) != (ca > cb))? 1 : 0);
		return r;
	}
};

// thread per element: cov[c * 36 + i * 6 + j] = (S^-1)(6c + i, 6c + j)
__global__ void k_camera_marginals(size_t C, const double *__restrict__ Ni, size_t ld, double *__restrict__ cov)
{
	size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
	if(i >= C * 36) return;
	const unsigned c = (unsigned)(i / 36), e = (unsigned)(i % 36);
	cov[i] = -minus_inv_at(Ni, ld, c * 6 + e / 6, c * 6 + e % 6);
}

// warp per landmark: the k^2 (a, b) pairs of its track are dealt to the lanes, every lane adds Y_a^T (S^-1)_ab Y_b to
// its own 3 x 3 accumulator, a fixed-shape shuffle tree sums the lanes (no atomics: reproducible), lane 0 adds D^-1
// (Measured alternative: only the k (k + 1) / 2 pairs a <= b with X + X^T for a < b, triangular index decoded per pair --
// correct, but the whole call went from 13.9 ms to 40 - 70 ms on the Venice shape; the same happened with 16-byte loads of
// the stored block columns (LDG.128 in the SASS, 22 - 67 ms). Both runs were erratic from call to call, which the kernel
// alone does not explain; not resolved within the round's GPU budget -- the next step is a per-kernel ncu timing of both.)
// The blocks (-S^-1)_ab come from an accessor: DenseMinusInverse (the dense path) or PanelInverse (selected inversion on
// the supernodal panels).
#define PM_WARPS 4
template <class Inv>
__global__ void __launch_bounds__(PM_WARPS * 32) k_point_marginals(size_t P, const uint32_t *__restrict__ pt_ptr,
	const uint32_t *__restrict__ obs_cam, const double *__restrict__ Y, const double *__restrict__ Cinv,
	const Inv inv, double *__restrict__ cov)
{
	const size_t p = blockIdx.x * (size_t)PM_WARPS + (threadIdx.x >> 5);
	if(p >= P) return;
	const unsigned lane = threadIdx.x & 31;
	const unsigned beg = pt_ptr[p], k = pt_ptr[p + 1] - beg;
	double acc[9];
	#pragma unroll
	for(int i = 0; i < 9; ++ i) acc[i] = 0;
	const unsigned long long n_pairs = (unsigned long long)k * k;
	for(unsigned long long q = lane; q < n_pairs; q += 32) {
		const unsigned a = (unsigned)(q / k), b = (unsigned)(q % k);
		const unsigned ca = obs_cam[beg + a], cb = obs_cam[beg + b];
		const double *Ya = Y + (size_t)(beg + a) * 18, *Yb = Y + (size_t)(beg + b) * 18; // column-major 6 x 3
		double yb[18];
		#pragma unroll
		for(int i = 0; i < 18; i += 2) {
			double2 t = *reinterpret_cast<const double2*>(Yb + i);
			yb[i] = t.x; yb[i + 1] = t.y;
		}
		double t[18]; // t = (-S^-1)_ab Y_b, 6 x 3 column-major
		#pragma unroll
		for(int i = 0; i < 18; ++ i) t[i] = 0;
		const typename Inv::Block blk = inv.block(ca, cb);
		#pragma unroll
		for(int j = 0; j < 6; ++ j) {
			#pragma unroll
			for(int i = 0; i < 6; ++ i) {
				const double m = blk(i, j);
				t[i] += m * yb[j];
				t[6 + i] += m * yb[6 + j];
				t[12 + i] += m * yb[12 + j];
			}
		}
		#pragma unroll
		for(int r = 0; r < 3; ++ r) {
			double ya[6];
			#pragma unroll
			for(int i = 0; i < 6; i += 2) {
				double2 v = *reinterpret_cast<const double2*>(Ya + r * 6 + i);
				ya[i] = v.x; ya[i + 1] = v.y;
			}
			#pragma unroll
			for(int c = 0; c < 3; ++ c) {
				double s = 0;
				#pragma unroll
				for(int i = 0; i < 6; ++ i)
					s += ya[i] * t[c * 6 + i];
				acc[r * 3 + c] -= s; // the matrix holds minus the inverse
			}
		}
	}
	#pragma unroll
	for(int i = 0; i < 9; ++ i) {
		#pragma unroll
		for(int off = 16; off; off >>= 1)
			acc[i] += __shfl_xor_sync(0xffffffffu, acc[i], off);
	}
	if(lane == 0) {
		const double *Ci = Cinv + p * 9;
		#pragma unroll
		for(int i = 0; i < 9; ++ i)
			cov[p * 9 + i] = Ci[i] + acc[i]; // symmetric: row- and column-major agree up to rounding
	}
}

// Marginals of the system currently held as (U, V, W): d_cam_cov [36 C], d_pt_cov [9 P] on the device (either may be
// null). Returns SPP_OK / SPP_NOT_POSDEF.
int schur_marginals_current(spp_ctx *ctx, double alpha, double *d_cam_cov, double *d_pt_cov)
{
	SchurSystem &s = ctx->sys;
	const size_t n = s.C * 6, ld = dense_chol_ld(n);
	schur_form_reduced_system(ctx, alpha, alpha, false); // Cinv, Y and the dense S at this damping
	s.Sinv.resize(2 * ld * ld);
	SPP_CUDA(cudaMemcpyAsync(s.Sinv.p(), s.S.p(), ld * ld * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
	int rc = dense_chol_inverse_device(ctx, s.Sinv.p(), n);
	if(rc != SPP_OK)
		return rc;
	if(d_cam_cov && s.C) {
		k_camera_marginals<<<n_blocks(s.C * 36, 256), 256, 0, ctx->stream>>>(s.C, s.Sinv.p(), ld, d_cam_cov);
		LAUNCH_CHECK(ctx);
	}
	if(d_pt_cov && s.P) {
		const DenseMinusInverse inv = {s.Sinv.p(), ld};
		k_point_marginals<<<n_blocks(s.P, PM_WARPS), PM_WARPS * 32, 0, ctx->stream>>>(s.P, s.pt_ptr.p(), s.obs_cam.p(),
			s.Y.p(), s.Cinv.p(), inv, d_pt_cov);
		LAUNCH_CHECK(ctx);
	}
	return SPP_OK;
}

// ---- block-sparse reduced camera system ----------------------------------------------------------------------
// The same marginals without a dense S^-1: supernodal factorisation of S (supernodal_chol.cu) and selected inversion of
// the factor (selinv.cu), which leaves the entries of S^-1 on the pattern of R in the panels. Every camera pair seen by
// one landmark is a block of S, so the panels hold every block the landmark sums need.

void snode_symbolic(spp_ctx *ctx, size_t n, const std::vector<uint32_t> &blk_row, const std::vector<uint32_t> &blk_col);
void schur_fetch_host_pattern(spp_ctx *ctx);
void snode_factor(spp_ctx *ctx, const double *d_Sblk, const double *d_b);
void snode_selected_inverse(spp_ctx *ctx);

// thread per element: cov[c * 36 + i * 6 + j] = Z(6c + i, 6c + j), the diagonal block read through its upper triangle
__global__ void k_camera_marginals_panels(size_t C, const double *__restrict__ L, const uint64_t *__restrict__ diag,
	const uint32_t *__restrict__ ld, double *__restrict__ cov)
{
	size_t k = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
	if(k >= C * 36) return;
	const size_t c = k / 36;
	const unsigned e = (unsigned)(k % 36), i = e / 6, j = e % 6;
	const double *P = L + diag[c];
	cov[k] = (i <= j)? P[(size_t)j * ld[c] + i] : P[(size_t)i * ld[c] + j];
}

// Marginals of the system held as (U, V, W) through the supernodal path, d_cam_cov [36 C], d_pt_cov [9 P] (either may be
// null). Re-forms the block list of S at this damping and overwrites the panels with Z: the last solve's S is gone, so
// the residual check of that solve is refused afterwards (sparse_solved); the next solve assembles its panels anew.
// ms_phases (optional, [5]): Schur forming, factorisation, selected inversion, cameras, points. Returns SPP_OK /
// SPP_NOT_POSDEF.
int schur_marginals_sparse_current(spp_ctx *ctx, double alpha, double *d_cam_cov, double *d_pt_cov, float *ms_phases)
{
	SchurSystem &s = ctx->sys;
	SupernodalChol &sc = ctx->snode;
	cudaStream_t st = ctx->stream;
	if(!sc.valid) { // as schur_solve_current makes it (one rank)
		schur_fetch_host_pattern(ctx);
		snode_symbolic(ctx, s.C, s.h_blk_row, s.h_blk_col);
	}
	cudaEvent_t *ev = ctx->ev + 10; // phase marks
	SPP_CUDA(cudaEventRecord(ev[0], st));
	schur_form_reduced_system(ctx, alpha, alpha, true); // Cinv, Y and the block list of S at this damping
	s.sparse_solved = false;
	SPP_CUDA(cudaEventRecord(ev[1], st));
	snode_factor(ctx, s.Sblk.p(), 0);
	SPP_CUDA(cudaEventRecord(ev[2], st));
	ctx->h_scalars.resize(16);
	int *h_info = reinterpret_cast<int*>(ctx->h_scalars.p());
	SPP_CUDA(cudaMemcpyAsync(h_info, sc.d_info.p(), sizeof(int), cudaMemcpyDeviceToHost, st));
	SPP_CUDA(cudaStreamSynchronize(st));
	if(*h_info != 0)
		return SPP_NOT_POSDEF;
	SPP_CUDA(cudaEventRecord(sc.ev_factor[sc.sn.n_super() - 1], st)); // "factorisation complete" for the side lanes
	snode_selected_inverse(ctx);
	SPP_CUDA(cudaEventRecord(ev[3], st));
	if(d_cam_cov && s.C) {
		k_camera_marginals_panels<<<n_blocks(s.C * 36, 256), 256, 0, st>>>(s.C, sc.d_L.p(), sc.d_cam_diag.p(), sc.d_cam_ld.p(), d_cam_cov);
		LAUNCH_CHECK(ctx);
	}
	SPP_CUDA(cudaEventRecord(ev[4], st));
	if(d_pt_cov && s.P) {
		const PanelInverse inv = {sc.d_L.p(), sc.d_csc_ptr.p(), sc.d_asm_dst.p(), sc.d_csc_row.p(), sc.d_csc_blk.p(), sc.d_asm_ld.p()};
		k_point_marginals<<<n_blocks(s.P, PM_WARPS), PM_WARPS * 32, 0, st>>>(s.P, s.pt_ptr.p(), s.obs_cam.p(), s.Y.p(), s.Cinv.p(),
			inv, d_pt_cov);
		LAUNCH_CHECK(ctx);
	}
	SPP_CUDA(cudaEventRecord(ev[5], st));
	if(ms_phases) {
		SPP_CUDA(cudaEventSynchronize(ev[5]));
		for(int i = 0; i < 5; ++ i)
			SPP_CUDA(cudaEventElapsedTime(ms_phases + i, ev[i], ev[i + 1]));
	}
	return SPP_OK;
}

// ---- off-diagonal blocks ---------------------------------------------------------------------------------------
// With Z = S^-1 and Y = W C^-1, the camera-landmark block of observation a = (c_a, p) is
//     Sigma_{c_a p} = -sum_{b in track(p)} Z_{c_a c_b} Y_b                       (6 x 3)
// (and Sigma_pp = C_p^-1 - sum_a Y_a^T Sigma_{c_a p}, what k_point_marginals sums). Every Z_{c_a c_b} needed is a block of
// S, so both paths have it: the dense S^-1, or the panels after the selected inversion. So is Z_ij of any covisible pair.

// thread per element: out[k * 36 + c * 6 + r] = Sigma(6 a_k + r, 6 b_k + c), column-major 6 x 6. Both accessors read a
// diagonal block through its upper triangle (as k_camera_marginals / _panels do) and give (j, i) as the exact
// transpose of (i, j).
template <class Inv>
__global__ void k_cam_pair_cov(size_t n, const uint32_t *__restrict__ cam_a, const uint32_t *__restrict__ cam_b, const Inv inv,
	double *__restrict__ out)
{
	const size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
	if(i >= n * 36) return;
	const size_t k = i / 36;
	const unsigned e = (unsigned)(i % 36), c = e / 6, r = e % 6;
	out[i] = -inv.block(cam_a[k], cam_b[k])(r, c);
}

// CP_LANES lanes per requested observation, strided over the track of its landmark: each lane adds (-Z)_{c_a c_b} Y_b
// to its own 6 x 3 accumulator, a fixed xor tree sums the lanes (no atomics: reproducible). k block gathers per
// observation, sum k^2 for all of them, as in k_point_marginals. obs (n entries): edge indices mapped to track positions
// through pos; null: the n = O observations in track order.
#define CP_LANES 8
#define CP_THREADS 128
template <class Inv>
__global__ void __launch_bounds__(CP_THREADS) k_cam_point_cov(size_t n, const uint32_t *__restrict__ obs,
	const uint32_t *__restrict__ pos, const uint32_t *__restrict__ obs_pt, const uint32_t *__restrict__ pt_ptr,
	const uint32_t *__restrict__ obs_cam, const double *__restrict__ Y, const Inv inv, double *__restrict__ out)
{
	const size_t q = (blockIdx.x * (size_t)blockDim.x + threadIdx.x) / CP_LANES;
	const unsigned g = threadIdx.x % CP_LANES;
	unsigned beg = 0, k = 0, ca = 0;
	if(q < n) { // lanes past the end still take part in the shuffles
		const uint32_t t = obs? pos[obs[q]] : (uint32_t)q;
		const uint32_t p = obs_pt[t];
		beg = pt_ptr[p];
		k = pt_ptr[p + 1] - beg;
		ca = obs_cam[t];
	}
	double acc[18];
	#pragma unroll
	for(int i = 0; i < 18; ++ i) acc[i] = 0;
	for(unsigned b = g; b < k; b += CP_LANES) {
		const double *Yb = Y + (size_t)(beg + b) * 18; // column-major 6 x 3
		double yb[18];
		#pragma unroll
		for(int i = 0; i < 18; i += 2) {
			double2 t = *reinterpret_cast<const double2*>(Yb + i);
			yb[i] = t.x; yb[i + 1] = t.y;
		}
		const typename Inv::Block blk = inv.block(ca, obs_cam[beg + b]);
		#pragma unroll
		for(int j = 0; j < 6; ++ j) {
			#pragma unroll
			for(int i = 0; i < 6; ++ i) {
				const double m = blk(i, j);
				acc[i] += m * yb[j];
				acc[6 + i] += m * yb[6 + j];
				acc[12 + i] += m * yb[12 + j];
			}
		}
	}
	#pragma unroll
	for(int i = 0; i < 18; ++ i) {
		#pragma unroll
		for(int off = CP_LANES / 2; off; off >>= 1)
			acc[i] += __shfl_xor_sync(0xffffffffu, acc[i], off);
	}
	if(q < n) {
		#pragma unroll
		for(int i = 0; i < 18; ++ i)
			if(i % CP_LANES == (int)g) out[q * 18 + i] = acc[i];
	}
}

// pos[obs_orig[t]] = t: edge insertion index -> track position
__global__ void k_invert_obs_orig(size_t O, const uint32_t *__restrict__ obs_orig, uint32_t *__restrict__ pos)
{
	const size_t t = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
	if(t < O) pos[obs_orig[t]] = (uint32_t)t;
}

// slot 1, the reverse of k_slot_gather: the covariance on the block pattern of lambda into the caller's value layout.
// cam [36 C] and pt [9 P] as the marginals write them (row-major, exactly / nearly symmetric), cp [18 O] column-major
// 6 x 3 in track order; a camera-landmark block that lambda stores 3 x 6 receives the transpose.
__global__ void k_slot_cov_scatter(size_t C, size_t P, size_t O, const double *__restrict__ cam, const double *__restrict__ pt,
	const double *__restrict__ cp, const uint64_t *__restrict__ u_src, const uint64_t *__restrict__ v_src,
	const uint64_t *__restrict__ w_src, const uint8_t *__restrict__ w_tr, double *__restrict__ vals)
{
	size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
	const size_t nU = C * 36, nV = P * 9, nW = O * 18;
	if(i < nU) {
		const size_t c = i / 36, e = i % 36;
		vals[u_src[c] + e] = cam[c * 36 + (e % 6) * 6 + e / 6];
		return;
	}
	i -= nU;
	if(i < nV) {
		const size_t p = i / 9, e = i % 9;
		vals[v_src[p] + e] = pt[p * 9 + (e % 3) * 3 + e / 3];
		return;
	}
	i -= nV;
	if(i < nW) {
		const size_t o = i / 18, k = i % 18, r = k % 6, c = k / 6;
		vals[w_src[o] + (w_tr[o]? r * 3 + c : k)] = cp[i];
	}
}

// ev[0 .. 2]: marks around the pair and the observation kernels
template <class Inv>
static void launch_cov_blocks(spp_ctx *ctx, const Inv &inv, size_t n_pairs, const uint32_t *d_cam_a, const uint32_t *d_cam_b,
	double *d_pair_cov, size_t n_obs, const uint32_t *d_obs, const uint32_t *d_pos, double *d_obs_cov, cudaEvent_t *ev)
{
	SchurSystem &s = ctx->sys;
	cudaStream_t st = ctx->stream;
	SPP_CUDA(cudaEventRecord(ev[0], st));
	if(n_pairs) {
		k_cam_pair_cov<<<n_blocks(n_pairs * 36, 256), 256, 0, st>>>(n_pairs, d_cam_a, d_cam_b, inv, d_pair_cov);
		LAUNCH_CHECK(ctx);
	}
	SPP_CUDA(cudaEventRecord(ev[1], st));
	if(n_obs) {
		k_cam_point_cov<<<n_blocks(n_obs * CP_LANES, CP_THREADS), CP_THREADS, 0, st>>>(n_obs, d_obs, d_pos, s.obs_pt.p(),
			s.pt_ptr.p(), s.obs_cam.p(), s.Y.p(), inv, d_obs_cov);
		LAUNCH_CHECK(ctx);
	}
	SPP_CUDA(cudaEventRecord(ev[2], st));
}

// Selected blocks of (lambda + alpha I)^-1 of the system held as (U, V, W), on the dense path (sparse == false: S^-1 in
// full) or the supernodal one (factorisation + selected inversion, same state rules as schur_marginals_sparse_current).
// Device arrays, each may be null with its count 0: d_cam_cov [36 C] / d_pt_cov [9 P] the block diagonal, bit-identical
// to the marginals of that path; d_pair_cov [36 n_pairs] Sigma(cam_a[k], cam_b[k]), column-major, every pair in the block
// pattern of S or diagonal (the caller checks); d_obs_cov [18 n_obs] Sigma(camera, point) of observation d_obs[k] (edge
// index, mapped through obs_orig; d_obs null: every observation in track order), column-major 6 x 3.
// ms_phases (optional, [8]): the five of schur_marginals_sparse_current (zero on the dense path, which keeps no phase
// marks of its own), the pair kernel, the observation kernel, and the whole path before them (forming, inverse, block
// diagonal). Returns SPP_OK / SPP_NOT_POSDEF.
int schur_covariance_blocks_current(spp_ctx *ctx, double alpha, bool sparse, double *d_cam_cov, double *d_pt_cov, size_t n_pairs,
	const uint32_t *d_cam_a, const uint32_t *d_cam_b, double *d_pair_cov, size_t n_obs, const uint32_t *d_obs, double *d_obs_cov,
	float *ms_phases)
{
	SchurSystem &s = ctx->sys;
	cudaStream_t st = ctx->stream;
	cudaEvent_t *ev = ctx->ev + 6; // [3]: start; [0 .. 2]: launch_cov_blocks
	SPP_CUDA(cudaEventRecord(ev[3], st));
	int rc = sparse? schur_marginals_sparse_current(ctx, alpha, d_cam_cov, d_pt_cov, ms_phases) :
		schur_marginals_current(ctx, alpha, d_cam_cov, d_pt_cov);
	if(rc != SPP_OK)
		return rc;
	const uint32_t *d_pos = 0;
	if(d_obs && n_obs) {
		s.cov_pos.resize(s.O);
		k_invert_obs_orig<<<n_blocks(s.O, 256), 256, 0, st>>>(s.O, ctx->ba.d_obs_orig.p(), s.cov_pos.p());
		LAUNCH_CHECK(ctx);
		d_pos = s.cov_pos.p();
	}
	if(sparse) {
		const SupernodalChol &sc = ctx->snode;
		const PanelInverse inv = {sc.d_L.p(), sc.d_csc_ptr.p(), sc.d_asm_dst.p(), sc.d_csc_row.p(), sc.d_csc_blk.p(), sc.d_asm_ld.p()};
		launch_cov_blocks(ctx, inv, n_pairs, d_cam_a, d_cam_b, d_pair_cov, n_obs, d_obs, d_pos, d_obs_cov, ev);
	} else {
		const DenseMinusInverse inv = {s.Sinv.p(), dense_chol_ld(s.C * 6)};
		launch_cov_blocks(ctx, inv, n_pairs, d_cam_a, d_cam_b, d_pair_cov, n_obs, d_obs, d_pos, d_obs_cov, ev);
	}
	if(ms_phases) {
		SPP_CUDA(cudaEventSynchronize(ev[2]));
		SPP_CUDA(cudaEventElapsedTime(ms_phases + 5, ev[0], ev[1]));
		SPP_CUDA(cudaEventElapsedTime(ms_phases + 6, ev[1], ev[2]));
		SPP_CUDA(cudaEventElapsedTime(ms_phases + 7, ev[3], ev[0]));
	}
	return SPP_OK;
}

// slot 1: the covariance on the block pattern of the caller's lambda, into d_vals [n_values] in its value layout;
// ms_phases as schur_covariance_blocks_current
int slot_covariance_pattern(spp_ctx *ctx, double alpha, bool sparse, double *d_vals, float *ms_phases)
{
	SchurSystem &s = ctx->sys;
	SchurSlot &sl = ctx->slot;
	s.cov_cam.resize(s.C * 36);
	s.cov_pt.resize(s.P * 9);
	s.cov_obs.resize(s.O * 18);
	int rc = schur_covariance_blocks_current(ctx, alpha, sparse, s.cov_cam.p(), s.cov_pt.p(), 0, 0, 0, 0, s.O, 0, s.cov_obs.p(),
		ms_phases);
	if(rc != SPP_OK)
		return rc;
	const size_t total = s.C * 36 + s.P * 9 + s.O * 18;
	k_slot_cov_scatter<<<n_blocks(total, 256), 256, 0, ctx->stream>>>(s.C, s.P, s.O, s.cov_cam.p(), s.cov_pt.p(), s.cov_obs.p(),
		sl.u_src.p(), sl.v_src.p(), sl.w_src.p(), sl.w_transposed.p(), d_vals);
	LAUNCH_CHECK(ctx);
	return SPP_OK;
}

// ---- pose graphs -------------------------------------------------------------------------------------------------
// Reference replaced: the marginals step of CNonlinearSolver_Lambda::Optimize() (NonlinearSolver_Lambda.h:669-767 ->
// CMarginals::Calculate_DenseMarginals_Recurrent_FBS on the Cholesky factor of lambda, policy mpart_Diagonal). The pose
// systems of the configurations in scope have at most a few thousand block columns: lambda is scattered into the
// dense solver's storage and inverted there.

__global__ void k_pose_blocks_to_dense(size_t n_vals, int dim, const double *__restrict__ vals,
	const uint32_t *__restrict__ blk_row, const uint32_t *__restrict__ blk_col, size_t ld, double *__restrict__ A)
{
	size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
	if(i >= n_vals) return;
	const size_t b = i / (dim * dim);
	const unsigned e = (unsigned)(i - b * (dim * dim)), r = blk_row[b] * dim + e % dim, c = blk_col[b] * dim + e / dim; // column-major blocks
	if(r <= c)
		A[(size_t)c * ld + r] = vals[i];
}

__global__ void k_pose_marginals(size_t N, int dim, const double *__restrict__ Ni, size_t ld, double *__restrict__ cov)
{
	size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
	if(i >= N * dim * dim) return;
	const unsigned v = (unsigned)(i / (dim * dim)), e = (unsigned)(i % (dim * dim));
	cov[i] = -minus_inv_at(Ni, ld, v * dim + e / dim, v * dim + e % dim);
}

// d_cov [N dim^2] on the device; lambda must be current (pose_linearise). Returns SPP_OK / SPP_NOT_POSDEF.
int pose_marginals(spp_ctx *ctx, double *d_cov)
{
	PoseProblem &pp = ctx->pose;
	const size_t n = pp.N * pp.dim, ld = dense_chol_ld(n);
	std::vector<uint32_t> h_row(pp.n_blocks), h_col(pp.n_blocks);
	for(size_t c = 0; c < pp.N; ++ c) {
		for(uint64_t k = pp.h_col_ptr[c]; k < pp.h_col_ptr[c + 1]; ++ k) {
			h_row[k] = (uint32_t)pp.h_row_idx[k];
			h_col[k] = (uint32_t)c;
		}
	}
	DBuf<uint32_t> d_row, d_col;
	d_row.upload(h_row, ctx->stream);
	d_col.upload(h_col, ctx->stream);
	DBuf<double> &A = ctx->sys.Sinv;
	A.resize(2 * ld * ld);
	SPP_CUDA(cudaMemsetAsync(A.p(), 0, ld * ld * sizeof(double), ctx->stream));
	const size_t n_vals = pp.n_blocks * pp.dim * pp.dim;
	k_pose_blocks_to_dense<<<n_blocks(n_vals, 256), 256, 0, ctx->stream>>>(n_vals, pp.dim, pp.vals.p(), d_row.p(), d_col.p(), ld, A.p());
	LAUNCH_CHECK(ctx);
	int rc = dense_chol_inverse_device(ctx, A.p(), n); // synchronises: the index arrays may go
	if(rc != SPP_OK)
		return rc;
	k_pose_marginals<<<n_blocks(pp.N * pp.dim * pp.dim, 256), 256, 0, ctx->stream>>>(pp.N, pp.dim, A.p(), ld, d_cov);
	LAUNCH_CHECK(ctx);
	return SPP_OK;
}

} // namespace spp

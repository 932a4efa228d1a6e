// dense_chol.cu -- stage 3 of the hot path for a dense reduced camera system: FP64 Cholesky S = R^T R of
// the upper triangle, and the two triangular solves.
//
// Reference function replaced (SURVEY 8(a) row a14): CLinearSolver_DenseEigen::Solve_PosDef
// (src/slam/LinearSolver_Schur.cpp:2314-2333) = Convert_to_Dense + Eigen::LLT<MatrixXd, Eigen::Upper>::compute
// (reads the upper triangle only, fails on a non-positive pivot) + LLT::solve (two triangular solves).
//
// Layout: column-major, leading dimension ld = n rounded up to a multiple of the panel width (128); the
// padding carries an identity diagonal so that no kernel needs bounds checks. The right-hand side rides along
// as an extra column block right of the matrix: the panel solve and the trailing update turn it into
// y = R^-T b for free (augmented-matrix trick), which leaves one backward solve R x = y.
//
// Blocked right-looking factorisation, panel width 128, one-step look-ahead on two streams:
//   k_potrf128      one CTA: 128x128 diagonal block in shared memory, 32-wide sub-blocks (register Cholesky in
//                   one warp, sub-row solve, rank-32 update), then the inverse of the triangular factor
//   k_gemm_tn<TRSM> block row right of the diagonal: P <- Rinv_kk^T P        (FP64 tensor cores)
//   k_gemm_tn<SYRK> trailing update C -= P^T P, upper tiles only             (FP64 tensor cores)
//                   critical stream: the tile row that the next panel needs (64x64 tiles, look-ahead)
//                   bulk stream    : everything below it (128x64 tiles)
// The GEMM kernel stages K-contiguous operand tiles with a 3-deep cp.async pipeline and issues
// mma.sync.m8n8k4.f64 (DMMA); tcgen05 has no FP64 kind, so this is the tensor path for FP64 on sm_100a.
// Backward solve: one persistent CTA per block row consumes x_j as soon as block row j publishes it and
// finishes with the inverse diagonal block computed by k_potrf128.

#include "spp_ctx.h"
#include <cuda_pipeline_primitives.h>
#include <stdlib.h>
#include <algorithm>

namespace spp {

#define LAUNCH_CHECK(ctx) do { ++ (ctx)->n_launches; SPP_CUDA(cudaGetLastError()); } while(0)

#define CH_NB 128          // panel width = K of every GEMM
#define CH_BK 16           // k-chunk staged in shared memory
#define CH_LDS (CH_BK + 4) // padded row length: conflict-free DMMA fragment loads
#define CH_STAGES 3

#include "potrf128.cuh"
#include "chol_dataflow.cuh"

static const size_t POTRF_SMEM_EXCLUSIVE = 227 * 1024; // the opt-in maximum per CTA: nothing else fits on the SM

// ---- FP64 tensor-core GEMM: C (op)= A^T B with K = 128, operands K-contiguous ---------------------------

enum { GEMM_SYRK = 0, GEMM_TRSM = 1, GEMM_GRAM = 2 };

// SYRK: C(i0.., j0..) -= P(:, i0..)^T P(:, j0..), P = rows k0..k0+127 of A; tiles with i0 > j0 are skipped.
//       grid.x = column tile (from column cbase), grid.y = row tile (from row rbase).
// TRSM: P(:, j0..) <- Rinv^T P(:, j0..) in place; BM must be 128 (a CTA owns whole columns of the panel).
// GRAM: SYRK with the operand rows taken from another matrix Z of the same leading dimension (passed in the Rinv
//       slot): C(i0.., j0..) -= Z(k0.., i0..)^T Z(k0.., j0..) -- the inverse of a factored matrix as Z^T Z, Z = R^-T.
// WM x WN is the warp tile (multiples of 8): 32 x 32 for the bulk updates, smaller for the few tiles on the critical
// chain, where more warps with shorter DMMA chains finish sooner.
template <int MODE, int BM, int BN, int WM = 32, int WN = 32, int STAGES = CH_STAGES>
__global__ void __launch_bounds__((BM / WM) * (BN / WN) * 32) k_gemm_tn(double *__restrict__ A, size_t ld, size_t k0,
	size_t rbase, size_t cbase, const double *__restrict__ Rinv)
{
	constexpr int WARPS_N = BN / WN, NT = (BM / WM) * (BN / WN) * 32, MA = WM / 8, NB = WN / 8;
	constexpr bool SYRK_LIKE = MODE != GEMM_TRSM;
	size_t i0, j0;
	if(SYRK_LIKE) {
		i0 = rbase + blockIdx.y * (size_t)BM;
		j0 = cbase + blockIdx.x * (size_t)BN;
		if(i0 > j0 + (BN - 1))
			return; // strictly below the diagonal
	} else {
		i0 = 0;
		j0 = cbase + blockIdx.x * (size_t)BN;
	}
	extern __shared__ double smem[];
	double (*As)[BM][CH_LDS] = reinterpret_cast<double (*)[BM][CH_LDS]>(smem);
	double (*Bs)[BN][CH_LDS] = reinterpret_cast<double (*)[BN][CH_LDS]>(smem + STAGES * BM * CH_LDS);
	const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
	const int wi = (warp / WARPS_N) * WM, wj = (warp % WARPS_N) * WN;
	const int g = lane >> 2, t = lane & 3;

	// operand pointers: element (k, m) at base[m * stride + k]
	const double *pa; size_t sa;
	if(MODE == GEMM_SYRK) { pa = A + i0 * ld + k0; sa = ld; }
	else if(MODE == GEMM_GRAM) { pa = Rinv + i0 * ld + k0; sa = ld; }
	else { pa = Rinv; sa = CH_NB; }
	const double *pb = ((MODE == GEMM_GRAM)? Rinv : A) + j0 * ld + k0;

	auto stage_load = [&](int st, int kc) {
		// BM (BN) rows x 8 chunks of 16 bytes
		for(int idx = tid; idx < BM * 8; idx += NT) {
			const int m = idx >> 3, q = idx & 7;
			__pipeline_memcpy_async(&As[st][m][q * 2], pa + (size_t)m * sa + kc * CH_BK + q * 2, 16);
		}
		for(int idx = tid; idx < BN * 8; idx += NT) {
			const int m = idx >> 3, q = idx & 7;
			__pipeline_memcpy_async(&Bs[st][m][q * 2], pb + (size_t)m * ld + kc * CH_BK + q * 2, 16);
		}
	};

	double acc[MA][NB][2];

	constexpr int KT = CH_NB / CH_BK;
	#pragma unroll
	for(int s = 0; s < STAGES - 1; ++ s) {
		stage_load(s, s);
		__pipeline_commit();
	}
	// SYRK: the accumulators start from the C tile (its loads overlap the pipeline fill) and the A fragments
	// are negated, so the epilogue is a plain store instead of a read-modify-write
	#pragma unroll
	for(int a = 0; a < MA; ++ a) {
		#pragma unroll
		for(int b = 0; b < NB; ++ b) {
			if(SYRK_LIKE) {
				const size_t c = j0 + wj + b * 8 + 2 * t, r = i0 + wi + a * 8 + g;
				acc[a][b][0] = A[c * ld + r];
				acc[a][b][1] = A[(c + 1) * ld + r];
			} else
				acc[a][b][0] = acc[a][b][1] = 0;
		}
	}
	for(int kt = 0; kt < KT; ++ kt) {
		__pipeline_wait_prior(STAGES - 2);
		__syncthreads();
		if(kt + STAGES - 1 < KT)
			stage_load((kt + STAGES - 1) % STAGES, kt + STAGES - 1);
		__pipeline_commit();
		const int st = kt % STAGES;
		#pragma unroll
		for(int k4 = 0; k4 < CH_BK; k4 += 4) {
			double fa[MA], fb[NB];
			#pragma unroll
			for(int a = 0; a < MA; ++ a)
				fa[a] = SYRK_LIKE? -As[st][wi + a * 8 + g][k4 + t] : As[st][wi + a * 8 + g][k4 + t];
			#pragma unroll
			for(int b = 0; b < NB; ++ b)
				fb[b] = Bs[st][wj + b * 8 + g][k4 + t];
			#pragma unroll
			for(int a = 0; a < MA; ++ a)
				#pragma unroll
				for(int b = 0; b < NB; ++ b)
					dmma_m8n8k4(acc[a][b][0], acc[a][b][1], fa[a], fb[b]);
		}
	}
	__pipeline_wait_prior(0);
	if(MODE == GEMM_TRSM)
		__syncthreads(); // every warp is done reading the panel (through smem) before anyone overwrites it
	#pragma unroll
	for(int a = 0; a < MA; ++ a) {
		#pragma unroll
		for(int b = 0; b < NB; ++ b) {
			const size_t c = j0 + wj + b * 8 + 2 * t;
			if(SYRK_LIKE) {
				const size_t r = i0 + wi + a * 8 + g;
				A[c * ld + r] = acc[a][b][0];
				A[(c + 1) * ld + r] = acc[a][b][1];
			} else {
				const size_t r = k0 + wi + a * 8 + g;
				A[c * ld + r] = acc[a][b][0];
				A[(c + 1) * ld + r] = acc[a][b][1];
			}
		}
	}
}

template <int BM, int BN, int STAGES = CH_STAGES>
constexpr size_t gemm_smem() { return (size_t)STAGES * (BM + BN) * CH_LDS * sizeof(double); }

// ---- backward solve R x = y ---------------------------------------------------------------------------

// One CTA per block row (blockIdx 0 = last block row), 256 threads: thread (r, h) owns row r, column half h. The chain
// x_j -> block row j - 1 -> x_{j-1} is all latency: the CTA's own inverse diagonal block waits in shared memory, the
// matrix entries of the next step are fetched before the flag is polled, and one thread publishes (release) after
// the CTA barrier.
__global__ void __launch_bounds__(256) k_backsolve(const double *__restrict__ A, size_t ld, size_t n_blk,
	const double *__restrict__ Rinv, double *y /* in: y, out: x */, int *flags)
{
	extern __shared__ __align__(16) double ri_s[]; // Rinv_ii, column-major 128 x 128
	__shared__ double xs[2][CH_NB];
	__shared__ double part[2][CH_NB];
	const size_t bi = n_blk - 1 - blockIdx.x;
	const int r = threadIdx.x & 127, h = threadIdx.x >> 7;
	{
		const double *Ri = Rinv + bi * (size_t)(CH_NB * CH_NB);
		for(int idx = threadIdx.x; idx < CH_NB * CH_NB / 2; idx += 256)
			__pipeline_memcpy_async(ri_s + 2 * idx, Ri + 2 * idx, 16);
		__pipeline_commit();
	}
	double acc = (h == 0)? y[bi * CH_NB + r] : 0.0;
	int p = 0;
	for(size_t bj = n_blk - 1; bj > bi; -- bj, p ^= 1) {
		// the 64 matrix entries of this thread do not depend on x_j: fetch them before waiting
		const double *row = A + (bj * CH_NB + h * 64) * ld + bi * CH_NB + r;
		double m[64];
		#pragma unroll
		for(int c = 0; c < 64; ++ c)
			m[c] = __ldg(row + (size_t)c * ld);
		if(threadIdx.x == 0) {
			while(df::ld_acquire(flags + bj) == 0)
				;
		}
		__syncthreads();
		if(threadIdx.x < CH_NB)
			xs[p][threadIdx.x] = __ldcg(y + bj * CH_NB + threadIdx.x);
		__syncthreads();
		double s0 = 0, s1 = 0, s2 = 0, s3 = 0;
		#pragma unroll
		for(int c = 0; c < 64; c += 4) {
			s0 += m[c] * xs[p][h * 64 + c];
			s1 += m[c + 1] * xs[p][h * 64 + c + 1];
			s2 += m[c + 2] * xs[p][h * 64 + c + 2];
			s3 += m[c + 3] * xs[p][h * 64 + c + 3];
		}
		acc -= (s0 + s1) + (s2 + s3);
	}
	__pipeline_wait_prior(0);
	part[h][r] = acc;
	__syncthreads();
	if(threadIdx.x < CH_NB)
		xs[p][threadIdx.x] = part[0][threadIdx.x] + part[1][threadIdx.x];
	__syncthreads();
	// x_i = Rinv_ii (upper triangular, zeros stored below the diagonal) * acc
	double s0 = 0, s1 = 0, s2 = 0, s3 = 0;
	#pragma unroll 4
	for(int c = h * 64; c < h * 64 + 64; c += 4) {
		s0 += ri_s[c * CH_NB + r] * xs[p][c];
		s1 += ri_s[(c + 1) * CH_NB + r] * xs[p][c + 1];
		s2 += ri_s[(c + 2) * CH_NB + r] * xs[p][c + 2];
		s3 += ri_s[(c + 3) * CH_NB + r] * xs[p][c + 3];
	}
	__syncthreads();
	part[h][r] = (s0 + s1) + (s2 + s3);
	__syncthreads();
	if(threadIdx.x < CH_NB)
		y[bi * CH_NB + threadIdx.x] = part[0][threadIdx.x] + part[1][threadIdx.x];
	__syncthreads();
	if(threadIdx.x == 0)
		df::st_release(flags + bi, 1);
}

static const size_t BACKSOLVE_SMEM = (size_t)CH_NB * CH_NB * sizeof(double);

__global__ void k_pad_identity(double *__restrict__ A, size_t ld, size_t n, size_t n_pad)
{
	size_t i = n + blockIdx.x * (size_t)blockDim.x + threadIdx.x;
	if(i < n_pad)
		A[i * ld + i] = 1.0;
}

__global__ void k_copy_rhs(double *__restrict__ dst, const double *__restrict__ src, size_t n)
{
	size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
	if(i < n)
		dst[i] = src[i];
}

// ---------------------------------------------------------------------------------------------------

size_t dense_chol_ld(size_t n)
{
	return (n + CH_NB - 1) / CH_NB * CH_NB;
}

// number of doubles of the augmented storage: ld x (ld + 128)
size_t dense_chol_storage(size_t n)
{
	size_t ld = dense_chol_ld(n);
	return ld * (ld + CH_NB);
}

static void chol_init_attributes(int device)
{
	static bool done[64] = {false}; // the attribute belongs to the (kernel, device) pair
	if(device < 0 || device >= 64 || done[device]) return;
	SPP_CUDA(cudaFuncSetAttribute(k_potrf128, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)POTRF_SMEM_EXCLUSIVE));
	SPP_CUDA(cudaFuncSetAttribute(k_backsolve, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)BACKSOLVE_SMEM));
	SPP_CUDA(cudaFuncSetAttribute(k_gemm_tn<GEMM_SYRK, 128, 64>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)gemm_smem<128, 64>()));
	SPP_CUDA(cudaFuncSetAttribute(k_gemm_tn<GEMM_SYRK, 64, 64>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)gemm_smem<64, 64>()));
	SPP_CUDA(cudaFuncSetAttribute(k_gemm_tn<GEMM_TRSM, 128, 64>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)gemm_smem<128, 64>()));
	SPP_CUDA(cudaFuncSetAttribute(k_gemm_tn<GEMM_GRAM, 128, 64>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)gemm_smem<128, 64>()));
	SPP_CUDA(cudaFuncSetAttribute(k_gemm_tn<GEMM_GRAM, 64, 64>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)gemm_smem<64, 64>()));
	SPP_CUDA(cudaFuncSetAttribute((k_gemm_tn<GEMM_TRSM, 128, 16, 32, 16, 8>), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)gemm_smem<128, 16, 8>()));
	SPP_CUDA(cudaFuncSetAttribute((k_gemm_tn<GEMM_SYRK, 32, 32, 16, 16, 8>), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)gemm_smem<32, 32, 8>()));
	done[device] = true;
}

static void chol_init_streams(spp_ctx *ctx)
{
	DenseChol &ch = ctx->chol;
	chol_init_attributes(ctx->device);
	if(ch.bulk_stream)
		return;
	// the context stream carries the critical chain (created with the highest priority in spp_create); the
	// look-ahead row is next, the bulk updates yield to both whenever an SM frees up
	int prio_lo = 0, prio_hi = 0;
	SPP_CUDA(cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
	SPP_CUDA(cudaStreamCreateWithPriority(&ch.bulk_stream, cudaStreamNonBlocking, prio_lo));
	SPP_CUDA(cudaStreamCreateWithPriority(&ch.row_stream, cudaStreamNonBlocking, (prio_hi + 1 <= prio_lo)? prio_hi + 1 : prio_hi));
	for(int i = 0; i < 2; ++ i) {
		SPP_CUDA(cudaEventCreateWithFlags(&ch.ev_potrf[i], cudaEventDisableTiming));
		SPP_CUDA(cudaEventCreateWithFlags(&ch.ev_first[i], cudaEventDisableTiming));
		SPP_CUDA(cudaEventCreateWithFlags(&ch.ev_panel[i], cudaEventDisableTiming));
		SPP_CUDA(cudaEventCreateWithFlags(&ch.ev_bulk[i], cudaEventDisableTiming));
		SPP_CUDA(cudaEventCreateWithFlags(&ch.ev_row[i], cudaEventDisableTiming));
	}
}

// Partial right-looking factorisation of a block ROW panel: A is column-major with ld rows (a multiple of 128) and
// n_cols >= ld + 128 columns (a multiple of 128). The leading ld x ld upper triangle is factored (R11), the columns
// right of it receive R11^-T A12 (block row of the factor / forward-solved right-hand sides). A dense matrix with its
// right-hand side block is the case n_cols = ld + 128; a supernode of the block-sparse factorisation
// (supernodal_chol.cu) is the case "ld = its own columns, n_cols - ld = its row structure + right-hand side".
// Rinv receives the inverses of the ld / 128 diagonal blocks of R11; *info the first non-positive pivot (1-based).
// Asynchronous: everything is ordered on (or joined back into) the context's stream.
// identity_tail: the columns right of R11 start as the identity (the inverse, dense_chol_inverse_device): block row b of
// them is zero right of column block b until panel b has been applied, so panel b only touches the first b + 1 of them.
void dense_chol_factor_panel(spp_ctx *ctx, double *A, size_t ld, size_t n_cols_all, double *Rinv, int *info, bool identity_tail)
{
	DenseChol &ch = ctx->chol;
	chol_init_streams(ctx);
	const size_t n_blk = ld / CH_NB;
	// factorisation with one-step look-ahead on three streams:
	//   sA (critical): potrf(b) -> trsm(b) -> update of the next diagonal tile -> potrf(b+1) ...
	//   sC           : update of the rest of the next panel's tile row (needed by trsm(b+1) only)
	//   sB (bulk)    : update of everything below that row, overlapping potrf/trsm of the next panel
	cudaStream_t sA = ctx->stream, sB = ch.bulk_stream, sC = ch.row_stream;
	// C(rows r0.., cols c0..) -= P^T P on the upper tiles of a (n_r x n_c) region, in 128 x 64 or 64 x 64 tiles
	auto syrk = [&](cudaStream_t s, size_t k0, size_t r0, size_t c0, size_t n_r, size_t n_c, bool tile128) {
		if(tile128) {
			dim3 grid((unsigned)(n_c / 64), (unsigned)(n_r / 128));
			k_gemm_tn<GEMM_SYRK, 128, 64><<<grid, 256, gemm_smem<128, 64>(), s>>>(A, ld, k0, r0, c0, 0);
		} else {
			dim3 grid((unsigned)(n_c / 64), (unsigned)(n_r / 64));
			k_gemm_tn<GEMM_SYRK, 64, 64><<<grid, 128, gemm_smem<64, 64>(), s>>>(A, ld, k0, r0, c0, 0);
		}
		LAUNCH_CHECK(ctx);
	};
	// Measured and rejected: bulk updates in pairs -- the bulk update of an even panel deferred and applied together with
	// the next panel's as one rank-256 pass (half the launches, half the read-modify-write traffic of the trailing matrix,
	// twice the K per tile). Bit-identical results, but slower on the Venice system (5226^2: 3.55 ms against 3.39 ms per
	// factorisation): the deferred update starts one panel later, so less of it hides behind the critical chain, and the
	// rank-256 look-ahead of the diagonal tile sits on that chain.
	bool bulk_in_flight = false, row_in_flight = false;
	int bulk_slot = 0; // the event the last bulk update was recorded in
	for(size_t b = 0; b < n_blk; ++ b) {
		const size_t k0 = b * CH_NB, c0 = k0 + CH_NB;
		const size_t n_cols = identity_tail? ld + (b + 1) * CH_NB : n_cols_all;
		const int e = int(b & 1);
		double *Rinv_b = Rinv + b * (size_t)(CH_NB * CH_NB);
		// the diagonal block asks for a whole SM's shared memory: co-resident update CTAs would compete for the FP64
		// pipe and stretch the critical chain (measured: 33 -> 45 us)
		k_potrf128<<<1, PT, POTRF_SMEM_EXCLUSIVE, sA>>>(A, ld, k0, Rinv_b, info, 0);
		LAUNCH_CHECK(ctx);
		SPP_CUDA(cudaEventRecord(ch.ev_potrf[e], sA));
		if(row_in_flight) { // tile row b was last updated by the look-ahead of panel b - 1 on sC
			SPP_CUDA(cudaStreamWaitEvent(sA, ch.ev_row[e ^ 1], 0));
			row_in_flight = false;
		}
		// panel solve, critical part: the tile right of the diagonal (the rhs block for the last panel)
		k_gemm_tn<GEMM_TRSM, 128, 16, 32, 16, 8><<<CH_NB / 16, 128, gemm_smem<128, 16, 8>(), sA>>>(A, ld, k0, 0, c0, Rinv_b);
		LAUNCH_CHECK(ctx);
		if(c0 >= ld) { // last diagonal block: what is left of its block row (more than the first tile only for a panel)
			if(n_cols > c0 + CH_NB) {
				k_gemm_tn<GEMM_TRSM, 128, 64><<<(unsigned)((n_cols - c0 - CH_NB) / 64), 256, gemm_smem<128, 64>(), sA>>>(A, ld, k0, 0,
					c0 + CH_NB, Rinv_b);
				LAUNCH_CHECK(ctx);
			}
			break;
		}
		SPP_CUDA(cudaEventRecord(ch.ev_first[e], sA));
		SPP_CUDA(cudaStreamWaitEvent(sC, ch.ev_potrf[e], 0));
		// panel solve, the rest of the block row (sC; its input was written by sC itself)
		k_gemm_tn<GEMM_TRSM, 128, 64><<<(unsigned)((n_cols - c0 - CH_NB) / 64), 256, gemm_smem<128, 64>(), sC>>>(A, ld, k0, 0,
			c0 + CH_NB, Rinv_b);
		LAUNCH_CHECK(ctx);
		SPP_CUDA(cudaEventRecord(ch.ev_panel[e], sC)); // panel b is final (together with ev_first)
		// the look-ahead updates write tile row b + 1, which the bulk update of step b - 1 also wrote
		if(bulk_in_flight) {
			SPP_CUDA(cudaStreamWaitEvent(sA, ch.ev_bulk[bulk_slot], 0));
			SPP_CUDA(cudaStreamWaitEvent(sC, ch.ev_bulk[bulk_slot], 0));
			bulk_in_flight = false;
		}
		// look-ahead, critical part: the next diagonal tile (32 x 32 tiles of four 16 x 16 warps: short chains)
		k_gemm_tn<GEMM_SYRK, 32, 32, 16, 16, 8><<<dim3(CH_NB / 32, CH_NB / 32), 128, gemm_smem<32, 32, 8>(), sA>>>(A, ld, k0, c0, c0, 0);
		LAUNCH_CHECK(ctx);
		// look-ahead, rest of the next panel's tile row (rhs block included)
		SPP_CUDA(cudaStreamWaitEvent(sC, ch.ev_first[e], 0));
		// 64 x 64 tiles while they are needed to occupy the SMs (a dense matrix), 128 x 64 for the long block rows of a
		// supernode panel
		syrk(sC, k0, c0, c0 + CH_NB, CH_NB, n_cols - (c0 + CH_NB), (n_cols - (c0 + CH_NB)) / 64 >= 148);
		SPP_CUDA(cudaEventRecord(ch.ev_row[e], sC));
		row_in_flight = true;
		const size_t r1 = c0 + CH_NB; // first row below the next panel's tile row
		if(r1 < ld) {
			SPP_CUDA(cudaStreamWaitEvent(sB, ch.ev_panel[e], 0));
			SPP_CUDA(cudaStreamWaitEvent(sB, ch.ev_first[e], 0));
			const size_t T = (ld - r1) / 128, n_tiles = T * (T + 1) / 2 + T;
			// 128 x 64 tiles (two CTAs per SM overlap each other's pipeline fill and epilogue: 5 % faster than 128 x 128
			// even on the largest trailing matrices), 64 x 64 when few tiles are left
			syrk(sB, k0, r1, r1, ld - r1, n_cols - r1, n_tiles >= 74);
			SPP_CUDA(cudaEventRecord(ch.ev_bulk[e], sB));
			bulk_in_flight = true;
			bulk_slot = e;
		}
	}
	for(int i = 0; i < 2; ++ i) { // join: whatever is still in flight on the side streams
		if(bulk_in_flight)
			SPP_CUDA(cudaStreamWaitEvent(sA, ch.ev_bulk[i], 0));
		if(row_in_flight)
			SPP_CUDA(cudaStreamWaitEvent(sA, ch.ev_row[i], 0));
	}
}

// ---- persistent dataflow factorisation (chol_dataflow.cuh): host side -----------------------------------

typedef CUresult (*spp_encode_tiled_fn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
	const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// TMA descriptor of a column-major FP64 matrix (n_rows contiguous, n_cols columns ld apart), boxes of box_rows x box_cols,
// 128-byte swizzle (box_rows = 16 doubles = one 128-byte line per column of the box)
static void make_tensor_map(CUtensorMap *map, const void *base, size_t n_rows, size_t n_cols, size_t ld, unsigned box_rows, unsigned box_cols)
{
	static spp_encode_tiled_fn encode = 0;
	if(!encode) {
		void *fn = 0;
		cudaDriverEntryPointQueryResult q;
		SPP_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q));
		if(q != cudaDriverEntryPointSuccess || !fn)
			throw cuda_error("cuTensorMapEncodeTiled is not available from this driver");
		encode = (spp_encode_tiled_fn)fn;
	}
	const cuuint64_t dims[2] = {(cuuint64_t)n_rows, (cuuint64_t)n_cols}, strides[1] = {(cuuint64_t)(ld * sizeof(double))};
	const cuuint32_t box[2] = {box_rows, box_cols}, elem[2] = {1, 1};
	CUresult r = encode(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, const_cast<void*>(base), dims, strides, box, elem, CU_TENSOR_MAP_INTERLEAVE_NONE,
		CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
	if(r != CUDA_SUCCESS) {
		char b[128];
		snprintf(b, sizeof(b), "cuTensorMapEncodeTiled failed (CUresult %d)", (int)r);
		throw cuda_error(b);
	}
}

bool dense_chol_dataflow_enabled()
{
	const char *e = getenv("SPP_CHOL_DATAFLOW"); // read at every call: tools / tests switch between the two paths in one process
	return !e || atoi(e) != 0;
}

// Factorisation of the leading ld x ld upper triangle of A (column-major, ld a multiple of 128) and forward solve of the
// n_cols - ld columns right of it (a multiple of 64), as dense_chol_factor_panel() without the identity tail, by the
// persistent dataflow kernel. Rinv / info as there; info = -1 reports the kernel's watchdog. Asynchronous on the
// context's stream.
void dense_chol_factor_dataflow(spp_ctx *ctx, double *A, size_t ld, size_t n_cols, double *Rinv, int *info)
{
	DenseChol &ch = ctx->chol;
	const size_t NB = ld / CH_NB, NJH = n_cols / 64;
	if(ld % CH_NB || n_cols % 64 || n_cols < ld || NB >= 0x8000 || NJH >= 0x10000)
		throw invalid_error("dense_chol_factor_dataflow: bad panel shape");
	cudaStream_t st = ctx->stream;
	if(!ch.n_sms) {
		SPP_CUDA(cudaDeviceGetAttribute(&ch.n_sms, cudaDevAttrMultiProcessorCount, ctx->device));
		SPP_CUDA(cudaFuncSetAttribute(k_chol_dataflow, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)df::SMEM_BYTES));
	}
	DenseChol::DfTaskList &tl = ch.df_tasks[((uint64_t)NB << 32) | NJH];
	if(!tl.n_tasks) {
		// Worker tasks in row-major order (row i, tile column j). The partial sums of the four half tiles on the chain itself
		// (the diagonal tile and the tile right of it) are queued one row early: a worker that takes them follows the
		// factorisation slab by slab and is one slab away from done when the chain gets there (their operands come later in
		// the queue: fine as long as there are more workers than the 8 open chain tasks; a starved launch ends in the
		// watchdog, not in a hang). Measured and rejected (profiles/r2d_*, r2e_*): queueing them 0, 2, 3, 4 or 6 rows early, and
		// skewing the row-major order to push the tiles far from the diagonal back behind the near-diagonal tiles of the
		// following rows.
		std::vector<std::pair<double, uint32_t> > keyed;
		for(size_t i = 0; i < NB; ++ i) {
			for(size_t jh = 2 * i; jh < NJH; ++ jh) {
				const size_t j = jh / 2;
				const bool chain = j == i || (j == i + 1 && j < NB);
				const double key = chain? (double)i - 1.5 : (double)i;
				keyed.push_back(std::make_pair(key, (uint32_t)((i << 16) | jh)));
			}
		}
		std::stable_sort(keyed.begin(), keyed.end(), [](const std::pair<double, uint32_t> &a, const std::pair<double, uint32_t> &b) { return a.first < b.first; });
		std::vector<uint32_t> tasks;
		for(size_t q = 0; q < keyed.size(); ++ q)
			tasks.push_back(keyed[q].second);
		tl.codes.upload(tasks, st);
		SPP_CUDA(cudaStreamSynchronize(st)); // the host vector goes out of scope
		tl.n_tasks = tasks.size();
	}
	if(ch.df_A != A || ch.df_ld != ld || ch.df_cols != n_cols || ch.df_Rinv != Rinv) {
		make_tensor_map(&ch.df_maps[0], A, ld, n_cols, ld, 16, 128);
		make_tensor_map(&ch.df_maps[1], A, ld, n_cols, ld, 16, 64);
		make_tensor_map(&ch.df_maps[2], A, ld, n_cols, ld, 16, 16);
		make_tensor_map(&ch.df_maps[3], Rinv, CH_NB, NB * CH_NB, CH_NB, 16, 128);
		make_tensor_map(&ch.df_maps[4], Rinv, CH_NB, NB * CH_NB, CH_NB, 16, 16);
		ch.df_A = A; ch.df_ld = ld; ch.df_cols = n_cols; ch.df_Rinv = Rinv;
	}
	const size_t n_flags = 4 + 4 * NB + 2 * NB * NJH;
	ch.df_flags.resize(n_flags);
	SPP_CUDA(cudaMemsetAsync(ch.df_flags.p(), 0, n_flags * sizeof(int), st));
	df::Args args;
	args.A = A; args.Rinv = Rinv; args.info = info; args.flags = ch.df_flags.p(); args.tasks = tl.codes.p();
	args.ld = ld; args.NB = (int)NB; args.NJH = (int)NJH; args.n_tasks = (int)tl.n_tasks;
	const size_t n_ctas = std::min((size_t)ch.n_sms, 1 + df::G + tl.n_tasks);
	static const bool timing = getenv("SPP_CHOL_TIMING") != 0;
	DBuf<unsigned long long> dbg;
	args.dbg = 0;
	if(timing) {
		dbg.resize(5 * NB + 8 * n_ctas);
		dbg.zero(st);
		args.dbg = dbg.p();
		SPP_CUDA(cudaEventRecord(ctx->ev[4], st));
	}
	if(ctx->async_mode) { // the LM loop reads this pair after its one synchronisation (ms_factor_kernel)
		if(!ctx->phase_ev[PH_CHOL_KERNEL][0]) {
			SPP_CUDA(cudaEventCreate(&ctx->phase_ev[PH_CHOL_KERNEL][0]));
			SPP_CUDA(cudaEventCreate(&ctx->phase_ev[PH_CHOL_KERNEL][1]));
		}
		SPP_CUDA(cudaEventRecord(ctx->phase_ev[PH_CHOL_KERNEL][0], st));
	}
	k_chol_dataflow<<<(unsigned)n_ctas, df::THREADS, df::SMEM_BYTES, st>>>(ch.df_maps[0], ch.df_maps[1], ch.df_maps[2], ch.df_maps[3], ch.df_maps[4], args);
	LAUNCH_CHECK(ctx);
	if(ctx->async_mode) {
		SPP_CUDA(cudaEventRecord(ctx->phase_ev[PH_CHOL_KERNEL][1], st));
		ctx->phase_used[PH_CHOL_KERNEL] = true;
	}
	if(timing) {
		SPP_CUDA(cudaEventRecord(ctx->ev[5], st));
		SPP_CUDA(cudaEventSynchronize(ctx->ev[5]));
		float ms;
		cudaEventElapsedTime(&ms, ctx->ev[4], ctx->ev[5]);
		int h[3];
		cudaMemcpy(h, ch.df_flags.p(), sizeof(h), cudaMemcpyDeviceToHost);
		fprintf(stderr, "[spp chol dataflow] ld %zu, %zu tile columns: %.3f ms = %.2f TFLOP/s (tasks taken %d, roles %d, watchdog %d)\n", ld, NJH,
			ms, (double)ld * ld * ld / 3 / ms * 1e-9, h[0], h[1], h[2]);
		std::vector<unsigned long long> d(dbg.size());
		cudaMemcpy(d.data(), dbg.p(), d.size() * 8, cudaMemcpyDeviceToHost);
		// the chain: for panel i, wait for the diagonal tile after H2(i-1), potrf + inverse, H1(i), H2(i)
		double s_wait = 0, s_potrf = 0, s_h1 = 0, s_h2 = 0;
		for(size_t i = 0; i < NB; ++ i) {
			const double t_wait = i? (double)(long long)(d[i] - d[3 * NB + i - 1]) * 1e-3 : 0, t_potrf = (double)(long long)(d[NB + i] - d[i]) * 1e-3;
			const double t_h1 = (i + 1 < NB)? (double)(long long)(d[2 * NB + i] - d[NB + i]) * 1e-3 : 0;
			const double t_h2 = (i + 1 < NB)? (double)(long long)(d[3 * NB + i] - d[2 * NB + i]) * 1e-3 : 0;
			s_wait += t_wait; s_potrf += t_potrf; s_h1 += t_h1; s_h2 += t_h2;
			if(i < 3 || i % 8 == 0 || i + 2 >= NB)
				fprintf(stderr, "[spp chol dataflow] panel %zu at %.1f us: flag->potrf %.1f, potrf %.1f, H1 %.1f, H2 %.1f\n", i,
					(double)(long long)(d[i] - d[0]) * 1e-3, t_wait, t_potrf, t_h1, t_h2);
		}
		fprintf(stderr, "[spp chol dataflow] chain %.1f us: flag->potrf %.1f, potrf until the helpers can start %.1f, H1 (incl. waiting for partial sums) %.1f, H2 %.1f\n",
			(double)(long long)(d[5 * NB - 1] - d[0]) * 1e-3, s_wait, s_potrf, s_h1, s_h2);
		double w_flags = 0, w_trsm = 0, w_pipe = 0, w_total = 0, t_end_min = 1e30, t_end_max = 0; size_t n_w = 0;
		for(size_t c = 0; c < n_ctas; ++ c) {
			const unsigned long long *w = &d[5 * NB + 8 * c];
			if(!w[3]) continue; // not a worker
			++ n_w;
			w_flags += (double)w[0]; w_trsm += (double)w[1]; w_pipe += (double)w[4]; w_total += (double)w[5];
			const double te = (double)(long long)(w[3] - d[0]) * 1e-3;
			t_end_min = std::min(t_end_min, te); t_end_max = std::max(t_end_max, te);
		}
		if(n_w)
			fprintf(stderr, "[spp chol dataflow] %zu workers: producer waits %.1f %% of the run for operand flags, %.1f %% for the diagonal block; "
				"consumer warp 0 waits %.1f %% for chunks; last task taken at %.1f .. %.1f us\n", n_w, 100 * w_flags / w_total, 100 * w_trsm / w_total,
				100 * w_pipe / w_total, t_end_min, t_end_max);
	}
}

// The same for a panel with ONE diagonal block (ld == 128) on a stream of the caller's choice: the diagonal-block
// kernel and the solve of the block row, no look-ahead needed -- the supernodal factorisation runs its many narrow
// supernodes side by side with this.
void dense_chol_factor_single_panel(spp_ctx *ctx, cudaStream_t stream, double *A, size_t n_cols, double *Rinv, int *info)
{
	chol_init_streams(ctx);
	k_potrf128<<<1, PT, POTRF_SMEM_EXCLUSIVE, stream>>>(A, CH_NB, 0, Rinv, info, 0);
	LAUNCH_CHECK(ctx);
	if(n_cols > CH_NB) {
		k_gemm_tn<GEMM_TRSM, 128, 64><<<(unsigned)((n_cols - CH_NB) / 64), 256, gemm_smem<128, 64>(), stream>>>(A, CH_NB, 0, 0, CH_NB, Rinv);
		LAUNCH_CHECK(ctx);
	}
}

// Backward solve R11 x = y on a factored panel (see dense_chol_factor_panel): y (ld doubles, in place) must not alias the
// panel's first ld columns; flags: ld / 128 ints, zero on entry.
void dense_chol_backsolve_panel(spp_ctx *ctx, cudaStream_t stream, const double *A, size_t ld, const double *Rinv, double *y, int *flags)
{
	chol_init_streams(ctx);
	k_backsolve<<<(unsigned)(ld / CH_NB), 256, BACKSOLVE_SMEM, stream>>>(A, ld, ld / CH_NB, Rinv, y, flags);
	LAUNCH_CHECK(ctx);
}

// A: device, augmented storage (upper triangle of the n x n matrix filled, everything else zero, rhs NOT yet
// placed). d_rhs_x: device vector of n doubles, rhs in, solution out. Returns SPP_OK / SPP_NOT_POSDEF.
int dense_chol_solve_device(spp_ctx *ctx, double *A, size_t n, double *d_rhs_x)
{
	DenseChol &ch = ctx->chol;
	const size_t ld = dense_chol_ld(n), n_blk = ld / CH_NB;
	cudaStream_t st = ctx->stream;
	chol_init_streams(ctx);
	ch.info.resize(1 + n_blk);
	SPP_CUDA(cudaMemsetAsync(ch.info.p(), 0, (1 + n_blk) * sizeof(int), st));
	if(ch.work.size() != n_blk * CH_NB * CH_NB) { // k_potrf128 writes the upper triangles only
		ch.work.resize(n_blk * CH_NB * CH_NB);
		ch.work.zero(st);
	}
	if(ld > n) {
		k_pad_identity<<<n_blocks(ld - n, 64), 64, 0, st>>>(A, ld, n, ld);
		LAUNCH_CHECK(ctx);
	}
	double *rhs_col = A + ld * ld; // first column of the rhs block
	k_copy_rhs<<<n_blocks(n, 256), 256, 0, st>>>(rhs_col, d_rhs_x, n);
	LAUNCH_CHECK(ctx);
	static const bool timing = getenv("SPP_CHOL_TIMING") != 0;
	if(timing)
		SPP_CUDA(cudaEventRecord(ctx->ev[6], st));
	if(dense_chol_dataflow_enabled()) // only the first 64 columns of the right-hand-side block are looked at
		dense_chol_factor_dataflow(ctx, A, ld, ld + 64, ch.work.p(), ch.info.p());
	else
		dense_chol_factor_panel(ctx, A, ld, ld + CH_NB, ch.work.p(), ch.info.p(), false);
	if(timing)
		SPP_CUDA(cudaEventRecord(ctx->ev[7], st));
	k_backsolve<<<(unsigned)n_blk, 256, BACKSOLVE_SMEM, st>>>(A, ld, n_blk, ch.work.p(), rhs_col, ch.info.p() + 1);
	LAUNCH_CHECK(ctx);
	if(timing) {
		SPP_CUDA(cudaEventRecord(ctx->ev[8], st));
		SPP_CUDA(cudaEventSynchronize(ctx->ev[8]));
		float ms_f, ms_b;
		cudaEventElapsedTime(&ms_f, ctx->ev[6], ctx->ev[7]);
		cudaEventElapsedTime(&ms_b, ctx->ev[7], ctx->ev[8]);
		fprintf(stderr, "[spp chol timing] n %zu: factor %.3f ms (%.2f TFLOP/s), backward solve %.3f ms\n", n, ms_f,
			(double)n * n * n / 3 / ms_f * 1e-9, ms_b);
	}
	k_copy_rhs<<<n_blocks(n, 256), 256, 0, st>>>(d_rhs_x, rhs_col, n);
	LAUNCH_CHECK(ctx);
	if(ctx->async_mode && ctx->async_info) { // the caller synchronises later and reads the status there
		SPP_CUDA(cudaMemcpyAsync(ctx->async_info, ch.info.p(), sizeof(int), cudaMemcpyDeviceToHost, st));
		return SPP_OK;
	}
	ctx->h_scalars.resize(16);
	int *h_info = reinterpret_cast<int*>(ctx->h_scalars.p());
	SPP_CUDA(cudaMemcpyAsync(h_info, ch.info.p(), sizeof(int), cudaMemcpyDeviceToHost, st));
	SPP_CUDA(cudaStreamSynchronize(st));
	if(*h_info < 0)
		throw cuda_error("dense Cholesky: the dataflow kernel's watchdog fired (a tile flag never arrived)");
	return (*h_info == 0)? SPP_OK : SPP_NOT_POSDEF;
}

__global__ void k_set_identity(double *__restrict__ Z, size_t ld)
{
	size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
	if(i < ld) Z[i * ld + i] = 1.0;
}

// Inverse of a dense SPD matrix through its Cholesky factor (marginal covariances of the reduced camera system:
// the reference recovers them from the factor of the Schur complement, include/slam/BAMarginals.h:579-760).
// A: device, column-major, ld = dense_chol_ld(n) rows and 2 * ld columns; on entry the upper triangle of the n x n
// matrix sits in the first ld columns (everything else there zero), the second ld columns are scratch. The panel
// factorisation of [A | I] leaves [R | Z], Z = R^-T (lower triangular); then the first ld columns are overwritten with
// MINUS the inverse, -Z^T Z, upper tiles (every 128 x 128 diagonal tile in full), 41 rank-128 DMMA updates that stop at
// the last non-zero block row of Z. Returns SPP_OK / SPP_NOT_POSDEF. Synchronises the stream.
int dense_chol_inverse_device(spp_ctx *ctx, double *A, size_t n)
{
	DenseChol &ch = ctx->chol;
	const size_t ld = dense_chol_ld(n), n_blk = ld / CH_NB;
	cudaStream_t st = ctx->stream;
	chol_init_streams(ctx);
	ch.info.resize(1 + n_blk);
	SPP_CUDA(cudaMemsetAsync(ch.info.p(), 0, (1 + n_blk) * sizeof(int), st));
	if(ch.work.size() != n_blk * CH_NB * CH_NB) {
		ch.work.resize(n_blk * CH_NB * CH_NB);
		ch.work.zero(st);
	}
	if(ld > n) {
		k_pad_identity<<<n_blocks(ld - n, 64), 64, 0, st>>>(A, ld, n, ld);
		LAUNCH_CHECK(ctx);
	}
	double *Z = A + ld * ld;
	SPP_CUDA(cudaMemsetAsync(Z, 0, ld * ld * sizeof(double), st));
	k_set_identity<<<n_blocks(ld, 256), 256, 0, st>>>(Z, ld);
	LAUNCH_CHECK(ctx);
	dense_chol_factor_panel(ctx, A, ld, 2 * ld, ch.work.p(), ch.info.p(), true);
	SPP_CUDA(cudaMemsetAsync(A, 0, ld * ld * sizeof(double), st));
	for(size_t kb = 0; kb < n_blk; ++ kb) { // block row kb of Z is non-zero in its first kb + 1 column blocks
		const size_t m = (kb + 1) * CH_NB;
		if((m / 128) * (m / 64) >= 148) {
			dim3 grid((unsigned)(m / 64), (unsigned)(m / 128));
			k_gemm_tn<GEMM_GRAM, 128, 64><<<grid, 256, gemm_smem<128, 64>(), st>>>(A, ld, kb * CH_NB, 0, 0, Z);
		} else {
			dim3 grid((unsigned)(m / 64), (unsigned)(m / 64));
			k_gemm_tn<GEMM_GRAM, 64, 64><<<grid, 128, gemm_smem<64, 64>(), st>>>(A, ld, kb * CH_NB, 0, 0, Z);
		}
		LAUNCH_CHECK(ctx);
	}
	ctx->h_scalars.resize(16);
	int *h_info = reinterpret_cast<int*>(ctx->h_scalars.p());
	SPP_CUDA(cudaMemcpyAsync(h_info, ch.info.p(), sizeof(int), cudaMemcpyDeviceToHost, st));
	SPP_CUDA(cudaStreamSynchronize(st));
	return (*h_info == 0)? SPP_OK : SPP_NOT_POSDEF;
}

} // namespace spp

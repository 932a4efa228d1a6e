// schur_kernels.cu -- stage 2 and 4 of the hot path: landmark-side Schur complement and back-substitution.
//
// Reference functions replaced (SURVEY 8(a) rows a9-a13, a16; all inside
// CLinearSolver_Schur::Solve_PosDef_Blocky, include/slam/LinearSolver_Schur.h:1623-1935):
//   Permute_UpperTriangular_To / SliceTo / TransposeTo  Schur.h:1687-1709   -> no-ops here: the system is
//                                                        stored as (U, V, W) in Schur order from the start
//   InverseOf_BlockDiag_FBS_Parallel + Scale(-1)        Schur.h:1720-1735, BlockMatrixFBS.inl:1749-1868
//   U.MultiplyToWith_FBS(C^-1)                          Schur.h:1743-1745   (Y = W C^-1, per observation)
//   (-U C^-1).MultiplyToWith_FBS(V, upper) + AddTo_FBS  Schur.h:1757-1767   (S = A - Y W^T, upper blocks)
//   PreMultiply_Add_FBS (rhs)                           Schur.h:1829-1830   (b = x - Y l)
//   PostMultiply_Add_FBS_Parallel + PreMultiply_Add     Schur.h:1867-1881   (dl = C^-1 (l - W^T dx))
//
// The product S_ij = A_ij - sum_p Y_ip W_jp^T is evaluated per destination block from a precomputed list of
// observation pairs sorted by landmark -- the reference's own accumulation order (BlockMatrixFBS.h:395-448)
// -- so there are no floating-point atomics and the result is bit-reproducible.

#include "spp_ctx.h"
#include <algorithm>

namespace spp {

size_t dense_chol_ld(size_t n);
size_t dense_chol_storage(size_t n);

#define LAUNCH_CHECK(ctx) do { ++ (ctx)->n_launches; SPP_CUDA(cudaGetLastError()); } while(0)

// warp per 32 consecutive landmarks: lane l inverts landmark p0 + l, Cinv = (V + alpha I)^-1 by cofactors (what
// Eigen's fixed 3x3 inverse() does, BlockMatrixBase.h:1256-1270); V is read and Cinv written as the warp's contiguous
// 32 x 9 range through shared memory. Then the warp walks the CONTIGUOUS W range of its 32 tracks in 16-byte units
// (coalesced loads, one double2 store of Y_o = W_o Cinv per unit). A lane's position (o, unit j of 9) advances by 32
// units = 3 observations + 5 units per step, so there is no division; obs_pt[o] names the unit's landmark.
#define LI_WARPS 8

__global__ void __launch_bounds__(LI_WARPS * 32) k_landmark_inverse(size_t P, double alpha, const uint32_t *__restrict__ pt_ptr,
	const uint32_t *__restrict__ obs_pt, const double *__restrict__ V, const double *__restrict__ W, double *__restrict__ Cinv,
	double *__restrict__ Y)
{
	__shared__ double sC[LI_WARPS][32 * 9];
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	const size_t p0 = (blockIdx.x * (size_t)LI_WARPS + warp) * 32;
	if(p0 >= P) return;
	const unsigned np = (unsigned)((P - p0 < 32)? P - p0 : 32);
	double *sc = sC[warp];
	for(unsigned i = lane; i < np * 9; i += 32)
		sc[i] = V[p0 * 9 + i];
	__syncwarp();
	if((unsigned)lane < np) {
		double *Vp = sc + lane * 9; // column-major; overwritten by this lane's inverse
		double m00 = Vp[0] + alpha, m10 = Vp[1], m20 = Vp[2];
		double m01 = Vp[3], m11 = Vp[4] + alpha, m21 = Vp[5];
		double m02 = Vp[6], m12 = Vp[7], m22 = Vp[8] + alpha;
		// cofactors
		double c00 = m11 * m22 - m12 * m21, c10 = m21 * m02 - m22 * m01, c20 = m01 * m12 - m02 * m11;
		double det = c00 * m00 + c10 * m10 + c20 * m20;
		double id = 1.0 / det;
		double inv[9]; // column-major
		inv[0] = c00 * id; inv[3] = c10 * id; inv[6] = c20 * id;
		inv[1] = (m12 * m20 - m10 * m22) * id; inv[4] = (m22 * m00 - m20 * m02) * id; inv[7] = (m02 * m10 - m00 * m12) * id;
		inv[2] = (m10 * m21 - m11 * m20) * id; inv[5] = (m20 * m01 - m21 * m00) * id; inv[8] = (m00 * m11 - m01 * m10) * id;
		#pragma unroll
		for(int i = 0; i < 9; ++ i)
			Vp[i] = inv[i];
	}
	__syncwarp();
	for(unsigned i = lane; i < np * 9; i += 32)
		Cinv[p0 * 9 + i] = sc[i];
	// unit j of a 6 x 3 column-major block holds rows r, r + 1 (r = 2 (j mod 3)) of column c = j / 3
	const unsigned o_end = pt_ptr[p0 + np];
	unsigned o = pt_ptr[p0] + lane / 9, j = lane % 9;
	while(o < o_end) {
		const unsigned c = j / 3, r = 2 * (j - 3 * c);
		const double *Ci = sc + (obs_pt[o] - (unsigned)p0) * 9 + c * 3;
		const double2 *Wo = reinterpret_cast<const double2*>(W + (size_t)o * 18 + r);
		const double2 w0 = Wo[0], w1 = Wo[3], w2 = Wo[6];
		*reinterpret_cast<double2*>(Y + (size_t)o * 18 + 2 * j) = make_double2(w0.x * Ci[0] + w1.x * Ci[1] + w2.x * Ci[2],
			w0.y * Ci[0] + w1.y * Ci[1] + w2.y * Ci[2]);
		o += 3; j += 5;
		if(j >= 9) { j -= 9; ++ o; }
	}
}

// ---- the Schur product ---------------------------------------------------------------------------------
// S(i,j) = [i == j] (U_i + alpha I) - sum_pairs Y_a W_b^T ; for i == j also b_i = gc_i - sum_a Y_a gp_{p(a)}
//
// Lane mapping: a warp is three groups of nine lanes (27 of 32 lanes work); group g of a warp takes pairs g, g + 3 * n_warps,
// ... of the list. Lane q = r3 + 3 k of a group owns the rows {2 r3, 2 r3 + 1} of the product and ONE value k of the
// summation index (a column of Y_a / W_b): per pair it loads its own 16-byte chunk of Y_a -- the nine lanes of a group
// cover the 144-byte block exactly once -- and the 48 bytes of column k of W_b, i.e. four 16-byte loads and ~10 L1
// wavefronts per pair (the kernel is L1-throughput bound); twelve accumulators per lane. No accumulator crosses a lane
// until the end, where the three k-partials of a row pair and then the three groups are added in a fixed order, so the
// result is bit-reproducible.
// (Measured alternatives, Venice shape: a lane owning a 2 x 2 sub-block of the product and all three k -- six 16-byte
// loads and ~16 L1 wavefronts per pair, L1 at 74 % of peak (profiles/r2q_full.csv). Against that mapping at 0.75 ms,
// one DMMA m8n8k4 per pair with one value per lane -- warp per block 1.15 ms, pair lists cut into 128-pair work items
// 1.25 ms: a pair is a dependent gather of two 144-byte blocks and the product is bound by the latency / L2 traffic of
// those gathers, not by the 108 FMAs.)
#define SB_WARPS 8
#define SB_UNROLL 4 // pairs in flight per lane group

struct SchurAccK {
	double s[2][6], b[2]; // (row 2 r3 + i, column c) partial over this lane's k; rhs rows
};

template <bool RHS>
__device__ __forceinline__ void schur_accumulate_k(uint64_t k0, uint64_t end, uint64_t stride, int r3, int kk,
	const uint32_t *__restrict__ pair_a, const uint32_t *__restrict__ pair_b, const double *__restrict__ Y,
	const double *__restrict__ W, const double *__restrict__ gp, const uint32_t *__restrict__ obs_pt, SchurAccK &acc)
{
	const double2 zero2 = make_double2(0.0, 0.0);
	// the observation indices of a trip are fetched one trip ahead, so that the dependent chain of a trip is one
	// memory round trip (the Y / W blocks) instead of two (index, then block)
	unsigned oa[SB_UNROLL], ob[SB_UNROLL];
	bool ok[SB_UNROLL];
	#pragma unroll
	for(int u = 0; u < SB_UNROLL; ++ u) {
		const uint64_t q = k0 + u * stride;
		ok[u] = q < end;
		oa[u] = ok[u]? pair_a[q] : 0u;
		ob[u] = RHS? oa[u] : (ok[u]? pair_b[q] : 0u);
	}
	for(uint64_t k = k0; k < end; k += SB_UNROLL * stride) {
		double2 y[SB_UNROLL], w[SB_UNROLL][3];
		double g[SB_UNROLL];
		#pragma unroll
		for(int u = 0; u < SB_UNROLL; ++ u) {
			const double2 *Wb = reinterpret_cast<const double2*>(W + (size_t)ob[u] * 18 + 6 * kk);
			y[u] = ok[u]? *reinterpret_cast<const double2*>(Y + (size_t)oa[u] * 18 + 6 * kk + 2 * r3) : zero2;
			#pragma unroll
			for(int q = 0; q < 3; ++ q)
				w[u][q] = ok[u]? Wb[q] : zero2;
			if(RHS)
				g[u] = ok[u]? gp[(size_t)obs_pt[oa[u]] * 3 + kk] : 0.0;
		}
		#pragma unroll
		for(int u = 0; u < SB_UNROLL; ++ u) { // next trip's indices
			const uint64_t q = k + (SB_UNROLL + u) * stride;
			ok[u] = q < end;
			oa[u] = ok[u]? pair_a[q] : 0u;
			ob[u] = RHS? oa[u] : (ok[u]? pair_b[q] : 0u);
		}
		#pragma unroll
		for(int u = 0; u < SB_UNROLL; ++ u) {
			#pragma unroll
			for(int q = 0; q < 3; ++ q) {
				acc.s[0][2 * q] += y[u].x * w[u][q].x;
				acc.s[0][2 * q + 1] += y[u].x * w[u][q].y;
				acc.s[1][2 * q] += y[u].y * w[u][q].x;
				acc.s[1][2 * q + 1] += y[u].y * w[u][q].y;
			}
			if(RHS) {
				acc.b[0] += y[u].x * g[u];
				acc.b[1] += y[u].y * g[u];
			}
		}
	}
}

// sums v over the three k-lanes of a row pair (lanes r3, r3 + 3, r3 + 6 of the group; k ascending), result valid in the k = 0 lane
__device__ __forceinline__ double sum_over_k(double v, int lane)
{
	const double v1 = __shfl_sync(0xffffffffu, v, (lane + 3) & 31), v2 = __shfl_sync(0xffffffffu, v, (lane + 6) & 31);
	return (v + v1) + v2;
}

// off-diagonal blocks (list entries first_blk ..): one warp per block. The pair lists differ a lot in length (1 .. several
// hundred pairs), so with a fixed block -> warp assignment a CTA lives as long as its longest list while its other
// warps idle (33 % of the warp slots active, profiles/r1k_full.csv); the warps of a persistent grid take block after
// block from the counter `queue` instead (with four pairs in flight per lane group: stage 1.26 -> 1.19 ms; the kernel
// is bound by the L2 sector traffic of its gathers, 2 x 144 bytes per pair, not by the imbalance). (Measured and
// rejected: the three lane groups sharing ONE pair, each taking one column of Y_a / W_b -- the minimum of L1 wavefronts
// per pair, but three times the index loads and loop trips per pair: 1.49 ms against 1.32 ms for the stage.)
__global__ void __launch_bounds__(SB_WARPS * 32, 2) k_schur_blocks_k(size_t first_blk, size_t n_blocks_total, size_t ld,
	const uint32_t *__restrict__ blk_row, const uint32_t *__restrict__ blk_col, const uint64_t *__restrict__ blk_ptr,
	const uint32_t *__restrict__ pair_a, const uint32_t *__restrict__ pair_b, const double *__restrict__ Y,
	const double *__restrict__ W, double *__restrict__ S, const uint32_t *__restrict__ slot, unsigned *__restrict__ queue)
{
	const int lane = threadIdx.x & 31;
	const int grp = lane / 9, q9 = lane - grp * 9, r3 = q9 % 3, kk = q9 / 3;
	for(;;) {
		unsigned idx = 0;
		if(lane == 0)
			idx = atomicAdd(queue, 1u);
		const size_t blk = first_blk + __shfl_sync(0xffffffffu, idx, 0);
		if(blk >= n_blocks_total) return;
		const unsigned bi = blk_row[blk], bj = blk_col[blk];
		SchurAccK acc;
		#pragma unroll
		for(int i = 0; i < 2; ++ i) {
			#pragma unroll
			for(int c = 0; c < 6; ++ c) acc.s[i][c] = 0;
			acc.b[i] = 0;
		}
		if(grp < 3)
			schur_accumulate_k<false>(blk_ptr[blk] + grp, blk_ptr[blk + 1], 3, r3, kk, pair_a, pair_b, Y, W, 0, 0, acc);
		#pragma unroll
		for(int i = 0; i < 2; ++ i) {
			#pragma unroll
			for(int c = 0; c < 6; ++ c) {
				double v = sum_over_k(acc.s[i][c], lane);
				const double v1 = __shfl_sync(0xffffffffu, v, (lane + 9) & 31), v2 = __shfl_sync(0xffffffffu, v, (lane + 18) & 31);
				acc.s[i][c] = (v + v1) + v2; // the three pair groups, fixed order
			}
		}
		if(lane < 3) { // k = 0 lanes of group 0: rows 2 r3, 2 r3 + 1
			const size_t ldo = ld? ld : 6;
			double *Sb = ld? S + ((size_t)bj * 6) * ld + (size_t)bi * 6 + 2 * r3 : S + (size_t)(slot? slot[blk] : blk) * 36 + 2 * r3;
			#pragma unroll
			for(int c = 0; c < 6; ++ c) {
				Sb[c * ldo] = -acc.s[0][c];
				Sb[c * ldo + 1] = -acc.s[1][c];
			}
		}
	}
}

// diagonal blocks (list entries 0 .. C-1, pairs (a, a) = the camera's observations): one CTA per camera, every
// warp group takes a strided share of the list, the 3 * SB_WARPS partial sums are added in a fixed order
__global__ void __launch_bounds__(SB_WARPS * 32, 2) k_schur_diag_k(size_t ld, double alpha, const uint64_t *__restrict__ blk_ptr,
	const uint32_t *__restrict__ pair_a, const double *__restrict__ Y, const double *__restrict__ W,
	const double *__restrict__ U, const double *__restrict__ gc, const double *__restrict__ gp,
	const uint32_t *__restrict__ obs_pt, double *__restrict__ S, double *__restrict__ b, const uint32_t *__restrict__ slot)
{
	__shared__ double part[3 * SB_WARPS][3][14]; // per lane group: rows 2 r3, 2 r3 + 1 x 6 columns, then the two rhs rows
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	const size_t bi = blockIdx.x;
	const int grp = lane / 9, q9 = lane - grp * 9, r3 = q9 % 3, kk = q9 / 3;
	SchurAccK acc;
	#pragma unroll
	for(int i = 0; i < 2; ++ i) {
		#pragma unroll
		for(int c = 0; c < 6; ++ c) acc.s[i][c] = 0;
		acc.b[i] = 0;
	}
	if(grp < 3)
		schur_accumulate_k<true>(blk_ptr[bi] + warp * 3 + grp, blk_ptr[bi + 1], 3 * SB_WARPS, r3, kk, pair_a, pair_a, Y, W, gp, obs_pt, acc);
	#pragma unroll
	for(int i = 0; i < 2; ++ i) {
		#pragma unroll
		for(int c = 0; c < 6; ++ c)
			acc.s[i][c] = sum_over_k(acc.s[i][c], lane);
		acc.b[i] = sum_over_k(acc.b[i], lane);
	}
	if(grp < 3 && kk == 0) {
		double *pp = part[warp * 3 + grp][r3];
		#pragma unroll
		for(int c = 0; c < 6; ++ c) {
			pp[2 * c] = acc.s[0][c];
			pp[2 * c + 1] = acc.s[1][c];
		}
		pp[12] = acc.b[0];
		pp[13] = acc.b[1];
	}
	__syncthreads();
	if(threadIdx.x < 42) { // 36 entries of the block (column-major: row pair r3, element e = 2 c + i), then the 6 rhs rows
		const int t = threadIdx.x;
		const int row = (t < 36)? t % 6 : t - 36, col = (t < 36)? t / 6 : 6;
		const int pr = row >> 1, e = (t < 36)? 2 * col + (row & 1) : 12 + (row & 1);
		double v = 0;
		for(int sgrp = 0; sgrp < 3 * SB_WARPS; ++ sgrp)
			v += part[sgrp][pr][e];
		if(t < 36) {
			const double u = U[bi * 36 + col * 6 + row] + ((row == col)? alpha : 0.0);
			double *Sb = ld? S + (bi * 6 + col) * ld + bi * 6 + row : S + (size_t)(slot? slot[bi] : bi) * 36 + col * 6 + row;
			*Sb = u - v;
		} else
			b[bi * 6 + row] = gc[bi * 6 + row] - v;
	}
}

// thread per landmark: dl = Cinv (gp - sum_o W_o^T dxc_{c(o)})
__global__ void k_backsubstitute(size_t P, const uint32_t *__restrict__ pt_ptr, const uint32_t *__restrict__ obs_cam,
	const double *__restrict__ W, const double *__restrict__ Cinv, const double *__restrict__ gp,
	const double *__restrict__ dxc, double *__restrict__ dxp)
{
	size_t p = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
	if(p >= P) return;
	double l0 = gp[p * 3], l1 = gp[p * 3 + 1], l2 = gp[p * 3 + 2];
	const unsigned beg = pt_ptr[p], end = pt_ptr[p + 1];
	for(unsigned o = beg; o < end; ++ o) {
		const unsigned c = obs_cam[o];
		const double *Wo = W + (size_t)o * 18;
		const double *d = dxc + (size_t)c * 6;
		double dd[6];
		#pragma unroll
		for(int i = 0; i < 6; i += 2) {
			double2 t = *reinterpret_cast<const double2*>(d + i);
			dd[i] = t.x; dd[i + 1] = t.y;
		}
		double w[18];
		#pragma unroll
		for(int i = 0; i < 18; i += 2) {
			double2 t = *reinterpret_cast<const double2*>(Wo + i);
			w[i] = t.x; w[i + 1] = t.y;
		}
		double s0 = 0, s1 = 0, s2 = 0;
		#pragma unroll
		for(int r = 0; r < 6; ++ r) {
			s0 += w[r] * dd[r];
			s1 += w[6 + r] * dd[r];
			s2 += w[12 + r] * dd[r];
		}
		l0 -= s0; l1 -= s1; l2 -= s2;
	}
	const double *Ci = Cinv + p * 9;
	dxp[p * 3 + 0] = Ci[0] * l0 + Ci[3] * l1 + Ci[6] * l2;
	dxp[p * 3 + 1] = Ci[1] * l0 + Ci[4] * l1 + Ci[7] * l2;
	dxp[p * 3 + 2] = Ci[2] * l0 + Ci[5] * l1 + Ci[8] * l2;
}

// ---------------------------------------------------------------------------------------------------

// forms Cinv, Y, the dense upper-triangular reduced camera system S and its right-hand side b
// alpha damps the landmark blocks of this rank; alpha_diag is what this rank adds to the camera diagonal (alpha on
// rank 0, zero elsewhere: the partial systems are summed over ranks)
// sparse_rcs: S goes to the compact block list s.Sblk (the supernodal solver scatters it into its panels)
void schur_form_reduced_system(spp_ctx *ctx, double alpha, double alpha_diag, bool sparse_rcs)
{
	SchurSystem &s = ctx->sys;
	const size_t n = s.C * 6;
	const size_t ld = sparse_rcs? 0 : dense_chol_ld(n); // S is written straight into the dense solver's padded storage
	s.Cinv.resize(s.P * 9);
	s.Y.resize(s.O * 18);
	const uint32_t *slot = (sparse_rcs && s.n_blocks_global)? s.blk_slot.p() : 0; // several ranks: the global block list
	if(sparse_rcs) {
		s.Sblk.resize((s.n_blocks_global? s.n_blocks_global : s.n_blocks) * 36);
		if(slot)
			s.Sblk.zero(ctx->stream); // blocks no landmark of this rank contributes to
	} else
		s.S.resize(dense_chol_storage(n));
	double *S_out = sparse_rcs? s.Sblk.p() : s.S.p();
	s.b.resize(n);
	if(s.P) {
		k_landmark_inverse<<<n_blocks(s.P, LI_WARPS * 32), LI_WARPS * 32, 0, ctx->stream>>>(s.P, alpha, s.pt_ptr.p(), s.obs_pt.p(),
			s.V.p(), s.W.p(), s.Cinv.p(), s.Y.p());
		LAUNCH_CHECK(ctx);
	}
	if(!sparse_rcs)
		s.S.zero(ctx->stream);
	if(s.C) { // list entries 0 .. C-1 are the diagonal blocks
		k_schur_diag_k<<<(unsigned)s.C, SB_WARPS * 32, 0, ctx->stream>>>(ld, alpha_diag, s.blk_ptr.p(), s.pair_a.p(), s.Y.p(),
			s.W.p(), s.U.p(), s.gc.p(), s.gp.p(), s.obs_pt.p(), S_out, s.b.p(), slot);
		LAUNCH_CHECK(ctx);
	}
	if(s.n_blocks > s.C) {
		static int n_sms = 0;
		if(!n_sms)
			SPP_CUDA(cudaDeviceGetAttribute(&n_sms, cudaDevAttrMultiProcessorCount, ctx->device));
		s.schur_queue.resize(1);
		SPP_CUDA(cudaMemsetAsync(s.schur_queue.p(), 0, sizeof(unsigned), ctx->stream));
		const unsigned grid = std::min(n_blocks(s.n_blocks - s.C, SB_WARPS), (unsigned)n_sms * 2u); // two CTAs per SM
		k_schur_blocks_k<<<grid, SB_WARPS * 32, 0, ctx->stream>>>(s.C, s.n_blocks, ld, s.blk_row.p(), s.blk_col.p(),
			s.blk_ptr.p(), s.pair_a.p(), s.pair_b.p(), s.Y.p(), s.W.p(), S_out, slot, s.schur_queue.p());
		LAUNCH_CHECK(ctx);
	}
}

void schur_backsubstitute(spp_ctx *ctx)
{
	SchurSystem &s = ctx->sys;
	s.dxp.resize(s.P * 3);
	if(s.P) {
		k_backsubstitute<<<n_blocks(s.P, 128), 128, 0, ctx->stream>>>(s.P, s.pt_ptr.p(), s.obs_cam.p(), s.W.p(),
			s.Cinv.p(), s.gp.p(), s.dxc.p(), s.dxp.p());
		LAUNCH_CHECK(ctx);
	}
}

} // namespace spp

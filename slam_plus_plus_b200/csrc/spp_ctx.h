// spp_ctx.h -- the solver context: device-resident system, symbolic structures, work buffers.
#pragma once

#include "spp_common.cuh"
#include "block_ordering.h"
#include <map>
#include <cuda.h> // CUtensorMap (types only: the encoder is fetched through cudaGetDriverEntryPoint)

namespace spp {

// landmark Schur system: the layout every BA stage kernel works on. Cameras and points are in the
// reference's guided Schur ordering (6-wide vertices first, then 3-wide, id order kept inside each group;
// src/slam/LinearSolver_Schur.cpp:771-838); observations are sorted by point so that a landmark's
// W / Y blocks are contiguous (a "track").
struct SchurSystem {
	size_t C, P, O; // cameras, points, observations
	// structure (device)
	DBuf<uint32_t> obs_cam, obs_pt;  // [O] local camera / point index of each observation (track order)
	DBuf<uint32_t> pt_ptr;           // [P+1] track of point p = observations pt_ptr[p] .. pt_ptr[p+1]
	DBuf<uint32_t> cam_ptr, cam_obs; // [C+1], [O] per camera: observation indices (edge insertion order)
	// reduced camera system structure: upper-triangular 6x6 block list and, per block, the pairs of
	// observations (a, b) of one landmark that contribute Y_a W_b^T (ascending landmark order)
	size_t n_blocks, n_pairs;
	DBuf<uint32_t> blk_row, blk_col; // [n_blocks] camera indices i <= j
	DBuf<uint64_t> blk_ptr;          // [n_blocks+1]
	DBuf<uint32_t> pair_a, pair_b;   // [n_pairs]
	std::vector<uint32_t> h_blk_row, h_blk_col; // host copy of the block pattern
	// several ranks + block-sparse reduced camera system: the block list of the WHOLE graph (identical on every rank)
	// and the position of this rank's blocks in it; n_blocks_global == 0 otherwise
	size_t n_blocks_global;
	std::vector<uint32_t> h_gblk_row, h_gblk_col;
	DBuf<uint32_t> blk_slot;         // [n_blocks] local block -> global block
	DBuf<uint32_t> gblk_row, gblk_col; // [n_blocks_global] the global block list on the device
	// values (device)
	DBuf<double> U;    // [C*36] camera diagonal blocks (column-major 6x6, undamped, incl. unary factor)
	DBuf<double> V;    // [P*9]  point diagonal blocks
	DBuf<double> W;    // [O*18] camera x point blocks J_c^T Sigma^-1 J_p (column-major 6x3), track order
	DBuf<double> gc, gp; // [6C], [3P] gradient eta
	DBuf<double> Cinv; // [P*9]  (V + alpha I)^-1
	DBuf<double> Y;    // [O*18] W C^-1
	DBuf<double> S;    // [n*n] dense column-major reduced camera system, n = 6C (upper triangle valid)
	DBuf<double> Sblk; // [n_blocks*36] the same as a compact block list (sparse reduced camera system), order of blk_row/col
	DBuf<double> S_copy; // optional copy kept for spp_schur_get_reduced_system
	DBuf<double> Sinv; // [ld * 2 ld] marginals: [S | I] -> [-S^-1 | R^-T] (marginals.cu)
	DBuf<double> cov_cam, cov_pt; // marginals: staging of the covariance blocks (kept: no allocation per call)
	DBuf<double> cov_pair, cov_obs; // covariance blocks: camera pairs, camera x point of observations
	DBuf<uint32_t> cov_cam_a, cov_cam_b, cov_obs_idx, cov_pos; // the requested pairs / observations; edge index -> track position
	// joint marginals (joint_marginals.cu), one batch at a time: compact right-hand sides / forward solves, the sets'
	// covariances, the batch's index arrays, set dimensions, set offsets and Gram problems
	DBuf<double> joint_F, joint_out;
	DBuf<uint32_t> joint_idx, joint_dim;
	DBuf<uint64_t> joint_off;
	DBuf<uint8_t> joint_jobs;
	DBuf<unsigned> schur_queue; // [1] work counter of k_schur_blocks_k
	DBuf<double> b, b_copy; // [n] reduced right-hand side / camera increment
	DBuf<double> dxc, dxp; // [6C], [3P] increments
	bool keep_reduced;
	bool sparse_solved;  // the last solve went through the block-sparse path and succeeded (Sblk, b_copy, dxc are consistent)
	SchurSystem() : C(0), P(0), O(0), n_blocks(0), n_pairs(0), n_blocks_global(0), keep_reduced(false), sparse_solved(false) {}
};

struct BAProblem {
	bool valid;
	size_t n_vertices;
	std::vector<uint8_t> vtype;          // per vertex id
	std::vector<uint32_t> vertex_local;  // vertex id -> camera / point index
	std::vector<uint32_t> cam_vertex, pt_vertex; // local index -> vertex id
	std::vector<uint32_t> obs_orig;      // track position -> original edge index (host copy, fetched on demand)
	std::vector<uint32_t> h_obs_cam, h_obs_pt; // host copies (track order, fetched on demand)
	DBuf<uint32_t> d_obs_orig;           // the same map on the device
	bool host_maps_valid;
	bool raw_on_device;                  // the caller's arrays (edge insertion order) are still staged on the device: the graph can be appended to
	size_t n_obs_raw;                    // observations staged
	int uf_is_cam; long uf_index;        // vertex id 0 carries the unary factor (-1: added by another rank)
	size_t P_global, pt_begin, pt_end;   // landmark slice of this rank (multi-GPU)
	int jac_mode;
	int loss_kind; double loss_scale;    // robust loss of the observations (SPP_LOSS_*, scale k), context state like jac_mode
	// device state
	DBuf<double> cam_state, cam_intr, pts;        // [6C], [5C], [3P]
	DBuf<double> cam_state_saved, pts_saved;
	DBuf<double> cam_state0, pts0;                // snapshot taken by spp_ba_set_graph
	DBuf<double> z, info;                         // [2O], [4O] track order
	DBuf<double> camRt;                           // [C*7*12] base + 6 perturbed [R|t]
	DBuf<double> camK;                            // [C*5] fx fy cx cy k
	DBuf<double> pt_rec;                          // [O*10] per observation: upper(Jp^T Sigma^-1 Jp) (6), Jp^T Sigma^-1 r (3), pad
	DBuf<double> partial;                         // reduction scratch
	DBuf<unsigned long long> maxdiag;             // [1] bits of the max per-edge Hessian diagonal
	DBuf<double> obs_err;                         // [2O] scratch of spp_ba_get_observation_errors (s2, w; edge insertion order)
	bool linearised;
	BAProblem() : valid(false), n_vertices(0), host_maps_valid(false), raw_on_device(false), n_obs_raw(0), uf_is_cam(1), uf_index(0), P_global(0), pt_begin(0),
		pt_end(0), jac_mode(0), loss_kind(0), loss_scale(1.0), linearised(false) {}
};

// slot-1 state: map from the caller's lambda values to the SchurSystem arrays
struct SchurSlot {
	bool valid;
	bool filled;                          // (U, V, W) hold the values of the last spp_schur_solve
	size_t n_bcols, n_scalars, n_values;
	std::vector<uint64_t> col_base;       // scalar offset of each block column
	std::vector<uint64_t> order;          // new position -> original block column
	size_t cut;
	DBuf<double> vals, eta;               // staging of the caller's arrays
	DBuf<uint64_t> u_src, v_src, w_src;   // value offsets of the U / V / W blocks
	DBuf<uint8_t> w_transposed;           // W block stored 3x6 in lambda (point id < camera id)
	DBuf<uint64_t> cam_eta_off, pt_eta_off; // scalar offsets in eta
	SchurSlot() : valid(false), filled(false), n_bcols(0), n_scalars(0), n_values(0), cut(0) {}
};

// scratch of the device-side symbolic analysis (symbolic_gpu.cu); grows only
struct SymbolicScratch {
	DBuf<uint8_t> cub_temp;
	DBuf<int> err;
	DBuf<uint32_t> iota, pos_of_edge, cnt, keys_out, cnt_lin, flag, rank, blk_of_lin, pkey, pkey_out;
	DBuf<uint64_t> cnt64, before, n_off, pair_off, pval, pval_out;
	DBuf<uint32_t> ocam, opt, vlocal;   // per-edge local indices (edge insertion order), vertex id -> local index
	DBuf<uint64_t> obs_pt_id, obs_cam_id; // staging of the caller's vertex ids
	DBuf<uint8_t> vtype;
	DBuf<double> z_in, info_in;         // staging of the caller's measurements (edge insertion order)
	DBuf<uint32_t> sl_flag, sl_pos, sl_kept, sl_ocam, sl_opt; // several ranks: compaction of this rank's edges
};

// block-sparse Cholesky (sparse_chol.cu): symbolic structures and the factor. The spp_chol_* slot and the pose path share
// it; owner names the one whose structure the analysis in memory was made for.
enum { SC_OWNER_NONE = 0, SC_OWNER_SLOT, SC_OWNER_POSE };
struct SparseChol {
	bool valid;
	int owner;                       // SC_OWNER_*
	size_t n, B, n_a_blocks, n_l_blocks;
	uint32_t n_levels, tail_level;
	int max_coop_ctas, coop_B;       // cooperative grid size, computed for the kernels of block size coop_B
	std::vector<uint32_t> h_order;   // new position -> caller's block column
	std::vector<uint64_t> h_lptr;    // column pointers of L
	std::vector<uint32_t> h_lrow, h_parent;
	DBuf<uint32_t> d_order, d_lrow, d_lcolof, d_rblk, d_ua, d_ub, d_lvl_ptr, d_lvl_cols, d_lvl_off_blk;
	DBuf<uint64_t> d_lptr, d_rptr, d_uptr, d_lvl_off_ptr;
	DBuf<int64_t> d_src;
	DBuf<double> d_L, d_Linv, d_y;
	DBuf<int> d_info;
	DBuf<double> slot_vals, slot_rhs, slot_x; // staging of the caller's arrays (slot use)
	size_t n_root, n_root_blocks;              // the columns of the narrow top levels form one dense root front
	std::vector<uint32_t> h_ridx;              // column -> index in the root front (0xffffffff: not in it)
	DBuf<uint32_t> d_root_blk, d_root_ua, d_root_ub, d_root_rblk, d_root_cols, d_ridx;
	DBuf<uint64_t> d_root_uptr, d_root_rptr;
	DBuf<double> d_root_S, d_root_rhs;
	SparseChol() : valid(false), owner(SC_OWNER_NONE), n(0), B(0), n_a_blocks(0), n_l_blocks(0), n_levels(0), tail_level(0),
		max_coop_ctas(0), coop_B(0), n_root(0), n_root_blocks(0) {}
};

// pose graph resident on the device (pose_kernels.cu)
struct PoseProblem {
	bool valid, symbolic_done, linearised;
	int dim;
	size_t N, E, n_blocks;
	long uf_block;                          // diagonal block of vertex 0 (unary factor)
	std::vector<uint64_t> h_col_ptr, h_row_idx, h_order_in; // structure of lambda (upper block CSC), optional ordering
	DBuf<double> states, states0, z, info, rec, vals, eta, dx, scratch;
	DBuf<uint32_t> e_from, e_to;
	DBuf<uint64_t> blk_src_ptr, blk_src, vec_src_ptr, vec_src;
	PoseProblem() : valid(false), symbolic_done(false), linearised(false), dim(0), N(0), E(0), n_blocks(0), uf_block(-1) {}
};

// supernodal block Cholesky of a reduced camera system that is too large to be dense (supernodal_chol.cu): every
// supernode owns a dense block-ROW panel of the upper factor R (R^T R = P S P^T), column-major, ld = its own columns
// rounded up to 128 (identity padding), followed by the columns of its row structure and one right-hand-side column
struct SnodeUpdate { // contribution of supernode s to its ancestor t: panel_t -= R_s[:, J]^T R_s[:, J..end]
	uint32_t s, t;
	uint32_t col0;    // first column of panel s of the suffix of its structure that starts inside t
	uint32_t M, N;    // scalar rows (the part of the suffix inside t's own columns) and columns (whole suffix + rhs)
	uint64_t map_off; // block positions in panel t of the suffix blocks, then of the rhs column
};

// selected inversion (selinv.cu): the structure of a supernode is padded to a multiple of SN_SEL_HP columns in its
// scratch; supernodes with one diagonal block and a structure of at most SN_SEL_LANE_MAX_H columns run on the side lanes
enum { SN_SEL_HP = 64, SN_SEL_LANE_MAX_H = 2048 };
inline bool selinv_on_lane(size_t ld, size_t hp) { return ld == 128 && hp <= SN_SEL_LANE_MAX_H; }

struct SupernodalChol {
	bool valid;
	int mode;                              // SPP_RCS_*
	size_t n;                              // block columns (cameras)
	std::vector<uint64_t> user_order;      // ordering given by the caller (spp_schur_set_rcs_ordering), may be empty
	std::vector<uint32_t> h_order;         // new position -> camera
	Supernodes sn;
	std::vector<uint64_t> panel_off;       // [ns] offset of panel s in d_L (doubles)
	std::vector<uint32_t> panel_ld, panel_cols, rinv_first;
	std::vector<SnodeUpdate> updates;      // grouped by s
	std::vector<uint64_t> upd_ptr;         // [ns + 1]
	size_t n_rinv_blocks, n_s_blocks, max_part;
	DBuf<uint32_t> d_cmap, d_rows, d_asm_ld, d_pad_ld, d_pad_n0, d_order;
	DBuf<uint64_t> d_asm_dst, d_rhs_dst, d_pad_off;
	DBuf<double> d_L, d_Rinv, d_x, d_part;
	DBuf<int> d_info;                      // [0] first non-positive pivot, [1..] backsolve flags
	// marginals (selinv.cu): the upper block CSC of S in camera order with the block id of every entry, so that a device
	// binary search finds the panel address of block (a, b) through d_asm_dst; the diagonal block of every camera
	DBuf<uint64_t> d_csc_ptr, d_cam_diag;  // [n + 1], [n]
	DBuf<uint32_t> d_csc_row, d_csc_blk, d_cam_ld;
	double selinv_flops;                   // selected inversion, 2 w^3 / 3 + 2 w^2 h + 2 w h^2 per supernode (padding excluded)
	size_t selinv_main_doubles, selinv_lane_doubles; // scratch: wide supernodes (main stream) / one side lane
	DBuf<double> d_sel_main, d_sel_lane;
	double factor_flops;                   // of the numeric phase as executed by THIS rank (amalgamation zeros included)
	double factor_flops_total;             // the same for the whole factorisation (equal on one rank)
	// several ranks: subtrees of the supernodal elimination tree belong to one rank each, the supernodes above them
	// (owner -1: "shared") are factored by every rank after the contributions to their panels have been summed
	// what the symbolic analysis in memory was made for: the same block list under the same ordering request on the same
	// rank layout needs no new one (the reference, too, orders and analyses only when the structure changed,
	// LinearSolver_Schur.h:1566-1606)
	std::vector<uint32_t> sym_row, sym_col;
	std::vector<uint64_t> sym_user_order;
	int sym_world, sym_rank;
	bool sym_kept;
	std::vector<int> owner;                // [ns] rank that factors supernode s, -1: every rank
	bool distributed;                      // some supernode has an owner
	DBuf<double> d_flag;                   // [1] "a non-positive pivot somewhere", summed over the ranks
	// side streams: the updates into one target panel all go to the same stream (fixed order: deterministic), the
	// updates of one supernode into different targets and the independent subtrees of the backward solve run side by side
	enum { N_STREAMS = 8 };
	cudaStream_t side[N_STREAMS];
	std::vector<cudaEvent_t> ev_factor, ev_target, ev_x;
	SupernodalChol() : valid(false), mode(0), n(0), n_rinv_blocks(0), n_s_blocks(0), max_part(0), selinv_flops(0),
		selinv_main_doubles(0), selinv_lane_doubles(0), factor_flops(0),
		factor_flops_total(0), sym_world(0), sym_rank(0), sym_kept(false), distributed(false)
	{
		for(int i = 0; i < N_STREAMS; ++ i) side[i] = 0;
	}
};

struct DenseChol {
	DBuf<double> work;        // inverse diagonal blocks, [n_blk][128 x 128]
	DBuf<int> info;           // [0] first non-positive pivot (1-based), [1..] block-row flags of the backsolve
	cudaStream_t bulk_stream; // trailing updates that overlap the next panel
	cudaStream_t row_stream;  // look-ahead update of the next panel's tile row
	cudaEvent_t ev_potrf[2], ev_first[2], ev_panel[2], ev_bulk[2], ev_row[2];
	// persistent dataflow factorisation (chol_dataflow.cuh)
	DBuf<int> df_flags;       // task / role counters, watchdog, tile flags (zeroed before every launch)
	struct DfTaskList { DBuf<uint32_t> codes; size_t n_tasks; DfTaskList() : n_tasks(0) {} };
	std::map<uint64_t, DfTaskList> df_tasks; // worker task lists by panel shape (panels << 32 | half-tile columns): built once per shape
	size_t df_nb, df_njh, df_n_tasks;
	CUtensorMap df_maps[5];   // TMA descriptors of (df_A, df_ld, df_cols) and df_Rinv
	const void *df_A, *df_Rinv;
	size_t df_ld, df_cols;
	int n_sms;
	DenseChol() : bulk_stream(0), row_stream(0), df_nb(0), df_njh(0),
		df_n_tasks(0), df_A(0), df_Rinv(0), df_ld(0), df_cols(0), n_sms(0) {}
};

} // namespace spp

// phases of one LM iteration; in asynchronous mode (the LM loop) their event pairs are recorded without host
// synchronisation and read after the one synchronisation of the iteration
enum { PH_LINEARISE = 0, PH_SCHUR, PH_FACTOR, PH_BACKSUBST, PH_UPDATE, PH_CHI2, PH_CHOL_KERNEL /* inside PH_FACTOR */, PH_COUNT };

struct spp_ctx {
	int device;
	bool async_mode;            // no host synchronisation inside the stages (the LM loop synchronises once per iteration)
	int *async_info;            // pinned slot that receives the factorisation status in asynchronous mode
	cudaEvent_t phase_ev[PH_COUNT][2];
	bool phase_used[PH_COUNT];
	cudaStream_t stream;
	cudaStream_t copy_stream;   // host-to-device copies that overlap the symbolic analysis (created on first use)
	cudaEvent_t copy_done;
	std::string last_error;
	std::string description;
	uint64_t n_launches;
	spp_allreduce_fn allreduce;
	void *allreduce_user;
	void *nccl_comm;            // ncclComm_t created by spp_set_nccl (the library's own NCCL path); 0: the hook is used
	int rank, world;
	spp::SchurSystem sys;
	spp::BAProblem ba;
	spp::SchurSlot slot;
	spp::DenseChol chol;
	spp::SymbolicScratch sym;
	spp::SparseChol schol;
	spp::SupernodalChol snode;
	spp::PoseProblem pose;
	spp::HPinned<double> h_scalars;
	cudaEvent_t ev[16];
};

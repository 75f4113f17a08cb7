// phb_ctx.cuh -- device context shared by the kernel translation units (internal).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "phb_cuda.h"

struct phbc_ctx {
	int device, T, N, S, C, P, root, tip_kind;
	cudaStream_t stream;
	int num_sms;
	size_t smem_optin, smem_sm;  // dynamic shared memory one CTA may ask for / shared memory of one SM

	// inputs
	uint8_t *d_tip_states;   // [T][P]
	double *d_tip_partials;  // [T][P][S]
	double *d_weights;       // [P]
	double *d_evec, *d_eval, *d_ivec;  // eigen system
	double *d_qmat;          // [S][S] Q = V diag(eval) V^-1 (rate matrix, for dP = Q P)
	double *d_freqs, *d_rates, *d_props;
	double *d_bl;            // [bl_cap][N]
	double *h_bl;            // pinned staging
	int bl_cap;
	bool have_eigen;
	double *d_ex, *h_ex;     // [N][C][S] host-computed exp(eval * t) of the branch lengths uploaded last (61-state parity), pinned staging
	int ex_cap, ex_count;    // samples the buffers hold / samples whose exponentials belong to the branch lengths uploaded last

	// node-at-a-time state
	double *d_P, *d_dP;      // [N][C][S*S]
	double *d_lower;         // [N-T][C][P][S]
	double *d_upper;         // [N][C][P][S]   (lazy)
	double *d_sf;            // [2N][P]        (lazy)
	bool lower_is_message;   // d_lower holds M_n = P_n L_n instead of L_n (tensor-core message form; the root's entry is L_root either way)
	double *d_dmma_img;      // packed matrix images of the tensor-core path [P | dP][N][C][IMG]
	size_t dmma_img_bytes;
	phbc_op *d_lower_ops, *d_upper_ops;
	phbc_op *d_sub_ops;      // op list of a partial re-evaluation (phbc_run_ops)
	int sub_ops_cap;
	double *d_branch;        // single-branch scratch: candidate lengths, matrices, per-CTA sums, results (phb_branch.cu)
	size_t branch_bytes;
	phbc_parent_op *d_parent_ops;
	int n_lower_ops, n_upper_ops, n_parent_ops;
	int *h_lower_level_off, *h_upper_level_off, *h_parent_level_off;
	int *h_lower_kind_off, *h_parent_kind_off;  // [levels][4]: within a level the device op lists are sorted by the number of tip children (0, 1, 2)
	int n_lower_levels, n_upper_levels;

	// fused walk state (phb_nuc4.cu)
	phbc_post_op *d_post_ops;
	phbc_pre_op *d_pre_ops;
	int n_post, n_pre, post_slots, pre_slots;
	int *d_post_tip_order, *d_pre_tip_order;    // [T]
	int post_first_tips, pre_first_tips;
	double *d_walk_mats;     // schedule-ordered transition matrices
	double *d_walk_lower;    // per-CTA lower-partial scratch
	double *d_walk_gacc;     // per-CTA gradient accumulators
	size_t walk_lower_bytes, walk_gacc_bytes, walk_mats_bytes;
	uint8_t *d_nuc4_codes;   // [2][tiles][T][PB] tip codes in post- and pre-order walk order
	int *d_nuc4_bad;
	bool nuc4_codes_valid, nuc4_codes_bad;
	double *d_nuc4_cta_lnl;
	int nuc4_grid;
	double *d_walk_gstat;    // per-(CTA, warp) expected-transition statistics [grid][warps][N][16] (GRAD = 2 walks)
	size_t walk_gstat_bytes;
	double *d_nuc4_G;        // [N][C][16] summed statistics; the root's entry holds the root term of the frequency gradient
	bool nuc4_G_valid;       // d_nuc4_G belongs to the current inputs (cleared by every other evaluation)
	double *d_walk_hacc;     // per-(CTA, warp) Hessian-diagonal rows [grid][warps][N] (GRAD = 3 walks)
	size_t walk_hacc_bytes;
	double *d_nuc4_hess;     // [N] summed Hessian diagonal of the last GRAD = 3 walk
	double *h_freqs, *h_qmat;  // host copies of small model constants (kernel parameter bank)

	// outputs
	double *d_pattern_lnl;   // [P]
	double *d_result;        // [result_cap][1+N]
	int result_cap;
	double *h_result;        // pinned host copy of the result slots
	size_t h_result_cap;
	double *d_cat_grad;      // [cat_grad_cap][N][C]
	int cat_grad_cap;
	double *d_reduce, *h_reduce;  // [N + 2] operand of a sharded evaluation's all-reduce: lnL, grad[N], inf flag (+ pinned host copy)
	double *d_scratch;       // reduction scratch
	double *d_rowmax;        // [op slot][C][n-split][P] row maxima left by the tensor-core kernels of a rescaled pass (phb_dmma.cu)
	size_t rowmax_bytes;
	int *d_upper_slot;       // [N] child -> 2 x (its parent's index within the sorted level of d_parent_ops) + (child is b)
	size_t scratch_bytes;

	// time-tree chain (phb_timetree.cu)
	double *d_tt_lowers;     // [N]
	int *d_tt_topo;          // parent[N] | preorder[N] | postorder[N]
	int *d_tt_bad;
	double *d_tt_ratios, *d_tt_rates, *d_tt_heights, *d_tt_adj, *d_tt_out;
	double *h_tt;            // pinned staging
	int tt_cap;

	int tune;                // kernel-geometry variant of the tensor-core message kernels (PHB_OPT_TUNE; 0 = shipped)
	int last_family;         // kernels of the last evaluation: 1 generic node-at-a-time, 2 fused 4-state walk, 3 FP64 tensor-core
	int dmma_pack_adjoint, dmma_pack_irf;  // how the dP images of internal nodes were packed last (phbc_download_matrices undoes it)
	uint8_t *d_enc_states;   // [T][P] 0/1 tip partials encoded as states for the message-form kernels (lazily; valid until the next tip upload)
	bool enc_states_valid, enc_states_bad;
	double *d_cherry_tab;    // [cherry ops of a launch][C][(S + 1)^2][S] messages of the state pairs (phb_dmma.cu, k_dmma_cherry_gather)
	size_t cherry_tab_bytes;
	phbc_op *d_cherry_ops;   // the launch's cherry ops re-pointed at the enumerated pairs
	int cherry_ops_cap;
	double *d_cherry_pairmax;  // rescaling: [cherry ops of a launch][C][(S + 1)^2] largest entry of the pair's L_n
	size_t cherry_pairmax_bytes;
	uint8_t *d_cherry_enum;  // [2][(S + 1)^2] the pairs as two rows of tip states
	int dmma_pack_tips;      // tips were packed as transposed gather images (2: derivative images frequency-weighted)

	// whole-tree tensor-core walk (phb_dwalk.cu)
	void *d_dw_post, *d_dw_pre;  // walk descriptors with global tip positions (DwPost / DwPre)
	int dw_nops;
	uint8_t *d_dw_codes;     // [2][tiles][T][TP] tip codes in post- / pre-order walk order, tile-major (one bulk copy per tip operand and tile)
	size_t dw_codes_bytes;
	int dw_codes_tp;         // patterns per tile the codes were laid out for (0: not valid)
	bool dw_codes_bad;       // tip partials that are not 0/1 vectors of a single state (or all ones): the walk declines
	int *d_dw_bad;
	double *d_dw_spill;      // [spilled slots][C][P][S] upper partials parked beyond the shared-memory slots
	size_t dw_spill_bytes;
	long long launches;
	long long node_evals;    // full evaluations that rewrote the node-at-a-time buffers (generic / tensor-core paths)

	// optional event timing of the dominant kernel(s)
	bool timing;
	cudaEvent_t *ev_beg, *ev_end;
	int ev_count, ev_cap;
	double timed_ms;
	long long timed_launches;
};

int phbc_time_begin(phbc_ctx *ctx);
int phbc_time_end(phbc_ctx *ctx);

extern thread_local char phbc_errbuf[512];

#define PHBC_CHECK(call)                                                                                     \
	do {                                                                                                     \
		cudaError_t e__ = (call);                                                                            \
		if (e__ != cudaSuccess) {                                                                            \
			snprintf(phbc_errbuf, sizeof(phbc_errbuf), "%s:%d: %s: %s", __FILE__, __LINE__, #call,          \
			         cudaGetErrorString(e__));                                                               \
			return -2;                                                                                       \
		}                                                                                                    \
	} while (0)

int phbc_ensure_scratch(phbc_ctx *ctx, size_t bytes);

// generic node-at-a-time path (phb_cuda.cu)
int phbc_generic_evaluate(phbc_ctx *ctx, const phbc_eval_opts *o);
// pieces of it shared with the tensor-core path (same buffers, same schedules)
struct Bufs {
	const uint8_t *tip_states;
	const double *tip_partials;
	double *lower;
	double *upper;
	double *sf;
	int T, N, S, C, P, tip_kind;
};
Bufs phbc_make_bufs(phbc_ctx *ctx);
int phbc_generic_prepare(phbc_ctx *ctx, const phbc_eval_opts *o);                       // buffers + transition matrices
int phbc_generic_buffers(phbc_ctx *ctx, const phbc_eval_opts *o);                       // buffers only (lazy)
int phbc_generic_scale_ops(phbc_ctx *ctx, const phbc_op *d_ops, int count, double threshold);  // K5 on one level
int phbc_generic_root(phbc_ctx *ctx, const phbc_eval_opts *o, double *result);           // K6, K7 -> result[0]
int phbc_generic_gradient(phbc_ctx *ctx, const phbc_eval_opts *o, double *result);       // K9, K10, A11 from materialised uppers
int phbc_gradient_from_partials(phbc_ctx *ctx, int tiles, double *result);               // cat_grad = sum of [N][C][tiles] scratch, A11
// FP64 tensor-core path, 20 / 61 states (phb_dmma.cu)
int phbc_dmma_evaluate(phbc_ctx *ctx, const phbc_eval_opts *o);
int phbc_dmma_matrix_gradient(phbc_ctx *ctx, const phbc_eval_opts *o, int nsets, const double *d_M, double *d_cat);  // node terms of calculate_dlnl_dQ, [nsets][N][C]
bool phbc_dmma_supported(const phbc_ctx *ctx, const phbc_eval_opts *o);
int phbc_dmma_pack(phbc_ctx *ctx);                                   // packed matrix images from d_P / d_dP
int phbc_dmma_lower_ops(phbc_ctx *ctx, const phbc_op *d_ops, int cnt);  // out = (P_a x_a) o (P_b x_b) for a device op list (one level)
// whole-tree walk on the FP64 tensor cores, 20 states (phb_dwalk.cu)
int phbc_dwalk_set_schedule(phbc_ctx *ctx, const phbc_schedule *s);
bool phbc_dwalk_supported(const phbc_ctx *ctx, const phbc_eval_opts *o);
int phbc_dwalk_usable(phbc_ctx *ctx, const phbc_eval_opts *o);                       // supported AND the tips encode as single states
int phbc_dwalk_passes(phbc_ctx *ctx, const phbc_eval_opts *o, double *result, int phases);  // 1: post-order walk + root, 2: pre-order walk + gradient sums
// fused 4-state walk path (phb_nuc4.cu)
int phbc_nuc4_evaluate(phbc_ctx *ctx, const phbc_eval_opts *o);
bool phbc_nuc4_supported(const phbc_ctx *ctx, const phbc_eval_opts *o);
int phbc_nuc4_matrix_gradient(phbc_ctx *ctx, const phbc_eval_opts *o, int nsets, const double *M_host, int skip_node, double *lnl, double *out_host);  // 1 = declined
int phbc_nuc4_root_frequency_gradient(phbc_ctx *ctx, double *out_host);
int phbc_nuc4_download_matrices(phbc_ctx *ctx, double *P, double *dP);  // what the last walk consumed, back in [N][C][4][4] form
int phbc_dmma_download_matrices(phbc_ctx *ctx, double *P, double *dP);  // the packed images, unpacked

// shared device helpers
__device__ __forceinline__ double phb_warp_sum(double v) {
#pragma unroll
	for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
	return v;
}

// generic partials addressing (node-at-a-time kernels)
__device__ __forceinline__ const double *partial_ptr(const Bufs &b, int idx, int c) {
	const size_t PS = (size_t)b.P * b.S;
	if (idx < b.T) return b.tip_partials + (size_t)idx * PS;
	if (idx < b.N) return b.lower + ((size_t)(idx - b.T) * b.C + c) * PS;
	return b.upper + ((size_t)(idx - b.N) * b.C + c) * PS;
}

__device__ __forceinline__ bool is_state_tip(const Bufs &b, int idx) { return idx < b.T && b.tip_kind == PHBC_TIP_STATES; }

// The dividing half of the rescaling kernels that decide with one thread per (pattern, category): m_s[k] is the maximum of pattern
// p0 + k where it is rescaled and 0 where it keeps its values.  A category's rows of consecutive patterns are contiguous, so the block
// sweeps them with coalesced accesses instead of each thread walking its own 8 S-byte row (that walk made the rescaling of upper
// partials, which happens at most levels, 11 of the 30 ms of a rescaled LG+G4 400 x 50k evaluation).  Same division, same values.
__device__ __forceinline__ void phbc_rescale_block(const Bufs &b, int out, int p0, int np, const double *m_s) {
	const int S = b.S, n = (np < b.P - p0 ? np : b.P - p0) * S;
	for (int c = 0; c < b.C; c++) {
		double *x = (double *)partial_ptr(b, out, c) + (size_t)p0 * S;
		for (int e = threadIdx.x; e < n; e += blockDim.x) {
			const double m = m_s[e / S];
			if (m > 0.0) x[e] /= m;
		}
	}
}

// message_i = sum_j M[i][j] x[j]; state tips gather a column, unknown states give 1 for probability
// matrices and the real row sum for derivative matrices (treelikelihoodX.c:166-289, 878-1001).
__device__ __forceinline__ double message(const Bufs &b, int idx, int c, const double *M, int p, int i, bool prob) {
	const int S = b.S;
	if (is_state_tip(b, idx)) {
		const int s = b.tip_states[(size_t)idx * b.P + p];
		if (s < S) return M[i * S + s];
		if (prob) return 1.0;
		double acc = 0.0;
		for (int j = 0; j < S; j++) acc += M[i * S + j];
		return acc;
	}
	const double *x = partial_ptr(b, idx, c) + (size_t)p * S;
	double acc = 0.0;
	for (int j = 0; j < S; j++) acc += M[i * S + j] * x[j];
	return acc;
}

// ---------------------------------------------------------------------------------------------
// PTX helpers: mbarrier + TMA bulk copy (global -> shared)
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
	asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
	asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar) {
	asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
	             "l"(src), "r"(bytes), "r"(smem_u32(bar))
	             : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
	uint32_t done;
	do {
		asm volatile(
		    "{\n"
		    ".reg .pred p;\n"
		    "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
		    "selp.u32 %0, 1, 0, p;\n"
		    "}\n"
		    : "=r"(done)
		    : "r"(smem_u32(bar)), "r"(parity)
		    : "memory");
	} while (!done);
}
__device__ __forceinline__ void red_add_f64(double *addr, double v) {
	asm volatile("red.global.add.f64 [%0], %1;" ::"l"(addr), "d"(v) : "memory");
}


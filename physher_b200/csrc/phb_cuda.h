/*
 * phb_cuda.h -- thin C-ABI layer between the C host code (phb_treelikelihood.c) and the sm_100a
 * kernels (phb_cuda.cu, phb_nuc4.cu, phb_dmma.cu).  Internal: the public ABI is include/physher_b200.h.
 *
 * The host side owns all control flow (dirty flags, caching, schedules, gradient assembly); this
 * layer owns device memory, the stream and the kernel launches.  No torch types anywhere.
 */
#ifndef PHB_CUDA_H
#define PHB_CUDA_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct phbc_ctx phbc_ctx;

/* tip representations on the device */
#define PHBC_TIP_STATES 0   /* uint8 [T][P]; >= S unknown                                         */
#define PHBC_TIP_PARTIALS 1 /* double [T][P][S] (category stride 0)                               */

/*
 * One partial-update op of the node-at-a-time ("generic") kernels; mirrors the reference's
 * update_partials(tlk, out, p1, m1, p2, m2) (treelikelihood.h:91): out = (M[m1] x[p1]) o (M[m2] x[p2]).
 * Buffer indices: < T tip, T..N-1 lower partials, N + node upper partials.  b < 0: single child.
 */
typedef struct phbc_op {
	int out;
	int a, a_mat;
	int b, b_mat;
	int flags; /* bit 0: multiply the result by the root frequencies (treelikelihood.c:2148-2153) */
} phbc_op;

/* Whole-tree walk schedules of the fused 4-state kernels (see phb_nuc4.cu). Ops are consumed in chunks of
 * PHBC_WALK_CHUNK (one TMA stage); tip operands are numbered in walk order so that the tip codes a chunk
 * needs are one contiguous range [chunk_tip0[ch], chunk_tip0[ch+1]) of a walk-ordered code array, and the
 * descriptors carry indices local to that range.  Operand kinds: */
#define PHBC_WALK_CHUNK 6
#define PHBC_W_TIP 0  /* idx = tip node id                                  */
#define PHBC_W_SLOT 1 /* idx = shared-memory slot                           */
#define PHBC_W_ROOT 2 /* pre-order only: the parent is the root (W = 1 or pi) */
#define PHBC_W_REG 3  /* the value is still in the registers of the preceding op   */
/* Cherry recomputation (unscaled gradient walks): the message M_b = P_b (m_a' o m_b') of a cherry b -- an internal node whose children
 * are both tips -- costs 24 FP64 operations to rebuild from its tips' matrix columns, against a 32-byte row written by the post-order
 * pass and read back by the pre-order pass per (pattern, category).  When b's pre-order op directly follows its parent's (it is the
 * parent's child b), the parent's op forms the two tip messages from the NEXT op's staged matrices and codes, leaves them in the
 * registers that op will read them from, and multiplies by P_b itself: the row of b is neither written nor read. */
#define PHBC_POST_NO_ROW 0x100   /* phbc_post_op.a_kind flag: the node's message row is not needed (recomputed by its parent's pre-order op) */
#define PHBC_PRE_B_RECOMPUTE 1   /* phbc_pre_op.flags: child b is a cherry and its op is the next one: rebuild M_b instead of loading b_row */
#define PHBC_PRE_TIPS_READY 2    /* phbc_pre_op.flags: this (tip-tip) op finds its two tip messages in registers, left by the preceding op */

typedef struct phbc_post_op { /* one internal node, DFS post-order; 32 bytes (TMA bulk-copy granule)   */
	int16_t a_kind, b_kind;  /* a tip child always comes first: kind = a_kind + b_kind in {0 tip-tip, 1 tip-internal, 2 internal-internal} */
	int a_idx, b_idx;        /* slot, or chunk-local index of the tip operand's code row           */
	int a_node, b_node;      /* node ids of the children (matrix owners)                          */
	int dst_slot;            /* slot receiving the result                                         */
	int node;                /* node id of the result; its lower-scratch row is the op's own index */
	int next_tips;           /* first op of a chunk: (first tip index << 5 | tip count) of the NEXT chunk */
} phbc_post_op;

#define PHBC_PF_DIST 3 /* L2 prefetch distance of the pre-order walk, in ops */
typedef struct phbc_pre_op { /* one internal node acting as parent, DFS pre-order; 48 bytes         */
	int16_t u_kind;          /* PHBC_W_SLOT, PHBC_W_REG or PHBC_W_ROOT                            */
	int16_t kind;            /* 0 tip-tip, 1 tip-internal (the tip is child a), 2 internal-internal */
	int next_tips;           /* as in phbc_post_op                                                */
	int16_t u_slot;          /* slot holding U_parent                                             */
	int16_t a_slot, b_slot;  /* slots receiving U_a / U_b for internal children (-1: not kept)    */
	int16_t a_code, b_code;  /* chunk-local index of a tip child's code row                       */
	int16_t flags;           /* PHBC_PRE_* (honoured by the unscaled gradient walk only)           */
	int node;                /* parent node id (matrix P_node when not the root)                  */
	int a_node, b_node;      /* children node ids                                                 */
	int a_row, b_row;        /* lower-scratch rows (post-order op index) of internal children     */
	int pf_a_row, pf_b_row;  /* a_row / b_row of the op PHBC_PF_DIST positions later (-1: none): L2 prefetch targets */
} phbc_pre_op;

/* One pre-order op of the tensor-core kernels: internal node `node` with children a, b.  The kernel turns
 * U_node (or the root message) into U_a, U_b and both branch-gradient terms.  Grouped by depth of `node`. */
typedef struct phbc_parent_op {
	int node, a, b;
	int flags; /* bit 0: node is the root */
} phbc_parent_op;

typedef struct phbc_schedule {
	int n_lower_ops, n_lower_levels;
	const phbc_op *lower_ops;   /* grouped by level, children before parents                      */
	const int *lower_level_off; /* [n_lower_levels + 1]                                           */
	int n_upper_ops, n_upper_levels;
	const phbc_op *upper_ops;   /* grouped by depth, parents before children                      */
	const int *upper_level_off;
	int n_parent_ops;                 /* internal nodes grouped by their own depth (root first)  */
	const phbc_parent_op *parent_ops;
	const int *parent_level_off;      /* [n_upper_levels + 1]: level d = parents at depth d       */
	int n_post, n_pre;
	const phbc_post_op *post_ops;
	const phbc_pre_op *pre_ops;
	int post_slots, pre_slots;  /* shared-memory slots the walks need                             */
	const int *post_tip_order;  /* [T] tip node ids in the order the post-order walk consumes them */
	const int *pre_tip_order;   /* [T] same for the pre-order walk                                 */
	int post_first_tips, pre_first_tips; /* tip count of chunk 0 of each walk (its first index is 0)  */
} phbc_schedule;

int phbc_device_count(void);
const char *phbc_last_error(void);

phbc_ctx *phbc_create(int device, int ntips, int nstate, int ncat, int npatterns, int root, int tip_kind);
void phbc_destroy(phbc_ctx *ctx);

int phbc_set_schedule(phbc_ctx *ctx, const phbc_schedule *s);
int phbc_set_root(phbc_ctx *ctx, int root); /* with a new schedule: topology moves */
int phbc_upload_tip_states(phbc_ctx *ctx, const uint8_t *states);
int phbc_upload_tip_partials(phbc_ctx *ctx, const double *partials);
int phbc_upload_weights(phbc_ctx *ctx, const double *w);
int phbc_upload_eigen(phbc_ctx *ctx, const double *evec, const double *eval, const double *ivec);
int phbc_upload_matrices(phbc_ctx *ctx, const double *P, const double *dP);
int phbc_upload_freqs(phbc_ctx *ctx, const double *freqs);
int phbc_upload_site_model(phbc_ctx *ctx, const double *rates, const double *props);
int phbc_upload_branch_lengths(phbc_ctx *ctx, const double *bl, int nbatch); /* [nbatch][N], pinned staging */
int phbc_upload_exponentials(phbc_ctx *ctx, const double *ex, int nbatch); /* [nbatch][N][C][S] exp(eval * bl * rate) from the host's libm, for the vectors uploaded last */
int phbc_download_branch_lengths(phbc_ctx *ctx, int nbatch, double *bl); /* [nbatch][N] as the device holds them */
/* device-to-device copy of the bulky inputs (tips, weights, explicit matrices, time-tree tables) between same-shaped contexts */
int phbc_copy_inputs(phbc_ctx *dst, phbc_ctx *src, int matrices, int time_tree);

typedef struct phbc_eval_opts {
	int kernels;                 /* PHB_KERNELS_*                                                  */
	int scale;                   /* rescaling on                                                   */
	double scaling_threshold;
	int include_root_freqs;
	int compat_scaled_gradient;
	int want_gradient;           /* 0 lnL, 1 + branch gradients, 2 + transition statistics, 3 + Hessian diagonal (fused 4-state walk only) */
	int explicit_matrices;       /* matrices were uploaded, do not rebuild them from the eigen system */
	int batch_index;             /* which uploaded branch-length vector (the first one of a batch)  */
	int materialize_uppers;      /* tensor-core path: store every upper partial (tips included) and reduce with the generic K9/K10 */
	int batch_count;             /* > 1: evaluate batch_index .. batch_index + batch_count - 1 (results in the matching slots) */
} phbc_eval_opts;

/*
 * One evaluation, asynchronous on the ctx stream: transition matrices, post-order pass, root
 * integration, and (want_gradient) the pre-order pass with the branch-gradient reductions.
 * Results stay on the device: result[0] = lnL, result[1..N] = d lnL / d bl by node id
 * (before the unrooted convention is applied), cat_grad [N][C].
 */
int phbc_evaluate(phbc_ctx *ctx, const phbc_eval_opts *o);
/* copy results of evaluation slot `batch_index` into out_device[0..N] on the stream (device to device) */
int phbc_result_to_device(phbc_ctx *ctx, int batch_index, double *out_device);
/* pattern-sharded evaluations: [lnL, grad[N], inf flag] of a result slot packed into the ctx's all-reduce operand (device pointer
 * returned, ordered on the ctx stream), and its blocking download through pinned memory */
int phbc_pack_reduce(phbc_ctx *ctx, int batch_index, double **out_device);
int phbc_download_reduce(phbc_ctx *ctx, double *host /* [N + 2] */);
/* blocking download of result slots [0, nbatch): lnl[b], grad[b][N] (either may be NULL) */
int phbc_download_results(phbc_ctx *ctx, int nbatch, double *lnl, double *grad);
int phbc_download_cat_grad(phbc_ctx *ctx, double *out);
int phbc_download_pattern_lnl(phbc_ctx *ctx, double *out);
int phbc_download_partials(phbc_ctx *ctx, int index, double *out);
int phbc_download_matrices(phbc_ctx *ctx, double *P, double *dP);
/* Partial re-evaluation on the resident node-at-a-time buffers (dirty-flag traversal, treelikelihood.c:1645-1734, 2164-2190):
 * host op list grouped by level; lower ops are followed by the root integration when do_root (lnl_host may be NULL). */
int phbc_run_ops(phbc_ctx *ctx, const phbc_eval_opts *o, int nops, const phbc_op *ops, int nlevels, const int *level_off, int rebuild_matrices,
                 int do_root, double *lnl_host);
/* d lnL / d pi_i at fixed partials from the resident root partial (root term of calculate_dlnl_dQ, treelikelihood.c:2371-2404) */
int phbc_root_frequency_gradient(phbc_ctx *ctx, double *out /* [S] */);
/* d lnL / d prop_c at fixed conditional likelihoods, from the same root partial (root term of gradient_pinv_sitemodel, treelikelihood.c:2943-3001) */
int phbc_root_category_gradient(phbc_ctx *ctx, double *out /* [C] */);
/* the node-at-a-time buffers, allocated lazily (zero-filled): lowers, uppers with want_gradient, scale factors with scale; -3 when the
 * device cannot hold them */
int phbc_generic_buffers(phbc_ctx *ctx, const phbc_eval_opts *o);
/* K9 / K10 / A11 over every branch from resident upper and lower partials (results in slot 0; lnL slot untouched) */
int phbc_resident_gradient(phbc_ctx *ctx, const phbc_eval_opts *o);
/* single-branch fast path (phb_branch.cu) on resident upper / lower partials: out [nitems][3] = lnL, d lnL/dt, d2 lnL/dt2 of the branch
 * above nodes[k] at length bl[k] -- one node repeated (candidate lengths) or every non-root node at its own length (Hessian diagonal) */
/* ex (may be NULL): [nitems][C][S] exp(eval * bl * rate) from the host's libm */
int phbc_branch_lnl(phbc_ctx *ctx, const phbc_eval_opts *o, int nitems, const int *nodes, const double *bl, const double *ex, double *out);
/* lnL, d lnL / d bl [N] and d2 lnL / d bl2 [N] (exact form, root entries 0, no unrooted convention) from ONE unscaled fused 4-state
 * walk (want_gradient = 3, phb_nuc4.cu); grad may be NULL.  Returns 1 (declined, nothing done) when the walk cannot serve the request:
 * not 4 states, a shape phbc_nuc4_supported refuses, rescaling, PHB_KERNELS_GENERIC, tip partials that are not 0/1 vectors, a batch. */
int phbc_nuc4_hessian(phbc_ctx *ctx, const phbc_eval_opts *o, double *lnl, double *grad, double *hess);
/* One nearest-neighbour interchange (phb_nni.cu): x and y exchanged across the branch above v = parent[y].  Buffer indices as in
 * phbc_op; matrix indices are entries of the call's matrix table (node n at its current length = entry n, move k's central length =
 * entry N + k). */
typedef struct phbc_nni_move {
	int x, y, keep; /* the exchanged subtrees and the child of v that stays                                          */
	int a, a_mat;   /* second factor of the upper side: N + p (U_p, matrix P_p) for an NNI below p, the child of w that stays
	                   for one across the root, a = -1 (a vector of ones) when p is the root                            */
	int w;          /* across the root: the root child w whose matrix closes the upper side; -1 otherwise               */
	int cmat;       /* table entry of the central branch (P, P', P")                                                   */
	int out;        /* output row                                                                                      */
} phbc_nni_move;
/* out [nmoves][3] = lnL, d lnL/dt_v, d2 lnL/dt_v2 of each exchanged tree from resident upper / lower partials; bl [N + nmoves] the matrix
 * table's lengths, ex (may be NULL) their exponentials [N + nmoves][C][S]; groups [ngroups][2] move pairs sharing (v, x), -1 = none
 * (the 4-state kernel's work items) */
int phbc_nni_scores(phbc_ctx *ctx, const phbc_eval_opts *o, int nmoves, const phbc_nni_move *moves, int ngroups, const int *groups,
                    const double *bl, const double *ex, double *out);
/* Subtree prune and regraft (phb_spr.cu): out [ntargets][3] = lnL, d lnL/dt_s, d2 lnL/dt_s2 of the subtree of s (p = parent[s])
 * regrafted on the branch above each target node, from the pruned tree's partials the caller left in the resident buffers (U~_e at
 * N + e, L~_e at e); bl [N + ntargets] the matrix table's lengths (node n = entry n, target k's pendant length = entry N + k), ex (may
 * be NULL) their exponentials [N + ntargets][C][S]. */
/* the call's matrix table and sums, allocated before the pruned pass changes anything: -1 when the state count needs more shared
 * memory than a CTA may have, -3 when the device cannot hold them */
int phbc_spr_reserve(phbc_ctx *ctx, int ntargets);
int phbc_spr_scores(phbc_ctx *ctx, const phbc_eval_opts *o, int s, int p, int ntargets, const int *targets, const double *bl, const double *ex,
                    double *out);
int phbc_matrix_gradient(phbc_ctx *ctx, const phbc_eval_opts *o, int nsets, const double *M_host, int skip_node, double *lnl, double *out_host);
/* time-tree chain, batched (phb_timetree.cu) */
int phbc_set_time_tree(phbc_ctx *ctx, const double *lowers, const int *parent, const int *preorder, const int *postorder);
int phbc_time_forward(phbc_ctx *ctx, int nbatch, const double *ratios, const double *rates, int nrates); /* 1: negative branch length */
int phbc_time_backward(phbc_ctx *ctx, int nbatch, int nrates, int include_jacobian, int want_gradient, double *lnl, double *logjac,
                       double *grad_ratios, double *grad_rates);
int phbc_synchronize(phbc_ctx *ctx);
void *phbc_stream(phbc_ctx *ctx);
long long phbc_launch_count(const phbc_ctx *ctx);
int phbc_last_family(const phbc_ctx *ctx); /* 1 generic, 2 fused walk, 3 tensor cores; 0 before the first evaluation */
long long phbc_node_eval_count(const phbc_ctx *ctx); /* full evaluations that rewrote the node-at-a-time partials buffers */
int phbc_set_timing(phbc_ctx *ctx, int on);
int phbc_set_tune(phbc_ctx *ctx, int variant); /* geometry variant of the tensor-core message kernels (profiling; 0 = shipped) */
int phbc_kernel_time(phbc_ctx *ctx, double *total_ms, long long *launches);

#ifdef __cplusplus
}
#endif
#endif

/*
 * phb_treelikelihood.c -- host side of the B200 tree likelihood, in C like the reference's host code.
 *
 * Mirrors the control flow of src/phyc/treelikelihood.c: construction (new_SingleTreeLikelihood,
 * :1007-1185), dirty flags and caching (_calculate_simple :1454-1526, update_* :1737-1771),
 * NaN / inf handling with the automatic switch to rescaling (:1489-1519), gradient entry points
 * (TreeLikelihood_initialize_gradient :237-318, TreeLikelihood_gradient :320-340) and the unrooted
 * convention (:3249-3255).  All numerics run on the device through the thin layer in phb_cuda.h;
 * this file contains no arithmetic on partials.
 *
 * It also turns the tree into the launch schedules the kernels consume:
 *   - level lists for the node-at-a-time kernels (children before parents / parents before children);
 *   - linear whole-tree walks for the fused kernels: a post-order walk ordered so that the number of
 *     live intermediate partials is the tree's Strahler number (larger-need child first) and a
 *     pre-order walk with the same property, each with its shared-memory slot assignment.
 */
#include "../../include/physher_b200.h"
#include "phb_cuda.h"

#include <math.h>
#include <nvtx3/nvToolsExt.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

struct phb_tlk {
	int T, N, S, C, P, root;
	int use_tip_states, device;
	int *left, *right, *parent;
	double *bl; /* [N] host copy, as Node_distance would return */
	phbc_ctx *ctx;

	/* tlk->update_nodes / update / update_upper (treelikelihood.h:79-80,114) */
	unsigned char *update_nodes;
	int update, update_upper;

	int scale; /* tlk->scale */
	double scaling_threshold;
	int include_root_freqs, compat_scaled_gradient, unrooted, kernels;

	int have_tips, have_weights, have_eigen, have_matrices, have_freqs, have_site, have_bl;
	int bl_dirty;

	double lk; /* tlk->lk */
	int prepared_gradient;
	double *gradient; /* owned, like tlk->gradient */
	size_t gradient_length;
	int gradient_valid;

	/* schedules (host copies kept for introspection) */
	phbc_op *lower_ops, *upper_ops;
	phbc_parent_op *parent_ops;
	int *lower_level_off, *upper_level_off, *parent_level_off;
	phbc_post_op *post_ops;
	phbc_pre_op *pre_ops;
	int n_lower_levels, n_upper_levels, post_slots, pre_slots;
	int *post_tip_order, *pre_tip_order, *post_chunk_tip0, *pre_chunk_tip0;
	int post_first_tips, pre_first_tips;
	int have_time_tree;
	int host_exp;  /* exponentials of the transition matrices from the host's libm (PHB_OPT_HOST_EXPONENTIALS; default on for >= 60 states) */
	double *ex_buf; /* [samples][N][C][S] */
	size_t ex_cap;
	int sweep_valid; /* the node-at-a-time buffers hold a full evaluation of the current inputs (phb_tlk_matrix_gradient) */

	/* resident node-at-a-time partials (PHB_OPT_INCREMENTAL): which device buffers hold values of the CURRENT inputs */
	int incremental, resident, all_dirty;
	int lower_stale;                    /* some lower_ok entries are 0 although update is clear (a fused gradient call consumed the dirty flags) */
	unsigned char *lower_ok, *upper_ok; /* [N] */
	int upper_irf;                      /* include_root_freqs value the valid uppers were built with */
	int *upper_op_of;                   /* [N] index into upper_ops */
	phbc_op *sub_ops;                   /* [2N] scratch op list */
	int *sub_level_off;                 /* [N + 2] */
	int *path;                          /* [N] scratch */

	/* host mirrors of the small model inputs + the stored state of store / restore (MCMC, treelikelihood.c:116-161) */
	double *h_evec, *h_eval, *h_ivec, *h_freqs, *h_rates, *h_props;
	int has_store;
	double *st_bl, *st_evec, *st_eval, *st_ivec, *st_freqs, *st_rates, *st_props;
	double st_lk;
	int st_update, st_scale, st_have_eigen;
	int eigen_changed, freqs_changed, site_changed, bl_changed; /* since the last store */
};

static _Thread_local char g_err[512] = "";

static int fail(int code, const char *fmt, ...) {
	va_list ap;
	va_start(ap, fmt);
	vsnprintf(g_err, sizeof(g_err), fmt, ap);
	va_end(ap);
	return code;
}

static int dev_fail(int rc) { return fail(rc == -3 ? PHB_ENOMEM : (rc == -1 ? PHB_EINVAL : (rc == -4 ? PHB_ESTATE : PHB_ECUDA)), "%s", phbc_last_error()); }

const char *phb_last_error(void) { return g_err; }

/* for the other host translation unit of the library (phb_group.c); not part of the ABI */
int phb_internal_fail(int code, const char *msg) { return fail(code, "%s", msg); }
int phb_device_count(void) { return phbc_device_count(); }
/* the kernel revision tag ties committed ncu captures (profiles/traffic.json) to the kernels they were taken on */
const char *phb_version(void) { return "physher_b200 0.2 (sm_100a; walk kernels r2w, level kernels r2z)"; }

/* ------------------------------------------------------------------------------------------- */
/* schedules                                                                                   */
/* ------------------------------------------------------------------------------------------- */

static int is_tip(const phb_tlk *t, int n) { return t->left[n] < 0; }

/* level lists: lower level = 1 + max(children levels) (tips 0); upper level = depth below the root */
static int build_level_schedules(phb_tlk *t) {
	const int N = t->N, T = t->T;
	int rc = PHB_OK;
	int *level = (int *)calloc(N, sizeof(int));
	int *depth = (int *)calloc(N, sizeof(int));
	int *order = (int *)malloc(sizeof(int) * N); /* pre-order */
	int *stack = (int *)malloc(sizeof(int) * (2 * (size_t)N + 2));
	int *fill = (int *)malloc(sizeof(int) * ((size_t)N + 2)); /* per-level fill counters (a level count never exceeds N) */
	if (!level || !depth || !order || !stack || !fill) {
		rc = fail(PHB_ENOMEM, "out of memory");
		goto done;
	}
	int sp = 0, cnt = 0;
	stack[sp++] = t->root;
	while (sp) {
		int n = stack[--sp];
		if (cnt >= N || level[n]) { /* a node reached twice: a cycle or a shared child (phb_tlk_set_topology hands over caller data) */
			cnt = N + 1;
			break;
		}
		level[n] = 1; /* visited mark; levels are assigned below */
		order[cnt++] = n;
		if (!is_tip(t, n)) {
			depth[t->left[n]] = depth[n] + 1;
			depth[t->right[n]] = depth[n] + 1;
			stack[sp++] = t->right[n];
			stack[sp++] = t->left[n];
		}
	}
	if (cnt != N) {
		rc = fail(PHB_EINVAL, "topology is not a rooted binary tree over %d nodes (visited %d)", N, cnt);
		goto done;
	}
	memset(level, 0, sizeof(int) * N); /* drop the visited marks: tips are level 0 */
	int maxlevel = 0, maxdepth = 0;
	for (int k = N - 1; k >= 0; k--) { /* reverse pre-order: children before parents */
		int n = order[k];
		if (!is_tip(t, n)) {
			int a = level[t->left[n]], b = level[t->right[n]];
			level[n] = 1 + (a > b ? a : b);
		}
		if (level[n] > maxlevel) maxlevel = level[n];
		if (depth[n] > maxdepth) maxdepth = depth[n];
	}
	t->n_lower_levels = maxlevel;
	t->n_upper_levels = maxdepth;
	t->lower_level_off = (int *)calloc(maxlevel + 2, sizeof(int));
	t->lower_ops = (phbc_op *)malloc(sizeof(phbc_op) * (N - T > 0 ? N - T : 1));
	t->upper_level_off = (int *)calloc(maxdepth + 2, sizeof(int));
	t->upper_ops = (phbc_op *)malloc(sizeof(phbc_op) * (N > 1 ? N - 1 : 1));
	t->parent_level_off = (int *)calloc(maxdepth + 2, sizeof(int));
	t->parent_ops = (phbc_parent_op *)malloc(sizeof(phbc_parent_op) * (N - T > 0 ? N - T : 1));
	if (!t->lower_level_off || !t->lower_ops || !t->upper_level_off || !t->upper_ops || !t->parent_level_off || !t->parent_ops) {
		rc = fail(PHB_ENOMEM, "out of memory"); /* whatever was allocated is released by free_schedules / phb_tlk_free */
		goto done;
	}
	/* lower ops: internal nodes grouped by level 1..maxlevel */
	for (int n = 0; n < N; n++)
		if (!is_tip(t, n)) t->lower_level_off[level[n]]++; /* count at index level (1-based) */
	{
		int acc = 0;
		for (int l = 1; l <= maxlevel; l++) {
			int c = t->lower_level_off[l];
			t->lower_level_off[l - 1] = acc;
			acc += c;
		}
		t->lower_level_off[maxlevel] = acc;
	}
	memset(fill, 0, sizeof(int) * ((size_t)N + 2));
	for (int n = 0; n < N; n++) {
		if (is_tip(t, n)) continue;
		int l = level[n] - 1;
		phbc_op *op = &t->lower_ops[t->lower_level_off[l] + fill[l]++];
		op->out = n;
		op->a = t->left[n];
		op->a_mat = t->left[n];
		op->b = t->right[n];
		op->b_mat = t->right[n];
		op->flags = 0;
	}
	/* upper ops: every non-root node, grouped by depth 1..maxdepth (update_upper_partials, treelikelihood.c:2129-2161) */
	for (int n = 0; n < N; n++)
		if (n != t->root) t->upper_level_off[depth[n]]++;
	{
		int acc = 0;
		for (int d = 1; d <= maxdepth; d++) {
			int c = t->upper_level_off[d];
			t->upper_level_off[d - 1] = acc;
			acc += c;
		}
		t->upper_level_off[maxdepth] = acc;
	}
	memset(fill, 0, sizeof(int) * ((size_t)N + 2));
	for (int n = 0; n < N; n++) {
		if (n == t->root) continue;
		int d = depth[n] - 1;
		int parent = t->parent[n];
		int sib = t->left[parent] == n ? t->right[parent] : t->left[parent];
		phbc_op *op = &t->upper_ops[t->upper_level_off[d] + fill[d]++];
		op->out = N + n;
		if (parent != t->root) { /* u_n = (P_p u_p) o (P_s L_s) */
			op->a = N + parent;
			op->a_mat = parent;
			op->b = sib;
			op->b_mat = sib;
			op->flags = 0;
		} else { /* u_n = P_s L_s [o pi] */
			op->a = sib;
			op->a_mat = sib;
			op->b = -1;
			op->b_mat = -1;
			op->flags = 1;
		}
	}
	/* parent ops: internal nodes grouped by their own depth 0..maxdepth-1 (their children sit one level deeper) */
	for (int n = 0; n < N; n++)
		if (!is_tip(t, n)) t->parent_level_off[depth[n] + 1]++;
	for (int d = 0; d < maxdepth; d++) t->parent_level_off[d + 1] += t->parent_level_off[d];
	memset(fill, 0, sizeof(int) * ((size_t)N + 2));
	for (int n = 0; n < N; n++) {
		if (is_tip(t, n)) continue;
		const int d = depth[n];
		phbc_parent_op *op = &t->parent_ops[t->parent_level_off[d] + fill[d]++];
		op->node = n;
		op->a = t->left[n];
		op->b = t->right[n];
		op->flags = n == t->root ? 1 : 0;
	}
done:
	free(fill);
	free(level);
	free(depth);
	free(order);
	free(stack);
	return rc;
}

/* Strahler-style register need of the subtree below n (tips need none) */
static void compute_need(const phb_tlk *t, int *need, int *size, int *stack /* [6N + 8] scratch of the caller */) {
	/* node ids are not guaranteed to be a post-order: iterate with an explicit stack */
	int sp = 0;
	stack[sp++] = t->root;
	stack[sp++] = 0;
	while (sp) {
		int state = stack[--sp];
		int n = stack[--sp];
		if (is_tip(t, n)) {
			need[n] = 0;
			size[n] = 1;
			continue;
		}
		if (state == 0) {
			stack[sp++] = n;
			stack[sp++] = 1;
			stack[sp++] = t->left[n];
			stack[sp++] = 0;
			stack[sp++] = t->right[n];
			stack[sp++] = 0;
		} else {
			int a = need[t->left[n]], b = need[t->right[n]];
			need[n] = a == b ? a + 1 : (a > b ? a : b);
			size[n] = 1 + size[t->left[n]] + size[t->right[n]];
		}
	}
}

typedef struct SlotPool {
	unsigned char *used;
	int cap, high;
} SlotPool;

static int slot_alloc(SlotPool *p) {
	for (int s = 0; s < p->cap; s++)
		if (!p->used[s]) {
			p->used[s] = 1;
			if (s + 1 > p->high) p->high = s + 1;
			return s;
		}
	return -1;
}

/*
 * Whole-tree walks for the fused kernels.
 *
 * Post-order: children commute in the product, so every op is normalised to one of three kinds
 *   0 tip-tip        (a tip, b tip)
 *   1 tip-internal   (a tip, b = the result of the IMMEDIATELY preceding op, still in registers)
 *   2 internal-int.  (a = an earlier result parked in a slot, b = the preceding op's result)
 * A result is parked in a shared-memory slot only when it is the first-visited child of a kind-2 parent;
 * visiting the child with the larger register need first keeps the number of live slots at the tree's
 * Strahler number.
 *
 * Pre-order over internal nodes (each op turns U_parent into U for both children and their branch
 * gradients): same three kinds; child b (when internal) is the node whose op comes NEXT, so its U stays in
 * registers; child a of a kind-2 op is parked in a slot until its own op comes up.
 */
static int build_walk_schedules(phb_tlk *t) {
	const int N = t->N, T = t->T;
	const int nint = N - T;
	int rc = PHB_OK;
	int *need = (int *)malloc(sizeof(int) * N);
	int *size = (int *)malloc(sizeof(int) * N);
	int *slot_of = (int *)malloc(sizeof(int) * N);
	int *row_of = (int *)malloc(sizeof(int) * N);
	int *parked = (int *)calloc(N, sizeof(int));
	int *pneed = (int *)calloc(N, sizeof(int));
	int *stack = (int *)malloc(sizeof(int) * (6 * (size_t)N + 8));
	SlotPool pool;
	pool.cap = N + 1;
	pool.used = (unsigned char *)calloc(pool.cap, 1);
	pool.high = 0;
	t->post_ops = (phbc_post_op *)malloc(sizeof(phbc_post_op) * (nint > 0 ? nint : 1));
	t->pre_ops = (phbc_pre_op *)malloc(sizeof(phbc_pre_op) * (nint > 0 ? nint : 1));
	if (!need || !size || !slot_of || !row_of || !parked || !pneed || !stack || !pool.used || !t->post_ops || !t->pre_ops) {
		rc = fail(PHB_ENOMEM, "out of memory");
		goto done;
	}
	compute_need(t, need, size, stack);

	/* ---- post-order: emit ops (larger-need child first), then assign slots in program order ---- */
	int sp = 0, nops = 0, prev = -1;
	stack[sp++] = t->root;
	stack[sp++] = 0;
	while (sp) {
		int state = stack[--sp];
		int n = stack[--sp];
		if (is_tip(t, n)) continue;
		int a = t->left[n], b = t->right[n];
		if (state == 0) {
			stack[sp++] = n;
			stack[sp++] = 1;
			int first = need[a] >= need[b] ? a : b;
			int second = first == a ? b : a;
			stack[sp++] = second; /* popped after `first` */
			stack[sp++] = 0;
			stack[sp++] = first;
			stack[sp++] = 0;
		} else {
			phbc_post_op *op = &t->post_ops[nops];
			if (!is_tip(t, a) && is_tip(t, b)) { /* a tip child comes first */
				int tmp = a; a = b; b = tmp;
			}
			if (!is_tip(t, a) && !is_tip(t, b) && a == prev) { /* the just-computed child is operand b */
				int tmp = a; a = b; b = tmp;
			}
			if (!is_tip(t, b) && b != prev) {
				rc = fail(PHB_EINVAL, "post-order walk: child %d of node %d was not computed by the preceding op", b, n);
				goto done;
			}
			op->node = n;
			op->a_node = a;
			op->b_node = b;
			op->a_kind = is_tip(t, a) ? PHBC_W_TIP : PHBC_W_SLOT;
			op->b_kind = is_tip(t, b) ? PHBC_W_TIP : PHBC_W_SLOT; /* SLOT here means "registers of the previous op" */
			op->a_idx = op->b_idx = -1;
			op->dst_slot = -1;
			op->next_tips = 0;
			if (op->a_kind == PHBC_W_SLOT) parked[a] = 1;
			row_of[n] = nops;
			prev = n;
			nops++;
		}
	}
	for (int k = 0; k < nops; k++) {
		phbc_post_op *op = &t->post_ops[k];
		if (op->a_kind == PHBC_W_SLOT) {
			op->a_idx = slot_of[op->a_node];
			pool.used[slot_of[op->a_node]] = 0; /* slots are thread-private: release before placing the result */
		}
		if (parked[op->node]) slot_of[op->node] = op->dst_slot = slot_alloc(&pool);
	}
	t->post_slots = pool.high > 0 ? pool.high : 1;

	/* ---- pre-order ---- */
	memset(pool.used, 0, pool.cap);
	pool.high = 0;
	for (int k = 0; k < nops; k++) { /* register need over the tree of INTERNAL nodes, children before parents */
		int n = t->post_ops[k].node;
		int a = t->left[n], b = t->right[n];
		int ia = !is_tip(t, a), ib = !is_tip(t, b);
		if (!ia && !ib) pneed[n] = 0;
		else if (ia && !ib) pneed[n] = pneed[a];
		else if (!ia && ib) pneed[n] = pneed[b];
		else {
			int lo = pneed[a] < pneed[b] ? pneed[a] : pneed[b];
			int hi = pneed[a] < pneed[b] ? pneed[b] : pneed[a];
			pneed[n] = lo + 1 > hi ? lo + 1 : hi;
		}
	}
	int npre = 0;
	sp = 0;
	prev = -1;
	stack[sp++] = t->root;
	while (sp) {
		int n = stack[--sp];
		int a = t->left[n], b = t->right[n];
		if (!is_tip(t, a) && is_tip(t, b)) { /* a tip child comes first */
			int tmp = a; a = b; b = tmp;
		}
		if (!is_tip(t, a) && !is_tip(t, b) && pneed[a] < pneed[b]) { /* b = visited next = the smaller need */
			int tmp = a; a = b; b = tmp;
		}
		phbc_pre_op *op = &t->pre_ops[npre++];
		const int a_tip = is_tip(t, a), b_tip = is_tip(t, b);
		op->node = n;
		op->a_node = a;
		op->b_node = b;
		op->kind = (int16_t)((a_tip ? 0 : 1) + (b_tip ? 0 : 1));
		op->next_tips = 0;
		op->u_slot = -1;
		op->pf_a_row = op->pf_b_row = -1;
		if (n == t->root) {
			op->u_kind = PHBC_W_ROOT;
		} else if (n == prev) {
			op->u_kind = PHBC_W_REG; /* U_n is still in the registers of the preceding op */
		} else {
			op->u_kind = PHBC_W_SLOT;
			op->u_slot = (int16_t)slot_of[n];
			pool.used[slot_of[n]] = 0;
		}
		op->a_slot = op->b_slot = -1;
		op->a_code = op->b_code = -1;
		op->a_row = a_tip ? -1 : row_of[a];
		op->b_row = b_tip ? -1 : row_of[b];
		if (op->kind == 2) {
			slot_of[a] = slot_alloc(&pool);
			op->a_slot = (int16_t)slot_of[a];
			stack[sp++] = a; /* parked, popped after b's whole subtree */
		}
		if (op->kind >= 1) {
			stack[sp++] = b;
			prev = b;
		} else {
			prev = -1;
		}
	}
	t->pre_slots = pool.high > 0 ? pool.high : 1;
	if (nops != nint || npre != nint) {
		rc = fail(PHB_EINVAL, "walk schedule covers %d/%d of %d internal nodes", nops, npre, nint);
		goto done;
	}

	/* number the tip operands in walk order and make the descriptors' tip indices local to their chunk */
	const int nch = (nint + PHBC_WALK_CHUNK - 1) / PHBC_WALK_CHUNK;
	t->post_tip_order = (int *)malloc(sizeof(int) * T);
	t->pre_tip_order = (int *)malloc(sizeof(int) * T);
	t->post_chunk_tip0 = (int *)calloc(nch + 2, sizeof(int));
	t->pre_chunk_tip0 = (int *)calloc(nch + 2, sizeof(int));
	if (!t->post_tip_order || !t->pre_tip_order || !t->post_chunk_tip0 || !t->pre_chunk_tip0) {
		rc = fail(PHB_ENOMEM, "out of memory");
		goto done;
	}
	int k = 0, q = 0;
	for (int i = 0; i < nint; i++) {
		if (i % PHBC_WALK_CHUNK == 0) {
			t->post_chunk_tip0[i / PHBC_WALK_CHUNK] = k;
			t->pre_chunk_tip0[i / PHBC_WALK_CHUNK] = q;
		}
		phbc_post_op *po = &t->post_ops[i];
		if (po->a_kind == PHBC_W_TIP) {
			t->post_tip_order[k] = po->a_node;
			po->a_idx = k++ - t->post_chunk_tip0[i / PHBC_WALK_CHUNK];
		}
		if (po->b_kind == PHBC_W_TIP) {
			t->post_tip_order[k] = po->b_node;
			po->b_idx = k++ - t->post_chunk_tip0[i / PHBC_WALK_CHUNK];
		}
		phbc_pre_op *qo = &t->pre_ops[i];
		if (qo->kind != 2) { /* child a is a tip */
			t->pre_tip_order[q] = qo->a_node;
			qo->a_code = (int16_t)(q++ - t->pre_chunk_tip0[i / PHBC_WALK_CHUNK]);
		}
		if (qo->kind == 0) {
			t->pre_tip_order[q] = qo->b_node;
			qo->b_code = (int16_t)(q++ - t->pre_chunk_tip0[i / PHBC_WALK_CHUNK]);
		}
	}
	t->post_chunk_tip0[nch] = k;
	t->pre_chunk_tip0[nch] = q;
	if (k != T || q != T) {
		rc = fail(PHB_EINVAL, "walk schedule consumes %d/%d of %d tips", k, q, T);
		goto done;
	}
	/* the first op of chunk ch announces the tip range of chunk ch + 1 (the kernel issues that load while it works on ch) */
	for (int ch = 0; ch + 1 < nch; ch++) {
		const int i = ch * PHBC_WALK_CHUNK;
		t->post_ops[i].next_tips = (t->post_chunk_tip0[ch + 1] << 5) | (t->post_chunk_tip0[ch + 2] - t->post_chunk_tip0[ch + 1]);
		t->pre_ops[i].next_tips = (t->pre_chunk_tip0[ch + 1] << 5) | (t->pre_chunk_tip0[ch + 2] - t->pre_chunk_tip0[ch + 1]);
	}
	for (int i = 0; i < nint; i++) { /* what the op PHBC_PF_DIST positions later will read: requested into L2 at this op */
		const int k2 = i + PHBC_PF_DIST;
		t->pre_ops[i].pf_a_row = k2 < nint ? t->pre_ops[k2].a_row : -1;
		t->pre_ops[i].pf_b_row = k2 < nint ? t->pre_ops[k2].b_row : -1;
		t->pre_ops[i].flags = 0;
	}
	/* cherry recomputation (see phb_cuda.h): op i + 1 is the op of op i's child b whenever b is internal; when that op is tip-tip, b's
	 * message is rebuilt by op i and its row is neither written nor read */
	for (int i = 0; i + 1 < nint; i++) {
		phbc_pre_op *po = &t->pre_ops[i], *nx = &t->pre_ops[i + 1];
		if (po->kind >= 1 && nx->kind == 0 && nx->node == po->b_node) {
			po->flags |= PHBC_PRE_B_RECOMPUTE;
			nx->flags |= PHBC_PRE_TIPS_READY;
			t->post_ops[po->b_row].a_kind |= PHBC_POST_NO_ROW;
		}
	}
	for (int i = 0; i < nint; i++) { /* a row that is never read needs no L2 hint */
		const int k2 = i + PHBC_PF_DIST;
		if (k2 < nint && (t->pre_ops[k2].flags & PHBC_PRE_B_RECOMPUTE)) t->pre_ops[i].pf_b_row = -1;
	}
	t->post_first_tips = nch > 0 ? t->post_chunk_tip0[1] : 0;
	t->pre_first_tips = nch > 0 ? t->pre_chunk_tip0[1] : 0;
done:
	free(pneed);
	free(parked);
	free(need);
	free(size);
	free(slot_of);
	free(row_of);
	free(stack);
	free(pool.used);
	return rc;
}

/* ------------------------------------------------------------------------------------------- */
/* construction                                                                                */
/* ------------------------------------------------------------------------------------------- */

/* hand the host schedules to the device context */
static int push_schedule(phb_tlk *t) {
	const int N = t->N, ntips = t->T;
	int rc;
	phbc_schedule s;
	memset(&s, 0, sizeof(s));
	s.n_lower_ops = N - ntips;
	s.n_lower_levels = t->n_lower_levels;
	s.lower_ops = t->lower_ops;
	s.lower_level_off = t->lower_level_off;
	s.n_upper_ops = N - 1;
	s.n_upper_levels = t->n_upper_levels;
	s.upper_ops = t->upper_ops;
	s.upper_level_off = t->upper_level_off;
	s.n_parent_ops = N - ntips;
	s.parent_ops = t->parent_ops;
	s.parent_level_off = t->parent_level_off;
	s.n_post = N - ntips;
	s.n_pre = N - ntips;
	s.post_ops = t->post_ops;
	s.pre_ops = t->pre_ops;
	s.post_slots = t->post_slots;
	s.pre_slots = t->pre_slots;
	s.post_tip_order = t->post_tip_order;
	s.pre_tip_order = t->pre_tip_order;
	s.post_first_tips = t->post_first_tips;
	s.pre_first_tips = t->pre_first_tips;
	if ((rc = phbc_set_schedule(t->ctx, &s))) return dev_fail(rc);
	return PHB_OK;
}

/* copies and checks a topology (node-id convention of tree.c:183-199) */
static int install_topology(phb_tlk *t, const int *left, const int *right, int root) {
	const int N = t->N, ntips = t->T;
	if (root < ntips || root >= N) return fail(PHB_EINVAL, "root %d is not an internal node", root);
	for (int n = 0; n < N; n++) {
		const int tip = left[n] < 0;
		if ((left[n] < 0) != (right[n] < 0) || (tip && n >= ntips) || (!tip && n < ntips) || left[n] >= N || right[n] >= N)
			return fail(PHB_EINVAL, "node %d breaks the id convention (tips 0..T-1, internal T..2T-2)", n);
	}
	for (int n = 0; n < N; n++) t->parent[n] = -1;
	for (int n = 0; n < N; n++) {
		t->left[n] = left[n];
		t->right[n] = right[n];
		if (left[n] >= 0) {
			t->parent[left[n]] = n;
			t->parent[right[n]] = n;
		}
	}
	t->root = root;
	return PHB_OK;
}

static void free_schedules(phb_tlk *t) {
	free(t->lower_ops), free(t->upper_ops), free(t->lower_level_off), free(t->upper_level_off), free(t->parent_ops), free(t->parent_level_off);
	free(t->post_ops), free(t->pre_ops), free(t->post_tip_order), free(t->pre_tip_order), free(t->post_chunk_tip0), free(t->pre_chunk_tip0);
	t->lower_ops = t->upper_ops = NULL;
	t->lower_level_off = t->upper_level_off = t->parent_level_off = NULL;
	t->parent_ops = NULL;
	t->post_ops = NULL;
	t->pre_ops = NULL;
	t->post_tip_order = t->pre_tip_order = t->post_chunk_tip0 = t->pre_chunk_tip0 = NULL;
}

/*
 * A topology move (NNI / SPR, nniopt.c:301-334, spropt.c:1548-1615): the reference re-reads the Tree pointers on every traversal and
 * only needs SingleTreeLikelihood_update_three_nodes; here the traversal order is compiled into schedules, so a changed tree is
 * handed over explicitly.  Same taxa, same node-id convention; data, model inputs, options and branch lengths (by node id) are
 * kept, every partial is dirty, the time-tree tables must be set again.  On failure the object keeps its previous topology.
 */
static int rebuild_schedules(phb_tlk *t) {
	const int N = t->N;
	free_schedules(t);
	int rc = build_level_schedules(t);
	if (rc == PHB_OK) rc = build_walk_schedules(t);
	if (rc != PHB_OK) return rc;
	for (int n = 0; n < N; n++) t->upper_op_of[n] = -1;
	for (int k = 0; k < N - 1; k++) t->upper_op_of[t->upper_ops[k].out - N] = k;
	if (phbc_set_root(t->ctx, t->root)) return fail(PHB_ECUDA, "%s", phbc_last_error());
	return push_schedule(t);
}

int phb_tlk_set_topology(phb_tlk *t, const int *left, const int *right, int root) {
	if (!left || !right) return fail(PHB_EINVAL, "left and right are required");
	const int N = t->N;
	int *old = (int *)malloc(sizeof(int) * 2 * (size_t)N);
	if (!old) return fail(PHB_ENOMEM, "out of memory");
	memcpy(old, t->left, sizeof(int) * N);
	memcpy(old + N, t->right, sizeof(int) * N);
	const int old_root = t->root;
	int rc = install_topology(t, left, right, root); /* validates before it touches the object */
	if (rc == PHB_OK && (rc = rebuild_schedules(t)) != PHB_OK) {
		char msg[sizeof(g_err)];
		memcpy(msg, g_err, sizeof(msg));
		install_topology(t, old, old + N, old_root);
		rebuild_schedules(t);
		memcpy(g_err, msg, sizeof(msg));
	}
	free(old);
	t->have_time_tree = 0;
	t->resident = 0;
	memset(t->lower_ok, 0, N);
	memset(t->upper_ok, 0, N);
	phb_tlk_update_all_nodes(t);
	return rc;
}

phb_tlk *phb_tlk_create(int ntips, int nstate, int ncat, int npatterns, const int *left, const int *right, int root,
                        int use_tip_states, int device) {
	if (ntips < 2 || nstate < 2 || ncat < 1 || npatterns < 1 || !left || !right) {
		fail(PHB_EINVAL, "phb_tlk_create: need ntips >= 2, nstate >= 2, ncat >= 1, npatterns >= 1 and a topology");
		return NULL;
	}
	if (use_tip_states && nstate > 255) {
		fail(PHB_EINVAL, "phb_tlk_create: uint8 tip states need nstate <= 255");
		return NULL;
	}
	const int N = 2 * ntips - 1;
	if (root < 0 || root >= N) {
		fail(PHB_EINVAL, "phb_tlk_create: root %d out of range", root);
		return NULL;
	}
	phb_tlk *t = (phb_tlk *)calloc(1, sizeof(phb_tlk));
	if (!t) return NULL;
	t->T = ntips;
	t->N = N;
	t->S = nstate;
	t->C = ncat;
	t->P = npatterns;
	t->root = root;
	t->use_tip_states = use_tip_states != 0;
	t->device = device;
	t->left = (int *)malloc(sizeof(int) * N);
	t->right = (int *)malloc(sizeof(int) * N);
	t->parent = (int *)malloc(sizeof(int) * N);
	t->bl = (double *)calloc(N, sizeof(double));
	t->update_nodes = (unsigned char *)malloc(N);
	t->lower_ok = (unsigned char *)calloc(N, 1);
	t->upper_ok = (unsigned char *)calloc(N, 1);
	t->upper_op_of = (int *)malloc(sizeof(int) * N);
	t->sub_ops = (phbc_op *)malloc(sizeof(phbc_op) * 2 * (size_t)N);
	t->sub_level_off = (int *)malloc(sizeof(int) * ((size_t)N + 2));
	t->path = (int *)malloc(sizeof(int) * N);
	t->all_dirty = 1;
	if (!t->left || !t->right || !t->parent || !t->bl || !t->update_nodes || !t->lower_ok || !t->upper_ok || !t->upper_op_of || !t->sub_ops ||
	    !t->sub_level_off || !t->path) {
		phb_tlk_free(t);
		fail(PHB_ENOMEM, "phb_tlk_create: out of memory");
		return NULL;
	}
	for (int n = 0; n < N; n++) t->parent[n] = -1;
	for (int n = 0; n < N; n++) {
		t->left[n] = left[n];
		t->right[n] = right[n];
		const int tip = left[n] < 0;
		if ((left[n] < 0) != (right[n] < 0) || (tip && n >= ntips) || (!tip && n < ntips) || left[n] >= N || right[n] >= N) {
			phb_tlk_free(t);
			fail(PHB_EINVAL, "phb_tlk_create: node %d breaks the id convention (tips 0..T-1, internal T..2T-2)", n);
			return NULL;
		}
		if (!tip) {
			t->parent[left[n]] = n;
			t->parent[right[n]] = n;
		}
	}
	memset(t->update_nodes, 1, N); /* treelikelihood.c:1054-1059 */
	t->update = 1;
	t->update_upper = 1;
	t->scale = 0;
	t->scaling_threshold = 1.e-40; /* treelikelihood.c:1121 */
	t->include_root_freqs = 0;
	t->compat_scaled_gradient = 0;
	t->unrooted = 1;
	t->kernels = PHB_KERNELS_AUTO;
	t->host_exp = nstate >= 60;
	int rc = build_level_schedules(t);
	if (rc == PHB_OK) rc = build_walk_schedules(t);
	if (rc == PHB_OK) {
		for (int n = 0; n < N; n++) t->upper_op_of[n] = -1;
		for (int k = 0; k < N - 1; k++) t->upper_op_of[t->upper_ops[k].out - N] = k;
	}
	if (rc != PHB_OK) {
		phb_tlk_free(t);
		return NULL;
	}
	t->ctx = phbc_create(device, ntips, nstate, ncat, npatterns, root, use_tip_states ? PHBC_TIP_STATES : PHBC_TIP_PARTIALS);
	if (!t->ctx) {
		fail(PHB_ECUDA, "%s", phbc_last_error());
		phb_tlk_free(t);
		return NULL;
	}
	if ((rc = push_schedule(t))) {
		phb_tlk_free(t);
		return NULL;
	}
	return t;
}

void phb_tlk_free(phb_tlk *t) {
	if (!t) return;
	if (t->ctx) phbc_destroy(t->ctx);
	free(t->left);
	free(t->right);
	free(t->parent);
	free(t->bl);
	free(t->update_nodes);
	free(t->gradient);
	free(t->lower_ops);
	free(t->upper_ops);
	free(t->lower_level_off);
	free(t->upper_level_off);
	free(t->parent_ops);
	free(t->parent_level_off);
	free(t->post_ops);
	free(t->pre_ops);
	free(t->post_tip_order);
	free(t->pre_tip_order);
	free(t->post_chunk_tip0);
	free(t->pre_chunk_tip0);
	free(t->lower_ok), free(t->upper_ok), free(t->upper_op_of), free(t->sub_ops), free(t->sub_level_off), free(t->path);
	free(t->ex_buf);
	free(t->h_evec), free(t->h_eval), free(t->h_ivec), free(t->h_freqs), free(t->h_rates), free(t->h_props);
	free(t->st_bl), free(t->st_evec), free(t->st_eval), free(t->st_ivec), free(t->st_freqs), free(t->st_rates), free(t->st_props);
	free(t);
}

/*
 * clone_SingleTreeLikelihood (treelikelihood.c:1241-1395; Model.clone :715-790): an independent object with the same topology,
 * data, model inputs, options and rescaling state -- what the reference's parallel users build per worker (gradascent.c:166-170).
 * Tips, weights, explicit matrices and the time-tree tables are copied device to device (`device` may differ from the
 * source's); partials are not copied: the clone starts with every node dirty, as a clone of a dirty reference object does.
 */
phb_tlk *phb_tlk_clone(phb_tlk *src, int device) {
	if (!src) {
		fail(PHB_EINVAL, "phb_tlk_clone: NULL source");
		return NULL;
	}
	phb_tlk *t = phb_tlk_create(src->T, src->S, src->C, src->P, src->left, src->right, src->root, src->use_tip_states, device);
	if (!t) return NULL;
	int rc = PHB_OK;
	if (src->have_tips || src->have_weights || src->have_matrices || src->have_time_tree) {
		const int drc = phbc_copy_inputs(t->ctx, src->ctx, src->have_matrices, src->have_time_tree);
		if (drc) rc = dev_fail(drc);
	}
	t->have_tips = src->have_tips;
	t->have_weights = src->have_weights;
	t->have_time_tree = src->have_time_tree;
	if (rc == PHB_OK && src->have_eigen && src->h_evec) rc = phb_tlk_set_eigen(t, src->h_evec, src->h_eval, src->h_ivec);
	if (rc == PHB_OK && src->have_matrices) t->have_matrices = 1, t->have_eigen = 0; /* explicit matrices win, as in the source */
	if (rc == PHB_OK && src->have_freqs && src->h_freqs) rc = phb_tlk_set_frequencies(t, src->h_freqs);
	if (rc == PHB_OK && src->have_site && src->h_rates) rc = phb_tlk_set_site_model(t, src->h_rates, src->h_props);
	if (rc == PHB_OK && src->have_bl) rc = phb_tlk_set_branch_lengths(t, src->bl);
	if (rc != PHB_OK) {
		phb_tlk_free(t);
		return NULL;
	}
	t->scale = src->scale;
	t->scaling_threshold = src->scaling_threshold;
	t->include_root_freqs = src->include_root_freqs;
	t->compat_scaled_gradient = src->compat_scaled_gradient;
	t->unrooted = src->unrooted;
	t->kernels = src->kernels;
	t->incremental = src->incremental;
	t->host_exp = src->host_exp;
	if (src->prepared_gradient) phb_tlk_initialize_gradient(t, src->prepared_gradient);
	t->eigen_changed = t->freqs_changed = t->site_changed = t->bl_changed = 0;
	phb_tlk_update_all_nodes(t);
	return t;
}

/* ------------------------------------------------------------------------------------------- */
/* inputs                                                                                      */
/* ------------------------------------------------------------------------------------------- */

void phb_tlk_update_all_nodes(phb_tlk *t) { /* treelikelihood.c:1737-1744 */
	memset(t->update_nodes, 1, t->N);
	t->update = 1;
	t->update_upper = 1;
	t->all_dirty = 1; /* resident partials (if any) are stale as a whole */
	t->sweep_valid = 0;
}

int phb_tlk_update_one_node(phb_tlk *t, int node) { /* treelikelihood.c:1747-1751 */
	if (node < 0 || node >= t->N) return fail(PHB_EINVAL, "node %d out of range", node);
	t->update_nodes[node] = 1;
	t->update = 1;
	t->update_upper = 1;
	t->sweep_valid = 0;
	return PHB_OK;
}

/* SingleTreeLikelihood_update_three_nodes (treelikelihood.c:1754-1771): a node and both its children (NNI / SPR moves) */
int phb_tlk_update_three_nodes(phb_tlk *t, int node) {
	int rc = phb_tlk_update_one_node(t, node);
	if (rc) return rc;
	if (!is_tip(t, node)) {
		t->update_nodes[t->left[node]] = 1;
		t->update_nodes[t->right[node]] = 1;
	}
	return PHB_OK;
}

int phb_tlk_set_tip_states(phb_tlk *t, const uint8_t *states) {
	if (!t->use_tip_states) return fail(PHB_ESTATE, "tlk was created with use_tip_states = false");
	int rc = phbc_upload_tip_states(t->ctx, states);
	if (rc) return dev_fail(rc);
	t->have_tips = 1;
	phb_tlk_update_all_nodes(t);
	return PHB_OK;
}

int phb_tlk_set_tip_partials(phb_tlk *t, const double *partials) {
	if (t->use_tip_states) return fail(PHB_ESTATE, "tlk was created with use_tip_states = true");
	int rc = phbc_upload_tip_partials(t->ctx, partials);
	if (rc) return dev_fail(rc);
	t->have_tips = 1;
	phb_tlk_update_all_nodes(t);
	return PHB_OK;
}

int phb_tlk_set_pattern_weights(phb_tlk *t, const double *w) {
	int rc = phbc_upload_weights(t->ctx, w);
	if (rc) return dev_fail(rc);
	t->have_weights = 1;
	phb_tlk_update_all_nodes(t);
	return PHB_OK;
}

int phb_tlk_set_eigen(phb_tlk *t, const double *evec, const double *eval, const double *ivec) {
	int rc = phbc_upload_eigen(t->ctx, evec, eval, ivec);
	if (rc) return dev_fail(rc);
	if (!t->h_evec) {
		t->h_evec = (double *)malloc(sizeof(double) * t->S * t->S);
		t->h_ivec = (double *)malloc(sizeof(double) * t->S * t->S);
		t->h_eval = (double *)malloc(sizeof(double) * t->S);
	}
	if (evec != t->h_evec) {
		memcpy(t->h_evec, evec, sizeof(double) * t->S * t->S);
		memcpy(t->h_ivec, ivec, sizeof(double) * t->S * t->S);
		memcpy(t->h_eval, eval, sizeof(double) * t->S);
	}
	t->eigen_changed = 1;
	t->have_eigen = 1;
	t->have_matrices = 0;
	phb_tlk_update_all_nodes(t); /* substitution model changed: _treelikelihood_handle_change, :73-114 */
	return PHB_OK;
}

int phb_tlk_set_matrices(phb_tlk *t, const double *P, const double *dP) {
	int rc = phbc_upload_matrices(t->ctx, P, dP);
	if (rc) return dev_fail(rc);
	t->have_matrices = 1;
	phb_tlk_update_all_nodes(t);
	return PHB_OK;
}

int phb_tlk_set_frequencies(phb_tlk *t, const double *freqs) {
	int rc = phbc_upload_freqs(t->ctx, freqs);
	if (rc) return dev_fail(rc);
	if (!t->h_freqs) t->h_freqs = (double *)malloc(sizeof(double) * t->S);
	if (freqs != t->h_freqs) memcpy(t->h_freqs, freqs, sizeof(double) * t->S);
	t->freqs_changed = 1;
	t->have_freqs = 1;
	phb_tlk_update_all_nodes(t);
	return PHB_OK;
}

int phb_tlk_set_site_model(phb_tlk *t, const double *rates, const double *props) {
	int rc = phbc_upload_site_model(t->ctx, rates, props);
	if (rc) return dev_fail(rc);
	if (!t->h_rates) {
		t->h_rates = (double *)malloc(sizeof(double) * t->C);
		t->h_props = (double *)malloc(sizeof(double) * t->C);
	}
	if (rates != t->h_rates) {
		memcpy(t->h_rates, rates, sizeof(double) * t->C);
		memcpy(t->h_props, props, sizeof(double) * t->C);
	}
	t->site_changed = 1;
	t->have_site = 1;
	phb_tlk_update_all_nodes(t);
	return PHB_OK;
}

int phb_tlk_set_branch_lengths(phb_tlk *t, const double *bl) {
	for (int n = 0; n < t->N; n++) {
		if (n != t->root && bl[n] < 0) /* treelikelihood.c:1659-1662 exits on a negative length */
			return fail(PHB_EINVAL, "calculate_partials: node %d branch length = %E", n, bl[n]);
	}
	if (t->incremental && t->resident && !t->all_dirty && t->have_bl && bl != t->bl) {
		/* resident partials: only the branches whose length differs are dirty (what the reference's per-node listener reports) */
		for (int n = 0; n < t->N; n++)
			if (n != t->root && bl[n] != t->bl[n]) {
				t->bl[n] = bl[n];
				t->update_nodes[n] = 1;
				t->update = 1;
				t->update_upper = 1;
			}
		t->bl_dirty = 1;
		t->bl_changed = 1;
		return PHB_OK;
	}
	if (bl != t->bl) memcpy(t->bl, bl, sizeof(double) * t->N);
	t->have_bl = 1;
	t->bl_dirty = 1;
	t->bl_changed = 1;
	phb_tlk_update_all_nodes(t);
	return PHB_OK;
}

int phb_tlk_set_branch_length(phb_tlk *t, int node, double bl) {
	if (node < 0 || node >= t->N) return fail(PHB_EINVAL, "node %d out of range", node);
	if (bl < 0) return fail(PHB_EINVAL, "calculate_partials: node %d branch length = %E", node, bl);
	t->bl[node] = bl;
	t->bl_dirty = 1;
	t->bl_changed = 1;
	return phb_tlk_update_one_node(t, node);
}

int phb_tlk_use_rescaling(phb_tlk *t, int use) { /* SingleTreeLikelihood_use_rescaling */
	t->scale = use != 0;
	phb_tlk_update_all_nodes(t);
	return PHB_OK;
}

int phb_tlk_rescaling(const phb_tlk *t) { return t->scale; }

int phb_tlk_set_option(phb_tlk *t, int option, int value) {
	switch (option) {
	/* an option set to the value it already has leaves the caches alone */
	case PHB_OPT_INCLUDE_ROOT_FREQS:
		if (t->include_root_freqs == (value != 0)) return PHB_OK;
		t->include_root_freqs = value != 0;
		break;
	case PHB_OPT_COMPAT_SCALED_GRADIENT:
		if (t->compat_scaled_gradient == (value != 0)) return PHB_OK;
		t->compat_scaled_gradient = value != 0;
		break;
	case PHB_OPT_UNROOTED:
		if (t->unrooted == (value != 0)) return PHB_OK;
		t->unrooted = value != 0;
		break;
	case PHB_OPT_KERNELS:
		if (value < PHB_KERNELS_AUTO || value > PHB_KERNELS_FUSED) return fail(PHB_EINVAL, "unknown kernel family %d", value);
		if (t->kernels == value) return PHB_OK;
		t->kernels = value;
		t->all_dirty = 1;
		break;
	case PHB_OPT_SCALING_THRESHOLD_EXP:
		t->scaling_threshold = pow(10.0, -(double)value);
		t->all_dirty = 1;
		break;
	case PHB_OPT_INCREMENTAL:
		if (t->incremental == (value != 0)) return PHB_OK;
		t->incremental = value != 0;
		t->resident = 0;
		phb_tlk_update_all_nodes(t);
		return PHB_OK;
	case PHB_OPT_HOST_EXPONENTIALS:
		if (t->host_exp == (value != 0)) return PHB_OK;
		t->host_exp = value != 0;
		t->all_dirty = 1;
		break;
	case PHB_OPT_TUNE: {
		int rc = phbc_set_tune(t->ctx, value);
		if (rc) return dev_fail(rc);
		phb_tlk_update_all_nodes(t);
		return PHB_OK;
	}
	case PHB_OPT_TIMING: {
		int rc = phbc_set_timing(t->ctx, value);
		if (rc) return dev_fail(rc);
		return PHB_OK;
	}
	default: return fail(PHB_EINVAL, "unknown option %d", option);
	}
	t->update_upper = 1;
	if (option != PHB_OPT_UNROOTED) t->update = 1;
	return PHB_OK;
}

/* ------------------------------------------------------------------------------------------- */
/* evaluation                                                                                  */
/* ------------------------------------------------------------------------------------------- */

static int check_ready(const phb_tlk *t) {
	if (!t->have_tips) return fail(PHB_ESTATE, "tip states / partials not set");
	if (!t->have_weights) return fail(PHB_ESTATE, "pattern weights not set");
	if (!t->have_eigen && !t->have_matrices) return fail(PHB_ESTATE, "substitution model not set");
	if (!t->have_freqs) return fail(PHB_ESTATE, "frequencies not set");
	if (!t->have_site) return fail(PHB_ESTATE, "site model not set");
	if (!t->have_bl) return fail(PHB_ESTATE, "branch lengths not set");
	return PHB_OK;
}

static void fill_opts(const phb_tlk *t, phbc_eval_opts *o, int want_gradient, int batch_index) {
	memset(o, 0, sizeof(*o));
	o->kernels = t->kernels;
	o->scale = t->scale;
	o->scaling_threshold = t->scaling_threshold;
	o->include_root_freqs = t->include_root_freqs;
	o->compat_scaled_gradient = t->compat_scaled_gradient;
	o->want_gradient = want_gradient;
	o->explicit_matrices = t->have_matrices;
	o->batch_index = batch_index;
}

/*
 * Branch lengths of a single evaluation to the device -- and, for models whose tiny transition probabilities come out of the eigen
 * sum by cancellation (61 states: codons two or three changes apart, P ~ t^2, t^3), the exponentials exp(eval_k * bl_n * rate_c) from
 * THIS host's libm, the one the reference calls (substmodel.c:539): a one-ulp difference between two correct exp implementations
 * moves those entries by 1e-9 relative and the gradient of a codon alignment by up to 3e-8, so 1e-10 parity needs the same exp.
 * N * C * S values per evaluation (12,139 at C5), nothing next to the evaluation itself.
 */
static int wants_host_exp(const phb_tlk *t) { return t->host_exp && t->have_eigen && !t->have_matrices && t->h_eval && t->h_rates; }

/* ex [n][C][S] = exp(eval_q * (bl[k] * rate_c)) for n lengths */
static void host_exponentials(const phb_tlk *t, size_t n, const double *bl, double *ex) {
	const int C = t->C, S = t->S;
	for (size_t k = 0; k < n; k++)
		for (int c = 0; c < C; c++)
			for (int q = 0; q < S; q++) ex[(k * C + c) * S + q] = exp(t->h_eval[q] * (bl[k] * t->h_rates[c]));
}

/* the exponentials of nbatch branch-length vectors, [nbatch][N][C][S], to the device */
static int upload_host_exponentials(phb_tlk *t, const double *bl, int nbatch) {
	const size_t need = (size_t)nbatch * t->N * t->C * t->S;
	if (need > t->ex_cap) {
		double *nb = (double *)realloc(t->ex_buf, sizeof(double) * need);
		if (!nb) return -3;
		t->ex_buf = nb;
		t->ex_cap = need;
	}
	host_exponentials(t, (size_t)nbatch * t->N, bl, t->ex_buf);
	return phbc_upload_exponentials(t->ctx, t->ex_buf, nbatch);
}

static int upload_bl(phb_tlk *t) {
	int rc = phbc_upload_branch_lengths(t->ctx, t->bl, 1);
	if (rc) return rc;
	if (wants_host_exp(t)) rc = upload_host_exponentials(t, t->bl, 1);
	return rc;
}

/* one full evaluation with the reference's NaN / inf handling (treelikelihood.c:1489-1519) */
static int evaluate_once(phb_tlk *t, int want_gradient, double *lnl, double *grad_out) {
	int rc = check_ready(t);
	if (rc) return rc;
	/* always: the upload is N doubles, and the batched entry points leave other samples' lengths in the device slots */
	if ((rc = upload_bl(t))) return dev_fail(rc);
	t->bl_dirty = 0;
	t->sweep_valid = 0; /* whatever phb_tlk_matrix_gradient left on the device is overwritten or outdated from here on */
	phbc_eval_opts o;
	for (int attempt = 0; attempt < 2; attempt++) {
		fill_opts(t, &o, want_gradient, 0);
		if ((rc = phbc_evaluate(t->ctx, &o))) return dev_fail(rc);
		if ((rc = phbc_download_results(t->ctx, 1, lnl, want_gradient ? grad_out : NULL))) return dev_fail(rc);
		if (isinf(*lnl) && !t->scale) {
			t->scale = 1;
			t->all_dirty = 1; /* resident unscaled partials are of no use any more */
			continue;
		}
		break;
	}
	return PHB_OK;
}


/* ------------------------------------------------------------------------------------------- */
/* resident partials: incremental evaluation and the single-branch fast path                   */
/* ------------------------------------------------------------------------------------------- */

/*
 * With PHB_OPT_INCREMENTAL the object keeps every lower (and, once asked for, upper) partial on the device between calls, like the
 * reference's tlk->partials, and an evaluation recomputes only what the dirty flags reach:
 *   lower partials   the proper ancestors of every node marked by update_one_node / set_branch_length -- the traversal of
 *                    _calculate_partials (treelikelihood.c:1645-1734), as per-level op lists;
 *   upper partials   U_x stays valid iff x lies on the root path of EVERY changed branch (U_x depends on everything outside the
 *                    subtree of x, and on the length of x's own branch not at all); the others are rebuilt lazily, top-down, for the
 *                    nodes a caller needs (update_upper_partials2, :2164-2190; the node-change logic of _calculate_uppper, :2592-2636).
 * Any other change (model, site model, tips, weights, options) marks the whole object dirty and the next evaluation is a full one.
 * These evaluations run on the node-at-a-time kernels (tensor-core kernels for 20 / 61 states); the fused 4-state walk keeps no
 * partials and is used only when the option is off.
 */
static void fill_opts_resident(const phb_tlk *t, phbc_eval_opts *o, int want_gradient) {
	fill_opts(t, o, want_gradient, 0);
	o->kernels = ((t->S == 20 || (t->S >= 60 && t->S <= 63)) && t->kernels != PHB_KERNELS_GENERIC) ? PHB_KERNELS_AUTO : PHB_KERNELS_GENERIC;
	o->materialize_uppers = 1;
}

/* PHB_OPT_INCREMENTAL on, for the calls that need resident partials */
static void resident_on(phb_tlk *t) {
	if (!t->incremental) {
		t->incremental = 1;
		t->resident = 0;
	}
}

static void mark_clean(phb_tlk *t) {
	memset(t->update_nodes, 0, t->N);
	t->update = 0;
}

/* full evaluation that leaves all lower partials (and with want_gradient all upper partials) resident */
static int resident_full(phb_tlk *t, int want_gradient, double *lnl, double *grad_out) {
	int rc = check_ready(t);
	if (rc) return rc;
	if ((rc = upload_bl(t))) return dev_fail(rc);
	t->bl_dirty = 0;
	t->resident = 0;
	t->sweep_valid = 0;
	for (int attempt = 0; attempt < 2; attempt++) {
		phbc_eval_opts o;
		fill_opts_resident(t, &o, want_gradient);
		if ((rc = phbc_evaluate(t->ctx, &o))) return dev_fail(rc);
		if ((rc = phbc_download_results(t->ctx, 1, lnl, want_gradient ? grad_out : NULL))) return dev_fail(rc);
		if (isinf(*lnl) && !t->scale) {
			t->scale = 1;
			continue;
		}
		break;
	}
	if (isnan(*lnl) || isinf(*lnl)) return PHB_OK; /* nothing is marked valid */
	for (int n = 0; n < t->N; n++) {
		t->lower_ok[n] = 1;
		t->upper_ok[n] = want_gradient != 0;
	}
	t->upper_irf = t->include_root_freqs;
	t->resident = 1;
	t->all_dirty = 0;
	t->lower_stale = 0;
	return PHB_OK;
}

/* fold the dirty flags into the validity maps: lowers of every proper ancestor of a changed branch, uppers everywhere except on the root
 * path of EVERY changed branch */
static void resident_invalidate(phb_tlk *t) {
	if (!t->resident || t->all_dirty) return;
	const int N = t->N;
	int ndirty = 0;
	int *cnt = t->path;
	memset(cnt, 0, sizeof(int) * N);
	for (int n = 0; n < N; n++) {
		if (!t->update_nodes[n] || n == t->root) continue;
		ndirty++;
		cnt[n]++;
		for (int a = t->parent[n]; a >= 0; a = t->parent[a]) {
			t->lower_ok[a] = 0;
			cnt[a]++;
		}
	}
	if (ndirty) {
		t->lower_stale = 1;
		for (int n = 0; n < N; n++)
			if (cnt[n] != ndirty) t->upper_ok[n] = 0;
	}
}

/* make lnL and every lower partial current; recomputes only the ancestors of changed branches when it can */
static int resident_calculate(phb_tlk *t, double *lnl) {
	if (!t->update && t->resident && !t->all_dirty && !t->lower_stale) {
		*lnl = t->lk;
		return PHB_OK;
	}
	int rc;
	if (!t->resident || t->all_dirty) {
		if ((rc = resident_full(t, 0, &t->lk, NULL))) return rc;
	} else {
		if ((rc = check_ready(t))) return rc;
		const int N = t->N;
		t->sweep_valid = 0;
		resident_invalidate(t);
		int nops = 0;
		for (int l = 0; l < t->n_lower_levels; l++) {
			t->sub_level_off[l] = nops;
			for (int k = t->lower_level_off[l]; k < t->lower_level_off[l + 1]; k++)
				if (!t->lower_ok[t->lower_ops[k].out]) t->sub_ops[nops++] = t->lower_ops[k];
		}
		t->sub_level_off[t->n_lower_levels] = nops;
		if ((rc = upload_bl(t))) return dev_fail(rc);
		t->bl_dirty = 0;
		phbc_eval_opts o;
		fill_opts_resident(t, &o, 0);
		if ((rc = phbc_run_ops(t->ctx, &o, nops, t->sub_ops, t->n_lower_levels, t->sub_level_off, 1, 1, &t->lk))) return dev_fail(rc);
		if (isinf(t->lk) && !t->scale) { /* treelikelihood.c:1496-1519: switch rescaling on and recompute everything */
			t->scale = 1;
			if ((rc = resident_full(t, 0, &t->lk, NULL))) return rc;
		} else if (!isnan(t->lk) && !isinf(t->lk)) {
			for (int n = 0; n < N; n++) t->lower_ok[n] = 1;
			t->lower_stale = 0;
		}
	}
	*lnl = t->lk;
	if (isnan(t->lk) || isinf(t->lk)) {
		if (isnan(t->lk)) phb_tlk_update_all_nodes(t); /* :1489-1495 */
		t->resident = 0;
		return PHB_OK;
	}
	mark_clean(t);
	t->update_upper = 1;
	return PHB_OK;
}

/* make U_node (node >= 0) or every upper partial (node < 0) current; lowers and matrices must be current */
static int resident_uppers(phb_tlk *t, int node, int irf) {
	const int N = t->N;
	if (t->upper_irf != irf) {
		memset(t->upper_ok, 0, N);
		t->upper_irf = irf;
	}
	int nops = 0, nlevels = 0;
	if (node >= 0) {
		int len = 0;
		for (int x = node; x != t->root; x = t->parent[x]) t->path[len++] = x;
		for (int k = len - 1; k >= 0; k--) { /* top-down: each op needs the one before it */
			const int x = t->path[k];
			if (t->upper_ok[x]) continue;
			t->sub_level_off[nlevels++] = nops;
			t->sub_ops[nops++] = t->upper_ops[t->upper_op_of[x]];
		}
		t->sub_level_off[nlevels] = nops;
	} else {
		for (int l = 0; l < t->n_upper_levels; l++) {
			t->sub_level_off[l] = nops;
			for (int k = t->upper_level_off[l]; k < t->upper_level_off[l + 1]; k++)
				if (!t->upper_ok[t->upper_ops[k].out - N]) t->sub_ops[nops++] = t->upper_ops[k];
		}
		nlevels = t->n_upper_levels;
		t->sub_level_off[nlevels] = nops;
	}
	if (nops == 0) return PHB_OK;
	phbc_eval_opts o;
	fill_opts_resident(t, &o, 1);
	o.include_root_freqs = irf;
	int rc = phbc_run_ops(t->ctx, &o, nops, t->sub_ops, nlevels, t->sub_level_off, 0, 0, NULL);
	if (rc) return dev_fail(rc);
	for (int k = 0; k < nops; k++) t->upper_ok[t->sub_ops[k].out - N] = 1;
	return PHB_OK;
}

/* SingleTreeLikelihood_update_uppers (treelikelihood.c:1530-1538): lnL, then every upper partial (root frequencies not folded in) */
static int phb_tlk_update_uppers_impl(phb_tlk *t) {
	resident_on(t);
	double lnl;
	int rc = resident_calculate(t, &lnl);
	if (rc) return rc;
	if (isnan(lnl) || isinf(lnl)) return fail(PHB_ESTATE, "update_uppers: lnL = %f", lnl);
	return resident_uppers(t, -1, 0);
}

/* lnL, d lnL/dt, d2 lnL/dt2 [nitems][3] of the branch above nodes[k] at length bl[k]; the uppers and lowers of those nodes are resident */
static int branch_items(phb_tlk *t, int nitems, const int *nodes, const double *bl, double *out) {
	phbc_eval_opts o;
	fill_opts_resident(t, &o, 1);
	double *ex = NULL;
	if (wants_host_exp(t)) { /* the item lengths get the host's exponentials like every other matrix of this model */
		ex = (double *)malloc(sizeof(double) * (size_t)nitems * t->C * t->S);
		if (!ex) return fail(PHB_ENOMEM, "out of memory");
		host_exponentials(t, (size_t)nitems, bl, ex);
	}
	const int rc = phbc_branch_lnl(t->ctx, &o, nitems, nodes, bl, ex, out);
	free(ex);
	return rc ? dev_fail(rc) : PHB_OK;
}

/* _calculate_uppper + calculate_dldt_uppper + d2lnldt2_uppper (treelikelihood.c:2592-2686, 2195-2335) at nbl candidate lengths */
static int phb_tlk_calculate_branch_impl(phb_tlk *t, int node, int nbl, const double *bl, double *lnl, double *dlnl, double *d2lnl) {
	if (node < 0 || node >= t->N || node == t->root) return fail(PHB_EINVAL, "calculate_branch: node %d is not a branch (root %d)", node, t->root);
	if (nbl < 1 || !bl) return fail(PHB_EINVAL, "calculate_branch: nbl >= 1 and bl are required");
	if (t->have_matrices) return fail(PHB_ESTATE, "calculate_branch needs the eigen system: explicit matrices cannot be re-evaluated at a new length");
	for (int k = 0; k < nbl; k++)
		if (bl[k] < 0) return fail(PHB_EINVAL, "calculate_partials: node %d branch length = %E", node, bl[k]);
	resident_on(t);
	double cur;
	int rc = resident_calculate(t, &cur);
	if (rc) return rc;
	if (isnan(cur) || isinf(cur)) {
		for (int k = 0; k < nbl; k++) {
			if (lnl) lnl[k] = cur;
			if (dlnl) dlnl[k] = NAN;
			if (d2lnl) d2lnl[k] = NAN;
		}
		return PHB_OK;
	}
	if ((rc = resident_uppers(t, node, 0))) return rc;
	int *nodes = (int *)malloc(sizeof(int) * (size_t)nbl);
	if (!nodes) return fail(PHB_ENOMEM, "out of memory");
	for (int k = 0; k < nbl; k++) nodes[k] = node;
	double *out = (double *)malloc(sizeof(double) * 3 * (size_t)nbl);
	if (!out) {
		free(nodes);
		return fail(PHB_ENOMEM, "out of memory");
	}
	rc = branch_items(t, nbl, nodes, bl, out);
	free(nodes);
	if (!rc)
		for (int k = 0; k < nbl; k++) {
			if (lnl) lnl[k] = out[3 * k];
			if (dlnl) dlnl[k] = out[3 * k + 1];
			if (d2lnl) d2lnl[k] = out[3 * k + 2];
		}
	free(out);
	return rc;
}

static void apply_unrooted(const phb_tlk *t, double *g);

/*
 * Diagonal of the branch-length Hessian (d2lnldt2_uppper, treelikelihood.c:2267-2335, for every branch at its current length), with
 * lnL and the gradient of the same pass.  Route 1: one unscaled fused 4-state walk that forms d2P/dt2 L = Q (Q m) next to the gradient
 * terms (phbc_nuc4_hessian).  Route 2, for everything the walk declines: lowers and uppers made resident (PHB_OPT_INCREMENTAL on, as
 * update_uppers does) and one launch of the single-branch kernels over the list (n, bl[n]) of every non-root node.
 */
static int phb_tlk_branch_hessian_diagonal_impl(phb_tlk *t, double *lnl, double *grad, double *hess) {
	if (!lnl || !hess) return fail(PHB_EINVAL, "branch_hessian_diagonal: lnl and hess are required");
	if (t->have_matrices) return fail(PHB_ESTATE, "branch_hessian_diagonal needs the eigen system: explicit matrices cannot be differentiated twice");
	int rc = check_ready(t);
	if (rc) return rc;
	const int N = t->N;
	double cur = 0.0;
	int done = 0;
	if (!t->incremental && !t->scale && t->kernels != PHB_KERNELS_GENERIC) {
		if ((rc = upload_bl(t))) return dev_fail(rc);
		t->bl_dirty = 0;
		t->sweep_valid = 0;
		phbc_eval_opts o;
		fill_opts(t, &o, 3, 0);
		rc = phbc_nuc4_hessian(t->ctx, &o, &cur, grad, hess);
		if (rc < 0) return dev_fail(rc);
		if (rc == 0) {
			if (isinf(cur)) { /* treelikelihood.c:1496-1519: rescaling on, recompute once -- on route 2, the walk route is unscaled */
				t->scale = 1;
				t->all_dirty = 1;
			} else {
				done = 1;
				t->lk = cur;
				if (isnan(cur)) {
					phb_tlk_update_all_nodes(t); /* :1489-1495 */
				} else {
					memset(t->update_nodes, 0, N);
					t->update = 0;
					t->update_upper = 1; /* the tlk-owned gradient buffer is not refreshed here */
				}
			}
		}
	}
	if (!done) {
		resident_on(t);
		if ((rc = resident_calculate(t, &cur))) return rc; /* retries with rescaling on itself */
		if (!isnan(cur) && !isinf(cur)) {
			if ((rc = resident_uppers(t, -1, 0))) return rc;
			int *nodes = (int *)malloc(sizeof(int) * (size_t)N);
			double *bl = (double *)malloc(sizeof(double) * (size_t)N);
			double *out = (double *)malloc(sizeof(double) * 3 * (size_t)N);
			if (!nodes || !bl || !out) {
				free(nodes), free(bl), free(out);
				return fail(PHB_ENOMEM, "out of memory");
			}
			int n_items = 0;
			for (int n = 0; n < N; n++)
				if (n != t->root) nodes[n_items] = n, bl[n_items++] = t->bl[n];
			rc = branch_items(t, n_items, nodes, bl, out);
			if (!rc) {
				for (int k = 0; k < n_items; k++) {
					if (grad) grad[nodes[k]] = out[3 * k + 1];
					hess[nodes[k]] = out[3 * k + 2];
				}
				if (grad) grad[t->root] = 0.0;
				hess[t->root] = 0.0;
			}
			free(nodes), free(bl), free(out);
			if (rc) return rc;
		}
	}
	*lnl = cur;
	if (isnan(cur) || isinf(cur)) { /* as phb_tlk_gradient, :328-332 */
		for (int n = 0; n < N; n++) {
			if (grad) grad[n] = NAN;
			hess[n] = NAN;
		}
		return PHB_OK;
	}
	if (grad) apply_unrooted(t, grad);
	apply_unrooted(t, hess);
	return PHB_OK;
}

/*
 * Nearest-neighbour interchanges (nniopt.c:301-334): move (x, y) exchanges the subtrees rooted at x and y across the branch above
 * v = parent[y].  Kind R (0): x is the sibling of v.  Kind C (1): v and w are the two children of the root, w is internal and x a child
 * of w -- the NNI across the root edge of the unrooted tree.  -1: not a move.
 */
static int sibling_of(const phb_tlk *t, int n) {
	const int p = t->parent[n];
	return t->left[p] == n ? t->right[p] : t->left[p];
}

static int nni_kind(const phb_tlk *t, int x, int y) {
	const int N = t->N;
	if (x < 0 || x >= N || y < 0 || y >= N || x == y) return -1;
	const int v = t->parent[y];
	if (v < 0 || v == t->root) return -1;
	const int p = t->parent[v];
	if (t->parent[x] == p && x != v) return 0;
	if (p == t->root) {
		const int w = sibling_of(t, v);
		if (!is_tip(t, w) && t->parent[x] == w) return 1;
	}
	return -1;
}

static int phb_tlk_nni_moves_impl(phb_tlk *t, int *moves) {
	int n = 0;
	for (int v = 0; v < t->N; v++) {
		if (is_tip(t, v) || v == t->root || (t->unrooted && t->parent[v] == t->root)) continue;
		const int s = sibling_of(t, v);
		if (moves) moves[2 * n] = s, moves[2 * n + 1] = t->left[v], moves[2 * n + 2] = s, moves[2 * n + 3] = t->right[v];
		n += 2;
	}
	const int r1 = t->left[t->root], r2 = t->right[t->root];
	if (t->unrooted && r1 >= 0 && !is_tip(t, r1) && !is_tip(t, r2)) {
		if (moves) moves[2 * n] = t->left[r1], moves[2 * n + 1] = t->left[r2], moves[2 * n + 2] = t->left[r1], moves[2 * n + 3] = t->right[r2];
		n += 2;
	}
	return n;
}

/* the matrix table of a score pass: every node at its current length (the root's entry unused, 0), then one length per candidate --
 * given[k], or the current length of node dflt[k * stride] */
static void table_lengths(const phb_tlk *t, int ncand, const double *given, const int *dflt, int dflt_stride, double *bl) {
	for (int n = 0; n < t->N; n++) bl[n] = n == t->root ? 0.0 : t->bl[n];
	for (int k = 0; k < ncand; k++) bl[t->N + k] = given ? given[k] : t->bl[dflt[(size_t)k * dflt_stride]];
}

/* launch order of the 4-state kernel's work items: by parent of v, so that the groups of two siblings are neighbours (U_p from L2) */
typedef struct NniKey {
	int pv, v, x, k; /* parent of v, v, x, move index */
} NniKey;
static int nni_order(const void *pa, const void *pb) {
	const NniKey *a = (const NniKey *)pa, *b = (const NniKey *)pb;
	const int ka[4] = {a->pv, a->v, a->x, a->k}, kb[4] = {b->pv, b->v, b->x, b->k};
	for (int i = 0; i < 4; i++)
		if (ka[i] != kb[i]) return ka[i] < kb[i] ? -1 : 1;
	return 0;
}

/* one pass of the scores on resident partials: every upper partial, the move descriptors, the (v, x) pairs, the matrix table and its
 * lengths */
typedef struct NniArgs {
	int nmoves;
	const int *moves;
	const double *t_central;
} NniArgs;
static int nni_pass(phb_tlk *t, const void *arg, double *out) {
	const NniArgs *a = (const NniArgs *)arg;
	const int N = t->N, C = t->C, S = t->S, nmoves = a->nmoves;
	const int *moves = a->moves;
	int rc = resident_uppers(t, -1, 0);
	if (rc) return rc;
	const size_t items = (size_t)N + nmoves;
	phbc_nni_move *desc = (phbc_nni_move *)malloc(sizeof(phbc_nni_move) * (size_t)nmoves);
	NniKey *order = (NniKey *)malloc(sizeof(NniKey) * (size_t)nmoves);
	int *groups = (int *)malloc(sizeof(int) * 2 * (size_t)nmoves);
	double *bl = (double *)malloc(sizeof(double) * items);
	double *ex = wants_host_exp(t) ? (double *)malloc(sizeof(double) * items * C * S) : NULL;
	if (!desc || !order || !groups || !bl || (wants_host_exp(t) && !ex)) {
		rc = fail(PHB_ENOMEM, "out of memory");
		goto done;
	}
	for (int k = 0; k < nmoves; k++) {
		const int x = moves[2 * k], y = moves[2 * k + 1], v = t->parent[y];
		phbc_nni_move *m = &desc[k];
		m->x = x, m->y = y, m->keep = sibling_of(t, y);
		if (nni_kind(t, x, y) == 0) {
			const int p = t->parent[v];
			m->a = p == t->root ? -1 : N + p, m->a_mat = p, m->w = -1;
		} else {
			m->w = t->parent[x];
			m->a = m->a_mat = sibling_of(t, x);
		}
		m->cmat = N + k, m->out = k;
		order[k] = (NniKey){t->parent[v], v, x, k};
	}
	table_lengths(t, nmoves, a->t_central, &order[0].v, sizeof(NniKey) / sizeof(int), bl); /* the central branch is v's */
	qsort(order, (size_t)nmoves, sizeof(NniKey), nni_order);
	int ngroups = 0;
	for (int i = 0; i < nmoves; ngroups++) {
		const NniKey *ka = &order[i], *kb = i + 1 < nmoves ? &order[i + 1] : NULL;
		const int pair = kb && ka->x == kb->x && ka->v == kb->v;
		groups[2 * ngroups] = ka->k, groups[2 * ngroups + 1] = pair ? kb->k : -1;
		i += pair ? 2 : 1;
	}
	if (ex) host_exponentials(t, items, bl, ex);
	phbc_eval_opts o;
	fill_opts_resident(t, &o, 1);
	if ((rc = phbc_nni_scores(t->ctx, &o, nmoves, desc, ngroups, groups, bl, ex, out))) rc = dev_fail(rc);
done:
	free(desc), free(order), free(groups), free(bl), free(ex);
	return rc;
}

/*
 * The score calls on resident partials (NNI, SPR): reserve the resident buffers (-3 with the object unchanged), make the lowers resident
 * (PHB_OPT_INCREMENTAL on), then one pass writing out [n][3].  NaN / inf as treelikelihood.c:1496-1519: an infinite lnL of the current
 * tree, or an output that is not finite while rescaling is off, switches rescaling on and scores once more; a current lnL still NaN or
 * infinite NaN-fills out.
 */
static int resident_scores(phb_tlk *t, int n, double *lnl, double *out, int (*pass)(phb_tlk *, const void *, double *), const void *arg) {
	phbc_eval_opts o;
	fill_opts(t, &o, 1, 0);
	int rc = phbc_generic_buffers(t->ctx, &o);
	if (rc) return dev_fail(rc);
	resident_on(t);
	double cur = 0.0;
	for (int attempt = 0; attempt < 2; attempt++) {
		if ((rc = resident_calculate(t, &cur))) return rc; /* retries with rescaling on itself */
		if (isnan(cur) || isinf(cur)) break;
		if ((rc = pass(t, arg, out))) return rc;
		int finite = 1;
		for (int k = 0; k < 3 * n; k++) finite &= isfinite(out[k]) != 0;
		if (finite || t->scale) break;
		t->scale = 1; /* something underflowed unscaled: rescale everything and score again */
		t->all_dirty = 1;
	}
	if (lnl) *lnl = cur;
	if (isnan(cur) || isinf(cur))
		for (int k = 0; k < 3 * n; k++) out[k] = NAN;
	return PHB_OK;
}

/* lnL and central-branch derivatives of every listed NNI neighbour from resident partials (phb_nni.cu) */
static int phb_tlk_nni_scores_impl(phb_tlk *t, int nmoves, const int *moves, const double *t_central, double *lnl, double *out) {
	if (!moves || !out) return fail(PHB_EINVAL, "nni_scores: moves and out are required");
	if (nmoves < 1) return fail(PHB_EINVAL, "nni_scores: %d moves (at least one is needed)", nmoves);
	for (int k = 0; k < nmoves; k++) {
		if (nni_kind(t, moves[2 * k], moves[2 * k + 1]) < 0)
			return fail(PHB_EINVAL, "nni_scores: move %d (%d, %d) is not a nearest-neighbour interchange of the current tree", k, moves[2 * k],
			            moves[2 * k + 1]);
		if (t_central && !(t_central[k] >= 0))
			return fail(PHB_EINVAL, "nni_scores: move %d central branch length = %E", k, t_central[k]);
	}
	if (t->have_matrices) return fail(PHB_ESTATE, "nni_scores needs the eigen system: explicit matrices cannot be re-evaluated at a new length");
	int rc = check_ready(t);
	if (rc) return rc;
	const NniArgs a = {nmoves, moves, t_central};
	return resident_scores(t, nmoves, lnl, out, nni_pass, &a);
}

/*
 * Subtree prune and regraft (spropt.c:1548-1615): the subtree of s is pruned together with p = parent[s] -- the sibling b of s takes
 * p's slot under g = parent[p] -- and regrafted on the branch above a target e of the pruned tree: p takes e's slot, e the slot of p
 * that is not s's.  s may be neither the root nor a child of the root; a target is any node outside the subtree of s other than p and
 * the root.  Regrafting on b gives back the current tree.
 */
static int spr_check_prune(const phb_tlk *t, const char *fn, int s) {
	if (s < 0 || s >= t->N || s == t->root || t->parent[s] == t->root)
		return fail(PHB_EINVAL, "%s: node %d cannot be pruned (it must be neither the root %d nor a child of the root)", fn, s, t->root);
	return PHB_OK;
}

/* mark [N] = 1 on the subtree of s, 0 elsewhere; stack [N] scratch */
static void mark_subtree(const phb_tlk *t, int s, unsigned char *mark, int *stack) {
	memset(mark, 0, t->N);
	int sp = 0;
	stack[sp++] = s;
	while (sp) {
		const int x = stack[--sp];
		mark[x] = 1;
		if (!is_tip(t, x)) stack[sp++] = t->left[x], stack[sp++] = t->right[x];
	}
}

static int phb_tlk_spr_targets_impl(phb_tlk *t, int s, int *targets) {
	int rc = spr_check_prune(t, "spr_targets", s);
	if (rc) return rc;
	unsigned char *mark = (unsigned char *)malloc(t->N);
	int *stack = (int *)malloc(sizeof(int) * t->N);
	if (!mark || !stack) {
		free(mark), free(stack);
		return fail(PHB_ENOMEM, "out of memory");
	}
	mark_subtree(t, s, mark, stack);
	const int p = t->parent[s], g = t->parent[p], b = sibling_of(t, s);
	/* unrooted: regrafting on q = sibling(p) when g is the root gives the current tree again (b and q then hang from the root, one
	 * unrooted edge), and the pruned tree's two root-child branches are one unrooted edge otherwise -- drop the right one */
	const int twin = !t->unrooted ? -1 : (g == t->root ? sibling_of(t, p) : t->right[t->root]);
	int n = 0;
	for (int e = 0; e < t->N; e++) {
		if (e == t->root || e == p || mark[e] || e == b || e == twin) continue;
		if (targets) targets[n] = e;
		n++;
	}
	free(mark), free(stack);
	return n;
}

/*
 * One pass of the SPR scores: the pruned tree's partials over the resident buffers, then the contraction of every target (phb_spr.cu).
 *   lowers  g's op becomes (b, b) o (q, q) on the side p had, every ancestor of g below the root takes its usual op (nothing when g is
 *           the root; the root's own lower partial is never written);
 *   uppers  the pruned tree's upper op of every node outside {p} and the subtree of s, grouped by their depth in the pruned tree.
 * Current matrices (no rebuild), no root integration.  The validity maps lose exactly what the pass overwrites: lower_ok of g and its
 * ancestors below the root (lower_stale: the next evaluation recomputes them, and the cached lnL stays that of the current tree) and
 * upper_ok of every node it wrote; the uppers of p and of the subtree of s are untouched.
 */
typedef struct SprArgs {
	int s, ntargets;
	const int *targets;
	const double *t_pendant;
} SprArgs;
static int spr_pass(phb_tlk *t, const void *arg, double *out) {
	const SprArgs *a = (const SprArgs *)arg;
	const int s = a->s, ntargets = a->ntargets;
	const int N = t->N, C = t->C, S = t->S, root = t->root;
	const int p = t->parent[s], g = t->parent[p], b = sibling_of(t, s);
	const size_t items = (size_t)N + ntargets;
	int *queue = (int *)malloc(sizeof(int) * N);
	int *depth = (int *)malloc(sizeof(int) * N);
	double *bl = (double *)malloc(sizeof(double) * items);
	double *ex = wants_host_exp(t) ? (double *)malloc(sizeof(double) * items * C * S) : NULL;
	int rc = PHB_OK;
	if (!queue || !depth || !bl || (wants_host_exp(t) && !ex)) {
		rc = fail(PHB_ENOMEM, "out of memory");
		goto done;
	}
	t->sweep_valid = 0;
	phbc_eval_opts o;
	int nops = 0;
	for (int x = g; x != root; x = t->parent[x]) { /* one level each, children before parents */
		int l = t->left[x], r = t->right[x];
		if (x == g) *(l == p ? &l : &r) = b;
		phbc_op *op = &t->sub_ops[nops];
		op->out = x, op->a = op->a_mat = l, op->b = op->b_mat = r, op->flags = 0;
		t->sub_level_off[nops] = nops;
		nops++;
		t->lower_ok[x] = 0;
	}
	t->sub_level_off[nops] = nops;
	if (nops) {
		t->lower_stale = 1;
		fill_opts_resident(t, &o, 0);
		if ((rc = phbc_run_ops(t->ctx, &o, nops, t->sub_ops, nops, t->sub_level_off, 0, 0, NULL))) {
			rc = dev_fail(rc);
			goto done;
		}
	}
	/* uppers: breadth first over the pruned tree (p replaced by b), so that the ops come grouped by depth */
	int head = 0, tail = 0, nlevels = 0;
	nops = 0;
	queue[tail++] = root;
	depth[root] = 0;
	while (head < tail) {
		const int n = queue[head++];
		if (is_tip(t, n)) continue;
		int ch[2] = {t->left[n], t->right[n]};
		for (int j = 0; j < 2; j++)
			if (ch[j] == p) ch[j] = b;
		for (int j = 0; j < 2; j++) {
			const int x = ch[j], sib = ch[1 - j];
			phbc_op *op = &t->sub_ops[nops++];
			op->out = N + x;
			if (n != root) /* u_x = (P_n u_n) o (P_sib L_sib) */
				op->a = N + n, op->a_mat = n, op->b = op->b_mat = sib, op->flags = 0;
			else /* u_x = P_sib L_sib */
				op->a = op->a_mat = sib, op->b = op->b_mat = -1, op->flags = 1;
			depth[x] = depth[n] + 1;
			queue[tail++] = x;
			t->upper_ok[x] = 0;
		}
	}
	for (int k = 0; k < nops; k++)
		if (k == 0 || depth[t->sub_ops[k].out - N] != depth[t->sub_ops[k - 1].out - N]) t->sub_level_off[nlevels++] = k;
	t->sub_level_off[nlevels] = nops;
	fill_opts_resident(t, &o, 1);
	o.include_root_freqs = 0;
	if ((rc = phbc_run_ops(t->ctx, &o, nops, t->sub_ops, nlevels, t->sub_level_off, 0, 0, NULL))) {
		rc = dev_fail(rc);
		goto done;
	}
	table_lengths(t, ntargets, a->t_pendant, &s, 0, bl); /* the pendant branch is s's */
	if (ex) host_exponentials(t, items, bl, ex);
	fill_opts_resident(t, &o, 1);
	if ((rc = phbc_spr_scores(t->ctx, &o, s, p, ntargets, a->targets, bl, ex, out))) rc = dev_fail(rc);
done:
	free(queue), free(depth), free(bl), free(ex);
	return rc;
}

/* lnL and pendant-branch derivatives of the subtree of s regrafted on each listed target, from one pass over the pruned tree (phb_spr.cu);
 * the matrix table is reserved with the resident buffers, before the pruned pass changes anything */
static int phb_tlk_spr_scores_impl(phb_tlk *t, int s, int ntargets, const int *targets, const double *t_pendant, double *lnl, double *out) {
	int rc = spr_check_prune(t, "spr_scores", s);
	if (rc) return rc;
	if (!targets || !out) return fail(PHB_EINVAL, "spr_scores: targets and out are required");
	if (ntargets < 1) return fail(PHB_EINVAL, "spr_scores: %d targets (at least one is needed)", ntargets);
	unsigned char *mark = (unsigned char *)malloc(t->N);
	int *stack = (int *)malloc(sizeof(int) * t->N);
	if (!mark || !stack) {
		free(mark), free(stack);
		return fail(PHB_ENOMEM, "out of memory");
	}
	mark_subtree(t, s, mark, stack);
	const int p = t->parent[s];
	for (int k = 0; k < ntargets && !rc; k++) {
		const int e = targets[k];
		if (e < 0 || e >= t->N || e == t->root || e == p || mark[e])
			rc = fail(PHB_EINVAL, "spr_scores: target %d (node %d) is not a regraft position of the subtree of %d", k, e, s);
		else if (t_pendant && !(t_pendant[k] >= 0))
			rc = fail(PHB_EINVAL, "spr_scores: target %d pendant branch length = %E", k, t_pendant[k]);
	}
	free(mark), free(stack);
	if (rc) return rc;
	if (t->have_matrices) return fail(PHB_ESTATE, "spr_scores needs the eigen system: explicit matrices cannot be re-evaluated at a new length");
	if ((rc = check_ready(t))) return rc;
	if ((rc = phbc_spr_reserve(t->ctx, ntargets))) return dev_fail(rc);
	const SprArgs a = {s, ntargets, targets, t_pendant};
	return resident_scores(t, ntargets, lnl, out, spr_pass, &a);
}

/*
 * tlk->update_partials(tlk, out, p1, m1, p2, m2) (treelikelihood.h:91; treelikelihoodX.c:1207 and friends): ONE partial update on the
 * resident buffers, by index like the reference's slot -- out = (P[m1] x[p1]) o (P[m2] x[p2]), p2 < 0: single child (the upper partial of
 * a child of the root, treelikelihood.c:2147).  Indices: < T tips, T..N-1 lower partials, N + node upper partials
 * (tlk->upper_partial_indexes, :2131).  This is what the callers that drive the slot themselves go through -- update_upper_partials[2]
 * (:2129-2190), the tripod optimisation of SPR (spropt.c:1578-1608), _calculate_partials (:1645-1734) -- once the glue has re-pointed
 * the slot.  Lower partials are made current first (whatever is dirty is recomputed with the current branch lengths), the
 * transition matrices are rebuilt from the current lengths, and `mirror` (may be NULL) receives a host copy of the result
 * [C][P][S], so that reference code reading tlk->partials directly (asr.c:60-69) sees what the device computed.
 */
static int phb_tlk_update_partials_impl(phb_tlk *t, int out, int p1, int m1, int p2, int m2, double *mirror) {
	const int N = t->N, T = t->T;
	if (out < T || out >= 2 * N || p1 < 0 || p1 >= 2 * N || m1 < 0 || m1 >= N || p2 >= 2 * N || (p2 >= 0 && (m2 < 0 || m2 >= N)))
		return fail(PHB_EINVAL, "update_partials(%d, %d, %d, %d, %d): index out of range", out, p1, m1, p2, m2);
	if (t->have_matrices) return fail(PHB_ESTATE, "update_partials needs the eigen system: explicit matrices belong to one set of branch lengths");
	resident_on(t);
	double cur;
	int rc = resident_calculate(t, &cur);
	if (rc) return rc;
	if (isnan(cur) || isinf(cur)) return fail(PHB_ESTATE, "update_partials: lnL = %f", cur);
	phbc_op op;
	op.out = out, op.a = p1, op.a_mat = m1, op.b = p2 < 0 ? -1 : p2, op.b_mat = p2 < 0 ? -1 : m2, op.flags = 0;
	const int off[2] = {0, 1};
	phbc_eval_opts o;
	fill_opts_resident(t, &o, out >= N);
	o.include_root_freqs = 0;
	if ((rc = phbc_run_ops(t->ctx, &o, 1, &op, 1, off, 1, 0, NULL))) return dev_fail(rc);
	if (out >= N) {
		if (t->upper_irf != 0) memset(t->upper_ok, 0, N);
		t->upper_irf = 0;
		t->upper_ok[out - N] = 1;
	}
	if (mirror && (rc = phbc_download_partials(t->ctx, out, mirror))) return dev_fail(rc);
	return PHB_OK;
}

/*
 * Gradient while partials are resident.  A gradient over ALL branches is a whole-tree job whatever changed (one changed branch
 * invalidates every upper partial outside its root path), and the fused kernels do the whole tree faster than the node-at-a-time
 * kernels can patch it (C2: 6.4 ms fused against 46 ms patched, round 1 h6) -- so the evaluation runs on the fast path.  The fused
 * 4-state walk leaves the resident buffers alone: the dirty flags are folded into the validity maps first and the next incremental
 * call recomputes only what they reach.  A path that rewrites the node-at-a-time buffers (tensor-core message form, generic) ends
 * residency; the next incremental call starts from a full lower pass.
 */
static int resident_gradient(phb_tlk *t, double *lnl, double *grad_out) {
	resident_invalidate(t);
	const long long before = phbc_node_eval_count(t->ctx);
	int rc = evaluate_once(t, 1, lnl, grad_out);
	if (rc) return rc;
	if (phbc_node_eval_count(t->ctx) != before || isnan(*lnl) || isinf(*lnl)) t->resident = 0;
	return PHB_OK;
}

static int phb_tlk_calculate_impl(phb_tlk *t, double *lnl) {
	if (!t->update) { /* cached, treelikelihood.c:1458-1460 */
		*lnl = t->lk;
		return PHB_OK;
	}
	if (t->incremental) return resident_calculate(t, lnl);
	int rc = evaluate_once(t, 0, &t->lk, NULL);
	if (rc) return rc;
	*lnl = t->lk;
	if (isnan(t->lk)) { /* :1489-1495 */
		phb_tlk_update_all_nodes(t);
		return PHB_OK;
	}
	memset(t->update_nodes, 0, t->N);
	t->update = 0;
	t->update_upper = 1;
	return PHB_OK;
}

int phb_tlk_pattern_log_likelihoods(phb_tlk *t, double *out) {
	double lnl;
	int rc = phb_tlk_calculate(t, &lnl);
	if (rc) return rc;
	if ((rc = phbc_download_pattern_lnl(t->ctx, out))) return dev_fail(rc);
	return PHB_OK;
}

size_t phb_tlk_initialize_gradient(phb_tlk *t, int flags) {
	if (flags == 0) flags = PHB_FLAG_TREE_MODEL;
	t->prepared_gradient = flags;
	size_t len = 0;
	if (flags & PHB_FLAG_TREE_MODEL) len += (size_t)t->N; /* branch-length trees: node count, treelikelihood.c:271-274 */
	if (t->gradient == NULL || t->gradient_length < len) {
		double *g = (double *)realloc(t->gradient, sizeof(double) * (len > 0 ? len : 1));
		if (!g) {
			fail(PHB_ENOMEM, "out of memory");
			return 0;
		}
		t->gradient = g;
	}
	t->gradient_length = len;
	t->update_upper = 1;
	return len;
}

static void apply_unrooted(const phb_tlk *t, double *g) {
	g[t->root] = 0.0;
	if (t->unrooted) g[t->right[t->root]] = 0.0; /* treelikelihood.c:3249-3255 */
}

static int phb_tlk_gradient_impl(phb_tlk *t, const double **grad) {
	if (t->gradient == NULL || !(t->prepared_gradient & PHB_FLAG_TREE_MODEL)) {
		if (phb_tlk_initialize_gradient(t, PHB_FLAG_TREE_MODEL) == 0) return PHB_ENOMEM;
	}
	if (t->update_upper || t->update) { /* treelikelihood.c:323 */
		double lnl;
		int rc = t->incremental ? resident_gradient(t, &lnl, t->gradient) : evaluate_once(t, 1, &lnl, t->gradient);
		if (rc) return rc;
		t->lk = lnl;
		if (isnan(lnl) || isinf(lnl)) { /* :328-332 */
			for (size_t i = 0; i < t->gradient_length; i++) t->gradient[i] = NAN;
			if (isnan(lnl)) phb_tlk_update_all_nodes(t);
		} else {
			apply_unrooted(t, t->gradient);
			memset(t->update_nodes, 0, t->N);
			t->update = 0;
			t->update_upper = 0;
		}
	}
	*grad = t->gradient;
	return PHB_OK;
}

int phb_tlk_cat_branch_gradient(phb_tlk *t, double *out) {
	int rc = phbc_download_cat_grad(t->ctx, out);
	if (rc) return dev_fail(rc);
	for (int c = 0; c < t->C; c++) {
		out[(size_t)t->root * t->C + c] = 0.0;
		if (t->unrooted) out[(size_t)t->right[t->root] * t->C + c] = 0.0;
	}
	return PHB_OK;
}

int phb_tlk_get_partials(phb_tlk *t, int index, double *out) {
	int rc;
	if (index >= t->T && t->incremental && t->resident && !t->all_dirty && (t->update || t->lower_stale)) {
		/* pending set_branch_length changes, or dirty flags a fused gradient call folded into the validity maps: recompute what they reach */
		double cur;
		if ((rc = resident_calculate(t, &cur))) return rc;
	}
	if (index >= t->T && !(t->incremental && t->resident && !t->all_dirty && !t->update && !t->lower_stale)) {
		/* tlk->partials as the reference holds them: a node-at-a-time evaluation with every upper partial materialised (the fused paths
		 * keep no partials, or keep messages P L in their place) */
		if ((rc = check_ready(t))) return rc;
		if ((rc = upload_bl(t))) return dev_fail(rc);
		phbc_eval_opts o;
		fill_opts_resident(t, &o, 1);
		t->resident = 0;
		t->sweep_valid = 0;
		if ((rc = phbc_evaluate(t->ctx, &o))) return dev_fail(rc);
	} else if (index >= t->N && t->incremental) {
		if ((rc = resident_uppers(t, index - t->N, t->upper_irf))) return rc;
	}
	rc = phbc_download_partials(t->ctx, index, out);
	if (rc) return dev_fail(rc);
	return PHB_OK;
}

int phb_tlk_get_matrices(phb_tlk *t, double *P, double *dP) {
	int rc = phbc_download_matrices(t->ctx, P, dP);
	if (rc) return dev_fail(rc);
	return PHB_OK;
}

static int phb_tlk_gradient_device_impl(phb_tlk *t, double *out_device) {
	int rc = check_ready(t);
	if (rc) return rc;
	if ((rc = upload_bl(t))) return dev_fail(rc);
	phbc_eval_opts o;
	fill_opts(t, &o, 1, 0);
	t->resident = 0;
	t->sweep_valid = 0;
	if ((rc = phbc_evaluate(t->ctx, &o))) return dev_fail(rc);
	if ((rc = phbc_result_to_device(t->ctx, 0, out_device))) return dev_fail(rc);
	/* the device copy holds raw per-shard sums; the caller applies the unrooted convention after the reduction */
	memset(t->update_nodes, 0, t->N);
	t->update = 1; /* lk is not known on the host: keep the object dirty */
	t->update_upper = 1;
	return PHB_OK;
}

/*
 * Split evaluation for single-process multi-GPU hosts (phb_group.c): launch queues one evaluation of the current inputs on the
 * tlk's stream and returns; collect blocks on that stream and returns the RAW sums of this object's patterns -- no inf / NaN /
 * unrooted policy, that belongs to whoever adds the shards up.  The object stays dirty (its lnL is not known here).
 */
static int phb_tlk_evaluate_launch_impl(phb_tlk *t, int want_gradient) {
	int rc = check_ready(t);
	if (rc) return rc;
	if ((rc = upload_bl(t))) return dev_fail(rc);
	t->bl_dirty = 0;
	phbc_eval_opts o;
	fill_opts(t, &o, want_gradient != 0, 0);
	t->resident = 0;
	t->sweep_valid = 0;
	if ((rc = phbc_evaluate(t->ctx, &o))) return dev_fail(rc);
	memset(t->update_nodes, 0, t->N);
	t->update = 1;
	t->update_upper = 1;
	return PHB_OK;
}

int phb_tlk_evaluate_collect(phb_tlk *t, double *lnl, double *grad) {
	int rc = phbc_download_results(t->ctx, 1, lnl, grad);
	if (rc) return dev_fail(rc);
	return PHB_OK;
}

/*
 * One process per GPU, patterns sharded across the ranks of `comm` (SURVEY.md 8e): this rank's evaluation, then ONE in-place
 * ncclAllReduce(sum) of [lnL, grad[N], inf flag] on the tlk's own stream -- kernels and collective are ordered by the stream, the host
 * does not wait in between.  The _device form only enqueues and hands back the device buffer (raw reduced sums, no policy).
 */
int phb_internal_allreduce(phb_comm *c, double *buf, size_t count, void *stream); /* phb_nccl.c */

static int phb_tlk_gradient_allreduce_device_impl(phb_tlk *t, phb_comm *comm, double **out_device) {
	int rc = check_ready(t);
	if (rc) return rc;
	if ((rc = upload_bl(t))) return dev_fail(rc);
	t->bl_dirty = 0;
	phbc_eval_opts o;
	fill_opts(t, &o, 1, 0);
	t->resident = 0;
	t->sweep_valid = 0;
	if ((rc = phbc_evaluate(t->ctx, &o))) return dev_fail(rc);
	double *buf = NULL;
	if ((rc = phbc_pack_reduce(t->ctx, 0, &buf))) return dev_fail(rc);
	if (comm && phb_comm_size(comm) > 1 && (rc = phb_internal_allreduce(comm, buf, (size_t)t->N + 2, phbc_stream(t->ctx)))) return rc;
	if (out_device) *out_device = buf;
	memset(t->update_nodes, 0, t->N);
	t->update = 1; /* lk is not known on the host: keep the object dirty */
	t->update_upper = 1;
	return PHB_OK;
}

/* the same with host results and the reference's conventions applied to the REDUCED values on every rank alike: +-inf lnL (or an
 * inf shard) switches rescaling on and recomputes (treelikelihood.c:1496-1519), NaN / inf NaN-fills the gradient (:328-332), the
 * unrooted convention zeroes the root's right child (:3249-3255).  *grad is owned by the tlk. */
static int phb_tlk_gradient_allreduce_impl(phb_tlk *t, phb_comm *comm, double *lnl, const double **grad) {
	if (!grad) return fail(PHB_EINVAL, "grad is required");
	if (t->gradient == NULL || !(t->prepared_gradient & PHB_FLAG_TREE_MODEL)) {
		if (phb_tlk_initialize_gradient(t, PHB_FLAG_TREE_MODEL) == 0) return PHB_ENOMEM;
	}
	const int N = t->N;
	double *h = (double *)malloc(sizeof(double) * ((size_t)N + 2));
	if (!h) return fail(PHB_ENOMEM, "out of memory");
	int rc = PHB_OK;
	for (int attempt = 0; attempt < 2; attempt++) {
		if ((rc = phb_tlk_gradient_allreduce_device(t, comm, NULL))) break;
		if ((rc = phbc_download_reduce(t->ctx, h))) {
			rc = dev_fail(rc);
			break;
		}
		if ((isinf(h[0]) || h[N + 1] > 0.0) && !t->scale) { /* every rank reads the same reduced values and takes the same branch */
			t->scale = 1;
			t->all_dirty = 1;
			continue;
		}
		break;
	}
	if (rc == PHB_OK) {
		t->lk = h[0];
		if (isnan(t->lk) || isinf(t->lk)) {
			for (int n = 0; n < N; n++) t->gradient[n] = NAN;
		} else {
			memcpy(t->gradient, h + 1, sizeof(double) * N);
			apply_unrooted(t, t->gradient);
		}
		if (lnl) *lnl = t->lk;
		*grad = t->gradient;
	}
	free(h);
	return rc;
}

/* for phb_group.c (one host thread, several devices): an evaluation queued with its result packed for the group's all-reduce */
int phb_internal_launch_packed(phb_tlk *t, int want_gradient, double **dev_buf, void **stream) {
	int rc = phb_tlk_evaluate_launch(t, want_gradient);
	if (rc) return rc;
	if ((rc = phbc_pack_reduce(t->ctx, 0, dev_buf))) return dev_fail(rc);
	*stream = phbc_stream(t->ctx);
	return PHB_OK;
}

int phb_internal_collect_packed(phb_tlk *t, double *host /* [N + 2] */) {
	int rc = phbc_download_reduce(t->ctx, host);
	if (rc) return dev_fail(rc);
	return PHB_OK;
}

void *phb_tlk_stream(phb_tlk *t) { return phbc_stream(t->ctx); }

int phb_tlk_synchronize(phb_tlk *t) {
	int rc = phbc_synchronize(t->ctx);
	if (rc) return dev_fail(rc);
	return PHB_OK;
}

static int phb_tlk_gradient_batch_impl(phb_tlk *t, int nbatch, const double *bl, double *lnl, double *grad) {
	if (nbatch < 1) return fail(PHB_EINVAL, "nbatch must be >= 1");
	/* inputs other than branch lengths must be in place */
	const int had_bl = t->have_bl;
	t->have_bl = 1;
	int rc = check_ready(t);
	t->have_bl = had_bl;
	if (rc) return rc;
	for (int b = 0; b < nbatch; b++)
		for (int n = 0; n < t->N; n++)
			if (n != t->root && bl[(size_t)b * t->N + n] < 0)
				return fail(PHB_EINVAL, "calculate_partials: sample %d node %d branch length = %E", b, n, bl[(size_t)b * t->N + n]);
	for (int attempt = 0; attempt < 2; attempt++) {
		if ((rc = phbc_upload_branch_lengths(t->ctx, bl, nbatch))) return dev_fail(rc);
		if (wants_host_exp(t) && (rc = upload_host_exponentials(t, bl, nbatch))) return dev_fail(rc);
		phbc_eval_opts o;
		fill_opts(t, &o, grad != NULL, 0);
		o.batch_count = nbatch; /* the fused 4-state walk takes the whole batch in one launch */
		if ((rc = phbc_evaluate(t->ctx, &o))) return dev_fail(rc);
		if ((rc = phbc_download_results(t->ctx, nbatch, lnl, grad))) return dev_fail(rc);
		int any_inf = 0;
		for (int b = 0; b < nbatch; b++) any_inf |= isinf(lnl[b]);
		if (any_inf && !t->scale) {
			t->scale = 1;
			continue;
		}
		break;
	}
	if (grad)
		for (int b = 0; b < nbatch; b++) {
			double *g = grad + (size_t)b * t->N;
			if (isnan(lnl[b]) || isinf(lnl[b])) {
				for (int n = 0; n < t->N; n++) g[n] = NAN;
			} else {
				apply_unrooted(t, g);
			}
		}
	/* the single-sample state (t->bl, t->lk) is untouched but device partials now belong to the last sample */
	phb_tlk_update_all_nodes(t);
	return PHB_OK;
}

/* node sweep of calculate_dlnl_dQ (treelikelihood.c:2337-2583) for `nsets` sets of per-node matrices, e.g. dP/d theta from m->dPdp */
static int phb_tlk_matrix_gradient_impl(phb_tlk *t, int nsets, const double *M, double *out) {
	if (nsets < 1 || !M || !out) return fail(PHB_EINVAL, "nsets >= 1, M and out are required");
	int rc = check_ready(t);
	if (rc) return rc;
	if ((rc = upload_bl(t))) return dev_fail(rc);
	t->bl_dirty = 0;
	for (int attempt = 0; attempt < 2; attempt++) {
		phbc_eval_opts o;
		fill_opts(t, &o, 1, 0);
		double lnl = 0.0;
		t->resident = 0; /* the sweep rebuilds every partial with its own options */
		if ((rc = phbc_matrix_gradient(t->ctx, &o, nsets, M, t->unrooted ? t->right[t->root] : -1, &lnl, out))) return dev_fail(rc);
		t->lk = lnl;
		if (isinf(lnl) && !t->scale) { /* treelikelihood.c:1496-1519 */
			t->scale = 1;
			continue;
		}
		break;
	}
	if (isnan(t->lk) || isinf(t->lk))
		for (int k = 0; k < nsets; k++) out[k] = NAN;
	t->update = isnan(t->lk) ? 1 : 0;
	t->update_upper = 1; /* the gradient buffer was not refreshed */
	t->sweep_valid = !(isnan(t->lk) || isinf(t->lk));
	return PHB_OK;
}

/* makes the root's lower partial (or the fused walk's root statistics) current on the device; *ok = 0 when lnL is NaN / inf */
static int ensure_root_partial(phb_tlk *t, int *ok) {
	int rc = check_ready(t);
	if (rc) return rc;
	if (t->incremental && t->resident && !t->all_dirty && (t->update || t->lower_stale)) {
		double cur;
		if ((rc = resident_calculate(t, &cur))) return rc;
	}
	const int resident_ok = t->incremental && t->resident && !t->all_dirty && !t->update && !t->lower_stale;
	*ok = 1;
	if (!resident_ok && (t->update || !t->sweep_valid)) { /* a node-at-a-time evaluation leaves the root partial on the device */
		if ((rc = upload_bl(t))) return dev_fail(rc);
		t->bl_dirty = 0;
		t->resident = 0;
		for (int attempt = 0; attempt < 2; attempt++) {
			phbc_eval_opts o;
			fill_opts_resident(t, &o, 0);
			if ((rc = phbc_evaluate(t->ctx, &o))) return dev_fail(rc);
			if ((rc = phbc_download_results(t->ctx, 1, &t->lk, NULL))) return dev_fail(rc);
			if (isinf(t->lk) && !t->scale) {
				t->scale = 1;
				continue;
			}
			break;
		}
		t->update = isnan(t->lk) ? 1 : 0;
		t->sweep_valid = !(isnan(t->lk) || isinf(t->lk));
		*ok = t->sweep_valid;
	}
	return PHB_OK;
}

/* root term of the frequency parameters in calculate_dlnl_dQ (treelikelihood.c:2371-2404): out[i] = d lnL / d pi_i at fixed partials */
int phb_tlk_root_frequency_gradient(phb_tlk *t, double *out) {
	if (!out) return fail(PHB_EINVAL, "out is required");
	int ok = 0, rc = ensure_root_partial(t, &ok);
	if (rc) return rc;
	if (!ok) {
		for (int i = 0; i < t->S; i++) out[i] = NAN;
		return PHB_OK;
	}
	if ((rc = phbc_root_frequency_gradient(t->ctx, out))) return dev_fail(rc);
	return PHB_OK;
}

/* d lnL / d prop_c at fixed conditional likelihoods: out[c] = sum_k w_k S_c(k) / L_k, S_c(k) the category's site likelihood.  The root
 * term of the invariant-site proportion (gradient_pinv_sitemodel / gradient_pinv_W_sitemodel, treelikelihood.c:2943-3001) is
 * out[0] - out[1], respectively out[0] - mean(out[1..]) */
int phb_tlk_category_gradient(phb_tlk *t, double *out) {
	if (!out) return fail(PHB_EINVAL, "out is required");
	int ok = 0, rc = ensure_root_partial(t, &ok);
	if (rc) return rc;
	if (!ok) {
		for (int c = 0; c < t->C; c++) out[c] = NAN;
		return PHB_OK;
	}
	if ((rc = phbc_root_category_gradient(t->ctx, out))) return dev_fail(rc);
	return PHB_OK;
}

/* ------------------------------------------------------------------------------------------- */
/* store / restore (MCMC accept / reject)                                                      */
/* ------------------------------------------------------------------------------------------- */

/*
 * _singleTreeLikelihood_store (treelikelihood.c:126-150): remember the state a rejected proposal returns to.  The reference
 * flips between two sets of partials and matrices; this backend recomputes every node per evaluation and keeps no partials
 * across calls (the fused walk has none), so the stored state is the inputs the likelihood is a function of -- branch
 * lengths, eigen system, frequencies, site model, rescaling flag -- and the cached lnL with its dirty flag.
 */
int phb_tlk_store(phb_tlk *t) {
	const size_t S = t->S, C = t->C, N = t->N;
	if (!t->st_bl) {
		t->st_bl = (double *)malloc(sizeof(double) * N);
		t->st_evec = (double *)malloc(sizeof(double) * S * S);
		t->st_ivec = (double *)malloc(sizeof(double) * S * S);
		t->st_eval = (double *)malloc(sizeof(double) * S);
		t->st_freqs = (double *)malloc(sizeof(double) * S);
		t->st_rates = (double *)malloc(sizeof(double) * C);
		t->st_props = (double *)malloc(sizeof(double) * C);
		if (!t->st_bl || !t->st_evec || !t->st_ivec || !t->st_eval || !t->st_freqs || !t->st_rates || !t->st_props) return fail(PHB_ENOMEM, "out of memory");
	}
	memcpy(t->st_bl, t->bl, sizeof(double) * N);
	t->st_have_eigen = t->have_eigen && t->h_evec != NULL;
	if (t->st_have_eigen) {
		memcpy(t->st_evec, t->h_evec, sizeof(double) * S * S);
		memcpy(t->st_ivec, t->h_ivec, sizeof(double) * S * S);
		memcpy(t->st_eval, t->h_eval, sizeof(double) * S);
	}
	if (t->h_freqs) memcpy(t->st_freqs, t->h_freqs, sizeof(double) * S);
	if (t->h_rates) {
		memcpy(t->st_rates, t->h_rates, sizeof(double) * C);
		memcpy(t->st_props, t->h_props, sizeof(double) * C);
	}
	t->st_lk = t->lk; /* tlk->stored_lk */
	t->st_update = t->update;
	t->st_scale = t->scale;
	t->eigen_changed = t->freqs_changed = t->site_changed = t->bl_changed = 0;
	t->has_store = 1;
	return PHB_OK;
}

/*
 * _singleTreeLikelihood_restore + _treelikelihood_handle_restore (treelikelihood.c:116-124, 152-161): back to the stored
 * state WITHOUT recomputation -- tlk->lk = tlk->stored_lk, and a following calculate() returns it from the cache.  Only the
 * inputs that changed since the store travel to the device again.  Models given as explicit matrices are not stored: after a
 * restore the caller sets them again (which marks the object dirty).
 */
int phb_tlk_restore(phb_tlk *t) {
	if (!t->has_store) return fail(PHB_ESTATE, "phb_tlk_restore without phb_tlk_store");
	int rc;
	if (t->bl_changed) {
		memcpy(t->bl, t->st_bl, sizeof(double) * t->N);
		t->bl_dirty = 1;
	}
	if (t->eigen_changed && t->st_have_eigen && (rc = phb_tlk_set_eigen(t, t->st_evec, t->st_eval, t->st_ivec))) return rc;
	if (t->freqs_changed && t->h_freqs && (rc = phb_tlk_set_frequencies(t, t->st_freqs))) return rc;
	if (t->site_changed && t->h_rates && (rc = phb_tlk_set_site_model(t, t->st_rates, t->st_props))) return rc;
	t->scale = t->st_scale;
	t->lk = t->st_lk;
	t->update = t->st_update || (t->eigen_changed && !t->st_have_eigen); /* explicit matrices were not stored */
	if (!t->update) memset(t->update_nodes, 0, t->N);
	t->update_upper = 1; /* the gradient buffer belongs to the rejected state */
	if (t->eigen_changed || t->freqs_changed || t->site_changed || t->bl_changed) t->all_dirty = 1; /* so do resident partials */
	t->eigen_changed = t->freqs_changed = t->site_changed = t->bl_changed = 0;
	return PHB_OK;
}

/* ------------------------------------------------------------------------------------------- */
/* time trees (batched chain on the device, phb_timetree.cu)                                   */
/* ------------------------------------------------------------------------------------------- */

int phb_tlk_set_time_tree(phb_tlk *t, const double *tip_heights) {
	const int N = t->N, T = t->T;
	double *lowers = (double *)malloc(sizeof(double) * N);
	int *pre = (int *)malloc(sizeof(int) * N), *post = (int *)malloc(sizeof(int) * N), *stack = (int *)malloc(sizeof(int) * N);
	if (!lowers || !pre || !post || !stack) {
		free(lowers), free(pre), free(post), free(stack);
		return fail(PHB_ENOMEM, "out of memory");
	}
	int sp = 0, cnt = 0;
	stack[sp++] = t->root;
	while (sp) { /* pre-order: parents before children */
		const int n = stack[--sp];
		pre[cnt++] = n;
		if (!is_tip(t, n)) {
			stack[sp++] = t->right[n];
			stack[sp++] = t->left[n];
		}
	}
	for (int k = 0; k < N; k++) post[k] = pre[N - 1 - k]; /* reversed pre-order: children before parents */
	/* lower bound of a node = the oldest sampling date below it (tree_transform_collect_lowers, treetransform.c:239-252) */
	for (int k = 0; k < N; k++) {
		const int n = post[k];
		if (is_tip(t, n)) lowers[n] = tip_heights[n];
		else lowers[n] = lowers[t->left[n]] > lowers[t->right[n]] ? lowers[t->left[n]] : lowers[t->right[n]];
	}
	(void)T;
	int rc = phbc_set_time_tree(t->ctx, lowers, t->parent, pre, post);
	free(lowers), free(pre), free(post), free(stack);
	if (rc) return dev_fail(rc);
	t->have_time_tree = 1;
	return PHB_OK;
}

static int phb_tlk_gradient_batch_time_impl(phb_tlk *t, int nbatch, const double *ratios, const double *rates, int nrates, int include_jacobian,
                                double *lnl, double *log_jacobian, double *grad_ratios, double *grad_rates) {
	if (nbatch < 1 || !ratios || !rates || !lnl) return fail(PHB_EINVAL, "nbatch >= 1, ratios, rates and lnl are required");
	if (nrates != 1 && nrates != t->N) return fail(PHB_EINVAL, "nrates must be 1 (strict clock) or N = %d (one rate per node)", t->N);
	if (!t->have_time_tree) return fail(PHB_ESTATE, "phb_tlk_set_time_tree has not been called");
	const int had_bl = t->have_bl;
	t->have_bl = 1;
	int rc = check_ready(t);
	t->have_bl = had_bl;
	if (rc) return rc;
	const int want_gradient = grad_ratios != NULL || grad_rates != NULL;
	rc = phbc_time_forward(t->ctx, nbatch, ratios, rates, nrates);
	if (rc == 1) return fail(PHB_EINVAL, "calculate_partials: a sample has a negative branch length (node older than its parent)");
	if (rc) return dev_fail(rc);
	if (wants_host_exp(t)) { /* the chain built the branch lengths on the device: fetch them for the host's exp (>= 60 states only) */
		double *hbl = (double *)malloc(sizeof(double) * (size_t)nbatch * t->N);
		if (!hbl) return fail(PHB_ENOMEM, "out of memory");
		rc = phbc_download_branch_lengths(t->ctx, nbatch, hbl);
		if (!rc) rc = upload_host_exponentials(t, hbl, nbatch);
		free(hbl);
		if (rc) return dev_fail(rc);
	}
	for (int attempt = 0; attempt < 2; attempt++) {
		phbc_eval_opts o;
		fill_opts(t, &o, want_gradient, 0);
		o.batch_count = nbatch;
		if ((rc = phbc_evaluate(t->ctx, &o))) return dev_fail(rc);
		if ((rc = phbc_time_backward(t->ctx, nbatch, nrates, include_jacobian, want_gradient, lnl, log_jacobian, grad_ratios, grad_rates)))
			return dev_fail(rc);
		int any_inf = 0;
		for (int b = 0; b < nbatch; b++) any_inf |= isinf(lnl[b]);
		if (any_inf && !t->scale) { /* treelikelihood.c:1496-1519 */
			t->scale = 1;
			continue;
		}
		break;
	}
	for (int b = 0; b < nbatch; b++) /* treelikelihood.c:328-332 */
		if (isnan(lnl[b]) || isinf(lnl[b])) {
			if (grad_ratios)
				for (int i = 0; i < t->T - 1; i++) grad_ratios[(size_t)b * (t->T - 1) + i] = NAN;
			if (grad_rates)
				for (int i = 0; i < nrates; i++) grad_rates[(size_t)b * nrates + i] = NAN;
		}
	phb_tlk_update_all_nodes(t); /* device partials now belong to the last sample */
	return PHB_OK;
}

int phb_tlk_kernel_time(phb_tlk *t, double *total_ms, long long *launches) {
	int rc = phbc_kernel_time(t->ctx, total_ms, launches);
	if (rc) return dev_fail(rc);
	return PHB_OK;
}

long long phb_tlk_launch_count(const phb_tlk *t) { return phbc_launch_count(t->ctx); }

int phb_tlk_last_kernels(const phb_tlk *t) { return phbc_last_family(t->ctx); }

/* ------------------------------------------------------------------------------------------- */
/* NVTX ranges at the C-ABI entry points that do device work (SURVEY.md 5): an nsys / ncu timeline   */
/* shows one named range per call of the reference-facing API, with the kernels nested inside   */
/* ------------------------------------------------------------------------------------------- */
int phb_tlk_calculate(phb_tlk *t, double *lnl) {
	nvtxRangePushA("phb_tlk_calculate");
	const int rc = phb_tlk_calculate_impl(t, lnl);
	nvtxRangePop();
	return rc;
}

int phb_tlk_gradient(phb_tlk *t, const double **grad) {
	nvtxRangePushA("phb_tlk_gradient");
	const int rc = phb_tlk_gradient_impl(t, grad);
	nvtxRangePop();
	return rc;
}

int phb_tlk_gradient_batch(phb_tlk *t, int nbatch, const double *bl, double *lnl, double *grad) {
	nvtxRangePushA("phb_tlk_gradient_batch");
	const int rc = phb_tlk_gradient_batch_impl(t, nbatch, bl, lnl, grad);
	nvtxRangePop();
	return rc;
}

int phb_tlk_gradient_batch_time(phb_tlk *t, int nbatch, const double *ratios, const double *rates, int nrates, int include_jacobian,
                                double *lnl, double *log_jacobian, double *grad_ratios, double *grad_rates) {
	nvtxRangePushA("phb_tlk_gradient_batch_time");
	const int rc = phb_tlk_gradient_batch_time_impl(t, nbatch, ratios, rates, nrates, include_jacobian, lnl, log_jacobian, grad_ratios, grad_rates);
	nvtxRangePop();
	return rc;
}

int phb_tlk_matrix_gradient(phb_tlk *t, int nsets, const double *M, double *out) {
	nvtxRangePushA("phb_tlk_matrix_gradient");
	const int rc = phb_tlk_matrix_gradient_impl(t, nsets, M, out);
	nvtxRangePop();
	return rc;
}

int phb_tlk_calculate_branch(phb_tlk *t, int node, int nbl, const double *bl, double *lnl, double *dlnl, double *d2lnl) {
	nvtxRangePushA("phb_tlk_calculate_branch");
	const int rc = phb_tlk_calculate_branch_impl(t, node, nbl, bl, lnl, dlnl, d2lnl);
	nvtxRangePop();
	return rc;
}

int phb_tlk_branch_hessian_diagonal(phb_tlk *t, double *lnl, double *grad, double *hess) {
	nvtxRangePushA("phb_tlk_branch_hessian_diagonal");
	const int rc = phb_tlk_branch_hessian_diagonal_impl(t, lnl, grad, hess);
	nvtxRangePop();
	return rc;
}

int phb_tlk_nni_moves(phb_tlk *t, int *moves) { return phb_tlk_nni_moves_impl(t, moves); }

int phb_tlk_nni_scores(phb_tlk *t, int nmoves, const int *moves, const double *t_central, double *lnl, double *out) {
	nvtxRangePushA("phb_tlk_nni_scores");
	const int rc = phb_tlk_nni_scores_impl(t, nmoves, moves, t_central, lnl, out);
	nvtxRangePop();
	return rc;
}

int phb_tlk_spr_targets(phb_tlk *t, int s, int *targets) { return phb_tlk_spr_targets_impl(t, s, targets); }

int phb_tlk_spr_scores(phb_tlk *t, int s, int ntargets, const int *targets, const double *t_pendant, double *lnl, double *out) {
	nvtxRangePushA("phb_tlk_spr_scores");
	const int rc = phb_tlk_spr_scores_impl(t, s, ntargets, targets, t_pendant, lnl, out);
	nvtxRangePop();
	return rc;
}

int phb_tlk_update_uppers(phb_tlk *t) {
	nvtxRangePushA("phb_tlk_update_uppers");
	const int rc = phb_tlk_update_uppers_impl(t);
	nvtxRangePop();
	return rc;
}

int phb_tlk_gradient_device(phb_tlk *t, double *out_device) {
	nvtxRangePushA("phb_tlk_gradient_device");
	const int rc = phb_tlk_gradient_device_impl(t, out_device);
	nvtxRangePop();
	return rc;
}

int phb_tlk_gradient_allreduce_device(phb_tlk *t, phb_comm *comm, double **out_device) {
	nvtxRangePushA("phb_tlk_gradient_allreduce_device");
	const int rc = phb_tlk_gradient_allreduce_device_impl(t, comm, out_device);
	nvtxRangePop();
	return rc;
}

int phb_tlk_gradient_allreduce(phb_tlk *t, phb_comm *comm, double *lnl, const double **grad) {
	nvtxRangePushA("phb_tlk_gradient_allreduce");
	const int rc = phb_tlk_gradient_allreduce_impl(t, comm, lnl, grad);
	nvtxRangePop();
	return rc;
}

int phb_tlk_evaluate_launch(phb_tlk *t, int want_gradient) {
	nvtxRangePushA("phb_tlk_evaluate_launch");
	const int rc = phb_tlk_evaluate_launch_impl(t, want_gradient);
	nvtxRangePop();
	return rc;
}

int phb_tlk_update_partials(phb_tlk *t, int out, int p1, int m1, int p2, int m2, double *mirror) {
	nvtxRangePushA("phb_tlk_update_partials");
	const int rc = phb_tlk_update_partials_impl(t, out, p1, m1, p2, m2, mirror);
	nvtxRangePop();
	return rc;
}

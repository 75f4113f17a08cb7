// phb_cuda.cu -- device context, uploads, transition-matrix kernel and the generic
// node-at-a-time kernels (any state count) of the B200 tree-likelihood path.
//
// The generic kernels restate, one launch per tree level, what the reference does one node at a
// time through tlk->update_partials / integrate_partials / node_log_likelihoods /
// calculate_per_cat_partials (treelikelihood.h:90-111).  They materialise upper partials like the
// reference (treelikelihood.c:2129-2161) and are the fallback for state counts without a
// specialised path, for explicit (closed-form) matrices and for phb_tlk_get_partials.
// The fast paths live in phb_nuc4.cu (4 states) and phb_dmma.cu (20 / 61 states).
#include "phb_ctx.cuh"

#include <math.h>
#include <stdlib.h>
#include <string.h>

thread_local char phbc_errbuf[512] = "";

extern "C" const char *phbc_last_error(void) { return phbc_errbuf; }

extern "C" int phbc_device_count(void) {
	int n = 0;
	if (cudaGetDeviceCount(&n) != cudaSuccess) {
		cudaGetLastError();
		return 0;
	}
	return n;
}

// ---------------------------------------------------------------------------------------------
// context
// ---------------------------------------------------------------------------------------------

template <typename T>
static int dev_alloc(T **p, size_t count) {
	PHBC_CHECK(cudaMalloc((void **)p, count * sizeof(T) > 0 ? count * sizeof(T) : 8));
	return 0;
}

extern "C" phbc_ctx *phbc_create(int device, int ntips, int nstate, int ncat, int npatterns, int root, int tip_kind) {
	int ndev = phbc_device_count();
	if (ndev <= 0) {
		snprintf(phbc_errbuf, sizeof(phbc_errbuf), "no CUDA device visible: the B200 path has no CPU fallback");
		return NULL;
	}
	if (device < 0 || device >= ndev) {
		snprintf(phbc_errbuf, sizeof(phbc_errbuf), "device %d out of range (%d visible)", device, ndev);
		return NULL;
	}
	if (cudaSetDevice(device) != cudaSuccess) {
		snprintf(phbc_errbuf, sizeof(phbc_errbuf), "cudaSetDevice(%d) failed", device);
		return NULL;
	}
	phbc_ctx *ctx = (phbc_ctx *)calloc(1, sizeof(phbc_ctx));
	if (!ctx) return NULL;
	ctx->device = device;
	ctx->T = ntips;
	ctx->N = 2 * ntips - 1;
	ctx->S = nstate;
	ctx->C = ncat;
	ctx->P = npatterns;
	ctx->root = root;
	ctx->tip_kind = tip_kind;
	cudaDeviceProp prop;
	cudaGetDeviceProperties(&prop, device);
	ctx->num_sms = prop.multiProcessorCount;
	ctx->smem_optin = prop.sharedMemPerBlockOptin;
	ctx->smem_sm = prop.sharedMemPerMultiprocessor;
	const size_t S = nstate, C = ncat, P = npatterns, N = ctx->N, T = ntips;
	bool ok = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) == cudaSuccess;
	ok = ok && dev_alloc(&ctx->d_weights, P) == 0;
	ok = ok && dev_alloc(&ctx->d_evec, S * S) == 0 && dev_alloc(&ctx->d_ivec, S * S) == 0 && dev_alloc(&ctx->d_eval, S) == 0;
	ok = ok && dev_alloc(&ctx->d_qmat, S * S) == 0;
	ok = ok && dev_alloc(&ctx->d_freqs, S) == 0 && dev_alloc(&ctx->d_rates, C) == 0 && dev_alloc(&ctx->d_props, C) == 0;
	ok = ok && dev_alloc(&ctx->d_pattern_lnl, P) == 0;
	ok = ok && dev_alloc(&ctx->d_cat_grad, N * C) == 0;
	ctx->cat_grad_cap = 1;
	ctx->result_cap = 1;
	ok = ok && dev_alloc(&ctx->d_result, (size_t)ctx->result_cap * (1 + N)) == 0;
	// [lnL, gradient[N]] travels to the host as one block, also after a likelihood-only evaluation: the gradient slots must be defined
	ok = ok && cudaMemset(ctx->d_result, 0, (size_t)ctx->result_cap * (1 + N) * sizeof(double)) == cudaSuccess;
	ctx->bl_cap = 1;
	ok = ok && dev_alloc(&ctx->d_bl, N) == 0;
	ok = ok && cudaMallocHost((void **)&ctx->h_bl, N * sizeof(double)) == cudaSuccess;
	if (tip_kind == PHBC_TIP_STATES)
		ok = ok && dev_alloc(&ctx->d_tip_states, T * P) == 0;
	else
		ok = ok && dev_alloc(&ctx->d_tip_partials, T * P * S + 64) == 0 &&
		     cudaMemset(ctx->d_tip_partials, 0, (T * P * S + 64) * sizeof(double)) == cudaSuccess;  // zeroed tail, see phbc_generic_prepare
	if (!ok) {
		if (!phbc_errbuf[0]) snprintf(phbc_errbuf, sizeof(phbc_errbuf), "device allocation failed");
		phbc_destroy(ctx);
		return NULL;
	}
	return ctx;
}

extern "C" void phbc_destroy(phbc_ctx *ctx) {
	if (!ctx) return;
	cudaSetDevice(ctx->device);
	if (ctx->stream) cudaStreamSynchronize(ctx->stream);
	void *bufs[] = {ctx->d_sub_ops, ctx->d_branch, ctx->d_tip_states, ctx->d_tip_partials, ctx->d_weights, ctx->d_evec, ctx->d_eval, ctx->d_ivec, ctx->d_qmat,
	                ctx->d_freqs, ctx->d_rates, ctx->d_props, ctx->d_bl, ctx->d_P, ctx->d_dP, ctx->d_lower, ctx->d_upper,
	                ctx->d_sf, ctx->d_lower_ops, ctx->d_upper_ops, ctx->d_parent_ops, ctx->d_post_ops, ctx->d_pre_ops, ctx->d_walk_mats,
	                ctx->d_walk_lower, ctx->d_walk_gacc, ctx->d_pattern_lnl, ctx->d_result, ctx->d_cat_grad, ctx->d_scratch,
	                ctx->d_nuc4_codes, ctx->d_nuc4_bad, ctx->d_nuc4_cta_lnl, ctx->d_walk_gstat, ctx->d_nuc4_G, ctx->d_walk_hacc, ctx->d_nuc4_hess, ctx->d_ex, ctx->d_post_tip_order, ctx->d_pre_tip_order, ctx->d_dmma_img, ctx->d_tt_lowers, ctx->d_tt_topo, ctx->d_tt_bad,
	                ctx->d_tt_ratios, ctx->d_tt_rates, ctx->d_tt_heights, ctx->d_tt_adj, ctx->d_tt_out, ctx->d_reduce,
	                ctx->d_dw_post, ctx->d_dw_pre, ctx->d_dw_codes, ctx->d_dw_bad, ctx->d_dw_spill, ctx->d_enc_states, ctx->d_rowmax, ctx->d_upper_slot, ctx->d_cherry_tab, ctx->d_cherry_ops, ctx->d_cherry_enum, ctx->d_cherry_pairmax};
	for (size_t i = 0; i < sizeof(bufs) / sizeof(bufs[0]); i++)
		if (bufs[i]) cudaFree(bufs[i]);
	if (ctx->ev_beg) {
		for (int i = 0; i < ctx->ev_cap; i++) {
			cudaEventDestroy(ctx->ev_beg[i]);
			cudaEventDestroy(ctx->ev_end[i]);
		}
		free(ctx->ev_beg);
		free(ctx->ev_end);
	}
	if (ctx->h_bl) cudaFreeHost(ctx->h_bl);
	if (ctx->h_ex) cudaFreeHost(ctx->h_ex);
	if (ctx->h_tt) cudaFreeHost(ctx->h_tt);
	if (ctx->h_reduce) cudaFreeHost(ctx->h_reduce);
	if (ctx->h_result) cudaFreeHost(ctx->h_result);
	free(ctx->h_freqs);
	free(ctx->h_qmat);
	free(ctx->h_lower_level_off);
	free(ctx->h_upper_level_off);
	free(ctx->h_parent_level_off);
	free(ctx->h_lower_kind_off);
	free(ctx->h_parent_kind_off);
	if (ctx->stream) cudaStreamDestroy(ctx->stream);
	free(ctx);
}

int phbc_ensure_scratch(phbc_ctx *ctx, size_t bytes) {
	if (bytes <= ctx->scratch_bytes) return 0;
	PHBC_CHECK(cudaStreamSynchronize(ctx->stream));
	if (ctx->d_scratch) cudaFree(ctx->d_scratch);
	ctx->d_scratch = NULL;
	ctx->scratch_bytes = 0;
	PHBC_CHECK(cudaMalloc((void **)&ctx->d_scratch, bytes));
	ctx->scratch_bytes = bytes;
	return 0;
}

template <typename T>
static int upload_array(phbc_ctx *ctx, T **dst, const T *src, size_t count) {
	PHBC_CHECK(cudaSetDevice(ctx->device));
	if (*dst) {
		PHBC_CHECK(cudaStreamSynchronize(ctx->stream));
		cudaFree(*dst);
		*dst = NULL;
	}
	if (count == 0) return 0;
	PHBC_CHECK(cudaMalloc((void **)dst, count * sizeof(T)));
	PHBC_CHECK(cudaMemcpy(*dst, src, count * sizeof(T), cudaMemcpyHostToDevice));
	return 0;
}

// stable sort of each level's ops by the number of tip children; kind_off [levels][4] = absolute offsets of the kind groups
template <typename OP, typename F>
static OP *sort_levels_by_kind(const OP *ops, int nops, int nlevels, const int *level_off, int *kind_off, F tips_of) {
	OP *out = (OP *)malloc(sizeof(OP) * (nops > 0 ? nops : 1));
	if (!out) return NULL;
	for (int l = 0; l < nlevels; l++) {
		int w = level_off[l];
		for (int kind = 0; kind < 3; kind++) {
			kind_off[4 * l + kind] = w;
			for (int k = level_off[l]; k < level_off[l + 1]; k++)
				if (tips_of(ops[k]) == kind) out[w++] = ops[k];
		}
		kind_off[4 * l + 3] = w;
	}
	return out;
}

extern "C" int phbc_set_root(phbc_ctx *ctx, int root) {
	if (root < ctx->T || root >= ctx->N) {
		snprintf(phbc_errbuf, sizeof(phbc_errbuf), "root %d is not an internal node", root);
		return -1;
	}
	ctx->root = root;
	ctx->nuc4_G_valid = false;
	return 0;
}

extern "C" int phbc_set_schedule(phbc_ctx *ctx, const phbc_schedule *s) {
	int rc;
	const int T = ctx->T;
	free(ctx->h_lower_kind_off);
	free(ctx->h_parent_kind_off);
	ctx->h_lower_kind_off = (int *)malloc(sizeof(int) * 4 * (s->n_lower_levels + 1));
	ctx->h_parent_kind_off = (int *)malloc(sizeof(int) * 4 * (s->n_upper_levels + 1));
	phbc_op *lsorted = sort_levels_by_kind(s->lower_ops, s->n_lower_ops, s->n_lower_levels, s->lower_level_off, ctx->h_lower_kind_off,
	                                       [T](const phbc_op &o) { return (o.a < T ? 1 : 0) + (o.b >= 0 && o.b < T ? 1 : 0); });
	phbc_parent_op *psorted = sort_levels_by_kind(s->parent_ops, s->n_parent_ops, s->n_upper_levels, s->parent_level_off, ctx->h_parent_kind_off,
	                                              [T](const phbc_parent_op &o) { return (o.a < T ? 1 : 0) + (o.b < T ? 1 : 0); });
	if (!lsorted || !psorted || !ctx->h_lower_kind_off || !ctx->h_parent_kind_off) {
		free(lsorted), free(psorted);
		return -3;
	}
	rc = upload_array(ctx, &ctx->d_lower_ops, lsorted, (size_t)s->n_lower_ops);
	if (!rc) rc = upload_array(ctx, &ctx->d_parent_ops, psorted, (size_t)s->n_parent_ops);
	if (!rc) {  // where each child's row maxima sit in its parent's launch (rescaled tensor-core passes)
		int *slot = (int *)calloc((size_t)ctx->N, sizeof(int));
		if (!slot) rc = -3;
		for (int l = 0; !rc && l < s->n_upper_levels; l++)
			for (int k = s->parent_level_off[l]; k < s->parent_level_off[l + 1]; k++) {
				slot[psorted[k].a] = 2 * (k - s->parent_level_off[l]);
				slot[psorted[k].b] = 2 * (k - s->parent_level_off[l]) + 1;
			}
		if (!rc) rc = upload_array(ctx, &ctx->d_upper_slot, slot, (size_t)ctx->N);
		free(slot);
	}
	free(lsorted), free(psorted);
	if (rc) return rc;
	if ((rc = upload_array(ctx, &ctx->d_upper_ops, s->upper_ops, (size_t)s->n_upper_ops))) return rc;
	ctx->n_parent_ops = s->n_parent_ops;
	if ((rc = upload_array(ctx, &ctx->d_post_ops, s->post_ops, (size_t)s->n_post))) return rc;
	if ((rc = upload_array(ctx, &ctx->d_pre_ops, s->pre_ops, (size_t)s->n_pre))) return rc;
	if ((rc = upload_array(ctx, &ctx->d_post_tip_order, s->post_tip_order, (size_t)ctx->T))) return rc;
	if ((rc = upload_array(ctx, &ctx->d_pre_tip_order, s->pre_tip_order, (size_t)ctx->T))) return rc;
	ctx->post_first_tips = s->post_first_tips;
	ctx->pre_first_tips = s->pre_first_tips;
	ctx->nuc4_codes_valid = false;
	if ((rc = phbc_dwalk_set_schedule(ctx, s))) return rc;
	ctx->n_lower_ops = s->n_lower_ops;
	ctx->n_upper_ops = s->n_upper_ops;
	ctx->n_lower_levels = s->n_lower_levels;
	ctx->n_upper_levels = s->n_upper_levels;
	ctx->n_post = s->n_post;
	ctx->n_pre = s->n_pre;
	ctx->post_slots = s->post_slots;
	ctx->pre_slots = s->pre_slots;
	free(ctx->h_lower_level_off);
	free(ctx->h_upper_level_off);
	ctx->h_lower_level_off = (int *)malloc(sizeof(int) * (s->n_lower_levels + 1));
	ctx->h_upper_level_off = (int *)malloc(sizeof(int) * (s->n_upper_levels + 1));
	memcpy(ctx->h_lower_level_off, s->lower_level_off, sizeof(int) * (s->n_lower_levels + 1));
	memcpy(ctx->h_upper_level_off, s->upper_level_off, sizeof(int) * (s->n_upper_levels + 1));
	free(ctx->h_parent_level_off);
	ctx->h_parent_level_off = (int *)malloc(sizeof(int) * (s->n_upper_levels + 1));
	memcpy(ctx->h_parent_level_off, s->parent_level_off, sizeof(int) * (s->n_upper_levels + 1));
	return 0;
}

#define UPLOAD(dst, src, count)                                                                                \
	do {                                                                                                       \
		PHBC_CHECK(cudaSetDevice(ctx->device));                                                                \
		PHBC_CHECK(cudaMemcpyAsync(dst, src, (count) * sizeof(*(src)), cudaMemcpyHostToDevice, ctx->stream));  \
		PHBC_CHECK(cudaStreamSynchronize(ctx->stream));                                                        \
	} while (0)

extern "C" int phbc_upload_tip_states(phbc_ctx *ctx, const uint8_t *states) {
	if (!ctx->d_tip_states) return -1;
	ctx->nuc4_codes_valid = false;
	ctx->dw_codes_tp = 0;
	ctx->enc_states_valid = false;
	UPLOAD(ctx->d_tip_states, states, (size_t)ctx->T * ctx->P);
	return 0;
}
extern "C" int phbc_upload_tip_partials(phbc_ctx *ctx, const double *partials) {
	if (!ctx->d_tip_partials) return -1;
	ctx->nuc4_codes_valid = false;
	ctx->dw_codes_tp = 0;
	ctx->enc_states_valid = false;
	UPLOAD(ctx->d_tip_partials, partials, (size_t)ctx->T * ctx->P * ctx->S);
	return 0;
}
extern "C" int phbc_upload_weights(phbc_ctx *ctx, const double *w) {
	UPLOAD(ctx->d_weights, w, (size_t)ctx->P);
	return 0;
}
extern "C" int phbc_upload_eigen(phbc_ctx *ctx, const double *evec, const double *eval, const double *ivec) {
	const int S = ctx->S;
	UPLOAD(ctx->d_evec, evec, (size_t)S * S);
	UPLOAD(ctx->d_eval, eval, (size_t)S);
	UPLOAD(ctx->d_ivec, ivec, (size_t)S * S);
	// Q = V diag(lambda) V^-1, used by the fused kernels as dP/dt = Q P(t)
	double *q = (double *)malloc(sizeof(double) * S * S);
	for (int i = 0; i < S; i++)
		for (int j = 0; j < S; j++) {
			double acc = 0;
			for (int k = 0; k < S; k++) acc += evec[i * S + k] * eval[k] * ivec[k * S + j];
			q[i * S + j] = acc;
		}
	cudaError_t e = cudaMemcpyAsync(ctx->d_qmat, q, sizeof(double) * S * S, cudaMemcpyHostToDevice, ctx->stream);
	if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
	free(ctx->h_qmat);
	ctx->h_qmat = q;
	PHBC_CHECK(e);
	ctx->have_eigen = true;
	return 0;
}
extern "C" int phbc_upload_freqs(phbc_ctx *ctx, const double *freqs) {
	UPLOAD(ctx->d_freqs, freqs, (size_t)ctx->S);
	if (!ctx->h_freqs) ctx->h_freqs = (double *)malloc(sizeof(double) * ctx->S);
	memcpy(ctx->h_freqs, freqs, sizeof(double) * ctx->S);
	return 0;
}
extern "C" int phbc_upload_site_model(phbc_ctx *ctx, const double *rates, const double *props) {
	UPLOAD(ctx->d_rates, rates, (size_t)ctx->C);
	UPLOAD(ctx->d_props, props, (size_t)ctx->C);
	return 0;
}

static int ensure_node_matrices(phbc_ctx *ctx) {
	const size_t n = (size_t)ctx->N * ctx->C * ctx->S * ctx->S;
	if (!ctx->d_P) PHBC_CHECK(cudaMalloc((void **)&ctx->d_P, n * sizeof(double)));
	if (!ctx->d_dP) PHBC_CHECK(cudaMalloc((void **)&ctx->d_dP, n * sizeof(double)));
	return 0;
}

extern "C" int phbc_upload_matrices(phbc_ctx *ctx, const double *P, const double *dP) {
	PHBC_CHECK(cudaSetDevice(ctx->device));
	int rc = ensure_node_matrices(ctx);
	if (rc) return rc;
	const size_t n = (size_t)ctx->N * ctx->C * ctx->S * ctx->S;
	UPLOAD(ctx->d_P, P, n);
	UPLOAD(ctx->d_dP, dP, n);
	return 0;
}

// Device-to-device copy of the bulky inputs of `src` into `dst` (same shape; any pair of devices): tip states / partials,
// pattern weights, explicit matrices and the time-tree tables.  The small model inputs are re-uploaded by the host layer.
extern "C" int phbc_copy_inputs(phbc_ctx *dst, phbc_ctx *src, int matrices, int time_tree) {
	if (dst->T != src->T || dst->S != src->S || dst->C != src->C || dst->P != src->P || dst->tip_kind != src->tip_kind) {
		snprintf(phbc_errbuf, sizeof(phbc_errbuf), "phbc_copy_inputs: shapes differ");
		return -1;
	}
	phbc_ctx *ctx = src;
	PHBC_CHECK(cudaSetDevice(src->device));
	PHBC_CHECK(cudaStreamSynchronize(src->stream));
	ctx = dst;
	PHBC_CHECK(cudaSetDevice(dst->device));
	const size_t T = src->T, P = src->P, S = src->S, N = src->N, C = src->C;
	if (src->d_tip_states) PHBC_CHECK(cudaMemcpyPeerAsync(dst->d_tip_states, dst->device, src->d_tip_states, src->device, T * P, dst->stream));
	if (src->d_tip_partials)
		PHBC_CHECK(cudaMemcpyPeerAsync(dst->d_tip_partials, dst->device, src->d_tip_partials, src->device, T * P * S * sizeof(double), dst->stream));
	PHBC_CHECK(cudaMemcpyPeerAsync(dst->d_weights, dst->device, src->d_weights, src->device, P * sizeof(double), dst->stream));
	dst->nuc4_codes_valid = false;
	dst->dw_codes_tp = 0;
	dst->enc_states_valid = false;
	if (matrices && src->d_P && src->d_dP) {
		int rc = ensure_node_matrices(dst);
		if (rc) return rc;
		PHBC_CHECK(cudaMemcpyPeerAsync(dst->d_P, dst->device, src->d_P, src->device, N * C * S * S * sizeof(double), dst->stream));
		PHBC_CHECK(cudaMemcpyPeerAsync(dst->d_dP, dst->device, src->d_dP, src->device, N * C * S * S * sizeof(double), dst->stream));
	}
	if (time_tree && src->d_tt_lowers) {
		if (!dst->d_tt_lowers) {
			PHBC_CHECK(cudaMalloc((void **)&dst->d_tt_lowers, N * sizeof(double)));
			PHBC_CHECK(cudaMalloc((void **)&dst->d_tt_topo, 3 * N * sizeof(int)));
			PHBC_CHECK(cudaMalloc((void **)&dst->d_tt_bad, sizeof(int)));
		}
		PHBC_CHECK(cudaMemcpyPeerAsync(dst->d_tt_lowers, dst->device, src->d_tt_lowers, src->device, N * sizeof(double), dst->stream));
		PHBC_CHECK(cudaMemcpyPeerAsync(dst->d_tt_topo, dst->device, src->d_tt_topo, src->device, 3 * N * sizeof(int), dst->stream));
	}
	PHBC_CHECK(cudaStreamSynchronize(dst->stream));
	return 0;
}

// exp(eval[k] * bl[n] * rates[c]) for the branch lengths uploaded LAST, [N][C][S], computed by the host (see k_transition_matrices);
// valid until the next branch-length upload
extern "C" int phbc_upload_exponentials(phbc_ctx *ctx, const double *ex, int nbatch) {
	PHBC_CHECK(cudaSetDevice(ctx->device));
	const size_t n = (size_t)ctx->N * ctx->C * ctx->S * (size_t)nbatch;
	if (nbatch > ctx->ex_cap) {
		PHBC_CHECK(cudaStreamSynchronize(ctx->stream));
		if (ctx->d_ex) cudaFree(ctx->d_ex);
		if (ctx->h_ex) cudaFreeHost(ctx->h_ex);
		ctx->d_ex = ctx->h_ex = NULL;
		ctx->ex_cap = 0;
		PHBC_CHECK(cudaMalloc((void **)&ctx->d_ex, n * sizeof(double)));
		PHBC_CHECK(cudaMallocHost((void **)&ctx->h_ex, n * sizeof(double)));
		ctx->ex_cap = nbatch;
	}
	PHBC_CHECK(cudaStreamSynchronize(ctx->stream));  // the previous copy out of the pinned staging buffer
	memcpy(ctx->h_ex, ex, n * sizeof(double));
	PHBC_CHECK(cudaMemcpyAsync(ctx->d_ex, ctx->h_ex, n * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
	ctx->ex_count = nbatch;
	return 0;
}

// branch lengths as the device holds them (the time-tree chain builds them there): [nbatch][N], blocking
extern "C" int phbc_download_branch_lengths(phbc_ctx *ctx, int nbatch, double *bl) {
	PHBC_CHECK(cudaSetDevice(ctx->device));
	if (nbatch > ctx->bl_cap) return -1;
	PHBC_CHECK(cudaMemcpyAsync(bl, ctx->d_bl, (size_t)nbatch * ctx->N * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
	PHBC_CHECK(cudaStreamSynchronize(ctx->stream));
	return 0;
}

extern "C" int phbc_upload_branch_lengths(phbc_ctx *ctx, const double *bl, int nbatch) {
	PHBC_CHECK(cudaSetDevice(ctx->device));
	const size_t N = ctx->N;
	ctx->ex_count = 0;
	if (nbatch > ctx->bl_cap) {
		PHBC_CHECK(cudaStreamSynchronize(ctx->stream));
		cudaFree(ctx->d_bl);
		cudaFreeHost(ctx->h_bl);
		ctx->d_bl = NULL;
		ctx->h_bl = NULL;
		PHBC_CHECK(cudaMalloc((void **)&ctx->d_bl, (size_t)nbatch * N * sizeof(double)));
		PHBC_CHECK(cudaMallocHost((void **)&ctx->h_bl, (size_t)nbatch * N * sizeof(double)));
		ctx->bl_cap = nbatch;
	}
	if (nbatch > ctx->result_cap) {
		PHBC_CHECK(cudaStreamSynchronize(ctx->stream));
		cudaFree(ctx->d_result);
		ctx->d_result = NULL;
		PHBC_CHECK(cudaMalloc((void **)&ctx->d_result, (size_t)nbatch * (1 + N) * sizeof(double)));
		PHBC_CHECK(cudaMemset(ctx->d_result, 0, (size_t)nbatch * (1 + N) * sizeof(double)));
		ctx->result_cap = nbatch;
	}
	// the previous async copy out of the pinned staging buffer must have completed
	PHBC_CHECK(cudaStreamSynchronize(ctx->stream));
	memcpy(ctx->h_bl, bl, (size_t)nbatch * N * sizeof(double));
	PHBC_CHECK(cudaMemcpyAsync(ctx->d_bl, ctx->h_bl, (size_t)nbatch * N * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
	return 0;
}

// ---------------------------------------------------------------------------------------------
// transition matrices:  P(t) = |V exp(L t) V^-1|,  dP/dt = V L exp(L t) V^-1   (substmodel.c:518-557, 695-723)
// one CTA per (node, category)
// ---------------------------------------------------------------------------------------------

__global__ void k_transition_matrices(int S, int C, int root, const double *__restrict__ evec, const double *__restrict__ eval,
                                      const double *__restrict__ ivec, const double *__restrict__ bl,
                                      const double *__restrict__ rates, double *__restrict__ Pm, double *__restrict__ dPm,
                                      const double *__restrict__ ex_host /* [N][C][S] exp(eval * t) from the host's libm, or NULL */) {
	extern __shared__ double sm[];
	double *ex = sm;       // exp(lambda_k t)
	double *lex = sm + S;  // lambda_k exp(lambda_k t)
	const int node = blockIdx.x, c = blockIdx.y;
	if (node == root) return;
	const double t = bl[node] * rates[c];
	for (int k = threadIdx.x; k < S; k += blockDim.x) {
		const double l = eval[k];
		// 61-state models have transition probabilities of order t^2, t^3 (codons two or three changes apart) that come out of this sum
		// by cancellation: one ulp in an exponential moves them by 1e-9 relative, so parity with the reference at 1e-10 needs ITS exp
		// (the host's libm, phb_treelikelihood.c:upload_bl), not just an equally good one
		const double e = ex_host ? ex_host[((size_t)node * C + c) * S + k] : exp(l * t);
		ex[k] = e;
		lex[k] = l * e;
	}
	__syncthreads();
	const size_t base = ((size_t)node * C + c) * S * S;
	for (int e = threadIdx.x; e < S * S; e += blockDim.x) {
		const int i = e / S, j = e % S;
		double p = 0.0, d = 0.0;
		// same operation order and rounding as substmodel.c:539-555 (no fused multiply-add):
		// PP[k][j] = Invevec[k][j] * exp(.), P[i][j] = sum_k PP[k][j] * evec[i][k]
		for (int k = 0; k < S; k++) {
			const double iv = ivec[k * S + j], ev = evec[i * S + k];
			p = __dadd_rn(p, __dmul_rn(__dmul_rn(iv, ex[k]), ev));
			d = __dadd_rn(d, __dmul_rn(__dmul_rn(iv, lex[k]), ev));
		}
		Pm[base + e] = fabs(p);
		dPm[base + e] = d;
	}
}

// ---------------------------------------------------------------------------------------------
// generic kernels
// ---------------------------------------------------------------------------------------------

// patterns per CTA of k_generic_combine: few states => many patterns, so that a CTA amortises its matrix staging over ~2k outputs
static inline int gen_pblk(int S) { return S <= 8 ? 512 : (S <= 32 ? 128 : 32); }

// out = (M_a x_a) o (M_b x_b) [o pi]; grid (ceil(P/pblk), C, ops in level)   -- K1-K4, K8
__global__ void k_generic_combine(Bufs b, const phbc_op *__restrict__ ops, const double *__restrict__ Pm,
                                  const double *__restrict__ freqs, int pblk) {
	extern __shared__ double sm[];
	const int S = b.S, SS = S * S;
	double *mA = sm, *mB = sm + SS;
	const phbc_op op = ops[blockIdx.z];
	const int c = blockIdx.y;
	for (int e = threadIdx.x; e < SS; e += blockDim.x) {
		mA[e] = Pm[((size_t)op.a_mat * b.C + c) * SS + e];
		if (op.b >= 0) mB[e] = Pm[((size_t)op.b_mat * b.C + c) * SS + e];
	}
	__syncthreads();
	double *out = (double *)partial_ptr(b, op.out, c);
	const int p0 = blockIdx.x * pblk;
	for (int e = threadIdx.x; e < pblk * S; e += blockDim.x) {
		const int p = p0 + e / S, i = e % S;
		if (p >= b.P) break;
		double v = message(b, op.a, c, mA, p, i, true);
		if (op.b >= 0) v *= message(b, op.b, c, mB, p, i, true);
		if ((op.flags & 1) && freqs != NULL) v *= freqs[i];
		out[(size_t)p * S + i] = v;
	}
}

// SingleTreeLikelihood_scalePartials (treelikelihood.c:1790-1836); grid (ceil(P/128), ops in level)   -- K5
__global__ void k_generic_scale(Bufs b, const phbc_op *__restrict__ ops, double threshold) {
	const phbc_op op = ops[blockIdx.y];
	const int p = blockIdx.x * blockDim.x + threadIdx.x;
	if (p >= b.P) return;
	const int S = b.S;
	double m = 0.0;
	for (int c = 0; c < b.C; c++) {
		const double *x = partial_ptr(b, op.out, c) + (size_t)p * S;
		for (int i = 0; i < S; i++) m = x[i] > m ? x[i] : m;
	}
	double sf = 0.0;
	if (m < threshold && m > 0.0) {  // m == 0: nothing to rescale (an upper partial the fused gradient path never wrote)
		for (int c = 0; c < b.C; c++) {
			double *x = (double *)partial_ptr(b, op.out, c) + (size_t)p * S;
			for (int i = 0; i < S; i++) x[i] /= m;
		}
		sf = log(m);
	}
	// children that own partials carry scaling factors; state tips do not (treelikelihood.c:1795-1796)
	if (!is_state_tip(b, op.a)) sf += b.sf[(size_t)op.a * b.P + p];
	if (op.b >= 0 && !is_state_tip(b, op.b)) sf += b.sf[(size_t)op.b * b.P + p];
	b.sf[(size_t)op.out * b.P + p] = sf;
}

// the same with one thread per (pattern, category), the C lanes of a pattern side by side: four times the loads in flight of the
// one-thread-per-pattern form (19 of the 33.8 ms of a rescaled LG+G4 400 x 50k evaluation were this kernel), the maximum over the
// categories by a butterfly over the lane group.  Same values, same factors.
__global__ void k_generic_scale_split(Bufs b, const phbc_op *__restrict__ ops, double threshold) {
	__shared__ double m_s[128];
	const phbc_op op = ops[blockIdx.y];
	const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
	const int C = b.C, S = b.S;
	const int p = (int)(t / C), c = (int)(t - (size_t)p * C);
	const bool live = p < b.P;  // whole lane groups are live or not: P * C is a multiple of C
	double m = 0.0;
	if (live) {
		const double *x = partial_ptr(b, op.out, c) + (size_t)p * S;
		for (int i = 0; i < S; i++) m = x[i] > m ? x[i] : m;
	}
	for (int off = C >> 1; off > 0; off >>= 1) m = fmax(m, __shfl_xor_sync(0xffffffffu, m, off));
	const bool rescaled = live && m < threshold && m > 0.0;
	if (c == 0) m_s[threadIdx.x / C] = rescaled ? m : 0.0;
	if (__syncthreads_or(rescaled)) phbc_rescale_block(b, op.out, (int)((size_t)blockIdx.x * blockDim.x / C), blockDim.x / C, m_s);
	if (live && c == 0) {
		double sf = rescaled ? log(m) : 0.0;
		if (!is_state_tip(b, op.a)) sf += b.sf[(size_t)op.a * b.P + p];
		if (op.b >= 0 && !is_state_tip(b, op.b)) sf += b.sf[(size_t)op.b * b.P + p];
		b.sf[(size_t)op.out * b.P + p] = sf;
	}
}

// integrate_partials + node_log_likelihoods + weighted sum (treelikelihoodX.c:104-164, treelikelihood.c:1482-1487)  -- K6, K7
__global__ void k_generic_root(Bufs b, int root, const double *__restrict__ freqs, const double *__restrict__ props,
                               const double *__restrict__ weights, int scale, double *__restrict__ pattern_lnl,
                               double *__restrict__ block_sums) {
	__shared__ double red[32];
	const int p = blockIdx.x * blockDim.x + threadIdx.x;
	double v = 0.0;
	if (p < b.P) {
		const int S = b.S;
		double site = 0.0;
		for (int i = 0; i < S; i++) {
			double r = 0.0;
			for (int c = 0; c < b.C; c++) {
				const double x = partial_ptr(b, root, c)[(size_t)p * S + i];
				r += (b.C == 1) ? x : x * props[c];
			}
			site += freqs[i] * r;
		}
		double plk = log(site);
		if (scale) plk += b.sf[(size_t)root * b.P + p];
		pattern_lnl[p] = plk;
		v = plk * weights[p];
	}
	v = phb_warp_sum(v);
	if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
	__syncthreads();
	if (threadIdx.x < 32) {
		double s = threadIdx.x < (blockDim.x >> 5) ? red[threadIdx.x] : 0.0;
		s = phb_warp_sum(s);
		if (threadIdx.x == 0) block_sums[blockIdx.x] = s;
	}
}

// deterministic final sum of n values by one CTA: out[0] = sum
__global__ void k_sum_blocks(const double *__restrict__ in, int n, double *__restrict__ out) {
	__shared__ double red[32];
	double v = 0.0;
	for (int i = threadIdx.x; i < n; i += blockDim.x) v += in[i];
	v = phb_warp_sum(v);
	if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
	__syncthreads();
	if (threadIdx.x < 32) {
		double s = threadIdx.x < (blockDim.x >> 5) ? red[threadIdx.x] : 0.0;
		s = phb_warp_sum(s);
		if (threadIdx.x == 0) out[0] = s;
	}
}

#define GEN_MAXC 32
#define GEN_PGRAD 256

// calculate_branch_partials + gradient_cat_branch_lengths (treelikelihoodX.c:878-1001, treelikelihood.c:2793-2941,
// 2715-2789); grid (ceil(P/256), non-root nodes y0 .. y0 + gridDim.y - 1), one thread per pattern       -- K9, K10
__global__ void k_generic_branch_gradient(Bufs b, int root, int y0, const double *__restrict__ Pm, const double *__restrict__ dPm,
                                          const double *__restrict__ freqs, const double *__restrict__ props,
                                          const double *__restrict__ weights, const double *__restrict__ pattern_lnl,
                                          int scale, int compat, int include_root_freqs, double *__restrict__ partial /* [N][C][tiles] */) {
	extern __shared__ double sm[];
	__shared__ double red[GEN_PGRAD / 32];
	const int S = b.S, SS = S * S;
	double *dM = sm, *M = sm + SS;
	int node = y0 + blockIdx.y;
	if (node >= root) node++;  // skip the root
	const int p = blockIdx.x * blockDim.x + threadIdx.x;
	const bool live = p < b.P;
	double numc[GEN_MAXC], denc[GEN_MAXC];
	for (int c = 0; c < b.C; c++) {
		__syncthreads();
		for (int e = threadIdx.x; e < SS; e += blockDim.x) {
			dM[e] = dPm[((size_t)node * b.C + c) * SS + e];
			if (scale) M[e] = Pm[((size_t)node * b.C + c) * SS + e];
		}
		__syncthreads();
		double num = 0.0, den = 0.0;
		if (live) {
			const double *U = partial_ptr(b, b.N + node, c) + (size_t)p * S;
			for (int i = 0; i < S; i++) {
				const double f = include_root_freqs ? 1.0 : freqs[i];
				const double u = f * U[i];
				num += u * message(b, node, c, dM, p, i, false);
				if (scale) den += u * message(b, node, c, M, p, i, false);
			}
		}
		numc[c] = num;
		denc[c] = den;
	}
	double den_all = 0.0;
	if (scale && !compat)
		for (int c = 0; c < b.C; c++) den_all += (b.C == 1 ? 1.0 : props[c]) * denc[c];
	const double w = live ? weights[p] : 0.0;
	const double lk = (live && !scale) ? exp(pattern_lnl[p]) : 1.0;  // pattern_likelihoods, treelikelihood.c:3207-3210
	for (int c = 0; c < b.C; c++) {
		double v = 0.0;
		if (live) {
			const double den = !scale ? lk : (compat ? denc[c] : den_all);
			v = numc[c] / den * w;
		}
		v = phb_warp_sum(v);
		__syncthreads();
		if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
		__syncthreads();
		if (threadIdx.x < 32) {
			double s = threadIdx.x < (blockDim.x >> 5) ? red[threadIdx.x] : 0.0;
			s = phb_warp_sum(s);
			if (threadIdx.x == 0) partial[((size_t)node * b.C + c) * gridDim.x + blockIdx.x] = s;
		}
	}
}

// cat_grad[n][c] = sum over tiles (fixed order); one thread per (node, category)
// one warp per (node, category) row of `tiles` partial sums: lanes stride through the row (coalesced), then a butterfly -- a fixed
// order, so the result is reproducible run to run.  (One thread per row streamed 9.5 kB each from rows 9.5 kB apart: 115 us for the
// 1184-wide rows of the tensor-core walk, 3 % of a 25k-pattern evaluation.)
__global__ void k_generic_gradient_reduce(int N, int C, int root, int tiles, const double *__restrict__ partial,
                                          double *__restrict__ cat_grad) {
	const int e = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
	if (e >= N * C) return;
	const int node = e / C;
	double s = 0.0;
	if (node != root)
		for (int t = lane; t < tiles; t += 32) s += partial[(size_t)e * tiles + t];
	s = phb_warp_sum(s);
	if (lane == 0) cat_grad[e] = s;
}

// gradient_branch_length_from_cat_inplace (treelikelihood.c:3129-3143): applied only when C > 1 (:3258-3266)
__global__ void k_collapse_categories(int N, int C, const double *__restrict__ cat_grad, const double *__restrict__ props,
                                      const double *__restrict__ rates, double *__restrict__ result /* [1+N] */) {
	const int n = blockIdx.x * blockDim.x + threadIdx.x;
	if (n >= N) return;
	double g;
	if (C == 1) {
		g = cat_grad[n];
	} else {
		g = cat_grad[(size_t)n * C] * props[0] * rates[0];
		for (int c = 1; c < C; c++) g += cat_grad[(size_t)n * C + c] * props[c] * rates[c];
	}
	result[1 + n] = g;
}

Bufs phbc_make_bufs(phbc_ctx *ctx) {
	Bufs b;
	b.tip_states = ctx->d_tip_states;
	b.tip_partials = ctx->d_tip_partials;
	b.lower = ctx->d_lower;
	b.upper = ctx->d_upper;
	b.sf = ctx->d_sf;
	b.T = ctx->T;
	b.N = ctx->N;
	b.S = ctx->S;
	b.C = ctx->C;
	b.P = ctx->P;
	b.tip_kind = ctx->tip_kind;
	return b;
}

static int phbc_launch_transition_matrices(phbc_ctx *ctx, int batch_index) {
	int rc = ensure_node_matrices(ctx);
	if (rc) return rc;
	const int S = ctx->S;
	dim3 grid(ctx->N, ctx->C);
	const int threads = S * S >= 256 ? 256 : (S * S >= 64 ? 64 : 32);
	k_transition_matrices<<<grid, threads, 2 * S * sizeof(double), ctx->stream>>>(
	    S, ctx->C, ctx->root, ctx->d_evec, ctx->d_eval, ctx->d_ivec, ctx->d_bl + (size_t)batch_index * ctx->N, ctx->d_rates,
	    ctx->d_P, ctx->d_dP, batch_index < ctx->ex_count ? ctx->d_ex + (size_t)batch_index * ctx->N * ctx->C * S : NULL);
	ctx->launches++;
	PHBC_CHECK(cudaGetLastError());
	return 0;
}

extern "C" int phbc_smem_check(const phbc_ctx *ctx, const char *what, int nmat) {
	const size_t need = (size_t)nmat * ctx->S * ctx->S * sizeof(double);
	if (need <= ctx->smem_optin) return 0;
	snprintf(phbc_errbuf, sizeof(phbc_errbuf), "%s: %d states need %zu bytes of shared memory for %d matrices (at most %zu)", what, ctx->S, need, nmat,
	         ctx->smem_optin);
	return -1;
}

int phbc_alloc(phbc_ctx *ctx, double **p, size_t count, bool zero) {
	const cudaError_t e = cudaMalloc((void **)p, count * sizeof(double));
	if (e == cudaErrorMemoryAllocation) {
		(void)cudaGetLastError();
		*p = NULL;
		snprintf(phbc_errbuf, sizeof(phbc_errbuf), "out of device memory: %.2f GB requested", count * 8.0 / 1e9);
		return -3;
	}
	PHBC_CHECK(e);
	if (zero) PHBC_CHECK(cudaMemsetAsync(*p, 0, count * sizeof(double), ctx->stream));
	return 0;
}

// buffers of the node-at-a-time paths (lazy) and the per-node transition matrices
int phbc_generic_buffers(phbc_ctx *ctx, const phbc_eval_opts *o) {
	PHBC_CHECK(cudaSetDevice(ctx->device));
	const size_t S = ctx->S, C = ctx->C, P = ctx->P, N = ctx->N, T = ctx->T;
	const size_t psize = C * P * S;
	// zero-initialised, with a zeroed tail: the tensor-core kernels stage whole k-chunks without predicates and may read a few
	// doubles past a row (into the next row / block) -- always finite values that meet zero-padded matrix columns
	const size_t tail = 64;
	int rc;
	if (!ctx->d_lower && (rc = phbc_alloc(ctx, &ctx->d_lower, (N - T) * psize + tail, true))) return rc;
	if (o->want_gradient && !ctx->d_upper && (rc = phbc_alloc(ctx, &ctx->d_upper, N * psize + tail, true))) return rc;
	if (o->scale && !ctx->d_sf && (rc = phbc_alloc(ctx, &ctx->d_sf, 2 * N * P, true))) return rc;
	return 0;
}

int phbc_generic_prepare(phbc_ctx *ctx, const phbc_eval_opts *o) {
	int brc = phbc_generic_buffers(ctx, o);
	if (brc) return brc;
	if (!o->explicit_matrices) {
		if (!ctx->have_eigen) {
			snprintf(phbc_errbuf, sizeof(phbc_errbuf), "no eigen system and no explicit matrices set");
			return -4;
		}
		return phbc_launch_transition_matrices(ctx, o->batch_index);
	}
	if (!ctx->d_P) {
		snprintf(phbc_errbuf, sizeof(phbc_errbuf), "explicit matrices requested but not uploaded");
		return -4;
	}
	return 0;
}

int phbc_generic_scale_ops(phbc_ctx *ctx, const phbc_op *d_ops, int count, double threshold) {
	Bufs b = phbc_make_bufs(ctx);
	const int C = ctx->C;
	const bool split = C <= 32 && (C & (C - 1)) == 0 && C > 1;  // one thread per (pattern, category): a power of two categories per lane group
	for (int z0 = 0; z0 < count; z0 += 65535) {
		const int zc = count - z0 < 65535 ? count - z0 : 65535;
		if (split) k_generic_scale_split<<<dim3((unsigned)(((size_t)ctx->P * C + 127) / 128), zc), 128, 0, ctx->stream>>>(b, d_ops + z0, threshold);
		else k_generic_scale<<<dim3((unsigned)((ctx->P + 127) / 128), zc), 128, 0, ctx->stream>>>(b, d_ops + z0, threshold);
		ctx->launches++;
	}
	PHBC_CHECK(cudaGetLastError());
	return 0;
}

int phbc_generic_root(phbc_ctx *ctx, const phbc_eval_opts *o, double *result) {
	Bufs b = phbc_make_bufs(ctx);
	const int rblocks = (ctx->P + 255) / 256;
	int rc;
	if ((rc = phbc_ensure_scratch(ctx, rblocks * sizeof(double)))) return rc;
	k_generic_root<<<rblocks, 256, 0, ctx->stream>>>(b, ctx->root, ctx->d_freqs, ctx->d_props, ctx->d_weights, o->scale,
	                                                  ctx->d_pattern_lnl, ctx->d_scratch);
	k_sum_blocks<<<1, 256, 0, ctx->stream>>>(ctx->d_scratch, rblocks, result);
	ctx->launches += 2;
	PHBC_CHECK(cudaGetLastError());
	return 0;
}

int phbc_gradient_from_partials(phbc_ctx *ctx, int tiles, double *result) {
	const int N = ctx->N, C = ctx->C;
	k_generic_gradient_reduce<<<(unsigned)(((size_t)N * C * 32 + 127) / 128), 128, 0, ctx->stream>>>(N, C, ctx->root, tiles, ctx->d_scratch, ctx->d_cat_grad);
	k_collapse_categories<<<(unsigned)((N + 127) / 128), 128, 0, ctx->stream>>>(N, C, ctx->d_cat_grad, ctx->d_props, ctx->d_rates, result);
	ctx->launches += 2;
	PHBC_CHECK(cudaGetLastError());
	return 0;
}

// k_generic_branch_gradient with dPm in the place of dP/dt over every non-root node into the [N][C][tiles] scratch: the nodes on grid.y,
// in launches of at most 65,535
static int gen_branch_gradient(phbc_ctx *ctx, const double *dPm, int scale, int compat, int include_root_freqs) {
	const size_t S = ctx->S, gtiles = ((size_t)ctx->P + GEN_PGRAD - 1) / GEN_PGRAD;
	const size_t smem = 2 * S * S * sizeof(double);
	if (smem > 48 * 1024) PHBC_CHECK(cudaFuncSetAttribute(k_generic_branch_gradient, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
	Bufs b = phbc_make_bufs(ctx);
	for (int y0 = 0; y0 < ctx->N - 1; y0 += 65535) {
		const int cnt = ctx->N - 1 - y0 < 65535 ? ctx->N - 1 - y0 : 65535;
		k_generic_branch_gradient<<<dim3((unsigned)gtiles, (unsigned)cnt), GEN_PGRAD, smem, ctx->stream>>>(
		    b, ctx->root, y0, ctx->d_P, dPm, ctx->d_freqs, ctx->d_props, ctx->d_weights, ctx->d_pattern_lnl, scale, compat, include_root_freqs,
		    ctx->d_scratch);
		ctx->launches++;
	}
	return 0;
}

int phbc_generic_gradient(phbc_ctx *ctx, const phbc_eval_opts *o, double *result) {
	const size_t C = ctx->C, P = ctx->P, N = ctx->N;
	const size_t gtiles = (P + GEN_PGRAD - 1) / GEN_PGRAD;
	int rc;
	if ((rc = phbc_ensure_scratch(ctx, N * C * gtiles * sizeof(double)))) return rc;
	if ((rc = gen_branch_gradient(ctx, ctx->d_dP, o->scale, o->compat_scaled_gradient, o->include_root_freqs))) return rc;
	return phbc_gradient_from_partials(ctx, (int)gtiles, result);
}

int phbc_generic_evaluate(phbc_ctx *ctx, const phbc_eval_opts *o) {
	const size_t S = ctx->S, C = ctx->C, P = ctx->P, N = ctx->N;
	if (C > GEN_MAXC) {
		snprintf(phbc_errbuf, sizeof(phbc_errbuf), "generic kernels support at most %d rate categories", GEN_MAXC);
		return -1;
	}
	int rc;
	if ((rc = phbc_smem_check(ctx, "generic kernels", 2))) return rc;
	if ((rc = phbc_generic_prepare(ctx, o))) return rc;
	ctx->lower_is_message = false;
	ctx->node_evals++;
	Bufs b = phbc_make_bufs(ctx);
	const size_t smem = 2 * S * S * sizeof(double);
	if (smem > 48 * 1024) PHBC_CHECK(cudaFuncSetAttribute(k_generic_combine, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
	const int pblk = gen_pblk((int)S), ptiles = (int)((P + pblk - 1) / pblk);
	if ((rc = phbc_time_begin(ctx))) return rc;
	// post-order, one launch per level
	for (int l = 0; l < ctx->n_lower_levels; l++) {
		const int beg = ctx->h_lower_level_off[l], cnt = ctx->h_lower_level_off[l + 1] - beg;
		if (cnt <= 0) continue;
		for (int z0 = 0; z0 < cnt; z0 += 65535) {
			const int zc = cnt - z0 < 65535 ? cnt - z0 : 65535;
			k_generic_combine<<<dim3(ptiles, (unsigned)C, zc), 128, smem, ctx->stream>>>(b, ctx->d_lower_ops + beg + z0, ctx->d_P, ctx->d_freqs, pblk);
			ctx->launches++;
		}
		if (o->scale && (rc = phbc_generic_scale_ops(ctx, ctx->d_lower_ops + beg, cnt, o->scaling_threshold))) return rc;
	}
	double *result = ctx->d_result + (size_t)o->batch_index * (1 + N);
	if ((rc = phbc_generic_root(ctx, o, result))) return rc;
	if (o->want_gradient) {
		for (int l = 0; l < ctx->n_upper_levels; l++) {
			const int beg = ctx->h_upper_level_off[l], cnt = ctx->h_upper_level_off[l + 1] - beg;
			if (cnt <= 0) continue;
			for (int z0 = 0; z0 < cnt; z0 += 65535) {
				const int zc = cnt - z0 < 65535 ? cnt - z0 : 65535;
				// op.flags bit 0 asks for the root frequencies; they are applied only under include_root_freqs
				k_generic_combine<<<dim3(ptiles, (unsigned)C, zc), 128, smem, ctx->stream>>>(b, ctx->d_upper_ops + beg + z0, ctx->d_P,
				                                                                           o->include_root_freqs ? ctx->d_freqs : NULL, pblk);
				ctx->launches++;
			}
			if (o->scale && (rc = phbc_generic_scale_ops(ctx, ctx->d_upper_ops + beg, cnt, o->scaling_threshold))) return rc;
		}
		if ((rc = phbc_generic_gradient(ctx, o, result))) return rc;
	}
	if ((rc = phbc_time_end(ctx))) return rc;
	PHBC_CHECK(cudaGetLastError());
	return 0;
}

// out[k] = sum over nodes n (not the root, not `skip`) and categories of props[c] * cat[k][n][c]  -- one block per set, fixed order
__global__ void k_matrix_gradient_sum(int N, int C, int root, int skip, const double *__restrict__ cat /* [nsets][N][C] */,
                                      const double *__restrict__ props, double *__restrict__ out) {
	__shared__ double red[256];
	const double *g = cat + (size_t)blockIdx.x * N * C;
	double s = 0.0;
	for (int e = threadIdx.x; e < N * C; e += blockDim.x) {
		const int n = e / C, c = e - n * C;
		if (n != root && n != skip) s += g[e] * (C == 1 ? 1.0 : props[c]);
	}
	red[threadIdx.x] = s;
	__syncthreads();
	for (int w = blockDim.x / 2; w > 0; w >>= 1) {
		if (threadIdx.x < w) red[threadIdx.x] += red[threadIdx.x + w];
		__syncthreads();
	}
	if (threadIdx.x == 0) out[blockIdx.x] = red[0];
}

/*
 * Node sweep of calculate_dlnl_dQ (treelikelihood.c:2337-2583): for each of `nsets` per-node matrix sets M (e.g. dP/d theta from
 * m->dPdp), out[k] = sum_n sum_p w_p / L_p sum_c prop_c sum_i f_i U_n[c,p,i] (M_k[n,c] L_n[c,p])_i over the non-root nodes
 * (and not `skip_node`: the root's right child of an unrooted tree, :2408).  Needs materialised upper partials, so the
 * evaluation runs on the node-at-a-time kernels (tensor-core lower / upper kernels for 20 / 61 states).
 */
extern "C" int phbc_matrix_gradient(phbc_ctx *ctx, const phbc_eval_opts *o, int nsets, const double *M_host, int skip_node, double *lnl,
                                    double *out_host) {
	PHBC_CHECK(cudaSetDevice(ctx->device));
	const size_t S = ctx->S, C = ctx->C, P = ctx->P, N = ctx->N;
	if (C > GEN_MAXC) {
		snprintf(phbc_errbuf, sizeof(phbc_errbuf), "generic kernels support at most %d rate categories", GEN_MAXC);
		return -1;
	}
	phbc_eval_opts e = *o;
	e.want_gradient = 1;
	e.materialize_uppers = 1;
	e.batch_count = 1;
	// 4 states, unscaled: the fused walk accumulates the per-branch statistics every set contracts with -- no materialised uppers
	ctx->nuc4_G_valid = false;
	{
		const int frc = phbc_nuc4_matrix_gradient(ctx, &e, nsets, M_host, skip_node, lnl, out_host);
		if (frc != 1) return frc;
	}
	const bool tensor = phbc_dmma_supported(ctx, &e) && e.kernels != 1;
	int rc;
	if (!tensor && (rc = phbc_smem_check(ctx, "generic kernels", 2))) return rc;
	ctx->last_family = tensor ? 3 : 1;
	rc = 0;
	const size_t set = N * C * S * S;
	double *d_M = NULL, *d_cat = NULL, *d_out = NULL;
	cudaError_t err = cudaMalloc((void **)&d_M, (size_t)nsets * set * sizeof(double));
	if (err == cudaSuccess) err = cudaMalloc((void **)&d_cat, (size_t)nsets * N * C * sizeof(double));
	if (err == cudaSuccess) err = cudaMalloc((void **)&d_out, (size_t)nsets * sizeof(double));
	if (err == cudaSuccess) err = cudaMemcpyAsync(d_M, M_host, (size_t)nsets * set * sizeof(double), cudaMemcpyHostToDevice, ctx->stream);
	if (err == cudaSuccess && tensor) {
		// 20 / 60..63 states: the forward phase once, one tensor-core gradient phase per set with the set in the place of dP/dt; no
		// materialised upper partials, no scalar S^2 products (round 2: GY94 100 x 250k, 2 sets, 899 ms -> see profiles/)
		rc = phbc_dmma_matrix_gradient(ctx, &e, nsets, d_M, d_cat);
		if (!rc) {
			k_matrix_gradient_sum<<<nsets, 256, 0, ctx->stream>>>((int)N, (int)C, ctx->root, skip_node, d_cat, ctx->d_props, d_out);
			ctx->launches++;
			err = cudaMemcpyAsync(out_host, d_out, (size_t)nsets * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream);
			if (err == cudaSuccess && lnl)
				err = cudaMemcpyAsync(lnl, ctx->d_result + (size_t)e.batch_index * (1 + N), sizeof(double), cudaMemcpyDeviceToHost, ctx->stream);
		}
		if (err == cudaSuccess) err = cudaStreamSynchronize(ctx->stream);
		if (err == cudaSuccess) err = cudaGetLastError();
		cudaFree(d_M), cudaFree(d_cat), cudaFree(d_out);
		if (rc) return rc;
		PHBC_CHECK(err);
		return 0;
	}
	if (err == cudaSuccess) rc = phbc_generic_evaluate(ctx, &e);
	if (rc) {
		cudaFree(d_M), cudaFree(d_cat), cudaFree(d_out);
		return rc;
	}
	const size_t gtiles = (P + GEN_PGRAD - 1) / GEN_PGRAD;
	if (err == cudaSuccess) {
		rc = phbc_ensure_scratch(ctx, N * C * gtiles * sizeof(double));
		for (int k = 0; k < nsets && !rc && err == cudaSuccess; k++) {
			rc = gen_branch_gradient(ctx, d_M + (size_t)k * set, e.scale, 0 /* one site denominator: dlikelihood / likelihood, :2464-2474 */,
			                         e.include_root_freqs);
			if (rc) break;
			k_generic_gradient_reduce<<<(unsigned)(((size_t)N * C * 32 + 127) / 128), 128, 0, ctx->stream>>>((int)N, (int)C, ctx->root, (int)gtiles, ctx->d_scratch,
			                                                                                 d_cat + (size_t)k * N * C);
			ctx->launches++;
		}
		if (!rc && err == cudaSuccess) {
			k_matrix_gradient_sum<<<nsets, 256, 0, ctx->stream>>>((int)N, (int)C, ctx->root, skip_node, d_cat, ctx->d_props, d_out);
			ctx->launches++;
			err = cudaMemcpyAsync(out_host, d_out, (size_t)nsets * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream);
			if (err == cudaSuccess && lnl)
				err = cudaMemcpyAsync(lnl, ctx->d_result + (size_t)e.batch_index * (1 + N), sizeof(double), cudaMemcpyDeviceToHost, ctx->stream);
		}
	}
	if (err == cudaSuccess) err = cudaStreamSynchronize(ctx->stream);
	if (err == cudaSuccess) err = cudaGetLastError();
	cudaFree(d_M), cudaFree(d_cat), cudaFree(d_out);
	if (rc) return rc;
	PHBC_CHECK(err);
	return 0;
}


/*
 * Partial re-evaluation on the resident node-at-a-time buffers: the dirty-flag traversal of _calculate_partials
 * (treelikelihood.c:1645-1734) and update_upper_partials2 (:2164-2190) as explicit op lists.  `ops` (host) is grouped by level
 * (level_off[nlevels + 1]); ops of one level are independent, levels run in order.  Lower ops (out < N) are followed by the root
 * integration when do_root; upper ops (out >= N) leave their results in the upper buffers.  Transition matrices of ALL nodes are
 * rebuilt from the uploaded branch lengths first when rebuild_matrices (N x C tiny CTAs: cheaper than tracking a subset).
 */
extern "C" int phbc_run_ops(phbc_ctx *ctx, const phbc_eval_opts *o, int nops, const phbc_op *ops, int nlevels, const int *level_off,
                            int rebuild_matrices, int do_root, double *lnl_host) {
	PHBC_CHECK(cudaSetDevice(ctx->device));
	const size_t S = ctx->S, C = ctx->C, P = ctx->P, N = ctx->N;
	int rc;
	if ((rc = phbc_smem_check(ctx, "generic kernels", 2))) return rc;
	phbc_eval_opts e = *o;
	e.batch_index = 0;
	e.batch_count = 1;
	ctx->nuc4_G_valid = false;
	for (int k = 0; k < nops; k++)
		if (ops[k].out >= (int)N) e.want_gradient = 1;  // upper buffers are needed
	if ((rc = phbc_generic_buffers(ctx, &e))) return rc;
	const bool dmma = e.kernels != 1 && phbc_dmma_supported(ctx, &e);
	ctx->last_family = 1;  // the op lists run on the node-at-a-time buffers and matrices (tensor-core products where the shape allows)
	if (rebuild_matrices) {
		if (!e.explicit_matrices) {
			if (!ctx->have_eigen) {
				snprintf(phbc_errbuf, sizeof(phbc_errbuf), "no eigen system and no explicit matrices set");
				return -4;
			}
			if ((rc = phbc_launch_transition_matrices(ctx, 0))) return rc;
		}
		if (dmma && (rc = phbc_dmma_pack(ctx))) return rc;
	}
	if (nops > 0) {
		// within a level: ops the tensor-core kernel takes (two operands, no frequency factor) first, the rest after them
		phbc_op *sorted = (phbc_op *)malloc(sizeof(phbc_op) * nops);
		int *split = (int *)malloc(sizeof(int) * (nlevels > 0 ? nlevels : 1));
		if (!sorted || !split) {
			free(sorted), free(split);
			return -3;
		}
		for (int l = 0; l < nlevels; l++) {
			int w = level_off[l];
			for (int pass = 0; pass < 2; pass++)
				for (int k = level_off[l]; k < level_off[l + 1]; k++) {
					const bool fast = dmma && ops[k].b >= 0 && !((ops[k].flags & 1) && e.include_root_freqs);
					if (fast == (pass == 0)) sorted[w++] = ops[k];
				}
			split[l] = level_off[l];
			for (int k = level_off[l]; k < level_off[l + 1]; k++)
				if (dmma && sorted[k].b >= 0 && !((sorted[k].flags & 1) && e.include_root_freqs)) split[l] = k + 1;
		}
		if (nops > ctx->sub_ops_cap) {
			PHBC_CHECK(cudaStreamSynchronize(ctx->stream));
			if (ctx->d_sub_ops) cudaFree(ctx->d_sub_ops);
			ctx->d_sub_ops = NULL;
			ctx->sub_ops_cap = 0;
			const int cap = nops > 2 * (int)N ? nops : 2 * (int)N;
			cudaError_t err = cudaMalloc((void **)&ctx->d_sub_ops, sizeof(phbc_op) * cap);
			if (err != cudaSuccess) {
				free(sorted), free(split);
				PHBC_CHECK(err);
			}
			ctx->sub_ops_cap = cap;
		}
		cudaError_t err = cudaMemcpyAsync(ctx->d_sub_ops, sorted, sizeof(phbc_op) * nops, cudaMemcpyHostToDevice, ctx->stream);
		if (err == cudaSuccess) err = cudaStreamSynchronize(ctx->stream);  // `sorted` is pageable and freed below
		free(sorted);
		if (err != cudaSuccess) {
			free(split);
			PHBC_CHECK(err);
		}
		Bufs b = phbc_make_bufs(ctx);
		const size_t smem = 2 * S * S * sizeof(double);
		if (smem > 48 * 1024) PHBC_CHECK(cudaFuncSetAttribute(k_generic_combine, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
		const int pblk = gen_pblk((int)S), ptiles = (int)((P + pblk - 1) / pblk);
		rc = 0;
		for (int l = 0; l < nlevels && !rc; l++) {
			const int beg = level_off[l], end = level_off[l + 1], mid = split[l];
			if (end <= beg) continue;
			if (mid > beg) rc = phbc_dmma_lower_ops(ctx, ctx->d_sub_ops + beg, mid - beg);
			for (int z0 = mid; z0 < end && !rc; z0 += 65535) {
				const int zc = end - z0 < 65535 ? end - z0 : 65535;
				k_generic_combine<<<dim3(ptiles, (unsigned)C, zc), 128, smem, ctx->stream>>>(b, ctx->d_sub_ops + z0, ctx->d_P,
				                                                                           e.include_root_freqs ? ctx->d_freqs : NULL, pblk);
				ctx->launches++;
			}
			if (!rc && e.scale) rc = phbc_generic_scale_ops(ctx, ctx->d_sub_ops + beg, end - beg, e.scaling_threshold);
		}
		free(split);
		if (rc) return rc;
	}
	if (do_root) {
		if ((rc = phbc_generic_root(ctx, &e, ctx->d_result))) return rc;
		if (lnl_host) {
			PHBC_CHECK(cudaMemcpyAsync(lnl_host, ctx->d_result, sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
			PHBC_CHECK(cudaStreamSynchronize(ctx->stream));
		}
	}
	PHBC_CHECK(cudaGetLastError());
	return 0;
}

// d lnL / d pi_i at fixed partials: G_i = sum_k w_k R[k,i] / L_k with R the category-integrated root partials -- the "root term" of the
// frequency parameters in calculate_dlnl_dQ (treelikelihood.c:2371-2404); under rescaling R and L_k carry the same factor (:2384-2392).
// grid (pattern tiles, S); partial [S][tiles]
__global__ void k_root_freq_gradient(Bufs b, int root, const double *__restrict__ freqs, const double *__restrict__ props,
                                     const double *__restrict__ weights, double *__restrict__ partial) {
	__shared__ double red[8];
	const int S = b.S, i = blockIdx.y;
	const int p = blockIdx.x * blockDim.x + threadIdx.x;
	double v = 0.0;
	if (p < b.P) {
		double L = 0.0, Ri = 0.0;
		for (int j = 0; j < S; j++) {
			double r = 0.0;
			for (int c = 0; c < b.C; c++) {
				const double x = partial_ptr(b, root, c)[(size_t)p * S + j];
				r += (b.C == 1) ? x : x * props[c];
			}
			L += freqs[j] * r;
			if (j == i) Ri = r;
		}
		v = weights[p] * Ri / L;
	}
	v = phb_warp_sum(v);
	if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
	__syncthreads();
	if (threadIdx.x == 0) {
		double s = 0.0;
		for (int w = 0; w < (int)(blockDim.x >> 5); w++) s += red[w];
		partial[(size_t)i * gridDim.x + blockIdx.x] = s;
	}
}
// d lnL / d prop_c at fixed conditional likelihoods: A_c = sum_k w_k S_c(k) / L_k with S_c(k) = sum_i pi_i L_root[c,k,i] and
// L_k = sum_c prop_c S_c(k) -- the root term of the invariant-site proportion in gradient_pinv_sitemodel / gradient_pinv_W_sitemodel
// (treelikelihood.c:2943-3001: sum_k w_k sum_i pi_i (R_0 - R_1)[k,i] / L_k = A_0 - A_1).  Numerator and denominator come from the same
// (possibly rescaled) root partial.  grid (pattern tiles, C); partial [C][tiles]
__global__ void k_root_cat_gradient(Bufs b, int root, const double *__restrict__ freqs, const double *__restrict__ props,
                                    const double *__restrict__ weights, double *__restrict__ partial) {
	__shared__ double red[8];
	const int S = b.S, cc = blockIdx.y;
	const int p = blockIdx.x * blockDim.x + threadIdx.x;
	double v = 0.0;
	if (p < b.P) {
		double L = 0.0, Sc = 0.0;
		for (int c = 0; c < b.C; c++) {
			const double *x = partial_ptr(b, root, c) + (size_t)p * S;
			double s = 0.0;
			for (int j = 0; j < S; j++) s += freqs[j] * x[j];
			L += (b.C == 1) ? s : s * props[c];
			if (c == cc) Sc = s;
		}
		v = weights[p] * Sc / L;
	}
	v = phb_warp_sum(v);
	if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
	__syncthreads();
	if (threadIdx.x == 0) {
		double s = 0.0;
		for (int w = 0; w < (int)(blockDim.x >> 5); w++) s += red[w];
		partial[(size_t)cc * gridDim.x + blockIdx.x] = s;
	}
}
__global__ void k_sum_rows(const double *__restrict__ partial, int n, double *__restrict__ out) {
	__shared__ double red[8];
	const double *in = partial + (size_t)blockIdx.x * n;
	double v = 0.0;
	for (int k = threadIdx.x; k < n; k += blockDim.x) v += in[k];
	v = phb_warp_sum(v);
	if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
	__syncthreads();
	if (threadIdx.x == 0) {
		double s = 0.0;
		for (int w = 0; w < (int)(blockDim.x >> 5); w++) s += red[w];
		out[blockIdx.x] = s;
	}
}

// the root's lower partial must be resident (any node-at-a-time evaluation of the current inputs)
extern "C" int phbc_root_frequency_gradient(phbc_ctx *ctx, double *out_host) {
	PHBC_CHECK(cudaSetDevice(ctx->device));
	if (ctx->nuc4_G_valid) return phbc_nuc4_root_frequency_gradient(ctx, out_host);
	if (!ctx->d_lower) {
		snprintf(phbc_errbuf, sizeof(phbc_errbuf), "lower partials are not resident");
		return -4;
	}
	const size_t S = ctx->S, P = ctx->P;
	const size_t tiles = (P + 255) / 256;
	int rc;
	if ((rc = phbc_ensure_scratch(ctx, (S * tiles + S) * sizeof(double)))) return rc;
	Bufs b = phbc_make_bufs(ctx);
	k_root_freq_gradient<<<dim3((unsigned)tiles, (unsigned)S), 256, 0, ctx->stream>>>(b, ctx->root, ctx->d_freqs, ctx->d_props, ctx->d_weights, ctx->d_scratch);
	k_sum_rows<<<(unsigned)S, 256, 0, ctx->stream>>>(ctx->d_scratch, (int)tiles, ctx->d_scratch + S * tiles);
	ctx->launches += 2;
	PHBC_CHECK(cudaGetLastError());
	PHBC_CHECK(cudaMemcpyAsync(out_host, ctx->d_scratch + S * tiles, S * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
	PHBC_CHECK(cudaStreamSynchronize(ctx->stream));
	return 0;
}

// the same root partial (or the root entry of the fused walk's statistics), per category: out[c] = d lnL / d prop_c
extern "C" int phbc_root_category_gradient(phbc_ctx *ctx, double *out_host) {
	PHBC_CHECK(cudaSetDevice(ctx->device));
	const size_t C = ctx->C, S = ctx->S, P = ctx->P;
	if (ctx->nuc4_G_valid) {  // G[root][c][i] = sum_k w_k / L_k L_root[c,k,i]
		double g[8 * 16];
		PHBC_CHECK(cudaMemcpyAsync(g, ctx->d_nuc4_G + (size_t)ctx->root * C * 16, C * 16 * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
		PHBC_CHECK(cudaStreamSynchronize(ctx->stream));
		for (size_t c = 0; c < C; c++) {
			double s = 0.0;
			for (int i = 0; i < 4; i++) s += ctx->h_freqs[i] * g[c * 16 + i];
			out_host[c] = s;
		}
		return 0;
	}
	if (!ctx->d_lower) {
		snprintf(phbc_errbuf, sizeof(phbc_errbuf), "lower partials are not resident");
		return -4;
	}
	(void)S;
	const size_t tiles = (P + 255) / 256;
	int rc;
	if ((rc = phbc_ensure_scratch(ctx, (C * tiles + C) * sizeof(double)))) return rc;
	Bufs b = phbc_make_bufs(ctx);
	k_root_cat_gradient<<<dim3((unsigned)tiles, (unsigned)C), 256, 0, ctx->stream>>>(b, ctx->root, ctx->d_freqs, ctx->d_props, ctx->d_weights, ctx->d_scratch);
	k_sum_rows<<<(unsigned)C, 256, 0, ctx->stream>>>(ctx->d_scratch, (int)tiles, ctx->d_scratch + C * tiles);
	ctx->launches += 2;
	PHBC_CHECK(cudaGetLastError());
	PHBC_CHECK(cudaMemcpyAsync(out_host, ctx->d_scratch + C * tiles, C * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
	PHBC_CHECK(cudaStreamSynchronize(ctx->stream));
	return 0;
}

// K9 / K10 / A11 over every branch from the resident upper and lower partials: result[1..N], cat_grad (lnL slot untouched)
extern "C" int phbc_resident_gradient(phbc_ctx *ctx, const phbc_eval_opts *o) {
	PHBC_CHECK(cudaSetDevice(ctx->device));
	if (!ctx->d_upper || !ctx->d_lower) {
		snprintf(phbc_errbuf, sizeof(phbc_errbuf), "upper / lower partials are not resident");
		return -4;
	}
	return phbc_generic_gradient(ctx, o, ctx->d_result);
}

extern "C" int phbc_evaluate(phbc_ctx *ctx, const phbc_eval_opts *o) {
	if (o->batch_index < 0 || o->batch_index >= ctx->bl_cap || o->batch_index >= ctx->result_cap) {
		snprintf(phbc_errbuf, sizeof(phbc_errbuf), "batch index %d out of range", o->batch_index);
		return -1;
	}
	ctx->nuc4_G_valid = false;
	const int count = o->batch_count > 1 ? o->batch_count : 1;
	if (o->batch_index + count > ctx->bl_cap || o->batch_index + count > ctx->result_cap) {
		snprintf(phbc_errbuf, sizeof(phbc_errbuf), "batch %d + %d out of range", o->batch_index, count);
		return -1;
	}
	if (o->kernels != 1 /* PHB_KERNELS_GENERIC */ && phbc_nuc4_supported(ctx, o)) return phbc_nuc4_evaluate(ctx, o);  // one launch for the whole batch (sets last_family itself: it may decline)
	if (count > 1) {  // node-at-a-time paths own one set of partials: samples run back to back
		phbc_eval_opts one = *o;
		one.batch_count = 1;
		for (int b = 0; b < count; b++) {
			one.batch_index = o->batch_index + b;
			int rc = phbc_evaluate(ctx, &one);
			if (rc) return rc;
		}
		return 0;
	}
	if (o->kernels != 1 /* PHB_KERNELS_GENERIC */ && phbc_dmma_supported(ctx, o)) {
		ctx->last_family = 3;
		return phbc_dmma_evaluate(ctx, o);
	}
	if (o->kernels == 2 /* PHB_KERNELS_FUSED */) {
		snprintf(phbc_errbuf, sizeof(phbc_errbuf), "fused kernels not available for this configuration (S=%d)", ctx->S);
		return -1;
	}
	ctx->last_family = 1;
	return phbc_generic_evaluate(ctx, o);
}

extern "C" int phbc_result_to_device(phbc_ctx *ctx, int batch_index, double *out_device) {
	PHBC_CHECK(cudaSetDevice(ctx->device));
	PHBC_CHECK(cudaMemcpyAsync(out_device, ctx->d_result + (size_t)batch_index * (1 + ctx->N), (1 + (size_t)ctx->N) * sizeof(double),
	                           cudaMemcpyDeviceToDevice, ctx->stream));
	return 0;
}

// [lnL, grad[N], 1 if this shard's lnL is +-inf] of result slot `batch_index` in a buffer of its own: the operand of the in-place
// all-reduce of a pattern-sharded evaluation (SURVEY.md 8e: the rescaling decision travels in the same collective as a flag slot)
__global__ void k_pack_reduce(const double *__restrict__ result, int N, double *__restrict__ out) {
	const int i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i <= N) out[i] = result[i];
	else if (i == N + 1) out[i] = isinf(result[0]) ? 1.0 : 0.0;
}

extern "C" int phbc_pack_reduce(phbc_ctx *ctx, int batch_index, double **out_device) {
	PHBC_CHECK(cudaSetDevice(ctx->device));
	const int N = ctx->N;
	if (!ctx->d_reduce) {
		PHBC_CHECK(cudaMalloc((void **)&ctx->d_reduce, (size_t)(N + 2) * sizeof(double)));
		PHBC_CHECK(cudaMallocHost((void **)&ctx->h_reduce, (size_t)(N + 2) * sizeof(double)));
	}
	k_pack_reduce<<<(N + 2 + 255) / 256, 256, 0, ctx->stream>>>(ctx->d_result + (size_t)batch_index * (1 + N), N, ctx->d_reduce);
	ctx->launches++;
	PHBC_CHECK(cudaGetLastError());
	*out_device = ctx->d_reduce;
	return 0;
}

extern "C" int phbc_download_reduce(phbc_ctx *ctx, double *host) {
	PHBC_CHECK(cudaSetDevice(ctx->device));
	if (!ctx->d_reduce) return -4;
	const size_t bytes = (size_t)(ctx->N + 2) * sizeof(double);
	PHBC_CHECK(cudaMemcpyAsync(ctx->h_reduce, ctx->d_reduce, bytes, cudaMemcpyDeviceToHost, ctx->stream));
	PHBC_CHECK(cudaStreamSynchronize(ctx->stream));
	memcpy(host, ctx->h_reduce, bytes);
	return 0;
}

extern "C" int phbc_download_results(phbc_ctx *ctx, int nbatch, double *lnl, double *grad) {
	PHBC_CHECK(cudaSetDevice(ctx->device));
	const size_t N = ctx->N, row = 1 + N;
	const size_t need = (size_t)nbatch * row;
	if (need > ctx->h_result_cap) {  // pinned: a pageable destination makes the copy a staged, synchronous one (C1 is all latency)
		if (ctx->h_result) cudaFreeHost(ctx->h_result);
		ctx->h_result = NULL;
		ctx->h_result_cap = 0;
		PHBC_CHECK(cudaMallocHost((void **)&ctx->h_result, need * sizeof(double)));
		ctx->h_result_cap = need;
	}
	double *h = ctx->h_result;
	PHBC_CHECK(cudaMemcpyAsync(h, ctx->d_result, need * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
	PHBC_CHECK(cudaStreamSynchronize(ctx->stream));
	for (int b = 0; b < nbatch; b++) {
		if (lnl) lnl[b] = h[b * row];
		if (grad) memcpy(grad + (size_t)b * N, h + b * row + 1, N * sizeof(double));
	}
	return 0;
}

#define DOWNLOAD(dst, src, count)                                                                              \
	do {                                                                                                       \
		PHBC_CHECK(cudaSetDevice(ctx->device));                                                                \
		PHBC_CHECK(cudaMemcpyAsync(dst, src, (count) * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));  \
		PHBC_CHECK(cudaStreamSynchronize(ctx->stream));                                                        \
	} while (0)

extern "C" int phbc_download_cat_grad(phbc_ctx *ctx, double *out) {
	DOWNLOAD(out, ctx->d_cat_grad, (size_t)ctx->N * ctx->C);
	return 0;
}
extern "C" int phbc_download_pattern_lnl(phbc_ctx *ctx, double *out) {
	DOWNLOAD(out, ctx->d_pattern_lnl, (size_t)ctx->P);
	return 0;
}
extern "C" int phbc_download_partials(phbc_ctx *ctx, int index, double *out) {
	const size_t psize = (size_t)ctx->C * ctx->P * ctx->S;
	if (index < 0 || index >= 2 * ctx->N) return -1;
	if (index < ctx->T) {
		if (!ctx->d_tip_partials) return -1;
		for (int c = 0; c < ctx->C; c++)
			DOWNLOAD(out + (size_t)c * ctx->P * ctx->S, ctx->d_tip_partials + (size_t)index * ctx->P * ctx->S, (size_t)ctx->P * ctx->S);
		return 0;
	}
	if (index < ctx->N) {
		if (!ctx->d_lower) return -4;
		if (ctx->lower_is_message && index != ctx->root) {
			snprintf(phbc_errbuf, sizeof(phbc_errbuf), "the last evaluation kept messages P L, not lower partials, on the device");
			return -4;
		}
		DOWNLOAD(out, ctx->d_lower + (size_t)(index - ctx->T) * psize, psize);
		return 0;
	}
	if (!ctx->d_upper) return -4;
	DOWNLOAD(out, ctx->d_upper + (size_t)(index - ctx->N) * psize, psize);
	return 0;
}
// the matrices the LAST evaluation's kernels consumed: the node-at-a-time arrays, the walk-ordered set of the fused 4-state walk
// or the packed images of the tensor-core path, each brought back to [N][C][S][S] (the root's entry is not a transition matrix)
extern "C" int phbc_download_matrices(phbc_ctx *ctx, double *P, double *dP) {
	if (ctx->last_family == 2) return phbc_nuc4_download_matrices(ctx, P, dP);
	if (ctx->last_family == 3) return phbc_dmma_download_matrices(ctx, P, dP);
	if (!ctx->d_P) return -4;
	const size_t n = (size_t)ctx->N * ctx->C * ctx->S * ctx->S;
	if (P) DOWNLOAD(P, ctx->d_P, n);
	if (dP) DOWNLOAD(dP, ctx->d_dP, n);
	return 0;
}
extern "C" int phbc_synchronize(phbc_ctx *ctx) {
	PHBC_CHECK(cudaSetDevice(ctx->device));
	PHBC_CHECK(cudaStreamSynchronize(ctx->stream));
	return 0;
}
extern "C" void *phbc_stream(phbc_ctx *ctx) { return (void *)ctx->stream; }

// --- optional event timing -------------------------------------------------------------------
static int drain_events(phbc_ctx *ctx) {
	if (ctx->ev_count == 0) return 0;
	PHBC_CHECK(cudaStreamSynchronize(ctx->stream));
	for (int i = 0; i < ctx->ev_count; i++) {
		float ms = 0.f;
		PHBC_CHECK(cudaEventElapsedTime(&ms, ctx->ev_beg[i], ctx->ev_end[i]));
		ctx->timed_ms += ms;
		ctx->timed_launches++;
	}
	ctx->ev_count = 0;
	return 0;
}
int phbc_time_begin(phbc_ctx *ctx) {
	if (!ctx->timing) return 0;
	if (ctx->ev_count == ctx->ev_cap) {
		int rc = drain_events(ctx);
		if (rc) return rc;
	}
	PHBC_CHECK(cudaEventRecord(ctx->ev_beg[ctx->ev_count], ctx->stream));
	return 0;
}
int phbc_time_end(phbc_ctx *ctx) {
	if (!ctx->timing) return 0;
	PHBC_CHECK(cudaEventRecord(ctx->ev_end[ctx->ev_count], ctx->stream));
	ctx->ev_count++;
	return 0;
}
extern "C" int phbc_set_timing(phbc_ctx *ctx, int on) {
	PHBC_CHECK(cudaSetDevice(ctx->device));
	if (on && !ctx->ev_beg) {
		ctx->ev_cap = 256;
		ctx->ev_beg = (cudaEvent_t *)calloc(ctx->ev_cap, sizeof(cudaEvent_t));
		ctx->ev_end = (cudaEvent_t *)calloc(ctx->ev_cap, sizeof(cudaEvent_t));
		for (int i = 0; i < ctx->ev_cap; i++) {
			PHBC_CHECK(cudaEventCreate(&ctx->ev_beg[i]));
			PHBC_CHECK(cudaEventCreate(&ctx->ev_end[i]));
		}
	}
	int rc = drain_events(ctx);
	if (rc) return rc;
	ctx->timing = on != 0;
	ctx->timed_ms = 0.0;
	ctx->timed_launches = 0;
	return 0;
}
extern "C" int phbc_set_tune(phbc_ctx *ctx, int variant) {
	if (variant < 0 || variant > 31) {
		snprintf(phbc_errbuf, sizeof(phbc_errbuf), "tuning variant %d out of range", variant);
		return -1;
	}
	ctx->tune = variant;
	return 0;
}
extern "C" int phbc_kernel_time(phbc_ctx *ctx, double *total_ms, long long *launches) {
	PHBC_CHECK(cudaSetDevice(ctx->device));
	int rc = drain_events(ctx);
	if (rc) return rc;
	if (total_ms) *total_ms = ctx->timed_ms;
	if (launches) *launches = ctx->timed_launches;
	return 0;
}
extern "C" long long phbc_launch_count(const phbc_ctx *ctx) { return ctx->launches; }
extern "C" long long phbc_node_eval_count(const phbc_ctx *ctx) { return ctx->node_evals; }
extern "C" int phbc_last_family(const phbc_ctx *ctx) { return ctx->last_family; }

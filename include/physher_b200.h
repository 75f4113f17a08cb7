/*
 * physher_b200.h -- C ABI of the B200-native tree-likelihood path.
 *
 * Drop-in boundary for physher's src/phyc/treelikelihood*.c (reference paths below are relative
 * to /root/reference/src/phyc/).  Plain pointers and sizes only; the caller keeps ownership of
 * every array it passes.  All arrays are host memory unless a name ends in `_device`.
 *
 * The object mirrors `struct _SingleTreeLikelihood` (treelikelihood.h:46-124).  Where the
 * reference reads its collaborators through raw struct pointers on every evaluation
 * (Tree*, SubstitutionModel*, SiteModel*, SitePattern*; treelikelihood.c:1007), this ABI takes the
 * same data as plain arrays through setters; a setter marks the matching state dirty exactly as
 * the reference's listener does (_treelikelihood_handle_change, treelikelihood.c:73-114).
 * INTEGRATION.md shows the glue a physher maintainer adds on top of these entry points.
 *
 * Node ids: tips 0..T-1, internal nodes T..2T-2 (tree.c:183-199); N = 2T-1.
 * Layouts: matrices [node][category][i = parent state][j = child state] row-major
 * (substmodel.c:547-555); partials [category][pattern][state] (treelikelihood.c:1028).
 *
 * Error convention: functions return PHB_OK (0) or a negative PHB_E* code and keep a message
 * retrievable with phb_last_error().  The reference has no error codes (stderr + exit(),
 * treelikelihood.c:1099-1100); the glue maps a non-zero return to that behaviour.  Numerical
 * conventions are kept: NaN lnL marks everything dirty, +-inf lnL switches rescaling on and
 * recomputes (treelikelihood.c:1489-1519); the gradient is NaN-filled when lnL is NaN/inf (:328-332).
 * There is NO CPU fallback: without a CUDA device every compute entry point fails with PHB_ECUDA.
 */
#ifndef PHYSHER_B200_H
#define PHYSHER_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PHB_OK 0
#define PHB_EINVAL (-1) /* bad argument                                   */
#define PHB_ECUDA (-2)  /* CUDA runtime error / no device                 */
#define PHB_ENOMEM (-3) /* host or device allocation failed               */
#define PHB_ESTATE (-4) /* call order: an input has not been set yet      */

/* gradient request flags == TREELIKELIHOOD_FLAG_* (treelikelihood.h:32-38) */
#define PHB_FLAG_TREE_MODEL (1 << 0)
#define PHB_FLAG_SITE_MODEL (1 << 1)
#define PHB_FLAG_SUBSTITUTION_MODEL (1 << 2)
#define PHB_FLAG_BRANCH_MODEL (1 << 6)

/* options for phb_tlk_set_option */
#define PHB_OPT_INCLUDE_ROOT_FREQS 1     /* tlk->include_root_freqs (treelikelihood.h:123); default 0 = exact form */
#define PHB_OPT_COMPAT_SCALED_GRADIENT 2 /* 1: per-category normalisation under rescaling as treelikelihood.c:2721-2738 */
#define PHB_OPT_UNROOTED 3               /* 1 (default): zero the root's right child gradient (treelikelihood.c:3249-3255) */
#define PHB_OPT_KERNELS 4                /* PHB_KERNELS_* : force a kernel family (testing / profiling) */
#define PHB_OPT_SCALING_THRESHOLD_EXP 5  /* tlk->scaling_threshold = 10^-value (default 40, treelikelihood.c:1121) */
#define PHB_OPT_TIMING 6                 /* 1: bracket the dominant kernel of every evaluation with CUDA events */
#define PHB_OPT_INCREMENTAL 7            /* 1: keep all partials resident between calls (like tlk->partials) and recompute only what
                                            update_one_node / set_branch_length dirtied (_calculate_partials, treelikelihood.c:1645-1734) */

#define PHB_OPT_HOST_EXPONENTIALS 8      /* 1: exp(eval * t) of the transition matrices comes from the host's libm -- the exp the reference calls
                                            (substmodel.c:539) -- instead of the device's: 61-state models have probabilities of order t^2, t^3
                                            that a one-ulp difference in an exponential moves by 1e-9.  Default 1 for >= 60 states, else 0; node-at-a-time
                                            and tensor-core paths, single evaluations (batches build their matrices on the device) */

#define PHB_OPT_TUNE 9                   /* profiling / tests: kernel variant of the tensor-core paths; 0 = the shipped choice, results do not depend
                                            on it beyond rounding.  1 ... 6: geometry of the level-batched message kernels (tile shape, cp.async ring
                                            depth and granule size; phb_dmma.cu MsgCfg).  20 states: 9 = the level-batched kernels instead of the
                                            whole-tree walk (phb_dwalk.cu); walk variants 11 = one shared-memory slot (parked values spill to HBM),
                                            12 / 14 = 8 / 4 consumer warps whatever the pattern count, 13 = 11 + 12, 15 = warp pairs take turns on
                                            the tensor pipe, 16 = 12 consumer warps x 8 patterns.  Level-batched message kernels: 20 / 21 =
                                            cherries by pairs of tip states always / never (default: from 4 (S + 1)^2 patterns on), 22 = rescaled
                                            evaluations on the node-at-a-time tensor-core kernels instead of the message form */

#define PHB_KERNELS_AUTO 0    /* by state count, like the function-pointer dispatch at treelikelihood.c:1067-1165 */
#define PHB_KERNELS_GENERIC 1 /* node-at-a-time kernels, any state count, materialised upper partials */
#define PHB_KERNELS_FUSED 2   /* whole-tree walk kernels (4 states; 20 states on the tensor cores) / level-batched tensor-core kernels (60 ... 63 states) */

typedef struct phb_tlk phb_tlk; /* mirrors SingleTreeLikelihood */

const char *phb_last_error(void);
int phb_device_count(void);
const char *phb_version(void);

/* new_SingleTreeLikelihood (treelikelihood.c:1007-1185).
 * left/right: [N] child ids (-1 for tips).  use_tip_states as the reference's argument:
 * non-zero => tips are uint8 states (state >= nstate is unknown), zero => tip partial vectors.
 * device: CUDA ordinal.  Returns NULL on failure (see phb_last_error). */
phb_tlk *phb_tlk_create(int ntips, int nstate, int ncat, int npatterns, const int *left, const int *right, int root,
                        int use_tip_states, int device);

/* free_SingleTreeLikelihood (treelikelihood.c:1187-1230) */
void phb_tlk_free(phb_tlk *tlk);

/* clone_SingleTreeLikelihood (treelikelihood.c:1241-1395; what Model.clone builds per worker, gradascent.c:166-170): an independent
 * object on `device` (may differ from the source's) with the same topology, data (copied device to device), model inputs,
 * options, rescaling state and gradient request.  Partials are not copied: the clone starts with every node dirty. */
phb_tlk *phb_tlk_clone(phb_tlk *tlk, int device);

/* Topology moves (NNI / SPR: nniopt.c:301-334, spropt.c:1548-1615).  The reference re-reads its Tree on every traversal; here the
 * traversal is compiled into schedules, so a changed tree (same taxa, same node-id convention) is handed over explicitly.  Data,
 * model inputs, options and branch lengths (by node id) are kept; every partial is dirty; phb_tlk_set_time_tree must be called
 * again.  On failure the previous topology stays in place. */
int phb_tlk_set_topology(phb_tlk *tlk, const int *left, const int *right, int root);

/* SitePattern inputs (sitepattern.h:68-82): patterns[taxon][pattern] by TIP NODE ID and weights[pattern] */
int phb_tlk_set_tip_states(phb_tlk *tlk, const uint8_t *states /* [T][P] */);
int phb_tlk_set_tip_partials(phb_tlk *tlk, const double *partials /* [T][P][S], sp->get_partials */);
int phb_tlk_set_pattern_weights(phb_tlk *tlk, const double *weights /* [P] */);

/* SubstitutionModel inputs: the host-side eigen decomposition (eigen.h EigenDecomposition) ... */
int phb_tlk_set_eigen(phb_tlk *tlk, const double *evec, const double *eval, const double *ivec);
/* ... or, for closed-form models (jc69.c:73, hky.c:230), explicit P and dP/dt [N][C][S][S] from m->p_t / m->dp_dt */
int phb_tlk_set_matrices(phb_tlk *tlk, const double *P, const double *dP);
/* tlk->get_root_frequencies (treelikelihood.c:1946-1953) */
int phb_tlk_set_frequencies(phb_tlk *tlk, const double *freqs /* [S] */);

/* SiteModel inputs: sm->get_rate(c) (already times mu) and sm->get_proportions (sitemodel.h:38-73) */
int phb_tlk_set_site_model(phb_tlk *tlk, const double *rates /* [C] */, const double *proportions /* [C] */);

/* branch lengths as _calculate_partials reads them (treelikelihood.c:1652-1663): Node_distance or rate*dt */
int phb_tlk_set_branch_lengths(phb_tlk *tlk, const double *bl /* [N], root entry ignored */);
int phb_tlk_set_branch_length(phb_tlk *tlk, int node, double bl); /* + SingleTreeLikelihood_update_one_node */

/* SingleTreeLikelihood_update_all_nodes / _update_one_node (treelikelihood.c:1737-1751) */
void phb_tlk_update_all_nodes(phb_tlk *tlk);
int phb_tlk_update_one_node(phb_tlk *tlk, int node);
/* SingleTreeLikelihood_update_three_nodes (treelikelihood.c:1754-1771): the node and both its children */
int phb_tlk_update_three_nodes(phb_tlk *tlk, int node);

/* Model.store / Model.restore of the tree likelihood (_singleTreeLikelihood_store / _restore, treelikelihood.c:116-161):
 * restore returns to the stored inputs and the stored lnL without recomputation (MCMC reject). */
int phb_tlk_store(phb_tlk *tlk);
int phb_tlk_restore(phb_tlk *tlk);

/* SingleTreeLikelihood_use_rescaling / _rescaling (treelikelihood.h:163-164) */
int phb_tlk_use_rescaling(phb_tlk *tlk, int use);
int phb_tlk_rescaling(const phb_tlk *tlk);

int phb_tlk_set_option(phb_tlk *tlk, int option, int value);

/* tlk->calculate (treelikelihood.c:1552 -> _calculate_simple :1454): cached unless something is dirty */
int phb_tlk_calculate(phb_tlk *tlk, double *lnl);

/* per-pattern log likelihoods, tlk->pattern_lk (treelikelihood.c:1480) */
int phb_tlk_pattern_log_likelihoods(phb_tlk *tlk, double *out /* [P] */);

/* TreeLikelihood_initialize_gradient (treelikelihood.c:237-318): returns the gradient length for `flags`.
 * Supported here: PHB_FLAG_TREE_MODEL on branch-length trees => N entries indexed by node id. */
size_t phb_tlk_initialize_gradient(phb_tlk *tlk, int flags);

/* TreeLikelihood_gradient (treelikelihood.c:320-340): lnL + pre-order pass + branch gradients.
 * *grad points at a buffer OWNED BY tlk (as in the reference), valid until the next call. */
int phb_tlk_gradient(phb_tlk *tlk, const double **grad);

/* cat_branch_gradient [N][C] of the last gradient call (gradient_cat_branch_lengths, treelikelihood.c:2793) */
int phb_tlk_cat_branch_gradient(phb_tlk *tlk, double *out /* [N][C] */);

/* Substitution-model parameter gradients: the node sweep of calculate_dlnl_dQ (treelikelihood.c:2337-2583).  M holds `nsets` sets of
 * per-node matrices [nsets][N][C][S][S] (row-major like P), e.g. dP/d theta_k from m->dPdp(m, k, mat, bl * rate_c)
 * (substmodel.c:469-489, :2421); out[k] = sum over non-root nodes (not the root's right child when unrooted, :2408) and patterns of
 * w_p / L_p * sum_c prop_c sum_i f_i U_n[c,p,i] (M_k[n,c] L_n[c,p])_i.  Honours PHB_OPT_INCLUDE_ROOT_FREQS and rescaling.
 * 4 states (under rescaling: exact weights and a reversible model): ONE launch of the fused walk accumulates the per-branch statistics G[n][c][i][j] =
 * sum_p w_p / L_p f_i U_n[c,p,i] L_n[c,p,j] and every set is a 16-element contraction per (node, category) -- no materialised upper
 * partials, cost independent of nsets.  Otherwise the node-at-a-time kernels (materialised upper partials, one sweep per set). */
int phb_tlk_matrix_gradient(phb_tlk *tlk, int nsets, const double *M, double *out /* [nsets] */);
/* The root term of the frequency parameters in calculate_dlnl_dQ (treelikelihood.c:2371-2404): out[i] = d lnL / d pi_i with the partials
 * held fixed = sum_p w_p R[p,i] / L_p, R the category-integrated root partials; the caller contracts it with d pi / d theta
 * (simplex->gradient, or a unit vector).  Reuses the partials phb_tlk_matrix_gradient left on the device when nothing changed since. */
int phb_tlk_root_frequency_gradient(phb_tlk *tlk, double *out /* [S] */);
/* The root term of the invariant-site proportion (gradient_pinv_sitemodel / gradient_pinv_W_sitemodel, treelikelihood.c:2943-3001), per
 * category: out[c] = d lnL / d prop_c with the conditional likelihoods held fixed = sum_p w_p S_c(p) / L_p, S_c(p) = sum_i pi_i
 * L_root[c,p,i].  The reference's pinv_grad is out[0] - out[1] (two categories) or out[0] - mean(out[1..]) (invariant + Weibull). */
int phb_tlk_category_gradient(phb_tlk *tlk, double *out /* [C] */);

/*
 * Single-branch fast path (tlk->use_upper: serial_brent_optimize_tree optimizer.c:111-152, NNI / SPR nniopt.c:301-334,
 * spropt.c:1548-1615, Model.d2logP treelikelihood.c:470-527).
 *
 * phb_tlk_update_uppers == SingleTreeLikelihood_update_uppers (treelikelihood.c:1530-1538): lnL, then every upper partial
 * (root frequencies not folded in), all kept on the device.  Switches PHB_OPT_INCREMENTAL on.
 *
 * phb_tlk_calculate_branch == _calculate_uppper (treelikelihood.c:2592-2686) + calculate_dldt_uppper (:2195-2262) +
 * d2lnldt2_uppper (:2267-2335): lnL and its first and second derivative with respect to the length of the branch above `node`,
 * at `nbl` candidate lengths in ONE launch, from the upper partial of `node`, its lower partial and fresh P, P', P" -- every other
 * branch at its current length (pending set_branch_length changes are applied first, recomputing only the partials they reach).
 * The object's own branch lengths are not changed; the caller keeps the length it chooses with phb_tlk_set_branch_length.
 * Output pointers may be NULL.
 */
int phb_tlk_update_uppers(phb_tlk *tlk);
int phb_tlk_calculate_branch(phb_tlk *tlk, int node, int nbl, const double *bl, double *lnl, double *dlnl, double *d2lnl);

/*
 * phb_tlk_branch_hessian_diagonal: in ONE call, lnL, d lnL / dt_n and d2 lnL / dt_n^2 for the branch above every node n (by node id), at
 * the current branch lengths -- the value phb_tlk_calculate_branch(tlk, n, 1, &t_n, ...) returns as d2lnl (d2lnldt2_uppper,
 * treelikelihood.c:2267-2335), for every branch at once (Newton steps over all branch lengths, Laplace approximations, diagonal
 * preconditioners).  With L_k, L'_k, L"_k the site likelihood and its first two derivatives in t_n (see phb_tlk_calculate_branch):
 *   hess[n] = sum_k w_k (L"_k / L_k - (L'_k / L_k)^2)
 * The derivatives are always the exact ones, like those of phb_tlk_calculate_branch: PHB_OPT_INCLUDE_ROOT_FREQS and
 * PHB_OPT_COMPAT_SCALED_GRADIENT do not apply.  hess[root] = 0 (and grad[root] = 0); with PHB_OPT_UNROOTED the root's right child is 0
 * in both.  NaN / inf follow phb_tlk_gradient: an infinite lnL switches rescaling on and recomputes once; a lnL still NaN or infinite
 * NaN-fills grad and hess.  Afterwards the object's cached lnL is *lnl (a following phb_tlk_calculate launches nothing); the
 * tlk-owned gradient buffer is not refreshed.  4-state models without rescaling run as one fused walk; every other case (20 / 61 /
 * any state count, rescaling, PHB_KERNELS_GENERIC, tip partials that are not 0/1 vectors, PHB_OPT_INCREMENTAL on) makes every
 * upper partial resident and switches PHB_OPT_INCREMENTAL on, as phb_tlk_update_uppers does.  grad may be NULL.
 * PHB_ESTATE with explicit matrices (phb_tlk_set_matrices): the second derivative needs the eigen system.
 */
int phb_tlk_branch_hessian_diagonal(phb_tlk *tlk, double *lnl, double *grad /* [N] or NULL */, double *hess /* [N] */);

/*
 * phb_tlk_update_partials == the struct slot tlk->update_partials(tlk, out, p1, m1, p2, m2) (treelikelihood.h:91), for the callers
 * that drive it themselves: update_upper_partials[2] (treelikelihood.c:2129-2190, i.e. the non-virtual
 * SingleTreeLikelihood_update_uppers[2]), the tripod optimisation of SPR (spropt.c:1578-1608).  ONE partial update on the resident
 * device buffers, by index as in the reference: out = (P[m1] x[p1]) o (P[m2] x[p2]); p2 < 0: single child; indices < T tips,
 * T..N-1 lower partials, N + node upper partials.  Lower partials are made current first and the matrices are rebuilt from the
 * current branch lengths; `mirror` (may be NULL) receives the result [C][P][S] on the host (what asr.c:60-69 reads from tlk->partials).
 * Switches PHB_OPT_INCREMENTAL on.
 */
int phb_tlk_update_partials(phb_tlk *tlk, int out, int p1, int m1, int p2, int m2, double *mirror);

/* Copy of one partials buffer [C][P][S]: index < N lower partials of that node, >= N upper partials of node
 * index-N (tlk->partials[..][index], treelikelihood.h:62; used by asr.c:60).  Generic kernels only. */
int phb_tlk_get_partials(phb_tlk *tlk, int index, double *out);
/* Transition matrices as the device built them, [N][C][S][S] each (either pointer may be NULL) */
int phb_tlk_get_matrices(phb_tlk *tlk, double *P, double *dP);

/*
 * Multi-GPU / batched entry points (no counterpart in the reference, SURVEY.md 3.4 and 8e).
 *
 * phb_tlk_gradient_device: same work as phb_tlk_gradient, result left ON THE DEVICE as
 * out_device[0] = lnL, out_device[1..N] = gradient by node id, ordered on the tlk's stream, so that a
 * pattern-sharded caller can all-reduce [lnL, grad] once (NCCL) without a host round trip.
 * The NaN / +-inf handling of phb_tlk_gradient is the caller's job here (it needs the reduced lnL).
 */
int phb_tlk_gradient_device(phb_tlk *tlk, double *out_device /* [1+N] */);
/* cudaStream_t the tlk launches on (as void*), for ordering external work after it */
void *phb_tlk_stream(phb_tlk *tlk);
int phb_tlk_synchronize(phb_tlk *tlk);

/*
 * NCCL inside the C library (SURVEY.md 8e: "one ncclAllReduce(sum, ncclDouble) over [lnL, grad] per evaluation, on the compute
 * stream").  One process per GPU: rank 0 calls phb_comm_unique_id, the PHB_NCCL_ID_BYTES bytes travel to the other ranks by
 * whatever the launcher offers (MPI_Bcast, a file, torch.distributed), every rank calls phb_comm_init_rank with its device.
 * NCCL is bound at run time (libnccl.so.2); phb_nccl_version() returns 0 when it cannot be loaded.
 *
 * phb_tlk_gradient_allreduce_device: this rank's evaluation of ITS pattern shard followed by one in-place all-reduce of
 * [lnL, grad[N], number of shards whose lnL is +-inf] (N + 2 doubles) on the tlk's stream; only enqueues.  *out_device (may be
 * NULL) receives the tlk-owned device buffer holding the reduced raw sums once the stream reaches that point.
 * phb_tlk_gradient_allreduce: the same, then the result on the host with the reference's conventions applied to the reduced
 * values on every rank alike (rescaling switch treelikelihood.c:1496-1519, NaN fill :328-332, unrooted :3249-3255).
 * comm == NULL or a communicator of size 1: no collective (single shard).
 */
#define PHB_NCCL_ID_BYTES 128
typedef struct phb_comm phb_comm;
int phb_nccl_version(void);
int phb_comm_unique_id(void *id /* [PHB_NCCL_ID_BYTES] */);
phb_comm *phb_comm_init_rank(int nranks, int rank, const void *id, int device);
void phb_comm_free(phb_comm *comm);
int phb_comm_size(const phb_comm *comm);
int phb_comm_rank(const phb_comm *comm);
int phb_tlk_gradient_allreduce_device(phb_tlk *tlk, phb_comm *comm, double **out_device /* [N + 2], tlk-owned */);
int phb_tlk_gradient_allreduce(phb_tlk *tlk, phb_comm *comm, double *lnl, const double **grad);

/*
 * The same for ONE host process driving several devices (physher itself is a single process): launch queues one evaluation of the
 * current inputs on the tlk's stream and returns, collect blocks on that stream and hands back the RAW sums of this object's
 * patterns (lnL and d lnL / d bl by node id; grad may be NULL) -- no inf / NaN / unrooted policy.
 */
int phb_tlk_evaluate_launch(phb_tlk *tlk, int want_gradient);
int phb_tlk_evaluate_collect(phb_tlk *tlk, double *lnl, double *grad /* [N] */);

/*
 * phb_group: one tree likelihood sharded over several GPUs from one host thread (SURVEY.md 8e).  Shard g owns the contiguous
 * pattern range [P g / G, P (g + 1) / G) on devices[g] (a device may appear more than once); pattern-indexed inputs are given
 * for the WHOLE alignment and sliced, model inputs are broadcast, an evaluation is launched on every shard before any result is
 * collected.  Reduction: when the shards sit on DISTINCT devices and NCCL is loadable, the group owns one communicator per device
 * (ncclCommInitAll) and every shard's [lnL, grad[N], inf flag] is all-reduced in place on the shard's own stream inside one NCCL
 * group call -- no host sum; only shard 0's copy travels to the host.  Otherwise (a device listed twice, no NCCL, or
 * PHB_GROUP_REDUCE_HOST requested: the cross-check of the tests) the G vectors are summed on the host in shard order.  The
 * reference's conventions are applied to
 * the REDUCED values: +-inf lnL switches rescaling on on every shard and recomputes (treelikelihood.c:1496-1519), a NaN / inf lnL
 * NaN-fills the gradient (:328-332), PHB_OPT_UNROOTED zeroes the root's right child (:3249-3255).  *grad is owned by the group.
 */
typedef struct phb_group phb_group;
phb_group *phb_group_create(int nshards, const int *devices, int ntips, int nstate, int ncat, int npatterns, const int *left,
                            const int *right, int root, int use_tip_states);
void phb_group_free(phb_group *g);
int phb_group_size(const phb_group *g);
phb_tlk *phb_group_shard(phb_group *g, int shard); /* borrowed: per-shard introspection */
int phb_group_shard_range(const phb_group *g, int shard, int *begin, int *end);
int phb_group_set_tip_states(phb_group *g, const uint8_t *states /* [T][P] */);
int phb_group_set_tip_partials(phb_group *g, const double *partials /* [T][P][S] */);
int phb_group_set_pattern_weights(phb_group *g, const double *weights /* [P] */);
int phb_group_set_eigen(phb_group *g, const double *evec, const double *eval, const double *ivec);
int phb_group_set_frequencies(phb_group *g, const double *freqs);
int phb_group_set_site_model(phb_group *g, const double *rates, const double *proportions);
int phb_group_set_branch_lengths(phb_group *g, const double *bl);
int phb_group_set_option(phb_group *g, int option, int value);
int phb_group_use_rescaling(phb_group *g, int use);
int phb_group_rescaling(const phb_group *g);
#define PHB_GROUP_REDUCE_HOST 0
#define PHB_GROUP_REDUCE_NCCL 1
int phb_group_set_reduction(phb_group *g, int how); /* PHB_ESTATE when NCCL cannot serve this device list */
int phb_group_reduction(const phb_group *g);
int phb_group_calculate(phb_group *g, double *lnl);
int phb_group_gradient(phb_group *g, double *lnl, const double **grad);

/* B branch-length vectors sharing topology, patterns and models: lnl[b], grad[b][N]. */
int phb_tlk_gradient_batch(phb_tlk *tlk, int nbatch, const double *bl /* [B][N] */, double *lnl /* [B] */,
                           double *grad /* [B][N] */);

/*
 * Time trees, batched (SURVEY.md 8f rank 1; the reference runs these O(N) recursions on the host around every evaluation).
 *
 * phb_tlk_set_time_tree: sampling dates of the tips as heights [T] by tip node id; the lower bounds of the ratio transform
 * are derived from them (tree_transform_collect_lowers, treetransform.c:239-252).
 *
 * phb_tlk_gradient_batch_time: B samples of the reparameterised tree -- ratios[b][class id] with the root height in the
 * root's entry (class id = node id - T, tree.c:183-199; TreeTransform parameters, treetransform.c:224-237) and clock rates
 * (nrates = 1: strict clock, nrates = N: one rate per node id, BranchModel.get) -- are turned into node heights and branch
 * lengths rate * (h_parent - h_node) (treelikelihood.c:1652-1663) on the device, evaluated in one fused launch, and the branch
 * gradients are chained back on the device to
 *   grad_ratios[b][T-1]  gradient_ratios (treelikelihood.c:3161-3171: gradient_heights + Tree_node_transform_jvp, plus the
 *                        gradient of the log Jacobian when include_jacobian, treetransform.c:95-120)
 *   grad_rates[b][nrates] gradient_clock (treelikelihood.c:3054-3075)
 * lnl[b] excludes the Jacobian (like tlk->calculate); log_jacobian[b] is TreeTransform.log_jacobian (treetransform.c:215-222),
 * what _singleTreeLikelihood_logP adds when tlk->include_jacobian (treelikelihood.c:163-172).  Any output pointer may be NULL.
 */
int phb_tlk_set_time_tree(phb_tlk *tlk, const double *tip_heights /* [T] */);
int phb_tlk_gradient_batch_time(phb_tlk *tlk, int nbatch, const double *ratios /* [B][T-1] */, const double *rates /* [B][nrates] */,
                                int nrates, int include_jacobian, double *lnl /* [B] */, double *log_jacobian /* [B] */,
                                double *grad_ratios /* [B][T-1] */, double *grad_rates /* [B][nrates] */);

/*
 * Site-pattern compression (SitePattern, sitepattern.h:68-82; new_SitePattern2 / _make_patterns, sitepattern.c:186-251, 731-754).
 * alignment: encoded states [ntaxa][nsites] (DataType.encoding, datatype.c:74-91), taxa in alignment order.
 * Out (malloc'd, release with phb_free): patterns [ntaxa][P] and weights [P] (multiplicities) in EXACTLY the order the
 * reference's hash table yields them (hashtable.c:199-312, 414-451; hashtable_size = its initial size request, 100 at
 * sitepattern.c:197), and optionally the pattern index of every site.  Integer work, bit-exact.
 */
int phb_compress_patterns(int device, int ntaxa, size_t nsites, const uint8_t *alignment, int hashtable_size, size_t *npatterns,
                          uint8_t **patterns, double **weights, int **site_to_pattern /* may be NULL */);
void phb_free(void *p);
const char *phb_patterns_last_error(void);

/* With PHB_OPT_TIMING on: device time (CUDA events on the tlk stream) and launch count of the dominant kernel
 * (the fused walk kernel, or the sum of the node-at-a-time kernels) since the option was set. Synchronises. */
int phb_tlk_kernel_time(phb_tlk *tlk, double *total_ms, long long *launches);

/* kernel family the last evaluation ran on (what the function-pointer dispatch of treelikelihood.c:1067-1165 decides by state count in
 * the reference): 0 none yet, PHB_RAN_GENERIC node-at-a-time kernels, PHB_RAN_WALK the fused 4-state walk, PHB_RAN_TENSOR the FP64
 * tensor-core kernels.  phb_tlk_get_matrices returns the matrices THAT family consumed (walk-ordered set / packed images, unpacked). */
#define PHB_RAN_GENERIC 1
#define PHB_RAN_WALK 2
#define PHB_RAN_TENSOR 3
int phb_tlk_last_kernels(const phb_tlk *tlk);

/* number of kernel launches issued by this tlk since creation (bench.py's gpu_launches) */
long long phb_tlk_launch_count(const phb_tlk *tlk);

#ifdef __cplusplus
}
#endif
#endif

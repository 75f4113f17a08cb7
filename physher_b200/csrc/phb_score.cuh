// phb_score.cuh -- the score passes on resident partials (internal): the single-branch path and the Hessian diagonal (phb_branch.cu),
// NNI scores (phb_nni.cu) and SPR scores (phb_spr.cu).
//
// Every pass has the same frame around its own score kernel:
//   phbc_score_scratch   ctx->d_branch carved as  bl [items] | out [nout][3] | mats [items][C][3][S*S] | part [nout][3][tiles] |
//                        ex [items][C][S] | the pass's descriptors
//   phbc_score_matrices  the lengths (and host exponentials) up, one k_branch_matrices launch: P, r P', r^2 P" of every table item
//   score kernel(s)      per-pattern terms (score_terms), block sums into part [row][3][tile] (score_block_sum)
//   phbc_score_finish    k_branch_sum over the tiles in a fixed order (bit-identical from run to run, no floating-point atomics) and
//                        the [nout][3] results down
#pragma once

#include "phb_ctx.cuh"

// phb_branch.cu
__global__ void k_branch_matrices(int S, int C, const double *__restrict__ evec, const double *__restrict__ eval, const double *__restrict__ ivec,
                                  const double *__restrict__ bl, const double *__restrict__ rates, const double *__restrict__ ex_host,
                                  double *__restrict__ mats);
__global__ void k_branch_sum(const double *__restrict__ partial, int n, double *__restrict__ out);

struct ScoreScratch {
	double *bl, *out, *mats, *part, *ex;
	void *desc;  // 8-byte aligned
};
int phbc_score_scratch(phbc_ctx *ctx, size_t items, size_t nout, size_t tiles, size_t desc_bytes, ScoreScratch *sc);
int phbc_score_matrices(phbc_ctx *ctx, const ScoreScratch &sc, size_t items, const double *bl_host, const double *ex_host);
int phbc_score_finish(phbc_ctx *ctx, const ScoreScratch &sc, size_t nout, size_t tiles, double *out_host);
// -4 unless the resident buffers the score kernels read are there: uppers, lowers, scale factors under rescaling, tip partials
int phbc_score_resident(const phbc_ctx *ctx, const phbc_eval_opts *o);

// The weighted terms of one pattern from its site likelihood L and the first two derivatives in one branch length: w lnL, w L'/L and
// w (L"/L - (L'/L)^2).  plk is log L plus the pattern's log scale factor, which each kernel adds in its own order.
// treelikelihood.c:2331 forms (L" L - L'^2) / L^2, which underflows to 0 / 0 once L < 1e-154 -- site likelihoods a tree of a thousand
// taxa reaches without rescaling; the ratio form is the same value and stays finite.
__device__ __forceinline__ void score_terms(double plk, double L, double dL, double d2L, double w, double *v) {
	const double r1 = dL / L;
	v[0] = plk * w;
	v[1] = r1 * w;
	v[2] = (d2L / L - r1 * r1) * w;
}

// Block sum of the three terms into partial [row][3][tiles]: red is shared [3][WARPS]; nwarps the warps of the block (<= WARPS), 0 for
// blockDim.x / 32.
template <int WARPS>
__device__ __forceinline__ void score_block_sum(double (*red)[WARPS], const double *v, int nwarps, int row, double *partial) {
	for (int q = 0; q < 3; q++) {
		const double s = phb_warp_sum(v[q]);
		if ((threadIdx.x & 31) == 0) red[q][threadIdx.x >> 5] = s;
	}
	__syncthreads();
	if (threadIdx.x < 3) {
		double s = 0.0;
		for (int w = 0; w < (nwarps ? nwarps : (int)(blockDim.x >> 5)); w++) s += red[threadIdx.x][w];
		partial[((size_t)row * 3 + threadIdx.x) * gridDim.x + blockIdx.x] = s;
	}
}

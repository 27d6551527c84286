/*
 * outerbase_b200_multi_percol.h -- C ABI of the multi-response objects of outerbase_b200_multi.h with an opt-in
 * per-column para: each response column gets its own noise scale (loglik_gauss_multi) and its own coefficient scale
 * (logpr_gauss_multi).  The hyper-parameters, the basis and the terms table stay shared.  Exported by the same library,
 * same types, conventions and error model.  para_per_column = 0 creates exactly the object of the plain _create call.
 *
 * Model (para_per_column = 1).  Column c is the single-response object at its own para:
 *   loglik_gauss_multi: npara = C; para[c] is column c's noise log-sd, default log(0.01 * var(Y[:,c])) (loglik_gauss's
 *     own default on that column, variance over all ranks' rows), paravar 1 for each entry.
 *   logpr_gauss_multi: npara = C; para[c] is column c's coefficient log-scale with logpr_gauss's para0 (6) and paravar (4).
 *   In each object: val and gradhyp are the column sums; gradpara[c] is column c's single-response gradpara; grad is
 *   K x C; hessmult is block-diagonal with column c's sd (or scale); diaghess and diaghessgradhyp are per column
 *   (column c's block is the single-response result at para[c]); diaghessgradpara is (K C) x C and block-diagonal.
 *   A para of any other length than C is refused (OB_ERR_INVALID).
 * ob_lpdfvec_create of two multi-response children with the same C may mix the two forms (e.g. per-column noise with a
 *   shared coefficient scale).  Its para is the concatenation in child order; column c's objective is the
 *   single-response lpdfvec at [child 0's entry for c, child 1's entry for c] -- a shared child's one entry serves every
 *   column -- including that column's own marginal adjustment.  ob_lpdf_optcg runs C independent CGs as for the shared
 *   form.  ob_lpdf_diaghessgradpara of such an lpdfvec forms the (K C) x npara matrix on request only.
 * ob_predictor_create on a loglik_gauss_multi that is per-column, or whose total Hessian diagonal was last set by an
 *   lpdfvec with a per-column child (e.g. a shared likelihood under a per-column prior: the columns' diagonals then
 *   differ): ob_predictor_mean writes N x C, and ob_predictor_var writes N x C as well (NOT one N-vector):
 *   column c = Phi^2 (1 / totdiaghess[:,c]) + exp(2 para_c), para_c the likelihood's entry for column c.
 *   ob_lpdf_get(loglik, "predvar_ncol") returns the number of columns ob_predictor_var will write for a predictor
 *   created from that likelihood now (C or 1).
 */
#ifndef OUTERBASE_B200_MULTI_PERCOL_H
#define OUTERBASE_B200_MULTI_PERCOL_H

#include "outerbase_b200_multi.h"

#ifdef __cplusplus
extern "C" {
#endif

/* C = 0 is refused (OB_ERR_INVALID). */
int ob_loglik_gauss_multi_create_ex(ob_ctx* ctx, ob_outermod* om, const uint64_t* terms, uint64_t K, const double* Y /* N x C */,
                                    uint64_t C, const double* x, uint64_t N, int para_per_column, ob_lpdf** out);
int ob_logpr_gauss_multi_create_ex(ob_ctx* ctx, ob_outermod* om, const uint64_t* terms, uint64_t K, uint64_t C,
                                   int para_per_column, ob_lpdf** out);

#ifdef __cplusplus
}
#endif
#endif /* OUTERBASE_B200_MULTI_PERCOL_H */

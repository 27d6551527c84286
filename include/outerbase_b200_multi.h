/*
 * outerbase_b200_multi.h -- C ABI of the multi-response extension: C responses observed at the same inputs, fitted on
 * one basis.  The reference has no counterpart, so these entry points are kept apart from outerbase_b200.h (the
 * drop-in boundary, whose every call names the reference interface it replaces and is mirrored by the CPU oracle);
 * they are exported by the same library and use its types, conventions and error model.
 *
 * Model.  loglik_gauss_multi(om, terms, Y, x): Y is N x C column-major; every column shares the basis, the terms table,
 * the hyper-parameters and para (noisescale).  Coefficients are K x C column-major, K*C entries, and every generic
 * ob_lpdf_* call operates on them (ob_lpdf_sizes reports nterms = K*C; "coeff", "grad", "totdiaghess" are K*C long).
 *   - val, gradhyp and gradpara are the sums over the columns of what loglik_gauss on Y[:,c] returns at coefficient
 *     column c; grad is K x C; hessmult is block-diagonal; diaghess and diaghessgradpara are loglik_gauss's repeated C
 *     times (diaghessgradhyp: each K x H column block repeated).
 *   - default para = log(0.01 * mean_c var(Y[:,c])), Armadillo two-pass variance over all ranks' rows (C = 1:
 *     loglik_gauss's default).  Rows are sharded over ranks like loglik_gauss.
 * logpr_gauss_multi(om, terms, C): an independent logpr_gauss on each coefficient column, shared coeffscale; its sums
 * are formed the same way.
 * ob_lpdfvec_create of two multi-response children with the same C (either order) is lpdfvec on the K*C-long
 * vectors: the marginal adjustment is C times the single-response one (up to summation order).  Mixing a
 * multi-response child with a single-response one, or two different C, is refused (OB_ERR_INVALID).
 * ob_lpdf_optcg on that lpdfvec runs C independent lpdf::optcg (src/fit.cpp:37-96): column c on column c's own objective
 * (its loglik, its prior, the single-response marginal adjustment) with its own step sizes and stop test; a column
 * that stops stays frozen.  They run as ONE column-batched loop on the device; the final update with gradients runs
 * once for the whole object.  ob_lpdf_get(..., "cg_iters") then returns C values, one per column, and
 * ob_lpdf_get(..., "ncol") returns C (1 on every single-response object of this library).
 * Refused on multi-response objects (OB_ERR_INVALID): the full Hessian (ob_lpdf_hess*, the full-Hessian branch of
 * lpdfvec), ob_lpdf_optnewton, and ob_lpdf_optcg outside lpdfvec(logpr_gauss_multi, loglik_gauss_multi).
 * ob_predictor_create on a loglik_gauss_multi: ob_predictor_mean writes N x C (Phi . coeff), ob_predictor_var writes
 * ONE N-vector shared by all columns (with shared para the total Hessian diagonal does not depend on the response).
 * outerbase_b200_multi_percol.h declares the variants with one para entry per column (its own noise scale and
 * coefficient scale for each response); when either child of the fit has them, ob_predictor_var writes N x C.
 */
#ifndef OUTERBASE_B200_MULTI_H
#define OUTERBASE_B200_MULTI_H

#include "outerbase_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

/* C = 0 is refused (OB_ERR_INVALID). */
int ob_loglik_gauss_multi_create(ob_ctx* ctx, ob_outermod* om, const uint64_t* terms, uint64_t K,
                                 const double* Y /* N x C */, uint64_t C, const double* x, uint64_t N, ob_lpdf** out);
int ob_logpr_gauss_multi_create(ob_ctx* ctx, ob_outermod* om, const uint64_t* terms, uint64_t K, uint64_t C,
                                ob_lpdf** out);

#ifdef __cplusplus
}
#endif
#endif /* OUTERBASE_B200_MULTI_H */

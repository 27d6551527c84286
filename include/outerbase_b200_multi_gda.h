/*
 * outerbase_b200_multi_gda.h -- C ABI of loglik_gda on C responses observed at the same inputs: the stage-1 likelihood
 * of a two-stage multi-response fit (a row subsample, with a per-row noise scale).  Exported by the same library, same
 * types, conventions and error model as outerbase_b200.h and outerbase_b200_multi.h.
 *
 * Model.  Y is N x C column-major; column c is exactly loglik_gda(om, terms, Y[:,c], x).
 *   Shared by the columns: the basis, the terms table, the hyper-parameters, the dodiag flag and both para entries
 *     (noise log-sd, log-scale of the diagonal adjustment).  The per-row noise sd obssd is one N-vector:
 *     obssd = sqrt(e^{2 p0} + e^{2 p1} residvar) with dodiag, sqrt(e^{2 p0}) without.
 *   val, gradhyp and gradpara are the sums of the single-response results over the columns, in column order.
 *   grad is K x C; hessmult is block-diagonal; yhat is N x C.
 *   diaghess, diaghessgradhyp and diaghessgradpara do not depend on the response: the single-response ones repeated
 *     C times ((K C) x 1, (K C) x H, (K C) x 2).
 *   Defaults: para0 = [0.5 log(0.01 mean_c var(Y[:,c])), 0], paravar = [4, 4] (C = 1: loglik_gda's own).
 * ob_lpdfvec_create(logpr_gauss_multi, loglik_gda_multi), in either order with the same C, is the lpdfvec of the
 *   K C-long vectors; ob_lpdf_optcg on it runs C independent CGs, one per column, as for loglik_gauss_multi.
 * ob_predictor_create on it: ob_predictor_mean writes N x C, ob_predictor_var one shared N-vector (pred_gda's);
 *   ob_lpdf_get(loglik, "predvar_ncol") is 1.
 * Refused (OB_ERR_INVALID): C = 0; an lpdfvec with a per-column logpr_gauss_multi, a single-response child or a
 *   different C; optnewton, the full Hessian, and optcg outside the lpdfvec above.  More than one rank is refused
 *   (OB_ERR_STATE).
 */
#ifndef OUTERBASE_B200_MULTI_GDA_H
#define OUTERBASE_B200_MULTI_GDA_H

#include "outerbase_b200_multi.h"

#ifdef __cplusplus
extern "C" {
#endif

int ob_loglik_gda_multi_create(ob_ctx* ctx, ob_outermod* om, const uint64_t* terms, uint64_t K, const double* Y /* N x C */,
                               uint64_t C, const double* x, uint64_t N, ob_lpdf** out);

#ifdef __cplusplus
}
#endif
#endif /* OUTERBASE_B200_MULTI_GDA_H */

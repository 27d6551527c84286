/*
 * outerbase_b200_sobol_pairs.h -- C ABI of the second-order sensitivity extension: which inputs of a fitted model
 * interact, and how much.  Model, measure, tables, conventions and refusals are those of outerbase_b200_sobol.h; this
 * entry point returns ob_sobol's four outputs (the same bits) and two forms per input pair.
 *
 * Pair factors of terms (k, k'), per dimension:  p_l = mu_l[t_kl] mu_l[t_k'l],  c_l = C_l[t_kl, t_k'l],  g_l = c_l + p_l.
 * Under the product measure the ANOVA component of f_b on the input set u has the variance
 *     sigma2_u,b = sum_{k,k'} coeff[k, b] coeff[k', b] prod_{j in u} c_j prod_{j not in u} p_j.
 * For each input pair l < m (P = d (d - 1) / 2 pairs, pair (l, m) at row r = l d - l (l + 1) / 2 + (m - l - 1)):
 *     second[r + P b] = sigma2_{lm}       = sum_{k,k'} coeff[k, b] coeff[k', b] c_l c_m prod_{j not in {l,m}} p_j
 *                                           (the pure second-order variance)
 *     supset[r + P b] = sum_{u >= {l,m}} sigma2_u
 *                                         = sum_{k,k'} coeff[k, b] coeff[k', b] c_l c_m prod_{j not in {l,m}} g_j
 *                                           (Liu-Owen superset importance: every interaction that involves both)
 * The closed second-order index is (first_l + first_m + second_lm) / var; second / var and supset / var are the
 * normalised pure and superset indices.  In exact arithmetic 0 <= second <= supset <= min(total_l, total_m),
 * sum first + sum second <= var, and for d = 2 second = supset = var - first_0 - first_1.
 *
 * Numerics.  As ob_sobol: no divisions and no differences of products.  Per term pair the product over
 * j not in {l, m} is a prefix product up to l, a middle product over l < j < m grown in ascending j as m advances, and a
 * suffix product after m, for p and for g.  The contraction over term pairs runs on the FP64 tensor cores in an order
 * fixed by K and d alone: a column's results do not depend on B or on the other columns, and are the same bits on
 * every run.
 *
 * Refused (OB_ERR_INVALID): whatever ob_sobol refuses, including more than one rank and d > 77.
 */
#ifndef OUTERBASE_B200_SOBOL_PAIRS_H
#define OUTERBASE_B200_SOBOL_PAIRS_H

#include "outerbase_b200_sobol.h"

#ifdef __cplusplus
extern "C" {
#endif

/* mean, var, first and total as ob_sobol; second and supset receive P x B (column-major), P = d (d - 1) / 2, pair
 * (l, m), l < m, at row l d - l (l + 1) / 2 + (m - l - 1); they may be null when P = 0 and are not written then */
int ob_sobol_pairs(ob_ctx* ctx, ob_outermod* om, const uint64_t* terms, uint64_t K, const double* coeff, uint64_t B,
                   const double* xq, uint64_t nq, double* mean, double* var, double* first, double* total,
                   double* second, double* supset);

#ifdef __cplusplus
}
#endif
#endif /* OUTERBASE_B200_SOBOL_PAIRS_H */

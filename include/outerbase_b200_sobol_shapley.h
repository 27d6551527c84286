/*
 * outerbase_b200_sobol_shapley.h -- C ABI of the Shapley-effect extension: how much of a fitted model's variance each
 * input accounts for, one number per input that adds up to the variance.  Model, measure, tables, conventions and
 * refusals are those of outerbase_b200_sobol.h; this entry point returns ob_sobol's four outputs (the same bits) and
 * the Shapley effect of every input.
 *
 * Pair factors of terms (k, k'), per dimension:  p_j = mu_j[t_kj] mu_j[t_k'j],  c_j = C_j[t_kj, t_k'j],  g_j = c_j + p_j.
 * Under the product measure the inputs are independent, and the ANOVA component of f_b on the input set u has the
 * variance
 *     sigma2_u,b = sum_{k,k'} coeff[k, b] coeff[k', b] prod_{j in u} c_j prod_{j not in u} p_j  (>= 0).
 * The Shapley effect (Owen 2014; Song, Nelson & Staum 2016) splits each component's variance equally among its inputs:
 *     shapley[l + d b] = Sh_l,b = sum_{u containing l} sigma2_u,b / |u|.
 * With h_j(z) = p_j + z c_j the sum over the subsets v of the other inputs, weighted 1 / (|v| + 1) = int_0^1 z^|v| dz, is
 *     Sh_l,b = sum_{k,k'} coeff[k, b] coeff[k', b] c_l int_0^1 prod_{j != l} h_j(z) dz.
 * The integrand is a polynomial of degree d - 1 in z; the n = max(1, ceil(d / 2))-node Gauss-Legendre rule on [0, 1],
 * nodes z_i and weights w_i (positive, adding up to 1), integrates it exactly:
 *     Sh_l,b = sum_{k,k'} coeff[k, b] coeff[k', b] c_l sum_i w_i prod_{j != l} h_j(z_i).
 * z = 0 gives first_l and z = 1 total_l.  In exact arithmetic:
 *     sum_l Sh_l = var           (sum_l c_l prod_{j != l} h_j(z) = d/dz prod_j h_j(z), whose integral is prod g - prod p)
 *     first_l <= Sh_l <= total_l (every sigma2_u >= 0)
 *     Sh_l = 0 for an input the function does not depend on.
 * shapley / var is the normalised Shapley effect; the normalised effects add up to 1.
 *
 * Numerics.  As ob_sobol: no divisions and no differences of products.  Per term pair and node, the product over
 * j != l is formed from prefix products of h_j in ascending j and suffix products in descending j, the nodes are added in
 * ascending order, and c_l multiplies the sum.  The contraction over term pairs runs on the FP64 tensor cores in an order
 * fixed by K and d alone: a column's results do not depend on B or on the other columns, and are the same bits on every
 * run.  The nodes and weights come from Newton's method on the Legendre recurrence in extended precision.
 *
 * Refused (OB_ERR_INVALID): whatever ob_sobol refuses, including more than one rank and d > 77.
 */
#ifndef OUTERBASE_B200_SOBOL_SHAPLEY_H
#define OUTERBASE_B200_SOBOL_SHAPLEY_H

#include "outerbase_b200_sobol.h"

#ifdef __cplusplus
extern "C" {
#endif

/* mean, var, first and total as ob_sobol; shapley receives d x B (column-major) */
int ob_sobol_shapley(ob_ctx* ctx, ob_outermod* om, const uint64_t* terms, uint64_t K, const double* coeff, uint64_t B,
                     const double* xq, uint64_t nq, double* mean, double* var, double* first, double* total,
                     double* shapley);

#ifdef __cplusplus
}
#endif
#endif /* OUTERBASE_B200_SOBOL_SHAPLEY_H */

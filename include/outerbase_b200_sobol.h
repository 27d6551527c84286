/*
 * outerbase_b200_sobol.h -- C ABI of the sensitivity extension: variance-based (Sobol) indices of a fitted model.
 * The reference has no counterpart, so this entry point is kept apart from outerbase_b200.h (the drop-in boundary); it is
 * exported by the same library and uses its types, conventions and error model.
 *
 * Model.  Column b of coeff (K x B, column-major) is the function f_b(x) = sum_k coeff[k, b] prod_l R_l(x_l, t_kl), with
 * t the terms table (K x d) and R_l(., j) column j of getbase(l + 1): basemat times the dimension's basescale factor.
 * Level 0 is included, so no separate basescale factor appears.
 *
 * Measure.  mu = prod_l mu_l, mu_l the empirical distribution of column l of xq (nq x d, column-major).  The pairing of
 * entries within a row of xq does not matter: the training inputs give the product of their empirical marginals,
 * independent uniform columns the usual indices on the unit box.
 *
 * Per-dimension table, for j, j' < mo_l = 1 + the highest level of dimension l in terms:
 *     mu_l[j]     = (1/nq) sum_q R_l(xq[q, l], j)
 *     C_l[j, j']  = (1/nq) sum_q (R_l(xq[q, l], j) - mu_l[j]) (R_l(xq[q, l], j') - mu_l[j'])   (centred)
 * Pair factors of terms (k, k'):  p_l = mu_l[t_kl] mu_l[t_k'l],  c_l = C_l[t_kl, t_k'l],  g_l = c_l + p_l.  Then
 *     mean[b]         = E f_b             = sum_k coeff[k, b] prod_l mu_l[t_kl]
 *     var[b]          = Var f_b           = sum_{k,k'} coeff[k, b] coeff[k', b] sum_l (prod_{j<l} g_j) c_l (prod_{j>l} p_j)
 *     first[l + d b]  = Var(E[f_b | x_l]) = sum_{k,k'} coeff[k, b] coeff[k', b] c_l prod_{j!=l} p_j
 *     total[l + d b]  = E[Var(f_b | x_-l)] = sum_{k,k'} coeff[k, b] coeff[k', b] c_l prod_{j!=l} g_j
 * The first-order index of dimension l is first / var, the total index total / var.  var uses the telescoping identity
 * prod g - prod p = sum_l (prod_{j<l} g_j) c_l (prod_{j>l} p_j): no pair subtracts two nearly equal products and nothing
 * divides by a table value.  In exact arithmetic 0 <= first_l <= total_l and sum_l first_l <= var <= sum_l total_l.
 *
 * Numerics.  The table is computed on the GPU with the means first and the moments centred at them; the forms sum over
 * k <= k' (off-diagonal pairs weighted 2).  Both reductions run in an order fixed by nq and K alone: a column's results
 * do not depend on B or on the other columns, and are the same bits on every run.
 *
 * Refused (OB_ERR_INVALID): B = 0; nq = 0; K = 0; levels beyond a dimension's knots; a context with more than one rank
 * (xq's rows would be rank-local).  The om must have its covariances and knots set.
 */
#ifndef OUTERBASE_B200_SOBOL_H
#define OUTERBASE_B200_SOBOL_H

#include "outerbase_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

/* mean and var receive B values, first and total d x B (column-major) */
int ob_sobol(ob_ctx* ctx, ob_outermod* om, const uint64_t* terms, uint64_t K, const double* coeff, uint64_t B,
             const double* xq, uint64_t nq, double* mean, double* var, double* first, double* total);

#ifdef __cplusplus
}
#endif
#endif /* OUTERBASE_B200_SOBOL_H */

/*
 * outerbase_b200_draws.h -- C ABI of the posterior-draws extension: S joint draws from the posterior of a fitted model.
 * The reference has no counterpart, so these entry points are kept apart from outerbase_b200.h (the drop-in boundary);
 * they are exported by the same library and use its types, conventions and error model.
 *
 * Model.  With the hyper-parameters, the terms and para of a fitted lpdfvec(logpr_gauss, loglik_gauss) (either child
 * order) held fixed, the coefficient posterior is N(mu, H^-1), H = Phi^T Phi / sigma^2 + D^-1, D = diag((coeffsd_k sca)^2),
 * sigma = exp(para of loglik_gauss), sca = exp(para of logpr_gauss).  Draw s is made by perturb-and-MAP: it is the
 * maximiser of
 *     -|y + sigma eps_s - Phi theta|^2 / (2 sigma^2) - (theta - delta_s)^T D^-1 (theta - delta_s) / 2,
 * eps_s ~ N(0, I_N), delta_s = coeffsd % sca xi_s ~ N(0, D), i.e. theta_s = H^-1 (Phi^T (y + sigma eps_s) / sigma^2 +
 * D^-1 delta_s), whose mean is mu and covariance H^-1 exactly.  The S maximisations are the S columns of
 * lpdfvec(logpr_gauss_multi(S) centred at delta, loglik_gauss_multi(S) on the perturbed responses), without the marginal
 * adjustment (it does not depend on theta), solved by the column-batched CG of outerbase_b200_multi.h from the fit's
 * coefficients (zero when the fit has none), each column with the reference's stop rule num < tol && valdiff < tol.  The
 * draws are exact only at convergence: tol = 0.001 is the reference's fitting tolerance, not a sampling guarantee.
 * The draws carry no hyper-parameter uncertainty, and predict gives draws of the latent function: observation noise at
 * new points (sigma N(0, 1)) is the caller's to add.
 *
 * Random numbers.  eps_s[i] and xi_s[k] are normal number i (k) of stream 0 (1), column s, of ob_debug_normals(seed, ...):
 * Philox4x32-10 with key = seed (low word first) and counter (index, stream, column, 0); each output gives two uniforms
 * u = ((x >> 11) + 1) 2^-53 in (0, 1] from the 64-bit words (v1 v0) and (v3 v2), and normals 2 index and 2 index + 1 by
 * Box-Muller, sqrt(-2 log u1) cos(2 pi u2) and sqrt(-2 log u1) sin(2 pi u2).  A draw depends on (seed, s) and the model
 * only: the first columns of a larger S are the draws of a smaller one.
 *
 * ob_draws_create snapshots the fit (its om, terms, para, y and x rows, coefficients); later changes to the om or the
 * logpdf do not affect the object.  Refused (OB_ERR_INVALID): anything but lpdfvec(logpr_gauss, loglik_gauss), i.e.
 * multi-response and per-column-para fits, loglik_gda and loglik_std fits; S = 0; a context with more than one rank.
 */
#ifndef OUTERBASE_B200_DRAWS_H
#define OUTERBASE_B200_DRAWS_H

#include "outerbase_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct ob_draws ob_draws;

int ob_draws_create(ob_lpdf* logpdf, uint64_t S, uint64_t seed, ob_draws** out);
int ob_draws_destroy(ob_draws* d);
/* runs the S solves from the fit's coefficients; may be called again (with another tol) */
int ob_draws_solve(ob_draws* d, double tol, uint64_t maxepch);
/* which: "coeff" (K x S, after solve), "cg_iters" (S, after solve), "y" (N x S perturbed responses), "prior_mean"
 * (K x S, the delta_s); *n receives the count, out may be null to ask for it */
int ob_draws_get(ob_draws* d, const char* which, double* out, uint64_t* n);
/* x is N x d (column-major); out is N x S: the draws of the latent function Phi(x) theta_s (after solve) */
int ob_draws_predict(ob_draws* d, const double* x, uint64_t N, double* out);
/* test hook, no GPU: n normals of (seed, stream, column) from index first on, by the host twin of the generator */
int ob_debug_normals(uint64_t seed, uint32_t stream, uint64_t column, uint64_t first, uint64_t n, double* out);
/* K x C prior means of a logpr_gauss_multi (n = K C), or none (n = 0): column c's prior is centred at mean[:, c] */
int ob_logpr_gauss_multi_set_mean(ob_lpdf* logpr, const double* mean, uint64_t n);

#ifdef __cplusplus
}
#endif
#endif /* OUTERBASE_B200_DRAWS_H */

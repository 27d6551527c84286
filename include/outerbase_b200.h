/*
 * outerbase_b200.h -- C ABI of the B200-native outerbase hot path.
 *
 * This is the drop-in boundary.  Every entry point names the reference
 * interface (file:line under the reference tree, MattPlumlee/outerbase 0.1.1)
 * whose body it replaces.  Conventions are the reference's own:
 *   - all matrices are column-major fp64 (Armadillo `mat`), vectors are dense
 *     fp64; `terms` is a K x d column-major table of 64-bit unsigned levels
 *     (Armadillo `umat`, src/linalg.cpp:73 treats level 0 as "skip");
 *   - every pointer argument is a HOST pointer unless its name ends in `_dev`;
 *   - output buffers are caller-owned and sized as documented per call.
 * No torch / Armadillo / Rcpp type appears in any signature.
 *
 * Error model (reference: C++ exceptions -> R errors, src/interfaceR.cpp:95-118,
 * src/fit.h:52-55): every call returns an int status, 0 on success.  The
 * message of the last failure on the calling thread is ob_last_error().
 * Non-finite model state is still signalled in-band (val = -inf), exactly as
 * src/fit.cpp:53-56 does.
 *
 * The identical ABI with prefix `orc_` is exported by the CPU oracle
 * (oracle/, test infrastructure only) so one test harness drives both.
 */
#ifndef OUTERBASE_B200_H
#define OUTERBASE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define OB_OK           0
#define OB_ERR_INVALID  1 /* std::range_error / std::invalid_argument in the reference */
#define OB_ERR_CUDA     2
#define OB_ERR_NCCL     3
#define OB_ERR_STATE    4 /* call order (e.g. knots before covfs, interfaceR.cpp:95) */
#define OB_ERR_NOGPU    5 /* no CUDA device: the product has NO CPU fallback */

typedef struct ob_ctx       ob_ctx;       /* one GPU: device, stream, optional NCCL communicator */
typedef struct ob_outermod  ob_outermod;  /* class outermod,  src/modandbase.h:9-54   (host)   */
typedef struct ob_outerbase ob_outerbase; /* class outerbase, src/modandbase.h:57-125 (device) */
typedef struct ob_lpdf      ob_lpdf;      /* class lpdf and children, src/fit.h:23-148,236-268 */
typedef struct ob_predictor ob_predictor; /* class predictor / pred_gauss, src/fit.h:352-361   */

const char* ob_last_error(void);
int ob_version(void);

/* ------------------------------------------------------------------ context
 * One context per GPU / per process rank.  Replaces the reference's implicit
 * "OpenMP team of nthreads" (src/modandbase.cpp:464,553). */
int ob_ctx_create(int device, ob_ctx** out);
int ob_ctx_destroy(ob_ctx* ctx);
int ob_ctx_synchronize(ob_ctx* ctx);
/* cudaStream_t all kernels of this context are launched on (for event timing). */
int ob_ctx_stream(ob_ctx* ctx, void** stream_out);
/* Row sharding over ranks: rows are partitioned by the CALLER (each rank builds
 * its outerbase from its own rows); every Phi^T-type result is summed over ranks
 * with one NCCL allreduce -- the reference's `#pragma omp critical  out += out_`
 * (src/linalg.cpp:334-335,438-442,616-617).  id is NCCL's 128-byte unique id. */
int ob_comm_get_unique_id(void* id128);
int ob_ctx_comm_init(ob_ctx* ctx, int nranks, int rank, const void* id128);
int ob_ctx_comm_info(ob_ctx* ctx, int* nranks, int* rank);
/* Sum buf_dev[0..n) over the ranks of the communicator, in place, on ctx's stream (not synchronised): the
 * cross-GPU form of the reference's `#pragma omp critical: out += out_` (src/linalg.cpp:334-335, 438-442, 616-617).
 * Every Phi^T-type call above does this itself; exposed for callers that keep their own row-sharded sums.
 * Up to 65536 doubles travel through the one-shot peer-memory kernel (option "p2p", default 1 when the ranks can
 * map each other's memory), larger payloads through ncclAllReduce.  All ranks must call it in the same order. */
int ob_ctx_allreduce_dev(ob_ctx* ctx, double* buf_dev, uint64_t n);
/* measured FP64 FMA peak of this GPU (TFLOP/s): the roofline denominator bench.py quotes. */
int ob_ctx_fp64_peak(ob_ctx* ctx, double* tflops);
/* test hook: number of CUDA kernels this context has launched so far. */
int ob_ctx_launch_count(ob_ctx* ctx, uint64_t* count);

/* ------------------------------------------------------------------ covf
 * covf_mat25 / covf_mat25pow / covf_mat25ang ::cov and ::cov_gradhyp,
 * src/covfuncs.cpp:113-126,134-150,197-212,220-243,285-310,318-347.
 * name in {"mat25","mat25pow","mat25ang"}; out is n1 x n2 (x numhyp slices). */
int ob_covf_numhyp(const char* name, uint64_t* numhyp);
int ob_covf_cov(ob_ctx* ctx, const char* name, const double* hyp,
                const double* x1, uint64_t n1, const double* x2, uint64_t n2, double* out);
int ob_covf_cov_gradhyp(ob_ctx* ctx, const char* name, const double* hyp,
                        const double* x1, uint64_t n1, const double* x2, uint64_t n2, double* out);

/* ------------------------------------------------------------------ outermod (host side, kept on the CPU)
 * new(outermod); setcovfs; setknot; gethyp  -- src/interfaceR.cpp:53-73,94-149,151-166
 * updatehyp=hyp_set :161; selectterms :387; getvar :350; getlvar_gradhyp :364;
 * hyplpdf :89; hyplpdf_grad :107 (all src/modandbase.cpp). */
int ob_outermod_create(ob_outermod** out);
int ob_outermod_destroy(ob_outermod* om);
int ob_outermod_setcovfs(ob_outermod* om, uint64_t d, const char* const* names);
/* knots: concatenation of the d knot vectors; lens[l] = length of vector l. */
int ob_outermod_setknot(ob_outermod* om, const double* knots, const uint64_t* lens);
int ob_outermod_updatehyp(ob_outermod* om, const double* hyp, uint64_t nhyp);
int ob_outermod_gethyp(ob_outermod* om, double* hyp /* nhyp */);
/* sizes: d, nhyp (H), nknot (M = sum of knot counts), nge (= knotptstge[d]). */
int ob_outermod_sizes(ob_outermod* om, uint64_t* d, uint64_t* nhyp, uint64_t* nknot, uint64_t* nge);
/* tie-break policy of selectterms (src/modandbase.cpp:406-409 shuffles with R's RNG,
 * which cannot be reproduced): seed == 0 -> lowest candidate index (default);
 * seed != 0 -> uniform choice from a SplitMix64 stream started at seed. */
int ob_outermod_set_select_seed(ob_outermod* om, uint64_t seed);
int ob_outermod_selectterms(ob_outermod* om, uint64_t numele, uint64_t* terms /* numele x d */);
int ob_outermod_getvar(ob_outermod* om, const uint64_t* terms, uint64_t K, double* out /* K */);
int ob_outermod_getlvar_gradhyp(ob_outermod* om, const uint64_t* terms, uint64_t K, double* out /* K x H */);
int ob_outermod_hyplpdf(ob_outermod* om, const double* hyp, uint64_t nhyp, double* out);
int ob_outermod_hyplpdf_grad(ob_outermod* om, const double* hyp, uint64_t nhyp, double* out /* H */);
/* index tables and eigenbasis, for parity tests of the integer-exact state
 * (SURVEY A1): which in {"knotptst"(d+1),"hypst"(d+1),"hypmatch"(H),"gest"(H+1),
 * "knotptstge"(d+1),"maxlevel"(d)} ; {"basisvar"(M),"knotpt"(M),
 * "logbasisvar_gradhyp"(nge),"rotmat"(mmax x M),"rotmat_gradhyp"(mmax x nge)}. */
int ob_outermod_get_index(ob_outermod* om, const char* which, int64_t* out, uint64_t* n);
int ob_outermod_get_real(ob_outermod* om, const char* which, double* out, uint64_t* nrow, uint64_t* ncol);

/* ------------------------------------------------------------------ outerbase (device resident)
 * new(outerbase, om, x) :459-483 ; build :547-626 ; getbase :634 ; getmat :649 ;
 * mm :677 ; tmm :700 ; mm_gradhyp :725 ; tmm_gradhyp :755 ; sqmm :784 ;
 * sqmm_gradhyp :798 ; sqtmm :816 ; sqtmmm :831 ; sqtmm_gradhyp :845 ;
 * sqcolsums :863 ; sqcolsums_gradhyp :875 (src/modandbase.cpp) and the
 * linalg.h kernels behind them (src/linalg.cpp:102-131,225-277,303-355,
 * 394-471,527-557,583-637,685-715).  x is N x d column-major and is copied. */
int ob_outerbase_create(ob_ctx* ctx, ob_outermod* om, const double* x, uint64_t N,
                        int dograd, ob_outerbase** out);
int ob_outerbase_destroy(ob_outerbase* ob);
int ob_outerbase_build(ob_outerbase* ob);
/* R-visible fields nthreads/vertpl/chunksize/loopsize (src/interfaceR.cpp:682-685):
 * accepted and reported with the reference's rule (modandbase.cpp:504-513),
 * ignored by the GPU path. */
int ob_outerbase_set_nthreads(ob_outerbase* ob, int nthreads);
int ob_outerbase_loopvals(ob_outerbase* ob, uint64_t* nthreads, uint64_t* chunksize,
                          uint64_t* loopsize, int* vertpl);
/* the matrices outerbase owns (public/private fields, modandbase.h:61,113-119): which in
 * {"basemat"(N x M),"basemat_gradhyp"(N x nge),"basescale"(N),"basescalemat"(N x d)};
 * out may be NULL to query the shape. */
int ob_outerbase_get_real(ob_outerbase* ob, const char* which, double* out, uint64_t* nrow, uint64_t* ncol);
int ob_outerbase_getbase(ob_outerbase* ob, uint64_t dim_1based, double* out /* N x m_dim */);
int ob_outerbase_getmat(ob_outerbase* ob, const uint64_t* terms, uint64_t K, double* out /* N x K */);
/* outerbase::getmat_gradhyp, src/modandbase.cpp:663-669 (C++ only, loglik_std's cube): N x K x H, slice after slice */
int ob_outerbase_getmat_gradhyp(ob_outerbase* ob, const uint64_t* terms, uint64_t K, double* out /* N x K x H */);
/* sq != 0 selects the squared operators (basematsq/basescalesq). */
int ob_outerbase_mm(ob_outerbase* ob, int sq, const uint64_t* terms, uint64_t K,
                    const double* a /* K */, double* out /* N */);
int ob_outerbase_tmm(ob_outerbase* ob, int sq, const uint64_t* terms, uint64_t K,
                     const double* a /* N */, double* out /* K */);
int ob_outerbase_mm_gradhyp(ob_outerbase* ob, int sq, const uint64_t* terms, uint64_t K,
                            const double* a, double* out /* N */, double* outge /* N x H */);
int ob_outerbase_tmm_gradhyp(ob_outerbase* ob, int sq, const uint64_t* terms, uint64_t K,
                             const double* a, double* out /* K */, double* outge /* K x H */);
/* multi right-hand-side versions, prodmm_(mat)/tprodmm_(mat) linalg.cpp:527-557,583-637 */
int ob_outerbase_mm_mat(ob_outerbase* ob, int sq, const uint64_t* terms, uint64_t K,
                        const double* A /* K x C */, uint64_t C, double* out /* N x C */);
int ob_outerbase_tmm_mat(ob_outerbase* ob, int sq, const uint64_t* terms, uint64_t K,
                         const double* A /* N x C */, uint64_t C, double* out /* K x C */);
/* outerbase::residvar / residvar_gradhyp (src/modandbase.cpp:889-922): variance of the terms left out of
 * the basis, 1 - sqmm(terms, getvar(terms)), and its hyper-gradient (N x H). */
int ob_outerbase_residvar(ob_outerbase* ob, const uint64_t* terms, uint64_t K, double* out /* N */);
int ob_outerbase_residvar_gradhyp(ob_outerbase* ob, const uint64_t* terms, uint64_t K, double* out /* N x H */);
/* Device-pointer forms of mm / tmm / mm_mat for callers that keep vectors in HBM
 * (the CG loop, bench.py's `value`).  All *_dev pointers are device memory on
 * ctx's GPU; work is enqueued on ctx's stream and NOT synchronised.
 * set_terms installs the terms table (K x d) they multiply with and must come first:
 * before it every *_dev call and terms_stats return OB_ERR_STATE and enqueue nothing.
 * Buffer lengths, with N the rows of the outerbase and K the terms installed:
 *   mm_dev      a_dev K,       out_dev N   (entries from N on are not written)
 *   tmm_dev     a_dev N,       out_dev K   (whatever follows a_dev's N entries, NaN included, never contributes)
 *   mm_mat_dev  A_dev K x C,   out_dev N x C, column-major, leading dimension N
 *   tmm_mat_dev A_dev N x C,   out_dev K x C, column-major, leading dimensions N and K
 * Any 8-byte-aligned device pointer is accepted: the library itself pads or realigns an
 * input that its kernels stage in whole row tiles. */
int ob_outerbase_set_terms(ob_outerbase* ob, const uint64_t* terms, uint64_t K);
int ob_outerbase_mm_dev(ob_outerbase* ob, int sq, const double* a_dev, double* out_dev);
int ob_outerbase_tmm_dev(ob_outerbase* ob, int sq, const double* a_dev, double* out_dev);
int ob_outerbase_mm_mat_dev(ob_outerbase* ob, int sq, const double* A_dev, uint64_t C, double* out_dev);
int ob_outerbase_tmm_mat_dev(ob_outerbase* ob, int sq, const double* A_dev, uint64_t C, double* out_dev);
/* statistics of the compiled terms program, for the roofline model (SURVEY 8d):
 * W = sum_k (nnz_k + 1), Lcols = distinct basis columns read, nodes = trie nodes. */
int ob_outerbase_terms_stats(ob_outerbase* ob, uint64_t* W, uint64_t* Lcols, uint64_t* nodes,
                             uint64_t* maxdepth);

/* ---- terms-specialised kernels (outerbase_b200/csrc/ob_spec.hpp, ob_spec_scaffold.inc).
 * A terms table stays fixed for every product of a fit (each CG iteration of each optcg,
 * src/fit.cpp:71-85), so the library can compile Phi a / Phi^T r kernels FOR that table at run
 * time (NVRTC, sm_100a): the table becomes straight-line FP64 code with its hot basis columns in
 * registers instead of being interpreted from shared memory.  The reference has no counterpart:
 * it is the GPU analogue of its `vertpl` / `chunksize` loop tuning (src/modandbase.cpp:504-513).
 * Policy, per context ("spec" option; environment OB_SPEC=0|1|auto sets the initial value):
 *   0  never        -- interpreter kernels only
 *   1  at first use -- compile when a table is first multiplied
 *   2  auto         -- (default) once a table has proven hot ("spec_work" row-terms, default
 *                      4e12) or when its module is already in the disk cache
 *                      ($OB_SPEC_CACHE, default ~/.cache/outerbase_b200, "0" disables)
 * ob_outerbase_specialize compiles NOW for one table (like planning an FFT) and reports the
 * seconds spent compiling (0 on a cache hit).  Results of the two kernel families agree to
 * rounding (<= 1e-12 relative), not bitwise: the summation trees differ.
 * Further options: "p2p" 1|0 -- the library's peer-memory allreduce or ncclAllReduce (see
 * ob_ctx_allreduce_dev; the same value on every rank); "dsweep" 0|1 (env OB_DSWEEP) -- the
 * hyper-gradients of a specialised table (prodmmge_ / sqmm_gradhyp contracted with row weights,
 * src/linalg.cpp:139-163, 225-277; loglik_gauss.cpp:127; fit.cpp:259-263) from ONE reverse-mode
 * sweep over the rows (kernel phi_d_spec) instead of one product per hyper-parameter.  dsweep is
 * on by default (same value on every rank; a rank whose module fails to build makes all ranks fall
 * back to the per-hyper products together); "device_cg" 1|0 (env OB_DEVICE_CG) -- lpdf::optcg
 * (src/fit.cpp:37-96) on lpdfvec(logpr_gauss, loglik_gauss) keeps every K-vector and scalar of the
 * loop in HBM (the host reads one stop flag per iteration); 0 = the host loop of round 1;
 * "overlap" 1|0 (env OB_OVERLAP) -- ob_outerbase_mm / _tmm on host buffers of 2^17 rows or more overlap
 * the transfer with the kernel (page-locked result written by the kernel, input vector streamed in
 * on a second stream); 0 = staged copies -- needed under tools that serialise kernels and copies
 * (ncu), where the kernel would wait for rows that cannot arrive (it traps after 20 s);
 * "tmap" 1|0 (env OB_TMAP) -- phi_a_spec stages a row tile with one 2-D tensor copy (cp.async.bulk.tensor) per
 * dimension of the model instead of one bulk copy per basis column. */
int ob_ctx_set_option(ob_ctx* ctx, const char* name, double value);
int ob_outerbase_specialize(ob_outerbase* ob, const uint64_t* terms, uint64_t K, double* compile_seconds);
/* 1: the specialised kernels serve this table, 0: interpreter kernels, -1: not specialisable */
int ob_outerbase_spec_state(ob_outerbase* ob, const uint64_t* terms, uint64_t K, int* state);
/* Test hook (no GPU needed): the CUDA source the generator emits for a table.  opts9 = {ra, qa,
 * tga, cache_a, wt, rt, pt, cache_t, acc_cap} or NULL for the defaults.  Call with buf = NULL to
 * get the length; info = {types, accumulators per thread, tile rows Phi a, tile rows Phi^T}. */
int ob_spec_source(const uint64_t* terms, uint64_t K, uint64_t d, const int* opts9, char* buf,
                   uint64_t* len, uint64_t* info /* 4 */);
/* Test hook (no GPU needed): the source of the hyper-gradient sweep kernel (phi_d_spec: gradhyp of
 * prodmmge_ / sqmm_gradhyp contracted with row weights, src/linalg.cpp:139-163, 225-277) for a table;
 * info = {coefficient slots, tile rows}. */
int ob_spec_source_dot(const uint64_t* terms, uint64_t K, uint64_t d, char* buf, uint64_t* len,
                       uint64_t* info /* 2 */);
/* Test hook (no GPU needed): the source of the transposed multi-right-hand-side kernel (phi_tm_spec: tprodmm_(mat),
 * src/linalg.cpp:583-637, on the FP64 tensor cores) for a table; info = {CTA types, most columns a type stages}. */
int ob_spec_source_tmat(const uint64_t* terms, uint64_t K, uint64_t d, char* buf, uint64_t* len,
                        uint64_t* info /* 2 */);
/* Test hook (no GPU needed): the source of the multi-right-hand-side kernel (phi_am_spec: prodmm_(mat),
 * src/linalg.cpp:527-557, on the FP64 tensor cores) for a table; info = {coefficient blocks per pass, tile rows}. */
int ob_spec_source_mat(const uint64_t* terms, uint64_t K, uint64_t d, char* buf, uint64_t* len,
                       uint64_t* info /* 2 */);
/* Test hook (no GPU needed): compile a source for sm_100a with NVRTC, bypassing the disk
 * cache; returns the cubin size. */
int ob_spec_compile_check(const char* source, uint64_t* cubin_bytes, double* seconds);

/* Host-side self check of the terms compiler (outerbase_b200/csrc/ob_terms.hpp): evaluates
 * ONE row on the CPU by interpreting the compiled warp programs -- bcols holds that row's
 * basemat (M values, knotptst layout).  out_phi_a = sum_k a_k prod_l B[t_kl] ;
 * out_phit[k] = b * prod_l B[t_kl].  aug_dim = -1 for the plain program.  Test hook only:
 * no product path calls it. */
int ob_debug_terms_eval(const uint64_t* terms, uint64_t K, uint64_t d, const uint64_t* knotptst,
                        int ngroups, int aug_dim, const double* bcols, const double* gcols0,
                        const double* a, double b, double* out_phi_a, double* out_phit,
                        uint64_t* stats /* W, Lcols, nodes, maxdepth, fast_ok, nslots, nwords_fwd, nwords_bwd */);
/* Test hook: the layout the interpreter Phi a (transpose = 0) or Phi^T (transpose = 1) kernel runs with for this
 * object's rows and a terms table (plain program, sq selects the squared operator).  out = {R rows per lane, tile
 * buffers, program in shared memory (1) or global memory (0), shared-memory bytes}; R = 0: the brute-force kernels
 * (a table the trie compiler refuses, or no layout fits in shared memory).  Specialised kernels are not reported. */
int ob_outerbase_debug_phi_geometry(ob_outerbase* ob, const uint64_t* terms, uint64_t K, int transpose, int sq,
                                    int* out /* 4 */);

/* ------------------------------------------------------------------ stateless linalg.h seam
 * Exactly the eight free functions of src/linalg.h:9-58: same argument meaning, host
 * buffers, basemat is N x M column-major.  getmge_ follows the reference's unchunked
 * branch for every shape (its row-chunked branch, linalg.cpp:788-810, cannot work:
 * dogetmge_ resizes the whole cube to one chunk and the chunk is never copied back).  vertpl/chunksize/loopsize/num_threads are
 * accepted and ignored.  These upload, run the same CUDA kernels, download. */
int ob_prodmm_vec(ob_ctx* ctx, double* out, const uint64_t* terms, uint64_t K, uint64_t d,
                  const double* a, const double* basemat, uint64_t N, uint64_t M,
                  const double* basescale, const uint64_t* knotptst);
int ob_tprodmm_vec(ob_ctx* ctx, double* out, const uint64_t* terms, uint64_t K, uint64_t d,
                   const double* a, const double* basemat, uint64_t N, uint64_t M,
                   const double* basescale, const uint64_t* knotptst);
int ob_prodmm_mat(ob_ctx* ctx, double* out, const uint64_t* terms, uint64_t K, uint64_t d,
                  const double* A, uint64_t C, const double* basemat, uint64_t N, uint64_t M,
                  const double* basescale, const uint64_t* knotptst);
int ob_tprodmm_mat(ob_ctx* ctx, double* out, const uint64_t* terms, uint64_t K, uint64_t d,
                   const double* A, uint64_t C, const double* basemat, uint64_t N, uint64_t M,
                   const double* basescale, const uint64_t* knotptst);
int ob_prodmmge(ob_ctx* ctx, double* out, double* outge, const uint64_t* terms, uint64_t K, uint64_t d,
                const double* a, const double* basemat, uint64_t N, uint64_t M,
                const double* basescale, const uint64_t* knotptst,
                const double* basematge, uint64_t Mge, const uint64_t* gest,
                const uint64_t* hypmatch, uint64_t H);
int ob_tprodmmge(ob_ctx* ctx, double* out, double* outge, const uint64_t* terms, uint64_t K, uint64_t d,
                 const double* a, const double* basemat, uint64_t N, uint64_t M,
                 const double* basescale, const uint64_t* knotptst,
                 const double* basematge, uint64_t Mge, const uint64_t* gest,
                 const uint64_t* hypmatch, uint64_t H);
int ob_getm(ob_ctx* ctx, double* out, const uint64_t* terms, uint64_t K, uint64_t d,
            const double* basemat, uint64_t N, uint64_t M,
            const double* basescale, const uint64_t* knotptst);
/* getmge_, src/linalg.cpp:724-822: outge is N x K x H (one slice per hyper-parameter). */
int ob_getmge(ob_ctx* ctx, double* outge, const uint64_t* terms, uint64_t K, uint64_t d,
              const double* basemat, uint64_t N, uint64_t M,
              const double* basescale, const uint64_t* knotptst,
              const double* basematge, uint64_t Mge, const uint64_t* gest,
              const uint64_t* hypmatch, uint64_t H);

/* ------------------------------------------------------------------ lpdf family
 * loglik_gauss  src/lpdfs/loglik_gauss.cpp:41-179   (device)
 * logpr_gauss   src/lpdfs/logpr_gauss.cpp:41-145    (K-vectors)
 * loglik_std    src/lpdfs/loglik_std.cpp:41-203     (device; full Hessian = tensor-core Phi^T Phi)
 * lpdfvec       src/fit.cpp:174-301,310-428,503-612 (diagonal and full-Hessian branches)
 * lpdf::optcg   src/fit.cpp:37-96 ; optnewton :98-131 ; paralpdf :133 ; paralpdf_grad :146. */
int ob_loglik_gauss_create(ob_ctx* ctx, ob_outermod* om, const uint64_t* terms, uint64_t K,
                           const double* y, const double* x, uint64_t N, ob_lpdf** out);
int ob_logpr_gauss_create(ob_ctx* ctx, ob_outermod* om, const uint64_t* terms, uint64_t K, ob_lpdf** out);
/* new(loglik_gda, om, terms, y, x) -- src/lpdfs/loglik_gda.cpp:47-239, src/interfaceR.cpp:745-750: the stage-1
 * likelihood of obfit (R/fitting.R:84), two parameters (noisescale, lik.coeffscale); flag "dodiag" = doda. */
int ob_loglik_gda_create(ob_ctx* ctx, ob_outermod* om, const uint64_t* terms, uint64_t K,
                         const double* y, const double* x, uint64_t N, ob_lpdf** out);
/* new(loglik_std, om, terms, y, x) -- src/lpdfs/loglik_std.cpp:41-59, src/interfaceR.cpp:733-737: loglik_gauss's model
 * with the K x K Hessian (hess / hessgradhyp / hessgradpara), what lpdf::optnewton needs.  The reference holds the
 * explicit N x K basis and its N x K x H gradient cube (getmge_, broken for row-chunked bases: linalg.cpp:788-810);
 * here values and gradients come from the implicit products and only the Hessians touch explicit matrices. */
int ob_loglik_std_create(ob_ctx* ctx, ob_outermod* om, const uint64_t* terms, uint64_t K,
                         const double* y, const double* x, uint64_t N, ob_lpdf** out);
/* new(lpdfvec, a, b): a is child 0 (grad/gradhyp are sized from it, fit.cpp:338-343). */
int ob_lpdfvec_create(ob_lpdf* a, ob_lpdf* b, ob_lpdf** out);
int ob_lpdf_destroy(ob_lpdf* l);
int ob_lpdf_setnthreads(ob_lpdf* l, int k);
int ob_lpdf_update(ob_lpdf* l, const double* coeff, uint64_t K);
int ob_lpdf_updateom(ob_lpdf* l);
int ob_lpdf_updatepara(ob_lpdf* l, const double* para, uint64_t npara);
int ob_lpdf_updateterms(ob_lpdf* l, const uint64_t* terms, uint64_t K);
int ob_lpdf_optcg(ob_lpdf* l, double tol, uint64_t maxepch);
/* lpdf::optnewton, src/fit.cpp:98-131: one Newton step coeff += solve(hess, grad); sets fullhess. */
int ob_lpdf_optnewton(ob_lpdf* l);
int ob_lpdf_hessmult(ob_lpdf* l, const double* g, double* out /* K */);
/* hess / hessgradhyp / hessgradpara (fit.h:86-88): K x K, K x K x H, K x K x npara column-major; an object without a
 * full Hessian (loglik_gauss, loglik_gda) returns n = 0 as the reference returns empty matrices. */
int ob_lpdf_hess(ob_lpdf* l, double* out /* K x K */, uint64_t* n);
int ob_lpdf_hessgradhyp(ob_lpdf* l, double* out /* K x K x H */, uint64_t* n);
int ob_lpdf_hessgradpara(ob_lpdf* l, double* out /* K x K x npara */, uint64_t* n);
int ob_lpdf_diaghess(ob_lpdf* l, double* out /* K */);
int ob_lpdf_diaghessgradhyp(ob_lpdf* l, double* out /* K x H */);
int ob_lpdf_diaghessgradpara(ob_lpdf* l, double* out /* K x npara */);
int ob_lpdf_paralpdf(ob_lpdf* l, const double* para, uint64_t npara, double* out);
int ob_lpdf_paralpdf_grad(ob_lpdf* l, const double* para, uint64_t npara, double* out);
/* flags: which in {"compute_val","compute_grad","compute_gradhyp","compute_gradpara",
 * "domarg", "fullhess"} -- the C++ member names (NOT the swapped R names, interfaceR.cpp:700-701). */
int ob_lpdf_set_flag(ob_lpdf* l, const char* which, int value);
int ob_lpdf_sizes(ob_lpdf* l, uint64_t* nterms, uint64_t* npara, uint64_t* nhyp, uint64_t* nrow);
/* which in {"val"(1),"grad"(K),"gradhyp"(H),"gradpara"(npara),"coeff"(K),"para"(npara),
 * "yhat"(N, loglik_gauss),"coeffsd"(K, logpr_gauss),"totdiaghess"(K),
 * "tothess"(K x K, after a full-Hessian build), "cg_iters"(1, iterations the last optcg ran)}. */
int ob_lpdf_get(ob_lpdf* l, const char* which, double* out, uint64_t* n);
/* set coeff (warm start, fit.cpp:45-48 keeps coeff across optcg calls). */
int ob_lpdf_set_coeff(ob_lpdf* l, const double* coeff, uint64_t K);

/* predictor(lpdf) / pred_gauss: src/lpdfs/loglik_gauss.cpp:196-227 ; pred_gda: loglik_gda.cpp:249-283 ;
 * predr_std: loglik_std.cpp:219-257 */
int ob_predictor_create(ob_lpdf* loglik, ob_predictor** out);
int ob_predictor_destroy(ob_predictor* p);
int ob_predictor_update(ob_predictor* p, const double* x, uint64_t N);
int ob_predictor_mean(ob_predictor* p, double* out /* N */);
int ob_predictor_var(ob_predictor* p, double* out /* N */);

#ifdef __cplusplus
}
#endif
#endif /* OUTERBASE_B200_H */

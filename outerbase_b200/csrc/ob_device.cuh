/*
 * ob_device.cuh -- device context, buffers and launcher declarations of the product.
 * sm_100a only; there is NO CPU fallback: every entry point fails with OB_ERR_NOGPU
 * when no CUDA device is present.
 */
#pragma once
#include <cuda_runtime.h>

#include <cstdint>
#include <cstdio>
#include <map>
#include <memory>
#include <stdexcept>
#include <string>
#include <vector>

#include "ob_model.hpp"
#include "ob_spec.hpp"
#include "ob_terms.hpp"

namespace obd {

using u64 = uint64_t;

struct CudaError : std::runtime_error { using std::runtime_error::runtime_error; };
struct NcclError : std::runtime_error { using std::runtime_error::runtime_error; };
struct NoGpuError : std::runtime_error { using std::runtime_error::runtime_error; };

#define OB_CUDA(expr)                                                                          \
  do {                                                                                         \
    cudaError_t e__ = (expr);                                                                  \
    if (e__ != cudaSuccess)                                                                    \
      throw obd::CudaError(std::string(#expr) + ": " + cudaGetErrorString(e__) + " (" + __FILE__ + ":" + std::to_string(__LINE__) + ")"); \
  } while (0)

/* ---- NCCL, bound at run time so that the library loads without it and shares the
 * libnccl.so.2 already mapped by the host process (e.g. torch's). */
struct NcclUid { char b[128]; }; /* ncclUniqueId, passed BY VALUE to ncclCommInitRank */
struct NcclApi {
  void* handle = nullptr;
  int (*GetUniqueId)(NcclUid*) = nullptr;
  int (*CommInitRank)(void**, int, NcclUid, int) = nullptr;
  int (*AllReduce)(const void*, void*, size_t, int, int, void*, cudaStream_t) = nullptr;
  int (*AllGather)(const void*, void*, size_t, int, void*, cudaStream_t) = nullptr;
  int (*CommDestroy)(void*) = nullptr;
  const char* (*GetErrorString)(int) = nullptr;
  static NcclApi& get();
};

struct Ctx {
  int device = 0;
  int sms = 148;
  size_t smem_optin = 0;
  cudaStream_t stream = nullptr;
  u64 launches = 0;
  void* comm = nullptr;
  int nranks = 1, rank = 0;
  double* pinned = nullptr; /* small pinned scratch for scalar read-back */
  /* one-shot allreduce over NVLink peer memory (p2p_allreduce_kernel): every rank stores its K-vector straight into
   * a slot of every peer's buffer and adds the slots it received in rank order.  Buffers are exchanged as CUDA IPC
   * handles over the NCCL communicator at comm_init; NCCL stays the path for payloads above kCap doubles and when
   * peer access is not available (p2p.G == 0). */
  struct P2P {
    static constexpr int kMaxRanks = 8;
    static constexpr size_t kCap = 65536;      /* elements (16 bytes each: value + tags) per slot */
    static constexpr int kThreads = 256;
    int G = 0;
    bool enabled = true;                       /* option "p2p": 0 sends everything through NCCL */
    void* local = nullptr;                     /* slots [parity 2][rank G][kCap] */
    void* peer[kMaxRanks] = {};                /* the same block of every rank, peer[rank] == local */
    unsigned seq = 0;                          /* tag of the current call (never 0) */
    unsigned long long timeout_ns = 300ull * 1000000000ull; /* a rank may sit in a run-time compile while its peers poll */
  } p2p;
  /* terms-specialised kernels (ob_spec.hpp): 0 never, 1 at first use, 2 once a table has proven hot
   * (spec_work row-terms processed by the interpreter kernels) or its module is in the disk cache */
  int spec_mode = 2;
  double spec_work = 4e12;
  /* hyper-gradients of a specialised table from one reverse-mode sweep (phi_d_spec) instead of one product per
   * hyper-parameter: option "dsweep" / env OB_DSWEEP (same value on every rank).  On by default: measured on a B200 in
   * round 2 (profiles/r02_dsweep.json: one C3 objective evaluation 43.4 -> 25.8 ms, parity 9e-16 against the per-hyper
   * path).  A rank that cannot run the sweep (module build failure) makes ALL ranks fall back together. */
  bool dsweep = true;
  explicit Ctx(int dev);
  ~Ctx();
  void sync() { OB_CUDA(cudaStreamSynchronize(stream)); }
  void allreduce_sum(double* buf_dev, size_t n);
  bool p2p_ok(size_t n) const;
  /* Fusion of a Phi^T product with the allreduce that follows it: fuse_allreduce(n) before the product asks the next
   * launch_phi_t_reduce to combine the ranks in the same launch; allreduce_after(out, n) afterwards does the plain
   * allreduce when the product did not end in that kernel (rows == 0, brute-force kernels). */
  size_t fuse_n = 0;
  bool fused = false;
  /* one more element rides on a fused Phi^T tail: the fixed-order sum of `fuse_extra_n` doubles (the per-CTA sums of
   * squared residuals of the preceding Phi a launch, loglik_gauss.cpp:122) lands in out[K]; extra_done tells the
   * caller whether the launch took care of it */
  const double* fuse_extra = nullptr;
  int fuse_extra_n = 0;
  bool extra_done = false;
  /* lpdf::optcg with every K-vector in HBM (option "device_cg", env OB_DEVICE_CG; on by default) */
  bool device_cg = true;
  /* host-pointer mm / tmm overlap their transfers with the kernel (option "overlap", env OB_OVERLAP; on by default).
   * Off under tools that serialise kernels and copies (ncu): the kernel would wait for rows that cannot arrive. */
  bool overlap = true;
  /* phi_a_spec stages its tiles with 2-D tensor copies (option "tmap", env OB_TMAP; on by default): 0 = one bulk copy
   * per column, as phi_t_spec does */
  bool tmap = true;
  void fuse_allreduce(size_t n) { fused = false; fuse_n = p2p_ok(n) ? n : 0; }
  void allreduce_after(double* buf_dev, size_t n) {
    fuse_n = 0;
    if (!fused) allreduce_sum(buf_dev, n);
    fused = false;
  }
  struct FuseScope { /* exception-safe request: a product that throws must not leave the request armed */
    Ctx& c;
    FuseScope(Ctx& c_, size_t n, const double* extra = nullptr, int extra_n = 0) : c(c_) {
      c.fuse_allreduce(n);
      c.fuse_extra = extra; c.fuse_extra_n = extra ? extra_n : 0; c.extra_done = false;
    }
    ~FuseScope() { c.fuse_n = 0; c.fuse_extra = nullptr; c.fuse_extra_n = 0; }
  };
  void p2p_init();  /* after the NCCL communicator exists; leaves p2p.G == 0 when peer memory cannot be mapped */
  void p2p_release();
  /* one call of the peer-memory protocol issued from another kernel (the fused tail of phi_t_spec): the slot blocks of
   * all ranks and the next sequence number */
  struct P2PCall { void* slots[P2P::kMaxRanks]; int G, rank; unsigned seq; unsigned long long timeout_ns; };
  P2PCall p2p_next_call();
  /* grid barrier of kernels that reduce in their own tail: a monotonic arrival counter, `sync_count` = arrivals
   * requested so far (the target a launch waits for) */
  unsigned* sync_ctr = nullptr;
  unsigned sync_count = 0;
  unsigned* grid_sync_counter();
  /* Host-pointer calls of the reference's interface (outerbase::tmm with a host vector) overlap the host -> device copy
   * with the kernel that consumes it: the copy runs in chunks on `copy_stream`, each followed by a 4-byte copy that
   * publishes the rows that have arrived in `rows_ready`; the Phi^T producers poll it before staging a tile.
   *   stream_rows_begin()        (main stream) reset the counter, returns its device address
   *   ... launch the consumer on the main stream ...
   *   stream_rows_copy(dst, src, n)   issue the chunked copy (after the launch: a pageable source blocks the host)
   *   stream_rows_end()          main stream waits for the copy */
  cudaStream_t copy_stream = nullptr;
  cudaEvent_t ev_main = nullptr, ev_copy = nullptr;
  unsigned* rows_ready = nullptr;
  unsigned* rows_table = nullptr; /* pinned: the values published after each chunk */
  const unsigned* stream_rows_begin();
  void stream_rows_copy(double* dst_dev, const double* src_host, size_t n);
  void stream_rows_end();
  /* device address of a caller's host buffer when it is page-locked and mapped (kernels then write results straight
   * into it, overlapping the device -> host transfer with the computation), else null */
  static double* mapped_host_pointer(double* host);
};

/* device buffer, grows on demand, never shrinks */
template <class T>
struct DevBuf {
  T* p = nullptr;
  size_t cap = 0;
  DevBuf() {}
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
  ~DevBuf() { if (p) cudaFree(p); }
  T* ensure(size_t n) {
    if (n > cap) {
      if (p) cudaFree(p);
      p = nullptr;
      OB_CUDA(cudaMalloc(&p, std::max<size_t>(n, 1) * sizeof(T)));
      cap = n;
    }
    return p;
  }
  void upload(const T* h, size_t n, cudaStream_t s) {
    ensure(n);
    if (n) OB_CUDA(cudaMemcpyAsync(p, h, n * sizeof(T), cudaMemcpyHostToDevice, s));
  }
  void upload(const std::vector<T>& h, cudaStream_t s) { upload(h.data(), h.size(), s); }
};

constexpr int kTileRowsMax = 128;

/* how one tile column is produced from what the bulk copies delivered */
enum ColOp : int { COL_COPY = 0, COL_SQUARE = 1, COL_TWO_G_B = 2 };

/* per (program, sq, hyper) pointer table: where each tile column is read from */
struct ColTable {
  DevBuf<const double*> load_src; /* ncol + naux base pointers (row 0 of the column) */
  DevBuf<int> col_op;             /* ncol entries: op | (auxcol << 8) */
  int ncol = 0, nload = 0;
  bool has_ops = false;
  std::vector<const double*> src_host; /* host image of load_src (tensor maps are encoded from it) */
  /* 2-D tensor maps of phi_a_spec's tile (one per run of adjacent columns), built at first use for one tile height */
  mutable DevBuf<unsigned char> tmaps;
  mutable int tmap_tr = 0, tmap_state = 0; /* 0 not built, 1 ready, -1 unavailable for this table */
};

/* compiled terms, resident on the device */
struct DevProgram {
  obt::Program host;
  DevBuf<uint32_t> fwd, bwd, fwd_off, bwd_off, slot_base, slot_real, csr_ptr, csr_col;
  DevBuf<int32_t> slot_term;
  void upload(cudaStream_t s);
};

enum PhiMode : int { PHI_PLAIN = 0, PHI_UPDATE = 1, PHI_HESS = 2, PHI_DOT = 3 };

struct PhiAArgs {
  const double* a = nullptr;       /* K coefficients (device) */
  double* out = nullptr;           /* N: yhat (PLAIN/UPDATE) ; may be null for HESS */
  double* w = nullptr;             /* N: UPDATE: -((yhat-y)/sd)/sd ; HESS: (yhat/sd)/sd */
  const double* y = nullptr;       /* UPDATE */
  double sd = 1.0;
  double* ssq_partial = nullptr;   /* UPDATE / DOT: one partial per CTA (device, >= grid entries) */
  /* DOT (specialised kernel only): partial += wdot[n] * (out_n + y[n] * yh[n]); nothing is stored */
  const double* wdot = nullptr;
  const double* yh = nullptr;
  int mode = PHI_PLAIN;
};

/* everything one Phi-type launch needs besides the vectors */
struct PhiPlan {
  const DevProgram* prog = nullptr;
  const ColTable* cols = nullptr;
  const double* scale = nullptr;   /* basescale (N) */
  int sq = 0;                      /* use scale^2 */
  u64 N = 0;
  u64 ld = 0;                      /* rows every column is allocated with (0: unknown -- no tensor maps) */
};

struct Workspace {
  DevBuf<double> partial;  /* Phi^T: grid x nslots partial sums */
  DevBuf<double> ssq;      /* per-CTA residual sums of squares */
};

int phi_grid(const Ctx& c, u64 N, int tile_rows);
/* Phi a (trie/Horner kernel, or the brute-force kernel when the program is not fast_ok) */
void launch_phi_a(Ctx& c, const PhiPlan& pl, const PhiAArgs& args, Workspace& ws, int* grid_out);
/* Phi^T w -> out (K, device); result is the LOCAL (this rank's rows) sum */
void launch_phi_t(Ctx& c, const PhiPlan& pl, const double* w, double* out, Workspace& ws);
void launch_phi_t_reduce(Ctx& c, const double* partial, int nblocks, int nslots, const int32_t* slot_term, double* out);
/* the layout launch_phi_a (is_a) / launch_phi_t picks for a plan: {rows per lane R, tile buffers, program in shared
 * memory, shared-memory bytes}; R == 0 means the brute-force kernels */
void phi_geometry_info(const Ctx& c, const PhiPlan& pl, bool is_a, int out[4]);
/* ---- terms-specialised kernels (ob_spec.hpp generator, ob_spec_scaffold.inc frame, ob_spec_rt.cu run time) */
struct SpecKernels;
bool spec_compiler_available();
obs::SpecOptions spec_default_options();
obs::SpecOptions spec_adapt_options(const Ctx& c, obs::SpecOptions o, int ncol, size_t nslots);
/* pa: program with G = opt.wa, pt: G = types * opt.wt.  only_if_cached: return null instead of compiling */
std::shared_ptr<SpecKernels> spec_build(Ctx& c, const obt::Program& pa, const obt::Program& pt, int types, const obs::SpecOptions& opt,
                                        bool only_if_cached);
double spec_compile_seconds(const SpecKernels& k);
std::string spec_compile_nocache(const std::string& src, double* seconds);
bool spec_fits(const Ctx& c, const SpecKernels& k, int ncol);
bool spec_uses_cluster(const SpecKernels& k);
bool launch_phi_tm_spec(Ctx& c, SpecKernels& k, const PhiPlan& pl, int types, const double* A, u64 lda, u64 C, double* out);
/* true when [p, p + bytes) lies inside one device allocation (cuMemGetAddressRange through the runtime's driver entry point) */
bool device_range_readable(const void* p, size_t bytes);
void launch_phi_a_spec(Ctx& c, SpecKernels& k, const PhiPlan& pl, const PhiAArgs& args, Workspace& ws, int* grid_out);
void launch_phi_t_spec(Ctx& c, SpecKernels& k, const PhiPlan& pl, const double* w, double* out, Workspace& ws, const unsigned* ready = nullptr);
/* Phi . A on the FP64 tensor cores (phi_am_spec): A is K x C column-major (device), out N x C with leading dimension ldo.
 * The module is generated and compiled at first use.  Returns false when the tile does not fit (caller: column loop). */
/* model-side tables of the hyper-gradient sweep (phi_d_spec): where the gradient columns of each hyper-parameter live */
struct DotArgs {
  const double* gmat = nullptr; /* basemat_gradhyp (leading dimension ld) */
  const double* bmat = nullptr; /* squared operator: the plain basemat, else null */
  u64 ld = 0;
  int H = 0, d = 0;
  const u64* hypst = nullptr;    /* d + 1 */
  const u64* gest = nullptr;     /* H + 1 */
  const u64* knotptst = nullptr; /* d + 1 */
};
bool launch_phi_d_spec(Ctx& c, SpecKernels& k, const PhiPlan& pl, const double* a_dev, const double* w_dev, const DotArgs& g, double* out_dev);
bool launch_phi_am_spec(Ctx& c, SpecKernels& k, const PhiPlan& pl, const double* A, u64 C, double* out, u64 ldo);
/* coefficient blocks in emit order, columns of odd rows swizzled (ob_spec_scaffold.inc, phi_am_spec) */
void launch_gather_coef_blocks(Ctx& c, const double* A, u64 K, u64 col0, int ncols, const int32_t* slot_term, int nslots, int nrows, double* out);
/* explicit Phi (N x K column-major, device), getm_ linalg.cpp:685-715 */
void launch_getmat(Ctx& c, const PhiPlan& pl, double* out, u64 ldo);
/* sum of n per-CTA partials, fixed order -> out[0] */
void launch_sum_partials(Ctx& c, const double* partial, int n, double* out);

/* ---- device-resident CG (lpdf::optcg, src/fit.cpp:37-96, on lpdfvec(logpr_gauss, loglik_gauss) in either order): the
 * K-vector algebra of one iteration between the Phi kernels, ONE single-CTA launch per stage, every vector and scalar
 * in HBM, so that an iteration never waits for the host.  Sums use one fixed tree order (deterministic; the reference's
 * two-accumulator `accu` order is sequential and would cost ~8 us per sum on one thread -- the iterates differ by
 * rounding, inside the 1e-8 budget of the fit). */
enum CgStage : int {
  CG_INIT = 0,              /* after the first update() (host path): rm = grad / m ; p = rm                         (:58-60)  */
  CG_FINISH_Q = 1,          /* q = hessmult(p) = lik part + p / (sd sca)^2 in child order                          (:59)     */
  CG_STEP = 2,              /* q as above; num = grad.rm ; stop test ; denom = q.p ; alpha ; coeff += alpha p ; valo (:72-77) */
  CG_POST_UPDATE = 3        /* grad, val ; valdiff ; rm ; num2 = -(alpha q).rm ; beta ; p = rm + beta p             (:79-83) */
};
/* Column-batched form (loglik_gauss_multi): the launch runs one CTA per column; coeff, grad, m, rm, p, q and red are K x C
 * column-major, scal holds CG_NSCAL scalars per column, sds is shared.  ncol = 1 with ssq = running = null is the
 * single-response launch.  Per-column para: CTA c reads entry c of sca_col, obssd_col and vma_col instead of the
 * scalar, for each of them that is set (uploaded once per optcg, not per iteration). */
struct CgParams {
  int K, stage, lik_first, domarg;
  double* coeff; double* grad; const double* m; double* rm; double* p; double* q;
  const double* red;    /* K + 1: likelihood part of grad (update) or of the Hessian product (hessmult) | sum of squared residuals */
  const double* sds;    /* K: coeffsd (logpr_gauss.cpp:57) */
  double sca, obssd, nglobal, val_margadj, tol;
  double* scal;         /* [0] num [1] denom [2] alpha [3] beta [4] val [5] valo [6] valdiff [7] stop [8] val_lik [9] val_pr [10] iter */
  const double* ssq = nullptr;  /* batched: per-column sums of squared residuals (red then holds K per column) */
  unsigned* running = nullptr;  /* batched: running[iter & 1] counts the columns that did not stop in CG_STEP of iteration iter */
  int iter = 0;
  const double* sca_col = nullptr;    /* batched, per-column coefficient scale: C entries replacing sca */
  const double* obssd_col = nullptr;  /* batched, per-column noise sd: C entries replacing obssd */
  const double* vma_col = nullptr;    /* batched, per-column marginal adjustment: C entries replacing val_margadj */
  /* loglik_gda_multi: the likelihood value is -0.5 ssq - sumlogsd (sumlogsd = sum_i log obssd_i, shared by the columns)
   * instead of -0.5 ssq - nglobal log obssd */
  int use_sumlogsd = 0;
  double sumlogsd = 0;
  /* posterior draws (DESIGN §3.9): K x C prior means; CG_POST_UPDATE takes (coeff - prior_mean) / sd for the prior's
   * value and gradient.  Null: every prior is centred at 0 (every other launch) */
  const double* prior_mean = nullptr;
};
enum { CG_NUM = 0, CG_DENOM, CG_ALPHA, CG_BETA, CG_VAL, CG_VALO, CG_VALDIFF, CG_STOP, CG_VAL_LIK, CG_VAL_PR, CG_ITER, CG_NSCAL = 16 };
void launch_cg_stage(Ctx& c, const CgParams& p, u64 ncol = 1);
/* after mm_mat_dev on C columns (leading dimension ld): update: w = -((yhat - y)/sd)/sd, ssq_out[c] = sum of
 * ((yhat - y)/sd)^2 over column c (fixed order); hessmult: w = (yhat/sd)/sd.  Pad rows of w are zero; yhat may alias w.
 * sd_cols (device, C entries), when set, gives column c the sd sd_cols[c] instead of sd; sd_rows (device, ld entries),
 * when set, gives row i of every column the sd sd_rows[i] (loglik_gda's per-row noise) instead of either. */
void launch_resid_multi(Ctx& c, const double* yhat, const double* y, double* w, u64 N, u64 ld, u64 C, double sd, bool update,
                        DevBuf<double>& partial, double* ssq_out, const double* sd_cols = nullptr, const double* sd_rows = nullptr);

/* ---- standard normals of the posterior draws (DESIGN §3.9), the same on the host and the device.
 * Philox4x32-10 (Salmon, Moraes, Dror, Shaw, SC'11; the constants of Random123) with key (seed low 32, seed high 32) and
 * counter (index, stream, column, 0).  One output gives two uniforms in (0, 1], u = ((x >> 11) + 1) 2^-53 with x the
 * 64-bit words (v1 v0) and (v3 v2), and two normals by Box-Muller: r cos(2 pi u2), r sin(2 pi u2), r = sqrt(-2 log u1).
 * Normal i of (seed, stream, column) is component i & 1 of index i >> 1, so a value depends on nothing but these four. */
enum DrawStream : uint32_t { DRAW_ROWS = 0 /* row noise eps */, DRAW_PRIOR = 1 /* prior noise xi */ };
__host__ __device__ inline uint32_t philox_mulhilo(uint32_t a, uint32_t b, uint32_t* lo) {
  *lo = a * b;
#ifdef __CUDA_ARCH__
  return __umulhi(a, b);
#else
  return (uint32_t)(((uint64_t)a * b) >> 32);
#endif
}
__host__ __device__ inline void philox4x32_10(uint32_t c[4], uint32_t k0, uint32_t k1) {
  for (int r = 0; r < 10; ++r) {
    if (r) { k0 += 0x9E3779B9u; k1 += 0xBB67AE85u; }
    uint32_t lo0, lo1;
    const uint32_t hi0 = philox_mulhilo(0xD2511F53u, c[0], &lo0), hi1 = philox_mulhilo(0xCD9E8D57u, c[2], &lo1);
    const uint32_t n0 = hi1 ^ c[1] ^ k0, n2 = hi0 ^ c[3] ^ k1;
    c[0] = n0; c[1] = lo1; c[2] = n2; c[3] = lo0;
  }
}
/* normals 2 index and 2 index + 1 of (seed, stream, column) */
__host__ __device__ inline void draw_normal_pair(uint64_t seed, uint32_t stream, uint32_t column, uint32_t index, double z[2]) {
  uint32_t c[4] = {index, stream, column, 0u};
  philox4x32_10(c, (uint32_t)seed, (uint32_t)(seed >> 32));
  const double u1 = (double)((((uint64_t)c[1] << 32 | c[0]) >> 11) + 1) * 0x1p-53;
  const double u2 = (double)((((uint64_t)c[3] << 32 | c[2]) >> 11) + 1) * 0x1p-53;
  const double r = sqrt(-2.0 * log(u1)), th = 6.283185307179586 * u2;
  z[0] = r * cos(th);
  z[1] = r * sin(th);
}
/* the perturbations of S posterior draws, one launch: y[i, s] = y0[i] + sigma eps_s[i] for the N rows (pad rows of the
 * ld x S y written 0) and delta[k, s] = (sds[k] sca) xi_s[k] (K x S), eps and xi the normals of streams DRAW_ROWS and
 * DRAW_PRIOR in column s */
void launch_draws_perturb(Ctx& c, const double* y0, u64 N, u64 ld, double sigma, const double* sds, double sca, u64 K, u64 S,
                          uint64_t seed, double* y, double* delta);

/* ---- Sobol sensitivity indices of a tensor-product model (DESIGN §3.10).  R_l(x, j) = basemat[x, col0 + j] scalemat[x, l]
 * is the basis of dimension l at level j; the tables are its mean mu_l[j] and centred second moment C_l[j, j'] over the
 * rows of X_q.  mu_l starts at mu_off of the mu table, C_l (mo x mo, column-major, symmetric) at c_off of the C table. */
struct SobolDim { int col0, mo, mu_off, c_off; };
constexpr int kSobolMomBlocks = 256; /* row slices of the moments kernel: partials per table entry */
constexpr size_t kSobolStageBytes = 48 * 1024; /* the forms kernel stages the tables in shared memory up to this size */
/* stage 0: musum[mu_off + j] = sum over the N rows of R_l(., j); stage 1: csum[c_off + j + mo j'] = sum of
 * (R_l(., j) - mu[mu_off + j]) (R_l(., j') - mu[mu_off + j']).  Fixed row partition (kSobolMomBlocks slices of 32-row
 * tiles), partials added in index order: the same bits on every run.  partial holds kSobolMomBlocks doubles per entry. */
void launch_sobol_moments(Ctx& c, int stage, const double* basemat, const double* scalemat, u64 N, u64 ld,
                          const std::vector<SobolDim>& dims, const SobolDim* dims_dev, const double* mu, double* partial,
                          double* out);
/* out[(b (2d + 1) + f)] for the B columns of coeff (K x B): f = 0 the variance form, 1 + l the first-order form of
 * dimension l, 1 + d + l its total-effect form, each sum_{k <= k'} w theta_kb theta_k'b F_f(k, k') with w = 2 off the
 * diagonal.  The pairs are cut into chunks and CTAs by K alone, so column b's result depends on nothing but column b
 * and is the same bits on every run.  The tables (mu_n + c_n doubles) are staged in shared memory when they take at
 * most kSobolStageBytes, read through the cache otherwise.  partial holds sobol_forms_partials(K) doubles per output. */
u64 sobol_forms_partials(u64 K);
void launch_sobol_forms(Ctx& c, const u64* terms, u64 K, u64 d, const SobolDim* dims_dev, const double* mu, u64 mu_n,
                        const double* cov, u64 c_n, const double* coeff, u64 B, double* partial, double* out);
/* Second-order forms (DESIGN §3.11), P = d (d - 1) / 2 input pairs (l, m), l < m, r = l d - l (l + 1) / 2 + m - l - 1:
 * out[b 2P + 2 r] = sum_{k <= k'} w theta_kb theta_k'b c_l c_m prod_{j not in {l, m}} p_j (pure second-order variance)
 * and out[b 2P + 2 r + 1] the same with g_j in the product (superset importance).  A GEMM over the term pairs on the
 * FP64 tensor cores; the term-pair chunks and output blocks depend on K and d alone, so column b's result depends on
 * nothing but column b and is the same bits on every run.  Nothing is launched when P = 0.  coeff_t holds the
 * coefficients transposed (B x K column-major: the B columns of term k are adjacent).  partial holds
 * sobol_pairs_partials(K, d) doubles per output. */
u64 sobol_pairs_partials(u64 K, u64 d);
void launch_sobol_pairs(Ctx& c, const u64* terms, u64 K, u64 d, const SobolDim* dims_dev, const double* mu, u64 mu_n,
                        const double* cov, u64 c_n, const double* coeff_t, u64 B, double* partial, double* out);
/* Shapley effects (DESIGN §3.12): out[b d + l] = sum_{k <= k'} w theta_kb theta_k'b c_l sum_i w_i prod_{j != l} h_j(z_i),
 * h_j(z) = p_j + z c_j, with nodes = z_0 .. z_{n-1}, w_0 .. w_{n-1} (device memory) a quadrature rule on [0, 1] exact
 * for degree d - 1.  A GEMM over the term pairs on the FP64 tensor cores; the term-pair chunks and the k-step split
 * depend on K and d alone, so column b's result depends on nothing but column b and is the same bits on every run.
 * coeff_t as launch_sobol_pairs.  partial holds sobol_shapley_partials(K) doubles per output. */
u64 sobol_shapley_partials(u64 K);
void launch_sobol_shapley(Ctx& c, const u64* terms, u64 K, u64 d, const SobolDim* dims_dev, const double* mu, u64 mu_n,
                          const double* cov, u64 c_n, const double* coeff_t, u64 B, const double* nodes, u64 n,
                          double* partial, double* out);

/* basis build: cov(x, knots) . rotmat, normalise (modandbase.cpp:285-327, 547-626) */
struct BuildDims {
  int kind; int m; int nh;
  int mo = 0;    /* leading columns (levels 0 .. mo-1) to build and store; 0 = all m */
  double hyp[2];
  u64 knot_off;  /* offset of this dim's knots in the transformed-knot arrays */
  u64 col_off;   /* knotptst[l] */
  u64 ge_off[2]; /* gest[h] for the dim's hypers */
  u64 rot_off;   /* column offset of the dim's block in rotmat */
  u64 rotg_off[2];
};
/* the kernel one dimension was built with: mma = 1 the DMMA kernel (tile = NT column tiles of 8), 0 the FMA kernel
 * (tile = ROWS rows per CTA); mo columns built; smem dynamic shared-memory bytes */
struct BuildGeom { int mma, tile, mo, smem; };
/* geom receives one entry per dimension.  Every dimension's kernel is chosen before any is launched: a dimension with
 * more knots than any kernel holds throws std::range_error and nothing is written. */
void launch_basis_build(Ctx& c, const std::vector<BuildDims>& dims, const double* x_dev, u64 N, u64 ld,
                        const double* knots_dev, const double* rot_dev, u64 rot_ld, const double* rotg_dev,
                        double* basemat, double* basematge, double* scalemat, double* scale, bool dograd,
                        std::vector<BuildGeom>& geom);
void launch_getbase(Ctx& c, const double* basemat, const double* scalemat_col, u64 N, u64 ld, u64 col0, u64 m, double* out);
void launch_cov(Ctx& c, int kind, const double* hyp, const double* x1, u64 n1, const double* x2, u64 n2,
                double* out, double* outg /* may be null */);
/* FP64 FMA peak of this GPU in TFLOP/s (micro-benchmark, ~50 ms) */
double measure_fp64_peak(Ctx& c);
/* C[:, j-1] = G[:, j] - G[:, 0] % B[:, j], j = 1..L: the factor the reference's domultgesub_ applies to
 * T_k^(-l) (linalg.cpp:139-163); sq: the same for the squared matrices, basematsq_gradhyp = 2 G % B
 * (modandbase.cpp:588-590): C_j = 2 B_j % (G_j - G_0 % B_j) */
void launch_gradcols(Ctx& c, const double* B, const double* G, u64 ld, u64 L, double* out, int sq = 0);
/* out[i] = in[i]^2 */
void launch_square(Ctx& c, const double* in, u64 n, double* out);
/* out[n] = c * g[n] * w[n] */
void launch_scaled_product(Ctx& c, double coef, const double* g, const double* w, u64 n, double* out);
/* out[k] = a[k] + (mask[k] ? b[k] : 0) */
void launch_masked_add(Ctx& c, const double* a, const double* b, const unsigned char* mask, u64 n, double* out);
/* elementwise helpers */
void launch_fill(Ctx& c, double* p, u64 n, double v);
void launch_rowdot(Ctx& c, const double* A, const double* B, u64 N, u64 K, u64 ld, double add, double* out);
/* outge[:,h] (N) dotted with w (N) -> out[h], deterministic two-stage */
void launch_dot_partials(Ctx& c, const double* a, const double* b, u64 n, double* partial, int* nblocks);

} // namespace obd

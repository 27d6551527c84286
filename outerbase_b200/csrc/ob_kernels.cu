/*
 * ob_kernels.cu -- hand-written sm_100a kernels of the outerbase hot path.
 *
 *   phi_a_kernel   Phi a  (+ fused loglik_gauss epilogues)   replaces prodmm_/domult_   src/linalg.cpp:57-131
 *   phi_t_kernel   Phi^T r                                    replaces tprodmm_/dotmultsub_ src/linalg.cpp:286-355
 *   (the same two kernels, fed augmented programs / gradient columns, give
 *    prodmmge_/tprodmmge_ src/linalg.cpp:139-277,364-471 and the squared operators
 *    of src/modandbase.cpp:784-879)
 *   *_simple       brute-force forms in the reference's own operation order
 *                  (fallback for programs the trie interpreter does not take, getm_ :685-715)
 *   basis_build    cov(x,knots) . rotmat, normalise          replaces outermod::buildob + outerbase::build
 *                                                             src/modandbase.cpp:285-327,547-626, covfuncs.cpp:113-347
 *
 * Layout in HBM: every N-row matrix is column-major with a leading dimension padded to
 * a multiple of 128 rows (pad rows are zero), so a (rows x column) tile segment is one
 * contiguous, 16-byte aligned run that a single cp.async.bulk (TMA, SASS UBLKCP) moves
 * into shared memory.  A CTA owns row tiles of 32*R rows; the tile's used basis columns
 * (Lcols ~ 75-100 of the M = 400-800 stored) are staged once, double buffered, and all
 * warps of the CTA interpret their share of the terms trie on it (ob_terms.hpp).
 */
#include <dlfcn.h>

#include "ob_device.cuh"

namespace obd {

using namespace obt;

/* ------------------------------------------------------------------ PTX helpers */
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE_%=;\n"
      "bra WAIT_%=;\n"
      "DONE_%=:\n"
      "}\n" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
/* 1-D bulk async copy global -> shared, completion on an mbarrier (TMA engine, SASS UBLKCP) */
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

/* ------------------------------------------------------------------ kernel parameters */
struct PhiKParams {
  const double* const* load_src;
  const int* col_op;
  int ncol, nload, has_ops;
  const uint32_t* prog;
  const uint32_t* prog_off;
  const uint32_t* slot_base;
  const uint32_t* slot_real;
  const int32_t* slot_term;
  int nslots, nwords, prog_in_smem;
  const double* scale;
  int sq;
  unsigned long long N;
  int ntiles, nbuf;
  unsigned off_tile, tile_doubles, off_vec, off_prog, off_part;
  int lt, ncs; /* TMEM kernels: columns [0,lt) in tensor memory, ncs = ncol - lt in shared memory */
  /* phi_a */
  const double* a;
  double* out;
  double* w;
  const double* y;
  double sd;
  double* ssq_partial;
  int mode;
  /* phi_t */
  const double* win;
  double* partial;
};

/* factor column -> registers.  tl = shared-space byte address of (tile base + this lane's first
 * row); a column is 32*R*8 bytes.  Explicit ld.shared.v2.f64: one LDS.128 per row pair. */
template <int R>
__device__ __forceinline__ void load_factor(double (&f)[R], uint32_t tl, uint32_t w) {
  const uint32_t addr = tl + ((w & 0xFFFFu) * (uint32_t)(32 * R * sizeof(double)));
  asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(f[0]), "=d"(f[1]) : "r"(addr));
  if constexpr (R == 4) asm volatile("ld.shared.v2.f64 {%0, %1}, [%2+512];" : "=d"(f[2]), "=d"(f[3]) : "r"(addr));
}
template <int R>
__device__ __forceinline__ int tile_row(int lane, int r) { return (r >> 1) * 64 + 2 * lane + (r & 1); }

/* The register stack (SD slots of R doubles) is indexed by a warp-uniform depth.  Every
 * access is a switch whose cases name fixed registers AND contain the consuming operation,
 * so nothing is selected speculatively on the hot (leaf) path. */
#define OB_CASES4(X) X(0) X(1) X(2) X(3)
#define OB_CASES_HI(X) X(4) X(5) X(6) X(7)

/* stage one row tile: nload columns of 32*R rows each, one bulk copy per column.  Called by
 * the producer warp only; UBLKCP takes uniform operands, so the copies are issued one by
 * one whatever the lane mapping -- lane 0 does them all. */
template <int R>
__device__ __forceinline__ void issue_tile(const PhiKParams& p, double* T, uint64_t* bar, unsigned long long row0, int lane) {
  constexpr uint32_t colbytes = 32 * R * sizeof(double);
  if (lane == 0) {
    fence_proxy_async();
    mbar_expect_tx(bar, colbytes * (uint32_t)p.nload);
#pragma unroll 1
    for (int c = 0; c < p.nload; ++c) bulk_g2s(T + (size_t)c * (32 * R), p.load_src[c] + row0, colbytes, bar);
  }
  __syncwarp();
}

template <int R>
__device__ __forceinline__ void transform_tile(const PhiKParams& p, double* T, int nthreads) {
  constexpr int TR = 32 * R;
  for (int idx = threadIdx.x; idx < p.ncol * TR; idx += nthreads) {
    const int c = idx / TR, r = idx - c * TR;
    const int op = p.col_op[c];
    const double x = T[idx];
    if ((op & 255) == COL_SQUARE) T[idx] = x * x;
    else if ((op & 255) == COL_TWO_G_B) T[idx] = 2.0 * (x * T[(op >> 8) * TR + r]);
  }
}

constexpr int kComputeWarps = 16;                      /* = term groups of a program (ob_terms.hpp G) */
constexpr int kPhiThreads = 32 * (kComputeWarps + 1);  /* + one producer warp issuing the bulk copies */

/* ------------------------------------------------------------------ Phi a
 * One compute warp = one term group; lanes x R = the tile's rows.  Backward (Horner) stream. */
template <int R, int SD, bool PS>
__global__ void __launch_bounds__(kPhiThreads, 1) phi_a_kernel(const PhiKParams p) {
  constexpr int TR = 32 * R;
  extern __shared__ __align__(128) unsigned char smem[];
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem);
  double* tiles = reinterpret_cast<double*>(smem + p.off_tile);
  double* a_sm = reinterpret_cast<double*>(smem + p.off_vec);
  uint32_t* prog_sm = reinterpret_cast<uint32_t*>(smem + p.off_prog);
  double* part = reinterpret_cast<double*>(smem + p.off_part);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const bool producer = warp == kComputeWarps;

  if (tid == 0) { mbar_init(&bars[0], 1); mbar_init(&bars[1], 1); fence_barrier_init(); }
  for (int i = tid; i < p.nslots; i += kPhiThreads) { const int t = p.slot_term[i]; a_sm[i] = t >= 0 ? p.a[t] : 0.0; }
  if (PS) for (int i = tid; i < p.nwords; i += kPhiThreads) prog_sm[i] = p.prog[i];
  __syncthreads();
  const uint32_t* pw0;
  if (PS) pw0 = prog_sm + (producer ? 0 : p.prog_off[warp]);
  else pw0 = p.prog + (producer ? 0 : p.prog_off[warp]);
  const int slot_hi = producer ? 0 : (int)p.slot_base[warp] + (int)p.slot_real[warp] - 1;

  int tile = blockIdx.x;
  if (producer && tile < p.ntiles) issue_tile<R>(p, tiles, &bars[0], (unsigned long long)tile * TR, lane);
  uint32_t phases = 0;
  double ssq_local = 0.0;
  for (int it = 0; tile < p.ntiles; tile += gridDim.x, ++it) {
    const int buf = (p.nbuf == 2) ? (it & 1) : 0;
    const int nxt = tile + gridDim.x;
    if (p.nbuf == 2 && producer && nxt < p.ntiles)
      issue_tile<R>(p, tiles + (size_t)(buf ^ 1) * p.tile_doubles, &bars[buf ^ 1], (unsigned long long)nxt * TR, lane);
    double* T = tiles + (size_t)buf * p.tile_doubles;
    if (!producer || p.has_ops) mbar_wait(&bars[buf], (phases >> buf) & 1u);
    phases ^= (1u << buf);
    if (p.has_ops) { transform_tile<R>(p, T, kPhiThreads); __syncthreads(); }

    if (!producer) {
      double cur[R], stk[SD][R];
#pragma unroll
      for (int r = 0; r < R; ++r) cur[r] = 0.0;
      const uint32_t tl = smem_u32(T) + 16u * (uint32_t)lane;
      const uint4* pq = reinterpret_cast<const uint4*>(pw0); /* streams are 16-byte aligned (ob_terms.hpp) */
      uint4 wq = pq[0];
      int slot = slot_hi;
/* one word of the backward stream; `goto a_done` on END */
#define OB_A_STEP(W)                                                                                     \
      {                                                                                                  \
        const uint32_t w = (W);                                                                          \
        if ((int32_t)w < 0) { /* B_LEAF: cur += B[col] * a[slot] */                                      \
          double f[R];                                                                                   \
          const double av = a_sm[slot--];                                                                \
          load_factor<R>(f, tl, w);                                                                      \
          _Pragma("unroll") for (int r = 0; r < R; ++r) cur[r] = fma(f[r], av, cur[r]);                  \
        } else {                                                                                         \
          const uint32_t op = w >> 28;                                                                   \
          if (op == B_END) goto a_done;                                                                  \
          const uint32_t e = (w >> 24) & 15u;                                                            \
          if (op == B_CLOSE_FRESH) {                                                                     \
            double f[R];                                                                                 \
            const double av = (w & (FLAG_HAS_A << 20)) ? a_sm[slot--] : 0.0;                             \
            load_factor<R>(f, tl, w);                                                                    \
            _Pragma("unroll") for (int r = 0; r < R; ++r) cur[r] = f[r] * (av + cur[r]);                 \
          } else if (op == B_CLOSE_LOAD) {                                                               \
            double f[R];                                                                                 \
            const double av = (w & (FLAG_HAS_A << 20)) ? a_sm[slot--] : 0.0;                             \
            load_factor<R>(f, tl, w);                                                                    \
            if constexpr (SD > 4) { switch (e) { OB_CASES4(OB_XA_LOAD) OB_CASES_HI(OB_XA_LOAD) default: break; } } \
            else { switch (e) { OB_CASES4(OB_XA_LOAD) default: break; } }                                \
          } else if (op == B_SAVE) {                                                                     \
            if constexpr (SD > 4) { switch (e) { OB_CASES4(OB_XA_SAVE) OB_CASES_HI(OB_XA_SAVE) default: break; } } \
            else { switch (e) { OB_CASES4(OB_XA_SAVE) default: break; } }                                \
          } else { /* B_ROOT */                                                                          \
            const double av = a_sm[slot--];                                                              \
            _Pragma("unroll") for (int r = 0; r < R; ++r) cur[r] += av;                                  \
          }                                                                                              \
        }                                                                                                \
      }
#define OB_XA_LOAD(i) case i + 1: _Pragma("unroll") for (int r = 0; r < R; ++r) cur[r] = fma(f[r], av + cur[r], stk[i][r]); break;
#define OB_XA_SAVE(i) case i: _Pragma("unroll") for (int r = 0; r < R; ++r) { stk[i][r] = cur[r]; cur[r] = 0.0; } break;
#pragma unroll 1
      for (;;) {
        const uint4 nq = pq[1]; /* next four words: the fetch never sits on the critical path */
        ++pq;
        if ((int32_t)(wq.x & wq.y & wq.z & wq.w) < 0) { /* four leaves: loads first, then 4R FMAs */
          double f0[R], f1[R], f2[R], f3[R];
          const double a0 = a_sm[slot], a1 = a_sm[slot - 1], a2 = a_sm[slot - 2], a3 = a_sm[slot - 3];
          slot -= 4;
          load_factor<R>(f0, tl, wq.x);
          load_factor<R>(f1, tl, wq.y);
          load_factor<R>(f2, tl, wq.z);
          load_factor<R>(f3, tl, wq.w);
#pragma unroll
          for (int r = 0; r < R; ++r) cur[r] = fma(f0[r], a0, cur[r]);
#pragma unroll
          for (int r = 0; r < R; ++r) cur[r] = fma(f1[r], a1, cur[r]);
#pragma unroll
          for (int r = 0; r < R; ++r) cur[r] = fma(f2[r], a2, cur[r]);
#pragma unroll
          for (int r = 0; r < R; ++r) cur[r] = fma(f3[r], a3, cur[r]);
        } else {
          OB_A_STEP(wq.x)
          OB_A_STEP(wq.y)
          OB_A_STEP(wq.z)
          OB_A_STEP(wq.w)
        }
        wq = nq;
      }
    a_done:;
#undef OB_A_STEP
#undef OB_XA_LOAD
#undef OB_XA_SAVE
#pragma unroll
      for (int r = 0; r < R; ++r) part[warp * TR + tile_row<R>(lane, r)] = cur[r];
    }
    __syncthreads();
    if (tid < TR) {
      const unsigned long long row = (unsigned long long)tile * TR + tid;
      if (row < p.N) {
        double s = 0.0;
#pragma unroll
        for (int g = 0; g < kComputeWarps; ++g) s += part[g * TR + tid];
        double sc = p.scale[row];
        if (p.sq) sc = sc * sc;
        const double yv = s * sc;
        if (p.mode == PHI_PLAIN) p.out[row] = yv;
        else if (p.mode == PHI_UPDATE) { /* loglik_gauss::update, loglik_gauss.cpp:121-125 */
          p.out[row] = yv;
          const double rt = (yv - p.y[row]) / p.sd;
          ssq_local += rt * rt;
          p.w[row] = -1. * (rt / p.sd);
        } else { /* loglik_gauss::hessmult, loglik_gauss.cpp:139-141 */
          p.w[row] = (yv / p.sd) / p.sd;
        }
      }
    }
    __syncthreads();
    if (p.nbuf == 1 && producer && nxt < p.ntiles) issue_tile<R>(p, tiles, &bars[0], (unsigned long long)nxt * TR, lane);
  }
  if (p.mode == PHI_UPDATE) { /* deterministic per-CTA sum of squared standardised residuals */
    __syncthreads();
    if (tid < TR) part[tid] = ssq_local;
    __syncthreads();
    if (tid == 0) {
      double s = 0.0;
      for (int i = 0; i < TR; ++i) s += part[i];
      p.ssq_partial[blockIdx.x] = s;
    }
  }
}

/* ------------------------------------------------------------------ Phi^T r
 * Forward (top-down) stream; per-term row sums are reduced across the warp with an
 * incremental 8-term butterfly and accumulated into CTA-private shared-memory slots;
 * every slot belongs to exactly one warp. */
__device__ __forceinline__ double shfl_xor_d(double v, int m) { return __shfl_xor_sync(0xffffffffu, v, m); }

/* Incremental 8-way butterfly.  Row sums of consecutive emits are paired as they arrive: two
 * pending sums are merged with ONE 64-bit exchange (each half of the lanes keeps one of them),
 * so eight emits cost 4+2+1 merging exchanges plus two plain ones instead of 8 x 5.  The
 * pending registers form a binary counter on the warp-uniform emit count, which keeps the
 * interpreter a single compact loop (no unrolling, no register indexing).
 * After the 8th emit every lane holds the full 32-lane sum of emit
 *   bit4(lane) + 2*bit3(lane) + 4*bit2(lane)   of the batch. */
struct EmitState {
  double p1, p2, p3;
  uint32_t cnt;
};
__device__ __forceinline__ double merge_xor(double first, double second, bool upper, int m) {
  const double keep = upper ? second : first;
  const double send = upper ? first : second;
  return keep + shfl_xor_d(send, m);
}
/* cur = (from stack ? stk[d-1] : cur) * f ; optional save to stk[d] */
#define OB_FWD_DESC()                                                                                   \
  {                                                                                                     \
    double f[R];                                                                                        \
    load_factor<R>(f, tl, w);                                            \
    if (op == F_DESC_STK) {                                                                             \
      OB_SWITCH(d, OB_X_MULSTK)                                                                         \
    } else {                                                                                            \
      _Pragma("unroll") for (int r = 0; r < R; ++r) cur[r] *= f[r];                                     \
    }                                                                                                   \
    if (w & (FLAG_SAVE << 20)) { OB_SWITCH(d, OB_X_SAVE) }                                              \
  }
#define OB_X_MULSTK(i) case i + 1: _Pragma("unroll") for (int r = 0; r < R; ++r) cur[r] = stk[i][r] * f[r]; break;
#define OB_X_SAVE(i) case i: _Pragma("unroll") for (int r = 0; r < R; ++r) stk[i][r] = cur[r]; break;
#define OB_X_LOAD(i) case i: _Pragma("unroll") for (int r = 0; r < R; ++r) cur[r] = stk[i][r]; break;
#define OB_SWITCH(sel, X)                                                       \
  if constexpr (SD > 4) { switch (sel) { OB_CASES4(X) OB_CASES_HI(X) default: break; } } \
  else { switch (sel) { OB_CASES4(X) default: break; } }

template <int R, int SD, bool PS>
__global__ void __launch_bounds__(kPhiThreads, 1) phi_t_kernel(const PhiKParams p) {
  constexpr int TR = 32 * R;
  extern __shared__ __align__(128) unsigned char smem[];
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem);
  double* tiles = reinterpret_cast<double*>(smem + p.off_tile);
  double* acc_sm = reinterpret_cast<double*>(smem + p.off_vec);
  uint32_t* prog_sm = reinterpret_cast<uint32_t*>(smem + p.off_prog);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const bool producer = warp == kComputeWarps;

  if (tid == 0) { mbar_init(&bars[0], 1); mbar_init(&bars[1], 1); fence_barrier_init(); }
  for (int i = tid; i < p.nslots; i += kPhiThreads) acc_sm[i] = 0.0;
  if (PS) for (int i = tid; i < p.nwords; i += kPhiThreads) prog_sm[i] = p.prog[i];
  __syncthreads();
  const uint32_t* pw0;
  if (PS) pw0 = prog_sm + (producer ? 0 : p.prog_off[warp]);
  else pw0 = p.prog + (producer ? 0 : p.prog_off[warp]);
  const int slot_lo = producer ? 0 : (int)p.slot_base[warp];
  /* which of the 8 emits of a batch this lane owns after the butterfly, and whether it stores */
  const int my_emit = ((lane >> 4) & 1) + ((lane >> 3) & 1) * 2 + ((lane >> 2) & 1) * 4;
  const bool storer = (lane & 3) == 0;
  const bool up16 = lane & 16, up8 = lane & 8, up4 = lane & 4;

  int tile = blockIdx.x;
  if (producer && tile < p.ntiles) issue_tile<R>(p, tiles, &bars[0], (unsigned long long)tile * TR, lane);
  uint32_t phases = 0;
  for (int it = 0; tile < p.ntiles; tile += gridDim.x, ++it) {
    const int buf = (p.nbuf == 2) ? (it & 1) : 0;
    const int nxt = tile + gridDim.x;
    if (p.nbuf == 2 && producer && nxt < p.ntiles)
      issue_tile<R>(p, tiles + (size_t)(buf ^ 1) * p.tile_doubles, &bars[buf ^ 1], (unsigned long long)nxt * TR, lane);
    /* b = basescale % a (linalg.cpp:312), zero beyond N */
    double cur[R], stk[SD][R];
    if (!producer) {
#pragma unroll
      for (int r = 0; r < R; ++r) {
        const unsigned long long row = (unsigned long long)tile * TR + tile_row<R>(lane, r);
        double b = 0.0;
        if (row < p.N) { double sc = p.scale[row]; if (p.sq) sc = sc * sc; b = sc * p.win[row]; }
        stk[0][r] = b;
        cur[r] = b;
      }
    }
    double* T = tiles + (size_t)buf * p.tile_doubles;
    if (!producer || p.has_ops) mbar_wait(&bars[buf], (phases >> buf) & 1u);
    phases ^= (1u << buf);
    if (p.has_ops) { transform_tile<R>(p, T, kPhiThreads); __syncthreads(); }

    if (!producer) {
      const uint32_t tl = smem_u32(T) + 16u * (uint32_t)lane;
      const uint32_t* pw = pw0;
      uint32_t w = pw[0], w1 = pw[1];
      int slot = slot_lo;
      EmitState es;
      es.p1 = es.p2 = es.p3 = 0.0;
      es.cnt = 0;
#pragma unroll 1
      for (;;) {
        const uint32_t w2 = pw[2];
        ++pw;
        double acc;
        if ((int32_t)w < 0) { /* F_LEAF: sum_r cur[r] * B[col][r] */
          double f[R];
          load_factor<R>(f, tl, w);
          acc = cur[0] * f[0];
#pragma unroll
          for (int r = 1; r < R; ++r) acc = fma(cur[r], f[r], acc);
        } else {
          const uint32_t op = w >> 28, d = (w >> 24) & 15u;
          if (op == F_END) break;
          acc = 0.0; /* F_EMITZERO */
          if (op == F_DESC_CUR || op == F_DESC_STK) {
            OB_FWD_DESC()
            acc = cur[0];
#pragma unroll
            for (int r = 1; r < R; ++r) acc += cur[r];
          } else if (op == F_ROOT) {
            acc = stk[0][0];
#pragma unroll
            for (int r = 1; r < R; ++r) acc += stk[0][r];
          } else if (op == F_LOADCUR) {
            OB_SWITCH(d, OB_X_LOAD)
          }
        }
        if (w & (FLAG_EMIT << 20)) {
          const uint32_t c = es.cnt++;
          if (!(c & 1u)) es.p1 = acc;
          else {
            const double h = merge_xor(es.p1, acc, up16, 16);
            if (!(c & 2u)) es.p2 = h;
            else {
              const double q = merge_xor(es.p2, h, up8, 8);
              if (!(c & 4u)) es.p3 = q;
              else {
                double v = merge_xor(es.p3, q, up4, 4);
                v += shfl_xor_d(v, 2);
                v += shfl_xor_d(v, 1);
                if (storer) acc_sm[slot + my_emit] += v;
                slot += 8;
              }
            }
          }
        }
        w = w1; w1 = w2;
      }
    }
    __syncthreads();
    if (p.nbuf == 1 && producer && nxt < p.ntiles) issue_tile<R>(p, tiles, &bars[0], (unsigned long long)nxt * TR, lane);
  }
  __syncthreads();
  for (int i = tid; i < p.nslots; i += kPhiThreads) p.partial[(size_t)blockIdx.x * p.nslots + i] = acc_sm[i];
}


/* out[term(slot)] = sum over CTAs, fixed order */
__global__ void phi_t_reduce_kernel(const double* __restrict__ partial, int nblocks, int nslots,
                                    const int32_t* __restrict__ slot_term, double* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nslots) return;
  const int t = slot_term[i];
  if (t < 0) return;
  double s = 0.0;
  for (int b = 0; b < nblocks; ++b) s += partial[(size_t)b * nslots + i];
  out[t] = s;
}

/* ------------------------------------------------------------------ brute-force forms
 * Operation order of the reference (linalg.cpp:70-75): temp = a_k; temp *= B columns
 * in ascending dimension; out += temp; finally out *= basescale.  __dmul_rn/__dadd_rn
 * keep the compiler from contracting to FMA, so phi_a_simple is BIT-EXACT against the
 * reference's row-chunk branch. */
__device__ __forceinline__ double col_value(const double* const* load_src, const int* col_op, uint32_t c, unsigned long long n) {
  const double x = load_src[c][n];
  const int op = col_op[c];
  if ((op & 255) == COL_SQUARE) return __dmul_rn(x, x);
  if ((op & 255) == COL_TWO_G_B) return __dmul_rn(2.0, __dmul_rn(x, load_src[op >> 8][n]));
  return x;
}

__global__ void phi_a_simple_kernel(const double* const* load_src, const int* col_op, const uint32_t* csr_ptr,
                                    const uint32_t* csr_col, int K, const double* a, const double* scale, int sq,
                                    unsigned long long N, double* out) {
  const unsigned long long n = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N) return;
  double acc = 0.0;
  for (int k = 0; k < K; ++k) {
    double t = a[k];
    for (uint32_t j = csr_ptr[k]; j < csr_ptr[k + 1]; ++j) t = __dmul_rn(t, col_value(load_src, col_op, csr_col[j], n));
    acc = __dadd_rn(acc, t);
  }
  double sc = scale[n];
  if (sq) sc = __dmul_rn(sc, sc);
  out[n] = __dmul_rn(acc, sc);
}

/* partial[k * gridDim.x + blockIdx.x] = this CTA's share of (Phi^T w)_k: rows in grid-stride order per thread, then the
 * warp butterfly, then the warps in index order.  blockIdx.y strides over the terms (few rows: more CTAs).  No atomics,
 * so the result is the same bits on every run; the CTA partials are added in index order by colsum_partials_kernel. */
constexpr int kSimpleTThreads = 512;
__global__ void __launch_bounds__(kSimpleTThreads) phi_t_simple_kernel(const double* const* load_src, const int* col_op,
                                                                       const uint32_t* csr_ptr, const uint32_t* csr_col, int K,
                                                                       const double* w, const double* scale, int sq,
                                                                       unsigned long long N, double* __restrict__ partial) {
  constexpr int kWarps = kSimpleTThreads / 32;
  __shared__ double warp_sum[2][kWarps]; /* double-buffered: one barrier per term */
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const unsigned long long stride = (unsigned long long)gridDim.x * kSimpleTThreads;
  for (int k = blockIdx.y, it = 0; k < K; k += gridDim.y, it ^= 1) {
    double s = 0.0;
    for (unsigned long long n = (unsigned long long)blockIdx.x * kSimpleTThreads + threadIdx.x; n < N; n += stride) {
      double sc = scale[n];
      if (sq) sc = __dmul_rn(sc, sc);
      double t = __dmul_rn(sc, w[n]);
      for (uint32_t j = csr_ptr[k]; j < csr_ptr[k + 1]; ++j) t = __dmul_rn(t, col_value(load_src, col_op, csr_col[j], n));
      s += t;
    }
#pragma unroll
    for (int m = 16; m > 0; m >>= 1) s += shfl_xor_d(s, m);
    if (lane == 0) warp_sum[it][warp] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
      double v = 0.0;
      for (int i = 0; i < kWarps; ++i) v += warp_sum[it][i];
      partial[(size_t)k * gridDim.x + blockIdx.x] = v;
    }
  }
}

/* out[c] = sum of column c's nb partials (partial[c * nb + i]), in index order */
__global__ void colsum_partials_kernel(const double* __restrict__ partial, int nb, double* __restrict__ out) {
  if (threadIdx.x != 0) return;
  double s = 0.0;
  for (int i = 0; i < nb; ++i) s += partial[(size_t)blockIdx.x * nb + i];
  out[blockIdx.x] = s;
}

/* Residuals of C columns after a plain product, the PHI_UPDATE / PHI_HESS epilogue of phi_a_kernel column by column
 * (same expressions, so a column's w equals the trie kernel's bit for bit given the same yhat and sd).  grid (nb, C);
 * rows N .. ld-1 of w are written as zero (phi_tm_spec and phi_t_spec read pad rows, they must be finite).  update:
 * partial[c * nb + b] = this CTA's sum of ((yhat - y) / sd)^2 over its rows of column c, fixed tree.  yhat may alias w.
 * sds, when set, holds one sd per column (per-column noise) and replaces the scalar sd.  rowsd, when set, holds one sd
 * per row shared by the columns (loglik_gda's obssd) and replaces both: the same expressions as LoglikGda::update /
 * hessmult with that row's sd. */
constexpr int kResidThreads = 256;
__global__ void __launch_bounds__(kResidThreads) resid_multi_kernel(const double* yhat, const double* __restrict__ y, double* w, u64 N,
                                                                   u64 ld, double sd0, const double* __restrict__ sds, int update,
                                                                   double* __restrict__ partial, const double* __restrict__ rowsd = nullptr) {
  __shared__ double sm[kResidThreads];
  const u64 col = blockIdx.y, base = col * ld;
  const double sdc = sds ? sds[col] : sd0;
  double s = 0.0;
  for (u64 i = (u64)blockIdx.x * kResidThreads + threadIdx.x; i < ld; i += (u64)gridDim.x * kResidThreads) {
    double wv = 0.0;
    if (i < N) {
      const double sd = rowsd ? rowsd[i] : sdc;
      const double yv = yhat[base + i];
      if (update) {
        const double rt = (yv - y[base + i]) / sd;
        s += rt * rt;
        wv = -1. * (rt / sd);
      } else wv = (yv / sd) / sd;
    }
    w[base + i] = wv;
  }
  if (!update) return;
  sm[threadIdx.x] = s;
  __syncthreads();
  for (int h = kResidThreads / 2; h > 0; h >>= 1) {
    if (threadIdx.x < h) sm[threadIdx.x] += sm[threadIdx.x + h];
    __syncthreads();
  }
  if (threadIdx.x == 0) partial[col * gridDim.x + blockIdx.x] = sm[0];
}

/* loglik_gda's per-row noise sd (LoglikGda::buildstd): v = v0, plus v1 (1 - phi2varc[i]) when phi2varc is set (dodiag;
 * phi2varc = Phi^2 varc, so that 1 - phi2varc is OuterBase::residvar), obssd = sqrt(v); rows N .. ld-1 are 1 */
__global__ void gda_obssd_kernel(const double* __restrict__ phi2varc, u64 N, u64 ld, double v0, double v1, double* __restrict__ obssd) {
  const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= ld) return;
  double v = 1.0;
  if (i < N) {
    v = v0;
    if (phi2varc) v += v1 * (1 - phi2varc[i]);
  }
  obssd[i] = sqrt(v);
}

__global__ void getmat_kernel(const double* const* load_src, const int* col_op, const uint32_t* csr_ptr,
                              const uint32_t* csr_col, int K, const double* scale, int sq, unsigned long long N,
                              double* out, unsigned long long ldo) {
  const unsigned long long n = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N) return;
  double sc = scale[n];
  if (sq) sc = __dmul_rn(sc, sc);
  for (int k = blockIdx.y; k < K; k += gridDim.y) {
    double t = 1.0;
    for (uint32_t j = csr_ptr[k]; j < csr_ptr[k + 1]; ++j) t = __dmul_rn(t, col_value(load_src, col_op, csr_col[j], n));
    out[n + (unsigned long long)k * ldo] = __dmul_rn(t, sc);
  }
}

__global__ void sum_partials_kernel(const double* partial, int n, double* out) {
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    double s = 0.0;
    for (int i = 0; i < n; ++i) s += partial[i];
    out[0] = s;
  }
}

__global__ void fill_kernel(double* p, unsigned long long n, double v) {
  const unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = v;
}

/* per-block partial dot products, fixed tree */
__global__ void dot_partials_kernel(const double* a, const double* b, unsigned long long n, double* partial) {
  __shared__ double sm[256];
  double s = 0.0;
  for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (unsigned long long)gridDim.x * blockDim.x)
    s = fma(a[i], b[i], s);
  sm[threadIdx.x] = s;
  __syncthreads();
  for (int st = 128; st > 0; st >>= 1) { if ((int)threadIdx.x < st) sm[threadIdx.x] += sm[threadIdx.x + st]; __syncthreads(); }
  if (threadIdx.x == 0) partial[blockIdx.x] = sm[0];
}

/* ------------------------------------------------------------------ covariance + basis build */
struct CovPt { double t, s; }; /* mat25/pow: t = transformed x, s = log(x)*t ; ang: t = sin/rho_s, s = cos/rho_c */

__device__ __forceinline__ CovPt cov_transform_dev(int kind, double h0, double h1, double x) {
  CovPt p;
  if (kind == obh::COV_MAT25) { p.t = x / exp(2. * h0); p.s = 0.0; }
  else if (kind == obh::COV_MAT25POW) {
    const double powv = exp(0.25 * h1);
    p.t = pow(x, powv) / exp(2. * h0 + 0.25 * h1);
    p.s = log(x) * p.t;
  } else { p.t = sin(x) / exp(2. * h0); p.s = cos(x) / exp(2. * h1); }
  return p;
}
/* covf_*::cov and cov_gradhyp for one pair, covfuncs.cpp:113-150,197-243,285-347 */
template <bool GRAD>
__device__ __forceinline__ void cov_pair_dev(int kind, double h1, const CovPt& a, const CovPt& b, double& v, double& g0, double& g1) {
  if (kind == obh::COV_MAT25ANG) {
    const double hs = a.t - b.t, hc = a.s - b.s;
    const double t = sqrt(hs * hs + hc * hc);
    const double e = exp(-t);
    v = (1 + t + (t * t) / 3) * e;
    if (GRAD) { const double wv = e * (t + 1); g0 = ((2. / 3) * (hs * hs)) * wv; g1 = ((2. / 3) * (hc * hc)) * wv; }
    return;
  }
  double h = a.t - b.t;
  const double ah = fabs(h), e = exp(-ah);
  v = (1 + ah + (ah * ah) / 3) * e;
  if (!GRAD) return;
  const double h2 = (h * (1 + ah)) * e;
  if (kind == obh::COV_MAT25) { g0 = (2. / 3) * (h * h2); g1 = 0.0; return; }
  const double powv = exp(0.25 * h1);
  double s1 = a.s - b.s;
  s1 *= (-(0.25 * powv / 3)) * h2;
  h *= h2;
  g1 = s1 + (0.25 / 3) * h;
  g0 = (2. / 3) * h;
}

__global__ void cov_kernel(int kind, double h0, double h1, const double* x1, unsigned long long n1, const double* x2,
                           unsigned long long n2, double* out, double* outg) {
  const unsigned long long idx = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= n1 * n2) return;
  const unsigned long long i = idx % n1, j = idx / n1;
  const CovPt a = cov_transform_dev(kind, h0, h1, x1[i]), b = cov_transform_dev(kind, h0, h1, x2[j]);
  double v, g0 = 0, g1 = 0;
  if (outg) cov_pair_dev<true>(kind, h1, a, b, v, g0, g1);
  else cov_pair_dev<false>(kind, h1, a, b, v, g0, g1);
  out[idx] = v;
  if (outg) {
    outg[idx] = g0;
    if (kind != obh::COV_MAT25) outg[idx + n1 * n2] = g1;
  }
}

struct BuildKParams {
  int kind, m, nh, mp; /* mp: padded row length of the transposed rotation blocks in smem */
  int mo;              /* columns built and stored (levels 0 .. mo-1 of the m): the contraction still runs over all m knots */
  double h0, h1;
  const double* knots;  /* this dim's m knots */
  const double* x;      /* this dim's column of x */
  const double* rot;    /* m x m block, column-major, ld rot_ld */
  const double* rotg0;
  const double* rotg1;
  unsigned long long rot_ld;
  double* bm;           /* basemat + col_off*ld */
  double* bg0;
  double* bg1;
  double* scalecol;     /* basescalemat column */
  unsigned long long N, ld;
  int dograd;
};

/* ROWS rows per CTA, 256 threads = ROWS x (256/ROWS) column groups, 4 columns per group step.
 * smem: rotT[(1+nh)][m][mp] (row p, column j contiguous), C[(1+nh)][m][ROWS], knot/row transforms. */
template <int ROWS>
__global__ void __launch_bounds__(256) basis_build_kernel(const BuildKParams p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  double* sm = reinterpret_cast<double*>(smem_raw);
  const int m = p.m, mp = p.mp, nh = p.dograd ? p.nh : 0;
  double* rotT = sm;                                   /* (1+nh) * m * mp */
  double* Cs = rotT + (size_t)(1 + nh) * m * mp;       /* (1+nh) * m * ROWS */
  double* kt = Cs + (size_t)(1 + nh) * m * ROWS;       /* 2*m knot transforms */
  double* xt = kt + 2 * m;                             /* 2*ROWS row transforms */
  const int tid = threadIdx.x;
  const unsigned long long row0 = (unsigned long long)blockIdx.x * ROWS;

  for (int idx = tid; idx < m * m; idx += 256) {
    const int pp = idx % m, j = idx / m; /* column-major source: element (pp, j) */
    rotT[(size_t)pp * mp + j] = p.rot[pp + (unsigned long long)j * p.rot_ld];
    if (nh > 0) rotT[(size_t)(m + pp) * mp + j] = p.rotg0[pp + (unsigned long long)j * p.rot_ld];
    if (nh > 1) rotT[(size_t)(2 * m + pp) * mp + j] = p.rotg1[pp + (unsigned long long)j * p.rot_ld];
  }
  for (int idx = tid; idx < m; idx += 256) {
    const CovPt c = cov_transform_dev(p.kind, p.h0, p.h1, p.knots[idx]);
    kt[idx] = c.t; kt[m + idx] = c.s;
  }
  for (int idx = tid; idx < ROWS; idx += 256) {
    const unsigned long long row = row0 + idx;
    CovPt c{0.0, 0.0};
    if (row < p.N) c = cov_transform_dev(p.kind, p.h0, p.h1, p.x[row]);
    xt[idx] = c.t; xt[ROWS + idx] = c.s;
  }
  __syncthreads();
  for (int idx = tid; idx < m * ROWS; idx += 256) {
    const int r = idx % ROWS, pp = idx / ROWS;
    const CovPt a{xt[r], xt[ROWS + r]}, b{kt[pp], kt[m + pp]};
    double v, g0 = 0, g1 = 0;
    if (nh > 0) cov_pair_dev<true>(p.kind, p.h1, a, b, v, g0, g1);
    else cov_pair_dev<false>(p.kind, p.h1, a, b, v, g0, g1);
    Cs[(size_t)pp * ROWS + r] = v;
    if (nh > 0) Cs[(size_t)(m + pp) * ROWS + r] = g0;
    if (nh > 1) Cs[(size_t)(2 * m + pp) * ROWS + r] = g1;
  }
  __syncthreads();

  constexpr int NCG = 256 / ROWS;
  const int r = tid % ROWS, cg = tid / ROWS;
  const unsigned long long row = row0 + r;
  const bool live = row < p.N;
  /* column 0 of the projected basis: the per-row scale P_l[:,0] (modandbase.cpp:297,572) */
  double p0 = 0.0;
  for (int pp = 0; pp < m; ++pp) p0 = fma(Cs[(size_t)pp * ROWS + r], rotT[(size_t)pp * mp], p0);
  if (cg == 0 && row < p.ld) p.scalecol[row] = live ? p0 : 0.0;
  for (int j0 = cg * 4; j0 < p.mo; j0 += NCG * 4) {
    double acc[4] = {0, 0, 0, 0}, s1[2][4] = {{0, 0, 0, 0}, {0, 0, 0, 0}}, s2[2][4] = {{0, 0, 0, 0}, {0, 0, 0, 0}};
    for (int pp = 0; pp < m; ++pp) {
      const double c = Cs[(size_t)pp * ROWS + r];
      const double* rr = rotT + (size_t)pp * mp + j0;
#pragma unroll
      for (int q = 0; q < 4; ++q) acc[q] = fma(c, rr[q], acc[q]);
      if (nh > 0) {
        const double cg0 = Cs[(size_t)(m + pp) * ROWS + r];
        const double* rg = rotT + (size_t)(m + pp) * mp + j0;
#pragma unroll
        for (int q = 0; q < 4; ++q) { s1[0][q] = fma(cg0, rr[q], s1[0][q]); s2[0][q] = fma(c, rg[q], s2[0][q]); }
      }
      if (nh > 1) {
        const double cg1 = Cs[(size_t)(2 * m + pp) * ROWS + r];
        const double* rg = rotT + (size_t)(2 * m + pp) * mp + j0;
#pragma unroll
        for (int q = 0; q < 4; ++q) { s1[1][q] = fma(cg1, rr[q], s1[1][q]); s2[1][q] = fma(c, rg[q], s2[1][q]); }
      }
    }
    if (row < p.ld) {
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int j = j0 + q;
        if (j >= p.mo) break;
        double v = 0.0;
        if (live) v = (j == 0) ? 1.0 : acc[q] / p0;
        p.bm[row + (unsigned long long)j * p.ld] = v;
        if (nh > 0) p.bg0[row + (unsigned long long)j * p.ld] = live ? (s1[0][q] + s2[0][q]) / p0 : 0.0;
        if (nh > 1) p.bg1[row + (unsigned long long)j * p.ld] = live ? (s1[1][q] + s2[1][q]) / p0 : 0.0;
      }
    }
  }
}

/* Tensor-core variant of the basis build: the m x m (+ gradient) contractions of buildob (modandbase.cpp:285-327) as
 * FP64 DMMAs (mma.sync.m8n8k4.f64).  64 rows per CTA, 8 warps = 8 row tiles; warp w contracts rows 8w..8w+7 against
 * all NT column tiles of the rotation blocks: per k-step 1 (+nh) A fragments from the covariance tile in shared
 * memory and (1+nh) NT B fragments from the rotation blocks, 1 + 2 nh DMMAs per column tile, with Rt = covg.rot +
 * cov.rotg accumulated in ONE tile.  Strides 72 / 44|76 doubles keep every fragment load at the minimum two
 * shared-memory wavefronts.  The existing FMA kernel stays for m > 72. */
__device__ __forceinline__ void dmma_f64(double& c0, double& c1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}
template <int NT>
__global__ void __launch_bounds__(256) basis_build_mma_kernel(const BuildKParams p) {
  constexpr int ROWS = 64, CS = ROWS + 8, RS = NT * 8 + 4;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  double* sm = reinterpret_cast<double*>(smem_raw);
  const int m = p.m, nh = p.dograd ? p.nh : 0, mk = (m + 3) & ~3;
  double* rotT = sm;                                    /* (1+nh) * mk * RS : element (p, j), zero padded */
  double* Cs = rotT + (size_t)(1 + nh) * mk * RS;       /* (1+nh) * mk * CS : element (p, row), zero padded */
  double* kt = Cs + (size_t)(1 + nh) * mk * CS;         /* 2*m knot transforms */
  double* xt = kt + 2 * m;                              /* 2*ROWS row transforms */
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int g = lane >> 2, k4 = lane & 3;
  const int mo = p.mo < NT * 8 ? p.mo : NT * 8;
  const int ntiles = (mo + 7) / 8;

  /* once per CTA: rotation blocks, knot transforms, zero padding (persistent CTAs walk the row tiles) */
  for (int idx = tid; idx < (1 + nh) * mk * RS; idx += 256) rotT[idx] = 0.0;
  for (int idx = tid; idx < (1 + nh) * mk * CS; idx += 256) Cs[idx] = 0.0;
  __syncthreads();
  for (int idx = tid; idx < m * mo; idx += 256) {
    const int pp = idx % m, j = idx / m; /* column-major source: element (pp, j), the first mo columns */
    rotT[(size_t)pp * RS + j] = p.rot[pp + (unsigned long long)j * p.rot_ld];
    if (nh > 0) rotT[(size_t)(mk + pp) * RS + j] = p.rotg0[pp + (unsigned long long)j * p.rot_ld];
    if (nh > 1) rotT[(size_t)(2 * mk + pp) * RS + j] = p.rotg1[pp + (unsigned long long)j * p.rot_ld];
  }
  for (int idx = tid; idx < m; idx += 256) {
    const CovPt c = cov_transform_dev(p.kind, p.h0, p.h1, p.knots[idx]);
    kt[idx] = c.t; kt[m + idx] = c.s;
  }
  const unsigned long long nrt = (p.ld + ROWS - 1) / ROWS;
  for (unsigned long long rt = blockIdx.x; rt < nrt; rt += gridDim.x) {
    const unsigned long long row0 = rt * ROWS;
    __syncthreads(); /* previous tile's fragments are consumed; knot transforms are visible */
    for (int idx = tid; idx < ROWS; idx += 256) {
      const unsigned long long row = row0 + idx;
      CovPt c{0.0, 0.0};
      if (row < p.N) c = cov_transform_dev(p.kind, p.h0, p.h1, p.x[row]);
      xt[idx] = c.t; xt[ROWS + idx] = c.s;
    }
    __syncthreads();
    for (int idx = tid; idx < m * ROWS; idx += 256) {
      const int r = idx % ROWS, pp = idx / ROWS;
      const CovPt a{xt[r], xt[ROWS + r]}, b{kt[pp], kt[m + pp]};
      double v, g0 = 0, g1 = 0;
      if (nh > 0) cov_pair_dev<true>(p.kind, p.h1, a, b, v, g0, g1);
      else cov_pair_dev<false>(p.kind, p.h1, a, b, v, g0, g1);
      Cs[(size_t)pp * CS + r] = v;
      if (nh > 0) Cs[(size_t)(mk + pp) * CS + r] = g0;
      if (nh > 1) Cs[(size_t)(2 * mk + pp) * CS + r] = g1;
    }
    __syncthreads();

    double acc[3][NT][2];
#pragma unroll
    for (int q = 0; q < 3; ++q)
#pragma unroll
      for (int jt = 0; jt < NT; ++jt) acc[q][jt][0] = acc[q][jt][1] = 0.0;
    for (int kk = 0; kk < mk / 4; ++kk) {
      const int pp = kk * 4 + k4;
      const double a0 = Cs[(size_t)pp * CS + warp * 8 + g];
      const double a1 = nh > 0 ? Cs[(size_t)(mk + pp) * CS + warp * 8 + g] : 0.0;
      const double a2 = nh > 1 ? Cs[(size_t)(2 * mk + pp) * CS + warp * 8 + g] : 0.0;
#pragma unroll
      for (int jt = 0; jt < NT; ++jt) {
        if (jt < ntiles) {
          const double b0 = rotT[(size_t)pp * RS + jt * 8 + g];
          dmma_f64(acc[0][jt][0], acc[0][jt][1], a0, b0);
          if (nh > 0) {
            const double b1 = rotT[(size_t)(mk + pp) * RS + jt * 8 + g];
            dmma_f64(acc[1][jt][0], acc[1][jt][1], a1, b0);
            dmma_f64(acc[1][jt][0], acc[1][jt][1], a0, b1);
          }
          if (nh > 1) {
            const double b2 = rotT[(size_t)(2 * mk + pp) * RS + jt * 8 + g];
            dmma_f64(acc[2][jt][0], acc[2][jt][1], a2, b0);
            dmma_f64(acc[2][jt][0], acc[2][jt][1], a0, b2);
          }
        }
      }
    }
    /* column 0 of the projected basis = the per-row scale P_l[:,0] (modandbase.cpp:297,572): C fragment element
     * (g, 0) lives in the first lane of every 4-lane group */
    const double p0 = __shfl_sync(0xffffffffu, acc[0][0][0], lane & ~3);
    const unsigned long long row = row0 + warp * 8 + g;
    const bool live = row < p.N;
    if (row < p.ld) {
      if (k4 == 0) p.scalecol[row] = live ? p0 : 0.0;
#pragma unroll
      for (int jt = 0; jt < NT; ++jt)
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          const int j = jt * 8 + 2 * k4 + e;
          if (j < mo) {
            double v = 0.0;
            if (live) v = (j == 0) ? 1.0 : acc[0][jt][e] / p0;
            p.bm[row + (unsigned long long)j * p.ld] = v;
            if (nh > 0) p.bg0[row + (unsigned long long)j * p.ld] = live ? acc[1][jt][e] / p0 : 0.0;
            if (nh > 1) p.bg1[row + (unsigned long long)j * p.ld] = live ? acc[2][jt][e] / p0 : 0.0;
          }
        }
    }
  }
}

/* basescale = prod_l P_l[:,0], multiplied in dimension order (modandbase.cpp:573) */
__global__ void basescale_kernel(const double* scalemat, unsigned long long ld, int d, unsigned long long N, double* scale) {
  const unsigned long long n = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= ld) return;
  double s = 1.0;
  for (int l = 0; l < d; ++l) s = __dmul_rn(s, scalemat[n + (unsigned long long)l * ld]);
  scale[n] = n < N ? s : 0.0;
}

__global__ void getbase_kernel(const double* basemat, const double* scalecol, unsigned long long N, unsigned long long ld,
                               unsigned long long col0, unsigned long long m, double* out) {
  const unsigned long long idx = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= N * m) return;
  const unsigned long long n = idx % N, j = idx / N;
  out[idx] = basemat[n + (col0 + j) * ld] * scalecol[n];
}

/* FP64 FMA micro-benchmark: the roofline denominator for the Phi kernels, measured on the
 * box the bench runs on (MEASURED_PEAKS.json has no FP64 entry).  16 independent DFMA chains
 * per thread, 8 warps x 4 CTAs per SM. */
__global__ void __launch_bounds__(256) fp64_peak_kernel(double* out, int iters, double seed) {
  double a[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) a[i] = seed + i + threadIdx.x * 1e-3;
  const double m = 1.0 - 1e-9, c = 1e-9;
  for (int it = 0; it < iters; ++it) {
#pragma unroll
    for (int i = 0; i < 16; ++i) a[i] = fma(a[i], m, c);
  }
  double s = 0;
#pragma unroll
  for (int i = 0; i < 16; ++i) s += a[i];
  if (s == 123.456) out[blockIdx.x] = s; /* never true: keeps the chains alive */
}

double measure_fp64_peak(Ctx& c) {
  DevBuf<double> sink;
  sink.ensure(4096);
  const int grid = c.sms * 8, iters = 20000;
  cudaEvent_t e0, e1;
  OB_CUDA(cudaEventCreate(&e0)); OB_CUDA(cudaEventCreate(&e1));
  fp64_peak_kernel<<<grid, 256, 0, c.stream>>>(sink.p, 2000, 1.0); /* warm-up */
  double best = 0;
  for (int rep = 0; rep < 3; ++rep) {
    OB_CUDA(cudaEventRecord(e0, c.stream));
    fp64_peak_kernel<<<grid, 256, 0, c.stream>>>(sink.p, iters, 1.0 + rep);
    OB_CUDA(cudaEventRecord(e1, c.stream));
    OB_CUDA(cudaEventSynchronize(e1));
    float ms = 0;
    OB_CUDA(cudaEventElapsedTime(&ms, e0, e1));
    const double flop = 2.0 * 16.0 * iters * 256.0 * grid;
    best = std::max(best, flop / (ms * 1e-3) / 1e12);
  }
  c.launches += 4;
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  return best;
}

/* ------------------------------------------------------------------ context */
NcclApi& NcclApi::get() {
  static NcclApi api;
  static bool tried = false;
  if (!tried) {
    tried = true;
    const char* names[] = {"libnccl.so.2", "libnccl.so"};
    for (const char* n : names) { api.handle = dlopen(n, RTLD_NOW | RTLD_GLOBAL); if (api.handle) break; }
    if (api.handle) {
      api.GetUniqueId = reinterpret_cast<decltype(api.GetUniqueId)>(dlsym(api.handle, "ncclGetUniqueId"));
      api.CommInitRank = reinterpret_cast<decltype(api.CommInitRank)>(dlsym(api.handle, "ncclCommInitRank"));
      api.AllReduce = reinterpret_cast<decltype(api.AllReduce)>(dlsym(api.handle, "ncclAllReduce"));
      api.AllGather = reinterpret_cast<decltype(api.AllGather)>(dlsym(api.handle, "ncclAllGather"));
      api.CommDestroy = reinterpret_cast<decltype(api.CommDestroy)>(dlsym(api.handle, "ncclCommDestroy"));
      api.GetErrorString = reinterpret_cast<decltype(api.GetErrorString)>(dlsym(api.handle, "ncclGetErrorString"));
    }
  }
  return api;
}

Ctx::Ctx(int dev) : device(dev) {
  int count = 0;
  const cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0)
    throw NoGpuError("no CUDA device visible: outerbase_b200 has no CPU fallback");
  if (dev < 0 || dev >= count) throw NoGpuError("CUDA device index out of range");
  OB_CUDA(cudaSetDevice(dev));
  cudaDeviceProp prop;
  OB_CUDA(cudaGetDeviceProperties(&prop, dev));
  if (prop.major < 10) throw NoGpuError(std::string("outerbase_b200 kernels are built for sm_100a only, found ") + prop.name);
  sms = prop.multiProcessorCount;
  smem_optin = prop.sharedMemPerBlockOptin;
  OB_CUDA(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
  OB_CUDA(cudaMallocHost(&pinned, 4096 * sizeof(double)));
  if (const char* e = getenv("OB_DSWEEP")) dsweep = std::string(e) != "0";
  if (const char* e = getenv("OB_DEVICE_CG")) device_cg = std::string(e) != "0";
  if (const char* e = getenv("OB_OVERLAP")) overlap = std::string(e) != "0";
  if (const char* e = getenv("OB_TMAP")) tmap = std::string(e) != "0";
  if (const char* e = getenv("OB_SPEC")) { /* 0 | 1 | auto */
    const std::string v(e);
    spec_mode = v == "0" ? 0 : (v == "1" ? 1 : 2);
  }
}

Ctx::~Ctx() {
  p2p_release();
  if (comm && NcclApi::get().CommDestroy) NcclApi::get().CommDestroy(comm);
  if (sync_ctr) cudaFree(sync_ctr);
  if (rows_ready) cudaFree(rows_ready);
  if (rows_table) cudaFreeHost(rows_table);
  if (ev_main) cudaEventDestroy(ev_main);
  if (ev_copy) cudaEventDestroy(ev_copy);
  if (copy_stream) cudaStreamDestroy(copy_stream);
  if (pinned) cudaFreeHost(pinned);
  if (stream) cudaStreamDestroy(stream);
}

/* ---- one-shot allreduce over NVLink peer memory (SURVEY 8e: the reference's `omp critical: out += out_`,
 * linalg.cpp:334-335, across GPUs).  A K-vector is 16 KB: the exchange is pure latency, so instead of a ring every
 * rank stores its values directly into slot [parity][rank] of EVERY peer's buffer (NVSwitch gives each pair full
 * bandwidth) and adds the G slots it receives in rank order -- all ranks add the same numbers in the same order, so the
 * result is bit-identical everywhere, as the replicated CG algebra needs.
 * Synchronisation is per ELEMENT and carried by the data itself: a double travels as two 8-byte words
 * {low half, tag}, {high half, tag} (8-byte stores are single-copy atomic over NVLink), tag = the call's sequence
 * number; the receiver polls an element until both tags match.  No flags, no system-scope fences (a
 * `fence.sys` behind remote stores costs a round trip per CTA: a first version with flags measured 26 us against
 * NCCL's 13 us at 2 ranks), no CTA barriers.  Slots alternate by the parity of the sequence number: a rank can only be
 * one call ahead of a peer (call s+1 completes only with every rank's s+1 data, sent after that rank finished call s),
 * so nobody overwrites an element that is still being polled. */
struct P2PArgs {
  uint4* slots[Ctx::P2P::kMaxRanks];
  int G, rank;
  unsigned seq;
  unsigned long long timeout_ns;
};

__device__ __forceinline__ void p2p_push(const P2PArgs& a, size_t at, double v) {
  const unsigned long long u = (unsigned long long)__double_as_longlong(v);
  const unsigned lo = (unsigned)u, hi = (unsigned)(u >> 32);
#pragma unroll 1
  for (int r = 0; r < a.G; ++r) { /* first stores spread over the peers */
    uint4* q = a.slots[(a.rank + r) % a.G] + at;
    asm volatile("st.volatile.global.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(q), "r"(lo), "r"(a.seq), "r"(hi), "r"(a.seq) : "memory");
  }
}

__device__ __forceinline__ double p2p_poll(const P2PArgs& a, const uint4* q) {
  unsigned lo, f0, hi, f1;
  unsigned long long t0 = 0, spins = 0;
  for (;;) {
    asm volatile("ld.volatile.global.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(lo), "=r"(f0), "=r"(hi), "=r"(f1) : "l"(q) : "memory");
    if (f0 == a.seq && f1 == a.seq) break;
    if ((++spins & 1023) == 0) { /* a peer that died must not hang this GPU for ever */
      unsigned long long now;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
      if (t0 == 0) t0 = now;
      else if (now - t0 > a.timeout_ns) __trap();
    }
  }
  return __longlong_as_double((long long)(((unsigned long long)hi << 32) | lo));
}

/* FUSED: the front end is phi_t_reduce_kernel (per-CTA partial sums of the Phi^T kernels added in CTA order, slot ->
 * term scatter) and its results go straight to the peers: Phi^T r's cross-CTA and cross-GPU reductions are ONE launch.
 * Ranks may mix the two variants within one call (a rank without rows has nothing to reduce). */
template <bool FUSED>
__global__ void __launch_bounds__(Ctx::P2P::kThreads) p2p_allreduce_kernel(const P2PArgs a, double* __restrict__ buf, int n,
                                                                            const double* __restrict__ partial, int nblocks,
                                                                            int nslots, const int32_t* __restrict__ slot_term) {
  constexpr size_t cap = Ctx::P2P::kCap;
  const int gtid = blockIdx.x * blockDim.x + threadIdx.x;
  const size_t par = (size_t)(a.seq & 1) * a.G;
  const size_t my_slot = (par + a.rank) * cap;
  if (FUSED) {
    for (int i = gtid; i < nslots; i += gridDim.x * blockDim.x) {
      const int t = slot_term[i];
      if (t < 0) continue;
      double v = 0.0;
      for (int b = 0; b < nblocks; ++b) v += partial[(size_t)b * nslots + i];
      p2p_push(a, my_slot + t, v);
    }
  } else if (gtid < n) {
    p2p_push(a, my_slot + gtid, buf[gtid]);
  }
  if (gtid < n) {
    const uint4* mine = a.slots[a.rank] + par * cap + gtid;
    double s = p2p_poll(a, mine);
    for (int r = 1; r < a.G; ++r) s += p2p_poll(a, mine + (size_t)r * cap);
    buf[gtid] = s;
  }
}

void Ctx::p2p_release() {
  for (int r = 0; r < P2P::kMaxRanks; ++r)
    if (p2p.peer[r] && p2p.peer[r] != p2p.local) cudaIpcCloseMemHandle(p2p.peer[r]);
  if (p2p.local) cudaFree(p2p.local);
  const bool en = p2p.enabled;
  p2p = P2P();
  p2p.enabled = en;
}

void Ctx::p2p_init() {
  NcclApi& api = NcclApi::get();
  if (const char* e = getenv("OB_P2P")) if (std::string(e) == "0") return;
  if (nranks < 2 || nranks > P2P::kMaxRanks || !comm || !api.AllGather) return;
  if (const char* e = getenv("OB_P2P_TIMEOUT_S")) p2p.timeout_ns = (unsigned long long)(atof(e) * 1e9);
  const size_t bytes = 2 * (size_t)nranks * P2P::kCap * sizeof(uint4);
  OB_CUDA(cudaMalloc(&p2p.local, bytes));
  OB_CUDA(cudaMemsetAsync(p2p.local, 0, bytes, stream));
  /* exchange the IPC handles (and whether this rank could export one) over the communicator */
  struct Rec { cudaIpcMemHandle_t h; int ok; int pad[15]; };
  static_assert(sizeof(Rec) == 128, "one record per rank");
  Rec mine{};
  mine.ok = cudaIpcGetMemHandle(&mine.h, p2p.local) == cudaSuccess ? 1 : 0;
  if (!mine.ok) cudaGetLastError();
  DevBuf<Rec> all;
  all.ensure((size_t)nranks);
  OB_CUDA(cudaMemcpyAsync(all.p + rank, &mine, sizeof(Rec), cudaMemcpyHostToDevice, stream));
  int rc = api.AllGather(all.p + rank, all.p, sizeof(Rec), /*ncclChar*/ 0, comm, stream);
  if (rc != 0) throw NcclError(std::string("ncclAllGather: ") + (api.GetErrorString ? api.GetErrorString(rc) : "error"));
  std::vector<Rec> recs((size_t)nranks);
  OB_CUDA(cudaMemcpyAsync(recs.data(), all.p, sizeof(Rec) * nranks, cudaMemcpyDeviceToHost, stream));
  sync();
  int ok = 1;
  for (int r = 0; r < nranks; ++r) ok &= recs[r].ok;
  for (int r = 0; r < nranks && ok; ++r) {
    if (r == rank) { p2p.peer[r] = p2p.local; continue; }
    if (cudaIpcOpenMemHandle(&p2p.peer[r], recs[r].h, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) {
      cudaGetLastError();
      p2p.peer[r] = nullptr;
      ok = 0;
    }
  }
  /* all ranks must take the same path: agree on the outcome (sum of ok flags == nranks) */
  double* agree = reinterpret_cast<double*>(all.p);
  const double okd = ok;
  OB_CUDA(cudaMemcpyAsync(agree, &okd, sizeof(double), cudaMemcpyHostToDevice, stream));
  rc = api.AllReduce(agree, agree, 1, /*ncclDouble*/ 8, /*ncclSum*/ 0, comm, stream);
  if (rc != 0) throw NcclError(std::string("ncclAllReduce: ") + (api.GetErrorString ? api.GetErrorString(rc) : "error"));
  double total = 0;
  OB_CUDA(cudaMemcpyAsync(&total, agree, sizeof(double), cudaMemcpyDeviceToHost, stream));
  sync();
  const bool verbose = getenv("OB_VERBOSE") != nullptr;
  if ((int)total != nranks) {
    if (verbose) fprintf(stderr, "[outerbase_b200] rank %d: peer memory not available (%d of %d ranks), allreduce stays on NCCL\n", rank, (int)total, nranks);
    p2p_release();
    return;
  }
  p2p.G = nranks;
  if (verbose) fprintf(stderr, "[outerbase_b200] rank %d: one-shot allreduce over peer memory, %d ranks\n", rank, nranks);
}

static void p2p_launch(Ctx& c, double* buf, size_t n, const double* partial, int nblocks, int nslots, const int32_t* slot_term) {
  P2PArgs a{};
  for (int r = 0; r < c.p2p.G; ++r) a.slots[r] = reinterpret_cast<uint4*>(c.p2p.peer[r]);
  if (++c.p2p.seq == 0) c.p2p.seq = 2; /* 0 is the tag of the zero-initialised buffer; keep the parity sequence */
  a.G = c.p2p.G; a.rank = c.rank; a.seq = c.p2p.seq; a.timeout_ns = c.p2p.timeout_ns;
  const int grid = (int)((n + Ctx::P2P::kThreads - 1) / Ctx::P2P::kThreads);
  if (slot_term) p2p_allreduce_kernel<true><<<grid, Ctx::P2P::kThreads, 0, c.stream>>>(a, buf, (int)n, partial, nblocks, nslots, slot_term);
  else p2p_allreduce_kernel<false><<<grid, Ctx::P2P::kThreads, 0, c.stream>>>(a, buf, (int)n, nullptr, 0, 0, nullptr);
  const cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) throw CudaError(std::string("p2p_allreduce_kernel: ") + cudaGetErrorString(e));
  ++c.launches;
}

bool Ctx::p2p_ok(size_t n) const { return p2p.G && p2p.enabled && n <= P2P::kCap; }

Ctx::P2PCall Ctx::p2p_next_call() {
  P2PCall a{};
  for (int r = 0; r < p2p.G; ++r) a.slots[r] = p2p.peer[r];
  if (++p2p.seq == 0) p2p.seq = 2; /* as p2p_launch: 0 is the tag of the zero-initialised buffer */
  a.G = p2p.G; a.rank = rank; a.seq = p2p.seq; a.timeout_ns = p2p.timeout_ns;
  return a;
}

const unsigned* Ctx::stream_rows_begin() {
  if (!copy_stream) {
    OB_CUDA(cudaStreamCreateWithFlags(&copy_stream, cudaStreamNonBlocking));
    OB_CUDA(cudaEventCreateWithFlags(&ev_main, cudaEventDisableTiming));
    OB_CUDA(cudaEventCreateWithFlags(&ev_copy, cudaEventDisableTiming));
    OB_CUDA(cudaMalloc(&rows_ready, sizeof(unsigned)));
    OB_CUDA(cudaMallocHost(&rows_table, 64 * sizeof(unsigned)));
  }
  OB_CUDA(cudaMemsetAsync(rows_ready, 0, sizeof(unsigned), stream));
  OB_CUDA(cudaEventRecord(ev_main, stream));
  OB_CUDA(cudaStreamWaitEvent(copy_stream, ev_main, 0));
  return rows_ready;
}

/* cuStreamWriteValue32 through the runtime's driver entry point: publishes the arrived-row count in stream order
 * without a second DMA transfer per chunk (falls back to a 4-byte copy) */
static bool stream_write_u32(cudaStream_t st, unsigned* dev, unsigned value) {
  using Fn = int (*)(cudaStream_t, unsigned long long, unsigned, unsigned);
  static Fn fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* f = nullptr;
    cudaDriverEntryPointQueryResult qr;
    if (!getenv("OB_OVERLAP_NOWRITEVALUE") &&
        cudaGetDriverEntryPoint("cuStreamWriteValue32", &f, cudaEnableDefault, &qr) == cudaSuccess && qr == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<Fn>(f);
  }
  return fn && fn(st, (unsigned long long)(uintptr_t)dev, value, 0u /* CU_STREAM_WRITE_VALUE_DEFAULT */) == 0;
}

void Ctx::stream_rows_copy(double* dst, const double* src, size_t n) {
  /* chunks: enough for the kernel to start on the first rows early, few enough that the fixed cost per DMA transfer
   * (several microseconds) stays below the kernel's own time (OB_OVERLAP_CHUNKS, tools/e2e_probe.py) */
  static const size_t want = [] { const char* e = getenv("OB_OVERLAP_CHUNKS"); return e ? (size_t)std::max(1, atoi(e)) : (size_t)16; }();
  const size_t chunks = std::min<size_t>(std::min<size_t>(want, 64), std::max<size_t>(1, n / 65536));
  const size_t per = ((n + chunks - 1) / chunks + 2047) / 2048 * 2048;
  size_t c = 0;
  for (size_t r0 = 0; r0 < n; r0 += per, ++c) {
    const size_t r1 = std::min(n, r0 + per);
    OB_CUDA(cudaMemcpyAsync(dst + r0, src + r0, (r1 - r0) * sizeof(double), cudaMemcpyHostToDevice, copy_stream));
    if (!stream_write_u32(copy_stream, rows_ready, (unsigned)r1)) {
      rows_table[c] = (unsigned)r1;
      OB_CUDA(cudaMemcpyAsync(rows_ready, rows_table + c, sizeof(unsigned), cudaMemcpyHostToDevice, copy_stream));
    }
  }
  OB_CUDA(cudaEventRecord(ev_copy, copy_stream));
}

void Ctx::stream_rows_end() { OB_CUDA(cudaStreamWaitEvent(stream, ev_copy, 0)); }

double* Ctx::mapped_host_pointer(double* host) {
  cudaPointerAttributes at{};
  if (cudaPointerGetAttributes(&at, host) != cudaSuccess) { (void)cudaGetLastError(); return nullptr; }
  if (at.type != cudaMemoryTypeHost || !at.devicePointer) return nullptr;
  return static_cast<double*>(at.devicePointer);
}

unsigned* Ctx::grid_sync_counter() {
  if (!sync_ctr) {
    OB_CUDA(cudaMalloc(&sync_ctr, sizeof(unsigned)));
    OB_CUDA(cudaMemsetAsync(sync_ctr, 0, sizeof(unsigned), stream));
    sync_count = 0;
  }
  return sync_ctr;
}

void Ctx::allreduce_sum(double* buf, size_t n) {
  if (nranks <= 1 || !comm || n == 0) return;
  if (p2p_ok(n)) { p2p_launch(*this, buf, n, nullptr, 0, 0, nullptr); return; }
  NcclApi& api = NcclApi::get();
  const int rc = api.AllReduce(buf, buf, n, /*ncclDouble*/ 8, /*ncclSum*/ 0, comm, stream);
  if (rc != 0) throw NcclError(std::string("ncclAllReduce: ") + (api.GetErrorString ? api.GetErrorString(rc) : "error"));
}

void DevProgram::upload(cudaStream_t s) {
  fwd.upload(host.fwd, s); bwd.upload(host.bwd, s);
  fwd_off.upload(host.fwd_off, s); bwd_off.upload(host.bwd_off, s);
  slot_base.upload(host.slot_base, s); slot_real.upload(host.slot_real, s);
  slot_term.upload(host.slot_term, s);
  csr_ptr.upload(host.csr_ptr, s); csr_col.upload(host.csr_col, s);
}

/* ------------------------------------------------------------------ launchers */
static void check_launch(Ctx& c, const char* what) {
  const cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) throw CudaError(std::string(what) + ": " + cudaGetErrorString(e));
  c.launches++;
}

int phi_grid(const Ctx& c, u64 N, int tile_rows) {
  const u64 ntiles = (N + tile_rows - 1) / tile_rows;
  return (int)std::max<u64>(1, std::min<u64>(ntiles, (u64)c.sms));
}

struct PhiGeom {
  int R = 0, nbuf = 0, G = 16;
  size_t smem = 0;
  unsigned off_tile, tile_doubles, off_vec, off_prog, off_part;
  int prog_in_smem = 0;
};

/* choose rows per lane / buffering so that the staged tile fits the 227 KB of the SM */
static PhiGeom phi_geometry(const Ctx& c, const DevProgram& pr, const ColTable& ct, bool is_a, u64 N) {
  const bool deep = (is_a ? pr.host.bwd_stack : pr.host.fwd_stack) > 4; /* R=4 with 8 stack slots spills */
  const size_t nwords = is_a ? pr.host.bwd.size() : pr.host.fwd.size();
  const size_t vec_bytes = ((pr.host.nslots() * sizeof(double) + 127) / 128) * 128;
  const int Rs[2] = {4, 2};
  for (int pass = 0; pass < 2; ++pass)      /* pass 0: program copied to smem too */
    for (int nbuf = 2; nbuf >= 1; --nbuf)
      for (int ri = 0; ri < 2; ++ri) {
        const int R = Rs[ri], TR = 32 * R;
        if (R == 4 && (deep || N <= (u64)c.sms * 64)) continue; /* small inputs: finer tiles fill more SMs */
        PhiGeom g;
        g.R = R; g.nbuf = nbuf; g.G = pr.host.G;
        g.off_tile = 128;
        g.tile_doubles = (unsigned)(ct.nload * TR);
        size_t off = g.off_tile + (size_t)nbuf * g.tile_doubles * sizeof(double);
        g.off_vec = (unsigned)off; off += vec_bytes;
        g.off_prog = (unsigned)off;
        g.prog_in_smem = (pass == 0);
        if (g.prog_in_smem) off += ((nwords * 4 + 127) / 128) * 128;
        g.off_part = (unsigned)off;
        if (is_a) off += (size_t)kComputeWarps * TR * sizeof(double);
        g.smem = off;
        if (g.smem <= c.smem_optin) return g;
      }
  PhiGeom none;
  return none;
}
/* the layout the interpreter kernel of a plan runs with; R == 0: the brute-force kernels */
static PhiGeom plan_geometry(const Ctx& c, const PhiPlan& pl, bool is_a) {
  if (!pl.prog->host.fast_ok) return PhiGeom();
  return phi_geometry(c, *pl.prog, *pl.cols, is_a, pl.N);
}
void phi_geometry_info(const Ctx& c, const PhiPlan& pl, bool is_a, int out[4]) {
  const PhiGeom g = plan_geometry(c, pl, is_a);
  out[0] = g.R; out[1] = g.nbuf; out[2] = g.prog_in_smem; out[3] = (int)g.smem;
}

static void fill_params(PhiKParams& p, const PhiPlan& pl, const PhiGeom& g, bool is_a) {
  const DevProgram& pr = *pl.prog;
  p.load_src = pl.cols->load_src.p; p.col_op = pl.cols->col_op.p;
  p.ncol = pl.cols->ncol; p.nload = pl.cols->nload; p.has_ops = pl.cols->has_ops ? 1 : 0;
  p.prog = is_a ? pr.bwd.p : pr.fwd.p;
  p.prog_off = is_a ? pr.bwd_off.p : pr.fwd_off.p;
  p.slot_base = pr.slot_base.p; p.slot_real = pr.slot_real.p; p.slot_term = pr.slot_term.p;
  p.nslots = (int)pr.host.nslots();
  p.nwords = (int)(is_a ? pr.host.bwd.size() : pr.host.fwd.size());
  p.prog_in_smem = g.prog_in_smem;
  p.scale = pl.scale; p.sq = pl.sq; p.N = pl.N;
  p.ntiles = (int)((pl.N + 32 * g.R - 1) / (32 * g.R));
  p.nbuf = g.nbuf;
  p.off_tile = g.off_tile; p.tile_doubles = g.tile_doubles; p.off_vec = g.off_vec; p.off_prog = g.off_prog; p.off_part = g.off_part;
}

template <class Kern>
static void set_smem(Kern k, size_t bytes) {
  OB_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
}

void launch_phi_a(Ctx& c, const PhiPlan& pl, const PhiAArgs& a, Workspace& ws, int* grid_out) {
  const DevProgram& pr = *pl.prog;
  if (pl.N == 0) { if (grid_out) *grid_out = 0; return; }
  const PhiGeom g = plan_geometry(c, pl, true);
  if (g.R == 0) { /* brute-force form; UPDATE / HESS: the trie kernel's epilogue follows as resid_multi_kernel */
    if (a.mode == PHI_DOT) throw std::logic_error("the dot epilogue needs the specialised kernel");
    double* yv = a.mode == PHI_HESS ? a.w : a.out; /* HESS stores no yhat: w holds it until the epilogue rewrites it */
    const int bs = 128;
    phi_a_simple_kernel<<<(unsigned)((pl.N + bs - 1) / bs), bs, 0, c.stream>>>(
        pl.cols->load_src.p, pl.cols->col_op.p, pr.csr_ptr.p, pr.csr_col.p, (int)pr.host.K, a.a, pl.scale, pl.sq, pl.N, yv);
    check_launch(c, "phi_a_simple_kernel");
    int nb = 0;
    if (a.mode != PHI_PLAIN) {
      /* at most one partial per SM, like the trie kernel's grid: ssq_partial buffers are sized for that */
      const u64 ld = std::max(pl.ld, pl.N);
      nb = (int)std::min<u64>((ld + kResidThreads - 1) / kResidThreads, (u64)c.sms);
      const bool update = a.mode == PHI_UPDATE;
      double* part = update ? (a.ssq_partial ? a.ssq_partial : ws.ssq.ensure(c.sms)) : nullptr;
      resid_multi_kernel<<<dim3((unsigned)nb, 1), kResidThreads, 0, c.stream>>>(yv, a.y, a.w, pl.N, ld, a.sd, nullptr, update ? 1 : 0, part);
      check_launch(c, "resid_multi_kernel");
    }
    if (grid_out) *grid_out = a.mode == PHI_UPDATE ? nb : 0;
    return;
  }
  PhiKParams p{};
  fill_params(p, pl, g, true);
  p.a = a.a; p.out = a.out; p.w = a.w; p.y = a.y; p.sd = a.sd; p.mode = a.mode;
  const int grid = phi_grid(c, pl.N, 32 * g.R);
  if (a.mode == PHI_UPDATE) p.ssq_partial = a.ssq_partial ? a.ssq_partial : ws.ssq.ensure(c.sms);
#define OB_LAUNCH_A(RR, SS, PP) { set_smem(phi_a_kernel<RR, SS, PP>, g.smem); phi_a_kernel<RR, SS, PP><<<grid, kPhiThreads, g.smem, c.stream>>>(p); }
#define OB_LAUNCH_A2(RR, SS) { if (g.prog_in_smem) OB_LAUNCH_A(RR, SS, true) else OB_LAUNCH_A(RR, SS, false) }
  const int sd = pr.host.bwd_stack;
  if (g.R == 4) { if (sd <= 4) OB_LAUNCH_A2(4, 4) else OB_LAUNCH_A2(4, 8) }
  else { if (sd <= 4) OB_LAUNCH_A2(2, 4) else OB_LAUNCH_A2(2, 8) }
#undef OB_LAUNCH_A2
#undef OB_LAUNCH_A
  check_launch(c, "phi_a_kernel");
  if (grid_out) *grid_out = grid;
}

void launch_phi_t(Ctx& c, const PhiPlan& pl, const double* w, double* out, Workspace& ws) {
  const DevProgram& pr = *pl.prog;
  const int K = (int)pr.host.K;
  if (K == 0) return;
  if (pl.N == 0) { launch_fill(c, out, K, 0.0); return; }
  const PhiGeom g = plan_geometry(c, pl, false);
  if (g.R == 0) { /* brute-force form: per-CTA partials, added in a fixed order */
    const u64 ctas = 2 * (u64)c.sms;
    const int nb = (int)std::max<u64>(1, std::min<u64>((pl.N + kSimpleTThreads - 1) / kSimpleTThreads, ctas));
    const unsigned nk = (unsigned)std::min<u64>({(u64)K, std::max<u64>(1, ctas / nb), 65535});
    double* part = ws.partial.ensure((size_t)nb * K);
    phi_t_simple_kernel<<<dim3((unsigned)nb, nk), kSimpleTThreads, 0, c.stream>>>(
        pl.cols->load_src.p, pl.cols->col_op.p, pr.csr_ptr.p, pr.csr_col.p, K, w, pl.scale, pl.sq, pl.N, part);
    check_launch(c, "phi_t_simple_kernel");
    colsum_partials_kernel<<<(unsigned)K, 32, 0, c.stream>>>(part, nb, out);
    check_launch(c, "colsum_partials_kernel");
    return;
  }
  PhiKParams p{};
  fill_params(p, pl, g, false);
  const int grid = phi_grid(c, pl.N, 32 * g.R);
  p.win = w;
  p.partial = ws.partial.ensure((size_t)grid * p.nslots);
#define OB_LAUNCH_T(RR, SS, PP) { set_smem(phi_t_kernel<RR, SS, PP>, g.smem); phi_t_kernel<RR, SS, PP><<<grid, kPhiThreads, g.smem, c.stream>>>(p); }
#define OB_LAUNCH_T2(RR, SS) { if (g.prog_in_smem) OB_LAUNCH_T(RR, SS, true) else OB_LAUNCH_T(RR, SS, false) }
  const int sd = pr.host.fwd_stack;
  if (g.R == 4) { if (sd <= 4) OB_LAUNCH_T2(4, 4) else OB_LAUNCH_T2(4, 8) }
  else { if (sd <= 4) OB_LAUNCH_T2(2, 4) else OB_LAUNCH_T2(2, 8) }
#undef OB_LAUNCH_T2
#undef OB_LAUNCH_T
  check_launch(c, "phi_t_kernel");
  launch_phi_t_reduce(c, p.partial, grid, p.nslots, pr.slot_term.p, out);
}

void launch_phi_t_reduce(Ctx& c, const double* partial, int nblocks, int nslots, const int32_t* slot_term, double* out) {
  if (c.fuse_n) { /* the caller's allreduce of out[0..fuse_n) rides on this launch (Ctx::fuse_allreduce) */
    p2p_launch(c, out, c.fuse_n, partial, nblocks, nslots, slot_term);
    c.fuse_n = 0;
    c.fused = true;
    return;
  }
  phi_t_reduce_kernel<<<(nslots + 127) / 128, 128, 0, c.stream>>>(partial, nblocks, nslots, slot_term, out);
  check_launch(c, "phi_t_reduce_kernel");
}

void launch_getmat(Ctx& c, const PhiPlan& pl, double* out, u64 ldo) {
  const DevProgram& pr = *pl.prog;
  if (pl.N == 0 || pr.host.K == 0) return;
  const int bs = 128;
  dim3 grid((unsigned)((pl.N + bs - 1) / bs), (unsigned)std::min<u64>(pr.host.K, 32768));
  getmat_kernel<<<grid, bs, 0, c.stream>>>(pl.cols->load_src.p, pl.cols->col_op.p, pr.csr_ptr.p, pr.csr_col.p, (int)pr.host.K,
                                          pl.scale, pl.sq, pl.N, out, ldo);
  check_launch(c, "getmat_kernel");
}

/* ------------------------------------------------------------------ device-resident CG stages (ob_device.cuh) */
constexpr int kCgThreads = 1024;
/* sum over the CTA in a fixed order: lanes by butterfly, warps in index order by thread 0; all threads get the result */
__device__ double cg_block_sum(double v, double* sm) {
#pragma unroll
  for (int m = 16; m > 0; m >>= 1) v += __shfl_xor_sync(0xffffffffu, v, m);
  __syncthreads(); /* sm may still be read from the previous sum */
  if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = v;
  __syncthreads();
  if (threadIdx.x == 0) {
    double s = 0.0;
    for (int w = 0; w < kCgThreads / 32; ++w) s += sm[w];
    sm[32] = s;
  }
  __syncthreads();
  return sm[32];
}

/* One CTA per column (blockIdx.x): the column's K-slices of every vector and its own CG_NSCAL scalars.  c.running is
 * set only by the column-batched caller; there a column whose stop test has passed is frozen (the reference `break`s,
 * fit.cpp:73) -- its stages return before touching anything. */
__global__ void __launch_bounds__(kCgThreads) cg_stage_kernel(CgParams c) {
  __shared__ double sm[33];
  const int K = c.K, tid = threadIdx.x;
  const size_t off = (size_t)blockIdx.x * (size_t)K;
  c.coeff += off; c.grad += off; c.m += off; c.rm += off; c.p += off; c.q += off; c.red += off;
  double* S = c.scal + (size_t)blockIdx.x * CG_NSCAL;
  if (c.running && S[CG_STOP] != 0.0) return;
  const double sca = c.sca_col ? c.sca_col[blockIdx.x] : c.sca;
  if (c.stage == CG_INIT) {
    for (int i = tid; i < K; i += kCgThreads) { const double rm = c.grad[i] / c.m[i]; c.rm[i] = rm; c.p[i] = rm; }
    return;
  }
  if (c.stage == CG_POST_UPDATE) {
    /* logpr_gauss::update (logpr_gauss.cpp:98-105) + loglik_gauss::update's scalars (loglik_gauss.cpp:121-128) +
     * lpdfvec::update's sums over the children in their order (fit.cpp:352-361) */
    double s1 = 0.0, s2 = 0.0;
    for (int i = tid; i < K; i += kCgThreads) {
      const double sd = c.sds[i] * sca;
      const double st = c.coeff[i] / sd;
      s1 += st * st;
      s2 += log(sd);
      const double gpr = -1. * st / sd, glik = c.red[i];
      c.grad[i] = c.lik_first ? (0.0 + glik) + gpr : (0.0 + gpr) + glik;
    }
    const double t1 = cg_block_sum(s1, sm), t2 = cg_block_sum(s2, sm);
    const double val_pr = -0.5 * t1 - t2;
    const double ssq = c.ssq ? c.ssq[blockIdx.x] : c.red[K];
    const double val_lik = c.use_sumlogsd ? -0.5 * ssq - c.sumlogsd : -0.5 * ssq - c.nglobal * log(c.obssd_col ? c.obssd_col[blockIdx.x] : c.obssd);
    double val = c.lik_first ? (0.0 + val_lik) + val_pr : (0.0 + val_pr) + val_lik;
    if (c.domarg) val += c.vma_col ? c.vma_col[blockIdx.x] : c.val_margadj;
    const double valo = S[CG_VALO], alpha = S[CG_ALPHA], num = S[CG_NUM];
    double s3 = 0.0;
    for (int i = tid; i < K; i += kCgThreads) {
      const double rm = c.grad[i] / c.m[i];
      c.rm[i] = rm;
      s3 += (alpha * c.q[i]) * rm;
    }
    const double num2 = -cg_block_sum(s3, sm);
    const double beta = num2 / num;
    for (int i = tid; i < K; i += kCgThreads) c.p[i] = c.rm[i] + beta * c.p[i];
    if (tid == 0) { S[CG_BETA] = beta; S[CG_VALDIFF] = val - valo; S[CG_VAL] = val; S[CG_VAL_LIK] = val_lik; S[CG_VAL_PR] = val_pr; }
    return;
  }
  /* q = hessmult(p): lpdfvec::hessmult sums the children in their order (fit.cpp:388-397); loglik part = red,
   * logpr_gauss::hessmult = p / (sd sca)^2 (logpr_gauss.cpp:112-114) */
  double sn = 0.0, sd_ = 0.0;
  for (int i = tid; i < K; i += kCgThreads) {
    const double sd = c.sds[i] * sca;
    const double hp = c.p[i] / (sd * sd), hl = c.red[i];
    const double q = c.lik_first ? hl + hp : hp + hl;
    c.q[i] = q;
    sn += c.grad[i] * c.rm[i];
    sd_ += q * c.p[i];
  }
  if (c.stage == CG_FINISH_Q) return;
  const double num = cg_block_sum(sn, sm), denom = cg_block_sum(sd_, sm);
  const bool stop = num < c.tol && S[CG_VALDIFF] < c.tol; /* fit.cpp:73 */
  const double alpha = num / denom;
  if (!stop)
    for (int i = tid; i < K; i += kCgThreads) c.coeff[i] += alpha * c.p[i];
  if (tid == 0) {
    S[CG_NUM] = num; S[CG_STOP] = stop ? 1.0 : 0.0;
    if (!stop) { S[CG_DENOM] = denom; S[CG_ALPHA] = alpha; S[CG_VALO] = S[CG_VAL]; }
    if (c.running) {
      if (stop) S[CG_ITER] = c.iter;
      else atomicAdd(c.running + (c.iter & 1), 1u);
    }
  }
}

void launch_cg_stage(Ctx& c, const CgParams& p, u64 ncol) {
  cg_stage_kernel<<<(unsigned)ncol, kCgThreads, 0, c.stream>>>(p);
  check_launch(c, "cg_stage_kernel");
}

void launch_resid_multi(Ctx& c, const double* yhat, const double* y, double* w, u64 N, u64 ld, u64 C, double sd, bool update,
                        DevBuf<double>& partial, double* ssq_out, const double* sd_cols, const double* sd_rows) {
  if (C == 0) return;
  if (ld == 0) { /* a rank without rows still takes part in the sums over ranks */
    if (update) OB_CUDA(cudaMemsetAsync(ssq_out, 0, C * sizeof(double), c.stream));
    return;
  }
  const int nb = (int)std::max<u64>(1, std::min<u64>((ld + kResidThreads - 1) / kResidThreads, std::max<u64>(1, (u64)c.sms * 8 / C)));
  if (update) partial.ensure((size_t)nb * C);
  resid_multi_kernel<<<dim3((unsigned)nb, (unsigned)C), kResidThreads, 0, c.stream>>>(yhat, y, w, N, ld, sd, sd_cols, update ? 1 : 0,
                                                                                      update ? partial.p : nullptr, sd_rows);
  check_launch(c, "resid_multi_kernel");
  if (!update) return;
  colsum_partials_kernel<<<(unsigned)C, 32, 0, c.stream>>>(partial.p, nb, ssq_out);
  check_launch(c, "colsum_partials_kernel");
}

void launch_sum_partials(Ctx& c, const double* partial, int n, double* out) {
  sum_partials_kernel<<<1, 32, 0, c.stream>>>(partial, n, out);
  check_launch(c, "sum_partials_kernel");
}

__global__ void gradcols_kernel(const double* __restrict__ B, const double* __restrict__ G, unsigned long long ld, unsigned long long L,
                                double* __restrict__ out, int sq) {
  const unsigned long long n = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= ld) return;
  const double g0 = G[n];
  for (unsigned long long j = 1; j <= L; ++j) {
    const double b = B[n + j * ld];
    const double c = G[n + j * ld] - g0 * b;
    out[n + (j - 1) * ld] = sq ? 2.0 * (b * c) : c;
  }
}
void launch_gradcols(Ctx& c, const double* B, const double* G, u64 ld, u64 L, double* out, int sq) {
  if (ld == 0 || L == 0) return;
  gradcols_kernel<<<(unsigned)((ld + 255) / 256), 256, 0, c.stream>>>(B, G, ld, L, out, sq);
  check_launch(c, "gradcols_kernel");
}
__global__ void square_kernel(const double* __restrict__ in, unsigned long long n, double* __restrict__ out) {
  for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (unsigned long long)gridDim.x * blockDim.x) {
    const double x = in[i];
    out[i] = x * x;
  }
}
void launch_square(Ctx& c, const double* in, u64 n, double* out) {
  if (n == 0) return;
  square_kernel<<<c.sms * 16, 256, 0, c.stream>>>(in, n, out);
  check_launch(c, "square_kernel");
}
__global__ void scaled_product_kernel(double coef, const double* __restrict__ g, const double* __restrict__ w, unsigned long long n,
                                      double* __restrict__ out) {
  const unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = coef * (g[i] * w[i]);
}
void launch_scaled_product(Ctx& c, double coef, const double* g, const double* w, u64 n, double* out) {
  if (n == 0) return;
  scaled_product_kernel<<<(unsigned)((n + 255) / 256), 256, 0, c.stream>>>(coef, g, w, n, out);
  check_launch(c, "scaled_product_kernel");
}
__global__ void masked_add_kernel(const double* __restrict__ a, const double* __restrict__ b, const unsigned char* __restrict__ mask,
                                  unsigned long long n, double* __restrict__ out) {
  const unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = mask[i] ? a[i] + b[i] : a[i];
}
void launch_masked_add(Ctx& c, const double* a, const double* b, const unsigned char* mask, u64 n, double* out) {
  if (n == 0) return;
  masked_add_kernel<<<(unsigned)((n + 255) / 256), 256, 0, c.stream>>>(a, b, mask, n, out);
  check_launch(c, "masked_add_kernel");
}

__global__ void gather_coef_blocks_kernel(const double* __restrict__ A, unsigned long long K, unsigned long long col0, int ncols,
                                         const int32_t* __restrict__ slot_term, int nslots, int nrows, double* __restrict__ out) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x; /* one thread per (slot, column) */
  if (idx >= nrows * 64) return;
  const int s = idx >> 6, c = idx & 63;
  double v = 0.0;
  if (s < nslots && c < ncols) { const int t = slot_term[s]; if (t >= 0) v = A[(unsigned long long)t + (col0 + c) * K]; }
  out[(size_t)s * 64 + (c ^ ((s & 3) << 2))] = v; /* phi_am_spec's bank swizzle */
}
void launch_gather_coef_blocks(Ctx& c, const double* A, u64 K, u64 col0, int ncols, const int32_t* slot_term, int nslots, int nrows, double* out) {
  const int n = nrows * 64;
  gather_coef_blocks_kernel<<<(n + 255) / 256, 256, 0, c.stream>>>(A, K, col0, ncols, slot_term, nslots, nrows, out);
  check_launch(c, "gather_coef_blocks_kernel");
}

/* out[n] = add + sum_k A[n, k] * B[n, k], k ascending (predr_std::var, loglik_std.cpp:251-257: sum(adj % basismat, 1)) */
__global__ void rowdot_kernel(const double* __restrict__ A, const double* __restrict__ B, unsigned long long N, unsigned long long K,
                              unsigned long long ld, double add, double* __restrict__ out) {
  const unsigned long long n = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N) return;
  double s = 0.0;
  for (unsigned long long k = 0; k < K; ++k) s += A[n + k * ld] * B[n + k * ld];
  out[n] = s + add;
}
void launch_rowdot(Ctx& c, const double* A, const double* B, u64 N, u64 K, u64 ld, double add, double* out) {
  if (N == 0) return;
  rowdot_kernel<<<(unsigned)((N + 255) / 256), 256, 0, c.stream>>>(A, B, N, K, ld, add, out);
  check_launch(c, "rowdot_kernel");
}

void launch_gda_obssd(Ctx& c, const double* phi2varc, u64 N, u64 ld, double v0, double v1, double* obssd) {
  if (ld == 0) return;
  gda_obssd_kernel<<<(unsigned)((ld + 255) / 256), 256, 0, c.stream>>>(phi2varc, N, ld, v0, v1, obssd);
  check_launch(c, "gda_obssd_kernel");
}

void launch_fill(Ctx& c, double* p, u64 n, double v) {
  if (n == 0) return;
  fill_kernel<<<(unsigned)((n + 255) / 256), 256, 0, c.stream>>>(p, n, v);
  check_launch(c, "fill_kernel");
}

void launch_dot_partials(Ctx& c, const double* a, const double* b, u64 n, double* partial, int* nblocks) {
  const int nb = (int)std::max<u64>(1, std::min<u64>((n + 255) / 256, (u64)c.sms * 4));
  dot_partials_kernel<<<nb, 256, 0, c.stream>>>(a, b, n, partial);
  check_launch(c, "dot_partials_kernel");
  *nblocks = nb;
}

void launch_cov(Ctx& c, int kind, const double* hyp, const double* x1, u64 n1, const double* x2, u64 n2, double* out, double* outg) {
  if (n1 * n2 == 0) return;
  const double h1 = (kind == obh::COV_MAT25) ? 0.0 : hyp[1];
  cov_kernel<<<(unsigned)((n1 * n2 + 255) / 256), 256, 0, c.stream>>>(kind, hyp[0], h1, x1, n1, x2, n2, out, outg);
  check_launch(c, "cov_kernel");
}

void launch_basis_build(Ctx& c, const std::vector<BuildDims>& dims, const double* x_dev, u64 N, u64 ld, const double* knots_dev,
                        const double* rot_dev, u64 rot_ld, const double* rotg_dev, double* basemat, double* basematge,
                        double* scalemat, double* scale, bool dograd) {
  if (ld == 0) return;
  for (size_t l = 0; l < dims.size(); ++l) {
    const BuildDims& D = dims[l];
    BuildKParams p{};
    p.kind = D.kind; p.m = D.m; p.nh = D.nh; p.mp = ((D.m + 3) / 4) * 4 + 4;
    p.h0 = D.hyp[0]; p.h1 = D.hyp[1];
    p.knots = knots_dev + D.knot_off;
    p.x = x_dev + l * ld;
    p.rot = rot_dev + D.rot_off * rot_ld;
    p.rot_ld = rot_ld;
    p.rotg0 = dograd && D.nh > 0 ? rotg_dev + D.rotg_off[0] * rot_ld : nullptr;
    p.rotg1 = dograd && D.nh > 1 ? rotg_dev + D.rotg_off[1] * rot_ld : nullptr;
    p.bm = basemat + D.col_off * ld;
    p.bg0 = dograd && D.nh > 0 ? basematge + D.ge_off[0] * ld : nullptr;
    p.bg1 = dograd && D.nh > 1 ? basematge + D.ge_off[1] * ld : nullptr;
    p.scalecol = scalemat + l * ld;
    p.N = N; p.ld = ld; p.dograd = dograd ? 1 : 0;
    p.mo = D.mo > 0 && D.mo < D.m ? D.mo : D.m;
    const int nh = dograd ? D.nh : 0;
    auto need = [&](int rows) {
      return ((size_t)(1 + nh) * D.m * p.mp + (size_t)(1 + nh) * D.m * rows + 2 * D.m + 2 * rows) * sizeof(double);
    };
    const int mk = (D.m + 3) & ~3;
    auto need_mma = [&](int nt) {
      return ((size_t)(1 + nh) * mk * (nt * 8 + 4) + (size_t)(1 + nh) * mk * 72 + 2 * D.m + 2 * 64) * sizeof(double);
    };
    static const bool use_mma = !(getenv("OB_BUILD") && std::string(getenv("OB_BUILD")) == "fma");
    /* column tiles of 8: the smallest instantiation that covers the columns to build (the accumulators of a tile
     * live in registers, so the count is a template argument); 2 CTAs per SM up to 5 tiles */
#define OB_BUILD_MMA(NT_, PER_SM)                                                                                   \
    {                                                                                                               \
      set_smem(basis_build_mma_kernel<NT_>, need_mma(NT_));                                                         \
      basis_build_mma_kernel<NT_><<<(unsigned)std::min<u64>((ld + 63) / 64, (u64)c.sms * PER_SM), 256, need_mma(NT_), c.stream>>>(p); \
    }
    const int nt = (p.mo + 7) / 8;
    if (use_mma && D.m <= 72 && nt <= 1 && need_mma(1) <= c.smem_optin) OB_BUILD_MMA(1, 2)
    else if (use_mma && D.m <= 72 && nt <= 2 && need_mma(2) <= c.smem_optin) OB_BUILD_MMA(2, 2)
    else if (use_mma && D.m <= 72 && nt <= 3 && need_mma(3) <= c.smem_optin) OB_BUILD_MMA(3, 2)
    else if (use_mma && D.m <= 72 && nt <= 5 && need_mma(5) <= c.smem_optin) OB_BUILD_MMA(5, 2)
    else if (use_mma && D.m <= 72 && need_mma(9) <= c.smem_optin) OB_BUILD_MMA(9, 1)
#undef OB_BUILD_MMA
    else if (need(64) <= c.smem_optin) {
      set_smem(basis_build_kernel<64>, need(64));
      basis_build_kernel<64><<<(unsigned)((ld + 63) / 64), 256, need(64), c.stream>>>(p);
    } else if (need(32) <= c.smem_optin) {
      set_smem(basis_build_kernel<32>, need(32));
      basis_build_kernel<32><<<(unsigned)((ld + 31) / 32), 256, need(32), c.stream>>>(p);
    } else throw std::range_error("too many knots in one dimension for the basis-build kernel");
    check_launch(c, "basis_build_kernel");
  }
  basescale_kernel<<<(unsigned)((ld + 255) / 256), 256, 0, c.stream>>>(scalemat, ld, (int)dims.size(), N, scale);
  check_launch(c, "basescale_kernel");
}

void launch_getbase(Ctx& c, const double* basemat, const double* scalecol, u64 N, u64 ld, u64 col0, u64 m, double* out) {
  if (N * m == 0) return;
  getbase_kernel<<<(unsigned)((N * m + 255) / 256), 256, 0, c.stream>>>(basemat, scalecol, N, ld, col0, m, out);
  check_launch(c, "getbase_kernel");
}

} // namespace obd

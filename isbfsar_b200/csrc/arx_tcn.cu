// tcgen05 cross-attention + distances for ANY tuple count N, tiled over blocks of 128 tuples
// (T=32 pairs N=496 -> 4 tiles, T=16 triples N=560 -> 5, T=32 triples N=4960 -> 39; also N <= 128 for other T).
//
// Reference semantics (modules/ar/utils/model.py:95-135), per (query window b, class c):
//   S = Kq.Kc^T / sqrt(D);  P = softmax(S, dim=-2)  -- normalised over the QUERY tuples, per support tuple s;
//   proto = P.Vc;  logit = -||Vq - proto||_F^2 / N.
// The softmax axis (q) is not the contraction axis of the prototype (s), so flash-attention's online rescaling does
// not apply (SURVEY 7.2-1): the normaliser Z[s] = sum_q exp(S[q,s]) needs ALL query tiles before any P can be formed.
// Two passes per (window, class), both on the schedule of the third-generation kernel (arx_tc3.cu):
//   pass A  for every pair of query tiles (qt0|qt1) and every support tile st:
//             MMA1  S^T[s, (q of qt0 | q of qt1)] = Kc[st] . Kq'^T   (M=128, N=256, K=128, fp16 operands)
//             the two softmax warpgroups take one 128-column half each: exp2, thread-local row sum (thread == TMEM
//             lane == support tuple s) accumulated into Z[st*128+s]
//   pass B  same tiles again: exp2 recomputed, P = E / Z[s] written to shared memory as the MN-major bf16 B operand,
//             MMA2  proto^T[d, q] += Vc^T[st][d, :] . P[q, :]   accumulated over st in TMEM (one accumulator per query
//             tile of the pair).  The accumulator does not start at zero but at -Vq^T: a SELECTION MMA  -Gv^T[d, (p,t)] .
//             Sel[q, (p,t)]^T  (one-hot rows: frame p of tuple q is t; Gv as hi + lo fp16 halves, K = 2cT) rebuilds
//             Vq[q][d] = sum_p Gv_p[frame_p(q)][d] on the tensor core, so after the last st the epilogue warps only form
//             sum_q acc[d][q]^2 -- no table, no gather (tuple features never exist; pad columns come out exactly 0).
// N <= 128 (one query tile) needs no pass A: the row sum of the only tile is the normaliser.
// The exponentials are computed twice (1.67x the exps of a single pass would need E kept on chip: N=496 alone is
// 512 KB of bf16 per class); MUFU.EX2 stays the co-limiting pipe exactly as in the N=120 kernel.
// MODE 1 (open-set head, model.py:323-324,196): same pipeline for the winning class only, with Uc = Wdr.Vc^T (rows l)
// in place of Vc^T, so the accumulator is sum_s P[q,s].(Wdr.Vc[s])[l] and the epilogue writes
//   y[q][l] = (Wdr.Vq[q] + bdr)[l] - acc[l][q]    (head by linearity, DESIGN 5-k4)
// straight into the fp16 activation image of discriminator.fc1.
// ROWMAX variant: subtracts a running row maximum before exp2 (online rescaling of Z across query tiles), for
// LayerNorm affines outside the static bound under which exp2 needs no shift (SURVEY 7.2-1).
// Episode mode (arx_score_episodes): every window has its own support classes, window w of a launch attends classes
// [cls_base + w*way, cls_base + (w+1)*way) of one pool of class tiles; the query side and the head are per window as always.
// Work unit = (window, class), round-robin over one persistent CTA per SM; 16 warps, warp-specialised; every
// mbarrier wait carries a watchdog (a protocol bug traps instead of hanging the GPU).
#include "arx_internal.cuh"
#include "arx_ptx.cuh"
#include <cuda_bf16.h>
#include <stdlib.h>

namespace {
using namespace ptx;

constexpr int DD = 128;
constexpr uint32_t IMG_BYTES = 128 * DD * 2;
constexpr uint32_t SUB_BYTES = 128 * 64 * 2;
constexpr int NTHREADS = 512;

constexpr uint32_t OFF_KQ = 0;                       // 64 KB: [sub0: t0 rows | t1 rows][sub1: t0 rows | t1 rows]
constexpr uint32_t OFF_KC = 2 * IMG_BYTES;           // 32 KB
constexpr uint32_t OFF_VCT = 3 * IMG_BYTES;          // 2 x 32 KB
constexpr uint32_t OFF_P = 5 * IMG_BYTES;            // 2 x 32 KB (one per softmax group / query tile of the pair)
constexpr uint32_t OFF_BAR = 7 * IMG_BYTES;
enum { B_FULL_KQ = 0, B_EMPTY_KQ = 1, B_FULL_KC = 2, B_EMPTY_KC = 3, B_FULL_VC = 4, B_EMPTY_VC = 6, B_S_FULL = 8, B_S_EMPTY = 9,
       B_P_FULL = 10, B_P_EMPTY = 12, B_O_FULL = 14, B_O_EMPTY = 16, B_XU = 18, B_COUNT = 20 };
constexpr uint32_t SMEM_BYTES = OFF_BAR + B_COUNT * 8 + 16 + 1024;

struct AttnNParams {
  const __half *kq_img;     // [n_win][nq] 32 KB tiles, K-major SW128, rows = query tuples (LayerNorm-ed, pre-scaled by log2e/sqrt(D))
  const __half *kc_img;     // [classes][ns] tiles, rows = support tuples
  const __half *vct_img;    // [classes][ns] tiles, rows = d (mode 0: Vc^T) or l (mode 1: Uc), cols = support tuples, bf16
  const __half *vq_img;     // [windows][nsel] 16 KB sub-tiles (128 rows x 64, fp16 K-major SW128): MINUS the per-frame table of the
                            // window, hi | lo halves, column h*c*T + p*T + t; rows = d (mode 0: V projections) or l (mode 1: head table)
  const __half *sel_img;    // [nq][nsel] 16 KB sub-tiles (128 query rows x 64): one-hot frame selection of every tuple, both halves
  int nsel;                 // 64-column sub-tiles of the selection operands = ceil(2*c*T / 64)
  const int32_t *chosen;    // mode 1: class of every window
  float *partial;           // mode 0: [n_win*way][4] squared-distance partials (one per epilogue warp)
  float *y;                 // mode 1: fp32 [n_win][N*L], or
  __half *y_img;            //         fp16 activation image [ceil(n_win/128)][y_nk][128 x 64]
  float *zscratch;          // [grid][2 unit parity][2 groups][2: Z | M][ns*128]
  int *diag;                // watchdog record (see mbar_wait_wd)
  long long *trace;         // optional timeline of CTA 0 (bring-up tool): [3 roles][64 steps][8 stamps] of clock64
  int n_win, way, N, T, c, nq, ns, mode, L, y_nk;
  int free_a;               // pass A: the softmax groups run free instead of taking turns on the MUFU phase
  int poly;                 // pass A: every other register pair takes the FMA-pipe exp2 polynomial
  int same_window;          // mode 1: every unit scores window 0 (against class chosen[u]); y row = u (streaming: the head of ALL classes at once)
  // class tiles of unit u: cls_base + u % cls_mod (mode 0), cls_base + u*cls_stride + chosen[u] (mode 1).  Ordinary launches:
  // cls_base = cls_stride = 0, cls_mod = way.  Episode mode (a pool of per-window support sets): window w of the launch attends
  // pool classes [cls_base + w*way, cls_base + (w+1)*way), so cls_mod = n_win*way (no wrap) and cls_stride = way
  // (`chosen` stays in [0, way): the argmax within the episode)
  int cls_base, cls_mod, cls_stride;
};

// Watchdog wait: a protocol bug must not hang the GPU.  On a timeout (~1 s) the first thread to notice records
// (barrier index, parity, role, step) in p.diag and every waiter of the CTA grid bails out; the launcher reports it.
__device__ __forceinline__ void mbar_wait_wd_(uint64_t *bar, uint32_t parity, int *diag, int code) {
  if (mbar_try_wait(bar, parity)) return;
  const long long t0 = clock64();
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if ((++spins & 1023u) == 0u) {
      if (*reinterpret_cast<volatile int *>(diag) != 0) return;
      if (clock64() - t0 > 2000000000LL) {
        if (atomicCAS(diag, 0, code | 0x40000000) == 0) { diag[1] = (int)blockIdx.x; diag[2] = (int)threadIdx.x; diag[3] = (int)parity; }
        return;
      }
    }
  }
}
#define TRACEN(role, step, slot) do { if (p.trace && blockIdx.x == 0 && (step) < 64) p.trace[(((role) * 64) + (step)) * 8 + (slot)] = clock64(); } while (0)
#define mbar_wait_wd(bar, parity) mbar_wait_wd_((bar), (parity), p.diag, (int)((bar) - bars) | (__LINE__ << 8))

__device__ __forceinline__ uint32_t ex2_bits(uint32_t x) {
  uint32_t y;
  asm volatile("ex2.approx.ftz.f32 %0, %1;" : "=r"(y) : "r"(x));
  return y;
}
__device__ __forceinline__ float ex2f(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// exp2 of two pre-scaled scores on the FMA pipe instead of the MUFU: round-to-nearest split x = n + f with the 1.5*2^23 magic
// constant, 2^f on [-0.5, 0.5] by a degree-3 polynomial (max relative error 7.5e-5), exponent add by an integer shift-add.
// Used for every other register pair of PASS A only: there the tile is summed, not stored, the FMA pipe is idle, and the MUFU
// (16 lanes/clk/SM) is the limiter -- in the single-pass N=120 kernel the same trick gained nothing because the FMA pipe was
// already busy with scaling and stores.  |x| < 100 by the LayerNorm bound (or after the row-max shift).
__device__ __forceinline__ void exp2_poly2(uint32_t &a, uint32_t &b) {
  const uint64_t MAGIC = pack2(12582912.0f, 12582912.0f);
  const uint64_t x = pack2u(a, b);
  const uint64_t t = add2(x, MAGIC);
  const uint64_t f = sub2(x, sub2(t, MAGIC));
  uint64_t p2 = fma2(f, pack2(0.0551716685f, 0.0551716685f), pack2(0.2426111251f, 0.2426111251f));
  p2 = fma2(p2, f, pack2(0.6932609677f, 0.6932609677f));
  p2 = fma2(p2, f, pack2(0.9999280572f, 0.9999280572f));
  a = (uint32_t)p2 + ((uint32_t)t << 23);
  b = (uint32_t)(p2 >> 32) + ((uint32_t)(t >> 32) << 23);
}

template <bool ROWMAX>
__global__ void __launch_bounds__(NTHREADS, 1) k_attn_tcn(const AttnNParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t *smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint64_t *bars = reinterpret_cast<uint64_t *>(smem + OFF_BAR);
  uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(smem + OFF_BAR + B_COUNT * 8);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const bool head = p.mode == 1;
  const int n_units = head ? p.n_win : p.n_win * p.way;
  const int my_units = n_units > (int)blockIdx.x ? (n_units - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x : 0;
  const int nq = p.nq, ns = p.ns, nqp = (nq + 1) >> 1;
  const int pass0 = nq == 1 ? 1 : 0;                   // a single query tile needs no normaliser pass

  if (threadIdx.x == 0) {
    mbar_init(&bars[B_FULL_KQ], 1); mbar_init(&bars[B_EMPTY_KQ], 1);
    mbar_init(&bars[B_FULL_KC], 1); mbar_init(&bars[B_EMPTY_KC], 1);
    mbar_init(&bars[B_S_FULL], 1); mbar_init(&bars[B_S_EMPTY], 256);
    for (int i = 0; i < 2; ++i) {
      mbar_init(&bars[B_FULL_VC + i], 1); mbar_init(&bars[B_EMPTY_VC + i], 1);
      mbar_init(&bars[B_P_FULL + i], 128); mbar_init(&bars[B_P_EMPTY + i], 1);
      mbar_init(&bars[B_O_FULL + i], 1); mbar_init(&bars[B_O_EMPTY + i], 128);
      mbar_init(&bars[B_XU + i], 128);
    }
    mbar_init_fence();
  }
  if (warp == 3) { tmem_alloc(tmem_slot, 512); tmem_relinquish(); }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  const uint32_t TM_S = tmem, TM_O = tmem + 256;

  if (warp < 4) {
    setmaxnreg_dec<40>();
    if (warp == 0) {
      if (elect_one()) {            // producer: class operands -- Kc every step (single-buffered), Vc^T/Uc in pass B (2-stage ring)
        int k = 0, kr = 0;                     // kr: items of the Vc ring (selection operands and Vc^T tiles alike)
        for (int ui = 0; ui < my_units; ++ui) {
          const int u = blockIdx.x + ui * gridDim.x;
          const size_t cls = (size_t)p.cls_base + (head ? (size_t)u * p.cls_stride + p.chosen[u] : (size_t)(u % p.cls_mod));
          const size_t win = head ? (p.same_window ? 0 : (size_t)u) : (size_t)(u / p.way);
          const uint8_t *kc0 = reinterpret_cast<const uint8_t *>(p.kc_img) + cls * ns * IMG_BYTES;
          const uint8_t *vc0 = reinterpret_cast<const uint8_t *>(p.vct_img) + cls * ns * IMG_BYTES;
          const uint8_t *vq0 = reinterpret_cast<const uint8_t *>(p.vq_img) + win * p.nsel * SUB_BYTES;
          for (int pass = pass0; pass < 2; ++pass)
            for (int qp = 0; qp < nqp; ++qp) {
              for (int st = 0; st < ns; ++st, ++k) {
                const uint8_t *kc = kc0 + (size_t)st * IMG_BYTES;
                mbar_wait_wd(&bars[B_EMPTY_KC], (k & 1) ^ 1);
                mbar_arrive_expect_tx(&bars[B_FULL_KC], IMG_BYTES);
                bulk_g2s(smem + OFF_KC, kc, SUB_BYTES, &bars[B_FULL_KC]);
                bulk_g2s(smem + OFF_KC + SUB_BYTES, kc + SUB_BYTES, SUB_BYTES, &bars[B_FULL_KC]);
                if (pass == 1 && st == 0) {
                  // selection operands of the pair's tiles: [ -Gv^T sub-tile j | Sel sub-tile j of the query tile ] per ring item.
                  // Issued AFTER the first Kc of the pair: the ring only drains once the epilogue has released the accumulators,
                  // and MMA1 of the new pair must not wait behind that.
                  const int nw = min(2, nq - 2 * qp);
                  for (int w = 0; w < nw; ++w)
                    for (int j = 0; j < p.nsel; ++j, ++kr) {
                      const int sg = kr & 1;
                      mbar_wait_wd(&bars[B_EMPTY_VC + sg], ((kr >> 1) & 1) ^ 1);
                      mbar_arrive_expect_tx(&bars[B_FULL_VC + sg], IMG_BYTES);
                      bulk_g2s(smem + OFF_VCT + sg * IMG_BYTES, vq0 + (size_t)j * SUB_BYTES, SUB_BYTES, &bars[B_FULL_VC + sg]);
                      bulk_g2s(smem + OFF_VCT + sg * IMG_BYTES + SUB_BYTES,
                               reinterpret_cast<const uint8_t *>(p.sel_img) + ((size_t)(2 * qp + w) * p.nsel + j) * SUB_BYTES, SUB_BYTES,
                               &bars[B_FULL_VC + sg]);
                    }
                }
                if (pass == 1) {
                  const uint8_t *vc = vc0 + (size_t)st * IMG_BYTES;
                  const int sg = kr & 1;
                  mbar_wait_wd(&bars[B_EMPTY_VC + sg], ((kr >> 1) & 1) ^ 1);
                  mbar_arrive_expect_tx(&bars[B_FULL_VC + sg], IMG_BYTES);
                  bulk_g2s(smem + OFF_VCT + sg * IMG_BYTES, vc, SUB_BYTES, &bars[B_FULL_VC + sg]);
                  bulk_g2s(smem + OFF_VCT + sg * IMG_BYTES + SUB_BYTES, vc + SUB_BYTES, SUB_BYTES, &bars[B_FULL_VC + sg]);
                  ++kr;
                }
              }
            }
        }
      }
    } else if (warp == 2) {
      if (elect_one()) {            // producer: the pair of query tiles, interleaved into one 256-row K-major B operand
        int kq = 0;
        for (int ui = 0; ui < my_units; ++ui) {
          const int u = blockIdx.x + ui * gridDim.x;
          const size_t win = head ? (p.same_window ? 0 : (size_t)u) : (size_t)(u / p.way);
          const uint8_t *q0 = reinterpret_cast<const uint8_t *>(p.kq_img) + win * nq * IMG_BYTES;
          for (int pass = pass0; pass < 2; ++pass)
            for (int qp = 0; qp < nqp; ++qp, ++kq) {
              const int nw = min(2, nq - 2 * qp);
              mbar_wait_wd(&bars[B_EMPTY_KQ], (kq & 1) ^ 1);
              mbar_arrive_expect_tx(&bars[B_FULL_KQ], nw * IMG_BYTES);
              for (int w = 0; w < nw; ++w) {
                const uint8_t *src = q0 + (size_t)(2 * qp + w) * IMG_BYTES;
                bulk_g2s(smem + OFF_KQ + w * SUB_BYTES, src, SUB_BYTES, &bars[B_FULL_KQ]);                              // d 0..63
                bulk_g2s(smem + OFF_KQ + 2 * SUB_BYTES + w * SUB_BYTES, src + SUB_BYTES, SUB_BYTES, &bars[B_FULL_KQ]);  // d 64..127
              }
              // the next pair is needed ns steps from now and its load is exposed (single buffer): have it wait in L2
              const int nqp_next = qp + 1 < nqp ? qp + 1 : 0;
              bulk_prefetch_l2(q0 + (size_t)(2 * nqp_next) * IMG_BYTES, min(2, nq - 2 * nqp_next) * IMG_BYTES);
            }
        }
      }
    } else if (warp == 1) {
      if (elect_one()) {            // MMA1 issuer: one N=256 (N=128 for an unpaired last tile) MMA sequence per step
        constexpr uint64_t DESC_K = smem_desc_sw128(16, 1024);
        const uint32_t sbase = smem_u32(smem);
        int k = 0, kq = 0;
        for (int ui = 0; ui < my_units; ++ui)
          for (int pass = pass0; pass < 2; ++pass)
            for (int qp = 0; qp < nqp; ++qp, ++kq) {
              const int nw = min(2, nq - 2 * qp);
              const uint32_t idesc = nw == 2 ? idesc_f16(128, 256, 0, 0) : idesc_f16(128, 128, 0, 0);
              TRACEN(0, k, 3);
              mbar_wait_wd(&bars[B_FULL_KQ], kq & 1);
              TRACEN(0, k, 4);
              for (int st = 0; st < ns; ++st, ++k) {
                TRACEN(0, k, 0);
                mbar_wait_wd(&bars[B_FULL_KC], k & 1);
                TRACEN(0, k, 1);
                mbar_wait_wd(&bars[B_S_EMPTY], (k & 1) ^ 1);
                tc_fence_after();
                TRACEN(0, k, 2);
#pragma unroll
                for (int kk = 0; kk < 8; ++kk) {
                  const uint32_t aoff = (kk >> 2) * SUB_BYTES + (kk & 3) * 32;
                  const uint32_t boff = (kk >> 2) * (2 * SUB_BYTES) + (kk & 3) * 32;
                  mma_f16_ss(TM_S, smem_desc_at(DESC_K, sbase + OFF_KC + aoff), smem_desc_at(DESC_K, sbase + OFF_KQ + boff), idesc, kk > 0);
                }
                mma_commit(&bars[B_S_FULL]);
                mma_commit(&bars[B_EMPTY_KC]);
                if (st == ns - 1) mma_commit(&bars[B_EMPTY_KQ]);
              }
            }
      }
    } else {
      if (elect_one()) {            // MMA2 issuer (pass B): proto^T[d, q of tile w] += Vc^T[st] . P_w, accumulated over st
        constexpr uint64_t DESC_K = smem_desc_sw128(16, 1024);
        constexpr uint64_t DESC_MN = smem_desc_sw128(16384, 1024);
        constexpr uint32_t IDESC2 = idesc_bf16(128, 128, 0, 1);
        const uint32_t sbase = smem_u32(smem);
        constexpr uint32_t IDESC_SEL = idesc_f16(128, 128, 0, 0);
        int kb = 0, kr = 0, ke = 0;
        for (int ui = 0; ui < my_units; ++ui)
          for (int qp = 0; qp < nqp; ++qp, ++ke) {
            const int nw = min(2, nq - 2 * qp);
            // the accumulators of the pair start at -Vq^T (selection MMA), once the epilogue has drained the previous pair's
            for (int w = 0; w < nw; ++w) {
              mbar_wait_wd(&bars[B_O_EMPTY + w], (ke & 1) ^ 1);
              for (int j = 0; j < p.nsel; ++j, ++kr) {
                const int sg = kr & 1;
                mbar_wait_wd(&bars[B_FULL_VC + sg], (kr >> 1) & 1);
                tc_fence_after();
#pragma unroll
                for (int kk = 0; kk < 4; ++kk)
                  mma_f16_ss(TM_O + w * 128, smem_desc_at(DESC_K, sbase + OFF_VCT + sg * IMG_BYTES + kk * 32),
                             smem_desc_at(DESC_K, sbase + OFF_VCT + sg * IMG_BYTES + SUB_BYTES + kk * 32), IDESC_SEL, (j > 0 || kk > 0) ? 1u : 0u);
                mma_commit(&bars[B_EMPTY_VC + sg]);
              }
            }
            if (nw == 1) mbar_wait_wd(&bars[B_O_EMPTY + 1], (ke & 1) ^ 1);      // the absent slot's barriers stay in phase (see below)
            for (int st = 0; st < ns; ++st, ++kb, ++kr) {
              const int sg = kr & 1;
              mbar_wait_wd(&bars[B_FULL_VC + sg], (kr >> 1) & 1);
              for (int w = 0; w < nw; ++w) {
                mbar_wait_wd(&bars[B_P_FULL + w], kb & 1);
                tc_fence_after();
#pragma unroll
                for (int kk = 0; kk < 8; ++kk) {
                  const uint32_t off = (kk >> 2) * SUB_BYTES + (kk & 3) * 32;
                  mma_f16_ss(TM_O + w * 128, smem_desc_at(DESC_K, sbase + OFF_VCT + sg * IMG_BYTES + off),
                             smem_desc_at(DESC_MN, sbase + OFF_P + w * IMG_BYTES + kk * 2048), IDESC2, 1u);
                }
                if (st == ns - 1) mma_commit(&bars[B_O_FULL + w]);
                mma_commit(&bars[B_P_EMPTY + w]);
              }
              if (nw == 1) {        // unpaired tile: slot 1's barriers complete the same phases, sequenced like a real tile (an
                                    // mbarrier parity wait cannot tell phase k from k+2: nothing may run two phases ahead of its waiter)
                mbar_wait_wd(&bars[B_P_FULL + 1], kb & 1);
                if (st == ns - 1) mbar_arrive(&bars[B_O_FULL + 1]);
                mbar_arrive(&bars[B_P_EMPTY + 1]);
              }
              mma_commit(&bars[B_EMPTY_VC + sg]);
            }
          }
      }
    }
  } else if (warp < 12) {
    // ---------------- softmax group g owns query tile g of every pair: S^T columns [128g, 128g+128), P buffer g
    setmaxnreg_inc<160>();
    const int g = (warp - 4) >> 2, quad = warp & 3;
    const int s = quad * 32 + lane;
    const uint32_t lane_base = (uint32_t)(quad * 32) << 16;
    uint8_t *prow = smem + OFF_P + g * IMG_BYTES + (s >> 3) * 1024 + (s & 7) * 128;
    const int NSP = ns * 128;
    int k = 0, kb = 0, kt = 0;               // kt: steps that took the MUFU token
    for (int ui = 0; ui < my_units; ++ui) {
      float *zme = p.zscratch + ((((size_t)blockIdx.x * 2 + (ui & 1)) * 2 + g) * 2) * NSP;      // this group's [Z | M]
      const float *zot = p.zscratch + ((((size_t)blockIdx.x * 2 + (ui & 1)) * 2 + (g ^ 1)) * 2) * NSP;
      for (int pass = pass0; pass < 2; ++pass) {
        if (pass == 1 && pass0 == 0) {         // both groups' normaliser partials must be visible before pass B reads them
          __threadfence_block();
          named_bar_sync(1, 256);
        }
        for (int qp = 0; qp < nqp; ++qp) {
          const int nw = min(2, nq - 2 * qp);
          const int nvalid = p.N - (2 * qp + g) * 128;       // valid query columns of this group's tile (>= 128: all)
          for (int st = 0; st < ns; ++st, ++k) {
            const int zi = st * 128 + s;
            const bool tok = pass == 1 || !p.free_a;
            // everything this step needs from the normaliser scratch is FETCHED here and USED after the exponentials: a global
            // load whose value is consumed right away sits on the softmax critical path (measured: +18 % on triples for zprev alone)
            float zinv = 0.f, mrow = 0.f, zprev = 0.f, za = 0.f, zb = 0.f, ma = 0.f, mb = 0.f;
            if (pass == 0 && qp > 0 && g < nw) zprev = zme[zi];   // running sum of the earlier query tiles
            if (pass == 1 && pass0 == 0 && g < nw) {          // normaliser of this support tuple over ALL query tiles (pass A)
              za = zme[zi]; zb = zot[zi];
              if constexpr (ROWMAX) { ma = zme[NSP + zi]; mb = zot[NSP + zi]; }
            }
            const bool trc = (threadIdx.x == 128 + g * 128);
            if (trc) TRACEN(1 + g, k, 0);
            mbar_wait_wd(&bars[B_S_FULL], k & 1);
            tc_fence_after();
            if (trc) TRACEN(1 + g, k, 1);
            if (g >= nw) {              // unpaired tile: this group has no columns, but its barriers keep their phase, in turn
              mbar_arrive(&bars[B_S_EMPTY]);
              if (tok) {
                mbar_wait_wd(&bars[B_XU + 0], kt & 1);
                mbar_arrive(&bars[B_XU + 1]);
                ++kt;
              }
              if (pass == 1) {          // sequenced like a real P tile: without the wait this barrier could complete two
                                        // phases while the MMA2 issuer is held up behind a slow epilogue (seen on the GPU)
                mbar_wait_wd(&bars[B_P_EMPTY + 1], (kb & 1) ^ 1);
                mbar_arrive(&bars[B_P_FULL + 1]);
                ++kb;
              }
              continue;
            }
            uint32_t r[128];
            tmem_ld32(TM_S + lane_base + g * 128 + 0, *reinterpret_cast<uint32_t(*)[32]>(&r[0]));
            tmem_ld32(TM_S + lane_base + g * 128 + 32, *reinterpret_cast<uint32_t(*)[32]>(&r[32]));
            tmem_ld32(TM_S + lane_base + g * 128 + 64, *reinterpret_cast<uint32_t(*)[32]>(&r[64]));
            tmem_ld32(TM_S + lane_base + g * 128 + 96, *reinterpret_cast<uint32_t(*)[32]>(&r[96]));
            tmem_ld_wait();
            tc_fence_before();
            mbar_arrive(&bars[B_S_EMPTY]);
            // MUFU token: the groups take turns on the exp phase so that one's loads / sums / stores run under the other's MUFU stream
            // (pass B only: in the normaliser pass a group has nothing but loads and sums around its exponentials, and two warps
            // per scheduler issuing MUFU together run the pipe at 8 clk per instruction instead of ~11 for one -- p.free_a)
            if (tok) {
              if (g == 0) { if (kt > 0) mbar_wait_wd(&bars[B_XU + 1], (kt - 1) & 1); }
              else mbar_wait_wd(&bars[B_XU + 0], kt & 1);
            }
            if (trc) TRACEN(1 + g, k, 2);
            float zscale = 0.f;             // ROWMAX pass A: factor that brings the running sum to the new maximum
            if constexpr (ROWMAX) {
              if (pass == 1 && pass0 == 0) mrow = fmaxf(ma, mb);
              if (pass == 0 || pass0 == 1) {
                float mt = -INFINITY;
                if (nvalid >= 128) {
#pragma unroll
                  for (int j = 0; j < 128; ++j) mt = fmaxf(mt, __uint_as_float(r[j]));
                } else {
#pragma unroll
                  for (int j = 0; j < 128; ++j) mt = fmaxf(mt, j < nvalid ? __uint_as_float(r[j]) : -INFINITY);
                }
                if (pass0 == 0 && qp > 0) {
                  const float mo = zme[NSP + zi];
                  mrow = fmaxf(mo, mt);
                  zscale = ex2f(mo - mrow);
                } else {
                  mrow = mt;
                }
              }
              const uint64_t mm = pack2(-mrow, -mrow);
#pragma unroll
              for (int j = 0; j < 128; j += 2) {
                const uint64_t v = add2(pack2u(r[j], r[j + 1]), mm);
                r[j] = (uint32_t)v; r[j + 1] = (uint32_t)(v >> 32);
              }
            }
            if (pass == 0 && p.poly) {
#pragma unroll
              for (int j = 0; j < 128; j += 4) {
                exp2_poly2(r[j], r[j + 1]);
                r[j + 2] = ex2_bits(r[j + 2]); r[j + 3] = ex2_bits(r[j + 3]);
              }
            } else {
#pragma unroll
              for (int j = 0; j < 128; ++j) r[j] = ex2_bits(r[j]);
            }
            if (tok) { mbar_arrive(&bars[B_XU + g]); ++kt; }
            if (trc) TRACEN(1 + g, k, 3);
            if (pass == 0 || pass0 == 1) {
              // row sum over the valid query columns (pad columns of the last tile have S = 0, exp = 1: masked out)
              if (nvalid < 128) {
#pragma unroll
                for (int j = 0; j < 128; ++j) r[j] = j < nvalid ? r[j] : 0u;
              }
              uint64_t z0 = 0ull, z1 = 0ull, z2 = 0ull, z3 = 0ull;
#pragma unroll
              for (int q = 0; q < 64; q += 4) {
                z0 = add2v(z0, pack2u(r[2 * q], r[2 * q + 1]));
                z1 = add2v(z1, pack2u(r[2 * q + 2], r[2 * q + 3]));
                z2 = add2v(z2, pack2u(r[2 * q + 4], r[2 * q + 5]));
                z3 = add2v(z3, pack2u(r[2 * q + 6], r[2 * q + 7]));
              }
              float zl, zh;
              unpack2(add2(add2(z0, z1), add2(z2, z3)), zl, zh);
              const float zs = zl + zh;
              if (pass == 0) {
                if constexpr (ROWMAX) {
                  zme[zi] = qp > 0 ? zprev * zscale + zs : zs;
                  zme[NSP + zi] = mrow;
                } else {
                  zme[zi] = qp > 0 ? zprev + zs : zs;
                }
                continue;
              }
              zinv = __frcp_rn(zs) * 1.0028177f;          // single query tile: the tile's own row sum is the normaliser
            } else {
              if constexpr (ROWMAX) zinv = __frcp_rn(za * ex2f(ma - mrow) + zb * ex2f(mb - mrow)) * 1.0028177f;
              else zinv = __frcp_rn(za + zb) * 1.0028177f;      // centred truncation to bf16, see arx_tc2.cu
              if (nvalid < 128) {           // pad query columns of the last tile: P = 0, so their accumulator columns stay exactly 0
#pragma unroll
                for (int j = 0; j < 128; ++j) r[j] = j < nvalid ? r[j] : 0u;
              }
            }
            const uint64_t zz = pack2(zinv, zinv);
            if (trc) TRACEN(1 + g, k, 4);
            mbar_wait_wd(&bars[B_P_EMPTY + g], (kb & 1) ^ 1);
            if (trc) TRACEN(1 + g, k, 5);
#pragma unroll
            for (int c16 = 0; c16 < 16; ++c16) {
              uint32_t hh[4];
#pragma unroll
              for (int q = 0; q < 4; ++q) {
                const uint64_t m = mul2(pack2u(r[c16 * 8 + 2 * q], r[c16 * 8 + 2 * q + 1]), zz);
                hh[q] = __byte_perm((uint32_t)m, (uint32_t)(m >> 32), 0x7632);
              }
              *reinterpret_cast<uint4 *>(prow + (c16 >> 3) * 16384 + (((c16 & 7) ^ (s & 7)) << 4)) = make_uint4(hh[0], hh[1], hh[2], hh[3]);
            }
            fence_proxy_async_smem();
            mbar_arrive(&bars[B_P_FULL + g]);
            if (trc) TRACEN(1 + g, k, 6);
            ++kb;
          }
        }
      }
    }
  } else {
    // ---------------- epilogue warps: thread == TMEM lane == output dimension d (mode 0) or head column l (mode 1)
    // The accumulator already holds proto - Vq (mode 0) or sum_s P.Uc - head table (mode 1): see the selection MMA.  Earlier
    // versions rebuilt Vq here from a per-frame table in global memory: even with the loads of a chunk batched the register
    // budget kept only a few in flight, a tile took 18-41 K clk (timeline trace, tools/trace_tcn.py) and stalled the next tile
    // pair's first MMA2 behind O_EMPTY -- at N=496 the epilogue cost as much as the sixteen steps of the unit; a thread-private
    // table in local memory was slower still (L1 is what shared memory leaves: nothing).
    setmaxnreg_inc<152>();
    const int quad = warp & 3;
    const int d = quad * 32 + lane;
    const uint32_t lane_base = (uint32_t)(quad * 32) << 16;
    int ke = 0;
    for (int ui = 0; ui < my_units; ++ui) {
      const int u = blockIdx.x + ui * gridDim.x;
      const int win = head ? u : u / p.way;                    // output row
      uint64_t acc2[4] = {0ull, 0ull, 0ull, 0ull};
      for (int qp = 0; qp < nqp; ++qp, ++ke) {
        const int nw = min(2, nq - 2 * qp);
        for (int w = 0; w < 2; ++w) {
          mbar_wait_wd(&bars[B_O_FULL + w], ke & 1);
          if (w >= nw) { mbar_arrive(&bars[B_O_EMPTY + w]); continue; }
          tc_fence_after();
          const int q0 = (2 * qp + w) * 128;
#pragma unroll 1
          for (int ch = 0; ch < 4; ch += 2) {
            uint32_t r[32], r2[32];
            tmem_ld32(TM_O + lane_base + w * 128 + ch * 32, r);
            tmem_ld32(TM_O + lane_base + w * 128 + ch * 32 + 32, r2);
            tmem_ld_wait();
            if (ch == 2) { tc_fence_before(); mbar_arrive(&bars[B_O_EMPTY + w]); }
            if (!head) {
#pragma unroll
              for (int jj = 0; jj < 32; jj += 2) {
                const uint64_t a = pack2u(r[jj], r[jj + 1]), b = pack2u(r2[jj], r2[jj + 1]);
                acc2[(jj >> 1) & 1] = fma2(a, a, acc2[(jj >> 1) & 1]);
                acc2[2 + ((jj >> 1) & 1)] = fma2(b, b, acc2[2 + ((jj >> 1) & 1)]);
              }
            } else if (d < p.L) {
#pragma unroll
              for (int jj = 0; jj < 64; ++jj) {
                const int q = q0 + ch * 32 + jj;
                if (q < p.N) {
                  const float df = -__uint_as_float(jj < 32 ? r[jj & 31] : r2[jj & 31]);
                  const int col = q * p.L + d;
                  if (p.y_img) {
                    uint8_t *dst = reinterpret_cast<uint8_t *>(p.y_img) + ((size_t)(win >> 7) * p.y_nk + (col >> 6)) * (128 * 128);
                    *reinterpret_cast<__half *>(dst + sw128_offset(win & 127, col & 63)) = __float2half_rn(df);
                  } else {
                    p.y[(size_t)win * p.N * p.L + col] = df;
                  }
                }
              }
            }
          }
        }
      }
      if (!head) {
        float al, ah;
        unpack2(add2(add2(acc2[0], acc2[1]), add2(acc2[2], acc2[3])), al, ah);
        float run = al + ah;
#pragma unroll
        for (int o = 16; o; o >>= 1) run += __shfl_xor_sync(0xffffffffu, run, o);
        if (lane == 0) p.partial[(size_t)u * 4 + quad] = run;
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 3) { tc_fence_after(); tmem_dealloc(tmem, 512); }
}

// ---- operand image builders (tiled) ---------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t pack_half2(float lo, float hi) {
  __half2 h = __floats2half2_rn(lo, hi);
  return *reinterpret_cast<uint32_t *>(&h);
}
__device__ __forceinline__ uint32_t pack_bf162(float lo, float hi) {
  __nv_bfloat162 h = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t *>(&h);
}

// Query K tiles: one warp per tuple row; K = LayerNorm(sum_p Gk_p[frame_p]) * alpha -> fp16, K-major SW128.  grid (n_win, nq)
__global__ void __launch_bounds__(256) k_prep_kq_tiles(const float *__restrict__ G, const uint32_t *__restrict__ tup, const float *__restrict__ ln_g,
                                                       const float *__restrict__ ln_b, __half *__restrict__ img, int T, int c, int N, int nq, int ldg,
                                                       float alpha) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const size_t seq = blockIdx.x;
  const int qt = blockIdx.y;
  uint8_t *out = reinterpret_cast<uint8_t *>(img) + (seq * nq + qt) * IMG_BYTES;
  const int d0 = lane * 4;
  const float4 g = *reinterpret_cast<const float4 *>(ln_g + d0);
  const float4 be = *reinterpret_cast<const float4 *>(ln_b + d0);
  for (int r = warp; r < 128; r += 8) {
    const int q = qt * 128 + r;
    uint2 packed = make_uint2(0u, 0u);
    if (q < N) {
      const uint32_t tp = tup[q];
      float4 k = make_float4(0, 0, 0, 0);
      for (int pp = 0; pp < c; ++pp) {
        const int fr = (tp >> (8 * pp)) & 0xff;
        const float4 a = *reinterpret_cast<const float4 *>(G + (seq * T + fr) * (size_t)ldg + pp * DD + d0);
        k.x += a.x; k.y += a.y; k.z += a.z; k.w += a.w;
      }
      float sm = k.x + k.y + k.z + k.w;
#pragma unroll
      for (int o = 16; o; o >>= 1) sm += __shfl_xor_sync(0xffffffffu, sm, o);
      const float mean = sm / DD;
      const float4 dl = make_float4(k.x - mean, k.y - mean, k.z - mean, k.w - mean);
      float qq = dl.x * dl.x + dl.y * dl.y + dl.z * dl.z + dl.w * dl.w;
#pragma unroll
      for (int o = 16; o; o >>= 1) qq += __shfl_xor_sync(0xffffffffu, qq, o);
      const float rstd = 1.0f / sqrtf(qq / DD + 1e-5f);
      packed.x = pack_half2((dl.x * rstd * g.x + be.x) * alpha, (dl.y * rstd * g.y + be.y) * alpha);
      packed.y = pack_half2((dl.z * rstd * g.z + be.z) * alpha, (dl.w * rstd * g.w + be.w) * alpha);
    }
    *reinterpret_cast<uint2 *>(out + (d0 >> 6) * SUB_BYTES + sw128_offset(r, d0 & 63)) = packed;
  }
}

// Support K tiles from fp32 ks (way, N, D): rows = s, cols = d.  grid (way, ns)
__global__ void __launch_bounds__(256) k_prep_kc_tiles(const float *__restrict__ ks, __half *__restrict__ img, int N, int ns) {
  const size_t cls = blockIdx.x;
  const int st = blockIdx.y;
  const float *k = ks + cls * (size_t)N * DD;
  uint8_t *out = reinterpret_cast<uint8_t *>(img) + (cls * ns + st) * IMG_BYTES;
  for (int e = threadIdx.x; e < 128 * 16; e += 256) {
    const int dc = e & 15, r = e >> 4, s = st * 128 + r;
    uint4 pk = make_uint4(0, 0, 0, 0);
    if (s < N) {
      const float4 x0 = *reinterpret_cast<const float4 *>(k + (size_t)s * DD + dc * 8);
      const float4 x1 = *reinterpret_cast<const float4 *>(k + (size_t)s * DD + dc * 8 + 4);
      pk.x = pack_half2(x0.x, x0.y); pk.y = pack_half2(x0.z, x0.w); pk.z = pack_half2(x1.x, x1.y); pk.w = pack_half2(x1.z, x1.w);
    }
    const int d0 = dc * 8;
    *reinterpret_cast<uint4 *>(out + (d0 >> 6) * SUB_BYTES + sw128_offset(r, d0 & 63)) = pk;
  }
}

// Support V^T tiles (bf16): rows = d, cols = support tuple of tile st (zero beyond N).  grid (way, ns)
__global__ void __launch_bounds__(256) k_prep_vct_tiles(const float *__restrict__ vs, __half *__restrict__ img, int N, int ns) {
  const size_t cls = blockIdx.x;
  const int st = blockIdx.y;
  const float *v = vs + cls * (size_t)N * DD;
  uint8_t *out = reinterpret_cast<uint8_t *>(img) + (cls * ns + st) * IMG_BYTES;
  for (int e = threadIdx.x; e < DD * 16; e += 256) {
    const int d = e & 127, sc = e >> 7;          // consecutive threads -> consecutive d (coalesced reads)
    float x[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int s = st * 128 + sc * 8 + i;
      x[i] = s < N ? v[(size_t)s * DD + d] : 0.f;
    }
    uint4 pk;
    pk.x = pack_bf162(x[0], x[1]); pk.y = pack_bf162(x[2], x[3]); pk.z = pack_bf162(x[4], x[5]); pk.w = pack_bf162(x[6], x[7]);
    const int s0 = sc * 8;
    *reinterpret_cast<uint4 *>(out + (s0 >> 6) * SUB_BYTES + sw128_offset(d, s0 & 63)) = pk;
  }
}

// Head operand Uc tiles (bf16): rows l < L hold sum_d Wdr[l][d].Vc[s][d], rows >= L are zero.  grid (way, ns), 128 threads (one per s).
// LMAX >= L: the rows one thread keeps in registers (32 for T <= 32, 64 for T <= 64; the 32-row instance is the one T <= 32 always ran)
template <int LMAX>
__global__ void __launch_bounds__(128) k_prep_uc_tiles(const float *__restrict__ vs, const float *__restrict__ dr_w, __half *__restrict__ img, int N,
                                                       int ns, int L) {
  extern __shared__ float w_s[];                 // [L][128]
  for (int e = threadIdx.x; e < L * 128; e += 128) w_s[e] = dr_w[e];
  __syncthreads();
  const size_t cls = blockIdx.x;
  const int st = blockIdx.y, r = threadIdx.x, s = st * 128 + r;
  uint8_t *out = reinterpret_cast<uint8_t *>(img) + (cls * ns + st) * IMG_BYTES;
  float acc[LMAX];
#pragma unroll
  for (int l = 0; l < LMAX; ++l) acc[l] = 0.f;
  if (s < N) {
    const float4 *v = reinterpret_cast<const float4 *>(vs + (cls * N + s) * DD);
    for (int d4 = 0; d4 < 32; ++d4) {
      const float4 x = v[d4];
#pragma unroll
      for (int l = 0; l < LMAX; ++l) {
        if (l < L) {
          const float4 ww = *reinterpret_cast<const float4 *>(&w_s[l * 128 + d4 * 4]);
          acc[l] += x.x * ww.x + x.y * ww.y + x.z * ww.z + x.w * ww.w;
        }
      }
    }
  }
  // column r of the tile for every row: rows l < L carry values, rows L..127 zero
  for (int l = 0; l < 128; ++l) {
    float val = 0.f;
#pragma unroll
    for (int m = 0; m < LMAX; ++m) if (m == l) val = acc[m];
    *reinterpret_cast<__nv_bfloat16 *>(out + (r >> 6) * SUB_BYTES + sw128_offset(l, r & 63)) = __float2bfloat16_rn(l < L ? val : 0.f);
  }
}

// Selection operand A of one window: MINUS its per-frame table as hi + lo fp16 halves, K-major SW128 sub-tiles of 64 columns.
// Column h*cT + p*T + t holds -(hi | lo)(tab[(win*T + t)*ld + off + p*pstride + row]); rows >= n_rows and columns >= 2cT are zero.
// grid (n_win, nsel), 256 threads: thread = (row, 8-column chunk).
__global__ void __launch_bounds__(256) k_prep_vq_img(const float *__restrict__ tab, int ld, int off, int pstride, int n_rows, int T, int c,
                                                     int nsel, __half *__restrict__ img) {
  const size_t win = blockIdx.x;
  const int sub = blockIdx.y, cT = c * T;
  uint8_t *out = reinterpret_cast<uint8_t *>(img) + (win * nsel + sub) * SUB_BYTES;
  for (int e = threadIdx.x; e < 128 * 8; e += 256) {
    const int row = e & 127, ch = e >> 7;             // consecutive threads -> consecutive rows (coalesced table reads)
    uint32_t pk[4];
#pragma unroll
    for (int i2 = 0; i2 < 4; ++i2) {
      float v[2];
#pragma unroll
      for (int i = 0; i < 2; ++i) {
        const int col = sub * 64 + ch * 8 + i2 * 2 + i;
        const int hh = col / cT, pt = col - hh * cT;
        float x = 0.f;
        if (hh < 2 && row < n_rows) {
          const int pp = pt / T, t = pt - pp * T;
          const float f = -__ldg(tab + (win * T + t) * (size_t)ld + off + pp * pstride + row);
          const float hi = __half2float(__float2half_rn(f));
          x = hh == 0 ? hi : f - hi;
        }
        v[i] = x;
      }
      pk[i2] = pack_half2(v[0], v[1]);
    }
    *reinterpret_cast<uint4 *>(out + sw128_offset(row, ch * 8)) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
  }
}

// Selection operand B of one query tile: Sel[q][h*cT + p*T + frame_p(q)] = 1 for both halves h, rows of pad tuples are zero.
// grid (nq, nsel), 256 threads.
__global__ void __launch_bounds__(256) k_prep_sel_tiles(const uint32_t *__restrict__ tup, int N, int T, int c, int nsel, __half *__restrict__ img) {
  const int qt = blockIdx.x, sub = blockIdx.y, cT = c * T;
  uint8_t *out = reinterpret_cast<uint8_t *>(img) + ((size_t)qt * nsel + sub) * SUB_BYTES;
  for (int e = threadIdx.x; e < 128 * 8; e += 256) {
    const int row = e >> 3, ch = e & 7, q = qt * 128 + row;
    const uint32_t tp = q < N ? tup[q] : 0u;
    uint32_t pk[4];
#pragma unroll
    for (int i2 = 0; i2 < 4; ++i2) {
      float v[2];
#pragma unroll
      for (int i = 0; i < 2; ++i) {
        const int col = sub * 64 + ch * 8 + i2 * 2 + i;
        const int hh = col / cT, pt = col - hh * cT;
        const int pp = pt / T, t = pt - pp * T;
        v[i] = (q < N && hh < 2 && (int)((tp >> (8 * pp)) & 0xffu) == t) ? 1.f : 0.f;
      }
      pk[i2] = pack_half2(v[0], v[1]);
    }
    *reinterpret_cast<uint4 *>(out + sw128_offset(row, ch * 8)) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
  }
}

// Head table: UAB[row][p*LP + l] = sum_d Wdr[l][d] . Gv_p[row][d] (+ bdr[l] for p == 0); rows = n_win*T, pair tuples, L <= LP
// columns per frame part (LP = 32 for T <= 32, 64 for T <= 64: arx_tcn_head_cols), row stride 2*LP.
// Persistent over groups of 256 / (2*LP) rows; Wdr is staged TRANSPOSED in shared memory once per CTA (the first version ran one CTA per
// row with every thread walking its own weight row in global memory: 32 sectors per load, 1.9 ms for 65 536 rows -- 15 % of a T=32 score).
// Same summation order as before (bias first, d ascending): bit-identical.
template <int LP>
__global__ void __launch_bounds__(256) k_head_uab(const float *__restrict__ G, int ldg, int voff, const float *__restrict__ dr_w,
                                                  const float *__restrict__ dr_b, float *__restrict__ uab, int64_t rows, int L) {
  constexpr int RG = 256 / (2 * LP);                // rows per group: one thread per (row, frame part, column)
  __shared__ float wT[DD][LP + 1];                  // wT[d][l], padded: the transposing store is conflict-free too
  __shared__ __align__(16) float g_s[RG][2 * DD];
  const int tid = threadIdx.x;
  for (int e = tid; e < LP * DD; e += 256) {
    const int l = e / DD, dd = e - l * DD;
    wT[dd][l] = l < L ? dr_w[(size_t)l * DD + dd] : 0.f;
  }
  const int slot = tid / (2 * LP), pp = (tid / LP) & 1, l = tid % LP;
  const float bias = (pp == 0 && l < L) ? dr_b[l] : 0.f;
  for (int64_t r0 = (int64_t)blockIdx.x * RG; r0 < rows; r0 += (int64_t)gridDim.x * RG) {
    __syncthreads();                                // the previous group's rows have been consumed (first pass: wT is complete)
    if (tid < RG * 64 && r0 + (tid >> 6) < rows)    // RG rows x 256 floats: one float4 per thread, coalesced
      *reinterpret_cast<float4 *>(&g_s[tid >> 6][(tid & 63) * 4]) = *reinterpret_cast<const float4 *>(G + (r0 + (tid >> 6)) * ldg + voff + (tid & 63) * 4);
    __syncthreads();
    if (r0 + slot < rows) {
      float a = bias;
      if (l < L) {
#pragma unroll 8
        for (int dd = 0; dd < DD; ++dd) a = fmaf(wT[dd][l], g_s[slot][pp * DD + dd], a);
      }
      uab[(r0 + slot) * (2 * LP) + pp * LP + l] = a;
    }
  }
}

__global__ void k_pack_tuples(const int32_t *__restrict__ tuples, uint32_t *__restrict__ out, int N, int c) {
  const int q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= N) return;
  uint32_t v = 0;
  for (int pp = 0; pp < c; ++pp) v |= (uint32_t)tuples[q * c + pp] << (8 * pp);
  out[q] = v;
}

__global__ void k_finish_n(const float *__restrict__ partial, float *__restrict__ logits, int32_t *__restrict__ chosen, int64_t n_win, int way,
                           int N) {
  const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= n_win) return;
  float best = -INFINITY;
  int bi = 0;
  for (int c = 0; c < way; ++c) {
    const float4 t = *reinterpret_cast<const float4 *>(partial + (b * way + c) * 4);
    const float lg = -(((t.x + t.y) + (t.z + t.w)) / (float)N);
    logits[b * way + c] = lg;
    if (lg > best) { best = lg; bi = c; }        // strict '>': the first maximum wins (torch.argmax, model.py:323)
  }
  if (chosen) chosen[b] = bi;
}

}  // namespace

bool arx_tcn_supported(const arx_handle *h, const ArxTransformer &tr) {
  return h->D == DD && h->T <= 255 && tr.c >= 2 && tr.c <= 3;
}
bool arx_tcn_head_supported(const arx_handle *h, const ArxTransformer &tr) { return tr.c == 2 && h->T <= 64; }
int arx_tcn_head_cols(int T) { return T <= 32 ? 32 : 64; }
// exp2 without a shift is only safe inside the overflow bound on the LayerNorm affine (SURVEY 7.2-1); past it the ROWMAX
// variant runs.  Only force_path = 2 gets there: by default weights past the tighter accuracy bound score on the fp32 kernels.
bool arx_tcn_needs_rowmax(const ArxTransformer &tr) { return !(tr.softmax_bound * ARX_SOFTMAX_LOG2E < 100.0f); }

int arx_tcn_prep_support(arx_handle *h, ArxTransformer &tr, int way, bool with_head, cudaStream_t st) {
  const int ns = tr.Npad / 128;
  const size_t bytes = (size_t)h->way_cap * ns * IMG_BYTES;
  if (!tr.kc_tiles) {
    ARX_CUDA(h, cudaMalloc(reinterpret_cast<void **>(&tr.kc_tiles), bytes));
    ARX_CUDA(h, cudaMalloc(reinterpret_cast<void **>(&tr.vct_tiles), bytes));
  }
  if (!tr.tup_packed) {
    ARX_CUDA(h, cudaMalloc(reinterpret_cast<void **>(&tr.tup_packed), (size_t)tr.N * sizeof(uint32_t)));
    k_pack_tuples<<<(tr.N + 127) / 128, 128, 0, st>>>(tr.tuples, tr.tup_packed, tr.N, tr.c);
    ARX_LAUNCH_CHECK(h);
    const int nsel = (2 * tr.c * h->T + 63) / 64;
    ARX_CUDA(h, cudaMalloc(reinterpret_cast<void **>(&tr.sel_tiles), (size_t)ns * nsel * SUB_BYTES));
    k_prep_sel_tiles<<<dim3(ns, nsel), 256, 0, st>>>(tr.tup_packed, tr.N, h->T, tr.c, nsel, tr.sel_tiles);
    ARX_LAUNCH_CHECK(h);
  }
  k_prep_kc_tiles<<<dim3(way, ns), 256, 0, st>>>(tr.ks, tr.kc_tiles, tr.N, ns);
  ARX_LAUNCH_CHECK(h);
  k_prep_vct_tiles<<<dim3(way, ns), 256, 0, st>>>(tr.vs, tr.vct_tiles, tr.N, ns);
  ARX_LAUNCH_CHECK(h);
  if (with_head) {
    if (!tr.uc_tiles) ARX_CUDA(h, cudaMalloc(reinterpret_cast<void **>(&tr.uc_tiles), bytes));
    auto kern = arx_tcn_head_cols(h->T) == 32 ? k_prep_uc_tiles<32> : k_prep_uc_tiles<64>;
    kern<<<dim3(way, ns), 128, h->T * 128 * sizeof(float), st>>>(tr.vs, h->dr_w, tr.uc_tiles, tr.N, ns, h->T);
    ARX_LAUNCH_CHECK(h);
  }
  return ARX_OK;
}

int arx_tcn_prep_query(arx_handle *h, const ArxTransformer &tr, const float *G, int ldg, int64_t n_win, __half *kq_tiles, cudaStream_t st) {
  const float alpha = ARX_SOFTMAX_LOG2E / sqrtf((float)h->D);
  const int nq = tr.Npad / 128;
  for (int64_t b0 = 0; b0 < n_win; b0 += 32768) {
    const int64_t nb = std::min<int64_t>(32768, n_win - b0);
    k_prep_kq_tiles<<<dim3((unsigned)nb, nq), 256, 0, st>>>(G + b0 * h->T * ldg, tr.tup_packed, tr.ln_g, tr.ln_b,
                                                           kq_tiles + (size_t)b0 * nq * 128 * DD, h->T, tr.c, tr.N, nq, ldg, alpha);
    ARX_LAUNCH_CHECK(h);
  }
  return ARX_OK;
}

static int tcn_launch(arx_handle *h, const ArxTransformer &tr, AttnNParams &p, int n_units, cudaStream_t st) {
  if (p.same_window && p.cls_stride) return arx_fail(h, ARX_ERR_INVALID, "tiled attention kernel: same_window and episode mode do not combine");
  const int grid = n_units < h->sm_count ? n_units : h->sm_count;
  // two regions: a head launch may run beside a main launch on another stream (streaming path)
  const size_t zhalf = (size_t)h->sm_count * 2 * 2 * 2 * tr.Npad, zbytes = 2 * zhalf * sizeof(float);
  if (h->zscratch_bytes < zbytes) {
    ARX_CUDA(h, cudaDeviceSynchronize());
    cudaFree(h->zscratch);
    h->zscratch = nullptr;
    h->zscratch_bytes = 0;
    ARX_CUDA(h, cudaMalloc(reinterpret_cast<void **>(&h->zscratch), zbytes));
    h->zscratch_bytes = zbytes;
  }
  p.zscratch = h->zscratch + (p.mode == 1 ? zhalf : 0);
  p.trace = h->trace_sel == 1 ? h->trace_buf : nullptr;
  p.free_a = h->tcn_free_a;
  p.poly = (h->tcn_poly && p.ns >= 8) ? 1 : 0;      // measured on B200: +3.4 % at N=4960 (MUFU-bound pass), -5 % at N=496 (latency-bound)
  if (!h->tcn_diag) {
    ARX_CUDA(h, cudaMalloc(reinterpret_cast<void **>(&h->tcn_diag), 8 * sizeof(int)));
    ARX_CUDA(h, cudaMemset(h->tcn_diag, 0, 8 * sizeof(int)));
  }
  p.diag = h->tcn_diag;
  const bool rowmax = arx_tcn_needs_rowmax(tr);
  auto kern = rowmax ? k_attn_tcn<true> : k_attn_tcn<false>;
  { const int rc_ = arx_func_smem(h, kern, (int)SMEM_BYTES); if (rc_) return rc_; }
  kern<<<grid, NTHREADS, SMEM_BYTES, st>>>(p);
  ARX_LAUNCH_CHECK(h);
  cudaStreamCaptureStatus cs_ = cudaStreamCaptureStatusNone;
  if (cudaStreamIsCapturing(st, &cs_) != cudaSuccess) { (void)cudaGetLastError(); cs_ = cudaStreamCaptureStatusNone; }
  if (getenv("ARX_TCN_CHECK") && cs_ == cudaStreamCaptureStatusNone) {            // bring-up: synchronise and report a watchdog record
    ARX_CUDA(h, cudaStreamSynchronize(st));
    int d[4] = {0, 0, 0, 0};
    ARX_CUDA(h, cudaMemcpy(d, h->tcn_diag, sizeof(d), cudaMemcpyDeviceToHost));
    if (d[0]) {
      cudaMemset(h->tcn_diag, 0, 8 * sizeof(int));
      return arx_fail(h, ARX_ERR_CUDA, "tiled attention kernel: mbarrier wait timed out (barrier %d, source line %d, parity %d, block %d, thread %d, mode %d, nq %d)",
                      d[0] & 0xff, (d[0] >> 8) & 0x3fffff, d[3], d[1], d[2], p.mode, p.nq);
    }
  }
  return ARX_OK;
}

static int tcn_nsel(const arx_handle *h, const ArxTransformer &tr) { return (2 * tr.c * h->T + 63) / 64; }

// selection operand A (minus the per-frame table, hi | lo) of n_win windows from a row-major table
static int tcn_prep_vq(arx_handle *h, const ArxTransformer &tr, const float *tab, int ld, int off, int pstride, int n_rows, int64_t n_win,
                       __half *vq, cudaStream_t st) {
  const int nsel = tcn_nsel(h, tr);
  for (int64_t b0 = 0; b0 < n_win; b0 += 32768) {
    const int64_t nb = std::min<int64_t>(32768, n_win - b0);
    k_prep_vq_img<<<dim3((unsigned)nb, nsel), 256, 0, st>>>(tab + (size_t)b0 * h->T * ld, ld, off, pstride, n_rows, h->T, tr.c, nsel,
                                                            vq + (size_t)b0 * nsel * 8192);
    ARX_LAUNCH_CHECK(h);
  }
  return ARX_OK;
}

// head table UAB of n_win windows (k_head_uab: rows = n_win*T, 2*LP columns) and selection operand A of the head from it
static int tcn_head_table(arx_handle *h, const ArxTransformer &tr, const float *G, int ldg, int64_t n_win, float *uab, __half *vq_ws, cudaStream_t st) {
  const int lp = arx_tcn_head_cols(h->T), rg = 256 / (2 * lp);
  const int64_t rows = n_win * h->T;
  auto kern = lp == 32 ? k_head_uab<32> : k_head_uab<64>;
  kern<<<(unsigned)std::min<int64_t>((rows + rg - 1) / rg, 4 * h->sm_count), 256, 0, st>>>(G, ldg, tr.c * h->D, h->dr_w, h->dr_b, uab, rows, h->T);
  ARX_LAUNCH_CHECK(h);
  return tcn_prep_vq(h, tr, uab, 2 * lp, 0, lp, h->T, n_win, vq_ws, st);
}

// squared-distance partials only (the streaming tail forms logits / argmax itself).  episodes: window w attends the pool
// classes [cls_base + w*way, cls_base + (w+1)*way) instead of classes [0, way)
int arx_tcn_attention_partial(arx_handle *h, const ArxTransformer &tr, const __half *kq_tiles, const float *G, int ldg, int64_t n_win, int way,
                              float *partial, __half *vq_ws, bool episodes, int64_t cls_base, cudaStream_t st) {
  int rc = tcn_prep_vq(h, tr, G, ldg, tr.c * h->D, h->D, 128, n_win, vq_ws, st);
  if (rc) return rc;
  AttnNParams p{};
  p.kq_img = kq_tiles; p.kc_img = tr.kc_tiles; p.vct_img = tr.vct_tiles; p.vq_img = vq_ws; p.sel_img = tr.sel_tiles; p.nsel = tcn_nsel(h, tr);
  p.partial = partial;
  p.n_win = (int)n_win; p.way = way; p.N = tr.N; p.T = h->T; p.c = tr.c; p.nq = p.ns = tr.Npad / 128;
  p.mode = 0;
  p.cls_base = episodes ? (int)cls_base : 0; p.cls_mod = episodes ? (int)n_win * way : way;
  return tcn_launch(h, tr, p, (int)n_win * way, st);
}

// logits (n_win, way) and chosen (n_win) of transformer `tr` from the query tiles; G = row-major per-frame projections
int arx_tcn_attention(arx_handle *h, const ArxTransformer &tr, const __half *kq_tiles, const float *G, int ldg, int64_t n_win, int way,
                      float *partial, float *logits, int32_t *chosen, __half *vq_ws, bool episodes, int64_t cls_base, cudaStream_t st) {
  int rc = arx_tcn_attention_partial(h, tr, kq_tiles, G, ldg, n_win, way, partial, vq_ws, episodes, cls_base, st);
  if (rc) return rc;
  k_finish_n<<<(unsigned)((n_win + 127) / 128), 128, 0, st>>>(partial, logits, chosen, n_win, way, tr.N);
  ARX_LAUNCH_CHECK(h);
  return ARX_OK;
}

// streaming: the head input of EVERY class of ONE window at once (y_all (way, N*L) fp32), so that it can run beside the main
// attention launch instead of after it; `iota` = device array 0..way-1
int arx_tcn_head_all(arx_handle *h, const ArxTransformer &tr, const __half *kq_tiles, const float *G, int ldg, int way, const int32_t *iota,
                     float *uab, float *y_all, __half *vq_ws, cudaStream_t st) {
  if (!arx_tcn_head_supported(h, tr) || !tr.uc_tiles) return arx_fail(h, ARX_ERR_INVALID, "tcn_head: pair tuples with T <= 64 only");
  int rc = tcn_head_table(h, tr, G, ldg, 1, uab, vq_ws, st);
  if (rc) return rc;
  AttnNParams p{};
  p.kq_img = kq_tiles; p.kc_img = tr.kc_tiles; p.vct_img = tr.uc_tiles; p.vq_img = vq_ws; p.sel_img = tr.sel_tiles; p.nsel = tcn_nsel(h, tr);
  p.chosen = iota;
  p.y = y_all; p.y_img = nullptr; p.y_nk = 0; p.L = h->T;
  p.n_win = way; p.way = 1; p.N = tr.N; p.T = h->T; p.c = tr.c; p.nq = p.ns = tr.Npad / 128;
  p.mode = 1; p.same_window = 1;
  return tcn_launch(h, tr, p, way, st);
}

// open-set head input y = dimensionality_reduction(diff of the winning class) (model.py:323-324,196), pair tuples.
// ep_way > 0: episode mode, window w's winner chosen[w] is class cls_base + w*ep_way + chosen[w] of the pool
int arx_tcn_head(arx_handle *h, const ArxTransformer &tr, const __half *kq_tiles, const float *G, int ldg, int64_t n_win, const int32_t *chosen,
                 float *uab, float *y, __half *y_img, int y_nk, __half *vq_ws, int ep_way, int64_t cls_base, cudaStream_t st) {
  if (!arx_tcn_head_supported(h, tr) || !tr.uc_tiles) return arx_fail(h, ARX_ERR_INVALID, "tcn_head: pair tuples with T <= 64 only");
  int rc = tcn_head_table(h, tr, G, ldg, n_win, uab, vq_ws, st);
  if (rc) return rc;
  AttnNParams p{};
  p.kq_img = kq_tiles; p.kc_img = tr.kc_tiles; p.vct_img = tr.uc_tiles; p.vq_img = vq_ws; p.sel_img = tr.sel_tiles; p.nsel = tcn_nsel(h, tr);
  p.chosen = chosen;
  p.y = y; p.y_img = y_img; p.y_nk = y_nk; p.L = h->T;
  p.n_win = (int)n_win; p.way = 1; p.N = tr.N; p.T = h->T; p.c = tr.c; p.nq = p.ns = tr.Npad / 128;
  p.mode = 1;
  p.cls_base = ep_way > 0 ? (int)cls_base : 0; p.cls_stride = ep_way > 0 ? ep_way : 0;
  return tcn_launch(h, tr, p, (int)n_win, st);
}

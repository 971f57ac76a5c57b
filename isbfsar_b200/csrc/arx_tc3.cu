// tcgen05 cross-attention + distance kernel, third generation (T=16 pair tuples, N=120).
// Same math / operand formats / slot order as arx_tc2.cu; the schedule changes again, following the timeline
// traces of the second generation (single P buffer chain, MMA2 queued behind look-ahead MMA1, shared-memory port):
//   * ONE MMA1 per class for BOTH windows of the group: S^T[s, (q of w0 | q of w1)] with N=256, so Kc is read
//     from shared memory once per two tiles and both softmax groups get their S tile from one accumulator;
//   * Kc is used exactly once per class, so it is single-buffered; the 32 KB it frees hold a second P buffer:
//     each softmax group owns its P buffer and its prototype accumulator -- nothing serialises on P any more;
//   * the two softmax groups are deliberately staggered by half a period, so that one group's TMEM loads, sums,
//     scaling and stores run under the other group's MUFU.EX2 stream (the co-limiting pipe);
//   * the epilogue keeps four independent fp32x2 accumulators.
// Shared memory: Kq 64 KB (both windows, laid out as one 256-row B operand) + Kc 32 KB + Vc^T 2 x 32 KB + P 2 x 32 KB.
// TMEM: S^T 256 columns (one accumulator), proto^T 2 x 128 columns.
#include "arx_internal.cuh"
#include "arx_ptx.cuh"
#include <utility>

namespace {
using namespace ptx;

constexpr int NTHREADS3 = 512;

constexpr uint32_t OFF_KQ = 0;                       // 64 KB: [sub0: w0 rows | w1 rows][sub1: w0 rows | w1 rows]
constexpr uint32_t OFF_KC = 2 * IMG_BYTES;           // 32 KB
constexpr uint32_t OFF_VCT = 3 * IMG_BYTES;          // 2 x 32 KB
constexpr uint32_t OFF_P = 5 * IMG_BYTES;            // 2 x 32 KB (one per softmax group / window slot)
constexpr uint32_t OFF_BAR = 7 * IMG_BYTES;
enum { B_FULL_KQ = 0, B_EMPTY_KQ = 1, B_FULL_KC = 2, B_EMPTY_KC = 3, B_FULL_VC = 4, B_EMPTY_VC = 6, B_S_FULL = 8, B_S_EMPTY = 9,
       B_P_FULL = 10, B_P_EMPTY = 12, B_O_FULL = 14, B_O_EMPTY = 16, B_XU = 18, B_COUNT = 20 };
constexpr uint32_t SMEM_BYTES = OFF_BAR + B_COUNT * 8 + 16 + 1024;

struct Attn3Params {
  const __half *kq_img, *kc_img, *vct_img;
  const float *G;
  float *partial;
  int n_win, way, ldg, voff;
  long long *trace;
  int stagger, token, gchunk;
  int ep;      // episode mode (train.py:110-120 call shape): every window has its OWN `way` classes at class index window*way + c; groups hold one window
};
#define ARX_TRACE_TILES 64
#define TRACE3(role, tile, k) do { if (p.trace && blockIdx.x == 0 && (tile) < ARX_TRACE_TILES) p.trace[(((role) * ARX_TRACE_TILES) + (tile)) * 8 + (k)] = clock64(); } while (0)

__device__ __forceinline__ uint32_t ex2_bits(uint32_t x) {
  uint32_t y;
  asm volatile("ex2.approx.ftz.f32 %0, %1;" : "=r"(y) : "r"(x));
  return y;
}

// exp2 of two pre-scaled scores on the FMA pipe instead of the MUFU (the co-limiting pipe): round-to-nearest split
// x = n + f with the 1.5*2^23 magic constant, 2^f on [-0.5, 0.5] by a degree-3 polynomial (max relative error
// 7.5e-5, far below the bf16 quantisation of P), exponent add by an integer shift-add.  |x| < 100 is guaranteed by
// the overflow bound on the LayerNorm affine checked at weight load (arx_tc_supported), which also holds under
// force_path = 2; by default the tighter accuracy bound (ARX_TC_ACCURACY_BOUND) keeps |x| far below it.
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

// one fp32x2 pair of the epilogue: columns Q, Q+1 (Q even) of chunk registers r; ACC selects one of four accumulators
template <int Q> __device__ __forceinline__ void epi_pair(const float (&a)[16], const uint64_t (&bb)[8], const uint32_t (&r)[32], uint64_t (&acc)[4]) {
  constexpr int I = arx_slot_i(Q), J = arx_slot_j(Q);
  static_assert(J % 2 == 0, "pairs start on an even j");
  uint64_t bj;
  if constexpr (J == I) bj = pack2(-a[I], __uint_as_float((uint32_t)(bb[J / 2] >> 32)));   // pad lane: a_i + (-a_i) == 0 == proto
  else bj = bb[J / 2];
  const uint64_t v = add2(pack2(a[I], a[I]), bj);
  const uint64_t d = sub2(v, pack2u(r[Q & 31], r[(Q & 31) + 1]));
  acc[(Q >> 1) & 3] = fma2(d, d, acc[(Q >> 1) & 3]);
}
template <int CH, int... Ks>
__device__ __forceinline__ void epi_chunk(const float (&a)[16], const uint64_t (&bb)[8], const uint32_t (&r)[32], uint64_t (&acc)[4],
                                          std::integer_sequence<int, Ks...>) {
  (epi_pair<CH * 32 + 2 * Ks>(a, bb, r, acc), ...);
}
template <int... Is> __device__ __forceinline__ void zero_pads(uint32_t (&r)[128], std::integer_sequence<int, Is...>) {
  ((r[arx_slot_row_start(2 * Is)] = 0u), ...);
}

// POLY: every POLY-th register pair of a score tile takes the polynomial exp2 (0 = all on the MUFU)
template <int POLY>
__global__ void __launch_bounds__(NTHREADS3, 1) k_attn_tc3(const Attn3Params p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t *smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint64_t *bars = reinterpret_cast<uint64_t *>(smem + OFF_BAR);
  uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(smem + OFF_BAR + B_COUNT * 8);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // this CTA's window groups: g = blockIdx.x, blockIdx.x + gridDim.x, ...; a group is 2 windows (the last may be 1)
  const int GW = p.ep ? 1 : 2;                     // windows per group
  const int n_groups = (p.n_win + GW - 1) / GW;
  const int my_groups = n_groups > (int)blockIdx.x ? (n_groups - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x : 0;
  auto group_nw = [&](int gi) { return min(GW, p.n_win - ((int)blockIdx.x + gi * (int)gridDim.x) * GW); };

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
      if (elect_one()) {            // producer: class operands -- Kc single-buffered (one MMA1 per class), Vc^T in a 2-stage ring
        int k = 0;
        for (int gi = 0; gi < my_groups; ++gi) {
          const size_t cbase = p.ep ? (size_t)(blockIdx.x + gi * gridDim.x) * p.way : 0;
          for (int c = 0; c < p.way; ++c, ++k) {
            const uint8_t *kc = reinterpret_cast<const uint8_t *>(p.kc_img) + (cbase + c) * IMG_BYTES;
            const uint8_t *vc = reinterpret_cast<const uint8_t *>(p.vct_img) + (cbase + c) * IMG_BYTES;
            mbar_wait(&bars[B_EMPTY_KC], (k & 1) ^ 1);
            mbar_arrive_expect_tx(&bars[B_FULL_KC], IMG_BYTES);
            bulk_g2s(smem + OFF_KC, kc, SUB_BYTES, &bars[B_FULL_KC]);
            bulk_g2s(smem + OFF_KC + SUB_BYTES, kc + SUB_BYTES, SUB_BYTES, &bars[B_FULL_KC]);
            const int st = k & 1;
            mbar_wait(&bars[B_EMPTY_VC + st], ((k >> 1) & 1) ^ 1);
            mbar_arrive_expect_tx(&bars[B_FULL_VC + st], IMG_BYTES);
            bulk_g2s(smem + OFF_VCT + st * IMG_BYTES, vc, SUB_BYTES, &bars[B_FULL_VC + st]);
            bulk_g2s(smem + OFF_VCT + st * IMG_BYTES + SUB_BYTES, vc + SUB_BYTES, SUB_BYTES, &bars[B_FULL_VC + st]);
          }
        }
      }
    } else if (warp == 2) {
      if (elect_one()) {            // producer: the group's Kq images, interleaved into one 256-row K-major operand
        for (int gi = 0; gi < my_groups; ++gi) {
          const int nw = group_nw(gi), g = blockIdx.x + gi * gridDim.x;
          mbar_wait(&bars[B_EMPTY_KQ], (gi & 1) ^ 1);
          mbar_arrive_expect_tx(&bars[B_FULL_KQ], nw * IMG_BYTES);
          for (int w = 0; w < nw; ++w) {
            const uint8_t *src = reinterpret_cast<const uint8_t *>(p.kq_img) + (size_t)(g * GW + w) * IMG_BYTES;
            bulk_g2s(smem + OFF_KQ + w * SUB_BYTES, src, SUB_BYTES, &bars[B_FULL_KQ]);                              // d 0..63
            bulk_g2s(smem + OFF_KQ + 2 * SUB_BYTES + w * SUB_BYTES, src + SUB_BYTES, SUB_BYTES, &bars[B_FULL_KQ]);  // d 64..127
          }
          // Kq is single-buffered, so the next group's load is exposed at the group boundary: have it wait in L2, not in HBM
          if (gi + 1 < my_groups) {
            const int nwn = group_nw(gi + 1);
            bulk_prefetch_l2(reinterpret_cast<const uint8_t *>(p.kq_img) + (size_t)((g + gridDim.x) * GW) * IMG_BYTES, nwn * IMG_BYTES);
          }
        }
      }
    } else if (warp == 1) {
      if (elect_one()) {            // MMA1 issuer: one N=256 (or 128 for a single-window tail group) MMA sequence per class
        constexpr uint64_t DESC_K = smem_desc_sw128(16, 1024);
        const uint32_t sbase = smem_u32(smem);
        int k = 0;
        for (int gi = 0; gi < my_groups; ++gi) {
          const int nw = group_nw(gi);
          const uint32_t idesc = nw == 2 ? idesc_f16(128, 256, 0, 0) : idesc_f16(128, 128, 0, 0);
          for (int c = 0; c < p.way; ++c, ++k) {
            if (c == 0) mbar_wait(&bars[B_FULL_KQ], gi & 1);
            mbar_wait(&bars[B_FULL_KC], k & 1);
            mbar_wait(&bars[B_S_EMPTY], (k & 1) ^ 1);
            tc_fence_after();
            TRACE3(0, k, 0);
#pragma unroll
            for (int kk = 0; kk < 8; ++kk) {
              const uint32_t aoff = (kk >> 2) * SUB_BYTES + (kk & 3) * 32;
              const uint32_t boff = (kk >> 2) * (2 * SUB_BYTES) + (kk & 3) * 32;
              mma_f16_ss(TM_S, smem_desc_at(DESC_K, sbase + OFF_KC + aoff), smem_desc_at(DESC_K, sbase + OFF_KQ + boff), idesc, kk > 0);
            }
            mma_commit(&bars[B_S_FULL]);
            mma_commit(&bars[B_EMPTY_KC]);
            if (c == p.way - 1) mma_commit(&bars[B_EMPTY_KQ]);
          }
        }
      }
    } else {
      if (elect_one()) {            // MMA2 issuer: proto^T = Vc^T . P for each window of the class
        constexpr uint64_t DESC_K = smem_desc_sw128(16, 1024);
        constexpr uint64_t DESC_MN = smem_desc_sw128(16384, 1024);
        constexpr uint32_t IDESC2 = idesc_bf16(128, 128, 0, 1);
        const uint32_t sbase = smem_u32(smem);
        int k = 0;
        for (int gi = 0; gi < my_groups; ++gi) {
          const int nw = group_nw(gi);
          for (int c = 0; c < p.way; ++c, ++k) {
            const int st = k & 1;
            mbar_wait(&bars[B_FULL_VC + st], (k >> 1) & 1);
            for (int w = 0; w < nw; ++w) {
              mbar_wait(&bars[B_P_FULL + w], k & 1);
              mbar_wait(&bars[B_O_EMPTY + w], (k & 1) ^ 1);
              tc_fence_after();
              TRACE3(0, k, 1 + w);
#pragma unroll
              for (int kk = 0; kk < 8; ++kk) {
                const uint32_t off = (kk >> 2) * SUB_BYTES + (kk & 3) * 32;
                mma_f16_ss(TM_O + w * 128, smem_desc_at(DESC_K, sbase + OFF_VCT + st * IMG_BYTES + off),
                           smem_desc_at(DESC_MN, sbase + OFF_P + w * IMG_BYTES + kk * 2048), IDESC2, kk > 0);
              }
              mma_commit(&bars[B_O_FULL + w]);
              mma_commit(&bars[B_P_EMPTY + w]);
            }
            // barriers of an absent second window keep their phase in step
            if (nw == 1) {          // sequenced like a real tile (see the parity note in the softmax branch)
              mbar_wait(&bars[B_O_EMPTY + 1], (k & 1) ^ 1);
              mbar_arrive(&bars[B_O_FULL + 1]);
              mbar_arrive(&bars[B_P_EMPTY + 1]);
            }
            mma_commit(&bars[B_EMPTY_VC + st]);
          }
        }
      }
    }
  } else if (warp < 12) {
    // ---------------- softmax group g owns window slot g of every group: S^T columns [128g, 128g+128), P buffer g
    setmaxnreg_inc<160>();
    const int g = (warp - 4) >> 2, quad = warp & 3;
    const int s = quad * 32 + lane;
    const uint32_t lane_base = (uint32_t)(quad * 32) << 16;
    uint8_t *prow = smem + OFF_P + g * IMG_BYTES + (s >> 3) * 1024 + (s & 7) * 128;
    const bool tr = (threadIdx.x == 128 + g * 128);
    int k = 0;
    for (int gi = 0; gi < my_groups; ++gi) {
      const int nw = group_nw(gi);
      for (int c = 0; c < p.way; ++c, ++k) {
        if (tr) TRACE3(1 + g, k, 0);
        mbar_wait(&bars[B_S_FULL], k & 1);
        tc_fence_after();
        if (tr) TRACE3(1 + g, k, 1);
        if (c == 0 && g == 1) {     // stagger: group 1 runs half a period behind group 0 (re-armed at every window group: the Kq reload resynchronises them), so that one
          const long long t0 = clock64();    // group's TMEM loads / sums / stores overlap the other group's MUFU stream
          while (clock64() - t0 < p.stagger) {}
        }
        if (g >= nw) {              // single-window tail group: slot 1 has no tile, but its barriers must keep their phase
          mbar_arrive(&bars[B_S_EMPTY]);
          // take the MUFU token in turn like a real tile: an mbarrier parity wait cannot tell phase k from k+2, so
          // no barrier may ever run two phases ahead of its waiter
          if (p.token) mbar_wait(&bars[B_XU + 0], k & 1);
          mbar_arrive(&bars[B_XU + 1]);
          mbar_arrive(&bars[B_P_FULL + 1]);
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
        // MUFU token: the groups take turns on the exp phase (group 0 of class k, group 1 of class k, group 0 of k+1, ...)
        // so that each one's loads / sums / scaling / stores run under the other's MUFU stream instead of beside it
        if (p.token) {
          if (g == 0) { if (k > 0) mbar_wait(&bars[B_XU + 1], (k - 1) & 1); }
          else mbar_wait(&bars[B_XU + 0], k & 1);
        }
        if (tr) TRACE3(1 + g, k, 2);
#pragma unroll
        for (int j = 0; j < 128; j += 2) {
          if (POLY > 0 && (j >> 1) % (POLY > 0 ? POLY : 1) == 0) exp2_poly2(r[j], r[j + 1]);
          else { r[j] = ex2_bits(r[j]); r[j + 1] = ex2_bits(r[j + 1]); }
        }
        mbar_arrive(&bars[B_XU + g]);
        zero_pads(r, std::make_integer_sequence<int, 8>{});
        // The sums stay BEHIND the whole MUFU stream (volatile adds): a warp issues in order, and an add that waits
        // for a fresh MUFU result holds back the next MUFU -- interleaved, the stream ran at ~12 clk per MUFU, not 8.
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
        const float zinv = __frcp_rn(zl + zh) * 1.0028177f;       // centred truncation to bf16, see arx_tc2.cu
        const uint64_t zz = pack2(zinv, zinv);
        if (tr) TRACE3(1 + g, k, 3);
        mbar_wait(&bars[B_P_EMPTY + g], (k & 1) ^ 1);
        if (tr) TRACE3(1 + g, k, 4);
#pragma unroll
        for (int c16 = 0; c16 < 16; ++c16) {
          uint32_t h[4];
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const uint64_t m = mul2(pack2u(r[c16 * 8 + 2 * q], r[c16 * 8 + 2 * q + 1]), zz);
            h[q] = __byte_perm((uint32_t)m, (uint32_t)(m >> 32), 0x7632);
          }
          *reinterpret_cast<uint4 *>(prow + (c16 >> 3) * 16384 + (((c16 & 7) ^ (s & 7)) << 4)) = make_uint4(h[0], h[1], h[2], h[3]);
        }
        if (tr) TRACE3(1 + g, k, 5);
        fence_proxy_async_smem();
        mbar_arrive(&bars[B_P_FULL + g]);
        if (tr) TRACE3(1 + g, k, 6);
      }
    }
  } else {
    // ---------------- epilogue warps: thread == output dimension d == TMEM lane; tiles (c, w0), (c, w1), (c+1, w0), ...
    setmaxnreg_inc<152>();
    const int quad = warp & 3;
    const int d = quad * 32 + lane;
    const uint32_t lane_base = (uint32_t)(quad * 32) << 16;
    float a0[16], a1[16];
    uint64_t bb0[8], bb1[8];
    // one flat loop over (group, class): the per-frame V projections are (re)loaded inside it at c == 0, which also
    // keeps the compiler from hoisting 32 loop-invariant register pairs per window out of a class loop and spilling them
    int gi = 0, c = 0, nw = my_groups ? group_nw(0) : 0, g = blockIdx.x;
    for (int k = 0; k < my_groups * p.way; ++k) {
      if (c == 0) {
        // per-frame V projections of the group's windows (v bias / positional table already inside).  Row-major
        // [frame][ldg] or the chunked layout of arx_gemm_p.cu (32-column chunks of 128 rows, 16-byte groups swizzled)
        auto load_ab = [&](int win, float (&a)[16], uint64_t (&bb)[8]) {
          if (p.gchunk) {
            const int r0 = (win & 7) * 16;
            const float *ca = p.G + ((size_t)(win >> 3) * 16 + ((p.voff + d) >> 5)) * 4096;
            const float *cb = ca + 4 * 4096;                                   // second V part: 128 columns = 4 chunks on
            const int qd = (d & 31) >> 2, e = d & 3;
#pragma unroll
            for (int i = 0; i < 16; ++i) a[i] = __ldg(ca + (r0 + i) * 32 + (((qd ^ (i & 7)) << 2) | e));
#pragma unroll
            for (int m = 0; m < 8; ++m)
              bb[m] = pack2(__ldg(cb + (r0 + 2 * m) * 32 + (((qd ^ ((2 * m) & 7)) << 2) | e)),
                            __ldg(cb + (r0 + 2 * m + 1) * 32 + (((qd ^ ((2 * m + 1) & 7)) << 2) | e)));
          } else {
            const float *g0 = p.G + (size_t)win * 16 * p.ldg + p.voff + d;
#pragma unroll
            for (int i = 0; i < 16; ++i) a[i] = __ldg(g0 + (size_t)i * p.ldg);
#pragma unroll
            for (int m = 0; m < 8; ++m) bb[m] = pack2(__ldg(g0 + (size_t)(2 * m) * p.ldg + DD), __ldg(g0 + (size_t)(2 * m + 1) * p.ldg + DD));
          }
        };
        load_ab(g * GW, a0, bb0);
        if (nw > 1) load_ab(g * GW + 1, a1, bb1);
      }
      // one tile: window slot w (compile-time, so a/bb stay in registers) of class c
      auto tile = [&](auto wc, const float (&a)[16], const uint64_t (&bb)[8]) {
        constexpr int w = decltype(wc)::value;
        mbar_wait(&bars[B_O_FULL + w], k & 1);
        if (w >= nw) { mbar_arrive(&bars[B_O_EMPTY + w]); return; }
        tc_fence_after();
        uint64_t acc[4] = {0ull, 0ull, 0ull, 0ull};
        uint32_t r[32], r2[32];
        tmem_ld32(TM_O + lane_base + w * 128 + 0, r);
        tmem_ld32(TM_O + lane_base + w * 128 + 32, r2);
        tmem_ld_wait();
        epi_chunk<0>(a, bb, r, acc, std::make_integer_sequence<int, 16>{});
        tmem_ld32(TM_O + lane_base + w * 128 + 64, r);
        epi_chunk<1>(a, bb, r2, acc, std::make_integer_sequence<int, 16>{});
        tmem_ld_wait();
        tmem_ld32(TM_O + lane_base + w * 128 + 96, r2);
        epi_chunk<2>(a, bb, r, acc, std::make_integer_sequence<int, 16>{});
        tmem_ld_wait();
        tc_fence_before();
        mbar_arrive(&bars[B_O_EMPTY + w]);
        epi_chunk<3>(a, bb, r2, acc, std::make_integer_sequence<int, 16>{});
        float al, ah;
        unpack2(add2(add2(acc[0], acc[1]), add2(acc[2], acc[3])), al, ah);
        float t = al + ah;
#pragma unroll
        for (int o = 16; o; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
        if (lane == 0) p.partial[((size_t)(g * GW + w) * p.way + c) * 4 + quad] = t;
      };
      tile(std::integral_constant<int, 0>{}, a0, bb0);
      tile(std::integral_constant<int, 1>{}, a1, bb1);
      if (++c == p.way) { c = 0; ++gi; g += gridDim.x; nw = gi < my_groups ? group_nw(gi) : 0; }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 3) { tc_fence_after(); tmem_dealloc(tmem, 512); }
}

}  // namespace

int arx_tc3_attention_launch(arx_handle *h, const ArxTransformer &tr, const __half *kq_img, const float *G, int64_t n_win, int way,
                             float *partial, int g_ld, int g_voff, bool g_chunked, bool episodes, cudaStream_t st) {
  Attn3Params p{};
  p.kq_img = kq_img; p.kc_img = tr.kc_tiles; p.vct_img = tr.vct_tiles; p.G = G; p.partial = partial;
  p.n_win = (int)n_win; p.way = way; p.ldg = g_ld; p.voff = g_voff; p.trace = h->trace_sel == 1 ? h->trace_buf : nullptr;
  p.gchunk = g_chunked ? 1 : 0;
  p.ep = episodes ? 1 : 0;
  p.token = h->attn_stagger < 0;
  p.stagger = h->attn_stagger < 0 ? 0 : h->attn_stagger;
  const int groups = episodes ? (int)n_win : (int)((n_win + 1) / 2);
  const int grid = groups < h->sm_count ? groups : h->sm_count;
  auto kern = h->attn_poly == 0 ? k_attn_tc3<0> : (h->attn_poly == 2 ? k_attn_tc3<2> : (h->attn_poly == 4 ? k_attn_tc3<4> : k_attn_tc3<3>));
  { const int rc_ = arx_func_smem(h, kern, (int)SMEM_BYTES); if (rc_) return rc_; }
  kern<<<grid, NTHREADS3, SMEM_BYTES, st>>>(p);
  ARX_LAUNCH_CHECK(h);
  return ARX_OK;
}

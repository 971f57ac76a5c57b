// Open-set head of the metric shape (T=16 pair tuples, N=120) by linearity, plus the padded-triangular slot order of
// the 120 query tuples shared with the attention kernel (arx_tc3.cu) and the tuple-image kernel (arx_gemm_p.cu):
// row i of the (i,j) triangle starts on an even j, so every fp32x2 operand pair is register-aligned; exactly 128 slots,
// 8 pads.  The order is internal to the kernels (the distance is a sum over tuples; y is written in lexicographic order).
#include "arx_internal.cuh"
#include "arx_ptx.cuh"
#include <utility>

namespace {
using namespace ptx;

constexpr int NTHREADS2 = 512;

}  // namespace

namespace {

__device__ __forceinline__ uint32_t ex2_bits(uint32_t x) {
  uint32_t y;
  asm volatile("ex2.approx.ftz.f32 %0, %1;" : "=r"(y) : "r"(x));
  return y;
}

template <int... Is> __device__ __forceinline__ void zero_pads(uint32_t (&r)[128], std::integer_sequence<int, Is...>) {
  ((r[arx_slot_row_start(2 * Is)] = 0u), ...);     // the pad slot of every even row
}

}  // namespace

// Host-side slot table (128 x 2): frame indices of every slot, -1 for pads; index math only.
void arx_tc2_slot_table(int32_t *out /* 256 */) {
  for (int q = 0; q < 128; ++q) {
    const int i = arx_slot_i(q), j = arx_slot_j(q);
    out[2 * q] = (j == i) ? -1 : i;
    out[2 * q + 1] = (j == i) ? -1 : j;
  }
}

// =====================================================================================================
// Open-set head pass, second generation (T=16 pair tuples).  For the winning class c* of every window
// (model.py:323-324) the discriminator input is y = Wdr.(Vq - proto)^T + bdr (model.py:196).  By linearity
//     y[q,l] = (Wdr.a_i)[l] + (Wdr.b_j)[l] + bdr[l]  -  sum_s P[q,s] * (Wdr.Vc[s])[l]
// so the pass needs no prototype MMA and no diff epilogue:
//   * UAB[frame][32] = {Wdr.a_i + bdr, Wdr.b_j}: 32 extra output columns of the frame projection GEMM
//     (composite weights Wdr.Wv, built at load time);
//   * Uc[l,s] = Wdr.Vc[s]: a 16 x 128 fp16 operand per class, built at set_support;
//   * MMA1 S^T = Kc.Kq'^T and the column softmax exactly as in k_attn_tc2, then ONE small MMA
//     Y[q,l] = sum_s P[q,s].Uc[l,s]  (M=128 q on TMEM lanes, N=16, K=128; A = P MN-major, 64 clk).
// Two softmax warpgroups with a P buffer each (200 KB of shared memory), so nothing serialises on P.
namespace {

constexpr uint32_t H2_OFF_KQ = 0;                       // 2 x 32 KB
constexpr uint32_t H2_OFF_KC = 2 * IMG_BYTES;           // 2 x 32 KB
constexpr uint32_t H2_OFF_P = 4 * IMG_BYTES;            // 2 x 32 KB (one per softmax group)
constexpr uint32_t H2_OFF_UC = 6 * IMG_BYTES;           // NUC x 4 KB
constexpr int NUC = 4;                                  // Uc ring: deeper than the Kq/Kc ring, see the producer
constexpr uint32_t UC_BYTES = 16 * DD * 2;
constexpr uint32_t H2_OFF_BAR = 6 * IMG_BYTES + NUC * UC_BYTES;
enum { H2_FULL_KK = 0, H2_EMPTY_KK = 2, H2_S_FULL = 4, H2_S_EMPTY = 6, H2_P_FULL = 8, H2_P_EMPTY = 10, H2_Y_FULL = 12, H2_Y_EMPTY = 14,
       H2_FULL_UC = 16, H2_EMPTY_UC = 16 + NUC, H2_COUNT = 16 + 2 * NUC };
constexpr uint32_t H2_SMEM_BYTES = H2_OFF_BAR + H2_COUNT * 8 + 16 + 1024;

struct Head2Params {
  const __half *kq_img, *kc_img, *uc_img;
  const float *uab;        // [n_win*16][32]
  const int32_t *chosen;
  __half *y_img;           // fp16 activation image [ceil(n_win/128)][y_nk][128 x 64]
  int n_win, y_nk;
  long long *trace;        // optional timeline of CTA 0 (bring-up): [3 roles: producer, softmax group 0, epilogue][64 windows][8 stamps]
  int l2_ahead;            // producer: L2 prefetch distance in windows of this CTA (huge = off)
  int cls_stride;          // episode mode: window b's classes start at b*cls_stride (0: one support set for all windows)
};

// per slot of the padded-triangular order: i | j << 8 | (lexicographic rank + 1) << 16 (0 = pad)
__constant__ uint32_t c_slot_info[128];

#define HTRACE(role, step, slot) do { if (p.trace && blockIdx.x == 0 && (step) < 64) p.trace[(((role) * 64) + (step)) * 8 + (slot)] = clock64(); } while (0)

__global__ void __launch_bounds__(NTHREADS2, 1) k_head2_tc(const Head2Params p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t *smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint64_t *bars = reinterpret_cast<uint64_t *>(smem + H2_OFF_BAR);
  uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(smem + H2_OFF_BAR + H2_COUNT * 8);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int ntiles = p.n_win > (int)blockIdx.x ? (p.n_win - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x : 0;
  if (threadIdx.x == 0) {
    for (int i = 0; i < 2; ++i) {
      mbar_init(&bars[H2_FULL_KK + i], 1); mbar_init(&bars[H2_EMPTY_KK + i], 1);
      mbar_init(&bars[H2_S_FULL + i], 1); mbar_init(&bars[H2_S_EMPTY + i], 128);
      mbar_init(&bars[H2_P_FULL + i], 128); mbar_init(&bars[H2_P_EMPTY + i], 1);
      mbar_init(&bars[H2_Y_FULL + i], 1); mbar_init(&bars[H2_Y_EMPTY + i], 128);
    }
    for (int i = 0; i < NUC; ++i) { mbar_init(&bars[H2_FULL_UC + i], 1); mbar_init(&bars[H2_EMPTY_UC + i], 1); }
    mbar_init_fence();
  }
  pdl_trigger();
  if (warp == 2) { tmem_alloc(tmem_slot, 512); tmem_relinquish(); }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  const uint32_t TM_S = tmem, TM_Y = tmem + 256;
  pdl_wait();

  if (warp < 4) {
    setmaxnreg_dec<40>();
    if (warp == 0) {
      if (elect_one()) {            // producer: {Kq[b], Kc[c*]} then Uc[c*] per tile, two stages
        for (int f = 1; f < p.l2_ahead && f < ntiles; ++f)
          bulk_prefetch_l2(reinterpret_cast<const uint8_t *>(p.kq_img) + (size_t)(blockIdx.x + f * gridDim.x) * IMG_BYTES, IMG_BYTES);
        // the class of the NEXT window is fetched while this window's copies are issued: a dependent load of `chosen` at the top
        // of every iteration put an L2 round trip on the producer's critical path
        int c_next = ntiles ? p.chosen[blockIdx.x] + (int)blockIdx.x * p.cls_stride : 0;
        for (int f = 0; f < ntiles; ++f) {
          const int b = blockIdx.x + f * gridDim.x, c = c_next, st = f & 1;
          if (f + 1 < ntiles) c_next = p.chosen[b + gridDim.x] + (b + (int)gridDim.x) * p.cls_stride;
          const uint8_t *kq = reinterpret_cast<const uint8_t *>(p.kq_img) + (size_t)b * IMG_BYTES;
          const uint8_t *kc = reinterpret_cast<const uint8_t *>(p.kc_img) + (size_t)c * IMG_BYTES;
          // the ring is two windows deep and a Kq image comes from HBM (the attention kernel read 134 MB since): with the DRAM
          // latency under load (~5 K clk) on every stage the kernel ran at ~3.1 K clk per window.  Pull the images of the windows
          // a few stages ahead into L2 now, so that the ring only sees the L2 latency.
          HTRACE(0, f, 0);
          if (f + p.l2_ahead < ntiles)
            bulk_prefetch_l2(reinterpret_cast<const uint8_t *>(p.kq_img) + (size_t)(b + p.l2_ahead * gridDim.x) * IMG_BYTES, IMG_BYTES);
          mbar_wait(&bars[H2_EMPTY_KK + st], ((f >> 1) & 1) ^ 1);
          HTRACE(0, f, 1);
          mbar_arrive_expect_tx(&bars[H2_FULL_KK + st], 2 * IMG_BYTES);
          bulk_g2s(smem + H2_OFF_KQ + st * IMG_BYTES, kq, SUB_BYTES, &bars[H2_FULL_KK + st]);
          bulk_g2s(smem + H2_OFF_KQ + st * IMG_BYTES + SUB_BYTES, kq + SUB_BYTES, SUB_BYTES, &bars[H2_FULL_KK + st]);
          bulk_g2s(smem + H2_OFF_KC + st * IMG_BYTES, kc, SUB_BYTES, &bars[H2_FULL_KK + st]);
          bulk_g2s(smem + H2_OFF_KC + st * IMG_BYTES + SUB_BYTES, kc + SUB_BYTES, SUB_BYTES, &bars[H2_FULL_KK + st]);
          HTRACE(0, f, 2);
          // A Uc stage is released by the Y MMA at the very END of a window's pipeline, a Kq/Kc stage by MMA1 at its start: with
          // two Uc stages this wait held back the NEXT window's Kq/Kc copies and exposed their latency on every other window
          // (timeline trace, tools/trace_head.py: 2.6 K clk per window).  Four 4 KB stages: the wait is always long satisfied.
          const int su = f % NUC;
          mbar_wait(&bars[H2_EMPTY_UC + su], ((f / NUC) & 1) ^ 1);
          HTRACE(0, f, 3);
          mbar_arrive_expect_tx(&bars[H2_FULL_UC + su], UC_BYTES);
          bulk_g2s(smem + H2_OFF_UC + su * UC_BYTES, reinterpret_cast<const uint8_t *>(p.uc_img) + (size_t)c * UC_BYTES, UC_BYTES,
                   &bars[H2_FULL_UC + su]);
        }
      }
    } else if (warp == 1) {
      if (elect_one()) {            // MMA1 issuer: S^T tiles
        constexpr uint64_t DESC_K = smem_desc_sw128(16, 1024);
        constexpr uint32_t IDESC1 = idesc_f16(128, 128, 0, 0);
        const uint32_t sbase = smem_u32(smem);
        for (int f = 0; f < ntiles; ++f) {
          const int st = f & 1;
          HTRACE(0, f, 4);
          mbar_wait(&bars[H2_FULL_KK + st], (f >> 1) & 1);
          HTRACE(0, f, 5);
          mbar_wait(&bars[H2_S_EMPTY + st], ((f >> 1) & 1) ^ 1);
          tc_fence_after();
          HTRACE(0, f, 6);
          const uint32_t a0 = sbase + H2_OFF_KC + st * IMG_BYTES, b0 = sbase + H2_OFF_KQ + st * IMG_BYTES;
#pragma unroll
          for (int kk = 0; kk < 8; ++kk) {
            const uint32_t off = (kk >> 2) * SUB_BYTES + (kk & 3) * 32;
            mma_f16_ss(TM_S + st * 128, smem_desc_at(DESC_K, a0 + off), smem_desc_at(DESC_K, b0 + off), IDESC1, kk > 0);
          }
          mma_commit(&bars[H2_S_FULL + st]);
          mma_commit(&bars[H2_EMPTY_KK + st]);
        }
      }
    } else if (warp == 3) {
      if (elect_one()) {            // Y issuer: Y[q,l] = sum_s P[q,s].Uc[l,s]
        constexpr uint64_t DESC_K = smem_desc_sw128(16, 1024);
        constexpr uint64_t DESC_MN = smem_desc_sw128(16384, 1024);
        constexpr uint32_t IDESCY = idesc_f16(128, 16, 1, 0);
        const uint32_t sbase = smem_u32(smem);
        for (int f = 0; f < ntiles; ++f) {
          const int st = f & 1;
          const int su = f % NUC;
          mbar_wait(&bars[H2_FULL_UC + su], (f / NUC) & 1);
          mbar_wait(&bars[H2_P_FULL + st], (f >> 1) & 1);
          mbar_wait(&bars[H2_Y_EMPTY + st], ((f >> 1) & 1) ^ 1);
          tc_fence_after();
#pragma unroll
          for (int kk = 0; kk < 8; ++kk) {
            const uint32_t boff = (kk >> 2) * (16 * 128) + (kk & 3) * 32;
            mma_f16_ss(TM_Y + st * 32, smem_desc_at(DESC_MN, sbase + H2_OFF_P + st * IMG_BYTES + kk * 2048),
                       smem_desc_at(DESC_K, sbase + H2_OFF_UC + su * UC_BYTES + boff), IDESCY, kk > 0);
          }
          mma_commit(&bars[H2_Y_FULL + st]);
          mma_commit(&bars[H2_P_EMPTY + st]);
          mma_commit(&bars[H2_EMPTY_UC + su]);
        }
      }
    }
  } else if (warp < 12) {
    setmaxnreg_inc<160>();
    const int g = (warp - 4) >> 2, quad = warp & 3;
    const int s = quad * 32 + lane;
    const uint32_t lane_base = (uint32_t)(quad * 32) << 16;
    uint8_t *prow = smem + H2_OFF_P + g * IMG_BYTES + (s >> 3) * 1024 + (s & 7) * 128;
    const bool trc = (threadIdx.x & 127) == 0;
    for (int f = g; f < ntiles; f += 2) {
      if (trc) HTRACE(1, f, 0);
      mbar_wait(&bars[H2_S_FULL + g], (f >> 1) & 1);
      tc_fence_after();
      if (trc) HTRACE(1, f, 1);
      uint32_t r[128];
      tmem_ld32(TM_S + lane_base + g * 128 + 0, *reinterpret_cast<uint32_t(*)[32]>(&r[0]));
      tmem_ld32(TM_S + lane_base + g * 128 + 32, *reinterpret_cast<uint32_t(*)[32]>(&r[32]));
      tmem_ld32(TM_S + lane_base + g * 128 + 64, *reinterpret_cast<uint32_t(*)[32]>(&r[64]));
      tmem_ld32(TM_S + lane_base + g * 128 + 96, *reinterpret_cast<uint32_t(*)[32]>(&r[96]));
      tmem_ld_wait();
      tc_fence_before();
      mbar_arrive(&bars[H2_S_EMPTY + g]);
      if (trc) HTRACE(1, f, 2);
#pragma unroll
      for (int j = 0; j < 128; ++j) r[j] = ex2_bits(r[j]);
      if (trc) HTRACE(1, f, 3);
      zero_pads(r, std::make_integer_sequence<int, 8>{});
      uint64_t z0 = 0ull, z1 = 0ull;
#pragma unroll
      for (int k = 0; k < 64; k += 2) {
        z0 = add2(z0, pack2u(r[2 * k], r[2 * k + 1]));
        z1 = add2(z1, pack2u(r[2 * k + 2], r[2 * k + 3]));
      }
      float zl, zh;
      unpack2(add2(z0, z1), zl, zh);
      const float zinv = __frcp_rn(zl + zh);
      const uint64_t zz = pack2(zinv, zinv);
      if (trc) HTRACE(1, f, 4);
      mbar_wait(&bars[H2_P_EMPTY + g], ((f >> 1) & 1) ^ 1);
      if (trc) HTRACE(1, f, 5);
#pragma unroll
      for (int c16 = 0; c16 < 16; ++c16) {
        uint32_t h[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          float lo, hi;
          unpack2(mul2(pack2u(r[c16 * 8 + 2 * k], r[c16 * 8 + 2 * k + 1]), zz), lo, hi);
          h[k] = pack_half2(lo, hi);
        }
        *reinterpret_cast<uint4 *>(prow + (c16 >> 3) * 16384 + (((c16 & 7) ^ (s & 7)) << 4)) = make_uint4(h[0], h[1], h[2], h[3]);
      }
      fence_proxy_async_smem();
      mbar_arrive(&bars[H2_P_FULL + g]);
      if (trc) HTRACE(1, f, 6);
    }
  } else {
    // ---------------- epilogue warps: thread == query-tuple slot q == TMEM lane of Y
    const int quad = warp & 3;
    const int q = quad * 32 + lane;
    const uint32_t lane_base = (uint32_t)(quad * 32) << 16;
    const uint32_t info = c_slot_info[q];
    const int fi = info & 0xff, fj = (info >> 8) & 0xff, rank = (int)(info >> 16) - 1;
    // the head-table rows of the NEXT window are fetched while this one is finished: loaded at the top of their own iteration
    // their L2 latency sat between the Y accumulator and the stores, ~1.9 K clk per window (timeline trace) -- the epilogue,
    // not the softmax groups, paced the kernel
    float4 ua[4], ub[4], na[4], nb[4];
    auto load_u = [&](int b, float4 (&a)[4], float4 (&bb)[4]) {
      const float4 *pa = reinterpret_cast<const float4 *>(p.uab + ((size_t)b * 16 + fi) * 32);
      const float4 *pb = reinterpret_cast<const float4 *>(p.uab + ((size_t)b * 16 + fj) * 32 + 16);
#pragma unroll
      for (int k = 0; k < 4; ++k) { a[k] = __ldg(pa + k); bb[k] = __ldg(pb + k); }
    };
    if (rank >= 0 && ntiles > 0) load_u(blockIdx.x, ua, ub);
    for (int f = 0; f < ntiles; ++f) {
      const int b = blockIdx.x + f * gridDim.x, st = f & 1;
      if (rank >= 0 && f + 1 < ntiles) load_u(b + gridDim.x, na, nb);
      if (q == 0) HTRACE(2, f, 0);
      mbar_wait(&bars[H2_Y_FULL + st], (f >> 1) & 1);
      tc_fence_after();
      if (q == 0) HTRACE(2, f, 1);
      uint32_t yv[16];
      tmem_ld16(TM_Y + lane_base + st * 32, yv);
      tmem_ld_wait();
      tc_fence_before();
      mbar_arrive(&bars[H2_Y_EMPTY + st]);
      if (rank >= 0) {
        const int col = rank * 16;
        uint8_t *dst = reinterpret_cast<uint8_t *>(p.y_img) + ((size_t)(b >> 7) * p.y_nk + (col >> 6)) * (128 * 128);
        float y[16];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          y[4 * k + 0] = ua[k].x + ub[k].x - __uint_as_float(yv[4 * k + 0]);
          y[4 * k + 1] = ua[k].y + ub[k].y - __uint_as_float(yv[4 * k + 1]);
          y[4 * k + 2] = ua[k].z + ub[k].z - __uint_as_float(yv[4 * k + 2]);
          y[4 * k + 3] = ua[k].w + ub[k].w - __uint_as_float(yv[4 * k + 3]);
        }
#pragma unroll
        for (int l = 0; l < 16; l += 8) {
          uint4 pk;
          pk.x = pack_half2(y[l + 0], y[l + 1]); pk.y = pack_half2(y[l + 2], y[l + 3]);
          pk.z = pack_half2(y[l + 4], y[l + 5]); pk.w = pack_half2(y[l + 6], y[l + 7]);
          *reinterpret_cast<uint4 *>(dst + sw128_offset(b & 127, (col & 63) + l)) = pk;
        }
      }
#pragma unroll
      for (int k = 0; k < 4; ++k) { ua[k] = na[k]; ub[k] = nb[k]; }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) { tc_fence_after(); tmem_dealloc(tmem, 512); }
}

// Uc[c][l][s] = sum_d Wdr[l][d] * Vc[c][s][d] as a K-major SW128 B operand (16 rows x 128 s, fp16); one block per class
__global__ void __launch_bounds__(128) k_support_uc(const float *__restrict__ vs, const float *__restrict__ dr_w, __half *__restrict__ uc_img, int N) {
  __shared__ float w[16 * 128];
  for (int e = threadIdx.x; e < 16 * 128; e += 128) w[e] = dr_w[e];
  __syncthreads();
  const size_t cls = blockIdx.x;
  const int s = threadIdx.x;
  float acc[16];
#pragma unroll
  for (int l = 0; l < 16; ++l) acc[l] = 0.f;
  if (s < N) {
    const float4 *v = reinterpret_cast<const float4 *>(vs + (cls * N + s) * 128);
    for (int d4 = 0; d4 < 32; ++d4) {
      const float4 x = v[d4];
#pragma unroll
      for (int l = 0; l < 16; ++l) {
        const float4 ww = *reinterpret_cast<const float4 *>(&w[l * 128 + d4 * 4]);
        acc[l] += x.x * ww.x + x.y * ww.y + x.z * ww.z + x.w * ww.w;
      }
    }
  }
  uint8_t *out = reinterpret_cast<uint8_t *>(uc_img) + cls * UC_BYTES;
#pragma unroll
  for (int l = 0; l < 16; ++l)
    *reinterpret_cast<__half *>(out + (s >> 6) * (16 * 128) + sw128_offset(l, s & 63)) = __float2half_rn(acc[l]);
}

// composite projection: Wc[p*16 + l][f] = sum_d Wdr[l][d] * Wv_p[d][f];  tc[t][p*16 + l] = sum_d Wdr[l][d] * table[t][(c+p)*128 + d] (+ bdr[l], p == 0)
__global__ void k_compose_head(const float *__restrict__ dr_w, const float *__restrict__ dr_b, const float *__restrict__ wp, const float *__restrict__ table,
                               float *__restrict__ wc, float *__restrict__ tc, int F, int ld, int voff, int T) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx < 32 * F) {
    const int row = idx / F, f = idx % F, pp = row >> 4, l = row & 15;
    float a = 0.f;
    for (int d = 0; d < 128; ++d) a += dr_w[l * 128 + d] * wp[(size_t)(voff + pp * 128 + d) * F + f];
    wc[idx] = a;
  }
  if (idx < T * 32) {
    const int t = idx / 32, col = idx % 32, pp = col >> 4, l = col & 15;
    float a = pp == 0 ? dr_b[l] : 0.f;
    for (int d = 0; d < 128; ++d) a += dr_w[l * 128 + d] * table[(size_t)t * ld + voff + pp * 128 + d];
    tc[idx] = a;
  }
}

}  // namespace

int arx_tc2_head_prepare_weights(arx_handle *h, ArxTransformer &tr, cudaStream_t st) {
  // composite weights / table for the 32 extra projection columns (only meaningful for T=16 pair tuples)
  if (!tr.wc) ARX_CUDA(h, cudaMalloc(reinterpret_cast<void **>(&tr.wc), (size_t)32 * h->F * sizeof(float)));
  if (!tr.tcomp) ARX_CUDA(h, cudaMalloc(reinterpret_cast<void **>(&tr.tcomp), (size_t)h->T * 32 * sizeof(float)));
  const int n = 32 * h->F;
  k_compose_head<<<(n + 127) / 128, 128, 0, st>>>(h->dr_w, h->dr_b, tr.wp, tr.bp, tr.wc, tr.tcomp, h->F, 2 * tr.c * h->D, tr.c * h->D, h->T);
  ARX_LAUNCH_CHECK(h);
  int rc = arx_tc_linear_prepare(h, tr.tl_uab, tr.wc, h->F, nullptr, 32, h->F, 32, st);
  if (rc) return rc;
  uint32_t info[128];
  for (int q = 0; q < 128; ++q) {
    const int i = arx_slot_i(q), j = arx_slot_j(q);
    const int rank = (j == i) ? -1 : i * (2 * 16 - i - 1) / 2 + (j - i - 1);
    info[q] = (uint32_t)i | ((uint32_t)j << 8) | ((uint32_t)(rank + 1) << 16);
  }
  ARX_CUDA(h, cudaMemcpyToSymbolAsync(c_slot_info, info, sizeof(info), 0, cudaMemcpyHostToDevice, st));
  return ARX_OK;
}

int arx_tc2_support_uc(arx_handle *h, ArxTransformer &tr, int way, cudaStream_t st) {
  if (!tr.uc_img) ARX_CUDA(h, cudaMalloc(reinterpret_cast<void **>(&tr.uc_img), (size_t)h->way_cap * UC_BYTES));
  k_support_uc<<<way, 128, 0, st>>>(tr.vs, h->dr_w, tr.uc_img, tr.N);
  ARX_LAUNCH_CHECK(h);
  return ARX_OK;
}

int arx_tc2_head_launch(arx_handle *h, const ArxTransformer &tr, const __half *kq_img, const float *uab, int64_t n_win, const int32_t *chosen,
                        __half *y_img, int y_nk, int cls_stride, cudaStream_t st) {
  Head2Params p{};
  p.kq_img = kq_img; p.kc_img = tr.kc_tiles; p.uc_img = tr.uc_img; p.uab = uab; p.chosen = chosen; p.y_img = y_img; p.n_win = (int)n_win; p.y_nk = y_nk; p.cls_stride = cls_stride;
  p.l2_ahead = (h->tc_variant & 16384) ? 1 << 30 : 4;
  p.trace = h->trace_sel == 3 ? h->trace_buf : nullptr;
  const int grid = n_win < h->sm_count ? (int)n_win : h->sm_count;
  { const int rc_ = arx_func_smem(h, k_head2_tc, (int)H2_SMEM_BYTES); if (rc_) return rc_; }
  ARX_CUDA(h, arx_launch_pdl(k_head2_tc, dim3(grid), dim3(NTHREADS2), H2_SMEM_BYTES, st, h->pdl, p));
  h->launches++;
  return ARX_OK;
}

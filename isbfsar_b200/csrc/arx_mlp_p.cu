// Fused frame MLP (modules/ar/utils/model.py:175-180): f = relu(fc2(relu(fc1(x)))) for a big batch of frames in ONE
// persistent tcgen05 kernel.  It replaces k_rows_to_img + k_gemm_p<192> + k_gemm_p<256>: the fp16 pose image and the
// hidden image never reach global memory (149 MB moved per 65 536 frames -> 66 MB: fp32 poses in, fp16 features out).
//   * one CTA per SM, persistent over 128-row tiles; BOTH weight images (48 + 96 KB) stay in shared memory;
//   * four loader warps read the next tile's poses (coalesced 8-byte loads, held in registers until the MMA has
//     released the operand buffer), round to fp16 and write the K-major SW128 operand image of fc1;
//   * one thread issues fc1 (N=192) into TMEM columns [0,192) and fc2 (N=256) into [256,512); fc2 starts on the
//     first 64 hidden columns while the epilogue is still producing the others, and fc1 of tile t+1 runs under the
//     second epilogue of tile t;
//   * eight epilogue warps (thread == row == TMEM lane, two warps per lane quadrant splitting the columns): bias + ReLU +
//     fp16 -> the hidden operand image in shared memory; then bias + ReLU + fp16 of fc2 into the SAME 48 KB (dead once fc2
//     has read it) as 4 KB staging blocks, written out with bulk stores -- the arithmetic (fp16 operands, fp32 accumulate,
//     round-to-nearest) is exactly that of the three kernels it replaces, so the feature image is bit-identical.
// The one-hot(frame position) sub-tile that carries the positional-encoding / bias table through the projection GEMM
// (arx_gemm_p.cu) is written here as well.
#include "arx_internal.cuh"
#include "arx_ptx.cuh"
#include <type_traits>

namespace {
using namespace ptx;

constexpr uint32_t SUB = 128 * 128;                   // one operand sub-tile: 128 rows x 64 fp16
constexpr int BN1 = 192, BN2 = 256, NK1 = 2, NK2 = 3;
constexpr uint32_t W1_BLK = BN1 * 128, W2_BLK = BN2 * 128;
constexpr uint32_t OFF_W1 = 0, OFF_W2 = NK1 * W1_BLK, OFF_X = OFF_W2 + NK2 * W2_BLK, OFF_H = OFF_X + NK1 * SUB, OFF_BAR = OFF_H + NK2 * SUB;
enum { B_W = 0, B_X_FULL, B_X_EMPTY, B_A1_FULL, B_A1_EMPTY, B_H_FULL /* NK2 of them */, B_A2_FULL = B_H_FULL + NK2, B_A2_EMPTY, B_COUNT };
constexpr uint32_t SMEM_BYTES = OFF_BAR + B_COUNT * 8 + 16 + 1024;
constexpr int M_THREADS = 448;                        // warps 0-7 epilogue, 8 weight producer, 9 MMA issuer, 10-13 pose loaders
constexpr int W_PROD = 8, W_MMA = 9, W_LOAD = 10;
static_assert(SMEM_BYTES <= 232448, "shared memory budget");

struct MlpParams {
  const void *x;              // [rows][2*PPR] poses, fp32 or fp16, rows contiguous
  const __half *w1_img;       // [NK1][BN1 x 64]
  const __half *w2_img;       // [NK2][BN2 x 64]
  __half *f_img;              // [m_tiles][c_nk][128 x 64]
  long long rows;
  long long *trace;           // optional timeline of CTA 0 (bring-up): [3 roles: MMA issuer, epilogue, loader][64 tiles][8 stamps]
  int m_tiles, c_nk, onehot_sub, k16_1;
  float b1[BN1], b2[BN2];     // zero padded; read as constant-bank operands
};

#define MTRACE(role, step, slot) do { if (p.trace && blockIdx.x == 0 && (step) < 64) p.trace[(((role) * 64) + (step)) * 8 + (slot)] = clock64(); } while (0)

__device__ __forceinline__ uint32_t pack_h2(float lo, float hi) {
  const __half2 h = __floats2half2_rn(lo, hi);
  return *reinterpret_cast<const uint32_t *>(&h);
}

// bias + ReLU + fp16 of one 32-column accumulator chunk (columns c0..c0+31 of layer LAYER) -> four 16-byte groups of a SW128 row;
// the bias is indexed in the kernel parameters directly, so it stays a constant-bank operand
template <int LAYER>
__device__ __forceinline__ void act_store(const MlpParams &p, const uint32_t (&v)[32], int c0, uint8_t *row, int lane) {
  const int half = (c0 >> 5) & 1;
#pragma unroll
  for (int ch = 0; ch < 4; ++ch) {
    float x[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) x[e] = fmaxf(__uint_as_float(v[ch * 8 + e]) + (LAYER == 1 ? p.b1[c0 + ch * 8 + e] : p.b2[c0 + ch * 8 + e]), 0.f);
    const uint4 pk = make_uint4(pack_h2(x[0], x[1]), pack_h2(x[2], x[3]), pack_h2(x[4], x[5]), pack_h2(x[6], x[7]));
    *reinterpret_cast<uint4 *>(row + (((half * 4 + ch) ^ (lane & 7)) << 4)) = pk;
  }
}

// PPR = element pairs per pose row (J3 / 2); TIn = float or __half
template <class TIn, int PPR>
__global__ void __launch_bounds__(M_THREADS, 1) k_mlp_p(const __grid_constant__ MlpParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t *smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint64_t *bars = reinterpret_cast<uint64_t *>(smem + OFF_BAR);
  uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(smem + OFF_BAR + B_COUNT * 8);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    mbar_init(&bars[B_W], 1);
    mbar_init(&bars[B_X_FULL], 128); mbar_init(&bars[B_X_EMPTY], 1);
    mbar_init(&bars[B_A1_FULL], 1); mbar_init(&bars[B_A1_EMPTY], 256);
    for (int i = 0; i < NK2; ++i) mbar_init(&bars[B_H_FULL + i], 256);
    mbar_init(&bars[B_A2_FULL], 1); mbar_init(&bars[B_A2_EMPTY], 256);
    mbar_init_fence();
  }
  if (warp == W_MMA) { tmem_alloc(tmem_slot, 512); tmem_relinquish(); }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  const uint32_t TM_1 = tmem, TM_2 = tmem + 256;

  if (warp == W_PROD) {
    if (elect_one()) {              // both weight images, once
      mbar_arrive_expect_tx(&bars[B_W], NK1 * W1_BLK + NK2 * W2_BLK);
      for (int ks = 0; ks < NK1; ++ks)
        bulk_g2s(smem + OFF_W1 + ks * W1_BLK, reinterpret_cast<const uint8_t *>(p.w1_img) + (size_t)ks * W1_BLK, W1_BLK, &bars[B_W]);
      for (int ks = 0; ks < NK2; ++ks)
        bulk_g2s(smem + OFF_W2 + ks * W2_BLK, reinterpret_cast<const uint8_t *>(p.w2_img) + (size_t)ks * W2_BLK, W2_BLK, &bars[B_W]);
    }
  } else if (warp == W_MMA) {
    if (elect_one()) {
      constexpr uint64_t DESC_K = smem_desc_sw128(16, 1024);
      constexpr uint32_t IDESC1 = idesc_f16(128, BN1, 0, 0), IDESC2 = idesc_f16(128, BN2, 0, 0);
      const uint32_t sbase = smem_u32(smem);
      mbar_wait(&bars[B_W], 0);
      int i = 0;
      for (int mt = blockIdx.x; mt < p.m_tiles; mt += gridDim.x, ++i) {
        MTRACE(0, i, 0);
        mbar_wait(&bars[B_X_FULL], i & 1);
        MTRACE(0, i, 1);
        mbar_wait(&bars[B_A1_EMPTY], (i & 1) ^ 1);
        tc_fence_after();
        for (int k = 0; k < p.k16_1; ++k)
          mma_f16_ss(TM_1, smem_desc_at(DESC_K, sbase + OFF_X + (k >> 2) * SUB + (k & 3) * 32),
                     smem_desc_at(DESC_K, sbase + OFF_W1 + (k >> 2) * W1_BLK + (k & 3) * 32), IDESC1, k != 0);
        mma_commit(&bars[B_X_EMPTY]);
        mma_commit(&bars[B_A1_FULL]);
        MTRACE(0, i, 2);
        mbar_wait(&bars[B_A2_EMPTY], (i & 1) ^ 1);
        MTRACE(0, i, 3);
        for (int ks = 0; ks < NK2; ++ks) {
          mbar_wait(&bars[B_H_FULL + ks], i & 1);
          MTRACE(0, i, 4 + ks);
          tc_fence_after();
#pragma unroll
          for (int kk = 0; kk < 4; ++kk)
            mma_f16_ss(TM_2, smem_desc_at(DESC_K, sbase + OFF_H + ks * SUB + kk * 32),
                       smem_desc_at(DESC_K, sbase + OFF_W2 + ks * W2_BLK + kk * 32), IDESC2, (ks | kk) != 0);
        }
        mma_commit(&bars[B_A2_FULL]);
        MTRACE(0, i, 7);
      }
    }
  } else if (warp >= W_LOAD) {
    // ---------------- pose loaders: thread t owns pairs t, t+128, ... of the tile's 128*PPR element pairs
    const int t = threadIdx.x - W_LOAD * 32;
    for (int e = t; e < (int)(NK1 * SUB / 16); e += 128) *reinterpret_cast<uint4 *>(smem + OFF_X + e * 16) = make_uint4(0u, 0u, 0u, 0u);   // pad columns stay zero
    __syncwarp();
    named_bar_sync(2, 128);
    int i = 0;
    for (int mt = blockIdx.x; mt < p.m_tiles; mt += gridDim.x, ++i) {
      const long long row0 = (long long)mt * 128;
      if (t == 0) MTRACE(2, i, 0);
      uint32_t v[PPR];
      // volatile loads: they must all be IN FLIGHT before the wait below (plain __ldg loads were partly scheduled behind it,
      // which put a DRAM latency on every tile's critical path -- ncu: the epilogue warps idle on the fc1 accumulator)
      if constexpr (sizeof(TIn) == 4) {
        float2 f[PPR];
        const float2 *src = reinterpret_cast<const float2 *>(p.x) + row0 * PPR;
#pragma unroll
        for (int k = 0; k < PPR; ++k) {
          const int pi = t + 128 * k;
          f[k] = make_float2(0.f, 0.f);
          if (row0 + pi / PPR < p.rows) asm volatile("ld.global.nc.v2.f32 {%0, %1}, [%2];" : "=f"(f[k].x), "=f"(f[k].y) : "l"(src + pi));
        }
#pragma unroll
        for (int k = 0; k < PPR; ++k) v[k] = pack_h2(f[k].x, f[k].y);
      } else {
        const uint32_t *src = reinterpret_cast<const uint32_t *>(p.x) + row0 * PPR;
#pragma unroll
        for (int k = 0; k < PPR; ++k) {
          const int pi = t + 128 * k;
          v[k] = 0u;
          if (row0 + pi / PPR < p.rows) asm volatile("ld.global.nc.b32 %0, [%1];" : "=r"(v[k]) : "l"(src + pi));
        }
      }
      if (t == 0) MTRACE(2, i, 1);
      mbar_wait(&bars[B_X_EMPTY], (i & 1) ^ 1);          // fc1 of the previous tile has read the operand buffer
#pragma unroll
      for (int k = 0; k < PPR; ++k) {
        const int pi = t + 128 * k, row = pi / PPR, col = 2 * (pi - row * PPR);
        *reinterpret_cast<uint32_t *>(smem + OFF_X + (col >> 6) * SUB + sw128_offset(row, col & 63)) = v[k];
      }
      if (t == 0) MTRACE(2, i, 2);
      fence_proxy_async_smem();
      mbar_arrive(&bars[B_X_FULL]);
      if (t == 0) MTRACE(2, i, 3);
    }
  } else {
    // ---------------- epilogue warps: thread == row of the tile == TMEM lane.  EIGHT warps, two per scheduler: warps q and q + 4
    // share TMEM lane quadrant q and split every 64-column sub-tile, `half` = which 32 columns.  The pair meets at a named barrier
    // where one of them speaks for both (bulk-store groups belong to the thread that committed them: lane 0 of the half-0 warp).
    // (Measured against four warps doing whole sub-tiles: the same ~1.5 K + 3 K clk per tile -- the chain is TMEM-load, fence,
    // barrier and bulk-store latencies, not instruction issue; kept because it halves the registers live per thread.)
    const int quad = warp & 3, half = warp >> 2;
    const int r = quad * 32 + lane;
    const uint32_t lane_base = (uint32_t)(quad * 32) << 16;
    uint8_t *hrow = smem + OFF_H + quad * 4096 + lane * 128;        // this row inside sub-tile / staging block 0
    const bool leader = half == 0 && lane == 0;
    auto pair_sync = [&]() { named_bar_sync(4 + quad, 64); };
    int i = 0;
    for (int mt = blockIdx.x; mt < p.m_tiles; mt += gridDim.x, ++i) {
      // fc1 epilogue -> hidden operand image, one 64-column K sub-tile of fc2 at a time; the next accumulator chunk is already on
      // its way from TMEM.  Staging blocks of the previous tile went out in the order 2, 0, 1, 2 (see below), so block ks only
      // needs all but the last (2 - ks) bulk stores to have left shared memory.
      if (threadIdx.x == 0) MTRACE(1, i, 0);
      mbar_wait(&bars[B_A1_FULL], i & 1);
      tc_fence_after();
      if (threadIdx.x == 0) MTRACE(1, i, 1);
      {
        uint32_t va[32], vb[32];
        auto step1 = [&](auto ksc, uint32_t (&cur)[32], uint32_t (&nxt)[32]) {
          constexpr int ks = decltype(ksc)::value;
          if (leader) { if (ks == 0) bulk_wait_read<2>(); else if (ks == 1) bulk_wait_read<1>(); else bulk_wait_read<0>(); }
          pair_sync();
          tmem_ld_wait();
          if (ks + 1 < BN1 / 64) tmem_ld32(TM_1 + lane_base + (ks + 1) * 64 + half * 32, nxt);
          else { tc_fence_before(); mbar_arrive(&bars[B_A1_EMPTY]); }
          act_store<1>(p, cur, ks * 64 + half * 32, hrow + ks * SUB, lane);
          fence_proxy_async_smem();                       // this warp's half of 64 hidden columns: fc2 may start once both are in
          mbar_arrive(&bars[B_H_FULL + ks]);
        };
        tmem_ld32(TM_1 + lane_base + half * 32, va);
        step1(std::integral_constant<int, 0>{}, va, vb);
        step1(std::integral_constant<int, 1>{}, vb, va);
        step1(std::integral_constant<int, 2>{}, va, vb);
      }
      // fc2 epilogue -> feature image; the hidden image is dead once fc2 has completed: its 48 KB are the staging blocks
      if (threadIdx.x == 0) MTRACE(1, i, 2);
      mbar_wait(&bars[B_A2_FULL], i & 1);
      tc_fence_after();
      if (threadIdx.x == 0) MTRACE(1, i, 3);
      {
        uint32_t va[32], vb[32];
        tmem_ld32(TM_2 + lane_base + half * 32, va);
        if (p.onehot_sub >= 0) {
          // extra K columns for the projection GEMM: one-hot(frame position) twice (against the hi and lo halves of the
          // positional-encoding / bias table), so that the table is added by the tensor core (model.py:27,75-78)
          uint8_t *dst = reinterpret_cast<uint8_t *>(p.f_img) + ((size_t)mt * p.c_nk + p.onehot_sub) * SUB;
          const int tt = r & 15;
#pragma unroll
          for (int c4 = 0; c4 < 4; ++c4) {                 // each warp of the pair writes half of the row
            const int ch = half * 4 + c4;
            uint4 pk = make_uint4(0u, 0u, 0u, 0u);
            if (ch == (tt >> 3) || ch == 2 + (tt >> 3)) {
              const uint32_t one = 0x3C00u << (16 * (tt & 1));
              const int w = (tt & 7) >> 1;
              pk.x = w == 0 ? one : 0u; pk.y = w == 1 ? one : 0u; pk.z = w == 2 ? one : 0u; pk.w = w == 3 ? one : 0u;
            }
            *reinterpret_cast<uint4 *>(dst + sw128_offset(r, ch * 8)) = pk;
          }
        }
        auto step2 = [&](auto sc, uint32_t (&cur)[32], uint32_t (&nxt)[32]) {
          constexpr int s4 = decltype(sc)::value;
          constexpr int sb = s4 == 0 ? 2 : (s4 == 1 ? 0 : (s4 == 2 ? 1 : 2));     // the block fc1's epilogue needs first is the one stored longest ago
          if (s4 == 3) {                                  // block 2 again: its first store must have left
            if (leader) bulk_wait_read<2>();
            pair_sync();
          }
          tmem_ld_wait();
          if (s4 + 1 < BN2 / 64) tmem_ld32(TM_2 + lane_base + (s4 + 1) * 64 + half * 32, nxt);
          else { tc_fence_before(); mbar_arrive(&bars[B_A2_EMPTY]); }
          act_store<2>(p, cur, s4 * 64 + half * 32, hrow + sb * SUB, lane);
          fence_proxy_async_smem();
          pair_sync();
          if (leader) {
            bulk_s2g(reinterpret_cast<uint8_t *>(p.f_img) + ((size_t)mt * p.c_nk + s4) * SUB + quad * 4096, smem + OFF_H + sb * SUB + quad * 4096, 4096);
            bulk_commit();
          }
        };
        step2(std::integral_constant<int, 0>{}, va, vb);
        step2(std::integral_constant<int, 1>{}, vb, va);
        step2(std::integral_constant<int, 2>{}, va, vb);
        step2(std::integral_constant<int, 3>{}, vb, va);
      }
      if (threadIdx.x == 0) MTRACE(1, i, 4);
    }
    if (leader) bulk_wait_all();
    tc_fence_before();
  }
  __syncthreads();
  if (warp == W_MMA) { tc_fence_after(); tmem_dealloc(tmem, 512); }
}

}  // namespace

// Can the fused kernel take this model / input?  (J3 = 90: 30 joints x 3; other shapes keep the three-kernel path.)
bool arx_mlp_fused_supported(const arx_handle *h, const void *x) {
  const ArxTcLinear &a = h->tl_fc1, &b = h->tl_fc2;
  return h->J3 == 90 && a.BN == BN1 && a.nk == NK1 && a.n_tiles == 1 && b.BN == BN2 && b.nk == NK2 && b.n_tiles == 1 && h->mlp_bias_host_ok &&
         (reinterpret_cast<uintptr_t>(x) & 7u) == 0;
}

// f_img[m_tiles][c_nk] = relu(fc2(relu(fc1(x)))) (+ the one-hot sub-tile at index onehot_sub, -1 = none); x (rows, J3) fp32, or fp16 when `f16`;
// persistent on at most `sms` SMs
int arx_mlp_fused(arx_handle *h, const void *x, bool f16, int64_t rows, __half *f_img, int c_nk, int onehot_sub, int sms, cudaStream_t st) {
  MlpParams p{};
  p.x = x; p.w1_img = h->tl_fc1.w_img; p.w2_img = h->tl_fc2.w_img; p.f_img = f_img; p.rows = rows;
  p.trace = h->trace_sel == 2 ? h->trace_buf : nullptr;
  p.m_tiles = (int)((rows + 127) / 128); p.c_nk = c_nk; p.onehot_sub = onehot_sub; p.k16_1 = (h->J3 + 15) / 16;
  memcpy(p.b1, h->mlp_bias_host, sizeof(p.b1));
  memcpy(p.b2, h->mlp_bias_host + BN1, sizeof(p.b2));
  const int grid = p.m_tiles < sms ? p.m_tiles : sms;
  if (f16) {
    auto kern = k_mlp_p<__half, 45>;
    { const int rc_ = arx_func_smem(h, kern, (int)SMEM_BYTES); if (rc_) return rc_; }
    kern<<<grid, M_THREADS, SMEM_BYTES, st>>>(p);
  } else {
    auto kern = k_mlp_p<float, 45>;
    { const int rc_ = arx_func_smem(h, kern, (int)SMEM_BYTES); if (rc_) return rc_; }
    kern<<<grid, M_THREADS, SMEM_BYTES, st>>>(p);
  }
  ARX_LAUNCH_CHECK(h);
  return ARX_OK;
}

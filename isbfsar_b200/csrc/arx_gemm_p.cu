// Persistent tcgen05 GEMM for the per-frame linear layers of a big batch, and the query tuple-image kernel.
//
// k_gemm_p:  C[M,N] = act(A[M,K] . W[N,K]^T + bias), same operand "images" as arx_gemm_tc.cu, but built for the
// shape these layers have at batch size -- M = 65536 rows against a weight matrix of a few hundred KB:
//   * one CTA per SM, persistent over the 128-row tiles of ONE column tile; the column tile's weights are loaded
//     into shared memory ONCE (up to 160 KB) instead of once per row tile (the non-persistent kernel re-read
//     240 KB of operands from L2 per CTA, which bounded it);
//   * activations stream through a ring of 16 KB stages (bulk copies + mbarriers);
//   * two TMEM accumulators (2 x 256 columns): the MMAs of tile t+1 run under the epilogue of tile t;
//   * the epilogue never stores from registers to global memory: each warp assembles its 32 rows x 128 B of every
//     32-column (fp32) / 64-column (fp16) block in shared memory, in the SW128 pattern (conflict-free), and one
//     lane issues a 4 KB bulk store.
// Outputs: fp16 activation images (next layer's A operand), or the CHUNKED fp32 projection buffer
//   Gc[row tile][32-column chunk][128 rows][32 floats, 16-byte groups XOR-swizzled by (row & 7)]
// which k_tuple_img and the attention epilogues read (model.py:75-78: k_linear/v_linear per frame, by linearity).
//
// k_tuple_img: Kq operand images from the chunked per-frame K projections (model.py:69-82): one CTA per window,
// THREAD == TUPLE SLOT, LayerNorm statistics thread-local, image assembled in shared memory, one 32 KB bulk store.
#include "arx_internal.cuh"
#include "arx_ptx.cuh"

namespace {
using namespace ptx;

constexpr uint32_t A_SUB = 128 * 128;       // 128 rows x 64 fp16
constexpr int P_THREADS = 192;
enum { POUT_IMG16 = 0, POUT_F32C = 1 };

struct GemmPParams {
  const __half *a_img;     // [m_tiles][a_nk][128 x 64]
  const __half *w_img;     // [n_tiles][nk][BN x 64]
  const float *bias;       // [n_tiles*BN] or null
  int nk, a_nk, nsta;
  int m_tiles, n_tiles;
  int act;
  __half *c_img;           // POUT_IMG16: [m_tiles][c_nk][128 x 64]
  int c_nk, onehot_sub;
  float *gc;               // POUT_F32C: chunked projections, n_tiles*BN/32 chunks per row tile
};

// NSTG = 4 KB staging blocks per epilogue warp: a bulk store takes ~1000 clocks to release its source, so a warp
// needs several blocks in flight unless the layer is HBM-bound anyway
template <int BN, int OUT, int NSTG>
__global__ void __launch_bounds__(P_THREADS, 1) k_gemm_p(const GemmPParams p) {
  constexpr uint32_t B_SUB = BN * 128;
  constexpr uint32_t P_STG = 4 * NSTG * 4096;
  extern __shared__ uint8_t smem_raw[];
  uint8_t *smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  const uint32_t off_a = p.nk * B_SUB, off_stg = off_a + p.nsta * A_SUB, off_bias = off_stg + P_STG, off_bar = off_bias + BN * 4;
  uint64_t *bars = reinterpret_cast<uint64_t *>(smem + off_bar);   // b_full, a_full[nsta], a_empty[nsta], acc_full[2], acc_empty[2]
  uint64_t *b_full = bars, *a_full = bars + 1, *a_empty = bars + 1 + p.nsta, *acc_full = bars + 1 + 2 * p.nsta, *acc_empty = acc_full + 2;
  uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(acc_empty + 2);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nt = blockIdx.x % p.n_tiles, m0 = blockIdx.x / p.n_tiles, m_stride = gridDim.x / p.n_tiles;
  if (threadIdx.x == 0) {
    mbar_init(b_full, 1);
    for (int i = 0; i < p.nsta; ++i) { mbar_init(&a_full[i], 1); mbar_init(&a_empty[i], 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(&acc_full[i], 1); mbar_init(&acc_empty[i], 128); }
    mbar_init_fence();
  }
  if (warp == 5) { tmem_alloc(tmem_slot, 512); tmem_relinquish(); }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;

  if (warp == 4) {
    if (elect_one()) {
      const uint8_t *w = reinterpret_cast<const uint8_t *>(p.w_img) + (size_t)nt * p.nk * B_SUB;
      mbar_arrive_expect_tx(b_full, p.nk * B_SUB);
      for (int ks = 0; ks < p.nk; ++ks) bulk_g2s(smem + ks * B_SUB, w + (size_t)ks * B_SUB, B_SUB, b_full);
      int it = 0;
      for (int mt = m0; mt < p.m_tiles; mt += m_stride) {
        const uint8_t *a = reinterpret_cast<const uint8_t *>(p.a_img) + (size_t)mt * p.a_nk * A_SUB;
        for (int ks = 0; ks < p.nk; ++ks, ++it) {
          const int st = it % p.nsta;
          mbar_wait(&a_empty[st], ((it / p.nsta) & 1) ^ 1);
          mbar_arrive_expect_tx(&a_full[st], A_SUB);
          bulk_g2s(smem + off_a + st * A_SUB, a + (size_t)ks * A_SUB, A_SUB, &a_full[st]);
        }
      }
    }
  } else if (warp == 5) {
    if (elect_one()) {
      constexpr uint64_t DESC_K = smem_desc_sw128(16, 1024);
      constexpr uint32_t IDESC = idesc_f16(128, BN, 0, 0);
      const uint32_t sbase = smem_u32(smem);
      mbar_wait(b_full, 0);
      int it = 0, t = 0;
      for (int mt = m0; mt < p.m_tiles; mt += m_stride, ++t) {
        const int buf = t & 1;
        mbar_wait(&acc_empty[buf], ((t >> 1) & 1) ^ 1);
        tc_fence_after();
        for (int ks = 0; ks < p.nk; ++ks, ++it) {
          const int st = it % p.nsta;
          mbar_wait(&a_full[st], (it / p.nsta) & 1);
          tc_fence_after();
#pragma unroll
          for (int kk = 0; kk < 4; ++kk)
            mma_f16_ss(tmem + buf * 256, smem_desc_at(DESC_K, sbase + off_a + st * A_SUB + kk * 32),
                       smem_desc_at(DESC_K, sbase + ks * B_SUB + kk * 32), IDESC, (ks | kk) != 0);
          mma_commit(&a_empty[st]);
        }
        mma_commit(&acc_full[buf]);
      }
    }
  } else {
    // epilogue: thread == row of the tile == TMEM lane; each warp owns 32 rows and a 4 KB staging block
    const int r = warp * 32 + lane;
    const uint32_t lane_base = (uint32_t)(warp * 32) << 16;
    uint8_t *stg0 = smem + off_stg + warp * (NSTG * 4096);
    float *sbias = reinterpret_cast<float *>(smem + off_bias);      // this column tile's bias: the L1 is tiny beside 220 KB of shared memory
    for (int i = threadIdx.x; i < BN; i += 128) sbias[i] = p.bias ? __ldg(p.bias + nt * BN + i) : 0.f;
    named_bar_sync(1, 128);
    int t = 0, sb = 0;                                              // sb: staging block in use
    for (int mt = m0; mt < p.m_tiles; mt += m_stride, ++t) {
      const int buf = t & 1;
      mbar_wait(&acc_full[buf], (t >> 1) & 1);
      tc_fence_after();
      if constexpr (OUT == POUT_IMG16) {
        if (p.onehot_sub >= 0 && nt == 0) {
          // extra K columns for the next GEMM: one-hot(frame position) twice (against the hi and lo halves of the
          // positional-encoding / bias table), so that the table is added by the tensor core (model.py:27,75-78)
          uint8_t *dst = reinterpret_cast<uint8_t *>(p.c_img) + ((size_t)mt * p.c_nk + p.onehot_sub) * A_SUB;
          const int tt = r & 15;
#pragma unroll
          for (int ch = 0; ch < 8; ++ch) {
            uint4 pk = make_uint4(0u, 0u, 0u, 0u);
            if (ch == (tt >> 3) || ch == 2 + (tt >> 3)) {
              const uint32_t one = 0x3C00u << (16 * (tt & 1));
              const int w = (tt & 7) >> 1;
              pk.x = w == 0 ? one : 0u; pk.y = w == 1 ? one : 0u; pk.z = w == 2 ? one : 0u; pk.w = w == 3 ? one : 0u;
            }
            *reinterpret_cast<uint4 *>(dst + sw128_offset(r, ch * 8)) = pk;
          }
        }
      }
#pragma unroll 1
      for (int c0 = 0; c0 < BN; c0 += 32) {
        uint32_t v[32];
        tmem_ld32(tmem + lane_base + buf * 256 + c0, v);
        const bool first = OUT == POUT_F32C || (c0 & 32) == 0;       // first chunk of a staging block: the bulk store
        if (first) {                                                  // issued NSTG blocks ago must have left it
          if (lane == 0) bulk_wait_read<NSTG - 1>();
          __syncwarp();
        }
        uint8_t *stg = stg0 + sb * 4096;
        uint8_t *srow = stg + lane * 128;
        tmem_ld_wait();
        if (c0 + 32 >= BN) {                                          // accumulator drained: the MMA warp may reuse it
          tc_fence_before();
          mbar_arrive(&acc_empty[buf]);
        }
        const int col0 = nt * BN + c0;
        if constexpr (OUT == POUT_F32C) {
#pragma unroll
          for (int j = 0; j < 8; ++j)
            *reinterpret_cast<uint4 *>(srow + ((j ^ (lane & 7)) << 4)) = make_uint4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
          fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) {
            float *dst = p.gc + (((size_t)mt * (p.n_tiles * (BN / 32)) + (col0 >> 5)) * 128 + warp * 32) * 32;
            bulk_s2g(dst, stg, 4096);
            bulk_commit();
          }
          sb = (sb + 1) % NSTG;
        } else {
          float x[32];
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            float tv = __uint_as_float(v[j]) + sbias[c0 + j];
            if (p.act == ARX_ACT_RELU) tv = fmaxf(tv, 0.f);
            x[j] = tv;
          }
#pragma unroll
          for (int ch = 0; ch < 4; ++ch) {
            uint4 pk;
            __half2 h0 = __floats2half2_rn(x[ch * 8 + 0], x[ch * 8 + 1]), h1 = __floats2half2_rn(x[ch * 8 + 2], x[ch * 8 + 3]);
            __half2 h2 = __floats2half2_rn(x[ch * 8 + 4], x[ch * 8 + 5]), h3 = __floats2half2_rn(x[ch * 8 + 6], x[ch * 8 + 7]);
            pk.x = *reinterpret_cast<uint32_t *>(&h0); pk.y = *reinterpret_cast<uint32_t *>(&h1);
            pk.z = *reinterpret_cast<uint32_t *>(&h2); pk.w = *reinterpret_cast<uint32_t *>(&h3);
            const int chunk = ((c0 & 32) >> 3) + ch;                  // 16-byte chunk of the 64-column sub-tile row
            *reinterpret_cast<uint4 *>(srow + ((chunk ^ (lane & 7)) << 4)) = pk;
          }
          if ((c0 & 32) != 0 || c0 + 32 >= BN) {                      // sub-tile complete
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) {
              uint8_t *dst = reinterpret_cast<uint8_t *>(p.c_img) + ((size_t)mt * p.c_nk + (col0 >> 6)) * A_SUB + warp * 4096;
              bulk_s2g(dst, stg, 4096);
              bulk_commit();
            }
            sb = (sb + 1) % NSTG;
          }
        }
      }
    }
    if (lane == 0) bulk_wait_all();
    tc_fence_before();
  }
  __syncthreads();
  if (warp == 5) { tc_fence_after(); tmem_dealloc(tmem, 512); }
}

// ------------------------------------------------------------------------------------------------ tuple images
constexpr int TI_STRIDE = 260;        // padded frame row (floats): 16 distinct rows hit every bank group twice, no worse

__constant__ int c_pslots[256];       // frame pair of every internal slot, -1 = pad

struct TupleParams {
  float gs[256];            // gamma*alpha [128] | beta*alpha [128]: read as constant-bank operands, not through the LSU
  const float *gc;
  __half *kq_img;
  int n_chunks, n_win;
};

// 256 threads: thread (slot s = tid & 127, HALF = tid >> 7) owns 64 of the 128 dimensions of tuple row s -- 16 warps
// per SM at <= 128 registers instead of 8 at 255.  HALF is warp-uniform and a template parameter of the body, so the
// LayerNorm affine stays a compile-time constant-bank operand; the two halves of a row exchange their sums of
// squares through shared memory under a barrier the loop needs anyway.
template <int HALF>
__device__ __forceinline__ void tuple_body(const TupleParams &p, const float *stg, float *sq, uint8_t *img0, int fi, int fj, bool live, int s,
                                           int it, int win) {
  const float4 *A = reinterpret_cast<const float4 *>(stg + (live ? fi : 0) * TI_STRIDE + HALF * 64);
  const float4 *B = reinterpret_cast<const float4 *>(stg + (live ? fj : 0) * TI_STRIDE + 128 + HALF * 64);
  uint64_t x[32];
  uint64_t q0 = 0ull, q1 = 0ull;
#pragma unroll
  for (int c = 0; c < 16; ++c) {
    const float4 a = A[c], b = B[c];
    x[2 * c] = add2(pack2(a.x, a.y), pack2(b.x, b.y));
    x[2 * c + 1] = add2(pack2(a.z, a.w), pack2(b.z, b.w));
    q0 = fma2(x[2 * c], x[2 * c], q0);
    q1 = fma2(x[2 * c + 1], x[2 * c + 1], q1);
  }
  float ql, qh;
  unpack2(add2(q0, q1), ql, qh);
  sq[HALF * 128 + s] = ql + qh;
  if (threadIdx.x == 0) bulk_wait_read<1>();        // the store that used this image buffer two windows ago has left it
  named_bar_sync(1, 256);                           // ... everybody is done with the staged rows, partial sums visible
  const float rstd = live ? rsqrtf((sq[s] + sq[128 + s]) * (1.0f / 128.0f) + 1e-5f) : 0.f;
  const uint64_t rr = pack2(rstd, rstd);
  uint8_t *img = img0 + (it & 1) * 32768;
  uint8_t *irow = img + HALF * 16384 + (s >> 3) * 1024 + (s & 7) * 128;
#pragma unroll
  for (int c = 0; c < 8; ++c) {
    uint32_t h[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      constexpr int D0 = HALF * 64;
      float lo, hi;
      unpack2(mul2(x[c * 4 + k], rr), lo, hi);
      const __half2 hh = __floats2half2_rn(fmaf(lo, p.gs[D0 + c * 8 + 2 * k], p.gs[128 + D0 + c * 8 + 2 * k]),
                                           fmaf(hi, p.gs[D0 + c * 8 + 2 * k + 1], p.gs[128 + D0 + c * 8 + 2 * k + 1]));
      h[k] = live ? *reinterpret_cast<const uint32_t *>(&hh) : 0u;
    }
    *reinterpret_cast<uint4 *>(irow + ((c ^ (s & 7)) << 4)) = make_uint4(h[0], h[1], h[2], h[3]);
  }
  fence_proxy_async_smem();
  named_bar_sync(1, 256);                           // (named: the two HALF bodies are different code paths)
  if (threadIdx.x == 0) {
    bulk_s2g(reinterpret_cast<uint8_t *>(p.kq_img) + (size_t)win * 32768, img, 32768);
    bulk_commit();
  }
}

__global__ void __launch_bounds__(256, 2) k_tuple_img(const __grid_constant__ TupleParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t *smem = smem_raw + ((128u - (smem_u32(smem_raw) & 127u)) & 127u);
  uint8_t *img0 = smem;                                                  // 2 x 32 KB, final swizzled layout
  float *stg = reinterpret_cast<float *>(smem + 65536);                 // [16 frames][260]: K part 1 | K part 2, centred
  float *sq = stg + 16 * TI_STRIDE;                                     // [2 halves][128 slots] partial sums of squares
  const int tid = threadIdx.x, s = tid & 127;
  const int fi = c_pslots[2 * s], fj = c_pslots[2 * s + 1];
  const bool live = fi >= 0;
  // the window's 16 x 256 K projections: 1024 float4, 4 per thread; a warp covers one (frame, part) per pass, so
  // the LayerNorm mean by linearity (mean(A_i + B_j) = mean(A_i) + mean(B_j)) is one warp reduction.  The loads
  // of the NEXT window are issued before this window's arithmetic (persistent CTA, software pipeline).
  float4 v[4];
  auto fetch = [&](int win) {
    const float4 *src = reinterpret_cast<const float4 *>(p.gc) + (size_t)(win >> 3) * p.n_chunks * 128 * 8;
    const int r0 = (win & 7) * 16;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int idx = k * 256 + tid;                // = frame * 64 + quad,  quad = 16-byte group of the 256 K columns
      const int row = r0 + (idx >> 6), quad = idx & 63;
      v[k] = __ldg(src + ((size_t)(quad >> 3) * 128 + row) * 8 + ((quad & 7) ^ (row & 7)));
    }
  };
  int win = blockIdx.x;
  if (win < p.n_win) fetch(win);
  for (int it = 0; win < p.n_win; win += gridDim.x, ++it) {
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      float sum = (v[k].x + v[k].y) + (v[k].z + v[k].w);
#pragma unroll
      for (int o = 16; o; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
      const float m = sum * (1.0f / 128.0f);
      const int idx = k * 256 + tid;
      *reinterpret_cast<float4 *>(stg + (idx >> 6) * TI_STRIDE + (idx & 63) * 4) = make_float4(v[k].x - m, v[k].y - m, v[k].z - m, v[k].w - m);
    }
    __syncthreads();
    if (win + (int)gridDim.x < p.n_win) fetch(win + gridDim.x);
    if (tid < 128) tuple_body<0>(p, stg, sq, img0, fi, fj, live, s, it, win);
    else tuple_body<1>(p, stg, sq, img0, fi, fj, live, s, it, win);
  }
  if (tid == 0) bulk_wait_all();
}

template <int BN, int OUT, int NSTG> int launch_p(arx_handle *h, GemmPParams &p, int sms, cudaStream_t st) {
  const uint32_t fixed = p.nk * BN * 128 + 4 * NSTG * 4096 + BN * 4 + 256 + 1024;
  const uint32_t cap = 232448;
  int nsta = (int)((cap - fixed) / A_SUB);
  if (nsta > 8) nsta = 8;
  if (nsta < 2) return arx_fail(h, ARX_ERR_INVALID, "gemm_p: weights of this layer do not fit in shared memory (nk=%d BN=%d)", p.nk, BN);
  p.nsta = nsta;
  const uint32_t smem = fixed + nsta * A_SUB;
  auto kern = k_gemm_p<BN, OUT, NSTG>;
  { const int rc_ = arx_func_smem(h, kern, (int)smem); if (rc_) return rc_; }
  int grid = (sms / p.n_tiles) * p.n_tiles;
  if (grid > p.m_tiles * p.n_tiles) grid = p.m_tiles * p.n_tiles;
  kern<<<grid, P_THREADS, smem, st>>>(p);
  ARX_LAUNCH_CHECK(h);
  return ARX_OK;
}

}  // namespace

bool arx_tcp_supported(const ArxTcLinear &L) { return (L.BN == 256 || L.BN == 192) && (size_t)L.nk * L.BN * 128 + 2 * A_SUB + 4 * 4096 + 4096 <= 232448; }

// act(A.W^T + b) -> fp16 activation image with c_nk K-sub-tiles per row tile (persistent kernel on `sms` SMs)
int arx_tcp_linear_img(arx_handle *h, const ArxTcLinear &L, const __half *a_img, int64_t M, int act, __half *c_img, int c_nk, int onehot_sub,
                       int sms, cudaStream_t st) {
  GemmPParams p{};
  p.a_img = a_img; p.w_img = L.w_img; p.bias = L.bias; p.nk = L.nk; p.a_nk = L.nk; p.m_tiles = (int)((M + 127) / 128); p.n_tiles = L.n_tiles;
  p.act = act; p.c_img = c_img; p.c_nk = c_nk; p.onehot_sub = onehot_sub;
  if (L.BN == 192) return launch_p<192, POUT_IMG16, 4>(h, p, sms, st);
  if (L.BN == 256) return launch_p<256, POUT_IMG16, 4>(h, p, sms, st);
  return arx_fail(h, ARX_ERR_INVALID, "tcp_linear_img: unsupported BN %d", L.BN);
}

// A.W^T -> chunked fp32 projections Gc (see the file header); the buffer holds ceil(M/128)*128 rows
int arx_tcp_linear_chunked(arx_handle *h, const ArxTcLinear &L, const __half *a_img, int a_nk, int64_t M, float *gc, int sms, cudaStream_t st) {
  GemmPParams p{};
  p.a_img = a_img; p.w_img = L.w_img; p.bias = nullptr; p.nk = L.nk; p.a_nk = a_nk; p.m_tiles = (int)((M + 127) / 128); p.n_tiles = L.n_tiles;
  p.act = ARX_ACT_NONE; p.gc = gc; p.onehot_sub = -1;
  if (L.BN == 256) return launch_p<256, POUT_F32C, 1>(h, p, sms, st);
  return arx_fail(h, ARX_ERR_INVALID, "tcp_linear_chunked: unsupported BN %d", L.BN);
}

// Kq operand images of n_win query windows from the chunked per-frame K projections (T=16 pair tuples, slot order)
int arx_tuple_img(arx_handle *h, const ArxTransformer &tr, const float *gc, int n_chunks, int64_t n_win, __half *kq_img, float alpha,
                  int sms, cudaStream_t st) {
  if (!(h->dev_init & ARX_INIT_PSLOTS)) {         // __constant__ symbols are per device: once per handle, not per process
    int32_t slots[256];
    arx_tc2_slot_table(slots);
    ARX_CUDA(h, cudaMemcpyToSymbol(c_pslots, slots, sizeof(slots)));
    h->dev_init |= ARX_INIT_PSLOTS;
  }
  const uint32_t smem = 65536 + 16 * TI_STRIDE * 4 + 1024 + 128;
  { const int rc_ = arx_func_smem(h, k_tuple_img, (int)smem); if (rc_) return rc_; }
  const int64_t grid = n_win < 2 * sms ? n_win : 2 * sms;
  TupleParams p{};
  for (int d = 0; d < 128; ++d) { p.gs[d] = tr.ln_host[d] * alpha; p.gs[128 + d] = tr.ln_host[128 + d] * alpha; }
  p.gc = gc; p.kq_img = kq_img; p.n_chunks = n_chunks; p.n_win = (int)n_win;
  k_tuple_img<<<(unsigned)grid, 256, smem, st>>>(p);
  ARX_LAUNCH_CHECK(h);
  return ARX_OK;
}

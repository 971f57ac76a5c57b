// tcgen05 GEMM for the per-frame linear layers and the discriminator MLP:
//   C[M,N] = act(A[M,K] . W[N,K]^T + bias)       fp16 operands, fp32 accumulation in TMEM
// (reference: MLP.forward model.py:175-180, k_linear/v_linear model.py:75-78 after folding the positional
//  encoding into a per-position bias table, Discriminator.forward model.py:197-203).
//
// Both operands live in HBM as pre-swizzled "images": [tile][k_sub][rows x 64 fp16, K-major SW128], so a
// 128x64 A block and a BNx64 W block are each ONE bulk copy into shared memory, directly usable by
// tcgen05.mma.  Producers of activations (this kernel's epilogue, the head kernel, k_rows_to_img) write
// that layout.  One CTA = one 128-row tile x one BN-column tile; 2 CTAs per SM overlap epilogue and mainloop.
#include "arx_internal.cuh"
#include "arx_ptx.cuh"

namespace {
using namespace ptx;

constexpr uint32_t A_SUB = 128 * 128;       // 128 rows x 64 fp16
constexpr int G_THREADS = 192;

enum { OUT_IMG16 = 0, OUT_F32 = 1, OUT_SIGMOID_DOT = 2 };

struct GemmParams {
  const __half *a_img;     // [m_tiles][nk][128 x 64]
  const __half *w_img;     // [n_tiles][nk][BN x 64]
  const float *bias;       // [n_tiles*BN] (zero padded) or null
  int nk;                  // K sub-tiles of 64 consumed by this GEMM
  int a_nk;                // sub-tiles per row tile of the A image (>= nk)
  int onehot_sub;          // OUT_IMG16: also write a one-hot(row % 16) sub-tile at this index of c_img (-1 = no)
  int64_t M;               // valid rows
  int act;                 // ARX_ACT_*
  // OUT_IMG16
  __half *c_img;           // [m_tiles][c_nk][128 x 64]
  int c_nk;
  // OUT_F32
  float *c;                // [M][ldc]
  int ldc, n_valid;
  const float *table;      // [T][ldc] added after activation (row % T), or null
  int T;
  // OUT_SIGMOID_DOT
  const float *w3, *b3;    // [BN], [1]
  float *out1;             // [M]
};

template <int BN, int OUT, int NST>
__global__ void __launch_bounds__(G_THREADS, 2) k_gemm_tc(const GemmParams p) {
  constexpr uint32_t B_SUB = BN * 128;
  constexpr uint32_t STAGE = A_SUB + B_SUB;
  constexpr uint32_t TM_COLS = BN <= 64 ? 64 : (BN <= 128 ? 128 : 256);
  extern __shared__ uint8_t smem_raw[];
  uint8_t *smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  constexpr uint32_t BAR_OFF = NST * STAGE;
  uint64_t *bars = reinterpret_cast<uint64_t *>(smem + BAR_OFF);     // full[NST], empty[NST], acc
  uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(smem + BAR_OFF + (2 * NST + 1) * 8);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int mt = blockIdx.x, nt = blockIdx.y;
  if (threadIdx.x == 0) {
    for (int i = 0; i < 2 * NST + 1; ++i) mbar_init(&bars[i], 1);
    mbar_init_fence();
  }
  pdl_trigger();
  if (warp == 5) { tmem_alloc(tmem_slot, TM_COLS); tmem_relinquish(); }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  pdl_wait();                       // everything above overlapped the previous kernel's tail

  if (warp == 4) {
    if (elect_one()) {
      const uint8_t *a = reinterpret_cast<const uint8_t *>(p.a_img) + (size_t)mt * p.a_nk * A_SUB;
      const uint8_t *w = reinterpret_cast<const uint8_t *>(p.w_img) + (size_t)nt * p.nk * B_SUB;
      for (int ks = 0; ks < p.nk; ++ks) {
        const int st = ks % NST;
        mbar_wait(&bars[NST + st], ((ks / NST) & 1) ^ 1);
        mbar_arrive_expect_tx(&bars[st], STAGE);
        bulk_g2s(smem + st * STAGE, a + (size_t)ks * A_SUB, A_SUB, &bars[st]);
        bulk_g2s(smem + st * STAGE + A_SUB, w + (size_t)ks * B_SUB, B_SUB, &bars[st]);
      }
    }
  } else if (warp == 5) {
    if (elect_one()) {
      constexpr uint64_t DESC_K = smem_desc_sw128(16, 1024);
      constexpr uint32_t IDESC = idesc_f16(128, BN, 0, 0);
      const uint32_t sbase = smem_u32(smem);
      for (int ks = 0; ks < p.nk; ++ks) {
        const int st = ks % NST;
        mbar_wait(&bars[st], (ks / NST) & 1);
        tc_fence_after();
#pragma unroll
        for (int kk = 0; kk < 4; ++kk)
          mma_f16_ss(tmem, smem_desc_at(DESC_K, sbase + st * STAGE + kk * 32), smem_desc_at(DESC_K, sbase + st * STAGE + A_SUB + kk * 32),
                     IDESC, (ks | kk) != 0);
        mma_commit(&bars[NST + st]);
      }
      mma_commit(&bars[2 * NST]);
    }
  } else {
    // epilogue: thread == row of the tile == TMEM lane
    const int r = warp * 32 + lane;
    const int64_t row = (int64_t)mt * 128 + r;
    const uint32_t lane_base = (uint32_t)(warp * 32) << 16;
    mbar_wait(&bars[2 * NST], 0);
    tc_fence_after();
    float dot = 0.f;
    if constexpr (OUT == OUT_IMG16) {
      if (p.onehot_sub >= 0 && nt == 0) {
        // extra K columns for the next GEMM: one-hot(frame position) twice (against the hi and lo halves of the
        // positional-encoding / bias table), so that the table is added by the tensor core (model.py:27,75-78)
        uint8_t *dst = reinterpret_cast<uint8_t *>(p.c_img) + ((size_t)mt * p.c_nk + p.onehot_sub) * A_SUB;
        const int t = r & 15;
#pragma unroll
        for (int ch = 0; ch < 8; ++ch) {
          uint4 pk = make_uint4(0u, 0u, 0u, 0u);
          if (ch == (t >> 3) || ch == 2 + (t >> 3)) {
            const uint32_t one = 0x3C00u << (16 * (t & 1));         // fp16 1.0 in the low or high half
            const int w = (t & 7) >> 1;
            pk.x = w == 0 ? one : 0u; pk.y = w == 1 ? one : 0u; pk.z = w == 2 ? one : 0u; pk.w = w == 3 ? one : 0u;
          }
          *reinterpret_cast<uint4 *>(dst + sw128_offset(r, ch * 8)) = pk;
        }
      }
    }
#pragma unroll 1
    for (int c0 = 0; c0 < BN; c0 += 32) {
      uint32_t v[32];
      tmem_ld32(tmem + lane_base + c0, v);
      tmem_ld_wait();
      const int col0 = nt * BN + c0;
      float x[32];
#pragma unroll
      for (int j = 0; j < 32; ++j) {
        float t = __uint_as_float(v[j]) + (p.bias ? __ldg(p.bias + col0 + j) : 0.f);
        if (p.act == ARX_ACT_RELU) t = fmaxf(t, 0.f);
        x[j] = t;
      }
      if constexpr (OUT == OUT_IMG16) {
        // next layer's A image: this tile's columns are K of the next GEMM
        uint8_t *dst = reinterpret_cast<uint8_t *>(p.c_img) + ((size_t)mt * p.c_nk + (col0 >> 6)) * A_SUB;
#pragma unroll
        for (int ch = 0; ch < 4; ++ch) {
          uint4 pk;
          __half2 h0 = __floats2half2_rn(x[ch * 8 + 0], x[ch * 8 + 1]), h1 = __floats2half2_rn(x[ch * 8 + 2], x[ch * 8 + 3]);
          __half2 h2 = __floats2half2_rn(x[ch * 8 + 4], x[ch * 8 + 5]), h3 = __floats2half2_rn(x[ch * 8 + 6], x[ch * 8 + 7]);
          pk.x = *reinterpret_cast<uint32_t *>(&h0); pk.y = *reinterpret_cast<uint32_t *>(&h1);
          pk.z = *reinterpret_cast<uint32_t *>(&h2); pk.w = *reinterpret_cast<uint32_t *>(&h3);
          *reinterpret_cast<uint4 *>(dst + sw128_offset(r, (col0 & 63) + ch * 8)) = pk;
        }
      } else if constexpr (OUT == OUT_F32) {
        if (row < p.M) {
          float *dst = p.c + row * (int64_t)p.ldc + col0;
          const float *tb = p.table ? p.table + (int64_t)(row % p.T) * p.ldc + col0 : nullptr;
#pragma unroll
          for (int j = 0; j < 32; j += 4) {
            if (col0 + j < p.n_valid) {
              float4 o = make_float4(x[j], x[j + 1], x[j + 2], x[j + 3]);
              if (tb) {
                const float4 tv = __ldg(reinterpret_cast<const float4 *>(tb + j));
                o.x += tv.x; o.y += tv.y; o.z += tv.z; o.w += tv.w;
              }
              *reinterpret_cast<float4 *>(dst + j) = o;
            }
          }
        }
      } else {
#pragma unroll
        for (int j = 0; j < 32; ++j) dot = fmaf(x[j], __ldg(p.w3 + col0 + j), dot);
      }
    }
    if constexpr (OUT == OUT_SIGMOID_DOT) {
      if (row < p.M) p.out1[row] = 1.f / (1.f + expf(-(dot + __ldg(p.b3))));
    }
    tc_fence_before();
  }
  __syncthreads();
  if (warp == 5) { tc_fence_after(); tmem_dealloc(tmem, TM_COLS); }
}

// fp32 (or fp16) row-major [M][lda] (K valid columns) -> fp16 activation image [ceil(M/128)][nk][128 x 64]; zero padded.
template <class TIn>
__global__ void __launch_bounds__(256) k_rows_to_img(const TIn *__restrict__ X, int lda, int K, int64_t M, __half *__restrict__ img, int nk,
                                                     int onehot_sub) {
  pdl_trigger();
  pdl_wait();
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;     // one 8-column chunk per thread
  const int chunks_per_row = nk * 8;
  const int64_t total = ((M + 127) / 128) * 128 * chunks_per_row;
  if (idx >= total) return;
  const int64_t row = idx / chunks_per_row;
  const int ch = (int)(idx % chunks_per_row);
  float x[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int k = ch * 8 + i;
    x[i] = (row < M && k < K) ? (float)X[row * (int64_t)lda + k] : 0.f;
    if (onehot_sub >= 0 && (ch >> 3) == onehot_sub) {          // one-hot(row % 16) at columns t and 16 + t of this sub-tile
      const int c = (ch & 7) * 8 + i;
      x[i] = (c < 32 && (c & 15) == (int)(row & 15)) ? 1.f : 0.f;
    }
  }
  uint4 pk;
  __half2 h0 = __floats2half2_rn(x[0], x[1]), h1 = __floats2half2_rn(x[2], x[3]), h2 = __floats2half2_rn(x[4], x[5]), h3 = __floats2half2_rn(x[6], x[7]);
  pk.x = *reinterpret_cast<uint32_t *>(&h0); pk.y = *reinterpret_cast<uint32_t *>(&h1);
  pk.z = *reinterpret_cast<uint32_t *>(&h2); pk.w = *reinterpret_cast<uint32_t *>(&h3);
  const int64_t mt = row >> 7;
  const int r = (int)(row & 127), ks = ch >> 3, c = (ch & 7) * 8;
  *reinterpret_cast<uint4 *>(reinterpret_cast<uint8_t *>(img) + ((size_t)mt * nk + ks) * A_SUB + sw128_offset(r, c)) = pk;
}

// fp32 weight [N][ldw] (K valid columns) -> fp16 image [n_tiles][nk][BN x 64]; zero padded.
__global__ void __launch_bounds__(256) k_weight_to_img(const float *__restrict__ W, int ldw, int N, int K, __half *__restrict__ img, int BN,
                                                       int n_tiles, int nk) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t total = (int64_t)n_tiles * BN * nk * 8;
  if (idx >= total) return;
  const int ch = (int)(idx % (nk * 8));
  const int64_t nrow = idx / (nk * 8);
  const int nt = (int)(nrow / BN), r = (int)(nrow % BN);
  float x[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int k = ch * 8 + i;
    x[i] = (nrow < N && k < K) ? W[nrow * (int64_t)ldw + k] : 0.f;
  }
  uint4 pk;
  __half2 h0 = __floats2half2_rn(x[0], x[1]), h1 = __floats2half2_rn(x[2], x[3]), h2 = __floats2half2_rn(x[4], x[5]), h3 = __floats2half2_rn(x[6], x[7]);
  pk.x = *reinterpret_cast<uint32_t *>(&h0); pk.y = *reinterpret_cast<uint32_t *>(&h1);
  pk.z = *reinterpret_cast<uint32_t *>(&h2); pk.w = *reinterpret_cast<uint32_t *>(&h3);
  const int ks = ch >> 3, c = (ch & 7) * 8;
  *reinterpret_cast<uint4 *>(reinterpret_cast<uint8_t *>(img) + ((size_t)nt * nk + ks) * ((size_t)BN * 128) + sw128_offset(r, c)) = pk;
}

// row sums of the (T, ld) positional-encoding/bias table over columns [0,128) and [128,256)
__global__ void k_table_sums(const float *__restrict__ table, int ld, float *__restrict__ out) {
  const int t = blockIdx.x, part = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float s = 0.f;
  for (int c = lane; c < 128; c += 32) s += table[(int64_t)t * ld + part * 128 + c];
#pragma unroll
  for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if (lane == 0) out[t * 2 + part] = s;
}

// extended projection weight (N, F+32): [ wp | hi(table)^T | lo(table)^T ] with hi = fp16(table), lo = table - hi
__global__ void k_build_wp_ext(const float *__restrict__ wp, const float *__restrict__ table, float *__restrict__ out, int N, int F) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  const int ld = F + 32;
  if (idx >= N * ld) return;
  const int n = idx / ld, c = idx % ld;
  float v;
  if (c < F) v = wp[(size_t)n * F + c];
  else {
    const int t = (c - F) & 15;
    const float x = table[(size_t)t * N + n];
    const float hi = __half2float(__float2half_rn(x));
    v = (c - F) < 16 ? hi : x - hi;
  }
  out[idx] = v;
}

__global__ void k_pad_bias(const float *__restrict__ b, int N, float *__restrict__ out, int Npad) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < Npad) out[i] = (b && i < N) ? b[i] : 0.f;
}

template <int BN, int OUT, int NST = 2> int launch_gemm(arx_handle *h, const GemmParams &p, int n_tiles, cudaStream_t st) {
  constexpr uint32_t body = NST * (A_SUB + BN * 128);
  constexpr uint32_t smem = body + (2 * NST + 1) * 8 + 16 + 1024;
  auto kern = k_gemm_tc<BN, OUT, NST>;
  { const int rc_ = arx_func_smem(h, kern, (int)smem); if (rc_) return rc_; }
  dim3 grid((unsigned)((p.M + 127) / 128), (unsigned)n_tiles);
  ARX_CUDA(h, arx_launch_pdl(kern, grid, dim3(G_THREADS), smem, st, h->pdl, p));
  h->launches++;
  return ARX_OK;
}

}  // namespace

int arx_tc_linear_prepare(arx_handle *h, ArxTcLinear &L, const float *W, int ldw, const float *bias, int N, int K, int BN, cudaStream_t st) {
  L.N = N; L.K = K; L.BN = BN; L.n_tiles = (N + BN - 1) / BN; L.nk = (K + 63) / 64;
  const size_t wbytes = (size_t)L.n_tiles * L.nk * BN * 128;
  if (!L.w_img) ARX_CUDA(h, cudaMalloc(reinterpret_cast<void **>(&L.w_img), wbytes));
  if (!L.bias) ARX_CUDA(h, cudaMalloc(reinterpret_cast<void **>(&L.bias), (size_t)L.n_tiles * BN * sizeof(float)));
  const int64_t total = (int64_t)L.n_tiles * BN * L.nk * 8;
  k_weight_to_img<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(W, ldw, N, K, L.w_img, BN, L.n_tiles, L.nk);
  ARX_LAUNCH_CHECK(h);
  k_pad_bias<<<(L.n_tiles * BN + 255) / 256, 256, 0, st>>>(bias, N, L.bias, L.n_tiles * BN);
  ARX_LAUNCH_CHECK(h);
  return ARX_OK;
}

int arx_tc_rows_to_img(arx_handle *h, const void *X, bool f16, int lda, int K, int64_t M, __half *img, int nk, int onehot_sub, cudaStream_t st) {
  const int64_t total = ((M + 127) / 128) * 128 * nk * 8;
  if (f16) {          // fp16 rows (arx_score_host*_f16): same image, no rounding step
    k_rows_to_img<__half><<<(unsigned)((total + 255) / 256), 256, 0, st>>>(static_cast<const __half *>(X), lda, K, M, img, nk, onehot_sub);
    ARX_LAUNCH_CHECK(h);
    return ARX_OK;
  }
  ARX_CUDA(h, arx_launch_pdl(k_rows_to_img<float>, dim3((unsigned)((total + 255) / 256)), dim3(256), 0, st, h->pdl,
                             static_cast<const float *>(X), lda, K, M, img, nk, onehot_sub));
  h->launches++;
  return ARX_OK;
}

// act(A.W^T + b) -> fp16 activation image with c_nk K-sub-tiles per row tile
int arx_tc_linear_img(arx_handle *h, const ArxTcLinear &L, const __half *a_img, int64_t M, int act, __half *c_img, int c_nk, int onehot_sub,
                      cudaStream_t st) {
  GemmParams p{};
  p.a_img = a_img; p.w_img = L.w_img; p.bias = L.bias; p.nk = L.nk; p.a_nk = L.nk; p.M = M; p.act = act; p.c_img = c_img; p.c_nk = c_nk;
  p.onehot_sub = onehot_sub;
  if (L.BN == 192) return launch_gemm<192, OUT_IMG16>(h, p, L.n_tiles, st);
  if (L.BN == 256) return launch_gemm<256, OUT_IMG16>(h, p, L.n_tiles, st);
  if (L.BN == 64) return launch_gemm<64, OUT_IMG16, 4>(h, p, L.n_tiles, st);     // deep-K layers: 4x the CTAs, 4-stage ring
  return arx_fail(h, ARX_ERR_INVALID, "tc_linear_img: unsupported BN %d", L.BN);
}

// A.W^T (+ table[row % T]) -> fp32 row-major
int arx_tc_linear_f32(arx_handle *h, const ArxTcLinear &L, const __half *a_img, int a_nk, int64_t M, float *C, int ldc, const float *table, int T,
                      cudaStream_t st, bool with_bias) {
  GemmParams p{};
  p.a_img = a_img; p.w_img = L.w_img; p.bias = with_bias ? L.bias : nullptr; p.nk = L.nk; p.a_nk = a_nk; p.M = M; p.act = ARX_ACT_NONE; p.c = C; p.ldc = ldc; p.n_valid = L.N;
  p.table = table; p.T = T;
  if (L.BN == 256) return launch_gemm<256, OUT_F32>(h, p, L.n_tiles, st);
  return arx_fail(h, ARX_ERR_INVALID, "tc_linear_f32: unsupported BN %d", L.BN);
}

// sigmoid(relu(A.W^T + b) . w3 + b3) -> out[M]     (discriminator fc2 + fc3, model.py:200-203)
int arx_tc_linear_sigmoid_dot(arx_handle *h, const ArxTcLinear &L, const __half *a_img, int64_t M, const float *w3, const float *b3, float *out,
                              cudaStream_t st) {
  GemmParams p{};
  p.a_img = a_img; p.w_img = L.w_img; p.bias = L.bias; p.nk = L.nk; p.a_nk = L.nk; p.M = M; p.act = ARX_ACT_RELU; p.w3 = w3; p.b3 = b3; p.out1 = out;
  if (L.BN == 64) return launch_gemm<64, OUT_SIGMOID_DOT>(h, p, 1, st);
  return arx_fail(h, ARX_ERR_INVALID, "tc_linear_sigmoid_dot: unsupported BN %d", L.BN);
}

// Fused K/V projection for T=16 pair tuples: Kq images (tuple gather + LayerNorm + scale, internal slot order)
// and the fp32 V projections [M][256], straight from the GEMM accumulator -- no `G` round trip.
int arx_tc_table_sums(arx_handle *h, const float *table, int T, int ld, float *out, cudaStream_t st) {
  k_table_sums<<<T, 64, 0, st>>>(table, ld, out);
  ARX_LAUNCH_CHECK(h);
  return ARX_OK;
}

// A.W^T + table[row % T] -> fp32 row-major for a narrow (32-column) layer
int arx_tc_linear_f32_small(arx_handle *h, const ArxTcLinear &L, const __half *a_img, int a_nk, int64_t M, float *C, int ldc, const float *table,
                            int T, cudaStream_t st) {
  GemmParams p{};
  p.a_img = a_img; p.w_img = L.w_img; p.bias = nullptr; p.nk = L.nk; p.a_nk = a_nk; p.M = M; p.act = ARX_ACT_NONE; p.c = C; p.ldc = ldc; p.n_valid = L.N;
  p.table = table; p.T = T;
  if (L.BN == 32) return launch_gemm<32, OUT_F32>(h, p, L.n_tiles, st);
  return arx_fail(h, ARX_ERR_INVALID, "tc_linear_f32_small: unsupported BN %d", L.BN);
}

int arx_tc_build_wp_ext(arx_handle *h, const float *wp, const float *table, float *out, int N, int F, cudaStream_t st) {
  const int total = N * (F + 32);
  k_build_wp_ext<<<(total + 255) / 256, 256, 0, st>>>(wp, table, out, N, F);
  ARX_LAUNCH_CHECK(h);
  return ARX_OK;
}

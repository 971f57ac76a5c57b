// Resident streaming scorer (reference modules/ar/ar.py:30-84, caller main.py:111): one camera frame per call.
// The reference re-embeds and re-projects all T frames of the sliding window on every call.  With the projection
// factorised per frame (SURVEY 8 a4) only ONE of the T frames is new: its MLP features and its position-INDEPENDENT
// projections W.f (K parts, V parts) are computed once and kept in a device ring buffer; the window's per-frame
// projections are then  G[t] = ring[(oldest + t) mod T] + table[t]  with table[t] = pe[t].W + bias (the positional
// encoding through the projection, arx_load_weights), and the window is scored by the tiled tcgen05 kernels.
// Three small kernels live here; the orchestration (CUDA graph per frame, pinned staging) is in arx_api.cu.
#include "arx_internal.cuh"
#include "arx_ptx.cuh"

namespace {
using namespace ptx;

constexpr int SF_THREADS = 512;

// rows [r0, r1) of y = act(W x + b), K <= 256: one warp per FOUR rows at a time with every load of the four rows issued
// before the first use (32 independent loads per lane: at one frame per call everything here is latency, not bandwidth);
// x in shared memory
__device__ __forceinline__ void warp_matvec4(const float *__restrict__ W, int ldw, const float *__restrict__ bias, const float *x_s, float *y,
                                             int r0, int r1, int K, bool relu) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  float xv[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) xv[i] = lane + 32 * i < K ? x_s[lane + 32 * i] : 0.f;
  for (int o = r0 + warp * 4; o < r1; o += nwarps * 4) {
    float wv[4][8];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
#pragma unroll
      for (int i = 0; i < 8; ++i) wv[u][i] = (o + u < r1 && lane + 32 * i < K) ? __ldg(W + (size_t)(o + u) * ldw + lane + 32 * i) : 0.f;
    }
    float a[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      float t0 = 0.f, t1 = 0.f;
#pragma unroll
      for (int i = 0; i < 8; i += 2) { t0 = fmaf(wv[u][i], xv[i], t0); t1 = fmaf(wv[u][i + 1], xv[i + 1], t1); }
      a[u] = t0 + t1;
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
#pragma unroll
      for (int s = 16; s; s >>= 1) a[u] += __shfl_xor_sync(0xffffffffu, a[u], s);
    }
    if (lane < 4 && o + lane < r1) {
      float v = (lane == 0 ? a[0] : lane == 1 ? a[1] : lane == 2 ? a[2] : a[3]) + (bias ? __ldg(bias + o + lane) : 0.f);
      y[o + lane] = relu ? fmaxf(v, 0.f) : v;
    }
  }
}

// New frame -> MLP features (model.py:175-180; every CTA computes them redundantly: 62 K MAC) -> this CTA's slice of the
// position-independent projections (model.py:75-78 without the positional term) -> ring slot *slot_next.
__global__ void __launch_bounds__(SF_THREADS) k_stream_frame(const float *__restrict__ x, const float *__restrict__ w1, const float *__restrict__ b1,
                                                            const float *__restrict__ w2, const float *__restrict__ b2, const float *__restrict__ wp,
                                                            float *__restrict__ ring, const int *__restrict__ slot_next, int J3, int H, int F, int NO) {
  extern __shared__ float sm[];
  float *x_s = sm, *h_s = sm + J3, *f_s = h_s + H;
  for (int i = threadIdx.x; i < J3; i += blockDim.x) x_s[i] = x[i];
  __syncthreads();
  warp_matvec4(w1, J3, b1, x_s, h_s, 0, H, J3, true);
  __syncthreads();
  warp_matvec4(w2, H, b2, h_s, f_s, 0, F, H, true);
  __syncthreads();
  const int per = (NO + gridDim.x - 1) / gridDim.x, o0 = blockIdx.x * per, o1 = min(NO, o0 + per);
  warp_matvec4(wp, F, nullptr, f_s, ring + (size_t)(*slot_next) * NO, o0, o1, F, false);
}


// Window formation + query tiles in one launch.  The window's frame t lives in ring slot (newest + 1 + t) mod T (newest =
// *slot_next, just written); its per-frame projections are ring + table[t] (table = positional encoding through the
// projection + biases).  Every CTA writes a slice of the row-major G (read by the attention epilogue and the head table) and
// eight rows of the LayerNorm-ed, pre-scaled fp16 query tiles (model.py:69-72,75,81): one warp per tuple row.
__global__ void __launch_bounds__(256) k_stream_tiles(const float *__restrict__ ring, const float *__restrict__ table, const uint32_t *__restrict__ tup,
                                                      const float *__restrict__ ln_g, const float *__restrict__ ln_b, const int *__restrict__ slot_next,
                                                      float *__restrict__ G, __half *__restrict__ kq, int T, int c, int N, int D, float alpha) {
  const int newest = *slot_next, NO = 2 * c * D;
  const int total = T * NO, per = (total + gridDim.x - 1) / gridDim.x;
  for (int e = blockIdx.x * per + threadIdx.x; e < min(total, (int)(blockIdx.x + 1) * per); e += blockDim.x) {
    const int t = e / NO, o = e - t * NO;
    G[e] = ring[(size_t)((newest + 1 + t) % T) * NO + o] + __ldg(table + e);
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int q = blockIdx.x * 8 + warp;                       // row of the tiled image: tile q / 128, row q % 128
  uint8_t *out = reinterpret_cast<uint8_t *>(kq) + (size_t)(q >> 7) * IMG_BYTES;
  const int r = q & 127, d0 = lane * 4;
  uint2 packed = make_uint2(0u, 0u);
  if (q < N) {
    const uint32_t tp = __ldg(tup + q);
    float4 k = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int pp = 0; pp < c; ++pp) {
      const int fr = (tp >> (8 * pp)) & 0xff;
      const float4 a = *reinterpret_cast<const float4 *>(ring + (size_t)((newest + 1 + fr) % T) * NO + pp * D + d0);
      const float4 b = __ldg(reinterpret_cast<const float4 *>(table + (size_t)fr * NO + pp * D + d0));
      k.x += a.x + b.x; k.y += a.y + b.y; k.z += a.z + b.z; k.w += a.w + b.w;
    }
    float sm_ = k.x + k.y + k.z + k.w;
#pragma unroll
    for (int s = 16; s; s >>= 1) sm_ += __shfl_xor_sync(0xffffffffu, sm_, s);
    const float mean = sm_ / D;
    const float4 dl = make_float4(k.x - mean, k.y - mean, k.z - mean, k.w - mean);
    float qq = dl.x * dl.x + dl.y * dl.y + dl.z * dl.z + dl.w * dl.w;
#pragma unroll
    for (int s = 16; s; s >>= 1) qq += __shfl_xor_sync(0xffffffffu, qq, s);
    const float rstd = 1.0f / sqrtf(qq / D + 1e-5f);
    const float4 g = __ldg(reinterpret_cast<const float4 *>(ln_g + d0)), be = __ldg(reinterpret_cast<const float4 *>(ln_b + d0));
    packed.x = pack_half2((dl.x * rstd * g.x + be.x) * alpha, (dl.y * rstd * g.y + be.y) * alpha);
    packed.y = pack_half2((dl.z * rstd * g.z + be.z) * alpha, (dl.w * rstd * g.w + be.w) * alpha);
  }
  *reinterpret_cast<uint2 *>(out + (d0 >> 6) * SUB_BYTES + sw128_offset(r, d0 & 63)) = packed;
}

// logits / argmax of ONE window from the distance partials (model.py:131-135,323: first maximum wins), then discriminator
// fc1 (model.py:198) on the winning class's head input: h1 = relu(W1 y + b1), 256 x (N*T).  One warp per output row, the
// row read as independent 16-byte loads (15 per lane at T=16).  Block 0 also publishes the logits.
// K = N*T = T^2 (T-1) / 2 is a multiple of 4 only for T = 0 (mod 4) or T = 1 (mod 8).  For other K the rows of W1 and y start
// at different offsets from a 16-byte boundary: a scalar head brings the row of W1 to its boundary, the body reads it as
// float4 and y as scalars, and a scalar tail ends the row.
__global__ void __launch_bounds__(256) k_stream_fc1(const float *__restrict__ partial, const float *__restrict__ y_all, const float *__restrict__ w,
                                                    const float *__restrict__ b, float *__restrict__ h1, float *__restrict__ logits, int K, int way,
                                                    int N, int has_disc) {
  float best = -INFINITY;
  int bi = 0;
  for (int c = 0; c < way; ++c) {
    const float4 t = __ldg(reinterpret_cast<const float4 *>(partial) + c);
    const float lg = -(((t.x + t.y) + (t.z + t.w)) / (float)N);
    if (blockIdx.x == 0 && threadIdx.x == 0) logits[c] = lg;
    if (lg > best) { best = lg; bi = c; }
  }
  if (!has_disc) return;
  const int lane = threadIdx.x & 31, row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= 256) return;
  float a0 = 0.f, a1 = 0.f;
  if ((K & 3) == 0) {
    const float4 *y = reinterpret_cast<const float4 *>(y_all + (size_t)bi * K);
    const float4 *wr = reinterpret_cast<const float4 *>(w + (size_t)row * K);
#pragma unroll 8
    for (int k = lane; k < K / 4; k += 32) {
      const float4 wv = __ldg(wr + k), yv = __ldg(y + k);
      a0 = fmaf(wv.x, yv.x, fmaf(wv.y, yv.y, a0));
      a1 = fmaf(wv.z, yv.z, fmaf(wv.w, yv.w, a1));
    }
  } else {
    const float *y = y_all + (size_t)bi * K, *wr = w + (size_t)row * K;
    const int hd = (int)((4u - (uint32_t)(((size_t)row * K) & 3u)) & 3u), nb = (K - hd) >> 2;   // w itself is 16-byte aligned
    if (lane < hd) a0 = __ldg(wr + lane) * __ldg(y + lane);
    const float4 *w4 = reinterpret_cast<const float4 *>(wr + hd);
    const float *yb = y + hd;
#pragma unroll 4
    for (int k = lane; k < nb; k += 32) {
      const float4 wv = __ldg(w4 + k);
      const float *yk = yb + 4 * k;
      a0 = fmaf(wv.x, __ldg(yk), fmaf(wv.y, __ldg(yk + 1), a0));
      a1 = fmaf(wv.z, __ldg(yk + 2), fmaf(wv.w, __ldg(yk + 3), a1));
    }
    const int k = hd + 4 * nb + lane;
    if (k < K) a1 = fmaf(__ldg(wr + k), __ldg(y + k), a1);
  }
  float a = a0 + a1;
#pragma unroll
  for (int s = 16; s; s >>= 1) a += __shfl_xor_sync(0xffffffffu, a, s);
  if (lane == 0) h1[row] = fmaxf(a + __ldg(b + row), 0.f);
}

// fc2 + fc3 + sigmoid (model.py:199-203), softmax over the class logits and the packed result (ar.py:77-78); finally the
// ring's slot pointer advances for the next frame.  One CTA.
__global__ void __launch_bounds__(256) k_stream_tail(const float *__restrict__ h1, const float *__restrict__ w2, const float *__restrict__ b2,
                                                     const float *__restrict__ w3, const float *__restrict__ b3, const float *__restrict__ logits,
                                                     float *__restrict__ out, int *__restrict__ slot_next, int way, int T, int has_disc) {
  __shared__ float h1_s[256], h2_s[64];
  if (has_disc) {
    h1_s[threadIdx.x] = h1[threadIdx.x];
    __syncthreads();
    warp_matvec4(w2, 256, b2, h1_s, h2_s, 0, 64, 256, true);
    __syncthreads();
  }
  if (threadIdx.x < 32) {
    float is_true = 0.f;
    if (has_disc) {
      float a = h2_s[threadIdx.x] * __ldg(w3 + threadIdx.x) + h2_s[threadIdx.x + 32] * __ldg(w3 + threadIdx.x + 32);
#pragma unroll
      for (int s = 16; s; s >>= 1) a += __shfl_xor_sync(0xffffffffu, a, s);
      is_true = 1.f / (1.f + expf(-(a + __ldg(b3))));
    }
    if (threadIdx.x == 0) {
      float m = -INFINITY;
      for (int c = 0; c < way; ++c) m = fmaxf(m, logits[c]);
      float sum = 0.f;
      for (int c = 0; c < way; ++c) sum += expf(logits[c] - m);
      for (int c = 0; c < way; ++c) out[c] = expf(logits[c] - m) / sum;
      out[way] = is_true;
      *slot_next = (*slot_next + 1) % T;
    }
  }
}

// Sliding windows over a frame stream (batch form): window w = frames w .. w+T-1.  From the per-frame position-independent
// projections P (n_frames, NO) and head columns U (n_frames, 32) forms every window's per-frame projections
//   G[w*T + t] = P[w + t] + table[t]      (table = positional encoding through the projection + biases)
// in the chunked layout of arx_gemm_p.cu (chunked != 0: [rows/128][NO/32 chunks][128 rows][32 floats], 16-byte groups XOR-
// swizzled by row & 7) or row-major, and  uab[w*T + t] = U[w + t] + tcomp[t].  One thread per (row, 4 columns).
__global__ void __launch_bounds__(256) k_form_windows(const float *__restrict__ P, const float *__restrict__ U, const float *__restrict__ table,
                                                      const float *__restrict__ tcomp, float *__restrict__ G, float *__restrict__ uab, int64_t n_win,
                                                      int T, int NO, int chunked) {
  const int gpr = NO / 4 + (U ? 8 : 0);                         // float4 groups per row: projections, then the 32 head columns
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= n_win * T * gpr) return;
  const int64_t row = idx / gpr;
  const int g4 = (int)(idx - row * gpr);
  const int64_t w = row / T;
  const int t = (int)(row - w * T);
  if (g4 < NO / 4) {
    const int c = g4 * 4;
    const float4 a = __ldg(reinterpret_cast<const float4 *>(P + (w + t) * NO + c));
    const float4 b = __ldg(reinterpret_cast<const float4 *>(table + (size_t)t * NO + c));
    const float4 o = make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w);
    if (chunked) {
      const int64_t tile = row >> 7;
      const int rr = (int)(row & 127), chunk = c >> 5, cc = c & 31;
      float *dst = G + ((size_t)tile * (NO / 32) + chunk) * 4096 + rr * 32 + ((((cc >> 2) ^ (rr & 7)) << 2));
      *reinterpret_cast<float4 *>(dst) = o;
    } else {
      *reinterpret_cast<float4 *>(G + row * NO + c) = o;
    }
  } else {
    const int c = (g4 - NO / 4) * 4;
    const float4 a = __ldg(reinterpret_cast<const float4 *>(U + (w + t) * 32 + c));
    const float4 b = __ldg(reinterpret_cast<const float4 *>(tcomp + (size_t)t * 32 + c));
    *reinterpret_cast<float4 *>(uab + row * 32 + c) = make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w);
  }
}

}  // namespace

int arx_stream_frame_launch(arx_handle *h, const ArxTransformer &tr, const float *x_dev, float *ring, int *slot_next, cudaStream_t st) {
  const int NO = 2 * tr.c * h->D;
  const size_t smem = (size_t)(h->J3 + h->H + h->F) * sizeof(float);
  k_stream_frame<<<16, SF_THREADS, smem, st>>>(x_dev, h->fc1_w, h->fc1_b, h->fc2_w, h->fc2_b, tr.wp, ring, slot_next, h->J3, h->H, h->F, NO);
  ARX_LAUNCH_CHECK(h);
  return ARX_OK;
}

// G (T, 2cD) row-major + the window's query tiles; the ring's newest frame is in slot *slot_next
int arx_stream_tiles_launch(arx_handle *h, const ArxTransformer &tr, const float *ring, const int *slot_next, float *G, __half *kq, cudaStream_t st) {
  const float alpha = ARX_SOFTMAX_LOG2E / sqrtf((float)h->D);
  k_stream_tiles<<<tr.Npad / 8, 256, 0, st>>>(ring, tr.bp, tr.tup_packed, tr.ln_g, tr.ln_b, slot_next, G, kq, h->T, tr.c, tr.N, h->D, alpha);
  ARX_LAUNCH_CHECK(h);
  return ARX_OK;
}

// logits + discriminator MLP for one window + softmax + packed result; advances the ring
int arx_stream_tail_launch(arx_handle *h, const ArxTransformer &tr, const float *partial, const float *y_all, float *h1, float *logits, float *out,
                           int *slot_next, int way, cudaStream_t st) {
  const int disc = h->cfg.has_discriminator ? 1 : 0;
  const int K1 = tr.N * h->T;
  k_stream_fc1<<<disc ? 32 : 1, 256, 0, st>>>(partial, y_all, h->d1_w, h->d1_b, h1, logits, K1, way, tr.N, disc);
  ARX_LAUNCH_CHECK(h);
  k_stream_tail<<<1, 256, 0, st>>>(h1, h->d2_w, h->d2_b, h->d3_w, h->d3_b, logits, out, slot_next, way, h->T, disc);
  ARX_LAUNCH_CHECK(h);
  return ARX_OK;
}

int arx_form_windows_launch(arx_handle *h, const ArxTransformer &tr, const float *P, const float *U, float *G, float *uab, int64_t n_win, bool chunked,
                            cudaStream_t st) {
  const int NO = 2 * tr.c * h->D;
  const int64_t total = n_win * h->T * (NO / 4 + (U ? 8 : 0));
  k_form_windows<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(P, U, tr.bp, tr.tcomp, G, uab, n_win, h->T, NO, chunked ? 1 : 0);
  ARX_LAUNCH_CHECK(h);
  return ARX_OK;
}

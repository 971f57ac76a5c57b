// The Kc / Vc^T class tiles that both tensor-core routes read (ArxTransformer::kc_tiles / vct_tiles): their allocation,
// their builders from the fp32 tuple tensors ks / vs (arx_import_support on either route, set_support on the tiled
// route), and the support side of the T=16 pair pipeline in one launch (tuple gather + LayerNorm + the single class
// tile of every class).  Also the logits / argmax finisher of both routes and the launcher of the pair pipeline's
// cross-attention kernel (arx_tc3.cu).
// Reference semantics (modules/ar/utils/model.py:69-84 for the support side, :130-146 and :323 for the finisher).
#include "arx_internal.cuh"
#include "arx_ptx.cuh"

namespace {
using namespace ptx;

constexpr int TILE = 128;

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

// Support side in ONE launch (model.py:69-84 for the support set): tuple gather, LayerNorm, fp32 K/V tuple tensors
// (general path, export blob) and, with class tiles, the single Kc (fp16) and Vc^T (bf16) tile of every class (N <= 128).
// One block per class.
__global__ void __launch_bounds__(256) k_support_build(const float *__restrict__ G, const int32_t *__restrict__ tuples,
                                                       const float *__restrict__ ln_g, const float *__restrict__ ln_b,
                                                       float *__restrict__ ks, float *__restrict__ vs, __half *__restrict__ kc_tiles,
                                                       __half *__restrict__ vct_tiles, int T, int c, int N, int ldg) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const size_t cls = blockIdx.x;
  const int d0 = lane * 4;
  const float4 g = *reinterpret_cast<const float4 *>(ln_g + d0);
  const float4 be = *reinterpret_cast<const float4 *>(ln_b + d0);
  uint8_t *kc = kc_tiles ? reinterpret_cast<uint8_t *>(kc_tiles) + cls * IMG_BYTES : nullptr;
  uint8_t *vb = vct_tiles ? reinterpret_cast<uint8_t *>(vct_tiles) + cls * IMG_BYTES : nullptr;
  const int rows = kc ? TILE : N;
  for (int r = blockIdx.y * 8 + warp; r < rows; r += 8 * gridDim.y) {
    float4 k = make_float4(0, 0, 0, 0), v = make_float4(0, 0, 0, 0);
    uint2 kpk = make_uint2(0u, 0u);
    if (r < N) {
      for (int pp = 0; pp < c; ++pp) {
        const int fr = tuples[r * c + pp];
        const float *row = G + (cls * T + fr) * (size_t)ldg;
        const float4 a = *reinterpret_cast<const float4 *>(row + pp * DD + d0);
        const float4 b = *reinterpret_cast<const float4 *>(row + (c + pp) * DD + d0);
        k.x += a.x; k.y += a.y; k.z += a.z; k.w += a.w;
        v.x += b.x; v.y += b.y; v.z += b.z; v.w += b.w;
      }
      float sum = k.x + k.y + k.z + k.w;
#pragma unroll
      for (int o = 16; o; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
      const float mean = sum / DD;
      const float4 dl = make_float4(k.x - mean, k.y - mean, k.z - mean, k.w - mean);
      float q = dl.x * dl.x + dl.y * dl.y + dl.z * dl.z + dl.w * dl.w;
#pragma unroll
      for (int o = 16; o; o >>= 1) q += __shfl_xor_sync(0xffffffffu, q, o);
      const float rstd = 1.0f / sqrtf(q / DD + 1e-5f);
      k = make_float4(dl.x * rstd * g.x + be.x, dl.y * rstd * g.y + be.y, dl.z * rstd * g.z + be.z, dl.w * rstd * g.w + be.w);
      *reinterpret_cast<float4 *>(ks + (cls * N + r) * DD + d0) = k;
      *reinterpret_cast<float4 *>(vs + (cls * N + r) * DD + d0) = v;
      kpk.x = pack_half2(k.x, k.y);
      kpk.y = pack_half2(k.z, k.w);
    }
    if (kc) {
      *reinterpret_cast<uint2 *>(kc + (d0 >> 6) * SUB_BYTES + sw128_offset(r, d0 & 63)) = kpk;      // row r (zero beyond N)
      const float vv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
      for (int e = 0; e < 4; ++e) {                                                                 // column r of Vc^T (zero beyond N)
        const uint32_t off = (r >> 6) * SUB_BYTES + sw128_offset(d0 + e, r & 63);
        *reinterpret_cast<__nv_bfloat16 *>(vb + off) = __float2bfloat16_rn(vv[e]);
      }
    }
  }
}

// logits / argmax from the squared-distance partials (n_win*way, 4) of either tensor-core route
__global__ void k_finish_tc(const float *__restrict__ partial, float *__restrict__ logits, int32_t *__restrict__ chosen, int64_t n_win,
                            int way, int N) {
  pdl_trigger();
  pdl_wait();
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

bool arx_tc_supported(const arx_handle *h, const ArxTransformer &tr) {
  // single-tile kernel: N <= 128; exp2 without max-subtraction needs the overflow bound on the LayerNorm affine
  return tr.N <= TILE && h->D == DD && tr.softmax_bound * ARX_SOFTMAX_LOG2E < 100.0f;
}

// the class tiles of transformer tr for way_cap classes, once per support capacity (free_support releases them)
static int class_tiles_alloc(arx_handle *h, ArxTransformer &tr) {
  if (tr.kc_tiles) return ARX_OK;
  const size_t bytes = (size_t)h->way_cap * (tr.Npad / 128) * IMG_BYTES;
  ARX_CUDA(h, cudaMalloc(reinterpret_cast<void **>(&tr.kc_tiles), bytes));
  ARX_CUDA(h, cudaMalloc(reinterpret_cast<void **>(&tr.vct_tiles), bytes));
  return ARX_OK;
}

int arx_tc_class_tiles(arx_handle *h, ArxTransformer &tr, int way, cudaStream_t st) {
  int rc = class_tiles_alloc(h, tr);
  if (rc) return rc;
  const int ns = tr.Npad / 128;
  k_prep_kc_tiles<<<dim3(way, ns), 256, 0, st>>>(tr.ks, tr.kc_tiles, tr.N, ns);
  ARX_LAUNCH_CHECK(h);
  k_prep_vct_tiles<<<dim3(way, ns), 256, 0, st>>>(tr.vs, tr.vct_tiles, tr.N, ns);
  ARX_LAUNCH_CHECK(h);
  return ARX_OK;
}

int arx_tc_finish(arx_handle *h, const float *partial, float *logits, int32_t *chosen, int64_t n_win, int way, int N, bool pdl, cudaStream_t st) {
  ARX_CUDA(h, arx_launch_pdl(k_finish_tc, dim3((unsigned)((n_win + 127) / 128)), dim3(128), 0, st, pdl, partial, logits, chosen, n_win, way, N));
  h->launches++;
  return ARX_OK;
}

// cross-attention + distances of the metric shape (T=16 pair tuples): third-generation kernel, then logits / argmax
int arx_tc_attention(arx_handle *h, const ArxTransformer &tr, const __half *kq_img, const float *G, int64_t n_win, int way, float *partial,
                     float *logits, int32_t *chosen, int g_ld, int g_voff, bool g_chunked, bool episodes, cudaStream_t st) {
  int rc = arx_tc3_attention_launch(h, tr, kq_img, G, n_win, way, partial, g_ld, g_voff, g_chunked, episodes, st);
  if (rc) return rc;
  return arx_tc_finish(h, partial, logits, chosen, n_win, way, tr.N, h->pdl, st);
}

// One-launch support build from the per-frame projections G (way*T, 2cD); with_tiles also fills the class tiles.
int arx_tc_support_build(arx_handle *h, ArxTransformer &tr, const float *G, int way, bool with_tiles, cudaStream_t st) {
  int rc;
  if (with_tiles && (rc = class_tiles_alloc(h, tr))) return rc;
  k_support_build<<<dim3(way, 8), 256, 0, st>>>(G, tr.tuples, tr.ln_g, tr.ln_b, tr.ks, tr.vs, with_tiles ? tr.kc_tiles : nullptr,
                                       with_tiles ? tr.vct_tiles : nullptr, h->T, tr.c, tr.N, 2 * tr.c * h->D);
  ARX_LAUNCH_CHECK(h);
  return ARX_OK;
}

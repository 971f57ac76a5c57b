// C ABI (include/arx.h): handle management, weight staging, support-set precompute and the
// scoring orchestration.  Host-side only; every kernel lives in the other translation units.
#include "arx_internal.cuh"
#include <stdarg.h>
#include <stdio.h>
#include <string.h>
#include <stdlib.h>
#include <math.h>
#include <algorithm>

static std::string g_create_err;
extern "C" { static void stream_free(arx_handle *h); }

int arx_fail(arx_handle *h, int code, const char *fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  if (h) h->err = buf;
  else g_create_err = buf;
  return code;
}

int arx_ws_reserve(arx_handle *h, size_t bytes) {
  if (bytes <= h->ws_bytes) return ARX_OK;
  if (h->ws) {
    ARX_CUDA(h, cudaDeviceSynchronize());
    ARX_CUDA(h, cudaFree(h->ws));
    h->ws = nullptr;
    h->ws_bytes = 0;
  }
  size_t want = bytes + (bytes >> 3);
  cudaError_t e = cudaMalloc(&h->ws, want);
  if (e != cudaSuccess) {
    want = bytes;
    e = cudaMalloc(&h->ws, want);
  }
  if (e != cudaSuccess) return arx_fail(h, ARX_ERR_NOMEM, "workspace cudaMalloc(%zu) failed: %s", want, cudaGetErrorString(e));
  h->ws_bytes = want;
  return ARX_OK;
}

namespace {

struct Carver {
  char *base;
  size_t off = 0;
  explicit Carver(void *p) : base(static_cast<char *>(p)) {}
  template <class Tp> Tp *take(size_t n) {
    off = (off + 255) & ~size_t(255);
    Tp *p = base ? reinterpret_cast<Tp *>(base + off) : nullptr;
    off += n * sizeof(Tp);
    return p;
  }
};

long long comb(int n, int k) {
  if (k < 0 || k > n) return 0;
  long long r = 1;
  for (int i = 1; i <= k; ++i) r = r * (n - k + i) / i;
  return r;
}

template <class Tp> int dev_alloc(arx_handle *h, Tp **p, size_t n) {
  ARX_CUDA(h, cudaMalloc(reinterpret_cast<void **>(p), std::max<size_t>(n, 1) * sizeof(Tp)));
  return ARX_OK;
}

int upload(arx_handle *h, float *dst, const float *src, size_t n, bool on_device, cudaStream_t st) {
  if (!src) return arx_fail(h, ARX_ERR_INVALID, "load_weights: missing tensor");
  ARX_CUDA(h, cudaMemcpyAsync(dst, src, n * sizeof(float), on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, st));
  return ARX_OK;
}

void free_support(arx_handle *h) {
  h->support_gen++;      // operand pointers change: cached score graphs no longer match
  for (int i = 0; i < h->cfg.n_transformers; ++i) {
    cudaFree(h->tr[i].ks); cudaFree(h->tr[i].vs);
    cudaFree(h->tr[i].ks_img); cudaFree(h->tr[i].vs_img); cudaFree(h->tr[i].vs_img_bf); cudaFree(h->tr[i].uc_img);
    cudaFree(h->tr[i].kc_tiles); cudaFree(h->tr[i].vct_tiles); cudaFree(h->tr[i].uc_tiles);
    h->tr[i].ks = h->tr[i].vs = nullptr;
    h->tr[i].ks_img = h->tr[i].vs_img = h->tr[i].vs_img_bf = h->tr[i].uc_img = nullptr;
    h->tr[i].kc_tiles = h->tr[i].vct_tiles = h->tr[i].uc_tiles = nullptr;
    h->tr[i].route = ARX_ROUTE_NONE;
  }
  cudaFree(h->ss_feat);
  cudaFree(h->ss_poses);
  h->ss_feat = nullptr;
  h->ss_poses = nullptr;
  h->way = h->way_cap = 0;
}

// What a scoring pass reads: pose windows (n, T, 3J), a frame stream (n + T - 1 frames of 3J; window w = frames w .. w+T-1)
// or feature windows (n, T, F).  Pose rows may be fp16 (arx_score_host*_f16); only routes with tc_front_end take them.
struct Query {
  enum Kind { WINDOWS, FRAMES, FEATURES };
  const void *rows;
  Kind kind;
  bool f16;
  bool poses() const { return kind != FEATURES; }
  // input rows that n windows read
  int64_t n_rows(const arx_handle *h, int64_t n) const { return kind == FRAMES ? n + h->T - 1 : n * h->T; }
  // the rows of the chunk that starts at window b0
  const void *at(const arx_handle *h, int64_t b0) const {
    const int64_t off = (kind == FRAMES ? b0 : b0 * h->T) * (poses() ? h->J3 : h->F);
    return static_cast<const char *>(rows) + off * (f16 ? sizeof(__half) : sizeof(float));
  }
  const float *f32(const arx_handle *h, int64_t b0) const { return static_cast<const float *>(at(h, b0)); }
};

// Where a pass writes: logits (n, way), is_true (n; null: no open-set head), chosen (n; null: argmax scratch in the
// workspace) and the debug outputs only the fp32 kernels write (probs (n, way, N, N), protos (n, way, N, D); null: none)
struct Outputs {
  float *logits, *is_true;
  int32_t *chosen;
  float *probs = nullptr, *protos = nullptr;
};

// per-window workspace of the T=16 pair pipeline
struct PairWs {
  __half *kq_img, *x_img, *h_img, *f_img, *y_img, *h1_img;
  float *uab, *G, *partial, *P, *U;     // P, U: frame-stream form: per-frame position-independent projections / head columns
  size_t bytes;
};
PairWs carve_pair(arx_handle *h, const ArxTransformer &tr, const Query &q, int64_t n, int way, bool disc, void *base) {
  Carver c(base);
  PairWs w{};
  const bool frames = q.kind == Query::FRAMES;
  const int64_t rows_pad = (n * h->T + 127) / 128 * 128, n_pad = (n + 127) / 128 * 128;
  w.kq_img = c.take<__half>(n * 128 * 128);
  w.x_img = q.poses() ? c.take<__half>(rows_pad * 128) : nullptr;
  w.h_img = q.poses() ? c.take<__half>(rows_pad * 192) : nullptr;
  w.f_img = c.take<__half>(rows_pad * 320);      // 4 feature sub-tiles + the one-hot sub-tile
  w.y_img = disc ? c.take<__half>(n_pad * (int64_t)h->tl_d1.nk * 64) : nullptr;
  w.h1_img = disc ? c.take<__half>(n_pad * 256) : nullptr;
  w.uab = disc ? c.take<float>(rows_pad * 32) : nullptr;
  w.G = c.take<float>(rows_pad * 2 * tr.c * h->D);     // chunked layout holds whole 128-row tiles
  w.partial = c.take<float>(n * way * 4);
  w.P = frames ? c.take<float>((n + h->T) * 2 * tr.c * h->D) : nullptr;
  w.U = frames ? c.take<float>((n + h->T) * 32) : nullptr;
  w.bytes = c.off + 256;
  return w;
}

// per-window workspace of the fp32 CUDA-core kernels
struct Fp32Ws {
  float *H1, *FE, *P, *G, *Kq, *Vq, *Z, *partial, *y, *h1, *h2;
  size_t bytes;
};
Fp32Ws carve_generic(arx_handle *h, const ArxTransformer &tr, const Query &q, int64_t n, int way, bool disc, void *base) {
  Carver c(base);
  Fp32Ws w{};
  const int64_t rows_in = q.n_rows(h, n);
  w.H1 = q.poses() ? c.take<float>(rows_in * h->H) : nullptr;
  w.FE = q.poses() ? c.take<float>(rows_in * h->F) : nullptr;
  w.P = q.kind == Query::FRAMES ? c.take<float>(rows_in * 2 * tr.c * h->D) : nullptr;
  w.G = c.take<float>(n * h->T * 2 * tr.c * h->D);
  w.Kq = c.take<float>(n * tr.N * h->D);
  w.Vq = c.take<float>(n * tr.N * h->D);
  w.Z = c.take<float>(n * way * tr.N * 2);
  w.partial = c.take<float>(n * way * ((tr.N + 63) / 64));
  w.y = disc ? c.take<float>(n * tr.N * h->T) : nullptr;
  w.h1 = disc ? c.take<float>(n * 256) : nullptr;
  w.h2 = disc ? c.take<float>(n * 64) : nullptr;
  w.bytes = c.off + 256;
  return w;
}

// Windows per pass: at most max_chunk (default 4096), and at most 3 GB of the layout carve(n, base)
template <class Carve> int64_t pass_windows(const arx_handle *h, int64_t n_windows, Carve &&carve) {
  const size_t per = carve(128, nullptr).bytes / 128 + 1;
  const int64_t cap = h->cfg.max_chunk > 0 ? h->cfg.max_chunk : 4096;
  const int64_t fit = (int64_t)(((size_t)3 << 30) / per);
  return std::max<int64_t>(1, std::min(std::min(cap, fit), n_windows));
}

// The workspace for passes of `chunk` windows and, without the caller's chosen buffer, the argmax scratch after it
template <class Ws, class Carve> int pass_reserve(arx_handle *h, int64_t chunk, const int32_t *chosen_dev, Carve &&carve, Ws *w, int32_t **chosen_ws) {
  const size_t bytes = carve(chunk, nullptr).bytes;
  const int rc = arx_ws_reserve(h, bytes + (chosen_dev ? 0 : (size_t)chunk * sizeof(int32_t) + 256));
  if (rc) return rc;
  *w = carve(chunk, h->ws);
  *chosen_ws = chosen_dev ? nullptr : reinterpret_cast<int32_t *>(static_cast<char *>(h->ws) + bytes);
  return ARX_OK;
}

// frames (n_seq*T, 3J) -> features (n_seq*T, F)             (model.py:164-180)
int embed_frames(arx_handle *h, const float *X, int64_t rows, float *H1, float *FE, cudaStream_t st) {
  int rc = arx_fp32_linear(h, X, h->J3, h->fc1_w, h->J3, h->fc1_b, H1, h->H, rows, h->H, h->J3, ARX_ACT_RELU, nullptr, 1, st);
  if (rc) return rc;
  return arx_fp32_linear(h, H1, h->H, h->fc2_w, h->H, h->fc2_b, FE, h->F, rows, h->F, h->H, ARX_ACT_RELU, nullptr, 1, st);
}

// the same on tensor cores, three launches: frames (fp32, or fp16 when `f16`) -> fp16 image x_img -> fc1 -> h_img -> fc2 ->
// feature image f_img (f_nk sub-tiles; f_onehot: the one-hot sub-tile of the positional table, or -1)
int embed_frames_tc(arx_handle *h, const void *X, bool f16, int64_t rows, __half *x_img, __half *h_img, __half *f_img, int f_nk, int f_onehot,
                    cudaStream_t st) {
  int rc;
  if ((rc = arx_tc_rows_to_img(h, X, f16, h->J3, h->J3, rows, x_img, h->tl_fc1.nk, -1, st))) return rc;
  if ((rc = arx_tc_linear_img(h, h->tl_fc1, x_img, rows, ARX_ACT_RELU, h_img, h->tl_fc2.nk, -1, st))) return rc;
  return arx_tc_linear_img(h, h->tl_fc2, h_img, rows, ARX_ACT_RELU, f_img, f_nk, f_onehot, st);
}

// discriminator MLP on the CUDA cores: head input y (n, N*T) -> d1 -> d2 -> d3 + sigmoid   (model.py:183-204)
int disc_tail_fp32(arx_handle *h, const ArxTransformer &tr, const float *y, float *h1, float *h2, int64_t n, float *is_true, cudaStream_t st) {
  const int K1 = tr.N * h->T;
  int rc;
  if ((rc = arx_fp32_linear(h, y, K1, h->d1_w, K1, h->d1_b, h1, 256, n, 256, K1, ARX_ACT_RELU, nullptr, 1, st))) return rc;
  if ((rc = arx_fp32_linear(h, h1, 256, h->d2_w, 256, h->d2_b, h2, 64, n, 64, 256, ARX_ACT_RELU, nullptr, 1, st))) return rc;
  return arx_fp32_linear(h, h2, 64, h->d3_w, 64, h->d3_b, is_true, 1, n, 1, 64, ARX_ACT_SIGMOID, nullptr, 1, st);
}

// the same on tensor cores from the head input image y_img: d1 -> h1_img, then d2 + d3 + sigmoid in one launch
int disc_tail_tc(arx_handle *h, const __half *y_img, __half *h1_img, int64_t n, float *is_true, cudaStream_t st) {
  const int rc = arx_tc_linear_img(h, h->tl_d1, y_img, n, ARX_ACT_RELU, h1_img, h->tl_d2.nk, -1, st);
  if (rc) return rc;
  return arx_tc_linear_sigmoid_dot(h, h->tl_d2, h1_img, n, h->d3_w, h->d3_b, is_true, st);
}

// features -> per-frame projections with the positional encoding folded into a per-position bias
// table: (f + pe[t]).Wp^T + bp = f.Wp^T + (pe[t].Wp^T + bp)   (model.py:65-66,75-78)
int project_frames(arx_handle *h, const ArxTransformer &tr, const float *FE, int64_t rows, float *G, cudaStream_t st) {
  return arx_fp32_linear(h, FE, h->F, tr.wp, h->F, nullptr, G, 2 * tr.c * h->D, rows, 2 * tr.c * h->D, h->F, ARX_ACT_NONE,
                         tr.bp /* (T, 2cD) table */, h->T, st);
}

}  // namespace

extern "C" {

int arx_abi_version(void) { return ARX_ABI_VERSION; }

const char *arx_last_error(const arx_handle *h) { return h ? h->err.c_str() : g_create_err.c_str(); }

int arx_create(const arx_config *cfg, arx_handle **out) {
  if (!cfg || !out) return arx_fail(nullptr, ARX_ERR_INVALID, "arx_create: null argument");
  *out = nullptr;
  if (cfg->seq_len < 2 || cfg->seq_len > 64) return arx_fail(nullptr, ARX_ERR_INVALID, "seq_len %d out of range [2,64]", cfg->seq_len);
  if (cfg->out_dim != 128) return arx_fail(nullptr, ARX_ERR_INVALID, "trans_linear_out_dim must be 128 (got %d)", cfg->out_dim);
  if (cfg->feat_dim <= 0 || cfg->feat_dim % 4) return arx_fail(nullptr, ARX_ERR_INVALID, "feat_dim must be a positive multiple of 4");
  if (cfg->n_joints <= 0) return arx_fail(nullptr, ARX_ERR_INVALID, "n_joints must be positive");
  if (cfg->n_transformers < 1 || cfg->n_transformers > ARX_MAX_TRANSFORMERS)
    return arx_fail(nullptr, ARX_ERR_INVALID, "n_transformers out of range");
  for (int i = 0; i < cfg->n_transformers; ++i)
    if (cfg->cardinality[i] < 1 || cfg->cardinality[i] > 4 || cfg->cardinality[i] > cfg->seq_len)
      return arx_fail(nullptr, ARX_ERR_INVALID, "temp_set[%d]=%d unsupported", i, cfg->cardinality[i]);
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return arx_fail(nullptr, ARX_ERR_CUDA, "no CUDA device: %s", cudaGetErrorString(e));
  cudaDeviceProp prop;
  e = cudaGetDeviceProperties(&prop, dev);
  if (e != cudaSuccess) return arx_fail(nullptr, ARX_ERR_CUDA, "cudaGetDeviceProperties: %s", cudaGetErrorString(e));
  if (prop.major != 10) return arx_fail(nullptr, ARX_ERR_INVALID, "libarx is built for sm_100a only (device is sm_%d%d)", prop.major, prop.minor);
  arx_handle *h = new arx_handle();
  h->cfg = *cfg;
  h->device = dev;
  h->sm_count = prop.multiProcessorCount;
  if (const char *e = getenv("ARX_SM_RESERVE")) h->sm_reserve_n = std::max(0, std::min(atoi(e), h->sm_count / 2));
  if (const char *e = getenv("ARX_VARIANT")) h->tc_variant = atoi(e);      // bring-up: initial value of debug key 0 (A/B runs of bench.py)
  h->T = cfg->seq_len;
  h->J3 = cfg->n_joints * 3;
  h->H = cfg->n_joints * 6;
  h->F = cfg->feat_dim;
  h->D = cfg->out_dim;
  int rc = ARX_OK;
  auto A = [&](float **p, size_t n) { if (rc == ARX_OK) rc = dev_alloc(h, p, n); };
  A(&h->fc1_w, (size_t)h->H * h->J3); A(&h->fc1_b, h->H);
  A(&h->fc2_w, (size_t)h->F * h->H); A(&h->fc2_b, h->F);
  for (int i = 0; i < cfg->n_transformers && rc == ARX_OK; ++i) {
    ArxTransformer &tr = h->tr[i];
    tr.c = cfg->cardinality[i];
    tr.N = (int)comb(h->T, tr.c);
    tr.Npad = (tr.N + 127) / 128 * 128;
    A(&tr.pe, (size_t)h->T * h->F);
    A(&tr.wp, (size_t)2 * tr.c * h->D * h->F);
    A(&tr.bp, (size_t)h->T * 2 * tr.c * h->D);
    A(&tr.bp_sums, (size_t)h->T * 2);
    A(&tr.ln_g, h->D); A(&tr.ln_b, h->D);
    if (rc == ARX_OK) rc = dev_alloc(h, &tr.tuples, (size_t)tr.N * tr.c);
    if (rc == ARX_OK) rc = arx_build_tuple_table(h, h->T, tr.c, tr.N, tr.tuples, 0);
  }
  if (cfg->has_discriminator) {
    const int n2 = h->T * (h->T - 1) / 2;
    A(&h->dr_w, (size_t)h->T * h->D); A(&h->dr_b, h->T);
    A(&h->d1_w, (size_t)256 * n2 * h->T); A(&h->d1_b, 256);
    A(&h->d2_w, 64 * 256); A(&h->d2_b, 64);
    A(&h->d3_w, 64); A(&h->d3_b, 1);
  }
  if (rc == ARX_OK && cudaDeviceSynchronize() != cudaSuccess) rc = arx_fail(h, ARX_ERR_CUDA, "create: sync failed");
  if (rc != ARX_OK) {
    g_create_err = h->err;
    arx_destroy(h);
    return rc;
  }
  *out = h;
  return ARX_OK;
}

void arx_destroy(arx_handle *h) {
  if (!h) return;
  cudaDeviceSynchronize();
  free_support(h);
  cudaFree(h->fc1_w); cudaFree(h->fc1_b); cudaFree(h->fc2_w); cudaFree(h->fc2_b);
  for (int i = 0; i < ARX_MAX_TRANSFORMERS; ++i) {
    ArxTransformer &tr = h->tr[i];
    cudaFree(tr.pe); cudaFree(tr.wp); cudaFree(tr.bp); cudaFree(tr.ln_g); cudaFree(tr.ln_b); cudaFree(tr.tuples); cudaFree(tr.bp_sums); cudaFree(tr.wp_ext);
    cudaFree(tr.tup_packed); cudaFree(tr.sel_tiles);
  }
  cudaFree(h->dr_w); cudaFree(h->dr_b); cudaFree(h->d1_w); cudaFree(h->d1_b);
  cudaFree(h->d2_w); cudaFree(h->d2_b); cudaFree(h->d3_w); cudaFree(h->d3_b);
  for (ArxTcLinear *L : {&h->tl_fc1, &h->tl_fc2, &h->tl_d1, &h->tl_d2, &h->tl_heads}) { cudaFree(L->w_img); cudaFree(L->bias); }
  for (int i = 0; i < ARX_MAX_TRANSFORMERS; ++i) {
    cudaFree(h->tr[i].tl_proj.w_img); cudaFree(h->tr[i].tl_proj.bias); cudaFree(h->tr[i].tl_proj_nt.w_img); cudaFree(h->tr[i].tl_proj_nt.bias); cudaFree(h->tr[i].tl_uab.w_img); cudaFree(h->tr[i].tl_uab.bias);
    cudaFree(h->tr[i].wc); cudaFree(h->tr[i].tcomp);
  }
  for (int i = 0; i < ARX_HOST_DEPTH; ++i) {
    cudaFree(h->hs_in[i]); cudaFree(h->hs_out[i]);
    if (h->hs_ev_h2d[i]) cudaEventDestroy(h->hs_ev_h2d[i]);
    if (h->hs_ev_comp[i]) cudaEventDestroy(h->hs_ev_comp[i]);
    if (h->hs_ev_done[i]) cudaEventDestroy(h->hs_ev_done[i]);
  }
  if (h->hs_h2d) { cudaStreamDestroy(h->hs_h2d); cudaStreamDestroy(h->hs_comp); cudaStreamDestroy(h->hs_d2h); }
  for (auto &g : h->graphs) for (int i = 0; i < 2; ++i) if (g.exec[i]) cudaGraphExecDestroy(g.exec[i]);
  if (h->side_stream) cudaStreamDestroy(h->side_stream);
  if (h->aux_stream) cudaStreamDestroy(h->aux_stream);
  if (h->ev_aux_fork) cudaEventDestroy(h->ev_aux_fork);
  if (h->ev_aux_done) cudaEventDestroy(h->ev_aux_done);
  if (h->ev_fork) cudaEventDestroy(h->ev_fork);
  if (h->ev_support_done) cudaEventDestroy(h->ev_support_done);
  if (h->ev_score_done) cudaEventDestroy(h->ev_score_done);
  stream_free(h);
  cudaFree(h->ws);
  cudaFree(h->zscratch);
  cudaFree(h->tcn_diag);
  cudaFree(h->ss_scratch);
  for (cudaEvent_t e : h->prof_events) cudaEventDestroy(e);
  for (int i = 0; i < 2; ++i) {
    cudaFree(h->dev_in[i]); cudaFree(h->dev_out[i]);
    if (h->own_stream[i]) cudaStreamDestroy(h->own_stream[i]);
    if (h->stage_ev[i]) cudaEventDestroy(h->stage_ev[i]);
  }
  delete h;
}

int arx_load_weights(arx_handle *h, const arx_weights *w, void *stream) {
  if (!h || !w) return arx_fail(h, ARX_ERR_INVALID, "load_weights: null argument");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const bool od = w->on_device != 0;
  int rc;
#define UP(dst, src, n) if ((rc = upload(h, dst, src, (n), od, st)) != ARX_OK) return rc
  UP(h->fc1_w, w->fc1_w, (size_t)h->H * h->J3); UP(h->fc1_b, w->fc1_b, h->H);
  UP(h->fc2_w, w->fc2_w, (size_t)h->F * h->H); UP(h->fc2_b, w->fc2_b, h->F);
  for (int i = 0; i < h->cfg.n_transformers; ++i) {
    ArxTransformer &tr = h->tr[i];
    const int D = h->D, F = h->F, c = tr.c;
    UP(tr.pe, w->pe[i], (size_t)h->T * F);                 // first T rows of (1, int(1.5T), F) (model.py:27)
    UP(tr.ln_g, w->ln_g[i], D); UP(tr.ln_b, w->ln_b[i], D);
    if (!w->k_w[i] || !w->v_w[i] || !w->k_b[i] || !w->v_b[i]) return arx_fail(h, ARX_ERR_INVALID, "load_weights: transformer %d tensors missing", i);
    // wp rows [p*D,(p+1)*D) = k_linear.weight[:, p*F:(p+1)*F]; rows [(c+p)*D, ...) = v_linear.weight[:, p*F:(p+1)*F]
    const cudaMemcpyKind kind = od ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
    for (int p = 0; p < c; ++p) {
      ARX_CUDA(h, cudaMemcpy2DAsync(tr.wp + (size_t)p * D * F, F * sizeof(float), w->k_w[i] + (size_t)p * F, (size_t)c * F * sizeof(float),
                                    F * sizeof(float), D, kind, st));
      ARX_CUDA(h, cudaMemcpy2DAsync(tr.wp + (size_t)(c + p) * D * F, F * sizeof(float), w->v_w[i] + (size_t)p * F, (size_t)c * F * sizeof(float),
                                    F * sizeof(float), D, kind, st));
    }
    // bias table bp (T, 2cD) = pe[t].wp^T + [k_b | 0.. | v_b | 0..]: computed with the linear kernel
    // (A = pe (T,F), W = wp, bias = flat bias (2cD)), staged through the workspace
    int rc2 = arx_ws_reserve(h, (size_t)2 * c * D * sizeof(float) + 256);
    if (rc2) return rc2;
    float *flat = static_cast<float *>(h->ws);
    ARX_CUDA(h, cudaMemsetAsync(flat, 0, (size_t)2 * c * D * sizeof(float), st));
    ARX_CUDA(h, cudaMemcpyAsync(flat, w->k_b[i], D * sizeof(float), kind, st));
    ARX_CUDA(h, cudaMemcpyAsync(flat + (size_t)c * D, w->v_b[i], D * sizeof(float), kind, st));
    rc = arx_fp32_linear(h, tr.pe, F, tr.wp, F, flat, tr.bp, 2 * c * D, h->T, 2 * c * D, F, ARX_ACT_NONE, nullptr, 1, st);
    if (rc) return rc;
    if (c >= 2 && (rc = arx_tc_table_sums(h, tr.bp, h->T, 2 * c * D, tr.bp_sums, st))) return rc;
    // static softmax bound from the LayerNorm affine (SURVEY.md 7.2-1): |S| <= (max|g| sqrt(D) + ||b||_2)^2 / sqrt(D)
    std::vector<float> g(D), b(D);
    ARX_CUDA(h, cudaMemcpyAsync(g.data(), tr.ln_g, D * sizeof(float), cudaMemcpyDeviceToHost, st));
    ARX_CUDA(h, cudaMemcpyAsync(b.data(), tr.ln_b, D * sizeof(float), cudaMemcpyDeviceToHost, st));
    ARX_CUDA(h, cudaStreamSynchronize(st));
    if (D == 128) { memcpy(tr.ln_host, g.data(), 128 * sizeof(float)); memcpy(tr.ln_host + 128, b.data(), 128 * sizeof(float)); }
    double gm = 0, bn = 0;
    for (int d = 0; d < D; ++d) { gm = std::max(gm, (double)fabsf(g[d])); bn += (double)b[d] * b[d]; }
    double r = gm * sqrt((double)D) + sqrt(bn);
    tr.softmax_bound = (float)(r * r / sqrt((double)D));
  }
  if (h->cfg.has_discriminator) {
    const int n2 = h->T * (h->T - 1) / 2;
    UP(h->dr_w, w->dr_w, (size_t)h->T * h->D); UP(h->dr_b, w->dr_b, h->T);
    UP(h->d1_w, w->d1_w, (size_t)256 * n2 * h->T); UP(h->d1_b, w->d1_b, 256);
    UP(h->d2_w, w->d2_w, 64 * 256); UP(h->d2_b, w->d2_b, 64);
    UP(h->d3_w, w->d3_w, 64); UP(h->d3_b, w->d3_b, 1);
  }
#undef UP
  // tensor-core images of the linear layers (fp16, pre-swizzled); shapes outside these bounds stay on the fp32 kernels
  h->tc_linears = false;
  if (h->cfg.force_path != 1 && h->F == 256 && h->H <= 192 && h->J3 <= 128) {
    if ((rc = arx_tc_linear_prepare(h, h->tl_fc1, h->fc1_w, h->J3, h->fc1_b, h->H, h->J3, 192, st))) return rc;
    if ((rc = arx_tc_linear_prepare(h, h->tl_fc2, h->fc2_w, h->H, h->fc2_b, h->F, h->H, 256, st))) return rc;
    for (int i = 0; i < h->cfg.n_transformers; ++i) {
      ArxTransformer &tr = h->tr[i];
      tr.table_in_gemm = (h->T == 16);
      if (tr.table_in_gemm) {
        // the positional-encoding / bias table rides through the GEMM: 32 one-hot K columns against hi/lo(table)
        if (!tr.wp_ext) ARX_CUDA(h, cudaMalloc(reinterpret_cast<void **>(&tr.wp_ext), (size_t)2 * tr.c * h->D * (h->F + 32) * sizeof(float)));
        if ((rc = arx_tc_build_wp_ext(h, tr.wp, tr.bp, tr.wp_ext, 2 * tr.c * h->D, h->F, st))) return rc;
        if ((rc = arx_tc_linear_prepare(h, tr.tl_proj, tr.wp_ext, h->F + 32, nullptr, 2 * tr.c * h->D, h->F + 32, 256, st))) return rc;
        if ((rc = arx_tc_linear_prepare(h, tr.tl_proj_nt, tr.wp, h->F, nullptr, 2 * tr.c * h->D, h->F, 256, st))) return rc;
      } else if ((rc = arx_tc_linear_prepare(h, tr.tl_proj, tr.wp, h->F, nullptr, 2 * tr.c * h->D, h->F, 256, st))) return rc;
    }
    if (h->cfg.has_discriminator) {
      const int K1 = h->T * (h->T - 1) / 2 * h->T;
      if ((rc = arx_tc_linear_prepare(h, h->tl_d1, h->d1_w, K1, h->d1_b, 256, K1, 64, st))) return rc;
      if ((rc = arx_tc_linear_prepare(h, h->tl_d2, h->d2_w, 256, h->d2_b, 64, 256, 64, st))) return rc;
      if (h->T == 16 && h->tr[0].c == 2 && (rc = arx_tc2_head_prepare_weights(h, h->tr[0], st))) return rc;
    }
    h->tc_linears = true;
  }
  h->mlp_bias_host_ok = false;
  if (h->tc_linears && h->tl_fc1.BN == 192 && h->tl_fc1.n_tiles == 1 && h->tl_fc2.BN == 256 && h->tl_fc2.n_tiles == 1) {
    ARX_CUDA(h, cudaMemcpyAsync(h->mlp_bias_host, h->tl_fc1.bias, 192 * sizeof(float), cudaMemcpyDeviceToHost, st));
    ARX_CUDA(h, cudaMemcpyAsync(h->mlp_bias_host + 192, h->tl_fc2.bias, 256 * sizeof(float), cudaMemcpyDeviceToHost, st));
    h->mlp_bias_host_ok = true;
  }
  ARX_CUDA(h, cudaStreamSynchronize(st));
  h->weights_loaded = true;
  h->weights_gen++;
  free_support(h);   // support operands depend on the weights
  return ARX_OK;
}

int arx_tuple_count(const arx_handle *h, int32_t ti) {
  if (!h || ti < 0 || ti >= h->cfg.n_transformers) return ARX_ERR_INVALID;
  return h->tr[ti].N;
}

int arx_tuple_table(arx_handle *h, int32_t ti, int32_t *out_dev, void *stream) {
  if (!h || !out_dev || ti < 0 || ti >= h->cfg.n_transformers) return arx_fail(h, ARX_ERR_INVALID, "tuple_table: bad argument");
  const ArxTransformer &tr = h->tr[ti];
  // rebuilt on device on every call (it is the kernel under test), not copied from the cached table
  return arx_build_tuple_table(h, h->T, tr.c, tr.N, out_dev, static_cast<cudaStream_t>(stream));
}

int arx_embed(arx_handle *h, const float *frames_dev, int64_t n_frames, float *feats_dev, void *stream) {
  if (!h || !frames_dev || !feats_dev || n_frames < 0) return arx_fail(h, ARX_ERR_INVALID, "embed: bad argument");
  if (!h->weights_loaded) return arx_fail(h, ARX_ERR_STATE, "embed: weights not loaded");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int64_t chunk = 1 << 16;
  int rc = arx_ws_reserve(h, (size_t)chunk * h->H * sizeof(float) + 256);
  if (rc) return rc;
  for (int64_t r0 = 0; r0 < n_frames; r0 += chunk) {
    int64_t r = std::min(chunk, n_frames - r0);
    rc = embed_frames(h, frames_dev + r0 * h->J3, r, static_cast<float *>(h->ws), feats_dev + r0 * h->F, st);
    if (rc) return rc;
  }
  return ARX_OK;
}

// ---- stream-capture awareness -------------------------------------------------------------------------------------
// A caller may capture whole steps (set_support + score + its own collectives) into ONE CUDA graph.  Inside a capture a
// stream may only wait on events recorded in the SAME capture, so every internal event remembers the capture it was
// recorded in (0 = recorded eagerly) and waits follow these rules:
//   same context (both eager, or same capture)      -> cudaStreamWaitEvent
//   capturing now, event recorded eagerly before     -> no node: nothing inside a capture may wait on (or even query) outside
//                                                       work; the work recorded eagerly before the capture began is ordered
//                                                       before the graph by whoever launches it (arx_stream_push waits for
//                                                       the support chain eagerly before it captures or replays; a caller
//                                                       capturing arx_score alone must have synchronised after set_support)
//   otherwise (event belongs to another capture)     -> nothing to wait for: replays are ordered by the launching stream
static unsigned long long capture_id(cudaStream_t st) {
  cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
  unsigned long long id = 0;
  if (cudaStreamGetCaptureInfo(st, &cs, &id) != cudaSuccess) { (void)cudaGetLastError(); return 0; }
  return cs == cudaStreamCaptureStatusActive ? (id ? id : 1ull) : 0ull;
}
static int wait_event_cap(arx_handle *h, cudaStream_t waiter, cudaEvent_t ev, unsigned long long ev_cid, unsigned long long cur_cid) {
  if (ev_cid == cur_cid) {
    ARX_CUDA(h, cudaStreamWaitEvent(waiter, ev, 0));
  }
  return ARX_OK;
}

// fork the support chain onto the side stream (after everything already queued on the caller's stream and after
// the last scoring pass that still reads the current operands)
static int support_fork(arx_handle *h, cudaStream_t st, cudaStream_t *side) {
  if (!h->side_stream) {
    ARX_CUDA(h, cudaStreamCreateWithFlags(&h->side_stream, cudaStreamNonBlocking));
    ARX_CUDA(h, cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming));
    ARX_CUDA(h, cudaEventCreateWithFlags(&h->ev_support_done, cudaEventDisableTiming));
    if (!h->ev_score_done) ARX_CUDA(h, cudaEventCreateWithFlags(&h->ev_score_done, cudaEventDisableTiming));
  }
  const unsigned long long cid = capture_id(st);
  ARX_CUDA(h, cudaEventRecord(h->ev_fork, st));
  ARX_CUDA(h, cudaStreamWaitEvent(h->side_stream, h->ev_fork, 0));
  // the last scoring pass still reads the current operands: on `st` itself it is already ordered before the fork
  if (h->score_recorded && h->last_score_stream != st) {
    const int rc = wait_event_cap(h, h->side_stream, h->ev_score_done, h->score_cid, cid);
    if (rc) return rc;
  }
  h->support_cid = cid;
  h->support_seq++;                 // a new support set is on its way: operands derived from the old one are stale
  *side = h->side_stream;
  return ARX_OK;
}
static int support_join_record(arx_handle *h) {
  ARX_CUDA(h, cudaEventRecord(h->ev_support_done, h->side_stream));
  h->support_recorded = true;
  h->support_inflight = true;
  return ARX_OK;
}
// consumers of the support operands on stream st
static int support_wait(arx_handle *h, cudaStream_t st) {
  h->support_inflight = false;
  if (h->support_recorded) return wait_event_cap(h, st, h->ev_support_done, h->support_cid, capture_id(st));
  return ARX_OK;
}
static int score_done_record(arx_handle *h, cudaStream_t st) {
  if (!h->ev_score_done) ARX_CUDA(h, cudaEventCreateWithFlags(&h->ev_score_done, cudaEventDisableTiming));
  ARX_CUDA(h, cudaEventRecord(h->ev_score_done, st));
  h->score_recorded = true;
  h->last_score_stream = st;
  h->score_cid = capture_id(st);
  return ARX_OK;
}
// the shared workspace may still be in use by streamed host requests or by a scoring pass on another stream
static int workspace_wait(arx_handle *h, cudaStream_t st) {
  const unsigned long long cid = capture_id(st);
  int rc;
  if (st != h->hs_comp && h->hs_submitted > 0 && (rc = wait_event_cap(h, st, h->hs_ev_comp[(h->hs_submitted - 1) % ARX_HOST_DEPTH], 0, cid))) return rc;
  if (h->score_recorded && h->last_score_stream != st && (rc = wait_event_cap(h, st, h->ev_score_done, h->score_cid, cid))) return rc;
  return ARX_OK;
}

// support tensors of `way` classes for transformers [0, n_tr) (n_tr < n_transformers: the episode pool of arx_score_episodes)
static int support_alloc(arx_handle *h, int way, int n_tr, cudaStream_t st) {
  if (way <= h->way_cap && h->tr[n_tr - 1].ks) return ARX_OK;
  ARX_CUDA(h, cudaStreamSynchronize(st));
  ARX_CUDA(h, cudaDeviceSynchronize());
  free_support(h);
  int rc;
  for (int i = 0; i < n_tr; ++i) {
    if ((rc = dev_alloc(h, &h->tr[i].ks, (size_t)way * h->tr[i].N * h->D))) return rc;
    if ((rc = dev_alloc(h, &h->tr[i].vs, (size_t)way * h->tr[i].N * h->D))) return rc;
  }
  if ((rc = dev_alloc(h, &h->ss_feat, (size_t)way * h->T * h->F))) return rc;
  if ((rc = dev_alloc(h, &h->ss_poses, (size_t)way * h->T * h->J3))) return rc;
  h->way_cap = way;
  return ARX_OK;
}

// scratch of the support path: [x_img | h_img | f_img | G], sized for way*T rows (padded to 128)
struct SupportScratch { __half *x_img, *h_img, *f_img; float *G; size_t bytes; };
static SupportScratch support_scratch(arx_handle *h, int way, void *base) {
  Carver c(base);
  SupportScratch s{};
  const int64_t rows_pad = ((int64_t)way * h->T + 127) / 128 * 128;
  int maxc = 1;
  for (int i = 0; i < h->cfg.n_transformers; ++i) maxc = std::max(maxc, h->tr[i].c);
  s.x_img = c.take<__half>(rows_pad * 128);
  s.h_img = c.take<__half>(rows_pad * 192);
  s.f_img = c.take<__half>(rows_pad * 320);
  s.G = c.take<float>(rows_pad * 2 * maxc * h->D);
  s.bytes = c.off + 256;
  return s;
}
static int support_scratch_reserve(arx_handle *h, int way, SupportScratch *out) {
  const size_t need = support_scratch(h, way, nullptr).bytes;
  if (need > h->ss_scratch_bytes) {
    ARX_CUDA(h, cudaDeviceSynchronize());
    cudaFree(h->ss_scratch);
    h->ss_scratch = nullptr;
    h->ss_scratch_bytes = 0;
    ARX_CUDA(h, cudaMalloc(&h->ss_scratch, need));
    h->ss_scratch_bytes = need;
  }
  *out = support_scratch(h, way, h->ss_scratch);
  return ARX_OK;
}

static float accuracy_bound(const ArxTransformer &tr) {
  return tr.N < ARX_TC_FEW_TUPLES ? ARX_TC_ACCURACY_BOUND_FEW_TUPLES : ARX_TC_ACCURACY_BOUND;
}
// The tensor-core routes may score transformer `tr`: its LayerNorm affine is inside the accuracy bound, or the caller
// forced them (force_path = 2) and accepts the reduced accuracy.
static bool tc_admitted(const arx_handle *h, const ArxTransformer &tr) {
  return h->cfg.force_path == 2 || tr.softmax_bound < accuracy_bound(tr);
}

// Which kernels score transformer `tr`:  the T=16 pair pipeline (arx_tc3.cu and friends: fused tuple images, head by
// linearity, graph replay), the tiled any-N tcgen05 kernels (arx_tcn.cu: T=32, triples, other T, and under force_path = 2
// LayerNorm affines past the overflow bound), or the fp32 CUDA-core kernels (forced, D != 128, LayerNorm affines past
// the accuracy bound; debug outputs take them at score time).
static ArxRoute support_route(const arx_handle *h, const ArxTransformer &tr) {
  // Past the accuracy bound the fp16 QK^T and bf16 P.V operands lose the 1e-3 tolerance well before exp2 can overflow
  // (DESIGN 4: the error grows with the bound).  Parity first: such weights score on the fp32 kernels unless the caller
  // forces the tensor-core routes, and the handle says so once on stderr.
  if (h->cfg.force_path == 1 || !tc_admitted(h, tr)) return ARX_ROUTE_FP32;
  if (arx_tc_supported(h, tr) && h->T == 16 && tr.c == 2 && h->tc_linears && (h->tc_variant & (4096 | 4)) == 0) return ARX_ROUTE_PAIR;
  if (arx_tcn_supported(h, tr)) return ARX_ROUTE_TILED;      // the ROWMAX variant past the overflow bound
  return ARX_ROUTE_FP32;
}
static void warn_fp32_fallback(arx_handle *h, int ti) {
  const ArxTransformer &tr = h->tr[ti];
  if (h->cfg.force_path == 1 || (h->warned & (1u << ti)) || !arx_tcn_supported(h, tr) || tc_admitted(h, tr)) return;
  h->warned |= 1u << ti;
  fprintf(stderr, "libarx: transformers[%d].norm_k has a LayerNorm affine outside the fp16 tensor-core bound (|S| <= %.1f; accuracy "
                  "bound %.1f, overflow bound %.1f): scoring on the fp32 CUDA-core kernels (about 30x slower) to stay within the "
                  "1e-3 tolerance; force_path=2 selects the tensor-core kernels at reduced accuracy\n",
          ti, (double)tr.softmax_bound, (double)accuracy_bound(tr), 100.0 / ARX_SOFTMAX_LOG2E);
}

// The tiled route builds the class tiles of the open-set head (Uc) for transformer i
static bool tiled_head(const arx_handle *h, int i) { return i == 0 && h->cfg.has_discriminator && arx_tcn_head_supported(h, h->tr[i]); }

// Decides transformer i's route and builds the support operands it reads: the tuple tensors ks/vs from the per-frame
// projections G (or, with G == nullptr, ks/vs are already in place: arx_import_support), the operand images and the
// head's Uc of the pair pipeline, the class tiles of the tiled kernels.
static int support_operands(arx_handle *h, int i, const float *G, int way, cudaStream_t st) {
  ArxTransformer &tr = h->tr[i];
  tr.route = support_route(h, tr);
  const bool imgs = tr.route == ARX_ROUTE_PAIR;
  int rc = ARX_OK;
  if (G && h->D == 128) rc = arx_tc_support_build(h, tr, G, way, imgs, st);      // tuples + LayerNorm + operand images, one launch
  else if (G) rc = arx_fp32_build_tuples(h, tr, G, way, tr.ks, tr.vs, st);
  else if (imgs) rc = arx_tc_prep_support(h, tr, way, st);
  if (rc) return rc;
  if (imgs && i == 0 && h->cfg.has_discriminator && (rc = arx_tc2_support_uc(h, tr, way, st))) return rc;
  if (tr.route == ARX_ROUTE_TILED) {
    if ((rc = arx_tcn_prep_support(h, tr, way, tiled_head(h, i), st))) return rc;
    h->tiles_gen[i] = h->support_seq + 1;
  }
  return ARX_OK;
}

// projection + tuple/LayerNorm/image build of the support set from frame features given as an fp16 image
// (tensor-core path) or as fp32 rows (general path), for transformers [0, n_tr); the others are left without operands
static int support_from_features(arx_handle *h, const __half *f_img, const float *feats32, int way, int n_tr, float *G, cudaStream_t st) {
  int rc;
  for (int i = n_tr; i < h->cfg.n_transformers; ++i) h->tr[i].route = ARX_ROUTE_NONE;
  for (int i = 0; i < n_tr; ++i) {
    ArxTransformer &tr = h->tr[i];
    const int64_t rows = (int64_t)way * h->T;
    if (f_img) {
      if ((rc = arx_tc_linear_f32(h, tr.tl_proj, f_img, h->tr[0].tl_proj.nk, rows, G, 2 * tr.c * h->D, tr.table_in_gemm ? nullptr : tr.bp, h->T, st)))
        return rc;
    } else {
      if ((rc = project_frames(h, tr, feats32, rows, G, st))) return rc;
    }
    if ((rc = support_operands(h, i, G, way, st))) return rc;
  }
  h->way = way;
  return ARX_OK;
}

static int set_support_features(arx_handle *h, const float *feats_dev, int32_t way, int n_tr, cudaStream_t st) {
  int rc;
  if ((rc = support_alloc(h, way, n_tr, st))) return rc;
  SupportScratch sc;
  if ((rc = support_scratch_reserve(h, way, &sc))) return rc;
  if ((rc = support_wait(h, st))) return rc;                       // a previous chain may still be writing ss_feat
  if (feats_dev != h->ss_feat)
    ARX_CUDA(h, cudaMemcpyAsync(h->ss_feat, feats_dev, (size_t)way * h->T * h->F * sizeof(float), cudaMemcpyDeviceToDevice, st));
  h->ss_feat_valid = true;
  cudaStream_t ss;
  if ((rc = support_fork(h, st, &ss))) return rc;                  // the caller's buffer is not touched past this point
  if (h->tc_linears) {
    if ((rc = arx_tc_rows_to_img(h, h->ss_feat, false, h->F, h->F, (int64_t)way * h->T, sc.f_img, h->tr[0].tl_proj.nk,
                                 h->tr[0].table_in_gemm ? h->tr[0].tl_proj.nk - 1 : -1, ss)))
      return rc;
    rc = support_from_features(h, sc.f_img, nullptr, way, n_tr, sc.G, ss);
  } else {
    rc = support_from_features(h, nullptr, h->ss_feat, way, n_tr, sc.G, ss);
  }
  if (rc) return rc;
  return support_join_record(h);
}

int arx_set_support_features(arx_handle *h, const float *feats_dev, int32_t way, void *stream) {
  if (!h || !feats_dev || way < 1) return arx_fail(h, ARX_ERR_INVALID, "set_support: bad argument");
  if (!h->weights_loaded) return arx_fail(h, ARX_ERR_STATE, "set_support: weights not loaded");
  return set_support_features(h, feats_dev, way, h->cfg.n_transformers, static_cast<cudaStream_t>(stream));
}

static int set_support_poses(arx_handle *h, const float *poses_dev, int32_t way, int n_tr, cudaStream_t st) {
  int rc;
  if ((rc = support_alloc(h, way, n_tr, st))) return rc;
  SupportScratch sc;
  if ((rc = support_scratch_reserve(h, way, &sc))) return rc;
  const int64_t rows = (int64_t)way * h->T;
  if ((rc = support_wait(h, st))) return rc;                       // a previous chain may still be reading ss_poses
  ARX_CUDA(h, cudaMemcpyAsync(h->ss_poses, poses_dev, (size_t)rows * h->J3 * sizeof(float), cudaMemcpyDeviceToDevice, st));
  h->ss_poses_valid = true;
  cudaStream_t ss;
  if ((rc = support_fork(h, st, &ss))) return rc;                  // the caller's buffer is not touched past this point
  if (h->tc_linears) {
    // same tensor-core pipeline as the query frames; the fp32 'support_features' are derived lazily on request
    h->ss_feat_valid = false;
    if ((rc = embed_frames_tc(h, h->ss_poses, false, rows, sc.x_img, sc.h_img, sc.f_img, h->tr[0].tl_proj.nk,
                              h->tr[0].table_in_gemm ? h->tr[0].tl_proj.nk - 1 : -1, ss)))
      return rc;
    rc = support_from_features(h, sc.f_img, nullptr, way, n_tr, sc.G, ss);
  } else {
    // general path: arx_embed stages through the shared workspace, so it stays on the caller's stream
    if ((rc = arx_embed(h, h->ss_poses, rows, h->ss_feat, st))) return rc;
    h->ss_feat_valid = true;
    if ((rc = support_fork(h, st, &ss))) return rc;
    rc = support_from_features(h, nullptr, h->ss_feat, way, n_tr, sc.G, ss);
  }
  if (rc) return rc;
  return support_join_record(h);
}

int arx_set_support_poses(arx_handle *h, const float *poses_dev, int32_t way, void *stream) {
  if (!h || !poses_dev || way < 1) return arx_fail(h, ARX_ERR_INVALID, "set_support: bad argument");
  if (!h->weights_loaded) return arx_fail(h, ARX_ERR_STATE, "set_support: weights not loaded");
  return set_support_poses(h, poses_dev, way, h->cfg.n_transformers, static_cast<cudaStream_t>(stream));
}

static int support_features_materialise(arx_handle *h, cudaStream_t st) {
  int rcw = support_wait(h, st);
  if (rcw) return rcw;
  if (h->ss_feat_valid) return ARX_OK;
  if (!h->ss_poses_valid)
    return arx_fail(h, ARX_ERR_STATE, "support features are not available: this handle received the support operands through arx_import_support");
  int rc = arx_embed(h, h->ss_poses, (int64_t)h->way * h->T, h->ss_feat, st);      // fp32 MLP (model.py:175-180)
  if (rc == ARX_OK) h->ss_feat_valid = true;
  return rc;
}

int arx_get_support_features(arx_handle *h, float *feats_dev, void *stream) {
  if (!h || !feats_dev) return arx_fail(h, ARX_ERR_INVALID, "get_support_features: bad argument");
  if (h->way < 1) return arx_fail(h, ARX_ERR_STATE, "get_support_features: no support set");
  int rcm = support_features_materialise(h, static_cast<cudaStream_t>(stream));
  if (rcm) return rcm;
  ARX_CUDA(h, cudaMemcpyAsync(feats_dev, h->ss_feat, (size_t)h->way * h->T * h->F * sizeof(float), cudaMemcpyDeviceToDevice,
                              static_cast<cudaStream_t>(stream)));
  return ARX_OK;
}

int arx_support_way(const arx_handle *h) { return h ? h->way : ARX_ERR_INVALID; }

int64_t arx_support_blob_bytes(const arx_handle *h, int32_t way) {
  if (!h || way < 1) return ARX_ERR_INVALID;
  int64_t n = 0;
  for (int i = 0; i < h->cfg.n_transformers; ++i) n += 2ll * way * h->tr[i].N * h->D;      // K (LayerNorm-ed) and V tuple tensors
  return n * (int64_t)sizeof(float);
}

// blob = for every transformer [ks (way,N,D) | vs (way,N,D)] fp32: the support-set tuple embeddings (SURVEY 8e)
int arx_export_support(arx_handle *h, void *blob_dev, void *stream) {
  if (!h || !blob_dev) return arx_fail(h, ARX_ERR_INVALID, "export_support: bad argument");
  if (h->way < 1) return arx_fail(h, ARX_ERR_STATE, "export_support: no support set");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  for (int i = 0; i < h->cfg.n_transformers; ++i)
    if (h->tr[i].route == ARX_ROUTE_NONE)
      return arx_fail(h, ARX_ERR_STATE, "export_support: transformers[%d] has no support operands (arx_score_episodes keeps those of "
                                        "transformers[0] only): set the support set again", i);
  int rc = support_wait(h, st);                       // the chain that produces ks/vs runs on the side stream
  if (rc) return rc;
  float *p = static_cast<float *>(blob_dev);
  for (int i = 0; i < h->cfg.n_transformers; ++i) {
    const size_t n = (size_t)h->way * h->tr[i].N * h->D;
    ARX_CUDA(h, cudaMemcpyAsync(p, h->tr[i].ks, n * sizeof(float), cudaMemcpyDeviceToDevice, st));
    p += n;
    ARX_CUDA(h, cudaMemcpyAsync(p, h->tr[i].vs, n * sizeof(float), cudaMemcpyDeviceToDevice, st));
    p += n;
  }
  return ARX_OK;
}

int arx_import_support(arx_handle *h, const void *blob_dev, int32_t way, void *stream) {
  if (!h || !blob_dev || way < 1) return arx_fail(h, ARX_ERR_INVALID, "import_support: bad argument");
  if (!h->weights_loaded) return arx_fail(h, ARX_ERR_STATE, "import_support: weights not loaded");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int rc = support_alloc(h, way, h->cfg.n_transformers, st);
  if (rc) return rc;
  // like set_support: the copies and the operand-image builds run on the side stream (after everything queued on
  // `st`, i.e. after the collective that filled the blob), overlapped with the query-side kernels of the next score
  cudaStream_t ss;
  if ((rc = support_fork(h, st, &ss))) return rc;
  h->ss_feat_valid = false;
  h->ss_poses_valid = false;
  const float *p = static_cast<const float *>(blob_dev);
  for (int i = 0; i < h->cfg.n_transformers; ++i) {
    ArxTransformer &tr = h->tr[i];
    const size_t n = (size_t)way * tr.N * h->D;
    ARX_CUDA(h, cudaMemcpyAsync(tr.ks, p, n * sizeof(float), cudaMemcpyDeviceToDevice, ss));
    p += n;
    ARX_CUDA(h, cudaMemcpyAsync(tr.vs, p, n * sizeof(float), cudaMemcpyDeviceToDevice, ss));
    p += n;
    if ((rc = support_operands(h, i, nullptr, way, ss))) return rc;
  }
  h->way = way;
  return support_join_record(h);
}

static int prof_mark(arx_handle *h, int idx, cudaStream_t st) {
  if (!h->prof_on) return ARX_OK;
  if (idx == 0) {
    if (h->prof_used + ARX_N_STAGES + 1 > h->prof_events.size()) {
      for (int i = 0; i < ARX_N_STAGES + 1; ++i) {
        cudaEvent_t e;
        ARX_CUDA(h, cudaEventCreate(&e));
        h->prof_events.push_back(e);
      }
    }
    h->prof_used += ARX_N_STAGES + 1;
  }
  ARX_CUDA(h, cudaEventRecord(h->prof_events[h->prof_used - (ARX_N_STAGES + 1) + idx], st));
  return ARX_OK;
}

// front end on the CUDA cores, the n windows from b0 -> row-major per-frame projections G.  Poses are embedded here (H1, FE).
// A frame stream embeds and projects every frame once without the positional table (P), and the windows are formed from
// that: k_linear adds the table after the accumulation, so either way G holds the same bits.
static int front_end_fp32(arx_handle *h, const ArxTransformer &tr, const Query &q, int64_t b0, int64_t n, float *H1, float *FE, float *P,
                          float *G, cudaStream_t st) {
  const int64_t rows = q.n_rows(h, n);
  const int ldg = 2 * tr.c * h->D;
  int rc;
  if (q.poses() && (rc = embed_frames(h, q.f32(h, b0), rows, H1, FE, st))) return rc;
  if ((rc = prof_mark(h, 1, st))) return rc;
  if (q.kind != Query::FRAMES) return project_frames(h, tr, q.poses() ? FE : q.f32(h, b0), rows, G, st);
  if ((rc = arx_fp32_linear(h, FE, h->F, tr.wp, h->F, nullptr, P, ldg, rows, ldg, h->F, ARX_ACT_NONE, nullptr, 1, st))) return rc;
  return arx_form_windows_launch(h, tr, P, nullptr, G, nullptr, n, false, st);
}

// The route runs its front end on the tensor-core linear layers: the one front end that reads fp16 pose rows
static bool tc_front_end(const arx_handle *h, ArxRoute route) {
  return (route == ARX_ROUTE_PAIR || route == ARX_ROUTE_TILED) && h->tc_linears && (h->tc_variant & 4) == 0;
}

extern "C++" {
static bool graphs_enabled(arx_handle *h) {
  if (h->graphs_on < 0) {
    const char *e = getenv("ARX_GRAPHS");
    h->graphs_on = (e && e[0] == '0') ? 0 : 1;
  }
  return h->graphs_on == 1;
}

static ArxScoreGraph *score_graph_lookup(arx_handle *h, const ArxScoreGraphKey &key) {
  h->graph_tick++;
  for (auto &g : h->graphs)
    if (g.key == key) { g.last_use = h->graph_tick; return &g; }
  if (h->graphs.size() >= 16) {                    // evict the least recently used entry
    size_t v = 0;
    for (size_t i = 1; i < h->graphs.size(); ++i) if (h->graphs[i].last_use < h->graphs[v].last_use) v = i;
    for (int i = 0; i < 2; ++i) if (h->graphs[v].exec[i]) cudaGraphExecDestroy(h->graphs[v].exec[i]);
    h->graphs.erase(h->graphs.begin() + v);
  }
  ArxScoreGraph g;
  g.key = key;
  g.last_use = h->graph_tick;
  h->graphs.push_back(g);
  return &h->graphs.back();
}

// Replay *exec on st, capturing body() on st into it first when it is empty.  The launches body() counts during the
// capture are recorded in *launches instead, and every replay adds them to the handle's launch count.
template <class F> static int graph_replay(arx_handle *h, cudaStream_t st, const char *what, cudaGraphExec_t *exec, int64_t *launches, F &&body) {
  if (!*exec) {
    const int64_t l0 = h->launches;
    ARX_CUDA(h, cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
    const int rc = body();
    cudaGraph_t graph = nullptr;
    const cudaError_t e = cudaStreamEndCapture(st, &graph);
    if (rc) { if (graph) cudaGraphDestroy(graph); return rc; }
    if (e != cudaSuccess || !graph) return arx_fail(h, ARX_ERR_CUDA, "%s: stream capture failed: %s", what, cudaGetErrorString(e));
    const cudaError_t e2 = cudaGraphInstantiate(exec, graph, 0);
    cudaGraphDestroy(graph);
    if (e2 != cudaSuccess) { *exec = nullptr; return arx_fail(h, ARX_ERR_CUDA, "%s: graph instantiation failed: %s", what, cudaGetErrorString(e2)); }
    *launches = h->launches - l0;
    h->launches = l0;
  }
  ARX_CUDA(h, cudaGraphLaunch(*exec, st));
  h->launches += *launches;
  return ARX_OK;
}

// Run one segment of the score chain: eagerly the first time a key is seen (one-time initialisation -- symbol
// uploads, function attributes, allocations -- must not happen under capture), captured into a graph the second
// time, replayed from then on.
template <class F> static int score_segment(arx_handle *h, ArxScoreGraph *g, int seg, cudaStream_t st, F &&body) {
  if (!g || g->seen < 1) return body();
  return graph_replay(h, st, "score", &g->exec[seg], &g->launches[seg], body);
}
}  // extern "C++"

// ---- scoring on the tiled any-N tcgen05 kernels (arx_tcn.cu) -----------------------------------------------------
struct TcnWs {
  __half *x_img, *h_img, *f_img, *kq, *y_img, *h1_img, *vq, *vq_head;
  float *H1, *FE, *G, *partial, *uab, *y, *h1, *h2, *P;
  size_t bytes;
};
static TcnWs carve_tcn(arx_handle *h, const ArxTransformer &tr, const Query &q, int64_t n, int way, bool disc, bool tcl, void *base) {
  Carver c(base);
  TcnWs w{};
  const int64_t rows = n * h->T, rows_pad = (rows + 127) / 128 * 128, n_pad = (n + 127) / 128 * 128;
  const int nq = tr.Npad / 128;
  w.x_img = (tcl && q.poses()) ? c.take<__half>(rows_pad * 128) : nullptr;
  w.h_img = (tcl && q.poses()) ? c.take<__half>(rows_pad * 192) : nullptr;
  w.f_img = tcl ? c.take<__half>(rows_pad * 320) : nullptr;
  w.H1 = (!tcl && q.poses()) ? c.take<float>(rows * h->H) : nullptr;
  w.FE = (!tcl && q.poses()) ? c.take<float>(rows * h->F) : nullptr;
  w.G = c.take<float>(rows_pad * 2 * tr.c * h->D);
  w.kq = c.take<__half>((size_t)n * nq * 128 * 128);
  w.partial = c.take<float>(n * way * 4);
  const int nsel = (2 * tr.c * h->T + 63) / 64;                     // selection operands: 16 KB sub-tiles per window
  w.vq = c.take<__half>((size_t)n * nsel * 8192);
  w.vq_head = disc ? c.take<__half>((size_t)n * nsel * 8192) : nullptr;
  if (disc) {
    const int64_t K1 = (int64_t)tr.N * h->T;
    w.uab = c.take<float>(rows * 2 * arx_tcn_head_cols(h->T) + 256);
    if (tcl) {
      w.y_img = c.take<__half>(n_pad * (int64_t)h->tl_d1.nk * 64);
      w.h1_img = c.take<__half>(n_pad * 256);
    } else {
      w.y = c.take<float>(n * K1);
      w.h1 = c.take<float>(n * 256);
      w.h2 = c.take<float>(n * 64);
    }
  }
  w.P = q.kind == Query::FRAMES ? c.take<float>((n + h->T) * 2 * tr.c * h->D) : nullptr;
  w.bytes = c.off + 256;
  return w;
}

// query tiles -> cross-attention -> logits / argmax -> open-set head, from the row-major per-frame projections w.G
// ep_way > 0: episode mode, window w of this pass attends pool classes [cls_base + w*way, cls_base + (w+1)*way)
static int tcn_backend(arx_handle *h, const ArxTransformer &tr, const TcnWs &w, int64_t n, int way, bool tcl, float *logits, float *is_true,
                       int32_t *ch, int ep_way, int64_t cls_base, cudaStream_t st) {
  const int ldg = 2 * tr.c * h->D;
  int rc;
  if ((rc = support_wait(h, st))) return rc;          // tup_packed and the class tiles come from the support chain
  if ((rc = arx_tcn_prep_query(h, tr, w.G, ldg, n, w.kq, st))) return rc;
  if ((rc = prof_mark(h, 3, st))) return rc;
  if ((rc = arx_tcn_attention(h, tr, w.kq, w.G, ldg, n, way, w.partial, logits, ch, w.vq, ep_way > 0, cls_base, st))) return rc;
  if ((rc = prof_mark(h, 4, st))) return rc;
  if (!is_true) return ARX_OK;
  if (tcl && ((int64_t)tr.N * h->T) % 64)       // fc1's K is padded to whole 64-column sub-tiles: the pad columns must be zero, not stale
    ARX_CUDA(h, cudaMemsetAsync(w.y_img, 0, (size_t)((n + 127) / 128 * 128) * h->tl_d1.nk * 64 * sizeof(__half), st));
  if ((rc = arx_tcn_head(h, tr, w.kq, w.G, ldg, n, ch, w.uab, w.y, w.y_img, tcl ? h->tl_d1.nk : 0, w.vq_head, ep_way, cls_base, st))) return rc;
  return tcl ? disc_tail_tc(h, w.y_img, w.h1_img, n, is_true, st) : disc_tail_fp32(h, tr, w.y, w.h1, w.h2, n, is_true, st);
}

// ep_way > 0: episode mode -- window b attends classes [b*ep_way, (b+1)*ep_way) of the support pool; the windows may
// still be split into several passes (the kernels take the pass's first pool class)
static int score_tcn(arx_handle *h, int ti, const Query &q, int64_t n_windows, const Outputs &out, cudaStream_t st, int ep_way) {
  const ArxTransformer &tr = h->tr[ti];
  const bool disc = out.is_true != nullptr, tcl = tc_front_end(h, ARX_ROUTE_TILED);
  const int way = ep_way > 0 ? ep_way : h->way;
  if (!tr.kc_tiles) return arx_fail(h, ARX_ERR_STATE, "score: support operands of the tiled kernels are missing (set the support set again)");
  if (disc && !tr.uc_tiles) return arx_fail(h, ARX_ERR_INVALID, "score: the open-set head of the tiled kernels needs pair tuples and T <= 64");
  auto carve = [&](int64_t n, void *base) { return carve_tcn(h, tr, q, n, way, disc, tcl, base); };
  const int64_t chunk = pass_windows(h, n_windows, carve);
  TcnWs w;
  int32_t *chosen_ws;
  int rc = pass_reserve(h, chunk, out.chosen, carve, &w, &chosen_ws);
  if (rc) return rc;
  const int ldg = 2 * tr.c * h->D;
  const int f_nk = tr.tl_proj.nk, f_onehot = tr.table_in_gemm ? f_nk - 1 : -1;     // feature image: + one-hot sub-tile
  h->last_path = ARX_ROUTE_TILED;
  for (int64_t b0 = 0; b0 < n_windows; b0 += chunk) {
    const int64_t n = std::min(chunk, n_windows - b0), rows = q.n_rows(h, n);
    if ((rc = prof_mark(h, 0, st))) return rc;
    if (!tcl) {
      if ((rc = front_end_fp32(h, tr, q, b0, n, w.H1, w.FE, w.P, w.G, st))) return rc;
    } else if (q.kind == Query::FRAMES) {
      // frame stream: embed and project every frame once (position-independent), then form the windows' projections
      const ArxTcLinear &L = tr.table_in_gemm ? tr.tl_proj_nt : tr.tl_proj;
      if ((rc = embed_frames_tc(h, q.at(h, b0), q.f16, rows, w.x_img, w.h_img, w.f_img, f_nk, -1, st))) return rc;
      if ((rc = prof_mark(h, 1, st))) return rc;
      if ((rc = arx_tc_linear_f32(h, L, w.f_img, f_nk, rows, w.P, ldg, nullptr, 1, st))) return rc;
      if ((rc = arx_form_windows_launch(h, tr, w.P, nullptr, w.G, nullptr, n, false, st))) return rc;
    } else {
      if (q.poses()) {
        if ((rc = embed_frames_tc(h, q.at(h, b0), q.f16, rows, w.x_img, w.h_img, w.f_img, f_nk, f_onehot, st))) return rc;
      } else if ((rc = arx_tc_rows_to_img(h, q.at(h, b0), false, h->F, h->F, rows, w.f_img, f_nk, f_onehot, st))) return rc;
      if ((rc = prof_mark(h, 1, st))) return rc;
      if ((rc = arx_tc_linear_f32(h, tr.tl_proj, w.f_img, f_nk, rows, w.G, ldg, tr.table_in_gemm ? nullptr : tr.bp, h->T, st))) return rc;
    }
    if ((rc = prof_mark(h, 2, st))) return rc;
    int32_t *ch = out.chosen ? out.chosen + b0 : chosen_ws;
    if ((rc = tcn_backend(h, tr, w, n, way, tcl, out.logits + b0 * way, disc ? out.is_true + b0 : nullptr, ch, ep_way, b0 * way, st)))
      return rc;
    if ((rc = prof_mark(h, 5, st))) return rc;
  }
  return ARX_OK;
}

// ---- the metric shape: T=16 pair tuples on the dedicated pipeline ---------------------------------------------------
// frames -> fp16 image -> fc1 -> fc2 (persistent weight-resident GEMMs) -> K/V projection into the chunked fp32 buffer ->
// tuple images (gather + LayerNorm + exp2 pre-scale) -> [join the support chain] -> cross-attention + distances ->
// logits / argmax -> open-set head by linearity -> fc1 -> fc2 + fc3 + sigmoid.  Replayed as two CUDA graphs (before /
// after the join) when the arguments recur.
static int score_gen3(arx_handle *h, int ti, const Query &q, int64_t n_windows, const Outputs &out, cudaStream_t st, int ep_way) {
  const ArxTransformer &tr = h->tr[ti];
  const bool disc = out.is_true != nullptr;
  const int way = ep_way > 0 ? ep_way : h->way;
  if (disc && (ti != 0 || !tr.uc_img)) return arx_fail(h, ARX_ERR_STATE, "score: open-set head operands missing (set the support set again)");
  const bool big_batch = n_windows * h->T >= 128ll * 2 * h->sm_count;             // persistent GEMMs pay off from ~2 tiles per SM
  const bool p_embed = big_batch && (h->tc_variant & 1024) == 0 && arx_tcp_supported(h->tl_fc1) && arx_tcp_supported(h->tl_fc2);
  auto carve = [&](int64_t n, void *base) { return carve_pair(h, tr, q, n, way, disc, base); };
  const int64_t chunk = pass_windows(h, n_windows, carve);
  // the episode-mode kernels take no pool class offset: arx_score_episodes sizes its passes to one chunk
  if (ep_way > 0 && chunk < n_windows) return arx_fail(h, ARX_ERR_INVALID, "score: an episode pass of the pair pipeline exceeds one chunk");
  PairWs w;
  int32_t *chosen_ws;
  int rc = pass_reserve(h, chunk, out.chosen, carve, &w, &chosen_ws);
  if (rc) return rc;
  h->last_path = ARX_ROUTE_PAIR;
  bool aux_pending = false;
  // A support chain still running on the side stream (set_support right before this pass) is six small dependent kernels;
  // the persistent front-end kernels own every SM with their shared memory, so the chain only advanced in the gaps between
  // them and the join below waited ~25 us for it.  The front end leaves it a few SMs of its own.
  const int reserve = (h->support_inflight && big_batch && (h->tc_variant & 32768) == 0) ? h->sm_reserve_n : 0;      // debug bit 32768: no reserved SMs
  const int sms = h->sm_count - reserve;
  ArxScoreGraph *sg = nullptr;
  bool capturable = st != nullptr && st != cudaStreamLegacy && st != cudaStreamPerThread && graphs_enabled(h);     // the default streams cannot be captured
  if (capturable && capture_id(st) != 0) capturable = false;      // a caller that is capturing this stream itself gets plain launches
  if (capturable && disc && q.kind == Query::WINDOWS && chunk >= n_windows && !h->prof_on && !h->trace_buf) {
    ArxScoreGraphKey key;
    key.q = q.rows; key.lo = out.logits; key.it = out.is_true; key.ch = out.chosen; key.ws = h->ws; key.n = n_windows; key.way = way;
    key.variant = h->tc_variant | (h->pdl ? (1 << 20) : 0) | (ep_way > 0 ? (1 << 21) : 0) | (q.f16 ? (1 << 22) : 0) | (reserve ? (1 << 23) : 0);
    key.poly = h->attn_poly; key.stagger = h->attn_stagger; key.sgen = h->support_gen; key.wgen = h->weights_gen;
    sg = score_graph_lookup(h, key);
  }
  const int f_nk = tr.tl_proj.nk, f_onehot = tr.table_in_gemm ? f_nk - 1 : -1;     // feature image: + one-hot sub-tile
  const int g_ld = 2 * tr.c * h->D, g_voff = tr.c * h->D;
  for (int64_t b0 = 0; b0 < n_windows; b0 += chunk) {
    const int64_t n = std::min(chunk, n_windows - b0), rows = q.n_rows(h, n);
    if ((rc = prof_mark(h, 0, st))) return rc;
    rc = score_segment(h, sg, 0, st, [&]() -> int {
      int rc = ARX_OK;
      const float alpha = ARX_SOFTMAX_LOG2E / sqrtf((float)h->D);
      const void *xq = q.at(h, b0);
      if (q.kind == Query::FRAMES) {
        // every frame is embedded and projected ONCE (position-independent); the windows are formed on the device
        if ((rc = embed_frames_tc(h, xq, q.f16, rows, w.x_img, w.h_img, w.f_img, f_nk, -1, st))) return rc;
        if ((rc = prof_mark(h, 1, st))) return rc;
        if ((rc = arx_tc_linear_f32(h, tr.tl_proj_nt, w.f_img, f_nk, rows, w.P, g_ld, nullptr, 1, st))) return rc;
        if (disc && (rc = arx_tc_linear_f32_small(h, tr.tl_uab, w.f_img, f_nk, rows, w.U, 32, nullptr, h->T, st))) return rc;
        if ((rc = arx_form_windows_launch(h, tr, w.P, disc ? w.U : nullptr, w.G, w.uab, n, true, st))) return rc;
        if ((rc = prof_mark(h, 2, st))) return rc;
        if ((rc = arx_tuple_img(h, tr, w.G, g_ld / 32, n, w.kq_img, alpha, sms, st))) return rc;
        return ARX_OK;
      }
      if (!q.poses()) {
        if ((rc = arx_tc_rows_to_img(h, xq, q.f16, h->F, h->F, rows, w.f_img, f_nk, f_onehot, st))) return rc;
      } else if (p_embed && (h->tc_variant & 8192) == 0 && arx_mlp_fused_supported(h, xq)) {
        if ((rc = arx_mlp_fused(h, xq, q.f16, rows, w.f_img, f_nk, f_onehot, sms, st))) return rc;      // one launch: poses -> feature image
      } else if (p_embed) {
        if ((rc = arx_tc_rows_to_img(h, xq, q.f16, h->J3, h->J3, rows, w.x_img, h->tl_fc1.nk, -1, st))) return rc;
        if ((rc = arx_tcp_linear_img(h, h->tl_fc1, w.x_img, rows, ARX_ACT_RELU, w.h_img, h->tl_fc2.nk, -1, sms, st))) return rc;
        if ((rc = arx_tcp_linear_img(h, h->tl_fc2, w.h_img, rows, ARX_ACT_RELU, w.f_img, f_nk, f_onehot, sms, st))) return rc;
      } else if ((rc = embed_frames_tc(h, xq, q.f16, rows, w.x_img, w.h_img, w.f_img, f_nk, f_onehot, st))) return rc;
      if ((rc = prof_mark(h, 1, st))) return rc;
      if ((rc = arx_tcp_linear_chunked(h, tr.tl_proj, w.f_img, f_nk, rows, w.G, sms, st))) return rc;
      if ((rc = prof_mark(h, 2, st))) return rc;
      if ((h->tc_variant & 64) == 0 && (rc = arx_tuple_img(h, tr, w.G, g_ld / 32, n, w.kq_img, alpha, sms, st))) return rc;   // bit 6: timing only
      if (disc) {
        // only the head pass reads these 32 columns: run them on a second stream, beside the tuple build + attention
        const bool aux = (h->tc_variant & 2048) == 0 && !h->prof_on && !sg;      // (a graph segment must end joined)
        cudaStream_t us = st;
        if (aux) {
          if (!h->aux_stream) {
            ARX_CUDA(h, cudaStreamCreateWithFlags(&h->aux_stream, cudaStreamNonBlocking));
            ARX_CUDA(h, cudaEventCreateWithFlags(&h->ev_aux_fork, cudaEventDisableTiming));
            ARX_CUDA(h, cudaEventCreateWithFlags(&h->ev_aux_done, cudaEventDisableTiming));
          }
          us = h->aux_stream;
          ARX_CUDA(h, cudaEventRecord(h->ev_aux_fork, st));
          ARX_CUDA(h, cudaStreamWaitEvent(us, h->ev_aux_fork, 0));
        }
        if ((rc = arx_tc_linear_f32_small(h, tr.tl_uab, w.f_img, f_nk, rows, w.uab, 32, tr.tcomp, h->T, us))) return rc;
        if (aux) { ARX_CUDA(h, cudaEventRecord(h->ev_aux_done, us)); aux_pending = true; }
      }
      return ARX_OK;
    });
    if (rc) return rc;
    if ((rc = support_wait(h, st))) return rc;                   // join the support chain (side stream) before its operands are read
    if ((rc = prof_mark(h, 3, st))) return rc;
    int32_t *ch = out.chosen ? out.chosen + b0 : chosen_ws;
    rc = score_segment(h, sg, 1, st, [&]() -> int {
      int rc = ARX_OK;
      if ((rc = arx_tc_attention(h, tr, w.kq_img, w.G, n, way, w.partial, out.logits + b0 * way, ch, g_ld, g_voff, true, ep_way > 0, st))) return rc;
      if ((rc = prof_mark(h, 4, st))) return rc;
      if (disc) {
        if (aux_pending) { ARX_CUDA(h, cudaStreamWaitEvent(st, h->ev_aux_done, 0)); aux_pending = false; }
        if ((rc = arx_tc2_head_launch(h, tr, w.kq_img, w.uab, n, ch, w.y_img, h->tl_d1.nk, ep_way, st))) return rc;
        if ((rc = disc_tail_tc(h, w.y_img, w.h1_img, n, out.is_true + b0, st))) return rc;
      }
      return ARX_OK;
    });
    if (rc) return rc;
    if ((rc = prof_mark(h, 5, st))) return rc;
  }
  if (sg) sg->seen++;
  return ARX_OK;
}

// ---- fp32 CUDA-core kernels: any shape, debug outputs (softmax scores, prototypes), forced path ---------------------
static int score_fp32(arx_handle *h, int ti, const Query &q, int64_t n_windows, const Outputs &out, cudaStream_t st) {
  const ArxTransformer &tr = h->tr[ti];
  const bool disc = out.is_true != nullptr;
  const int way = h->way;
  auto carve = [&](int64_t n, void *base) { return carve_generic(h, tr, q, n, way, disc, base); };
  const int64_t chunk = pass_windows(h, n_windows, carve);
  Fp32Ws w;
  int32_t *chosen_ws;
  int rc = pass_reserve(h, chunk, out.chosen, carve, &w, &chosen_ws);
  if (rc) return rc;
  h->last_path = ARX_ROUTE_FP32;
  const int64_t NN = (int64_t)tr.N * tr.N, ND = (int64_t)tr.N * h->D;
  for (int64_t b0 = 0; b0 < n_windows; b0 += chunk) {
    const int64_t n = std::min(chunk, n_windows - b0);
    if ((rc = prof_mark(h, 0, st))) return rc;
    if ((rc = front_end_fp32(h, tr, q, b0, n, w.H1, w.FE, w.P, w.G, st))) return rc;
    if ((rc = prof_mark(h, 2, st))) return rc;
    if ((rc = arx_fp32_build_tuples(h, tr, w.G, n, w.Kq, w.Vq, st))) return rc;
    if ((rc = support_wait(h, st))) return rc;
    if ((rc = prof_mark(h, 3, st))) return rc;
    int32_t *ch = out.chosen ? out.chosen + b0 : chosen_ws;
    if ((rc = arx_fp32_attention(h, tr, w.Kq, w.Vq, n, way, w.Z, w.partial, out.logits + b0 * way, ch, disc ? w.y : nullptr,
                                 out.probs ? out.probs + b0 * way * NN : nullptr, out.protos ? out.protos + b0 * way * ND : nullptr, st)))
      return rc;
    if ((rc = prof_mark(h, 4, st))) return rc;
    if (disc && (rc = disc_tail_fp32(h, tr, w.y, w.h1, w.h2, n, out.is_true + b0, st))) return rc;
    if ((rc = prof_mark(h, 5, st))) return rc;
  }
  return ARX_OK;
}

// ep_way > 0: episode mode -- window b is scored against classes [b*ep_way, (b+1)*ep_way) of the support pool
static int score_impl(arx_handle *h, int ti, const Query &q, int64_t n_windows, const Outputs &out, cudaStream_t st, int ep_way = 0) {
  if (!h->weights_loaded) return arx_fail(h, ARX_ERR_STATE, "score: weights not loaded");
  if (h->way < 1) return arx_fail(h, ARX_ERR_STATE, "score: support set not set");
  if (n_windows == 0) return ARX_OK;
  const ArxTransformer &tr = h->tr[ti];
  if (out.is_true && (!h->cfg.has_discriminator || ti != 0 || tr.c != 2))
    return arx_fail(h, ARX_ERR_INVALID, "score: the discriminator is sized for pair tuples of transformers[0] (model.py:283-285)");
  if (ep_way > 0 && (int64_t)ep_way * n_windows != h->way) return arx_fail(h, ARX_ERR_STATE, "score: episode pool does not match the batch");
  if (tr.route == ARX_ROUTE_NONE)
    return arx_fail(h, ARX_ERR_STATE, "score: transformers[%d] has no support operands (arx_score_episodes keeps those of transformers[0] "
                                      "only): set the support set again", ti);
  const bool debug_out = out.probs || out.protos;
  const ArxRoute route = debug_out ? ARX_ROUTE_FP32 : tr.route;      // only the fp32 kernels write the debug outputs
  int rc = workspace_wait(h, st);
  if (rc) return rc;
  if (route == ARX_ROUTE_PAIR)
    rc = score_gen3(h, ti, q, n_windows, out, st, ep_way);
  else if (route == ARX_ROUTE_TILED)
    rc = score_tcn(h, ti, q, n_windows, out, st, ep_way);
  else if (h->cfg.force_path == 2 && !debug_out)
    rc = arx_fail(h, ARX_ERR_INVALID, "score: force_path=2 but no tcgen05 path covers this shape (N=%d, D=%d)", tr.N, h->D);
  else {
    if (!debug_out) warn_fp32_fallback(h, ti);
    rc = score_fp32(h, ti, q, n_windows, out, st);
  }
  if (rc) return rc;
  return score_done_record(h, st);
}

int arx_score(arx_handle *h, const float *query_dev, int64_t n_windows, float *logits_dev, float *is_true_dev, int32_t *chosen_dev,
              void *stream) {
  if (!h || !query_dev || !logits_dev || n_windows < 0) return arx_fail(h, ARX_ERR_INVALID, "score: bad argument");
  if (!h->cfg.has_discriminator) is_true_dev = nullptr;
  return score_impl(h, 0, {query_dev, Query::WINDOWS, false}, n_windows, {logits_dev, is_true_dev, chosen_dev},
                    static_cast<cudaStream_t>(stream));
}

// Support pool of arx_score_episodes on the tiled route: a pass scores `piece` episodes against one pool of piece*way
// support classes, and piece is chosen so that the pool takes at most this many bytes (at most 256 episodes, at least one).
static const size_t ARX_EPISODE_POOL_BUDGET = (size_t)1 << 30;

// Device bytes of one class of that pool (transformer 0 only): the fp32 tuple tensors ks / vs, the class tiles Kc and
// Vc^T (and Uc for the open-set head), its rows of ss_feat and ss_poses, and its rows of the support scratch.  At T=32,
// F=256, 30 joints: pairs with the head (temp_set [2, 3], scratch sized for triples) 1 084 674 B, 49 episodes of 20-way
// per pass; triples (N=4960, temp_set [3]) 7 818 498 B, 6 episodes of 20-way per pass.  T=64 pairs with the head (N=2016,
// temp_set [2]): 3 938 818 B, 13 episodes of 20-way per pass.
static size_t tiled_pool_class_bytes(arx_handle *h) {
  const ArxTransformer &tr = h->tr[0];
  const size_t tile = 128 * 128 * sizeof(__half), ns = tr.Npad / 128;
  size_t b = 2 * (size_t)tr.N * h->D * sizeof(float);
  b += (tiled_head(h, 0) ? 3 : 2) * ns * tile;
  b += (size_t)h->T * (h->F + h->J3) * sizeof(float);
  b += support_scratch(h, 128, nullptr).bytes / 128;
  return b;
}

int arx_score_episodes(arx_handle *h, const float *support_dev, int32_t is_features, int32_t way, const float *query_dev, int64_t n_episodes,
                       float *logits_dev, float *is_true_dev, int32_t *chosen_dev, void *stream) {
  if (!h || !support_dev || !query_dev || !logits_dev || way < 1 || n_episodes < 0) return arx_fail(h, ARX_ERR_INVALID, "score_episodes: bad argument");
  if (!h->weights_loaded) return arx_fail(h, ARX_ERR_STATE, "score_episodes: weights not loaded");
  if (!h->cfg.has_discriminator) is_true_dev = nullptr;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const size_t per_class = (size_t)h->T * (is_features ? h->F : h->J3);
  // support operands of transformers[0] only: episodes are scored by it alone (model.py:320)
  auto set_support = [&](int64_t e0, int64_t n_classes) -> int {
    const float *sup = support_dev + (size_t)e0 * way * per_class;
    return is_features ? set_support_features(h, sup, (int32_t)n_classes, 1, st) : set_support_poses(h, sup, (int32_t)n_classes, 1, st);
  };
  const Query q{query_dev, Query::WINDOWS, false};
  // episodes [e0, e0 + m) against a pool of m*way support classes (ep_way = way), or one at a time against a support set of
  // their own (ep_way = 0: the same kernels as set_support + arx_score)
  auto score = [&](int64_t e0, int64_t m, int ep_way) -> int {
    const int rc = set_support(e0, m * way);
    if (rc) return rc;
    return score_impl(h, 0, {q.at(h, e0), Query::WINDOWS, false}, m,
                      {logits_dev + e0 * way, is_true_dev ? is_true_dev + e0 : nullptr, chosen_dev ? chosen_dev + e0 : nullptr},
                      st, ep_way);
  };
  auto one_at_a_time = [&](int64_t e0, int64_t e1) -> int {
    for (int64_t e = e0; e < e1; ++e)
      if (const int rc = score(e, 1, 0)) return rc;
    return ARX_OK;
  };
  // The route depends on the configuration and the weights only: decided before any pool is built.  The fp32 kernels
  // (force_path = 1, LayerNorm affines past the accuracy bound, D != 128) have no episode mode.
  const ArxRoute route = support_route(h, h->tr[0]);
  if (route == ARX_ROUTE_FP32) return one_at_a_time(0, n_episodes);
  // The pair pipeline keeps 256 episodes per pass; the tiled route sizes its pool by ARX_EPISODE_POOL_BUDGET.
  const int64_t piece = route == ARX_ROUTE_PAIR
                            ? 256
                            : std::max<int64_t>(1, std::min<int64_t>(256, (int64_t)(ARX_EPISODE_POOL_BUDGET / ((size_t)way * tiled_pool_class_bytes(h)))));
  const bool disc = is_true_dev != nullptr;
  for (int64_t e0 = 0; e0 < n_episodes; e0 += piece) {
    const int64_t m = std::min(piece, n_episodes - e0);
    // the episode-mode kernels of the pair pipeline take no pool class offset: a pass must fit one chunk
    const bool one_chunk = route != ARX_ROUTE_PAIR || pass_windows(h, m, [&](int64_t n, void *base) {
      return carve_pair(h, h->tr[0], q, n, way, disc, base);
    }) >= m;
    if (const int rc = one_chunk ? score(e0, m, way) : one_at_a_time(e0, e0 + m)) return rc;
  }
  return ARX_OK;
}

int arx_score_frames(arx_handle *h, const float *frames_dev, int64_t n_frames, float *logits_dev, float *is_true_dev, int32_t *chosen_dev,
                     void *stream) {
  if (!h || !frames_dev || !logits_dev || n_frames < 0) return arx_fail(h, ARX_ERR_INVALID, "score_frames: bad argument");
  if (!h->cfg.has_discriminator) is_true_dev = nullptr;
  const int64_t n_windows = n_frames - h->T + 1;
  if (n_windows <= 0) return ARX_OK;                      // fewer than seq_len frames: nothing to report (ar.py:43-44)
  return score_impl(h, 0, {frames_dev, Query::FRAMES, false}, n_windows, {logits_dev, is_true_dev, chosen_dev},
                    static_cast<cudaStream_t>(stream));
}

int arx_score_features(arx_handle *h, int32_t ti, const float *qfeats_dev, int64_t n_windows, float *logits_dev, void *stream) {
  if (!h || !qfeats_dev || !logits_dev || n_windows < 0 || ti < 0 || ti >= h->cfg.n_transformers)
    return arx_fail(h, ARX_ERR_INVALID, "score_features: bad argument");
  return score_impl(h, ti, {qfeats_dev, Query::FEATURES, false}, n_windows, {logits_dev, nullptr, nullptr},
                    static_cast<cudaStream_t>(stream));
}

int arx_debug_attention(arx_handle *h, const float *query_dev, int64_t n_windows, float *probs_dev, float *prototypes_dev, void *stream) {
  if (!h || !query_dev || n_windows < 0) return arx_fail(h, ARX_ERR_INVALID, "debug_attention: bad argument");
  if (h->way < 1) return arx_fail(h, ARX_ERR_STATE, "debug_attention: support set not set");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  float *logits = nullptr;
  ARX_CUDA(h, cudaMalloc(&logits, (size_t)std::max<int64_t>(1, n_windows) * h->way * sizeof(float)));
  int rc = score_impl(h, 0, {query_dev, Query::WINDOWS, false}, n_windows, {logits, nullptr, nullptr, probs_dev, prototypes_dev}, st);
  cudaStreamSynchronize(st);
  cudaFree(logits);
  return rc;
}

// fp16 host rows go straight into the fp16 operand image of the first GEMM (the fp32 path rounds to fp16 there anyway, so
// results are bit-identical for inputs that are representable in fp16)
static int score_host_impl(arx_handle *h, const void *query_host_v, bool f16, int64_t n_windows, float *logits_host, float *is_true_host,
                           int32_t *chosen_host) {
  if (!h || !query_host_v || !logits_host || n_windows < 0) return arx_fail(h, ARX_ERR_INVALID, "score_host: bad argument");
  if (h->way < 1) return arx_fail(h, ARX_ERR_STATE, "score_host: support set not set");
  if (n_windows == 0) return ARX_OK;
  if (f16 && !tc_front_end(h, h->tr[0].route)) return arx_fail(h, ARX_ERR_INVALID, "score_host_f16: fp16 rows need the tensor-core linear layers (this shape scores on the fp32 kernels)");
  const char *query_host = static_cast<const char *>(query_host_v);
  const bool disc = h->cfg.has_discriminator && is_true_host;
  const int way = h->way;
  const size_t in_per = (size_t)h->T * h->J3 * (f16 ? sizeof(__half) : sizeof(float));
  const size_t out_per = (size_t)(way + 2) * sizeof(float);   // logits | is_true | chosen
  // copy/compute overlap needs at least two chunks per call, but small chunks waste the GPU (fixed per-launch costs):
  // halve the batch (rounded to whole 128-row tiles), never below 1024 windows
  int64_t stage = h->cfg.max_chunk > 0 ? h->cfg.max_chunk : 4096;
  if (const char *e = getenv("ARX_HOST_STAGE")) stage = atoll(e);
  else stage = std::min<int64_t>(stage, std::max<int64_t>(1024, ((n_windows + 1) / 2 + 127) / 128 * 128));
  stage = std::max<int64_t>(1, std::min<int64_t>(stage, n_windows));
  if ((size_t)stage > h->stage_windows || way != h->stage_way) {
    // (re)allocate staging sized for `stage` windows at the current way
    ARX_CUDA(h, cudaDeviceSynchronize());
    for (int i = 0; i < 2; ++i) {
      cudaFree(h->dev_in[i]); cudaFree(h->dev_out[i]);
      h->dev_in[i] = h->dev_out[i] = nullptr;
      ARX_CUDA(h, cudaMalloc(&h->dev_in[i], stage * in_per));
      ARX_CUDA(h, cudaMalloc(&h->dev_out[i], stage * out_per));
      if (!h->own_stream[i]) ARX_CUDA(h, cudaStreamCreateWithFlags(&h->own_stream[i], cudaStreamNonBlocking));
      if (!h->stage_ev[i]) ARX_CUDA(h, cudaEventCreateWithFlags(&h->stage_ev[i], cudaEventDisableTiming));
    }
    h->stage_windows = (size_t)stage;
    h->stage_way = way;
  }
  // Two streams ping-pong over chunks: chunk i's H2D + compute + D2H run on stream i&1; the shared
  // workspace serialises the compute of consecutive chunks through stage_ev.
  int64_t i = 0;
  for (int64_t b0 = 0; b0 < n_windows; b0 += stage, ++i) {
    const int s = (int)(i & 1);
    const int64_t n = std::min(stage, n_windows - b0);
    cudaStream_t st = h->own_stream[s];
    float *din = static_cast<float *>(h->dev_in[s]);
    float *dlog = static_cast<float *>(h->dev_out[s]);
    float *dist = dlog + (size_t)stage * way;
    int32_t *dch = reinterpret_cast<int32_t *>(dist + stage);
    ARX_CUDA(h, cudaMemcpyAsync(din, query_host + b0 * in_per, n * in_per, cudaMemcpyHostToDevice, st));
    if (i > 0) ARX_CUDA(h, cudaStreamWaitEvent(st, h->stage_ev[s ^ 1], 0));   // previous chunk done with the workspace
    const int rc = score_impl(h, 0, {din, Query::WINDOWS, f16}, n, {dlog, disc ? dist : nullptr, dch}, st);
    if (rc) return rc;
    ARX_CUDA(h, cudaEventRecord(h->stage_ev[s], st));
    ARX_CUDA(h, cudaMemcpyAsync(logits_host + b0 * way, dlog, (size_t)n * way * sizeof(float), cudaMemcpyDeviceToHost, st));
    if (disc) ARX_CUDA(h, cudaMemcpyAsync(is_true_host + b0, dist, (size_t)n * sizeof(float), cudaMemcpyDeviceToHost, st));
    if (chosen_host) ARX_CUDA(h, cudaMemcpyAsync(chosen_host + b0, dch, (size_t)n * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  }
  ARX_CUDA(h, cudaStreamSynchronize(h->own_stream[0]));
  ARX_CUDA(h, cudaStreamSynchronize(h->own_stream[1]));
  return ARX_OK;
}

int arx_score_host(arx_handle *h, const float *query_host, int64_t n_windows, float *logits_host, float *is_true_host, int32_t *chosen_host) {
  return score_host_impl(h, query_host, false, n_windows, logits_host, is_true_host, chosen_host);
}
int arx_score_host_f16(arx_handle *h, const uint16_t *query_host_f16, int64_t n_windows, float *logits_host, float *is_true_host,
                       int32_t *chosen_host) {
  return score_host_impl(h, query_host_f16, true, n_windows, logits_host, is_true_host, chosen_host);
}

static int score_host_submit_impl(arx_handle *h, const void *query_host, bool f16, int64_t n_windows, float *logits_host, float *is_true_host,
                                  int32_t *chosen_host, int64_t *ticket) {
  if (!h || !query_host || !logits_host || !ticket || n_windows <= 0) return arx_fail(h, ARX_ERR_INVALID, "score_host_submit: bad argument");
  if (h->way < 1) return arx_fail(h, ARX_ERR_STATE, "score_host_submit: support set not set");
  if (f16 && !tc_front_end(h, h->tr[0].route)) return arx_fail(h, ARX_ERR_INVALID, "score_host_submit_f16: fp16 rows need the tensor-core linear layers");
  const bool disc = h->cfg.has_discriminator && is_true_host;
  const int way = h->way;
  const size_t in_per = (size_t)h->T * h->J3 * sizeof(float);          // staging is sized for fp32 rows (fp16 requests use half of it)
  const size_t in_bytes = (size_t)n_windows * h->T * h->J3 * (f16 ? sizeof(__half) : sizeof(float));
  const size_t out_per = (size_t)(way + 2) * sizeof(float);
  if (!h->hs_h2d) {
    ARX_CUDA(h, cudaStreamCreateWithFlags(&h->hs_h2d, cudaStreamNonBlocking));
    ARX_CUDA(h, cudaStreamCreateWithFlags(&h->hs_comp, cudaStreamNonBlocking));
    ARX_CUDA(h, cudaStreamCreateWithFlags(&h->hs_d2h, cudaStreamNonBlocking));
    for (int i = 0; i < ARX_HOST_DEPTH; ++i) {
      ARX_CUDA(h, cudaEventCreateWithFlags(&h->hs_ev_h2d[i], cudaEventDisableTiming));
      ARX_CUDA(h, cudaEventCreateWithFlags(&h->hs_ev_comp[i], cudaEventDisableTiming));
      ARX_CUDA(h, cudaEventCreateWithFlags(&h->hs_ev_done[i], cudaEventDisableTiming));
    }
  }
  if (n_windows > h->hs_cap_windows || way != h->hs_way) {
    ARX_CUDA(h, cudaDeviceSynchronize());
    for (int i = 0; i < ARX_HOST_DEPTH; ++i) {
      cudaFree(h->hs_in[i]); cudaFree(h->hs_out[i]);
      h->hs_in[i] = h->hs_out[i] = nullptr;
      ARX_CUDA(h, cudaMalloc(&h->hs_in[i], n_windows * in_per));
      ARX_CUDA(h, cudaMalloc(&h->hs_out[i], n_windows * out_per));
    }
    h->hs_cap_windows = n_windows;
    h->hs_way = way;
    h->hs_base = h->hs_submitted;      // ticket ids stay monotonic; everything before the device-wide sync above has completed
  }
  const int64_t id = h->hs_submitted;
  const int s = (int)(id % ARX_HOST_DEPTH);
  float *din = static_cast<float *>(h->hs_in[s]);
  float *dlog = static_cast<float *>(h->hs_out[s]);
  float *dist = dlog + (size_t)n_windows * way;
  int32_t *dch = reinterpret_cast<int32_t *>(dist + n_windows);
  // H2D of request id may start once the request that used this slot (id - DEPTH) has been scored
  const bool slot_used = id - h->hs_base >= ARX_HOST_DEPTH;     // this slot's buffers carried an earlier request since the last reallocation
  if (slot_used) ARX_CUDA(h, cudaStreamWaitEvent(h->hs_h2d, h->hs_ev_comp[s], 0));
  ARX_CUDA(h, cudaMemcpyAsync(din, query_host, in_bytes, cudaMemcpyHostToDevice, h->hs_h2d));
  ARX_CUDA(h, cudaEventRecord(h->hs_ev_h2d[s], h->hs_h2d));
  // scoring: after its inputs arrived and after the results previously held in this slot went back to the host
  ARX_CUDA(h, cudaStreamWaitEvent(h->hs_comp, h->hs_ev_h2d[s], 0));
  if (slot_used) ARX_CUDA(h, cudaStreamWaitEvent(h->hs_comp, h->hs_ev_done[s], 0));
  const int rc = score_impl(h, 0, {din, Query::WINDOWS, f16}, n_windows, {dlog, disc ? dist : nullptr, dch}, h->hs_comp);
  if (rc) return rc;
  ARX_CUDA(h, cudaEventRecord(h->hs_ev_comp[s], h->hs_comp));
  ARX_CUDA(h, cudaStreamWaitEvent(h->hs_d2h, h->hs_ev_comp[s], 0));
  ARX_CUDA(h, cudaMemcpyAsync(logits_host, dlog, (size_t)n_windows * way * sizeof(float), cudaMemcpyDeviceToHost, h->hs_d2h));
  if (disc) ARX_CUDA(h, cudaMemcpyAsync(is_true_host, dist, (size_t)n_windows * sizeof(float), cudaMemcpyDeviceToHost, h->hs_d2h));
  if (chosen_host) ARX_CUDA(h, cudaMemcpyAsync(chosen_host, dch, (size_t)n_windows * sizeof(int32_t), cudaMemcpyDeviceToHost, h->hs_d2h));
  ARX_CUDA(h, cudaEventRecord(h->hs_ev_done[s], h->hs_d2h));
  *ticket = id;
  h->hs_submitted = id + 1;
  return ARX_OK;
}

int arx_score_host_submit(arx_handle *h, const float *query_host, int64_t n_windows, float *logits_host, float *is_true_host,
                          int32_t *chosen_host, int64_t *ticket) {
  return score_host_submit_impl(h, query_host, false, n_windows, logits_host, is_true_host, chosen_host, ticket);
}
int arx_score_host_submit_f16(arx_handle *h, const uint16_t *query_host_f16, int64_t n_windows, float *logits_host, float *is_true_host,
                              int32_t *chosen_host, int64_t *ticket) {
  return score_host_submit_impl(h, query_host_f16, true, n_windows, logits_host, is_true_host, chosen_host, ticket);
}

int arx_score_host_wait(arx_handle *h, int64_t ticket) {
  if (!h || ticket < 0 || ticket >= h->hs_submitted) return arx_fail(h, ARX_ERR_INVALID, "score_host_wait: unknown ticket");
  if (ticket < h->hs_base) return ARX_OK;       // submitted before a staging reallocation, which synchronised the device
  // The slot's event may have been re-recorded for a newer request (submit never blocks the host): the copy-back
  // stream is in order, so that newer record completing implies this ticket's copies have landed too.
  ARX_CUDA(h, cudaEventSynchronize(h->hs_ev_done[ticket % ARX_HOST_DEPTH]));
  return ARX_OK;
}

// ---- resident streaming scorer (ar.py:30-84) ------------------------------------------------------------------------
static void stream_free(arx_handle *h) {
  ArxStream &s = h->stream;
  if (s.exec) cudaGraphExecDestroy(s.exec);
  cudaFree(s.ring); cudaFree(s.slot); cudaFree(s.x_dev); cudaFree(s.out_dev); cudaFree(s.logits);
  cudaFree(s.ws); cudaFree(s.iota); cudaFree(s.y_all);
  if (s.st2) { cudaStreamDestroy(s.st2); cudaEventDestroy(s.ev_fork); cudaEventDestroy(s.ev_join); }
  if (s.pin_in) cudaFreeHost(s.pin_in);
  if (s.pin_out) cudaFreeHost(s.pin_out);
  if (s.st) cudaStreamDestroy(s.st);
  s = ArxStream();
}

int arx_stream_reset(arx_handle *h) {
  if (!h) return ARX_ERR_INVALID;
  ArxStream &s = h->stream;
  s.count = 0;
  if (s.ring) {
    ARX_CUDA(h, cudaStreamSynchronize(s.st));
    ARX_CUDA(h, cudaMemsetAsync(s.ring, 0, (size_t)h->T * 2 * h->tr[0].c * h->D * sizeof(float), s.st));
    ARX_CUDA(h, cudaMemsetAsync(s.slot, 0, sizeof(int), s.st));
  }
  return ARX_OK;
}

int arx_stream_push(arx_handle *h, const float *frame_host, float *result_host, int32_t *valid) {
  if (!h || !frame_host || !result_host) return arx_fail(h, ARX_ERR_INVALID, "stream_push: bad argument");
  if (!h->weights_loaded) return arx_fail(h, ARX_ERR_STATE, "stream_push: weights not loaded");
  if (h->way < 1) return arx_fail(h, ARX_ERR_STATE, "stream_push: support set not set");
  ArxTransformer &tr = h->tr[0];
  const int way = h->way, NO = 2 * tr.c * h->D;
  const bool disc = h->cfg.has_discriminator != 0;
  if (h->cfg.force_path == 1 || !tc_admitted(h, tr) || !arx_tcn_supported(h, tr) || arx_tcn_needs_rowmax(tr) || tr.c != 2 ||
      h->J3 > 256 || h->H > 256 || h->F > 256)
    return arx_fail(h, ARX_ERR_INVALID, "stream_push: the resident streaming path covers pair tuples on the tiled tcgen05 kernels only");
  ArxStream &s = h->stream;
  int rc;
  if (!s.ring) {
    ARX_CUDA(h, cudaStreamCreateWithFlags(&s.st, cudaStreamNonBlocking));
    ARX_CUDA(h, cudaMalloc(reinterpret_cast<void **>(&s.ring), (size_t)h->T * NO * sizeof(float)));
    ARX_CUDA(h, cudaMalloc(reinterpret_cast<void **>(&s.slot), sizeof(int)));
    ARX_CUDA(h, cudaMalloc(reinterpret_cast<void **>(&s.x_dev), (size_t)h->J3 * sizeof(float)));
    ARX_CUDA(h, cudaMallocHost(reinterpret_cast<void **>(&s.pin_in), (size_t)h->J3 * sizeof(float)));
    ARX_CUDA(h, cudaMemsetAsync(s.ring, 0, (size_t)h->T * NO * sizeof(float), s.st));
    ARX_CUDA(h, cudaMemsetAsync(s.slot, 0, sizeof(int), s.st));
    s.count = 0;
  }
  const bool stale = s.way != way || s.sgen != h->support_seq || s.wgen != h->weights_gen;
  if (stale) {
    ARX_CUDA(h, cudaStreamSynchronize(s.st));
    if (s.exec) { cudaGraphExecDestroy(s.exec); s.exec = nullptr; }
    s.seen = 0;
    if (s.way != way) {
      cudaFree(s.out_dev); cudaFree(s.logits);
      if (s.pin_out) cudaFreeHost(s.pin_out);
      s.out_dev = s.logits = s.pin_out = nullptr;
      ARX_CUDA(h, cudaMalloc(reinterpret_cast<void **>(&s.out_dev), (size_t)(way + 1) * sizeof(float)));
      ARX_CUDA(h, cudaMalloc(reinterpret_cast<void **>(&s.logits), (size_t)way * sizeof(float)));
      ARX_CUDA(h, cudaMallocHost(reinterpret_cast<void **>(&s.pin_out), (size_t)(way + 1) * sizeof(float)));
      cudaFree(s.iota); cudaFree(s.y_all);
      s.iota = nullptr; s.y_all = nullptr;
      std::vector<int32_t> io(way);
      for (int i = 0; i < way; ++i) io[i] = i;
      ARX_CUDA(h, cudaMalloc(reinterpret_cast<void **>(&s.iota), (size_t)way * sizeof(int32_t)));
      ARX_CUDA(h, cudaMemcpy(s.iota, io.data(), (size_t)way * sizeof(int32_t), cudaMemcpyHostToDevice));
      ARX_CUDA(h, cudaMalloc(reinterpret_cast<void **>(&s.y_all), (size_t)way * tr.N * h->T * sizeof(float) + 256));
      if (!s.st2) {
        ARX_CUDA(h, cudaStreamCreateWithFlags(&s.st2, cudaStreamNonBlocking));
        ARX_CUDA(h, cudaEventCreateWithFlags(&s.ev_fork, cudaEventDisableTiming));
        ARX_CUDA(h, cudaEventCreateWithFlags(&s.ev_join, cudaEventDisableTiming));
      }
    }
    const size_t need = carve_tcn(h, tr, {nullptr, Query::FEATURES, false}, 1, way, disc, false, nullptr).bytes;      // fp32 head buffers (one window: matvec kernels)
    if (need > s.ws_bytes) {
      cudaFree(s.ws);
      s.ws = nullptr;
      ARX_CUDA(h, cudaMalloc(&s.ws, need));
      s.ws_bytes = need;
    }
    // the tiled class operands (the T=16 pair pipeline of arx_score builds its own images): from the fp32 tuple tensors
    if (h->tiles_gen[0] != h->support_seq + 1) {
      if ((rc = support_wait(h, s.st))) return rc;
      if ((rc = arx_tcn_prep_support(h, tr, way, disc, s.st))) return rc;
      h->tiles_gen[0] = h->support_seq + 1;
    }
    s.way = way; s.sgen = h->support_seq; s.wgen = h->weights_gen;
  }
  TcnWs w = carve_tcn(h, tr, {nullptr, Query::FEATURES, false}, 1, way, disc, false, s.ws);
  auto body = [&]() -> int {
    int rc;
    if ((rc = prof_mark(h, 0, s.st))) return rc;          // stage timers: 0 H2D + frame MLP/projection, 1 window + query tiles, 2 -, 3 attention, 4 head + D2H
    ARX_CUDA(h, cudaMemcpyAsync(s.x_dev, s.pin_in, (size_t)h->J3 * sizeof(float), cudaMemcpyHostToDevice, s.st));
    if ((rc = arx_stream_frame_launch(h, tr, s.x_dev, s.ring, s.slot, s.st))) return rc;
    if ((rc = prof_mark(h, 1, s.st))) return rc;
    if ((rc = arx_stream_tiles_launch(h, tr, s.ring, s.slot, w.G, w.kq, s.st))) return rc;
    if ((rc = prof_mark(h, 2, s.st))) return rc;
    if ((rc = prof_mark(h, 3, s.st))) return rc;
    const int ldg = 2 * tr.c * h->D;
    // the open-set head input of EVERY class runs on a second stream beside the main attention launch (5 + 5 CTAs): the
    // winner is only known afterwards, and at one window per call the kernels are all latency
    if (disc) {
      ARX_CUDA(h, cudaEventRecord(s.ev_fork, s.st));
      ARX_CUDA(h, cudaStreamWaitEvent(s.st2, s.ev_fork, 0));
      if ((rc = arx_tcn_head_all(h, tr, w.kq, w.G, ldg, way, s.iota, w.uab, s.y_all, w.vq_head, s.st2))) return rc;
      ARX_CUDA(h, cudaEventRecord(s.ev_join, s.st2));
    }
    if ((rc = arx_tcn_attention_partial(h, tr, w.kq, w.G, ldg, 1, way, w.partial, w.vq, false, 0, s.st))) return rc;
    if ((rc = prof_mark(h, 4, s.st))) return rc;
    if (disc) ARX_CUDA(h, cudaStreamWaitEvent(s.st, s.ev_join, 0));
    if ((rc = arx_stream_tail_launch(h, tr, w.partial, s.y_all, w.h1, s.logits, s.out_dev, s.slot, way, s.st))) return rc;
    ARX_CUDA(h, cudaMemcpyAsync(s.pin_out, s.out_dev, (size_t)(way + 1) * sizeof(float), cudaMemcpyDeviceToHost, s.st));
    if ((rc = prof_mark(h, 5, s.st))) return rc;
    return ARX_OK;
  };
  memcpy(s.pin_in, frame_host, (size_t)h->J3 * sizeof(float));
  if ((rc = support_wait(h, s.st))) return rc;            // eagerly, before any capture / replay: the support chain runs on its own stream
  const bool prof = h->prof_on;
  if (s.seen < 1 || prof || !graphs_enabled(h)) {
    if ((rc = body())) return rc;                       // first sighting: eager (allocations, one-time initialisation)
    s.seen++;
  } else if ((rc = graph_replay(h, s.st, "stream_push", &s.exec, &s.launches, body))) return rc;
  ARX_CUDA(h, cudaStreamSynchronize(s.st));
  memcpy(result_host, s.pin_out, (size_t)(way + 1) * sizeof(float));
  s.count++;
  if (valid) *valid = s.count >= h->T ? 1 : 0;            // ar.py:43-44: nothing to report before seq_len frames were seen
  h->last_path = ARX_ROUTE_TILED;
  return ARX_OK;
}

// ---- MetrABS heads: Linear(1280 -> 288) over the (8,8) feature map (modules/hpe/setup/4_create_heads_onnx.py:7-16) -----
int arx_heads_load(arx_handle *h, const float *weight, const float *bias, int32_t on_device, void *stream) {
  if (!h || !weight || !bias) return arx_fail(h, ARX_ERR_INVALID, "heads_load: bad argument");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int N = 288, K = 1280;
  float *w = nullptr, *b = nullptr;
  ARX_CUDA(h, cudaMalloc(reinterpret_cast<void **>(&w), (size_t)N * K * sizeof(float)));
  ARX_CUDA(h, cudaMalloc(reinterpret_cast<void **>(&b), (size_t)N * sizeof(float)));
  const cudaMemcpyKind kind = on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
  cudaError_t e = cudaMemcpyAsync(w, weight, (size_t)N * K * sizeof(float), kind, st);
  if (e == cudaSuccess) e = cudaMemcpyAsync(b, bias, (size_t)N * sizeof(float), kind, st);
  int rc = e == cudaSuccess ? arx_tc_linear_prepare(h, h->tl_heads, w, K, b, N, K, 256, st) : arx_fail(h, ARX_ERR_CUDA, "heads_load: %s", cudaGetErrorString(e));
  cudaStreamSynchronize(st);
  cudaFree(w);
  cudaFree(b);
  if (rc == ARX_OK) h->heads_loaded = true;
  return rc;
}

int arx_heads_forward(arx_handle *h, const float *feats_dev, int64_t n_frames, float *logits_dev, void *stream) {
  if (!h || !feats_dev || !logits_dev || n_frames < 0) return arx_fail(h, ARX_ERR_INVALID, "heads_forward: bad argument");
  if (!h->heads_loaded) return arx_fail(h, ARX_ERR_STATE, "heads_forward: heads weights not loaded");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int K = 1280, N = 288, nk = h->tl_heads.nk;
  int rc = workspace_wait(h, st);
  if (rc) return rc;
  const int64_t chunk = 512;                                  // frames per pass: 32768 rows, 84 MB of fp16 operand image
  if ((rc = arx_ws_reserve(h, (size_t)chunk * 64 * nk * 64 * sizeof(__half) + 256))) return rc;
  __half *img = static_cast<__half *>(h->ws);
  for (int64_t f0 = 0; f0 < n_frames; f0 += chunk) {
    const int64_t rows = std::min(chunk, n_frames - f0) * 64;
    if ((rc = arx_tc_rows_to_img(h, feats_dev + f0 * 64 * K, false, K, K, rows, img, nk, -1, st))) return rc;
    if ((rc = arx_tc_linear_f32(h, h->tl_heads, img, nk, rows, logits_dev + f0 * 64 * N, N, nullptr, 1, st, true))) return rc;
  }
  return score_done_record(h, st);
}

int arx_decode_heatmaps_cams(arx_handle *h, const float *logits_dev, int64_t n_frames, const float *expand_dev, int32_t n_out,
                             const float *new_K_dev, const float *homo_inv_dev, float *poses_dev, uint8_t *valid_dev, void *stream) {
  if (!h || !logits_dev || !expand_dev || !new_K_dev || !homo_inv_dev || !poses_dev || !valid_dev || n_frames < 0 || n_out < 1)
    return arx_fail(h, ARX_ERR_INVALID, "decode_heatmaps_cams: bad argument");
  return arx_decode_launch(h, logits_dev, n_frames, expand_dev, n_out, nullptr, nullptr, poses_dev, valid_dev, static_cast<cudaStream_t>(stream),
                           new_K_dev, homo_inv_dev);
}

int arx_decode_heatmaps(arx_handle *h, const float *logits_dev, int64_t n_frames, const float *expand_dev, int32_t n_out,
                        const float *new_K_host9, const float *homo_inv_host9, float *poses_dev, uint8_t *valid_dev, void *stream) {
  if (!h || !logits_dev || !expand_dev || !new_K_host9 || !homo_inv_host9 || !poses_dev || !valid_dev || n_frames < 0 || n_out < 1)
    return arx_fail(h, ARX_ERR_INVALID, "decode_heatmaps: bad argument");
  return arx_decode_launch(h, logits_dev, n_frames, expand_dev, n_out, new_K_host9, homo_inv_host9, poses_dev, valid_dev,
                           static_cast<cudaStream_t>(stream));
}

int arx_profile_enable(arx_handle *h, int32_t on) {
  if (!h) return ARX_ERR_INVALID;
  h->prof_on = on != 0;
  return ARX_OK;
}

int arx_profile_read(arx_handle *h, double *ms, int64_t *chunks, int32_t reset) {
  if (!h) return ARX_ERR_INVALID;
  const size_t per = ARX_N_STAGES + 1;
  for (size_t c = 0; c + per <= h->prof_used; c += per) {
    ARX_CUDA(h, cudaEventSynchronize(h->prof_events[c + ARX_N_STAGES]));
    for (int s = 0; s < ARX_N_STAGES; ++s) {
      float t = 0.f;
      ARX_CUDA(h, cudaEventElapsedTime(&t, h->prof_events[c + s], h->prof_events[c + s + 1]));
      h->prof_ms[s] += t;
    }
    h->prof_chunks++;
  }
  h->prof_used = 0;
  if (ms) for (int s = 0; s < ARX_N_STAGES; ++s) ms[s] = h->prof_ms[s];
  if (chunks) *chunks = h->prof_chunks;
  if (reset) {
    for (int s = 0; s < ARX_N_STAGES; ++s) h->prof_ms[s] = 0;
    h->prof_chunks = 0;
  }
  return ARX_OK;
}

int arx_debug_set(arx_handle *h, int32_t key, int32_t value) {
  if (!h) return ARX_ERR_INVALID;
  if (key == 0) { h->tc_variant = value; return ARX_OK; }
  if (key == 2) { h->pdl = value != 0; return ARX_OK; }
  if (key == 3) { h->attn_stagger = (int)value; return ARX_OK; }
  if (key == 4) { h->attn_poly = (int)value; return ARX_OK; }
  if (key == 5) { h->graphs_on = value != 0; return ARX_OK; }
  if (key == 6) { h->tcn_poly = value != 0; return ARX_OK; }
  if (key == 7) { h->tcn_free_a = value != 0; return ARX_OK; }
  if (key == 1) {   // allocate (value != 0) / free the kernel timeline trace buffer: 3 roles x 64 tiles x 8 stamps
    if (value && !h->trace_buf) {
      ARX_CUDA(h, cudaMalloc(reinterpret_cast<void **>(&h->trace_buf), 3 * 64 * 8 * sizeof(long long)));
      ARX_CUDA(h, cudaMemset(h->trace_buf, 0, 3 * 64 * 8 * sizeof(long long)));
    } else if (!value && h->trace_buf) {
      cudaFree(h->trace_buf);
      h->trace_buf = nullptr;
    }
    h->trace_sel = value;        // 1: attention kernels, 2: fused frame MLP, 3: head kernel
    return ARX_OK;
  }
  return arx_fail(h, ARX_ERR_INVALID, "debug_set: unknown key %d", key);
}

int arx_debug_read_trace(arx_handle *h, long long *host_out) {
  if (!h || !host_out || !h->trace_buf) return ARX_ERR_INVALID;
  ARX_CUDA(h, cudaMemcpy(host_out, h->trace_buf, 3 * 64 * 8 * sizeof(long long), cudaMemcpyDeviceToHost));
  return ARX_OK;
}

int64_t arx_launch_count(const arx_handle *h) { return h ? h->launches : 0; }
int arx_last_path(const arx_handle *h) { return h ? h->last_path : 0; }

}  // extern "C"

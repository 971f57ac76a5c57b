// Internal declarations shared by the translation units of libarx.so.
#pragma once
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include <string>
#include <vector>
#include <unordered_map>
#include "../../include/arx.h"

#define ARX_SOFTMAX_LOG2E 1.4426950408889634f
// Two limits on the static softmax bound |S| <= (max|gamma| sqrt(D) + ||beta||_2)^2 / sqrt(D) of norm_k's LayerNorm
// affine (ArxTransformer::softmax_bound):
//   overflow: |S| log2(e) < 100 keeps exp2 without max-subtraction inside fp32 range.  It picks the row-max variant of
//             the tiled kernels and bounds what the kernels without it may run on (arx_tc_supported, arx_tcn_needs_rowmax);
//   accuracy: |S| below these keeps the fp16 QK^T and bf16 P.V operands within the 1e-3 relative tolerance.  It
//             admits weights to the tensor-core routes by default (support_route, arx_stream_push).  Set from the B200
//             sweep in profiles/r03_ln_bound_sweep.txt.  A logit averages the rounding error over the N query tuples, so
//             at equal bound it falls like 1/sqrt(N), and the limit depends on N (DESIGN 4):
//               N >= 120 (T=16 pairs and larger): the largest swept bound whose worst error is <= 0.6e-3 (19.1), headroom
//                        for inputs the sweep did not draw;
//               N < 120 (T=8 pairs): 2.5x the error at equal bound, 7e-4 already at gamma = 1 (11.3) and 1.1e-3 at 16.3;
//                        this limit keeps gamma = 1 on the tensor cores and holds the tolerance itself, not 0.6e-3.
#define ARX_TC_ACCURACY_BOUND 19.0f
#define ARX_TC_ACCURACY_BOUND_FEW_TUPLES 12.0f
#define ARX_TC_FEW_TUPLES 120
// Below this many query tuples nothing averages the operand rounding at all, whatever the affine: at gamma = 1 the tiled
// route errs 1.05e-3 at N = 21 (T=7 pairs), 2.5e-3 at N = 10 and 1.3e-2 at N = 1, against 7.2e-4 at N = 28 (T=8 pairs)
// (B200, 1000 W power limit; profiles/r04_few_tuples_accuracy.txt, DESIGN 4).  Such transformers score on the fp32 kernels by default, and a handle none of
// whose transformers reaches it runs its front end (support side included) on the fp32 CUDA cores too.
#define ARX_TC_MIN_TUPLES 28

// A linear layer prepared for the tcgen05 GEMM: fp16 weight image [n_tiles][nk][BN x 64] + zero-padded bias
struct ArxTcLinear {
  __half *w_img = nullptr;
  float *bias = nullptr;
  int N = 0, K = 0, BN = 0, n_tiles = 0, nk = 0;
};

// Which kernels score a transformer; the values are those arx_last_path reports.  Decided when the support operands are
// built (arx_api.cu: support_route), because each route needs operands of its own.
enum ArxRoute {
  ARX_ROUTE_NONE = 0,    // no support operands yet
  ARX_ROUTE_FP32 = 1,    // fp32 CUDA-core kernels (arx_fp32.cu)
  ARX_ROUTE_PAIR = 2,    // T=16 pair pipeline (arx_tc3.cu and friends)
  ARX_ROUTE_TILED = 3,   // tiled any-N tcgen05 kernels (arx_tcn.cu)
};

struct ArxTransformer {
  int c = 0;            // tuple cardinality
  int N = 0;            // C(T,c)
  int Npad = 0;         // N rounded up to 128 (tcgen05 tile rows)
  float *pe = nullptr;      // (T,F) slice of the reference buffer
  float *wp = nullptr;      // (2cD, F): K parts then V parts of k_linear/v_linear (model.py:41-44)
  float *bp = nullptr;      // (T, 2cD) table: positional encoding through the projection + biases
  float *bp_sums = nullptr; // (T, 2) row sums of the table over the two K parts
  float *wp_ext = nullptr;  // (2cD, F+32): wp | hi(table)^T | lo(table)^T -- the table enters the GEMM through one-hot K columns (T == 16)
  bool table_in_gemm = false;
  float *ln_g = nullptr, *ln_b = nullptr;
  float ln_host[256] = {};  // host copy [gamma(128) | beta(128)] when D == 128: kernel-parameter operands of k_tuple_img
  int32_t *tuples = nullptr; // (N,c) int32, built on device
  ArxRoute route = ARX_ROUTE_NONE;   // the route the support operands below were built for
  // support operands, fp32 generic path: (W,N,D) each
  float *ks = nullptr, *vs = nullptr;
  // class operands of both tensor-core routes (arx_tc.cu): [way_cap][Npad/128] 32 KB K-major SW128 tiles, Kc fp16 (rows =
  // support tuples) and Vc^T bf16 (rows = d); the T=16 pair pipeline has one tile per class
  __half *kc_tiles = nullptr, *vct_tiles = nullptr;
  float softmax_bound = 0.f; // static |S| bound from LayerNorm affine (SURVEY 7.2-1)
  ArxTcLinear tl_proj;       // K/V projection (2cD x F) on tensor cores
  ArxTcLinear tl_proj_nt;    // the same without the positional-table columns (frame streams: the table is added per window position)
  ArxTcLinear tl_uab;        // 32 composite columns Wdr.Wv of the second-generation head pass
  float *wc = nullptr, *tcomp = nullptr;   // composite weights (32,F) and table (T,32)
  __half *uc_img = nullptr;  // pair pipeline's head: per class Wdr.Vc^T (16 x 128 fp16 B operand)
  // operands of the tiled any-N kernels only (arx_tcn.cu)
  __half *uc_tiles = nullptr;       // head: per class Wdr.Vc^T, [way_cap][Npad/128] 32 KB bf16 tiles
  uint32_t *tup_packed = nullptr;   // (N) tuple frames packed one byte each
  __half *sel_tiles = nullptr;      // one-hot frame-selection operand of every query tile (selection MMA of arx_tcn.cu)
};

// Replayable CUDA graphs of the arx_score kernel chain for one (buffers, batch, support geometry, weights) key: the
// ~14 launches of a score become two graph launches (before / after the join with the support chain), which takes
// the host off the critical path when several ranks share the box's cores.
struct ArxScoreGraphKey {
  const void *q = nullptr, *lo = nullptr, *it = nullptr, *ch = nullptr, *ws = nullptr;
  int64_t n = 0;
  int way = 0, variant = 0, poly = 0, stagger = 0;
  uint64_t sgen = 0, wgen = 0;
  bool operator==(const ArxScoreGraphKey &o) const {
    return q == o.q && lo == o.lo && it == o.it && ch == o.ch && ws == o.ws && n == o.n && way == o.way && variant == o.variant &&
           poly == o.poly && stagger == o.stagger && sgen == o.sgen && wgen == o.wgen;
  }
};
struct ArxScoreGraph {
  ArxScoreGraphKey key;
  cudaGraphExec_t exec[2] = {nullptr, nullptr};
  int64_t launches[2] = {0, 0};
  int seen = 0;
  uint64_t last_use = 0;
};

// Resident streaming scorer state (arx_stream_push): device ring of per-frame projections, its own workspace, stream,
// pinned staging and the per-frame CUDA graph.
struct ArxStream {
  float *ring = nullptr;            // (T, 2cD) position-independent projections of the last T frames
  int *slot = nullptr;              // device: ring slot the next frame goes to
  float *x_dev = nullptr, *out_dev = nullptr, *logits = nullptr;
  int32_t *iota = nullptr;
  float *y_all = nullptr;
  cudaStream_t st2 = nullptr;       // the head of all classes runs beside the main attention launch
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  float *pin_in = nullptr, *pin_out = nullptr;
  void *ws = nullptr;
  size_t ws_bytes = 0;
  cudaStream_t st = nullptr;
  cudaGraphExec_t exec = nullptr;
  int64_t launches = 0;             // kernel launches one replay of exec stands for
  uint64_t sgen = 0, wgen = 0;      // support / weights generation the graph (and the tiled operands) were built for
  int way = 0, seen = 0;
  int64_t count = 0;                // frames pushed since the last reset
};

struct arx_handle {
  arx_config cfg{};
  int device = 0;
  int sm_count = 0;
  int T = 0, J3 = 0, H = 0, F = 0, D = 0;
  bool weights_loaded = false;
  // MLP (model.py:164-180)
  float *fc1_w = nullptr, *fc1_b = nullptr, *fc2_w = nullptr, *fc2_b = nullptr;
  ArxTransformer tr[ARX_MAX_TRANSFORMERS];
  // discriminator (model.py:183-204)
  float *dr_w = nullptr, *dr_b = nullptr, *d1_w = nullptr, *d1_b = nullptr;
  float *d2_w = nullptr, *d2_b = nullptr, *d3_w = nullptr, *d3_b = nullptr;
  ArxTcLinear tl_fc1, tl_fc2, tl_d1, tl_d2;
  ArxTcLinear tl_heads;        // MetrABS heads Linear(1280 -> 288) in front of the heatmap decoder (arx_heads_*)
  bool heads_loaded = false;
  bool tc_linears = false;     // frame MLP / projection / discriminator MLP run on tensor cores
  // support set
  int way = 0;
  int way_cap = 0;
  float *ss_feat = nullptr;   // (W,T,F)
  void *ss_scratch = nullptr;
  size_t ss_scratch_bytes = 0;
  // the support chain runs on an internal side stream, overlapped with the query-side frame kernels of the next
  // arx_score; consumers join on ev_support_done, producers wait for ev_score_done (operands still being read)
  cudaStream_t side_stream = nullptr;
  cudaEvent_t ev_fork = nullptr, ev_support_done = nullptr, ev_score_done = nullptr;
  // second side stream inside arx_score: the 32-column head projection runs beside the K/V projection and attention
  cudaStream_t aux_stream = nullptr;
  cudaEvent_t ev_aux_fork = nullptr, ev_aux_done = nullptr;
  bool support_recorded = false, score_recorded = false;
  unsigned long long support_cid = 0, score_cid = 0;   // capture the events were last recorded in (0 = eagerly), see arx_api.cu
  cudaStream_t last_score_stream = nullptr;   // stream of the last scoring pass (ev_score_done was recorded there)
  float *ss_poses = nullptr;       // copy of the support poses when the features were produced on tensor cores
  bool ss_poses_valid = false;
  bool ss_feat_valid = false;      // ss_feat holds fp32 features (else they are derived lazily from ss_poses)
  // workspace (grown on demand)
  void *ws = nullptr;
  size_t ws_bytes = 0;
  // device staging for arx_score_host
  void *dev_in[2] = {nullptr, nullptr};
  void *dev_out[2] = {nullptr, nullptr};
  size_t stage_windows = 0;
  int stage_way = 0;
  cudaStream_t own_stream[2] = {nullptr, nullptr};
  cudaEvent_t stage_ev[2] = {nullptr, nullptr};
  // streaming host path (arx_score_host_submit / _wait)
  cudaStream_t hs_h2d = nullptr, hs_comp = nullptr, hs_d2h = nullptr;
  void *hs_in[ARX_HOST_DEPTH] = {nullptr, nullptr};
  void *hs_out[ARX_HOST_DEPTH] = {nullptr, nullptr};
  cudaEvent_t hs_ev_h2d[ARX_HOST_DEPTH] = {nullptr, nullptr}, hs_ev_comp[ARX_HOST_DEPTH] = {nullptr, nullptr}, hs_ev_done[ARX_HOST_DEPTH] = {nullptr, nullptr};
  int64_t hs_cap_windows = 0, hs_submitted = 0, hs_base = 0;   // tickets below hs_base predate the last staging reallocation
  int hs_way = 0;
  int64_t launches = 0;
  // stage timers (arx_profile_*)
  bool prof_on = false;
  std::vector<cudaEvent_t> prof_events;   // ARX_N_STAGES+1 events per recorded chunk
  size_t prof_used = 0;
  double prof_ms[ARX_N_STAGES] = {0, 0, 0, 0, 0};
  int64_t prof_chunks = 0;
  int last_path = 0;
  std::vector<ArxScoreGraph> graphs;     // small LRU cache (arx_score with recurring arguments)
  uint64_t graph_tick = 0, support_gen = 0, weights_gen = 0;
  uint64_t support_seq = 0;              // increments whenever a new support set is set / imported
  int graphs_on = -1;                    // -1: from the environment (ARX_GRAPHS=0 disables), else 0/1 (debug key 5)
  // one-time per-DEVICE initialisation done by this handle (__constant__ tables, function attributes): kept per handle,
  // not process-wide, so a second handle on another GPU of the same process initialises its own device
  uint32_t dev_init = 0;
  uint32_t warned = 0;              // per-transformer: the fp32-fallback notice was printed
  std::unordered_map<const void *, int> smem_attr;   // dynamic shared-memory limit already set per kernel (saves a driver call per launch)
  float *zscratch = nullptr;        // softmax normaliser partials of the tiled attention kernel (arx_tcn.cu), per CTA
  size_t zscratch_bytes = 0;
  ArxStream stream;
  uint64_t tiles_gen[ARX_MAX_TRANSFORMERS] = {0, 0, 0, 0};   // support generation the tiled route's extras (tables, Uc tiles) were built for (+1)
  float mlp_bias_host[192 + 256] = {};   // host copies of the (zero padded) fc1 / fc2 biases: kernel-parameter operands of k_mlp_p
  bool mlp_bias_host_ok = false;
  bool support_inflight = false;    // a support chain was forked onto the side stream and no scoring pass has joined it yet
  int sm_reserve_n = 4;             // SMs the persistent front-end kernels leave free for that chain (environment variable ARX_SM_RESERVE overrides)
  int tcn_free_a = 1;               // tiled attention, pass A: softmax groups free-running (debug key 7)
  int tcn_poly = 1;                 // tiled attention, pass A: half of the exponentials on the FMA pipe (debug key 6)
  int *tcn_diag = nullptr;          // watchdog record of the tiled attention kernel
  long long *trace_buf = nullptr;   // debug: device buffer for kernel timeline traces (arx_debug_set key 1)
  int trace_sel = 0;                // which kernel writes it: 1 attention kernels, 2 fused frame MLP, 3 head kernel
  int attn_stagger = -1;     // k_attn_tc3 softmax groups: < 0 = take turns on the MUFU phase (token), >= 0 = free-running, group 1 this many clocks behind (debug key 3)
  int attn_poly = 0;         // k_attn_tc3: every attn_poly-th register pair takes the FMA-pipe exp2 polynomial (0 = none; debug key 4)
  bool pdl = false;     // programmatic dependent launch for the arx_score kernel chain (debug key 2; measured: no gain, off by default)
  int tc_variant = 0;   // debug key 0: kernel-variant bit mask (include/arx.h)
  std::string err;
};

int arx_fail(arx_handle *h, int code, const char *fmt, ...);
#define ARX_CUDA(h, expr)                                                              \
  do {                                                                                 \
    cudaError_t _e = (expr);                                                           \
    if (_e != cudaSuccess)                                                             \
      return arx_fail((h), ARX_ERR_CUDA, "%s failed: %s (%s:%d)", #expr,               \
                      cudaGetErrorString(_e), __FILE__, __LINE__);                     \
  } while (0)
#define ARX_LAUNCH_CHECK(h)                                                            \
  do {                                                                                 \
    (h)->launches++;                                                                   \
    ARX_CUDA((h), cudaGetLastError());                                                 \
  } while (0)

int arx_ws_reserve(arx_handle *h, size_t bytes);
enum ArxDevInit { ARX_INIT_PSLOTS = 1 };

// cudaFuncSetAttribute(MaxDynamicSharedMemorySize) once per kernel and size instead of once per launch
template <class K> inline int arx_func_smem(arx_handle *h, K kern, int bytes) {
  const void *key = reinterpret_cast<const void *>(kern);
  auto it = h->smem_attr.find(key);
  if (it != h->smem_attr.end() && it->second == bytes) return ARX_OK;
  ARX_CUDA(h, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
  h->smem_attr[key] = bytes;
  return ARX_OK;
}

// Launch with programmatic stream serialization (PDL): the kernel may start while its predecessor in the stream is
// still running; it must execute griddepcontrol.wait before touching the predecessor's output.
template <class... KArgs, class... Args>
static inline cudaError_t arx_launch_pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, bool pdl, Args... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr; cfg.numAttrs = pdl ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kern, KArgs(args)...);
}

// ---- fp32 generic kernels (arx_fp32.cu) ------------------------------------------
enum ArxAct { ARX_ACT_NONE = 0, ARX_ACT_RELU = 1, ARX_ACT_SIGMOID = 2 };
// C[M,N] = act(A[M,K] * W[N,K]^T + bias[N]) (+ pe[(row % peT), N] after act when pe != nullptr)
int arx_fp32_linear(arx_handle *h, const float *A, int lda, const float *W, int ldw, const float *bias,
                    float *C, int ldc, int64_t M, int N, int K, int act, const float *pe, int peT,
                    cudaStream_t st);
// tuple K (LayerNorm-ed) and V from per-frame projections G (rows = n_seq*T, 2cD)
int arx_fp32_build_tuples(arx_handle *h, const ArxTransformer &tr, const float *G, int64_t n_seq,
                          float *K, float *V, cudaStream_t st);
// attention + distances (two passes), see arx_fp32.cu
int arx_fp32_attention(arx_handle *h, const ArxTransformer &tr, const float *Kq, const float *Vq,
                       int64_t n_win, int way, float *Z, float *partial, float *logits, int32_t *chosen,
                       float *y /* (n_win, N*T) or null */, float *probs, float *protos, cudaStream_t st);


// ---- tcgen05 kernels (arx_tc.cu) -------------------------------------------------
bool arx_tc_supported(const arx_handle *h, const ArxTransformer &tr);
// Kc / Vc^T class tiles of `way` classes from the fp32 tuple tensors ks / vs
int arx_tc_class_tiles(arx_handle *h, ArxTransformer &tr, int way, cudaStream_t st);
// ks / vs (and with_tiles: the single class tile of every class) from the per-frame projections G, one launch
int arx_tc_support_build(arx_handle *h, ArxTransformer &tr, const float *G, int way, bool with_tiles, cudaStream_t st);
// logits (n_win, way) and chosen (n_win) from the squared-distance partials (n_win*way, 4) of either tensor-core route
int arx_tc_finish(arx_handle *h, const float *partial, float *logits, int32_t *chosen, int64_t n_win, int way, int N, bool pdl, cudaStream_t st);
int arx_tc_attention(arx_handle *h, const ArxTransformer &tr, const __half *kq_img, const float *G, int64_t n_win, int way, float *partial,
                     float *logits, int32_t *chosen, int g_ld, int g_voff, bool g_chunked, bool episodes, cudaStream_t st);

// ---- tcgen05 GEMM (arx_gemm_tc.cu) ------------------------------------------------
int arx_tc_linear_prepare(arx_handle *h, ArxTcLinear &L, const float *W, int ldw, const float *bias, int N, int K, int BN, cudaStream_t st);
// 64-column sub-tiles per row tile that the fp16 image epilogues of layer L write: every column of its n_tiles column tiles
inline int arx_tc_img_nk(const ArxTcLinear &L) { return L.n_tiles * L.BN / 64; }
// rows X (M, K; fp32, or fp16 when `f16`) -> fp16 operand image
int arx_tc_rows_to_img(arx_handle *h, const void *X, bool f16, int lda, int K, int64_t M, __half *img, int nk, int onehot_sub, cudaStream_t st);
// Activation image of one layer for the next: a_img has a_nk >= L.nk sub-tiles per row tile; c_img gets c_nk sub-tiles per row
// tile, at least the n_tiles * BN / 64 this layer writes (arx_tc_img_nk), or a row tile's pad columns land in the next one
int arx_tc_linear_img(arx_handle *h, const ArxTcLinear &L, const __half *a_img, int a_nk, int64_t M, int act, __half *c_img, int c_nk,
                      int onehot_sub, cudaStream_t st);
int arx_tc_linear_f32(arx_handle *h, const ArxTcLinear &L, const __half *a_img, int a_nk, int64_t M, float *C, int ldc, const float *table, int T,
                      cudaStream_t st, bool with_bias = false);
int arx_tc_linear_sigmoid_dot(arx_handle *h, const ArxTcLinear &L, const __half *a_img, int64_t M, const float *w3, const float *b3, float *out,
                              cudaStream_t st);

// ---- padded-triangular slot order of the C(16,2) pairs (shared with the host-side slot table) ---------
// row i: i even -> slots for j = i..15 (the j == i slot is a pad), i odd -> j = i+1..15; every row has even length.
__host__ __device__ constexpr int arx_slot_row_len(int i) { return (i % 2 == 0) ? 16 - i : 15 - i; }
__host__ __device__ constexpr int arx_slot_row_start(int i) {
  int s = 0;
  for (int k = 0; k < i; ++k) s += arx_slot_row_len(k);
  return s;
}
__host__ __device__ constexpr int arx_slot_i(int q) {
  int i = 0;
  while (q >= arx_slot_row_start(i + 1)) ++i;
  return i;
}
__host__ __device__ constexpr int arx_slot_j(int q) {   // == i for a pad slot
  const int i = arx_slot_i(q), off = q - arx_slot_row_start(i);
  return (i % 2 == 0) ? i + off : i + 1 + off;
}
static_assert(arx_slot_row_start(16) == 128, "slot layout must fill the 128-column tile exactly");

void arx_tc2_slot_table(int32_t *out /* 256 */);
int arx_tc_table_sums(arx_handle *h, const float *table, int T, int ld, float *out, cudaStream_t st);

int arx_tc2_head_prepare_weights(arx_handle *h, ArxTransformer &tr, cudaStream_t st);
int arx_tc2_support_uc(arx_handle *h, ArxTransformer &tr, int way, cudaStream_t st);
int arx_tc2_head_launch(arx_handle *h, const ArxTransformer &tr, const __half *kq_img, const float *uab, int64_t n_win, const int32_t *chosen,
                        __half *y_img, int y_nk, int cls_stride, cudaStream_t st);
int arx_tc_linear_f32_small(arx_handle *h, const ArxTcLinear &L, const __half *a_img, int a_nk, int64_t M, float *C, int ldc, const float *table,
                            int T, cudaStream_t st);

int arx_tc_build_wp_ext(arx_handle *h, const float *wp, const float *table, float *out, int N, int F, cudaStream_t st);

int arx_tc3_attention_launch(arx_handle *h, const ArxTransformer &tr, const __half *kq_img, const float *G, int64_t n_win, int way,
                             float *partial, int g_ld, int g_voff, bool g_chunked, bool episodes, cudaStream_t st);
// ---- persistent GEMM + tuple images (arx_gemm_p.cu)
bool arx_tcp_supported(const ArxTcLinear &L);
// The persistent kernels below run on at most `sms` SMs (fewer than sm_count leave room to a support chain in flight).
// fused frame MLP (arx_mlp_p.cu)
bool arx_mlp_fused_supported(const arx_handle *h, const void *x);
int arx_mlp_fused(arx_handle *h, const void *x, bool f16, int64_t rows, __half *f_img, int c_nk, int onehot_sub, int sms, cudaStream_t st);
int arx_tcp_linear_img(arx_handle *h, const ArxTcLinear &L, const __half *a_img, int a_nk, int64_t M, int act, __half *c_img, int c_nk,
                       int onehot_sub, int sms, cudaStream_t st);
int arx_tcp_linear_chunked(arx_handle *h, const ArxTcLinear &L, const __half *a_img, int a_nk, int64_t M, float *gc, int sms, cudaStream_t st);
int arx_tuple_img(arx_handle *h, const ArxTransformer &tr, const float *gc, int n_chunks, int64_t n_win, __half *kq_img, float alpha,
                  int sms, cudaStream_t st);

// ---- tiled any-N tcgen05 attention (arx_tcn.cu)
bool arx_tcn_supported(const arx_handle *h, const ArxTransformer &tr);
bool arx_tcn_needs_rowmax(const ArxTransformer &tr);
// the open-set head on the tiled kernels: pair tuples, head columns L = T <= 64 (TMEM lanes of the MODE 1 accumulator)
bool arx_tcn_head_supported(const arx_handle *h, const ArxTransformer &tr);
// columns per frame part of the head table UAB (row stride 2x this): 32 for T <= 32, 64 above
int arx_tcn_head_cols(int T);
// the tiled route's own support-side operands: packed tuples and selection tiles (once per handle), with_head the Uc tiles
int arx_tcn_prep_extras(arx_handle *h, ArxTransformer &tr, int way, bool with_head, cudaStream_t st);
int arx_tcn_prep_query(arx_handle *h, const ArxTransformer &tr, const float *G, int ldg, int64_t n_win, __half *kq_tiles, cudaStream_t st);
int arx_tcn_attention(arx_handle *h, const ArxTransformer &tr, const __half *kq_tiles, const float *G, int ldg, int64_t n_win, int way,
                      float *partial, float *logits, int32_t *chosen, __half *vq_ws, bool episodes, int64_t cls_base, cudaStream_t st);
int arx_tcn_head(arx_handle *h, const ArxTransformer &tr, const __half *kq_tiles, const float *G, int ldg, int64_t n_win, const int32_t *chosen,
                 float *uab, float *y, __half *y_img, int y_nk, __half *vq_ws, int ep_way, int64_t cls_base, cudaStream_t st);

int arx_tcn_head_all(arx_handle *h, const ArxTransformer &tr, const __half *kq_tiles, const float *G, int ldg, int way, const int32_t *iota,
                     float *uab, float *y_all, __half *vq_ws, cudaStream_t st);
int arx_tcn_attention_partial(arx_handle *h, const ArxTransformer &tr, const __half *kq_tiles, const float *G, int ldg, int64_t n_win, int way,
                              float *partial, __half *vq_ws, bool episodes, int64_t cls_base, cudaStream_t st);

// ---- streaming kernels (arx_stream.cu)
int arx_stream_frame_launch(arx_handle *h, const ArxTransformer &tr, const float *x_dev, float *ring, int *slot_next, cudaStream_t st);
int arx_stream_tiles_launch(arx_handle *h, const ArxTransformer &tr, const float *ring, const int *slot_next, float *G, __half *kq, cudaStream_t st);
int arx_stream_tail_launch(arx_handle *h, const ArxTransformer &tr, const float *partial, const float *y_all, float *h1, float *logits, float *out,
                           int *slot_next, int way, cudaStream_t st);

int arx_form_windows_launch(arx_handle *h, const ArxTransformer &tr, const float *P, const float *U, float *G, float *uab, int64_t n_win, bool chunked,
                            cudaStream_t st);

// ---- tuple table (arx_tuples.cu) -------------------------------------------------
int arx_build_tuple_table(arx_handle *h, int T, int c, int N, int32_t *out_dev, cudaStream_t st);

// ---- decode (arx_decode.cu) ------------------------------------------------------
int arx_decode_launch(arx_handle *h, const float *logits, int64_t n_frames, const float *expand, int n_out,
                      const float *K9, const float *R9, float *poses, uint8_t *valid, cudaStream_t st, const float *Ks_dev = nullptr,
                      const float *Rs_dev = nullptr);

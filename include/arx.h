/*
 * arx.h -- C ABI of the B200-native ISBFSAR action-recognition scoring path.
 *
 * The reference (steb6/ISBFSAR) has no native/FFI boundary: the path sits behind
 * its Python API (modules/ar/utils/model.py, modules/ar/ar.py).  This header is
 * the boundary a binding would use; isbfsar_b200/_lib.py binds it with ctypes
 * and isbfsar_b200/{model,ar}.py mirror the reference classes on top of it.
 * Each entry point cites the reference code it replaces (paths relative to the
 * reference root).
 *
 * Conventions
 *   - every function returns 0 on success or a negative arx_status; nothing
 *     throws across the boundary; arx_last_error() gives the message.
 *   - all pointers named *_dev are CUDA device pointers on the handle's device,
 *     fp32 unless stated, C-contiguous in the reference's own layouts.
 *   - all work is enqueued on the caller's stream (a cudaStream_t passed as
 *     void*); no hidden synchronisation except in the *_host entry points.
 *   - the caller owns every I/O buffer; the handle owns weight copies, the
 *     support-set operands and the scratch workspace.  One handle per device,
 *     not thread-safe (the reference is single-threaded, main.py:111).
 *   - inference only (the reference calls it under torch.no_grad(), ar.py:68).
 */
#ifndef ARX_H
#define ARX_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ARX_ABI_VERSION 1
#if defined(__GNUC__)
#define ARX_API __attribute__((visibility("default")))
#else
#define ARX_API
#endif
#define ARX_MAX_TRANSFORMERS 4

typedef enum arx_status {
  ARX_OK = 0,
  ARX_ERR_INVALID = -1,   /* bad argument / unsupported configuration */
  ARX_ERR_CUDA = -2,      /* a CUDA runtime call failed               */
  ARX_ERR_STATE = -3,     /* call order (weights/support not set)     */
  ARX_ERR_NOMEM = -4
} arx_status;

/* Mirror of the TRXConfig fields the path reads (utils/params.py:50-95). */
typedef struct arx_config {
  int32_t seq_len;        /* T; 16 (utils/params.py:8)                                   */
  int32_t n_joints;       /* J; MLP input = 3*J, hidden = 6*J (model.py:269)             */
  int32_t feat_dim;       /* F = trans_linear_in_dim = MLP output = 256                  */
  int32_t out_dim;        /* D = trans_linear_out_dim = 128                              */
  int32_t n_transformers; /* len(temp_set) (model.py:279)                                */
  int32_t cardinality[ARX_MAX_TRANSFORMERS]; /* temp_set entries, 2 or 3                 */
  int32_t has_discriminator; /* 1 for model="DISC" (model.py:282-285)                    */
  int32_t max_chunk;      /* windows processed per internal pass (0 = default)           */
  int32_t force_path;     /* 0 = auto, 1 = fp32 CUDA-core kernels, 2 = tcgen05 kernels   *
                           * (also for LayerNorm affines past the accuracy bound, DESIGN 4) */
} arx_config;

/* Weights in the reference state_dict layouts (SURVEY.md 8b); host or device fp32. */
typedef struct arx_weights {
  int32_t on_device;                     /* 1: pointers are device pointers             */
  const float *fc1_w, *fc1_b;            /* features_extractor.sk.fc1 (6J,3J),(6J)      */
  const float *fc2_w, *fc2_b;            /* features_extractor.sk.fc2 (F,6J),(F)        */
  const float *pe[ARX_MAX_TRANSFORMERS];     /* transformers.i.pe.pe (1,int(1.5T),F)    */
  const float *k_w[ARX_MAX_TRANSFORMERS];    /* transformers.i.k_linear.weight (D,c*F)  */
  const float *k_b[ARX_MAX_TRANSFORMERS];
  const float *v_w[ARX_MAX_TRANSFORMERS];    /* transformers.i.v_linear.weight (D,c*F)  */
  const float *v_b[ARX_MAX_TRANSFORMERS];
  const float *ln_g[ARX_MAX_TRANSFORMERS];   /* transformers.i.norm_k.weight (D)        */
  const float *ln_b[ARX_MAX_TRANSFORMERS];
  const float *dr_w, *dr_b;              /* discriminator.dimensionality_reduction (T,D)*/
  const float *d1_w, *d1_b;              /* discriminator.fc1 (256, C(T,2)*T)           */
  const float *d2_w, *d2_b;              /* discriminator.fc2 (64,256)                  */
  const float *d3_w, *d3_b;              /* discriminator.fc3 (1,64)                    */
} arx_weights;

typedef struct arx_handle arx_handle;

/* TRXOS.__init__ (model.py:261-289): allocate a scorer on the current CUDA device. */
ARX_API int arx_create(const arx_config *cfg, arx_handle **out);
ARX_API void arx_destroy(arx_handle *h);
ARX_API const char *arx_last_error(const arx_handle *h);   /* h may be NULL: last create error */
ARX_API int arx_abi_version(void);

/* nn.Module.load_state_dict for the skeleton path (ar.py:17-19). */
ARX_API int arx_load_weights(arx_handle *h, const arx_weights *w, void *stream);

/* TemporalCrossTransformer.__init__ tuple table (model.py:51-55): writes the
 * C(T,c) x c lexicographic combinations as int32, built on device. */
ARX_API int arx_tuple_count(const arx_handle *h, int32_t ti);
ARX_API int arx_tuple_table(arx_handle *h, int32_t ti, int32_t *out_dev, void *stream);

/* MLP.forward (model.py:164-180) over n_frames rows of 3J -> F. */
ARX_API int arx_embed(arx_handle *h, const float *frames_dev, int64_t n_frames, float *feats_dev, void *stream);

/* Support side of TemporalCrossTransformer.forward (model.py:65,69,71,75,77,81)
 * done ONCE per support-set change instead of per call (ar.py:56-67).
 *   poses_dev (W,T,3J) -> MLP -> features; or feats_dev (W,T,F) given directly
 *   (the ss_features argument of TRXOS.forward, model.py:291,307).
 * Class order is the caller's (ss_labels[0] already applied). */
ARX_API int arx_set_support_poses(arx_handle *h, const float *poses_dev, int32_t way, void *stream);
ARX_API int arx_set_support_features(arx_handle *h, const float *feats_dev, int32_t way, void *stream);
/* out (W,T,F): the 'support_features' entry of the return dict (model.py:327-328). */
ARX_API int arx_get_support_features(arx_handle *h, float *feats_dev, void *stream);
ARX_API int arx_support_way(const arx_handle *h);

/* Support-set tuple embeddings (LayerNorm-ed K and V tuple tensors of every transformer, fp32) as one flat device
 * blob, for the NCCL broadcast across ranks (SURVEY.md 8e).  export/import must use handles with identical
 * config+weights.  import rebuilds the tensor-core operand images on the handle's side stream; a handle that
 * imported its support set cannot return 'support_features' (arx_get_support_features -> ARX_ERR_STATE). */
ARX_API int64_t arx_support_blob_bytes(const arx_handle *h, int32_t way);
ARX_API int arx_export_support(arx_handle *h, void *blob_dev, void *stream);
ARX_API int arx_import_support(arx_handle *h, const void *blob_dev, int32_t way, void *stream);

/* TRXOS.forward (model.py:291-328) for B query windows against the current
 * support set, transformers[0] + discriminator:
 *   query_dev (B,T,3J) -> logits_dev (B,W) [= -distance], is_true_dev (B) in (0,1)
 *   [may be NULL / ignored without discriminator], chosen_dev (B) int32 argmax
 *   (first maximum on ties, model.py:323) [may be NULL].
 * The discriminator is sized for pair tuples (model.py:282-285): is_true needs temp_set[0] = 2.  On the tiled tcgen05
 * kernels the open-set head covers every seq_len the handle accepts (2..64); the head's T columns are accumulator lanes
 * of the attention kernel's head mode. */
ARX_API int arx_score(arx_handle *h, const float *query_dev, int64_t n_windows,
              float *logits_dev, float *is_true_dev, int32_t *chosen_dev, void *stream);

/* Frame-stream form of arx_score: frames_dev (n_frames, 3J) is a sequence of camera frames and EVERY sliding window of
 * seq_len consecutive frames is scored (window w = frames w .. w+T-1, what n_frames successive ActionRecognizer.inference
 * calls see, ar.py:42-50): logits_dev (n_frames-T+1, W), is_true_dev (n_frames-T+1).  On every route each frame is embedded
 * and projected ONCE (the projection is position-independent; the positional table is added per window position when the
 * windows are formed on the device), and a caller uploads 3J floats per window instead of T*3J. */
ARX_API int arx_score_frames(arx_handle *h, const float *frames_dev, int64_t n_frames,
                     float *logits_dev, float *is_true_dev, int32_t *chosen_dev, void *stream);

/* TRXOS.forward in the training / evaluation call shape (modules/ar/utils/train.py:110-120,
 * modules/ar/utils/test/compute_fsos.py:89-98): every batch row is its own EPISODE -- query i is scored against
 * ITS OWN `way` support classes (model.py:59-148 never mixes batch rows).  On both tensor-core routes (the T=16 pair
 * pipeline and the tiled kernels: T=32, other T, triples, debug bit 4096, force_path = 2 past the overflow bound)
 * episodes go through the batched kernels a pass at a time: the support operands of the pass's episodes*way classes
 * form one pool, and window i attends classes [i*way, (i+1)*way) of it.  A pass holds 256 episodes on the pair
 * pipeline; on the tiled kernels as many as keep the pool within 1 GiB (at least one, at most 256).  The fp32 route
 * (force_path = 1, LayerNorm affines past the accuracy bound, D != 128) scores one episode at a time.
 * The pool holds the support operands of transformers[0] only, the transformer that scores episodes (model.py:320).
 *   support_dev (n_episodes, way, T, 3J) poses, or (n_episodes, way, T, F) frame features when is_features != 0
 *   (the ss_features argument); query_dev (n_episodes, T, 3J); outputs as arx_score.
 * REPLACES the handle's current support set (by the pool of the last pass, transformers[0] only): call
 * arx_set_support_* again before the next arx_score; until then arx_score_features(ti >= 1) and arx_export_support
 * return ARX_ERR_STATE. */
ARX_API int arx_score_episodes(arx_handle *h, const float *support_dev, int32_t is_features, int32_t way, const float *query_dev,
                       int64_t n_episodes, float *logits_dev, float *is_true_dev, int32_t *chosen_dev, void *stream);

/* TemporalCrossTransformer(args, temp_set[ti]).forward(...)['logits'] (model.py:59-148)
 * from precomputed frame features qfeats_dev (B,T,F); used for the cardinality-3
 * transformer that TRXOS.forward never calls (model.py:320). */
ARX_API int arx_score_features(arx_handle *h, int32_t ti, const float *qfeats_dev, int64_t n_windows,
                       float *logits_dev, void *stream);

/* Debug outputs (model.py:110-111,126,146): softmax scores P (B,W,N,N) and
 * prototypes (B,W,N,D) of transformers[0] for a SMALL batch; either may be NULL. */
ARX_API int arx_debug_attention(arx_handle *h, const float *query_dev, int64_t n_windows,
                        float *probs_dev, float *prototypes_dev, void *stream);

/* End-to-end convenience: HOST buffers in, HOST buffers out; chunks are staged
 * through pinned memory with copies overlapped with compute.  Synchronises. */
ARX_API int arx_score_host(arx_handle *h, const float *query_host, int64_t n_windows,
                   float *logits_host, float *is_true_host, int32_t *chosen_host);

/* fp16 HOST rows (IEEE binary16, same (B,T,3J) layout): half the PCIe bytes of the fp32 entry points.  The first GEMM's
 * operand image is fp16 in any case, so for inputs representable in fp16 the results are bit-identical to the fp32 entry
 * points.  Available where the linear layers run on tensor cores (all BASELINE configs); ARX_ERR_INVALID otherwise. */
ARX_API int arx_score_host_f16(arx_handle *h, const uint16_t *query_host_f16, int64_t n_windows,
                       float *logits_host, float *is_true_host, int32_t *chosen_host);

/* Streaming variant of arx_score_host: returns as soon as the copies and kernels are enqueued on the handle's
 * internal copy/compute streams; up to ARX_HOST_DEPTH requests may be in flight, so the H2D copy of request i+1
 * overlaps the scoring of request i.  arx_score_host_wait blocks until request `ticket` (returned by submit)
 * has landed in the host output buffers.  Host buffers must stay valid (and should be pinned) until then. */
#define ARX_HOST_DEPTH 2
ARX_API int arx_score_host_submit(arx_handle *h, const float *query_host, int64_t n_windows,
                          float *logits_host, float *is_true_host, int32_t *chosen_host, int64_t *ticket);
ARX_API int arx_score_host_submit_f16(arx_handle *h, const uint16_t *query_host_f16, int64_t n_windows,
                              float *logits_host, float *is_true_host, int32_t *chosen_host, int64_t *ticket);
ARX_API int arx_score_host_wait(arx_handle *h, int64_t ticket);

/* Resident streaming scorer: ActionRecognizer.inference (modules/ar/ar.py:30-84, called once per camera frame from
 * main.py:111).  The handle keeps the sliding window on the device: arx_stream_push takes ONE new frame (3J floats, HOST),
 * computes its MLP features and its position-independent K/V projections once, stores them in a ring of T frames, forms the
 * window's per-frame projections as ring + positional table, scores the window against the current support set
 * (transformers[0] + discriminator) and returns result_host[0..way) = softmax(logits) (ar.py:77), result_host[way] = is_true
 * (ar.py:78).  *valid = 0 until seq_len frames have been pushed since the last reset (ar.py:43-44).  One H2D (the frame),
 * one CUDA-graph launch and one D2H per call; synchronises the handle's internal stream.  Pair tuples only (with or
 * without the discriminator, any seq_len up to 64), on the tiled tcgen05 kernels.
 * arx_stream_reset forgets the window (previous_frames = []). */
ARX_API int arx_stream_push(arx_handle *h, const float *frame_host, float *result_host, int32_t *valid);
ARX_API int arx_stream_reset(arx_handle *h);

/* MetrABS-style heatmap decode (modules/hpe/hpe.py:108-169 + main.py:103-105):
 *   logits_dev (B,8,8,32+8*32) fp32 -> poses_dev (B,3*n_out) fp32 root-centred,
 *   valid_dev (B) uint8 (0 where the reference returns None, hpe.py:152-153).
 *   expand_dev (32,n_out) fp32 = column-selected assets/32_to_122.npy,
 *   new_K (3x3 row-major) and homo_inv (3x3) as produced by misc.py:homography. */
ARX_API int arx_decode_heatmaps(arx_handle *h, const float *logits_dev, int64_t n_frames,
                        const float *expand_dev, int32_t n_out,
                        const float *new_K_host9, const float *homo_inv_host9,
                        float *poses_dev, uint8_t *valid_dev, void *stream);

/* Same decode with a camera PER FRAME: new_K_dev / homo_inv_dev are (n_frames,3,3) fp32 device arrays.  This is the
 * test-time-augmentation call shape (hpe.py:88-93, misc.py:310-327): every augmented crop of a camera frame has its own
 * scaled intrinsics and its own rotation/flip to undo. */
ARX_API int arx_decode_heatmaps_cams(arx_handle *h, const float *logits_dev, int64_t n_frames, const float *expand_dev, int32_t n_out,
                             const float *new_K_dev, const float *homo_inv_dev, float *poses_dev, uint8_t *valid_dev, void *stream);

/* MetrABS heads that produce those logits: Linear(1280 -> 288) applied to every cell of the (8,8,1280) backbone feature map
 * (modules/hpe/setup/4_create_heads_onnx.py:7-16; the reference runs it as a TensorRT fp16 engine, hpe.py:106).  tcgen05 GEMM,
 * fp16 operands / fp32 accumulate.  weight (288,1280) and bias (288) fp32, host or device; feats_dev (n_frames,8,8,1280) fp32 ->
 * logits_dev (n_frames,8,8,288) fp32, the input of arx_decode_heatmaps. */
ARX_API int arx_heads_load(arx_handle *h, const float *weight, const float *bias, int32_t on_device, void *stream);
ARX_API int arx_heads_forward(arx_handle *h, const float *feats_dev, int64_t n_frames, float *logits_dev, void *stream);

/* Stage timers for roofline reporting: CUDA events recorded on the caller's stream around the
 * stages of arx_score (0 frame embedding MLP, 1 per-frame K/V projection, 2 tuple build + LayerNorm,
 * 3 cross-attention + distances, 4 open-set head).  arx_profile_read synchronises the events,
 * adds the elapsed milliseconds per stage into ms[ARX_N_STAGES] and returns the number of
 * arx_score chunks covered in *chunks; reset != 0 clears the accumulators. */
#define ARX_N_STAGES 5
ARX_API int arx_profile_enable(arx_handle *h, int32_t on);
ARX_API int arx_profile_read(arx_handle *h, double *ms, int64_t *chunks, int32_t reset);

/* Debug knobs for kernel bring-up and tests.
 *  key 0: kernel-variant bit mask -- 4 fp32 CUDA-core linear layers in front of the tiled tcgen05 attention (T=16 pair
 *         tuples leave their dedicated pipeline), 64 timing only: skip the tuple build, 1024 one-tile-per-CTA GEMMs for
 *         the frame MLP, 2048 head projection on the caller's stream, 4096 T=16 pair tuples on the tiled any-N kernels.
 *         8192 frame MLP as three launches (pose image, fc1, fc2) instead of the fused kernel, 16384 no L2 prefetch ahead of the
 *         head kernel's operand ring, 32768 the persistent front-end kernels take every SM even while a support chain is in flight.
 *         Bits 4 and 4096 choose the kernels of the T=16 pairs when the support set is built (they decide which support
 *         operands are built): set them BEFORE the support set.  Scoring keeps the kernels the current support operands
 *         were built for; only the front end of the tiled kernels follows bit 4 at once.
 *  key 1: arm a timeline trace of CTA 0 of the attention kernel (value 1) of the fused frame-MLP kernel (value 2) or of the head kernel (value 3); 0 frees it.
 *  key 2: programmatic dependent launch for the score kernel chain.
 *  key 3: softmax-group scheduling of the attention kernel: < 0 the groups take turns on the MUFU phase
 *         (default), >= 0 free-running with group 1 started this many clocks late.
 *  key 4: attention kernel: every value-th register pair of a score tile takes the FMA-pipe exp2 polynomial
 *         instead of MUFU.EX2 (0 = none (default), 2, 3, 4; measured: no gain on B200, the packed FMA ops cost
 *         as much pipe time as the MUFU they replace).
 *  key 5: CUDA-graph replay of the arx_score kernel chain when its arguments recur (default on; the environment
 *         variable ARX_GRAPHS=0 disables it too).
 *  key 6: tiled attention kernels, normaliser pass: half of the exponentials on the FMA pipe (default 1; 0 = all on the MUFU).
 *  key 7: tiled attention kernels, normaliser pass: softmax groups free-running (default 1) instead of taking turns on the MUFU. */
ARX_API int arx_debug_set(arx_handle *h, int32_t key, int32_t value);
/* key 1 (value != 0) arms a timeline trace of CTA 0 of the attention kernel; this reads it back:
 * host_out[3 roles][64 tiles][8 stamps] of SM clock values (bring-up tool). */
ARX_API int arx_debug_read_trace(arx_handle *h, long long *host_out);

/* Introspection for tests/bench: kernel launches issued by this handle so far,
 * and which attention path the last arx_score used: 1 = fp32 CUDA-core kernels, 2 = tcgen05 pipeline of the
 * metric shape (T=16 pair tuples), 3 = tiled any-N tcgen05 kernels (T=32, triples, other T, ROWMAX variant). */
ARX_API int64_t arx_launch_count(const arx_handle *h);
ARX_API int arx_last_path(const arx_handle *h);

#ifdef __cplusplus
}
#endif
#endif /* ARX_H */

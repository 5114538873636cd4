/*
 * gitb200 -- C ABI of the B200-native GIT captioning hot path.
 *
 * The reference (farazali7/real-time-video-captioning) has no FFI: its boundary for this path is the
 * Python class surface of /root/reference/src/models/model.py.  Each entry point below names the
 * reference interface whose arithmetic it replaces; the Python mirror in
 * real-time-video-captioning_b200/model.py binds them with ctypes (see INTEGRATION.md).
 *
 * Conventions: plain pointers and sizes only; every call returns 0 on success or a negative
 * gitb200_status, never throws; `gitb200_last_error` gives the message.  Pointers named *_dev are
 * device pointers on the context's GPU, *_host are host pointers.  All work is enqueued on `stream`
 * (a cudaStream_t passed as void*; NULL = legacy default stream) and is asynchronous unless stated.
 * One context per GPU; a context is not thread-safe.  There is no CPU fallback: without a usable
 * sm_100 device every compute call fails with GITB200_ERR_CUDA.
 */
#ifndef GITB200_H_
#define GITB200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct gitb200_ctx gitb200_ctx;

typedef enum {
  GITB200_OK = 0,
  GITB200_ERR_INVALID = -1,  /* bad argument / unsupported shape */
  GITB200_ERR_CUDA = -2,     /* CUDA runtime or driver error (message has the detail) */
  GITB200_ERR_STATE = -3,    /* call order violated (weights not finalised, no visual features, ...) */
  GITB200_ERR_MISSING = -4   /* a required weight was never loaded */
} gitb200_status;

/* Model hyper-parameters: get_git_model(tokenizer, param), model.py:681-718. */
typedef struct {
  int vit_width, vit_layers, vit_heads, patch, resolution; /* CLIPViT_B_16: 768,12,12,16,224; CLIPViT_L_14: 1024,24,16,14,224 */
  int hidden, dec_layers, dec_heads, ffn;                   /* 768, 6, 12, 3072            (model.py:690-693) */
  int vocab, max_positions;                                 /* 30522, 1024                 (model.py:689,694) */
  int num_image_with_embedding;                             /* param['num_image_with_embedding'] (model.py:368) */
  float vit_ln_eps, proj_ln_eps, embed_ln_eps, bert_ln_eps; /* 1e-5, 1e-5, 1e-8, 1e-12 */
  int sos, eos;                                             /* tokenizer.cls_token_id / sep_token_id (model.py:363-364) */
} gitb200_config;

/* GeneratorWithBeamSearchV2(...) + search(...) arguments, model.py:702-708 and :479-480. */
typedef struct {
  int beam_size;          /* 4  (model.py:706) */
  int max_steps;          /* 15 (model.py:704): captions hold at most max_steps tokens incl. SOS */
  int per_node_beam_size; /* 2  (upstream default) */
  int num_keep_best;      /* 1  (model.py:479) */
  float length_penalty;   /* 0.6 (model.py:707) */
  int reorder_cache;      /* 0 = reference behaviour: decoder cache rows are NOT re-indexed after a beam
                             re-order (model.py:623-634 is commented out); 1 = re-index by parent beam */
} gitb200_search_params;

/* ---- lifetime ------------------------------------------------------------------------------- */
int gitb200_create(const gitb200_config* cfg, int device, gitb200_ctx** out);
void gitb200_destroy(gitb200_ctx* ctx);
/* Message of the last failure on this context (ctx may be NULL for create failures). */
const char* gitb200_last_error(const gitb200_ctx* ctx);
/* Library build info, e.g. "gitb200 0.1 sm_100a". */
const char* gitb200_version(void);

/* ---- weights: load_state_dict(self.model, ckpt['model']), model.py:736-738 -------------------
 * `name` is the upstream state-dict key (image_encoder.conv1.weight, textual.transformer.encoder.
 * layer.0.attention.self.query.weight, img_temperal_embedding.0, ...); `data` is fp32, host or device.
 * Unknown names are ignored (upstream's loader is tolerant); finalize repacks everything once:
 * bf16 K-major matrices, fused decoder QKV, vocabulary padded to a multiple of 256. */
int gitb200_load_weight(gitb200_ctx* ctx, const char* name, const float* data, int ndim, const int64_t* shape);
int gitb200_finalize_weights(gitb200_ctx* ctx);

/* Pre-size every workspace and the KV cache (optional; calls grow them on demand). */
int gitb200_reserve(gitb200_ctx* ctx, int max_clips, int max_frames, int max_rows_per_clip, int max_text_len);

/* Geometry helpers. */
int gitb200_tokens_per_frame(const gitb200_ctx* ctx); /* T = (resolution/patch)^2 + 1 */
int gitb200_logits_ld(const gitb200_ctx* ctx);        /* leading dimension of every logits buffer (vocab rounded up to 256) */

/* ---- image encoder: self.image_encoder(frames) + temporal embeddings + concat, model.py:378-382 -
 * frames_dev: fp32 [n_clips, n_frames, 3, R, R].  Frames beyond num_image_with_embedding are dropped
 * (zip truncation, model.py:380).  Keeps the bf16 visual features inside the context for the calls
 * below and, if visual_features_dev != NULL, also writes them as fp32 [n_clips, F'*T, Dv]. */
int gitb200_encode(gitb200_ctx* ctx, const float* frames_dev, int n_clips, int n_frames, float* visual_features_dev,
                   void* stream);
/* Single-image branch of the same forward (batch['image'] is a tensor, not a list: model.py:387-388):
 * images_dev fp32 [n_images, 3, R, R] -> visual features [n_images, T, Dv], NO temporal embedding. */
int gitb200_encode_images(gitb200_ctx* ctx, const float* images_dev, int n_images, float* visual_features_dev, void* stream);
/* Forward hooks on image_encoder.transformer.resblocks[i] (registered at model.py:847, read at :912-913): while taps are
 * set, every encode (gitb200_encode / _forward_logits / _caption) also writes the OUTPUT of each listed resblock as fp32
 * [n_layers, n_clips, F', T, Dv] to out_dev (the reference's hook sees the same values as [T, F', Dv] per clip).
 * layers_host: resblock indices on the host; n_layers = 0 removes the taps.  out_dev must stay valid while taps are set. */
int gitb200_set_vit_taps(gitb200_ctx* ctx, const int32_t* layers_host, int n_layers, float* out_dev);
/* Use caller-provided visual features (infer(batch, visual_features, ...), model.py:426). fp32 [n_clips, nv, Dv]. */
int gitb200_set_visual_features(gitb200_ctx* ctx, const float* visual_features_dev, int n_clips, int nv, void* stream);

/* ---- caption search: infer + GeneratorWithBeamSearchV2.search, model.py:426-462, :479-678 -----
 * Runs on the context's current visual features.  tokens_dev: int32 [n_clips, num_keep_best, max_steps]
 * (eos padded, SOS first); logprobs_dev: fp32 [n_clips, num_keep_best]; logits_dev (optional): fp32
 * [max_steps-1, n_clips*beam_size, logits_ld] = the per-step scores the reference copies to the host at
 * model.py:521 (kept on the device here). */
int gitb200_decode(gitb200_ctx* ctx, const gitb200_search_params* sp, int32_t* tokens_dev, float* logprobs_dev,
                   float* logits_dev, void* stream);
/* encode + decode.  For small batches (<= 8 clips) on a non-default stream, the second call with identical buffers,
 * shapes and search parameters is captured into a CUDA graph and later identical calls replay it (latency mode). */
int gitb200_caption(gitb200_ctx* ctx, const float* frames_dev, int n_clips, int n_frames,
                    const gitb200_search_params* sp, int32_t* tokens_dev, float* logprobs_dev, float* logits_dev,
                    void* stream);
/* The reference leaves its step loop as soon as every clip's search is finished (`if all(done): break`, model.py:640).
 * The device search counts finished clips; every `every_steps` decode steps (default 4; 0 = never, the call then stays
 * fully asynchronous) the host reads that count (4 bytes + one stream synchronisation) and stops enqueueing steps when
 * it equals n_clips.  Finished clips never change again, so tokens / scores are identical either way; only calls that
 * are being captured into a CUDA graph always run all steps.  gitb200_last_decode_steps: steps the last decode enqueued
 * (= len(saved_logits) of the reference; rows of logits_dev beyond it are not written). */
int gitb200_set_early_exit(gitb200_ctx* ctx, int every_steps);
int gitb200_last_decode_steps(const gitb200_ctx* ctx);
/* Latency mode of the search loop (default on): the search of ONE clip (gitb200_caption / _decode / _stream_caption with one
 * clip, beam_size <= 4, no saved logits) runs as one persistent cooperative kernel -- every decode step's embedding, decoder
 * layers, vocabulary head and search step (model.py:518-640) are phases of a grid that stays resident, separated by
 * grid-wide barriers instead of ~42 kernel launches per step.  Bit-identical to the launch sequence (0 selects it). */
int gitb200_set_persistent_decode(gitb200_ctx* ctx, int enable);
/* Profiling aid: while enabled, CTA 0 of the persistent decode kernel adds the SM cycles it spends in each phase to 32
 * counters (0-6: QKV, attention, out-proj, fc1, fc2, vocabulary head, search -- its own work; 16-22: the wait in the grid
 * barrier that ends the phase; 15: launches).  Copies the counters to out32 (may be NULL), then enables / disables (both
 * reset them).  Synchronises the device. */
int gitb200_debug_persistent_decode_trace(gitb200_ctx* ctx, unsigned long long* out32, int enable);
/* gitb200_caption calls of up to `max_clips` clips are captured into CUDA graphs (default 8: the launch-bound latency
 * mode).  Larger values also graph throughput-sized batches once gitb200_reserve has pinned the workspaces. */
int gitb200_set_graph_max_clips(gitb200_ctx* ctx, int max_clips);
/* Batches above that size are graphed in pieces that do not depend on the caller's output pointers (default on): encode +
 * visual pass per frame buffer (host paths: per staged chunk), the decode loop per segment of `every_steps` steps with the
 * finished-clip poll between segments.  The ~1200 launches of a 512-clip step reach the GPU as a handful of graph launches.
 * Calls on the legacy default stream run on the context's own stream, forked from / joined into the caller's.  0 = eager. */
int gitb200_set_graph_segments(gitb200_ctx* ctx, int enable);

/* Opt-in (default off): ViT ln_1 / ln_2 folded into the following QKV / fc1 GEMM: the GEMM reads the raw residual stream, its
 * weights carry gamma, its bias carries W*beta, and its epilogue applies rstd*(acc - mean*colsum) from row statistics
 * emitted by the previous residual GEMM's epilogue.  0 restores the separate LayerNorm kernels (same result within the
 * bf16 tolerance; the folded form skips one bf16 rounding of the normalised activations).  Measured on B200: the 24
 * LayerNorm launches disappear (4.5 % of the step) but the heavier GEMM epilogues give most of it back (+1 % net), and
 * the atomically accumulated statistics make results run-to-run non-bit-exact, hence off by default. */
int gitb200_set_fold_layernorm(gitb200_ctx* ctx, int enable);
/* Opt-in (default off: measured 1 % slower than the separate LayerNorm kernels at the bench geometry, profiles/r02_layernorm_fusion.md):
 * for sweeps of >= 1024 rows the LayerNorm that FOLLOWS a residual GEMM -- ViT ln_2 after the out-projection, the
 * next block's ln_1 after fc2, the decoder's visual_projection LayerNorm and its two post-LNs per layer over the visual rows --
 * is produced by that GEMM as a second output: the CTA pair owns whole 256-row blocks, accumulates the rows' statistics over its
 * N / 256 tiles in a fixed order and writes the normalised rows itself.  Bit-reproducible. */
int gitb200_set_fuse_layernorm(gitb200_ctx* ctx, int enable);

/* Large batches walk the ViT and the decoder's pass over the visual tokens in sub-batches of about `rows` token rows
 * (default 151296 = 128 six-frame ViT-B/16 clips; 0 = the whole batch in one sweep), so that the row-sized scratch
 * (ViT activations, decoder visual hidden states, MLP buffers) is held for one sub-batch only: 4.4 instead of 17.6 GB at
 * 512 clips.  Clips are independent on this part of the path (the reference encodes them one by one, model.py:752-759),
 * every sub-batch writes its own slice of the visual features / visual K/V cache, and results are bit-identical whenever
 * every sub-batch takes the same GEMM kernel as the whole batch (>= 1024 rows; a smaller ragged tail differs by bf16
 * rounding only).  Throughput-neutral from 128 clips per sub-batch up (measured A/B on one B200); call it before
 * gitb200_reserve. */
int gitb200_set_sweep_rows(gitb200_ctx* ctx, int rows);

/* Opt-in large-batch pipelining of gitb200_caption / gitb200_caption_host: clips per chunk (0 = off, the default;
 * -1 = automatic: a quarter of the batch clamped to [32, 128]).  Chunks alternate between two internal streams / workspace sets so that one
 * chunk's decode steps overlap the next chunk's ViT.  When a call is pipelined, the context does not keep the visual
 * features of the whole batch resident afterwards.  Measured SLOWER than the single-stream schedule on B200 (kernel-
 * granularity interleaving stretches the latency-bound decode chain behind 100-250 us GEMM kernels): kept for experiments. */
int gitb200_set_pipeline(gitb200_ctx* ctx, int chunk_clips);

/* Same with HOST buffers (frames_host should be pinned for full PCIe speed): chunks of `chunk_clips`
 * clips are copied host->device on a side stream while the previous chunk computes; tokens and
 * logprobs are copied back; returns after everything has completed (synchronous). */
int gitb200_caption_host(gitb200_ctx* ctx, const float* frames_host, int n_clips, int n_frames, int chunk_clips,
                         const gitb200_search_params* sp, int32_t* tokens_host, float* logprobs_host);
/* Host frames in, DEVICE results out -- what GenerativeImageTextModel.forward returns for a batch handed over on the host
 * (model.py:768-780: predictions, logprobs, the per-step logits of logits_dict, visual_features).  Same chunked,
 * copy-overlapped encode as gitb200_caption_host; logits_dev (fp32 [max_steps-1, n_clips*beam, logits_ld]) and
 * visual_features_dev (fp32 [n_clips, F*T, vit_width]) are optional.  Asynchronous: the work runs on the context's own
 * streams and `stream` is made to wait for the results; frames_host must stay valid until then. */
int gitb200_caption_from_host(gitb200_ctx* ctx, const float* frames_host, int n_clips, int n_frames, int chunk_clips,
                              const gitb200_search_params* sp, int32_t* tokens_dev, float* logprobs_dev, float* logits_dev,
                              float* visual_features_dev, void* stream);

/* ---- teacher-forced logits: forward_one_custom, model.py:371-424 ------------------------------
 * tokens_dev: int32 [n_clips, L].  If frames_dev == NULL the current visual features are used.
 * logits_dev: fp32 [n_clips*L, logits_ld].  hidden_states_dev (optional): fp32
 * [n_clips, dec_layers+1, nv+L, hidden] (the 7 stacked hidden states of model.py:419-423).
 * visual_features_dev (optional): fp32 [n_clips, nv, Dv]. */
int gitb200_forward_logits(gitb200_ctx* ctx, const float* frames_dev, int n_clips, int n_frames,
                           const int32_t* tokens_dev, int L, float* logits_dev, float* hidden_states_dev,
                           float* visual_features_dev, void* stream);

/* ---- step-wise decoding: CaptioningModel.decoding_step bound at model.py:442-445 --------------
 * For callers that drive their own search loop through the generic `step(input_ids)` callable.
 * begin: runs the decoder over the visual tokens (the first-call branch of decoding_step) for
 * n_clips * rows_per_clip rows; step: feeds one token per row at text position `pos` and writes
 * fp32 logits [rows, logits_ld]; reorder: optional cache re-index by beam_idx (int32 [rows]). */
int gitb200_decode_begin(gitb200_ctx* ctx, int rows_per_clip, void* stream);
int gitb200_decode_step(gitb200_ctx* ctx, const int32_t* tokens_dev, int pos, float* logits_dev, void* stream);
int gitb200_decode_reorder(gitb200_ctx* ctx, const int32_t* beam_idx_dev, int pos, void* stream);

/* ---- streaming window: the webcam loop of src/real_time_inference.py:38-61 --------------------------------------
 * push: encode ONE preprocessed frame (fp32 [3, R, R]) with the ViT as it arrives and keep its features (after ln_post,
 * before the temporal embedding) in a ring of num_image_with_embedding frames; caption: add the temporal embeddings in
 * arrival order (oldest frame = position 0), run the decoder + search on the frames currently in the window
 * (tokens_dev int32 [1, num_keep_best, max_steps]).  The caption after 6 pushes equals gitb200_caption on those 6
 * frames, but only one frame's ViT (35 of 211 GFLOP) stands between the last frame and its caption.  reset empties the
 * window (the reference clears its frame list after every caption: non-overlapping windows; not clearing it gives a
 * sliding window with per-frame feature reuse). */
int gitb200_stream_reset(gitb200_ctx* ctx);
int gitb200_stream_push(gitb200_ctx* ctx, const float* frame_dev, void* stream);
/* gitb200_stream_push for a raw webcam frame: frame_dev uint8 [height, width, 3] BGR HWC on the device (what
 * cv2.VideoCapture.read() returns, real_time_inference.py:49-57); image_transform() runs fused into the patch-embed loader. */
int gitb200_stream_push_u8(gitb200_ctx* ctx, const uint8_t* frame_dev, int height, int width, void* stream);
int gitb200_stream_frames(const gitb200_ctx* ctx);
int gitb200_stream_caption(gitb200_ctx* ctx, const gitb200_search_params* sp, int32_t* tokens_dev, float* logprobs_dev,
                           void* stream);

/* ---- multi-stream pool: many cameras on one context ------------------------------------------------------------
 * A pool of n_streams windows next to the single window above (which it does not touch), each window the same ring of
 * num_image_with_embedding per-frame ViT features: bf16 [n_streams][cap][T][Dv] (GIT-base, 6 frames: 1.82 MB per stream).
 * Stream ids are 0 .. n_streams-1.  configure empties every window; a different count also reallocates the pool.
 * Every call below checks its id list on the host before it enqueues anything and fails, naming the offending id, on an
 * unknown id or an id given twice (GITB200_ERR_INVALID), k < 1 (GITB200_ERR_INVALID), or a call before configure
 * (GITB200_ERR_STATE); a rejected call changes no window.  Which frames each window holds is host-side bookkeeping. */
int gitb200_streams_configure(gitb200_ctx* ctx, int n_streams);
/* ONE frame for each of k distinct streams, encoded as one ViT batch (the launch sequence of gitb200_encode_images on the same
 * k frames, in sub-batches of gitb200_set_sweep_rows): ln_post writes each frame's T rows straight into its stream's ring
 * slot.  frames_dev fp32 [k, 3, R, R] (preprocessed) or, for _u8, uint8 [k, height, width, 3] BGR with image_transform()
 * fused into the patch-embed loader (as gitb200_stream_push_u8); ids_host int32 [k]: frame j goes to stream ids_host[j].
 * Calls of up to gitb200_set_graph_max_clips frames (larger ones too while graph segments are on) on a non-default stream
 * are captured into a CUDA graph keyed by shape only (k, frame buffer, height / width): the same shape replays whichever
 * streams it pushes to, because the per-call slot table is copied (cudaMemcpyAsync, from host memory the call owns) into a
 * context-owned device buffer before the graph launch. */
int gitb200_streams_push(gitb200_ctx* ctx, const int32_t* ids_host, int k, const float* frames_dev, void* stream);
int gitb200_streams_push_u8(gitb200_ctx* ctx, const int32_t* ids_host, int k, const uint8_t* frames_dev, int height, int width,
                            void* stream);
/* Decoder + search over the windows of k distinct streams that hold the SAME number of frames n (temporal embeddings by
 * arrival order, oldest = position 0, exactly as gitb200_stream_caption): tokens_dev int32 [k, num_keep_best, max_steps],
 * logprobs_dev fp32 [k, num_keep_best], row j = stream ids_host[j].  Fails with GITB200_ERR_STATE on an empty stream and
 * GITB200_ERR_INVALID when the streams hold different frame counts (caption those in separate calls).  Afterwards the
 * context's current visual features are these k windows [k, n*T, Dv], as after gitb200_stream_caption.  Up to
 * gitb200_set_graph_max_clips windows the whole call is one CUDA graph (one window with beam <= 4 takes the persistent
 * decode kernel); larger calls graph the window assembly + visual pass and the decode segments.  The caption of a stream
 * does not depend on which other streams share the call or in which order. */
int gitb200_streams_caption(gitb200_ctx* ctx, const int32_t* ids_host, int k, const gitb200_search_params* sp,
                            int32_t* tokens_dev, float* logprobs_dev, void* stream);
/* Empties the windows of k distinct streams (the reference's frames.clear() after a caption, real_time_inference.py:61). */
int gitb200_streams_reset(gitb200_ctx* ctx, const int32_t* ids_host, int k);
/* Frames held by one stream's window (0 .. num_image_with_embedding); GITB200_ERR_INVALID for an unknown id. */
int gitb200_streams_frames(const gitb200_ctx* ctx, int stream_id);
/* One stream's window as the decoder sees it: temporal embeddings added, bf16 values written as fp32 [n*T, Dv] (the
 * visual features gitb200_streams_caption decodes for that stream).  Does not change the context's current features. */
int gitb200_streams_window(gitb200_ctx* ctx, int stream_id, float* out_dev, void* stream);

/* ---- frame preprocessing: image_transform(), src/utils/dataloader.py:18-32 (= real_time_inference.py:16-28) ----
 * frames_dev: uint8 [n_frames, height, width, 3] in OpenCV's BGR HWC layout; out_dev: fp32 [n_frames, 3, size, size]
 * (RGB, CLIP-normalised): bicubic resize of the smaller edge to `size` (no antialias, like the pinned torchvision
 * 0.16 on tensors), centre crop, channel flip, normalise -- ready for gitb200_encode / gitb200_caption. */
int gitb200_preprocess(const uint8_t* frames_dev, int n_frames, int height, int width, int size, float* out_dev,
                       void* stream);

/* Host path for RAW video frames (SURVEY 8f rank 1; the caller's side is real_time_inference.py:49-57 and the dataset's
 * cv2 frame reads, dataloader.py:61-75): frames_host uint8 [n_clips, n_frames, height, width, 3] BGR HWC (pinned
 * recommended) -> host tokens / log-probs exactly as gitb200_caption_host.  Frames cross PCIe as bytes in chunks of
 * `chunk_clips` clips (copy of chunk i+1 overlaps chunk i's work), image_transform() runs on the device fused into the
 * patch-embed loader (gitb200_preprocess's arithmetic, written as bf16 straight into the patch matrix of the conv1 GEMM:
 * no fp32 frames exist on the device), then one batched decode.  Same result, bit for bit, as gitb200_preprocess +
 * gitb200_caption on the same frames.  Synchronous. */
int gitb200_caption_host_u8(gitb200_ctx* ctx, const uint8_t* frames_host, int n_clips, int n_frames, int height, int width,
                            int chunk_clips, const gitb200_search_params* sp, int32_t* tokens_host, float* logprobs_host);

/* ---- student decoder (SURVEY 8f rank 3): the decoder half of StudentCandidateV1, model.py:50-187 ---------------------
 * nn.Embedding + PositionalEncoding + post-LN nn.TransformerDecoder (causal / padding-masked self-attention, cross-attention
 * to the F frame tokens of `memory`, ReLU feed-forward) + the vocabulary nn.Linear.  The TinyViT image encoder that
 * produces `memory` (timm, model.py:35-48) is NOT part of this library: memory fp32 [B, F, d_model] is an input.
 * Weights use the reference's state-dict names (decoder.layers.N.{self_attn,multihead_attn}.{in_proj_weight,in_proj_bias,
 * out_proj.weight,out_proj.bias}, .linear1/.linear2/.norm1-3.{weight,bias}, embed.weight, linear.{weight,bias}) plus
 * "pos_enc.pe" = the [max_len, d_model] sinusoidal table of PositionalEncoding (model.py:324-335). */
typedef struct gitb200_student gitb200_student;
typedef struct {
  int d_model, n_head, d_ffn, n_layers; /* config.py:80-84: 576, 8, 1024, 2 */
  int vocab, max_len;                   /* tokenizer vocabulary (30522), PositionalEncoding max_len (500) */
  int cls, sep, pad;                    /* 101, 102 (model.py:82-83), create_padding_mask's padding_token 0 (masking.py:4) */
  float ln_eps;                         /* nn.LayerNorm default 1e-5 */
} gitb200_student_config;
int gitb200_student_create(const gitb200_student_config* cfg, int device, gitb200_student** out);
void gitb200_student_destroy(gitb200_student* s);
const char* gitb200_student_last_error(const gitb200_student* s);
int gitb200_student_load_weight(gitb200_student* s, const char* name, const float* data, int ndim, const int64_t* shape);
int gitb200_student_finalize(gitb200_student* s);
int gitb200_student_logits_ld(const gitb200_student* s); /* vocabulary rounded up to 256 */
/* ---- distillation training step of the student decoder (BASELINE.json configs[4]; DistillationTrainer.training_step,
 * model.py:880-983, optimizer model.py:1105, DDP train.py:217-221) -------------------------------------------------------
 * loss = KLDivLoss(batchmean)(log_softmax(student/T), softmax(teacher/T)) * T^2 + CrossEntropyLoss(ignore_index=0)(student[:, :-1],
 * y[:, 1:]).  Parameters live in ONE flat fp32 vector (padded to the GEMM tile multiples; the vocabulary head first); the
 * caller supplies a gradient vector of the same length (n = return value of _train_begin) and all-reduces it between
 * _train_backward and _train_apply -- [0, head_floats) may be reduced as soon as phase 0 has been enqueued, while phase 1
 * runs.  Dropout is not applied (parity oracle: torch.autograd on the same modules with dropout off).
 *   _set_training(1) before the weights are loaded keeps their fp32 values for the master copy;
 *   _train_forward: tokens_dev int32 [B, L], memory_dev fp32 [B, M, d_model], teacher_logits_dev fp32 [B*L, ld_teacher]
 *                   -> loss_dev fp32 [3] = (total, KL, CE); activations are kept for the backward pass;
 *   _train_backward: phase 0 = vocabulary head, phase 1 = decoder layers + embedding (+ d loss / d memory fp32 [B, M, d_model]);
 *   _train_apply: torch.optim.Adam on grads * grad_scale, then the bf16 operand copies are refreshed;
 *   _train_export: parameter (which = 0) or gradient (which = 1) `name` in the reference's tensor shape. */
int gitb200_student_set_training(gitb200_student* s, int enable);
long long gitb200_student_train_begin(gitb200_student* s, float lr, float beta1, float beta2, float eps);
long long gitb200_student_train_head_floats(const gitb200_student* s);
int gitb200_student_train_forward(gitb200_student* s, const int32_t* tokens_dev, const float* memory_dev, const float* teacher_logits_dev,
                                  int ld_teacher, int B, int L, int M, float temperature, float* loss_dev, void* stream);
int gitb200_student_train_backward(gitb200_student* s, int phase, float* grads_dev, float* d_memory_dev, void* stream);
int gitb200_student_train_apply(gitb200_student* s, const float* grads_dev, float grad_scale, void* stream);
int gitb200_student_train_export(gitb200_student* s, const char* name, int which, const float* grads_dev, float* out_dev, void* stream);

/* forward_decoder(y, memory), model.py:135-154: tokens_dev int32 [B, L], memory_dev fp32 [B, M, d_model] ->
 * logits_dev fp32 [B*L, logits_ld] (teacher-forced, every position). */
int gitb200_student_forward_decoder(gitb200_student* s, const int32_t* tokens_dev, const float* memory_dev, int B, int L, int M,
                                    float* logits_dev, void* stream);
/* greedy_decode, model.py:156-187, on a given memory, with a K/V cache instead of the reference's full re-decode per step.
 * tokens_dev int32 [B, max_len + 1] (CLS first); *out_len_dev = length of the reference's returned sequence: it stops only
 * when EVERY row emitted SEP in the same step (model.py:184), columns >= *out_len_dev are not part of the result. */
int gitb200_student_greedy_decode(gitb200_student* s, const float* memory_dev, int B, int M, int max_len, int32_t* tokens_dev,
                                  int32_t* out_len_dev, void* stream);

/* ---- single operators (used by the parity tests; same kernels the pipeline launches) ---------- */
/* out = act(A[M,K] * W[N,K]^T + bias) + residual; bf16 in/out (uint16 storage), fp32 bias. act: 0 none,
 * 1 QuickGELU, 2 erf-GELU, 3 ReLU.  tile_n: 0 auto, 128 or 256. */
int gitb200_op_gemm(const void* a_dev, const void* w_dev, int M, int N, int K, const float* bias_dev,
                    const void* residual_dev, int act, void* out_bf16_dev, float* out_f32_dev, int tile_n,
                    void* stream);
/* C = A W^T + bias + residual (bf16) AND LayerNorm(C) * gamma + beta as a second bf16 output, both from the CTA-pair tcgen05 GEMM
 * (M >= 1024, N a multiple of 256 up to 1024): the operator behind gitb200_set_fuse_layernorm. */
int gitb200_op_gemm_ln(const void* a_dev, const void* w_dev, int M, int N, int K, const float* bias_dev, const void* residual_dev,
                       const float* gamma_dev, const float* beta_dev, float eps, void* out_bf16_dev, void* ln_out_bf16_dev, void* stream);
int gitb200_op_layernorm(const void* x_dev, int rows, int cols, const float* gamma_dev, const float* beta_dev,
                         float eps, void* out_bf16_dev, void* stream);
/* qkv: bf16 [n_groups*group_len, 3*heads*64] -> out bf16 [n_groups*group_len, heads*64] */
int gitb200_op_attention_groups(const void* qkv_dev, void* out_dev, int n_groups, int group_len, int heads,
                                float scale, void* stream);
/* the same operator on the warp-level mma.sync path (the kernel the tcgen05 one replaced; kept as a cross-check) */
int gitb200_op_attention_groups_mma(const void* qkv_dev, void* out_dev, int n_groups, int group_len, int heads,
                                    float scale, void* stream);
/* Decode-step / text-row attention (SURVEY K11; the attention of model.py:1056-1075's text rows over the clip's visual keys and
 * their own text history): q bf16 [n_clips*rows_per_clip, heads*64]; vis_kv bf16 [n_clips*n_vis, 2*heads*64] (K | V);
 * txt_kv bf16 [n_text][n_clips*rows_per_clip][2*heads*64]; anc int32 [rows, n_text] (slot of the row's ancestor at each text
 * position, NULL = the row itself); every row sees all n_vis visual keys of its clip and n_text text keys.  splits >= 1 key
 * splits (partials combined by a second kernel).  out bf16 [rows, heads*64]. */
int gitb200_op_text_attention(const void* q_dev, const void* vis_kv_dev, const void* txt_kv_dev, const int32_t* anc_dev, int n_clips,
                              int rows_per_clip, int heads, int n_vis, int n_text, int splits, float scale, void* out_dev, void* stream);
/* Search on a pre-computed score sequence: logits_dev fp32 [max_steps-1, n_clips*beam, ld]. */
int gitb200_op_search(const float* logits_dev, int ld, int vocab, int n_clips, int sos, int eos,
                      const gitb200_search_params* sp, int32_t* tokens_dev, float* logprobs_dev, void* stream);

/* Per-launch timing of the tcgen05 GEMM kernel with CUDA events recorded on the launching stream
 * (enable != 0 resets the counters).  read: summed milliseconds, summed 2*M*N*K flops, launches. */
void gitb200_profile_gemm(int enable);
void gitb200_profile_gemm_read(double* ms, double* flops, long long* launches);
/* Same switch, second counter: the decode-step attention launches (text_attention_kernel, the HBM-bound kernel of the
 * path): summed CUDA-event time, summed ALGORITHMIC bytes (each clip's visual K/V once + every row's text K/V) and the
 * number of launches since gitb200_profile_gemm(1). */
void gitb200_profile_decode_attention_read(double* ms, double* bytes, long long* launches);

/* Number of caption calls served by replaying the captured CUDA graph. */
long long gitb200_graph_launches(const gitb200_ctx* ctx);

/* Number of kernels this library has launched since the last call with reset != 0 (bench.py's gpu_launches). */
long long gitb200_launch_count(int reset);

#ifdef __cplusplus
}
#endif
#endif /* GITB200_H_ */

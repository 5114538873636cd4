// C-ABI (include/gitb200.h) and the host-side engine of the captioning path: weight repacking,
// workspace / KV-cache management in HBM, and the launch sequences for
//   encode  (CLIP ViT over every frame + temporal embeddings)          -- model.py:378-382
//   visual pass of the prefix-LM decoder (fills the visual K/V cache)  -- first call of decoding_step
//   decode steps + device-side beam / greedy search                    -- model.py:426-462, :479-678
//   teacher-forced logits (forward_one_custom)                         -- model.py:371-424
//
// HBM layout (all activations bf16, row-major, rows = tokens):
//   ViT:      x/ln [n_clips*F*T, W], qkv [.., 3W], attn [.., W], mlp [.., 4W]
//   decoder:  hv [n_clips*Nv, H] visual hidden states; kv[l] [n_clips*Nv, 3H] = this layer's q|k|v of the
//             visual tokens -- columns [H, 3H) ARE the visual K/V cache that every decode step of every
//             beam of the clip reads (pages = one clip's contiguous Nv rows, shared by all beams);
//             txt_kv[l] [max_len][rows][2H] text K/V cache, one slot per beam row and position, re-ordered
//             through the ancestor table instead of being copied.
#include <cuda_runtime.h>
#include <math.h>
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>

#include <atomic>
#include <map>
#include <string>
#include <vector>

#include "../../include/gitb200.h"
#include "kernels.h"

static std::atomic<long long> g_launches{0};
void note_launch(int n) { g_launches += n; }

namespace {

std::string g_create_err;

struct DevF32 {
  float* p = nullptr;
  std::vector<int64_t> shape;
  size_t numel() const {
    size_t n = 1;
    for (auto d : shape) n *= (size_t)d;
    return n;
  }
};

struct VitLayer {
  float *ln1_g, *ln1_b, *ln2_g, *ln2_b, *b_qkv, *b_out, *b_fc1, *b_fc2;
  bf16 *w_qkv, *w_out, *w_fc1, *w_fc2;
  // ln_1 folded into the QKV projection and ln_2 into fc1 (W * diag(gamma), bias + W beta, column sums of W')
  bf16 *wf_qkv, *wf_fc1;
  float *bf_qkv, *bf_fc1, *cs_qkv, *cs_fc1;
};
struct DecLayer {
  float *b_qkv, *b_out, *lna_g, *lna_b, *b_fc1, *b_fc2, *lno_g, *lno_b;
  bf16 *w_qkv, *w_out, *w_fc1, *w_fc2;
};

template <typename T>
struct Buf {
  T* p = nullptr;
  size_t cap = 0;  // elements
};

}  // namespace

struct gitb200_ctx {
  gitb200_config cfg;
  int device = 0;
  std::string err;
  bool finalized = false;
  std::map<std::string, DevF32> raw;  // staged fp32 weights (freed by finalize)
  std::vector<void*> weight_allocs;

  // geometry
  int T = 0, kpad = 0, vocab_pad = 0, n_temporal = 0;

  // repacked weights
  bf16 *w_patch = nullptr, *pos_bf16 = nullptr;
  float *cls = nullptr, *ln_pre_g = nullptr, *ln_pre_b = nullptr, *ln_post_g = nullptr, *ln_post_b = nullptr;
  float* temporal = nullptr;  // [n_temporal, W]
  std::vector<VitLayer> vit;
  bf16* w_proj = nullptr;
  float *b_proj = nullptr, *lnp_g = nullptr, *lnp_b = nullptr;
  float *words_f32 = nullptr, *pos_f32 = nullptr, *lne_g = nullptr, *lne_b = nullptr;
  std::vector<DecLayer> dec;
  bf16* w_vocab = nullptr;
  float* b_vocab = nullptr;

  // workspaces
  Buf<bf16> patches, x, lnb, qkv, attn, mlp, vf, hv, hvb, hvc, vattn, vmlp;
  std::vector<Buf<bf16>> kv;      // per decoder layer: [n_clips*Nv, 3H]
  std::vector<Buf<bf16>> txt_kv;  // per decoder layer: [max_len][rows][2H]
  Buf<bf16> tx, tq, ta, tb, tc, tf;
  Buf<float> logits, partial, vf_in_f32, stats_a, stats_b;  // stats_*: [rows, 2 W / 256, 2] partial row sums for the folded LayerNorms
  Buf<int> ibuf;       // search ints
  Buf<double> dbuf;    // search doubles
  Buf<float> fbuf;     // search floats
  Buf<int> pos_arr, ntext_arr, tok_arr;
  Buf<float> stage[2];  // host-path frame staging
  Buf<uint8_t> stage_u8[2];  // host-path staging of raw uint8 video frames (gitb200_caption_host_u8)
  Buf<int> out_tok;
  Buf<float> out_lp;
  cudaStream_t copy_stream = nullptr, comp_stream = nullptr;
  // The caller's stream that last received work of this context (every entry point with a `stream` argument is asynchronous).
  // The host-frame entry points run on the context's private NON-BLOCKING streams, which nothing orders behind that stream --
  // not even the legacy default stream does -- so they wait for it explicitly (order_after_caller_work): without that a
  // gitb200_caption(...) immediately followed by gitb200_caption_host*(...) ran both on the same workspaces at once.
  cudaStream_t last_stream = nullptr;
  bool last_stream_valid = false;
  cudaEvent_t ev_copy[2] = {nullptr, nullptr}, ev_done[2] = {nullptr, nullptr}, ev_user = nullptr;

  // CUDA graphs for the launch-bound small-batch calls (latency mode): a call signature is captured on its second
  // occurrence and replayed afterwards.  kind: 0 caption (small batch, whole call), 1 stream_push, 2 stream_caption, 3 stream_push_u8,
  // 5 decode-step segment, 6 encode + visual pass of a device-resident batch, 7 / 8 encode of a host chunk (fp32 / raw uint8), 9 visual pass.
  struct GraphKey {
    int kind = -1;
    const void *p0 = nullptr, *p1 = nullptr, *p2 = nullptr;
    int i0 = 0, i1 = 0, i2 = 0, i3 = 0, i4 = 0, i5 = 0;
    gitb200_search_params sp{};
    bool operator==(const GraphKey& o) const {
      return kind == o.kind && p0 == o.p0 && p1 == o.p1 && p2 == o.p2 && i0 == o.i0 && i1 == o.i1 && i2 == o.i2 && i3 == o.i3 &&
             i4 == o.i4 && i5 == o.i5 && memcmp(&sp, &o.sp, sizeof(sp)) == 0;
    }
  };
  struct GraphEntry {
    GraphKey key;
    cudaGraphExec_t exec = nullptr;  // nullptr: seen once, not captured yet
    unsigned long long gen = 0;      // workspace generation the graph was captured under
  };
  std::vector<GraphEntry> graphs;
  // A captured graph bakes in the workspace pointers (x / qkv / kv / txt_kv / ibuf ...) and the launch sequence the
  // switches select.  Whenever a workspace is actually reallocated (ensure(): cudaFree + cudaMalloc for a larger call or
  // gitb200_reserve) or a switch that changes the launch sequence flips (fold_ln, sweep_rows, pipeline), the generation
  // moves on and every graph captured under an older generation is destroyed before it can be replayed.
  unsigned long long ws_gen = 0;
  bool graphs_enabled = true;
  long long graph_launches = 0;

  // Two-stream chunk pipeline for large batches: chunk i runs encode + decode on stream i & 1 with workspace set
  // i & 1 (this context / its twin, which shares the weights), offset by one phase so that the HBM / latency bound
  // decode of one chunk overlaps the tensor bound encode of the next.
  gitb200_ctx* twin = nullptr;
  bool is_twin = false;
  bool fold_ln = false;     // ViT ln_1 / ln_2 folded into the QKV / fc1 GEMMs (rows >= 1024); the row statistics are partial sums per
                            // 128-column half tile stored by the producing GEMM and added in slot order by the consumer: bit-reproducible
  // Opt-in: the LayerNorm that follows a residual GEMM (ViT ln_2 / next block's ln_1, the decoder's three post-LNs over the visual
  // rows) written by that GEMM as a second output (gemm2 LNOUT, rows >= 1024): no separate LayerNorm kernel, bit-reproducible --
  // and measured 1 % SLOWER than the separate kernels (profiles/r02_layernorm_fusion.md): default off.
  bool fuse_ln = false;
  int pipeline_chunk = 0;   // 0 off (default: measured slower, see DESIGN.md), -1 auto, > 0 clips per chunk
  // Large batches walk the ViT / the decoder's visual pass in sub-batches of about this many token rows (0: one sweep).
  // 151296 = 128 six-frame GIT-base clips.  Throughput-neutral from 128 clips up (A/B on one box, 512 clips per step:
  // 2431 / 2432 / 2430 / 2384 clips/s for one sweep / 128 / 256 / 64 clips per sub-batch), but the row-sized scratch
  // shrinks with it: 17.6 -> 4.4 GB at 512 clips, so larger batches fit.
  int sweep_rows = 151296;
  cudaStream_t pipe_stream[2] = {nullptr, nullptr};
  cudaEvent_t ev_fork = nullptr, ev_enc0 = nullptr, ev_join[2] = {nullptr, nullptr};

  // streaming window (real_time_inference.py:38-61): per-frame ViT features (after ln_post, before the temporal
  // embedding) of the last `num_image_with_embedding` frames
  Buf<bf16> ring;
  int ring_count = 0, ring_head = 0;

  // multi-stream pool (gitb200_streams_*): one window of num_image_with_embedding frames per camera stream, bf16
  // [pool_streams][cap][T][W], same per-frame features as `ring`.  head / count of every window are kept here on the host.
  // The per-call tables (ln_post output row of every pushed frame, oldest ring slot of every captioned window) are copied
  // into pool_rows / pool_oldest at fixed addresses, so a captured graph replays for any set of streams of the same shape.
  Buf<bf16> pool;
  int pool_streams = 0;
  std::vector<int> pool_head, pool_count;
  Buf<int> pool_rows, pool_oldest;

  // forward-hook taps on image_encoder.transformer.resblocks[i] (model.py:847): outputs copied out by the next encodes
  std::vector<int> tap_layers;
  float* tap_out = nullptr;

  // decode loop early exit (model.py:640): poll the device's done count every N steps (0 = never: fully asynchronous)
  int early_exit_every = 4;
  bool persistent_decode = true;     // single-clip searches run as ONE persistent cooperative kernel (decode_mega.cu)
  Buf<unsigned int> mega_bar;        // its grid-barrier counter
  Buf<unsigned long long> mega_trace;  // optional per-phase cycle counters (gitb200_debug_persistent_decode_trace)
  bool mega_trace_on = false;
  int* h_done = nullptr;             // pinned
  int last_decode_steps = 0;         // decode steps the last gitb200_decode / _caption call enqueued
  int graph_max_clips = 8;           // calls of up to this many clips are captured into ONE CUDA graph (latency mode)
  // Larger batches are graphed in pieces that do not depend on the caller's output pointers: encode (+ visual pass) per
  // frame buffer, and the decode loop in segments of `early_exit_every` steps with the finished-clip poll between them --
  // the ~1200 launches of a step reach the GPU as a handful of graph launches (+2-4 % at 512 clips, same-box A/B).
  bool graph_segments = true;
  cudaEvent_t ev_gfork = nullptr, ev_gjoin = nullptr;

  // current state
  int cur_clips = 0, cur_nv = 0;     // visual features held in vf
  int step_rows_per_clip = 0;        // step-wise decoding state
  bool visual_pass_done = false;
  int visual_pass_full = 0;
  int anc_parity = 0;
  bool step_anc_used = false;
};

namespace {

int fail(gitb200_ctx* c, int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  if (c)
    c->err = buf;
  else
    g_create_err = buf;
  return code;
}

#define CUDA_OK(c, expr)                                                                                   \
  do {                                                                                                     \
    cudaError_t e_ = (expr);                                                                               \
    if (e_ != cudaSuccess)                                                                                 \
      return fail(c, GITB200_ERR_CUDA, "%s failed: %s [%s] (%s:%d)", #expr, cudaGetErrorString(e_),        \
                  gemm_last_error(), __FILE__, __LINE__);                                                  \
  } while (0)

// Debug aid (GITB200_POISON=1 in the environment): every fresh device allocation is filled with 0xFF bytes (NaN as bf16 and
// as fp32, -1 as int), so a kernel that consumes memory nobody wrote shows up as NaN / a fault instead of depending on
// whatever the allocator hands out (a fresh process gets zero pages, a long-running one gets its own freed buffers).
bool poison_allocs() {
  static const bool on = [] { const char* e = getenv("GITB200_POISON"); return e != nullptr && e[0] != '\0' && e[0] != '0'; }();
  return on;
}

template <typename T>
int ensure(gitb200_ctx* c, Buf<T>& b, size_t n) {
  if (b.cap >= n) return 0;
  if (b.p) {
    CUDA_OK(c, cudaFree(b.p));
    if (c) c->ws_gen++;  // captured graphs hold the freed pointer: they are stale from here on (see gitb200_ctx::ws_gen)
  }
  b.p = nullptr;
  b.cap = 0;
  CUDA_OK(c, cudaMalloc(&b.p, n * sizeof(T)));
  if (poison_allocs()) CUDA_OK(c, cudaMemset(b.p, 0xFF, n * sizeof(T)));
  b.cap = n;
  return 0;
}
#define ENSURE(c, b, n)                   \
  do {                                    \
    int r_ = ensure(c, b, (size_t)(n));   \
    if (r_) return r_;                    \
  } while (0)

template <typename T>
int walloc(gitb200_ctx* c, T** p, size_t n) {
  CUDA_OK(c, cudaMalloc(p, n * sizeof(T)));
  if (poison_allocs()) CUDA_OK(c, cudaMemset(*p, 0xFF, n * sizeof(T)));
  c->weight_allocs.push_back(*p);
  return 0;
}

const DevF32* find(gitb200_ctx* c, const std::string& name) {
  auto it = c->raw.find(name);
  return it == c->raw.end() ? nullptr : &it->second;
}

// fp32 [rows, cols] -> bf16 [dst_rows, dst_cols] zero padded
int to_bf16(gitb200_ctx* c, const std::string& name, int rows, int cols, int dst_rows, int dst_cols, bf16** out) {
  const DevF32* w = find(c, name);
  if (!w) return fail(c, GITB200_ERR_MISSING, "missing weight %s", name.c_str());
  if (w->numel() != (size_t)rows * cols)
    return fail(c, GITB200_ERR_INVALID, "weight %s has %zu elements, expected %d x %d", name.c_str(), w->numel(), rows, cols);
  int r = walloc(c, out, (size_t)dst_rows * dst_cols);
  if (r) return r;
  CUDA_OK(c, cast_f32_to_bf16(w->p, rows, cols, cols, *out, dst_cols, dst_rows, dst_cols, 0));
  return 0;
}
// fp32 vector copy (optionally zero padded)
int to_f32(gitb200_ctx* c, const std::string& name, size_t n, size_t n_pad, float** out) {
  const DevF32* w = find(c, name);
  if (!w) return fail(c, GITB200_ERR_MISSING, "missing weight %s", name.c_str());
  if (w->numel() != n) return fail(c, GITB200_ERR_INVALID, "weight %s has %zu elements, expected %zu", name.c_str(), w->numel(), n);
  int r = walloc(c, out, n_pad);
  if (r) return r;
  if (n_pad > n) CUDA_OK(c, cudaMemset(*out, 0, n_pad * sizeof(float)));
  CUDA_OK(c, cudaMemcpy(*out, w->p, n * sizeof(float), cudaMemcpyDeviceToDevice));
  return 0;
}
#define TRY(expr)          \
  do {                     \
    int r_ = (expr);       \
    if (r_) return r_;     \
  } while (0)

int gemm(gitb200_ctx* c, const GemmArgs& g, cudaStream_t s) {
  CUDA_OK(c, gemm_bf16(g, s, 0));
  return 0;
}

GemmArgs linear(const bf16* A, int lda, const bf16* W, int K, int M, int N, const float* bias, bf16* out, int ldo) {
  GemmArgs g;
  g.A = A; g.lda = lda; g.W = W; g.ldw = K; g.M = M; g.N = N; g.K = K; g.bias = bias; g.out = out; g.ldo = ldo;
  return g;
}

int ln(gitb200_ctx* c, const bf16* x, int rows, int cols, const float* g, const float* b, float eps, bf16* out,
       cudaStream_t s, const float* addend = nullptr, int add_group = 1, int add_period = 1, float* out32 = nullptr) {
  LayerNormArgs a;
  a.x = x; a.ldx = cols; a.rows = rows; a.cols = cols; a.gamma = g; a.beta = b; a.eps = eps; a.out = out; a.ldo = cols;
  a.addend = addend; a.add_group = add_group; a.add_period = add_period; a.out_f32 = out32; a.ldo32 = cols;
  CUDA_OK(c, layernorm_bf16(a, s));
  return 0;
}

// Clips per sub-batch of a sweep over `n_clips` clips of `rows_per_clip` token rows: at most sweep_rows rows, and the
// sub-batches balanced (32 clips at 24 per sub-batch run as 16 + 16, not 24 + 8: every launch keeps the SMs equally full).
int sweep_clips(int sweep_rows, int rows_per_clip, int n_clips) {
  if (sweep_rows <= 0 || n_clips <= 1) return n_clips;
  int sub = sweep_rows / rows_per_clip;
  if (sub < 1) sub = 1;
  if (sub >= n_clips) return n_clips;
  const int n_sub = (n_clips + sub - 1) / sub;
  return (n_clips + n_sub - 1) / n_sub;
}

// ------------------------------------------------------------------ encode
// clip_offset / total_clips: the visual features of this call land at clip index `clip_offset` of a buffer sized for
// `total_clips` clips (host path: chunks are encoded as their frames arrive, then decoded together).
// frame_out != nullptr: streaming mode -- write ln_post(x) WITHOUT temporal embeddings to frame_out and leave the
// context's visual features untouched.  out_rows != nullptr (device table, one entry per frame): frame f's T rows go to
// frame_out rows out_rows[f] .. out_rows[f] + T - 1 (a multi-stream push: each frame straight into its stream's ring slot).
// raw != nullptr: `frames` is ignored and the patch matrix is filled straight from raw uint8 BGR video frames
// (image_transform() fused into the patch-embed loader, preprocess.cu).
struct RawFrames {
  const uint8_t* p;  // [n_clips, n_frames, height, width, 3] on the device
  int height, width;
};

int run_encode(gitb200_ctx* c, const float* frames, int n_clips, int n_frames, cudaStream_t s, int clip_offset = 0, int total_clips = 0,
               bf16* frame_out = nullptr, bool temporal = true, const RawFrames* raw = nullptr, const int* out_rows = nullptr) {
  const gitb200_config& k = c->cfg;
  const int W = k.vit_width, T = c->T, G = k.resolution / k.patch;
  // zip() truncation of model.py:380: frames beyond the temporal-embedding list are dropped
  const int F = (temporal && k.num_image_with_embedding > 0 && n_frames > k.num_image_with_embedding) ? k.num_image_with_embedding : n_frames;
  const int rows = n_clips * F * T;
  const int prow = n_clips * F * G * G;
  ENSURE(c, c->patches, (size_t)prow * c->kpad);
  ENSURE(c, c->x, (size_t)rows * W);
  ENSURE(c, c->lnb, (size_t)rows * W);
  ENSURE(c, c->qkv, (size_t)rows * 3 * W);
  ENSURE(c, c->attn, (size_t)rows * W);
  ENSURE(c, c->mlp, (size_t)rows * 4 * W);
  if (total_clips < clip_offset + n_clips) total_clips = clip_offset + n_clips;
  if (frame_out != nullptr) {
  } else if (clip_offset == 0) ENSURE(c, c->vf, (size_t)total_clips * F * T * W);  // later chunks must not reallocate it
  else if (c->vf.cap < (size_t)total_clips * F * T * W) return fail(c, GITB200_ERR_STATE, "visual feature buffer too small for chunked encode");

  const size_t frame_elems = (size_t)3 * k.resolution * k.resolution;
  if (raw != nullptr) {
    const size_t raw_frame = (size_t)raw->height * raw->width * 3;
    if (F == n_frames) {
      CUDA_OK(c, preprocess_frames_u8_to_patches(raw->p, n_clips * F, raw->height, raw->width, k.resolution, k.patch, c->kpad, c->patches.p, s));
    } else {
      for (int i = 0; i < n_clips; ++i)
        CUDA_OK(c, preprocess_frames_u8_to_patches(raw->p + (size_t)i * n_frames * raw_frame, F, raw->height, raw->width, k.resolution,
                                                   k.patch, c->kpad, c->patches.p + (size_t)i * F * G * G * c->kpad, s));
    }
  } else if (F == n_frames) {
    CUDA_OK(c, im2col_patches(frames, n_clips * F, k.resolution, k.patch, c->kpad, c->patches.p, s));
  } else {
    for (int i = 0; i < n_clips; ++i)
      CUDA_OK(c, im2col_patches(frames + (size_t)i * n_frames * frame_elems, F, k.resolution, k.patch, c->kpad,
                                c->patches.p + (size_t)i * F * G * G * c->kpad, s));
  }
  // patch embedding (conv1 as GEMM) + positional embedding, rows shifted to leave the CLS slot of every frame
  {
    GemmArgs g = linear(c->patches.p, c->kpad, c->w_patch, c->kpad, prow, W, nullptr, c->x.p, W);
    g.residual = c->pos_bf16; g.ldr = W; g.res_periodic = 1; g.gin = G * G; g.gout = T; g.goff = 1;
    TRY(gemm(c, g, s));
  }
  CUDA_OK(c, write_cls_rows(c->cls, c->pos_bf16, n_clips * F, T, W, c->x.p, s));
  // ln_pre (in place semantics: x <- ln_pre(x)); the residual stream starts from the normalised tokens
  const bool fold = c->fold_ln && rows >= 1024;  // the folded-LayerNorm epilogue lives in the CTA-pair GEMM
  const bool fuse = c->fuse_ln && !fold && rows >= 1024 && W <= 1024;  // LayerNorm as the residual GEMM's second output (CTA-pair GEMM)
  if (fold) {
    ENSURE(c, c->stats_a, (size_t)rows * 2 * (2 * W / 256));
    ENSURE(c, c->stats_b, (size_t)rows * 2 * (2 * W / 256));
  }
  {
    LayerNormArgs a;
    a.x = c->x.p; a.ldx = W; a.rows = rows; a.cols = W; a.gamma = c->ln_pre_g; a.beta = c->ln_pre_b; a.eps = k.vit_ln_eps;
    a.out = c->lnb.p; a.ldo = W; a.stats_out = fold ? c->stats_a.p : nullptr; a.stats_slots = 2 * W / 256;
    CUDA_OK(c, layernorm_bf16(a, s));
  }
  std::swap(c->x.p, c->lnb.p);
  std::swap(c->x.cap, c->lnb.cap);
  const float scale = 1.0f / sqrtf((float)(W / k.vit_heads));
  // resblock output taps: fp32 [n_taps, rows, W] (rows = (clip, frame, token))
  auto emit_tap = [&](int l) -> int {
    if (c->tap_out == nullptr || frame_out != nullptr) return 0;
    for (size_t i = 0; i < c->tap_layers.size(); ++i)
      if (c->tap_layers[i] == l)
        CUDA_OK(c, cast_bf16_to_f32(c->x.p, rows, W, W, c->tap_out + ((size_t)i * total_clips + clip_offset) * F * T * W, W, s));
    return 0;
  };
  for (int l = 0; l < k.vit_layers; ++l) {
    const VitLayer& L = c->vit[l];
    if (fold) {
      // ln_1 and ln_2 never materialise: the QKV / fc1 GEMMs read the raw residual stream and normalise in their
      // epilogue from the row statistics the previous residual GEMM (or ln_pre) produced.
      {
        GemmArgs g = linear(c->x.p, W, L.wf_qkv, W, rows, 3 * W, L.bf_qkv, c->qkv.p, 3 * W);
        g.ln_stats = c->stats_a.p; g.ln_colsum = L.cs_qkv; g.ln_eps = k.vit_ln_eps;
        TRY(gemm(c, g, s));
      }
      CUDA_OK(c, attention_groups_tc(c->qkv.p, 3 * W, c->attn.p, W, n_clips * F, T, k.vit_heads, scale, s));
      {
        GemmArgs g = linear(c->attn.p, W, L.w_out, W, rows, W, L.b_out, c->x.p, W);
        g.residual = c->x.p; g.ldr = W; g.stats_out = c->stats_b.p;
        TRY(gemm(c, g, s));
      }
      {
        GemmArgs g = linear(c->x.p, W, L.wf_fc1, W, rows, 4 * W, L.bf_fc1, c->mlp.p, 4 * W);
        g.act = ACT_QUICK_GELU; g.ln_stats = c->stats_b.p; g.ln_colsum = L.cs_fc1; g.ln_eps = k.vit_ln_eps;
        TRY(gemm(c, g, s));
      }
      {
        GemmArgs g = linear(c->mlp.p, 4 * W, L.w_fc2, 4 * W, rows, W, L.b_fc2, c->x.p, W);
        g.residual = c->x.p; g.ldr = W; g.stats_out = c->stats_a.p;
        TRY(gemm(c, g, s));
      }
      TRY(emit_tap(l));
      continue;
    }
    // ln_1: a kernel of its own for the first block; afterwards the previous block's fc2 GEMM has written it (fused)
    if (!(fuse && l > 0)) TRY(ln(c, c->x.p, rows, W, L.ln1_g, L.ln1_b, k.vit_ln_eps, c->lnb.p, s));
    TRY(gemm(c, linear(c->lnb.p, W, L.w_qkv, W, rows, 3 * W, L.b_qkv, c->qkv.p, 3 * W), s));
    CUDA_OK(c, attention_groups_tc(c->qkv.p, 3 * W, c->attn.p, W, n_clips * F, T, k.vit_heads, scale, s));
    {
      GemmArgs g = linear(c->attn.p, W, L.w_out, W, rows, W, L.b_out, c->x.p, W);
      g.residual = c->x.p; g.ldr = W;  // x += out_proj(attn): each element is read then written by one thread
      if (fuse) {  // ... and ln_2(x) leaves the same GEMM as its second output
        g.lnout = c->lnb.p; g.lnout_ld = W; g.lnout_gamma = L.ln2_g; g.lnout_beta = L.ln2_b; g.lnout_eps = k.vit_ln_eps;
      }
      TRY(gemm(c, g, s));
    }
    if (!fuse) TRY(ln(c, c->x.p, rows, W, L.ln2_g, L.ln2_b, k.vit_ln_eps, c->lnb.p, s));
    {
      GemmArgs g = linear(c->lnb.p, W, L.w_fc1, W, rows, 4 * W, L.b_fc1, c->mlp.p, 4 * W);
      g.act = ACT_QUICK_GELU;
      TRY(gemm(c, g, s));
    }
    {
      GemmArgs g = linear(c->mlp.p, 4 * W, L.w_fc2, 4 * W, rows, W, L.b_fc2, c->x.p, W);
      g.residual = c->x.p; g.ldr = W;
      if (fuse && l + 1 < k.vit_layers) {  // the next block's ln_1
        const VitLayer& Ln = c->vit[l + 1];
        g.lnout = c->lnb.p; g.lnout_ld = W; g.lnout_gamma = Ln.ln1_g; g.lnout_beta = Ln.ln1_b; g.lnout_eps = k.vit_ln_eps;
      }
      TRY(gemm(c, g, s));
    }
    TRY(emit_tap(l));
  }
  // ln_post on all tokens + temporal embedding of the frame (frame index = (row / T) % F)
  if (frame_out != nullptr) {
    LayerNormArgs a;
    a.x = c->x.p; a.ldx = W; a.rows = rows; a.cols = W; a.gamma = c->ln_post_g; a.beta = c->ln_post_b; a.eps = k.vit_ln_eps;
    a.out = frame_out; a.ldo = W; a.out_row_base = out_rows; a.out_group = T;
    CUDA_OK(c, layernorm_bf16(a, s));
    return 0;
  }
  TRY(ln(c, c->x.p, rows, W, c->ln_post_g, c->ln_post_b, k.vit_ln_eps, c->vf.p + (size_t)clip_offset * F * T * W, s,
         (temporal && k.num_image_with_embedding > 0) ? c->temporal : nullptr, T, F));
  c->cur_clips = clip_offset + n_clips;
  c->cur_nv = F * T;
  c->visual_pass_done = false;
  c->step_rows_per_clip = 0;  // a step-wise decoding state set up for the previous features is void
  return 0;
}

// ------------------------------------------------------------------ decoder over the visual tokens
// full_last: also run attention/FFN of the last layer on the visual rows (needed only for hidden-state output)
int run_visual_pass(gitb200_ctx* c, bool full_last, float* hidden_out, int L_text, cudaStream_t s) {
  const gitb200_config& k = c->cfg;
  const int H = k.hidden, Nv = c->cur_nv, Ball = c->cur_clips;
  if (Ball <= 0 || Nv <= 0) return fail(c, GITB200_ERR_STATE, "no visual features: call gitb200_encode or gitb200_set_visual_features first");
  // Clips are independent here, so a large batch walks the layers in sub-batches of ~`sweep_rows` token rows: every
  // row-sized scratch buffer is then allocated for one sub-batch only (4x less at 512 clips; throughput-neutral from
  // 128 clips per sub-batch up).  Row results do not depend on the sub-batch they are computed in (tests: bit-exact).
  const int Bsub = sweep_clips(c->sweep_rows, Nv, Ball);
  const int Msub = Bsub * Nv;
  ENSURE(c, c->hv, (size_t)Msub * H);
  ENSURE(c, c->hvb, (size_t)Msub * H);
  ENSURE(c, c->hvc, (size_t)Msub * H);
  ENSURE(c, c->vattn, (size_t)Msub * H);
  ENSURE(c, c->vmlp, (size_t)Msub * k.ffn);
  if ((int)c->kv.size() != k.dec_layers) c->kv.resize(k.dec_layers);
  for (int l = 0; l < k.dec_layers; ++l) ENSURE(c, c->kv[l], (size_t)Ball * Nv * 3 * H);
  const float scale = 1.0f / sqrtf((float)(H / k.dec_heads));

 for (int b0 = 0; b0 < Ball; b0 += Bsub) {
  const int B = (Ball - b0) < Bsub ? (Ball - b0) : Bsub, M = B * Nv;
  const size_t kvoff = (size_t)b0 * Nv * 3 * H;
  auto emit_hidden = [&](int idx) -> int {
    if (!hidden_out) return 0;
    // hidden_out: [B, layers+1, Nv+L, H]; visual rows of clip b, state idx
    const size_t per_state = (size_t)(Nv + L_text) * H;
    for (int b = 0; b < B; ++b)
      CUDA_OK(c, cast_bf16_to_f32(c->hv.p + (size_t)b * Nv * H, Nv, H, H,
                                  hidden_out + ((size_t)(b0 + b) * (k.dec_layers + 1) + idx) * per_state, H, s));
    return 0;
  };

  // visual_projection = Linear + LayerNorm
  const bool fuse = c->fuse_ln && M >= 1024;  // the LayerNorms leave the GEMMs that feed them as a second output (CTA-pair GEMM)
  {
    GemmArgs g = linear(c->vf.p + (size_t)b0 * Nv * k.vit_width, k.vit_width, c->w_proj, k.vit_width, M, H, c->b_proj, c->hvb.p, H);
    if (fuse) {
      g.lnout = c->hv.p; g.lnout_ld = H; g.lnout_gamma = c->lnp_g; g.lnout_beta = c->lnp_b; g.lnout_eps = k.proj_ln_eps;
    }
    TRY(gemm(c, g, s));
  }
  if (!fuse) TRY(ln(c, c->hvb.p, M, H, c->lnp_g, c->lnp_b, k.proj_ln_eps, c->hv.p, s));
  TRY(emit_hidden(0));
  for (int l = 0; l < k.dec_layers; ++l) {
    const DecLayer& L = c->dec[l];
    const bool full = (l + 1 < k.dec_layers) || full_last;
    bf16* kvl = c->kv[l].p + kvoff;
    if (full) {
      TRY(gemm(c, linear(c->hv.p, H, L.w_qkv, H, M, 3 * H, L.b_qkv, kvl, 3 * H), s));
    } else {
      // last layer: only K and V of the visual tokens are ever read again
      TRY(gemm(c, linear(c->hv.p, H, L.w_qkv + (size_t)H * H, H, M, 2 * H, L.b_qkv + H, kvl + H, 3 * H), s));
      break;
    }
    CUDA_OK(c, attention_groups_tc(kvl, 3 * H, c->vattn.p, H, B, Nv, k.dec_heads, scale, s));
    {
      GemmArgs g = linear(c->vattn.p, H, L.w_out, H, M, H, L.b_out, c->hvb.p, H);
      g.residual = c->hv.p; g.ldr = H;
      if (fuse) {
        g.lnout = c->hvc.p; g.lnout_ld = H; g.lnout_gamma = L.lna_g; g.lnout_beta = L.lna_b; g.lnout_eps = k.bert_ln_eps;
      }
      TRY(gemm(c, g, s));
    }
    if (!fuse) TRY(ln(c, c->hvb.p, M, H, L.lna_g, L.lna_b, k.bert_ln_eps, c->hvc.p, s));
    {
      GemmArgs g = linear(c->hvc.p, H, L.w_fc1, H, M, k.ffn, L.b_fc1, c->vmlp.p, k.ffn);
      g.act = ACT_GELU_ERF;
      TRY(gemm(c, g, s));
    }
    {
      GemmArgs g = linear(c->vmlp.p, k.ffn, L.w_fc2, k.ffn, M, H, L.b_fc2, c->hvb.p, H);
      g.residual = c->hvc.p; g.ldr = H;
      if (fuse) {
        g.lnout = c->hv.p; g.lnout_ld = H; g.lnout_gamma = L.lno_g; g.lnout_beta = L.lno_b; g.lnout_eps = k.bert_ln_eps;
      }
      TRY(gemm(c, g, s));
    }
    if (!fuse) TRY(ln(c, c->hvb.p, M, H, L.lno_g, L.lno_b, k.bert_ln_eps, c->hv.p, s));
    TRY(emit_hidden(l + 1));
  }
 }
  c->visual_pass_done = true;
  c->visual_pass_full = full_last ? 1 : 0;
  return 0;
}

// ------------------------------------------------------------------ text rows through the decoder
struct TextPass {
  int n_clips, rows_per_clip, max_len;
  const int* tokens;     // [rows]
  const int* positions;  // [rows] or nullptr -> pos_const
  int pos_const;
  const int* n_text;     // [rows] or nullptr -> n_text_const
  int n_text_const;
  const int* anc;        // ancestor table or nullptr
  int slot_div, n_slots, slot_is_clip;
  float* logits;         // [rows, vocab_pad]
  float* hidden_out;     // optional fp32 [B, layers+1, Nv+L, H] (text rows written)
};

int ensure_text(gitb200_ctx* c, int rows, int n_slots, int max_len) {
  const gitb200_config& k = c->cfg;
  const int H = k.hidden;
  ENSURE(c, c->tx, (size_t)rows * H);
  ENSURE(c, c->tq, (size_t)rows * 3 * H);
  ENSURE(c, c->ta, (size_t)rows * H);
  ENSURE(c, c->tb, (size_t)rows * H);
  ENSURE(c, c->tc, (size_t)rows * H);
  ENSURE(c, c->tf, (size_t)rows * k.ffn);
  if ((int)c->txt_kv.size() != k.dec_layers) c->txt_kv.resize(k.dec_layers);
  for (int l = 0; l < k.dec_layers; ++l) ENSURE(c, c->txt_kv[l], (size_t)max_len * n_slots * 2 * H);
  return 0;
}

// Live timing of the decode-step attention launches (the HBM-bound kernel of the path) with CUDA events on the launching
// stream, switched together with the GEMM profile (gitb200_profile_gemm); read with gitb200_profile_decode_attention_read.
struct DecAttnProf {
  std::vector<cudaEvent_t> ev;  // pairs
  std::vector<double> bytes;
  size_t used = 0;
  double ms = 0, by = 0;
  long long n = 0;
} g_dap;

int dap_begin(cudaStream_t s) {
  if (!gemm_profile_enabled()) return -1;
  if (g_dap.ev.empty()) {
    g_dap.ev.resize(2 * 2048);
    g_dap.bytes.resize(2048);
    for (auto& e : g_dap.ev) cudaEventCreate(&e);
  }
  if (g_dap.used >= g_dap.bytes.size()) return -1;
  const int slot = (int)g_dap.used++;
  g_dap.bytes[slot] = 0;
  cudaEventRecord(g_dap.ev[2 * slot], s);
  return slot;
}

void dap_end(int slot, cudaStream_t s, double bytes) {
  cudaEventRecord(g_dap.ev[2 * slot + 1], s);
  g_dap.bytes[slot] = bytes;
}

void dap_drain() {
  for (size_t i = 0; i < g_dap.used; ++i) {
    float t = 0;
    if (g_dap.bytes[i] > 0 && cudaEventSynchronize(g_dap.ev[2 * i + 1]) == cudaSuccess &&
        cudaEventElapsedTime(&t, g_dap.ev[2 * i], g_dap.ev[2 * i + 1]) == cudaSuccess) {
      g_dap.ms += t;
      g_dap.by += g_dap.bytes[i];
      ++g_dap.n;
    }
  }
  g_dap.used = 0;
}

int run_text_pass(gitb200_ctx* c, const TextPass& t, cudaStream_t s) {
  const gitb200_config& k = c->cfg;
  const int H = k.hidden, rows = t.n_clips * t.rows_per_clip, Nv = c->cur_nv;
  const float scale = 1.0f / sqrtf((float)(H / k.dec_heads));
  // split the visual keys over several CTAs when there are too few (clip, head) pairs to fill 148 SMs
  const int chunks = (t.rows_per_clip + 3) / 4;
  int splits = (2 * 148 + t.n_clips * chunks * k.dec_heads - 1) / (t.n_clips * chunks * k.dec_heads);
  if (splits > 16) splits = 16;
  while (splits > 1 && Nv / splits < 64) --splits;
  if (splits < 1) splits = 1;
  if (splits > 1) ENSURE(c, c->partial, text_attention_workspace_floats(rows, k.dec_heads, splits));

  auto emit_hidden = [&](int idx) -> int {
    if (!t.hidden_out) return 0;
    const int L = t.rows_per_clip;
    const size_t per_state = (size_t)(Nv + L) * H;
    for (int b = 0; b < t.n_clips; ++b)
      CUDA_OK(c, cast_bf16_to_f32(c->tx.p + (size_t)b * L * H, L, H, H,
                                  t.hidden_out + ((size_t)b * (k.dec_layers + 1) + idx) * per_state + (size_t)Nv * H, H, s));
    return 0;
  };

  CUDA_OK(c, embed_text(t.tokens, t.positions, t.pos_const, rows, c->words_f32, c->pos_f32, c->lne_g, c->lne_b,
                        k.embed_ln_eps, H, c->tx.p, s));
  TRY(emit_hidden(0));
  // Latency mode (<= 4 rows: one clip greedy or beam 4, nothing else reads the hidden states): the two LayerNorms of a layer
  // run inside the skinny GEMMs that consume them (normalise-on-load, CTA 0 stores the normalised rows for the residuals)
  // and the K/V scatter inside the QKV projection: 6 launches per layer instead of 9 (a decode step is launch-latency
  // bound: ~5 us per dependent kernel against a 24 us weight-streaming floor).
  static const bool no_fused = [] { const char* e = getenv("GITB200_NO_FUSED_STEP"); return e != nullptr && e[0] == '1'; }();  // debug switch
  const bool fused = rows <= 4 && t.hidden_out == nullptr && H == 768 && !no_fused;
  for (int l = 0; l < k.dec_layers; ++l) {
    const DecLayer& L = c->dec[l];
    {
      // fused, l > 0: tb holds the previous layer's un-normalised output; its output LayerNorm runs here and lands in tx
      GemmArgs g = linear(fused && l > 0 ? c->tb.p : c->tx.p, H, L.w_qkv, H, rows, 3 * H, L.b_qkv, c->tq.p, 3 * H);
      if (fused) {
        if (l > 0) {
          g.lnl_gamma = c->dec[l - 1].lno_g; g.lnl_beta = c->dec[l - 1].lno_b; g.lnl_eps = k.bert_ln_eps; g.lnl_out = c->tx.p; g.lnl_ldo = H;
        }
        g.sc_kv = c->txt_kv[l].p; g.sc_q_width = H; g.sc_kv_width = 2 * H; g.sc_pos = t.positions; g.sc_pos_const = t.pos_const;
        g.sc_slot_div = t.slot_div; g.sc_n_slots = t.n_slots;
      }
      TRY(gemm(c, g, s));
    }
    if (!fused)
      CUDA_OK(c, store_text_kv(c->tq.p, 3 * H, rows, 2 * H, H, t.positions, t.pos_const, t.slot_div, t.n_slots,
                               c->txt_kv[l].p, s));
    TextAttnArgs a;
    a.q = c->tq.p; a.ldq = 3 * H; a.n_clips = t.n_clips; a.rows_per_clip = t.rows_per_clip; a.heads = k.dec_heads;
    a.vis_kv = c->kv[l].p; a.ld_vis = 3 * H; a.k_off = H; a.v_off = 2 * H; a.Nv = Nv;
    a.txt_kv = c->txt_kv[l].p; a.txt_slots = t.n_slots; a.text_slot_is_clip = t.slot_is_clip;
    a.anc = t.anc; a.anc_ld = t.max_len; a.n_text = t.n_text; a.n_text_const = t.n_text_const; a.max_text = t.max_len;
    a.scale = scale; a.out = c->ta.p; a.ldo = H; a.partial = c->partial.p; a.splits = splits;
    const int pslot = dap_begin(s);
    CUDA_OK(c, text_attention(a, s));
    // algorithmic bytes of this launch: every clip's visual K/V once (shared by its beam rows) + the text K/V of every row
    if (pslot >= 0)
      dap_end(pslot, s, (double)t.n_clips * Nv * 2 * H * sizeof(bf16) +
                            (double)rows * (t.n_text ? t.max_len : t.n_text_const) * 2 * H * sizeof(bf16));
    {
      GemmArgs g = linear(c->ta.p, H, L.w_out, H, rows, H, L.b_out, c->tb.p, H);
      g.residual = c->tx.p; g.ldr = H;
      TRY(gemm(c, g, s));
    }
    if (!fused) TRY(ln(c, c->tb.p, rows, H, L.lna_g, L.lna_b, k.bert_ln_eps, c->tc.p, s));
    {
      GemmArgs g = linear(fused ? c->tb.p : c->tc.p, H, L.w_fc1, H, rows, k.ffn, L.b_fc1, c->tf.p, k.ffn);
      g.act = ACT_GELU_ERF;
      if (fused) {
        g.lnl_gamma = L.lna_g; g.lnl_beta = L.lna_b; g.lnl_eps = k.bert_ln_eps; g.lnl_out = c->tc.p; g.lnl_ldo = H;
      }
      TRY(gemm(c, g, s));
    }
    {
      GemmArgs g = linear(c->tf.p, k.ffn, L.w_fc2, k.ffn, rows, H, L.b_fc2, c->tb.p, H);
      g.residual = c->tc.p; g.ldr = H;
      TRY(gemm(c, g, s));
    }
    if (!fused) {
      TRY(ln(c, c->tb.p, rows, H, L.lno_g, L.lno_b, k.bert_ln_eps, c->tx.p, s));
      TRY(emit_hidden(l + 1));
    }
  }
  {
    GemmArgs g = linear(fused ? c->tb.p : c->tx.p, H, c->w_vocab, H, rows, c->vocab_pad, c->b_vocab, nullptr, 0);
    g.out_f32 = t.logits; g.ldo32 = c->vocab_pad;
    if (fused) {  // the last layer's output LayerNorm runs inside the vocabulary head
      const DecLayer& L = c->dec[k.dec_layers - 1];
      g.lnl_gamma = L.lno_g; g.lnl_beta = L.lno_b; g.lnl_eps = k.bert_ln_eps; g.lnl_out = nullptr;
    }
    TRY(gemm(c, g, s));
  }
  return 0;
}

bool graph_stream_ok(cudaStream_t s) { return s != nullptr && s != cudaStreamLegacy && s != cudaStreamPerThread; }

// Runs `body` (a sequence of launches on stream s).  First occurrence of `key`: eager.  Second: captured into a graph,
// instantiated and launched.  Later: replayed.  Any capture failure disables graphs for this context (eager for good).
template <class Body>
int run_graphed(gitb200_ctx* c, const gitb200_ctx::GraphKey& key, cudaStream_t s, bool eligible, Body&& body) {
  if (!eligible || !c->graphs_enabled || !c->tap_layers.empty() || !graph_stream_ok(s) || gemm_profile_enabled()) return body();
  {  // inside somebody else's capture (the whole-call graph of the latency mode): just contribute the launches
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    if (cudaStreamIsCapturing(s, &cs) != cudaSuccess || cs != cudaStreamCaptureStatusNone) {
      cudaGetLastError();
      return body();
    }
  }
  // drop every graph captured before the last workspace reallocation / launch-sequence switch
  for (size_t i = 0; i < c->graphs.size();) {
    if (c->graphs[i].gen != c->ws_gen) {
      if (c->graphs[i].exec) cudaGraphExecDestroy(c->graphs[i].exec);
      c->graphs.erase(c->graphs.begin() + i);
    } else {
      ++i;
    }
  }
  gitb200_ctx::GraphEntry* ent = nullptr;
  for (auto& g : c->graphs)
    if (g.key == key) ent = &g;
  if (ent && ent->exec) {
    CUDA_OK(c, cudaGraphLaunch(ent->exec, s));
    c->graph_launches++;
    return 1;  // replayed: the caller restores whatever host-side state `body` would have left
  }
  if (!ent) {
    if (c->graphs.size() >= 64) {
      for (auto& g : c->graphs)
        if (g.exec) cudaGraphExecDestroy(g.exec);
      c->graphs.clear();
    }
    gitb200_ctx::GraphEntry e;
    e.key = key;
    const int r = body();  // every workspace gets sized by this eager run
    e.gen = c->ws_gen;     // (read after the run: its own first-time allocations do not count against it)
    c->graphs.push_back(e);
    return r;
  }
  cudaGraph_t graph = nullptr;
  const unsigned long long gen0 = c->ws_gen;
  if (cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal) == cudaSuccess) {
    const int r = body();
    const cudaError_t e = cudaStreamEndCapture(s, &graph);
    if (c->ws_gen != gen0) {
      // a workspace moved while capturing (cannot happen after the sizing run, but never keep such a graph): run eagerly
      if (graph) cudaGraphDestroy(graph);
      cudaGetLastError();
      ent->gen = c->ws_gen;
      return body();
    }
    if (r == 0 && e == cudaSuccess && graph && cudaGraphInstantiate(&ent->exec, graph, 0) == cudaSuccess) {
      cudaGraphDestroy(graph);
      CUDA_OK(c, cudaGraphLaunch(ent->exec, s));
      c->graph_launches++;
      return 0;
    }
    if (graph) cudaGraphDestroy(graph);
  }
  cudaGetLastError();
  ent->exec = nullptr;
  c->graphs_enabled = false;
  return body();
}


int make_search_state(gitb200_ctx* c, int n_clips, int V, int ldl, int sos_unused, int eos, const gitb200_search_params& sp,
                      SearchState* st) {
  (void)sos_unused;
  const int nb = sp.beam_size, rows = n_clips * nb, ml = sp.max_steps, nk = sp.num_keep_best;
  if (nb < 1 || nb > 8 || sp.per_node_beam_size < 1 || nb * sp.per_node_beam_size > 16 || nk < 1 || nk > 15 || ml < 2)
    return fail(c, GITB200_ERR_INVALID, "unsupported search parameters (beam %d, per-node %d, keep %d, max_steps %d)", nb,
                sp.per_node_beam_size, nk, ml);
  const int cand = nb * sp.per_node_beam_size;
  const size_t n_int = (size_t)rows * ml * 4 + (size_t)n_clips * 2 + 1 + rows + (size_t)n_clips * (nk + 1) * (1 + ml) + (size_t)rows * cand;
  ENSURE(c, c->ibuf, n_int);
  ENSURE(c, c->dbuf, (size_t)n_clips * (nk + 2));
  ENSURE(c, c->fbuf, (size_t)rows * (1 + cand));
  int* ip = c->ibuf.p;
  st->n_clips = n_clips; st->nb = nb; st->cand = nb * sp.per_node_beam_size; st->V = V; st->ldl = ldl; st->max_len = ml;
  st->eos = eos; st->n_keep = nk; st->length_penalty = sp.length_penalty; st->reorder_cache = sp.reorder_cache;
  st->tokens = ip; ip += (size_t)rows * ml;
  st->tokens_tmp = ip; ip += (size_t)rows * ml;
  st->anc = ip; ip += (size_t)rows * ml;
  st->anc_tmp = ip; ip += (size_t)rows * ml;
  st->done = ip; ip += n_clips;
  st->hyp_count = ip; ip += n_clips;
  st->done_count = ip; ip += 1;
  st->cur_tok = ip; ip += rows;
  st->hyp_len = ip; ip += (size_t)n_clips * (nk + 1);
  st->hyp_tok = ip; ip += (size_t)n_clips * (nk + 1) * ml;
  st->row_cand_idx = ip;
  st->row_cand_score = c->fbuf.p + rows;
  st->hyp_score = c->dbuf.p;
  st->worst = c->dbuf.p + (size_t)n_clips * (nk + 1);
  st->beam_scores = c->fbuf.p;
  return 0;
}

int run_decode(gitb200_ctx* c, const gitb200_search_params& sp, int32_t* tokens_out, float* logprobs_out, float* logits_out,
               cudaStream_t s) {
  const gitb200_config& k = c->cfg;
  const int B = c->cur_clips, nb = sp.beam_size, rows = B * nb;
  if (sp.max_steps > k.max_positions) return fail(c, GITB200_ERR_INVALID, "max_steps %d exceeds the %d text positions", sp.max_steps, k.max_positions);
  SearchState st;
  TRY(make_search_state(c, B, k.vocab, c->vocab_pad, k.sos, k.eos, sp, &st));
  if (!c->visual_pass_done) TRY(run_visual_pass(c, false, nullptr, 0, s));
  TRY(ensure_text(c, rows, rows, sp.max_steps));
  if (!logits_out) ENSURE(c, c->logits, (size_t)rows * c->vocab_pad);
  // Latency mode: ONE clip (rows = its beams <= 4).  The whole step loop -- embedding, decoder layers, vocabulary head and
  // search step of every step -- runs as one persistent cooperative kernel whose phases are separated by grid barriers
  // instead of kernel boundaries (decode_mega.cu; bit-identical to the launch sequence below, which remains the path for
  // everything else and for devices that cannot keep the grid resident).  It leaves its loop itself once the clip is done.
  if (c->persistent_decode && B == 1 && rows <= 4 && logits_out == nullptr && k.hidden == 768 && k.dec_layers <= MEGA_MAX_LAYERS &&
      !gemm_profile_enabled()) {
    MegaArgs m;
    memset(&m, 0, sizeof(m));
    m.n_layers = k.dec_layers; m.rows = rows; m.hidden = k.hidden; m.heads = k.dec_heads; m.ffn = k.ffn; m.Nv = c->cur_nv;
    decode_mega_attention_geometry(rows, k.dec_heads, c->cur_nv, sp.max_steps, &m.splits, &m.kcap);
    m.vocab_pad = c->vocab_pad; m.steps = sp.max_steps - 1;
    m.words = c->words_f32; m.pos_table = c->pos_f32; m.lne_g = c->lne_g; m.lne_b = c->lne_b;
    m.embed_eps = k.embed_ln_eps; m.ln_eps = k.bert_ln_eps;
    m.scale_log2 = (1.0f / sqrtf((float)(k.hidden / k.dec_heads))) * 1.4426950408889634f;
    m.w_vocab = c->w_vocab; m.b_vocab = c->b_vocab;
    m.logits = c->logits.p; m.logits_step_stride = 0;
    m.st = st;
    if (decode_mega_supported(m)) {
      if (m.splits > 1) ENSURE(c, c->partial, text_attention_workspace_floats(rows, k.dec_heads, m.splits));
      ENSURE(c, c->mega_bar, 32 + 2 * 128);  // [0]: barrier counter; [32, 160): candidate scores; [160, 288): candidate ids
      for (int l = 0; l < k.dec_layers; ++l) {
        const DecLayer& L = c->dec[l];
        MegaLayer& ml = m.layer[l];
        ml.w_qkv = L.w_qkv; ml.w_out = L.w_out; ml.w_fc1 = L.w_fc1; ml.w_fc2 = L.w_fc2;
        ml.b_qkv = L.b_qkv; ml.b_out = L.b_out; ml.b_fc1 = L.b_fc1; ml.b_fc2 = L.b_fc2;
        ml.lna_g = L.lna_g; ml.lna_b = L.lna_b; ml.lno_g = L.lno_g; ml.lno_b = L.lno_b;
        ml.vis_kv = c->kv[l].p; ml.txt_kv = c->txt_kv[l].p;
      }
      m.trace = c->mega_trace_on ? c->mega_trace.p : nullptr;
      m.tq = c->tq.p; m.ta = c->ta.p; m.tb = c->tb.p; m.tf = c->tf.p; m.partial = c->partial.p; m.barrier = c->mega_bar.p; m.attn_cnt = reinterpret_cast<int*>(c->mega_bar.p + 8);
      m.cand_score = reinterpret_cast<float*>(c->mega_bar.p + 32); m.cand_idx = reinterpret_cast<int*>(c->mega_bar.p + 160);
      CUDA_OK(c, search_init(st, k.sos, s));
      const cudaError_t e = decode_mega(m, s);
      if (e == cudaSuccess) {
        c->last_decode_steps = sp.max_steps - 1;
        CUDA_OK(c, search_finalize(st, tokens_out, logprobs_out, s));
        return 0;
      }
      if (e != cudaErrorNotSupported) CUDA_OK(c, e);
      cudaGetLastError();
    }
  }
  // model.py:640 `if all(done): break`: every `early_exit_every` steps the host reads the device's count of finished clips
  // (4 bytes, one stream synchronisation) and stops enqueueing decode steps once every clip is done.  Finished clips no
  // longer change, so the result is the same as running all steps; skipped while the stream is being captured into a graph.
  bool poll_done = c->early_exit_every > 0;
  if (poll_done) {
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    if (cudaStreamIsCapturing(s, &cs) != cudaSuccess || cs != cudaStreamCaptureStatusNone) poll_done = false;
    cudaGetLastError();
    if (poll_done && !c->h_done) CUDA_OK(c, cudaMallocHost(&c->h_done, sizeof(int)));
  }
  c->last_decode_steps = 0;
  const int steps = sp.max_steps - 1;  // model.py:518: while cur_len < max_length, cur_len = t + 1
  // The loop runs in segments of `early_exit_every` steps (all steps when polling is off).  A segment touches only
  // context-owned buffers, so it is captured into a CUDA graph on its second occurrence and replayed from then on; the
  // poll of the finished-clip count sits between segments.  Saved logits go to a caller buffer: its address is part of the
  // graph key (a caller that hands in the same buffer again -- torch's caching allocator does -- replays; another buffer is
  // another graph, and the cache is bounded).
  const int seg = (poll_done && c->early_exit_every < steps) ? c->early_exit_every : steps;
  const bool graphable = c->graph_segments && B > c->graph_max_clips;
  for (int t0 = 0; t0 < steps; t0 += seg) {
    const int n = steps - t0 < seg ? steps - t0 : seg;
    gitb200_ctx::GraphKey key;
    key.kind = 5; key.i0 = B; key.i1 = t0; key.i2 = n; key.i3 = c->cur_nv; key.sp = sp; key.p0 = logits_out;
    const int r = run_graphed(c, key, s, graphable, [&]() -> int {
      if (t0 == 0) CUDA_OK(c, search_init(st, k.sos, s));
      for (int t = t0; t < t0 + n; ++t) {
        const int parity = t & 1;
        TextPass tp;
        tp.n_clips = B; tp.rows_per_clip = nb; tp.max_len = sp.max_steps;
        tp.tokens = st.cur_tok; tp.positions = nullptr; tp.pos_const = t;
        tp.n_text = nullptr; tp.n_text_const = t + 1;
        tp.anc = sp.reorder_cache ? (parity ? st.anc_tmp : st.anc) : nullptr;
        tp.slot_div = 1; tp.n_slots = rows; tp.slot_is_clip = 0;
        tp.logits = logits_out ? logits_out + (size_t)t * rows * c->vocab_pad : c->logits.p;
        tp.hidden_out = nullptr;
        TRY(run_text_pass(c, tp, s));
        CUDA_OK(c, search_step(st, tp.logits, t + 1, parity, s));
      }
      return 0;
    });
    if (r != 0 && r != 1) return r;
    c->last_decode_steps = t0 + n;
    if (poll_done && t0 + n < steps) {
      CUDA_OK(c, cudaMemcpyAsync(c->h_done, st.done_count, sizeof(int), cudaMemcpyDeviceToHost, s));
      CUDA_OK(c, cudaStreamSynchronize(s));
      if (*c->h_done >= B) break;
    }
  }
  CUDA_OK(c, search_finalize(st, tokens_out, logprobs_out, s));
  return 0;
}

void free_workspaces(gitb200_ctx* c) {
  auto fr = [](auto& b) { if (b.p) cudaFree(b.p); b.p = nullptr; b.cap = 0; };
  fr(c->patches); fr(c->x); fr(c->lnb); fr(c->qkv); fr(c->attn); fr(c->mlp); fr(c->vf); fr(c->hv); fr(c->hvb); fr(c->hvc);
  fr(c->vattn); fr(c->vmlp);
  for (auto& b : c->kv) fr(b);
  for (auto& b : c->txt_kv) fr(b);
  fr(c->tx); fr(c->tq); fr(c->ta); fr(c->tb); fr(c->tc); fr(c->tf); fr(c->logits); fr(c->partial); fr(c->vf_in_f32);
  fr(c->ibuf); fr(c->dbuf); fr(c->fbuf); fr(c->pos_arr); fr(c->ntext_arr); fr(c->tok_arr); fr(c->stage[0]); fr(c->stage[1]); fr(c->stage_u8[0]); fr(c->stage_u8[1]);
  fr(c->out_tok); fr(c->out_lp); fr(c->stats_a); fr(c->stats_b); fr(c->ring);
  fr(c->pool); fr(c->pool_rows); fr(c->pool_oldest);
}

// second workspace set that shares this context's (read-only) weights
gitb200_ctx* make_twin(gitb200_ctx* c) {
  gitb200_ctx* t = new gitb200_ctx();
  t->cfg = c->cfg; t->device = c->device; t->finalized = true; t->is_twin = true; t->graphs_enabled = false; t->pipeline_chunk = 0;
  t->fold_ln = c->fold_ln; t->fuse_ln = c->fuse_ln; t->sweep_rows = c->sweep_rows;
  t->T = c->T; t->kpad = c->kpad; t->vocab_pad = c->vocab_pad; t->n_temporal = c->n_temporal;
  t->w_patch = c->w_patch; t->pos_bf16 = c->pos_bf16; t->cls = c->cls; t->ln_pre_g = c->ln_pre_g; t->ln_pre_b = c->ln_pre_b;
  t->ln_post_g = c->ln_post_g; t->ln_post_b = c->ln_post_b; t->temporal = c->temporal; t->vit = c->vit;
  t->w_proj = c->w_proj; t->b_proj = c->b_proj; t->lnp_g = c->lnp_g; t->lnp_b = c->lnp_b;
  t->words_f32 = c->words_f32; t->pos_f32 = c->pos_f32; t->lne_g = c->lne_g; t->lne_b = c->lne_b; t->dec = c->dec;
  t->w_vocab = c->w_vocab; t->b_vocab = c->b_vocab;
  return t;
}

int ensure_pipeline(gitb200_ctx* c) {
  if (!c->twin) c->twin = make_twin(c);
  if (!c->pipe_stream[0]) {
    for (int i = 0; i < 2; ++i) {
      CUDA_OK(c, cudaStreamCreateWithFlags(&c->pipe_stream[i], cudaStreamNonBlocking));
      CUDA_OK(c, cudaEventCreateWithFlags(&c->ev_join[i], cudaEventDisableTiming));
    }
    CUDA_OK(c, cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming));
    CUDA_OK(c, cudaEventCreateWithFlags(&c->ev_enc0, cudaEventDisableTiming));
  }
  return 0;
}

int pipeline_chunk_for(const gitb200_ctx* c, int n_clips) {
  if (c->pipeline_chunk == 0 || c->is_twin) return 0;
  int chunk = c->pipeline_chunk > 0 ? c->pipeline_chunk : (n_clips + 3) / 4;
  if (c->pipeline_chunk < 0) {
    if (chunk < 32) chunk = 32;
    if (chunk > 128) chunk = 128;
  }
  return n_clips >= 2 * chunk ? chunk : 0;
}

// Device-resident frames, chunk pipeline on the two internal streams, joined back into `caller`.
int caption_pipelined(gitb200_ctx* c, const float* frames, int n_clips, int n_frames, const gitb200_search_params& sp,
                      int32_t* tokens, float* logprobs, cudaStream_t caller, int chunk) {
  TRY(ensure_pipeline(c));
  const size_t clip_elems = (size_t)n_frames * 3 * c->cfg.resolution * c->cfg.resolution;
  const int per_clip_tok = sp.num_keep_best * sp.max_steps;
  CUDA_OK(c, cudaEventRecord(c->ev_fork, caller));
  for (int i = 0; i < 2; ++i) CUDA_OK(c, cudaStreamWaitEvent(c->pipe_stream[i], c->ev_fork, 0));
  int done = 0;
  for (int i = 0; done < n_clips; ++i) {
    const int w = i & 1;
    gitb200_ctx* cw = w ? c->twin : c;
    cudaStream_t s = c->pipe_stream[w];
    const int nc = (n_clips - done) < chunk ? (n_clips - done) : chunk;
    if (i == 1) CUDA_OK(c, cudaStreamWaitEvent(s, c->ev_enc0, 0));  // one phase behind: its encode meets chunk 0's decode
    int r = run_encode(cw, frames + (size_t)done * clip_elems, nc, n_frames, s);
    if (r == 0 && i == 0) CUDA_OK(c, cudaEventRecord(c->ev_enc0, s));
    if (r == 0) r = run_decode(cw, sp, tokens + (size_t)done * per_clip_tok, logprobs + (size_t)done * sp.num_keep_best, nullptr, s);
    if (r) {
      if (w) c->err = c->twin->err;
      return r;
    }
    done += nc;
  }
  for (int i = 0; i < 2; ++i) {
    CUDA_OK(c, cudaEventRecord(c->ev_join[i], c->pipe_stream[i]));
    CUDA_OK(c, cudaStreamWaitEvent(caller, c->ev_join[i], 0));
  }
  return 0;
}

int effective_frames(const gitb200_ctx* c, int n_frames) {
  const int n = c->cfg.num_image_with_embedding;
  return (n > 0 && n_frames > n) ? n : n_frames;
}

int ensure_host_streams(gitb200_ctx* c) {
  if (!c->copy_stream) {
    CUDA_OK(c, cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking));
    for (int i = 0; i < 2; ++i) {
      CUDA_OK(c, cudaEventCreateWithFlags(&c->ev_copy[i], cudaEventDisableTiming));
      CUDA_OK(c, cudaEventCreateWithFlags(&c->ev_done[i], cudaEventDisableTiming));
    }
  }
  // the legacy default stream would serialise with the copy stream; compute runs on a private one
  if (!c->comp_stream) CUDA_OK(c, cudaStreamCreateWithFlags(&c->comp_stream, cudaStreamNonBlocking));
  if (!c->ev_user) CUDA_OK(c, cudaEventCreateWithFlags(&c->ev_user, cudaEventDisableTiming));
  if (!c->ev_gfork) CUDA_OK(c, cudaEventCreateWithFlags(&c->ev_gfork, cudaEventDisableTiming));
  if (!c->ev_gjoin) CUDA_OK(c, cudaEventCreateWithFlags(&c->ev_gjoin, cudaEventDisableTiming));
  return 0;
}

cudaStream_t caller_stream(gitb200_ctx* c, void* stream) {
  if (c) {
    c->last_stream = (cudaStream_t)stream;
    c->last_stream_valid = true;
  }
  return (cudaStream_t)stream;
}

// The context's private streams wait for whatever this context last enqueued on a caller's stream (see gitb200_ctx::last_stream).
int order_after_caller_work(gitb200_ctx* c) {
  if (!c->last_stream_valid) return 0;
  TRY(ensure_host_streams(c));
  if (cudaEventRecord(c->ev_user, c->last_stream) != cudaSuccess) {
    cudaGetLastError();  // the caller's stream no longer exists: everything it was given has to be complete, the blunt way
    CUDA_OK(c, cudaDeviceSynchronize());
  } else {
    CUDA_OK(c, cudaStreamWaitEvent(c->comp_stream, c->ev_user, 0));
    CUDA_OK(c, cudaStreamWaitEvent(c->copy_stream, c->ev_user, 0));
  }
  c->last_stream_valid = false;
  return 0;
}

// The decoder's pass over the visual tokens of the clips now held in vf (fills the visual K/V cache), graphed for large batches.
int visual_pass_graphed(gitb200_ctx* c, cudaStream_t s) {
  gitb200_ctx::GraphKey key;
  key.kind = 9; key.i0 = c->cur_clips; key.i1 = c->cur_nv;
  const int r = run_graphed(c, key, s, c->graph_segments && c->cur_clips > c->graph_max_clips,
                            [&]() { return run_visual_pass(c, false, nullptr, 0, s); });
  if (r == 1) {  // replayed: host-side state the eager run would have left
    c->visual_pass_done = true;
    c->visual_pass_full = 0;
    return 0;
  }
  return r;
}

// Frames from the HOST (fp32 preprocessed, or raw uint8 BGR): chunks of `chunk_clips` clips are copied on the copy stream into
// two staging buffers and encoded on `comp` as they arrive (the copy of chunk i+1 overlaps the ViT of chunk i; a small first
// chunk keeps the un-overlapped head of the transfer short); then the decoder's visual pass over all clips.  For large
// batches every chunk's encode and the visual pass are CUDA graphs (the staging buffers are context-owned: stable pointers).
int encode_from_host(gitb200_ctx* c, const float* f32_host, const uint8_t* u8_host, int height, int width, int n_clips, int n_frames,
                     int chunk_clips, cudaStream_t comp) {
  const size_t clip_elems = u8_host ? (size_t)n_frames * height * width * 3 : (size_t)n_frames * 3 * c->cfg.resolution * c->cfg.resolution;
  const size_t elem = u8_host ? 1 : sizeof(float);
  for (int i = 0; i < 2; ++i) {
    if (u8_host) ENSURE(c, c->stage_u8[i], (size_t)chunk_clips * clip_elems);
    else ENSURE(c, c->stage[i], (size_t)chunk_clips * clip_elems);
  }
  const bool graphs = c->graph_segments && n_clips > c->graph_max_clips;
  const int F = effective_frames(c, n_frames);
  int done = 0, ch = 0;
  while (done < n_clips) {
    const int b = ch & 1;
    int nc = ch == 0 ? (chunk_clips + 1) / 2 : chunk_clips;
    if (nc > n_clips - done) nc = n_clips - done;
    void* stage = u8_host ? (void*)c->stage_u8[b].p : (void*)c->stage[b].p;
    const void* src = u8_host ? (const void*)(u8_host + (size_t)done * clip_elems) : (const void*)(f32_host + (size_t)done * clip_elems);
    if (ch >= 2) CUDA_OK(c, cudaStreamWaitEvent(c->copy_stream, c->ev_done[b], 0));  // staging buffer free again
    CUDA_OK(c, cudaMemcpyAsync(stage, src, (size_t)nc * clip_elems * elem, cudaMemcpyHostToDevice, c->copy_stream));
    CUDA_OK(c, cudaEventRecord(c->ev_copy[b], c->copy_stream));
    CUDA_OK(c, cudaStreamWaitEvent(comp, c->ev_copy[b], 0));
    gitb200_ctx::GraphKey key;
    key.kind = u8_host ? 8 : 7; key.p0 = stage; key.i0 = nc; key.i1 = done; key.i2 = n_clips; key.i3 = n_frames; key.i4 = height; key.i5 = width;
    const RawFrames raw{c->stage_u8[b].p, height, width};
    const int r = run_graphed(c, key, comp, graphs, [&]() {
      return run_encode(c, u8_host ? nullptr : c->stage[b].p, nc, n_frames, comp, done, n_clips, nullptr, true, u8_host ? &raw : nullptr);
    });
    if (r == 1) {  // replayed: host-side state the eager run would have left
      c->cur_clips = done + nc; c->cur_nv = F * c->T; c->visual_pass_done = false; c->step_rows_per_clip = 0;
    } else if (r != 0) {
      return r;
    }
    CUDA_OK(c, cudaEventRecord(c->ev_done[b], comp));
    done += nc;
    ++ch;
  }
  return visual_pass_graphed(c, comp);
}

}  // namespace

// ==================================================================== C ABI
extern "C" {

const char* gitb200_version(void) { return "gitb200 0.1 (sm_100a: tcgen05/TMEM GEMM + TMA, CUDA 12.9)"; }

long long gitb200_launch_count(int reset) {
  const long long v = g_launches.load();
  if (reset) g_launches = 0;
  return v;
}

void gitb200_profile_gemm(int enable) {
  if (enable) {
    dap_drain();
    g_dap.ms = g_dap.by = 0;
    g_dap.n = 0;
  }
  gemm_profile_enable(enable);
}

void gitb200_profile_decode_attention_read(double* ms, double* bytes, long long* launches) {
  dap_drain();
  if (ms) *ms = g_dap.ms;
  if (bytes) *bytes = g_dap.by;
  if (launches) *launches = g_dap.n;
}
long long gitb200_graph_launches(const gitb200_ctx* c) { return c ? c->graph_launches : 0; }
void gitb200_profile_gemm_read(double* ms, double* flops, long long* launches) {
  double a = 0, b = 0;
  long long n = 0;
  gemm_profile_read(&a, &b, &n);
  if (ms) *ms = a;
  if (flops) *flops = b;
  if (launches) *launches = n;
}

const char* gitb200_last_error(const gitb200_ctx* ctx) { return ctx ? ctx->err.c_str() : g_create_err.c_str(); }

int gitb200_create(const gitb200_config* cfg, int device, gitb200_ctx** out) {
  if (!cfg || !out) return fail(nullptr, GITB200_ERR_INVALID, "null argument");
  *out = nullptr;
  int n_dev = 0;
  cudaError_t e = cudaGetDeviceCount(&n_dev);
  if (e != cudaSuccess || n_dev <= 0)
    return fail(nullptr, GITB200_ERR_CUDA, "no CUDA device available (%s): gitb200 has no CPU fallback", cudaGetErrorString(e));
  if (device < 0 || device >= n_dev) return fail(nullptr, GITB200_ERR_INVALID, "device %d out of range (%d devices)", device, n_dev);
  cudaDeviceProp prop;
  e = cudaGetDeviceProperties(&prop, device);
  if (e != cudaSuccess) return fail(nullptr, GITB200_ERR_CUDA, "cudaGetDeviceProperties: %s", cudaGetErrorString(e));
  if (prop.major != 10)
    return fail(nullptr, GITB200_ERR_CUDA, "device %d is sm_%d%d; gitb200 kernels are built for sm_100a only", device, prop.major, prop.minor);
  if (cfg->vit_width % 256 != 0 || cfg->vit_width / cfg->vit_heads != 64 || cfg->hidden != 768 || cfg->hidden / cfg->dec_heads != 64 ||
      cfg->ffn % 256 != 0 || cfg->resolution % cfg->patch != 0 || cfg->vit_layers < 1 || cfg->dec_layers < 1 ||
      (cfg->vit_width != 768 && cfg->vit_width != 1024))
    return fail(nullptr, GITB200_ERR_INVALID, "unsupported model geometry (need head dim 64, hidden 768, ViT width 768 or 1024)");
  gitb200_ctx* c = new gitb200_ctx();
  c->cfg = *cfg;
  c->device = device;
  const int G = cfg->resolution / cfg->patch;
  c->T = G * G + 1;
  c->kpad = ((3 * cfg->patch * cfg->patch + 63) / 64) * 64;
  c->vocab_pad = ((cfg->vocab + 255) / 256) * 256;
  c->n_temporal = cfg->num_image_with_embedding;
  *out = c;
  return GITB200_OK;
}

void gitb200_destroy(gitb200_ctx* c) {
  if (!c) return;
  cudaSetDevice(c->device);
  cudaDeviceSynchronize();
  for (auto& kv : c->raw) cudaFree(kv.second.p);
  for (void* p : c->weight_allocs) cudaFree(p);
  free_workspaces(c);
  if (c->twin) {
    free_workspaces(c->twin);
    delete c->twin;
  }
  for (int i = 0; i < 2; ++i) {
    if (c->pipe_stream[i]) cudaStreamDestroy(c->pipe_stream[i]);
    if (c->ev_join[i]) cudaEventDestroy(c->ev_join[i]);
  }
  if (c->ev_fork) cudaEventDestroy(c->ev_fork);
  if (c->ev_enc0) cudaEventDestroy(c->ev_enc0);
  for (auto& g : c->graphs)
    if (g.exec) cudaGraphExecDestroy(g.exec);
  if (c->h_done) cudaFreeHost(c->h_done);
  if (c->ev_user) cudaEventDestroy(c->ev_user);
  if (c->ev_gfork) cudaEventDestroy(c->ev_gfork);
  if (c->ev_gjoin) cudaEventDestroy(c->ev_gjoin);
  if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
  if (c->comp_stream) cudaStreamDestroy(c->comp_stream);
  for (int i = 0; i < 2; ++i) {
    if (c->ev_copy[i]) cudaEventDestroy(c->ev_copy[i]);
    if (c->ev_done[i]) cudaEventDestroy(c->ev_done[i]);
  }
  delete c;
}

int gitb200_load_weight(gitb200_ctx* c, const char* name, const float* data, int ndim, const int64_t* shape) {
  if (!c || !name || !data || ndim < 0 || ndim > 8) return fail(c, GITB200_ERR_INVALID, "bad load_weight argument");
  if (c->finalized) return fail(c, GITB200_ERR_STATE, "weights already finalised");
  CUDA_OK(c, cudaSetDevice(c->device));
  DevF32 w;
  for (int i = 0; i < ndim; ++i) w.shape.push_back(shape[i]);
  const size_t n = w.numel();
  if (n == 0) return fail(c, GITB200_ERR_INVALID, "empty weight %s", name);
  auto it = c->raw.find(name);
  if (it != c->raw.end()) {
    cudaFree(it->second.p);
    c->raw.erase(it);
  }
  CUDA_OK(c, cudaMalloc(&w.p, n * sizeof(float)));
  CUDA_OK(c, cudaMemcpy(w.p, data, n * sizeof(float), cudaMemcpyDefault));
  c->raw[name] = w;
  return GITB200_OK;
}

int gitb200_finalize_weights(gitb200_ctx* c) {
  if (!c) return GITB200_ERR_INVALID;
  if (c->finalized) return GITB200_OK;
  CUDA_OK(c, cudaSetDevice(c->device));
  const gitb200_config& k = c->cfg;
  const int W = k.vit_width, H = k.hidden, P = k.patch, T = c->T;
  const std::string ie = "image_encoder.";
  TRY(to_bf16(c, ie + "conv1.weight", W, 3 * P * P, W, c->kpad, &c->w_patch));
  TRY(to_f32(c, ie + "class_embedding", W, W, &c->cls));
  TRY(to_bf16(c, ie + "positional_embedding", T, W, T, W, &c->pos_bf16));
  TRY(to_f32(c, ie + "ln_pre.weight", W, W, &c->ln_pre_g));
  TRY(to_f32(c, ie + "ln_pre.bias", W, W, &c->ln_pre_b));
  TRY(to_f32(c, ie + "ln_post.weight", W, W, &c->ln_post_g));
  TRY(to_f32(c, ie + "ln_post.bias", W, W, &c->ln_post_b));
  c->vit.resize(k.vit_layers);
  for (int l = 0; l < k.vit_layers; ++l) {
    const std::string b = ie + "transformer.resblocks." + std::to_string(l) + ".";
    VitLayer& L = c->vit[l];
    TRY(to_f32(c, b + "ln_1.weight", W, W, &L.ln1_g));
    TRY(to_f32(c, b + "ln_1.bias", W, W, &L.ln1_b));
    TRY(to_bf16(c, b + "attn.in_proj_weight", 3 * W, W, 3 * W, W, &L.w_qkv));
    TRY(to_f32(c, b + "attn.in_proj_bias", 3 * W, 3 * W, &L.b_qkv));
    TRY(to_bf16(c, b + "attn.out_proj.weight", W, W, W, W, &L.w_out));
    TRY(to_f32(c, b + "attn.out_proj.bias", W, W, &L.b_out));
    TRY(to_f32(c, b + "ln_2.weight", W, W, &L.ln2_g));
    TRY(to_f32(c, b + "ln_2.bias", W, W, &L.ln2_b));
    TRY(to_bf16(c, b + "mlp.c_fc.weight", 4 * W, W, 4 * W, W, &L.w_fc1));
    TRY(to_f32(c, b + "mlp.c_fc.bias", 4 * W, 4 * W, &L.b_fc1));
    TRY(to_bf16(c, b + "mlp.c_proj.weight", W, 4 * W, W, 4 * W, &L.w_fc2));
    TRY(to_f32(c, b + "mlp.c_proj.bias", W, W, &L.b_fc2));
    TRY(walloc(c, &L.wf_qkv, (size_t)3 * W * W));
    TRY(walloc(c, &L.bf_qkv, (size_t)3 * W));
    TRY(walloc(c, &L.cs_qkv, (size_t)3 * W));
    TRY(walloc(c, &L.wf_fc1, (size_t)4 * W * W));
    TRY(walloc(c, &L.bf_fc1, (size_t)4 * W));
    TRY(walloc(c, &L.cs_fc1, (size_t)4 * W));
    CUDA_OK(c, ln_fold_weight(find(c, b + "attn.in_proj_weight")->p, 3 * W, W, L.ln1_g, L.ln1_b, L.b_qkv, L.wf_qkv, L.cs_qkv, L.bf_qkv, 0));
    CUDA_OK(c, ln_fold_weight(find(c, b + "mlp.c_fc.weight")->p, 4 * W, W, L.ln2_g, L.ln2_b, L.b_fc1, L.wf_fc1, L.cs_fc1, L.bf_fc1, 0));
  }
  if (c->n_temporal > 0) {
    TRY(walloc(c, &c->temporal, (size_t)c->n_temporal * W));
    for (int i = 0; i < c->n_temporal; ++i) {
      const DevF32* w = find(c, "img_temperal_embedding." + std::to_string(i));
      if (!w) return fail(c, GITB200_ERR_MISSING, "missing weight img_temperal_embedding.%d", i);
      if (w->numel() != (size_t)W) return fail(c, GITB200_ERR_INVALID, "img_temperal_embedding.%d has %zu elements", i, w->numel());
      CUDA_OK(c, cudaMemcpy(c->temporal + (size_t)i * W, w->p, W * sizeof(float), cudaMemcpyDeviceToDevice));
    }
  }
  const std::string tx = "textual.";
  TRY(to_bf16(c, tx + "visual_projection.0.weight", H, W, H, W, &c->w_proj));
  TRY(to_f32(c, tx + "visual_projection.0.bias", H, H, &c->b_proj));
  TRY(to_f32(c, tx + "visual_projection.1.weight", H, H, &c->lnp_g));
  TRY(to_f32(c, tx + "visual_projection.1.bias", H, H, &c->lnp_b));
  TRY(to_f32(c, tx + "embedding.words.weight", (size_t)k.vocab * H, (size_t)k.vocab * H, &c->words_f32));
  TRY(to_f32(c, tx + "embedding.positions.weight", (size_t)k.max_positions * H, (size_t)k.max_positions * H, &c->pos_f32));
  TRY(to_f32(c, tx + "embedding.layer_norm.weight", H, H, &c->lne_g));
  TRY(to_f32(c, tx + "embedding.layer_norm.bias", H, H, &c->lne_b));
  c->dec.resize(k.dec_layers);
  for (int l = 0; l < k.dec_layers; ++l) {
    const std::string b = tx + "transformer.encoder.layer." + std::to_string(l) + ".";
    DecLayer& L = c->dec[l];
    // fused q|k|v projection
    TRY(walloc(c, &L.w_qkv, (size_t)3 * H * H));
    TRY(walloc(c, &L.b_qkv, (size_t)3 * H));
    const char* names[3] = {"query", "key", "value"};
    for (int j = 0; j < 3; ++j) {
      const DevF32* w = find(c, b + "attention.self." + names[j] + ".weight");
      const DevF32* bi = find(c, b + "attention.self." + names[j] + ".bias");
      if (!w || !bi) return fail(c, GITB200_ERR_MISSING, "missing weight %sattention.self.%s.*", b.c_str(), names[j]);
      if (w->numel() != (size_t)H * H || bi->numel() != (size_t)H) return fail(c, GITB200_ERR_INVALID, "bad shape for %sattention.self.%s", b.c_str(), names[j]);
      CUDA_OK(c, cast_f32_to_bf16(w->p, H, H, H, L.w_qkv + (size_t)j * H * H, H, H, H, 0));
      CUDA_OK(c, cudaMemcpy(L.b_qkv + (size_t)j * H, bi->p, H * sizeof(float), cudaMemcpyDeviceToDevice));
    }
    TRY(to_bf16(c, b + "attention.output.dense.weight", H, H, H, H, &L.w_out));
    TRY(to_f32(c, b + "attention.output.dense.bias", H, H, &L.b_out));
    TRY(to_f32(c, b + "attention.output.LayerNorm.weight", H, H, &L.lna_g));
    TRY(to_f32(c, b + "attention.output.LayerNorm.bias", H, H, &L.lna_b));
    TRY(to_bf16(c, b + "intermediate.dense.weight", k.ffn, H, k.ffn, H, &L.w_fc1));
    TRY(to_f32(c, b + "intermediate.dense.bias", k.ffn, k.ffn, &L.b_fc1));
    TRY(to_bf16(c, b + "output.dense.weight", H, k.ffn, H, k.ffn, &L.w_fc2));
    TRY(to_f32(c, b + "output.dense.bias", H, H, &L.b_fc2));
    TRY(to_f32(c, b + "output.LayerNorm.weight", H, H, &L.lno_g));
    TRY(to_f32(c, b + "output.LayerNorm.bias", H, H, &L.lno_b));
  }
  // vocabulary head: upstream ties output.weight to embedding.words.weight; accept either
  const std::string ow = find(c, tx + "output.weight") ? tx + "output.weight" : tx + "embedding.words.weight";
  TRY(to_bf16(c, ow, k.vocab, H, c->vocab_pad, H, &c->w_vocab));
  if (find(c, tx + "output.bias")) {
    TRY(to_f32(c, tx + "output.bias", k.vocab, c->vocab_pad, &c->b_vocab));
  } else {
    TRY(walloc(c, &c->b_vocab, (size_t)c->vocab_pad));
    CUDA_OK(c, cudaMemset(c->b_vocab, 0, c->vocab_pad * sizeof(float)));
  }
  CUDA_OK(c, cudaDeviceSynchronize());
  for (auto& kv : c->raw) cudaFree(kv.second.p);
  c->raw.clear();
  c->finalized = true;
  return GITB200_OK;
}

int gitb200_tokens_per_frame(const gitb200_ctx* c) { return c ? c->T : 0; }
int gitb200_logits_ld(const gitb200_ctx* c) { return c ? c->vocab_pad : 0; }

int gitb200_reserve(gitb200_ctx* c, int max_clips, int max_frames, int max_rows_per_clip, int max_text_len) {
  if (!c || max_clips < 1 || max_frames < 1 || max_rows_per_clip < 1 || max_text_len < 1) return fail(c, GITB200_ERR_INVALID, "bad reserve argument");
  CUDA_OK(c, cudaSetDevice(c->device));
  const gitb200_config& k = c->cfg;
  const int F = (k.num_image_with_embedding > 0 && max_frames > k.num_image_with_embedding) ? k.num_image_with_embedding : max_frames;
  const int W = k.vit_width, H = k.hidden, G = k.resolution / k.patch;
  const size_t rows = (size_t)max_clips * F * c->T;
  // row-sized scratch is needed for one sub-batch of the sweeps only (gitb200_ctx::sweep_rows); the visual features and
  // the visual K/V cache are per clip and stay whole
  const int sub_clips = sweep_clips(c->sweep_rows, F * c->T, max_clips);
  const size_t srows = (size_t)sub_clips * F * c->T;
  ENSURE(c, c->patches, (size_t)sub_clips * F * G * G * c->kpad);
  ENSURE(c, c->x, srows * W);
  ENSURE(c, c->lnb, srows * W);
  ENSURE(c, c->qkv, srows * 3 * W);
  ENSURE(c, c->attn, srows * W);
  ENSURE(c, c->mlp, srows * 4 * W);
  ENSURE(c, c->vf, rows * W);
  ENSURE(c, c->hv, srows * H);
  ENSURE(c, c->hvb, srows * H);
  ENSURE(c, c->hvc, srows * H);
  ENSURE(c, c->vattn, srows * H);
  ENSURE(c, c->vmlp, srows * k.ffn);
  c->kv.resize(k.dec_layers);
  for (int l = 0; l < k.dec_layers; ++l) ENSURE(c, c->kv[l], rows * 3 * H);
  const int trows = max_clips * max_rows_per_clip;
  TRY(ensure_text(c, trows, trows, max_text_len));
  ENSURE(c, c->logits, (size_t)trows * c->vocab_pad);
  return GITB200_OK;
}

// run_encode over `n_clips` clips in sub-batches of ~sweep_rows token rows (see gitb200_ctx::sweep_rows); every sub-batch
// writes its slice of the visual features (or, with frame_out / out_rows, its frames' rows), so the result is the one
// sweep's, bit for bit.  raw != nullptr: raw uint8 frames instead of `frames` (see run_encode).
static int run_encode_sweeps(gitb200_ctx* c, const float* frames, int n_clips, int n_frames, cudaStream_t s, bool temporal = true,
                             bf16* frame_out = nullptr, const int* out_rows = nullptr, const RawFrames* raw = nullptr) {
  const gitb200_config& k = c->cfg;
  const int F = (temporal && k.num_image_with_embedding > 0 && n_frames > k.num_image_with_embedding) ? k.num_image_with_embedding : n_frames;
  const int sub = sweep_clips(c->sweep_rows, F * c->T, n_clips);
  if (sub >= n_clips) return run_encode(c, frames, n_clips, n_frames, s, 0, 0, frame_out, temporal, raw, out_rows);
  const size_t clip_elems = (size_t)n_frames * 3 * k.resolution * k.resolution;
  for (int done = 0; done < n_clips; done += sub) {
    const int nc = (n_clips - done) < sub ? (n_clips - done) : sub;
    RawFrames part{};
    if (raw) part = RawFrames{raw->p + (size_t)done * n_frames * raw->height * raw->width * 3, raw->height, raw->width};
    TRY(run_encode(c, frames ? frames + (size_t)done * clip_elems : nullptr, nc, n_frames, s, done, n_clips, frame_out, temporal,
                   raw ? &part : nullptr, out_rows ? out_rows + (size_t)done * F : nullptr));
  }
  return 0;
}

int gitb200_set_sweep_rows(gitb200_ctx* c, int rows) {
  if (!c || rows < 0) return fail(c, GITB200_ERR_INVALID, "gitb200_set_sweep_rows: rows must be >= 0");
  if (c->sweep_rows != rows) c->ws_gen++;  // captured graphs replay the old sub-batch walk
  c->sweep_rows = rows;
  if (c->twin) c->twin->sweep_rows = rows;
  return GITB200_OK;
}

int gitb200_encode(gitb200_ctx* c, const float* frames, int n_clips, int n_frames, float* vf_out, void* stream) {
  if (!c || !frames || n_clips < 1 || n_frames < 1) return fail(c, GITB200_ERR_INVALID, "bad encode argument");
  if (!c->finalized) return fail(c, GITB200_ERR_STATE, "call gitb200_finalize_weights first");
  CUDA_OK(c, cudaSetDevice(c->device));
  cudaStream_t s = caller_stream(c, stream);
  TRY(run_encode_sweeps(c, frames, n_clips, n_frames, s));
  if (vf_out) CUDA_OK(c, cast_bf16_to_f32(c->vf.p, n_clips * c->cur_nv, c->cfg.vit_width, c->cfg.vit_width, vf_out, c->cfg.vit_width, s));
  return GITB200_OK;
}

int gitb200_encode_images(gitb200_ctx* c, const float* images, int n_images, float* vf_out, void* stream) {
  if (!c || !images || n_images < 1) return fail(c, GITB200_ERR_INVALID, "bad encode_images argument");
  if (!c->finalized) return fail(c, GITB200_ERR_STATE, "call gitb200_finalize_weights first");
  CUDA_OK(c, cudaSetDevice(c->device));
  cudaStream_t s = caller_stream(c, stream);
  TRY(run_encode_sweeps(c, images, n_images, 1, s, /*temporal=*/false));
  if (vf_out) CUDA_OK(c, cast_bf16_to_f32(c->vf.p, n_images * c->cur_nv, c->cfg.vit_width, c->cfg.vit_width, vf_out, c->cfg.vit_width, s));
  return GITB200_OK;
}

int gitb200_set_vit_taps(gitb200_ctx* c, const int32_t* layers_host, int n_layers, float* out_dev) {
  if (!c) return GITB200_ERR_INVALID;
  if (n_layers < 0 || (n_layers > 0 && (layers_host == nullptr || out_dev == nullptr)))
    return fail(c, GITB200_ERR_INVALID, "gitb200_set_vit_taps: bad arguments");
  for (int i = 0; i < n_layers; ++i)
    if (layers_host[i] < 0 || layers_host[i] >= c->cfg.vit_layers)
      return fail(c, GITB200_ERR_INVALID, "gitb200_set_vit_taps: layer %d outside [0, %d)", layers_host[i], c->cfg.vit_layers);
  c->tap_layers.assign(layers_host, layers_host + n_layers);
  c->tap_out = n_layers > 0 ? out_dev : nullptr;
  return 0;
}

int gitb200_set_visual_features(gitb200_ctx* c, const float* vf, int n_clips, int nv, void* stream) {
  if (!c || !vf || n_clips < 1 || nv < 1) return fail(c, GITB200_ERR_INVALID, "bad set_visual_features argument");
  if (!c->finalized) return fail(c, GITB200_ERR_STATE, "call gitb200_finalize_weights first");
  CUDA_OK(c, cudaSetDevice(c->device));
  const int W = c->cfg.vit_width;
  ENSURE(c, c->vf, (size_t)n_clips * nv * W);
  CUDA_OK(c, cast_f32_to_bf16(vf, n_clips * nv, W, W, c->vf.p, W, n_clips * nv, W, caller_stream(c, stream)));
  c->cur_clips = n_clips;
  c->cur_nv = nv;
  c->visual_pass_done = false;
  c->step_rows_per_clip = 0;
  return GITB200_OK;
}

int gitb200_decode(gitb200_ctx* c, const gitb200_search_params* sp, int32_t* tokens, float* logprobs, float* logits, void* stream) {
  if (!c || !sp || !tokens || !logprobs) return fail(c, GITB200_ERR_INVALID, "bad decode argument");
  if (!c->finalized) return fail(c, GITB200_ERR_STATE, "call gitb200_finalize_weights first");
  if (c->cur_clips <= 0) return fail(c, GITB200_ERR_STATE, "no visual features: call gitb200_encode or gitb200_set_visual_features first");
  CUDA_OK(c, cudaSetDevice(c->device));
  return run_decode(c, *sp, tokens, logprobs, logits, caller_stream(c, stream));
}

static int caption_eager(gitb200_ctx* c, const float* frames, int n_clips, int n_frames, const gitb200_search_params* sp,
                         int32_t* tokens, float* logprobs, float* logits, void* stream) {
  int r = gitb200_encode(c, frames, n_clips, n_frames, nullptr, stream);
  if (r) return r;
  return gitb200_decode(c, sp, tokens, logprobs, logits, stream);
}

int gitb200_caption(gitb200_ctx* c, const float* frames, int n_clips, int n_frames, const gitb200_search_params* sp,
                    int32_t* tokens, float* logprobs, float* logits, void* stream) {
  if (!c || !sp) return fail(c, GITB200_ERR_INVALID, "bad caption argument");
  // Latency mode: a small batch is launch-bound (~850 kernels per caption), so the second call with the same
  // buffers / shapes on a capturable stream is recorded into a CUDA graph and later calls replay it.
  cudaStream_t s = caller_stream(c, stream);
  if (n_clips > 0 && n_clips <= c->graph_max_clips && frames && tokens && logprobs && c->finalized) {
    gitb200_ctx::GraphKey key;
    key.kind = 0; key.p0 = frames; key.p1 = tokens; key.p2 = logprobs; key.i0 = n_clips; key.i1 = n_frames;
    key.i2 = logits != nullptr; key.sp = *sp;
    CUDA_OK(c, cudaSetDevice(c->device));
    const int r = run_graphed(c, key, s, logits == nullptr, [&]() { return caption_eager(c, frames, n_clips, n_frames, sp, tokens, logprobs, logits, stream); });
    if (r == 1) {  // replayed: host-side state the eager path would have left behind
      const int F = (c->cfg.num_image_with_embedding > 0 && n_frames > c->cfg.num_image_with_embedding) ? c->cfg.num_image_with_embedding : n_frames;
      c->cur_clips = n_clips; c->cur_nv = F * c->T; c->visual_pass_done = true; c->visual_pass_full = 0; c->step_rows_per_clip = 0;
      c->last_decode_steps = sp->max_steps - 1;
      return GITB200_OK;
    }
    return r;
  }
  if (logits == nullptr && frames && tokens && logprobs && c->finalized && n_clips > 0 && n_frames > 0) {
    const int chunk = pipeline_chunk_for(c, n_clips);
    if (chunk > 0) {
      CUDA_OK(c, cudaSetDevice(c->device));
      return caption_pipelined(c, frames, n_clips, n_frames, *sp, tokens, logprobs, s, chunk);
    }
    if (c->graph_segments && c->graphs_enabled && c->tap_layers.empty() && !gemm_profile_enabled() && n_clips > c->graph_max_clips) {
      // Throughput-sized batch: encode + visual pass replay as one CUDA graph per frame buffer, the decode loop as one graph per
      // segment of steps (run_decode); nothing in them depends on the caller's output pointers.  The legacy default stream
      // cannot be captured: the work then runs on the context's compute stream, forked from / joined back into the caller's.
      CUDA_OK(c, cudaSetDevice(c->device));
      cudaStream_t gs = s;
      const bool forked = !graph_stream_ok(s);
      if (forked) {
        TRY(ensure_host_streams(c));
        gs = c->comp_stream;
        CUDA_OK(c, cudaEventRecord(c->ev_gfork, s));
        CUDA_OK(c, cudaStreamWaitEvent(gs, c->ev_gfork, 0));
      }
      gitb200_ctx::GraphKey key;
      key.kind = 6; key.p0 = frames; key.i0 = n_clips; key.i1 = n_frames;
      const int r = run_graphed(c, key, gs, true, [&]() -> int {
        TRY(run_encode_sweeps(c, frames, n_clips, n_frames, gs));
        return run_visual_pass(c, false, nullptr, 0, gs);
      });
      if (r == 1) {  // replayed: host-side state the eager run would have left
        c->cur_clips = n_clips; c->cur_nv = effective_frames(c, n_frames) * c->T; c->visual_pass_done = true; c->visual_pass_full = 0;
        c->step_rows_per_clip = 0;
      } else if (r != 0) {
        return r;
      }
      TRY(run_decode(c, *sp, tokens, logprobs, nullptr, gs));
      if (forked) {
        CUDA_OK(c, cudaEventRecord(c->ev_gjoin, gs));
        CUDA_OK(c, cudaStreamWaitEvent(s, c->ev_gjoin, 0));
      }
      return GITB200_OK;
    }
  }
  return caption_eager(c, frames, n_clips, n_frames, sp, tokens, logprobs, logits, stream);
}

int gitb200_stream_reset(gitb200_ctx* c) {
  if (!c) return GITB200_ERR_INVALID;
  c->ring_count = 0;
  c->ring_head = 0;
  return GITB200_OK;
}

int gitb200_stream_push(gitb200_ctx* c, const float* frame, void* stream) {
  if (!c || !frame) return fail(c, GITB200_ERR_INVALID, "bad stream_push argument");
  if (!c->finalized) return fail(c, GITB200_ERR_STATE, "call gitb200_finalize_weights first");
  const int cap = c->cfg.num_image_with_embedding;
  if (cap < 1) return fail(c, GITB200_ERR_STATE, "streaming needs num_image_with_embedding >= 1 (the window length)");
  CUDA_OK(c, cudaSetDevice(c->device));
  const size_t per_frame = (size_t)c->T * c->cfg.vit_width;
  ENSURE(c, c->ring, (size_t)cap * per_frame);
  {
    gitb200_ctx::GraphKey key;
    key.kind = 1; key.p0 = frame; key.i0 = c->ring_head;
    bf16* dst = c->ring.p + (size_t)c->ring_head * per_frame;
    const int r = run_graphed(c, key, caller_stream(c, stream), true, [&]() { return run_encode(c, frame, 1, 1, caller_stream(c, stream), 0, 0, dst); });
    if (r != 0 && r != 1) return r;
  }
  c->ring_head = (c->ring_head + 1) % cap;
  if (c->ring_count < cap) c->ring_count++;
  return GITB200_OK;
}

// The same for a RAW webcam frame (uint8 BGR HWC on the device, real_time_inference.py:49-57): image_transform() runs
// fused into the patch-embed loader, so a push is the ViT's own launches and nothing else.
int gitb200_stream_push_u8(gitb200_ctx* c, const uint8_t* frame, int height, int width, void* stream) {
  if (!c || !frame || height < 1 || width < 1) return fail(c, GITB200_ERR_INVALID, "bad stream_push_u8 argument");
  if (!c->finalized) return fail(c, GITB200_ERR_STATE, "call gitb200_finalize_weights first");
  const int cap = c->cfg.num_image_with_embedding;
  if (cap < 1) return fail(c, GITB200_ERR_STATE, "streaming needs num_image_with_embedding >= 1 (the window length)");
  CUDA_OK(c, cudaSetDevice(c->device));
  const size_t per_frame = (size_t)c->T * c->cfg.vit_width;
  ENSURE(c, c->ring, (size_t)cap * per_frame);
  {
    gitb200_ctx::GraphKey key;
    key.kind = 3; key.p0 = frame; key.i0 = c->ring_head; key.i1 = height; key.i2 = width;
    bf16* dst = c->ring.p + (size_t)c->ring_head * per_frame;
    const RawFrames raw{frame, height, width};
    const int r = run_graphed(c, key, caller_stream(c, stream), true,
                              [&]() { return run_encode(c, nullptr, 1, 1, caller_stream(c, stream), 0, 0, dst, true, &raw); });
    if (r != 0 && r != 1) return r;
  }
  c->ring_head = (c->ring_head + 1) % cap;
  if (c->ring_count < cap) c->ring_count++;
  return GITB200_OK;
}

int gitb200_stream_frames(const gitb200_ctx* c) { return c ? c->ring_count : 0; }

int gitb200_stream_caption(gitb200_ctx* c, const gitb200_search_params* sp, int32_t* tokens, float* logprobs, void* stream) {
  if (!c || !sp || !tokens || !logprobs) return fail(c, GITB200_ERR_INVALID, "bad stream_caption argument");
  if (c->ring_count < 1) return fail(c, GITB200_ERR_STATE, "no frames in the streaming window: call gitb200_stream_push first");
  CUDA_OK(c, cudaSetDevice(c->device));
  cudaStream_t s = caller_stream(c, stream);
  const int cap = c->cfg.num_image_with_embedding, n = c->ring_count, T = c->T, W = c->cfg.vit_width;
  ENSURE(c, c->vf, (size_t)n * T * W);
  const int first = (c->ring_head - n + cap) % cap;  // oldest frame -> temporal position 0
  gitb200_ctx::GraphKey key;
  key.kind = 2; key.p0 = tokens; key.p1 = logprobs; key.i0 = n; key.i1 = first; key.sp = *sp;
  const int r = run_graphed(c, key, s, true, [&]() {
    CUDA_OK(c, assemble_window(c->ring.p, first, cap, n, T, W, c->temporal, c->vf.p, s));
    c->cur_clips = 1;
    c->cur_nv = n * T;
    c->visual_pass_done = false;
    c->step_rows_per_clip = 0;
    return run_decode(c, *sp, tokens, logprobs, nullptr, s);
  });
  if (r == 1) {
    c->cur_clips = 1; c->cur_nv = n * T; c->visual_pass_done = true; c->visual_pass_full = 0; c->step_rows_per_clip = 0;
    return GITB200_OK;
  }
  return r;
}

// ---- multi-stream pool: one window per camera stream, pushes and captions batched over streams
// Host-side checks of a stream-id list, before anything is enqueued: the pool exists, k >= 1, every id is known and distinct.
static int pool_check_ids(gitb200_ctx* c, const char* what, const int32_t* ids, int k) {
  if (c->pool_streams < 1) return fail(c, GITB200_ERR_STATE, "%s: no stream pool: call gitb200_streams_configure first", what);
  if (k < 1 || ids == nullptr) return fail(c, GITB200_ERR_INVALID, "%s: need k >= 1 stream ids (k = %d)", what, k);
  std::vector<char> seen((size_t)c->pool_streams, 0);
  for (int j = 0; j < k; ++j) {
    const int id = ids[j];
    if (id < 0 || id >= c->pool_streams)
      return fail(c, GITB200_ERR_INVALID, "%s: unknown stream id %d (the pool has ids 0..%d)", what, id, c->pool_streams - 1);
    if (seen[id]) return fail(c, GITB200_ERR_INVALID, "%s: stream id %d appears twice in one call", what, id);
    seen[id] = 1;
  }
  return 0;
}

// The per-call tables sit at fixed device addresses: a call on another stream than this context's previous call first waits
// for that stream, so that a table (or a window) is not rewritten while the previous call still reads it.
static int pool_order_after_last_stream(gitb200_ctx* c, cudaStream_t s) {
  if (!c->last_stream_valid || c->last_stream == s) return 0;
  if (!c->ev_user) CUDA_OK(c, cudaEventCreateWithFlags(&c->ev_user, cudaEventDisableTiming));
  if (cudaEventRecord(c->ev_user, c->last_stream) != cudaSuccess) {
    cudaGetLastError();  // that stream no longer exists: everything it was given has to be complete
    CUDA_OK(c, cudaDeviceSynchronize());
  } else {
    CUDA_OK(c, cudaStreamWaitEvent(s, c->ev_user, 0));
  }
  return 0;
}

int gitb200_streams_configure(gitb200_ctx* c, int n_streams) {
  if (!c) return GITB200_ERR_INVALID;
  if (n_streams < 1) return fail(c, GITB200_ERR_INVALID, "gitb200_streams_configure: n_streams must be >= 1 (got %d)", n_streams);
  const int cap = c->cfg.num_image_with_embedding;
  if (cap < 1) return fail(c, GITB200_ERR_STATE, "streaming needs num_image_with_embedding >= 1 (the window length)");
  CUDA_OK(c, cudaSetDevice(c->device));
  if (n_streams != c->pool_streams) {
    for (void* p : {(void*)c->pool.p, (void*)c->pool_rows.p, (void*)c->pool_oldest.p})
      if (p) {
        CUDA_OK(c, cudaFree(p));
        c->ws_gen++;  // captured graphs hold the freed pointers
      }
    c->pool = Buf<bf16>{}; c->pool_rows = Buf<int>{}; c->pool_oldest = Buf<int>{};
    c->pool_streams = 0;
    c->pool_head.clear(); c->pool_count.clear();
    ENSURE(c, c->pool, (size_t)n_streams * cap * c->T * c->cfg.vit_width);
    ENSURE(c, c->pool_rows, (size_t)n_streams);
    ENSURE(c, c->pool_oldest, (size_t)n_streams);
    c->pool_streams = n_streams;
  }
  c->pool_head.assign((size_t)n_streams, 0);
  c->pool_count.assign((size_t)n_streams, 0);
  return GITB200_OK;
}

static int streams_push_any(gitb200_ctx* c, const int32_t* ids, int k, const float* frames, const uint8_t* raw, int height, int width,
                            void* stream) {
  const char* what = raw ? "gitb200_streams_push_u8" : "gitb200_streams_push";
  if (!c) return GITB200_ERR_INVALID;
  if (!c->finalized) return fail(c, GITB200_ERR_STATE, "call gitb200_finalize_weights first");
  TRY(pool_check_ids(c, what, ids, k));
  if ((raw == nullptr && frames == nullptr) || (raw != nullptr && (height < 1 || width < 1)))
    return fail(c, GITB200_ERR_INVALID, "%s: bad frame buffer / size", what);
  CUDA_OK(c, cudaSetDevice(c->device));
  const cudaStream_t s = (cudaStream_t)stream;
  TRY(pool_order_after_last_stream(c, s));
  caller_stream(c, stream);
  const int cap = c->cfg.num_image_with_embedding, T = c->T;
  std::vector<int> rows((size_t)k);
  for (int j = 0; j < k; ++j) rows[j] = (ids[j] * cap + c->pool_head[ids[j]]) * T;
  CUDA_OK(c, cudaMemcpyAsync(c->pool_rows.p, rows.data(), (size_t)k * sizeof(int), cudaMemcpyHostToDevice, s));
  // the launch sequence of gitb200_encode_images on the same k frames, except that ln_post writes through the row table
  gitb200_ctx::GraphKey key;
  key.kind = raw ? 11 : 10; key.p0 = raw ? (const void*)raw : (const void*)frames; key.i0 = k; key.i1 = height; key.i2 = width;
  const RawFrames rf{raw, height, width};
  const int r = run_graphed(c, key, s, k <= c->graph_max_clips || c->graph_segments, [&]() {
    return run_encode_sweeps(c, frames, k, 1, s, /*temporal=*/false, c->pool.p, c->pool_rows.p, raw ? &rf : nullptr);
  });
  if (r != 0 && r != 1) return r;
  for (int j = 0; j < k; ++j) {
    const int id = ids[j];
    c->pool_head[id] = (c->pool_head[id] + 1) % cap;
    if (c->pool_count[id] < cap) c->pool_count[id]++;
  }
  return GITB200_OK;
}

int gitb200_streams_push(gitb200_ctx* c, const int32_t* ids, int k, const float* frames, void* stream) {
  return streams_push_any(c, ids, k, frames, nullptr, 0, 0, stream);
}

int gitb200_streams_push_u8(gitb200_ctx* c, const int32_t* ids, int k, const uint8_t* frames, int height, int width, void* stream) {
  if (!frames) return fail(c, GITB200_ERR_INVALID, "gitb200_streams_push_u8: null frame buffer");
  return streams_push_any(c, ids, k, nullptr, frames, height, width, stream);
}

int gitb200_streams_caption(gitb200_ctx* c, const int32_t* ids, int k, const gitb200_search_params* sp, int32_t* tokens,
                            float* logprobs, void* stream) {
  if (!c || !sp || !tokens || !logprobs) return fail(c, GITB200_ERR_INVALID, "bad streams_caption argument");
  if (!c->finalized) return fail(c, GITB200_ERR_STATE, "call gitb200_finalize_weights first");
  TRY(pool_check_ids(c, "gitb200_streams_caption", ids, k));
  const int n = c->pool_count[ids[0]];
  for (int j = 0; j < k; ++j) {
    if (c->pool_count[ids[j]] < 1)
      return fail(c, GITB200_ERR_STATE, "gitb200_streams_caption: stream id %d holds no frames: push first", ids[j]);
    if (c->pool_count[ids[j]] != n)
      return fail(c, GITB200_ERR_INVALID, "gitb200_streams_caption: stream id %d holds %d frames but stream id %d holds %d: "
                  "windows of different lengths go in separate calls", ids[j], c->pool_count[ids[j]], ids[0], n);
  }
  CUDA_OK(c, cudaSetDevice(c->device));
  const cudaStream_t s = (cudaStream_t)stream;
  TRY(pool_order_after_last_stream(c, s));
  caller_stream(c, stream);
  const int cap = c->cfg.num_image_with_embedding, T = c->T, W = c->cfg.vit_width;
  ENSURE(c, c->vf, (size_t)k * n * T * W);
  std::vector<int> oldest((size_t)k);
  for (int j = 0; j < k; ++j) oldest[j] = ids[j] * cap + (c->pool_head[ids[j]] - n + cap) % cap;  // temporal position 0
  CUDA_OK(c, cudaMemcpyAsync(c->pool_oldest.p, oldest.data(), (size_t)k * sizeof(int), cudaMemcpyHostToDevice, s));
  auto assemble = [&]() -> int {
    CUDA_OK(c, assemble_windows(c->pool.p, c->pool_oldest.p, 0, k, n, cap, T, W, c->temporal, c->vf.p, nullptr, s));
    c->cur_clips = k; c->cur_nv = n * T; c->visual_pass_done = false; c->step_rows_per_clip = 0;
    return 0;
  };
  gitb200_ctx::GraphKey key;
  key.i0 = k; key.i1 = n;
  if (k <= c->graph_max_clips) {  // latency mode: the whole call as one graph (k == 1, beam <= 4: the persistent decode kernel)
    key.kind = 12; key.p0 = tokens; key.p1 = logprobs; key.sp = *sp;
    const int r = run_graphed(c, key, s, true, [&]() -> int {
      TRY(assemble());
      return run_decode(c, *sp, tokens, logprobs, nullptr, s);
    });
    if (r == 1) {  // replayed: host-side state the eager run would have left
      c->cur_clips = k; c->cur_nv = n * T; c->visual_pass_done = true; c->visual_pass_full = 0; c->step_rows_per_clip = 0;
      c->last_decode_steps = sp->max_steps - 1;
      return GITB200_OK;
    }
    return r;
  }
  // throughput-sized: window assembly + the decoder's visual pass as one graph, then the graphed decode segments of run_decode
  key.kind = 13;
  const int r = run_graphed(c, key, s, c->graph_segments, [&]() -> int {
    TRY(assemble());
    return run_visual_pass(c, false, nullptr, 0, s);
  });
  if (r == 1) {
    c->cur_clips = k; c->cur_nv = n * T; c->visual_pass_done = true; c->visual_pass_full = 0; c->step_rows_per_clip = 0;
  } else if (r != 0) {
    return r;
  }
  return run_decode(c, *sp, tokens, logprobs, nullptr, s);
}

int gitb200_streams_reset(gitb200_ctx* c, const int32_t* ids, int k) {
  if (!c) return GITB200_ERR_INVALID;
  TRY(pool_check_ids(c, "gitb200_streams_reset", ids, k));
  for (int j = 0; j < k; ++j) c->pool_head[ids[j]] = c->pool_count[ids[j]] = 0;
  return GITB200_OK;
}

int gitb200_streams_frames(const gitb200_ctx* c, int id) {
  if (!c || id < 0 || id >= c->pool_streams) return GITB200_ERR_INVALID;
  return c->pool_count[id];
}

int gitb200_streams_window(gitb200_ctx* c, int id, float* out, void* stream) {
  if (!c || !out) return fail(c, GITB200_ERR_INVALID, "bad streams_window argument");
  if (c->pool_streams < 1) return fail(c, GITB200_ERR_STATE, "gitb200_streams_window: no stream pool: call gitb200_streams_configure first");
  if (id < 0 || id >= c->pool_streams)
    return fail(c, GITB200_ERR_INVALID, "gitb200_streams_window: unknown stream id %d (the pool has ids 0..%d)", id, c->pool_streams - 1);
  const int n = c->pool_count[id];
  if (n < 1) return fail(c, GITB200_ERR_STATE, "gitb200_streams_window: stream id %d holds no frames", id);
  CUDA_OK(c, cudaSetDevice(c->device));
  const cudaStream_t s = (cudaStream_t)stream;
  TRY(pool_order_after_last_stream(c, s));
  caller_stream(c, stream);
  const int cap = c->cfg.num_image_with_embedding;
  CUDA_OK(c, assemble_windows(c->pool.p, nullptr, id * cap + (c->pool_head[id] - n + cap) % cap, 1, n, cap, c->T, c->cfg.vit_width,
                              c->temporal, nullptr, out, s));
  return GITB200_OK;
}

int gitb200_set_fold_layernorm(gitb200_ctx* c, int enable) {
  if (!c) return GITB200_ERR_INVALID;
  if (c->fold_ln != (enable != 0)) c->ws_gen++;  // captured graphs replay the other launch sequence
  c->fold_ln = enable != 0;
  if (c->twin) c->twin->fold_ln = c->fold_ln;
  return GITB200_OK;
}

int gitb200_set_early_exit(gitb200_ctx* c, int every_steps) {
  if (!c || every_steps < 0) return fail(c, GITB200_ERR_INVALID, "gitb200_set_early_exit: every_steps must be >= 0");
  c->early_exit_every = every_steps;
  return GITB200_OK;
}

int gitb200_set_persistent_decode(gitb200_ctx* c, int enable) {
  if (!c) return GITB200_ERR_INVALID;
  if (c->persistent_decode != (enable != 0)) c->ws_gen++;  // captured small-batch graphs hold the other launch sequence
  c->persistent_decode = enable != 0;
  return GITB200_OK;
}

int gitb200_debug_persistent_decode_trace(gitb200_ctx* c, unsigned long long* out32, int enable) {
  if (!c) return GITB200_ERR_INVALID;
  CUDA_OK(c, cudaSetDevice(c->device));
  CUDA_OK(c, cudaDeviceSynchronize());
  if (c->mega_trace.p == nullptr) {
    ENSURE(c, c->mega_trace, 32);
    CUDA_OK(c, cudaMemset(c->mega_trace.p, 0, 32 * sizeof(unsigned long long)));
  }
  if (out32) CUDA_OK(c, cudaMemcpy(out32, c->mega_trace.p, 32 * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
  if ((enable != 0) != c->mega_trace_on) {
    c->ws_gen++;  // captured graphs hold the kernel's arguments
    CUDA_OK(c, cudaMemset(c->mega_trace.p, 0, 32 * sizeof(unsigned long long)));
  }
  c->mega_trace_on = enable != 0;
  return GITB200_OK;
}

int gitb200_last_decode_steps(const gitb200_ctx* c) { return c ? c->last_decode_steps : 0; }

int gitb200_set_graph_max_clips(gitb200_ctx* c, int max_clips) {
  if (!c || max_clips < 0) return fail(c, GITB200_ERR_INVALID, "gitb200_set_graph_max_clips: max_clips must be >= 0");
  c->graph_max_clips = max_clips;
  return GITB200_OK;
}

int gitb200_set_fuse_layernorm(gitb200_ctx* c, int enable) {
  if (!c) return GITB200_ERR_INVALID;
  if (c->fuse_ln != (enable != 0)) c->ws_gen++;  // captured graphs replay the other launch sequence
  c->fuse_ln = enable != 0;
  if (c->twin) c->twin->fuse_ln = c->fuse_ln;
  return GITB200_OK;
}

int gitb200_set_graph_segments(gitb200_ctx* c, int enable) {
  if (!c) return GITB200_ERR_INVALID;
  c->graph_segments = enable != 0;
  return GITB200_OK;
}

int gitb200_set_pipeline(gitb200_ctx* c, int chunk_clips) {
  if (!c) return GITB200_ERR_INVALID;
  if (c->pipeline_chunk != chunk_clips) c->ws_gen++;
  c->pipeline_chunk = chunk_clips;
  return GITB200_OK;
}

int gitb200_caption_host(gitb200_ctx* c, const float* frames_host, int n_clips, int n_frames, int chunk_clips,
                         const gitb200_search_params* sp, int32_t* tokens_host, float* logprobs_host) {
  if (!c || !frames_host || !sp || !tokens_host || !logprobs_host || n_clips < 1 || n_frames < 1)
    return fail(c, GITB200_ERR_INVALID, "bad caption_host argument");
  if (!c->finalized) return fail(c, GITB200_ERR_STATE, "call gitb200_finalize_weights first");
  CUDA_OK(c, cudaSetDevice(c->device));
  if (chunk_clips < 1) chunk_clips = n_clips < 32 ? n_clips : 32;
  const size_t clip_elems = (size_t)n_frames * 3 * c->cfg.resolution * c->cfg.resolution;
  const int per_clip_tok = sp->num_keep_best * sp->max_steps;
  TRY(ensure_host_streams(c));
  TRY(order_after_caller_work(c));
  cudaStream_t comp = c->comp_stream;
  ENSURE(c, c->out_tok, (size_t)n_clips * per_clip_tok);
  ENSURE(c, c->out_lp, (size_t)n_clips * sp->num_keep_best);
  if (c->pipeline_chunk != 0) {
    // opt-in two-stream variant: chunk i is copied, then encoded + decoded on pipeline stream i & 1 (workspace set i & 1)
    for (int i = 0; i < 2; ++i) ENSURE(c, c->stage[i], (size_t)chunk_clips * clip_elems);
    TRY(ensure_pipeline(c));
    int done = 0;
    for (int ch = 0; done < n_clips; ++ch) {
      const int b = ch & 1;
      gitb200_ctx* cw = b ? c->twin : c;
      cudaStream_t s = c->pipe_stream[b];
      int nc = ch == 0 ? (chunk_clips + 1) / 2 : chunk_clips;
      if (nc > n_clips - done) nc = n_clips - done;
      if (ch >= 2) CUDA_OK(c, cudaStreamWaitEvent(c->copy_stream, c->ev_done[b], 0));  // staging buffer free again
      CUDA_OK(c, cudaMemcpyAsync(c->stage[b].p, frames_host + (size_t)done * clip_elems, (size_t)nc * clip_elems * sizeof(float),
                                 cudaMemcpyHostToDevice, c->copy_stream));
      CUDA_OK(c, cudaEventRecord(c->ev_copy[b], c->copy_stream));
      CUDA_OK(c, cudaStreamWaitEvent(s, c->ev_copy[b], 0));
      if (ch == 1) CUDA_OK(c, cudaStreamWaitEvent(s, c->ev_enc0, 0));
      int r = run_encode(cw, c->stage[b].p, nc, n_frames, s);
      if (r == 0) CUDA_OK(c, cudaEventRecord(c->ev_done[b], s));
      if (r == 0 && ch == 0) CUDA_OK(c, cudaEventRecord(c->ev_enc0, s));
      if (r == 0) r = run_decode(cw, *sp, c->out_tok.p + (size_t)done * per_clip_tok, c->out_lp.p + (size_t)done * sp->num_keep_best, nullptr, s);
      if (r) {
        if (b) c->err = c->twin->err;
        return r;
      }
      done += nc;
    }
    for (int i = 0; i < 2; ++i) {
      CUDA_OK(c, cudaEventRecord(c->ev_join[i], c->pipe_stream[i]));
      CUDA_OK(c, cudaStreamWaitEvent(comp, c->ev_join[i], 0));
    }
  } else {
    // Encode chunk by chunk as the frames arrive, then run the decoder once over all clips: the decode steps have a fixed
    // cost per launch that is amortised over the whole batch.
    TRY(encode_from_host(c, frames_host, nullptr, 0, 0, n_clips, n_frames, chunk_clips, comp));
    TRY(run_decode(c, *sp, c->out_tok.p, c->out_lp.p, nullptr, comp));
  }
  CUDA_OK(c, cudaMemcpyAsync(tokens_host, c->out_tok.p, (size_t)n_clips * per_clip_tok * sizeof(int32_t), cudaMemcpyDeviceToHost, comp));
  CUDA_OK(c, cudaMemcpyAsync(logprobs_host, c->out_lp.p, (size_t)n_clips * sp->num_keep_best * sizeof(float), cudaMemcpyDeviceToHost, comp));
  CUDA_OK(c, cudaStreamSynchronize(comp));
  return GITB200_OK;
}

// Host frames in, DEVICE results out: the chunked, copy-overlapped encode of gitb200_caption_host, then one decode whose
// tokens / log-probabilities / per-step logits / visual features stay on the device (what GenerativeImageTextModel.forward
// returns, model.py:768-780).  Work runs on the context's private streams; `stream` (the caller's) waits for the results.
int gitb200_caption_from_host(gitb200_ctx* c, const float* frames_host, int n_clips, int n_frames, int chunk_clips,
                              const gitb200_search_params* sp, int32_t* tokens_dev, float* logprobs_dev, float* logits_dev,
                              float* vf_dev, void* stream) {
  if (!c || !frames_host || !sp || !tokens_dev || !logprobs_dev || n_clips < 1 || n_frames < 1)
    return fail(c, GITB200_ERR_INVALID, "bad caption_from_host argument");
  if (!c->finalized) return fail(c, GITB200_ERR_STATE, "call gitb200_finalize_weights first");
  CUDA_OK(c, cudaSetDevice(c->device));
  if (chunk_clips < 1) chunk_clips = n_clips < 32 ? n_clips : 32;
  TRY(ensure_host_streams(c));
  TRY(order_after_caller_work(c));  // (work given to ANOTHER stream before this call)
  cudaStream_t comp = c->comp_stream, user = caller_stream(c, stream);
  // the caller's earlier work on its stream (e.g. the allocation of the output tensors) is ordered before ours
  CUDA_OK(c, cudaEventRecord(c->ev_user, user));
  CUDA_OK(c, cudaStreamWaitEvent(comp, c->ev_user, 0));
  CUDA_OK(c, cudaStreamWaitEvent(c->copy_stream, c->ev_user, 0));
  TRY(encode_from_host(c, frames_host, nullptr, 0, 0, n_clips, n_frames, chunk_clips, comp));
  if (vf_dev) CUDA_OK(c, cast_bf16_to_f32(c->vf.p, n_clips * c->cur_nv, c->cfg.vit_width, c->cfg.vit_width, vf_dev, c->cfg.vit_width, comp));
  TRY(run_decode(c, *sp, tokens_dev, logprobs_dev, logits_dev, comp));
  CUDA_OK(c, cudaEventRecord(c->ev_user, comp));
  CUDA_OK(c, cudaStreamWaitEvent(user, c->ev_user, 0));
  return GITB200_OK;
}

// Raw video frames from the host: uint8 BGR HWC, as cv2.VideoCapture / cv2.resize deliver them (real_time_inference.py:49-57,
// dataloader.py:61-75).  A chunk's frames cross PCIe as bytes (height*width*3 per frame instead of 3*R*R*4 after the
// host-side image_transform) and are resized / cropped / normalised by preprocess_kernel<true> straight into the bf16 patch
// matrix of the patch-embedding GEMM (no fp32 frames on the device at all); the copy of chunk i+1 overlaps chunk i's ViT.
int gitb200_caption_host_u8(gitb200_ctx* c, const uint8_t* frames_host, int n_clips, int n_frames, int height, int width,
                            int chunk_clips, const gitb200_search_params* sp, int32_t* tokens_host, float* logprobs_host) {
  if (!c || !frames_host || !sp || !tokens_host || !logprobs_host || n_clips < 1 || n_frames < 1 || height < 1 || width < 1)
    return fail(c, GITB200_ERR_INVALID, "bad caption_host_u8 argument");
  if (!c->finalized) return fail(c, GITB200_ERR_STATE, "call gitb200_finalize_weights first");
  CUDA_OK(c, cudaSetDevice(c->device));
  if (chunk_clips < 1) chunk_clips = n_clips < 32 ? n_clips : 32;
  const int per_clip_tok = sp->num_keep_best * sp->max_steps;
  TRY(ensure_host_streams(c));
  TRY(order_after_caller_work(c));
  cudaStream_t comp = c->comp_stream;
  ENSURE(c, c->out_tok, (size_t)n_clips * per_clip_tok);
  ENSURE(c, c->out_lp, (size_t)n_clips * sp->num_keep_best);
  TRY(encode_from_host(c, nullptr, frames_host, height, width, n_clips, n_frames, chunk_clips, comp));  // a chunk's first kernel consumes the bytes
  TRY(run_decode(c, *sp, c->out_tok.p, c->out_lp.p, nullptr, comp));
  CUDA_OK(c, cudaMemcpyAsync(tokens_host, c->out_tok.p, (size_t)n_clips * per_clip_tok * sizeof(int32_t), cudaMemcpyDeviceToHost, comp));
  CUDA_OK(c, cudaMemcpyAsync(logprobs_host, c->out_lp.p, (size_t)n_clips * sp->num_keep_best * sizeof(float), cudaMemcpyDeviceToHost, comp));
  CUDA_OK(c, cudaStreamSynchronize(comp));
  return GITB200_OK;
}

int gitb200_forward_logits(gitb200_ctx* c, const float* frames, int n_clips, int n_frames, const int32_t* tokens, int L,
                           float* logits, float* hidden, float* vf_out, void* stream) {
  if (!c || !tokens || !logits || L < 1) return fail(c, GITB200_ERR_INVALID, "bad forward_logits argument");
  if (!c->finalized) return fail(c, GITB200_ERR_STATE, "call gitb200_finalize_weights first");
  if (L > c->cfg.max_positions) return fail(c, GITB200_ERR_INVALID, "caption length %d exceeds %d positions", L, c->cfg.max_positions);
  CUDA_OK(c, cudaSetDevice(c->device));
  cudaStream_t s = caller_stream(c, stream);
  if (frames) {
    if (n_clips < 1 || n_frames < 1) return fail(c, GITB200_ERR_INVALID, "bad forward_logits argument");
    TRY(run_encode_sweeps(c, frames, n_clips, n_frames, s));
  }
  if (c->cur_clips <= 0) return fail(c, GITB200_ERR_STATE, "no visual features");
  const int B = c->cur_clips, rows = B * L, W = c->cfg.vit_width;
  if (vf_out) CUDA_OK(c, cast_bf16_to_f32(c->vf.p, B * c->cur_nv, W, W, vf_out, W, s));
  const bool want_full = hidden != nullptr;
  if (!c->visual_pass_done || (want_full && !c->visual_pass_full) || hidden) TRY(run_visual_pass(c, want_full, hidden, L, s));
  TRY(ensure_text(c, rows, B, L));
  ENSURE(c, c->pos_arr, rows);
  ENSURE(c, c->ntext_arr, rows);
  CUDA_OK(c, fill_positions(c->pos_arr.p, c->ntext_arr.p, rows, L, s));
  TextPass tp;
  tp.n_clips = B; tp.rows_per_clip = L; tp.max_len = L;
  tp.tokens = tokens; tp.positions = c->pos_arr.p; tp.pos_const = 0;
  tp.n_text = c->ntext_arr.p; tp.n_text_const = 0; tp.anc = nullptr;
  tp.slot_div = L; tp.n_slots = B; tp.slot_is_clip = 1;
  tp.logits = logits; tp.hidden_out = hidden;
  return run_text_pass(c, tp, s);
}

int gitb200_decode_begin(gitb200_ctx* c, int rows_per_clip, void* stream) {
  if (!c || rows_per_clip < 1) return fail(c, GITB200_ERR_INVALID, "bad decode_begin argument");
  if (!c->finalized) return fail(c, GITB200_ERR_STATE, "call gitb200_finalize_weights first");
  CUDA_OK(c, cudaSetDevice(c->device));
  cudaStream_t s = caller_stream(c, stream);
  if (!c->visual_pass_done) TRY(run_visual_pass(c, false, nullptr, 0, s));
  const int rows = c->cur_clips * rows_per_clip, ml = c->cfg.max_positions < 64 ? c->cfg.max_positions : 64;
  TRY(ensure_text(c, rows, rows, ml));
  ENSURE(c, c->ibuf, (size_t)rows * ml * 2);
  c->step_rows_per_clip = rows_per_clip;
  c->anc_parity = 0;
  c->step_anc_used = false;
  return GITB200_OK;
}

int gitb200_decode_step(gitb200_ctx* c, const int32_t* tokens, int pos, float* logits, void* stream) {
  if (!c || !tokens || !logits || pos < 0) return fail(c, GITB200_ERR_INVALID, "bad decode_step argument");
  if (c->step_rows_per_clip < 1 || !c->visual_pass_done) return fail(c, GITB200_ERR_STATE, "call gitb200_decode_begin first");
  const int ml = c->cfg.max_positions < 64 ? c->cfg.max_positions : 64;
  if (pos >= ml) return fail(c, GITB200_ERR_INVALID, "step-wise decoding supports up to %d text positions", ml);
  CUDA_OK(c, cudaSetDevice(c->device));
  const int rows = c->cur_clips * c->step_rows_per_clip;
  TextPass tp;
  tp.n_clips = c->cur_clips; tp.rows_per_clip = c->step_rows_per_clip; tp.max_len = ml;
  tp.tokens = tokens; tp.positions = nullptr; tp.pos_const = pos; tp.n_text = nullptr; tp.n_text_const = pos + 1;
  tp.anc = c->step_anc_used ? c->ibuf.p + (size_t)c->anc_parity * rows * ml : nullptr;
  tp.slot_div = 1; tp.n_slots = rows; tp.slot_is_clip = 0; tp.logits = logits; tp.hidden_out = nullptr;
  return run_text_pass(c, tp, caller_stream(c, stream));
}

int gitb200_decode_reorder(gitb200_ctx* c, const int32_t* beam_idx, int pos, void* stream) {
  if (!c || !beam_idx || pos < 0) return fail(c, GITB200_ERR_INVALID, "bad decode_reorder argument");
  if (c->step_rows_per_clip < 1) return fail(c, GITB200_ERR_STATE, "call gitb200_decode_begin first");
  CUDA_OK(c, cudaSetDevice(c->device));
  const int rows = c->cur_clips * c->step_rows_per_clip, ml = c->cfg.max_positions < 64 ? c->cfg.max_positions : 64;
  int* a0 = c->ibuf.p + (size_t)c->anc_parity * rows * ml;
  int* a1 = c->ibuf.p + (size_t)(c->anc_parity ^ 1) * rows * ml;
  CUDA_OK(c, anc_reorder(c->step_anc_used ? a0 : nullptr, a1, beam_idx, rows, ml, pos, caller_stream(c, stream)));
  c->anc_parity ^= 1;
  c->step_anc_used = true;
  return GITB200_OK;
}

// ---- single operators
int gitb200_op_gemm(const void* a, const void* w, int M, int N, int K, const float* bias, const void* residual, int act,
                    void* out_bf16, float* out_f32, int tile_n, void* stream) {
  GemmArgs g;
  g.A = (const bf16*)a; g.lda = K; g.W = (const bf16*)w; g.ldw = K; g.M = M; g.N = N; g.K = K; g.bias = bias;
  g.residual = (const bf16*)residual; g.ldr = N; g.act = act; g.out = (bf16*)out_bf16; g.ldo = N; g.out_f32 = out_f32; g.ldo32 = N;
  cudaError_t e = gemm_bf16(g, (cudaStream_t)stream, tile_n);
  if (e != cudaSuccess) return fail(nullptr, GITB200_ERR_CUDA, "gemm: %s [%s]", cudaGetErrorString(e), gemm_last_error());
  return GITB200_OK;
}

int gitb200_op_gemm_ln(const void* a, const void* w, int M, int N, int K, const float* bias, const void* residual, const float* gamma,
                       const float* beta, float eps, void* out_bf16, void* ln_out_bf16, void* stream) {
  GemmArgs g;
  g.A = (const bf16*)a; g.lda = K; g.W = (const bf16*)w; g.ldw = K; g.M = M; g.N = N; g.K = K; g.bias = bias;
  g.residual = (const bf16*)residual; g.ldr = N; g.out = (bf16*)out_bf16; g.ldo = N;
  g.lnout = (bf16*)ln_out_bf16; g.lnout_ld = N; g.lnout_gamma = gamma; g.lnout_beta = beta; g.lnout_eps = eps;
  cudaError_t e = gemm_bf16(g, (cudaStream_t)stream, 0);
  if (e != cudaSuccess) return fail(nullptr, GITB200_ERR_CUDA, "gemm_ln: %s [%s]", cudaGetErrorString(e), gemm_last_error());
  return GITB200_OK;
}

int gitb200_op_layernorm(const void* x, int rows, int cols, const float* gamma, const float* beta, float eps, void* out, void* stream) {
  LayerNormArgs a;
  a.x = (const bf16*)x; a.ldx = cols; a.rows = rows; a.cols = cols; a.gamma = gamma; a.beta = beta; a.eps = eps; a.out = (bf16*)out; a.ldo = cols;
  cudaError_t e = layernorm_bf16(a, (cudaStream_t)stream);
  if (e != cudaSuccess) return fail(nullptr, GITB200_ERR_CUDA, "layernorm: %s", cudaGetErrorString(e));
  return GITB200_OK;
}

int gitb200_op_attention_groups(const void* qkv, void* out, int n_groups, int group_len, int heads, float scale, void* stream) {
  cudaError_t e = attention_groups_tc((const bf16*)qkv, 3 * heads * 64, (bf16*)out, heads * 64, n_groups, group_len, heads, scale, (cudaStream_t)stream);
  if (e != cudaSuccess) return fail(nullptr, GITB200_ERR_CUDA, "attention_groups_tc: %s [%s]", cudaGetErrorString(e), gemm_last_error());
  return GITB200_OK;
}

int gitb200_op_attention_groups_mma(const void* qkv, void* out, int n_groups, int group_len, int heads, float scale, void* stream) {
  cudaError_t e = attention_groups((const bf16*)qkv, 3 * heads * 64, (bf16*)out, heads * 64, n_groups, group_len, heads, scale, (cudaStream_t)stream);
  if (e != cudaSuccess) return fail(nullptr, GITB200_ERR_CUDA, "attention_groups: %s", cudaGetErrorString(e));
  return GITB200_OK;
}

int gitb200_op_text_attention(const void* q, const void* vis_kv, const void* txt_kv, const int32_t* anc, int n_clips, int rows_per_clip,
                              int heads, int n_vis, int n_text, int splits, float scale, void* out, void* stream) {
  if (!q || !vis_kv || !out || n_clips < 1 || rows_per_clip < 1 || heads < 1 || n_vis < 0 || n_text < 0 || (n_text > 0 && !txt_kv) ||
      splits < 1 || splits > 16)
    return fail(nullptr, GITB200_ERR_INVALID, "bad op_text_attention argument");
  TextAttnArgs a;
  const int width = heads * 64, rows = n_clips * rows_per_clip;
  a.q = (const bf16*)q; a.ldq = width;
  a.n_clips = n_clips; a.rows_per_clip = rows_per_clip; a.heads = heads;
  a.vis_kv = (const bf16*)vis_kv; a.ld_vis = 2 * width; a.k_off = 0; a.v_off = width; a.Nv = n_vis;
  a.txt_kv = (const bf16*)txt_kv; a.txt_slots = rows;
  a.anc = anc; a.anc_ld = n_text;
  a.n_text_const = n_text; a.max_text = n_text;
  a.scale = scale;
  a.out = (bf16*)out; a.ldo = width;
  a.splits = splits;
  float* partial = nullptr;
  if (splits > 1 && cudaMalloc(&partial, text_attention_workspace_floats(rows, heads, splits) * sizeof(float)) != cudaSuccess)
    return fail(nullptr, GITB200_ERR_CUDA, "op_text_attention: workspace allocation failed");
  a.partial = partial;
  cudaError_t e = text_attention(a, (cudaStream_t)stream);
  if (partial) {
    if (e == cudaSuccess) e = cudaStreamSynchronize((cudaStream_t)stream);
    cudaFree(partial);
  }
  if (e != cudaSuccess) return fail(nullptr, GITB200_ERR_CUDA, "text_attention: %s", cudaGetErrorString(e));
  return GITB200_OK;
}

int gitb200_preprocess(const uint8_t* frames, int n_frames, int height, int width, int size, float* out, void* stream) {
  if (!frames || !out) return fail(nullptr, GITB200_ERR_INVALID, "bad preprocess argument");
  cudaError_t e = preprocess_frames_u8(frames, n_frames, height, width, size, out, (cudaStream_t)stream);
  if (e != cudaSuccess) return fail(nullptr, GITB200_ERR_CUDA, "preprocess: %s", cudaGetErrorString(e));
  return GITB200_OK;
}

int gitb200_op_search(const float* logits, int ld, int vocab, int n_clips, int sos, int eos, const gitb200_search_params* sp,
                      int32_t* tokens, float* logprobs, void* stream) {
  if (!logits || !sp || !tokens || !logprobs || n_clips < 1) return fail(nullptr, GITB200_ERR_INVALID, "bad op_search argument");
  gitb200_ctx tmp;  // scratch owner for the search buffers
  cudaGetDevice(&tmp.device);
  SearchState st;
  int r = make_search_state(&tmp, n_clips, vocab, ld, sos, eos, *sp, &st);
  cudaStream_t s = (cudaStream_t)stream;
  cudaError_t e = cudaSuccess;
  if (!r) {
    const int rows = n_clips * sp->beam_size;
    e = search_init(st, sos, s);
    int parity = 0;
    for (int t = 0; e == cudaSuccess && t + 1 < sp->max_steps; ++t) {
      e = search_step(st, logits + (size_t)t * rows * ld, t + 1, parity, s);
      parity ^= 1;
    }
    if (e == cudaSuccess) e = search_finalize(st, tokens, logprobs, s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
  }
  if (tmp.ibuf.p) cudaFree(tmp.ibuf.p);
  if (tmp.dbuf.p) cudaFree(tmp.dbuf.p);
  if (tmp.fbuf.p) cudaFree(tmp.fbuf.p);
  if (r) return fail(nullptr, r, "%s", tmp.err.c_str());
  if (e != cudaSuccess) return fail(nullptr, GITB200_ERR_CUDA, "search: %s", cudaGetErrorString(e));
  return GITB200_OK;
}

}  // extern "C"

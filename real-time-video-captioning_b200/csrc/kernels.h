// Host-side launch interface of the sm_100a kernels (internal C++; the public C-ABI is
// include/gitb200.h, implemented in api.cu on top of these).
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

typedef __nv_bfloat16 bf16;

enum { ACT_NONE = 0, ACT_QUICK_GELU = 1, ACT_GELU_ERF = 2, ACT_RELU = 3 };

// every host wrapper below reports the kernels it enqueues (gitb200_launch_count)
void note_launch(int n = 1);

// C[M,N] = act(A[M,K] * W[N,K]^T + bias) + residual, bf16 operands, fp32 accumulation in TMEM.
struct GemmArgs {
  const bf16* A = nullptr;  // row-major [M, K], leading dimension lda (elements, multiple of 8)
  int lda = 0;
  const bf16* W = nullptr;  // row-major [N, K] (the nn.Linear layout), leading dimension ldw
  int ldw = 0;
  int M = 0, N = 0, K = 0;        // N % 128 == 0, K % 8 == 0
  const float* bias = nullptr;    // [N] fp32, optional
  const bf16* residual = nullptr; // optional addend, leading dimension ldr
  int ldr = 0;
  int res_periodic = 0;  // 1: residual row = (r % gin) + goff (positional-embedding table), 0: output row
  int act = ACT_NONE;
  bf16* out = nullptr;  // optional bf16 output, leading dimension ldo
  int ldo = 0;
  float* out_f32 = nullptr;  // optional fp32 output, leading dimension ldo32
  int ldo32 = 0;
  // Output row remap: out_row = (r / gin) * gout + (r % gin) + goff when gin > 0 (used to leave a
  // gap for the CLS row of every frame in the patch-embedding GEMM).
  int gin = 0, gout = 0, goff = 0;
  // LayerNorm folded into this GEMM (pre-LN blocks): A holds the UN-normalised rows x, W already carries gamma
  // (W' = W * diag(gamma)), bias already carries W * beta, and the epilogue applies
  //     rstd_r * (acc - mean_r * ln_colsum[n]) + bias[n]      with (sum, sum of squares) of row r = the sum over the row's
  //     2 * K / 256 partial slots in ln_stats (one per 128-column half tile of the GEMM that produced A; added in slot order).
  const float* ln_stats = nullptr;   // [M, 2 * K / 256, 2] fp32
  const float* ln_colsum = nullptr;  // [N] fp32: sum_k W'[n, k]
  float ln_eps = 1e-5f;
  // Optional: (sum, sum of squares) of every OUTPUT row (bf16-rounded values), one partial pair per 128-column half tile, stored
  // (not accumulated: deterministic, nothing to zero) into stats_out[r][2 * N / 256][2] -- what the next folded LayerNorm needs.
  float* stats_out = nullptr;
  // LayerNorm of the OUTPUT rows as a second output (CTA-pair kernel only, N <= 1024, bf16 `out` required):
  //     lnout[r, :] = LN(out[r, :]) * lnout_gamma + lnout_beta      (statistics of the bf16-rounded output row, fp32)
  // -- the LayerNorm that follows a residual GEMM, written by the GEMM itself (see gemm2_tcgen05.cu, LNOUT).
  bf16* lnout = nullptr;
  int lnout_ld = 0;
  const float* lnout_gamma = nullptr;
  const float* lnout_beta = nullptr;
  float lnout_eps = 1e-5f;
  // ---- weight-streaming skinny kernel only (M <= 8 decode rows; gemm_bf16 rejects them on the tensor-core kernels) ----
  // LayerNorm of the A rows ON LOAD (M <= 4, K == 768): A holds the UN-normalised rows; every warp normalises them exactly
  // like layernorm_kernel (fp32 statistics, result rounded to bf16) before its dot products, and CTA 0 also stores the
  // normalised rows to lnl_out (the residual of a later sub-layer).  Removes one launch per LayerNorm from a decode step.
  const float* lnl_gamma = nullptr;
  const float* lnl_beta = nullptr;
  float lnl_eps = 0.f;
  bf16* lnl_out = nullptr;
  int lnl_ldo = 0;
  // Output columns >= sc_q_width are ALSO scattered into the text K/V plane (the store_text_kv kernel fused into the QKV
  // projection): sc_kv[(pos(m) * sc_n_slots + m / sc_slot_div) * sc_kv_width + (n - sc_q_width)].
  bf16* sc_kv = nullptr;
  int sc_q_width = 0, sc_kv_width = 0;
  const int* sc_pos = nullptr;
  int sc_pos_const = 0, sc_slot_div = 1, sc_n_slots = 0;
};
// force_bn: 0 = heuristic, 128 or 256 = tile width override (tests / tuning).
cudaError_t gemm_bf16(const GemmArgs& a, cudaStream_t stream, int force_bn = 0);
const char* gemm_last_error();
// per-launch CUDA-event timing of the GEMM kernel (bench.py roofline): enable resets the counters
void gemm_profile_enable(int on);
bool gemm_profile_enabled();
void gemm_profile_read(double* ms, double* flops, long long* launches);

// out[r,:] = LN(x[r,:]) * gamma + beta (+ addend[((r / add_group) % add_period), :]); fp32 statistics.
struct LayerNormArgs {
  const bf16* x = nullptr;
  int ldx = 0;
  int rows = 0, cols = 0;  // cols == 768 or 1024 (layernorm_bf16 returns cudaErrorInvalidValue for any other width)
  const float* gamma = nullptr;
  const float* beta = nullptr;
  float eps = 1e-5f;
  const float* addend = nullptr;  // optional [add_period, cols] fp32 (temporal embedding)
  int add_group = 1, add_period = 1;
  bf16* out = nullptr;
  int ldo = 0;
  float* out_f32 = nullptr;  // optional fp32 copy
  int ldo32 = 0;
  float* stats_out = nullptr;  // optional [rows, stats_slots, 2]: (sum, sum of squares) of the bf16-rounded output row in slot 0, zeros elsewhere
  int stats_slots = 1;
  // optional device table: input rows [g * out_group, (g + 1) * out_group) are written to output rows out_row_base[g] + 0,
  // 1, ... (ln_post of a multi-stream push straight into each frame's ring slot); null = output row r for input row r
  const int* out_row_base = nullptr;
  int out_group = 0;
};
cudaError_t layernorm_bf16(const LayerNormArgs& a, cudaStream_t stream);

// frames fp32 NCHW [n_frames, 3, res, res] -> patches bf16 [n_frames * grid * grid, kpad], k = c*p*p + ky*p + kx
cudaError_t im2col_patches(const float* frames, int n_frames, int res, int patch, int kpad, bf16* out,
                           cudaStream_t stream);
// x[f*T + 0, :] = cls[:] + pos[0, :]   (bf16 residual stream)
cudaError_t write_cls_rows(const float* cls, const bf16* pos, int n_frames, int T, int width, bf16* x,
                           cudaStream_t stream);

// Bidirectional self-attention over fixed-length groups of rows (ViT frames: len 197/257; decoder
// visual pass: len Nv).  qkv: [rows, 3*H*64] bf16 laid out [q | k | v], out: [rows, H*64] bf16.
cudaError_t attention_groups(const bf16* qkv, int ld_qkv, bf16* out, int ldo, int n_groups, int group_len,
                             int heads, float scale, cudaStream_t stream);
// Same contract on the tcgen05 path (S and PV accumulators in TMEM, TMA-fed): the kernel the pipeline uses.
cudaError_t attention_groups_tc(const bf16* qkv, int ld_qkv, bf16* out, int ldo, int n_groups, int group_len,
                                int heads, float scale, cudaStream_t stream);

// Text rows attending to the visual keys of their clip plus their causal text prefix.
struct TextAttnArgs {
  const bf16* q = nullptr;  // [n_rows, ldq] : query of text row r (first H*64 columns used)
  int ldq = 0;
  int n_clips = 0, rows_per_clip = 0;  // row r belongs to clip r / rows_per_clip
  int heads = 0;
  const bf16* vis_kv = nullptr;  // this layer's visual K|V: [n_clips * Nv, ld_vis], K at col k_off, V at col v_off
  int ld_vis = 0, k_off = 0, v_off = 0, Nv = 0;
  const bf16* txt_kv = nullptr;  // this layer's text K|V plane: [max_pos][txt_slots][2*H*64]  (K then V)
  int txt_slots = 0;             // slots per position: n_rows (decode: one per beam row) or n_clips (teacher forcing)
  int text_slot_is_clip = 0;     // 1: every text key of row r lives in slot (r / rows_per_clip)  (teacher forcing)
  const int* anc = nullptr;      // [n_rows, anc_ld]: slot of row r's ancestor at text position s < n_text-1 (null = r)
  int anc_ld = 0;
  const int* n_text = nullptr;   // [n_rows] number of visible text keys (pos+1); null = n_text_const
  int n_text_const = 0;
  int max_text = 0;              // upper bound of the visible text keys of any row (sizes the score buffer)
  float scale = 0.125f;
  bf16* out = nullptr;  // [n_rows, ldo]
  int ldo = 0;
  float* partial = nullptr;  // workspace: [n_rows * heads * splits * (64 + 2)] fp32
  int splits = 1;
};
cudaError_t text_attention(const TextAttnArgs& a, cudaStream_t stream);
size_t text_attention_workspace_floats(int n_rows, int heads, int splits);

// words[tok] + positions[pos] -> LN(eps) -> out bf16   (fp32 tables; positions == nullptr -> pos_const)
cudaError_t embed_text(const int* tokens, const int* positions, int pos_const, int n_rows, const float* words,
                       const float* pos_table, const float* gamma, const float* beta, float eps, int width, bf16* out,
                       cudaStream_t stream);

// Scatter this step's K|V (columns [q_width, q_width + kv_width) of qkv) into the text KV plane:
// txt_kv[(pos(r) * n_slots + r / slot_div) * kv_width + c];  pos(r) = pos ? pos[r] : pos_const.
cudaError_t store_text_kv(const bf16* qkv, int ld_qkv, int n_rows, int kv_width, int q_width, const int* pos,
                          int pos_const, int slot_div, int n_slots, bf16* txt_kv, cudaStream_t stream);

cudaError_t cast_f32_to_bf16(const float* src, int rows, int cols, int lds, bf16* dst, int ldd, int dst_rows,
                             int dst_cols, cudaStream_t stream);
cudaError_t cast_bf16_to_f32(const bf16* src, int rows, int cols, int lds, float* dst, int ldd, cudaStream_t stream);

// Beam / greedy search state, all device resident (semantics: reference model.py:479-678).
struct SearchState {
  int n_clips, nb, cand, V, ldl, max_len, eos, n_keep;
  float length_penalty;
  int* tokens;        // [n_rows, max_len]   current partial captions (input_ids)
  int* tokens_tmp;    // [n_rows, max_len]
  float* beam_scores; // [n_rows]
  int* done;          // [n_clips]
  int* done_count;    // [1] number of clips whose search is finished (model.py:640 `if all(done): break`)
  int* anc;           // [n_rows, max_len] ancestor slot per text position
  int* anc_tmp;
  int* cur_tok;       // [n_rows] token fed to the next step
  // hypotheses: per clip up to n_keep (+1 scratch)
  double* hyp_score;  // [n_clips, n_keep + 1]  (Python float arithmetic in the reference -> double)
  int* hyp_len;       // [n_clips, n_keep + 1]
  int* hyp_tok;       // [n_clips, n_keep + 1, max_len]
  int* hyp_count;     // [n_clips]
  double* worst;      // [n_clips]
  int reorder_cache;  // 0 = reference behaviour (cache rows never re-indexed), 1 = re-index by parent
  // beam search: every row's own top `cand` candidates [n_rows, cand] (search_step: one CTA per ROW selects, one per clip merges
  // and walks); null = one CTA per clip does both
  float* row_cand_score = nullptr;
  int* row_cand_idx = nullptr;
};
// One search step: log-softmax over logits [n_rows, ldl] (fp32), + beam score, top-(cand) per clip,
// then the reference's candidate walk; cur_len = current caption length before this step.
// parity: which of the (tokens, tokens_tmp) / (anc, anc_tmp) pairs currently holds the live state
// (0: tokens/anc are read and *_tmp written; 1: the reverse).  The caller flips it after every step.
cudaError_t search_step(const SearchState& s, const float* logits, int cur_len, int parity, cudaStream_t stream);
cudaError_t search_init(const SearchState& s, int sos, cudaStream_t stream);
// search_init with a prompt of P tokens (model.py:432-437, batch['prefix']): prompt is device int [clips][P] and row r belongs
// to clip r / rows_per_clip; its history is that clip's P tokens and it feeds the last of them to the first step.
// The history goes to the token buffer that the first step (t0 = P - 1) reads: tokens for even t0, tokens_tmp for odd.
// P >= max_len: no step runs and the prompt (which does not fit) is not written.
cudaError_t search_init_prefix(const SearchState& s, const int* prompt, int P, int rows_per_clip, cudaStream_t stream);
// decoded [n_clips, n_keep, max_len] (eos padded), logprobs [n_clips, n_keep]
cudaError_t search_finalize(const SearchState& s, int* decoded, float* logprobs, cudaStream_t stream);
// Extended search step (model.py:524-554): repetition penalty, and with do_sample temperature, top-k / top-p filtering
// (min_tokens_to_keep = 2) and per_node_beam_size draws without replacement per beam row.  The search "clips" of `s` are
// entries e = clip * nrs + j (return sequence j of clip `clip`), nb rows each.
struct SampleState {
  int do_sample, top_k, nrs, pnb;
  float top_p, temperature, rp;
  const unsigned long long* seed;  // device word: the Philox key
  // Optional device table of one Philox key per clip (entry e draws with keys[e / nrs] and counter word 3 = 0, so a clip's
  // draws do not depend on its position in the call).  nullptr: key *seed, counter word 3 = the clip index e / nrs.
  const unsigned long long* keys;
};
// Bytes of dynamic shared memory a row of `V` logits needs (the limit the caller checks before enqueueing anything).
size_t sample_step_smem(int V);
// step = t for cur_len = t + 1 (the Philox counter's step word)
cudaError_t sample_step(const SearchState& s, const SampleState& p, const float* logits, int cur_len, int parity, int step,
                        cudaStream_t stream);

// ---- persistent single-clip decode kernel (decode_mega.cu): the whole search of ONE clip (rows = beams <= 4) in one launch
constexpr int MEGA_MAX_LAYERS = 8;
struct MegaLayer {
  const bf16 *w_qkv, *w_out, *w_fc1, *w_fc2;  // [3H, H], [H, H], [ffn, H], [H, ffn]
  const float *b_qkv, *b_out, *b_fc1, *b_fc2, *lna_g, *lna_b, *lno_g, *lno_b;
  const bf16* vis_kv;  // the clip's visual q|k|v rows of this layer: [Nv, 3H]
  bf16* txt_kv;        // this layer's text K|V plane: [max_len][rows][2H]
};
struct MegaArgs {
  MegaLayer layer[MEGA_MAX_LAYERS];
  int n_layers, rows, hidden, heads, ffn, Nv, splits, kcap, vocab_pad, steps;
  int first_step;                                  // the loop runs t = first_step .. steps - 1 (a prompt of P tokens: P - 1)
  const float *words, *pos_table, *lne_g, *lne_b;  // fp32 embedding tables, embedding LayerNorm
  float embed_eps, ln_eps, scale_log2;
  const bf16* w_vocab;   // [vocab_pad, H]
  const float* b_vocab;  // [vocab_pad]
  float* logits;         // [steps or 1][rows, vocab_pad] (step t's logits at logits + t * logits_step_stride)
  long long logits_step_stride;  // floats between the logits of consecutive steps (0: one buffer reused)
  bf16 *tq, *ta, *tb, *tf;  // scratch rows: [rows, 3H], [rows, H], [rows, H], [rows, ffn]
  float* partial;           // key-split partials of the attention
  unsigned int* barrier;    // grid barrier counter (reset by the launcher together with attn_cnt: 32 words from here)
  int* attn_cnt;            // [row chunks * heads <= 24] finished key splits per (row chunk, head): the last one combines
  unsigned long long* trace;  // optional [32]: SM cycles of CTA 0 per phase (0-7: work, 16-23: barrier wait; 15: launches)
  float* cand_score;        // [rows * st.cand] every beam row's own top candidates (search step, part 1 -> part 2)
  int* cand_idx;
  SearchState st;
};
bool decode_mega_supported(const MegaArgs& a);
void decode_mega_attention_geometry(int rows, int heads, int Nv, int max_text, int* splits, int* kcap);
cudaError_t decode_mega(const MegaArgs& a, cudaStream_t stream);

// Prompt K/V into the decode plane: dst[(p * n_clips * rows_per_clip + r) * width + c] = src[(p * n_clips + r / rows_per_clip) *
// width + c] for p < n_pos (src: the teacher-forced plane [n_pos][n_clips][width]; width % 8 == 0)
cudaError_t fanout_prefix_kv(const bf16* src, bf16* dst, int n_pos, int n_clips, int rows_per_clip, int width, cudaStream_t stream);
// pos[r] = r % L, n_text[r] = r % L + 1 (teacher-forced text rows)
cudaError_t fill_positions(int* pos, int* n_text, int rows, int L, cudaStream_t stream);
// Step-wise decoding cache re-index: out[r][s] = in ? in[beam_idx[r]][s] : beam_idx[r] for s < pos; out[r][pos] = beam_idx[r].
cudaError_t anc_reorder(const int* anc_in, int* anc_out, const int* beam_idx, int rows, int ld, int pos, cudaStream_t stream);

// uint8 BGR HWC frames [n, H, W, 3] -> fp32 RGB NCHW [n, 3, size, size]: bicubic resize of the smaller edge to `size`,
// centre crop, CLIP normalisation (the reference's image_transform(), src/utils/dataloader.py:18-32).
cudaError_t preprocess_frames_u8(const uint8_t* frames, int n, int H, int W, int size, float* out, cudaStream_t stream);
// same pixels written as bf16 into the patch-embedding GEMM's A matrix (im2col layout, K padded to kpad): no fp32 frames in between
cudaError_t preprocess_frames_u8_to_patches(const uint8_t* frames, int n, int H, int W, int size, int patch, int kpad,
                                            bf16* patches, cudaStream_t stream);

// LayerNorm folding at weight-load time: wf[n,k] = bf16(w[n,k] * gamma[k]); colsum[n] = sum_k float(wf[n,k]);
// bias_f[n] = bias[n] + sum_k w[n,k] * beta[k].
cudaError_t ln_fold_weight(const float* w, int N, int K, const float* gamma, const float* beta, const float* bias, bf16* wf,
                           float* colsum, float* bias_f, cudaStream_t stream);

// Streaming window: vf[i*T + t, :] = ring[((first + i) % cap)*T + t, :] + temporal[i, :]  for i < n  (bf16, fp32 temporal)
cudaError_t assemble_window(const bf16* ring, int first, int cap, int n, int T, int W, const float* temporal, bf16* vf,
                            cudaStream_t stream);
// Multi-stream pool: the k windows of n frames each, vf[(w*n + i)*T + t, :] = ring[slot(w, i)*T + t, :] + temporal[i, :] with
// slot(w, i) = base + (first + i) % cap and oldest[w] = base + first (device table; nullptr: oldest_const for the one window).
// Writes bf16 vf, or, if vf32 != nullptr, the same bf16-rounded values as fp32 to vf32 instead.
cudaError_t assemble_windows(const bf16* ring, const int* oldest, int oldest_const, int k, int n, int cap, int T, int W,
                             const float* temporal, bf16* vf, float* vf32, cudaStream_t stream);

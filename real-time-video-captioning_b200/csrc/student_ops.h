// Host-side launchers of the student decoder's kernels (student.cu: inference, student_train.cu: the distillation step).
// Host-only: it includes nothing but kernels.h, so a host compiler can build against it (tests/cuda/student_ops.cpp).
// Every launcher enqueues on stream s, reports its kernels through note_launch and returns 0 or a GITB200_ERR_* code (the
// message in gitb200_student_last_error).  Scratch buffers are arguments: no launcher allocates or reads the training state.
#pragma once
#include "kernels.h"

struct gitb200_student;

namespace sdet {

// One dropout site of the distillation step (mask: philox.cuh, dropout_scale): key `seed`, counter word `step` (the dropout
// step, mod 2^32) and `site` = 6 * layer + k; p in (0, 1), inv_keep = 1 / (1 - p) in fp32.
struct SDrop {
  unsigned long long seed;
  unsigned step;
  unsigned site;
  float p, inv_keep;
};

// ---- forward (student.cu)
// out = A W^T + bias (+ residual), act; bf16 out and / or fp32 out32 (gemm_bf16)
int s_gemm(gitb200_student* c, const bf16* A, int lda, const bf16* W, int K, int M, int N, const float* bias, const bf16* residual,
           int ldr, int act, bf16* out, int ldo, float* out32, int ldo32, cudaStream_t s);
// out[r, :] = LN(x[r, :]) * g + b over d_model columns, eps = cfg.ln_eps
int s_ln(gitb200_student* c, const bf16* x, int ldx, int rows, const float* g, const float* b, bf16* out, int ldo, cudaStream_t s);
// out[r, :d] (leading dimension dp) = (embed[tok] + pe[pos0 + r % L]) / sqrt(d), tok = tokens[(r / L) * tok_ld + pos0 + r % L]
// clamped to [0, vocab)
int s_embed(gitb200_student* c, const int* tokens, int tok_ld, int L, int pos0, int rows, bf16* out, cudaStream_t s);
// softmax(q k^T / sqrt(hd) + mask) v, one warp per (query row, head); query r sits at position pos0 + r % Lq.  causal: keys
// 0 .. pos0 + r % Lq; tokens != nullptr: key j of sequence b masked when tokens[b * tok_ld + j] == cfg.pad.  n_keys <= 128.
int s_attn(gitb200_student* c, const bf16* q, int ldq, int Lq, int pos0, const bf16* kv, int kv_rows, int ldkv, int k_off, int v_off,
           int n_keys, int causal, const int* tokens, int tok_ld, int rows, bf16* out, int ldo, cudaStream_t s);
// s_attn with dropout on the probabilities (distillation step only): out = (D o P) V, D the mask of site dr over the element
// index ((b * H + h) * Lq + i) * n_keys + j, b = r / Lq, i = r % Lq.  pos0 = 0.
int s_attn_dropout(gitb200_student* c, const bf16* q, int ldq, int Lq, const bf16* kv, int kv_rows, int ldkv, int k_off, int v_off,
                   int n_keys, int causal, const int* tokens, int tok_ld, int rows, bf16* out, int ldo, const SDrop& dr, cudaStream_t s);

// ---- distillation backward (student_train.cu)
// dst[c * R_pad + r] = src[r * ld_src + c] for r < R, c < C; zero for R <= r < R_pad or C <= c < C_pad
int t_transpose(gitb200_student* c, const bf16* src, int ld_src, int R, int C, bf16* dst, int R_pad, int C_pad, cudaStream_t s);
// out[c] = sum_r x[r, c], fp32, rows in order
int t_colsum(gitb200_student* c, const bf16* x, int ld, int R, int C, float* out, cudaStream_t s);
// dW [n_pad, k_pad] fp32 = dY^T X over R rows through the bf16 transposes tA [n_pad, round_up(R, 64)] and
// tB [k_pad, round_up(R, 64)] (X columns x_cols .. k_pad and rows R .. round_up(R, 64) are zero)
int t_weight_grad(gitb200_student* c, const bf16* dY, int ldy, int n_pad, const bf16* X, int ldx, int x_cols, int k_pad, int R, float* dW,
                  bf16* tA, bf16* tB, cudaStream_t s);
// LayerNorm backward over d_model columns (leading dimension dp): y = LN input, dx = d loss / d LN output;
// dy = d loss / d y, dgamma / dbeta = column sums; stats [2 * rows] fp32 scratch (mean, rstd per row)
int t_ln_bwd(gitb200_student* c, const bf16* y, const bf16* dx, int rows, const float* gamma, bf16* dy, float* dgamma, float* dbeta,
             float* stats, cudaStream_t s);
// attention backward, one CTA per (sequence, head) over B sequences of Lq queries and n_keys keys (<= 64 each); layouts as
// s_attn with pos0 = 0, dO at leading dimension dp; dq like q, dk / dv at dkv + dk_off / dv_off
int t_attn_bwd(gitb200_student* c, const bf16* q, int ldq, int Lq, const bf16* kv, int kv_rows, int ldkv, int k_off, int v_off, int n_keys,
               int causal, const int* tokens, int tok_ld, int B, const bf16* dO, bf16* dq, int lddq, bf16* dkv, int lddkv, int dk_off,
               int dv_off, cudaStream_t s);
// KL(batchmean)(log_softmax(s / T), softmax(t / T)) T^2 + CE(ignore_index 0)(s[:, :-1], tokens[:, 1:]) over B x L rows of
// vocab logits: dlogits bf16 [B * L, vp] (columns vocab .. vp zero); n_valid (1 int) and loss (2 * B * L floats: the rows'
// KL and CE parts) scratch; loss_out (3 floats) = (KL + CE, KL, CE), the parts summed in a fixed order.  No valid CE target:
// CE = 0 and no CE gradient.
int t_distill_loss(gitb200_student* c, const float* s_logits, int ld_s, const float* t_logits, int ld_t, const int* tokens, int B, int L,
                   float temperature, int* n_valid, bf16* dlogits, float* loss, float* loss_out, cudaStream_t s);
// dh[i] = 0 where !(h[i] > 0), i < n
int t_relu_bwd(gitb200_student* c, const bf16* h, bf16* dh, size_t n, cudaStream_t s);
// ---- dropout sites of the distillation step (student_train.cu); element index r * cols + c over the logical columns
// y = x + D o z (bf16, kept for the LayerNorm backward) and out = LN(y) * g + b over d_model columns (leading dimension dp),
// one warp per row; D = mask of site dr
int t_dropout_add_ln(gitb200_student* c, const bf16* x, const bf16* z, int rows, const float* g, const float* b, bf16* y, bf16* out,
                     const SDrop& dr, cudaStream_t s);
// h[r, c] *= D[r, c] in place for r < rows, c < cols (cols % 4 == 0), leading dimension ld
int t_dropout_inplace(gitb200_student* c, bf16* h, int ld, int rows, int cols, const SDrop& dr, cudaStream_t s);
// t_ln_bwd with a second output dz = D o dy (bf16 of the rounded dy), D = mask of site dr
int t_ln_bwd_dropout(gitb200_student* c, const bf16* y, const bf16* dx, int rows, const float* gamma, bf16* dy, bf16* dz, float* dgamma,
                     float* dbeta, float* stats, const SDrop& dr, cudaStream_t s);
// t_attn_bwd for out = (D o P) V: dV = (D o P)^T dO, dP = D o (dO V^T), dS = P o (dP - rowsum(P o dP)); D over the element
// index ((b * H + h) * Lq + i) * n_keys + j
int t_attn_bwd_dropout(gitb200_student* c, const bf16* q, int ldq, int Lq, const bf16* kv, int kv_rows, int ldkv, int k_off, int v_off,
                       int n_keys, int causal, const int* tokens, int tok_ld, int B, const bf16* dO, bf16* dq, int lddq, bf16* dkv, int lddkv,
                       int dk_off, int dv_off, const SDrop& dr, cudaStream_t s);
// ReLU backward through h' = D o relu(.): dh[i] = h'[i] > 0 ? dh[i] * inv_keep : 0, i < n (exact: where D = 0, h' = 0)
int t_relu_bwd_dropout(gitb200_student* c, const bf16* h, bf16* dh, size_t n, float inv_keep, cudaStream_t s);
// dembed[tok, :] = sum over the rows r with tokens[r] == tok (clamped to [0, vocab)), in row order, of dx[r, :d] / sqrt(d);
// rows of tokens that do not occur are left untouched
int t_embed_bwd(gitb200_student* c, const int* tokens, int rows, const bf16* dx, int ld, float* dembed, cudaStream_t s);

}  // namespace sdet

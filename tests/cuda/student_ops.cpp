// Test-only C entry points over the student decoder's kernel launchers (csrc/student_ops.h), so that the operator tests can
// run each forward and distillation-backward kernel on their own inputs: embedding, LayerNorm, attention (self, cross and the
// cached-decode layout), the loss, LayerNorm / attention / ReLU / embedding backward, column sums, transposes and the weight
// gradient.
//
// Host-only C++: it compiles no kernel, allocates nothing and makes no CUDA runtime call.  `h` is the gitb200_student* of a
// StudentCandidateV1 in training mode (its `_h`); the launchers read only its configuration and, for the forward kernels, its
// embedding and positional tables.  The caller owns every buffer, scratch included, and passes device pointers and a stream;
// every function returns the launcher's status (0 or a GITB200_ERR_* code).  Built and loaded by tests/op_modes_shim.py.
#include "student_ops.h"

using namespace sdet;

#define H ((gitb200_student*)h)
#define S ((cudaStream_t)stream)

extern "C" {

int sto_embed(void* h, const int* tokens, int tok_ld, int L, int pos0, int rows, void* out, void* stream) {
  return s_embed(H, tokens, tok_ld, L, pos0, rows, (bf16*)out, S);
}

int sto_ln(void* h, const void* x, int ldx, int rows, const float* g, const float* b, void* out, int ldo, void* stream) {
  return s_ln(H, (const bf16*)x, ldx, rows, g, b, (bf16*)out, ldo, S);
}

int sto_attn(void* h, const void* q, int ldq, int Lq, int pos0, const void* kv, int kv_rows, int ldkv, int k_off, int v_off, int n_keys,
             int causal, const int* tokens, int tok_ld, int rows, void* out, int ldo, void* stream) {
  return s_attn(H, (const bf16*)q, ldq, Lq, pos0, (const bf16*)kv, kv_rows, ldkv, k_off, v_off, n_keys, causal, tokens, tok_ld, rows,
                (bf16*)out, ldo, S);
}

int sto_transpose(void* h, const void* src, int ld_src, int R, int C, void* dst, int R_pad, int C_pad, void* stream) {
  return t_transpose(H, (const bf16*)src, ld_src, R, C, (bf16*)dst, R_pad, C_pad, S);
}

int sto_colsum(void* h, const void* x, int ld, int R, int C, float* out, void* stream) {
  return t_colsum(H, (const bf16*)x, ld, R, C, out, S);
}

int sto_weight_grad(void* h, const void* dY, int ldy, int n_pad, const void* X, int ldx, int x_cols, int k_pad, int R, float* dW, void* tA,
                    void* tB, void* stream) {
  return t_weight_grad(H, (const bf16*)dY, ldy, n_pad, (const bf16*)X, ldx, x_cols, k_pad, R, dW, (bf16*)tA, (bf16*)tB, S);
}

int sto_ln_bwd(void* h, const void* y, const void* dx, int rows, const float* gamma, void* dy, float* dgamma, float* dbeta, float* stats,
               void* stream) {
  return t_ln_bwd(H, (const bf16*)y, (const bf16*)dx, rows, gamma, (bf16*)dy, dgamma, dbeta, stats, S);
}

int sto_attn_bwd(void* h, const void* q, int ldq, int Lq, const void* kv, int kv_rows, int ldkv, int k_off, int v_off, int n_keys, int causal,
                 const int* tokens, int tok_ld, int B, const void* dO, void* dq, int lddq, void* dkv, int lddkv, int dk_off, int dv_off,
                 void* stream) {
  return t_attn_bwd(H, (const bf16*)q, ldq, Lq, (const bf16*)kv, kv_rows, ldkv, k_off, v_off, n_keys, causal, tokens, tok_ld, B,
                    (const bf16*)dO, (bf16*)dq, lddq, (bf16*)dkv, lddkv, dk_off, dv_off, S);
}

int sto_distill_loss(void* h, const float* s_logits, int ld_s, const float* t_logits, int ld_t, const int* tokens, int B, int L,
                     float temperature, int* n_valid, void* dlogits, float* loss, float* loss_out, void* stream) {
  return t_distill_loss(H, s_logits, ld_s, t_logits, ld_t, tokens, B, L, temperature, n_valid, (bf16*)dlogits, loss, loss_out, S);
}

int sto_relu_bwd(void* h, const void* act, void* dh, long long n, void* stream) {
  return t_relu_bwd(H, (const bf16*)act, (bf16*)dh, (size_t)n, S);
}

int sto_embed_bwd(void* h, const int* tokens, int rows, const void* dx, int ld, float* dembed, void* stream) {
  return t_embed_bwd(H, tokens, rows, (const bf16*)dx, ld, dembed, S);
}

}  // extern "C"

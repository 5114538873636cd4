// Test-only C entry points over the student decoder's dropout launchers (csrc/student_ops.h), so that the operator tests can
// run each dropout kernel of the distillation step on their own inputs: attention forward and backward with dropout on the
// probabilities, the fused dropout-add-LayerNorm, the in-place mask and the dropout-ReLU backward.
//
// Host-only C++, like tests/cuda/student_ops.cpp: no kernel, no allocation, no CUDA runtime call.  `h` is the gitb200_student*
// of a StudentCandidateV1 in training mode; (seed, step, site, p) name the mask (philox.cuh, dropout_scale).  Built and loaded
// by tests/op_modes_shim.py's load().
#include "student_ops.h"

using namespace sdet;

#define H ((gitb200_student*)h)
#define S ((cudaStream_t)stream)

static SDrop mask(unsigned long long seed, long long step, int site, float p) {
  return SDrop{seed, (unsigned)step, (unsigned)site, p, 1.f / (1.f - p)};
}

extern "C" {

int sdo_attn(void* h, const void* q, int ldq, int Lq, const void* kv, int kv_rows, int ldkv, int k_off, int v_off, int n_keys, int causal,
             const int* tokens, int tok_ld, int rows, void* out, int ldo, unsigned long long seed, long long step, int site, float p,
             void* stream) {
  return s_attn_dropout(H, (const bf16*)q, ldq, Lq, (const bf16*)kv, kv_rows, ldkv, k_off, v_off, n_keys, causal, tokens, tok_ld, rows,
                        (bf16*)out, ldo, mask(seed, step, site, p), S);
}

int sdo_attn_bwd(void* h, const void* q, int ldq, int Lq, const void* kv, int kv_rows, int ldkv, int k_off, int v_off, int n_keys, int causal,
                 const int* tokens, int tok_ld, int B, const void* dO, void* dq, int lddq, void* dkv, int lddkv, int dk_off, int dv_off,
                 unsigned long long seed, long long step, int site, float p, void* stream) {
  return t_attn_bwd_dropout(H, (const bf16*)q, ldq, Lq, (const bf16*)kv, kv_rows, ldkv, k_off, v_off, n_keys, causal, tokens, tok_ld, B,
                            (const bf16*)dO, (bf16*)dq, lddq, (bf16*)dkv, lddkv, dk_off, dv_off, mask(seed, step, site, p), S);
}

int sdo_add_ln(void* h, const void* x, const void* z, int rows, const float* g, const float* b, void* y, void* out, unsigned long long seed,
               long long step, int site, float p, void* stream) {
  return t_dropout_add_ln(H, (const bf16*)x, (const bf16*)z, rows, g, b, (bf16*)y, (bf16*)out, mask(seed, step, site, p), S);
}

int sdo_inplace(void* h, void* x, int ld, int rows, int cols, unsigned long long seed, long long step, int site, float p, void* stream) {
  return t_dropout_inplace(H, (bf16*)x, ld, rows, cols, mask(seed, step, site, p), S);
}

int sdo_ln_bwd(void* h, const void* y, const void* dx, int rows, const float* gamma, void* dy, void* dz, float* dgamma, float* dbeta,
               float* stats, unsigned long long seed, long long step, int site, float p, void* stream) {
  return t_ln_bwd_dropout(H, (const bf16*)y, (const bf16*)dx, rows, gamma, (bf16*)dy, (bf16*)dz, dgamma, dbeta, stats,
                          mask(seed, step, site, p), S);
}

int sdo_relu_bwd(void* h, const void* act, void* dh, long long n, float p, void* stream) {
  return t_relu_bwd_dropout(H, (const bf16*)act, (bf16*)dh, (size_t)n, 1.f / (1.f - p), S);
}

}  // extern "C"

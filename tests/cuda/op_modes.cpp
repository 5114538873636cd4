// Test-only C entry points over the internal launchers of libgitb200.so (csrc/kernels.h), so that the operator tests can reach
// every mode the engine's launch sequences use: row remap + periodic residual, fp32-only output, in-place residual, leading
// dimensions wider than the rows, LayerNorm-on-load and K/V scatter in the skinny GEMM, LayerNorm addend / output-row table /
// row statistics, and the decode attention in the engine's own layouts.  The public C ABI (gitb200_op_*) sets only the plain
// subset of each argument struct.
//
// Host-only C++: it compiles no kernel, allocates nothing and makes no CUDA runtime call.  The caller owns every buffer
// (including the text-attention split workspace) and passes device pointers and a stream; every function returns the
// launcher's cudaError_t as an int.  Built and loaded by tests/op_modes_shim.py.
#include "kernels.h"

extern "C" {

int opm_gemm(const void* A, int lda, const void* W, int ldw, int M, int N, int K, const float* bias, const void* residual, int ldr,
             int res_periodic, int act, void* out, int ldo, float* out_f32, int ldo32, int gin, int gout, int goff,
             const float* lnl_gamma, const float* lnl_beta, float lnl_eps, void* lnl_out, int lnl_ldo, void* sc_kv, int sc_q_width,
             int sc_kv_width, const int* sc_pos, int sc_pos_const, int sc_slot_div, int sc_n_slots, int force_bn, void* stream) {
  GemmArgs g;
  g.A = (const bf16*)A; g.lda = lda; g.W = (const bf16*)W; g.ldw = ldw; g.M = M; g.N = N; g.K = K; g.bias = bias;
  g.residual = (const bf16*)residual; g.ldr = ldr; g.res_periodic = res_periodic; g.act = act;
  g.out = (bf16*)out; g.ldo = ldo; g.out_f32 = out_f32; g.ldo32 = ldo32; g.gin = gin; g.gout = gout; g.goff = goff;
  g.lnl_gamma = lnl_gamma; g.lnl_beta = lnl_beta; g.lnl_eps = lnl_eps; g.lnl_out = (bf16*)lnl_out; g.lnl_ldo = lnl_ldo;
  g.sc_kv = (bf16*)sc_kv; g.sc_q_width = sc_q_width; g.sc_kv_width = sc_kv_width; g.sc_pos = sc_pos; g.sc_pos_const = sc_pos_const;
  g.sc_slot_div = sc_slot_div; g.sc_n_slots = sc_n_slots;
  return (int)gemm_bf16(g, (cudaStream_t)stream, force_bn);
}

int opm_layernorm(const void* x, int ldx, int rows, int cols, const float* gamma, const float* beta, float eps, const float* addend,
                  int add_group, int add_period, void* out, int ldo, float* out_f32, int ldo32, float* stats_out, int stats_slots,
                  const int* out_row_base, int out_group, void* stream) {
  LayerNormArgs a;
  a.x = (const bf16*)x; a.ldx = ldx; a.rows = rows; a.cols = cols; a.gamma = gamma; a.beta = beta; a.eps = eps;
  a.addend = addend; a.add_group = add_group; a.add_period = add_period; a.out = (bf16*)out; a.ldo = ldo;
  a.out_f32 = out_f32; a.ldo32 = ldo32; a.stats_out = stats_out; a.stats_slots = stats_slots;
  a.out_row_base = out_row_base; a.out_group = out_group;
  return (int)layernorm_bf16(a, (cudaStream_t)stream);
}

int opm_text_attention(const void* q, int ldq, int n_clips, int rows_per_clip, int heads, const void* vis_kv, int ld_vis, int k_off,
                       int v_off, int Nv, const void* txt_kv, int txt_slots, int text_slot_is_clip, const int* anc, int anc_ld,
                       const int* n_text, int n_text_const, int max_text, float scale, void* out, int ldo, float* partial, int splits,
                       void* stream) {
  TextAttnArgs a;
  a.q = (const bf16*)q; a.ldq = ldq; a.n_clips = n_clips; a.rows_per_clip = rows_per_clip; a.heads = heads;
  a.vis_kv = (const bf16*)vis_kv; a.ld_vis = ld_vis; a.k_off = k_off; a.v_off = v_off; a.Nv = Nv;
  a.txt_kv = (const bf16*)txt_kv; a.txt_slots = txt_slots; a.text_slot_is_clip = text_slot_is_clip;
  a.anc = anc; a.anc_ld = anc_ld; a.n_text = n_text; a.n_text_const = n_text_const; a.max_text = max_text;
  a.scale = scale; a.out = (bf16*)out; a.ldo = ldo; a.partial = partial; a.splits = splits;
  return (int)text_attention(a, (cudaStream_t)stream);
}

long long opm_text_attention_workspace_floats(int n_rows, int heads, int splits) {
  return (long long)text_attention_workspace_floats(n_rows, heads, splits);
}

int opm_store_text_kv(const void* qkv, int ld_qkv, int n_rows, int kv_width, int q_width, const int* pos, int pos_const, int slot_div,
                      int n_slots, void* txt_kv, void* stream) {
  return (int)store_text_kv((const bf16*)qkv, ld_qkv, n_rows, kv_width, q_width, pos, pos_const, slot_div, n_slots, (bf16*)txt_kv,
                            (cudaStream_t)stream);
}

}  // extern "C"

// Internal state of the student decoder (shared by student.cu: inference, and student_train.cu: the distillation step).
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <stdarg.h>
#include <stdio.h>

#include <map>
#include <string>
#include <vector>

#include "../../include/gitb200.h"
#include "common.cuh"
#include "kernels.h"
#include "philox.cuh"
#include "student_ops.h"

namespace sdet {

struct SLayer {
  bf16 *w_sa_in, *w_sa_out, *w_ca_q, *w_ca_kv, *w_ca_out, *w_ff1, *w_ff2;
  float *b_sa_in, *b_sa_out, *b_ca_q, *b_ca_kv, *b_ca_out, *b_ff1, *b_ff2;
  float *n1_g, *n1_b, *n2_g, *n2_b, *n3_g, *n3_b;
};
struct RawW {
  float* p = nullptr;
  std::vector<int64_t> shape;
  size_t numel() const {
    size_t n = 1;
    for (auto d : shape) n *= (size_t)d;
    return n;
  }
};
template <typename T>
struct SBuf {
  T* p = nullptr;
  size_t cap = 0;
};
struct STrain;  // student_train.cu

}  // namespace sdet

struct gitb200_student {
  gitb200_student_config cfg;
  int device = 0;
  std::string err;
  bool finalized = false;
  std::map<std::string, sdet::RawW> raw;
  std::vector<void*> allocs;
  int dp = 0, fp = 0, vp = 0, hd = 0;  // padded d_model / d_ffn / vocab, head dim
  float *embed = nullptr, *pe = nullptr, *b_vocab = nullptr;
  bf16* w_vocab = nullptr;
  std::vector<sdet::SLayer> layers;
  // workspaces
  sdet::SBuf<bf16> x, y, a, q2, h, mem;
  std::vector<sdet::SBuf<bf16>> cache, memkv;
  sdet::SBuf<float> logits;
  sdet::SBuf<int> toks;
  // distillation training state (student_train.cu); nullptr until gitb200_student_train_begin
  bool keep_raw = false;  // finalize keeps the staged fp32 weights: the fp32 master copy of the optimizer is built from them
  sdet::STrain* train = nullptr;
};

namespace sdet {

int sfail(gitb200_student* c, int code, const char* fmt, ...);
#define S_CUDA_OK(c, expr)                                                                                            \
  do {                                                                                                                \
    cudaError_t e_ = (expr);                                                                                          \
    if (e_ != cudaSuccess)                                                                                            \
      return sdet::sfail(c, GITB200_ERR_CUDA, "%s failed: %s [%s] (%s:%d)", #expr, cudaGetErrorString(e_), gemm_last_error(), \
                         __FILE__, __LINE__);                                                                         \
  } while (0)
#define S_TRY(expr)      \
  do {                   \
    int r_ = (expr);     \
    if (r_) return r_;   \
  } while (0)

template <typename T>
int sensure(gitb200_student* c, SBuf<T>& b, size_t n) {
  if (b.cap >= n) return 0;
  if (b.p) S_CUDA_OK(c, cudaFree(b.p));
  b.p = nullptr;
  b.cap = 0;
  S_CUDA_OK(c, cudaMalloc(&b.p, n * sizeof(T)));
  S_CUDA_OK(c, cudaMemset(b.p, 0, n * sizeof(T)));  // padded columns are never written by the glue kernels: keep them finite
  b.cap = n;
  return 0;
}
inline int round_up(int v, int m) { return (v + m - 1) / m * m; }

// the kernel launchers (s_*: student.cu, t_*: student_train.cu) are declared in student_ops.h
void student_train_destroy(gitb200_student* c);

}  // namespace sdet

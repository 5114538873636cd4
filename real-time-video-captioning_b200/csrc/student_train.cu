// Distillation training step of the student decoder (SURVEY 8f rank 3, BASELINE.json configs[4]):
// DistillationTrainer.training_step of the reference (/root/reference/src/models/model.py:880-983) for the decoder half of
// StudentCandidateV1 -- forward_decoder(y, memory) (model.py:135-154), the loss
//     KLDivLoss(batchmean)(log_softmax(student / T), softmax(teacher / T)) * T^2      (model.py:922-928)
//   + CrossEntropyLoss(ignore_index = 0)(student[:, :-1], y[:, 1:])                    (model.py:930-935, :983)
// its backward pass through the vocabulary head, the post-LN nn.TransformerDecoder layers (self-attention under the causal +
// padding mask, cross-attention to the memory tokens, ReLU feed-forward) and the embedding, and torch.optim.Adam
// (model.py:1105).  The image encoder that produces `memory` (timm TinyViT) is not part of this library: memory is an input and
// d loss / d memory is an output, so an external encoder can continue the backward pass.
//
// Layout: ONE flat fp32 parameter vector P (master weights, padded to the GEMM tile multiples the inference path uses:
// d_model 576 -> 640 etc.; padding stays exactly zero), a gradient vector G of the same layout supplied by the caller (a
// torch tensor, so that torch.distributed can all-reduce it in place: reference = Lightning DDP, train.py:217-221), and the
// Adam moments.  The vocabulary head comes first in the layout: its gradients are complete after phase 0 of the backward
// pass, and the caller starts their all-reduce while phase 1 (the decoder layers and the embedding) is still running.
// Every contraction -- forward, dX = dY W and dW = dY^T X -- runs on the tcgen05 GEMM of the inference path (C = A W^T with
// both operands K-major): dX uses a transposed bf16 copy of W kept next to W, dW uses explicit bf16 transposes of the two
// (small: B*L = 160 rows) activation matrices.  Activations and activation gradients are bf16, weight gradients fp32.
// Dropout (nn.TransformerDecoderLayer's six sites per layer, p = 0.3 in config.py:83) is opt-in: gitb200_student_train_set_dropout
// gives p and a Philox seed.  The masks are regenerated in the backward pass, never stored (mask: philox.cuh, dropout_scale);
// where dropout is on, the three residual sites' GEMMs write z without the residual and dropout_add_ln_kernel forms x + D o z.
#include "student_internal.cuh"

using namespace sdet;

namespace sdet {

struct PEntry {
  std::string name;   // reference state-dict key
  int src_row0;       // first row of the torch tensor this block holds (fused in_proj weights are split into q | k | v blocks)
  int rows, cols;     // block shape in the torch tensor (vectors: cols = 1)
  int rows_pad, cols_pad;
  size_t off;         // offset in the flat vectors
  // bf16 operand copies refreshed after every optimizer step (matrices only)
  bf16* w = nullptr;  // [rows_pad, w_ld] row-major, first w_cols columns
  int w_ld = 0, w_cols = 0;
  bf16* wt = nullptr; // transposed: element (r, c) at wt[c * wt_ld + r]
  int wt_ld = 0;
};

struct LayerAct {
  SBuf<bf16> x0, qkv, a, y1, x1, q2, memkv, a2, y2, x2, h, y3;
};
struct LayerT {
  bf16 *sa_in = nullptr, *sa_out = nullptr, *ca_q = nullptr, *ca_kv = nullptr, *ca_out = nullptr, *ff1 = nullptr, *ff2 = nullptr;
};

struct STrain {
  std::vector<PEntry> entries;
  size_t n_floats = 0, head_floats = 0;
  float *P = nullptr, *M1 = nullptr, *M2 = nullptr;
  long long step = 0;
  float lr = 1e-4f, beta1 = 0.9f, beta2 = 0.999f, eps = 1e-8f;
  std::vector<LayerT> lt;
  bf16* wt_vocab = nullptr;
  std::vector<LayerAct> acts;
  SBuf<bf16> xo, mem, dlogits, tA, tB, dx, dy, da, dqkv, dh, dmemkv, dmem;
  SBuf<bf16> z, dz;  // dropout only: the residual sites' dropped addend (forward scratch) and its gradient D o dy
  // dropout (off while drop_p == 0): drop_step counts the forwards that applied it; the backward pass replays fwd_step's masks
  float drop_p = 0.f;
  unsigned long long drop_seed = 0;
  long long drop_step = 0, fwd_step = 0;
  bool fwd_drop = false;
  SBuf<float> logits, stats, loss;
  SBuf<int> nvalid, toks;
  int B = 0, L = 0, M = 0;
  bool have_forward = false, have_head = false;
};

}  // namespace sdet

namespace {

constexpr int T_MAX_SEQ = 64;  // training sequences / memory tokens per clip (reference: 20 caption tokens, 6 memory tokens)

// ------------------------------------------------------------------ kernels
// dst[c * ld_dst + r] = (r < R && c < C) ? src[r * ld_src + c] : 0   for c < C_pad, r < R_pad  (bf16 transpose with zero padding)
__global__ void transpose_pad_kernel(const bf16* __restrict__ src, int ld_src, int R, int C, bf16* __restrict__ dst, int ld_dst, int R_pad,
                                     int C_pad) {
  __shared__ bf16 tile[32][33];
  const int c0 = blockIdx.x * 32, r0 = blockIdx.y * 32;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int r = r0 + i, c = c0 + threadIdx.x;
    tile[i][threadIdx.x] = (r < R && c < C) ? src[(size_t)r * ld_src + c] : __float2bfloat16(0.f);
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int c = c0 + i, r = r0 + threadIdx.x;
    if (c < C_pad && r < R_pad) dst[(size_t)c * ld_dst + r] = tile[threadIdx.x][i];
  }
}

// out[c] = sum_r x[r, c]  (bias gradients; R is a few hundred rows)
__global__ void colsum_kernel(const bf16* __restrict__ x, int ld, int R, int C, float* __restrict__ out) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  float s = 0.f;
  for (int r = 0; r < R; ++r) s += __bfloat162float(x[(size_t)r * ld + c]);
  out[c] = s;
}

// n_valid = #{(b, i) : i >= 1, tokens[b, i] != ignore}  -- the denominator of CrossEntropyLoss(ignore_index) (model.py:931-935)
__global__ void count_valid_kernel(const int* __restrict__ tokens, int B, int L, int ignore, int* __restrict__ n_valid) {
  __shared__ int acc;
  if (threadIdx.x == 0) acc = 0;
  __syncthreads();
  int n = 0;
  for (int i = threadIdx.x; i < B * L; i += blockDim.x)
    if (i % L >= 1 && tokens[i] != ignore) ++n;
  atomicAdd(&acc, n);
  __syncthreads();
  if (threadIdx.x == 0) *n_valid = acc;
}

__device__ __forceinline__ float block_reduce(float v, float* sh, bool is_max) {
  v = is_max ? warp_max(v) : warp_sum(v);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
  __syncthreads();
  if (lane == 0) sh[warp] = v;
  __syncthreads();
  float r = sh[0];
  for (int w = 1; w < nw; ++w) r = is_max ? fmaxf(r, sh[w]) : r + sh[w];
  return r;
}

// One CTA per row r = (b, i): KL(batchmean) * T^2 + CE(ignore_index) and d loss / d student-logits (model.py:922-935, :983).
//   loss[r] = KL_row / B * T^2, loss[R + r] = CE_row / n_valid (0 without a CE target);
//   dlogits[r, v] = T (p_s - p_t) / B + [CE row] (p_s1 - onehot) / n_valid  where p_s = softmax(s / T), p_t = softmax(t / T),
//   p_s1 = softmax(s).  loss_total_kernel sums the rows' parts in a fixed order.
__global__ void __launch_bounds__(256) distill_loss_kernel(const float* __restrict__ s_logits, int ld_s, const float* __restrict__ t_logits,
                                                           int ld_t, const int* __restrict__ tokens, int B, int L, int V, int Vp, int ignore,
                                                           float temperature, const int* __restrict__ n_valid, bf16* __restrict__ dlogits,
                                                           float* __restrict__ loss) {
  __shared__ float sh[8];
  const int r = blockIdx.x, b = r / L, i = r % L;
  const float* s = s_logits + (size_t)r * ld_s;
  const float* t = t_logits + (size_t)r * ld_t;
  const float invT = 1.f / temperature;
  float ms = -INFINITY, mt = -INFINITY;
  for (int v = threadIdx.x; v < V; v += blockDim.x) {
    ms = fmaxf(ms, s[v]);
    mt = fmaxf(mt, t[v]);
  }
  ms = block_reduce(ms, sh, true);
  mt = block_reduce(mt, sh, true);
  float zs = 0.f, zt = 0.f, z1 = 0.f;
  for (int v = threadIdx.x; v < V; v += blockDim.x) {
    zs += __expf((s[v] - ms) * invT);
    zt += __expf((t[v] - mt) * invT);
    z1 += __expf(s[v] - ms);
  }
  zs = block_reduce(zs, sh, false);
  zt = block_reduce(zt, sh, false);
  z1 = block_reduce(z1, sh, false);
  const float ls = logf(zs), lt = logf(zt), l1 = logf(z1);
  const int tgt = (i + 1 < L) ? tokens[b * L + i + 1] : ignore;
  const bool ce_row = (i + 1 < L) && tgt != ignore;
  const int nv = *n_valid;
  const float w_kl = temperature / (float)B, w_ce = ce_row && nv > 0 ? 1.f / (float)nv : 0.f;
  float kl = 0.f;
  for (int v = threadIdx.x; v < Vp; v += blockDim.x) {
    float g = 0.f;
    if (v < V) {
      const float lps = (s[v] - ms) * invT - ls, lpt = (t[v] - mt) * invT - lt;
      const float ps = __expf(lps), pt = __expf(lpt);
      if (pt > 0.f) kl += pt * (lpt - lps);
      g = w_kl * (ps - pt);
      if (ce_row) g += w_ce * (__expf(s[v] - ms - l1) - (v == tgt ? 1.f : 0.f));
    }
    dlogits[(size_t)r * Vp + v] = __float2bfloat16(g);
  }
  kl = block_reduce(kl, sh, false);
  if (threadIdx.x == 0) {
    loss[r] = kl * temperature * temperature / (float)B;
    loss[gridDim.x + r] = (ce_row && nv > 0) ? -(s[tgt] - ms - l1) / (float)nv : 0.f;
  }
}

// LayerNorm backward, one warp per row: y = LN input (pre-norm), dx = gradient of the LN output.
//   dy = rstd * (g - mean(g) - xhat * mean(g * xhat)),  g = dx * gamma;  stats[r] = (mean, rstd) for the parameter-gradient kernel
//   DROP: also dz = D o dy (D = dropout mask of `site`, element index warp * cols + c): the gradient of the dropped addend
template <bool DROP>
__global__ void ln_bwd_kernel(const bf16* __restrict__ y, const bf16* __restrict__ dx, int ld, int rows, int cols,
                              const float* __restrict__ gamma, float eps, bf16* __restrict__ dy, float* __restrict__ stats,
                              bf16* __restrict__ dz, SDrop site) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= rows) return;
  const bf16* yr = y + (size_t)warp * ld;
  const bf16* dr = dx + (size_t)warp * ld;
  float s = 0.f;
  for (int c = lane; c < cols; c += 32) s += __bfloat162float(yr[c]);
  const float mean = warp_sum(s) / (float)cols;
  float q = 0.f;
  for (int c = lane; c < cols; c += 32) {
    const float v = __bfloat162float(yr[c]) - mean;
    q += v * v;
  }
  const float rstd = rsqrtf(warp_sum(q) / (float)cols + eps);
  float s1 = 0.f, s2 = 0.f;
  for (int c = lane; c < cols; c += 32) {
    const float xh = (__bfloat162float(yr[c]) - mean) * rstd, g = __bfloat162float(dr[c]) * gamma[c];
    s1 += g;
    s2 += g * xh;
  }
  const float c1 = warp_sum(s1) / (float)cols, c2 = warp_sum(s2) / (float)cols;
  for (int c = lane; c < cols; c += 32) {
    const float xh = (__bfloat162float(yr[c]) - mean) * rstd, g = __bfloat162float(dr[c]) * gamma[c];
    const bf16 v = __float2bfloat16(rstd * (g - c1 - xh * c2));
    dy[(size_t)warp * ld + c] = v;
    if constexpr (DROP)
      dz[(size_t)warp * ld + c] =
          __float2bfloat16(__bfloat162float(v) * dropout_scale(site.seed, site.step, site.site, (unsigned)(warp * cols + c), site.p, site.inv_keep));
  }
  if (lane == 0) {
    stats[2 * warp] = mean;
    stats[2 * warp + 1] = rstd;
  }
}
// dgamma[c] = sum_r dx[r, c] * xhat[r, c], dbeta[c] = sum_r dx[r, c]   (one thread per column: deterministic)
__global__ void ln_param_grad_kernel(const bf16* __restrict__ y, const bf16* __restrict__ dx, int ld, int rows, int cols,
                                     const float* __restrict__ stats, float* __restrict__ dgamma, float* __restrict__ dbeta) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= cols) return;
  float dg = 0.f, db = 0.f;
  for (int r = 0; r < rows; ++r) {
    const float d = __bfloat162float(dx[(size_t)r * ld + c]);
    dg += d * (__bfloat162float(y[(size_t)r * ld + c]) - stats[2 * r]) * stats[2 * r + 1];
    db += d;
  }
  dgamma[c] = dg;
  dbeta[c] = db;
}

// dh[r, c] = h[r, c] > 0 ? dh[r, c] : 0   (ReLU backward; h is the stored post-activation)
__global__ void relu_bwd_kernel(const bf16* __restrict__ h, bf16* __restrict__ dh, size_t n) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n && !(__bfloat162float(h[i]) > 0.f)) dh[i] = __float2bfloat16(0.f);
}
// dh[r, c] = h'[r, c] > 0 ? dh[r, c] * inv_keep : 0   (h' = D o relu(.), the stored post-dropout activation)
__global__ void relu_bwd_dropout_kernel(const bf16* __restrict__ h, bf16* __restrict__ dh, size_t n, float inv_keep) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dh[i] = __bfloat162float(h[i]) > 0.f ? __float2bfloat16(__bfloat162float(dh[i]) * inv_keep) : __float2bfloat16(0.f);
}

// h[r, c] *= D[r, c] for c < cols (cols % 4 == 0): one thread per 4 consecutive elements, one Philox call each
__global__ void dropout_inplace_kernel(bf16* __restrict__ h, int ld, int rows, int cols, SDrop dr) {
  const size_t g = (size_t)blockIdx.x * blockDim.x + threadIdx.x, quads = (size_t)rows * (cols >> 2);
  if (g >= quads) return;
  const unsigned idx = (unsigned)(g * 4);
  const int r = (int)(idx / cols), c = (int)(idx % cols);
  const Philox4 w = dropout_words(dr.seed, dr.step, dr.site, idx);
  bf16* p = h + (size_t)r * ld + c;
  for (int k = 0; k < 4; ++k) p[k] = __float2bfloat16(__bfloat162float(p[k]) * dropout_keep(w.x[k], dr.p, dr.inv_keep));
}

// y = x + D o z (bf16), out = LN(y) * gamma + beta over `cols` columns (cols % 4 == 0); one warp per row, each lane owns
// groups of 4 consecutive columns (one Philox call each).  The statistics are those of student_ln_kernel on the stored y.
__global__ void dropout_add_ln_kernel(const bf16* __restrict__ x, const bf16* __restrict__ z, int ld, int rows, int cols,
                                      const float* __restrict__ gamma, const float* __restrict__ beta, float eps, bf16* __restrict__ y,
                                      bf16* __restrict__ out, SDrop dr) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= rows) return;
  const size_t row = (size_t)warp * ld;
  for (int c = 4 * lane; c < cols; c += 128) {
    const Philox4 w = dropout_words(dr.seed, dr.step, dr.site, (unsigned)(warp * cols + c));
    for (int k = 0; k < 4; ++k)
      y[row + c + k] = __float2bfloat16(__bfloat162float(x[row + c + k]) +
                                        __bfloat162float(z[row + c + k]) * dropout_keep(w.x[k], dr.p, dr.inv_keep));
  }
  __syncwarp();
  const bf16* yr = y + row;
  float s = 0.f;
  for (int c = lane; c < cols; c += 32) s += __bfloat162float(yr[c]);
  const float mean = warp_sum(s) / (float)cols;
  float q = 0.f;
  for (int c = lane; c < cols; c += 32) {
    const float v = __bfloat162float(yr[c]) - mean;
    q += v * v;
  }
  const float rstd = rsqrtf(warp_sum(q) / (float)cols + eps);
  for (int c = lane; c < cols; c += 32) out[row + c] = __float2bfloat16((__bfloat162float(yr[c]) - mean) * rstd * gamma[c] + beta[c]);
}

// Attention backward for one (sequence b, head h): recomputes P = softmax(scale Q K^T + mask) and returns dQ, dK, dV.
//   q row (b * Lq + i) at q[.. * ldq + h * hd]; key / value j at kv[(b * kv_rows + j) * ldkv + {k_off, v_off} + h * hd]
//   dO like the forward output; dq like q (leading dimension lddq); dk / dv like k / v in dkv (lddkv, dk_off, dv_off)
//   causal: key j visible to query i iff j <= i; tokens != nullptr: key j masked when tokens[b * tok_ld + j] == pad
//   DROP: the forward was (D o P) V, D the dropout mask of site dr over ((b * H + h) * Lq + i) * n_keys + j (kept in shared
//   memory): dV = (D o P)^T dO, dP = D o (dO V^T), dS = P o (dP - rowsum(P o dP)) with P the undropped probabilities
template <bool DROP>
__global__ void __launch_bounds__(128) attn_bwd_kernel(const bf16* __restrict__ q, int ldq, int Lq, const bf16* __restrict__ kv, int kv_rows,
                                                       int ldkv, int k_off, int v_off, int n_keys, int causal,
                                                       const int* __restrict__ tokens, int tok_ld, int pad, int hd, float scale,
                                                       const bf16* __restrict__ dO, int lddo, bf16* __restrict__ dq, int lddq,
                                                       bf16* __restrict__ dkv, int lddkv, int dk_off, int dv_off, SDrop dr) {
  extern __shared__ float sm[];
  const int b = blockIdx.x, h = blockIdx.y, tid = threadIdx.x, nt = blockDim.x;
  const int hs = hd + 1, ps = n_keys + 1;
  float* Q = sm;                    // [Lq][hs]
  float* K = Q + Lq * hs;           // [n_keys][hs]
  float* Vv = K + n_keys * hs;      // [n_keys][hs]
  float* G = Vv + n_keys * hs;      // [Lq][hs]   dO
  float* P = G + Lq * hs;           // [Lq][ps]
  float* S = P + Lq * ps;           // [Lq][ps]   dP, then dS
  float* D = S + Lq * ps;           // [Lq][ps]   dropout scales (DROP only)
  for (int e = tid; e < Lq * hd; e += nt) {
    const int i = e / hd, c = e % hd;
    Q[i * hs + c] = __bfloat162float(q[(size_t)(b * Lq + i) * ldq + h * hd + c]);
    G[i * hs + c] = __bfloat162float(dO[(size_t)(b * Lq + i) * lddo + h * hd + c]);
  }
  for (int e = tid; e < n_keys * hd; e += nt) {
    const int j = e / hd, c = e % hd;
    const bf16* row = kv + (size_t)(b * kv_rows + j) * ldkv + h * hd + c;
    K[j * hs + c] = __bfloat162float(row[k_off]);
    Vv[j * hs + c] = __bfloat162float(row[v_off]);
  }
  __syncthreads();
  for (int e = tid; e < Lq * n_keys; e += nt) {
    const int i = e / n_keys, j = e % n_keys;
    float s = 0.f, g = 0.f;
    for (int c = 0; c < hd; ++c) {
      s = fmaf(Q[i * hs + c], K[j * hs + c], s);
      g = fmaf(G[i * hs + c], Vv[j * hs + c], g);
    }
    const bool masked = (causal && j > i) || (tokens != nullptr && tokens[(size_t)b * tok_ld + j] == pad);
    P[i * ps + j] = masked ? -INFINITY : s * scale;
    if constexpr (DROP) {
      const float m = dropout_scale(dr.seed, dr.step, dr.site, (unsigned)(((b * gridDim.y + h) * Lq + i) * n_keys + j), dr.p, dr.inv_keep);
      D[i * ps + j] = m;
      S[i * ps + j] = g * m;  // dP of the undropped probabilities
    } else {
      S[i * ps + j] = g;  // dP
    }
  }
  __syncthreads();
  for (int i = tid; i < Lq; i += nt) {
    float mx = -INFINITY;
    for (int j = 0; j < n_keys; ++j) mx = fmaxf(mx, P[i * ps + j]);
    float z = 0.f;
    for (int j = 0; j < n_keys; ++j) {
      const float p = __expf(P[i * ps + j] - mx);
      P[i * ps + j] = p;
      z += p;
    }
    const float inv = 1.f / z;
    float dsum = 0.f;
    for (int j = 0; j < n_keys; ++j) {
      const float p = P[i * ps + j] * inv;
      P[i * ps + j] = p;
      dsum += p * S[i * ps + j];
    }
    for (int j = 0; j < n_keys; ++j) S[i * ps + j] = P[i * ps + j] * (S[i * ps + j] - dsum);  // dS
  }
  __syncthreads();
  for (int e = tid; e < Lq * hd; e += nt) {
    const int i = e / hd, c = e % hd;
    float a = 0.f;
    for (int j = 0; j < n_keys; ++j) a = fmaf(S[i * ps + j], K[j * hs + c], a);
    dq[(size_t)(b * Lq + i) * lddq + h * hd + c] = __float2bfloat16(a * scale);
  }
  for (int e = tid; e < n_keys * hd; e += nt) {
    const int j = e / hd, c = e % hd;
    float dk = 0.f, dv = 0.f;
    for (int i = 0; i < Lq; ++i) {
      dk = fmaf(S[i * ps + j], Q[i * hs + c], dk);
      dv = fmaf(DROP ? P[i * ps + j] * D[i * ps + j] : P[i * ps + j], G[i * hs + c], dv);
    }
    bf16* row = dkv + (size_t)(b * kv_rows + j) * lddkv + h * hd + c;
    row[dk_off] = __float2bfloat16(dk * scale);
    row[dv_off] = __float2bfloat16(dv);
  }
}

// d embed[tok, c] = sum over the rows r with tok(r) == tok of dx0[r, c] / sqrt(d)   (model.py:144-148: the embedding sum is divided
// by sqrt(d) after adding pe).  One CTA per row; the CTA of a token's first row sums that token's rows in row order and stores
// the result (every token repeats: CLS starts each sequence), so the gradient does not depend on block scheduling.  The rows
// of the token are gathered, in order, 32 * EMB_WARPS at a time into a shared list (ballot compaction); the column loop then
// reads only those rows.  acc: d floats of dynamic shared memory, one column per thread and pass.
constexpr int EMB_WARPS = 4;
__global__ void __launch_bounds__(32 * EMB_WARPS) embed_bwd_kernel(const int* __restrict__ tokens, int rows, const bf16* __restrict__ dx,
                                                                   int ld, int d, int vocab, float inv_sqrt_d, float* __restrict__ dembed) {
  extern __shared__ float acc[];
  __shared__ int list[32 * EMB_WARPS];
  __shared__ int wcnt[EMB_WARPS];
  const int r = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (r >= rows) return;
  const int tok = min(max(tokens[r], 0), vocab - 1);
  bool seen = false;
  for (int j = tid; j < r && !seen; j += blockDim.x) seen = min(max(tokens[j], 0), vocab - 1) == tok;
  if (__syncthreads_or(seen)) return;
  for (int c = tid; c < d; c += blockDim.x) acc[c] = 0.f;
  for (int base = r; base < rows; base += blockDim.x) {
    const int j = base + tid;
    const bool m = j < rows && min(max(tokens[j], 0), vocab - 1) == tok;
    const unsigned bal = __ballot_sync(0xffffffffu, m);
    if (lane == 0) wcnt[warp] = __popc(bal);
    __syncthreads();
    int off = 0, n = 0;
    for (int w = 0; w < EMB_WARPS; ++w) {
      off += w < warp ? wcnt[w] : 0;
      n += wcnt[w];
    }
    if (m) list[off + __popc(bal & ((1u << lane) - 1u))] = j;
    __syncthreads();
    for (int c = tid; c < d; c += blockDim.x) {
      float a = acc[c];
      for (int k = 0; k < n; ++k) a = __fadd_rn(a, __fmul_rn(__bfloat162float(dx[(size_t)list[k] * ld + c]), inv_sqrt_d));
      acc[c] = a;
    }
    __syncthreads();
  }
  for (int c = tid; c < d; c += blockDim.x) dembed[(size_t)tok * d + c] = acc[c];
}

// torch.optim.Adam (no weight decay, no amsgrad): one element per thread over the flat vectors
__global__ void adam_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v, size_t n,
                            float grad_scale, float lr, float b1, float b2, float eps, float bc1, float bc2_sqrt) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float gi = g[i] * grad_scale;
  const float mi = b1 * m[i] + (1.f - b1) * gi;
  const float vi = b2 * v[i] + (1.f - b2) * gi * gi;
  m[i] = mi;
  v[i] = vi;
  p[i] -= (lr / bc1) * mi / (sqrtf(vi) / bc2_sqrt + eps);
}

// fp32 master block [rows_pad, cols_pad] -> bf16 operand w [rows_pad, w_ld] (first w_cols columns) and its transpose
__global__ void repack_kernel(const float* __restrict__ p, int rows_pad, int cols_pad, bf16* __restrict__ w, int w_ld, int w_cols,
                              bf16* __restrict__ wt, int wt_ld) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (size_t)rows_pad * cols_pad) return;
  const int r = (int)(i / cols_pad), c = (int)(i % cols_pad);
  const bf16 v = __float2bfloat16(p[i]);
  if (c < w_cols) w[(size_t)r * w_ld + c] = v;
  if (wt) wt[(size_t)c * wt_ld + r] = v;
}

// out = (KL + CE, KL, CE) from the per-row parts [2][R], summed by one warp in a fixed order (run-to-run identical)
__global__ void loss_total_kernel(const float* __restrict__ parts, int R, float* __restrict__ out) {
  float kl = 0.f, ce = 0.f;
  for (int r = threadIdx.x; r < R; r += 32) {
    kl += parts[r];
    ce += parts[R + r];
  }
  kl = warp_sum(kl);
  ce = warp_sum(ce);
  if (threadIdx.x == 0) {
    out[0] = kl + ce;
    out[1] = kl;
    out[2] = ce;
  }
}

}  // namespace

// ------------------------------------------------------------------ launchers (student_ops.h)
namespace sdet {

int t_transpose(gitb200_student* c, const bf16* src, int ld_src, int R, int C, bf16* dst, int R_pad, int C_pad, cudaStream_t s) {
  dim3 grid((C_pad + 31) / 32, (R_pad + 31) / 32), block(32, 8);
  transpose_pad_kernel<<<grid, block, 0, s>>>(src, ld_src, R, C, dst, R_pad, R_pad, C_pad);
  note_launch();
  S_CUDA_OK(c, cudaGetLastError());
  return 0;
}
int t_colsum(gitb200_student* c, const bf16* x, int ld, int R, int C, float* out, cudaStream_t s) {
  colsum_kernel<<<(C + 127) / 128, 128, 0, s>>>(x, ld, R, C, out);
  note_launch();
  S_CUDA_OK(c, cudaGetLastError());
  return 0;
}

int t_weight_grad(gitb200_student* c, const bf16* dY, int ldy, int n_pad, const bf16* X, int ldx, int x_cols, int k_pad, int R, float* dW,
                  bf16* tA, bf16* tB, cudaStream_t s) {
  const int Rp = round_up(R, 64);
  S_TRY(t_transpose(c, dY, ldy, R, n_pad, tA, Rp, n_pad, s));
  S_TRY(t_transpose(c, X, ldx, R, x_cols, tB, Rp, k_pad, s));
  return s_gemm(c, tA, Rp, tB, Rp, n_pad, k_pad, nullptr, nullptr, 0, ACT_NONE, nullptr, 0, dW, k_pad, s);
}

template <bool DROP>
static int ln_bwd_launch(gitb200_student* c, const bf16* y, const bf16* dx, int rows, const float* gamma, bf16* dy, bf16* dz, float* dgamma,
                         float* dbeta, float* stats, const SDrop& dr, cudaStream_t s) {
  const int d = c->cfg.d_model, dp = c->dp;
  ln_bwd_kernel<DROP><<<(rows * 32 + 255) / 256, 256, 0, s>>>(y, dx, dp, rows, d, gamma, c->cfg.ln_eps, dy, stats, dz, dr);
  ln_param_grad_kernel<<<(d + 127) / 128, 128, 0, s>>>(y, dx, dp, rows, d, stats, dgamma, dbeta);
  note_launch(2);
  S_CUDA_OK(c, cudaGetLastError());
  return 0;
}
int t_ln_bwd(gitb200_student* c, const bf16* y, const bf16* dx, int rows, const float* gamma, bf16* dy, float* dgamma, float* dbeta,
             float* stats, cudaStream_t s) {
  return ln_bwd_launch<false>(c, y, dx, rows, gamma, dy, nullptr, dgamma, dbeta, stats, SDrop{}, s);
}
int t_ln_bwd_dropout(gitb200_student* c, const bf16* y, const bf16* dx, int rows, const float* gamma, bf16* dy, bf16* dz, float* dgamma,
                     float* dbeta, float* stats, const SDrop& dr, cudaStream_t s) {
  return ln_bwd_launch<true>(c, y, dx, rows, gamma, dy, dz, dgamma, dbeta, stats, dr, s);
}

template <bool DROP>
static int attn_bwd_launch(gitb200_student* c, const bf16* q, int ldq, int Lq, const bf16* kv, int kv_rows, int ldkv, int k_off, int v_off,
                           int n_keys, int causal, const int* tokens, int tok_ld, int B, const bf16* dO, bf16* dq, int lddq, bf16* dkv,
                           int lddkv, int dk_off, int dv_off, const SDrop& dr, cudaStream_t s) {
  if (Lq < 1 || Lq > T_MAX_SEQ || n_keys < 1 || n_keys > T_MAX_SEQ)
    return sfail(c, GITB200_ERR_INVALID, "attention backward over %d queries x %d keys (1 .. %d each)", Lq, n_keys, T_MAX_SEQ);
  const int hd = c->hd;
  const size_t smem = ((size_t)(2 * Lq + 2 * n_keys) * (hd + 1) + (size_t)(DROP ? 3 : 2) * Lq * (n_keys + 1)) * sizeof(float);
  static size_t attr = 0;  // per instantiation, process-wide, not per device: one process trains on one GPU (dist.py)
  if (smem > 48 * 1024 && smem > attr) {
    S_CUDA_OK(c, cudaFuncSetAttribute(attn_bwd_kernel<DROP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attr = smem;
  }
  attn_bwd_kernel<DROP><<<dim3(B, c->cfg.n_head), 128, smem, s>>>(q, ldq, Lq, kv, kv_rows, ldkv, k_off, v_off, n_keys, causal, tokens,
                                                                  tok_ld, c->cfg.pad, hd, 1.0f / sqrtf((float)hd), dO, c->dp, dq, lddq, dkv,
                                                                  lddkv, dk_off, dv_off, dr);
  note_launch();
  S_CUDA_OK(c, cudaGetLastError());
  return 0;
}
int t_attn_bwd(gitb200_student* c, const bf16* q, int ldq, int Lq, const bf16* kv, int kv_rows, int ldkv, int k_off, int v_off, int n_keys,
               int causal, const int* tokens, int tok_ld, int B, const bf16* dO, bf16* dq, int lddq, bf16* dkv, int lddkv, int dk_off,
               int dv_off, cudaStream_t s) {
  return attn_bwd_launch<false>(c, q, ldq, Lq, kv, kv_rows, ldkv, k_off, v_off, n_keys, causal, tokens, tok_ld, B, dO, dq, lddq, dkv, lddkv,
                                dk_off, dv_off, SDrop{}, s);
}
int t_attn_bwd_dropout(gitb200_student* c, const bf16* q, int ldq, int Lq, const bf16* kv, int kv_rows, int ldkv, int k_off, int v_off,
                       int n_keys, int causal, const int* tokens, int tok_ld, int B, const bf16* dO, bf16* dq, int lddq, bf16* dkv, int lddkv,
                       int dk_off, int dv_off, const SDrop& dr, cudaStream_t s) {
  return attn_bwd_launch<true>(c, q, ldq, Lq, kv, kv_rows, ldkv, k_off, v_off, n_keys, causal, tokens, tok_ld, B, dO, dq, lddq, dkv, lddkv,
                               dk_off, dv_off, dr, s);
}

int t_dropout_add_ln(gitb200_student* c, const bf16* x, const bf16* z, int rows, const float* g, const float* b, bf16* y, bf16* out,
                     const SDrop& dr, cudaStream_t s) {
  const int d = c->cfg.d_model;
  if (d % 4 != 0) return sfail(c, GITB200_ERR_INVALID, "dropout-add-LayerNorm needs d_model %% 4 == 0, not %d", d);
  dropout_add_ln_kernel<<<(rows * 32 + 255) / 256, 256, 0, s>>>(x, z, c->dp, rows, d, g, b, c->cfg.ln_eps, y, out, dr);
  note_launch();
  S_CUDA_OK(c, cudaGetLastError());
  return 0;
}

int t_dropout_inplace(gitb200_student* c, bf16* h, int ld, int rows, int cols, const SDrop& dr, cudaStream_t s) {
  if (cols % 4 != 0) return sfail(c, GITB200_ERR_INVALID, "dropout over %d columns (a multiple of 4)", cols);
  const size_t quads = (size_t)rows * (cols / 4);
  dropout_inplace_kernel<<<(unsigned)((quads + 255) / 256), 256, 0, s>>>(h, ld, rows, cols, dr);
  note_launch();
  S_CUDA_OK(c, cudaGetLastError());
  return 0;
}

int t_distill_loss(gitb200_student* c, const float* s_logits, int ld_s, const float* t_logits, int ld_t, const int* tokens, int B, int L,
                   float temperature, int* n_valid, bf16* dlogits, float* loss, float* loss_out, cudaStream_t s) {
  count_valid_kernel<<<1, 256, 0, s>>>(tokens, B, L, 0, n_valid);
  distill_loss_kernel<<<B * L, 256, 0, s>>>(s_logits, ld_s, t_logits, ld_t, tokens, B, L, c->cfg.vocab, c->vp, 0, temperature, n_valid,
                                            dlogits, loss);
  note_launch(2);
  S_CUDA_OK(c, cudaGetLastError());
  loss_total_kernel<<<1, 32, 0, s>>>(loss, B * L, loss_out);  // (KL + CE, KL, CE)
  note_launch();
  S_CUDA_OK(c, cudaGetLastError());
  return 0;
}

int t_relu_bwd(gitb200_student* c, const bf16* h, bf16* dh, size_t n, cudaStream_t s) {
  relu_bwd_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(h, dh, n);
  note_launch();
  S_CUDA_OK(c, cudaGetLastError());
  return 0;
}

int t_relu_bwd_dropout(gitb200_student* c, const bf16* h, bf16* dh, size_t n, float inv_keep, cudaStream_t s) {
  relu_bwd_dropout_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(h, dh, n, inv_keep);
  note_launch();
  S_CUDA_OK(c, cudaGetLastError());
  return 0;
}

int t_embed_bwd(gitb200_student* c, const int* tokens, int rows, const bf16* dx, int ld, float* dembed, cudaStream_t s) {
  const int d = c->cfg.d_model;
  const size_t smem = (size_t)d * sizeof(float);  // the accumulators of one token's row of the table
  if (smem > 48 * 1024) return sfail(c, GITB200_ERR_INVALID, "embedding backward holds at most %d columns, not %d", 48 * 1024 / 4, d);
  embed_bwd_kernel<<<rows, 32 * EMB_WARPS, smem, s>>>(tokens, rows, dx, ld, d, c->cfg.vocab, 1.0f / sqrtf((float)d), dembed);
  note_launch();
  S_CUDA_OK(c, cudaGetLastError());
  return 0;
}

}  // namespace sdet

namespace {

PEntry* find_entry(STrain* t, const std::string& name, int src_row0 = 0) {
  for (auto& e : t->entries)
    if (e.name == name && e.src_row0 == src_row0) return &e;
  return nullptr;
}
float* G_of(STrain* t, float* G, const std::string& name, int src_row0 = 0) { return G + find_entry(t, name, src_row0)->off; }

int repack_all(gitb200_student* c, cudaStream_t s) {
  STrain* t = c->train;
  for (auto& e : t->entries) {
    if (!e.w) continue;
    const size_t n = (size_t)e.rows_pad * e.cols_pad;
    repack_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(t->P + e.off, e.rows_pad, e.cols_pad, e.w, e.w_ld, e.w_cols, e.wt, e.wt_ld);
    note_launch();
  }
  S_CUDA_OK(c, cudaGetLastError());
  return 0;
}

template <typename T>
int t_alloc(gitb200_student* c, T** p, size_t n) {
  S_CUDA_OK(c, cudaMalloc(p, n * sizeof(T)));
  S_CUDA_OK(c, cudaMemset(*p, 0, n * sizeof(T)));
  c->allocs.push_back(*p);
  return 0;
}

}  // namespace

namespace sdet {
void student_train_destroy(gitb200_student* c) {
  STrain* t = c->train;
  if (!t) return;
  cudaFree(t->P);
  cudaFree(t->M1);
  cudaFree(t->M2);
  for (auto& a : t->acts)
    for (auto* b : {&a.x0, &a.qkv, &a.a, &a.y1, &a.x1, &a.q2, &a.memkv, &a.a2, &a.y2, &a.x2, &a.h, &a.y3}) cudaFree(b->p);
  for (auto* b : {&t->xo, &t->mem, &t->dlogits, &t->tA, &t->tB, &t->dx, &t->dy, &t->da, &t->dqkv, &t->dh, &t->dmemkv, &t->dmem, &t->z, &t->dz})
    cudaFree(b->p);
  cudaFree(t->logits.p);
  cudaFree(t->stats.p);
  cudaFree(t->loss.p);
  cudaFree(t->nvalid.p);
  cudaFree(t->toks.p);
  delete t;
  c->train = nullptr;
}
}  // namespace sdet

extern "C" {

int gitb200_student_set_training(gitb200_student* c, int enable) {
  if (!c) return GITB200_ERR_INVALID;
  if (c->finalized && enable && !c->keep_raw)
    return sfail(c, GITB200_ERR_STATE, "gitb200_student_set_training must be called before gitb200_student_finalize (the fp32 weights are gone)");
  c->keep_raw = enable != 0;
  return GITB200_OK;
}

// Build the flat fp32 master vector from the staged fp32 weights, re-point the inference path's fp32 vectors (biases, LayerNorm
// affines, embedding table) into it and create the transposed bf16 operand copies.  Returns the length of the flat vectors.
long long gitb200_student_train_begin(gitb200_student* c, float lr, float beta1, float beta2, float eps) {
  if (!c) return -1;
  if (!c->finalized || !c->keep_raw || c->raw.empty()) {
    sfail(c, GITB200_ERR_STATE, "training needs gitb200_student_set_training(1) before the weights are loaded and finalised");
    return -1;
  }
  if (cudaSetDevice(c->device) != cudaSuccess) return -1;
  if (c->train) student_train_destroy(c);
  STrain* t = new STrain();
  c->train = t;
  t->lr = lr; t->beta1 = beta1; t->beta2 = beta2; t->eps = eps;
  const gitb200_student_config& k = c->cfg;
  const int d = k.d_model, dp = c->dp, f = k.d_ffn, fp = c->fp, vp = c->vp;
  size_t off = 0;
  auto add = [&](const std::string& name, int src_row0, int rows, int cols, int rows_pad, int cols_pad) -> PEntry& {
    PEntry e;
    e.name = name; e.src_row0 = src_row0; e.rows = rows; e.cols = cols; e.rows_pad = rows_pad; e.cols_pad = cols_pad; e.off = off;
    off += (size_t)rows_pad * cols_pad;
    off = (off + 63) / 64 * 64;  // 256-byte aligned blocks (GEMM fp32 outputs, vector loads)
    t->entries.push_back(e);
    return t->entries.back();
  };
  // ---- bucket 0: the vocabulary head (its gradients are complete after phase 0 of the backward pass)
  add("linear.weight", 0, k.vocab, d, vp, dp);
  add("linear.bias", 0, k.vocab, 1, vp, 1);
  t->head_floats = off;
  // ---- bucket 1: decoder layers, then the embedding table
  for (int l = 0; l < k.n_layers; ++l) {
    const std::string p = "decoder.layers." + std::to_string(l) + ".";
    for (int b = 0; b < 3; ++b) add(p + "self_attn.in_proj_weight", b * d, d, d, dp, dp);
    for (int b = 0; b < 3; ++b) add(p + "self_attn.in_proj_bias", b * d, d, 1, dp, 1);
    add(p + "self_attn.out_proj.weight", 0, d, d, dp, dp);
    add(p + "self_attn.out_proj.bias", 0, d, 1, dp, 1);
    for (int b = 0; b < 3; ++b) add(p + "multihead_attn.in_proj_weight", b * d, d, d, dp, dp);
    for (int b = 0; b < 3; ++b) add(p + "multihead_attn.in_proj_bias", b * d, d, 1, dp, 1);
    add(p + "multihead_attn.out_proj.weight", 0, d, d, dp, dp);
    add(p + "multihead_attn.out_proj.bias", 0, d, 1, dp, 1);
    add(p + "linear1.weight", 0, f, d, fp, dp);
    add(p + "linear1.bias", 0, f, 1, fp, 1);
    add(p + "linear2.weight", 0, d, f, dp, fp);
    add(p + "linear2.bias", 0, d, 1, dp, 1);
    for (const char* n : {"norm1.weight", "norm1.bias", "norm2.weight", "norm2.bias", "norm3.weight", "norm3.bias"}) add(p + n, 0, d, 1, d, 1);
  }
  add("embed.weight", 0, k.vocab, d, k.vocab, d);
  t->n_floats = off;
  if (cudaMalloc(&t->P, off * sizeof(float)) != cudaSuccess || cudaMalloc(&t->M1, off * sizeof(float)) != cudaSuccess ||
      cudaMalloc(&t->M2, off * sizeof(float)) != cudaSuccess) {
    sfail(c, GITB200_ERR_CUDA, "cudaMalloc of the optimizer state (%zu floats x 3) failed", off);
    return -1;
  }
  cudaMemset(t->P, 0, off * sizeof(float));
  cudaMemset(t->M1, 0, off * sizeof(float));
  cudaMemset(t->M2, 0, off * sizeof(float));
  for (auto& e : t->entries) {
    auto it = c->raw.find(e.name);
    if (it == c->raw.end() || (int64_t)it->second.numel() < (int64_t)(e.src_row0 + e.rows) * e.cols) {
      sfail(c, GITB200_ERR_MISSING, "missing or short weight %s", e.name.c_str());
      return -1;
    }
    if (cudaMemcpy2D(t->P + e.off, (size_t)e.cols_pad * sizeof(float), it->second.p + (size_t)e.src_row0 * e.cols, (size_t)e.cols * sizeof(float),
                     (size_t)e.cols * sizeof(float), e.rows, cudaMemcpyDeviceToDevice) != cudaSuccess) {
      sfail(c, GITB200_ERR_CUDA, "copy of %s into the master vector failed", e.name.c_str());
      return -1;
    }
  }
  // ---- operand copies: existing bf16 weights stay where the inference path expects them; transposed twins are new
  t->lt.assign(k.n_layers, LayerT{});
  auto tr = [&](bf16** p, size_t n) { return t_alloc(c, p, n); };
  if (tr(&t->wt_vocab, (size_t)dp * vp)) return -1;
  {
    PEntry* e = find_entry(t, "linear.weight");
    e->w = c->w_vocab; e->w_ld = d; e->w_cols = d; e->wt = t->wt_vocab; e->wt_ld = vp;
  }
  c->b_vocab = t->P + find_entry(t, "linear.bias")->off;
  for (int l = 0; l < k.n_layers; ++l) {
    const std::string p = "decoder.layers." + std::to_string(l) + ".";
    SLayer& W = c->layers[l];
    LayerT& T = t->lt[l];
    if (tr(&T.sa_in, (size_t)dp * 3 * dp) || tr(&T.sa_out, (size_t)dp * dp) || tr(&T.ca_q, (size_t)dp * dp) || tr(&T.ca_kv, (size_t)dp * 2 * dp) ||
        tr(&T.ca_out, (size_t)dp * dp) || tr(&T.ff1, (size_t)dp * fp) || tr(&T.ff2, (size_t)fp * dp))
      return -1;
    for (int b = 0; b < 3; ++b) {
      PEntry* e = find_entry(t, p + "self_attn.in_proj_weight", b * d);
      e->w = W.w_sa_in + (size_t)b * dp * d; e->w_ld = d; e->w_cols = d; e->wt = T.sa_in + (size_t)b * dp; e->wt_ld = 3 * dp;
    }
    {
      PEntry* e = find_entry(t, p + "self_attn.out_proj.weight");
      e->w = W.w_sa_out; e->w_ld = d; e->w_cols = d; e->wt = T.sa_out; e->wt_ld = dp;
      e = find_entry(t, p + "multihead_attn.in_proj_weight", 0);
      e->w = W.w_ca_q; e->w_ld = d; e->w_cols = d; e->wt = T.ca_q; e->wt_ld = dp;
      for (int b = 0; b < 2; ++b) {
        e = find_entry(t, p + "multihead_attn.in_proj_weight", (b + 1) * d);
        e->w = W.w_ca_kv + (size_t)b * dp * d; e->w_ld = d; e->w_cols = d; e->wt = T.ca_kv + (size_t)b * dp; e->wt_ld = 2 * dp;
      }
      e = find_entry(t, p + "multihead_attn.out_proj.weight");
      e->w = W.w_ca_out; e->w_ld = d; e->w_cols = d; e->wt = T.ca_out; e->wt_ld = dp;
      e = find_entry(t, p + "linear1.weight");
      e->w = W.w_ff1; e->w_ld = d; e->w_cols = d; e->wt = T.ff1; e->wt_ld = fp;
      e = find_entry(t, p + "linear2.weight");
      e->w = W.w_ff2; e->w_ld = fp; e->w_cols = fp; e->wt = T.ff2; e->wt_ld = dp;
    }
    // fp32 vectors: the inference kernels now read the live master copies.  The fused q|k|v bias blocks are contiguous in the
    // layout (3 blocks of dp floats, each a multiple of 64), like the [3*dp] vector the forward expects.
    W.b_sa_in = t->P + find_entry(t, p + "self_attn.in_proj_bias", 0)->off;
    W.b_sa_out = t->P + find_entry(t, p + "self_attn.out_proj.bias")->off;
    W.b_ca_q = t->P + find_entry(t, p + "multihead_attn.in_proj_bias", 0)->off;
    W.b_ca_kv = t->P + find_entry(t, p + "multihead_attn.in_proj_bias", d)->off;
    W.b_ca_out = t->P + find_entry(t, p + "multihead_attn.out_proj.bias")->off;
    W.b_ff1 = t->P + find_entry(t, p + "linear1.bias")->off;
    W.b_ff2 = t->P + find_entry(t, p + "linear2.bias")->off;
    W.n1_g = t->P + find_entry(t, p + "norm1.weight")->off;
    W.n1_b = t->P + find_entry(t, p + "norm1.bias")->off;
    W.n2_g = t->P + find_entry(t, p + "norm2.weight")->off;
    W.n2_b = t->P + find_entry(t, p + "norm2.bias")->off;
    W.n3_g = t->P + find_entry(t, p + "norm3.weight")->off;
    W.n3_b = t->P + find_entry(t, p + "norm3.bias")->off;
  }
  c->embed = t->P + find_entry(t, "embed.weight")->off;
  if (repack_all(c, 0)) return -1;
  if (cudaDeviceSynchronize() != cudaSuccess) {
    sfail(c, GITB200_ERR_CUDA, "train_begin: %s", cudaGetErrorString(cudaGetLastError()));
    return -1;
  }
  t->acts.resize(k.n_layers);
  return (long long)t->n_floats;
}

int gitb200_student_train_set_dropout(gitb200_student* c, float p, uint64_t seed, long long step) {
  if (!c) return GITB200_ERR_INVALID;
  if (!(p >= 0.f && p < 1.f) || step < 0)
    return sfail(c, GITB200_ERR_INVALID, "dropout p must lie in [0, 1) and the step be >= 0 (got p = %g, step = %lld)", (double)p, step);
  STrain* t = c->train;
  if (!t) return sfail(c, GITB200_ERR_STATE, "call gitb200_student_train_begin first");
  t->drop_p = p;
  t->drop_seed = seed;
  t->drop_step = step;
  return GITB200_OK;
}

int gitb200_student_train_get_dropout(const gitb200_student* c, float* p, uint64_t* seed, long long* step) {
  if (!c || !c->train) return GITB200_ERR_STATE;
  if (p) *p = c->train->drop_p;
  if (seed) *seed = c->train->drop_seed;
  if (step) *step = c->train->drop_step;
  return GITB200_OK;
}

long long gitb200_student_train_head_floats(const gitb200_student* c) { return (c && c->train) ? (long long)c->train->head_floats : -1; }

// Forward with stored activations + loss + d loss / d logits.  tokens int32 [B, L]; memory fp32 [B, M, d_model]; teacher_logits fp32
// [B*L, ld_teacher] (first `vocab` columns).  loss_out (device, 3 floats): total, KL term, CE term.
int gitb200_student_train_forward(gitb200_student* c, const int32_t* tokens, const float* memory, const float* teacher_logits, int ld_teacher,
                                  int B, int L, int M, float temperature, float* loss_out, void* stream) {
  if (!c || !tokens || !memory || !teacher_logits || !loss_out) return sfail(c, GITB200_ERR_INVALID, "bad train_forward argument");
  STrain* t = c->train;
  if (!t) return sfail(c, GITB200_ERR_STATE, "call gitb200_student_train_begin first");
  const gitb200_student_config& k = c->cfg;
  if (B < 1 || L < 2 || M < 1 || L > T_MAX_SEQ || M > T_MAX_SEQ || L > k.max_len || ld_teacher < k.vocab || temperature <= 0.f)
    return sfail(c, GITB200_ERR_INVALID, "train_forward: need 2 <= L <= %d, 1 <= M <= %d, teacher rows of >= %d logits", T_MAX_SEQ, T_MAX_SEQ, k.vocab);
  S_CUDA_OK(c, cudaSetDevice(c->device));
  cudaStream_t s = (cudaStream_t)stream;
  const int d = k.d_model, dp = c->dp, fp = c->fp, vp = c->vp, R = B * L, Rm = B * M;
  const int Rp = round_up(R, 64), Rmp = round_up(Rm, 64), Rmax = Rp > Rmp ? Rp : Rmp;
  for (auto& a : t->acts) {
    S_TRY(sensure(c, a.x0, (size_t)R * dp));
    S_TRY(sensure(c, a.qkv, (size_t)R * 3 * dp));
    S_TRY(sensure(c, a.a, (size_t)R * dp));
    S_TRY(sensure(c, a.y1, (size_t)R * dp));
    S_TRY(sensure(c, a.x1, (size_t)R * dp));
    S_TRY(sensure(c, a.q2, (size_t)R * dp));
    S_TRY(sensure(c, a.memkv, (size_t)Rm * 2 * dp));
    S_TRY(sensure(c, a.a2, (size_t)R * dp));
    S_TRY(sensure(c, a.y2, (size_t)R * dp));
    S_TRY(sensure(c, a.x2, (size_t)R * dp));
    S_TRY(sensure(c, a.h, (size_t)R * fp));
    S_TRY(sensure(c, a.y3, (size_t)R * dp));
  }
  S_TRY(sensure(c, t->xo, (size_t)R * dp));
  S_TRY(sensure(c, t->mem, (size_t)Rm * d));
  S_TRY(sensure(c, t->logits, (size_t)R * vp));
  S_TRY(sensure(c, t->dlogits, (size_t)R * vp));
  const int widest = vp > 3 * dp ? vp : 3 * dp;
  S_TRY(sensure(c, t->tA, (size_t)(widest > fp ? widest : fp) * Rmax));
  S_TRY(sensure(c, t->tB, (size_t)(dp > fp ? dp : fp) * Rmax));
  S_TRY(sensure(c, t->dx, (size_t)R * dp));
  S_TRY(sensure(c, t->dy, (size_t)R * dp));
  S_TRY(sensure(c, t->da, (size_t)R * dp));
  S_TRY(sensure(c, t->dqkv, (size_t)R * 3 * dp));
  S_TRY(sensure(c, t->dh, (size_t)R * fp));
  S_TRY(sensure(c, t->dmemkv, (size_t)Rm * 2 * dp));
  S_TRY(sensure(c, t->dmem, (size_t)Rm * dp));
  S_TRY(sensure(c, t->stats, (size_t)2 * R));
  S_TRY(sensure(c, t->loss, (size_t)2 * R));
  S_TRY(sensure(c, t->nvalid, 1));
  S_TRY(sensure(c, t->toks, (size_t)R));
  const bool drop = t->drop_p > 0.f;
  if (drop) {
    S_TRY(sensure(c, t->z, (size_t)R * dp));
    S_TRY(sensure(c, t->dz, (size_t)R * dp));
  }
  auto site = [&](int l, int k) { return SDrop{t->drop_seed, (unsigned)t->drop_step, (unsigned)(6 * l + k), t->drop_p, 1.f / (1.f - t->drop_p)}; };
  S_CUDA_OK(c, cudaMemcpyAsync(t->toks.p, tokens, (size_t)R * sizeof(int), cudaMemcpyDeviceToDevice, s));  // the backward pass reads them again
  S_CUDA_OK(c, cast_f32_to_bf16(memory, Rm, d, d, t->mem.p, d, Rm, d, s));
  S_TRY(s_embed(c, t->toks.p, L, L, 0, R, t->acts[0].x0.p, s));
  for (int l = 0; l < k.n_layers; ++l) {
    const SLayer& W = c->layers[l];
    LayerAct& A = t->acts[l];
    bf16* x3 = (l + 1 < k.n_layers) ? t->acts[l + 1].x0.p : t->xo.p;
    S_TRY(s_gemm(c, A.x0.p, dp, W.w_sa_in, d, R, 3 * dp, W.b_sa_in, nullptr, 0, ACT_NONE, A.qkv.p, 3 * dp, nullptr, 0, s));
    if (drop) {  // the six sites of nn.TransformerDecoderLayer, in its call order: site 6 l + k
      S_TRY(s_attn_dropout(c, A.qkv.p, 3 * dp, L, A.qkv.p, L, 3 * dp, dp, 2 * dp, L, 1, t->toks.p, L, R, A.a.p, dp, site(l, 0), s));
      S_TRY(s_gemm(c, A.a.p, dp, W.w_sa_out, d, R, dp, W.b_sa_out, nullptr, 0, ACT_NONE, t->z.p, dp, nullptr, 0, s));
      S_TRY(t_dropout_add_ln(c, A.x0.p, t->z.p, R, W.n1_g, W.n1_b, A.y1.p, A.x1.p, site(l, 1), s));
      S_TRY(s_gemm(c, A.x1.p, dp, W.w_ca_q, d, R, dp, W.b_ca_q, nullptr, 0, ACT_NONE, A.q2.p, dp, nullptr, 0, s));
      S_TRY(s_gemm(c, t->mem.p, d, W.w_ca_kv, d, Rm, 2 * dp, W.b_ca_kv, nullptr, 0, ACT_NONE, A.memkv.p, 2 * dp, nullptr, 0, s));
      S_TRY(s_attn_dropout(c, A.q2.p, dp, L, A.memkv.p, M, 2 * dp, 0, dp, M, 0, nullptr, 0, R, A.a2.p, dp, site(l, 2), s));
      S_TRY(s_gemm(c, A.a2.p, dp, W.w_ca_out, d, R, dp, W.b_ca_out, nullptr, 0, ACT_NONE, t->z.p, dp, nullptr, 0, s));
      S_TRY(t_dropout_add_ln(c, A.x1.p, t->z.p, R, W.n2_g, W.n2_b, A.y2.p, A.x2.p, site(l, 3), s));
      S_TRY(s_gemm(c, A.x2.p, dp, W.w_ff1, d, R, fp, W.b_ff1, nullptr, 0, ACT_RELU, A.h.p, fp, nullptr, 0, s));
      S_TRY(t_dropout_inplace(c, A.h.p, fp, R, k.d_ffn, site(l, 4), s));
      S_TRY(s_gemm(c, A.h.p, fp, W.w_ff2, fp, R, dp, W.b_ff2, nullptr, 0, ACT_NONE, t->z.p, dp, nullptr, 0, s));
      S_TRY(t_dropout_add_ln(c, A.x2.p, t->z.p, R, W.n3_g, W.n3_b, A.y3.p, x3, site(l, 5), s));
      continue;
    }
    S_TRY(s_attn(c, A.qkv.p, 3 * dp, L, 0, A.qkv.p, L, 3 * dp, dp, 2 * dp, L, 1, t->toks.p, L, R, A.a.p, dp, s));
    S_TRY(s_gemm(c, A.a.p, dp, W.w_sa_out, d, R, dp, W.b_sa_out, A.x0.p, dp, ACT_NONE, A.y1.p, dp, nullptr, 0, s));
    S_TRY(s_ln(c, A.y1.p, dp, R, W.n1_g, W.n1_b, A.x1.p, dp, s));
    S_TRY(s_gemm(c, A.x1.p, dp, W.w_ca_q, d, R, dp, W.b_ca_q, nullptr, 0, ACT_NONE, A.q2.p, dp, nullptr, 0, s));
    S_TRY(s_gemm(c, t->mem.p, d, W.w_ca_kv, d, Rm, 2 * dp, W.b_ca_kv, nullptr, 0, ACT_NONE, A.memkv.p, 2 * dp, nullptr, 0, s));
    S_TRY(s_attn(c, A.q2.p, dp, L, 0, A.memkv.p, M, 2 * dp, 0, dp, M, 0, nullptr, 0, R, A.a2.p, dp, s));
    S_TRY(s_gemm(c, A.a2.p, dp, W.w_ca_out, d, R, dp, W.b_ca_out, A.x1.p, dp, ACT_NONE, A.y2.p, dp, nullptr, 0, s));
    S_TRY(s_ln(c, A.y2.p, dp, R, W.n2_g, W.n2_b, A.x2.p, dp, s));
    S_TRY(s_gemm(c, A.x2.p, dp, W.w_ff1, d, R, fp, W.b_ff1, nullptr, 0, ACT_RELU, A.h.p, fp, nullptr, 0, s));
    S_TRY(s_gemm(c, A.h.p, fp, W.w_ff2, fp, R, dp, W.b_ff2, A.x2.p, dp, ACT_NONE, A.y3.p, dp, nullptr, 0, s));
    S_TRY(s_ln(c, A.y3.p, dp, R, W.n3_g, W.n3_b, x3, dp, s));
  }
  S_TRY(s_gemm(c, t->xo.p, dp, c->w_vocab, d, R, vp, c->b_vocab, nullptr, 0, ACT_NONE, nullptr, 0, t->logits.p, vp, s));
  S_TRY(t_distill_loss(c, t->logits.p, vp, teacher_logits, ld_teacher, t->toks.p, B, L, temperature, t->nvalid.p, t->dlogits.p, t->loss.p,
                       loss_out, s));
  t->B = B; t->L = L; t->M = M;
  t->fwd_drop = drop;
  t->fwd_step = t->drop_step;
  if (drop) t->drop_step += 1;
  t->have_forward = true;
  t->have_head = false;
  return GITB200_OK;
}

// Backward pass.  phase 0: vocabulary head (dW, db into grads[0, head_floats), d loss / d decoder output kept internally);
// phase 1: decoder layers + embedding (grads[head_floats, n_floats)) and, optionally, d loss / d memory fp32 [B, M, d_model].
int gitb200_student_train_backward(gitb200_student* c, int phase, float* grads, float* d_memory, void* stream) {
  if (!c || !grads || (phase != 0 && phase != 1)) return sfail(c, GITB200_ERR_INVALID, "bad train_backward argument");
  STrain* t = c->train;
  if (!t || !t->have_forward) return sfail(c, GITB200_ERR_STATE, "call gitb200_student_train_forward first");
  if (phase == 1 && !t->have_head) return sfail(c, GITB200_ERR_STATE, "backward phase 0 (vocabulary head) must run before phase 1");
  S_CUDA_OK(c, cudaSetDevice(c->device));
  cudaStream_t s = (cudaStream_t)stream;
  const gitb200_student_config& k = c->cfg;
  const int d = k.d_model, dp = c->dp, fp = c->fp, vp = c->vp, B = t->B, L = t->L, M = t->M, R = B * L, Rm = B * M;
  if (phase == 0) {
    // logits = xo W_v^T + b_v
    S_TRY(t_weight_grad(c, t->dlogits.p, vp, vp, t->xo.p, dp, dp, dp, R, G_of(t, grads, "linear.weight"), t->tA.p, t->tB.p, s));
    S_TRY(t_colsum(c, t->dlogits.p, vp, R, vp, G_of(t, grads, "linear.bias"), s));
    S_TRY(s_gemm(c, t->dlogits.p, vp, t->wt_vocab, vp, R, dp, nullptr, nullptr, 0, ACT_NONE, t->dx.p, dp, nullptr, 0, s));
    t->have_head = true;
    return GITB200_OK;
  }
  // embed_bwd_kernel stores the rows of the tokens that occur; the rows of the others must read as zero
  {
    PEntry* e = find_entry(t, "embed.weight");
    S_CUDA_OK(c, cudaMemsetAsync(grads + e->off, 0, (size_t)e->rows_pad * e->cols_pad * sizeof(float), s));
  }
  // dropout: the residual sites' LayerNorm backward also gives dz = D o dy, the gradient of the dropped addend, which feeds the
  // out-projection's gradients; dy itself still goes to the residual addend.  Without dropout dz is dy.
  const bool drop = t->fwd_drop;
  const float inv_keep = drop ? 1.f / (1.f - t->drop_p) : 1.f;
  auto site = [&](int l, int kk) { return SDrop{t->drop_seed, (unsigned)t->fwd_step, (unsigned)(6 * l + kk), t->drop_p, inv_keep}; };
  bf16* dz = drop ? t->dz.p : t->dy.p;
  auto ln_bwd = [&](const bf16* y, int l, int kk, const float* gamma, const std::string& name) {
    float *dg = G_of(t, grads, name + ".weight"), *db = G_of(t, grads, name + ".bias");
    return drop ? t_ln_bwd_dropout(c, y, t->dx.p, R, gamma, t->dy.p, dz, dg, db, t->stats.p, site(l, kk), s)
                : t_ln_bwd(c, y, t->dx.p, R, gamma, t->dy.p, dg, db, t->stats.p, s);
  };
  for (int l = k.n_layers - 1; l >= 0; --l) {
    const std::string p = "decoder.layers." + std::to_string(l) + ".";
    const SLayer& W = c->layers[l];
    const LayerT& T = t->lt[l];
    LayerAct& A = t->acts[l];
    // ---- x3 = norm3(y3), y3 = h W2^T + b2 + x2, h = relu(x2 W1^T + b1)              (dx holds d loss / d x3)
    S_TRY(ln_bwd(A.y3.p, l, 5, W.n3_g, p + "norm3"));
    S_TRY(t_weight_grad(c, dz, dp, dp, A.h.p, fp, fp, fp, R, G_of(t, grads, p + "linear2.weight"), t->tA.p, t->tB.p, s));
    S_TRY(t_colsum(c, dz, dp, R, dp, G_of(t, grads, p + "linear2.bias"), s));
    S_TRY(s_gemm(c, dz, dp, T.ff2, dp, R, fp, nullptr, nullptr, 0, ACT_NONE, t->dh.p, fp, nullptr, 0, s));
    if (drop)
      S_TRY(t_relu_bwd_dropout(c, A.h.p, t->dh.p, (size_t)R * fp, inv_keep, s));
    else
      S_TRY(t_relu_bwd(c, A.h.p, t->dh.p, (size_t)R * fp, s));
    S_TRY(t_weight_grad(c, t->dh.p, fp, fp, A.x2.p, dp, dp, dp, R, G_of(t, grads, p + "linear1.weight"), t->tA.p, t->tB.p, s));
    S_TRY(t_colsum(c, t->dh.p, fp, R, fp, G_of(t, grads, p + "linear1.bias"), s));
    S_TRY(s_gemm(c, t->dh.p, fp, T.ff1, fp, R, dp, nullptr, t->dy.p, dp, ACT_NONE, t->dx.p, dp, nullptr, 0, s));  // d x2 = dh W1 + d y3
    // ---- x2 = norm2(y2), y2 = a2 Wo^T + bo + x1, a2 = attn(q2, memkv), q2 = x1 Wq^T + bq, memkv = mem Wkv^T + bkv
    S_TRY(ln_bwd(A.y2.p, l, 3, W.n2_g, p + "norm2"));
    S_TRY(t_weight_grad(c, dz, dp, dp, A.a2.p, dp, dp, dp, R, G_of(t, grads, p + "multihead_attn.out_proj.weight"), t->tA.p, t->tB.p, s));
    S_TRY(t_colsum(c, dz, dp, R, dp, G_of(t, grads, p + "multihead_attn.out_proj.bias"), s));
    S_TRY(s_gemm(c, dz, dp, T.ca_out, dp, R, dp, nullptr, nullptr, 0, ACT_NONE, t->da.p, dp, nullptr, 0, s));
    if (drop)
      S_TRY(t_attn_bwd_dropout(c, A.q2.p, dp, L, A.memkv.p, M, 2 * dp, 0, dp, M, 0, nullptr, 0, B, t->da.p, t->dqkv.p, dp, t->dmemkv.p, 2 * dp, 0,
                               dp, site(l, 2), s));
    else
      S_TRY(t_attn_bwd(c, A.q2.p, dp, L, A.memkv.p, M, 2 * dp, 0, dp, M, 0, nullptr, 0, B, t->da.p, t->dqkv.p, dp, t->dmemkv.p, 2 * dp, 0, dp, s));
    S_TRY(t_weight_grad(c, t->dqkv.p, dp, dp, A.x1.p, dp, dp, dp, R, G_of(t, grads, p + "multihead_attn.in_proj_weight", 0), t->tA.p, t->tB.p, s));
    S_TRY(t_colsum(c, t->dqkv.p, dp, R, dp, G_of(t, grads, p + "multihead_attn.in_proj_bias", 0), s));
    S_TRY(s_gemm(c, t->dqkv.p, dp, T.ca_q, dp, R, dp, nullptr, t->dy.p, dp, ACT_NONE, t->dx.p, dp, nullptr, 0, s));  // d x1 = dq2 Wq + d y2
    // the k | v blocks of in_proj are adjacent in the layout ([2*dp, dp] fp32): one GEMM fills both
    S_TRY(t_weight_grad(c, t->dmemkv.p, 2 * dp, 2 * dp, t->mem.p, d, d, dp, Rm, G_of(t, grads, p + "multihead_attn.in_proj_weight", d), t->tA.p,
                        t->tB.p, s));
    S_TRY(t_colsum(c, t->dmemkv.p, 2 * dp, Rm, 2 * dp, G_of(t, grads, p + "multihead_attn.in_proj_bias", d), s));
    S_TRY(s_gemm(c, t->dmemkv.p, 2 * dp, T.ca_kv, 2 * dp, Rm, dp, nullptr, l + 1 < k.n_layers ? t->dmem.p : nullptr, dp, ACT_NONE, t->dmem.p, dp,
                 nullptr, 0, s));  // d memory accumulates over the layers
    // ---- x1 = norm1(y1), y1 = a Wo^T + bo + x0, a = self-attn(qkv), qkv = x0 Win^T + bin
    S_TRY(ln_bwd(A.y1.p, l, 1, W.n1_g, p + "norm1"));
    S_TRY(t_weight_grad(c, dz, dp, dp, A.a.p, dp, dp, dp, R, G_of(t, grads, p + "self_attn.out_proj.weight"), t->tA.p, t->tB.p, s));
    S_TRY(t_colsum(c, dz, dp, R, dp, G_of(t, grads, p + "self_attn.out_proj.bias"), s));
    S_TRY(s_gemm(c, dz, dp, T.sa_out, dp, R, dp, nullptr, nullptr, 0, ACT_NONE, t->da.p, dp, nullptr, 0, s));
    if (drop)
      S_TRY(t_attn_bwd_dropout(c, A.qkv.p, 3 * dp, L, A.qkv.p, L, 3 * dp, dp, 2 * dp, L, 1, t->toks.p, L, B, t->da.p, t->dqkv.p, 3 * dp, t->dqkv.p,
                               3 * dp, dp, 2 * dp, site(l, 0), s));
    else
      S_TRY(t_attn_bwd(c, A.qkv.p, 3 * dp, L, A.qkv.p, L, 3 * dp, dp, 2 * dp, L, 1, t->toks.p, L, B, t->da.p, t->dqkv.p, 3 * dp, t->dqkv.p, 3 * dp,
                       dp, 2 * dp, s));
    // q | k | v blocks are adjacent in the layout ([3*dp, dp] fp32): one GEMM fills all three
    S_TRY(t_weight_grad(c, t->dqkv.p, 3 * dp, 3 * dp, A.x0.p, dp, dp, dp, R, G_of(t, grads, p + "self_attn.in_proj_weight", 0), t->tA.p, t->tB.p, s));
    S_TRY(t_colsum(c, t->dqkv.p, 3 * dp, R, 3 * dp, G_of(t, grads, p + "self_attn.in_proj_bias", 0), s));
    S_TRY(s_gemm(c, t->dqkv.p, 3 * dp, T.sa_in, 3 * dp, R, dp, nullptr, t->dy.p, dp, ACT_NONE, t->dx.p, dp, nullptr, 0, s));  // d x0 = dqkv Win + d y1
  }
  S_TRY(t_embed_bwd(c, t->toks.p, R, t->dx.p, dp, G_of(t, grads, "embed.weight"), s));
  if (d_memory) S_CUDA_OK(c, cast_bf16_to_f32(t->dmem.p, Rm, d, dp, d_memory, d, s));
  t->have_forward = false;
  return GITB200_OK;
}

// torch.optim.Adam step on the flat master vector with grads * grad_scale (1 / world size after a SUM all-reduce), then the
// bf16 operand copies (and their transposes) are refreshed from the master.
int gitb200_student_train_apply(gitb200_student* c, const float* grads, float grad_scale, void* stream) {
  if (!c || !grads) return sfail(c, GITB200_ERR_INVALID, "bad train_apply argument");
  STrain* t = c->train;
  if (!t) return sfail(c, GITB200_ERR_STATE, "call gitb200_student_train_begin first");
  S_CUDA_OK(c, cudaSetDevice(c->device));
  cudaStream_t s = (cudaStream_t)stream;
  t->step += 1;
  const float bc1 = 1.f - powf(t->beta1, (float)t->step), bc2 = 1.f - powf(t->beta2, (float)t->step);
  adam_kernel<<<(unsigned)((t->n_floats + 255) / 256), 256, 0, s>>>(t->P, grads, t->M1, t->M2, t->n_floats, grad_scale, t->lr, t->beta1, t->beta2,
                                                                     t->eps, bc1, sqrtf(bc2));
  note_launch();
  S_CUDA_OK(c, cudaGetLastError());
  return repack_all(c, s);
}

// which = 0: parameter (master copy), 1: gradient (from the flat vector `grads`).  out: fp32 tensor of the reference's shape for `name`.
int gitb200_student_train_export(gitb200_student* c, const char* name, int which, const float* grads, float* out, void* stream) {
  if (!c || !name || !out || (which == 1 && !grads)) return sfail(c, GITB200_ERR_INVALID, "bad train_export argument");
  STrain* t = c->train;
  if (!t) return sfail(c, GITB200_ERR_STATE, "call gitb200_student_train_begin first");
  S_CUDA_OK(c, cudaSetDevice(c->device));
  bool any = false;
  for (auto& e : t->entries) {
    if (e.name != name) continue;
    any = true;
    const float* src = (which == 0 ? t->P : grads) + e.off;
    S_CUDA_OK(c, cudaMemcpy2DAsync(out + (size_t)e.src_row0 * e.cols, (size_t)e.cols * sizeof(float), src, (size_t)e.cols_pad * sizeof(float),
                                   (size_t)e.cols * sizeof(float), e.rows, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  }
  if (!any) return sfail(c, GITB200_ERR_MISSING, "no trainable parameter named %s", name);
  return GITB200_OK;
}

}  // extern "C"

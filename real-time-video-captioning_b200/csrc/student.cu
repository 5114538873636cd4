// Student decoder on the GPU (SURVEY 8f rank 3): the decoder half of StudentCandidateV1
// (/root/reference/src/models/model.py:50-187) -- nn.Embedding + sinusoidal PositionalEncoding, a post-LN
// nn.TransformerDecoder (self-attention under the causal + padding mask, cross-attention to the F frame tokens of
// `memory`, ReLU feed-forward) and the vocabulary nn.Linear -- as
//   * forward_decoder(y, memory)            (model.py:135-154, teacher-forced, all positions)
//   * greedy_decode on a given memory       (model.py:156-187) with a K/V cache: the reference re-decodes the whole
//     growing sequence every step (O(n^2) decoder passes); causal masking makes the cached form identical.
// All contractions go through the tcgen05 / weight-streaming GEMMs of the teacher path (weights zero-padded to tile
// multiples: d_model 576 -> 640); the small glue kernels below are plain CUDA-core kernels (a few KB per row).
// The QKV projection writes straight into the per-layer cache [B][Lmax][3*dp] (GEMM output leading dimension =
// Lmax*3*dp, base offset pos*3*dp), so no K/V scatter kernel exists.
#include "student_internal.cuh"

using namespace sdet;

namespace sdet {

std::string g_student_err;

int sfail(gitb200_student* c, int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  if (c) c->err = buf;
  else g_student_err = buf;
  return code;
}

}  // namespace sdet

namespace {

// ------------------------------------------------------------------ kernels
// x[r, :] = (embed[tok(r)] + pe[pos(r)]) / sqrt(d)        (model.py:144-148: the scaling is applied AFTER adding pe)
// tok(r) = tokens[(r / L) * tok_ld + tok_off + r % L], pos(r) = pos0 + r % L
__global__ void student_embed_kernel(const int* __restrict__ tokens, int tok_ld, int tok_off, int L, int pos0, int rows,
                                     const float* __restrict__ embed, const float* __restrict__ pe, int d, int vocab,
                                     float inv_sqrt_d, bf16* __restrict__ out, int ldo) {
  const int r = blockIdx.x;
  if (r >= rows) return;
  const int b = r / L, i = r % L;
  int tok = tokens[(size_t)b * tok_ld + tok_off + i];
  tok = min(max(tok, 0), vocab - 1);
  const float* e = embed + (size_t)tok * d;
  const float* p = pe + (size_t)(pos0 + i) * d;
  for (int c = threadIdx.x; c < d; c += blockDim.x) out[(size_t)r * ldo + c] = __float2bfloat16((e[c] + p[c]) * inv_sqrt_d);
}

// out[r, :] = LN(x[r, :]) * gamma + beta over `cols` columns (one warp per row, fp32 statistics)
__global__ void student_ln_kernel(const bf16* __restrict__ x, int ldx, int rows, int cols, const float* __restrict__ gamma,
                                  const float* __restrict__ beta, float eps, bf16* __restrict__ out, int ldo) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= rows) return;
  const bf16* xr = x + (size_t)warp * ldx;
  float s = 0.f;
  for (int c = lane; c < cols; c += 32) s += __bfloat162float(xr[c]);
  const float mean = warp_sum(s) / (float)cols;
  float q = 0.f;
  for (int c = lane; c < cols; c += 32) {
    const float v = __bfloat162float(xr[c]) - mean;
    q += v * v;
  }
  const float rstd = rsqrtf(warp_sum(q) / (float)cols + eps);
  for (int c = lane; c < cols; c += 32)
    out[(size_t)warp * ldo + c] = __float2bfloat16((__bfloat162float(xr[c]) - mean) * rstd * gamma[c] + beta[c]);
}

// One warp per (query row, head): softmax(q k^T * scale + mask) v over a handful of keys (<= 128).
//   q row r at q[r * ldq + h * hd]; key / value j of batch b at kv[(b * kv_rows + j) * ldkv + {k_off, v_off} + h * hd]
//   causal != 0: keys 0 .. pos0 + (r % Lq) (the query's own position included); else all n_keys
//   tokens != nullptr: key j is masked when tokens[b * tok_ld + j] == pad (tgt_key_padding_mask, masking.py:14)
//   DROP (distillation step only): out = (D o P) v with D the dropout mask of site dr over the element index
//   ((b * gridDim.y + h) * Lq + i) * n_keys + j; the softmax sum is over the undropped probabilities
constexpr int S_MAX_KEYS = 128, S_MAX_HD = 128;
template <bool DROP>
__global__ void __launch_bounds__(32) student_attn_kernel(const bf16* __restrict__ q, int ldq, int Lq, int pos0,
                                                          const bf16* __restrict__ kv, int kv_rows, int ldkv, int k_off, int v_off,
                                                          int n_keys, int causal, const int* __restrict__ tokens, int tok_ld, int pad,
                                                          int hd, float scale, bf16* __restrict__ out, int ldo, SDrop dr) {
  __shared__ float sq[S_MAX_HD];
  __shared__ float sp[S_MAX_KEYS];
  const int r = blockIdx.x, h = blockIdx.y, lane = threadIdx.x;
  const int b = r / Lq, i = r % Lq;
  const int nk = causal ? min(pos0 + i + 1, n_keys) : n_keys;
  for (int c = lane; c < hd; c += 32) sq[c] = __bfloat162float(q[(size_t)r * ldq + h * hd + c]) * scale;
  __syncwarp();
  float mx = -INFINITY;
  for (int j = lane; j < nk; j += 32) {
    const bf16* kr = kv + ((size_t)b * kv_rows + j) * ldkv + k_off + h * hd;
    float s = 0.f;
    for (int c = 0; c < hd; c += 2) {
      const float2 k2 = __bfloat1622float2(*reinterpret_cast<const bf162*>(kr + c));
      s = fmaf(sq[c], k2.x, s);
      s = fmaf(sq[c + 1], k2.y, s);
    }
    if (tokens != nullptr && tokens[(size_t)b * tok_ld + j] == pad) s = -INFINITY;
    sp[j] = s;
    mx = fmaxf(mx, s);
  }
  mx = warp_max(mx);
  float sum = 0.f;
  for (int j = lane; j < nk; j += 32) {
    const float p = __expf(sp[j] - mx);
    sum += p;
    if constexpr (DROP)
      sp[j] = p * dropout_scale(dr.seed, dr.step, dr.site, (unsigned)(((b * gridDim.y + h) * Lq + i) * n_keys + j), dr.p, dr.inv_keep);
    else
      sp[j] = p;
  }
  sum = warp_sum(sum);
  __syncwarp();
  const float inv = 1.f / sum;
  for (int c = lane; c < hd; c += 32) {
    float acc = 0.f;
    for (int j = 0; j < nk; ++j)
      acc = fmaf(sp[j], __bfloat162float(kv[((size_t)b * kv_rows + j) * ldkv + v_off + h * hd + c]), acc);
    out[(size_t)r * ldo + h * hd + c] = __float2bfloat16(acc * inv);
  }
}

// tokens[b * tok_ld + pos + 1] = argmax_v logits[b, v]  (first maximum, like torch.argmax); one CTA per row
__global__ void __launch_bounds__(256) student_argmax_kernel(const float* __restrict__ logits, int ld, int vocab, int* __restrict__ tokens,
                                                             int tok_ld, int pos) {
  __shared__ float sv[8];
  __shared__ int si[8];
  const int b = blockIdx.x;
  const float* row = logits + (size_t)b * ld;
  float best = -INFINITY;
  int bi = 0x7fffffff;
  for (int v = threadIdx.x; v < vocab; v += blockDim.x) {
    const float x = row[v];
    if (x > best) {
      best = x;
      bi = v;
    }
  }
  for (int o = 16; o > 0; o >>= 1) {
    const float ob = __shfl_xor_sync(0xffffffffu, best, o);
    const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
    if (ob > best || (ob == best && oi < bi)) {
      best = ob;
      bi = oi;
    }
  }
  if ((threadIdx.x & 31) == 0) {
    sv[threadIdx.x >> 5] = best;
    si[threadIdx.x >> 5] = bi;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < 8; ++w)
      if (sv[w] > best || (sv[w] == best && si[w] < bi)) {
        best = sv[w];
        bi = si[w];
      }
    tokens[(size_t)b * tok_ld + pos + 1] = bi;
  }
}

__global__ void student_init_tokens_kernel(int* tokens, int n, int tok_ld, int cls) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b < n) tokens[(size_t)b * tok_ld] = cls;
}
// out_len = 1 + (first step s whose tokens[:, s + 1] are ALL sep, + 1), else max_len + 1   (model.py:184)
__global__ void student_finish_kernel(const int* __restrict__ tokens, int B, int tok_ld, int max_len, int sep, int* out_len) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  int len = max_len + 1;
  for (int s = 0; s < max_len; ++s) {
    bool all = true;
    for (int b = 0; b < B && all; ++b) all = tokens[(size_t)b * tok_ld + s + 1] == sep;
    if (all) {
      len = s + 2;
      break;
    }
  }
  *out_len = len;
}
__global__ void student_copy_tokens_kernel(const int* __restrict__ src, int src_ld, int* __restrict__ dst, int dst_ld, int B, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < B * n) dst[(size_t)(i / n) * dst_ld + i % n] = src[(size_t)(i / n) * src_ld + i % n];
}

// ------------------------------------------------------------------ host helpers
}  // namespace

namespace sdet {

int s_gemm(gitb200_student* c, const bf16* A, int lda, const bf16* W, int K, int M, int N, const float* bias, const bf16* residual,
           int ldr, int act, bf16* out, int ldo, float* out32, int ldo32, cudaStream_t s) {
  GemmArgs g;
  g.A = A; g.lda = lda; g.W = W; g.ldw = K; g.M = M; g.N = N; g.K = K; g.bias = bias; g.residual = residual; g.ldr = ldr;
  g.act = act; g.out = out; g.ldo = ldo; g.out_f32 = out32; g.ldo32 = ldo32;
  S_CUDA_OK(c, gemm_bf16(g, s, 0));
  return 0;
}
int s_ln(gitb200_student* c, const bf16* x, int ldx, int rows, const float* g, const float* b, bf16* out, int ldo, cudaStream_t s) {
  student_ln_kernel<<<(rows * 32 + 255) / 256, 256, 0, s>>>(x, ldx, rows, c->cfg.d_model, g, b, c->cfg.ln_eps, out, ldo);
  note_launch();
  S_CUDA_OK(c, cudaGetLastError());
  return 0;
}
// embedding of positions pos0 .. pos0 + L - 1 of every sequence (teacher forcing: pos0 = 0; cached decoding: L = 1)
int s_embed(gitb200_student* c, const int* tokens, int tok_ld, int L, int pos0, int rows, bf16* out, cudaStream_t s) {
  student_embed_kernel<<<rows, 128, 0, s>>>(tokens, tok_ld, pos0, L, pos0, rows, c->embed, c->pe, c->cfg.d_model, c->cfg.vocab,
                                            1.0f / sqrtf((float)c->cfg.d_model), out, c->dp);
  note_launch();
  S_CUDA_OK(c, cudaGetLastError());
  return 0;
}
int s_attn(gitb200_student* c, const bf16* q, int ldq, int Lq, int pos0, const bf16* kv, int kv_rows, int ldkv, int k_off, int v_off,
           int n_keys, int causal, const int* tokens, int tok_ld, int rows, bf16* out, int ldo, cudaStream_t s) {
  if (n_keys < 1 || n_keys > S_MAX_KEYS) return sfail(c, GITB200_ERR_INVALID, "student attention over %d keys (1 .. %d)", n_keys, S_MAX_KEYS);
  student_attn_kernel<false><<<dim3(rows, c->cfg.n_head), 32, 0, s>>>(q, ldq, Lq, pos0, kv, kv_rows, ldkv, k_off, v_off, n_keys, causal,
                                                                      tokens, tok_ld, c->cfg.pad, c->hd, 1.0f / sqrtf((float)c->hd), out, ldo,
                                                                      SDrop{});
  note_launch();
  S_CUDA_OK(c, cudaGetLastError());
  return 0;
}
int s_attn_dropout(gitb200_student* c, const bf16* q, int ldq, int Lq, const bf16* kv, int kv_rows, int ldkv, int k_off, int v_off,
                   int n_keys, int causal, const int* tokens, int tok_ld, int rows, bf16* out, int ldo, const SDrop& dr, cudaStream_t s) {
  if (n_keys < 1 || n_keys > S_MAX_KEYS) return sfail(c, GITB200_ERR_INVALID, "student attention over %d keys (1 .. %d)", n_keys, S_MAX_KEYS);
  student_attn_kernel<true><<<dim3(rows, c->cfg.n_head), 32, 0, s>>>(q, ldq, Lq, 0, kv, kv_rows, ldkv, k_off, v_off, n_keys, causal, tokens,
                                                                     tok_ld, c->cfg.pad, c->hd, 1.0f / sqrtf((float)c->hd), out, ldo, dr);
  note_launch();
  S_CUDA_OK(c, cudaGetLastError());
  return 0;
}

}  // namespace sdet

namespace {

const RawW* sfind(gitb200_student* c, const std::string& n) {
  auto it = c->raw.find(n);
  return it == c->raw.end() ? nullptr : &it->second;
}
// fp32 rows [r0, r0 + rows) x cols of `name` -> bf16 [dst_rows, cols] at *out + row offset (zero padded)
int s_w(gitb200_student* c, const std::string& name, int r0, int rows, int cols, bf16* dst, int dst_rows) {
  const RawW* w = sfind(c, name);
  if (!w) return sfail(c, GITB200_ERR_MISSING, "missing weight %s", name.c_str());
  if (w->shape.size() != 2 || w->shape[1] != cols || w->shape[0] < r0 + rows)
    return sfail(c, GITB200_ERR_INVALID, "weight %s has the wrong shape", name.c_str());
  S_CUDA_OK(c, cast_f32_to_bf16(w->p + (size_t)r0 * cols, rows, cols, cols, dst, cols, dst_rows, cols, 0));
  return 0;
}
int s_v(gitb200_student* c, const std::string& name, int off, int n, float* dst) {
  const RawW* w = sfind(c, name);
  if (!w) return sfail(c, GITB200_ERR_MISSING, "missing weight %s", name.c_str());
  if ((int64_t)w->numel() < off + n) return sfail(c, GITB200_ERR_INVALID, "weight %s is too short", name.c_str());
  S_CUDA_OK(c, cudaMemcpy(dst, w->p + off, (size_t)n * sizeof(float), cudaMemcpyDeviceToDevice));
  return 0;
}
template <typename T>
int s_alloc(gitb200_student* c, T** p, size_t n) {
  S_CUDA_OK(c, cudaMalloc(p, n * sizeof(T)));
  S_CUDA_OK(c, cudaMemset(*p, 0, n * sizeof(T)));
  c->allocs.push_back(*p);
  return 0;
}

// The decoder stack over `rows` = B * L query rows at positions pos0 .. pos0 + L - 1 of caches sized for Lmax positions.
// tokens: int [B, tok_ld] (the ids at every position up to pos0 + L - 1; used for the embedding and the padding mask).
int run_layers(gitb200_student* c, int B, int L, int pos0, int Lmax, const int* tokens, int tok_ld, int M, float* logits, cudaStream_t s) {
  const gitb200_student_config& k = c->cfg;
  const int d = k.d_model, dp = c->dp, fp = c->fp, rows = B * L;
  if (pos0 + L > Lmax || Lmax > S_MAX_KEYS || M > S_MAX_KEYS) return sfail(c, GITB200_ERR_INVALID, "sequence / memory longer than %d", S_MAX_KEYS);
  S_TRY(sensure(c, c->x, (size_t)rows * dp));
  S_TRY(sensure(c, c->y, (size_t)rows * dp));
  S_TRY(sensure(c, c->a, (size_t)rows * dp));
  S_TRY(sensure(c, c->q2, (size_t)rows * dp));
  S_TRY(sensure(c, c->h, (size_t)rows * fp));
  S_TRY(s_embed(c, tokens, tok_ld, L, pos0, rows, c->x.p, s));
  for (int l = 0; l < k.n_layers; ++l) {
    const SLayer& W = c->layers[l];
    bf16* cache = c->cache[l].p;
    // self-attention block: x = norm1(x + out_proj(attn(in_proj(x))))
    if (L == Lmax && pos0 == 0) {
      S_TRY(s_gemm(c, c->x.p, dp, W.w_sa_in, d, rows, 3 * dp, W.b_sa_in, nullptr, 0, ACT_NONE, cache, 3 * dp, nullptr, 0, s));
    } else {  // one position per sequence: row b lands at cache[b][pos0]
      if (L != 1) return sfail(c, GITB200_ERR_INVALID, "cached decoding feeds one position at a time");
      S_TRY(s_gemm(c, c->x.p, dp, W.w_sa_in, d, rows, 3 * dp, W.b_sa_in, nullptr, 0, ACT_NONE, cache + (size_t)pos0 * 3 * dp,
                   Lmax * 3 * dp, nullptr, 0, s));
    }
    {
      const bf16* qp = (L == Lmax && pos0 == 0) ? cache : cache + (size_t)pos0 * 3 * dp;
      const int ldq = (L == Lmax && pos0 == 0) ? 3 * dp : Lmax * 3 * dp;
      S_TRY(s_attn(c, qp, ldq, L, pos0, cache, Lmax, 3 * dp, dp, 2 * dp, pos0 + L, 1, tokens, tok_ld, rows, c->a.p, dp, s));
    }
    S_TRY(s_gemm(c, c->a.p, dp, W.w_sa_out, d, rows, dp, W.b_sa_out, c->x.p, dp, ACT_NONE, c->y.p, dp, nullptr, 0, s));
    S_TRY(s_ln(c, c->y.p, dp, rows, W.n1_g, W.n1_b, c->x.p, dp, s));
    // cross-attention block: x = norm2(x + out_proj(attn(q(x), kv(memory))))
    S_TRY(s_gemm(c, c->x.p, dp, W.w_ca_q, d, rows, dp, W.b_ca_q, nullptr, 0, ACT_NONE, c->q2.p, dp, nullptr, 0, s));
    S_TRY(s_attn(c, c->q2.p, dp, L, 0, c->memkv[l].p, M, 2 * dp, 0, dp, M, 0, nullptr, 0, rows, c->a.p, dp, s));
    S_TRY(s_gemm(c, c->a.p, dp, W.w_ca_out, d, rows, dp, W.b_ca_out, c->x.p, dp, ACT_NONE, c->y.p, dp, nullptr, 0, s));
    S_TRY(s_ln(c, c->y.p, dp, rows, W.n2_g, W.n2_b, c->x.p, dp, s));
    // feed-forward block: x = norm3(x + linear2(relu(linear1(x))))
    S_TRY(s_gemm(c, c->x.p, dp, W.w_ff1, d, rows, fp, W.b_ff1, nullptr, 0, ACT_RELU, c->h.p, fp, nullptr, 0, s));
    S_TRY(s_gemm(c, c->h.p, fp, W.w_ff2, fp, rows, dp, W.b_ff2, c->x.p, dp, ACT_NONE, c->y.p, dp, nullptr, 0, s));
    S_TRY(s_ln(c, c->y.p, dp, rows, W.n3_g, W.n3_b, c->x.p, dp, s));
  }
  // vocabulary head (model.py:152)
  S_TRY(s_gemm(c, c->x.p, dp, c->w_vocab, d, rows, c->vp, c->b_vocab, nullptr, 0, ACT_NONE, nullptr, 0, logits, c->vp, s));
  return 0;
}

// memory fp32 [B, M, d] -> per-layer cross-attention K|V [B*M, 2*dp]; caches sized [B][Lmax][3*dp]
int prepare(gitb200_student* c, const float* memory, int B, int M, int Lmax, cudaStream_t s) {
  const gitb200_student_config& k = c->cfg;
  const int d = k.d_model, dp = c->dp;
  if (B < 1 || M < 1 || Lmax < 1) return sfail(c, GITB200_ERR_INVALID, "bad student shapes");
  if (Lmax > k.max_len) return sfail(c, GITB200_ERR_INVALID, "sequence of %d positions exceeds the %d-row positional table", Lmax, k.max_len);
  S_TRY(sensure(c, c->mem, (size_t)B * M * d));
  S_CUDA_OK(c, cast_f32_to_bf16(memory, B * M, d, d, c->mem.p, d, B * M, d, s));
  if ((int)c->cache.size() != k.n_layers) {
    c->cache.resize(k.n_layers);
    c->memkv.resize(k.n_layers);
  }
  for (int l = 0; l < k.n_layers; ++l) {
    S_TRY(sensure(c, c->cache[l], (size_t)B * Lmax * 3 * dp));
    S_TRY(sensure(c, c->memkv[l], (size_t)B * M * 2 * dp));
    S_TRY(s_gemm(c, c->mem.p, d, c->layers[l].w_ca_kv, d, B * M, 2 * dp, c->layers[l].b_ca_kv, nullptr, 0, ACT_NONE, c->memkv[l].p, 2 * dp,
                 nullptr, 0, s));
  }
  return 0;
}

}  // namespace

extern "C" {

const char* gitb200_student_last_error(const gitb200_student* s) { return s ? s->err.c_str() : g_student_err.c_str(); }

int gitb200_student_create(const gitb200_student_config* cfg, int device, gitb200_student** out) {
  if (!cfg || !out) return sfail(nullptr, GITB200_ERR_INVALID, "null argument");
  if (cfg->d_model < 8 || cfg->d_model % 8 != 0 || cfg->n_head < 1 || cfg->d_model % cfg->n_head != 0 ||
      (cfg->d_model / cfg->n_head) % 2 != 0 || cfg->d_model / cfg->n_head > S_MAX_HD || cfg->d_ffn % 8 != 0 || cfg->n_layers < 1 ||
      cfg->vocab < 2 || cfg->max_len < 2)
    return sfail(nullptr, GITB200_ERR_INVALID, "unsupported student configuration");
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess || device < 0 || device >= count)
    return sfail(nullptr, GITB200_ERR_CUDA, "no usable CUDA device %d (the student decoder has no CPU fallback)", device);
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess || prop.major != 10)
    return sfail(nullptr, GITB200_ERR_CUDA, "device %d is not an sm_100 GPU", device);
  gitb200_student* c = new gitb200_student();
  c->cfg = *cfg;
  c->device = device;
  c->dp = round_up(cfg->d_model, 128);
  c->fp = round_up(cfg->d_ffn, 128);
  c->vp = round_up(cfg->vocab, 256);
  c->hd = cfg->d_model / cfg->n_head;
  *out = c;
  return GITB200_OK;
}

void gitb200_student_destroy(gitb200_student* c) {
  if (!c) return;
  cudaSetDevice(c->device);
  for (auto& kv : c->raw) cudaFree(kv.second.p);
  for (void* p : c->allocs) cudaFree(p);
  for (auto* b : {&c->x, &c->y, &c->a, &c->q2, &c->h, &c->mem}) cudaFree(b->p);
  for (auto& b : c->cache) cudaFree(b.p);
  for (auto& b : c->memkv) cudaFree(b.p);
  cudaFree(c->logits.p);
  cudaFree(c->toks.p);
  sdet::student_train_destroy(c);
  delete c;
}

int gitb200_student_load_weight(gitb200_student* c, const char* name, const float* data, int ndim, const int64_t* shape) {
  if (!c || !name || !data || ndim < 1 || !shape) return sfail(c, GITB200_ERR_INVALID, "bad load_weight argument");
  S_CUDA_OK(c, cudaSetDevice(c->device));
  RawW w;
  w.shape.assign(shape, shape + ndim);
  S_CUDA_OK(c, cudaMalloc(&w.p, w.numel() * sizeof(float)));
  S_CUDA_OK(c, cudaMemcpy(w.p, data, w.numel() * sizeof(float), cudaMemcpyDefault));
  auto it = c->raw.find(name);
  if (it != c->raw.end()) cudaFree(it->second.p);
  c->raw[name] = w;
  c->finalized = false;
  return GITB200_OK;
}

int gitb200_student_finalize(gitb200_student* c) {
  if (!c) return GITB200_ERR_INVALID;
  S_CUDA_OK(c, cudaSetDevice(c->device));
  const gitb200_student_config& k = c->cfg;
  const int d = k.d_model, dp = c->dp, fp = c->fp, f = k.d_ffn;
  c->layers.assign(k.n_layers, SLayer{});
  for (int l = 0; l < k.n_layers; ++l) {
    SLayer& W = c->layers[l];
    const std::string p = "decoder.layers." + std::to_string(l) + ".";
    // self-attention in_proj [3d, d] -> q | k | v blocks of dp rows each
    S_TRY(s_alloc(c, &W.w_sa_in, (size_t)3 * dp * d));
    S_TRY(s_alloc(c, &W.b_sa_in, (size_t)3 * dp));
    for (int t = 0; t < 3; ++t) {
      S_TRY(s_w(c, p + "self_attn.in_proj_weight", t * d, d, d, W.w_sa_in + (size_t)t * dp * d, dp));
      S_TRY(s_v(c, p + "self_attn.in_proj_bias", t * d, d, W.b_sa_in + (size_t)t * dp));
    }
    S_TRY(s_alloc(c, &W.w_sa_out, (size_t)dp * d));
    S_TRY(s_alloc(c, &W.b_sa_out, (size_t)dp));
    S_TRY(s_w(c, p + "self_attn.out_proj.weight", 0, d, d, W.w_sa_out, dp));
    S_TRY(s_v(c, p + "self_attn.out_proj.bias", 0, d, W.b_sa_out));
    // cross-attention: q from the text rows, k | v from memory
    S_TRY(s_alloc(c, &W.w_ca_q, (size_t)dp * d));
    S_TRY(s_alloc(c, &W.b_ca_q, (size_t)dp));
    S_TRY(s_w(c, p + "multihead_attn.in_proj_weight", 0, d, d, W.w_ca_q, dp));
    S_TRY(s_v(c, p + "multihead_attn.in_proj_bias", 0, d, W.b_ca_q));
    S_TRY(s_alloc(c, &W.w_ca_kv, (size_t)2 * dp * d));
    S_TRY(s_alloc(c, &W.b_ca_kv, (size_t)2 * dp));
    for (int t = 0; t < 2; ++t) {
      S_TRY(s_w(c, p + "multihead_attn.in_proj_weight", (t + 1) * d, d, d, W.w_ca_kv + (size_t)t * dp * d, dp));
      S_TRY(s_v(c, p + "multihead_attn.in_proj_bias", (t + 1) * d, d, W.b_ca_kv + (size_t)t * dp));
    }
    S_TRY(s_alloc(c, &W.w_ca_out, (size_t)dp * d));
    S_TRY(s_alloc(c, &W.b_ca_out, (size_t)dp));
    S_TRY(s_w(c, p + "multihead_attn.out_proj.weight", 0, d, d, W.w_ca_out, dp));
    S_TRY(s_v(c, p + "multihead_attn.out_proj.bias", 0, d, W.b_ca_out));
    // feed-forward: linear1 [f, d] -> [fp, d]; linear2 [d, f] -> [dp, fp] (K padded with zero columns)
    S_TRY(s_alloc(c, &W.w_ff1, (size_t)fp * d));
    S_TRY(s_alloc(c, &W.b_ff1, (size_t)fp));
    S_TRY(s_w(c, p + "linear1.weight", 0, f, d, W.w_ff1, fp));
    S_TRY(s_v(c, p + "linear1.bias", 0, f, W.b_ff1));
    S_TRY(s_alloc(c, &W.w_ff2, (size_t)dp * fp));
    S_TRY(s_alloc(c, &W.b_ff2, (size_t)dp));
    {
      const RawW* w = sfind(c, p + "linear2.weight");
      if (!w) return sfail(c, GITB200_ERR_MISSING, "missing weight %slinear2.weight", p.c_str());
      if (w->shape.size() != 2 || w->shape[0] != d || w->shape[1] != f) return sfail(c, GITB200_ERR_INVALID, "linear2.weight has the wrong shape");
      S_CUDA_OK(c, cast_f32_to_bf16(w->p, d, f, f, W.w_ff2, fp, dp, fp, 0));
    }
    S_TRY(s_v(c, p + "linear2.bias", 0, d, W.b_ff2));
    float** ln[6] = {&W.n1_g, &W.n1_b, &W.n2_g, &W.n2_b, &W.n3_g, &W.n3_b};
    const char* names[6] = {"norm1.weight", "norm1.bias", "norm2.weight", "norm2.bias", "norm3.weight", "norm3.bias"};
    for (int i = 0; i < 6; ++i) {
      S_TRY(s_alloc(c, ln[i], (size_t)d));
      S_TRY(s_v(c, p + names[i], 0, d, *ln[i]));
    }
  }
  S_TRY(s_alloc(c, &c->embed, (size_t)k.vocab * d));
  S_TRY(s_v(c, "embed.weight", 0, k.vocab * d, c->embed));
  S_TRY(s_alloc(c, &c->pe, (size_t)k.max_len * d));
  S_TRY(s_v(c, "pos_enc.pe", 0, k.max_len * d, c->pe));
  S_TRY(s_alloc(c, &c->w_vocab, (size_t)c->vp * d));
  S_TRY(s_alloc(c, &c->b_vocab, (size_t)c->vp));
  S_TRY(s_w(c, "linear.weight", 0, k.vocab, d, c->w_vocab, c->vp));
  S_TRY(s_v(c, "linear.bias", 0, k.vocab, c->b_vocab));
  S_CUDA_OK(c, cudaDeviceSynchronize());
  if (!c->keep_raw) {
    for (auto& kv : c->raw) cudaFree(kv.second.p);
    c->raw.clear();
  }
  c->finalized = true;
  return GITB200_OK;
}

int gitb200_student_logits_ld(const gitb200_student* c) { return c ? c->vp : 0; }

int gitb200_student_forward_decoder(gitb200_student* c, const int32_t* tokens, const float* memory, int B, int L, int M, float* logits,
                                    void* stream) {
  if (!c || !tokens || !memory || !logits) return sfail(c, GITB200_ERR_INVALID, "bad forward_decoder argument");
  if (!c->finalized) return sfail(c, GITB200_ERR_STATE, "call gitb200_student_finalize first");
  S_CUDA_OK(c, cudaSetDevice(c->device));
  cudaStream_t s = (cudaStream_t)stream;
  S_TRY(prepare(c, memory, B, M, L, s));
  return run_layers(c, B, L, 0, L, tokens, L, M, logits, s);
}

int gitb200_student_greedy_decode(gitb200_student* c, const float* memory, int B, int M, int max_len, int32_t* tokens_out, int32_t* out_len,
                                  void* stream) {
  if (!c || !memory || !tokens_out || !out_len || max_len < 1) return sfail(c, GITB200_ERR_INVALID, "bad greedy_decode argument");
  if (!c->finalized) return sfail(c, GITB200_ERR_STATE, "call gitb200_student_finalize first");
  S_CUDA_OK(c, cudaSetDevice(c->device));
  cudaStream_t s = (cudaStream_t)stream;
  const int Lmax = max_len + 1;  // CLS + max_len generated tokens; the last one is never fed back
  S_TRY(prepare(c, memory, B, M, Lmax, s));
  S_TRY(sensure(c, c->logits, (size_t)B * c->vp));
  S_TRY(sensure(c, c->toks, (size_t)B * Lmax));
  S_CUDA_OK(c, cudaMemsetAsync(c->toks.p, 0, (size_t)B * Lmax * sizeof(int), s));
  student_init_tokens_kernel<<<(B + 127) / 128, 128, 0, s>>>(c->toks.p, B, Lmax, c->cfg.cls);
  note_launch();
  for (int t = 0; t < max_len; ++t) {  // model.py:173: every step feeds the newest token; all rows keep decoding
    S_TRY(run_layers(c, B, 1, t, Lmax, c->toks.p, Lmax, M, c->logits.p, s));
    student_argmax_kernel<<<B, 256, 0, s>>>(c->logits.p, c->vp, c->cfg.vocab, c->toks.p, Lmax, t);
    note_launch();
  }
  student_finish_kernel<<<1, 32, 0, s>>>(c->toks.p, B, Lmax, max_len, c->cfg.sep, out_len);
  student_copy_tokens_kernel<<<(B * Lmax + 255) / 256, 256, 0, s>>>(c->toks.p, Lmax, tokens_out, Lmax, B, Lmax);
  note_launch(2);
  S_CUDA_OK(c, cudaGetLastError());
  return GITB200_OK;
}

}  // extern "C"

// HBM-bound helper kernels of the captioning path: LayerNorm (SURVEY K2/K7 tail), patch im2col +
// bf16 cast (K1 front), CLS rows, text embedding + LN (K8), text K/V scatter, dtype casts.
// All are one-pass, 16-byte vectorised, one warp per row where a row reduction is needed.
#include "common.cuh"
#include "kernels.h"

namespace {

// ------------------------------------------------------------------ LayerNorm: one warp per row
// Persistent: the grid is sized to the machine and every warp walks rows with a grid stride, the next row's 16-byte loads
// are issued before the current row is reduced, and gamma / beta sit in shared memory (loaded once per CTA; the first
// version re-read 6 KB of them from L1 for every 1.5 KB row and started one 8-row CTA per 12 KB of traffic).
// REMAP: output rows go through LayerNormArgs::out_row_base (a separate instantiation, so the plain kernel is untouched).
template <int VECS, bool REMAP>  // 16-byte vectors per lane: cols = 32 * 8 * VECS  (768 -> 3, 1024 -> 4)
__global__ void __launch_bounds__(256, 3) layernorm_kernel(LayerNormArgs a) {
  __shared__ float4 sg[VECS * 64], sb[VECS * 64];  // gamma / beta as float4: index (i * 32 + lane) * 2 + {0, 1}
  for (int i = threadIdx.x; i < VECS * 64; i += blockDim.x) {
    sg[i] = __ldg(reinterpret_cast<const float4*>(a.gamma) + i);
    sb[i] = __ldg(reinterpret_cast<const float4*>(a.beta) + i);
  }
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const int n_warps = (gridDim.x * blockDim.x) >> 5;
  int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  uint4 nxt[VECS];
  if (warp < a.rows) {
#pragma unroll
    for (int i = 0; i < VECS; ++i) nxt[i] = *reinterpret_cast<const uint4*>(a.x + (size_t)warp * a.ldx + (i * 32 + lane) * 8);
  }
  for (; warp < a.rows; warp += n_warps) {
  float v[VECS * 8];
#pragma unroll
  for (int i = 0; i < VECS; ++i) {
    const uint4 u = nxt[i];
    const float2 f0 = unpack_bf16(u.x), f1 = unpack_bf16(u.y), f2 = unpack_bf16(u.z), f3 = unpack_bf16(u.w);
    v[i * 8 + 0] = f0.x; v[i * 8 + 1] = f0.y; v[i * 8 + 2] = f1.x; v[i * 8 + 3] = f1.y;
    v[i * 8 + 4] = f2.x; v[i * 8 + 5] = f2.y; v[i * 8 + 6] = f3.x; v[i * 8 + 7] = f3.y;
  }
  if (warp + n_warps < a.rows) {  // next row of this warp: in flight while this one is reduced and written
#pragma unroll
    for (int i = 0; i < VECS; ++i) nxt[i] = *reinterpret_cast<const uint4*>(a.x + (size_t)(warp + n_warps) * a.ldx + (i * 32 + lane) * 8);
  }
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < VECS * 8; ++i) s += v[i];
  const float mean = warp_sum(s) / (float)a.cols;
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < VECS * 8; ++i) {
    const float d = v[i] - mean;
    q += d * d;
  }
  const float rstd = rsqrtf(warp_sum(q) / (float)a.cols + a.eps);
  const float* add = a.addend ? a.addend + (size_t)((warp / a.add_group) % a.add_period) * a.cols : nullptr;
  const size_t orow = REMAP ? (size_t)a.out_row_base[warp / a.out_group] + warp % a.out_group : (size_t)warp;
  float st1 = 0.f, st2 = 0.f;
#pragma unroll
  for (int i = 0; i < VECS; ++i) {
    const int c = (i * 32 + lane) * 8;
    const float4 g0 = sg[(i * 32 + lane) * 2], g1 = sg[(i * 32 + lane) * 2 + 1];
    const float4 b0 = sb[(i * 32 + lane) * 2], b1 = sb[(i * 32 + lane) * 2 + 1];
    float o[8];
    o[0] = (v[i * 8 + 0] - mean) * rstd * g0.x + b0.x;
    o[1] = (v[i * 8 + 1] - mean) * rstd * g0.y + b0.y;
    o[2] = (v[i * 8 + 2] - mean) * rstd * g0.z + b0.z;
    o[3] = (v[i * 8 + 3] - mean) * rstd * g0.w + b0.w;
    o[4] = (v[i * 8 + 4] - mean) * rstd * g1.x + b1.x;
    o[5] = (v[i * 8 + 5] - mean) * rstd * g1.y + b1.y;
    o[6] = (v[i * 8 + 6] - mean) * rstd * g1.z + b1.z;
    o[7] = (v[i * 8 + 7] - mean) * rstd * g1.w + b1.w;
    if (add) {
      const float4 a0 = __ldg(reinterpret_cast<const float4*>(add + c));
      const float4 a1 = __ldg(reinterpret_cast<const float4*>(add + c + 4));
      o[0] += a0.x; o[1] += a0.y; o[2] += a0.z; o[3] += a0.w;
      o[4] += a1.x; o[5] += a1.y; o[6] += a1.z; o[7] += a1.w;
    }
    if (a.out) {
      uint4 u;
      u.x = pack_bf16(o[0], o[1]); u.y = pack_bf16(o[2], o[3]); u.z = pack_bf16(o[4], o[5]); u.w = pack_bf16(o[6], o[7]);
      *reinterpret_cast<uint4*>(a.out + orow * a.ldo + c) = u;
      if (a.stats_out) {
        const float2 r0 = unpack_bf16(u.x), r1 = unpack_bf16(u.y), r2 = unpack_bf16(u.z), r3 = unpack_bf16(u.w);
        st1 += (r0.x + r0.y) + (r1.x + r1.y) + (r2.x + r2.y) + (r3.x + r3.y);
        st2 += r0.x * r0.x + r0.y * r0.y + r1.x * r1.x + r1.y * r1.y + r2.x * r2.x + r2.y * r2.y + r3.x * r3.x + r3.y * r3.y;
      }
    }
    if (a.out_f32) {
      float4* p = reinterpret_cast<float4*>(a.out_f32 + orow * a.ldo32 + c);
      p[0] = make_float4(o[0], o[1], o[2], o[3]);
      p[1] = make_float4(o[4], o[5], o[6], o[7]);
    }
  }
  if (a.stats_out) {
    st1 = warp_sum(st1);
    st2 = warp_sum(st2);
    // slot 0 of the row's `stats_slots` partial-sum slots holds the whole row, the others are zero (the consuming GEMM adds all)
    for (int sl = lane; sl < a.stats_slots; sl += 32)
      reinterpret_cast<float2*>(a.stats_out)[(size_t)warp * a.stats_slots + sl] = sl == 0 ? make_float2(st1, st2) : make_float2(0.f, 0.f);
  }
  }
}

// one warp per output row n: fold gamma into the weights, beta into the bias, and compute the column sums
__global__ void ln_fold_weight_kernel(const float* __restrict__ w, int N, int K, const float* __restrict__ gamma,
                                      const float* __restrict__ beta, const float* __restrict__ bias, bf16* __restrict__ wf,
                                      float* __restrict__ colsum, float* __restrict__ bias_f) {
  const int n = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (n >= N) return;
  float cs = 0.f, bs = 0.f;
  for (int k = lane; k < K; k += 32) {
    const float wv = w[(size_t)n * K + k];
    const bf16 r = __float2bfloat16(wv * gamma[k]);
    wf[(size_t)n * K + k] = r;
    cs += __bfloat162float(r);
    bs += wv * beta[k];
  }
  cs = warp_sum(cs);
  bs = warp_sum(bs);
  if (lane == 0) {
    colsum[n] = cs;
    bias_f[n] = bias[n] + bs;
  }
}

// ------------------------------------------------------------------ patch im2col + cast
// out[(f*G*G + gy*G + gx), c*P*P + ky*P + kx] = frames[f, c, gy*P + ky, gx*P + kx]; columns >= 3*P*P are zero.
__global__ void __launch_bounds__(256) im2col_kernel(const float* __restrict__ frames, int n_frames, int res, int P,
                                                     int kpad, bf16* __restrict__ out) {
  const int G = res / P;
  const int kreal = 3 * P * P;
  const int chunks_per_row = kpad / 8;
  const size_t total = (size_t)n_frames * G * G * chunks_per_row;
  for (size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
    const int chunk = (int)(idx % chunks_per_row);
    const size_t row = idx / chunks_per_row;
    const int gx = (int)(row % G);
    const int gy = (int)((row / G) % G);
    const int f = (int)(row / ((size_t)G * G));
    float v[8];
    if (P % 8 == 0 && res % 4 == 0) {
      // 8 consecutive k share (channel, patch row): one aligned 32-byte run of the source row -> two 16-byte loads
      // (ViT-B/16; the scalar path below, 8 loads + 8 index decompositions per thread, ran at 26 % of the HBM bandwidth)
      const int k = chunk * 8;
      if (k < kreal) {
        const int c = k / (P * P);
        const int rem = k - c * P * P;
        const int ky = rem / P;
        const int kx = rem - ky * P;
        const float4* src = reinterpret_cast<const float4*>(frames + (((size_t)f * 3 + c) * res + (gy * P + ky)) * res + gx * P + kx);
        const float4 a = __ldg(src), b = __ldg(src + 1);
        v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
      } else {
#pragma unroll
        for (int j = 0; j < 8; ++j) v[j] = 0.f;
      }
    } else
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int k = chunk * 8 + j;
      float val = 0.f;
      if (k < kreal) {
        const int c = k / (P * P);
        const int rem = k - c * P * P;
        const int ky = rem / P;
        const int kx = rem - ky * P;
        val = __ldg(frames + (((size_t)f * 3 + c) * res + (gy * P + ky)) * res + gx * P + kx);
      }
      v[j] = val;
    }
    uint4 u;
    u.x = pack_bf16(v[0], v[1]); u.y = pack_bf16(v[2], v[3]); u.z = pack_bf16(v[4], v[5]); u.w = pack_bf16(v[6], v[7]);
    *reinterpret_cast<uint4*>(out + row * kpad + chunk * 8) = u;
  }
}

__global__ void cls_rows_kernel(const float* __restrict__ cls, const bf16* __restrict__ pos, int n_frames, int T,
                                int width, bf16* __restrict__ x) {
  const int f = blockIdx.x;
  for (int c = threadIdx.x; c < width; c += blockDim.x)
    x[(size_t)f * T * width + c] = __float2bfloat16(cls[c] + __bfloat162float(pos[c]));
}

// ------------------------------------------------------------------ text embedding + LayerNorm (one warp per row)
template <int VECS>
__global__ void __launch_bounds__(128) embed_text_kernel(const int* __restrict__ tokens, const int* __restrict__ positions,
                                                         int pos_const, int n_rows, const float* __restrict__ words,
                                                         const float* __restrict__ pos_table,
                                                         const float* __restrict__ gamma, const float* __restrict__ beta,
                                                         float eps, int width, bf16* __restrict__ out) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (warp >= n_rows) return;
  const int tok = tokens[warp];
  const int pos = positions ? positions[warp] : pos_const;
  const float* w = words + (size_t)tok * width;
  const float* p = pos_table + (size_t)pos * width;
  float v[VECS * 8];
#pragma unroll
  for (int i = 0; i < VECS * 2; ++i) {
    const int c = (i * 32 + lane) * 4;
    const float4 a = __ldg(reinterpret_cast<const float4*>(w + c));
    const float4 b = __ldg(reinterpret_cast<const float4*>(p + c));
    v[i * 4 + 0] = a.x + b.x; v[i * 4 + 1] = a.y + b.y; v[i * 4 + 2] = a.z + b.z; v[i * 4 + 3] = a.w + b.w;
  }
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < VECS * 8; ++i) s += v[i];
  const float mean = warp_sum(s) / (float)width;
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < VECS * 8; ++i) q += (v[i] - mean) * (v[i] - mean);
  const float rstd = rsqrtf(warp_sum(q) / (float)width + eps);
#pragma unroll
  for (int i = 0; i < VECS * 2; ++i) {
    const int c = (i * 32 + lane) * 4;
    const float4 g = __ldg(reinterpret_cast<const float4*>(gamma + c));
    const float4 b = __ldg(reinterpret_cast<const float4*>(beta + c));
    uint2 u;
    u.x = pack_bf16((v[i * 4 + 0] - mean) * rstd * g.x + b.x, (v[i * 4 + 1] - mean) * rstd * g.y + b.y);
    u.y = pack_bf16((v[i * 4 + 2] - mean) * rstd * g.z + b.z, (v[i * 4 + 3] - mean) * rstd * g.w + b.w);
    *reinterpret_cast<uint2*>(out + (size_t)warp * width + c) = u;
  }
}

// txt_kv[(pos * n_slots + r / slot_div) * kv_width + c] = qkv[r * ld + q_width + c]
__global__ void store_text_kv_kernel(const bf16* __restrict__ qkv, int ld_qkv, int n_rows, int kv_width, int q_width,
                                     const int* __restrict__ pos, int pos_const, int slot_div, int n_slots,
                                     bf16* __restrict__ txt_kv) {
  const int chunks = kv_width / 8;
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= n_rows * chunks) return;
  const int r = idx / chunks, c = (idx % chunks) * 8;
  const int p = pos ? pos[r] : pos_const;
  *reinterpret_cast<uint4*>(txt_kv + ((size_t)p * n_slots + r / slot_div) * kv_width + c) =
      *reinterpret_cast<const uint4*>(qkv + (size_t)r * ld_qkv + q_width + c);
}

__global__ void cast_f32_bf16_kernel(const float* __restrict__ src, int rows, int cols, int lds, bf16* __restrict__ dst,
                                     int ldd, int dst_rows, int dst_cols) {
  // dst is [dst_rows, dst_cols] (ldd); region outside [rows, cols] is zero padded
  const size_t total = (size_t)dst_rows * dst_cols;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int r = (int)(i / dst_cols), c = (int)(i % dst_cols);
    const float v = (r < rows && c < cols) ? src[(size_t)r * lds + c] : 0.f;
    dst[(size_t)r * ldd + c] = __float2bfloat16(v);
  }
}
__global__ void cast_bf16_f32_kernel(const bf16* __restrict__ src, int rows, int cols, int lds, float* __restrict__ dst,
                                     int ldd) {
  const size_t total = (size_t)rows * cols;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int r = (int)(i / cols), c = (int)(i % cols);
    dst[(size_t)r * ldd + c] = __bfloat162float(src[(size_t)r * lds + c]);
  }
}

__global__ void assemble_window_kernel(const bf16* __restrict__ ring, int first, int cap, int n, int T, int W,
                                       const float* __restrict__ temporal, bf16* __restrict__ vf) {
  const size_t chunks_per_row = W / 8;
  const size_t total = (size_t)n * T * chunks_per_row;
  for (size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
    const int c = (int)(idx % chunks_per_row) * 8;
    const size_t row = idx / chunks_per_row;
    const int i = (int)(row / T), t = (int)(row % T);
    const int slot = (first + i) % cap;
    const uint4 u = *reinterpret_cast<const uint4*>(ring + ((size_t)slot * T + t) * W + c);
    float2 a = unpack_bf16(u.x), b = unpack_bf16(u.y), d = unpack_bf16(u.z), e = unpack_bf16(u.w);
    if (temporal) {
      const float4 t0 = __ldg(reinterpret_cast<const float4*>(temporal + (size_t)i * W + c));
      const float4 t1 = __ldg(reinterpret_cast<const float4*>(temporal + (size_t)i * W + c + 4));
      a.x += t0.x; a.y += t0.y; b.x += t0.z; b.y += t0.w; d.x += t1.x; d.y += t1.y; e.x += t1.z; e.y += t1.w;
    }
    uint4 o;
    o.x = pack_bf16(a.x, a.y); o.y = pack_bf16(b.x, b.y); o.z = pack_bf16(d.x, d.y); o.w = pack_bf16(e.x, e.y);
    *reinterpret_cast<uint4*>(vf + row * W + c) = o;
  }
}

// The windows of k streams of the multi-stream pool, n frames each: window w, frame i (0 = oldest), token t is
//   vf[(w * n + i) * T + t, :] = bf16(ring[(base + (first + i) % cap) * T + t, :] + temporal[i, :])
// with oldest[w] = base + first (base = the stream's first ring slot, a multiple of cap); oldest == nullptr: oldest_const.
// The arithmetic of assemble_window_kernel; vf32 != nullptr writes the bf16-rounded values as fp32 instead of vf.
__global__ void assemble_windows_kernel(const bf16* __restrict__ ring, const int* __restrict__ oldest, int oldest_const, int k,
                                        int n, int cap, int T, int W, const float* __restrict__ temporal, bf16* __restrict__ vf,
                                        float* __restrict__ vf32) {
  const size_t chunks_per_row = W / 8;
  const size_t total = (size_t)k * n * T * chunks_per_row;
  for (size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
    const int c = (int)(idx % chunks_per_row) * 8;
    const size_t row = idx / chunks_per_row;
    const int w = (int)(row / ((size_t)n * T));
    const int r = (int)(row % ((size_t)n * T));
    const int i = r / T, t = r % T;
    const int o = oldest ? oldest[w] : oldest_const;
    const int first = o % cap;
    const int slot = o - first + (first + i) % cap;
    const uint4 u = *reinterpret_cast<const uint4*>(ring + ((size_t)slot * T + t) * W + c);
    float2 a = unpack_bf16(u.x), b = unpack_bf16(u.y), d = unpack_bf16(u.z), e = unpack_bf16(u.w);
    const float4 t0 = __ldg(reinterpret_cast<const float4*>(temporal + (size_t)i * W + c));
    const float4 t1 = __ldg(reinterpret_cast<const float4*>(temporal + (size_t)i * W + c + 4));
    a.x += t0.x; a.y += t0.y; b.x += t0.z; b.y += t0.w; d.x += t1.x; d.y += t1.y; e.x += t1.z; e.y += t1.w;
    uint4 q;
    q.x = pack_bf16(a.x, a.y); q.y = pack_bf16(b.x, b.y); q.z = pack_bf16(d.x, d.y); q.w = pack_bf16(e.x, e.y);
    if (vf32) {
      const float2 r0 = unpack_bf16(q.x), r1 = unpack_bf16(q.y), r2 = unpack_bf16(q.z), r3 = unpack_bf16(q.w);
      float4* p = reinterpret_cast<float4*>(vf32 + row * W + c);
      p[0] = make_float4(r0.x, r0.y, r1.x, r1.y);
      p[1] = make_float4(r2.x, r2.y, r3.x, r3.y);
    } else {
      *reinterpret_cast<uint4*>(vf + row * W + c) = q;
    }
  }
}

__global__ void fill_positions_kernel(int* pos, int* n_text, int rows, int L) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r < rows) {
    pos[r] = r % L;
    n_text[r] = r % L + 1;
  }
}

// Prompt K/V fan-out: dst[(p * rows + r) * width + c] = src[(p * n_clips + r / rows_per_clip) * width + c] for text positions
// p < n_pos; 16-byte chunks (width % 8 == 0).  Every decode row gets its clip's prompt K/V in its OWN slot, so that both ways
// of following the beams (ancestor table or not) read the prompt wherever they look.
__global__ void fanout_prefix_kv_kernel(const bf16* __restrict__ src, bf16* __restrict__ dst, int n_pos, int n_clips,
                                        int rows_per_clip, int width) {
  const int w8 = width / 8, rows = n_clips * rows_per_clip;
  const size_t total = (size_t)n_pos * rows * w8;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int c = (int)(i % w8);
    const size_t pr = i / w8;
    const int r = (int)(pr % rows), p = (int)(pr / rows);
    reinterpret_cast<uint4*>(dst)[i] = __ldg(reinterpret_cast<const uint4*>(src) + ((size_t)p * n_clips + r / rows_per_clip) * w8 + c);
  }
}

}  // namespace

cudaError_t fanout_prefix_kv(const bf16* src, bf16* dst, int n_pos, int n_clips, int rows_per_clip, int width, cudaStream_t stream) {
  if (width % 8 != 0 || n_clips < 0 || rows_per_clip < 1) return cudaErrorInvalidValue;
  const size_t total = (size_t)n_pos * n_clips * rows_per_clip * (width / 8);
  if (n_pos <= 0 || total == 0) return cudaSuccess;
  const size_t want = (total + 255) / 256;
  fanout_prefix_kv_kernel<<<(int)(want < 148 * 16 ? want : 148 * 16), 256, 0, stream>>>(src, dst, n_pos, n_clips, rows_per_clip, width);
  note_launch();
  return cudaGetLastError();
}

cudaError_t assemble_window(const bf16* ring, int first, int cap, int n, int T, int W, const float* temporal, bf16* vf,
                            cudaStream_t stream) {
  const size_t total = (size_t)n * T * (W / 8);
  if (total == 0) return cudaSuccess;
  assemble_window_kernel<<<(int)((total + 255) / 256), 256, 0, stream>>>(ring, first, cap, n, T, W, temporal, vf);
  note_launch();
  return cudaGetLastError();
}

cudaError_t assemble_windows(const bf16* ring, const int* oldest, int oldest_const, int k, int n, int cap, int T, int W,
                             const float* temporal, bf16* vf, float* vf32, cudaStream_t stream) {
  const size_t total = (size_t)k * n * T * (W / 8);
  if (total == 0) return cudaSuccess;
  const size_t blocks = (total + 255) / 256;
  assemble_windows_kernel<<<(int)(blocks > 148 * 32 ? 148 * 32 : blocks), 256, 0, stream>>>(ring, oldest, oldest_const, k, n, cap, T, W,
                                                                                          temporal, vf, vf32);
  note_launch();
  return cudaGetLastError();
}

cudaError_t fill_positions(int* pos, int* n_text, int rows, int L, cudaStream_t stream) {
  if (rows <= 0) return cudaSuccess;
  fill_positions_kernel<<<(rows + 255) / 256, 256, 0, stream>>>(pos, n_text, rows, L);
  note_launch();
  return cudaGetLastError();
}

cudaError_t ln_fold_weight(const float* w, int N, int K, const float* gamma, const float* beta, const float* bias, bf16* wf,
                           float* colsum, float* bias_f, cudaStream_t stream) {
  if (N <= 0) return cudaSuccess;
  ln_fold_weight_kernel<<<(N * 32 + 255) / 256, 256, 0, stream>>>(w, N, K, gamma, beta, bias, wf, colsum, bias_f);
  note_launch();
  return cudaGetLastError();
}

cudaError_t layernorm_bf16(const LayerNormArgs& a, cudaStream_t stream) {
  if (a.rows <= 0) return cudaSuccess;
  int blocks = (a.rows * 32 + 255) / 256;
  const int max_blocks = 148 * 3;  // three 256-thread CTAs per SM (two rows in flight per warp), grid-stride over the rows
  if (blocks > max_blocks) blocks = max_blocks;
  const bool remap = a.out_row_base != nullptr;
  if (remap && a.out_group < 1) return cudaErrorInvalidValue;
  if (a.cols == 768 && !remap)
    layernorm_kernel<3, false><<<blocks, 256, 0, stream>>>(a);
  else if (a.cols == 1024 && !remap)
    layernorm_kernel<4, false><<<blocks, 256, 0, stream>>>(a);
  else if (a.cols == 768)
    layernorm_kernel<3, true><<<blocks, 256, 0, stream>>>(a);
  else if (a.cols == 1024)
    layernorm_kernel<4, true><<<blocks, 256, 0, stream>>>(a);
  else
    return cudaErrorInvalidValue;
  note_launch();
  return cudaGetLastError();
}

cudaError_t im2col_patches(const float* frames, int n_frames, int res, int patch, int kpad, bf16* out,
                           cudaStream_t stream) {
  const int G = res / patch;
  const size_t total = (size_t)n_frames * G * G * (kpad / 8);
  if (total == 0) return cudaSuccess;
  const int blocks = (int)((total + 255) / 256 > 148 * 16 ? 148 * 16 : (total + 255) / 256);
  im2col_kernel<<<blocks, 256, 0, stream>>>(frames, n_frames, res, patch, kpad, out);
  note_launch();
  return cudaGetLastError();
}

cudaError_t write_cls_rows(const float* cls, const bf16* pos, int n_frames, int T, int width, bf16* x,
                           cudaStream_t stream) {
  if (n_frames <= 0) return cudaSuccess;
  cls_rows_kernel<<<n_frames, 256, 0, stream>>>(cls, pos, n_frames, T, width, x);
  note_launch();
  return cudaGetLastError();
}

cudaError_t embed_text(const int* tokens, const int* positions, int pos_const, int n_rows, const float* words,
                       const float* pos_table, const float* gamma, const float* beta, float eps, int width, bf16* out,
                       cudaStream_t stream) {
  if (n_rows <= 0) return cudaSuccess;
  if (width != 768) return cudaErrorInvalidValue;
  embed_text_kernel<3><<<(n_rows * 32 + 127) / 128, 128, 0, stream>>>(tokens, positions, pos_const, n_rows, words,
                                                                      pos_table, gamma, beta, eps, width, out);
  note_launch();
  return cudaGetLastError();
}

cudaError_t store_text_kv(const bf16* qkv, int ld_qkv, int n_rows, int kv_width, int q_width, const int* pos,
                          int pos_const, int slot_div, int n_slots, bf16* txt_kv, cudaStream_t stream) {
  const int total = n_rows * (kv_width / 8);
  if (total <= 0) return cudaSuccess;
  store_text_kv_kernel<<<(total + 255) / 256, 256, 0, stream>>>(qkv, ld_qkv, n_rows, kv_width, q_width, pos, pos_const,
                                                                slot_div, n_slots, txt_kv);
  note_launch();
  return cudaGetLastError();
}

cudaError_t cast_f32_to_bf16(const float* src, int rows, int cols, int lds, bf16* dst, int ldd, int dst_rows,
                             int dst_cols, cudaStream_t stream) {
  const size_t total = (size_t)dst_rows * dst_cols;
  if (total == 0) return cudaSuccess;
  const int blocks = (int)((total + 255) / 256 > 148 * 32 ? 148 * 32 : (total + 255) / 256);
  cast_f32_bf16_kernel<<<blocks, 256, 0, stream>>>(src, rows, cols, lds, dst, ldd, dst_rows, dst_cols);
  note_launch();
  return cudaGetLastError();
}

cudaError_t cast_bf16_to_f32(const bf16* src, int rows, int cols, int lds, float* dst, int ldd, cudaStream_t stream) {
  const size_t total = (size_t)rows * cols;
  if (total == 0) return cudaSuccess;
  const int blocks = (int)((total + 255) / 256 > 148 * 32 ? 148 * 32 : (total + 255) / 256);
  cast_bf16_f32_kernel<<<blocks, 256, 0, stream>>>(src, rows, cols, lds, dst, ldd);
  note_launch();
  return cudaGetLastError();
}

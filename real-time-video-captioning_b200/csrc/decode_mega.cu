// Persistent single-clip decode kernel (latency mode; SURVEY K8-K15 for one clip): the WHOLE caption search of one clip --
// every decode step's embedding, 6 decoder layers, vocabulary head and search step -- runs inside ONE cooperative launch.
//
// Why: a single-clip decode step is ~42 dependent launches of 1-5 us of work each (131.8 MB of weights = ~20 us of HBM
// time per step against 284 us measured, CUDA-graph replay included): the step is bound by launch / drain latency between
// dependent kernels, not by bytes.  Here the dependent kernels become PHASES of one grid that stays resident (one CTA of 512
// threads per SM); a phase boundary is a grid-wide barrier on one global counter (~1-2 us) instead of a kernel boundary.
//
// Phases of a decode step (rows M <= 4 = the beams of the clip; H = 768):
//   per layer   A  x = LN_o(previous layer) or the embedding, redundantly per CTA; QKV: one output column per warp; q -> tq,
//                  this step's K | V straight into the text K/V plane
//               B  attention: the launch path's 128-thread CTA body run as "virtual CTAs" (head x row chunk x key split),
//                  up to four per CTA, partial (m, l, o) per split -> global
//               C  split combine (redundantly per participating CTA) + output projection + residual -> tb
//               D  c = LN_a(tb) redundantly per CTA; fc1 + GELU: one column per warp -> tf
//               E  fc2 (K = 3072 split over 8 warps per column group, fixed-order reduction) + residual c -> tb
//   head           x = LN_o(tb); vocabulary head: ~13 columns per warp, loads of the next column group in flight -> logits
//   search         CTA 0: the launch path's search step (search_step.cuh) on the first 256 threads
// 32 grid barriers per step.  Buffers exchanged between CTAs inside the launch are read with ld.global.cg.
//
// Arithmetic: every dot product, LayerNorm, softmax, combine and search statement is executed with the SAME operand order as
// the launch path's kernels (gemv_skinny.cu, elementwise.cu, text_attention_dev.cuh, search_step.cuh), so the tokens,
// log-probabilities and logits are BIT-IDENTICAL to it (tests/test_decode_mega.py) -- only the work distribution differs.
#include <math.h>

#include "common.cuh"
#include "kernels.h"
#include "search_step.cuh"
#include "text_attention_dev.cuh"

namespace {

constexpr int MEGA_THREADS = 512;
constexpr int MEGA_WARPS = MEGA_THREADS / 32;
constexpr int H = 768;            // decoder width (3 slices of 256 per warp pass)
constexpr int HV = H / 8;         // 16-byte vectors per row
constexpr int VCTAS = MEGA_THREADS / text_attn_dev::TA_THREADS;  // virtual attention CTAs per CTA

#ifndef GITB200_MEGA_SPIN_LIMIT
#define GITB200_MEGA_SPIN_LIMIT (2000000000LL)  // ~1 s: a barrier that never completes traps instead of hanging the GPU
#endif

// ---- grid-wide barrier: one monotonically increasing counter, every CTA adds 1 per barrier instance
__device__ __forceinline__ void grid_barrier(unsigned int* counter, unsigned int& target, unsigned int n_ctas) {
  __syncthreads();
  if (threadIdx.x == 0) {
    target += n_ctas;
    // release (cumulative over what the bar.sync above ordered before this thread) ... acquire: no separate fences needed
    asm volatile("red.release.gpu.global.add.u32 [%0], 1;" ::"l"(counter) : "memory");
    unsigned int v;
    const long long t0 = clock64();
    for (;;) {
      asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(counter) : "memory");
      if (v >= target) break;
      if (clock64() - t0 > GITB200_MEGA_SPIN_LIMIT) {
        printf("gitb200: decode_mega grid barrier timed out (block %d, counter %u, target %u)\n", (int)blockIdx.x, v, target);
        __trap();
      }
    }
  }
  __syncthreads();
}

__device__ __forceinline__ void named_barrier(int id, int n_threads) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(n_threads) : "memory"); }

__device__ __forceinline__ void unpack8(const uint4& u, float (&f)[8]) {
  const float2 a = unpack_bf16(u.x), b = unpack_bf16(u.y), c = unpack_bf16(u.z), d = unpack_bf16(u.w);
  f[0] = a.x; f[1] = a.y; f[2] = b.x; f[3] = b.y; f[4] = c.x; f[5] = c.y; f[6] = d.x; f[7] = d.y;
}

// ---- LayerNorm of one 768-wide bf16 row by one warp, result (rounded to bf16) into shared memory.
// Same arithmetic and lane -> column assignment as layernorm_kernel / gemv_skinny's normalise-on-load.
__device__ __forceinline__ void ln_row_to_smem(const bf16* __restrict__ src, const float* __restrict__ gamma, const float* __restrict__ beta,
                                               float eps, uint4* dst, int lane) {
  float v[24];
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    const uint4 u = __ldcg(reinterpret_cast<const uint4*>(src + (i * 32 + lane) * 8));
    const float2 a = unpack_bf16(u.x), b = unpack_bf16(u.y), c2 = unpack_bf16(u.z), d = unpack_bf16(u.w);
    v[i * 8 + 0] = a.x; v[i * 8 + 1] = a.y; v[i * 8 + 2] = b.x; v[i * 8 + 3] = b.y;
    v[i * 8 + 4] = c2.x; v[i * 8 + 5] = c2.y; v[i * 8 + 6] = d.x; v[i * 8 + 7] = d.y;
  }
  float sum = 0.f;
#pragma unroll
  for (int i = 0; i < 24; ++i) sum += v[i];
  const float mean = warp_sum(sum) / (float)H;
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < 24; ++i) {
    const float dlt = v[i] - mean;
    q += dlt * dlt;
  }
  const float rstd = rsqrtf(warp_sum(q) / (float)H + eps);
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    const int c = (i * 32 + lane) * 8;
    const float4 g0 = __ldg(reinterpret_cast<const float4*>(gamma + c)), g1 = __ldg(reinterpret_cast<const float4*>(gamma + c + 4));
    const float4 b0 = __ldg(reinterpret_cast<const float4*>(beta + c)), b1 = __ldg(reinterpret_cast<const float4*>(beta + c + 4));
    float o[8];
    o[0] = (v[i * 8 + 0] - mean) * rstd * g0.x + b0.x;
    o[1] = (v[i * 8 + 1] - mean) * rstd * g0.y + b0.y;
    o[2] = (v[i * 8 + 2] - mean) * rstd * g0.z + b0.z;
    o[3] = (v[i * 8 + 3] - mean) * rstd * g0.w + b0.w;
    o[4] = (v[i * 8 + 4] - mean) * rstd * g1.x + b1.x;
    o[5] = (v[i * 8 + 5] - mean) * rstd * g1.y + b1.y;
    o[6] = (v[i * 8 + 6] - mean) * rstd * g1.z + b1.z;
    o[7] = (v[i * 8 + 7] - mean) * rstd * g1.w + b1.w;
    uint4 u;
    u.x = pack_bf16(o[0], o[1]); u.y = pack_bf16(o[2], o[3]); u.z = pack_bf16(o[4], o[5]); u.w = pack_bf16(o[6], o[7]);
    dst[i * 32 + lane] = u;
  }
}

// ---- words[tok] + positions[pos] -> LayerNorm -> bf16 row in shared memory (embed_text_kernel<3>'s arithmetic)
__device__ __forceinline__ void embed_row_to_smem(const float* __restrict__ w, const float* __restrict__ p, const float* __restrict__ gamma,
                                                  const float* __restrict__ beta, float eps, bf16* dst, int lane) {
  float v[24];
#pragma unroll
  for (int i = 0; i < 6; ++i) {
    const int c = (i * 32 + lane) * 4;
    const float4 a = __ldg(reinterpret_cast<const float4*>(w + c));
    const float4 b = __ldg(reinterpret_cast<const float4*>(p + c));
    v[i * 4 + 0] = a.x + b.x; v[i * 4 + 1] = a.y + b.y; v[i * 4 + 2] = a.z + b.z; v[i * 4 + 3] = a.w + b.w;
  }
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < 24; ++i) s += v[i];
  const float mean = warp_sum(s) / (float)H;
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < 24; ++i) q += (v[i] - mean) * (v[i] - mean);
  const float rstd = rsqrtf(warp_sum(q) / (float)H + eps);
#pragma unroll
  for (int i = 0; i < 6; ++i) {
    const int c = (i * 32 + lane) * 4;
    const float4 g = __ldg(reinterpret_cast<const float4*>(gamma + c));
    const float4 b = __ldg(reinterpret_cast<const float4*>(beta + c));
    uint2 u;
    u.x = pack_bf16((v[i * 4 + 0] - mean) * rstd * g.x + b.x, (v[i * 4 + 1] - mean) * rstd * g.y + b.y);
    u.y = pack_bf16((v[i * 4 + 2] - mean) * rstd * g.z + b.z, (v[i * 4 + 3] - mean) * rstd * g.w + b.w);
    *reinterpret_cast<uint2*>(dst + c) = u;
  }
}

// ---- NC output columns of a K = 768 contraction by one warp: acc[m][c] = sum_k x[m][k] * W[n_c][k], lane owns
// k = lane * 8 + it * 256 (it = 0, 1, 2 in this order; 8 sequential FMAs per slice) -- gemv_skinny's non-split-K order.
// load768 issues all 3 * NC weight loads; they are static data, so a phase's first columns are fetched BEFORE the grid
// barrier that precedes the phase and the HBM latency hides behind the barrier and the phase's prologue.
// wrow[c] == nullptr: column absent (result ignored).
template <int NC>
__device__ __forceinline__ void load768(const bf16* const (&wrow)[NC], int lane, uint4 (&wv)[NC][3]) {
#pragma unroll
  for (int c = 0; c < NC; ++c)
#pragma unroll
    for (int it = 0; it < 3; ++it)
      wv[c][it] = wrow[c] != nullptr ? __ldg(reinterpret_cast<const uint4*>(wrow[c]) + it * 32 + lane) : make_uint4(0, 0, 0, 0);
}
template <int MT, int NC>
__device__ __forceinline__ void fma768(const uint4 (&wv)[NC][3], const uint4* xs /* [MT][HV] shared */, int lane, float (&acc)[MT][NC]) {
#pragma unroll
  for (int m = 0; m < MT; ++m)
#pragma unroll
    for (int c = 0; c < NC; ++c) acc[m][c] = 0.f;
#pragma unroll
  for (int it = 0; it < 3; ++it) {
    float xf[MT][8];
#pragma unroll
    for (int m = 0; m < MT; ++m) unpack8(xs[m * HV + it * 32 + lane], xf[m]);
#pragma unroll
    for (int c = 0; c < NC; ++c) {
      float wf[8];
      unpack8(wv[c][it], wf);
#pragma unroll
      for (int m = 0; m < MT; ++m)
#pragma unroll
        for (int i = 0; i < 8; ++i) acc[m][c] = fmaf(xf[m][i], wf[i], acc[m][c]);
    }
  }
#pragma unroll
  for (int m = 0; m < MT; ++m)
#pragma unroll
    for (int c = 0; c < NC; ++c) acc[m][c] = warp_sum(acc[m][c]);
}

// value (m, c) of a fully reduced acc[][] without dynamic register indexing
template <int MT, int NC>
__device__ __forceinline__ float pick(const float (&acc)[MT][NC], int m, int c) {
  float v = 0.f;
#pragma unroll
  for (int mm = 0; mm < MT; ++mm)
#pragma unroll
    for (int cc = 0; cc < NC; ++cc)
      if (mm == m && cc == c) v = acc[mm][cc];
  return v;
}

// ---- phase B: the launch path's decode-step attention CTA as "virtual CTAs" of 128 threads 
template <int NB>
__device__ __forceinline__ void attention_phase(const MegaArgs& a, const MegaLayer& L, float* attn_smem, int attn_floats, int t, int parity,
                                             int M, int chunks, int n_vcta) {
  const int tid = threadIdx.x, G = gridDim.x, b = blockIdx.x;
  TextAttnArgs ta;
  ta.q = a.tq; ta.ldq = 3 * H; ta.n_clips = 1; ta.rows_per_clip = M; ta.heads = a.heads;
  ta.vis_kv = L.vis_kv; ta.ld_vis = 3 * H; ta.k_off = H; ta.v_off = 2 * H; ta.Nv = a.Nv;
  ta.txt_kv = L.txt_kv; ta.txt_slots = M; ta.text_slot_is_clip = 0;
  ta.anc = a.st.reorder_cache ? (parity ? a.st.anc_tmp : a.st.anc) : nullptr;
  ta.anc_ld = a.st.max_len; ta.n_text = nullptr; ta.n_text_const = t + 1; ta.max_text = a.st.max_len;
  ta.out = a.ta; ta.ldo = H; ta.partial = a.partial; ta.splits = a.splits;
  const int vslot = tid >> 7, vtid = tid & 127;
  float* scratch = attn_smem + (size_t)vslot * attn_floats;
  for (int v = b + G * vslot; v < n_vcta; v += G * VCTAS) {
    const int h = v % a.heads, rest = v / a.heads;
    const int chunk = rest % chunks;
    text_attn_dev::text_attention_body<NB, true>(ta, a.scale_log2, a.kcap, scratch, 0, chunk, h, rest / chunks, vtid,
                                                 [vslot] { named_barrier(1 + vslot, text_attn_dev::TA_THREADS); });
    if (a.splits > 1) {
      // The LAST virtual CTA of this (row chunk, head) to finish combines the key splits' partials right here (the launch
      // path's combine kernel, same arithmetic) and writes the attention output rows -- instead of every CTA of the next phase
      // combining every (row, head) for itself, which at beam 4 cost more than the projection it fed.
      __shared__ int s_ticket[VCTAS];
      __threadfence();  // this thread's partials are visible GPU-wide before the ticket is drawn
      named_barrier(1 + vslot, text_attn_dev::TA_THREADS);
      if (vtid == 0) s_ticket[vslot] = atomicAdd(a.attn_cnt + chunk * a.heads + h, 1);
      named_barrier(1 + vslot, text_attn_dev::TA_THREADS);
      if (s_ticket[vslot] == a.splits - 1) {
        __threadfence();
        const int n_loc = min(NB, M - chunk * NB);
        for (int r = vtid >> 5; r < n_loc; r += text_attn_dev::TA_THREADS / 32) {
          const int row = chunk * NB + r;
          const uint32_t u = text_attn_dev::combine_partials<true>(a.partial + ((size_t)row * a.heads + h) * a.splits * (text_attn_dev::HD + 2),
                                                                   a.splits, vtid & 31);
          reinterpret_cast<uint32_t*>(a.ta + (size_t)row * H + h * text_attn_dev::HD)[vtid & 31] = u;
        }
        if (vtid == 0) a.attn_cnt[chunk * a.heads + h] = 0;  // ready for the next layer (grid barriers lie in between)
      }
    }
    named_barrier(1 + vslot, text_attn_dev::TA_THREADS);  // scratch reuse by the next virtual CTA of this slot
  }
}

// ---- search step, part 1: beam row `row` from the staged logits (all threads of the CTA)
__device__ __forceinline__ void search_row_phase(const MegaArgs& a, const float* stage, float thread_max, int row, search_dev::SearchSmem& sh,
                                                 float* wred) {
  const int tid = threadIdx.x, C = a.st.cand;
  search_dev::search_row_staged(a.st, stage, thread_max, row, 0, tid, MEGA_THREADS, [] { __syncthreads(); },
                                [] { named_barrier(6, search_dev::SS_THREADS); }, sh, wred);
  if (tid < C) {
    a.cand_score[row * C + tid] = sh.cand_score[tid];
    a.cand_idx[row * C + tid] = sh.cand_idx[tid];
  }
}

// ---- search step, part 2 (CTA 0): merge of the rows' candidate lists, candidate walk, re-ordering
__device__ __forceinline__ void search_walk_phase(const MegaArgs& a, int M, int t, int parity, search_dev::SearchSmem& sh) {
  const int tid = threadIdx.x, C = a.st.cand;
  __shared__ float all_s[4 * search_dev::MAX_CAND];
  __shared__ int all_i[4 * search_dev::MAX_CAND];
  if (tid < M * C) {
    all_s[tid] = __ldcg(a.cand_score + tid);
    all_i[tid] = __ldcg(a.cand_idx + tid);
  }
  named_barrier(6, search_dev::SS_THREADS);
  if (tid == 0) {
    int head[search_dev::MAX_NB];
    for (int r = 0; r < M; ++r) head[r] = 0;
    for (int c = 0; c < C; ++c) {  // M sorted lists of C candidates -> the best C of all, in `better` order
      int br = -1;
      float bs = 0.f;
      int bi = 0;
      for (int r = 0; r < M; ++r) {
        if (head[r] >= C) continue;
        const float s2 = all_s[r * C + head[r]];
        const int i2 = all_i[r * C + head[r]];
        if (br < 0 || search_dev::better(s2, i2, bs, bi)) {
          br = r;
          bs = s2;
          bi = i2;
        }
      }
      sh.cand_score[c] = bs;
      sh.cand_idx[c] = bi;
      ++head[br];
    }
  }
  named_barrier(6, search_dev::SS_THREADS);
  search_dev::search_walk_reorder(a.st, t + 1, parity, 0, tid, [] { named_barrier(6, search_dev::SS_THREADS); }, sh);
}

__device__ __forceinline__ void preload_qkv(const MegaArgs& a, int l, int gw, int lane, uint4 (&wA)[1][3], float& bA) {
  bA = __ldg(a.layer[l].b_qkv + min(gw, 3 * H - 1));
  // UNCONDITIONAL (out-of-range warps re-read the last column): a conditional definition would keep the registers alive
  // around the whole layer loop in the compiler's view
  const bf16* const wr[1] = {a.layer[l].w_qkv + (size_t)min(gw, 3 * H - 1) * H};
  load768<1>(wr, lane, wA);
}
// fc2 weights of one CTA column block: 3 columns of this warp's column group x its (at most) two 256-wide K slices
__device__ __forceinline__ void load_fc2(const bf16* __restrict__ w_fc2, int ffn, int c0, int vw, int lane, uint4 (&w)[3][2]) {
#pragma unroll
  for (int c = 0; c < 3; ++c)
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      const int k0 = (vw + 8 * r) * 256 + lane * 8;
      w[c][r] = (c0 + c < H && k0 < ffn) ? __ldg(reinterpret_cast<const uint4*>(w_fc2 + (size_t)(c0 + c) * ffn + k0)) : make_uint4(0, 0, 0, 0);
    }
}

struct Smem {
  uint4* xs;     // [4][HV] layer input (normalised), the attention sub-layer's residual
  uint4* cs;     // [4][HV] LN_a output: fc1 input, fc2 residual
  uint4* as;     // [4][HV] attention output (combined)
  uint4* tfs;    // [4][ffn / 8] fc1 output
  float* red2;   // [2][8][4][3] fc2 partials
  float* attn;   // VCTAS x attention scratch
};

template <int MT>
__device__ __forceinline__ void mega_body(const MegaArgs& a, const Smem& sm, int attn_floats) {
  const int tid = threadIdx.x, wid = tid >> 5, lane = tid & 31;
  const int G = gridDim.x, b = blockIdx.x;
  const int M = a.rows;
  const int gw = b * MEGA_WARPS + wid, n_gw = G * MEGA_WARPS;
  unsigned int bar_target = 0;
  const int ffn = a.ffn;
  constexpr int NB = MT >= 4 ? 4 : (MT >= 2 ? 2 : 1);
  const int chunks = (M + NB - 1) / NB;
  const int n_vcta = a.heads * chunks * a.splits;
  __shared__ search_dev::SearchSmem sh;
  __shared__ float wred[MEGA_WARPS];
  // optional phase trace (gitb200_debug_persistent_decode_trace): SM cycles CTA 0 spends working in / waiting after each phase
  const bool tracing = a.trace != nullptr && b == 0 && tid == 0;
  long long t_prev = tracing ? clock64() : 0;
  auto mark = [&](int slot) {
    if (tracing) {
      const long long now = clock64();
      a.trace[slot] += (unsigned long long)(now - t_prev);
      t_prev = now;
    }
  };
  auto barrier = [&](int slot) {
    __syncthreads();
    mark(slot);          // work of this phase (CTA 0's share)
    grid_barrier(a.barrier, bar_target, G);
    mark(slot + 16);     // waiting for the other CTAs + the barrier itself
  };

  // weights of a phase's first columns, fetched before the barrier in front of the phase
  uint4 wA[1][3], wC[1][3], wD[2][3], wE[3][2], wV[4][3];
  float bA = 0.f, bC = 0.f, bD = 0.f, bE = 0.f, bV = 0.f;  // ... and the bias values this thread's epilogues will add
  const int cols_per_cta = 6, n_cta_cols = (H + cols_per_cta - 1) / cols_per_cta;  // fc2: columns per CTA
  const int vw = wid & 7, cg = wid >> 3;                                             // fc2: K-slice warp, column group
  preload_qkv(a, 0, gw, lane, wA, bA);

  for (int t = a.first_step; t < a.steps; ++t) {
    const int parity = t & 1;
    // ------------------------------------------------------------------ embedding (every CTA, its own copy)
    if (wid < M) {
      const int tok = __ldcg(a.st.cur_tok + wid);
      embed_row_to_smem(a.words + (size_t)tok * H, a.pos_table + (size_t)t * H, a.lne_g, a.lne_b, a.embed_eps,
                        reinterpret_cast<bf16*>(sm.xs + wid * HV), lane);
    } else if (wid < MT) {
      for (int i = lane; i < HV; i += 32) sm.xs[wid * HV + i] = make_uint4(0, 0, 0, 0);
    }
    __syncthreads();

    for (int l = 0; l < a.n_layers; ++l) {
      const MegaLayer& L = a.layer[l];
      // ---------------------------------------------------------------- A: x = LN_o(previous layer's output); QKV
      if (l > 0) {
        const MegaLayer& Lp = a.layer[l - 1];
        if (wid < M) ln_row_to_smem(a.tb + (size_t)wid * H, Lp.lno_g, Lp.lno_b, a.ln_eps, sm.xs + wid * HV, lane);
        __syncthreads();
      }
      for (int n = gw; n < 3 * H; n += n_gw) {
        if (n != gw) {
          const bf16* const wr[1] = {L.w_qkv + (size_t)n * H};
          load768<1>(wr, lane, wA);
          bA = __ldg(L.b_qkv + n);
        }
        float acc[MT][1];
        fma768<MT, 1>(wA, sm.xs, lane, acc);
        if (lane < M) {
          const float v = pick<MT, 1>(acc, lane, 0) + bA;
          const bf16 o = __float2bfloat16(v);
          a.tq[(size_t)lane * 3 * H + n] = o;
          if (n >= H) L.txt_kv[((size_t)t * M + lane) * 2 * H + (n - H)] = o;
        }
      }
      barrier(0);

      // ---------------------------------------------------------------- B: attention (virtual 128-thread CTAs)
      attention_phase<NB>(a, L, sm.attn, attn_floats, t, parity, M, chunks, n_vcta);
      {
        const bf16* const wr[1] = {L.w_out + (size_t)min(gw, H - 1) * H};
        load768<1>(wr, lane, wC);
        bC = __ldg(L.b_out + min(gw, H - 1));
      }
      barrier(1);

      // ---------------------------------------------------------------- C: combine + output projection + residual x
      if (b * MEGA_WARPS < H) {
        for (int i = tid; i < M * HV; i += MEGA_THREADS) sm.as[i] = __ldcg(reinterpret_cast<const uint4*>(a.ta) + i);
        if (MT > M)
          for (int i = tid; i < (MT - M) * HV; i += MEGA_THREADS) sm.as[M * HV + i] = make_uint4(0, 0, 0, 0);
        __syncthreads();
        for (int n = gw; n < H; n += n_gw) {
          if (n != gw) {
            const bf16* const wr[1] = {L.w_out + (size_t)n * H};
            load768<1>(wr, lane, wC);
            bC = __ldg(L.b_out + n);
          }
          float acc[MT][1];
          fma768<MT, 1>(wC, sm.as, lane, acc);
          if (lane < M) {
            float v = pick<MT, 1>(acc, lane, 0) + bC;
            v += __bfloat162float(reinterpret_cast<const bf16*>(sm.xs + lane * HV)[n]);
            a.tb[(size_t)lane * H + n] = __float2bfloat16(v);
          }
        }
      }
      {
        const bf16* const wr[2] = {L.w_fc1 + (size_t)min(gw, ffn - 1) * H, L.w_fc1 + (size_t)min(gw + n_gw, ffn - 1) * H};
        load768<2>(wr, lane, wD);
        bD = __ldg(L.b_fc1 + min(gw + (lane & 1) * n_gw, ffn - 1));  // lane -> (row lane >> 1, column lane & 1)
      }
      barrier(2);

      // ---------------------------------------------------------------- D: c = LN_a(tb); fc1 + GELU
      if (wid < M) ln_row_to_smem(a.tb + (size_t)wid * H, L.lna_g, L.lna_b, a.ln_eps, sm.cs + wid * HV, lane);
      else if (wid < MT)
        for (int i = lane; i < HV; i += 32) sm.cs[wid * HV + i] = make_uint4(0, 0, 0, 0);
      __syncthreads();
      for (int n = gw; n < ffn; n += 2 * n_gw) {
        const int n2 = n + n_gw;
        if (n != gw) {
          const bf16* const wr[2] = {L.w_fc1 + (size_t)n * H, n2 < ffn ? L.w_fc1 + (size_t)n2 * H : nullptr};
          load768<2>(wr, lane, wD);
          bD = __ldg(L.b_fc1 + min(n + (lane & 1) * n_gw, ffn - 1));
        }
        float acc[MT][2];
        fma768<MT, 2>(wD, sm.cs, lane, acc);
        if (lane < 2 * M) {
          const int m = lane >> 1, c = lane & 1, nn = c ? n2 : n;
          if (nn < ffn) a.tf[(size_t)m * ffn + nn] = __float2bfloat16(gelu_erf(pick<MT, 2>(acc, m, c) + bD));
        }
      }
      load_fc2(L.w_fc2, ffn, min(b, n_cta_cols - 1) * cols_per_cta + cg * 3, vw, lane, wE);
      bE = __ldg(L.b_fc2 + min(min(b, n_cta_cols - 1) * cols_per_cta + tid % cols_per_cta, H - 1));  // column of the finalising thread
      barrier(3);

      // ---------------------------------------------------------------- E: fc2 (split K, fixed-order reduction) + residual c
      {
        // columns of this CTA: 3 per 8-warp half, the same warp -> K-slice assignment as gemv_skinny's split-K kernel
        // (virtual warp w takes the 256-wide slices w, w + 8, ...; partials added in the order w = 0 .. 7)
        for (int cb = b; cb < n_cta_cols; cb += G) {
          for (int i = tid; i < M * (ffn / 8); i += MEGA_THREADS) sm.tfs[i] = __ldcg(reinterpret_cast<const uint4*>(a.tf) + i);
          if (cb != b) {
            load_fc2(L.w_fc2, ffn, cb * cols_per_cta + cg * 3, vw, lane, wE);
            bE = __ldg(L.b_fc2 + min(cb * cols_per_cta + tid % cols_per_cta, H - 1));
          }
          __syncthreads();
          float acc[MT][3];
#pragma unroll
          for (int m = 0; m < MT; ++m)
#pragma unroll
            for (int c = 0; c < 3; ++c) acc[m][c] = 0.f;
#pragma unroll
          for (int r = 0; r < 2; ++r) {  // slices vw, vw + 8 (ffn <= 4096: at most two per virtual warp)
            const int k0 = (vw + 8 * r) * 256 + lane * 8;
            if (k0 < ffn) {
              float xf[MT][8];
#pragma unroll
              for (int m = 0; m < MT; ++m) {
                if (m < M) unpack8(sm.tfs[m * (ffn / 8) + (k0 >> 3)], xf[m]);
                else {
#pragma unroll
                  for (int i = 0; i < 8; ++i) xf[m][i] = 0.f;
                }
              }
#pragma unroll
              for (int c = 0; c < 3; ++c) {
                float wf[8];
                unpack8(wE[c][r], wf);
#pragma unroll
                for (int m = 0; m < MT; ++m)
#pragma unroll
                  for (int i = 0; i < 8; ++i) acc[m][c] = fmaf(xf[m][i], wf[i], acc[m][c]);
              }
            }
          }
#pragma unroll
          for (int m = 0; m < MT; ++m)
#pragma unroll
            for (int c = 0; c < 3; ++c) {
              const float v = warp_sum(acc[m][c]);
              if (lane == 0) sm.red2[((cg * 8 + vw) * 4 + m) * 3 + c] = v;
            }
          __syncthreads();
          if (tid < cols_per_cta * M) {
            const int j = tid % cols_per_cta, m = tid / cols_per_cta;
            const int n = cb * cols_per_cta + j;
            if (n < H) {
              float v = 0.f;
              for (int w2 = 0; w2 < 8; ++w2) v += sm.red2[(((j / 3) * 8 + w2) * 4 + m) * 3 + (j % 3)];
              v += bE;
              v += __bfloat162float(reinterpret_cast<const bf16*>(sm.cs + m * HV)[n]);
              a.tb[(size_t)m * H + n] = __float2bfloat16(v);
            }
          }
          __syncthreads();
        }
      }
      if (l + 1 < a.n_layers) {
        preload_qkv(a, l + 1, gw, lane, wA, bA);
        barrier(4);
      }
    }
    {  // (the last layer's closing barrier, with the vocabulary head's first weights in flight)
      const int n = min(gw * 4, a.vocab_pad - 4);
      const bf16* const wrc[4] = {a.w_vocab + (size_t)n * H, a.w_vocab + (size_t)(n + 1) * H, a.w_vocab + (size_t)(n + 2) * H,
                                  a.w_vocab + (size_t)(n + 3) * H};
      load768<4>(wrc, lane, wV);
      bV = __ldg(a.b_vocab + n + (lane & 3));  // lane -> (row lane >> 2, column lane & 3)
      barrier(4);
    }

    // ------------------------------------------------------------------ vocabulary head: x = LN_o(tb); logits
    {
      const MegaLayer& Ll = a.layer[a.n_layers - 1];
      if (wid < M) ln_row_to_smem(a.tb + (size_t)wid * H, Ll.lno_g, Ll.lno_b, a.ln_eps, sm.xs + wid * HV, lane);
      __syncthreads();
      float* logits = a.logits + (size_t)t * a.logits_step_stride;
      // groups of 4 consecutive columns dealt round-robin to all warps of the grid (7680 groups over 2368 warps: 3-4 each)
      const int n_end = a.vocab_pad;
      for (int n = gw * 4; n < n_end; n += n_gw * 4) {
        if (n != gw * 4) {
          const bf16* const wrc[4] = {a.w_vocab + (size_t)n * H, a.w_vocab + (size_t)(n + 1) * H, a.w_vocab + (size_t)(n + 2) * H,
                                      a.w_vocab + (size_t)(n + 3) * H};
          load768<4>(wrc, lane, wV);
          bV = __ldg(a.b_vocab + n + (lane & 3));
        }
        float acc[MT][4];
        fma768<MT, 4>(wV, sm.xs, lane, acc);
        if (lane < 4 * M) {
          const int m = lane >> 2, c = lane & 3;
          logits[(size_t)m * a.vocab_pad + n + c] = pick<MT, 4>(acc, m, c) + bV;
        }
      }
      barrier(5);

      // ---------------------------------------------------------------- search step, part 1: one CTA per beam row.
      // The launch path's per-clip search CTA walks the rows' 30522 logits three times from L2 with 256 threads (latency
      // bound: 67 us greedy / 270 us beam 4 per step when run as one CTA here).  Instead CTA r stages row r in shared memory
      // (one round of 16-byte loads by all 512 threads), computes its log-softmax statistics and its exact top-C there -- the
      // SAME arithmetic in the same order -- and publishes C candidates; the clip's top-C is the top-C of the rows' top-Cs.
      if (b < M) {
        float* stage = reinterpret_cast<float*>(sm.xs);  // the whole dynamic shared memory: nothing in it is live here
        const float4* xr = reinterpret_cast<const float4*>(logits + (size_t)b * a.vocab_pad);
        const int n4 = (a.st.V + 3) / 4;
        float tmax = -INFINITY;  // maximum of the logits this thread stages (row maximum + selection threshold, search_row_staged)
        for (int i0 = tid; i0 < n4; i0 += 8 * MEGA_THREADS) {  // 8 independent 16-byte loads per thread in flight
          float4 v8[8];
#pragma unroll
          for (int j = 0; j < 8; ++j)
            if (i0 + j * MEGA_THREADS < n4) v8[j] = __ldcg(xr + i0 + j * MEGA_THREADS);
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const int i4 = i0 + j * MEGA_THREADS;
            if (i4 < n4) {
              reinterpret_cast<float4*>(stage)[i4] = v8[j];
              const int i = 4 * i4;  // elements beyond V (the padded tail of the last vector) do not count
              if (i < a.st.V) tmax = fmaxf(tmax, v8[j].x);
              if (i + 1 < a.st.V) tmax = fmaxf(tmax, v8[j].y);
              if (i + 2 < a.st.V) tmax = fmaxf(tmax, v8[j].z);
              if (i + 3 < a.st.V) tmax = fmaxf(tmax, v8[j].w);
            }
          }
        }
        __syncthreads();
        search_row_phase(a, stage, tmax, b, sh, wred);
      }
      barrier(6);
      // ---------------------------------------------------------------- part 2 (CTA 0): merge, candidate walk, re-order
      if (b == 0 && tid < search_dev::SS_THREADS) search_walk_phase(a, M, t, parity, sh);
      preload_qkv(a, 0, gw, lane, wA, bA);  // the next step's first weights
      barrier(7);
    }
    // model.py:640 `if all(done): break`: the clip's search is finished, later steps would not change anything
    if (__ldcg(a.st.done) != 0) break;
  }
  if (tracing) a.trace[15] += 1;
}

template <int MT>  // rows padded to 1 / 2 / 4: one kernel each (own register allocation)
__global__ void __launch_bounds__(MEGA_THREADS, 1) decode_mega_kernel(const __grid_constant__ MegaArgs a, int attn_floats) {
  extern __shared__ uint4 smem_mega[];
  Smem sm;
  sm.xs = smem_mega;
  sm.cs = sm.xs + 4 * HV;
  sm.as = sm.cs + 4 * HV;
  sm.tfs = sm.as + 4 * HV;
  sm.red2 = reinterpret_cast<float*>(sm.tfs + 4 * (a.ffn / 8));
  sm.attn = sm.red2 + 2 * 8 * 4 * 3;
  mega_body<MT>(a, sm, attn_floats);
}

size_t mega_smem_bytes(const MegaArgs& a, int* attn_floats) {
  const int nb = a.rows > 2 ? 4 : (a.rows == 2 ? 2 : 1);  // = NB of mega_body<MT> (3 rows share one 4-row virtual CTA: per-row arithmetic does not depend on it)
  *attn_floats = text_attn_dev::ta_smem_floats(nb, a.kcap);
  const size_t layers = (size_t)(3 * 4 * HV + 4 * (a.ffn / 8)) * sizeof(uint4) + (size_t)(2 * 8 * 4 * 3 + VCTAS * *attn_floats) * sizeof(float);
  const size_t search = (size_t)((a.st.V + 3) / 4) * sizeof(float4);  // one staged logits row
  return layers > search ? layers : search;
}

}  // namespace

// Key-split factor and score-buffer width the launch path uses for ONE clip of `rows` beam rows (api.cu: run_text_pass,
// attention.cu: text_attention) -- the persistent kernel must split the keys identically to stay bit-identical.
void decode_mega_attention_geometry(int rows, int heads, int Nv, int max_text, int* splits, int* kcap) {
  const int chunks = (rows + 3) / 4;
  int s = (2 * 148 + chunks * heads - 1) / (chunks * heads);
  if (s > 16) s = 16;
  while (s > 1 && Nv / s < 64) --s;
  if (s < 1) s = 1;
  const int per = (Nv + s - 1) / s;
  *splits = s;
  *kcap = ((per + max_text + 3) / 4) * 4;
}

bool decode_mega_supported(const MegaArgs& a) {
  int af = 0;
  if (a.rows < 1 || a.rows > 4 || a.hidden != H || a.heads * text_attn_dev::HD != H || a.ffn % 256 != 0 || a.ffn < 2048 || a.ffn > 4096 ||
      a.n_layers < 1 || a.n_layers > MEGA_MAX_LAYERS || a.vocab_pad % 4 != 0 || a.st.n_clips != 1 || a.st.nb != a.rows ||
      a.first_step < 0 || a.first_step >= a.steps)
    return false;
  return mega_smem_bytes(a, &af) <= 200 * 1024;
}

// Enqueues: reset of the barrier counter, then the cooperative launch (one CTA per SM).  cudaErrorNotSupported when the device
// cannot keep the whole grid resident (the caller then uses the launch-per-kernel path).
cudaError_t decode_mega(const MegaArgs& a, cudaStream_t stream) {
  if (!decode_mega_supported(a)) return cudaErrorNotSupported;
  int attn_floats = 0;
  const size_t smem = mega_smem_bytes(a, &attn_floats);
  static int n_sm = 0, coop = 0;
  static bool attr_set = false;
  if (!attr_set) {
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, dev);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(decode_mega_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(decode_mega_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(decode_mega_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    if (e != cudaSuccess) return e;
    attr_set = true;
  }
  if (!coop || n_sm < 8) return cudaErrorNotSupported;
  void (*kernel)(const MegaArgs, int) = a.rows <= 1 ? decode_mega_kernel<1> : (a.rows <= 2 ? decode_mega_kernel<2> : decode_mega_kernel<4>);
  int per_sm = 0;
  cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, MEGA_THREADS, smem);
  if (e != cudaSuccess) return e;
  if (per_sm < 1) return cudaErrorNotSupported;
  e = cudaMemsetAsync(a.barrier, 0, 32 * sizeof(unsigned int), stream);  // [0]: barrier counter; [8, 32): attention tickets (attn_cnt)
  if (e != cudaSuccess) return e;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(n_sm);
  cfg.blockDim = dim3(MEGA_THREADS);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeCooperative;
  at[0].val.cooperative = 1;
  cfg.attrs = at;
  cfg.numAttrs = 1;
  e = cudaLaunchKernelEx(&cfg, kernel, a, attn_floats);
  if (e != cudaSuccess) return e;
  note_launch();
  return cudaGetLastError();
}

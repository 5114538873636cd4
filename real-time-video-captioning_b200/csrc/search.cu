// Device-resident caption search (SURVEY K13/K14): the reference's GeneratorWithBeamSearchV2.search
// (/root/reference/src/models/model.py:479-678, greedy-beam branch) and the upstream BeamHypotheses it
// uses, executed by one CTA per clip so that no logits, scores or indices ever cross PCIe per step.
//
//   step kernel:  log-softmax of every beam row (block reduce with warp shuffles), + running beam score,
//                 exact top-(per_node_beam_size * num_beams) over the clip's num_beams * V candidates,
//                 then thread 0 walks the candidates exactly like model.py:573-611 (EOS / last-step
//                 hypotheses, next beam content) and all threads re-order token rows and the text-KV
//                 ancestor table by the chosen parents.
#include <math.h>

#include "common.cuh"
#include "kernels.h"

#include "philox.cuh"
#include "search_step.cuh"

namespace {

using search_dev::MAX_CAND;
using search_dev::MAX_NB;
using search_dev::SS_THREADS;

__global__ void __launch_bounds__(SS_THREADS) search_step_kernel(SearchState st, const float* __restrict__ logits, int cur_len, int parity) {
  __shared__ search_dev::SearchSmem sh;
  search_dev::search_step_device<false>(st, logits, cur_len, parity, blockIdx.x, threadIdx.x, [] { __syncthreads(); }, sh);
}

// Beam search at batch size: one CTA per beam ROW for the log-softmax statistics and the row's own top candidates (the one-CTA-
// per-clip kernel walks a clip's rows one after the other: 244 us per step at 256 clips x 4 beams, 1.7 waves of 4-pass CTAs),
// then one CTA per clip merges its rows' sorted lists and does the candidate walk.  The top `cand` of a clip lie inside the union
// of its rows' top `cand`, and the order `better` is total: same candidates in the same order, bit for bit.
__global__ void __launch_bounds__(SS_THREADS) search_rows_kernel(SearchState st, const float* __restrict__ logits) {
  __shared__ search_dev::SearchSmem sh;
  const int b = blockIdx.x, clip = blockIdx.y, nb = st.nb, ldl = st.ldl, C = st.cand;
  auto load = [=](int bb, int i) { return logits[(size_t)(clip * nb + bb) * ldl + i]; };
  search_dev::search_topc_rows(st, load, b, b + 1, clip, threadIdx.x, [] { __syncthreads(); }, sh);
  if (threadIdx.x < C) {
    st.row_cand_score[(size_t)(clip * nb + b) * C + threadIdx.x] = sh.cand_score[threadIdx.x];
    st.row_cand_idx[(size_t)(clip * nb + b) * C + threadIdx.x] = sh.cand_idx[threadIdx.x];
  }
}

__global__ void __launch_bounds__(SS_THREADS) search_merge_walk_kernel(SearchState st, int cur_len, int parity) {
  __shared__ search_dev::SearchSmem sh;
  __shared__ float all_s[search_dev::MAX_NB * search_dev::MAX_CAND];
  __shared__ int all_i[search_dev::MAX_NB * search_dev::MAX_CAND];
  const int clip = blockIdx.x, tid = threadIdx.x, nb = st.nb, C = st.cand;
  if (tid < nb * C) {
    all_s[tid] = st.row_cand_score[(size_t)clip * nb * C + tid];
    all_i[tid] = st.row_cand_idx[(size_t)clip * nb * C + tid];
  }
  __syncthreads();
  if (tid == 0) {
    int head[search_dev::MAX_NB];
    for (int r = 0; r < nb; ++r) head[r] = 0;
    for (int c = 0; c < C; ++c) {  // nb sorted lists of C candidates -> the best C of all, in `better` order
      int br = -1, bi = 0;
      float bs = 0.f;
      for (int r = 0; r < nb; ++r) {
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
  __syncthreads();
  search_dev::search_walk_reorder(st, cur_len, parity, clip, tid, [] { __syncthreads(); }, sh);
}

// ---------------------------------------------------------------- extended step: repetition penalty, sampling (model.py:524-554)
// One CTA per beam row stages the row's logits in shared memory and patches them there (the logits buffer -- the saved,
// pre-penalty scores of model.py:521 -- is never written).  Without do_sample the penalised row goes through the exact
// top-C of the beam path (search_row_staged) and the clip's merge + walk; with do_sample the row is tempered, filtered and
// sampled, and a per-entry kernel walks the candidates in sample order.
struct SampleSmem {
  search_dev::SearchSmem sh;
  float wred[SS_THREADS / 32];
  int wred_i[SS_THREADS / 32];
  unsigned int hist[256];
  unsigned long long mass[256];  // fixed-point softmax mass per radix bin: integer sums, so the result is order-independent
  unsigned int bc_u[3];
  unsigned long long bc_m;
  int bc_i;
  float bc_f;
};

// order-preserving float -> uint32 (larger float, larger key)
__device__ __forceinline__ unsigned int fkey(float x) {
  const unsigned int u = __float_as_uint(x);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

// exp(x - m) in 2^-40 units (m = row maximum, so every weight is <= 2^40 and a row's sum stays below 2^56)
__device__ __forceinline__ unsigned long long fixed_weight(float x, float m) {
  return x == -INFINITY ? 0ull : __double2ull_rn((double)expf(x - m) * 1099511627776.0);
}

// Radix selection over the keys of xs[0, V), 8 bits per pass.
//   MASS = false: K = the k-th largest key, counting duplicates (torch.topk(...)[0][..., -1]).
//   MASS = true:  K = the smallest key whose strictly larger keys hold a mass (fixed_weight) <= P.
// Returns K, the count and mass of the keys > K, and the number of keys == K.
template <bool MASS>
__device__ void radix_select(const float* xs, int V, float m, unsigned int k, double P, int tid, SampleSmem& s, unsigned int* key,
                             unsigned int* above, unsigned long long* above_mass, unsigned int* ties) {
  unsigned int prefix = 0, mask = 0, n_above = 0, n_ties = 0;
  unsigned long long m_above = 0;
  for (int shift = 24; shift >= 0; shift -= 8) {
    for (int d = tid; d < 256; d += SS_THREADS) {
      s.hist[d] = 0;
      s.mass[d] = 0;
    }
    __syncthreads();
    for (int i = tid; i < V; i += SS_THREADS) {
      const float x = xs[i];
      const unsigned int kx = fkey(x);
      if ((kx & mask) == prefix) {
        const int d = (kx >> shift) & 255;
        atomicAdd(&s.hist[d], 1u);
        if (MASS) atomicAdd(&s.mass[d], fixed_weight(x, m));
      }
    }
    __syncthreads();
    if (tid == 0) {
      int pick = -1;
      if (MASS) {
        // the lowest non-empty bin whose largest key still qualifies (the mass above a bin grows as the bin goes down)
        unsigned long long acc = m_above;
        unsigned int acc_n = n_above;
        for (int d = 255; d >= 0; --d) {
          if (s.hist[d] == 0) continue;
          if ((double)acc > P) break;
          pick = d;
          m_above = acc;
          n_above = acc_n;
          acc += s.mass[d];
          acc_n += s.hist[d];
        }
      } else {
        for (int d = 255; d >= 0; --d) {
          if (n_above + s.hist[d] >= k) {
            pick = d;
            break;
          }
          n_above += s.hist[d];
        }
      }
      if (pick < 0) pick = 0;  // (unreachable: the bin of the largest key always qualifies)
      s.bc_u[0] = prefix | ((unsigned int)pick << shift);
      s.bc_u[1] = n_above;
      s.bc_u[2] = s.hist[pick];
      s.bc_m = m_above;
    }
    __syncthreads();
    prefix = s.bc_u[0];
    n_above = s.bc_u[1];
    n_ties = s.bc_u[2];
    m_above = s.bc_m;
    mask |= 255u << shift;
    __syncthreads();
  }
  *key = prefix;
  *above = n_above;
  *above_mass = m_above;
  *ties = n_ties;
}

__device__ __forceinline__ float block_max(float v, int tid, SampleSmem& s) {
  v = warp_max(v);
  if ((tid & 31) == 0) s.wred[tid >> 5] = v;
  __syncthreads();
  float r = s.wred[0];
  for (int w = 1; w < SS_THREADS / 32; ++w) r = fmaxf(r, s.wred[w]);
  __syncthreads();
  return r;
}

// block-wide best (score, index) in the order `better`
__device__ __forceinline__ void block_argmax(float& bs, int& bi, int tid, SampleSmem& s) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float s2 = __shfl_xor_sync(0xffffffffu, bs, o);
    const int i2 = __shfl_xor_sync(0xffffffffu, bi, o);
    if (search_dev::better(s2, i2, bs, bi)) {
      bs = s2;
      bi = i2;
    }
  }
  if ((tid & 31) == 0) {
    s.wred[tid >> 5] = bs;
    s.wred_i[tid >> 5] = bi;
  }
  __syncthreads();
  bs = s.wred[0];
  bi = s.wred_i[0];
  for (int w = 1; w < SS_THREADS / 32; ++w)
    if (search_dev::better(s.wred[w], s.wred_i[w], bs, bi)) {
      bs = s.wred[w];
      bi = s.wred_i[w];
    }
  __syncthreads();
}

__global__ void __launch_bounds__(SS_THREADS) sample_rows_kernel(SearchState st, SampleState p, const float* __restrict__ logits,
                                                                 int cur_len, int parity, int step) {
  extern __shared__ float xs[];  // [V]
  __shared__ SampleSmem s;
  const int b = blockIdx.x, e = blockIdx.y, tid = threadIdx.x, nb = st.nb, V = st.V;
  const int row = e * nb + b;
  const float* src = logits + (size_t)row * st.ldl;
  for (int i = tid; i < V; i += SS_THREADS) xs[i] = src[i];
  __syncthreads();

  // ---- repetition penalty (model.py:524-531): every DISTINCT token of the row's input_ids once, in fp32
  if (p.rp != 1.f) {
    const int* hist = (parity ? st.tokens_tmp : st.tokens) + (size_t)row * st.max_len;
    for (int t = tid; t < cur_len; t += SS_THREADS) {
      const int tok = hist[t];
      bool first = tok >= 0 && tok < V;
      for (int u = 0; u < t && first; ++u) first = hist[u] != tok;
      if (first) {
        const float x = xs[tok];
        xs[tok] = x < 0.f ? __fmul_rn(x, p.rp) : __fdiv_rn(x, p.rp);
      }
    }
    __syncthreads();
  }

  if (!p.do_sample) {  // ---- beam / greedy on the penalised row: the exact top-C of the beam path
    float tmax = -INFINITY;
    for (int i = tid; i < V; i += SS_THREADS) tmax = fmaxf(tmax, xs[i]);
    auto sync = [] { __syncthreads(); };
    search_dev::search_row_staged(st, xs, tmax, b, e, tid, SS_THREADS, sync, sync, s.sh, s.wred);
    if (tid < st.cand) {
      st.row_cand_score[(size_t)row * st.cand + tid] = s.sh.cand_score[tid];
      st.row_cand_idx[(size_t)row * st.cand + tid] = s.sh.cand_idx[tid];
    }
    return;
  }

  // ---- temperature (model.py:535): a true division, as torch's `scores / temperature`
  if (p.temperature != 1.f) {
    for (int i = tid; i < V; i += SS_THREADS) xs[i] = __fdiv_rn(xs[i], p.temperature);
    __syncthreads();
  }
  unsigned int key, above, ties;
  unsigned long long above_m;
  // ---- top-k (model.py:537, k = max(top_k, min_tokens_to_keep = 2)): keep every value >= the k-th largest, ties included
  if (p.top_k > 0) {
    const int kk = min(max(p.top_k, 2), V);
    radix_select<false>(xs, V, 0.f, (unsigned int)kk, 0.0, tid, s, &key, &above, &above_m, &ties);
    for (int i = tid; i < V; i += SS_THREADS)
      if (fkey(xs[i]) < key) xs[i] = -INFINITY;
    __syncthreads();
  }
  float m = -INFINITY;
  for (int i = tid; i < V; i += SS_THREADS) m = fmaxf(m, xs[i]);
  m = block_max(m, tid, s);  // the row maximum is never filtered
  // ---- top-p: sorted descending (ties: lower index first), a token is kept when the softmax mass BEFORE it is <= top_p;
  // the first min_tokens_to_keep + 1 = 3 sorted tokens always stay (upstream zeroes the first two removal flags and then
  // shifts the flags right by one)
  if (p.top_p < 1.f) {
    unsigned long long z = 0;
    for (int i = tid; i < V; i += SS_THREADS) z += fixed_weight(xs[i], m);
    if (tid == 0) s.bc_m = 0;
    __syncthreads();
    atomicAdd(&s.bc_m, z);
    __syncthreads();
    const double P = (double)p.top_p * (double)s.bc_m;
    __syncthreads();
    radix_select<true>(xs, V, m, 0u, P, tid, s, &key, &above, &above_m, &ties);
    // ties of the cut value K are kept in index order while the mass before them stays <= P
    const float xk = __uint_as_float((key & 0x80000000u) ? (key & 0x7fffffffu) : ~key);
    const unsigned long long w = fixed_weight(xk, m);
    unsigned int keep_t = ties;
    if (w > 0) {
      const double q = floor((P - (double)above_m) / (double)w) + 1.0;
      if (q < (double)ties) keep_t = (unsigned int)q;
    }
    unsigned int need = keep_t;
    if (above + keep_t < 3u) {  // the kept prefix is shorter than 3: the cut is the 3rd sorted token
      const unsigned int k3 = V < 3 ? (unsigned int)V : 3u;
      radix_select<false>(xs, V, 0.f, k3, 0.0, tid, s, &key, &above, &above_m, &ties);
      need = k3 - above;
    }
    int cut_idx = 0x7fffffff;
    if (need < ties) {  // only part of a run of equal values stays: find the need-th of them by index (rare: one thread)
      if (tid == 0) {
        unsigned int n = 0;
        int idx = 0x7fffffff;
        for (int i = 0; i < V; ++i)
          if (fkey(xs[i]) == key && ++n == need) {
            idx = i;
            break;
          }
        s.bc_i = idx;
      }
      __syncthreads();
      cut_idx = s.bc_i;
    }
    for (int i = tid; i < V; i += SS_THREADS) {
      const unsigned int kx = fkey(xs[i]);
      if (kx < key || (kx == key && i > cut_idx)) xs[i] = -INFINITY;
    }
    __syncthreads();
  }
  // ---- log_softmax over the kept tokens (model.py:543)
  float sum = 0.f;
  for (int i = tid; i < V; i += SS_THREADS) sum += expf(xs[i] - m);
  sum = warp_sum(sum);
  if ((tid & 31) == 0) s.wred[tid >> 5] = sum;
  __syncthreads();
  if (tid == 0) {
    float t = 0.f;
    for (int w = 0; w < SS_THREADS / 32; ++w) t += s.wred[w];
    s.bc_f = logf(t);
  }
  __syncthreads();
  const float l = s.bc_f;
  const float bs = __ldcg(st.beam_scores + row);
  // ---- per_node_beam_size draws without replacement (model.py:540): the exponential race -- the largest
  // (x - m) - log(-log u) in order, u = Philox4x32-10(counter (i / 4, step, j * nb + b, clip), key = seed) word i % 4;
  // with a key table, counter (i / 4, step, j * nb + b, 0) and key = keys[clip].
  // When the filters keep fewer tokens than per_node_beam_size (only a top-p cut can: check_sample rejects top-k below it),
  // the reference's torch.multinomial raises; here the missing draws are removed tokens in index order, with score -inf.
  const int clip = e / p.nrs;
  const unsigned long long seed = p.keys ? p.keys[clip] : *p.seed;
  const uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
  const uint32_t c2 = (uint32_t)((e % p.nrs) * nb + b), c3 = p.keys ? 0u : (uint32_t)clip;
  float prev_s = INFINITY;
  int prev_i = -1;
  for (int r = 0; r < p.pnb; ++r) {
    float best_s = -INFINITY;
    int best_i = 0x7fffffff;
    for (int g = tid; 4 * g < V; g += SS_THREADS) {
      const Philox4 ph = philox4x32_10((uint32_t)g, (uint32_t)step, c2, c3, k0, k1);
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int i = 4 * g + q;
        if (i < V) {
          const float x = xs[i];
          const float kx = x == -INFINITY ? -INFINITY : (x - m) + philox_gumbel(ph.x[q]);
          if (search_dev::better(prev_s, prev_i, kx, i) && search_dev::better(kx, i, best_s, best_i)) {
            best_s = kx;
            best_i = i;
          }
        }
      }
    }
    block_argmax(best_s, best_i, tid, s);
    if (tid == 0) {
      st.row_cand_score[(size_t)row * st.cand + r] = ((xs[best_i] - m) - l) + bs;
      st.row_cand_idx[(size_t)row * st.cand + r] = best_i;
    }
    prev_s = best_s;
    prev_i = best_i;
  }
}

// model.py:548-553: candidate j of an entry carries the word and score drawn from its beam row j / pnb, but the beam id
// j % nb (the reference adds arange(nb) * V repeated pnb times); the walk goes in this order, is_done on the maximum.
__global__ void __launch_bounds__(SS_THREADS) sample_walk_kernel(SearchState st, int pnb, int cur_len, int parity) {
  __shared__ search_dev::SearchSmem sh;
  const int e = blockIdx.x, tid = threadIdx.x, nb = st.nb, C = st.cand;
  if (tid < C) {
    const size_t src = (size_t)(e * nb + tid / pnb) * C + tid % pnb;
    sh.cand_score[tid] = st.row_cand_score[src];
    sh.cand_idx[tid] = (tid % nb) * st.V + st.row_cand_idx[src];
  }
  __syncthreads();
  search_dev::search_walk_reorder(st, cur_len, parity, e, tid, [] { __syncthreads(); }, sh, true);
}

__global__ void search_init_kernel(SearchState st, int sos) {
  const int row = blockIdx.x * blockDim.x + threadIdx.x;
  const int n_rows = st.n_clips * st.nb;
  if (row < n_rows) {
    st.tokens[(size_t)row * st.max_len] = sos;
    st.cur_tok[row] = sos;
    st.beam_scores[row] = (row % st.nb == 0) ? 0.f : -1e9f;  // model.py:508-510
    for (int t = 0; t < st.max_len; ++t) {
      st.anc[(size_t)row * st.max_len + t] = row;
      st.anc_tmp[(size_t)row * st.max_len + t] = row;
    }
  }
  if (row == 0) *st.done_count = 0;
  if (row < st.n_clips) {
    st.done[row] = 0;
    st.hyp_count[row] = 0;
    st.worst[row] = 1e9;
  }
}

// search_init_kernel with the prompt as every row's history (model.py:432-437, :481-495); see search_init_prefix
__global__ void search_init_prefix_kernel(SearchState st, const int* __restrict__ prompt, int P, int rows_per_clip) {
  const int row = blockIdx.x * blockDim.x + threadIdx.x;
  const int n_rows = st.n_clips * st.nb;
  if (row < n_rows) {
    const int* src = prompt + (size_t)(row / rows_per_clip) * P;
    if (P < st.max_len) {
      int* dst = (((P - 1) & 1) ? st.tokens_tmp : st.tokens) + (size_t)row * st.max_len;
      for (int t = 0; t < P; ++t) dst[t] = src[t];
    }
    st.cur_tok[row] = src[P - 1];
    st.beam_scores[row] = (row % st.nb == 0) ? 0.f : -1e9f;  // model.py:508-510
    for (int t = 0; t < st.max_len; ++t) {
      st.anc[(size_t)row * st.max_len + t] = row;
      st.anc_tmp[(size_t)row * st.max_len + t] = row;
    }
  }
  if (row == 0) *st.done_count = 0;
  if (row < st.n_clips) {
    st.done[row] = 0;
    st.hyp_count[row] = 0;
    st.worst[row] = 1e9;
  }
}

// model.py:653-677: best n_keep hypotheses per clip, eos padded, + one eos appended
__global__ void search_finalize_kernel(SearchState st, int* decoded, float* logprobs) {
  const int clip = blockIdx.x * blockDim.x + threadIdx.x;
  if (clip >= st.n_clips) return;
  const int nk = st.n_keep, max_len = st.max_len;
  const double* hs = st.hyp_score + (size_t)clip * (nk + 1);
  const int* hl = st.hyp_len + (size_t)clip * (nk + 1);
  const int* ht = st.hyp_tok + (size_t)clip * (nk + 1) * max_len;
  const int cnt = st.hyp_count[clip];
  bool used[MAX_CAND];
  for (int k = 0; k < cnt && k < MAX_CAND; ++k) used[k] = false;
  for (int k = 0; k < nk; ++k) {
    int* dst = decoded + ((size_t)clip * nk + k) * max_len;
    for (int t = 0; t < max_len; ++t) dst[t] = st.eos;
    logprobs[(size_t)clip * nk + k] = -1e5f;
    if (k >= cnt) continue;
    int best = -1;  // torch.topk over float32 scores: largest first, earliest index on ties
    for (int j = 0; j < cnt; ++j)
      if (!used[j] && (best < 0 || (float)hs[j] > (float)hs[best])) best = j;
    used[best] = true;
    for (int t = 0; t < hl[best]; ++t) dst[t] = ht[(size_t)best * max_len + t];
    logprobs[(size_t)clip * nk + k] = (float)hs[best];
  }
}

__global__ void anc_reorder_kernel(const int* __restrict__ in, int* __restrict__ out, const int* __restrict__ beam_idx,
                                   int rows, int ld, int pos) {
  const int r = blockIdx.x;
  if (r >= rows) return;
  const int p = beam_idx[r];
  for (int s = threadIdx.x; s < pos; s += blockDim.x) out[(size_t)r * ld + s] = in ? in[(size_t)p * ld + s] : p;
  if (threadIdx.x == 0) out[(size_t)r * ld + pos] = p;
}

}  // namespace

cudaError_t anc_reorder(const int* anc_in, int* anc_out, const int* beam_idx, int rows, int ld, int pos, cudaStream_t stream) {
  if (rows <= 0) return cudaSuccess;
  anc_reorder_kernel<<<rows, 64, 0, stream>>>(anc_in, anc_out, beam_idx, rows, ld, pos);
  note_launch();
  return cudaGetLastError();
}

cudaError_t search_init(const SearchState& s, int sos, cudaStream_t stream) {
  const int n = s.n_clips * s.nb;
  if (n <= 0) return cudaSuccess;
  if (s.nb > MAX_NB || s.cand > MAX_CAND || s.n_keep + 1 > MAX_CAND) return cudaErrorInvalidValue;
  search_init_kernel<<<(n + 127) / 128, 128, 0, stream>>>(s, sos);
  note_launch();
  return cudaGetLastError();
}

cudaError_t search_init_prefix(const SearchState& s, const int* prompt, int P, int rows_per_clip, cudaStream_t stream) {
  const int n = s.n_clips * s.nb;
  if (n <= 0) return cudaSuccess;
  if (s.nb > MAX_NB || s.cand > MAX_CAND || s.n_keep + 1 > MAX_CAND || prompt == nullptr || P < 1 || rows_per_clip < 1)
    return cudaErrorInvalidValue;
  search_init_prefix_kernel<<<(n + 127) / 128, 128, 0, stream>>>(s, prompt, P, rows_per_clip);
  note_launch();
  return cudaGetLastError();
}

cudaError_t search_step(const SearchState& s, const float* logits, int cur_len, int parity, cudaStream_t stream) {
  if (s.n_clips <= 0) return cudaSuccess;
  if (s.nb > MAX_NB || s.cand > MAX_CAND || cur_len + 1 > s.max_len) return cudaErrorInvalidValue;
  if (s.nb > 1 && s.row_cand_score != nullptr && s.row_cand_idx != nullptr && s.n_clips <= 65535) {
    search_rows_kernel<<<dim3(s.nb, s.n_clips), SS_THREADS, 0, stream>>>(s, logits);
    note_launch();
    search_merge_walk_kernel<<<s.n_clips, SS_THREADS, 0, stream>>>(s, cur_len, parity);
  } else {
    search_step_kernel<<<s.n_clips, SS_THREADS, 0, stream>>>(s, logits, cur_len, parity);
  }
  note_launch();
  return cudaGetLastError();
}

cudaError_t search_finalize(const SearchState& s, int* decoded, float* logprobs, cudaStream_t stream) {
  if (s.n_clips <= 0) return cudaSuccess;
  search_finalize_kernel<<<(s.n_clips + 63) / 64, 64, 0, stream>>>(s, decoded, logprobs);
  note_launch();
  return cudaGetLastError();
}

size_t sample_step_smem(int V) { return (size_t)V * sizeof(float); }

cudaError_t sample_step(const SearchState& s, const SampleState& p, const float* logits, int cur_len, int parity, int step,
                        cudaStream_t stream) {
  if (s.n_clips <= 0) return cudaSuccess;
  if (s.nb > MAX_NB || s.cand > MAX_CAND || cur_len + 1 > s.max_len || s.n_clips > 65535 || p.nrs < 1 || p.pnb < 1 ||
      s.row_cand_score == nullptr || s.row_cand_idx == nullptr || (p.do_sample && p.seed == nullptr && p.keys == nullptr))
    return cudaErrorInvalidValue;
  const size_t smem = sample_step_smem(s.V);
  cudaError_t e = cudaFuncSetAttribute(sample_rows_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  sample_rows_kernel<<<dim3(s.nb, s.n_clips), SS_THREADS, smem, stream>>>(s, p, logits, cur_len, parity, step);
  note_launch();
  if (p.do_sample)
    sample_walk_kernel<<<s.n_clips, SS_THREADS, 0, stream>>>(s, p.pnb, cur_len, parity);
  else
    search_merge_walk_kernel<<<s.n_clips, SS_THREADS, 0, stream>>>(s, cur_len, parity);
  note_launch();
  return cudaGetLastError();
}

// Device-side body of one caption-search step (shared by search.cu's kernel and the persistent decode kernel, decode_mega.cu).
#pragma once
#include <math.h>

#include "common.cuh"
#include "kernels.h"

namespace search_dev {

constexpr int SS_THREADS = 256;
constexpr int MAX_CAND = 16;  // per_node_beam_size * num_beams upper bound
constexpr int MAX_NB = 8;

__device__ __forceinline__ bool better(float s1, int i1, float s2, int i2) { return s1 > s2 || (s1 == s2 && i1 < i2); }

struct SearchSmem {
  float red_f[SS_THREADS / 32];
  int red_i[SS_THREADS / 32];
  float row_lse_max[MAX_NB], row_lse[MAX_NB];
  float cand_score[MAX_CAND];
  int cand_idx[MAX_CAND];
  int nxt_parent[MAX_NB], nxt_word[MAX_NB];
  float nxt_score[MAX_NB];
  float bc_f;
  int bc_i;
  static constexpr int LIST_CAP = 192;  // candidates at or above the selection threshold (expected: C plus a few)
  int list_n;
  float list_s[LIST_CAP];
  int list_i[LIST_CAP];
};

// Parts 1 + 2 of a search step for the beam rows [b_begin, b_end) of clip `clip`: log-softmax statistics of every row, then
// the exact top-C (C = st.cand) of (log_softmax + beam_score) over those rows' V candidates each, ordered by `better`, into
// sh.cand_score / sh.cand_idx (candidate id = b * V + word).  load(b, i) returns logit i of beam row b.
// Executed by SS_THREADS threads (tid = 0 .. SS_THREADS-1) that meet in sync().
// prof (optional, debugging): thread 0 adds the SM cycles of the five sections to prof[0..4].
template <class Load, class Sync>
__device__ __forceinline__ void search_topc_rows(const SearchState& st, Load load, int b_begin, int b_end, int clip, int tid, Sync sync,
                                                 SearchSmem& sh, unsigned long long* prof = nullptr) {
  const int warp = tid >> 5, lane = tid & 31;
  const int nb = st.nb, V = st.V, C = st.cand;
  long long t_prof = (prof != nullptr && tid == 0) ? clock64() : 0;
  auto section = [&](int k) {
    if (prof != nullptr && tid == 0) {
      const long long now = clock64();
      prof[k] += (unsigned long long)(now - t_prof);
      t_prof = now;
    }
  };
  // ---- 1. log-softmax statistics per beam row: max, then log(sum(exp(x - max)))   (model.py:557)
  for (int b = b_begin; b < b_end; ++b) {
    // (the loops below fetch 8 logits per thread before using them: the loads are independent, the uses keep their order)
    float m = -INFINITY;
    for (int i0 = tid; i0 < V; i0 += 8 * SS_THREADS) {
      float x8[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) x8[j] = i0 + j * SS_THREADS < V ? load(b, i0 + j * SS_THREADS) : -INFINITY;
#pragma unroll
      for (int j = 0; j < 8; ++j) m = fmaxf(m, x8[j]);
    }
    m = warp_max(m);
    if (lane == 0) sh.red_f[warp] = m;
    sync();
    if (tid == 0) {
      float mm = sh.red_f[0];
      for (int w = 1; w < SS_THREADS / 32; ++w) mm = fmaxf(mm, sh.red_f[w]);
      sh.bc_f = mm;
    }
    sync();
    m = sh.bc_f;
    float s = 0.f;
    for (int i0 = tid; i0 < V; i0 += 8 * SS_THREADS) {
      float x8[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) x8[j] = i0 + j * SS_THREADS < V ? load(b, i0 + j * SS_THREADS) : 0.f;
#pragma unroll
      for (int j = 0; j < 8; ++j)
        if (i0 + j * SS_THREADS < V) s += expf(x8[j] - m);
    }
    s = warp_sum(s);
    sync();
    if (lane == 0) sh.red_f[warp] = s;
    sync();
    if (tid == 0) {
      float ss = 0.f;
      for (int w = 0; w < SS_THREADS / 32; ++w) ss += sh.red_f[w];
      sh.row_lse_max[b] = m;
      sh.row_lse[b] = logf(ss);
    }
    sync();
  }

  section(0);
  // ---- 2. top-C of (log_softmax + beam_score) over the rows' V candidates each     (model.py:561-565)
  // Exact selection in three sweeps without per-thread sorted lists (a sorted insertion by ANY lane stalls its whole warp, and
  // with C = 8 some lane inserts at nearly every element):
  //   a. every thread's single best candidate, in registers;
  //   b. C rounds of block-wide argmax over those 256 bests -> T = the C-th of them: at least C candidates are >= T, so the
  //      top-C all lie at or above T;
  //   c. every candidate at or above T (a handful) is appended to a shared list; each list entry's rank among the list
  //      (number of entries that beat it in the total order `better`) places it: ranks 0 .. C-1 are the answer, in order.
  // The order `better` is total (ids are unique), so the result is THE top-C in THE order: the same as any other exact method.
  const auto score_of = [&](int b, int i, float m, float l, float bs) { return ((load(b, i) - m) - l) + bs; };
  float best_s = -INFINITY;
  int best_i = 0x7fffffff;
  for (int b = b_begin; b < b_end; ++b) {
    const float m = sh.row_lse_max[b], l = sh.row_lse[b], bs = __ldcg(st.beam_scores + clip * nb + b);
    for (int i0 = tid; i0 < V; i0 += 8 * SS_THREADS) {
      float x8[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) x8[j] = i0 + j * SS_THREADS < V ? load(b, i0 + j * SS_THREADS) : 0.f;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const int i = i0 + j * SS_THREADS;
        if (i < V) {
          const float sc = ((x8[j] - m) - l) + bs;
          if (better(sc, b * V + i, best_s, best_i)) {
            best_s = sc;
            best_i = b * V + i;
          }
        }
      }
    }
  }
  section(1);
  float thr_s = -INFINITY;
  int thr_i = 0x7fffffff;
  for (int c = 0; c < C; ++c) {
    float bs_ = best_s;
    int bi_ = best_i;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float s2 = __shfl_xor_sync(0xffffffffu, bs_, o);
      const int i2 = __shfl_xor_sync(0xffffffffu, bi_, o);
      if (better(s2, i2, bs_, bi_)) {
        bs_ = s2;
        bi_ = i2;
      }
    }
    if (lane == 0) {
      sh.red_f[warp] = bs_;
      sh.red_i[warp] = bi_;
    }
    sync();
    if (tid == 0) {
      float s = sh.red_f[0];
      int i = sh.red_i[0];
      for (int w = 1; w < SS_THREADS / 32; ++w)
        if (better(sh.red_f[w], sh.red_i[w], s, i)) {
          s = sh.red_f[w];
          i = sh.red_i[w];
        }
      sh.bc_f = s;
      sh.bc_i = i;
    }
    sync();
    thr_s = sh.bc_f;
    thr_i = sh.bc_i;
    if (best_i == thr_i) {  // this thread's best was taken (ids are unique): it leaves the contest
      best_s = -INFINITY;
      best_i = 0x7fffffff;
    }
    sync();
  }
  section(2);
  if (tid == 0) sh.list_n = 0;
  sync();
  for (int b = b_begin; b < b_end; ++b) {
    const float m = sh.row_lse_max[b], l = sh.row_lse[b], bs = __ldcg(st.beam_scores + clip * nb + b);
    for (int i0 = tid; i0 < V; i0 += 8 * SS_THREADS) {
      float x8[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) x8[j] = i0 + j * SS_THREADS < V ? load(b, i0 + j * SS_THREADS) : 0.f;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const int i = i0 + j * SS_THREADS;
        if (i < V) {
          const float sc = ((x8[j] - m) - l) + bs;
          if (!better(thr_s, thr_i, sc, b * V + i)) {  // at or above the threshold
            const int slot = atomicAdd(&sh.list_n, 1);
            if (slot < SearchSmem::LIST_CAP) {
              sh.list_s[slot] = sc;
              sh.list_i[slot] = b * V + i;
            }
          }
        }
      }
    }
  }
  sync();
  section(3);
  const int n_list = sh.list_n;
  if (n_list <= SearchSmem::LIST_CAP) {
    for (int e = tid; e < n_list; e += SS_THREADS) {
      const float se = sh.list_s[e];
      const int ie = sh.list_i[e];
      int rank = 0;
      for (int f = 0; f < n_list; ++f) rank += better(sh.list_s[f], sh.list_i[f], se, ie) ? 1 : 0;
      if (rank < C) {
        sh.cand_score[rank] = se;
        sh.cand_idx[rank] = ie;
      }
    }
  } else {
    // (never seen: more than LIST_CAP candidates above the C-th best thread maximum)  Exact fallback: C rounds of block-wide
    // argmax over ALL candidates below the previous pick.
    float prev_s = INFINITY;
    int prev_i = -1;
    for (int c = 0; c < C; ++c) {
      float bs_ = -INFINITY;
      int bi_ = 0x7fffffff;
      for (int b = b_begin; b < b_end; ++b) {
        const float m = sh.row_lse_max[b], l = sh.row_lse[b], bs = __ldcg(st.beam_scores + clip * nb + b);
        for (int i = tid; i < V; i += SS_THREADS) {
          const float sc = score_of(b, i, m, l, bs);
          const int id = b * V + i;
          if (better(prev_s, prev_i, sc, id) && better(sc, id, bs_, bi_)) {
            bs_ = sc;
            bi_ = id;
          }
        }
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const float s2 = __shfl_xor_sync(0xffffffffu, bs_, o);
        const int i2 = __shfl_xor_sync(0xffffffffu, bi_, o);
        if (better(s2, i2, bs_, bi_)) {
          bs_ = s2;
          bi_ = i2;
        }
      }
      if (lane == 0) {
        sh.red_f[warp] = bs_;
        sh.red_i[warp] = bi_;
      }
      sync();
      if (tid == 0) {
        float s = sh.red_f[0];
        int i = sh.red_i[0];
        for (int w = 1; w < SS_THREADS / 32; ++w)
          if (better(sh.red_f[w], sh.red_i[w], s, i)) {
            s = sh.red_f[w];
            i = sh.red_i[w];
          }
        sh.cand_score[c] = s;
        sh.cand_idx[c] = i;
      }
      sync();
      prev_s = sh.cand_score[c];
      prev_i = sh.cand_idx[c];
      sync();
    }
  }
  sync();
  section(4);
}

// Parts 1 + 2 for ONE beam row whose V logits sit in shared memory (persistent single-clip decode kernel: one CTA per row),
// executed by ALL n_threads threads of the CTA (n_threads >= SS_THREADS, tid = 0 .. n_threads-1, meeting in sync_all();
// sync_ss() is a barrier over the first SS_THREADS threads only).  thread_max = the maximum of the logits THIS thread staged.
// Same results as search_topc_rows over that row, bit for bit:
//   * the row maximum is exact whatever the order; the sum of exponentials runs on the first SS_THREADS threads in
//     search_topc_rows' order (thread t adds elements t, t + SS_THREADS, ... in this order, then the same tree);
//   * selection: x -> ((x - m) - l) + bs is monotone, so with T = the C-th largest of the threads' maxima at least C candidates
//     score >= score(T), and every member of the top-C does; those few candidates are ranked in the total order `better`.
template <class SyncAll, class SyncSS>
__device__ __forceinline__ void search_row_staged(const SearchState& st, const float* xs /* shared: [V] */, float thread_max, int b, int clip,
                                                  int tid, int n_threads, SyncAll sync_all, SyncSS sync_ss, SearchSmem& sh, float* wred /* shared: [n_threads / 32] */) {
  const int warp = tid >> 5, lane = tid & 31, n_warps = n_threads >> 5;
  const int nb = st.nb, V = st.V, C = st.cand;
  // ---- row maximum, and T = the C-th largest thread maximum (C rounds of block-wide max; the winner leaves the contest)
  float mine = thread_max, m = 0.f, thr_x = 0.f;
  for (int c = 0; c < C; ++c) {
    float v = warp_max(mine);
    if (lane == 0) wred[warp] = v;
    sync_all();
    float top = wred[0];
    for (int w = 1; w < n_warps; ++w) top = fmaxf(top, wred[w]);
    if (c == 0) m = top;
    thr_x = top;
    // exactly one thread among those holding `top` retires per round (ties: the lowest thread index)
    const unsigned holders = __ballot_sync(0xffffffffu, mine == top);
    sync_all();
    if (holders != 0 && lane == __ffs(holders) - 1) wred[warp] = (float)tid; else if (lane == 0 && holders == 0) wred[warp] = 3.0e38f;
    sync_all();
    float first = wred[0];
    for (int w = 1; w < n_warps; ++w) first = fminf(first, wred[w]);
    if ((float)tid == first) mine = -INFINITY;
    sync_all();
  }
  // ---- log(sum(exp(x - m))): search_topc_rows' summation order on the first SS_THREADS threads
  if (tid < SS_THREADS) {
    float s = 0.f;
    for (int i0 = tid; i0 < V; i0 += 8 * SS_THREADS) {
      float x8[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) x8[j] = i0 + j * SS_THREADS < V ? xs[i0 + j * SS_THREADS] : 0.f;
#pragma unroll
      for (int j = 0; j < 8; ++j)
        if (i0 + j * SS_THREADS < V) s += expf(x8[j] - m);
    }
    s = warp_sum(s);
    if (lane == 0) sh.red_f[warp] = s;
    sync_ss();
    if (tid == 0) {
      float ss = 0.f;
      for (int w = 0; w < SS_THREADS / 32; ++w) ss += sh.red_f[w];
      sh.row_lse_max[b] = m;
      sh.row_lse[b] = logf(ss);
      sh.list_n = 0;
    }
  }
  sync_all();
  // ---- candidates at or above score(T), then their ranks
  const float l = sh.row_lse[b], bs = __ldcg(st.beam_scores + clip * nb + b);
  const float thr_s = ((thr_x - m) - l) + bs;
  for (int i0 = tid; i0 < V; i0 += 8 * n_threads) {
    float x8[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) x8[j] = i0 + j * n_threads < V ? xs[i0 + j * n_threads] : -INFINITY;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float sc = ((x8[j] - m) - l) + bs;
      if (sc >= thr_s && i0 + j * n_threads < V) {
        const int slot = atomicAdd(&sh.list_n, 1);
        if (slot < SearchSmem::LIST_CAP) {
          sh.list_s[slot] = sc;
          sh.list_i[slot] = b * V + i0 + j * n_threads;
        }
      }
    }
  }
  sync_all();
  const int n_list = sh.list_n;
  if (n_list <= SearchSmem::LIST_CAP) {
    for (int e = tid; e < n_list; e += n_threads) {
      const float se = sh.list_s[e];
      const int ie = sh.list_i[e];
      int rank = 0;
      for (int f = 0; f < n_list; ++f) rank += better(sh.list_s[f], sh.list_i[f], se, ie) ? 1 : 0;
      if (rank < C) {
        sh.cand_score[rank] = se;
        sh.cand_idx[rank] = ie;
      }
    }
    sync_all();
  } else {
    // (never seen: a long run of equal logits)  the general routine, on the first SS_THREADS threads
    if (tid < SS_THREADS) search_topc_rows(st, [xs](int, int i) { return xs[i]; }, b, b + 1, clip, tid, sync_ss, sh);
    sync_all();
  }
}

// Parts 3 + 4 of a search step: the reference's candidate walk over sh.cand_score / sh.cand_idx (the clip's top-C, ordered),
// then the re-ordering of token rows / the ancestor table.  Same thread / sync contract as above.
// done_on_max: is_done sees the maximum candidate score (the sampling branch, whose candidates are in sample order); otherwise
// candidate 0, which is the maximum of a sorted top-C.
template <class Sync>
__device__ __forceinline__ void search_walk_reorder(const SearchState& st, int cur_len, int parity, int clip, int tid, Sync sync,
                                                    SearchSmem& sh, bool done_on_max = false) {
  const int nb = st.nb, V = st.V, C = st.cand;
  const int* tok_in = parity ? st.tokens_tmp : st.tokens;
  int* tok_out = parity ? st.tokens : st.tokens_tmp;
  const int* anc_in = parity ? st.anc_tmp : st.anc;
  int* anc_out = parity ? st.anc : st.anc_tmp;
  float* cand_score = sh.cand_score;
  int* cand_idx = sh.cand_idx;
  int* nxt_parent = sh.nxt_parent;
  int* nxt_word = sh.nxt_word;
  float* nxt_score = sh.nxt_score;

  // ---- 3. candidate walk (thread 0), exactly the reference's control flow           (model.py:573-611)
  if (tid == 0) {
    const int max_len = st.max_len;
    const int nk = st.n_keep;
    double* hs = st.hyp_score + (size_t)clip * (nk + 1);
    int* hl = st.hyp_len + (size_t)clip * (nk + 1);
    int* ht = st.hyp_tok + (size_t)clip * (nk + 1) * max_len;
    int cnt = st.hyp_count[clip];
    double worst = st.worst[clip];
    int is_done = st.done[clip];
    if (!is_done) {
      // BeamHypotheses.is_done(best_sum_logprobs) with early_stopping=False
      float best = cand_score[0];
      if (done_on_max)
        for (int c = 1; c < C; ++c) best = fmaxf(best, cand_score[c]);
      if (cnt >= nk) is_done = worst >= (double)best / pow((double)(max_len - 1), (double)st.length_penalty);
    }
    int n_next = 0;
    if (!is_done) {
      for (int c = 0; c < C; ++c) {
        const int beam_id = cand_idx[c] / V, word = cand_idx[c] % V;
        const int prow = clip * nb + beam_id;
        if (word == st.eos || cur_len + 1 == max_len) {
          // BeamHypotheses.add(input_ids[prow, :cur_len], score)
          const double score = (double)cand_score[c] / pow((double)cur_len, (double)st.length_penalty);
          if (cnt < nk || score > worst) {
            hs[cnt] = score;
            hl[cnt] = cur_len;
            for (int t = 0; t < cur_len; ++t) ht[(size_t)cnt * max_len + t] = tok_in[(size_t)prow * max_len + t];
            ++cnt;
            if (cnt > nk) {
              // drop the worst (first minimum in (score, index) order), keep insertion order of the rest
              int w0 = 0;
              for (int k = 1; k < cnt; ++k)
                if (hs[k] < hs[w0]) w0 = k;
              for (int k = w0; k + 1 < cnt; ++k) {
                hs[k] = hs[k + 1];
                hl[k] = hl[k + 1];
                for (int t = 0; t < max_len; ++t) ht[(size_t)k * max_len + t] = ht[(size_t)(k + 1) * max_len + t];
              }
              --cnt;
              double w1 = hs[0];
              for (int k = 1; k < cnt; ++k) w1 = fmin(w1, hs[k]);
              worst = w1;
            } else {
              worst = fmin(score, worst);
            }
          }
        } else {
          nxt_score[n_next] = cand_score[c];
          nxt_word[n_next] = word;
          nxt_parent[n_next] = prow;
          ++n_next;
        }
        if (n_next == nb) break;
      }
    }
    if (n_next != nb) {
      // done clip, or the final step: "pad the batch" (model.py:578, :609).  The reference pads with global
      // row 0 as parent; the padded rows are never read again, so the clip's own row is used instead.
      for (int b = 0; b < nb; ++b) {
        nxt_score[b] = 0.f;
        nxt_word[b] = st.eos;
        nxt_parent[b] = clip * nb + b;
      }
    }
    st.hyp_count[clip] = cnt;
    st.worst[clip] = worst;
    if (is_done && !st.done[clip]) atomicAdd(st.done_count, 1);  // the host polls this to leave the step loop early
    st.done[clip] = is_done;
  }
  sync();

  // ---- 4. re-order token rows (model.py:615-621) and, optionally, the text-KV ancestor table
  for (int b = 0; b < nb; ++b) {
    const int row = clip * nb + b, prow = nxt_parent[b];
    for (int t = tid; t < cur_len; t += SS_THREADS) tok_out[(size_t)row * st.max_len + t] = tok_in[(size_t)prow * st.max_len + t];
    if (st.reorder_cache) {
      // ancestors of text positions 0 .. cur_len-2 are inherited; position cur_len-1 was computed by the parent itself
      for (int t = tid; t < cur_len - 1; t += SS_THREADS) anc_out[(size_t)row * st.max_len + t] = anc_in[(size_t)prow * st.max_len + t];
      if (tid == 0) anc_out[(size_t)row * st.max_len + cur_len - 1] = prow;
    }
    if (tid == 0) {
      tok_out[(size_t)row * st.max_len + cur_len] = nxt_word[b];
      st.cur_tok[row] = nxt_word[b];
      st.beam_scores[row] = nxt_score[b];
    }
  }
}

// One search step of clip `clip` by one group of SS_THREADS threads (search_step_kernel: one CTA per clip).
// COHERENT: the logits were written by other CTAs of the same launch.
template <bool COHERENT, class Sync>
__device__ __forceinline__ void search_step_device(const SearchState& st, const float* __restrict__ logits, int cur_len, int parity,
                                                   int clip, int tid, Sync sync, SearchSmem& sh) {
  const int nb = st.nb, ldl = st.ldl;
  auto load = [=](int b, int i) { const float* q = logits + (size_t)(clip * nb + b) * ldl + i; return COHERENT ? __ldcg(q) : *q; };
  search_topc_rows(st, load, 0, nb, clip, tid, sync, sh);
  search_walk_reorder(st, cur_len, parity, clip, tid, sync, sh);
}

}  // namespace search_dev

"""Host-side references for the device sampling search: a numpy Philox4x32-10, the exponential-race draw the device uses in
place of ``torch.multinomial``, and a restatement of ``oracle.search_oracle.search``'s sampling branch with switches that
each break one rule on purpose (negative controls)."""
from __future__ import annotations

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import search_oracle as so

M0, M1, W0, W1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57), np.uint64(0x9E3779B9), np.uint64(0xBB67AE85)
MASK = np.uint64(0xFFFFFFFF)
FILTER = so.top_k_top_p_filtering  # the oracle's filter, bound before any test replaces it with RaceSampler.filtering


def philox4x32_10(c0, c1, c2, c3, k0, k1):
    """Vectorised Philox4x32-10 over uint32 counter arrays (broadcast) -> 4 uint32 arrays."""
    c = [np.asarray(x, dtype=np.uint64) & MASK for x in (c0, c1, c2, c3)]
    c = list(np.broadcast_arrays(*c))
    k0, k1 = np.uint64(k0) & MASK, np.uint64(k1) & MASK
    for r in range(10):
        if r:
            k0, k1 = (k0 + W0) & MASK, (k1 + W1) & MASK
        p0, p1 = M0 * c[0], M1 * c[2]
        hi0, lo0, hi1, lo1 = p0 >> np.uint64(32), p0 & MASK, p1 >> np.uint64(32), p1 & MASK
        c = [hi1 ^ c[1] ^ k0, lo1, hi0 ^ c[3] ^ k1, lo0]
    return [x.astype(np.uint32) for x in c]


def uniform(x):
    """Philox word(s) -> ((x >> 8) + 0.5) * 2^-24 in float64 (exact, strictly inside (0, 1)), as philox_uniform."""
    return ((np.asarray(x, dtype=np.uint32) >> 8).astype(np.float64) + 0.5) * 2.0 ** -24


def gumbel(u):
    """-log(-log u) in float64, rounded to float32, as philox_gumbel."""
    return (-np.log(-np.log(u))).astype(np.float32)


def uniforms(V, step, c2, clip, seed):
    """u[i] for vocabulary index i = word i % 4 of Philox(counter (i / 4, step, c2, clip), key = seed), in (0, 1)."""
    g = np.arange((V + 3) // 4, dtype=np.uint64)
    w = philox4x32_10(g, step, c2, clip, seed & 0xFFFFFFFF, seed >> 32)
    return uniform(np.stack(w, axis=1).reshape(-1)[:V])


class RaceSampler:
    """Stand-in for ``torch.multinomial(probs, n)`` inside the oracle's search: the top-n of log p - log(-log u) with the
    device's Philox uniforms.  Records, per search entry, how close its decisions were: the smallest relative gap between
    consecutive keys around the draws, and whether a token whose top-p keep decision was marginal (cumulative mass before it
    within tol of top_p, relative) would have been drawn had that decision gone the other way."""

    def __init__(self, nb, nrs, seed, top_p=1.0, tol=1e-4):
        self.nb, self.nrs, self.seed, self.top_p, self.tol = nb, nrs, seed, top_p, tol
        self.step = 0
        self.key_margin = {}
        self.p_margin = {}
        self.marginal = {}  # row -> [(token, log-probability it would have among the kept tokens)]

    def _note(self, d, e, v):
        d[e] = min(d.get(e, np.inf), v)

    def multinomial(self, probs, num_samples):
        R, V = probs.shape
        out = np.zeros((R, num_samples), dtype=np.int64)
        lp = np.log(probs.double().cpu().numpy()).astype(np.float32)
        for r in range(R):
            e, b = divmod(r, self.nb)
            clip, j = divmod(e, self.nrs)
            u = uniforms(V, self.step, j * self.nb + b, clip, self.seed)
            with np.errstate(invalid="ignore"):  # log p = -inf for filtered tokens: key -inf
                key = (lp[r] + gumbel(u)).astype(np.float32)
            order = np.lexsort((np.arange(V), -key.astype(np.float64)))
            out[r] = order[:num_samples]
            kth = float(key[order[num_samples - 1]])
            for tok, lp_tok in self.marginal.get(r, ()):
                k_tok = float(lp_tok + gumbel(u[tok]))
                if k_tok >= kth - self.tol * max(1.0, abs(kth)):
                    self._note(self.p_margin, e, 0.0)
            k = key[order[:num_samples + 1]].astype(np.float64)
            fin = np.isfinite(k)
            gaps = [(k[q] - k[q + 1]) / max(1.0, abs(k[q])) for q in range(num_samples) if fin[q] and fin[q + 1]]
            if gaps:
                self._note(self.key_margin, e, min(gaps))
        self.step += 1
        self.marginal = {}
        return torch.from_numpy(out).to(probs.device)

    def filtering(self, logits, top_k=0, top_p=1.0, filter_value=-float("Inf"), min_tokens_to_keep=1):
        self.marginal = {}
        if top_p < 1.0:
            x = FILTER(logits.clone(), top_k=top_k, top_p=1.0, min_tokens_to_keep=min_tokens_to_keep)
            srt, idx = torch.sort(x, descending=True)
            prob = F.softmax(srt.double(), dim=-1)
            cum = torch.cumsum(prob, dim=-1)
            for r in range(x.shape[0]):
                # the keep flag of sorted position q + 1 is cum[q] > top_p, for q >= min_tokens_to_keep
                q = np.flatnonzero((cum[r] - top_p).abs().numpy() <= self.tol * top_p)
                q = q[q >= min_tokens_to_keep]
                if len(q):
                    kept_mass = cum[r, max(int(np.searchsorted(cum[r].numpy(), top_p, side="right")), min_tokens_to_keep)].item()
                    self.marginal[r] = [(int(idx[r, j + 1]), float(np.log(prob[r, j + 1].item()) - np.log(kept_mass)))
                                        for j in q if j + 1 < x.shape[1]]
        return FILTER(logits, top_k=top_k, top_p=top_p, filter_value=filter_value, min_tokens_to_keep=min_tokens_to_keep)

    def unsure(self, tol=1e-4):
        """Search entries with a decision closer than tol (relative)."""
        return {e for d in (self.key_margin, self.p_margin) for e, v in d.items() if v <= tol}


def oracle_search(logits, n_clips, *, V, eos, sos, max_steps, nb, pnb, keep, lp, do_sample, top_k, top_p,
                  temperature, rp, nrs, seed):
    """oracle/search_oracle.search on the device's per-step logits [steps, n_clips*nrs*nb, >= V] with the race sampler.
    Returns (decoded [n_clips*nrs, keep, max_steps], logprobs, sampler)."""
    smp = RaceSampler(nb, nrs, seed, top_p if top_p is not None else 1.0)
    steps = iter(range(logits.shape[0]))

    def step(input_ids):
        return logits[next(steps), :, :V].clone()

    start = torch.full((n_clips, 1), sos, dtype=torch.long)
    with pytest.MonkeyPatch.context() as mp:  # only inside this call: torch.multinomial is not reproducible on the device
        mp.setattr(torch, "multinomial", smp.multinomial)
        mp.setattr(so, "top_k_top_p_filtering", smp.filtering)
        dec, lps, _ = so.search(start, step, eos_index=eos, max_steps=max_steps, beam_size=nb, length_penalty=lp,
                                per_node_beam_size=pnb, num_keep_best=keep, save_logits=False, do_sample=do_sample,
                                top_k=top_k, top_p=top_p, num_return_sequences=nrs, repetition_penalty=rp,
                                temperature=temperature)
    if keep == 1:
        dec = dec.unsqueeze(1)
    return dec, lps, smp


def broken_search(logits, n_clips, *, V, eos, sos, max_steps, nb, pnb, keep, lp, top_k, top_p, temperature, rp, nrs, seed,
                  break_rule=None):
    """The oracle's sampling branch (model.py:518-678, do_sample) restated with the race sampler, where ``break_rule``
    breaks one rule: "offsets_j_div_pnb", "no_shift", "penalty_per_occurrence", "penalty_after_filter", "done_on_first".
    With break_rule None it equals oracle_search."""
    B = n_clips * nrs
    ids = torch.full((B * nb, 1), sos, dtype=torch.long)
    hyps = [so.BeamHypotheses(keep, max_steps, lp, early_stopping=False) for _ in range(B)]
    beam_scores = torch.zeros(B, nb)
    beam_scores[:, 1:] = -1e9
    beam_scores = beam_scores.view(-1)
    done = [False] * B
    smp = RaceSampler(nb, nrs, seed)
    cur_len = 1

    def penalise(s):
        for i in range(B * nb):
            toks = ids[i].tolist() if break_rule == "penalty_per_occurrence" else set(ids[i].tolist())
            for t in toks:
                s[i, t] = s[i, t] * rp if s[i, t] < 0 else s[i, t] / rp

    def filt(s):
        if break_rule != "no_shift" or top_p >= 1.0:
            return so.top_k_top_p_filtering(s, top_k=top_k, top_p=top_p, min_tokens_to_keep=2)
        s = so.top_k_top_p_filtering(s, top_k=top_k, top_p=1.0, min_tokens_to_keep=2)
        srt, idx = torch.sort(s, descending=True)
        rem = torch.cumsum(F.softmax(srt, dim=-1), dim=-1) > top_p
        rem[..., :2] = False
        s[rem.scatter(1, idx, rem)] = -float("inf")
        return s

    t = 0
    while cur_len < max_steps:
        s = logits[t, :, :V].clone()
        t += 1
        if rp != 1.0 and break_rule != "penalty_after_filter":
            penalise(s)
        if temperature != 1.0:
            s = s / temperature
        s = filt(s)
        if rp != 1.0 and break_rule == "penalty_after_filter":
            penalise(s)
        words = smp.multinomial(F.softmax(s, dim=-1), pnb)
        sc = torch.gather(F.log_softmax(s, dim=-1), -1, words) + beam_scores[:, None]
        if break_rule == "offsets_j_div_pnb":
            offs = (torch.arange(nb * pnb) // pnb * V).repeat(B, 1)
        else:
            offs = (torch.arange(nb) * V).repeat(B, pnb)
        nw = words.view(B, pnb * nb) + offs
        ns = sc.view(B, pnb * nb)
        nxt = []
        for b in range(B):
            best = ns[b, 0].item() if break_rule == "done_on_first" else ns[b].max().item()
            done[b] = done[b] or hyps[b].is_done(best)
            if done[b]:
                nxt.extend([(0, eos, 0)] * nb)
                continue
            beam = []
            for idx, score in zip(nw[b].tolist(), ns[b].tolist()):
                bid, w = idx // V, idx % V
                if w == eos or cur_len + 1 == max_steps:
                    hyps[b].add(ids[b * nb + bid, :cur_len].clone(), score)
                else:
                    beam.append((score, w, b * nb + bid))
                if len(beam) == nb:
                    break
            nxt.extend(beam if beam else [(0, eos, 0)] * nb)
        beam_scores = torch.tensor([x[0] for x in nxt], dtype=torch.float)
        ids = torch.cat([ids[torch.tensor([x[2] for x in nxt])], torch.tensor([x[1] for x in nxt])[:, None]], dim=-1)
        cur_len += 1
        if all(done):
            break
    dec = torch.full((B, keep, max_steps), eos, dtype=torch.long)
    lps = torch.full((B, keep), -1e5)
    for i, h in enumerate(hyps):
        order = torch.topk(torch.tensor([x[0] for x in h.hyp]), min(keep, len(h.hyp)))[1].tolist()
        for j, hi in enumerate(order):
            conf, best = h.hyp[hi]
            lps[i, j] = conf
            dec[i, j, :len(best)] = best
    return dec, lps

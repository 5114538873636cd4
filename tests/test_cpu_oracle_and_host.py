"""CPU suite (-m "not gpu"): the oracle against its golden fixtures and hand-worked cases, the host-side logic of
the package, and the C-ABI library (loads, exports every symbol include/gitb200.h declares, fails loudly without
a GPU).  No compute call reaches the CUDA library here."""
import ctypes
import importlib
import math
import os
import re

import numpy as np
import pytest
import torch

from oracle import bleu_oracle, git_oracle as go, make_golden, search_oracle as so

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
g = importlib.import_module("real-time-video-captioning_b200")


# ------------------------------------------------------------------------------------------ golden fixtures
@pytest.mark.slow
def test_oracle_reproduces_golden_fixture():
    """tests/golden/git_base_f2.npz was produced by oracle/make_golden.py; the oracle must still reproduce it."""
    gold = np.load(os.path.join(ROOT, "tests", "golden", "git_base_f2.npz"))
    now = make_golden.compute()
    assert set(gold.files) == set(now)
    for k in gold.files:
        a, b = gold[k], np.asarray(now[k])
        if a.dtype.kind in "iu":
            assert np.array_equal(a, b), k
        else:
            assert np.allclose(a, b, rtol=2e-4, atol=2e-4), (k, np.abs(a - b).max())


# ------------------------------------------------------------------------------------------ search semantics
def _scripted(steps, vocab=12):
    """step() that returns scripted score rows: steps[t] is a [rows, vocab] tensor."""
    it = iter(steps)
    return lambda ids: next(it).clone()


def test_beam_hypotheses_matches_legacy_semantics():
    h = so.BeamHypotheses(2, 10, 0.6, early_stopping=False)
    assert not h.is_done(-1.0)
    h.add(torch.tensor([101, 5, 6]), -3.0)
    h.add(torch.tensor([101, 5]), -1.0)
    assert len(h) == 2 and math.isclose(h.worst_score, -3.0 / 3 ** 0.6)
    h.add(torch.tensor([101, 7, 8, 9]), -2.0)  # better than the worst: evicts it
    assert len(h) == 2 and math.isclose(h.worst_score, min(-1.0 / 2 ** 0.6, -2.0 / 4 ** 0.6))
    assert h.is_done(-100.0) and not h.is_done(-0.1)
    p = g.BeamHypotheses(2, 10, 0.6, early_stopping=False)  # product's host copy must behave identically
    for hyp, s in ((torch.tensor([101, 5, 6]), -3.0), (torch.tensor([101, 5]), -1.0), (torch.tensor([101, 7, 8, 9]), -2.0)):
        p.add(hyp, s)
    assert [round(s, 12) for s, _ in p.hyp] == [round(s, 12) for s, _ in h.hyp] and p.worst_score == h.worst_score


def test_greedy_is_not_plain_argmax_eos_at_rank1_continues_with_rank2():
    """SURVEY Appendix B.3: with beam_size=1 two candidates are considered; EOS at rank 1 stores a hypothesis and the
    rank-2 word continues the beam (model.py:585-600)."""
    V, eos, sos = 12, 2, 1
    s0 = torch.full((1, V), -5.0); s0[0, eos] = 3.0; s0[0, 7] = 2.0
    s1 = torch.full((1, V), -5.0); s1[0, 4] = 1.0
    s2 = torch.full((1, V), -5.0); s2[0, 9] = 1.0
    dec, lp, _ = so.search(torch.tensor([[sos]]), _scripted([s0, s1, s2]), eos_index=eos, max_steps=4, beam_size=1,
                           length_penalty=0.6, save_logits=False)
    # hypothesis [sos] (score log p(eos)/1^0.6) is stored at step 0; is_done() then compares it with the best
    # continuation: log p(eos) is the larger number so the clip is finished immediately at step 1.
    assert dec.tolist() == [[sos, eos, eos, eos]]
    assert math.isclose(lp.item(), torch.log_softmax(s0, -1)[0, eos].item(), rel_tol=1e-6)


def test_last_step_word_is_scored_but_dropped():
    """SURVEY Appendix B.2: at cur_len + 1 == max_length every candidate becomes a hypothesis WITHOUT the new word."""
    V, eos, sos = 12, 2, 1
    steps = [torch.full((1, V), -5.0) for _ in range(3)]
    steps[0][0, 5] = 4.0; steps[1][0, 6] = 4.0; steps[2][0, 7] = 4.0
    dec, lp, saved = so.search(torch.tensor([[sos]]), _scripted(steps), eos_index=eos, max_steps=4, beam_size=1,
                               length_penalty=0.6)
    assert dec.tolist() == [[sos, 5, 6, eos]] and len(saved) == 3 and saved[0][0].shape == (V,)
    total = sum(torch.log_softmax(s, -1)[0].max().item() for s in steps)
    assert math.isclose(lp.item(), total / 3 ** 0.6, rel_tol=1e-5)


def test_host_search_equals_oracle_search_on_random_scores():
    """The product's generic GeneratorWithBeamSearchV2.search (host control flow) == the line-by-line oracle."""
    V, eos, sos, n, nb, ms = 50, 2, 1, 3, 4, 9
    gen = torch.Generator().manual_seed(3)
    steps = [torch.randn(n * nb, V, generator=gen) * 2 for _ in range(ms - 1)]
    for s in steps:
        s[:, eos] += 2.5 * torch.rand(n * nb, generator=gen)
    ref = so.search(torch.full((n, 1), sos), _scripted(steps), eos_index=eos, max_steps=ms, beam_size=nb, length_penalty=0.6,
                    num_keep_best=2, save_logits=False)
    dec = g.GeneratorWithBeamSearchV2(eos, ms, nb, 0.6).search(torch.full((n, 1), sos), _scripted(steps), num_keep_best=2)
    assert torch.equal(dec[0], ref[0]) and torch.allclose(dec[1], ref[1], atol=1e-6)


@pytest.mark.parametrize("top_k,top_p,temperature,rep,nrs", [(5, 1.0, 1.0, 1.0, 1), (0, 0.8, 0.7, 1.0, 1), (8, 0.9, 1.3, 1.2, 2)])
def test_sampling_branch_equals_oracle(top_k, top_p, temperature, rep, nrs):
    """search(do_sample=True) (model.py:532-554: temperature, top_k_top_p_filtering, multinomial, the reference's beam-offset
    layout) and the repetition penalty (:524-531) / num_return_sequences (:481-484) paths: product == oracle under the same
    torch RNG seed on the same scripted scores."""
    V, eos, sos, n, nb, ms = 40, 2, 1, 2, 3, 8
    gen = torch.Generator().manual_seed(11)
    steps = [torch.randn(n * nrs * nb, V, generator=gen) * 2 for _ in range(ms - 1)]
    start = torch.full((n, 1), sos)
    torch.manual_seed(5)
    ref = so.search(start, _scripted([s.clone() for s in steps]), eos_index=eos, max_steps=ms, beam_size=nb, length_penalty=0.6,
                    save_logits=False, do_sample=True, top_k=top_k, top_p=top_p, num_return_sequences=nrs,
                    repetition_penalty=rep, temperature=temperature)
    torch.manual_seed(5)
    dec = g.GeneratorWithBeamSearchV2(eos, ms, nb, 0.6, repetition_penalty=rep, temperature=temperature).search(
        start, _scripted([s.clone() for s in steps]), do_sample=True, top_k=top_k, top_p=top_p, num_return_sequences=nrs)
    assert dec[0].shape == (n * nrs, ms)
    assert torch.equal(dec[0], ref[0]) and torch.allclose(dec[1], ref[1], atol=1e-6)


def test_top_k_top_p_filtering_hand_case_and_upstream_error_behaviour():
    m = importlib.import_module("real-time-video-captioning_b200.model")
    logits = torch.log(torch.tensor([[0.5, 0.25, 0.15, 0.07, 0.03]]))
    for f in (m.top_k_top_p_filtering, so.top_k_top_p_filtering):
        out = f(logits.clone(), top_k=3, top_p=1.0)
        assert torch.isinf(out[0, 3:]).all() and torch.isfinite(out[0, :3]).all()
        out = f(logits.clone(), top_k=0, top_p=0.7)          # 0.5 + 0.25 crosses 0.7 at the second token: it is kept
        assert torch.isfinite(out[0, :2]).all() and torch.isinf(out[0, 2:]).all()
        out = f(logits.clone(), top_k=1, top_p=0.1, min_tokens_to_keep=2)
        assert torch.isfinite(out[0, :2]).all() and torch.isinf(out[0, 2:]).all()
        with pytest.raises(TypeError):                       # upstream compares None > 0 (search's default arguments)
            f(logits.clone(), top_k=None, top_p=None)


def test_prefix_lm_mask_and_frame_truncation():
    m = go.prefix_lm_mask(3, 2)
    assert (m[:3, :3] == 0).all() and torch.isinf(m[:3, 3:]).all() and (m[3:, :3] == 0).all()
    assert m[3, 3] == 0 and torch.isinf(m[3, 4]) and m[4, 3] == 0 and m[4, 4] == 0
    cfg = go.GitConfig(num_image_with_embedding=1, resolution=32)
    sd = go.init_state_dict(cfg, seed=1)
    vf = go.encode_clip(sd, cfg, torch.randn(3, 3, 32, 32))  # 3 frames, 1 temporal embedding -> zip drops 2 frames
    assert vf.shape == (1, cfg.tokens_per_frame, 768)


def test_reorder_modes_differ_only_for_beams():
    """Appendix B.1: the reference never re-indexes the cache; greedy is unaffected, beam search may differ."""
    cfg = go.GitConfig(num_image_with_embedding=1, resolution=32, tie_output=False)
    sd = go.init_state_dict(cfg, seed=2)
    vf = go.encode_clip(sd, cfg, torch.randn(1, 3, 32, 32, generator=torch.Generator().manual_seed(0)))
    with torch.no_grad():
        a = so.infer(sd, cfg, vf, beam_size=1, max_steps=6, reorder_cache=False, save_logits=False)
        b = so.infer(sd, cfg, vf, beam_size=1, max_steps=6, reorder_cache=True, save_logits=False)
    assert torch.equal(a["predictions"], b["predictions"]) and torch.allclose(a["logprobs"], b["logprobs"])


# ------------------------------------------------------------------------------------------ metric
def test_bleu_is_character_level_and_matches_hand_computation():
    # identical strings -> 100
    assert math.isclose(bleu_oracle.calculate_bleu_score_corpus([["a cat"]], ["a cat"]), 100.0)
    # hand computation on characters: hyp "abcd", ref "abce": p1=3/4 p2=2/3 p3=1/2 p4 -> 0 matches -> float_min (method0)
    import sys
    want = 100 * math.exp(0.25 * (math.log(3 / 4) + math.log(2 / 3) + math.log(1 / 2) + math.log(sys.float_info.min)))
    assert math.isclose(bleu_oracle.calculate_bleu_score_corpus([["abce"]], ["abcd"]), want, rel_tol=1e-12)
    # word-level BLEU of these would be 0 (no 2-gram overlap); character-level is clearly positive
    v = bleu_oracle.calculate_bleu_score_corpus([["a man speaks."]], ["a man is speaking"])
    assert 30 < v < 80
    # brevity penalty: shorter hypothesis, closest reference length with ties to the shorter reference
    refs, hyp = [["aaaaaaaa", "aaaaaa"]], ["aaaaaaa"]  # lengths 8, 6 vs 7 -> tie -> 6 -> no penalty
    assert math.isclose(bleu_oracle.calculate_bleu_score_corpus(refs, hyp), 100.0)
    assert math.isclose(bleu_oracle.calculate_bleu_score_corpus([["aaaaaaaa"]], ["aaaaaa"]), 100.0 * math.exp(1 - 8 / 6))
    assert bleu_oracle.calculate_bleu_score_corpus([["xyz"]], ["abc"]) == 0  # no unigram match
    with pytest.raises(AssertionError):
        bleu_oracle.calculate_bleu_score_corpus([["a"]], ["a", "b"])


def test_product_metric_equals_oracle_on_the_reference_test_inputs():
    """Inputs of /root/reference/tests/test_metrics.py:17-18 (the reference's only test; it asserts nothing)."""
    cand = ["a man is speaking", "rain falls"]
    ref = [["a man speaks.", "someone speaks.", "a man is speaking while a bird is chirping in the background"],
           ["rain is falling hard on a surface"]]
    a = g.calculate_bleu_score_corpus(ref, cand)
    b = bleu_oracle.calculate_bleu_score_corpus(ref, cand)
    assert a == pytest.approx(b, rel=1e-12) and 0 < a < 100
    rng = np.random.default_rng(0)
    words = ["a", "man", "is", "the", "dog", "runs", "on", "grass", "t101", "t2045"]
    for _ in range(20):
        refs = [[" ".join(rng.choice(words, rng.integers(2, 8))) for _ in range(rng.integers(1, 4))] for _ in range(5)]
        cands = [" ".join(rng.choice(words, rng.integers(1, 8))) for _ in range(5)]
        assert g.calculate_bleu_score_corpus(refs, cands) == pytest.approx(bleu_oracle.calculate_bleu_score_corpus(refs, cands), rel=1e-12)


# ------------------------------------------------------------------------------------------ C ABI / package
def _header_symbols():
    text = open(os.path.join(ROOT, "include", "gitb200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(gitb200_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol_and_binding_covers_them():
    lib_mod = importlib.import_module("real-time-video-captioning_b200._lib")
    assert os.path.exists(lib_mod.LIB_PATH), "libgitb200.so missing: run python __graft_entry__.py"
    syms = _header_symbols()
    assert len(syms) >= 20
    lib = lib_mod.load()
    for s in syms:
        assert hasattr(lib, s), f"{s} declared in include/gitb200.h but not exported"
    assert sorted(lib_mod.SIGNATURES) == syms, set(lib_mod.SIGNATURES) ^ set(syms)
    assert b"sm_100a" in lib.gitb200_version()


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_no_gpu_means_loud_failure_not_fallback():
    lib_mod = importlib.import_module("real-time-video-captioning_b200._lib")
    lib = lib_mod.load()
    cfg = g.make_config({"num_image_with_embedding": 6}, 101, 102)
    h = ctypes.c_void_p()
    rc = lib.gitb200_create(ctypes.byref(cfg), 0, ctypes.byref(h))
    assert rc == -2 and b"no CPU fallback" in lib.gitb200_last_error(None)
    with pytest.raises(g.GitB200Error):
        g.Engine(cfg, 0)
    m = g.get_git_model(g.SyntheticTokenizer(), {"num_image_with_embedding": 2})
    with pytest.raises(RuntimeError):
        m.eval()({"image": [torch.zeros(1, 3, 224, 224)] * 2})
    with pytest.raises(RuntimeError):
        m.image_encoder.conv1(torch.zeros(1))  # parameter containers have no torch forward


def test_product_never_imports_the_oracle():
    """oracle/ is test infrastructure: nothing in the package, the public header, or the development tools outside tests/
    may import, link or execute it (only tests/, __graft_entry__.smoke() and bench.py's CPU legs do)."""
    for top in ("real-time-video-captioning_b200", "tools", "include"):
        for dp, _, fs in os.walk(os.path.join(ROOT, top)):
            for f in fs:
                if f.endswith((".py", ".cu", ".cuh", ".h")):
                    src = open(os.path.join(dp, f)).read()
                    assert not re.search(r"^\s*(from|import)\s+\.*oracle\b", src, flags=re.M), f
                    assert "import_module(\"oracle" not in src and "dlopen" not in src, f


def test_bench_touches_the_oracle_only_in_its_cpu_legs():
    """bench.py may execute oracle/ only as the CPU baseline (`cpu_baseline`, `--impl reference`): every oracle import sits
    inside run_reference_cpu(), and the GPU arm builds its weights through the package."""
    import ast
    src = open(os.path.join(ROOT, "bench.py")).read()
    tree = ast.parse(src)
    offenders = []
    for fn in [n for n in ast.walk(tree) if isinstance(n, (ast.FunctionDef, ast.Module))]:
        for node in (fn.body if isinstance(fn, ast.Module) else ast.walk(fn)):
            names = []
            if isinstance(node, ast.ImportFrom) and node.module:
                names = [node.module]
            elif isinstance(node, ast.Import):
                names = [a.name for a in node.names]
            if any(n == "oracle" or n.startswith("oracle.") for n in names):
                where = "module" if isinstance(fn, ast.Module) else fn.name
                if where != "run_reference_cpu":
                    offenders.append((where, node.lineno))
    assert not offenders, offenders
    assert "import_module(\"oracle" not in src


def test_bench_emits_exactly_one_json_line_on_stdout(tmp_path):
    """Whatever libraries print to file descriptor 1 after claim_stdout() (NCCL's version banner did) lands on stderr; the
    JSON line goes to the real stdout."""
    import subprocess
    import sys
    code = ("import os, sys; sys.path.insert(0, %r); import bench; bench.claim_stdout(); os.write(1, b'NCCL version banner\\n'); "
            "print('chatter'); bench.emit({'metric': 'm', 'value': 1})") % ROOT
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    assert r.stdout.strip().splitlines() == ['{"metric": "m", "value": 1}'], r.stdout
    assert "NCCL version banner" in r.stderr and "chatter" in r.stderr


def test_bench_dump_outputs_round_trips_tokens_and_scores(tmp_path):
    """--dump-outputs: the gathered tokens (int32) come back exactly as float64, the log-probabilities bit for bit as float32."""
    import bench
    tok = torch.tensor([[[101, 30521, 2 ** 31 - 1, 102]], [[101, 7, 102, 102]]], dtype=torch.int32)
    lp = torch.tensor([[-1.25], [-0.1]])
    bench.dump_outputs(str(tmp_path / "out"), tok, lp)
    t, l = np.load(tmp_path / "out" / "tokens.npy"), np.load(tmp_path / "out" / "logprobs.npy")
    assert t.dtype == np.float64 and l.dtype == np.float32 and t.shape == (2, 1, 4) and l.shape == (2, 1)
    assert np.array_equal(t.astype(np.int64), tok.numpy()) and np.array_equal(l, lp.numpy())


def test_module_tree_and_state_dict_names_match_upstream():
    m = g.get_git_model(g.SyntheticTokenizer(), {"num_image_with_embedding": 6})
    sd = m.state_dict()
    osd = go.init_state_dict(go.GitConfig(), seed=0)
    assert set(sd) == set(osd)
    for k in sd:
        assert tuple(sd[k].shape) == tuple(osd[k].shape), k
    # attributes the reference's callers touch (SURVEY 8b)
    assert len(m.image_encoder.transformer.resblocks) == 12 and len(m.textual.transformer.encoder.layer) == 6
    assert hasattr(m.textual.transformer.encoder.layer[3], "output") and m.sos_index == 101 and m.eos_index == 102
    assert m.decoder.beam_size == 4 and m.decoder.max_steps == 15 and m.decoder.length_penalty == 0.6
    assert m.textual.output.weight is m.textual.embedding.words.weight  # tied head
    m.load_state_dict(osd)
    big = g.get_git_model(g.SyntheticTokenizer(), {"image_encoder_type": "CLIPViT_L_14", "visual_feature_size": 1024,
                                                   "num_image_with_embedding": 6})
    assert big.image_encoder.positional_embedding.shape == (257, 1024) and len(big.image_encoder.transformer.resblocks) == 24
    with pytest.raises(ValueError):
        g.make_config({"image_encoder_type": "CLIPViT_L_14", "visual_feature_size": 768}, 101, 102)


def test_lazy_logits_and_tokenizer_and_shards():
    ll = g.LazyLogits(torch.arange(2 * 3 * 8, dtype=torch.float32).view(2, 3, 8), vocab=5)
    assert len(ll) == 2 and len(ll[0]) == 3 and ll[1][2].shape == (5,) and ll[1][2][0] == 40
    assert g.SyntheticTokenizer().decode([101, 2023, 7, 102, 102]) == "t2023 t7"
    assert [g.shard_range(10, r, 4) for r in range(4)] == [(0, 3), (3, 6), (6, 9), (9, 10)]
    assert [g.shard_range(2, r, 4) for r in range(4)] == [(0, 1), (1, 2), (2, 2), (2, 2)]
    tok, lp = g.caption_sharded(lambda b, e: (torch.arange(b, e).view(-1, 1, 1).int(), torch.arange(b, e).view(-1, 1).float()), 5)
    assert tok.flatten().tolist() == [0, 1, 2, 3, 4]


# ------------------------------------------------------------------------------------------ preprocessing oracle
@pytest.mark.parametrize("h,w", [(240, 320), (360, 640), (224, 224), (500, 300), (100, 180)])
def test_preprocess_oracle_matches_torchvision_transforms(h, w):
    """Pin oracle/preprocess_oracle.py against torchvision itself: the reference's Compose (dataloader.py:18-32) applied to
    a tensor with the pinned torchvision 0.16 semantics (bicubic, antialias off)."""
    tv = pytest.importorskip("torchvision")
    from torchvision.transforms import v2
    from oracle import preprocess_oracle as po
    frame = torch.randint(0, 256, (h, w, 3), dtype=torch.uint8, generator=torch.Generator().manual_seed(h * 1000 + w))
    x = frame.permute(2, 0, 1).float() / 255.0                                                     # ToTensor
    x = v2.functional.resize(x, [224], interpolation=v2.InterpolationMode.BICUBIC, antialias=False)  # Resize(224, BICUBIC)
    x = v2.functional.center_crop(x, [224, 224])                                                   # CenterCrop(224)
    x = x[[2, 1, 0], ...]                                                                          # BGR2RGBTransform
    x = v2.functional.normalize(x, po.CLIP_MEAN, po.CLIP_STD)                                      # Normalize
    got = po.preprocess_frames(frame[None])[0]
    assert got.shape == x.shape == (3, 224, 224)
    assert torch.allclose(got, x, atol=1e-5, rtol=1e-5), (got - x).abs().max()

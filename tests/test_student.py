"""Student decoder (SURVEY 8f rank 3; /root/reference/src/models/model.py:50-187).

CPU part: the oracle's hand-written glue (positional encoding, masks, scaling order, cached-vs-recomputed decoding, the
all-rows-SEP stop rule) against the stock torch.nn modules it wraps.  GPU part: csrc/student.cu through the C ABI against the
oracle.  Tolerances (bf16 weights / activations, fp32 accumulation, fp32 oracle): logits max |delta| < 0.15 sigma(logits),
mean < 0.03 sigma; greedy tokens must equal the oracle's wherever the oracle's own top-2 margin exceeds that logit tolerance;
inside it (a near-tie) the CUDA choice must score within the tolerance of the oracle's maximum."""
import importlib
import math

import pytest
import torch

from oracle import student_oracle as st

g = importlib.import_module("real-time-video-captioning_b200")


def _small_cfg():
    return st.StudentConfig(d_model=64, n_head=4, d_ffn=128, num_decoder_layers=2, vocab_length=50, cls_token_id=1, sep_token_id=2)


def test_positional_encoding_matches_closed_form():
    pe = st.positional_encoding(16, 10)
    for pos in (0, 3, 9):
        for i in (0, 2, 14):
            w = math.exp(-math.log(10000.0) * i / 16)
            assert math.isclose(pe[pos, i].item(), math.sin(pos * w), abs_tol=1e-6)
            assert math.isclose(pe[pos, i + 1].item(), math.cos(pos * w), abs_tol=1e-6)
    m = importlib.import_module("real-time-video-captioning_b200.student")
    assert torch.equal(m.PositionalEncoding(16, 10).pe[0], pe)


def test_oracle_forward_is_the_stock_modules_with_the_reference_glue():
    """forward_decoder == embedding + pe, THEN / sqrt(d) (model.py:144-148), stock nn.TransformerDecoder with the causal and
    padding masks, stock nn.Linear -- evaluated here step by step with explicit mask tensors."""
    cfg = _small_cfg()
    m = st.init_student(cfg, seed=1)
    y = torch.tensor([[1, 7, 0, 9], [1, 3, 4, 0]])
    mem = torch.randn(2, 3, 64, generator=torch.Generator().manual_seed(2))
    out = m.forward_decoder(y, mem)
    x = (m.embed.weight[y] + st.positional_encoding(64, 500)[:4]) / math.sqrt(64)
    causal = torch.full((4, 4), float("-inf")).triu(1)
    pad = torch.zeros(2, 4).masked_fill(y == 0, float("-inf"))
    with torch.no_grad():
        ref = m.linear(m.decoder(x, mem, tgt_mask=causal, tgt_key_padding_mask=pad))
    assert torch.allclose(out, ref, atol=1e-5)


def test_causal_masking_makes_cached_decoding_identical_to_the_reference_redecode():
    """Position p's logits do not depend on later tokens, so feeding one new position per step over cached keys / values
    (what the CUDA path does) reproduces the reference's full re-decode of the growing sequence (model.py:173-182)."""
    cfg = _small_cfg()
    m = st.init_student(cfg, seed=4)
    mem = torch.randn(3, 6, 64, generator=torch.Generator().manual_seed(5))
    full = m.greedy_decode_from_memory(mem, max_len=7)
    lo = m.forward_decoder(full[:, :-1], mem)
    assert torch.equal(lo.argmax(-1), full[:, 1:])          # every prefix's argmax is the next token
    lo_short = m.forward_decoder(full[:, :3], mem)
    assert torch.allclose(lo_short, lo[:, :3], atol=1e-5)   # ... and does not change when the sequence grows


def test_greedy_stops_only_when_every_row_emits_sep_in_the_same_step():
    cfg = _small_cfg()
    m = st.init_student(cfg, seed=6)
    with torch.no_grad():
        m.linear.bias[cfg.sep_token_id] += 100.0   # every row emits SEP immediately
    out = m.greedy_decode_from_memory(torch.randn(2, 6, 64), max_len=9)
    assert out.shape == (2, 2) and (out[:, 1] == cfg.sep_token_id).all()


def test_state_dict_names_follow_the_reference_student():
    cfg = _small_cfg()
    sd = st.state_dict_of(st.init_student(cfg))
    s = g.StudentCandidateV1(None, 64, 4, 128, 0.3, 2, 50, 1, 2)
    own = {k for k in s.state_dict() if k != "pos_enc.pe"}
    assert own == set(sd)
    assert all(s.state_dict()[k].shape == sd[k].shape for k in sd)
    with pytest.raises(RuntimeError, match="CUDA"):
        s.forward_decoder(torch.zeros(1, 2, dtype=torch.long), torch.zeros(1, 6, 64))
    with pytest.raises(RuntimeError, match="image encoder"):
        s.greedy_decode(torch.zeros(1, 6, 3, 8, 8), 3)


def test_beam_search_host_logic_equals_the_reference_loop():
    """StudentCandidateV1.beam_search (model.py:189-316): the product's batched tensor form against the statement-by-statement
    restatement, both driven by the same CPU forward_decoder (the oracle module's)."""
    cfg = _small_cfg()
    m = st.init_student(cfg, seed=10)
    mem = torch.randn(4, 6, 64, generator=torch.Generator().manual_seed(11))
    ref = st.beam_search_from_memory(m.forward_decoder, mem, cfg.cls_token_id, max_len=7, k=3)
    s = g.StudentCandidateV1(None, 64, 4, 128, 0.3, 2, 50, cfg.cls_token_id, cfg.sep_token_id)
    out = s.beam_search_from_memory(mem, max_len=7, k=3, forward_decoder=m.forward_decoder)
    assert out.shape == (4, 7) and torch.equal(out, ref)


# ------------------------------------------------------------------------------------------ GPU parity
def _gpu_student(cfg, seed):
    m = st.init_student(cfg, seed=seed)
    s = g.StudentCandidateV1(None, cfg.d_model, cfg.n_head, cfg.d_ffn, cfg.dropout, cfg.num_decoder_layers, cfg.vocab_length,
                             cfg.cls_token_id, cfg.sep_token_id)
    s.load_state_dict(st.state_dict_of(m))
    return m, s.to("cuda")


@pytest.mark.gpu
@pytest.mark.parametrize("B,L,F", [(1, 1, 6), (3, 9, 6), (16, 26, 6), (2, 5, 1)])
def test_student_forward_decoder_matches_oracle(B, L, F):
    cfg = st.StudentConfig()   # config.py:76-84: d_model 576, 8 heads (head dim 72), d_ffn 1024, 2 layers
    m, s = _gpu_student(cfg, seed=7)
    gen = torch.Generator().manual_seed(B * 100 + L)
    y = torch.randint(1, cfg.vocab_length, (B, L), generator=gen)
    y[:, 0] = cfg.cls_token_id
    if L > 3:
        y[0, L - 2:] = 0      # padded tail: masked as keys for every later query (masking.py:14)
    mem = torch.randn(B, F, cfg.d_model, generator=gen)
    ref = m.forward_decoder(y, mem)
    out = s.forward_decoder(y, mem).cpu()
    assert out.shape == ref.shape
    sigma = ref.std().item()
    err = (out - ref).abs()
    assert err.max().item() < 0.15 * sigma and err.mean().item() < 0.03 * sigma, (err.max().item() / sigma, err.mean().item() / sigma)


@pytest.mark.gpu
@pytest.mark.parametrize("B,max_len", [(1, 12), (5, 25), (64, 10)])
def test_student_greedy_decode_matches_oracle(B, max_len):
    cfg = st.StudentConfig()
    m, s = _gpu_student(cfg, seed=8)
    mem = torch.randn(B, 6, cfg.d_model, generator=torch.Generator().manual_seed(B))
    out = s.greedy_decode_from_memory(mem, max_len).cpu()
    assert out.shape[0] == B and out.shape[1] <= max_len + 1 and (out[:, 0] == cfg.cls_token_id).all()
    # teacher-force the CUDA tokens through the oracle: every token must be the oracle's argmax for its prefix, or tie with it
    lo = m.forward_decoder(out[:, :-1], mem)
    sigma = lo.std().item()
    top2 = lo.topk(2, dim=-1)
    chosen = torch.gather(lo, -1, out[:, 1:, None]).squeeze(-1)
    exact = out[:, 1:] == top2.indices[..., 0]
    near_tie = (top2.values[..., 0] - chosen) < 0.15 * sigma
    assert (exact | near_tie).all()
    clear = (top2.values[..., 0] - top2.values[..., 1]) >= 0.15 * sigma   # the oracle's own choice is outside the logit tolerance
    assert exact[clear].all() and clear.float().mean().item() > 0.5
    assert exact.float().mean().item() >= 0.95   # random-init logits over 30522 words: a few per cent of the steps are near-ties
    if exact.all():   # no near-tie taken: the whole run (including the stop rule) must equal the oracle's
        assert torch.equal(out, m.greedy_decode_from_memory(mem, max_len))


@pytest.mark.gpu
def test_student_greedy_stop_rule_and_reference_facade():
    cfg = st.StudentConfig()
    m, s = _gpu_student(cfg, seed=9)
    with torch.no_grad():
        m.linear.bias[cfg.sep_token_id] += 50.0
    s.load_state_dict(st.state_dict_of(m))
    s = s.to("cuda")
    mem = torch.randn(4, 6, cfg.d_model)
    out = s.greedy_decode_from_memory(mem, 8)
    assert out.shape == (4, 2) and (out[:, 1] == cfg.sep_token_id).all()

    class FakeEncoder(torch.nn.Module):  # stands in for the timm TinyViT: returns the list of stage feature maps
        def forward(self, x):
            return [x.mean(dim=1, keepdim=True), x[:, :1].repeat(1, 576, 1, 1)]

    s.image_encoder = FakeEncoder()
    src = torch.randn(2, 6, 3, 8, 8, device="cuda")
    tok = s.greedy_decode(src, 5)
    _, memory = s.forward_image_enc(src)
    assert memory.shape == (2, 6, 576) and torch.equal(tok.cpu(), m.greedy_decode_from_memory(memory.cpu(), 5))


@pytest.mark.gpu
def test_student_beam_search_on_the_gpu_decoder():
    """beam_search on the CUDA decoder: the returned sequence, scored by the ORACLE decoder, must be within the logit tolerance
    of the oracle's own beam-search winner (random-init margins are small, so the two may pick different near-tied beams)."""
    cfg = st.StudentConfig()
    m, s = _gpu_student(cfg, seed=12)
    mem = torch.randn(3, 6, cfg.d_model, generator=torch.Generator().manual_seed(13))
    out = s.beam_search_from_memory(mem.cuda(), max_len=6, k=3).cpu()
    ref = st.beam_search_from_memory(m.forward_decoder, mem, cfg.cls_token_id, max_len=6, k=3)
    assert out.shape == ref.shape == (3, 6) and (out[:, 0] == cfg.cls_token_id).all()

    def seq_score(seq):
        lp = torch.log_softmax(m.forward_decoder(seq[:, :-1], mem), dim=-1)
        return torch.gather(lp, -1, seq[:, 1:, None]).squeeze(-1).sum(-1)

    sigma = m.forward_decoder(ref[:, :-1], mem).std().item()
    assert (seq_score(ref) - seq_score(out) < 5 * 0.15 * sigma).all()


# ------------------------------------------------------------------------------------------ distillation training step
def _train_inputs(cfg, B, L, F, seed, pads=True):
    gen = torch.Generator().manual_seed(seed)
    y = torch.randint(1000, cfg.vocab_length, (B, L), generator=gen)
    y[:, 0] = cfg.cls_token_id
    if pads and L > 4:  # padded tails: masked keys (masking.py:14) and ignored CE targets (ignore_index=0, model.py:935)
        y[0, L - 3:] = 0
        y[B - 1, L - 1:] = 0
    mem = torch.randn(B, F, cfg.d_model, generator=gen)
    teacher = torch.randn(B, L, cfg.vocab_length, generator=gen) * 1.5
    return y, mem, teacher


def record(name, **vals):
    import json
    import os
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    os.makedirs(os.path.join(root, "gpurun_out"), exist_ok=True)
    with open(os.path.join(root, "gpurun_out", "parity_metrics.jsonl"), "a") as fh:
        fh.write(json.dumps({"test": name, **{k: (float(v) if isinstance(v, (int, float)) else v) for k, v in vals.items()}}) + "\n")


def _rel(a, b):
    return ((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-30)).item()


@pytest.mark.gpu
@pytest.mark.parametrize("B,L,F,temperature", [(8, 20, 6, 1.0), (3, 7, 2, 2.0)])
def test_distillation_step_gradients_match_autograd(B, L, F, temperature):
    """BASELINE.json configs[4] (8 clips x 20 caption tokens per GPU, student decoder of config.py:76-84): loss and every
    parameter gradient of gitb200_student_train_forward / _backward against torch.autograd on the stock nn modules the
    reference instantiates (oracle/student_oracle.py: KLDivLoss(batchmean) * T^2 + CrossEntropyLoss(ignore_index=0),
    model.py:922-935, :983).  bf16 activations / activation gradients, fp32 weight gradients: relative Frobenius error
    < 3e-2 over all parameters together, < 8e-2 for any single tensor (the step is bit-reproducible, so these seeded cases
    measure the same every run: worst tensor linear1.weight of layer 1, 6.6e-2 in the 21-row case, 4.9e-2 at 8 x 20)."""
    cfg = st.StudentConfig()
    m, s = _gpu_student(cfg, seed=21)
    y, mem, teacher = _train_inputs(cfg, B, L, F, seed=B * 10 + L)
    info, ref_grads, ref_dmem = st.distillation_step(m, y, mem, teacher, temperature)
    s.enable_training(lr=1e-4)
    out = s.distillation_step(y, mem, teacher, temperature=temperature, apply=False, want_memory_grad=True)
    loss, kl, ce = out["loss"].item(), out["kl"].item(), out["ce"].item()
    assert abs(loss - (kl + ce)) < 1e-5 * abs(loss)
    assert abs(kl - info["kl"]) < 2e-2 * abs(info["kl"]) and abs(ce - info["ce"]) < 2e-2 * abs(info["ce"]), (kl, info["kl"], ce, info["ce"])
    grads = {k: v.cpu() for k, v in s.gradients().items()}
    assert set(grads) == set(ref_grads)
    worst, num, den, per = ("", 0.0), 0.0, 0.0, {}
    for k, ref in ref_grads.items():
        e = per[k] = _rel(grads[k], ref)
        num += (grads[k].double() - ref.double()).pow(2).sum().item()
        den += ref.double().pow(2).sum().item()
        if e > worst[1]:
            worst = (k, e)
        assert e < 8e-2, (k, e)
    total = (num / den) ** 0.5
    e_mem = _rel(out["d_memory"].cpu(), ref_dmem)
    record("distillation_step_grads", B=B, L=L, temperature=temperature, loss=loss, ref_loss=info["loss"], all_params_rel_fro=total,
           worst_tensor=worst[0], worst_rel_fro=worst[1], d_memory_rel_fro=e_mem, per_tensor_rel_fro=per)
    assert total < 3e-2, total
    assert e_mem < 6e-2, e_mem
    # rows of the embedding table that do not occur in y get exactly zero gradient
    unused = torch.ones(cfg.vocab_length, dtype=torch.bool)
    unused[y.flatten()] = False
    assert (grads["embed.weight"][unused] == 0).all()


@pytest.mark.gpu
def test_distillation_adam_step_matches_torch_optim_and_loss_goes_down():
    """gitb200_student_train_apply == torch.optim.Adam(lr=1e-4) (model.py:1105) fed the SAME gradients, for three steps; the
    refreshed bf16 operand copies are live (the forward after the step uses them): the loss on a fixed batch decreases; the
    inference entry points keep working on the trained weights and state_dict() returns them."""
    cfg = st.StudentConfig()
    m, s = _gpu_student(cfg, seed=22)
    y, mem, teacher = _train_inputs(cfg, 8, 20, 6, seed=5)
    s.enable_training(lr=1e-4)
    names = [k for k, _ in s.named_parameters() if k.startswith(("decoder.layers.", "embed.", "linear."))]
    ref_params = {k: p.detach().clone().cuda().requires_grad_(True) for k, p in s.named_parameters() if k in names}
    opt = torch.optim.Adam(list(ref_params.values()), lr=1e-4)
    losses = []
    for step in range(3):
        out = s.distillation_step(y, mem, teacher, apply=False)
        losses.append(out["loss"].item())
        g = s.gradients()
        import ctypes
        rc = s._lib.gitb200_student_train_apply(s._h, ctypes.c_void_p(s._grads.data_ptr()), ctypes.c_float(1.0), s._stream())
        assert rc == 0
        s._params_dirty = True
        for k in names:
            ref_params[k].grad = g[k].clone()
        opt.step()
        for k in names:
            got = s._export(k, 0)
            assert torch.allclose(got, ref_params[k].detach(), atol=2e-7, rtol=1e-5), (step, k, (got - ref_params[k]).abs().max().item())
    for _ in range(12):
        out = s.distillation_step(y, mem, teacher)
        losses.append(out["loss"].item())
    assert losses[-1] < losses[0] - 0.05, losses
    sd = s.state_dict()
    assert not torch.equal(sd["linear.bias"].cpu(), st.state_dict_of(m)["linear.bias"])   # trained weights, not the initial ones
    logits = s.forward_decoder(y, mem)                                                    # inference path on the trained weights
    m2 = st.init_student(cfg, seed=22)
    m2.load_state_dict({k: v.cpu() for k, v in sd.items() if k in st.state_dict_of(m2)}, strict=False)
    ref = m2.forward_decoder(y, mem)
    sigma = ref.std().item()
    assert (logits.cpu() - ref).abs().max().item() < 0.15 * sigma


@pytest.mark.gpu
def test_distillation_trainer_step_with_the_git_teacher():
    """DistillationTrainer.training_step (model.py:880-983) end to end for the decoder: the frozen GIT teacher's teacher-forced
    logits (forward_output_logits, :896) feed the KL term; one step returns a finite loss equal to the oracle's on the same
    teacher logits."""
    tcfg_param = {"num_image_with_embedding": 2}
    teacher = g.GenerativeImageTextTeacher.from_random_init(tcfg_param)
    cfg = st.StudentConfig()
    m, s = _gpu_student(cfg, seed=23)
    trainer = g.DistillationTrainer(teacher, s, lr=1e-4)
    gen = torch.Generator().manual_seed(3)
    x = torch.randn(2, 2, 3, 224, 224, generator=gen)
    y = torch.randint(1000, 30000, (2, 6), generator=gen)
    y[:, 0] = 101
    mem = torch.randn(2, 2, cfg.d_model, generator=gen)
    t_logits = trainer.teacher_logits(x, y)
    assert t_logits.shape == (2, 6, 30522)
    info, _, _ = st.distillation_step(m, y, mem, t_logits.cpu().float())
    loss = trainer.training_step({"frames": x, "caption": y, "memory": mem})
    assert torch.isfinite(loss) and abs(loss.item() - info["loss"]) < 2e-2 * abs(info["loss"]), (loss.item(), info["loss"])
    assert trainer.last["d_memory"].shape == mem.shape


def _allreduce_worker(rank, world, port, q):
    import os
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    flat = torch.arange(10, dtype=torch.float32) * (rank + 1)
    h0 = g.all_reduce_bucket(flat, 0, 4)        # the "vocabulary head" bucket first ...
    h1 = g.all_reduce_bucket(flat, 4, 10)       # ... then the rest, both in flight
    scale = g.finish_all_reduce([h0, h1])
    q.put((rank, (flat * scale).tolist()))
    dist.destroy_process_group()


def test_gradient_buckets_all_reduce_to_the_ddp_average_on_two_gloo_ranks():
    """The distillation step's collective (SURVEY 2.3 C1): two in-place bucket all-reduces + the 1/world scaling = the DDP
    gradient average, on a world of 2 (gloo, CPU)."""
    import socket
    import torch.multiprocessing as mp
    sock = socket.socket()
    sock.bind(("127.0.0.1", 0))
    port = sock.getsockname()[1]
    sock.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    ps = [ctx.Process(target=_allreduce_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in ps:
        p.start()
    out = [q.get(timeout=120) for _ in ps]
    for p in ps:
        p.join(timeout=60)
        assert p.exitcode == 0
    want = [i * 1.5 for i in range(10)]   # (1 + 2) / 2 * i
    for rank, vals in out:
        assert vals == want, (rank, vals)
    assert g.finish_all_reduce([None, None]) == 1.0 and g.all_reduce_bucket(torch.zeros(4), 0, 4) is None   # no process group: no-ops

"""Pin the oracle's layer arithmetic against an independent implementation: transformers.GitForCausalLM (HF port of GIT).
tests/golden/hf_git.npz holds what HF computed on the oracle's seeded weights (upstream -> HF key map from SURVEY.md
section 8b, oracle/make_hf_golden.py): strided samples of the visual features and text-row logits, which must agree to fp32
round-off, and per-row norms, sums and argmax over the full arrays.
The reference itself cannot be imported here (SURVEY.md section 8c), so this is the strongest external
anchor available for the un-vendored generativeimage2text arithmetic."""
import numpy as np
import pytest
import torch

from oracle import git_oracle as go
from oracle import make_hf_golden as mh


@pytest.fixture(scope="module")
def hf():
    return np.load(mh.PATH, allow_pickle=False)


@pytest.mark.parametrize("encoder", mh.ENCODERS)
def test_oracle_matches_hf_git_forward(hf, encoder):
    """Both vision towers the reference can be configured with (model.py:682-685): ViT-B/16 (GIT-base, BASELINE configs
    1-3) and ViT-L/14 (the shipped teacher, data/teacher_configs/GIT_LARGE_MSRVTT/parameter.yaml; BASELINE configs 4-5)."""
    torch.manual_seed(0)
    F_, L = mh.FWD["n_frames"], len(mh.FWD["tokens"])
    large = encoder == "CLIPViT_L_14"
    cfg, sd, frames, tokens = mh.forward_inputs(encoder)
    with torch.no_grad():
        logits, vf, hidden = go.forward_one_custom(sd, cfg, frames, tokens)
    nv = vf.shape[1]
    assert nv == F_ * (257 if large else 197)
    assert list(vf.shape) == hf[f"{encoder}.visual_features_shape"].tolist()
    hf_vis = torch.from_numpy(hf[f"{encoder}.visual_features"])
    vs = vf[:, ::mh.VIS_ROW, ::mh.VIS_COL]
    assert torch.allclose(vs, hf_vis, atol=2e-4, rtol=1e-4), (vs - hf_vis).abs().max()
    assert list(logits.shape) == hf[f"{encoder}.logits_shape"].tolist() == [1, L, cfg.vocab_size]
    err = (logits[..., ::mh.LOGIT_COL] - torch.from_numpy(hf[f"{encoder}.logits"])).abs().max().item()
    assert err < 2e-3 * max(1.0, logits.abs().max().item()), err
    assert torch.equal(logits.argmax(-1), torch.from_numpy(hf[f"{encoder}.logits_argmax"]))
    # every value, unsampled, through per-row aggregates (fp32 round-off leaves them at ~2e-7 relative / ~1e-4 absolute)
    for name, a, sum_atol in (("visual_features", vf, 2e-3), ("logits", logits, 1e-2)):
        norms, sums = a.double().norm(dim=-1), a.double().sum(dim=-1)
        assert torch.allclose(norms, torch.from_numpy(hf[f"{encoder}.{name}_row_norms"]), rtol=1e-5, atol=0), name
        assert torch.allclose(sums, torch.from_numpy(hf[f"{encoder}.{name}_row_sums"]), rtol=0, atol=sum_atol), name
    assert hidden.shape == (7, nv + L, 768)


def test_history_cache_equals_full_forward():
    """The upstream hidden-state history path must be arithmetically identical to a full re-forward."""
    cfg = go.GitConfig(num_image_with_embedding=1, resolution=32, image_encoder_type="CLIPViT_B_16")
    sd = go.init_state_dict(cfg, seed=5)
    g = torch.Generator().manual_seed(2)
    vf = go.encode_clip(sd, cfg, torch.randn(1, 3, 32, 32, generator=g))
    toks = torch.tensor([[101, 7, 9, 11]])
    with torch.no_grad():
        full, _ = go.textual_forward(sd, cfg, vf, toks)
        st = go.DecodingState(sd, cfg, vf)
        outs = [st(toks[:, :t + 1]) for t in range(toks.shape[1])]
    for t, o in enumerate(outs):
        assert torch.allclose(o, full[:, t], atol=1e-4), (t, (o - full[:, t]).abs().max())


def test_oracle_greedy_search_matches_hf_generate_on_a_single_image(hf):
    """An independent END-TO-END check of encode + decoding + greedy search: HuggingFace's ``GitForCausalLM.generate`` (its own
    generation loop) against the oracle's ``infer`` (the reference's ``GeneratorWithBeamSearchV2.search`` restated line by line,
    beam_size 1, over the upstream hidden-state history cache) on the single-image branch (model.py:387-388; HF's generation
    cannot take videos: SURVEY Appendix C).  Untied random head, so the tokens are not the trivial copy.  HF ran its
    un-cached loop (``use_cache=False``, oracle/make_hf_golden.py): in transformers 5.5 HF's CACHED GIT generation disagrees
    with HF's own full forward from the second step on ([101, 18861, 24035, ...] cached vs [101, 18861, 29428, ...] for both its
    un-cached loop and its teacher-forced forward on this input); the un-cached loop re-runs the full forward the other test
    pins the oracle against, inside HF's loop.
    The reference's loop scores ``max_steps - 1`` steps, keeps the first ``max_steps - 2`` words and appends EOS (model.py:585-596,
    :653-677): those words must be HF's greedy continuation."""
    from oracle import search_oracle as so

    torch.manual_seed(0)
    cfg, sd, image = mh.greedy_inputs()
    max_steps = mh.GREEDY["max_steps"]
    with torch.no_grad():
        vf = go.vit_forward(sd, cfg, image)                                   # [1, 197, 768]: no temporal embedding
        ref = so.infer(sd, cfg, vf, beam_size=1, max_steps=max_steps, save_logits=False)["predictions"][0]
    out = torch.from_numpy(hf["greedy.tokens"])
    words = ref[1:max_steps - 1]
    assert ref[0].item() == 101 and ref[max_steps - 1].item() == 102
    assert 102 not in words.tolist()                                          # random head: nobody emits EOS in 7 steps
    assert out.shape == (max_steps - 1,)
    assert out[0].item() == 101 and torch.equal(out[1:], words), (out, ref)

"""Generate tests/golden/hf_git.npz: what transformers.GitForCausalLM (the HuggingFace port of GIT, an implementation
independent of the oracle) computes on the oracle's seeded weights (TEST INFRASTRUCTURE; see oracle/git_oracle.py header).

tests/test_oracle_vs_hf.py compares the oracle's layer arithmetic and greedy search against these numbers, so the
comparison runs without transformers installed.  Generated with transformers 5.5.0 and torch 2.11 on CPU; everything is
seeded, and re-running this script must reproduce the file within fp32 round-off.

    python -m oracle.make_hf_golden          # needs transformers; writes tests/golden/hf_git.npz (~0.3 MB)
"""
import os

import numpy as np
import torch

from . import git_oracle as go

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PATH = os.path.join(ROOT, "tests", "golden", "hf_git.npz")
ENCODERS = ("CLIPViT_B_16", "CLIPViT_L_14")
# forward: 2 frames, a 5-token caption.  The full arrays are several MB: stored are every VIS_ROW-th visual token at every
# VIS_COL-th channel and every LOGIT_COL-th vocabulary column, and, over ALL channels / the whole vocabulary, each row's
# float64 norm and sum (every visual token, every text row) and each text row's argmax
FWD = dict(weights_seed=3, frames_seed=1, n_frames=2, tokens=[101, 2023, 2003, 1037, 3231])
VIS_ROW, VIS_COL, LOGIT_COL = 5, 4, 8
# greedy: one image without temporal embedding, untied head, the reference search scores max_steps - 1 = 8 steps
GREEDY = dict(weights_seed=9, image_seed=4, max_steps=9)


def forward_config(encoder):
    """HF uses one LayerNorm eps (1e-12) for embeddings too: the oracle is aligned to it for this comparison only."""
    large = encoder == "CLIPViT_L_14"
    return go.GitConfig(num_image_with_embedding=FWD["n_frames"], embedding_ln_eps=1e-12, image_encoder_type=encoder,
                        visual_feature_size=1024 if large else 768)


def forward_inputs(encoder):
    cfg = forward_config(encoder)
    sd = go.init_state_dict(cfg, seed=FWD["weights_seed"], temporal_std=0.02, perturb=True)
    frames = torch.randn(FWD["n_frames"], 3, 224, 224, generator=torch.Generator().manual_seed(FWD["frames_seed"]))
    return cfg, sd, frames, torch.tensor([FWD["tokens"]])


def greedy_inputs():
    cfg = go.GitConfig(num_image_with_embedding=0, embedding_ln_eps=1e-12, tie_output=False)
    sd = go.init_state_dict(cfg, seed=GREEDY["weights_seed"], temporal_std=0.0, perturb=True)
    image = torch.randn(1, 3, 224, 224, generator=torch.Generator().manual_seed(GREEDY["image_seed"]))
    return cfg, sd, image


def to_hf_state_dict(sd, cfg):
    """Upstream GIT state-dict names -> HF GitForCausalLM names (SURVEY.md section 8b)."""
    out = {}
    v = cfg.vit
    W = v["width"]
    vm = "git.image_encoder.vision_model."
    out[vm + "embeddings.patch_embedding.weight"] = sd["image_encoder.conv1.weight"]
    out[vm + "embeddings.class_embedding"] = sd["image_encoder.class_embedding"]
    out[vm + "embeddings.position_embedding.weight"] = sd["image_encoder.positional_embedding"]
    for a, b in (("ln_pre", "pre_layrnorm"), ("ln_post", "post_layernorm")):
        out[vm + b + ".weight"] = sd[f"image_encoder.{a}.weight"]
        out[vm + b + ".bias"] = sd[f"image_encoder.{a}.bias"]
    for i in range(v["layers"]):
        s = f"image_encoder.transformer.resblocks.{i}."
        d = f"{vm}encoder.layers.{i}."
        for j, nm in enumerate(("q_proj", "k_proj", "v_proj")):
            out[d + f"self_attn.{nm}.weight"] = sd[s + "attn.in_proj_weight"][j * W:(j + 1) * W]
            out[d + f"self_attn.{nm}.bias"] = sd[s + "attn.in_proj_bias"][j * W:(j + 1) * W]
        for a, b in (("attn.out_proj", "self_attn.out_proj"), ("ln_1", "layer_norm1"), ("ln_2", "layer_norm2"),
                     ("mlp.c_fc", "mlp.fc1"), ("mlp.c_proj", "mlp.fc2")):
            out[d + b + ".weight"] = sd[s + a + ".weight"]
            out[d + b + ".bias"] = sd[s + a + ".bias"]
    for k, val in sd.items():
        if k.startswith("textual.visual_projection."):
            out["git.visual_projection.visual_projection." + k[len("textual.visual_projection."):]] = val
        elif k.startswith("textual.transformer.encoder."):
            out["git.encoder." + k[len("textual.transformer.encoder."):]] = val
        elif k.startswith("img_temperal_embedding."):
            out["git.img_temporal_embedding." + k.split(".")[-1]] = val
    out["git.embeddings.word_embeddings.weight"] = sd["textual.embedding.words.weight"]
    out["git.embeddings.position_embeddings.weight"] = sd["textual.embedding.positions.weight"]
    out["git.embeddings.LayerNorm.weight"] = sd["textual.embedding.layer_norm.weight"]
    out["git.embeddings.LayerNorm.bias"] = sd["textual.embedding.layer_norm.bias"]
    out["output.weight"] = sd["textual.output.weight"]
    out["output.bias"] = sd["textual.output.bias"]
    return out


def _load_hf(hf, sd, cfg):
    missing, unexpected = hf.load_state_dict(to_hf_state_dict(sd, cfg), strict=False)
    missing = [m for m in missing if "position_ids" not in m]
    assert not missing and not unexpected, (missing, unexpected)   # every HF weight comes from the oracle's state dict
    return hf


def compute():
    from transformers import GitConfig as HFGitConfig, GitForCausalLM

    torch.set_num_threads(max(1, min(8, os.cpu_count() or 1)))
    out = {}
    for encoder in ENCODERS:
        cfg, sd, frames, tokens = forward_inputs(encoder)
        large = encoder == "CLIPViT_L_14"
        vision = dict(hidden_size=1024, intermediate_size=4096, num_hidden_layers=24, num_attention_heads=16, patch_size=14,
                      image_size=224) if large else {}
        hf_cfg = HFGitConfig(num_image_with_embedding=FWD["n_frames"], layer_norm_eps=1e-12, tie_word_embeddings=False,
                             vision_config=vision or None)
        hf = _load_hf(GitForCausalLM(hf_cfg).eval(), sd, cfg)
        with torch.no_grad():
            logits = hf(input_ids=tokens, pixel_values=frames[None], output_hidden_states=False).logits
            vis = torch.cat([hf.git.image_encoder(frames[i:i + 1]).last_hidden_state + hf.git.img_temporal_embedding[i]
                             for i in range(FWD["n_frames"])], dim=1)
        nv = vis.shape[1]
        if logits.shape[1] == nv + tokens.shape[1]:  # HF returns every row; upstream keeps the text rows
            logits = logits[:, nv:]
        for name, a in (("visual_features", vis), ("logits", logits)):
            out[f"{encoder}.{name}_shape"] = np.array(a.shape)
            out[f"{encoder}.{name}_row_norms"] = a.double().norm(dim=-1).numpy()
            out[f"{encoder}.{name}_row_sums"] = a.double().sum(dim=-1).numpy()
        out[f"{encoder}.visual_features"] = vis[:, ::VIS_ROW, ::VIS_COL].numpy()
        out[f"{encoder}.logits"] = logits[..., ::LOGIT_COL].numpy()
        out[f"{encoder}.logits_argmax"] = logits.argmax(dim=-1).numpy()

    cfg, sd, image = greedy_inputs()
    hf_cfg = HFGitConfig(num_image_with_embedding=None, layer_norm_eps=1e-12, tie_word_embeddings=False,
                         bos_token_id=101, eos_token_id=102, pad_token_id=0)
    hf = _load_hf(GitForCausalLM(hf_cfg).eval(), sd, cfg)
    with torch.no_grad():
        # use_cache=False: in transformers 5.5 HF's CACHED GIT generation disagrees with HF's own full forward from the second
        # step on; the un-cached loop re-runs the full forward the forward comparison pins the oracle against
        gen = hf.generate(pixel_values=image, input_ids=torch.tensor([[101]]), max_length=GREEDY["max_steps"] - 1, do_sample=False,
                          num_beams=1, use_cache=False)[0]
    out["greedy.tokens"] = gen.numpy()
    return out


def main():
    np.savez_compressed(PATH, **compute())
    print(PATH, os.path.getsize(PATH))


if __name__ == "__main__":
    main()

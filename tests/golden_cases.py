"""Definitions of the golden cases shared by tools/make_goldens.py (which runs the UNMODIFIED reference in
the build container and writes tests/golden/*.npz) and by the tests that replay them against oracle/
and against the CUDA path.  Inputs are regenerated from seeds (mug_diffusion_b200.synth), only reference
OUTPUTS are stored."""
from __future__ import annotations

import numpy as np
import torch

from mug_diffusion_b200 import synth

U = "model.unet_model."
D = "model.first_stage_model.decoder."

# per-block cases at z_length 96 (levels 96/48/24/12), batch 2.
# kind, module path inside the reference DDPM (attribute path), state_dict prefix, input channels, ds
BLOCK_CASES = {
    "res_skipconv_l0":  dict(kind="res",  path="model.unet_model.input_blocks.2.0",  prefix=U + "input_blocks.2.0.",  cin=384, ds=1),
    "res_identity_l0":  dict(kind="res",  path="model.unet_model.input_blocks.3.0",  prefix=U + "input_blocks.3.0.",  cin=128, ds=1),
    "res_up_l3":        dict(kind="res",  path="model.unet_model.output_blocks.1.0", prefix=U + "output_blocks.1.0.", cin=1536, ds=8),
    "attn_l1":          dict(kind="attn", path="model.unet_model.input_blocks.6.1",  prefix=U + "input_blocks.6.1.",  cin=256, ds=2),
    "attn_l2":          dict(kind="attn", path="model.unet_model.input_blocks.10.1", prefix=U + "input_blocks.10.1.", cin=384, ds=4),
    "attn_mid":         dict(kind="attn", path="model.unet_model.middle_block.1",    prefix=U + "middle_block.1.",    cin=512, ds=8),
    "s4_l0":            dict(kind="s4",   path="model.unet_model.input_blocks.2.1",  prefix=U + "input_blocks.2.1.",  cin=128, ds=1),
    "s4_l2":            dict(kind="s4",   path="model.unet_model.input_blocks.10.2", prefix=U + "input_blocks.10.2.", cin=384, ds=4),
    "down_l0":          dict(kind="down", path="model.unet_model.input_blocks.4.0",  prefix=U + "input_blocks.4.0.",  cin=128, ds=1),
    "up_l1":            dict(kind="up",   path="model.unet_model.output_blocks.11.2", prefix=U + "output_blocks.11.2.", cin=256, ds=2),
    "dec_res_256_128":  dict(kind="dec_res", path="model.first_stage_model.decoder.up.1.block.0", prefix=D + "up.1.block.0.", cin=256, ds=1),
}
BLOCK_L = 96
BLOCK_B = 2

# self/cross attention cores (CrossAttention modules) -- [B, L, C] inputs
ATTN_CORE_CASES = {
    "self_d32":  dict(path="model.unet_model.input_blocks.6.1.transformer_blocks.0.attn1", prefix=U + "input_blocks.6.1.transformer_blocks.0.attn1.", C=256, L=48, cross=False),
    "cross_d48": dict(path="model.unet_model.input_blocks.10.1.transformer_blocks.0.attn2", prefix=U + "input_blocks.10.1.transformer_blocks.0.attn2.", C=384, L=24, cross=True),
    "self_d64_long": dict(path="model.unet_model.middle_block.1.transformer_blocks.0.attn1", prefix=U + "middle_block.1.transformer_blocks.0.attn1.", C=512, L=200, cross=False),
}

# whole-network cases: (z_length, batch, timesteps)
UNET_CASES = {
    "unet_L96_B2":  dict(L=96,  B=2, t=[981, 1]),
    "unet_L512_B2": dict(L=512, B=2, t=[501, 21]),
    "unet_L992_B1": dict(L=992, B=1, t=[741]),
}

# DDIM trajectories: (z_length, batch, S, cfg scale)
DDIM_CASES = {
    "ddim_L96_B1_S10_nocfg": dict(L=96,  B=1, S=10, scale=1.0),
    "ddim_L96_B2_S10_cfg5":  dict(L=96,  B=2, S=10, scale=5.0),
    "ddim_L512_B1_S50_cfg5": dict(L=512, B=1, S=50, scale=5.0),
}


def block_input(name: str, case: dict) -> torch.Tensor:
    L = BLOCK_L // case["ds"]
    rng = synth._rng(77, "block:" + name)
    return synth._gauss(rng, (BLOCK_B, case["cin"], L))


def block_emb(name: str) -> torch.Tensor:
    return synth._gauss(synth._rng(77, "emb:" + name), (BLOCK_B, 512))


def block_context(name: str) -> torch.Tensor:
    return synth._gauss(synth._rng(77, "ctx:" + name), (BLOCK_B, 128, 21))


def attn_core_inputs(name: str, case: dict):
    x = synth._gauss(synth._rng(78, "x:" + name), (BLOCK_B, case["L"], case["C"]))
    ctx = synth._gauss(synth._rng(78, "c:" + name), (BLOCK_B, 21, 128)) if case["cross"] else None
    return x, ctx


def load_golden(path):
    with np.load(path) as z:
        return {k: torch.from_numpy(z[k]) for k in z.files}


def synthetic_note_logits(B: int = 3, T: int = 700, seed: int = 9) -> torch.Tensor:
    """[B,16,T] logits that hit the corner cases of array_to_objects: dense starts, long notes that run into the last
    frame, a start on the last frame, holds interrupted by a new start, offsets outside [0,1] (clipped)."""
    x = synth._gauss(synth._rng(seed, "notes"), (B, 16, T)) * 1.5
    x[:, 0:4] -= 1.2                       # starts are sparse
    x[:, 8:12] += 0.8                      # holds are common -> long notes
    x[:, 4:8] = x[:, 4:8] * 2.0            # offsets beyond [0,1] -> clip
    x[0, 0, T - 1] = 2.0                   # start on the last frame
    x[1, 1, T - 40:] = -1.0
    x[1, 1, T - 40] = 3.0                  # long note running to the end
    x[1, 9, T - 39:] = 2.0
    x[2, 2, 10:20] = 1.0                   # back-to-back starts
    return x


# ---- prompt path (SURVEY 8f N3): feature dicts whose ids / embeddings are pinned to the reference in tests/golden/prompt.json
PROMPT_DICTS = [
    {},                                                        # the unconditional prompt (webui uc)
    {"sr": 6.4, "ln_ratio": 0.0, "rc": True},                  # the reference's own examples, mug/util.py:164-179
    {"sr": 6.2, "ln_ratio": 0.5, "rc": False},
    {"sr": 0, "ln_ratio": 0.5, "rc": True},                    # below min -> clamped
    {"sr": 0.6, "hb": True},
    {"sr": 99.0, "ln_ratio": 1.0, "ett": 35, "stamina_ett": 5},      # above max / at the edges
    {"sr": 3, "rank_status": "ranked", "rc": 1, "ln_ratio": 0},      # the SURVEY 8d bench prompt
    {"sr": 4.19999, "rank_status": "graveyard", "ln": False, "stamina": True, "stream_ett": 17.9},
    {"sr": 7.999, "rank_status": "loved", "hb": 0, "ln_ratio": 0.95},
]

# a spec that exercises what the shipped yaml does not: count > 1 and non-integer bin edges
PROMPT_SPEC_COUNT = [
    {"name": "a", "type": "numeric", "min": 0.5, "max": 2.0, "interval": 0.25, "count": 3},
    {"name": "b", "type": "category", "category": ["x", "y"], "count": 2},
    {"name": "c", "type": "bool"},
    {"name": "d", "type": "numeric", "min": -3, "max": 3, "interval": 1},
]


def random_feature_dicts(spec, n, rnd):
    """n feature dicts drawn from ``rnd`` (a random.Random): features left out, values below / above the range, at its
    edges and inside it; the ids the reference gives them are in tests/golden/prompt_random.json"""
    out = []
    for _ in range(n):
        d = {}
        for x in spec:
            if rnd.random() < 0.4:
                continue
            if x["type"] == "numeric":
                span = x["max"] - x["min"]
                d[x["name"]] = rnd.choice([x["min"] - 1, x["max"] + 1, x["min"] + span * rnd.random(), x["min"], x["max"]])
            elif x["type"] == "bool":
                d[x["name"]] = rnd.choice([True, False, 0, 1])
            else:
                d[x["name"]] = rnd.choice(x["category"])
        out.append(d)
    return out

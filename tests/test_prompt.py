"""Prompt path (SURVEY 8f N3): feature dict -> embedding ids -> [B,128,21] conditioning.
CPU: the oracle restatement and the product's host function against ids produced by the UNMODIFIED reference
(tests/golden/prompt.json, tools/make_goldens.py --only prompt; tests/golden/prompt_random.json, --only prompt_random).
GPU: the gather kernel behind ``model.model.cond_stage_model`` bit-exact against the reference embedder's output."""
import json
import os
import random
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import golden_cases as gc  # noqa: E402
from mug_diffusion_b200 import prompt as P  # noqa: E402
from oracle import mug_oracle as orc  # noqa: E402

SPEC_COUNT = gc.PROMPT_SPEC_COUNT


@pytest.fixture(scope="module")
def gold(golden_dir):
    return json.load(open(os.path.join(golden_dir, "prompt.json")))


def test_ids_match_reference_golden(gold):
    assert gold["dicts"] == gc.PROMPT_DICTS
    for d, want in zip(gold["dicts"], gold["ids"]):
        assert orc.feature_ids(d, gold["spec"]) == want
        assert P.feature_dict_to_embedding_ids(d, gold["spec"]) == want
    assert P.count_beatmap_features(gold["spec"]) == gold["n_embed"] == 329
    assert len(gold["ids"][0]) == 21 and gold["ids"][0] == orc.feature_ids({}, gold["spec"])      # uc: every slot "missing"


def test_count_slots_and_errors():
    dicts = [{}, {"a": 1.3, "b": "y", "c": True, "d": -7}, {"a": 2.0, "b": "x", "c": 0, "d": 2.9}, {"a": 0.74999}]
    for d in dicts:
        ids = P.feature_dict_to_embedding_ids(d, SPEC_COUNT)
        assert ids == orc.feature_ids(d, SPEC_COUNT)
        assert len(ids) == 3 + 2 + 1 + 1 and max(ids) < P.count_beatmap_features(SPEC_COUNT)
    # slots of one feature share the bin but own consecutive row blocks
    ids = P.feature_dict_to_embedding_ids({"a": 1.3}, SPEC_COUNT)
    w = P.count_beatmap_features_embedding(SPEC_COUNT[0])
    assert ids[1] - ids[0] == w and ids[2] - ids[1] == w
    for fn in (P.feature_dict_to_embedding_ids, orc.feature_ids):
        with pytest.raises(ValueError):                       # the reference's list.index raises ValueError too
            fn({"b": "not-a-category"}, SPEC_COUNT)
    with pytest.raises(ValueError):
        P.count_beatmap_features([{"name": "z", "type": "weird"}])


def test_oracle_embed_matches_reference_golden(gold, golden_dir):
    g = gc.load_golden(os.path.join(golden_dir, "prompt_embed.npz"))
    ids = torch.tensor(np.asarray(gold["ids"]), dtype=torch.float32)          # float ids, as webui.py:191 passes them
    assert torch.equal(orc.prompt_embed(g["table"], ids), g["out"])


def test_ids_match_live_reference_on_random_dicts(gold, golden_dir):
    """300 seeded random dicts per spec against the ids the reference's feature_dict_to_embedding_ids gave them"""
    cases = json.load(open(os.path.join(golden_dir, "prompt_random.json")))
    rnd = random.Random(5)
    assert len(cases) == 2
    for spec, case in zip((gold["spec"], SPEC_COUNT), cases):
        assert case["spec"] == spec
        dicts = gc.random_feature_dicts(spec, 300, rnd)
        assert dicts == case["dicts"]
        assert P.count_beatmap_features(spec) == case["n_embed"]
        for d, want in zip(dicts, case["ids"]):
            assert P.feature_dict_to_embedding_ids(d, spec) == want
            assert orc.feature_ids(d, spec) == want


# ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_gpu_embedder_bit_exact_and_wired(gold, golden_dir):
    from mug_diffusion_b200 import synth
    from mug_diffusion_b200.config import ModelConfig
    from mug_diffusion_b200.sampler import PROMPT_TABLE_KEY, MugDiffusionB200
    g = gc.load_golden(os.path.join(golden_dir, "prompt_embed.npz"))
    sd = synth.synthetic_state_dict(gc.BLOCK_L)
    sd[PROMPT_TABLE_KEY] = g["table"]
    model = MugDiffusionB200(sd, ModelConfig(), z_length=gc.BLOCK_L, device="cuda:0")
    ids = torch.tensor(np.asarray(gold["ids"]), dtype=torch.float32, device="cuda")        # webui.py:190-193
    c = model.model.cond_stage_model(ids)
    assert c.shape == (len(gold["ids"]), 128, 21) and c.dtype == torch.float32
    assert torch.equal(c.cpu(), g["out"])
    with pytest.raises(IndexError):
        model.model.cond_stage_model(torch.full((1, 21), 329.0))
    # the conditioning feeds the U-Net like the reference's: same eps as with the golden tensor handed over from the host
    x = synth._gauss(synth._rng(3, "px"), (2, 16, gc.BLOCK_L))
    w = [synth._gauss(synth._rng(4, f"pw{i}"), (2, ch, gc.BLOCK_L >> i)).cuda() for i, ch in enumerate((256, 512, 512, 512))]
    t = torch.tensor([500, 20])
    e1 = model.model.forward(x.cuda(), t.cuda(), c[1:3], w)
    e2 = model.model.forward(x.cuda(), t.cuda(), g["out"][1:3].cuda(), w)
    assert torch.equal(e1, e2)
    # a model built without the table says so
    bare = MugDiffusionB200(synth.synthetic_state_dict(gc.BLOCK_L), ModelConfig(), z_length=gc.BLOCK_L, device="cuda:0")
    with pytest.raises(RuntimeError):
        bare.model.cond_stage_model(ids)

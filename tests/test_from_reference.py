"""The drop-in constructor reads the architecture off a live reference DDPM.  The reference's side is replayed from
tests/golden/ref_model.json (tools/make_goldens.py --only refmodel): the attributes config_from_reference reads and the name
and shape of every state_dict entry of a DDPM built from the reference's shipped yaml."""
import json
import os
from types import SimpleNamespace

import torch

from mug_diffusion_b200 import netspec
from mug_diffusion_b200.config import ModelConfig
from mug_diffusion_b200.sampler import MugDiffusionB200


class _Module(SimpleNamespace):
    """attributes plus a state_dict() of zero-strided tensors with the recorded shapes (no weight memory)"""

    def __init__(self, shapes, prefix, **attrs):
        super().__init__(**attrs)
        self._shapes = {k[len(prefix):]: s for k, s in shapes.items() if k.startswith(prefix)}

    def state_dict(self):
        return {k: torch.zeros(()).expand(s) for k, s in self._shapes.items()}


def _reference_ddpm(golden_dir):
    g = json.load(open(os.path.join(golden_dir, "ref_model.json")))
    sd = g["state_dict"]
    dec = g["decoder"]
    decoder = SimpleNamespace(num_resolutions=dec["num_resolutions"], num_res_blocks=dec["num_res_blocks"],
                              norm_out=SimpleNamespace(num_groups=dec["norm_out_num_groups"]))
    model = SimpleNamespace(unet_model=_Module(sd, "model.unet_model.", **g["unet"]),
                            first_stage_model=SimpleNamespace(decoder=decoder, **g["first_stage"]))
    return _Module(sd, "", model=model, **g["ddpm"])


def test_config_from_reference_matches_shipped_yaml(golden_dir):
    sd, cfg = MugDiffusionB200.config_from_reference(_reference_ddpm(golden_dir))
    want = ModelConfig()
    assert cfg.unet == want.unet
    assert cfg.decoder == want.decoder
    assert (cfg.z_channels, cfg.timesteps, cfg.linear_start, cfg.linear_end) == (16, 1000, 1e-4, 2e-2)
    # every tensor the packer needs is present in the reference state_dict under the names netspec generates
    need = {**netspec.unet_param_specs(cfg.unet), **netspec.decoder_param_specs(cfg.decoder)}
    assert all(k in sd and tuple(sd[k].shape) == tuple(shape) for k, (shape, _) in need.items())

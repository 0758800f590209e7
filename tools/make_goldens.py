"""Generate tests/golden/*.npz by running the UNMODIFIED reference (/root/reference, CPU fp32, via
tools/ref_shim.py) on the seeded synthetic weights/inputs of mug_diffusion_b200.synth.

Run in the build container only (the GPU box has no /root/reference):
    python tools/make_goldens.py [--only blocks|unet|ddim|s4len|wave|notes|prompt|prompt_random|refmodel]
"""
import argparse
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.path.insert(0, os.path.join(ROOT, "tests"))

import golden_cases as gc  # noqa: E402
import ref_shim  # noqa: E402
from mug_diffusion_b200 import synth  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")


def get_module(model, path):
    m = model
    for part in path.split("."):
        m = m[int(part)] if part.isdigit() else getattr(m, part)
    return m


def fresh_model(z_length):
    """A new reference model per config (S4 mutates its state on first use of a length, SURVEY H2)."""
    model, _ = ref_shim.load_reference_model(z_length=z_length)
    sd = synth.synthetic_state_dict(z_length)
    missing, unexpected = model.load_state_dict(sd, strict=False)
    bad = [k for k in missing if k.startswith("model.unet_model.") or k.startswith("model.first_stage_model.decoder.")]
    assert not bad and not unexpected, (bad[:5], unexpected[:5])
    return model, sd


def save(name, **arrs):
    np.savez_compressed(os.path.join(GOLD, name + ".npz"), **{k: np.asarray(v, dtype=np.float32) for k, v in arrs.items()})
    print("wrote", name, {k: tuple(np.shape(v)) for k, v in arrs.items()})


@torch.no_grad()
def make_blocks():
    model, _ = fresh_model(gc.BLOCK_L)
    out = {}
    for name, case in gc.BLOCK_CASES.items():
        mod = get_module(model, case["path"])
        x = gc.block_input(name, case)
        if case["kind"] == "res":
            y = mod(x, gc.block_emb(name))
        elif case["kind"] == "attn":
            y = mod(x, gc.block_context(name))
        else:
            y = mod(x)
        out[name] = y.numpy()
        if case["kind"] == "s4":
            k, _ = mod.s4_model.kernel(L=x.shape[-1])
            out[name + ".K"] = k[0].numpy()
    for name, case in gc.ATTN_CORE_CASES.items():
        mod = get_module(model, case["path"])
        x, ctx = gc.attn_core_inputs(name, case)
        out["core." + name] = mod(x, context=ctx).numpy()
    save("blocks_L96", **out)


@torch.no_grad()
def make_unet():
    for name, case in gc.UNET_CASES.items():
        model, _ = fresh_model(case["L"])
        inp = synth.synthetic_inputs(case["B"], case["L"])
        t = torch.tensor(case["t"], dtype=torch.long)
        t0 = time.time()
        eps = model.model.forward(inp["x_T"], t, inp["c"], synth.wave_list(inp["w"]))
        print(name, "ref eval %.2fs" % (time.time() - t0))
        save(name, eps=eps.numpy())


@torch.no_grad()
def make_ddim():
    from mug.diffusion.ddim import DDIMSampler

    for name, case in gc.DDIM_CASES.items():
        model, _ = fresh_model(case["L"])
        model.z_length = case["L"]
        inp = synth.synthetic_inputs(case["B"], case["L"])
        sampler = DDIMSampler(model)
        pred = []
        t0 = time.time()
        z, inter = sampler.sample(S=case["S"], c=inp["c"], w=synth.wave_list(inp["w"]), batch_size=case["B"],
                                  shape=None, verbose=False, x_T=inp["x_T"], eta=0.0,
                                  unconditional_guidance_scale=case["scale"],
                                  unconditional_conditioning=inp["uc"],
                                  img_callback=lambda p, i: pred.append(p.clone()))
        logits = model.model.decode(z)
        print(name, "ref sample+decode %.2fs" % (time.time() - t0))
        save(name, z=z.numpy(), logits=logits.numpy(), pred_x0_first=pred[0].numpy(), pred_x0_last=pred[-1].numpy())


@torch.no_grad()
def make_s4_lengthen():
    """C~ lengthening (s4.py:557-584): a layer persisted at L=48 asked for L=96 (doubling), then 4x (two doublings),
    and a never-run layer (L buffer 0) initialised at 96."""
    out = {}
    for tag, L_state, L_req in (("double", 48, 96), ("double2", 24, 96), ("init", 0, 96)):
        model, _ = fresh_model(max(L_state, 8) if L_state else 96)
        mod = get_module(model, "model.unet_model.input_blocks.2.1").s4_model.kernel.kernel
        mod.L.fill_(L_state)
        k, _ = mod(L=L_req)
        out[tag + ".C"] = mod.C.detach().numpy().copy()
        out[tag + ".L"] = np.asarray([int(mod.L.item())], dtype=np.float32)
        out[tag + ".K"] = k[0].numpy().copy()
    save("s4_lengthen", **out)
    # whole U-Net: weights persisted at z_length 48 (S4 buffers 48/24/12/6), evaluated at 96 -> every S4 layer doubles
    model, _ = fresh_model(48)
    inp = synth.synthetic_inputs(2, 96)
    eps = model.model.forward(inp["x_T"], torch.tensor([981, 1]), inp["c"], synth.wave_list(inp["w"]))
    save("unet_L96_from48", eps=eps.numpy())



@torch.no_grad()
def make_wave():
    """the reference audio encoder (wave.py:398-467) on a synthetic mel, T = 64 * 96 frames: last four level outputs"""
    from mug_diffusion_b200 import wave as mwave
    model, _ = ref_shim.load_reference_model()
    wsd = mwave.synthetic_wave_state_dict()
    missing, unexpected = model.load_state_dict(wsd, strict=False)
    assert not [k for k in missing if k.startswith("model.wave_model.")] and not unexpected
    mel = mwave.synthetic_mel(2, 64 * 96)
    hs = model.model.wave_model(mel)
    save("wave_T6144_B2", **{f"h{i}": hs[i].numpy() for i in range(6, 10)})
    print([tuple(h.shape) for h in hs])


def make_prompt():
    """Prompt path (SURVEY 8f N3): the reference's feature_dict_to_embedding_ids on a set of feature dicts (its own examples,
    mug/util.py:164-179, plus clamping / missing / count>1 / category cases) and BeatmapFeatureEmbedder.forward on those ids
    with a seeded table.  The parsed feature spec travels with the golden (the GPU box has no /root/reference)."""
    import json
    import yaml
    ref_shim.install_shims()
    from mug.cond.feature import BeatmapFeatureEmbedder
    from mug.util import count_beatmap_features, feature_dict_to_embedding_ids
    ypath = os.path.join(ref_shim.REF_ROOT, "configs", "mug", "mania_beatmap_features.yaml")
    spec = yaml.safe_load(open(ypath))
    ids = [feature_dict_to_embedding_ids(d, spec) for d in gc.PROMPT_DICTS]
    emb = BeatmapFeatureEmbedder(ypath, 128)
    g = torch.Generator().manual_seed(77)
    with torch.no_grad():
        emb.embedding.weight.copy_(torch.randn(emb.embedding.weight.shape, generator=g))
        out = emb(torch.tensor(np.asarray(ids), dtype=torch.float32))       # float ids, as webui.py:191 passes them
    json.dump(dict(spec=spec, dicts=gc.PROMPT_DICTS, ids=ids, n_embed=count_beatmap_features(spec)),
              open(os.path.join(GOLD, "prompt.json"), "w"), indent=1)
    save("prompt_embed", table=emb.embedding.weight.detach().numpy(), out=out.numpy())
    print("prompt:", len(ids), "dicts,", len(ids[0]), "slots, table", tuple(emb.embedding.weight.shape))


def make_prompt_random():
    """The reference's count_beatmap_features and feature_dict_to_embedding_ids on 300 seeded random feature dicts for the
    shipped spec (from prompt.json) and for a spec with count > 1 slots."""
    import json
    import random
    ref_shim.install_shims()
    from mug.util import count_beatmap_features, feature_dict_to_embedding_ids
    rnd = random.Random(5)
    out = []
    for spec in (json.load(open(os.path.join(GOLD, "prompt.json")))["spec"], gc.PROMPT_SPEC_COUNT):
        dicts = gc.random_feature_dicts(spec, 300, rnd)
        out.append(dict(spec=spec, n_embed=count_beatmap_features(spec), dicts=dicts,
                        ids=[feature_dict_to_embedding_ids(d, spec) for d in dicts]))
    with open(os.path.join(GOLD, "prompt_random.json"), "w") as f:
        json.dump(out, f)
    print("wrote prompt_random.json", [len(c["dicts"]) for c in out])


def make_reference_model():
    """What MugDiffusionB200.config_from_reference reads off a reference DDPM built from the shipped yaml: the module
    attributes and the name and shape of every state_dict entry."""
    import json
    model, _ = ref_shim.load_reference_model()
    unet, fs = model.model.unet_model, model.model.first_stage_model
    out = dict(
        ddpm=dict(z_channels=int(model.z_channels), num_timesteps=int(model.num_timesteps),
                  linear_start=float(model.linear_start), linear_end=float(model.linear_end)),
        unet={a: (list(getattr(unet, a)) if isinstance(getattr(unet, a), (list, tuple)) else int(getattr(unet, a)))
              for a in ("in_channels", "model_channels", "out_channels", "num_res_blocks", "attention_resolutions",
                        "channel_mult", "num_heads")},
        first_stage=dict(scale=float(fs.scale)),
        decoder=dict(num_resolutions=int(fs.decoder.num_resolutions), num_res_blocks=int(fs.decoder.num_res_blocks),
                     norm_out_num_groups=int(fs.decoder.norm_out.num_groups)),
        state_dict={k: list(v.shape) for k, v in model.state_dict().items()})
    with open(os.path.join(GOLD, "ref_model.json"), "w") as f:
        json.dump(out, f)
    print("wrote ref_model.json:", len(out["state_dict"]), "state_dict entries")


def make_hit_objects():
    """OsuManiaConvertor.array_to_objects of the UNMODIFIED reference on the golden decoder logits (and on a synthetic
    logit array that exercises long notes running to the last frame, back-to-back starts and clipped offsets)."""
    import json
    ref_shim.install_shims()
    from mug.data.convertor import BeatmapMeta, OsuManiaConvertor
    frame_ms = 512 / 4 / 22050 * 8 * 1000          # webui.py:341-342 hop 128 @ 22.05 kHz x audio_note_window_ratio 8
    conv = OsuManiaConvertor(frame_ms=frame_ms, max_frame=4096, from_logits=True)
    meta = BeatmapMeta(path="", cs=4)
    out = {"frame_ms": frame_ms}
    for name in ("ddim_L512_B1_S50_cfg5", "ddim_L96_B2_S10_cfg5"):
        lg = gc.load_golden(os.path.join(GOLD, name + ".npz"))["logits"].numpy()
        out[name] = [conv.array_to_objects(lg[b], meta) for b in range(lg.shape[0])]
    syn = gc.synthetic_note_logits().numpy()
    out["synthetic"] = [conv.array_to_objects(syn[b], meta) for b in range(syn.shape[0])]
    with open(os.path.join(GOLD, "hit_objects.json"), "w") as f:
        json.dump(out, f)
    print("wrote hit_objects.json", {k: (len(v) if isinstance(v, list) else v) for k, v in out.items()}, [len(c) for c in out["synthetic"]])


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--only", default=None)
    a = ap.parse_args()
    torch.set_num_threads(os.cpu_count())
    os.makedirs(GOLD, exist_ok=True)
    if a.only in (None, "blocks"):
        make_blocks()
    if a.only in (None, "unet"):
        make_unet()
    if a.only in (None, "ddim"):
        make_ddim()
    if a.only in (None, "s4len"):
        make_s4_lengthen()
    if a.only in (None, "wave"):
        make_wave()
    if a.only in (None, "notes"):
        make_hit_objects()
    if a.only in (None, "prompt"):
        make_prompt()
    if a.only in (None, "prompt_random"):
        make_prompt_random()
    if a.only in (None, "refmodel"):
        make_reference_model()



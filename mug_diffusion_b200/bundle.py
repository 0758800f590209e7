"""Export one compiled sampling request as a bundle a host WITHOUT Python can run (examples/host_c/sample_host.c):

    python -m mug_diffusion_b200.bundle --out /tmp/bundle --L 96 --B 1 --S 10 --scale 5

The network -> launch-plan compiler is Python (engine.py); what it produces is plain data: arrays of mugd_op whose pointers fall
into a handful of device allocations.  The bundle holds
    manifest.txt        region table (name, bytes, initial contents), the plans in execution order, test inputs, expected outputs
    *.plan              mugd_plan_save files (pointers stored as region + offset)
    *.bin               region contents: the packed weight blob as it is resident (hi in place) + its lo buffer, the S4 convolution kernels, the per-request tables (timestep
                        sinusoids and DDIM coefficients for the chosen S -- host float math, kept out of the C demo), test vectors
Request flow = DDIMSampler.sample + model.decode (ddim.py:56-196, diffusion.py:49-50):
    emb (time-embedding table) -> ctx (cross-attention K|V) -> audio (concat slots) -> loadx -> S x {eval graph ; update ; advance}
    -> readz -> decode -> readlogits
"""
from __future__ import annotations

import argparse
import ctypes as C
import os
from typing import Dict, List

import numpy as np
import torch

from . import lib as L_
from .engine import OpList
from .runtime import Plan, _ptr


def _save_plan(eng, ops: OpList, regions: List[L_.Region], path: str) -> Plan:
    pl = Plan(eng, ops)
    arr = (L_.Region * len(regions))(*regions)
    L_.check(eng.lib.mugd_plan_save(pl.handle, arr, len(regions), path.encode()), f"plan_save {path}")
    return pl


def export_bundle(model, inp: Dict[str, torch.Tensor], S: int, scale: float, out_dir: str) -> Dict[str, torch.Tensor]:
    """Compile the request (inp: x_T, c, uc, w[4] on the host), write the bundle, run it once through the very same plans and
    return the results (z, logits) that the C host must reproduce."""
    from .sampler import DDIMSampler

    os.makedirs(out_dir, exist_ok=True)
    eng = model.engine
    dev = eng.device
    cfg = eng.cfg
    B, Cz, Lz = inp["x_T"].shape
    cfg_on = scale != 1.0
    Beff = 2 * B if cfg_on else B
    sampler = DDIMSampler(model)
    sampler.make_schedule(S, verbose=False)
    ts = np.flip(sampler.ddim_timesteps)
    total = len(ts)

    with eng.lock:
        sess = eng.session(Beff, Lz, per_sample_t=False)
        dec = eng.decoder_session(B, Lz)
        T = inp["c"].shape[2]
        if T != sess.ctx_tokens:
            sess.ctx_tokens = T
            sess._build(sess.comp)
        # ---- staging buffers of the caller (inputs / outputs in the reference's NCL layout) ----
        st = dict(in_x=inp["x_T"].to(dev).contiguous(), in_c=inp["c"].to(dev).contiguous(), in_uc=inp["uc"].to(dev).contiguous(),
                  pred=torch.zeros(B * Lz * Cz, device=dev), out_z=torch.zeros(B, Cz, Lz, device=dev),
                  out_logits=torch.zeros(B, cfg.decoder.x_channels, dec.Lout, device=dev))
        w4 = [w.to(dev).contiguous() for w in list(inp["w"])[-cfg.unet.levels:]]
        for i, w in enumerate(w4):
            st[f"in_w{i}"] = w
        # per-request host tables for this S
        sess.set_timestep_table(ts.copy())
        coef = np.stack([np.asarray(a, dtype=np.float32) for a in (sampler.ddim_alphas, sampler.ddim_alphas_prev, sampler.ddim_sigmas,
                                                                   sampler.ddim_sqrt_one_minus_alphas)], axis=1)
        sess.coef.zero_()
        sess.coef[:total].copy_(torch.from_numpy(np.ascontiguousarray(coef)).to(dev))

        # ---- regions: every device allocation a plan may point into ----
        tensors: Dict[str, torch.Tensor] = dict(weights=eng.weights, weights_lo=eng.weights_lo, arena=sess.arena_t, emb_table=sess.emb_table, temb=sess.temb,
                                                emb_h1=sess.emb_h1, emb_h2=sess.emb_h2, step=sess.step, coef=sess.coef, ctx=sess.ctx,
                                                tc_ws=eng.tc_ws, dec_arena=dec.arena_t)
        for i, t in enumerate(sess.ctx_kv):
            tensors[f"ctx_kv{i}"] = t
        for i, (_, t) in enumerate(sorted(sess.s4_kt.items())):
            tensors[f"s4_kt{i}"] = t
        tensors.update(st)
        contents = {"weights", "weights_lo", "temb", "coef"} | {k for k in tensors if k.startswith("s4_kt")}       # saved; everything else starts zeroed
        inputs = {k for k in st if k.startswith("in_")}
        names = list(tensors)
        keep = [n.encode() for n in names]
        regions = [L_.Region(keep[i], _ptr(tensors[n]), tensors[n].numel() * tensors[n].element_size()) for i, n in enumerate(names)]

        # ---- the plans ----
        upd = L_.DdimUpdate()
        upd.x = sess.xin.ptr
        upd.x_dup = sess.xin.r(B * Lz, 2 * B * Lz).ptr if cfg_on else None
        upd.eps, upd.pred_x0, upd.coef, upd.step = sess.eps.ptr, _ptr(st["pred"]), _ptr(sess.coef), _ptr(sess.step)
        upd.S, upd.n, upd.cfg, upd.scale, upd.temperature = total, B * Lz * Cz, int(cfg_on), float(scale), 1.0
        adv = L_.StepAdvance()
        adv.step = _ptr(sess.step)
        tail = OpList()
        tail.add(L_.OP_DDIM_UPDATE, upd)
        tail.add(L_.OP_STEP_ADVANCE, adv)
        readz = OpList()
        readz.transpose(sess.xin.ptr, _ptr(st["out_z"]), sess.xin.ld, 0, B, Cz, Lz, False)
        dec_in = OpList()
        assert cfg.decoder.scale == 1.0, "bundle export assumes first-stage scale 1 (the shipped config)"
        dec_in.transpose(_ptr(st["out_z"]), dec.zin.ptr, 0, dec.zin.ld, B, cfg.decoder.z_channels, Lz, True)
        dec_out = OpList()
        dec_out.transpose(dec.logits.ptr, _ptr(st["out_logits"]), dec.logits.ld, 0, B, cfg.decoder.x_channels, dec.Lout, False)
        ctx_parts = [(_ptr(st["in_uc"]), B), (_ptr(st["in_c"]), B)] if cfg_on else [(_ptr(st["in_c"]), B)]
        seq = [("emb", sess.timestep_ops(total), "run"), ("ctx", sess.context_ops(ctx_parts, T), "run"),
               ("audio", sess.audio_ops([_ptr(w) for w in w4], cfg_on), "run"), ("loadx", sess.loadx_ops(_ptr(st["in_x"]), B, cfg_on), "run"),
               ("eval", None, "graph"), ("tail", tail, "tail"), ("readz", readz, "run"), ("dec_in", dec_in, "run"), ("dec", None, "graph"),
               ("dec_out", dec_out, "run")]
        plans = {}
        lines = ["mugd_bundle 1", f"# z_length {Lz} batch {B} guidance {scale} steps {total} (S={S})"]
        for n in names:
            t = tensors[n]
            nbytes = t.numel() * t.element_size()
            if n in contents or n in inputs:
                t.detach().cpu().contiguous().numpy().tofile(os.path.join(out_dir, n + ".bin"))
                lines.append(f"region {n} {nbytes} file {n}.bin")
            else:
                lines.append(f"region {n} {nbytes} zero -")
        for name, ops, mode in seq:
            path = os.path.join(out_dir, name + ".plan")
            if ops is None:
                pl = sess.plan if name == "eval" else dec.plan
                arr = (L_.Region * len(regions))(*regions)
                L_.check(eng.lib.mugd_plan_save(pl.handle, arr, len(regions), path.encode()), f"plan_save {name}")
            else:
                pl = _save_plan(eng, ops, regions, path)
            plans[name] = pl
            if mode == "tail":
                continue
            if name == "eval":
                lines.append(f"sample eval.plan tail.plan {total}")
            else:
                lines.append(f"plan {name}.plan {mode}")

        # ---- run the request once through these very plans: the expected outputs ----
        sess.set_step(0)
        for name in ("emb", "ctx", "audio", "loadx"):
            plans[name].run()
        sess.run_steps(total, tail)
        for name in ("readz", "dec_in"):
            plans[name].run()
        if not dec.plan.captured:
            dec.plan.run()
            dec.plan.capture()
        dec.plan.replay(1)
        plans["dec_out"].run()
        torch.cuda.synchronize()
        for n in ("out_z", "out_logits"):
            st[n].cpu().numpy().tofile(os.path.join(out_dir, n + ".expected.bin"))
            lines.append(f"expect {n} {st[n].numel() * 4} {n}.expected.bin")
        open(os.path.join(out_dir, "manifest.txt"), "w").write("\n".join(lines) + "\n")
        return dict(z=st["out_z"].clone(), logits=st["out_logits"].clone())


def main():
    from . import synth
    from .sampler import MugDiffusionB200

    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--L", type=int, default=96)
    ap.add_argument("--B", type=int, default=1)
    ap.add_argument("--S", type=int, default=10)
    ap.add_argument("--scale", type=float, default=5.0)
    a = ap.parse_args()
    model = MugDiffusionB200.from_state_dict(synth.synthetic_state_dict(a.L), z_length=a.L)
    inp = synth.synthetic_inputs(a.B, a.L)
    res = export_bundle(model, inp, a.S, a.scale, a.out)
    print("bundle written to", a.out, "| z", tuple(res["z"].shape), "logits", tuple(res["logits"].shape))


if __name__ == "__main__":
    main()

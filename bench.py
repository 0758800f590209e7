#!/usr/bin/env python
"""Benchmark of the denoising hot path (BASELINE.json metric: denoising-steps/sec).

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--workload NAME] [--no-secondary] [--dump-outputs DIR]

One "step" = one DDIM step of the workload's whole per-GPU batch: Beff U-Net evaluations (2B with
classifier-free guidance) + the CFG/DDIM update.  Default workload = BASELINE.json configs[1]:
3-min audio (z_length 512), 4 charts, webui-default CFG scale 5 (effective U-Net batch 8), 50-step schedule.
Multi-GPU: every rank runs the same per-GPU batch on different samples after one NCCL weight broadcast
(weak scaling, no per-step collective); value = N*K / max-over-ranks time.

The ONE JSON line (rank 0) carries, besides the contract keys,
  roofline / cpu_baseline / e2e            for the headline workload,
  secondary.workloads                      the same measurements for BASELINE configs 3 (L512_B32) and 5 (L992_B8) at N=1,
                                           and for config 4's per-GPU batch (32 charts / GPU) at every N.
--impl reference times the CPU oracle port of the reference path (oracle/mug_oracle.py: torch CPU fp32) on the same workload.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: z_length, per-GPU batch, CFG scale, schedule length S
    "L512_B4_cfg5_S50": dict(L=512, B=4, scale=5.0, S=50),          # BASELINE config 2 (headline)
    "L512_B4_nocfg_S50": dict(L=512, B=4, scale=1.0, S=50),
    "L512_B32_cfg5_S50": dict(L=512, B=32, scale=5.0, S=50),        # BASELINE config 3; per-GPU batch of config 4 (256 / 8 GPUs)
    "L992_B8_cfg5_S100": dict(L=992, B=8, scale=5.0, S=100),        # BASELINE config 5
    "L96_B1_cfg5_S10": dict(L=96, B=1, scale=5.0, S=10),            # BASELINE config 1 shape
}
GFLOP_PER_EVAL = {96: 4.19, 512: 22.46, 992: 44.37}        # BASELINE.md §3, per sample-eval
METRIC = "denoising-steps/sec"
UNIT = "DDIM steps/s (whole per-GPU batch per step, summed over GPUs)"
MIN_REGION_S = 0.6          # steps are replayed for at least this long before the timed K steps so the clock sampler sees the load


def config_of(name, wl, world=1, **extra):
    """the keys BOTH arms print, so the driver can compare configs"""
    Beff = wl["B"] * (2 if wl["scale"] != 1.0 else 1)
    d = dict(workload=name, z_length=wl["L"], per_gpu_batch=wl["B"], global_batch=wl["B"] * world, unet_batch_per_gpu=Beff,
             cfg_scale=wl["scale"], schedule_S=wl["S"])
    d.update(extra)
    return d


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(tflops=float(d.get("bf16_tflops_sustained", d.get("bf16_tflops", 1590.0))), hbm=float(d.get("hbm_gbs", 6650.0)),
                    src="measured (MEASURED_PEAKS.json bf16_tflops_sustained)")
    return dict(tflops=1400.0, hbm=6650.0, src="fallback (B200_PROFILING.md)")


def ncu_step_traffic(name):
    """Whole-step DRAM traffic from the committed ncu capture of ONE graphed-plan evaluation of this workload
    (profiles/r02_step_traffic.json, written by tools/summarize_step_ncu.py): every launch of the eval, --cache-control none."""
    p = os.path.join(ROOT, "profiles", "r02_step_traffic.json")
    try:
        return json.load(open(p)).get(name)
    except Exception:
        return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons while the step loop runs (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows, self.proc, self.gpu = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50",
                                          "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"], samples=0)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = [float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = set()
        for r in self.rows:
            if len(r) >= 9:
                for n, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
        return dict(sm_mhz=float(np.median(sm)) if sm else None, sm_max_mhz=max(mx) if mx else None,
                    reasons=sorted(reasons), samples=len(sm),
                    note="sampled every 50 ms from the sustain phase (same step loop, >= 0.6 s) through the timed K steps")


def make_inputs(wl, rank):
    from mug_diffusion_b200 import synth

    return synth.synthetic_inputs(wl["B"], wl["L"], seed=1234 + rank)


# ---------------------------------------------------------------------------------------------------
# reference arm / cpu_baseline : the oracle port of the reference path on the host cores
# ---------------------------------------------------------------------------------------------------
def time_oracle_steps(wl, steps, warmup, repeats=3, sd=None, budget_s=120.0):
    """DDIM steps of the CPU oracle (full workload batch, CFG as configured).  One protocol for both the reference arm and the
    cpu_baseline leg: probe the thread count, `warmup` untimed steps, then `repeats` timed blocks of `steps` steps; the MEDIAN block
    is reported.  Returns dict(value, threads, host_cores, seconds, blocks)."""
    from mug_diffusion_b200 import synth
    from oracle import mug_oracle as orc

    sd = sd or synth.synthetic_state_dict(wl["L"], decoder=False)
    inp = make_inputs(wl, 0)
    # Give the CPU arm its best thread count: torch's default (= all cores) oversubscribes the many small
    # ops of this network on big hosts (128 threads ran 100x slower than 16 on the GPU box), so probe a few
    # counts on one eval of the workload's shape and keep the fastest.
    ncpu = os.cpu_count() or 1
    cands = sorted({c for c in (8, 16, 32, 64, ncpu) if c <= ncpu})
    pb = min(wl["B"] * (2 if wl["scale"] != 1.0 else 1), 8)
    reps_p = (pb + wl["B"] - 1) // wl["B"]
    px = torch.cat([inp["x_T"]] * reps_p)[:pb]
    pc = torch.cat([inp["c"]] * reps_p)[:pb]
    pw = [torch.cat([w] * reps_p)[:pb] for w in inp["w"]]
    probe_t = torch.full((pb,), 500, dtype=torch.long)
    best, best_dt = cands[0], float("inf")
    torch.set_num_threads(cands[0])
    with torch.no_grad():                      # untimed first call (allocator / oneDNN primitive caches)
        orc.unet_forward(sd, px, probe_t, pc, pw)
    for c in cands:
        torch.set_num_threads(c)
        d = float("inf")
        for _ in range(2):
            with torch.no_grad():
                t0 = time.perf_counter()
                orc.unet_forward(sd, px, probe_t, pc, pw)
                d = min(d, time.perf_counter() - t0)
        if d < best_dt:
            best, best_dt = c, d
        if d > 3 * best_dt:
            break
    torch.set_num_threads(best)
    sch = orc.make_schedule(wl["S"])
    ts = np.flip(sch["timesteps"])
    x = inp["x_T"]
    B = wl["B"]
    cfg = wl["scale"] != 1.0

    def one(i, x):
        t = torch.full((B,), int(ts[i % len(ts)]), dtype=torch.long)
        with torch.no_grad():
            if cfg:
                e = orc.unet_forward(sd, torch.cat([x, x]), torch.cat([t, t]), torch.cat([inp["uc"], inp["c"]]),
                                     [torch.cat([w, w]) for w in inp["w"]])
                eu, ec = e.chunk(2)
                e = eu + wl["scale"] * (ec - eu)
            else:
                e = orc.unet_forward(sd, x, t, inp["c"], inp["w"])
        idx = len(ts) - 1 - (i % len(ts))
        a_t, a_prev = float(sch["alphas"][idx]), float(sch["alphas_prev"][idx])
        pred = (x - float(sch["sqrt_one_minus_alphas"][idx]) * e) / a_t ** 0.5
        return a_prev ** 0.5 * pred + (1 - a_prev) ** 0.5 * e

    k = 0
    for _ in range(warmup):
        x = one(k, x)
        k += 1
    blocks = []
    t_all = time.perf_counter()
    for r in range(repeats):
        t0 = time.perf_counter()
        for _ in range(steps):
            x = one(k, x)
            k += 1
        blocks.append(time.perf_counter() - t0)
        if time.perf_counter() - t_all > budget_s:      # bounded sample: never let the CPU leg run away on a slow host
            break
    dt = float(np.median(blocks))
    return dict(value=steps / dt, threads=torch.get_num_threads(), host_cores=ncpu, seconds=dt, blocks=[round(b, 3) for b in blocks])


def cpu_baseline_dict(r, steps, warmup):
    return dict(value=r["value"], unit=UNIT, cores=r["threads"], host_cores=r["host_cores"], kind="port",
                sample=f"median of {len(r['blocks'])} blocks of {steps} full DDIM steps of the workload (+{warmup} warm-up) on the CPU oracle "
                       f"port; {r['threads']} torch threads (probed best of 8/16/32/64/all) on a host with {r['host_cores']} logical cores; "
                       f"block seconds {r['blocks']}")


def run_reference(args, wl, name):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    r = time_oracle_steps(wl, args.steps, args.warmup)
    v = r["value"]
    line = dict(metric=METRIC, value=v, unit=UNIT, n_gpus=args.gpus, steps=args.steps, warmup=args.warmup,
                ms_per_step=1000.0 / v, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f32", data="synthetic",
                impl="reference",
                config=config_of(name, wl, args.gpus),        # identical keys and values to the B200 arm's `config`
                info=dict(note="CPU oracle port of the reference PyTorch path (oracle/mug_oracle.py, bit-identical to the reference on "
                               "tests/golden); S4 kernels regenerated every eval like the reference.  One host runs ONE per-GPU batch: at "
                               "--gpus N > 1 only rank 0 measures one per-GPU batch, so the driver's ratio compares N GPUs with one CPU host"),
                cpu_baseline=cpu_baseline_dict(r, args.steps, args.warmup),
                e2e=dict(value=v, unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=0), gpu_launches=0)
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------------------
# the B200 arm
# ---------------------------------------------------------------------------------------------------
class _NoBar:
    def __init__(self, it, **kw):
        self.it = it

    def __iter__(self):
        return iter(self.it)


def build_model(L, world, rank, dev, gemm):
    import torch.distributed as dist

    from mug_diffusion_b200 import synth
    from mug_diffusion_b200.config import ModelConfig
    from mug_diffusion_b200.dist import broadcast_blob
    from mug_diffusion_b200.sampler import MugDiffusionB200

    cfg = ModelConfig()
    if world > 1:                                  # rank 0 builds + packs, ONE NCCL broadcast of the blob
        sd = synth.synthetic_state_dict(L) if rank == 0 else None
        blob = broadcast_blob(sd, cfg, dev)
        return MugDiffusionB200(None, cfg, z_length=L, device=dev, gemm_impl=gemm, blob=blob), sd
    sd = synth.synthetic_state_dict(L)
    return MugDiffusionB200(sd, cfg, z_length=L, device=dev, gemm_impl=gemm, fold_ln={"0": False, "1": True}.get(os.environ.get("MUGD_FOLD_LN", ""))), sd


def measure(model, name, wl, steps, warmup, world, rank, dev, with_roofline=True, sustain=True):
    """value (device-resident loop, CUDA events, max over ranks), roofline of the GEMM family, e2e through the public API."""
    import torch.distributed as dist

    from mug_diffusion_b200 import lib as L_
    from mug_diffusion_b200.engine import OpList
    from mug_diffusion_b200.sampler import DDIMSampler, _ptr

    eng = model.engine
    L, B, S = wl["L"], wl["B"], wl["S"]
    cfg_on = wl["scale"] != 1.0
    Beff = 2 * B if cfg_on else B
    inp = make_inputs(wl, rank)
    sampler = DDIMSampler(model)

    # ---- device-resident timed loop ("value") -----------------------------------------------------
    # Set the request up exactly as sample() does, then drive steps of (graph replay + update) by hand.
    sampler.make_schedule(S, verbose=False)
    sess = eng.session(Beff, L, per_sample_t=False)
    ts = np.flip(sampler.ddim_timesteps)
    rows = 1000
    reps = rows // len(ts) + 1
    sess.set_timestep_table(np.tile(ts, reps)[:rows])
    sess.set_context([inp["uc"].to(dev), inp["c"].to(dev)] if cfg_on else inp["c"].to(dev))
    sess.set_audio([w.to(dev) for w in inp["w"]], dup=cfg_on)
    coef = np.stack([np.asarray(a, dtype=np.float32) for a in (sampler.ddim_alphas, sampler.ddim_alphas_prev, sampler.ddim_sigmas,
                                                               sampler.ddim_sqrt_one_minus_alphas)], axis=1)
    # the step counter cycles through the rows; replicate the coefficient table so row (rows-1-i) is valid
    sess.coef[:rows].copy_(torch.from_numpy(np.ascontiguousarray(np.tile(coef, (reps, 1))[:rows])).to(dev))
    n = B * L * 16
    upd = L_.DdimUpdate()
    upd.x = sess.xin.ptr
    upd.x_dup = sess.xin.r(B * L, 2 * B * L).ptr if cfg_on else None
    upd.eps, upd.coef, upd.step = sess.eps.ptr, _ptr(sess.coef), _ptr(sess.step)
    upd.S, upd.n, upd.cfg, upd.scale, upd.temperature = rows, n, int(cfg_on), float(wl["scale"]), 1.0
    adv = L_.StepAdvance()
    adv.step = _ptr(sess.step)
    tail = OpList()
    tail.add(L_.OP_DDIM_UPDATE, upd)
    tail.add(L_.OP_STEP_ADVANCE, adv)
    budget = [0]

    def restart():
        sess.load_x(inp["x_T"].to(dev), dup=cfg_on)
        sess.set_step(0)
        budget[0] = rows

    def step():
        if budget[0] == 0:
            restart()
        budget[0] -= 1
        sess.eval(graph=True)
        eng.run_ops(tail)

    restart()
    for _ in range(max(warmup, 3)):
        step()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    clocks = ClockSampler(dev.index or 0)
    if rank == 0:
        clocks.start()
    # sustain phase: the same loop, untimed, long enough for the 50 ms clock sampler to see the load the timed steps run under
    if sustain:
        t0 = time.perf_counter()
        while time.perf_counter() - t0 < MIN_REGION_S:
            for _ in range(10):
                step()
            torch.cuda.synchronize()
    restart()                                   # the timed steps start from x_T at step 0, whatever the sustain phase ran
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0.record()
    for _ in range(steps):                      # EXACTLY K timed steps
        step()
    e1.record()
    torch.cuda.synchronize()
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.barrier()
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms = float(ms.item())
    clock_info = clocks.stop() if rank == 0 else None
    launches_per_step = sess.plan.launches + 2
    value = world * steps / (ms / 1000.0)
    # what the last timed step computed: the latent after its DDIM update and the U-Net output it used (read here: the
    # roofline below reuses the session's buffers)
    outputs = dict(x=sess.read_rows(sess.xin.r(0, B * L), B, 16, L).cpu(), eps=sess.read_rows(sess.eps, Beff, 16, L).cpu())
    finite = bool(torch.isfinite(outputs["eps"]).all())

    # ---- roofline of the dominant kernel family (GEMM) -----------------------------------------------------
    # Device time per kernel family, measured live with CUDA events: the ops of one family are put in their own
    # launch plan, captured as a CUDA graph (no host launch overhead in the number) and replayed back to back.
    roof = None
    if rank == 0 and with_roofline:
        from mug_diffusion_b200.runtime import Plan
        ops_all = sess.plan._arr
        names = {1: "gemm", 2: "groupnorm", 3: "layernorm", 4: "attention", 5: "s4conv", 7: "transpose", 8: "copy2d"}
        fam_ms, fam_n = {}, {}
        gemm_flops = 0.0
        for kind in sorted({ops_all[i].kind for i in range(sess.plan.n_ops)}):
            sub = OpList()
            for i in range(sess.plan.n_ops):
                if ops_all[i].kind == kind:
                    sub.ops.append(ops_all[i])
                    if kind == L_.OP_GEMM:
                        g = ops_all[i].u.gemm
                        gemm_flops += 2.0 * g.M * g.N * (g.K * g.taps + g.K2)
            pl = Plan(eng, sub)
            pl.run()
            pl.capture()
            pl.replay(2)
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            a0.record()
            pl.replay(5)
            a1.record()
            torch.cuda.synchronize()
            fam_ms[kind] = a0.elapsed_time(a1) / 5
            fam_n[kind] = pl.launches
        pk = measured_peaks()
        gemm_ms, gemm_n = fam_ms[L_.OP_GEMM], fam_n[L_.OP_GEMM]
        ach = gemm_flops / (gemm_ms * 1e-3) / 1e12
        tr = ncu_step_traffic(name)
        roof = dict(bound="tensor", kernel=f"gemm_tc_kernel (tcgen05 3xTF32; impl={eng.gemm_impl})", achieved=ach, peak=pk["tflops"],
                    unit="TFLOP/s", frac=ach / pk["tflops"], frac_of_3xtf32_ceiling=ach / (pk["tflops"] / 6.0),
                    traffic=(tr or {}).get("gemm_bytes_per_launch"), peak_source=pk["src"], launches=gemm_n,
                    traffic_note=("profiles/r02_step_traffic.json: dram__bytes_read+write summed over EVERY gemm_tc launch of one whole eval "
                                  "of this workload (ncu --cache-control none), divided by the launches; whole-step sum and the ratio to the "
                                  "algorithmic bytes are in `step_traffic`") if tr else "no committed whole-step ncu capture for this workload",
                    step_traffic=tr,
                    avg_launch_us=1000.0 * gemm_ms / max(gemm_n, 1), algorithmic_gflop_per_step=gemm_flops / 1e9,
                    note="3xTF32 issues 3 tensor-core products per fp32 product and TF32 runs at half the bf16 rate: "
                         "the fp32-exact ceiling is peak/6",
                    family_ms_in_graph={names.get(k, str(k)): round(v, 4) for k, v in sorted(fam_ms.items())},
                    family_launches={names.get(k, str(k)): fam_n[k] for k in sorted(fam_n)})

    # ---- end to end through the public API with HOST (pinned) inputs ----------------------------------
    # ONE full request of the workload: its own S-step schedule (not K), inputs in pinned host memory, logits back in pinned host
    # memory; the copies are inside the timed region.
    host = dict(x_T=inp["x_T"].pin_memory(), c=inp["c"].pin_memory(), uc=inp["uc"].pin_memory(), w=[w.pin_memory() for w in inp["w"]])
    h2d = sum(t.numel() * 4 for t in [host["x_T"], host["c"], host["uc"]] + host["w"])
    out_host = torch.empty(B, 16, 8 * L).pin_memory()
    trace = os.environ.get("BENCH_E2E_TRACE") == "1"      # phase wall times (adds syncs: not for the reported number)

    def request():
        tt = [time.perf_counter()]

        def mark():
            if trace:
                torch.cuda.synchronize()
                tt.append(time.perf_counter())
        c = host["c"].to(dev, non_blocking=True)
        uc = host["uc"].to(dev, non_blocking=True)
        w = [t.to(dev, non_blocking=True) for t in host["w"]]
        xT = host["x_T"].to(dev, non_blocking=True)
        mark()
        z, _ = sampler.sample(S=S, c=c, w=w, batch_size=B, shape=(16, L), verbose=False, x_T=xT, eta=0.0,
                              unconditional_guidance_scale=wl["scale"], unconditional_conditioning=uc, tqdm_class=_NoBar)
        mark()
        logits = model.model.decode(z)
        mark()
        out_host.copy_(logits, non_blocking=True)
        torch.cuda.synchronize()
        mark()
        if trace and rank == 0:
            print(f"e2e phases ms ({name}; h2d, sample, decode, d2h):", [round(1e3 * (b - a), 2) for a, b in zip(tt, tt[1:])], file=sys.stderr)
        return out_host

    request()                                   # warm (decoder plan + graph)
    torch.cuda.synchronize()
    times = []
    for _ in range(3):                          # three whole requests, the median one is reported (a single request is ~0.2 s:
        if world > 1:                           # one host hiccup would otherwise be the number)
            dist.barrier()
        t0 = time.perf_counter()
        out = request()
        dt = torch.tensor([time.perf_counter() - t0], device=dev)
        if world > 1:
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        times.append(float(dt.item()))
    dt = torch.tensor([sorted(times)[1]], device=dev)
    n_steps_e2e = len(sampler.ddim_timesteps)
    outputs["e2e_logits"] = out.clone()
    e2e = dict(value=world * n_steps_e2e / float(dt.item()), unit=UNIT, h2d_bytes_per_step=h2d / n_steps_e2e,
               d2h_bytes_per_step=out.numel() * 4 / n_steps_e2e, request_ms=1000.0 * float(dt.item()), request_ms_all=[round(1000.0 * t, 2) for t in times], steps_in_request=n_steps_e2e,
               note=f"median of 3 sampler.sample(S={S}) + decode requests per GPU from pinned host inputs to pinned host logits; "
                    f"{n_steps_e2e} DDIM steps; per-step bytes = request bytes / steps")
    return dict(value=value, ms_per_step=ms / steps, e2e=e2e, roofline=roof, launches_per_step=launches_per_step, clocks=clock_info,
                finite=finite, sampler=sampler, host=host, Beff=Beff, outputs=outputs)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="L512_B4_cfg5_S50", choices=list(WORKLOADS))
    ap.add_argument("--gemm", default=os.environ.get("MUGD_GEMM", "auto"), choices=["auto", "simt", "tc", "tc_tf32"],
                    help="tc_tf32 = opt-in single-pass TF32 (NOT fp32-accurate; for characterisation only)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the secondary workloads (configs 3/4/5)")
    ap.add_argument("--cpu-steps", type=int, default=10)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write rank 0's outputs of the headline workload as float32 DIR/<name>.npy: x (latent after the last timed "
                         "step), eps (U-Net output of that step) and e2e_logits (decoder logits of the last end-to-end request)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to --impl b200")
    name = args.workload
    wl = WORKLOADS[name]
    if args.impl == "reference":
        return run_reference(args, wl, name)

    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torchrun"
    dev = torch.device(f"cuda:{local}")
    torch.cuda.set_device(dev)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    L, B, S = wl["L"], wl["B"], wl["S"]

    model, sd = build_model(L, world, rank, dev, args.gemm)
    eng = model.engine
    m = measure(model, name, wl, args.steps, args.warmup, world, rank, dev)
    if args.dump_outputs and rank == 0:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for k, v in m["outputs"].items():
            np.save(os.path.join(args.dump_outputs, k + ".npy"), v.numpy())

    # ---- secondary numbers: the same loop without guidance, the decode, and the other BASELINE configs -----------------------
    secondary = None
    if not args.no_secondary:
        sampler, host = m["sampler"], m["host"]
        secondary = {}
        if rank == 0:
            def timed_request(scale, S2):
                c = host["c"].to(dev); uc = host["uc"].to(dev); w = [t.to(dev) for t in host["w"]]; xT = host["x_T"].to(dev)
                sampler.sample(S=2, c=c, w=w, batch_size=B, shape=(16, L), verbose=False, x_T=xT, eta=0.0, unconditional_guidance_scale=scale,
                               unconditional_conditioning=uc, tqdm_class=_NoBar)                      # session build + capture
                b0, b1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                torch.cuda.synchronize()
                b0.record()
                z, _ = sampler.sample(S=S2, c=c, w=w, batch_size=B, shape=(16, L), verbose=False, x_T=xT, eta=0.0,
                                      unconditional_guidance_scale=scale, unconditional_conditioning=uc, tqdm_class=_NoBar)
                b1.record()
                torch.cuda.synchronize()
                return z, len(sampler.ddim_timesteps) / (b0.elapsed_time(b1) / 1000.0)
            z, v_nocfg = timed_request(1.0, 50)
            model.model.decode(z)
            d0, d1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            d0.record()
            for _ in range(5):
                model.model.decode(z)
            d1.record()
            torch.cuda.synchronize()
            secondary.update(steps_per_s_without_cfg=v_nocfg, unet_batch_without_cfg=B,
                             note_steps="sampler.sample(S=50, scale=1.0) through the public API incl. per-request setup",
                             decode_ms=d0.elapsed_time(d1) / 5,
                             decode_note=f"model.model.decode of {B} latents [16,{L}] -> logits [16,{8 * L}] (CUDA graph + boundary transposes)")
        # Other BASELINE configs.  N = 1: configs 3 and 5.  N > 1: config 4's per-GPU batch (32 charts per GPU) on every rank.
        others = ["L512_B32_cfg5_S50"] if world > 1 else ["L512_B32_cfg5_S50", "L992_B8_cfg5_S100"]
        wls = {}
        for oname in others:
            if oname == name:
                continue
            owl = WORKLOADS[oname]
            if owl["L"] == L:
                omodel = model
            else:
                del model, eng
                model = eng = None
                torch.cuda.empty_cache()
                omodel, _ = build_model(owl["L"], world, rank, dev, args.gemm)
            osteps = max(10, min(args.steps, 30))
            om = measure(omodel, oname, owl, osteps, 3, world, rank, dev, sustain=True)
            wls[oname] = dict(value=om["value"], unit=UNIT, ms_per_step=om["ms_per_step"], steps=osteps, n_gpus=world,
                              config=config_of(oname, owl, world), chart_steps_per_s=om["value"] * owl["B"],
                              e2e=om["e2e"], roofline=om["roofline"], launches_per_step=om["launches_per_step"], clocks=om["clocks"],
                              outputs_finite=om["finite"])
            if owl["L"] != L:
                del omodel
                torch.cuda.empty_cache()
        secondary["workloads"] = wls
        if world > 1:
            secondary["note_multi_gpu"] = ("L512_B32_cfg5_S50 at N GPUs is BASELINE config 4's shape (32 charts per GPU; 256 charts at N=8), "
                                           "sharded by sample with no per-step collective")

    # ---- CPU baseline (rank 0, N=1 only, bounded sample): the SAME protocol as --impl reference ---------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        r = time_oracle_steps(wl, args.cpu_steps, 2, repeats=3, budget_s=45.0,
                              sd={k: v for k, v in sd.items() if k.startswith("model.unet_model.")})
        cpu = cpu_baseline_dict(r, args.cpu_steps, 2)

    if rank == 0:
        Beff = m["Beff"]
        line = dict(metric=METRIC, value=m["value"], unit=UNIT, n_gpus=world, steps=args.steps, warmup=max(args.warmup, 3),
                    ms_per_step=m["ms_per_step"], higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f32", data="synthetic",
                    config=config_of(name, wl, world),
                    info=dict(gemm_impl=args.gemm, parallelism=f"replica-sharded batch x{world}",
                              l2="working set exceeds L2: ~0.8 GB of TF32 hi/lo weight operands are streamed every step",
                              gflop_per_step=Beff * GFLOP_PER_EVAL.get(L, 0.0), outputs_finite=m["finite"]),
                    roofline=m["roofline"], cpu_baseline=cpu, e2e=m["e2e"], secondary=secondary,
                    gpu_launches=m["launches_per_step"] * args.steps, launches_per_step=m["launches_per_step"], clocks=m["clocks"])
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()

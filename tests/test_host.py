"""CPU-only checks of the host logic: netspec keys, packer layouts, plan compiler bookkeeping, schedule,
and that libmugd.so loads and exports every symbol include/mugd.h declares (no compute without a GPU)."""
import ctypes as C
import json
import os
import re

import numpy as np
import pytest
import torch

from mug_diffusion_b200 import lib as L_
from mug_diffusion_b200 import netspec, packer, sampler, synth
from mug_diffusion_b200.config import ModelConfig
from mug_diffusion_b200.engine import Arena, DecoderCompiler, UNetCompiler, View
from oracle import mug_oracle as orc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_netspec_keys_match_reference_state_dict(golden_dir):
    ref = json.load(open(os.path.join(golden_dir, "ref_keys.json")))
    cfg = ModelConfig()
    mine = {**netspec.unet_param_specs(cfg.unet), **netspec.decoder_param_specs(cfg.decoder)}
    assert set(mine) == set(ref)
    for k, (shape, _) in mine.items():
        assert list(shape) == ref[k], k


def test_library_loads_and_exports_header_symbols():
    lib = L_.load()
    hdr = open(os.path.join(ROOT, "include", "mugd.h")).read()
    declared = set(re.findall(r"\b(mugd_[a-z0-9_]+)\s*\(", hdr))
    assert declared == set(L_.EXPORTED_SYMBOLS)
    for sym in declared:
        assert hasattr(lib, sym), sym
    assert lib.mugd_abi_version() == L_.ABI_VERSION


def test_no_cpu_fallback_without_gpu():
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    lib = L_.load()
    h = C.c_void_p()
    assert lib.mugd_create(0, C.byref(h)) == 3          # MUGD_ERR_NO_DEVICE
    assert b"no CPU fallback" in lib.mugd_last_error()
    with pytest.raises(L_.MugdError):
        sampler.MugDiffusionB200.from_state_dict({}, z_length=96)


def test_schedule_tables_equal_oracle():
    for S, eta in ((50, 0.0), (10, 0.0), (30, 0.0), (20, 0.7)):
        o = orc.make_schedule(S, eta)
        sch = sampler.register_schedule()
        ts = sampler.ddim_timesteps_uniform(S, 1000)
        sig, al, alp = sampler.ddim_parameters(sch["alphas_cumprod"], ts, eta)
        assert np.array_equal(ts, o["timesteps"])
        assert np.array_equal(np.asarray(al), np.asarray(o["alphas"]))
        assert np.array_equal(np.asarray(alp), np.asarray(o["alphas_prev"]))
        assert np.array_equal(np.asarray(sig), np.asarray(o["sigmas"]))


@pytest.fixture(scope="module")
def packed():
    cfg = ModelConfig()
    sd = synth.synthetic_state_dict(96)
    return cfg, sd, packer.pack_model(sd, cfg.unet, cfg.decoder)


def test_packer_layouts(packed):
    cfg, sd, blob = packed
    p = "model.unet_model.input_blocks.2.0."
    w = sd[p + "in_layers.2.weight"]
    pw = blob.view(p + "in_layers.2.weight")
    assert pw.shape == (128, 3 * 384)
    assert torch.equal(pw.view(128, 3, 384)[:, 1, :], w[:, :, 1])
    t = "model.unet_model.input_blocks.6.1.transformer_blocks.0."
    qkv = blob.view(t + "attn1.qkv.weight")
    assert torch.equal(qkv[256:512], sd[t + "attn1.to_k.weight"])
    ff = blob.view(t + "ff.net.0.proj.weight")
    assert torch.equal(ff[0::2], sd[t + "ff.net.0.proj.weight"][:1024]) and torch.equal(ff[1::2], sd[t + "ff.net.0.proj.weight"][1024:])
    assert blob.meta["emb_total"] == 7424
    assert all(e.offset % 64 == 0 for e in blob.entries.values())
    assert blob.meta["model.unet_model.input_blocks.6.2.s4_model.kernel.kernel.L"] == 48


def _fake_ext(comp, Beff, Lz):
    blocks = [b for e in comp.lay.input + [comp.lay.middle] + comp.lay.output if not isinstance(e, tuple) for b in e]
    return dict(emb_table=1 << 40, step=(1 << 40) + 4096, ctx_tokens=21,
                ctx_kv=[View((1 << 41) + i * (1 << 24), 2 * b.cin, Beff * 21, 2 * b.cin) for i, b in enumerate(x for x in blocks if x.kind == "attn")],
                s4_kt={b.prefix: View((1 << 42) + i * (1 << 24), b.cin, Lz // b.ds, b.cin) for i, b in enumerate(x for x in blocks if x.kind == "s4")})


@pytest.mark.parametrize("fuse", [False, True], ids=["plain", "ln_folded"])
@pytest.mark.parametrize("Beff,Lz", [(2, 96), (8, 512), (1, 992)])
def test_unet_plan_compiles_and_is_consistent(packed, Beff, Lz, fuse):
    cfg, sd, blob = packed
    comp = UNetCompiler(cfg.unet, blob, 1 << 30)
    arena = Arena(1 << 32)
    res = comp.compile(arena, Beff, Lz, _fake_ext(comp, Beff, Lz), False, fuse)
    ops = res["ops"].ops
    kinds = [o.kind for o in ops]
    gemms = [o.u.gemm for o in ops if o.kind == L_.OP_GEMM]
    # 22 ResBlocks, 16 transformers, 16 S4 layers (SURVEY §8a)
    assert kinds.count(L_.OP_S4CONV) == 16 and kinds.count(L_.OP_ATTENTION) == 32
    assert kinds.count(L_.OP_GROUPNORM) == 44 + 16 + 16 + 1
    assert len(res["audio_slots"]) == 8
    if fuse:
        # all 48 LayerNorms ride in the epilogue of the Linear behind them; the producer of each one's input delivers row moments
        assert kinds.count(L_.OP_LAYERNORM) == 0 and sum(1 for g in gemms if g.ln_stats) == 48
        assert sum(1 for g in gemms if g.row_moments) == 48
        assert kinds[0] == L_.OP_COPY2D and kinds.count(L_.OP_COPY2D) == 5   # first op zeroes the row-moment block
    else:
        assert kinds.count(L_.OP_LAYERNORM) == 48 and not any(g.row_moments or g.ln_stats for g in gemms)
        assert kinds.count(L_.OP_COPY2D) == 4                     # only the 4 doubly-homed skip tensors are copied
    # by default the fold is chosen by size: below 8192 token rows (Beff * Lz)
    auto = comp.compile(Arena(1 << 32), Beff, Lz, _fake_ext(comp, Beff, Lz), False)
    assert auto["ln_folded"] == (Beff * Lz < 8192)
    # every GEMM's output stays inside the arena; deterministic recompile gives identical addresses
    arena2 = Arena(1 << 32)
    res2 = comp.compile(arena2, Beff, Lz, _fake_ext(comp, Beff, Lz), False, fuse)
    assert arena.high == arena2.high
    for o, o2 in zip(ops, res2["ops"].ops):
        if o.kind == L_.OP_GEMM:
            assert o.u.gemm.C == o2.u.gemm.C and (1 << 32) <= o.u.gemm.C < (1 << 32) + arena.high
            g = o.u.gemm
            assert g.K % 16 == 0 and g.N % 4 == 0 and g.M % g.Lout == 0
    # the parity-split Upsample convs (CONV_TAPS) do 2/3 of the literal FLOPs: count them at the reference's cost
    flops = sum(2.0 * o.u.gemm.M * o.u.gemm.N * (o.u.gemm.K * o.u.gemm.taps * (1.5 if (o.u.gemm.conv_mode == L_.CONV_TAPS and o.u.gemm.taps == 2) else 1.0) + o.u.gemm.K2)
                for o in ops if o.kind == L_.OP_GEMM)
    # the 16 skip_connection convs and the 16 proj_out convs ride as second sources of other GEMMs
    assert sum(1 for o in ops if o.kind == L_.OP_GEMM and o.u.gemm.K2 > 0) == 32
    if Lz == 512:
        # GEMM-class work per sample-eval (BASELINE.md §3: 21.80 GFLOP) minus the hoisted emb / ctx-KV projections
        assert abs(flops / Beff / 1e9 - 21.8) < 0.3


def test_decoder_plan_compiles(packed):
    cfg, sd, blob = packed
    comp = DecoderCompiler(cfg.decoder, blob, 1 << 30)
    res = comp.compile(Arena(1 << 32), 2, 96)
    kinds = [o.kind for o in res["ops"].ops]
    assert kinds.count(L_.OP_GROUPNORM) == 21 and res["Lout"] == 768
    flops = sum(2.0 * o.u.gemm.M * o.u.gemm.N * o.u.gemm.K * o.u.gemm.taps * (1.5 if (o.u.gemm.conv_mode == L_.CONV_TAPS and o.u.gemm.taps == 2) else 1.0)
                for o in res["ops"].ops if o.kind == L_.OP_GEMM)
    assert abs(flops / 2 / 1e9 - 1.23) < 0.05                 # BASELINE.md: 1.23 GFLOP per chart at L=96


def test_synthetic_streams_are_stable():
    """the seeded generators must not drift: goldens depend on them"""
    sd = synth.synthetic_state_dict(96, decoder=False)
    w = sd["model.unet_model.input_blocks.0.0.weight"]
    assert abs(float(w.double().sum()) - (-17.870057)) < 1e-3, float(w.double().sum())
    x = synth.synthetic_inputs(1, 96)["x_T"]
    assert abs(float(x.double().sum()) - -30.42121) < 1e-3, float(x.double().sum())


@pytest.mark.parametrize("Beff,Lz", [(2, 96), (8, 512), (64, 512), (16, 992)])
def test_tensor_core_planner_invariants(packed, Beff, Lz):
    """tile / split-K planning of the tcgen05 GEMM (pure host code in libmugd, no GPU needed) over every GEMM of real plans:
    what it takes it must be able to run with the engine's fixed 32 MB workspace."""
    import ctypes as C
    cfg, sd, blob = packed
    lib = L_.load()
    comp = UNetCompiler(cfg.unet, blob, 1 << 30)
    res = comp.compile(Arena(1 << 32), Beff, Lz, _fake_ext(comp, Beff, Lz), False)
    n_tc = n_split = 0
    for o in res["ops"].ops:
        if o.kind != L_.OP_GEMM:
            continue
        g = o.u.gemm
        ok, sp, nt, ws = C.c_int32(), C.c_int32(), C.c_int32(), C.c_int64()
        assert lib.mugd_gemm_tc_query(None, C.byref(g), 148, C.byref(ok), C.byref(sp), C.byref(ws), C.byref(nt)) == 0
        small = g.K % 32 != 0 or g.N < 16                       # conv_in (K = 16 per tap) stays on the FFMA kernel
        assert bool(ok.value) == (not small), (g.M, g.N, g.K)
        if not ok.value:
            assert sp.value == 0 and ws.value == 0
            assert not g.W_hi                                    # FFMA GEMMs must read a weight the device-side TF32 split left alone
            continue
        assert g.W_hi == g.W                                     # hi lives where the plain weight was: no fp32 duplicate is resident
        n_tc += 1
        ksteps = g.taps * (g.K // 32) + g.K2 // 32
        assert 1 <= sp.value <= ksteps and 1 <= nt.value <= 4096
        if sp.value > 1:
            n_split += 1
            assert nt.value * sp.value <= 2 * 148               # bounds the workspace: fewer than 2 partial tiles per SM
            assert ksteps // sp.value >= 2                       # a split never leaves a CTA with a single k-step
            assert 0 < ws.value <= 32 << 20
            assert ws.value % (128 * 64 * 4) == 0                # whole 128-row partial tiles
        else:
            assert ws.value == 0
        # a machine with fewer SMs never gets more CTAs than twice its size out of a split either
        sp2, nt2 = C.c_int32(), C.c_int32()
        lib.mugd_gemm_tc_query(None, C.byref(g), 64, None, C.byref(sp2), None, C.byref(nt2))
        assert sp2.value == 1 or nt2.value * sp2.value <= 2 * 64
    assert n_tc >= 190          # 228 - 32 (fused second-source GEMMs) + 1
    if Beff <= 8:
        assert n_split > 100                                     # small batches underfill 148 SMs: most GEMMs are split
    if Beff == 64:
        assert n_split < n_tc // 2


@pytest.mark.parametrize("Beff,Lz", [(8, 512), (64, 512), (16, 992)])
def test_tensor_core_variant_rule(packed, Beff, Lz):
    """which GEMM kernel variant the planner picks (pure host code): the two-CTAs-per-SM variant only for unsplit GEMMs with more
    128-wide tiles than SMs, never more than 2 x SMs CTAs; small batches never see it except for their widest GEMMs"""
    import ctypes as C
    cfg, sd, blob = packed
    lib = L_.load()
    comp = UNetCompiler(cfg.unet, blob, 1 << 30)
    res = comp.compile(Arena(1 << 32), Beff, Lz, _fake_ext(comp, Beff, Lz), False)
    n_two = n_tc = 0
    for o in res["ops"].ops:
        if o.kind != L_.OP_GEMM:
            continue
        g = o.u.gemm
        bn, occ, ctas = C.c_int32(), C.c_int32(), C.c_int32()
        assert lib.mugd_gemm_tc_variant(C.byref(g), 148, C.byref(bn), C.byref(occ), C.byref(ctas)) == 0
        if bn.value == 0:
            assert g.K % 32 != 0                                  # only conv_in stays on the FFMA kernel
            continue
        n_tc += 1
        sp, nt = C.c_int32(), C.c_int32()
        lib.mugd_gemm_tc_query(None, C.byref(g), 148, None, C.byref(sp), None, C.byref(nt))
        assert bn.value in (64, 128, 256) and occ.value in (1, 2)
        if occ.value == 2:
            n_two += 1
            assert bn.value == 128 and sp.value == 1 and nt.value > 148 and ctas.value == min(nt.value, 296)
        else:
            assert ctas.value == nt.value * sp.value
    assert n_tc >= 190
    if Beff == 64:
        assert n_two >= 60                                        # the big batch runs most of its GEMM time on the two-CTA variant
    if Beff == 8:
        assert n_two <= 20                                        # only the widest feed-forward GEMMs have more tiles than SMs

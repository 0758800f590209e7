"""Runtime: ``MugEngine`` (handle + weights on one GPU) and ``Session`` (compiled state for one shape)."""
from __future__ import annotations

import ctypes as C
import threading
from collections import OrderedDict
from typing import Dict, List, Optional, Sequence

import numpy as np
import torch

from . import lib as L_
from .config import ModelConfig
from .engine import (Arena, CTX_TOKENS_MAX, DecoderCompiler, MAX_STEPS, OpList, UNetCompiler, View, tc_weight_map)
from .netspec import s4_blocks
from .packer import WeightBlob, pack_model


def _ptr(t: torch.Tensor) -> int:
    return t.data_ptr()


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


class Plan:
    def __init__(self, engine: "MugEngine", ops: OpList):
        self.engine = engine
        self.n_ops = len(ops.ops)
        engine.attach_workspace(ops)
        self._arr = ops.array()
        self.handle = C.c_void_p()
        L_.check(engine.lib.mugd_plan_create(engine.handle, self._arr, self.n_ops, C.byref(self.handle)), "plan_create")
        self.captured = False
        self.launches = 0

    def run(self):
        L_.check(self.engine.lib.mugd_plan_run(self.handle, _stream()), "plan_run")
        self.launches = self.engine.lib.mugd_plan_launch_count(self.handle)

    def capture(self):
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            L_.check(self.engine.lib.mugd_plan_capture(self.handle, side.cuda_stream), "plan_capture")
        torch.cuda.current_stream().wait_stream(side)
        self.launches = self.engine.lib.mugd_plan_launch_count(self.handle)
        self.captured = True

    def replay(self, times: int = 1):
        L_.check(self.engine.lib.mugd_plan_replay(self.handle, times, _stream()), "plan_replay")

    def __del__(self):
        try:
            if self.handle:
                self.engine.lib.mugd_plan_destroy(self.handle)
        except Exception:
            pass


class MugEngine:
    """One GPU: libmugd handle + packed weights.  Thread-safe through a single lock (the reference is not
    re-entrant either: webui.py:355-356 mutates model.z_length per request)."""

    def __init__(self, state_dict: Dict[str, torch.Tensor], cfg: Optional[ModelConfig] = None,
                 device: Optional[torch.device] = None, gemm_impl: str = "auto", blob: Optional[WeightBlob] = None,
                 max_sessions: int = 4, fold_ln: Optional[bool] = None):
        if not torch.cuda.is_available():
            raise L_.MugdError("mug_diffusion_b200 needs an sm_100 (B200) GPU; there is no CPU fallback")
        self.cfg = cfg or ModelConfig()
        self.device = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
        torch.cuda.set_device(self.device)
        self.lib = L_.load()
        self.handle = C.c_void_p()
        L_.check(self.lib.mugd_create(self.device.index or 0, C.byref(self.handle)), "mugd_create")
        self.blob = blob if blob is not None else pack_model(state_dict, self.cfg.unet, self.cfg.decoder)
        self.weights = self.blob.data.to(self.device)          # every weight once, fp32 (0.56 GB); tensor-core weights become hi in place
        self.wbase = self.weights.data_ptr()
        self.weights_lo: Optional[torch.Tensor] = None         # the lo operands of the tensor-core weights (second buffer)
        self.tc_split_done = False
        self.lock = threading.RLock()
        # split-K scratch of the tensor-core GEMM: all ops run in stream order, so one buffer serves every plan
        # (bound: tiles*splits < 2*SMs tiles of 128x128 fp32)
        self.tc_ws = torch.zeros(8 * 1024 * 1024, device=self.device)          # 32 MB
        # Compiled shapes are cached in small LRUs: webui derives z_length from each audio's duration (any multiple of
        # 32, webui.py:349-356), so an unbounded cache would grow by one ~1.5 GB arena + CUDA graph per new shape.
        self.sessions: "OrderedDict[tuple, Session]" = OrderedDict()
        self.dec_sessions: "OrderedDict[tuple, object]" = OrderedDict()
        self.max_sessions = max_sessions
        self.fold_ln = fold_ln                # LayerNorm folded into the next Linear: None = below 8192 token rows, True / False = forced
        # internal S4 kernel length per layer (SSKernelNPLR's `L` buffer, s4.py:557-584).  It is ENGINE state: lengthening
        # rewrites this engine's device copy of C~, so the length that goes with it must not live in the shared host blob.
        self.s4_L: Dict[str, int] = {k: int(v) for k, v in self.blob.meta.items() if k.endswith("kernel.kernel.L")}
        self.set_gemm_impl(gemm_impl)

    def set_gemm_impl(self, impl: str):
        # "tc_tf32" is an opt-in speed mode: single-pass TF32 tensor-core products (~2^-11 per product) instead of the
        # fp32-accurate 3xTF32 split.  Per-handle state; never used by the parity tests or bench.py.
        code = {"auto": L_.GEMM_TC, "simt": L_.GEMM_SIMT, "tc": L_.GEMM_TC, "tc_tf32": L_.GEMM_TC}[impl]
        L_.check(self.lib.mugd_set_gemm_impl(self.handle, code), "set_gemm_impl")
        if impl == "simt":
            # the exact-fp32 FFMA path needs the plain weights: restore them if this engine had already split them in place
            if self.tc_split_done:
                if self.blob.data.device.type != "cpu":
                    raise L_.MugdError("this engine's weights were split in place and no host copy exists: build a new engine for gemm_impl='simt'")
                self.weights.copy_(self.blob.data)
                self.tc_split_done = False
            self.blob.lo_bases[self.wbase] = 0
        else:
            self._split_tc_weights()
        L_.check(self.lib.mugd_set_tc_single_pass_tf32(self.handle, 1 if impl == "tc_tf32" else 0), "set_tc_single_pass_tf32")
        self.gemm_impl = impl
        self.sessions.clear()
        self.dec_sessions.clear()

    def _split_tc_weights(self):
        """TF32 hi / lo operands of every tensor-core weight, computed on the device: hi over the plain weight, lo in a second buffer"""
        shared = getattr(self.blob, "_lo_tensors", None)
        if shared is None:
            shared = self.blob._lo_tensors = {}
        if not self.tc_split_done and self.wbase in shared:
            # the blob already lives on this device (broadcast_blob over NCCL) and another engine split it in place: share its lo buffer
            self.weights_lo, self.tc_split_done = shared[self.wbase], True
        if not self.tc_split_done:
            if self.weights_lo is None:
                self.weights_lo = torch.zeros(max(self.blob.tc_lo_numel, 4), device=self.device)
            if self.weights is self.blob.data:
                shared[self.wbase] = self.weights_lo
            ops = OpList()
            for _, off, n, lo in self.blob.tc:
                d = L_.Tf32Split()
                d.w_hi, d.lo, d.n = self.wbase + 4 * off, self.weights_lo.data_ptr() + 4 * lo, n
                ops.add(L_.OP_TF32_SPLIT, d)
            st = _stream()
            for op in ops.ops:
                L_.check(self.lib.mugd_op_run(self.handle, C.byref(op), st), "tf32_split")
            self.tc_split_done = True
        self.blob.lo_bases[self.wbase] = self.weights_lo.data_ptr()

    def attach_workspace(self, ops: OpList):
        for op in ops.ops:
            if op.kind == L_.OP_GEMM:
                g = op.u.gemm
                g.workspace, g.workspace_bytes = self.tc_ws.data_ptr(), self.tc_ws.numel() * 4

    def run_ops(self, ops: OpList):
        self.attach_workspace(ops)
        st = _stream()
        for op in ops.ops:
            L_.check(self.lib.mugd_op_run(self.handle, C.byref(op), st), f"op kind {op.kind}")

    def _lru_get(self, cache: OrderedDict, key, make):
        s = cache.get(key)
        if s is None:
            while len(cache) >= max(1, self.max_sessions):
                _, old = cache.popitem(last=False)          # least recently used: frees its arena, plan and graph
                if hasattr(old, "release"):
                    old.release()
                del old
            s = make()
            cache[key] = s
        else:
            cache.move_to_end(key)
        return s

    def session(self, Beff: int, Lz: int, per_sample_t: bool = False) -> "Session":
        return self._lru_get(self.sessions, (Beff, Lz, per_sample_t), lambda: Session(self, Beff, Lz, per_sample_t))

    def wave_session(self, B: int, T: int):
        """Audio encoder plan for B mel-spectrograms of T frames (SURVEY §8f N1); needs wave weights in the blob."""
        if "wave_cfg" not in self.blob.meta:
            raise L_.MugdError("this engine was packed without model.wave_model.* weights")
        from .wave import WaveSession
        return self._lru_get(self.dec_sessions, ("wave", B, T), lambda: WaveSession(self, B, T))

    def decoder_session(self, B: int, Lz: int) -> "DecoderSession":
        return self._lru_get(self.dec_sessions, (B, Lz), lambda: DecoderSession(self, B, Lz))

    def __del__(self):
        try:
            self.sessions.clear()
            self.dec_sessions.clear()
            if self.handle:
                self.lib.mugd_destroy(self.handle)
        except Exception:
            pass


class Session:
    """Compiled U-Net evaluation for Beff samples of length Lz (Beff = 2B under classifier-free guidance)."""

    def __init__(self, engine: MugEngine, Beff: int, Lz: int, per_sample_t: bool):
        self.engine, self.Beff, self.Lz, self.per_sample_t = engine, Beff, Lz, per_sample_t
        cfg = engine.cfg.unet
        dev = engine.device
        comp = UNetCompiler(cfg, engine.blob, engine.wbase)
        self.comp = comp
        emb_total = engine.blob.meta["emb_total"]
        n_attn = sum(1 for b in _all_blocks(comp) if b.kind == "attn")
        attn_blocks = [b for b in _all_blocks(comp) if b.kind == "attn"]
        s4b = [b for b in _all_blocks(comp) if b.kind == "s4"]

        # ---- side buffers (owned torch tensors) ----------------------------------------------
        emb_rows = Beff if per_sample_t else MAX_STEPS
        self.emb_table = torch.zeros(emb_rows, emb_total, device=dev)
        self.temb = torch.zeros(emb_rows, cfg.model_channels, device=dev)
        self.emb_h1 = torch.zeros(emb_rows, cfg.time_embed_dim, device=dev)
        self.emb_h2 = torch.zeros(emb_rows, cfg.time_embed_dim, device=dev)
        self.step = torch.zeros(1, dtype=torch.int32, device=dev)
        self.coef = torch.zeros(MAX_STEPS, 4, device=dev)
        self.ctx = torch.zeros(Beff * CTX_TOKENS_MAX, cfg.context_dim, device=dev)
        self.ctx_kv = [torch.zeros(Beff * CTX_TOKENS_MAX, 2 * b.cin, device=dev) for b in attn_blocks]
        self.ctx_tokens = 21
        self.s4_kt = {b.prefix: torch.zeros(Lz // b.ds, b.cin, device=dev) for b in s4b}
        self._gen_s4_kernels(s4b)
        self._build(comp)

    # S4 convolution kernels for this length: SSKernelNPLR.forward once per (model, L)  (s4.py:706-832)
    def _gen_s4_kernels(self, s4b):
        eng = self.engine
        N = eng.cfg.unet.s4_state // 2
        ws = None
        for b in s4b:
            k = b.prefix + "s4_model.kernel.kernel."
            L_int = int(eng.s4_L[k + "L"])
            L_req = self.Lz // b.ds
            if L_req > L_int:
                # same one-time, persistent mutation the reference performs in SSKernelNPLR._setup_C (s4.py:557-584):
                # lengthen C~ on the host, store it back into the weight blob and remember the new internal length
                from . import s4_setup

                def grab(n):
                    e = eng.blob.entries[k + n]
                    cnt = int(np.prod(e.shape))
                    return eng.weights[e.offset:e.offset + cnt].view(e.shape).detach().cpu()

                params = {n: grab(n) for n in ("C", "log_dt", "P", "inv_w_real", "w_imag")}
                C_new, L_int = s4_setup.lengthen(params, L_int, L_req)
                e = eng.blob.entries[k + "C"]
                eng.weights[e.offset:e.offset + C_new.numel()].copy_(C_new.reshape(-1).to(eng.device))
                eng.s4_L[k + "L"] = L_int
            need = 16 * b.cin * (L_int // 2 + 1)
            if ws is None or ws.numel() * 8 < need:
                ws = torch.empty(need // 8 + 2, dtype=torch.float64, device=eng.device)

            def w(n):
                return eng.wbase + 4 * eng.blob.offset(k + n)

            om = s4_fft_nodes(L_int).to(eng.device)
            L_.check(eng.lib.mugd_s4_kernel_gen(eng.handle, w("log_dt"), w("B"), w("C"), w("P"), w("inv_w_real"), w("w_imag"),
                                                _ptr(om), b.cin, N, L_int, L_req, _ptr(self.s4_kt[b.prefix]), _ptr(ws), ws.numel() * 8,
                                                _stream()), "s4_kernel_gen")
        torch.cuda.current_stream().synchronize()

    def _ext(self, base_ctx_tokens: int) -> dict:
        return dict(
            emb_table=_ptr(self.emb_table), step=_ptr(self.step), ctx_tokens=base_ctx_tokens,
            ctx_kv=[View(_ptr(t), t.shape[1], self.Beff * base_ctx_tokens, t.shape[1]) for t in self.ctx_kv],
            s4_kt={p: View(_ptr(t), t.shape[1], t.shape[0], t.shape[1]) for p, t in self.s4_kt.items()},
        )

    def _build(self, comp: UNetCompiler):
        # the LayerNorm fold lives in the tensor-core GEMM epilogues; the exact-fp32 FFMA path keeps the stand-alone LayerNorm
        # kernels and doubles as the referee of the folded plan.  engine.fold_ln: None = by size, True / False = forced (A/B, tests)
        fold = False if self.engine.gemm_impl == "simt" else self.engine.fold_ln
        dry = Arena(0)
        comp.compile(dry, self.Beff, self.Lz, self._ext(self.ctx_tokens), self.per_sample_t, fold)
        nbytes = dry.high + 1024
        self.arena_t = torch.zeros(nbytes // 4 + 64, device=self.engine.device)
        base = (self.arena_t.data_ptr() + 255) // 256 * 256
        arena = Arena(base, nbytes)
        res = comp.compile(arena, self.Beff, self.Lz, self._ext(self.ctx_tokens), self.per_sample_t, fold)
        self.xin: View = res["xin"]
        self.eps: View = res["eps"]
        self.audio_slots = res["audio_slots"]
        self.ln_folded = res["ln_folded"]
        self.plan = Plan(self.engine, res["ops"])
        self.arena_bytes = nbytes
        self._captured_for = None

    # ---- per-request preparation ---------------------------------------------------------------
    def set_timestep_table(self, timesteps: Sequence[int]):
        """Time-embedding MLP + all ResBlock emb projections for the given timesteps, one row each
        (unet.py:335-339, 166-172; model/util.py:156-176).  The sinusoid is evaluated on the host exactly
        as the reference does; the three GEMMs run on the GPU."""
        cfg = self.engine.cfg.unet
        eng = self.engine
        t = torch.as_tensor(np.asarray(timesteps), dtype=torch.long)
        R = t.shape[0]
        assert R <= self.temb.shape[0]
        half = cfg.model_channels // 2
        import math
        freqs = torch.exp(-math.log(10000.0) * torch.arange(0, half, dtype=torch.float32) / half)
        args = t[:, None].float() * freqs[None]
        emb = torch.cat([torch.cos(args), torch.sin(args)], dim=-1)
        self.temb[:R].copy_(emb.to(eng.device))
        eng.run_ops(self.timestep_ops(R))

    def timestep_ops(self, R: int) -> OpList:
        """the three GEMMs that turn R sinusoid rows (self.temb) into R rows of the fused ResBlock embedding table"""
        cfg = self.engine.cfg.unet
        eng = self.engine
        ops = OpList(tc_weight_map(eng.blob, eng.wbase))
        up = self.comp.prefix
        tv = View(_ptr(self.temb), cfg.model_channels, R, cfg.model_channels)
        h1 = View(_ptr(self.emb_h1), cfg.time_embed_dim, R, cfg.time_embed_dim)
        h2 = View(_ptr(self.emb_h2), cfg.time_embed_dim, R, cfg.time_embed_dim)
        et = View(_ptr(self.emb_table), self.emb_table.shape[1], R, self.emb_table.shape[1])
        w = self.comp.w
        ops.gemm(tv, w(up + "time_embed.0.weight"), cfg.time_embed_dim, cfg.model_channels, h1, bias=w(up + "time_embed.0.bias"),
                 act=L_.ACT_SILU)
        # emb is only ever consumed through emb_layers = SiLU -> Linear, so SiLU(emb) is stored
        ops.gemm(h1, w(up + "time_embed.2.weight"), cfg.time_embed_dim, cfg.time_embed_dim, h2, bias=w(up + "time_embed.2.bias"),
                 act=L_.ACT_SILU)
        ops.gemm(h2, w(up + "emb_all.weight"), self.emb_table.shape[1], cfg.time_embed_dim, et, bias=w(up + "emb_all.bias"))
        return ops

    def set_context(self, context):
        """context [Beff, ctx_dim, T] (reference layout; or a list of such tensors that follow each other along the batch, e.g.
        [uc, c] under classifier-free guidance, ddim.py:173) -> per-layer cross-attention K|V projections (attention.py:97-98),
        constant over the DDIM steps."""
        eng = self.engine
        cfg = eng.cfg.unet
        parts = list(context) if isinstance(context, (list, tuple)) else [context]
        parts = [c.to(eng.device, torch.float32).contiguous() for c in parts]
        Bc = sum(int(c.shape[0]) for c in parts)
        _, Cd, T = parts[0].shape
        assert Bc == self.Beff and Cd == cfg.context_dim and T <= CTX_TOKENS_MAX and all(c.shape[1:] == parts[0].shape[1:] for c in parts)
        if T != self.ctx_tokens:
            self.ctx_tokens = T
            self._build(self.comp)            # Lk is baked into the attention ops
        eng.run_ops(self.context_ops([(_ptr(c), int(c.shape[0])) for c in parts], T))
        self._keep = parts

    def context_ops(self, parts: Sequence, T: int) -> OpList:
        """parts: (device address of a [b, ctx_dim, T] tensor, b) in batch order -> transposes + the 16 K|V projections"""
        eng = self.engine
        cfg = eng.cfg.unet
        Cd = cfg.context_dim
        Bc = sum(b for _, b in parts)
        ops = OpList(tc_weight_map(eng.blob, eng.wbase))
        row = 0
        for addr, bpart in parts:
            ops.transpose(addr, _ptr(self.ctx) + 4 * row * Cd, 0, Cd, bpart, Cd, T, True)
            row += bpart * T
        cv = View(_ptr(self.ctx), Cd, Bc * T, Cd)
        blocks = [b for b in _all_blocks(self.comp) if b.kind == "attn"]
        for b, kv in zip(blocks, self.ctx_kv):
            o = View(_ptr(kv), kv.shape[1], Bc * T, kv.shape[1])
            ops.gemm(cv, self.comp.w(b.prefix + "transformer_blocks.0.attn2.kv.weight"), 2 * b.cin, Cd, o, Lout=T)
        return ops

    def set_audio(self, audios: Sequence[torch.Tensor], dup: bool = False):
        """The last ``levels`` entries of the wave-encoder output list (unet.py:527-543), NCL layout, written
        (transposed) into every concat slot that holds them.  ``dup``: the tensors hold Beff/2 samples and both halves of the
        batch get them (the reference concatenates them with themselves under classifier-free guidance, ddim.py:171-174)."""
        cfg = self.engine.cfg.unet
        w4 = [a.to(self.engine.device, torch.float32).contiguous() for a in list(audios)[-cfg.levels:]]
        Bh = self.Beff // 2 if dup else self.Beff
        for lvl in range(cfg.levels):
            assert w4[lvl].shape == (Bh, cfg.audio_channels[lvl], self.Lz >> lvl), (w4[lvl].shape, lvl)
        self.engine.run_ops(self.audio_ops([_ptr(a) for a in w4], dup))
        self._keep_audio = w4

    def audio_ops(self, addrs: Sequence[int], dup: bool) -> OpList:
        """addrs[lvl] = device address of the [Beff (or Beff/2 when dup), C_lvl, L_lvl] audio feature map of level lvl"""
        cfg = self.engine.cfg.unet
        Bh = self.Beff // 2 if dup else self.Beff
        ops = OpList()
        for lvl, view in self.audio_slots:
            Cc, Lr = cfg.audio_channels[lvl], self.Lz >> lvl
            ops.transpose(addrs[lvl], view.ptr, 0, view.ld, Bh, Cc, Lr, True)
            if dup:
                ops.transpose(addrs[lvl], view.r(Bh * Lr, 2 * Bh * Lr).ptr, 0, view.ld, Bh, Cc, Lr, True)
        return ops

    def load_x(self, x: torch.Tensor, dup: bool):
        """x [B,C,L] -> xin rows (both halves when dup)."""
        x = x.to(self.engine.device, torch.float32).contiguous()
        B, Cc, Lr = x.shape
        self.engine.run_ops(self.loadx_ops(_ptr(x), B, dup))
        self._keep_x = x

    def loadx_ops(self, addr: int, B: int, dup: bool) -> OpList:
        Cc, Lr = self.engine.cfg.unet.in_channels, self.Lz
        ops = OpList()
        ops.transpose(addr, self.xin.ptr, 0, self.xin.ld, B, Cc, Lr, True)
        if dup:
            ops.transpose(addr, self.xin.r(B * Lr, 2 * B * Lr).ptr, 0, self.xin.ld, B, Cc, Lr, True)
        return ops

    def read_rows(self, view: View, B: int, Cc: int, Lr: int) -> torch.Tensor:
        out = torch.empty(B, Cc, Lr, device=self.engine.device)
        ops = OpList()
        ops.transpose(view.ptr, _ptr(out), view.ld, 0, B, Cc, Lr, False)
        self.engine.run_ops(ops)
        return out

    def eval(self, graph: bool = True):
        if graph:
            if not self.plan.captured:
                self.plan.run()               # warm-up (lazy module load) outside capture
                self.plan.capture()
            self.plan.replay(1)
        else:
            self.plan.run()

    def run_steps(self, n: int, tail: OpList):
        """n DDIM steps from ONE C call (mugd_sample): n x {graph replay of the evaluation ; the tail ops (update, step advance)}"""
        if not self.plan.captured:
            self.plan.run()                   # warm-up (lazy module load) outside capture
            self.plan.capture()
        self.engine.attach_workspace(tail)
        arr = tail.array()
        L_.check(self.engine.lib.mugd_sample(self.plan.handle, arr, len(tail.ops), n, _stream()), "mugd_sample")

    def set_step(self, value: int):
        L_.check(self.engine.lib.mugd_fill_i32(_ptr(self.step), value, _stream()), "fill_i32")


class DecoderSession:
    def __init__(self, engine: MugEngine, B: int, Lz: int):
        self.engine, self.B, self.Lz = engine, B, Lz
        comp = DecoderCompiler(engine.cfg.decoder, engine.blob, engine.wbase)
        dry = Arena(0)
        comp.compile(dry, B, Lz)
        nbytes = dry.high + 1024
        self.arena_t = torch.zeros(nbytes // 4 + 64, device=engine.device)
        base = (self.arena_t.data_ptr() + 255) // 256 * 256
        res = comp.compile(Arena(base, nbytes), B, Lz)
        self.zin, self.logits, self.Lout = res["zin"], res["logits"], res["Lout"]
        self.plan = Plan(engine, res["ops"])
        self.arena_bytes = nbytes

    def notes(self, frame_ms: float, key_count: int = 4):
        """Note extraction on the logits of the last ``decode`` (still resident, channels-last): returns
        (count [B,K], start_ms [B,K,T], end_ms [B,K,T]) as CPU int32 tensors; only count and the used prefixes matter."""
        eng = self.engine
        B, T, K = self.B, self.Lout, key_count
        assert 4 * K == eng.cfg.decoder.x_channels
        cnt = torch.zeros(B, K, dtype=torch.int32, device=eng.device)
        st = torch.full((B, K, T), -1, dtype=torch.int32, device=eng.device)
        en = torch.full((B, K, T), -1, dtype=torch.int32, device=eng.device)
        d = L_.Notes()
        d.logits, d.ld = self.logits.ptr, self.logits.ld
        d.count, d.start_ms, d.end_ms = _ptr(cnt), _ptr(st), _ptr(en)
        d.frame_ms, d.B, d.T, d.K = float(frame_ms), B, T, K
        ops = OpList()
        ops.add(L_.OP_NOTES, d)
        eng.run_ops(ops)
        cnt_c = cnt.cpu()
        nmax = int(cnt_c.max()) if cnt_c.numel() else 0
        return cnt_c, st[:, :, :max(nmax, 1)].cpu(), en[:, :, :max(nmax, 1)].cpu()

    def decode(self, z: torch.Tensor) -> torch.Tensor:
        eng = self.engine
        cfg = eng.cfg.decoder
        z = z.to(eng.device, torch.float32)
        if cfg.scale != 1.0:
            z = z / cfg.scale                 # autoencoder.py:76
        z = z.contiguous()
        ops = OpList()
        ops.transpose(_ptr(z), self.zin.ptr, 0, self.zin.ld, self.B, cfg.z_channels, self.Lz, True)
        eng.run_ops(ops)
        if not self.plan.captured:
            self.plan.run()                   # warm-up (lazy module load) outside capture
            self.plan.capture()
        self.plan.replay(1)
        out = torch.empty(self.B, cfg.x_channels, self.Lout, device=eng.device)
        ops = OpList()
        ops.transpose(self.logits.ptr, _ptr(out), self.logits.ld, 0, self.B, cfg.x_channels, self.Lout, False)
        eng.run_ops(ops)
        return out


_NODE_CACHE: Dict[int, torch.Tensor] = {}


def s4_fft_nodes(L_int: int) -> torch.Tensor:
    """omega_f for f = 0..L/2 evaluated the way the reference does (SSKernelNPLR._omega, s4.py:586-604):
    a complex64 base raised to integer powers on the host.  This is a parameter-free constant table like the
    timestep sinusoid; feeding the same nodes to the fp64 kernel generator reproduces the reference's kernel
    to ~2e-6 instead of ~1e-4 (the complex64 power drifts by up to 5e-6 at f = L/2).  Returns [L/2+1, 2] fp32."""
    t = _NODE_CACHE.get(L_int)
    if t is None:
        base = torch.tensor(np.exp(-2j * np.pi / L_int), dtype=torch.complex64)
        t = torch.view_as_real(base ** torch.arange(0, L_int // 2 + 1)).contiguous()
        _NODE_CACHE[L_int] = t
    return t


def hit_object_lines(count, start_ms, end_ms, key_count: int):
    """Per chart: the .osu hit-object lines of OsuManiaConvertor.array_to_objects (convertor.py:257-264) from the
    compact (column, frame-ordered) note lists the GPU produced; sorted by start time with a stable sort, like the reference."""
    width = int(512 / key_count)
    charts = []
    for b in range(count.shape[0]):
        items = []
        for col in range(key_count):
            n = int(count[b, col])
            x = int(round((col + 0.5) * width))
            for s_, e_ in zip(start_ms[b, col, :n].tolist(), end_ms[b, col, :n].tolist()):
                line = f"{x},192,{s_},1,0,0:0:0:0:" if e_ == -1 else f"{x},192,{s_},128,0,{e_}:0:0:0:0:"
                items.append((line, s_))
        items.sort(key=lambda t: t[1])
        charts.append([t[0] for t in items])
    return charts


def _all_blocks(comp: UNetCompiler):
    lay = comp.lay
    for entry in lay.input + [lay.middle] + lay.output:
        if isinstance(entry, tuple):
            continue
        for b in entry:
            yield b

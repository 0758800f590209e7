"""Launch-plan compiler and runtime of the B200 sampler.

``MugEngine`` owns a libmugd handle and the packed weight blob on one GPU.  ``Session`` is the compiled
state for one (effective batch, z_length): an activation arena, the S4 convolution kernels for that
length, the U-Net launch plan captured as a CUDA graph and the decoder plan.  All device memory is torch
storage; libmugd only ever sees raw pointers (include/mugd.h).

Data layout: channels-last ``[B*L, C]`` fp32 with a leading dimension.  Every ``torch.cat`` of the
reference U-Net (AudioConcatBlock unet.py:114-118, skip concat unet.py:545) is a column range of a wider
buffer that producers write into directly, so no concat copy runs per step except the four per-level
tensors that belong to two concat buffers at once.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import lib as L_
from .config import DecoderConfig, ModelConfig, UNetConfig
from .netspec import Block, decoder_layout, unet_layout
from .packer import WeightBlob, pack_model

GN_EPS = 1e-6     # models.py:11
LN_EPS = 1e-5     # nn.LayerNorm default, attention.py:136-138
MAX_STEPS = 1000
CTX_TOKENS_MAX = 64


@dataclass
class View:
    """rows x cols window of a row-major fp32 buffer."""
    ptr: int      # device address in bytes
    ld: int       # leading dimension in floats
    rows: int
    cols: int

    def c(self, c0: int, c1: int) -> "View":
        assert 0 <= c0 < c1 <= self.cols, (c0, c1, self.cols)
        return View(self.ptr + 4 * c0, self.ld, self.rows, c1 - c0)

    def r(self, r0: int, r1: int) -> "View":
        assert 0 <= r0 < r1 <= self.rows
        return View(self.ptr + 4 * r0 * self.ld, self.ld, r1 - r0, self.cols)


class Arena:
    """Bump allocator over one torch buffer.  ``mark``/``release`` give stack-scoped scratch so the
    temporaries of every block reuse the same (L2-resident) addresses."""

    def __init__(self, base: int = 0, capacity: Optional[int] = None):
        self.base = base
        self.capacity = capacity
        self.top = 0
        self.high = 0

    def alloc(self, rows: int, cols: int) -> View:
        n = rows * cols * 4
        start = (self.top + 255) // 256 * 256
        self.top = start + n
        self.high = max(self.high, self.top)
        if self.capacity is not None:
            assert self.top <= self.capacity, "arena overflow"
        return View(self.base + start, cols, rows, cols)

    def mark(self) -> int:
        return self.top

    def release(self, mark: int):
        self.top = mark


class OpList:
    def __init__(self, tc_map: Optional[Dict[int, Tuple[int, int]]] = None):
        self.ops: List[L_.Op] = []
        self.tc_map = tc_map or {}         # W pointer -> (W_hi, W_lo) pointers of the TF32 split

    def add(self, kind: int, desc, tag: int = 0):
        self.ops.append(L_.make_op(kind, desc, tag))

    def array(self):
        arr = (L_.Op * len(self.ops))(*self.ops)
        return arr

    # ---- op constructors ---------------------------------------------------------------------
    def gemm(self, A: View, W: int, N: int, K: int, out: View, *, bias: int = 0, taps: int = 1,
             mode: int = L_.CONV_NONE, Lin: int = 0, Lout: int = 0, act: int = L_.ACT_NONE,
             gate: int = L_.GATE_NONE, residual: Optional[View] = None, rowvec: int = 0,
             rowvec_b_stride: int = 0, rowvec_step_stride: int = 0, step: int = 0, impl: int = L_.GEMM_AUTO,
             W_hi: int = 0, W_lo: int = 0, split_k: int = 0, tc_variant: int = L_.TC_AUTO, tap_shift: int = 0, dilation: int = 1,
             tag: int = 0, A2: Optional[View] = None, ln: Optional[Tuple[int, int, float]] = None) -> int:
        g = L_.Gemm()
        M = out.rows
        g.A, g.lda = A.ptr, A.ld
        if not W_hi and W in self.tc_map:
            W_hi, W_lo = self.tc_map[W]
        g.W, g.W_hi, g.W_lo, g.bias = W, W_hi or None, W_lo or None, bias or None
        g.split_k, g.tc_variant = split_k, tc_variant
        g.tap_shift = tap_shift
        g.tap_dilation = dilation
        g.rowvec, g.rowvec_b_stride, g.rowvec_step_stride = rowvec or None, rowvec_b_stride, rowvec_step_stride
        g.step = step or None
        if residual is not None:
            g.residual, g.ldr = residual.ptr, residual.ld
        if A2 is not None:                     # second activation source: K2 more channels at the output row (1x1 term)
            assert A2.rows == out.rows, (A2.rows, out.rows)
            g.A2, g.lda2, g.K2 = A2.ptr, A2.ld, A2.cols
        g.C, g.ldc = out.ptr, out.ld
        g.M, g.N, g.K = M, N, K
        g.taps, g.conv_mode = taps, mode
        g.Lout = Lout or M
        g.Lin = Lin or g.Lout
        g.act, g.gate, g.impl = act, gate, impl
        if ln is not None:                     # LayerNorm folded in: (row moments of A, column sums of the gamma-scaled weight, eps)
            g.ln_stats, g.ln_colsum, g.ln_eps = ln[0], ln[1], float(ln[2])
        nout = N // 2 if gate else N
        assert out.cols == nout, (out.cols, nout)
        assert A.cols == K, (A.cols, K)
        self.add(L_.OP_GEMM, g, tag)
        return len(self.ops) - 1

    def can_deliver_row_moments(self, i: int) -> bool:
        """can GEMM op i also accumulate the row moments of its output?  (tensor-core path with a plain epilogue)"""
        op = self.ops[i]
        if op.kind != L_.OP_GEMM:
            return False
        g = op.u.gemm
        tc = bool(g.W_hi) and g.K % 32 == 0 and g.K2 % 32 == 0 and g.N >= 16 and g.impl != L_.GEMM_SIMT and g.conv_mode != L_.CONV_UP
        return tc and g.act == L_.ACT_NONE and g.gate == L_.GATE_NONE and not g.ln_stats and not g.row_moments

    def groupnorm(self, x: View, y: View, gamma: int, beta: int, B: int, Lrows: int, G: int, silu: bool, tag: int = 0) -> int:
        d = L_.GroupNorm()
        d.x, d.ldx, d.y, d.ldy = x.ptr, x.ld, y.ptr, y.ld
        d.gamma, d.beta = gamma, beta
        d.B, d.L, d.C, d.G = B, Lrows, x.cols, G
        d.eps, d.silu = GN_EPS, int(silu)
        assert x.rows == B * Lrows and y.cols == x.cols
        self.add(L_.OP_GROUPNORM, d, tag)
        return len(self.ops) - 1

    def layernorm(self, x: View, y: View, gamma: int, beta: int, tag: int = 0):
        d = L_.LayerNorm()
        d.x, d.ldx, d.y, d.ldy = x.ptr, x.ld, y.ptr, y.ld
        d.gamma, d.beta = gamma, beta
        d.rows, d.C, d.eps = x.rows, x.cols, LN_EPS
        self.add(L_.OP_LAYERNORM, d, tag)
        return len(self.ops) - 1

    def attention(self, q: View, k: View, v: View, o: View, relpos: int, cgain: int, B: int, H: int, Lq: int,
                  Lk: int, pos_max: int, tag: int = 0):
        d = L_.Attention()
        D = q.cols // H
        d.q, d.ldq, d.k, d.ldk, d.v, d.ldv, d.o, d.ldo = q.ptr, q.ld, k.ptr, k.ld, v.ptr, v.ld, o.ptr, o.ld
        d.relpos, d.cgain = relpos, cgain
        d.B, d.H, d.D, d.Lq, d.Lk, d.pos_max = B, H, D, Lq, Lk, pos_max
        d.scale = float(D) ** -0.5
        self.add(L_.OP_ATTENTION, d, tag)

    def s4conv(self, u: View, Kt: int, Dp: int, y: View, B: int, Lrows: int, tag: int = 0):
        d = L_.S4Conv()
        d.u, d.ldu, d.Kt, d.D, d.y, d.ldy = u.ptr, u.ld, Kt, Dp, y.ptr, y.ld
        d.B, d.L, d.H = B, Lrows, u.cols
        self.add(L_.OP_S4CONV, d, tag)

    def transpose(self, inp: int, out: int, ldi: int, ldo: int, B: int, Cc: int, Lrows: int, to_nlc: bool, tag: int = 0):
        d = L_.Transpose()
        d.inp, d.out, d.ldi, d.ldo = inp, out, ldi, ldo
        d.B, d.C, d.L, d.to_nlc = B, Cc, Lrows, int(to_nlc)
        self.add(L_.OP_TRANSPOSE, d, tag)

    def copy2d(self, src: View, dst: View, tag: int = 0):
        d = L_.Copy2D()
        assert src.rows == dst.rows and src.cols == dst.cols
        d.src, d.lds, d.dst, d.ldd, d.rows, d.cols = src.ptr, src.ld, dst.ptr, dst.ld, src.rows, src.cols
        self.add(L_.OP_COPY2D, d, tag)


def emit_upsample_conv(ops: "OpList", blob: WeightBlob, wfn, prefix: str, x: View, out: View, Lin: int, cin: int, cout: int, tag: int):
    """Upsample (nearest x2) + conv3 (models.py:66-70).  With the parity-split weights of the packer this is two 2-tap
    GEMMs over the Lin input rows writing the even / odd output rows (row stride 2*ld) -- 2/3 of the FLOPs of the
    literal form and eligible for the tensor-core kernel; otherwise the generic MUGD_CONV_UP addressing is used."""
    idx = []
    if (prefix + "conv.up_even.weight") in blob.entries:
        for parity, name, shift in ((0, "conv.up_even.weight", -1), (1, "conv.up_odd.weight", 0)):
            dst = View(out.ptr + 4 * parity * out.ld, 2 * out.ld, x.rows, out.cols)
            idx.append(ops.gemm(x, wfn(prefix + name), cout, cin, dst, bias=wfn(prefix + "conv.bias"), taps=2, mode=L_.CONV_TAPS,
                                Lin=Lin, Lout=Lin, tap_shift=shift, tag=tag))
    else:
        idx.append(ops.gemm(x, wfn(prefix + "conv.weight"), cout, cin, out, bias=wfn(prefix + "conv.bias"), taps=3, mode=L_.CONV_UP,
                            Lin=Lin, Lout=2 * Lin, tag=tag))
    return idx


def tc_weight_map(blob: WeightBlob, wbase: int) -> Dict[int, Tuple[int, int]]:
    """address of every tensor-core GEMM weight -> (hi address, lo address).  After the engine's device-side split (runtime.MugEngine)
    hi lives where the plain weight was and lo in the engine's second buffer (``blob.lo_bases[wbase]``; 0 = this engine keeps plain
    fp32 weights for the exact-fp32 FFMA path: empty map).  A base nobody registered (plan compilation without a device, CPU tests)
    gets a virtual lo buffer behind the blob."""
    lo_base = blob.lo_bases.get(wbase, wbase + 4 * blob.numel)
    if lo_base == 0:
        return {}
    cached = getattr(blob, "_tc_maps", None)
    if cached is None:
        cached = blob._tc_maps = {}
    key = (wbase, lo_base)
    if key not in cached:
        cached[key] = {wbase + 4 * off: (wbase + 4 * off, lo_base + 4 * lo) for _, off, _, lo in blob.tc}
    return cached[key]


# tags (profiling labels carried in mugd_op.tag)
TAG_RES, TAG_ATTN, TAG_S4, TAG_UPDOWN, TAG_IO = 1, 2, 3, 4, 5


class UNetCompiler:
    """Emit the op list of one U-Net evaluation (unet.py:511-550) for Beff samples of length L."""

    def __init__(self, cfg: UNetConfig, blob: WeightBlob, wbase: int, prefix: str = "model.unet_model."):
        self.cfg, self.blob, self.wbase, self.prefix = cfg, blob, wbase, prefix
        self.lay = unet_layout(cfg, prefix)

    def w(self, name: str) -> int:
        return self.wbase + 4 * self.blob.offset(name)

    def compile(self, arena: Arena, Beff: int, Lz: int, ext: Dict[str, int], per_sample_t: bool, fold_ln: Optional[bool] = None) -> dict:
        """fold_ln: every LayerNorm of the transformer blocks is folded into the Linear behind it (the producer of its input delivers
        the row moments, the Linear corrects in its epilogue; no LayerNorm kernel, the normalised tensor is never written).  Worth
        1.2 % at Beff = 8 and -0.8 % at Beff = 64 (profiles/r02_norm_fusion_ab.md), so None = fold below 8192 token rows.
        False = stand-alone LayerNorm kernels (the referee path, and what the exact-fp32 FFMA GEMM uses)."""
        cfg = self.cfg
        ops = OpList(tc_weight_map(self.blob, self.wbase))
        nlev = cfg.levels
        assert Lz % (1 << (nlev - 1)) == 0 and (Lz >> (nlev - 1)) % 4 == 0, "z_length must be a multiple of 32"
        rows = [Beff * (Lz >> l) for l in range(nlev)]
        lens = [Lz >> l for l in range(nlev)]
        mc = cfg.model_channels
        G = cfg.gn_groups
        if fold_ln is None:
            fold_ln = rows[0] < 8192
        fuse_ln = fold_ln and any(k.endswith("qkv_ln.weight") for k in self.blob.entries)

        # ---- row-moment block: [live | zeros] fp64, `live` re-armed by the first op of every evaluation ----
        all_blocks = [b for e in self.lay.input + [self.lay.middle] + self.lay.output if not isinstance(e, tuple) for b in e]
        lvl_of_ds = {1 << l: l for l in range(nlev)}
        ln_rows = sum(3 * rows[lvl_of_ds[b.ds]] for b in all_blocks if b.kind == "attn")
        stat_doubles = ln_rows * 2 if fuse_ln else 0
        stat_floats = (2 * stat_doubles + 63) // 64 * 64
        live = arena.alloc(1, stat_floats) if fuse_ln else None
        zeros = arena.alloc(1, stat_floats) if fuse_ln else None          # never written: the arena starts zeroed
        stat_top = [0]                        # doubles handed out

        def stat_alloc(n_doubles: int) -> int:
            o = stat_top[0]
            stat_top[0] += (n_doubles + 1) // 2 * 2
            assert stat_top[0] <= stat_doubles, "row-moment block overflow"
            return live.ptr + 8 * o

        if fuse_ln:
            ops.copy2d(zeros, live, TAG_IO)

        # ---- persistent buffers --------------------------------------------------------------
        xin = arena.alloc(rows[0], cfg.in_channels)
        eps = arena.alloc(rows[0], cfg.out_channels)
        ctx_tokens = ext["ctx_tokens"]
        # down-path concat buffers [h | audio_l]
        down_cat = []
        ch = mc
        ch_in_level = []
        for l in range(nlev):
            ch_in_level.append(ch)
            down_cat.append(arena.alloc(rows[l], ch + cfg.audio_channels[l]))
            ch = cfg.channel_mult[l] * mc
        # up-path concat buffers, one per output block: [h | audio (first block of a level) | skip]
        up_blocks = [e for e in self.lay.output if not isinstance(e, tuple)]
        up_cat: List[View] = []
        up_parts: List[Tuple[int, int, int]] = []     # (ch_h, ch_audio, ch_skip)
        skip_ch = list(self.lay.skip_channels)
        ch = cfg.channel_mult[-1] * mc
        bi = 0
        for level in reversed(range(nlev)):
            for i in range(cfg.num_res_blocks + 1):
                ich = skip_ch.pop()
                ca = cfg.audio_channels[level] if i == 0 else 0
                up_cat.append(arena.alloc(rows[level], ch + ca + ich))
                up_parts.append((ch, ca, ich))
                assert up_blocks[bi][0].cin == ch + ca + ich, (up_blocks[bi][0].cin, ch, ca, ich)
                ch = cfg.channel_mult[level] * mc
                bi += 1
        # home of every skip tensor = skip slice of the up block that pops it (LIFO)
        n_skips = len(self.lay.skip_channels)
        skip_home: List[View] = [None] * n_skips
        for k in range(n_skips):           # k-th pushed is popped by up block (n_skips-1-k)
            ub = n_skips - 1 - k
            ch_h, ca, ich = up_parts[ub]
            assert ich == self.lay.skip_channels[k]
            skip_home[k] = up_cat[ub].c(ch_h + ca, ch_h + ca + ich)
        audio_slots: List[Tuple[int, View]] = []       # (level, view) every place audio_l must be written
        for l in range(nlev):
            audio_slots.append((l, down_cat[l].c(ch_in_level[l], ch_in_level[l] + cfg.audio_channels[l])))
        bi = 0
        for level in reversed(range(nlev)):
            ch_h, ca, ich = up_parts[bi]
            audio_slots.append((level, up_cat[bi].c(ch_h, ch_h + ca)))
            bi += cfg.num_res_blocks + 1

        emb_total = self.blob.meta["emb_total"]
        emb_off = self.blob.meta["emb_offsets"]
        E = ext["emb_table"]
        step = ext["step"]

        gemm = ops.gemm

        def copy(src: View, dst: View, tag: int):
            ops.copy2d(src, dst, tag)

        def groupnorm(x: View, y: View, gamma: int, beta: int, Lr: int, silu: bool, tag: int):
            ops.groupnorm(x, y, gamma, beta, Beff, Lr, G, silu, tag)

        # ---- block emitters ------------------------------------------------------------------
        def emit_res(b: Block, x: View, out: View, lvl: int):
            Lr = lens[lvl]
            m = arena.mark()
            p = b.prefix
            t1 = arena.alloc(x.rows, b.cin)
            groupnorm(x, t1, self.w(p + "in_layers.0.weight"), self.w(p + "in_layers.0.bias"), Lr, True, TAG_RES)
            t2 = arena.alloc(x.rows, b.cout)
            gemm(t1, self.w(p + "in_layers.2.weight"), b.cout, b.cin, t2, bias=self.w(p + "in_layers.2.bias"), taps=3,
                 mode=L_.CONV_SAME, Lin=Lr, Lout=Lr, rowvec=E + 4 * emb_off[p],
                 rowvec_b_stride=emb_total if per_sample_t else 0,
                 rowvec_step_stride=0 if per_sample_t else emb_total, step=0 if per_sample_t else step, tag=TAG_RES)
            t3 = arena.alloc(x.rows, b.cout)
            groupnorm(t2, t3, self.w(p + "out_layers.0.weight"), self.w(p + "out_layers.0.bias"), Lr, True, TAG_RES)
            if b.has_skip_conv:
                # conv3(t3) + skip_connection(x) as ONE GEMM: the 1x1 skip runs as extra k-steps on a second source
                gemm(t3, self.w(p + "out_skip.weight"), b.cout, b.cout, out, bias=self.w(p + "out_skip.bias"), taps=3,
                     mode=L_.CONV_SAME, Lin=Lr, Lout=Lr, A2=x, tag=TAG_RES)
            else:
                gemm(t3, self.w(p + "out_layers.3.weight"), b.cout, b.cout, out, bias=self.w(p + "out_layers.3.bias"), taps=3,
                     mode=L_.CONV_SAME, Lin=Lr, Lout=Lr, residual=x, tag=TAG_RES)
            arena.release(m)

        attn_index = [0]

        def emit_attn(b: Block, x: View, out: View, lvl: int):
            Lr, Cc, H = lens[lvl], b.cin, b.heads
            m = arena.mark()
            p = b.prefix
            t = p + "transformer_blocks.0."
            kv = ext["ctx_kv"][attn_index[0]]          # View [Beff*ctx_tokens, 2C] filled at prepare()
            attn_index[0] += 1
            g = arena.alloc(x.rows, Cc)
            groupnorm(x, g, self.w(p + "norm.weight"), self.w(p + "norm.bias"), Lr, False, TAG_ATTN)
            h0 = arena.alloc(x.rows, Cc)
            i_h0 = gemm(g, self.w(p + "proj_in.weight"), Cc, Cc, h0, bias=self.w(p + "proj_in.bias"), Lout=Lr, tag=TAG_ATTN)

            def normed_linear(src: View, i_src: int, norm: str, lin: str, N: int, dst: View, gate: int = L_.GATE_NONE, has_bias: bool = False):
                """Linear(LayerNorm(src)) (attention.py:147-151).  Folded: the producer of src (op i_src) delivers the row moments,
                the Linear runs on the raw rows with gamma-scaled weights and corrects in its epilogue; else LayerNorm kernel + Linear."""
                if fuse_ln and ops.can_deliver_row_moments(i_src):
                    lv = stat_alloc(src.rows * 2)
                    ops.ops[i_src].u.gemm.row_moments = lv
                    gemm(src, self.w(t + lin + "_ln.weight"), N, Cc, dst, bias=self.w(t + lin + "_ln.bias"), gate=gate, Lout=Lr,
                         ln=(lv, self.w(t + lin + "_ln.colsum"), LN_EPS), tag=TAG_ATTN)
                else:
                    n = arena.alloc(src.rows, Cc)
                    ops.layernorm(src, n, self.w(t + norm + ".weight"), self.w(t + norm + ".bias"), TAG_ATTN)
                    gemm(n, self.w(t + lin + ".weight"), N, Cc, dst, bias=self.w(t + lin + ".bias") if has_bias else 0, gate=gate,
                         Lout=Lr, tag=TAG_ATTN)

            qkv = arena.alloc(x.rows, 3 * Cc)
            normed_linear(h0, i_h0, "norm1", "attn1.qkv", 3 * Cc, qkv)
            ao = arena.alloc(x.rows, Cc)
            ops.attention(qkv.c(0, Cc), qkv.c(Cc, 2 * Cc), qkv.c(2 * Cc, 3 * Cc), ao,
                          self.w(t + "attn1.relative_position_embedding"), self.w(t + "attn1.C_embedding"),
                          Beff, H, Lr, Lr, cfg.pos_max, TAG_ATTN)
            h1 = arena.alloc(x.rows, Cc)
            i_h1 = gemm(ao, self.w(t + "attn1.to_out.0.weight"), Cc, Cc, h1, bias=self.w(t + "attn1.to_out.0.bias"),
                        residual=h0, Lout=Lr, tag=TAG_ATTN)
            q2 = arena.alloc(x.rows, Cc)
            normed_linear(h1, i_h1, "norm2", "attn2.to_q", Cc, q2)
            ops.attention(q2, kv.c(0, Cc), kv.c(Cc, 2 * Cc), ao,
                          self.w(t + "attn2.relative_position_embedding"), self.w(t + "attn2.C_embedding"),
                          Beff, H, Lr, ctx_tokens, cfg.pos_max, TAG_ATTN)
            h2 = h0                                    # h0 is dead after the first residual add
            i_h2 = gemm(ao, self.w(t + "attn2.to_out.0.weight"), Cc, Cc, h2, bias=self.w(t + "attn2.to_out.0.bias"),
                        residual=h1, Lout=Lr, tag=TAG_ATTN)
            ff = arena.alloc(x.rows, 4 * Cc)
            normed_linear(h2, i_h2, "norm3", "ff.net.0.proj", 8 * Cc, ff, gate=L_.GATE_GEGLU, has_bias=True)
            # proj_out(ff.net.2(ff) + h2) + x as ONE GEMM over [ff | h2] with the packer-composed weight [Wp Wf | Wp]
            gemm(ff, self.w(p + "ff_out.weight"), Cc, 4 * Cc, out, bias=self.w(p + "ff_out.bias"), residual=x, Lout=Lr,
                 A2=h2, tag=TAG_ATTN)
            arena.release(m)

        def emit_s4(b: Block, x: View, out: View, lvl: int):
            Lr, Hc = lens[lvl], b.cin
            m = arena.mark()
            p = b.prefix
            s_ = p + "s4_model."
            g = arena.alloc(x.rows, Hc)
            groupnorm(x, g, self.w(p + "norm.weight"), self.w(p + "norm.bias"), Lr, False, TAG_S4)
            y = arena.alloc(x.rows, Hc)
            ops.s4conv(g, ext["s4_kt"][p].ptr, self.w(s_ + "D"), y, Beff, Lr, TAG_S4)
            z = g
            gemm(y, self.w(s_ + "output_linear.0.weight"), 2 * Hc, Hc, z, bias=self.w(s_ + "output_linear.0.bias"),
                 gate=L_.GATE_GLU, Lout=Lr, tag=TAG_S4)
            gemm(z, self.w(p + "out_layer.weight"), Hc, Hc, out, bias=self.w(p + "out_layer.bias"), taps=3,
                 mode=L_.CONV_SAME, Lin=Lr, Lout=Lr, residual=x, tag=TAG_S4)
            arena.release(m)

        def run_blocks(blocks: List[Block], x: View, final_out: Optional[View], lvl: int) -> Tuple[View, int]:
            """Run a TimestepEmbedSequential; the last block writes into final_out (if given)."""
            cur = x
            for j, b in enumerate(blocks):
                last = j == len(blocks) - 1
                if b.kind == "up":
                    tgt_rows = rows[lvl - 1]
                    out = final_out if (last and final_out is not None) else arena.alloc(tgt_rows, b.cout)
                    emit_upsample_conv(ops, self.blob, self.w, b.prefix, cur, out, lens[lvl], b.cin, b.cout, TAG_UPDOWN)
                    lvl -= 1
                    cur = out
                    continue
                out = final_out if (last and final_out is not None) else arena.alloc(cur.rows, b.cout)
                if b.kind == "res":
                    emit_res(b, cur, out, lvl)
                elif b.kind == "attn":
                    emit_attn(b, cur, out, lvl)
                elif b.kind == "s4":
                    emit_s4(b, cur, out, lvl)
                else:
                    raise ValueError(b.kind)
                cur = out
            return cur, lvl

        # ---- input blocks --------------------------------------------------------------------
        k = 0            # skip push counter
        lvl = 0
        h: Optional[View] = None
        for entry in self.lay.input:
            if isinstance(entry, tuple):          # AudioConcatBlock: h already sits in down_cat[lvl][:, :ch]
                h = down_cat[lvl]
                continue
            b0 = entry[0]
            if b0.kind == "conv_in":
                dst = down_cat[0].c(0, mc)
                gemm(xin, self.w(b0.prefix + "weight"), b0.cout, b0.cin, dst, bias=self.w(b0.prefix + "bias"), taps=3,
                     mode=L_.CONV_SAME, Lin=lens[0], Lout=lens[0], tag=TAG_IO)
                copy(dst, skip_home[k], TAG_IO)
                k += 1
                h = dst
            elif b0.kind == "down":
                dst = down_cat[lvl + 1].c(0, b0.cout)
                gemm(h, self.w(b0.prefix + "conv.weight"), b0.cout, b0.cin, dst, bias=self.w(b0.prefix + "conv.bias"),
                     taps=3, mode=L_.CONV_DOWN, Lin=lens[lvl], Lout=lens[lvl + 1], tag=TAG_UPDOWN)
                copy(dst, skip_home[k], TAG_UPDOWN)
                k += 1
                lvl += 1
                h = dst
            else:
                # persistent intermediates inside the sequential are tiny; write the block result
                # straight into its skip home and continue reading it from there
                h, lvl = run_blocks(entry, h, skip_home[k], lvl)
                k += 1
        assert k == n_skips and lvl == nlev - 1

        # ---- middle --------------------------------------------------------------------------
        h, lvl = run_blocks(self.lay.middle, h, up_cat[0].c(0, up_parts[0][0]), lvl)

        # ---- output blocks -------------------------------------------------------------------
        ub = 0
        final = arena.alloc(rows[0], mc)
        for entry in self.lay.output:
            if isinstance(entry, tuple):
                continue
            if ub + 1 < len(up_cat):
                nxt = up_cat[ub + 1].c(0, up_parts[ub + 1][0])
            else:
                nxt = final
            h, lvl = run_blocks(entry, up_cat[ub], nxt, lvl)
            ub += 1
        assert lvl == 0

        # ---- out: GN32 -> SiLU -> conv3 128->16 ------------------------------------------------
        ob = self.lay.out
        m = arena.mark()
        t = arena.alloc(rows[0], mc)
        groupnorm(final, t, self.w(ob.prefix + "0.weight"), self.w(ob.prefix + "0.bias"), lens[0], True, TAG_IO)
        gemm(t, self.w(ob.prefix + "2.weight"), ob.cout, ob.cin, eps, bias=self.w(ob.prefix + "2.bias"), taps=3,
             mode=L_.CONV_SAME, Lin=lens[0], Lout=lens[0], tag=TAG_IO)
        arena.release(m)
        return dict(ops=ops, xin=xin, eps=eps, audio_slots=audio_slots, ln_folded=fuse_ln)


class DecoderCompiler:
    """Decoder.forward (autoencoder.py:329-354) on channels-last rows."""

    def __init__(self, cfg: DecoderConfig, blob: WeightBlob, wbase: int, prefix: str = "model.first_stage_model.decoder."):
        self.cfg, self.blob, self.wbase, self.prefix = cfg, blob, wbase, prefix
        self.seq = decoder_layout(cfg, prefix)

    def w(self, name: str) -> int:
        return self.wbase + 4 * self.blob.offset(name)

    def compile(self, arena: Arena, B: int, Lz: int) -> dict:
        cfg = self.cfg
        ops = OpList(tc_weight_map(self.blob, self.wbase))
        G = cfg.num_groups
        zin = arena.alloc(B * Lz, cfg.z_channels)
        cur = zin
        out_view = None
        for b in self.seq:
            Lr = Lz * b.mul
            p = b.prefix
            if b.kind == "dec_conv_in":
                o = arena.alloc(B * Lr, b.cout)
                ops.gemm(cur, self.w(p + "weight"), b.cout, b.cin, o, bias=self.w(p + "bias"), taps=3, mode=L_.CONV_SAME,
                         Lin=Lr, Lout=Lr, tag=TAG_IO)
                cur = o
            elif b.kind == "dec_res":
                o = arena.alloc(B * Lr, b.cout)
                m = arena.mark()
                t1 = arena.alloc(B * Lr, b.cin)
                ops.groupnorm(cur, t1, self.w(p + "norm1.weight"), self.w(p + "norm1.bias"), B, Lr, G, True, TAG_RES)
                t2 = arena.alloc(B * Lr, b.cout)
                ops.gemm(t1, self.w(p + "conv1.weight"), b.cout, b.cin, t2, bias=self.w(p + "conv1.bias"), taps=3,
                         mode=L_.CONV_SAME, Lin=Lr, Lout=Lr, tag=TAG_RES)
                t3 = arena.alloc(B * Lr, b.cout)
                ops.groupnorm(t2, t3, self.w(p + "norm2.weight"), self.w(p + "norm2.bias"), B, Lr, G, True, TAG_RES)
                if b.has_skip_conv:
                    ops.gemm(t3, self.w(p + "out_skip.weight"), b.cout, b.cout, o, bias=self.w(p + "out_skip.bias"), taps=3,
                             mode=L_.CONV_SAME, Lin=Lr, Lout=Lr, A2=cur, tag=TAG_RES)
                else:
                    ops.gemm(t3, self.w(p + "conv2.weight"), b.cout, b.cout, o, bias=self.w(p + "conv2.bias"), taps=3,
                             mode=L_.CONV_SAME, Lin=Lr, Lout=Lr, residual=cur, tag=TAG_RES)
                arena.release(m)
                cur = o
            elif b.kind == "up":
                o = arena.alloc(B * Lr * 2, b.cout)
                emit_upsample_conv(ops, self.blob, self.w, p, cur, o, Lr, b.cin, b.cout, TAG_UPDOWN)
                cur = o
            elif b.kind == "dec_out":
                t = arena.alloc(B * Lr, b.cin)
                ops.groupnorm(cur, t, self.w(p + "norm_out.weight"), self.w(p + "norm_out.bias"), B, Lr, G, True, TAG_IO)
                out_view = arena.alloc(B * Lr, b.cout)
                ops.gemm(t, self.w(p + "conv_out.weight"), b.cout, b.cin, out_view, bias=self.w(p + "conv_out.bias"), taps=3,
                         mode=L_.CONV_SAME, Lin=Lr, Lout=Lr, tag=TAG_IO)
        return dict(ops=ops, zin=zin, logits=out_view, Lout=Lz * self.seq[-1].mul)

"""Every planned form of the tcgen05 GEMM (gemm_tc.cu / gemm_tc.cuh), one table case per path, each pinned to its kernel.

A tensor-core GEMM runs as one of four tile variants (64 / 128 / 256 wide, or 128 wide with two CTAs per SM walking a tile list), unsplit
(fused epilogue in tc_store_tile) or split-K (epilogue in gemm_tc_reduce_kernel), with one of the eight TcEpi epilogue instantiations,
one A-operand addressing form and optional operands.  The op-level tests in test_gpu_gemm_tc.py let the cost model choose the variant,
so they drift away from the paths their shapes were chosen for; here every case FORCES its variant and split and checks the plan.

GPU cases: plan == expected (at the device's SM count), output == fp64 torch statement (1e-5 of max|ref|, folded LayerNorm 2e-5, row
moments 1e-6 of the fp64 row sums of the stored output), nothing written outside the output view, second run bit-identical.
CPU tests (run by a plain `pytest`): every table case plans as stated, and every tensor-core GEMM of the real U-Net / decoder / wave
encoder / time-embedding plans runs on a (variant, split, epilogue, addressing, operands) signature that some table case covers."""
import ctypes as C
import collections
from dataclasses import dataclass

import pytest
import torch
import torch.nn.functional as F

from mug_diffusion_b200 import lib as L_
from mug_diffusion_b200.engine import LN_EPS, OpList, View
from mug_diffusion_b200.packer import tf32_split

PLAN_SMS = 148                     # B200: the production plans are checked against the table at this SM count
TOL, TOL_LN, TOL_SINK = 1e-5, 2e-5, 1e-6
EPI_NAMES = ("NONE", "GEGLU", "GLU", "SILU", "GELU", "SINK", "LN", "LN_GEGLU")        # enum TcEpi, gemm_tc.cuh
EPI_ACT_GATE = {"NONE": (L_.ACT_NONE, L_.GATE_NONE), "GEGLU": (L_.ACT_NONE, L_.GATE_GEGLU), "GLU": (L_.ACT_NONE, L_.GATE_GLU),
                "SILU": (L_.ACT_SILU, L_.GATE_NONE), "GELU": (L_.ACT_GELU, L_.GATE_NONE), "SINK": (L_.ACT_NONE, L_.GATE_NONE),
                "LN": (L_.ACT_NONE, L_.GATE_NONE), "LN_GEGLU": (L_.ACT_NONE, L_.GATE_GEGLU)}
MODE_NAMES = {L_.CONV_NONE: "linear", L_.CONV_SAME: "same", L_.CONV_DOWN: "down", L_.CONV_UP: "up", L_.CONV_TAPS: "taps"}
PAD = 4                            # every operand is a column window PAD columns into a wider buffer; C also has a row above and below
STEPS, STEP = 3, 2                 # per-step row vector: table of STEPS steps, device step counter = STEP


# ---------------------------------------------------------------------------------------------------------------------------------
# the case table
# ---------------------------------------------------------------------------------------------------------------------------------
@dataclass(frozen=True)
class Case:
    name: str
    variant: int          # forced mugd_gemm.tc_variant
    split: int            # forced mugd_gemm.split_k (1 = unsplit)
    expect: tuple         # planned (tile_n, ctas_per_sm, splits)
    N: int                # weight rows (gated: twice the output columns)
    K: int                # channels per tap
    L: int                # output rows per sample (Linear: rows per sample of the row vector; up2: input rows per sample)
    Bs: int = 1           # samples
    form: str = "linear"  # linear / same / down / up2 (Upsample as its two 2-tap parity GEMMs) / dil (3 taps, tap_shift -1, dilation)
    dil: int = 1
    K2: int = 0           # channels of the second source A2
    epi: str = "NONE"
    bias: bool = True
    res: bool = False
    rowvec: str = ""      # "" / "sample" / "step"

    @property
    def taps(self):
        return {"linear": 1, "same": 3, "down": 3, "up2": 2, "dil": 3}[self.form]

    @property
    def Lin(self):
        return 2 * self.L if self.form == "down" else self.L

    @property
    def rows_out(self):
        return self.Bs * self.L * (2 if self.form == "up2" else 1)

    @property
    def nout(self):
        return self.N // 2 if EPI_ACT_GATE[self.epi][1] else self.N


SPLIT = {64: 3, 128: 4, 256: 2}


def _variants():
    """(label, forced tc_variant, forced split_k, planned (tile_n, ctas_per_sm, splits)): each width unsplit and split-K, and the
    two-CTA variant (unsplit only: it has no split-K form)"""
    for bn, tv in ((64, L_.TC_N64), (128, L_.TC_N128), (256, L_.TC_N256)):
        yield f"n{bn}", bn, tv, 1, (bn, 1, 1)
        yield f"n{bn}s{SPLIT[bn]}", bn, tv, SPLIT[bn], (bn, 1, SPLIT[bn])
    yield "2cta", "2cta", L_.TC_N128_2CTA, 1, (128, 2, 1)


# Linear shapes of the epilogue sweep (M, N, K): partial last row tile and partial last column tile everywhere; gated half widths
# 56 / 100 / 164 / 260 are not multiples of the half tile; k-step counts 5 / 7 / 5 make the forced splits uneven.  The two-CTA
# shape has 76 x 5 = 380 tiles: more than 2 x 148, every CTA walks at least two.
EPI_SHAPE = {64: (200, 112, 160), 128: (300, 200, 224), 256: (260, 328, 160), "2cta": (9637, 520, 64)}
# conv shapes of the addressing sweep: N per width (partial last column tile for 128 / 256), samples of 160 rows (two row tiles, the
# second partial) or packed (24 rows: 5 samples per tile; 12 rows: 10 per tile) with a sample count that is not a multiple of that
FORM_N = {64: 96, 128: 136, 256: 264, "2cta": 136}
FORM_BS = {False: {160: 3}, True: {24: 7, 12: 13}}
FORM_BS_2CTA = {False: {160: 120}, True: {24: 751, 12: 1501}}    # >= 300 tiles (Linear 150 x 2): more than 2 x 148


def _ops_label(c_bias, c_res, rowvec="", K2=0):
    return ("b" if c_bias else "") + ("r" if c_res else "") + ({"sample": "v", "step": "t"}[rowvec] if rowvec else "") + ("2" if K2 else "")


def build_table():
    cases = []

    def add(**kw):
        cases.append(Case(**kw))

    for lab, w, tv, sp, exp in _variants():
        # every epilogue instantiation on a Linear: no operands, bias, bias + residual
        M, N, K = EPI_SHAPE[w]
        for epi in EPI_NAMES:
            for bias, res in ((False, False), (True, False), (True, True)):
                add(name=f"{lab}-{epi}-linear-{_ops_label(bias, res) or 'plain'}", variant=tv, split=sp, expect=exp, N=N, K=K, L=M, epi=epi,
                    bias=bias, res=res)
        # every addressing form, packed samples and not, with bias and with bias + residual
        Nf = FORM_N[w]
        forms = [("linear", 1, 96, False), ("same", 1, 0, True), ("same", 1, 96, True), ("down", 1, 0, True), ("up2", 1, 0, True),
                 ("dil", 2, 0, True), ("dil", 4, 0, True), ("dil", 8, 0, True)]
        for form, d, K2, packable in forms:
            for packed in ((False, True) if packable else (False,)):
                L = (12 if form == "dil" else 24) if packed else 160
                Bs = (FORM_BS_2CTA if w == "2cta" else FORM_BS)[packed][L]
                for res in ((False,) if form == "up2" else (False, True)):
                    add(name=f"{lab}-{form}{d if form == 'dil' else ''}-L{L}x{Bs}-{_ops_label(True, res, K2=K2)}", variant=tv, split=sp,
                        expect=exp, N=Nf, K=64, L=L, Bs=Bs, form=form, dil=d, K2=K2, res=res)
        # a dilation longer than the sample: the outer taps read nothing but the zero fill
        Bs = (FORM_BS_2CTA if w == "2cta" else FORM_BS)[True][12]
        add(name=f"{lab}-dil16-L12x{Bs}-b", variant=tv, split=sp, expect=exp, N=Nf, K=64, L=12, Bs=Bs, form="dil", dil=16)
        # the per-sample and the per-step row vector (time embedding), packed and not, with and without a residual
        for rv in ("sample", "step"):
            for packed in (False, True):
                L = 24 if packed else 160
                Bs = (FORM_BS_2CTA if w == "2cta" else FORM_BS)[packed][L]
                for res in (False, True):
                    add(name=f"{lab}-same-L{L}x{Bs}-{_ops_label(True, res, rv)}", variant=tv, split=sp, expect=exp, N=Nf, K=64, L=L, Bs=Bs,
                        form="same", res=res, rowvec=rv)
    # narrow outputs on the 64-wide tile (zero-filled weight rows beyond N)
    for N in (16, 40):
        for sp in (1, 3):
            add(name=f"n64{'s3' if sp > 1 else ''}-NONE-linear-N{N}-br", variant=L_.TC_N64, split=sp, expect=(64, 1, sp), N=N, K=96, L=300,
                res=True)
    # two-CTA variant with between 148 and 2 x 148 tiles (100 x 2): some CTAs walk two tiles, some one
    add(name="2cta-NONE-linear-200tiles-br", variant=L_.TC_N128_2CTA, split=1, expect=(128, 2, 1), N=136, K=64, L=12800, res=True)
    # the two-CTA variant has no split-K form: with a forced split it falls back to the 128-wide tile with that split
    add(name="2cta-forced-split2-falls-back-to-n128s2", variant=L_.TC_N128_2CTA, split=2, expect=(128, 1, 2), N=256, K=128, L=1000,
        res=True)
    return cases


CASES = build_table()


# ---------------------------------------------------------------------------------------------------------------------------------
# one case as launch ops (real tensors on the GPU, placeholder addresses for the planner on the CPU)
# ---------------------------------------------------------------------------------------------------------------------------------
class Buffers:
    """the operand buffers of one case: torch tensors on `device`, or (device None) distinct 1 KB-aligned placeholder addresses that
    only the planner sees"""

    def __init__(self, device=None):
        self.device, self.t, self._next = device, {}, 1 << 36

    def __call__(self, name, rows, cols, dtype=torch.float32):
        if self.device is None:
            addr, self._next = self._next, self._next + (1 << 34)
            return addr
        self.t[name] = torch.empty(rows, cols, dtype=dtype, device=self.device)
        return self.t[name].data_ptr()


def case_ops(c: Case, buf: Buffers) -> OpList:
    act, gate = EPI_ACT_GATE[c.epi]
    rows_in = c.Bs * c.Lin
    a = buf("A", rows_in, c.K + 2 * PAD)
    A = View(a + 4 * PAD, c.K + 2 * PAD, rows_in, c.K)
    ldc = c.nout + 2 * PAD
    out = View(buf("C", c.rows_out + 2, ldc) + 4 * (ldc + PAD), ldc, c.rows_out, c.nout)
    kw = dict(act=act, gate=gate, impl=L_.GEMM_TC, split_k=c.split, tc_variant=c.variant)
    if c.bias:
        kw["bias"] = buf("bias", 1, c.N)
    if c.res:
        ldr = c.nout + 2 * PAD
        kw["residual"] = View(buf("res", c.rows_out, ldr) + 4 * PAD, ldr, c.rows_out, c.nout)
    if c.rowvec:
        rvs = c.N + PAD
        kw.update(rowvec=buf("rowvec", (STEPS if c.rowvec == "step" else 1) * c.Bs, rvs), rowvec_b_stride=rvs)
        if c.rowvec == "step":
            kw.update(rowvec_step_stride=c.Bs * rvs, step=buf("step", 1, 1, torch.int32))
    if c.epi.startswith("LN"):
        kw["ln"] = (buf("ln_stats", rows_in, 2, torch.float64), buf("colsum", 1, c.N), LN_EPS)
    if c.K2:
        a2 = buf("A2", c.rows_out, c.K2 + 2 * PAD)
        kw["A2"] = View(a2 + 4 * PAD, c.K2 + 2 * PAD, c.rows_out, c.K2)
    ops = OpList()
    if c.form == "up2":
        for parity, shift in ((0, -1), (1, 0)):
            dst = View(out.ptr + 4 * parity * out.ld, 2 * out.ld, c.Bs * c.L, c.nout)
            ops.gemm(A, buf(f"W{parity}", c.N, 2 * c.K), c.N, c.K, dst, W_hi=buf(f"W{parity}hi", c.N, 2 * c.K),
                     W_lo=buf(f"W{parity}lo", c.N, 2 * c.K), taps=2, mode=L_.CONV_TAPS, Lin=c.L, Lout=c.L, tap_shift=shift, **kw)
    else:
        kt = c.taps * c.K + c.K2
        mode = {"linear": L_.CONV_NONE, "same": L_.CONV_SAME, "down": L_.CONV_DOWN, "dil": L_.CONV_TAPS}[c.form]
        if c.form == "dil":
            kw.update(tap_shift=-1, dilation=c.dil)
        ops.gemm(A, buf("W", c.N, kt), c.N, c.K, out, W_hi=buf("Whi", c.N, kt), W_lo=buf("Wlo", c.N, kt), taps=c.taps, mode=mode,
                 Lin=c.Lin, Lout=c.L, **kw)
    if c.epi == "SINK":
        sink = buf("sink", c.rows_out, 2, torch.float64)
        for op in ops.ops:
            op.u.gemm.row_moments = sink
    return ops


# ---------------------------------------------------------------------------------------------------------------------------------
# the planner's view of a GEMM
# ---------------------------------------------------------------------------------------------------------------------------------
def planned(lib, g, sms):
    """(tile_n, ctas_per_sm, splits, tiles, workspace bytes) the library plans for this GEMM on `sms` SMs (tile_n 0: not tensor-core)"""
    bn, occ = C.c_int32(), C.c_int32()
    L_.check(lib.mugd_gemm_tc_variant(C.byref(g), sms, C.byref(bn), C.byref(occ), None), "tc_variant")
    ok, sp, nt, ws = C.c_int32(), C.c_int32(), C.c_int32(), C.c_int64()
    L_.check(lib.mugd_gemm_tc_query(None, C.byref(g), sms, C.byref(ok), C.byref(sp), C.byref(ws), C.byref(nt)), "tc_query")
    return bn.value, occ.value, sp.value, nt.value, ws.value


def epi_of(g):
    """TcEpi instantiation of a GEMM (tc_epi_of, gemm_tc.cuh)"""
    if g.ln_stats:
        return "LN_GEGLU" if g.gate == L_.GATE_GEGLU else "LN"
    if g.row_moments:
        return "SINK"
    if g.gate:
        return {L_.GATE_GEGLU: "GEGLU", L_.GATE_GLU: "GLU"}[g.gate]
    return {L_.ACT_NONE: "NONE", L_.ACT_SILU: "SILU", L_.ACT_GELU: "GELU"}[g.act]


def signature(lib, g, sms=PLAN_SMS):
    """the path a GEMM takes through the tensor-core kernels, or None if it does not take them"""
    bn, occ, splits, _, _ = planned(lib, g, sms)
    if bn == 0 or not g.W_hi:
        return None
    return (bn, occ, splits > 1, epi_of(g), MODE_NAMES[g.conv_mode], g.conv_mode == L_.CONV_TAPS and g.tap_dilation > 1,
            g.conv_mode != L_.CONV_NONE and g.Lout < 128, bool(g.bias), bool(g.residual),
            "step" if g.step else ("sample" if g.rowvec else ""), g.K2 > 0)


def _sig_text(s):
    bn, occ, split, epi, mode, dil, packed, bias, res, rv, a2 = s
    ops = [n for n, f in (("bias", bias), ("residual", res), (f"{rv} rowvec", rv), ("A2", a2)) if f]
    return (f"{bn}{'x2cta' if occ == 2 else ''}{' split-K' if split else ''} {epi} {mode}{' dilated' if dil else ''}"
            f"{' packed' if packed else ''} [{', '.join(ops)}]")


# ---------------------------------------------------------------------------------------------------------------------------------
# CPU: the table plans as stated and covers every tensor-core GEMM of the real plans
# ---------------------------------------------------------------------------------------------------------------------------------
def test_table_cases_plan_as_expected():
    lib = L_.load()
    assert len({c.name for c in CASES}) == len(CASES)
    two_cta_tiles = []
    for c in CASES:
        for op in case_ops(c, Buffers()).ops:
            bn, occ, sp, tiles, _ = planned(lib, op.u.gemm, PLAN_SMS)
            assert (bn, occ, sp) == c.expect, c.name
            assert epi_of(op.u.gemm) == c.epi, c.name
            if occ == 2:
                two_cta_tiles.append(tiles)
    assert min(two_cta_tiles) > PLAN_SMS and any(t <= 2 * PLAN_SMS for t in two_cta_tiles)
    assert sum(t > 2 * PLAN_SMS for t in two_cta_tiles) >= len(two_cta_tiles) - 1       # all but one walk at least two tiles per CTA


def _production_gemms():
    """every GEMM of the U-Net (per-step / per-sample time embedding, LayerNorm folded or not), decoder, wave encoder and time-embedding
    plans at the shapes the sampler runs"""
    from mug_diffusion_b200 import packer, synth, wave
    from mug_diffusion_b200.config import ModelConfig
    from mug_diffusion_b200.engine import Arena, DecoderCompiler, UNetCompiler
    from test_host import _fake_ext

    cfg = ModelConfig()
    blob = packer.pack_model(synth.synthetic_state_dict(96), cfg.unet, cfg.decoder)
    for Beff, Lz in ((2, 96), (8, 512), (64, 512), (16, 992), (8, 992), (32, 256)):
        for per_sample_t in (False, True):
            for fold in (False, True):
                comp = UNetCompiler(cfg.unet, blob, 1 << 30)
                ops = comp.compile(Arena(1 << 32), Beff, Lz, _fake_ext(comp, Beff, Lz), per_sample_t, fold)["ops"].ops
                yield from (o.u.gemm for o in ops if o.kind == L_.OP_GEMM)
    for B, Lz in ((4, 512), (32, 512), (8, 992)):
        yield from (o.u.gemm for o in DecoderCompiler(cfg.decoder, blob, 1 << 30).compile(Arena(1 << 32), B, Lz)["ops"].ops
                    if o.kind == L_.OP_GEMM)
    wcfg = wave.WaveConfig()
    wb = packer.WeightBlob()
    wave.pack_wave(wb, wave.synthetic_wave_state_dict(wcfg), wcfg)
    wb.finalize()
    for B, T in ((1, 32768), (8, 32768), (2, 6144)):
        yield from (o.u.gemm for o in wave.WaveCompiler(wcfg, wb, 1 << 30).compile(Arena(1 << 34), B, T)["ops"].ops if o.kind == L_.OP_GEMM)
    # runtime.UNetSession.timestep_ops: sinusoid -> SiLU(Linear) -> SiLU(Linear) -> Linear into the fused ResBlock embedding table
    P, d0, d1, d2 = 1 << 32, cfg.unet.model_channels, cfg.unet.time_embed_dim, blob.meta["emb_total"]
    for R in (8, 50, 100, 1000):
        ops = OpList()
        ops.gemm(View(P, d0, R, d0), P, d1, d0, View(P, d1, R, d1), W_hi=P, W_lo=P, bias=P, act=L_.ACT_SILU)
        ops.gemm(View(P, d1, R, d1), P, d1, d1, View(P, d1, R, d1), W_hi=P, W_lo=P, bias=P, act=L_.ACT_SILU)
        ops.gemm(View(P, d1, R, d1), P, d2, d1, View(P, d2, R, d2), W_hi=P, W_lo=P, bias=P)
        yield from (o.u.gemm for o in ops.ops)


def test_every_production_gemm_path_is_in_the_table():
    lib = L_.load()
    table = {signature(lib, op.u.gemm) for c in CASES for op in case_ops(c, Buffers()).ops}
    uses = collections.Counter(s for s in (signature(lib, g) for g in _production_gemms()) if s is not None)
    assert len(uses) > 40
    missing = sorted((s for s in uses if s not in table), key=lambda s: -uses[s])
    assert not missing, "tensor-core GEMM paths of real plans that no table case runs:\n" + "\n".join(
        f"  {uses[s]:4d} x {_sig_text(s)}" for s in missing)


# ---------------------------------------------------------------------------------------------------------------------------------
# GPU: each case against fp64
# ---------------------------------------------------------------------------------------------------------------------------------
class Device:
    def __init__(self):
        self.lib = L_.load()
        self.handle = C.c_void_p()
        L_.check(self.lib.mugd_create(torch.cuda.current_device(), C.byref(self.handle)), "mugd_create")
        sms, major, minor = C.c_int32(), C.c_int32(), C.c_int32()
        L_.check(self.lib.mugd_device_info(self.handle, C.byref(sms), C.byref(major), C.byref(minor)), "device_info")
        self.sms = sms.value

    def run(self, ops: OpList):
        st = torch.cuda.current_stream().cuda_stream
        for op in ops.ops:
            L_.check(self.lib.mugd_op_run(self.handle, C.byref(op), st), "gemm")
        torch.cuda.synchronize()


@pytest.fixture(scope="module")
def dev():
    d = Device()
    yield d
    d.lib.mugd_destroy(d.handle)


def _fill(c: Case, buf: Buffers, gen):
    """seeded operands; returns the fp64 reference of the output view (and the 3-tap weight of up2)"""
    t = buf.t

    def rnd(name, scale=1.0, shift=0.0):
        x = t[name]
        x.copy_(torch.randn(x.shape, generator=gen, device=x.device) * scale + shift)

    rnd("A", shift=2.0 if c.epi.startswith("LN") else 0.0)         # LayerNorm: row means of 2 sigma, the cancellation case
    if c.K2:
        rnd("A2")
    kt = c.taps * c.K + c.K2
    w3 = None
    if c.form == "up2":
        w3 = torch.randn(c.N, c.K, 3, generator=gen, device=buf.device) / (3 * c.K) ** 0.5
        w0, w1, w2 = w3[:, :, 0], w3[:, :, 1], w3[:, :, 2]
        for parity, w in ((0, torch.cat([w0, w1 + w2], 1)), (1, torch.cat([w0 + w1, w2], 1))):
            hi, lo = tf32_split(w)
            t[f"W{parity}"].copy_(w), t[f"W{parity}hi"].copy_(hi), t[f"W{parity}lo"].copy_(lo)
    else:
        rnd("W", kt ** -0.5)
        hi, lo = tf32_split(t["W"])
        t["Whi"].copy_(hi), t["Wlo"].copy_(lo)
    for name, scale in (("bias", 0.1), ("res", 1.0), ("rowvec", 0.5)):
        if name in t:
            rnd(name, scale)
    if "step" in t:
        t["step"].fill_(STEP)
    t["C"].fill_(float("nan"))
    A = t["A"][:, PAD:PAD + c.K].double()
    if c.epi.startswith("LN"):
        t["ln_stats"].copy_(torch.stack([A.sum(1), (A * A).sum(1)], 1))
        t["colsum"].copy_(t["W"].double().sum(1).float()[None])
    return reference(c, buf, w3)


def reference(c: Case, buf: Buffers, w3=None) -> torch.Tensor:
    t = buf.t
    A = t["A"][:, PAD:PAD + c.K].double()
    if c.epi.startswith("LN"):
        A = F.layer_norm(A, (c.K,), eps=LN_EPS)
    if c.form == "up2":
        W = None
    else:
        W = t["W"].double()
    if c.form == "linear":
        acc = A @ W[:, :c.K].T
    else:
        x = A.reshape(c.Bs, c.Lin, c.K).permute(0, 2, 1)                  # [Bs, K, Lin]
        if c.form == "up2":
            y = F.conv1d(x.repeat_interleave(2, dim=-1), w3.double(), padding=1)
        else:
            w = W[:, :3 * c.K].reshape(c.N, 3, c.K).permute(0, 2, 1)      # [N, K, 3]: tap t of the packed [N][t][K] weight
            if c.form == "same":
                y = F.conv1d(x, w, padding=1)
            elif c.form == "down":
                y = F.conv1d(F.pad(x, (0, 1)), w, stride=2)
            else:
                y = F.conv1d(x, w, padding=c.dil, dilation=c.dil)
        acc = y.permute(0, 2, 1).reshape(c.rows_out, c.N)
    if c.K2:
        acc = acc + t["A2"][:, PAD:PAD + c.K2].double() @ W[:, c.taps * c.K:].T
    if c.bias:
        acc = acc + t["bias"].double()
    if c.rowvec:
        rows = t["rowvec"][:, :c.N].double()
        if c.rowvec == "step":
            rows = rows[STEP * c.Bs:(STEP + 1) * c.Bs]
        acc = acc + rows.repeat_interleave(c.rows_out // c.Bs, dim=0)
    act, gate = EPI_ACT_GATE[c.epi]
    if act == L_.ACT_SILU:
        acc = F.silu(acc)
    elif act == L_.ACT_GELU:
        acc = F.gelu(acc)
    if gate:                                                              # weight rows interleave (value_j, gate_j)
        v, g = acc[:, 0::2], acc[:, 1::2]
        acc = v * (F.gelu(g) if gate == L_.GATE_GEGLU else torch.sigmoid(g))
    if c.res:
        acc = acc + t["res"][:, PAD:PAD + c.nout].double()
    return acc


def _prepare(dev, c: Case, seed: int):
    buf = Buffers("cuda")
    ops = case_ops(c, buf)
    gen = torch.Generator(device="cuda")
    gen.manual_seed(seed)
    ref = _fill(c, buf, gen)
    # split-K workspace sized by the planner for this GEMM (forced splits are not bounded like the automatic ones)
    ws_bytes = max(planned(dev.lib, op.u.gemm, dev.sms)[4] for op in ops.ops)
    ws = torch.full((max(ws_bytes // 4, 4),), float("nan"), device="cuda")
    for op in ops.ops:
        op.u.gemm.workspace, op.u.gemm.workspace_bytes = ws.data_ptr(), ws_bytes
    return buf, ops, ref, ws


@pytest.mark.gpu
@pytest.mark.parametrize("c", CASES, ids=lambda c: c.name)
def test_tc_gemm_case(dev, c):
    buf, ops, ref, ws = _prepare(dev, c, seed=CASES.index(c))
    for op in ops.ops:
        bn, occ, sp, tiles, _ = planned(dev.lib, op.u.gemm, dev.sms)
        assert (bn, occ, sp) == c.expect
    runs = []
    for _ in range(2):
        if "sink" in buf.t:
            buf.t["sink"].zero_()
        dev.run(ops)
        runs.append(buf.t["C"].clone())
    Cb = runs[0]
    inside = torch.zeros_like(Cb, dtype=torch.bool)
    inside[1:1 + c.rows_out, PAD:PAD + c.nout] = True
    out = Cb[inside].view(c.rows_out, c.nout)
    assert bool(torch.isnan(Cb[~inside]).all()), "written outside the output view"
    assert bool(torch.isfinite(out).all()), "output view not fully written"
    err = float((out.double() - ref).abs().max() / ref.abs().max())
    assert err < (TOL_LN if c.epi.startswith("LN") else TOL), err
    if c.epi == "SINK":
        o = out.double()
        exp = torch.stack([o.sum(1), (o * o).sum(1)], 1)
        assert float((buf.t["sink"] - exp).abs().max() / exp.abs().max()) < TOL_SINK
    assert torch.equal(runs[0].view(torch.int32), runs[1].view(torch.int32)), "second run differs"


@pytest.mark.gpu
def test_split_workspace_one_tile_short_is_refused(dev):
    c = next(c for c in CASES if c.name == "n128s4-NONE-linear-br")
    buf, ops, _, ws = _prepare(dev, c, seed=0)
    g = ops.ops[0].u.gemm
    g.workspace_bytes -= 128 * c.expect[0] * 4
    with pytest.raises(L_.MugdError, match="workspace too small"):
        dev.run(ops)
    assert bool(torch.isnan(buf.t["C"]).all())

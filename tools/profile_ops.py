"""Where does one U-Net evaluation spend its device time?  Times every distinct op signature of the real launch plan
in its own CUDA graph (REPS copies back to back, inputs warm in L2) and prints count x us per signature.
usage (on the GPU box): python tools/profile_ops.py [--B 4] [--L 512] [--nocfg] [--tile 128x2]"""
import argparse
import collections
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from mug_diffusion_b200 import lib as L_, synth  # noqa: E402
from mug_diffusion_b200.config import ModelConfig  # noqa: E402
from mug_diffusion_b200.engine import OpList  # noqa: E402
from mug_diffusion_b200.runtime import Plan  # noqa: E402
from mug_diffusion_b200.sampler import MugDiffusionB200  # noqa: E402

NAMES = {1: "gemm", 2: "groupnorm", 3: "layernorm", 4: "attention", 5: "s4conv", 7: "transpose", 8: "copy2d"}
TILES = {"auto": L_.TC_AUTO, "64": L_.TC_N64, "128": L_.TC_N128, "256": L_.TC_N256, "128x2": L_.TC_N128_2CTA}


def signature(op):
    k = op.kind
    if k == L_.OP_GEMM:
        g = op.u.gemm
        return ("gemm", g.M, g.N, g.K, g.taps, g.conv_mode, g.gate, g.act, int(bool(g.residual)), int(bool(g.rowvec)), f"K2={g.K2}",
                f"rowmom={int(bool(g.row_moments))}", f"ln={int(bool(g.ln_stats))}")
    if k == L_.OP_GROUPNORM:
        g = op.u.gn
        return ("groupnorm", g.B, g.L, g.C, g.G, g.silu)
    if k == L_.OP_LAYERNORM:
        g = op.u.ln
        return ("layernorm", g.rows, g.C)
    if k == L_.OP_ATTENTION:
        a = op.u.attn
        return ("attention", a.B, a.H, a.Lq, a.Lk, a.D)
    if k == L_.OP_S4CONV:
        s = op.u.s4
        return ("s4conv", s.B, s.L, s.H)
    return (NAMES.get(k, str(k)),)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--B", type=int, default=4)
    ap.add_argument("--L", type=int, default=512)
    ap.add_argument("--nocfg", action="store_true")
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--gemm", default="auto")
    ap.add_argument("--fuse", type=int, default=1, help="0: stand-alone LayerNorm kernels")
    ap.add_argument("--attn", type=int, default=1, help="0: exact-fp32 FFMA attention kernel instead of the tcgen05 one")
    ap.add_argument("--only", default="", help="only ops whose family name contains this")
    ap.add_argument("--tile", choices=list(TILES), default="auto",
                    help="force this tensor-core GEMM tile variant where the shape allows it (128x2: 128 wide, two CTAs per SM)")
    a = ap.parse_args()
    dev = torch.device("cuda:0")
    cfg = ModelConfig()
    model = MugDiffusionB200(synth.synthetic_state_dict(a.L), cfg, z_length=a.L, device=dev, gemm_impl=a.gemm, fold_ln=bool(a.fuse))
    eng = model.engine
    eng.lib.mugd_set_attention_impl(eng.handle, a.attn)
    Beff = a.B if a.nocfg else 2 * a.B
    sess = eng.session(Beff, a.L, per_sample_t=False)
    arr, n = sess.plan._arr, sess.plan.n_ops
    groups = collections.OrderedDict()
    for i in range(n):
        groups.setdefault(signature(arr[i]), []).append(i)
    rows = []
    for sig, idx in groups.items():
        if a.only and a.only not in sig[0]:
            continue
        sub = OpList()
        if sig[0] == "gemm":
            arr[idx[0]].u.gemm.tc_variant = TILES[a.tile]
        for _ in range(a.reps):
            sub.ops.append(arr[idx[0]])
        pl = Plan(eng, sub)
        pl.run()
        pl.capture()
        pl.replay(2)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        pl.replay(5)
        e1.record()
        torch.cuda.synchronize()
        us = e0.elapsed_time(e1) * 1000 / (5 * a.reps)
        launches = pl.launches / a.reps
        extra = ""
        if sig[0] == "gemm":
            import ctypes as C
            sp, ok, nt = C.c_int32(), C.c_int32(), C.c_int32()
            g = arr[idx[0]].u.gemm
            try:
                eng.lib.mugd_gemm_tc_query(eng.handle, C.byref(g), 148, C.byref(ok), C.byref(sp), None, C.byref(nt))
                bn, occ = C.c_int32(), C.c_int32()
                eng.lib.mugd_gemm_tc_variant(C.byref(g), 148, C.byref(bn), C.byref(occ), None)
                extra = (f"tc={ok.value} tiles={nt.value} split={sp.value} bn={bn.value}x{occ.value} "
                         f"TF/s={2.0*g.M*g.N*(g.K*g.taps+g.K2)/us/1e6:.0f}")
            except Exception as e:       # noqa: BLE001
                extra = str(e)
        rows.append((us * len(idx), len(idx), us, launches, sig, extra))
    tot = sum(r[0] for r in rows)
    print(f"B={a.B} L={a.L} cfg={'off' if a.nocfg else 'on'}: {n} ops, sum of isolated op times {tot/1e3:.3f} ms")
    print(f"{'total us':>9s} {'share':>6s} {'n':>4s} {'us/op':>7s} {'k/op':>4s}  signature")
    for t, c, us, ln, sig, extra in sorted(rows, key=lambda r: -r[0]):
        print(f"{t:9.1f} {100*t/tot:5.1f}% {c:4d} {us:7.2f} {ln:4.1f}  {sig} {extra}")


if __name__ == "__main__":
    main()

"""Per-k-step timeline of CTA (0,0,0) of the tensor-core GEMM (globaltimer stamps written by the kernel's debug hooks).
usage: python tools/build_variant.py timeline -DMUGD_TC_TIMELINE   (here), then on the GPU box
       MUGD_LIB=mug_diffusion_b200/libmugd_timeline.so python tools/gemm_timeline.py"""
import ctypes as C
import math
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from gpu_util import OpRunner, ptr, view  # noqa: E402
from mug_diffusion_b200 import lib as L_  # noqa: E402
from mug_diffusion_b200.engine import OpList  # noqa: E402
from mug_diffusion_b200.packer import tf32_split  # noqa: E402

# (label, B, L, Cin, Cout, taps, split, tile variant)
SHAPES = [
    ("tiny 1x1 128->128 M4096 bn128", 8, 512, 128, 128, 1, 1, L_.TC_N128),
    ("tiny 1x1 128->128 M4096 bn128 split2", 8, 512, 128, 128, 1, 2, L_.TC_N128),
    ("1x1 256->256 M2048 bn128", 8, 256, 256, 256, 1, 1, L_.TC_N128),
    ("1x1 256->256 M2048 bn64", 8, 256, 256, 256, 1, 1, L_.TC_N64),
    ("1x1 384->384 M1024 bn128 unsplit", 8, 128, 384, 384, 1, 1, L_.TC_N128),
    ("conv3 640->256 B64 bn256", 64, 256, 640, 256, 3, 1, L_.TC_N256),
    ("conv3 640->256 B64 bn128", 64, 256, 640, 256, 3, 1, L_.TC_N128),
    ("ff1 512->4096 M512 bn256", 8, 64, 512, 4096, 1, 1, L_.TC_N256),
]


def main():
    R = OpRunner()
    st = torch.cuda.current_stream().cuda_stream
    for label, B, L, Cin, Cout, taps, split, variant in SHAPES:
        M = B * L
        x = torch.randn(M, Cin, device="cuda")
        w = torch.randn(Cout, taps * Cin) / math.sqrt(taps * Cin)
        hi, lo = tf32_split(w)
        wc, hc, lc = w.cuda(), hi.cuda(), lo.cuda()
        out = torch.zeros(M, Cout, device="cuda")
        ops = OpList()
        ops.gemm(view(x), ptr(wc), Cout, Cin, view(out), W_hi=ptr(hc), W_lo=ptr(lc), taps=taps,
                 mode=L_.CONV_SAME if taps == 3 else L_.CONV_NONE, Lin=L, Lout=L, impl=L_.GEMM_TC, split_k=split,
                 tc_variant=variant)
        for _ in range(3):
            R.run(ops)                      # warm: weights and activations in L2
        buf = torch.zeros(8 + 24 * 6, dtype=torch.int64, device="cuda")
        R.lib.mugd_debug_set_tc_timing(buf.data_ptr())
        L_.check(R.lib.mugd_op_run(R.handle, C.byref(ops.ops[0]), st), "op")
        torch.cuda.synchronize()
        R.lib.mugd_debug_set_tc_timing(None)
        t = buf.cpu().tolist()
        t0 = t[0]
        print(f"\n== {label}: M={M} N={Cout} K={taps*Cin}  [ns after kernel entry] setup done {t[1]-t0}, accum ready {t[2]-t0}, staged {t[3]-t0}, "
              f"phase-2 start {t[5]-t0}, done {t[4]-t0}")
        print("   k | tma issued  full seen  conv done  mma start  mma commit | empty seen (producer)")
        nk = min(24, taps * Cin // 32)
        for i in range(nk):
            r = [t[8 + i * 6 + j] for j in range(6)]
            print(f"  {i:2d} | " + " ".join(f"{(v - t0) if v else -1:10d}" for v in r[:5]) + f" | {(r[5]-t0) if r[5] else -1:10d}")


if __name__ == "__main__":
    main()

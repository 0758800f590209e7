"""Helpers for the -m gpu tests: run single libmugd ops on torch CUDA tensors through the C ABI."""
import ctypes as C

import torch

from mug_diffusion_b200 import lib as L_
from mug_diffusion_b200.engine import OpList, View


class OpRunner:
    def __init__(self):
        self.lib = L_.load()
        self.handle = C.c_void_p()
        L_.check(self.lib.mugd_create(0, C.byref(self.handle)), "mugd_create")

        self.ws = torch.zeros(16 * 1024 * 1024, device="cuda")

    def run(self, ops: OpList):
        for op in ops.ops:
            if op.kind == L_.OP_GEMM:
                g = op.u.gemm
                g.workspace, g.workspace_bytes = self.ws.data_ptr(), self.ws.numel() * 4
        st = torch.cuda.current_stream().cuda_stream
        for op in ops.ops:
            L_.check(self.lib.mugd_op_run(self.handle, C.byref(op), st), f"op {op.kind}")
        torch.cuda.synchronize()

    def set_impl(self, name):
        L_.check(self.lib.mugd_set_gemm_impl(self.handle, {"simt": L_.GEMM_SIMT, "tc": L_.GEMM_TC}[name]), "impl")


def view(t: torch.Tensor, c0: int = 0, c1: int = None) -> View:
    """2-D row-major CUDA tensor (optionally a column window of it) as a View."""
    assert t.dim() == 2 and t.is_contiguous()
    c1 = t.shape[1] if c1 is None else c1
    return View(t.data_ptr() + 4 * c0, t.shape[1], t.shape[0], c1 - c0)


def ptr(t: torch.Tensor) -> int:
    return t.data_ptr()


def nlc(x: torch.Tensor) -> torch.Tensor:
    """[B,C,L] -> [B*L, C] contiguous"""
    B, Cc, L = x.shape
    return x.permute(0, 2, 1).reshape(B * L, Cc).contiguous()


def ncl(x2: torch.Tensor, B: int) -> torch.Tensor:
    """[B*L, C] -> [B,C,L]"""
    M, Cc = x2.shape
    return x2.reshape(B, M // B, Cc).permute(0, 2, 1).contiguous()


def rel_err(a: torch.Tensor, b: torch.Tensor) -> float:
    a, b = a.detach().float().cpu(), b.detach().float().cpu()
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))

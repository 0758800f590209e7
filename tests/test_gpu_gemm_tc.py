"""tcgen05 3xTF32 GEMM (gemm_tc.cu) through the C ABI against an fp64 torch statement of the same contraction.
Tolerance 1e-5 of the output's max magnitude (the exact-fp32 FFMA kernel sits at ~1e-6; a single-pass TF32
GEMM would be ~5e-4 and fails this test by construction)."""
import math

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

from mug_diffusion_b200 import lib as L_  # noqa: E402
from mug_diffusion_b200 import synth  # noqa: E402
from mug_diffusion_b200.engine import OpList  # noqa: E402
from mug_diffusion_b200.packer import _interleave_halves, tf32_split  # noqa: E402

from gpu_util import OpRunner, ncl, nlc, ptr, rel_err, view  # noqa: E402

TOL = 1e-5


@pytest.fixture(scope="module")
def R():
    return OpRunner()


def g(name, shape, seed=9):
    return synth._gauss(synth._rng(seed, name), shape)


def run_tc(R, A, W2d, N, K, out, **kw):
    hi, lo = tf32_split(W2d)
    wc, hc, lc = W2d.cuda(), hi.cuda(), lo.cuda()
    ops = OpList()
    ops.gemm(A, ptr(wc), N, K, out, W_hi=ptr(hc), W_lo=ptr(lc), impl=L_.GEMM_TC, **kw)
    R.run(ops)
    return ops


def test_tf32_split_is_exact_enough():
    w = g("w", (257, 96)) * 3
    hi, lo = tf32_split(w)
    assert float(((hi + lo) - w).abs().max() / w.abs().max()) < 2.0 ** -21
    assert int((hi.view(torch.int32) & 0x1FFF).abs().max()) == 0 and int((lo.view(torch.int32) & 0x1FFF).abs().max()) == 0


@pytest.mark.parametrize("M,K,N", [(256, 128, 128), (100, 256, 192), (300, 64, 64), (1024, 512, 1536), (4096, 128, 384), (37, 32, 64),
                                   (4096, 128, 16), (700, 256, 40), (16384, 384, 3072)])     # narrow N (zero-filled weight rows), two-CTA variant
def test_tc_linear(R, M, K, N):
    x, w, b = g("x", (M, K)), g("w", (N, K)) / math.sqrt(K), 0.1 * g("b", (N,))
    ref = F.linear(x.double(), w.double(), b.double())
    xc, bc, out = x.cuda(), b.cuda(), torch.zeros(M, N).cuda()
    run_tc(R, view(xc), w, N, K, view(out), bias=ptr(bc))
    e = rel_err(out, ref)
    print(f"tc_linear M={M} K={K} N={N} rel_err={e:.2e}")
    assert e < TOL


@pytest.mark.parametrize("B,L,Cin,Cout", [(4, 64, 128, 128), (2, 512, 384, 128), (3, 124, 512, 512), (4, 62, 64, 64), (1, 992, 128, 128),
                                          (8, 64, 1536, 512), (5, 32, 256, 384), (2, 256, 640, 256), (8, 512, 128, 16), (64, 512, 128, 256)])
def test_tc_conv3_same(R, B, L, Cin, Cout):
    x, w, b = g("cx", (B, Cin, L)), g("cw", (Cout, Cin, 3)) / math.sqrt(3 * Cin), 0.1 * g("cb", (Cout,))
    emb, res = g("ce", (B, Cout)), g("cr", (B, Cout, L))
    ref = F.conv1d(x.double(), w.double(), b.double(), padding=1) + emb.double()[:, :, None] + res.double()
    wp = w.permute(0, 2, 1).contiguous().reshape(Cout, 3 * Cin)
    xc, bc, ec, rc = nlc(x).cuda(), b.cuda(), emb.cuda(), nlc(res).cuda()
    out = torch.zeros(B * L, Cout).cuda()
    run_tc(R, view(xc), wp, Cout, Cin, view(out), bias=ptr(bc), taps=3, mode=L_.CONV_SAME, Lin=L, Lout=L, rowvec=ptr(ec),
           rowvec_b_stride=Cout, residual=view(rc))
    e = rel_err(ncl(out.cpu(), B), ref)
    print(f"tc_conv3 B={B} L={L} Cin={Cin} Cout={Cout} rel_err={e:.2e}")
    assert e < TOL


@pytest.mark.parametrize("split", [2, 3, 7])
def test_tc_forced_split_k_is_deterministic(R, split):
    B, L, Cin, Cout = 2, 64, 512, 256
    x, w = g("sx", (B, Cin, L)), g("sw", (Cout, Cin, 3)) / math.sqrt(3 * Cin)
    ref = F.conv1d(x.double(), w.double(), None, padding=1)
    wp = w.permute(0, 2, 1).contiguous().reshape(Cout, 3 * Cin)
    xc = nlc(x).cuda()
    outs = []
    for _ in range(2):
        out = torch.zeros(B * L, Cout).cuda()
        run_tc(R, view(xc), wp, Cout, Cin, view(out), taps=3, mode=L_.CONV_SAME, Lin=L, Lout=L, split_k=split)
        outs.append(out.clone())
    assert rel_err(ncl(outs[0].cpu(), B), ref) < TOL
    assert torch.equal(outs[0], outs[1])


@pytest.mark.parametrize("gate", [L_.GATE_GEGLU, L_.GATE_GLU])
def test_tc_gated_and_strided(R, gate):
    M, K, Hh = 260, 256, 512
    x, w, b, res = g("gx", (M, K)), g("gw", (2 * Hh, K)) / math.sqrt(K), 0.1 * g("gb", (2 * Hh,)), g("gr", (M, Hh))
    proj = F.linear(x.double(), w.double(), b.double())
    a, gt = proj.chunk(2, dim=-1)
    ref = (a * F.gelu(gt) if gate == L_.GATE_GEGLU else a * torch.sigmoid(gt)) + res.double()
    wide_in = torch.zeros(M, K + 64).cuda()
    wide_in[:, 32:32 + K] = x.cuda()
    wide_out = torch.full((M, Hh + 128), 7.0).cuda()
    bi, rc = _interleave_halves(b).cuda(), res.cuda()
    run_tc(R, view(wide_in, 32, 32 + K), _interleave_halves(w), 2 * Hh, K, view(wide_out, 64, 64 + Hh), bias=ptr(bi), gate=gate,
           residual=view(rc))
    assert rel_err(wide_out[:, 64:64 + Hh], ref) < TOL
    assert float((wide_out[:, :64] - 7).abs().max()) == 0 and float((wide_out[:, 64 + Hh:] - 7).abs().max()) == 0


def test_tc_matches_simt_closely_and_beats_plain_tf32(R):
    """3xTF32 must sit at fp32 accuracy: compare error of tc vs simt against fp64 on a long-K conv"""
    B, L, Cin, Cout = 2, 128, 1536, 512
    x, w = g("mx", (B, Cin, L)), g("mw", (Cout, Cin, 3)) / math.sqrt(3 * Cin)
    ref = F.conv1d(x.double(), w.double(), None, padding=1)
    wp = w.permute(0, 2, 1).contiguous().reshape(Cout, 3 * Cin)
    xc = nlc(x).cuda()
    out_tc = torch.zeros(B * L, Cout).cuda()
    run_tc(R, view(xc), wp, Cout, Cin, view(out_tc), taps=3, mode=L_.CONV_SAME, Lin=L, Lout=L)
    out_si = torch.zeros(B * L, Cout).cuda()
    wc = wp.cuda()
    ops = OpList()
    ops.gemm(view(xc), ptr(wc), Cout, Cin, view(out_si), taps=3, mode=L_.CONV_SAME, Lin=L, Lout=L, impl=L_.GEMM_SIMT)
    R.run(ops)
    e_tc, e_si = rel_err(ncl(out_tc.cpu(), B), ref), rel_err(ncl(out_si.cpu(), B), ref)
    print(f"long-K conv: tc err {e_tc:.2e}  simt err {e_si:.2e}")
    assert e_tc < 5e-6 and e_si < 5e-6


@pytest.mark.parametrize("B,L,C", [(2, 512, 128), (4, 256, 256), (3, 128, 384), (8, 64, 64)])
def test_tc_downsample(R, B, L, C):
    """models.py:84-91: right-pad 1, conv3 stride 2 -- one strided TMA tensor map per tap"""
    x, w, b = g("dx", (B, C, L)), g("dw", (C, C, 3)) / math.sqrt(3 * C), 0.1 * g("db", (C,))
    ref = F.conv1d(F.pad(x.double(), (0, 1)), w.double(), b.double(), stride=2)
    wp = w.permute(0, 2, 1).contiguous().reshape(C, 3 * C)
    xc, bc = nlc(x).cuda(), b.cuda()
    out = torch.zeros(B * L // 2, C).cuda()
    run_tc(R, view(xc), wp, C, C, view(out), bias=ptr(bc), taps=3, mode=L_.CONV_DOWN, Lin=L, Lout=L // 2)
    e = rel_err(ncl(out.cpu(), B), ref)
    print(f"tc_down B={B} L={L} C={C} rel_err={e:.2e}")
    assert e < TOL


@pytest.mark.parametrize("impl", [L_.GEMM_TC, L_.GEMM_SIMT])
@pytest.mark.parametrize("B,L,C", [(2, 128, 256), (3, 64, 512), (2, 256, 64)])
def test_upsample_as_two_parity_gemms(R, impl, B, L, C):
    """models.py:66-70 nearest x2 + conv3 == y[2j] = W0 x[j-1] + (W1+W2) x[j], y[2j+1] = (W0+W1) x[j] + W2 x[j+1]"""
    from mug_diffusion_b200.engine import View
    x, w, b = g("ux", (B, C, L)), g("uw", (C, C, 3)) / math.sqrt(3 * C), 0.1 * g("ub", (C,))
    ref = F.conv1d(x.double().repeat_interleave(2, dim=-1), w.double(), b.double(), padding=1)
    w0, w1, w2 = w[:, :, 0], w[:, :, 1], w[:, :, 2]
    we, wo = torch.cat([w0, w1 + w2], dim=1).contiguous(), torch.cat([w0 + w1, w2], dim=1).contiguous()
    xc, bc = nlc(x).cuda(), b.cuda()
    out = torch.zeros(B * 2 * L, C).cuda()
    keep = []
    ops = OpList()
    for parity, wt, shift in ((0, we, -1), (1, wo, 0)):
        hi, lo = tf32_split(wt)
        wc, hc, lc = wt.cuda(), hi.cuda(), lo.cuda()
        keep += [wc, hc, lc]
        dst = View(out.data_ptr() + 4 * parity * C, 2 * C, B * L, C)
        ops.gemm(view(xc), ptr(wc), C, C, dst, W_hi=ptr(hc), W_lo=ptr(lc), bias=ptr(bc), taps=2, mode=L_.CONV_TAPS, Lin=L, Lout=L,
                 tap_shift=shift, impl=impl)
    R.run(ops)
    e = rel_err(ncl(out.cpu(), B), ref)
    print(f"upsample parity impl={impl} B={B} L={L} C={C} rel_err={e:.2e}")
    assert e < TOL


@pytest.mark.parametrize("kind", ["linear", "conv3"])
def test_tc_oversubscribed_grid(R, kind):
    """grids with more tiles than the 148 SMs, as the cost model plans them (both cases run the 128-wide two-CTA variant; the
    256-wide tiles are pinned in test_gpu_gemm_matrix.py): same numbers as the fp64 reference"""
    if kind == "linear":
        M, K, N = 296 * 128, 128, 256
        x, w, b = g("mcx", (M, K)), g("mcw", (N, K)) / math.sqrt(K), 0.1 * g("mcb", (N,))
        ref = F.linear(x.double(), w.double(), b.double())
        xc, bc, out = x.cuda(), b.cuda(), torch.zeros(M, N).cuda()
        run_tc(R, view(xc), w, N, K, view(out), bias=ptr(bc))
        assert rel_err(out, ref) < TOL
    else:
        B, L, Cin, Cout = 64, 512, 128, 128
        x, w = g("mcx3", (B, Cin, L)), g("mcw3", (Cout, Cin, 3)) / math.sqrt(3 * Cin)
        ref = F.conv1d(x.double(), w.double(), None, padding=1)
        wp = w.permute(0, 2, 1).contiguous().reshape(Cout, 3 * Cin)
        xc = nlc(x).cuda()
        out = torch.zeros(B * L, Cout).cuda()
        run_tc(R, view(xc), wp, Cout, Cin, view(out), taps=3, mode=L_.CONV_SAME, Lin=L, Lout=L)
        assert rel_err(ncl(out.cpu(), B), ref) < TOL


@pytest.mark.parametrize("impl", [L_.GEMM_TC, L_.GEMM_SIMT], ids=["tc", "simt"])
@pytest.mark.parametrize("B,L,C1,C2,Cout,split", [(2, 64, 512, 1536, 512, 0), (3, 128, 256, 768, 256, 0), (8, 512, 128, 384, 128, 0),
                                                   (2, 12, 64, 96, 64, 0), (2, 64, 512, 1536, 512, 5)])
def test_gemm_conv3_plus_skip_second_source(R, impl, B, L, C1, C2, Cout, split):
    """conv3(t3) + skip_connection(x) of a TimestepResBlock (unet.py:187-193,237-239) as ONE GEMM: the 1x1 term runs as extra
    k-steps on a second activation source; split-K ranges that straddle the two sources included"""
    t3, x = g("d_t3", (B, C1, L)), g("d_x", (B, C2, L))
    w3, w1 = g("d_w3", (Cout, C1, 3)) / math.sqrt(3 * C1), g("d_w1", (Cout, C2, 1)) / math.sqrt(C2)
    b = 0.1 * g("d_b", (Cout,))
    ref = F.conv1d(t3.double(), w3.double(), b.double(), padding=1) + F.conv1d(x.double(), w1.double())
    wcat = torch.cat([w3.permute(0, 2, 1).reshape(Cout, 3 * C1), w1.reshape(Cout, C2)], dim=1).contiguous()
    hi, lo = tf32_split(wcat)
    wc, hc, lc, bc = wcat.cuda(), hi.cuda(), lo.cuda(), b.cuda()
    tc_, xc = nlc(t3).cuda(), nlc(x).cuda()
    out = torch.zeros(B * L, Cout).cuda()
    ops = OpList()
    ops.gemm(view(tc_), ptr(wc), Cout, C1, view(out), W_hi=ptr(hc), W_lo=ptr(lc), bias=ptr(bc), taps=3, mode=L_.CONV_SAME, Lin=L, Lout=L,
             A2=view(xc), impl=impl, split_k=split)
    R.run(ops)
    e = rel_err(ncl(out.cpu(), B), ref)
    print(f"conv3+skip impl={impl} B={B} L={L} rel_err={e:.2e}")
    assert e < TOL


@pytest.mark.parametrize("impl", [L_.GEMM_TC, L_.GEMM_SIMT], ids=["tc", "simt"])
def test_gemm_ff_out_composed(R, impl):
    """proj_out(ff.net.2(f) + h) + x (attention.py:57-65,194-199) as one GEMM over [f | h] with the composed weight [Wp Wf | Wp]"""
    M, C = 1024, 256
    f, h, x = g("c_f", (M, 4 * C)), g("c_h", (M, C)), g("c_x", (M, C))
    wf, bf = g("c_wf", (C, 4 * C)) / math.sqrt(4 * C), 0.1 * g("c_bf", (C,))
    wp, bp = g("c_wp", (C, C)) / math.sqrt(C), 0.1 * g("c_bp", (C,))
    ref = F.linear(F.linear(f.double(), wf.double(), bf.double()) + h.double(), wp.double(), bp.double()) + x.double()
    wcat = torch.cat([wp.double() @ wf.double(), wp.double()], dim=1).float().contiguous()
    bcat = (wp.double() @ bf.double() + bp.double()).float()
    hi, lo = tf32_split(wcat)
    wc, hc, lc, bc = wcat.cuda(), hi.cuda(), lo.cuda(), bcat.cuda()
    fc, hcc, xc = f.cuda(), h.cuda(), x.cuda()
    out = torch.zeros(M, C).cuda()
    ops = OpList()
    ops.gemm(view(fc), ptr(wc), C, 4 * C, view(out), W_hi=ptr(hc), W_lo=ptr(lc), bias=ptr(bc), residual=view(xc), A2=view(hcc), impl=impl)
    R.run(ops)
    assert rel_err(out, ref) < TOL


@pytest.mark.parametrize("case", ["linear_bias", "conv3_rowvec_residual", "geglu", "ragged"])
def test_forced_two_cta_variant_walks_its_tile_list(R, case):
    """the 128-wide variant built for two CTAs per SM (TcSmem<128, 2>): at most 2 x SMs CTAs walk the tile list with running barrier
    rings -- forced through the op's tc_variant so that every CTA runs several tiles (the planner picks it by itself for GEMMs with
    more tiles than SMs)"""
    import ctypes as C
    two = L_.TC_N128_2CTA
    if case == "linear_bias":
        M, K, N = 12288, 256, 1024                                     # 96 x 8 = 768 tiles over 296 CTAs
        x, w, b = g("ox", (M, K)), g("ow", (N, K)) / math.sqrt(K), 0.1 * g("ob", (N,))
        ref = F.linear(x.double(), w.double(), b.double())
        xc, bc, out = x.cuda(), b.cuda(), torch.zeros(M, N).cuda()
        ops = run_tc(R, view(xc), w, N, K, view(out), bias=ptr(bc), tc_variant=two)
        got = out
    elif case == "conv3_rowvec_residual":
        B, L, Cin, Cout = 48, 512, 128, 256                            # 192 x 2 = 384 tiles
        x, w, b = g("px", (B, Cin, L)), g("pw", (Cout, Cin, 3)) / math.sqrt(3 * Cin), 0.1 * g("pb", (Cout,))
        emb, res = g("pe", (B, Cout)), g("pr", (B, Cout, L))
        ref = F.conv1d(x.double(), w.double(), b.double(), padding=1) + emb.double()[:, :, None] + res.double()
        wp = w.permute(0, 2, 1).contiguous().reshape(Cout, 3 * Cin)
        xc, bc, ec, rc = nlc(x).cuda(), b.cuda(), emb.cuda(), nlc(res).cuda()
        out = torch.zeros(B * L, Cout).cuda()
        ops = run_tc(R, view(xc), wp, Cout, Cin, view(out), bias=ptr(bc), taps=3, mode=L_.CONV_SAME, Lin=L, Lout=L, rowvec=ptr(ec),
                     rowvec_b_stride=Cout, residual=view(rc), tc_variant=two)
        got, ref = ncl(out.cpu(), B), ref
    elif case == "geglu":
        M, K, Hh = 8192, 128, 512                                      # N = 1024: 64 x 8 = 512 tiles
        x, w, b = g("qx", (M, K)), g("qw", (2 * Hh, K)) / math.sqrt(K), 0.1 * g("qb", (2 * Hh,))
        a, gt = F.linear(x.double(), w.double(), b.double()).chunk(2, dim=-1)
        ref = a * F.gelu(gt)
        xc, bi, out = x.cuda(), _interleave_halves(b).cuda(), torch.zeros(M, Hh).cuda()
        ops = run_tc(R, view(xc), _interleave_halves(w), 2 * Hh, K, view(out), bias=ptr(bi), gate=L_.GATE_GEGLU, tc_variant=two)
        got = out
    else:
        M, K, N = 20000, 96, 328                                       # 157 x 3 tiles; last row tile and last column tile are partial
        x, w = g("rx", (M, K)), g("rw", (N, K)) / math.sqrt(K)
        ref = F.linear(x.double(), w.double())
        xc, out = x.cuda(), torch.zeros(M, N).cuda()
        ops = run_tc(R, view(xc), w, N, K, view(out), tc_variant=two)
        got = out
    gm = ops.ops[0].u.gemm
    ok, sp, nt, ws = C.c_int32(), C.c_int32(), C.c_int32(), C.c_int64()
    R.lib.mugd_gemm_tc_query(None, C.byref(gm), 148, C.byref(ok), C.byref(sp), C.byref(ws), C.byref(nt))
    assert ok.value and sp.value == 1 and nt.value > 2 * 148            # more tiles than resident CTAs: the walk is exercised
    bn, occ = C.c_int32(), C.c_int32()
    R.lib.mugd_gemm_tc_variant(C.byref(gm), 148, C.byref(bn), C.byref(occ), None)
    assert (bn.value, occ.value) == (128, 2)
    assert rel_err(got.cpu() if got.is_cuda else got, ref) < TOL
    first = out.clone()
    R.run(ops)
    assert torch.equal(first, out)

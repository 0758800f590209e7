// Exact-fp32 (FFMA) implicit-GEMM for every dense contraction on the hot path:
//   nn.Linear, 1x1 conv, conv k=3 pad 1, Downsample (right-pad, stride 2), Upsample (nearest x2 + conv3)
// on channels-last activations, with the fused epilogues the U-Net needs (bias, time-embedding row add,
// SiLU / GELU, GEGLU / GLU gates, residual add, strided output into a concat buffer).
//
//   C[m, n] = epi( sum_{t < taps} sum_{k < K} A[row(m, t), k] * W[n, t*K + k] )
//
// This is the bit-faithful fp32 path (also the numerical referee for the tcgen05 3xTF32 kernel in
// gemm_tc.cu).  Tiles 64x64 or 128x128, BK = 16, 256 threads, register-prefetch double buffering.
//
// Reference call sites: unet.py:153-157,174-181,187-193 (ResBlock convs/skip), attention.py:38-65,
// 77-89,166-182 (Linear/1x1), models.py:55-91 (Up/Downsample), s4.py:1463-1469 (output_linear + GLU).
#include "common.cuh"

namespace mugd {

constexpr int SG_THREADS = 256;
constexpr int SG_BK = 16;

struct GemmParams {
    mugd_gemm g;
    int nk;  // total k-steps = (taps*K + K2)/16
};

__device__ __forceinline__ int conv_src_row(int mode, int l, int t, int Lin, int Lout, int tap_shift, int dil) {
    // returns source row inside the sample or -1 for the zero padding
    if (mode == MUGD_CONV_NONE) return l;
    if (mode == MUGD_CONV_SAME) {
        const int r = l + t - 1;
        return (r >= 0 && r < Lin) ? r : -1;
    }
    if (mode == MUGD_CONV_DOWN) {
        const int r = 2 * l + t;
        return (r < Lin) ? r : -1;
    }
    if (mode == MUGD_CONV_TAPS) {
        const int r = l + (t + tap_shift) * dil;
        return (r >= 0 && r < Lin) ? r : -1;
    }
    // MUGD_CONV_UP: index on the x2-upsampled axis, then halve
    const int r = l + t - 1;
    return (r >= 0 && r < Lout) ? (r >> 1) : -1;
}

template <int RM, int RN>
__global__ void __launch_bounds__(SG_THREADS)
gemm_simt_kernel(const GemmParams p) {
    constexpr int BM = 64 * RM, BN = 64 * RN;
    constexpr int SA = BM + 4, SW = BN + 4;
    __shared__ __align__(16) float As[2][SG_BK][SA];
    __shared__ __align__(16) float Ws[2][SG_BK][SW];

    pdl_wait();
    const mugd_gemm& g = p.g;
    const int tid = threadIdx.x;
    const int tx = tid & 15, ty = tid >> 4;
    const int m0 = blockIdx.y * BM, n0 = blockIdx.x * BN;

    // ---- global->register tile loaders -----------------------------------------------------------
    int a_row[RM], a_b[RM], a_l[RM];
    const int a_kq = tid & 3;
#pragma unroll
    for (int r = 0; r < RM; ++r) {
        const int row = (tid >> 2) + r * 64;
        a_row[r] = row;
        const int m = m0 + row;
        if (m < g.M) { a_b[r] = m / g.Lout; a_l[r] = m - a_b[r] * g.Lout; }
        else { a_b[r] = -1; a_l[r] = 0; }
    }
    int w_row[RN];
    bool w_ok[RN];
#pragma unroll
    for (int r = 0; r < RN; ++r) {
        w_row[r] = (tid >> 2) + r * 64;
        w_ok[r] = (n0 + w_row[r]) < g.N;
    }
    const int64_t wld = (int64_t)g.taps * g.K + g.K2;
    const int k_main = g.taps * g.K;

    float4 ra[RM], rw[RN];
    auto load_tile = [&](int kt) {
        const int kk = kt * SG_BK;
        const bool second = kk >= k_main;         // k-steps of the second source (1x1 term at the output row)
        const int t = second ? 0 : kk / g.K;
        const int k0 = second ? kk - k_main : kk - t * g.K;
#pragma unroll
        for (int r = 0; r < RM; ++r) {
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (a_b[r] >= 0) {
                if (second) {
                    v = ld_f4(g.A2 + ((int64_t)a_b[r] * g.Lout + a_l[r]) * g.lda2 + k0 + a_kq * 4);
                } else {
                    const int src = conv_src_row(g.conv_mode, a_l[r], t, g.Lin, g.Lout, g.tap_shift, g.tap_dilation > 1 ? g.tap_dilation : 1);
                    if (src >= 0) v = ld_f4(g.A + ((int64_t)a_b[r] * g.Lin + src) * g.lda + k0 + a_kq * 4);
                }
            }
            ra[r] = v;
        }
#pragma unroll
        for (int r = 0; r < RN; ++r) {
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (w_ok[r]) v = ld_f4(g.W + (int64_t)(n0 + w_row[r]) * wld + kk + a_kq * 4);
            rw[r] = v;
        }
    };
    auto store_tile = [&](int buf) {
#pragma unroll
        for (int r = 0; r < RM; ++r) {
            As[buf][a_kq * 4 + 0][a_row[r]] = ra[r].x;
            As[buf][a_kq * 4 + 1][a_row[r]] = ra[r].y;
            As[buf][a_kq * 4 + 2][a_row[r]] = ra[r].z;
            As[buf][a_kq * 4 + 3][a_row[r]] = ra[r].w;
        }
#pragma unroll
        for (int r = 0; r < RN; ++r) {
            Ws[buf][a_kq * 4 + 0][w_row[r]] = rw[r].x;
            Ws[buf][a_kq * 4 + 1][w_row[r]] = rw[r].y;
            Ws[buf][a_kq * 4 + 2][w_row[r]] = rw[r].z;
            Ws[buf][a_kq * 4 + 3][w_row[r]] = rw[r].w;
        }
    };

    float acc[RM][4][RN][4];
#pragma unroll
    for (int a = 0; a < RM; ++a)
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int b = 0; b < RN; ++b)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[a][i][b][j] = 0.f;

    load_tile(0);
    store_tile(0);
    __syncthreads();
    for (int kt = 0; kt < p.nk; ++kt) {
        const int buf = kt & 1;
        if (kt + 1 < p.nk) load_tile(kt + 1);
#pragma unroll
        for (int k = 0; k < SG_BK; ++k) {
            float4 av[RM], wv[RN];
#pragma unroll
            for (int a = 0; a < RM; ++a) av[a] = *reinterpret_cast<const float4*>(&As[buf][k][a * 64 + ty * 4]);
#pragma unroll
            for (int b = 0; b < RN; ++b) wv[b] = *reinterpret_cast<const float4*>(&Ws[buf][k][b * 64 + tx * 4]);
#pragma unroll
            for (int a = 0; a < RM; ++a) {
                const float af[4] = {av[a].x, av[a].y, av[a].z, av[a].w};
#pragma unroll
                for (int b = 0; b < RN; ++b) {
                    const float wf[4] = {wv[b].x, wv[b].y, wv[b].z, wv[b].w};
#pragma unroll
                    for (int i = 0; i < 4; ++i)
#pragma unroll
                        for (int j = 0; j < 4; ++j) acc[a][i][b][j] = fmaf(af[i], wf[j], acc[a][i][b][j]);
                }
            }
        }
        if (kt + 1 < p.nk) store_tile(buf ^ 1);
        __syncthreads();
    }

    // ---- epilogue --------------------------------------------------------------------------------
    const int step = g.step ? *g.step : 0;
    const float* rowvec = g.rowvec ? g.rowvec + (int64_t)step * g.rowvec_step_stride : nullptr;
#pragma unroll
    for (int a = 0; a < RM; ++a) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int m = m0 + a * 64 + ty * 4 + i;
            if (m >= g.M) continue;
            const int bidx = m / g.Lout;
#pragma unroll
            for (int b = 0; b < RN; ++b) {
                const int n = n0 + b * 64 + tx * 4;
                if (n >= g.N) continue;
                float v[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) v[j] = acc[a][i][b][j];
                if (g.bias) {
                    const float4 bb = ld_f4(g.bias + n);
                    v[0] += bb.x; v[1] += bb.y; v[2] += bb.z; v[3] += bb.w;
                }
                if (rowvec) {
                    const float4 rv = ld_f4(rowvec + (int64_t)bidx * g.rowvec_b_stride + n);
                    v[0] += rv.x; v[1] += rv.y; v[2] += rv.z; v[3] += rv.w;
                }
                if (g.act == MUGD_ACT_SILU) {
#pragma unroll
                    for (int j = 0; j < 4; ++j) v[j] = silu_f(v[j]);
                } else if (g.act == MUGD_ACT_GELU) {
#pragma unroll
                    for (int j = 0; j < 4; ++j) v[j] = gelu_f(v[j]);
                }
                if (g.gate == MUGD_GATE_NONE) {
                    if (g.residual) {
                        const float4 rr = ld_f4(g.residual + (int64_t)m * g.ldr + n);
                        v[0] += rr.x; v[1] += rr.y; v[2] += rr.z; v[3] += rr.w;
                    }
                    st_f4(g.C + (int64_t)m * g.ldc + n, make_float4(v[0], v[1], v[2], v[3]));
                } else {
                    float o0, o1;
                    if (g.gate == MUGD_GATE_GEGLU) { o0 = v[0] * gelu_f(v[1]); o1 = v[2] * gelu_f(v[3]); }
                    else { o0 = v[0] * sigmoid_f(v[1]); o1 = v[2] * sigmoid_f(v[3]); }
                    const int no = n >> 1;
                    if (g.residual) {
                        const float2 rr = *reinterpret_cast<const float2*>(g.residual + (int64_t)m * g.ldr + no);
                        o0 += rr.x; o1 += rr.y;
                    }
                    *reinterpret_cast<float2*>(g.C + (int64_t)m * g.ldc + no) = make_float2(o0, o1);
                }
            }
        }
    }
}

static int validate_gemm(const mugd_gemm& g) {
    MUGD_REQUIRE(g.M > 0 && g.N > 0 && g.K > 0, "gemm: empty shape M=%d N=%d K=%d", g.M, g.N, g.K);
    MUGD_REQUIRE(g.K % 16 == 0, "gemm: K=%d must be a multiple of 16", g.K);
    MUGD_REQUIRE(g.N % 4 == 0, "gemm: N=%d must be a multiple of 4", g.N);
    MUGD_REQUIRE(g.taps >= 1 && g.taps <= 3, "gemm: taps=%d must be 1..3", g.taps);
    if (g.conv_mode == MUGD_CONV_TAPS) MUGD_REQUIRE(g.Lin == g.Lout, "gemm: CONV_TAPS needs Lin == Lout");
    else MUGD_REQUIRE((g.conv_mode == MUGD_CONV_NONE) ? (g.taps == 1) : (g.taps == 3), "gemm: conv_mode %d inconsistent with taps %d", g.conv_mode, g.taps);
    MUGD_REQUIRE(g.Lout > 0 && g.Lin > 0 && g.M % g.Lout == 0, "gemm: M=%d not a multiple of Lout=%d", g.M, g.Lout);
    if (g.conv_mode == MUGD_CONV_NONE || g.conv_mode == MUGD_CONV_SAME)
        MUGD_REQUIRE(g.Lin == g.Lout, "gemm: Lin must equal Lout for conv_mode %d", g.conv_mode);
    if (g.conv_mode == MUGD_CONV_DOWN) MUGD_REQUIRE(g.Lin == 2 * g.Lout, "gemm: Downsample needs Lin == 2*Lout");
    if (g.conv_mode == MUGD_CONV_UP) MUGD_REQUIRE(g.Lout == 2 * g.Lin, "gemm: Upsample needs Lout == 2*Lin");
    MUGD_REQUIRE(g.A && g.W && g.C, "gemm: null operand");
    MUGD_REQUIRE(g.K2 >= 0 && (g.K2 == 0) == (g.A2 == nullptr), "gemm: A2 / K2 inconsistent");
    if (g.K2 > 0)
        MUGD_REQUIRE(g.K2 % 16 == 0 && aligned16(g.A2) && g.lda2 % 4 == 0 && g.lda2 >= g.K2 && g.conv_mode != MUGD_CONV_DOWN &&
                         g.conv_mode != MUGD_CONV_UP, "gemm: second source needs K2 %% 16 == 0, aligned A2 and an unstrided conv mode");
    MUGD_REQUIRE(aligned16(g.A) && aligned16(g.W) && g.lda % 4 == 0 && g.lda >= g.K, "gemm: A/W alignment or lda");
    MUGD_REQUIRE(!g.bias || aligned16(g.bias), "gemm: bias alignment");
    MUGD_REQUIRE(!g.rowvec || (aligned16(g.rowvec) && g.rowvec_b_stride % 4 == 0 && g.rowvec_step_stride % 4 == 0), "gemm: rowvec alignment");
    const int nout = g.gate == MUGD_GATE_NONE ? g.N : g.N / 2;
    const int al = g.gate == MUGD_GATE_NONE ? 4 : 2;
    MUGD_REQUIRE(g.ldc >= nout && g.ldc % al == 0 && (reinterpret_cast<uintptr_t>(g.C) % (4 * al)) == 0, "gemm: C alignment/ldc");
    MUGD_REQUIRE(!g.residual || (g.ldr >= nout && g.ldr % al == 0 && (reinterpret_cast<uintptr_t>(g.residual) % (4 * al)) == 0), "gemm: residual alignment/ldr");
    MUGD_REQUIRE(g.act >= 0 && g.act <= 2 && g.gate >= 0 && g.gate <= 2, "gemm: bad act/gate");
    return MUGD_OK;
}

int launch_gemm(const DeviceInfo& dev, const mugd_gemm& g, int default_impl, cudaStream_t st, int* launches) {
    int rc = validate_gemm(g);
    if (rc != MUGD_OK) return rc;
    int impl = g.impl == MUGD_GEMM_AUTO ? default_impl : g.impl;
    if (impl == MUGD_GEMM_TC) {
        if (gemm_tc_supported(g)) return launch_gemm_tc(dev, g, st, launches);
        MUGD_REQUIRE(g.impl != MUGD_GEMM_TC, "gemm: tensor-core path requested but shape unsupported (M=%d N=%d K=%d)", g.M, g.N, g.K);
    }
    // a weight that was split in place (W_hi == W) no longer holds fp32 values: the FFMA kernel must never read it
    MUGD_REQUIRE(!(g.W_hi && g.W_hi == g.W), "gemm: W was split into TF32 hi/lo in place, the FFMA kernel needs the plain fp32 weight (M=%d N=%d K=%d)", g.M, g.N, g.K);
    MUGD_REQUIRE(!g.row_moments && !g.ln_stats,
                 "gemm: the row-moment sink / folded LayerNorm exist on the tensor-core path only (M=%d N=%d K=%d fell to the FFMA kernel)", g.M, g.N, g.K);
    GemmParams p;
    p.g = g;
    p.nk = (g.taps * g.K + g.K2) / SG_BK;
    // big tiles only when they still fill the machine
    const long tiles128 = (long)((g.M + 127) / 128) * ((g.N + 127) / 128);
    if (tiles128 >= 2L * dev.sm_count) {
        dim3 grid((g.N + 127) / 128, (g.M + 127) / 128);
        MUGD_CHECK_CUDA(launch_k(gemm_simt_kernel<2, 2>, grid, dim3(SG_THREADS), 0, st, p));
    } else {
        dim3 grid((g.N + 63) / 64, (g.M + 63) / 64);
        MUGD_CHECK_CUDA(launch_k(gemm_simt_kernel<1, 1>, grid, dim3(SG_THREADS), 0, st, p));
    }
    MUGD_CHECK_CUDA(cudaGetLastError());
    if (launches) *launches += 1;
    return MUGD_OK;
}

}  // namespace mugd

// S4 layer pieces (mug/model/s4.py):
//
// (1) s4conv: the per-step part of S4.forward (s4.py:1503-1532).  The reference multiplies rfft(u, 2L)
//     by rfft(K, 2L) and keeps the first L samples of the inverse -- i.e. the causal convolution
//         y[b, l, h] = sum_{j <= l} K[h, j] * u[b, l - j, h]
//     which is evaluated here directly in fp32 (agrees with the FFT form to ~4e-7, SURVEY §8a a9), fused
//     with the D*u skip (s4.py:1514) and the exact-erf GELU (s4.py:1532).
//
// (2) s4 kernel generation: SSKernelNPLR.forward (s4.py:706-832) for rank 1 / channels 1 / rate 1 /
//     no state, with the NON-conjugate Cauchy sum `cauchy_naive` (s4.py:140-147) the reference falls back
//     to.  The reference regenerates K on every forward although it depends on parameters only; here it
//     runs once per (model, L) in fp64 and is checked tap-for-tap against the reference's K.
#include "common.cuh"

#include <math.h>

namespace mugd {

// =====================================================================================================
// (1) causal long convolution on the FFMA lanes.
//
// Why not tensor cores: the Toeplitz matrix is per CHANNEL, so a GEMM formulation has N = batch (8..64 columns) and must build a
// 128 x 32 operand tile per (channel, k-step) by hand; DFT-as-GEMM shares its matrix across channels but costs 8x the FLOPs at
// 3xTF32.  A direct kernel that keeps the FMA pipe fed wins: the round-1 kernel ran at ~18 % of the FFMA peak (per-load bounds
// checks, a register window copied every chunk); this one has no predicate in the inner loop and runs 16 loads per 64 FMAs.
//
// One CTA = 16 channels of one sample (x a share of the output blocks when nsplit > 1); u and K tiles live in shared memory with
// zero padding on both sides, so the inner loop never tests an index.  A warp computes a "super block" of 16 consecutive outputs:
// lanes 0-15 take outputs l0..l0+7 of channels 0..15, lanes 16-31 take l0+8..l0+15 of the same channels (both halves run the
// same number of chunks; the row pitch of 18 floats puts the two halves on disjoint banks, the tap loads are broadcasts).
// Per chunk of 8 taps a lane loads 8 new window values + 8 taps and issues 64 FMAs; the 15-wide window lives in two register
// arrays whose roles alternate (no copies).
// =====================================================================================================
constexpr int S4_WARPS = 16;       // 4 warps per scheduler hide the shared-memory latency of the dependent load -> FMA chains
constexpr int S4_R = 8;          // outputs per lane and taps per chunk
constexpr int S4_CH = 16;        // channels per CTA
constexpr int S4_PITCH = 18;     // floats per time step in shared memory (8 * 18 = 144 = 16 mod 32: the halves hit disjoint banks)
constexpr int S4_PAD = 32;       // zero rows in front of u (last chunk of the lower half: u[-16 .. -9]; the prefetch reaches 16 rows further)

__device__ __forceinline__ void s4_chunk(float (&acc)[S4_R], const float (&lo)[S4_R], const float (&hi)[S4_R], const float (&kk)[S4_R]) {
    // window W(t) = t < 8 ? lo[t] : hi[t - 8];  acc[r] += K[jc + i] * W(8 + r - i)
#pragma unroll
    for (int i = 0; i < S4_R; ++i) {
#pragma unroll
        for (int r = 0; r < S4_R; ++r) {
            const int t = S4_R + r - i;
            acc[r] = fmaf(kk[i], t < S4_R ? lo[t] : hi[t - S4_R], acc[r]);
        }
    }
}

template <bool INTERLEAVE>
__global__ void __launch_bounds__(32 * S4_WARPS)
s4conv_kernel(const mugd_s4conv s, int nsplit, int Lpad) {
    extern __shared__ float smem_s4[];
    float* us = smem_s4;                                        // [S4_PAD + Lpad][S4_PITCH], row S4_PAD = time 0
    float* ks = smem_s4 + (size_t)(S4_PAD + Lpad) * S4_PITCH;   // [Lpad + 3 * S4_R][S4_PITCH], zero beyond L
    pdl_wait();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int ch = lane & (S4_CH - 1), half = lane >> 4;
    const int c0 = blockIdx.x * S4_CH;
    const int b = blockIdx.y;
    const int L = s.L;
    const float* ub = s.u + (int64_t)b * L * s.ldu + c0;
    const float* Kc = s.Kt + c0;                                // tap j of channel c at Kc[j*H + c]
    // ---- tiles (zero padded) ----
    for (int i = threadIdx.x; i < (S4_PAD + Lpad) * S4_CH; i += 32 * S4_WARPS) {
        const int row = i / S4_CH, c = i % S4_CH;
        const int l = row - S4_PAD;
        us[row * S4_PITCH + c] = (l >= 0 && l < L) ? ub[(int64_t)l * s.ldu + c] : 0.f;
    }
    for (int i = threadIdx.x; i < (Lpad + 3 * S4_R) * S4_CH; i += 32 * S4_WARPS) {
        const int j = i / S4_CH, c = i % S4_CH;
        ks[j * S4_PITCH + c] = (j < L) ? Kc[(int64_t)j * s.H + c] : 0.f;
    }
    __syncthreads();

    const int h = c0 + ch;
    const float Dh = s.D[h];
    float* yb = s.y + (int64_t)b * L * s.ldy + h;
    const float* uz = us + S4_PAD * S4_PITCH + ch;              // uz[l * PITCH] = u[l, ch], valid for l >= -S4_PAD
    const float* kz = ks + ch;
    const int nsb = Lpad / (2 * S4_R);                          // super blocks of 16 outputs
    const int npairs = (nsb + 1) / 2;
    // blocked worker ids normally; interleaved (host's choice) when at most half of the workers get a pair, so that every CTA of the split keeps some
    const int worker = INTERLEAVE ? warp * nsplit + (int)blockIdx.z : (int)blockIdx.z * S4_WARPS + warp;
    const int nworkers = nsplit * S4_WARPS;
    // the cost of super block sb grows linearly with sb (causal): pairing sb with nsb-1-sb gives every worker the same work
    for (int p = worker; p < npairs; p += nworkers) {
#pragma unroll 1
        for (int which = 0; which < 2; ++which) {
            const int sb = which == 0 ? (nsb - 1 - p) : p;
            if (which == 1 && sb == nsb - 1 - p) break;
            const int l0 = sb * 2 * S4_R + half * S4_R;          // this lane's first output
            float acc[S4_R], wa[S4_R], wb[S4_R], wc[S4_R], ka[S4_R], kb[S4_R];
            // both halves run chunks jc = 0, 8, ..., sb*16 + 8 (the lower half's last chunk multiplies zeros)
            const int nchunks = sb * 2 + 2;
            const float* up = uz + (l0 - S4_R) * S4_PITCH;       // window rows l0 - jc - 8 + r
            const float* kp = kz;
#pragma unroll
            for (int r = 0; r < S4_R; ++r) { acc[r] = 0.f; wb[r] = uz[(l0 + r) * S4_PITCH]; wa[r] = up[r * S4_PITCH]; ka[r] = kp[r * S4_PITCH]; }
            // software pipeline: the window rows and taps of chunk c+1 are loaded before the 64 FMAs of chunk c are issued (the
            // rows of the padding in front of u / behind K make the last prefetch harmless)
#pragma unroll 1
            for (int c = 0; c < nchunks; c += 2) {
                up -= S4_R * S4_PITCH; kp += S4_R * S4_PITCH;
#pragma unroll
                for (int r = 0; r < S4_R; ++r) { wc[r] = up[r * S4_PITCH]; kb[r] = kp[r * S4_PITCH]; }
                s4_chunk(acc, wa, wb, ka);                       // lo = wa, hi = wb
                up -= S4_R * S4_PITCH; kp += S4_R * S4_PITCH;
#pragma unroll
                for (int r = 0; r < S4_R; ++r) { wb[r] = up[r * S4_PITCH]; ka[r] = kp[r * S4_PITCH]; }
                s4_chunk(acc, wc, wa, kb);                       // lo = wc, hi = wa
#pragma unroll
                for (int r = 0; r < S4_R; ++r) { const float t = wa[r]; wa[r] = wb[r]; wb[r] = wc[r]; (void)t; }
            }
#pragma unroll
            for (int r = 0; r < S4_R; ++r) {
                const int li = l0 + r;
                if (li < L) yb[(int64_t)li * s.ldy] = gelu_f(acc[r] + Dh * uz[li * S4_PITCH]);
            }
        }
    }
}

// the byte count grows with L: allow what the device allows, the launcher checks each launch against it
int configure_s4_kernels(const DeviceInfo& dev) {
    MUGD_CHECK_CUDA(cudaFuncSetAttribute(s4conv_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, dev.max_smem_optin));
    MUGD_CHECK_CUDA(cudaFuncSetAttribute(s4conv_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, dev.max_smem_optin));
    return MUGD_OK;
}

int launch_s4conv(const DeviceInfo& dev, const mugd_s4conv& s, cudaStream_t st, int* launches) {
    MUGD_REQUIRE(s.B > 0 && s.L > 0 && s.H > 0 && s.H % S4_CH == 0, "s4conv: H=%d must be a positive multiple of %d", s.H, S4_CH);
    MUGD_REQUIRE(s.ldu >= s.H && s.ldy >= s.H, "s4conv: ld < H");
    const int Lpad = (s.L + 2 * S4_R - 1) / (2 * S4_R) * (2 * S4_R);
    const size_t smem = ((size_t)(S4_PAD + Lpad) + (size_t)(Lpad + 3 * S4_R)) * S4_PITCH * sizeof(float);
    MUGD_REQUIRE((int)smem <= dev.max_smem_optin, "s4conv: L=%d needs %zu B of shared memory (max %d)", s.L, smem, dev.max_smem_optin);
    const int base = (s.H / S4_CH) * s.B;
    const int npairs = (Lpad / (2 * S4_R) + 1) / 2;
    int nsplit = 1;
    // A pair of super blocks is the unit of work (constant cost).  Output blocks are split over more CTAs while every worker (warp) still
    // gets two pairs -- and, as long as there are fewer CTAs than SMs, even when the doubled CTAs leave half of their warps without
    // a pair: the busy warps then share a scheduler with fewer others (Beff = 8, L = 512, H = 128: 64 -> 128 CTAs, 20.3 -> 13.6 us;
    // with the machine already full the same step costs time: Beff = 16, L = 496: 37.2 -> 39.8 us).
    while (nsplit < 16 && ((base * nsplit < 2 * dev.sm_count && nsplit * 2 * S4_WARPS <= npairs) ||
                           (base * nsplit < dev.sm_count && nsplit * S4_WARPS <= npairs)))
        nsplit *= 2;
    dim3 grid(s.H / S4_CH, s.B, nsplit);
    if (2 * npairs <= nsplit * S4_WARPS) MUGD_CHECK_CUDA(launch_k(s4conv_kernel<true>, grid, dim3(32 * S4_WARPS), smem, st, s, nsplit, Lpad));
    else MUGD_CHECK_CUDA(launch_k(s4conv_kernel<false>, grid, dim3(32 * S4_WARPS), smem, st, s, nsplit, Lpad));
    if (launches) *launches += 1;
    return MUGD_OK;
}

// =====================================================================================================
// (2) kernel generation (fp64).  With w' = w*dt, omega_f = exp(-2 pi i f / L):
//   reference:  z = 2(1-omega)/(1+omega);  r_xy = dt * sum_n v_xy[n] / (z - w'_n)
//               k_f = (r00 - r01 r10 / (1 + r11)) * 2 / (1 + omega);   K = irfft(k_f, L)[:L_out]
//   Multiplying numerator and denominator by (1+omega) -- an identity for ANY omega, exact or not --
//   removes the 0/0 at the Nyquist node (where the reference relies on rounding noise of its complex64
//   omega^f):
//               s_xy = dt * sum_n v_xy[n] / (2(1-omega) - w'_n (1+omega)),     r_xy = (1+omega) s_xy
//               k_f  = 2 * ( s00 - (1+omega) s01 s10 / (1 + (1+omega) s11) )
//   v00 = B*C, v01 = B*conj(P), v10 = P*C, v11 = P*conj(P)              (s4.py:771-778)
// =====================================================================================================
struct cd { double re, im; };
__device__ __forceinline__ cd cmul(cd a, cd b) { return {a.re * b.re - a.im * b.im, a.re * b.im + a.im * b.re}; }
__device__ __forceinline__ cd cadd(cd a, cd b) { return {a.re + b.re, a.im + b.im}; }
__device__ __forceinline__ cd csub(cd a, cd b) { return {a.re - b.re, a.im - b.im}; }
__device__ __forceinline__ cd cdiv(cd a, cd b) {
    const double d = b.re * b.re + b.im * b.im;
    return {(a.re * b.re + a.im * b.im) / d, (a.im * b.re - a.re * b.im) / d};
}

__global__ void s4_kf_kernel(const float* __restrict__ log_dt, const float* __restrict__ Bri,
                             const float* __restrict__ Cri, const float* __restrict__ Pri,
                             const float* __restrict__ inv_w_real, const float* __restrict__ w_imag,
                             const float* __restrict__ omega_ri, int H, int N, int Lint, double2* __restrict__ kf) {
    const int nf = Lint / 2 + 1;
    const int f = blockIdx.x * blockDim.x + threadIdx.x;
    const int h = blockIdx.y;
    if (f >= nf) return;
    const double dt = exp((double)log_dt[h]);
    // FFT nodes: the caller's table (the reference evaluates omega^f as a complex64 power, s4.py:595-598,
    // which is off by up to ~5e-6 at f = L/2; using the same nodes reproduces its kernel to ~2e-6) or exact.
    cd om;
    if (omega_ri) {
        om = {(double)omega_ri[2 * f], (double)omega_ri[2 * f + 1]};
    } else {
        double sn, cs;
        sincospi(-2.0 * (double)f / (double)Lint, &sn, &cs);
        om = {cs, sn};
    }
    const cd one_m = {2.0 * (1.0 - om.re), -2.0 * om.im};     // 2(1-omega)
    const cd one_p = {1.0 + om.re, om.im};                    // 1+omega
    cd s00 = {0, 0}, s01 = {0, 0}, s10 = {0, 0}, s11 = {0, 0};
    for (int n = 0; n < N; ++n) {
        const int64_t o = ((int64_t)h * N + n);
        const cd w = {-exp((double)inv_w_real[o]) * dt, (double)w_imag[o] * dt};
        const cd Bc = {(double)Bri[2 * o], (double)Bri[2 * o + 1]};
        const cd Cc = {(double)Cri[2 * o], (double)Cri[2 * o + 1]};
        const cd Pc = {(double)Pri[2 * o], (double)Pri[2 * o + 1]};
        const cd Qc = {Pc.re, -Pc.im};
        const cd den = csub(one_m, cmul(w, one_p));
        const cd inv = cdiv({1.0, 0.0}, den);
        s00 = cadd(s00, cmul(cmul(Bc, Cc), inv));
        s01 = cadd(s01, cmul(cmul(Bc, Qc), inv));
        s10 = cadd(s10, cmul(cmul(Pc, Cc), inv));
        s11 = cadd(s11, cmul(cmul(Pc, Qc), inv));
    }
    s00 = {s00.re * dt, s00.im * dt}; s01 = {s01.re * dt, s01.im * dt};
    s10 = {s10.re * dt, s10.im * dt}; s11 = {s11.re * dt, s11.im * dt};
    const cd num = cmul(one_p, cmul(s01, s10));
    const cd den = cadd({1.0, 0.0}, cmul(one_p, s11));
    const cd k = csub(s00, cdiv(num, den));
    kf[(int64_t)h * nf + f] = make_double2(2.0 * k.re, 2.0 * k.im);
}

// inverse real DFT of length Lint (C2R semantics of torch.fft.irfft: imaginary parts of the DC and
// Nyquist bins are ignored), truncated to L_out taps, written tap-major Kt[l][h].
__global__ void s4_irfft_kernel(const double2* __restrict__ kf, int H, int Lint, int Lout, float* __restrict__ Kt) {
    extern __shared__ double2 sm[];       // [nf] spectrum of this h, then [Lint] twiddles
    const int nf = Lint / 2 + 1;
    double2* X = sm;
    double2* tw = sm + nf;
    const int h = blockIdx.x;
    for (int f = threadIdx.x; f < nf; f += blockDim.x) X[f] = kf[(int64_t)h * nf + f];
    for (int m = threadIdx.x; m < Lint; m += blockDim.x) {
        double sn, cs;
        sincospi(2.0 * (double)m / (double)Lint, &sn, &cs);
        tw[m] = make_double2(cs, sn);
    }
    __syncthreads();
    const bool even = (Lint % 2) == 0;
    const int fmax = even ? nf - 1 : nf;  // exclusive upper bound of the doubled interior bins
    for (int l = threadIdx.x; l < Lout; l += blockDim.x) {
        double acc = X[0].x;
        int ph = 0;
        for (int f = 1; f < fmax; ++f) {
            ph += l;
            if (ph >= Lint) ph -= Lint;
            acc += 2.0 * (X[f].x * tw[ph].x - X[f].y * tw[ph].y);
        }
        if (even) acc += (l & 1) ? -X[nf - 1].x : X[nf - 1].x;
        Kt[(int64_t)l * H + h] = (float)(acc / (double)Lint);
    }
}

}  // namespace mugd

extern "C" int mugd_s4_kernel_gen(mugd_handle*, const float* log_dt, const float* Bri, const float* Cri,
                                  const float* Pri, const float* inv_w_real, const float* w_imag,
                                  const float* omega_ri, int32_t H, int32_t N, int32_t L_internal, int32_t L_out,
                                  float* Kt, void* workspace, int64_t workspace_bytes, void* stream) {
    using namespace mugd;
    MUGD_REQUIRE(H > 0 && N > 0 && L_internal > 0 && L_out > 0 && L_out <= L_internal,
                 "s4_kernel_gen: bad shape H=%d N=%d L_internal=%d L_out=%d (L_out must be <= L_internal; lengthen C~ with "
                 "the host-side setup first, s4.py:557-584)", H, N, L_internal, L_out);
    const int nf = L_internal / 2 + 1;
    MUGD_REQUIRE(workspace && workspace_bytes >= (int64_t)sizeof(double2) * H * nf, "s4_kernel_gen: workspace too small");
    MUGD_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 15u) == 0, "s4_kernel_gen: workspace alignment");
    cudaStream_t st = (cudaStream_t)stream;
    double2* kf = (double2*)workspace;
    dim3 g1((nf + 127) / 128, H);
    s4_kf_kernel<<<g1, 128, 0, st>>>(log_dt, Bri, Cri, Pri, inv_w_real, w_imag, omega_ri, H, N, L_internal, kf);
    MUGD_CHECK_CUDA(cudaGetLastError());
    const size_t smem = sizeof(double2) * (size_t)(nf + L_internal);
    MUGD_REQUIRE(smem <= 200 * 1024, "s4_kernel_gen: L_internal=%d too long for the one-shot DFT", L_internal);
    if (smem > 48 * 1024)
        MUGD_CHECK_CUDA(cudaFuncSetAttribute(s4_irfft_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    s4_irfft_kernel<<<H, 256, smem, st>>>(kf, H, L_internal, L_out, Kt);
    MUGD_CHECK_CUDA(cudaGetLastError());
    return MUGD_OK;
}

// GroupNorm(+SiLU) and LayerNorm on channels-last activations.  HBM/L2-bandwidth kernels:
// 128-bit vector loads, per-thread fp64 partial moments, warp-shuffle + one smem hop block reduction.
//
// Reference semantics:
//   Normalize = GroupNorm(num_groups, C, eps=1e-6, affine)      mug/model/models.py:10-13
//   followed by SiLU in TimestepResBlock / ResnetBlock / out     mug/diffusion/unet.py:153-157,174-181,489-491
//   nn.LayerNorm(dim) eps=1e-5                                   mug/model/attention.py:136-138
#include "common.cuh"

namespace mugd {

// One CTA per (group, sample).  The (L x cg) slab of a group is read ONCE: every thread pulls its float4s into registers with all
// loads in flight together (one memory round trip), the block reduces the fp64 moments, and the values are normalised straight from
// the registers.  Slabs of more than GN_MAXV float4 per thread (L * cg > 32768 elements) take the two-pass form below.
// cg is a multiple of 4 so every float4 belongs to one group.
constexpr int GN_THREADS = 256;
constexpr int GN_MAXV = 32;

__device__ __forceinline__ void gn_block_stats(double s, double ss, double inv_n, float eps, float& mean, float& rstd) {
    __shared__ double red[2][GN_THREADS / 32];
    s = warp_sum(s);
    ss = warp_sum(ss);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (lane == 0) { red[0][warp] = s; red[1][warp] = ss; }
    __syncthreads();
    // every thread adds the eight warp partials itself (broadcast reads, same order everywhere): one barrier instead of
    // barrier -> thread 0 -> barrier on the critical path of a 3 us kernel
    double ts = 0.0, tss = 0.0;
#pragma unroll
    for (int w = 0; w < GN_THREADS / 32; ++w) { ts += red[0][w]; tss += red[1][w]; }
    // the variance is formed in fp64 (E[x^2] - mean^2 cancels); its reciprocal square root in fp32 with one Newton step (~1 ulp)
    // instead of the ~100-deep fp64 sqrt + divide chain
    const double m = ts * inv_n;
    const double var = tss * inv_n - m * m;
    const float v = fmaxf((float)var, 0.f) + eps;
    float r = rsqrtf(v);
    r = r * (1.5f - 0.5f * v * r * r);
    mean = (float)m;
    rstd = r;
}

template <int NV>
__global__ void __launch_bounds__(GN_THREADS)
groupnorm_silu_reg_kernel(const float* __restrict__ x, int64_t ldx, float* __restrict__ y, int64_t ldy,
                          const float* __restrict__ gamma, const float* __restrict__ beta,
                          int L, int C, int G, float eps, int silu) {
    pdl_wait();
    const int g = blockIdx.x, b = blockIdx.y;
    const int cg = C / G;
    const int q = cg >> 2;                 // float4 per row of this group
    const int total = L * q;
    const double inv_n = 1.0 / ((double)L * cg);       // requested before the loads: off the chain behind the block reduction
    const float* xb = x + (int64_t)b * L * ldx + (int64_t)g * cg;
    float* yb = y + (int64_t)b * L * ldy + (int64_t)g * cg;
    float4 v[NV];
#pragma unroll
    for (int u = 0; u < NV; ++u) {
        const int i = (int)threadIdx.x + u * GN_THREADS;
        v[u] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (i < total) {
            const int row = i / q, qq = i - row * q;
            v[u] = ld_f4(xb + (int64_t)row * ldx + qq * 4);
        }
    }
    double s = 0.0, ss = 0.0;
#pragma unroll
    for (int u = 0; u < NV; ++u) {          // (slots past `total` hold zeros)
        s += (double)v[u].x + (double)v[u].y + (double)v[u].z + (double)v[u].w;
        ss += (double)v[u].x * v[u].x + (double)v[u].y * v[u].y + (double)v[u].z * v[u].z + (double)v[u].w * v[u].w;
    }
    // gamma / beta do not depend on the moments: request them before the block reduction (NV <= 8: registers are cheap there)
    const float* gm = gamma + g * cg;
    const float* bt = beta + g * cg;
    constexpr bool PRE = NV <= 8;
    float4 gav[PRE ? NV : 1], bev[PRE ? NV : 1];
    if constexpr (PRE) {
#pragma unroll
        for (int u = 0; u < NV; ++u) {
            const int i = (int)threadIdx.x + u * GN_THREADS;
            const int qq = i < total ? i % q : 0;
            gav[u] = ld_f4(gm + qq * 4);
            bev[u] = ld_f4(bt + qq * 4);
        }
    }
    float mean, rstd;
    gn_block_stats(s, ss, inv_n, eps, mean, rstd);
#pragma unroll
    for (int u = 0; u < NV; ++u) {
        const int i = (int)threadIdx.x + u * GN_THREADS;
        if (i < total) {
            const int row = i / q, qq = i - row * q;
            float4 ga, be;
            if constexpr (PRE) { ga = gav[u]; be = bev[u]; }
            else { ga = ld_f4(gm + qq * 4); be = ld_f4(bt + qq * 4); }
            float4 o;
            o.x = (v[u].x - mean) * rstd * ga.x + be.x;
            o.y = (v[u].y - mean) * rstd * ga.y + be.y;
            o.z = (v[u].z - mean) * rstd * ga.z + be.z;
            o.w = (v[u].w - mean) * rstd * ga.w + be.w;
            if (silu) { o.x = silu_f(o.x); o.y = silu_f(o.y); o.z = silu_f(o.z); o.w = silu_f(o.w); }
            st_f4(yb + (int64_t)row * ldy + qq * 4, o);
        }
    }
}

// two-pass form for slabs that do not fit the registers: moments, then apply (the second read is served by L1/L2)
__global__ void __launch_bounds__(GN_THREADS)
groupnorm_silu_kernel(const float* __restrict__ x, int64_t ldx, float* __restrict__ y, int64_t ldy,
                      const float* __restrict__ gamma, const float* __restrict__ beta,
                      int L, int C, int G, float eps, int silu) {
    pdl_wait();
    const int g = blockIdx.x, b = blockIdx.y;
    const int cg = C / G;
    const int q = cg >> 2;
    const int total = L * q;
    const double inv_n = 1.0 / ((double)L * cg);       // requested before the loads: off the chain behind the block reduction
    const float* xb = x + (int64_t)b * L * ldx + (int64_t)g * cg;
    float* yb = y + (int64_t)b * L * ldy + (int64_t)g * cg;

    double s = 0.0, ss = 0.0;
    for (int i = threadIdx.x; i < total; i += GN_THREADS) {
        const int row = i / q, qq = i - row * q;
        const float4 v = ld_f4(xb + (int64_t)row * ldx + qq * 4);
        s += (double)v.x + (double)v.y + (double)v.z + (double)v.w;
        ss += (double)v.x * v.x + (double)v.y * v.y + (double)v.z * v.z + (double)v.w * v.w;
    }
    float mean, rstd;
    gn_block_stats(s, ss, inv_n, eps, mean, rstd);
    const float* gm = gamma + g * cg;
    const float* bt = beta + g * cg;
    for (int i = threadIdx.x; i < total; i += GN_THREADS) {
        const int row = i / q, qq = i - row * q;
        const float4 v = ld_f4(xb + (int64_t)row * ldx + qq * 4);
        const float4 ga = ld_f4(gm + qq * 4);
        const float4 be = ld_f4(bt + qq * 4);
        float4 o;
        o.x = (v.x - mean) * rstd * ga.x + be.x;
        o.y = (v.y - mean) * rstd * ga.y + be.y;
        o.z = (v.z - mean) * rstd * ga.z + be.z;
        o.w = (v.w - mean) * rstd * ga.w + be.w;
        if (silu) { o.x = silu_f(o.x); o.y = silu_f(o.y); o.z = silu_f(o.z); o.w = silu_f(o.w); }
        st_f4(yb + (int64_t)row * ldy + qq * 4, o);
    }
}

// A second form -- one thread-block CLUSTER per sample, CTAs owning bands of whole rows (fully coalesced, gamma / beta per thread,
// band moments exchanged through distributed shared memory) -- was built and measured in round 2 and lost almost everywhere
// (profiles/r02_groupnorm_ab.md: 0.30 -> 0.49 ms per step at Beff = 8, 1.29 -> 1.36 at Beff = 64, 0.77 -> 1.03 at L = 992): inside the
// graph the slabs come out of L2, where the 16..48-byte pieces of this kernel cost little, while two cluster barriers + the DSMEM
// exchange sit on every launch's critical path.  Removed.
int launch_groupnorm(const DeviceInfo&, const mugd_groupnorm& g, cudaStream_t st, int* launches) {
    MUGD_REQUIRE(g.B > 0 && g.L > 0 && g.C > 0 && g.G > 0, "groupnorm: empty shape B=%d L=%d C=%d G=%d", g.B, g.L, g.C, g.G);
    MUGD_REQUIRE(g.C % g.G == 0 && (g.C / g.G) % 4 == 0, "groupnorm: C/G must be a multiple of 4 (C=%d G=%d)", g.C, g.G);
    MUGD_REQUIRE(g.ldx % 4 == 0 && g.ldy % 4 == 0 && aligned16(g.x) && aligned16(g.y) && aligned16(g.gamma) && aligned16(g.beta),
                 "groupnorm: operands must be 16-byte aligned with ld %% 4 == 0");
    MUGD_REQUIRE(g.ldx >= g.C && g.ldy >= g.C, "groupnorm: leading dimension smaller than C");
    dim3 grid(g.G, g.B);
    const int per_thread = (g.L * (g.C / g.G / 4) + GN_THREADS - 1) / GN_THREADS;     // float4 per thread
#define GN_GO(K) MUGD_CHECK_CUDA(launch_k(K, grid, dim3(GN_THREADS), 0, st, g.x, g.ldx, g.y, g.ldy, g.gamma, g.beta, g.L, g.C, g.G, g.eps, g.silu))
    if (per_thread <= 2) GN_GO(groupnorm_silu_reg_kernel<2>);
    else if (per_thread <= 4) GN_GO(groupnorm_silu_reg_kernel<4>);
    else if (per_thread <= 8) GN_GO(groupnorm_silu_reg_kernel<8>);
    else if (per_thread <= 16) GN_GO(groupnorm_silu_reg_kernel<16>);
    else if (per_thread <= GN_MAXV) GN_GO(groupnorm_silu_reg_kernel<GN_MAXV>);
    else GN_GO(groupnorm_silu_kernel);
#undef GN_GO
    if (launches) *launches += 1;
    return MUGD_OK;
}

// ---- LayerNorm: one warp per row, row held in registers (C <= 1024) --------------------------------
constexpr int LN_WARPS = 8;
constexpr int LN_MAXQ = 8;   // float4 per lane

__global__ void __launch_bounds__(LN_WARPS * 32)
layernorm_kernel(const float* __restrict__ x, int64_t ldx, float* __restrict__ y, int64_t ldy,
                 const float* __restrict__ gamma, const float* __restrict__ beta, int rows, int C, float eps) {
    pdl_wait();
    const int row = blockIdx.x * LN_WARPS + (threadIdx.x >> 5);
    if (row >= rows) return;
    const int lane = threadIdx.x & 31;
    const int nq = C >> 2;
    const float* xr = x + (int64_t)row * ldx;
    float4 v[LN_MAXQ];
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < LN_MAXQ; ++i) {
        const int qi = lane + i * 32;
        if (qi < nq) {
            v[i] = ld_f4(xr + qi * 4);
            s += (v[i].x + v[i].y) + (v[i].z + v[i].w);
        } else {
            v[i] = make_float4(0.f, 0.f, 0.f, 0.f);
        }
    }
    const float mean = warp_sum(s) / (float)C;
    float ss = 0.f;
#pragma unroll
    for (int i = 0; i < LN_MAXQ; ++i) {
        const int qi = lane + i * 32;
        if (qi < nq) {
            const float a = v[i].x - mean, b = v[i].y - mean, c = v[i].z - mean, d = v[i].w - mean;
            ss += (a * a + b * b) + (c * c + d * d);
        }
    }
    const float rstd = rsqrtf(warp_sum(ss) / (float)C + eps);
    float* yr = y + (int64_t)row * ldy;
#pragma unroll
    for (int i = 0; i < LN_MAXQ; ++i) {
        const int qi = lane + i * 32;
        if (qi < nq) {
            const float4 ga = ld_f4(gamma + qi * 4), be = ld_f4(beta + qi * 4);
            float4 o;
            o.x = (v[i].x - mean) * rstd * ga.x + be.x;
            o.y = (v[i].y - mean) * rstd * ga.y + be.y;
            o.z = (v[i].z - mean) * rstd * ga.z + be.z;
            o.w = (v[i].w - mean) * rstd * ga.w + be.w;
            st_f4(yr + qi * 4, o);
        }
    }
}

int launch_layernorm(const DeviceInfo&, const mugd_layernorm& g, cudaStream_t st, int* launches) {
    MUGD_REQUIRE(g.rows > 0 && g.C > 0, "layernorm: empty shape");
    MUGD_REQUIRE(g.C % 4 == 0 && g.C <= LN_MAXQ * 128, "layernorm: C=%d must be a multiple of 4 and <= %d", g.C, LN_MAXQ * 128);
    MUGD_REQUIRE(g.ldx % 4 == 0 && g.ldy % 4 == 0 && aligned16(g.x) && aligned16(g.y) && aligned16(g.gamma) && aligned16(g.beta),
                 "layernorm: operands must be 16-byte aligned with ld %% 4 == 0");
    const int blocks = (g.rows + LN_WARPS - 1) / LN_WARPS;
    MUGD_CHECK_CUDA(launch_k(layernorm_kernel, dim3(blocks), dim3(LN_WARPS * 32), 0, st, g.x, g.ldx, g.y, g.ldy, g.gamma, g.beta, g.rows,
                             g.C, g.eps));
    if (launches) *launches += 1;
    return MUGD_OK;
}

}  // namespace mugd

// Attention of mug/model/attention.py:91-126 (CrossAttention.forward) with both contractions on the tcgen05 tensor
// cores, fp32 in / fp32 out through the same 3xTF32 split as gemm_tc.cu:
//
//     idx_ij = clamp(j - i, -P, P) + P
//     s_ij   = (q_i . k_j + relpos[idx_ij, h]) * scale                 S = Q K^T   : tcgen05.mma, A = Q from TMEM
//     o_i    = sum_j softmax_j(s_i)_j * cgain[idx_ij, h] * v_j         O = P V     : tcgen05.mma, A = P from TMEM
//
// One CTA owns 128 queries of one (sample, head) and streams 128-key tiles (flash style: no [Lq, Lk] matrix in
// memory, running max / sum per query row).  Thread t and thread t+128 share query row (t & 127) = TMEM lane:
//   * Q is split into q_hi / q_lo once and lives in tensor memory for the whole CTA (A operand, "TS" form);
//   * the raw K and V head slices of a key tile arrive by TMA (3-D tensor maps (channel, key, sample), 128B swizzle,
//     keys past Lk zero-filled by the TMA bounds check), one tile ahead of the math when two stages fit (head dim 32);
//     the key tile is split in place into k_hi / k_lo (row = key, 128 bytes of channels: the K-major B operand of
//     S = Q K^T); the value tile is split and transposed shared -> shared into V^T hi / lo (row = channel, keys
//     contiguous: the K-major B operand of O = P V) -- tcgen05 takes MN-major TF32 operands only in a different
//     swizzle, so the transpose is done by hand, one conflict-free 32-key x 4-channel block per warp step;
//   * S lands in TMEM columns [0,128); each thread pulls its half of the row into registers, applies the
//     relative-position bias, scale and key mask, and the two halves combine max / sum through shared memory;
//   * P * gain is split into hi / lo and written back to tensor memory (hi over the S columns it came from, lo next
//     to it): the second MMA consumes it from there, so P never touches shared or global memory;
//   * the per-tile O lands in TMEM and is folded into the register accumulator with the usual exp(m_old - m_new).
// The FFMA kernel in attention.cu stays as the exact-fp32 referee (mugd_set_attention_impl(0)).
#include <cuda.h>

#include "common.cuh"

#include <math.h>

namespace mugd {
namespace atc {

constexpr int THREADS = 256;
constexpr int BQ = 128;
constexpr int BKV = 128;
constexpr uint32_t SLAB = BKV * 128;          // 128 keys x (32 fp32 channels = 128 B): one swizzle-atom column of a tile

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
// bounded wait: a protocol bug traps (CUDA error) instead of hanging the GPU
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t done = 0;
    const long long t0 = clock64();
    while (true) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(bar), "r"(parity)
            : "memory");
        if (done) break;
        if (clock64() - t0 > 4000000000LL) __trap();
    }
}
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1, int c2) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
        ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1), "r"(c2)
        : "memory");
}
__device__ __forceinline__ void umma_tf32_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}"
        ::"r"(d_tmem), "r"(a_tmem), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// one lane of a converged warp (see gemm_tc.cu: uniform-datapath instructions must not sit in a lane-divergent branch)
__device__ __forceinline__ bool elect_one() {
    uint32_t pred = 0;
    asm volatile(
        "{\n\t.reg .b32 rx;\n\t.reg .pred px;\n\t"
        "elect.sync rx|px, 0xffffffff;\n\t"
        "selp.u32 %0, 1, 0, px;\n\t}"
        : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// K-major SWIZZLE_128B shared-memory matrix descriptor (cute::UMMA::SmemDescriptor bit layout, version 1, same encoding as
// gemm_tc.cu): rows of 128 bytes, 8-row groups 1024 B apart (SBO), LBO unused.
__device__ __forceinline__ uint64_t umma_desc_kmajor(uint32_t saddr) {
    return (uint64_t)((saddr >> 4) & 0x3FFFu) | (1ull << 16) | (64ull << 32) | (1ull << 46) | (2ull << 61);
}
__device__ __forceinline__ float to_tf32(float x) {
    uint32_t r;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
    return __uint_as_float(r);
}
// 8 consecutive 32-bit TMEM columns of this thread's lane
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, float* v) {
    uint32_t r[8];
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr));
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const float* v) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};"
                 ::"r"(taddr), "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])),
                   "r"(__float_as_uint(v[3])), "r"(__float_as_uint(v[4])), "r"(__float_as_uint(v[5])),
                   "r"(__float_as_uint(v[6])), "r"(__float_as_uint(v[7]))
                 : "memory");
}
__device__ __forceinline__ void fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ float4 lds_f4(uint32_t addr) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
    return v;
}
__device__ __forceinline__ void sts_f1(uint32_t addr, float v) {
    asm volatile("st.shared.f32 [%0], %1;" ::"r"(addr), "f"(v) : "memory");
}
__device__ __forceinline__ void sts_f4(uint32_t addr, float4 v) {
    asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}

template <int D>
struct Smem {
    static constexpr int KSLABS = (D + 31) / 32;           // 32-channel slabs per head slice (head dim 48: 1.5 used)
    static constexpr int STAGES = (D == 64) ? 1 : 2;       // two key tiles in flight do not fit for head dim 64
    static constexpr uint32_t OPER = KSLABS * SLAB;        // one [128 keys x head slice] tile
    static constexpr uint32_t STAGE_BYTES = 2 * OPER;      // k raw -> k_hi in place | v raw
    static constexpr uint32_t VT_SLAB = D * 128;           // V^T: D channel rows x (32 keys = 128 B)
    static constexpr uint32_t VT_BYTES = (BKV / 32) * VT_SLAB;
    static constexpr uint32_t TILE_BYTES = STAGES * STAGE_BYTES + OPER + 2 * VT_BYTES;   // + k_lo + V^T hi + V^T lo
    static constexpr uint32_t AUX_BYTES = 64 + 4 * BQ * 4; // mbarriers + tmem slot | mx[2][128] rs[2][128]
    static size_t total(int pos_max) { return TILE_BYTES + AUX_BYTES + 2 * (2 * pos_max + 1) * 4 + 1024; }
};

template <int D>
__global__ void __launch_bounds__(THREADS, 1)
attention_tc_kernel(const __grid_constant__ CUtensorMap tmK, const __grid_constant__ CUtensorMap tmV, const mugd_attention a) {
    using S = Smem<D>;
    constexpr int HC = D / 2;                               // Q / O columns owned by one thread of a row pair
    constexpr int STAGES = S::STAGES;
    constexpr uint32_t TM_S = 0, TM_PLO = 128, TM_O = 256, TM_QHI = 320, TM_QLO = 384, TM_COLS = 512;
    extern __shared__ uint8_t smem_raw[];
    const uint32_t raw = smem_u32(smem_raw);
    const uint32_t base = (raw + 1023u) & ~1023u;           // SWIZZLE_128B operands need 1024-byte alignment
    auto k_hi = [&](int s) { return base + (uint32_t)s * S::STAGE_BYTES; };
    auto v_raw = [&](int s) { return base + (uint32_t)s * S::STAGE_BYTES + S::OPER; };
    const uint32_t k_lo = base + STAGES * S::STAGE_BYTES, vt_hi = k_lo + S::OPER, vt_lo = vt_hi + S::VT_BYTES;
    const uint32_t aux = base + S::TILE_BYTES;
    auto bar_full = [&](int s) { return aux + 8u * s; };
    const uint32_t bar_s = aux + 16, bar_o = aux + 24, tmem_slot = aux + 32;
    float* red = reinterpret_cast<float*>(smem_raw + (aux - raw) + 64);   // mx[2][128], rs[2][128]
    float* rel = red + 4 * BQ;
    const int P = a.pos_max, NT = 2 * P + 1;
    float* cg = rel + NT;

    const int tid = threadIdx.x, warp = tid >> 5;
    const int g = tid >> 7, r = tid & 127;                  // thread group (column half), query row = TMEM lane
    const int b = blockIdx.z, h = blockIdx.y, q0 = blockIdx.x * BQ;
    const int ntiles = (a.Lk + BKV - 1) / BKV;

    if (tid == 0) {
        for (int s = 0; s < STAGES; ++s) mbar_init(bar_full(s), 1);
        mbar_init(bar_s, 1);
        mbar_init(bar_o, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"(TM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    fence_before();
    __syncthreads();
    fence_after();
    uint32_t tmem_base;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));
    const uint32_t lane_addr = tmem_base + ((uint32_t)((warp & 3) * 32) << 16);
    pdl_wait();

    // raw K / V head slices of key tile t -> stage t % STAGES (keys >= Lk and channels >= H*D arrive as zeros)
    auto issue_tile = [&](int t) {
        const int s = t % STAGES;
        mbar_expect_tx(bar_full(s), 2u * S::OPER);
#pragma unroll
        for (int sl = 0; sl < S::KSLABS; ++sl) {
            tma_load_3d(k_hi(s) + sl * SLAB, &tmK, bar_full(s), h * D + sl * 32, t * BKV, b);
            tma_load_3d(v_raw(s) + sl * SLAB, &tmV, bar_full(s), h * D + sl * 32, t * BKV, b);
        }
    };
    if (warp == 0) {
        if (elect_one()) {
            issue_tile(0);
            if (STAGES > 1 && ntiles > 1) issue_tile(1);
        }
        __syncwarp();
    }
    for (int t = tid; t < NT; t += THREADS) {
        rel[t] = a.relpos[t * a.H + h] * a.scale;      // (s + rel) * scale == fma(s, scale, rel * scale) up to one rounding
        cg[t] = a.cgain[t * a.H + h];
    }
    // ---- Q row half -> q_hi / q_lo in tensor memory --------------------------------------------------------
    const int qi = q0 + r;
    {
        const float* qp = a.q + ((int64_t)b * a.Lq + qi) * a.ldq + h * D + g * HC;
#pragma unroll
        for (int c = 0; c < HC / 8; ++c) {
            float hi[8], lo[8];
            float4 x0 = make_float4(0.f, 0.f, 0.f, 0.f), x1 = x0;
            if (qi < a.Lq) { x0 = ld_f4(qp + c * 8); x1 = ld_f4(qp + c * 8 + 4); }
            const float x[8] = {x0.x, x0.y, x0.z, x0.w, x1.x, x1.y, x1.z, x1.w};
#pragma unroll
            for (int j = 0; j < 8; ++j) { hi[j] = to_tf32(x[j]); lo[j] = to_tf32(x[j] - hi[j]); }
            tmem_st8(lane_addr + TM_QHI + g * HC + c * 8, hi);
            tmem_st8(lane_addr + TM_QLO + g * HC + c * 8, lo);
        }
        tmem_wait_st();
    }
    float m_i = -INFINITY, l_i = 0.f, o[HC];
#pragma unroll
    for (int c = 0; c < HC; ++c) o[c] = 0.f;
    // instruction descriptor: D=F32 [4,6)=1, A=TF32 [7,10)=2, B=TF32 [10,13)=2, K-major A/B, N>>3 at [17,23), M>>4 at [24,29)
    const uint32_t idesc0 = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(BQ >> 4) << 24);
    uint32_t ph = 0;

    for (int t = 0; t < ntiles; ++t) {
        const int s = t % STAGES;
        const int j0 = t * BKV;
        const int nk = min(BKV, a.Lk - j0);
        const int NK = (nk + 15) & ~15;                     // MMA N (S) and K extent (PV): padded keys are zero / masked
        mbar_wait(bar_full(s), (uint32_t)(t / STAGES) & 1u);
        // ---- key tile: raw -> k_hi in place, k_lo beside it (elementwise, so swizzle-agnostic) -------------------
        for (int f = tid; f < S::KSLABS * 1024; f += THREADS) {
            const int row = (f & 1023) >> 3;                // key within the tile
            if (row >= NK) continue;
            float4 x = lds_f4(k_hi(s) + (uint32_t)f * 16u);
            if (row >= nk) x = make_float4(0.f, 0.f, 0.f, 0.f);
            float4 hi, lo;
            hi.x = to_tf32(x.x); hi.y = to_tf32(x.y); hi.z = to_tf32(x.z); hi.w = to_tf32(x.w);
            lo.x = to_tf32(x.x - hi.x); lo.y = to_tf32(x.y - hi.y); lo.z = to_tf32(x.z - hi.z); lo.w = to_tf32(x.w - hi.w);
            sts_f4(k_hi(s) + (uint32_t)f * 16u, hi);
            sts_f4(k_lo + (uint32_t)f * 16u, lo);
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy smem writes -> visible to the MMA / TMA
        fence_before();
        __syncthreads();
        // ---- S = Q K^T ----------------------------------------------------------------------------------------
        if (warp == 0) {
            fence_after();
            if (elect_one()) {
            const uint32_t idesc = idesc0 | ((uint32_t)(NK >> 3) << 17);
#pragma unroll
            for (int kk = 0; kk < D / 8; ++kk) {
                const uint32_t so = (uint32_t)(kk >> 2) * SLAB;
                const uint64_t ko = (uint64_t)((kk & 3) * 2);          // 8 channels = 32 bytes = 2 x 16-byte units
                const uint64_t dh = umma_desc_kmajor(k_hi(s) + so) + ko, dl = umma_desc_kmajor(k_lo + so) + ko;
                umma_tf32_ts(tmem_base + TM_S, tmem_base + TM_QLO + kk * 8, dh, idesc, kk > 0 ? 1u : 0u);
                umma_tf32_ts(tmem_base + TM_S, tmem_base + TM_QHI + kk * 8, dl, idesc, 1u);
                umma_tf32_ts(tmem_base + TM_S, tmem_base + TM_QHI + kk * 8, dh, idesc, 1u);
            }
            umma_commit(bar_s);
            }
            __syncwarp();
        }
        // ---- value tile (needed by the SECOND contraction only, so it is prepared while the tensor cores work on S): split + transpose
        // into V^T (row = channel, 32-key slabs).  One warp step = 32 keys x one 16-byte channel chunk: the reads hit 8 distinct
        // swizzled chunks per quarter warp and the 32 lanes of each scalar store fill one 128-byte row, so both sides are
        // bank-conflict free.
        for (int it = warp; it < D; it += THREADS / 32) {
            const int kg = it / (D / 4), c = it - kg * (D / 4);
            const int key = kg * 32 + (tid & 31);
            if (key >= NK) continue;
            float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
            if (key < nk) x = lds_f4(v_raw(s) + (uint32_t)(c >> 3) * SLAB + (uint32_t)key * 128u + (uint32_t)(((c & 7) ^ (key & 7)) << 4));
            const float xs[4] = {x.x, x.y, x.z, x.w};
            const uint32_t col = (uint32_t)kg * S::VT_SLAB + (uint32_t)((key & 3) << 2);
            const int kc = (key & 31) >> 2;                 // 16-byte chunk of this key inside its 32-key slab row
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int d = c * 4 + j;
                const float hi = to_tf32(xs[j]), lo = to_tf32(xs[j] - hi);
                const uint32_t off = col + (uint32_t)d * 128u + (uint32_t)((kc ^ (d & 7)) << 4);
                sts_f1(vt_hi + off, hi);
                sts_f1(vt_lo + off, lo);
            }
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // V^T writes -> visible to the PV MMAs (issued behind the next barriers)
        mbar_wait(bar_s, ph);
        fence_after();
        // ---- bias, scale, mask, online softmax on this thread's half of the row (logits stay in registers) -------
        const int split = min(NK, ((NK >> 4) + 1) / 2 * 16);
        const int c_lo = g == 0 ? 0 : split, c_hi = g == 0 ? split : NK;
        float sv[64];
        float mx = -INFINITY;
#pragma unroll
        for (int ci = 0; ci < 4; ++ci) {
            const int c0 = c_lo + ci * 16;
            if (c0 < c_hi) {                                // uniform over the warp (g, NK are)
                float v[16];
                tmem_ld8(lane_addr + TM_S + c0, v);
                tmem_ld8(lane_addr + TM_S + c0 + 8, v + 8);
                tmem_wait_ld();
#pragma unroll
                for (int j = 0; j < 16; ++j) {
                    const int kj = j0 + c0 + j;
                    const int idx = max(-P, min(P, kj - qi)) + P;
                    const float sc = (kj < a.Lk) ? fmaf(v[j], a.scale, rel[idx]) : -INFINITY;
                    sv[ci * 16 + j] = sc;
                    mx = fmaxf(mx, sc);
                }
            }
        }
        red[g * BQ + r] = mx;
        __syncthreads();
        const float mnew = fmaxf(m_i, fmaxf(red[r], red[BQ + r]));     // finite: key j0 is always valid
        const float corr = expf(m_i - mnew);
        float rs = 0.f;
#pragma unroll
        for (int ci = 0; ci < 4; ++ci) {
            const int c0 = c_lo + ci * 16;
            if (c0 < c_hi) {
                float phi[16], plo[16];
#pragma unroll
                for (int j = 0; j < 16; ++j) {
                    const int idx = max(-P, min(P, j0 + c0 + j - qi)) + P;
                    const float pe = expf(sv[ci * 16 + j] - mnew);      // 0 for masked keys
                    rs += pe;
                    const float pg = pe * cg[idx];
                    phi[j] = to_tf32(pg);
                    plo[j] = to_tf32(pg - phi[j]);
                }
                tmem_st8(lane_addr + TM_S + c0, phi);                   // p_hi overwrites the logits it was made from
                tmem_st8(lane_addr + TM_S + c0 + 8, phi + 8);
                tmem_st8(lane_addr + TM_PLO + c0, plo);
                tmem_st8(lane_addr + TM_PLO + c0 + 8, plo + 8);
            }
        }
        tmem_wait_st();
        red[2 * BQ + g * BQ + r] = rs;
        fence_before();
        __syncthreads();
        l_i = l_i * corr + (red[2 * BQ + r] + red[3 * BQ + r]);
        m_i = mnew;
        // ---- O_tile = P V ----------------------------------------------------------------------------------------
        if (warp == 0) {
            fence_after();
            if (elect_one()) {
            const uint32_t idesc = idesc0 | ((uint32_t)(D >> 3) << 17);
            for (int kk = 0; kk < NK / 8; ++kk) {
                const uint32_t so = (uint32_t)(kk >> 2) * S::VT_SLAB;
                const uint64_t ko = (uint64_t)((kk & 3) * 2);           // 8 keys = 32 bytes = 2 x 16-byte units
                const uint64_t dh = umma_desc_kmajor(vt_hi + so) + ko, dl = umma_desc_kmajor(vt_lo + so) + ko;
                umma_tf32_ts(tmem_base + TM_O, tmem_base + TM_PLO + kk * 8, dh, idesc, kk > 0 ? 1u : 0u);
                umma_tf32_ts(tmem_base + TM_O, tmem_base + TM_S + kk * 8, dl, idesc, 1u);
                umma_tf32_ts(tmem_base + TM_O, tmem_base + TM_S + kk * 8, dh, idesc, 1u);
            }
            umma_commit(bar_o);
            }
            __syncwarp();
        }
        mbar_wait(bar_o, ph);
        fence_after();
        // every MMA that read stage s has retired: refill it (the split's generic writes were fenced above)
        if (warp == 0 && t + STAGES < ntiles) {
            __syncwarp();
            if (elect_one()) issue_tile(t + STAGES);
            __syncwarp();
        }
#pragma unroll
        for (int c = 0; c < HC / 8; ++c) {
            float ot[8];
            tmem_ld8(lane_addr + TM_O + g * HC + c * 8, ot);
            tmem_wait_ld();
#pragma unroll
            for (int j = 0; j < 8; ++j) o[c * 8 + j] = fmaf(o[c * 8 + j], corr, ot[j]);
        }
        ph ^= 1u;
        fence_before();                                     // orders these TMEM reads before the next tile's MMAs
    }
    if (qi < a.Lq) {
        const float inv = 1.0f / l_i;
        float* op = a.o + ((int64_t)b * a.Lq + qi) * a.ldo + h * D + g * HC;
#pragma unroll
        for (int c = 0; c < HC / 4; ++c)
            st_f4(op + c * 4, make_float4(o[c * 4] * inv, o[c * 4 + 1] * inv, o[c * 4 + 2] * inv, o[c * 4 + 3] * inv));
    }
    fence_before();
    __syncthreads();
    if (warp == 0) {
        fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TM_COLS) : "memory");
    }
}

// (channel, key, sample) view of a [B*Lk, ld] row-major buffer whose first H*D columns are the head slices
static int encode_kv(EncodeTiledFn enc, CUtensorMap* tm, const float* p, int64_t ld, int cols, int Lk, int B) {
    cuuint64_t dims[3] = {(cuuint64_t)cols, (cuuint64_t)Lk, (cuuint64_t)B};
    cuuint64_t strides[2] = {(cuuint64_t)ld * 4, (cuuint64_t)Lk * (cuuint64_t)ld * 4};
    cuuint32_t box[3] = {32, (cuuint32_t)BKV, 1};
    cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = enc(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float*>(p), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    MUGD_REQUIRE(r == CUDA_SUCCESS, "attention_tc: cuTensorMapEncodeTiled failed with %d (cols=%d Lk=%d B=%d ld=%lld)", (int)r, cols, Lk, B,
                 (long long)ld);
    return MUGD_OK;
}

template <int D>
static int launch(const DeviceInfo& dev, const mugd_attention& a, cudaStream_t st) {
    EncodeTiledFn enc = get_encode();
    MUGD_REQUIRE(enc != nullptr, "attention_tc: cuTensorMapEncodeTiled entry point not available");
    CUtensorMap tmK, tmV;
    int rc = encode_kv(enc, &tmK, a.k, a.ldk, a.H * D, a.Lk, a.B);
    if (rc != MUGD_OK) return rc;
    rc = encode_kv(enc, &tmV, a.v, a.ldv, a.H * D, a.Lk, a.B);
    if (rc != MUGD_OK) return rc;
    const size_t bytes = Smem<D>::total(a.pos_max);
    MUGD_REQUIRE(bytes <= (size_t)dev.max_smem_optin, "attention_tc: pos_max=%d needs %zu B of shared memory (max %d)", a.pos_max, bytes,
                 dev.max_smem_optin);
    dim3 grid((a.Lq + BQ - 1) / BQ, a.H, a.B);
    MUGD_CHECK_CUDA(launch_k(attention_tc_kernel<D>, grid, dim3(THREADS), bytes, st, tmK, tmV, a));
    return MUGD_OK;
}

}  // namespace atc

// the byte count grows with pos_max: allow what the device allows, the launcher checks each launch against it
int configure_attention_tc_kernels(const DeviceInfo& dev) {
    MUGD_CHECK_CUDA(cudaFuncSetAttribute(atc::attention_tc_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, dev.max_smem_optin));
    MUGD_CHECK_CUDA(cudaFuncSetAttribute(atc::attention_tc_kernel<48>, cudaFuncAttributeMaxDynamicSharedMemorySize, dev.max_smem_optin));
    MUGD_CHECK_CUDA(cudaFuncSetAttribute(atc::attention_tc_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, dev.max_smem_optin));
    return MUGD_OK;
}

int launch_attention_tc(const DeviceInfo& dev, const mugd_attention& a, cudaStream_t st) {
    return (a.D == 32) ? atc::launch<32>(dev, a, st) : (a.D == 48) ? atc::launch<48>(dev, a, st) : atc::launch<64>(dev, a, st);
}

}  // namespace mugd

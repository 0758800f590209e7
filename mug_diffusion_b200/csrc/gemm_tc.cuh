// Device side of the tcgen05 (5th-generation tensor core) implicit GEMM, shared by the stand-alone kernels of gemm_tc.cu and any
// kernel that embeds GEMM tiles.  fp32 in / fp32 out with the 3xTF32 split so results stay at fp32 accuracy
// (DESIGN.md §4 "Precision"):
//
//     a = a_hi + a_lo (both exactly representable in TF32, round-to-nearest),   w = w_hi + w_lo
//     acc += a_lo*w_hi + a_hi*w_lo + a_hi*w_hi          (fp32 accumulation in TMEM, dropped term ~2^-22)
//
// One call of gemm_tc_tile<BN>() computes one 128 x BN output tile (or its split-K partial) with the 8 warps of a CTA:
//   warp 0      TMA producer : per k-step (32 fp32 = one 128-byte swizzle row) loads the raw A tile through a 3-D tensor map
//                              (k, l, b) -- the conv k=3 halo is the TMA out-of-bounds zero fill on the l axis, so no im2col /
//                              padding copy exists -- plus the pre-split W_hi / W_lo tiles; completion on an mbarrier.
//   warp 3      second producer (256-wide tiles only: the weight ring is decoupled from the activation ring)
//   warps 4-7   converter    : thread = tile row = TMEM lane; splits the raw row into a_hi / a_lo (cvt.rna.tf32) and writes them
//                              straight into tensor memory (tcgen05.st); the MMAs take A from TMEM (".kind::tf32" TS form).
//   warp 1      MMA issuer   : one elected lane issues 12 tcgen05.mma.kind::tf32 (M128 x BN x K8) per k-step; tcgen05.commit
//                              releases the stage and, after the last k-step, hands the accumulator to the epilogue.
//   warps 4-7   epilogue 1   : tcgen05.ld 32x32b -> shared memory (row pitch BN+4)
//   all warps   epilogue 2   : bias / time-embedding row / SiLU / GELU / GEGLU / GLU / residual, row-contiguous coalesced stores;
//                              with split-K the partial tile goes to an L2-resident workspace and tc_reduce_item() sums the
//                              splits in fixed order (deterministic) and runs the same fused epilogue.
//
// Variants that were built and measured slower on B200 in round 1 (operands both from shared memory, weight-tile TMA multicast over
// clusters, split-K reduction through DSMEM / by the last-arriving CTA / by a cooperative rendezvous, explicit PDL triggers) were
// removed in round 2; their numbers stay in DESIGN.md §4.
#pragma once
#include <cuda.h>

#include <type_traits>

#include "common.cuh"

namespace mugd {

constexpr int TC_BM = 128;
constexpr int TC_BK = 32;                 // fp32 elements per k-step = 128 bytes = one swizzle row
constexpr int TC_THREADS = 256;
constexpr uint32_t TC_A_BYTES = TC_BM * TC_BK * 4;   // 16 KB

struct TcParams {
    // What the tile prologue and the TMA producer read before the first load leaves, packed into the first 64 bytes: kernel
    // parameters live in constant memory, a fresh launch misses on every line it touches, and those misses are serial on the
    // producer's critical path (tools/gemm_timeline.py: ~0.4 us between kernel entry and the first TMA were parameter fetches).
    struct Hot {
        int32_t Lrows, Bs, box_l, box_b, tiles_per_sample, it_base, it_rem, it_main, kblocks, total_it, splits, single_pass,
            conv_mode, tap_shift, tap_dilation, gx;
    } hot;
    mugd_gemm g;
    float* ws;                // split-K partial tiles [tile][split][128][BN]
    int32_t splits;
    int32_t total_it;         // (taps * K + K2) / 32
    int32_t kblocks;          // K / 32
    int32_t it_main;          // taps * K / 32: k-steps >= it_main read the second source (A2, 1x1 term)
    int32_t Lrows, Bs;        // row structure of the A tensor map (Lrows = rows per sample, Bs samples)
    int32_t box_l, box_b;     // TMA box: box_l rows of box_b consecutive samples (box_l*box_b <= 128)
    int32_t tiles_per_sample; // when Lrows >= 128
    int32_t single_pass;      // 1: plain TF32 (a_hi*w_hi only, ~2^-11 relative) -- opt-in speed mode, NOT used for parity/bench
    int32_t BN, gx, gy;       // tile width and tile grid (gx column tiles x gy row tiles x splits)
    int32_t occ;              // CTAs per SM the kernel variant is built for (1; 2 = the two-stage 128-wide variant)
    int32_t sm_count;
    double ln_invK;           // 1 / K (folded LayerNorm: moments -> mean / variance)
    int32_t it_base, it_rem;  // split z owns k-steps [z*it_base + min(z, it_rem), +it_base + (z < it_rem)): no division on the device
#ifdef MUGD_TC_TIMELINE
    long long* dbg;           // CTA (0,0,0) writes globaltimer stamps (tools/gemm_timeline.py)
#endif
};

#ifdef __CUDACC__
// ---- raw PTX helpers ---------------------------------------------------------------------------------
__device__ __forceinline__ long long gtimer() {
    long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t) :: "memory");
    return t;
}
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_inval(uint32_t bar) {
    asm volatile("mbarrier.inval.shared::cta.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
// bounded wait: a protocol bug traps (CUDA error) instead of hanging the GPU
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t done = 0;
    long long t0 = 0;                 // the clock is read only after a probe has failed: the common case costs one try_wait
    while (true) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(bar), "r"(parity)
            : "memory");
        if (done) break;
        const long long now = clock64();
        if (t0 == 0) t0 = now;
        else if (now - t0 > 4000000000LL) __trap();
    }
}
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1, int c2) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
        ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1), "r"(c2)
        : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1)
        : "memory");
}
// A operand from tensor memory (lane = row, one 32-bit column per K element), B from shared memory
__device__ __forceinline__ void umma_tf32_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}"
        ::"r"(d_tmem), "r"(a_tmem), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const float* v) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
        "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
        "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
        ::"r"(taddr), "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])), "r"(__float_as_uint(v[3])),
          "r"(__float_as_uint(v[4])), "r"(__float_as_uint(v[5])), "r"(__float_as_uint(v[6])), "r"(__float_as_uint(v[7])),
          "r"(__float_as_uint(v[8])), "r"(__float_as_uint(v[9])), "r"(__float_as_uint(v[10])), "r"(__float_as_uint(v[11])),
          "r"(__float_as_uint(v[12])), "r"(__float_as_uint(v[13])), "r"(__float_as_uint(v[14])), "r"(__float_as_uint(v[15])),
          "r"(__float_as_uint(v[16])), "r"(__float_as_uint(v[17])), "r"(__float_as_uint(v[18])), "r"(__float_as_uint(v[19])),
          "r"(__float_as_uint(v[20])), "r"(__float_as_uint(v[21])), "r"(__float_as_uint(v[22])), "r"(__float_as_uint(v[23])),
          "r"(__float_as_uint(v[24])), "r"(__float_as_uint(v[25])), "r"(__float_as_uint(v[26])), "r"(__float_as_uint(v[27])),
          "r"(__float_as_uint(v[28])), "r"(__float_as_uint(v[29])), "r"(__float_as_uint(v[30])), "r"(__float_as_uint(v[31]))
        : "memory");
}
// One lane of a converged warp.  tcgen05.mma / tcgen05.commit / cp.async.bulk.tensor are uniform-datapath instructions: issued
// from a lane-divergent branch (`if (lane == 0)`) ptxas wraps every one of them in an elect-and-branch loop (~95 cycles per
// MMA measured, which starved the tensor pipe); guarded by elect.sync in a converged warp they issue back to back.
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
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float* v) {
    uint32_t r[32];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
          "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
          "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ float to_tf32(float x) {
    uint32_t r;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
    return __uint_as_float(r);
}
// K-major, SWIZZLE_128B shared-memory matrix descriptor (cute::UMMA::SmemDescriptor bit layout):
// start>>4 [0,14) | LBO>>4 [16,30) (unused for swizzled K-major, 1) | SBO>>4 [32,46) = 1024 B between 8-row
// groups | version=1 [46,48) | layout_type=SWIZZLE_128B(2) [61,64)
__device__ __forceinline__ uint64_t umma_desc(uint32_t saddr) {
    return (uint64_t)((saddr >> 4) & 0x3FFFu) | (1ull << 16) | (64ull << 32) | (1ull << 46) | (2ull << 61);
}

// OCC = CTAs resident per SM.  OCC 2 (128-wide tiles only) halves the pipeline to two 48 KB stages and the tensor memory to 256
// columns so that TWO CTAs share an SM: the same four stages are in flight per SM, but while one CTA drains its accumulator
// (tcgen05.ld, bias / activation / gate math, global stores: 3-4 us in which its tensor pipe used to idle) the other one's main
// loop keeps the tensor cores busy.  For GEMMs with more tiles than SMs (big batches).
template <int BN, int OCC = 1>
struct TcSmem {
    static_assert(OCC == 1 || (OCC == 2 && BN == 128), "two CTAs per SM exist for 128-wide tiles");
    static constexpr uint32_t B_BYTES = BN * TC_BK * 4;
    static constexpr uint32_t STAGE_BYTES = TC_A_BYTES + 2 * B_BYTES;     // raw A tile + W_hi + W_lo (a_hi / a_lo live in TMEM)
    static constexpr int STAGES = OCC == 2 ? 2 : ((BN == 256) ? 2 : (BN == 128 ? 4 : 6));
    // Decoupled rings (256-wide tiles): only two 80 KB coupled stages would fit, and tied to the A tile the weight tile sat idle
    // while the activations were fetched and split.  Decoupled, the A side is a 2-deep smem ring feeding a 4-deep ring of TMEM
    // operand slots and runs ahead, and the freed shared memory holds a THIRD weight stage; a weight stage is occupied only from
    // its TMA to the retirement of its MMAs (k-step 1.10 -> 1.00 us on the Beff=64 convs).
    static constexpr bool DEC = BN == 256;
    static constexpr int SAS = DEC ? 2 : STAGES;           // raw activation tiles in shared memory
    static constexpr int SA = DEC ? 4 : STAGES;            // split activation tiles in tensor memory
    static constexpr int SW = DEC ? 3 : STAGES;            // weight stages (hi + lo)
    static constexpr uint32_t TILE_BYTES = DEC ? SAS * TC_A_BYTES + SW * 2 * B_BYTES : STAGES * STAGE_BYTES;
    static constexpr uint32_t BAR_BYTES = 256;
    static constexpr uint32_t TOTAL = TILE_BYTES + 1024 /*align slack*/ + BAR_BYTES;
    static constexpr int TMEM_NEED = BN + SA * 64;         // accumulator + per slot 32 columns a_hi + 32 columns a_lo
    static constexpr int TMEM_COLS = TMEM_NEED <= 64 ? 64 : (TMEM_NEED <= 128 ? 128 : (TMEM_NEED <= 256 ? 256 : 512));
    static_assert(TMEM_NEED <= 512 && TMEM_COLS * OCC <= 512, "tensor memory budget");
    static_assert((TOTAL + 1024) * OCC <= 227u * 1024u, "shared memory budget");
    static_assert(128u * (BN + 4) * 4u + 1024u <= TILE_BYTES, "the staged accumulator tile + row statistics must fit the pipeline buffers");
};

// ---- row moments of the OUTPUT for the LayerNorm that follows, accumulated while the tile is written (mugd_gemm.row_moments) ----
// The SEG lanes that hold one output row of this tile reduce with shuffles (fp32: at
// most 128 values), the segment leader adds the tile's share of the row to the row's two doubles -- one address per row, so no
// contention.  Every lane of the warp must call it (inactive: v = 0, m < 0).
template <int SEG>
__device__ __forceinline__ void tc_row_sink(double* buf, int m, float4 v) {
    float s = (v.x + v.y) + (v.z + v.w);
    float ss = (v.x * v.x + v.y * v.y) + (v.z * v.z + v.w * v.w);
#pragma unroll
    for (int o = SEG / 2; o > 0; o >>= 1) {
        s += __shfl_xor_sync(0xffffffffu, s, o);
        ss += __shfl_xor_sync(0xffffffffu, ss, o);
    }
    if ((threadIdx.x & (SEG - 1)) == 0 && m >= 0) {
        atomicAdd(buf + (int64_t)m * 2, (double)s);
        atomicAdd(buf + (int64_t)m * 2 + 1, (double)ss);
    }
}
// mean / rstd of a row from its two moments (LayerNorm folded into the GEMM, mugd_gemm.ln_stats).  The variance is formed in fp64
// (E[x^2] - mean^2 cancels), the reciprocal square root in fp32 with one Newton step (~1 ulp): a handful of instructions instead of the
// ~100-deep fp64 divide / sqrt chains, which sat on the critical path between the main loop and the epilogue.
__device__ __forceinline__ float2 tc_ln_from_moments(double s, double ss, double invK, float eps) {
    const double mean = s * invK;
    double var = ss * invK - mean * mean;
    const float v = fmaxf((float)var, 0.f) + eps;
    float r = rsqrtf(v);
    r = r * (1.5f - 0.5f * v * r * r);
    return make_float2((float)mean, r);
}

// epilogue modes of a tile / reduce pass
constexpr int TC_EPI_PLAIN = 0, TC_EPI_SINK = 1 /* act == gate == NONE + row moments of the output */, TC_EPI_LN = 2 /* LayerNorm folded in */;

// Fused epilogue math on 4 consecutive accumulator columns.  ACT / GATE are compile-time so that the compiler
// cannot if-convert the branches into "compute SiLU, GELU and both gates for every element, then select"
// (which it did, costing ~4 us per tile); callers dispatch once per tile on the (uniform) act/gate values.
// LNF: acc is A W'^T of the un-normalised rows; (acc - mean*colsum)*rstd is the product with the LayerNorm'd rows.
// Returns the stored float4 (GATE_NONE) for the row-moment sink.
template <int ACT, int GATE, bool LNF>
__device__ __forceinline__ float4 tc_finish4(const mugd_gemm& g, float* dst, float4 acc, float4 bia, float4 rvv, float4 res, float4 cs, float2 ln,
                                             int m, int no) {
    // dst = &C[m][no]  (no = output column: the accumulator column, or half of it for gated epilogues)
    float x[4];
    if constexpr (LNF) {
        x[0] = (acc.x - ln.x * cs.x) * ln.y + bia.x + rvv.x; x[1] = (acc.y - ln.x * cs.y) * ln.y + bia.y + rvv.y;
        x[2] = (acc.z - ln.x * cs.z) * ln.y + bia.z + rvv.z; x[3] = (acc.w - ln.x * cs.w) * ln.y + bia.w + rvv.w;
    } else {
        x[0] = acc.x + bia.x + rvv.x; x[1] = acc.y + bia.y + rvv.y; x[2] = acc.z + bia.z + rvv.z; x[3] = acc.w + bia.w + rvv.w;
    }
    if constexpr (ACT == MUGD_ACT_SILU) {
#pragma unroll
        for (int j = 0; j < 4; ++j) x[j] = silu_f(x[j]);
    } else if constexpr (ACT == MUGD_ACT_GELU) {
#pragma unroll
        for (int j = 0; j < 4; ++j) x[j] = gelu_f(x[j]);
    }
    if constexpr (GATE == MUGD_GATE_NONE) {
        const float4 o = make_float4(x[0] + res.x, x[1] + res.y, x[2] + res.z, x[3] + res.w);
        st_f4(dst, o);
        return o;
    } else {
        float o0, o1;
        if constexpr (GATE == MUGD_GATE_GEGLU) { o0 = x[0] * gelu_f(x[1]); o1 = x[2] * gelu_f(x[3]); }
        else { o0 = x[0] * sigmoid_f(x[1]); o1 = x[2] * sigmoid_f(x[3]); }
        if (g.residual) {
            const float2 rr = *reinterpret_cast<const float2*>(g.residual + (int64_t)m * g.ldr + no);
            o0 += rr.x; o1 += rr.y;
        }
        *reinterpret_cast<float2*>(dst) = make_float2(o0, o1);
        return make_float4(o0, o1, 0.f, 0.f);
    }
}

// phase 2 of the epilogue for one CTA: read the staged accumulator tile from shared memory (row pitch BN+4) and
// finish it with coalesced global traffic; U float4 per thread in flight, every global load issued before any use.
// MODE = TC_EPI_LN reads the (mean, rstd) of tile row r from shared memory at rowstat + 8*r (written in phase 1).
template <int BN, int ACT, int GATE, int MODE, int UMAX = 16>
__device__ __forceinline__ void tc_store_tile(const mugd_gemm& g, uint32_t stage, int m_base, int n0, int rows_valid, const float* rowvec,
                                              uint32_t rowstat, float4 bia, float4 cs) {
    constexpr int SP = BN + 4;
    constexpr int C4 = BN / 4;
    constexpr int NU = TC_BM * C4 / TC_THREADS;          // float4 per thread: 8 / 16 / 32 for BN = 64 / 128 / 256
    constexpr int U = NU < UMAX ? NU : UMAX;             // in flight together (two CTAs per SM: 8, the register file is split in two)
    constexpr int SEG = C4 < 32 ? C4 : 32;
    static_assert(TC_THREADS % C4 == 0, "a thread keeps its column quad for the whole tile");
    // this thread's column quad is the same for every row it visits: bias / column sums (bia, cs) were loaded once, before the main loop
    const int c4 = (int)threadIdx.x % C4;
    const int nn = n0 + c4 * 4;
    const bool col_ok = nn < g.N;
    const bool has_res = GATE == MUGD_GATE_NONE && g.residual != nullptr;
    // Row bookkeeping is incremental (the SASS of the first version spent ~75 instructions per float4 on it: 64-bit address products,
    // an integer division per row for the time-embedding row): a thread's rows are row0, row0 + RPP, ... ; pointers advance by
    // RPP rows; the sample of a row (for the per-sample row vector) is found by ONE division and then by comparison.
    constexpr int RPP = TC_THREADS / C4;                 // rows between two float4s of a thread
    const int row0 = (int)threadIdx.x / C4;
    const int n_rows = min(rows_valid, g.M - m_base);    // rows of this tile that exist
    const int no = (GATE == MUGD_GATE_NONE) ? nn : (nn >> 1);
    float* cp = g.C + (int64_t)(m_base + row0) * g.ldc + no;
    const float* rp = has_res ? g.residual + (int64_t)(m_base + row0) * g.ldr + nn : nullptr;
    const int64_t c_step = (int64_t)RPP * g.ldc, r_step = (int64_t)RPP * g.ldr;
    int smp = 0, smp_end = 0;                            // sample of the current row, first row (tile-relative... absolute m) of the next sample
    if (rowvec) { smp = (m_base + row0) / g.Lout; smp_end = (smp + 1) * g.Lout; }
    // A tile that lies fully inside the matrix (the common case) runs the loop without any per-element predicate, so that the
    // compiler can put all shared-memory reads of a pass in flight; edge tiles take the predicated copy.
    auto pass = [&](auto full_tag) {
        constexpr bool FULL = decltype(full_tag)::value;
#pragma unroll 1
        for (int i0 = 0; i0 < NU; i0 += U) {
            // every global load of this pass is issued before anything is consumed: ONE memory round trip per 16 rows
            float4 res[U], rvv[U];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int row = row0 + (i0 + u) * RPP;
                res[u] = rvv[u] = make_float4(0.f, 0.f, 0.f, 0.f);
                if (FULL || (row < n_rows && col_ok)) {
                    if (has_res) res[u] = ld_f4(rp + (int64_t)(i0 + u) * r_step);
                    if (rowvec) {
                        const int m = m_base + row;
                        while (m >= smp_end) { ++smp; smp_end += g.Lout; }
                        rvv[u] = ld_f4(rowvec + (int64_t)smp * g.rowvec_b_stride + nn);
                    }
                }
            }
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int row = row0 + (i0 + u) * RPP;
                const int m = m_base + row;
                const bool ok = FULL || (row < n_rows && col_ok);
                float4 acc;
                asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(acc.x), "=f"(acc.y), "=f"(acc.z), "=f"(acc.w)
                             : "r"(stage + (uint32_t)(row * SP + c4 * 4) * 4u));
                float2 ln = make_float2(0.f, 1.f);
                if constexpr (MODE == TC_EPI_LN)
                    asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(ln.x), "=f"(ln.y) : "r"(rowstat + (uint32_t)row * 8u));
                float4 o = make_float4(0.f, 0.f, 0.f, 0.f);
                if (ok) o = tc_finish4<ACT, GATE, MODE == TC_EPI_LN>(g, cp + (int64_t)(i0 + u) * c_step, acc, bia, rvv[u], res[u], cs, ln, m, no);
                if constexpr (MODE == TC_EPI_SINK) tc_row_sink<SEG>(g.row_moments, ok ? m : -1, o);
            }
        }
    };
    if (n_rows >= TC_BM && n0 + BN <= g.N) pass(std::true_type{});
    else pass(std::false_type{});
}

// Epilogue variant of a kernel instantiation.  Every variant is its own kernel (template parameter), so a launch only carries the
// store loop it executes: with all eight variants inlined in one kernel the hot kernel grew by 60 % and every GEMM of the step
// got ~0.5 us slower (instruction fetch), fused or not.
enum TcEpi { TC_E_NONE = 0, TC_E_GEGLU, TC_E_GLU, TC_E_SILU, TC_E_GELU, TC_E_SINK, TC_E_LN, TC_E_LN_GEGLU, TC_E_COUNT };
template <int EPI> struct TcEpiTraits;
template <> struct TcEpiTraits<TC_E_NONE>     { static constexpr int ACT = MUGD_ACT_NONE, GATE = MUGD_GATE_NONE,  MODE = TC_EPI_PLAIN; };
template <> struct TcEpiTraits<TC_E_GEGLU>    { static constexpr int ACT = MUGD_ACT_NONE, GATE = MUGD_GATE_GEGLU, MODE = TC_EPI_PLAIN; };
template <> struct TcEpiTraits<TC_E_GLU>      { static constexpr int ACT = MUGD_ACT_NONE, GATE = MUGD_GATE_GLU,   MODE = TC_EPI_PLAIN; };
template <> struct TcEpiTraits<TC_E_SILU>     { static constexpr int ACT = MUGD_ACT_SILU, GATE = MUGD_GATE_NONE,  MODE = TC_EPI_PLAIN; };
template <> struct TcEpiTraits<TC_E_GELU>     { static constexpr int ACT = MUGD_ACT_GELU, GATE = MUGD_GATE_NONE,  MODE = TC_EPI_PLAIN; };
template <> struct TcEpiTraits<TC_E_SINK>     { static constexpr int ACT = MUGD_ACT_NONE, GATE = MUGD_GATE_NONE,  MODE = TC_EPI_SINK; };
template <> struct TcEpiTraits<TC_E_LN>       { static constexpr int ACT = MUGD_ACT_NONE, GATE = MUGD_GATE_NONE,  MODE = TC_EPI_LN; };
template <> struct TcEpiTraits<TC_E_LN_GEGLU> { static constexpr int ACT = MUGD_ACT_NONE, GATE = MUGD_GATE_GEGLU, MODE = TC_EPI_LN; };

inline int tc_epi_of(const mugd_gemm& g) {
    if (g.ln_stats) return g.gate == MUGD_GATE_GEGLU ? TC_E_LN_GEGLU : TC_E_LN;
    if (g.row_moments) return TC_E_SINK;
    if (g.gate == MUGD_GATE_GEGLU) return TC_E_GEGLU;
    if (g.gate == MUGD_GATE_GLU) return TC_E_GLU;
    if (g.act == MUGD_ACT_SILU) return TC_E_SILU;
    if (g.act == MUGD_ACT_GELU) return TC_E_GELU;
    return TC_E_NONE;
}

// rows of output tile `by`
__device__ __forceinline__ void tc_tile_rows(const TcParams& p, int by, int& b_base, int& l_base, int& rows_valid) {
    const TcParams::Hot& h = p.hot;
    if (h.Lrows >= TC_BM) {
        b_base = by / h.tiles_per_sample;
        l_base = (by % h.tiles_per_sample) * TC_BM;
        rows_valid = min(TC_BM, h.Lrows - l_base);
    } else {
        b_base = by * h.box_b;
        l_base = 0;
        rows_valid = min(h.box_b, h.Bs - b_base) * h.Lrows;
    }
}

// Barrier block of one CTA (at base + TILE_BYTES): full[SAS] conv[SA] empty[SA], decoupled rings add afree[SAS] wfull[SW]
// wfree[SW]; then accum and the tmem-pointer slot.
template <int BN, int OCC = 1>
struct TcBars {
    using S = TcSmem<BN, OCC>;
    static constexpr int N_DEC = S::DEC ? S::SAS + 2 * S::SW : 0;
    static constexpr int COUNT = S::SAS + 2 * S::SA + N_DEC + 1;
    static_assert(8 * (COUNT + 1) <= (int)S::BAR_BYTES, "barrier block");
    uint32_t bars;
    __device__ __forceinline__ explicit TcBars(uint32_t base) : bars(base + S::TILE_BYTES) {}
    __device__ __forceinline__ uint32_t full(int s) const { return bars + 8u * s; }                                    // raw A tile (coupled: + W) landed
    __device__ __forceinline__ uint32_t conv(int s) const { return bars + 8u * (S::SAS + s); }                         // split A in its TMEM slot
    __device__ __forceinline__ uint32_t empty(int s) const { return bars + 8u * (S::SAS + S::SA + s); }                // coupled: stage free; decoupled: TMEM slot retired
    __device__ __forceinline__ uint32_t afree(int s) const { return bars + 8u * (S::SAS + 2 * S::SA + s); }            // decoupled: raw A tile consumed
    __device__ __forceinline__ uint32_t wfull(int s) const { return bars + 8u * (2 * S::SAS + 2 * S::SA + s); }        // decoupled: weight stage landed
    __device__ __forceinline__ uint32_t wfree(int s) const { return bars + 8u * (2 * S::SAS + 2 * S::SA + S::SW + s); }
    __device__ __forceinline__ uint32_t accum() const { return bars + 8u * (COUNT - 1); }
    __device__ __forceinline__ uint32_t tmem_slot() const { return bars + 8u * COUNT; }
    // arm every barrier for one tile: thread t (t < COUNT) arms barrier t; call from the first warp(s), then sync the CTA
    __device__ __forceinline__ void init_parallel(int t) const {
        if (t >= COUNT) return;
        uint32_t count = 1;
        if (t >= S::SAS && t < S::SAS + S::SA) count = 4;                                         // conv: one arrival per converter warp
        if (S::DEC && t >= S::SAS + 2 * S::SA && t < 2 * S::SAS + 2 * S::SA) count = 4;           // afree
        mbar_init(bars + 8u * t, count);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
};

// One 128 x BN output tile (bx, by) of split bz.  `base` = 1024-byte aligned shared-memory address of the CTA's tile pool
// (TcSmem<BN>::TILE_BYTES + barrier block), `tmem_base` = allocated tensor memory (>= TcSmem<BN>::TMEM_NEED columns), barriers
// armed by the caller (TcBars::init) and visible to all threads.  All 256 threads call it; on return every TMA has landed, every
// MMA has retired and been observed, and the tile (or its partial) is on its way to global memory.
// The producer side executes griddepcontrol.wait (PDL) before touching activations.
template <int BN, int EPI, int OCC = 1>
__device__ __forceinline__ void gemm_tc_tile(const CUtensorMap* tmA, const CUtensorMap* tmA1, const CUtensorMap* tmA2, const CUtensorMap* tmB,
                                             const CUtensorMap* tmWhi, const CUtensorMap* tmWlo, const TcParams& p, int bx, int by, int bz,
                                             uint32_t base, uint32_t tmem_base, int it0 = 0, uint32_t acc_phase = 0) {
    // it0 / acc_phase: a CTA that runs several tiles one after the other (two-CTAs-per-SM variant) does not re-arm its barriers:
    // the stage rings simply keep turning -- it0 = k-steps this CTA has already pushed through them, acc_phase = tiles done & 1.
    using S = TcSmem<BN, OCC>;
    constexpr bool DEC = S::DEC;
    constexpr int SAS = S::SAS, SA = S::SA, SW = S::SW;
    const TcBars<BN, OCC> B(base);
    auto a_raw = [&](int s) { return DEC ? base + s * TC_A_BYTES : base + s * S::STAGE_BYTES; };
    auto b_hi = [&](int s) { return DEC ? base + SAS * TC_A_BYTES + s * 2 * S::B_BYTES : base + s * S::STAGE_BYTES + TC_A_BYTES; };
    auto b_lo = [&](int s) { return b_hi(s) + S::B_BYTES; };

    const mugd_gemm& g = p.g;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n0 = bx * BN;
    int b_base, l_base, rows_valid;
    tc_tile_rows(p, by, b_base, l_base, rows_valid);
    const int m_base = b_base * p.hot.Lrows + l_base;
    const int it_begin = bz * p.hot.it_base + min(bz, p.hot.it_rem);
    const int nit = p.hot.it_base + (bz < p.hot.it_rem ? 1 : 0);
#ifdef MUGD_TC_TIMELINE
    const bool dbg_cta = p.dbg && bx == 0 && by == 0 && bz == 0;
#define TC_STAMP(cond, slot) do { if (dbg_cta && (cond)) p.dbg[slot] = gtimer(); } while (0)
#else
#define TC_STAMP(cond, slot) do { } while (0)
#endif
    TC_STAMP(threadIdx.x == 0, 1);
    // Epilogue operands that do not depend on the accumulator are requested NOW, so that their memory latency hides behind the main
    // loop: the device step counter (selects the time-embedding row) and this thread's bias / column-sum quad (its column quad is the
    // same for every row of the tile).  Warps 0-3 have nothing else to do with their registers; for warps 4-7 it is 9 registers.
    int epi_step = 0;
    float4 epi_bias = make_float4(0.f, 0.f, 0.f, 0.f), epi_cs = epi_bias;
    auto request_epilogue_operands = [&]() {
        if (p.hot.splits != 1) return;
        const int nn = n0 + ((int)threadIdx.x % (BN / 4)) * 4;
        if (g.step || (g.bias && nn < g.N)) {
            pdl_wait();                                          // the step counter is written by the previous kernels
            if (g.step) epi_step = *g.step;
            if (g.bias && nn < g.N) epi_bias = ld_f4(g.bias + nn);
        }
        if constexpr (TcEpiTraits<EPI>::MODE == TC_EPI_LN) {
            if (nn < g.N) epi_cs = ld_f4(g.ln_colsum + nn);
        }
    };
    if (warp != 0) request_epilogue_operands();      // the producer warp first gets its loads out (it asks after its loop)

    if (warp == 0) {
        // ===================================== TMA producer =====================================
        // the whole warp walks the loop converged; one elected lane issues the copies
        const TcParams::Hot& h = p.hot;
        const uint32_t a_tx = (uint32_t)(h.box_l * h.box_b) * TC_BK * 4;
        const uint32_t w_tx = (h.single_pass ? 1u : 2u) * S::B_BYTES;
        for (int i = 0; i < nit; ++i) {
            const int gi = it0 + i;
            const int s = gi % SAS;
            const uint32_t ph = (uint32_t)(gi / SAS) & 1u;
            if constexpr (DEC) mbar_wait(B.afree(s), ph ^ 1u);
            else mbar_wait(B.empty(s), ph ^ 1u);
            if (elect_one()) {
                TC_STAMP(i < 24, 8 + i * 6 + 5);
                const int it = it_begin + i;
                mbar_expect_tx(B.full(s), DEC ? a_tx : a_tx + w_tx);
                if constexpr (!DEC) {
                    // weights first: they do not depend on the previous kernel / op.  W columns are in k-step order.
                    tma_load_2d(b_hi(s), tmWhi, B.full(s), it * TC_BK, n0);
                    if (!h.single_pass) tma_load_2d(b_lo(s), tmWlo, B.full(s), it * TC_BK, n0);
                }
                if (i == 0) pdl_wait();             // activations written by the previous kernel are touched from here on
                if (it < h.it_main) {
                    const int t = it / h.kblocks;
                    const int kb = it - t * h.kblocks;
                    // row addressing per tap: SAME = l+t-1, TAPS = l+(t+shift)*dilation (zero fill outside the sample by TMA
                    // bounds); DOWN (stride 2, right pad) uses one strided tensor map per tap (row l of map t = source row 2l+t)
                    const CUtensorMap* ma = tmA;
                    int lshift = 0;
                    if (h.conv_mode == MUGD_CONV_SAME) lshift = t - 1;
                    else if (h.conv_mode == MUGD_CONV_TAPS) lshift = (t + h.tap_shift) * (h.tap_dilation > 1 ? h.tap_dilation : 1);
                    else if (h.conv_mode == MUGD_CONV_DOWN) ma = (t == 0) ? tmA : (t == 1 ? tmA1 : tmA2);
                    tma_load_3d(a_raw(s), ma, B.full(s), kb * TC_BK, l_base + lshift, b_base);
                } else {
                    tma_load_3d(a_raw(s), tmB, B.full(s), (it - h.it_main) * TC_BK, l_base, b_base);   // second source: 1x1 term
                }
                TC_STAMP(i < 24, 8 + i * 6 + 0);
            }
            __syncwarp();
        }
        request_epilogue_operands();
    } else if (DEC && warp == 3) {
        // ===================================== weight producer (decoupled rings) ================
        for (int i = 0; i < nit; ++i) {
            const int gi = it0 + i;
            const int s = gi % SW;
            const uint32_t ph = (uint32_t)(gi / SW) & 1u;
            mbar_wait(B.wfree(s), ph ^ 1u);
            if (elect_one()) {
                const int it = it_begin + i;
                mbar_expect_tx(B.wfull(s), (p.single_pass ? 1u : 2u) * S::B_BYTES);
                tma_load_2d(b_hi(s), tmWhi, B.wfull(s), it * TC_BK, n0);
                if (!p.single_pass) tma_load_2d(b_lo(s), tmWlo, B.wfull(s), it * TC_BK, n0);
            }
            __syncwarp();
        }
    } else if (warp == 1) {
        // ===================================== MMA issuer =======================================
        // instruction descriptor (cute::UMMA::InstrDescriptor): D=F32 [4,6)=1, A=TF32 [7,10)=2, B=TF32 [10,13)=2,
        // A/B K-major (bits 15,16 = 0), N>>3 at [17,23), M>>4 at [24,29)
        const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(TC_BM >> 4) << 24);
        for (int i = 0; i < nit; ++i) {
            const int gi = it0 + i;
            const int s = gi % SA;
            const uint32_t ph = (uint32_t)(gi / SA) & 1u;
            const int sw = DEC ? gi % SW : s;
            mbar_wait(B.conv(s), ph);
            if constexpr (DEC) mbar_wait(B.wfull(sw), (uint32_t)(gi / SW) & 1u);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            if (elect_one()) {
                TC_STAMP(i < 24, 8 + i * 6 + 3);
                const uint64_t dbh = umma_desc(b_hi(sw)), dbl = umma_desc(b_lo(sw));
                const uint32_t ta_hi = tmem_base + (uint32_t)(BN + s * 64), ta_lo = ta_hi + 32u;
#pragma unroll
                for (int kk = 0; kk < TC_BK / 8; ++kk) {
                    const uint64_t ko = (uint64_t)(kk * 2);     // 8 fp32 = 32 bytes = 2 x 16-byte units
                    if (p.single_pass) {
                        umma_tf32_ts(tmem_base, ta_hi + kk * 8, dbh + ko, idesc, (i > 0 || kk > 0) ? 1u : 0u);
                    } else {
                        umma_tf32_ts(tmem_base, ta_lo + kk * 8, dbh + ko, idesc, (i > 0 || kk > 0) ? 1u : 0u);
                        umma_tf32_ts(tmem_base, ta_hi + kk * 8, dbl + ko, idesc, 1u);
                        umma_tf32_ts(tmem_base, ta_hi + kk * 8, dbh + ko, idesc, 1u);
                    }
                }
                umma_commit(B.empty(s));                      // stage (decoupled: TMEM operand slot) reusable once these MMAs retire
                if constexpr (DEC) umma_commit(B.wfree(sw));  // ... and the weight stage
                TC_STAMP(i < 24, 8 + i * 6 + 4);
            }
            __syncwarp();
        }
        if (elect_one()) umma_commit(B.accum());
        __syncwarp();
        // drain: observe the release of the last use of every stage, so that no commit is still on its way to a barrier when the
        // caller re-arms them for the next tile (persistent kernel) or the CTA exits
        for (int i = (nit > SA ? nit - SA : 0); i < nit; ++i) mbar_wait(B.empty((it0 + i) % SA), (uint32_t)((it0 + i) / SA) & 1u);
        if constexpr (DEC) {
            for (int i = (nit > SW ? nit - SW : 0); i < nit; ++i) mbar_wait(B.wfree((it0 + i) % SW), (uint32_t)((it0 + i) / SW) & 1u);
        }
    } else if (warp >= 4) {
        // ===================================== converter ========================================
        // LayerNorm folded into this GEMM: fetch the moments of this thread's row now (written by earlier kernels), use them after the loop
        double ln_s = 0.0, ln_ss = 0.0;
        if constexpr (TcEpiTraits<EPI>::MODE == TC_EPI_LN) {
            pdl_wait();
            const int rr = (warp & 3) * 32 + lane;
            if (rr < rows_valid && m_base + rr < g.M) {
                const double2 mo = *reinterpret_cast<const double2*>(g.ln_stats + (int64_t)(m_base + rr) * 2);
                ln_s = mo.x; ln_ss = mo.y;
            }
        }
        for (int i = 0; i < nit; ++i) {
            const int gi = it0 + i;
            const int s = gi % SA;                                    // TMEM operand slot
            const int sm = gi % SAS;                                  // raw tile in shared memory
            mbar_wait(B.full(sm), (uint32_t)(gi / SAS) & 1u);
            if constexpr (DEC) {
                mbar_wait(B.empty(s), ((uint32_t)(gi / SA) & 1u) ^ 1u);  // the MMAs that read TMEM slot s last time have retired
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            }
            TC_STAMP(threadIdx.x == 128 && i < 24, 8 + i * 6 + 1);
            // thread = tile row (= TMEM lane): read the row's 128 bytes out of the 128B-swizzled tile (16-byte chunk c
            // of row r sits at chunk c ^ (r & 7)), split, and store hi / lo to this slot's TMEM columns
            const int r = (warp & 3) * 32 + lane;
            const uint32_t rowaddr = a_raw(sm) + (uint32_t)r * 128u;
            float hi[32], lo[32];
#pragma unroll
            for (int c = 0; c < 8; ++c) {
                float4 x;
                asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(x.x), "=f"(x.y), "=f"(x.z), "=f"(x.w)
                             : "r"(rowaddr + (uint32_t)((c ^ (r & 7)) * 16)));
                hi[c * 4] = to_tf32(x.x); hi[c * 4 + 1] = to_tf32(x.y); hi[c * 4 + 2] = to_tf32(x.z); hi[c * 4 + 3] = to_tf32(x.w);
                lo[c * 4] = to_tf32(x.x - hi[c * 4]); lo[c * 4 + 1] = to_tf32(x.y - hi[c * 4 + 1]);
                lo[c * 4 + 2] = to_tf32(x.z - hi[c * 4 + 2]); lo[c * 4 + 3] = to_tf32(x.w - hi[c * 4 + 3]);
            }
            const uint32_t ta = tmem_base + ((uint32_t)((warp & 3) * 32) << 16) + (uint32_t)(BN + s * 64);
            tmem_st32(ta, hi);
            tmem_st32(ta + 32u, lo);
            asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            __syncwarp();
            if (lane == 0) {
                mbar_arrive(B.conv(s));
                if constexpr (DEC) mbar_arrive(B.afree(sm));          // the raw tile has been read: its smem slot may be refilled
            }
            TC_STAMP(threadIdx.x == 128 && i < 24, 8 + i * 6 + 2);
        }
        // LayerNorm folded into this GEMM: the moments of this thread's row (written by the previous kernels) -> mean / rstd
        float2 lnrow = make_float2(0.f, 1.f);
        if constexpr (TcEpiTraits<EPI>::MODE == TC_EPI_LN) lnrow = tc_ln_from_moments(ln_s, ln_ss, p.ln_invK, g.ln_eps);
        // ===================================== epilogue, phase 1 ================================
        mbar_wait(B.accum(), acc_phase);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        TC_STAMP(threadIdx.x == 128, 2);
        const int q = warp & 3;                                        // TMEM lane quarter this warp may read
        const int r = q * 32 + lane;                                   // tile row == TMEM lane
        const uint32_t trow = tmem_base + ((uint32_t)(q * 32) << 16);
        // TMEM -> registers -> shared (the pipeline buffers are free: every TMA landed, every MMA retired).
        // Row pitch BN+4 floats keeps the per-row float4 stores and the row-contiguous reads below conflict-free.
        constexpr int SP = BN + 4;
        float v[32];
#pragma unroll 1
        for (int c0 = 0; c0 < BN; c0 += 32) {
            tmem_ld32(trow + (uint32_t)c0, v);
#pragma unroll
            for (int j = 0; j < 8; ++j)
                asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(base + (uint32_t)(r * SP + c0 + j * 4) * 4u), "f"(v[j * 4]),
                             "f"(v[j * 4 + 1]), "f"(v[j * 4 + 2]), "f"(v[j * 4 + 3]) : "memory");
        }
        if constexpr (TcEpiTraits<EPI>::MODE == TC_EPI_LN)      // (mean, rstd) of tile row r for phase 2, in the last KB of the (now idle) pipeline buffers
            asm volatile("st.shared.v2.f32 [%0], {%1, %2};" ::"r"(base + S::TILE_BYTES - 1024u + (uint32_t)r * 8u), "f"(lnrow.x), "f"(lnrow.y) : "memory");
        TC_STAMP(threadIdx.x == 128, 3);
    }
    // ---- phase 2 (all 8 warps): consecutive threads take consecutive float4 of a row -> coalesced global traffic.
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    TC_STAMP(threadIdx.x == 0, 5);
    {
        const float* rowvec = g.rowvec ? g.rowvec + (int64_t)epi_step * g.rowvec_step_stride : nullptr;
        if (p.splits > 1) {
            const int tile_lin = by * p.gx + bx;
            float* wsp = p.ws + ((int64_t)tile_lin * p.splits + bz) * (TC_BM * BN);
            constexpr int SP = BN + 4;
            constexpr int C4 = BN / 4;
            constexpr int U = 8;
#pragma unroll 1
            for (int i0 = 0; i0 < TC_BM * C4; i0 += TC_THREADS * U) {
                float4 acc[U];
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    const int idx = i0 + u * TC_THREADS + (int)threadIdx.x;
                    const int row = idx / C4, c4 = idx - row * C4;
                    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(acc[u].x), "=f"(acc[u].y), "=f"(acc[u].z), "=f"(acc[u].w)
                                 : "r"(base + (uint32_t)(row * SP + c4 * 4) * 4u));
                }
#pragma unroll
                for (int u = 0; u < U; ++u) st_f4(wsp + (i0 + u * TC_THREADS + (int)threadIdx.x) * 4, acc[u]);   // [row][BN] dense
            }
        } else {
            using E = TcEpiTraits<EPI>;
            tc_store_tile<BN, E::ACT, E::GATE, E::MODE, OCC == 2 ? 8 : 16>(g, base, m_base, n0, rows_valid, rowvec, base + S::TILE_BYTES - 1024u, epi_bias,
                                                                           epi_cs);
        }
    }
    TC_STAMP(threadIdx.x == 0, 4);
#undef TC_STAMP
}

// split-K second pass.  One call = one thread's share of reduce block `blk`: TC_RED_R output rows x one 4-column group.  A block of
// 256 threads covers RPB = TC_RED_R * (256 / (BN/4)) rows of one tile; the partial tiles are summed in fixed split order
// (deterministic), then the fused epilogue (+ row-moment sink / folded LayerNorm) runs.  One row per thread: the reduce of a small
// GEMM is latency-bound, more and smaller blocks finish sooner (4 rows per thread cost +0.45 ms per step at Beff = 8).
constexpr int TC_RED_R = 1;
template <int BN>
struct TcReduceGeom {
    static constexpr int C4 = BN / 4;
    static constexpr int RPP = TC_THREADS / C4;       // rows per pass
    static constexpr int RPB = TC_RED_R * RPP;        // rows per block
    static constexpr int BPT = TC_BM / RPB;           // blocks per tile
    static_assert(TC_BM % RPB == 0, "reduce geometry");
};

template <int BN, int ACT, int GATE, int MODE>
__device__ __forceinline__ void tc_reduce_rows(const TcParams& p, int tile_lin, int rb) {
    using G = TcReduceGeom<BN>;
    static_assert(TC_RED_R == 1, "one output row per thread");
    constexpr int C4 = G::C4;
    constexpr int SEG = C4 < 32 ? C4 : 32;
    constexpr int ZU = 8;                              // partial tiles in flight per thread
    const mugd_gemm& g = p.g;
    const int bx = tile_lin % p.gx, by = tile_lin / p.gx;
    int b_base, l_base, rows_valid;
    tc_tile_rows(p, by, b_base, l_base, rows_valid);
    const int m_base = b_base * p.Lrows + l_base;
    const int c4 = (int)threadIdx.x % C4;
    const int r = rb * G::RPB + (int)threadIdx.x / C4;
    const int n = bx * BN + c4 * 4;
    const int m = m_base + r;
    const bool ok = r < rows_valid && m < g.M && n < g.N;
    // The kernel is one dependent chain of memory round trips; everything that can be asked for early is: bias / column sums are
    // weights (requested before the wait for the GEMM), then -- behind the wait -- the step counter, the residual quad and the row's
    // LayerNorm moments go out BEFORE the partial tiles, and up to 8 partial tiles are in flight together.
    float4 bia = make_float4(0.f, 0.f, 0.f, 0.f), rvv = bia, res = bia, cs = bia;
    if (ok && g.bias) bia = ld_f4(g.bias + n);
    if constexpr (MODE == TC_EPI_LN) {
        if (ok) cs = ld_f4(g.ln_colsum + n);
    }
    pdl_wait();
    int step = 0;
    if (g.step) step = *g.step;
    if (GATE == MUGD_GATE_NONE && g.residual && ok) res = ld_f4(g.residual + (int64_t)m * g.ldr + n);
    double2 mo = make_double2(0.0, 1.0);
    if constexpr (MODE == TC_EPI_LN) {
        if (ok) mo = *reinterpret_cast<const double2*>(g.ln_stats + (int64_t)m * 2);
    }
    const float* src = p.ws + ((long long)tile_lin * p.splits) * (TC_BM * BN) + (long long)r * BN + c4 * 4;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int z0 = 0; z0 < p.splits; z0 += ZU) {                            // fixed order -> deterministic
        float4 t4[ZU];
#pragma unroll
        for (int u = 0; u < ZU; ++u) {
            t4[u] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (ok && z0 + u < p.splits) t4[u] = __ldcg(reinterpret_cast<const float4*>(src + (long long)(z0 + u) * (TC_BM * BN)));
        }
        if (z0 == 0 && g.rowvec && ok)                                      // needs the step counter: by now it has arrived
            rvv = ld_f4(g.rowvec + (int64_t)step * g.rowvec_step_stride + (int64_t)(m / g.Lout) * g.rowvec_b_stride + n);
#pragma unroll
        for (int u = 0; u < ZU; ++u) { acc.x += t4[u].x; acc.y += t4[u].y; acc.z += t4[u].z; acc.w += t4[u].w; }
    }
    float4 o = make_float4(0.f, 0.f, 0.f, 0.f);
    if (ok) {
        float2 ln = make_float2(0.f, 1.f);
        if constexpr (MODE == TC_EPI_LN) ln = tc_ln_from_moments(mo.x, mo.y, p.ln_invK, g.ln_eps);
        const int no = (GATE == MUGD_GATE_NONE) ? n : (n >> 1);
        o = tc_finish4<ACT, GATE, MODE == TC_EPI_LN>(g, g.C + (int64_t)m * g.ldc + no, acc, bia, rvv, res, cs, ln, m, no);
    }
    if constexpr (MODE == TC_EPI_SINK) tc_row_sink<SEG>(g.row_moments, ok ? m : -1, o);
}

template <int BN, int EPI>
__device__ __forceinline__ void tc_reduce_block(const TcParams& p, int blk) {
    using G = TcReduceGeom<BN>;
    using E = TcEpiTraits<EPI>;
    tc_reduce_rows<BN, E::ACT, E::GATE, E::MODE>(p, blk / G::BPT, blk % G::BPT);
}
#endif  // __CUDACC__

// ---- host side (gemm_tc.cu) -------------------------------------------------------------------------
struct TcGeometry {
    int BN, occ, splits, gx, gy, Lrows, Bs, box_l, box_b, tiles_per_sample, total_it;
    int64_t ws_floats;
};
// one planned tensor-core GEMM: kernel parameters + its six tensor maps (A taps 0..2, second source, W_hi, W_lo)
struct alignas(64) TcPlanned {
    CUtensorMap maps[6];
    TcParams p;
};
TcGeometry tc_geometry(const mugd_gemm& g, int sm_count, int forced_split);
int tc_plan(const DeviceInfo& dev, const mugd_gemm& g, TcPlanned* out);     // validates, picks the geometry, encodes the maps

}  // namespace mugd

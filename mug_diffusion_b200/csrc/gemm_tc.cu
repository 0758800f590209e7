// tcgen05 implicit GEMM: stand-alone kernels + host side (geometry planner, tensor-map encoding, launch).
// The device code lives in gemm_tc.cuh (shared with other kernels that embed GEMM tiles).
//
// Reference call sites are the same as gemm_simt.cu (which remains the exact-fp32 referee and the fallback for
// shapes this kernel does not take: K % 32 != 0, N < 16, generic upsampling addressing).
#include "gemm_tc.cuh"

namespace mugd {

template <int BN, int EPI, int OCC = 1>
__global__ void __launch_bounds__(TC_THREADS, OCC)
gemm_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmA1,
               const __grid_constant__ CUtensorMap tmA2, const __grid_constant__ CUtensorMap tmB, const __grid_constant__ CUtensorMap tmWhi,
               const __grid_constant__ CUtensorMap tmWlo, const __grid_constant__ TcParams p) {
    using S = TcSmem<BN, OCC>;
    extern __shared__ uint8_t smem_raw[];
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;       // SWIZZLE_128B needs 1024-B alignment
    const TcBars<BN, OCC> B(base);
    const int warp = threadIdx.x >> 5;
#ifdef MUGD_TC_TIMELINE
    if (p.dbg && blockIdx.x == 0 && blockIdx.y == 0 && blockIdx.z == 0 && threadIdx.x == 0) p.dbg[0] = gtimer();
#endif
    // ---- one-time setup: barriers, tensor memory; nothing here touches memory written by the previous kernel ----
    // The producer warp arms the barriers itself and starts fetching operands at once: it only ARRIVES at the setup rendezvous
    // (named barrier 1), the other seven warps wait there for it and for the tensor-memory allocation.  The first TMA leaves
    // ~0.8 us earlier than behind a CTA-wide __syncthreads (tools/gemm_timeline.py: setup took 0.86 us, first TMA at 1.4 us).
    uint32_t tmem_base = 0;
    if (warp == 0) {
        B.init_parallel((int)threadIdx.x);
        __syncwarp();
        asm volatile("bar.arrive 1, %0;" ::"n"(TC_THREADS) : "memory");
    } else {
        if (threadIdx.x >= 32 && threadIdx.x < 38) {
            // warm the TMA descriptor cache while the barriers / tensor memory are set up
            const CUtensorMap* m = threadIdx.x == 32 ? &tmA : threadIdx.x == 33 ? &tmA1 : threadIdx.x == 34 ? &tmA2
                                 : threadIdx.x == 35 ? &tmB : threadIdx.x == 36 ? &tmWhi : &tmWlo;
            asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
        }
        if (warp == 2) {
            asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(B.tmem_slot()), "r"((uint32_t)S::TMEM_COLS) : "memory");
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
            // Kernel parameters live in constant memory and a fresh launch misses on every 64-byte line it touches; the epilogue reads
            // fields from five of them one after the other (tools/gemm_timeline.py: a bias-free 128x128 tile took 3.2 us to store
            // against 1.0 us for a split-K partial, which reads two).  This otherwise idle warp touches every line of the block now, so
            // that the misses overlap the main loop instead of stretching the epilogue.
            constexpr int LINES = (int)((sizeof(TcParams) + 63) / 64);
            const int* pw = reinterpret_cast<const int*>(&p);
#pragma unroll
            for (int k = 0; k < LINES; ++k) {
                const int v = pw[k * 16];
                asm volatile("" ::"r"(v));
            }
        }
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        asm volatile("bar.sync 1, %0;" ::"n"(TC_THREADS) : "memory");
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(B.tmem_slot()));
        // the producer warp waits for the previous kernel (griddepcontrol.wait) before its first activation load; every other
        // global access of this kernel (epilogue) is ordered behind data that went through that load
        pdl_wait();
    }
    if constexpr (OCC == 2) {
        // Two residents per SM, launched as at most 2 x SMs CTAs: a CTA walks the tile list with stride gridDim.x (consecutive CTAs
        // take neighbouring column tiles of one row band: the band's activations are fetched once into L2) and keeps its tensor
        // memory, its tensor-map cache lines and its warm instruction cache from tile to tile; the barrier rings keep turning
        // (it0 / acc_phase of gemm_tc_tile), nothing is re-armed.
        const int n_tiles = p.gx * p.gy;
        int done = 0;
        for (int tile = (int)blockIdx.x; tile < n_tiles; tile += (int)gridDim.x, ++done) {
            gemm_tc_tile<BN, EPI, OCC>(&tmA, &tmA1, &tmA2, &tmB, &tmWhi, &tmWlo, p, tile % p.gx, tile / p.gx, 0, base, tmem_base,
                                       done * p.hot.total_it, (uint32_t)done & 1u);
            __syncthreads();         // the staged tile has been read: the next tile's TMA may overwrite the pipeline buffers
        }
    } else {
        gemm_tc_tile<BN, EPI, OCC>(&tmA, &tmA1, &tmA2, &tmB, &tmWhi, &tmWlo, p, blockIdx.x, blockIdx.y, blockIdx.z, base, tmem_base);
    }
    // ---- teardown (all tcgen05.ld completed before the phase-2 barrier inside the tile function) ----
    __syncthreads();
    if (warp == 2) {
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)S::TMEM_COLS) : "memory");
    }
}

// split-K second pass: fully parallel over the GPU and L2-resident (see tc_reduce_rows).
template <int BN, int EPI>
__global__ void __launch_bounds__(TC_THREADS)
gemm_tc_reduce_kernel(const __grid_constant__ TcParams p) {
    tc_reduce_block<BN, EPI>(p, blockIdx.x);           // waits for the GEMM (griddepcontrol.wait) after requesting its weight-side operands
}

#ifdef MUGD_TC_TIMELINE
static long long* g_tc_dbg = nullptr;
#endif
// planner constants: us per k-step of a 128- / 256-wide tile (tools/bench_gemm.py), us per split-K round trip (workspace + reduce
// launch).  The split cost was 4.0 in round 1; with the slimmer kernels of round 2 a bench.py sweep of it (299 / 303 / 312 / 312
// steps/s at 5.0 / 4.0 / 3.0 / 2.0) favours splitting a little more.
// The two-CTAs-per-SM variant (TcSmem<128, 2>) is taken when its estimate -- tiles per SM x k-steps x the 128-wide k-step, two residents
// sharing one tensor pipe -- beats the best single-resident estimate by more than k_tc_cost[3].  That constant is a CREDIT (negative):
// the single-resident estimates carry 1.0 us of fill per wave because only their differences matter to the split decision, while a
// wave really exposes ~7 us of prologue + accumulator drain that two residents hide behind each other's main loop.  Fitted on the
// per-op tables of Beff = 64 / L = 512 and Beff = 16 / L = 992 (tools/compare_ops.py): every GEMM it picks was measured faster
// (0.71-0.98x), the ones it leaves alone (fewer tiles than SMs, or long K with < 2 tiles per SM) were slower or even.
constexpr float k_tc_cost[4] = {0.55f, 0.9f, 3.0f, -6.5f};

// =====================================================================================================
// host side
// =====================================================================================================
static bool tc_shape_ok(const mugd_gemm& g) {
    if (!(g.conv_mode == MUGD_CONV_NONE || g.conv_mode == MUGD_CONV_SAME || g.conv_mode == MUGD_CONV_DOWN ||
          g.conv_mode == MUGD_CONV_TAPS)) return false;
    if (g.conv_mode == MUGD_CONV_DOWN && g.Lout < 2) return false;
    if (g.K2 % TC_BK != 0 || (g.K2 > 0 && g.conv_mode == MUGD_CONV_DOWN)) return false;
    return g.K % TC_BK == 0 && g.N >= 16 && g.N % 4 == 0;      // narrow outputs (the 16-channel output convs) take a 64-wide tile: the TMA zero-fills the missing weight rows
}

bool gemm_tc_supported(const mugd_gemm& g) {
    if (!tc_shape_ok(g)) return false;
    if (!g.W_hi || !g.W_lo) return false;
    if (g.lda % 4 != 0 || !aligned16(g.A) || !aligned16(g.W_hi) || !aligned16(g.W_lo)) return false;
    if (g.K2 > 0 && (!g.A2 || g.lda2 % 4 != 0 || !aligned16(g.A2))) return false;
    return true;
}

// the row-moment sink and the folded LayerNorm exist on the tensor-core path only
static int tc_validate_fusions(const mugd_gemm& g) {
    if (g.row_moments)
        MUGD_REQUIRE(g.act == MUGD_ACT_NONE && g.gate == MUGD_GATE_NONE && !g.ln_stats && (reinterpret_cast<uintptr_t>(g.row_moments) & 15u) == 0,
                     "gemm: row_moments needs act == gate == NONE, no folded LayerNorm and a 16-byte aligned buffer");
    if (g.ln_stats) {
        MUGD_REQUIRE(g.ln_colsum && aligned16(g.ln_colsum) && (reinterpret_cast<uintptr_t>(g.ln_stats) & 15u) == 0 && g.taps == 1 && g.K2 == 0 &&
                         g.act == MUGD_ACT_NONE && (g.gate == MUGD_GATE_NONE || g.gate == MUGD_GATE_GEGLU) && !g.rowvec,
                     "gemm: folded LayerNorm needs a single-source Linear with act NONE and gate NONE/GEGLU");
    }
    return MUGD_OK;
}

TcGeometry tc_geometry(const mugd_gemm& g, int sm_count, int forced_split) {
    TcGeometry t;
    t.BN = (g.N >= 128) ? 128 : 64;
    t.occ = 1;
    if (g.conv_mode == MUGD_CONV_NONE) { t.Lrows = g.M; t.Bs = 1; }
    else { t.Lrows = g.Lout; t.Bs = g.M / g.Lout; }
    if (t.Lrows >= TC_BM) {
        t.box_l = TC_BM; t.box_b = 1;
        t.tiles_per_sample = (t.Lrows + TC_BM - 1) / TC_BM;
        t.gy = t.tiles_per_sample * t.Bs;
    } else {
        t.box_l = t.Lrows;
        t.box_b = TC_BM / t.Lrows;
        if (t.box_b > t.Bs) t.box_b = t.Bs;
        t.tiles_per_sample = 1;
        t.gy = (t.Bs + t.box_b - 1) / t.box_b;
    }
    t.total_it = g.taps * (g.K / TC_BK) + g.K2 / TC_BK;
    // Cost model from the B200 micro-benchmark (tools/bench_gemm.py): a CTA needs ~1 us to fill its pipeline and
    // ~0.55 us per k-step with 128-wide tiles (~0.9 us with 256-wide tiles, which do twice the math per step);
    // splitting K adds the workspace round trip and a second (reduce) launch, ~4 us.
    // Candidates: tile width 64 for narrow N, 128, 256 when N allows it, each with its best K split.
    int splits = 1;
    float best = 1e30f;
    static const int cands[4] = {64, 128, 256, 130 /* 128 wide, two CTAs per SM */};
    // a forced variant (mugd_gemm.tc_variant) in the same codes; 0 = cost model.  The two-CTA variant has no split-K form: with a
    // forced split it falls back to the 128-wide one-CTA-per-SM tile, which honours the split.
    int force = (g.tc_variant >= MUGD_TC_N64 && g.tc_variant <= MUGD_TC_N128_2CTA) ? cands[g.tc_variant - MUGD_TC_N64] : 0;
    if (force == 130 && forced_split > 1) force = 128;
    for (int cand = 0; cand < 4; ++cand) {
        const int code = cands[cand];
        const int bn = code == 130 ? 128 : code;
        const int occ = code == 130 ? 2 : 1;
        if (bn > 64 && g.N < bn) continue;
        if (bn == 64 && g.N >= 128 && force != 64) continue;
        if (force && code != force && !((force == 256 ? 256 : 128) > g.N && code == (g.N >= 128 ? 128 : 64))) continue;
        const int gx = (g.N + bn - 1) / bn;
        const int tiles = gx * t.gy;
        if (occ == 2) {
            // two residents per SM share one tensor pipe: n tiles per SM back to back, one exposed prologue + epilogue
            if (forced_split > 1 || (tiles <= sm_count && force != 130)) continue;
            const int n = (tiles + sm_count - 1) / sm_count;
            const float est = k_tc_cost[3] + n * k_tc_cost[0] * t.total_it;
            if (est < best - 0.25f || force == 130) { best = est; splits = 1; t.BN = 128; t.occ = 2; }
            continue;
        }
        const float kstep = bn == 256 ? k_tc_cost[1] : (bn == 128 ? k_tc_cost[0] : 0.4f);
        // 256-wide tiles only pay off unsplit (measured: l1/l2 FF1 and the B=64 convs gain 15-25 %, split cases lose)
        const int sp_max = forced_split > 0 ? forced_split : ((tiles < sm_count && bn != 256) ? 16 : 1);
        for (int sp = forced_split > 0 ? forced_split : 1; sp <= sp_max && sp <= t.total_it; ++sp) {
            const int per = (t.total_it + sp - 1) / sp;
            if (forced_split <= 0 && sp > 1 && per < 2) break;
            if (forced_split <= 0 && sp > 1 && tiles * sp > 2 * sm_count) break;   // bounds the workspace: < 2*SMs partial tiles
            const int waves = (tiles * sp + sm_count - 1) / sm_count;
            const float est = waves * (1.0f + kstep * per) + (sp > 1 ? k_tc_cost[2] : 0.0f);
            if (est < best - 0.25f) { best = est; splits = sp; t.BN = bn; t.occ = 1; }
        }
    }
    t.gx = (g.N + t.BN - 1) / t.BN;
    const int tiles = t.gx * t.gy;
    if (splits > t.total_it) splits = t.total_it;
    if (splits < 1) splits = 1;
    t.splits = splits;
    t.ws_floats = splits > 1 ? (int64_t)tiles * splits * TC_BM * t.BN : 0;
    return t;
}

int tc_plan(const DeviceInfo& dev, const mugd_gemm& g, TcPlanned* out) {
    MUGD_REQUIRE(gemm_tc_supported(g), "gemm_tc: unsupported shape/operands");
    MUGD_REQUIRE(g.tc_variant >= MUGD_TC_AUTO && g.tc_variant <= MUGD_TC_N128_2CTA, "gemm_tc: tc_variant %d", g.tc_variant);
    {
        const int rc = tc_validate_fusions(g);
        if (rc != MUGD_OK) return rc;
    }
    EncodeTiledFn enc = get_encode();
    MUGD_REQUIRE(enc != nullptr, "gemm_tc: cuTensorMapEncodeTiled not available from the driver");
    const TcGeometry t = tc_geometry(g, dev.sm_count, g.split_k);
    if (t.splits > 1) {
        MUGD_REQUIRE(g.workspace, "gemm_tc: split-K needs a workspace");
        MUGD_REQUIRE(g.workspace_bytes >= t.ws_floats * 4, "gemm_tc: workspace too small (%lld < %lld)", (long long)g.workspace_bytes,
                     (long long)t.ws_floats * 4);
    }
    for (int tap = 0; tap < 3; ++tap) {
        if (tap > 0 && g.conv_mode != MUGD_CONV_DOWN) { out->maps[tap] = out->maps[0]; continue; }
        const bool down = g.conv_mode == MUGD_CONV_DOWN;
        // DOWN: row l of the map of tap t is source row 2l+t; the last row of tap 2 is the right padding -> out of bounds
        const cuuint64_t rows = down ? (cuuint64_t)(t.Lrows - (tap == 2 ? 1 : 0)) : (cuuint64_t)t.Lrows;
        const cuuint64_t sample_rows = down ? (cuuint64_t)g.Lin : (cuuint64_t)t.Lrows;
        cuuint64_t dims[3] = {(cuuint64_t)g.K, rows, (cuuint64_t)t.Bs};
        cuuint64_t strides[2] = {(cuuint64_t)g.lda * 4 * (down ? 2 : 1), sample_rows * (cuuint64_t)g.lda * 4};
        cuuint32_t box[3] = {(cuuint32_t)TC_BK, (cuuint32_t)t.box_l, (cuuint32_t)t.box_b};
        cuuint32_t estr[3] = {1, 1, 1};
        const float* basep = g.A + (down ? (int64_t)tap * g.lda : 0);
        CUresult r = enc(&out->maps[tap], CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float*>(basep), dims, strides, box, estr,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        MUGD_REQUIRE(r == CUDA_SUCCESS, "gemm_tc: cuTensorMapEncodeTiled(A) failed with %d (K=%d L=%d B=%d lda=%lld)", (int)r, g.K,
                     t.Lrows, t.Bs, (long long)g.lda);
    }
    if (g.K2 > 0) {
        // second source: same row structure as the output (Lrows rows per sample), no tap shift
        cuuint64_t dims[3] = {(cuuint64_t)g.K2, (cuuint64_t)t.Lrows, (cuuint64_t)t.Bs};
        cuuint64_t strides[2] = {(cuuint64_t)g.lda2 * 4, (cuuint64_t)t.Lrows * (cuuint64_t)g.lda2 * 4};
        cuuint32_t box[3] = {(cuuint32_t)TC_BK, (cuuint32_t)t.box_l, (cuuint32_t)t.box_b};
        cuuint32_t estr[3] = {1, 1, 1};
        CUresult r = enc(&out->maps[3], CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float*>(g.A2), dims, strides, box, estr,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        MUGD_REQUIRE(r == CUDA_SUCCESS, "gemm_tc: cuTensorMapEncodeTiled(A2) failed with %d (K2=%d lda2=%lld)", (int)r, g.K2, (long long)g.lda2);
    } else {
        out->maps[3] = out->maps[0];
    }
    for (int w = 0; w < 2; ++w) {
        const cuuint64_t ktot = (cuuint64_t)g.taps * g.K + g.K2;
        cuuint64_t dims[2] = {ktot, (cuuint64_t)g.N};
        cuuint64_t strides[1] = {ktot * 4};
        cuuint32_t box[2] = {(cuuint32_t)TC_BK, (cuuint32_t)t.BN};
        cuuint32_t estr[2] = {1, 1};
        CUresult r = enc(&out->maps[4 + w], CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(w == 0 ? g.W_hi : g.W_lo), dims,
                         strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                         CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        MUGD_REQUIRE(r == CUDA_SUCCESS, "gemm_tc: cuTensorMapEncodeTiled(W) failed with %d", (int)r);
    }
    TcParams& p = out->p;
    memset(&p, 0, sizeof(p));
    p.g = g;
    p.ws = (float*)g.workspace;
    p.splits = t.splits;
    p.total_it = t.total_it;
    p.kblocks = g.K / TC_BK;
    p.it_main = g.taps * (g.K / TC_BK);
    p.Lrows = t.Lrows;
    p.Bs = t.Bs;
    p.box_l = t.box_l;
    p.box_b = t.box_b;
    p.tiles_per_sample = t.tiles_per_sample;
    p.single_pass = dev.tc_single_pass ? 1 : 0;
    p.BN = t.BN;
    p.occ = t.occ;
    p.sm_count = dev.sm_count;
    p.gx = t.gx;
    p.gy = t.gy;
    p.ln_invK = 1.0 / (double)g.K;
    p.it_base = t.total_it / t.splits;
    p.it_rem = t.total_it % t.splits;
    p.hot = {p.Lrows, p.Bs, p.box_l, p.box_b, p.tiles_per_sample, p.it_base, p.it_rem, p.it_main, p.kblocks, p.total_it, p.splits, p.single_pass,
             g.conv_mode, g.tap_shift, g.tap_dilation, p.gx};
#ifdef MUGD_TC_TIMELINE
    p.dbg = g_tc_dbg;
#endif
    return MUGD_OK;
}

template <int BN, int EPI>
static int tc_launch(const TcPlanned& pl, cudaStream_t st) {
    const TcParams& p = pl.p;
    if (p.splits > 1) {
        // the main kernel only writes partial tiles: it runs the smallest instantiation, the epilogue variant lives in the reduce
        MUGD_CHECK_CUDA(launch_k(gemm_tc_kernel<BN, TC_E_NONE>, dim3(p.gx, p.gy, p.splits), dim3(TC_THREADS), TcSmem<BN>::TOTAL, st, pl.maps[0],
                                 pl.maps[1], pl.maps[2], pl.maps[3], pl.maps[4], pl.maps[5], p));
        MUGD_CHECK_CUDA(launch_k(gemm_tc_reduce_kernel<BN, EPI>, dim3((unsigned)(p.gx * p.gy * TcReduceGeom<BN>::BPT)), dim3(TC_THREADS), 0, st, p));
        return MUGD_OK;
    }
    if constexpr (BN == 128) {
        if (p.occ == 2) {
            const int n_tiles = p.gx * p.gy;
            const int ctas = n_tiles < 2 * p.sm_count ? n_tiles : 2 * p.sm_count;
            MUGD_CHECK_CUDA(launch_k(gemm_tc_kernel<BN, EPI, 2>, dim3(ctas, 1, 1), dim3(TC_THREADS), TcSmem<BN, 2>::TOTAL, st, pl.maps[0], pl.maps[1],
                                     pl.maps[2], pl.maps[3], pl.maps[4], pl.maps[5], p));
            return MUGD_OK;
        }
    }
    MUGD_CHECK_CUDA(launch_k(gemm_tc_kernel<BN, EPI>, dim3(p.gx, p.gy, 1), dim3(TC_THREADS), TcSmem<BN>::TOTAL, st, pl.maps[0], pl.maps[1],
                             pl.maps[2], pl.maps[3], pl.maps[4], pl.maps[5], p));
    return MUGD_OK;
}

template <int BN>
static int tc_launch_bn(const TcPlanned& pl, cudaStream_t st) {
    switch (tc_epi_of(pl.p.g)) {
        case TC_E_GEGLU: return tc_launch<BN, TC_E_GEGLU>(pl, st);
        case TC_E_GLU: return tc_launch<BN, TC_E_GLU>(pl, st);
        case TC_E_SILU: return tc_launch<BN, TC_E_SILU>(pl, st);
        case TC_E_GELU: return tc_launch<BN, TC_E_GELU>(pl, st);
        case TC_E_SINK: return tc_launch<BN, TC_E_SINK>(pl, st);
        case TC_E_LN: return tc_launch<BN, TC_E_LN>(pl, st);
        case TC_E_LN_GEGLU: return tc_launch<BN, TC_E_LN_GEGLU>(pl, st);
        default: return tc_launch<BN, TC_E_NONE>(pl, st);
    }
}

template <int BN, int OCC, int... EPI>
static cudaError_t tc_configure(std::integer_sequence<int, EPI...>) {
    cudaError_t e = cudaSuccess;
    ((e = e != cudaSuccess ? e : cudaFuncSetAttribute(gemm_tc_kernel<BN, EPI, OCC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TcSmem<BN, OCC>::TOTAL)), ...);
    if constexpr (OCC == 2) ((e = e != cudaSuccess ? e : cudaFuncSetAttribute(gemm_tc_kernel<BN, EPI, OCC>, cudaFuncAttributePreferredSharedMemoryCarveout, 100)), ...);
    return e;
}

// every instantiation tc_launch can pick: 64 / 128 / 256 wide with each epilogue, and the 128-wide two-CTAs-per-SM variant
int configure_gemm_tc_kernels(const DeviceInfo&) {
    using Epis = std::make_integer_sequence<int, TC_E_COUNT>;
    MUGD_CHECK_CUDA((tc_configure<64, 1>(Epis{})));
    MUGD_CHECK_CUDA((tc_configure<128, 1>(Epis{})));
    MUGD_CHECK_CUDA((tc_configure<256, 1>(Epis{})));
    MUGD_CHECK_CUDA((tc_configure<128, 2>(Epis{})));
    return MUGD_OK;
}

int launch_gemm_tc(const DeviceInfo& dev, const mugd_gemm& g, cudaStream_t st, int* launches) {
    TcPlanned pl;
    int rc = tc_plan(dev, g, &pl);
    if (rc != MUGD_OK) return rc;
    if (pl.p.BN == 256) rc = tc_launch_bn<256>(pl, st);
    else if (pl.p.BN == 128) rc = tc_launch_bn<128>(pl, st);
    else rc = tc_launch_bn<64>(pl, st);
    if (rc != MUGD_OK) return rc;
    if (launches) *launches += pl.p.splits > 1 ? 2 : 1;
    return MUGD_OK;
}

}  // namespace mugd

extern "C" int mugd_debug_set_tc_timing(long long* device_buf) {
#ifdef MUGD_TC_TIMELINE
    mugd::g_tc_dbg = device_buf;
    return MUGD_OK;
#else
    (void)device_buf;
    mugd::set_error("mugd_debug_set_tc_timing: this build has no timeline hooks (rebuild with -DMUGD_TC_TIMELINE, tools/build_variant.py)");
    return MUGD_ERR_INVALID;
#endif
}

extern "C" int mugd_gemm_tc_variant(const mugd_gemm* g, int32_t sm_count, int32_t* tile_n, int32_t* ctas_per_sm, int32_t* grid_ctas) {
    using namespace mugd;
    MUGD_REQUIRE(g, "gemm_tc_variant: null");
    if (!tc_shape_ok(*g)) {
        if (tile_n) *tile_n = 0;
        if (ctas_per_sm) *ctas_per_sm = 0;
        if (grid_ctas) *grid_ctas = 0;
        return MUGD_OK;
    }
    const int sms = sm_count > 0 ? sm_count : 148;
    const TcGeometry t = tc_geometry(*g, sms, g->split_k);
    const int tiles = t.gx * t.gy;
    if (tile_n) *tile_n = t.BN;
    if (ctas_per_sm) *ctas_per_sm = t.occ;
    if (grid_ctas) *grid_ctas = t.occ == 2 ? (tiles < 2 * sms ? tiles : 2 * sms) : tiles * t.splits;
    return MUGD_OK;
}

extern "C" int mugd_gemm_tc_query(mugd_handle*, const mugd_gemm* g, int32_t sm_count, int32_t* supported, int32_t* splits,
                                  int64_t* workspace_bytes, int32_t* n_tiles) {
    using namespace mugd;
    MUGD_REQUIRE(g, "gemm_tc_query: null");
    const bool ok = tc_shape_ok(*g);
    if (supported) *supported = ok ? 1 : 0;
    if (!ok) {
        if (splits) *splits = 0;
        if (workspace_bytes) *workspace_bytes = 0;
        if (n_tiles) *n_tiles = 0;
        return MUGD_OK;
    }
    const TcGeometry t = tc_geometry(*g, sm_count > 0 ? sm_count : 148, g->split_k);
    if (splits) *splits = t.splits;
    if (workspace_bytes) *workspace_bytes = t.ws_floats * 4;
    if (n_tiles) *n_tiles = t.gx * t.gy;
    return MUGD_OK;
}

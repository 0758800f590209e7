// Attention of mug/model/attention.py:91-126 (CrossAttention.forward), fp32, flash-style (no [Lq,Lk]
// matrix in memory):
//     idx_ij = clamp(j - i, -P, P) + P
//     s_ij   = (q_i . k_j + relpos[idx_ij, h]) * scale
//     o_i    = sum_j softmax_j(s_i)_j * cgain[idx_ij, h] * v_j
// The post-softmax gain multiplies the numerator only; the softmax denominator accumulates plain p.
// Self attention (Lk = Lq) and cross attention to the 21 prompt tokens (Lk = 21) share the kernel.
//
// Register-tiled FFMA formulation: a CTA of 256 threads (16 x 16) owns 64 queries of one (sample, head) and
// streams 64-key tiles.  S = Q K^T is a 64x64xD smem-tiled product with 4x4 micro-tiles (operands stored
// k-major so both are read as conflict-free float4), the online softmax runs on the micro-tile with
// 16-lane shuffle reductions, P*gain goes back to shared memory transposed, and O += P V is a second
// 64 x D x 64 product.  Exact fp32 (expf, IEEE division): this is 2.6 % of the FLOPs, the parity-critical
// part (non-standard bias + gain) rather than the fast part of the network.
#include "common.cuh"

#include <math.h>

namespace mugd {

constexpr int AT_BQ = 64;
constexpr int AT_BK = 64;
constexpr int AT_PAD = 4;
constexpr int AT_THREADS = 256;

template <int D>
struct AttSmem {
    static constexpr int QT = D * (AT_BQ + AT_PAD);
    static constexpr int KT = D * (AT_BK + AT_PAD);
    static constexpr int VS = AT_BK * D;
    static constexpr int PT = AT_BK * (AT_BQ + AT_PAD);
    static constexpr int FLOATS = QT + KT + VS + PT;
};

template <int D>
__global__ void __launch_bounds__(AT_THREADS)
attention_kernel(const mugd_attention a) {
    constexpr int DC = D / 16;                 // output columns per thread
    constexpr int SQ = AT_BQ + AT_PAD, SK = AT_BK + AT_PAD;
    extern __shared__ __align__(16) float sm[];
    float* Qt = sm;                            // [D][SQ]   Qt[k][row]
    float* Kt = Qt + AttSmem<D>::QT;           // [D][SK]   Kt[k][col]
    float* Vs = Kt + AttSmem<D>::KT;           // [BK][D]
    float* Pt = Vs + AttSmem<D>::VS;           // [BK][SQ]  Pt[key][row] = p * gain
    float* rel = Pt + AttSmem<D>::PT;          // [2P+1]
    const int P = a.pos_max, NT = 2 * P + 1;
    float* cg = rel + NT;

    pdl_wait();
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    const int b = blockIdx.z, h = blockIdx.y;
    const int q0 = blockIdx.x * AT_BQ;
    for (int t = tid; t < NT; t += AT_THREADS) {
        rel[t] = a.relpos[t * a.H + h];
        cg[t] = a.cgain[t * a.H + h];
    }
    constexpr int QD = D / 4;
    {
        const float* qb = a.q + (int64_t)b * a.Lq * a.ldq + h * D;
        for (int t = tid; t < AT_BQ * QD; t += AT_THREADS) {
            const int r = t / QD, c = (t - r * QD) * 4;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (q0 + r < a.Lq) v = ld_f4(qb + (int64_t)(q0 + r) * a.ldq + c);
            Qt[(c + 0) * SQ + r] = v.x; Qt[(c + 1) * SQ + r] = v.y; Qt[(c + 2) * SQ + r] = v.z; Qt[(c + 3) * SQ + r] = v.w;
        }
    }
    float m_i[4], l_i[4], o[4][DC];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        m_i[i] = -INFINITY; l_i[i] = 0.f;
#pragma unroll
        for (int c = 0; c < DC; ++c) o[i][c] = 0.f;
    }
    const float* kb = a.k + (int64_t)b * a.Lk * a.ldk + h * D;
    const float* vb = a.v + (int64_t)b * a.Lk * a.ldv + h * D;

    for (int j0 = 0; j0 < a.Lk; j0 += AT_BK) {
        __syncthreads();                       // previous tile consumed (first pass: Qt / tables written)
        for (int t = tid; t < AT_BK * QD; t += AT_THREADS) {
            const int r = t / QD, c = (t - r * QD) * 4;
            float4 kv = make_float4(0.f, 0.f, 0.f, 0.f), vv = kv;
            if (j0 + r < a.Lk) {
                kv = ld_f4(kb + (int64_t)(j0 + r) * a.ldk + c);
                vv = ld_f4(vb + (int64_t)(j0 + r) * a.ldv + c);
            }
            Kt[(c + 0) * SK + r] = kv.x; Kt[(c + 1) * SK + r] = kv.y; Kt[(c + 2) * SK + r] = kv.z; Kt[(c + 3) * SK + r] = kv.w;
            *reinterpret_cast<float4*>(&Vs[r * D + c]) = vv;
        }
        __syncthreads();
        // ---- S = Q K^T on a 4x4 micro-tile ---------------------------------------------------------------
        float s[4][4];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) s[i][j] = 0.f;
#pragma unroll 8
        for (int kk = 0; kk < D; ++kk) {
            const float4 qa = *reinterpret_cast<const float4*>(&Qt[kk * SQ + ty * 4]);
            const float4 kv = *reinterpret_cast<const float4*>(&Kt[kk * SK + tx * 4]);
            const float qf[4] = {qa.x, qa.y, qa.z, qa.w}, kf[4] = {kv.x, kv.y, kv.z, kv.w};
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) s[i][j] = fmaf(qf[i], kf[j], s[i][j]);
        }
        // ---- bias, scale, mask, online softmax ------------------------------------------------------------
        float pc[4][4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int qi = q0 + ty * 4 + i;
            float mx = -INFINITY;
            int idx[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int kj = j0 + tx * 4 + j;
                idx[j] = max(-P, min(P, kj - qi)) + P;
                s[i][j] = (kj < a.Lk) ? (s[i][j] + rel[idx[j]]) * a.scale : -INFINITY;
                mx = fmaxf(mx, s[i][j]);
            }
#pragma unroll
            for (int off = 8; off > 0; off >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, off));
            const float mnew = fmaxf(m_i[i], mx);          // finite: column j0 of every tile is a valid key
            const float corr = expf(m_i[i] - mnew);
            float rs = 0.f;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const float pe = expf(s[i][j] - mnew);      // 0 for masked keys
                rs += pe;
                pc[i][j] = pe * cg[idx[j]];
            }
#pragma unroll
            for (int off = 8; off > 0; off >>= 1) rs += __shfl_xor_sync(0xffffffffu, rs, off);
            l_i[i] = l_i[i] * corr + rs;
            m_i[i] = mnew;
#pragma unroll
            for (int c = 0; c < DC; ++c) o[i][c] *= corr;
        }
#pragma unroll
        for (int j = 0; j < 4; ++j)
            *reinterpret_cast<float4*>(&Pt[(tx * 4 + j) * SQ + ty * 4]) = make_float4(pc[0][j], pc[1][j], pc[2][j], pc[3][j]);
        __syncthreads();
        // ---- O += P V ----------------------------------------------------------------------------------------
        const int nk = min(AT_BK, a.Lk - j0);
#pragma unroll 4
        for (int kk = 0; kk < nk; ++kk) {
            const float4 pa = *reinterpret_cast<const float4*>(&Pt[kk * SQ + ty * 4]);
            const float pf[4] = {pa.x, pa.y, pa.z, pa.w};
            float vf[DC];
#pragma unroll
            for (int c = 0; c < DC; ++c) vf[c] = Vs[kk * D + tx * DC + c];
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int c = 0; c < DC; ++c) o[i][c] = fmaf(pf[i], vf[c], o[i][c]);
        }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int qi = q0 + ty * 4 + i;
        if (qi < a.Lq) {
            const float inv = 1.0f / l_i[i];
            float* op = a.o + ((int64_t)b * a.Lq + qi) * a.ldo + h * D + tx * DC;
#pragma unroll
            for (int c = 0; c < DC; ++c) op[c] = o[i][c] * inv;
        }
    }
}

template <int D>
static int attention_launch(const DeviceInfo& dev, const mugd_attention& a, cudaStream_t st) {
    const size_t bytes = sizeof(float) * (AttSmem<D>::FLOATS + 2 * (2 * a.pos_max + 1));
    MUGD_REQUIRE(bytes <= (size_t)dev.max_smem_optin, "attention: pos_max=%d needs %zu B of shared memory (max %d)", a.pos_max, bytes,
                 dev.max_smem_optin);
    dim3 grid((a.Lq + AT_BQ - 1) / AT_BQ, a.H, a.B);
    MUGD_CHECK_CUDA(launch_k(attention_kernel<D>, grid, dim3(AT_THREADS), bytes, st, a));
    return MUGD_OK;
}

// the byte count grows with pos_max: allow what the device allows, the launcher checks each launch against it
int configure_attention_kernels(const DeviceInfo& dev) {
    MUGD_CHECK_CUDA(cudaFuncSetAttribute(attention_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, dev.max_smem_optin));
    MUGD_CHECK_CUDA(cudaFuncSetAttribute(attention_kernel<48>, cudaFuncAttributeMaxDynamicSharedMemorySize, dev.max_smem_optin));
    MUGD_CHECK_CUDA(cudaFuncSetAttribute(attention_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, dev.max_smem_optin));
    return MUGD_OK;
}

// =====================================================================================================
// Few keys (Lk <= 32): the cross attention to the 21 prompt tokens, 16 of the 32 attention launches of an evaluation.
// A 128-key tensor-core tile would be 5/6 zero fill behind ~5 us of fixed cost (tensor-memory allocation, TMA, operand splits);
// here ONE LANE OWNS ONE KEY: lane j keeps k_j in registers, a warp takes four query rows at a time (four independent dependency
// chains) -- the rows are read back from shared memory as broadcast float4s for the D-long dot products, max / sum are warp shuffles, and for O = (P*gain) V lane d owns output
// channels d, d+32 and receives p_j from lane j by shuffle.  Exact fp32, same formula order as the FFMA referee above.
// =====================================================================================================
constexpr int ASK_WARPS = 8;
constexpr int ASK_RW = 4;         // query rows a warp carries together
constexpr int ASK_ROWS = ASK_WARPS * ASK_RW;      // query rows per CTA

template <int D>
__global__ void __launch_bounds__(ASK_WARPS * 32)
attention_smallk_kernel(const mugd_attention a) {
    constexpr int DV = (D + 31) / 32;                 // output channels per lane
    constexpr int KP = D + 1;                         // K row pitch: lane j reads row j, the odd pitch keeps the lanes on distinct banks
    constexpr int QD = D / 4;
    extern __shared__ __align__(16) float sm[];
    float* Ks = sm;                                   // [32][KP]
    float* Vs = Ks + 32 * KP;                         // [32][D]
    float* Qs = Vs + 32 * D;                          // [ASK_ROWS][D]
    pdl_wait();
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int b = blockIdx.z, h = blockIdx.y, q0 = blockIdx.x * ASK_ROWS;
    const int P = a.pos_max;
    const int qbase = q0 + warp * ASK_RW;             // the warp's ASK_RW query rows go through the kernel together
    const bool key_ok = lane < a.Lk;
    // everything this thread needs from global memory is requested up front, in one round trip with the K / V fill: its slice of
    // the warp's query rows and the bias / gain of (its key, each row) -- 2 x ASK_RW table entries, not the whole 2P+1 table
    float qpre[ASK_RW][DV], relv[ASK_RW], cgv[ASK_RW];
#pragma unroll
    for (int i = 0; i < ASK_RW; ++i) {
        const int qi = min(qbase + i, a.Lq - 1);      // rows past the end recompute the last row (never stored)
        const float* qp = a.q + ((int64_t)b * a.Lq + qi) * a.ldq + h * D;
#pragma unroll
        for (int c = 0; c < DV; ++c) qpre[i][c] = (lane + c * 32 < D) ? qp[lane + c * 32] : 0.f;
        const int idx = max(-P, min(P, lane - (qbase + i))) + P;
        relv[i] = a.relpos[idx * a.H + h];
        cgv[i] = a.cgain[idx * a.H + h];
    }
    const float* kb = a.k + (int64_t)b * a.Lk * a.ldk + h * D;
    const float* vb = a.v + (int64_t)b * a.Lk * a.ldv + h * D;
    for (int t = tid; t < 32 * QD; t += ASK_WARPS * 32) {
        const int r = t / QD, c = (t - r * QD) * 4;
        float4 kv = make_float4(0.f, 0.f, 0.f, 0.f), vv = kv;
        if (r < a.Lk) {
            kv = ld_f4(kb + (int64_t)r * a.ldk + c);
            vv = ld_f4(vb + (int64_t)r * a.ldv + c);
        }
        Ks[r * KP + c] = kv.x; Ks[r * KP + c + 1] = kv.y; Ks[r * KP + c + 2] = kv.z; Ks[r * KP + c + 3] = kv.w;
        *reinterpret_cast<float4*>(&Vs[r * D + c]) = vv;
    }
    float* qrows = Qs + warp * ASK_RW * D;
#pragma unroll
    for (int i = 0; i < ASK_RW; ++i)
#pragma unroll
        for (int c = 0; c < DV; ++c)
            if (lane + c * 32 < D) qrows[i * D + lane + c * 32] = qpre[i][c];
    __syncthreads();
    if (qbase >= a.Lq) return;                        // uniform over the warp; no barrier follows
    float kreg[D];
#pragma unroll
    for (int d = 0; d < D; ++d) kreg[d] = Ks[lane * KP + d];
    float s[ASK_RW];
#pragma unroll
    for (int i = 0; i < ASK_RW; ++i) s[i] = 0.f;
#pragma unroll
    for (int c = 0; c < QD; ++c) {
#pragma unroll
        for (int i = 0; i < ASK_RW; ++i) {
            const float4 qv = *reinterpret_cast<const float4*>(&qrows[i * D + c * 4]);       // broadcast
            s[i] = fmaf(qv.x, kreg[c * 4], s[i]); s[i] = fmaf(qv.y, kreg[c * 4 + 1], s[i]);
            s[i] = fmaf(qv.z, kreg[c * 4 + 2], s[i]); s[i] = fmaf(qv.w, kreg[c * 4 + 3], s[i]);
        }
    }
    float mx[ASK_RW], pe[ASK_RW], sum[ASK_RW], pg[ASK_RW];
#pragma unroll
    for (int i = 0; i < ASK_RW; ++i) {
        s[i] = key_ok ? (s[i] + relv[i]) * a.scale : -INFINITY;
        mx[i] = s[i];
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1)
#pragma unroll
        for (int i = 0; i < ASK_RW; ++i) mx[i] = fmaxf(mx[i], __shfl_xor_sync(0xffffffffu, mx[i], off));
#pragma unroll
    for (int i = 0; i < ASK_RW; ++i) { pe[i] = expf(s[i] - mx[i]); sum[i] = pe[i]; pg[i] = pe[i] * cgv[i]; }   // pe = 0 for lanes without a key
#pragma unroll
    for (int off = 16; off > 0; off >>= 1)
#pragma unroll
        for (int i = 0; i < ASK_RW; ++i) sum[i] += __shfl_xor_sync(0xffffffffu, sum[i], off);
    float o[ASK_RW][DV];
#pragma unroll
    for (int i = 0; i < ASK_RW; ++i)
#pragma unroll
        for (int c = 0; c < DV; ++c) o[i][c] = 0.f;
    for (int j = 0; j < a.Lk; ++j) {
        float vj[DV];
#pragma unroll
        for (int c = 0; c < DV; ++c) vj[c] = (lane + c * 32 < D) ? Vs[j * D + lane + c * 32] : 0.f;
#pragma unroll
        for (int i = 0; i < ASK_RW; ++i) {
            const float pj = __shfl_sync(0xffffffffu, pg[i], j);
#pragma unroll
            for (int c = 0; c < DV; ++c) o[i][c] = fmaf(pj, vj[c], o[i][c]);
        }
    }
#pragma unroll
    for (int i = 0; i < ASK_RW; ++i) {
        const int qi = qbase + i;
        if (qi < a.Lq) {
            const float inv = 1.0f / sum[i];
            float* op = a.o + ((int64_t)b * a.Lq + qi) * a.ldo + h * D;
#pragma unroll
            for (int c = 0; c < DV; ++c)
                if (lane + c * 32 < D) op[lane + c * 32] = o[i][c] * inv;
        }
    }
}

template <int D>
static int attention_smallk_launch(const mugd_attention& a, cudaStream_t st) {
    const size_t bytes = sizeof(float) * (32 * (D + 1) + 32 * D + ASK_ROWS * D + 4);
    dim3 grid((a.Lq + ASK_ROWS - 1) / ASK_ROWS, a.H, a.B);      // (more rows per CTA -- fewer re-reads of K / V -- measured slower)
    MUGD_CHECK_CUDA(launch_k(attention_smallk_kernel<D>, grid, dim3(ASK_WARPS * 32), bytes, st, a));
    return MUGD_OK;
}

int launch_attention_tc(const DeviceInfo& dev, const mugd_attention& a, cudaStream_t st);   // attention_tc.cu
// 1 (default): both contractions on the tcgen05 tensor cores (attention_tc.cu), a lane-per-key kernel when there are at most 32 keys;
// 0: the tiled FFMA kernel above for everything (referee)
int launch_attention(const DeviceInfo& dev, const mugd_attention& a, cudaStream_t st, int* launches) {
    MUGD_REQUIRE(a.B > 0 && a.H > 0 && a.Lq > 0 && a.Lk > 0, "attention: empty shape");
    MUGD_REQUIRE(a.D == 32 || a.D == 48 || a.D == 64, "attention: head dim %d not in {32,48,64}", a.D);
    MUGD_REQUIRE(a.pos_max >= 0 && a.pos_max <= 1024, "attention: pos_max %d", a.pos_max);
    MUGD_REQUIRE(aligned16(a.q) && aligned16(a.k) && aligned16(a.v) && aligned16(a.o) && a.ldq % 4 == 0 && a.ldk % 4 == 0 &&
                     a.ldv % 4 == 0 && a.ldo % 4 == 0, "attention: alignment");
    MUGD_REQUIRE(a.ldq >= a.H * a.D && a.ldk >= a.H * a.D && a.ldv >= a.H * a.D && a.ldo >= a.H * a.D, "attention: ld < H*D");
    MUGD_REQUIRE(a.relpos && a.cgain, "attention: tables missing");
    int rc;
    // measured per shape (tools/profile_ops.py --only attention): with head dim 32 (Lq = 256 at the default length) the rows are many
    // and short and the FFMA lanes saturate (6.9 vs 5.8 us at Beff = 8); with head dim 48 / 64 the lane-per-key kernel wins
    // (5.7 vs 7.6, 4.2 vs 6.5 us at Beff = 8; 26.8 vs 28.0, 17.3 vs 23.9 us at Beff = 64)
    if (dev.attention_impl == 1 && a.Lk <= 32 && a.D >= 48)
        rc = (a.D == 48) ? attention_smallk_launch<48>(a, st) : attention_smallk_launch<64>(a, st);
    else if (dev.attention_impl == 1) rc = launch_attention_tc(dev, a, st);
    else rc = (a.D == 32) ? attention_launch<32>(dev, a, st) : (a.D == 48) ? attention_launch<48>(dev, a, st) : attention_launch<64>(dev, a, st);
    if (rc != MUGD_OK) return rc;
    if (launches) *launches += 1;
    return MUGD_OK;
}

}  // namespace mugd


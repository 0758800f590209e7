// Small fused elementwise kernels of the sampler loop:
//   ddim_update : classifier-free-guidance combine + DDIM x_{t-1} update   mug/diffusion/ddim.py:170-195
//   transpose   : [B,C,L] <-> channels-last [B*L, ld] at the Python boundary (reference tensors are NCL)
//   copy2d      : strided row copy (the 4 per-level tensors that live in two concat buffers)
//   step_advance: device-side step counter so one CUDA graph serves every DDIM step
#include "common.cuh"

namespace mugd {

// x_prev = sqrt(a_prev) * (x - sqrt(1-a_t) e)/sqrt(a_t) + sqrt(1 - a_prev - sigma^2) e + sigma*noise*T
// written with explicit _rn intrinsics: same operation order and roundings as the reference's separate
// ATen ops (no FMA contraction), so given identical eps the update is bit-identical.
__global__ void __launch_bounds__(256)
ddim_update_kernel(const mugd_ddim_update d) {
    pdl_wait();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= d.n) return;
    const int step = d.step ? *d.step : 0;
    const int index = d.S - 1 - step;                     // ddim.py:138
    const float* cf = d.coef + 4 * index;
    const float a_t = cf[0], a_prev = cf[1], sigma = cf[2], s1m = cf[3];
    float e;
    if (d.cfg) {
        const float eu = d.eps[i], ec = d.eps[(int64_t)d.n + i];
        e = __fadd_rn(eu, __fmul_rn(d.scale, __fsub_rn(ec, eu)));   // ddim.py:175
    } else {
        e = d.eps[i];
    }
    const float x = d.x[i];
    const float pred = __fdiv_rn(__fsub_rn(x, __fmul_rn(s1m, e)), __fsqrt_rn(a_t));            // :189
    const float dir = __fmul_rn(__fsqrt_rn(__fsub_rn(__fsub_rn(1.0f, a_prev), __fmul_rn(sigma, sigma))), e);  // :191
    float xp = __fadd_rn(__fmul_rn(__fsqrt_rn(a_prev), pred), dir);
    const float nz = d.noise ? __fmul_rn(__fmul_rn(sigma, d.noise[i]), d.temperature) : 0.0f;  // :192
    xp = __fadd_rn(xp, nz);                                                                     // :195
    d.x[i] = xp;
    if (d.x_dup) d.x_dup[i] = xp;
    if (d.pred_x0) d.pred_x0[i] = pred;
}

int launch_ddim_update(const DeviceInfo&, const mugd_ddim_update& d, cudaStream_t st, int* launches) {
    MUGD_REQUIRE(d.n > 0 && d.S > 0 && d.x && d.eps && d.coef, "ddim_update: bad arguments");
    MUGD_CHECK_CUDA(launch_k(ddim_update_kernel, dim3((d.n + 255) / 256), dim3(256), 0, st, d));
    if (launches) *launches += 1;
    return MUGD_OK;
}

// 32x32 smem-tiled transpose, coalesced on both sides.
__global__ void __launch_bounds__(256)
transpose_kernel(const mugd_transpose t) {
    __shared__ float tile[32][33];
    pdl_wait();
    const int b = blockIdx.z;
    const int c0 = blockIdx.y * 32, l0 = blockIdx.x * 32;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;   // 32 x 8
    if (t.to_nlc) {
        const float* in = t.in + (int64_t)b * t.C * t.L;
#pragma unroll
        for (int r = ty; r < 32; r += 8) {
            const int c = c0 + r, l = l0 + tx;
            tile[r][tx] = (c < t.C && l < t.L) ? in[(int64_t)c * t.L + l] : 0.f;
        }
        __syncthreads();
        float* out = t.out + (int64_t)b * t.L * t.ldo;
#pragma unroll
        for (int r = ty; r < 32; r += 8) {
            const int l = l0 + r, c = c0 + tx;
            if (c < t.C && l < t.L) out[(int64_t)l * t.ldo + c] = tile[tx][r];
        }
    } else {
        const float* in = t.in + (int64_t)b * t.L * t.ldi;
#pragma unroll
        for (int r = ty; r < 32; r += 8) {
            const int l = l0 + r, c = c0 + tx;
            tile[r][tx] = (c < t.C && l < t.L) ? in[(int64_t)l * t.ldi + c] : 0.f;
        }
        __syncthreads();
        float* out = t.out + (int64_t)b * t.C * t.L;
#pragma unroll
        for (int r = ty; r < 32; r += 8) {
            const int c = c0 + r, l = l0 + tx;
            if (c < t.C && l < t.L) out[(int64_t)c * t.L + l] = tile[tx][r];
        }
    }
}

int launch_transpose(const DeviceInfo&, const mugd_transpose& t, cudaStream_t st, int* launches) {
    MUGD_REQUIRE(t.B > 0 && t.C > 0 && t.L > 0 && t.in && t.out, "transpose: bad arguments");
    MUGD_REQUIRE(t.B <= 65535 && (t.C + 31) / 32 <= 65535, "transpose: grid too large");
    if (t.to_nlc) MUGD_REQUIRE(t.ldo >= t.C, "transpose: ldo < C");
    else MUGD_REQUIRE(t.ldi >= t.C, "transpose: ldi < C");
    dim3 grid((t.L + 31) / 32, (t.C + 31) / 32, t.B);
    MUGD_CHECK_CUDA(launch_k(transpose_kernel, grid, dim3(256), 0, st, t));
    if (launches) *launches += 1;
    return MUGD_OK;
}

__global__ void __launch_bounds__(256)
copy2d_kernel(const mugd_copy2d c) {
    pdl_wait();
    const int q = c.cols >> 2;
    const int64_t total = (int64_t)c.rows * q;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = i / q;
        const int cc = (int)(i - r * q) * 4;
        st_f4(c.dst + r * c.ldd + cc, ld_f4(c.src + r * c.lds + cc));
    }
}

int launch_copy2d(const DeviceInfo& dev, const mugd_copy2d& c, cudaStream_t st, int* launches) {
    MUGD_REQUIRE(c.rows > 0 && c.cols > 0 && c.cols % 4 == 0 && c.lds % 4 == 0 && c.ldd % 4 == 0 && aligned16(c.src) && aligned16(c.dst),
                 "copy2d: shape/alignment");
    const int64_t total = (int64_t)c.rows * (c.cols / 4);
    int blocks = (int)((total + 255) / 256);
    if (blocks > dev.sm_count * 8) blocks = dev.sm_count * 8;
    MUGD_CHECK_CUDA(launch_k(copy2d_kernel, dim3(blocks), dim3(256), 0, st, c));
    if (launches) *launches += 1;
    return MUGD_OK;
}

// weight preprocessing for the 3xTF32 GEMM: hi over w, lo beside it (same roundings as the converter warps apply to activations)
__global__ void __launch_bounds__(256)
tf32_split_kernel(float* __restrict__ w_hi, float* __restrict__ lo, int64_t n4) {
    pdl_wait();
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
        const float4 w = ld_f4(w_hi + i * 4);
        float4 h, l;
        uint32_t r;
#define MUGD_RNA(dst, src) asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(src)); dst = __uint_as_float(r)
        MUGD_RNA(h.x, w.x); MUGD_RNA(h.y, w.y); MUGD_RNA(h.z, w.z); MUGD_RNA(h.w, w.w);
        MUGD_RNA(l.x, w.x - h.x); MUGD_RNA(l.y, w.y - h.y); MUGD_RNA(l.z, w.z - h.z); MUGD_RNA(l.w, w.w - h.w);
#undef MUGD_RNA
        st_f4(w_hi + i * 4, h);
        st_f4(lo + i * 4, l);
    }
}

int launch_tf32_split(const DeviceInfo& dev, const mugd_tf32_split& s, cudaStream_t st, int* launches) {
    MUGD_REQUIRE(s.w_hi && s.lo && s.n > 0 && s.n % 4 == 0 && aligned16(s.w_hi) && aligned16(s.lo), "tf32_split: needs 16-byte aligned buffers and n %% 4 == 0");
    const int64_t n4 = s.n / 4;
    int blocks = (int)((n4 + 255) / 256);
    if (blocks > dev.sm_count * 16) blocks = dev.sm_count * 16;
    MUGD_CHECK_CUDA(launch_k(tf32_split_kernel, dim3(blocks), dim3(256), 0, st, s.w_hi, s.lo, n4));
    if (launches) *launches += 1;
    return MUGD_OK;
}

__global__ void step_advance_kernel(int32_t* step) {
    pdl_wait();
    *step += 1;
}
__global__ void fill_i32_kernel(int32_t* p, int32_t v) { *p = v; }

int launch_step_advance(const DeviceInfo&, const mugd_step_advance& a, cudaStream_t st, int* launches) {
    MUGD_REQUIRE(a.step, "step_advance: null counter");
    MUGD_CHECK_CUDA(launch_k(step_advance_kernel, dim3(1), dim3(1), 0, st, a.step));
    if (launches) *launches += 1;
    return MUGD_OK;
}

// ---- note extraction (SURVEY §8f N2): OsuManiaConvertor.array_to_objects, mug/data/convertor.py:232-264 -------------
// One CTA per (key column, chart).  Frames are visited in order in chunks of 256; the notes found in a chunk are
// compacted with a ballot/prefix scan so the output is ordered by frame like the reference's np.where loop.
__global__ void __launch_bounds__(256)
notes_kernel(const mugd_notes n) {
    pdl_wait();
    const int c = blockIdx.x, b = blockIdx.y;
    const int K = n.K, T = n.T;
    const float* Lg = n.logits + (int64_t)b * T * n.ld;
    int32_t* st_out = n.start_ms + ((int64_t)b * K + c) * T;
    int32_t* en_out = n.end_ms + ((int64_t)b * K + c) * T;
    __shared__ int warp_cnt[8];
    __shared__ int base_s;
    if (threadIdx.x == 0) base_s = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int t0 = 0; t0 < T; t0 += 256) {
        const int t = t0 + threadIdx.x;
        bool is = false;
        int start = 0, end = -1;
        if (t < T && Lg[(int64_t)t * n.ld + c] > 0.f) {
            is = true;
            const float so = fminf(fmaxf(Lg[(int64_t)t * n.ld + K + c], 0.f), 1.f);
            start = (int)rint(((double)t + (double)so) * n.frame_ms);           // python round(): half to even
            if (t != T - 1) {
                int i = t + 1;
                while (i < T && Lg[(int64_t)i * n.ld + 2 * K + c] > 0.f && !(Lg[(int64_t)i * n.ld + c] > 0.f)) ++i;
                const int ei = i - 1;
                if (ei != t) {
                    const float eo = fminf(fmaxf(Lg[(int64_t)ei * n.ld + 3 * K + c], 0.f), 1.f);
                    end = (int)rint(((double)ei + (double)eo) * n.frame_ms);
                }
            }
        }
        const unsigned m = __ballot_sync(0xffffffffu, is);
        if (lane == 0) warp_cnt[warp] = __popc(m);
        __syncthreads();
        int off = base_s;
        for (int w = 0; w < warp; ++w) off += warp_cnt[w];
        if (is) {
            const int pos = off + __popc(m & ((1u << lane) - 1u));
            st_out[pos] = start;
            en_out[pos] = end;
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            int tot = 0;
            for (int w = 0; w < 8; ++w) tot += warp_cnt[w];
            base_s += tot;
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) n.count[b * K + c] = base_s;
}

int launch_notes(const DeviceInfo&, const mugd_notes& n, cudaStream_t st, int* launches) {
    MUGD_REQUIRE(n.B > 0 && n.T > 0 && n.K > 0 && n.K <= 16 && n.ld >= 4 * n.K, "notes: bad shape B=%d T=%d K=%d", n.B, n.T, n.K);
    MUGD_REQUIRE(n.logits && n.count && n.start_ms && n.end_ms && n.frame_ms > 0, "notes: null argument");
    MUGD_CHECK_CUDA(launch_k(notes_kernel, dim3(n.K, n.B), dim3(256), 0, st, n));
    if (launches) *launches += 1;
    return MUGD_OK;
}

// ---- prompt embedding (mug/cond/feature.py:15-21): gather + "b f h -> b h f" ------------------------------------------
// One CTA per (sample, feature slot): the table row is read coalesced, the store is strided by F (21 slots x 128 channels per
// sample: 10 KB per request, latency only).
__global__ void __launch_bounds__(128)
embed_kernel(const mugd_embed e) {
    pdl_wait();
    const int f = blockIdx.x, b = blockIdx.y;
    const int id = e.ids[b * e.F + f];
    const float* row = e.table + (int64_t)id * e.H;
    float* out = e.out + (int64_t)b * e.H * e.F + f;
    for (int h = threadIdx.x; h < e.H; h += blockDim.x) out[(int64_t)h * e.F] = row[h];
}

int launch_embed(const DeviceInfo&, const mugd_embed& e, cudaStream_t st, int* launches) {
    MUGD_REQUIRE(e.B > 0 && e.F > 0 && e.H > 0 && e.n_embed > 0, "embed: bad shape B=%d F=%d H=%d n=%d", e.B, e.F, e.H, e.n_embed);
    MUGD_REQUIRE(e.table && e.ids && e.out, "embed: null argument");
    MUGD_REQUIRE(e.B <= 65535, "embed: B=%d too large for one launch", e.B);
    MUGD_CHECK_CUDA(launch_k(embed_kernel, dim3(e.F, e.B), dim3(128), 0, st, e));
    if (launches) *launches += 1;
    return MUGD_OK;
}

}  // namespace mugd

extern "C" int mugd_fill_i32(int32_t* dst, int32_t value, void* stream) {
    using namespace mugd;
    MUGD_REQUIRE(dst, "fill_i32: null");
    fill_i32_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(dst, value);
    MUGD_CHECK_CUDA(cudaGetLastError());
    return MUGD_OK;
}

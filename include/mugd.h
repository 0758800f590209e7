/*
 * mugd.h -- C ABI of libmugd.so, the sm_100a (B200) denoising engine for Mug-Diffusion.
 *
 * The reference (Keytoyze/Mug-Diffusion) has no FFI: its hot path is Python calling ATen.  The boundary
 * this library replaces is therefore the set of Python call sites
 *     DDIMSampler.sample / ddim_sampling / p_sample_ddim   mug/diffusion/ddim.py:56-196
 *     MugDiffusionWrapper.forward -> UNetModel.forward       mug/diffusion/diffusion.py:52-54, unet.py:511-550
 *     MugDiffusionWrapper.decode  -> Decoder.forward         mug/diffusion/diffusion.py:49-50, autoencoder.py:329-354
 * and the entry points below are what a ctypes binding on the reference side would call
 * (INTEGRATION.md shows that binding).  Plain pointers and sizes only: every pointer is a DEVICE pointer
 * into memory the caller owns (torch allocations in the Python host), `stream` is a cudaStream_t passed
 * as void*.  No CPU fallback exists: mugd_create fails on anything that is not compute capability 10.x.
 *
 * Execution model: the host "compiles" a network evaluation into a flat launch plan (array of mugd_op,
 * pointers fully resolved), the library validates it, optionally captures it into a CUDA graph, and
 * replays it once per DDIM step with zero host synchronisation.  Step-dependent data (time-embedding
 * rows, DDIM coefficients) is indexed on the device through a step counter, so one graph serves all steps.
 *
 * Activation layout: channels-last  [B * L, C]  fp32 row-major with explicit leading dimension, so a
 * channel concat is a column range of a wider buffer (unet.py:114-118,545 torch.cat -> zero copies).
 */
#ifndef MUGD_H
#define MUGD_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MUGD_ABI_VERSION 13

typedef struct mugd_handle mugd_handle;   /* one device + scratch state            */
typedef struct mugd_plan mugd_plan;       /* validated launch plan (+ CUDA graph)  */

enum mugd_status {
    MUGD_OK = 0,
    MUGD_ERR_INVALID = 1,      /* bad argument / unsupported shape            */
    MUGD_ERR_CUDA = 2,         /* CUDA runtime error (see mugd_last_error)    */
    MUGD_ERR_NO_DEVICE = 3,    /* not an sm_100 device; there is no fallback  */
    MUGD_ERR_OOM = 4
};

enum mugd_op_kind {
    MUGD_OP_GEMM = 1,          /* Linear / 1x1 conv / conv3 / strided conv / upsample+conv, fused epilogue */
    MUGD_OP_GROUPNORM = 2,     /* GroupNorm(eps) [+ SiLU]                                                    */
    MUGD_OP_LAYERNORM = 3,
    MUGD_OP_ATTENTION = 4,     /* rel-pos-biased softmax attention with post-softmax gain                   */
    MUGD_OP_S4CONV = 5,        /* causal long convolution + D*u + GELU                                       */
    MUGD_OP_DDIM_UPDATE = 6,   /* CFG combine + x_{t-1} update                                              */
    MUGD_OP_TRANSPOSE = 7,     /* [B,C,L] <-> [B,L,C] with leading dimensions                                */
    MUGD_OP_COPY2D = 8,        /* strided row copy                                                           */
    MUGD_OP_STEP_ADVANCE = 9,  /* *step += 1                                                                 */
    MUGD_OP_NOTES = 10,        /* decoder logits -> ordered note list (OsuManiaConvertor.array_to_objects)   */
    MUGD_OP_EMBED = 11,        /* prompt ids -> [B, H, F] embedding (BeatmapFeatureEmbedder.forward)         */
    MUGD_OP_TF32_SPLIT = 12    /* weight preprocessing: w -> (hi in place, lo) for the 3xTF32 tensor-core GEMM */
};

/* A-operand row addressing of MUGD_OP_GEMM (rows are tokens of B samples, Lout output rows each) */
enum mugd_conv_mode {
    MUGD_CONV_NONE = 0,        /* taps=1: Linear / 1x1 conv (unet.py skip_connection, attention.py proj_in)  */
    MUGD_CONV_SAME = 1,        /* taps=3, pad 1: nn.Conv1d(k=3,padding=1)                                    */
    MUGD_CONV_DOWN = 2,        /* taps=3, right-pad 1, stride 2: models.py:84-91 Downsample                  */
    MUGD_CONV_UP = 3,          /* nearest x2 then taps=3 pad 1: models.py:66-70 Upsample                     */
    MUGD_CONV_TAPS = 4         /* `taps` consecutive rows l+tap_shift .. (zero outside the sample), Lin == Lout: the
                                  two parity halves of Upsample (y[2j] = W0 x[j-1] + (W1+W2) x[j],
                                  y[2j+1] = (W0+W1) x[j] + W2 x[j+1]) run as 2-tap GEMMs on half the rows         */
};
enum mugd_act { MUGD_ACT_NONE = 0, MUGD_ACT_SILU = 1, MUGD_ACT_GELU = 2 };
/* gated epilogues: weight rows are interleaved (value_j, gate_j) by the packer; output has N/2 columns */
enum mugd_gate { MUGD_GATE_NONE = 0, MUGD_GATE_GEGLU = 1 /* a*gelu(g), attention.py:38-45 */,
                 MUGD_GATE_GLU = 2 /* a*sigmoid(g), s4.py:191-192,1536 */ };
enum mugd_gemm_impl { MUGD_GEMM_AUTO = 0, MUGD_GEMM_SIMT = 1 /* exact fp32 FMA */,
                      MUGD_GEMM_TC = 2 /* tcgen05 3xTF32 split, fp32 accumulate in TMEM */ };
/* tile variant of the tensor-core GEMM (mugd_gemm.tc_variant): AUTO = the planner's cost model; the others force a variant where
 * the shape allows it (a tile wider than N falls back to the 128- or 64-wide tile; N128_2CTA together with split_k > 1 falls back to
 * the 128-wide one-CTA-per-SM tile with that split) */
enum mugd_tc_variant { MUGD_TC_AUTO = 0, MUGD_TC_N64 = 1, MUGD_TC_N128 = 2, MUGD_TC_N256 = 3,
                       MUGD_TC_N128_2CTA = 4 /* 128 wide, two CTAs per SM walking a tile list */ };

typedef struct mugd_gemm {
    const float* A;  int64_t lda;          /* [B*Lin, K] activations                                       */
    const float* W;                        /* [N][taps*K], K-major per tap (conv weight [Cout][k][Cin])    */
    const float* W_hi;                     /* optional: W rounded to TF32 (rna)            } tensor-core path, */
    const float* W_lo;                     /* optional: rna_tf32(W - W_hi)                 } same layout as W  */
    const float* bias;                     /* [N] or NULL                                                  */
    const float* rowvec;                   /* per-sample row vector added before act: time embedding       */
    int64_t rowvec_b_stride;               /*   rowvec[step*step_stride + b*b_stride + n]                  */
    int64_t rowvec_step_stride;
    const int32_t* step;                   /* device step counter or NULL (=0)                             */
    const float* residual; int64_t ldr;    /* added after act/gate, or NULL                                */
    float* C;        int64_t ldc;          /* [B*Lout, N] (N/2 when gated)                                 */
    int32_t M, N, K;                       /* M = B*Lout rows, N weight rows, K channels per tap           */
    int32_t taps, conv_mode, Lin, Lout;
    int32_t act, gate, impl;
    int32_t split_k;                       /* tensor-core path: 0 = auto, >0 forces the K split            */
    int32_t tap_shift;                     /* MUGD_CONV_TAPS: source row of tap t is l + (t + tap_shift) * dilation */
    int32_t tap_dilation;                  /* MUGD_CONV_TAPS: 0/1 = dense taps; d = dilated conv (wave.py:425-433)  */
    void* workspace; int64_t workspace_bytes; /* split-K partial tiles (see mugd_gemm_tc_query)            */
    /* optional SECOND activation source: K2 more channels read at the output row itself (a 1x1 term), weights in columns
     * taps*K .. taps*K+K2 of every W row.  One GEMM then computes  conv3(A) + conv1(A2):  out_layers conv + skip_connection
     * of a TimestepResBlock (unet.py:187-193,237-239), and  proj_out(ff.net.2(ff) + h) = (Wp Wf) ff + Wp h  of the transformer
     * block (attention.py:57-65,194-199) with the packer-composed weight.  NULL / 0 = single source. */
    const float* A2; int64_t lda2;         /* [B*Lout, K2]                                                 */
    int32_t K2;
    int32_t tc_variant;                    /* tensor-core path: enum mugd_tc_variant, 0 = auto             */
    /* Row moments of the OUTPUT for a LayerNorm that follows (tensor-core path, act == gate == NONE only): while the tile is stored,
     * row_moments[m*2 + {0,1}] += {sum, sum of squares} of the columns of output row m (fp64 atomics; the plan zeroes the buffer at
     * the start of every evaluation).  Round 2 also built GroupNorm-moment sinks + a single-pass apply kernel; they lost at every batch
     * size (profiles/r02_norm_fusion_ab.md) and were removed. */
    double* row_moments;
    /* LayerNorm folded into this GEMM (attention.py:147-151: norm_i followed by a Linear): with W' = W diag(gamma) packed as the
     * weight, colsum[n] = sum_k W'[n][k] and bias' = W beta + b,   C = rstd_m * (A W'^T - mean_m * colsum) + bias'   where mean_m,
     * rstd_m come from the row moments ln_stats[m*2 + {0,1}] = {sum, sum of squares} over the K channels of A's row m (the row_moments
     * of A's producer).  The normalised tensor is never materialised.  NULL = plain GEMM. */
    const double* ln_stats; const float* ln_colsum; float ln_eps; int32_t reserved2_;
} mugd_gemm;

typedef struct mugd_groupnorm {
    const float* x; int64_t ldx; float* y; int64_t ldy;
    const float* gamma; const float* beta;
    int32_t B, L, C, G; float eps; int32_t silu;
} mugd_groupnorm;

typedef struct mugd_layernorm {
    const float* x; int64_t ldx; float* y; int64_t ldy;
    const float* gamma; const float* beta;
    int32_t rows, C; float eps;
} mugd_layernorm;

typedef struct mugd_attention {
    const float* q; int64_t ldq;           /* [B*Lq, H*D] head h at columns h*D..                          */
    const float* k; int64_t ldk;           /* [B*Lk, H*D]                                                  */
    const float* v; int64_t ldv;
    float* o; int64_t ldo;
    const float* relpos;                   /* [2*pos_max+1][H] additive, inside the scale (attention.py:113) */
    const float* cgain;                    /* [2*pos_max+1][H] post-softmax multiplier (attention.py:122)   */
    int32_t B, H, D, Lq, Lk, pos_max; float scale;
} mugd_attention;

typedef struct mugd_s4conv {
    const float* u; int64_t ldu;           /* [B*L, H]                                                     */
    const float* Kt;                       /* [L][H] kernel taps, tap-major (from mugd_s4_kernel_gen)      */
    const float* D;                        /* [H]                                                          */
    float* y; int64_t ldy;                 /* gelu(conv + D*u)                                             */
    int32_t B, L, H;
} mugd_s4conv;

typedef struct mugd_ddim_update {
    float* x;                              /* [B*L, C] in place -> x_{t-1}                                  */
    float* x_dup;                          /* optional second copy of x_{t-1} (the cfg half of the 2B batch) */
    const float* eps;                      /* [Beff*L, C]; Beff = 2B when cfg (uncond first, ddim.py:173)   */
    const float* noise;                    /* [B*L, C] or NULL (sigma = 0)                                  */
    float* pred_x0;                        /* [B*L, C] or NULL                                              */
    const float* coef;                     /* [S][4] = a_t, a_prev, sigma_t, sqrt(1-a_t) per DDIM index     */
    const int32_t* step;                   /* device step counter i; row used = S-1-i (ddim.py:138)         */
    int32_t S; int32_t n;                  /* n = B*L*C elements                                            */
    int32_t cfg; float scale; float temperature;
} mugd_ddim_update;

typedef struct mugd_transpose {            /* to_nlc=1: in [B,C,L] (contiguous) -> out [B*L, ldo] cols 0..C  */
    const float* in; float* out;           /* to_nlc=0: in [B*L, ldi] -> out [B,C,L]                          */
    int64_t ldi, ldo; int32_t B, C, L, to_nlc;
} mugd_transpose;

typedef struct mugd_copy2d {
    const float* src; int64_t lds; float* dst; int64_t ldd; int32_t rows, cols;
} mugd_copy2d;

typedef struct mugd_step_advance { int32_t* step; } mugd_step_advance;

/* Note extraction, mug/data/convertor.py:232-264 (from_logits): for key column c of chart b a note starts at every frame
 * t with logit[t][c] > 0; start = round((t + clip(logit[t][K+c],0,1)) * frame_ms); it is a long note when the following
 * frames have logit[.][2K+c] > 0 and no new start, end = round((t_end + clip(logit[t_end][3K+c],0,1)) * frame_ms), else -1.
 * Output is compact and ordered by frame per (chart, column): count[b*K+c], start_ms/end_ms[(b*K+c)*T + i]. */
typedef struct mugd_notes {
    const float* logits; int64_t ld;       /* [B*T, 4K] channels-last decoder output                        */
    int32_t* count; int32_t* start_ms; int32_t* end_ms;
    double frame_ms;
    int32_t B, T, K;
} mugd_notes;

/* Prompt embedding, mug/cond/feature.py:15-21 (BeatmapFeatureEmbedder.forward): out[b][h][f] = table[ids[b][f]][h], the
 * nn.Embedding lookup followed by rearrange "b f h -> b h f".  ids must lie in [0, n_embed) (the host checks, like torch). */
typedef struct mugd_embed {
    const float* table;                    /* [n_embed, H] row-major                                         */
    const int32_t* ids;                    /* [B, F]                                                         */
    float* out;                            /* [B, H, F]                                                      */
    int32_t B, F, H, n_embed;
} mugd_embed;

/* hi = rna_tf32(w) written over w, lo = rna_tf32(w - hi): the two TF32 operands whose products reconstruct an fp32 weight.
 * Run once per engine after the (plain fp32) weight blob has reached the device -- the blob that is packed, stored and broadcast holds
 * every weight once; the resident copy holds hi + lo of the tensor-core weights and no plain duplicate. */
typedef struct mugd_tf32_split { float* w_hi; float* lo; int64_t n; } mugd_tf32_split;

typedef struct mugd_op {
    int32_t kind;
    int32_t tag;                           /* free for the host (profiling labels)                          */
    union {
        mugd_gemm gemm; mugd_groupnorm gn; mugd_layernorm ln; mugd_attention attn; mugd_s4conv s4;
        mugd_ddim_update ddim; mugd_transpose tr; mugd_copy2d cp; mugd_step_advance adv; mugd_notes notes;
        mugd_embed embed; mugd_tf32_split split;
    } u;
} mugd_op;

/* ---- lifecycle -------------------------------------------------------------------------------- */
int  mugd_abi_version(void);
const char* mugd_last_error(void);                         /* thread-local message of the last failure */
int  mugd_create(int device, mugd_handle** out);           /* MUGD_ERR_NO_DEVICE unless sm_100          */
void mugd_destroy(mugd_handle* h);
int  mugd_device_info(mugd_handle* h, int32_t* sm_count, int32_t* cc_major, int32_t* cc_minor);
int  mugd_set_gemm_impl(mugd_handle* h, int impl);         /* default for ops with impl == AUTO         */

/* ---- single op (parity tests call every kernel through this) ---------------------------------- */
int  mugd_op_run(mugd_handle* h, const mugd_op* op, void* stream);

/* ---- plans ------------------------------------------------------------------------------------ */
int  mugd_plan_create(mugd_handle* h, const mugd_op* ops, int32_t n_ops, mugd_plan** out);
int  mugd_plan_run(mugd_plan* p, void* stream);            /* eager launches                            */
int  mugd_plan_capture(mugd_plan* p, void* stream);        /* build + instantiate a CUDA graph          */
int  mugd_plan_replay(mugd_plan* p, int32_t times, void* stream); /* launch the graph `times` times     */
int  mugd_plan_launch_count(mugd_plan* p);                 /* kernels launched by one run of the plan   */
void mugd_plan_destroy(mugd_plan* p);

/* ---- the sampler loop from ONE call: DDIMSampler.ddim_sampling's for-loop (ddim.py:136-157) -------------------------------
 * n_steps x { replay the captured evaluation plan (one CUDA graph = Beff U-Net evaluations) ; run the `tail` ops eagerly on the same
 * stream: MUGD_OP_DDIM_UPDATE (CFG combine + x_{t-1}) and MUGD_OP_STEP_ADVANCE (device step counter) }.  Nothing synchronises; the
 * step-dependent rows (time embedding, DDIM coefficients) are selected on the device by the counter.  `eval_plan` must be captured. */
int  mugd_sample(mugd_plan* eval_plan, const mugd_op* tail, int32_t n_tail, int32_t n_steps, void* stream);

/* ---- plans on disk: a host without Python (examples/host_c) loads what the Python plan compiler produced ---------------------
 * Every pointer of a plan lies in one of a few device allocations ("regions": weight blob, activation arena, side tables, the
 * caller's staging buffers).  mugd_plan_save stores each pointer as (region, offset); mugd_plan_load resolves them against the
 * loader's allocations, matched by name (each at least as large as recorded).  Region contents are the caller's business. */
typedef struct mugd_region { const char* name; void* base; int64_t bytes; } mugd_region;
int  mugd_plan_save(mugd_plan* p, const mugd_region* regions, int32_t n_regions, const char* path);
int  mugd_plan_load(mugd_handle* h, const char* path, const mugd_region* regions, int32_t n_regions, mugd_plan** out);
/* the (relocated) ops of a plan, e.g. to hand a loaded update/advance plan to mugd_sample as its tail; owned by the plan */
int  mugd_plan_ops(mugd_plan* p, const mugd_op** ops, int32_t* n_ops);
/* names and sizes of the regions a plan file refers to (names[i] receives the text, out[i].name points at it); n_regions always set */
int  mugd_plan_regions(const char* path, mugd_region* out, char (*names)[48], int32_t max_regions, int32_t* n_regions);

/* ---- S4 kernel generation: SSKernelNPLR.forward, s4.py:706-832 (once per model and length) ----- */
int  mugd_s4_kernel_gen(mugd_handle* h,
                        const float* log_dt,      /* [H]        */
                        const float* Bri,         /* [H][N][2]  */
                        const float* Cri,         /* [H][N][2]  */
                        const float* Pri,         /* [H][N][2]  */
                        const float* inv_w_real,  /* [H][N]     */
                        const float* w_imag,      /* [H][N]     */
                        const float* omega_ri,    /* [L_internal/2+1][2] FFT nodes as the reference computes them
                                                     (complex64 omega**arange, s4.py:595-598) or NULL = exact */
                        int32_t H, int32_t N, int32_t L_internal, int32_t L_out,
                        float* Kt,                /* [L_out][H] */
                        void* workspace, int64_t workspace_bytes, /* >= 16*H*(L_internal/2+1) bytes */
                        void* stream);

/* ---- tensor-core GEMM planning: is this GEMM taken by the tcgen05 kernel, with which K split, and how much
 * split-K workspace does it need (the host allocates it once per plan) ------ */
int  mugd_gemm_tc_query(mugd_handle* h, const mugd_gemm* g, int32_t sm_count, int32_t* supported, int32_t* splits,
                        int64_t* workspace_bytes, int32_t* n_tiles);
/* which kernel variant the planner picks for this GEMM on a machine with sm_count SMs: tile width (64 / 128 / 256; 0 = not taken by the
 * tensor-core kernel), CTAs per SM it is built for (1, or 2 = the 128-wide variant whose CTAs walk a tile list), CTAs launched */
int  mugd_gemm_tc_variant(const mugd_gemm* g, int32_t sm_count, int32_t* tile_n, int32_t* ctas_per_sm, int32_t* grid_ctas);

/* ---- per-handle switches -------------------------------------------------------------------------
 * OPT-IN speed mode of the tensor-core GEMM: 1 = plain TF32 products (a_hi*w_hi only, ~2^-11 relative error per product, like
 * cuDNN's allow_tf32 that the reference's own GPU path uses for convs); 0 (default) = 3xTF32, fp32-accurate.  Parity tests and
 * bench.py use 0.  Plans created (and graphs captured) earlier keep the mode they were created with. */
int  mugd_set_tc_single_pass_tf32(mugd_handle* h, int enabled);

/* attention kernel: 1 (default) = QK^T and PV on the tcgen05 tensor cores (3xTF32, fp32 accuracy); 0 = exact-fp32 FFMA kernel
 * (the referee of the parity tests).  Replaces the einsum/softmax body of CrossAttention.forward, attention.py:99-121 */
int  mugd_set_attention_impl(mugd_handle* h, int impl);

/* ---- measurement aid ------------------------------------------------------------------------------------
 * builds with -DMUGD_TC_TIMELINE only (tools/build_variant.py): CTA (0,0,0) of every tensor-core GEMM launch writes
 * %globaltimer stamps into the device buffer (tools/gemm_timeline.py); otherwise returns MUGD_ERR_INVALID */
int  mugd_debug_set_tc_timing(long long* device_buf);

/* ---- utility ---------------------------------------------------------------------------------- */
int  mugd_fill_i32(int32_t* dst, int32_t value, void* stream);
/* sizeof() of {mugd_op, mugd_gemm, mugd_groupnorm, mugd_layernorm, mugd_attention, mugd_s4conv,
 * mugd_ddim_update, mugd_transpose, mugd_copy2d, mugd_notes, mugd_embed, mugd_tf32_split} so a foreign-language mirror can verify its layout */
int  mugd_abi_sizes(int32_t* out, int32_t n);

#ifdef __cplusplus
}
#endif
#endif /* MUGD_H */

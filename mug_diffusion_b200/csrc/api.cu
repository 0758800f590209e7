// C ABI glue of libmugd: handle, op dispatch, launch plans and CUDA-graph capture/replay.
#include <stdarg.h>
#include <string.h>

#include <vector>

#include "common.cuh"

namespace mugd {

static thread_local char g_err[1024] = "";

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

}  // namespace mugd

struct mugd_handle {
    mugd::DeviceInfo dev;
    int default_gemm_impl = MUGD_GEMM_SIMT;
};

struct mugd_plan {
    mugd_handle* h = nullptr;
    std::vector<mugd_op> ops;
    cudaGraph_t graph = nullptr;
    cudaGraphExec_t exec = nullptr;
    int launches = 0;
};

namespace mugd {

const std::vector<mugd_op>& plan_ops(const mugd_plan* p) { return p->ops; }
int plan_from_ops(mugd_handle* h, const mugd_op* ops, int32_t n, mugd_plan** out) { return mugd_plan_create(h, ops, n, out); }

static int dispatch(mugd_handle* h, const mugd_op& op, cudaStream_t st, int* launches) {
    switch (op.kind) {
        case MUGD_OP_GEMM: return launch_gemm(h->dev, op.u.gemm, h->default_gemm_impl, st, launches);
        case MUGD_OP_GROUPNORM: return launch_groupnorm(h->dev, op.u.gn, st, launches);
        case MUGD_OP_LAYERNORM: return launch_layernorm(h->dev, op.u.ln, st, launches);
        case MUGD_OP_ATTENTION: return launch_attention(h->dev, op.u.attn, st, launches);
        case MUGD_OP_S4CONV: return launch_s4conv(h->dev, op.u.s4, st, launches);
        case MUGD_OP_DDIM_UPDATE: return launch_ddim_update(h->dev, op.u.ddim, st, launches);
        case MUGD_OP_TRANSPOSE: return launch_transpose(h->dev, op.u.tr, st, launches);
        case MUGD_OP_COPY2D: return launch_copy2d(h->dev, op.u.cp, st, launches);
        case MUGD_OP_STEP_ADVANCE: return launch_step_advance(h->dev, op.u.adv, st, launches);
        case MUGD_OP_NOTES: return launch_notes(h->dev, op.u.notes, st, launches);
        case MUGD_OP_EMBED: return launch_embed(h->dev, op.u.embed, st, launches);
        case MUGD_OP_TF32_SPLIT: return launch_tf32_split(h->dev, op.u.split, st, launches);
        default:
            set_error("unknown op kind %d", op.kind);
            return MUGD_ERR_INVALID;
    }
}

}  // namespace mugd

using namespace mugd;

extern "C" {

int mugd_abi_version(void) { return MUGD_ABI_VERSION; }

const char* mugd_last_error(void) { return g_err; }

int mugd_create(int device, mugd_handle** out) {
    MUGD_REQUIRE(out, "mugd_create: null out");
    *out = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n <= 0 || device < 0 || device >= n) {
        set_error("mugd_create: no CUDA device %d (count=%d, %s). libmugd has no CPU fallback.", device, n,
                  e == cudaSuccess ? "ok" : cudaGetErrorString(e));
        return MUGD_ERR_NO_DEVICE;
    }
    cudaDeviceProp prop;
    MUGD_CHECK_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) {
        set_error("mugd_create: device %d is sm_%d%d; libmugd is built for sm_100a (B200) only", device, prop.major, prop.minor);
        return MUGD_ERR_NO_DEVICE;
    }
    MUGD_CHECK_CUDA(cudaSetDevice(device));
    DeviceInfo dev;
    dev.device = device;
    dev.sm_count = prop.multiProcessorCount;
    dev.cc_major = prop.major;
    dev.cc_minor = prop.minor;
    dev.max_smem_optin = (int)prop.sharedMemPerBlockOptin;
    int rc = configure_gemm_tc_kernels(dev);
    if (rc == MUGD_OK) rc = configure_attention_kernels(dev);
    if (rc == MUGD_OK) rc = configure_attention_tc_kernels(dev);
    if (rc == MUGD_OK) rc = configure_s4_kernels(dev);
    if (rc != MUGD_OK) return rc;
    mugd_handle* h = new mugd_handle();
    h->dev = dev;
    *out = h;
    return MUGD_OK;
}

void mugd_destroy(mugd_handle* h) { delete h; }

int mugd_device_info(mugd_handle* h, int32_t* sm_count, int32_t* cc_major, int32_t* cc_minor) {
    MUGD_REQUIRE(h, "null handle");
    if (sm_count) *sm_count = h->dev.sm_count;
    if (cc_major) *cc_major = h->dev.cc_major;
    if (cc_minor) *cc_minor = h->dev.cc_minor;
    return MUGD_OK;
}

int mugd_set_gemm_impl(mugd_handle* h, int impl) {
    MUGD_REQUIRE(h, "null handle");
    MUGD_REQUIRE(impl == MUGD_GEMM_SIMT || impl == MUGD_GEMM_TC, "set_gemm_impl: %d", impl);
    h->default_gemm_impl = impl;
    return MUGD_OK;
}

int mugd_set_tc_single_pass_tf32(mugd_handle* h, int enabled) {
    MUGD_REQUIRE(h, "null handle");
    h->dev.tc_single_pass = enabled ? 1 : 0;
    return MUGD_OK;
}

int mugd_set_attention_impl(mugd_handle* h, int impl) {
    MUGD_REQUIRE(h, "null handle");
    h->dev.attention_impl = impl ? 1 : 0;
    return MUGD_OK;
}

int mugd_op_run(mugd_handle* h, const mugd_op* op, void* stream) {
    MUGD_REQUIRE(h && op, "mugd_op_run: null argument");
    return dispatch(h, *op, (cudaStream_t)stream, nullptr);
}

int mugd_plan_create(mugd_handle* h, const mugd_op* ops, int32_t n_ops, mugd_plan** out) {
    MUGD_REQUIRE(h && ops && out && n_ops > 0, "mugd_plan_create: bad arguments");
    mugd_plan* p = new mugd_plan();
    p->h = h;
    p->ops.assign(ops, ops + n_ops);
    *out = p;
    return MUGD_OK;
}

int mugd_plan_run(mugd_plan* p, void* stream) {
    MUGD_REQUIRE(p, "null plan");
    int launches = 0;
    for (size_t i = 0; i < p->ops.size(); ++i) {
        int rc = dispatch(p->h, p->ops[i], (cudaStream_t)stream, &launches);
        if (rc != MUGD_OK) {
            char prev[900];
            strncpy(prev, g_err, sizeof(prev) - 1);
            prev[sizeof(prev) - 1] = 0;
            set_error("plan op %zu (kind %d, tag %d): %s", i, p->ops[i].kind, p->ops[i].tag, prev);
            return rc;
        }
    }
    p->launches = launches;
    return MUGD_OK;
}

int mugd_plan_capture(mugd_plan* p, void* stream) {
    MUGD_REQUIRE(p, "null plan");
    cudaStream_t st = (cudaStream_t)stream;
    MUGD_REQUIRE(st != nullptr, "plan_capture: needs a non-default stream");
    if (p->exec) { cudaGraphExecDestroy(p->exec); p->exec = nullptr; }
    if (p->graph) { cudaGraphDestroy(p->graph); p->graph = nullptr; }
    MUGD_CHECK_CUDA(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
    int rc = mugd_plan_run(p, stream);
    cudaGraph_t g = nullptr;
    cudaError_t e = cudaStreamEndCapture(st, &g);
    if (rc != MUGD_OK) {
        if (g) cudaGraphDestroy(g);
        return rc;
    }
    if (e != cudaSuccess) {
        set_error("cudaStreamEndCapture: %s", cudaGetErrorString(e));
        return MUGD_ERR_CUDA;
    }
    p->graph = g;
    MUGD_CHECK_CUDA(cudaGraphInstantiate(&p->exec, p->graph, 0));
    return MUGD_OK;
}

int mugd_plan_replay(mugd_plan* p, int32_t times, void* stream) {
    MUGD_REQUIRE(p && p->exec, "plan_replay: plan not captured");
    for (int i = 0; i < times; ++i) MUGD_CHECK_CUDA(cudaGraphLaunch(p->exec, (cudaStream_t)stream));
    return MUGD_OK;
}

int mugd_sample(mugd_plan* eval_plan, const mugd_op* tail, int32_t n_tail, int32_t n_steps, void* stream) {
    MUGD_REQUIRE(eval_plan && eval_plan->exec, "mugd_sample: the evaluation plan must be captured (mugd_plan_capture)");
    MUGD_REQUIRE(n_steps >= 0 && n_tail >= 0 && (n_tail == 0 || tail), "mugd_sample: bad arguments");
    cudaStream_t st = (cudaStream_t)stream;
    for (int i = 0; i < n_steps; ++i) {
        MUGD_CHECK_CUDA(cudaGraphLaunch(eval_plan->exec, st));
        for (int k = 0; k < n_tail; ++k) {
            int rc = dispatch(eval_plan->h, tail[k], st, nullptr);
            if (rc != MUGD_OK) return rc;
        }
    }
    return MUGD_OK;
}

int mugd_abi_sizes(int32_t* out, int32_t n) {
    MUGD_REQUIRE(out && n >= 12, "abi_sizes: need room for 12 entries");
    out[0] = sizeof(mugd_op); out[1] = sizeof(mugd_gemm); out[2] = sizeof(mugd_groupnorm);
    out[3] = sizeof(mugd_layernorm); out[4] = sizeof(mugd_attention); out[5] = sizeof(mugd_s4conv);
    out[6] = sizeof(mugd_ddim_update); out[7] = sizeof(mugd_transpose); out[8] = sizeof(mugd_copy2d);
    out[9] = sizeof(mugd_notes); out[10] = sizeof(mugd_embed); out[11] = sizeof(mugd_tf32_split);
    return MUGD_OK;
}

int mugd_plan_ops(mugd_plan* p, const mugd_op** ops, int32_t* n_ops) {
    MUGD_REQUIRE(p && ops && n_ops, "plan_ops: bad arguments");
    *ops = p->ops.data();
    *n_ops = (int32_t)p->ops.size();
    return MUGD_OK;
}

int mugd_plan_launch_count(mugd_plan* p) { return p ? p->launches : 0; }

void mugd_plan_destroy(mugd_plan* p) {
    if (!p) return;
    if (p->exec) cudaGraphExecDestroy(p->exec);
    if (p->graph) cudaGraphDestroy(p->graph);
    delete p;
}

}  // extern "C"

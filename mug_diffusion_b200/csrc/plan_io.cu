// Launch plans on disk: mugd_plan_save / mugd_plan_load, so that a host WITHOUT Python can run the sampler.
//
// The plan compiler (which network op becomes which launch, where every tensor lives) is Python (mug_diffusion_b200/engine.py).
// A compiled plan, however, is just an array of mugd_op whose pointers all fall into a handful of device allocations ("regions":
// the weight blob, the activation arena, the per-request side tables, the staging buffers of the caller).  Saving rewrites every
// pointer as (region, offset); loading resolves them against the loader's own allocations of the same names.  Region CONTENTS
// (weights, S4 kernels) are the caller's business -- tools/export_bundle.py writes them next to the plans, examples/host_c loads them.
//
// File layout (little endian): magic "MUGDPLN1" | abi u32 | n_regions u32 | n_ops u32 | n_reloc u32 | sizeof(mugd_op) u32 | pad u32
//   n_regions x { char name[48]; i64 bytes }   n_ops x mugd_op (pointer fields hold offsets)   n_reloc x { u32 op; u32 field; u32 region; u32 pad }
#include <stddef.h>
#include <stdio.h>

#include <vector>

#include "common.cuh"

namespace mugd {

struct PtrField { int kind; size_t off; };
#define PF(kind, member) {kind, offsetof(mugd_op, u.member)}
static const PtrField k_ptr_fields[] = {
    PF(MUGD_OP_GEMM, gemm.A), PF(MUGD_OP_GEMM, gemm.W), PF(MUGD_OP_GEMM, gemm.W_hi), PF(MUGD_OP_GEMM, gemm.W_lo), PF(MUGD_OP_GEMM, gemm.bias),
    PF(MUGD_OP_GEMM, gemm.rowvec), PF(MUGD_OP_GEMM, gemm.step), PF(MUGD_OP_GEMM, gemm.residual), PF(MUGD_OP_GEMM, gemm.C),
    PF(MUGD_OP_GEMM, gemm.workspace), PF(MUGD_OP_GEMM, gemm.A2), PF(MUGD_OP_GEMM, gemm.row_moments),
    PF(MUGD_OP_GEMM, gemm.ln_stats), PF(MUGD_OP_GEMM, gemm.ln_colsum),
    PF(MUGD_OP_GROUPNORM, gn.x), PF(MUGD_OP_GROUPNORM, gn.y), PF(MUGD_OP_GROUPNORM, gn.gamma), PF(MUGD_OP_GROUPNORM, gn.beta),
    PF(MUGD_OP_LAYERNORM, ln.x), PF(MUGD_OP_LAYERNORM, ln.y), PF(MUGD_OP_LAYERNORM, ln.gamma), PF(MUGD_OP_LAYERNORM, ln.beta),
    PF(MUGD_OP_ATTENTION, attn.q), PF(MUGD_OP_ATTENTION, attn.k), PF(MUGD_OP_ATTENTION, attn.v), PF(MUGD_OP_ATTENTION, attn.o),
    PF(MUGD_OP_ATTENTION, attn.relpos), PF(MUGD_OP_ATTENTION, attn.cgain),
    PF(MUGD_OP_S4CONV, s4.u), PF(MUGD_OP_S4CONV, s4.Kt), PF(MUGD_OP_S4CONV, s4.D), PF(MUGD_OP_S4CONV, s4.y),
    PF(MUGD_OP_DDIM_UPDATE, ddim.x), PF(MUGD_OP_DDIM_UPDATE, ddim.x_dup), PF(MUGD_OP_DDIM_UPDATE, ddim.eps), PF(MUGD_OP_DDIM_UPDATE, ddim.noise),
    PF(MUGD_OP_DDIM_UPDATE, ddim.pred_x0), PF(MUGD_OP_DDIM_UPDATE, ddim.coef), PF(MUGD_OP_DDIM_UPDATE, ddim.step),
    PF(MUGD_OP_TRANSPOSE, tr.in), PF(MUGD_OP_TRANSPOSE, tr.out),
    PF(MUGD_OP_COPY2D, cp.src), PF(MUGD_OP_COPY2D, cp.dst),
    PF(MUGD_OP_STEP_ADVANCE, adv.step),
    PF(MUGD_OP_NOTES, notes.logits), PF(MUGD_OP_NOTES, notes.count), PF(MUGD_OP_NOTES, notes.start_ms), PF(MUGD_OP_NOTES, notes.end_ms),
    PF(MUGD_OP_EMBED, embed.table), PF(MUGD_OP_EMBED, embed.ids), PF(MUGD_OP_EMBED, embed.out),
    PF(MUGD_OP_TF32_SPLIT, split.w_hi), PF(MUGD_OP_TF32_SPLIT, split.lo),
};
#undef PF

struct FileHeader { char magic[8]; uint32_t abi, n_regions, n_ops, n_reloc, op_size, pad; };
struct FileRegion { char name[48]; int64_t bytes; };
struct FileReloc { uint32_t op, field, region, pad; };

static uintptr_t& ptr_at(mugd_op& op, size_t off) { return *reinterpret_cast<uintptr_t*>(reinterpret_cast<char*>(&op) + off); }

const std::vector<mugd_op>& plan_ops(const mugd_plan* p);                               // api.cu
int plan_from_ops(mugd_handle* h, const mugd_op* ops, int32_t n, mugd_plan** out);      // api.cu

}  // namespace mugd

using namespace mugd;

extern "C" int mugd_plan_save(mugd_plan* p, const mugd_region* regions, int32_t n_regions, const char* path) {
    MUGD_REQUIRE(p && regions && n_regions > 0 && path, "plan_save: bad arguments");
    std::vector<mugd_op> ops = plan_ops(p);
    std::vector<FileReloc> rel;
    for (size_t i = 0; i < ops.size(); ++i) {
        for (const PtrField& f : k_ptr_fields) {
            if (f.kind != ops[i].kind) continue;
            uintptr_t& v = ptr_at(ops[i], f.off);
            if (!v) continue;
            int found = -1;
            for (int r = 0; r < n_regions; ++r) {
                const uintptr_t b = reinterpret_cast<uintptr_t>(regions[r].base);
                if (v >= b && v < b + (uintptr_t)regions[r].bytes) { found = r; break; }
            }
            MUGD_REQUIRE(found >= 0, "plan_save: op %zu (kind %d) has a pointer (field offset %zu) outside every registered region", i, ops[i].kind, f.off);
            v -= reinterpret_cast<uintptr_t>(regions[found].base);
            rel.push_back({(uint32_t)i, (uint32_t)f.off, (uint32_t)found, 0u});
        }
    }
    FILE* fp = fopen(path, "wb");
    MUGD_REQUIRE(fp, "plan_save: cannot open %s", path);
    FileHeader h = {{'M', 'U', 'G', 'D', 'P', 'L', 'N', '1'}, MUGD_ABI_VERSION, (uint32_t)n_regions, (uint32_t)ops.size(), (uint32_t)rel.size(),
                    (uint32_t)sizeof(mugd_op), 0u};
    bool ok = fwrite(&h, sizeof(h), 1, fp) == 1;
    for (int r = 0; r < n_regions && ok; ++r) {
        FileRegion fr;
        memset(&fr, 0, sizeof(fr));
        strncpy(fr.name, regions[r].name ? regions[r].name : "", sizeof(fr.name) - 1);
        fr.bytes = regions[r].bytes;
        ok = fwrite(&fr, sizeof(fr), 1, fp) == 1;
    }
    ok = ok && fwrite(ops.data(), sizeof(mugd_op), ops.size(), fp) == ops.size();
    ok = ok && (rel.empty() || fwrite(rel.data(), sizeof(FileReloc), rel.size(), fp) == rel.size());
    fclose(fp);
    MUGD_REQUIRE(ok, "plan_save: short write to %s", path);
    return MUGD_OK;
}

extern "C" int mugd_plan_load(mugd_handle* h, const char* path, const mugd_region* regions, int32_t n_regions, mugd_plan** out) {
    MUGD_REQUIRE(h && path && regions && out, "plan_load: bad arguments");
    *out = nullptr;
    FILE* fp = fopen(path, "rb");
    MUGD_REQUIRE(fp, "plan_load: cannot open %s", path);
    FileHeader fh;
    bool ok = fread(&fh, sizeof(fh), 1, fp) == 1 && memcmp(fh.magic, "MUGDPLN1", 8) == 0;
    if (!ok) { fclose(fp); MUGD_REQUIRE(false, "plan_load: %s is not a libmugd plan file", path); }
    if (fh.abi != MUGD_ABI_VERSION || fh.op_size != sizeof(mugd_op)) {
        fclose(fp);
        MUGD_REQUIRE(false, "plan_load: %s was written by ABI %u (op size %u), this library is ABI %d (op size %zu)", path, fh.abi, fh.op_size,
                     MUGD_ABI_VERSION, sizeof(mugd_op));
    }
    std::vector<FileRegion> fr(fh.n_regions);
    std::vector<mugd_op> ops(fh.n_ops);
    std::vector<FileReloc> rel(fh.n_reloc);
    ok = fread(fr.data(), sizeof(FileRegion), fr.size(), fp) == fr.size() && fread(ops.data(), sizeof(mugd_op), ops.size(), fp) == ops.size() &&
         (rel.empty() || fread(rel.data(), sizeof(FileReloc), rel.size(), fp) == rel.size());
    fclose(fp);
    MUGD_REQUIRE(ok, "plan_load: %s is truncated", path);
    // resolve the file's regions by name against the caller's allocations
    std::vector<int> map(fr.size(), -1);
    for (size_t i = 0; i < fr.size(); ++i) {
        for (int r = 0; r < n_regions; ++r)
            if (regions[r].name && strncmp(fr[i].name, regions[r].name, sizeof(fr[i].name)) == 0) { map[i] = r; break; }
    }
    for (const FileReloc& e : rel) {
        MUGD_REQUIRE(e.op < ops.size() && e.region < fr.size() && e.field + sizeof(uintptr_t) <= sizeof(mugd_op), "plan_load: corrupt relocation");
        const int r = map[e.region];
        MUGD_REQUIRE(r >= 0, "plan_load: region '%s' of %s was not provided", fr[e.region].name, path);
        MUGD_REQUIRE(regions[r].bytes >= fr[e.region].bytes, "plan_load: region '%s' is %lld bytes, the plan needs %lld", fr[e.region].name,
                     (long long)regions[r].bytes, (long long)fr[e.region].bytes);
        uintptr_t& v = ptr_at(ops[e.op], e.field);
        MUGD_REQUIRE((int64_t)v < fr[e.region].bytes, "plan_load: offset outside region '%s'", fr[e.region].name);
        v += reinterpret_cast<uintptr_t>(regions[r].base);
    }
    return plan_from_ops(h, ops.data(), (int32_t)ops.size(), out);
}

extern "C" int mugd_plan_regions(const char* path, mugd_region* out, char (*names)[48], int32_t max_regions, int32_t* n_regions) {
    MUGD_REQUIRE(path && n_regions, "plan_regions: bad arguments");
    FILE* fp = fopen(path, "rb");
    MUGD_REQUIRE(fp, "plan_regions: cannot open %s", path);
    FileHeader fh;
    bool ok = fread(&fh, sizeof(fh), 1, fp) == 1 && memcmp(fh.magic, "MUGDPLN1", 8) == 0;
    if (ok) {
        *n_regions = (int32_t)fh.n_regions;
        for (uint32_t i = 0; i < fh.n_regions && ok; ++i) {
            FileRegion fr;
            ok = fread(&fr, sizeof(fr), 1, fp) == 1;
            if (ok && out && names && (int32_t)i < max_regions) {
                memcpy(names[i], fr.name, 48);
                out[i].name = names[i];
                out[i].base = nullptr;
                out[i].bytes = fr.bytes;
            }
        }
    }
    fclose(fp);
    MUGD_REQUIRE(ok, "plan_regions: %s is not a libmugd plan file", path);
    return MUGD_OK;
}

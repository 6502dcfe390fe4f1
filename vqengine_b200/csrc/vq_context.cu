// vq_context.cu — context lifetime, error plumbing, packed-layout helpers and the host-side
// FidelityFX constant setup (== the A_CPU functions the engine calls, PostProcess.cpp:39-99).
#include "vq_common.cuh"
#include <stdlib.h>
#include <stdarg.h>
#include <string.h>
#include <math.h>
#include <new>

std::atomic<uint64_t> g_vq_launches{0};
static thread_local char t_err[512] = "";

void vq_set_error(const char* fmt, ...) {
    va_list ap; va_start(ap, fmt);
    vsnprintf(t_err, sizeof(t_err), fmt, ap);
    va_end(ap);
}

int vq_enter(VqContext* ctx) {
    if (!ctx) { vq_set_error("null context"); return VQ_ERR_INVALID_ARG; }
    VQ_CUDA_OK(cudaSetDevice(ctx->device));
    return VQ_OK;
}
int vq_check_launch(const char* what) {
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { vq_set_error("%s launch failed: %s", what, cudaGetErrorString(e)); return VQ_ERR_CUDA; }
    vq_count_launch();
    return VQ_OK;
}

int vq_fill_peer_sync(const VqPeerSignal* sig, PeerSync* out) {
    memset(out, 0, sizeof(*out));
    if (!sig || sig->n_ranks <= 1) return VQ_OK;
    VQ_REQUIRE(sig->n_ranks <= 8 && sig->my_index >= 0 && sig->my_index < sig->n_ranks, "bad peer signal descriptor");
    for (int k = 0; k < sig->n_ranks; ++k) { VQ_REQUIRE(sig->flags[k], "null flag array in the peer signal"); out->flags[k] = sig->flags[k]; }
    out->n = sig->n_ranks; out->myIndex = sig->my_index; out->epoch = sig->epoch;
    return VQ_OK;
}

extern "C" {

const char* vq_last_error(void) { return t_err; }
const char* vq_version(void) { return "vqcuda 0.1 (sm_100a)"; }
uint64_t vq_launch_count(void) { return g_vq_launches.load(); }

int vq_ctx_create(int device, VqContext** out_ctx) {
    if (!out_ctx) { vq_set_error("out_ctx is null"); return VQ_ERR_INVALID_ARG; }
    *out_ctx = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) {
        // no CPU fallback by design: fail loudly
        vq_set_error("no CUDA device available (%s): this backend has no CPU path", e == cudaSuccess ? "count=0" : cudaGetErrorString(e));
        return VQ_ERR_NO_DEVICE;
    }
    if (device < 0 || device >= n) { vq_set_error("device %d out of range [0,%d)", device, n); return VQ_ERR_INVALID_ARG; }
    VQ_CUDA_OK(cudaSetDevice(device));
    cudaDeviceProp prop;
    VQ_CUDA_OK(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10) {
        vq_set_error("device %d is sm_%d%d; this library only carries sm_100a code", device, prop.major, prop.minor);
        return VQ_ERR_UNSUPPORTED;
    }
    VqContext* c = new (std::nothrow) VqContext();
    if (!c) return VQ_ERR_OUT_OF_MEMORY;
    memset(c, 0, sizeof(*c));
    c->device = device;
    c->sm_count = prop.multiProcessorCount;
    c->l2_bytes = prop.l2CacheSize;
    if (cudaMalloc(&c->spd_counter, 2 * VQ_SPD_SLOTS * sizeof(uint32_t)) != cudaSuccess) { delete c; vq_set_error("cudaMalloc failed"); return VQ_ERR_OUT_OF_MEMORY; }
    cudaMemset(c->spd_counter, 0, 2 * VQ_SPD_SLOTS * sizeof(uint32_t));
    c->spd_next = new std::atomic<uint32_t>(0u);
    c->mu = new std::recursive_mutex();
    *out_ctx = c;
    return VQ_OK;
}

int vq_ctx_destroy(VqContext* ctx) {
    if (!ctx) return VQ_OK;
    cudaSetDevice(ctx->device);
    if (ctx->streams_ready) {
        for (auto& s : ctx->streams) cudaStreamDestroy(s);
        for (auto& e : ctx->events) cudaEventDestroy(e);
    }
    if (ctx->stage_dev) cudaFree(ctx->stage_dev);
    for (void* p : {ctx->env_all, ctx->tmp_diff, ctx->tmp_spec, ctx->tmp_lut, ctx->resize_mid, ctx->resize_tab, ctx->depth_pad, ctx->shadow_rec}) if (p) cudaFree(p);
    if (ctx->spd_counter) cudaFree(ctx->spd_counter);
    delete ctx->spd_next; delete ctx->mu;
    delete ctx;
    return VQ_OK;
}

static int ctx_resize_locked(VqContext* ctx, int width, int height);
int vq_ctx_resize(VqContext* ctx, int width, int height) {
    int rc = vq_enter(ctx); if (rc) return rc;
    VqScratchLock lock(ctx);
    return ctx_resize_locked(ctx, width, height);
}
int vq_ctx_resize_locked(VqContext* ctx, int width, int height) { return ctx_resize_locked(ctx, width, height); }
static int ctx_resize_locked(VqContext* ctx, int width, int height) {
    VQ_REQUIRE(width > 0 && height > 0, "resolution must be positive");
    const size_t need = (size_t)width * height * 16 * 4;   // 3 G-buffer planes + output
    if (ctx->stage_dev_bytes < need) {
        if (ctx->stage_dev) cudaFree(ctx->stage_dev);
        ctx->stage_dev = nullptr; ctx->stage_dev_bytes = 0;
        if (cudaMalloc(&ctx->stage_dev, need) != cudaSuccess) { cudaGetLastError(); vq_set_error("staging cudaMalloc(%zu) failed", need); return VQ_ERR_OUT_OF_MEMORY; }
        ctx->stage_dev_bytes = need;
    }
    if (!ctx->streams_ready) {
        for (auto& s : ctx->streams) VQ_CUDA_OK(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
        for (auto& e : ctx->events) VQ_CUDA_OK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        ctx->streams_ready = 1;
    }
    return VQ_OK;
}

// ---- packed layouts ---------------------------------------------------------------------------
int vq_mip_level_count(uint64_t w, uint64_t h) {   // Image::CalculateMipLevelCount, Image.cpp:231-241
    int mips = 0;
    while (w >= 1 && h >= 1) { ++mips; w >>= 1; h >>= 1; }
    return mips;
}
uint64_t vq_cubemap_texel_count(int res, int mips) {
    uint64_t o = 0;
    for (int m = 0; m < mips; ++m) { const uint64_t r = (uint64_t)(res >> m); o += 6 * r * r; }
    return o;
}
uint64_t vq_cubemap_offset(int res, int mip, int face) {
    const uint64_t r = (uint64_t)(res >> mip);
    return vq_cubemap_texel_count(res, mip) + (uint64_t)face * r * r;
}
int vq_cubemap_row_count(int res, int mips) {
    int n = 0;
    for (int m = 0; m < mips; ++m) n += 6 * (res >> m);
    return n;
}
uint64_t vq_pyramid_texel_count(int width, int height, int levels) {
    uint64_t o = 0;
    for (int l = 0; l < levels; ++l) o += (uint64_t)(width >> l) * (uint64_t)(height >> l);
    return o;
}
uint64_t vq_pyramid_offset(int width, int height, int level) { return vq_pyramid_texel_count(width, height, level); }

// ---- FidelityFX constant setup (host) ------------------------------------------------------------
static inline uint32_t fbits(float f) { uint32_t u; memcpy(&u, &f, 4); return u; }

// float -> half bits, truncating, denormal-aware, +-INF/NaN -> +-65504 (the rule behind the
// reference's AU1_AH1_AF1 tables, FSR1.0/ffx_a.h:482-550)
static uint32_t half_bits_trunc(float f) {
    const uint32_t u = fbits(f);
    const uint32_t se = u >> 23, e = se & 0xffu, sign = (se >> 8) << 15;
    uint32_t base, shift;
    if (e < 103u)       { base = 0u;                    shift = 24u; }
    else if (e < 113u)  { base = 0x0400u >> (113u - e); shift = 126u - e; }
    else if (e <= 142u) { base = (e - 112u) << 10;      shift = 13u; }
    else                { base = 0x7bffu;               shift = 24u; }
    return (base | sign) + ((u & 0x7fffffu) >> shift);
}

void vq_fsr_easu_con(uint32_t con[16], float vpw, float vph, float inw, float inh, float outw, float outh) {
    // FsrEasuCon, ffx_fsr1.h:156-202 (ARcpF1(a) = 1.0f/a on the CPU, ffx_a.h:326)
    const float rx = 1.0f / outw, ry = 1.0f / outh, rix = 1.0f / inw, riy = 1.0f / inh;
    con[0] = fbits(vpw * rx);
    con[1] = fbits(vph * ry);
    con[2] = fbits(0.5f * vpw * rx - 0.5f);
    con[3] = fbits(0.5f * vph * ry - 0.5f);
    con[4] = fbits(rix);
    con[5] = fbits(riy);
    con[6] = fbits(1.0f * rix);
    con[7] = fbits(-1.0f * riy);
    con[8] = fbits(-1.0f * rix);
    con[9] = fbits(2.0f * riy);
    con[10] = fbits(1.0f * rix);
    con[11] = fbits(2.0f * riy);
    con[12] = fbits(0.0f * rix);
    con[13] = fbits(4.0f * riy);
    con[14] = con[15] = 0;
}

void vq_fsr_rcas_con(uint32_t con[4], float sharpness_stops) {
    // FsrRcasCon, ffx_fsr1.h:662-672
    const float s = exp2f(-sharpness_stops);
    con[0] = fbits(s);
    con[1] = half_bits_trunc(s) + (half_bits_trunc(s) << 16);
    con[2] = 0; con[3] = 0;
}

void vq_cas_setup(uint32_t con[8], float sharpness, float inw, float inh, float outw, float outh) {
    // CasSetup, ffx_cas.h:375-394; ALerpF1(a,b,c) = b*c + (-a*c + a), ffx_a.h:298
    const float rx = 1.0f / outw, ry = 1.0f / outh;
    con[0] = fbits(inw * rx);
    con[1] = fbits(inh * ry);
    con[2] = fbits(0.5f * inw * rx - 0.5f);
    con[3] = fbits(0.5f * inh * ry - 0.5f);
    const float c = fminf(1.0f, fmaxf(0.0f, sharpness));
    const float l = 5.0f * c + (-8.0f * c + 8.0f);
    const float sharp = -(1.0f / l);
    con[4] = fbits(sharp);
    con[5] = half_bits_trunc(sharp) + (half_bits_trunc(0.0f) << 16);
    con[6] = fbits(8.0f * inw * rx);
    con[7] = 0;
}

void vq_spd_setup(uint32_t dispatch_xy[2], VqSpdConstants* constants, const uint32_t rect[4], int mips) {
    // SpdSetup, ffx_spd.h:327-351
    constants->workGroupOffset[0] = rect[0] / 64;
    constants->workGroupOffset[1] = rect[1] / 64;
    const uint32_t endX = (rect[0] + rect[2] - 1) / 64;
    const uint32_t endY = (rect[1] + rect[3] - 1) / 64;
    dispatch_xy[0] = endX + 1 - constants->workGroupOffset[0];
    dispatch_xy[1] = endY + 1 - constants->workGroupOffset[1];
    constants->numWorkGroups = dispatch_xy[0] * dispatch_xy[1];
    if (mips >= 0) constants->mips = (uint32_t)mips;
    else {
        const uint32_t res = rect[2] > rect[3] ? rect[2] : rect[3];
        constants->mips = (uint32_t)fminf(floorf(log2f((float)res)), 12.0f);
    }
}

}  // extern "C"

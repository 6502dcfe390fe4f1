// vq_shadow.cu — SURVEY §8(f).4: shadowed casters and the hierarchical MIN depth pyramid.
//
//   vq_forward_lighting_shadowed   PSMain with the shadow maps bound (ForwardLighting.hlsl:321-377): the caster lists and a
//                                  shadowing directional light multiplied by their PCF tests (Lighting.hlsl:79-272)
//   vq_depth_min_pyramid           DownsampleDepth.hlsl:50-119 (FidelityFX SPD with the MIN reduction over a D3D mip chain)
//
// Checked against the oracle (oracle/oracle_shadow.cpp, itself pinned bit for bit to the reference's shader text,
// tests/test_hlsl_ref.py) on a B200: tests/test_shadow_gpu.py (-m gpu), memcheck clean (profiles/r02_shadow_first_run.txt).
//
// Structure of the shadowed pass: the PCF tests are DISCRETE decisions (a texel index, a depth comparison), the light terms they
// multiply are continuous. So shadow_pcf_kernel runs only the tests, with every fp32 operation rounded as the oracle rounds it,
// and stores per pixel the number of shadowed taps of every caster (5 bits each in one 64-bit record: 8 B/pixel); the SHADOWED
// instantiation of K1 (vq_forward.cu) then shades the caster lights in its own packed light loop with weight * (1 - taps/N).
// (Round 2's first version re-evaluated the whole BRDF per caster with correctly rounded divisions in a second full-frame pass:
// 5100 instructions per pixel, 2.0 ms at 4K; profiles/r02_shadow_a_summary.txt.)
//
// The per-pixel math lives in vq_shadow_math.cuh, which also compiles for the HOST: tests/test_shadow_math_host.py checks it
// against the oracle bit for bit on the CPU.
#include "vq_common.cuh"
#include "vq_shadow_math.cuh"
#include <string.h>

namespace {

struct PcfParams {
    ImgV pos, nrm;
    uint2* rec; int recPitch;          // records of rows [rowBegin, rowBegin + rows), recPitch per row
    int rowBegin, rows, width;
    vqshadow::ShadowLights L;
};

__device__ __forceinline__ vqshadow::Px4 px4(float4 v) { vqshadow::Px4 r; r.x = v.x; r.y = v.y; r.z = v.z; r.w = v.w; return r; }

// One thread per pixel; rows strided over the grid. 32 B/pixel in (position, normal), 8 B/pixel out; the shadow maps are
// L2-resident side data. Bound by instruction issue: ~45 instructions per cube tap (face selection, two correctly rounded
// quotients, texel address, depth comparison), ~10 per 2-D tap.
constexpr int PCF_MIN_BLOCKS = 8;
__global__ void __launch_bounds__(128, PCF_MIN_BLOCKS) shadow_pcf_kernel(const __grid_constant__ PcfParams P) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    const int cx = min(x, P.width - 1);          // whole warps stay alive (pcf_record votes across the warp): a lane past the row's end
    for (int r = blockIdx.y; r < P.rows; r += gridDim.y) {   // re-computes the last pixel and stores nothing
        const int y = P.rowBegin + r;
        const float4 p4 = vq::ld_stream(P.pos.row(y) + cx), n4 = vq::ld_stream(P.nrm.row(y) + cx);
        const unsigned long long rec = vqshadow::pcf_record(P.L, px4(p4), px4(n4));
        if (x < P.width) P.rec[(size_t)r * P.recPitch + x] = make_uint2((uint32_t)rec, (uint32_t)(rec >> 32));
    }
}

// ---- MIN depth pyramid: SIX levels per launch (a 4K pyramid = 2 launches; it was a copy + 11 one-level launches) ----------
// Level l of the padded domain is ceil-halved (see the oracle) and a texel outside a level reads 0, so dst(x,y) = min of the
// zero-padded 2x2 block of the level above. A CTA owns a 64x64 tile of the source level S and reduces it to 1x1 (levels S+1 ..
// S+6): the hierarchy is tile-local because ceil-halving keeps 2^k-aligned blocks aligned, and a texel outside level k comes out
// as min(0,0,0,0) = 0 on its own once the loads outside S return 0. Each level is stored clipped to its D3D size
// max(1, w>>l) x max(1, h>>l); the LAST level of the launch is also kept in the padded domain (`pad`) for the next launch.
// HBM-bound: level 0 read once and copied once (8 B/texel) + 4/3 B/texel of levels.
struct DepthArgs {
    const float* src; int srcPitch, sw, sh;     // source level in the padded domain (sw x sh valid texels)
    float* copy;                                // != nullptr: also copy the source tightly packed (level 0 of the output)
    float* dst[6]; int lw[6], lh[6];            // stored levels S+1 .. S+n, clipped sizes
    int n;
    float* pad; int padW, padH;                 // padded-domain copy of level S+n (nullptr: not needed)
};

__global__ void __launch_bounds__(256) depth_min6_kernel(const __grid_constant__ DepthArgs A) {
    __shared__ float sm[2][16][16];
    const int t = threadIdx.x, px = t & 15, py = t >> 4;
    const int x0 = blockIdx.x * 64 + px * 4, y0 = blockIdx.y * 64 + py * 4;          // 4x4 source patch of this thread
    float v4[4][4];
    const bool vecIn = ((A.srcPitch & 3) == 0) && (((uintptr_t)A.src & 15) == 0) && x0 + 4 <= A.sw;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int y = y0 + k;
        if (y < A.sh && vecIn) {
            const float4 r = __ldg((const float4*)(A.src + (size_t)y * A.srcPitch + x0));
            v4[k][0] = r.x; v4[k][1] = r.y; v4[k][2] = r.z; v4[k][3] = r.w;
        } else {
#pragma unroll
            for (int i = 0; i < 4; ++i) v4[k][i] = (y < A.sh && x0 + i < A.sw) ? __ldg(A.src + (size_t)y * A.srcPitch + x0 + i) : 0.0f;
        }
    }
    if (A.copy) {
        const bool vecOut = ((A.sw & 3) == 0) && (((uintptr_t)A.copy & 15) == 0) && x0 + 4 <= A.sw;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int y = y0 + k;
            if (y >= A.sh) continue;
            float* d = A.copy + (size_t)y * A.sw + x0;
            if (vecOut) *(float4*)d = make_float4(v4[k][0], v4[k][1], v4[k][2], v4[k][3]);
            else {
#pragma unroll
                for (int i = 0; i < 4; ++i) if (x0 + i < A.sw) d[i] = v4[k][i];
            }
        }
    }
    auto keep_pad = [&](int lvl, int X, int Y, float m) {        // level index inside this launch (0-based)
        if (A.pad && lvl == A.n - 1 && X < A.padW && Y < A.padH) A.pad[(size_t)Y * A.padW + X] = m;
    };
    // level +1: 2x2 texels per thread (same association as depth_min_texel: min(min(a,b), min(c,d)))
    float l1[2][2];
#pragma unroll
    for (int j = 0; j < 2; ++j)
#pragma unroll
        for (int i = 0; i < 2; ++i) {
            const float m = fminf(fminf(v4[2 * j][2 * i], v4[2 * j][2 * i + 1]), fminf(v4[2 * j + 1][2 * i], v4[2 * j + 1][2 * i + 1]));
            l1[j][i] = m;
            const int X = (x0 >> 1) + i, Y = (y0 >> 1) + j;
            if (X < A.lw[0] && Y < A.lh[0]) A.dst[0][(size_t)Y * A.lw[0] + X] = m;
            keep_pad(0, X, Y, m);
        }
    if (A.n < 2) return;
    float v = fminf(fminf(l1[0][0], l1[0][1]), fminf(l1[1][0], l1[1][1]));             // level +2: one texel per thread
    {
        const int X = x0 >> 2, Y = y0 >> 2;
        if (X < A.lw[1] && Y < A.lh[1]) A.dst[1][(size_t)Y * A.lw[1] + X] = v;
        keep_pad(1, X, Y, v);
    }
    sm[0][py][px] = v;
    int side = 8, cur = 0;                                                            // levels +3 .. +6: 8x8 .. 1x1 texels of this tile
#pragma unroll
    for (int lvl = 2; lvl < 6; ++lvl, side >>= 1, cur ^= 1) {
        if (lvl >= A.n) return;                                                       // uniform across the block
        __syncthreads();
        if (t < side * side) {
            const int qx = t % side, qy = t / side;
            v = fminf(fminf(sm[cur][2 * qy][2 * qx], sm[cur][2 * qy][2 * qx + 1]), fminf(sm[cur][2 * qy + 1][2 * qx], sm[cur][2 * qy + 1][2 * qx + 1]));
            sm[cur ^ 1][qy][qx] = v;
            const int X = blockIdx.x * side + qx, Y = blockIdx.y * side + qy;
            if (X < A.lw[lvl] && Y < A.lh[lvl]) A.dst[lvl][(size_t)Y * A.lw[lvl] + X] = v;
            keep_pad(lvl, X, Y, v);
        }
    }
}

int ensure_scratch(void** ptr, size_t* have, size_t need) {
    if (*have >= need && *ptr) return VQ_OK;
    if (*ptr) cudaFree(*ptr);
    *ptr = nullptr; *have = 0;
    if (cudaMalloc(ptr, need) != cudaSuccess) { cudaGetLastError(); vq_set_error("cudaMalloc(%zu) failed", need); return VQ_ERR_OUT_OF_MEMORY; }
    *have = need;
    return VQ_OK;
}

}  // namespace

extern "C" int vq_forward_lighting_shadowed(VqContext* ctx, const VqPerFrameData* pf, const VqPerViewLightingData* pv,
                                            const VqGBuffer* gb, const VqEnvironmentMaps* env, const VqShadowMaps* sm,
                                            VqImage out, int row_begin, int row_end, void* stream) {
    int rc = vq_enter(ctx); if (rc) return rc;
    VQ_MARK("RenderSceneColor");
    VQ_REQUIRE(pf && pv && gb && env && sm, "null parameter block");
    const VqSceneLighting& L = pf->Lights;
    VQ_REQUIRE(L.numPointCasters >= 0 && L.numPointCasters <= VQ_NUM_SHADOWING_LIGHTS_POINT &&
               L.numSpotCasters >= 0 && L.numSpotCasters <= VQ_NUM_SHADOWING_LIGHTS_SPOT, "caster counts exceed the cbuffer arrays");
    // texel indices inside one map are 32-bit in the kernel
    if (sm->point_cubes) VQ_REQUIRE(sm->point_res > 0 && sm->point_res <= 16384, "point shadow cubes need a resolution in 1..16384");
    if (sm->spot_maps) VQ_REQUIRE(sm->spot_width > 0 && sm->spot_height > 0 && (uint64_t)sm->spot_width * sm->spot_height < (1ull << 31), "spot shadow maps need positive dimensions (< 2^31 texels)");
    if (sm->directional_map) VQ_REQUIRE(sm->directional_width > 0 && sm->directional_height > 0 && (uint64_t)sm->directional_width * sm->directional_height < (1ull << 31), "directional shadow map needs positive dimensions (< 2^31 texels)");
    const bool anyTest = (sm->point_cubes && L.numPointCasters > 0) || (sm->spot_maps && L.numSpotCasters > 0) ||
                         (sm->directional_map && L.directional.enabled && L.directional.shadowing);
    if (!anyTest || row_begin >= row_end)          // no test runs: every factor is 1, which is what the plain kernel computes
        return vq_forward_launch(ctx, pf, pv, gb, env, out, row_begin, row_end, (cudaStream_t)stream);
    VQ_REQUIRE(gb->position_ao.ptr && vq_image_ok(gb->position_ao) && vq_image_ok(gb->normal_roughness) &&
               gb->normal_roughness.width == gb->position_ao.width && gb->normal_roughness.height == gb->position_ao.height,
               "bad G-buffer planes");
    VQ_REQUIRE(row_begin >= 0 && row_end <= gb->position_ao.height, "row range out of bounds");

    PcfParams P;
    memset(&P, 0, sizeof(P));
    P.pos = make_view(gb->position_ao); P.nrm = make_view(gb->normal_roughness);
    P.rowBegin = row_begin; P.rows = row_end - row_begin; P.width = gb->position_ao.width;
    vqshadow::fill_shadow_lights(P.L, *pf, *pv, *sm);
    VqScratchLock lock(ctx);                       // the records are context scratch (vqcuda.h lists the call as not re-entrant per context)
    rc = ensure_scratch(&ctx->shadow_rec, &ctx->shadow_rec_bytes, (size_t)P.width * P.rows * sizeof(uint2)); if (rc) return rc;
    P.rec = (uint2*)ctx->shadow_rec; P.recPitch = P.width;

    const unsigned gx = (unsigned)((P.width + 127) / 128);
    unsigned gy = (unsigned)(ctx->sm_count * PCF_MIN_BLOCKS) / gx;
    if (gy < 1) gy = 1;
    if (gy > (unsigned)P.rows) gy = (unsigned)P.rows;
    if (gy > 65535u) gy = 65535u;
    shadow_pcf_kernel<<<dim3(gx, gy), 128, 0, (cudaStream_t)stream>>>(P);
    rc = vq_check_launch("shadow_pcf"); if (rc) return rc;

    vq::ShadowRecV V;
    V.p = P.rec; V.pitch = P.recPitch;
    V.nPointCasters = L.numPointCasters; V.nSpotCasters = L.numSpotCasters;
    V.dirSlot = (sm->directional_map && L.directional.enabled && L.directional.shadowing) ? L.numPointCasters + L.numSpotCasters : -1;
    return vq_forward_launch(ctx, pf, pv, gb, env, out, row_begin, row_end, (cudaStream_t)stream, &V);
}

extern "C" int vq_depth_pyramid_level_count(int width, int height) { return vqshadow::depth_level_count(width, height); }
extern "C" uint64_t vq_depth_pyramid_texel_count(int width, int height, int levels) {
    uint64_t t = 0;
    for (int l = 0; l < levels; ++l) t += (uint64_t)((width >> l) > 0 ? (width >> l) : 1) * (uint64_t)((height >> l) > 0 ? (height >> l) : 1);
    return t;
}

extern "C" int vq_depth_min_pyramid(VqContext* ctx, VqImage depth, void* levels, int n_levels, void* stream_) {
    int rc = vq_enter(ctx); if (rc) return rc;
    VQ_MARK("DownsampleDepth");
    cudaStream_t stream = (cudaStream_t)stream_;
    VQ_REQUIRE(vq_image_ok(depth, 4), "bad depth image descriptor (R32F)");
    VQ_REQUIRE(levels && ((uintptr_t)levels % 4) == 0, "levels buffer is null or misaligned");
    const int W = depth.width, H = depth.height;
    VQ_REQUIRE(n_levels >= 1 && n_levels <= vq_depth_pyramid_level_count(W, H), "level count out of range");
    vqshadow::DepthLevelPlan plan[13];
    vqshadow::depth_pyramid_plan(W, H, n_levels, plan);
    // padded-domain copies of levels 6 and 12 (what a following launch reads): level 6 is at most ceil(W/64) x ceil(H/64)
    const size_t padTexels = (size_t)((W + 63) / 64) * ((H + 63) / 64);
    VqScratchLock lock(ctx);
    rc = ensure_scratch(&ctx->depth_pad, &ctx->depth_pad_bytes, padTexels * 2 * 4 > 16 ? padTexels * 2 * 4 : 16); if (rc) return rc;
    float* pads[2] = {(float*)ctx->depth_pad, (float*)ctx->depth_pad + padTexels};
    float* out = (float*)levels;
    DepthArgs A;
    A.src = (const float*)depth.ptr; A.srcPitch = (int)(depth.pitch_bytes / 4); A.sw = W; A.sh = H;
    A.copy = out;
    int launch = 0;
    for (int l0 = 0; l0 == 0 || l0 + 1 < n_levels; l0 += 6, ++launch) {   // source level l0 -> levels l0+1 .. l0+6 (level 0 alone: the copy)
        A.n = n_levels - 1 - l0 < 6 ? n_levels - 1 - l0 : 6;
        for (int j = 0; j < 6; ++j) {
            const bool on = j < A.n;
            A.dst[j] = on ? out + plan[l0 + 1 + j].out_offset : nullptr;
            A.lw[j] = on ? plan[l0 + 1 + j].lw : 0; A.lh[j] = on ? plan[l0 + 1 + j].lh : 0;
        }
        const bool more = l0 + 6 + 1 < n_levels;                         // another launch reads level l0+6 in the padded domain
        A.pad = more ? pads[launch & 1] : nullptr;
        A.padW = more ? plan[l0 + 6].pw : 0; A.padH = more ? plan[l0 + 6].ph : 0;
        depth_min6_kernel<<<dim3((A.sw + 63) / 64, (A.sh + 63) / 64), 256, 0, stream>>>(A);
        rc = vq_check_launch("depth_min6"); if (rc) return rc;
        if (!more) break;
        A.src = A.pad; A.srcPitch = A.padW; A.sw = A.padW; A.sh = A.padH; A.copy = nullptr;
    }
    return VQ_OK;
}

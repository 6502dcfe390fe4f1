// vq_surface.cu — SURVEY.md §8(f).1: the part of PSMain BEFORE lighting (ForwardLighting.hlsl:226-283) as a kernel that
// fills the G-buffer K1 consumes, plus the RGBA8 box mip chain the engine builds on the CPU for material textures
// (DXGIUtils.cpp:250-287).
//
// Bound: HBM. Algorithmic bytes per pixel = 3 float4 attribute planes in + 3 (4 with emissive) float4 G-buffer planes out
// = 96 (112) B/px (+4 with the SSAO plane); material textures are L2-resident side data (like K1's cubemaps).
//
// Sampling semantics (identical in oracle/oracle_surface.cpp, DESIGN.md §3.6): implicit derivatives = fine finite
// differences inside the pixel's aligned 2x2 quad, exchanged with warp shuffles (a warp shades a 16x2 pixel strip, so
// lane^1 is the horizontal and lane^16 the vertical quad partner); isotropic trilinear, WRAP; texel = byte/255.
#include "vq_common.cuh"
#include <stdlib.h>

using namespace vq;

namespace {

// device copy of one texture descriptor: 16 B = one LDG.128. Level offsets are recomputed in registers (a short loop over
// the levels below the sampled one) instead of being looked up: a table would add a dependent memory round trip per map.
struct DevTex {
    const uint32_t* p;       // RGBA8 texels, packed levels; nullptr = null SRV
    int32_t w;
    uint32_t h_levels;       // height in bits 0..26, level count in bits 27..31
};
static_assert(sizeof(DevTex) == 16, "DevTex layout");

// One 16-byte RECORD per texel of a material whose maps all have the same size (how shipped material sets look): the bytes
// PSMain reads of every map, interleaved, so that one LDG.128 per trilinear tap fetches the texel of ALL maps:
//   x = diffuse RGBA | y = normal RGB, local-AO R | z = emissive RGB, roughness R | w = metalness R, ORM G, ORM B, 0
// (a null map contributes zeros, which is what a null SRV reads). Built once per table by record_build_kernel from the maps'
// own mip chains, level by level (same packed-level offsets); the K1 sampling copies of the cubemaps are the same idea.
struct DevMaterial {         // 80 + 7*16 + 16 = 208 B
    VqMaterialData c;
    DevTex t[7];
    DevTex rec;              // p = uint4 records (nullptr: this material samples its maps one by one), w, h_levels
};
static_assert(sizeof(DevMaterial) == 208, "DevMaterial layout");

}  // namespace

struct VqMaterialTable {
    DevMaterial* dev;
    int count;
    void* records;           // one allocation holding every material's texel records (nullptr: none)
    size_t record_bytes;
};

namespace {

// ---------------------------------------------------------------------------------------------
// RGBA8 2x2 box, per channel (a+b+c+d)/4 truncating.  One thread = 4 destination texels (16 B store, two 32 B loads).
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t box4(uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
    // per-byte sums need 10 bits: split even/odd bytes into 16-bit lanes
    const uint32_t lo = (a & 0x00ff00ffu) + (b & 0x00ff00ffu) + (c & 0x00ff00ffu) + (d & 0x00ff00ffu);
    const uint32_t hi = ((a >> 8) & 0x00ff00ffu) + ((b >> 8) & 0x00ff00ffu) + ((c >> 8) & 0x00ff00ffu) + ((d >> 8) & 0x00ff00ffu);
    return ((lo >> 2) & 0x00ff00ffu) | (((hi >> 2) & 0x00ff00ffu) << 8);
}

// Six levels per launch: a block reduces one 64x64 tile of the source level all the way to 1x1 (levels +1 .. +6), so a
// 4096^2 chain is 2 launches instead of 12 and every level is read at most once from HBM. Floor-halved level sizes keep
// the hierarchy tile-local: a valid texel of level k only depends on valid texels of level k-1 (2X+1 < 2*(w>>k) <= w>>(k-1)).
struct MipArgs {
    const uint32_t* src; int sw, sh;       // source level
    uint32_t* dst[6]; int n;               // destination levels (n <= 6), level j is (sw >> (j+1)) x (sh >> (j+1))
};

__global__ void __launch_bounds__(256) tex_mip6_kernel(const __grid_constant__ MipArgs A) {
    __shared__ uint32_t sm[2][16][16];
    const int t = threadIdx.x, px = t & 15, py = t >> 4;
    const int x0 = blockIdx.x * 64 + px * 4, y0 = blockIdx.y * 64 + py * 4;          // 4x4 source patch of this thread
    const int w1 = A.sw >> 1, h1 = A.sh >> 1;
    uint32_t l1[2][2] = {{0u, 0u}, {0u, 0u}};
    const bool vec = ((A.sw & 3) == 0) && (((uintptr_t)A.src & 15) == 0) && x0 + 4 <= A.sw && y0 + 4 <= A.sh;
    if (vec) {
        uint4 r[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) r[k] = __ldg((const uint4*)(A.src + (size_t)(y0 + k) * A.sw + x0));
        l1[0][0] = box4(r[0].x, r[0].y, r[1].x, r[1].y); l1[0][1] = box4(r[0].z, r[0].w, r[1].z, r[1].w);
        l1[1][0] = box4(r[2].x, r[2].y, r[3].x, r[3].y); l1[1][1] = box4(r[2].z, r[2].w, r[3].z, r[3].w);
    } else {
#pragma unroll
        for (int j = 0; j < 2; ++j)
#pragma unroll
            for (int i = 0; i < 2; ++i) {
                const int X = (x0 >> 1) + i, Y = (y0 >> 1) + j;
                if (X < w1 && Y < h1) {
                    const uint32_t* q = A.src + (size_t)(2 * Y) * A.sw + 2 * X;
                    l1[j][i] = box4(__ldg(q), __ldg(q + 1), __ldg(q + A.sw), __ldg(q + A.sw + 1));
                }
            }
    }
    {   // level +1: 2x2 texels per thread
        const int X = x0 >> 1, Y = y0 >> 1;
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            if (Y + j >= h1) continue;
            uint32_t* d = A.dst[0] + (size_t)(Y + j) * w1 + X;
            if (X + 1 < w1 && (((uintptr_t)d) & 7) == 0) *(uint2*)d = make_uint2(l1[j][0], l1[j][1]);
            else { if (X < w1) d[0] = l1[j][0]; if (X + 1 < w1) d[1] = l1[j][1]; }
        }
    }
    if (A.n < 2) return;
    uint32_t v = box4(l1[0][0], l1[0][1], l1[1][0], l1[1][1]);                       // level +2: one texel per thread
    {
        const int w2 = A.sw >> 2, h2 = A.sh >> 2, X = x0 >> 2, Y = y0 >> 2;
        if (X < w2 && Y < h2) A.dst[1][(size_t)Y * w2 + X] = v;
    }
    sm[0][py][px] = v;
    // levels +3 .. +6: 8x8, 4x4, 2x2, 1x1 texels of this tile, ping-pong through shared memory
    int side = 8, cur = 0;
#pragma unroll
    for (int lvl = 2; lvl < 6; ++lvl, side >>= 1, cur ^= 1) {
        if (lvl >= A.n) return;                                                      // uniform across the block
        __syncthreads();
        if (t < side * side) {
            const int qx = t % side, qy = t / side;
            v = box4(sm[cur][2 * qy][2 * qx], sm[cur][2 * qy][2 * qx + 1], sm[cur][2 * qy + 1][2 * qx], sm[cur][2 * qy + 1][2 * qx + 1]);
            sm[cur ^ 1][qy][qx] = v;
            const int wl = A.sw >> (lvl + 1), hl = A.sh >> (lvl + 1);
            const int X = blockIdx.x * side + qx, Y = blockIdx.y * side + qy;
            if (X < wl && Y < hl) A.dst[lvl][(size_t)Y * wl + X] = v;
        }
    }
}

// ---------------------------------------------------------------------------------------------
// texture sampling
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ int wrap_index(int i, int n) {           // general modulo (uv is unbounded: tiling)
    int r = i % n;
    return r < 0 ? r + n : r;
}

constexpr int SURF_MIN_BLOCKS = 4;
struct TexR { const uint32_t* p; int w, h, levels; };               // a descriptor in registers
__device__ __forceinline__ TexR load_tex(const DevTex* d) {
    const uint4 v = __ldg((const uint4*)d);
    TexR t;
    t.p = (const uint32_t*)(((uint64_t)v.y << 32) | v.x);
    t.w = (int)v.z; t.h = (int)(v.w & 0x07ffffffu); t.levels = (int)(v.w >> 27);
    return t;
}

// Sampler state of one Sample()/SampleBias() call: everything that depends only on (uv, derivatives, texture dimensions,
// bias) — the two mip levels, the trilinear fraction, the four tap offsets (level offset included) and the bilinear
// weights per level. A material's maps are usually all the same size, so consecutive textures reuse it (only the texel
// pointer differs) and the ~70 instructions of address math are paid once per pixel, not once per map.
struct Taps {
    int32_t w, h, levels; float bias;      // key
    uint32_t i[2][4];                      // [level slot][t00, t10, t01, t11]
    float fx[2], fy[2];
    float f;                               // trilinear fraction (0 -> slot 1 repeats slot 0)
};

__device__ __forceinline__ void level_taps(int W, int H, uint32_t o, float u, float v, uint32_t (&idx)[4], float& fx, float& fy) {
    // two roundings, as the oracle writes it: the weights multiply full-contrast byte data, so the coordinate must match
    const float x = __fsub_rn(__fmul_rn(u, (float)W), 0.5f), y = __fsub_rn(__fmul_rn(v, (float)H), 0.5f);
    const float x0 = floorf(x), y0 = floorf(y);
    fx = __fsub_rn(x, x0); fy = __fsub_rn(y, y0);
    const bool pow2 = ((W & (W - 1)) | (H & (H - 1))) == 0;
    int ix0, iy0;
    if (pow2) { ix0 = (int)x0 & (W - 1); iy0 = (int)y0 & (H - 1); }
    else      { ix0 = wrap_index((int)x0, W); iy0 = wrap_index((int)y0, H); }
    const int ix1 = ix0 + 1 == W ? 0 : ix0 + 1, iy1 = iy0 + 1 == H ? 0 : iy0 + 1;
    const uint32_t r0 = o + (uint32_t)(iy0 * W), r1 = o + (uint32_t)(iy1 * W);
    idx[0] = r0 + ix0; idx[1] = r0 + ix1; idx[2] = r1 + ix0; idx[3] = r1 + ix1;
}

__device__ __forceinline__ void make_taps(Taps& T, const TexR& t, float u, float v, float dudx, float dvdx, float dudy,
                                          float dvdy, float bias) {
    if (t.w == T.w && t.h == T.h && t.levels == T.levels && bias == T.bias) return;      // same sampler state as the previous map
    T.w = t.w; T.h = t.h; T.levels = t.levels; T.bias = bias;
    const float W = (float)t.w, H = (float)t.h;
    const float ax = dudx * W, ay = dvdx * H, bx = dudy * W, by = dvdy * H;
    const float m = fmaxf(fmaf(ax, ax, ay * ay), fmaf(bx, bx, by * by));
    float lod = (m > 0.0f ? 0.5f * __log2f(m) : -126.0f) + bias;
    lod = fminf(fmaxf(lod, 0.0f), (float)(t.levels - 1));
    const float l0f = floorf(lod);
    const int l0 = (int)l0f;
    T.f = (l0 + 1 < t.levels) ? lod - l0f : 0.0f;
    uint32_t o = 0;                                                   // texel offset of level l0 (vq_pyramid_offset)
    if (t.w == t.h && (t.w & (t.w - 1)) == 0 && t.w <= 16384) {       // square power of two: sum_{l<l0} (w>>l)^2 = 4 (w^2 - (w>>l0)^2) / 3
        const uint32_t wl = (uint32_t)t.w >> l0;
        o = (4u * ((uint32_t)t.w * (uint32_t)t.w - wl * wl)) / 3u;
    } else {
        for (int l = 0; l < l0; ++l) o += (uint32_t)((t.w >> l) * (t.h >> l));
    }
    const int W0 = t.w >> l0, H0 = t.h >> l0;
    level_taps(W0, H0, o, u, v, T.i[0], T.fx[0], T.fy[0]);
    // the second level is fetched unconditionally so that all 8 taps of a Sample() are independent loads in flight at once;
    // when the fraction is 0 it re-reads the first level's taps (L1 hits) and the lerp returns them unchanged
    if (T.f != 0.0f) level_taps(W0 >> 1, H0 >> 1, o + (uint32_t)(W0 * H0), u, v, T.i[1], T.fx[1], T.fy[1]);
    else {
#pragma unroll
        for (int k = 0; k < 4; ++k) T.i[1][k] = T.i[0][k];
        T.fx[1] = T.fx[0]; T.fy[1] = T.fy[0];
    }
}

// byte c of a packed RGBA8 texel as a float in [0,255]: PRMT drops the byte into the mantissa of 2^23 (ALU pipe) and one
// FADD removes the bias — instead of shift/mask + I2F, which issues on the quarter-rate XU pipe (39 % busy before).
template <int C>
__device__ __forceinline__ float byte_to_float(uint32_t texel) {
    return __uint_as_float(__byte_perm(texel, 0x4B000000u, 0x7650 + C)) - 8388608.0f;
}

template <int NCH>
__device__ __forceinline__ void bilinear_lerp(uint32_t t00, uint32_t t10, uint32_t t01, uint32_t t11, float fx, float fy,
                                              float (&out)[NCH]) {
#define VQ_CH(C)                                                                                   \
    if (C < NCH) {                                                                                 \
        const float a = byte_to_float<C>(t00), b = byte_to_float<C>(t10);                          \
        const float d = byte_to_float<C>(t01), e = byte_to_float<C>(t11);                          \
        const float top = fmaf(fx, b - a, a), bot = fmaf(fx, e - d, d);                            \
        out[C < NCH ? C : 0] = fmaf(fy, bot - top, top);                                           \
    }
    VQ_CH(0) VQ_CH(1) VQ_CH(2) VQ_CH(3)
#undef VQ_CH
}

// L2 residency hints (no instruction cost: the policy rides in the LDG/STG descriptor). Material texels are re-read by
// many blocks and should survive in L2; the interpolant planes and the G-buffer are touched exactly once and must not
// push them out (before: 40 % of the texel sectors that missed L1 also missed L2 with a 58 MB texture set).
__device__ __forceinline__ uint64_t l2_policy_evict_last() {
    uint64_t p; asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p)); return p;
}
__device__ __forceinline__ uint64_t l2_policy_evict_first() {
    uint64_t p; asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p)); return p;
}
__device__ __forceinline__ uint32_t ld_texel(const uint32_t* p, uint64_t pol) {
    uint32_t r; asm volatile("ld.global.nc.L2::cache_hint.b32 %0, [%1], %2;" : "=r"(r) : "l"(p), "l"(pol)); return r;
}
__device__ __forceinline__ float4 ld_once(const float4* p, uint64_t pol) {
    float4 v;
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v4.f32 {%0,%1,%2,%3}, [%4], %5;"
                 : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p), "l"(pol));
    return v;
}
__device__ __forceinline__ void st_once(float4* p, float4 v, uint64_t pol) {
    asm volatile("st.global.L1::no_allocate.L2::cache_hint.v4.f32 [%0], {%1,%2,%3,%4}, %5;"
                 :: "l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w), "l"(pol) : "memory");
}

// ---- record path: every map of the material in one 16-byte texel record ---------------------------------------------------
// byte C of a texel word as the float 2^23 + byte (PRMT only); differences of two such values are the exact byte differences,
// so only the lerp's base operand needs the bias removed — and the arithmetic runs on channel PAIRS (FADD2 / FFMA2).
template <int C>
__device__ __forceinline__ float byte_biased(uint32_t texel) { return __uint_as_float(__byte_perm(texel, 0x4B000000u, 0x7650 + C)); }

// bilinear blend of channels (C0, C1) of four texel words, in [0,255]; the same operations, in the same order, as bilinear_lerp
template <int C0, int C1>
__device__ __forceinline__ f2 bilinear2(uint32_t t00, uint32_t t10, uint32_t t01, uint32_t t11, f2 fx, f2 fy) {
    const f2 unbias = bc(-8388608.0f);
    const f2 a = mk(byte_biased<C0>(t00), byte_biased<C1>(t00)), b = mk(byte_biased<C0>(t10), byte_biased<C1>(t10));
    const f2 d = mk(byte_biased<C0>(t01), byte_biased<C1>(t01)), e = mk(byte_biased<C0>(t11), byte_biased<C1>(t11));
    const f2 top = fma2(fx, b - a, a + unbias), bot = fma2(fx, e - d, d + unbias);
    return fma2(fy, bot - top, top);
}
// trilinear sample of the four channels of one record word -> [0,1]; w0[] = the word at the four taps of the lower level,
// w1[] = of the upper one (read only when the fraction is not 0: f == 0 returns the lower level's blend unchanged, as sample8 does)
__device__ __forceinline__ void sample_word(const uint32_t (&w0)[4], const uint32_t (&w1)[4], const Taps& T, bool two, float (&out)[4]) {
    f2 lo01 = bilinear2<0, 1>(w0[0], w0[1], w0[2], w0[3], bc(T.fx[0]), bc(T.fy[0]));
    f2 lo23 = bilinear2<2, 3>(w0[0], w0[1], w0[2], w0[3], bc(T.fx[0]), bc(T.fy[0]));
    if (two) {
        const f2 hi01 = bilinear2<0, 1>(w1[0], w1[1], w1[2], w1[3], bc(T.fx[1]), bc(T.fy[1]));
        const f2 hi23 = bilinear2<2, 3>(w1[0], w1[1], w1[2], w1[3], bc(T.fx[1]), bc(T.fy[1]));
        lo01 = fma2(bc(T.f), hi01 - lo01, lo01);
        lo23 = fma2(bc(T.f), hi23 - lo23, lo23);
    }
    lo01 = lo01 * bc(1.0f / 255.0f); lo23 = lo23 * bc(1.0f / 255.0f);
    out[0] = lo01.v.x; out[1] = lo01.v.y; out[2] = lo23.v.x; out[3] = lo23.v.y;
}
__device__ __forceinline__ uint4 ld_record(const uint4* p, uint64_t pol) {
    uint4 r;
    asm volatile("ld.global.nc.L2::cache_hint.v4.u32 {%0,%1,%2,%3}, [%4], %5;" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p), "l"(pol));
    return r;
}

// Texture2D.Sample / SampleBias of ONE RGBA8 map: isotropic trilinear, WRAP; channels in [0,1]. Two or more channels are
// filtered as packed pairs (bilinear2); the operations per channel are those of bilinear_lerp either way.
template <int NCH>
__device__ __forceinline__ void sample8(Taps& T, const TexR& t, float u, float v, float dudx, float dvdx, float dudy,
                                        float dvdy, float bias, float (&out)[NCH]) {
    make_taps(T, t, u, v, dudx, dvdx, dudy, dvdy, bias);
    const uint32_t* p = t.p;
    const uint64_t keep = l2_policy_evict_last();
    uint32_t q[8];
#pragma unroll
    for (int k = 0; k < 4; ++k) { q[k] = ld_texel(p + T.i[0][k], keep); q[4 + k] = ld_texel(p + T.i[1][k], keep); }
    if (NCH == 1) {
        float lo[1], hi[1];
        bilinear_lerp<1>(q[0], q[1], q[2], q[3], T.fx[0], T.fy[0], lo);
        bilinear_lerp<1>(q[4], q[5], q[6], q[7], T.fx[1], T.fy[1], hi);
        out[0] = fmaf(T.f, hi[0] - lo[0], lo[0]) * (1.0f / 255.0f);
    } else {
        const uint32_t w0[4] = {q[0], q[1], q[2], q[3]}, w1[4] = {q[4], q[5], q[6], q[7]};
        float o[4];
        sample_word(w0, w1, T, true, o);                             // f == 0: the upper level repeats the lower one's taps
#pragma unroll
        for (int c = 0; c < NCH; ++c) out[c] = o[c];
    }
}

// what PSMain's Sample() calls return for one pixel (zeros where a map is not sampled or its SRV is null)
struct Sampled {
    float d[4];              // diffuse RGBA
    float n[3];              // tangent-space normal RGB
    float e[3];              // emissive RGB
    float ao, rg, mt;        // local AO .r, roughness .r, metalness .r
    float og, ob;            // ORM .g, .b
    bool nrm;                // a normal map is bound
};

__device__ __forceinline__ float pow22(float c) {                   // SRGBToLinear, ShadingMath.hlsl:65; c in [0,1]
    // lg2.approx / ex2.approx (2 ulp each) without exp2f()'s scaling for denormal results: c^2.2 of a sampled byte blend is either 0
    // (log2(0) = -inf -> ex2 = 0) or >= (1/255/2^20)^2.2, far above the denormal range
    float r; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(2.2f * __log2f(c))); return r;
}

struct SurfArgs {
    ImgV posU, nrmV, tanM;
    const float* ssao; int ssaoPitch;       // floats
    ImgV outPos, outNrm, outAlb, outEmi;    // outEmi.p == nullptr -> no emissive plane
    const DevMaterial* mats; int nMats;
    float ambient;
    int alphaMask;
    int rowBegin, rowEnd, tileY0;           // tileY0 = rowBegin & ~1 (quads are aligned to absolute even rows)
};

// One pixel of PSMain before lighting, from its interpolants (pu, nv, tm), its material index and the fine quad derivatives of
// the raw uv. Early returns = the alpha-mask discard.
__device__ __forceinline__ void shade_surface_pixel(const SurfArgs& A, int x, int y, int mi, float4 pu, float4 nv, float4 tm, float ssao,
                                                    float dRawUdx, float dRawVdx, float dRawUdy, float dRawVdy, uint64_t once) {
    const float ru = pu.w, rv = nv.w;
    const DevMaterial& M = A.mats[mi];
    const float4 c0 = __ldg((const float4*)&M.c), c1 = __ldg((const float4*)&M.c + 1);
    const float4 c2 = __ldg((const float4*)&M.c + 2), c3 = __ldg((const float4*)&M.c + 3), c4 = __ldg((const float4*)&M.c + 4);
    const uint4 rd = __ldg((const uint4*)&M.rec);                   // texel records of this material (pointer 0: none)
    // c0 = diffuse.rgb, alpha | c1 = emissiveColor.rgb, emissiveIntensity | c2 = specular.rgb, normalMapMipBias
    // c3 = uvScaleOffset | c4 = roughness, metalness, displacement, textureConfig
    const int cfg = (int)c4.w;

    const float u = __fadd_rn(__fmul_rn(ru, c3.x), c3.z), v = __fadd_rn(__fmul_rn(rv, c3.y), c3.w);   // :226
    const float dudx = dRawUdx * c3.x, dvdx = dRawVdx * c3.y, dudy = dRawUdy * c3.x, dvdy = dRawVdy * c3.y;

    Sampled S;
    S.d[0] = S.d[1] = S.d[2] = S.d[3] = 0.0f; S.n[0] = S.n[1] = S.n[2] = 0.0f; S.e[0] = S.e[1] = S.e[2] = 0.0f;
    S.ao = S.rg = S.mt = S.og = S.ob = 0.0f; S.nrm = false;
    Taps T;
    T.w = T.h = T.levels = -1; T.bias = 0.0f; T.f = 0.0f;

    if (rd.x | rd.y) {
        // ---- record path: the maps share one size, so ONE sampler state and 8 x LDG.128 serve every Sample() of the pixel ----
        TexR tr;
        tr.p = nullptr; tr.w = (int)(rd.z & 0x00ffffffu); tr.h = (int)(rd.w & 0x07ffffffu); tr.levels = (int)(rd.w >> 27);
        const uint4* R = (const uint4*)(((uint64_t)rd.y << 32) | rd.x);
        const uint32_t present = rd.z >> 24;                                // bit k: map k is bound
        S.nrm = (present & 2u) != 0u;
        make_taps(T, tr, u, v, dudx, dvdx, dudy, dvdy, 0.0f);
        const uint64_t keep = l2_policy_evict_last();
        const bool two = T.f != 0.0f;
        uint4 q[8];
#pragma unroll
        for (int k = 0; k < 4; ++k) q[k] = ld_record(R + T.i[0][k], keep);
        if (two) {
#pragma unroll
            for (int k = 0; k < 4; ++k) q[4 + k] = ld_record(R + T.i[1][k], keep);
        } else {
#pragma unroll
            for (int k = 0; k < 4; ++k) q[4 + k] = q[k];
        }
        const bool biasedNormal = S.nrm && c2.w != 0.0f;                    // SampleBias with its own LOD: a second set of taps
        uint32_t nq[8];
        Taps TN;
        bool twoN = false;
        if (biasedNormal) {
            TN.w = -1; TN.h = TN.levels = -1; TN.bias = 0.0f; TN.f = 0.0f;
            make_taps(TN, tr, u, v, dudx, dvdx, dudy, dvdy, c2.w);
            twoN = TN.f != 0.0f;
            const uint32_t* Rw = (const uint32_t*)R + 1;                    // word y of a record
#pragma unroll
            for (int k = 0; k < 4; ++k) { nq[k] = ld_texel(Rw + 4 * (size_t)TN.i[0][k], keep); nq[4 + k] = ld_texel(Rw + 4 * (size_t)TN.i[1][k], keep); }
        }
        float o[4];
        if (cfg & VQ_TEXCFG_DIFFUSE) {
            const uint32_t w0[4] = {q[0].x, q[1].x, q[2].x, q[3].x}, w1[4] = {q[4].x, q[5].x, q[6].x, q[7].x};
            sample_word(w0, w1, T, two, o);
            S.d[0] = o[0]; S.d[1] = o[1]; S.d[2] = o[2]; S.d[3] = o[3];
        }
        if ((S.nrm && !biasedNormal) || (cfg & VQ_TEXCFG_AO)) {
            const uint32_t w0[4] = {q[0].y, q[1].y, q[2].y, q[3].y}, w1[4] = {q[4].y, q[5].y, q[6].y, q[7].y};
            sample_word(w0, w1, T, two, o);
            S.n[0] = o[0]; S.n[1] = o[1]; S.n[2] = o[2]; S.ao = o[3];
        }
        if (biasedNormal) {
            const uint32_t w0[4] = {nq[0], nq[1], nq[2], nq[3]}, w1[4] = {nq[4], nq[5], nq[6], nq[7]};
            sample_word(w0, w1, TN, twoN, o);
            S.n[0] = o[0]; S.n[1] = o[1]; S.n[2] = o[2];
        }
        if (cfg & (VQ_TEXCFG_EMISSIVE | VQ_TEXCFG_ROUGHNESS)) {
            const uint32_t w0[4] = {q[0].z, q[1].z, q[2].z, q[3].z}, w1[4] = {q[4].z, q[5].z, q[6].z, q[7].z};
            sample_word(w0, w1, T, two, o);
            S.e[0] = o[0]; S.e[1] = o[1]; S.e[2] = o[2]; S.rg = o[3];
        }
        if (cfg & (VQ_TEXCFG_METALLIC | VQ_TEXCFG_ORM)) {
            const uint32_t w0[4] = {q[0].w, q[1].w, q[2].w, q[3].w}, w1[4] = {q[4].w, q[5].w, q[6].w, q[7].w};
            sample_word(w0, w1, T, two, o);
            S.mt = o[0]; S.og = o[1]; S.ob = o[2];
        }
    } else {
        // ---- one map at a time (maps of different sizes): a Sample() = 8 x LDG.32 ----
        // (one looped copy of the sampler instead of these seven inlined ones shrinks the kernel from 92 KB to 36 KB of code but
        //  executes 11 % more instructions — four channels for every map, routing by slot: 0.415 ms against 0.371, not kept)
        if (cfg & VQ_TEXCFG_DIFFUSE) {
            const TexR tDiff = load_tex(&M.t[0]);
            if (tDiff.p) {
                if (A.alphaMask) sample8<4>(T, tDiff, u, v, dudx, dvdx, dudy, dvdy, 0.0f, S.d);
                else { float s3[3]; sample8<3>(T, tDiff, u, v, dudx, dvdx, dudy, dvdy, 0.0f, s3); S.d[0] = s3[0]; S.d[1] = s3[1]; S.d[2] = s3[2]; }
            }
            if (A.alphaMask && S.d[3] < 0.01f) return;                                                // discard before the other maps are read
        }
        if (cfg & VQ_TEXCFG_EMISSIVE) {
            const TexR tEmi = load_tex(&M.t[2]);
            if (tEmi.p) sample8<3>(T, tEmi, u, v, dudx, dvdx, dudy, dvdy, 0.0f, S.e);
        }
        const TexR tNrm = load_tex(&M.t[1]);                                                          // sampled whatever the config says
        if (tNrm.p) { S.nrm = true; sample8<3>(T, tNrm, u, v, dudx, dvdx, dudy, dvdy, c2.w, S.n); }
        if (cfg & VQ_TEXCFG_AO)        { float s[1] = {0.f}; const TexR t = load_tex(&M.t[6]); if (t.p) sample8<1>(T, t, u, v, dudx, dvdx, dudy, dvdy, 0.0f, s); S.ao = s[0]; }
        if (cfg & VQ_TEXCFG_ROUGHNESS) { float s[1] = {0.f}; const TexR t = load_tex(&M.t[4]); if (t.p) sample8<1>(T, t, u, v, dudx, dvdx, dudy, dvdy, 0.0f, s); S.rg = s[0]; }
        if (cfg & VQ_TEXCFG_METALLIC)  { float s[1] = {0.f}; const TexR t = load_tex(&M.t[3]); if (t.p) sample8<1>(T, t, u, v, dudx, dvdx, dudy, dvdy, 0.0f, s); S.mt = s[0]; }
        if (cfg & VQ_TEXCFG_ORM) {
            float s[3] = {0.f, 0.f, 0.f};
            const TexR t = load_tex(&M.t[5]);
            if (t.p) sample8<3>(T, t, u, v, dudx, dvdx, dudy, dvdy, 0.0f, s);
            S.og = s[1]; S.ob = s[2];
        }
    }

    // --- diffuse (+alpha for the ENABLE_ALPHA_MASK variant, :237-240) ---
    float3 diffuseColor = f3(c0.x, c0.y, c0.z);
    if (cfg & VQ_TEXCFG_DIFFUSE) {
        if (A.alphaMask && S.d[3] < 0.01f) return;                                                    // discard
        diffuseColor = f3(pow22(S.d[0]) * c0.x, pow22(S.d[1]) * c0.y, pow22(S.d[2]) * c0.z);          // :243,249
    }
    // --- emissive ---
    float3 emissiveColor = f3(c1.x, c1.y, c1.z);
    if (cfg & VQ_TEXCFG_EMISSIVE) emissiveColor = f3(pow22(S.e[0]) * c1.x, pow22(S.e[1]) * c1.y, pow22(S.e[2]) * c1.z);   // :244,250
    float roughness = c4.x, metalness = c4.y;                                                         // :252-253
    float ao = A.ambient;                                                                             // :247

    // --- normal: N / T from the interpolants, tangent-space normal whenever the sample is not ~0 (:265-267) ---
    const float3 Nw = f3(nv.x, nv.y, nv.z), Tw = f3(tm.x, tm.y, tm.z);
    const float3 N = Nw * rsqrtf(dot(Nw, Nw));
    float3 Nout = N;
    if (S.nrm) {
        const float* s = S.n;
        if (sqrtf(s[0] * s[0] + s[1] * s[1] + s[2] * s[2]) >= 0.01f) {
            const float3 T0 = Tw * rsqrtf(dot(Tw, Tw));
            float3 sn = f3(s[0] * 2.0f - 1.0f, s[1] * 2.0f - 1.0f, s[2] * 2.0f - 1.0f);               // ShadingMath.hlsl:46
            sn = sn * rsqrtf(dot(sn, sn));
            float3 T = T0 - N * dot(N, T0);                                                           // :47
            T = T * rsqrtf(dot(T, T));
            const float3 Nn = N * rsqrtf(dot(N, N));                                                  // :48 (N is already unit)
            float3 B = cross(T, Nn);                                                                  // :49
            B = B * rsqrtf(dot(B, B));
            Nout = T * sn.x + B * sn.y + Nn * sn.z;                                                   // :50-51
        }
    }
    if (cfg & VQ_TEXCFG_AO)        ao *= S.ao;                                                        // :269
    if (cfg & VQ_TEXCFG_ROUGHNESS) roughness *= S.rg;                                                 // :270
    if (cfg & VQ_TEXCFG_METALLIC)  metalness *= S.mt;                                                 // :271
    if (cfg & VQ_TEXCFG_ORM) { roughness *= S.og; metalness *= S.ob; }                                // :272-277
    ao *= ssao;                                                                                       // :280-281 (1 when no SSAO plane is bound)

    st_once(A.outPos.row(y) + x, make_float4(pu.x, pu.y, pu.z, ao), once);
    st_once(A.outNrm.row(y) + x, make_float4(Nout.x, Nout.y, Nout.z, roughness), once);
    st_once(A.outAlb.row(y) + x, make_float4(diffuseColor.x, diffuseColor.y, diffuseColor.z, metalness), once);
    if (A.outEmi.p) st_once(A.outEmi.row(y) + x, make_float4(emissiveColor.x, emissiveColor.y, emissiveColor.z, c1.w), once);
}

// block = 256 threads = 8 warps; a warp shades 16x2 pixels (one row of 2x2 quads), a block 32x8.
// Three restructurings of this launch were measured and NOT kept (profiles/r02_surface_variants.txt): queueing a warp's minority-
// material pixels for a second pass inside the block (0.49 ms) or for a second small launch (0.45 ms) against 0.37 ms in place —
// the majority paths dominate the instruction count, not the stray lanes; and a persistent kernel with the interpolant planes on a
// TMA / mbarrier ring like K1's (0.49 ms) — the waits are on the texel and SSAO loads, not on the interpolants, and 92 KB of code
// with every warp of an SM somewhere else in it stalls on instruction fetch. Several tiles per block, each prefetching the
// next tile's interpolants, were slower too: the extra live registers spill (profiles/r02_surface_variants.txt).
struct SurfTexels { float4 pu, nv, tm; float ssao; };
__device__ __forceinline__ SurfTexels surface_fetch(const SurfArgs& A, int x, int y, uint64_t once) {
    const int W = A.posU.w, H = A.posU.h;
    // threads outside the image re-read the clamped texel: their uv equals the in-image partner's -> derivative 0,
    // exactly the oracle's "partner clamped to the image"
    const int cx = min(x, W - 1), cy = min(y, H - 1);
    SurfTexels t;
    t.pu = ld_once(A.posU.row(cy) + cx, once);
    t.nv = ld_once(A.nrmV.row(cy) + cx, once);
    t.tm = ld_once(A.tanM.row(cy) + cx, once);
    // the SSAO texel (x+1, y+1, WRAP; :280-281) depends on nothing but the pixel: fetched with the interpolants, not at the point
    // of use after the whole sampling chain (where it was 17 % of the kernel's long-scoreboard stalls)
    t.ssao = 1.0f;
    if (A.ssao) {
        const int sxp = cx + 1 == W ? 0 : cx + 1, syp = cy + 1 == H ? 0 : cy + 1;
        t.ssao = __ldg(A.ssao + (size_t)syp * A.ssaoPitch + sxp);
    }
    return t;
}

__global__ void __launch_bounds__(256, SURF_MIN_BLOCKS) surface_kernel(const __grid_constant__ SurfArgs A) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int x = blockIdx.x * 32 + (warp & 1) * 16 + (lane & 15);
    const int y = A.tileY0 + blockIdx.y * 8 + (warp >> 1) * 2 + (lane >> 4);
    const int W = A.posU.w, H = A.posU.h;
    const uint64_t once = l2_policy_evict_first();
    const SurfTexels cur = surface_fetch(A, x, y, once);
    const float ru = cur.pu.w, rv = cur.nv.w;
    // fine quad derivatives of the RAW uv: horizontal partner = lane^1, vertical = lane^16
    const float ruX = __shfl_xor_sync(0xffffffffu, ru, 1), rvX = __shfl_xor_sync(0xffffffffu, rv, 1);
    const float ruY = __shfl_xor_sync(0xffffffffu, ru, 16), rvY = __shfl_xor_sync(0xffffffffu, rv, 16);
    const float sx = (lane & 1) ? -1.0f : 1.0f, sy = (lane & 16) ? -1.0f : 1.0f;   // (odd - even) regardless of which I am
    const float dRawUdx = (ruX - ru) * sx, dRawVdx = (rvX - rv) * sx;
    const float dRawUdy = (ruY - ru) * sy, dRawVdy = (rvY - rv) * sy;
    if (x < W && y < H && y >= A.rowBegin && y < A.rowEnd) {
        const int mi = min(max((int)cur.tm.w, 0), A.nMats - 1);
        shade_surface_pixel(A, x, y, mi, cur.pu, cur.nv, cur.tm, cur.ssao, dRawUdx, dRawVdx, dRawUdy, dRawVdy, once);
    }
}

// interleaves the texels of a material's seven maps (same size, same level count; nullptr = null SRV = zeros) into records
struct RecBuildArgs { const uint32_t* src[7]; uint4* dst; uint32_t n; };
__global__ void __launch_bounds__(256) record_build_kernel(const __grid_constant__ RecBuildArgs A) {
    const uint32_t i = blockIdx.x * 256u + threadIdx.x;
    if (i >= A.n) return;
    uint32_t t[7];
#pragma unroll
    for (int k = 0; k < 7; ++k) t[k] = A.src[k] ? __ldg(A.src[k] + i) : 0u;
    // slots: 0 diffuse, 1 normals, 2 emissive, 3 metalness, 4 roughness, 5 occl_rough_metal, 6 local_ao
    A.dst[i] = make_uint4(t[0], (t[1] & 0x00ffffffu) | (t[6] << 24), (t[2] & 0x00ffffffu) | (t[4] << 24), (t[3] & 0xffu) | (t[5] & 0x00ffff00u));
}

static bool tex_ok(const VqTexture2D& t) {
    if (!t.ptr) return true;     // null SRV
    return t.width > 0 && t.height > 0 && t.levels >= 1 && t.levels <= vq_mip_level_count((uint64_t)t.width, (uint64_t)t.height) &&
           t.levels <= 31 && t.height < (1 << 27) && ((uintptr_t)t.ptr % 4) == 0;
}

}  // namespace

extern "C" int vq_texture_build_mips(VqContext* ctx, VqTexture2D tex, void* stream) {
    int rc = vq_enter(ctx); if (rc) return rc;
    VQ_REQUIRE(tex.ptr && tex_ok(tex), "bad texture descriptor");
    uint32_t* base = (uint32_t*)tex.ptr;
    for (int l0 = 0; l0 + 1 < tex.levels; l0 += 6) {                   // source level l0 -> levels l0+1 .. l0+6
        MipArgs A;
        A.src = base + vq_pyramid_offset(tex.width, tex.height, l0);
        A.sw = tex.width >> l0; A.sh = tex.height >> l0;
        A.n = tex.levels - 1 - l0 < 6 ? tex.levels - 1 - l0 : 6;
        for (int j = 0; j < 6; ++j) A.dst[j] = j < A.n ? base + vq_pyramid_offset(tex.width, tex.height, l0 + 1 + j) : nullptr;
        const dim3 grid((A.sw + 63) / 64, (A.sh + 63) / 64);
        tex_mip6_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(A);
        rc = vq_check_launch("texture_build_mips"); if (rc) return rc;
    }
    return VQ_OK;
}

extern "C" int vq_material_table_create(VqContext* ctx, const VqMaterialData* materials, const VqMaterialTextures* textures,
                                        int count, VqMaterialTable** out_table) {
    int rc = vq_enter(ctx); if (rc) return rc;
    VQ_REQUIRE(materials && textures && out_table, "null argument");
    VQ_REQUIRE(count >= 1 && count <= (1 << 20), "material count out of range");
    DevMaterial* host = (DevMaterial*)calloc((size_t)count, sizeof(DevMaterial));
    if (!host) { vq_set_error("out of host memory"); return VQ_ERR_OUT_OF_MEMORY; }
    for (int i = 0; i < count; ++i) {
        host[i].c = materials[i];
        const VqTexture2D* src = &textures[i].diffuse;     // 7 consecutive descriptors
        for (int k = 0; k < 7; ++k) {
            if (!tex_ok(src[k])) { free(host); vq_set_error("invalid argument: material %d texture %d descriptor", i, k); return VQ_ERR_INVALID_ARG; }
            DevTex& d = host[i].t[k];
            if (!src[k].ptr) continue;                                  // null SRV: p = nullptr, reads 0
            if (vq_pyramid_texel_count(src[k].width, src[k].height, src[k].levels) > 0xffffffffull) {
                free(host); vq_set_error("invalid argument: texture too large for 32-bit texel offsets"); return VQ_ERR_INVALID_ARG;
            }
            d.p = (const uint32_t*)src[k].ptr; d.w = src[k].width;
            d.h_levels = (uint32_t)src[k].height | ((uint32_t)src[k].levels << 27);
        }
    }
    // texel records (see DevMaterial): a material qualifies when at least two maps are bound and every bound map has the same
    // width, height and level count. VQ_SURFACE_RECORDS=0 in the environment keeps every material on the map-by-map path.
    const char* recEnv = getenv("VQ_SURFACE_RECORDS");
    const bool wantRecords = !(recEnv && recEnv[0] == '0');
    uint64_t recTexels = 0;
    uint64_t* recOffset = (uint64_t*)calloc((size_t)count, sizeof(uint64_t));
    uint64_t* recCount = (uint64_t*)calloc((size_t)count, sizeof(uint64_t));
    if (!recOffset || !recCount) { free(host); free(recOffset); free(recCount); vq_set_error("out of host memory"); return VQ_ERR_OUT_OF_MEMORY; }
    for (int i = 0; wantRecords && i < count; ++i) {
        const VqTexture2D* src = &textures[i].diffuse;
        int bound = 0, first = -1; bool same = true;
        for (int k = 0; k < 7; ++k) {
            if (!src[k].ptr) continue;
            if (first < 0) first = k;
            else same = same && src[k].width == src[first].width && src[k].height == src[first].height && src[k].levels == src[first].levels;
            ++bound;
        }
        if (bound < 2 || !same || src[first].width >= (1 << 24)) continue;
        recOffset[i] = recTexels;
        recCount[i] = vq_pyramid_texel_count(src[first].width, src[first].height, src[first].levels);
        recTexels += recCount[i];
    }
    VqMaterialTable* t = (VqMaterialTable*)calloc(1, sizeof(VqMaterialTable));
    if (!t) { free(host); free(recOffset); free(recCount); vq_set_error("out of host memory"); return VQ_ERR_OUT_OF_MEMORY; }
    cudaError_t e = cudaSuccess;
    if (recTexels) {
        // a sampling copy is an optimisation: when it does not fit, the materials simply stay on the map-by-map path
        if (cudaMalloc(&t->records, (size_t)recTexels * 16) != cudaSuccess) { cudaGetLastError(); t->records = nullptr; recTexels = 0; }
        else t->record_bytes = (size_t)recTexels * 16;
    }
    if (t->records) {
        e = cudaDeviceSynchronize();                                    // mip chains may still be in flight on the caller's streams
        for (int i = 0; e == cudaSuccess && i < count; ++i) {
            if (!recCount[i]) continue;
            const VqTexture2D* src = &textures[i].diffuse;
            RecBuildArgs B;
            uint32_t present = 0; int first = -1;
            for (int k = 0; k < 7; ++k) { B.src[k] = (const uint32_t*)src[k].ptr; if (src[k].ptr) { present |= 1u << k; if (first < 0) first = k; } }
            B.dst = (uint4*)t->records + recOffset[i]; B.n = (uint32_t)recCount[i];
            record_build_kernel<<<(unsigned)((recCount[i] + 255) / 256), 256>>>(B);
            vq_count_launch();
            e = cudaGetLastError();
            host[i].rec.p = (const uint32_t*)B.dst;
            host[i].rec.w = src[first].width | (int32_t)(present << 24);
            host[i].rec.h_levels = (uint32_t)src[first].height | ((uint32_t)src[first].levels << 27);
        }
        if (e == cudaSuccess) e = cudaDeviceSynchronize();
    }
    free(recOffset); free(recCount);
    if (e == cudaSuccess) e = cudaMalloc(&t->dev, (size_t)count * sizeof(DevMaterial));
    if (e == cudaSuccess) e = cudaMemcpy(t->dev, host, (size_t)count * sizeof(DevMaterial), cudaMemcpyHostToDevice);
    free(host);
    if (e != cudaSuccess) {
        if (t->dev) cudaFree(t->dev);
        if (t->records) cudaFree(t->records);
        free(t);
        vq_set_error("material table upload failed: %s", cudaGetErrorString(e));
        return e == cudaErrorMemoryAllocation ? VQ_ERR_OUT_OF_MEMORY : VQ_ERR_CUDA;
    }
    t->count = count;
    *out_table = t;
    return VQ_OK;
}

extern "C" int vq_material_table_destroy(VqContext* ctx, VqMaterialTable* table) {
    int rc = vq_enter(ctx); if (rc) return rc;
    if (!table) return VQ_OK;
    if (table->dev) cudaFree(table->dev);
    if (table->records) cudaFree(table->records);
    free(table);
    return VQ_OK;
}

extern "C" int vq_gbuffer_from_materials(VqContext* ctx, const VqSurfaceInputs* in, const VqMaterialTable* table,
                                         float ambient_factor, int alpha_mask, const VqGBuffer* out,
                                         int row_begin, int row_end, void* stream) {
    int rc = vq_enter(ctx); if (rc) return rc;
    VQ_MARK("Geometry");
    VQ_REQUIRE(in && table && out, "null argument");
    VQ_REQUIRE(table->dev && table->count >= 1, "empty material table");
    const int W = in->position_u.width, H = in->position_u.height;
    VQ_REQUIRE(vq_image_ok(in->position_u) && vq_image_ok(in->normal_v) && vq_image_ok(in->tangent_m), "bad attribute plane");
    VQ_REQUIRE(in->normal_v.width == W && in->normal_v.height == H && in->tangent_m.width == W && in->tangent_m.height == H,
               "attribute planes differ in size");
    VQ_REQUIRE(vq_image_ok(out->position_ao) && vq_image_ok(out->normal_roughness) && vq_image_ok(out->albedo_metalness), "bad G-buffer plane");
    VQ_REQUIRE(out->position_ao.width == W && out->position_ao.height == H && out->normal_roughness.width == W &&
               out->normal_roughness.height == H && out->albedo_metalness.width == W && out->albedo_metalness.height == H,
               "G-buffer planes differ in size from the attribute planes");
    if (out->emissive.ptr)
        VQ_REQUIRE(vq_image_ok(out->emissive) && out->emissive.width == W && out->emissive.height == H, "bad emissive plane");
    if (in->ssao.ptr)
        VQ_REQUIRE(vq_image_ok(in->ssao, 4) && in->ssao.width == W && in->ssao.height == H, "bad SSAO plane");
    VQ_REQUIRE(row_begin >= 0 && row_end <= H && row_begin <= row_end, "row range out of bounds");
    if (row_begin == row_end) return VQ_OK;

    SurfArgs A;
    A.posU = make_view(in->position_u); A.nrmV = make_view(in->normal_v); A.tanM = make_view(in->tangent_m);
    A.ssao = (const float*)in->ssao.ptr; A.ssaoPitch = in->ssao.ptr ? (int)(in->ssao.pitch_bytes / 4) : 0;
    A.outPos = make_view(out->position_ao); A.outNrm = make_view(out->normal_roughness); A.outAlb = make_view(out->albedo_metalness);
    if (out->emissive.ptr) A.outEmi = make_view(out->emissive); else { A.outEmi.p = nullptr; A.outEmi.w = A.outEmi.h = A.outEmi.pitch4 = 0; }
    A.mats = table->dev; A.nMats = table->count;
    A.ambient = ambient_factor; A.alphaMask = alpha_mask;
    A.rowBegin = row_begin; A.rowEnd = row_end; A.tileY0 = row_begin & ~1;
    const dim3 grid((W + 31) / 32, (row_end - A.tileY0 + 7) / 8);
    surface_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(A);
    return vq_check_launch("gbuffer_from_materials");
}

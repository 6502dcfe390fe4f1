// vq_forward.cu — K1 forward PBR lighting for sm_100a.
//
// Replaces VQRenderer::RenderSceneColor (SceneRendering.cpp:1619-1851) + PSMain
// (ForwardLighting.hlsl:285-380) over a G-buffer of three float4 planes (+ optional emissive):
//   64 B/pixel of HBM traffic: the three planes arrive as 4 KB row segments through a TMA (cp.async.bulk) /
//   mbarrier ring in shared memory, the result leaves as one STG.128 per pixel; one thread shades TWO pixels with packed
//   fp32x2 arithmetic (FFMA2/FMUL2/FADD2: half the issue slots of the light loop); the light array is staged once per
//   CTA into shared memory; the IBL cubemaps and the BRDF LUT are gathered from L2-resident sampling copies
//   (pair / footprint records, 102 MB at the reference sizes) with five 256-bit loads per pixel, because the
//   L1 data pipe — one wavefront per distinct line of a divergent gather — is what bounds this kernel (DESIGN.md §4).
// The math is PSMain's with per-pixel invariants hoisted out of the light loops (N, V, N.V, the
// Smith-G term of V, F0, kD factors). Discontinuities are evaluated exactly as the oracle does:
//   * `D < l.range` uses an unfused |L-P|^2 and a per-light threshold on the squared distance that is
//     equivalent to the correctly-rounded sqrt compare;
//   * the specular mip is int(roughness * MAX_LOD) (one fp32 multiply);
//   * cubemap taps are seamless across face edges, so face selection is not a discontinuity.
#include "vq_common.cuh"
#include <stdlib.h>

using namespace vq;

namespace {


// Sampling copy of a cubemap. Every face of every mip is a (N+2)x(N+2) grid of bordered texel positions, the 1-texel
// border holding the neighbouring faces' edge texels (corners: the mean of the three texels that meet there), so
// that the seamless bilinear footprint never leaves the face. Each position (i,j) stores the PAIR {t(i,j), t(i+1,j)}
// as one 32-byte record: a bilinear footprint is two 256-bit loads (LDG.E.256, sm_100) instead of four 128-bit ones.
// K1 is bound by the L1 data pipe (one wavefront per distinct 128-byte line a warp-wide load touches, ~20-30 for a
// gather whose lanes go to unrelated texels), so the number of gather INSTRUCTIONS per pixel is what the layout
// minimises: 12 -> 5. mipOffset[] are record offsets of face 0 per mip.
struct CubeV { const float4* p; int res, mips; uint32_t mipOffset[16]; };
// Footprint copy of the BRDF LUT: record (cx,cy), cx = clamp(x0+1, 0, W), holds the CLAMP-addressed 2x2 footprint
// {p(x0,y0), p(x0+1,y0), p(x0,y0+1), p(x0+1,y0+1)} as 4 x float2 = 32 bytes: one 256-bit load per pixel.
struct LutV { const float4* q; int w, h; };
struct F8 { float4 a, b; };

struct SPoint { float3 pos; float d2Limit; float3 color; float brightness; };
struct SDir { float3 wi; float pad0; float3 radiance; float pad1; };
struct SSpot { float3 pos; float outer; float3 color; float brightness; float3 dir; float inner; float invCone; float pad[3]; };
constexpr int FWD_MAX_POINT = VQ_NUM_LIGHTS_POINT + VQ_NUM_SHADOWING_LIGHTS_POINT, FWD_MAX_SPOT = VQ_NUM_LIGHTS_SPOT + VQ_NUM_SHADOWING_LIGHTS_SPOT;

struct FwdParams {
    // the frame's lights, conditioned on the host (exact range thresholds, normalised directions, radiance) and read by the kernel
    // straight from the constant bank with warp-uniform indices: no shared-memory staging, no LDS in the light loop (the L1/MIO
    // pipe that the environment gathers keep busy is left alone)
    SPoint pts[FWD_MAX_POINT];         // point lights, then (unshadowed) point casters
    SSpot spots[FWD_MAX_SPOT];         // spot lights, then spot casters
    SDir dir;
    int numPoint, numSpot, dirEnabled;
    float3 cam;
    float cosB, sinB;                  // GetHDRIRotationMatrix (Lighting.hlsl:348-358), cos/sin(-offset)
    int maxLod;                        // int(MaxEnvMapLODLevels)
    int diffuseOnly;
    int hasEmissive;
    ImgV pos, nrm, alb, emi;
    ImgV outs[8];                      // destinations: the local frame and, for the fused gather, the peers' frames (NVLink P2P)
    int nOut, dstRowOffset;            // every shaded pixel goes to row dstRowOffset+y of every destination
    CubeV diff, spec;
    LutV lut;
    PeerSync sync;                     // MULTI: optional end-of-pass rendezvous run by the last CTA (n == 0: none)
    uint32_t* ticket;                  // MULTI: retired-CTA count (zero between launches)
    float diffHalfN;                   // res/2 of the diffuse cube
    uint32_t diffMaxRec, specMaxRec;   // last record a footprint may start at (address clamp for non-finite directions)
    int rowBegin, rows, width;
    // SHADOWED instantiation only (vq_forward_lighting_shadowed): PCF tap counts per pixel and caster; the caster lights are the
    // LAST nPointCasters / nSpotCasters entries of pts[] / spots[]
    ShadowRecV shadow;
};

// ---------------------------------------------------------------------------------------------
// cubemap sampling: bilinear, seamless (SURVEY.md §9; identical rule in oracle/oracle_shading.cpp)
// ---------------------------------------------------------------------------------------------
// D3D face selection (largest |component|; ties X > Y > Z as in the oracle) written with selects so that a warp never
// diverges on it:  face, and the face-plane coordinates sx (right), sy (up) in [-1,1]
__device__ __forceinline__ void dir_to_face(float3 d, int& face, float& sx, float& sy) {
    const float ax = fabsf(d.x), ay = fabsf(d.y), az = fabsf(d.z);
    const bool isX = ax >= ay && ax >= az;
    const bool isY = !isX && ay >= az;
    const float ma = isX ? ax : (isY ? ay : az);
    const float mv = isX ? d.x : (isY ? d.y : d.z);          // signed major component
    const bool pos = mv > 0.0f;
    const float r = rcp_fast(ma);
    // +X: (-z, y)  -X: (z, y)  +Y: (x, -z)  -Y: (x, z)  +Z: (x, y)  -Z: (-x, y)
    const float u = isX ? (pos ? -d.z : d.z) : (isY ? d.x : (pos ? d.x : -d.x));
    const float v = isY ? (pos ? -d.z : d.z) : d.y;
    sx = u * r; sy = v * r;
    face = (isX ? 0 : (isY ? 2 : 4)) + (pos ? 0 : 1);
}

// integer-only neighbour lookup for a tap one texel outside the face (see DESIGN.md "cube edges"); used only by
// the border-padding kernel, never per pixel
__device__ void cube_resolve_edge(int N, int face, int i, int j, int& of, int& oi, int& oj) {
    const int A = 2 * i + 1 - N, B = N - 1 - 2 * j, C = N;
    int dx, dy, dz;
    switch (face) {
        case 0: dx = C;  dy = B;  dz = -A; break;
        case 1: dx = -C; dy = B;  dz = A;  break;
        case 2: dx = A;  dy = C;  dz = -B; break;
        case 3: dx = A;  dy = -C; dz = B;  break;
        case 4: dx = A;  dy = B;  dz = C;  break;
        default: dx = -A; dy = B; dz = -C; break;
    }
    const int M = N + 1;
    int nsx, nsy;
    if (dx == M)       { of = 0; nsx = -dz; nsy = dy; }
    else if (dx == -M) { of = 1; nsx = dz;  nsy = dy; }
    else if (dy == M)  { of = 2; nsx = dx;  nsy = -dz; }
    else if (dy == -M) { of = 3; nsx = dx;  nsy = dz; }
    else if (dz == M)  { of = 4; nsx = dx;  nsy = dy; }
    else               { of = 5; nsx = -dx; nsy = dy; }
    oi = min(max(((nsx + M) * N) / (2 * M), 0), N - 1);
    oj = min(max(((M - nsy) * N) / (2 * M), 0), N - 1);
}

// value of bordered position `idx` (flattened over mips, faces, (N+2)^2 positions) of a packed cube
__device__ float4 bordered_texel(const float4* __restrict__ src, int res, int mips, uint32_t idx) {
    uint32_t rem = idx, srcOff = 0; int m = 0, N = res;
    for (; m < mips; ++m) {
        N = res >> m;
        const uint32_t sz = 6u * (uint32_t)(N + 2) * (uint32_t)(N + 2);
        if (rem < sz) break;
        rem -= sz; srcOff += 6u * (uint32_t)N * (uint32_t)N;
    }
    const int P = N + 2;
    const int face = (int)(rem / (uint32_t)(P * P));
    const int r2 = (int)(rem % (uint32_t)(P * P));
    const int i = r2 % P - 1, j = r2 / P - 1;           // face-relative texel, -1..N
    const float4* sm = src + srcOff;
    auto fetch = [&](int f, int x, int y) { return __ldg(sm + (size_t)f * N * N + (size_t)y * N + x); };
    auto edge = [&](int x, int y) { int f2, i2, j2; cube_resolve_edge(N, face, x, y, f2, i2, j2); return fetch(f2, i2, j2); };
    const bool oi = (i < 0 || i >= N), oj = (j < 0 || j >= N);
    if (!oi && !oj) return fetch(face, i, j);
    if (oi != oj) return edge(i, j);
    // cube corner: mean of the three texels meeting there (own corner + the two edge neighbours)
    const int ci = i < 0 ? 0 : N - 1, cj = j < 0 ? 0 : N - 1;
    const float4 a = fetch(face, ci, cj), b = edge(i, cj), c = edge(ci, j);
    return make_float4((a.x + b.x + c.x) * (1.0f / 3.0f), (a.y + b.y + c.y) * (1.0f / 3.0f),
                       (a.z + b.z + c.z) * (1.0f / 3.0f), (a.w + b.w + c.w) * (1.0f / 3.0f));
}
// packed cube (mip-major / face-minor, N x N faces) -> sampling copy: one {t(i,j), t(i+1,j)} record per bordered position
// (the last position of a row repeats itself; it is never the left tap of a footprint)
__global__ void __launch_bounds__(256) cube_pad_kernel(const float4* __restrict__ src, float4* __restrict__ dst,
                                                        int res, int mips, uint32_t totalPadded) {
    for (uint32_t idx = blockIdx.x * 256u + threadIdx.x; idx < totalPadded; idx += gridDim.x * 256u) {
        // is idx the last position of its row?  rows are (N+2) long and faces/mips are whole rows, so walk the mips
        uint32_t rem = idx; int P = res + 2;
        for (int m = 0; m < mips; ++m) {
            P = (res >> m) + 2;
            const uint32_t sz = 6u * (uint32_t)P * (uint32_t)P;
            if (rem < sz) break;
            rem -= sz;
        }
        const bool last = (rem % (uint32_t)P) == (uint32_t)(P - 1);
        const float4 v0 = bordered_texel(src, res, mips, idx);
        const float4 v1 = last ? v0 : bordered_texel(src, res, mips, idx + 1u);
        dst[2 * (size_t)idx] = v0;
        dst[2 * (size_t)idx + 1] = v1;
    }
}

// BRDF LUT (float2, pitched) -> footprint records (see LutV): (W+1) x (H+1) records of 32 bytes
__global__ void __launch_bounds__(256) lut_footprint_kernel(const float2* __restrict__ src, int pitch2, int W, int H, float4* __restrict__ dst) {
    const uint32_t total = (uint32_t)(W + 1) * (uint32_t)(H + 1);
    for (uint32_t idx = blockIdx.x * 256u + threadIdx.x; idx < total; idx += gridDim.x * 256u) {
        const int cx = (int)(idx % (uint32_t)(W + 1)), cy = (int)(idx / (uint32_t)(W + 1));
        const int x0 = max(cx - 1, 0), x1 = min(cx, W - 1), y0 = max(cy - 1, 0), y1 = min(cy, H - 1);
        const float2 p00 = __ldg(src + (size_t)y0 * pitch2 + x0), p10 = __ldg(src + (size_t)y0 * pitch2 + x1);
        const float2 p01 = __ldg(src + (size_t)y1 * pitch2 + x0), p11 = __ldg(src + (size_t)y1 * pitch2 + x1);
        dst[2 * (size_t)idx] = make_float4(p00.x, p00.y, p10.x, p10.y);
        dst[2 * (size_t)idx + 1] = make_float4(p01.x, p01.y, p11.x, p11.y);
    }
}

// ---------------------------------------------------------------------------------------------
// packed fp32x2 arithmetic (FADD2 / FMUL2 / FFMA2, new on sm_100)
// ---------------------------------------------------------------------------------------------
// K1 is bound by instruction issue (profiles/r01_forward_g_summary.txt: 904 warp-instructions per 32 pixels, more than half of
// them FADD/FMUL/FFMA), so one thread shades TWO pixels and every quantity of the light loop is a pair {pixel A, pixel B} in
// an aligned 64-bit register pair: one packed instruction does the work of two at one issue slot. Lane .x of every f2
// is pixel A (column x0 + tid), lane .y pixel B (column x0 + 128 + tid). MUFU, compares, selects and min/max have no packed
// form and stay per lane (profiles/r02_forward_*: 80 -> 42 issue slots per pixel and light).

// ---------------------------------------------------------------------------------------------
// per-pixel-pair shading state with everything that does not depend on the light hoisted
// ---------------------------------------------------------------------------------------------
struct Px2 {
    float3 PA, PB;                // positions of the two pixels (scalar: every use is a first-touch subtraction)
    f2 Nx, Ny, Nz;                // normalize(Ns)                                   (BRDF.hlsl:167)
    f2 Vx, Vy, Vz;                // normalize(cam - P)                              (ForwardLighting.hlsl:285)
    f2 nsLen;                     // |Ns|: dot(Ns,Wi) = nsLen * dot(Nn,Wi)           (Lighting.hlsl:316 uses the raw s.N)
    f2 nv, nv4;                   // dot(Nn,V), 4*saturate(dot(Nn,V))
    f2 a2m1;                      // roughness^4 - 1 (unfused, feeds the exact t)
    f2 a2gV, gV;                  // a2 * G1(V), G1(V) = Smith-Schlick-GGX of the view vector (BRDF.hlsl:82-97)
    f2 k4, omk;                   // k + 0.0001, 1 - k with k = (roughness+1)^2 / 8
    uint32_t texA, texB;          // shared-memory addresses of the two pixels' position texels (planes follow at FWD_PLANE)
    uint64_t recA, recB;          // SHADOWED only: the two pixels' PCF records (ShadowRecV, vq_common.cuh)
};
struct Acc2 { f2 ax, ay, az, bx, by, bz, cx, cy, cz; };   // sum over lights of w*col * {(1-fc), fc*spec, spec}

// ---- exact re-evaluation of N.H -------------------------------------------------------------------
// GGX's t = nh2*(a2-1)+1 cancels catastrophically near a highlight on a smooth surface (t ~ a2 ~ 1e-5),
// so D amplifies a 1-ulp difference in N.H by up to 1e4. Where t is small the kernel therefore recomputes
// N.H with the oracle's exact operation sequence (correctly rounded div/sqrt, no FMA contraction): V, Wo,
// N, Wi, H as BRDF.hlsl:166-169 / Lighting.hlsl:312 write them. T_EXACT = 0.02 bounds the fast path's
// relative error in D by 2*dt/t <= 2*5e-7/0.02 = 5e-5; the slow path runs for < 1 % of pixel-light pairs.
constexpr float T_EXACT = 0.02f;

// dot_u, sqrt_rn_inrange, rcp_rn_prepare / div_rn_inrange, len2_inrange: vq_common.cuh (shared with the PCF kernel)
// v / sqrt(dot(v,v)) with correctly rounded sqrt and divisions (== the oracle's normalize)
__device__ __noinline__ float3 normalize_u_generic(float3 v) {
    const float l = __fsqrt_rn(dot_u(v, v));
    return f3(__fdiv_rn(v.x, l), __fdiv_rn(v.y, l), __fdiv_rn(v.z, l));
}
__device__ __forceinline__ float3 normalize_u(float3 v) {
    const float d = dot_u(v, v);
    if (!len2_inrange(d)) return normalize_u_generic(v);                          // never taken for sane geometry
    const RcpRn r = rcp_rn_prepare(sqrt_rn_inrange(d));
    return f3(div_rn_inrange(v.x, r), div_rn_inrange(v.y, r), div_rn_inrange(v.z, r));
}

// nrmTexel: the pixel's raw {N.xyz, roughness} texel in the shared-memory stage (still valid: the stage is released
// after the pixel is finished)
__device__ __noinline__ float exact_ndoth(float3 cam, float3 P, uint32_t nrmTexel, float3 wiSrc, float wiLenSq) {
    float4 nr;
    asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(nr.x), "=f"(nr.y), "=f"(nr.z), "=f"(nr.w) : "r"(nrmTexel));
    const float3 Ns = f3(nr.x, nr.y, nr.z);
    const float3 Vv = f3(__fsub_rn(cam.x, P.x), __fsub_rn(cam.y, P.y), __fsub_rn(cam.z, P.z));
    const float3 V = normalize_u(Vv);                 // ForwardLighting.hlsl:285
    const float3 Wo = normalize_u(V);                 // BRDF.hlsl:166
    const float3 N = normalize_u(Ns);                 // BRDF.hlsl:167
    float3 Wi;                                        // Lighting.hlsl:312: Lv / length(Lv)
    if (len2_inrange(wiLenSq)) {
        const RcpRn r = rcp_rn_prepare(sqrt_rn_inrange(wiLenSq));
        Wi = f3(div_rn_inrange(wiSrc.x, r), div_rn_inrange(wiSrc.y, r), div_rn_inrange(wiSrc.z, r));
    } else {
        const float w2 = __fsqrt_rn(wiLenSq);
        Wi = f3(__fdiv_rn(wiSrc.x, w2), __fdiv_rn(wiSrc.y, w2), __fdiv_rn(wiSrc.z, w2));
    }
    const float3 Hs = f3(__fadd_rn(Wo.x, Wi.x), __fadd_rn(Wo.y, Wi.y), __fadd_rn(Wo.z, Wi.z));
    const float3 H = normalize_u(Hs);                 // BRDF.hlsl:168
    return saturate(dot_u(N, H));
}

// ---- exact re-evaluation of N.V ---------------------------------------------------------------------
// `denom = max(4*NdotV*NdotL, 0.0001)` (BRDF.hlsl:186): once the clamp is active the specular term is PROPORTIONAL to NdotV
// (the G1(V) factor no longer cancels) with a gain of 1e4, and NdotV ~ 0 comes out of a cancellation: a 2e-7 difference in
// dot(N, Wo) is a 2e-3 difference in D*G*F/denom. Found by the full-frame parity test at 1920x1080 (4 pixels in 2 M, all with
// |N.V| < 5e-5, profiles/r02_diag_fullsize.txt). Grazing pixels therefore recompute N.V with the oracle's operation sequence.
constexpr float NV_EXACT = 1e-3f;
__device__ __noinline__ float exact_nv(float3 cam, float3 P, uint32_t nrmTexel) {
    float4 nr;
    asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(nr.x), "=f"(nr.y), "=f"(nr.z), "=f"(nr.w) : "r"(nrmTexel));
    const float3 Vv = f3(__fsub_rn(cam.x, P.x), __fsub_rn(cam.y, P.y), __fsub_rn(cam.z, P.z));
    const float3 Wo = normalize_u(normalize_u(Vv));                 // ForwardLighting.hlsl:285, BRDF.hlsl:166
    const float3 N = normalize_u(f3(nr.x, nr.y, nr.z));             // BRDF.hlsl:167
    return dot_u(N, Wo);
}

constexpr int FWD_THREADS = 128;
constexpr int FWD_TILE = 2 * FWD_THREADS;          // pixels per tile: 256 consecutive pixels of one row (4 KB per G-buffer plane)
constexpr uint32_t FWD_PLANE = FWD_TILE * 16u;     // bytes between the planes of one stage

// One light for the pixel pair: accumulates BRDF(s, Wi, V) * radiance * NdotL (BRDF.hlsl:163-194, Lighting.hlsl:308-345) in the
// factored form  r = K1*(1-fc) + omF0*(fc*spec) + F0*spec  with  F = F0 + (1-F0)*fc.
//   L, d2 : un-normalised light vector and its squared length (Wi = L/sqrt(d2)),  invD = 1/sqrt(d2)
//   scale : attenuation * brightness * spot intensity (0 when the light is out of range);  col : light colour
// H = normalize(V+Wi) is never formed: |V+Wi|^2 = 2+2c with c = V.Wi, so N.H = (N.V+N.Wi)*rh and
// H.V = (1+c)*rh with rh = rsqrt(2+2c).
// The body is branch-free (a light that does not contribute gets weight 0); only the rare exact-N.H slow path branches.
// TINY: the `denom < EPSILON -> D = 1` escape of NormalDistributionGGX (BRDF.hlsl:77) can only trigger when
// PI*(1+min(a2-1,0))^2 < 1e-12, i.e. roughness < 0.024: the caller picks the instantiation per warp, so ordinary
// materials never pay for the selects.
template <bool TINY>
__device__ __forceinline__ void shade_light2(const Px2& s, Acc2& acc, float3 cam, f2 Lx, f2 Ly, f2 Lz, f2 d2, f2 invD,
                                             f2 scale, float3 col) {
    const f2 nl = dot3(s.Nx, s.Ny, s.Nz, Lx, Ly, Lz) * invD;
    const f2 c = dot3(s.Vx, s.Vy, s.Vz, Lx, Ly, Lz) * invD;
    const f2 rh = rsq2(max2(fma2(bc(2.0f), c, bc(2.0f)), 1e-12f));
    f2 NdotH = mulsat2(s.nv + nl, rh);
    const f2 HV = mulsat2(bc(1.0f) + c, rh);              // (1+c)*rh = cos of the half angle: in [0,1] up to rounding
    const f2 omh = bc(1.0f) - HV;
    const f2 omh2 = omh * omh;
    const f2 fc = omh2 * omh2 * omh;                      // Fresnel_Schlick (BRDF.hlsl:132-136)
    f2 t = fma2(NdotH * NdotH, s.a2m1, bc(1.0f));         // NormalDistributionGGX (BRDF.hlsl:65-79)
    const f2 NL = sat2(nl);                               // saturate(N.L) == max(0,N.L) for unit vectors
    const f2 w = mulsat2(s.nsLen, nl) * scale;            // NdotL of the raw s.N (Lighting.hlsl:316) * radiance scale
    if (fminf(t.v.x, t.v.y) < T_EXACT) {                  // < 1 % of pixel-light pairs
        if (t.v.x < T_EXACT && w.v.x > 0.0f) {
            const float nh = exact_ndoth(cam, s.PA, s.texA + FWD_PLANE, f3(Lx.v.x, Ly.v.x, Lz.v.x), d2.v.x);
            t.v.x = __fadd_rn(__fmul_rn(__fmul_rn(nh, nh), s.a2m1.v.x), 1.0f);
        }
        if (t.v.y < T_EXACT && w.v.y > 0.0f) {
            const float nh = exact_ndoth(cam, s.PB, s.texB + FWD_PLANE, f3(Lx.v.y, Ly.v.y, Lz.v.y), d2.v.y);
            t.v.y = __fadd_rn(__fmul_rn(__fmul_rn(nh, nh), s.a2m1.v.y), 1.0f);
        }
    }
    f2 dDen = bc(PI) * (t * t);
    const f2 gDen = fma2(NL, s.omk, s.k4);                // Geometry_Smiths_SchlickGGX of L (BRDF.hlsl:82-97)
    const f2 sDen = max2(s.nv4 * NL, 0.0001f);            // max(4*NdotV*NdotL, 0.0001)
    f2 num;
    if (TINY) {                                           // `denom < EPSILON -> D = 1` (BRDF.hlsl:77)
        const bool ta = dDen.v.x < 0.000000000001f, tb = dDen.v.y < 0.000000000001f;
        num = mk(ta ? s.gV.v.x : s.a2gV.v.x, tb ? s.gV.v.y : s.a2gV.v.y) * NL;
        dDen = mk(ta ? 1.0f : dDen.v.x, tb ? 1.0f : dDen.v.y);
    } else {
        num = s.a2gV * NL;
    }
    const f2 spec = num * rcp2(dDen * gDen * sDen);       // D*G/denom with ONE reciprocal (den >= 1e-20)
    const f2 wa = (bc(1.0f) - fc) * w, wc = spec * w, wb = fc * wc;
    const f2 cr = bc(col.x), cg = bc(col.y), cb = bc(col.z);
    acc.ax = fma2(wa, cr, acc.ax); acc.ay = fma2(wa, cg, acc.ay); acc.az = fma2(wa, cb, acc.az);
    acc.bx = fma2(wb, cr, acc.bx); acc.by = fma2(wb, cg, acc.by); acc.bz = fma2(wb, cb, acc.bz);
    acc.cx = fma2(wc, cr, acc.cx); acc.cy = fma2(wc, cg, acc.cy); acc.cz = fma2(wc, cb, acc.cz);
}

// un-normalised light vector of a positional light and its squared length, |L-P|^2 exactly as the oracle's dot():
// (x*x + y*y) + z*z with every operation rounded
struct LightVec2 { f2 x, y, z, d2, invD; };
__device__ __forceinline__ LightVec2 light_vector2(const Px2& s, float3 pos) {
    LightVec2 L;
    // two scalar subtractions write straight into a register pair: cheaper than packing P once more per light
    L.x = mk(pos.x - s.PA.x, pos.x - s.PB.x); L.y = mk(pos.y - s.PA.y, pos.y - s.PB.y); L.z = mk(pos.z - s.PA.z, pos.z - s.PB.z);
    L.d2 = add_rn2(add_rn2(mul_rn2(L.x, L.x), mul_rn2(L.y, L.y)), mul_rn2(L.z, L.z));
    L.invD = rsq2(L.d2 + bc(1e-30f));                     // == rsqrt(d2) for every d2 >= 1e-22; finite at d2 = 0
    return L;
}

// SHADOWED: the shadow factor pair {pixel A, pixel B} of caster slot c = 1 - taps/n (Lighting.hlsl:162-164, :207-209), taps from the
// pixels' PCF records; a continuous factor of the light's weight, so one FFMA2 instead of the reference's division
__device__ __forceinline__ f2 shadow_factor2(const Px2& s, int slot, float invTaps) {
    const float ca = (float)((uint32_t)(s.recA >> (5 * slot)) & 31u), cb = (float)((uint32_t)(s.recB >> (5 * slot)) & 31u);
    return fma2(mk(ca, cb), bc(-invTaps), bc(1.0f));
}

// every light of the frame for one pixel pair, in PSMain's order
template <bool TINY, bool SHADOWED>
__device__ __forceinline__ void shade_all_lights(const Px2& s, Acc2& acc, const FwdParams& P) {
    const float3 cam = P.cam;
    const int numPoint = P.numPoint, numSpot = P.numSpot;
    // ---- point lights, then point casters (Lighting.hlsl:308-322; PSMain :310-313,321-340):
    //      in range <=> d2 < d2Limit (== length(Lw-P) < l.range, exactly) ----
    // one light at a time: interleaving two buys ILP for the dependent MUFU/FMA chains at ~20 more registers
#pragma unroll 1
    for (int i = 0; i < numPoint; ++i) {
        const SPoint l = P.pts[i];                                       // constant bank, warp-uniform index
        const LightVec2 L = light_vector2(s, l.pos);
        const f2 att = (L.invD * L.invD) * bc(l.brightness);               // AttenuationBRDF = 1/D^2
        f2 scale = mk(L.d2.v.x < l.d2Limit ? att.v.x : 0.0f, L.d2.v.y < l.d2Limit ? att.v.y : 0.0f);
        if (SHADOWED) {                                                   // OmnidirectionalShadowTestPCF: 20 taps
            const int c = i - (numPoint - P.shadow.nPointCasters);
            if (c >= 0) scale = scale * shadow_factor2(s, c, 1.0f / 20.0f);
        }
        shade_light2<TINY>(s, acc, cam, L.x, L.y, L.z, L.d2, L.invD, scale, l.color);
    }
    // ---- spot lights, then spot casters (Lighting.hlsl:57-73,323-333) ----
    for (int k = 0; k < numSpot; ++k) {
        const SSpot l = P.spots[k];
        const LightVec2 L = light_vector2(s, l.pos);
        const f2 cosT = dot3(L.x, L.y, L.z, bc(l.dir.x), bc(l.dir.y), bc(l.dir.z)) * L.invD;   // pixel direction = -Wi
        float inten[2];
#pragma unroll
        for (int q = 0; q < 2; ++q) {
            const float theta = acosf(fminf(fmaxf(-(q ? cosT.v.y : cosT.v.x), -1.0f), 1.0f));
            const float lin = 1.0f - (theta - l.inner) * l.invCone;
            inten[q] = theta > l.outer ? 0.0f : (theta <= l.inner ? 1.0f : lin);
        }
        f2 scale = mk(inten[0], inten[1]) * bc(l.brightness) * (L.invD * L.invD);
        if (SHADOWED) {                                                   // ShadowTestPCF: 5x5 taps
            const int c = k - (numSpot - P.shadow.nSpotCasters);
            if (c >= 0) scale = scale * shadow_factor2(s, P.shadow.nPointCasters + c, 1.0f / 25.0f);
        }
        shade_light2<TINY>(s, acc, cam, L.x, L.y, L.z, L.d2, L.invD, scale, l.color);
    }
    // ---- directional (PSMain :360-377; ShadowingFactor = 1 unless SHADOWED and the light casts) ----
    if (P.dirEnabled) {
        const SDir d = P.dir;
        f2 scale = bc(1.0f);
        if (SHADOWED) { if (P.shadow.dirSlot >= 0) scale = shadow_factor2(s, P.shadow.dirSlot, 1.0f / 25.0f); }
        shade_light2<TINY>(s, acc, cam, bc(d.wi.x), bc(d.wi.y), bc(d.wi.z), bc(1.0f), bc(1.0f), scale, d.radiance);
    }
}

// ---------------------------------------------------------------------------------------------
// TMA (bulk async copy) + mbarrier plumbing, raw PTX for sm_100a
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" :: "r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t done;
    do {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(done) : "r"(bar), "r"(parity) : "memory");
    } while (!done);
}
__device__ __forceinline__ void mbar_wait_backoff(uint32_t bar, uint32_t parity) {   // single-thread waits: do not steal issue slots
    uint32_t done;
    for (;;) {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(done) : "r"(bar), "r"(parity) : "memory");
        if (done) break;
        __nanosleep(128);
    }
}
__device__ __forceinline__ uint64_t l2_evict_first_policy() {
    uint64_t pol; asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol)); return pol;
}
// one contiguous row segment global -> shared through the TMA unit; completion is counted in bytes on `bar`
__device__ __forceinline__ void tma_load_row(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar, uint64_t pol) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;"
                 :: "r"(dst), "l"(src), "r"(bytes), "r"(bar), "l"(pol) : "memory");
}
__device__ __forceinline__ float4 lds128(uint32_t addr) {       // volatile: the load stays where it is written (register diet)
    float4 r;
    asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "r"(addr) : "memory");
    return r;
}
__device__ __forceinline__ float lds32(uint32_t addr) {
    float r; asm volatile("ld.shared.f32 %0, [%1];" : "=f"(r) : "r"(addr) : "memory"); return r;
}
__device__ __forceinline__ void st_stream_hint(float4* p, float4 v, uint64_t pol) {
    asm volatile("st.global.L1::no_allocate.L2::cache_hint.v4.f32 [%0], {%1,%2,%3,%4}, %5;"
                 :: "l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w), "l"(pol) : "memory");
}

// K1 is a persistent kernel: FWD_CTAS_PER_SM CTAs of 128 threads per SM, each walking the tile list
// (tile = 256 consecutive pixels of one row = one 4 KB row segment per G-buffer plane; two pixels per thread) with stride
// gridDim.y over the rows. The G-buffer arrives through a FWD_STAGES-deep TMA pipeline in shared memory: thread 0 issues one bulk
// copy per plane for the tile FWD_AHEAD iterations ahead (full[] mbarriers count the bytes), every thread reads
// ITS texels back with LDS when it needs them and releases the stage (empty[] mbarriers) when its pixels are
// stored. Nothing of the G-buffer is live in registers across the light loop: albedo/metalness/ao, the raw
// normal and the emissive texel are (re-)read from the stage after it.
constexpr int FWD_STAGES = 2;          // shared-memory stages
constexpr int FWD_AHEAD = 1;           // tiles requested ahead of the one being shaded (< FWD_STAGES)
constexpr int FWD_CTAS_PER_SM = 4;
static_assert(FWD_AHEAD >= 1 && FWD_AHEAD < FWD_STAGES, "the lookahead must leave at least one stage for the tile being shaded");

// ---- environment taps -----------------------------------------------------------------------------------
// per (mip, face) constants of the specular sampling copy, staged once per CTA: one LDS.128 replaces the shifts, the
// int->float conversions and the mipOffset[] constant-bank indexing of a per-pixel mip
struct FaceRec { uint32_t base; uint32_t P; float halfN; float c0; };     // first record of the face, row stride, N/2, N/2 - 0.5
static_assert(sizeof(FaceRec) == 16, "one LDS.128");

// L1 policy of a gather (A/B on B200): the diffuse cube's gathers allocate in L1, the specular cube's and the LUT's do not
template <bool NO_ALLOCATE>
__device__ __forceinline__ F8 ldg256(const float4* p) {             // 32-byte aligned, read-only path (LDG.E.256)
    F8 r;
    if (NO_ALLOCATE)
        asm("ld.global.nc.L1::no_allocate.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
            : "=f"(r.a.x), "=f"(r.a.y), "=f"(r.a.z), "=f"(r.a.w), "=f"(r.b.x), "=f"(r.b.y), "=f"(r.b.z), "=f"(r.b.w) : "l"(p));
    else
        asm("ld.global.nc.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
            : "=f"(r.a.x), "=f"(r.a.y), "=f"(r.a.z), "=f"(r.a.w), "=f"(r.b.x), "=f"(r.b.y), "=f"(r.b.z), "=f"(r.b.w) : "l"(p));
    return r;
}
// A/B on B200 (profiles/r02_forward_variants_b.txt): a lane-pair variant — column-major records so that the two rows of a footprint
// are adjacent, lanes 2q/2q+1 fetching one footprint together and swapping halves with shuffles — touches fewer 128-byte lines per
// instruction (tools/ubench_gather.cu: 16 lines cost 20 L1 wavefronts, 32 cost 33) but measured 268 us against 258 us for this
// form: the five shuffles per footprint and the lost line sharing between neighbouring lanes (row-major records of neighbouring
// pixels share lines) cost more than the pairing saves.
struct CubeLoad { F8 r0, r1; float fx, fy; };                     // rows j0 and j0+1: {t(i0), t(i0+1)} each
// A gather is split into "issue" (address + the 256-bit loads) and "finish" (the lerps) so that the loads of several
// gathers are in flight before the first one is consumed.
// maxRec: last record a footprint may start at (clamps the address for NaN/inf directions: no surface => no normal)
template <bool NO_ALLOCATE>
__device__ __forceinline__ CubeLoad cube_issue(const float4* __restrict__ recs, FaceRec f, uint32_t maxRec, float sx, float sy) {
    const float x = fmaf(sx, f.halfN, f.c0), y = fmaf(-sy, f.halfN, f.c0);       // texel space: (s*0.5+0.5)*N - 0.5
    const float xf = floorf(x), yf = floorf(y);                                  // in [-1, N-1] for every finite direction
    CubeLoad L;
    L.fx = x - xf; L.fy = y - yf;
    const uint32_t off = min(f.base + (uint32_t)((int)yf + 1) * f.P + (uint32_t)((int)xf + 1), maxRec);
    const float4* p = recs + 2u * off;
    L.r0 = ldg256<NO_ALLOCATE>(p); L.r1 = ldg256<NO_ALLOCATE>(p + 2u * f.P);
    return L;
}
// bilinear blend of the footprint as packed pairs {x,y}, {z,w} of one pixel: 12 packed operations instead of 18 scalar ones
__device__ __forceinline__ float3 cube_finish(const CubeLoad& L) {
    const f2 fx = bc(L.fx), fy = bc(L.fy);
    const f2 a0 = mk(L.r0.a.x, L.r0.a.y), a1 = mk(L.r0.a.z, L.r0.a.w), b0 = mk(L.r0.b.x, L.r0.b.y), b1 = mk(L.r0.b.z, L.r0.b.w);
    const f2 c0 = mk(L.r1.a.x, L.r1.a.y), c1 = mk(L.r1.a.z, L.r1.a.w), d0 = mk(L.r1.b.x, L.r1.b.y), d1 = mk(L.r1.b.z, L.r1.b.w);
    const f2 t0 = fma2(fx, b0 - a0, a0), t1 = fma2(fx, b1 - a1, a1);
    const f2 u0 = fma2(fx, d0 - c0, c0), u1 = fma2(fx, d1 - c1, c1);
    const f2 r0 = fma2(fy, u0 - t0, t0), r1 = fma2(fy, u1 - t1, t1);
    return f3(r0.v.x, r0.v.y, r1.v.x);
}
struct LutLoad { F8 q; float fx, fy; };
__device__ __forceinline__ LutLoad lut_issue(const LutV& l, float u, float v) {   // bilinear, CLAMP
    const float x = fmaf(u, (float)l.w, -0.5f), y = fmaf(v, (float)l.h, -0.5f);
    const float x0 = floorf(x), y0 = floorf(y);
    LutLoad L;
    L.fx = x - x0; L.fy = y - y0;
    const int cx = min(max((int)x0 + 1, 0), l.w), cy = min(max((int)y0 + 1, 0), l.h);
    L.q = ldg256<true>(l.q + 2u * (uint32_t)(cy * (l.w + 1) + cx));
    return L;
}
__device__ __forceinline__ float2 lut_finish(const LutLoad& L) {    // record = {p00, p10 | p01, p11} as float2 each
    const f2 fx = bc(L.fx), fy = bc(L.fy);
    const f2 p00 = mk(L.q.a.x, L.q.a.y), p10 = mk(L.q.a.z, L.q.a.w), p01 = mk(L.q.b.x, L.q.b.y), p11 = mk(L.q.b.z, L.q.b.w);
    const f2 t = fma2(fx, p10 - p00, p00), u = fma2(fx, p11 - p01, p01);
    return fma2(fy, u - t, t).v;
}

// the environment lookups and the final composition of ONE pixel (PSMain :290-293, Lighting.hlsl:360-395, BRDF.hlsl:177-207)
//   texel : shared-memory address of the pixel's position texel,  V/nsnv : normalize(cam-P), saturate(dot(s.N, V))
//   la/lb/lc : the light sums  sum w*col*{(1-fc), fc*spec, spec}
//   Ns : the surface normal as normalize(Ns)*|Ns| (within an ulp of the raw texel; it only steers the two cube lookups)
// The environment lookups of one pixel, split into "issue" (the five 256-bit gathers: diffuse cube x2, specular cube x2, LUT, with
// their bilinear weights) and "compose" (the blends + the final composition), so that the kernel can put BOTH pixels' gathers in
// flight before it consumes either: a thread then waits for the L2/HBM latency once per pair instead of once per
// pixel (ncu: a third of all stall samples sit on the first use of pixel A's taps and again on pixel B's). Ten 256-bit loads in
// flight need ~160 registers, i.e. three CTAs per SM instead of four: A/B in profiles/r02_forward_variants_e.txt.
struct EnvLoads { CubeLoad D, S; LutLoad L; };
template <bool ROT, bool SPEC>
__device__ __forceinline__ void env_issue(EnvLoads& E, const FwdParams& P, const FaceRec* __restrict__ sFace, float3 V, float nsnv, float3 Ns, float roughness) {
    const float3 Nr = ROT ? f3(Ns.x * P.cosB - Ns.z * P.sinB, Ns.y, Ns.x * P.sinB + Ns.z * P.cosB) : Ns;
    int face; float sx, sy;
    dir_to_face(Nr, face, sx, sy);
    FaceRec fd; fd.P = (uint32_t)P.diff.res + 2u; fd.base = (uint32_t)face * fd.P * fd.P; fd.halfN = P.diffHalfN; fd.c0 = P.diffHalfN - 0.5f;
    E.D = cube_issue<false>(P.diff.p, fd, P.diffMaxRec, sx, sy);
    if (SPEC) {
        const float3 R0 = reflect(-V, Ns);
        const float3 R = ROT ? f3(R0.x * P.cosB - R0.z * P.sinB, R0.y, R0.x * P.sinB + R0.z * P.cosB) : R0;
        dir_to_face(R, face, sx, sy);
        const int mip = min(max((int)(roughness * (float)P.maxLod), 0), P.spec.mips - 1);
        E.S = cube_issue<true>(P.spec.p, sFace[face * 16 + mip], P.specMaxRec, sx, sy);
        E.L = lut_issue(P.lut, nsnv, roughness);                                 // (saturate(dot(s.N, V)), roughness)
    }
}
// the final composition of the pixel (PSMain :290-293, Lighting.hlsl:360-395, BRDF.hlsl:177-207)
//   texel : shared-memory address of the pixel's position texel,  nsnv : saturate(dot(s.N, V))
//   la/lb/lc : the light sums  sum w*col*{(1-fc), fc*spec, spec}
__device__ __forceinline__ float4 compose_values(const FwdParams& P, uint32_t texel, float nsnv, float roughness, float ao,
                                                 float3 la, float3 lb, float3 lc, float3 diffIrr, float3 specCol, float2 sb) {
    // ---- the rest of the G-buffer texel comes out of the stage only now ----
    const float4 am = lds128(texel + 2u * FWD_PLANE);
    const float3 albedo = xyz(am);
    const float metalness = am.w;
    float3 I = albedo * ao;                                  // ForwardLighting.hlsl:290-293 (the ambient factor rides in position.w)
    if (P.hasEmissive) {
        const float4 em = lds128(texel + 3u * FWD_PLANE);
        I += xyz(em) * em.w;
    }
    const float3 F0 = lerp(f3(0.04f), albedo, metalness);    // BRDF.hlsl:177
    {   // K1 = (1-F0)*(1-metal)*albedo/PI (BRDF.hlsl:189-191)
        const float3 omF0 = f3(1.0f) - F0;
        const float3 K1 = omF0 * albedo * ((1.0f - metalness) * (1.0f / PI));
        I.x += fmaf(K1.x, la.x, fmaf(omF0.x, lb.x, F0.x * lc.x));
        I.y += fmaf(K1.y, la.y, fmaf(omF0.y, lb.y, F0.y * lc.y));
        I.z += fmaf(K1.z, la.z, fmaf(omF0.z, lb.z, F0.z * lc.z));
    }
    {   // ---- EnvironmentBRDF (BRDF.hlsl:196-207) on the gathered taps ----
        const float fr = pow5(1.0f - nsnv);                      // FresnelWithRoughness(saturate(dot(s.N, V))), BRDF.hlsl:152-156
        const float omr = 1.0f - roughness;
        const float3 Ks = f3(fmaf(fmaxf(omr, F0.x) - F0.x, fr, F0.x),
                             fmaf(fmaxf(omr, F0.y) - F0.y, fr, F0.y),
                             fmaf(fmaxf(omr, F0.z) - F0.z, fr, F0.z));
        const float om = 1.0f - metalness;
        I.x += (1.0f - Ks.x) * om * (diffIrr.x * albedo.x) + specCol.x * fmaf(Ks.x, sb.x, sb.y);
        I.y += (1.0f - Ks.y) * om * (diffIrr.y * albedo.y) + specCol.y * fmaf(Ks.y, sb.x, sb.y);
        I.z += (1.0f - Ks.z) * om * (diffIrr.z * albedo.z) + specCol.z * fmaf(Ks.z, sb.x, sb.y);
    }
    return make_float4(I.x, I.y, I.z, roughness);                // :380
}
template <bool SPEC>
__device__ __forceinline__ float4 compose_pixel(const FwdParams& P, uint32_t texel, float nsnv, float roughness, float ao,
                                                float3 la, float3 lb, float3 lc, const EnvLoads& E) {
    float3 specCol = f3(0.0f); float2 sb = make_float2(0.0f, 0.0f);
    if (SPEC) { specCol = cube_finish(E.S); sb = lut_finish(E.L); }
    const float3 diffIrr = cube_finish(E.D);
    return compose_values(P, texel, nsnv, roughness, ao, la, lb, lc, diffIrr, specCol, sb);
}

// everything after the light loop for the pixel pair: environment taps, composition, stores
template <bool MULTI, bool ROT, bool SPEC>
__device__ __forceinline__ void finish_pair(const FwdParams& P, const FaceRec* __restrict__ sFace, const Px2& s, const Acc2& acc, f2 roughness, f2 ao,
                                            int y, int xA, int xB, bool validA, bool validB) {
    const f2 nsnv = mulsat2(s.nsLen, s.nv);                      // saturate(dot(s.N, V)) of the raw normal
    const f2 Nrx = s.Nx * s.nsLen, Nry = s.Ny * s.nsLen, Nrz = s.Nz * s.nsLen;
    EnvLoads eA, eB;
    env_issue<ROT, SPEC>(eA, P, sFace, f3(s.Vx.v.x, s.Vy.v.x, s.Vz.v.x), nsnv.v.x, f3(Nrx.v.x, Nry.v.x, Nrz.v.x), roughness.v.x);
    env_issue<ROT, SPEC>(eB, P, sFace, f3(s.Vx.v.y, s.Vy.v.y, s.Vz.v.y), nsnv.v.y, f3(Nrx.v.y, Nry.v.y, Nrz.v.y), roughness.v.y);
    const float4 oA = compose_pixel<SPEC>(P, s.texA, nsnv.v.x, roughness.v.x, ao.v.x, f3(acc.ax.v.x, acc.ay.v.x, acc.az.v.x),
                                          f3(acc.bx.v.x, acc.by.v.x, acc.bz.v.x), f3(acc.cx.v.x, acc.cy.v.x, acc.cz.v.x), eA);
    if (validA) {   // one STG.128 per destination; peer destinations are mapped NVLink addresses (fused compute + gather)
        if (MULTI) { for (int q = 0; q < P.nOut; ++q) st_stream(P.outs[q].row(P.dstRowOffset + y) + xA, oA); }
        else st_stream_hint(P.outs[0].row(P.dstRowOffset + y) + xA, oA, l2_evict_first_policy());
    }
    const float4 oB = compose_pixel<SPEC>(P, s.texB, nsnv.v.y, roughness.v.y, ao.v.y, f3(acc.ax.v.y, acc.ay.v.y, acc.az.v.y),
                                          f3(acc.bx.v.y, acc.by.v.y, acc.bz.v.y), f3(acc.cx.v.y, acc.cy.v.y, acc.cz.v.y), eB);
    if (validB) {
        if (MULTI) { for (int q = 0; q < P.nOut; ++q) st_stream(P.outs[q].row(P.dstRowOffset + y) + xB, oB); }
        else st_stream_hint(P.outs[0].row(P.dstRowOffset + y) + xB, oB, l2_evict_first_policy());
    }
}

// per-pixel-pair set-up (everything the lights share) and the light loops: fills s, acc, roughness, ao from the staged texels
template <bool SHADOWED>
__device__ __forceinline__ void shade_pair_lights(const FwdParams& P, Px2& s, Acc2& acc, f2& roughness, f2& ao) {
    {
        const float4 pa = lds128(s.texA), pb = lds128(s.texB);
        ao = mk(pa.w, pb.w);
        const float4 na = lds128(s.texA + FWD_PLANE), nb = lds128(s.texB + FWD_PLANE);
        s.PA = xyz(pa); s.PB = xyz(pb);
        const f2 Nsx = mk(na.x, nb.x), Nsy = mk(na.y, nb.y), Nsz = mk(na.z, nb.z);
        roughness = mk(na.w, nb.w);
        const f2 Vx = mk(P.cam.x - pa.x, P.cam.x - pb.x), Vy = mk(P.cam.y - pa.y, P.cam.y - pb.y), Vz = mk(P.cam.z - pa.z, P.cam.z - pb.z);
        const f2 rv = rsq2(dot3(Vx, Vy, Vz, Vx, Vy, Vz));
        s.Vx = Vx * rv; s.Vy = Vy * rv; s.Vz = Vz * rv;          // ForwardLighting.hlsl:285
        const f2 n2 = dot3(Nsx, Nsy, Nsz, Nsx, Nsy, Nsz), rn = rsq2(n2);
        s.Nx = Nsx * rn; s.Ny = Nsy * rn; s.Nz = Nsz * rn;       // BRDF.hlsl:167
        s.nsLen = n2 * rn;
    }
    const f2 a = roughness * roughness;
    const f2 a2 = mul_rn2(a, a);
    s.a2m1 = add_rn2(a2, bc(-1.0f));                             // no contraction: feeds the exact t
    const f2 rp1 = roughness + bc(1.0f);
    const f2 k = (rp1 * rp1) * bc(0.125f);
    s.omk = bc(1.0f) - k; s.k4 = k + bc(0.0001f);
    s.nv = dot3(s.Nx, s.Ny, s.Nz, s.Vx, s.Vy, s.Vz);
    if (fminf(fabsf(s.nv.v.x), fabsf(s.nv.v.y)) < NV_EXACT) {     // grazing view: ~0.1 % of pixels
        if (fabsf(s.nv.v.x) < NV_EXACT) s.nv.v.x = exact_nv(P.cam, s.PA, s.texA + FWD_PLANE);
        if (fabsf(s.nv.v.y) < NV_EXACT) s.nv.v.y = exact_nv(P.cam, s.PB, s.texB + FWD_PLANE);
    }
    const f2 NdotV = sat2(s.nv);
    s.gV = NdotV * rcp2(fma2(NdotV, s.omk, s.k4));
    s.a2gV = a2 * s.gV;
    s.nv4 = NdotV * bc(4.0f);

    acc.ax = acc.ay = acc.az = acc.bx = acc.by = acc.bz = acc.cx = acc.cy = acc.cz = bc(0.0f);
    // can `PI*t*t < 1e-12` ever hold for one of this warp's pixels?  t >= 1 + min(a2-1, 0), rounding is monotone
    const f2 tmin = bc(1.0f) + mk(fminf(s.a2m1.v.x, 0.0f), fminf(s.a2m1.v.y, 0.0f));
    const f2 dmin = bc(PI) * (tmin * tmin);
    if (__any_sync(0xffffffffu, fminf(dmin.v.x, dmin.v.y) < 2e-12f))
        shade_all_lights<true, SHADOWED>(s, acc, P);
    else
        shade_all_lights<false, SHADOWED>(s, acc, P);
}

template <bool MULTI, bool ROT, bool SHADOWED = false>
__global__ void __launch_bounds__(FWD_THREADS, FWD_CTAS_PER_SM) forward_kernel(const __grid_constant__ FwdParams P) {
    extern __shared__ __align__(128) unsigned char smemRaw[];
    const int nPl = P.hasEmissive ? 4 : 3;
    const int tid = threadIdx.x;
    // shared-memory layout: [FWD_STAGES][nPl][FWD_TILE] float4 | full[S], empty[S] mbarriers | FaceRec[8*16]
    const uint32_t stageBytes = (uint32_t)nPl * FWD_PLANE;
    uint64_t* bars = (uint64_t*)(smemRaw + FWD_STAGES * stageBytes);
    FaceRec* sFace = (FaceRec*)(bars + 2 * FWD_STAGES);
    const uint32_t stage0 = smem_u32(smemRaw), bar0 = smem_u32(bars);
    auto fullBar = [&](int st) { return bar0 + 8u * (uint32_t)st; };
    auto emptyBar = [&](int st) { return bar0 + 8u * (uint32_t)(FWD_STAGES + st); };

    // ---- tile schedule: the grid is (tiles per row) x (row groups); a CTA keeps its column and strides rows, so the
    //      only loop state is the row, the stage index and the stage's use count ----
    const int x0 = (int)blockIdx.x * FWD_TILE;
    const int rowStep = (int)gridDim.y;
    const uint32_t tileBytes = (uint32_t)min(FWD_TILE, P.width - x0) * 16u;
    // thread 0: request the tile of row `r` into stage `sIdx`, which has been used `useCount` times before
    auto request = [&](int r, int sIdx, uint32_t useCount) {
        if (r >= P.rows) return;
        if (useCount > 0) mbar_wait_backoff(emptyBar(sIdx), (useCount - 1u) & 1u);   // every thread is done with the previous use
        const uint64_t pol = l2_evict_first_policy();                 // the G-buffer is touched once: first out of L2
        const uint32_t dst = stage0 + (uint32_t)sIdx * stageBytes, bar = fullBar(sIdx);
        const size_t y = (size_t)(P.rowBegin + r);
        mbar_expect_tx(bar, tileBytes * (uint32_t)nPl);
        tma_load_row(dst, P.pos.p + y * P.pos.pitch4 + x0, tileBytes, bar, pol);
        tma_load_row(dst + FWD_PLANE, P.nrm.p + y * P.nrm.pitch4 + x0, tileBytes, bar, pol);
        tma_load_row(dst + 2u * FWD_PLANE, P.alb.p + y * P.alb.pitch4 + x0, tileBytes, bar, pol);
        if (nPl == 4) tma_load_row(dst + 3u * FWD_PLANE, P.emi.p + y * P.emi.pitch4 + x0, tileBytes, bar, pol);
    };
    if (tid == 0) {
        for (int s = 0; s < FWD_STAGES; ++s) { mbar_init(fullBar(s), 1u); mbar_init(emptyBar(s), (uint32_t)FWD_THREADS); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        for (int s = 0; s < FWD_AHEAD; ++s) request((int)blockIdx.y + s * rowStep, s, 0u);   // prologue: FWD_AHEAD tiles in flight
    }

    // ---- stage the specular cube's face table, once per CTA ----
    for (int i = tid; i < 16 * 8; i += FWD_THREADS) {
        // index = face*16 + mip: the lanes of a warp mostly share the face and differ in the mip (per-pixel roughness), so the
        // entries they read are ADJACENT 16-byte words in different banks (mip*8+face measured 19 wavefronts per LDS.128, ideal 4)
        const int mip = i & 15, face = i >> 4;
        FaceRec f; f.base = 0u; f.P = 3u; f.halfN = 0.5f; f.c0 = 0.0f;
        if (!P.diffuseOnly && mip < P.spec.mips && face < 6) {
            const int N = P.spec.res >> mip;
            f.P = (uint32_t)N + 2u; f.base = P.spec.mipOffset[mip] + (uint32_t)face * f.P * f.P;
            f.halfN = 0.5f * (float)N; f.c0 = f.halfN - 0.5f;
        }
        sFace[i] = f;
    }
    __syncthreads();                                              // face table staged, mbarriers initialised

    int st = 0; uint32_t use = 0;                                 // stage of the current tile, completed uses of that stage
    const int xA = x0 + tid, xB = xA + FWD_THREADS;
    const bool validA = xA < P.width, validB = xB < P.width;      // a ragged last tile: B (or both) fall off the row
    for (int row = (int)blockIdx.y; row < P.rows; row += rowStep) {
        if (tid == 0) {                                           // request the tile FWD_AHEAD iterations ahead
            const int ps = st + FWD_AHEAD;
            if (ps < FWD_STAGES) request(row + FWD_AHEAD * rowStep, ps, use);
            else request(row + FWD_AHEAD * rowStep, ps - FWD_STAGES, use + 1u);
        }
        mbar_wait(fullBar(st), use & 1u);                         // this tile has landed
        const int y = P.rowBegin + row;
        {   // every lane shades (the warp votes below need whole warps): pixels off the end of a ragged row are aliased to the
            // row's last pixel and simply not stored
            Px2 s;
            const uint32_t stageBase = stage0 + (uint32_t)st * stageBytes;
            s.texA = stageBase + (uint32_t)(min(xA, P.width - 1) - x0) * 16u;
            s.texB = stageBase + (uint32_t)(min(xB, P.width - 1) - x0) * 16u;
            f2 roughness, ao;
            Acc2 acc;
            if (SHADOWED) {                                       // the pair's PCF records: two coalesced 8-byte loads, consumed in the light loop
                const uint2* rr = P.shadow.p + (size_t)row * P.shadow.pitch;
                const uint2 ra = __ldg(rr + min(xA, P.width - 1)), rb = __ldg(rr + min(xB, P.width - 1));
                s.recA = ((uint64_t)ra.y << 32) | ra.x; s.recB = ((uint64_t)rb.y << 32) | rb.x;
            }
            shade_pair_lights<SHADOWED>(P, s, acc, roughness, ao);
            if (P.diffuseOnly) finish_pair<MULTI, ROT, false>(P, sFace, s, acc, roughness, ao, y, xA, xB, validA, validB);
            else finish_pair<MULTI, ROT, true>(P, sFace, s, acc, roughness, ao, y, xA, xB, validA, validB);
        }
        mbar_arrive(emptyBar(st));                               // this thread is done with the stage
        if (++st == FWD_STAGES) { st = 0; ++use; }
    }
    if (MULTI && P.sync.n > 1) {       // fused gather: the last CTA to retire signals the peers and waits for theirs (one kernel = one step)
        __threadfence_system();        // this CTA's peer stores are ordered before its retirement
        __syncthreads();
        if (tid == 0) {
            const uint32_t done = atomicAdd(P.ticket, 1u);
            if (done == gridDim.x * gridDim.y - 1u) {
                *P.ticket = 0u;
                __threadfence_system();
                peer_rendezvous(P.sync);
            }
        }
    }
}

uint64_t padded_texels(int res, int mips) {
    uint64_t n = 0;
    for (int m = 0; m < mips; ++m) { const uint64_t p = (uint64_t)(res >> m) + 2; n += 6 * p * p; }
    return n;
}
// bytes of a sampling copy: the records plus one mip-0 row of slack, so that a footprint whose first record was clamped to
// the last record (a non-finite direction: pixels without a surface carry a zero normal) still reads inside the allocation
size_t padded_bytes(int res, int mips) { return (size_t)(padded_texels(res, mips) + (uint64_t)res + 3u) * 32u; }
bool cube_desc_ok(const VqCubemap& c) {
    return c.ptr && c.res >= 1 && c.mips >= 1 && c.mips <= 16 && (c.res >> (c.mips - 1)) >= 1 &&
           padded_texels(c.res, c.mips) < (1ull << 30);
}
// builds the sampling copy of `c` into `dst` (padded_texels() records of 32 bytes) on `stream`
int pad_cube(const VqCubemap& c, float4* dst, cudaStream_t stream) {
    const uint32_t total = (uint32_t)padded_texels(c.res, c.mips);
    unsigned blocks = (total + 255u) / 256u;
    if (blocks > 148u * 16u) blocks = 148u * 16u;
    cube_pad_kernel<<<blocks, 256, 0, stream>>>((const float4*)c.ptr, dst, c.res, c.mips, total);
    return vq_check_launch("cube_pad");
}
void fill_cube_view(const VqCubemap& c, const float4* padded, CubeV& v) {
    v.p = padded; v.res = c.res; v.mips = c.mips;
    uint32_t off = 0;
    for (int m = 0; m < 16; ++m) {
        v.mipOffset[m] = m < c.mips ? off : 0u;
        if (m < c.mips) { const uint32_t p = (uint32_t)(c.res >> m) + 2u; off += 6u * p * p; }
    }
}
bool same_cube(const VqCubemap& a, const VqCubemap& b) { return a.ptr == b.ptr && a.res == b.res && a.mips == b.mips; }
bool same_image(const VqImage& a, const VqImage& b) { return a.ptr == b.ptr && a.width == b.width && a.height == b.height && a.pitch_bytes == b.pitch_bytes; }
size_t lut_footprint_bytes(const VqImage& lut) { return (size_t)(lut.width + 1) * (size_t)(lut.height + 1) * 32; }
// builds the footprint copy of the BRDF LUT into `dst` on `stream`
int footprint_lut(const VqImage& lut, float4* dst, cudaStream_t stream) {
    const uint32_t total = (uint32_t)(lut.width + 1) * (uint32_t)(lut.height + 1);
    unsigned blocks = (total + 255u) / 256u;
    if (blocks > 148u * 16u) blocks = 148u * 16u;
    lut_footprint_kernel<<<blocks, 256, 0, stream>>>((const float2*)lut.ptr, (int)(lut.pitch_bytes / 8), lut.width, lut.height, dst);
    return vq_check_launch("lut_footprint");
}

int ensure_bytes(void** ptr, size_t* have, size_t need) {
    if (*have >= need && *ptr) return VQ_OK;
    if (*ptr) cudaFree(*ptr);
    *ptr = nullptr; *have = 0;
    if (cudaMalloc(ptr, need) != cudaSuccess) { cudaGetLastError(); vq_set_error("cudaMalloc(%zu) failed", need); return VQ_ERR_OUT_OF_MEMORY; }
    *have = need;
    return VQ_OK;
}

}  // namespace

// Scene::GatherLightData's arrays -> what the kernel reads per light, on the host in IEEE fp32 (every operation rounded on its
// own: the same bits the oracle's normalize() / length() produce):
//   point: smallest d2 with sqrt_rn(d2) >= range, so that (d2 < limit) == (sqrt_rn(d2) < range) exactly  (Lighting.hlsl:308-322)
//   spot : normalize(l.spotDir) (Lighting.hlsl:60), 1/(outer - inner);  directional: Wi = normalize(-dir), radiance = color*brightness
static void normalize_host(const float v[3], float out[3]) {
    volatile float xx = v[0] * v[0], yy = v[1] * v[1], zz = v[2] * v[2];
    volatile float s = xx + yy; s = s + zz;
    const float l = sqrtf(s);
    out[0] = v[0] / l; out[1] = v[1] / l; out[2] = v[2] / l;
}
static void condition_lights(const VqSceneLighting& L, FwdParams& P) {
    const int nP = L.numPointLights, nPC = L.numPointCasters, nS = L.numSpotLights, nSC = L.numSpotCasters;
    P.numPoint = nP + nPC; P.numSpot = nS + nSC;
    for (int i = 0; i < P.numPoint; ++i) {
        const VqPointLight& l = i < nP ? L.point_lights[i] : L.point_casters[i - nP];
        SPoint& s = P.pts[i];
        s.pos = make_float3(l.position.x, l.position.y, l.position.z);
        s.color = make_float3(l.color.x, l.color.y, l.color.z);
        s.brightness = l.brightness;
        volatile float lim = l.range * l.range;
        if (!(l.range > 0.0f)) lim = 0.0f;
        else {
            auto bits = [](float f) { uint32_t u; memcpy(&u, &f, 4); return u; };
            auto flt = [](uint32_t u) { float f; memcpy(&f, &u, 4); return f; };
            while (sqrtf(lim) >= l.range && lim > 0.0f) lim = flt(bits(lim) - 1u);
            while (sqrtf(lim) < l.range) lim = flt(bits(lim) + 1u);
        }
        s.d2Limit = lim;
    }
    for (int i = 0; i < P.numSpot; ++i) {
        const VqSpotLight& l = i < nS ? L.spot_lights[i] : L.spot_casters[i - nS];
        SSpot& s = P.spots[i];
        s.pos = make_float3(l.position.x, l.position.y, l.position.z);
        s.color = make_float3(l.color.x, l.color.y, l.color.z);
        s.brightness = l.brightness;
        const float d[3] = {l.spotDir.x, l.spotDir.y, l.spotDir.z};
        float n[3]; normalize_host(d, n);
        s.dir = make_float3(n[0], n[1], n[2]);
        s.outer = l.outerConeAngle; s.inner = l.innerConeAngle;
        s.invCone = 1.0f / (l.outerConeAngle - l.innerConeAngle);
    }
    P.dirEnabled = L.directional.enabled != 0;
    if (P.dirEnabled) {
        const float d[3] = {-L.directional.lightDirection.x, -L.directional.lightDirection.y, -L.directional.lightDirection.z};
        float n[3]; normalize_host(d, n);
        P.dir.wi = make_float3(n[0], n[1], n[2]);
        P.dir.radiance = make_float3(L.directional.color.x * L.directional.brightness, L.directional.color.y * L.directional.brightness,
                                     L.directional.color.z * L.directional.brightness);
    }
}

int vq_forward_launch_multi(VqContext* ctx, const VqPerFrameData* pf, const VqPerViewLightingData* pv,
                            const VqGBuffer* gb, const VqEnvironmentMaps* env, const VqImage* outs, int n_outs,
                            int dst_row_offset, int row_begin, int row_end, const VqPeerSignal* sig, cudaStream_t stream,
                            const ShadowRecV* shadow = nullptr) {
    VQ_REQUIRE(pf && pv && gb && env && outs, "null parameter block");
    VQ_REQUIRE(n_outs >= 1 && n_outs <= 8, "1..8 destinations");
    VQ_REQUIRE(vq_image_ok(gb->position_ao) && vq_image_ok(gb->normal_roughness) && vq_image_ok(gb->albedo_metalness), "bad image descriptor");
    const int W = gb->position_ao.width, H = gb->position_ao.height;
    VQ_REQUIRE(gb->normal_roughness.width == W && gb->albedo_metalness.width == W &&
               gb->normal_roughness.height == H && gb->albedo_metalness.height == H, "G-buffer planes must have the same size");
    VQ_REQUIRE(dst_row_offset >= 0, "negative destination row offset");
    for (int k = 0; k < n_outs; ++k)
        VQ_REQUIRE(vq_image_ok(outs[k]) && outs[k].width == W && outs[k].height >= dst_row_offset + H,
                   "every destination must be as wide as the G-buffer and hold dst_row_offset + height rows");
    VQ_REQUIRE(row_begin >= 0 && row_end <= H && row_begin <= row_end, "row range out of bounds");
    const VqSceneLighting& L = pf->Lights;
    VQ_REQUIRE(L.numPointLights >= 0 && L.numPointLights <= VQ_NUM_LIGHTS_POINT &&
               L.numSpotLights >= 0 && L.numSpotLights <= VQ_NUM_LIGHTS_SPOT &&
               L.numPointCasters >= 0 && L.numPointCasters <= VQ_NUM_SHADOWING_LIGHTS_POINT &&
               L.numSpotCasters >= 0 && L.numSpotCasters <= VQ_NUM_SHADOWING_LIGHTS_SPOT, "light counts exceed the cbuffer arrays");
    VQ_REQUIRE(row_begin < row_end || !(sig && sig->n_ranks > 1), "a rendezvous needs a non-empty row range (the kernel runs it)");
    if (row_begin == row_end) return VQ_OK;
    VqScratchLock lock(ctx);           // env_* registration and the per-call tmp_* sampling copies are the context's

    FwdParams P;
    memset(&P, 0, sizeof(P));
    condition_lights(L, P);
    P.cam = make_float3(pv->CameraPosition.x, pv->CameraPosition.y, pv->CameraPosition.z);
    P.cosB = cosf(-pf->fHDRIOffsetInRadians);
    P.sinB = sinf(-pf->fHDRIOffsetInRadians);
    P.maxLod = (int)pv->MaxEnvMapLODLevels;
    P.diffuseOnly = pv->EnvironmentMapDiffuseOnlyIllumination != 0;
    P.pos = make_view(gb->position_ao); P.nrm = make_view(gb->normal_roughness); P.alb = make_view(gb->albedo_metalness);
    for (int k = 0; k < n_outs; ++k) P.outs[k] = make_view(outs[k]);
    P.nOut = n_outs; P.dstRowOffset = dst_row_offset;
    P.hasEmissive = gb->emissive.ptr != nullptr;
    if (P.hasEmissive) {
        VQ_REQUIRE(vq_image_ok(gb->emissive) && gb->emissive.width == W && gb->emissive.height == H, "bad emissive plane");
        P.emi = make_view(gb->emissive);
    }
    VQ_REQUIRE(cube_desc_ok(env->irradiance_diffuse), "bad cubemap descriptor (irradiance_diffuse)");
    if (!P.diffuseOnly) {
        VQ_REQUIRE(cube_desc_ok(env->irradiance_specular), "bad cubemap descriptor (irradiance_specular)");
        VQ_REQUIRE(vq_image_ok(env->brdf_lut, 8), "bad BRDF LUT descriptor");
        VQ_REQUIRE(env->brdf_lut.width <= 8192 && env->brdf_lut.height <= 8192, "BRDF LUT larger than 8192^2");
        P.lut.w = env->brdf_lut.width; P.lut.h = env->brdf_lut.height;
    }
    // bordered sampling copies: from the prepared environment when it matches, else padded now on this stream
    int rc;
    const bool prepared = ctx->env_valid && same_cube(ctx->env_key.irradiance_diffuse, env->irradiance_diffuse) &&
                          (P.diffuseOnly || (same_cube(ctx->env_key.irradiance_specular, env->irradiance_specular) &&
                                             same_image(ctx->env_key.brdf_lut, env->brdf_lut) && ctx->env_lut));
    if (prepared) {
        fill_cube_view(env->irradiance_diffuse, (const float4*)ctx->env_diff, P.diff);
        if (!P.diffuseOnly) {
            fill_cube_view(env->irradiance_specular, (const float4*)ctx->env_spec, P.spec);
            P.lut.q = (const float4*)ctx->env_lut;
        }
    } else {
        rc = ensure_bytes(&ctx->tmp_diff, &ctx->tmp_diff_bytes, padded_bytes(env->irradiance_diffuse.res, env->irradiance_diffuse.mips)); if (rc) return rc;
        rc = pad_cube(env->irradiance_diffuse, (float4*)ctx->tmp_diff, stream); if (rc) return rc;
        fill_cube_view(env->irradiance_diffuse, (const float4*)ctx->tmp_diff, P.diff);
        if (!P.diffuseOnly) {
            rc = ensure_bytes(&ctx->tmp_spec, &ctx->tmp_spec_bytes, padded_bytes(env->irradiance_specular.res, env->irradiance_specular.mips)); if (rc) return rc;
            rc = pad_cube(env->irradiance_specular, (float4*)ctx->tmp_spec, stream); if (rc) return rc;
            fill_cube_view(env->irradiance_specular, (const float4*)ctx->tmp_spec, P.spec);
            rc = ensure_bytes(&ctx->tmp_lut, &ctx->tmp_lut_bytes, lut_footprint_bytes(env->brdf_lut)); if (rc) return rc;
            rc = footprint_lut(env->brdf_lut, (float4*)ctx->tmp_lut, stream); if (rc) return rc;
            P.lut.q = (const float4*)ctx->tmp_lut;
        }
    }
    P.rowBegin = row_begin; P.rows = row_end - row_begin; P.width = W;
    const bool shadowed = shadow && shadow->p;
    if (shadowed) {
        VQ_REQUIRE(n_outs == 1, "the shadowed pass writes one destination");
        VQ_REQUIRE(shadow->nPointCasters == L.numPointCasters && shadow->nSpotCasters == L.numSpotCasters && shadow->pitch >= W,
                   "PCF records do not match the frame's caster lists");
        P.shadow = *shadow;
    }

    rc = vq_fill_peer_sync(sig, &P.sync); if (rc) return rc;
    VQ_REQUIRE(P.sync.n == 0 || n_outs > 1, "a rendezvous only makes sense with peer destinations");
    P.ticket = P.sync.n > 1 ? vq_ticket_pair(ctx) : nullptr;
    P.diffHalfN = 0.5f * (float)env->irradiance_diffuse.res;
    P.diffMaxRec = (uint32_t)padded_texels(env->irradiance_diffuse.res, 1) - 1u;      // K1 samples mip 0 of the diffuse cube only
    P.specMaxRec = P.diffuseOnly ? 0u : (uint32_t)padded_texels(env->irradiance_specular.res, env->irradiance_specular.mips) - 1u;

    // persistent grid: x = the row's 256-pixel tiles, y = row groups striding the rows
    const unsigned gx = (unsigned)((W + FWD_TILE - 1) / FWD_TILE);
    unsigned gy = (unsigned)(ctx->sm_count * FWD_CTAS_PER_SM) / gx;
    if (gy < 1) gy = 1;
    if (gy > (unsigned)P.rows) gy = (unsigned)P.rows;
    VQ_REQUIRE(gy <= 65535u, "frame too tall for the launch grid");
    const int nPl = P.hasEmissive ? 4 : 3;
    const size_t smem = (size_t)FWD_STAGES * nPl * FWD_PLANE + 2 * FWD_STAGES * sizeof(uint64_t) + 16 * 8 * sizeof(FaceRec);
    const bool rot = P.sinB != 0.0f || P.cosB != 1.0f;            // yaw offset 0 is the common case: compiled out
    static std::atomic<bool> attrSet{false};                      // process-wide and idempotent: every instantiation, once
    if (!attrSet.load(std::memory_order_acquire)) {
        VQ_CUDA_OK(cudaFuncSetAttribute(forward_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024));
        VQ_CUDA_OK(cudaFuncSetAttribute(forward_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024));
        VQ_CUDA_OK(cudaFuncSetAttribute(forward_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024));
        VQ_CUDA_OK(cudaFuncSetAttribute(forward_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024));
        VQ_CUDA_OK(cudaFuncSetAttribute(forward_kernel<false, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024));
        VQ_CUDA_OK(cudaFuncSetAttribute(forward_kernel<false, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024));
        attrSet.store(true, std::memory_order_release);
    }
    auto launch = [&](auto kernel) { kernel<<<dim3(gx, gy), FWD_THREADS, smem, stream>>>(P); };
    VQ_REQUIRE(smem <= 96 * 1024, "stage layout exceeds the shared-memory budget");
    if (shadowed) rot ? launch(forward_kernel<false, true, true>) : launch(forward_kernel<false, false, true>);
    else if (n_outs > 1) rot ? launch(forward_kernel<true, true>) : launch(forward_kernel<true, false>);
    else rot ? launch(forward_kernel<false, true>) : launch(forward_kernel<false, false>);
    return vq_check_launch("forward_lighting");
}

int vq_forward_launch(VqContext* ctx, const VqPerFrameData* pf, const VqPerViewLightingData* pv,
                      const VqGBuffer* gb, const VqEnvironmentMaps* env, VqImage out,
                      int row_begin, int row_end, cudaStream_t stream, const ShadowRecV* shadow) {
    VQ_REQUIRE(gb && vq_image_ok(out) && out.height == gb->position_ao.height, "G-buffer planes and output must have the same size");
    return vq_forward_launch_multi(ctx, pf, pv, gb, env, &out, 1, 0, row_begin, row_end, nullptr, stream, shadow);
}

extern "C" int vq_forward_lighting(VqContext* ctx, const VqPerFrameData* pf, const VqPerViewLightingData* pv,
                                   const VqGBuffer* gb, const VqEnvironmentMaps* env, VqImage out,
                                   int row_begin, int row_end, void* stream) {
    int rc = vq_enter(ctx); if (rc) return rc;
    VQ_MARK("RenderSceneColor");
    return vq_forward_launch(ctx, pf, pv, gb, env, out, row_begin, row_end, (cudaStream_t)stream);
}

extern "C" int vq_forward_lighting_multi(VqContext* ctx, const VqPerFrameData* pf, const VqPerViewLightingData* pv,
                                         const VqGBuffer* gb, const VqEnvironmentMaps* env, const VqImage* outs, int n_outs,
                                         int dst_row_offset, int row_begin, int row_end, void* stream) {
    int rc = vq_enter(ctx); if (rc) return rc;
    VQ_MARK("RenderSceneColor");
    return vq_forward_launch_multi(ctx, pf, pv, gb, env, outs, n_outs, dst_row_offset, row_begin, row_end, nullptr, (cudaStream_t)stream);
}

// the same, with the cross-rank rendezvous run by the kernel's last CTA (VqPeerSignal): one kernel = shade + gather + barrier
extern "C" int vq_forward_lighting_multi_signal(VqContext* ctx, const VqPerFrameData* pf, const VqPerViewLightingData* pv,
                                                const VqGBuffer* gb, const VqEnvironmentMaps* env, const VqImage* outs, int n_outs,
                                                int dst_row_offset, int row_begin, int row_end, const VqPeerSignal* signal, void* stream) {
    int rc = vq_enter(ctx); if (rc) return rc;
    VQ_MARK("RenderSceneColor");
    return vq_forward_launch_multi(ctx, pf, pv, gb, env, outs, n_outs, dst_row_offset, row_begin, row_end, signal, (cudaStream_t)stream);
}

// The IBL cubemaps and the BRDF LUT are sampled from footprint-friendly copies (see CubeV, LutV).
// vq_environment_prepare builds them once and registers them in the context: the analogue of the RENDER_TARGET -> PIXEL_SHADER_RESOURCE transition the engine
// records after prefiltering (EnvironmentMapRendering.cpp:466-472). Call it again whenever the maps' contents change.
// Without it vq_forward_lighting rebuilds the copies on every call (always correct, slower: see tools/perf_forward.py).
extern "C" int vq_environment_prepare(VqContext* ctx, const VqEnvironmentMaps* env, void* stream) {
    int rc = vq_enter(ctx); if (rc) return rc;
    VQ_MARK("TransitionForSceneRendering");
    VQ_REQUIRE(env, "env is null");
    VQ_REQUIRE(cube_desc_ok(env->irradiance_diffuse), "bad cubemap descriptor (irradiance_diffuse)");
    VqScratchLock lock(ctx);
    ctx->env_valid = 0;
    const bool hasSpec = env->irradiance_specular.ptr != nullptr, hasLut = env->brdf_lut.ptr != nullptr;
    if (hasSpec) VQ_REQUIRE(cube_desc_ok(env->irradiance_specular), "bad cubemap descriptor (irradiance_specular)");
    if (hasLut) VQ_REQUIRE(vq_image_ok(env->brdf_lut, 8) && env->brdf_lut.width <= 8192 && env->brdf_lut.height <= 8192, "bad BRDF LUT descriptor");
    // ONE allocation for the three sampling copies (diffuse | specular | LUT footprints, 256-byte aligned parts): one buffer
    // to grow and free instead of three, regrown only when the three together outgrow it
    auto up = [](size_t b) { return (b + 255) & ~(size_t)255; };
    const size_t bD = up(padded_bytes(env->irradiance_diffuse.res, env->irradiance_diffuse.mips));
    const size_t bS = hasSpec ? up(padded_bytes(env->irradiance_specular.res, env->irradiance_specular.mips)) : 0;
    const size_t bL = hasLut ? up(lut_footprint_bytes(env->brdf_lut)) : 0;
    rc = ensure_bytes(&ctx->env_all, &ctx->env_all_bytes, bD + bS + bL); if (rc) return rc;
    ctx->env_diff = ctx->env_all;
    ctx->env_spec = hasSpec ? (char*)ctx->env_all + bD : nullptr;
    ctx->env_lut = hasLut ? (char*)ctx->env_all + bD + bS : nullptr;
    rc = pad_cube(env->irradiance_diffuse, (float4*)ctx->env_diff, (cudaStream_t)stream); if (rc) return rc;
    ctx->env_key = *env;
    if (hasSpec) { rc = pad_cube(env->irradiance_specular, (float4*)ctx->env_spec, (cudaStream_t)stream); if (rc) return rc; }
    if (hasLut) { rc = footprint_lut(env->brdf_lut, (float4*)ctx->env_lut, (cudaStream_t)stream); if (rc) return rc; }
    ctx->env_valid = 1;
    return VQ_OK;
}
extern "C" int vq_environment_invalidate(VqContext* ctx) {
    if (!ctx) { vq_set_error("null context"); return VQ_ERR_INVALID_ARG; }
    VqScratchLock lock(ctx);
    ctx->env_valid = 0;    return VQ_OK;
}

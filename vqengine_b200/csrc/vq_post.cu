// vq_post.cu — post chain kernels for sm_100a: Tonemapper (K6), separable Gaussian blur (K5),
// FidelityFX CAS (K7), FSR1 EASU (K8) / RCAS (K9), SPD (K10).
//
// All are streaming kernels over RGBA32F rows: float4 (LDG.128/STG.128) coalesced accesses, inputs
// that are read once bypass L1 allocation, stencil inputs are staged in shared memory (blur) or
// served by L1 (3x3 / 12-tap stencils). Math follows the HLSL the engine ships (file:line cited per
// kernel); parity against oracle/ is tested in tests/test_post_gpu.py.
#include "vq_common.cuh"

using namespace vq;

// =============================================================================================
// K6 Tonemapper — Shaders/Tonemapper.hlsl:110-151, Shaders/HDR.hlsl:76-119
// =============================================================================================
// pow(x, e) for x >= 0 as ex2(e * lg2(x)) on the SFU (MUFU.LG2 + MUFU.EX2): |rel err| <~ 3e-7 * max(1, e), far inside the
// 1e-4 budget even for the PQ exponent 78.84; powf() costs ~40 instructions per call and made the pass ALU-bound.
__device__ __forceinline__ float pow_sfu(float x, float e) { return exp2f(e * __log2f(x)); }
__device__ __forceinline__ float linear_to_srgb(float c) {          // HDR.hlsl:76-80
    return c < 0.0031308f ? 12.92f * c : fmaf(1.055f, pow_sfu(fabsf(c), 1.0f / 2.4f), -0.055f);
}
__device__ __forceinline__ float linear_to_st2084(float c) {        // HDR.hlsl:110-119
    const float m1 = 2610.0f / 4096.0f / 4, m2 = 2523.0f / 4096.0f * 128;
    const float c1 = 3424.0f / 4096.0f, c2 = 2413.0f / 4096.0f * 32, c3 = 2392.0f / 4096.0f * 32;
    const float cp = pow_sfu(fabsf(c), m1);
    return pow_sfu(__fdividef(fmaf(c2, cp, c1), fmaf(c3, cp, 1.0f)), m2);
}

template <int CURVE, bool GAMMA, bool TO2020>
__device__ __forceinline__ float4 tonemap_px(float4 in, float hdrScalar) {
    float3 o;
    if (CURVE == VQ_DISPLAY_CURVE_SRGB) {
        // Tonemap_Reinhard (Tonemapper.hlsl:24-27): c / (c + 1)
        o = f3(__fdividef(in.x, in.x + 1.0f), __fdividef(in.y, in.y + 1.0f), __fdividef(in.z, in.z + 1.0f));
        if (GAMMA) o = f3(linear_to_srgb(o.x), linear_to_srgb(o.y), linear_to_srgb(o.z));
    } else if (CURVE == VQ_DISPLAY_CURVE_ST2084) {
        o = xyz(in);
        if (TO2020) {   // Rec709ToRec2020, HDR.hlsl:88-97 (rows dot colour)
            const float3 c = o;
            o.x = 0.627402f * c.x + 0.329292f * c.y + 0.043306f * c.z;
            o.y = 0.069095f * c.x + 0.919544f * c.y + 0.011360f * c.z;
            o.z = 0.016394f * c.x + 0.088028f * c.y + 0.895578f * c.z;
        }
        o = f3(linear_to_st2084(o.x * hdrScalar), linear_to_st2084(o.y * hdrScalar), linear_to_st2084(o.z * hdrScalar));
    } else if (CURVE == VQ_DISPLAY_CURVE_LINEAR) {
        o = xyz(in);
    } else {
        o = f3(1.0f, 1.0f, 0.0f);
    }
    return make_float4(o.x, o.y, o.z, in.w);
}

constexpr int TM_THREADS = 256;
constexpr int TM_PX = 4;   // pixels per thread, loads issued back to back for memory-level parallelism

template <int CURVE, bool GAMMA, bool TO2020>
__global__ void __launch_bounds__(TM_THREADS) tonemap_kernel(ImgV in, ImgV out, float hdrScalar) {
    const int y = blockIdx.y;
    const int x0 = blockIdx.x * (TM_THREADS * TM_PX) + threadIdx.x;
    const float4* __restrict__ src = in.row(y);
    float4* __restrict__ dst = out.row(y);
    float4 v[TM_PX];
#pragma unroll
    for (int i = 0; i < TM_PX; ++i) {
        const int x = x0 + i * TM_THREADS;
        if (x < in.w) v[i] = ld_stream(src + x);
    }
#pragma unroll
    for (int i = 0; i < TM_PX; ++i) {
        const int x = x0 + i * TM_THREADS;
        if (x < in.w) st_stream(dst + x, tonemap_px<CURVE, GAMMA, TO2020>(v[i], hdrScalar));
    }
}

extern "C" int vq_tonemap(VqContext* ctx, const VqTonemapperParams* p, VqImage in, VqImage out, void* stream) {
    int rc = vq_enter(ctx); if (rc) return rc;
    VQ_MARK("TonemapperCS");
    VQ_REQUIRE(p, "params is null");
    VQ_REQUIRE(vq_image_ok(in) && vq_image_ok(out), "bad image descriptor");
    VQ_REQUIRE(in.width == out.width && in.height == out.height, "tonemap: in/out size mismatch");
    const dim3 grid((in.width + TM_THREADS * TM_PX - 1) / (TM_THREADS * TM_PX), in.height);
    const ImgV vi = make_view(in), vo = make_view(out);
    cudaStream_t s = (cudaStream_t)stream;
    const float hdrScalar = p->DisplayReferenceBrightnessLevel / 10000.0f;   // ST2084_MAX, HDR.hlsl:43
    switch (p->OutputDisplayCurve) {
        case VQ_DISPLAY_CURVE_SRGB:
            if (p->ToggleGammaCorrection) tonemap_kernel<VQ_DISPLAY_CURVE_SRGB, true, false><<<grid, TM_THREADS, 0, s>>>(vi, vo, hdrScalar);
            else                          tonemap_kernel<VQ_DISPLAY_CURVE_SRGB, false, false><<<grid, TM_THREADS, 0, s>>>(vi, vo, hdrScalar);
            break;
        case VQ_DISPLAY_CURVE_ST2084:
            if (p->ContentColorSpace == VQ_COLOR_SPACE_REC_709) tonemap_kernel<VQ_DISPLAY_CURVE_ST2084, false, true><<<grid, TM_THREADS, 0, s>>>(vi, vo, hdrScalar);
            else                                                 tonemap_kernel<VQ_DISPLAY_CURVE_ST2084, false, false><<<grid, TM_THREADS, 0, s>>>(vi, vo, hdrScalar);
            break;
        case VQ_DISPLAY_CURVE_LINEAR:
            tonemap_kernel<VQ_DISPLAY_CURVE_LINEAR, false, false><<<grid, TM_THREADS, 0, s>>>(vi, vo, hdrScalar);
            break;
        default:   // Tonemapper.hlsl:143-145: unknown curve paints yellow
            tonemap_kernel<3, false, false><<<grid, TM_THREADS, 0, s>>>(vi, vo, hdrScalar);
            break;
    }
    return vq_check_launch("tonemap");
}

// =============================================================================================
// K5 Gaussian blur — Shaders/GaussianBlur.hlsl:74-186, KERNEL_DIMENSION 21, clamp-to-edge, alpha = 1
// =============================================================================================
__constant__ float c_gauss[11] = {0.224716f, 0.191756f, 0.119146f, 0.053897f, 0.017746f, 0.004252f,
                                  0.000741f, 0.000094f, 0.000009f, 0.000001f, 0.0f};   // GaussianBlur.hlsl:110

// X pass: a CTA owns a 512-pixel column strip and walks BX_XR consecutive rows. Each row's BX_W+24 pixels are staged into
// PLANAR shared memory (R,G,B planes) so that each thread reads its 28-value window with conflict-free LDS.128 and
// produces 4 adjacent pixels from registers (sliding window: 7 LDS.128 per channel per 4 pixels). The next row's global
// loads are issued into registers before the current row is filtered (software pipelining), results leave through a
// shared-memory transpose so that the stores are coalesced.
constexpr int BX_T = 128;            // threads per CTA (4 autonomous warps)
constexpr int BX_XR = 4;             // consecutive rows per CTA (software-pipelined)
constexpr int BX_WW = 128;           // output pixels per warp per row (4 per lane)
constexpr int BX_W = BX_WW * (BX_T / 32);   // per CTA
constexpr int BX_SM = BX_WW + 24;    // staged per warp: [-12, BX_WW+12)
constexpr int BX_LD = (BX_SM + 31) / 32;    // float4 loads per lane per row (5)

__global__ void __launch_bounds__(BX_T) blur_x_kernel(ImgV in, ImgV out, int sizeX, int sizeY) {
    // every warp owns its sub-strip end to end (private staging + private output tile): only __syncwarp(), so warps
    // drift apart and overlap each other's load / filter / store phases instead of meeting at CTA barriers
    __shared__ __align__(16) float sm[BX_T / 32][3][BX_SM];
    __shared__ float4 so[BX_T / 32][BX_WW];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int xBase = blockIdx.x * BX_W + warp * BX_WW;
    const int row0 = blockIdx.y * BX_XR;
    if (xBase >= sizeX) return;
    float4 pre[BX_LD];
    auto load_row = [&](int y) {
        const float4* __restrict__ src = in.row(y);
#pragma unroll
        for (int q = 0; q < BX_LD; ++q) {
            const int i = lane + q * 32;
            const int sx = min(max(xBase - 12 + i, 0), sizeX - 1);       // sampleCoord clamp, GaussianBlur.hlsl:144
            if (i < BX_SM) pre[q] = __ldg(src + sx);
        }
    };
    if (row0 < sizeY) load_row(row0);
    float (*buf)[BX_SM] = sm[warp];
    for (int r = 0; r < BX_XR; ++r) {
        const int y = row0 + r;
        if (y >= sizeY) break;
#pragma unroll
        for (int q = 0; q < BX_LD; ++q) {
            const int i = lane + q * 32;
            if (i < BX_SM) { buf[0][i] = pre[q].x; buf[1][i] = pre[q].y; buf[2][i] = pre[q].z; }
        }
        __syncwarp();
        if (r + 1 < BX_XR && y + 1 < sizeY) load_row(y + 1);             // in flight while this row is filtered
        float acc[3][4];
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            float win[28];                                               // staged positions 4l .. 4l+27 == image x-12 .. x+15
            const float4* p = reinterpret_cast<const float4*>(&buf[c][lane * 4]);
#pragma unroll
            for (int q = 0; q < 7; ++q) { const float4 v = p[q]; win[4 * q] = v.x; win[4 * q + 1] = v.y; win[4 * q + 2] = v.z; win[4 * q + 3] = v.w; }
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                float a = 0.0f;
#pragma unroll
                for (int k = 0; k < 21; ++k) {                           // kernelIt order 0..20 as in the HLSL loop
                    const int ki = k < 10 ? 10 - k : k - 10;
                    a = fmaf(win[j + 2 + k], c_gauss[ki], a);            // tap at x+j-10+k -> window index j+2+k
                }
                acc[c][j] = a;
            }
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) so[warp][lane * 4 + j] = make_float4(acc[0][j], acc[1][j], acc[2][j], 1.0f);
        __syncwarp();
        float4* __restrict__ dst = out.row(y);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int lx = lane + k * 32;
            if (xBase + lx < sizeX) st_stream(dst + xBase + lx, so[warp][lx]);
        }
        __syncwarp();                                                    // so[] and buf[] free for the next row
    }
}

// Y pass: no shared memory. A thread owns one column and marches down BYM_ROWS output rows keeping the last 21 input
// rows of its column in a REGISTER ring (the loop is unrolled by 21 so that every ring index is a compile-time constant):
// one coalesced LDG.128 and one STG.128 per output pixel, 63 FMAs, no barriers. Lanes are adjacent columns, so every
// warp instruction moves 512 contiguous bytes. Segments overlap by 20 rows (re-read through L2).
constexpr int BYM_T = 128;          // threads per CTA = columns per CTA
// A/B on B200 at 4K (us): rows/prefetch 21/21: 47.9 | 42/21: 49.2 | 63/21: 51.0 | 63/7: 57.2 | 126/7: 65.3 | 252/7: 62.5
// (the shared-memory tile version it replaces: 67.5)
constexpr int BYM_ROWS = 21;        // output rows per thread (multiple of 21)
constexpr int BYM_PRE = 21;         // rows requested ahead of use (divides 21): memory-level parallelism per thread

__global__ void __launch_bounds__(BYM_T) blur_y_kernel(ImgV in, ImgV out, int sizeX, int sizeY) {
    const int x = blockIdx.x * BYM_T + threadIdx.x;
    if (x >= sizeX) return;
    const int y0 = blockIdx.y * BYM_ROWS;
    const float4* __restrict__ src = in.p + x;
    float4* __restrict__ dst = out.p + x;
    const int pin = in.pitch4, pout = out.pitch4;
    float3 ring[21], pre[BYM_PRE];
    // rows y0-10 .. y0+9 (clamped) fill ring slots 0..19; slot k holds input row (y0 - 10 + k)
#pragma unroll
    for (int k = 0; k < 20; ++k) {
        const int sy = min(max(y0 - 10 + k, 0), sizeY - 1);          // GaussianBlur.hlsl:180
        ring[k] = xyz(__ldg(src + (size_t)sy * pin));
    }
#pragma unroll
    for (int k = 0; k < BYM_PRE; ++k) pre[k] = xyz(__ldg(src + (size_t)min(y0 + 10 + k, sizeY - 1) * pin));
    for (int base = 0; base < BYM_ROWS && y0 + base < sizeY; base += 21) {
#pragma unroll
        for (int u = 0; u < 21; ++u) {
            const int y = y0 + base + u;              // no early exit inside the unrolled body: loads stay hoistable
            // newest row y+10 (requested BYM_PRE iterations ago) goes to slot (20+u)%21; request row y+10+BYM_PRE
            ring[(20 + u) % 21] = pre[u % BYM_PRE];
            pre[u % BYM_PRE] = xyz(__ldg(src + (size_t)min(y + 10 + BYM_PRE, sizeY - 1) * pin));
            float3 a = f3(0.0f);
#pragma unroll
            for (int k = 0; k < 21; ++k) {                           // kernelIt order 0..20 as in the HLSL loop
                const float w = c_gauss[k < 10 ? 10 - k : k - 10];
                const float3 v = ring[(u + k) % 21];
                a.x = fmaf(v.x, w, a.x); a.y = fmaf(v.y, w, a.y); a.z = fmaf(v.z, w, a.z);
            }
            if (y < sizeY) st_stream(dst + (size_t)y * pout, make_float4(a.x, a.y, a.z, 1.0f));
        }
    }
}

static int blur_common(VqContext* ctx, const VqBlurParams* p, VqImage in, VqImage out, void* stream, bool vertical) {
    int rc = vq_enter(ctx); if (rc) return rc;
    VQ_REQUIRE(p, "params is null");
    VQ_REQUIRE(vq_image_ok(in) && vq_image_ok(out), "bad image descriptor");
    VQ_REQUIRE(p->iImageSizeX > 0 && p->iImageSizeY > 0, "blur: image size must be positive");
    VQ_REQUIRE(p->iImageSizeX <= in.width && p->iImageSizeY <= in.height &&
               p->iImageSizeX <= out.width && p->iImageSizeY <= out.height, "blur: iImageSize exceeds the images");
    VQ_REQUIRE(in.ptr != out.ptr, "blur: in-place is not supported (the engine ping-pongs too)");
    const ImgV vi = make_view(in), vo = make_view(out);
    cudaStream_t s = (cudaStream_t)stream;
    if (!vertical) {
        const dim3 grid((p->iImageSizeX + BX_W - 1) / BX_W, (p->iImageSizeY + BX_XR - 1) / BX_XR);
        blur_x_kernel<<<grid, BX_T, 0, s>>>(vi, vo, p->iImageSizeX, p->iImageSizeY);
    } else {
        const dim3 grid((p->iImageSizeX + BYM_T - 1) / BYM_T, (p->iImageSizeY + BYM_ROWS - 1) / BYM_ROWS);
        blur_y_kernel<<<grid, BYM_T, 0, s>>>(vi, vo, p->iImageSizeX, p->iImageSizeY);
    }
    return vq_check_launch(vertical ? "gaussian_blur_y" : "gaussian_blur_x");
}
extern "C" int vq_gaussian_blur_x(VqContext* ctx, const VqBlurParams* p, VqImage in, VqImage out, void* stream) { VQ_MARK("BlurX"); return blur_common(ctx, p, in, out, stream, false); }
extern "C" int vq_gaussian_blur_y(VqContext* ctx, const VqBlurParams* p, VqImage in, VqImage out, void* stream) { VQ_MARK("BlurY"); return blur_common(ctx, p, in, out, stream, true); }

// =============================================================================================
// FidelityFX scalar helpers — FSR1.0/ffx_a.h:1842-1845 (integer bit tricks: reproduced exactly)
// =============================================================================================
__device__ __forceinline__ float APrxLoSqrtF1(float a) { return __uint_as_float((__float_as_uint(a) >> 1u) + 0x1fbc4639u); }
__device__ __forceinline__ float APrxLoRcpF1(float a)  { return __uint_as_float(0x7ef07ebbu - __float_as_uint(a)); }
__device__ __forceinline__ float APrxMedRcpF1(float a) { const float b = __uint_as_float(0x7ef19fffu - __float_as_uint(a)); return b * fmaf(-b, a, 2.0f); }
__device__ __forceinline__ float APrxLoRsqF1(float a)  { return __uint_as_float(0x5f347d74u - (__float_as_uint(a) >> 1u)); }
__device__ __forceinline__ float min3f(float a, float b, float c) { return fminf(a, fminf(b, c)); }
__device__ __forceinline__ float max3f(float a, float b, float c) { return fmaxf(a, fmaxf(b, c)); }

// Texture.Load semantics: out-of-range reads return 0 (SURVEY.md §9)
__device__ __forceinline__ float3 load_zero_border(const ImgV& im, int x, int y) {
    if ((unsigned)x >= (unsigned)im.w || (unsigned)y >= (unsigned)im.h) return f3(0.0f);
    return xyz(__ldg(im.row(y) + x));
}

// =============================================================================================
// K7 CAS sharpen-only — CAS/ffx_cas.h:408-537 (noScaling), wrapper AMDFidelityFX.hlsl:122-174
// =============================================================================================
constexpr int ST_BX = 32, ST_BY = 8;   // 3x3 stencil kernels: 32x8 pixel blocks, rows shared through L1

__global__ void __launch_bounds__(ST_BX * ST_BY) cas_kernel(ImgV in, ImgV out, float peak) {
    const int x = blockIdx.x * ST_BX + threadIdx.x, y = blockIdx.y * ST_BY + threadIdx.y;
    if (x >= out.w || y >= out.h) return;
    const float3 b = load_zero_border(in, x, y - 1);
    const float3 d = load_zero_border(in, x - 1, y);
    const float3 e = load_zero_border(in, x, y);
    const float3 f = load_zero_border(in, x + 1, y);
    const float3 h = load_zero_border(in, x, y + 1);
    // only the green channel's weight survives without CAS_SLOW (ffx_cas.h:511-519)
    const float mnG = min3f(min3f(d.y, e.y, f.y), b.y, h.y);
    const float mxG = max3f(max3f(d.y, e.y, f.y), b.y, h.y);
    const float rcpMG = APrxLoRcpF1(mxG);
    float ampG = saturate(fminf(mnG, 1.0f - mxG) * rcpMG);
    ampG = APrxLoSqrtF1(ampG);
    const float wG = ampG * peak;
    const float rcpWeight = APrxMedRcpF1(fmaf(4.0f, wG, 1.0f));
    float3 o;
    o.x = saturate((b.x * wG + d.x * wG + f.x * wG + h.x * wG + e.x) * rcpWeight);
    o.y = saturate((b.y * wG + d.y * wG + f.y * wG + h.y * wG + e.y) * rcpWeight);
    o.z = saturate((b.z * wG + d.z * wG + f.z * wG + h.z * wG + e.z) * rcpWeight);
    st_stream(out.row(y) + x, make_float4(o.x, o.y, o.z, 1.0f));
}

extern "C" int vq_cas(VqContext* ctx, const uint32_t cas_const[8], VqImage in, VqImage out, void* stream) {
    int rc = vq_enter(ctx); if (rc) return rc;
    VQ_MARK("FFX-CAS CS");
    VQ_REQUIRE(cas_const, "cas_const is null");
    VQ_REQUIRE(vq_image_ok(in) && vq_image_ok(out), "bad image descriptor");
    VQ_REQUIRE(in.width == out.width && in.height == out.height, "cas: sharpen-only path needs equal sizes (FFXCAS_NO_UPSCALING)");
    VQ_REQUIRE(in.ptr != out.ptr, "cas: in-place is not supported");
    float peak; memcpy(&peak, &cas_const[4], 4);     // const1.x
    const dim3 grid((out.width + ST_BX - 1) / ST_BX, (out.height + ST_BY - 1) / ST_BY);
    cas_kernel<<<grid, dim3(ST_BX, ST_BY), 0, (cudaStream_t)stream>>>(make_view(in), make_view(out), peak);
    return vq_check_launch("cas");
}

// =============================================================================================
// K9 RCAS — FSR1.0/ffx_fsr1.h:684-769, wrapper AMDFidelityFX.hlsl:335-376
// =============================================================================================
__global__ void __launch_bounds__(ST_BX * ST_BY) rcas_kernel(ImgV in, ImgV out, float sharp) {
    const int x = blockIdx.x * ST_BX + threadIdx.x, y = blockIdx.y * ST_BY + threadIdx.y;
    if (x >= out.w || y >= out.h) return;
    const float3 b = load_zero_border(in, x, y - 1);
    const float3 d = load_zero_border(in, x - 1, y);
    const float3 e = load_zero_border(in, x, y);
    const float3 f = load_zero_border(in, x + 1, y);
    const float3 h = load_zero_border(in, x, y + 1);
    const float3 mn4 = f3(fminf(min3f(b.x, d.x, f.x), h.x), fminf(min3f(b.y, d.y, f.y), h.y), fminf(min3f(b.z, d.z, f.z), h.z));
    const float3 mx4 = f3(fmaxf(max3f(b.x, d.x, f.x), h.x), fmaxf(max3f(b.y, d.y, f.y), h.y), fmaxf(max3f(b.z, d.z, f.z), h.z));
    // limiters use the full-precision rcp of the HLSL (ffx_fsr1.h:749-755), i.e. the hardware reciprocal (1 ulp)
    const float hitMinR = mn4.x * rcp_fast(4.0f * mx4.x);
    const float hitMinG = mn4.y * rcp_fast(4.0f * mx4.y);
    const float hitMinB = mn4.z * rcp_fast(4.0f * mx4.z);
    const float hitMaxR = (1.0f - mx4.x) * rcp_fast(fmaf(4.0f, mn4.x, -4.0f));
    const float hitMaxG = (1.0f - mx4.y) * rcp_fast(fmaf(4.0f, mn4.y, -4.0f));
    const float hitMaxB = (1.0f - mx4.z) * rcp_fast(fmaf(4.0f, mn4.z, -4.0f));
    const float lobeR = fmaxf(-hitMinR, hitMaxR);
    const float lobeG = fmaxf(-hitMinG, hitMaxG);
    const float lobeB = fmaxf(-hitMinB, hitMaxB);
    const float FSR_RCAS_LIMIT = 0.25f - (1.0f / 16.0f);   // ffx_fsr1.h:654
    const float lobe = fmaxf(-FSR_RCAS_LIMIT, fminf(max3f(lobeR, lobeG, lobeB), 0.0f)) * sharp;
    const float rcpL = APrxMedRcpF1(fmaf(4.0f, lobe, 1.0f));
    float3 o;
    o.x = (lobe * b.x + lobe * d.x + lobe * h.x + lobe * f.x + e.x) * rcpL;
    o.y = (lobe * b.y + lobe * d.y + lobe * h.y + lobe * f.y + e.y) * rcpL;
    o.z = (lobe * b.z + lobe * d.z + lobe * h.z + lobe * f.z + e.z) * rcpL;
    st_stream(out.row(y) + x, make_float4(o.x, o.y, o.z, 1.0f));
}

extern "C" int vq_fsr_rcas(VqContext* ctx, const uint32_t rcas_const[4], VqImage in, VqImage out, void* stream) {
    int rc = vq_enter(ctx); if (rc) return rc;
    VQ_MARK("FSR-RCAS CS");
    VQ_REQUIRE(rcas_const, "rcas_const is null");
    VQ_REQUIRE(vq_image_ok(in) && vq_image_ok(out), "bad image descriptor");
    VQ_REQUIRE(in.width == out.width && in.height == out.height, "rcas: in/out size mismatch");
    VQ_REQUIRE(in.ptr != out.ptr, "rcas: in-place is not supported");
    float sharp; memcpy(&sharp, &rcas_const[0], 4);
    const dim3 grid((out.width + ST_BX - 1) / ST_BX, (out.height + ST_BY - 1) / ST_BY);
    rcas_kernel<<<grid, dim3(ST_BX, ST_BY), 0, (cudaStream_t)stream>>>(make_view(in), make_view(out), sharp);
    return vq_check_launch("fsr_rcas");
}

// =============================================================================================
// K8 EASU — FSR1.0/ffx_fsr1.h:239-437, wrapper AMDFidelityFX.hlsl:247-288.
// FsrEasuCon puts every Gather4 coordinate on a texel corner, so the 4 gathers are 12 integer texel
// fetches around (fx,fy) = floor(ip*con0.xy + con0.zw) under the sampler's addressing mode.
// =============================================================================================
template <int ADDR>
__device__ __forceinline__ float3 load_addr(const ImgV& im, int x, int y) {
    if (ADDR == VQ_ADDRESS_WRAP) {
        // taps lie within [-2, size+2]: one conditional add/sub wraps them (the general % only for images < 3 wide)
        if (im.w >= 3) { x = x < 0 ? x + im.w : (x >= im.w ? x - im.w : x); } else { x %= im.w; if (x < 0) x += im.w; }
        if (im.h >= 3) { y = y < 0 ? y + im.h : (y >= im.h ? y - im.h : y); } else { y %= im.h; if (y < 0) y += im.h; }
    } else {
        x = min(max(x, 0), im.w - 1);
        y = min(max(y, 0), im.h - 1);
    }
    return xyz(__ldg(im.row(y) + x));
}

__device__ __forceinline__ void easu_set(float2& dir, float& len, float w, float lA, float lB, float lC, float lD, float lE) {
    // FsrEasuSetF, ffx_fsr1.h:275-313 (w = the bilinear weight selected by biS/biT/biU/biV)
    const float dc = lD - lC, cb = lC - lB;
    float lenX = fmaxf(fabsf(dc), fabsf(cb));
    lenX = APrxLoRcpF1(lenX);
    const float dirX = lD - lB;
    dir.x = fmaf(dirX, w, dir.x);
    lenX = saturate(fabsf(dirX) * lenX);
    lenX *= lenX;
    len = fmaf(lenX, w, len);
    const float ec = lE - lC, ca = lC - lA;
    float lenY = fmaxf(fabsf(ec), fabsf(ca));
    lenY = APrxLoRcpF1(lenY);
    const float dirY = lE - lA;
    dir.y = fmaf(dirY, w, dir.y);
    lenY = saturate(fabsf(dirY) * lenY);
    lenY *= lenY;
    len = fmaf(lenY, w, len);
}
__device__ __forceinline__ void easu_tap(float3& aC, float& aW, float offx, float offy, float2 dir, float2 len, float lob, float clp, float3 c) {
    // FsrEasuTapF, ffx_fsr1.h:239-272
    float vx = offx * dir.x + offy * dir.y;
    float vy = offx * (-dir.y) + offy * dir.x;
    vx *= len.x; vy *= len.y;
    float d2 = vx * vx + vy * vy;
    d2 = fminf(d2, clp);
    float wB = fmaf(2.0f / 5.0f, d2, -1.0f);
    float wA = fmaf(lob, d2, -1.0f);
    wB *= wB; wA *= wA;
    wB = fmaf(25.0f / 16.0f, wB, -(25.0f / 16.0f - 1.0f));
    const float w = wB * wA;
    aC.x = fmaf(c.x, w, aC.x); aC.y = fmaf(c.y, w, aC.y); aC.z = fmaf(c.z, w, aC.z);
    aW += w;
}
__device__ __forceinline__ float luma2(float3 c) { return fmaf(c.z, 0.5f, fmaf(c.x, 0.5f, c.y)); }

struct EasuCon { float c0x, c0y, c0z, c0w; };

// position of 'f' for output coordinate o (ffx_fsr1.h:323-326). Unfused mul+add so floor() sees the oracle's value.
__device__ __forceinline__ float easu_pos(int o, float scale, float bias) { return __fadd_rn(__fmul_rn((float)o, scale), bias); }

// The 12-tap kernel + analysis for one output pixel; tap(dx,dy) returns the texel at (fx+dx, fy+dy).
template <class Tap>
__device__ __forceinline__ float3 easu_filter(float ppx, float ppy, Tap tap) {
    const float3 b = tap(0, -1), c = tap(1, -1);
    const float3 e = tap(-1, 0), f = tap(0, 0), g = tap(1, 0), h = tap(2, 0);
    const float3 i = tap(-1, 1), j = tap(0, 1), k = tap(1, 1), l = tap(2, 1);
    const float3 n = tap(0, 2), o = tap(1, 2);
    const float bL = luma2(b), cL = luma2(c), eL = luma2(e), fL = luma2(f), gL = luma2(g), hL = luma2(h);
    const float iL = luma2(i), jL = luma2(j), kL = luma2(k), lL = luma2(l), nL = luma2(n), oL = luma2(o);
    float2 dir = make_float2(0.0f, 0.0f);
    float len = 0.0f;
    easu_set(dir, len, (1.0f - ppx) * (1.0f - ppy), bL, eL, fL, gL, jL);
    easu_set(dir, len, ppx * (1.0f - ppy), cL, fL, gL, hL, kL);
    easu_set(dir, len, (1.0f - ppx) * ppy, fL, iL, jL, kL, nL);
    easu_set(dir, len, ppx * ppy, gL, jL, kL, lL, oL);
    float dirR = dir.x * dir.x + dir.y * dir.y;
    const bool zro = dirR < (1.0f / 32768.0f);
    dirR = APrxLoRsqF1(dirR);
    dirR = zro ? 1.0f : dirR;
    dir.x = zro ? 1.0f : dir.x;
    dir.x *= dirR; dir.y *= dirR;
    len = len * 0.5f;
    len *= len;
    const float stretch = (dir.x * dir.x + dir.y * dir.y) * APrxLoRcpF1(fmaxf(fabsf(dir.x), fabsf(dir.y)));
    const float2 len2 = make_float2(fmaf(stretch - 1.0f, len, 1.0f), fmaf(-0.5f, len, 1.0f));
    const float lob = fmaf((1.0f / 4.0f - 0.04f) - 0.5f, len, 0.5f);
    const float clp = APrxLoRcpF1(lob);
    const float3 min4 = fmin3(fmin3(f, fmin3(g, j)), k);
    const float3 max4 = fmax3(fmax3(f, fmax3(g, j)), k);
    float3 aC = f3(0.0f);
    float aW = 0.0f;
    easu_tap(aC, aW, 0.0f - ppx, -1.0f - ppy, dir, len2, lob, clp, b);
    easu_tap(aC, aW, 1.0f - ppx, -1.0f - ppy, dir, len2, lob, clp, c);
    easu_tap(aC, aW, -1.0f - ppx, 1.0f - ppy, dir, len2, lob, clp, i);
    easu_tap(aC, aW, 0.0f - ppx, 1.0f - ppy, dir, len2, lob, clp, j);
    easu_tap(aC, aW, 0.0f - ppx, 0.0f - ppy, dir, len2, lob, clp, f);
    easu_tap(aC, aW, -1.0f - ppx, 0.0f - ppy, dir, len2, lob, clp, e);
    easu_tap(aC, aW, 1.0f - ppx, 1.0f - ppy, dir, len2, lob, clp, k);
    easu_tap(aC, aW, 2.0f - ppx, 1.0f - ppy, dir, len2, lob, clp, l);
    easu_tap(aC, aW, 2.0f - ppx, 0.0f - ppy, dir, len2, lob, clp, h);
    easu_tap(aC, aW, 1.0f - ppx, 0.0f - ppy, dir, len2, lob, clp, g);
    easu_tap(aC, aW, 1.0f - ppx, 2.0f - ppy, dir, len2, lob, clp, o);
    easu_tap(aC, aW, 0.0f - ppx, 2.0f - ppy, dir, len2, lob, clp, n);
    const float rw = rcp_fast(aW);   // ARcpF1 = rcp() in the HLSL
    return fmin3(max4, fmax3(min4, aC * rw));
}

// Generic path (any scale): taps fetched straight from global memory through L1.
template <int ADDR>
__global__ void __launch_bounds__(ST_BX * ST_BY) easu_kernel(ImgV in, ImgV out, EasuCon con) {
    const int x = blockIdx.x * ST_BX + threadIdx.x, y = blockIdx.y * ST_BY + threadIdx.y;
    if (x >= out.w || y >= out.h) return;
    float ppx = easu_pos(x, con.c0x, con.c0z), ppy = easu_pos(y, con.c0y, con.c0w);
    const float fpx = floorf(ppx), fpy = floorf(ppy);
    ppx -= fpx; ppy -= fpy;
    const int fx = (int)fpx, fy = (int)fpy;
    const float3 pix = easu_filter(ppx, ppy, [&](int dx, int dy) { return load_addr<ADDR>(in, fx + dx, fy + dy); });
    st_stream(out.row(y) + x, make_float4(pix.x, pix.y, pix.z, 1.0f));
}

// Upscaling path (input/output ratio <= 1, the FSR use case), two phases per CTA of 32x8 OUTPUT pixels:
//   stage  : the CTA's input footprint (<= 36x12 texels) goes to shared memory once, sampler addressing applied,
//            with the tap's luma in .w;
//   phase 1: one thread per candidate 'f' texel (<= 32x8) evaluates the four FsrEasuSetF analyses — they depend only
//            on the 12 lumas around 'f', so every output pixel that resolves to the same texel shares them (4 outputs
//            per texel at 2x) — and parks them in shared memory;
//   phase 2: one thread per output pixel blends the four analyses with its bilinear weights and runs the 12 taps with
//            incrementally updated rotated offsets (v(i,j) = v(0,0) + i*A + j*B instead of two dot products per tap).
// ncu r01: the per-output kernel executed 505 instructions per output pixel; this organisation needs ~60 % of that.
constexpr int EU_BX = 32, EU_BY = 8;
constexpr int EU_TW = EU_BX + 4, EU_TH = EU_BY + 4;

struct EasuSet { float dirX, dirY, lenX, lenY; };
__device__ __forceinline__ EasuSet easu_set_shared(float lA, float lB, float lC, float lD, float lE) {
    // the weight-independent half of FsrEasuSetF (ffx_fsr1.h:291-312)
    EasuSet r;
    const float dc = lD - lC, cb = lC - lB;
    float lenX = APrxLoRcpF1(fmaxf(fabsf(dc), fabsf(cb)));
    r.dirX = lD - lB;
    lenX = saturate(fabsf(r.dirX) * lenX);
    r.lenX = lenX * lenX;
    const float ec = lE - lC, ca = lC - lA;
    float lenY = APrxLoRcpF1(fmaxf(fabsf(ec), fabsf(ca)));
    r.dirY = lE - lA;
    lenY = saturate(fabsf(r.dirY) * lenY);
    r.lenY = lenY * lenY;
    return r;
}
__device__ __forceinline__ void easu_set_blend(float2& dir, float& len, float w, const float4& a) {   // a = {dirX,dirY,lenX,lenY}
    dir.x = fmaf(a.x, w, dir.x); len = fmaf(a.z, w, len);
    dir.y = fmaf(a.y, w, dir.y); len = fmaf(a.w, w, len);
}
// weight of a tap at rotated, anisotropically scaled offset (vx,vy) (the second half of FsrEasuTapF)
__device__ __forceinline__ void easu_tap_v(float3& aC, float& aW, float vx, float vy, float lob, float clp, float4 c) {
    float d2 = fminf(fmaf(vx, vx, vy * vy), clp);
    float wB = fmaf(2.0f / 5.0f, d2, -1.0f);
    float wA = fmaf(lob, d2, -1.0f);
    wB *= wB; wA *= wA;
    wB = fmaf(25.0f / 16.0f, wB, -(25.0f / 16.0f - 1.0f));
    const float w = wB * wA;
    aC.x = fmaf(c.x, w, aC.x); aC.y = fmaf(c.y, w, aC.y); aC.z = fmaf(c.z, w, aC.z);
    aW += w;
}

template <int ADDR>
__global__ void __launch_bounds__(EU_BX * EU_BY, 4) easu_up_kernel(ImgV in, ImgV out, EasuCon con) {
    __shared__ float4 tile[EU_TH][EU_TW];          // rgb + luma
    __shared__ float4 sets[4][EU_BY][EU_BX];       // S,T,U,V analyses of candidate texel (fy-fyFirst, fx-fxFirst); SoA: conflict-free
    const int ox0 = blockIdx.x * EU_BX, oy0 = blockIdx.y * EU_BY;
    const int fxFirst = (int)floorf(easu_pos(ox0, con.c0x, con.c0z));
    const int fyFirst = (int)floorf(easu_pos(oy0, con.c0y, con.c0w));
    const int tx0 = fxFirst - 1, ty0 = fyFirst - 1;
    // candidate 'f' texels of this tile: local (cx,cy) in [0,ncx) x [0,ncy); the staged footprint is (ncx+3) x (ncy+3)
    const int oxl = min(ox0 + EU_BX - 1, out.w - 1), oyl = min(oy0 + EU_BY - 1, out.h - 1);
    const int ncx = (int)floorf(easu_pos(oxl, con.c0x, con.c0z)) - fxFirst + 1;
    const int ncy = (int)floorf(easu_pos(oyl, con.c0y, con.c0w)) - fyFirst + 1;
    if (threadIdx.x < ncx + 3) {                               // only the footprint this ratio needs (20x8 texels at 2x, not 36x12)
        for (int ly = threadIdx.y; ly < ncy + 3; ly += EU_BY) {
            const float3 v = load_addr<ADDR>(in, tx0 + (int)threadIdx.x, ty0 + ly);
            tile[ly][threadIdx.x] = make_float4(v.x, v.y, v.z, luma2(v));
        }
    }
    if (threadIdx.x < 4 && (int)threadIdx.x + EU_BX < ncx + 3) {   // columns 32..35 of the footprint (ratio close to 1)
        for (int ly = threadIdx.y; ly < ncy + 3; ly += EU_BY) {
            const float3 v = load_addr<ADDR>(in, tx0 + (int)threadIdx.x + EU_BX, ty0 + ly);
            tile[ly][threadIdx.x + EU_BX] = make_float4(v.x, v.y, v.z, luma2(v));
        }
    }
    __syncthreads();
    // ---- phase 1 ----
    {
        const int cx = threadIdx.x, cy = threadIdx.y;
        if (cx < ncx && cy < ncy) {
            const float4* t = &tile[cy + 1][cx + 1];                   // 'f'
            const float bL = t[-EU_TW].w, cL = t[-EU_TW + 1].w;
            const float eL = t[-1].w, fL = t[0].w, gL = t[1].w, hL = t[2].w;
            const float iL = t[EU_TW - 1].w, jL = t[EU_TW].w, kL = t[EU_TW + 1].w, lL = t[EU_TW + 2].w;
            const float nL = t[2 * EU_TW].w, oL = t[2 * EU_TW + 1].w;
            const EasuSet sS = easu_set_shared(bL, eL, fL, gL, jL), sT = easu_set_shared(cL, fL, gL, hL, kL);
            const EasuSet sU = easu_set_shared(fL, iL, jL, kL, nL), sV = easu_set_shared(gL, jL, kL, lL, oL);
            sets[0][cy][cx] = make_float4(sS.dirX, sS.dirY, sS.lenX, sS.lenY);
            sets[1][cy][cx] = make_float4(sT.dirX, sT.dirY, sT.lenX, sT.lenY);
            sets[2][cy][cx] = make_float4(sU.dirX, sU.dirY, sU.lenX, sU.lenY);
            sets[3][cy][cx] = make_float4(sV.dirX, sV.dirY, sV.lenX, sV.lenY);
        }
    }
    __syncthreads();
    // ---- phase 2: one output pixel per thread ----
    const int x = ox0 + threadIdx.x, y = oy0 + threadIdx.y;
    if (x >= out.w || y >= out.h) return;
    float ppx = easu_pos(x, con.c0x, con.c0z), ppy = easu_pos(y, con.c0y, con.c0w);
    const float fpx = floorf(ppx), fpy = floorf(ppy);
    ppx -= fpx; ppy -= fpy;
    const int cx = (int)fpx - fxFirst, cy = (int)fpy - fyFirst;
    float2 dir = make_float2(0.0f, 0.0f);
    float len = 0.0f;
    easu_set_blend(dir, len, (1.0f - ppx) * (1.0f - ppy), sets[0][cy][cx]);
    easu_set_blend(dir, len, ppx * (1.0f - ppy), sets[1][cy][cx]);
    easu_set_blend(dir, len, (1.0f - ppx) * ppy, sets[2][cy][cx]);
    easu_set_blend(dir, len, ppx * ppy, sets[3][cy][cx]);
    float dirR = dir.x * dir.x + dir.y * dir.y;
    const bool zro = dirR < (1.0f / 32768.0f);
    dirR = APrxLoRsqF1(dirR);
    dirR = zro ? 1.0f : dirR;
    dir.x = zro ? 1.0f : dir.x;
    dir.x *= dirR; dir.y *= dirR;
    len = len * 0.5f;
    len *= len;
    const float stretch = (dir.x * dir.x + dir.y * dir.y) * APrxLoRcpF1(fmaxf(fabsf(dir.x), fabsf(dir.y)));
    const float lenx = fmaf(stretch - 1.0f, len, 1.0f), leny = fmaf(-0.5f, len, 1.0f);
    const float lob = fmaf((1.0f / 4.0f - 0.04f) - 0.5f, len, 0.5f);
    const float clp = APrxLoRcpF1(lob);
    // rotated + scaled offset of tap (i,j):  vx = ((i-ppx)*dir.x + (j-ppy)*dir.y)*lenx,  vy = (-(i-ppx)*dir.y + (j-ppy)*dir.x)*leny
    const float Ax = dir.x * lenx, Bx = dir.y * lenx;        // d vx / d i , d vx / d j
    const float Ay = -dir.y * leny, By = dir.x * leny;       // d vy / d i , d vy / d j
    const float vx00 = -(ppx * Ax + ppy * Bx), vy00 = -(ppx * Ay + ppy * By);
    const float4* t = &tile[cy + 1][cx + 1];                 // 'f'
    const float4 tf = t[0], tg = t[1], tj = t[EU_TW], tk = t[EU_TW + 1];
    const float3 min4 = fmin3(fmin3(xyz(tf), fmin3(xyz(tg), xyz(tj))), xyz(tk));
    const float3 max4 = fmax3(fmax3(xyz(tf), fmax3(xyz(tg), xyz(tj))), xyz(tk));
    float3 aC = f3(0.0f);
    float aW = 0.0f;
    // rows j = -1, 0, 1, 2 of the 12-tap cross; offsets built by additions only
    const float vxm = vx00 - Bx, vym = vy00 - By;                               // (0,-1)
    easu_tap_v(aC, aW, vxm, vym, lob, clp, t[-EU_TW]);                           // b (0,-1)
    easu_tap_v(aC, aW, vxm + Ax, vym + Ay, lob, clp, t[-EU_TW + 1]);             // c (1,-1)
    easu_tap_v(aC, aW, vx00 - Ax, vy00 - Ay, lob, clp, t[-1]);                   // e (-1,0)
    easu_tap_v(aC, aW, vx00, vy00, lob, clp, tf);                                // f (0,0)
    easu_tap_v(aC, aW, vx00 + Ax, vy00 + Ay, lob, clp, tg);                      // g (1,0)
    easu_tap_v(aC, aW, fmaf(2.0f, Ax, vx00), fmaf(2.0f, Ay, vy00), lob, clp, t[2]);   // h (2,0)
    const float vx1 = vx00 + Bx, vy1 = vy00 + By;                                // (0,1)
    easu_tap_v(aC, aW, vx1 - Ax, vy1 - Ay, lob, clp, t[EU_TW - 1]);              // i (-1,1)
    easu_tap_v(aC, aW, vx1, vy1, lob, clp, tj);                                  // j (0,1)
    easu_tap_v(aC, aW, vx1 + Ax, vy1 + Ay, lob, clp, tk);                        // k (1,1)
    easu_tap_v(aC, aW, fmaf(2.0f, Ax, vx1), fmaf(2.0f, Ay, vy1), lob, clp, t[EU_TW + 2]);   // l (2,1)
    const float vx2 = fmaf(2.0f, Bx, vx00), vy2 = fmaf(2.0f, By, vy00);          // (0,2)
    easu_tap_v(aC, aW, vx2, vy2, lob, clp, t[2 * EU_TW]);                        // n (0,2)
    easu_tap_v(aC, aW, vx2 + Ax, vy2 + Ay, lob, clp, t[2 * EU_TW + 1]);          // o (1,2)
    const float rw = rcp_fast(aW);
    const float3 pix = fmin3(max4, fmax3(min4, aC * rw));
    st_stream(out.row(y) + x, make_float4(pix.x, pix.y, pix.z, 1.0f));
}

// Exact 2x upscale (the FSR1 "performance" preset, BASELINE config 4): con0 = (0.5, 0.5, -0.25, -0.25), so the output pixels
// (2k+1, 2m+1), (2k+2, 2m+1), (2k+1, 2m+2), (2k+2, 2m+2) all resolve to input texel 'f' = (k, m) with pp = (.25|.75, .25|.75).
// One THREAD per input texel therefore owns a 2x2 output quad: it reads the 12 texels once, evaluates the four FsrEasuSetF analyses
// once, and only the blend of the analyses + the 12 tap weights are per pixel — and those run as packed fp32x2 pairs
// {left pixel, right pixel} (FFMA2/FMUL2/FADD2: one issue slot for two pixels). ncu r01: the one-pixel-per-thread kernel issued
// 485 instructions per output pixel at 77 % issue utilisation (0.62 ms 4K->8K); this one issues ~150.
// Texels k = -1 and k = W-1 (m likewise) own quads that hang over the image edge: those stores are predicated off.
constexpr int E2_BX = 32, E2_BY = 4;                   // input texels ('f' candidates) per CTA -> 64 x 2*E2_BY output pixels
constexpr int E2_MINB = 8;
constexpr int E2_TW = E2_BX + 3, E2_TH = E2_BY + 3;    // staged footprint: columns k-1 .. k+2, rows m-1 .. m+2

struct EasuPx2 { f2 dirx, diry, lenx, leny, lob, clp; };
// dir/len of an output pair from the four shared analyses and the pair's constant bilinear weights (ffx_fsr1.h:349-384)
__device__ __forceinline__ EasuPx2 easu2_direction(const EasuSet& S, const EasuSet& T, const EasuSet& U, const EasuSet& V,
                                                   f2 wS, f2 wT, f2 wU, f2 wV) {
    f2 dx = bc(S.dirX) * wS, dy = bc(S.dirY) * wS, len = bc(S.lenX) * wS;
    len = fma2(bc(S.lenY), wS, len);
    dx = fma2(bc(T.dirX), wT, dx); len = fma2(bc(T.lenX), wT, len); dy = fma2(bc(T.dirY), wT, dy); len = fma2(bc(T.lenY), wT, len);
    dx = fma2(bc(U.dirX), wU, dx); len = fma2(bc(U.lenX), wU, len); dy = fma2(bc(U.dirY), wU, dy); len = fma2(bc(U.lenY), wU, len);
    dx = fma2(bc(V.dirX), wV, dx); len = fma2(bc(V.lenX), wV, len); dy = fma2(bc(V.dirY), wV, dy); len = fma2(bc(V.lenY), wV, len);
    const f2 dirR0 = fma2(dx, dx, dy * dy);
    const bool z0 = dirR0.v.x < (1.0f / 32768.0f), z1 = dirR0.v.y < (1.0f / 32768.0f);
    const f2 dirR = mk(z0 ? 1.0f : APrxLoRsqF1(dirR0.v.x), z1 ? 1.0f : APrxLoRsqF1(dirR0.v.y));
    dx = mk(z0 ? 1.0f : dx.v.x, z1 ? 1.0f : dx.v.y);
    dx = dx * dirR; dy = dy * dirR;
    len = len * bc(0.5f);
    len = len * len;
    const f2 mxd = mk(APrxLoRcpF1(fmaxf(fabsf(dx.v.x), fabsf(dy.v.x))), APrxLoRcpF1(fmaxf(fabsf(dx.v.y), fabsf(dy.v.y))));
    const f2 stretch = fma2(dx, dx, dy * dy) * mxd;
    EasuPx2 r;
    r.dirx = dx; r.diry = dy;
    r.lenx = fma2(stretch - bc(1.0f), len, bc(1.0f));
    r.leny = fma2(bc(-0.5f), len, bc(1.0f));
    r.lob = fma2(bc((1.0f / 4.0f - 0.04f) - 0.5f), len, bc(0.5f));
    r.clp = mk(APrxLoRcpF1(r.lob.v.x), APrxLoRcpF1(r.lob.v.y));
    return r;
}
struct EasuAcc2 { f2 r, g, b, w; };
// one tap for an output pair: weight at the rotated, anisotropically scaled offset (vx, vy) (second half of FsrEasuTapF)
__device__ __forceinline__ void easu2_tap(EasuAcc2& A, f2 vx, f2 vy, const EasuPx2& P, float4 c) {
    const f2 d0 = fma2(vx, vx, vy * vy);
    const f2 d2 = mk(fminf(d0.v.x, P.clp.v.x), fminf(d0.v.y, P.clp.v.y));
    f2 wB = fma2(bc(2.0f / 5.0f), d2, bc(-1.0f));
    f2 wA = fma2(P.lob, d2, bc(-1.0f));
    wB = wB * wB; wA = wA * wA;
    wB = fma2(bc(25.0f / 16.0f), wB, bc(-(25.0f / 16.0f - 1.0f)));
    const f2 w = wB * wA;
    A.r = fma2(bc(c.x), w, A.r); A.g = fma2(bc(c.y), w, A.g); A.b = fma2(bc(c.z), w, A.b);
    A.w = A.w + w;
}

template <int ADDR>
__global__ void __launch_bounds__(E2_BX * E2_BY, E2_MINB) easu_2x_kernel(ImgV in, ImgV out) {
    __shared__ float4 tile[E2_TH][E2_TW];          // rgb + luma
    // 'f' texels of this CTA: k in [k0, k0+32), m in [m0, m0+8) with k0 = 32*bx - 1 (k = -1 owns output column 0)
    const int k0 = (int)blockIdx.x * E2_BX - 1, m0 = (int)blockIdx.y * E2_BY - 1;
    for (int i = threadIdx.y * E2_BX + threadIdx.x; i < E2_TH * E2_TW; i += E2_BX * E2_BY) {
        const int ly = i / E2_TW, lx = i - ly * E2_TW;
        const float3 v = load_addr<ADDR>(in, k0 - 1 + lx, m0 - 1 + ly);
        tile[ly][lx] = make_float4(v.x, v.y, v.z, luma2(v));
    }
    __syncthreads();
    const int k = k0 + (int)threadIdx.x, m = m0 + (int)threadIdx.y;
    const int ox = 2 * k + 1, oy = 2 * m + 1;                        // top-left pixel of the quad
    if (ox >= out.w || oy >= out.h) return;                          // (k, m) beyond the last owning texel
    const float4* t = &tile[threadIdx.y + 1][threadIdx.x + 1];      // 'f'
    float3 min4, max4;
    EasuSet S, T, U, V;
    {   // the four analyses need only the lumas; the colours are re-read from shared memory tap by tap below, so that the 12
        // texels are not live in registers across the whole kernel (48 registers: 2 CTAs per SM became 6)
        const float bL = t[-E2_TW].w, cL = t[-E2_TW + 1].w, eL = t[-1].w, hL = t[2].w;
        const float iL = t[E2_TW - 1].w, lL = t[E2_TW + 2].w, nL = t[2 * E2_TW].w, oL = t[2 * E2_TW + 1].w;
        const float4 tf = t[0], tg = t[1], tj = t[E2_TW], tk = t[E2_TW + 1];
        S = easu_set_shared(bL, eL, tf.w, tg.w, tj.w); T = easu_set_shared(cL, tf.w, tg.w, hL, tk.w);
        U = easu_set_shared(tf.w, iL, tj.w, tk.w, nL); V = easu_set_shared(tg.w, tj.w, tk.w, lL, oL);
        // clamp range of the quad: min/max of f, g, j, k (ffx_fsr1.h:395-398)
        min4 = fmin3(fmin3(xyz(tf), fmin3(xyz(tg), xyz(tj))), xyz(tk));
        max4 = fmax3(fmax3(xyz(tf), fmax3(xyz(tg), xyz(tj))), xyz(tk));
    }
    // the two output rows one after the other: one pair's state live at a time (A/B in profiles/r02_post_variants.txt)
#pragma unroll 1
    for (int row = 0; row < 2; ++row) {                              // output rows oy (pp.y = .25) and oy+1 (pp.y = .75)
        const float ppy = row ? 0.75f : 0.25f;
        const int y = oy + row;
        if (y < 0 || y >= out.h) continue;
        // bilinear weights of the four analyses for {left, right}: (1-ppx)(1-ppy), ppx(1-ppy), (1-ppx)ppy, ppx ppy — exact constants
        const f2 wS = mk(0.75f * (1.0f - ppy), 0.25f * (1.0f - ppy)), wT = mk(0.25f * (1.0f - ppy), 0.75f * (1.0f - ppy));
        const f2 wU = mk(0.75f * ppy, 0.25f * ppy), wV = mk(0.25f * ppy, 0.75f * ppy);
        const EasuPx2 P = easu2_direction(S, T, U, V, wS, wT, wU, wV);
        // rotated + scaled offset of tap (i,j):  vx = ((i-ppx)*dir.x + (j-ppy)*dir.y)*lenx,  vy = (-(i-ppx)*dir.y + (j-ppy)*dir.x)*leny
        const f2 Ax = P.dirx * P.lenx, Bx = P.diry * P.lenx;         // d vx / d i , d vx / d j
        const f2 Ay = mk(-P.diry.v.x, -P.diry.v.y) * P.leny, By = P.dirx * P.leny;
        const f2 nppy = bc(-ppy);
        const f2 vx00 = fma2(nppy, Bx, mk(-0.25f, -0.75f) * Ax), vy00 = fma2(nppy, By, mk(-0.25f, -0.75f) * Ay);
        EasuAcc2 A; A.r = A.g = A.b = A.w = bc(0.0f);
        const f2 vxm = vx00 - Bx, vym = vy00 - By;                                        // (0,-1)
        easu2_tap(A, vxm, vym, P, t[-E2_TW]);                                                     // b (0,-1)
        easu2_tap(A, vxm + Ax, vym + Ay, P, t[-E2_TW + 1]);                                           // c (1,-1)
        easu2_tap(A, vx00 - Ax, vy00 - Ay, P, t[-1]);                                         // e (-1,0)
        easu2_tap(A, vx00, vy00, P, t[0]);                                                   // f (0,0)
        easu2_tap(A, vx00 + Ax, vy00 + Ay, P, t[1]);                                         // g (1,0)
        easu2_tap(A, fma2(bc(2.0f), Ax, vx00), fma2(bc(2.0f), Ay, vy00), P, t[2]);           // h (2,0)
        const f2 vx1 = vx00 + Bx, vy1 = vy00 + By;                                         // (0,1)
        easu2_tap(A, vx1 - Ax, vy1 - Ay, P, t[E2_TW - 1]);                                           // i (-1,1)
        easu2_tap(A, vx1, vy1, P, t[E2_TW]);                                                     // j (0,1)
        easu2_tap(A, vx1 + Ax, vy1 + Ay, P, t[E2_TW + 1]);                                           // k (1,1)
        easu2_tap(A, fma2(bc(2.0f), Ax, vx1), fma2(bc(2.0f), Ay, vy1), P, t[E2_TW + 2]);             // l (2,1)
        const f2 vx2 = fma2(bc(2.0f), Bx, vx00), vy2 = fma2(bc(2.0f), By, vy00);           // (0,2)
        easu2_tap(A, vx2, vy2, P, t[2 * E2_TW]);                                                     // n (0,2)
        easu2_tap(A, vx2 + Ax, vy2 + Ay, P, t[2 * E2_TW + 1]);                                           // o (1,2)
        const f2 rw = rcp2(A.w);                                                           // ARcpF1 = rcp() in the HLSL
        const f2 cr = A.r * rw, cg = A.g * rw, cb = A.b * rw;
        float4* dst = out.row(y);
        if (ox >= 0) st_stream(dst + ox, make_float4(fminf(max4.x, fmaxf(min4.x, cr.v.x)), fminf(max4.y, fmaxf(min4.y, cg.v.x)),
                                                     fminf(max4.z, fmaxf(min4.z, cb.v.x)), 1.0f));
        if (ox + 1 < out.w) st_stream(dst + ox + 1, make_float4(fminf(max4.x, fmaxf(min4.x, cr.v.y)), fminf(max4.y, fmaxf(min4.y, cg.v.y)),
                                                                fminf(max4.z, fmaxf(min4.z, cb.v.y)), 1.0f));
    }
}

extern "C" int vq_fsr_easu(VqContext* ctx, const uint32_t con[16], int address_mode, VqImage in, VqImage out, void* stream) {
    int rc = vq_enter(ctx); if (rc) return rc;
    VQ_MARK("FSR-EASU CS");
    VQ_REQUIRE(con, "easu_const is null");
    VQ_REQUIRE(vq_image_ok(in) && vq_image_ok(out), "bad image descriptor");
    VQ_REQUIRE(address_mode == VQ_ADDRESS_WRAP || address_mode == VQ_ADDRESS_CLAMP, "easu: unknown address mode");
    VQ_REQUIRE(in.ptr != out.ptr, "easu: in-place is not supported");
    EasuCon c; memcpy(&c, con, 16);
    cudaStream_t st = (cudaStream_t)stream;
    // ratio <= 1 (upscale or 1:1) and the footprint of a 32x16 output tile fits the staged tile: shared-memory path
    const bool up = c.c0x > 0.0f && c.c0y > 0.0f && c.c0x <= 1.0f && c.c0y <= 1.0f;
    // exact 2x (FsrEasuCon(w, h, w, h, 2w, 2h)): one thread per input texel, a 2x2 output quad each
    const bool x2 = c.c0x == 0.5f && c.c0y == 0.5f && c.c0z == -0.25f && c.c0w == -0.25f && out.width == 2 * in.width && out.height == 2 * in.height;
    if (x2) {
        // 'f' texels k = -1 .. W-1, m = -1 .. H-1
        const dim3 grid((in.width + 1 + E2_BX - 1) / E2_BX, (in.height + 1 + E2_BY - 1) / E2_BY);
        if (address_mode == VQ_ADDRESS_WRAP) easu_2x_kernel<VQ_ADDRESS_WRAP><<<grid, dim3(E2_BX, E2_BY), 0, st>>>(make_view(in), make_view(out));
        else                                 easu_2x_kernel<VQ_ADDRESS_CLAMP><<<grid, dim3(E2_BX, E2_BY), 0, st>>>(make_view(in), make_view(out));
    } else if (up) {
        const dim3 grid((out.width + EU_BX - 1) / EU_BX, (out.height + EU_BY - 1) / EU_BY);
        if (address_mode == VQ_ADDRESS_WRAP) easu_up_kernel<VQ_ADDRESS_WRAP><<<grid, dim3(EU_BX, EU_BY), 0, st>>>(make_view(in), make_view(out), c);
        else                                 easu_up_kernel<VQ_ADDRESS_CLAMP><<<grid, dim3(EU_BX, EU_BY), 0, st>>>(make_view(in), make_view(out), c);
    } else {
        const dim3 grid((out.width + ST_BX - 1) / ST_BX, (out.height + ST_BY - 1) / ST_BY);
        if (address_mode == VQ_ADDRESS_WRAP) easu_kernel<VQ_ADDRESS_WRAP><<<grid, dim3(ST_BX, ST_BY), 0, st>>>(make_view(in), make_view(out), c);
        else                                 easu_kernel<VQ_ADDRESS_CLAMP><<<grid, dim3(ST_BX, ST_BY), 0, st>>>(make_view(in), make_view(out), c);
    }
    return vq_check_launch("fsr_easu");
}

// =============================================================================================
// K10 SPD — SPD/ffx_spd.h:557-835 (LDS ordering), reduction (v0+v1+v2+v3)*0.25 (AMDFidelityFX.hlsl:463-466)
//
// One 256-thread block per 64x64 source tile. Thread t owns a 4x4 source patch; patches are laid out
// in Morton order inside each warp, so levels 1-2 are pure register work and levels 3-4 are warp
// shuffles; levels 5-6 go through 1 KB of shared memory. A global ticket (atomicAdd + __threadfence)
// elects the last block, which reduces level 6 -> 7..12 out of shared memory.
// Operand order per level (SURVEY.md §9): levels 1 and 7 sum (x,y),(x,y+1),(x+1,y),(x+1,y+1);
// every other level sums (x,y),(x+1,y),(x,y+1),(x+1,y+1).
// =============================================================================================
struct SpdLevels { float4* p[12]; int w[12], h[12], pitch4[12]; };

// SpdReduce4 is the callback the integration supplies: the engine's colour wrapper averages (AMDFidelityFX.hlsl:463-466),
// its live depth-pyramid use takes a MIN (DownsampleDepth.hlsl:72) and the CPU HDRI mip filter this backend also routes
// through the same kernel is min(rgb), alpha = 1 (DXGIUtils.cpp:305-311).
enum { SPD_AVG = 0, SPD_MIN_RGB_A1 = 1 };
template <int OP>
__device__ __forceinline__ float4 spd_reduce4(float4 v0, float4 v1, float4 v2, float4 v3) {
    if (OP == SPD_AVG)
        return make_float4(((v0.x + v1.x) + v2.x + v3.x) * 0.25f, ((v0.y + v1.y) + v2.y + v3.y) * 0.25f,
                           ((v0.z + v1.z) + v2.z + v3.z) * 0.25f, ((v0.w + v1.w) + v2.w + v3.w) * 0.25f);
    return make_float4(fminf(v0.x, fminf(v1.x, fminf(v2.x, v3.x))), fminf(v0.y, fminf(v1.y, fminf(v2.y, v3.y))),
                       fminf(v0.z, fminf(v1.z, fminf(v2.z, v3.z))), 1.0f);
}
__device__ __forceinline__ float4 shfl4(float4 v, int lane) {
    return make_float4(__shfl_sync(0xffffffffu, v.x, lane), __shfl_sync(0xffffffffu, v.y, lane),
                       __shfl_sync(0xffffffffu, v.z, lane), __shfl_sync(0xffffffffu, v.w, lane));
}
__device__ __forceinline__ void spd_store(const SpdLevels& L, int lvl /*1-based*/, int mips, int x, int y, float4 v) {
    if (lvl <= mips && x < L.w[lvl - 1] && y < L.h[lvl - 1]) L.p[lvl - 1][(size_t)y * L.pitch4[lvl - 1] + x] = v;
}

template <int OP>
__global__ void __launch_bounds__(256) spd_kernel(ImgV src, SpdLevels L, int mips, uint32_t numWorkGroups,
                                                  uint32_t offX, uint32_t offY, uint32_t* counter) {
    __shared__ float4 s4[4][4];        // level-4 texels of this tile
    __shared__ float4 s5[2][2];
    __shared__ uint32_t sTicket;
    __shared__ float4 sTail[32 * 32];  // level 7 and beyond, ping-pong halves handled by index ranges
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    // Morton decode of the lane (5 bits: x0 y0 x1 y1 x2) -> 8 wide x 4 high patches per warp
    const int lx = (lane & 1) | ((lane >> 1) & 2) | ((lane >> 2) & 4);
    const int ly = ((lane >> 1) & 1) | ((lane >> 2) & 2);
    // warps tile the 16x16 patch grid as 2 columns x 4 rows of 8x4 patch blocks
    const int px = (warp & 1) * 8 + lx, py = (warp >> 1) * 4 + ly;          // patch coords in the tile
    const int tileX = blockIdx.x + offX, tileY = blockIdx.y + offY;
    const int sx0 = tileX * 64 + px * 4, sy0 = tileY * 64 + py * 4;        // source texel of the patch

    // ---- load the 4x4 patch (zeros outside the image: they only ever feed dropped texels) ----
    float4 t[4][4];
#pragma unroll
    for (int j = 0; j < 4; ++j)
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int sx = sx0 + i, sy = sy0 + j;
            t[j][i] = (sx < src.w && sy < src.h) ? ld_stream(src.row(sy) + sx) : make_float4(0, 0, 0, 0);   // (A/B: through L1 is 8 % slower)
        }
    // ---- level 1: 2x2 per thread, column-major operand order (ffx_spd.h:468-476) ----
    float4 l1[2][2];
#pragma unroll
    for (int j = 0; j < 2; ++j)
#pragma unroll
        for (int i = 0; i < 2; ++i) {
            l1[j][i] = spd_reduce4<OP>(t[2 * j][2 * i], t[2 * j + 1][2 * i], t[2 * j][2 * i + 1], t[2 * j + 1][2 * i + 1]);
            spd_store(L, 1, mips, tileX * 32 + px * 2 + i, tileY * 32 + py * 2 + j, l1[j][i]);
        }
    if (mips <= 1) return;
    // ---- level 2: 1 per thread, row-major operand order (ffx_spd.h:590-595) ----
    const float4 l2 = spd_reduce4<OP>(l1[0][0], l1[0][1], l1[1][0], l1[1][1]);
    spd_store(L, 2, mips, tileX * 16 + px, tileY * 16 + py, l2);
    // ---- level 3: quad of lanes (Morton bits 0,1) ----
    const int q = lane & ~3;
    const float4 l3 = spd_reduce4<OP>(shfl4(l2, q), shfl4(l2, q | 1), shfl4(l2, q | 2), shfl4(l2, q | 3));
    if (mips >= 3 && (lane & 3) == 0) spd_store(L, 3, mips, tileX * 8 + (px >> 1), tileY * 8 + (py >> 1), l3);
    // ---- level 4: 16 lanes (Morton bits 2,3) ----
    const int g = lane & ~15;
    const float4 l4 = spd_reduce4<OP>(shfl4(l3, g), shfl4(l3, g | 4), shfl4(l3, g | 8), shfl4(l3, g | 12));
    if ((lane & 15) == 0) {
        if (mips >= 4) spd_store(L, 4, mips, tileX * 4 + (px >> 2), tileY * 4 + (py >> 2), l4);
        s4[py >> 2][px >> 2] = l4;
    }
    __syncthreads();
    // ---- level 5 and 6 through shared memory ----
    if (tid < 4 && mips >= 5) {
        const int x = tid & 1, y = tid >> 1;
        const float4 v = spd_reduce4<OP>(s4[2 * y][2 * x], s4[2 * y][2 * x + 1], s4[2 * y + 1][2 * x], s4[2 * y + 1][2 * x + 1]);
        spd_store(L, 5, mips, tileX * 2 + x, tileY * 2 + y, v);
        s5[y][x] = v;
    }
    __syncthreads();
    if (tid == 0 && mips >= 6) {
        const float4 v = spd_reduce4<OP>(s5[0][0], s5[0][1], s5[1][0], s5[1][1]);
        spd_store(L, 6, mips, tileX, tileY, v);
    }
    if (mips <= 6) return;

    // ---- elect the last block (SpdExitWorkgroup, ffx_spd.h:391-400) ----
    __threadfence();                       // publish this block's level-6 texel device-wide
    __syncthreads();
    if (tid == 0) sTicket = atomicAdd(counter, 1u);
    __syncthreads();
    if (sTicket != numWorkGroups - 1) return;
    if (tid == 0) *counter = 0;            // SpdResetAtomicCounter: ready for the next launch
    __threadfence();

    // ---- tail: level 6 (<= 64x64, read through L2) -> 7 (column-major order), then 8..12 row-major ----
    const int w6 = L.w[5], h6 = L.h[5];
    const float4* p6 = L.p[5];
    const int pitch6 = L.pitch4[5];
    int cw = L.w[6], ch = L.h[6];          // level 7 size
    for (int idx = tid; idx < cw * ch; idx += 256) {
        const int x = idx % cw, y = idx / cw;
        const float4 v0 = __ldcg(p6 + (size_t)(2 * y) * pitch6 + 2 * x);
        const float4 v1 = __ldcg(p6 + (size_t)(2 * y + 1) * pitch6 + 2 * x);
        const float4 v2 = __ldcg(p6 + (size_t)(2 * y) * pitch6 + 2 * x + 1);
        const float4 v3 = __ldcg(p6 + (size_t)(2 * y + 1) * pitch6 + 2 * x + 1);
        const float4 v = spd_reduce4<OP>(v0, v1, v2, v3);
        spd_store(L, 7, mips, x, y, v);
        sTail[y * 32 + x] = v;
    }
    (void)w6; (void)h6;
    __syncthreads();
    // levels 8.. : source rows live at stride 32 in sTail; results overwrite in place after a barrier
    for (int lvl = 8; lvl <= mips; ++lvl) {
        const int nw = L.w[lvl - 1], nh = L.h[lvl - 1];
        float4 v = make_float4(0, 0, 0, 0);
        const bool active = tid < nw * nh;             // nw*nh <= 16*16
        int x = 0, y = 0;
        if (active) {
            x = tid % nw; y = tid / nw;
            v = spd_reduce4<OP>(sTail[(2 * y) * 32 + 2 * x], sTail[(2 * y) * 32 + 2 * x + 1],
                            sTail[(2 * y + 1) * 32 + 2 * x], sTail[(2 * y + 1) * 32 + 2 * x + 1]);
            spd_store(L, lvl, mips, x, y, v);
        }
        __syncthreads();
        if (active) sTail[y * 32 + x] = v;
        __syncthreads();
    }
}

extern "C" int vq_spd_downsample(VqContext* ctx, const VqSpdConstants* c, VqImage src, const VqImage* mips, void* stream) {
    int rc = vq_enter(ctx); if (rc) return rc;
    VQ_MARK("FFX-SPD CS");
    VQ_REQUIRE(c && mips, "constants/mips is null");
    VQ_REQUIRE(vq_image_ok(src), "bad source image");
    VQ_REQUIRE(c->mips >= 1 && c->mips <= 12, "spd: 1..12 destination mips");
    VQ_REQUIRE(src.width <= 4096 && src.height <= 4096, "spd: source up to 4096^2 (ffx_spd.h limit)");
    SpdLevels L; memset(&L, 0, sizeof(L));
    for (uint32_t i = 0; i < c->mips; ++i) {
        VQ_REQUIRE(vq_image_ok(mips[i]), "bad mip image");
        VQ_REQUIRE(mips[i].width == (src.width >> (i + 1)) && mips[i].height == (src.height >> (i + 1)),
                   "spd: mip i must be floor-halved (src >> (i+1))");
        L.p[i] = (float4*)mips[i].ptr; L.w[i] = mips[i].width; L.h[i] = mips[i].height; L.pitch4[i] = (int)(mips[i].pitch_bytes / 16);
    }
    // group grid: same arithmetic as SpdSetup (ffx_spd.h:336-343) for a full-image rect at the given offset
    const uint32_t gx = (uint32_t)(src.width + 63) / 64 - c->workGroupOffset[0];
    const uint32_t gy = (uint32_t)(src.height + 63) / 64 - c->workGroupOffset[1];
    VQ_REQUIRE(gx >= 1 && gy >= 1 && gx * gy == c->numWorkGroups, "spd: numWorkGroups does not match the image / offset (use vq_spd_setup)");
    spd_kernel<SPD_AVG><<<dim3(gx, gy), 256, 0, (cudaStream_t)stream>>>(make_view(src), L, (int)c->mips, c->numWorkGroups,
                                                               c->workGroupOffset[0], c->workGroupOffset[1], vq_spd_ticket(ctx));
    return vq_check_launch("spd_downsample");
}

// K11 through the SPD kernel: the whole HDRI min-pyramid in ONE launch (levels 1..levels-1 of the packed pyramid).
int vq_spd_min_pyramid(VqContext* ctx, VqPyramid hd, cudaStream_t stream) {
    SpdLevels L; memset(&L, 0, sizeof(L));
    const int mips = hd.levels - 1;
    float4* base = (float4*)hd.ptr;
    for (int i = 0; i < mips; ++i) {
        L.p[i] = base + vq_pyramid_offset(hd.width, hd.height, i + 1);
        L.w[i] = hd.width >> (i + 1); L.h[i] = hd.height >> (i + 1); L.pitch4[i] = L.w[i];
    }
    ImgV src; src.p = base; src.w = hd.width; src.h = hd.height; src.pitch4 = hd.width;
    const unsigned gx = (unsigned)(hd.width + 63) / 64, gy = (unsigned)(hd.height + 63) / 64;
    spd_kernel<SPD_MIN_RGB_A1><<<dim3(gx, gy), 256, 0, stream>>>(src, L, mips, gx * gy, 0u, 0u, vq_spd_ticket(ctx));
    return vq_check_launch("hdri_build_mips(spd)");
}

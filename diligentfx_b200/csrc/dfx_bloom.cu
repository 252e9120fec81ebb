// dfx_bloom.cu — Bloom B1-B4 as sm_100a kernels.
// Reference: PostProcess/Bloom/src/Bloom.cpp:288-393 (one draw per level: :324-337 down, :355-375 up, :387-391 composite) +
//            Shaders/PostProcess/Bloom/private/Bloom_Compute{Prefiltered,Downsampled,Upsampled}Texture.fx.
//
// Three kernel families:
//   * generic (any size ratio): one thread per output texel, the shader's 13 / 9 bilinear taps gathered from HBM;
//   * streaming (exact 2:1 levels — every large level of the pyramid): a WARP walks down a column band; each lane loads its
//     own texels with 128-bit coalesced loads exactly once and receives its horizontal neighbours' through warp shuffles, the
//     vertical filter runs over a register sliding window. No shared memory, no barriers: the kernels are bound by HBM;
//   * tail (levels of <= 2K texels, a dozen dependent launches in the reference): ONE thread-block cluster runs all of them,
//     down to the top of the pyramid and back up, with a cluster barrier between levels (the planes stay in L2).
#include "dfx_common.cuh"
#include "dfx_tonemap.cuh"
#include <cooperative_groups.h>
#include <algorithm>
#include <atomic>

namespace dfx
{

// =====================================================================================================================
// Bloom. Levels are RGBA32F planes (rgb used). B1/B2 sample with linear + border(0) addressing, B3/B4 with linear + clamp.
// The output pixel centre in UV is (p + 0.5) / output size; taps are offset by whole input texels.
// =====================================================================================================================
template <bool BORDER>
DFX_HD float3 tap3(const View<const float4>& t, float u, float v)
{
    return xyz(BORDER ? sample_linear_border(t, u, v) : sample_linear_clamp(t, u, v));
}

struct Taps13
{
    float3 A, B, C, D, E, F, G, H, I, J, K, L, M;
};
DFX_HD Taps13 taps13(const View<const float4>& in, float u, float v)
{
    const float tx = 1.0f / float(in.w), ty = 1.0f / float(in.h);
    Taps13      t;
    t.A = tap3<true>(in, u + tx * -2.0f, v + ty * +2.0f);
    t.B = tap3<true>(in, u + tx * +0.0f, v + ty * +2.0f);
    t.C = tap3<true>(in, u + tx * +2.0f, v + ty * +2.0f);
    t.D = tap3<true>(in, u + tx * -2.0f, v + ty * +0.0f);
    t.E = tap3<true>(in, u + tx * +0.0f, v + ty * +0.0f);
    t.F = tap3<true>(in, u + tx * +2.0f, v + ty * +0.0f);
    t.G = tap3<true>(in, u + tx * -2.0f, v + ty * -2.0f);
    t.H = tap3<true>(in, u + tx * +0.0f, v + ty * -2.0f);
    t.I = tap3<true>(in, u + tx * +2.0f, v + ty * -2.0f);
    t.J = tap3<true>(in, u + tx * -1.0f, v + ty * +1.0f);
    t.K = tap3<true>(in, u + tx * +1.0f, v + ty * +1.0f);
    t.L = tap3<true>(in, u + tx * -1.0f, v + ty * -1.0f);
    t.M = tap3<true>(in, u + tx * +1.0f, v + ty * -1.0f);
    return t;
}

// B1: Bloom_ComputePrefilteredTexture.fx:37-83 — 13 taps in 5 Karis-weighted groups, soft-knee threshold
__global__ void __launch_bounds__(256) bloom_prefilter_kernel(dfx_bloom_attribs A, View<const float4> in, View<float4> out, int y0, int y1)
{
    const PixelXY pix = cta_pixel(y0);
    const int     x = pix.x, y = pix.y;
    if (x >= out.w || y >= y1) return;
    const float  u = (float(x) + 0.5f) / float(out.w), v = (float(y) + 0.5f) / float(out.h);
    const Taps13 t = taps13(in, u, v);
    float3       g[5];
    g[0] = (t.A + t.B + t.D + t.E) / 4.0f;
    g[1] = (t.B + t.C + t.E + t.F) / 4.0f;
    g[2] = (t.D + t.E + t.G + t.H) / 4.0f;
    g[3] = (t.E + t.F + t.H + t.I) / 4.0f;
    g[4] = (t.J + t.K + t.L + t.M) / 4.0f;
    float3 csum = make_float3(0.f, 0.f, 0.f);
    float  wsum = 0.0f;
#pragma unroll
    for (int i = 0; i < 5; ++i)
    {
        const float w = (i == 4 ? 0.5f : 0.125f) * (1.0f / (1.0f + luminance(g[i])));
        csum = csum + g[i] * w;
        wsum += 1.0f * w;
    }
    const float3 c = csum / (wsum + 1.0e-5f);
    // Prefilter :24-35
    const float brightness = fmaxf(c.x, fmaxf(c.y, c.z));
    const float knee       = A.Threshold * A.SoftTreshold;
    float       soft       = brightness - A.Threshold + knee;
    soft                   = fminf(fmaxf(soft, 0.0f), 2.0f * knee);
    soft                   = soft * soft * 0.25f / (knee + 1.0e-5f);
    float contribution     = fmaxf(soft, brightness - A.Threshold);
    contribution /= fmaxf(brightness, 1.0e-5f);
    out.at(x, y) = f4(c * contribution, 0.0f);
}

// B2: Bloom_ComputeDownsampledTexture.fx:11-41 — 13-tap downsample, weights 1/32, 1/16, 1/8
__global__ void __launch_bounds__(256) bloom_downsample_kernel(View<const float4> in, View<float4> out, int y0, int y1)
{
    const PixelXY pix = cta_pixel(y0);
    const int     x = pix.x, y = pix.y;
    if (x >= out.w || y >= y1) return;
    const float  u = (float(x) + 0.5f) / float(out.w), v = (float(y) + 0.5f) / float(out.h);
    const Taps13 t = taps13(in, u, v);
    float3       o = make_float3(0.f, 0.f, 0.f);
    o = o + (t.A + t.C + t.G + t.I) * 0.03125f;
    o = o + (t.B + t.D + t.F + t.H) * 0.0625f;
    o = o + (t.E + t.J + t.K + t.L + t.M) * 0.125f;
    out.at(x, y) = f4(o, 0.0f);
}

DFX_HD float3 tent9(const View<const float4>& lo, float u, float v)
{
    const float  tx = 1.0f / float(lo.w), ty = 1.0f / float(lo.h);
    const float3 A = tap3<false>(lo, u - tx, v + ty), B = tap3<false>(lo, u, v + ty), C = tap3<false>(lo, u + tx, v + ty);
    const float3 D = tap3<false>(lo, u - tx, v), E = tap3<false>(lo, u, v), F = tap3<false>(lo, u + tx, v);
    const float3 G = tap3<false>(lo, u - tx, v - ty), H = tap3<false>(lo, u, v - ty), I = tap3<false>(lo, u + tx, v - ty);
    float3       s = E * 0.25f;
    s = s + (B + D + F + H) * 0.125f;
    s = s + (A + C + G + I) * 0.0625f;
    return s;
}

// B3: Bloom_ComputeUpsampledTexture.fx:20-54 (uInstID == 0): same-level downsample + 3x3 tent of the coarser level
__global__ void __launch_bounds__(256) bloom_upsample_kernel(View<const float4> same, View<const float4> coarser, View<float4> out, int y0, int y1)
{
    const PixelXY pix = cta_pixel(y0);
    const int     x = pix.x, y = pix.y;
    if (x >= out.w || y >= y1) return;
    const float  u = (float(x) + 0.5f) / float(out.w), v = (float(y) + 0.5f) / float(out.h);
    const float3 s = tent9(coarser, u, v);
    const float3 c = tap3<false>(same, u, v);
    out.at(x, y)   = f4(c + s, 0.0f);
}

// B4: final composite (uInstID != 0), :45-48
__global__ void __launch_bounds__(256) bloom_composite_kernel(dfx_bloom_attribs A, View<const float4> color, View<const float4> up0,
                                                              View<float4> out, int y0, int y1)
{
    const PixelXY pix = cta_pixel(y0);
    const int     x = pix.x, y = pix.y;
    if (x >= out.w || y >= y1) return;
    const float  u = (float(x) + 0.5f) / float(out.w), v = (float(y) + 0.5f) / float(out.h);
    const float3 s = tent9(up0, u, v);
    const float3 c = tap3<false>(color, u, v);
    st_cs(&out.at(x, y), f4(lerp3(c, c + A.Intensity * s, A.AlphaInterpolation), 0.0f));
}

// ---------------------------------------------------------------------------------------------------------------------
// Exact-2:1 fast paths. When the finer plane is exactly twice the coarser one in both dimensions (every large level of the
// pyramid: 3840x2160 -> 1920x1080 -> 960x540 -> 480x270 -> 240x135), all sample positions fall on texel corners
// (down-sampling) or on quarter-texel offsets (up-sampling), exactly representable in the sampler's 8 sub-texel bits. The
// bilinear weights are then the constants 1/4 (corner average) resp. {1/4, 3/4}, so the taps can be evaluated from a
// shared-memory tile of the source with fixed weights instead of 13x4 / 9x4 gathered texels per pixel.
// ---------------------------------------------------------------------------------------------------------------------
constexpr int kDnTileW = 68, kDnTileH = 20; // source texels staged for a 32x8 output tile of B1/B2: (2*32 + 4) x (2*8 + 4)
constexpr int kDnCornW = 67, kDnCornH = 19; // texel corners inside that tile

// B1 / B2 on an exact 2:1 level. Stage 1: the CTA stages the 68x20 source tile (out-of-range texels = 0: border addressing).
// Stage 2: the 67x19 corner averages (each bilinear tap of the shader IS one corner average). Stage 3: 13 taps per output.
// stages 2 and 3, from a staged source tile
template <bool PREFILTER>
__device__ __forceinline__ void bloom_down2x_from_tile(const dfx_bloom_attribs& A, const float4 (&tile)[kDnTileH][kDnTileW], float4 (&corner)[kDnCornH][kDnCornW],
                                                       View<float4> out, int ox0, int oy0, int y1)
{
    const int tid = threadIdx.y * 32 + threadIdx.x;
    for (int i = tid; i < kDnCornW * kDnCornH; i += 256)
    {
        const int    ly = i / kDnCornW, lx = i - ly * kDnCornW;
        const float4 a = tile[ly][lx], b = tile[ly][lx + 1], c = tile[ly + 1][lx], d = tile[ly + 1][lx + 1];
        corner[ly][lx] = (a * 0.25f + b * 0.25f) + (c * 0.25f + d * 0.25f);
    }
    __syncthreads();
    const int x = ox0 + threadIdx.x, y = oy0 + threadIdx.y;
    if (x >= out.w || y >= y1) return;
    // output centre = corner (2*lx + 2, 2*ly + 2) of the tile; tap offset (i, j) texels -> corner (cx + i, cy + j)
    const int cx = 2 * threadIdx.x + 2, cy = 2 * threadIdx.y + 2;
    auto      T  = [&](int i, int j) { return xyz(corner[cy + j][cx + i]); };
    const float3 tA = T(-2, +2), tB = T(0, +2), tC = T(+2, +2), tD = T(-2, 0), tE = T(0, 0), tF = T(+2, 0), tG = T(-2, -2), tH = T(0, -2), tI = T(+2, -2);
    const float3 tJ = T(-1, +1), tK = T(+1, +1), tL = T(-1, -1), tM = T(+1, -1);
    if (!PREFILTER)
    {
        float3 o = make_float3(0.f, 0.f, 0.f);
        o = o + (tA + tC + tG + tI) * 0.03125f;
        o = o + (tB + tD + tF + tH) * 0.0625f;
        o = o + (tE + tJ + tK + tL + tM) * 0.125f;
        out.at(x, y) = f4(o, 0.0f);
        return;
    }
    float3 g[5];
    g[0] = (tA + tB + tD + tE) * 0.25f;
    g[1] = (tB + tC + tE + tF) * 0.25f;
    g[2] = (tD + tE + tG + tH) * 0.25f;
    g[3] = (tE + tF + tH + tI) * 0.25f;
    g[4] = (tJ + tK + tL + tM) * 0.25f;
    float3 csum = make_float3(0.f, 0.f, 0.f);
    float  wsum = 0.0f;
#pragma unroll
    for (int i = 0; i < 5; ++i)
    {
        const float w = (i == 4 ? 0.5f : 0.125f) * frcp(1.0f + luminance(g[i]));
        csum = csum + g[i] * w;
        wsum += w;
    }
    const float3 c = csum * frcp(wsum + 1.0e-5f);
    const float brightness = fmaxf(c.x, fmaxf(c.y, c.z));
    const float knee       = A.Threshold * A.SoftTreshold;
    float       soft       = fminf(fmaxf(brightness - A.Threshold + knee, 0.0f), 2.0f * knee);
    soft                   = soft * soft * 0.25f * frcp(knee + 1.0e-5f);
    const float contribution = fmaxf(soft, brightness - A.Threshold) * frcp(fmaxf(brightness, 1.0e-5f));
    out.at(x, y) = f4(c * contribution, 0.0f);
}

template <bool PREFILTER>
__global__ void __launch_bounds__(256) bloom_down2x_kernel(dfx_bloom_attribs A, View<const float4> in, View<float4> out, int y0, int y1)
{
    __shared__ float4 tile[kDnTileH][kDnTileW];
    __shared__ float4 corner[kDnCornH][kDnCornW];
    const int tid = threadIdx.y * 32 + threadIdx.x;
    const int ox0 = blockIdx.x * 32, oy0 = y0 + blockIdx.y * 8;
    const int sx0 = 2 * ox0 - 2, sy0 = 2 * oy0 - 2;
    for (int i = tid; i < kDnTileW * kDnTileH; i += 256)
    {
        const int ly = i / kDnTileW, lx = i - ly * kDnTileW;
        tile[ly][lx] = load0(in, sx0 + lx, sy0 + ly);
    }
    __syncthreads();
    bloom_down2x_from_tile<PREFILTER>(A, tile, corner, out, ox0, oy0, y1);
}


// B3 / B4 on an exact 1:2 level: the 3x3 tent of bilinear taps of the coarser level collapses to a separable 4-tap filter
// whose weights depend only on the parity of the output coordinate:
//   even x = 2k : texels k-2..k+1 weigh (1, 5, 7, 3)/16      odd x = 2k+1 : texels k-1..k+2 weigh (3, 7, 5, 1)/16
// (position x/2 - 1/4 resp. + 1/4 -> bilinear {1/4, 3/4}, convolved with the tent {1/4, 1/2, 1/4}). Clamp addressing is
// applied when the 20x8 coarse tile is staged. COMPOSITE selects B4 (lerp with Intensity) instead of B3 (plain add).

template <bool COMPOSITE, bool TONEMAP = false, bool LUM_DEV = false>
__global__ void __launch_bounds__(256) bloom_up2x_kernel(dfx_bloom_attribs A, View<const float4> fine, View<const float4> coarser, View<float4> out, int y0, int y1,
                                                         ToneMapIn tm = ToneMapIn{})
{
    if (LUM_DEV) tm.ave_log_lum = fmaxf(0.05f, __ldg(tm.ave_log_lum_dev)); // GetAverageSceneLuminance (AtmosphereShadersCommon.fxh:188-197)
    // A CTA of 256 threads produces 64x16 outputs; every thread a 2x2 block that shares one 5x5 coarse footprint, so the
    // shared-memory traffic is 25 LDS.128 per four outputs (the kernel would otherwise be bound by smem bandwidth, not HBM).
    __shared__ float4 tile[12][36];
    const int tid = threadIdx.y * 32 + threadIdx.x;
    const int ox0 = blockIdx.x * 64, oy0 = y0 + blockIdx.y * 16; // y0 is even for whole-level launches (checked by the caller)
    const int cx0 = (ox0 >> 1) - 2, cy0 = (oy0 >> 1) - 2;
    for (int i = tid; i < 12 * 36; i += 256)
    {
        const int ly = i / 36, lx = i - ly * 36;
        tile[ly][lx] = loadc(coarser, cx0 + lx, cy0 + ly);
    }
    __syncthreads();
    const int x = ox0 + 2 * threadIdx.x, y = oy0 + 2 * threadIdx.y;
    if (x >= out.w || y >= y1) return;
    float3 E[5], O[5]; // per coarse row: the horizontal 4-tap result for the even / odd output column
#pragma unroll
    for (int j = 0; j < 5; ++j)
    {
        const float3 c0 = xyz(tile[threadIdx.y + j][threadIdx.x]), c1 = xyz(tile[threadIdx.y + j][threadIdx.x + 1]), c2 = xyz(tile[threadIdx.y + j][threadIdx.x + 2]);
        const float3 c3 = xyz(tile[threadIdx.y + j][threadIdx.x + 3]), c4 = xyz(tile[threadIdx.y + j][threadIdx.x + 4]);
        E[j] = c0 * (1.f / 16) + c1 * (5.f / 16) + c2 * (7.f / 16) + c3 * (3.f / 16);
        O[j] = c1 * (3.f / 16) + c2 * (7.f / 16) + c3 * (5.f / 16) + c4 * (1.f / 16);
    }
    const float3 s00 = E[0] * (1.f / 16) + E[1] * (5.f / 16) + E[2] * (7.f / 16) + E[3] * (3.f / 16);
    const float3 s10 = O[0] * (1.f / 16) + O[1] * (5.f / 16) + O[2] * (7.f / 16) + O[3] * (3.f / 16);
    const float3 s01 = E[1] * (3.f / 16) + E[2] * (7.f / 16) + E[3] * (5.f / 16) + E[4] * (1.f / 16);
    const float3 s11 = O[1] * (3.f / 16) + O[2] * (7.f / 16) + O[3] * (5.f / 16) + O[4] * (1.f / 16);
    auto emit = [&](int px, int py, float3 s) {
        if (px >= out.w || py >= y1) return;
        const float3 c = xyz(__ldg(&fine.at(px, py))); // linear sampler at the texel centre == the texel
        if (COMPOSITE)
        {
            float3 o = lerp3(c, c + A.Intensity * s, A.AlphaInterpolation);
            if (TONEMAP)
            {
                o = tone_map_rt(tm.attribs.iToneMappingMode, o, tm.attribs, tm.ave_log_lum);
                if (tm.to_srgb) o = linear_to_srgb(o);
            }
            st_cs(&out.at(px, py), f4(o, 0.0f));
        }
        else
            out.at(px, py) = f4(c + s, 0.0f);
    };
    emit(x, y, s00), emit(x + 1, y, s10), emit(x, y + 1, s01), emit(x + 1, y + 1, s11);
}

// =====================================================================================================================
// Streaming kernels for exact 2:1 levels.
//
// Down (B1 / B2). With in = 2 x out every bilinear tap of the shader sits on a texel corner, i.e. it IS the average of a 2x2
// texel block, and each of the five tap groups of Bloom_ComputePrefilteredTexture.fx:62-80 (four corner groups A+B+D+E ...,
// centre group J+K+L+M) is the average of a 4x4 texel box; the 13-tap kernel of Bloom_ComputeDownsampledTexture.fx:36-40 is
// 0.125 * (four corner boxes) + 0.5 * (centre box). Box sums are separable: a lane holding texels (2x, 2x+1) of a source row
// builds the three horizontal 4-sums it needs (starting at 2x-2, 2x-1, 2x) from its own pair and its neighbours' (shuffles),
// and the vertical 4-sums slide down the rows in registers. Lanes 0 and 31 only feed their neighbours: a warp emits 30 columns.
// Texels outside the plane read as 0 (the border addressing of these taps, Bloom.cpp:185, :219).
// =====================================================================================================================
DFX_HD float3 shfl_up3(float3 v) { return make_float3(__shfl_up_sync(0xffffffffu, v.x, 1), __shfl_up_sync(0xffffffffu, v.y, 1), __shfl_up_sync(0xffffffffu, v.z, 1)); }
DFX_HD float3 shfl_dn3(float3 v) { return make_float3(__shfl_down_sync(0xffffffffu, v.x, 1), __shfl_down_sync(0xffffffffu, v.y, 1), __shfl_down_sync(0xffffffffu, v.z, 1)); }
DFX_HD float3 shfl3(float3 v, int src) { return make_float3(__shfl_sync(0xffffffffu, v.x, src), __shfl_sync(0xffffffffu, v.y, src), __shfl_sync(0xffffffffu, v.z, src)); }

constexpr int kDnCols = 30; // output columns per warp
constexpr int kStreamWarps = 4;
// Rows per warp are chosen per launch (stream_rows_per_warp): as few as keep the whole level in ONE wave of resident warps, so that a
// large level streams at full bandwidth without a tail wave (measured: 1.05 waves cost 2x) and a small level is spread over as many
// warps as the GPU has (a warp walks its rows sequentially: one memory latency per row pair).

struct RowPair // texels (sx, sx + 1) of the source rows 2k and 2k + 1
{
    float4 a0, a1, b0, b1;
};
struct PairSums
{
    float3 Rl, Rr;       // 4-wide horizontal sums starting at sx - 2 resp. sx, summed over the two rows
    float3 ce, co, cc;   // 4-wide horizontal sum starting at sx - 1: even row, odd row, both
};
DFX_HD PairSums pair_sums(const RowPair& p)
{
    const float3 ea = xyz(p.a0), oa = xyz(p.a1), eb = xyz(p.b0), ob = xyz(p.b1);
    const float3 Pa = ea + oa, Pb = eb + ob, P2 = Pa + Pb;
    PairSums s;
    s.Rl = shfl_up3(P2) + P2;
    s.Rr = P2 + shfl_dn3(P2);
    s.ce = (shfl_up3(oa) + Pa) + shfl_dn3(ea);
    s.co = (shfl_up3(ob) + Pb) + shfl_dn3(eb);
    s.cc = s.ce + s.co;
    return s;
}

// One warp's share of a streaming down-sample: output columns [ox0, ox0 + kDnCols) x rows [oyb, oye). CG: loads bypass L1 (ld.global.cg), for
// source levels written earlier in the SAME launch by other SMs (bloom_levels_kernel).
template <bool PREFILTER, bool CG>
__device__ __forceinline__ void down2x_stream_item(const dfx_bloom_attribs& A, const View<const float4>& in, const View<float4>& out, int ox0, int oyb, int oye, int lane)
{
    const int  ox = ox0 + lane - 1, sx = 2 * ox;
    const bool col_ok = sx >= 0 && sx < in.w; // in.w == 2 * out.w: sx + 1 is inside whenever sx is
    auto ld = [&](const float4* q) { return CG ? __ldcg(q) : __ldg(q); };
    auto load_pair = [&](int k) {
        RowPair   p;
        const int r = 2 * k; // in.h == 2 * out.h: rows 2k and 2k + 1 are inside or outside together
        if (col_ok && r >= 0 && r < in.h)
        {
            const float4* q = in.row(r) + sx;
            p.a0 = ld(q), p.a1 = ld(q + 1), p.b0 = ld(q + in.pitch), p.b1 = ld(q + in.pitch + 1);
        }
        else
            p.a0 = p.a1 = p.b0 = p.b1 = make_float4(0.f, 0.f, 0.f, 0.f);
        return p;
    };
    // warm-up: pairs oyb - 1 and oyb; `next` always holds the pair one iteration ahead (loads in flight while this one computes)
    RowPair        next = load_pair(oyb + 1);
    const PairSums s0 = pair_sums(load_pair(oyb - 1)), s1 = pair_sums(load_pair(oyb));
    float3         Rl0 = s0.Rl, Rr0 = s0.Rr, Rl1 = s1.Rl, Rr1 = s1.Rr, oddPrev = s0.co, oddCur = s1.co, ccCur = s1.cc;
    for (int oy = oyb; oy < oye; ++oy)
    {
        const RowPair cur = next;
        if (oy + 2 <= oye) next = load_pair(oy + 2);
        const PairSums s = pair_sums(cur); // rows 2 oy + 2, 2 oy + 3
        // 4x4 box sums: corner boxes over rows [2oy-2, 2oy+1] / [2oy, 2oy+3], centre box over rows [2oy-1, 2oy+2]
        const float3 bUL = Rl0 + Rl1, bUR = Rr0 + Rr1, bLL = Rl1 + s.Rl, bLR = Rr1 + s.Rr, bC = (oddPrev + ccCur) + s.ce;
        if (lane >= 1 && lane <= kDnCols && ox < out.w)
        {
            if (!PREFILTER)
                out.at(ox, oy) = f4(((bUL + bUR) + (bLL + bLR)) * (0.125f / 16.0f) + bC * (0.5f / 16.0f), 0.0f);
            else
            {
                float3 g[5] = {bUL * (1.0f / 16.0f), bUR * (1.0f / 16.0f), bLL * (1.0f / 16.0f), bLR * (1.0f / 16.0f), bC * (1.0f / 16.0f)};
                float3 csum = make_float3(0.f, 0.f, 0.f);
                float  wsum = 0.0f;
#pragma unroll
                for (int i = 0; i < 5; ++i)
                {
                    const float w = (i == 4 ? 0.5f : 0.125f) * frcp(1.0f + luminance(g[i])); // KarisAverage :19-22
                    csum = csum + g[i] * w;
                    wsum += w;
                }
                const float3 c = csum * frcp(wsum + 1.0e-5f);
                // Prefilter :24-35
                const float brightness   = fmaxf(c.x, fmaxf(c.y, c.z));
                const float knee         = A.Threshold * A.SoftTreshold;
                float       soft         = fminf(fmaxf(brightness - A.Threshold + knee, 0.0f), 2.0f * knee);
                soft                     = soft * soft * 0.25f * frcp(knee + 1.0e-5f);
                const float contribution = fmaxf(soft, brightness - A.Threshold) * frcp(fmaxf(brightness, 1.0e-5f));
                out.at(ox, oy) = f4(c * contribution, 0.0f);
            }
        }
        Rl0 = Rl1, Rr0 = Rr1, Rl1 = s.Rl, Rr1 = s.Rr, oddPrev = oddCur, oddCur = s.co, ccCur = s.cc;
    }
}

template <bool PREFILTER>
__global__ void __launch_bounds__(32 * kStreamWarps) bloom_down2x_stream_kernel(dfx_bloom_attribs A, View<const float4> in, View<float4> out, int y0, int y1, int rows_per_warp)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int ox0 = (blockIdx.x * kStreamWarps + warp) * kDnCols;
    const int oyb = y0 + blockIdx.y * rows_per_warp, oye = min(oyb + rows_per_warp, y1);
    if (ox0 >= out.w || oyb >= oye) return; // warp-uniform
    down2x_stream_item<PREFILTER, false>(A, in, out, ox0, oyb, oye, lane);
}

// Up (B3 / B4). With out = 2 x coarser the 3x3 tent of bilinear taps (Bloom_ComputeUpsampledTexture.fx:27-43) collapses to a
// separable 4-tap filter whose weights depend only on the parity of the output coordinate:
//   even x = 2k : coarse texels k-2..k+1 weigh (1, 5, 7, 3)/16      odd x = 2k+1 : k-1..k+2 weigh (3, 7, 5, 1)/16
// (position x/2 -+ 1/4 -> bilinear {1/4, 3/4}, convolved with the tent {1/4, 1/2, 1/4}); clamp addressing. A warp owns 32 output
// columns: lanes 0..19 load the 20 coarse texels of a coarse row that the 32 columns touch, every lane gathers its four by
// shuffle, and the vertical filter slides over five coarse rows in registers, emitting two output rows per coarse row. The
// fine-level texel (same-level down-sample for B3, the scene colour for B4) is read once, fully coalesced, and so is the store.

// TM: -1 = no tone map, otherwise the tone-mapping operator (a compile-time parameter: one operator's code per instantiation, and its
// per-frame constants - exposure scale, white-point normalisation - are hoisted out of the row loop by the compiler).
// One warp's share: output columns [fx0, fx0 + 32) x rows [fyb, fye), fyb even; y1 = end of the caller's row range.
template <bool COMPOSITE, int TM, bool CG>
__device__ __forceinline__ void up2x_stream_item(const dfx_bloom_attribs& A, const View<const float4>& fine, const View<const float4>& coarser, const View<float4>& out,
                                                 int fx0, int fyb, int fye, int y1, int lane, const ToneMapIn& tm)
{
    const int   x = fx0 + lane;
    const bool  xin = x < out.w;
    const int   ck = min(max((fx0 >> 1) - 2 + lane, 0), coarser.w - 1);
    const int   s0 = (lane >> 1) + (lane & 1);
    const bool  odd = lane & 1;
    const float w0 = odd ? 3.f / 16 : 1.f / 16, w1 = odd ? 7.f / 16 : 5.f / 16, w2 = odd ? 5.f / 16 : 7.f / 16, w3 = odd ? 1.f / 16 : 3.f / 16;
    auto ld = [&](const float4* q) { return CG ? __ldcg(q) : __ldg(q); };
    auto load_coarse = [&](int j) { // this lane's texel of the coarse row j (clamped); lanes 20..31 hold nothing
        const int cj = min(max(j, 0), coarser.h - 1);
        return lane < 20 ? xyz(ld(&coarser.at(ck, cj))) : make_float3(0.f, 0.f, 0.f);
    };
    auto hfilter = [&](float3 c) { return shfl3(c, s0) * w0 + shfl3(c, s0 + 1) * w1 + shfl3(c, s0 + 2) * w2 + shfl3(c, s0 + 3) * w3; }; // horizontal 4-tap
    auto load_fine = [&](int y) { return (xin && y < y1) ? ld(&fine.at(x, y)) : make_float4(0.f, 0.f, 0.f, 0.f); };
    auto emit = [&](int y, float3 s, float4 f) {
        if (!xin || y >= y1) return;
        const float3 c = xyz(f); // linear sampler at the texel centre == the texel
        if (COMPOSITE)
        {
            float3 o = lerp3(c, c + A.Intensity * s, A.AlphaInterpolation);
            if (TM >= 0)
            {
                o = tone_map<(TM < 0 ? 0 : TM)>(o, tm.attribs, tm.ave_log_lum);
                if (tm.to_srgb) o = linear_to_srgb(o);
            }
            st_cs(&out.at(x, y), f4(o, 0.0f));
        }
        else
            out.at(x, y) = f4(c + s, 0.0f);
    };
    // Software pipeline: the fine texels and the coarse row of the NEXT step are in flight while this step computes. (Two steps ahead
    // was measured slower: 0.079 vs 0.064 ms for the 4K composite, profiles/r2i.)
    const int jb = fyb >> 1;
    float4    f0 = load_fine(fyb), f1 = load_fine(fyb + 1);
    float3    cnext = load_coarse(jb + 2);
    float3    H0 = hfilter(load_coarse(jb - 2)), H1 = hfilter(load_coarse(jb - 1)), H2 = hfilter(load_coarse(jb)), H3 = hfilter(load_coarse(jb + 1));
    for (int j = jb; 2 * j < fye; ++j)
    {
        const float4 c0 = f0, c1 = f1;
        const float3 ccur = cnext;
        f0 = load_fine(2 * j + 2), f1 = load_fine(2 * j + 3);
        cnext = load_coarse(j + 3);
        const float3 H4 = hfilter(ccur);
        emit(2 * j, H0 * (1.f / 16) + H1 * (5.f / 16) + H2 * (7.f / 16) + H3 * (3.f / 16), c0);
        emit(2 * j + 1, H1 * (3.f / 16) + H2 * (7.f / 16) + H3 * (5.f / 16) + H4 * (1.f / 16), c1);
        H0 = H1, H1 = H2, H2 = H3, H3 = H4;
    }
}

template <bool COMPOSITE, int TM, bool LUM_DEV = false>
__global__ void __launch_bounds__(32 * kStreamWarps) bloom_up2x_stream_kernel(dfx_bloom_attribs A, View<const float4> fine, View<const float4> coarser, View<float4> out,
                                                                              int y0, int y1, int coarse_rows_per_warp, ToneMapIn tm)
{
    if (LUM_DEV) tm.ave_log_lum = fmaxf(0.05f, __ldg(tm.ave_log_lum_dev)); // GetAverageSceneLuminance (AtmosphereShadersCommon.fxh:188-197)
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int fx0 = (blockIdx.x * kStreamWarps + warp) * 32;
    const int fyb = y0 + blockIdx.y * (2 * coarse_rows_per_warp), fye = min(fyb + 2 * coarse_rows_per_warp, y1); // y0 is even (checked by the caller)
    if (fx0 >= out.w || fyb >= fye) return; // warp-uniform
    up2x_stream_item<COMPOSITE, TM, false>(A, fine, coarser, out, fx0, fyb, fye, y1, lane, tm);
}

// =====================================================================================================================
// Tail: every level with at most kTailTexels texels (60x33 and below at 4K), down to the top of the pyramid and back up, in ONE launch
// of one thread-block cluster (8 CTAs x 512 threads, co-scheduled on one GPC). Levels are separated by a cluster barrier
// (release / acquire at cluster scope); planes written inside the kernel are re-read with ld.global.cg (L2, never a stale L1 line).
// Per texel the arithmetic is the generic kernels' (same taps, same order): the tail is bit-identical to the per-level launches.
// =====================================================================================================================
constexpr int kTailTexels  = 2048; // one cluster = 8 SMs: larger levels are faster as ordinary launches over the whole GPU (measured)
constexpr int kTailDefault = 0;    // dfx_tune("bloom_tail"): measured at 4K (profiles/r2k1) the tail wins as a pass (0.035 ms against 0.049 ms for the two
                                   // launches it replaces) and loses as a frame (2.30 vs 2.24 ms): the cluster holds 8 SMs of one GPC for 35 us of
                                   // dependent latency on the Bloom stream, the per-level launches interleave with the next frame's front half
constexpr int kTailThreads = 512;
constexpr int kTailCluster = 8;

struct TailArgs
{
    View<float4> down[DFX_BLOOM_MAX_LEVELS], up[DFX_BLOOM_MAX_LEVELS];
    int          first, mips; // computes down[first .. mips-1] from down[first-1], then up[mips-2 .. first-1]
};

template <bool BORDER>
DFX_HD float3 tap3_cg(const View<float4>& t, float u, float v)
{
    const float px = snap8(u * float(t.w) - 0.5f), py = snap8(v * float(t.h) - 0.5f);
    const float fx0 = floorf(px), fy0 = floorf(py);
    const int   x0 = (int)fx0, y0 = (int)fy0;
    const float fx = px - fx0, fy = py - fy0;
    auto ld = [&](int x, int y) {
        if (BORDER)
            return ((unsigned)x < (unsigned)t.w && (unsigned)y < (unsigned)t.h) ? __ldcg(&t.at(x, y)) : make_float4(0.f, 0.f, 0.f, 0.f);
        return __ldcg(&t.at(min(max(x, 0), t.w - 1), min(max(y, 0), t.h - 1)));
    };
    const float4 a = ld(x0, y0), b = ld(x0 + 1, y0), c = ld(x0, y0 + 1), d = ld(x0 + 1, y0 + 1);
    return xyz(a * ((1.0f - fx) * (1.0f - fy)) + b * (fx * (1.0f - fy)) + c * ((1.0f - fx) * fy) + d * (fx * fy));
}

// B2 (generic level) and B3 (generic level) over a flat range of threads; every load is ld.global.cg
__device__ __forceinline__ void generic_down_level(const View<float4>& in, const View<float4>& out, int tid, int nth)
{
    for (int idx = tid; idx < out.w * out.h; idx += nth)
    {
        const int   y = idx / out.w, x = idx - y * out.w;
        const float u = (float(x) + 0.5f) / float(out.w), v = (float(y) + 0.5f) / float(out.h);
        const float tx = 1.0f / float(in.w), ty = 1.0f / float(in.h);
        auto        T = [&](float i_, float j_) { return tap3_cg<true>(in, u + tx * i_, v + ty * j_); };
        const float3 tA = T(-2, +2), tB = T(0, +2), tC = T(+2, +2), tD = T(-2, 0), tE = T(0, 0), tF = T(+2, 0), tG = T(-2, -2), tH = T(0, -2), tI = T(+2, -2);
        const float3 tJ = T(-1, +1), tK = T(+1, +1), tL = T(-1, -1), tM = T(+1, -1);
        float3 o = make_float3(0.f, 0.f, 0.f);
        o = o + (tA + tC + tG + tI) * 0.03125f;
        o = o + (tB + tD + tF + tH) * 0.0625f;
        o = o + (tE + tJ + tK + tL + tM) * 0.125f;
        out.at(x, y) = f4(o, 0.0f);
    }
}
__device__ __forceinline__ void generic_up_level(const View<float4>& same, const View<float4>& lo, const View<float4>& out, int tid, int nth)
{
    for (int idx = tid; idx < out.w * out.h; idx += nth)
    {
        const int   y = idx / out.w, x = idx - y * out.w;
        const float u = (float(x) + 0.5f) / float(out.w), v = (float(y) + 0.5f) / float(out.h);
        const float tx = 1.0f / float(lo.w), ty = 1.0f / float(lo.h);
        const float3 tA = tap3_cg<false>(lo, u - tx, v + ty), tB = tap3_cg<false>(lo, u, v + ty), tC = tap3_cg<false>(lo, u + tx, v + ty);
        const float3 tD = tap3_cg<false>(lo, u - tx, v), tE = tap3_cg<false>(lo, u, v), tF = tap3_cg<false>(lo, u + tx, v);
        const float3 tG = tap3_cg<false>(lo, u - tx, v - ty), tH = tap3_cg<false>(lo, u, v - ty), tI = tap3_cg<false>(lo, u + tx, v - ty);
        float3 s = tE * 0.25f;
        s = s + (tB + tD + tF + tH) * 0.125f;
        s = s + (tA + tC + tG + tI) * 0.0625f;
        out.at(x, y) = f4(tap3_cg<false>(same, u, v) + s, 0.0f);
    }
}

__global__ void __cluster_dims__(kTailCluster, 1, 1) __launch_bounds__(kTailThreads) bloom_tail_kernel(TailArgs a)
{
    namespace cg = cooperative_groups;
    cg::cluster_group cluster = cg::this_cluster();
    const int tid = int(cluster.block_rank()) * kTailThreads + int(threadIdx.x), nth = kTailCluster * kTailThreads;
    for (int i = a.first; i < a.mips; ++i) // B2
    {
        generic_down_level(a.down[i - 1], a.down[i], tid, nth);
        cluster.sync();
    }
    const int top = a.mips - 1;
    for (int i = top; i >= a.first; --i) // B3: up[i-1] = down[i-1] + tent(i == top ? down[i] : up[i])
    {
        generic_up_level(a.down[i - 1], i == top ? a.down[i] : a.up[i], a.up[i - 1], tid, nth);
        if (i > a.first) cluster.sync();
    }
}

// =====================================================================================================================
// Levels: EVERY level after the prefilter - down to the top of the pyramid and back up to level 0 - in ONE cooperative launch over the
// whole GPU (dfx_pass_bloom_levels). The per-level launches of B2 / B3 are a chain of 9-11 dependent kernels of 5-15 us each on planes
// that fit in L2: launch gaps and the 8-SM cluster of the tail were half of their time. Here a level is a phase of a persistent grid
// (as many CTAs as are co-resident), phases are separated by a grid-wide barrier (arrive counter in global memory, release / acquire at
// GPU scope), and a phase is either the streaming shuffle code of an exact 2:1 level (work items = warp column x row chunk, dealt
// round-robin to the grid's warps) or the generic gather code. Planes written inside the launch are read with ld.global.cg. Per texel
// the arithmetic is that of the per-level kernels (same taps, same order; the compiler's FMA contraction may differ in the last bit).
// Measured at 4K (profiles/r2j): 0.104 ms against 0.118 ms for the nine per-level launches and 20 instead of 28 launches per frame,
// but the whole frame is SLOWER under async compute (2.34 vs 2.28 ms): a cooperative grid needs every SM at once, so it cannot
// slip into the gaps of the next frame's front half the way the small per-level launches do. Opt-in: dfx_tune("bloom_levels") = 1.
// The launch is cooperative (all CTAs co-resident or the launch fails), so two such kernels on two streams cannot starve each other at
// the barrier; a barrier that is not reached within ~2 s raises the error word of the workspace instead of hanging the GPU.
// =====================================================================================================================
constexpr int                kLevelsThreads = 256;
constexpr unsigned long long kLevelsSpinLimit = 4000000000ull; // cycles
struct LevelsArgs
{
    TailArgs  t;
    unsigned* ws; // [0] barrier arrivals, [1] exit tickets, [2] error; all zero between launches
};

__device__ __forceinline__ unsigned ld_acquire_gpu(const unsigned* p)
{
    unsigned v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void grid_barrier(unsigned* ws, unsigned target)
{
    __syncthreads();
    if (threadIdx.x == 0)
    {
        __threadfence();
        atomicAdd(&ws[0], 1u);
        const long long t0 = clock64();
        while (ld_acquire_gpu(&ws[0]) < target)
        {
            if (ld_acquire_gpu(&ws[2]) != 0u) break; // another CTA gave up: do not wait for it
            if ((unsigned long long)(clock64() - t0) > kLevelsSpinLimit)
            {
                atomicExch(&ws[2], 1u);
                break;
            }
        }
        __threadfence();
    }
    __syncthreads();
}
__device__ __forceinline__ View<const float4> as_const(const View<float4>& v) { return View<const float4>{v.p, v.pitch, v.w, v.h}; }
__device__ __forceinline__ int cdiv(int a, int b) { return (a + b - 1) / b; }

__global__ void __launch_bounds__(kLevelsThreads, 3) bloom_levels_kernel(const __grid_constant__ LevelsArgs a)
{
    const int lane = threadIdx.x & 31;
    const int gwarp = (blockIdx.x * kLevelsThreads + threadIdx.x) >> 5, nwarps = (gridDim.x * kLevelsThreads) >> 5;
    const int tid = blockIdx.x * kLevelsThreads + threadIdx.x, nth = gridDim.x * kLevelsThreads;
    unsigned  phase = 0;
    const dfx_bloom_attribs A{};
    const ToneMapIn         tm{};
    for (int i = a.t.first; i < a.t.mips; ++i) // B2
    {
        const View<float4>&in = a.t.down[i - 1], &out = a.t.down[i];
        if (in.w == 2 * out.w && in.h == 2 * out.h)
        {
            // rows per item: as few as give every warp of the grid at most one item (at least 2: each item re-reads two source row pairs)
            const int cols = cdiv(out.w, kDnCols), per_col = max(nwarps / cols, 1), rpw = max(cdiv(out.h, per_col), 2), chunks = cdiv(out.h, rpw);
            for (int item = gwarp; item < cols * chunks; item += nwarps)
            {
                const int c = item % cols, r = item / cols;
                down2x_stream_item<false, true>(A, as_const(in), out, c * kDnCols, r * rpw, min((r + 1) * rpw, out.h), lane);
            }
        }
        else
            generic_down_level(in, out, tid, nth);
        grid_barrier(a.ws, ++phase * gridDim.x);
    }
    const int top = a.t.mips - 1;
    for (int i = top; i >= a.t.first; --i) // B3: up[i-1] = down[i-1] + tent(i == top ? down[i] : up[i])
    {
        const View<float4>&same = a.t.down[i - 1], &lo = i == top ? a.t.down[i] : a.t.up[i], &out = a.t.up[i - 1];
        if (out.w == 2 * lo.w && out.h == 2 * lo.h)
        {
            const int cols = cdiv(out.w, 32), per_col = max(nwarps / cols, 1), cpw = min(max(cdiv(lo.h, per_col), 1), 4), chunks = cdiv(lo.h, cpw);
            for (int item = gwarp; item < cols * chunks; item += nwarps)
            {
                const int c = item % cols, r = item / cols;
                up2x_stream_item<false, -1, true>(A, as_const(same), as_const(lo), out, c * 32, 2 * r * cpw, min(2 * (r + 1) * cpw, out.h), out.h, lane, tm);
            }
        }
        else
            generic_up_level(same, lo, out, tid, nth);
        if (i > a.t.first) grid_barrier(a.ws, ++phase * gridDim.x);
    }
    // leave the workspace zeroed for the next launch: the last CTA out knows that every other CTA is past the last barrier
    __syncthreads();
    if (threadIdx.x == 0 && atomicAdd(&a.ws[1], 1u) == gridDim.x - 1)
    {
        a.ws[0] = 0u, a.ws[1] = 0u;
        __threadfence();
    }
}

} // namespace dfx

using namespace dfx;

#define DFX_GRID(w, rows) dim3 block(32, 8), grid(div_up(w, 32), div_up(rows.y1 - rows.y0, 8))

// dfx_tune("bloom_impl"): 1 (default) = streaming shuffle kernels on exact 2:1 levels, 0 = the round-1 shared-memory tile kernels
// (kept for A/B timing), 2 = generic gather kernels everywhere.
static int bloom_impl() { return dfx_tune_get("bloom_impl", 1); }

// Rows per warp of a streaming launch: the fewest that fit the level into one wave of resident warps (at least `min_rows`).
template <class K>
static int stream_rows_per_warp(K kernel, int warp_columns, int rows, int min_rows)
{
    // resident warps of this kernel (one static per kernel instantiation). Cached once per process: the GPUs of a node are identical, and
    // two threads racing here store the same value.
    static std::atomic<int> cached{0};
    int                     slots = cached.load(std::memory_order_relaxed);
    if (slots == 0)
    {
        int dev = 0, sms = 148, blocks = 4;
        (void)cudaGetDevice(&dev);
        (void)cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&blocks, kernel, 32 * kStreamWarps, 0) != cudaSuccess || blocks < 1) blocks = 4;
        slots = sms * blocks * kStreamWarps;
        cached.store(slots, std::memory_order_relaxed);
    }
    const int per_column = std::max(slots / std::max(warp_columns, 1), 1);
    return std::max(div_up(rows, per_column), min_rows);
}

static dfx_status launch_down(void* stream, bool prefilter, const dfx_bloom_attribs& A, const View<const float4>& in, const View<float4>& out, dfx_rows rows)
{
    cudaStream_t s     = as_stream(stream);
    const bool   exact = in.w == 2 * out.w && in.h == 2 * out.h;
    const int    impl  = bloom_impl();
    if (exact && impl == 1)
    {
        const int  bx = div_up(out.w, kDnCols * kStreamWarps), n = rows.y1 - rows.y0;
        const int  rpw = prefilter ? stream_rows_per_warp(bloom_down2x_stream_kernel<true>, bx * kStreamWarps, n, 2) : stream_rows_per_warp(bloom_down2x_stream_kernel<false>, bx * kStreamWarps, n, 2);
        const dim3 grid(bx, div_up(n, rpw));
        if (prefilter)
            bloom_down2x_stream_kernel<true><<<grid, 32 * kStreamWarps, 0, s>>>(A, in, out, rows.y0, rows.y1, rpw);
        else
            bloom_down2x_stream_kernel<false><<<grid, 32 * kStreamWarps, 0, s>>>(A, in, out, rows.y0, rows.y1, rpw);
    }
    else
    {
        DFX_GRID(out.w, rows);
        if (exact && impl == 0)
        {
            if (prefilter)
                bloom_down2x_kernel<true><<<grid, block, 0, s>>>(A, in, out, rows.y0, rows.y1);
            else
                bloom_down2x_kernel<false><<<grid, block, 0, s>>>(A, in, out, rows.y0, rows.y1);
        }
        else if (prefilter)
            bloom_prefilter_kernel<<<grid, block, 0, s>>>(A, in, out, rows.y0, rows.y1);
        else
            bloom_downsample_kernel<<<grid, block, 0, s>>>(in, out, rows.y0, rows.y1);
    }
    DFX_LAUNCHED("bloom down-sampling kernel");
    return DFX_OK;
}

extern "C" dfx_status dfx_pass_bloom_prefilter(void* stream, const dfx_bloom_attribs* attribs, const dfx_plane* color, const dfx_plane* out_level0, dfx_rows rows)
{
    DFX_PROFILE(stream, "bloom_prefilter");
    DFX_REQUIRE(attribs, "null argument");
    DFX_VIEW(const float4, in, color, DFX_FORMAT_RGBA32F);
    DFX_VIEW(float4, out, out_level0, DFX_FORMAT_RGBA32F);
    DFX_REQUIRE(out.w == max(in.w / 2, 1) && out.h == max(in.h / 2, 1), "level 0 must be half the input size");
    DFX_REQUIRE(rows_ok(rows, out.h), "bad row range (rows are in output-plane coordinates)");
    if (rows.y1 == rows.y0) return DFX_OK;
    return launch_down(stream, true, *attribs, in, out, rows);
}

extern "C" dfx_status dfx_pass_bloom_downsample(void* stream, const dfx_plane* in_, const dfx_plane* out_, dfx_rows rows)
{
    DFX_PROFILE(stream, "bloom_downsample");
    DFX_VIEW(const float4, in, in_, DFX_FORMAT_RGBA32F);
    DFX_VIEW(float4, out, out_, DFX_FORMAT_RGBA32F);
    DFX_REQUIRE(out.w == max(in.w / 2, 1) && out.h == max(in.h / 2, 1), "output must be half the input size");
    DFX_REQUIRE(rows_ok(rows, out.h), "bad row range (rows are in output-plane coordinates)");
    if (rows.y1 == rows.y0) return DFX_OK;
    return launch_down(stream, false, dfx_bloom_attribs{}, in, out, rows);
}

// B3 / B4 (+ M1 / M2): mode 0 = up-sample, 1 = composite, 2 = composite + tone map
static dfx_status launch_up(void* stream, int mode, const dfx_bloom_attribs& A, const View<const float4>& fine, const View<const float4>& lo, const View<float4>& out,
                            dfx_rows rows, const ToneMapIn& tm)
{
    cudaStream_t s     = as_stream(stream);
    const bool   exact = out.w == 2 * lo.w && out.h == 2 * lo.h && (rows.y0 & 1) == 0;
    const int    impl  = bloom_impl();
    if (mode == 2 && !exact) return set_error(DFX_ERR_UNSUPPORTED, "fused composite+tonemap needs an exact 2:1 level");
    if (exact && impl == 1)
    {
        const int bx = div_up(out.w, 32 * kStreamWarps), n = div_up(rows.y1 - rows.y0, 2); // coarse rows
        // coarse rows per warp: dfx_tune("bloom_up_rows"), 0 = as few as fill one wave. Measured at 4K (profiles/r2i): 4 rows 0.062 ms for the
        // composite, 8 rows 0.064, 16 rows 0.066, one wave (25 rows) 0.070 - unlike the down-sampling, short warps win here.
        const int fixed_rows = dfx_tune_get("bloom_up_rows", 4);
#define DFX_UP_LAUNCH_(COMP, TMODE, LD)                                                                                                              \
    do {                                                                                                                                             \
        const int  cpw = fixed_rows > 0 ? fixed_rows : stream_rows_per_warp(bloom_up2x_stream_kernel<COMP, TMODE, LD>, bx * kStreamWarps, n, 1);     \
        const dim3 grid(bx, div_up(n, cpw));                                                                                                         \
        bloom_up2x_stream_kernel<COMP, TMODE, LD><<<grid, 32 * kStreamWarps, 0, s>>>(A, fine, lo, out, rows.y0, rows.y1, cpw, tm);                   \
    } while (0)
#define DFX_UP_LAUNCH(COMP, TMODE)                                                                                                                   \
    do {                                                                                                                                             \
        if (TMODE >= 0 && tm.ave_log_lum_dev) DFX_UP_LAUNCH_(COMP, TMODE, true);                                                                     \
        else DFX_UP_LAUNCH_(COMP, TMODE, false);                                                                                                     \
    } while (0)
        if (mode == 0) DFX_UP_LAUNCH(false, -1);
        else if (mode == 1) DFX_UP_LAUNCH(true, -1);
        else
            switch (tm.attribs.iToneMappingMode)
            {
                case DFX_TONE_MAPPING_MODE_NONE: DFX_UP_LAUNCH(true, DFX_TONE_MAPPING_MODE_NONE); break;
                case DFX_TONE_MAPPING_MODE_EXP: DFX_UP_LAUNCH(true, DFX_TONE_MAPPING_MODE_EXP); break;
                case DFX_TONE_MAPPING_MODE_REINHARD: DFX_UP_LAUNCH(true, DFX_TONE_MAPPING_MODE_REINHARD); break;
                case DFX_TONE_MAPPING_MODE_REINHARD_MOD: DFX_UP_LAUNCH(true, DFX_TONE_MAPPING_MODE_REINHARD_MOD); break;
                case DFX_TONE_MAPPING_MODE_UNCHARTED2: DFX_UP_LAUNCH(true, DFX_TONE_MAPPING_MODE_UNCHARTED2); break;
                case DFX_TONE_MAPPING_MODE_FILMIC_ALU: DFX_UP_LAUNCH(true, DFX_TONE_MAPPING_MODE_FILMIC_ALU); break;
                case DFX_TONE_MAPPING_MODE_LOGARITHMIC: DFX_UP_LAUNCH(true, DFX_TONE_MAPPING_MODE_LOGARITHMIC); break;
                case DFX_TONE_MAPPING_MODE_ADAPTIVE_LOG: DFX_UP_LAUNCH(true, DFX_TONE_MAPPING_MODE_ADAPTIVE_LOG); break;
                case DFX_TONE_MAPPING_MODE_AGX: DFX_UP_LAUNCH(true, DFX_TONE_MAPPING_MODE_AGX); break;
                case DFX_TONE_MAPPING_MODE_AGX_CUSTOM: DFX_UP_LAUNCH(true, DFX_TONE_MAPPING_MODE_AGX_CUSTOM); break;
                case DFX_TONE_MAPPING_MODE_PBR_NEUTRAL: DFX_UP_LAUNCH(true, DFX_TONE_MAPPING_MODE_PBR_NEUTRAL); break;
                default: DFX_UP_LAUNCH(true, DFX_TONE_MAPPING_MODE_COMMERCE); break;
            }
#undef DFX_UP_LAUNCH
#undef DFX_UP_LAUNCH_
    }
    else if (exact && (impl == 0 || mode == 2))
    {
        const dim3 grid(div_up(out.w, 64), div_up(rows.y1 - rows.y0, 16)), block(32, 8);
        if (mode == 0) bloom_up2x_kernel<false><<<grid, block, 0, s>>>(A, fine, lo, out, rows.y0, rows.y1);
        if (mode == 1) bloom_up2x_kernel<true><<<grid, block, 0, s>>>(A, fine, lo, out, rows.y0, rows.y1);
        if (mode == 2 && !tm.ave_log_lum_dev) bloom_up2x_kernel<true, true><<<grid, block, 0, s>>>(A, fine, lo, out, rows.y0, rows.y1, tm);
        if (mode == 2 && tm.ave_log_lum_dev) bloom_up2x_kernel<true, true, true><<<grid, block, 0, s>>>(A, fine, lo, out, rows.y0, rows.y1, tm);
    }
    else
    {
        DFX_GRID(out.w, rows);
        if (mode == 0)
            bloom_upsample_kernel<<<grid, block, 0, s>>>(fine, lo, out, rows.y0, rows.y1);
        else
            bloom_composite_kernel<<<grid, block, 0, s>>>(A, fine, lo, out, rows.y0, rows.y1);
    }
    DFX_LAUNCHED("bloom up-sampling kernel");
    return DFX_OK;
}

extern "C" dfx_status dfx_pass_bloom_upsample(void* stream, const dfx_plane* same_level_down, const dfx_plane* coarser, const dfx_plane* out_, dfx_rows rows)
{
    DFX_PROFILE(stream, "bloom_upsample");
    DFX_VIEW(const float4, same, same_level_down, DFX_FORMAT_RGBA32F);
    DFX_VIEW(const float4, lo, coarser, DFX_FORMAT_RGBA32F);
    DFX_VIEW(float4, out, out_, DFX_FORMAT_RGBA32F);
    DFX_SAME_SIZE(same, out);
    DFX_REQUIRE(rows_ok(rows, out.h), "bad row range (rows are in output-plane coordinates)");
    if (rows.y1 == rows.y0) return DFX_OK;
    return launch_up(stream, 0, dfx_bloom_attribs{}, same, lo, out, rows, ToneMapIn{});
}

extern "C" dfx_status dfx_pass_bloom_composite(void* stream, const dfx_bloom_attribs* attribs, const dfx_plane* color, const dfx_plane* up0,
                                               const dfx_plane* out_, dfx_rows rows)
{
    DFX_PROFILE(stream, "bloom_composite");
    DFX_REQUIRE(attribs, "null argument");
    DFX_VIEW(const float4, c, color, DFX_FORMAT_RGBA32F);
    DFX_VIEW(const float4, u, up0, DFX_FORMAT_RGBA32F);
    DFX_VIEW(float4, out, out_, DFX_FORMAT_RGBA32F);
    DFX_SAME_SIZE(c, out);
    DFX_REQUIRE(rows_ok(rows, out.h), "bad row range");
    if (rows.y1 == rows.y0) return DFX_OK;
    return launch_up(stream, 1, *attribs, c, u, out, rows, ToneMapIn{});
}

// B4 + M1/M2 in one kernel (only on exact 2:1 levels: the caller falls back to the two separate passes otherwise).
extern "C" dfx_status dfx_pass_bloom_composite_tonemap(void* stream, const dfx_bloom_attribs* attribs, const dfx_tonemap_attribs* tonemap, float ave_log_lum,
                                                       int32_t convert_to_srgb, const dfx_plane* color, const dfx_plane* up0, const dfx_plane* ldr_out, dfx_rows rows)
{
    DFX_PROFILE(stream, "bloom_composite_tonemap");
    DFX_REQUIRE(attribs && tonemap, "null argument");
    DFX_VIEW(const float4, c, color, DFX_FORMAT_RGBA32F);
    DFX_VIEW(const float4, u, up0, DFX_FORMAT_RGBA32F);
    DFX_VIEW(float4, out, ldr_out, DFX_FORMAT_RGBA32F);
    DFX_SAME_SIZE(c, out);
    DFX_REQUIRE(rows_ok(rows, out.h), "bad row range");
    DFX_REQUIRE(tonemap->iToneMappingMode >= 0 && tonemap->iToneMappingMode <= DFX_TONE_MAPPING_MODE_COMMERCE, "unknown tone mapping mode %d", tonemap->iToneMappingMode);
    if (rows.y1 == rows.y0) return DFX_OK;
    return launch_up(stream, 2, *attribs, c, u, out, rows, ToneMapIn{*tonemap, ave_log_lum, convert_to_srgb});
}

// the same with fAveLogLum = max(0.05, *ave_log_lum_dev), read by the kernel (the average-luminance state of dfx_exposure.cu)
extern "C" dfx_status dfx_pass_bloom_composite_tonemap_dev(void* stream, const dfx_bloom_attribs* attribs, const dfx_tonemap_attribs* tonemap,
                                                           const float* ave_log_lum_dev, int32_t convert_to_srgb, const dfx_plane* color, const dfx_plane* up0,
                                                           const dfx_plane* ldr_out, dfx_rows rows)
{
    DFX_PROFILE(stream, "bloom_composite_tonemap");
    DFX_REQUIRE(attribs && tonemap && ave_log_lum_dev, "null argument");
    DFX_VIEW(const float4, c, color, DFX_FORMAT_RGBA32F);
    DFX_VIEW(const float4, u, up0, DFX_FORMAT_RGBA32F);
    DFX_VIEW(float4, out, ldr_out, DFX_FORMAT_RGBA32F);
    DFX_SAME_SIZE(c, out);
    DFX_REQUIRE(rows_ok(rows, out.h), "bad row range");
    DFX_REQUIRE(tonemap->iToneMappingMode >= 0 && tonemap->iToneMappingMode <= DFX_TONE_MAPPING_MODE_COMMERCE, "unknown tone mapping mode %d", tonemap->iToneMappingMode);
    if (rows.y1 == rows.y0) return DFX_OK;
    return launch_up(stream, 2, *attribs, c, u, out, rows, ToneMapIn{*tonemap, 0.0f, convert_to_srgb, ave_log_lum_dev});
}

// First level the tail kernel takes over: the first one with at most kTailTexels texels (never level 0: it needs a source level).
extern "C" int32_t dfx_bloom_tail_first_level(const dfx_plane* down, int32_t mips)
{
    if (!down || mips < 2 || dfx_tune_get("bloom_tail", kTailDefault) == 0) return mips;
    const long long limit = dfx_tune_get("bloom_tail_texels", kTailTexels);
    for (int i = 1; i < mips; ++i)
        if ((long long)down[i].width * down[i].height <= limit) return i;
    return mips;
}

// B2 for the levels first .. mips-1 and B3 for the levels mips-2 .. first-1, in one launch (see bloom_tail_kernel).
extern "C" dfx_status dfx_pass_bloom_tail(void* stream, const dfx_plane* down, const dfx_plane* up, int32_t first, int32_t mips)
{
    DFX_PROFILE(stream, "bloom_tail");
    DFX_REQUIRE(down && up, "null argument");
    DFX_REQUIRE(mips >= 2 && mips <= DFX_BLOOM_MAX_LEVELS && first >= 1 && first < mips, "bad level range: first %d of %d levels", first, mips);
    TailArgs a;
    a.first = first, a.mips = mips;
    for (int i = first - 1; i < mips; ++i)
    {
        DFX_REQUIRE(make_view<float4>(&down[i], DFX_FORMAT_RGBA32F, a.down[i]), "bad down-sampled level %d", i);
        if (i > first - 1) DFX_REQUIRE(a.down[i].w == max(a.down[i - 1].w / 2, 1) && a.down[i].h == max(a.down[i - 1].h / 2, 1), "level %d must be half of level %d", i, i - 1);
        if (i < mips - 1)
        {
            DFX_REQUIRE(make_view<float4>(&up[i], DFX_FORMAT_RGBA32F, a.up[i]), "bad up-sampled level %d", i);
            DFX_REQUIRE(a.up[i].w == a.down[i].w && a.up[i].h == a.down[i].h, "up-sampled level %d must have the size of the down-sampled one", i);
        }
    }
    bloom_tail_kernel<<<kTailCluster, kTailThreads, 0, as_stream(stream)>>>(a);
    DFX_LAUNCHED("bloom_tail_kernel");
    return DFX_OK;
}

// B2 for the levels first .. mips-1 and B3 for the levels mips-2 .. first-1 in one cooperative launch over the whole GPU (bloom_levels_kernel).
extern "C" dfx_status dfx_pass_bloom_levels(void* stream, const dfx_plane* down, const dfx_plane* up, int32_t first, int32_t mips, void* workspace)
{
    DFX_PROFILE(stream, "bloom_levels");
    DFX_REQUIRE(down && up && workspace, "null argument");
    DFX_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 15) == 0, "workspace must be 16-byte aligned");
    DFX_REQUIRE(mips >= 2 && mips <= DFX_BLOOM_MAX_LEVELS && first >= 1 && first < mips, "bad level range: first %d of %d levels", first, mips);
    LevelsArgs a;
    a.t.first = first, a.t.mips = mips, a.ws = static_cast<unsigned*>(workspace);
    for (int i = first - 1; i < mips; ++i)
    {
        DFX_REQUIRE(make_view<float4>(&down[i], DFX_FORMAT_RGBA32F, a.t.down[i]), "bad down-sampled level %d", i);
        if (i > first - 1) DFX_REQUIRE(a.t.down[i].w == max(a.t.down[i - 1].w / 2, 1) && a.t.down[i].h == max(a.t.down[i - 1].h / 2, 1), "level %d must be half of level %d", i, i - 1);
        if (i < mips - 1)
        {
            DFX_REQUIRE(make_view<float4>(&up[i], DFX_FORMAT_RGBA32F, a.t.up[i]), "bad up-sampled level %d", i);
            DFX_REQUIRE(a.t.up[i].w == a.t.down[i].w && a.t.up[i].h == a.t.down[i].h, "up-sampled level %d must have the size of the down-sampled one", i);
        }
    }
    static std::atomic<int> cached_grid{0}; // co-resident CTAs of the kernel (identical GPUs: see stream_rows_per_warp)
    int                     grid = cached_grid.load(std::memory_order_relaxed);
    if (grid == 0)
    {
        int dev = 0, sms = 0, blocks = 0, coop = 0;
        DFX_CUDA(cudaGetDevice(&dev));
        DFX_CUDA(cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, dev));
        DFX_REQUIRE(coop, "the device does not support cooperative launches");
        DFX_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
        DFX_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&blocks, bloom_levels_kernel, kLevelsThreads, 0));
        DFX_REQUIRE(blocks >= 1, "bloom_levels_kernel does not fit on an SM");
        grid = sms * blocks;
        cached_grid.store(grid, std::memory_order_relaxed);
    }
    cudaLaunchConfig_t   cfg{};
    cudaLaunchAttribute  attr{};
    attr.id              = cudaLaunchAttributeCooperative;
    attr.val.cooperative = 1;
    cfg.gridDim = dim3(grid), cfg.blockDim = dim3(kLevelsThreads), cfg.dynamicSmemBytes = 0, cfg.stream = as_stream(stream), cfg.attrs = &attr, cfg.numAttrs = 1;
    DFX_CUDA(cudaLaunchKernelEx(&cfg, bloom_levels_kernel, a));
    DFX_LAUNCHED("bloom_levels_kernel");
    return DFX_OK;
}

// 1 if a launch of dfx_pass_bloom_levels on this workspace gave up at a barrier (synchronises with the device)
extern "C" dfx_status dfx_bloom_levels_check(const void* workspace, int32_t* timed_out)
{
    DFX_REQUIRE(workspace && timed_out, "null argument");
    unsigned w[4] = {0, 0, 0, 0};
    DFX_CUDA(cudaMemcpy(w, workspace, sizeof(w), cudaMemcpyDeviceToHost));
    *timed_out = w[2] != 0u;
    return DFX_OK;
}

// dfx_taa_tonemap.cu — TAA T1, compose, ToneMap M1/M2 as sm_100a kernels.
// Reference: PostProcess/TemporalAntiAliasing/src/TemporalAntiAliasing.cpp:260-289 + TAA_ComputeTemporalAccumulation.fx;
//            Shaders/PostProcess/ToneMapping/public/ToneMapping.fxh; Hydrogent/shaders/HnPostProcess.psh:145-185, HnCopyFrame.psh:32-62.
#include "dfx_common.cuh"
#include "dfx_tonemap.cuh"

namespace dfx
{

// =====================================================================================================================
// TAA — TAA_ComputeTemporalAccumulation.fx:229-261
// =====================================================================================================================
template <bool YCOCG>
DFX_HD float3 rgb_to_ycocg(float3 c)
{
    if (!YCOCG) return c;
    float co = c.x - c.z, tmp = c.z + 0.5f * co, cg = c.y - tmp, yy = tmp + 0.5f * cg;
    return make_float3(yy, co, cg);
}
template <bool YCOCG>
DFX_HD float3 ycocg_to_rgb(float3 c)
{
    if (!YCOCG) return c;
    float tmp = c.x - 0.5f * c.z, g = c.z + tmp, b = tmp - 0.5f * c.y, r = b + c.y;
    return make_float3(r, g, b);
}
DFX_HD float3 hdr_to_sdr(float3 c) { return make_float3(c.x * frcp(1.0f + c.x), c.y * frcp(1.0f + c.y), c.z * frcp(1.0f + c.z)); }
DFX_HD float3 sdr_to_hdr(float3 c)
{
    return make_float3(c.x * frcp(1.0f - c.x + kFltEps), c.y * frcp(1.0f - c.y + kFltEps), c.z * frcp(1.0f - c.z + kFltEps));
}

// ClipToAABB :98-106. Less/GreaterEqual are 0/1 selectors fed to lerp(a,b,t) = a + t*(b-a); fminf ignores NaN operands.
DFX_HD float3 clip_to_aabb(float3 prev, float3 curr, float3 centre, float3 ext)
{
    const float  maxT = 10.0f;
    const float3 dir  = curr - prev;
    const float  ix = fdiv((centre.x - signf(dir.x) * ext.x) - prev.x, dir.x); // x/0 -> +-inf, 0/0 -> NaN as in IEEE division
    const float  iy = fdiv((centre.y - signf(dir.y) * ext.y) - prev.y, dir.y);
    const float  iz = fdiv((centre.z - signf(dir.z) * ext.z) - prev.z, dir.z);
    const float  px = lerpf(maxT + 1.0f, ix, ix >= 0.0f ? 1.0f : 0.0f);
    const float  py = lerpf(maxT + 1.0f, iy, iy >= 0.0f ? 1.0f : 0.0f);
    const float  pz = lerpf(maxT + 1.0f, iz, iz >= 0.0f ? 1.0f : 0.0f);
    const float  T  = fminf(maxT, fminf(px, fminf(py, pz)));
    const float  lt = T < maxT ? 1.0f : 0.0f;
    return lerp3(prev, prev + dir * T, lt);
}

struct TaaCam
{
    CamS c, p;
};

// The compose step (rgb += ssr.rgb * ssr.a * scale; rgb *= lerp(1, ao, scale)) evaluated where the composed colour is
// consumed, so that the composed frame never makes a round trip through HBM (same arithmetic as compose_kernel).
struct ComposeIn
{
    View<const float4> ssr;
    View<const float>  ao;
    float              ssr_scale, ssao_scale;
};
template <bool COMPOSE, class TexC>
DFX_HD float3 load_scene_colour(const TexC& color, const ComposeIn& ci, int gx, int gy)
{
    float3 c = xyz(color.ld(gx, gy));
    if (COMPOSE)
    {
        if (ci.ssr.p && ci.ssr_scale > 0.0f)
        {
            const float4 s = __ldg(&ci.ssr.at(gx, gy));
            c              = c + xyz(s) * s.w * ci.ssr_scale;
        }
        if (ci.ao.p && ci.ssao_scale > 0.0f) c = c * lerpf(1.0f, __ldg(&ci.ao.at(gx, gy)), ci.ssao_scale);
    }
    return c;
}

template <bool BICUBIC, bool YCOCG, bool GAUSS, bool COMPOSE, bool C16>
__global__ void __launch_bounds__(256, DFX_OCC_TAA) taa_kernel(const dfx_camera_attribs* __restrict__ cams, dfx_taa_attribs A, TexRGBA<C16> curr_color,
                                                  ComposeIn ci, View<const float4> prev_accum, View<const float2> motion, View<const float> curr_depth,
                                                  View<const float> prev_depth, View<float4> out, int y0, int y1)
{
    // 32x8 pixel tile + 1-pixel halo of the current colour, converted ONCE per texel to the clipping space (Reinhard SDR,
    // optionally YCoCg) and shared through smem: the 3x3 statistics then cost 9 LDS instead of 9 LDG + 9 conversions.
    __shared__ TaaCam S;
    __shared__ float4 tile[10][34];
    if (threadIdx.x == 0 && threadIdx.y == 0) load_cam(S.c, &cams[0]), load_cam(S.p, &cams[1]);
    {
        const int tx0 = blockIdx.x * 32 - 1, ty0 = y0 + blockIdx.y * 8 - 1;
        for (int i = threadIdx.y * 32 + threadIdx.x; i < 340; i += 256)
        {
            const int    ly = i / 34, lx = i - ly * 34;
            const int    gx = min(max(tx0 + lx, 0), curr_color.w - 1), gy = min(max(ty0 + ly, 0), curr_color.h - 1); // ClampScreenCoord
            const float3 sdr = rgb_to_ycocg<YCOCG>(hdr_to_sdr(max0(load_scene_colour<COMPOSE>(curr_color, ci, gx, gy))));
            tile[ly][lx]     = f4(sdr, 0.0f);
        }
    }
    __syncthreads();
    const CamS& cam = S.c;
    const int   x = blockIdx.x * blockDim.x + threadIdx.x;
    const int   y = y0 + blockIdx.y * blockDim.y + threadIdx.y;
    if (x >= out.w || y >= y1) return;

    const float posx = float(x) + 0.5f, posy = float(y) + 0.5f;
    float2      mv   = __ldg(&motion.at(x, y));
    mv.x *= 0.5f, mv.y *= -0.5f;
    const float ppx = posx - mv.x * cam.vw, ppy = posy - mv.y * cam.vh;
    const float3 currHDR = max0(load_scene_colour<COMPOSE>(curr_color, ci, x, y));

    if (!(ppx >= 0.0f && ppy >= 0.0f && ppx < cam.vw && ppy < cam.vh) || A.ResetAccumulation)
    {
        st_cs(&out.at(x, y), f4(currHDR, 0.5f));
        return;
    }
    const float aspect = cam.vw * cam.ivh;
    const float mf     = saturate(1.0f - fsqrt((mv.x * aspect) * (mv.x * aspect) + mv.y * mv.y) * 256.0f);

    // ComputeDepthDisocclusion :117-136 (unclamped loads)
    float depthFactor;
    {
        const int   pix = (int)ppx, piy = (int)ppy;
        const float cd  = __ldg(&curr_depth.at(x, y));
        const float lc  = fabsf(depth_to_camz(cd, cam));
        // max_i exp(-r_i) > 0.9  <=>  min_i r_i < -ln(0.9): the predicate is evaluated without the nine exp()
        float rmin = kFltMax;
#pragma unroll
        for (int dy = -1; dy <= 1; ++dy)
#pragma unroll
            for (int dx = -1; dx <= 1; ++dx)
            {
                const float pd = load0(prev_depth, pix + dx, piy + dy);
                const float lp = fabsf(fdiv(S.p.m32 - pd * S.p.m33, pd * S.p.m23 - S.p.m22));
                rmin           = fminf(rmin, fdiv(fabsf(lc - lp), fmaxf(fmaxf(lc, lp), 1e-6f)));
            }
        depthFactor = rmin < 0.105360516f ? 1.0f : 0.0f;
    }

    float4 prevHDR;
    if (BICUBIC)
    {
        // SamplePrevColorCatmullRom :138-173 (5 bilinear taps)
        const float cx = floorf(ppx - 0.5f) + 0.5f, cy = floorf(ppy - 0.5f) + 0.5f;
        const float fx = ppx - cx, fy = ppy - cy;
        const float fx2 = fx * fx, fy2 = fy * fy, fx3 = fx2 * fx, fy3 = fy2 * fy;
        const float w0x = -0.5f * fx3 + fx2 - 0.5f * fx, w0y = -0.5f * fy3 + fy2 - 0.5f * fy;
        const float w1x = 1.5f * fx3 - 2.5f * fx2 + 1.0f, w1y = 1.5f * fy3 - 2.5f * fy2 + 1.0f;
        const float w2x = -1.5f * fx3 + 2.0f * fx2 + 0.5f * fx, w2y = -1.5f * fy3 + 2.0f * fy2 + 0.5f * fy;
        const float w3x = 0.5f * fx3 - 0.5f * fx2, w3y = 0.5f * fy3 - 0.5f * fy2;
        const float w12x = w1x + w2x, w12y = w1y + w2y;
        const float t0x = (cx - 1.0f) * cam.ivw, t0y = (cy - 1.0f) * cam.ivh;
        const float t3x = (cx + 2.0f) * cam.ivw, t3y = (cy + 2.0f) * cam.ivh;
        const float t12x = (cx + fdiv(w2x, w12x)) * cam.ivw, t12y = (cy + fdiv(w2y, w12y)) * cam.ivh;
        const float p0 = w12x * w0y, p1 = w0x * w12y, p2 = w12x * w12y, p3 = w3x * w12y, p4 = w12x * w3y;
        // The five bilinear taps touch 12 texels, not 20: the "0" and "3" coordinates are exact texel centres (after the
        // sampler's 1/256 snap their second bilinear weight is exactly 0), only the "12" coordinate blends two texels.
        const int   PW = prev_accum.w, PH = prev_accum.h;
        const float fpw = float(PW), fph = float(PH);
        const float sx12 = snap8(t12x * fpw - 0.5f), sy12 = snap8(t12y * fph - 0.5f);
        const float bx = floorf(sx12), by = floorf(sy12);
        const float qx = sx12 - bx, qy = sy12 - by; // weights of the right / lower texel of the "12" pair
        auto cxi = [&](int v) { return min(max(v, 0), PW - 1); };
        auto cyi = [&](int v) { return min(max(v, 0), PH - 1); };
        const int xa = cxi((int)bx), xb = cxi((int)bx + 1), ya = cyi((int)by), yb = cyi((int)by + 1);
        const int x0 = cxi((int)rintf(snap8(t0x * fpw - 0.5f))), x3 = cxi((int)rintf(snap8(t3x * fpw - 0.5f)));
        const int y0i = cyi((int)rintf(snap8(t0y * fph - 0.5f))), y3i = cyi((int)rintf(snap8(t3y * fph - 0.5f)));
        auto ld = [&](int tx, int ty) { return __ldg(&prev_accum.at(tx, ty)); };
        auto mixx = [&](int ty) { return ld(xa, ty) * (1.0f - qx) + ld(xb, ty) * qx; };
        const float4 rowa = mixx(ya), rowb = mixx(yb);
        float4       r    = mixx(y0i) * p0;                                        // (12, 0)
        r = r + (ld(x0, ya) * (1.0f - qy) + ld(x0, yb) * qy) * p1;                 // (0, 12)
        r = r + (rowa * (1.0f - qy) + rowb * qy) * p2;                             // (12, 12)
        r = r + (ld(x3, ya) * (1.0f - qy) + ld(x3, yb) * qy) * p3;                 // (3, 12)
        r = r + mixx(y3i) * p4;                                                    // (12, 3)
        prevHDR = max0(r * frcp(p0 + p1 + p2 + p3 + p4));
    }
    else
    {
        prevHDR = max0(sample_linear_clamp(prev_accum, ppx * cam.ivw, ppy * cam.ivh));
    }

    const float3 currSDR = rgb_to_ycocg<YCOCG>(hdr_to_sdr(currHDR));
    const float3 prevSDR = rgb_to_ycocg<YCOCG>(hdr_to_sdr(xyz(prevHDR)));
    auto corrected_alpha = [&](float a) { return fminf(A.TemporalStabilityFactor, saturate(frcp(2.0f - a))); };

    if (A.SkipRejection)
    {
        const float3 o = sdr_to_hdr(ycocg_to_rgb<YCOCG>(lerp3(currSDR, prevSDR, prevHDR.w)));
        st_cs(&out.at(x, y), f4(o, corrected_alpha(prevHDR.w)));
        return;
    }

    const float gamma = lerpf(0.75f, 2.5f, mf * mf);
    // ComputePixelStatisticYCoCgSDR :191-222
    float3 m1 = make_float3(0.f, 0.f, 0.f), m2 = m1;
    float  wsum = 0.0f;
#pragma unroll
    for (int dx = -1; dx <= 1; ++dx)
#pragma unroll
        for (int dy = -1; dy <= 1; ++dy)
        {
            const float3 sdr = xyz(tile[threadIdx.y + 1 + dy][threadIdx.x + 1 + dx]);
            // exp(-3 r^2 / 4), r^2 in {0, 1, 2}: compile-time constants after unrolling
            const float  w   = GAUSS ? ((dx * dx + dy * dy) == 0 ? 1.0f : (dx * dx + dy * dy) == 1 ? 0.472366553f : 0.223130160f) : 1.0f;
            m1 = m1 + sdr * w, m2 = m2 + sdr * sdr * w;
            wsum += w;
        }
    const float3 mean = m1 * frcp(wsum);
    const float3 var  = m2 * frcp(wsum) - (mean * mean);
    const float3 sd   = make_float3(fsqrt(fmaxf(var.x, 0.f)), fsqrt(fmaxf(var.y, 0.f)), fsqrt(fmaxf(var.z, 0.f)));
    const float3 clipped = clip_to_aabb(prevSDR, currSDR, mean, gamma * sd);
    const float  alpha   = prevHDR.w * mf * depthFactor;
    const float3 o       = sdr_to_hdr(ycocg_to_rgb<YCOCG>(lerp3(currSDR, clipped, alpha)));
    st_cs(&out.at(x, y), f4(o, corrected_alpha(alpha)));
}

// =====================================================================================================================
// compose (reduced form of HnPostProcess.psh:145-185): rgb += ssr.rgb*ssr.a*scale ; rgb *= lerp(1, ao, scale)
// =====================================================================================================================
template <bool C16>
__global__ void __launch_bounds__(256) compose_kernel(TexRGBA<C16> color, View<const float4> ssr, View<const float> ao, float ssr_scale,
                                                      float ssao_scale, View<float4> out, int y0, int y1)
{
    const PixelXY pix = cta_pixel(y0);
    const int     x = pix.x, y = pix.y;
    if (x >= out.w || y >= y1) return;
    const float4 C = color.ld(x, y);
    float3       c = xyz(C);
    if (ssr.p && ssr_scale > 0.0f)
    {
        const float4 s = __ldg(&ssr.at(x, y));
        c              = c + xyz(s) * s.w * ssr_scale;
    }
    if (ao.p && ssao_scale > 0.0f) c = c * lerpf(1.0f, __ldg(&ao.at(x, y)), ssao_scale);
    st_cs(&out.at(x, y), f4(c, C.w));
}

// =====================================================================================================================
// ToneMap — ToneMapping.fxh:87-226 (all 11 operators) + LinearToSRGB (SRGBUtilities.fxh:27-33)
// =====================================================================================================================
template <int MODE>
__global__ void __launch_bounds__(256) tonemap_kernel(dfx_tonemap_attribs A, float aveLogLum, int to_srgb, View<const float4> in, View<float4> out,
                                                      int y0, int y1)
{
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    const int y = y0 + blockIdx.y;
    if (x >= out.w || y >= y1) return;
    const float4 C = __ldg(&in.at(x, y));
    float3       c = tone_map<MODE>(xyz(C), A, aveLogLum);
    if (to_srgb) c = linear_to_srgb(c);
    st_cs(&out.at(x, y), f4(c, C.w));
}
// the same with fAveLogLum = max(0.05, *lum_dev) (GetAverageSceneLuminance, AtmosphereShadersCommon.fxh:188-197), read on the device
template <int MODE>
__global__ void __launch_bounds__(256) tonemap_dev_kernel(dfx_tonemap_attribs A, const float* lum_dev, int to_srgb, View<const float4> in, View<float4> out,
                                                          int y0, int y1)
{
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    const int y = y0 + blockIdx.y;
    if (x >= out.w || y >= y1) return;
    const float  aveLogLum = fmaxf(0.05f, __ldg(lum_dev));
    const float4 C = __ldg(&in.at(x, y));
    float3       c = tone_map<MODE>(xyz(C), A, aveLogLum);
    if (to_srgb) c = linear_to_srgb(c);
    st_cs(&out.at(x, y), f4(c, C.w));
}

} // namespace dfx

using namespace dfx;

#define DFX_GRID(w, rows) dim3 block(32, 8), grid(div_up(w, 32), div_up(rows.y1 - rows.y0, 8))

static dfx_status launch_taa(void* stream, const dfx_camera_attribs* cameras_dev, const dfx_taa_attribs* attribs, uint32_t flags, bool compose,
                             const dfx_plane* ssr, const dfx_plane* ao, float ssr_scale, float ssao_scale, const dfx_plane* curr_color,
                             const dfx_plane* prev_accum, const dfx_plane* closest_motion, const dfx_plane* reprojected_depth,
                             const dfx_plane* previous_depth, const dfx_plane* out_accum, dfx_rows rows)
{
    DFX_REQUIRE(cameras_dev && attribs, "null argument");
    DFX_TEX4(cc, curr_color);
    DFX_VIEW(const float4, pa, prev_accum, DFX_FORMAT_RGBA32F);
    DFX_VIEW(const float2, mv, closest_motion, DFX_FORMAT_RG32F);
    DFX_VIEW(const float, cd, reprojected_depth, DFX_FORMAT_R32F);
    DFX_VIEW(const float, pd, previous_depth, DFX_FORMAT_R32F);
    DFX_VIEW(float4, out, out_accum, DFX_FORMAT_RGBA32F);
    DFX_SAME_SIZE(cc, pa);
    DFX_SAME_SIZE(cc, mv);
    DFX_SAME_SIZE(cc, cd);
    DFX_SAME_SIZE(cc, pd);
    DFX_SAME_SIZE(cc, out);
    DFX_REQUIRE(rows_ok(rows, out.h), "bad row range");
    if (rows.y1 == rows.y0) return DFX_OK;
    ComposeIn ci{View<const float4>{nullptr, 0, 0, 0}, View<const float>{nullptr, 0, 0, 0}, ssr_scale, ssao_scale};
    if (compose && ssr) DFX_REQUIRE(make_view<const float4>(ssr, DFX_FORMAT_RGBA32F, ci.ssr) && ci.ssr.w == cc.w && ci.ssr.h == cc.h, "bad ssr plane");
    if (compose && ao) DFX_REQUIRE(make_view<const float>(ao, DFX_FORMAT_R32F, ci.ao) && ci.ao.w == cc.w && ci.ao.h == cc.h, "bad ao plane");
    DFX_GRID(out.w, rows);
    cudaStream_t s = as_stream(stream);
#define TAA_LAUNCH(B, Y, G)                                                                                                            \
    do {                                                                                                                               \
        if (compose)                                                                                                                   \
            DFX_FMT16(is16(cc), C16, taa_kernel<B, Y, G, true, C16><<<grid, block, 0, s>>>(cameras_dev, *attribs, cc, ci, pa, mv, cd, pd, out, rows.y0, rows.y1));    \
        else                                                                                                                           \
            DFX_FMT16(is16(cc), C16, taa_kernel<B, Y, G, false, C16><<<grid, block, 0, s>>>(cameras_dev, *attribs, cc, ci, pa, mv, cd, pd, out, rows.y0, rows.y1));   \
    } while (0)
    switch (flags & 7u)
    {
        case 0: TAA_LAUNCH(false, false, false); break;
        case 1: TAA_LAUNCH(false, false, true); break;
        case 2: TAA_LAUNCH(true, false, false); break;
        case 3: TAA_LAUNCH(true, false, true); break;
        case 4: TAA_LAUNCH(false, true, false); break;
        case 5: TAA_LAUNCH(false, true, true); break;
        case 6: TAA_LAUNCH(true, true, false); break;
        case 7: TAA_LAUNCH(true, true, true); break;
    }
#undef TAA_LAUNCH
    DFX_LAUNCHED("taa_kernel");
    return DFX_OK;
}

extern "C" dfx_status dfx_pass_taa(void* stream, const dfx_camera_attribs* cameras_dev, const dfx_taa_attribs* attribs, uint32_t flags,
                                   const dfx_plane* curr_color, const dfx_plane* prev_accum, const dfx_plane* closest_motion,
                                   const dfx_plane* reprojected_depth, const dfx_plane* previous_depth, const dfx_plane* out_accum, dfx_rows rows)
{
    DFX_PROFILE(stream, "taa");
    return launch_taa(stream, cameras_dev, attribs, flags, false, nullptr, nullptr, 0.0f, 0.0f, curr_color, prev_accum, closest_motion, reprojected_depth,
                      previous_depth, out_accum, rows);
}

extern "C" dfx_status dfx_pass_compose_taa(void* stream, const dfx_camera_attribs* cameras_dev, const dfx_taa_attribs* attribs, uint32_t flags,
                                           const dfx_plane* color, const dfx_plane* ssr, const dfx_plane* ao, float ssr_scale, float ssao_scale,
                                           const dfx_plane* prev_accum, const dfx_plane* closest_motion, const dfx_plane* reprojected_depth,
                                           const dfx_plane* previous_depth, const dfx_plane* out_accum, dfx_rows rows)
{
    DFX_PROFILE(stream, "compose_taa");
    return launch_taa(stream, cameras_dev, attribs, flags, true, ssr, ao, ssr_scale, ssao_scale, color, prev_accum, closest_motion, reprojected_depth,
                      previous_depth, out_accum, rows);
}

extern "C" dfx_status dfx_pass_compose(void* stream, const dfx_plane* color, const dfx_plane* ssr, const dfx_plane* ao, float ssr_scale,
                                       float ssao_scale, const dfx_plane* out_, dfx_rows rows)
{
    DFX_PROFILE(stream, "compose");
    DFX_TEX4(c, color);
    DFX_VIEW(float4, out, out_, DFX_FORMAT_RGBA32F);
    DFX_SAME_SIZE(c, out);
    View<const float4> s{nullptr, 0, 0, 0};
    View<const float>  a{nullptr, 0, 0, 0};
    if (ssr)
    {
        DFX_REQUIRE(make_view<const float4>(ssr, DFX_FORMAT_RGBA32F, s) && s.w == c.w && s.h == c.h, "bad ssr plane");
    }
    if (ao)
    {
        DFX_REQUIRE(make_view<const float>(ao, DFX_FORMAT_R32F, a) && a.w == c.w && a.h == c.h, "bad ao plane");
    }
    DFX_REQUIRE(rows_ok(rows, out.h), "bad row range");
    if (rows.y1 == rows.y0) return DFX_OK;
    DFX_GRID(out.w, rows);
    DFX_FMT16(is16(c), C16, compose_kernel<C16><<<grid, block, 0, as_stream(stream)>>>(c, s, a, ssr_scale, ssao_scale, out, rows.y0, rows.y1));
    DFX_LAUNCHED("compose_kernel");
    return DFX_OK;
}

extern "C" dfx_status dfx_pass_tonemap(void* stream, const dfx_tonemap_attribs* attribs, float ave_log_lum, int32_t convert_to_srgb,
                                       const dfx_plane* color, const dfx_plane* out_, dfx_rows rows)
{
    DFX_PROFILE(stream, "tonemap");
    DFX_REQUIRE(attribs, "null argument");
    DFX_VIEW(const float4, c, color, DFX_FORMAT_RGBA32F);
    DFX_VIEW(float4, out, out_, DFX_FORMAT_RGBA32F);
    DFX_SAME_SIZE(c, out);
    DFX_REQUIRE(rows_ok(rows, out.h), "bad row range");
    if (rows.y1 == rows.y0) return DFX_OK;
    dim3         block(256), grid(div_up(out.w, 256), rows.y1 - rows.y0);
    cudaStream_t s = as_stream(stream);
#define TM_LAUNCH(M) tonemap_kernel<M><<<grid, block, 0, s>>>(*attribs, ave_log_lum, convert_to_srgb, c, out, rows.y0, rows.y1)
    switch (attribs->iToneMappingMode)
    {
        case DFX_TONE_MAPPING_MODE_NONE: TM_LAUNCH(DFX_TONE_MAPPING_MODE_NONE); break;
        case DFX_TONE_MAPPING_MODE_EXP: TM_LAUNCH(DFX_TONE_MAPPING_MODE_EXP); break;
        case DFX_TONE_MAPPING_MODE_REINHARD: TM_LAUNCH(DFX_TONE_MAPPING_MODE_REINHARD); break;
        case DFX_TONE_MAPPING_MODE_REINHARD_MOD: TM_LAUNCH(DFX_TONE_MAPPING_MODE_REINHARD_MOD); break;
        case DFX_TONE_MAPPING_MODE_UNCHARTED2: TM_LAUNCH(DFX_TONE_MAPPING_MODE_UNCHARTED2); break;
        case DFX_TONE_MAPPING_MODE_FILMIC_ALU: TM_LAUNCH(DFX_TONE_MAPPING_MODE_FILMIC_ALU); break;
        case DFX_TONE_MAPPING_MODE_LOGARITHMIC: TM_LAUNCH(DFX_TONE_MAPPING_MODE_LOGARITHMIC); break;
        case DFX_TONE_MAPPING_MODE_ADAPTIVE_LOG: TM_LAUNCH(DFX_TONE_MAPPING_MODE_ADAPTIVE_LOG); break;
        case DFX_TONE_MAPPING_MODE_AGX: TM_LAUNCH(DFX_TONE_MAPPING_MODE_AGX); break;
        case DFX_TONE_MAPPING_MODE_AGX_CUSTOM: TM_LAUNCH(DFX_TONE_MAPPING_MODE_AGX_CUSTOM); break;
        case DFX_TONE_MAPPING_MODE_PBR_NEUTRAL: TM_LAUNCH(DFX_TONE_MAPPING_MODE_PBR_NEUTRAL); break;
        case DFX_TONE_MAPPING_MODE_COMMERCE: TM_LAUNCH(DFX_TONE_MAPPING_MODE_COMMERCE); break;
        default: return set_error(DFX_ERR_INVALID_ARG, "unknown tone mapping mode %d", attribs->iToneMappingMode);
    }
#undef TM_LAUNCH
    DFX_LAUNCHED("tonemap_kernel");
    return DFX_OK;
}

extern "C" dfx_status dfx_pass_tonemap_dev(void* stream, const dfx_tonemap_attribs* attribs, const float* ave_log_lum_dev, int32_t convert_to_srgb,
                                           const dfx_plane* color, const dfx_plane* out_, dfx_rows rows)
{
    DFX_PROFILE(stream, "tonemap");
    DFX_REQUIRE(attribs && ave_log_lum_dev, "null argument");
    DFX_VIEW(const float4, c, color, DFX_FORMAT_RGBA32F);
    DFX_VIEW(float4, out, out_, DFX_FORMAT_RGBA32F);
    DFX_SAME_SIZE(c, out);
    DFX_REQUIRE(rows_ok(rows, out.h), "bad row range");
    DFX_REQUIRE(attribs->iToneMappingMode >= 0 && attribs->iToneMappingMode <= DFX_TONE_MAPPING_MODE_COMMERCE, "unknown tone mapping mode %d", attribs->iToneMappingMode);
    if (rows.y1 == rows.y0) return DFX_OK;
    dim3         block(256), grid(div_up(out.w, 256), rows.y1 - rows.y0);
    cudaStream_t s = as_stream(stream);
#define TM_LAUNCH(M) tonemap_dev_kernel<M><<<grid, block, 0, s>>>(*attribs, ave_log_lum_dev, convert_to_srgb, c, out, rows.y0, rows.y1)
    switch (attribs->iToneMappingMode)
    {
        case DFX_TONE_MAPPING_MODE_NONE: TM_LAUNCH(DFX_TONE_MAPPING_MODE_NONE); break;
        case DFX_TONE_MAPPING_MODE_EXP: TM_LAUNCH(DFX_TONE_MAPPING_MODE_EXP); break;
        case DFX_TONE_MAPPING_MODE_REINHARD: TM_LAUNCH(DFX_TONE_MAPPING_MODE_REINHARD); break;
        case DFX_TONE_MAPPING_MODE_REINHARD_MOD: TM_LAUNCH(DFX_TONE_MAPPING_MODE_REINHARD_MOD); break;
        case DFX_TONE_MAPPING_MODE_UNCHARTED2: TM_LAUNCH(DFX_TONE_MAPPING_MODE_UNCHARTED2); break;
        case DFX_TONE_MAPPING_MODE_FILMIC_ALU: TM_LAUNCH(DFX_TONE_MAPPING_MODE_FILMIC_ALU); break;
        case DFX_TONE_MAPPING_MODE_LOGARITHMIC: TM_LAUNCH(DFX_TONE_MAPPING_MODE_LOGARITHMIC); break;
        case DFX_TONE_MAPPING_MODE_ADAPTIVE_LOG: TM_LAUNCH(DFX_TONE_MAPPING_MODE_ADAPTIVE_LOG); break;
        case DFX_TONE_MAPPING_MODE_AGX: TM_LAUNCH(DFX_TONE_MAPPING_MODE_AGX); break;
        case DFX_TONE_MAPPING_MODE_AGX_CUSTOM: TM_LAUNCH(DFX_TONE_MAPPING_MODE_AGX_CUSTOM); break;
        case DFX_TONE_MAPPING_MODE_PBR_NEUTRAL: TM_LAUNCH(DFX_TONE_MAPPING_MODE_PBR_NEUTRAL); break;
        default: TM_LAUNCH(DFX_TONE_MAPPING_MODE_COMMERCE); break;
    }
#undef TM_LAUNCH
    DFX_LAUNCHED("tonemap_dev_kernel");
    return DFX_OK;
}

// ORACLE — TEST INFRASTRUCTURE ONLY (see oracle_math.h). Pinned against the reference's own shaders (oracle/refshader/build_exposure.py,
// harness exposure.inc; tests/test_auto_exposure_cpu.py).
// Auto exposure with light adaptation as EpipolarLightScattering computes it (the shaders have no dependence on the atmosphere;
// without light scattering the inscattering term is 0 and the extinction 1):
//   GetWeightedLogLum          AtmosphereShadersCommon.fxh:199-205 (MinLuminance 0.01: UnwarpEpipolarScattering.fx:305)
//   64x64 RG16F target         point samples of the colour (Sam_PointClamp, EpipolarLightScattering.cpp:1751; :863-883)
//   GenerateMips               down to 1x1 (…cpp:2469, :2503): fp32 mean of the four texels, rounded to half (DESIGN.md §2)
//   UpdateAverageLuminancePS   UpdateAverageLuminance.fx:12-29, output alpha-blended into the 1x1 R16F state (…cpp:1823-1827)
// and the every-pixel variant of the product (DFX_LUMINANCE_SAMPLING_FULL), with an fp64 sum.
#include "oracle_exposure.h"
#include "oracle_quant.h"
#include <algorithm>
#include <cmath>

namespace orc
{

float2 weighted_log_lum(float3 color, float min_luminance)
{
    const float lum = color.x * 0.212671f + color.y * 0.715160f + color.z * 0.072169f; // dot(Color, RGB_TO_LUMINANCE), left to right
    const float w   = saturate((lum - min_luminance) / min_luminance);
    const float ll  = std::log(std::max(lum, 1e-5f));
    return float2(ll * w, w);
}

float2 update_average_luminance_ps(float2 loglum_w, float elapsed, bool light_adaptation)
{
    float weight = 1.0f;
    if (light_adaptation)
    {
        const float rate = 1.0f;
        weight           = 1.0f - std::exp(-rate * elapsed);
    }
    const float log_lum = loglum_w.x / std::max(loglum_w.y, 1e-6f);
    weight *= saturate(loglum_w.y / 1e-3f);
    return float2(std::exp(log_lum), weight);
}

void blend_average_luminance(LumState& s, float measured, float weight)
{
    // BS_AlphaBlend: dst = src * a + dst * (1 - a), stored in R16F
    s.value       = q_half(measured * weight + s.value * (1.0f - weight));
    s.ave_log_lum = std::max(0.05f, s.value);
    s.measured    = measured;
    s.weight      = weight;
}

float2 luminance_reference_level(const Tex<float4>& color)
{
    constexpr int N = 64;
    std::vector<float2> lv(N * N);
    for (int j = 0; j < N; ++j)
        for (int i = 0; i < N; ++i)
        {
            const float2 uv((float(i) + 0.5f) * (1.0f / N), (float(j) + 0.5f) * (1.0f / N));
            const float4 c = sample_point_clamp(color, uv);
            const float2 l = weighted_log_lum(float3(c.x, c.y, c.z), kExposureMinLuminance);
            lv[j * N + i]  = float2(q_half(l.x), q_half(l.y));
        }
    for (int n = N / 2; n >= 1; n >>= 1)
    {
        std::vector<float2> nx(n * n);
        const int           src = 2 * n;
        for (int j = 0; j < n; ++j)
            for (int i = 0; i < n; ++i)
            {
                const float2 a = lv[(2 * j) * src + 2 * i], b = lv[(2 * j) * src + 2 * i + 1];
                const float2 c = lv[(2 * j + 1) * src + 2 * i], d = lv[(2 * j + 1) * src + 2 * i + 1];
                nx[j * n + i]  = float2(q_half((a.x + b.x + c.x + d.x) * 0.25f), q_half((a.y + b.y + c.y + d.y) * 0.25f));
            }
        lv.swap(nx);
    }
    return lv[0];
}

void update_average_luminance(const Tex<float4>& color, int sampling, float elapsed, bool light_adaptation, LumState& s)
{
    if (sampling == 1)
    {
        const float2 top = luminance_reference_level(color);
        const float2 o   = update_average_luminance_ps(top, elapsed, light_adaptation);
        blend_average_luminance(s, o.x, o.y);
        return;
    }
    // every pixel: fp32 per pixel, fp64 sum; the means are what the 1x1 level of a full-resolution mip chain holds
    double swl = 0.0, sw = 0.0;
    for (const float4& c : color.d)
    {
        const float2 l = weighted_log_lum(float3(c.x, c.y, c.z), kExposureMinLuminance);
        swl += double(l.x), sw += double(l.y);
    }
    const double n = double(color.w) * double(color.h), mwl = swl / n, mw = sw / n;
    const float  measured = float(std::exp(mwl / std::max(mw, 1e-6)));
    float        weight   = light_adaptation ? 1.0f - std::exp(-elapsed) : 1.0f;
    weight *= saturate(float(mw) / 1e-3f);
    blend_average_luminance(s, measured, weight);
}

} // namespace orc

// ---------------------------------------------------------------------------------------------------------------------------------
// C API (ctypes, oracle/exposure_py.py). This file is its own library (oracle/_build/liboracle_exposure.so), next to liboracle.so.
// ---------------------------------------------------------------------------------------------------------------------------------
#define ORC_EXPOSURE_API extern "C" __attribute__((visibility("default")))
using namespace orc;

ORC_EXPOSURE_API void orc_weighted_log_lum(const float* rgb, float* out2, int n)
{
    for (int i = 0; i < n; ++i)
    {
        const float2 l = weighted_log_lum(float3(rgb[3 * i], rgb[3 * i + 1], rgb[3 * i + 2]), kExposureMinLuminance);
        out2[2 * i] = l.x, out2[2 * i + 1] = l.y;
    }
}
ORC_EXPOSURE_API void orc_update_average_luminance_ps(const float* loglum_w, const float* elapsed, int light_adaptation, float* out2, int n)
{
    for (int i = 0; i < n; ++i)
    {
        const float2 o = update_average_luminance_ps(float2(loglum_w[2 * i], loglum_w[2 * i + 1]), elapsed[i], light_adaptation != 0);
        out2[2 * i] = o.x, out2[2 * i + 1] = o.y;
    }
}
// one update of `state4` (value, ave_log_lum, measured, weight) from an RGBA frame; sampling 1 = reference, 2 = every pixel
ORC_EXPOSURE_API int orc_update_average_luminance(const float* rgba, int w, int hgt, int sampling, float elapsed, int light_adaptation, float* state4)
{
    if (w <= 0 || hgt <= 0 || (sampling != 1 && sampling != 2)) return 1;
    Tex<float4> t(w, hgt);
    for (size_t i = 0; i < t.d.size(); ++i) t.d[i] = float4(rgba[4 * i], rgba[4 * i + 1], rgba[4 * i + 2], rgba[4 * i + 3]);
    LumState s{state4[0], state4[1], state4[2], state4[3]};
    update_average_luminance(t, sampling, elapsed, light_adaptation != 0, s);
    state4[0] = s.value, state4[1] = s.ave_log_lum, state4[2] = s.measured, state4[3] = s.weight;
    return 0;
}

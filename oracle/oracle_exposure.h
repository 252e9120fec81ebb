// ORACLE — TEST INFRASTRUCTURE ONLY. Auto exposure with light adaptation (oracle_exposure.cpp).
#pragma once
#include "oracle_common.h"
#include "oracle_tex.h"

namespace orc
{
constexpr float kExposureMinLuminance = 0.01f; // UnwarpEpipolarScattering.fx:305

struct LumState // the 1x1 R16F average-luminance target (cleared to 0.1 at creation, EpipolarLightScattering.cpp:885-905)
{
    float value = 0.0999755859375f, ave_log_lum = 0.0999755859375f; // half-rounded state (R16F holds 0.1 as this), max(0.05, state)
    float measured = 0.0f, weight = 0.0f;   // the last update's exp(mean wlogL / mean w) and blend weight
};

float2 weighted_log_lum(float3 color, float min_luminance);                                 // AtmosphereShadersCommon.fxh:199-205
float2 update_average_luminance_ps(float2 loglum_w, float elapsed, bool light_adaptation);  // UpdateAverageLuminance.fx:12-29 -> (exp(LogLum), weight)
void   blend_average_luminance(LumState& s, float measured, float weight);                 // BS_AlphaBlend into R16F
float2 luminance_reference_level(const Tex<float4>& color);                                // the 1x1 level of the 64x64 RG16F chain
// sampling 1 = the reference's 64x64 point samples, 2 = every pixel (fp64 sum)
void update_average_luminance(const Tex<float4>& color, int sampling, float elapsed, bool light_adaptation, LumState& s);
} // namespace orc

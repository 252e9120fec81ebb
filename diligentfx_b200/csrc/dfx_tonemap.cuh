// dfx_tonemap.cuh — ToneMap M1 (all 11 operators, ToneMapping.fxh:87-226) + LinearToSRGB (SRGBUtilities.fxh:27-33) as device
// functions, shared by the stand-alone tone-map pass (dfx_taa_tonemap.cu) and the Bloom composite that fuses it (dfx_bloom.cu).
#pragma once
#include "dfx_common.cuh"

namespace dfx
{
DFX_HD float3 max0(float3 c) { return make_float3(fmaxf(c.x, 0.f), fmaxf(c.y, 0.f), fmaxf(c.z, 0.f)); }
DFX_HD float4 max0(float4 c) { return make_float4(fmaxf(c.x, 0.f), fmaxf(c.y, 0.f), fmaxf(c.z, 0.f), fmaxf(c.w, 0.f)); }

DFX_HD float3 uncharted2(float3 x) // :8-19
{
    const float A = 0.15f, B = 0.50f, C = 0.10f, D = 0.20f, E = 0.02f, F = 0.30f;
    auto        f = [&](float v) { return fdiv(v * (A * v + C * B) + D * E, v * (A * v + B) + D * F) - E / F; };
    return make_float3(f(x.x), f(x.y), f(x.z));
}
// pow via MUFU lg2/ex2 (relative error ~1e-6 at these exponents): the tone map is a full-screen element-wise pass that
// the correctly-rounded powf() would make ALU-bound instead of HBM-bound
DFX_HD float fpow(float v, float e) { return __powf(v, e); }
DFX_HD float3 pow3(float3 v, float e) { return make_float3(fpow(v.x, e), fpow(v.y, e), fpow(v.z, e)); }
DFX_HD float3 srgb_to_linear(float3 s)
{
    auto f = [](float v) {
        float hi = fpow(saturate((v + 0.055f) * (1.0f / 1.055f)), 2.4f);
        return lerpf(v / 12.92f, hi, v >= 0.04045f ? 1.0f : 0.0f);
    };
    return make_float3(f(s.x), f(s.y), f(s.z));
}
DFX_HD float3 linear_to_srgb(float3 c)
{
    auto f = [](float v) {
        float hi = fpow(v, 1.0f / 2.4f) * 1.055f - 0.055f;
        return lerpf(v * 12.92f, hi, v >= 0.0031308f ? 1.0f : 0.0f);
    };
    return make_float3(f(c.x), f(c.y), f(c.z));
}
DFX_HD float3 agx(float3 c) // :36-58
{
    float3 t = make_float3(0.842479062253094f * c.x + 0.0784335999999992f * c.y + 0.0792237451477643f * c.z,
                           0.0423282422610123f * c.x + 0.878468636469772f * c.y + 0.0791661274605434f * c.z,
                           0.0423756549057051f * c.x + 0.0784336f * c.y + 0.879142973793104f * c.z);
    const float mn = -12.47393f, mx = 4.026069f;
    auto        enc = [&](float v) { return (fminf(fmaxf(log2f(v), mn), mx) - mn) / (mx - mn); };
    t               = make_float3(enc(t.x), enc(t.y), enc(t.z));
    auto poly = [](float x) {
        float x2 = x * x, x4 = x2 * x2;
        return 15.5f * x4 * x2 - 40.14f * x4 * x + 31.96f * x4 - 6.868f * x2 * x + 0.4298f * x2 + 0.1191f * x - 0.00232f;
    };
    return make_float3(poly(t.x), poly(t.y), poly(t.z));
}
DFX_HD float3 agx_eotf(float3 c) // :60-74
{
    float3 t = make_float3(+1.19687900512017f * c.x - 0.0980208811401368f * c.y - 0.0990297440797205f * c.z,
                           -0.0528968517574562f * c.x + 1.15190312990417f * c.y - 0.0989611768448433f * c.z,
                           -0.0529716355144438f * c.x - 0.0980434501171241f * c.y + 1.15107367264116f * c.z);
    return srgb_to_linear(t);
}

template <int MODE>
DFX_HD float3 tone_map(float3 color, const dfx_tonemap_attribs& A, float aveLogLum)
{
    const float3 lumw  = make_float3(0.212671f, 0.715160f, 0.072169f);
    const float  scale = A.fMiddleGray / aveLogLum;
    color              = max0(color);
    const float  lum0  = fmaxf(dot(lumw, color), 1e-10f);
    const float  lumS  = lum0 * scale;
    const float3 cS    = color * scale;
    const float  wp    = A.fWhitePoint;
    if (MODE == DFX_TONE_MAPPING_MODE_EXP) return (1.0f - expf(-lumS)) * pow3(color / lum0, A.fLuminanceSaturation);
    if (MODE == DFX_TONE_MAPPING_MODE_REINHARD) return (lumS / (1.0f + lumS)) * pow3(color / lum0, A.fLuminanceSaturation);
    if (MODE == DFX_TONE_MAPPING_MODE_REINHARD_MOD) return (lumS * (1.0f + lumS / (wp * wp)) / (1.0f + lumS)) * pow3(color / lum0, A.fLuminanceSaturation);
    if (MODE == DFX_TONE_MAPPING_MODE_UNCHARTED2)
    {
        const float3 curr = uncharted2(2.0f * cS);
        const float3 w    = uncharted2(make_float3(wp, wp, wp));
        return curr * make_float3(frcp(w.x), frcp(w.y), frcp(w.z));
    }
    if (MODE == DFX_TONE_MAPPING_MODE_FILMIC_ALU)
    {
        auto f = [](float v) {
            v = fmaxf(v - 0.004f, 0.0f);
            v = (v * (6.2f * v + 0.5f)) / (v * (6.2f * v + 1.7f) + 0.06f);
            return powf(v, 2.2f);
        };
        return make_float3(f(cS.x), f(cS.y), f(cS.z));
    }
    if (MODE == DFX_TONE_MAPPING_MODE_LOGARITHMIC) return (log10f(1.0f + lumS) / log10f(1.0f + wp)) * pow3(color / lum0, A.fLuminanceSaturation);
    if (MODE == DFX_TONE_MAPPING_MODE_ADAPTIVE_LOG)
    {
        const float l = 1.0f / log10f(1.0f + wp) * logf(1.0f + lumS) / logf(2.0f + 8.0f * powf(lumS / wp, logf(0.85f) / logf(0.5f)));
        return l * pow3(color / lum0, A.fLuminanceSaturation);
    }
    if (MODE == DFX_TONE_MAPPING_MODE_AGX) return agx_eotf(agx(cS));
    if (MODE == DFX_TONE_MAPPING_MODE_AGX_CUSTOM)
    {
        float3      c   = agx(cS);
        const float lum = dot(c, lumw);
        c               = pow3(c * A.AgXSlope + make_float3(A.AgXOffset, A.AgXOffset, A.AgXOffset), A.AgXPower);
        c               = make_float3(lum, lum, lum) + A.AgXSaturation * (c - make_float3(lum, lum, lum));
        return agx_eotf(c);
    }
    if (MODE == DFX_TONE_MAPPING_MODE_PBR_NEUTRAL)
    {
        float3      c   = color * (0.3f / aveLogLum);
        const float sc  = 0.8f - 0.04f, desat = 0.15f;
        const float mn  = fminf(c.x, fminf(c.y, c.z));
        const float off = mn < 0.08f ? mn - 6.25f * mn * mn : 0.04f;
        c               = c - make_float3(off, off, off);
        const float peak = fmaxf(c.x, fmaxf(c.y, c.z));
        if (peak >= sc)
        {
            const float d = 1.0f - sc, np = 1.0f - d * d / (peak + d - sc);
            c             = c * (np / peak);
            const float g = 1.0f - 1.0f / (desat * (peak - np) + 1.0f);
            c             = lerp3(c, make_float3(np, np, np), g);
        }
        return c;
    }
    if (MODE == DFX_TONE_MAPPING_MODE_COMMERCE)
    {
        float3      c  = color * (0.3f / aveLogLum);
        const float sc = 0.8f, desat = 0.5f, d = 1.0f - sc;
        const float peak = fmaxf(c.x, fmaxf(c.y, c.z));
        if (peak >= sc)
        {
            const float np = 1.0f - d * d / (peak + d - sc), ip = 1.0f / peak;
            const float3 e = c * (1.0f - sc * ip);
            const float extra = e.x * 1.0f + e.y * 1.0f + e.z * 1.0f;
            c             = c * (np * ip);
            const float g = 1.0f - 3.0f / (desat * extra + 3.0f);
            c             = lerp3(c, make_float3(1.f, 1.f, 1.f), g);
        }
        return c;
    }
    return color;
}

DFX_HD float3 tone_map_rt(int mode, float3 color, const dfx_tonemap_attribs& A, float aveLogLum)
{
    switch (mode) // warp-uniform
    {
        case DFX_TONE_MAPPING_MODE_EXP: return tone_map<DFX_TONE_MAPPING_MODE_EXP>(color, A, aveLogLum);
        case DFX_TONE_MAPPING_MODE_REINHARD: return tone_map<DFX_TONE_MAPPING_MODE_REINHARD>(color, A, aveLogLum);
        case DFX_TONE_MAPPING_MODE_REINHARD_MOD: return tone_map<DFX_TONE_MAPPING_MODE_REINHARD_MOD>(color, A, aveLogLum);
        case DFX_TONE_MAPPING_MODE_UNCHARTED2: return tone_map<DFX_TONE_MAPPING_MODE_UNCHARTED2>(color, A, aveLogLum);
        case DFX_TONE_MAPPING_MODE_FILMIC_ALU: return tone_map<DFX_TONE_MAPPING_MODE_FILMIC_ALU>(color, A, aveLogLum);
        case DFX_TONE_MAPPING_MODE_LOGARITHMIC: return tone_map<DFX_TONE_MAPPING_MODE_LOGARITHMIC>(color, A, aveLogLum);
        case DFX_TONE_MAPPING_MODE_ADAPTIVE_LOG: return tone_map<DFX_TONE_MAPPING_MODE_ADAPTIVE_LOG>(color, A, aveLogLum);
        case DFX_TONE_MAPPING_MODE_AGX: return tone_map<DFX_TONE_MAPPING_MODE_AGX>(color, A, aveLogLum);
        case DFX_TONE_MAPPING_MODE_AGX_CUSTOM: return tone_map<DFX_TONE_MAPPING_MODE_AGX_CUSTOM>(color, A, aveLogLum);
        case DFX_TONE_MAPPING_MODE_PBR_NEUTRAL: return tone_map<DFX_TONE_MAPPING_MODE_PBR_NEUTRAL>(color, A, aveLogLum);
        case DFX_TONE_MAPPING_MODE_COMMERCE: return tone_map<DFX_TONE_MAPPING_MODE_COMMERCE>(color, A, aveLogLum);
        default: return tone_map<DFX_TONE_MAPPING_MODE_NONE>(color, A, aveLogLum);
    }
}

struct ToneMapIn // what the Bloom composite needs to apply the final ToneMap(+sRGB) in its epilogue
{
    dfx_tonemap_attribs attribs;
    float               ave_log_lum;
    int                 to_srgb;
    const float*        ave_log_lum_dev = nullptr; // the *_dev entries: fAveLogLum = max(0.05, *ave_log_lum_dev) instead of ave_log_lum
};

} // namespace dfx

// PostProcessEffects.hpp — ScreenSpaceAmbientOcclusion, ScreenSpaceReflection, Bloom, TemporalAntiAliasing and ToneMap()
// with the reference's public signatures, implemented over the C-ABI:
//   PostProcess/ScreenSpaceAmbientOcclusion/interface/ScreenSpaceAmbientOcclusion.hpp:59-136
//   PostProcess/ScreenSpaceReflection/interface/ScreenSpaceReflection.hpp:64-139
//   PostProcess/Bloom/interface/Bloom.hpp:60-114
//   PostProcess/TemporalAntiAliasing/interface/TemporalAntiAliasing.hpp:62-156
//   Shaders/PostProcess/ToneMapping/public/ToneMapping.fxh:87-226 (a shader include in the reference: no class exists)
// Call protocol is the reference's: every frame PostFXContext::PrepareResources -> each effect's PrepareResources ->
// PostFXContext::Execute -> effects' Execute. Returns are void, nothing throws; problems are logged (LOG_ERROR_MESSAGE
// behaviour) and the effect's output is left untouched. UpdateUI() (ImGui panels) is out of scope and returns false.
#pragma once
#include "PostFXContext.hpp"

namespace Diligent
{

// =====================================================================================================================
class ScreenSpaceAmbientOcclusion
{
public:
    enum FEATURE_FLAGS : Uint32
    {
        FEATURE_FLAG_NONE                 = 0u,
        FEATURE_FLAG_HALF_PRECISION_DEPTH = 1u << 0u, // AO self-occlusion offset 0.005; planes stay fp32 here
        FEATURE_FLAG_HALF_RESOLUTION      = 1u << 1u  // AO at half resolution + bilateral upsampling
    };
    enum ALGORITHM_TYPE : Uint32
    {
        ALGORITHM_TYPE_GTAO = 0,
        ALGORITHM_TYPE_HBAO = 1,
        ALGORITHM_TYPE_VBAO = 2
    };
    struct RenderAttributes
    {
        IRenderDevice*                                  pDevice          = nullptr;
        IRenderStateCache*                              pStateCache      = nullptr;
        IDeviceContext*                                 pDeviceContext   = nullptr;
        PostFXContext*                                  pPostFXContext   = nullptr;
        ITextureView*                                   pDepthBufferSRV  = nullptr; // R32_FLOAT
        ITextureView*                                   pNormalBufferSRV = nullptr; // RGBA32_FLOAT, xyz = world-space normal
        const HLSL::ScreenSpaceAmbientOcclusionAttribs* pSSAOAttribs     = nullptr;
    };
    struct CreateInfo
    {
        bool EnableAsyncCreation = false;
    };

    ScreenSpaceAmbientOcclusion(IRenderDevice* pDevice, const CreateInfo& CI)
    {
        (void)pDevice, (void)CI;
        detail::Check(dfx_ssao_create(&m_Fx), "dfx_ssao_create");
        if (m_Fx) dfx_ssao_set_alpha_interpolation(m_Fx, -1.0f); // reference behaviour: fade in over the first second (m_FrameTimer); SetAlphaInterpolation() pins it
    }
    ~ScreenSpaceAmbientOcclusion() { dfx_ssao_destroy(m_Fx); }
    ScreenSpaceAmbientOcclusion(const ScreenSpaceAmbientOcclusion&)            = delete;
    ScreenSpaceAmbientOcclusion& operator=(const ScreenSpaceAmbientOcclusion&) = delete;

    void PrepareResources(IRenderDevice* pDevice, IDeviceContext* pDeviceContext, PostFXContext* pPostFXContext, FEATURE_FLAGS FeatureFlags)
    {
        (void)pDeviceContext;
        DFX_DEV_CHECK_ERR(pDevice != nullptr, "pDevice must not be null");
        DFX_DEV_CHECK_ERR(pPostFXContext != nullptr, "pPostFXContext must not be null");
        if (pPostFXContext) detail::Check(dfx_ssao_prepare(m_Fx, pPostFXContext->GetHandle(), static_cast<uint32_t>(FeatureFlags)), "ScreenSpaceAmbientOcclusion::PrepareResources");
    }
    void Execute(const RenderAttributes& RenderAttribs)
    {
        DFX_DEV_CHECK_ERR(RenderAttribs.pDevice != nullptr, "RenderAttribs.pDevice must not be null");
        DFX_DEV_CHECK_ERR(RenderAttribs.pDeviceContext != nullptr, "RenderAttribs.pDeviceContext must not be null");
        DFX_DEV_CHECK_ERR(RenderAttribs.pPostFXContext != nullptr, "RenderAttribs.pPostFXContext must not be null");
        DFX_DEV_CHECK_ERR(RenderAttribs.pDepthBufferSRV != nullptr, "RenderAttribs.pDepthBufferSRV must not be null");
        DFX_DEV_CHECK_ERR(RenderAttribs.pNormalBufferSRV != nullptr, "RenderAttribs.pNormalBufferSRV must not be null");
        DFX_DEV_CHECK_ERR(RenderAttribs.pSSAOAttribs != nullptr, "RenderAttribs.pSSAOAttribs must not be null");
        dfx_ssao_render_attribs a{};
        a.stream  = detail::StreamOf(RenderAttribs.pDeviceContext);
        a.postfx  = RenderAttribs.pPostFXContext ? RenderAttribs.pPostFXContext->GetHandle() : nullptr;
        a.depth   = RenderAttribs.pDepthBufferSRV ? RenderAttribs.pDepthBufferSRV->GetPlane() : nullptr;
        a.normal  = RenderAttribs.pNormalBufferSRV ? RenderAttribs.pNormalBufferSRV->GetPlane() : nullptr;
        a.attribs = RenderAttribs.pSSAOAttribs;
        detail::Check(dfx_ssao_execute(m_Fx, &a), "ScreenSpaceAmbientOcclusion::Execute");
    }
    static bool UpdateUI(HLSL::ScreenSpaceAmbientOcclusionAttribs&, FEATURE_FLAGS&) { return false; }

    ITextureView* GetAmbientOcclusionSRV() const
    {
        dfx_plane p{};
        return dfx_ssao_get_plane(m_Fx, DFX_SSAO_PLANE_OUTPUT, &p) == DFX_OK ? m_Out.Update(p) : nullptr;
    }
    // The reference fades the effect in over the first second of wall-clock time (AlphaInterpolation,
    // ScreenSpaceAmbientOcclusion.cpp:793-795), and so does this class. Tests pin it (>= 0); a negative value restores the fade.
    void SetAlphaInterpolation(float Alpha) { dfx_ssao_set_alpha_interpolation(m_Fx, Alpha); }
    dfx_ssao* GetHandle() const { return m_Fx; }

private:
    dfx_ssao*                 m_Fx = nullptr;
    mutable detail::PlaneView m_Out;
};
DEFINE_FLAG_ENUM_OPERATORS(ScreenSpaceAmbientOcclusion::FEATURE_FLAGS)

// =====================================================================================================================
class ScreenSpaceReflection
{
public:
    enum FEATURE_FLAGS : Uint32
    {
        FEATURE_FLAG_NONE            = 0u,
        FEATURE_FLAG_PREVIOUS_FRAME  = 1u << 0u,
        FEATURE_FLAG_HALF_RESOLUTION = 1u << 1u // one ray per 2x2 block, half-size intersect targets
    };
    struct RenderAttributes
    {
        IRenderDevice*                            pDevice            = nullptr;
        IRenderStateCache*                        pStateCache        = nullptr;
        IDeviceContext*                           pDeviceContext     = nullptr;
        PostFXContext*                            pPostFXContext     = nullptr;
        ITextureView*                             pColorBufferSRV    = nullptr; // RGBA32_FLOAT
        ITextureView*                             pDepthBufferSRV    = nullptr; // R32_FLOAT
        ITextureView*                             pNormalBufferSRV   = nullptr; // RGBA32_FLOAT
        ITextureView*                             pMaterialBufferSRV = nullptr; // RGBA32_FLOAT, roughness in pSSRAttribs->RoughnessChannel
        ITextureView*                             pMotionVectorsSRV  = nullptr; // RG32_FLOAT
        const HLSL::ScreenSpaceReflectionAttribs* pSSRAttribs        = nullptr;
    };
    struct CreateInfo
    {
        bool EnableAsyncCreation = false;
    };

    ScreenSpaceReflection(IRenderDevice* pDevice, const CreateInfo& CI)
    {
        (void)pDevice, (void)CI;
        detail::Check(dfx_ssr_create(&m_Fx), "dfx_ssr_create");
        if (m_Fx) dfx_ssr_set_alpha_interpolation(m_Fx, -1.0f); // reference behaviour: fade in over the first second (m_FrameTimer); SetAlphaInterpolation() pins it
    }
    ~ScreenSpaceReflection() { dfx_ssr_destroy(m_Fx); }
    ScreenSpaceReflection(const ScreenSpaceReflection&)            = delete;
    ScreenSpaceReflection& operator=(const ScreenSpaceReflection&) = delete;

    void PrepareResources(IRenderDevice* pDevice, IDeviceContext* pDeviceContext, PostFXContext* pPostFXContext, FEATURE_FLAGS FeatureFlags)
    {
        (void)pDeviceContext;
        DFX_DEV_CHECK_ERR(pDevice != nullptr, "pDevice must not be null");
        DFX_DEV_CHECK_ERR(pPostFXContext != nullptr, "pPostFXContext must not be null");
        if (pPostFXContext) detail::Check(dfx_ssr_prepare(m_Fx, pPostFXContext->GetHandle(), static_cast<uint32_t>(FeatureFlags)), "ScreenSpaceReflection::PrepareResources");
    }
    void Execute(const RenderAttributes& RenderAttribs)
    {
        DFX_DEV_CHECK_ERR(RenderAttribs.pDevice != nullptr, "RenderAttribs.pDevice must not be null");
        DFX_DEV_CHECK_ERR(RenderAttribs.pDeviceContext != nullptr, "RenderAttribs.pDeviceContext must not be null");
        DFX_DEV_CHECK_ERR(RenderAttribs.pPostFXContext != nullptr, "RenderAttribs.pPostFXContext must not be null");
        DFX_DEV_CHECK_ERR(RenderAttribs.pColorBufferSRV != nullptr, "RenderAttribs.pColorBufferSRV must not be null");
        DFX_DEV_CHECK_ERR(RenderAttribs.pDepthBufferSRV != nullptr, "RenderAttribs.pDepthBufferSRV must not be null");
        DFX_DEV_CHECK_ERR(RenderAttribs.pNormalBufferSRV != nullptr, "RenderAttribs.pNormalBufferSRV must not be null");
        DFX_DEV_CHECK_ERR(RenderAttribs.pMaterialBufferSRV != nullptr, "RenderAttribs.pMaterialBufferSRV must not be null");
        DFX_DEV_CHECK_ERR(RenderAttribs.pMotionVectorsSRV != nullptr, "RenderAttribs.pMotionBufferSRV must not be null");
        DFX_DEV_CHECK_ERR(RenderAttribs.pSSRAttribs != nullptr, "RenderAttribs.pSSRAttribs must not be null");
        auto plane = [](ITextureView* v) { return v ? v->GetPlane() : nullptr; };
        dfx_ssr_render_attribs a{};
        a.stream   = detail::StreamOf(RenderAttribs.pDeviceContext);
        a.postfx   = RenderAttribs.pPostFXContext ? RenderAttribs.pPostFXContext->GetHandle() : nullptr;
        a.color    = plane(RenderAttribs.pColorBufferSRV);
        a.depth    = plane(RenderAttribs.pDepthBufferSRV);
        a.normal   = plane(RenderAttribs.pNormalBufferSRV);
        a.material = plane(RenderAttribs.pMaterialBufferSRV);
        a.motion   = plane(RenderAttribs.pMotionVectorsSRV);
        a.attribs  = RenderAttribs.pSSRAttribs;
        detail::Check(dfx_ssr_execute(m_Fx, &a), "ScreenSpaceReflection::Execute");
    }
    static bool UpdateUI(HLSL::ScreenSpaceReflectionAttribs&, FEATURE_FLAGS&, Uint32&) { return false; }

    ITextureView* GetSSRRadianceSRV() const
    {
        dfx_plane p{};
        return dfx_ssr_get_plane(m_Fx, DFX_SSR_PLANE_OUTPUT, &p) == DFX_OK ? m_Out.Update(p) : nullptr;
    }
    void     SetAlphaInterpolation(float Alpha) { dfx_ssr_set_alpha_interpolation(m_Fx, Alpha); }
    dfx_ssr* GetHandle() const { return m_Fx; }

private:
    dfx_ssr*                  m_Fx = nullptr;
    mutable detail::PlaneView m_Out;
};
DEFINE_FLAG_ENUM_OPERATORS(ScreenSpaceReflection::FEATURE_FLAGS)

// =====================================================================================================================
class Bloom
{
public:
    enum FEATURE_FLAGS : Uint32
    {
        FEATURE_FLAG_NONE = 0u
    };
    struct RenderAttributes
    {
        IRenderDevice*            pDevice         = nullptr;
        IRenderStateCache*        pStateCache     = nullptr;
        IDeviceContext*           pDeviceContext  = nullptr;
        PostFXContext*            pPostFXContext  = nullptr;
        ITextureView*             pColorBufferSRV = nullptr; // RGBA32_FLOAT
        const HLSL::BloomAttribs* pBloomAttribs   = nullptr;
    };
    struct CreateInfo
    {
        bool EnableAsyncCreation = false;
    };

    Bloom(IRenderDevice* pDevice, const CreateInfo& CI)
    {
        (void)pDevice, (void)CI;
        detail::Check(dfx_bloom_create(&m_Fx), "dfx_bloom_create");
        if (m_Fx) dfx_bloom_set_alpha_interpolation(m_Fx, -1.0f); // reference behaviour: fade in over the first second (m_FrameTimer); SetAlphaInterpolation() pins it
    }
    ~Bloom() { dfx_bloom_destroy(m_Fx); }
    Bloom(const Bloom&)            = delete;
    Bloom& operator=(const Bloom&) = delete;

    void PrepareResources(IRenderDevice* pDevice, IDeviceContext* pDeviceContext, PostFXContext* pPostFXContext, FEATURE_FLAGS FeatureFlags)
    {
        (void)pDeviceContext;
        DFX_DEV_CHECK_ERR(pDevice != nullptr, "pDevice must not be null");
        DFX_DEV_CHECK_ERR(pPostFXContext != nullptr, "pPostFXContext must not be null");
        if (pPostFXContext) detail::Check(dfx_bloom_prepare(m_Fx, pPostFXContext->GetHandle(), static_cast<uint32_t>(FeatureFlags)), "Bloom::PrepareResources");
    }
    void Execute(const RenderAttributes& RenderAttribs)
    {
        DFX_DEV_CHECK_ERR(RenderAttribs.pDevice != nullptr, "RenderAttribs.pDevice must not be null");
        DFX_DEV_CHECK_ERR(RenderAttribs.pDeviceContext != nullptr, "RenderAttribs.pDeviceContext must not be null");
        DFX_DEV_CHECK_ERR(RenderAttribs.pPostFXContext != nullptr, "RenderAttribs.pPostFXContext must not be null");
        DFX_DEV_CHECK_ERR(RenderAttribs.pColorBufferSRV != nullptr, "RenderAttribs.pColorBufferSRV must not be null");
        DFX_DEV_CHECK_ERR(RenderAttribs.pBloomAttribs != nullptr, "RenderAttribs.pBloomAttribs must not be null");
        dfx_bloom_render_attribs a{};
        a.stream  = detail::StreamOf(RenderAttribs.pDeviceContext);
        a.postfx  = RenderAttribs.pPostFXContext ? RenderAttribs.pPostFXContext->GetHandle() : nullptr;
        a.color   = RenderAttribs.pColorBufferSRV ? RenderAttribs.pColorBufferSRV->GetPlane() : nullptr;
        a.attribs = RenderAttribs.pBloomAttribs;
        detail::Check(dfx_bloom_execute(m_Fx, &a), "Bloom::Execute");
    }
    static bool UpdateUI(HLSL::BloomAttribs&, FEATURE_FLAGS&) { return false; }

    ITextureView* GetBloomTextureSRV() const
    {
        dfx_plane p{};
        return dfx_bloom_get_plane(m_Fx, DFX_BLOOM_PLANE_OUTPUT, &p) == DFX_OK ? m_Out.Update(p) : nullptr;
    }
    void       SetAlphaInterpolation(float Alpha) { dfx_bloom_set_alpha_interpolation(m_Fx, Alpha); }
    dfx_bloom* GetHandle() const { return m_Fx; }

private:
    dfx_bloom*                m_Fx = nullptr;
    mutable detail::PlaneView m_Out;
};

// =====================================================================================================================
// PostProcess/DepthOfField/interface/DepthOfField.hpp:59-125
class DepthOfField
{
public:
    enum FEATURE_FLAGS : Uint32
    {
        FEATURE_FLAG_NONE                      = 0u,
        FEATURE_FLAG_ENABLE_TEMPORAL_SMOOTHING = 1u << 0u,
        FEATURE_FLAG_ENABLE_KARIS_INVERSE      = 1u << 1u
    };
    struct RenderAttributes
    {
        IRenderDevice*                   pDevice         = nullptr;
        IRenderStateCache*               pStateCache     = nullptr;
        IDeviceContext*                  pDeviceContext  = nullptr;
        PostFXContext*                   pPostFXContext  = nullptr;
        ITextureView*                    pColorBufferSRV = nullptr; // RGBA32_FLOAT
        ITextureView*                    pDepthBufferSRV = nullptr; // R32_FLOAT
        const HLSL::DepthOfFieldAttribs* pDOFAttribs     = nullptr;
    };
    struct CreateInfo
    {
        bool EnableAsyncCreation = false;
    };

    DepthOfField(IRenderDevice* pDevice, const CreateInfo& CI)
    {
        (void)pDevice, (void)CI;
        detail::Check(dfx_dof_create(&m_Fx), "dfx_dof_create");
        if (m_Fx) dfx_dof_set_alpha_interpolation(m_Fx, -1.0f); // reference behaviour: fade in over the first second (m_FrameTimer); SetAlphaInterpolation() pins it
    }
    ~DepthOfField() { dfx_dof_destroy(m_Fx); }
    DepthOfField(const DepthOfField&)            = delete;
    DepthOfField& operator=(const DepthOfField&) = delete;

    void PrepareResources(IRenderDevice* pDevice, IDeviceContext* pDeviceContext, PostFXContext* pPostFXContext, FEATURE_FLAGS FeatureFlags)
    {
        (void)pDeviceContext;
        DFX_DEV_CHECK_ERR(pDevice != nullptr, "pDevice must not be null");
        DFX_DEV_CHECK_ERR(pPostFXContext != nullptr, "pPostFXContext must not be null");
        if (pPostFXContext) detail::Check(dfx_dof_prepare(m_Fx, pPostFXContext->GetHandle(), static_cast<uint32_t>(FeatureFlags)), "DepthOfField::PrepareResources");
    }
    void Execute(const RenderAttributes& RenderAttribs)
    {
        DFX_DEV_CHECK_ERR(RenderAttribs.pDevice != nullptr, "RenderAttribs.pDevice must not be null");
        DFX_DEV_CHECK_ERR(RenderAttribs.pDeviceContext != nullptr, "RenderAttribs.pDeviceContext must not be null");
        DFX_DEV_CHECK_ERR(RenderAttribs.pPostFXContext != nullptr, "RenderAttribs.pPostFXContext must not be null");
        DFX_DEV_CHECK_ERR(RenderAttribs.pColorBufferSRV != nullptr, "RenderAttribs.pColorBufferSRV must not be null");
        DFX_DEV_CHECK_ERR(RenderAttribs.pDepthBufferSRV != nullptr, "RenderAttribs.pDepthBufferSRV must not be null");
        DFX_DEV_CHECK_ERR(RenderAttribs.pDOFAttribs != nullptr, "RenderAttribs.pDOFAttribs must not be null");
        dfx_dof_render_attribs a{};
        a.stream  = detail::StreamOf(RenderAttribs.pDeviceContext);
        a.postfx  = RenderAttribs.pPostFXContext ? RenderAttribs.pPostFXContext->GetHandle() : nullptr;
        a.color   = RenderAttribs.pColorBufferSRV ? RenderAttribs.pColorBufferSRV->GetPlane() : nullptr;
        a.depth   = RenderAttribs.pDepthBufferSRV ? RenderAttribs.pDepthBufferSRV->GetPlane() : nullptr;
        a.attribs = RenderAttribs.pDOFAttribs;
        detail::Check(dfx_dof_execute(m_Fx, &a), "DepthOfField::Execute");
    }
    static bool UpdateUI(HLSL::DepthOfFieldAttribs&, FEATURE_FLAGS&) { return false; }

    ITextureView* GetDepthOfFieldTextureSRV() const
    {
        dfx_plane p{};
        return dfx_dof_get_plane(m_Fx, DFX_DOF_PLANE_OUTPUT, &p) == DFX_OK ? m_Out.Update(p) : nullptr;
    }
    void     SetAlphaInterpolation(float Alpha) { dfx_dof_set_alpha_interpolation(m_Fx, Alpha); }
    dfx_dof* GetHandle() const { return m_Fx; }

private:
    dfx_dof*                  m_Fx = nullptr;
    mutable detail::PlaneView m_Out;
};
DEFINE_FLAG_ENUM_OPERATORS(DepthOfField::FEATURE_FLAGS)

// =====================================================================================================================
class TemporalAntiAliasing
{
public:
    enum FEATURE_FLAGS : Uint32
    {
        FEATURE_FLAG_NONE               = 0u,
        FEATURE_FLAG_GAUSSIAN_WEIGHTING = 1u << 0u,
        FEATURE_FLAG_BICUBIC_FILTER     = 1u << 1u,
        FEATURE_FLAG_YCOCG_COLOR_SPACE  = 1u << 2u
    };
    struct RenderAttributes
    {
        IRenderDevice*                           pDevice               = nullptr;
        IRenderStateCache*                       pStateCache           = nullptr;
        IDeviceContext*                          pDeviceContext        = nullptr;
        PostFXContext*                           pPostFXContext        = nullptr;
        ITextureView*                            pColorBufferSRV       = nullptr; // RGBA32_FLOAT, rendered with the jittered projection
        const HLSL::TemporalAntiAliasingAttribs* pTAAAttribs           = nullptr;
        Uint32                                   AccumulationBufferIdx = 0;
    };
    struct CreateInfo
    {
        bool EnableAsyncCreation = false;
    };

    TemporalAntiAliasing(IRenderDevice* pDevice, const CreateInfo& CI)
    {
        (void)pDevice, (void)CI;
        detail::Check(dfx_taa_create(&m_Fx), "dfx_taa_create");
    }
    ~TemporalAntiAliasing() { dfx_taa_destroy(m_Fx); }
    TemporalAntiAliasing(const TemporalAntiAliasing&)            = delete;
    TemporalAntiAliasing& operator=(const TemporalAntiAliasing&) = delete;

    float2 GetJitterOffset(Uint32 AccumulationBufferIdx = 0) const
    {
        float j[2] = {0.0f, 0.0f};
        dfx_taa_get_jitter_offset(m_Fx, AccumulationBufferIdx, j);
        return float2{j[0], j[1]};
    }
    void PrepareResources(IRenderDevice* pDevice, IDeviceContext* pDeviceContext, PostFXContext* pPostFXContext, FEATURE_FLAGS FeatureFlag,
                          Uint32 AccumulationBufferIdx = 0)
    {
        (void)pDeviceContext;
        DFX_DEV_CHECK_ERR(pDevice != nullptr, "pDevice must not be null");
        DFX_DEV_CHECK_ERR(pPostFXContext != nullptr, "pPostFXContext must not be null");
        if (pPostFXContext)
            detail::Check(dfx_taa_prepare(m_Fx, pPostFXContext->GetHandle(), static_cast<uint32_t>(FeatureFlag), AccumulationBufferIdx), "TemporalAntiAliasing::PrepareResources");
    }
    void Execute(const RenderAttributes& RenderAttribs)
    {
        DFX_DEV_CHECK_ERR(RenderAttribs.pDevice != nullptr, "RenderAttribs.pDevice must not be null");
        DFX_DEV_CHECK_ERR(RenderAttribs.pDeviceContext != nullptr, "RenderAttribs.pDeviceContext must not be null");
        DFX_DEV_CHECK_ERR(RenderAttribs.pPostFXContext != nullptr, "RenderAttribs.pPostFXContext must not be null");
        DFX_DEV_CHECK_ERR(RenderAttribs.pColorBufferSRV != nullptr, "RenderAttribs.pColorBufferSRV must not be null");
        DFX_DEV_CHECK_ERR(RenderAttribs.pTAAAttribs != nullptr, "RenderAttribs.pTAAAttribs must not be null");
        dfx_taa_render_attribs a{};
        a.stream                  = detail::StreamOf(RenderAttribs.pDeviceContext);
        a.postfx                  = RenderAttribs.pPostFXContext ? RenderAttribs.pPostFXContext->GetHandle() : nullptr;
        a.color                   = RenderAttribs.pColorBufferSRV ? RenderAttribs.pColorBufferSRV->GetPlane() : nullptr;
        a.attribs                 = RenderAttribs.pTAAAttribs;
        a.accumulation_buffer_idx = RenderAttribs.AccumulationBufferIdx;
        // An unknown accumulation buffer is logged and the call returns, as in TemporalAntiAliasing.cpp:178-183.
        detail::Check(dfx_taa_execute(m_Fx, &a), "TemporalAntiAliasing::Execute");
    }
    static bool UpdateUI(HLSL::TemporalAntiAliasingAttribs&, FEATURE_FLAGS&) { return false; }

    ITextureView* GetAccumulatedFrameSRV(bool IsPrevFrame = false, Uint32 AccumulationBufferIdx = 0) const
    {
        dfx_plane p{};
        if (dfx_taa_get_plane(m_Fx, IsPrevFrame ? DFX_TAA_PLANE_ACCUMULATED_PREV : DFX_TAA_PLANE_ACCUMULATED_CURR, AccumulationBufferIdx, &p) != DFX_OK)
        {
            DFX_LOG_ERROR_MESSAGE("Accumulation buffer with index %u is not found.", AccumulationBufferIdx);
            return nullptr;
        }
        return m_Out[IsPrevFrame ? 1 : 0].Update(p);
    }
    // TemporalAntiAliasing.hpp:138-156
    static inline float4x4 GetJitteredProjMatrix(float4x4 Proj, const float2& Jitter)
    {
        if (Proj.m33 == 0.f)
        {
            Proj.m20 += Jitter.x; // perspective: proportional to z, constant in screen space
            Proj.m21 += Jitter.y;
        }
        else
        {
            Proj.m30 += Jitter.x; // orthographic
            Proj.m31 += Jitter.y;
        }
        return Proj;
    }
    dfx_taa* GetHandle() const { return m_Fx; }

private:
    dfx_taa*                  m_Fx = nullptr;
    mutable detail::PlaneView m_Out[2];
};
DEFINE_FLAG_ENUM_OPERATORS(TemporalAntiAliasing::FEATURE_FLAGS)

// =====================================================================================================================
// ToneMap(): in the reference this is an HLSL function callers splice into their own final-blit shader
// (Hydrogent/shaders/HnCopyFrame.psh:32-62). Here it is one full-screen pass: Dst = [LinearToSRGB](ToneMap(Src, Attribs, fAveLogLum)).
inline void ToneMap(IDeviceContext* pDeviceContext, ITextureView* pSrcColorSRV, ITextureView* pDstColorRTV, const HLSL::ToneMappingAttribs& Attribs,
                    float fAveLogLum, bool ConvertOutputToSRGB)
{
    DFX_DEV_CHECK_ERR(pSrcColorSRV != nullptr && pDstColorRTV != nullptr, "source and destination views must not be null");
    if (!pSrcColorSRV || !pDstColorRTV) return;
    const dfx_plane* src = pSrcColorSRV->GetPlane();
    detail::Check(dfx_pass_tonemap(detail::StreamOf(pDeviceContext), &Attribs, fAveLogLum, ConvertOutputToSRGB ? 1 : 0, src, pDstColorRTV->GetPlane(),
                                   dfx_rows{0, src ? src->height : 0}),
                  "ToneMap");
}

// ToneMap() with fAveLogLum = max(0.05, *pAveLogLumDev) read on the device (GetAverageSceneLuminance, AtmosphereShadersCommon.fxh:188-197):
// pass AverageLuminance::GetStateDev() below, or any device float the caller keeps.
inline void ToneMap(IDeviceContext* pDeviceContext, ITextureView* pSrcColorSRV, ITextureView* pDstColorRTV, const HLSL::ToneMappingAttribs& Attribs,
                    const float* pAveLogLumDev, bool ConvertOutputToSRGB)
{
    DFX_DEV_CHECK_ERR(pSrcColorSRV != nullptr && pDstColorRTV != nullptr && pAveLogLumDev != nullptr, "views and luminance must not be null");
    if (!pSrcColorSRV || !pDstColorRTV || !pAveLogLumDev) return;
    const dfx_plane* src = pSrcColorSRV->GetPlane();
    detail::Check(dfx_pass_tonemap_dev(detail::StreamOf(pDeviceContext), &Attribs, pAveLogLumDev, ConvertOutputToSRGB ? 1 : 0, src, pDstColorRTV->GetPlane(),
                                       dfx_rows{0, src ? src->height : 0}),
                  "ToneMap");
}

// Auto exposure with light adaptation, the part of EpipolarLightScattering that ToneMappingAttribs::bAutoExposure / bLightAdaptation
// switch on (EpipolarLightScattering.cpp:2463-2481, UpdateAverageLuminance.fx): owns the persistent average-luminance state (the 1x1
// R16F target of the reference, cleared to 0.1) and updates it from a colour view once per frame. Update() measures when
// Attribs.bAutoExposure is set and adapts over dElapsedTime (FrameAttribs.dElapsedTime) when Attribs.bLightAdaptation is set.
class AverageLuminance
{
public:
    enum SAMPLING : int32_t
    {
        SAMPLING_REFERENCE = DFX_LUMINANCE_SAMPLING_REFERENCE, // 64x64 point samples, half-rounded mip chain: the reference's numbers
        SAMPLING_FULL      = DFX_LUMINANCE_SAMPLING_FULL       // every pixel (a small highlight cannot be missed)
    };
    explicit AverageLuminance(SAMPLING Sampling = SAMPLING_FULL) : m_Sampling(Sampling)
    {
        if (detail::Check(dfx_plane_alloc(DFX_AVERAGE_LUMINANCE_STATE_FLOATS, 1, DFX_FORMAT_R32F, &m_State), "AverageLuminance"))
            Reset(nullptr);
    }
    ~AverageLuminance() { dfx_plane_free(&m_State); }
    AverageLuminance(const AverageLuminance&)            = delete;
    AverageLuminance& operator=(const AverageLuminance&) = delete;

    void Reset(IDeviceContext* pDeviceContext)
    {
        detail::Check(dfx_pass_reset_average_luminance(detail::StreamOf(pDeviceContext), GetStateDev()), "AverageLuminance::Reset");
    }
    void Update(IDeviceContext* pDeviceContext, ITextureView* pColorSRV, const HLSL::ToneMappingAttribs& Attribs, double dElapsedTime)
    {
        DFX_DEV_CHECK_ERR(pColorSRV != nullptr, "pColorSRV must not be null");
        if (!pColorSRV || !Attribs.bAutoExposure) return;
        detail::Check(dfx_pass_update_average_luminance(detail::StreamOf(pDeviceContext), &Attribs, m_Sampling, static_cast<float>(dElapsedTime),
                                                        pColorSRV->GetPlane(), GetStateDev()),
                      "AverageLuminance::Update");
    }
    float* GetStateDev() const { return static_cast<float*>(m_State.ptr); }

private:
    SAMPLING  m_Sampling;
    dfx_plane m_State{};
};

// ToneMap() with the adapted luminance of `Lum` when Attribs.bAutoExposure is set, with fAveLogLum otherwise.
inline void ToneMap(IDeviceContext* pDeviceContext, ITextureView* pSrcColorSRV, ITextureView* pDstColorRTV, const HLSL::ToneMappingAttribs& Attribs,
                    const AverageLuminance& Lum, float fAveLogLum, bool ConvertOutputToSRGB)
{
    if (Attribs.bAutoExposure)
        ToneMap(pDeviceContext, pSrcColorSRV, pDstColorRTV, Attribs, static_cast<const float*>(Lum.GetStateDev()), ConvertOutputToSRGB);
    else
        ToneMap(pDeviceContext, pSrcColorSRV, pDstColorRTV, Attribs, fAveLogLum, ConvertOutputToSRGB);
}

// The compose step that sits between SSAO and TAA in the reference integration (reduced form, SURVEY.md §8f rank 1).
inline void ComposeSSRAndSSAO(IDeviceContext* pDeviceContext, ITextureView* pColorSRV, ITextureView* pSSRRadianceSRV, ITextureView* pAmbientOcclusionSRV,
                              float SSRScale, float SSAOScale, ITextureView* pDstColorRTV)
{
    if (!pColorSRV || !pDstColorRTV) return;
    detail::Check(dfx_pass_compose(detail::StreamOf(pDeviceContext), pColorSRV->GetPlane(), pSSRRadianceSRV ? pSSRRadianceSRV->GetPlane() : nullptr,
                                   pAmbientOcclusionSRV ? pAmbientOcclusionSRV->GetPlane() : nullptr, SSRScale, SSAOScale, pDstColorRTV->GetPlane(),
                                   dfx_rows{0, pColorSRV->GetPlane()->height}),
                  "ComposeSSRAndSSAO");
}

} // namespace Diligent

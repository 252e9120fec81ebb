/* dfx_b200.h — C-ABI of the B200-native DiligentFX PostProcess chain.
 *
 * This is the drop-in boundary (SURVEY.md §8b): every entry point is `extern "C"`, takes plain pointers /
 * sizes / POD structs, never throws and returns a dfx_status. It replaces, for the PostProcess hot path only,
 * what the reference records through DiligentCore's IDeviceContext inside
 *   PostFXContext::Execute                 (PostProcess/Common/src/PostFXContext.cpp:287-338)
 *   ScreenSpaceAmbientOcclusion::Execute   (PostProcess/ScreenSpaceAmbientOcclusion/src/ScreenSpaceAmbientOcclusion.cpp:348-387)
 *   ScreenSpaceReflection::Execute         (PostProcess/ScreenSpaceReflection/src/ScreenSpaceReflection.cpp:300-341)
 *   Bloom::Execute                         (PostProcess/Bloom/src/Bloom.cpp:407-436)
 *   TemporalAntiAliasing::Execute          (PostProcess/TemporalAntiAliasing/src/TemporalAntiAliasing.cpp:169-201)
 *   ToneMap()                              (Shaders/PostProcess/ToneMapping/public/ToneMapping.fxh:87-226)
 *
 * Two layers:
 *   1. pass level   `dfx_pass_*`  — one stateless call per reference render pass (or fused pass group); every
 *                                   plane is passed explicitly. This is what the parity tests drive.
 *   2. effect level `dfx_<effect>_{create,prepare,execute,get_plane,destroy}` — owns the effect's internal
 *                                   planes (history ping-pong, pyramids) exactly like the reference classes own
 *                                   their textures; the C++ headers under include/dfx/ wrap these in C++ classes with the
 *                                   reference's own signatures.
 *
 * All device pointers are CUDA device pointers on the current device; `stream` is a cudaStream_t passed as void*.
 * There is no CPU fallback: every entry fails with DFX_ERR_CUDA when no sm_100 device/driver is usable.
 */
#ifndef DFX_B200_H
#define DFX_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DFX_API __attribute__((visibility("default")))

/* ------------------------------------------------------------------------------------------------------------ */
/* status                                                                                                       */
typedef enum dfx_status
{
    DFX_OK               = 0,
    DFX_ERR_INVALID_ARG  = 1, /* null pointer, bad format, mismatched size (reference: DEV_CHECK_ERR)        */
    DFX_ERR_CUDA         = 2, /* a CUDA runtime call or launch failed; see dfx_last_error()                   */
    DFX_ERR_NOT_PREPARED = 3, /* execute before prepare (reference: TemporalAntiAliasing.cpp:178-183)         */
    DFX_ERR_UNSUPPORTED  = 4  /* unknown feature-flag bits, or a combination this build has no kernel for   */
} dfx_status;

DFX_API const char* dfx_last_error(void);           /* thread-local message of the last non-OK status      */
DFX_API int         dfx_version(void);              /* 10000*major + 100*minor + patch                     */
DFX_API uint64_t    dfx_launch_count(void);         /* kernels launched by this library so far (process)   */

/* ------------------------------------------------------------------------------------------------------------ */
/* planes                                                                                                       */
typedef enum dfx_format
{
    DFX_FORMAT_UNKNOWN = 0,
    DFX_FORMAT_R32F    = 1, /* depth, AO, history length, variance, roughness …            4 B/texel */
    DFX_FORMAT_RG32F   = 2, /* motion vectors, blue noise                                  8 B/texel */
    DFX_FORMAT_RGBA32F = 3, /* colour, normal (xyz_), material, radiance, bloom levels    16 B/texel */
    DFX_FORMAT_R8U     = 4, /* SSR reflection mask (stands in for the D16 stencil mask)    1 B/texel */
    /* transfer formats (dfx_pass_unpack_plane / dfx_pass_pack_ldr8 only; the passes compute on the fp32 formats above) */
    DFX_FORMAT_RGBA16F = 5, /* scene colour, normal as the G-buffer stores them             8 B/texel */
    DFX_FORMAT_RG16F   = 6, /* motion vectors                                               4 B/texel */
    DFX_FORMAT_RG8U    = 7, /* material (roughness, metallic) UNORM                         2 B/texel */
    DFX_FORMAT_RGBA8U  = 8  /* tone-mapped sRGB frame as a swap chain stores it             4 B/texel */
} dfx_format;

/* A pitched 2-D array in HBM: row y starts at (char*)ptr + y*pitch_bytes. Stands in for ITextureView. */
typedef struct dfx_plane
{
    void*    ptr;
    size_t   pitch_bytes;
    int32_t  width;
    int32_t  height;
    int32_t  format; /* dfx_format */
    int32_t  flags;  /* DFX_PLANE_FLAG_*; 0 for every plane but a reversed depth buffer */
} dfx_plane;
/* A DEPTH plane (or level 0 of a depth pyramid) that stores reversed depth: near = 1, far = 0. Stands in for
 * PostFXContext::FEATURE_FLAG_REVERSED_DEPTH (PostFXContext.hpp:54) at the pass level, where the reference compiles the
 * POSTFX/SSAO/SSR_OPTION_INVERTED_DEPTH shader variants (ComputeClosestMotion.fx:5-9,36-40; SSAO_Common.fxh:6-23;
 * SSR_Common.fxh:6-12,48-55; SSR_ComputeIntersection.fx:109-124): the passes that read the plane take the closest depth
 * as the maximum, the far plane as 0 and the background test as depth < 1e-6. The effect-level objects set it themselves
 * from the PostFX feature flag.                                                                                  */
#define DFX_PLANE_FLAG_REVERSED_DEPTH 1
/* A depth plane (level 0 of the SSAO prefiltered-depth pyramid) that the reference would keep in R16_UNORM
 * (ScreenSpaceAmbientOcclusion::FEATURE_FLAG_HALF_PRECISION_DEPTH, …cpp:96-97). The plane stays fp32 here — this library
 * models none of the reference's narrow storage formats — but the AO pass uses the larger self-occlusion offset the
 * reference compiles in for that mode (0.005 instead of 0.00001, SSAO_ComputeAmbientOcclusion.fx:145-150).          */
#define DFX_PLANE_FLAG_HALF_PRECISION_DEPTH 2

#define DFX_MAX_MIPS 8
/* A mip chain of planes (level i is max(w>>i,1) x max(h>>i,1)). Stands in for a mip-mapped ITexture. */
typedef struct dfx_pyramid
{
    dfx_plane level[DFX_MAX_MIPS];
    int32_t   levels;
    int32_t   reserved;
} dfx_pyramid;

/* Row range [y0, y1) of the full frame that a call computes. {0, height} = whole frame. Used by the row-strip
 * multi-GPU path (SURVEY.md §8e): every GPU holds full-size planes and computes only its strip; halo rows are
 * exchanged between calls. For pyramid passes y0/y1 must be multiples of 64 (or y1 == height).               */
typedef struct dfx_rows
{
    int32_t y0;
    int32_t y1;
} dfx_rows;

/* ------------------------------------------------------------------------------------------------------------ */
/* constant blocks — byte-identical to the reference's shared C++/HLSL structs                                  */

typedef struct dfx_float4x4 { float m[4][4]; } dfx_float4x4; /* row-major, row-vector convention mul(v, M) */

/* == HLSL::CameraAttribs, Shaders/Common/public/BasicStructures.fxh:84-149 (576 bytes) */
typedef struct dfx_camera_attribs
{
    float f4Position[4];
    float f4ViewportSize[4]; /* (width, height, 1/width, 1/height) */
    float fNearPlaneZ, fFarPlaneZ, fNearPlaneDepth, fFarPlaneDepth;
    float fSceneNearZ, fSceneFarZ, fSceneNearDepth, fSceneFarDepth;
    float    fHandness;
    uint32_t uiFrameIndex;
    float    Padding0, Padding1;
    float fFocusDistance, fFStop, fFocalLength, fSensorWidth;
    float fSensorHeight, fExposure;
    float f2Jitter[2];
    dfx_float4x4 mView, mProj, mViewProj, mViewInv, mProjInv, mViewProjInv;
    float f4ExtraData[5][4];
} dfx_camera_attribs;

/* == HLSL::ScreenSpaceAmbientOcclusionAttribs, …/ScreenSpaceAmbientOcclusionStructures.fxh:64-98 (48 bytes) */
typedef struct dfx_ssao_attribs
{
    float    EffectRadius;                /* 1.0   */
    float    EffectFalloffRange;          /* 0.615 */
    float    RadiusMultiplier;            /* 1.457 */
    float    DepthMIPSamplingOffset;      /* 3.3   */
    float    TemporalStabilityFactor;     /* 0.9   */
    float    SpatialReconstructionRadius; /* 4.0   */
    int32_t  ResetAccumulation;           /* FALSE */
    float    AlphaInterpolation;          /* 1.0   */
    float    BitmaskThickness;            /* 0.5   */
    uint32_t Algorithm;                   /* DFX_SSAO_ALGORITHM_GTAO */
    float    Padding0, Padding1;
} dfx_ssao_attribs;
#define DFX_SSAO_ALGORITHM_GTAO 0
#define DFX_SSAO_ALGORITHM_HBAO 1
#define DFX_SSAO_ALGORITHM_VBAO 2

/* == HLSL::ScreenSpaceReflectionAttribs, …/ScreenSpaceReflectionStructures.fxh:43-80 (48 bytes) */
typedef struct dfx_ssr_attribs
{
    float    DepthBufferThickness;               /* 0.025 */
    float    RoughnessThreshold;                 /* 0.2   */
    uint32_t MostDetailedMip;                    /* 0     */
    int32_t  IsRoughnessPerceptual;              /* TRUE  */
    uint32_t RoughnessChannel;                   /* 0     */
    uint32_t MaxTraversalIntersections;          /* 128   */
    float    GGXImportanceSampleBias;            /* 0.3   */
    float    SpatialReconstructionRadius;        /* 4.0   */
    float    TemporalRadianceStabilityFactor;    /* 1.0   */
    float    TemporalVarianceStabilityFactor;    /* 0.9   */
    float    BilateralCleanupSpatialSigmaFactor; /* 0.9   */
    float    AlphaInterpolation;                 /* 1.0   */
} dfx_ssr_attribs;

/* == HLSL::BloomAttribs, …/BloomStructures.fxh:12-34 (32 bytes) */
typedef struct dfx_bloom_attribs
{
    float Intensity;          /* 0.15  */
    float Threshold;          /* 1.0   */
    float SoftTreshold;       /* 0.125 */
    float Radius;             /* 0.75  */
    float AlphaInterpolation; /* 1.0   */
    float Padding0, Padding1, Padding2;
} dfx_bloom_attribs;

/* == HLSL::TemporalAntiAliasingAttribs, …/TemporalAntiAliasingStructures.fxh:35-46 (16 bytes) */
typedef struct dfx_taa_attribs
{
    float   TemporalStabilityFactor; /* 0.9375 */
    int32_t ResetAccumulation;       /* FALSE  */
    int32_t SkipRejection;           /* FALSE  */
    float   Padding0;
} dfx_taa_attribs;

/* == HLSL::DepthOfFieldAttribs, Shaders/PostProcess/DepthOfField/public/DepthOfFieldStructures.fxh:31-56 (32 bytes) */
typedef struct dfx_dof_attribs
{
    float   MaxCircleOfConfusion;    /* 0.01   : largest CoC in texture coordinates                    */
    float   TemporalStabilityFactor; /* 0.9375                                                         */
    int32_t BokehKernelRingCount;    /* 5      : rings of the Octaweb kernel (2..5)                    */
    int32_t BokehKernelRingDensity;  /* 7      : samples per ring step (2..7)                          */
    float   AlphaInterpolation;      /* 1.0                                                            */
    float   Padding0, Padding1, Padding2;
} dfx_dof_attribs;
#define DFX_DOF_FEATURE_FLAG_NONE                      0u
#define DFX_DOF_FEATURE_FLAG_ENABLE_TEMPORAL_SMOOTHING (1u << 0) /* D2 (DepthOfField.hpp:65) */
#define DFX_DOF_FEATURE_FLAG_ENABLE_KARIS_INVERSE      (1u << 1) /* HDR-weighted gather in D8 (:67) */

/* == HLSL::ToneMappingAttribs (+AgXAttribs), …/ToneMappingStructures.fxh:24-52 (48 bytes) */
typedef struct dfx_tonemap_attribs
{
    int32_t  iToneMappingMode;     /* DFX_TONE_MAPPING_MODE_UNCHARTED2 */
    int32_t  bAutoExposure;        /* TRUE  */
    float    fMiddleGray;          /* 0.18  */
    int32_t  bLightAdaptation;     /* TRUE  */
    float    fWhitePoint;          /* 3.0   */
    float    fLuminanceSaturation; /* 1.0   */
    uint32_t Padding0, Padding1;
    float    AgXSaturation, AgXSlope, AgXPower, AgXOffset; /* 1,1,1,0 */
} dfx_tonemap_attribs;
#define DFX_TONE_MAPPING_MODE_NONE          0
#define DFX_TONE_MAPPING_MODE_EXP           1
#define DFX_TONE_MAPPING_MODE_REINHARD      2
#define DFX_TONE_MAPPING_MODE_REINHARD_MOD  3
#define DFX_TONE_MAPPING_MODE_UNCHARTED2    4
#define DFX_TONE_MAPPING_MODE_FILMIC_ALU    5
#define DFX_TONE_MAPPING_MODE_LOGARITHMIC   6
#define DFX_TONE_MAPPING_MODE_ADAPTIVE_LOG  7
#define DFX_TONE_MAPPING_MODE_AGX           8
#define DFX_TONE_MAPPING_MODE_AGX_CUSTOM    9
#define DFX_TONE_MAPPING_MODE_PBR_NEUTRAL  10
#define DFX_TONE_MAPPING_MODE_COMMERCE     11

/* Default-initialisers (the reference's DEFAULT_VALUE()s). */
DFX_API void dfx_ssao_attribs_default(dfx_ssao_attribs* a);
DFX_API void dfx_ssr_attribs_default(dfx_ssr_attribs* a);
DFX_API void dfx_bloom_attribs_default(dfx_bloom_attribs* a);
DFX_API void dfx_dof_attribs_default(dfx_dof_attribs* a);
DFX_API void dfx_taa_attribs_default(dfx_taa_attribs* a);
DFX_API void dfx_tonemap_attribs_default(dfx_tonemap_attribs* a);

/* == PostFXContext::FrameDesc, PostProcess/Common/interface/PostFXContext.hpp:68-84 */
typedef struct dfx_frame_desc
{
    uint32_t Index;
    uint32_t Width;
    uint32_t Height;
    uint32_t OutputWidth;
    uint32_t OutputHeight;
} dfx_frame_desc;

/* feature flags: numeric values of the reference enums */
#define DFX_POSTFX_FEATURE_FLAG_NONE                 0u
#define DFX_POSTFX_FEATURE_FLAG_REVERSED_DEPTH       (1u << 0) /* depth: near = 1, far = 0 (see DFX_PLANE_FLAG_REVERSED_DEPTH) */
#define DFX_POSTFX_FEATURE_FLAG_HALF_PRECISION_DEPTH (1u << 1) /* accepted; selects a storage format only, planes stay fp32 */
#define DFX_POSTFX_FEATURE_FLAG_TEMPORAL_UPSCALING   (1u << 2) /* Bloom runs at FrameDesc.OutputWidth x OutputHeight (Bloom.cpp:84-85) */
#define DFX_SSAO_FEATURE_FLAG_NONE                   0u
#define DFX_SSAO_FEATURE_FLAG_HALF_PRECISION_DEPTH   (1u << 0) /* AO self-occlusion offset 0.005; planes stay fp32 */
#define DFX_SSAO_FEATURE_FLAG_HALF_RESOLUTION        (1u << 1) /* A0 + A1-A3 at width/2 x height/2 + A4 */
#define DFX_SSR_FEATURE_FLAG_NONE                    0u
#define DFX_SSR_FEATURE_FLAG_PREVIOUS_FRAME          (1u << 0)
#define DFX_SSR_FEATURE_FLAG_HALF_RESOLUTION         (1u << 1) /* S3 + S4 at width/2 x height/2 */
#define DFX_BLOOM_FEATURE_FLAG_NONE                  0u
#define DFX_TAA_FEATURE_FLAG_NONE                    0u
#define DFX_TAA_FEATURE_FLAG_GAUSSIAN_WEIGHTING      (1u << 0)
#define DFX_TAA_FEATURE_FLAG_BICUBIC_FILTER          (1u << 1)
#define DFX_TAA_FEATURE_FLAG_YCOCG_COLOR_SPACE       (1u << 2)

/* ============================================================================================================ */
/* 1. pass level                                                                                                */
/* ============================================================================================================ */

/* P0 ComputeBlueNoiseTexture (PostFXContext.cpp:567-609; Shaders/Common/private/ComputeBlueNoiseTexture.fx:81-89).
 * tables: device pointer to the 131,328-byte blob (Sobol_256d[256] ++ ScramblingTile[128*128*8]).
 * xy, zw: 128x128 RG32F.                                                                                       */
DFX_API dfx_status dfx_pass_blue_noise(void* stream, const uint8_t* tables, uint32_t frame_index,
                                       const dfx_plane* xy, const dfx_plane* zw);

/* P1+P2+P3 fused: ComputeReprojectedDepth (ComputeReprojectedDepth.fx:18-30), ComputeClosestMotion
 * (ComputeClosestMotion.fx:24-55), ComputePreviousDepth (PostFXContext.cpp:657-676).
 * cameras: device pointer to dfx_camera_attribs[2] = {curr, prev}.                                             */
DFX_API dfx_status dfx_pass_postfx_prepare(void* stream, const dfx_camera_attribs* cameras_dev,
                                           const dfx_plane* curr_depth, const dfx_plane* prev_depth_in,
                                           const dfx_plane* motion,
                                           const dfx_plane* reprojected_depth, const dfx_plane* closest_motion,
                                           const dfx_plane* previous_depth, dfx_rows rows);

/* A1+A2 ComputePrefilteredDepth (ScreenSpaceAmbientOcclusion.cpp:843-957; SSAO_ComputePrefilteredDepthBuffer.fx:79-122).
 * pyr->level[0] aliases the input depth (the reference's CopyTextureDepth into mip 0 is elided); levels 1..4 written. */
DFX_API dfx_status dfx_pass_ssao_prefilter_depth(void* stream, const dfx_camera_attribs* cameras_dev,
                                                 const dfx_ssao_attribs* attribs, const dfx_pyramid* pyr, dfx_rows rows);

/* FEATURE_FLAG_HALF_RESOLUTION (ScreenSpaceAmbientOcclusion.hpp:59-82): A0 builds a width/2 x height/2 checkerboard of the 2x2
 * min / max depth, A1-A3 run on it (the prefiltered pyramid, hence the occlusion target, is half size: A3 recognises the
 * mode by a pyramid of half the normal plane's size and doubles GetInvViewportSize(), SSAO_ComputeAmbientOcclusion.fx:68-75),
 * and A4 brings the occlusion back to full resolution for A5-A8.
 * A0 ComputeDepthCheckerboard (…cpp:818-841; SSAO_ComputeDownsampledDepth.fx:8-29). `rows`: rows of the half-size plane. */
DFX_API dfx_status dfx_pass_ssao_downsample_depth(void* stream, const dfx_plane* depth, const dfx_plane* out_half, dfx_rows rows);
/* A4 ComputeBilateralUpsampling (…cpp:992-1020; SSAO_ComputeBilateralUpsampling.fx:62-139): 3x3 joint-bilateral filter of
 * the half-size occlusion guided by the full-resolution depth; background pixels get 1.0.                        */
DFX_API dfx_status dfx_pass_ssao_upsample(void* stream, const dfx_camera_attribs* cameras_dev, const dfx_plane* depth,
                                          const dfx_plane* occlusion_half, const dfx_plane* out_occlusion, dfx_rows rows);

/* A3 ComputeAmbientOcclusion (…cpp:961-990; SSAO_ComputeAmbientOcclusion.fx:132-231). Includes the clear to 1.0. */
DFX_API dfx_status dfx_pass_ssao_ambient_occlusion(void* stream, const dfx_camera_attribs* cameras_dev,
                                                   const dfx_ssao_attribs* attribs, const dfx_pyramid* prefiltered_depth,
                                                   const dfx_plane* normal, const dfx_plane* blue_noise_zw,
                                                   const dfx_plane* occlusion, dfx_rows rows);

/* A5 ComputeTemporalAccumulation (…cpp:1032-1073; SSAO_ComputeTemporalAccumulation.fx:151-182). Includes the
 * clears of both targets to 1.0 (background pixels keep 1.0).                                                  */
DFX_API dfx_status dfx_pass_ssao_temporal(void* stream, const dfx_camera_attribs* cameras_dev,
                                          const dfx_ssao_attribs* attribs,
                                          const dfx_plane* curr_occlusion, const dfx_plane* prev_occlusion,
                                          const dfx_plane* prev_history_length, const dfx_plane* reprojected_depth,
                                          const dfx_plane* previous_depth, const dfx_plane* closest_motion,
                                          const dfx_plane* out_occlusion, const dfx_plane* out_history_length,
                                          dfx_rows rows);

/* A6 ComputeConvolutedDepthHistory (…cpp:1075-1255; SSAO_ComputeConvolutedDepthHistory.fx:93-109).
 * level[0] of both pyramids are inputs (accumulated AO, depth); levels 1..4 written.                           */
DFX_API dfx_status dfx_pass_ssao_convolute(void* stream, const dfx_pyramid* occlusion_pyr, const dfx_pyramid* depth_pyr,
                                           dfx_rows rows);

/* A7 ComputeResampledHistory (…cpp:1257-1286; SSAO_ComputeResampledHistory.fx:56-115). */
DFX_API dfx_status dfx_pass_ssao_resample(void* stream, const dfx_camera_attribs* cameras_dev,
                                          const dfx_pyramid* occlusion_pyr, const dfx_pyramid* depth_pyr,
                                          const dfx_plane* history_length, const dfx_plane* normal,
                                          const dfx_plane* out_occlusion, dfx_rows rows);

/* A8 ComputeSpatialReconstruction (…cpp:1288-1329; SSAO_ComputeSpatialReconstruction.fx:49-100). The reference's
 * CopyTexture(resolved -> history[curr]) is elided: `out_occlusion` IS history[curr].                          */
DFX_API dfx_status dfx_pass_ssao_spatial(void* stream, const dfx_camera_attribs* cameras_dev,
                                         const dfx_ssao_attribs* attribs,
                                         const dfx_plane* occlusion, const dfx_plane* history_length,
                                         const dfx_plane* depth, const dfx_plane* normal,
                                         const dfx_plane* out_occlusion, dfx_rows rows);

/* S1 ComputeHierarchicalDepthBuffer (ScreenSpaceReflection.cpp:777-902; SSR_ComputeHierarchicalDepthBuffer.fx:30-73).
 * level[0] aliases the input depth; levels 1..6 written.                                                       */
DFX_API dfx_status dfx_pass_ssr_hiz(void* stream, const dfx_pyramid* pyr, dfx_rows rows);

/* S2 ComputeStencilMaskAndExtractRoughness (…cpp:904-932; SSR_ComputeStencilMaskAndExtractRoughness.fx:13-40).
 * mask (R8U): 1 where the pixel is a reflection sample, 0 elsewhere; roughness written only where mask==1.     */
DFX_API dfx_status dfx_pass_ssr_mask_roughness(void* stream, const dfx_ssr_attribs* attribs,
                                               const dfx_plane* material, const dfx_plane* depth,
                                               const dfx_plane* roughness, const dfx_plane* mask, dfx_rows rows);

/* FEATURE_FLAG_HALF_RESOLUTION (ScreenSpaceReflection.hpp:64-76): S3 downsamples the mask, S4 traces one ray per 2x2 block
 * into width/2 x height/2 targets (which of the four pixels: a 4x4 pattern, PostFX_Common.fxh:45-55), S5 gathers from the
 * half-size targets; S6 / S7 are unchanged. S4 and S5 recognise the mode by intersect planes of half the frame size.
 * S3 ComputeDownsampledStencilMask (…cpp:934-961; SSR_ComputeDownsampledStencilMask.fx:13-61): 1 where the closest depth
 * and the largest roughness of the 2x2 (+ odd row / column) footprint pass IsReflectionSample. `rows`: of the half-size mask. */
DFX_API dfx_status dfx_pass_ssr_downsample_mask(void* stream, const dfx_ssr_attribs* attribs, const dfx_plane* roughness,
                                                const dfx_plane* depth, const dfx_plane* mask_half, dfx_rows rows);

/* S4 ComputeIntersection (…cpp:963-999; SSR_ComputeIntersection.fx:281-325). Includes both clears to 0.
 * motion may be NULL unless DFX_SSR_FEATURE_FLAG_PREVIOUS_FRAME is set in `flags`.                             */
DFX_API dfx_status dfx_pass_ssr_intersect(void* stream, const dfx_camera_attribs* cameras_dev,
                                          const dfx_ssr_attribs* attribs, uint32_t flags,
                                          const dfx_plane* color, const dfx_plane* normal, const dfx_plane* roughness,
                                          const dfx_plane* mask, const dfx_plane* blue_noise_xy,
                                          const dfx_pyramid* hiz, const dfx_plane* motion,
                                          const dfx_plane* out_radiance, const dfx_plane* out_raydir_pdf, dfx_rows rows);

/* S4 for one frame split into row strips over several GPUs of an NVLink / NVSwitch box (SURVEY.md §8e). The march of a ray may
 * cross the whole screen. The Hi-Z pyramid `hiz` (depth included) must be COMPLETE on this GPU - the march walks it in a dependent
 * chain of ~36 loads per ray, which must not cross the link (measured; the strips executor all-gathers it by peer stores) - while
 * the colour and the normal at the hit, two independent loads per ray, are loaded straight from the GPU that OWNS the row (peer
 * loads; every GPU holds full-size RGBA32F planes at the same pitch, valid on its own rows only). `color`, `normal` describe the
 * local planes; `peers` gives, per rank, the base pointer of the same plane as mapped into this process (cudaIpcOpenMemHandle, or a
 * plain pointer when one process drives all GPUs; base[own rank] = the local pointer; the `hiz` entries are not used).
 * row_begin[r] .. row_begin[r+1] are the rows rank r owns; every boundary but the last is a multiple of 64. Output is bit-identical
 * to dfx_pass_ssr_intersect on complete planes. DFX_SSR_FEATURE_FLAG_PREVIOUS_FRAME is not supported. The caller orders the
 * producers on all GPUs before this launch (stream-ordered barrier) and this launch before the next frame's writers. No reference
 * counterpart: the reference renders a frame on one device.                                                        */
#define DFX_MAX_PEERS 8
typedef struct dfx_peer_set {
    int32_t     count;                                  /* GPUs sharing the frame, 1..DFX_MAX_PEERS                    */
    int32_t     row_begin[DFX_MAX_PEERS + 1];
    const void* color[DFX_MAX_PEERS];
    const void* normal[DFX_MAX_PEERS];
    const void* hiz[DFX_MAX_MIPS][DFX_MAX_PEERS];       /* level 0 = the depth plane                                   */
} dfx_peer_set;
/* The same frame-sharding description in the form the strips executor (section 4) uses: every rank holds ALL planes at the same
 * offsets of an identically laid-out slab; base[r] is rank r's slab as mapped into this process (dfx_ipc_open), so the copy of any
 * plane on rank r is at (plane pointer - base[rank] + base[r]). Rows are owned in 64-row blocks: rank r owns [row_begin[r], row_begin[r+1]). */
typedef struct dfx_peer_map {
    int32_t     count, rank;
    int32_t     row_begin[DFX_MAX_PEERS + 1];
    const void* base[DFX_MAX_PEERS];
} dfx_peer_map;
DFX_API dfx_status dfx_pass_ssr_intersect_peer(void* stream, const dfx_camera_attribs* cameras_dev,
                                               const dfx_ssr_attribs* attribs, uint32_t flags, const dfx_peer_set* peers,
                                               const dfx_plane* color, const dfx_plane* normal, const dfx_plane* roughness,
                                               const dfx_plane* mask, const dfx_plane* blue_noise_xy, const dfx_pyramid* hiz,
                                               const dfx_plane* out_radiance, const dfx_plane* out_raydir_pdf, dfx_rows rows);
/* cudaDeviceEnablePeerAccess(peer_device) for the current device; OK if already enabled, DFX_ERR_UNSUPPORTED if the
 * two devices have no peer path.                                                                                   */
DFX_API dfx_status dfx_enable_peer_access(int32_t peer_device);
/* Device memory another process on the same box can map (one process per GPU): dfx_ipc_alloc = cudaMalloc +
 * cudaIpcGetMemHandle on the current device; the 64-byte handle travels over any host channel; dfx_ipc_open maps it into
 * the CURRENT device's address space (cudaIpcMemLazyEnablePeerAccess), so kernels of the opening process may load from
 * it over NVLink. The owner keeps the allocation alive until every peer has called dfx_ipc_close.                  */
#define DFX_IPC_HANDLE_BYTES 64
DFX_API dfx_status dfx_ipc_alloc(size_t bytes, void** out_ptr, uint8_t handle[DFX_IPC_HANDLE_BYTES]);
DFX_API dfx_status dfx_ipc_free(void* ptr);
DFX_API dfx_status dfx_ipc_open(const uint8_t handle[DFX_IPC_HANDLE_BYTES], void** out_ptr);
DFX_API dfx_status dfx_ipc_close(void* mapped);

/* S5 ComputeSpatialReconstruction (…cpp:1001-1031; SSR_ComputeSpatialReconstruction.fx:114-172). Masked writes. */
DFX_API dfx_status dfx_pass_ssr_spatial(void* stream, const dfx_camera_attribs* cameras_dev,
                                        const dfx_ssr_attribs* attribs,
                                        const dfx_plane* roughness, const dfx_plane* mask, const dfx_plane* normal,
                                        const dfx_plane* depth, const dfx_plane* raydir_pdf, const dfx_plane* radiance,
                                        const dfx_plane* out_resolved_radiance, const dfx_plane* out_resolved_variance,
                                        const dfx_plane* out_resolved_depth, dfx_rows rows);

/* S6 ComputeTemporalAccumulation (…cpp:1033-1069; SSR_ComputeTemporalAccumulation.fx:224-263). Masked writes. */
DFX_API dfx_status dfx_pass_ssr_temporal(void* stream, const dfx_camera_attribs* cameras_dev,
                                         const dfx_ssr_attribs* attribs, const dfx_plane* mask,
                                         const dfx_plane* motion, const dfx_plane* hit_depth,
                                         const dfx_plane* reprojected_depth, const dfx_plane* curr_radiance,
                                         const dfx_plane* curr_variance, const dfx_plane* previous_depth,
                                         const dfx_plane* prev_radiance, const dfx_plane* prev_variance,
                                         const dfx_plane* out_radiance, const dfx_plane* out_variance, dfx_rows rows);

/* S6 on a row strip of a frame sharded over several GPUs: the previous-frame planes (previous depth, radiance and variance history),
 * which the pass reads at reprojected positions that no fixed halo bounds, are loaded from the GPU that owns the row. The three planes
 * must lie in the caller's slab (peers->base[peers->rank]). Bit-identical to dfx_pass_ssr_temporal on complete planes. */
DFX_API dfx_status dfx_pass_ssr_temporal_peer(void* stream, const dfx_camera_attribs* cameras_dev, const dfx_ssr_attribs* attribs,
                                              const dfx_peer_map* peers, const dfx_plane* mask, const dfx_plane* motion,
                                              const dfx_plane* hit_depth, const dfx_plane* reprojected_depth,
                                              const dfx_plane* curr_radiance, const dfx_plane* curr_variance,
                                              const dfx_plane* previous_depth, const dfx_plane* prev_radiance,
                                              const dfx_plane* prev_variance, const dfx_plane* out_radiance,
                                              const dfx_plane* out_variance, dfx_rows rows);

/* S7 ComputeBilateralCleanup (…cpp:1071-1104; SSR_ComputeBilateralCleanup.fx:49-97). Includes the clear to 0. */
DFX_API dfx_status dfx_pass_ssr_bilateral(void* stream, const dfx_camera_attribs* cameras_dev,
                                          const dfx_ssr_attribs* attribs, const dfx_plane* mask,
                                          const dfx_plane* depth, const dfx_plane* normal, const dfx_plane* roughness,
                                          const dfx_plane* radiance, const dfx_plane* variance,
                                          const dfx_plane* out, dfx_rows rows);

/* Bloom passes: `rows` is a row range of the OUTPUT plane of the call (the pyramid level being written), not of the
 * full-resolution frame — the levels have their own heights.
 * B1 ComputePrefilteredTexture (Bloom.cpp:288-311; Bloom_ComputePrefilteredTexture.fx:37-83). */
DFX_API dfx_status dfx_pass_bloom_prefilter(void* stream, const dfx_bloom_attribs* attribs,
                                            const dfx_plane* color, const dfx_plane* out_level0, dfx_rows rows);
/* B2 ComputeDownsampledTexture (Bloom.cpp:313-337; Bloom_ComputeDownsampledTexture.fx:11-41). */
DFX_API dfx_status dfx_pass_bloom_downsample(void* stream, const dfx_plane* in, const dfx_plane* out, dfx_rows rows);
/* B3 ComputeUpsampledTexture, uInstID==0 (Bloom.cpp:339-375; Bloom_ComputeUpsampledTexture.fx:20-54). */
DFX_API dfx_status dfx_pass_bloom_upsample(void* stream, const dfx_plane* same_level_down, const dfx_plane* coarser,
                                           const dfx_plane* out, dfx_rows rows);
/* B4 final composite, uInstID!=0 (Bloom.cpp:373-393; Bloom_ComputeUpsampledTexture.fx:45-48). */
DFX_API dfx_status dfx_pass_bloom_composite(void* stream, const dfx_bloom_attribs* attribs,
                                            const dfx_plane* color, const dfx_plane* up0, const dfx_plane* out, dfx_rows rows);

/* B2 for the levels first .. mips-1 followed by B3 for the levels mips-2 .. first-1, in ONE launch of one thread-block cluster
 * (the reference issues one draw per level, Bloom.cpp:324-337 and :355-375; on the small levels of the pyramid those dependent
 * launches cost more than the work). `down` / `up` are arrays of `mips` planes (level i = max(level0 >> i, 1)); reads
 * down[first-1], writes down[first..mips-1] and up[first-1..mips-2]. Results are bit-identical to the per-level passes.
 * dfx_bloom_tail_first_level: the level the effect object hands over to this pass (`mips` = none). Off by default (dfx_tune "bloom_tail" =
 * 1 switches it on: first level with <= "bloom_tail_texels" = 2048 texels): as a pass the cluster launch beats the per-level launches of the
 * same levels, but a cluster occupies 8 SMs of one GPC for 35 us, and under async compute the whole frame is 2 % faster without it
 * (profiles/r2k1). */
#define DFX_BLOOM_MAX_LEVELS 16
DFX_API dfx_status dfx_pass_bloom_tail(void* stream, const dfx_plane* down, const dfx_plane* up, int32_t first, int32_t mips);
DFX_API int32_t    dfx_bloom_tail_first_level(const dfx_plane* down, int32_t mips);
/* The same contract as dfx_pass_bloom_tail for levels of ANY size, in one cooperative launch over the whole GPU: a level is a phase
 * of a persistent grid, phases are separated by a grid-wide barrier (replaces the 5 + 5 draws of Bloom.cpp:324-337 / :355-375 at 4K).
 * `workspace`: 64 bytes of device memory, 16-byte aligned, zeroed once by the caller and used by one launch at a time (the kernel
 * leaves it zeroed). A barrier that is not reached within ~2 s raises an error word in the workspace instead of hanging the GPU:
 * dfx_bloom_levels_check reads it back (synchronises). Same taps in the same order as the per-level passes (results agree to the last
 * bit or two: FMA contraction). The effect object uses it when dfx_tune "bloom_levels" is 1; default 0 - under async compute the per-level
 * launches overlap the next frame better than a grid that needs the whole GPU (profiles/r2j). */
DFX_API dfx_status dfx_pass_bloom_levels(void* stream, const dfx_plane* down, const dfx_plane* up, int32_t first, int32_t mips, void* workspace);
DFX_API dfx_status dfx_bloom_levels_check(const void* workspace, int32_t* timed_out);

/* T1 ComputeTemporalAccumulation (TemporalAntiAliasing.cpp:260-289; TAA_ComputeTemporalAccumulation.fx:229-261). */
DFX_API dfx_status dfx_pass_taa(void* stream, const dfx_camera_attribs* cameras_dev, const dfx_taa_attribs* attribs,
                                uint32_t flags, const dfx_plane* curr_color, const dfx_plane* prev_accum,
                                const dfx_plane* closest_motion, const dfx_plane* reprojected_depth,
                                const dfx_plane* previous_depth, const dfx_plane* out_accum, dfx_rows rows);

/* Compose step between SSAO and TAA, reduced form (SURVEY.md §8f rank 1; Hydrogent/shaders/HnPostProcess.psh:145-185):
 *   rgb += ssr.rgb * ssr.a * ssr_scale;  rgb *= lerp(1, ao, ssao_scale);  alpha passes through.
 * ssr / ao may be NULL (scale treated as 0).                                                                   */
DFX_API dfx_status dfx_pass_compose(void* stream, const dfx_plane* color, const dfx_plane* ssr, const dfx_plane* ao,
                                    float ssr_scale, float ssao_scale, const dfx_plane* out, dfx_rows rows);

/* DepthOfField (PostProcess/DepthOfField/src/DepthOfField.cpp:292-331; Shaders/PostProcess/DepthOfField/private/DOF_*.fx), the
 * eleven passes in execution order. `rows` is always a row range of the OUTPUT plane of the call. Sizes: CoC planes
 * W x H; dilation level k (W >> k) x (H >> k), k = 0..3; prefiltered / bokeh planes (W/2) x (H/2), alpha = CoC of the layer.
 *   D1  coc            signed circle of confusion in [-1, 1] from depth and the lens fields of the camera (…CircleOfConfusion.fx:24-39)
 *   D2  temporal_coc   history reprojected by the closest motion, clamped to mean +- 2.5 sigma (…TemporalCircleOfConfusion.fx:54-92)
 *   D3  separated_coc  near field |CoC| (CoC < 0) -> dilation level 0 (…SeparatedCircleOfConfusion.fx:5-11)
 *   D4  dilation       2x2 (+ odd row / column) maximum, called for levels 1..3 (…DilationCircleOfConfusion.fx:16-52)
 *   D5/6 blur_coc      13-tap Gaussian (radius 6, sigma 5), horizontal into an intermediate plane, vertical back (…BlurredCoC.fx:8-28)
 *   D7  prefilter      SDR-weighted 2x2 mean -> foreground (alpha: blurred dilation, linear) and background (alpha: max far CoC)
 *   D8  bokeh, first   gather over the Octaweb kernel (rings, density from attribs), optional HDR ("Karis inverse") weights
 *   D9  bokeh, second  flood fill with the small 3 x 5 kernel (component-wise maximum)
 *   D10 postfilter     2x2 tent
 *   D11 combine        far layer, then near layer over the full-resolution colour by smoothstep(0.1, 1, alpha)            */
DFX_API dfx_status dfx_pass_dof_coc(void* stream, const dfx_camera_attribs* cameras_dev, const dfx_dof_attribs* attribs,
                                    const dfx_plane* depth, const dfx_plane* out_coc, dfx_rows rows);
DFX_API dfx_status dfx_pass_dof_temporal_coc(void* stream, const dfx_camera_attribs* cameras_dev, const dfx_dof_attribs* attribs,
                                             const dfx_plane* curr_coc, const dfx_plane* prev_coc, const dfx_plane* closest_motion,
                                             const dfx_plane* out_coc, dfx_rows rows);
DFX_API dfx_status dfx_pass_dof_separated_coc(void* stream, const dfx_plane* coc, const dfx_plane* out, dfx_rows rows);
DFX_API dfx_status dfx_pass_dof_dilation(void* stream, const dfx_plane* last, const dfx_plane* out, dfx_rows rows);
DFX_API dfx_status dfx_pass_dof_blur_coc(void* stream, const dfx_plane* coc, int32_t vertical, const dfx_plane* out, dfx_rows rows);
DFX_API dfx_status dfx_pass_dof_prefilter(void* stream, const dfx_plane* color, const dfx_plane* coc, const dfx_plane* dilation,
                                          const dfx_plane* out_fg, const dfx_plane* out_bg, dfx_rows rows);
/* radiance (the full-resolution colour) is read only with DFX_DOF_FEATURE_FLAG_ENABLE_KARIS_INVERSE in `flags`; may be NULL otherwise */
DFX_API dfx_status dfx_pass_dof_bokeh(void* stream, const dfx_camera_attribs* cameras_dev, const dfx_dof_attribs* attribs, uint32_t flags,
                                      int32_t second_pass, const dfx_plane* fg, const dfx_plane* bg, const dfx_plane* radiance,
                                      const dfx_plane* out_fg, const dfx_plane* out_bg, dfx_rows rows);
DFX_API dfx_status dfx_pass_dof_postfilter(void* stream, const dfx_plane* fg, const dfx_plane* bg, const dfx_plane* out_fg,
                                           const dfx_plane* out_bg, dfx_rows rows);
DFX_API dfx_status dfx_pass_dof_combine(void* stream, const dfx_dof_attribs* attribs, const dfx_plane* color, const dfx_plane* dof_near,
                                        const dfx_plane* dof_far, const dfx_plane* out, dfx_rows rows);

/* Compose step, full form (Hydrogent/shaders/HnPostProcess.psh:145-185; host HnPostProcessTask.cpp:834-869). With
 * Opacity = color.a:
 *   rgb += (GetSpecularIBL_GGX(surface, view, ssr.rgb) - specular_ibl.rgb) * ssr.a * ssr_scale * Opacity
 *   rgb *= lerp(1, ao, ssao_scale * Opacity);                       alpha passes through
 * i.e. the reflection is re-weighted by the split-sum BRDF of the surface (metallic-roughness workflow, PBR_Shading.fxh:
 * 220-302 with USE_IBL_MULTIPLE_SCATTERING = 1, :429-451; material.x = roughness, material.y = metallic) and exchanged for
 * the image-based specular term the renderer had already added. `brdf_lut` = dfx_pass_precompute_brdf_lut (RG32F, sampled
 * linear-clamp at (N.V, roughness)). ssr == NULL skips the first line (the five planes it needs may then be NULL too);
 * ao == NULL skips the second.                                                                                     */
DFX_API dfx_status dfx_pass_compose_ibl(void* stream, const dfx_camera_attribs* cameras_dev, const dfx_plane* color,
                                        const dfx_plane* ssr, const dfx_plane* ao, const dfx_plane* specular_ibl,
                                        const dfx_plane* normal, const dfx_plane* base_color, const dfx_plane* material,
                                        const dfx_plane* brdf_lut, float ssr_scale, float ssao_scale, const dfx_plane* out,
                                        dfx_rows rows);
/* Pre-integrated GGX table (Shaders/PBR/private/PrecomputeBRDF.psh:10-48; PBR_Renderer.cpp:548-625 builds it once at
 * 512 x 512 with 512 samples): texel (x, y) = (scale, bias) of the split sum at N.V = (x + .5)/w, roughness = (y + .5)/h. */
DFX_API dfx_status dfx_pass_precompute_brdf_lut(void* stream, uint32_t num_samples, const dfx_plane* out_lut);

/* M1+M2 ToneMap() (ToneMapping.fxh:87-226) + optional LinearToSRGB (SRGBUtilities.fxh:27-33), as used by
 * Hydrogent/shaders/HnCopyFrame.psh:32-62. ave_log_lum is the already exposure-scaled fAveLogLum argument.     */
DFX_API dfx_status dfx_pass_tonemap(void* stream, const dfx_tonemap_attribs* attribs, float ave_log_lum,
                                    int32_t convert_to_srgb, const dfx_plane* color, const dfx_plane* out, dfx_rows rows);

/* Fused variants (B200-first: an element-wise pass is evaluated inside the kernel that consumes / produces its plane, so the
 * intermediate frame never makes a round trip through HBM). Same arithmetic per pixel as the separate passes.
 *   compose + T1 : `color` is the un-composed scene colour; the composed colour is computed on the fly.
 *   B4 + M1/M2   : writes the tone-mapped LDR frame directly; only for exact 2:1 levels (DFX_ERR_UNSUPPORTED otherwise). */
DFX_API dfx_status dfx_pass_compose_taa(void* stream, const dfx_camera_attribs* cameras_dev, const dfx_taa_attribs* attribs, uint32_t flags,
                                        const dfx_plane* color, const dfx_plane* ssr, const dfx_plane* ao, float ssr_scale, float ssao_scale,
                                        const dfx_plane* prev_accum, const dfx_plane* closest_motion, const dfx_plane* reprojected_depth,
                                        const dfx_plane* previous_depth, const dfx_plane* out_accum, dfx_rows rows);
DFX_API dfx_status dfx_pass_bloom_composite_tonemap(void* stream, const dfx_bloom_attribs* attribs, const dfx_tonemap_attribs* tonemap, float ave_log_lum,
                                                    int32_t convert_to_srgb, const dfx_plane* color, const dfx_plane* up0, const dfx_plane* ldr_out,
                                                    dfx_rows rows);

/* Auto exposure with light adaptation (ToneMappingAttribs.bAutoExposure / bLightAdaptation, ToneMappingStructures.fxh:37,41). The
 * reference implements it in EpipolarLightScattering: a 64x64 RG16F target of GetWeightedLogLum (AtmosphereShadersCommon.fxh:199-205,
 * UnwarpEpipolarScattering.fx:285-307, point samples), GenerateMips down to 1x1 (EpipolarLightScattering.cpp:2469, :2503),
 * UpdateAverageLuminancePS (UpdateAverageLuminance.fx:12-29) alpha-blended into a persistent 1x1 R16F cleared to 0.1
 * (…cpp:1823-1827, :885-905), and the consumer max(0.05, state) -> ToneMap() (GetAverageSceneLuminance, AtmosphereShadersCommon.fxh:188-197).
 *
 * The state is a device buffer of DFX_AVERAGE_LUMINANCE_STATE_FLOATS floats, 16-byte aligned, owned by the caller:
 *   [0] the adapted luminance, rounded to half as the R16F target holds it     [1] max(0.05, [0]): the fAveLogLum the tone map uses
 *   [2] this frame's measurement exp(mean wlogL / mean w) (fp32, not rounded)  [3] the blend weight it entered with
 *   [4..] scratch of the full-frame mode (a ticket word and the per-CTA partials; left ready for the next launch).
 * dfx_pass_reset_average_luminance must run once before the first update. One update at a time per buffer (stream order).        */
#define DFX_LUMINANCE_SAMPLING_REFERENCE 1 /* 64x64 point samples, half-rounded mip chain: the reference bit for bit; one CTA         */
#define DFX_LUMINANCE_SAMPLING_FULL      2 /* every pixel, fp32 per CTA, fp64 fixed-order total; deterministic                     */
#define DFX_AVERAGE_LUMINANCE_MAX_PARTIALS 512
#define DFX_AVERAGE_LUMINANCE_STATE_FLOATS (8 + 2 * DFX_AVERAGE_LUMINANCE_MAX_PARTIALS)
/* Measures `color` (RGBA32F or RGBA16F, any size) and blends the measurement into the state: weight
 * (1 - exp(-elapsed_seconds)) * saturate(mean w / 1e-3) with attribs->bLightAdaptation, saturate(mean w / 1e-3) without.
 * Replaces the luminance branch of ApplyInscatteredRadiancePS, GenerateMips and UpdateAverageLuminancePS (EpipolarLightScattering.cpp:2463-2481). */
DFX_API dfx_status dfx_pass_update_average_luminance(void* stream, const dfx_tonemap_attribs* attribs, int32_t sampling, float elapsed_seconds,
                                                     const dfx_plane* color, float* state_dev);
/* state := 0.1 as R16F holds it (0.0999755859375; the clear of EpipolarLightScattering.cpp:885-905), scratch words zeroed. */
DFX_API dfx_status dfx_pass_reset_average_luminance(void* stream, float* state_dev);
/* dfx_pass_tonemap / dfx_pass_bloom_composite_tonemap with fAveLogLum = max(0.05, *ave_log_lum_dev) read on the device (pass the state
 * buffer itself): bit-identical to the scalar entries given max(0.05, that value).                                                   */
DFX_API dfx_status dfx_pass_tonemap_dev(void* stream, const dfx_tonemap_attribs* attribs, const float* ave_log_lum_dev,
                                        int32_t convert_to_srgb, const dfx_plane* color, const dfx_plane* out, dfx_rows rows);
DFX_API dfx_status dfx_pass_bloom_composite_tonemap_dev(void* stream, const dfx_bloom_attribs* attribs, const dfx_tonemap_attribs* tonemap,
                                                        const float* ave_log_lum_dev, int32_t convert_to_srgb, const dfx_plane* color,
                                                        const dfx_plane* up0, const dfx_plane* ldr_out, dfx_rows rows);

/* Host-side pieces that the reference computes on the CPU. */
/* TemporalAntiAliasing::GetJitterOffset (TemporalAntiAliasing.cpp:63-78, Halton(2,3) x16). */
DFX_API void dfx_taa_jitter_offset(uint32_t frame_index, uint32_t width, uint32_t height, float out_jitter[2]);
/* Bloom::ComputeMipCount (Bloom.cpp:152-156) applied to the half-resolution level-0 size. */
DFX_API int32_t dfx_bloom_mip_count(uint32_t width, uint32_t height, float radius);

/* Implementation switches for A/B measurements (tools/, bench.py --tune): every value of a knob computes the same pass, through a
 * different kernel. Unknown names read as `fallback`. Also settable at load time: DFX_TUNE="name=value,name=value". */
DFX_API void    dfx_tune_set(const char* name, int32_t value);
DFX_API int32_t dfx_tune_get(const char* name, int32_t fallback);
DFX_API void    dfx_tune_unset(const char* name); /* back to the built-in default (NULL: every knob) */

/* ============================================================================================================ */
/* 2. effect level                                                                                              */
/* ============================================================================================================ */

typedef struct dfx_postfx dfx_postfx;
typedef struct dfx_ssao   dfx_ssao;
typedef struct dfx_ssr    dfx_ssr;
typedef struct dfx_bloom  dfx_bloom;
typedef struct dfx_taa    dfx_taa;

/* plane ids for dfx_*_get_plane */
enum
{
    DFX_POSTFX_PLANE_BLUE_NOISE_XY     = 0,
    DFX_POSTFX_PLANE_BLUE_NOISE_ZW     = 1,
    DFX_POSTFX_PLANE_REPROJECTED_DEPTH = 2,
    DFX_POSTFX_PLANE_PREVIOUS_DEPTH    = 3,
    DFX_POSTFX_PLANE_CLOSEST_MOTION    = 4
};
enum
{
    DFX_SSAO_PLANE_OUTPUT            = 0,  /* == GetAmbientOcclusionSRV()                       */
    DFX_SSAO_PLANE_OCCLUSION         = 1,  /* raw AO (A3)                                       */
    DFX_SSAO_PLANE_ACCUMULATED       = 2,  /* A5 output == convoluted-AO mip 0                  */
    DFX_SSAO_PLANE_HISTORY_LENGTH    = 3,  /* A5 history length of the current frame            */
    DFX_SSAO_PLANE_RESAMPLED         = 4,  /* A7                                                */
    DFX_SSAO_PLANE_UPSAMPLED         = 5,  /* A4 (half resolution only); OCCLUSION is then width/2 x height/2 */
    DFX_SSAO_PLANE_PREFILTERED_MIP0  = 10, /* +i : prefiltered depth mip i (0..4)               */
    DFX_SSAO_PLANE_CONV_AO_MIP0      = 20, /* +i : convoluted AO mip i (0..4)                   */
    DFX_SSAO_PLANE_CONV_DEPTH_MIP0   = 30  /* +i : convoluted depth mip i (0..4)                */
};
enum
{
    DFX_SSR_PLANE_OUTPUT            = 0,  /* == GetSSRRadianceSRV()                             */
    DFX_SSR_PLANE_ROUGHNESS         = 1,
    DFX_SSR_PLANE_MASK              = 2,
    DFX_SSR_PLANE_RADIANCE          = 3,
    DFX_SSR_PLANE_RAYDIR_PDF        = 4,
    DFX_SSR_PLANE_RESOLVED_RADIANCE = 5,
    DFX_SSR_PLANE_RESOLVED_VARIANCE = 6,
    DFX_SSR_PLANE_RESOLVED_DEPTH    = 7,
    DFX_SSR_PLANE_RADIANCE_HISTORY  = 8,  /* current frame's slot                               */
    DFX_SSR_PLANE_VARIANCE_HISTORY  = 9,
    DFX_SSR_PLANE_HIZ_MIP0          = 10, /* +i : Hi-Z mip i (0..6)                             */
    DFX_SSR_PLANE_MASK_HALF         = 20  /* S3 (half resolution only); RADIANCE / RAYDIR_PDF are then half size */
};
enum
{
    DFX_BLOOM_PLANE_OUTPUT    = 0,   /* == GetBloomTextureSRV()                                 */
    DFX_BLOOM_PLANE_DOWN0     = 10,  /* +i : downsampled level i                                */
    DFX_BLOOM_PLANE_UP0       = 30   /* +i : upsampled level i                                  */
};
enum
{
    DFX_TAA_PLANE_ACCUMULATED_CURR = 0, /* == GetAccumulatedFrameSRV(false)                     */
    DFX_TAA_PLANE_ACCUMULATED_PREV = 1  /* == GetAccumulatedFrameSRV(true)                      */
};

/* ---- PostFXContext (PostProcess/Common/interface/PostFXContext.hpp:51-172) ---- */
typedef struct dfx_postfx_render_attribs
{
    void*                     stream;          /* stands in for pDeviceContext                   */
    const dfx_plane*          curr_depth;      /* pCurrDepthBufferSRV  R32F                      */
    const dfx_plane*          prev_depth;      /* pPrevDepthBufferSRV  R32F                      */
    const dfx_plane*          motion_vectors;  /* pMotionVectorsSRV    RG32F                     */
    const dfx_camera_attribs* curr_camera;     /* host pointers, uploaded like PostFXContext.cpp:302-319 */
    const dfx_camera_attribs* prev_camera;
} dfx_postfx_render_attribs;

DFX_API dfx_status dfx_postfx_create(dfx_postfx** out);
DFX_API void       dfx_postfx_destroy(dfx_postfx* ctx);
DFX_API dfx_status dfx_postfx_prepare(dfx_postfx* ctx, const dfx_frame_desc* desc, uint32_t feature_flags);
DFX_API dfx_status dfx_postfx_execute(dfx_postfx* ctx, const dfx_postfx_render_attribs* attribs);
DFX_API dfx_status dfx_postfx_get_plane(const dfx_postfx* ctx, int32_t id, dfx_plane* out);
DFX_API dfx_status dfx_postfx_get_frame_desc(const dfx_postfx* ctx, dfx_frame_desc* out);
DFX_API const dfx_camera_attribs* dfx_postfx_get_camera_attribs_dev(const dfx_postfx* ctx); /* GetCameraAttribsCB */

/* ---- ScreenSpaceAmbientOcclusion (…/ScreenSpaceAmbientOcclusion.hpp:59-136) ---- */
typedef struct dfx_ssao_render_attribs
{
    void*                   stream;
    dfx_postfx*             postfx;  /* pPostFXContext   */
    const dfx_plane*        depth;   /* pDepthBufferSRV  R32F    */
    const dfx_plane*        normal;  /* pNormalBufferSRV RGBA32F (xyz world-space normal) */
    const dfx_ssao_attribs* attribs; /* pSSAOAttribs     */
} dfx_ssao_render_attribs;

DFX_API dfx_status dfx_ssao_create(dfx_ssao** out);
DFX_API void       dfx_ssao_destroy(dfx_ssao* fx);
DFX_API dfx_status dfx_ssao_prepare(dfx_ssao* fx, dfx_postfx* postfx, uint32_t feature_flags);
/* The reference fades the effect in with wall-clock time (AlphaInterpolation, …cpp:793-795). `alpha < 0`
 * restores that behaviour; parity runs pin it (default after create: pinned to 1.0).                            */
DFX_API dfx_status dfx_ssao_set_alpha_interpolation(dfx_ssao* fx, float alpha);
DFX_API dfx_status dfx_ssao_execute(dfx_ssao* fx, const dfx_ssao_render_attribs* attribs);
DFX_API dfx_status dfx_ssao_get_plane(const dfx_ssao* fx, int32_t id, dfx_plane* out);

/* ---- ScreenSpaceReflection (…/ScreenSpaceReflection.hpp:64-139) ---- */
typedef struct dfx_ssr_render_attribs
{
    void*                  stream;
    dfx_postfx*            postfx;
    const dfx_plane*       color;     /* pColorBufferSRV    RGBA32F */
    const dfx_plane*       depth;     /* pDepthBufferSRV    R32F    */
    const dfx_plane*       normal;    /* pNormalBufferSRV   RGBA32F */
    const dfx_plane*       material;  /* pMaterialBufferSRV RGBA32F */
    const dfx_plane*       motion;    /* pMotionVectorsSRV  RG32F   */
    const dfx_ssr_attribs* attribs;   /* pSSRAttribs        */
} dfx_ssr_render_attribs;

DFX_API dfx_status dfx_ssr_create(dfx_ssr** out);
DFX_API void       dfx_ssr_destroy(dfx_ssr* fx);
DFX_API dfx_status dfx_ssr_prepare(dfx_ssr* fx, dfx_postfx* postfx, uint32_t feature_flags);
DFX_API dfx_status dfx_ssr_set_alpha_interpolation(dfx_ssr* fx, float alpha);
DFX_API dfx_status dfx_ssr_execute(dfx_ssr* fx, const dfx_ssr_render_attribs* attribs);
DFX_API dfx_status dfx_ssr_get_plane(const dfx_ssr* fx, int32_t id, dfx_plane* out);

/* ---- Bloom (…/Bloom.hpp:60-114) ---- */
typedef struct dfx_bloom_render_attribs
{
    void*                    stream;
    dfx_postfx*              postfx;
    const dfx_plane*         color;   /* pColorBufferSRV RGBA32F */
    const dfx_bloom_attribs* attribs; /* pBloomAttribs   */
} dfx_bloom_render_attribs;

DFX_API dfx_status dfx_bloom_create(dfx_bloom** out);
DFX_API void       dfx_bloom_destroy(dfx_bloom* fx);
DFX_API dfx_status dfx_bloom_prepare(dfx_bloom* fx, dfx_postfx* postfx, uint32_t feature_flags);
DFX_API dfx_status dfx_bloom_set_alpha_interpolation(dfx_bloom* fx, float alpha);
DFX_API dfx_status dfx_bloom_execute(dfx_bloom* fx, const dfx_bloom_render_attribs* attribs);
DFX_API dfx_status dfx_bloom_get_plane(const dfx_bloom* fx, int32_t id, dfx_plane* out);
/* Bloom + final ToneMap(+sRGB) with the last two kernels fused; writes `ldr_out`, does not update the bloom output plane. */
DFX_API dfx_status dfx_bloom_execute_tonemapped(dfx_bloom* fx, const dfx_bloom_render_attribs* attribs, const dfx_tonemap_attribs* tonemap,
                                                float ave_log_lum, int32_t convert_to_srgb, const dfx_plane* ldr_out);

/* ---- DepthOfField (PostProcess/DepthOfField/interface/DepthOfField.hpp:59-125) ---- */
typedef struct dfx_dof dfx_dof;
typedef struct dfx_dof_render_attribs
{
    void*                  stream;
    dfx_postfx*            postfx;  /* camera (lens fields included), frame index, closest motion */
    const dfx_plane*       color;   /* pColorBufferSRV RGBA32F */
    const dfx_plane*       depth;   /* pDepthBufferSRV R32F    */
    const dfx_dof_attribs* attribs; /* pDOFAttribs             */
} dfx_dof_render_attribs;
typedef enum dfx_dof_plane_id
{
    DFX_DOF_PLANE_OUTPUT        = 0,  /* == GetDepthOfFieldTextureSRV(): combined colour, alpha of the input kept */
    DFX_DOF_PLANE_COC           = 1,  /* D1                                                   */
    DFX_DOF_PLANE_COC_TEMPORAL  = 2,  /* D2, current frame's slot (temporal smoothing only)   */
    DFX_DOF_PLANE_DILATION_MIP0 = 10, /* +k : dilation level k (0..3); level 3 is blurred     */
    DFX_DOF_PLANE_PREFILTERED0  = 20, /* +i : foreground (0) / background (1) after D9        */
    DFX_DOF_PLANE_BOKEH0        = 22  /* +i : foreground (0) / background (1) after D10       */
} dfx_dof_plane_id;
DFX_API dfx_status dfx_dof_create(dfx_dof** out);
DFX_API void       dfx_dof_destroy(dfx_dof* fx);
DFX_API dfx_status dfx_dof_prepare(dfx_dof* fx, dfx_postfx* postfx, uint32_t feature_flags);
DFX_API dfx_status dfx_dof_set_alpha_interpolation(dfx_dof* fx, float alpha);
DFX_API dfx_status dfx_dof_execute(dfx_dof* fx, const dfx_dof_render_attribs* attribs);
DFX_API dfx_status dfx_dof_get_plane(const dfx_dof* fx, int32_t id, dfx_plane* out);

/* ---- TemporalAntiAliasing (…/TemporalAntiAliasing.hpp:62-156) ---- */
typedef struct dfx_taa_render_attribs
{
    void*                  stream;
    dfx_postfx*            postfx;
    const dfx_plane*       color;   /* pColorBufferSRV RGBA32F */
    const dfx_taa_attribs* attribs; /* pTAAAttribs     */
    uint32_t               accumulation_buffer_idx;
} dfx_taa_render_attribs;

DFX_API dfx_status dfx_taa_create(dfx_taa** out);
DFX_API void       dfx_taa_destroy(dfx_taa* fx);
DFX_API dfx_status dfx_taa_prepare(dfx_taa* fx, dfx_postfx* postfx, uint32_t feature_flags, uint32_t accumulation_buffer_idx);
DFX_API dfx_status dfx_taa_execute(dfx_taa* fx, const dfx_taa_render_attribs* attribs);
/* TAA with the compose step evaluated on the fly (attribs->color = un-composed scene colour; ssr / ao may be NULL). */
DFX_API dfx_status dfx_taa_execute_composed(dfx_taa* fx, const dfx_taa_render_attribs* attribs, const dfx_plane* ssr, const dfx_plane* ao,
                                            float ssr_scale, float ssao_scale);
DFX_API dfx_status dfx_taa_get_plane(const dfx_taa* fx, int32_t id, uint32_t accumulation_buffer_idx, dfx_plane* out);
DFX_API dfx_status dfx_taa_get_jitter_offset(const dfx_taa* fx, uint32_t accumulation_buffer_idx, float out_jitter[2]);

/* ============================================================================================================ */
/* Ingest / egress in the reference's render-target formats (Hydrogent/src/Tasks/HnBeginFrameTask.cpp:63-69: scene colour
 * and normal RGBA16_FLOAT, motion RG16_FLOAT, material RG8_UNORM; the final target is an 8-bit sRGB swap chain). The
 * passes keep fp32 planes in HBM; these two entries convert at the PCIe boundary so that the narrow formats are what
 * travels (30 B/px in, 4 B/px out instead of 64 / 16). Widening is exact.
 *   unpack: RGBA16F -> RGBA32F, RG16F -> RG32F, RG8U -> RGBA32F (x, y = c/255; z = w = 0)
 *   pack  : RGBA32F -> RGBA8U, D3D UNORM rule: saturate, * 255, + 0.5, truncate (NaN -> 0)                        */
DFX_API dfx_status dfx_pass_unpack_plane(void* stream, const dfx_plane* src, const dfx_plane* dst, dfx_rows rows);
DFX_API dfx_status dfx_pass_pack_ldr8(void* stream, const dfx_plane* src_rgba32f, const dfx_plane* dst_rgba8u, dfx_rows rows);

/* ============================================================================================================ */
/* plane helpers (device memory owned by the library; used by the C++ shim and the tests)                       */
DFX_API dfx_status dfx_plane_alloc(int32_t width, int32_t height, int32_t format, dfx_plane* out);
DFX_API void       dfx_plane_free(dfx_plane* p);
DFX_API dfx_status dfx_plane_upload(void* stream, const dfx_plane* dst, const void* host_src, size_t host_pitch_bytes);
DFX_API dfx_status dfx_plane_download(void* stream, const dfx_plane* src, void* host_dst, size_t host_pitch_bytes);
DFX_API dfx_status dfx_plane_fill(void* stream, const dfx_plane* dst, const float value[4]);
DFX_API dfx_status dfx_stream_synchronize(void* stream);

/* Optional per-pass device timing (stands in for the reference's ScopedDebugGroup markers, e.g. ScreenSpaceAmbientOcclusion.cpp:363):
 * while enabled every dfx_pass_* call is bracketed by two CUDA events on its stream. Not thread-safe; one stream at a time. */
DFX_API void       dfx_profile_enable(int32_t on);
DFX_API dfx_status dfx_profile_collect(void);                 /* waits for the recorded events, folds them into per-pass totals */
DFX_API void       dfx_profile_reset(void);
DFX_API int32_t    dfx_profile_count(void);
DFX_API dfx_status dfx_profile_entry(int32_t i, char* name, int32_t name_cap, double* total_ms, int32_t* calls);

/* ============================================================================================================ */
/* 3. chain level: the whole PostProcess chain of one view, one call per frame                                    */
/* ============================================================================================================ */
/* Owns one PostFXContext, SSAO, SSR, TAA, DepthOfField and Bloom object and runs them in the order of the reference's only in-tree
 * integration (Hydrogent/src/Tasks/HnPostProcessTask.cpp: Prepare :591-683, Execute :743-947):
 *   PostFXContext -> SSR -> SSAO -> compose -> TAA -> [DepthOfField] -> Bloom -> ToneMap(+sRGB).
 * The SSAO passes run beside the SSR passes on a second stream, Bloom + ToneMap of frame f beside the front half of frame f+1
 * on a third; in steady state (consecutive frame indices, no history reset, constant attributes) the launches are replayed
 * from CUDA graphs cached per (input planes, ping-pong parity, configuration). Results are bit-identical whichever way a frame
 * is issued. Not thread-safe: one chain per view / stream of frames, like the reference's effect objects. */
#define DFX_CHAIN_STAGE_POSTFX  1u
#define DFX_CHAIN_STAGE_SSR     2u
#define DFX_CHAIN_STAGE_SSAO    4u
#define DFX_CHAIN_STAGE_COMPOSE 8u
#define DFX_CHAIN_STAGE_TAA     16u
#define DFX_CHAIN_STAGE_BLOOM   32u
#define DFX_CHAIN_STAGE_TONEMAP 64u
#define DFX_CHAIN_STAGE_ALL     127u

typedef struct dfx_chain_config
{
    dfx_ssao_attribs    ssao;
    dfx_ssr_attribs     ssr;
    dfx_bloom_attribs   bloom;
    dfx_taa_attribs     taa;
    dfx_tonemap_attribs tonemap;
    dfx_dof_attribs     dof;
    uint32_t postfx_flags, ssao_flags, ssr_flags, taa_flags, dof_flags; /* DFX_*_FEATURE_FLAG_* */
    uint32_t stages;      /* DFX_CHAIN_STAGE_* mask                                                                          */
    int32_t  enable_dof;  /* DepthOfField between TAA and Bloom (HnPostProcessTask.cpp:899-909)                                */
    int32_t  fuse;        /* compose inside TAA, ToneMap inside the Bloom composite (same arithmetic, two HBM round trips fewer) */
    int32_t  overlap;     /* async compute on three streams                                                                  */
    int32_t  use_graph;   /* replay steady-state frames from CUDA graphs                                                     */
    int32_t  to_srgb;     /* LinearToSRGB after the tone map (HnCopyFrame.psh:60-62)                                         */
    float    ave_log_lum; /* HnPostProcessTask.hpp:88                                                                        */
    float    ssr_scale, ssao_scale; /* compose: rgb += ssr.rgb * ssr.a * ssr_scale; rgb *= lerp(1, ao, ssao_scale)           */
    /* 0: the constant ave_log_lum (HnCopyFrame.psh:35). 1 / 2 (DFX_LUMINANCE_SAMPLING_*): measure the colour Bloom receives and
     * tone-map with the adapted luminance, when tonemap.bAutoExposure is set (else the constant); tonemap.bLightAdaptation and
     * dfx_chain_set_elapsed_time drive the adaptation. The state restarts at 0.1 whenever the histories reset.               */
    int32_t  auto_exposure;
} dfx_chain_config;

typedef struct dfx_chain_frame
{
    uint32_t                  frame_index;  /* FrameDesc.Index: consecutive, or the histories reset                          */
    int32_t                   defer_post;   /* 1: return without making `stream` wait for Bloom + ToneMap (dfx_chain_join)    */
    const dfx_camera_attribs* curr_camera;  /* host pointers                                                                 */
    const dfx_camera_attribs* prev_camera;
    const dfx_plane*          depth;        /* R32F    */
    const dfx_plane*          prev_depth;   /* R32F    */
    const dfx_plane*          motion;       /* RG32F   */
    const dfx_plane*          normal;       /* RGBA32F */
    const dfx_plane*          color;        /* RGBA32F */
    const dfx_plane*          material;     /* RGBA32F */
    const dfx_plane*          ldr_out;      /* RGBA32F: the tone-mapped frame                                                */
} dfx_chain_frame;

typedef struct dfx_chain_stats
{
    uint64_t frames_eager, frames_replayed, graphs_built, graph_failures;
} dfx_chain_stats;

typedef enum dfx_chain_effect_id
{
    DFX_CHAIN_EFFECT_POSTFX = 0, DFX_CHAIN_EFFECT_SSAO = 1, DFX_CHAIN_EFFECT_SSR = 2, DFX_CHAIN_EFFECT_BLOOM = 3, DFX_CHAIN_EFFECT_TAA = 4, DFX_CHAIN_EFFECT_DOF = 5
} dfx_chain_effect_id;

typedef struct dfx_chain dfx_chain;
DFX_API void       dfx_chain_config_default(dfx_chain_config* config); /* reference struct defaults, Hydrogent's TAA flags, every stage, fused, async, graphs */
DFX_API dfx_status dfx_chain_create(int32_t width, int32_t height, const dfx_chain_config* config /* NULL = defaults */, dfx_chain** out);
DFX_API void       dfx_chain_destroy(dfx_chain* chain);
DFX_API dfx_status dfx_chain_set_config(dfx_chain* chain, const dfx_chain_config* config);
DFX_API dfx_status dfx_chain_get_config(const dfx_chain* chain, dfx_chain_config* out);
/* Runs one frame, ordered after the work already on `stream`; the frame's LDR plane is complete in stream order when the call
 * returns (defer_post = 0) or after dfx_chain_join (defer_post = 1). */
DFX_API dfx_status dfx_chain_execute(dfx_chain* chain, void* stream, const dfx_chain_frame* frame);
DFX_API dfx_status dfx_chain_join(dfx_chain* chain, void* stream);
/* The effect objects (dfx_postfx*, dfx_ssao*, ...) for dfx_*_get_plane / dfx_*_set_alpha_interpolation; owned by the chain. */
DFX_API void*      dfx_chain_effect(dfx_chain* chain, int32_t which /* dfx_chain_effect_id */);
/* The stream Bloom + ToneMap run on when `overlap` is set (to order a read-back after a deferred frame). */
DFX_API void*      dfx_chain_post_stream(dfx_chain* chain);
DFX_API dfx_status dfx_chain_get_stats(const dfx_chain* chain, dfx_chain_stats* out);
/* Seconds since the previous frame (FrameAttribs.dElapsedTime of the reference) for light adaptation, from the next dfx_chain_execute
 * on; it travels with the cameras, so it may change every frame while frames keep replaying from graphs. Default 0. */
DFX_API dfx_status dfx_chain_set_elapsed_time(dfx_chain* chain, float seconds);
/* The chain's average-luminance state (layout above dfx_pass_update_average_luminance); valid in the post stream's order. */
DFX_API const float* dfx_chain_average_luminance_dev(const dfx_chain* chain);

/* ============================================================================================================ */
/* 4. one frame split into row strips over the GPUs of a box (no reference counterpart)                          */
/* ============================================================================================================ */
/* ScreenSpaceReflection S1-S7 (+ the PostFXContext planes they read) on the strip [row_begin[rank], row_begin[rank+1]) of a frame
 * whose other strips are computed by other GPUs (BASELINE.json config 4). Every rank allocates one slab of
 * dfx_ssr_strips_slab_bytes() bytes (dfx_ipc_alloc), maps the other ranks' slabs (dfx_ipc_open) and hands all base addresses
 * over in a dfx_peer_map; all planes live in the slab at offsets that depend on the frame size only. Halo rows of bounded taps are
 * pushed into the neighbours' slabs by a copy kernel and announced through flags in peer memory; the ray march and the temporal
 * pass load what they need beyond the strip from the owning GPU directly (NVLink peer loads); there is no host synchronisation and
 * no NCCL call per frame. The sharded frame is bit-identical to the unsharded one. Several ranks may also live in one process on
 * one device (plain cudaMalloc slabs, one stream per rank): that is how the single-GPU tests cover this path. */
typedef enum dfx_ssr_strips_plane_id
{
    /* inputs: the caller writes its own rows */
    DFX_SSR_STRIPS_PLANE_DEPTH = 0, DFX_SSR_STRIPS_PLANE_PREV_DEPTH_IN = 1, DFX_SSR_STRIPS_PLANE_MOTION = 2, DFX_SSR_STRIPS_PLANE_NORMAL = 3,
    DFX_SSR_STRIPS_PLANE_COLOR = 4, DFX_SSR_STRIPS_PLANE_MATERIAL = 5,
    /* PostFXContext */
    DFX_SSR_STRIPS_PLANE_REPROJECTED_DEPTH = 6, DFX_SSR_STRIPS_PLANE_CLOSEST_MOTION = 7, DFX_SSR_STRIPS_PLANE_PREVIOUS_DEPTH = 8,
    /* SSR */
    DFX_SSR_STRIPS_PLANE_HIZ1 = 9, /* .. HIZ6 = 14 */
    DFX_SSR_STRIPS_PLANE_ROUGHNESS = 15, DFX_SSR_STRIPS_PLANE_MASK = 16, DFX_SSR_STRIPS_PLANE_RADIANCE = 17, DFX_SSR_STRIPS_PLANE_RAYDIR = 18,
    DFX_SSR_STRIPS_PLANE_RESOLVED_RADIANCE = 19, DFX_SSR_STRIPS_PLANE_RESOLVED_VARIANCE = 20, DFX_SSR_STRIPS_PLANE_RESOLVED_DEPTH = 21,
    DFX_SSR_STRIPS_PLANE_RADIANCE_HISTORY0 = 22, DFX_SSR_STRIPS_PLANE_RADIANCE_HISTORY1 = 23, DFX_SSR_STRIPS_PLANE_VARIANCE_HISTORY0 = 24,
    DFX_SSR_STRIPS_PLANE_VARIANCE_HISTORY1 = 25,
    DFX_SSR_STRIPS_PLANE_OUTPUT = 26, /* == GetSSRRadianceSRV(), valid on the own rows */
    DFX_SSR_STRIPS_PLANE_COUNT = 27
} dfx_ssr_strips_plane_id;

typedef struct dfx_ssr_strips dfx_ssr_strips;
DFX_API size_t     dfx_ssr_strips_slab_bytes(int32_t width, int32_t height);
/* peers->base[peers->rank] is this rank's slab (zeroed by this call: make sure no peer touches it before all ranks have returned);
 * blue_noise_tables: the 131,328-byte Sobol + scrambling-tile blob (host memory). */
DFX_API dfx_status dfx_ssr_strips_create(int32_t width, int32_t height, const dfx_peer_map* peers, const uint8_t* blue_noise_tables, dfx_ssr_strips** out);
DFX_API void       dfx_ssr_strips_destroy(dfx_ssr_strips* strips);
DFX_API dfx_status dfx_ssr_strips_plane(const dfx_ssr_strips* strips, int32_t id, dfx_plane* out);
DFX_API dfx_status dfx_ssr_strips_rows(const dfx_ssr_strips* strips, dfx_rows* out);
/* One frame on this rank's strip; every rank of the map calls it for every frame. Ends with an all-rank barrier in stream order. */
DFX_API dfx_status dfx_ssr_strips_execute(dfx_ssr_strips* strips, void* stream, uint32_t frame_index, const dfx_camera_attribs* curr_camera,
                                          const dfx_camera_attribs* prev_camera, const dfx_ssr_attribs* attribs);
/* *timed_out = 1 if a flag wait of an earlier frame gave up after ~2 s (a peer never signalled). Synchronises the device. */
DFX_API dfx_status dfx_ssr_strips_check(const dfx_ssr_strips* strips, int32_t* timed_out);

#ifdef __cplusplus
} /* extern "C" */
#endif
#endif /* DFX_B200_H */

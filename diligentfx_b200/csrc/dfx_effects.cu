// dfx_effects.cu — effect-level objects of the C-ABI: they own the internal planes (pyramids, history ping-pong) and
// sequence the pass-level entries exactly like the reference classes sequence their draws:
//   PostFXContext::Execute                 PostProcess/Common/src/PostFXContext.cpp:287-338
//   ScreenSpaceAmbientOcclusion::Execute   …/ScreenSpaceAmbientOcclusion.cpp:348-387 (+ UpdateConstantBuffer :790-816)
//   ScreenSpaceReflection::Execute         …/ScreenSpaceReflection.cpp:300-341
//   Bloom::Execute                         …/Bloom.cpp:407-436
//   TemporalAntiAliasing::Execute          …/TemporalAntiAliasing.cpp:169-201 (+ UpdateConstantBuffer :123-141)
#include "dfx_common.cuh"
#include <chrono>
#include <cstring>
#include <string>
#include <map>
#include <new>
#include <vector>

#include "_gen/blue_noise_tables.inc" // static const unsigned char kBlueNoiseTables[131328] (generated at build time from data/blue_noise_tables.bin)

using namespace dfx;

namespace
{
using Clock = std::chrono::steady_clock;

struct PlaneOwner
{
    dfx_plane p{};
    ~PlaneOwner() { dfx_plane_free(&p); }
    dfx_status alloc(int w, int h, int fmt)
    {
        dfx_plane_free(&p);
        return dfx_plane_alloc(w, h, fmt, &p);
    }
};

dfx_status clear_plane(cudaStream_t s, const dfx_plane& p, float v)
{
    const float c[4] = {v, v, v, v};
    return dfx_plane_fill(s, &p, c);
}

// AlphaInterpolation = clamp(seconds since the effect became ready, 0, 1) unless pinned (SURVEY.md Appendix B.9)
struct AlphaTimer
{
    float             pinned = 1.0f; // < 0 -> wall clock
    bool              started = false;
    Clock::time_point t0;
    float             value()
    {
        if (pinned >= 0.0f) return pinned;
        if (!started) started = true, t0 = Clock::now();
        float s = std::chrono::duration<float>(Clock::now() - t0).count();
        return s < 0.0f ? 0.0f : (s > 1.0f ? 1.0f : s);
    }
};
} // namespace

// =====================================================================================================================
// PostFXContext
// =====================================================================================================================
struct dfx_postfx
{
    dfx_frame_desc      desc{};
    uint32_t            flags    = 0;
    bool                prepared = false, executed = false;
    uint8_t*            tables_dev = nullptr;
    dfx_camera_attribs* cams_dev   = nullptr; // {curr, prev} followed by the frame index (uint32) the blue-noise pass reads and,
    uint32_t*           frame_dev  = nullptr; // in the two words after it, the chain's elapsed time per ping-pong parity (float)
    PlaneOwner          bn_xy, bn_zw, reproj, prev_depth, closest;
    int                 w = 0, h = 0;
    ~dfx_postfx()
    {
        cudaFree(tables_dev);
        cudaFree(cams_dev);
    }
};

extern "C" dfx_status dfx_postfx_create(dfx_postfx** out)
{
    DFX_REQUIRE(out, "out must not be null");
    dfx_postfx* c = new (std::nothrow) dfx_postfx;
    DFX_REQUIRE(c, "out of memory");
    cudaError_t e = cudaMalloc((void**)&c->tables_dev, sizeof(kBlueNoiseTables));
    if (e == cudaSuccess) e = cudaMemcpy(c->tables_dev, kBlueNoiseTables, sizeof(kBlueNoiseTables), cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMalloc((void**)&c->cams_dev, 2 * sizeof(dfx_camera_attribs) + 16);
    if (e == cudaSuccess) c->frame_dev = reinterpret_cast<uint32_t*>(c->cams_dev + 2);
    dfx_status st = DFX_OK;
    if (e != cudaSuccess) st = check_cuda(e, "dfx_postfx_create");
    if (st == DFX_OK) st = c->bn_xy.alloc(128, 128, DFX_FORMAT_RG32F);
    if (st == DFX_OK) st = c->bn_zw.alloc(128, 128, DFX_FORMAT_RG32F);
    if (st != DFX_OK)
    {
        delete c;
        return st;
    }
    *out = c;
    return DFX_OK;
}
extern "C" void dfx_postfx_destroy(dfx_postfx* c) { delete c; }

extern "C" dfx_status dfx_postfx_prepare(dfx_postfx* c, const dfx_frame_desc* desc, uint32_t flags)
{
    DFX_REQUIRE(c && desc, "null argument");
    // HALF_PRECISION_DEPTH only selects R16_UNORM for the reprojected / previous depth textures (PostFXContext.cpp:259, :270); this
    // library keeps every plane in fp32 and models none of the reference's narrow formats (DESIGN.md §2), so the flag is accepted
    // and changes nothing here.
    if (flags & ~(DFX_POSTFX_FEATURE_FLAG_REVERSED_DEPTH | DFX_POSTFX_FEATURE_FLAG_TEMPORAL_UPSCALING | DFX_POSTFX_FEATURE_FLAG_HALF_PRECISION_DEPTH))
        return set_error(DFX_ERR_UNSUPPORTED, "unknown PostFX feature flags 0x%x", flags);
    DFX_REQUIRE(!(flags & DFX_POSTFX_FEATURE_FLAG_TEMPORAL_UPSCALING) || (desc->OutputWidth > 0 && desc->OutputHeight > 0),
                "temporal upscaling needs FrameDesc.OutputWidth / OutputHeight");
    DFX_REQUIRE(desc->Width > 0 && desc->Height > 0, "empty frame");
    c->desc  = *desc;
    c->flags = flags;
    if (c->w != (int)desc->Width || c->h != (int)desc->Height)
    {
        c->w = desc->Width, c->h = desc->Height;
        dfx_status st;
        if ((st = c->reproj.alloc(c->w, c->h, DFX_FORMAT_R32F)) != DFX_OK) return st;
        if ((st = c->prev_depth.alloc(c->w, c->h, DFX_FORMAT_R32F)) != DFX_OK) return st;
        if ((st = c->closest.alloc(c->w, c->h, DFX_FORMAT_RG32F)) != DFX_OK) return st;
    }
    // the context's own depth planes carry the encoding of the depth buffer they are derived from (PostFXContext.cpp:515)
    c->reproj.p.flags = c->prev_depth.p.flags = (flags & DFX_POSTFX_FEATURE_FLAG_REVERSED_DEPTH) ? DFX_PLANE_FLAG_REVERSED_DEPTH : 0;
    c->prepared = true;
    return DFX_OK;
}

namespace dfx
{
dfx_status launch_blue_noise(void* stream, const uint8_t* tables, uint32_t frame_index, const uint32_t* frame_index_dev, const dfx_plane* xy, const dfx_plane* zw);
dfx_status launch_upload_cameras(void* stream, const dfx_camera_attribs* curr, const dfx_camera_attribs* prev, uint32_t frame_index, dfx_camera_attribs* dst_cams,
                                 uint32_t* dst_frame);
dfx_status launch_upload_cameras(void* stream, const dfx_camera_attribs* curr, const dfx_camera_attribs* prev, uint32_t frame_index, dfx_camera_attribs* dst_cams,
                                 uint32_t* dst_frame, float elapsed, float* dst_elapsed);
dfx_status launch_update_average_luminance(void* stream, int adapt, int32_t sampling, float dt, const float* dt_dev, const dfx_plane* color, float* state);
dfx_status launch_reset_average_luminance(void* stream, float* state);
}
// upload {curr, prev} like the map-discard of PostFXContext.cpp:310-318, plus the frame index (as kernel parameters: dfx_postfx.cu)
static dfx_status postfx_upload(dfx_postfx* c, cudaStream_t s, const dfx_camera_attribs* curr, const dfx_camera_attribs* prev)
{
    return launch_upload_cameras(s, curr, prev, c->desc.Index, c->cams_dev, c->frame_dev);
}
// the kernels of PostFXContext::Execute (everything they read per frame comes from device memory: the launches can be replayed from a graph)
static dfx_status postfx_launch(dfx_postfx* c, cudaStream_t s, const dfx_plane* curr_depth, const dfx_plane* prev_depth, const dfx_plane* motion)
{
    EffectRange nvtx_range("PreparePostFX");
    dfx_status st;
    if ((st = launch_blue_noise(s, c->tables_dev, c->desc.Index, c->frame_dev, &c->bn_xy.p, &c->bn_zw.p)) != DFX_OK) return st;
    dfx_rows  all{0, c->h};
    dfx_plane depth = *curr_depth;
    depth.flags |= c->reproj.p.flags;
    if ((st = dfx_pass_postfx_prepare(s, c->cams_dev, &depth, prev_depth, motion, &c->reproj.p, &c->closest.p, &c->prev_depth.p, all)) != DFX_OK) return st;
    c->executed = true;
    return DFX_OK;
}

extern "C" dfx_status dfx_postfx_execute(dfx_postfx* c, const dfx_postfx_render_attribs* a)
{
    DFX_REQUIRE(c && a, "null argument");
    if (!c->prepared) return set_error(DFX_ERR_NOT_PREPARED, "dfx_postfx_prepare was not called");
    DFX_REQUIRE(a->curr_depth && a->prev_depth && a->motion_vectors, "depth / motion planes must not be null");
    DFX_REQUIRE(a->curr_camera && a->prev_camera, "camera attribs must not be null");
    cudaStream_t s = as_stream(a->stream);
    dfx_status   st;
    if ((st = postfx_upload(c, s, a->curr_camera, a->prev_camera)) != DFX_OK) return st;
    return postfx_launch(c, s, a->curr_depth, a->prev_depth, a->motion_vectors);
}

extern "C" dfx_status dfx_postfx_get_plane(const dfx_postfx* c, int32_t id, dfx_plane* out)
{
    DFX_REQUIRE(c && out, "null argument");
    switch (id)
    {
        case DFX_POSTFX_PLANE_BLUE_NOISE_XY: *out = c->bn_xy.p; break;
        case DFX_POSTFX_PLANE_BLUE_NOISE_ZW: *out = c->bn_zw.p; break;
        case DFX_POSTFX_PLANE_REPROJECTED_DEPTH: *out = c->reproj.p; break;
        case DFX_POSTFX_PLANE_PREVIOUS_DEPTH: *out = c->prev_depth.p; break;
        case DFX_POSTFX_PLANE_CLOSEST_MOTION: *out = c->closest.p; break;
        default: return set_error(DFX_ERR_INVALID_ARG, "unknown PostFX plane id %d", id);
    }
    DFX_REQUIRE(out->ptr != nullptr, "plane %d is not allocated yet (prepare first)", id);
    return DFX_OK;
}
extern "C" dfx_status dfx_postfx_get_frame_desc(const dfx_postfx* c, dfx_frame_desc* out)
{
    DFX_REQUIRE(c && out, "null argument");
    *out = c->desc;
    return DFX_OK;
}
extern "C" const dfx_camera_attribs* dfx_postfx_get_camera_attribs_dev(const dfx_postfx* c) { return c ? c->cams_dev : nullptr; }

// =====================================================================================================================
// ScreenSpaceAmbientOcclusion
// =====================================================================================================================
struct dfx_ssao
{
    int        w = 0, h = 0, levels = 0;
    uint32_t   flags = 0, last_frame = ~0u, curr_frame = 0;
    bool       prepared = false;
    AlphaTimer alpha;
    PlaneOwner pre[5];      // [0] unused: level 0 aliases the input depth
    PlaneOwner conv_occ[5]; // [0] = accumulated AO (A5 output)
    PlaneOwner conv_depth[5]; // [0] unused: aliases the input depth
    PlaneOwner occ, resampled, hist[2], histlen[2];
    PlaneOwner checker, occ_up; // FEATURE_FLAG_HALF_RESOLUTION: A0 output (prefiltered level 0) and A4 output
    dfx_plane  last_depth{}; // input depth of the last Execute (for get_plane of the aliased levels)
};

extern "C" dfx_status dfx_ssao_create(dfx_ssao** out)
{
    DFX_REQUIRE(out, "out must not be null");
    *out = new (std::nothrow) dfx_ssao;
    DFX_REQUIRE(*out, "out of memory");
    return DFX_OK;
}
extern "C" void dfx_ssao_destroy(dfx_ssao* fx) { delete fx; }
extern "C" dfx_status dfx_ssao_set_alpha_interpolation(dfx_ssao* fx, float alpha)
{
    DFX_REQUIRE(fx, "null argument");
    fx->alpha.pinned  = alpha;
    fx->alpha.started = false;
    return DFX_OK;
}

static int mip_levels_count(int w, int h)
{
    int m = w > h ? w : h, n = 0;
    while (m > 0) ++n, m >>= 1;
    return n;
}

extern "C" dfx_status dfx_ssao_prepare(dfx_ssao* fx, dfx_postfx* postfx, uint32_t flags)
{
    DFX_REQUIRE(fx && postfx, "null argument");
    if (flags & ~(DFX_SSAO_FEATURE_FLAG_HALF_RESOLUTION | DFX_SSAO_FEATURE_FLAG_HALF_PRECISION_DEPTH))
        return set_error(DFX_ERR_UNSUPPORTED, "unknown SSAO feature flags 0x%x", flags);
    if (!postfx->prepared) return set_error(DFX_ERR_NOT_PREPARED, "PostFXContext is not prepared");
    fx->curr_frame = postfx->desc.Index;
    if (fx->w == postfx->w && fx->h == postfx->h && fx->prepared && fx->flags == flags) return DFX_OK;
    // a change of the resolution mode resets the temporal state, like the reference's ResetStateFeatureMask (…cpp:453)
    fx->flags = flags, fx->last_frame = ~0u;
    fx->w = postfx->w, fx->h = postfx->h;
    fx->levels = std::min(mip_levels_count(fx->w, fx->h), 5);
    const bool half = (flags & DFX_SSAO_FEATURE_FLAG_HALF_RESOLUTION) != 0;
    const int  pw = half ? fx->w / 2 : fx->w, ph = half ? fx->h / 2 : fx->h; // prefiltered depth / raw occlusion (…cpp:109-110, :273-274)
    DFX_REQUIRE(pw > 0 && ph > 0, "frame too small for half-resolution SSAO");
    dfx_status st;
    for (int i = 1; i < fx->levels; ++i)
    {
        const int mw = std::max(fx->w >> i, 1), mh = std::max(fx->h >> i, 1);
        if ((st = fx->pre[i].alloc(std::max(pw >> i, 1), std::max(ph >> i, 1), DFX_FORMAT_R32F)) != DFX_OK) return st;
        if ((st = fx->conv_occ[i].alloc(mw, mh, DFX_FORMAT_R32F)) != DFX_OK) return st;
        if ((st = fx->conv_depth[i].alloc(mw, mh, DFX_FORMAT_R32F)) != DFX_OK) return st;
    }
    if (half)
    {
        if ((st = fx->checker.alloc(pw, ph, DFX_FORMAT_R32F)) != DFX_OK) return st;
        if ((st = fx->occ_up.alloc(fx->w, fx->h, DFX_FORMAT_R32F)) != DFX_OK) return st;
    }
    if ((st = fx->conv_occ[0].alloc(fx->w, fx->h, DFX_FORMAT_R32F)) != DFX_OK) return st;
    if ((st = fx->occ.alloc(pw, ph, DFX_FORMAT_R32F)) != DFX_OK) return st;
    if ((st = fx->resampled.alloc(fx->w, fx->h, DFX_FORMAT_R32F)) != DFX_OK) return st;
    for (int i = 0; i < 2; ++i)
    {
        if ((st = fx->hist[i].alloc(fx->w, fx->h, DFX_FORMAT_R32F)) != DFX_OK) return st;
        if ((st = fx->histlen[i].alloc(fx->w, fx->h, DFX_FORMAT_R32F)) != DFX_OK) return st;
        // cleared to 1.0 at creation (…SSAO.cpp:304-305, :320-321)
        if ((st = clear_plane(nullptr, fx->hist[i].p, 1.0f)) != DFX_OK) return st;
        if ((st = clear_plane(nullptr, fx->histlen[i].p, 1.0f)) != DFX_OK) return st;
    }
    DFX_CUDA(cudaStreamSynchronize(nullptr));
    fx->last_frame = ~0u;
    fx->prepared   = true;
    return DFX_OK;
}

extern "C" dfx_status dfx_ssao_execute(dfx_ssao* fx, const dfx_ssao_render_attribs* a)
{
    EffectRange nvtx_range("ScreenSpaceAmbientOcclusion");
    DFX_REQUIRE(fx && a, "null argument");
    if (!fx->prepared) return set_error(DFX_ERR_NOT_PREPARED, "dfx_ssao_prepare was not called");
    DFX_REQUIRE(a->postfx && a->depth && a->normal && a->attribs, "postfx / depth / normal / attribs must not be null");
    dfx_postfx* pfx = a->postfx;
    if (!pfx->executed) return set_error(DFX_ERR_NOT_PREPARED, "PostFXContext::Execute must run before SSAO");
    DFX_REQUIRE(a->depth->width == fx->w && a->depth->height == fx->h, "depth size does not match the prepared frame size");
    cudaStream_t s = as_stream(a->stream);

    // UpdateConstantBuffer (…SSAO.cpp:790-816)
    dfx_ssao_attribs A = *a->attribs;
    const bool reset   = fx->last_frame == ~0u || fx->curr_frame != fx->last_frame + 1u || a->attribs->ResetAccumulation != 0;
    A.ResetAccumulation  = reset ? 1 : 0;
    A.AlphaInterpolation = fx->alpha.value();
    fx->last_frame       = fx->curr_frame;

    const uint32_t cur = fx->curr_frame & 1u, prv = (fx->curr_frame + 1u) & 1u;
    const dfx_rows all{0, fx->h};
    dfx_plane depth = *a->depth; // SSAO_OPTION_INVERTED_DEPTH follows the PostFX feature flag (ScreenSpaceAmbientOcclusion.cpp:72, :471)
    depth.flags |= pfx->reproj.p.flags;
    fx->last_depth = depth;

    dfx_pyramid pre{}, cocc{}, cdep{};
    pre.levels = cocc.levels = cdep.levels = fx->levels;
    const bool half = (fx->flags & DFX_SSAO_FEATURE_FLAG_HALF_RESOLUTION) != 0;
    // HALF_PRECISION_DEPTH: the pyramids stay fp32 (no narrow format is modelled); what the shaders see of the flag is the larger
    // self-occlusion offset of the AO pass, keyed on the plane flag (SSAO_ComputeAmbientOcclusion.fx:145-150)
    if (fx->flags & DFX_SSAO_FEATURE_FLAG_HALF_PRECISION_DEPTH) depth.flags |= DFX_PLANE_FLAG_HALF_PRECISION_DEPTH;
    pre.level[0] = depth, cocc.level[0] = fx->conv_occ[0].p, cdep.level[0] = depth;
    for (int i = 1; i < fx->levels; ++i) pre.level[i] = fx->pre[i].p, cocc.level[i] = fx->conv_occ[i].p, cdep.level[i] = fx->conv_depth[i].p;

    dfx_status st;
    dfx_rows   pre_rows = all;
    if (half)
    {
        // A0, then A1-A3 on the half-size checkerboard (…cpp:818-857); the checkerboard keeps the depth buffer's encoding
        pre_rows = dfx_rows{0, fx->h / 2};
        fx->checker.p.flags = depth.flags;
        if ((st = dfx_pass_ssao_downsample_depth(s, &depth, &fx->checker.p, pre_rows)) != DFX_OK) return st;
        pre.level[0] = fx->checker.p;
    }
    if ((st = dfx_pass_ssao_prefilter_depth(s, pfx->cams_dev, &A, &pre, pre_rows)) != DFX_OK) return st;
    if ((st = dfx_pass_ssao_ambient_occlusion(s, pfx->cams_dev, &A, &pre, a->normal, &pfx->bn_zw.p, &fx->occ.p, pre_rows)) != DFX_OK) return st;
    if (half && (st = dfx_pass_ssao_upsample(s, pfx->cams_dev, &depth, &fx->occ.p, &fx->occ_up.p, all)) != DFX_OK) return st;
    if ((st = dfx_pass_ssao_temporal(s, pfx->cams_dev, &A, half ? &fx->occ_up.p : &fx->occ.p, &fx->hist[prv].p, &fx->histlen[prv].p, &pfx->reproj.p, &pfx->prev_depth.p,
                                     &pfx->closest.p, &fx->conv_occ[0].p, &fx->histlen[cur].p, all)) != DFX_OK)
        return st;
    if ((st = dfx_pass_ssao_convolute(s, &cocc, &cdep, all)) != DFX_OK) return st;
    if ((st = dfx_pass_ssao_resample(s, pfx->cams_dev, &cocc, &cdep, &fx->histlen[cur].p, a->normal, &fx->resampled.p, all)) != DFX_OK) return st;
    if ((st = dfx_pass_ssao_spatial(s, pfx->cams_dev, &A, &fx->resampled.p, &fx->histlen[cur].p, &depth, a->normal, &fx->hist[cur].p, all)) != DFX_OK) return st;
    return DFX_OK;
}

extern "C" dfx_status dfx_ssao_get_plane(const dfx_ssao* fx, int32_t id, dfx_plane* out)
{
    DFX_REQUIRE(fx && out, "null argument");
    if (!fx->prepared) return set_error(DFX_ERR_NOT_PREPARED, "dfx_ssao_prepare was not called");
    const uint32_t cur = fx->curr_frame & 1u;
    if (id == DFX_SSAO_PLANE_OUTPUT) *out = fx->hist[cur].p;
    else if (id == DFX_SSAO_PLANE_OCCLUSION) *out = fx->occ.p;
    else if (id == DFX_SSAO_PLANE_ACCUMULATED) *out = fx->conv_occ[0].p;
    else if (id == DFX_SSAO_PLANE_HISTORY_LENGTH) *out = fx->histlen[cur].p;
    else if (id == DFX_SSAO_PLANE_RESAMPLED) *out = fx->resampled.p;
    else if (id == DFX_SSAO_PLANE_UPSAMPLED) *out = fx->occ_up.p;
    else if (id >= DFX_SSAO_PLANE_PREFILTERED_MIP0 && id < DFX_SSAO_PLANE_PREFILTERED_MIP0 + fx->levels)
        *out = id == DFX_SSAO_PLANE_PREFILTERED_MIP0 ? ((fx->flags & DFX_SSAO_FEATURE_FLAG_HALF_RESOLUTION) ? fx->checker.p : fx->last_depth)
                                                     : fx->pre[id - DFX_SSAO_PLANE_PREFILTERED_MIP0].p;
    else if (id >= DFX_SSAO_PLANE_CONV_AO_MIP0 && id < DFX_SSAO_PLANE_CONV_AO_MIP0 + fx->levels) *out = fx->conv_occ[id - DFX_SSAO_PLANE_CONV_AO_MIP0].p;
    else if (id >= DFX_SSAO_PLANE_CONV_DEPTH_MIP0 && id < DFX_SSAO_PLANE_CONV_DEPTH_MIP0 + fx->levels)
        *out = id == DFX_SSAO_PLANE_CONV_DEPTH_MIP0 ? fx->last_depth : fx->conv_depth[id - DFX_SSAO_PLANE_CONV_DEPTH_MIP0].p;
    else
        return set_error(DFX_ERR_INVALID_ARG, "unknown SSAO plane id %d", id);
    DFX_REQUIRE(out->ptr != nullptr, "plane %d is not available yet", id);
    return DFX_OK;
}

// =====================================================================================================================
// ScreenSpaceReflection
// =====================================================================================================================
struct dfx_ssr
{
    int        w = 0, h = 0, levels = 0;
    uint32_t   flags = 0, curr_frame = 0;
    bool       prepared = false;
    AlphaTimer alpha;
    PlaneOwner hiz[7]; // [0] unused: aliases the input depth
    PlaneOwner roughness, mask, radiance, raydir, res_rad, res_var, res_depth, radhist[2], varhist[2], out;
    PlaneOwner mask_half; // FEATURE_FLAG_HALF_RESOLUTION: S3 output; radiance / raydir are then width/2 x height/2
    dfx_plane  last_depth{};
};

extern "C" dfx_status dfx_ssr_create(dfx_ssr** out)
{
    DFX_REQUIRE(out, "out must not be null");
    *out = new (std::nothrow) dfx_ssr;
    DFX_REQUIRE(*out, "out of memory");
    return DFX_OK;
}
extern "C" void dfx_ssr_destroy(dfx_ssr* fx) { delete fx; }
extern "C" dfx_status dfx_ssr_set_alpha_interpolation(dfx_ssr* fx, float alpha)
{
    DFX_REQUIRE(fx, "null argument");
    fx->alpha.pinned  = alpha;
    fx->alpha.started = false;
    return DFX_OK;
}

extern "C" dfx_status dfx_ssr_prepare(dfx_ssr* fx, dfx_postfx* postfx, uint32_t flags)
{
    DFX_REQUIRE(fx && postfx, "null argument");
    if (flags & ~(DFX_SSR_FEATURE_FLAG_PREVIOUS_FRAME | DFX_SSR_FEATURE_FLAG_HALF_RESOLUTION))
        return set_error(DFX_ERR_UNSUPPORTED, "unknown SSR feature flags 0x%x", flags);
    if (!postfx->prepared) return set_error(DFX_ERR_NOT_PREPARED, "PostFXContext is not prepared");
    fx->curr_frame = postfx->desc.Index;
    const bool half = (flags & DFX_SSR_FEATURE_FLAG_HALF_RESOLUTION) != 0;
    const bool same_mode = ((fx->flags ^ flags) & DFX_SSR_FEATURE_FLAG_HALF_RESOLUTION) == 0;
    fx->flags = flags;
    if (fx->w == postfx->w && fx->h == postfx->h && fx->prepared && same_mode) return DFX_OK;
    fx->w = postfx->w, fx->h = postfx->h;
    const int pw = half ? fx->w / 2 : fx->w, ph = half ? fx->h / 2 : fx->h; // intersect targets (…cpp:201-213)
    DFX_REQUIRE(pw > 0 && ph > 0, "frame too small for half-resolution SSR");
    fx->levels = std::min(mip_levels_count(fx->w, fx->h), 7);
    dfx_status st;
    for (int i = 1; i < fx->levels; ++i)
        if ((st = fx->hiz[i].alloc(std::max(fx->w >> i, 1), std::max(fx->h >> i, 1), DFX_FORMAT_R32F)) != DFX_OK) return st;
    struct { PlaneOwner* p; int fmt; } planes[] = {
        {&fx->roughness, DFX_FORMAT_R32F}, {&fx->mask, DFX_FORMAT_R8U}, {&fx->radiance, DFX_FORMAT_RGBA32F}, {&fx->raydir, DFX_FORMAT_RGBA32F},
        {&fx->res_rad, DFX_FORMAT_RGBA32F}, {&fx->res_var, DFX_FORMAT_R32F}, {&fx->res_depth, DFX_FORMAT_R32F},
        {&fx->radhist[0], DFX_FORMAT_RGBA32F}, {&fx->radhist[1], DFX_FORMAT_RGBA32F}, {&fx->varhist[0], DFX_FORMAT_R32F}, {&fx->varhist[1], DFX_FORMAT_R32F},
        {&fx->out, DFX_FORMAT_RGBA32F}};
    for (auto& pl : planes)
    {
        const bool target = pl.p == &fx->radiance || pl.p == &fx->raydir;
        if ((st = pl.p->alloc(target ? pw : fx->w, target ? ph : fx->h, pl.fmt)) != DFX_OK) return st;
        // history / output are cleared to 0 at creation (ScreenSpaceReflection.cpp:263-264, :279-280, :294-295); the targets the
        // reference never clears (roughness, resolved *) start from zeroed memory here so runs are deterministic.
        DFX_CUDA(cudaMemset2D(pl.p->p.ptr, pl.p->p.pitch_bytes, 0, pl.p->p.pitch_bytes, pl.p->p.height));
    }
    if (half && (st = fx->mask_half.alloc(pw, ph, DFX_FORMAT_R8U)) != DFX_OK) return st;
    fx->prepared = true;
    return DFX_OK;
}

extern "C" dfx_status dfx_ssr_execute(dfx_ssr* fx, const dfx_ssr_render_attribs* a)
{
    EffectRange nvtx_range("ScreenSpaceReflection");
    DFX_REQUIRE(fx && a, "null argument");
    if (!fx->prepared) return set_error(DFX_ERR_NOT_PREPARED, "dfx_ssr_prepare was not called");
    DFX_REQUIRE(a->postfx && a->color && a->depth && a->normal && a->material && a->motion && a->attribs, "all SSR inputs must not be null");
    dfx_postfx* pfx = a->postfx;
    if (!pfx->executed) return set_error(DFX_ERR_NOT_PREPARED, "PostFXContext::Execute must run before SSR");
    DFX_REQUIRE(a->depth->width == fx->w && a->depth->height == fx->h, "depth size does not match the prepared frame size");
    cudaStream_t s = as_stream(a->stream);

    dfx_ssr_attribs A    = *a->attribs; // UpdateConstantBuffer (…cpp:755-776)
    A.AlphaInterpolation = fx->alpha.value();
    const uint32_t cur = fx->curr_frame & 1u, prv = (fx->curr_frame + 1u) & 1u;
    const dfx_rows all{0, fx->h};
    dfx_plane depth = *a->depth; // SSR_OPTION_INVERTED_DEPTH follows the PostFX feature flag (ScreenSpaceReflection.cpp:73, :473)
    depth.flags |= pfx->reproj.p.flags;
    fx->last_depth = depth;

    dfx_pyramid hz{};
    hz.levels   = fx->levels;
    hz.level[0] = depth;
    for (int i = 1; i < fx->levels; ++i) hz.level[i] = fx->hiz[i].p;

    dfx_status st;
    if ((st = dfx_pass_ssr_hiz(s, &hz, all)) != DFX_OK) return st;
    if ((st = dfx_pass_ssr_mask_roughness(s, &A, a->material, &depth, &fx->roughness.p, &fx->mask.p, all)) != DFX_OK) return st;
    const bool half = (fx->flags & DFX_SSR_FEATURE_FLAG_HALF_RESOLUTION) != 0;
    const dfx_rows trows = half ? dfx_rows{0, fx->h / 2} : all;
    if (half && (st = dfx_pass_ssr_downsample_mask(s, &A, &fx->roughness.p, &depth, &fx->mask_half.p, trows)) != DFX_OK) return st;
    if ((st = dfx_pass_ssr_intersect(s, pfx->cams_dev, &A, fx->flags, a->color, a->normal, &fx->roughness.p, half ? &fx->mask_half.p : &fx->mask.p,
                                     &pfx->bn_xy.p, &hz, a->motion, &fx->radiance.p, &fx->raydir.p, trows)) != DFX_OK)
        return st;
    if ((st = dfx_pass_ssr_spatial(s, pfx->cams_dev, &A, &fx->roughness.p, &fx->mask.p, a->normal, &depth, &fx->raydir.p, &fx->radiance.p, &fx->res_rad.p,
                                   &fx->res_var.p, &fx->res_depth.p, all)) != DFX_OK)
        return st;
    if ((st = dfx_pass_ssr_temporal(s, pfx->cams_dev, &A, &fx->mask.p, a->motion, &fx->res_depth.p, &pfx->reproj.p, &fx->res_rad.p, &fx->res_var.p,
                                    &pfx->prev_depth.p, &fx->radhist[prv].p, &fx->varhist[prv].p, &fx->radhist[cur].p, &fx->varhist[cur].p, all)) != DFX_OK)
        return st;
    if ((st = dfx_pass_ssr_bilateral(s, pfx->cams_dev, &A, &fx->mask.p, &depth, a->normal, &fx->roughness.p, &fx->radhist[cur].p, &fx->varhist[cur].p,
                                     &fx->out.p, all)) != DFX_OK)
        return st;
    return DFX_OK;
}

extern "C" dfx_status dfx_ssr_get_plane(const dfx_ssr* fx, int32_t id, dfx_plane* out)
{
    DFX_REQUIRE(fx && out, "null argument");
    if (!fx->prepared) return set_error(DFX_ERR_NOT_PREPARED, "dfx_ssr_prepare was not called");
    const uint32_t cur = fx->curr_frame & 1u;
    switch (id)
    {
        case DFX_SSR_PLANE_OUTPUT: *out = fx->out.p; break;
        case DFX_SSR_PLANE_ROUGHNESS: *out = fx->roughness.p; break;
        case DFX_SSR_PLANE_MASK: *out = fx->mask.p; break;
        case DFX_SSR_PLANE_MASK_HALF: *out = fx->mask_half.p; break;
        case DFX_SSR_PLANE_RADIANCE: *out = fx->radiance.p; break;
        case DFX_SSR_PLANE_RAYDIR_PDF: *out = fx->raydir.p; break;
        case DFX_SSR_PLANE_RESOLVED_RADIANCE: *out = fx->res_rad.p; break;
        case DFX_SSR_PLANE_RESOLVED_VARIANCE: *out = fx->res_var.p; break;
        case DFX_SSR_PLANE_RESOLVED_DEPTH: *out = fx->res_depth.p; break;
        case DFX_SSR_PLANE_RADIANCE_HISTORY: *out = fx->radhist[cur].p; break;
        case DFX_SSR_PLANE_VARIANCE_HISTORY: *out = fx->varhist[cur].p; break;
        default:
            if (id >= DFX_SSR_PLANE_HIZ_MIP0 && id < DFX_SSR_PLANE_HIZ_MIP0 + fx->levels)
                *out = id == DFX_SSR_PLANE_HIZ_MIP0 ? fx->last_depth : fx->hiz[id - DFX_SSR_PLANE_HIZ_MIP0].p;
            else
                return set_error(DFX_ERR_INVALID_ARG, "unknown SSR plane id %d", id);
    }
    DFX_REQUIRE(out->ptr != nullptr, "plane %d is not available yet", id);
    return DFX_OK;
}

// =====================================================================================================================
// Bloom
// =====================================================================================================================
#ifndef DFX_BLOOM_LEVELS_DEFAULT
#define DFX_BLOOM_LEVELS_DEFAULT 0
#endif
struct dfx_bloom
{
    int                     w = 0, h = 0;
    bool                    prepared = false;
    AlphaTimer              alpha;
    std::vector<PlaneOwner> down, up;
    PlaneOwner              out;
    PlaneOwner              levels_ws; // barrier words of dfx_pass_bloom_levels (zero between launches)
};

extern "C" dfx_status dfx_bloom_create(dfx_bloom** out)
{
    DFX_REQUIRE(out, "out must not be null");
    *out = new (std::nothrow) dfx_bloom;
    DFX_REQUIRE(*out, "out of memory");
    return DFX_OK;
}
extern "C" void dfx_bloom_destroy(dfx_bloom* fx) { delete fx; }
extern "C" dfx_status dfx_bloom_set_alpha_interpolation(dfx_bloom* fx, float alpha)
{
    DFX_REQUIRE(fx, "null argument");
    fx->alpha.pinned  = alpha;
    fx->alpha.started = false;
    return DFX_OK;
}

extern "C" dfx_status dfx_bloom_prepare(dfx_bloom* fx, dfx_postfx* postfx, uint32_t flags)
{
    DFX_REQUIRE(fx && postfx, "null argument");
    if (flags != DFX_BLOOM_FEATURE_FLAG_NONE) return set_error(DFX_ERR_UNSUPPORTED, "unknown Bloom feature flags 0x%x", flags);
    if (!postfx->prepared) return set_error(DFX_ERR_NOT_PREPARED, "PostFXContext is not prepared");
    // Bloom runs after the temporal upscaler when there is one: on the OUTPUT resolution of the frame (Bloom.cpp:84-85)
    const bool upscaled = (postfx->flags & DFX_POSTFX_FEATURE_FLAG_TEMPORAL_UPSCALING) != 0;
    const int  bw = upscaled ? (int)postfx->desc.OutputWidth : postfx->w, bh = upscaled ? (int)postfx->desc.OutputHeight : postfx->h;
    if (fx->w == bw && fx->h == bh && fx->prepared) return DFX_OK;
    fx->w = bw, fx->h = bh;
    // Bloom.cpp:96-128: TextureCount = ComputeMipLevelsCount(W/2, H/2), level i = max(half >> i, 1)
    const int hw = std::max(fx->w / 2, 1), hh = std::max(fx->h / 2, 1);
    const int count = mip_levels_count(hw, hh);
    fx->down = std::vector<PlaneOwner>(count);
    fx->up   = std::vector<PlaneOwner>(count);
    dfx_status st;
    for (int i = 0; i < count; ++i)
    {
        if ((st = fx->down[i].alloc(std::max(hw >> i, 1), std::max(hh >> i, 1), DFX_FORMAT_RGBA32F)) != DFX_OK) return st;
        if ((st = fx->up[i].alloc(std::max(hw >> i, 1), std::max(hh >> i, 1), DFX_FORMAT_RGBA32F)) != DFX_OK) return st;
    }
    if ((st = fx->out.alloc(fx->w, fx->h, DFX_FORMAT_RGBA32F)) != DFX_OK) return st;
    if ((st = fx->levels_ws.alloc(16, 1, DFX_FORMAT_R32F)) != DFX_OK) return st;
    DFX_CUDA(cudaMemset(fx->levels_ws.p.ptr, 0, 64));
    fx->prepared = true;
    return DFX_OK;
}

static dfx_status bloom_execute_impl(dfx_bloom* fx, const dfx_bloom_render_attribs* a, const dfx_tonemap_attribs* tonemap, float ave_log_lum,
                                     int32_t to_srgb, const dfx_plane* ldr_out, const float* ave_log_lum_dev = nullptr);

extern "C" dfx_status dfx_bloom_execute(dfx_bloom* fx, const dfx_bloom_render_attribs* a) { return bloom_execute_impl(fx, a, nullptr, 0.0f, 0, nullptr); }

// Bloom followed by the final ToneMap(+sRGB) (HnPostProcessTask.cpp:911-925) with the composite and the tone map fused into
// one kernel: the HDR bloom output never touches HBM (GetBloomTextureSRV() is NOT updated by this call).
extern "C" dfx_status dfx_bloom_execute_tonemapped(dfx_bloom* fx, const dfx_bloom_render_attribs* a, const dfx_tonemap_attribs* tonemap, float ave_log_lum,
                                                   int32_t convert_to_srgb, const dfx_plane* ldr_out)
{
    DFX_REQUIRE(tonemap && ldr_out, "tonemap attribs / output plane must not be null");
    return bloom_execute_impl(fx, a, tonemap, ave_log_lum, convert_to_srgb, ldr_out);
}
// the same with fAveLogLum = max(0.05, *ave_log_lum_dev) (auto exposure: the chain's average-luminance state)
static dfx_status dfx_bloom_execute_tonemapped_dev(dfx_bloom* fx, const dfx_bloom_render_attribs* a, const dfx_tonemap_attribs* tonemap, const float* ave_log_lum_dev,
                                                   int32_t convert_to_srgb, const dfx_plane* ldr_out)
{
    DFX_REQUIRE(tonemap && ldr_out && ave_log_lum_dev, "tonemap attribs / luminance / output plane must not be null");
    return bloom_execute_impl(fx, a, tonemap, 0.0f, convert_to_srgb, ldr_out, ave_log_lum_dev);
}

static dfx_status bloom_execute_impl(dfx_bloom* fx, const dfx_bloom_render_attribs* a, const dfx_tonemap_attribs* tonemap, float ave_log_lum,
                                     int32_t to_srgb, const dfx_plane* ldr_out, const float* ave_log_lum_dev)
{
    EffectRange nvtx_range("Bloom");
    DFX_REQUIRE(fx && a, "null argument");
    if (!fx->prepared) return set_error(DFX_ERR_NOT_PREPARED, "dfx_bloom_prepare was not called");
    DFX_REQUIRE(a->color && a->attribs, "color / attribs must not be null");
    DFX_REQUIRE(a->color->width == fx->w && a->color->height == fx->h, "color size does not match the prepared frame size");
    cudaStream_t      s = as_stream(a->stream);
    dfx_bloom_attribs A = *a->attribs; // UpdateConstantBuffer (Bloom.cpp:270-286)
    A.AlphaInterpolation = fx->alpha.value();

    const int mips = std::min<int>(dfx_bloom_mip_count(fx->down[0].p.width, fx->down[0].p.height, A.Radius), (int)fx->down.size());
    DFX_REQUIRE(mips >= 2, "Bloom radius %.3f leaves fewer than two pyramid levels", A.Radius);
    auto rows = [](const dfx_plane& p) { return dfx_rows{0, p.height}; };
    dfx_status st;
    // The reference draws one level per pass (Bloom.cpp:324-337 down, :355-375 up), and by default so does this: under async compute
    // the small per-level launches interleave with the next frame's front half, and the frame is fastest that way (profiles/r2k1,
    // r2j). Two fused forms exist and win as isolated passes: dfx_tune "bloom_tail" = 1 (the levels of <= 2K texels, down and up, in one
    // thread-block-cluster launch) and "bloom_levels" = 1 (every level after the prefilter in one cooperative launch over the GPU).
    dfx_plane down[DFX_BLOOM_MAX_LEVELS], up[DFX_BLOOM_MAX_LEVELS];
    DFX_REQUIRE(mips <= DFX_BLOOM_MAX_LEVELS, "too many Bloom levels");
    for (int i = 0; i < mips; ++i) down[i] = fx->down[i].p, up[i] = fx->up[i].p;
    if ((st = dfx_pass_bloom_prefilter(s, &A, a->color, &down[0], rows(down[0]))) != DFX_OK) return st;
    if (dfx_tune_get("bloom_levels", DFX_BLOOM_LEVELS_DEFAULT))
    {
        if ((st = dfx_pass_bloom_levels(s, down, up, 1, mips, fx->levels_ws.p.ptr)) != DFX_OK) return st;
    }
    else
    {
        const int first = dfx_bloom_tail_first_level(down, mips);
        for (int i = 1; i < first; ++i)
            if ((st = dfx_pass_bloom_downsample(s, &down[i - 1], &down[i], rows(down[i]))) != DFX_OK) return st;
        if (first < mips && (st = dfx_pass_bloom_tail(s, down, up, first, mips)) != DFX_OK) return st;
        const int top = mips - 1;
        for (int i = std::min(top, first - 1); i > 0; --i)
            if ((st = dfx_pass_bloom_upsample(s, &down[i - 1], i != top ? &up[i] : &down[i], &up[i - 1], rows(up[i - 1]))) != DFX_OK) return st;
    }
    if (tonemap)
    {
        const dfx_plane& u0 = fx->up[0].p;
        if (fx->w == 2 * u0.width && fx->h == 2 * u0.height)
            return ave_log_lum_dev ? dfx_pass_bloom_composite_tonemap_dev(s, &A, tonemap, ave_log_lum_dev, to_srgb, a->color, &u0, ldr_out, rows(fx->out.p))
                                   : dfx_pass_bloom_composite_tonemap(s, &A, tonemap, ave_log_lum, to_srgb, a->color, &u0, ldr_out, rows(fx->out.p));
        if ((st = dfx_pass_bloom_composite(s, &A, a->color, &u0, &fx->out.p, rows(fx->out.p))) != DFX_OK) return st;
        return ave_log_lum_dev ? dfx_pass_tonemap_dev(s, tonemap, ave_log_lum_dev, to_srgb, &fx->out.p, ldr_out, rows(fx->out.p))
                               : dfx_pass_tonemap(s, tonemap, ave_log_lum, to_srgb, &fx->out.p, ldr_out, rows(fx->out.p));
    }
    return dfx_pass_bloom_composite(s, &A, a->color, &fx->up[0].p, &fx->out.p, rows(fx->out.p));
}

extern "C" dfx_status dfx_bloom_get_plane(const dfx_bloom* fx, int32_t id, dfx_plane* out)
{
    DFX_REQUIRE(fx && out, "null argument");
    if (!fx->prepared) return set_error(DFX_ERR_NOT_PREPARED, "dfx_bloom_prepare was not called");
    const int n = (int)fx->down.size();
    if (id == DFX_BLOOM_PLANE_OUTPUT) *out = fx->out.p;
    else if (id >= DFX_BLOOM_PLANE_DOWN0 && id < DFX_BLOOM_PLANE_DOWN0 + n) *out = fx->down[id - DFX_BLOOM_PLANE_DOWN0].p;
    else if (id >= DFX_BLOOM_PLANE_UP0 && id < DFX_BLOOM_PLANE_UP0 + n) *out = fx->up[id - DFX_BLOOM_PLANE_UP0].p;
    else
        return set_error(DFX_ERR_INVALID_ARG, "unknown Bloom plane id %d", id);
    return DFX_OK;
}

// =====================================================================================================================
// TemporalAntiAliasing
// =====================================================================================================================
struct TaaBuffer
{
    int        w = 0, h = 0;
    uint32_t   flags = 0, last_frame = ~0u, curr_frame = 0;
    PlaneOwner accum[2];
};
struct dfx_taa
{
    std::map<uint32_t, TaaBuffer> buffers;
};

extern "C" dfx_status dfx_taa_create(dfx_taa** out)
{
    DFX_REQUIRE(out, "out must not be null");
    *out = new (std::nothrow) dfx_taa;
    DFX_REQUIRE(*out, "out of memory");
    return DFX_OK;
}
extern "C" void dfx_taa_destroy(dfx_taa* fx) { delete fx; }

extern "C" dfx_status dfx_taa_prepare(dfx_taa* fx, dfx_postfx* postfx, uint32_t flags, uint32_t idx)
{
    DFX_REQUIRE(fx && postfx, "null argument");
    if (flags & ~7u) return set_error(DFX_ERR_UNSUPPORTED, "unknown TAA feature flags 0x%x", flags);
    if (!postfx->prepared) return set_error(DFX_ERR_NOT_PREPARED, "PostFXContext is not prepared");
    TaaBuffer& b = fx->buffers[idx];
    b.flags      = flags;
    b.curr_frame = postfx->desc.Index;
    if (b.w == postfx->w && b.h == postfx->h) return DFX_OK;
    b.w = postfx->w, b.h = postfx->h;
    dfx_status st;
    for (int i = 0; i < 2; ++i)
    {
        if ((st = b.accum[i].alloc(b.w, b.h, DFX_FORMAT_RGBA32F)) != DFX_OK) return st;
        DFX_CUDA(cudaMemset2D(b.accum[i].p.ptr, b.accum[i].p.pitch_bytes, 0, b.accum[i].p.pitch_bytes, b.h)); // cleared to 0 (TemporalAntiAliasing.cpp:112-116)
    }
    b.last_frame = ~0u;
    return DFX_OK;
}

static dfx_status taa_execute_impl(dfx_taa* fx, const dfx_taa_render_attribs* a, bool compose, const dfx_plane* ssr, const dfx_plane* ao, float ssr_scale,
                                   float ssao_scale);

extern "C" dfx_status dfx_taa_execute(dfx_taa* fx, const dfx_taa_render_attribs* a) { return taa_execute_impl(fx, a, false, nullptr, nullptr, 0.0f, 0.0f); }

// TAA with the compose step (HnPostProcessTask.cpp:834-895) evaluated on the fly: attribs->color is the UN-composed scene colour.
extern "C" dfx_status dfx_taa_execute_composed(dfx_taa* fx, const dfx_taa_render_attribs* a, const dfx_plane* ssr, const dfx_plane* ao, float ssr_scale,
                                               float ssao_scale)
{
    return taa_execute_impl(fx, a, true, ssr, ao, ssr_scale, ssao_scale);
}

static dfx_status taa_execute_impl(dfx_taa* fx, const dfx_taa_render_attribs* a, bool compose, const dfx_plane* ssr, const dfx_plane* ao, float ssr_scale,
                                   float ssao_scale)
{
    DFX_REQUIRE(fx && a, "null argument");
    DFX_REQUIRE(a->postfx && a->color && a->attribs, "postfx / color / attribs must not be null");
    auto it = fx->buffers.find(a->accumulation_buffer_idx);
    if (it == fx->buffers.end())
        return set_error(DFX_ERR_NOT_PREPARED, "Accumulation buffer with index %u is not found, which indicates that PrepareResources() method was not called.",
                         a->accumulation_buffer_idx);
    TaaBuffer&  b   = it->second;
    dfx_postfx* pfx = a->postfx;
    if (!pfx->executed) return set_error(DFX_ERR_NOT_PREPARED, "PostFXContext::Execute must run before TAA");
    DFX_REQUIRE(a->color->width == b.w && a->color->height == b.h, "color size does not match the prepared frame size");

    // AccumulationBufferInfo::UpdateConstantBuffer (TemporalAntiAliasing.cpp:123-141)
    dfx_taa_attribs A  = *a->attribs;
    const bool reset   = b.last_frame == ~0u || b.curr_frame != b.last_frame + 1u || a->attribs->ResetAccumulation != 0;
    A.ResetAccumulation = reset ? 1 : 0;
    b.last_frame        = b.curr_frame;
    const uint32_t cur = b.curr_frame & 1u, prv = (b.curr_frame + 1u) & 1u;
    if (compose)
        return dfx_pass_compose_taa(as_stream(a->stream), pfx->cams_dev, &A, b.flags, a->color, ssr, ao, ssr_scale, ssao_scale, &b.accum[prv].p, &pfx->closest.p,
                                    &pfx->reproj.p, &pfx->prev_depth.p, &b.accum[cur].p, dfx_rows{0, b.h});
    return dfx_pass_taa(as_stream(a->stream), pfx->cams_dev, &A, b.flags, a->color, &b.accum[prv].p, &pfx->closest.p, &pfx->reproj.p, &pfx->prev_depth.p,
                        &b.accum[cur].p, dfx_rows{0, b.h});
}

extern "C" dfx_status dfx_taa_get_plane(const dfx_taa* fx, int32_t id, uint32_t idx, dfx_plane* out)
{
    DFX_REQUIRE(fx && out, "null argument");
    auto it = fx->buffers.find(idx);
    if (it == fx->buffers.end()) return set_error(DFX_ERR_NOT_PREPARED, "Accumulation buffer with index %u is not found.", idx);
    const TaaBuffer& b = it->second;
    // GetAccumulatedFrameSRV (TemporalAntiAliasing.cpp:203-214)
    if (id == DFX_TAA_PLANE_ACCUMULATED_CURR) *out = b.accum[b.curr_frame & 1u].p;
    else if (id == DFX_TAA_PLANE_ACCUMULATED_PREV) *out = b.accum[(b.curr_frame + 1u) & 1u].p;
    else
        return set_error(DFX_ERR_INVALID_ARG, "unknown TAA plane id %d", id);
    return DFX_OK;
}

extern "C" dfx_status dfx_taa_get_jitter_offset(const dfx_taa* fx, uint32_t idx, float out[2])
{
    DFX_REQUIRE(fx && out, "null argument");
    out[0] = out[1] = 0.0f;
    auto it = fx->buffers.find(idx);
    if (it == fx->buffers.end() || it->second.w == 0 || it->second.h == 0) return DFX_OK; // TemporalAntiAliasing.cpp:65-72
    dfx_taa_jitter_offset(it->second.curr_frame, it->second.w, it->second.h, out);
    return DFX_OK;
}

// =====================================================================================================================
// DepthOfField (PostProcess/DepthOfField/src/DepthOfField.cpp; interface/DepthOfField.hpp:59-125)
// =====================================================================================================================
struct dfx_dof
{
    int        w = 0, h = 0;
    uint32_t   flags = 0, curr_frame = 0;
    bool       prepared = false;
    AlphaTimer alpha;
    PlaneOwner coc, coc_temporal[2], dilation[4], dilation_tmp, pre[2], bokeh[2], out;
};

extern "C" dfx_status dfx_dof_create(dfx_dof** out)
{
    DFX_REQUIRE(out, "out must not be null");
    *out = new (std::nothrow) dfx_dof;
    DFX_REQUIRE(*out, "out of memory");
    return DFX_OK;
}
extern "C" void dfx_dof_destroy(dfx_dof* fx) { delete fx; }
extern "C" dfx_status dfx_dof_set_alpha_interpolation(dfx_dof* fx, float alpha)
{
    DFX_REQUIRE(fx, "null argument");
    fx->alpha.pinned  = alpha;
    fx->alpha.started = false;
    return DFX_OK;
}

// DepthOfField::PrepareResources (…cpp:152-290)
extern "C" dfx_status dfx_dof_prepare(dfx_dof* fx, dfx_postfx* postfx, uint32_t flags)
{
    DFX_REQUIRE(fx && postfx, "null argument");
    if (flags & ~(DFX_DOF_FEATURE_FLAG_ENABLE_TEMPORAL_SMOOTHING | DFX_DOF_FEATURE_FLAG_ENABLE_KARIS_INVERSE))
        return set_error(DFX_ERR_UNSUPPORTED, "unknown DepthOfField feature flags 0x%x", flags);
    if (!postfx->prepared) return set_error(DFX_ERR_NOT_PREPARED, "PostFXContext is not prepared");
    fx->curr_frame = postfx->desc.Index;
    if (fx->w == postfx->w && fx->h == postfx->h && fx->flags == flags && fx->prepared) return DFX_OK;
    fx->w = postfx->w, fx->h = postfx->h, fx->flags = flags;
    DFX_REQUIRE((fx->w >> 3) > 0 && (fx->h >> 3) > 0, "frame too small for the dilation chain (needs width, height >= 8)");
    dfx_status st;
    if ((st = fx->coc.alloc(fx->w, fx->h, DFX_FORMAT_R32F)) != DFX_OK) return st;
    if (flags & DFX_DOF_FEATURE_FLAG_ENABLE_TEMPORAL_SMOOTHING)
        for (auto& t : fx->coc_temporal)
        {
            if ((st = t.alloc(fx->w, fx->h, DFX_FORMAT_R32F)) != DFX_OK) return st;
            if ((st = clear_plane(nullptr, t.p, 0.0f)) != DFX_OK) return st; // cleared to 0 at creation (…cpp:187-189)
        }
    for (int k = 0; k < 4; ++k)
        if ((st = fx->dilation[k].alloc(fx->w >> k, fx->h >> k, DFX_FORMAT_R32F)) != DFX_OK) return st;
    if ((st = fx->dilation_tmp.alloc(fx->w >> 3, fx->h >> 3, DFX_FORMAT_R32F)) != DFX_OK) return st;
    for (int i = 0; i < 2; ++i)
    {
        if ((st = fx->pre[i].alloc(fx->w / 2, fx->h / 2, DFX_FORMAT_RGBA32F)) != DFX_OK) return st;
        if ((st = fx->bokeh[i].alloc(fx->w / 2, fx->h / 2, DFX_FORMAT_RGBA32F)) != DFX_OK) return st;
    }
    if ((st = fx->out.alloc(fx->w, fx->h, DFX_FORMAT_RGBA32F)) != DFX_OK) return st;
    DFX_CUDA(cudaStreamSynchronize(nullptr));
    fx->prepared = true;
    return DFX_OK;
}

// DepthOfField::Execute (…cpp:292-331)
extern "C" dfx_status dfx_dof_execute(dfx_dof* fx, const dfx_dof_render_attribs* a)
{
    EffectRange nvtx_range("DepthOfField");
    DFX_REQUIRE(fx && a, "null argument");
    if (!fx->prepared) return set_error(DFX_ERR_NOT_PREPARED, "dfx_dof_prepare was not called");
    DFX_REQUIRE(a->postfx && a->color && a->depth && a->attribs, "postfx / color / depth / attribs must not be null");
    dfx_postfx* pfx = a->postfx;
    if (!pfx->executed) return set_error(DFX_ERR_NOT_PREPARED, "PostFXContext::Execute must run before DepthOfField");
    DFX_REQUIRE(a->color->width == fx->w && a->color->height == fx->h, "color size does not match the prepared frame size");
    cudaStream_t    s = as_stream(a->stream);
    dfx_dof_attribs A = *a->attribs; // UpdateConstantBuffers (…cpp:792-818)
    A.AlphaInterpolation = fx->alpha.value();
    const bool     temporal = (fx->flags & DFX_DOF_FEATURE_FLAG_ENABLE_TEMPORAL_SMOOTHING) != 0;
    const uint32_t cur = fx->curr_frame & 1u, prv = (fx->curr_frame + 1u) & 1u;
    const auto     rows = [](const dfx_plane& p) { return dfx_rows{0, p.height}; };
    dfx_status     st;
    if ((st = dfx_pass_dof_coc(s, pfx->cams_dev, &A, a->depth, &fx->coc.p, rows(fx->coc.p))) != DFX_OK) return st;
    const dfx_plane* coc = &fx->coc.p;
    if (temporal)
    {
        if ((st = dfx_pass_dof_temporal_coc(s, pfx->cams_dev, &A, &fx->coc.p, &fx->coc_temporal[prv].p, &pfx->closest.p, &fx->coc_temporal[cur].p,
                                            rows(fx->coc.p))) != DFX_OK)
            return st;
        coc = &fx->coc_temporal[cur].p;
    }
    if ((st = dfx_pass_dof_separated_coc(s, coc, &fx->dilation[0].p, rows(fx->dilation[0].p))) != DFX_OK) return st;
    for (int k = 1; k < 4; ++k)
        if ((st = dfx_pass_dof_dilation(s, &fx->dilation[k - 1].p, &fx->dilation[k].p, rows(fx->dilation[k].p))) != DFX_OK) return st;
    if ((st = dfx_pass_dof_blur_coc(s, &fx->dilation[3].p, 0, &fx->dilation_tmp.p, rows(fx->dilation_tmp.p))) != DFX_OK) return st;
    if ((st = dfx_pass_dof_blur_coc(s, &fx->dilation_tmp.p, 1, &fx->dilation[3].p, rows(fx->dilation[3].p))) != DFX_OK) return st;
    if ((st = dfx_pass_dof_prefilter(s, a->color, coc, &fx->dilation[3].p, &fx->pre[0].p, &fx->pre[1].p, rows(fx->pre[0].p))) != DFX_OK) return st;
    if ((st = dfx_pass_dof_bokeh(s, pfx->cams_dev, &A, fx->flags, 0, &fx->pre[0].p, &fx->pre[1].p, a->color, &fx->bokeh[0].p, &fx->bokeh[1].p,
                                 rows(fx->bokeh[0].p))) != DFX_OK)
        return st;
    if ((st = dfx_pass_dof_bokeh(s, pfx->cams_dev, &A, fx->flags, 1, &fx->bokeh[0].p, &fx->bokeh[1].p, nullptr, &fx->pre[0].p, &fx->pre[1].p,
                                 rows(fx->pre[0].p))) != DFX_OK)
        return st;
    if ((st = dfx_pass_dof_postfilter(s, &fx->pre[0].p, &fx->pre[1].p, &fx->bokeh[0].p, &fx->bokeh[1].p, rows(fx->bokeh[0].p))) != DFX_OK) return st;
    return dfx_pass_dof_combine(s, &A, a->color, &fx->bokeh[0].p, &fx->bokeh[1].p, &fx->out.p, rows(fx->out.p));
}

extern "C" dfx_status dfx_dof_get_plane(const dfx_dof* fx, int32_t id, dfx_plane* out)
{
    DFX_REQUIRE(fx && out, "null argument");
    if (!fx->prepared) return set_error(DFX_ERR_NOT_PREPARED, "dfx_dof_prepare was not called");
    if (id == DFX_DOF_PLANE_OUTPUT) *out = fx->out.p;
    else if (id == DFX_DOF_PLANE_COC) *out = fx->coc.p;
    else if (id == DFX_DOF_PLANE_COC_TEMPORAL) *out = fx->coc_temporal[fx->curr_frame & 1u].p;
    else if (id >= DFX_DOF_PLANE_DILATION_MIP0 && id < DFX_DOF_PLANE_DILATION_MIP0 + 4) *out = fx->dilation[id - DFX_DOF_PLANE_DILATION_MIP0].p;
    else if (id >= DFX_DOF_PLANE_PREFILTERED0 && id < DFX_DOF_PLANE_PREFILTERED0 + 2) *out = fx->pre[id - DFX_DOF_PLANE_PREFILTERED0].p;
    else if (id >= DFX_DOF_PLANE_BOKEH0 && id < DFX_DOF_PLANE_BOKEH0 + 2) *out = fx->bokeh[id - DFX_DOF_PLANE_BOKEH0].p;
    else
        return set_error(DFX_ERR_INVALID_ARG, "unknown DepthOfField plane id %d", id);
    DFX_REQUIRE(out->ptr != nullptr, "plane %d is not available (temporal smoothing off?)", id);
    return DFX_OK;
}

// =====================================================================================================================
// Chain executor: the whole PostProcess chain of one view as ONE call per frame.
//
// Sequence and wiring follow the reference's only in-tree integration, Hydrogent's HnPostProcessTask (Prepare :591-683, Execute
// :743-947): PostFXContext -> SSR -> SSAO -> compose -> TAA -> [DepthOfField] -> Bloom -> ToneMap(+sRGB). What is added here is
// how the launches reach the GPU:
//   * async compute: the SSAO passes run on a second stream beside the SSR passes (they share read-only inputs), and Bloom +
//     ToneMap of frame f run on a third stream beside the front half of frame f+1 (they share only the ping-pong TAA accumulator);
//   * CUDA graphs: in steady state (consecutive frame indices, no history reset, constant attributes) the ~25 launches of the
//     front half and the ~8 of the back half are replayed from two instantiated graphs, cached per (input planes, ping-pong
//     parity, attributes). Everything that changes from frame to frame - both cameras and the frame index - lives in device
//     memory and is refreshed before the replay by a one-block kernel that receives them as launch parameters. A frame that resets a history, the first
//     frames, or a profiling run take the eager path (same kernels, same streams).
// =====================================================================================================================
namespace dfx
{
bool profiling_enabled();
void set_async_compute_hint(bool on);
}

namespace
{
struct GraphPair
{
    cudaGraphExec_t front = nullptr, post = nullptr;
    int             kernels = 0; // kernel nodes of the two graphs: what one replay adds to dfx_launch_count()
};
void append_bytes(std::string& k, const void* p, size_t n) { k.append(static_cast<const char*>(p), n); }
void append_plane(std::string& k, const dfx_plane* p)
{
    static const dfx_plane none{};
    append_bytes(k, p ? p : &none, sizeof(dfx_plane));
}
} // namespace

static_assert(sizeof(dfx_chain_config) == 284, "dfx_chain_config layout (mirrored by diligentfx_b200/capi.py ChainConfigC)");
struct dfx_chain
{
    dfx_chain_config cfg{};
    int              w = 0, h = 0;
    dfx_postfx*      pfx   = nullptr;
    dfx_ssao*        ssao  = nullptr;
    dfx_ssr*         ssr   = nullptr;
    dfx_bloom*       bloom = nullptr;
    dfx_taa*         taa   = nullptr;
    dfx_dof*         dof   = nullptr;
    cudaStream_t     ao_stream = nullptr, post_stream = nullptr, cap_stream = nullptr;
    cudaEvent_t      ev_fork = nullptr, ev_ao_done = nullptr, ev_front_done = nullptr, post_done[2] = {nullptr, nullptr};
    bool             post_pending[2] = {false, false};
    PlaneOwner       composed;
    float*           lum_state = nullptr; // average-luminance state of auto exposure (DFX_AVERAGE_LUMINANCE_STATE_FLOATS, dfx_exposure.cu)
    float            elapsed   = 0.0f;    // dfx_chain_set_elapsed_time
    uint32_t         last_frame = ~0u;
    bool             graphs_ok  = true;
    std::map<std::string, GraphPair> graphs;
    dfx_chain_stats  stats{};

    void drop_graphs()
    {
        for (auto& g : graphs)
        {
            if (g.second.front) cudaGraphExecDestroy(g.second.front);
            if (g.second.post) cudaGraphExecDestroy(g.second.post);
        }
        graphs.clear();
    }
    ~dfx_chain()
    {
        cudaDeviceSynchronize();
        drop_graphs();
        dfx_dof_destroy(dof), dfx_taa_destroy(taa), dfx_bloom_destroy(bloom), dfx_ssr_destroy(ssr), dfx_ssao_destroy(ssao), dfx_postfx_destroy(pfx);
        for (cudaEvent_t e : {ev_fork, ev_ao_done, ev_front_done, post_done[0], post_done[1]})
            if (e) cudaEventDestroy(e);
        for (cudaStream_t s : {ao_stream, post_stream, cap_stream})
            if (s) cudaStreamDestroy(s);
        cudaFree(lum_state);
    }
};

extern "C" void dfx_chain_config_default(dfx_chain_config* c)
{
    if (!c) return;
    memset(c, 0, sizeof(*c));
    dfx_ssao_attribs_default(&c->ssao), dfx_ssr_attribs_default(&c->ssr), dfx_bloom_attribs_default(&c->bloom), dfx_taa_attribs_default(&c->taa);
    dfx_tonemap_attribs_default(&c->tonemap), dfx_dof_attribs_default(&c->dof);
    c->taa_flags   = DFX_TAA_FEATURE_FLAG_BICUBIC_FILTER; // Hydrogent default (HnPostProcessTask.hpp:109)
    c->stages      = DFX_CHAIN_STAGE_ALL;
    c->fuse        = 1;
    c->overlap     = 1;
    c->use_graph   = 1;
    c->to_srgb     = 1;
    c->ave_log_lum = 0.3f; // HnPostProcessTask.hpp:88, fExposure 0
    c->ssr_scale = c->ssao_scale = 1.0f;
}

extern "C" dfx_status dfx_chain_create(int32_t width, int32_t height, const dfx_chain_config* config, dfx_chain** out)
{
    DFX_REQUIRE(out && width > 0 && height > 0, "bad arguments");
    dfx_chain* c = new (std::nothrow) dfx_chain;
    DFX_REQUIRE(c, "out of memory");
    c->w = width, c->h = height;
    if (config)
        c->cfg = *config;
    else
        dfx_chain_config_default(&c->cfg);
    dfx_status st = DFX_OK;
    if (st == DFX_OK) st = dfx_postfx_create(&c->pfx);
    if (st == DFX_OK) st = dfx_ssao_create(&c->ssao);
    if (st == DFX_OK) st = dfx_ssr_create(&c->ssr);
    if (st == DFX_OK) st = dfx_bloom_create(&c->bloom);
    if (st == DFX_OK) st = dfx_taa_create(&c->taa);
    if (st == DFX_OK) st = dfx_dof_create(&c->dof);
    cudaError_t e = cudaSuccess;
    for (cudaStream_t* s : {&c->ao_stream, &c->post_stream, &c->cap_stream})
        if (e == cudaSuccess) e = cudaStreamCreateWithFlags(s, cudaStreamNonBlocking);
    for (cudaEvent_t* ev : {&c->ev_fork, &c->ev_ao_done, &c->ev_front_done, &c->post_done[0], &c->post_done[1]})
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(ev, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaMalloc((void**)&c->lum_state, DFX_AVERAGE_LUMINANCE_STATE_FLOATS * sizeof(float));
    if (st == DFX_OK && e != cudaSuccess) st = check_cuda(e, "dfx_chain_create");
    if (st == DFX_OK) st = launch_reset_average_luminance(c->post_stream, c->lum_state);
    if (st == DFX_OK && (e = cudaStreamSynchronize(c->post_stream)) != cudaSuccess) st = check_cuda(e, "dfx_chain_create");
    if (st != DFX_OK)
    {
        delete c;
        return st;
    }
    *out = c;
    return DFX_OK;
}
extern "C" void dfx_chain_destroy(dfx_chain* c) { delete c; }

extern "C" dfx_status dfx_chain_set_config(dfx_chain* c, const dfx_chain_config* config)
{
    DFX_REQUIRE(c && config, "null argument");
    // The graph cache is keyed by the configuration bytes, so a change of attribute values just stops hitting the old entries. A
    // change of feature flags or stages, however, makes the effects re-create their planes: every recorded graph then points at
    // freed memory and must go.
    const dfx_chain_config& o = c->cfg;
    const bool realloc = o.postfx_flags != config->postfx_flags || o.ssao_flags != config->ssao_flags || o.ssr_flags != config->ssr_flags || o.taa_flags != config->taa_flags ||
                         o.dof_flags != config->dof_flags || o.enable_dof != config->enable_dof || o.stages != config->stages || o.fuse != config->fuse;
    if (realloc || c->graphs.size() > 16)
    {
        DFX_CUDA(cudaDeviceSynchronize()); // a graph that is still executing must not be destroyed
        c->drop_graphs();
    }
    c->cfg = *config;
    return DFX_OK;
}
extern "C" dfx_status dfx_chain_get_config(const dfx_chain* c, dfx_chain_config* out)
{
    DFX_REQUIRE(c && out, "null argument");
    *out = c->cfg;
    return DFX_OK;
}
extern "C" void* dfx_chain_effect(dfx_chain* c, int32_t which)
{
    if (!c) return nullptr;
    switch (which)
    {
        case DFX_CHAIN_EFFECT_POSTFX: return c->pfx;
        case DFX_CHAIN_EFFECT_SSAO: return c->ssao;
        case DFX_CHAIN_EFFECT_SSR: return c->ssr;
        case DFX_CHAIN_EFFECT_BLOOM: return c->bloom;
        case DFX_CHAIN_EFFECT_TAA: return c->taa;
        case DFX_CHAIN_EFFECT_DOF: return c->dof;
        default: return nullptr;
    }
}
extern "C" void* dfx_chain_post_stream(dfx_chain* c) { return c ? c->post_stream : nullptr; }
extern "C" dfx_status dfx_chain_set_elapsed_time(dfx_chain* c, float seconds)
{
    DFX_REQUIRE(c, "null argument");
    DFX_REQUIRE(seconds >= 0.0f && seconds < INFINITY, "elapsed time must be finite and >= 0 (got %g)", seconds);
    c->elapsed = seconds;
    return DFX_OK;
}
extern "C" const float* dfx_chain_average_luminance_dev(const dfx_chain* c) { return c ? c->lum_state : nullptr; }
extern "C" dfx_status dfx_chain_get_stats(const dfx_chain* c, dfx_chain_stats* out)
{
    DFX_REQUIRE(c && out, "null argument");
    *out = c->stats;
    return DFX_OK;
}

// Makes `stream` wait for the Bloom + ToneMap work that dfx_chain_execute(defer_post = 1) left running on the chain's own stream.
extern "C" dfx_status dfx_chain_join(dfx_chain* c, void* stream)
{
    DFX_REQUIRE(c, "null argument");
    for (int i = 0; i < 2; ++i)
        if (c->post_pending[i]) DFX_CUDA(cudaStreamWaitEvent(as_stream(stream), c->post_done[i], 0));
    return DFX_OK;
}

namespace
{
struct FrameCtx
{
    dfx_chain*             c;
    const dfx_chain_frame* f;
    uint32_t               st;
    bool                   side_ao, side_post, fuse_compose, fuse_tonemap, with_dof;
    bool                   exposure, reset_lum; // auto exposure this frame; restart its state at 0.1 first (histories reset)
};

// PostFX .. TAA [.. DoF] on `s` (the SSAO passes fork to the chain's second stream and join before the compose). `*color_out` = what Bloom reads.
dfx_status record_front(const FrameCtx& x, cudaStream_t s, dfx_plane* color_out)
{
    dfx_chain*             c   = x.c;
    const dfx_chain_frame* f   = x.f;
    const dfx_chain_config& cfg = c->cfg;
    dfx_status             st;
    if (x.st & DFX_CHAIN_STAGE_POSTFX)
        if ((st = postfx_launch(c->pfx, s, f->depth, f->prev_depth, f->motion)) != DFX_OK) return st;
    if (x.side_ao)
    {
        DFX_CUDA(cudaEventRecord(c->ev_fork, s));
        DFX_CUDA(cudaStreamWaitEvent(c->ao_stream, c->ev_fork, 0));
    }
    if (x.st & DFX_CHAIN_STAGE_SSR)
    {
        dfx_ssr_render_attribs a{s, c->pfx, f->color, f->depth, f->normal, f->material, f->motion, &cfg.ssr};
        if ((st = dfx_ssr_execute(c->ssr, &a)) != DFX_OK) return st;
    }
    if (x.st & DFX_CHAIN_STAGE_SSAO)
    {
        dfx_ssao_render_attribs a{x.side_ao ? c->ao_stream : s, c->pfx, f->depth, f->normal, &cfg.ssao};
        if ((st = dfx_ssao_execute(c->ssao, &a)) != DFX_OK) return st;
    }
    if (x.side_ao)
    {
        DFX_CUDA(cudaEventRecord(c->ev_ao_done, c->ao_stream));
        DFX_CUDA(cudaStreamWaitEvent(s, c->ev_ao_done, 0));
    }
    dfx_plane        color = *f->color, ssr_out{}, ao_out{};
    const dfx_plane *pssr = nullptr, *pao = nullptr;
    if (x.st & DFX_CHAIN_STAGE_COMPOSE)
    {
        if (x.st & DFX_CHAIN_STAGE_SSR)
        {
            if ((st = dfx_ssr_get_plane(c->ssr, DFX_SSR_PLANE_OUTPUT, &ssr_out)) != DFX_OK) return st;
            pssr = &ssr_out;
        }
        if (x.st & DFX_CHAIN_STAGE_SSAO)
        {
            if ((st = dfx_ssao_get_plane(c->ssao, DFX_SSAO_PLANE_OUTPUT, &ao_out)) != DFX_OK) return st;
            pao = &ao_out;
        }
        if (!x.fuse_compose)
        {
            if ((st = dfx_pass_compose(s, &color, pssr, pao, cfg.ssr_scale, cfg.ssao_scale, &c->composed.p, dfx_rows{0, c->h})) != DFX_OK) return st;
            color = c->composed.p;
        }
    }
    if (x.st & DFX_CHAIN_STAGE_TAA)
    {
        dfx_taa_render_attribs a{s, c->pfx, &color, &cfg.taa, 0};
        st = x.fuse_compose ? dfx_taa_execute_composed(c->taa, &a, pssr, pao, cfg.ssr_scale, cfg.ssao_scale) : dfx_taa_execute(c->taa, &a);
        if (st != DFX_OK) return st;
        if ((st = dfx_taa_get_plane(c->taa, DFX_TAA_PLANE_ACCUMULATED_CURR, 0, &color)) != DFX_OK) return st;
    }
    if (x.with_dof)
    {
        dfx_dof_render_attribs a{s, c->pfx, &color, f->depth, &cfg.dof};
        if ((st = dfx_dof_execute(c->dof, &a)) != DFX_OK) return st;
        if ((st = dfx_dof_get_plane(c->dof, DFX_DOF_PLANE_OUTPUT, &color)) != DFX_OK) return st;
    }
    *color_out = color;
    return DFX_OK;
}

// Bloom + ToneMap(+sRGB) on `s`
dfx_status record_post(const FrameCtx& x, cudaStream_t s, dfx_plane color)
{
    dfx_chain*              c   = x.c;
    const dfx_chain_config& cfg = c->cfg;
    dfx_status              st;
    if (x.exposure)
    {
        // the scene luminance of the plane Bloom receives, measured and adapted before the composite reads it (EpipolarLightScattering.cpp:
        // 2463-2481); the elapsed time is the word of this frame's parity that the camera upload wrote
        if (x.reset_lum && (st = launch_reset_average_luminance(s, c->lum_state)) != DFX_OK) return st;
        const float* dt_dev = reinterpret_cast<const float*>(c->pfx->frame_dev) + 1 + (x.f->frame_index & 1u);
        if ((st = launch_update_average_luminance(s, cfg.tonemap.bLightAdaptation != 0, cfg.auto_exposure, 0.0f, dt_dev, &color, c->lum_state)) != DFX_OK) return st;
    }
    if (x.st & DFX_CHAIN_STAGE_BLOOM)
    {
        dfx_bloom_render_attribs a{s, c->pfx, &color, &cfg.bloom};
        if (x.fuse_tonemap && x.exposure) return dfx_bloom_execute_tonemapped_dev(c->bloom, &a, &cfg.tonemap, c->lum_state, cfg.to_srgb, x.f->ldr_out);
        if (x.fuse_tonemap) return dfx_bloom_execute_tonemapped(c->bloom, &a, &cfg.tonemap, cfg.ave_log_lum, cfg.to_srgb, x.f->ldr_out);
        if ((st = dfx_bloom_execute(c->bloom, &a)) != DFX_OK) return st;
        if ((st = dfx_bloom_get_plane(c->bloom, DFX_BLOOM_PLANE_OUTPUT, &color)) != DFX_OK) return st;
    }
    if ((x.st & DFX_CHAIN_STAGE_TONEMAP) && x.exposure)
        return dfx_pass_tonemap_dev(s, &cfg.tonemap, c->lum_state, cfg.to_srgb, &color, x.f->ldr_out, dfx_rows{0, c->h});
    if (x.st & DFX_CHAIN_STAGE_TONEMAP) return dfx_pass_tonemap(s, &cfg.tonemap, cfg.ave_log_lum, cfg.to_srgb, &color, x.f->ldr_out, dfx_rows{0, c->h});
    return DFX_OK;
}

// what TAA's output plane will be for this frame (needed by the replay path, which never calls record_front)
bool alpha_constant(AlphaTimer& a) { return a.pinned >= 0.0f || a.value() >= 1.0f; }
} // namespace

extern "C" dfx_status dfx_chain_execute(dfx_chain* c, void* stream, const dfx_chain_frame* f)
{
    DFX_REQUIRE(c && f, "null argument");
    DFX_REQUIRE(f->curr_camera && f->prev_camera, "camera attribs must not be null");
    DFX_REQUIRE(f->depth && f->prev_depth && f->motion && f->normal && f->color && f->material, "all six G-buffer planes must be given");
    const dfx_chain_config& cfg = c->cfg;
    const uint32_t          st  = cfg.stages;
    DFX_REQUIRE(!(st & (DFX_CHAIN_STAGE_TONEMAP)) || f->ldr_out, "the tone-mapped output plane must be given");
    cudaStream_t main = as_stream(stream);
    FrameCtx     x{c, f, st, false, false, false, false, false, false, false};
    DFX_REQUIRE(cfg.auto_exposure >= 0 && cfg.auto_exposure <= DFX_LUMINANCE_SAMPLING_FULL, "unknown auto_exposure mode %d", cfg.auto_exposure);
    // auto exposure is opt-in: the default configuration carries the reference's bAutoExposure = TRUE, and the constant ave_log_lum
    // stays what a chain computes unless auto_exposure asks for the measurement
    x.exposure  = cfg.auto_exposure != 0 && cfg.tonemap.bAutoExposure != 0 && (st & DFX_CHAIN_STAGE_TONEMAP);
    x.reset_lum = c->last_frame == ~0u || f->frame_index != c->last_frame + 1u; // the histories' reset rule (SURVEY.md §8b)
    x.with_dof     = cfg.enable_dof != 0;
    x.side_ao      = cfg.overlap && (st & DFX_CHAIN_STAGE_SSAO) && (st & DFX_CHAIN_STAGE_SSR);
    x.side_post    = cfg.overlap && (st & DFX_CHAIN_STAGE_BLOOM) && (st & DFX_CHAIN_STAGE_TAA) && !x.with_dof;
    x.fuse_compose = cfg.fuse && (st & DFX_CHAIN_STAGE_COMPOSE) && (st & DFX_CHAIN_STAGE_TAA);
    x.fuse_tonemap = cfg.fuse && (st & DFX_CHAIN_STAGE_BLOOM) && (st & DFX_CHAIN_STAGE_TONEMAP) && (c->w % 2 == 0) && (c->h % 2 == 0);
    // launch shapes that depend on whether the two halves of the frame share the GPU (dfx_pyramid.cuh: build_pyramid) read this while
    // the frame is issued or recorded; it is part of the graph key through cfg.overlap
    struct AsyncHint
    {
        explicit AsyncHint(bool on) { set_async_compute_hint(on); }
        ~AsyncHint() { set_async_compute_hint(false); }
    } async_hint(x.side_ao);

    // ---- Prepare (HnPostProcessTask.cpp:671-683): host bookkeeping; allocates on the first frame / on a size change
    dfx_status     s;
    dfx_frame_desc desc{f->frame_index, (uint32_t)c->w, (uint32_t)c->h, (uint32_t)c->w, (uint32_t)c->h};
    if ((s = dfx_postfx_prepare(c->pfx, &desc, cfg.postfx_flags)) != DFX_OK) return s;
    if ((st & DFX_CHAIN_STAGE_SSAO) && (s = dfx_ssao_prepare(c->ssao, c->pfx, cfg.ssao_flags)) != DFX_OK) return s;
    if ((st & DFX_CHAIN_STAGE_SSR) && (s = dfx_ssr_prepare(c->ssr, c->pfx, cfg.ssr_flags)) != DFX_OK) return s;
    if ((st & DFX_CHAIN_STAGE_TAA) && (s = dfx_taa_prepare(c->taa, c->pfx, cfg.taa_flags, 0)) != DFX_OK) return s;
    if ((st & DFX_CHAIN_STAGE_BLOOM) && (s = dfx_bloom_prepare(c->bloom, c->pfx, 0)) != DFX_OK) return s;
    if (x.with_dof && (s = dfx_dof_prepare(c->dof, c->pfx, cfg.dof_flags)) != DFX_OK) return s;
    if ((st & DFX_CHAIN_STAGE_COMPOSE) && !x.fuse_compose && !c->composed.p.ptr && (s = c->composed.alloc(c->w, c->h, DFX_FORMAT_RGBA32F)) != DFX_OK) return s;

    // ---- can this frame be replayed from a graph?
    const uint32_t par    = f->frame_index & 1u;
    bool           steady = cfg.use_graph && c->graphs_ok && !profiling_enabled() && c->last_frame != ~0u && f->frame_index == c->last_frame + 1u;
    if (steady && (st & DFX_CHAIN_STAGE_SSAO))
        steady = c->ssao->last_frame != ~0u && c->ssao->curr_frame == c->ssao->last_frame + 1u && !cfg.ssao.ResetAccumulation && alpha_constant(c->ssao->alpha);
    if (steady && (st & DFX_CHAIN_STAGE_SSR)) steady = alpha_constant(c->ssr->alpha);
    if (steady && (st & DFX_CHAIN_STAGE_BLOOM)) steady = alpha_constant(c->bloom->alpha);
    if (steady && x.with_dof) steady = alpha_constant(c->dof->alpha);
    if (steady && (st & DFX_CHAIN_STAGE_TAA))
    {
        const TaaBuffer& b = c->taa->buffers[0];
        steady             = b.last_frame != ~0u && b.curr_frame == b.last_frame + 1u && !cfg.taa.ResetAccumulation;
    }

    // ---- TAA of this frame overwrites the accumulator that Bloom of frame f-2 read on the chain's third stream
    if (c->post_pending[par])
    {
        DFX_CUDA(cudaStreamWaitEvent(main, c->post_done[par], 0));
        c->post_pending[par] = false;
    }
    // ---- cameras + frame index -> device memory (kernel parameters, no copy engine; outside the recorded graphs: they change every frame)
    // the elapsed time goes to the word of this frame's parity: Bloom + ToneMap of the previous frame may still read the other one
    // on the chain's third stream (the wait on post_done[par] above orders the frame before last)
    if (((st & DFX_CHAIN_STAGE_POSTFX) || x.exposure) &&
        (s = launch_upload_cameras(main, f->curr_camera, f->prev_camera, f->frame_index, c->pfx->cams_dev, c->pfx->frame_dev, c->elapsed,
                                   reinterpret_cast<float*>(c->pfx->frame_dev) + 1 + par)) != DFX_OK)
        return s;

    dfx_plane color{};
    bool      replayed = false;
    if (steady)
    {
        std::string key;
        key.reserve(1024);
        append_bytes(key, &par, sizeof(par));
        append_bytes(key, &cfg, sizeof(cfg));
        for (const dfx_plane* p : {f->depth, f->prev_depth, f->motion, f->normal, f->color, f->material, f->ldr_out}) append_plane(key, p);
        const float alphas[4] = {c->ssao->alpha.value(), c->ssr->alpha.value(), c->bloom->alpha.value(), c->dof->alpha.value()};
        append_bytes(key, alphas, sizeof(alphas));
        GraphPair& g = c->graphs[key];
        if (!g.front)
        {
            // capture on the chain's own stream (the caller's may be the legacy default stream, which cannot capture)
            cudaGraph_t    graph    = nullptr;
            const uint64_t counted0 = dfx_launch_count();
            cudaError_t    e        = cudaStreamBeginCapture(c->cap_stream, cudaStreamCaptureModeThreadLocal);
            dfx_status  rs    = e == cudaSuccess ? record_front(x, c->cap_stream, &color) : check_cuda(e, "cudaStreamBeginCapture");
            if (rs == DFX_OK && !x.side_post) rs = record_post(x, c->cap_stream, color);
            if (e == cudaSuccess) e = cudaStreamEndCapture(c->cap_stream, &graph);
            if (rs == DFX_OK && e == cudaSuccess) e = cudaGraphInstantiate(&g.front, graph, 0);
            if (graph) cudaGraphDestroy(graph);
            if (rs == DFX_OK && e == cudaSuccess && x.side_post)
            {
                graph = nullptr;
                e     = cudaStreamBeginCapture(c->cap_stream, cudaStreamCaptureModeThreadLocal);
                rs    = e == cudaSuccess ? record_post(x, c->cap_stream, color) : check_cuda(e, "cudaStreamBeginCapture");
                if (e == cudaSuccess) e = cudaStreamEndCapture(c->cap_stream, &graph);
                if (rs == DFX_OK && e == cudaSuccess) e = cudaGraphInstantiate(&g.post, graph, 0);
                if (graph) cudaGraphDestroy(graph);
            }
            if (rs != DFX_OK || e != cudaSuccess)
            {
                // a capture that failed leaves nothing on the GPU: run this frame (and every later one) eagerly
                (void)cudaGetLastError();
                if (g.front) cudaGraphExecDestroy(g.front);
                if (g.post) cudaGraphExecDestroy(g.post);
                c->graphs.erase(key);
                c->graphs_ok = false;
                c->stats.graph_failures += 1;
                steady = false;
            }
            else
            {
                c->stats.graphs_built += 1;
                g.kernels = int(dfx_launch_count() - counted0);
            }
            count_launch(-int(dfx_launch_count() - counted0)); // recorded, not launched
            if (c->graphs.size() > 64) c->drop_graphs(), steady = false; // runaway key churn (a caller that never reuses its planes): stay eager
        }
        if (steady)
        {
            GraphPair& gg = c->graphs[key];
            DFX_CUDA(cudaGraphLaunch(gg.front, main));
            if (x.side_post)
            {
                DFX_CUDA(cudaEventRecord(c->ev_front_done, main));
                DFX_CUDA(cudaStreamWaitEvent(c->post_stream, c->ev_front_done, 0));
                DFX_CUDA(cudaGraphLaunch(gg.post, c->post_stream));
            }
            // the host-side state the effects' Execute() would have advanced
            c->pfx->executed = true;
            if (st & DFX_CHAIN_STAGE_SSAO) c->ssao->last_frame = c->ssao->curr_frame;
            if (st & DFX_CHAIN_STAGE_TAA) c->taa->buffers[0].last_frame = c->taa->buffers[0].curr_frame;
            count_launch(gg.kernels);
            c->stats.frames_replayed += 1;
            replayed = true;
        }
    }
    if (!replayed)
    {
        if ((s = record_front(x, main, &color)) != DFX_OK) return s;
        if (x.side_post)
        {
            DFX_CUDA(cudaEventRecord(c->ev_front_done, main));
            DFX_CUDA(cudaStreamWaitEvent(c->post_stream, c->ev_front_done, 0));
        }
        if ((s = record_post(x, x.side_post ? c->post_stream : main, color)) != DFX_OK) return s;
        c->stats.frames_eager += 1;
    }
    if (x.side_post)
    {
        DFX_CUDA(cudaEventRecord(c->post_done[par], c->post_stream));
        c->post_pending[par] = true;
        if (!f->defer_post)
        {
            DFX_CUDA(cudaStreamWaitEvent(main, c->post_done[par], 0));
            c->post_pending[par] = false;
        }
    }
    c->last_frame = f->frame_index;
    return DFX_OK;
}

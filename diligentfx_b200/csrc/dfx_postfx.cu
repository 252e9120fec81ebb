// dfx_postfx.cu — PostFXContext passes: P0 blue noise, P1+P2+P3 fused prepare kernel.
// Reference: PostProcess/Common/src/PostFXContext.cpp:567-676; Shaders/Common/private/ComputeBlueNoiseTexture.fx,
// ComputeReprojectedDepth.fx, ComputeClosestMotion.fx.
#include "dfx_common.cuh"

namespace dfx
{

// ---------------------------------------------------------------------------------------------------------------------
// P0: Heitz blue-noise sampler (Sobol ^ scrambling tile) + R1 shift -> XY ; Hilbert-indexed R2 sequence -> ZW
// ---------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ float bn_random_number(const uint8_t* __restrict__ tables, uint32_t x, uint32_t y, uint32_t dim)
{
    uint32_t value = tables[dim & 255u];
    uint32_t idx   = (dim & 7u) + ((x & 127u) + (y & 127u) * 128u) * 8u;
    value ^= (uint32_t)tables[256u + idx];
    return (float(value) + 0.5f) / 256.0f;
}

__device__ __forceinline__ uint32_t hilbert_index_128(uint32_t x, uint32_t y)
{
    x &= 127u, y &= 127u;
    uint32_t index = 0u;
#pragma unroll
    for (uint32_t level = 64u; level > 0u; level >>= 1)
    {
        uint32_t rx = (x & level) ? 1u : 0u, ry = (y & level) ? 1u : 0u;
        index += level * level * ((3u * rx) ^ ry);
        if (ry == 0u)
        {
            if (rx == 1u) x = 127u - x, y = 127u - y;
            uint32_t t = x;
            x = y, y = t;
        }
    }
    return index;
}

// `frame_dev` (optional) overrides `frame`: a launch recorded into a CUDA graph reads the frame index of the frame being replayed
__global__ void __launch_bounds__(128) blue_noise_kernel(const uint8_t* __restrict__ tables, uint32_t frame, const uint32_t* __restrict__ frame_dev, View<float2> xy,
                                                         View<float2> zw)
{
    if (frame_dev) frame = *frame_dev;
    uint32_t x = threadIdx.x, y = blockIdx.x;
    // R1 sequence shift (golden ratio)
    float alpha = 0.5f + (1.0f / 1.61803398875f) * float(frame & 0xFFu);
    xy.at(x, y) = make_float2(fracf(bn_random_number(tables, x, y, 0u) + alpha), fracf(bn_random_number(tables, x, y, 1u) + alpha));
    // R2 sequence over the Hilbert curve index
    uint32_t index = hilbert_index_128(x, y) + frame;
    index += 288u * (frame & 127u);
    const float g  = 1.32471795724474602596f;
    const float a1 = 1.0f / g, a2 = 1.0f / (g * g);
    zw.at(x, y)    = make_float2(fracf(0.5f + float(index) * a1), fracf(0.5f + float(index) * a2));
}

// ---------------------------------------------------------------------------------------------------------------------
// P1 + P2 + P3 in one pass over the frame: every input plane is read once, every output written once.
//   reprojected depth: unproject (uv + jitter, depth) with curr mViewProjInv, project with prev mViewProj, keep z
//   closest motion   : motion at the 3x3 neighbour with the smallest depth (unclamped loads: out of bounds reads 0)
//   previous depth   : copy
// ---------------------------------------------------------------------------------------------------------------------
struct PrepCam
{
    float ivw, ivh, jx, jy;
    Mat4  curr_vp_inv, prev_vp;
};

template <bool M16>
__global__ void __launch_bounds__(256) postfx_prepare_kernel(const dfx_camera_attribs* __restrict__ cams, View<const float> depth,
                                                             View<const float> prev_in, TexRG<M16> motion, View<float> reproj,
                                                             View<float2> closest, View<float> prev_out, int y0, int y1, int rev)
{
    __shared__ PrepCam cam;
    if (threadIdx.x == 0 && threadIdx.y == 0)
    {
        cam.ivw = cams[0].f4ViewportSize[2], cam.ivh = cams[0].f4ViewportSize[3];
        cam.jx = cams[0].f2Jitter[0], cam.jy = cams[0].f2Jitter[1];
        load_mat(cam.curr_vp_inv, cams[0].mViewProjInv);
        load_mat(cam.prev_vp, cams[1].mViewProj);
    }
    __syncthreads();
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    const int y = y0 + blockIdx.y * blockDim.y + threadIdx.y;
    if (x >= depth.w || y >= y1) return;

    // 3x3 closest depth; iteration order x outer, y inner, strict '<' (first minimum wins) as in the shader; reversed depth:
    // far plane 0 and strict '>' (ComputeClosestMotion.fx:5-9, 36-40)
    float d_c = 0.0f, closest_d = rev ? 0.0f : 1.0f;
    int   ox = 0, oy = 0;
#pragma unroll
    for (int dx = -1; dx <= 1; ++dx)
#pragma unroll
        for (int dy = -1; dy <= 1; ++dy)
        {
            float nd = load0(depth, x + dx, y + dy);
            if (dx == 0 && dy == 0) d_c = nd;
            if (rev ? nd > closest_d : nd < closest_d) closest_d = nd, ox = dx, oy = dy;
        }
    st_cs(&closest.at(x, y), load0(motion, x + ox, y + oy));

    float  u  = (float(x) + 0.5f) * cam.ivw + 0.5f * cam.jx;
    float  v  = (float(y) + 0.5f) * cam.ivh - 0.5f * cam.jy;
    float3 wp = inv_project_position(u, v, d_c, cam.curr_vp_inv);
    float4 c  = mul_point(wp, cam.prev_vp);
    st_cs(&reproj.at(x, y), c.z / c.w);

    st_cs(&prev_out.at(x, y), __ldg(&prev_in.at(x, y)));
}

} // namespace dfx

using namespace dfx;

namespace dfx
{
// Both cameras + the frame index travel as KERNEL PARAMETERS (1.2 KB) and are written to device memory by the kernel: no copy engine
// is involved, so the per-frame constants never queue behind a bulk host-to-device transfer of the next frame's G-buffer (a pinned
// cudaMemcpyAsync does: measured 4.1 -> 6.0 ms per streamed 4K frame), and the source needs no pinned staging ring.
struct CameraUpload
{
    dfx_camera_attribs cams[2];
    uint32_t           frame;
    float              elapsed; // seconds since the previous frame (light adaptation, dfx_exposure.cu)
};
__global__ void __launch_bounds__(320) upload_cameras_kernel(const __grid_constant__ CameraUpload u, uint32_t* __restrict__ dst_cams, uint32_t* __restrict__ dst_frame,
                                                             float* __restrict__ dst_elapsed)
{
    constexpr int  kWords = int(2 * sizeof(dfx_camera_attribs) / 4);
    const uint32_t* src   = reinterpret_cast<const uint32_t*>(&u);
    if (threadIdx.x < kWords) dst_cams[threadIdx.x] = src[threadIdx.x];
    if (threadIdx.x == 0 && dst_frame) *dst_frame = u.frame;
    if (threadIdx.x == 0 && dst_elapsed) *dst_elapsed = u.elapsed;
}
dfx_status launch_upload_cameras(void* stream, const dfx_camera_attribs* curr, const dfx_camera_attribs* prev, uint32_t frame_index, dfx_camera_attribs* dst_cams,
                                 uint32_t* dst_frame, float elapsed, float* dst_elapsed)
{
    static_assert(2 * sizeof(dfx_camera_attribs) / 4 <= 320, "one thread per word");
    CameraUpload u;
    u.cams[0] = *curr, u.cams[1] = *prev, u.frame = frame_index, u.elapsed = elapsed;
    upload_cameras_kernel<<<1, 320, 0, as_stream(stream)>>>(u, reinterpret_cast<uint32_t*>(dst_cams), dst_frame, dst_elapsed);
    DFX_LAUNCHED("upload_cameras_kernel");
    return DFX_OK;
}
dfx_status launch_upload_cameras(void* stream, const dfx_camera_attribs* curr, const dfx_camera_attribs* prev, uint32_t frame_index, dfx_camera_attribs* dst_cams,
                                 uint32_t* dst_frame)
{
    return launch_upload_cameras(stream, curr, prev, frame_index, dst_cams, dst_frame, 0.0f, nullptr);
}

void preload_postfx_kernels() // force the lazily-loaded kernels of this file in (see dfx_strips.cu)
{
    cudaFuncAttributes fa;
    (void)cudaFuncGetAttributes(&fa, upload_cameras_kernel);
    (void)cudaFuncGetAttributes(&fa, blue_noise_kernel);
    (void)cudaFuncGetAttributes(&fa, postfx_prepare_kernel<false>);
}

dfx_status launch_blue_noise(void* stream, const uint8_t* tables, uint32_t frame_index, const uint32_t* frame_index_dev, const dfx_plane* xy, const dfx_plane* zw)
{
    DFX_PROFILE(stream, "blue_noise");
    DFX_REQUIRE(tables != nullptr, "tables must not be null");
    DFX_VIEW(float2, vxy, xy, DFX_FORMAT_RG32F);
    DFX_VIEW(float2, vzw, zw, DFX_FORMAT_RG32F);
    DFX_REQUIRE(vxy.w == 128 && vxy.h == 128 && vzw.w == 128 && vzw.h == 128, "blue-noise planes must be 128x128");
    blue_noise_kernel<<<128, 128, 0, as_stream(stream)>>>(tables, frame_index, frame_index_dev, vxy, vzw);
    DFX_LAUNCHED("blue_noise_kernel");
    return DFX_OK;
}
} // namespace dfx

extern "C" dfx_status dfx_pass_blue_noise(void* stream, const uint8_t* tables, uint32_t frame_index, const dfx_plane* xy, const dfx_plane* zw)
{
    return launch_blue_noise(stream, tables, frame_index, nullptr, xy, zw);
}

extern "C" dfx_status dfx_pass_postfx_prepare(void* stream, const dfx_camera_attribs* cameras_dev, const dfx_plane* curr_depth,
                                              const dfx_plane* prev_depth_in, const dfx_plane* motion, const dfx_plane* reprojected_depth,
                                              const dfx_plane* closest_motion, const dfx_plane* previous_depth, dfx_rows rows)
{
    DFX_PROFILE(stream, "postfx_prepare");
    DFX_REQUIRE(cameras_dev != nullptr, "cameras_dev must not be null");
    DFX_VIEW(const float, d, curr_depth, DFX_FORMAT_R32F);
    DFX_VIEW(const float, pin, prev_depth_in, DFX_FORMAT_R32F);
    DFX_TEX2(m, motion);
    DFX_VIEW(float, rp, reprojected_depth, DFX_FORMAT_R32F);
    DFX_VIEW(float2, cm, closest_motion, DFX_FORMAT_RG32F);
    DFX_VIEW(float, pout, previous_depth, DFX_FORMAT_R32F);
    DFX_SAME_SIZE(d, pin);
    DFX_SAME_SIZE(d, m);
    DFX_SAME_SIZE(d, rp);
    DFX_SAME_SIZE(d, cm);
    DFX_SAME_SIZE(d, pout);
    DFX_REQUIRE(rows_ok(rows, d.h), "bad row range");
    if (rows.y1 == rows.y0) return DFX_OK;
    dim3 block(32, 8), grid(div_up(d.w, 32), div_up(rows.y1 - rows.y0, 8));
    DFX_FMT16(is16(m), M16, postfx_prepare_kernel<M16><<<grid, block, 0, as_stream(stream)>>>(cameras_dev, d, pin, m, rp, cm, pout, rows.y0, rows.y1, reversed_depth(curr_depth)));
    DFX_LAUNCHED("postfx_prepare_kernel");
    return DFX_OK;
}

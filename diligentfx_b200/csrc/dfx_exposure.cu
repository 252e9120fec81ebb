// dfx_exposure.cu — auto exposure with light adaptation: the scene's average luminance, measured on the device, kept in a small
// device buffer and read by the tone-map kernels (ToneMap(c, attribs, fAveLogLum)) without a host round trip.
//
// The reference implements it inside EpipolarLightScattering (the shaders have no dependence on the atmosphere; with no light
// scattering the inscattering term is 0 and the extinction 1, so the luminance pass reads the scene colour itself):
//   GetWeightedLogLum           AtmosphereShadersCommon.fxh:199-205 (MinLuminance 0.01, UnwarpEpipolarScattering.fx:285-307)
//                               into a 64x64 RG16F target with point samples (EpipolarLightScattering.cpp:863-883, :1751)
//   GenerateMips                the box mip chain down to 1x1 (…cpp:2469, :2503)
//   UpdateAverageLuminancePS    UpdateAverageLuminance.fx:12-29 (LIGHT_ADAPTATION, fElapsedTime = FrameAttribs.dElapsedTime)
//                               alpha-blended into a persistent 1x1 R16F cleared to 0.1 at creation (…cpp:1823-1827, :885-905)
//   GetAverageSceneLuminance    max(0.05, state) (AtmosphereShadersCommon.fxh:188-197)
//
// Two sampling modes:
//   DFX_LUMINANCE_SAMPLING_REFERENCE  the reference's arithmetic bit for bit (fixed-function parts as stated in DESIGN.md §2): one CTA.
//   DFX_LUMINANCE_SAMPLING_FULL       every pixel: a grid-stride read of the colour plane (RGBA32F or RGBA16F, Tex4T loaders), fp32 per
//                                     pixel and per CTA, the per-CTA partials summed in fp64 in a fixed order by the last CTA to finish
//                                     (a ticket, no float atomics): the result is bit-identical run to run, eager or replayed.
// Both end with the same adaptation step and the same half-rounded state update.
#include "dfx_common.cuh"

namespace dfx
{
namespace
{
constexpr float kMinLuminance = 0.01f; // UnwarpEpipolarScattering.fx:305
constexpr int   kRefSize      = 64;    // sm_iLowResLuminanceMips = 7 -> 64 x 64 (EpipolarLightScattering.hpp:255)
constexpr int   kRefThreads   = 1024;
constexpr int   kFullThreads  = 256;
constexpr int   kFullCtas     = DFX_AVERAGE_LUMINANCE_MAX_PARTIALS;

// state layout (DFX_AVERAGE_LUMINANCE_STATE_FLOATS floats): see dfx_b200.h
constexpr int kStValue = 0, kStAveLogLum = 1, kStMeasured = 2, kStWeight = 3, kStTicket = 4, kStPartials = 8;

__device__ __forceinline__ float half_rn(float v) { return __half2float(__float2half_rn(v)); }
__device__ __forceinline__ float sat(float v) { return fminf(fmaxf(v, 0.0f), 1.0f); }
// log / exp correctly rounded to fp32 (evaluated in fp64): the reference mode must agree with the CPU restatement after the
// half rounding of every stored value, and in a one-CTA pass this costs nothing.
__device__ __forceinline__ float log_rn(float v) { return float(log(double(v))); }
__device__ __forceinline__ float exp_rn(float v) { return float(exp(double(v))); }

// GetWeightedLogLum (AtmosphereShadersCommon.fxh:199-205), every operation rounded separately (no contraction)
__device__ __forceinline__ float2 weighted_log_lum(float3 c)
{
    const float lum = __fadd_rn(__fadd_rn(__fmul_rn(c.x, 0.212671f), __fmul_rn(c.y, 0.715160f)), __fmul_rn(c.z, 0.072169f));
    const float w   = sat(__fdiv_rn(__fsub_rn(lum, kMinLuminance), kMinLuminance));
    const float ll  = log_rn(fmaxf(lum, 1e-5f));
    return make_float2(__fmul_rn(ll, w), w);
}

// UpdateAverageLuminancePS (UpdateAverageLuminance.fx:12-29) + the BS_AlphaBlend of its output into the R16F state:
// `wl`, `w` = the 1x1 level (means over the samples). Writes the state and the value the tone map reads.
__device__ void update_state(float* state, float measured, float w, float dt, int adapt)
{
    float a = adapt ? __fsub_rn(1.0f, exp_rn(-dt)) : 1.0f; // fAdaptationRate = 1.0
    a       = __fmul_rn(a, sat(__fdiv_rn(w, 1e-3f)));
    const float dst = state[kStValue];
    const float v   = half_rn(__fadd_rn(__fmul_rn(measured, a), __fmul_rn(dst, __fsub_rn(1.0f, a))));
    state[kStValue]     = v;
    state[kStAveLogLum] = fmaxf(0.05f, v);
    state[kStMeasured]  = measured;
    state[kStWeight]    = a;
}

__device__ __forceinline__ float elapsed(const float* dt_dev, float dt) { return dt_dev ? *dt_dev : dt; }

template <int FMT>
__global__ void __launch_bounds__(kRefThreads) luminance_reference_kernel(Tex4T<FMT> color, float* state, const float* dt_dev, float dt, int adapt)
{
    __shared__ float2 lv[kRefSize * kRefSize];
    const int tid = threadIdx.x;
    // level 0: 64 x 64 point samples at uv = ((i + .5) / 64, (j + .5) / 64), texel = floor(uv * size) (clamp addressing)
    for (int s = tid; s < kRefSize * kRefSize; s += kRefThreads)
    {
        const int   i = s % kRefSize, j = s / kRefSize;
        const float u = __fmul_rn(float(i) + 0.5f, 1.0f / kRefSize), v = __fmul_rn(float(j) + 0.5f, 1.0f / kRefSize);
        const int   x = min(max(int(floorf(__fmul_rn(u, float(color.w)))), 0), color.w - 1);
        const int   y = min(max(int(floorf(__fmul_rn(v, float(color.h)))), 0), color.h - 1);
        const float4 c = color.ld(x, y);
        const float2 l = weighted_log_lum(make_float3(c.x, c.y, c.z));
        lv[s] = make_float2(half_rn(l.x), half_rn(l.y)); // RG16F render target
    }
    __syncthreads();
    // GenerateMips: six 2x2 box levels, each the fp32 mean of four rounded to RG16F (in place: level k lives in the first n*n entries)
    for (int n = kRefSize / 2; n >= 1; n >>= 1)
    {
        float2 m = make_float2(0.f, 0.f);
        const bool active = tid < n * n;
        if (active)
        {
            const int    i = tid % n, j = tid / n, src = 2 * n;
            const float2 a = lv[(2 * j) * src + 2 * i], b = lv[(2 * j) * src + 2 * i + 1];
            const float2 c = lv[(2 * j + 1) * src + 2 * i], d = lv[(2 * j + 1) * src + 2 * i + 1];
            m.x = half_rn(__fmul_rn(__fadd_rn(__fadd_rn(__fadd_rn(a.x, b.x), c.x), d.x), 0.25f));
            m.y = half_rn(__fmul_rn(__fadd_rn(__fadd_rn(__fadd_rn(a.y, b.y), c.y), d.y), 0.25f));
        }
        __syncthreads();
        if (active) lv[tid] = m;
        __syncthreads();
    }
    if (tid == 0)
    {
        const float2 t        = lv[0];
        const float  measured = exp_rn(__fdiv_rn(t.x, fmaxf(t.y, 1e-6f)));
        update_state(state, measured, t.y, elapsed(dt_dev, dt), adapt);
    }
}

template <class T>
__device__ __forceinline__ T block_sum(T v, T* red) // fixed order: butterfly within warps, then warp 0 over the warp sums
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    __syncthreads();
    if (lane == 0) red[warp] = v;
    __syncthreads();
    if (warp == 0)
    {
        v = lane < int(blockDim.x >> 5) ? red[lane] : T(0);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    }
    return v; // valid in thread 0
}

template <int FMT>
__global__ void __launch_bounds__(kFullThreads) luminance_full_kernel(Tex4T<FMT> color, float* state, const float* dt_dev, float dt, int adapt)
{
    __shared__ float  redf[kFullThreads / 32];
    __shared__ double redd[kFullThreads / 32];
    __shared__ bool   last;
    float swl = 0.0f, sw = 0.0f;
    for (int y = blockIdx.x; y < color.h; y += gridDim.x)
    {
#pragma unroll 4
        for (int x = threadIdx.x; x < color.w; x += kFullThreads)
        {
            const float4 c   = color.ld(x, y);
            const float  lum = c.x * 0.212671f + c.y * 0.715160f + c.z * 0.072169f;
            const float  w   = sat((lum - kMinLuminance) * (1.0f / kMinLuminance));
            swl += logf(fmaxf(lum, 1e-5f)) * w;
            sw += w;
        }
    }
    swl = block_sum(swl, redf);
    sw  = block_sum(sw, redf);
    float2*   partials = reinterpret_cast<float2*>(state + kStPartials);
    unsigned* ticket   = reinterpret_cast<unsigned*>(state + kStTicket);
    if (threadIdx.x == 0)
    {
        partials[blockIdx.x] = make_float2(swl, sw);
        __threadfence();
        last = atomicAdd(ticket, 1u) == gridDim.x - 1;
    }
    __syncthreads();
    if (!last) return;
    __threadfence();
    // the last CTA: the partials in index order, in fp64
    double dwl = 0.0, dw = 0.0;
    for (int i = threadIdx.x; i < int(gridDim.x); i += kFullThreads)
    {
        const float2 p = __ldcg(&partials[i]);
        dwl += double(p.x), dw += double(p.y);
    }
    dwl = block_sum(dwl, redd);
    dw  = block_sum(dw, redd);
    if (threadIdx.x == 0)
    {
        const double n        = double(color.w) * double(color.h);
        const double mwl = dwl / n, mw = dw / n; // what the 1x1 level of a full-resolution mip chain would hold
        const float  measured = float(exp(mwl / fmax(mw, 1e-6)));
        update_state(state, measured, float(mw), elapsed(dt_dev, dt), adapt);
        *ticket = 0u; // ready for the next launch
    }
}

__global__ void luminance_reset_kernel(float* state)
{
    state[kStValue] = state[kStAveLogLum] = half_rn(0.1f); // the R16F target cleared to 0.1 (EpipolarLightScattering.cpp:885-905)
    state[kStMeasured] = state[kStWeight] = 0.0f;
    reinterpret_cast<unsigned*>(state)[kStTicket] = 0u;
}
} // namespace

dfx_status launch_update_average_luminance(void* stream, int adapt, int32_t sampling, float dt, const float* dt_dev, const dfx_plane* color_, float* state)
{
    DFX_REQUIRE(state, "null state buffer");
    DFX_REQUIRE(sampling == DFX_LUMINANCE_SAMPLING_REFERENCE || sampling == DFX_LUMINANCE_SAMPLING_FULL, "unknown luminance sampling %d", sampling);
    DFX_REQUIRE(reinterpret_cast<uintptr_t>(state) % 16 == 0, "the state buffer must be 16-byte aligned");
    DFX_TEX4(c, color_);
    cudaStream_t s = as_stream(stream);
    if (sampling == DFX_LUMINANCE_SAMPLING_REFERENCE)
    {
        DFX_FMT16(is16(c), H, luminance_reference_kernel<H ? DFX_FORMAT_RGBA16F : DFX_FORMAT_RGBA32F><<<1, kRefThreads, 0, s>>>(c, state, dt_dev, dt, adapt));
        DFX_LAUNCHED("luminance_reference_kernel");
    }
    else
    {
        const int ctas = min(c.h, kFullCtas);
        DFX_FMT16(is16(c), H, luminance_full_kernel<H ? DFX_FORMAT_RGBA16F : DFX_FORMAT_RGBA32F><<<ctas, kFullThreads, 0, s>>>(c, state, dt_dev, dt, adapt));
        DFX_LAUNCHED("luminance_full_kernel");
    }
    return DFX_OK;
}

dfx_status launch_reset_average_luminance(void* stream, float* state)
{
    DFX_REQUIRE(state, "null state buffer");
    DFX_REQUIRE(reinterpret_cast<uintptr_t>(state) % 16 == 0, "the state buffer must be 16-byte aligned");
    luminance_reset_kernel<<<1, 1, 0, as_stream(stream)>>>(state);
    DFX_LAUNCHED("luminance_reset_kernel");
    return DFX_OK;
}
} // namespace dfx

using namespace dfx;

extern "C" dfx_status dfx_pass_update_average_luminance(void* stream, const dfx_tonemap_attribs* attribs, int32_t sampling, float elapsed_seconds,
                                                        const dfx_plane* color, float* state_dev)
{
    DFX_PROFILE(stream, "update_average_luminance");
    DFX_REQUIRE(attribs, "null argument");
    DFX_REQUIRE(elapsed_seconds >= 0.0f, "elapsed time must be >= 0 (got %g)", elapsed_seconds);
    return launch_update_average_luminance(stream, attribs->bLightAdaptation != 0, sampling, elapsed_seconds, nullptr, color, state_dev);
}

extern "C" dfx_status dfx_pass_reset_average_luminance(void* stream, float* state_dev)
{
    DFX_PROFILE(stream, "reset_average_luminance");
    return launch_reset_average_luminance(stream, state_dev);
}

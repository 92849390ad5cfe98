// The small ops at the end of the render inside one `-O` train step (SURVEY.md 8f row 2), each as ONE launch instead of
// the reference's chains of eager elementwise kernels (the optimizer step after it is csrc/adam.cu):
//
//   * ngp_blend_background_forward/backward: `image + (1 - weights_sum) * bg`, the depth normalisation and the
//     hit mask at the end of run_cuda (nerf/renderer.py:535-557).
//   * ngp_entropy_loss_forward/backward: the opacity-entropy regulariser of train_step (nerf/utils.py:389-394).
//
// All of it is streaming fp32 work, no tensor cores.
#include <math.h>

#include "common.cuh"

namespace ngp {
namespace step {

// ---- background blend ---------------------------------------------------------------------------------------------
// image_out = image + (1 - ws) * bg ; depth_out = clamp(depth - near, 0) / (far - near) ; mask = near < far
__global__ void __launch_bounds__(256) blend_forward_kernel(const float* __restrict__ image, const float* __restrict__ ws,
                                                            const float* __restrict__ depth, const float* __restrict__ bg,
                                                            int bg_stride, const float* __restrict__ nears,
                                                            const float* __restrict__ fars, uint32_t N, float* __restrict__ image_out,
                                                            float* __restrict__ depth_out, uint8_t* __restrict__ mask) {
    const uint32_t n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    const float one_minus = 1.f - ws[n];
    const float* b = bg + (size_t)n * bg_stride;  // bg_stride 0: one broadcast colour
#pragma unroll
    for (int c = 0; c < 3; ++c) image_out[(size_t)n * 3 + c] = image[(size_t)n * 3 + c] + one_minus * b[c];
    const float nr = nears[n], fr = fars[n];
    if (depth_out) depth_out[n] = fmaxf(depth[n] - nr, 0.f) / (fr - nr);  // NaN for box misses, as the reference (0/0)
    if (mask) mask[n] = nr < fr ? 1 : 0;
}

// d_image = g ; d_ws = -sum_c g_c bg_c ; d_bg = (1 - ws) g   (d_image aliases g: nothing to write)
__global__ void __launch_bounds__(256) blend_backward_kernel(const float* __restrict__ g, const float* __restrict__ ws,
                                                             const float* __restrict__ bg, int bg_stride, uint32_t N,
                                                             float* __restrict__ d_ws, float* __restrict__ d_bg) {
    const uint32_t n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    const float one_minus = 1.f - ws[n];
    const float* b = bg + (size_t)n * bg_stride;
    float acc = 0.f;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        const float gc = g[(size_t)n * 3 + c];
        acc += gc * b[c];
        if (d_bg) d_bg[(size_t)n * 3 + c] = one_minus * gc;
    }
    d_ws[n] = -acc;
}

// ---- opacity entropy ------------------------------------------------------------------------------------------------
// loss = lam * mean(-a log2 a - (1 - a) log2(1 - a)),  a = clamp(ws, 1e-5, 1 - 1e-5)   (nerf/utils.py:389-394)
// One block: deterministic, and N is a ray count (<= a few 10^5).
constexpr float kAlphaLo = 1e-5f, kAlphaHi = 1.f - 1e-5f;

__global__ void __launch_bounds__(1024) entropy_forward_kernel(const float* __restrict__ ws, uint32_t N, float lam,
                                                               float* __restrict__ loss) {
    __shared__ float s_part[32];
    float acc = 0.f;
    for (uint32_t n = threadIdx.x; n < N; n += blockDim.x) {
        const float a = fminf(fmaxf(ws[n], kAlphaLo), kAlphaHi);
        acc += -a * log2f(a) - (1.f - a) * log2f(1.f - a);
    }
    acc = warp_sum(acc);
    if ((threadIdx.x & 31) == 0) s_part[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x < 32) {
        float v = threadIdx.x < (blockDim.x >> 5) ? s_part[threadIdx.x] : 0.f;
        v = warp_sum(v);
        if (threadIdx.x == 0) *loss = lam * (v / (float)N);
    }
}

// d_ws (+)= g * lam / N * (log2(1 - a) - log2(a)) inside the clamp range, 0 outside (clamp's subgradient).
// `g` is a device scalar (the upstream gradient of the loss, e.g. the GradScaler's scale).
__global__ void __launch_bounds__(256) entropy_backward_kernel(const float* __restrict__ ws, uint32_t N, float lam,
                                                               const float* __restrict__ g, float* __restrict__ d_ws,
                                                               int accumulate) {
    const uint32_t n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    const float w = ws[n];
    float d = 0.f;
    if (w >= kAlphaLo && w <= kAlphaHi) d = (*g) * (lam / (float)N) * (log2f(1.f - w) - log2f(w));
    d_ws[n] = accumulate ? d_ws[n] + d : d;
}

}  // namespace step
}  // namespace ngp

using namespace ngp;

extern "C" int ngp_blend_background_forward(const float* image, const float* weights_sum, const float* depth, const float* bg,
                                            int bg_per_ray, const float* nears, const float* fars, uint32_t N, float* image_out,
                                            float* depth_out, uint8_t* mask, void* stream) {
    if (!image || !weights_sum || !bg || !nears || !fars || !image_out || (depth_out && !depth)) return NGP_ERR_BAD_ARG;
    if (N == 0) return NGP_OK;
    step::blend_forward_kernel<<<cdiv(N, 256), 256, 0, as_stream(stream)>>>(image, weights_sum, depth, bg, bg_per_ray ? 3 : 0,
                                                                          nears, fars, N, image_out, depth_out, mask);
    return launch_status();
}

extern "C" int ngp_blend_background_backward(const float* grad_image, const float* weights_sum, const float* bg, int bg_per_ray,
                                             uint32_t N, float* grad_weights_sum, float* grad_bg, void* stream) {
    if (!grad_image || !weights_sum || !bg || !grad_weights_sum) return NGP_ERR_BAD_ARG;
    if (N == 0) return NGP_OK;
    step::blend_backward_kernel<<<cdiv(N, 256), 256, 0, as_stream(stream)>>>(grad_image, weights_sum, bg, bg_per_ray ? 3 : 0, N,
                                                                           grad_weights_sum, bg_per_ray ? grad_bg : nullptr);
    return launch_status();
}

extern "C" int ngp_entropy_loss_forward(const float* weights_sum, uint32_t N, float lambda, float* loss, void* stream) {
    if (!weights_sum || !loss || N == 0) return NGP_ERR_BAD_ARG;
    step::entropy_forward_kernel<<<1, 1024, 0, as_stream(stream)>>>(weights_sum, N, lambda, loss);
    return launch_status();
}

extern "C" int ngp_entropy_loss_backward(const float* weights_sum, uint32_t N, float lambda, const float* grad_loss,
                                         float* grad_weights_sum, int accumulate, void* stream) {
    if (!weights_sum || !grad_loss || !grad_weights_sum || N == 0) return NGP_ERR_BAD_ARG;
    step::entropy_backward_kernel<<<cdiv(N, 256), 256, 0, as_stream(stream)>>>(weights_sum, N, lambda, grad_loss,
                                                                              grad_weights_sum, accumulate);
    return launch_status();
}

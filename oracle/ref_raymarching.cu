// TEST INFRASTRUCTURE: oracle_composite_rays (ngp_oracle.c, raymarching.cu:843-899) as a CUDA kernel.  The reference takes
// alpha from __expf (the device's ex2.approx), which only a device produces; every fused multiply-add is spelled out with
// fmaf as in the oracle, and oracle/build.py compiles this file with -fmad=false so that no other one is formed.
// Used by oracle/ref_standin.py.
#include <cstdint>
#include <cuda_runtime.h>

__global__ void oracle_composite_rays_kernel(uint32_t n_alive, uint32_t n_step, float T_thresh, int* rays_alive, float* rays_t,
                                             const float* sigmas, const float* rgbs, const float* deltas, float* weights_sum,
                                             float* depth, float* image) {
    const uint32_t n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= n_alive) return;
    const int index = rays_alive[n];
    const float* s = sigmas + (uint64_t)n * n_step;
    const float* c = rgbs + (uint64_t)n * n_step * 3;
    const float* dl = deltas + (uint64_t)n * n_step * 2;
    float t = rays_t[index];
    float weight_sum = weights_sum[index], d = depth[index];
    float r = image[index * 3], g = image[index * 3 + 1], b = image[index * 3 + 2];
    uint32_t step = 0;
    while (step < n_step) {
        if (dl[0] == 0) break;
        const float alpha = 1.0f - __expf(-s[0] * dl[0]);
        const float T = 1 - weight_sum;
        const float weight = alpha * T;
        weight_sum += weight;
        t += dl[1];
        d = fmaf(weight, t, d);
        r = fmaf(weight, c[0], r);
        g = fmaf(weight, c[1], g);
        b = fmaf(weight, c[2], b);
        if (T < T_thresh) break;
        s++; c += 3; dl += 2; step++;
    }
    if (step < n_step) rays_alive[n] = -1; else rays_t[index] = t;
    weights_sum[index] = weight_sum; depth[index] = d;
    image[index * 3] = r; image[index * 3 + 1] = g; image[index * 3 + 2] = b;
}

extern "C" int oracle_composite_rays_cuda(uint32_t n_alive, uint32_t n_step, float T_thresh, int* rays_alive, float* rays_t,
                                          const float* sigmas, const float* rgbs, const float* deltas, float* weights_sum,
                                          float* depth, float* image, void* stream) {
    if (n_alive == 0) return 0;
    oracle_composite_rays_kernel<<<(n_alive + 127) / 128, 128, 0, (cudaStream_t)stream>>>(
        n_alive, n_step, T_thresh, rays_alive, rays_t, sigmas, rgbs, deltas, weights_sum, depth, image);
    return (int)cudaGetLastError();
}

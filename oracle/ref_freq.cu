// TEST INFRASTRUCTURE: oracle_freq_encode_forward (ngp_oracle.c, freqencoder.cu:30-58) as a CUDA kernel.  The reference
// builds its freqencoder with --use_fast_math (freqencoder/backend.py:9), so its sinf is the device's sin.approx, which
// only a device produces; oracle/build.py compiles this file the same way.  Used by oracle/ref_standin.py.
#include <cstdint>
#include <cuda_runtime.h>

__global__ void oracle_freq_forward_kernel(const float* inputs, uint32_t B, uint32_t D, uint32_t C, float* outputs) {
    const uint64_t t = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (t >= (uint64_t)B * C) return;
    const uint32_t b = (uint32_t)(t / C), c = (uint32_t)(t % C);
    const float* in = inputs + (uint64_t)b * D;
    float v;
    if (c < D) {
        v = in[c];
    } else {
        const uint32_t col = c / D - 1, d = c % D, freq = col / 2;
        const float phase_shift = (float)(col % 2) * (3.141592653589793f / 2);
        v = sinf(ldexpf(in[d], (int)freq) + phase_shift);
    }
    outputs[t] = v;
}

extern "C" int oracle_freq_encode_forward_cuda(const float* inputs, uint32_t B, uint32_t D, uint32_t C, float* outputs,
                                               void* stream) {
    const uint64_t n = (uint64_t)B * C;
    if (n == 0) return 0;
    oracle_freq_forward_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(inputs, B, D, C, outputs);
    return (int)cudaGetLastError();
}

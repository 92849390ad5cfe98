// Shading path of the grid field as a 7-point stencil (SURVEY 8f-4): finite-difference normals + Lambertian / textureless /
// normal colouring, forward and backward.
//
// Behavioural contract: nerf/network_grid.py:90-144.  The reference evaluates the field SEVEN times per shaded sample -
// common_forward(x) plus common_forward((x +- eps e_i).clamp(-bound, bound)) for the three axes (:93-98), each a separate
// encoder launch + 3 GEMMs + ~10 elementwise kernels - and SIX more for the smoothness regulariser's normal(x + noise)
// (nerf/renderer.py:491).  Here the stencil points of a sample are laid out as K CONSECUTIVE rows of ONE batch
// (K = 7 with the centre, 6 without): one fused-field launch evaluates all of them, the K points of a sample sit within
// 2 eps = 0.02 of each other, so at every level coarser than that they hit the same grid cell - the corner fetches come
// from L1 and the warp-aggregated scatter of the backward merges their updates before they reach L2 - and two small
// kernels here turn the K densities into normal / colour and back-propagate through them.
//
// Arithmetic under fp16 autocast, mirrored: densities are fp32 (trunc_exp returns float); grad = 0.5 * (s+ - s-) / eps
// in fp32 (a division by a python scalar multiplies by the fp32 reciprocal); safe_normalize clamps the squared norm at
// 1e-20, NaNs -> 0; `normal @ l` runs as a half matrix-vector product (operands rounded to half, fp32 accumulate, half
// result); ratio + (1 - ratio) * clamp(., 0) and albedo * lambertian are half operations (each rounds to half).
//
// The hand-scheduled train step (ngp_b200/trainer.py) runs the same arithmetic on fixed-capacity buffers with the sample
// count read on the device: stencil_points_kernel with a count pointer writes 7 M for the field kernels, the *_step kernels
// below read / write the chain's ordinary per-sample rows (sigma [M], rgb [M,3] for ngp_train_ray_loss, and its gradients)
// and the backward adds the orientation regulariser of nerf/renderer.py:485-486 and its gradient.  The light direction is
// read from device memory (ngp_train_light, csrc/raymarch.cu, draws it per step).
#include "common.cuh"

namespace ngp {
namespace shade {

constexpr float kRcpEps100 = 100.0f;   // fl(1 / fl(0.01)) in fp32

NGP_DEVINL float clampf(float x, float lo, float hi) { return fminf(hi, fmaxf(lo, x)); }
NGP_DEVINL float h16(float x) { return __half2float(__float2half_rn(x)); }

// K rows per sample: [x,] x + eps e_x, x - eps e_x, x + eps e_y, ... (the reference's dx_pos, dx_neg, dy_pos, ... order).
// count_ptr (optional): M = min(*count_ptr, M_cap) samples, read on the device; count_out (optional) receives K * M.
__global__ void stencil_points_kernel(const float* __restrict__ xyzs, uint32_t M_cap, const int* __restrict__ count_ptr,
                                      float eps, float bound, int with_centre, float* __restrict__ out, int* __restrict__ count_out) {
    const uint32_t K = with_centre ? 7u : 6u;
    const uint32_t M = count_ptr ? min((uint32_t)max(*count_ptr, 0), M_cap) : M_cap;
    if (count_out && blockIdx.x == 0 && threadIdx.x == 0) *count_out = (int)(K * M);
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < M; i += gridDim.x * blockDim.x) {
        const float x[3] = {xyzs[(size_t)i * 3], xyzs[(size_t)i * 3 + 1], xyzs[(size_t)i * 3 + 2]};
        float* o = out + (size_t)i * K * 3;
        if (with_centre) { o[0] = x[0]; o[1] = x[1]; o[2] = x[2]; o += 3; }
#pragma unroll
        for (int a = 0; a < 3; ++a) {
#pragma unroll
            for (int s = 0; s < 2; ++s) {
                float p[3] = {x[0], x[1], x[2]};
                p[a] = __fadd_rn(p[a], s == 0 ? eps : -eps);
                // (x + offset).clamp(-bound, bound): all three coordinates are clamped (network_grid.py:93-98)
                o[0] = clampf(p[0], -bound, bound); o[1] = clampf(p[1], -bound, bound); o[2] = clampf(p[2], -bound, bound);
                o += 3;
            }
        }
    }
}

struct Normal {
    float g[3];     // -0.5 (s+ - s-) / eps  (finite_difference_normal)
    float n[3];     // safe_normalize(g), NaN -> 0
    float inv;      // 1 / sqrt(max(|g|^2, 1e-20))
    bool clamped;   // |g|^2 < 1e-20: the norm is the constant 1e-10
    bool nan[3];
};
NGP_DEVINL Normal normal_of(const float* __restrict__ s6) {
    Normal r;
#pragma unroll
    for (int a = 0; a < 3; ++a) r.g[a] = -(__fmul_rn(__fmul_rn(0.5f, __fsub_rn(s6[2 * a], s6[2 * a + 1])), kRcpEps100));
    const float nn = __fadd_rn(__fadd_rn(__fmul_rn(r.g[0], r.g[0]), __fmul_rn(r.g[1], r.g[1])), __fmul_rn(r.g[2], r.g[2]));
    r.clamped = !(nn >= 1e-20f);          // (NaN compares false: treated like the clamp for the backward; values become 0)
    r.inv = 1.0f / sqrtf(fmaxf(nn, 1e-20f));
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        float v = __fdiv_rn(r.g[a], sqrtf(fmaxf(nn, 1e-20f)));
        r.nan[a] = v != v;
        r.n[a] = r.nan[a] ? 0.f : v;      // normal[torch.isnan(normal)] = 0
    }
    return r;
}

// colour of a shaded sample from its normal (network_grid.py:126-140); mode: 0 = lambertian, 1 = textureless, 2 = normal.
// alb: the centre row's albedo (fp32 holding half values; read in mode 0 only).
NGP_DEVINL void shade_color(const Normal& nm, const float* __restrict__ light, float ratio, int mode, const float* __restrict__ alb,
                            float c[3]) {
    if (mode == 2) {                      // (normal + 1) / 2, fp32
#pragma unroll
        for (int a = 0; a < 3; ++a) c[a] = __fmul_rn(__fadd_rn(nm.n[a], 1.0f), 0.5f);
        return;
    }
    // lambertian = ratio + (1 - ratio) * (normal @ l).clamp(min=0), in half (see the header)
    float dot = 0.f;
#pragma unroll
    for (int a = 0; a < 3; ++a) dot = fmaf(h16(nm.n[a]), h16(light[a]), dot);
    const float dh = fmaxf(h16(dot), 0.f);
    const float lam = h16(ratio + h16((1.0f - ratio) * dh));
    if (mode == 1) { c[0] = lam; c[1] = lam; c[2] = lam; return; }
#pragma unroll
    for (int a = 0; a < 3; ++a) c[a] = h16(alb[a] * lam);
}

// d_color [3] -> dn [3] += its share of the normal's gradient; d_alb [3] = d(albedo) (mode 0, else left alone)
NGP_DEVINL void shade_color_backward(const Normal& nm, const float* __restrict__ light, float ratio, int mode,
                                     const float* __restrict__ alb, const float dc[3], float dn[3], float d_alb[3]) {
    if (mode == 2) {
#pragma unroll
        for (int a = 0; a < 3; ++a) dn[a] += 0.5f * dc[a];
        return;
    }
    float dot = 0.f;
#pragma unroll
    for (int a = 0; a < 3; ++a) dot = fmaf(h16(nm.n[a]), h16(light[a]), dot);
    const float dh = h16(dot);
    const float lam = h16(ratio + h16((1.0f - ratio) * fmaxf(dh, 0.f)));
    float d_lam;
    if (mode == 1) {
        d_lam = dc[0] + dc[1] + dc[2];
    } else {
        d_lam = dc[0] * alb[0] + dc[1] * alb[1] + dc[2] * alb[2];
#pragma unroll
        for (int a = 0; a < 3; ++a) d_alb[a] = dc[a] * lam;
    }
    if (dh >= 0.f) {                      // clamp(min=0) passes the gradient where input >= 0 (torch: grad * (x >= min))
        const float d_dot = d_lam * (1.0f - ratio);
#pragma unroll
        for (int a = 0; a < 3; ++a) dn[a] += d_dot * light[a];
    }
}

// through normal[isnan] = 0 and safe_normalize (n = g * inv, inv = max(|g|^2, 1e-20)^-1/2) and the central difference:
// d(s+) of axis a = ds[a], d(s-) = -ds[a]  (NaN -> 0)
NGP_DEVINL void normal_backward(const Normal& nm, const float dn[3], float ds[3]) {
    float dnm[3], dg[3];
#pragma unroll
    for (int a = 0; a < 3; ++a) dnm[a] = nm.nan[a] ? 0.f : dn[a];
    if (nm.clamped) {
#pragma unroll
        for (int a = 0; a < 3; ++a) dg[a] = dnm[a] * nm.inv;
    } else {
        const float proj = nm.n[0] * dnm[0] + nm.n[1] * dnm[1] + nm.n[2] * dnm[2];
#pragma unroll
        for (int a = 0; a < 3; ++a) dg[a] = (dnm[a] - nm.n[a] * proj) * nm.inv;
    }
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        float v = -0.5f * kRcpEps100 * dg[a];
        if (v != v) v = 0.f;
        ds[a] = v;
    }
}

// mode: 0 = lambertian, 1 = textureless, 2 = normal ; K = 7 (centre first) or 6 (normal only: color == nullptr)
__global__ void shade_forward_kernel(const float* __restrict__ sigma_all, const float* __restrict__ rgb_all, uint32_t M, uint32_t K,
                                     const float* __restrict__ light, float ratio, int mode, float* __restrict__ normal_out,
                                     float* __restrict__ color_out) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= M) return;
    const float* s = sigma_all + (size_t)i * K + (K == 7 ? 1 : 0);
    float s6[6];
#pragma unroll
    for (int k = 0; k < 6; ++k) s6[k] = s[k];
    const Normal nm = normal_of(s6);
    normal_out[(size_t)i * 3] = nm.n[0]; normal_out[(size_t)i * 3 + 1] = nm.n[1]; normal_out[(size_t)i * 3 + 2] = nm.n[2];
    if (!color_out) return;
    float c[3];
    shade_color(nm, light, ratio, mode, rgb_all + (size_t)i * K * 3, c);
    color_out[(size_t)i * 3] = c[0]; color_out[(size_t)i * 3 + 1] = c[1]; color_out[(size_t)i * 3 + 2] = c[2];
}

// d_sigma_all [M*K] (the centre's entry, k = 0 of K = 7, is written as 0: its own gradient arrives through the sigma
// output), d_rgb_all [M*K,3] (non-zero only in the centre row, lambertian mode); either may be nullptr.
__global__ void shade_backward_kernel(const float* __restrict__ sigma_all, const float* __restrict__ rgb_all, uint32_t M, uint32_t K,
                                      const float* __restrict__ light, float ratio, int mode, const float* __restrict__ d_normal,
                                      const float* __restrict__ d_color, float* __restrict__ d_sigma_all,
                                      float* __restrict__ d_rgb_all) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= M) return;
    const uint32_t c0 = (K == 7 ? 1u : 0u);
    const float* s = sigma_all + (size_t)i * K + c0;
    float s6[6];
#pragma unroll
    for (int k = 0; k < 6; ++k) s6[k] = s[k];
    const Normal nm = normal_of(s6);
    float dn[3] = {0.f, 0.f, 0.f};
    if (d_normal) { dn[0] = d_normal[(size_t)i * 3]; dn[1] = d_normal[(size_t)i * 3 + 1]; dn[2] = d_normal[(size_t)i * 3 + 2]; }
    float d_alb[3] = {0.f, 0.f, 0.f};
    if (d_color) {
        const float dc[3] = {d_color[(size_t)i * 3], d_color[(size_t)i * 3 + 1], d_color[(size_t)i * 3 + 2]};
        shade_color_backward(nm, light, ratio, mode, rgb_all + (size_t)i * K * 3, dc, dn, d_alb);
    }
    float dsa[3];
    normal_backward(nm, dn, dsa);
    if (d_sigma_all) {
        float* ds = d_sigma_all + (size_t)i * K;
        if (K == 7) ds[0] = 0.f;
#pragma unroll
        for (int a = 0; a < 3; ++a) { ds[c0 + 2 * a] = dsa[a]; ds[c0 + 2 * a + 1] = -dsa[a]; }
    }
    if (d_rgb_all) {
        float* dr = d_rgb_all + (size_t)i * K * 3;
        for (uint32_t k = 0; k < K * 3; ++k) dr[k] = 0.f;
        if (K == 7 && mode == 0) { dr[0] = d_alb[0]; dr[1] = d_alb[1]; dr[2] = d_alb[2]; }
    }
}

// ---- the hand-scheduled train step's pair (7 rows per sample, device-side count) -----------------------------------------
NGP_DEVINL uint32_t device_count(const int* count_ptr, uint32_t cap) { return min((uint32_t)max(*count_ptr, 0), cap); }

// sigma_all [7 cap] / rgb_all [7 cap,3] -> sigma [cap] (the centre density) and rgb [cap,3] (the shaded colour), rows < M
__global__ void shade_forward_step_kernel(const float* __restrict__ sigma_all, const float* __restrict__ rgb_all, uint32_t M_cap,
                                          const int* __restrict__ count_ptr, const float* __restrict__ light, float ratio, int mode,
                                          float* __restrict__ sigma, float* __restrict__ rgb) {
    const uint32_t M = device_count(count_ptr, M_cap);
    const float l[3] = {light[0], light[1], light[2]};
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < M; i += gridDim.x * blockDim.x) {
        const float* s = sigma_all + (size_t)i * 7;
        float s6[6];
#pragma unroll
        for (int k = 0; k < 6; ++k) s6[k] = s[1 + k];
        const Normal nm = normal_of(s6);
        float c[3];
        shade_color(nm, l, ratio, mode, rgb_all + (size_t)i * 21, c);
        sigma[i] = s[0];
        rgb[(size_t)i * 3] = c[0]; rgb[(size_t)i * 3 + 1] = c[1]; rgb[(size_t)i * 3 + 2] = c[2];
    }
}

// Composite gradients d_sigma [cap] / d_rgb [cap,3] of the per-sample rows -> d_sigma_all [7 cap] (centre row: d_sigma;
// stencil rows: the normal's gradient) and d_rgb_all [7 cap,3] (centre row: d(albedo) in mode 0; 0 elsewhere), with the
// orientation regulariser folded in: loss_orient = (1 - exp(-sigma)).detach() * clamp(n . d, 0)^2 averaged over the
// step's samples (the sum of counters[2c], c < n_counters: every chain of the step), *loss += lambda * mean, and its
// gradient times *scale (the GradScaler scale) joins the normal's gradient ahead of the colour's (renderer.py:485-486).
__global__ void __launch_bounds__(256) shade_backward_step_kernel(
    const float* __restrict__ sigma_all, const float* __restrict__ rgb_all, uint32_t M_cap, const int* __restrict__ count_ptr,
    const int* __restrict__ counters, uint32_t n_counters, const float* __restrict__ dirs, const float* __restrict__ light,
    float ratio, int mode, const float* __restrict__ d_sigma, const float* __restrict__ d_rgb, float lambda_orient,
    const float* __restrict__ scale, float* __restrict__ d_sigma_all, float* __restrict__ d_rgb_all, float* __restrict__ loss) {
    __shared__ float s_loss[8];
    const uint32_t M = device_count(count_ptr, M_cap);
    uint32_t total = 0;
    for (uint32_t c = 0; c < n_counters; ++c) total += (uint32_t)max(counters[2 * c], 0);
    const float coef = lambda_orient / (float)max(total, 1u);
    const float g_scale = (scale ? *scale : 1.f) * coef;
    const float l[3] = {light[0], light[1], light[2]};
    float acc = 0.f;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < M; i += gridDim.x * blockDim.x) {
        const float* s = sigma_all + (size_t)i * 7;
        float s6[6];
#pragma unroll
        for (int k = 0; k < 6; ++k) s6[k] = s[1 + k];
        const Normal nm = normal_of(s6);
        const float d[3] = {dirs[(size_t)i * 3], dirs[(size_t)i * 3 + 1], dirs[(size_t)i * 3 + 2]};
        // orientation term: weights = 1 - exp(-sigma) (fp32, detached), (normals * dirs).sum(-1).clamp(min=0) ** 2
        const float w = 1.0f - expf(-s[0]);
        const float nd = fmaxf(__fadd_rn(__fadd_rn(__fmul_rn(nm.n[0], d[0]), __fmul_rn(nm.n[1], d[1])), __fmul_rn(nm.n[2], d[2])), 0.f);
        acc += w * (nd * nd);
        const float g_nd = g_scale * w * 2.f * nd;      // d(scale * lambda * mean) / d(n . d); 0 where n . d < 0
        float dn[3] = {g_nd * d[0], g_nd * d[1], g_nd * d[2]};
        float d_alb[3] = {0.f, 0.f, 0.f};
        const float dc[3] = {d_rgb[(size_t)i * 3], d_rgb[(size_t)i * 3 + 1], d_rgb[(size_t)i * 3 + 2]};
        shade_color_backward(nm, l, ratio, mode, rgb_all + (size_t)i * 21, dc, dn, d_alb);
        float dsa[3];
        normal_backward(nm, dn, dsa);
        float* ds = d_sigma_all + (size_t)i * 7;
        ds[0] = d_sigma[i];
#pragma unroll
        for (int a = 0; a < 3; ++a) { ds[1 + 2 * a] = dsa[a]; ds[2 + 2 * a] = -dsa[a]; }
        float* dr = d_rgb_all + (size_t)i * 21;
        dr[0] = d_alb[0]; dr[1] = d_alb[1]; dr[2] = d_alb[2];
#pragma unroll
        for (int k = 3; k < 21; ++k) dr[k] = 0.f;
    }
    if (!loss) return;
    acc = warp_sum(acc);
    if ((threadIdx.x & 31) == 0) s_loss[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        float v = 0.f;
        for (uint32_t w = 0; w < (blockDim.x >> 5); ++w) v += s_loss[w];
        if (v != 0.f) atomicAdd(loss, v * coef);
    }
}

}  // namespace shade
}  // namespace ngp

using namespace ngp;

// grid of the count-driven kernels: sized from the capacity, at most 8 blocks of 256 per SM; the kernels walk it grid-stride
static int step_grid(uint32_t cap) { return (int)min((long long)cdiv(cap, 256), (long long)num_sms() * 8); }

extern "C" int ngp_stencil_points(const float* xyzs, uint32_t M, const int* count_ptr, float eps, float bound, int with_centre,
                                  float* out, int* count_out, void* stream) {
    if (!xyzs || !out) return NGP_ERR_BAD_ARG;
    if (count_out && (uint64_t)M * (with_centre ? 7u : 6u) > 0x7fffffffull) return NGP_ERR_BAD_ARG;
    if (M == 0 && !count_out) return NGP_OK;   // (with count_out, one block still writes the count)
    const int grid = count_ptr ? step_grid(M ? M : 1) : (M ? cdiv(M, 256) : 1);
    shade::stencil_points_kernel<<<grid, 256, 0, as_stream(stream)>>>(xyzs, M, count_ptr, eps, bound, with_centre, out, count_out);
    return launch_status();
}

extern "C" int ngp_shade_forward(const float* sigma_all, const float* rgb_all, uint32_t M, uint32_t K, const float* light, float ratio,
                                 int mode, float* normal_out, float* color_out, void* stream) {
    if (!sigma_all || !normal_out || (K != 6 && K != 7)) return NGP_ERR_BAD_ARG;
    if (color_out && (K != 7 || mode < 0 || mode > 2 || (mode != 2 && !light) || (mode == 0 && !rgb_all))) return NGP_ERR_BAD_ARG;
    if (M == 0) return NGP_OK;
    shade::shade_forward_kernel<<<cdiv(M, 256), 256, 0, as_stream(stream)>>>(sigma_all, rgb_all, M, K, light, ratio, mode, normal_out,
                                                                             color_out);
    return launch_status();
}

extern "C" int ngp_shade_backward(const float* sigma_all, const float* rgb_all, uint32_t M, uint32_t K, const float* light, float ratio,
                                  int mode, const float* d_normal, const float* d_color, float* d_sigma_all, float* d_rgb_all,
                                  void* stream) {
    if (!sigma_all || (K != 6 && K != 7)) return NGP_ERR_BAD_ARG;
    if (d_color && (K != 7 || mode < 0 || mode > 2 || (mode != 2 && !light) || (mode == 0 && !rgb_all))) return NGP_ERR_BAD_ARG;
    if (M == 0) return NGP_OK;
    shade::shade_backward_kernel<<<cdiv(M, 256), 256, 0, as_stream(stream)>>>(sigma_all, rgb_all, M, K, light, ratio, mode, d_normal,
                                                                              d_color, d_sigma_all, d_rgb_all);
    return launch_status();
}

extern "C" int ngp_shade_forward_step(const float* sigma_all, const float* rgb_all, uint32_t M_cap, const int* count_ptr,
                                      const float* light, float ratio, int mode, float* sigma, float* rgb, void* stream) {
    if (!sigma_all || !rgb_all || !count_ptr || !light || !sigma || !rgb || mode < 0 || mode > 2) return NGP_ERR_BAD_ARG;
    if ((uint64_t)M_cap * 7 > 0xffffffffull) return NGP_ERR_BAD_ARG;
    if (M_cap == 0) return NGP_OK;
    shade::shade_forward_step_kernel<<<step_grid(M_cap), 256, 0, as_stream(stream)>>>(sigma_all, rgb_all, M_cap, count_ptr, light,
                                                                                      ratio, mode, sigma, rgb);
    return launch_status();
}

extern "C" int ngp_shade_backward_step(const float* sigma_all, const float* rgb_all, uint32_t M_cap, const int* count_ptr,
                                       const int* counters, uint32_t n_counters, const float* dirs, const float* light, float ratio,
                                       int mode, const float* d_sigma, const float* d_rgb, float lambda_orient, const float* scale,
                                       float* d_sigma_all, float* d_rgb_all, float* loss, void* stream) {
    if (!sigma_all || !rgb_all || !count_ptr || !counters || n_counters == 0 || !dirs || !light || !d_sigma || !d_rgb ||
        !d_sigma_all || !d_rgb_all || mode < 0 || mode > 2)
        return NGP_ERR_BAD_ARG;
    if ((uint64_t)M_cap * 7 > 0xffffffffull) return NGP_ERR_BAD_ARG;
    if (M_cap == 0) return NGP_OK;
    shade::shade_backward_step_kernel<<<step_grid(M_cap), 256, 0, as_stream(stream)>>>(
        sigma_all, rgb_all, M_cap, count_ptr, counters, n_counters, dirs, light, ratio, mode, d_sigma, d_rgb, lambda_orient, scale,
        d_sigma_all, d_rgb_all, loss);
    return launch_status();
}

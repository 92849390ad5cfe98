/*
 * ngp_oracle.c - TEST INFRASTRUCTURE.  A plain-C, single-threaded CPU restatement of the reference's
 * NeRF hot-path kernels.  Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
 * --impl reference legs may load this; the product (libngp_b200.so) never does.
 *
 * Every function follows one reference kernel (file:line cited, relative to the reference tree)
 * and reproduces its floating-point evaluation ORDER.  The reference is compiled by nvcc with
 * the default -fmad=true, so wherever its source has `a * b + c` in fp32 the device executes one
 * fused multiply-add; those places use fmaf() here explicitly (checked against the SASS of the
 * reference extensions built for sm_100: FFMA for ray points, cell exits `fma(mip_bound,u,-x)`,
 * `fma(exp2, H, -1)`, `fma(x, scale, .5)` and the interpolation accumulate).  This file must be
 * built with -ffp-contract=off so the host compiler fuses nothing else.
 *
 * Known, documented deviations from device arithmetic (CPU cannot reproduce SFU approximations):
 *   - exp2f(level*S): device = raw MUFU.EX2 (<=2 ulp).  Callers may pass the device-computed
 *     per-level scales (`scale_override`) to remove this from a comparison.
 *   - __expf / __sinf: device = ex2.approx / sin.approx; here expf / sinf.
 * Pinned against: the reference's own CUDA extensions on a B200 (tests/test_ref_parity_gpu.py) and
 * the committed golden vectors generated from them (tests/golden/, oracle/make_golden.py).
 */
#include <float.h>
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#define ORACLE_F32 0
#define ORACLE_F16 1

/* ---------------------------------------------------------------------------------------------
 * IEEE binary16 <-> binary32 (round-to-nearest-even), bit-level; no reliance on _Float16.
 * --------------------------------------------------------------------------------------------- */
static float h2f(uint16_t h) {
    uint32_t sign = (uint32_t)(h & 0x8000u) << 16;
    uint32_t exp = (h >> 10) & 0x1fu;
    uint32_t man = h & 0x3ffu;
    uint32_t bits;
    if (exp == 0) {
        if (man == 0) {
            bits = sign;
        } else { /* subnormal: normalise */
            int e = -1;
            do { e++; man <<= 1; } while ((man & 0x400u) == 0);
            man &= 0x3ffu;
            bits = sign | (uint32_t)(127 - 15 - e) << 23 | (man << 13);
        }
    } else if (exp == 31) {
        bits = sign | 0x7f800000u | (man << 13);
    } else {
        bits = sign | ((exp + 127 - 15) << 23) | (man << 13);
    }
    float f;
    memcpy(&f, &bits, 4);
    return f;
}

static uint16_t f2h(float f) {
    uint32_t x;
    memcpy(&x, &f, 4);
    uint32_t sign = (x >> 16) & 0x8000u;
    uint32_t absx = x & 0x7fffffffu;
    if (absx >= 0x7f800000u) { /* inf / nan */
        return (uint16_t)(sign | 0x7c00u | ((absx > 0x7f800000u) ? 0x200u : 0));
    }
    if (absx >= 0x477ff000u) { /* rounds to >= 65520 -> inf */
        return (uint16_t)(sign | 0x7c00u);
    }
    if (absx < 0x33000001u) { /* < 2^-25 (or == 2^-25 -> ties to even 0) */
        return (uint16_t)sign;
    }
    int e = (int)(absx >> 23) - 127;
    uint32_t man = (absx & 0x7fffffu) | 0x800000u;
    int shift;
    uint32_t hexp;
    if (e < -14) { /* subnormal half */
        shift = 13 + (-14 - e);
        hexp = 0;
    } else {
        shift = 13;
        hexp = (uint32_t)(e + 15);
    }
    uint32_t hman = man >> shift;
    uint32_t rem = man & ((1u << shift) - 1);
    uint32_t half = 1u << (shift - 1);
    if (rem > half || (rem == half && (hman & 1u))) hman++;
    uint32_t out;
    if (hexp == 0) {
        out = hman; /* may carry into exponent 1: still correct */
    } else {
        out = (hexp << 10) + (hman - 0x400u); /* mantissa carry propagates into exponent */
    }
    return (uint16_t)(sign | out);
}

static float round_h(float v) { return h2f(f2h(v)); }

void oracle_f2h(const float* in, uint16_t* out, uint64_t n) { for (uint64_t i = 0; i < n; ++i) out[i] = f2h(in[i]); }
void oracle_h2f(const uint16_t* in, float* out, uint64_t n) { for (uint64_t i = 0; i < n; ++i) out[i] = h2f(in[i]); }

/* ---------------------------------------------------------------------------------------------
 * gridencoder  (gridencoder/src/gridencoder.cu)
 * --------------------------------------------------------------------------------------------- */
static const uint32_t kPrimes[7] = {1u, 2654435761u, 805459861u, 3674653429u, 2097192037u, 1434869437u, 2165219737u};

/* gridencoder.cu:35-51 */
static uint32_t fast_hash(const uint32_t* p, uint32_t D) {
    uint32_t r = 0;
    for (uint32_t i = 0; i < D; ++i) r ^= p[i] * kPrimes[i];
    return r;
}

/* gridencoder.cu:54-72 (row index only, i.e. without `* C + ch`) */
static uint32_t grid_row(uint32_t gridtype, int align_corners, uint32_t hashmap_size, uint32_t resolution,
                         const uint32_t* p, uint32_t D) {
    uint32_t stride = 1, index = 0;
    for (uint32_t d = 0; d < D && stride <= hashmap_size; d++) {
        index += p[d] * stride;
        stride *= align_corners ? resolution : (resolution + 1);
    }
    if (gridtype == 0 && stride > hashmap_size) index = fast_hash(p, D);
    return index % hashmap_size;
}

/* gridencoder.cu:125-126.  scale = fma(exp2f(level*S), H, -1) (one FFMA on the device). */
void oracle_grid_level_params(uint32_t L, float S, uint32_t H, float* scales, uint32_t* resolutions) {
    for (uint32_t level = 0; level < L; ++level) {
        float e = exp2f((float)level * S);
        float scale = fmaf(e, (float)H, -1.0f);
        scales[level] = scale;
        resolutions[level] = (uint32_t)ceilf(scale) + 1;
    }
}

static float load_elem(const void* base, uint64_t idx, int dtype) {
    return dtype == ORACLE_F16 ? h2f(((const uint16_t*)base)[idx]) : ((const float*)base)[idx];
}
static void store_elem(void* base, uint64_t idx, int dtype, float v) {
    if (dtype == ORACLE_F16) ((uint16_t*)base)[idx] = f2h(v); else ((float*)base)[idx] = v;
}

/* kernel_grid, gridencoder.cu:76-223.  out_layout 0 = [L,B,C] (reference), 1 = [B,L*C]. */
int oracle_grid_encode_forward(const float* inputs, const void* embeddings, const int* offsets, void* outputs,
                               uint32_t B, uint32_t D, uint32_t C, uint32_t L, float S, uint32_t H, void* dy_dx,
                               uint32_t gridtype, int align_corners, int dtype, int out_layout,
                               const float* scale_override) {
    if (D < 1 || D > 5 || C > 8) return -2;
    float* scales = (float*)malloc(sizeof(float) * L);
    uint32_t* ress = (uint32_t*)malloc(sizeof(uint32_t) * L);
    oracle_grid_level_params(L, S, H, scales, ress);
    if (scale_override) {
        for (uint32_t l = 0; l < L; ++l) { scales[l] = scale_override[l]; ress[l] = (uint32_t)ceilf(scales[l]) + 1; }
    }
    for (uint32_t level = 0; level < L; ++level) {
        const uint64_t tbl = (uint64_t)(uint32_t)offsets[level] * C;
        const uint32_t hashmap_size = (uint32_t)offsets[level + 1] - (uint32_t)offsets[level];
        const float scale = scales[level];
        const uint32_t resolution = ress[level];
        for (uint32_t b = 0; b < B; ++b) {
            const float* x = inputs + (uint64_t)b * D;
            const uint64_t o = out_layout ? ((uint64_t)b * L + level) * C : ((uint64_t)level * B + b) * C;
            const uint64_t jo = ((uint64_t)b * L + level) * D * C;
            int oob = 0;
            for (uint32_t d = 0; d < D; ++d) if (x[d] < 0 || x[d] > 1) oob = 1;
            if (oob) { /* :106-122 */
                for (uint32_t c = 0; c < C; ++c) store_elem(outputs, o + c, dtype, 0.f);
                if (dy_dx) for (uint32_t k = 0; k < D * C; ++k) store_elem(dy_dx, jo + k, dtype, 0.f);
                continue;
            }
            float pos[5];
            uint32_t pg[5];
            for (uint32_t d = 0; d < D; ++d) { /* :132-137 */
                float p = fmaf(x[d], scale, align_corners ? 0.0f : 0.5f);
                pg[d] = (uint32_t)floorf(p);
                pos[d] = p - (float)pg[d];
            }
            float res[8] = {0};
            for (uint32_t idx = 0; idx < (1u << D); ++idx) { /* :145-169 */
                float w = 1;
                uint32_t pl[5];
                for (uint32_t d = 0; d < D; ++d) {
                    if ((idx & (1u << d)) == 0) { w *= 1 - pos[d]; pl[d] = pg[d]; }
                    else                        { w *= pos[d];     pl[d] = pg[d] + 1; }
                }
                const uint64_t row = grid_row(gridtype, align_corners, hashmap_size, resolution, pl, D);
                for (uint32_t c = 0; c < C; ++c) {
                    const float g = load_elem(embeddings, tbl + row * C + c, dtype);
                    if (dtype == ORACLE_F16) res[c] = round_h(res[c] + round_h(w * g)); /* c10::Half += float */
                    else res[c] = fmaf(w, g, res[c]);
                }
            }
            for (uint32_t c = 0; c < C; ++c) store_elem(outputs, o + c, dtype, res[c]);

            if (dy_dx) { /* :179-222 */
                for (uint32_t gd = 0; gd < D; ++gd) {
                    float rg[8] = {0};
                    for (uint32_t idx = 0; idx < (1u << (D - 1)); ++idx) {
                        float w = scale;
                        uint32_t pl[5];
                        for (uint32_t nd = 0; nd + 1 < D; ++nd) {
                            const uint32_t d = (nd >= gd) ? (nd + 1) : nd;
                            if ((idx & (1u << nd)) == 0) { w *= 1 - pos[d]; pl[d] = pg[d]; }
                            else                         { w *= pos[d];     pl[d] = pg[d] + 1; }
                        }
                        pl[gd] = pg[gd];
                        const uint64_t left = grid_row(gridtype, align_corners, hashmap_size, resolution, pl, D);
                        pl[gd] = pg[gd] + 1;
                        const uint64_t right = grid_row(gridtype, align_corners, hashmap_size, resolution, pl, D);
                        for (uint32_t c = 0; c < C; ++c) {
                            const float gl = load_elem(embeddings, tbl + left * C + c, dtype);
                            const float gr = load_elem(embeddings, tbl + right * C + c, dtype);
                            if (dtype == ORACLE_F16) rg[c] = round_h(rg[c] + round_h(w * round_h(gr - gl)));
                            else rg[c] = fmaf(w, gr - gl, rg[c]);
                        }
                    }
                    for (uint32_t c = 0; c < C; ++c) store_elem(dy_dx, jo + gd * C + c, dtype, rg[c]);
                }
            }
        }
    }
    free(scales);
    free(ress);
    return 0;
}

/* kernel_grid_backward, gridencoder.cu:227-313.  The reference scatters with order-nondeterministic
 * atomics (fp16 table under autocast); the oracle accumulates the same per-corner addends
 * (w * grad, rounded to half first iff round_addend_to_half) into a DOUBLE table = the exact sum
 * (accumulate 0), or, like the reference's atomics in sample order, rounds the running sum to
 * float (accumulate 1) or half (accumulate 2) after every add. */
int oracle_grid_encode_backward(const void* grad, const float* inputs, const int* offsets, double* grad_table,
                                uint32_t B, uint32_t D, uint32_t C, uint32_t L, float S, uint32_t H,
                                uint32_t gridtype, int align_corners, int dtype, int grad_layout,
                                int round_addend_to_half, int accumulate, const float* scale_override) {
    if (D < 1 || D > 5 || C > 8) return -2;
    float* scales = (float*)malloc(sizeof(float) * L);
    uint32_t* ress = (uint32_t*)malloc(sizeof(uint32_t) * L);
    oracle_grid_level_params(L, S, H, scales, ress);
    if (scale_override) {
        for (uint32_t l = 0; l < L; ++l) { scales[l] = scale_override[l]; ress[l] = (uint32_t)ceilf(scales[l]) + 1; }
    }
    for (uint32_t level = 0; level < L; ++level) {
        const uint64_t tbl = (uint64_t)(uint32_t)offsets[level] * C;
        const uint32_t hashmap_size = (uint32_t)offsets[level + 1] - (uint32_t)offsets[level];
        const float scale = scales[level];
        const uint32_t resolution = ress[level];
        for (uint32_t b = 0; b < B; ++b) {
            const float* x = inputs + (uint64_t)b * D;
            int oob = 0;
            for (uint32_t d = 0; d < D; ++d) if (x[d] < 0 || x[d] > 1) oob = 1;
            if (oob) continue; /* :253-258 */
            const uint64_t go = grad_layout ? ((uint64_t)b * L + level) * C : ((uint64_t)level * B + b) * C;
            float pos[5];
            uint32_t pg[5];
            for (uint32_t d = 0; d < D; ++d) {
                float p = fmaf(x[d], scale, align_corners ? 0.0f : 0.5f);
                pg[d] = (uint32_t)floorf(p);
                pos[d] = p - (float)pg[d];
            }
            for (uint32_t idx = 0; idx < (1u << D); ++idx) {
                float w = 1;
                uint32_t pl[5];
                for (uint32_t d = 0; d < D; ++d) {
                    if ((idx & (1u << d)) == 0) { w *= 1 - pos[d]; pl[d] = pg[d]; }
                    else                        { w *= pos[d];     pl[d] = pg[d] + 1; }
                }
                const uint64_t row = grid_row(gridtype, align_corners, hashmap_size, resolution, pl, D);
                for (uint32_t c = 0; c < C; ++c) {
                    float v = w * load_elem(grad, go + c, dtype);
                    if (round_addend_to_half) v = round_h(v); /* :302 */
                    double* t = grad_table + tbl + row * C + c;
                    if (accumulate == 1)      *t = (double)((float)*t + v);
                    else if (accumulate == 2) *t = (double)round_h((float)*t + v);
                    else                      *t += (double)v;
                }
            }
        }
    }
    free(scales);
    free(ress);
    return 0;
}

/* kernel_input_backward, gridencoder.cu:317-342 */
void oracle_grid_input_backward(const void* grad, const void* dy_dx, void* grad_inputs, uint32_t B, uint32_t D,
                                uint32_t C, uint32_t L, int dtype, int grad_layout) {
    for (uint32_t b = 0; b < B; ++b)
        for (uint32_t d = 0; d < D; ++d) {
            float acc = 0;
            for (uint32_t l = 0; l < L; ++l)
                for (uint32_t c = 0; c < C; ++c) {
                    const uint64_t go = grad_layout ? ((uint64_t)b * L + l) * C + c : ((uint64_t)l * B + b) * C + c;
                    const float g = load_elem(grad, go, dtype);
                    const float j = load_elem(dy_dx, (((uint64_t)b * L + l) * D + d) * C + c, dtype);
                    if (dtype == ORACLE_F16) acc = round_h(acc + round_h(g * j));
                    else acc = fmaf(g, j, acc);
                }
            store_elem(grad_inputs, (uint64_t)b * D + d, dtype, acc);
        }
}

/* ---------------------------------------------------------------------------------------------
 * raymarching  (raymarching/src/raymarching.cu)
 * --------------------------------------------------------------------------------------------- */
static float clampf(float x, float lo, float hi) { return fminf(hi, fmaxf(lo, x)); } /* :34 */

static uint32_t expand_bits(uint32_t v) { /* :56-63 */
    v = (v * 0x00010001u) & 0xFF0000FFu;
    v = (v * 0x00000101u) & 0x0F00F00Fu;
    v = (v * 0x00000011u) & 0xC30C30C3u;
    v = (v * 0x00000005u) & 0x49249249u;
    return v;
}
static uint32_t morton3d(uint32_t x, uint32_t y, uint32_t z) { /* :65-71 */
    return expand_bits(x) | (expand_bits(y) << 1) | (expand_bits(z) << 2);
}
static uint32_t morton3d_invert(uint32_t x) { /* :73-81 */
    x = x & 0x49249249u;
    x = (x | (x >> 2)) & 0xc30c30c3u;
    x = (x | (x >> 4)) & 0x0f00f00fu;
    x = (x | (x >> 8)) & 0xff0000ffu;
    x = (x | (x >> 16)) & 0x0000ffffu;
    return x;
}

static int mip_from_pos(float x, float y, float z, float max_cascade) { /* :42-47 */
    const float mx = fmaxf(fabsf(x), fmaxf(fabsf(y), fabsf(z)));
    int e;
    frexpf(mx, &e);
    return (int)fminf(max_cascade - 1, fmaxf(0, (float)e));
}
static int mip_from_dt(float dt, float H, float max_cascade) { /* :49-54; `* 0.5` in double is exact */
    const float mx = (float)((double)(dt * H) * 0.5);
    int e;
    frexpf(mx, &e);
    return (int)fminf(max_cascade - 1, fmaxf(0, (float)e));
}

/* kernel_near_far_from_aabb, :92-145 */
void oracle_near_far_from_aabb(const float* rays_o, const float* rays_d, const float* aabb, uint32_t N,
                               float min_near, float* nears, float* fars) {
    for (uint32_t n = 0; n < N; ++n) {
        const float ox = rays_o[n * 3], oy = rays_o[n * 3 + 1], oz = rays_o[n * 3 + 2];
        const float rdx = 1 / rays_d[n * 3], rdy = 1 / rays_d[n * 3 + 1], rdz = 1 / rays_d[n * 3 + 2];
        float near = (aabb[0] - ox) * rdx, far = (aabb[3] - ox) * rdx, t;
        if (near > far) { t = near; near = far; far = t; }
        float near_y = (aabb[1] - oy) * rdy, far_y = (aabb[4] - oy) * rdy;
        if (near_y > far_y) { t = near_y; near_y = far_y; far_y = t; }
        if (near > far_y || near_y > far) { nears[n] = fars[n] = FLT_MAX; continue; }
        if (near_y > near) near = near_y;
        if (far_y < far) far = far_y;
        float near_z = (aabb[2] - oz) * rdz, far_z = (aabb[5] - oz) * rdz;
        if (near_z > far_z) { t = near_z; near_z = far_z; far_z = t; }
        if (near > far_z || near_z > far) { nears[n] = fars[n] = FLT_MAX; continue; }
        if (near_z > near) near = near_z;
        if (far_z < far) far = far_z;
        if (near < min_near) near = min_near;
        nears[n] = near;
        fars[n] = far;
    }
}

/* kernel_sph_from_ray, :163-198 */
void oracle_sph_from_ray(const float* rays_o, const float* rays_d, float radius, uint32_t N, float* coords) {
    for (uint32_t n = 0; n < N; ++n) {
        const float ox = rays_o[n * 3], oy = rays_o[n * 3 + 1], oz = rays_o[n * 3 + 2];
        const float dx = rays_d[n * 3], dy = rays_d[n * 3 + 1], dz = rays_d[n * 3 + 2];
        const float A = fmaf(dz, dz, fmaf(dy, dy, dx * dx));
        const float Bh = fmaf(oz, dz, fmaf(oy, dy, ox * dx));
        const float Cq = fmaf(-radius, radius, fmaf(oz, oz, fmaf(oy, oy, ox * ox)));
        const float t = (-Bh + sqrtf(fmaf(Bh, Bh, -(A * Cq)))) / A;
        const float x = fmaf(t, dx, ox), y = fmaf(t, dy, oy), z = fmaf(t, dz, oz);
        const float theta = atan2f(sqrtf(fmaf(z, z, x * x)), y);
        const float phi = atan2f(z, x);
        coords[n * 2] = fmaf(2 * theta, 0.3183098861837907f, -1.0f);
        coords[n * 2 + 1] = phi * 0.3183098861837907f;
    }
}

void oracle_morton3D(const int* coords, uint32_t N, int* indices) { /* :214-226 */
    for (uint32_t n = 0; n < N; ++n)
        indices[n] = (int)morton3d((uint32_t)coords[n * 3], (uint32_t)coords[n * 3 + 1], (uint32_t)coords[n * 3 + 2]);
}
void oracle_morton3D_invert(const int* indices, uint32_t N, int* coords) { /* :237-254 */
    for (uint32_t n = 0; n < N; ++n) {
        const int ind = indices[n];
        coords[n * 3] = (int)morton3d_invert((uint32_t)(ind >> 0));
        coords[n * 3 + 1] = (int)morton3d_invert((uint32_t)(ind >> 1));
        coords[n * 3 + 2] = (int)morton3d_invert((uint32_t)(ind >> 2));
    }
}
void oracle_packbits(const float* grid, uint32_t N, float thresh, uint8_t* bitfield) { /* :268-289 */
    for (uint32_t n = 0; n < N; ++n) {
        uint8_t bits = 0;
        for (int i = 0; i < 8; ++i) bits |= (grid[(uint64_t)n * 8 + i] > thresh) ? (uint8_t)(1u << i) : 0;
        bitfield[n] = bits;
    }
}

typedef struct {
    const uint8_t* grid;
    float bound, dt_gamma, dt_min, dt_max, rH, H3, Hf, Cf, Hm1;
    uint32_t H;
} march_consts;

static march_consts make_consts(const uint8_t* grid, float bound, float dt_gamma, uint32_t max_steps, uint32_t C,
                                uint32_t H) {
    march_consts p;
    p.grid = grid; p.bound = bound; p.dt_gamma = dt_gamma;
    p.dt_min = (2 * 1.7320508075688772f) / (float)max_steps;               /* :345 */
    p.dt_max = ((2 * 1.7320508075688772f) * (float)(1 << (C - 1))) / (float)H; /* :346 */
    p.rH = 1 / (float)H;
    p.H3 = (float)(H * H * H);
    p.Hf = (float)H; p.Cf = (float)C; p.Hm1 = (float)(H - 1); p.H = H;
    return p;
}

/* One iteration of the marching loop (:360-399).  Returns 1 when the cell is occupied (x,y,z,dt set;
 * the caller advances t by dt), else advances t past the empty cell and returns 0. */
static int march_probe(const march_consts* p, float ox, float oy, float oz, float dx, float dy, float dz, float rdx,
                       float rdy, float rdz, float* t, float* px, float* py, float* pz, float* pdt) {
    const float x = clampf(fmaf(*t, dx, ox), -p->bound, p->bound);
    const float y = clampf(fmaf(*t, dy, oy), -p->bound, p->bound);
    const float z = clampf(fmaf(*t, dz, oz), -p->bound, p->bound);
    const float dt = clampf(*t * p->dt_gamma, p->dt_min, p->dt_max);
    const int a = mip_from_pos(x, y, z, p->Cf), b = mip_from_dt(dt, p->Hf, p->Cf);
    const int level = a > b ? a : b;
    const float mip_bound = fminf(ldexpf(1.0f, level), p->bound);
    const float mip_rbound = 1 / mip_bound;
    /* `0.5 * (x * mip_rbound + 1) * H`: fp32 fma, then double multiplies, then round to float (:374) */
    const int nx = (int)clampf((float)(0.5 * (double)fmaf(x, mip_rbound, 1.0f) * (double)p->H), 0.0f, p->Hm1);
    const int ny = (int)clampf((float)(0.5 * (double)fmaf(y, mip_rbound, 1.0f) * (double)p->H), 0.0f, p->Hm1);
    const int nz = (int)clampf((float)(0.5 * (double)fmaf(z, mip_rbound, 1.0f) * (double)p->H), 0.0f, p->Hm1);
    const uint32_t index = (uint32_t)fmaf((float)level, p->H3, (float)morton3d((uint32_t)nx, (uint32_t)ny, (uint32_t)nz));
    const int occ = p->grid[index / 8] & (1 << (index % 8));
    *px = x; *py = y; *pz = z; *pdt = dt;
    if (occ) return 1;
    /* :390-398 */
    const float sx = copysignf(1.0f, dx), sy = copysignf(1.0f, dy), sz = copysignf(1.0f, dz);
    const float tx = fmaf(fmaf(fmaf(0.5f, sx, (float)nx + 0.5f) * p->rH, 2.0f, -1.0f), mip_bound, -x) * rdx;
    const float ty = fmaf(fmaf(fmaf(0.5f, sy, (float)ny + 0.5f) * p->rH, 2.0f, -1.0f), mip_bound, -y) * rdy;
    const float tz = fmaf(fmaf(fmaf(0.5f, sz, (float)nz + 0.5f) * p->rH, 2.0f, -1.0f), mip_bound, -z) * rdz;
    const float tt = *t + fmaxf(0.0f, fminf(tx, fminf(ty, tz)));
    do {
        *t += clampf(*t * p->dt_gamma, p->dt_min, p->dt_max);
    } while (*t < tt);
    return 0;
}

/* kernel_march_rays_train, :312-480, with the reference's atomic slot allocation replaced by its
 * canonical (ray-ordered) outcome: rays[n] = (n, exclusive prefix of counts + counter[0], count). */
void oracle_march_rays_train(const float* rays_o, const float* rays_d, const uint8_t* grid, float bound,
                             float dt_gamma, uint32_t max_steps, uint32_t N, uint32_t C, uint32_t H, uint32_t M,
                             const float* nears, const float* fars, float* xyzs, float* dirs, float* deltas,
                             int* rays, int* counter, const float* noises) {
    const march_consts p = make_consts(grid, bound, dt_gamma, max_steps, C, H);
    uint32_t point_index = (uint32_t)counter[0];
    for (uint32_t n = 0; n < N; ++n) {
        const float ox = rays_o[n * 3], oy = rays_o[n * 3 + 1], oz = rays_o[n * 3 + 2];
        const float dx = rays_d[n * 3], dy = rays_d[n * 3 + 1], dz = rays_d[n * 3 + 2];
        const float rdx = 1 / dx, rdy = 1 / dy, rdz = 1 / dz;
        const float near = nears[n], far = fars[n], noise = noises[n];
        float t0 = near;
        t0 = fmaf(clampf(t0 * dt_gamma, p.dt_min, p.dt_max), noise, t0); /* :351 */
        float t = t0, x, y, z, dt;
        uint32_t num_steps = 0;
        while (t < far && num_steps < max_steps) {
            if (march_probe(&p, ox, oy, oz, dx, dy, dz, rdx, rdy, rdz, &t, &x, &y, &z, &dt)) { num_steps++; t += dt; }
        }
        rays[n * 3] = (int)n;
        rays[n * 3 + 1] = (int)point_index;
        rays[n * 3 + 2] = (int)num_steps;
        const uint32_t offset = point_index;
        point_index += num_steps;
        if (num_steps == 0) continue;
        if (offset + num_steps > M) continue; /* :416 */
        t = t0;
        uint32_t step = 0;
        float last_t = t;
        float* px = xyzs + (uint64_t)offset * 3;
        float* pd = dirs + (uint64_t)offset * 3;
        float* pl = deltas + (uint64_t)offset * 2;
        while (t < far && step < num_steps) {
            if (march_probe(&p, ox, oy, oz, dx, dy, dz, rdx, rdy, rdz, &t, &x, &y, &z, &dt)) {
                px[0] = x; px[1] = y; px[2] = z;
                pd[0] = dx; pd[1] = dy; pd[2] = dz;
                t += dt;
                pl[0] = dt;
                pl[1] = t - last_t;
                last_t = t;
                px += 3; pd += 3; pl += 2;
                step++;
            }
        }
    }
    counter[0] = (int)point_index;
    counter[1] += (int)N;
}

/* kernel_composite_rays_train_forward, :501-577 */
void oracle_composite_rays_train_forward(const float* sigmas, const float* rgbs, const float* deltas,
                                         const int* rays, uint32_t M, uint32_t N, float T_thresh,
                                         float* weights_sum, float* depth, float* image) {
    for (uint32_t n = 0; n < N; ++n) {
        const uint32_t index = (uint32_t)rays[n * 3], offset = (uint32_t)rays[n * 3 + 1], num_steps = (uint32_t)rays[n * 3 + 2];
        if (num_steps == 0 || offset + num_steps > M) {
            weights_sum[index] = 0; depth[index] = 0;
            image[index * 3] = image[index * 3 + 1] = image[index * 3 + 2] = 0;
            continue;
        }
        const float* s = sigmas + offset;
        const float* c = rgbs + (uint64_t)offset * 3;
        const float* dl = deltas + (uint64_t)offset * 2;
        float T = 1.0f, r = 0, g = 0, b = 0, ws = 0, t = 0, d = 0;
        for (uint32_t step = 0; step < num_steps; ++step) {
            const float alpha = 1.0f - expf(-s[0] * dl[0]);
            const float weight = alpha * T;
            r = fmaf(weight, c[0], r);
            g = fmaf(weight, c[1], g);
            b = fmaf(weight, c[2], b);
            t += dl[1];
            d = fmaf(weight, t, d);
            ws += weight;
            T *= 1.0f - alpha;
            if (T < T_thresh) break;
            s++; c += 3; dl += 2;
        }
        weights_sum[index] = ws; depth[index] = d;
        image[index * 3] = r; image[index * 3 + 1] = g; image[index * 3 + 2] = b;
    }
}

/* kernel_composite_rays_train_backward, :602-682.  grad_sigmas / grad_rgbs must be zero-filled. */
void oracle_composite_rays_train_backward(const float* grad_weights_sum, const float* grad_image,
                                          const float* sigmas, const float* rgbs, const float* deltas,
                                          const int* rays, const float* weights_sum, const float* image, uint32_t M,
                                          uint32_t N, float T_thresh, float* grad_sigmas, float* grad_rgbs) {
    for (uint32_t n = 0; n < N; ++n) {
        const uint32_t index = (uint32_t)rays[n * 3], offset = (uint32_t)rays[n * 3 + 1], num_steps = (uint32_t)rays[n * 3 + 2];
        if (num_steps == 0 || offset + num_steps > M) continue;
        const float gws = grad_weights_sum[index];
        const float* gi = grad_image + (uint64_t)index * 3;
        const float ws_final = weights_sum[index];
        const float r_final = image[index * 3], g_final = image[index * 3 + 1], b_final = image[index * 3 + 2];
        const float* s = sigmas + offset;
        const float* c = rgbs + (uint64_t)offset * 3;
        const float* dl = deltas + (uint64_t)offset * 2;
        float* gs = grad_sigmas + offset;
        float* gc = grad_rgbs + (uint64_t)offset * 3;
        float T = 1.0f, r = 0, g = 0, b = 0, ws = 0;
        for (uint32_t step = 0; step < num_steps; ++step) {
            const float alpha = 1.0f - expf(-s[0] * dl[0]);
            const float weight = alpha * T;
            r = fmaf(weight, c[0], r);
            g = fmaf(weight, c[1], g);
            b = fmaf(weight, c[2], b);
            ws += weight;
            T *= 1.0f - alpha;
            gc[0] = gi[0] * weight; gc[1] = gi[1] * weight; gc[2] = gi[2] * weight;
            /* :662-667, evaluated in double here (the device's own contraction order only changes the last ulp) */
            gs[0] = (float)((double)dl[0] * ((double)gi[0] * ((double)T * c[0] - ((double)r_final - r)) +
                                             (double)gi[1] * ((double)T * c[1] - ((double)g_final - g)) +
                                             (double)gi[2] * ((double)T * c[2] - ((double)b_final - b)) +
                                             (double)gws * (1.0 - (double)ws_final)));
            if (T < T_thresh) break;
            s++; c += 3; dl += 2; gs++; gc += 3;
        }
    }
}

/* kernel_march_rays, :701-805 (inference).  Outputs must be zero-filled. */
void oracle_march_rays(uint32_t n_alive, uint32_t n_step, const int* rays_alive, const float* rays_t,
                       const float* rays_o, const float* rays_d, float bound, float dt_gamma, uint32_t max_steps,
                       uint32_t C, uint32_t H, const uint8_t* grid, const float* nears, const float* fars, float* xyzs,
                       float* dirs, float* deltas, const float* noises) {
    (void)nears;
    const march_consts p = make_consts(grid, bound, dt_gamma, max_steps, C, H);
    for (uint32_t n = 0; n < n_alive; ++n) {
        const int index = rays_alive[n];
        const float noise = noises[n];
        const float ox = rays_o[index * 3], oy = rays_o[index * 3 + 1], oz = rays_o[index * 3 + 2];
        const float dx = rays_d[index * 3], dy = rays_d[index * 3 + 1], dz = rays_d[index * 3 + 2];
        const float rdx = 1 / dx, rdy = 1 / dy, rdz = 1 / dz;
        float t = rays_t[index];
        const float far = fars[index];
        t = fmaf(clampf(t * dt_gamma, p.dt_min, p.dt_max), noise, t); /* :746 */
        float last_t = t, x, y, z, dt;
        float* px = xyzs + (uint64_t)n * n_step * 3;
        float* pd = dirs + (uint64_t)n * n_step * 3;
        float* pl = deltas + (uint64_t)n * n_step * 2;
        uint32_t step = 0;
        while (t < far && step < n_step) {
            if (march_probe(&p, ox, oy, oz, dx, dy, dz, rdx, rdy, rdz, &t, &x, &y, &z, &dt)) {
                px[0] = x; px[1] = y; px[2] = z;
                pd[0] = dx; pd[1] = dy; pd[2] = dz;
                t += dt;
                pl[0] = dt;
                pl[1] = t - last_t;
                last_t = t;
                px += 3; pd += 3; pl += 2;
                step++;
            }
        }
    }
}

/* kernel_composite_rays, :819-905 (inference, in place) */
void oracle_composite_rays(uint32_t n_alive, uint32_t n_step, float T_thresh, int* rays_alive, float* rays_t,
                           const float* sigmas, const float* rgbs, const float* deltas, float* weights_sum,
                           float* depth, float* image) {
    for (uint32_t n = 0; n < n_alive; ++n) {
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
            const float alpha = 1.0f - expf(-s[0] * dl[0]);
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
}

/* `rays_alive = rays_alive[rays_alive >= 0]`, nerf/renderer.py:529 */
uint32_t oracle_compact_alive(const int* rays_alive, uint32_t n, int* out) {
    uint32_t k = 0;
    for (uint32_t i = 0; i < n; ++i) if (rays_alive[i] >= 0) out[k++] = rays_alive[i];
    return k;
}

/* ---------------------------------------------------------------------------------------------
 * freqencoder  (freqencoder/src/freqencoder.cu)
 * --------------------------------------------------------------------------------------------- */
void oracle_freq_encode_forward(const float* inputs, uint32_t B, uint32_t D, uint32_t deg, uint32_t C, float* outputs) {
    (void)deg;
    for (uint32_t b = 0; b < B; ++b)
        for (uint32_t c = 0; c < C; ++c) { /* :30-58 */
            const float* in = inputs + (uint64_t)b * D;
            float v;
            if (c < D) {
                v = in[c];
            } else {
                const uint32_t col = c / D - 1, d = c % D, freq = col / 2;
                const float phase_shift = (float)(col % 2) * (3.141592653589793f / 2);
                v = sinf(ldexpf(in[d], (int)freq) + phase_shift);
            }
            outputs[(uint64_t)b * C + c] = v;
        }
}

void oracle_freq_encode_backward(const float* grad, const float* outputs, uint32_t B, uint32_t D, uint32_t deg,
                                 uint32_t C, float* grad_inputs) {
    for (uint32_t b = 0; b < B; ++b)
        for (uint32_t d = 0; d < D; ++d) { /* :63-94 */
            const float* g = grad + (uint64_t)b * C;
            const float* o = outputs + (uint64_t)b * C;
            float result = g[d];
            g += D; o += D;
            for (uint32_t f = 0; f < deg; ++f) {
                result = fmaf(ldexpf(1.0f, (int)f), fmaf(g[d], o[D + d], -(g[D + d] * o[d])), result);
                g += 2 * D; o += 2 * D;
            }
            grad_inputs[(uint64_t)b * D + d] = result;
        }
}

/* ---------------------------------------------------------------------------------------------
 * occupancy-grid update  (NeRFRenderer.update_extra_state, nerf/renderer.py:562-613)
 * --------------------------------------------------------------------------------------------- */
/* renderer.py:581-593 for one cascade; noise in linear (x,y,z) cell order, output in Morton order.
 * torch's CUDA `tensor / python_scalar` multiplies by the fp32 reciprocal, reproduced here. */
void oracle_occupancy_cell_points(uint32_t H, float cell_scale, float half_cell, const float* noise, float* xyzs) {
    const uint32_t n_cells = H * H * H;
    const float inv_hm1 = 1.0f / (float)(H - 1);
    for (uint32_t m = 0; m < n_cells; ++m) {
        const uint32_t c[3] = {morton3d_invert(m), morton3d_invert(m >> 1), morton3d_invert(m >> 2)};
        const uint64_t lin = ((uint64_t)c[0] * H + c[1]) * H + c[2];
        for (int a = 0; a < 3; ++a) {
            const float centre = ((2.0f * (float)c[a]) * inv_hm1) - 1.0f;
            const float scaled = centre * cell_scale;
            const float jitter = ((noise[lin * 3 + a] * 2.0f) - 1.0f) * half_cell;
            xyzs[(uint64_t)m * 3 + a] = scaled + jitter;
        }
    }
}

/* renderer.py:600-607: EMA-max over valid cells, mean, threshold = python min(mean, thresh), packbits. */
void oracle_update_density_grid(float* grid, const float* tmp_grid, uint32_t n_cells, float decay,
                                float density_thresh, float* mean_out, uint8_t* bitfield) {
    double sum = 0.0;
    uint64_t cnt = 0;
    for (uint32_t i = 0; i < n_cells; ++i) {
        float g = grid[i];
        if (g >= 0) {
            const float a = g * decay, b = tmp_grid[i];
            g = (a != a || b != b) ? NAN : fmaxf(a, b);
            grid[i] = g;
            sum += (double)g;
            cnt++;
        }
    }
    const float mean = (float)(sum / (double)cnt);
    const float thresh = (density_thresh < mean) ? density_thresh : mean;
    *mean_out = mean;
    oracle_packbits(grid, n_cells / 8, thresh, bitfield);
}

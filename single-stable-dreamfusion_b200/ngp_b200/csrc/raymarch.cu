// Occupancy-grid ray marching and volume compositing for sm_100a.
//
// Behavioural contract: raymarching/src/raymarching.cu of the reference.  Sample positions, step
// sizes, per-ray counts and bitfields must be BIT-EXACT with it, so every floating-point
// expression that decides a sample keeps the reference's operand order (cited inline); the
// parallel structure is new:
//   * training march = count pass -> block-wide exclusive scan in ray order -> write pass, which
//     replaces the reference's two global atomics per ray (raymarching.cu:405-406) and makes the
//     sample layout deterministic (ray n owns rows [offset_n, offset_n + count_n));
//   * compositing runs one WARP per ray: 32 samples per step, alpha/exp evaluated in parallel, the
//     transmittance chain rebuilt with warp shuffles in the reference's multiplication order (so
//     the early-termination decision is the reference's), colour/weight sums by warp reduction.
#include <float.h>
#include <stdio.h>
#include <string.h>

#include "common.cuh"

namespace ngp {
namespace march {

// test / profiling switch (ngp_march_set_option 0): 1 = the reference's decomposition, one thread per ray
bool g_thread_per_ray = false;
bool g_infer_warp_march = false;  // ngp_march_set_option 1: warp-per-ray walk for one-sample inference calls
// ngp_march_set_option 2: launches of at least this many rays with dt_gamma == 0 use the thread-per-ray walk with closed-form
// lattice jumps (fewer instructions, but a ray is one serial ~0.2 ms chain); smaller ones keep the warp-per-ray walk.
// 0 = never (the default: measured 0.314 vs 0.310 ms at 32768 rays, 0.232 vs 0.066 ms at 4096).
uint32_t g_thread_march_min_rays = 0;

NGP_DEVINL float clampf(float x, float lo, float hi) { return fminf(hi, fmaxf(lo, x)); }  // raymarching.cu:34

// 10-bit-per-axis Morton interleave (raymarching.cu:56-71): the classic magic-multiply spread.
NGP_DEVINL uint32_t spread3(uint32_t v) {
    v = (v * 0x00010001u) & 0xFF0000FFu;
    v = (v * 0x00000101u) & 0x0F00F00Fu;
    v = (v * 0x00000011u) & 0xC30C30C3u;
    v = (v * 0x00000005u) & 0x49249249u;
    return v;
}
NGP_DEVINL uint32_t morton_encode(uint32_t x, uint32_t y, uint32_t z) {
    return spread3(x) | (spread3(y) << 1) | (spread3(z) << 2);
}
NGP_DEVINL uint32_t compact3(uint32_t x) {  // raymarching.cu:73-81
    x &= 0x49249249u;
    x = (x | (x >> 2)) & 0xc30c30c3u;
    x = (x | (x >> 4)) & 0x0f00f00fu;
    x = (x | (x >> 8)) & 0xff0000ffu;
    x = (x | (x >> 16)) & 0x0000ffffu;
    return x;
}

// Cascade level of a position / of a step size (raymarching.cu:42-54).  frexpf exponent, clamped.
NGP_DEVINL int level_from_pos(float x, float y, float z, float n_cascades) {
    const float mx = fmaxf(fabsf(x), fmaxf(fabsf(y), fabsf(z)));
    int e;
    frexpf(mx, &e);
    return (int)fminf(n_cascades - 1, fmaxf(0.f, (float)e));
}
NGP_DEVINL int level_from_dt(float dt, float H, float n_cascades) {
    const float mx = (dt * H) * 0.5f;  // the reference's `* 0.5` is a double multiply by a power of two: exact
    int e;
    frexpf(mx, &e);
    return (int)fminf(n_cascades - 1, fmaxf(0.f, (float)e));
}

struct MarchParams {
    const uint8_t* __restrict__ grid;
    float bound, dt_gamma, dt_min, dt_max, rH, H3, Hf, Cf, Hm1;
    // one cascade (bound <= 1, the -O default): the level is 0 for every position and every step size, so the cascade
    // selection (two frexpf, a scalbnf, a division) collapses to these two per-launch constants - same values, hoisted
    bool single;
    float mip_bound0, mip_rbound0;
    // optional shared-memory table spread3(i), i < H (the warp-per-ray marcher: its LSU is idle, its issue slots are not -
    // three LDS replace 24 multiply / mask instructions of the bit interleave)
    const uint32_t* lut;
};

NGP_DEVINL MarchParams make_params(const uint8_t* grid, float bound, float dt_gamma, uint32_t max_steps, uint32_t C,
                                   uint32_t H) {
    MarchParams p;
    p.grid = grid;
    p.bound = bound;
    p.dt_gamma = dt_gamma;
    p.dt_min = 2 * 1.7320508075688772f / max_steps;            // raymarching.cu:345
    p.dt_max = 2 * 1.7320508075688772f * (1 << (C - 1)) / H;   // raymarching.cu:346
    p.rH = 1 / (float)H;
    p.H3 = H * H * H;                                          // uint32 product converted to float (:339)
    p.Hf = (float)H;
    p.Cf = (float)C;
    p.Hm1 = (float)(H - 1);
    p.lut = nullptr;
    p.single = (C == 1);
    p.mip_bound0 = fminf(scalbnf(1.0f, 0), bound);
    p.mip_rbound0 = 1 / p.mip_bound0;
    // (opaque to the optimiser: otherwise it merges this division with classify()'s per-point `1 / mip_bound` of the
    //  multi-cascade path and re-evaluates the reciprocal for every lattice point of single-cascade scenes too)
    asm volatile("" : "+f"(p.mip_rbound0));
    return p;
}

struct Ray {
    float ox, oy, oz, dx, dy, dz, rdx, rdy, rdz;
};
NGP_DEVINL Ray load_ray(const float* __restrict__ rays_o, const float* __restrict__ rays_d, uint32_t n) {
    Ray r;
    r.ox = rays_o[n * 3 + 0]; r.oy = rays_o[n * 3 + 1]; r.oz = rays_o[n * 3 + 2];
    r.dx = rays_d[n * 3 + 0]; r.dy = rays_d[n * 3 + 1]; r.dz = rays_d[n * 3 + 2];
    r.rdx = 1 / r.dx; r.rdy = 1 / r.dy; r.rdz = 1 / r.dz;  // IEEE division: this TU is never built with fast-math
    return r;
}

// Cell under parameter t (raymarching.cu:360-379): sample position, step size, cascade and occupancy bit.
struct Cell {
    float x, y, z, dt, mip_bound;
    int nx, ny, nz;
    bool occ;
};
NGP_DEVINL Cell classify(const MarchParams& p, const Ray& r, float t, uint32_t* cached_index = nullptr, bool* cached_occ = nullptr) {
    Cell c;
    c.x = clampf(r.ox + t * r.dx, -p.bound, p.bound);
    c.y = clampf(r.oy + t * r.dy, -p.bound, p.bound);
    c.z = clampf(r.oz + t * r.dz, -p.bound, p.bound);
    c.dt = clampf(t * p.dt_gamma, p.dt_min, p.dt_max);

    int level = 0;
    float mip_rbound = p.mip_rbound0;
    c.mip_bound = p.mip_bound0;
    if (!p.single) {   // (warp-uniform)
        level = max(level_from_pos(c.x, c.y, c.z, p.Cf), level_from_dt(c.dt, p.Hf, p.Cf));
        c.mip_bound = fminf(scalbnf(1.0f, level), p.bound);
        mip_rbound = 1 / c.mip_bound;
    }

    // `0.5 * (x*rb + 1) * H` is evaluated in double by the reference; both factors are exactly
    // representable so the float product below rounds to the same value (DESIGN.md "marcher").
    c.nx = (int)clampf(__fmul_rn(0.5f * (c.x * mip_rbound + 1), p.Hf), 0.0f, p.Hm1);
    c.ny = (int)clampf(__fmul_rn(0.5f * (c.y * mip_rbound + 1), p.Hf), 0.0f, p.Hm1);
    c.nz = (int)clampf(__fmul_rn(0.5f * (c.z * mip_rbound + 1), p.Hf), 0.0f, p.Hm1);

    const uint32_t morton = p.lut ? (p.lut[c.nx] | (p.lut[c.ny] << 1) | (p.lut[c.nz] << 2)) : morton_encode(c.nx, c.ny, c.nz);
    const uint32_t index = level * p.H3 + morton;  // float arithmetic, as in :378
    if (cached_index) {       // (serial walks: the previous point's cell is usually this point's cell)
        if (index != *cached_index) { *cached_index = index; *cached_occ = p.grid[index / 8] & (1 << (index % 8)); }
        c.occ = *cached_occ;
        return c;
    }
    c.occ = p.grid[index / 8] & (1 << (index % 8));
    return c;
}
// Parameter at which the ray leaves the (empty) cell (raymarching.cu:390-394).
NGP_DEVINL float cell_exit(const MarchParams& p, const Ray& r, const Cell& c, float t) {
    const float tx = (((c.nx + 0.5f + 0.5f * copysignf(1.0f, r.dx)) * p.rH * 2 - 1) * c.mip_bound - c.x) * r.rdx;
    const float ty = (((c.ny + 0.5f + 0.5f * copysignf(1.0f, r.dy)) * p.rH * 2 - 1) * c.mip_bound - c.y) * r.rdy;
    const float tz = (((c.nz + 0.5f + 0.5f * copysignf(1.0f, r.dz)) * p.rH * 2 - 1) * c.mip_bound - c.z) * r.rdz;
    return t + fmaxf(0.0f, fminf(tx, fminf(ty, tz)));
}

// One iteration of the reference's serial loop (raymarching.cu:360-399): either report an occupied sample
// (returns true; x,y,z,dt valid) or step the fixed t-lattice until the empty cell has been crossed (:396-398).
NGP_DEVINL bool probe(const MarchParams& p, const Ray& r, float& t, float& x, float& y, float& z, float& dt) {
    const Cell c = classify(p, r, t);
    x = c.x; y = c.y; z = c.z; dt = c.dt;
    if (c.occ) return true;
    const float tt = cell_exit(p, r, c, t);
    do {
        t += clampf(t * p.dt_gamma, p.dt_min, p.dt_max);
    } while (t < tt);
    return false;
}

// Per-binade constants of the jump, recomputed only when t enters another binade (at most five times per ray)
struct Binade {
    int key;        // sign + exponent bits of the t they were derived for (-1: none yet)
    uint32_t m;     // lattice step in units of the binade's ulp
    float inv_m;
    bool ok;        // closed form applies (no tie, m >= 1, sane exponent)
};
NGP_DEVINL void binade_setup(int tb, float dtc, Binade& b) {
    b.key = tb >> 23;
    b.ok = false; b.m = 1u; b.inv_m = 1.f;
    const int e = ((tb >> 23) & 0xff) - 127;
    if (tb > 0 && e > -100 && e < 100) {
        const float rr = scalbnf(dtc, 23 - e);              // dt / u, exact
        const float fl = floorf(rr);
        if (rr < 4194304.f && (rr - fl) != 0.5f && rr >= 0.5f) {
            b.m = (uint32_t)__float2int_rn(rr);
            b.inv_m = __frcp_rn((float)b.m);
            b.ok = true;
        }
    }
}
// floor(a / m) and ceil(a / m) for a < 2^23 through one float multiply and exact integer fix-ups (the estimate is within
// one of the quotient): the 32-bit integer division they replace is ~20 dependent instructions on the ray's serial chain
NGP_DEVINL uint32_t floor_div(uint32_t a, uint32_t m, float inv_m) {
    uint32_t q = (uint32_t)(__uint2float_rz(a) * inv_m);
    if (q * m > a) --q;
    if (q * m > a) --q;
    if ((q + 1u) * m <= a) ++q;
    return q;
}
NGP_DEVINL uint32_t ceil_div(uint32_t a, uint32_t m, float inv_m) {
    const uint32_t f = floor_div(a, m, inv_m);
    return f * m == a ? f : f + 1u;
}
// -------------------------------------------------------------------------------------------------
// Warp-per-ray walk.  The candidate parameters of a ray form a FIXED lattice T_0 = t0,
// T_{k+1} = T_k + clamp(T_k * dt_gamma, dt_min, dt_max): both branches of the reference loop advance t by exactly
// that increment, occupancy only decides which lattice points are visited (an empty cell jumps to the first T_j >=
// its exit parameter).  So 32 lanes evaluate 32 consecutive lattice points (each lane re-doing the serial additions
// from the window base, which keeps every T bit-identical), classify their cells in parallel, turn "where do I go
// next" into a pointer per lane and resolve the visited chain with 5 rounds of pointer doubling.
// Returns the number of emitted samples (<= limit); WRITE == 1 stores them at rows [0, n) of the given pointers,
// WRITE == 2 only records their lattice parameters T in `xyzs` (a shared-memory buffer of `limit` floats: position, step
// and delta of a sample are functions of T and of the previous sample's T, see march_packed_kernel).
// -------------------------------------------------------------------------------------------------
template <int WRITE>
NGP_DEVINL uint32_t walk_ray_warp(const MarchParams& p, const Ray& r, float t0, float far, uint32_t limit, int lane,
                                  float* __restrict__ xyzs, float* __restrict__ dirs, float* __restrict__ deltas) {
    constexpr unsigned FULL = 0xffffffffu;
    const uint32_t lt_mask = (1u << lane) - 1u;
    float Tb = t0;               // lattice value of lane 0 of the current window
    float pending = -FLT_MAX;    // the next visited point is the first with T >= pending
    float last_t = t0;           // t after the previously emitted sample (raymarching.cu:425,462)
    uint32_t emitted = 0;
    Binade bn;
    bn.key = -1; bn.m = 1u; bn.inv_m = 1.f; bn.ok = false;
    while (Tb < far && emitted < limit) {
        // lane i holds lattice point i of the window: T = Tb advanced i times
        float T, T_next;
        bool closed_form = false;
        int tb = 0;
        if (p.dt_gamma == 0.f) {
            // Constant step dtc.  Inside one binade [2^e, 2^(e+1)) every float is a multiple of u = 2^(e-23), so the
            // rounded sum fl(T + dtc) equals T + m*u with m = rn(dtc / u) for EVERY T of the binade (no tie) - the
            // serial additions collapse to integer arithmetic on the bit pattern.  Ties and binade crossings (a
            // handful of windows per ray) fall back to the serial loop below.  (m is cached per binade.)
            tb = __float_as_int(Tb);
            if ((tb >> 23) != bn.key) binade_setup(tb, clampf(0.f, p.dt_min, p.dt_max), bn);
            if (bn.ok && ((uint32_t)tb & 0x7fffffu) + 32u * bn.m <= 0x7fffffu) {   // all 33 values stay inside the binade
                T = __int_as_float(tb + lane * (int)bn.m);
                T_next = __int_as_float(tb + (lane + 1) * (int)bn.m);
                closed_form = true;
            }
        }
        if (!closed_form) {
            T = Tb;
#pragma unroll 1
            for (int j = 0; j < 31; ++j) {
                const float Tn = T + clampf(T * p.dt_gamma, p.dt_min, p.dt_max);
                if (j < lane) T = Tn;
            }
            T_next = T + clampf(T * p.dt_gamma, p.dt_min, p.dt_max);  // == T of lane+1
        }
        const bool in_range = T < far;
        const unsigned valid = __ballot_sync(FULL, in_range);
        const unsigned start_mask = __ballot_sync(FULL, T >= pending);
        if (start_mask == 0u) {       // the pending cell exit lies beyond this window
            if (valid != FULL) break;
            Tb = __shfl_sync(FULL, T_next, 31);
            continue;
        }
        Cell c;
        c.occ = false; c.x = c.y = c.z = c.dt = 0.f;
        float tt = 0.f;
        if (in_range) {
            c = classify(p, r, T);
            if (!c.occ) tt = cell_exit(p, r, c, T);
        }
        // next pointer: lower_bound over the lanes above me of T >= tt (the do-while always advances once)
        uint32_t lo = lane + 1, hi = 32;
        if (closed_form) {
            // the window's lattice is tb + j * m in bit patterns (positive floats order like their bits): the first j with
            // T_j >= tt is ceil((bits(tt) - tb) / m), exact through one float multiply and integer fix-ups
            const int tti = __float_as_int(tt);
            if (tti > tb) {
                const uint32_t diff = (uint32_t)(tti - tb);
                const uint32_t j = diff >= 32u * bn.m ? 32u : ceil_div(diff, bn.m, bn.inv_m);
                lo = max(lo, j);
            }
        } else {
#pragma unroll
            for (int it = 0; it < 5; ++it) {
                const uint32_t mid = (lo + hi) >> 1;
                const float Tm = __shfl_sync(FULL, T, mid & 31);
                if (lo < hi) {
                    if (Tm >= tt) hi = mid; else lo = mid + 1;
                }
            }
        }
        // (lo == hi now, except for the degenerate single-candidate case handled by the loop above)
        uint32_t nxt = !in_range ? 32u : (c.occ ? (uint32_t)lane + 1u : lo);
        // visited = everything reachable from the start lane (pointer doubling, 2^5 >= 32 hops)
        unsigned vis = 1u << (__ffs(start_mask) - 1);
        uint32_t hop = nxt;
#pragma unroll
        for (int it = 0; it < 5; ++it) {   // (leaving the loop as soon as a round adds nothing was measured SLOWER: 0.323 vs 0.310 ms)
            const unsigned contrib = (((vis >> lane) & 1u) && hop < 32u) ? (1u << hop) : 0u;
            vis |= __reduce_or_sync(FULL, contrib);
            const uint32_t h2 = __shfl_sync(FULL, hop, hop & 31);
            hop = hop < 32u ? h2 : 32u;
        }
        vis &= valid;
        const unsigned occ_mask = __ballot_sync(FULL, c.occ);
        unsigned emit_mask = vis & occ_mask;
        if (emit_mask) {            // (warp-uniform: most windows of a ray cross empty space and emit nothing)
            const uint32_t room = limit - emitted;
            if ((uint32_t)__popc(emit_mask) > room) {   // keep the first `room` samples only (max_steps cap)
                const uint32_t last = __fns(emit_mask, 0, (int)room);
                emit_mask &= (last >= 31u) ? FULL : ((2u << last) - 1u);
            }
            if (WRITE == 2) {
                if ((emit_mask >> lane) & 1u) xyzs[emitted + __popc(emit_mask & lt_mask)] = T;
            } else if (WRITE == 1) {
                const unsigned below = emit_mask & lt_mask;
                const int prev = below ? (31 - __clz(below)) : 0;
                const float prev_after = __shfl_sync(FULL, T_next, prev);
                if ((emit_mask >> lane) & 1u) {
                    const size_t row = emitted + __popc(below);
                    xyzs[row * 3 + 0] = c.x; xyzs[row * 3 + 1] = c.y; xyzs[row * 3 + 2] = c.z;
                    if (dirs) { dirs[row * 3 + 0] = r.dx; dirs[row * 3 + 1] = r.dy; dirs[row * 3 + 2] = r.dz; }
                    deltas[row * 2 + 0] = c.dt;
                    deltas[row * 2 + 1] = T_next - (below ? prev_after : last_t);  // t - last_t (:461)
                }
            }
            if (emit_mask) {
                last_t = __shfl_sync(FULL, T_next, 31 - __clz(emit_mask));
                emitted += __popc(emit_mask);
            }
        }
        if (valid != FULL || vis == 0u) break;   // the lattice passed `far` inside this window
        // carry: the last visited lane points past the window; if it was empty its exit parameter is pending
        const int last_vis = 31 - __clz(vis);
        const float tt_last = __shfl_sync(FULL, tt, last_vis);
        const bool occ_last = (occ_mask >> last_vis) & 1u;
        pending = occ_last ? -FLT_MAX : tt_last;
        Tb = __shfl_sync(FULL, T_next, 31);
    }
    return emitted;
}

// -------------------------------------------------------------------------------------------------
// utils
// -------------------------------------------------------------------------------------------------
// slab test, axis by axis (raymarching.cu:113-141); a miss reports FLT_MAX for both
NGP_DEVINL void near_far_of(const Ray& r, const float* __restrict__ aabb, float min_near, float& near, float& far) {
    float lo = (aabb[0] - r.ox) * r.rdx, hi = (aabb[3] - r.ox) * r.rdx;
    if (lo > hi) { float s = lo; lo = hi; hi = s; }
    float lo_y = (aabb[1] - r.oy) * r.rdy, hi_y = (aabb[4] - r.oy) * r.rdy;
    if (lo_y > hi_y) { float s = lo_y; lo_y = hi_y; hi_y = s; }
    bool miss = (lo > hi_y || lo_y > hi);
    if (!miss) {
        if (lo_y > lo) lo = lo_y;
        if (hi_y < hi) hi = hi_y;
        float lo_z = (aabb[2] - r.oz) * r.rdz, hi_z = (aabb[5] - r.oz) * r.rdz;
        if (lo_z > hi_z) { float s = lo_z; lo_z = hi_z; hi_z = s; }
        miss = (lo > hi_z || lo_z > hi);
        if (!miss) {
            if (lo_z > lo) lo = lo_z;
            if (hi_z < hi) hi = hi_z;
            if (lo < min_near) lo = min_near;
        }
    }
    near = miss ? FLT_MAX : lo;
    far = miss ? FLT_MAX : hi;
}

__global__ void near_far_kernel(const float* __restrict__ rays_o, const float* __restrict__ rays_d,
                                const float* __restrict__ aabb, uint32_t N, float min_near, float* nears,
                                float* fars) {
    const uint32_t n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    const Ray r = load_ray(rays_o, rays_d, n);
    float lo, hi;
    near_far_of(r, aabb, min_near, lo, hi);
    nears[n] = lo;
    fars[n] = hi;
}

// First kernel of the hand-scheduled train step (ngp_train_prologue): near/far of every ray plus the step's device-side
// bookkeeping, so no separate fill launches are needed: zero the sample-counter pairs and the loss accumulator; open the
// step's row of run_cuda's 16-step counter window (nerf/renderer.py:466-467): *cur_row = *local_step % 16,
// step_counter[*cur_row] = 0, ++*local_step.
// Per-ray march jitter on the device (the reference draws torch.rand(N) per call, raymarching.py:213-216): a counter-based
// generator keyed by (seed, step counter, ray) - three rounds of a 32-bit avalanche mix, top 24 bits -> [0, 1) like
// torch.rand.  Drawing it here removes the uniform_ launch from the step and, in graph mode, the two seed / offset fill
// kernels torch enqueues before every replay of a graph that contains one of its generators.
// rng = u64[3]: seed, step counter, (low word) block-election counter.  Thread 0 of every block reads the counter before it
// signs off; the LAST block to sign off advances it, so every ray of a step sees the same counter and steps never repeat.
NGP_DEVINL uint32_t mix32(uint32_t x) {
    x ^= x >> 16; x *= 0x7feb352du; x ^= x >> 15; x *= 0x846ca68bu; x ^= x >> 16;
    return x;
}
NGP_DEVINL float ray_noise(unsigned long long seed, unsigned long long ctr, uint32_t n) {
    uint32_t x = mix32(n ^ (uint32_t)seed);
    x = mix32(x + (uint32_t)ctr * 0x9E3779B9u + (uint32_t)(ctr >> 32));
    x = mix32(x ^ (uint32_t)(seed >> 32));
    return (float)(x >> 8) * (1.0f / 16777216.0f);
}
NGP_DEVINL void rng_step_done(unsigned long long* rng, unsigned long long ctr) {   // thread 0 of every block, after its reads
    __threadfence();
    unsigned int* done = reinterpret_cast<unsigned int*>(rng + 2);
    if (atomicAdd(done, 1u) == gridDim.x - 1) {
        rng[1] = ctr + 1ull;
        *done = 0u;
    }
}

__global__ void train_prologue_kernel(const float* __restrict__ rays_o, const float* __restrict__ rays_d,
                                      const float* __restrict__ aabb, uint32_t N, float min_near, float* nears,
                                      float* fars, int* counters, uint32_t n_counters, float* loss, int* step_counter,
                                      int* local_step, int* cur_row, float* noises, unsigned long long* rng) {
    __shared__ unsigned long long s_rng[2];
    const uint32_t n = blockIdx.x * blockDim.x + threadIdx.x;
    if (noises) {
        if (threadIdx.x == 0) { s_rng[0] = rng[0]; s_rng[1] = rng[1]; }
        __syncthreads();
    }
    if (n == 0) {
        for (uint32_t i = 0; counters && i < n_counters; ++i) counters[i] = 0;
        if (loss) *loss = 0.f;
        if (step_counter && local_step && cur_row) {
            const int row = (*local_step) & 15;
            *cur_row = row;
            step_counter[row * 2] = 0;
            step_counter[row * 2 + 1] = 0;
            *local_step += 1;
        }
    }
    if (n < N) {
        const Ray r = load_ray(rays_o, rays_d, n);
        float lo, hi;
        near_far_of(r, aabb, min_near, lo, hi);
        nears[n] = lo;
        fars[n] = hi;
        if (noises) noises[n] = ray_noise(s_rng[0], s_rng[1], n);
    }
    if (noises && threadIdx.x == 0) rng_step_done(rng, s_rng[1]);
}

// -------------------------------------------------------------------------------------------------
// Ray generation on the device (nerf/utils.py:43-106 get_rays, the N = -1 branch the dataset uses, provider.py:227): pixel
// centres at +0.5, camera-space direction ((i - cx) / fx, (j - cy) / fy, 1) normalised with safe_normalize (clamp of the
// squared norm at 1e-20, :33-36), rotated by the pose's 3x3 block (rays_d = directions @ R^T), origin = the pose's
// translation.  Sharded views: this launch produces `n_rows` image rows  row0, row0 + row_stride, ...  of every view
// (parallel.shard_rows), rows of one view contiguous.
// -------------------------------------------------------------------------------------------------
struct RayGen {
    const float* poses;        // [B, 4, 4] row-major cam2world
    const float* intrinsics;   // [B, 4] or [1, 4]: fx, fy, cx, cy
    uint32_t B, W, n_rows, row0, row_stride, intr_per_view;
};
NGP_DEVINL Ray generate_ray(const RayGen& g, uint32_t n) {
    const uint32_t per_view = g.n_rows * g.W;
    const uint32_t b = n / per_view, p = n - b * per_view;
    const uint32_t rl = p / g.W, col = p - rl * g.W;
    const uint32_t row = g.row0 + rl * g.row_stride;
    const float* K = g.intrinsics + (g.intr_per_view ? (size_t)b * 4 : 0);
    const float* P = g.poses + (size_t)b * 16;
    const float x = __fdiv_rn(__fsub_rn(__fadd_rn((float)col, 0.5f), K[2]), K[0]);
    const float y = __fdiv_rn(__fsub_rn(__fadd_rn((float)row, 0.5f), K[3]), K[1]);
    const float z = 1.0f;
    const float nrm = sqrtf(fmaxf(__fadd_rn(__fadd_rn(__fmul_rn(x, x), __fmul_rn(y, y)), __fmul_rn(z, z)), 1e-20f));
    const float dx = __fdiv_rn(x, nrm), dy = __fdiv_rn(y, nrm), dz = __fdiv_rn(z, nrm);
    Ray r;
    r.dx = dx * P[0] + dy * P[1] + dz * P[2];
    r.dy = dx * P[4] + dy * P[5] + dz * P[6];
    r.dz = dx * P[8] + dy * P[9] + dz * P[10];
    r.ox = P[3]; r.oy = P[7]; r.oz = P[11];
    r.rdx = 1 / r.dx; r.rdy = 1 / r.dy; r.rdz = 1 / r.dz;
    return r;
}

__global__ void get_rays_kernel(const RayGen g, float* __restrict__ rays_o, float* __restrict__ rays_d) {
    const uint32_t n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= g.B * g.n_rows * g.W) return;
    const Ray r = generate_ray(g, n);
    rays_o[n * 3] = r.ox; rays_o[n * 3 + 1] = r.oy; rays_o[n * 3 + 2] = r.oz;
    rays_d[n * 3] = r.dx; rays_d[n * 3 + 1] = r.dy; rays_d[n * 3 + 2] = r.dz;
}

// train_prologue_kernel with the rays generated in place of loaded: a step's input is B poses + intrinsics (+ G)
__global__ void train_prologue_rays_kernel(const RayGen g, float* __restrict__ rays_o, float* __restrict__ rays_d,
                                           const float* __restrict__ aabb, float min_near, float* nears, float* fars,
                                           int* counters, uint32_t n_counters, float* loss, int* step_counter, int* local_step,
                                           int* cur_row, float* noises, unsigned long long* rng) {
    __shared__ unsigned long long s_rng[2];
    const uint32_t n = blockIdx.x * blockDim.x + threadIdx.x;
    if (noises) {
        if (threadIdx.x == 0) { s_rng[0] = rng[0]; s_rng[1] = rng[1]; }
        __syncthreads();
    }
    if (n == 0) {
        for (uint32_t i = 0; counters && i < n_counters; ++i) counters[i] = 0;
        if (loss) *loss = 0.f;
        if (step_counter && local_step && cur_row) {
            const int row = (*local_step) & 15;
            *cur_row = row;
            step_counter[row * 2] = 0;
            step_counter[row * 2 + 1] = 0;
            *local_step += 1;
        }
    }
    if (n < g.B * g.n_rows * g.W) {
        const Ray r = generate_ray(g, n);
        rays_o[n * 3] = r.ox; rays_o[n * 3 + 1] = r.oy; rays_o[n * 3 + 2] = r.oz;
        rays_d[n * 3] = r.dx; rays_d[n * 3 + 1] = r.dy; rays_d[n * 3 + 2] = r.dz;
        float lo, hi;
        near_far_of(r, aabb, min_near, lo, hi);
        nears[n] = lo;
        fars[n] = hi;
        if (noises) noises[n] = ray_noise(s_rng[0], s_rng[1], n);
    }
    if (noises && threadIdx.x == 0) rng_step_done(rng, s_rng[1]);
}

// Light direction of a shaded train step (nerf/renderer.py:461-464): light_d = safe_normalize(rays_o[0] + randn(3)), with
// the three normal draws taken from the same counter-based generator as the march jitter, on keys no ray uses: ray_noise at
// "ray" indices 2^32 - 1 ... 2^32 - 4 (four uniforms -> two Box-Muller pairs, three of the four normals used).  One thread.
// advance == 0: a prologue launch of this step drew the jitter and advanced the counter, so the step's counter is rng[1] - 1;
// advance == 1: no jitter was drawn, the step's counter is rng[1] and this launch advances it.
__global__ void train_light_kernel(const float* __restrict__ rays_o, unsigned long long* rng, int advance, float* __restrict__ light) {
    if (blockIdx.x != 0 || threadIdx.x != 0) return;
    const unsigned long long seed = rng[0], ctr = advance ? rng[1] : rng[1] - 1ull;
    float u[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) u[j] = ray_noise(seed, ctr, 0xFFFFFFFFu - (uint32_t)j);
    // 1 - u lies in [2^-24, 1]: the logarithm is finite
    const float r0 = sqrtf(-2.0f * logf(1.0f - u[0])), r1 = sqrtf(-2.0f * logf(1.0f - u[2]));
    float s0, c0, s1, c1;
    sincospif(2.0f * u[1], &s0, &c0);
    sincospif(2.0f * u[3], &s1, &c1);
    const float z[3] = {r0 * c0, r0 * s0, r1 * c1};
    float x[3];
#pragma unroll
    for (int a = 0; a < 3; ++a) x[a] = __fadd_rn(rays_o[a], z[a]);
    const float nn = __fadd_rn(__fadd_rn(__fmul_rn(x[0], x[0]), __fmul_rn(x[1], x[1])), __fmul_rn(x[2], x[2]));
    const float nrm = sqrtf(fmaxf(nn, 1e-20f));
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        light[a] = __fdiv_rn(x[a], nrm);
        light[3 + a] = z[a];
    }
    if (advance) rng[1] = ctr + 1ull;
}

__global__ void sph_from_ray_kernel(const float* __restrict__ rays_o, const float* __restrict__ rays_d, float radius,
                                    uint32_t N, float* coords) {
    const uint32_t n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    const float ox = rays_o[n * 3], oy = rays_o[n * 3 + 1], oz = rays_o[n * 3 + 2];
    const float dx = rays_d[n * 3], dy = rays_d[n * 3 + 1], dz = rays_d[n * 3 + 2];
    // |o + t d| = radius, larger root (raymarching.cu:184-188)
    const float A = dx * dx + dy * dy + dz * dz;
    const float Bh = ox * dx + oy * dy + oz * dz;
    const float Cq = ox * ox + oy * oy + oz * oz - radius * radius;
    const float t = (-Bh + sqrtf(Bh * Bh - A * Cq)) / A;
    const float x = ox + t * dx, y = oy + t * dy, z = oz + t * dz;
    const float theta = atan2f(sqrtf(x * x + z * z), y);
    const float phi = atan2f(z, x);
    const float inv_pi = 0.3183098861837907f;
    coords[n * 2] = 2 * theta * inv_pi - 1;
    coords[n * 2 + 1] = phi * inv_pi;
}

__global__ void morton_kernel(const int* __restrict__ coords, uint32_t N, int* indices) {
    const uint32_t n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    indices[n] = (int)morton_encode(coords[n * 3], coords[n * 3 + 1], coords[n * 3 + 2]);
}
__global__ void morton_invert_kernel(const int* __restrict__ indices, uint32_t N, int* coords) {
    const uint32_t n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    const int m = indices[n];
    coords[n * 3 + 0] = (int)compact3(m >> 0);
    coords[n * 3 + 1] = (int)compact3(m >> 1);
    coords[n * 3 + 2] = (int)compact3(m >> 2);
}

// One thread packs one byte from two 16-byte loads (raymarching.cu:268-289).
__global__ void packbits_kernel(const float* __restrict__ grid, uint32_t N, float thresh, uint8_t* bitfield) {
    const uint32_t n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    const float4 a = __ldg(reinterpret_cast<const float4*>(grid) + 2 * (size_t)n);
    const float4 b = __ldg(reinterpret_cast<const float4*>(grid) + 2 * (size_t)n + 1);
    uint32_t bits = 0;
    bits |= (a.x > thresh) ? 1u : 0u;   bits |= (a.y > thresh) ? 2u : 0u;
    bits |= (a.z > thresh) ? 4u : 0u;   bits |= (a.w > thresh) ? 8u : 0u;
    bits |= (b.x > thresh) ? 16u : 0u;  bits |= (b.y > thresh) ? 32u : 0u;
    bits |= (b.z > thresh) ? 64u : 0u;  bits |= (b.w > thresh) ? 128u : 0u;
    bitfield[n] = (uint8_t)bits;
}

// -------------------------------------------------------------------------------------------------
// training march
// -------------------------------------------------------------------------------------------------
NGP_DEVINL float perturbed_start(const MarchParams& p, float near, float noise) {
    float t0 = near;
    t0 += clampf(t0 * p.dt_gamma, p.dt_min, p.dt_max) * noise;  // raymarching.cu:351
    return t0;
}

__global__ void __launch_bounds__(128) march_count_kernel(const float* __restrict__ rays_o, const float* __restrict__ rays_d,
                                                          const uint8_t* __restrict__ grid, float bound, float dt_gamma,
                                                          uint32_t max_steps, uint32_t N, uint32_t C, uint32_t H,
                                                          const float* __restrict__ nears, const float* __restrict__ fars,
                                                          const float* __restrict__ noises, int* __restrict__ counts) {
    const uint32_t n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    const MarchParams p = make_params(grid, bound, dt_gamma, max_steps, C, H);
    const Ray r = load_ray(rays_o, rays_d, n);
    const float far = fars[n];
    float t = perturbed_start(p, nears[n], noises[n]);
    uint32_t steps = 0;
    float x, y, z, dt;
    while (t < far && steps < max_steps) {
        if (probe(p, r, t, x, y, z, dt)) { ++steps; t += dt; }
    }
    counts[n] = (int)steps;
}

// warp-per-ray variants of the count / write passes (see walk_ray_warp)
__global__ void __launch_bounds__(128) march_count_warp_kernel(const float* __restrict__ rays_o, const float* __restrict__ rays_d,
                                                               const uint8_t* __restrict__ grid, float bound, float dt_gamma,
                                                               uint32_t max_steps, uint32_t N, uint32_t C, uint32_t H,
                                                               const float* __restrict__ nears, const float* __restrict__ fars,
                                                               const float* __restrict__ noises, int* __restrict__ counts) {
    const uint32_t n = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (n >= N) return;
    const MarchParams p = make_params(grid, bound, dt_gamma, max_steps, C, H);
    const Ray r = load_ray(rays_o, rays_d, n);
    const float t0 = perturbed_start(p, nears[n], noises[n]);
    const uint32_t steps = walk_ray_warp<0>(p, r, t0, fars[n], max_steps, lane, nullptr, nullptr, nullptr);
    if (lane == 0) counts[n] = (int)steps;
}

__global__ void __launch_bounds__(128) march_write_warp_kernel(const float* __restrict__ rays_o, const float* __restrict__ rays_d,
                                                               const uint8_t* __restrict__ grid, float bound, float dt_gamma,
                                                               uint32_t max_steps, uint32_t N, uint32_t C, uint32_t H, uint32_t M,
                                                               const float* __restrict__ nears, const float* __restrict__ fars,
                                                               const float* __restrict__ noises, const int* __restrict__ counts,
                                                               const int* __restrict__ rays, float* __restrict__ xyzs,
                                                               float* __restrict__ dirs, float* __restrict__ deltas) {
    const uint32_t n = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (n >= N) return;
    const uint32_t num_steps = (uint32_t)counts[n];
    if (num_steps == 0) return;
    const uint32_t offset = (uint32_t)rays[(size_t)n * 3 + 1];
    if (offset + num_steps > M) return;  // raymarching.cu:416
    const MarchParams p = make_params(grid, bound, dt_gamma, max_steps, C, H);
    const Ray r = load_ray(rays_o, rays_d, n);
    const float t0 = perturbed_start(p, nears[n], noises[n]);
    walk_ray_warp<1>(p, r, t0, fars[n], num_steps, lane, xyzs + (size_t)offset * 3, dirs ? dirs + (size_t)offset * 3 : nullptr,
                        deltas + (size_t)offset * 2);
}

__device__ void scan_ray_counts(const int* __restrict__ counts, uint32_t N, int* __restrict__ rays, int* __restrict__ counter,
                                int* s_warp);

// Single-pass variant: walk every ray ONCE, writing its samples into a private slab of max_steps rows, then (after
// the scan has assigned the final offsets) copy the slabs to their packed positions.
__global__ void __launch_bounds__(128) march_slab_kernel(const float* __restrict__ rays_o, const float* __restrict__ rays_d,
                                                         const uint8_t* __restrict__ grid, float bound, float dt_gamma,
                                                         uint32_t max_steps, uint32_t N, uint32_t C, uint32_t H,
                                                         const float* __restrict__ nears, const float* __restrict__ fars,
                                                         const float* __restrict__ noises, int* __restrict__ counts,
                                                         float* __restrict__ slab_xyz, float* __restrict__ slab_delta,
                                                         unsigned int* __restrict__ blocks_done, int* __restrict__ rays,
                                                         int* __restrict__ counter) {
    __shared__ int s_warp[32];
    __shared__ bool s_last;
    __shared__ uint32_t s_lut[1024];
    const bool use_lut = H <= 1024u;
    if (use_lut) {
        for (uint32_t i = threadIdx.x; i < H; i += blockDim.x) s_lut[i] = spread3(i);
        __syncthreads();
    }
    const uint32_t n = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (n < N) {
        MarchParams p = make_params(grid, bound, dt_gamma, max_steps, C, H);
        if (use_lut) p.lut = s_lut;
        const Ray r = load_ray(rays_o, rays_d, n);
        const float t0 = perturbed_start(p, nears[n], noises[n]);
        const uint32_t steps = walk_ray_warp<1>(p, r, t0, fars[n], max_steps, lane, slab_xyz + (size_t)n * max_steps * 3, nullptr,
                                                   slab_delta + (size_t)n * max_steps * 2);
        if (lane == 0) counts[n] = (int)steps;
    }
    if (!blocks_done) return;
    // the LAST block to finish scans the counts (it used to be a separate single-CTA launch): a release / acquire pair
    // on the election counter makes every block's counts visible to it
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        s_last = atomicAdd(blocks_done, 1u) == gridDim.x - 1;
    }
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    scan_ray_counts(counts, N, rays, counter, s_warp);
    if (threadIdx.x == 0) *blocks_done = 0u;     // ready for the next launch on this workspace
}

// Single-pass, slab-free variant ("packed"): the warp walks its ray ONCE, parking the lattice parameter T of every emitted
// sample in shared memory (4 bytes per sample: the clamped position is o + T d, the step clamp(T dt_gamma), and
// deltas[1] = (T + step) - (previous sample's T + step), raymarching.cu:425,461), then claims its rows with ONE
// atomicAdd on the sample counter - the reference's own slot allocation (raymarching.cu:405-406) - and writes them straight
// to their final place.  No per-ray slab (N x max_steps rows of scratch), no scan launch, no compaction copy; the price is
// the reference's row order: rays land in completion order (each ray's samples stay contiguous, rays[n] still describes
// ray n), which every consumer of `rays` accepts.
__global__ void __launch_bounds__(128) march_packed_kernel(const float* __restrict__ rays_o, const float* __restrict__ rays_d,
                                                           const uint8_t* __restrict__ grid, float bound, float dt_gamma,
                                                           uint32_t max_steps, uint32_t N, uint32_t C, uint32_t H, uint32_t M,
                                                           const float* __restrict__ nears, const float* __restrict__ fars,
                                                           const float* __restrict__ noises, float* __restrict__ xyzs,
                                                           float* __restrict__ dirs, float* __restrict__ deltas,
                                                           int* __restrict__ rays, int* __restrict__ counter) {
    extern __shared__ float s_T[];          // [4 warps][max_steps]
    __shared__ uint32_t s_lut[1024];
    const bool use_lut = H <= 1024u;
    if (use_lut) {
        for (uint32_t i = threadIdx.x; i < H; i += blockDim.x) s_lut[i] = spread3(i);
        __syncthreads();
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(counter + 1, (int)N);   // rays seen (raymarching.cu:406)
    const uint32_t n = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (n >= N) return;
    MarchParams p = make_params(grid, bound, dt_gamma, max_steps, C, H);
    if (use_lut) p.lut = s_lut;
    const Ray r = load_ray(rays_o, rays_d, n);
    const float t0 = perturbed_start(p, nears[n], noises[n]);
    float* sT = s_T + (threadIdx.x >> 5) * max_steps;
    const uint32_t steps = walk_ray_warp<2>(p, r, t0, fars[n], max_steps, lane, sT, nullptr, nullptr);
    __syncwarp();
    uint32_t offset = 0;
    if (lane == 0) {
        if (steps) offset = (uint32_t)atomicAdd(counter, (int)steps);
        rays[(size_t)n * 3 + 0] = (int)n;
        rays[(size_t)n * 3 + 1] = (int)offset;
        rays[(size_t)n * 3 + 2] = (int)steps;
    }
    offset = __shfl_sync(0xffffffffu, offset, 0);
    if (steps == 0 || offset + steps > M) return;     // raymarching.cu:415-416
    float* ox = xyzs + (size_t)offset * 3;
    float2* od = reinterpret_cast<float2*>(deltas) + offset;
    for (uint32_t i = lane; i < steps; i += 32) {
        const float T = sT[i];
        const float dt = clampf(T * p.dt_gamma, p.dt_min, p.dt_max);
        float prev_after = t0;                               // t after the previous sample's step (t0 before the first)
        if (i) { const float Tp = sT[i - 1]; prev_after = Tp + clampf(Tp * p.dt_gamma, p.dt_min, p.dt_max); }
        ox[i * 3 + 0] = clampf(__fmaf_rn(T, r.dx, r.ox), -p.bound, p.bound);   // = classify()'s position
        ox[i * 3 + 1] = clampf(__fmaf_rn(T, r.dy, r.oy), -p.bound, p.bound);
        ox[i * 3 + 2] = clampf(__fmaf_rn(T, r.dz, r.oz), -p.bound, p.bound);
        od[i] = make_float2(dt, (T + dt) - prev_after);
        if (dirs) { float* pd = dirs + ((size_t)offset + i) * 3; pd[0] = r.dx; pd[1] = r.dy; pd[2] = r.dz; }
    }
}

// -------------------------------------------------------------------------------------------------
// Thread-per-ray walk with CLOSED-FORM lattice jumps (constant step, dt_gamma == 0: the -O configuration).
// The warp-per-ray walk above classifies all 32 lattice points of a window although, in empty space, only the first point
// of each cell is visited (a 128^3 cell is ~4.6 steps long): ~8 k warp instructions per ray.  Here one thread follows the
// reference's own serial chain - classify, then either emit + one real `t += dt`, or jump out of the empty cell - but the
// reference's inner `do t += dt; while (t < tt)` (raymarching.cu:396-398) is collapsed: inside a binade every float is a
// multiple of u = 2^(e-23) and fl(t + dt) = t + m u with m = rn(dt / u) for every t of the binade (unless dt / u is an exact
// tie), so n steps add n * m to the bit pattern.  The jump takes the n = ceil((tt - t) / (m u)) >= 1 steps the loop would,
// as long as they stay inside the binade; a binade crossing (at most four per ray) or a tie is one REAL float addition.
// Same lattice, same visited points, same bits - at ~1/15 of the instructions; the price is latency (a ray is one serial
// chain), so small launches keep the warp-per-ray walk.
// -------------------------------------------------------------------------------------------------
NGP_DEVINL float lattice_jump(float t, float tt, float dtc, Binade& b) {
    const int tti = __float_as_int(tt);          // tt >= t > 0 or +inf: the bit patterns order like the values
    do {
        const int tb = __float_as_int(t);
        if ((tb >> 23) != b.key) binade_setup(tb, dtc, b);
        if (b.ok) {
            const uint32_t avail = 0x7fffffu - ((uint32_t)tb & 0x7fffffu);            // ulps left in the binade
            uint32_t need_ulps = b.m;                                                 // the do-while always steps once
            bool inside = true;
            if (tti > tb) {
                const uint32_t diff = (uint32_t)(tti - tb);
                inside = diff <= avail;                                               // (otherwise tt lies beyond the binade)
                if (inside) need_ulps = max(ceil_div(diff, b.m, b.inv_m), 1u) * b.m;   // first lattice point >= tt
            }
            if (inside && need_ulps <= avail) return __int_as_float(tb + (int)need_ulps);
            t = __int_as_float(tb + (int)(floor_div(avail, b.m, b.inv_m) * b.m));     // the last point of the binade: still < tt
        }
        t += dtc;        // the crossing (or tie / denormal) step, in float arithmetic as the reference
    } while (t < tt);
    return t;
}

// slab row = (x, y, z, t after the sample's step): ONE 16-byte store per sample; dt is the constant step and
// deltas[1] = t_after - previous t_after (raymarching.cu:461) are rebuilt by march_compact4_kernel.
__global__ void __launch_bounds__(128) march_slab_thread_kernel(const float* __restrict__ rays_o, const float* __restrict__ rays_d,
                                                                const uint8_t* __restrict__ grid, float bound, uint32_t max_steps,
                                                                uint32_t N, uint32_t C, uint32_t H, const float* __restrict__ nears,
                                                                const float* __restrict__ fars, const float* __restrict__ noises,
                                                                int* __restrict__ counts, float4* __restrict__ slab,
                                                                unsigned int* __restrict__ blocks_done, int* __restrict__ rays,
                                                                int* __restrict__ counter) {
    __shared__ int s_warp[32];
    __shared__ bool s_last;
    __shared__ uint32_t s_lut[1024];
    const bool use_lut = H <= 1024u;
    if (use_lut) {
        for (uint32_t i = threadIdx.x; i < H; i += blockDim.x) s_lut[i] = spread3(i);
        __syncthreads();
    }
    const uint32_t n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n < N) {
        MarchParams p = make_params(grid, bound, 0.f, max_steps, C, H);
        if (use_lut) p.lut = s_lut;
        const Ray r = load_ray(rays_o, rays_d, n);
        const float far = fars[n];
        const float dtc = clampf(0.f, p.dt_min, p.dt_max);
        float t = perturbed_start(p, nears[n], noises[n]);
        float4* row = slab + (size_t)n * max_steps;
        uint32_t steps = 0;
        Binade bn;
        bn.key = -1; bn.m = 1u; bn.inv_m = 1.f; bn.ok = false;
        uint32_t last_index = 0xffffffffu;   // consecutive samples stay ~4 steps in a cell: its bit is fetched once
        bool last_occ = false;
        while (t < far && steps < max_steps) {
            const Cell c = classify(p, r, t, &last_index, &last_occ);
            if (c.occ) {
                t += c.dt;                                   // (c.dt == dtc; raymarching.cu:425)
                row[steps++] = make_float4(c.x, c.y, c.z, t);
            } else {
                t = lattice_jump(t, cell_exit(p, r, c, t), dtc, bn);
            }
        }
        counts[n] = (int)steps;
    }
    if (!blocks_done) return;
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        s_last = atomicAdd(blocks_done, 1u) == gridDim.x - 1;
    }
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    scan_ray_counts(counts, N, rays, counter, s_warp);
    if (threadIdx.x == 0) *blocks_done = 0u;
}

__global__ void __launch_bounds__(256) march_compact4_kernel(const float* __restrict__ rays_d, const int* __restrict__ rays,
                                                             const float4* __restrict__ slab, const float* __restrict__ nears,
                                                             const float* __restrict__ noises, uint32_t max_steps, uint32_t N,
                                                             uint32_t M, uint32_t C, uint32_t H, float* __restrict__ xyzs,
                                                             float* __restrict__ dirs, float* __restrict__ deltas) {
    const uint32_t n = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint32_t lane = threadIdx.x & 31;
    if (n >= N) return;
    const uint32_t offset = (uint32_t)rays[(size_t)n * 3 + 1], count = (uint32_t)rays[(size_t)n * 3 + 2];
    if (count == 0 || offset + count > M) return;  // raymarching.cu:415-416
    const MarchParams p = make_params(nullptr, 1.f, 0.f, max_steps, C, H);
    const float dtc = clampf(0.f, p.dt_min, p.dt_max);
    const float t0 = perturbed_start(p, nears[n], noises[n]);     // last_t before the first sample (raymarching.cu:351,425)
    const float4* src = slab + (size_t)n * max_steps;
    float* ox = xyzs + (size_t)offset * 3;
    float2* od = reinterpret_cast<float2*>(deltas) + offset;
    float d0 = 0.f, d1 = 0.f, d2 = 0.f;
    if (dirs) { d0 = rays_d[n * 3]; d1 = rays_d[n * 3 + 1]; d2 = rays_d[n * 3 + 2]; }
    for (uint32_t i = lane; i < count; i += 32) {
        const float4 v = src[i];
        const float prev = i ? src[i - 1].w : t0;
        ox[i * 3] = v.x; ox[i * 3 + 1] = v.y; ox[i * 3 + 2] = v.z;
        od[i] = make_float2(dtc, v.w - prev);
        if (dirs) { float* pd = dirs + ((size_t)offset + i) * 3; pd[0] = d0; pd[1] = d1; pd[2] = d2; }
    }
}

__global__ void __launch_bounds__(256) march_compact_kernel(const float* __restrict__ rays_d, const int* __restrict__ rays,
                                                            const float* __restrict__ slab_xyz, const float* __restrict__ slab_delta,
                                                            uint32_t max_steps, uint32_t N, uint32_t M, float* __restrict__ xyzs,
                                                            float* __restrict__ dirs, float* __restrict__ deltas) {
    const uint32_t n = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint32_t lane = threadIdx.x & 31;
    if (n >= N) return;
    const uint32_t offset = (uint32_t)rays[(size_t)n * 3 + 1], count = (uint32_t)rays[(size_t)n * 3 + 2];
    if (count == 0 || offset + count > M) return;  // raymarching.cu:415-416
    const float* sx = slab_xyz + (size_t)n * max_steps * 3;
    const float* sd = slab_delta + (size_t)n * max_steps * 2;
    float* ox = xyzs + (size_t)offset * 3;
    float* od = deltas + (size_t)offset * 2;
    for (uint32_t i = lane; i < count * 3; i += 32) ox[i] = sx[i];
    for (uint32_t i = lane; i < count * 2; i += 32) od[i] = sd[i];
    if (dirs) {
        const float d0 = rays_d[n * 3], d1 = rays_d[n * 3 + 1], d2 = rays_d[n * 3 + 2];
        float* pd = dirs + (size_t)offset * 3;
        for (uint32_t i = lane; i < count * 3; i += 32) { const uint32_t a = i % 3; pd[i] = a == 0 ? d0 : (a == 1 ? d1 : d2); }
    }
}

// Block-wide exclusive scan of the per-ray counts, in ray order (any block size that is a multiple of 32, <= 1024).  Writes
// the (id, offset, count) rows (row n <-> ray n; offsets start at the incoming counter[0], as the reference's atomicAdd
// would) and bumps the two counters the way the reference's atomics do in aggregate.
// One pass: thread t owns the `per` consecutive rays [t * per, (t + 1) * per) - local sum, one block-wide scan of the
// thread sums, then the rows - so the cost is two barriers whatever N is.
__device__ void scan_ray_counts(const int* __restrict__ counts, uint32_t N, int* __restrict__ rays, int* __restrict__ counter,
                                int* s_warp /* [32] shared */) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, n_warps = blockDim.x >> 5;
    const uint32_t per = ((N + blockDim.x - 1) / blockDim.x + 3u) & ~3u;  // multiple of 4: 16-byte loads, 48-byte row groups
    const uint32_t first = threadIdx.x * per;
    // N % 4 == 0: every group of 4 rays is either fully inside or fully outside [0, N)
    const bool vec = (N % 4 == 0) && ((reinterpret_cast<uintptr_t>(counts) | reinterpret_cast<uintptr_t>(rays)) & 15) == 0;
    int sum = 0;
    if (vec) {
        for (uint32_t i = 0; i < per; i += 4)
            if (first + i < N) {
                const int4 c = __ldcg(reinterpret_cast<const int4*>(counts + first + i));   // L2: written by other blocks
                sum += c.x + c.y + c.z + c.w;
            }
    } else {
        for (uint32_t i = 0; i < per; ++i)
            if (first + i < N) sum += __ldcg(counts + first + i);
    }
    int incl = warp_incl_scan_i(sum, lane);
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        const int v = lane < n_warps ? s_warp[lane] : 0;
        s_warp[lane] = warp_incl_scan_i(v, lane);
    }
    __syncthreads();
    const int carry = counter[0];  // read by every thread BEFORE the last thread overwrites it (barrier below)
    int offset = carry + (warp ? s_warp[warp - 1] : 0) + incl - sum;
    if (vec) {
        for (uint32_t i = 0; i < per; i += 4)
            if (first + i < N) {
                const uint32_t n = first + i;
                const int4 c = __ldcg(reinterpret_cast<const int4*>(counts + n));
                const int o0 = offset, o1 = o0 + c.x, o2 = o1 + c.y, o3 = o2 + c.z;
                int4* row = reinterpret_cast<int4*>(rays + (size_t)n * 3);  // 4 rows = 48 bytes, 16-byte aligned
                row[0] = make_int4((int)n, o0, c.x, (int)n + 1);
                row[1] = make_int4(o1, c.y, (int)n + 2, o2);
                row[2] = make_int4(c.z, (int)n + 3, o3, c.w);
                offset = o3 + c.w;
            }
    } else {
        for (uint32_t i = 0; i < per; ++i)
            if (first + i < N) {
                const uint32_t n = first + i;
                const int c = __ldcg(counts + n);
                rays[(size_t)n * 3 + 0] = (int)n;
                rays[(size_t)n * 3 + 1] = offset;
                rays[(size_t)n * 3 + 2] = c;
                offset += c;
            }
    }
    __syncthreads();
    if (threadIdx.x == blockDim.x - 1) {
        counter[0] = carry + s_warp[31];
        counter[1] += (int)N;
    }
}

__global__ void __launch_bounds__(1024) march_scan_kernel(const int* __restrict__ counts, uint32_t N, int* __restrict__ rays,
                                                          int* __restrict__ counter) {
    __shared__ int s_warp[32];
    scan_ray_counts(counts, N, rays, counter, s_warp);
}

__global__ void __launch_bounds__(128) march_write_kernel(const float* __restrict__ rays_o, const float* __restrict__ rays_d,
                                                          const uint8_t* __restrict__ grid, float bound, float dt_gamma,
                                                          uint32_t max_steps, uint32_t N, uint32_t C, uint32_t H, uint32_t M,
                                                          const float* __restrict__ nears, const float* __restrict__ fars,
                                                          const float* __restrict__ noises, const int* __restrict__ counts,
                                                          const int* __restrict__ rays, float* __restrict__ xyzs,
                                                          float* __restrict__ dirs, float* __restrict__ deltas) {
    const uint32_t n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    const uint32_t num_steps = (uint32_t)counts[n];
    if (num_steps == 0) return;
    const uint32_t offset = (uint32_t)rays[(size_t)n * 3 + 1];
    if (offset + num_steps > M) return;  // raymarching.cu:416

    const MarchParams p = make_params(grid, bound, dt_gamma, max_steps, C, H);
    const Ray r = load_ray(rays_o, rays_d, n);
    const float far = fars[n];
    float t = perturbed_start(p, nears[n], noises[n]);
    float last_t = t;
    float* px = xyzs + (size_t)offset * 3;
    float* pd = dirs ? dirs + (size_t)offset * 3 : nullptr;  // dirs may be omitted (albedo shading never reads them)
    float* pl = deltas + (size_t)offset * 2;
    uint32_t step = 0;
    float x, y, z, dt;
    while (t < far && step < num_steps) {
        if (probe(p, r, t, x, y, z, dt)) {
            px[0] = x; px[1] = y; px[2] = z;
            if (pd) { pd[0] = r.dx; pd[1] = r.dy; pd[2] = r.dz; pd += 3; }
            t += dt;
            pl[0] = dt;
            pl[1] = t - last_t;  // raymarching.cu:461
            last_t = t;
            px += 3; pl += 2;
            ++step;
        }
    }
}

// -------------------------------------------------------------------------------------------------
// training composite: one warp per ray
// -------------------------------------------------------------------------------------------------
struct RaySpan { uint32_t id, offset, count; bool live; };
NGP_DEVINL RaySpan load_span(const int* __restrict__ rays, uint32_t n, uint32_t M) {
    RaySpan s;
    s.id = (uint32_t)rays[n * 3]; s.offset = (uint32_t)rays[n * 3 + 1]; s.count = (uint32_t)rays[n * 3 + 2];
    s.live = !(s.count == 0 || s.offset + s.count > M);  // raymarching.cu:521
    return s;
}

// For the 32 samples [base, base+32) of one ray: per-lane transmittance BEFORE the sample, rebuilt in
// the reference's left-to-right multiplication order (T *= 1 - alpha, raymarching.cu:554), and the
// running depth parameter t (t += deltas[1], :549).  Returns the lane's own (1 - alpha).
NGP_DEVINL void serial_prefix(float om, float d1, int lane, float T_in, float t_in, float& T_before, float& t_incl) {
    float T = T_in, tt = t_in;
#pragma unroll
    for (int j = 0; j < 32; ++j) {
        const float om_j = __shfl_sync(0xffffffffu, om, j);
        const float d_j = __shfl_sync(0xffffffffu, d1, j);
        if (j < lane) T *= om_j;
        if (j <= lane) tt += d_j;
    }
    T_before = T;
    t_incl = tt;
}

__global__ void __launch_bounds__(256) composite_train_fwd_kernel(const float* __restrict__ sigmas, const float* __restrict__ rgbs,
                                                                  const float* __restrict__ deltas, const int* __restrict__ rays,
                                                                  uint32_t M, uint32_t N, float T_thresh, float* weights_sum,
                                                                  float* depth, float* image) {
    const uint32_t n = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (n >= N) return;
    const RaySpan s = load_span(rays, n, M);
    float r = 0, g = 0, b = 0, ws = 0, d = 0;
    if (s.live) {
        float T_carry = 1.0f, t_carry = 0.f;
        for (uint32_t base = 0; base < s.count; base += 32) {
            const uint32_t i = base + lane;
            const bool valid = i < s.count;
            float om = 1.0f, d1 = 0.f, alpha = 0.f, cr = 0.f, cg = 0.f, cb = 0.f;
            if (valid) {
                const size_t m = (size_t)s.offset + i;
                const float sigma = __ldg(sigmas + m);
                const float2 dl = __ldg(reinterpret_cast<const float2*>(deltas) + m);
                alpha = 1.0f - __expf(-sigma * dl.x);  // raymarching.cu:542
                om = 1.0f - alpha;
                d1 = dl.y;
                cr = __ldg(rgbs + m * 3); cg = __ldg(rgbs + m * 3 + 1); cb = __ldg(rgbs + m * 3 + 2);
            }
            float T_before, t_incl;
            serial_prefix(om, d1, lane, T_carry, t_carry, T_before, t_incl);
            const float T_after = T_before * om;
            // first sample after which the ray is opaque enough (:557): it is still accumulated
            const unsigned stop_mask = __ballot_sync(0xffffffffu, valid && (T_after < T_thresh));
            const int stop_lane = stop_mask ? (__ffs(stop_mask) - 1) : 31;
            if (valid && lane <= stop_lane) {
                const float w = alpha * T_before;
                r += w * cr; g += w * cg; b += w * cb;
                d += w * t_incl;
                ws += w;
            }
            if (stop_mask) break;
            T_carry = __shfl_sync(0xffffffffu, T_after, 31);
            t_carry = __shfl_sync(0xffffffffu, t_incl, 31);
        }
        r = warp_sum(r); g = warp_sum(g); b = warp_sum(b); ws = warp_sum(ws); d = warp_sum(d);
    }
    if (lane == 0) {
        weights_sum[s.id] = ws;
        depth[s.id] = d;
        image[s.id * 3] = r; image[s.id * 3 + 1] = g; image[s.id * 3 + 2] = b;
    }
}

NGP_DEVINL float warp_incl_scan_f(float v, int lane) {
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const float t = __shfl_up_sync(0xffffffffu, v, o);
        if (lane >= o) v += t;
    }
    return v;
}

// raymarching.cu:602-682.  ZERO_TAIL additionally writes zeros for the samples of a live ray that lie
// behind the early-termination point, so the caller need not pre-zero rows owned by live rays.
template <bool ZERO_TAIL>
__global__ void __launch_bounds__(256) composite_train_bwd_kernel(
    const float* __restrict__ grad_ws, const float* __restrict__ grad_image, const float* __restrict__ sigmas,
    const float* __restrict__ rgbs, const float* __restrict__ deltas, const int* __restrict__ rays,
    const float* __restrict__ weights_sum, const float* __restrict__ image, uint32_t M, uint32_t N, float T_thresh,
    float* __restrict__ grad_sigmas, float* __restrict__ grad_rgbs) {
    const uint32_t n = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (n >= N) return;
    const RaySpan s = load_span(rays, n, M);
    if (!s.live) return;
    const float gi0 = grad_image[s.id * 3], gi1 = grad_image[s.id * 3 + 1], gi2 = grad_image[s.id * 3 + 2];
    const float gws = grad_ws[s.id];
    const float r_final = image[s.id * 3], g_final = image[s.id * 3 + 1], b_final = image[s.id * 3 + 2];
    const float ws_final = weights_sum[s.id];

    float T_carry = 1.0f, r_carry = 0.f, g_carry = 0.f, b_carry = 0.f;
    bool stopped = false;
    for (uint32_t base = 0; base < s.count; base += 32) {
        const uint32_t i = base + lane;
        const bool valid = i < s.count;
        const size_t m = (size_t)s.offset + i;
        if (stopped) {  // warp-uniform
            if (ZERO_TAIL && valid) {
                grad_sigmas[m] = 0.f;
                grad_rgbs[m * 3] = 0.f; grad_rgbs[m * 3 + 1] = 0.f; grad_rgbs[m * 3 + 2] = 0.f;
            }
            continue;
        }
        float om = 1.0f, alpha = 0.f, d0 = 0.f, cr = 0.f, cg = 0.f, cb = 0.f;
        if (valid) {
            const float sigma = __ldg(sigmas + m);
            d0 = __ldg(deltas + m * 2);
            alpha = 1.0f - __expf(-sigma * d0);
            om = 1.0f - alpha;
            cr = __ldg(rgbs + m * 3); cg = __ldg(rgbs + m * 3 + 1); cb = __ldg(rgbs + m * 3 + 2);
        }
        float T_before, unused_t;
        serial_prefix(om, 0.f, lane, T_carry, 0.f, T_before, unused_t);
        const float T_after = T_before * om;
        const unsigned stop_mask = __ballot_sync(0xffffffffu, valid && (T_after < T_thresh));
        const int stop_lane = stop_mask ? (__ffs(stop_mask) - 1) : 31;
        const bool active = valid && lane <= stop_lane;
        const float w = active ? alpha * T_before : 0.f;
        // running colour INCLUDING this sample (:648-650)
        const float r_run = r_carry + warp_incl_scan_f(w * cr, lane);
        const float g_run = g_carry + warp_incl_scan_f(w * cg, lane);
        const float b_run = b_carry + warp_incl_scan_f(w * cb, lane);
        if (active) {
            grad_rgbs[m * 3] = gi0 * w; grad_rgbs[m * 3 + 1] = gi1 * w; grad_rgbs[m * 3 + 2] = gi2 * w;
            grad_sigmas[m] = d0 * (gi0 * (T_after * cr - (r_final - r_run)) + gi1 * (T_after * cg - (g_final - g_run)) +
                                   gi2 * (T_after * cb - (b_final - b_run)) + gws * (1 - ws_final));
        } else if (ZERO_TAIL && valid) {
            grad_sigmas[m] = 0.f;
            grad_rgbs[m * 3] = 0.f; grad_rgbs[m * 3 + 1] = 0.f; grad_rgbs[m * 3 + 2] = 0.f;
        }
        if (stop_mask) { stopped = true; continue; }
        T_carry = __shfl_sync(0xffffffffu, T_after, 31);
        r_carry = __shfl_sync(0xffffffffu, r_run, 31);
        g_carry = __shfl_sync(0xffffffffu, g_run, 31);
        b_carry = __shfl_sync(0xffffffffu, b_run, 31);
    }
}

// -------------------------------------------------------------------------------------------------
// Hand-scheduled train step: everything between "the field has been evaluated on the marched samples" and "the
// gradients of sigma / rgb are known" for ONE ray, in one warp, in one launch (ngp_train_ray_loss):
//   composite forward (raymarching.cu:501-588)  ->  background blend (nerf/renderer.py:541-545)
//   -> loss gradients at the ray: the guidance gradient G of the blended pixel (nerf/sd.py:115, applied unscaled) and
//      the opacity-entropy regulariser times the GradScaler scale (nerf/utils.py:389-394,708)
//   -> composite backward (raymarching.cu:602-693) over the same samples, still hot in L1/L2.
// The reference spends ~45 launches on this part of a step (two extension kernels + eager elementwise chains either way).
// Arithmetic of both composite passes is the code of the two kernels above, so results are identical to running them
// back to back with the same upstream gradients.
// -------------------------------------------------------------------------------------------------
struct RayLossArgs {
    const float *sigmas, *rgbs, *deltas;
    const int* rays;
    uint32_t M, N;
    float T_thresh;
    const __half* bg;      // [N,3] background colour per ray (bg_net output) or nullptr: the constant bg_const
    float bg_const;
    const float* G;        // gradient wrt the blended image: [B,3,hw] (NCHW, hw = H*W pixels per view) or [N,3] if hw == 0
    uint32_t hw;
    float lambda;          // entropy weight; the mean runs over the N rays of this launch
    const float* scale;    // device scalar multiplying the entropy term's gradient (GradScaler scale) or nullptr (1)
    float *weights_sum, *depth, *image;   // [N], [N], [N,3]: what composite_rays_train returns (image BEFORE the blend)
    float* d_bg;           // [N,3] gradient wrt the background colour, or nullptr
    float *grad_sigmas, *grad_rgbs;       // [M], [M,3]
    float* loss;           // += lambda * mean entropy (zeroed by the prologue)
    // A launch may cover a CHUNK of the step's rays (chunks run on parallel streams): ray_base = index of its first ray
    // among all rays of the step (for the NCHW lookup of G), n_total = rays of the whole step (the entropy mean)
    uint32_t ray_base, n_total;
    // optional device-side bookkeeping of run_cuda / the bench (done by one thread, atomically - chunks run concurrently):
    // samples_total += counter[0]; step_counter[*cur_row] += counter   (row opened by the prologue)
    const int* counter;
    unsigned long long* samples_total;
    int* step_counter;
    const int* cur_row;
};

constexpr float kAlphaLoR = 1e-5f, kAlphaHiR = 1.f - 1e-5f;

struct RaySample { float sigma, d0, d1, r, g, b; };
// sample i of the ray's span (zeros past its end)
NGP_DEVINL RaySample load_ray_sample(const RayLossArgs& a, const RaySpan& s, uint32_t i) {
    RaySample v = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    if (i < s.count) {
        const size_t m = (size_t)s.offset + i;
        v.sigma = a.sigmas[m];
        const float2 dl = *(reinterpret_cast<const float2*>(a.deltas) + m);
        v.d0 = dl.x; v.d1 = dl.y;
        v.r = a.rgbs[m * 3]; v.g = a.rgbs[m * 3 + 1]; v.b = a.rgbs[m * 3 + 2];
    }
    return v;
}

// The same prefix as serial_prefix() - same operations in the same order, so the same bits - with the 32 per-lane values
// exchanged through shared memory: 2 STS + 16 broadcast LDS.128 instead of 64 SHFL (the kernel was bound by the shuffle
// pipe: one warp-wide shuffle per cycle per SM).  s_om / s_d1: this warp's 32-float rows.
NGP_DEVINL void serial_prefix_smem(float om, float d1, int lane, float T_in, float t_in, float* s_om, float* s_d1,
                                   float& T_before, float& t_incl) {
    s_om[lane] = om;
    s_d1[lane] = d1;
    __syncwarp();
    float T = T_in, tt = t_in;
#pragma unroll
    for (int q = 0; q < 8; ++q) {
        const float4 o4 = reinterpret_cast<const float4*>(s_om)[q];
        const float4 d4 = reinterpret_cast<const float4*>(s_d1)[q];
        const float oj[4] = {o4.x, o4.y, o4.z, o4.w}, dj[4] = {d4.x, d4.y, d4.z, d4.w};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int j = q * 4 + k;
            if (j < lane) T *= oj[k];
            if (j <= lane) tt += dj[k];
        }
    }
    __syncwarp();   // everyone has read the rows before the next chunk overwrites them
    T_before = T;
    t_incl = tt;
}

__global__ void __launch_bounds__(256) train_ray_loss_kernel(const RayLossArgs a) {
    __shared__ float s_loss[8];
    __shared__ __align__(16) float s_om[8][32];
    __shared__ __align__(16) float s_d1[8][32];
    const uint32_t n = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    float entropy = 0.f;
    if (blockIdx.x == 0 && threadIdx.x == 0 && a.counter) {
        if (a.samples_total) atomicAdd(a.samples_total, (unsigned long long)a.counter[0]);
        if (a.step_counter && a.cur_row) {
            const int row = (*a.cur_row) & 15;
            atomicAdd(a.step_counter + row * 2, a.counter[0]);
            atomicAdd(a.step_counter + row * 2 + 1, a.counter[1]);
        }
    }
    if (n < a.N) {
        const RaySpan s = load_span(a.rays, n, a.M);
        // ---- pass 1: composite forward ------------------------------------------------------------------------
        // The transmittance BEFORE each sample is parked in grad_sigmas[m] (the row pass 2 overwrites with the gradient):
        // pass 2 re-reads it - written by this very thread - instead of rebuilding the serial product.
        float r = 0, g = 0, b = 0, ws = 0, d = 0;
        if (s.live) {
            float T_carry = 1.0f, t_carry = 0.f;
            // the ray's samples are walked 32 at a time and each chunk depends on the previous one (transmittance), so the
            // loads of chunk k+1 are issued before chunk k is processed: the walk is bound by load latency otherwise
            RaySample nxt = load_ray_sample(a, s, lane);
            for (uint32_t base = 0; base < s.count; base += 32) {
                const RaySample cur = nxt;
                if (base + 32 < s.count) nxt = load_ray_sample(a, s, base + 32 + lane);
                const bool valid = base + lane < s.count;
                float om = 1.0f, d1 = 0.f, alpha = 0.f, cr = 0.f, cg = 0.f, cb = 0.f;
                if (valid) {
                    alpha = 1.0f - __expf(-cur.sigma * cur.d0);
                    om = 1.0f - alpha;
                    d1 = cur.d1;
                    cr = cur.r; cg = cur.g; cb = cur.b;
                }
                float T_before, t_incl;
                serial_prefix_smem(om, d1, lane, T_carry, t_carry, s_om[warp], s_d1[warp], T_before, t_incl);
                if (valid) a.grad_sigmas[(size_t)s.offset + base + lane] = T_before;
                const float T_after = T_before * om;
                const unsigned stop_mask = __ballot_sync(0xffffffffu, valid && (T_after < a.T_thresh));
                const int stop_lane = stop_mask ? (__ffs(stop_mask) - 1) : 31;
                if (valid && lane <= stop_lane) {
                    const float w = alpha * T_before;
                    r += w * cr; g += w * cg; b += w * cb;
                    d += w * t_incl;
                    ws += w;
                }
                if (stop_mask) break;
                T_carry = __shfl_sync(0xffffffffu, T_after, 31);
                t_carry = __shfl_sync(0xffffffffu, t_incl, 31);
            }
            r = warp_sum(r); g = warp_sum(g); b = warp_sum(b); ws = warp_sum(ws); d = warp_sum(d);
        }
        // ---- the ray's loss terms (every lane computes the same values) -----------------------------------------
        const uint32_t id = s.id;
        float bgc[3] = {a.bg_const, a.bg_const, a.bg_const};
        if (a.bg) {
#pragma unroll
            for (int c = 0; c < 3; ++c) bgc[c] = __half2float(a.bg[(size_t)id * 3 + c]);
        }
        float gi[3];
        if (a.hw) {
            const uint32_t gid = id + a.ray_base;
            const uint32_t view = gid / a.hw, pix = gid % a.hw;
#pragma unroll
            for (int c = 0; c < 3; ++c) gi[c] = a.G[((size_t)view * 3 + c) * a.hw + pix];
        } else {
#pragma unroll
            for (int c = 0; c < 3; ++c) gi[c] = a.G[(size_t)id * 3 + c];
        }
        // blend backward: d_ws = -sum_c g_c bg_c, d_bg = (1 - ws) g  (train_step.cu blend_backward_kernel)
        float gws = -(gi[0] * bgc[0] + gi[1] * bgc[1] + gi[2] * bgc[2]);
        // entropy of the clamped opacity and its gradient (train_step.cu entropy_*_kernel)
        const float al = fminf(fmaxf(ws, kAlphaLoR), kAlphaHiR);
        entropy = -al * log2f(al) - (1.f - al) * log2f(1.f - al);
        if (ws >= kAlphaLoR && ws <= kAlphaHiR) {
            const float up = a.scale ? *a.scale : 1.f;
            gws += up * (a.lambda / (float)a.n_total) * (log2f(1.f - ws) - log2f(ws));
        }
        if (lane == 0) {
            a.weights_sum[id] = ws;
            a.depth[id] = d;
            a.image[(size_t)id * 3] = r; a.image[(size_t)id * 3 + 1] = g; a.image[(size_t)id * 3 + 2] = b;
            if (a.d_bg) {
                const float one_minus = 1.f - ws;
#pragma unroll
                for (int c = 0; c < 3; ++c) a.d_bg[(size_t)id * 3 + c] = one_minus * gi[c];
            }
        }
        // ---- pass 2: composite backward --------------------------------------------------------------------------
        if (s.live) {
            const float r_final = r, g_final = g, b_final = b, ws_final = ws;
            float r_carry = 0.f, g_carry = 0.f, b_carry = 0.f;
            bool stopped = false;
            RaySample nxt = load_ray_sample(a, s, lane);
            float T_nxt = (uint32_t)lane < s.count ? a.grad_sigmas[(size_t)s.offset + lane] : 1.0f;   // parked by pass 1
            for (uint32_t base = 0; base < s.count; base += 32) {
                const uint32_t i = base + lane;
                const bool valid = i < s.count;
                const size_t m = (size_t)s.offset + i;
                if (stopped) {  // warp-uniform: rows behind the early-termination point get zero gradients
                    if (valid) {
                        a.grad_sigmas[m] = 0.f;
                        a.grad_rgbs[m * 3] = 0.f; a.grad_rgbs[m * 3 + 1] = 0.f; a.grad_rgbs[m * 3 + 2] = 0.f;
                    }
                    continue;
                }
                const RaySample cur = nxt;
                const float T_before = T_nxt;
                if (base + 32 < s.count) {
                    nxt = load_ray_sample(a, s, base + 32 + lane);
                    // (rows behind the stop chunk were never parked: whatever is read there is discarded with `stopped`)
                    T_nxt = (base + 32 + lane < s.count) ? a.grad_sigmas[m + 32] : 1.0f;
                }
                float om = 1.0f, alpha = 0.f, d0 = 0.f, cr = 0.f, cg = 0.f, cb = 0.f;
                if (valid) {
                    d0 = cur.d0;
                    alpha = 1.0f - __expf(-cur.sigma * d0);
                    om = 1.0f - alpha;
                    cr = cur.r; cg = cur.g; cb = cur.b;
                }
                const float T_after = T_before * om;
                const unsigned stop_mask = __ballot_sync(0xffffffffu, valid && (T_after < a.T_thresh));
                const int stop_lane = stop_mask ? (__ffs(stop_mask) - 1) : 31;
                const bool active = valid && lane <= stop_lane;
                const float w = active ? alpha * T_before : 0.f;
                const float r_run = r_carry + warp_incl_scan_f(w * cr, lane);
                const float g_run = g_carry + warp_incl_scan_f(w * cg, lane);
                const float b_run = b_carry + warp_incl_scan_f(w * cb, lane);
                if (active) {
                    a.grad_rgbs[m * 3] = gi[0] * w; a.grad_rgbs[m * 3 + 1] = gi[1] * w; a.grad_rgbs[m * 3 + 2] = gi[2] * w;
                    a.grad_sigmas[m] = d0 * (gi[0] * (T_after * cr - (r_final - r_run)) + gi[1] * (T_after * cg - (g_final - g_run)) +
                                             gi[2] * (T_after * cb - (b_final - b_run)) + gws * (1 - ws_final));
                } else if (valid) {
                    a.grad_sigmas[m] = 0.f;
                    a.grad_rgbs[m * 3] = 0.f; a.grad_rgbs[m * 3 + 1] = 0.f; a.grad_rgbs[m * 3 + 2] = 0.f;
                }
                if (stop_mask) { stopped = true; continue; }
                r_carry = __shfl_sync(0xffffffffu, r_run, 31);
                g_carry = __shfl_sync(0xffffffffu, g_run, 31);
                b_carry = __shfl_sync(0xffffffffu, b_run, 31);
            }
        }
    }
    // loss: one atomic per block
    if (lane == 0) s_loss[warp] = entropy;
    __syncthreads();
    if (threadIdx.x == 0 && a.loss) {
        float v = 0.f;
        for (uint32_t w = 0; w < (blockDim.x >> 5); ++w) v += s_loss[w];
        atomicAdd(a.loss, v * (a.lambda / (float)a.n_total));
    }
}

// -------------------------------------------------------------------------------------------------
// inference march / composite (raymarching.cu:701-905): few steps per call, one thread per ray
// -------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) march_infer_kernel(uint32_t n_alive, uint32_t n_step, const int* __restrict__ rays_alive,
                                                          const float* __restrict__ rays_t, const float* __restrict__ rays_o,
                                                          const float* __restrict__ rays_d, float bound, float dt_gamma,
                                                          uint32_t max_steps, uint32_t C, uint32_t H,
                                                          const uint8_t* __restrict__ grid, const float* __restrict__ nears,
                                                          const float* __restrict__ fars, float* __restrict__ xyzs,
                                                          float* __restrict__ dirs, float* __restrict__ deltas,
                                                          const float* __restrict__ noises) {
    const uint32_t n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= n_alive) return;
    const int id = rays_alive[n];
    const MarchParams p = make_params(grid, bound, dt_gamma, max_steps, C, H);
    const Ray r = load_ray(rays_o, rays_d, (uint32_t)id);
    const float far = fars[id];
    float t = rays_t[id];
    t += clampf(t * p.dt_gamma, p.dt_min, p.dt_max) * noises[n];  // raymarching.cu:746
    float last_t = t;
    float* px = xyzs + (size_t)n * n_step * 3;
    float* pd = dirs + (size_t)n * n_step * 3;
    float* pl = deltas + (size_t)n * n_step * 2;
    uint32_t step = 0;
    float x, y, z, dt;
    while (t < far && step < n_step) {
        if (probe(p, r, t, x, y, z, dt)) {
            px[0] = x; px[1] = y; px[2] = z;
            pd[0] = r.dx; pd[1] = r.dy; pd[2] = r.dz;
            t += dt;
            pl[0] = dt;
            pl[1] = t - last_t;
            last_t = t;
            px += 3; pd += 3; pl += 2;
            ++step;
        }
    }
}

// Warp-per-ray variant for ONE sample per ray (the first iterations of a frame, n_step == 1 while most rays are alive):
// there every ray first crosses the empty space in front of the object - hundreds of lattice points - before it emits its
// sample, and one thread per ray walks them serially.  walk_ray_warp classifies 32 lattice points per iteration and is
// bit-identical to the serial loop (it is the training marcher's walk, checked against the reference there).
__global__ void __launch_bounds__(128) march_infer_warp_kernel(uint32_t n_alive, uint32_t n_step, const int* __restrict__ rays_alive,
                                                               const float* __restrict__ rays_t, const float* __restrict__ rays_o,
                                                               const float* __restrict__ rays_d, float bound, float dt_gamma,
                                                               uint32_t max_steps, uint32_t C, uint32_t H,
                                                               const uint8_t* __restrict__ grid, const float* __restrict__ fars,
                                                               float* __restrict__ xyzs, float* __restrict__ dirs,
                                                               float* __restrict__ deltas, const float* __restrict__ noises) {
    const int lane = threadIdx.x & 31;
    const uint32_t warps = (gridDim.x * blockDim.x) >> 5;
    const MarchParams p = make_params(grid, bound, dt_gamma, max_steps, C, H);
    for (uint32_t n = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; n < n_alive; n += warps) {
        const int id = rays_alive[n];
        const Ray r = load_ray(rays_o, rays_d, (uint32_t)id);
        float t = rays_t[id];
        t += clampf(t * p.dt_gamma, p.dt_min, p.dt_max) * (noises ? noises[n] : 0.f);
        walk_ray_warp<1>(p, r, t, fars[id], n_step, lane, xyzs + (size_t)n * n_step * 3, dirs ? dirs + (size_t)n * n_step * 3 : nullptr,
                            deltas + (size_t)n * n_step * 2);
    }
}

__global__ void __launch_bounds__(128) composite_infer_kernel(uint32_t n_alive, uint32_t n_step, float T_thresh, int* rays_alive,
                                                              float* rays_t, const float* __restrict__ sigmas,
                                                              const float* __restrict__ rgbs, const float* __restrict__ deltas,
                                                              float* weights_sum, float* depth, float* image) {
    const uint32_t n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= n_alive) return;
    const int id = rays_alive[n];
    const float* ps = sigmas + (size_t)n * n_step;
    const float* pc = rgbs + (size_t)n * n_step * 3;
    const float* pl = deltas + (size_t)n * n_step * 2;
    float t = rays_t[id];
    float wsum = weights_sum[id], d = depth[id];
    float r = image[id * 3], g = image[id * 3 + 1], b = image[id * 3 + 2];
    uint32_t step = 0;
    while (step < n_step) {
        if (pl[0] == 0) break;  // unused slot: the marcher ran out of ray (raymarching.cu:858)
        const float alpha = 1.0f - __expf(-ps[0] * pl[0]);
        const float T = 1 - wsum;  // transmittance from the running alpha sum (:868)
        const float w = alpha * T;
        wsum += w;
        t += pl[1];
        d += w * t;
        r += w * pc[0]; g += w * pc[1]; b += w * pc[2];
        if (T < T_thresh) break;
        ++ps; pc += 3; pl += 2; ++step;
    }
    if (step < n_step) rays_alive[n] = -1; else rays_t[id] = t;  // :894-898
    weights_sum[id] = wsum;
    depth[id] = d;
    image[id * 3] = r; image[id * 3 + 1] = g; image[id * 3 + 2] = b;
}

// -------------------------------------------------------------------------------------------------
// stable compaction of alive rays (device-side replacement for the boolean-mask indexing)
// -------------------------------------------------------------------------------------------------
constexpr int kCompactBlock = 1024;
__global__ void __launch_bounds__(kCompactBlock) compact_count_kernel(const int* __restrict__ rays_alive, uint32_t n,
                                                                      int* __restrict__ block_counts) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    const int keep = (i < n && rays_alive[i] >= 0) ? 1 : 0;
    const int total = __syncthreads_count(keep);
    if (threadIdx.x == 0) block_counts[blockIdx.x] = total;
}
__global__ void __launch_bounds__(kCompactBlock) compact_scatter_kernel(const int* __restrict__ rays_alive, uint32_t n,
                                                                        const int* __restrict__ block_counts, int* __restrict__ out,
                                                                        int* __restrict__ n_out) {
    __shared__ int s_warp[32];
    __shared__ int s_base;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    // prefix of the preceding blocks' counts (grid is small: <= n/1024 entries)
    int part = 0;
    for (uint32_t j = threadIdx.x; j < blockIdx.x; j += blockDim.x) part += block_counts[j];
    part = warp_sum_i(part);
    if (lane == 0) s_warp[warp] = part;
    __syncthreads();
    if (warp == 0) {
        int v = s_warp[lane];
        v = warp_sum_i(v);
        if (lane == 0) s_base = v;
    }
    __syncthreads();
    const int base = s_base;
    __syncthreads();
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    const int v = i < n ? rays_alive[i] : -1;
    const int keep = v >= 0 ? 1 : 0;
    const int incl = warp_incl_scan_i(keep, lane);
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        int w = s_warp[lane];
        w = warp_incl_scan_i(w, lane);
        s_warp[lane] = w;
    }
    __syncthreads();
    const int pos = base + (warp ? s_warp[warp - 1] : 0) + incl - keep;
    if (keep) out[pos] = v;
    if (blockIdx.x == gridDim.x - 1 && threadIdx.x == blockDim.x - 1) *n_out = base + s_warp[31];
}


// -------------------------------------------------------------------------------------------------
// Device-driven inference loop.  The reference's eval branch (nerf/renderer.py:496-532) is a HOST while-loop: count
// the alive rays (a device->host sync), pick n_step = clamp(N / n_alive, 1, 8), march, evaluate the field, composite,
// compact.  Here the loop state lives on the device and the loop itself is a CUDA-graph conditional WHILE node
// (ngp_render_infer_loop): the kernels below read n_alive / n_step from `InferState`, the last kernel of the body
// advances the state and sets the loop condition - no host round trip per iteration.  Arithmetic and visiting order
// are those of march_infer_kernel / composite_infer_kernel above (so results equal the host loop's bit for bit).
// -------------------------------------------------------------------------------------------------
struct InferState {
    int n_alive;      // rays in alive[cur]
    int n_step;       // samples marched per alive ray this iteration
    int step;         // sum of the n_step of completed iterations (the reference's `step`)
    int cur;          // which of the two alive buffers is current
    int iters;        // completed iterations
    int rows;         // n_alive * n_step: field rows of this iteration
    int n_next;       // compaction output count
    int pad;
};

NGP_DEVINL int plan_n_step(int N, int n_alive) { return max(min(N / max(n_alive, 1), 8), 1); }  // renderer.py:521

__global__ void infer_init_kernel(uint32_t N, const float* __restrict__ nears, int* __restrict__ alive0, float* __restrict__ rays_t,
                                  float* __restrict__ weights_sum, float* __restrict__ depth, float* __restrict__ image,
                                  InferState* st) {
    const uint32_t n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n == 0) {
        st->n_alive = (int)N; st->n_step = plan_n_step((int)N, (int)N); st->step = 0; st->cur = 0; st->iters = 0;
        st->rows = (int)N * st->n_step; st->n_next = 0;
    }
    if (n >= N) return;
    alive0[n] = (int)n;              // rays_alive = arange(N), rays_t = nears.clone()  (renderer.py:505-507)
    rays_t[n] = nears[n];
    weights_sum[n] = 0.f; depth[n] = 0.f;
    image[n * 3] = 0.f; image[n * 3 + 1] = 0.f; image[n * 3 + 2] = 0.f;
}

__global__ void __launch_bounds__(128) infer_march_kernel(const InferState* __restrict__ st, uint32_t N, int* __restrict__ alive_buf,
                                                          const float* __restrict__ rays_t, const float* __restrict__ rays_o,
                                                          const float* __restrict__ rays_d, float bound, float dt_gamma,
                                                          uint32_t max_steps, uint32_t C, uint32_t H,
                                                          const uint8_t* __restrict__ grid, const float* __restrict__ fars,
                                                          float* __restrict__ xyzs, float* __restrict__ deltas,
                                                          const float* __restrict__ noises) {
    const uint32_t n_alive = (uint32_t)st->n_alive, n_step = (uint32_t)st->n_step;
    const int* __restrict__ rays_alive = alive_buf + (size_t)st->cur * N;
    const bool first = st->step == 0;
    const MarchParams p = make_params(grid, bound, dt_gamma, max_steps, C, H);
    if (first && n_step == 1 && n_alive <= 16384u) {
        // first iteration of a SMALL frame: every ray starts at its near plane and crosses the empty space in front of the
        // object (hundreds of lattice points) before its first sample, and there are too few rays to fill the machine with
        // one thread each - one WARP per ray, 32 lattice points classified per iteration (see march_infer_warp_kernel).
        // The warp walk spends ~10x the lane-time of the serial walk, so with many rays (800x800: 640 000) a thread per ray
        // wins (measured: 13.5 vs 9.35 ms per frame), as it does on later iterations that start next to the last sample.
        const int lane = threadIdx.x & 31;
        const uint32_t warps = (gridDim.x * blockDim.x) >> 5;
        for (uint32_t n = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; n < n_alive; n += warps) {
            const int id = rays_alive[n];
            const Ray r = load_ray(rays_o, rays_d, (uint32_t)id);
            float t = rays_t[id];
            t += clampf(t * p.dt_gamma, p.dt_min, p.dt_max) * ((first && noises) ? noises[n] : 0.f);
            const uint32_t got = walk_ray_warp<1>(p, r, t, fars[id], 1u, lane, xyzs + (size_t)n * 3, nullptr, deltas + (size_t)n * 2);
            if (got == 0 && lane == 0) {
                xyzs[(size_t)n * 3] = 0.f; xyzs[(size_t)n * 3 + 1] = 0.f; xyzs[(size_t)n * 3 + 2] = 0.f;
                deltas[(size_t)n * 2] = 0.f; deltas[(size_t)n * 2 + 1] = 0.f;
            }
        }
        return;
    }
    for (uint32_t n = blockIdx.x * blockDim.x + threadIdx.x; n < n_alive; n += gridDim.x * blockDim.x) {
        const int id = rays_alive[n];
        const Ray r = load_ray(rays_o, rays_d, (uint32_t)id);
        const float far = fars[id];
        float t = rays_t[id];
        const float noise = (first && noises) ? noises[n] : 0.f;      // perturb only on the first call (renderer.py:523)
        t += clampf(t * p.dt_gamma, p.dt_min, p.dt_max) * noise;
        float last_t = t;
        float* px = xyzs + (size_t)n * n_step * 3;
        float* pl = deltas + (size_t)n * n_step * 2;
        uint32_t step = 0;
        float x, y, z, dt;
        while (t < far && step < n_step) {
            if (probe(p, r, t, x, y, z, dt)) {
                px[0] = x; px[1] = y; px[2] = z;
                t += dt;
                pl[0] = dt;
                pl[1] = t - last_t;
                last_t = t;
                px += 3; pl += 2;
                ++step;
            }
        }
        // unused slots: what the reference's zero-filled buffers hold (delta 0 terminates the composite, :858)
        for (; step < n_step; ++step) { px[0] = 0.f; px[1] = 0.f; px[2] = 0.f; pl[0] = 0.f; pl[1] = 0.f; px += 3; pl += 2; }
    }
}

__global__ void __launch_bounds__(128) infer_composite_kernel(const InferState* __restrict__ st, uint32_t N, float T_thresh,
                                                              int* __restrict__ alive_buf, float* __restrict__ rays_t,
                                                              const float* __restrict__ sigmas, const float* __restrict__ rgbs,
                                                              const float* __restrict__ deltas, float* weights_sum, float* depth,
                                                              float* image) {
    const uint32_t n_alive = (uint32_t)st->n_alive, n_step = (uint32_t)st->n_step;
    int* __restrict__ rays_alive = alive_buf + (size_t)st->cur * N;
    for (uint32_t n = blockIdx.x * blockDim.x + threadIdx.x; n < n_alive; n += gridDim.x * blockDim.x) {
        const int id = rays_alive[n];
        const float* ps = sigmas + (size_t)n * n_step;
        const float* pc = rgbs + (size_t)n * n_step * 3;
        const float* pl = deltas + (size_t)n * n_step * 2;
        float t = rays_t[id];
        float wsum = weights_sum[id], d = depth[id];
        float r = image[id * 3], g = image[id * 3 + 1], b = image[id * 3 + 2];
        uint32_t step = 0;
        while (step < n_step) {
            if (pl[0] == 0) break;
            const float alpha = 1.0f - __expf(-ps[0] * pl[0]);
            const float T = 1 - wsum;
            const float w = alpha * T;
            wsum += w;
            t += pl[1];
            d += w * t;
            r += w * pc[0]; g += w * pc[1]; b += w * pc[2];
            if (T < T_thresh) break;
            ++ps; pc += 3; pl += 2; ++step;
        }
        if (step < n_step) rays_alive[n] = -1; else rays_t[id] = t;
        weights_sum[id] = wsum;
        depth[id] = d;
        image[id * 3] = r; image[id * 3 + 1] = g; image[id * 3 + 2] = b;
    }
}

// stable compaction alive[cur] -> alive[cur ^ 1] with a device-side length: per-block counts, then scatter
__global__ void __launch_bounds__(kCompactBlock) infer_compact_count_kernel(const InferState* __restrict__ st, uint32_t N,
                                                                            const int* __restrict__ alive_buf,
                                                                            int* __restrict__ block_counts) {
    const uint32_t n_alive = (uint32_t)st->n_alive;
    const int* __restrict__ rays_alive = alive_buf + (size_t)st->cur * N;
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    const int keep = (i < n_alive && rays_alive[i] >= 0) ? 1 : 0;
    const int total = __syncthreads_count(keep);
    if (threadIdx.x == 0) block_counts[blockIdx.x] = total;
}
__global__ void __launch_bounds__(kCompactBlock) infer_compact_scatter_kernel(InferState* st, uint32_t N, int* __restrict__ alive_buf,
                                                                              const int* __restrict__ block_counts) {
    __shared__ int s_warp[32];
    __shared__ int s_base;
    const uint32_t n_alive = (uint32_t)st->n_alive;
    const int* __restrict__ rays_alive = alive_buf + (size_t)st->cur * N;
    int* __restrict__ out = alive_buf + (size_t)(st->cur ^ 1) * N;
    if (blockIdx.x * blockDim.x >= n_alive && blockIdx.x != 0) return;   // (block 0 always runs: it publishes an empty result)
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int part = 0;
    for (uint32_t j = threadIdx.x; j < blockIdx.x; j += blockDim.x) part += block_counts[j];
    part = warp_sum_i(part);
    if (lane == 0) s_warp[warp] = part;
    __syncthreads();
    if (warp == 0) {
        int v = s_warp[lane];
        v = warp_sum_i(v);
        if (lane == 0) s_base = v;
    }
    __syncthreads();
    const int base = s_base;
    __syncthreads();
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    const int v = i < n_alive ? rays_alive[i] : -1;
    const int keep = v >= 0 ? 1 : 0;
    const int incl = warp_incl_scan_i(keep, lane);
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        int w = s_warp[lane];
        w = warp_incl_scan_i(w, lane);
        s_warp[lane] = w;
    }
    __syncthreads();
    const int pos = base + (warp ? s_warp[warp - 1] : 0) + incl - keep;
    if (keep) out[pos] = v;
    // the block holding the last alive slot publishes the total
    const uint32_t last_block = n_alive ? (n_alive - 1) / blockDim.x : 0u;
    if (blockIdx.x == last_block && threadIdx.x == blockDim.x - 1) st->n_next = base + s_warp[31];
}

// last kernel of the loop body: advance the loop state and decide whether the body runs again
__global__ void infer_plan_kernel(InferState* st, uint32_t N, uint32_t max_steps, cudaGraphConditionalHandle handle,
                                  int use_handle) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    st->step += st->n_step;                         // renderer.py:532
    st->n_alive = st->n_next;                       // rays_alive = rays_alive[rays_alive >= 0]  (:529)
    st->cur ^= 1;
    st->iters += 1;
    st->n_step = plan_n_step((int)N, st->n_alive);
    st->rows = st->n_alive * st->n_step;
    const bool again = st->n_alive > 0 && st->step < (int)max_steps;   // `while step < max_steps` / `if n_alive <= 0: break`
    if (use_handle) cudaGraphSetConditional(handle, again ? 1u : 0u);
}

}  // namespace march
}  // namespace ngp

using namespace ngp;

extern "C" int ngp_near_far_from_aabb(const float* rays_o, const float* rays_d, const float* aabb, uint32_t N,
                                      float min_near, float* nears, float* fars, void* stream) {
    if (!rays_o || !rays_d || !aabb || !nears || !fars) return NGP_ERR_BAD_ARG;
    if (N == 0) return NGP_OK;
    march::near_far_kernel<<<cdiv(N, 128), 128, 0, as_stream(stream)>>>(rays_o, rays_d, aabb, N, min_near, nears, fars);
    return launch_status();
}

extern "C" int ngp_sph_from_ray(const float* rays_o, const float* rays_d, float radius, uint32_t N, float* coords,
                                void* stream) {
    if (!rays_o || !rays_d || !coords) return NGP_ERR_BAD_ARG;
    if (N == 0) return NGP_OK;
    march::sph_from_ray_kernel<<<cdiv(N, 128), 128, 0, as_stream(stream)>>>(rays_o, rays_d, radius, N, coords);
    return launch_status();
}

extern "C" int ngp_morton3D(const int* coords, uint32_t N, int* indices, void* stream) {
    if (!coords || !indices) return NGP_ERR_BAD_ARG;
    if (N == 0) return NGP_OK;
    march::morton_kernel<<<cdiv(N, 256), 256, 0, as_stream(stream)>>>(coords, N, indices);
    return launch_status();
}

extern "C" int ngp_morton3D_invert(const int* indices, uint32_t N, int* coords, void* stream) {
    if (!coords || !indices) return NGP_ERR_BAD_ARG;
    if (N == 0) return NGP_OK;
    march::morton_invert_kernel<<<cdiv(N, 256), 256, 0, as_stream(stream)>>>(indices, N, coords);
    return launch_status();
}

extern "C" int ngp_packbits(const float* grid, uint32_t N, float density_thresh, uint8_t* bitfield, void* stream) {
    if (!grid || !bitfield) return NGP_ERR_BAD_ARG;
    if (N == 0) return NGP_OK;
    march::packbits_kernel<<<cdiv(N, 256), 256, 0, as_stream(stream)>>>(grid, N, density_thresh, bitfield);
    return launch_status();
}

extern "C" int ngp_march_set_option(int option, int value) {
    if (option == 0) { march::g_thread_per_ray = (value != 0); return NGP_OK; }
    if (option == 1) { march::g_infer_warp_march = (value != 0); return NGP_OK; }
    if (option == 2 && value >= 0) { march::g_thread_march_min_rays = (uint32_t)value; return NGP_OK; }
    return NGP_ERR_BAD_ARG;
}

extern "C" uint64_t ngp_march_rays_train_workspace(uint32_t N, uint32_t max_steps) {
    // election counter (256 B) + per-ray counts + (warp-per-ray walk) a private slab of max_steps rows (xyz 12 B + deltas 8 B)
    return 256 + (((uint64_t)N * sizeof(int) + 255) / 256) * 256 + (uint64_t)N * max_steps * 20 + 256;
}

extern "C" int ngp_march_rays_train(const float* rays_o, const float* rays_d, const uint8_t* grid, float bound,
                                    float dt_gamma, uint32_t max_steps, uint32_t N, uint32_t C, uint32_t H, uint32_t M,
                                    const float* nears, const float* fars, float* xyzs, float* dirs, float* deltas,
                                    int* rays, int* counter, const float* noises, void* workspace,
                                    uint64_t workspace_bytes, void* stream) {
    if (!rays_o || !rays_d || !grid || !nears || !fars || !xyzs || !deltas || !rays || !counter || !noises)
        return NGP_ERR_BAD_ARG;
    if (C == 0 || H == 0 || max_steps == 0) return NGP_ERR_BAD_ARG;
    if (!workspace || workspace_bytes < ngp_march_rays_train_workspace(N, max_steps)) return NGP_ERR_WORKSPACE;
    if (N == 0) return NGP_OK;
    cudaStream_t st = as_stream(stream);
    unsigned int* blocks_done = static_cast<unsigned int*>(workspace);
    int* counts = reinterpret_cast<int*>(static_cast<uint8_t*>(workspace) + 256);
    if (march::g_thread_per_ray) {
        march::march_count_kernel<<<cdiv(N, 128), 128, 0, st>>>(rays_o, rays_d, grid, bound, dt_gamma, max_steps, N, C, H, nears,
                                                                fars, noises, counts);
        march::march_scan_kernel<<<1, 1024, 0, st>>>(counts, N, rays, counter);
        march::march_write_kernel<<<cdiv(N, 128), 128, 0, st>>>(rays_o, rays_d, grid, bound, dt_gamma, max_steps, N, C, H, M,
                                                                nears, fars, noises, counts, rays, xyzs, dirs, deltas);
    } else {
        // warp per ray, single walk into per-ray slabs (scratch after the counts), scan, packed copy
        float* slab_xyz = reinterpret_cast<float*>(static_cast<uint8_t*>(workspace) + 256 + (((size_t)N * sizeof(int) + 255) / 256) * 256);
        float* slab_delta = slab_xyz + (size_t)N * max_steps * 3;
        const int blocks = cdiv((uint64_t)N * 32, 128);
        if (dt_gamma == 0.f && march::g_thread_march_min_rays && N >= march::g_thread_march_min_rays) {
            float4* slab4 = reinterpret_cast<float4*>(slab_xyz);   // (256-byte aligned; 16 of the 20 bytes per row are used)
            march::march_slab_thread_kernel<<<cdiv(N, 128), 128, 0, st>>>(rays_o, rays_d, grid, bound, max_steps, N, C, H, nears, fars,
                                                                         noises, counts, slab4, nullptr, rays, counter);
            march::march_scan_kernel<<<1, 1024, 0, st>>>(counts, N, rays, counter);
            march::march_compact4_kernel<<<cdiv((uint64_t)N * 32, 256), 256, 0, st>>>(rays_d, rays, slab4, nears, noises, max_steps, N, M,
                                                                                     C, H, xyzs, dirs, deltas);
            return launch_status();
        }
        if (N <= 8192) {
            // few rays per launch (a data-parallel rank's chain): the LAST block of the walk scans the counts - one launch
            // and one dependent-launch gap less.  The election counter (first word of the workspace) must be zero on entry:
            // the caller zero-fills the head of a NEW workspace once, the electing block leaves it zero again (a memset
            // node per call cost 2-4 us on the step's critical path)
            march::march_slab_kernel<<<blocks, 128, 0, st>>>(rays_o, rays_d, grid, bound, dt_gamma, max_steps, N, C, H, nears, fars,
                                                             noises, counts, slab_xyz, slab_delta, blocks_done, rays, counter);
        } else {
            // many rays: a 1024-thread scan kernel beats 128 threads of the last walking block
            march::march_slab_kernel<<<blocks, 128, 0, st>>>(rays_o, rays_d, grid, bound, dt_gamma, max_steps, N, C, H, nears, fars,
                                                             noises, counts, slab_xyz, slab_delta, nullptr, rays, counter);
            march::march_scan_kernel<<<1, 1024, 0, st>>>(counts, N, rays, counter);
        }
        march::march_compact_kernel<<<cdiv((uint64_t)N * 32, 256), 256, 0, st>>>(rays_d, rays, slab_xyz, slab_delta, max_steps, N, M,
                                                                                 xyzs, dirs, deltas);
    }
    return launch_status();
}

extern "C" int ngp_march_rays_train_packed(const float* rays_o, const float* rays_d, const uint8_t* grid, float bound,
                                           float dt_gamma, uint32_t max_steps, uint32_t N, uint32_t C, uint32_t H, uint32_t M,
                                           const float* nears, const float* fars, float* xyzs, float* dirs, float* deltas,
                                           int* rays, int* counter, const float* noises, void* stream) {
    if (!rays_o || !rays_d || !grid || !nears || !fars || !xyzs || !deltas || !rays || !counter || !noises)
        return NGP_ERR_BAD_ARG;
    if (C == 0 || H == 0 || max_steps == 0) return NGP_ERR_BAD_ARG;
    if (max_steps > 2048 || (reinterpret_cast<uintptr_t>(deltas) & 7)) return NGP_ERR_UNSUPPORTED;   // 4 x max_steps floats of smem
    if (N == 0) return NGP_OK;
    march::march_packed_kernel<<<cdiv((uint64_t)N * 32, 128), 128, 4 * max_steps * sizeof(float), as_stream(stream)>>>(
        rays_o, rays_d, grid, bound, dt_gamma, max_steps, N, C, H, M, nears, fars, noises, xyzs, dirs, deltas, rays, counter);
    return launch_status();
}

extern "C" int ngp_composite_rays_train_forward(const float* sigmas, const float* rgbs, const float* deltas,
                                                const int* rays, uint32_t M, uint32_t N, float T_thresh,
                                                float* weights_sum, float* depth, float* image, void* stream) {
    if (!sigmas || !rgbs || !deltas || !rays || !weights_sum || !depth || !image) return NGP_ERR_BAD_ARG;
    if (N == 0) return NGP_OK;
    march::composite_train_fwd_kernel<<<cdiv((uint64_t)N * 32, 256), 256, 0, as_stream(stream)>>>(
        sigmas, rgbs, deltas, rays, M, N, T_thresh, weights_sum, depth, image);
    return launch_status();
}

extern "C" int ngp_composite_rays_train_backward(const float* grad_weights_sum, const float* grad_image,
                                                 const float* sigmas, const float* rgbs, const float* deltas,
                                                 const int* rays, const float* weights_sum, const float* image,
                                                 uint32_t M, uint32_t N, float T_thresh, float* grad_sigmas,
                                                 float* grad_rgbs, void* stream) {
    if (!grad_weights_sum || !grad_image || !sigmas || !rgbs || !deltas || !rays || !weights_sum || !image ||
        !grad_sigmas || !grad_rgbs)
        return NGP_ERR_BAD_ARG;
    if (N == 0) return NGP_OK;
    march::composite_train_bwd_kernel<true><<<cdiv((uint64_t)N * 32, 256), 256, 0, as_stream(stream)>>>(
        grad_weights_sum, grad_image, sigmas, rgbs, deltas, rays, weights_sum, image, M, N, T_thresh, grad_sigmas,
        grad_rgbs);
    return launch_status();
}

extern "C" int ngp_train_prologue(const float* rays_o, const float* rays_d, const float* aabb, uint32_t N, float min_near,
                                  float* nears, float* fars, int* counters, uint32_t n_counters, float* loss,
                                  int* step_counter, int* local_step, int* cur_row, float* noises, uint64_t* rng,
                                  void* stream) {
    if (!rays_o || !rays_d || !aabb || !nears || !fars || (noises && !rng)) return NGP_ERR_BAD_ARG;
    march::train_prologue_kernel<<<N ? cdiv(N, 128) : 1, 128, 0, as_stream(stream)>>>(
        rays_o, rays_d, aabb, N, min_near, nears, fars, counters, n_counters, loss, step_counter, local_step, cur_row, noises,
        reinterpret_cast<unsigned long long*>(rng));
    return launch_status();
}

static int make_raygen(march::RayGen& g, const float* poses, const float* intrinsics, uint32_t B, uint32_t H, uint32_t W,
                       uint32_t row0, uint32_t row_stride, uint32_t n_rows, int intrinsics_per_view) {
    if (!poses || !intrinsics) return NGP_ERR_BAD_ARG;
    if (row_stride == 0) row_stride = 1;
    if (n_rows == 0) n_rows = (H - row0 + row_stride - 1) / row_stride;
    if (B == 0 || W == 0 || row0 >= H || row0 + (uint64_t)(n_rows - 1) * row_stride >= H) return NGP_ERR_BAD_ARG;
    if ((uint64_t)B * n_rows * W > 0x7fffffffull) return NGP_ERR_BAD_ARG;
    g.poses = poses; g.intrinsics = intrinsics; g.B = B; g.W = W; g.n_rows = n_rows; g.row0 = row0; g.row_stride = row_stride;
    g.intr_per_view = intrinsics_per_view ? 1u : 0u;
    return NGP_OK;
}

extern "C" int ngp_get_rays(const float* poses, const float* intrinsics, int intrinsics_per_view, uint32_t B, uint32_t H,
                            uint32_t W, uint32_t row0, uint32_t row_stride, uint32_t n_rows, float* rays_o, float* rays_d,
                            void* stream) {
    if (!rays_o || !rays_d) return NGP_ERR_BAD_ARG;
    march::RayGen g;
    const int rc = make_raygen(g, poses, intrinsics, B, H, W, row0, row_stride, n_rows, intrinsics_per_view);
    if (rc != NGP_OK) return rc;
    const uint32_t N = g.B * g.n_rows * g.W;
    march::get_rays_kernel<<<cdiv(N, 256), 256, 0, as_stream(stream)>>>(g, rays_o, rays_d);
    return launch_status();
}

extern "C" int ngp_train_prologue_rays(const float* poses, const float* intrinsics, int intrinsics_per_view, uint32_t B,
                                       uint32_t H, uint32_t W, uint32_t row0, uint32_t row_stride, uint32_t n_rows,
                                       float* rays_o, float* rays_d, const float* aabb, float min_near, float* nears,
                                       float* fars, int* counters, uint32_t n_counters, float* loss, int* step_counter,
                                       int* local_step, int* cur_row, float* noises, uint64_t* rng, void* stream) {
    if (!rays_o || !rays_d || !aabb || !nears || !fars || (noises && !rng)) return NGP_ERR_BAD_ARG;
    march::RayGen g;
    const int rc = make_raygen(g, poses, intrinsics, B, H, W, row0, row_stride, n_rows, intrinsics_per_view);
    if (rc != NGP_OK) return rc;
    const uint32_t N = g.B * g.n_rows * g.W;
    march::train_prologue_rays_kernel<<<cdiv(N, 128), 128, 0, as_stream(stream)>>>(
        g, rays_o, rays_d, aabb, min_near, nears, fars, counters, n_counters, loss, step_counter, local_step, cur_row, noises,
        reinterpret_cast<unsigned long long*>(rng));
    return launch_status();
}

extern "C" int ngp_train_light(const float* rays_o, uint64_t* rng, int advance, float* light, void* stream) {
    if (!rays_o || !rng || !light) return NGP_ERR_BAD_ARG;
    march::train_light_kernel<<<1, 32, 0, as_stream(stream)>>>(rays_o, reinterpret_cast<unsigned long long*>(rng), advance, light);
    return launch_status();
}

extern "C" int ngp_train_ray_loss(const float* sigmas, const float* rgbs, const float* deltas, const int* rays, uint32_t M,
                                  uint32_t N, float T_thresh, const void* bg_half, float bg_const, const float* grad_pred,
                                  uint32_t pixels_per_view, uint32_t ray_base, uint32_t n_rays_total, float lambda_entropy,
                                  const float* scale, float* weights_sum, float* depth, float* image, float* grad_bg,
                                  float* grad_sigmas, float* grad_rgbs, float* loss, const int* counter,
                                  unsigned long long* samples_total, int* step_counter, const int* cur_row, void* stream) {
    if (!sigmas || !rgbs || !deltas || !rays || !grad_pred || !weights_sum || !depth || !image || !grad_sigmas || !grad_rgbs)
        return NGP_ERR_BAD_ARG;
    if (n_rays_total == 0) n_rays_total = N;
    if ((uint64_t)ray_base + N > n_rays_total) return NGP_ERR_BAD_ARG;
    if (pixels_per_view && n_rays_total % pixels_per_view != 0) return NGP_ERR_BAD_ARG;
    if (N == 0) return NGP_OK;
    march::RayLossArgs a;
    a.sigmas = sigmas; a.rgbs = rgbs; a.deltas = deltas; a.rays = rays; a.M = M; a.N = N; a.T_thresh = T_thresh;
    a.bg = static_cast<const __half*>(bg_half); a.bg_const = bg_const; a.G = grad_pred; a.hw = pixels_per_view;
    a.ray_base = ray_base; a.n_total = n_rays_total;
    a.lambda = lambda_entropy; a.scale = scale; a.weights_sum = weights_sum; a.depth = depth; a.image = image;
    a.d_bg = grad_bg; a.grad_sigmas = grad_sigmas; a.grad_rgbs = grad_rgbs; a.loss = loss; a.counter = counter;
    a.samples_total = samples_total; a.step_counter = step_counter; a.cur_row = cur_row;
    march::train_ray_loss_kernel<<<cdiv((uint64_t)N * 32, 256), 256, 0, as_stream(stream)>>>(a);
    return launch_status();
}

extern "C" int ngp_march_rays(uint32_t n_alive, uint32_t n_step, const int* rays_alive, const float* rays_t,
                              const float* rays_o, const float* rays_d, float bound, float dt_gamma,
                              uint32_t max_steps, uint32_t C, uint32_t H, const uint8_t* grid, const float* nears,
                              const float* fars, float* xyzs, float* dirs, float* deltas, const float* noises,
                              void* stream) {
    if (!rays_alive || !rays_t || !rays_o || !rays_d || !grid || !nears || !fars || !xyzs || !dirs || !deltas || !noises)
        return NGP_ERR_BAD_ARG;
    if (C == 0 || H == 0 || max_steps == 0) return NGP_ERR_BAD_ARG;
    if (n_alive == 0 || n_step == 0) return NGP_OK;
    if (n_step == 1 && march::g_infer_warp_march) {   // opt-in (ngp_march_set_option 1): pays only when the rays start far from
        //                                                  the object, i.e. on a frame's FIRST call; the device-driven loop
        //                                                  (ngp_render_infer_loop) selects it there by itself
        // (the caller's buffers are zero-filled, raymarching.py:334-336: rays that emit nothing leave their slot untouched)
        const int blocks = min(cdiv((uint64_t)n_alive * 32, 128), num_sms() * 16);
        march::march_infer_warp_kernel<<<blocks, 128, 0, as_stream(stream)>>>(n_alive, n_step, rays_alive, rays_t, rays_o, rays_d, bound,
                                                                               dt_gamma, max_steps, C, H, grid, fars, xyzs, dirs, deltas,
                                                                               noises);
        return launch_status();
    }
    march::march_infer_kernel<<<cdiv(n_alive, 128), 128, 0, as_stream(stream)>>>(
        n_alive, n_step, rays_alive, rays_t, rays_o, rays_d, bound, dt_gamma, max_steps, C, H, grid, nears, fars, xyzs, dirs,
        deltas, noises);
    return launch_status();
}

extern "C" int ngp_composite_rays(uint32_t n_alive, uint32_t n_step, float T_thresh, int* rays_alive, float* rays_t,
                                  const float* sigmas, const float* rgbs, const float* deltas, float* weights_sum,
                                  float* depth, float* image, void* stream) {
    if (!rays_alive || !rays_t || !sigmas || !rgbs || !deltas || !weights_sum || !depth || !image) return NGP_ERR_BAD_ARG;
    if (n_alive == 0) return NGP_OK;
    march::composite_infer_kernel<<<cdiv(n_alive, 128), 128, 0, as_stream(stream)>>>(
        n_alive, n_step, T_thresh, rays_alive, rays_t, sigmas, rgbs, deltas, weights_sum, depth, image);
    return launch_status();
}

extern "C" uint64_t ngp_compact_alive_workspace(uint32_t n_alive) {
    return (uint64_t)cdiv(n_alive > 0 ? n_alive : 1, march::kCompactBlock) * sizeof(int);
}

extern "C" int ngp_compact_alive(const int* rays_alive, uint32_t n_alive, int* out, int* n_out, void* workspace,
                                 uint64_t workspace_bytes, void* stream) {
    if (!rays_alive || !out || !n_out) return NGP_ERR_BAD_ARG;
    cudaStream_t st = as_stream(stream);
    if (n_alive == 0) { cudaMemsetAsync(n_out, 0, sizeof(int), st); return launch_status(); }
    if (!workspace || workspace_bytes < ngp_compact_alive_workspace(n_alive)) return NGP_ERR_WORKSPACE;
    const int blocks = cdiv(n_alive, march::kCompactBlock);
    int* block_counts = static_cast<int*>(workspace);
    march::compact_count_kernel<<<blocks, march::kCompactBlock, 0, st>>>(rays_alive, n_alive, block_counts);
    march::compact_scatter_kernel<<<blocks, march::kCompactBlock, 0, st>>>(rays_alive, n_alive, block_counts, out, n_out);
    return launch_status();
}

// -------------------------------------------------------------------------------------------------
// ngp_render_infer_loop: the whole inference loop of run_cuda as ONE graph launch (init node -> conditional WHILE node
// whose body is march -> fused field -> composite -> compaction -> plan).  The executable graph is cached per argument
// set (pointers and scalars are baked into its nodes), so callers keep their buffers in a persistent workspace.
// -------------------------------------------------------------------------------------------------
namespace {
struct InferLoopKey {
    const void* p[20];
    uint32_t u[10];
    float f[4];
    int dev;
    bool operator==(const InferLoopKey& o) const { return memcmp(this, &o, sizeof(InferLoopKey)) == 0; }
};
struct InferLoopEntry {
    InferLoopKey key;
    cudaGraph_t graph = nullptr;
    cudaGraphExec_t exec = nullptr;
    uint64_t stamp = 0;
    bool valid = false;
};
constexpr int kInferCache = 8;
InferLoopEntry g_infer_cache[kInferCache];
uint64_t g_infer_stamp = 0;

inline uint64_t align_up(uint64_t v, uint64_t a) { return (v + a - 1) / a * a; }
struct InferLayout {
    uint64_t state, alive, rays_t, xyzs, deltas, sigma, rgb, blocks, total;
};
inline InferLayout infer_layout(uint32_t N) {
    InferLayout l;
    const uint64_t cap = align_up((uint64_t)N, 128) + 128;   // field tiles are 128 rows
    uint64_t o = 0;
    l.state = o; o += 256;
    l.alive = o; o += align_up((uint64_t)2 * N * 4, 256);
    l.rays_t = o; o += align_up((uint64_t)N * 4, 256);
    l.xyzs = o; o += align_up(cap * 12, 256);
    l.deltas = o; o += align_up(cap * 8, 256);
    l.sigma = o; o += align_up(cap * 4, 256);
    l.rgb = o; o += align_up(cap * 12, 256);
    l.blocks = o; o += align_up((uint64_t)cdiv(N ? N : 1, march::kCompactBlock) * 4, 256);
    l.total = o;
    return l;
}
}  // namespace

extern "C" uint64_t ngp_render_infer_workspace(uint32_t N) { return infer_layout(N).total; }

static int render_infer_loop_impl(const float* rays_o, const float* rays_d, const float* nears, const float* fars, uint32_t N,
                                  float bound, float dt_gamma, uint32_t max_steps, uint32_t C, uint32_t H,
                                  const uint8_t* grid, float T_thresh, const float* noises, const void* table, const void* quads,
                                  const int* offsets, uint32_t L, uint32_t Cfeat, float S, uint32_t Hres, uint32_t gridtype,
                                  int align_corners, const void* w1, const void* b1, const void* w2, const void* b2,
                                  const void* w3, const void* b3, uint32_t hidden, uint32_t out_dim, float* weights_sum,
                                  float* depth, float* image, void* workspace, uint64_t workspace_bytes, void* stream) {
    if (!rays_o || !rays_d || !nears || !fars || !grid || !table || !offsets || !w1 || !b1 || !w2 || !b2 || !w3 || !b3 ||
        !weights_sum || !depth || !image)
        return NGP_ERR_BAD_ARG;
    if (C == 0 || H == 0 || max_steps == 0) return NGP_ERR_BAD_ARG;
    if (L != 16 || Cfeat != 2 || hidden != 64 || out_dim != 4) return NGP_ERR_UNSUPPORTED;
    if (N == 0) return NGP_OK;
    const InferLayout lay = infer_layout(N);
    if (!workspace || workspace_bytes < lay.total) return NGP_ERR_WORKSPACE;
    uint8_t* ws = static_cast<uint8_t*>(workspace);
    march::InferState* st = reinterpret_cast<march::InferState*>(ws + lay.state);
    int* alive = reinterpret_cast<int*>(ws + lay.alive);
    float* rays_t = reinterpret_cast<float*>(ws + lay.rays_t);
    float* xyzs = reinterpret_cast<float*>(ws + lay.xyzs);
    float* deltas = reinterpret_cast<float*>(ws + lay.deltas);
    float* sigma = reinterpret_cast<float*>(ws + lay.sigma);
    float* rgb = reinterpret_cast<float*>(ws + lay.rgb);
    int* blocks = reinterpret_cast<int*>(ws + lay.blocks);

    InferLoopKey key;
    memset(&key, 0, sizeof(key));
    const void* ptrs[] = {rays_o, rays_d, nears, fars, grid, noises, table, offsets, w1, b1, w2, b2, w3, b3, weights_sum, depth,
                          image, workspace, quads};
    for (size_t i = 0; i < sizeof(ptrs) / sizeof(ptrs[0]); ++i) key.p[i] = ptrs[i];
    const uint32_t us[] = {N, max_steps, C, H, L, Cfeat, Hres, gridtype, (uint32_t)(align_corners != 0), 0u};
    for (size_t i = 0; i < 10; ++i) key.u[i] = us[i];
    key.f[0] = bound; key.f[1] = dt_gamma; key.f[2] = T_thresh; key.f[3] = S;
    if (cudaGetDevice(&key.dev) != cudaSuccess) return launch_status();

    InferLoopEntry* hit = nullptr;
    InferLoopEntry* victim = &g_infer_cache[0];
    for (int i = 0; i < kInferCache; ++i) {
        InferLoopEntry& e = g_infer_cache[i];
        if (e.valid && e.key == key) { hit = &e; break; }
        if (!e.valid || e.stamp < victim->stamp || (victim->valid && !e.valid)) victim = &e;
    }
    if (!hit) {
        if (victim->valid) {
            cudaGraphExecDestroy(victim->exec);
            cudaGraphDestroy(victim->graph);
            victim->valid = false;
        }
        cudaGraph_t graph = nullptr;
        cudaGraphExec_t exec = nullptr;
        cudaStream_t cs = nullptr;
        cudaError_t e = cudaGraphCreate(&graph, 0);
        int rc = NGP_OK;
        do {
            if (e != cudaSuccess) break;
            // node 1: loop state + accumulators
            cudaGraphNode_t init_node;
            {
                cudaKernelNodeParams kp;
                memset(&kp, 0, sizeof(kp));
                void* args[] = {(void*)&N, (void*)&nears, (void*)&alive, (void*)&rays_t, (void*)&weights_sum, (void*)&depth,
                                (void*)&image, (void*)&st};
                kp.func = reinterpret_cast<void*>(march::infer_init_kernel);
                kp.gridDim = dim3(cdiv(N, 256));
                kp.blockDim = dim3(256);
                kp.kernelParams = args;
                if ((e = cudaGraphAddKernelNode(&init_node, graph, nullptr, 0, &kp)) != cudaSuccess) break;
            }
            // node 2: WHILE (condition defaults to 1 at every launch; infer_plan_kernel sets it at the end of each pass)
            cudaGraphConditionalHandle handle;
            if ((e = cudaGraphConditionalHandleCreate(&handle, graph, 1, cudaGraphCondAssignDefault)) != cudaSuccess) break;
            cudaGraphNodeParams cp = {cudaGraphNodeTypeConditional};
            cp.conditional.handle = handle;
            cp.conditional.type = cudaGraphCondTypeWhile;
            cp.conditional.size = 1;
            cudaGraphNode_t while_node;
            if ((e = cudaGraphAddNode(&while_node, graph, &init_node, 1, &cp)) != cudaSuccess) break;
            cudaGraph_t body = cp.conditional.phGraph_out[0];
            if ((e = cudaStreamCreateWithFlags(&cs, cudaStreamNonBlocking)) != cudaSuccess) break;
            if ((e = cudaStreamBeginCaptureToGraph(cs, body, nullptr, nullptr, 0, cudaStreamCaptureModeThreadLocal)) != cudaSuccess) break;
            const int persistent = num_sms() * 8;
            const int g128 = min(cdiv(N, 128), persistent);
            const int g_march = N <= 16384u ? min(cdiv((uint64_t)N * 32, 128), num_sms() * 16) : g128;   // (warp-per-ray first pass)
            march::infer_march_kernel<<<g_march, 128, 0, cs>>>(st, N, alive, rays_t, rays_o, rays_d, bound, dt_gamma, max_steps, C, H, grid,
                                                            fars, xyzs, deltas, noises);
            rc = quads ? ngp_field_forward_quads(xyzs, (uint32_t)(align_up((uint64_t)N, 128)), &st->rows, table, quads, offsets, L, Cfeat,
                                                 S, Hres, gridtype, align_corners, bound, w1, b1, w2, b2, w3, b3, hidden, out_dim, sigma,
                                                 rgb, nullptr, nullptr, nullptr, cs)
                       : ngp_field_forward(xyzs, (uint32_t)(align_up((uint64_t)N, 128)), &st->rows, table, offsets, L, Cfeat, S, Hres,
                                           gridtype, align_corners, bound, w1, b1, w2, b2, w3, b3, hidden, out_dim, sigma, rgb, nullptr,
                                           nullptr, nullptr, cs);
            march::infer_composite_kernel<<<g128, 128, 0, cs>>>(st, N, T_thresh, alive, rays_t, sigma, rgb, deltas, weights_sum, depth,
                                                                image);
            const int cblocks = cdiv(N, march::kCompactBlock);
            march::infer_compact_count_kernel<<<cblocks, march::kCompactBlock, 0, cs>>>(st, N, alive, blocks);
            march::infer_compact_scatter_kernel<<<cblocks, march::kCompactBlock, 0, cs>>>(st, N, alive, blocks);
            march::infer_plan_kernel<<<1, 32, 0, cs>>>(st, N, max_steps, handle, 1);
            cudaGraph_t captured = nullptr;
            e = cudaStreamEndCapture(cs, &captured);
            if (e != cudaSuccess || rc != NGP_OK) break;
            if ((e = cudaGraphInstantiate(&exec, graph, 0)) != cudaSuccess) break;
        } while (false);
        if (cs) cudaStreamDestroy(cs);
        if (e != cudaSuccess || rc != NGP_OK || !exec) {
            if (exec) cudaGraphExecDestroy(exec);
            if (graph) cudaGraphDestroy(graph);
            cudaGetLastError();
            fprintf(stderr, "[ngp_b200] ngp_render_infer_loop: conditional graph not built (%s, rc %d); the caller runs the host loop\n",
                    e != cudaSuccess ? cudaGetErrorString(e) : "no error", rc);
            return NGP_ERR_UNSUPPORTED;
        }
        victim->key = key; victim->graph = graph; victim->exec = exec; victim->valid = true;
        hit = victim;
    }
    hit->stamp = ++g_infer_stamp;
    const cudaError_t le = cudaGraphLaunch(hit->exec, as_stream(stream));
    if (le != cudaSuccess) { cudaGetLastError(); return (int)le; }
    return launch_status();
}

extern "C" int ngp_render_infer_loop(const float* rays_o, const float* rays_d, const float* nears, const float* fars, uint32_t N,
                                     float bound, float dt_gamma, uint32_t max_steps, uint32_t C, uint32_t H,
                                     const uint8_t* grid, float T_thresh, const float* noises, const void* table,
                                     const int* offsets, uint32_t L, uint32_t Cfeat, float S, uint32_t Hres, uint32_t gridtype,
                                     int align_corners, const void* w1, const void* b1, const void* w2, const void* b2,
                                     const void* w3, const void* b3, uint32_t hidden, uint32_t out_dim, float* weights_sum,
                                     float* depth, float* image, void* workspace, uint64_t workspace_bytes, void* stream) {
    return render_infer_loop_impl(rays_o, rays_d, nears, fars, N, bound, dt_gamma, max_steps, C, H, grid, T_thresh, noises, table,
                                  nullptr, offsets, L, Cfeat, S, Hres, gridtype, align_corners, w1, b1, w2, b2, w3, b3, hidden, out_dim,
                                  weights_sum, depth, image, workspace, workspace_bytes, stream);
}

// the same loop with the field reading the embeddings through a quad table (ngp_grid_quad_table, built by the caller from
// the SAME fp16 table before the launch)
extern "C" int ngp_render_infer_loop_quads(const float* rays_o, const float* rays_d, const float* nears, const float* fars,
                                           uint32_t N, float bound, float dt_gamma, uint32_t max_steps, uint32_t C, uint32_t H,
                                           const uint8_t* grid, float T_thresh, const float* noises, const void* table,
                                           const void* quads, const int* offsets, uint32_t L, uint32_t Cfeat, float S,
                                           uint32_t Hres, uint32_t gridtype, int align_corners, const void* w1, const void* b1,
                                           const void* w2, const void* b2, const void* w3, const void* b3, uint32_t hidden,
                                           uint32_t out_dim, float* weights_sum, float* depth, float* image, void* workspace,
                                           uint64_t workspace_bytes, void* stream) {
    if (!quads) return NGP_ERR_BAD_ARG;
    return render_infer_loop_impl(rays_o, rays_d, nears, fars, N, bound, dt_gamma, max_steps, C, H, grid, T_thresh, noises, table,
                                  quads, offsets, L, Cfeat, S, Hres, gridtype, align_corners, w1, b1, w2, b2, w3, b3, hidden, out_dim,
                                  weights_sum, depth, image, workspace, workspace_bytes, stream);
}

// device int[8] view of the loop state after the last launch on this workspace: n_alive, n_step, step, cur, iters, ...
extern "C" int ngp_render_infer_state(const void* workspace, int* state_host, void* stream) {
    if (!workspace || !state_host) return NGP_ERR_BAD_ARG;
    cudaError_t e = cudaMemcpyAsync(state_host, workspace, sizeof(march::InferState), cudaMemcpyDeviceToHost, as_stream(stream));
    if (e == cudaSuccess) e = cudaStreamSynchronize(as_stream(stream));
    return e == cudaSuccess ? NGP_OK : (int)e;
}

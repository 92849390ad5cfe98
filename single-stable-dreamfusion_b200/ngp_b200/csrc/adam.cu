// The optimisation step of the `-O` train step: GradScaler.unscale_ / found_inf + Adam (betas, eps, per-group lr, LambdaLR
// decay) + GradScaler.update + refresh of the fp16 shadow of the parameters + zero-fill of the gradient bucket, over ONE
// flat fp32 buffer, as two launches:
//
//   ngp_check_finite / ngp_check_finite_fold   found_inf of the bucket -> state[3] (the fold variant first adds the
//                                              odd-frame twin of the table gradient into the bucket)
//   ngp_adam_step     (adam_step_kernel)       the update on one GPU, or after an NCCL all-reduce of the bucket
//   ngp_adam_step_dp  (adam_dp_kernel)         world > 1 over NVLink peer memory, with the gradient all-reduce fused in
//
// Reference semantics: `scaler.step(optimizer); scaler.update()` on Adam(betas (0.9, 0.99), eps 1e-15) with per-group lr
// and LambdaLR (main.py:128-131, network_grid.py:170-181, nerf/utils.py:708-713); with world > 1 the gradients are
// reduced over ranks as DistributedDataParallel (the reference's dormant wrap, nerf/utils.py:200-202) would.
//
// Both update kernels take one Args and share the step coefficients, the per-element update, the fp16 packing, the
// last-block election and the GradScaler tail below, so that from the same summed gradient they compute the same bits.
//
// adam_dp_kernel: every rank checks its OWN bucket first (ngp_check_finite: a sum of <= 8 finite fp32 gradients is finite,
// so the reduced gradient is non-finite iff an addend is) and the verdict rides on B0's flag exchange: after B0 every block
// of every rank knows the global found_inf.  Block b then owns sub-slice b of its rank's slice end to end:
//     B0(b)  flags of block b of all ranks (payload: local found_inf | error)
//     P      per element: `world` P2P loads (or one multimem.ld_reduce) -> sum -> Adam -> new parameter + fp16 shadow
//            stored to every replica (or one multimem.st each).  The moments are sharded: rank r keeps slice r of exp_avg /
//            exp_avg_sq, and the all-gather half of the all-reduce moves parameters instead of gradients, so the optimizer
//            arithmetic is done once per element, not `world` times
//     B2(b)  every rank's block b is done: its reads of MY bucket and its writes to MY replica have completed
//     Z      zero sub-slice b of ALL `world` slices of my bucket (exactly what the peers' blocks b have finished reading)
// No block ever waits for another block of its own grid, so the grid can be small (it runs beside the next step's ray
// marching in pipelined mode) and needs no co-residency guarantee.
//
// Cross-GPU barriers are flag exchanges in peer memory (st.release.sys / ld.acquire.sys), one slot per (barrier, block,
// source rank), carrying a monotonically increasing epoch kept on the device, so the kernel is CUDA-graph replayable.
// Every spin is bounded by a wall-clock timeout (default 20 s, ngp_dp_set_option(0, milliseconds)): a lost peer raises
// the sticky error flag state[5] instead of hanging the GPU; blocks that learn of it apply nothing and every later launch
// returns at once.  TrainStep polls the flag and raises.
#include <math.h>

#include "common.cuh"

namespace ngp {
namespace adam {

constexpr uint32_t kMaxWorld = NGP_DP_MAX_WORLD;
constexpr uint32_t kMaxBlocks = NGP_DP_MAX_BLOCKS;
uint64_t g_spin_timeout_ns = 20ull * 1000 * 1000 * 1000;  // 20 s; ngp_dp_set_option(0, ms)
int g_blocks = 0;                                          // adam_dp_kernel grid, 0 = sized from the slice; ngp_dp_set_option(1, blocks)

struct Args {
    float* p;          // parameters (flat fp32), this rank's replica
    float* g;          // gradient bucket (flat fp32), scaled by state[0]
    float* m;          // exp_avg      (adam_dp_kernel: only this rank's slice is maintained)
    float* v;          // exp_avg_sq
    __half* h;         // optional fp16 shadow of p
    uint64_t n;
    uint32_t n_seg;
    uint64_t seg_end[NGP_ADAM_MAX_SEGMENTS];  // exclusive end of each lr group in the flat buffer
    float seg_lr[NGP_ADAM_MAX_SEGMENTS];
    float beta1, beta2, eps;
    float grad_div;    // extra divisor for the gradients (data-parallel world size for a mean)
    float lr_decay_ln; // lr multiplier = exp(lr_decay_ln * min(step, lr_decay_steps))  (LambdaLR 0.1^(it/iters))
    float lr_decay_steps;
    float growth, backoff;
    uint32_t growth_interval;
    float* state;      // [0] scale [1] growth tracker [2] steps [3] found_inf [4] skipped [5] error flag [6] armed
    int deferred;      // 1: a launch that finds state[6] == 0 applies nothing and only raises state[6] (pipelined step)
    uint32_t* sync;    // [0] block election (zero between launches), adam_dp_kernel: [1] barrier epoch
    int zero_grads;    // adam_step_kernel: zero-fill the bucket on the way out (adam_dp_kernel always does)
    // adam_dp_kernel only
    uint32_t rank, world;
    float* peer_g[kMaxWorld];
    float* peer_p[kMaxWorld];
    __half* peer_h[kMaxWorld];
    uint32_t* peer_flags[kMaxWorld];  // each: [3][kMaxBlocks][kMaxWorld] uint32, zero-initialised
    // optional NVLink SHARP (NVLS) multicast views of the same three buffers: one multimem.ld_reduce returns the sum of an
    // element over all replicas (added inside the switch), one multimem.st writes an element to every replica
    float* mc_g;
    float* mc_p;
    __half* mc_h;
    uint64_t timeout_ns;
};

// ---- shared by both update kernels ---------------------------------------------------------------------------------
// Adam's bias corrections of step step0 + 1 and the LambdaLR factor: the same expressions as torch's fused Adam (evaluated
// in double, then narrowed).  Once per block by one thread: two double-precision pow() per THREAD made adam_step_kernel
// 35 us instead of 23 (fp64 is slow here).
NGP_DEVINL void step_coefficients(const Args& a, float step0, float* coef) {
    const float t = step0 + 1.f;
    coef[0] = (float)(1.0 - pow((double)a.beta1, (double)t));
    coef[1] = (float)sqrt(1.0 - pow((double)a.beta2, (double)t));
    coef[2] = a.lr_decay_ln != 0.f ? expf(a.lr_decay_ln * fminf(step0, a.lr_decay_steps)) : 1.f;
}

// the per-launch constants of the update: the step coefficients and the unscale factor
struct Update {
    float bc1, bc2_sqrt, lr_mult, inv, w1, w2;
    NGP_DEVINL Update(const Args& a, const float* coef, float scale)
        : bc1(coef[0]), bc2_sqrt(coef[1]), lr_mult(coef[2]), inv(1.0f / (scale * a.grad_div)), w1(1.f - a.beta1),
          w2(1.f - a.beta2) {}
};

// Adam on elements e0 .. e0 + 3; g holds their scaled (summed) gradients
NGP_DEVINL void adam4(const Args& a, const Update& u, uint64_t e0, const float g[4], float p[4], float m[4], float v[4]) {
#pragma unroll
    for (uint32_t j = 0; j < 4; ++j) {
        // learning-rate group of this element (groups are few and long; segments may split a float4)
        float lr = a.seg_lr[0];
#pragma unroll
        for (uint32_t s = 1; s < NGP_ADAM_MAX_SEGMENTS; ++s)
            if (s < a.n_seg && e0 + j >= a.seg_end[s - 1]) lr = a.seg_lr[s];
        const float step_size = lr * u.lr_mult / u.bc1;
        const float gr = g[j] * u.inv;
        m[j] = fmaf(u.w1, gr - m[j], m[j]);                 // exp_avg.lerp_(grad, 1 - beta1)
        v[j] = a.beta2 * v[j] + u.w2 * gr * gr;
        const float denom = sqrtf(v[j]) / u.bc2_sqrt + a.eps;
        p[j] -= step_size * m[j] / denom;
    }
}

NGP_DEVINL uint2 pack_half4(const float p[4]) {
    __half2 h0 = __floats2half2_rn(p[0], p[1]), h1 = __floats2half2_rn(p[2], p[3]);
    uint2 raw;
    raw.x = *reinterpret_cast<uint32_t*>(&h0); raw.y = *reinterpret_cast<uint32_t*>(&h1);
    return raw;
}

// Every block signs off once all its threads are past their last read of the step's state; true in the last block, whose
// thread 0 then applies the scaler update and resets sync[0].
NGP_DEVINL bool last_block(uint32_t* done) {
    __shared__ bool s_last;
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        s_last = atomicAdd(done, 1u) == gridDim.x - 1;
    }
    __syncthreads();
    return s_last;
}

// GradScaler.update() + the step count (torch/amp/grad_scaler.py: _amp_update_scale_); one thread of the last block
NGP_DEVINL void scaler_update(const Args& a, float scale, float step0, bool skip) {
    float tracker = a.state[1];
    float new_scale = scale;
    if (skip) {
        new_scale = scale * a.backoff;
        tracker = 0.f;
        a.state[4] += 1.f;
    } else {
        a.state[2] = step0 + 1.f;
        tracker += 1.f;
        if (tracker >= (float)a.growth_interval) {
            const float grown = scale * a.growth;
            if (isfinite(grown)) new_scale = grown;
            tracker = 0.f;
        }
    }
    a.state[0] = new_scale;
    a.state[1] = tracker;
    a.state[3] = 0.f;
}

// ---- found_inf -------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) check_finite_kernel(const float4* __restrict__ g4, const float* __restrict__ g,
                                                           uint64_t n, float* __restrict__ found_inf) {
    const uint64_t n4 = n / 4;
    bool bad = false;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (uint64_t)gridDim.x * blockDim.x) {
        const float4 v = __ldg(g4 + i);
        // x - x is 0 for finite x and NaN for +-inf / NaN
        const float s = (v.x - v.x) + (v.y - v.y) + (v.z - v.z) + (v.w - v.w);
        bad = bad || (s != 0.f);
    }
    if (blockIdx.x == 0 && threadIdx.x < (n & 3)) {
        const float v = g[n4 * 4 + threadIdx.x];
        bad = bad || ((v - v) != 0.f);
    }
    if (__any_sync(0xffffffffu, bad) && (threadIdx.x & 31) == 0) *found_inf = 1.0f;
}

// found_inf of the bucket with the odd-frame twin of the table gradient (ngp_grid_scatter_samples_split) folded in on the
// way: g[t_lo2 .. t_hi2) += odd, odd = 0 (float2 units; the twin is 8-byte aligned) - one pass over the bucket instead of a
// fold launch followed by a check launch on the critical path of the step
__global__ void __launch_bounds__(256) check_finite_fold_kernel(float2* __restrict__ g2, uint64_t n2, uint64_t t_lo2, uint64_t t_hi2,
                                                                float2* __restrict__ odd2, float* __restrict__ found_inf) {
    bool bad = false;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n2; i += (uint64_t)gridDim.x * blockDim.x) {
        float2 v = g2[i];
        if (i >= t_lo2 && i < t_hi2) {
            const float2 o = odd2[i - t_lo2];
            if (o.x != 0.f || o.y != 0.f) {
                v.x += o.x; v.y += o.y;
                g2[i] = v;
                odd2[i - t_lo2] = make_float2(0.f, 0.f);
            }
        }
        bad = bad || (((v.x - v.x) + (v.y - v.y)) != 0.f);
    }
    if (__any_sync(0xffffffffu, bad) && (threadIdx.x & 31) == 0) *found_inf = 1.0f;
}

// ---- one GPU -------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) adam_step_kernel(const Args a) {
    if (a.deferred && *(volatile float*)(a.state + 6) == 0.f) {
        // deferred mode, nothing pending yet: every block reads the flag before it signs off, the last one raises it
        if (last_block(a.sync) && threadIdx.x == 0) { a.state[3] = 0.f; a.state[6] = 1.f; a.sync[0] = 0u; }
        return;
    }
    const float scale = a.state[0];
    const float step0 = a.state[2];
    const bool skip = a.state[3] != 0.f;
    __shared__ float s_coef[3];
    if (threadIdx.x == 0) step_coefficients(a, step0, s_coef);
    __syncthreads();
    const Update u(a, s_coef, scale);

    const uint64_t n4 = a.n / 4;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4 + (a.n & 3 ? 1 : 0);
         i += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t e0 = i * 4;
        const uint32_t cnt = (uint32_t)((a.n - e0) < 4 ? (a.n - e0) : 4);
        float g[4], p[4], m[4], v[4];
        if (cnt == 4) {
            const float4 g4 = *reinterpret_cast<const float4*>(a.g + e0);
            g[0] = g4.x; g[1] = g4.y; g[2] = g4.z; g[3] = g4.w;
        } else {
            for (uint32_t j = 0; j < 4; ++j) g[j] = j < cnt ? a.g[e0 + j] : 0.f;
        }
        if (a.zero_grads) {
            if (cnt == 4) *reinterpret_cast<float4*>(a.g + e0) = make_float4(0.f, 0.f, 0.f, 0.f);
            else for (uint32_t j = 0; j < cnt; ++j) a.g[e0 + j] = 0.f;
        }
        if (skip) continue;
        if (cnt == 4) {
            const float4 p4 = *reinterpret_cast<const float4*>(a.p + e0);
            const float4 m4 = *reinterpret_cast<const float4*>(a.m + e0);
            const float4 v4 = *reinterpret_cast<const float4*>(a.v + e0);
            p[0] = p4.x; p[1] = p4.y; p[2] = p4.z; p[3] = p4.w;
            m[0] = m4.x; m[1] = m4.y; m[2] = m4.z; m[3] = m4.w;
            v[0] = v4.x; v[1] = v4.y; v[2] = v4.z; v[3] = v4.w;
        } else {
            for (uint32_t j = 0; j < 4; ++j) {
                p[j] = j < cnt ? a.p[e0 + j] : 0.f; m[j] = j < cnt ? a.m[e0 + j] : 0.f; v[j] = j < cnt ? a.v[e0 + j] : 0.f;
            }
        }
        adam4(a, u, e0, g, p, m, v);
        if (cnt == 4) {
            *reinterpret_cast<float4*>(a.p + e0) = make_float4(p[0], p[1], p[2], p[3]);
            *reinterpret_cast<float4*>(a.m + e0) = make_float4(m[0], m[1], m[2], m[3]);
            *reinterpret_cast<float4*>(a.v + e0) = make_float4(v[0], v[1], v[2], v[3]);
            if (a.h) *reinterpret_cast<uint2*>(a.h + e0) = pack_half4(p);
        } else {
            for (uint32_t j = 0; j < cnt; ++j) {
                a.p[e0 + j] = p[j]; a.m[e0 + j] = m[j]; a.v[e0 + j] = v[j];
                if (a.h) a.h[e0 + j] = __float2half_rn(p[j]);
            }
        }
    }
    if (last_block(a.sync) && threadIdx.x == 0) {
        scaler_update(a, scale, step0, skip);
        a.sync[0] = 0u;
    }
}

// ---- world > 1 over peer memory --------------------------------------------------------------------------------------
NGP_DEVINL void st_release_sys(uint32_t* p, uint32_t v) { asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory"); }
NGP_DEVINL uint32_t ld_acquire_sys(const uint32_t* p) {
    uint32_t v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
NGP_DEVINL float4 ld_relaxed_sys_f4(const float* p) {
    float4 v;
    asm volatile("ld.relaxed.sys.global.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p) : "memory");
    return v;
}
NGP_DEVINL float4 multimem_ld_reduce_add_f4(const float* mc) {
    float4 v;
    asm volatile("multimem.ld_reduce.relaxed.sys.global.add.v4.f32 {%0, %1, %2, %3}, [%4];"
                 : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(mc) : "memory");
    return v;
}
NGP_DEVINL void multimem_st_f4(float* mc, float4 v) {
    asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(mc), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
NGP_DEVINL void multimem_st_b64(void* mc, uint2 v) {  // 8 bytes moved as two f32 lanes (a store: the bit patterns pass through)
    asm volatile("multimem.st.relaxed.sys.global.v2.f32 [%0], {%1, %2};" ::"l"(mc), "f"(__uint_as_float(v.x)), "f"(__uint_as_float(v.y)) : "memory");
}
NGP_DEVINL uint64_t now_ns() {
    uint64_t t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}

NGP_DEVINL uint32_t* flag_slot(uint32_t* pad, uint32_t barrier, uint32_t block, uint32_t src) {
    return pad + ((size_t)barrier * kMaxBlocks + block) * kMaxWorld + src;
}

// Block-level barrier across ranks: block b of every rank meets block b of every other rank.  `payload` (2 bits) is
// OR-ed over the ranks and returned to every thread of the block.  A timed-out wait sets the sticky error flag state[5]
// and reports payload bit 1 (kPayloadError).
constexpr uint32_t kPayloadInf = 1u, kPayloadError = 2u;
// coef (optional, shared float[3]): while the first `world` threads exchange flags, the block's last thread evaluates the
// step coefficients into it (microseconds on one thread, hidden behind the wait for the peers)
NGP_DEVINL uint32_t xrank_barrier(const Args& a, uint32_t barrier, uint32_t block, uint32_t epoch, uint32_t payload,
                                  float* coef = nullptr, float step0 = 0.f) {
    __shared__ uint32_t s_or;
    if (threadIdx.x == 0) s_or = 0u;
    __syncthreads();
    if (coef && threadIdx.x == blockDim.x - 1) step_coefficients(a, step0, coef);
    if (threadIdx.x < a.world) {
        const uint32_t q = threadIdx.x;
        uint32_t got = 0;
        __threadfence_system();
        st_release_sys(flag_slot(a.peer_flags[q], barrier, block, a.rank), epoch * 4 + (payload & 3u));
        const uint32_t* mine = flag_slot(a.peer_flags[a.rank], barrier, block, q);
        const uint64_t t0 = now_ns();
        for (;;) {
            const uint32_t f = ld_acquire_sys(mine);
            if ((int32_t)((f >> 2) - epoch) >= 0) { got = f & 3u; break; }
            if (now_ns() - t0 > a.timeout_ns) { *(volatile float*)(a.state + 5) = 1.f; got = kPayloadError; break; }
        }
        if (got) atomicOr(&s_or, got);
    }
    __syncthreads();
    const uint32_t r = s_or;
    __syncthreads();   // s_or may be re-initialised by the next barrier of this block
    return r;
}

__global__ void __launch_bounds__(512) adam_dp_kernel(const Args a) {
    if (*(volatile float*)(a.state + 5) != 0.f) return;                 // sticky: a peer was lost in an earlier launch
    const bool arm_only = a.deferred && *(volatile float*)(a.state + 6) == 0.f;   // deferred mode, nothing pending yet
    const float scale = a.state[0];
    const float step0 = a.state[2];
    const uint32_t epoch = a.sync[1] + 1;
    bool skip = false, broken = false;
    if (!arm_only) {
        const uint64_t n4 = a.n / 4;
        const uint64_t per = (n4 + a.world - 1) / a.world;
        const uint64_t lo = per * a.rank < n4 ? per * a.rank : n4;
        const uint64_t hi = lo + per < n4 ? lo + per : n4;
        const uint64_t chunk = (per + gridDim.x - 1) / gridDim.x;       // float4s of a slice that one block owns
        const uint64_t b_lo = lo + chunk * blockIdx.x < hi ? lo + chunk * blockIdx.x : hi;
        const uint64_t b_hi = b_lo + chunk < hi ? b_lo + chunk : hi;

        const uint32_t mine = (*(volatile float*)(a.state + 3) != 0.f ? kPayloadInf : 0u);
        __shared__ float s_coef[3];
        const uint32_t any = xrank_barrier(a, 0, blockIdx.x, epoch, mine, s_coef, step0);      // B0 (+ the step coefficients)
        broken = (any & kPayloadError) != 0u;
        skip = (any & kPayloadInf) != 0u;
        if (!broken) {
            if (!skip) {
                const Update u(a, s_coef, scale);
                for (uint64_t i = b_lo + threadIdx.x; i < b_hi; i += blockDim.x) {
                    const uint64_t e0 = i * 4;
                    float4 s;
                    if (a.mc_g) {
                        s = multimem_ld_reduce_add_f4(a.mc_g + e0);   // summed in the NVSwitch: 1/world of the P2P ingress
                    } else {
                        // all `world` loads are issued before the first add: one NVLink round trip per element, not `world`
                        float4 v[kMaxWorld];
#pragma unroll
                        for (uint32_t q = 0; q < kMaxWorld; ++q)
                            if (q < a.world) v[q] = ld_relaxed_sys_f4(a.peer_g[q] + e0);
                        s = v[0];
#pragma unroll
                        for (uint32_t q = 1; q < kMaxWorld; ++q)
                            if (q < a.world) { s.x += v[q].x; s.y += v[q].y; s.z += v[q].z; s.w += v[q].w; }   // fixed rank order
                    }
                    const float4 p4 = *reinterpret_cast<const float4*>(a.p + e0);
                    const float4 m4 = *reinterpret_cast<const float4*>(a.m + e0);
                    const float4 v4 = *reinterpret_cast<const float4*>(a.v + e0);
                    const float g[4] = {s.x, s.y, s.z, s.w};
                    float p[4] = {p4.x, p4.y, p4.z, p4.w}, m[4] = {m4.x, m4.y, m4.z, m4.w}, v[4] = {v4.x, v4.y, v4.z, v4.w};
                    adam4(a, u, e0, g, p, m, v);
                    *reinterpret_cast<float4*>(a.m + e0) = make_float4(m[0], m[1], m[2], m[3]);
                    *reinterpret_cast<float4*>(a.v + e0) = make_float4(v[0], v[1], v[2], v[3]);
                    const float4 pn = make_float4(p[0], p[1], p[2], p[3]);
                    const uint2 raw = pack_half4(p);
                    if (a.mc_p) {
                        multimem_st_f4(a.mc_p + e0, pn);             // one store, replicated by the switch to every rank
                        if (a.h) multimem_st_b64(a.mc_h + e0, raw);
                    } else {
                        for (uint32_t q = 0; q < a.world; ++q) {
                            const uint32_t dst = (a.rank + q) % a.world;   // start with the own replica, spread the link load
                            *reinterpret_cast<float4*>(a.peer_p[dst] + e0) = pn;
                            if (a.h) *reinterpret_cast<uint2*>(a.peer_h[dst] + e0) = raw;
                        }
                    }
                }
            }
            const uint32_t late = xrank_barrier(a, 2, blockIdx.x, epoch, 0);     // B2
            broken = (late & kPayloadError) != 0u;
            if (!broken) {
                // every rank's block b has finished reading sub-slice b of "its" slice of my bucket: clear those
                for (uint32_t q = 0; q < a.world; ++q) {
                    const uint64_t q_lo = per * q < n4 ? per * q : n4;
                    const uint64_t q_hi = q_lo + per < n4 ? q_lo + per : n4;
                    const uint64_t z_lo = q_lo + chunk * blockIdx.x < q_hi ? q_lo + chunk * blockIdx.x : q_hi;
                    const uint64_t z_hi = z_lo + chunk < q_hi ? z_lo + chunk : q_hi;
                    for (uint64_t i = z_lo + threadIdx.x; i < z_hi; i += blockDim.x)
                        *reinterpret_cast<float4*>(a.g + i * 4) = make_float4(0.f, 0.f, 0.f, 0.f);
                }
            }
        }
    }
    // ---- last block: GradScaler.update() + step count + epoch (or: arm the deferred mode) ---------------------------------
    if (last_block(a.sync) && threadIdx.x == 0) {
        a.sync[0] = 0u;
        if (arm_only) { a.state[6] = 1.f; return; }
        if (*(volatile float*)(a.state + 5) != 0.f) return;      // broken exchange: scaler state and epoch stay as they are
        scaler_update(a, scale, step0, skip);
        a.sync[1] = epoch;
    }
}

}  // namespace adam
}  // namespace ngp

using namespace ngp;

// The arguments both update entry points share: pointer and alignment checks, the lr groups padded to
// NGP_ADAM_MAX_SEGMENTS, the hyperparameters.  The data-parallel fields are left zero.
static int fill_args(adam::Args& a, float* params, float* grads, float* exp_avg, float* exp_avg_sq, void* half_shadow, uint64_t n,
                     uint32_t n_segments, const uint64_t* seg_end, const float* seg_lr, float beta1, float beta2, float eps,
                     float grad_div, float lr_decay_ln, float lr_decay_steps, float growth_factor, float backoff_factor,
                     uint32_t growth_interval, float* state, uint32_t* sync) {
    if (!params || !grads || !exp_avg || !exp_avg_sq || !state || !sync || !seg_end || !seg_lr) return NGP_ERR_BAD_ARG;
    if (n_segments == 0 || n_segments > NGP_ADAM_MAX_SEGMENTS || seg_end[n_segments - 1] != n) return NGP_ERR_BAD_ARG;
    const uintptr_t al = reinterpret_cast<uintptr_t>(params) | reinterpret_cast<uintptr_t>(grads) |
                         reinterpret_cast<uintptr_t>(exp_avg) | reinterpret_cast<uintptr_t>(exp_avg_sq);
    if ((al & 15) != 0 || (reinterpret_cast<uintptr_t>(half_shadow) & 7) != 0) return NGP_ERR_BAD_ARG;
    a = adam::Args{};
    a.p = params; a.g = grads; a.m = exp_avg; a.v = exp_avg_sq; a.h = static_cast<__half*>(half_shadow); a.n = n;
    a.n_seg = n_segments;
    for (uint32_t s = 0; s < NGP_ADAM_MAX_SEGMENTS; ++s) {
        a.seg_end[s] = s < n_segments ? seg_end[s] : n;
        a.seg_lr[s] = s < n_segments ? seg_lr[s] : 0.f;
    }
    a.beta1 = beta1; a.beta2 = beta2; a.eps = eps; a.grad_div = grad_div > 0.f ? grad_div : 1.f;
    a.lr_decay_ln = lr_decay_ln; a.lr_decay_steps = lr_decay_steps;
    a.growth = growth_factor; a.backoff = backoff_factor; a.growth_interval = growth_interval;
    a.state = state; a.sync = sync;
    return NGP_OK;
}

extern "C" int ngp_check_finite(const float* grads, uint64_t n, float* found_inf, void* stream) {
    if (!grads || !found_inf) return NGP_ERR_BAD_ARG;
    if (n == 0) return NGP_OK;
    if ((reinterpret_cast<uintptr_t>(grads) & 15) != 0) return NGP_ERR_BAD_ARG;
    const uint64_t want = (n / 4 + 255) / 256 + 1, cap = (uint64_t)num_sms() * 8;
    const int blocks = (int)(want < cap ? want : cap);
    adam::check_finite_kernel<<<blocks, 256, 0, as_stream(stream)>>>(reinterpret_cast<const float4*>(grads), grads, n, found_inf);
    return launch_status();
}

extern "C" int ngp_check_finite_fold(float* grads, uint64_t n, float* grad_table, float* grad_table_odd, uint64_t table_n,
                                     float* found_inf, void* stream) {
    if (!grads || !found_inf || !grad_table || !grad_table_odd) return NGP_ERR_BAD_ARG;
    if ((n & 1) || (table_n & 1) || grad_table < grads || grad_table + table_n > grads + n) return NGP_ERR_BAD_ARG;
    if (((reinterpret_cast<uintptr_t>(grads) | reinterpret_cast<uintptr_t>(grad_table) | reinterpret_cast<uintptr_t>(grad_table_odd)) & 7) != 0)
        return NGP_ERR_BAD_ARG;
    if (n == 0) return NGP_OK;
    const uint64_t n2 = n / 2, t_lo2 = (uint64_t)(grad_table - grads) / 2, t_hi2 = t_lo2 + table_n / 2;
    const uint64_t want = (n2 + 255) / 256, cap = (uint64_t)num_sms() * 8;
    const int blocks = (int)(want < cap ? want : cap);
    adam::check_finite_fold_kernel<<<blocks, 256, 0, as_stream(stream)>>>(reinterpret_cast<float2*>(grads), n2, t_lo2, t_hi2,
                                                                         reinterpret_cast<float2*>(grad_table_odd), found_inf);
    return launch_status();
}

extern "C" int ngp_adam_step(float* params, float* grads, float* exp_avg, float* exp_avg_sq, void* half_shadow, uint64_t n,
                             uint32_t n_segments, const uint64_t* seg_end, const float* seg_lr, float beta1, float beta2,
                             float eps, float grad_div, float lr_decay_ln, float lr_decay_steps, float growth_factor,
                             float backoff_factor, uint32_t growth_interval, int zero_grads, float* state,
                             uint32_t* blocks_done, void* stream) {
    adam::Args a;
    const int rc = fill_args(a, params, grads, exp_avg, exp_avg_sq, half_shadow, n, n_segments, seg_end, seg_lr, beta1, beta2, eps,
                             grad_div, lr_decay_ln, lr_decay_steps, growth_factor, backoff_factor, growth_interval, state, blocks_done);
    if (rc != NGP_OK) return rc;
    if (n == 0) return NGP_OK;
    a.zero_grads = zero_grads & 1; a.deferred = (zero_grads >> 1) & 1;
    const uint64_t want = (n / 4 + 255) / 256 + 1, cap = (uint64_t)num_sms() * 8;
    const int blocks = (int)(want < cap ? want : cap);
    adam::adam_step_kernel<<<blocks, 256, 0, as_stream(stream)>>>(a);
    return launch_status();
}

extern "C" uint64_t ngp_dp_flags_bytes(void) { return (uint64_t)3 * adam::kMaxBlocks * adam::kMaxWorld * sizeof(uint32_t); }

extern "C" int ngp_enable_peer_access(int peer_device) {
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return (int)e;
    if (peer_device == dev) return NGP_OK;
    int can = 0;
    e = cudaDeviceCanAccessPeer(&can, dev, peer_device);
    if (e != cudaSuccess) return (int)e;
    if (!can) return NGP_ERR_UNSUPPORTED;
    e = cudaDeviceEnablePeerAccess(peer_device, 0);
    if (e == cudaErrorPeerAccessAlreadyEnabled) { cudaGetLastError(); return NGP_OK; }
    return e == cudaSuccess ? NGP_OK : (int)e;
}

// 0: spin timeout of the cross-GPU waits in milliseconds (>= 1); 1: blocks of the ngp_adam_step_dp grid (0 = sized from the slice)
extern "C" int ngp_dp_set_option(int option, int value) {
    if (option == 0 && value >= 1) { adam::g_spin_timeout_ns = (uint64_t)value * 1000000ull; return NGP_OK; }
    if (option == 1 && value >= 0 && value <= (int)adam::kMaxBlocks) { adam::g_blocks = value; return NGP_OK; }
    return NGP_ERR_BAD_ARG;
}

// world > 1 only, and the caller must have run ngp_check_finite(grads, n, state + 3) on the same stream first (see
// adam_dp_kernel).
extern "C" int ngp_adam_step_dp(float* params, float* grads, float* exp_avg, float* exp_avg_sq, void* half_shadow, uint64_t n,
                                uint32_t n_segments, const uint64_t* seg_end, const float* seg_lr, float beta1, float beta2,
                                float eps, float grad_div, float lr_decay_ln, float lr_decay_steps, float growth_factor,
                                float backoff_factor, uint32_t growth_interval, int deferred, float* state, uint32_t* sync,
                                uint32_t rank, uint32_t world, const uint64_t* peer_grads, const uint64_t* peer_params,
                                const uint64_t* peer_half, const uint64_t* peer_flags, const uint64_t* multicast, void* stream) {
    adam::Args a;
    const int rc = fill_args(a, params, grads, exp_avg, exp_avg_sq, half_shadow, n, n_segments, seg_end, seg_lr, beta1, beta2, eps,
                             grad_div, lr_decay_ln, lr_decay_steps, growth_factor, backoff_factor, growth_interval, state, sync);
    if (rc != NGP_OK) return rc;
    if (n == 0 || (n & 3) != 0) return NGP_ERR_BAD_ARG;
    if (world < 2 || world > adam::kMaxWorld || rank >= world) return NGP_ERR_BAD_ARG;
    if (!peer_grads || !peer_params || !peer_flags || (half_shadow && !peer_half)) return NGP_ERR_BAD_ARG;
    a.deferred = deferred; a.rank = rank; a.world = world;
    for (uint32_t q = 0; q < world; ++q) {
        a.peer_g[q] = reinterpret_cast<float*>(peer_grads[q]);
        a.peer_p[q] = reinterpret_cast<float*>(peer_params[q]);
        a.peer_h[q] = peer_half ? reinterpret_cast<__half*>(peer_half[q]) : nullptr;
        a.peer_flags[q] = reinterpret_cast<uint32_t*>(peer_flags[q]);
        if (!a.peer_g[q] || !a.peer_p[q] || !a.peer_flags[q]) return NGP_ERR_BAD_ARG;
    }
    const bool mc = multicast && multicast[0] && multicast[1] && (!half_shadow || multicast[2]);
    a.mc_g = mc ? reinterpret_cast<float*>(multicast[0]) : nullptr;
    a.mc_p = mc ? reinterpret_cast<float*>(multicast[1]) : nullptr;
    a.mc_h = mc && half_shadow ? reinterpret_cast<__half*>(multicast[2]) : nullptr;
    a.timeout_ns = adam::g_spin_timeout_ns;
    // a rank's slice is n / (4 world) float4s; ~4 per thread keeps `world` x 4 peer loads in flight per thread
    const uint64_t per = (n / 4 + world - 1) / world;
    int blocks = adam::g_blocks > 0 ? adam::g_blocks : (int)((per + 512 * 4 - 1) / (512 * 4));
    if (blocks < 8) blocks = 8;
    if (blocks > num_sms()) blocks = num_sms();
    if (blocks > (int)adam::kMaxBlocks) blocks = (int)adam::kMaxBlocks;
    adam::adam_dp_kernel<<<blocks, 512, 0, as_stream(stream)>>>(a);
    return launch_status();
}

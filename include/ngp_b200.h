/*
 * ngp_b200.h - C ABI of libngp_b200.so: the B200 (sm_100a) NeRF rendering hot path of
 * stable-dreamfusion (hash-grid encode, occupancy-grid ray marching, volume compositing,
 * occupancy-grid update, frequency encode, fused 64-wide field MLP).
 *
 * This is the drop-in boundary.  Every entry point replaces one native function that the
 * reference binds through pybind11 (file:line given per function, relative to the reference
 * tree) and keeps its argument order and meaning.  Differences from the pybind surface:
 *   - at::Tensor arguments become raw DEVICE pointers (the caller owns, allocates and - where
 *     noted - zero-fills every buffer, exactly as the reference's Python wrappers do);
 *   - a dtype code replaces AT_DISPATCH (NGP_F32 / NGP_F16);
 *   - a trailing `stream` (a cudaStream_t passed as void*) replaces the reference's implicit
 *     legacy default stream; kernels are launched on the CURRENT device of the calling thread;
 *   - every function returns an int: NGP_OK (0), a negative NGP_ERR_* argument error, or a
 *     positive cudaError_t from the launch.  Nothing is thrown, allocated or synchronised
 *     unless stated.
 * No torch / pybind / C++ types appear in any signature.
 */
#ifndef NGP_B200_H_
#define NGP_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NGP_OK 0
#define NGP_ERR_BAD_ARG (-1)     /* null pointer / inconsistent sizes */
#define NGP_ERR_UNSUPPORTED (-2) /* D, C or dtype outside what the reference instantiates */
#define NGP_ERR_WORKSPACE (-3)   /* workspace too small */

#define NGP_F32 0
#define NGP_F16 1

/* grid-encode output / grad layouts */
#define NGP_LAYOUT_LBC 0 /* [L, B, C] - the reference kernel's native layout (gridencoder.cu:361) */
#define NGP_LAYOUT_BLC 1 /* [B, L*C] - what grid.py:52 permutes to; written directly (fused permute) */

#define NGP_GRID_HASH 0  /* gridencoder/grid.py:14-17 */
#define NGP_GRID_TILED 1

int ngp_version(void);
/* Human-readable text for a return code (static storage). */
const char* ngp_error_string(int code);
/* Name of the device the library is running on + SM count (host call, no launch). */
int ngp_device_info(char* name, int name_len, int* sm_count, int* cc_major, int* cc_minor);

/* ------------------------------------------------------------------------------------------
 * gridencoder  (reference: gridencoder/src/gridencoder.h:12-13, gridencoder.cu:424-479)
 * ------------------------------------------------------------------------------------------ */

/* Replaces grid_encode_forward (gridencoder.cu:424).  inputs f32[B,D] in [0,1]; embeddings
 * dtype[sO,C]; offsets i32[L+1]; outputs dtype, layout per out_layout; dy_dx dtype[B,L,D,C] or
 * NULL; S = log2(per_level_scale); H = base resolution.  D in 1..5, C in {1,2,4,8}
 * (gridencoder.cu:354,372); dtype NGP_F32 or NGP_F16 (double is not built: NGP_ERR_UNSUPPORTED). */
int ngp_grid_encode_forward(const float* inputs, const void* embeddings, const int* offsets, void* outputs,
                            uint32_t B, uint32_t D, uint32_t C, uint32_t L, float S, uint32_t H, void* dy_dx,
                            uint32_t gridtype, int align_corners, int dtype, int out_layout, void* stream);

/* Replaces grid_encode_backward (gridencoder.cu:449).  grad dtype in grad_layout; grad_embeddings
 * [sO,C] MUST be zero-filled by the caller (grid.py:72); its element type is grad_emb_dtype:
 * NGP_F16 reproduces the reference's half2 atomics, NGP_F32 accumulates in fp32 (what the Python
 * host uses: more accurate, same API-visible result after autograd's cast).  dy_dx/grad_inputs
 * (dtype[B,L,D,C] / dtype[B,D]) may be NULL. */
int ngp_grid_encode_backward(const void* grad, const float* inputs, const void* embeddings, const int* offsets,
                             void* grad_embeddings, uint32_t B, uint32_t D, uint32_t C, uint32_t L, float S,
                             uint32_t H, const void* dy_dx, void* grad_inputs, uint32_t gridtype,
                             int align_corners, int dtype, int grad_layout, int grad_emb_dtype, void* stream);

/* Tuning / test switches.  option 0: value != 0 disables the warp-aggregated scatter of the backward (every
 * sample then issues its own atomics, like the reference).  option 1: value != 0 makes ngp_grid_scatter_samples run
 * its counting build (measurement only): every red instruction a lane issues AFTER warp aggregation is counted.
 * option 2: longest run of neighbouring lanes ngp_grid_scatter_samples[_split] sums before issuing the reds (4, 8, 16 or
 * 32 = a whole warp): shorter runs mean fewer shuffle steps and a few more reds at the coarse levels. */
int ngp_grid_set_option(int option, int value);
/* Reads (and optionally resets) that counter into *lane_ops (HOST pointer); synchronises the device. */
int ngp_grid_red_count(uint64_t* lane_ops, int reset);

/* Device-computed per-level (scale, resolution) exactly as gridencoder.cu:125-126 evaluates them
 * (exp2f on the device).  scales f32[L], resolutions u32[L] are DEVICE buffers. */
int ngp_grid_level_params(uint32_t L, float S, uint32_t H, float* scales, uint32_t* resolutions, void* stream);

/* ------------------------------------------------------------------------------------------
 * raymarching  (reference: raymarching/src/raymarching.h:7-17)
 * All floating tensors are f32 (the wrappers force-cast: raymarching.py custom_fwd(cast_inputs=float32)).
 * ------------------------------------------------------------------------------------------ */

/* raymarching.cu:148  rays_o/rays_d f32[N,3], aabb f32[6] -> nears/fars f32[N] (miss: FLT_MAX both). */
int ngp_near_far_from_aabb(const float* rays_o, const float* rays_d, const float* aabb, uint32_t N,
                           float min_near, float* nears, float* fars, void* stream);
/* raymarching.cu:201  coords f32[N,2] */
int ngp_sph_from_ray(const float* rays_o, const float* rays_d, float radius, uint32_t N, float* coords,
                     void* stream);
/* raymarching.cu:229  coords i32[N,3] -> indices i32[N] */
int ngp_morton3D(const int* coords, uint32_t N, int* indices, void* stream);
/* raymarching.cu:257  indices i32[N] -> coords i32[N,3] */
int ngp_morton3D_invert(const int* indices, uint32_t N, int* coords, void* stream);
/* raymarching.cu:292  grid f32[N*8] -> bitfield u8[N]; bit i of byte n = grid[8n+i] > thresh */
int ngp_packbits(const float* grid, uint32_t N, float density_thresh, uint8_t* bitfield, void* stream);

/* raymarching.cu:482.  Outputs xyzs f32[M,3], dirs f32[M,3], deltas f32[M,2] (rows not written stay
 * untouched: the caller zero-fills as raymarching.py:205-207 does, or relies on `rays`), rays
 * i32[N,3] = (ray id, offset, count), counter i32[2] += (sum count, N).  Unlike the reference's
 * nondeterministic atomic slot allocation (raymarching.cu:405-406) rows are emitted in ray order:
 * rays[n] describes ray n and offsets are an exclusive prefix sum - one of the orders the
 * reference itself can produce.  A ray whose offset+count > M is recorded in `rays` but writes no
 * samples (raymarching.cu:416).  workspace: device scratch of >=
 * ngp_march_rays_train_workspace(N, max_steps) bytes (per-ray counts + one max_steps-row slab per ray).  The first 256
 * bytes of a NEW workspace must be zero-filled once by the caller (block-election word); every call leaves them zero. */
int ngp_march_rays_train(const float* rays_o, const float* rays_d, const uint8_t* grid, float bound,
                         float dt_gamma, uint32_t max_steps, uint32_t N, uint32_t C, uint32_t H, uint32_t M,
                         const float* nears, const float* fars, float* xyzs, float* dirs, float* deltas,
                         int* rays, int* counter, const float* noises, void* workspace,
                         uint64_t workspace_bytes, void* stream);
/* (dirs may be NULL: the albedo-shaded training path never reads the per-sample directions.) */
uint64_t ngp_march_rays_train_workspace(uint32_t N, uint32_t max_steps);
/* The same marcher as ONE launch without scratch: each ray is walked once (its samples' lattice parameters parked in shared
 * memory), claims its rows with one atomicAdd on counter[0] - the reference's slot allocation, raymarching.cu:405-406 - and
 * writes them in place.  Same samples per ray, bit for bit; rays[n] = (n, offset, count) still describes ray n, but offsets
 * follow completion order instead of ray order (as in the reference).  max_steps <= 2048 (else NGP_ERR_UNSUPPORTED: use
 * ngp_march_rays_train).  The hand-scheduled train step uses this one. */
int ngp_march_rays_train_packed(const float* rays_o, const float* rays_d, const uint8_t* grid, float bound,
                                float dt_gamma, uint32_t max_steps, uint32_t N, uint32_t C, uint32_t H, uint32_t M,
                                const float* nears, const float* fars, float* xyzs, float* dirs, float* deltas,
                                int* rays, int* counter, const float* noises, void* stream);
/* option 0: value != 0 selects the one-thread-per-ray count / write kernels (the reference's decomposition) instead of
 * the default walks; option 1: warp-per-ray walk for one-sample inference calls; option 2: ngp_march_rays_train launches of
 * at least `value` rays with dt_gamma == 0 use the thread-per-ray walk with closed-form lattice jumps, smaller ones the
 * warp-per-ray walk (0 = never, the default: it is not faster).  Results are bit-identical in every mode. */
int ngp_march_set_option(int option, int value);

/* raymarching.cu:580 */
int ngp_composite_rays_train_forward(const float* sigmas, const float* rgbs, const float* deltas,
                                     const int* rays, uint32_t M, uint32_t N, float T_thresh,
                                     float* weights_sum, float* depth, float* image, void* stream);
/* raymarching.cu:685.  grad_sigmas f32[M], grad_rgbs f32[M,3] zero-filled by the caller
 * (raymarching.py:283-284). */
int ngp_composite_rays_train_backward(const float* grad_weights_sum, const float* grad_image,
                                      const float* sigmas, const float* rgbs, const float* deltas,
                                      const int* rays, const float* weights_sum, const float* image,
                                      uint32_t M, uint32_t N, float T_thresh, float* grad_sigmas,
                                      float* grad_rgbs, void* stream);

/* raymarching.cu:808 (inference).  Outputs are slot-major [n_alive*n_step (+pad), ...], zero-filled
 * by the caller (raymarching.py:334-336). */
int ngp_march_rays(uint32_t n_alive, uint32_t n_step, const int* rays_alive, const float* rays_t,
                   const float* rays_o, const float* rays_d, float bound, float dt_gamma, uint32_t max_steps,
                   uint32_t C, uint32_t H, const uint8_t* grid, const float* nears, const float* fars,
                   float* xyzs, float* dirs, float* deltas, const float* noises, void* stream);
/* raymarching.cu:908 (inference, in place). */
int ngp_composite_rays(uint32_t n_alive, uint32_t n_step, float T_thresh, int* rays_alive, float* rays_t,
                       const float* sigmas, const float* rgbs, const float* deltas, float* weights_sum,
                       float* depth, float* image, void* stream);

/* Device-side replacement for `rays_alive = rays_alive[rays_alive >= 0]` (nerf/renderer.py:529):
 * stable compaction of the first n_alive entries of rays_alive into out; *n_out (device i32)
 * receives the new count.  workspace >= ngp_compact_alive_workspace(n_alive) bytes. */
int ngp_compact_alive(const int* rays_alive, uint32_t n_alive, int* out, int* n_out, void* workspace,
                      uint64_t workspace_bytes, void* stream);
uint64_t ngp_compact_alive_workspace(uint32_t n_alive);

/* ------------------------------------------------------------------------------------------
 * freqencoder  (reference: freqencoder/src/freqencoder.h:7,10; freqencoder.cu:97,114)
 * ------------------------------------------------------------------------------------------ */
int ngp_freq_encode_forward(const float* inputs, uint32_t B, uint32_t D, uint32_t deg, uint32_t C,
                            float* outputs, void* stream);
int ngp_freq_encode_backward(const float* grad, const float* outputs, uint32_t B, uint32_t D, uint32_t deg,
                             uint32_t C, float* grad_inputs, void* stream);

/* ------------------------------------------------------------------------------------------
 * Occupancy-grid update  (reference: NeRFRenderer.update_extra_state, nerf/renderer.py:562-613)
 * ------------------------------------------------------------------------------------------ */

/* Cell centres + jitter for one cascade (renderer.py:581-593): for morton-ordered cell m in
 * [0,H^3): coords = morton3D_invert(m); xyz = (2*coords/(H-1) - 1)*cell_scale + (2*noise-1)*half_cell
 * where the host passes cell_scale = fp32(bound_c - bound_c/H) and half_cell = fp32(bound_c/H).
 * noise f32[H^3,3] is indexed by the LINEAR cell id x*H*H+y*H+z (the order torch.rand_like is
 * consumed in); out xyzs f32[H^3,3] is in MORTON order so the density query result lands directly
 * in density_grid order (renderer.py:597). */
int ngp_occupancy_cell_points(uint32_t H, float cell_scale, float half_cell, const float* noise, float* xyzs,
                              void* stream);
/* One rank's share of a data-parallel refresh: the query points of Morton cells [first, first + count) only, jitter from
 * noise f32[count,3] indexed by (cell - first); xyzs f32[count,3]. */
int ngp_occupancy_cell_points_range(uint32_t H, float cell_scale, float half_cell, const float* noise, uint32_t first,
                                    uint32_t count, float* xyzs, void* stream);

/* EMA-max + mean + bitfield (renderer.py:600-607).  grid f32[n_cells] updated in place where
 * grid >= 0: grid = max(grid*decay, tmp).  mean_out f32[1] = mean over valid cells.  bitfield
 * u8[n_cells/8] = grid > min(mean, density_thresh).  workspace >= 16 bytes, zeroed by the call. */
int ngp_update_density_grid(float* grid, const float* tmp_grid, uint32_t n_cells, float decay,
                            float density_thresh, float* mean_out, uint8_t* bitfield, void* workspace,
                            uint64_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * Fused field network  (reference: NeRFNetwork.common_forward, nerf/network_grid.py:76-87, under fp16
 * autocast: GridEncoder -> Linear(32,64)+ReLU -> Linear(64,64)+ReLU -> Linear(64,4) -> trunc_exp / sigmoid;
 * activation.py:4-17).  The three GEMMs run on tcgen05 tensor cores inside one kernel per direction.
 * Only the reference's own shape is built: L=16 levels x C=2 features, D=3, hidden 64, 4 outputs
 * (anything else: NGP_ERR_UNSUPPORTED - the host then uses the unfused ops).
 * ------------------------------------------------------------------------------------------ */

/* xyzs f32[M,3] in [-bound,bound]; table f16[rows,2]; w1..w3 and b1..b3 are the fp16 casts of the nn.Linear weights
 * ([out,in] row-major) and biases; count_ptr (optional, device i32) limits the rows actually processed.
 * Outputs: sigma f32[M]; rgb f32[M,3] (the fp16-rounded sigmoid, widened).  enc_save / h1_save / h2_save are optional
 * (NULL for inference) and feed ngp_field_backward: OPAQUE buffers of ceil(M/128)*128 rows x 32 / 64 / 64 fp16
 * (16-byte aligned), written one whole 128-sample tile at a time in the kernels' shared-memory tile layout (one
 * bulk copy per tile) - not row-major. */
int ngp_field_forward(const float* xyzs, uint32_t M, const int* count_ptr, const void* table, const int* offsets,
                      uint32_t L, uint32_t C, float S, uint32_t H, uint32_t gridtype, int align_corners, float bound,
                      const void* w1, const void* b1, const void* w2, const void* b2, const void* w3, const void* b3,
                      uint32_t hidden, uint32_t out_dim, float* sigma, float* rgb, void* enc_save, void* h1_save,
                      void* h2_save, void* stream);
/* The same forward reading the table through a QUAD table: quads u32[rows,4] (16-byte aligned), row r of a linear / tiled
 * level = the fp16x2 features of rows r, r+1, r+stride_y, r+stride_y+1 of that level (wrapped as gridencoder.cu:54-72 wraps
 * them) = the four corners of one z slice of the cell whose base corner is row r, so a level costs one or two 16-byte
 * gathers per sample instead of four to eight 4-byte ones.  Same values in the same order: bit-equal outputs.  Built from
 * the fp16 table by ngp_grid_quad_table (rows = offsets[L]; 16 bytes per row) - rebuild after every parameter update. */
int ngp_grid_quad_table(const void* table, const int* offsets, uint32_t L, uint32_t total_rows, float S, uint32_t H,
                        uint32_t gridtype, int align_corners, void* quads, void* stream);
int ngp_field_forward_quads(const float* xyzs, uint32_t M, const int* count_ptr, const void* table, const void* quads,
                            const int* offsets, uint32_t L, uint32_t C, float S, uint32_t H, uint32_t gridtype,
                            int align_corners, float bound, const void* w1, const void* b1, const void* w2, const void* b2,
                            const void* w3, const void* b3, uint32_t hidden, uint32_t out_dim, float* sigma, float* rgb,
                            void* enc_save, void* h1_save, void* h2_save, void* stream);

/* Backward of the MLP part: from d_sigma f32[M], d_rgb f32[M,3] (+ the forward outputs and saves) to
 * d_enc f16[M,32] (gradient wrt the grid encoding - feed it to ngp_grid_encode_backward) and the fp32 weight /
 * bias gradients gw1[64,32] gb1[64] gw2[64,64] gb2[64] gw3[4,64] gb3[4], which are ACCUMULATED (+=). */
int ngp_field_backward(uint32_t M, const int* count_ptr, const void* w1, const void* w2, const void* w3,
                       uint32_t hidden, uint32_t out_dim, const float* d_sigma, const float* d_rgb, const float* sigma,
                       const float* rgb, const void* enc_save, const void* h1_save, const void* h2_save, void* d_enc,
                       float* gw1, float* gb1, float* gw2, float* gb2, float* gw3, float* gb3, void* stream);

/* Tuning switch for the fused field kernels (profiling support): option 0 = forward CTAs per SM (1..7),
 * option 1 = forward shared-memory carveout percent (-1: driver default). */
int ngp_field_set_option(int option, int value);

/* Table-gradient scatter for the sync-free training path: like ngp_grid_encode_backward for D=3, C=2, fp16
 * [M, L*C] gradients and an fp32 table, but (a) only the first *count_ptr rows (device i32, may be NULL) of the
 * M_cap-row buffers are processed and (b) positions are world coordinates in [-bound, bound], mapped to [0,1]
 * inside the kernel as GridEncoder.forward does (grid.py:142).  grad_table is accumulated into (+=). */
int ngp_grid_scatter_samples(const void* d_enc, const float* xyzs, float bound, const int* count_ptr, uint32_t M_cap,
                             const int* offsets, uint32_t L, uint32_t C, float S, uint32_t H, uint32_t gridtype,
                             int align_corners, float* grad_table, void* stream);

/* The same scatter with the table gradient split over two fp32 buffers (no reference counterpart; it replaces the
 * per-corner atomicAdd of gridencoder.cu:298-310 like the call above).  The SM issues vector reds at a fixed rate per
 * lane whatever their width, so the two x-neighbours of a corner pair go out as ONE 16-byte red - which needs the pair
 * 16-byte aligned.  Pairs starting on an even table row are aligned in grad_table; pairs starting on an odd row are
 * aligned in grad_table_odd, a buffer indexed exactly like grad_table whose address is 8 bytes off a 16-byte boundary.
 * gradient = grad_table + grad_table_odd: fold with ngp_grid_fold_odd before anything reads it. */
int ngp_grid_scatter_samples_split(const void* d_enc, const float* xyzs, float bound, const int* count_ptr, uint32_t M_cap,
                                   const int* offsets, uint32_t L, uint32_t C, float S, uint32_t H, uint32_t gridtype,
                                   int align_corners, float* grad_table, float* grad_table_odd, void* stream);

/* grad_table[i] += grad_table_odd[i]; grad_table_odd[i] = 0 for i < n (n even; both buffers 8-byte aligned). */
int ngp_grid_fold_odd(float* grad_table, float* grad_table_odd, uint64_t n, void* stream);

/* ------------------------------------------------------------------------------------------
 * The steps either side of the render inside one train step (SURVEY.md 8f rows 1-2).  The reference runs these as
 * chains of eager PyTorch kernels; each entry point below is one launch.
 * ------------------------------------------------------------------------------------------ */
#define NGP_ADAM_MAX_SEGMENTS 8

/* GradScaler's inf/nan check (torch.amp.GradScaler.unscale_, called from nerf/utils.py:709 scaler.step):
 * sets *found_inf = 1.0f (device f32, never cleared here) if any of grads f32[n] is not finite.  grads 16-byte aligned. */
int ngp_check_finite(const float* grads, uint64_t n, float* found_inf, void* stream);
/* The same verdict with the odd-frame twin of the table gradient (ngp_grid_scatter_samples_split) folded into the bucket on
 * the way: grad_table (a sub-range of grads, table_n floats) += grad_table_odd, grad_table_odd = 0 - what ngp_grid_fold_odd
 * followed by ngp_check_finite do, in one pass. */
int ngp_check_finite_fold(float* grads, uint64_t n, float* grad_table, float* grad_table_odd, uint64_t table_n,
                          float* found_inf, void* stream);

/* scaler.step(optimizer) + scaler.update() for Adam over ONE flat parameter buffer (main.py:128 Adam betas
 * (0.9,0.99) eps 1e-15; network_grid.py:170-181 lr groups; main.py:131 LambdaLR 0.1^(iter/iters);
 * nerf/utils.py:709-710).  All pointers are device pointers except seg_end / seg_lr (HOST arrays of n_segments
 * entries: exclusive end index of each learning-rate group in the flat buffer, and its base lr).
 *   state f32[5]: [0] loss scale, [1] growth tracker, [2] optimizer steps taken, [3] found_inf (from
 *   ngp_check_finite), [4] skipped steps.  If state[3] != 0 the parameters are left untouched and the scale is
 *   multiplied by backoff_factor; otherwise grads are divided by state[0] * grad_div, Adam is applied with
 *   lr * exp(lr_decay_ln * min(steps, lr_decay_steps)), and the scale grows by growth_factor every
 *   growth_interval clean steps.  half_shadow (optional f16[n]) receives the fp16 cast of the new parameters (what
 *   autocast re-derives every forward, gridencoder/grid.py:38-39); zero_grads != 0 zero-fills grads on the way out
 *   (optimizer.zero_grad, nerf/utils.py:700).  blocks_done: zero-initialised device u32 scratch (left zero).
 *   zero_grads is a bit set: bit 0 = zero-fill the gradients; bit 1 = deferred (state must then have 7 entries): a launch
 *   that finds state[6] == 0 applies nothing and only sets state[6] = 1 - the update of step k launched at the start of
 *   step k + 1, where the very first launch has nothing to apply (TrainStep(pipelined=True)). */
int ngp_adam_step(float* params, float* grads, float* exp_avg, float* exp_avg_sq, void* half_shadow, uint64_t n,
                  uint32_t n_segments, const uint64_t* seg_end, const float* seg_lr, float beta1, float beta2, float eps,
                  float grad_div, float lr_decay_ln, float lr_decay_steps, float growth_factor, float backoff_factor,
                  uint32_t growth_interval, int zero_grads, float* state, uint32_t* blocks_done, void* stream);

/* Background colour network (nerf/network_grid.py:54-62,158-167 under fp16 autocast): FreqEncoder(degree 6) ->
 * Linear(39,64)+ReLU -> Linear(64,3) -> sigmoid, one launch.  dirs f32[N,3]; w1 f16[64,39], b1 f16[64], w2 f16[3,64],
 * b2 f16[3] (the fp16 casts of bg_net.net.{0,1}); out_rgb f16[N,3].  Only degree 6 / hidden 64 is built. */
int ngp_bg_forward(const float* dirs, uint32_t N, const void* w1, const void* b1, const void* w2, const void* b2,
                   uint32_t degree, uint32_t hidden, void* out_rgb, void* stream);
/* Its backward wrt the parameters (the forward is recomputed per ray): grad_rgb f32[N,3]; gw1 f32[64,39], gb1 f32[64],
 * gw2 f32[3,64], gb2 f32[3] are ACCUMULATED (+=). */
int ngp_bg_backward(const float* dirs, const float* grad_rgb, uint32_t N, const void* w1, const void* b1, const void* w2,
                    const void* b2, uint32_t degree, uint32_t hidden, float* gw1, float* gb1, float* gw2, float* gb2,
                    void* stream);

/* ngp_adam_step for world > 1 ranks with the data-parallel gradient all-reduce fused in over NVLink peer memory
 * (csrc/adam.cu): the all_reduce DistributedDataParallel would issue for the reference's dormant wrap
 * (nerf/utils.py:200-202) and the update in one plain launch of independent blocks (block b owns sub-slice b of its
 * rank's slice: flag exchange - P2P / multimem reduce - Adam - parameter broadcast - flag exchange - clear).  The
 * GradScaler verdict comes from each rank's OWN bucket: the caller runs ngp_check_finite(grads, n, state + 3) on the same
 * stream first (a sum of <= 8 finite fp32 gradients is finite), and it travels with the first flag exchange.  Arguments as
 * ngp_adam_step, and:
 *   state f32[8]: as ngp_adam_step, plus [5] = 1 if a cross-GPU wait timed out (sticky: from then on the step is a no-op
 *   on every rank that saw the flag - nothing is reduced, updated, broadcast or cleared).  sync u32[2], zero-initialised:
 *   [0] block election, [1] barrier epoch.  n must be a multiple of 4, 2 <= world <= NGP_DP_MAX_WORLD.
 *   peer_* are HOST arrays of `world` device addresses (this rank's own buffers included, in rank order) of every rank's
 *   gradient bucket, parameter buffer, fp16 shadow (may be NULL without half_shadow) and flag pad (ngp_dp_flags_bytes()
 *   bytes, zeroed once), all mapped into this process (symmetric memory / CUDA IPC).  Each rank reduces and updates slice
 *   `rank` and writes the new parameters to every replica; exp_avg / exp_avg_sq are maintained for that slice only.  The
 *   gradient bucket is always zero-filled on the way out.  All ranks must launch the same sequence of calls.
 *   multicast: NULL, or a HOST array of 3 NVLS multicast addresses of the gradient bucket, the parameters and the shadow
 *   (the same symmetric allocation mapped through the NVSwitch): the reduce-scatter then is one multimem.ld_reduce per
 *   element (summed inside the switch) and the parameter broadcast one multimem.st instead of `world` P2P stores.
 *   deferred != 0: for a trainer that applies step k's update at the START of step k+1 (overlapped with that step's ray
 *   marching): a launch that finds state[6] == 0 applies nothing and sets state[6] = 1 ("gradients will be pending next
 *   time"); the caller clears state[6] after flushing the last pending update. */
#define NGP_DP_MAX_WORLD 8
#define NGP_DP_MAX_BLOCKS 256
int ngp_adam_step_dp(float* params, float* grads, float* exp_avg, float* exp_avg_sq, void* half_shadow, uint64_t n,
                     uint32_t n_segments, const uint64_t* seg_end, const float* seg_lr, float beta1, float beta2, float eps,
                     float grad_div, float lr_decay_ln, float lr_decay_steps, float growth_factor, float backoff_factor,
                     uint32_t growth_interval, int deferred, float* state, uint32_t* sync, uint32_t rank, uint32_t world,
                     const uint64_t* peer_grads, const uint64_t* peer_params, const uint64_t* peer_half, const uint64_t* peer_flags,
                     const uint64_t* multicast, void* stream);
uint64_t ngp_dp_flags_bytes(void);
/* option 0: timeout of the cross-GPU waits in milliseconds (default 20000); option 1: blocks of the ngp_adam_step_dp grid
 * (0 = sized from the slice, the default). */
int ngp_dp_set_option(int option, int value);
/* cudaDeviceEnablePeerAccess(peer_device) from the current device (idempotent). */
int ngp_enable_peer_access(int peer_device);

/* First and middle kernels of the hand-scheduled train step (ngp_b200/trainer.py).
 * ngp_train_prologue: near_far_from_aabb (raymarching.cu:92-156) for N rays + the step's device-side bookkeeping: zero-fill
 * of counters i32[n_counters] and loss f32[1]; opens the step's row of run_cuda's 16-step window (nerf/renderer.py:466-467):
 * *cur_row = *local_step % 16, step_counter[*cur_row] = (0, 0), ++*local_step.  Each pointer group may be NULL.
 * noises (optional, f32[N]) + rng (u64[3]: seed, step counter, scratch - zero the scratch once): the per-ray march jitter the
 * reference draws with torch.rand(N) (raymarching.py:213-216), from a counter-based generator keyed by (seed, counter, ray);
 * the launch advances the counter by one, so consecutive steps draw fresh, reproducible noise without a generator launch.
 * ngp_train_ray_loss: per ray, in one launch: composite_rays_train forward (raymarching.cu:501-588), the background blend
 * (nerf/renderer.py:541-545), the gradients of the two losses of Trainer.train_step at the ray - grad_pred (the guidance
 * gradient wrt the blended image, [B,3,pixels_per_view] NCHW as nerf/sd.py:115 passes it, or [N,3] if pixels_per_view is
 * 0) and lambda * mean opacity entropy times *scale (nerf/utils.py:389-394,708) - and composite_rays_train backward
 * (raymarching.cu:602-693).  The launch may cover a chunk of the step's rays: its N rays are rays ray_base .. ray_base+N-1
 * of n_rays_total (0 = N); all per-ray pointers are the chunk's.  Outputs: weights_sum[N], depth[N], image[N,3] (before the
 * blend), grad_bg[N,3] (optional), grad_sigmas[M], grad_rgbs[M,3]; *loss += the chunk's share of the entropy loss.
 * bg_half: f16[N,3] or NULL (then the colour bg_const).  Optional bookkeeping when counter != NULL (atomic):
 * *samples_total += counter[0]; step_counter[*cur_row] += counter.
 * ngp_train_light: the light direction of a shaded train step (nerf/renderer.py:461-464), one thread:
 * light f32[6] = (safe_normalize(rays_o[0..2] + z), z) with z three N(0, 1) draws (Box-Muller) from the generator of rng
 * (u64[3], as above) at keys no ray's jitter uses.  advance = 0: call it after a prologue launch that drew noise (it takes
 * that launch's counter, rng[1] - 1); advance = 1: it takes rng[1] and advances the counter itself.  So the light is
 * reproducible for a given (seed, step) and fresh on every step, graph replays included. */
int ngp_train_prologue(const float* rays_o, const float* rays_d, const float* aabb, uint32_t N, float min_near, float* nears,
                       float* fars, int* counters, uint32_t n_counters, float* loss, int* step_counter, int* local_step,
                       int* cur_row, float* noises, uint64_t* rng, void* stream);
int ngp_train_ray_loss(const float* sigmas, const float* rgbs, const float* deltas, const int* rays, uint32_t M, uint32_t N,
                       float T_thresh, const void* bg_half, float bg_const, const float* grad_pred, uint32_t pixels_per_view,
                       uint32_t ray_base, uint32_t n_rays_total, float lambda_entropy, const float* scale, float* weights_sum,
                       float* depth, float* image, float* grad_bg, float* grad_sigmas, float* grad_rgbs, float* loss,
                       const int* counter, unsigned long long* samples_total, int* step_counter, const int* cur_row,
                       void* stream);
int ngp_train_light(const float* rays_o, uint64_t* rng, int advance, float* light, void* stream);

/* Shading path as a 7-point stencil (nerf/network_grid.py:90-144; csrc/shading.cu).  ngp_stencil_points: xyzs f32[M,3] ->
 * out f32[M*K,3], K = 7 (x, x+eps e_x, x-eps e_x, x+eps e_y, ...) or 6 (with_centre == 0), shifted points clamped to
 * [-bound, bound] (:93-98): the K points of a sample are K consecutive rows of ONE field batch.  count_ptr (optional, as
 * ngp_field_forward takes it): M is then the capacity and min(*count_ptr, M) samples are read on the device; count_out
 * (optional) receives K times that count, for the field kernels that follow (K * M must fit an int).  NULL / NULL: all M.
 * ngp_shade_forward: the K
 * densities (sigma_all f32[M*K]) -> normal f32[M,3] = safe_normalize(-0.5 (s+ - s-) / eps), NaN -> 0 (:100-114) and, for
 * K = 7 and color_out != NULL, the colour of mode 0 lambertian (albedo * (ratio + (1 - ratio) max(n.l, 0)), albedo = the
 * centre row of rgb_all f32[M*K,3]), 1 textureless, 2 normal ((n + 1) / 2) with autocast's half roundings (:126-140).
 * ngp_shade_backward: d_normal f32[M,3] and / or d_color f32[M,3] -> d_sigma_all f32[M*K] (0 for the centre row) and
 * d_rgb_all f32[M*K,3] (centre row only; may be NULL). */
int ngp_stencil_points(const float* xyzs, uint32_t M, const int* count_ptr, float eps, float bound, int with_centre, float* out,
                       int* count_out, void* stream);
int ngp_shade_forward(const float* sigma_all, const float* rgb_all, uint32_t M, uint32_t K, const float* light, float ratio, int mode,
                      float* normal_out, float* color_out, void* stream);
int ngp_shade_backward(const float* sigma_all, const float* rgb_all, uint32_t M, uint32_t K, const float* light, float ratio, int mode,
                       const float* d_normal, const float* d_color, float* d_sigma_all, float* d_rgb_all, void* stream);
/* The same pair for the hand-scheduled shaded train step (K = 7, the sample count M = min(*count_ptr, M_cap) read on the
 * device, light f32[3] in device memory).  Rows >= M of every output are left untouched.
 * ngp_shade_forward_step: sigma_all f32[7 M_cap] / rgb_all f32[7 M_cap,3] -> sigma f32[M_cap] (the centre row's density)
 * and rgb f32[M_cap,3] (the colour of ngp_shade_forward, same arithmetic): the per-sample rows ngp_train_ray_loss reads.
 * ngp_shade_backward_step: the composite gradients d_sigma f32[M_cap] / d_rgb f32[M_cap,3] (ngp_train_ray_loss) ->
 * d_sigma_all f32[7 M_cap] (centre row: d_sigma; the six stencil rows: the normal's gradient) and d_rgb_all f32[7 M_cap,3]
 * (centre row: d(albedo) in mode 0, else 0; the stencil rows 0), with the orientation regulariser of
 * nerf/renderer.py:485-486 fused in: loss_orient = (1 - exp(-sigma)).detach() * clamp(n . d, 0)^2 (dirs f32[M_cap,3]: the
 * per-sample ray directions), averaged over the step's samples - the sum of counters[2c], c < n_counters, the i32[n,2]
 * counters of every ray chain of the step, so all their marches must be complete - and *loss += lambda_orient * mean (one
 * atomic per block).  Its gradient is multiplied by *scale (the GradScaler scale; NULL = 1) and joins the normal's
 * gradient ahead of the colour's.  loss may be NULL. */
int ngp_shade_forward_step(const float* sigma_all, const float* rgb_all, uint32_t M_cap, const int* count_ptr, const float* light,
                           float ratio, int mode, float* sigma, float* rgb, void* stream);
int ngp_shade_backward_step(const float* sigma_all, const float* rgb_all, uint32_t M_cap, const int* count_ptr, const int* counters,
                            uint32_t n_counters, const float* dirs, const float* light, float ratio, int mode, const float* d_sigma,
                            const float* d_rgb, float lambda_orient, const float* scale, float* d_sigma_all, float* d_rgb_all,
                            float* loss, void* stream);

/* The inference branch of run_cuda (nerf/renderer.py:496-532) as ONE launch: the reference's host loop - count alive rays
 * (a device->host sync per iteration), n_step = clamp(N / n_alive, 1, 8), march_rays, field, composite_rays, mask-compact -
 * becomes a CUDA-graph conditional WHILE node whose body is march -> fused field (ngp_field_forward) -> composite ->
 * device compaction -> a one-thread kernel that advances the loop state and sets the loop condition.  Same kernels'
 * arithmetic as ngp_march_rays / ngp_composite_rays (albedo shading), so weights_sum[N] / depth[N] / image[N,3] (zeroed
 * here, BEFORE the background blend and depth normalisation) equal the host loop's.  noises: f32[N] perturbation of the
 * first iteration, or NULL.  workspace: ngp_render_infer_workspace(N) bytes of device memory the caller keeps alive; the
 * executable graph is cached per argument set (keep pointers stable across frames).  Returns NGP_ERR_UNSUPPORTED if the
 * driver cannot build the conditional graph (callers then run the host loop).
 * ngp_render_infer_state copies the final loop state (int[8]: n_alive, n_step, step, cur, iterations, rows, -, -) to the host. */
uint64_t ngp_render_infer_workspace(uint32_t N);
int ngp_render_infer_loop(const float* rays_o, const float* rays_d, const float* nears, const float* fars, uint32_t N, float bound,
                          float dt_gamma, uint32_t max_steps, uint32_t C, uint32_t H, const uint8_t* grid, float T_thresh,
                          const float* noises, const void* table, const int* offsets, uint32_t L, uint32_t Cfeat, float S,
                          uint32_t Hres, uint32_t gridtype, int align_corners, const void* w1, const void* b1, const void* w2,
                          const void* b2, const void* w3, const void* b3, uint32_t hidden, uint32_t out_dim, float* weights_sum,
                          float* depth, float* image, void* workspace, uint64_t workspace_bytes, void* stream);
/* The same loop with the field forward reading the embeddings through a quad table (ngp_grid_quad_table over the same fp16
 * table, built by the caller before the launch; see ngp_field_forward_quads): bit-equal results. */
int ngp_render_infer_loop_quads(const float* rays_o, const float* rays_d, const float* nears, const float* fars, uint32_t N, float bound,
                          float dt_gamma, uint32_t max_steps, uint32_t C, uint32_t H, const uint8_t* grid, float T_thresh,
                          const float* noises, const void* table, const void* quads, const int* offsets, uint32_t L, uint32_t Cfeat, float S,
                          uint32_t Hres, uint32_t gridtype, int align_corners, const void* w1, const void* b1, const void* w2,
                          const void* b2, const void* w3, const void* b3, uint32_t hidden, uint32_t out_dim, float* weights_sum,
                          float* depth, float* image, void* workspace, uint64_t workspace_bytes, void* stream);
int ngp_render_infer_state(const void* workspace, int* state_host, void* stream);

/* Ray generation on the device: nerf/utils.py:43-106 get_rays (the N = -1 full-image branch, as nerf/provider.py:227 calls
 * it).  poses f32[B,4,4] row-major cam2world; intrinsics f32[4] = (fx, fy, cx, cy), or f32[B,4] when intrinsics_per_view
 * != 0 (one random focal per training view, provider.py:209-213).  Produces image rows row0, row0 + row_stride, ...
 * (n_rows of them; 0 = all that fit; row_stride 0 = 1) of every view: rays_o, rays_d f32[B, n_rows * W, 3].
 * ngp_train_prologue_rays = ngp_train_prologue with the rays generated instead of loaded (one launch; the rays are also
 * written out, the marcher and the background net read them). */
int ngp_get_rays(const float* poses, const float* intrinsics, int intrinsics_per_view, uint32_t B, uint32_t H, uint32_t W,
                 uint32_t row0, uint32_t row_stride, uint32_t n_rows, float* rays_o, float* rays_d, void* stream);
int ngp_train_prologue_rays(const float* poses, const float* intrinsics, int intrinsics_per_view, uint32_t B, uint32_t H,
                            uint32_t W, uint32_t row0, uint32_t row_stride, uint32_t n_rows, float* rays_o, float* rays_d,
                            const float* aabb, float min_near, float* nears, float* fars, int* counters, uint32_t n_counters,
                            float* loss, int* step_counter, int* local_step, int* cur_row, float* noises, uint64_t* rng,
                            void* stream);

/* End of run_cuda (nerf/renderer.py:535-557): image_out = image + (1 - weights_sum) * bg, depth_out =
 * clamp(depth - nears, 0) / (fars - nears) (NaN where the ray misses the box, as the reference), mask = nears < fars.
 * bg is f32[N,3] (bg_per_ray != 0) or one f32[3] colour.  depth_out / mask may be NULL. */
int ngp_blend_background_forward(const float* image, const float* weights_sum, const float* depth, const float* bg,
                                 int bg_per_ray, const float* nears, const float* fars, uint32_t N, float* image_out,
                                 float* depth_out, uint8_t* mask, void* stream);
/* Its backward: grad_weights_sum[n] = -sum_c grad_image[n,c] * bg[n,c]; grad_bg = (1 - weights_sum) * grad_image
 * (only when bg_per_ray; may be NULL).  The gradient wrt `image` is grad_image itself. */
int ngp_blend_background_backward(const float* grad_image, const float* weights_sum, const float* bg, int bg_per_ray,
                                  uint32_t N, float* grad_weights_sum, float* grad_bg, void* stream);

/* Opacity-entropy regulariser of train_step (nerf/utils.py:389-394): *loss = lambda * mean(-a log2 a - (1-a) log2(1-a)),
 * a = clamp(weights_sum, 1e-5, 1 - 1e-5).  Deterministic single-block reduction. */
int ngp_entropy_loss_forward(const float* weights_sum, uint32_t N, float lambda, float* loss, void* stream);
/* grad_weights_sum[n] (= or +=, per `accumulate`) (*grad_loss) * d loss / d weights_sum[n]; grad_loss is a DEVICE
 * scalar (the GradScaler's scale when the loss is scaled). */
int ngp_entropy_loss_backward(const float* weights_sum, uint32_t N, float lambda, const float* grad_loss,
                              float* grad_weights_sum, int accumulate, void* stream);

/* ------------------------------------------------------------------------------------------
 * Roofline micro-benchmarks (measurement support; SURVEY 8d asks for a measured L2 peak)
 * ------------------------------------------------------------------------------------------ */
/* Random 4-byte gathers: each of n_threads threads performs `iters` x 8 independent loads from
 * table u32[table_words] (table_words a power of two) and writes a checksum to sink u32[n_threads]. */
int ngp_bench_gather4(const uint32_t* table, uint32_t table_words, uint32_t* sink, uint32_t n_threads,
                      uint32_t iters, uint32_t seed, void* stream);
/* Random 8-byte red.global.add.v2.f32 into table f32[table_words]. */
int ngp_bench_red8(float* table, uint32_t table_words, uint32_t n_threads, uint32_t iters, uint32_t seed,
                   void* stream);

/* Random red.global.add of `width` (1, 2 or 4) consecutive floats per op; only every lane_stride-th lane of a warp
 * issues (1 = all 32 lanes).  Separates the per-lane issue cost from the L2 cost of the scatter. */
int ngp_bench_red_width(float* table, uint32_t table_words, uint32_t n_threads, uint32_t iters, uint32_t seed,
                        uint32_t width, uint32_t lane_stride, void* stream);

/* cudaGraphLaunch of an instantiated graph (cudaGraphExec_t) on `stream`.  The host framework's own replay call also
 * enqueues two fill kernels per replay for its random generators; a captured hand-scheduled step draws its noise on the
 * device (ngp_train_prologue), so it is launched bare. */
int ngp_graph_launch(void* graph_exec, void* stream);

/* Timeline support: writes the device's nanosecond clock (%globaltimer) to *slot when `stream` reaches this launch.
 * Capturable; NGP_TRACE-style tools bracket every entry point of a graphed step with two stamps (profiles/tools/timeline.py). */
int ngp_stamp(uint64_t* slot, void* stream);

/* Hardware self-test of the hand-written tcgen05 path (one CTA, one small fp16 GEMM with fp32 accumulate):
 * mode 0: D[128,N] = A[128,K] B[N,K]^T ; mode 1: D[M,N] = A[128,M]^T B[128,N] (M in {64,128}) ;
 * mode 2: D[128,N] = A[128,K] B[K,N].  A, B row-major fp16, D row-major fp32, N,K multiples of 16 <= 128. */
int ngp_tc_selftest(int mode, const void* A, const void* B, float* D, uint32_t M, uint32_t N, uint32_t K,
                    void* stream);

#ifdef __cplusplus
}
#endif
#endif /* NGP_B200_H_ */

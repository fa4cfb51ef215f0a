/*
 * drqv2_b200.h — C ABI of libdrqv2_b200.so: the DrQ-v2 agent-update hot path
 * as hand-written sm_100a CUDA kernels.
 *
 * The reference (johannah/drqv2) is pure Python/PyTorch and has no FFI of its
 * own; its plug-in point is the duck-typed agent class named in
 * cfgs/config.yaml:35 (`_target_: drqv2.DrQV2Agent`).  This header is the
 * boundary a maintainer binds (ctypes, see INTEGRATION.md) to replace the ATen
 * library kernels that drqv2.py / utils.py / replay_buffer.py launch.  Every
 * entry point cites the reference lines whose arithmetic it replaces.
 *
 * Conventions
 *   - plain pointers and sizes only; every pointer is a DEVICE pointer unless
 *     the name ends in `_host`.  The caller owns all memory.
 *   - every function enqueues work on `stream` (a cudaStream_t passed as
 *     void*) and returns immediately: no sync, no allocation, no host reads.
 *     All entry points are CUDA-graph capturable.
 *   - return value: 0 = ok; non-zero = error, text via drq_last_error().
 *   - there is NO CPU fallback: without a CUDA device every compute entry
 *     point fails with DRQ_ERR_CUDA.
 *
 * Layouts
 *   - parameters, gradients and Adam state are fp32 in the reference's own
 *     layouts (conv [Cout,Cin,3,3]; linear [out,in]), so state_dict tensors
 *     can alias them.
 *   - encoder activations use the "wide plane" layout: [N][32][DRQ_PLANE]
 *     with a fixed row stride of DRQ_PW = 41 elements for every layer (conv1's
 *     true output width).  Layer l's valid region is rows/cols < 41,39,37,35;
 *     other positions are don't-care in forward buffers and exactly zero in
 *     gradient buffers.  A 3x3 stride-1 tap (ky,kx) is then the constant
 *     offset ky*41+kx, which makes forward and dgrad the same shifted GEMM.
 *   - features handed to the heads are compact NCHW-flattened [N][39200],
 *     exactly drqv2.py:66 `h.view(h.shape[0], -1)`.
 */
#ifndef DRQV2_B200_H
#define DRQV2_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DRQ_SCAL_SLOT 32   /* floats per slot of the per-update host scalar ring (drq_scalars_fetch) */
#define DRQ_ABI_VERSION 2

#define DRQ_OK 0
#define DRQ_ERR_INVALID 1 /* bad argument */
#define DRQ_ERR_CUDA 2    /* CUDA runtime / launch failure */

#define DRQ_IMG 84          /* input frame height = width (dmc.py pixels wrapper) */
#define DRQ_PW 41           /* wide-plane row stride */
#define DRQ_PLANE 1696      /* wide-plane stride per channel (41*41=1681, padded) */
#define DRQ_CONV_CH 32      /* drqv2.py:55 */
#define DRQ_REPR_DIM 39200  /* drqv2.py:53 32*35*35 */

/* bf16 tensor-core mode: "WB" activation layout [4 channel-blocks][N*DRQ_PLB + DRQ_WB_SLACK pixel rows][8 ch]
 * (bf16); image n's wide position p is pixel row n*DRQ_PLB + DRQ_GUARD + p. */
#define DRQ_PLB 1776
#define DRQ_GUARD 88
#define DRQ_WB_SLACK 128

/* GEMM epilogues (drq_gemm_f32) */
#define DRQ_EPI_NONE 0       /* C = acc (+bias) */
#define DRQ_EPI_RELU 1       /* C = relu(acc + bias)            nn.ReLU in drqv2.py:77-81,103-111 */
#define DRQ_EPI_MASK 2       /* C = acc * (mask > 0)            ReLU backward */
#define DRQ_EPI_MASK_WIDE 3  /* as MASK, N index = compact feature k -> scatter into wide plane */

int drq_abi_version(void);
const char* drq_last_error(void);
/* number of SMs of the current device (0 if none) — used to size persistent grids */
int drq_device_sm_count(void);
/* SMs the persistent kernels (convs, GEMMs) size their grids for: 148 (default) or fewer.  A data-parallel update
 * leaves a few SMs to the NCCL all-reduce that runs beside the encoder backward - a persistent kernel keeps every SM it
 * got until it ends, so a collective that finds none free would either wait for it or make its late CTAs run their
 * (statically assigned) tiles after everyone else.  Read at launch time; the per-CTA workspaces are sized for 148. */
int drq_set_sm_limit(int sms);
/* on: drq_gemm_bf16 launches of the K-major / K-MN modes with 64-wide tiles use a two-stage pipeline (<= 66 KB of shared
 * memory) so that their CTAs fit on an SM BESIDE two resident CTAs of the persistent conv kernels (148 KB) - set by the
 * host around the launches of the actor pass, which runs beside the encoder backward.  Read at launch time. */
int drq_set_gemm_small(int on);
/* which kernel drq_conv3x3_fwd_bf16 / drq_conv3x3_dgrad_bf16 launch: 0 = one output pixel per accumulator row (N = 32
 * UMMAs, csrc/conv_tc.cu); 1 = a column of four output pixels per row (N = 32 / 64 / 96 UMMAs over the 6x3 input window,
 * tensor-map TMA loads; csrc/conv4x1_tc.cu) for launches of >= 48 images and the former below; 2 = the latter always;
 * 3 (default) = as 1 for the forward, the former for the data gradient (which runs beside other streams' kernels and
 * must leave them room on the SM); 4 = as 1 for the data gradient only.  Same arguments, layouts and results (to fp32
 * accumulation order).  Returns the previous mode; a value outside 0..4 only queries. */
int drq_set_conv4x1(int mode);
/* which kernel drq_conv1_fwd_bf16[_ring] launch: 0 = an im2col tile of 96 entries per output position is built in shared
 * memory; 1 (default) = for launches of >= 48 images the input pixels are converted once into parity planes and the nine
 * taps are descriptor offsets into them (9 UMMAs of K = 16 per tile of three output rows; csrc/conv1_tc.cu, both), the
 * former below; 2 = the latter always.  Same arguments, layouts and results (to fp32 accumulation order).  Returns the
 * previous value; a value outside 0..2 only queries. */
int drq_set_conv1_planes(int on);

/* ------------------------------------------------------------------ replay */

/* n-step gather from the GPU-resident uint8 ring.
 * Replaces ReplayBuffer._sample (replay_buffer.py:142-160) + default-collate +
 * utils.to_torch (utils.py:48-49).
 * Ring: one slot per environment step; slot s holds the newest frame
 * frames[s] u8[frame_c,84,84], action[s] f32[A], reward[s], discount[s].  An episode occupies
 * consecutive slots modulo `capacity`, row 0 being the reset step.
 * Sample i is (ep_start[i], idx[i]): first slot of its episode and the row
 * `idx` of replay_buffer.py:150.  Produces
 *   obs[i]      = stack of rows max(idx-1-(S-1-j),0), j=0..S-1   (dmc.py:86-109)
 *   next_obs[i] = same for row idx+nstep-1
 *   action[i]   = action[idx];  reward/discount = the fp32 chain of
 *                 replay_buffer.py:154-159, un-fused (bit-exact).
 * frame_c = channels per frame (3), stack = frames per observation (3). */
int drq_ring_gather_nstep(const uint8_t* frames, const float* action, const float* reward,
                          const float* discount, int64_t capacity, int frame_c, int stack, int A,
                          const int32_t* ep_start, const int32_t* idx, int B, int nstep,
                          float gamma, uint8_t* obs_out, uint8_t* next_obs_out,
                          float* action_out, float* reward_out, float* discount_out,
                          void* stream);

/* Device-side sampler: episode ~ U{0..E-1} then idx ~ U{1..len-nstep+1}
 * (replay_buffer.py:96-98,150).  ep_table is int32 [E][2] = (start slot, len)
 * with len = transitions in the episode (rows-1); E = *n_episodes is read on
 * the device so that a captured graph follows the ring as it fills.
 * Philox4x32-10 keyed by (seed, *counter); the kernel does not advance the
 * counter. */
int drq_ring_sample(const int32_t* ep_table, const int32_t* n_episodes, int nstep, uint64_t seed,
                    const uint64_t* counter, int32_t* ep_start_out, int32_t* idx_out, int B,
                    void* stream);

/* ------------------------------------------------------------------ RNG */

/* Every draw is Philox4x32-10 with key `seed` and counter (element index lo, index hi, word lo, word hi) where
 * word = (*counter << 3) | stream.  Streams: 0 = replay sample (the loader's seed), 1 = shifts, 3 = the update's
 * noise, 5 = drq_rng_normal_f32.  Integers are multiply-shift reductions of a word w: (w * range) >> 32 - the
 * sample's episode from word 0 (range E), its idx - 1 from word 1 (range len - nstep + 1); shift_obs (x, y) from
 * words 0, 1 and shift_next (x, y) from words 2, 3 of element b (range 2 * pad + 1).  Normals are Box-Muller on
 * the pair i >> 1: u = ((float)(w >> 8) + 0.5f) * 2^-24 in fp32, so above 2^23 the + 0.5 rounds to even and u
 * lies on a 2^-23 grid, and w >> 8 == 0xFFFFFF gives u1 = 1.0 exactly: a normal of +0 or -0.  Element i is
 * sqrt(-2 ln u1) * cos(2 pi u2), sin when i is odd; eps_critic takes words 0 (u1) and 1 (u2), eps_actor
 * words 2 and 3, drq_rng_normal_f32 words 0 and 1.  A launch writes elements [0, B) / [0, B*A) / [0, n) and
 * nothing past them (tests/test_gpu_draws.py holds every producer to this, tests/helpers.py restates it). */

/* Per-update random draws, in the reference's order (drqv2.py:241-242 shifts,
 * utils.py:119 noise x2): shift_obs/shift_next int32 [B][2] = (x, y) in
 * [0, 2*pad], eps_critic/eps_actor f32 [B][A] ~ N(0,1).  Keyed by
 * (seed, *counter) on streams 1 and 3; the kernel does not advance `counter` (drq_counter_advance does). */
int drq_rng_update_draws(uint64_t seed, const uint64_t* counter, int pad, int32_t* shift_obs,
                         int32_t* shift_next, float* eps_critic, float* eps_actor, int B, int A,
                         void* stream);
/* out[0..n) ~ N(0,1): the exploration noise of act() (drqv2.py:172, utils.py:119). */
int drq_rng_normal_f32(uint64_t seed, const uint64_t* counter, float* out, int n, void* stream);
int drq_counter_advance(uint64_t* counter, void* stream);

/* Per-update host scalars for graph replays: out[0..DRQ_SCAL_SLOT) = ring[*cursor % slots][..], then *cursor += 1.
 * One slot: Adam scalars (8 floats, see drq_adam_step) of critic_opt at [0, 8), stddev(step) at [8], encoder_opt at
 * [16, 24), actor_opt at [24, 32) - torch.optim.Adam keeps a step count per optimiser (drqv2.py:148-150).
 * `ring` is pinned (device-visible) host memory of slots x DRQ_SCAL_SLOT floats that the host fills ahead of the device -
 * the Adam bias corrections of torch/optim/adam.py:531-547 and the exploration stddev of utils.py:130-146 change
 * every update, a captured graph cannot take new arguments, and a single staging buffer would be overwritten by
 * a host that enqueues updates faster than the device runs them.  `cursor` is a device counter. */
int drq_scalars_fetch(const float* ring, int slots, uint64_t* cursor, float* out, void* stream);

/* A sampled batch as a view of the replay ring: everything the sampler and the consumers of one batch need, so that
 * the frame stacks never have to be materialised (north_star (1)/(2): "builds the frame stack by index", "augmented
 * frames are never materialised").  Filled by the host once per (ring, loader); all pointers are device pointers.
 * Reference: ReplayBuffer._sample replay_buffer.py:142-160 and the stack layout of dmc.py:86-109. */
typedef struct {
    const uint8_t* frames; const float* action; const float* reward; const float* discount;   /* ring arrays */
    int64_t capacity;                     /* ring slots */
    int32_t frame_c, stack, A, nstep;     /* channels per frame, frames per stack, action dim, n-step */
    float gamma; int32_t reserved;
    const int32_t* ep_table; const int32_t* n_episodes;   /* sampler input: (start slot, rows) per eligible episode */
    uint64_t seed; uint64_t* counter;                     /* sampler key and draw counter (device) */
    int32_t* ep_start; int32_t* idx;                      /* [B] sampled (episode start slot, idx) - written by the
                                                             prologue, read by the conv1 loaders */
} drq_ring_src;

/* drq_update_prologue + drq_ring_sample_step + the action / n-step reward / discount part of drq_ring_gather_nstep in
 * ONE one-block launch: the head of a ring-fed update.  The frame stacks are not gathered: drq_conv1_*_bf16_ring read
 * them from the ring through (ep_start, idx).  Results are bit-identical to the three separate calls. */
int drq_update_prologue_ring(const float* scal_ring, int slots, uint64_t* cursor, float* scal_out, uint64_t seed,
                             uint64_t* counter, int pad, int32_t* shift_obs, int32_t* shift_next, float* eps_critic,
                             float* eps_actor, int B, int A, const drq_ring_src* src, float* action_out,
                             float* reward_out, float* discount_out, void* stream);

/* The same in two launches: part 1 = what the encoder's first kernel waits for (the two shift draws and the replay
 * sample (ep_start, idx)); part 2 = the rest (host scalars, the two noise draws, action copy, n-step reward / discount),
 * launched after part 1 - on a side stream it runs beside conv1.  part 3 = drq_update_prologue_ring.  Bit-identical.
 * Part 1 advances the sampler's counter only: it reads *counter but leaves it and the scalar cursor to part 2. */
int drq_update_prologue_ring_part(const float* scal_ring, int slots, uint64_t* cursor, float* scal_out, uint64_t seed,
                                  uint64_t* counter, int pad, int32_t* shift_obs, int32_t* shift_next, float* eps_critic,
                                  float* eps_actor, int B, int A, const drq_ring_src* src, float* action_out,
                                  float* reward_out, float* discount_out, int part, void* stream);

/* drq_ring_sample followed by *counter += 1 in one launch (one block). */
int drq_ring_sample_step(const int32_t* ep_table, const int32_t* n_episodes, int nstep, uint64_t seed, uint64_t* counter,
                         int32_t* ep_start_out, int32_t* idx_out, int B, void* stream);

/* everything an update needs before its first real kernel, in one launch (one block): drq_scalars_fetch, then -
 * unless shift_obs == NULL (injected draws) - drq_rng_update_draws and *counter += 1.  With shift_obs == NULL no draw
 * buffer is written and the counter is neither read nor advanced (also in drq_update_prologue_ring[_part]). */
int drq_update_prologue(const float* scal_ring, int slots, uint64_t* cursor, float* scal_out, uint64_t seed, uint64_t* counter,
                        int pad, int32_t* shift_obs, int32_t* shift_next, float* eps_critic, float* eps_actor, int B, int A,
                        void* stream);

/* ------------------------------------------------------------------ augmentation */

/* RandomShiftsAug as an exact integer shift (drqv2.py:19-45 in intent):
 * out[n,c,r,col] = in[n,c,clamp(r+sy-pad,0,H-1),clamp(col+sx-pad,0,W-1)],
 * shift[n] = (sx, sy).  Stand-alone (materialising) form used by the
 * RandomShiftsAug module; the update path uses the fused conv1 loader. */
int drq_random_shift_f32(const float* in, const int32_t* shift, float* out, int N, int C, int H,
                         int W, int pad, void* stream);

/* Its transpose, the backward of the RandomShiftsAug module w.r.t. its input: dx[n,c,i,j] = sum of dout[n,c,r,col]
 * over every (r, col) with clamp(r+sy-pad,0,H-1) = i and clamp(col+sx-pad,0,W-1) = j, summed in fp32 in ascending
 * (r, col) order (deterministic, no atomics).  A pixel takes none, one or several: the first / last rows and columns
 * take the whole clamped run, and on the side the image moves away from there are pixels that take none - those are
 * written as +0.  Reads dout [N][C][H][W] and shift [N][2] (x, y), and nothing else; writes every element of dx
 * [N][C][H][W] exactly once and nothing else. */
int drq_random_shift_bwd_f32(const float* dout, const int32_t* shift, float* dx, int N, int C, int H, int W, int pad,
                             void* stream);

/* ------------------------------------------------------------------ encoder, fp32 */

/* conv1 of drqv2.py:55 (Cin->32, k3, stride 2) + ReLU, with RandomShiftsAug
 * (integer shift, pad 4) and `obs / 255.0 - 0.5` (drqv2.py:64) fused into the
 * loader.  obs u8 [N][cin][84][84]; shift int32 [N][2] (x,y) or NULL for no
 * augmentation (act path).  out: wide plane [N][32][DRQ_PLANE]; writes positions [0, 1681) of each
 * plane (the 41 x 41 output) and nothing else - the plane's slack [1681, DRQ_PLANE) is left as it was. */
int drq_conv1_fwd_f32(const uint8_t* obs, const int32_t* shift, const float* w, const float* b,
                      float* out, int N, int cin, int pad, void* stream);

/* weight/bias gradient of conv1: dw [32][cin][3][3], db [32] from
 * dpre (wide, gradient w.r.t. the pre-ReLU output; read on [0, 1681) of each plane only).
 * partial: workspace of drq_conv_wgrad_ws_floats(cin) floats. */
int drq_conv1_wgrad_f32(const uint8_t* obs, const int32_t* shift, const float* dpre,
                        float* partial, float* dw, float* db, int N, int cin, int pad,
                        void* stream);

/* The same two from real-valued pixels: obs fp32 [N][cin][84][84] on the 0..255 scale, already augmented (no shift),
 * any value (no range, integrality or finiteness check).  The loader computes x/255 - 0.5 exactly as the u8 loader
 * does, so integer-valued pixels give the bits of drq_conv1_{fwd,wgrad}_f32 with shift = NULL.  Same outputs, same
 * write sets; the wgrad reads dpre on [0, 1681) of each plane only. */
int drq_conv1_fwd_f32_from_f32(const float* obs, const float* w, const float* b, float* out, int N, int cin,
                               void* stream);
int drq_conv1_wgrad_f32_from_f32(const float* obs, const float* dpre, float* partial, float* dw, float* db, int N,
                                 int cin, void* stream);

/* conv1's data gradient w.r.t. the pixels (the backward of drqv2.py:64-65 through conv1, 1/255 included):
 * dx[n][c][iy][ix] = (sum over taps (ky, kx) with iy = 2oy+ky, ix = 2ox+kx, oy, ox < 41, and over co, of
 * w[co][c][ky][kx] * dpre[n][co][oy*41 + ox]) / 255 - at most 2 x 2 taps x 32 channels per pixel; row and column 83
 * take no tap.  dpre: wide, gradient w.r.t. conv1's pre-ReLU output, read on [0, 1681) of each plane only; w fp32
 * [32][cin][3][3].  Writes every element of dx fp32 [N][cin][84][84] exactly once (+0 at row 83) and nothing else.
 * CUDA cores, fixed summation order (taps ascending, co ascending within a tap), then one division by 255. */
int drq_conv1_dgrad_f32(const float* dpre, const float* w, float* dx, int N, int cin, void* stream);

/* conv2..4 of drqv2.py:56-59 (32->32, k3, stride 1) + ReLU.
 * in: wide plane; hout = valid output rows = cols (39, 37 or 35).
 * compact_out == 0: writes positions [0, hout*41) of each plane of the wide
 * out (rows < hout, all 41 columns; columns >= hout hold values without
 * meaning), nothing else.  compact_out != 0: writes exactly out[N][32][hout][hout]
 * (the flattened features of drqv2.py:66) instead.  Valid outputs read `in`
 * only inside hin x hin (hin = hout + 2); the rest of the plane may hold
 * anything, NaN included. */
int drq_conv3x3_fwd_f32(const float* in, const float* w, const float* b, float* out, int N,
                        int hout, int compact_out, void* stream);

/* data gradient: din_pre[ci][q] = relu'(act_in[ci][q]) * sum_{co,tap} w[co][ci][tap] dout[co][q-off].
 * dout: wide, gradient w.r.t. this layer's PRE-ReLU output.  It is read on
 * positions [0, (hout+2)*41) of each plane, and there it must be +0 outside
 * the valid hout x hout region: in rows hout, hout+1 and in columns >= hout.
 * Rows >= hout+2 and the slack are not read.  act_in: this layer's input
 * activation (post-ReLU output of the layer below), used as the ReLU mask and
 * read inside hin x hin (hin = hout + 2) only.  din: wide, gradient w.r.t. the
 * layer below's pre-ReLU output; written on [0, (hout+2)*41) of each plane -
 * rows < hout+2, with +0 at columns >= hout+2 - and nowhere else: its rows
 * >= hout+2 and its slack are left as they were, so a caller that passes din
 * on as the next layer's dout (hout' = hout+2) keeps its rows hout', hout'+1
 * at +0 itself (drqv2.py's workspace allocates them zeroed and no kernel
 * writes them). */
int drq_conv3x3_dgrad_f32(const float* dout, const float* w, const float* act_in, float* din,
                          int N, int hout, void* stream);

/* weight/bias gradient of a 32->32 layer.  in: wide input activation, read on
 * the whole plane [0, DRQ_PLANE): outside hin x hin it must be finite (it
 * meets zeros of dpre there, and 0 * NaN is NaN).  dpre: wide gradient w.r.t.
 * the pre-ReLU output, read on [0, hout*41) only, and +0 there outside the
 * valid hout x hout region (columns >= hout).  partial: workspace of
 * drq_conv_wgrad_ws_floats(32) floats. */
int drq_conv3x3_wgrad_f32(const float* in, const float* dpre, float* partial, float* dw,
                          float* db, int N, int hout, void* stream);
int64_t drq_conv_wgrad_ws_floats(int cin);

/* conv4's pre-ReLU gradient from an arbitrary gradient of the features (the backward of the autograd Encoder,
 * drqv2.py:66-67: whatever losses consumed the features, their gradients already summed).  dfeat and feat are
 * compact [N][39200] (c*1225 + y*35 + x; feat = conv4's post-ReLU output, the mask); dpre is wide [N][32][DRQ_PLANE]:
 * dpre[n][c][y*41 + x] = feat > 0 ? dfeat : +0 inside 35 x 35, and +0 at rows 35-36 and at columns 35-40 of rows
 * < 35.  Writes exactly positions [0, 37*41) of each plane - the set drq_conv3x3_dgrad_f32 reads at hout = 35, with
 * the zeros it requires - and nothing else.  DRQ_EPI_MASK_WIDE does the same fused into the trunk's data-gradient
 * GEMM, for one consumer and without the zero rows. */
int drq_feature_grad_wide_f32(const float* dfeat, const float* feat, float* dpre, int N, void* stream);

/* ------------------------------------------------------------------ encoder, bf16 tensor cores */

/* bf16 elements of a WB buffer holding n_images images. */
int64_t drq_wb_elems(int n_images);

/* fp32 conv weight [32][32][3][3] -> the two packed bf16 UMMA B operands ([36][32][8] each)
 * used by the forward and data-gradient kernels. */
int drq_pack_conv_w_bf16(const float* w, uint16_t* w_fwd, uint16_t* w_dgrad, void* stream);

/* conv2..4 (drqv2.py:56-59) + bias + ReLU on tcgen05 tensor cores, bf16 in / fp32 accumulate
 * (TMEM) / bf16 out.  in, out: WB buffers of N images.  nhwc_out == 1: out is the compact NHWC
 * feature matrix [N][hout*hout][32]; nhwc_out == 2: out is the TB feature matrix the tensor-core
 * trunk consumes (feature (c/8)*hout*hout*8 + (y*hout+x)*8 + c%8, feat_rpad = units per row = hout*hout*4); image n is row n
 * for n < feat_half and row n - feat_half + feat_half_row after it (the next_obs half of an update starts
 * on its own 128-row block); feat_half <= 0: row = image.  What is written: WB out = rows < hout of images < N - the
 * four-pixel-column kernel stores columns < hout only, the one-pixel kernel whole 41-pixel rows (columns hout..40 then
 * hold values no later kernel reads); NHWC = images < N; TB = the rows of images < N.  Nothing else (guard rows, slack,
 * TB rows of no image) is touched.  The data gradient writes rows < hout + 2 of images < N, all 41 columns, with exact
 * zeros past column hout + 1. */
int drq_conv3x3_fwd_bf16(const uint16_t* in, const uint16_t* w_fwd, const float* bias, uint16_t* out,
                         int N, int hout, int nhwc_out, int64_t feat_rpad, int feat_half, int feat_half_row,
                         void* stream);

/* data gradient on tensor cores; dout/din: WB buffers of N images (zero guard rows);
 * act_in: WB buffer of n_act >= N images holding the layer's input activation (ReLU mask). */
int drq_conv3x3_dgrad_bf16(const uint16_t* dout, const uint16_t* w_dgrad, const uint16_t* act_in,
                           int n_act, uint16_t* din, int N, int hout, void* stream);

/* weight + bias gradient of a 32->32 layer on tensor cores (fp32 accumulation in TMEM, fp32
 * output in the reference layout dw [32][32][3][3], db [32]).  in: WB buffer of n_in >= N images
 * (input activation), dpre: WB buffer of N images.  partial: drq_conv_wgrad_bf16_ws_floats(). */
int drq_conv3x3_wgrad_bf16(const uint16_t* in, int n_in, const uint16_t* dpre, float* partial, float* dw,
                           float* db, int N, int hout, void* stream);
int64_t drq_conv_wgrad_bf16_ws_floats(void);

/* conv1 (drqv2.py:55, stride 2) with RandomShiftsAug + obs/255-0.5 fused into the loader, tensor
 * cores.  The im2col entries are the exact integers x-128 in bf16 (built from the uint8 pixels by byte
 * permutes); the affine map x/255-0.5 is applied in the epilogue: out = relu(acc/255 + b'),
 * b' = b + (128/255-0.5) sum_k bf16(W[co][k]).  w_packed: drq_conv1_w_packed_elems() uint16 elements =
 * bf16 weights [12 K units][32][8] (K = cin*9 padded to 96) followed by float b'[32].  cin*9+1 <= 96. */
int64_t drq_conv1_w_packed_elems(void);
int drq_pack_conv1_w_bf16(const float* w, const float* bias, uint16_t* out, int cin, void* stream);
int drq_conv1_fwd_bf16(const uint8_t* obs, const int32_t* shift, const uint16_t* w_packed, uint16_t* out, int N,
                       int cin, int pad, void* stream);
/* conv1 weight + bias gradient (fp32, reference layout) from dpre (WB bf16 of N images). */
int drq_conv1_wgrad_bf16(const uint8_t* obs, const int32_t* shift, const uint16_t* dpre, float* partial,
                         float* dw, float* db, int N, int cin, int pad, void* stream);
/* The same two kernels with the row producer addressing the replay ring directly: image n < B is the stack of
 * sample n at rows idx-1 (obs), image n >= B the stack of sample n-B at rows idx+nstep-1 (next_obs), channel
 * c = frame (c / frame_c) of the stack = ring frame max(t - (stack-1-j), 0) of the episode (dmc.py:98-109,
 * replay_buffer.py:151,153).  cin = frame_c * stack.  Bit-identical to drq_ring_gather_nstep followed by the
 * plain kernels (tests/test_gpu_ring_direct.py). */
int drq_conv1_fwd_bf16_ring(const drq_ring_src* src, int B, const int32_t* shift, const uint16_t* w_packed,
                            uint16_t* out, int N, int pad, void* stream);
int drq_conv1_wgrad_bf16_ring(const drq_ring_src* src, int B, const int32_t* shift, const uint16_t* dpre,
                              float* partial, float* dw, float* db, int N, int pad, void* stream);

int64_t drq_conv1_wgrad_bf16_ws_floats(void);

/* The same two from real-valued pixels: obs fp32 [N][cin][84][84] on the 0..255 scale, already augmented (no shift),
 * any value (no range, integrality or finiteness check), through the im2col kernel at every batch size.  The im2col
 * entries are RN-bf16(RN-fp32(x - 128)) - the pixel's rounding point: exact for integers in 0..255 (so integer-valued
 * pixels give the bits of the im2col selection of drq_conv1_{fwd,wgrad}_bf16, drq_set_conv1_planes(0), with shift =
 * NULL), 8 significant bits otherwise - and the epilogues are those of the u8 kernels.  Same outputs and write sets.
 * The wgrad's partial holds drq_conv1_wgrad_bf16_ws_floats() floats; dw and db are required. */
int drq_conv1_fwd_bf16_from_f32(const float* obs, const uint16_t* w_packed, uint16_t* out, int N, int cin,
                                void* stream);
int drq_conv1_wgrad_bf16_from_f32(const float* obs, const uint16_t* dpre, float* partial, float* dw, float* db, int N,
                                  int cin, void* stream);

/* conv1's data gradient w.r.t. the pixels on tcgen05 tensor cores: per tile of three output rows, col[p][9c + tap] =
 * sum_co dpre[p][co] * W[co][9c + tap] (M = 128 positions, N = 96, K = 32; bf16 operands, fp32 accumulation in TMEM),
 * then col2im in the epilogue: dx[n][c][iy][ix] = (sum of the <= 4 col entries of the pixel) / 255, fp32, summed from
 * +0 with taps (ky, kx) ascending - except input rows 6t (t = 1..13), which two tiles share: their sum starts with the
 * ky = 2 taps of tile t-1 (kx ascending), carried in shared memory, and adds the ky = 0 taps of tile t (kx
 * ascending).  Row 83 and column 83 take no tap (+0).  A CTA walks whole images, tiles in order (deterministic, no
 * atomics, no global scratch).
 *   dpre: WB bf16 buffer of N images, conv1's pre-ReLU gradient.  Read: pixel rows n*DRQ_PLB + DRQ_GUARD + [0, 1727)
 *     of every channel block (positions 1681.. reach only accumulator rows that are never stored: they may hold
 *     anything, NaN included; the last image's reads end inside the buffer's slack).
 *   w_packed: the packed conv1 operand of drq_pack_conv1_w_bf16; its bf16 weights [12][32][8] are read (entries of
 *     k >= cin*9 reach only unused columns: anything), the fused biases behind them are not.
 *   dx: fp32 [N][cin][84][84]; every element written exactly once, nothing else.
 * Grid min(N, 2 x the SM budget) CTAs of 128 threads. */
int drq_conv1_dgrad_bf16(const uint16_t* dpre, const uint16_t* w_packed, float* dx, int N, int cin, void* stream);

/* ------------------------------------------------------------------ dense, bf16 tensor cores */

/* Tile-blocked "TB" layout of every bf16 matrix the tensor-core heads touch (activations, gradients,
 * packed weights):  X_tb[row / R][feature / 8][row % R][feature % 8]  - 16-byte units of 8 consecutive
 * features, R rows per unit block, the `units` (= padded features / 8, features padded to a multiple
 * of 16) unit blocks of one row block adjacent; rows zero padded to a multiple of R.  R = DRQ_TB_ACT
 * for activations / gradients, DRQ_TB_W for weights.  The same buffer is a K-major operand when the
 * contraction runs over the feature dim and an MN-major operand when it runs over the rows (weight
 * and data gradients), and every operand tile is one contiguous span (one bulk-async copy). */
#define DRQ_TB_ACT 128
#define DRQ_TB_W 64

/* operand modes of drq_gemm_bf16 */
#define DRQ_GEMM_KK 0    /* A activation, contraction over its features; B weight, over its features (Linear forward)   */
#define DRQ_GEMM_KMN 1   /* A activation, over its features; B weight, contraction over its rows (data gradient)         */
#define DRQ_GEMM_MNMN 2  /* A and B activations, contraction over their rows (weight gradient: M = A features)          */

/* epilogues of drq_gemm_bf16 */
#define DRQ_TEPI_F32 0          /* C(fp32 row-major, stride ldc) = acc (+bias) (+C if accumulate)   */
#define DRQ_TEPI_RELU_BF16 1    /* C(TB bf16 activation, units = ldc) = relu(acc + bias)             */
#define DRQ_TEPI_MASK_BF16 2    /* C(TB bf16) = acc * (mask > 0), mask TB activation with units_mask  */
#define DRQ_TEPI_TRUNK_WGRAD 3  /* C(fp32)[m][ref(n)] = acc: encoder-output feature column -> reference order */
#define DRQ_TEPI_TRUNK_DGRAD 4  /* C(WB bf16 of conv4's gradient) = acc * (feature > 0), scattered; ldc = WB block stride in rows; mask = TB features */

/* C[M,N] = sum_k A(m,k) B(n,k) on tcgen05 tensor cores, bf16 TB operands, fp32 accumulate (TMEM).
 * units_a / units_b: units per row of the operand buffers.  TB outputs write feature columns
 * [0, max(N, n_store)) with zeros beyond N; n_store may not lie past the last N tile (ceil(N / bn) * bn).  batch > 1: grid z = zo * batch_inner + zi, operand z at
 * offset zi * strides[0..4] + zo * strides[5..9] (elements; a, b, c, bias, mask; strides == NULL: 0;
 * strides has 11 entries).  splitk > 1 (DRQ_GEMM_KK, fp32): plane s of C (stride strides[10]) receives
 * the partial sum of K chunk s (bias is not applied); grid z = batch entry * splitk + s.
 * bn = N tile: 64 (all modes) or 128 (KMN, MNMN).
 * What a launch reads:  a K-major operand (contraction over its features: A of KK / KMN, B of KK) is read up to
 * ceil(K/16)*16 features of each chunk; an MN-major operand (contraction over its rows: B of KMN, A and B of MNMN) is
 * read as whole row blocks (128 rows, weights 64), of which only the first ceil(K/16)*16 rows enter the UMMAs.  Rows
 * of a K-major operand past M (N), and features of an MN-major operand past M (N), reach only outputs that are not
 * stored: they may hold anything.  Padding INSIDE the read extent must be zero: features [K, ceil(K/16)*16) of K-major
 * operands and rows [K, ceil(K/16)*16) of MN-major ones (the rows [B, ceil(B/16)*16) of every activation or gradient
 * contracted over the batch).  The library keeps that: its TB buffers start zeroed and every producer of one (these
 * epilogues, drq_ln_tanh_fwd*, drq_ln_tanh_bwd, drq_actor_sample_bwd, drq_policy_head_fwd_bf16, the conv4 feature
 * epilogue) writes rows < B only.  (tests/test_gpu_gemm_edges.py fills everything past the extent with NaN.) */
int drq_gemm_bf16(const uint16_t* A, int units_a, const uint16_t* B, int units_b, int mode, void* C, int64_t ldc,
                  int n_store, const float* bias, const uint16_t* mask, int units_mask, int M, int N, int K,
                  int epilogue, int accumulate, int batch, int batch_inner, const int64_t* strides, int splitk,
                  int bn, void* stream);

/* debug aid: clock64 timeline of block (0,0,0) of every later drq_gemm_bf16 launch into buf (>= 16
 * int64, device memory); NULL switches it off. */
int drq_debug_gemm_stamps(int64_t* buf);
/* the same for drq_conv3x3_{fwd,dgrad}_bf16: [0] producer wait-for-empty, [1] producer total, [2] issuer
 * wait-for-accumulator, [3] issuer wait-for-data, [4] issuer total, [5] epilogue wait-for-accumulator (cycles). */
int drq_debug_conv_stamps(int64_t* buf);
/* 6 words of MAPPED HOST memory (cudaHostAlloc / torch pin_memory; readable after the context died), or null: a bounded
 * mbarrier wait that gives up writes {1 = plain / 2 = sleeping wait, block size, thread, barrier shared-memory address,
 * parity, block} there before it traps - tells which role of which kernel stopped making progress */
int drq_debug_trap_note(uint32_t* mapped_host_words);
/* 12 clock64 totals of block 0 of the four-pixel-column conv kernels (device buffer, or null = off): producer {wait
 * stage, -, -, total}, UMMA warp {wait accumulator, wait stage, issue, total}, first epilogue warp {wait accumulator,
 * TMEM load, math + stores, total} */
int drq_debug_conv4x1_stamps(int64_t* buf);
/* drq_conv1_fwd_bf16 builders (threads 0 / 128 of block 0 at [0..4] / [8..12]): wait-for-rows, re-pitch,
 * barrier, wait-for-free-tile, build (cycles). */
int drq_debug_conv1_stamps(int64_t* buf);

/* fp32 nn.Linear weight [rows][cols] -> TB(DRQ_TB_W) bf16 [ceil(rows/64)][ceil16(cols)/8][64][8]. */
int drq_pack_linear_tb(const float* w, uint16_t* out, int rows, int cols, void* stream);
/* trunk Linear(39200->rows) weight -> TB(DRQ_TB_W) bf16 in the feature order (c/8)*9800 + (y*35+x)*8 + c%8
 * of the bf16 encoder output (reference column c*1225+y*35+x, drqv2.py:66). */
int drq_pack_trunk_tb(const float* w, uint16_t* out, int rows, void* stream);
/* encoded features fp32 [rows][39200] in the reference's flatten order (drqv2.py:66) -> TB(DRQ_TB_ACT) bf16 in the
 * encoder-output feature order; `out` points at a 128-row block boundary of the feature operand.  Behind the stage
 * API DrQV2Agent.update_critic / update_actor (drqv2.py:177,206), which take features, in the tensor-core mode. */
int drq_pack_features_tb(const float* feat, uint16_t* out, int rows, void* stream);

/* all bf16 operand re-packs of one optimiser phase in one launch.  kind LINEAR: drq_pack_linear_tb(w, out,
 * rows, cols); TRUNK: drq_pack_trunk_tb(w, out, rows); CONV: drq_pack_conv_w_bf16(w, out, out2);
 * CONV1: drq_pack_conv1_w_bf16(w, bias, out, cin = cols). */
#define DRQ_PACK_LINEAR 0
#define DRQ_PACK_TRUNK 1
#define DRQ_PACK_CONV 2
#define DRQ_PACK_CONV1 3
#define DRQ_PACK_MAX_JOBS 12
typedef struct { int32_t kind; int32_t rows; int32_t cols; int32_t reserved; const float* w; const float* bias; uint16_t* out; uint16_t* out2; } drq_pack_job;
int drq_pack_multi(const drq_pack_job* jobs, int njobs, void* stream);

/* all bias gradients (column sums over the batch rows) of one backward pass in one launch: out[n] =
 * sum_m X[m][n], X fp32 row-major with row stride ld (tb == 0) or a TB bf16 activation with ld units per
 * row (tb != 0).  With Y (fp32 jobs) the sum runs over the elementwise product - LayerNorm's dgamma. */
#define DRQ_COLSUM_MAX_JOBS 8
typedef struct { const void* X; int64_t ld; float* out; int32_t M; int32_t N; int32_t tb; int32_t reserved;
                 const float* Y; /* fp32 jobs: nullable, same shape/ld as X: out[n] = sum_m X[m][n] * Y[m][n] */ } drq_colsum_job;
int drq_colsum_multi(const drq_colsum_job* jobs, int njobs, void* stream);

/* all weight/bias-gradient reductions of the encoder backward in one launch: drq_conv3x3_wgrad_bf16 /
 * drq_conv1_wgrad_bf16 called with dw == db == NULL leave their per-CTA partials in `partial`; this call
 * reduces them (fixed order) into dw / db.  cin > 0: a conv1 job (N images); cin == 0: a conv3x3 job (N, hout). */
#define DRQ_WGRAD_REDUCE_MAX_JOBS 4
typedef struct { const float* partial; float* dw; float* db; int32_t n_images; int32_t hout; int32_t cin; int32_t reserved; } drq_wgrad_reduce_job;
int drq_conv_wgrad_reduce_multi(const drq_wgrad_reduce_job* jobs, int njobs, void* stream);

/* ------------------------------------------------------------------ dense, fp32 */

/* C[z][m][n] = epi( sum_k A[z](m,k) * B[z](k,n) + bias[z][n] ), general strides.
 * A(m,k) = A[m*sa_m + k*sa_k], B(k,n) = B[k*sb_k + n*sb_n], C row stride ldc.
 * batch > 1: independent problems at pointer strides (bs_a, bs_b, bs_c,
 * bs_bias, bs_mask) — the twin Q heads of drqv2.py:103-111.
 * splitk > 1 (batch must be 1): K is cut in `splitk` chunks and chunk s writes
 * its raw partial sum to C + s*bs_c (bias/epilogue ignored) — reduced in fixed
 * order by drq_ln_tanh_fwd.
 * accumulate != 0: C += result (after epilogue).  DRQ_EPI_MASK: mask(m, n) =
 * mask[m*ldmask + n] (at mask + z*bs_mask per batch entry).  DRQ_EPI_MASK_WIDE
 * (N = 39200): the mask is the compact feature matrix [M][ldmask] and column n
 * = c*1225 + y*35 + x is stored at C[m*ldc + c*DRQ_PLANE + y*41 + x] - only
 * those compact->wide positions are written; columns and rows 35..40 of each
 * plane and its slack are left as they were.  Every epilogue writes rows < M,
 * columns < N (split planes z < splitk) and nothing else. */
int drq_gemm_f32(const float* A, int64_t sa_m, int64_t sa_k, const float* B, int64_t sb_k,
                 int64_t sb_n, float* C, int64_t ldc, const float* bias, const float* mask,
                 int64_t ldmask, int M, int N, int K, int epilogue, int accumulate, int batch,
                 int64_t bs_a, int64_t bs_b, int64_t bs_c, int64_t bs_bias, int64_t bs_mask,
                 int splitk, void* stream);

/* out[z][n] = sum_m X[z][m*ld + n]  — bias gradients. */
int drq_colsum_f32(const float* X, int64_t ld, float* out, int M, int N, int batch, int64_t bs_x,
                   int64_t bs_out, void* stream);

/* trunk tail: z = sum_s partial[s] + bias; LayerNorm(F, eps) affine; tanh
 * (drqv2.py:74-75,100-101).  h written at h_out[b*ld_h + f] (so it can land in
 * the [h, action] concat buffer of drqv2.py:117).  xhat [B][F] and rstd [B]
 * are saved for backward when non-NULL; h_bf16 (nullable, TB activation layout, rpad_hb = units per row) receives a bf16 copy of h for the tensor-core heads. */
int drq_ln_tanh_fwd(const float* partial, int S, int64_t split_stride, const float* bias,
                    const float* gamma, const float* beta, float* h_out, int64_t ld_h,
                    float* xhat, float* rstd, uint16_t* h_bf16, int64_t rpad_hb, int B, int F, float eps,
                    void* stream);

/* the same for several (network, row range) pairs in one launch - the five trunk forwards of an
 * update (drqv2.py:182-184,187,210,213) read only two feature matrices.  partial row stride is
 * ld_partial (the job's columns start at `partial`); the bf16 copy lands at TB rows row0_bf16 + b. */
#define DRQ_LN_MAX_JOBS 4
typedef struct {
    const float* partial; int64_t ld_partial; int64_t split_stride; int32_t S;
    const float* bias; const float* gamma; const float* beta;
    float* h_out; int64_t ld_h; float* xhat; float* rstd;
    uint16_t* h_bf16; int64_t units_bf16; int64_t row0_bf16;
    const float* tail; int64_t ld_tail; int32_t n_tail;   /* nullable: tail[b][0..n_tail) is appended at feature F of the bf16 row
                                                             (the action of torch.cat([h, action]), drqv2.py:117);
                                                             F + n_tail <= 8 * units_bf16 */
} drq_ln_job;
int drq_ln_tanh_fwd_multi(const drq_ln_job* jobs, int njobs, int B, int F, float eps, void* stream);

/* dh may arrive as n_planes partial planes (plane_stride floats apart) that are summed on the fly - the
 * per-head / split-K partial products of the Q heads' first-layer data gradient.
 * backward of tanh∘LayerNorm: dh (ld_dh) -> dz (gradient w.r.t. the Linear
 * output), dgamma[F], dbeta[F].  h is the saved tanh output (ld_h).
 * dz must hold 2*B*F floats: [0,B*F) receives dz, [B*F,2*B*F) receives dy = dh * tanh'.
 * dgamma == NULL: only the row kernel runs; dgamma = colsum(dy * xhat) and dbeta = colsum(dy) are then left to
 * drq_colsum_multi. */
int drq_ln_tanh_bwd(const float* dh, int64_t ld_dh, const float* h, int64_t ld_h,
                    const float* xhat, const float* rstd, const float* gamma, float* dz,
                    float* dgamma, float* dbeta, uint16_t* dz_bf16, int64_t rpad_zb, int B, int F,
                    int n_planes, int64_t plane_stride, void* stream);

/* ------------------------------------------------------------------ heads */

/* Actor tail (drqv2.py:88-92 + utils.py:112-126): mu = tanh(mu_pre);
 * e = eps*std; if clip > 0: e = clamp(e,-clip,clip); a = clamp(mu+e, -1+1e-6, 1-1e-6).
 * std is read from the device scalar *std_dev.  eps == NULL -> a = mu (eval
 * mode mean).  Writes a at action_out[b*ld_a + j] and mu at mu_out (nullable).
 * metrics (nullable) [2]: mean_b sum_j log_prob, mean_b sum_j entropy
 * (drqv2.py:212,226). */
int drq_actor_sample(const float* mu_pre, const float* eps, const float* std_dev, float clip,
                     float* action_out, int64_t ld_a, float* mu_out, float* metrics, int B, int A, void* stream);

/* Policy head of the tensor-core mode in one launch (drqv2.py:81,88-92 + utils.py:112-126): mu_pre[m][a] =
 * p2[m][:] . bf16(w4[a][:]) + b4[a] for the M rows of the TB activation p2 (units per row), and - by the thread that
 * holds each value - drq_actor_sample's arithmetic on up to DRQ_POLICY_MAX_JOBS row ranges.  1 <= A <= DRQ_POLICY_MAX_A,
 * H % 8 == 0; the actions are split into ceil(A / 32) balanced groups, and one group's ceil(A / groups) x H fp32 weights
 * must fit a block's opt-in shared memory (128 KB at A = 32 or 128, H = 1024).  At most one job carries metrics (it
 * needs eps); `scratch` then is 1 + ceil(M / 8) * ceil(A / 32) (at most 1 + DRQ_POLICY_MAX_PARTIALS) zero-initialised
 * 32-bit words (block ticket + per-block log-prob sums) that the kernel leaves zeroed.  Replaces a 128 x 64 tensor-core
 * tile that was > 75 % padding (A <= 32 outputs) followed by one or two sampling launches. */
#define DRQ_POLICY_MAX_JOBS 2
#define DRQ_POLICY_MAX_A 128
#define DRQ_POLICY_MAX_PARTIALS 16384   /* M <= 32768 at every A <= 128 */
typedef struct { int32_t row0; int32_t rows; const float* eps; float* action_out; int64_t ld_a; float* mu_out;
                 float* metrics; uint16_t* a_bf16; int64_t units_a; int32_t feat_off; int32_t reserved; } drq_policy_sample;
int drq_policy_head_fwd_bf16(const uint16_t* p2, int64_t units, const float* w4, const float* b4, float* mu_pre, int M,
                             int H, int A, const drq_policy_sample* jobs, int njobs, const float* std_dev, float clip,
                             uint32_t* scratch, void* stream);

/* d(mu_pre) = d(action) * (1 - mu^2)   (straight-through clamp, utils.py:113-116) */
int drq_actor_sample_bwd(const float* daction, int64_t ld_da, const float* mu, float* dmu_pre,
                         uint16_t* dmu_bf16, int64_t rpad_mb, int B, int A, int n_planes, int64_t plane_stride,
                         void* stream);

/* TD target + critic loss (drqv2.py:185-189): tq = r + d*min(tq1,tq2);
 * loss = mean((q1-tq)^2) + mean((q2-tq)^2); dq1 = 2(q1-tq)/B, dq2 likewise.
 * metrics [5]: batch_reward, critic_target_q, critic_q1, critic_q2, critic_loss
 * (drqv2.py:192-195,249).  target_q_out nullable [B]. */
int drq_critic_loss(const float* q1, const float* q2, const float* tq1, const float* tq2,
                    const float* reward, const float* discount, float* dq1, float* dq2,
                    float* target_q_out, float* metrics, int B, void* stream);

/* actor loss (drqv2.py:213-216): L = -mean(min(q1,q2)); dq1/dq2 = -1/B on the
 * smaller head (split evenly on exact ties, as torch.minimum's backward).
 * metrics [1]: actor_loss. */
int drq_actor_loss(const float* q1, const float* q2, float* dq1, float* dq2, float* metrics,
                   int B, void* stream);

/* dst[r*ld_dst + c] = src[r*ld_src + c]  (the `torch.cat([h, action])` of drqv2.py:117) */
int drq_copy2d_f32(const float* src, int64_t ld_src, float* dst, int64_t ld_dst, int rows, int cols,
                   void* stream);

/* bf16-mode helpers of the heads (TB activation layout; every `rpad` argument = units per row) */
/* final Linear(hidden,1) of the Q heads (drqv2.py:106,111) on an FB hidden activation c2 (head z at
 * c2 + z*bs_c2): q[z][b] = c2[z][b].w3[z] + b3[z]; w3/b3 of head z at w3 + z*w_stride / b3 + z*w_stride. */
int drq_q_head_fwd_bf16(const uint16_t* c2, int64_t rpad, int64_t bs_c2, const float* w3, const float* b3,
                        float* q, int B, int H, int heads, int64_t w_stride, int heads_inner, int64_t w_stride_outer,
                        void* stream);
/* its backward, with the loss gradient computed in place: dc2 = dq w3 (c2 > 0) as TB bf16, dw3 / db3 (nullable) in
 * fp32 at the same strides, where dq comes from loss = 1: critic loss of
 * drqv2.py:185-189 from q[2][B], tq[2][B], reward, discount (metrics[0..4] and target_q_out as drq_critic_loss);
 * loss = 2: actor loss of drqv2.py:213-216 from q[2][B] (metrics[0] = actor_loss).  Two heads. */
int drq_q_head_bwd_loss_bf16(int loss, const float* q, const float* tq, const float* reward, const float* discount,
                             float* target_q_out, float* metrics, const uint16_t* c2, int64_t rpad, int64_t bs_c2,
                             const float* w3, uint16_t* dc2, float* dw3, float* db3, int B, int H, int64_t w_stride,
                             void* stream);

/* drq_q_head_bwd_loss_bf16's backward from given upstream gradients (the autograd Critic of differentiable="bf16",
 * drqv2.py:115-121): dq1 / dq2 [B] fp32, each nullable - a null one skips its head, whose outputs are then left alone.
 * Head z (0 = Q1, 1 = Q2) reads c2 + z*bs_c2 and w3 + z*w_stride and writes dc2 + z*bs_c2 = RN-bf16(dq w3 (c2 > 0))
 * at rows < B of its TB activation (rpad = units per row; features < H), and (each nullable) dw3 + z*w_stride [H]
 * = sum_b dq c2, db3 + z*w_stride = sum_b dq - the sums of the loss modes, in the same fixed order. */
int drq_q_head_bwd_bf16(const float* dq1, const float* dq2, const uint16_t* c2, int64_t rpad, int64_t bs_c2,
                        const float* w3, uint16_t* dc2, float* dw3, float* db3, int B, int H, int64_t w_stride,
                        void* stream);

/* ------------------------------------------------------------------ autograd module boundary, bf16 tensor cores */

/* Rows a feature conversion takes: one grid row per feature row, the same bound drq_pack_features_tb's grid has
 * (511 blocks of DRQ_TB_ACT rows). */
#define DRQ_FEATURE_MAX_ROWS 65408

/* Features back to the reference's flatten order (drqv2.py:66): out [rows][39200] fp32, column c*1225 + y*35 + x,
 * from src in the encoder-output order (c/8)*9800 + (y*35+x)*8 + c%8 - src_tb != 0: TB(DRQ_TB_ACT) bf16 rows (conv4's
 * feature operand; `src` at a 128-row block boundary), exact; src_tb == 0: fp32 [rows][39200] (the trunk's data
 * gradient from drq_gemm_bf16 KMN / DRQ_TEPI_F32, ldc = 39200).  Writes exactly out[0 .. rows*39200).  The inverse
 * of drq_pack_features_tb on bf16-representable rows. */
int drq_features_to_ref(const void* src, int src_tb, float* out, int rows, void* stream);

/* The bf16 twin of drq_feature_grad_wide_f32: conv4's pre-ReLU gradient as the WB buffer of N images
 * (drq_wb_elems(N) bf16) from an arbitrary gradient of the features.  dfeat and feat are compact fp32 [N][39200] in
 * the reference order (feat = conv4's post-ReLU output, the mask).  dpre = RN-bf16(feat > 0 ? dfeat : +0) at the
 * 35 x 35 pixels of every image and +0 at every other element of the buffer (guard rows, rows 35-40, columns 35-40,
 * slack): every element of the N-image buffer is written, so that the zeros drq_conv3x3_dgrad_bf16 and
 * drq_conv3x3_wgrad_bf16 require hold whatever the buffer held before. */
int drq_feature_grad_wide_bf16(const float* dfeat, const float* feat, uint16_t* dpre, int N, void* stream);

/* out[r*ld_out + c] = 0 + sum over s = 0, 1, .. n_planes-1 (in that order) of planes[s*plane_stride + r*ld + c], for
 * r < rows, c < cols; writes exactly those elements.  The critic's action gradient: the split-K / per-head planes of
 * its first layer's data gradient at the action columns (planes + F), summed in the order drq_ln_tanh_bwd and
 * drq_actor_sample_bwd sum the same planes. */
int drq_plane_sum_f32(const float* planes, int64_t ld, int64_t plane_stride, int n_planes, float* out, int64_t ld_out,
                      int rows, int cols, void* stream);

/* ------------------------------------------------------------------ optimiser */

/* scalars (device, float[8]): [0] 1-beta1, [1] beta2, [2] 1-beta2,
 * [3] sqrt(1-beta2^t), [4] eps, [5] -lr/(1-beta1^t)  — computed on the host in
 * float64 exactly as torch/optim/adam.py:531-547 and cast to fp32.
 * One launch updates the contiguous range p[0..n): torch.optim.Adam x3 of
 * drqv2.py:148-150,201-202,221 over the flat parameter arena. */
int drq_adam_step(float* p, const float* g, float* m, float* v, int64_t n, const float* scalars,
                  void* stream);

/* The producer of those scalars on the device (DrQV2Agent(capturable=True)): one thread, stream-ordered and
 * capturable, so that every replay of a captured optimiser step advances its own step count.  t = ++*step, then
 * scalars[0..8) = utils.adam_scalars(lr, t, beta1, beta2, eps): [0] 1-beta1, [1] beta2, [2] 1-beta2,
 * [3] pow(1-pow(beta2,t), 0.5), [4] eps, [5] -(lr/(1-pow(beta1,t))), each computed in fp64 and rounded once to fp32,
 * [6] = [7] = 0.  Writes *step and those 8 floats, nothing else.  Equal to the host's values bit for bit at every t
 * in 1..4096 and at 1000 t up to 10^7 on a B200 (tests/test_gpu_capture.py), although CUDA's fp64 pow and glibc's need not
 * agree in the last fp64 place. */
int drq_adam_scalars_advance(int64_t* step, double lr, double beta1, double beta2, double eps, float* scalars,
                             void* stream);

/* soft target update (utils.py:42-45): tp = tau*p + (1-tau)*tp, two rounded
 * multiplies then an add (bit-exact). */
int drq_soft_update(const float* p, float* tp, int64_t n, float tau, float one_minus_tau,
                    void* stream);

/* fused: Adam over p[0..n_adam) and soft update of target from src[0..n_ema)
 * in one launch (K17+K18 of SURVEY §2.1). */
int drq_adam_ema_step(float* p, const float* g, float* m, float* v, int64_t n_adam,
                      const float* scalars, const float* ema_src, float* ema_dst, int64_t n_ema,
                      float tau, float one_minus_tau, void* stream);

/* Optimiser step and bf16 operand refresh in one launch (bf16 mode): every tensor of an optimiser phase is a
 * segment; the kernel applies Adam (ema == 0: p/g/m/v[off .. off+n)) or the soft target update (ema == 1:
 * ema_dst[off ..] = tau*ema_src[off ..] + (1-tau)*ema_dst[off ..]) and writes the bf16 copy the tensor-core
 * kernels read straight from the updated value - what drq_adam_ema_step followed by drq_pack_multi produce,
 * bit for bit, without reading the fp32 parameters a second time.
 *   DRQ_OPT_PLAIN : no bf16 copy (biases, LayerNorm, the scalar Q heads)
 *   DRQ_OPT_LINEAR: nn.Linear weight [rows][cols]            -> out as drq_pack_linear_tb
 *   DRQ_OPT_TRUNK : trunk weight [rows][32*35*35]            -> out as drq_pack_trunk_tb
 *   DRQ_OPT_CONV  : conv weight [32][32][3][3] (n = 9216)    -> out (fwd), out2 (dgrad) as drq_pack_conv_w_bf16
 *   DRQ_OPT_CONV1 : conv1 weight [32][rows=cin][3][3] and its bias, adjacent (n = 288*cin + 32)
 *                                                            -> out as drq_pack_conv1_w_bf16 */
#define DRQ_OPT_PLAIN 0
#define DRQ_OPT_LINEAR 1
#define DRQ_OPT_TRUNK 2
#define DRQ_OPT_CONV 3
#define DRQ_OPT_CONV1 4
#define DRQ_OPT_MAX_SEGS 32
typedef struct { int32_t kind; int32_t ema; int32_t rows; int32_t cols; int64_t off; int64_t n;
                 uint16_t* out; uint16_t* out2; } drq_opt_seg;
int drq_adam_pack_step(float* p, const float* g, float* m, float* v, const float* scalars,
                       const float* ema_src, float* ema_dst, float tau, float one_minus_tau,
                       const drq_opt_seg* segs, int nsegs, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DRQV2_B200_H */

// GPU-resident replay ring: n-step gather, device-side sampler, per-update RNG draws.
// Reference arithmetic: replay_buffer.py:142-160 (sample), dmc.py:86-109 (frame stack).
#include <stdarg.h>
#include <stdio.h>

#include "common.cuh"

namespace drq {

static thread_local char g_err[512] = "";
int g_sm_limit = 148;

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

void* tensor_map_encoder() {
    static void* fn = nullptr;
    if (!fn) {
        cudaDriverEntryPointQueryResult q;
        void* p = nullptr;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess) fn = p;
    }
    return fn;
}

int check_launch(const char* what) {
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        set_error("%s: %s", what, cudaGetErrorString(e));
        return DRQ_ERR_CUDA;
    }
    return DRQ_OK;
}

int ensure_smem(const void* kernel, size_t bytes, const char* what) {
    // the opt-in is a per-device function attribute: the cache is keyed by (device, kernel)
    constexpr int kMax = 512;
    static const void* seen_fn[kMax];
    static size_t seen_bytes[kMax];
    static int seen_dev[kMax];
    static int n_seen = 0;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) { cudaGetLastError(); dev = 0; }
    for (int i = 0; i < n_seen; ++i)
        if (seen_fn[i] == kernel && seen_dev[i] == dev && seen_bytes[i] >= bytes) return DRQ_OK;
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (e != cudaSuccess) {
        set_error("%s: cudaFuncSetAttribute(%zu): %s", what, bytes, cudaGetErrorString(e));
        return DRQ_ERR_CUDA;
    }
    int slot = -1;
    for (int i = 0; i < n_seen; ++i)
        if (seen_fn[i] == kernel && seen_dev[i] == dev) slot = i;
    if (slot < 0 && n_seen < kMax) slot = n_seen++;
    if (slot >= 0) { seen_fn[slot] = kernel; seen_bytes[slot] = bytes; seen_dev[slot] = dev; }
    return DRQ_OK;
}

// grid (B, 2*stack + 1).  y < 2*stack: copy one frame of obs / next_obs with 16-byte
// vectors; y == 2*stack: action copy + the un-fused fp32 n-step chain.
__global__ void __launch_bounds__(256)
ring_gather_kernel(const uint8_t* __restrict__ frames, const float* __restrict__ action,
                   const float* __restrict__ reward, const float* __restrict__ discount,
                   long long capacity, int frame_bytes, int stack, int A,
                   const int* __restrict__ ep_start, const int* __restrict__ idx, int nstep,
                   float gamma, uint8_t* __restrict__ obs_out, uint8_t* __restrict__ next_out,
                   float* __restrict__ action_out, float* __restrict__ reward_out,
                   float* __restrict__ discount_out) {
    const int b = blockIdx.x;
    const int y = blockIdx.y;
    const long long start = ep_start[b];
    const int row = idx[b];
    if (y < 2 * stack) {
        const bool is_next = y >= stack;
        const int j = is_next ? y - stack : y;
        const int t = is_next ? row + nstep - 1 : row - 1;  // replay_buffer.py:151,153
        int r = t - (stack - 1 - j);                        // dmc.py:98-109: deque of last `stack` frames
        r = r < 0 ? 0 : r;                                  // reset repeats the first frame
        const long long slot = (start + r) % capacity;
        const int4* src = reinterpret_cast<const int4*>(frames + slot * (long long)frame_bytes);
        uint8_t* dst_base = (is_next ? next_out : obs_out) +
                            ((long long)b * stack + j) * (long long)frame_bytes;
        int4* dst = reinterpret_cast<int4*>(dst_base);
        const int nvec = frame_bytes >> 4;
        for (int i = threadIdx.x; i < nvec; i += blockDim.x) dst[i] = __ldg(src + i);
        // tail (frame_bytes % 16 != 0 never happens for 3x84x84 but stay general)
        for (int i = (nvec << 4) + threadIdx.x; i < frame_bytes; i += blockDim.x)
            dst_base[i] = frames[slot * (long long)frame_bytes + i];
    } else {
        const long long s0 = (start + row) % capacity;
        for (int a = threadIdx.x; a < A; a += blockDim.x)
            action_out[(long long)b * A + a] = action[s0 * A + a];  // replay_buffer.py:152
        if (threadIdx.x == 0) {
            float rew = 0.f, disc = 1.f;  // replay_buffer.py:154-155
            for (int i = 0; i < nstep; ++i) {
                const long long s = (start + row + i) % capacity;
                rew = __fadd_rn(rew, __fmul_rn(disc, reward[s]));             // :158
                disc = __fmul_rn(disc, __fmul_rn(discount[s], gamma));        // :159
            }
            reward_out[b] = rew;
            discount_out[b] = disc;
        }
    }
}

__device__ __forceinline__ void ring_sample_elem(const int* __restrict__ ep_table, int E, int nstep, unsigned long long seed,
                                                 unsigned long long c, int* __restrict__ ep_start_out, int* __restrict__ idx_out, int b) {
    uint32_t r[4];
    Philox::gen(seed, (c << 3) | 0ull, (uint64_t)b, r);
    // unbiased enough for E, len << 2^32: multiply-shift range reduction
    const int e = (int)(((uint64_t)r[0] * (uint64_t)E) >> 32);
    const int start = ep_table[2 * e], len = ep_table[2 * e + 1];
    const int span = len - nstep + 1;  // np.random.randint(0, len - nstep + 1) + 1
    const int i = (int)(((uint64_t)r[1] * (uint64_t)span) >> 32) + 1;
    ep_start_out[b] = start;
    idx_out[b] = i;
}

__global__ void ring_sample_kernel(const int* __restrict__ ep_table, const int* __restrict__ n_episodes, int nstep,
                                   unsigned long long seed, const unsigned long long* counter,
                                   int* __restrict__ ep_start_out, int* __restrict__ idx_out, int B) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    ring_sample_elem(ep_table, *n_episodes, nstep, seed, *counter, ep_start_out, idx_out, b);
}

// the same draw followed by counter += 1: one block, so that the increment can follow every read
__global__ void __launch_bounds__(256) ring_sample_step_kernel(const int* __restrict__ ep_table, const int* __restrict__ n_episodes,
                                                               int nstep, unsigned long long seed, unsigned long long* counter,
                                                               int* __restrict__ ep_start_out, int* __restrict__ idx_out, int B) {
    const unsigned long long c = *counter;
    const int E = *n_episodes;
    for (int b = threadIdx.x; b < B; b += blockDim.x) ring_sample_elem(ep_table, E, nstep, seed, c, ep_start_out, idx_out, b);
    __syncthreads();
    if (threadIdx.x == 0) *counter = c + 1ull;
}

// stream ids: 1 shift_obs, 2 shift_next, 3 eps_critic, 4 eps_actor
__device__ __forceinline__ float box_muller(uint32_t a, uint32_t b, bool odd) {
    const float u1 = ((float)(a >> 8) + 0.5f) * (1.0f / 16777216.0f);
    const float u2 = ((float)(b >> 8) + 0.5f) * (1.0f / 16777216.0f);
    const float rad = sqrtf(-2.0f * logf(u1));
    float s, co;
    sincospif(2.0f * u2, &s, &co);
    return odd ? rad * s : rad * co;
}

__device__ __forceinline__ void update_draws_elem(unsigned long long seed, unsigned long long c, int pad, int* __restrict__ shift_obs,
                                                  int* __restrict__ shift_next, float* __restrict__ eps_c,
                                                  float* __restrict__ eps_a, int B, int A, int i) {
    const unsigned range = 2 * pad + 1;
    if (shift_obs && i < B) {
        uint32_t r[4];
        Philox::gen(seed, (c << 3) | 1ull, (uint64_t)i, r);
        shift_obs[2 * i] = (int)(((uint64_t)r[0] * range) >> 32);
        shift_obs[2 * i + 1] = (int)(((uint64_t)r[1] * range) >> 32);
        shift_next[2 * i] = (int)(((uint64_t)r[2] * range) >> 32);
        shift_next[2 * i + 1] = (int)(((uint64_t)r[3] * range) >> 32);
    }
    // Box-Muller: 4 words -> 2 pairs -> 4 normals; element i uses pair (i>>1) of stream 3/4.
    if (eps_c && i < B * A) {
        uint32_t r[4];
        Philox::gen(seed, (c << 3) | 3ull, (uint64_t)(i >> 1), r);
        eps_c[i] = box_muller(r[0], r[1], i & 1);
        eps_a[i] = box_muller(r[2], r[3], i & 1);
    }
}

__global__ void rng_update_draws_kernel(unsigned long long seed, const unsigned long long* counter,
                                        int pad, int* __restrict__ shift_obs,
                                        int* __restrict__ shift_next, float* __restrict__ eps_c,
                                        float* __restrict__ eps_a, int B, int A) {
    update_draws_elem(seed, *counter, pad, shift_obs, shift_next, eps_c, eps_a, B, A, blockIdx.x * blockDim.x + threadIdx.x);
}

// Everything an update needs before its first real kernel, in one block: the per-update host scalars
// (scalars_fetch_kernel), the four random draws (rng_update_draws_kernel) and counter += 1.
__global__ void __launch_bounds__(1024) update_prologue_kernel(const float* scal_ring, int slots, unsigned long long* cursor,
                                                               float* scal_out, unsigned long long seed, unsigned long long* counter,
                                                               int pad, int* __restrict__ shift_obs, int* __restrict__ shift_next,
                                                               float* __restrict__ eps_c, float* __restrict__ eps_a, int B, int A) {
    if (threadIdx.x < DRQ_SCAL_SLOT) {
        const unsigned long long cur = *cursor;
        scal_out[threadIdx.x] = *reinterpret_cast<const volatile float*>(scal_ring + (cur % (unsigned long long)slots) * DRQ_SCAL_SLOT + threadIdx.x);
        __syncwarp();
        if (threadIdx.x == 0) *cursor = cur + 1ull;
    }
    if (shift_obs) {
        const unsigned long long c = *counter;
        const int n = B * A > B ? B * A : B;
        for (int i = threadIdx.x; i < n; i += blockDim.x) update_draws_elem(seed, c, pad, shift_obs, shift_next, eps_c, eps_a, B, A, i);
        __syncthreads();
        if (threadIdx.x == 0) *counter = c + 1ull;
    }
}

// The head of a ring-fed update in one block: update_prologue_kernel, then ring_sample_step_kernel, then the scalar
// part of ring_gather_kernel (action copy + un-fused fp32 n-step chain) on the indices just drawn.  The frame stacks
// stay in the ring (conv1_tc_kernel's row producer reads them through ep_start / idx).
// `part`: 3 = everything; 1 = only what the encoder's first kernel waits for (the two shift draws, the replay sample);
// 2 = the rest (host scalars, the two noise draws, n-step reward / discount, action copy), launched after part 1 on a side
// stream (drq_update_prologue_ring_part).  Same values either way: every draw is a function of (seed, counter, element).
__global__ void __launch_bounds__(1024) update_prologue_ring_kernel(const float* scal_ring, int slots, unsigned long long* cursor,
                                                                    float* scal_out, unsigned long long seed, unsigned long long* counter,
                                                                    int pad, int* __restrict__ shift_obs, int* __restrict__ shift_next,
                                                                    float* __restrict__ eps_c, float* __restrict__ eps_a, int B, int A,
                                                                    const drq_ring_src src, float* __restrict__ action_out,
                                                                    float* __restrict__ reward_out, float* __restrict__ discount_out,
                                                                    int part) {
    const bool head = part & 1, rest = part & 2;
    if (rest && threadIdx.x < DRQ_SCAL_SLOT) {
        const unsigned long long cur = *cursor;
        scal_out[threadIdx.x] = *reinterpret_cast<const volatile float*>(scal_ring + (cur % (unsigned long long)slots) * DRQ_SCAL_SLOT + threadIdx.x);
        __syncwarp();
        if (threadIdx.x == 0) *cursor = cur + 1ull;
    }
    unsigned long long c = 0;
    if (shift_obs) {
        c = *counter;
        // update_draws_elem writes the shifts of element i < B and the noise of element i < B * A
        const int n = rest ? (B * A > B ? B * A : B) : B;
        for (int i = threadIdx.x; i < n; i += blockDim.x)
            update_draws_elem(seed, c, pad, head ? shift_obs : nullptr, shift_next, rest ? eps_c : nullptr, eps_a, B, A, i);
    }
    unsigned long long cs = 0;
    if (head) {
        cs = *src.counter;
        const int E = *src.n_episodes;
        for (int b = threadIdx.x; b < B; b += blockDim.x) ring_sample_elem(src.ep_table, E, src.nstep, src.seed, cs, src.ep_start, src.idx, b);
    }
    __syncthreads();                                  // indices visible to the block; every counter read is done
    if (threadIdx.x == 0) {
        if (shift_obs && rest) *counter = c + 1ull;   // (part 1 reads the counter part 2 advances)
        if (head) *src.counter = cs + 1ull;
    }
    if (!rest) return;
    for (int b = threadIdx.x; b < B; b += blockDim.x) {
        const long long start = src.ep_start[b];
        const int row = src.idx[b];
        float rew = 0.f, disc = 1.f;                  // replay_buffer.py:154-159
        for (int i = 0; i < src.nstep; ++i) {
            const long long sl = (start + row + i) % src.capacity;
            rew = __fadd_rn(rew, __fmul_rn(disc, src.reward[sl]));
            disc = __fmul_rn(disc, __fmul_rn(src.discount[sl], src.gamma));
        }
        reward_out[b] = rew;
        discount_out[b] = disc;
    }
    for (int i = threadIdx.x; i < B * A; i += blockDim.x) {
        const int b = i / A, a = i - b * A;
        const long long s0 = ((long long)src.ep_start[b] + src.idx[b]) % src.capacity;
        action_out[i] = src.action[s0 * A + a];       // replay_buffer.py:152
    }
}

// out[i] ~ N(0,1): stream 5, Box-Muller on pair (i >> 1)
__global__ void rng_normal_kernel(unsigned long long seed, const unsigned long long* counter,
                                  float* __restrict__ out, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t r[4];
    Philox::gen(seed, (*counter << 3) | 5ull, (uint64_t)(i >> 1), r);
    const float u1 = ((float)(r[0] >> 8) + 0.5f) * (1.0f / 16777216.0f);
    const float u2 = ((float)(r[1] >> 8) + 0.5f) * (1.0f / 16777216.0f);
    const float rad = sqrtf(-2.0f * logf(u1));
    float s, co;
    sincospif(2.0f * u2, &s, &co);
    out[i] = (i & 1) ? rad * s : rad * co;
}

__global__ void counter_advance_kernel(unsigned long long* counter) { *counter += 1ull; }

// out[0..DRQ_SCAL_SLOT) = ring[cursor % slots][..]; cursor += 1.  The ring is pinned host memory the host fills one
// update ahead of the device: a CUDA graph cannot take new scalars per replay, and a fixed staging buffer
// would be overwritten by a host that enqueues updates faster than the device runs them.
__global__ void scalars_fetch_kernel(const float* ring, int slots, unsigned long long* cursor, float* out) {
    const unsigned long long c = *cursor;
    const float v = *reinterpret_cast<const volatile float*>(ring + (c % (unsigned long long)slots) * DRQ_SCAL_SLOT + threadIdx.x);
    out[threadIdx.x] = v;
    __syncwarp();
    if (threadIdx.x == 0) *cursor = c + 1ull;
}

// out[n,c,r,col] = in[n,c,clamp(r+sy-pad),clamp(col+sx-pad)]
__global__ void random_shift_f32_kernel(const float* __restrict__ in, const int* __restrict__ shift,
                                        float* __restrict__ out, int C, int H, int W, int pad) {
    const int n = blockIdx.y;
    const int sx = shift[2 * n], sy = shift[2 * n + 1];
    const long long per = (long long)C * H * W;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < per;
         i += (long long)gridDim.x * blockDim.x) {
        const int col = (int)(i % W);
        const int r = (int)((i / W) % H);
        const int c = (int)(i / ((long long)W * H));
        const int sr = clampi(r + sy - pad, 0, H - 1), sc = clampi(col + sx - pad, 0, W - 1);
        out[n * per + i] = in[n * per + ((long long)c * H + sr) * W + sc];
    }
}

// its transpose: dx[n,c,i,j] = sum of dout[n,c,r,col] over every (r, col) whose clamped source is (i, j), in ascending
// (r, col) order.  Separable: the rows are r = i - dy (dy = sy - pad) in the interior, r <= -dy at i = 0 and
// r >= H-1-dy at i = H-1, each range cut to [0, H); the columns likewise.  An empty range gives +0.
// Grid: (pixel blocks of a plane, N * C planes); consecutive threads take consecutive columns, whose sources are
// consecutive too away from the clamped edges.
__global__ void random_shift_bwd_f32_kernel(const float* __restrict__ dout, const int* __restrict__ shift,
                                            float* __restrict__ dx, int planes, int C, int H, int W, int pad) {
  for (int plane = blockIdx.y; plane < planes; plane += gridDim.y) {
    const int n = plane / C;
    const int dxs = __ldg(shift + 2 * n) - pad, dys = __ldg(shift + 2 * n + 1) - pad;
    const int hw = H * W;
    const float* src = dout + (long long)plane * hw;
    float* dst = dx + (long long)plane * hw;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < hw; i += gridDim.x * blockDim.x) {
        const int r = i / W, col = i - r * W;
        const int rlo = max(r == 0 ? 0 : r - dys, 0), rhi = min(r == H - 1 ? H - 1 : r - dys, H - 1);
        const int clo = max(col == 0 ? 0 : col - dxs, 0), chi = min(col == W - 1 ? W - 1 : col - dxs, W - 1);
        float acc = 0.f;
        for (int rr = rlo; rr <= rhi; ++rr)
            for (int cc = clo; cc <= chi; ++cc) acc += __ldg(src + rr * W + cc);
        dst[i] = acc;
    }
  }
}

__global__ void copy2d_kernel(const float* __restrict__ src, long long ld_src, float* __restrict__ dst,
                              long long ld_dst, int rows, int cols) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= rows * cols) return;
    const int r = i / cols, c = i - r * cols;
    dst[r * ld_dst + c] = src[r * ld_src + c];
}

}  // namespace drq

using namespace drq;

extern "C" {

int drq_set_sm_limit(int sms) {
    DRQ_REQUIRE(sms >= 1 && sms <= 148, "set_sm_limit: 1..148");
    drq::g_sm_limit = sms;
    return DRQ_OK;
}

int drq_abi_version(void) { return DRQ_ABI_VERSION; }
const char* drq_last_error(void) { return drq::g_err; }

int drq_device_sm_count(void) {
    int dev = 0, n = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) { cudaGetLastError(); return 0; }
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n < drq::g_sm_limit ? n : drq::g_sm_limit;
}

int drq_ring_gather_nstep(const uint8_t* frames, const float* action, const float* reward,
                          const float* discount, int64_t capacity, int frame_c, int stack, int A,
                          const int32_t* ep_start, const int32_t* idx, int B, int nstep, float gamma,
                          uint8_t* obs_out, uint8_t* next_obs_out, float* action_out,
                          float* reward_out, float* discount_out, void* stream) {
    DRQ_REQUIRE(frames && action && reward && discount && ep_start && idx, "ring_gather: null input");
    DRQ_REQUIRE(obs_out && next_obs_out && action_out && reward_out && discount_out,
                "ring_gather: null output");
    DRQ_REQUIRE(capacity > 0 && frame_c > 0 && stack > 0 && A > 0 && nstep > 0, "ring_gather: bad dims");
    if (B == 0) return DRQ_OK;
    DRQ_REQUIRE(B > 0, "ring_gather: negative batch");
    const int frame_bytes = frame_c * kImg * kImg;
    DRQ_REQUIRE(frame_bytes % 16 == 0 && ((uintptr_t)frames % 16) == 0 &&
                    ((uintptr_t)obs_out % 16) == 0 && ((uintptr_t)next_obs_out % 16) == 0,
                "ring_gather: frames must be 16-byte aligned");
    dim3 grid(B, 2 * stack + 1);
    ring_gather_kernel<<<grid, 256, 0, as_stream(stream)>>>(
        frames, action, reward, discount, (long long)capacity, frame_bytes, stack, A, ep_start, idx,
        nstep, gamma, obs_out, next_obs_out, action_out, reward_out, discount_out);
    return check_launch("ring_gather_kernel");
}

int drq_ring_sample(const int32_t* ep_table, const int32_t* n_episodes, int nstep, uint64_t seed,
                    const uint64_t* counter, int32_t* ep_start_out, int32_t* idx_out, int B, void* stream) {
    DRQ_REQUIRE(ep_table && n_episodes && counter && ep_start_out && idx_out, "ring_sample: null pointer");
    DRQ_REQUIRE(nstep > 0 && B > 0, "ring_sample: bad dims");
    ring_sample_kernel<<<(B + 127) / 128, 128, 0, as_stream(stream)>>>(
        ep_table, n_episodes, nstep, (unsigned long long)seed, (const unsigned long long*)counter,
        ep_start_out, idx_out, B);
    return check_launch("ring_sample_kernel");
}

int drq_rng_update_draws(uint64_t seed, const uint64_t* counter, int pad, int32_t* shift_obs,
                         int32_t* shift_next, float* eps_critic, float* eps_actor, int B, int A,
                         void* stream) {
    DRQ_REQUIRE(counter && shift_obs && shift_next && eps_critic && eps_actor, "rng: null pointer");
    DRQ_REQUIRE(B > 0 && A > 0 && pad >= 0, "rng: bad dims");
    const int n = B * A > B ? B * A : B;
    rng_update_draws_kernel<<<(n + 127) / 128, 128, 0, as_stream(stream)>>>(
        (unsigned long long)seed, (const unsigned long long*)counter, pad, shift_obs, shift_next,
        eps_critic, eps_actor, B, A);
    return check_launch("rng_update_draws_kernel");
}

int drq_copy2d_f32(const float* src, int64_t ld_src, float* dst, int64_t ld_dst, int rows, int cols,
                   void* stream) {
    DRQ_REQUIRE(src && dst && rows > 0 && cols > 0, "copy2d: bad args");
    copy2d_kernel<<<(rows * cols + 255) / 256, 256, 0, as_stream(stream)>>>(src, ld_src, dst, ld_dst, rows, cols);
    return check_launch("copy2d_kernel");
}

int drq_rng_normal_f32(uint64_t seed, const uint64_t* counter, float* out, int n, void* stream) {
    DRQ_REQUIRE(counter && out && n > 0, "rng_normal: bad args");
    rng_normal_kernel<<<(n + 127) / 128, 128, 0, as_stream(stream)>>>(
        (unsigned long long)seed, (const unsigned long long*)counter, out, n);
    return check_launch("rng_normal_kernel");
}

int drq_counter_advance(uint64_t* counter, void* stream) {
    DRQ_REQUIRE(counter, "counter_advance: null pointer");
    counter_advance_kernel<<<1, 1, 0, as_stream(stream)>>>((unsigned long long*)counter);
    return check_launch("counter_advance_kernel");
}

int drq_ring_sample_step(const int32_t* ep_table, const int32_t* n_episodes, int nstep, uint64_t seed, uint64_t* counter,
                         int32_t* ep_start_out, int32_t* idx_out, int B, void* stream) {
    DRQ_REQUIRE(ep_table && n_episodes && counter && ep_start_out && idx_out, "ring_sample_step: null pointer");
    DRQ_REQUIRE(B > 0 && nstep > 0, "ring_sample_step: bad dims");
    ring_sample_step_kernel<<<1, 256, 0, as_stream(stream)>>>(ep_table, n_episodes, nstep, (unsigned long long)seed,
             (unsigned long long*)counter, ep_start_out, idx_out, B);
    return check_launch("ring_sample_step_kernel");
}

int drq_update_prologue(const float* scal_ring, int slots, uint64_t* cursor, float* scal_out, uint64_t seed, uint64_t* counter,
                        int pad, int32_t* shift_obs, int32_t* shift_next, float* eps_critic, float* eps_actor, int B, int A,
                        void* stream) {
    DRQ_REQUIRE(scal_ring && cursor && scal_out && slots > 0, "update_prologue: bad scalar ring");
    const bool draws = shift_obs != nullptr;
    DRQ_REQUIRE(!draws || (counter && shift_next && eps_critic && eps_actor && B > 0 && A > 0 && pad >= 0), "update_prologue: bad draw arguments");
    update_prologue_kernel<<<1, 1024, 0, as_stream(stream)>>>(scal_ring, slots, (unsigned long long*)cursor, scal_out,
             (unsigned long long)seed, (unsigned long long*)counter, pad, shift_obs, shift_next, eps_critic, eps_actor, B, A);
    return check_launch("update_prologue_kernel");
}

int drq_update_prologue_ring_part(const float* scal_ring, int slots, uint64_t* cursor, float* scal_out, uint64_t seed,
                                  uint64_t* counter, int pad, int32_t* shift_obs, int32_t* shift_next, float* eps_critic,
                                  float* eps_actor, int B, int A, const drq_ring_src* src, float* action_out,
                                  float* reward_out, float* discount_out, int part, void* stream) {
    DRQ_REQUIRE(part >= 1 && part <= 3, "update_prologue_ring: part is 1 (shifts + sample), 2 (the rest) or 3 (both)");
    DRQ_REQUIRE(scal_ring && cursor && scal_out && slots > 0, "update_prologue_ring: bad scalar ring");
    DRQ_REQUIRE(!shift_obs || (counter && shift_next && eps_critic && eps_actor && pad >= 0), "update_prologue_ring: bad draw arguments");
    DRQ_REQUIRE(src && src->action && src->reward && src->discount && src->ep_table && src->n_episodes && src->counter &&
                    src->ep_start && src->idx, "update_prologue_ring: incomplete ring source");
    DRQ_REQUIRE(B > 0 && A > 0 && A == src->A && src->capacity > 0 && src->nstep > 0, "update_prologue_ring: bad dims");
    DRQ_REQUIRE(action_out && reward_out && discount_out, "update_prologue_ring: null output");
    update_prologue_ring_kernel<<<1, 1024, 0, as_stream(stream)>>>(scal_ring, slots, (unsigned long long*)cursor, scal_out,
             (unsigned long long)seed, (unsigned long long*)counter, pad, shift_obs, shift_next, eps_critic, eps_actor, B, A,
             *src, action_out, reward_out, discount_out, part);
    return check_launch("update_prologue_ring_kernel");
}

int drq_update_prologue_ring(const float* scal_ring, int slots, uint64_t* cursor, float* scal_out, uint64_t seed,
                             uint64_t* counter, int pad, int32_t* shift_obs, int32_t* shift_next, float* eps_critic,
                             float* eps_actor, int B, int A, const drq_ring_src* src, float* action_out,
                             float* reward_out, float* discount_out, void* stream) {
    return drq_update_prologue_ring_part(scal_ring, slots, cursor, scal_out, seed, counter, pad, shift_obs, shift_next, eps_critic,
                                         eps_actor, B, A, src, action_out, reward_out, discount_out, 3, stream);
}

int drq_scalars_fetch(const float* ring, int slots, uint64_t* cursor, float* out, void* stream) {
    DRQ_REQUIRE(ring && cursor && out && slots > 0, "scalars_fetch: bad arguments");
    scalars_fetch_kernel<<<1, DRQ_SCAL_SLOT, 0, as_stream(stream)>>>(ring, slots, (unsigned long long*)cursor, out);
    return check_launch("scalars_fetch_kernel");
}

int drq_random_shift_f32(const float* in, const int32_t* shift, float* out, int N, int C, int H,
                         int W, int pad, void* stream) {
    DRQ_REQUIRE(in && shift && out, "random_shift: null pointer");
    DRQ_REQUIRE(N >= 0 && C > 0 && H > 0 && W > 0 && pad >= 0, "random_shift: bad dims");
    DRQ_REQUIRE(H == W, "random_shift: h != w (drqv2.py:21)");
    if (N == 0) return DRQ_OK;
    const long long per = (long long)C * H * W;
    int gx = (int)((per + 255) / 256);
    if (gx > 64) gx = 64;
    random_shift_f32_kernel<<<dim3(gx, N), 256, 0, as_stream(stream)>>>(in, shift, out, C, H, W, pad);
    return check_launch("random_shift_f32_kernel");
}

int drq_random_shift_bwd_f32(const float* dout, const int32_t* shift, float* dx, int N, int C, int H, int W, int pad,
                             void* stream) {
    DRQ_REQUIRE(dout && shift && dx, "random_shift_bwd: null pointer");
    DRQ_REQUIRE(N >= 0 && C > 0 && H > 0 && W > 0 && pad >= 0, "random_shift_bwd: bad dims");
    DRQ_REQUIRE(H == W, "random_shift_bwd: h != w (drqv2.py:21)");
    DRQ_REQUIRE((long long)H * W < (1ll << 31) && (long long)N * C < (1ll << 31), "random_shift_bwd: too large");
    if (N == 0) return DRQ_OK;
    int gx = (H * W + 255) / 256;
    if (gx > 1024) gx = 1024;
    const int planes = N * C, gy = planes < 65535 ? planes : 65535;
    random_shift_bwd_f32_kernel<<<dim3(gx, gy), 256, 0, as_stream(stream)>>>(dout, shift, dx, planes, C, H, W, pad);
    return check_launch("random_shift_bwd_f32_kernel");
}

}  // extern "C"

namespace drq {
int trap_note_conv(unsigned int*); int trap_note_conv1(unsigned int*); int trap_note_conv4x1(unsigned int*); int trap_note_gemm(unsigned int*);
}
extern "C" int drq_debug_trap_note(uint32_t* mapped_host_words) {
    unsigned int* p = mapped_host_words;
    if (drq::trap_note_conv(p) | drq::trap_note_conv1(p) | drq::trap_note_conv4x1(p) | drq::trap_note_gemm(p)) {
        drq::set_error("drq_debug_trap_note: cudaMemcpyToSymbol failed");
        return DRQ_ERR_CUDA;
    }
    return DRQ_OK;
}

// conv1 of the encoder (drqv2.py:55: Cin->32, k3, stride 2) on tensor cores, with
// RandomShiftsAug (integer shift, drqv2.py:19-45) and obs/255-0.5 (drqv2.py:64) fused into
// the loader: builder warps gather the augmented 3x3xCin patch of every output position
// straight from the uint8 frame stack into an im2col tile in shared memory (canonical
// no-swizzle UMMA layout [K unit][position][16 B]); the augmented image never exists in HBM.
//
//   forward : out[p][co] = relu(b'[co] + (1/255) sum_k im2col[p][k] * W[co][k])   M=128 pos, N=32, K=96
//   wgrad   : S[co][k]   = sum_p d[p][co] * im2col[p][k]                          M=64(co), N=96, K=pos
//
// The im2col entries are the exact integers x - 128 in bf16 (|x - 128| <= 128 has at most 8 significant
// bits, so no rounding of the pixels): a byte permute with 0x4B000000 turns a uint8 into the float
// 2^23 + x, one subtract centres it, one cvt packs two of them.  The affine map x/255 - 0.5 = (x - 128)/255 + (128/255 - 0.5) moves to the epilogues:
//   forward : b'[co] = b[co] + (128/255 - 0.5) sum_k bf16(W[co][k])   (pack kernel), accumulator scaled by 1/255
//   wgrad   : dW[co][k] = S[co][k]/255 + (128/255 - 0.5) db[co],  db[co] = S[co][cin*9]
// K = cin*9 is padded to 96; slot k = cin*9 holds the constant 1.0 so that column cin*9 of the
// weight-gradient GEMM is the bias gradient (the forward weight there is zero).  (kind::f16 needs both
// operands in the same 16-bit format - mixing an fp16 im2col with the bf16 gradient tile traps - hence
// bf16 rather than the cheaper fp16 construction.)
//
// Loader: the (vertically clamped) source rows of a tile are staged per channel as replicate-padded
// rows [4 | 84 | 4] bytes, so the horizontal shift is an address offset and the three kx taps of one
// (channel, ky) are three consecutive bytes: two aligned 32-bit loads + a funnel shift per group of
// three K entries instead of a byte load and a table lookup per entry.
//
// Warp roles (704 threads): warps 0..15 re-pitch the rows + build im2col tiles (4 threads per output
// position), warp 16 issues UMMAs (and bulk-loads the gradient tile in wgrad), warps 17..20 run the
// epilogue, warp 21 bulk-copies the source rows of the next tiles (4 stages ahead).
#include <cuda.h>
#include <cuda_fp16.h>

#include "pack.cuh"
#include "wgrad_reduce.cuh"

namespace drq {

DRQ_TRAP_NOTE_HOOK(trap_note_conv1)

using namespace tc;

constexpr int kC1K = 96, kC1Units = kC1K / 8;
constexpr int kC1Tile = 128;
constexpr int kC1ABytes = kC1Units * kC1Tile * 16;     // 24576
constexpr int kC1Stages = 3;
constexpr int kC1WBytes = kC1Units * 32 * 16;          // weights [12][32][16 B] (+ 32 fused biases behind them)
constexpr int kC1Builders = 512;                        // 16 builder warps: 4 threads per output position
constexpr int kC1Threads = kC1Builders + 6 * 32;       // + UMMA warp, 4 epilogue warps, row producer warp
constexpr int kC1DBytes = 4 * kC1Tile * 16;            // wgrad: d tile [4 blocks][128][16 B]
constexpr int kC1Acc = 4;
constexpr float kC1Scale = 1.0f / 255.0f;
constexpr float kC1Shift = 128.0f / 255.0f - 0.5f;     // (x - 128)/255 + kC1Shift == x/255 - 0.5

struct Conv1TcArgs {
    const uint8_t* obs; const int* shift; int cin, pad;
    const __nv_bfloat16* w;       // fwd: packed bf16 [12][32][8], then float bias'[32]
    __nv_bfloat16* out; long long cs_out;          // fwd: WB output
    const __nv_bfloat16* d; long long cs_d;        // wgrad: WB gradient (N images)
    float* partial;                                // wgrad: [grid][32][96]
    int n_images;
    long long* stamps;                             // debug: builder cycle totals of block 0 (or null)
    // rows straight from the replay ring (ring_frames != null; obs unused): see drq_conv1_fwd_bf16_ring
    const uint8_t* ring_frames; const int* ring_ep_start; const int* ring_idx;
    long long ring_capacity; int ring_B, ring_nstep, ring_stack, ring_frame_c;
    const float* fobs;            // real-valued pixels [N][cin][84][84] (the *_from_f32 entry points; obs unused)
};

// first byte of channel `c` of image `n`: the gathered stack, or the ring frame the stack is made of
// (replay_buffer.py:151,153 rows idx-1 / idx+nstep-1; dmc.py:98-109 stack of the last frames, reset frame repeated)
__device__ __forceinline__ const uint8_t* channel_plane(const Conv1TcArgs& a, int n, int c) {
    if (!a.ring_frames) return a.obs + ((long long)n * a.cin + c) * (kImg * kImg);
    const int j = c / a.ring_frame_c, cc = c - j * a.ring_frame_c;
    const bool is_next = n >= a.ring_B;
    const int b = is_next ? n - a.ring_B : n;
    const int t = is_next ? a.ring_idx[b] + a.ring_nstep - 1 : a.ring_idx[b] - 1;
    int r = t - (a.ring_stack - 1 - j);
    r = r < 0 ? 0 : r;
    const long long slot = ((long long)a.ring_ep_start[b] + r) % a.ring_capacity;
    return a.ring_frames + (slot * a.ring_frame_c + cc) * (long long)(kImg * kImg);
}

static long long* g_c1_stamps = nullptr;
#ifdef DRQ_STAMPS
#define C1_T() (a.stamps ? clock64() : 0ll)
#else
#define C1_T() 0ll
#endif

// Input rows of one tile staged in shared memory: per channel up to 11 (clamped) source rows, each as a
// replicate-padded row of kC1RowBytes.
constexpr int kC1RowWords = kImg / 4;                 // 21 source words per row
constexpr int kC1MaxRows = 11;
constexpr int kC1RowBytes = 96;                       // [4 pad | 84 | 4 pad | 4 slack]
constexpr int kC1ChBytes = kC1MaxRows * kC1RowBytes;  // 1056
constexpr int kC1ChWords = kC1MaxRows * kC1RowWords;  // 231 source words per channel
constexpr int kC1InBytes = 10 * kC1ChBytes;           // one padded-row buffer (cin <= 10)
constexpr int kC1RawSlot = 960;                       // raw rows of one channel: <= 15 + 11 * 84 bytes, 16-byte granular
constexpr int kC1RawBytes = 10 * kC1RawSlot;          // one raw stage
constexpr int kC1RawStages = 4;

struct TileGeom { int n, p0, rlo, nrows; };

__device__ __forceinline__ TileGeom tile_geom(int t, const int* __restrict__ shift, int pad) {
    constexpr int TILES_PER_IMG = (kPW * kPW + kC1Tile - 1) / kC1Tile;
    TileGeom g;
    g.n = t / TILES_PER_IMG;
    g.p0 = (t - g.n * TILES_PER_IMG) * kC1Tile;
    const int sy = shift ? shift[2 * g.n + 1] : pad;
    const int oy_min = g.p0 / kPW;
    const int oy_max = min(g.p0 + kC1Tile - 1, kPW * kPW - 1) / kPW;
    g.rlo = clampi(2 * oy_min + sy - pad, 0, kImg - 1);
    const int rhi = clampi(2 * oy_max + 2 + sy - pad, 0, kImg - 1);
    g.nrows = rhi - g.rlo + 1;
    return g;
}

// The row producer warp lands the tile's (vertically clamped) source rows of every channel in shared
// memory with one bulk-async copy per channel (the rows of a channel are contiguous in the frame stack);
// the builders then re-pitch them as replicate-padded rows (drqv2.py:26 F.pad(mode='replicate'),
// horizontally).  Thread (channel ci, word jw) walks the rows: no index arithmetic in the loop.
__device__ __forceinline__ void pad_rows(const uint8_t* __restrict__ raw, uint8_t* __restrict__ stage, int off0, int nrows,
                                         int cin, int b) {
    constexpr int RW = kC1RowBytes / 4;
    if (b < cin * kC1RowWords) {
        // thread (channel ci, word jw): copy the 84 pixel bytes of every row to byte 4 of the padded row
        const int ci = b / kC1RowWords, jw = b - ci * kC1RowWords;
        const uint32_t* src = reinterpret_cast<const uint32_t*>(raw + ci * kC1RawSlot + off0) + jw;
        uint32_t* dst = reinterpret_cast<uint32_t*>(stage + ci * kC1ChBytes) + 1 + jw;
#pragma unroll 4
        for (int r = 0; r < nrows; ++r) dst[r * RW] = src[r * kC1RowWords];
    } else if (b < cin * kC1RowWords + 2 * cin) {
        // thread (channel ci, side): the replicate pad words - pixel 0 x4 on the left, pixel 83 x4 on the right
        const int e = b - cin * kC1RowWords, ci = e >> 1, side = e & 1;
        const uint32_t* src = reinterpret_cast<const uint32_t*>(raw + ci * kC1RawSlot + off0) + (side ? kC1RowWords - 1 : 0);
        uint32_t* dst = reinterpret_cast<uint32_t*>(stage + ci * kC1ChBytes) + (side ? 1 + kC1RowWords : 0);
        const uint32_t sel = side ? 0x3333u : 0x0000u;
#pragma unroll 4
        for (int r = 0; r < nrows; ++r) dst[r * RW] = __byte_perm(src[r * kC1RowWords], 0, sel);
    }
}

// bf16 pair (x_A - 128, x_B - 128) from byte bA of group word gA (low half) and byte bB of gB (high half):
// a byte permute with 0x4B000000 makes the float 2^23 + x, subtracting 2^23 + 128 is exact, and so is the
// conversion to bf16 (|x - 128| <= 128 has at most 8 significant bits).
__device__ __forceinline__ float centred(uint32_t g, int b) {
    return __uint_as_float(__byte_perm(g, 0x4B000000u, (uint32_t)b | 0x7650u)) - 8388736.0f;
}
__device__ __forceinline__ uint32_t pair_from(uint32_t gA, int bA, uint32_t gB, int bB) {
    return pack_bf16x2(centred(gA, bA), centred(gB, bB));
}
__device__ __forceinline__ uint32_t one_from(uint32_t gA, int bA) {              // low half x - 128, high half 0
    return pack_bf16x2(centred(gA, bA), 0.f);
}

// One builder thread: position r of the tile, K units [U0, U0 + 3).  K entry k = 9*c + 3*ky + kx; group
// i = k / 3 = 3*c + ky is three consecutive bytes of channel c's staged row ky at byte offset g.
template <int U0, int CIN>                             // CIN = compile-time channel count, 0 = use cin
__device__ __forceinline__ void build_part(uint8_t* tile, const uint8_t* __restrict__ stage, int cin, int r,
                                           const int (&rowoff)[3], int g) {
    constexpr int G0 = U0 * 8 / 3;                     // first group of this quarter (0, 8, 16, 24)
    constexpr int NG = 8;                              // 24 K entries = 8 groups
    const int kmax = CIN ? CIN * 9 : cin * 9;
    uint32_t grp[NG];
    const int sh = (g & 3) * 8;
    const uint8_t* base[3];
#pragma unroll
    for (int ky = 0; ky < 3; ++ky) base[ky] = stage + rowoff[ky] + (g & ~3);
#pragma unroll
    for (int i = 0; i < NG; ++i) {
        const int gi = G0 + i, c = gi / 3, ky = gi % 3;
        uint32_t v = 0;
        if (gi * 3 < kmax) {
            const uint32_t* p = reinterpret_cast<const uint32_t*>(base[ky] + c * kC1ChBytes);
            v = __funnelshift_r(p[0], p[1], sh);
        }
        grp[i] = v;
    }
#pragma unroll
    for (int u = 0; u < 3; ++u) {
        uint32_t w[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const int kA = (U0 + u) * 8 + 2 * e, kB = kA + 1;
            const int iA = kA / 3 - G0, iB = kB / 3 - G0;
            uint32_t v = 0;
            if (kB < kmax) v = pair_from(grp[iA], kA % 3, grp[iB], kB % 3);
            else if (kA < kmax) v = one_from(grp[iA], kA % 3) | (kB == kmax ? 0x3F800000u : 0u);   // data | 1.0
            else if (kA == kmax) v = 0x00003F80u;                                                    // 1.0 | 0
            w[e] = v;
        }
        *reinterpret_cast<uint4*>(tile + (U0 + u) * (kC1Tile * 16) + r * 16) = make_uint4(w[0], w[1], w[2], w[3]);
    }
}

// The same K units from real-valued pixels (FSRC): entry k < cin*9 is RN-bf16(RN-fp32(x - 128)) of the pixel
// x = fobs[n][c][2*oy + ky][2*ox + kx] (already augmented, no shift), entry cin*9 the constant 1.0, the rest 0.  On
// integer pixels in 0..255 these are the bits build_part makes.
template <int U0>
__device__ __forceinline__ void build_part_f32(uint8_t* tile, const float* __restrict__ img, int kmax, int r, int oy, int ox) {
    auto entry = [&](int k) -> float {
        if (k >= kmax) return k == kmax ? 1.f : 0.f;
        const int c = k / 9, ky = (k % 9) / 3, kx = k % 3;
        return __fsub_rn(__ldg(img + (c * kImg + 2 * oy + ky) * kImg + 2 * ox + kx), 128.f);
    };
#pragma unroll
    for (int u = 0; u < 3; ++u) {
        uint32_t w[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const int kA = (U0 + u) * 8 + 2 * e;
            w[e] = pack_bf16x2(entry(kA), entry(kA + 1));
        }
        *reinterpret_cast<uint4*>(tile + (U0 + u) * (kC1Tile * 16) + r * 16) = make_uint4(w[0], w[1], w[2], w[3]);
    }
}

template <bool WGRAD, int CIN, bool FSRC = false>
__global__ void __launch_bounds__(kC1Threads, 1) conv1_tc_kernel(Conv1TcArgs a) {
    extern __shared__ __align__(128) uint8_t smem[];
    constexpr int STAGE = kC1ABytes + (WGRAD ? kC1DBytes : 0);
    uint8_t* w_s = smem;                                    // fwd only: packed weights
    float* bias_s = reinterpret_cast<float*>(smem + kC1WBytes);   // fwd only: fused bias'
    uint8_t* in_s = smem + kC1WBytes + 128;                 // 2 builder groups x 2 padded-row buffers
    uint8_t* raw_s = in_s + 4 * kC1InBytes;                 // kC1RawStages x raw rows (bulk-copy destinations)
    uint8_t* st_s = raw_s + kC1RawStages * kC1RawBytes;
    uint64_t* bars = reinterpret_cast<uint64_t*>(st_s + kC1Stages * STAGE + (WGRAD ? kC1DBytes : 0));
    uint64_t* full = bars;                     // one builder group (256 arrivals)
    uint64_t* empty = bars + kC1Stages;
    uint64_t* dfull = bars + 2 * kC1Stages;    // wgrad: bulk copy of the d tile
    uint64_t* tfull = bars + 3 * kC1Stages;
    uint64_t* tempty = bars + 3 * kC1Stages + kC1Acc;
    uint64_t* done = bars + 3 * kC1Stages + 2 * kC1Acc;
    uint64_t* rfull = done + 1;                // raw rows landed (cin producer lanes announce their bytes)
    uint64_t* rempty = rfull + kC1RawStages;   // raw stage re-pitched by the 256 builders of a group
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(rempty + kC1RawStages);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    constexpr int TILES_PER_IMG = (kPW * kPW + kC1Tile - 1) / kC1Tile;   // 14
    const int total_tiles = a.n_images * TILES_PER_IMG;

    if (threadIdx.x == 0) {
        for (int i = 0; i < kC1Stages; ++i) { mbar_init(full + i, kC1Builders / 2); mbar_init(empty + i, 1); mbar_init(dfull + i, 1); }
        for (int i = 0; i < kC1Acc; ++i) { mbar_init(tfull + i, 1); mbar_init(tempty + i, 4); }
        mbar_init(done, 1);
        for (int i = 0; i < kC1RawStages; ++i) { mbar_init(rfull + i, a.cin); mbar_init(rempty + i, kC1Builders / 2); }
        fence_barrier_init();
    }
    if (warp == 16) {
        tmem_alloc(tmem_slot, 128);
        tmem_relinquish();
    }
    if (!WGRAD) {
        const uint4* src = reinterpret_cast<const uint4*>(a.w);
        uint4* dst = reinterpret_cast<uint4*>(w_s);
        for (int i = threadIdx.x; i < (kC1WBytes + 128) / 16; i += kC1Threads) dst[i] = __ldg(src + i);
    }
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp < 16) {
        // ------------------------------------------------ row re-pitch + im2col builders
        // Two groups of 8 warps work on alternate tiles (group 0: tiles 0, 2, 4, ... of this CTA; group 1: 1, 3, ...)
        // so that one group's re-pitch / barrier latency overlaps the other's build.  Ring positions follow
        // from the tile ordinal.
        const int group = warp >> 3, gb = threadIdx.x & 255, r = gb & 127, half = gb >> 7;
        int it = 0;
        for (int ord = group; blockIdx.x + ord * (int)gridDim.x < total_tiles; ord += 2, ++it) {
            const int t = blockIdx.x + ord * gridDim.x;
            const int stage = ord % kC1Stages; const uint32_t phase = (ord / kC1Stages) & 1;
            const int rs = ord % kC1RawStages; const uint32_t rphase = (ord / kC1RawStages) & 1;
            const TileGeom cur = tile_geom(t, a.shift, a.pad);
            uint8_t* stg = in_s + (group * 2 + (it & 1)) * kC1InBytes;
            if (!FSRC) {
                mbar_wait(rfull + rs, rphase);
                pad_rows(raw_s + rs * kC1RawBytes, stg, (cur.rlo * kImg) & 15, cur.nrows, a.cin, gb);
                mbar_arrive(rempty + rs);
                if (group == 0) asm volatile("bar.sync 1, 256;" ::: "memory");      // padded rows visible to the group
                else            asm volatile("bar.sync 2, 256;" ::: "memory");
            }
            // Positions past the image (last tile) build from clamped, valid addresses in the forward (their rows
            // are never stored); in wgrad their im2col rows are zeroed below (the gradient tile's rows there
            // belong to the next image).
            const int p = min(cur.p0 + r, kPW * kPW - 1);
            const bool live = !WGRAD || cur.p0 + r < kPW * kPW;
            const int oy = p / kPW, ox = p - oy * kPW;
            const int sx = a.shift ? a.shift[2 * cur.n] : a.pad, sy = a.shift ? a.shift[2 * cur.n + 1] : a.pad;
            int rowoff[3];
#pragma unroll
            for (int ky = 0; ky < 3; ++ky)
                rowoff[ky] = (clampi(2 * oy + ky + sy - a.pad, 0, kImg - 1) - cur.rlo) * kC1RowBytes;
            // aug column j = src[clamp(j + sx - pad)] = padded[j + sx + (4 - pad)]; the three kx taps start at j = 2*ox
            const int gofs = 2 * ox + sx + (4 - a.pad);
            mbar_wait(empty + stage, phase ^ 1);
            uint8_t* tile = st_s + stage * STAGE;
            if (!live) {
#pragma unroll
                for (int u = 0; u < 6; ++u)
                    *reinterpret_cast<uint4*>(tile + (half * 6 + u) * (kC1Tile * 16) + r * 16) = make_uint4(0, 0, 0, 0);
            } else if (FSRC) {
                const float* img = a.fobs + (long long)cur.n * a.cin * (kImg * kImg);
                if (half == 0) { build_part_f32<0>(tile, img, a.cin * 9, r, oy, ox); build_part_f32<3>(tile, img, a.cin * 9, r, oy, ox); }
                else           { build_part_f32<6>(tile, img, a.cin * 9, r, oy, ox); build_part_f32<9>(tile, img, a.cin * 9, r, oy, ox); }
            } else if (half == 0) {
                build_part<0, CIN>(tile, stg, a.cin, r, rowoff, gofs);
                build_part<3, CIN>(tile, stg, a.cin, r, rowoff, gofs);
            } else {
                build_part<6, CIN>(tile, stg, a.cin, r, rowoff, gofs);
                build_part<9, CIN>(tile, stg, a.cin, r, rowoff, gofs);
            }
            fence_proxy_async();
            mbar_arrive(full + stage);
        }
    } else if (warp == 16) {
        // ------------------------------------------------ UMMA issuer (+ d-tile producer in wgrad)
        int stage = 0; uint32_t phase = 0; int acc = 0; uint32_t acc_phase = 0;
        bool first = true;
        if (WGRAD && elect_one()) {
            // prefetch the d tiles of the first kC1Stages tiles
            int s2 = 0;
            for (int t = blockIdx.x; t < total_tiles && s2 < kC1Stages; t += gridDim.x, ++s2) {
                const int n = t / TILES_PER_IMG, p0 = (t - n * TILES_PER_IMG) * kC1Tile;
                const long long row0 = (long long)n * DRQ_PLB + DRQ_GUARD + p0;
                mbar_arrive_expect_tx(dfull + s2, kC1DBytes);
                for (int c = 0; c < 4; ++c)
                    bulk_g2s(st_s + s2 * STAGE + kC1ABytes + c * kC1Tile * 16, a.d + (c * a.cs_d + row0) * 8, kC1Tile * 16, dfull + s2);
            }
        }
        __syncwarp();
        // descriptors: per-stage base + compile-time (address >> 4) offsets
        const uint64_t da0 = WGRAD ? make_smem_desc(smem_u32(st_s) + kC1ABytes, 128, kC1Tile * 16)     // d^T, MN-major
                                   : make_smem_desc(smem_u32(st_s), kC1Tile * 16, 128);               // im2col, K-major
        const uint64_t db0 = WGRAD ? make_smem_desc(smem_u32(st_s), 128, kC1Tile * 16)                 // im2col, MN-major
                                   : make_smem_desc(smem_u32(w_s), 512, 128);                         // weights, K-major
        for (int t = blockIdx.x; t < total_tiles; t += gridDim.x) {
            if (!WGRAD) mbar_wait(tempty + acc, acc_phase ^ 1);
            mbar_wait(full + stage, phase);
            if (WGRAD) mbar_wait(dfull + stage, phase);
            tc_fence_after();
            if (elect_one()) {
                const uint64_t so = (uint64_t)(stage * (STAGE >> 4));
                if (!WGRAD) {
                    constexpr uint32_t idesc = make_idesc_bf16(128, 32, false, false);
#pragma unroll
                    for (int ks = 0; ks < kC1K / 16; ++ks)
                        umma_bf16(tmem_base + acc * 32, da0 + so + (uint64_t)(ks * 2 * kC1Tile), db0 + (uint64_t)(ks * 2 * 32), idesc,
                                  ks ? 1u : 0u);
                    umma_commit(empty + stage);
                    umma_commit(tfull + acc);
                } else {
                    // S[co (64)][k (96)] += d^T[co][pos] * im2col[pos][k]; both operands MN-major, K = 16 positions
                    constexpr uint32_t idesc = make_idesc_bf16(64, kC1K, true, true);
#pragma unroll
                    for (int ks = 0; ks < kC1Tile / 16; ++ks)
                        umma_bf16(tmem_base, da0 + so + (uint64_t)(ks * 16), db0 + so + (uint64_t)(ks * 16), idesc,
                                  (first && ks == 0) ? 0u : 1u);
                    umma_commit(empty + stage);
                }
            }
            __syncwarp();
            first = false;
            if (WGRAD) {
                // refill this stage's d tile for the tile kC1Stages ahead, once the UMMAs reading it retire
                const int tn = t + kC1Stages * gridDim.x;
                if (tn < total_tiles && elect_one()) {
                    mbar_wait(empty + stage, phase);
                    const int n = tn / TILES_PER_IMG, p0 = (tn - n * TILES_PER_IMG) * kC1Tile;
                    const long long row0 = (long long)n * DRQ_PLB + DRQ_GUARD + p0;
                    mbar_arrive_expect_tx(dfull + stage, kC1DBytes);
                    for (int c = 0; c < 4; ++c)
                        bulk_g2s(st_s + stage * STAGE + kC1ABytes + c * kC1Tile * 16, a.d + (c * a.cs_d + row0) * 8, kC1Tile * 16, dfull + stage);
                }
                __syncwarp();
            }
            if (++stage == kC1Stages) { stage = 0; phase ^= 1; }
            if (++acc == kC1Acc) { acc = 0; acc_phase ^= 1; }
        }
        if (WGRAD) {
            if (elect_one()) umma_commit(done);
            __syncwarp();
        }
    } else if (warp == 21) {
        // ------------------------------------------------ row producer: lane c copies channel c's rows of the tile
        if (!FSRC && lane < a.cin) {
            int rs = 0; uint32_t rphase = 0;
            // As in conv1_planes_kernel's producer: the image's shift, ring index and episode start are requested
            // kAhead tiles ahead (their round trip to L2, and a 64-bit modulo per tile, were on this warp's serial path:
            // ~1.3 us per tile), the ring slot is a compare-and-subtract, the lane's frame / channel are loop constants.
            constexpr int kAhead = 4;
            constexpr int TPI = (kPW * kPW + kC1Tile - 1) / kC1Tile;
            const bool ring = a.ring_frames != nullptr;
            const int fj = ring ? lane / a.ring_frame_c : 0, fcc = ring ? lane - fj * a.ring_frame_c : 0;
            const int cap = (int)a.ring_capacity;
            int q_sy[kAhead], q_idx[kAhead], q_ep[kAhead];
            auto fetch = [&](int t, int& sy, int& idx, int& ep) {
                sy = a.pad; idx = 0; ep = 0;
                if (t >= total_tiles) return;
                const int n = t / TPI;
                if (a.shift) sy = a.shift[2 * n + 1];
                if (ring) {
                    const int b = n >= a.ring_B ? n - a.ring_B : n;
                    idx = a.ring_idx[b];
                    ep = a.ring_ep_start[b];
                }
            };
#pragma unroll
            for (int d = 0; d < kAhead; ++d) fetch(blockIdx.x + d * gridDim.x, q_sy[d], q_idx[d], q_ep[d]);
            for (int t0 = blockIdx.x; t0 < total_tiles; t0 += kAhead * gridDim.x) {
#pragma unroll
                for (int d = 0; d < kAhead; ++d) {
                    const int t = t0 + d * gridDim.x;
                    if (t >= total_tiles) break;
                    const int sy1[2] = {0, q_sy[d]};                 // tile_geom reads shift[2 * n + 1]: hand it element 1 of a pair
                    const TileGeom g0 = tile_geom(t - (t / TPI) * TPI, sy1, a.pad);   // image 0's tile of the same index: same rows
                    const int n = t / TPI;
                    const uint8_t* plane;
                    if (!ring) {
                        plane = a.obs + ((long long)n * a.cin + lane) * (kImg * kImg);
                    } else {
                        const int tt = n >= a.ring_B ? q_idx[d] + a.ring_nstep - 1 : q_idx[d] - 1;
                        int r = tt - (a.ring_stack - 1 - fj);
                        r = r < 0 ? 0 : r;
                        int slot = q_ep[d] + r;
                        while (slot >= cap) slot -= cap;
                        plane = a.ring_frames + ((long long)slot * a.ring_frame_c + fcc) * (long long)(kImg * kImg);
                    }
                    fetch(t + kAhead * gridDim.x, q_sy[d], q_idx[d], q_ep[d]);
                    const uint8_t* src = plane + g0.rlo * kImg;
                    const int off0 = (g0.rlo * kImg) & 15;           // every channel plane starts 16-byte aligned
                    const uint32_t nbytes = (uint32_t)((off0 + g0.nrows * kImg + 15) & ~15);
                    mbar_wait(rempty + rs, rphase ^ 1);
                    mbar_arrive_expect_tx(rfull + rs, nbytes);
                    bulk_g2s(raw_s + rs * kC1RawBytes + lane * kC1RawSlot, src - off0, nbytes, rfull + rs);
                    if (++rs == kC1RawStages) { rs = 0; rphase ^= 1; }
                }
            }
        }
    } else {
        // ------------------------------------------------ epilogue warps 17..20 -> lane quarters 1,2,3,0
        const int q = warp & 3;
        if (!WGRAD) {
            int acc = 0; uint32_t acc_phase = 0;
            float bias_r[32];                       // registers: shared-memory reads per tile were bank-conflict wavefronts
#pragma unroll
            for (int i = 0; i < 32; ++i) bias_r[i] = bias_s[i];
            for (int t = blockIdx.x; t < total_tiles; t += gridDim.x) {
                const int n = t / TILES_PER_IMG, p0 = (t - n * TILES_PER_IMG) * kC1Tile;
                mbar_wait(tfull + acc, acc_phase);
                tc_fence_after();
                float v[32];
                tmem_ld_32x32(tmem_base + ((uint32_t)(q * 32) << 16) + acc * 32, v);
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(tempty + acc);
                if (++acc == kC1Acc) { acc = 0; acc_phase ^= 1; }
                const int p = p0 + q * 32 + lane;
                if (p >= kPW * kPW) continue;
                const long long row = (long long)n * DRQ_PLB + DRQ_GUARD + p;
                uint32_t packed[16];
#pragma unroll
                for (int i = 0; i < 16; ++i)
                    packed[i] = pack_bf16x2(fmaxf(fmaf(v[2 * i], kC1Scale, bias_r[2 * i]), 0.f),
                                            fmaxf(fmaf(v[2 * i + 1], kC1Scale, bias_r[2 * i + 1]), 0.f));
#pragma unroll
                for (int c = 0; c < 4; ++c)
                    *reinterpret_cast<uint4*>(a.out + (c * a.cs_out + row) * 8) =
                        make_uint4(packed[4 * c], packed[4 * c + 1], packed[4 * c + 2], packed[4 * c + 3]);
            }
        } else {
            mbar_wait(done, 0);
            tc_fence_after();
            if (q < 2) {
                float* out = a.partial + (long long)blockIdx.x * (32 * kC1K);
#pragma unroll
                for (int c0 = 0; c0 < kC1K; c0 += 32) {
                    float v[32];
                    tmem_ld_32x32(tmem_base + ((uint32_t)(q * 32) << 16) + c0, v);
                    if (lane < 16) {
                        float4* dst = reinterpret_cast<float4*>(out + (q * 16 + lane) * kC1K + c0);
#pragma unroll
                        for (int i = 0; i < 8; ++i) dst[i] = make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
                    }
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 16) tmem_dealloc(tmem_base, 128);
}

__global__ void __launch_bounds__(256)
pack_conv1_w_kernel(const float* __restrict__ w, const float* __restrict__ bias, __nv_bfloat16* __restrict__ out, int cin) {
    __shared__ float part[32][9];
    pack_conv1_w_block(w, bias, out, cin, threadIdx.x, part);
}

// dw[co][k] = S[co][k]/255 + (128/255 - 0.5) db[co] (k < cin*9), db[co] = S[co][cin*9], S = sum of the per-CTA
// partials [32][96].  Block = 32 outputs x 8 slices of the G partials, combined in fixed order.
__global__ void __launch_bounds__(256)
conv1_wgrad_reduce_kernel(const float* __restrict__ partial, int G, int cin, float* __restrict__ dw, float* __restrict__ db) {
    __shared__ float red[8][33], redb[8][33];
    conv1_reduce_block(partial, G, cin, dw, db, blockIdx.x, red, redb);
}

// ---------------------------------------------------------------- forward, second formulation: parity planes
// The im2col tile above costs 96 built entries per output position (9 taps x 9 channels, padded), and building them is
// what the kernel spends its time on.  The stride-2 conv is a stride-1 conv over the four row/column parity planes of
// the augmented image V (plane (py, px)[i][j] = V[2i+py][2j+px]): tap (ky, kx) of output (y, x) is plane (ky&1, kx&1)
// at [y + ky/2][x + kx/2].  So the builders convert every pixel of the tile's 7 V rows ONCE, pixel-major - K unit 0 =
// channels 0..7, K unit 1 = channels 8.. (zero padded) - into [K unit][py][px][4 plane rows][42 columns][16 B], and tap
// (ky, kx) of 126 consecutive (row, column) positions is the K-major operand at the constant offset
// (ky/2)*42 + kx/2 of its plane: 9 UMMAs of M128 N32 K16 per tile of 3 output rows, 10 converted values per input
// pixel instead of 96 per output pixel.  A builder thread owns one plane column of one V row (two pixels): consecutive
// lanes write consecutive 16-byte slots (no bank conflicts) and read the bulk-copied source rows directly - the shift
// and the replicate padding are a clamped byte address and a byte selector, there is no re-pitch pass.  Same
// exact-integer entries, same epilogue (scale 1/255, fused bias), same results up to fp32 summation order.
#ifndef P1_RELAXED_WAIT
#define P1_RELAXED_WAIT mbar_wait_relaxed<128u>
#endif
#ifndef P1_HINT
#define P1_HINT 1000000u        // suspend-time hint of the kernel's mbarrier waits (measured: no effect between 0 and 1 ms)
#endif
constexpr int kP1Pitch = 42;                      // plane columns j = 0..41 (V columns 2j + px)
constexpr int kP1Rows = 3;                        // output rows per tile
constexpr int kP1TilesPerImg = (kPW + kP1Rows - 1) / kP1Rows;     // 14
constexpr int kP1Live = kP1Rows * kP1Pitch;       // 126 accumulator rows carry positions (column 41 is a dummy)
constexpr int kP1Region = 4 * kP1Pitch * 16;      // one (K unit, py, px): 4 plane rows
constexpr int kP1StageBytes = 8 * kP1Region;      // 21,504
constexpr int kP1Stages = 6;
constexpr int kP1VRows = 2 * kP1Rows + 1;         // V rows per tile
constexpr int kP1WBytes = 9 * 2 * 32 * 16;        // [tap][2 K units][32 co][16 B]
constexpr int kP1Units = kP1VRows * (kImg / 4);   // builder work units: (V row, 4 columns) = 147
constexpr int kP1Group = 160;                     // builder threads per group
constexpr int kP1Groups = 3;                      // groups take tiles round robin
constexpr int kP1Acc = 4;                         // accumulator ring: 4 x 32 TMEM columns
constexpr int kP1Threads = kP1Groups * kP1Group + 10 * 32; // + UMMA warp, 8 epilogue warps (two per TMEM lane quarter), row producer warp
constexpr int kP1RawSlot = 640;                   // raw rows of one channel: 7 * 84 bytes + the word a funnel shift may touch, 128-byte granular
constexpr int kP1BoxWords = kP1RawSlot / 4;       // TMA box: 160 words of a channel plane from the tile's first source row
constexpr int kP1RawBytes = 10 * kP1RawSlot;
constexpr int kP1RawStages = 8;

struct P1Geom { int n, y0, rlo, nrows; };
__device__ __forceinline__ P1Geom p1_geom(int t, int sy, int pad) {
    P1Geom g;
    g.n = t / kP1TilesPerImg;
    g.y0 = (t - g.n * kP1TilesPerImg) * kP1Rows;
    g.rlo = clampi(2 * g.y0 + sy - pad, 0, kImg - 1);
    const int rhi = clampi(2 * g.y0 + kP1VRows - 1 + sy - pad, 0, kImg - 1);
    g.nrows = rhi - g.rlo + 1;
    return g;
}

// fp16 pairs (x_A - 128, x_B - 128) of two pixels at once: `ab` = [A px0, B px0, A px1, B px1] bytes (one PRMT from the
// two channel words); 0x6400 | x is the fp16 1024 + x, one packed subtract centres both halves exactly.  (The im2col
// kernel feeds bf16 because its weight-gradient twin multiplies the same tile with a bf16 gradient and kind::f16 wants
// one format for both operands; the forward alone is free to use fp16 pixels x fp16 copies of the bf16-rounded weights,
// which is 1.25 instructions per entry instead of 2.5.)
__device__ __forceinline__ uint32_t centred_h2(uint32_t ab, uint32_t sel) {
    const uint32_t h = __byte_perm(ab, 0x64646464u, sel);
    const __half2 c = __hsub2(*reinterpret_cast<const __half2*>(&h), __half2half2(__ushort_as_half((unsigned short)0x6480)));   // 1024 + 128
    return *reinterpret_cast<const uint32_t*>(&c);
}

__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, int c0, int c1, uint64_t* bar) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
                 ::"r"(dst), "l"(map), "r"(c0), "r"(c1), "r"(smem_u32(bar)) : "memory");
}

// `map`: the source as (1764 words of a channel plane) x (channel planes): the gathered stacks [N * cin planes], or the
// ring's frames [capacity * frame_c planes]; box = (kP1BoxWords, cin) resp. (kP1BoxWords, frame_c)
template <int CIN>                                // compile-time channel count, 0 = use a.cin (<= 10)
__global__ void __launch_bounds__(kP1Threads, 1) conv1_planes_kernel(const __grid_constant__ CUtensorMap map, Conv1TcArgs a) {
    extern __shared__ __align__(128) uint8_t smem[];
    uint8_t* w_s = smem;                                    // [tap][2][32][16 B]
    float* bias_s = reinterpret_cast<float*>(smem + kP1WBytes);
    uint8_t* raw_s = smem + kP1WBytes + 128;                // kP1RawStages x raw rows (bulk-copy destinations)
    uint8_t* st_s = raw_s + kP1RawStages * kP1RawBytes;
    uint64_t* bars = reinterpret_cast<uint64_t*>(st_s + kP1Stages * kP1StageBytes + 128);
    uint64_t* full = bars;
    uint64_t* empty = bars + kP1Stages;
    uint64_t* tfull = bars + 2 * kP1Stages;
    uint64_t* tempty = bars + 2 * kP1Stages + kP1Acc;
    uint64_t* rfull = bars + 2 * kP1Stages + 2 * kP1Acc;
    uint64_t* rempty = rfull + kP1RawStages;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(rempty + kP1RawStages);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    constexpr int kBuildWarps = kP1Groups * kP1Group / 32;  // warps 0..14 build, 15 issues UMMAs, 16..23 epilogue, 24 copies rows
    const int cin = CIN ? CIN : a.cin;
    const int total_tiles = a.n_images * kP1TilesPerImg;

    if (threadIdx.x == 0) {
        for (int i = 0; i < kP1Stages; ++i) { mbar_init(full + i, kP1Group); mbar_init(empty + i, 1); }
        for (int i = 0; i < kP1Acc; ++i) { mbar_init(tfull + i, 1); mbar_init(tempty + i, 4); }
        for (int i = 0; i < kP1RawStages; ++i) { mbar_init(rfull + i, a.ring_frames ? a.ring_stack : 1); mbar_init(rempty + i, kP1Group); }
        fence_barrier_init();
    }
    if (warp == kBuildWarps) {
        tmem_alloc(tmem_slot, kP1Acc * 32);
        tmem_relinquish();
    }
    // plane stages start as zeros: the never written fourth row of the odd-row planes must read as finite values
    for (int i = threadIdx.x; i < kP1Stages * kP1StageBytes / 16; i += kP1Threads) reinterpret_cast<uint4*>(st_s)[i] = make_uint4(0, 0, 0, 0);
    {
        // B operands from the packed im2col weights [k / 8][co][k % 8], k = 9 * c + tap: [tap][c / 8][co][c % 8].  The packed
        // block is staged in the (not yet used) raw-row buffer with 16-byte loads and re-ordered from there: 2-byte gathers
        // straight from global memory were a chain of L2 round trips per thread.
        const uint4* src = reinterpret_cast<const uint4*>(a.w);
        uint4* tmp = reinterpret_cast<uint4*>(raw_s);
        for (int i = threadIdx.x; i < (kC1WBytes + 128) / 16; i += kP1Threads) tmp[i] = __ldg(src + i);
        __syncthreads();
        // (fp16 copies of the bf16 weights: exact but for magnitudes below 2^-14, which lose bits to fp16 subnormals)
        const __nv_bfloat16* wp = reinterpret_cast<const __nv_bfloat16*>(raw_s);
        __half* dst = reinterpret_cast<__half*>(w_s);
        for (int i = threadIdx.x; i < 9 * 2 * 32 * 8; i += kP1Threads) {
            const int e = i & 7, co = (i >> 3) & 31, u = (i >> 8) & 1, tap = i >> 9;
            const int c = u * 8 + e, k = 9 * c + tap;
            dst[i] = __float2half_rn(c < cin ? __bfloat162float(wp[((k >> 3) * 32 + co) * 8 + (k & 7)]) : 0.f);
        }
        if (threadIdx.x < 32) bias_s[threadIdx.x] = reinterpret_cast<const float*>(wp + kC1Units * 32 * 8)[threadIdx.x];
    }
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();            // also: the staged weights are read before the row producer overwrites the raw buffer
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp < kBuildWarps) {
        // ------------------------------------------------ plane builders; three groups of 5 warps take tiles round robin
        const int group = threadIdx.x / kP1Group, gb = threadIdx.x - group * kP1Group;
        const int k = gb / (kImg / 4), g = gb - k * (kImg / 4);          // work unit: V row k of the tile, V columns 4g..4g+3
        const bool worker = gb < kP1Units;
        long long s_raw = 0, s_empty = 0, s_build = 0, s_fence = 0;
        const long long s_begin = clock64();
        // the shifts of a tile's image are fetched one tile ahead: a dependent global load per tile was most of the loop
        int2 sh_next = make_int2(a.pad, a.pad);
        {
            const int t0 = blockIdx.x + group * (int)gridDim.x;
            if (a.shift && t0 < total_tiles) sh_next = *reinterpret_cast<const int2*>(a.shift + 2 * (t0 / kP1TilesPerImg));
        }
        for (int ord = group; blockIdx.x + ord * (int)gridDim.x < total_tiles; ord += kP1Groups) {
            const long long c0 = clock64();
            const int t = blockIdx.x + ord * gridDim.x;
            const int stage = ord % kP1Stages; const uint32_t phase = (ord / kP1Stages) & 1;
            const int rs = ord % kP1RawStages; const uint32_t rphase = (ord / kP1RawStages) & 1;
            const int sx = sh_next.x, sy = sh_next.y;
            {
                const int tn = t + kP1Groups * (int)gridDim.x;
                if (a.shift && tn < total_tiles) sh_next = *reinterpret_cast<const int2*>(a.shift + 2 * (tn / kP1TilesPerImg));
            }
            const P1Geom cur = p1_geom(t, sy, a.pad);
            P1_RELAXED_WAIT(rfull + rs, rphase);
            const long long c1 = clock64();
            P1_RELAXED_WAIT(empty + stage, phase ^ 1);
            const long long c2 = clock64();
            if (worker) {
                // V row 2*y0 + k = source row clamp(. + sy - pad) (a V row past the image only feeds output rows past it);
                // V columns 4g + i = source columns s_i = clamp(. + sx - pad): the bytes s_0 + b_i of the row, b_i = s_i - s_0
                // (consecutive, or repeated at an edge).  (Two plane columns 21 apart per thread instead - consecutive lanes on
                // consecutive 16-byte slots, no two-pass stores - measured slower: twice the loads.)
                const int sr = clampi(min(2 * cur.y0 + k, kImg - 1) + sy - a.pad, 0, kImg - 1) - cur.rlo;
                const int x0 = 4 * g + sx - a.pad;
                const int s0 = clampi(x0, 0, kImg - 1);
                const uint32_t b1 = (uint32_t)(clampi(x0 + 1, 0, kImg - 1) - s0), b2 = (uint32_t)(clampi(x0 + 2, 0, kImg - 1) - s0),
                               b3 = (uint32_t)(clampi(x0 + 3, 0, kImg - 1) - s0);
                const int ab = ((cur.rlo * kImg) & 15) + sr * kImg + s0;
                const int sh = (ab & 3) * 8;
                // pixel pairs (0, 2) -> plane column 2g and (1, 3) -> 2g + 1 of the even / odd column planes:
                // [A b_i, B b_i, A b_j, B b_j] from the two channel words A, B
                const uint32_t sel02 = 0u | (4u << 4) | (b2 << 8) | ((4u + b2) << 12);
                const uint32_t sel13 = b1 | ((4u + b1) << 4) | (b3 << 8) | ((4u + b3) << 12);
                const uint8_t* base = raw_s + rs * kP1RawBytes + (ab & ~3);
                uint32_t v[10];
#pragma unroll
                for (int c = 0; c < 10; ++c) {
                    v[c] = 0x80808080u;                                   // pixel 128 = entry 0 (its weights are zero anyway)
                    if (c < cin) {
                        const uint32_t* p = reinterpret_cast<const uint32_t*>(base + c * kP1RawSlot);
                        v[c] = __funnelshift_r(p[0], p[1], sh);
                    }
                }
                // h[px][pair][q]: channel pair q of the pixel at plane column 2g + pair of column plane px
                uint32_t h[2][2][5];
#pragma unroll
                for (int q = 0; q < 5; ++q) {
                    const uint32_t e = __byte_perm(v[2 * q], v[2 * q + 1], sel02), o = __byte_perm(v[2 * q], v[2 * q + 1], sel13);
                    h[0][0][q] = centred_h2(e, 0x4140u); h[0][1][q] = centred_h2(e, 0x4342u);
                    h[1][0][q] = centred_h2(o, 0x4140u); h[1][1][q] = centred_h2(o, 0x4342u);
                }
                // a lane owns two adjacent 16-byte slots per plane; lanes 4..7 of every eight write theirs in the other order,
                // so that each store instruction of a quarter warp hits eight different bank groups (lane g and g + 4 own
                // slots 128 bytes apart: ncu counted 2.0 M conflict wavefronts of 4.2 M with the straight order)
                const int flip = (g >> 2) & 1;
                uint8_t* dst = st_s + stage * kP1StageBytes + (k & 1) * (2 * kP1Region) + ((k >> 1) * kP1Pitch + 2 * g) * 16;
#pragma unroll
                for (int px = 0; px < 2; ++px)
#pragma unroll
                    for (int o = 0; o < 2; ++o) {
                        const int pr = o ^ flip;
                        uint8_t* d = dst + px * kP1Region + pr * 16;
                        *reinterpret_cast<uint4*>(d) = make_uint4(pr ? h[px][1][0] : h[px][0][0], pr ? h[px][1][1] : h[px][0][1],
                                                                  pr ? h[px][1][2] : h[px][0][2], pr ? h[px][1][3] : h[px][0][3]);
                        *reinterpret_cast<uint4*>(d + 4 * kP1Region) = make_uint4(pr ? h[px][1][4] : h[px][0][4], 0, 0, 0);
                    }
            }
            mbar_arrive(rempty + rs);
            const long long c3 = clock64();
            fence_proxy_async();
            mbar_arrive(full + stage);
            const long long c4 = clock64();
            s_raw += c1 - c0; s_empty += c2 - c1; s_build += c3 - c2; s_fence += c4 - c3;
        }
        if (a.stamps && blockIdx.x == 0 && threadIdx.x == 0) {
            a.stamps[0] = s_raw; a.stamps[1] = 0; a.stamps[2] = s_empty; a.stamps[3] = s_build; a.stamps[4] = s_fence;
            a.stamps[5] = clock64() - s_begin;
        }
    } else if (warp == kBuildWarps) {
        // ------------------------------------------------ UMMA issuer: tap (ky, kx) = plane (ky&1, kx&1) at row offset (ky/2)*42 + kx/2
        int stage = 0; uint32_t phase = 0; int acc = 0; uint32_t acc_phase = 0;
        const uint64_t da0 = make_smem_desc(smem_u32(st_s), 4 * kP1Region, 128);
        const uint64_t db0 = make_smem_desc(smem_u32(w_s), 512, 128);
        constexpr uint32_t idesc = make_idesc_bf16(128, 32, false, false) & ~((1u << 7) | (1u << 10));     // A, B format fp16 (0)
        long long s_tempty = 0, s_full = 0;
        const long long s_begin = clock64();
        for (int t = blockIdx.x; t < total_tiles; t += gridDim.x) {
            const long long c0 = clock64();
            mbar_wait<P1_HINT>(tempty + acc, acc_phase ^ 1);
            const long long c1 = clock64();
            mbar_wait<P1_HINT>(full + stage, phase);
            s_tempty += c1 - c0; s_full += clock64() - c1;
            tc_fence_after();
            if (elect_one()) {
                const uint64_t da = da0 + (uint64_t)(stage * (kP1StageBytes >> 4));
#pragma unroll
                for (int tap = 0; tap < 9; ++tap) {
                    const int ky = tap / 3, kx = tap % 3;
                    umma_bf16(tmem_base + acc * 32,
                              da + (uint64_t)(((ky & 1) * 2 + (kx & 1)) * (kP1Region >> 4) + (ky >> 1) * kP1Pitch + (kx >> 1)),
                              db0 + (uint64_t)(tap * 64), idesc, tap ? 1u : 0u);
                }
                umma_commit(empty + stage);
                umma_commit(tfull + acc);
            }
            __syncwarp();
            if (++stage == kP1Stages) { stage = 0; phase ^= 1; }
            if (++acc == kP1Acc) { acc = 0; acc_phase ^= 1; }
        }
        // drain: the commits' arrivals on the last stages' `empty` barriers are asynchronous and nobody else waits for them;
        // the CTA must not exit (and hand its shared memory to the next CTA) while one is still in flight
        for (int j = 0; j < kP1Stages; ++j) {
            int s2 = stage - 1 - j; uint32_t ph = phase;
            if (s2 < 0) { s2 += kP1Stages; ph ^= 1; }
            // slot s2 was last committed in "wrap" ph (never used at all if the CTA had fewer tiles: its phase 0 never
            // completes - skip those)
            const int used = (int)((total_tiles - 1 - (int)blockIdx.x) / (int)gridDim.x) + 1;     // tiles of this CTA
            if (j < used) mbar_wait<P1_HINT>(empty + s2, ph);
        }
        if (a.stamps && blockIdx.x == 0 && lane == 0) { a.stamps[6] = s_tempty; a.stamps[7] = s_full; a.stamps[8] = clock64() - s_begin; }
    } else if (warp == kBuildWarps + 9) {
        // ------------------------------------------------ row producer: one tensor-map copy per tile (gathered stacks) or
        // one per ring frame - every channel's 7 source rows (588 contiguous bytes of its plane) in one box.  (One
        // 1-d bulk copy per channel, as the im2col kernel does, was the bottleneck here: ~85 ns per copy issued by a warp.)
        const int n_src = a.ring_frames ? a.ring_stack : 1;
        if (lane < n_src) {
            int rs = 0; uint32_t rphase = 0;
            const int planes_per_src = a.ring_frames ? a.ring_frame_c : a.cin;
            const uint32_t nbytes = (uint32_t)(planes_per_src * kP1RawSlot);
            // The tile's geometry needs the image's shift, its ring index and episode start: global loads whose latency
            // (and, before, a 64-bit modulo per tile) sat on this lane's serial path - one tile of this loop could not be
            // shorter than a round trip to L2.  The raw values are requested kP1Ahead tiles ahead and only used - clamps,
            // ring slot by compare-and-subtract (ep_start < capacity, row < capacity) - when their tile comes up.
            constexpr int kP1Ahead = 4;
            int q_sy[kP1Ahead], q_idx[kP1Ahead], q_ep[kP1Ahead];
            auto fetch = [&](int t, int& sy, int& idx, int& ep) {
                sy = a.pad; idx = 0; ep = 0;
                if (t >= total_tiles) return;
                const int n = t / kP1TilesPerImg;
                if (a.shift) sy = a.shift[2 * n + 1];
                if (a.ring_frames) {
                    const int b = n >= a.ring_B ? n - a.ring_B : n;
                    idx = a.ring_idx[b];
                    ep = a.ring_ep_start[b];
                }
            };
#pragma unroll
            for (int d = 0; d < kP1Ahead; ++d) fetch(blockIdx.x + d * gridDim.x, q_sy[d], q_idx[d], q_ep[d]);
            const int cap = (int)a.ring_capacity;
            long long p_wait = 0; const long long p_begin = clock64();
            for (int t0 = blockIdx.x; t0 < total_tiles; t0 += kP1Ahead * gridDim.x) {
#pragma unroll
                for (int d = 0; d < kP1Ahead; ++d) {
                    const int t = t0 + d * gridDim.x;
                    if (t >= total_tiles) break;
                    const int n = t / kP1TilesPerImg;
                    const P1Geom g = p1_geom(t, q_sy[d], a.pad);
                    const int word0 = (g.rlo * (kImg / 4)) & ~3;    // boxes start on 16-byte boundaries; the builders add (rlo * 84) % 16
                    int plane0 = n * a.cin;
                    if (a.ring_frames) {
                        // frame `lane` of image n's stack (channel_plane)
                        const int tt = n >= a.ring_B ? q_idx[d] + a.ring_nstep - 1 : q_idx[d] - 1;
                        int r = tt - (a.ring_stack - 1 - lane);
                        r = r < 0 ? 0 : r;
                        int slot = q_ep[d] + r;
                        while (slot >= cap) slot -= cap;
                        plane0 = slot * a.ring_frame_c;
                    }
                    fetch(t + kP1Ahead * gridDim.x, q_sy[d], q_idx[d], q_ep[d]);
                    const long long p0 = clock64();
                    P1_RELAXED_WAIT(rempty + rs, rphase ^ 1);
                    p_wait += clock64() - p0;
                    mbar_arrive_expect_tx(rfull + rs, nbytes);
                    tma_load_2d(smem_u32(raw_s + rs * kP1RawBytes + lane * planes_per_src * kP1RawSlot), &map, word0, plane0, rfull + rs);
                    if (++rs == kP1RawStages) { rs = 0; rphase ^= 1; }
                }
            }
            if (a.stamps && blockIdx.x == 0 && lane == 0) { a.stamps[9] = p_wait; a.stamps[10] = clock64() - p_begin; }
        }
    } else {
        // ------------------------------------------------ epilogue warps 16..23: lane quarter warp % 4, two warps per quarter on
        // alternate tiles (one warp per quarter needs ~1000 cycles per tile between the TMEM load, 80 arithmetic
        // instructions and its share of the issue slots; the UMMAs of a tile take 400)
        const int q = warp & 3, par = (warp - kBuildWarps - 1) >> 2;
        const int m = q * 32 + lane;
        const int r = m / kP1Pitch, x = m - r * kP1Pitch;
        float bias_r[32];
#pragma unroll
        for (int i = 0; i < 32; ++i) bias_r[i] = bias_s[i];
        int ord = par;
        for (int t = blockIdx.x + par * (int)gridDim.x; t < total_tiles; t += 2 * gridDim.x, ord += 2) {
            const int acc = ord % kP1Acc; const uint32_t acc_phase = (ord / kP1Acc) & 1;
            const int n = t / kP1TilesPerImg, y = (t - n * kP1TilesPerImg) * kP1Rows + r;
            mbar_wait<P1_HINT>(tfull + acc, acc_phase);
            tc_fence_after();
            float v[32];
            tmem_ld_32x32(tmem_base + ((uint32_t)(q * 32) << 16) + acc * 32, v);
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(tempty + acc);
            if (m >= kP1Live || x >= kPW || y >= kPW) continue;
            const long long row = (long long)n * DRQ_PLB + DRQ_GUARD + y * kPW + x;
            uint32_t packed[16];
#pragma unroll
            for (int i = 0; i < 16; ++i)
                packed[i] = pack_bf16x2(fmaxf(fmaf(v[2 * i], kC1Scale, bias_r[2 * i]), 0.f),
                                        fmaxf(fmaf(v[2 * i + 1], kC1Scale, bias_r[2 * i + 1]), 0.f));
#pragma unroll
            for (int c = 0; c < 4; ++c)
                *reinterpret_cast<uint4*>(a.out + (c * a.cs_out + row) * 8) =
                    make_uint4(packed[4 * c], packed[4 * c + 1], packed[4 * c + 2], packed[4 * c + 3]);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == kBuildWarps) tmem_dealloc(tmem_base, kP1Acc * 32);
}

// ---------------------------------------------------------------- data gradient
// d(pixels) of conv1 from its pre-ReLU gradient dY (WB bf16, K-major over co exactly as conv2's forward reads conv1's
// output): per tile of three output rows (positions p0 = 123 t .. p0 + 127 of the image, rows 123.. unused)
//   col[p][k] = sum_co dY[p][co] * W[co][k]                        M = 128 positions, N = 96 (k = 9c + tap), K = 32 co
// one UMMA pair (two K16 steps) into 96 TMEM columns.  The packed conv1 weights [12 k units][32 co][8 k] are the
// canonical MN-major B operand of this product (MN = k, K = co) as they stand.  Col2im in the epilogue: the tile's col
// goes through shared memory and every input pixel sums its <= 4 entries, taps (ky, kx) ascending (the carried row:
// ky = 2 of the previous tile first, then ky = 0 of this one).  A CTA takes whole
// images and their 14 tiles in order: tile t completes input rows 6t .. 6t+5; row 6t+6 also takes taps of the next
// tile, so its partial sum (ky = 2 of output row 3t+2) is carried in shared memory and the next tile adds its ky = 0
// taps to it.  Row 83 takes no tap and is written as +0.  Fixed order, no atomics, no global scratch.
constexpr int kDgTiles = 14;
constexpr int kDgColPitch = 97;                 // fp32 col row pitch in shared memory (conflict-free gathers)
constexpr int kDgThreads = 128;
constexpr int kDgABytes = 4 * kC1Tile * 16;     // [4 co blocks][128 positions][16 B]
constexpr size_t kDgOffA = kC1WBytes;
constexpr size_t kDgOffCol = kDgOffA + 2 * kDgABytes;
constexpr size_t kDgOffCarry = kDgOffCol + (size_t)kC1Tile * kDgColPitch * 4;
constexpr size_t kDgOffBars = kDgOffCarry + 2 * 10 * kImg * 4;
constexpr size_t kConv1DgradSmem = kDgOffBars + 4 * 8 + 16;

__global__ void __launch_bounds__(kDgThreads) conv1_dgrad_tc_kernel(const __nv_bfloat16* __restrict__ d, long long cs_d,
                                                                    const __nv_bfloat16* __restrict__ w_packed,
                                                                    float* __restrict__ dx, int n_images, int cin) {
    extern __shared__ __align__(128) uint8_t smem[];
    uint8_t* w_s = smem;
    uint8_t* a_s = smem + kDgOffA;
    float* col_s = reinterpret_cast<float*>(smem + kDgOffCol);
    float* carry_s = reinterpret_cast<float*>(smem + kDgOffCarry);      // [2][cin][84]
    uint64_t* full = reinterpret_cast<uint64_t*>(smem + kDgOffBars);   // [2]
    uint64_t* mma = full + 2;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(mma + 1);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

    if (tid == 0) {
        mbar_init(full, 1); mbar_init(full + 1, 1); mbar_init(mma, 1);
        fence_barrier_init();
    }
    if (warp == 0) {
        tmem_alloc(tmem_slot, 128);
        tmem_relinquish();
    }
    {
        const uint4* src = reinterpret_cast<const uint4*>(w_packed);
        for (int i = tid; i < kC1WBytes / 16; i += kDgThreads) reinterpret_cast<uint4*>(w_s)[i] = __ldg(src + i);
    }
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    // tile j of this CTA: image blockIdx.x + (j / 14) * gridDim.x, tile j % 14
    auto load = [&](int j) {
        const int n = blockIdx.x + (j / kDgTiles) * (int)gridDim.x, t = j % kDgTiles;
        const int s = j & 1;
        const long long row0 = (long long)n * DRQ_PLB + DRQ_GUARD + t * 3 * kPW;
        mbar_arrive_expect_tx(full + s, kDgABytes);
        for (int c = 0; c < 4; ++c)
            bulk_g2s(a_s + s * kDgABytes + c * kC1Tile * 16, d + (c * cs_d + row0) * 8, kC1Tile * 16, full + s);
    };
    const int my_images = blockIdx.x < n_images ? (n_images - 1 - (int)blockIdx.x) / (int)gridDim.x + 1 : 0;
    const int my_tiles = my_images * kDgTiles;
    if (tid == 0 && my_tiles > 0) load(0);
    const uint64_t da0 = make_smem_desc(smem_u32(a_s), kC1Tile * 16, 128);   // dY, K-major (K = co)
    const uint64_t db0 = make_smem_desc(smem_u32(w_s), 128, 512);            // W, MN-major (MN = k, K = co)
    constexpr uint32_t idesc = make_idesc_bf16(128, kC1K, false, true);

    for (int j = 0; j < my_tiles; ++j) {
        const int n = blockIdx.x + (j / kDgTiles) * (int)gridDim.x, t = j % kDgTiles;
        const int s = j & 1;
        // the other stage's UMMAs retired before the previous tile's epilogue started
        if (tid == 0 && j + 1 < my_tiles) load(j + 1);
        mbar_wait(full + s, (j >> 1) & 1);
        tc_fence_after();
        if (warp == 0) {
            if (elect_one()) {
#pragma unroll
                for (int ks = 0; ks < 2; ++ks)
                    umma_bf16(tmem_base, da0 + (uint64_t)(s * (kDgABytes >> 4) + ks * 2 * kC1Tile), db0 + (uint64_t)(ks * 16),
                              idesc, ks ? 1u : 0u);
                umma_commit(mma);
            }
            __syncwarp();
        }
        mbar_wait(mma, j & 1);
        tc_fence_after();
#pragma unroll
        for (int c0 = 0; c0 < kC1K; c0 += 32) {
            float v[32];
            tmem_ld_32x32(tmem_base + ((uint32_t)(warp * 32) << 16) + c0, v);
            float* dst = col_s + (warp * 32 + lane) * kDgColPitch + c0;
#pragma unroll
            for (int i = 0; i < 32; ++i) dst[i] = v[i];
        }
        tc_fence_before();
        __syncthreads();
        // col2im of output rows oy0 .. oy0 + R - 1 into input rows 2 oy0 .. 2 oy0 + 2R (the last one carried unless t = 13)
        const int oy0 = 3 * t, R = min(3, kPW - oy0), nrows = 2 * R + 1;
        const float* carry_in = carry_s + ((t + 1) & 1) * (10 * kImg);
        float* carry_out = carry_s + (t & 1) * (10 * kImg);
        float* dx_n = dx + (long long)n * cin * (kImg * kImg);
        for (int i = tid; i < cin * nrows * kImg; i += kDgThreads) {
            const int c = i / (nrows * kImg), rem = i - c * (nrows * kImg), rl = rem / kImg, ix = rem - rl * kImg;
            const int iy = 2 * oy0 + rl;
            float acc = (rl == 0 && t > 0) ? carry_in[c * kImg + ix] : 0.f;
#pragma unroll
            for (int ky = 0; ky < 3; ++ky) {
                const int oy2 = rl - ky;                       // 2 (oy - oy0)
                if (oy2 < 0 || (oy2 & 1) || (oy2 >> 1) >= R) continue;
#pragma unroll
                for (int kx = 0; kx < 3; ++kx) {
                    const int ox2 = ix - kx;
                    if (ox2 < 0 || (ox2 & 1) || (ox2 >> 1) >= kPW) continue;
                    acc += col_s[((oy2 >> 1) * kPW + (ox2 >> 1)) * kDgColPitch + c * 9 + ky * 3 + kx];
                }
            }
            if (rl == nrows - 1 && t < kDgTiles - 1) carry_out[c * kImg + ix] = acc;
            else dx_n[(c * kImg + iy) * kImg + ix] = __fdiv_rn(acc, 255.0f);
        }
        if (t == kDgTiles - 1)
            for (int i = tid; i < cin * kImg; i += kDgThreads)
                dx_n[((i / kImg) * kImg + kImg - 1) * kImg + i % kImg] = 0.f;
        tc_fence_before();
        __syncthreads();                 // col_s and the carry are re-written by the next tile; TMEM is re-accumulated
        tc_fence_after();
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem_base, 128);
}

constexpr size_t kConv1PlanesSmem = kP1WBytes + 128 + kP1RawStages * kP1RawBytes + kP1Stages * kP1StageBytes + 128 +
                                    (2 * kP1Stages + 2 * kP1Acc + 2 * kP1RawStages) * 8 + 16;
static_assert(kC1WBytes + 128 <= kP1RawStages * kP1RawBytes, "the packed weights are staged in the raw-row buffer");
// 0 = im2col kernel, 1 (default) = parity planes for launches that fill the machine (>= 48 images, the same rule and the
// same kernel family as the conv3x3 forward that follows it: csrc/conv_tc.cu), 2 = parity planes always (tests)
static int g_conv1_planes = 1;
constexpr int kP1MinImages = 48;

constexpr size_t kConv1FwdSmem = kC1WBytes + 128 + 4 * kC1InBytes + kC1RawStages * kC1RawBytes + kC1Stages * kC1ABytes +
                                 (3 * kC1Stages + 2 * kC1Acc + 1 + 2 * kC1RawStages) * 8 + 16;
// wgrad: + one extra d-tile worth of tail padding (rows 32..63 of the M=64 operand read 4 blocks past the tile)
constexpr size_t kConv1WgSmem = kC1WBytes + 128 + 4 * kC1InBytes + kC1RawStages * kC1RawBytes + kC1Stages * (kC1ABytes + kC1DBytes) +
                                kC1DBytes + (3 * kC1Stages + 2 * kC1Acc + 1 + 2 * kC1RawStages) * 8 + 16;

}  // namespace drq

using namespace drq;

extern "C" {

int drq_debug_conv1_stamps(int64_t* buf) { g_c1_stamps = reinterpret_cast<long long*>(buf); return DRQ_OK; }

int drq_set_conv1_planes(int on) {
    const int prev = g_conv1_planes;
    if (on >= 0 && on <= 2) g_conv1_planes = on;
    return prev;
}

int64_t drq_conv1_w_packed_elems(void) { return kC1Units * 32 * 8 + 64; }

int drq_pack_conv1_w_bf16(const float* w, const float* bias, uint16_t* out, int cin, void* stream) {
    DRQ_REQUIRE(w && bias && out && cin > 0 && cin * 9 + 1 <= kC1K, "pack_conv1_w: bad args (cin <= 10)");
    pack_conv1_w_kernel<<<1, 256, 0, as_stream(stream)>>>(w, bias, reinterpret_cast<__nv_bfloat16*>(out), cin);
    return check_launch("pack_conv1_w_kernel");
}

// the ring view of a batch as kernel arguments
static int ring_args(Conv1TcArgs& a, const drq_ring_src* src, int B, int N) {
    DRQ_REQUIRE(src && src->frames && src->ep_start && src->idx, "conv1_*_ring: incomplete ring source");
    DRQ_REQUIRE(src->capacity > 0 && src->frame_c > 0 && src->stack > 0 && src->nstep > 0, "conv1_*_ring: bad ring dims");
    // the row producers compute the ring slot in 32 bits: episode start + row < 2 * capacity
    DRQ_REQUIRE(src->capacity <= (1ll << 30), "conv1_*_ring: ring capacity above 2^30 slots");
    DRQ_REQUIRE(B > 0 && N > 0 && N <= 2 * B, "conv1_*_ring: N images must be B (obs) or 2B (obs | next_obs)");
    DRQ_REQUIRE(((uintptr_t)src->frames % 16) == 0, "conv1_*_ring: ring frames must be 16-byte aligned");
    a.ring_frames = src->frames; a.ring_ep_start = src->ep_start; a.ring_idx = src->idx;
    a.ring_capacity = src->capacity; a.ring_B = B; a.ring_nstep = src->nstep; a.ring_stack = src->stack;
    a.ring_frame_c = src->frame_c;
    a.cin = src->frame_c * src->stack;
    return DRQ_OK;
}

static int conv1_fwd_launch(Conv1TcArgs& a, const int32_t* shift, const uint16_t* w_packed, uint16_t* out, int N, int pad,
                            cudaStream_t stream);
static int conv1_wgrad_launch(Conv1TcArgs& a, const int32_t* shift, const uint16_t* dpre, float* partial, float* dw, float* db,
                              int N, int pad, cudaStream_t stream);

int drq_conv1_fwd_bf16_ring(const drq_ring_src* src, int B, const int32_t* shift, const uint16_t* w_packed,
                            uint16_t* out, int N, int pad, void* stream) {
    Conv1TcArgs a{};
    if (int rc = ring_args(a, src, B, N)) return rc;
    return conv1_fwd_launch(a, shift, w_packed, out, N, pad, as_stream(stream));
}

int drq_conv1_wgrad_bf16_ring(const drq_ring_src* src, int B, const int32_t* shift, const uint16_t* dpre,
                              float* partial, float* dw, float* db, int N, int pad, void* stream) {
    Conv1TcArgs a{};
    if (int rc = ring_args(a, src, B, N)) return rc;
    return conv1_wgrad_launch(a, shift, dpre, partial, dw, db, N, pad, as_stream(stream));
}

int drq_conv1_fwd_bf16(const uint8_t* obs, const int32_t* shift, const uint16_t* w_packed, uint16_t* out, int N,
                       int cin, int pad, void* stream) {
    DRQ_REQUIRE(obs, "conv1_fwd_bf16: null pointer");
    Conv1TcArgs a{};
    a.obs = obs; a.cin = cin;
    return conv1_fwd_launch(a, shift, w_packed, out, N, pad, as_stream(stream));
}

static int conv1_fwd_launch(Conv1TcArgs& a, const int32_t* shift, const uint16_t* w_packed, uint16_t* out, int N, int pad,
                            cudaStream_t stream) {
    const int cin = a.cin;
    DRQ_REQUIRE(w_packed && out, "conv1_fwd_bf16: null pointer");
    DRQ_REQUIRE(N > 0 && cin > 0 && cin * 9 + 1 <= kC1K && pad >= 0 && pad <= 4, "conv1_fwd_bf16: bad dims (cin <= 10, pad <= 4)");
    if (int rc = ensure_smem((const void*)conv1_tc_kernel<false, 9>, kConv1FwdSmem, "conv1_fwd_bf16")) return rc;
    if (int rc = ensure_smem((const void*)conv1_tc_kernel<false, 0>, kConv1FwdSmem, "conv1_fwd_bf16")) return rc;
    a.shift = shift; a.pad = pad;
    a.w = reinterpret_cast<const __nv_bfloat16*>(w_packed);
    a.out = reinterpret_cast<__nv_bfloat16*>(out);
    a.cs_out = (long long)N * DRQ_PLB + DRQ_WB_SLACK;
    a.n_images = N;
    a.stamps = g_c1_stamps;
    if (g_conv1_planes == 2 || (g_conv1_planes == 1 && N >= kP1MinImages)) {
        typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                     const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
        EncodeFn encode = reinterpret_cast<EncodeFn>(tensor_map_encoder());
        DRQ_REQUIRE(encode, "conv1_fwd_bf16: cuTensorMapEncodeTiled is not available");
        // the source as (words of a channel plane) x (channel planes); a box = the tile's source rows of the planes of one
        // stack (gathered) or of one ring frame
        const bool ring = a.ring_frames != nullptr;
        const void* base = ring ? (const void*)a.ring_frames : (const void*)a.obs;
        const long long planes = ring ? a.ring_capacity * a.ring_frame_c : (long long)N * cin;
        const int box_planes = ring ? a.ring_frame_c : cin;
        DRQ_REQUIRE(((uintptr_t)base % 16) == 0 && planes < (1ll << 31) && box_planes * a.ring_stack * (ring ? 1 : 0) <= 10 && box_planes <= 10,
                    "conv1_fwd_bf16: source must be 16-byte aligned, <= 10 channels");
        CUtensorMap map;
        const cuuint64_t gdim[2] = {(cuuint64_t)(kImg * kImg / 4), (cuuint64_t)planes};
        const cuuint64_t gstr[1] = {(cuuint64_t)(kImg * kImg)};
        const cuuint32_t box[2] = {(cuuint32_t)kP1BoxWords, (cuuint32_t)box_planes};
        const cuuint32_t estr[2] = {1, 1};
        const CUresult r = encode(&map, CU_TENSOR_MAP_DATA_TYPE_UINT32, 2, const_cast<void*>(base), gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                                  CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        DRQ_REQUIRE(r == CUDA_SUCCESS, "conv1_fwd_bf16: cuTensorMapEncodeTiled failed (%d)", (int)r);
        if (int rc = ensure_smem((const void*)conv1_planes_kernel<9>, kConv1PlanesSmem, "conv1_fwd_bf16")) return rc;
        if (int rc = ensure_smem((const void*)conv1_planes_kernel<0>, kConv1PlanesSmem, "conv1_fwd_bf16")) return rc;
        const int ptiles = N * kP1TilesPerImg;
        const int G = ptiles < sm_budget() ? ptiles : sm_budget();
        if (cin == 9) conv1_planes_kernel<9><<<G, kP1Threads, kConv1PlanesSmem, stream>>>(map, a);
        else conv1_planes_kernel<0><<<G, kP1Threads, kConv1PlanesSmem, stream>>>(map, a);
        return check_launch("conv1_planes_kernel");
    }
    const int tiles = N * 14;
    const int G = tiles < sm_budget() ? tiles : sm_budget();
    if (cin == 9) conv1_tc_kernel<false, 9><<<G, kC1Threads, kConv1FwdSmem, stream>>>(a);
    else conv1_tc_kernel<false, 0><<<G, kC1Threads, kConv1FwdSmem, stream>>>(a);
    return check_launch("conv1_tc_kernel<fwd>");
}

int64_t drq_conv1_wgrad_bf16_ws_floats(void) { return 148ll * 32 * kC1K; }

int drq_conv1_wgrad_bf16(const uint8_t* obs, const int32_t* shift, const uint16_t* dpre, float* partial,
                         float* dw, float* db, int N, int cin, int pad, void* stream) {
    DRQ_REQUIRE(obs, "conv1_wgrad_bf16: null pointer");
    Conv1TcArgs a{};
    a.obs = obs; a.cin = cin;
    return conv1_wgrad_launch(a, shift, dpre, partial, dw, db, N, pad, as_stream(stream));
}

static int conv1_wgrad_launch(Conv1TcArgs& a, const int32_t* shift, const uint16_t* dpre, float* partial, float* dw, float* db,
                              int N, int pad, cudaStream_t stream) {
    const int cin = a.cin;
    DRQ_REQUIRE(dpre && partial && (dw != nullptr) == (db != nullptr), "conv1_wgrad_bf16: null pointer");
    DRQ_REQUIRE(N > 0 && cin > 0 && cin * 9 + 1 <= kC1K && pad >= 0 && pad <= 4, "conv1_wgrad_bf16: bad dims (cin <= 10, pad <= 4)");
    if (int rc = ensure_smem((const void*)conv1_tc_kernel<true, 9>, kConv1WgSmem, "conv1_wgrad_bf16")) return rc;
    if (int rc = ensure_smem((const void*)conv1_tc_kernel<true, 0>, kConv1WgSmem, "conv1_wgrad_bf16")) return rc;
    a.shift = shift; a.pad = pad;
    a.d = reinterpret_cast<const __nv_bfloat16*>(dpre);
    a.cs_d = (long long)N * DRQ_PLB + DRQ_WB_SLACK;
    a.partial = partial;
    a.n_images = N;
    const int G = conv1_wgrad_ctas(N);
    if (cin == 9) conv1_tc_kernel<true, 9><<<G, kC1Threads, kConv1WgSmem, stream>>>(a);
    else conv1_tc_kernel<true, 0><<<G, kC1Threads, kConv1WgSmem, stream>>>(a);
    if (int rc = check_launch("conv1_tc_kernel<wgrad>")) return rc;
    if (!dw) return DRQ_OK;                                   // partials only: reduced later by drq_conv_wgrad_reduce_multi
    conv1_wgrad_reduce_kernel<<<kC1ReduceBlocks, 256, 0, stream>>>(partial, G, cin, dw, db);
    return check_launch("conv1_wgrad_reduce_kernel");
}

int drq_conv1_dgrad_bf16(const uint16_t* dpre, const uint16_t* w_packed, float* dx, int N, int cin, void* stream) {
    DRQ_REQUIRE(dpre && w_packed && dx, "conv1_dgrad_bf16: null pointer");
    DRQ_REQUIRE(N >= 0 && cin > 0 && cin * 9 + 1 <= kC1K, "conv1_dgrad_bf16: bad dims (cin <= 10)");
    if (N == 0) return DRQ_OK;
    if (int rc = ensure_smem((const void*)conv1_dgrad_tc_kernel, kConv1DgradSmem, "conv1_dgrad_bf16")) return rc;
    const int G = N < 2 * sm_budget() ? N : 2 * sm_budget();
    conv1_dgrad_tc_kernel<<<G, kDgThreads, kConv1DgradSmem, as_stream(stream)>>>(
        reinterpret_cast<const __nv_bfloat16*>(dpre), (long long)N * DRQ_PLB + DRQ_WB_SLACK,
        reinterpret_cast<const __nv_bfloat16*>(w_packed), dx, N, cin);
    return check_launch("conv1_dgrad_tc_kernel");
}

int drq_conv1_fwd_bf16_from_f32(const float* obs, const uint16_t* w_packed, uint16_t* out, int N, int cin, void* stream) {
    DRQ_REQUIRE(obs && w_packed && out, "conv1_fwd_bf16_from_f32: null pointer");
    DRQ_REQUIRE(N > 0 && cin > 0 && cin * 9 + 1 <= kC1K, "conv1_fwd_bf16_from_f32: bad dims (cin <= 10)");
    if (int rc = ensure_smem((const void*)conv1_tc_kernel<false, 0, true>, kConv1FwdSmem, "conv1_fwd_bf16_from_f32")) return rc;
    Conv1TcArgs a{};
    a.fobs = obs; a.cin = cin;
    a.w = reinterpret_cast<const __nv_bfloat16*>(w_packed);
    a.out = reinterpret_cast<__nv_bfloat16*>(out);
    a.cs_out = (long long)N * DRQ_PLB + DRQ_WB_SLACK;
    a.n_images = N;
    const int tiles = N * 14;
    const int G = tiles < sm_budget() ? tiles : sm_budget();
    conv1_tc_kernel<false, 0, true><<<G, kC1Threads, kConv1FwdSmem, as_stream(stream)>>>(a);
    return check_launch("conv1_tc_kernel<fwd, f32 pixels>");
}

int drq_conv1_wgrad_bf16_from_f32(const float* obs, const uint16_t* dpre, float* partial, float* dw, float* db, int N,
                                  int cin, void* stream) {
    DRQ_REQUIRE(obs && dpre && partial && dw && db, "conv1_wgrad_bf16_from_f32: null pointer");
    DRQ_REQUIRE(N > 0 && cin > 0 && cin * 9 + 1 <= kC1K, "conv1_wgrad_bf16_from_f32: bad dims (cin <= 10)");
    if (int rc = ensure_smem((const void*)conv1_tc_kernel<true, 0, true>, kConv1WgSmem, "conv1_wgrad_bf16_from_f32")) return rc;
    Conv1TcArgs a{};
    a.fobs = obs; a.cin = cin;
    a.d = reinterpret_cast<const __nv_bfloat16*>(dpre);
    a.cs_d = (long long)N * DRQ_PLB + DRQ_WB_SLACK;
    a.partial = partial;
    a.n_images = N;
    const int G = conv1_wgrad_ctas(N);
    conv1_tc_kernel<true, 0, true><<<G, kC1Threads, kConv1WgSmem, as_stream(stream)>>>(a);
    if (int rc = check_launch("conv1_tc_kernel<wgrad, f32 pixels>")) return rc;
    conv1_wgrad_reduce_kernel<<<kC1ReduceBlocks, 256, 0, as_stream(stream)>>>(partial, G, cin, dw, db);
    return check_launch("conv1_wgrad_reduce_kernel");
}

}  // extern "C"

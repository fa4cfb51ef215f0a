// 3x3 stride-1 convolutions of Encoder (drqv2.py:56-59), forward and data gradient, as implicit GEMMs whose accumulator
// row is a COLUMN OF FOUR output pixels (tcgen05 + TMEM + tensor-map TMA, sm_100a only).
//
// Why: a tcgen05.mma M128 K16 costs 44.6 cycles at N = 32, 48.1 at N = 64, ~56 at N = 96 and 64.1 at N = 128
// (tools/ub/ub_mma.cu: the operand bytes read from shared memory, (A + B) / 128 B per cycle), so the one-pixel-per-row
// kernel of conv_tc.cu (N = 32 output channels, 18 UMMAs per 128 pixels = 6.3 cycles per pixel) cannot pass 36 % of the
// tensor peak.  Here accumulator row m is the pixel column (4i+oy, x), oy = 0..3, its 128 columns are (oy, co), and the
// contraction runs over the 6x3 input window of that column: window row wy reaches the outputs oy with 0 <= wy-oy <= 2 -
// one, two or three ADJACENT column groups - so every window element is one UMMA of N = 32 / 64 / 96 with no padding:
// 36 UMMAs per 128 columns = 512 pixels, 1784 cycles = 3.5 cycles per pixel.
//
// The activations stay in the WB layout (conv_tc.cu).  Window row wy of pixel column (i, x) is image row 4i+wy, i.e. row
// block i + wy/4 of the "row plane" wy%4, and a row plane is whole image rows (41 pixels x 16 B = 656 contiguous bytes per
// channel block): one 5-d tensor-map TMA per tile - box (656 B, 4 row blocks, 4 planes, 1 image, 4 channel blocks) -
// lands the [channel block][plane][row block][x] windows of three block rows in shared memory, where window element
// (wy, wx) of 128 consecutive pixel columns is plane wy%4 at the constant row offset (wy/4)*41 + wx: one K-major
// no-swizzle descriptor plus an offset per UMMA, as in conv_tc.cu.  (A first version split 2x2 output blocks into four
// row/column parity planes with 16-byte cp.async copies: correct, and slower than conv_tc.cu - 2432 LSU requests per
// tile kept a loader warp issuing for 2500 cycles per 1800-cycle tile; git history, DESIGN.md §6.)  Row blocks outside
// the image are zero-filled by the TMA; the data gradient relies, like conv_tc.cu, on the gradient buffer being zero
// outside its valid region.
//
// The weights arrive in the compact operand layout of pack_conv_w_elem ([tap*4 + k/8][n][k%8], 18 KB) and are expanded
// per CTA into the 18 per-window-element B operands (72 KB of shared memory) while the first tiles load.
//
// Tiles are per image: three block rows = 123 pixel columns of the 41-wide rows (5 accumulator rows idle).
// Warp roles (320 threads, one CTA per SM): warp 0 = UMMA issuer, warp 1 = TMA producer, warps 2..9 = epilogue (TMEM
// lane quarter = warp % 4, output rows oy in {0,1} or {2,3} = (warp - 2) / 4).
#include <cuda.h>

#include "tc_common.cuh"

namespace drq {

DRQ_TRAP_NOTE_HOOK(trap_note_conv4x1)

using namespace tc;

namespace c4 {

constexpr int kPLB = DRQ_PLB;
constexpr int kGuard = DRQ_GUARD;
constexpr int kRowBytes = kPW * 16;           // one image row of one channel block
constexpr int kBoxRows = 4;                   // row blocks per box: three block rows of outputs + the window's extra one
constexpr int kTileRows = 3;
constexpr int kTileCols = kTileRows * kPW;    // 123 live accumulator rows
constexpr int kRegion = kBoxRows * kRowBytes; // bytes of one (channel block, plane)
constexpr int kStageBytes = 16 * kRegion;     // 41,984
constexpr int kStages = 3;
constexpr int kAcc = 4;                       // accumulator ring: 4 x 128 TMEM columns
constexpr int kWUnits = 3 * 12 * 128;         // 16-byte units of the expanded weights: per wx, sum over wy of 4 K units x 32 * cnt(wy)
constexpr int kWBytes = kWUnits * 16;
constexpr int kThreads = 10 * 32;
constexpr int kExpanders = kThreads - 32;     // everyone but the producer warp
constexpr int kRowBlocks = 11;                // row blocks of a 41-row image (rows 0..43: the tail lies in the next image's guard)

struct Args {
    const __nv_bfloat16* w;                         // compact [36][32][8]
    const float* bias;                              // fwd
    const __nv_bfloat16* mask; long long cs_mask;   // dgrad: the layer's input activation (WB)
    __nv_bfloat16* out; long long cs_out;
    int n_images, tiles_per_image, total_tiles;
    int h_out;                                      // valid height = width of the output
    int out_mode;                                   // 0 WB, 1 compact NHWC, 2 TB features
    uint32_t m_tiles;                               // floor(2^32 / tiles_per_image) + 1
    long long feat_rpad; int feat_half, feat_half_row;
    long long* stamps;                              // drq_debug_conv4x1_stamps: per-role clock64 totals of block 0, or null
};

__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }

__device__ __forceinline__ void tma_load_5d(uint32_t dst, const CUtensorMap* map, int c0, int c1, int c2, int c3, int c4, uint64_t* bar) {
    asm volatile("cp.async.bulk.tensor.5d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5, %6}], [%7];"
                 ::"r"(dst), "l"(map), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4), "r"(smem_u32(bar)) : "memory");
}

// window row wy reaches the outputs oy_min(wy) .. oy_min(wy) + cnt(wy) - 1
__host__ __device__ constexpr int win_cnt(int wy) { return wy == 0 || wy == 5 ? 1 : wy == 1 || wy == 4 ? 2 : 3; }
__host__ __device__ constexpr int win_oy0(int wy) { return wy < 2 ? 0 : wy - 2; }
__host__ __device__ constexpr int win_prefix(int wy) { return wy == 0 ? 0 : wy == 1 ? 1 : wy == 2 ? 3 : wy == 3 ? 6 : wy == 4 ? 9 : 11; }
// first 16-byte unit of the B operand of window element (wy, wx): [4 K units][32 * cnt n][8]
__host__ __device__ constexpr int win_unit0(int wy, int wx) { return wx * 1536 + 128 * win_prefix(wy); }

template <bool DGRAD>
__device__ __forceinline__ void expand_weights(const __nv_bfloat16* __restrict__ w, uint8_t* w_s, int e) {
    const uint4* src = reinterpret_cast<const uint4*>(w);
    // unrolled: the 16 units of a thread are independent address chains (a lone warp per scheduler runs a dependent
    // chain at ~5 cycles per instruction)
#pragma unroll
    for (int k = 0; k < kWUnits / kExpanders; ++k) {
        const int u = e + k * kExpanders;
        const int wx = u / 1536, rem = u - wx * 1536;
        const int s = rem >> 7;                                     // 0..11 = prefix slot
        const int wy = s < 1 ? 0 : s < 3 ? 1 : s < 6 ? 2 : s < 9 ? 3 : s < 11 ? 4 : 5;
        const int cnt = win_cnt(wy), n32 = 32 * cnt;
        const int r2 = rem - 128 * win_prefix(wy);
        const int ku = r2 / n32, n = r2 - ku * n32;
        const int oy = win_oy0(wy) + (n >> 5), co = n & 31;
        const int dy = DGRAD ? oy + 2 - wy : wy - oy;
        const int dx = DGRAD ? 2 - wx : wx;
        cp_async16(smem_u32(w_s) + u * 16, src + ((dy * 3 + dx) * 4 + ku) * 32 + co);
    }
    cp_async_commit();
    cp_async_wait_all();
}
static_assert(kWUnits % kExpanders == 0, "expansion loop has no tail");

template <bool DGRAD>
__global__ void __maxnreg__(128) conv4x1_tc_kernel(const __grid_constant__ CUtensorMap map, const Args a) {
    extern __shared__ __align__(128) uint8_t smem[];
    uint8_t* w_s = smem;
    uint8_t* a_s = smem + kWBytes;
    uint64_t* bars = reinterpret_cast<uint64_t*>(a_s + kStages * kStageBytes + 128);
    uint64_t* full = bars;
    uint64_t* empty = bars + kStages;
    uint64_t* tfull = bars + 2 * kStages;
    uint64_t* tempty = bars + 2 * kStages + kAcc;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * kStages + 2 * kAcc);
    float* bias_s = reinterpret_cast<float*>(tmem_slot + 4);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) {
        for (int i = 0; i < kStages; ++i) { mbar_init(full + i, 1); mbar_init(empty + i, 1); }
        for (int i = 0; i < kAcc; ++i) { mbar_init(tfull + i, 1); mbar_init(tempty + i, 8); }
        fence_barrier_init();
    }
    if (warp == 0) {
        tmem_alloc(tmem_slot, kAcc * 128);
        tmem_relinquish();
    }
    if (!DGRAD && threadIdx.x < 32) bias_s[threadIdx.x] = a.bias[threadIdx.x];
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 1) {
        // ------------------------------------------------ TMA producer: one box per tile
        if (lane == 0) {
            int stage = 0; uint32_t phase = 0;
            long long st_empty = 0;
            const long long st_begin = clock64();
            for (int t = blockIdx.x; t < a.total_tiles; t += gridDim.x) {
                const int n = (int)__umulhi((uint32_t)t, a.m_tiles);
                const int i0 = (t - n * a.tiles_per_image) * kTileRows;
                const long long c0 = clock64();
                mbar_wait(empty + stage, phase ^ 1);
                st_empty += clock64() - c0;
                mbar_arrive_expect_tx(full + stage, kStageBytes);
                tma_load_5d(smem_u32(a_s + stage * kStageBytes), &map, 0, i0 - (DGRAD ? 1 : 0), 0, n, 0, full + stage);
                if (++stage == kStages) { stage = 0; phase ^= 1; }
            }
            if (a.stamps && blockIdx.x == 0) { a.stamps[0] = st_empty; a.stamps[3] = clock64() - st_begin; }
        }
        __syncwarp();
    } else {
        // ------------------------------------------------ everyone else first expands the weights
        expand_weights<DGRAD>(a.w, w_s, warp == 0 ? lane : threadIdx.x - 32);
        fence_proxy_async();
        asm volatile("bar.sync 1, %0;" ::"n"(kExpanders) : "memory");
        if (warp == 0) {
            // -------------------------------------------- UMMA issuer
            // A: K-major, 16-byte K units (channel blocks) 4 regions apart; B: K-major, K units 32 * cnt rows apart
            const uint64_t da0 = make_smem_desc(smem_u32(a_s), 4 * kRegion, 128);
            const uint64_t db32 = make_smem_desc(smem_u32(w_s), 32 * 16, 128);
            const uint64_t db64 = make_smem_desc(smem_u32(w_s), 64 * 16, 128);
            const uint64_t db96 = make_smem_desc(smem_u32(w_s), 96 * 16, 128);
            constexpr uint32_t idesc32 = make_idesc_bf16(128, 32, false, false);
            constexpr uint32_t idesc64 = make_idesc_bf16(128, 64, false, false);
            constexpr uint32_t idesc96 = make_idesc_bf16(128, 96, false, false);
            int stage = 0; uint32_t phase = 0; int acc = 0; uint32_t acc_phase = 0;
            long long st_tempty = 0, st_full = 0, st_mma = 0;
            const long long st_begin = clock64();
            for (int t = blockIdx.x; t < a.total_tiles; t += gridDim.x) {
                const long long c0 = clock64();
                mbar_wait(tempty + acc, acc_phase ^ 1);
                const long long c1 = clock64();
                mbar_wait(full + stage, phase);
                const long long c2 = clock64();
                st_tempty += c1 - c0; st_full += c2 - c1;
                tc_fence_after();
                if (elect_one()) {
                    const uint64_t da = da0 + (uint64_t)(stage * (kStageBytes >> 4));
                    const uint32_t d_tmem = tmem_base + acc * 128;
                    // wy = 2 writes columns 0..95 first, wy = 5 columns 96..127; everything else accumulates
#pragma unroll
                    for (int o = 0; o < 6; ++o) {
                        const int wy = o == 0 ? 2 : o == 1 ? 5 : o == 2 ? 3 : o == 3 ? 1 : o == 4 ? 4 : 0;
                        // forward: image row 4i+wy = row block i + wy/4 of plane wy%4, columns x..x+2
                        // data gradient: gradient row 4i-2+wy = row block i-1 + (wy>=2) of plane (wy+2)%4 (the box starts one row
                        // block earlier), columns x-2..x
                        const int plane = DGRAD ? (wy + 2) & 3 : wy & 3;
                        const int down = DGRAD ? (wy >= 2) : (wy >> 2);
                        const int cnt = win_cnt(wy);
                        const uint64_t dbn = cnt == 1 ? db32 : cnt == 2 ? db64 : db96;
                        const uint32_t idesc = cnt == 1 ? idesc32 : cnt == 2 ? idesc64 : idesc96;
#pragma unroll
                        for (int wx = 0; wx < 3; ++wx)
#pragma unroll
                            for (int h = 0; h < 2; ++h)
                                umma_bf16(d_tmem + 32 * win_oy0(wy),
                                          da + (uint64_t)(int64_t)(plane * (kRegion >> 4) + down * kPW + wx - (DGRAD ? 2 : 0) + h * 2 * 4 * (kRegion >> 4)),
                                          dbn + (uint64_t)(win_unit0(wy, wx) + h * 2 * 32 * cnt), idesc, (o < 2 && wx == 0 && h == 0) ? 0u : 1u);
                    }
                    umma_commit(empty + stage);
                    umma_commit(tfull + acc);
                }
                __syncwarp();
                st_mma += clock64() - c2;
                if (++stage == kStages) { stage = 0; phase ^= 1; }
                if (++acc == kAcc) { acc = 0; acc_phase ^= 1; }
            }
            if (a.stamps && blockIdx.x == 0 && lane == 0) {
                a.stamps[4] = st_tempty; a.stamps[5] = st_full; a.stamps[6] = st_mma; a.stamps[7] = clock64() - st_begin;
            }
        } else {
            // -------------------------------------------- epilogue: TMEM lane quarter q, output rows oy = 2*half, 2*half + 1
            const int q = warp & 3, half = (warp - 2) >> 2;
            const int m = q * 32 + lane;
            const int r = (m >= kPW) + (m >= 2 * kPW), x = m - r * kPW;
            const bool live = m < kTileCols;
            int acc = 0; uint32_t acc_phase = 0;
            float bias_r[DGRAD ? 1 : 32];
            if (!DGRAD) {
#pragma unroll
                for (int i = 0; i < 32; ++i) bias_r[i] = bias_s[i];
            }
            long long st_tfull = 0, st_ld = 0, st_rest = 0;
            const long long st_begin = clock64();
            long long e_prev = st_begin;
            // data gradient: the ReLU mask (the layer's input activation at the output pixels) of tile t is fetched one tile
            // ahead - issued after the previous tile's accumulator has been read, consumed after this tile's
            uint4 mk[DGRAD ? 2 : 1][4], mk_next[DGRAD ? 2 : 1][4];
            auto load_mask = [&](int t, uint4 (&m4)[DGRAD ? 2 : 1][4]) {
                if (t >= a.total_tiles) return;
                const int n = (int)__umulhi((uint32_t)t, a.m_tiles);
                const int y0 = 4 * ((t - n * a.tiles_per_image) * kTileRows + r) + 2 * half;
                const long long row0 = (long long)n * kPLB + kGuard + y0 * kPW + x;
                const bool colok = live && x < a.h_out;
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    m4[0][c] = (colok && y0 < a.h_out) ? __ldg(reinterpret_cast<const uint4*>(a.mask + (c * a.cs_mask + row0) * 8)) : make_uint4(0, 0, 0, 0);
                    m4[DGRAD ? 1 : 0][c] = (colok && y0 + 1 < a.h_out) ? __ldg(reinterpret_cast<const uint4*>(a.mask + (c * a.cs_mask + row0 + kPW) * 8))
                                                                       : make_uint4(0, 0, 0, 0);
                }
            };
            if (DGRAD) load_mask(blockIdx.x, mk_next);
            for (int t = blockIdx.x; t < a.total_tiles; t += gridDim.x) {
                const int n = (int)__umulhi((uint32_t)t, a.m_tiles);
                const int i0 = (t - n * a.tiles_per_image) * kTileRows;
                const int y0 = 4 * (i0 + r) + 2 * half;
                const long long row0 = (long long)n * kPLB + kGuard + y0 * kPW + x;
                // data gradient: every column of a valid row is written (zeros beyond the valid width: the next layer's
                // windows read them); forward: valid pixels only
                const bool ok0 = live && y0 < a.h_out && (DGRAD || x < a.h_out);
                const bool ok1 = live && y0 + 1 < a.h_out && (DGRAD || x < a.h_out);
                if (DGRAD) {
#pragma unroll
                    for (int c = 0; c < 4; ++c) { mk[0][c] = mk_next[0][c]; mk[DGRAD ? 1 : 0][c] = mk_next[DGRAD ? 1 : 0][c]; }
                }
                const long long e0 = clock64();
                mbar_wait(tfull + acc, acc_phase);
                const long long e1 = clock64();
                st_rest += e0 - e_prev; st_tfull += e1 - e0;
                tc_fence_after();
                uint32_t raw[2][32];
                const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + acc * 128 + half * 64;
                tmem_ld_32x32_raw(taddr, raw[0]);
                tmem_ld_32x32_raw(taddr + 32, raw[1]);
                tmem_wait_ld();
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(tempty + acc);
                if (++acc == kAcc) { acc = 0; acc_phase ^= 1; }
                e_prev = clock64();
                st_ld += e_prev - e1;
                if (DGRAD) load_mask(t + gridDim.x, mk_next);

#pragma unroll
                for (int o = 0; o < 2; ++o) {
                    if (!(o ? ok1 : ok0)) continue;
                    uint32_t packed[16];
                    if (!DGRAD) {
#pragma unroll
                        for (int k = 0; k < 16; ++k)
                            packed[k] = pack_bf16x2(fmaxf(__uint_as_float(raw[o][2 * k]) + bias_r[DGRAD ? 0 : 2 * k], 0.f),
                                                    fmaxf(__uint_as_float(raw[o][2 * k + 1]) + bias_r[DGRAD ? 0 : 2 * k + 1], 0.f));
                    } else {
#pragma unroll
                        for (int c = 0; c < 4; ++c) {
                            const uint32_t mw[4] = {mk[DGRAD ? o : 0][c].x, mk[DGRAD ? o : 0][c].y, mk[DGRAD ? o : 0][c].z, mk[DGRAD ? o : 0][c].w};
#pragma unroll
                            for (int k = 0; k < 4; ++k)
                                packed[4 * c + k] = pack_bf16x2(bf16_lo(mw[k]) > 0.f ? __uint_as_float(raw[o][8 * c + 2 * k]) : 0.f,
                                                                bf16_hi(mw[k]) > 0.f ? __uint_as_float(raw[o][8 * c + 2 * k + 1]) : 0.f);
                        }
                    }
                    const int y = y0 + o;
                    if (!DGRAD && a.out_mode == 2) {
                        // TB feature matrix, channel-group-major feature order (conv_tc.cu): unit (c/8)*h*h + y*h + x
                        const long long hw = (long long)a.h_out * a.h_out;
                        const long long u0 = (long long)y * a.h_out + x;
                        const int fr = n < a.feat_half ? n : n - a.feat_half + a.feat_half_row;
#pragma unroll
                        for (int c = 0; c < 4; ++c)
                            *reinterpret_cast<uint4*>(a.out + ((((long long)(fr >> 7)) * a.feat_rpad + c * hw + u0) * DRQ_TB_ACT + (fr & 127)) * 8) =
                                make_uint4(packed[4 * c], packed[4 * c + 1], packed[4 * c + 2], packed[4 * c + 3]);
                    } else if (!DGRAD && a.out_mode == 1) {
                        uint4* dst = reinterpret_cast<uint4*>(a.out + (((long long)n * a.h_out + y) * a.h_out + x) * 32);
#pragma unroll
                        for (int c = 0; c < 4; ++c) dst[c] = make_uint4(packed[4 * c], packed[4 * c + 1], packed[4 * c + 2], packed[4 * c + 3]);
                    } else {
#pragma unroll
                        for (int c = 0; c < 4; ++c)
                            *reinterpret_cast<uint4*>(a.out + (c * a.cs_out + row0 + o * kPW) * 8) =
                                make_uint4(packed[4 * c], packed[4 * c + 1], packed[4 * c + 2], packed[4 * c + 3]);
                    }
                }
            }
            if (a.stamps && blockIdx.x == 0 && threadIdx.x == 2 * 32) {
                a.stamps[8] = st_tfull; a.stamps[9] = st_ld; a.stamps[10] = st_rest + (clock64() - e_prev); a.stamps[11] = clock64() - st_begin;
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem_base, kAcc * 128);
}

constexpr size_t kSmem = kWBytes + kStages * kStageBytes + 128 + (2 * kStages + 2 * kAcc) * 8 + 16 + 128;

long long* g_stamps = nullptr;

typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                             const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeFn encode_fn() { return reinterpret_cast<EncodeFn>(tensor_map_encoder()); }

}  // namespace c4

// Forward (dgrad = 0): in = the layer's input activation (valid h_out + 2), out per out_mode.  Data gradient (dgrad = 1):
// in = the gradient of the layer's output (valid h_layer_out, zero elsewhere), out = the gradient of its input (valid
// h_layer_out + 2), masked by the input activation.
int conv4x1_launch(bool dgrad, const __nv_bfloat16* in, long long cs_in, const __nv_bfloat16* w, const float* bias,
                   const __nv_bfloat16* mask, long long cs_mask, __nv_bfloat16* out, long long cs_out, int N, int h_layer_out,
                   int out_mode, long long feat_rpad, int feat_half, int feat_half_row, cudaStream_t stream) {
    using namespace c4;
    EncodeFn encode = encode_fn();
    if (!encode) {
        set_error("conv4x1: cuTensorMapEncodeTiled is not available");
        return DRQ_ERR_CUDA;
    }
    // the WB buffer as (164 x u32 = one image row of one channel block, row blocks, row planes, images, channel blocks)
    CUtensorMap map;
    const cuuint64_t gdim[5] = {(cuuint64_t)(kRowBytes / 4), (cuuint64_t)kRowBlocks, 4, (cuuint64_t)N, 4};
    const cuuint64_t gstr[4] = {(cuuint64_t)(4 * kRowBytes), (cuuint64_t)kRowBytes, (cuuint64_t)kPLB * 16, (cuuint64_t)cs_in * 16};
    const cuuint32_t box[5] = {(cuuint32_t)(kRowBytes / 4), (cuuint32_t)kBoxRows, 4, 1, 4};
    const cuuint32_t estr[5] = {1, 1, 1, 1, 1};
    const CUresult r = encode(&map, CU_TENSOR_MAP_DATA_TYPE_UINT32, 5, const_cast<__nv_bfloat16*>(in) + kGuard * 8, gdim, gstr, box, estr,
                              CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_error("conv4x1: cuTensorMapEncodeTiled failed (%d)", (int)r);
        return DRQ_ERR_CUDA;
    }
    Args a{};
    a.w = w; a.bias = bias; a.mask = mask; a.cs_mask = cs_mask; a.out = out; a.cs_out = cs_out;
    a.n_images = N;
    a.h_out = dgrad ? h_layer_out + 2 : h_layer_out;
    const int block_rows = (a.h_out + 3) / 4;
    a.tiles_per_image = (block_rows + kTileRows - 1) / kTileRows;
    a.total_tiles = N * a.tiles_per_image;
    a.m_tiles = (uint32_t)((1ull << 32) / (uint32_t)a.tiles_per_image) + 1u;
    a.out_mode = out_mode;
    a.feat_rpad = feat_rpad; a.feat_half = feat_half; a.feat_half_row = feat_half_row;
    a.stamps = g_stamps;
    if (a.h_out > kPW || (long long)a.total_tiles * a.tiles_per_image >= (1ll << 31)) {
        set_error("conv4x1: bad dims N=%d hout=%d", N, h_layer_out);
        return DRQ_ERR_INVALID;
    }
    const int grid = a.total_tiles < sm_budget() ? a.total_tiles : sm_budget();
    if (dgrad) {
        if (int rc = ensure_smem((const void*)conv4x1_tc_kernel<true>, kSmem, "conv4x1_dgrad")) return rc;
        conv4x1_tc_kernel<true><<<grid, kThreads, kSmem, stream>>>(map, a);
        return check_launch("conv4x1_tc_kernel<dgrad>");
    }
    if (int rc = ensure_smem((const void*)conv4x1_tc_kernel<false>, kSmem, "conv4x1_fwd")) return rc;
    conv4x1_tc_kernel<false><<<grid, kThreads, kSmem, stream>>>(map, a);
    return check_launch("conv4x1_tc_kernel<fwd>");
}

}  // namespace drq

extern "C" int drq_debug_conv4x1_stamps(int64_t* buf) { drq::c4::g_stamps = reinterpret_cast<long long*>(buf); return DRQ_OK; }

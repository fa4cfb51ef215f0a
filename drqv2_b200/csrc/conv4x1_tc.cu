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
// channel block).  A tile has three slots of 41 accumulator rows (123 live, 5 idle): three block rows of one image, or
// - where 10 block rows would leave a fourth tile one-third full (39 and 37 output rows) - the last block row of three
// images.  Its stage is six regions, one per window row wy, each [channel block][slot][41 px]; three 5-d tensor-map TMA
// boxes of two row planes (656 B x 3 row blocks or 3 images x 4 channel blocks x 2 planes) fill them: forward planes 0-3
// of the slots' row blocks and planes 0-1 of the next ones, data gradient (window two rows higher) planes 2-3 of the
// previous row blocks and planes 0-3 of the slots'.  Window element (wy, wx) of the 128 pixel columns is then region wy
// at offset wx: one K-major no-swizzle descriptor (K units = channel blocks one slab apart) plus an offset per UMMA, as
// in conv_tc.cu.  (A first version split 2x2 output blocks into four row/column parity planes with 16-byte cp.async
// copies: correct, and slower than conv_tc.cu - 2432 LSU requests per tile kept a loader warp issuing for 2500 cycles
// per 1800-cycle tile; git history, DESIGN.md §6.)  Row blocks outside the image and images past N are zero-filled by
// the TMA; the data gradient relies, like conv_tc.cu, on the gradient buffer being zero outside its valid region (its
// x - 2 of slot 0 reads columns 39-40 of the slab before, or the zeros in front of the stages).
//
// The weights arrive in the compact operand layout of pack_conv_w_elem ([tap*4 + k/8][n][k%8], 18 KB) and are reordered
// per CTA, while the first tiles load, into [wx][k/8][j][n][k%8] (18 KB): position j holds tap row dy = 2 - j (data
// gradient: dy = j).  Window row wy reaches the outputs oy0 .. oy0 + cnt - 1 through tap rows that are consecutive
// positions j = 2 - wy + oy, so the B operand of every window element (wy, wx) - N = 32 * cnt columns (oy, co) - is one
// K-major descriptor over the same 18 KB: start (wx * 12 + 2 - wy + oy0) * 32 units, K units 96 rows apart.
//
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
constexpr int kTileRows = 3;                  // slots of a tile: block rows of one image, or one block row of three images
constexpr int kTileCols = kTileRows * kPW;    // 123 live accumulator rows
constexpr int kSlab = kTileRows * kRowBytes;  // one (region, channel block): three slots, 1,968 B
constexpr int kRegion = 4 * kSlab;            // one window row wy: [channel block][slot][41 px]
constexpr int kBoxBytes = 2 * kRegion;        // one TMA box: two row planes
constexpr int kStageBytes = 6 * kRegion;      // 47,232
constexpr int kPad = 128;                     // zeros in front of stage 0: the data gradient's x - 2 of slot 0 reads them
constexpr int kStages = 3;
constexpr int kAcc = 4;                       // accumulator ring: 4 x 128 TMEM columns
constexpr int kWUnits = 3 * 4 * 3 * 32;       // 16-byte units of the reordered weights [wx][k/8][j][n]
constexpr int kWBytes = kWUnits * 16;
constexpr int kThreads = 10 * 32;
constexpr int kExpanders = kThreads - 32;     // everyone but the producer warp

struct Args {
    const __nv_bfloat16* w;                         // compact [36][32][8]
    const float* bias;                              // fwd
    const __nv_bfloat16* mask; long long cs_mask;   // dgrad: the layer's input activation (WB)
    __nv_bfloat16* out; long long cs_out;
    int n_images, tiles_per_image, total_tiles;     // tiles_per_image: per-image tiles, three block rows each
    int block_rows;
    int image_tiles;                                // N * tiles_per_image; the grouped tiles follow
    int pair_tiles;                                 // tiles of the images 0 .. (N & ~1) - 1
    int pair_rounds;                                // tile pairs every CTA takes before the single tiles of the tail
    int h_out;                                      // valid height = width of the output
    int out_mode;                                   // 0 WB, 1 compact NHWC, 2 TB features
    uint32_t m_pair;                                // floor(2^32 / (2 * tiles_per_image)) + 1
    long long feat_rpad; int feat_half, feat_half_row;
    long long* stamps;                              // drq_debug_conv4x1_stamps: per-role clock64 totals of block 0, or null
};

// Tile t < image_tiles is block rows i0 .. i0 + 2 of image n (slot s = block row i0 + s), numbered image-pair-major:
// t = 2 * (p * tiles_per_image + i0 / 3) + (n & 1) for n = 2p + (n & 1) < (N & ~1), then the tiles of an odd N's last
// image.  Tiles 2u and 2u + 1 (u < pair_tiles / 2) are the same block rows of two adjacent images.  A grouped tile
// t = image_tiles + g (only when block_rows % 3 == 1) is the last block row i0 = block_rows - 1 of images n = 3g .. 3g + 2
// (slot s = image n + s; images >= N are zero-filled by the TMA and not stored).
__device__ __forceinline__ bool tile_pos(const Args& a, int t, int& n, int& i0) {
    if (t < a.pair_tiles) {
        const int p = (int)__umulhi((uint32_t)t, a.m_pair);
        const int rem = t - p * 2 * a.tiles_per_image;
        i0 = (rem >> 1) * kTileRows;
        n = 2 * p + (rem & 1);
        return false;
    }
    if (t < a.image_tiles) {
        n = a.n_images - 1;
        i0 = (t - a.pair_tiles) * kTileRows;
        return false;
    }
    n = (t - a.image_tiles) * kTileRows;
    i0 = a.block_rows - 1;
    return true;
}

// The k-th tile of this CTA (>= total_tiles: done): pair_rounds pairs of consecutive tiles 2u, 2u + 1, u = blockIdx.x +
// j * gridDim.x, then one tile at a time over what is left - as many tiles per CTA as a plain round robin, and the TB
// epilogue sees both images of a pair in one CTA.
__device__ __forceinline__ int tile_at(const Args& a, int k) {
    const int q2 = 2 * a.pair_rounds;
    return k < q2 ? 2 * ((int)blockIdx.x + (k >> 1) * (int)gridDim.x) + (k & 1)
                  : q2 * (int)gridDim.x + (int)blockIdx.x + (k - q2) * (int)gridDim.x;
}

__device__ __forceinline__ void st_global_v8(void* p, const uint32_t* lo, const uint32_t* hi) {
    asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};"
                 ::"l"(p), "r"(lo[0]), "r"(lo[1]), "r"(lo[2]), "r"(lo[3]), "r"(hi[0]), "r"(hi[1]), "r"(hi[2]), "r"(hi[3]) : "memory");
}

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
// first 16-byte unit of the B operand of window element (wy, wx) in [wx][k/8][j][n][k%8]
__host__ __device__ constexpr int win_unit0(int wy, int wx) { return (wx * 12 + 2 - wy + win_oy0(wy)) * 32; }

template <bool DGRAD>
__device__ __forceinline__ void expand_weights(const __nv_bfloat16* __restrict__ w, uint8_t* w_s, int e) {
    const uint4* src = reinterpret_cast<const uint4*>(w);
    // unrolled: the units of a thread are independent address chains (a lone warp per scheduler runs a dependent chain
    // at ~5 cycles per instruction)
#pragma unroll
    for (int k = 0; k < kWUnits / kExpanders; ++k) {
        const int u = e + k * kExpanders;
        const int co = u & 31, r = u >> 5;                          // r = (wx * 4 + ku) * 3 + j
        const int wk = r / 3, j = r - wk * 3;
        const int wx = wk >> 2, ku = wk & 3;
        const int dy = DGRAD ? j : 2 - j;
        const int dx = DGRAD ? 2 - wx : wx;
        cp_async16(smem_u32(w_s) + u * 16, src + ((dy * 3 + dx) * 4 + ku) * 32 + co);
    }
    cp_async_commit();
    cp_async_wait_all();
}
static_assert(kWUnits % kExpanders == 0, "expansion loop has no tail");

template <bool DGRAD>
__global__ void __maxnreg__(128) conv4x1_tc_kernel(const __grid_constant__ CUtensorMap map_rows, const __grid_constant__ CUtensorMap map_imgs,
                                                   const Args a) {
    extern __shared__ __align__(128) uint8_t smem[];
    uint8_t* w_s = smem;
    uint8_t* a_s = smem + kWBytes + kPad;
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
        // ------------------------------------------------ TMA producer: three boxes of two row planes per tile, region
        // pair b = window rows 2b, 2b + 1.  Forward: planes 0-1 and 2-3 of the slots' row blocks, planes 0-1 of the next
        // row block; data gradient (the window starts two image rows higher): planes 2-3 of the previous row block, planes
        // 0-1 and 2-3 of the slots' row blocks.
        if (lane == 0) {
            int stage = 0; uint32_t phase = 0;
            long long st_empty = 0;
            const long long st_begin = clock64();
            for (int k = 0, t; (t = tile_at(a, k)) < a.total_tiles; ++k) {
                int n, i0;
                const bool grouped = tile_pos(a, t, n, i0);
                const long long c0 = clock64();
                mbar_wait(empty + stage, phase ^ 1);
                st_empty += clock64() - c0;
                mbar_arrive_expect_tx(full + stage, kStageBytes);
#pragma unroll
                for (int b = 0; b < 3; ++b) {
                    const int plane = DGRAD ? (b == 1 ? 0 : 2) : (b == 1 ? 2 : 0);
                    const int rb = i0 + (DGRAD ? (b == 0 ? -1 : 0) : (b == 2 ? 1 : 0));
                    const uint32_t dst = smem_u32(a_s + stage * kStageBytes + b * kBoxBytes);
                    if (grouped) tma_load_5d(dst, &map_imgs, 0, n, 0, plane, rb, full + stage);
                    else tma_load_5d(dst, &map_rows, 0, rb, 0, plane, n, full + stage);
                }
                if (++stage == kStages) { stage = 0; phase ^= 1; }
            }
            if (a.stamps && blockIdx.x == 0) { a.stamps[0] = st_empty; a.stamps[3] = clock64() - st_begin; }
        }
        __syncwarp();
    } else {
        // ------------------------------------------------ everyone else first expands the weights
        expand_weights<DGRAD>(a.w, w_s, warp == 0 ? lane : threadIdx.x - 32);
        if (threadIdx.x < kPad / 16) reinterpret_cast<uint4*>(a_s - kPad)[threadIdx.x] = make_uint4(0, 0, 0, 0);
        fence_proxy_async();
        asm volatile("bar.sync 1, %0;" ::"n"(kExpanders) : "memory");
        if (warp == 0) {
            // -------------------------------------------- UMMA issuer
            // A: K-major, 16-byte K units (channel blocks) one slab apart; B: K-major, K units 96 rows apart
            const uint64_t da0 = make_smem_desc(smem_u32(a_s), kSlab, 128);
            const uint64_t db = make_smem_desc(smem_u32(w_s), 96 * 16, 128);
            constexpr uint32_t idesc32 = make_idesc_bf16(128, 32, false, false);
            constexpr uint32_t idesc64 = make_idesc_bf16(128, 64, false, false);
            constexpr uint32_t idesc96 = make_idesc_bf16(128, 96, false, false);
            int stage = 0; uint32_t phase = 0; int acc = 0; uint32_t acc_phase = 0;
            long long st_tempty = 0, st_full = 0, st_mma = 0;
            const long long st_begin = clock64();
            for (int k = 0; tile_at(a, k) < a.total_tiles; ++k) {
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
                        // region wy holds window row wy of every slot: forward image row 4i+wy, columns x..x+2; data
                        // gradient: gradient row 4i-2+wy, columns x-2..x
                        const int cnt = win_cnt(wy);
                        const uint32_t idesc = cnt == 1 ? idesc32 : cnt == 2 ? idesc64 : idesc96;
#pragma unroll
                        for (int wx = 0; wx < 3; ++wx)
#pragma unroll
                            for (int h = 0; h < 2; ++h)
                                umma_bf16(d_tmem + 32 * win_oy0(wy),
                                          da + (uint64_t)(int64_t)(wy * (kRegion >> 4) + wx - (DGRAD ? 2 : 0) + h * 2 * (kSlab >> 4)),
                                          db + (uint64_t)(win_unit0(wy, wx) + h * 2 * 96), idesc, (o < 2 && wx == 0 && h == 0) ? 0u : 1u);
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
            long long st_tfull = 0, st_ld = 0, st_rest = 0;
            const long long st_begin = clock64();
            long long e_prev = st_begin;
            // data gradient: the ReLU mask (the layer's input activation at the output pixels) of tile t is fetched one tile
            // ahead - issued after the previous tile's accumulator has been read, consumed after this tile's
            uint4 mk[DGRAD ? 2 : 1][4], mk_next[DGRAD ? 2 : 1][4];
            auto load_mask = [&](int t, uint4 (&m4)[DGRAD ? 2 : 1][4]) {
                if (t >= a.total_tiles) return;
                int n, i0;
                const bool grouped = tile_pos(a, t, n, i0);
                if (grouped) n += r; else i0 += r;
                const int y0 = 4 * i0 + 2 * half;
                const long long row0 = (long long)n * kPLB + kGuard + y0 * kPW + x;
                const bool colok = live && x < a.h_out && n < a.n_images;
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    m4[0][c] = (colok && y0 < a.h_out) ? __ldg(reinterpret_cast<const uint4*>(a.mask + (c * a.cs_mask + row0) * 8)) : make_uint4(0, 0, 0, 0);
                    m4[DGRAD ? 1 : 0][c] = (colok && y0 + 1 < a.h_out) ? __ldg(reinterpret_cast<const uint4*>(a.mask + (c * a.cs_mask + row0 + kPW) * 8))
                                                                       : make_uint4(0, 0, 0, 0);
                }
            };
            // the bias is read from shared memory (broadcast) here: 32 registers held across the loop make it spill
            auto pack_fwd = [&](const uint32_t (&raw)[32], uint32_t (&packed)[16]) {
#pragma unroll
                for (int k = 0; k < 8; ++k) {
                    const float4 b = reinterpret_cast<const float4*>(bias_s)[k];
                    packed[2 * k] = pack_bf16x2(fmaxf(__uint_as_float(raw[4 * k]) + b.x, 0.f), fmaxf(__uint_as_float(raw[4 * k + 1]) + b.y, 0.f));
                    packed[2 * k + 1] = pack_bf16x2(fmaxf(__uint_as_float(raw[4 * k + 2]) + b.z, 0.f), fmaxf(__uint_as_float(raw[4 * k + 3]) + b.w, 0.f));
                }
            };
            // TB feature matrix, channel-group-major feature order (conv_tc.cu): 16-byte unit (c/8)*h*h + y*h + x of row fr
            const long long hw = (long long)a.h_out * a.h_out;
            auto tb_row = [&](int n) { return n < a.feat_half ? n : n - a.feat_half + a.feat_half_row; };
            auto tb_unit = [&](int fr, int c, long long u) { return a.out + ((((long long)(fr >> 7)) * a.feat_rpad + c * hw + u) * DRQ_TB_ACT + (fr & 127)) * 8; };
            const uint32_t tq = tmem_base + ((uint32_t)(q * 32) << 16) + half * 64;
            if (DGRAD) load_mask(tile_at(a, 0), mk_next);
            for (int k = 0, t; (t = tile_at(a, k)) < a.total_tiles; ++k) {
                int n, i0;
                const bool grouped = tile_pos(a, t, n, i0);
                // TB features: tiles t, t + 1 of a pair round are the same pixels of images n, n + 1.  Where their feature
                // rows are an aligned pair of adjacent 16-byte units, one 32-byte store (a whole sector) writes both: lanes,
                // consecutive x, are 2 KB apart, so a 16-byte store is half a sector.  Otherwise the two go one at a time.
                const bool two = !DGRAD && a.out_mode == 2 && !(k & 1) && k < 2 * a.pair_rounds && t < a.pair_tiles &&
                                 tb_row(n + 1) == tb_row(n) + 1 && !(tb_row(n) & 1);
                // this thread's slot r: image n + r of a grouped tile, block row i0 + r of a per-image one
                if (grouped) n += r; else i0 += r;
                const int y0 = 4 * i0 + 2 * half;
                const long long row0 = (long long)n * kPLB + kGuard + y0 * kPW + x;
                // data gradient: every column of a valid row is written (zeros beyond the valid width: the next layer's
                // windows read them); forward: valid pixels only
                const bool okp = live && n < a.n_images && (DGRAD || x < a.h_out);
                const bool ok0 = okp && y0 < a.h_out;
                const bool ok1 = okp && y0 + 1 < a.h_out;
                if (DGRAD) {
#pragma unroll
                    for (int c = 0; c < 4; ++c) { mk[0][c] = mk_next[0][c]; mk[DGRAD ? 1 : 0][c] = mk_next[DGRAD ? 1 : 0][c]; }
                }
                const int acc1 = two ? (acc + 1) % kAcc : acc;
                const long long e0 = clock64();
                mbar_wait(tfull + acc, acc_phase);
                if (two) mbar_wait(tfull + acc1, acc1 == 0 ? acc_phase ^ 1 : acc_phase);
                const long long e1 = clock64();
                st_rest += e0 - e_prev; st_tfull += e1 - e0;
                tc_fence_after();
                // one tile: raw = output rows 2*half, 2*half + 1 in one pass; a pair: raw = one output row of both images per pass
#pragma unroll 1
                for (int pass = 0; pass < (two ? 2 : 1); ++pass) {
                    uint32_t raw[2][32];
                    tmem_ld_32x32_raw(tq + acc * 128 + (two ? 32 * pass : 0), raw[0]);
                    tmem_ld_32x32_raw(tq + acc1 * 128 + (two ? 32 * pass : 32), raw[1]);
                    tmem_wait_ld();
                    if (pass == (two ? 1 : 0)) {
                        tc_fence_before();
                        __syncwarp();
                        if (lane == 0) {
                            mbar_arrive(tempty + acc);
                            if (two) mbar_arrive(tempty + acc1);
                        }
                        for (int i = 0; i < (two ? 2 : 1); ++i)
                            if (++acc == kAcc) { acc = 0; acc_phase ^= 1; }
                        e_prev = clock64();
                        st_ld += e_prev - e1;
                        if (DGRAD) load_mask(tile_at(a, k + 1), mk_next);
                    }
                    if (two) {
                        if (!(pass ? ok1 : ok0)) continue;
                        const long long u = (long long)(y0 + pass) * a.h_out + x;
                        const int fa = tb_row(n);
#pragma unroll
                        for (int c = 0; c < 4; ++c) {
                            uint32_t pa[4], pb[4];
#pragma unroll
                            for (int j = 0; j < 4; ++j) {
                                const float2 b = reinterpret_cast<const float2*>(bias_s)[4 * c + j];
                                pa[j] = pack_bf16x2(fmaxf(__uint_as_float(raw[0][8 * c + 2 * j]) + b.x, 0.f), fmaxf(__uint_as_float(raw[0][8 * c + 2 * j + 1]) + b.y, 0.f));
                                pb[j] = pack_bf16x2(fmaxf(__uint_as_float(raw[1][8 * c + 2 * j]) + b.x, 0.f), fmaxf(__uint_as_float(raw[1][8 * c + 2 * j + 1]) + b.y, 0.f));
                            }
                            st_global_v8(tb_unit(fa, c, u), pa, pb);
                        }
                        continue;
                    }
#pragma unroll
                    for (int o = 0; o < 2; ++o) {
                        if (!(o ? ok1 : ok0)) continue;
                        uint32_t packed[16];
                        if (!DGRAD) {
                            pack_fwd(raw[o], packed);
                        } else {
#pragma unroll
                            for (int c = 0; c < 4; ++c) {
                                const uint32_t mw[4] = {mk[DGRAD ? o : 0][c].x, mk[DGRAD ? o : 0][c].y, mk[DGRAD ? o : 0][c].z, mk[DGRAD ? o : 0][c].w};
#pragma unroll
                                for (int j = 0; j < 4; ++j)
                                    packed[4 * c + j] = pack_bf16x2(bf16_lo(mw[j]) > 0.f ? __uint_as_float(raw[o][8 * c + 2 * j]) : 0.f,
                                                                    bf16_hi(mw[j]) > 0.f ? __uint_as_float(raw[o][8 * c + 2 * j + 1]) : 0.f);
                            }
                        }
                        const int y = y0 + o;
                        if (!DGRAD && a.out_mode == 2) {
                            // a tile without a partner image in this CTA (the tail past the pair rounds, an odd N's last image)
                            const long long u = (long long)y * a.h_out + x;
#pragma unroll
                            for (int c = 0; c < 4; ++c)
                                *reinterpret_cast<uint4*>(tb_unit(tb_row(n), c, u)) = make_uint4(packed[4 * c], packed[4 * c + 1], packed[4 * c + 2], packed[4 * c + 3]);
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
                if (two) ++k;
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

constexpr size_t kSmem = kWBytes + kPad + kStages * kStageBytes + 128 + (2 * kStages + 2 * kAcc) * 8 + 16 + 128;

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
    // the WB buffer as 164 x u32 = one image row of one channel block, then row blocks / images, channel blocks, row planes,
    // images / row blocks: a box of two row planes lands [plane][channel block][slot][656 B], three row blocks of one image
    // (map_rows) or one row block of three images (map_imgs) as the slots
    // Row blocks: those holding the valid input rows, so that the rest reads as zeros.  Image rows 41..43 would be the next
    // image's guard and first pixels, and the data gradient's x - 2 of slot 0 reads columns 39-40 of whatever row block
    // precedes it in shared memory.
    CUtensorMap maps[2];
    const cuuint64_t row_blocks = (cuuint64_t)(((dgrad ? h_layer_out : h_layer_out + 2) + 3) / 4);
    const cuuint64_t s_img = (cuuint64_t)kPLB * 16, s_rb = 4 * kRowBytes;
    const cuuint64_t gdim[2][5] = {{(cuuint64_t)(kRowBytes / 4), row_blocks, 4, 4, (cuuint64_t)N},
                                   {(cuuint64_t)(kRowBytes / 4), (cuuint64_t)N, 4, 4, row_blocks}};
    const cuuint64_t gstr[2][4] = {{s_rb, (cuuint64_t)cs_in * 16, (cuuint64_t)kRowBytes, s_img},
                                   {s_img, (cuuint64_t)cs_in * 16, (cuuint64_t)kRowBytes, s_rb}};
    const cuuint32_t box[5] = {(cuuint32_t)(kRowBytes / 4), (cuuint32_t)kTileRows, 4, 2, 1};
    const cuuint32_t estr[5] = {1, 1, 1, 1, 1};
    static_assert(kBoxBytes == kRowBytes * kTileRows * 4 * 2, "a box fills two regions");
    for (int i = 0; i < 2; ++i) {
        const CUresult r = encode(&maps[i], CU_TENSOR_MAP_DATA_TYPE_UINT32, 5, const_cast<__nv_bfloat16*>(in) + kGuard * 8, gdim[i], gstr[i], box,
                                  estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) {
            set_error("conv4x1: cuTensorMapEncodeTiled failed (%d)", (int)r);
            return DRQ_ERR_CUDA;
        }
    }
    Args a{};
    a.w = w; a.bias = bias; a.mask = mask; a.cs_mask = cs_mask; a.out = out; a.cs_out = cs_out;
    a.n_images = N;
    a.h_out = dgrad ? h_layer_out + 2 : h_layer_out;
    a.block_rows = (a.h_out + 3) / 4;
    // a last block row that would be a tile of its own shares one with those of the next two images: 39 and 37 output
    // rows = 10 block rows = 3 tiles per image + one per three images instead of 4 per image
    const bool grouped = a.block_rows % kTileRows == 1;
    a.tiles_per_image = grouped ? a.block_rows / kTileRows : (a.block_rows + kTileRows - 1) / kTileRows;
    a.image_tiles = N * a.tiles_per_image;
    a.total_tiles = a.image_tiles + (grouped ? (N + kTileRows - 1) / kTileRows : 0);
    a.pair_tiles = (N & ~1) * a.tiles_per_image;
    a.m_pair = a.tiles_per_image ? (uint32_t)((1ull << 32) / (uint32_t)(2 * a.tiles_per_image)) + 1u : 0u;
    a.out_mode = out_mode;
    a.feat_rpad = feat_rpad; a.feat_half = feat_half; a.feat_half_row = feat_half_row;
    a.stamps = g_stamps;
    if (a.h_out > kPW || (long long)a.total_tiles * 2 * (a.tiles_per_image + 1) >= (1ll << 31)) {
        set_error("conv4x1: bad dims N=%d hout=%d", N, h_layer_out);
        return DRQ_ERR_INVALID;
    }
    const int grid = a.total_tiles < sm_budget() ? a.total_tiles : sm_budget();
    a.pair_rounds = a.total_tiles / (2 * grid);
    if (dgrad) {
        if (int rc = ensure_smem((const void*)conv4x1_tc_kernel<true>, kSmem, "conv4x1_dgrad")) return rc;
        conv4x1_tc_kernel<true><<<grid, kThreads, kSmem, stream>>>(maps[0], maps[1], a);
        return check_launch("conv4x1_tc_kernel<dgrad>");
    }
    if (int rc = ensure_smem((const void*)conv4x1_tc_kernel<false>, kSmem, "conv4x1_fwd")) return rc;
    conv4x1_tc_kernel<false><<<grid, kThreads, kSmem, stream>>>(maps[0], maps[1], a);
    return check_launch("conv4x1_tc_kernel<fwd>");
}

}  // namespace drq

extern "C" int drq_debug_conv4x1_stamps(int64_t* buf) { drq::c4::g_stamps = reinterpret_cast<long long*>(buf); return DRQ_OK; }

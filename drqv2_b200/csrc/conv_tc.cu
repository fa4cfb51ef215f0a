// bf16 tensor-core encoder kernels (tcgen05 + TMEM + bulk-async loads), sm_100a only.
// Reference ops: the 3x3 stride-1 convolutions of Encoder (drqv2.py:56-59) forward, and
// their data gradients.
//
// Layout "WB" (wide, blocked, bf16): [4 channel-blocks][N images * kPLB pixel rows + slack][8 ch].
// Image n's wide position p (row stride 41, see encoder_f32.cu) is pixel row n*kPLB + kGuard + p;
// the kGuard leading rows of every image stay zero in gradient buffers so that dgrad's
// negative tap offsets read zeros.  One pixel row of one block is 16 bytes = one K unit of a
// K-major (no-swizzle) UMMA operand, so a [128 + 84]-row window staged once in shared memory
// serves all nine taps: tap (ky,kx) is the same descriptor advanced by (ky*41+kx)*16 bytes.
//
//   out[p][:] = sum_tap  A_tap[128 x 32] * W_tap[32 x 32]      (18 UMMAs of M128 N32 K16 per tile)
//
// Warp roles (192 threads): warp 0 = bulk-copy producer, warp 1 = UMMA issuer, warps 2..5 =
// epilogue (TMEM -> registers -> bias/ReLU or ReLU-mask -> bf16 -> coalesced 16-byte stores).
#include "pack.cuh"
#include "wgrad_reduce.cuh"

namespace drq {

DRQ_TRAP_NOTE_HOOK(trap_note_conv)

constexpr int kPLB = DRQ_PLB;        // pixel rows per image in WB buffers
constexpr int kGuard = DRQ_GUARD;    // zero rows in front of every image
constexpr int kSlack = DRQ_WB_SLACK; // rows after the last image of each block
constexpr int kTM = 128;             // output positions per tile
constexpr int kHaloTC = 2 * kPW + 2; // 84
constexpr int kWinRows = kTM + kHaloTC;      // 212 rows loaded per block
constexpr int kStageRows = 216;              // smem rows per block (8-row aligned)
constexpr int kStageBytes = 4 * kStageRows * 16;
constexpr int kStagesTC = 4;
constexpr int kAccStages = 4;
constexpr int kWBytes = 36 * 32 * 16;        // 9 taps x 4 K units x 32 n x 16 B
constexpr int kThreadsTC = 192;

using namespace tc;

struct ConvTcArgs {
    const __nv_bfloat16* in; long long cs_in;       // chunk stride in pixel rows
    const __nv_bfloat16* w;                         // packed [36][32][8]
    const float* bias;                              // fwd
    const __nv_bfloat16* mask; long long cs_mask;   // dgrad: input activation (WB)
    __nv_bfloat16* out; long long cs_out;
    int n_images, ntiles, n_pos, w_valid, nhwc_out;   // nhwc_out: 0 WB, 1 compact NHWC, 2 TB features (feat_rpad = units per row)
    long long* stamps;        // debug: per-role wait / work cycle totals of block 0, or null
    long long feat_rpad; int feat_half, feat_half_row;   // TB features: image n >= feat_half lands at row n - feat_half + feat_half_row
};

static long long* g_conv_stamps = nullptr;

// conv4x1_tc.cu: four output pixels (a column) per accumulator row.  0 = off, 1 = for launches that fill the machine,
// 2 = always (tests), 3 (default) = as 1 for the forward only, 4 = as 1 for the data gradient only.  Measured on the
// B = 256 update (gpurun_out/ab_conv4x1_*): alone the new kernels are faster (graph nodes, warm: forward 27.6 vs 28.9 us,
// data gradient 16.7 vs 20.1 us; one-stream update 1719 vs 1672 updates/s), but in the three-stream schedule the data
// gradient runs on the encoder stream beside the critic's optimiser step and the actor pass, and its one 200 KB /
// 54 K-register CTA per SM leaves no room for their blocks (the old kernel's two 74 KB CTAs do): 1798 updates/s with it,
// 1858 without, 1868 with the forward alone.
int conv4x1_launch(bool dgrad, const __nv_bfloat16* in, long long cs_in, const __nv_bfloat16* w, const float* bias,
                   const __nv_bfloat16* mask, long long cs_mask, __nv_bfloat16* out, long long cs_out, int N, int h_layer_out,
                   int out_mode, long long feat_rpad, int feat_half, int feat_half_row, cudaStream_t stream);
static int g_conv4x1 = 3;
constexpr int kConv4x1MinImages = 48;      // ~148 tiles: below that the one-pixel-per-row kernel's 18 KB set-up wins
static bool use_conv4x1(int N, bool dgrad) {
    if (g_conv4x1 == 3 && dgrad) return false;      // 3 / 4: forward only / data gradient only (A/B measurements)
    if (g_conv4x1 == 4 && !dgrad) return false;
    return g_conv4x1 == 2 || (g_conv4x1 >= 1 && N >= kConv4x1MinImages);
}
#ifdef DRQ_STAMPS
#define CV_T() (a.stamps ? clock64() : 0ll)
#define CV_STAMPS(x) x
#else
#define CV_T() 0ll
#define CV_STAMPS(x)
#endif

template <bool DGRAD>
__global__ void __launch_bounds__(kThreadsTC, 2) conv3x3_tc_kernel(ConvTcArgs a) {
    extern __shared__ __align__(128) uint8_t smem[];
    uint8_t* w_s = smem;
    uint8_t* a_s = smem + kWBytes;
    uint64_t* bars = reinterpret_cast<uint64_t*>(a_s + kStagesTC * kStageBytes);
    uint64_t* full = bars;
    uint64_t* empty = bars + kStagesTC;
    uint64_t* tfull = bars + 2 * kStagesTC;
    uint64_t* tempty = bars + 2 * kStagesTC + kAccStages;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * kStagesTC + 2 * kAccStages);
    float* bias_s = reinterpret_cast<float*>(tmem_slot + 4);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int total_tiles = a.n_images * a.ntiles;
    if (threadIdx.x == 0) {
        for (int i = 0; i < kStagesTC; ++i) { mbar_init(full + i, 1); mbar_init(empty + i, 1); }
        for (int i = 0; i < kAccStages; ++i) { mbar_init(tfull + i, 1); mbar_init(tempty + i, 4); }
        fence_barrier_init();
    }
    if (warp == 1) {
        tmem_alloc(tmem_slot, kAccStages * 32);
        tmem_relinquish();
    }
    if (!DGRAD && threadIdx.x < 32) bias_s[threadIdx.x] = a.bias[threadIdx.x];

    // packed weights -> smem (same byte layout)
    {
        const uint4* src = reinterpret_cast<const uint4*>(a.w);
        uint4* dst = reinterpret_cast<uint4*>(w_s);
        for (int i = threadIdx.x; i < kWBytes / 16; i += kThreadsTC) dst[i] = __ldg(src + i);
    }
    fence_proxy_async();      // generic-proxy smem writes (weights) -> visible to the async proxy (UMMA)
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ------------------------------------------------ producer: lanes 0..3 issue one channel block each
        {
            int stage = 0; uint32_t phase = 0;
            long long w_empty = 0;
            const long long t_begin = CV_T();
            for (int t = blockIdx.x; t < total_tiles; t += gridDim.x) {
                const int n = t / a.ntiles, p0 = (t - n * a.ntiles) * kTM;
                const long long c0 = CV_T();
                mbar_wait(empty + stage, phase ^ 1);
                w_empty += CV_T() - c0;
                if (lane == 0) mbar_arrive_expect_tx(full + stage, 4 * kWinRows * 16);
                __syncwarp();
                const long long row0 = (long long)n * kPLB + kGuard + p0 - (DGRAD ? kHaloTC : 0);
                uint8_t* dst = a_s + stage * kStageBytes;
                if (lane < 4)
                    bulk_g2s(dst + lane * kStageRows * 16, a.in + (lane * a.cs_in + row0) * 8, kWinRows * 16, full + stage);
                if (++stage == kStagesTC) { stage = 0; phase ^= 1; }
            }
            CV_STAMPS(if (a.stamps && blockIdx.x == 0 && lane == 0) { a.stamps[0] = w_empty; a.stamps[1] = CV_T() - t_begin; })
        }
    } else if (warp == 1) {
        // ------------------------------------------------ UMMA issuer.  One thread issues 18 UMMAs per tile; the
        // descriptors are a per-stage base plus compile-time (address >> 4) offsets so that the issue
        // loop is two adds and the instruction per UMMA (a dependent ALU op costs the lone thread ~4
        // cycles; the M128 N32 K16 UMMA itself retires every ~45 cycles, tools/ub/ub_mma.cu).
        constexpr uint32_t idesc = make_idesc_bf16(128, 32, false, false);
        int stage = 0; uint32_t phase = 0; int acc = 0; uint32_t acc_phase = 0;
        const uint64_t da0 = make_smem_desc(smem_u32(a_s), kStageRows * 16, 128);
        const uint64_t db0 = make_smem_desc(smem_u32(w_s), 512, 128);
        long long w_tempty = 0, w_full = 0;
        const long long t_begin = CV_T();
        for (int t = blockIdx.x; t < total_tiles; t += gridDim.x) {
            const long long c0 = CV_T();
            mbar_wait(tempty + acc, acc_phase ^ 1);
            const long long c1 = CV_T();
            mbar_wait(full + stage, phase);
            const long long c2 = CV_T();
            w_tempty += c1 - c0; w_full += c2 - c1;
            tc_fence_after();
            if (elect_one()) {
                const uint64_t da = da0 + (uint64_t)(stage * (kStageBytes >> 4));
                const uint32_t d_tmem = tmem_base + acc * 32;
#pragma unroll
                for (int tap = 0; tap < 9; ++tap) {
                    const int off = (tap / 3) * kPW + (tap % 3);
                    const int o = DGRAD ? kHaloTC - off : off;
#pragma unroll
                    for (int h = 0; h < 2; ++h)
                        umma_bf16(d_tmem, da + (uint64_t)(o + h * 2 * kStageRows), db0 + (uint64_t)((tap * 4 + h * 2) * 32), idesc,
                                  (tap | h) ? 1u : 0u);
                }
                umma_commit(empty + stage);    // smem stage reusable once these UMMAs retire
                umma_commit(tfull + acc);      // accumulator ready for the epilogue
            }
            __syncwarp();
            if (++stage == kStagesTC) { stage = 0; phase ^= 1; }
            if (++acc == kAccStages) { acc = 0; acc_phase ^= 1; }
        }
        // drain the last stages' `empty` arrivals (asynchronous, waited for by nobody else) before the CTA may exit
        {
            const int used = blockIdx.x < (unsigned)total_tiles ? (total_tiles - 1 - (int)blockIdx.x) / (int)gridDim.x + 1 : 0;
            for (int j = 0; j < kStagesTC && j < used; ++j) {
                int s2 = stage - 1 - j; uint32_t ph = phase;
                if (s2 < 0) { s2 += kStagesTC; ph ^= 1; }
                mbar_wait(empty + s2, ph);
            }
        }
        CV_STAMPS(if (a.stamps && blockIdx.x == 0 && lane == 0) { a.stamps[2] = w_tempty; a.stamps[3] = w_full; a.stamps[4] = CV_T() - t_begin; })
    } else {
        // ------------------------------------------------ epilogue (warps 2..5 -> TMEM lane quarters 2,3,0,1)
        const int q = warp & 3;
        int acc = 0; uint32_t acc_phase = 0;
        uint4 mk[4], mk_next[4];
        auto load_mask = [&](int t, uint4 (&m4)[4]) {     // ReLU mask (the layer's input activation) of tile t
            const int n = t / a.ntiles, p = (t - n * a.ntiles) * kTM + q * 32 + lane;
            if (t < total_tiles && p < a.n_pos) {
                const long long row = (long long)n * kPLB + kGuard + p;
#pragma unroll
                for (int c = 0; c < 4; ++c) m4[c] = __ldg(reinterpret_cast<const uint4*>(a.mask + (c * a.cs_mask + row) * 8));
            }
        };
        if (DGRAD) load_mask(blockIdx.x, mk_next);
        // the bias in registers: read per tile from shared memory it was 80 % of the kernel's shared-memory wavefronts
        // (ncu r2: 2.0 M bank-conflict wavefronts of 2.5 M, against 63 k in the data-gradient variant)
        float bias_r[DGRAD ? 1 : 32];
        if (!DGRAD) {
#pragma unroll
            for (int i = 0; i < 32; ++i) bias_r[i] = bias_s[i];
        }
        for (int t = blockIdx.x; t < total_tiles; t += gridDim.x) {
            const int n = t / a.ntiles, p0 = (t - n * a.ntiles) * kTM;
            const int p = p0 + q * 32 + lane;
            const long long row = (long long)n * kPLB + kGuard + p;
            if (DGRAD) {        // this tile's mask was fetched one tile ago; start the next tile's loads now
#pragma unroll
                for (int c = 0; c < 4; ++c) mk[c] = mk_next[c];
                load_mask(t + gridDim.x, mk_next);
            }
            const long long e0 = CV_T();
            mbar_wait(tfull + acc, acc_phase);
            CV_STAMPS(if (a.stamps && blockIdx.x == 0 && threadIdx.x == 64) a.stamps[5] += CV_T() - e0;)
            tc_fence_after();
            float v[32];
            tmem_ld_32x32(tmem_base + ((uint32_t)(q * 32) << 16) + acc * 32, v);
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(tempty + acc);
            if (++acc == kAccStages) { acc = 0; acc_phase ^= 1; }

            if (p >= a.n_pos) continue;
            const int y = p / kPW, x = p - y * kPW;
            uint32_t packed[16];
            if (!DGRAD) {
#pragma unroll
                for (int i = 0; i < 16; ++i) {
                    const float lo = fmaxf(v[2 * i] + bias_r[DGRAD ? 0 : 2 * i], 0.f);
                    const float hi = fmaxf(v[2 * i + 1] + bias_r[DGRAD ? 0 : 2 * i + 1], 0.f);
                    packed[i] = pack_bf16x2(lo, hi);
                }
                if (a.nhwc_out == 2) {
                    // TB feature matrix, channel-group-major feature order: unit (c/8)*w*w + y*w + x, row = image
                    // (128-row blocks of feat_rpad units)
                    if (x < a.w_valid) {
                        const long long hw = (long long)a.w_valid * a.w_valid;
                        const long long u0 = (long long)y * a.w_valid + x;
                        const int fr = n < a.feat_half ? n : n - a.feat_half + a.feat_half_row;
#pragma unroll
                        for (int c = 0; c < 4; ++c)
                            *reinterpret_cast<uint4*>(a.out + ((((long long)(fr >> 7)) * a.feat_rpad + c * hw + u0) * DRQ_TB_ACT + (fr & 127)) * 8) =
                                make_uint4(packed[4 * c], packed[4 * c + 1], packed[4 * c + 2], packed[4 * c + 3]);
                    }
                    continue;
                }
                if (a.nhwc_out) {
                    if (x < a.w_valid) {
                        uint4* dst = reinterpret_cast<uint4*>(a.out + (((long long)n * a.w_valid + y) * a.w_valid + x) * 32);
#pragma unroll
                        for (int c = 0; c < 4; ++c)
                            dst[c] = make_uint4(packed[4 * c], packed[4 * c + 1], packed[4 * c + 2], packed[4 * c + 3]);
                    }
                    continue;
                }
            } else {
                const bool col_ok = x < a.w_valid;
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    const uint32_t mw[4] = {mk[c].x, mk[c].y, mk[c].z, mk[c].w};
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const float lo = (col_ok && bf16_lo(mw[j]) > 0.f) ? v[8 * c + 2 * j] : 0.f;
                        const float hi = (col_ok && bf16_hi(mw[j]) > 0.f) ? v[8 * c + 2 * j + 1] : 0.f;
                        packed[4 * c + j] = pack_bf16x2(lo, hi);
                    }
                }
            }
#pragma unroll
            for (int c = 0; c < 4; ++c)
                *reinterpret_cast<uint4*>(a.out + (c * a.cs_out + row) * 8) =
                    make_uint4(packed[4 * c], packed[4 * c + 1], packed[4 * c + 2], packed[4 * c + 3]);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem_base, kAccStages * 32);
}

__global__ void pack_conv_w_kernel(const float* __restrict__ w, __nv_bfloat16* __restrict__ w_fwd,
                                   __nv_bfloat16* __restrict__ w_dgrad) {
    pack_conv_w_elem(w, w_fwd, w_dgrad, blockIdx.x * blockDim.x + threadIdx.x);
}


// ---------------------------------------------------------------- conv 32->32 weight gradient
// dW[tap][ci][co] = sum_{n,p} in[n][p + off(tap)][ci] * d[n][p][co]: GEMMs with K = positions whose operands
// are read straight from WB-layout windows as MN-major UMMA operands (8 channels = one 16-byte unit,
// consecutive positions 16 bytes apart = consecutive K).
// A UMMA of this shape is bound by the shared-memory bytes of its operands ((A + B) / 128 B per cycle,
// tools/ub/ub_mma.cu), so the three horizontal taps share one instruction: the input window is staged three
// times, shifted by 0 / 1 / 2 positions, as 12 consecutive MN units, a 13th unit holds bf16 ones (its rows
// give the bias gradient) and one M = 128 UMMA per vertical tap and K step multiplies all of them by the
// gradient tile: 3 UMMAs of 5 KB per K step instead of 10 of 3 KB.  Units 13..15 read whatever follows
// in shared memory; their accumulator rows are ignored.  Every CTA keeps its 3 accumulators (96 TMEM columns)
// across all of its tiles and writes one fp32 partial at the end; partials are reduced in fixed order.
constexpr int kWgStages = 3;
constexpr int kWgDRows = kTM;                              // d tile rows per block
constexpr int kWgPlane = kStageRows * 16;                  // one MN unit: 216 positions x 8 channels
constexpr int kWgABytes = 13 * kWgPlane;                   // 3 shifted windows x 4 channel blocks + ones
constexpr int kWgStageBytes = kWgABytes + 4 * kWgDRows * 16;
constexpr int kWgAcc = 10;
constexpr int kWgPartial = kWgAcc * 32 * 32;
static_assert(kWgPartial == kWgPartialFloats, "wgrad_reduce.cuh");               // floats per CTA: [9 taps + bias][ci][co]

struct WgradTcArgs {
    const __nv_bfloat16* in; long long cs_in;
    const __nv_bfloat16* d; long long cs_d;
    float* partial;
    int n_images, ntiles;
};

__global__ void __launch_bounds__(kThreadsTC, 1) conv3x3_wgrad_tc_kernel(WgradTcArgs a) {
    extern __shared__ __align__(128) uint8_t smem[];
    uint8_t* st_s = smem;
    uint64_t* bars = reinterpret_cast<uint64_t*>(st_s + kWgStages * kWgStageBytes + 3 * kWgPlane);
    uint64_t* full = bars;
    uint64_t* empty = bars + kWgStages;
    uint64_t* done = bars + 2 * kWgStages;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * kWgStages + 1);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int total_tiles = a.n_images * a.ntiles;
    const int cta = blockIdx.x, ncta = gridDim.x;
    for (int i = threadIdx.x; i < kWgStages * (kWgPlane / 4); i += kThreadsTC) {
        const int st = i / (kWgPlane / 4), w = i - st * (kWgPlane / 4);
        reinterpret_cast<uint32_t*>(st_s + st * kWgStageBytes + 12 * kWgPlane)[w] = 0x3F803F80u;    // bf16 1.0 x2
    }
    if (threadIdx.x == 0) {
        for (int i = 0; i < kWgStages; ++i) { mbar_init(full + i, 1); mbar_init(empty + i, 1); }
        mbar_init(done, 1);
        fence_barrier_init();
    }
    if (warp == 1) {
        tmem_alloc(tmem_slot, 128);
        tmem_relinquish();
    }
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // lanes 0..11: input window, shift lane / 4, channel block lane % 4; lanes 12..15: gradient tile channel blocks
        int stage = 0; uint32_t phase = 0;
        for (int t = cta; t < total_tiles; t += ncta) {
            const int n = t / a.ntiles, p0 = (t - n * a.ntiles) * kTM;
            mbar_wait(empty + stage, phase ^ 1);
            if (lane == 0) mbar_arrive_expect_tx(full + stage, (12 * kWinRows + 4 * kWgDRows) * 16);
            __syncwarp();
            const long long row0 = (long long)n * kPLB + kGuard + p0;
            uint8_t* dst = st_s + stage * kWgStageBytes;
            if (lane < 12)
                bulk_g2s(dst + lane * kWgPlane, a.in + ((lane & 3) * a.cs_in + row0 + (lane >> 2)) * 8, kWinRows * 16, full + stage);
            else if (lane < 16)
                bulk_g2s(dst + kWgABytes + (lane - 12) * kWgDRows * 16, a.d + ((lane - 12) * a.cs_d + row0) * 8, kWgDRows * 16, full + stage);
            if (++stage == kWgStages) { stage = 0; phase ^= 1; }
        }
    } else if (warp == 1) {
        constexpr uint32_t idesc = make_idesc_bf16(128, 32, true, true);
        int stage = 0; uint32_t phase = 0;
        bool first = true;
        // descriptors = per-stage base + compile-time (address >> 4) offsets (cheap issue loop)
        const uint64_t da0 = make_smem_desc(smem_u32(st_s), 128, kWgPlane);
        const uint64_t db0 = make_smem_desc(smem_u32(st_s) + kWgABytes, 128, kWgDRows * 16);
        for (int t = cta; t < total_tiles; t += ncta) {
            mbar_wait(full + stage, phase);
            tc_fence_after();
            if (elect_one()) {
                const uint64_t so = (uint64_t)(stage * (kWgStageBytes >> 4));
#pragma unroll 1
                for (int ks = 0; ks < kTM / 16; ++ks) {
                    const uint64_t db = db0 + so + (uint64_t)(ks * 16);
                    const uint64_t da = da0 + so + (uint64_t)(ks * 16);
                    const uint32_t accum = (first && ks == 0) ? 0u : 1u;
#pragma unroll
                    for (int dy = 0; dy < 3; ++dy)
                        umma_bf16(tmem_base + dy * 32, da + (uint64_t)(dy * kPW), db, idesc, accum);
                }
                umma_commit(empty + stage);
            }
            __syncwarp();
            first = false;
            if (++stage == kWgStages) { stage = 0; phase ^= 1; }
        }
        if (elect_one()) umma_commit(done);
        __syncwarp();
    } else {
        // accumulator row = MN unit * 8 + channel: lane quarter q < 3 holds the horizontal tap q (row = ci), quarter 3
        // the ones unit (row 96 = bias gradient)
        const int q = warp & 3;
        mbar_wait(done, 0);
        tc_fence_after();
        float* out = a.partial + (long long)cta * kWgPartial;
        for (int dy = 0; dy < 3; ++dy) {
            float v[32];
            tmem_ld_32x32(tmem_base + ((uint32_t)(q * 32) << 16) + dy * 32, v);
            float4* dst = nullptr;
            if (q < 3) dst = reinterpret_cast<float4*>(out + ((dy * 3 + q) * 32 + lane) * 32);
            else if (dy == 0 && lane == 0) dst = reinterpret_cast<float4*>(out + 9 * 32 * 32);
            if (dst) {
#pragma unroll
                for (int i = 0; i < 8; ++i) dst[i] = make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem_base, 128);
}

__global__ void __launch_bounds__(256) wgrad_tc_reduce_kernel(const float* __restrict__ partial, int G, float* __restrict__ dw,
                                                              float* __restrict__ db) {
    __shared__ float red[8][33];
    wgrad3x3_reduce_block(partial, G, dw, db, blockIdx.x, red);
}

// + 3 planes of tail padding: MN units 13..15 of the last stage's A operand (results ignored) must stay inside
// the allocation
constexpr size_t kWgradTcSmem = kWgStages * kWgStageBytes + 3 * kWgPlane + (2 * kWgStages + 1) * 8 + 16;

constexpr size_t kConvTcSmem = kWBytes + kStagesTC * kStageBytes + (2 * kStagesTC + 2 * kAccStages) * 8 + 16 + 128;

// ctas_per_sm = 2 for forward / dgrad (74 KB smem, 128 TMEM columns each): independent pipelines per SM
// keep the tensor pipe fed while one CTA's issuing thread waits for data or a free accumulator
static int conv_tc_grid(int total_tiles, int ctas_per_sm = 1) {
    const int slots = sm_budget() * ctas_per_sm;
    return total_tiles < slots ? total_tiles : slots;
}

}  // namespace drq

using namespace drq;

extern "C" {

int drq_debug_conv_stamps(int64_t* buf) { g_conv_stamps = reinterpret_cast<long long*>(buf); return DRQ_OK; }

int drq_set_conv4x1(int mode) {
    const int prev = g_conv4x1;
    if (mode >= 0 && mode <= 4) g_conv4x1 = mode;
    return prev;
}

int64_t drq_wb_elems(int n_images) { return 4ll * ((long long)n_images * kPLB + kSlack) * 8; }

int drq_pack_conv_w_bf16(const float* w, uint16_t* w_fwd, uint16_t* w_dgrad, void* stream) {
    DRQ_REQUIRE(w && w_fwd && w_dgrad, "pack_conv_w: null pointer");
    pack_conv_w_kernel<<<(9216 + 255) / 256, 256, 0, as_stream(stream)>>>(
        w, reinterpret_cast<__nv_bfloat16*>(w_fwd), reinterpret_cast<__nv_bfloat16*>(w_dgrad));
    return check_launch("pack_conv_w_kernel");
}

int drq_conv3x3_fwd_bf16(const uint16_t* in, const uint16_t* w_fwd, const float* bias, uint16_t* out, int N,
                         int hout, int nhwc_out, int64_t feat_rpad, int feat_half, int feat_half_row, void* stream) {
    DRQ_REQUIRE(in && w_fwd && bias && out, "conv3x3_fwd_bf16: null pointer");
    DRQ_REQUIRE(N > 0 && hout > 0 && hout <= kPW - 2, "conv3x3_fwd_bf16: bad dims");
    if (int rc = ensure_smem((const void*)conv3x3_tc_kernel<false>, kConvTcSmem, "conv3x3_fwd_bf16")) return rc;
    ConvTcArgs a{};
    a.in = reinterpret_cast<const __nv_bfloat16*>(in);
    a.cs_in = (long long)N * kPLB + kSlack;
    a.w = reinterpret_cast<const __nv_bfloat16*>(w_fwd);
    a.bias = bias;
    a.out = reinterpret_cast<__nv_bfloat16*>(out);
    a.cs_out = a.cs_in;
    a.n_images = N;
    a.n_pos = hout * kPW;
    a.ntiles = (a.n_pos + kTM - 1) / kTM;
    a.w_valid = hout;
    a.nhwc_out = nhwc_out;
    a.feat_rpad = feat_rpad;
    a.stamps = g_conv_stamps;
    a.feat_half = feat_half > 0 ? feat_half : N;
    a.feat_half_row = feat_half_row;
    DRQ_REQUIRE(nhwc_out != 2 || feat_rpad == (int64_t)hout * hout * 4, "conv3x3_fwd_bf16: TB feature units must be hout*hout*4");
    if (use_conv4x1(N, false))
        return conv4x1_launch(false, a.in, a.cs_in, a.w, bias, nullptr, 0, a.out, a.cs_out, N, hout, nhwc_out, feat_rpad, a.feat_half,
                              feat_half_row, as_stream(stream));
    conv3x3_tc_kernel<false><<<conv_tc_grid(N * a.ntiles, 2), kThreadsTC, kConvTcSmem, as_stream(stream)>>>(a);
    return check_launch("conv3x3_tc_kernel<fwd>");
}

int drq_conv3x3_dgrad_bf16(const uint16_t* dout, const uint16_t* w_dgrad, const uint16_t* act_in, int n_act,
                           uint16_t* din, int N, int hout, void* stream) {
    DRQ_REQUIRE(dout && w_dgrad && act_in && din, "conv3x3_dgrad_bf16: null pointer");
    DRQ_REQUIRE(N > 0 && n_act >= N && hout > 0 && hout <= kPW - 2, "conv3x3_dgrad_bf16: bad dims");
    if (int rc = ensure_smem((const void*)conv3x3_tc_kernel<true>, kConvTcSmem, "conv3x3_dgrad_bf16")) return rc;
    ConvTcArgs a{};
    a.in = reinterpret_cast<const __nv_bfloat16*>(dout);
    a.cs_in = (long long)N * kPLB + kSlack;
    a.w = reinterpret_cast<const __nv_bfloat16*>(w_dgrad);
    a.mask = reinterpret_cast<const __nv_bfloat16*>(act_in);
    a.cs_mask = (long long)n_act * kPLB + kSlack;
    a.out = reinterpret_cast<__nv_bfloat16*>(din);
    a.cs_out = a.cs_in;
    a.n_images = N;
    const int hin = hout + 2;
    a.n_pos = hin * kPW;
    a.ntiles = (a.n_pos + kTM - 1) / kTM;
    a.w_valid = hin;
    a.nhwc_out = 0;
    a.stamps = g_conv_stamps;
    if (use_conv4x1(N, true))
        return conv4x1_launch(true, a.in, a.cs_in, a.w, nullptr, a.mask, a.cs_mask, a.out, a.cs_out, N, hout, 0, 0, 0, 0, as_stream(stream));
    conv3x3_tc_kernel<true><<<conv_tc_grid(N * a.ntiles, 2), kThreadsTC, kConvTcSmem, as_stream(stream)>>>(a);
    return check_launch("conv3x3_tc_kernel<dgrad>");
}

int64_t drq_conv_wgrad_bf16_ws_floats(void) { return 148ll * kWgPartial; }

int drq_conv3x3_wgrad_bf16(const uint16_t* in, int n_in, const uint16_t* dpre, float* partial, float* dw,
                           float* db, int N, int hout, void* stream) {
    DRQ_REQUIRE(in && dpre && partial && (dw != nullptr) == (db != nullptr), "conv3x3_wgrad_bf16: null pointer");
    DRQ_REQUIRE(N > 0 && n_in >= N && hout > 0 && hout <= kPW - 2, "conv3x3_wgrad_bf16: bad dims");
    if (int rc = ensure_smem((const void*)conv3x3_wgrad_tc_kernel, kWgradTcSmem, "conv3x3_wgrad_bf16")) return rc;
    WgradTcArgs a{};
    a.in = reinterpret_cast<const __nv_bfloat16*>(in);
    a.cs_in = (long long)n_in * kPLB + kSlack;
    a.d = reinterpret_cast<const __nv_bfloat16*>(dpre);
    a.cs_d = (long long)N * kPLB + kSlack;
    a.partial = partial;
    a.n_images = N;
    a.ntiles = (hout * kPW + kTM - 1) / kTM;
    const int G = conv_wgrad_ctas(N, hout);                   // tile walkers, one per SM
    conv3x3_wgrad_tc_kernel<<<G, kThreadsTC, kWgradTcSmem, as_stream(stream)>>>(a);
    if (int rc = check_launch("conv3x3_wgrad_tc_kernel")) return rc;
    if (!dw) return DRQ_OK;                                   // partials only: reduced later by drq_conv_wgrad_reduce_multi
    wgrad_tc_reduce_kernel<<<kWgReduceBlocks, 256, 0, as_stream(stream)>>>(partial, G, dw, db);
    return check_launch("wgrad_tc_reduce_kernel");
}

}  // extern "C"

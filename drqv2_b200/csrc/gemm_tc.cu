// bf16 tensor-core GEMM (tcgen05 + TMEM + bulk-async copies) for the heads in bf16 mode: trunk
// Linear(39200->F) forward (split-K) / weight gradient / data gradient and the actor / twin-Q MLP
// layers.  Reference ops: nn.Linear forward/backward of drqv2.py:74-81,100-111.
//
//   C[M,N] = sum_k A(m,k) * B(n,k),  bf16 operands, fp32 accumulation in TMEM.
//
// Operands live in HBM in the tile-blocked layout "TB" (include/drqv2_b200.h):
//   X_tb[row / R][feature / 8][row % R][feature % 8],  R = 128 for activations, 64 for weights,
// i.e. 16-byte units of 8 consecutive features, R rows per unit block, unit blocks of one row block
// adjacent.  Every operand tile of every GEMM of the update is then ONE contiguous 8-32 KB span that
// a single bulk-async copy (TMA engine, mbarrier complete_tx) lands in shared memory already in the
// canonical no-swizzle UMMA layout [unit][row][16 B]:
//   * contraction over features (K-major): units k0/8 .. of row block m0/R;
//   * contraction over rows (MN-major, weight gradients / data gradients): the K chunk is one row
//     block, the M/N extent a run of units.
// (Measured on B200: the copy engine of an SM retires a bulk copy in ~33 ns + bytes / 105 GB/s, so
// 2 KB pieces cap a CTA at ~40 GB/s while 16 KB pieces reach ~85 GB/s; tools/ub/ub_bulk.cu.)
//
// Warp roles (192 threads): warp 0 = copy producer, warp 1 = UMMA issuer, warps 2..5 = epilogue
// (TMEM lane quarters 2,3,0,1).  The code is kept small on purpose (epilogue variant and operand
// mode are template parameters, loops stay rolled): these kernels run for a few microseconds and
// every instruction executes from a cold instruction cache.
#include "pack.cuh"

namespace drq {

DRQ_TRAP_NOTE_HOOK(trap_note_gemm)

using namespace tc;

constexpr int GT_BM = 128, GT_THREADS = 192;
constexpr int RA = DRQ_TB_ACT, RW = DRQ_TB_W;      // rows per block: activations 128, weights 64
constexpr int MODE_KK = DRQ_GEMM_KK, MODE_KMN = DRQ_GEMM_KMN, MODE_MNMN = DRQ_GEMM_MNMN;

struct GemmTcArgs {
    const __nv_bfloat16* A; int units_a;
    const __nv_bfloat16* B; int units_b;
    int M, N, K;
    int batch_inner; long long bs[11];               // inner / outer batch strides: a, b, c, bias, mask; [10] split-K plane stride
    int splitk, k_chunk, nz;                         // nz = batch entries x split-K chunks
    int grid3d;                                      // 1: grid = (n tiles, m tiles, nz), one tile per CTA; 0: persistent 1-D grid
    int accumulate;
    float* Cf; __nv_bfloat16* Cb; long long ldc;     // ldc: fp32 row stride, units of a TB output, WB block stride
    int n_store;                                     // TB outputs: feature columns to write (>= N, zero filled)
    const float* bias;
    const __nv_bfloat16* mask; int units_mask;
    long long* stamps;                               // debug: clock64 timeline of block (0,0,0), or null
};

static long long* g_stamps = nullptr;
#ifdef DRQ_STAMPS
#define GT_STAMP(i) do { if (g.stamps && (blockIdx.x | blockIdx.y | blockIdx.z) == 0) g.stamps[i] = clock64(); } while (0)
#else
#define GT_STAMP(i) do { } while (0)
#endif

// SMALL: a two-stage pipeline (<= 66 KB of shared memory instead of <= 196 KB) for the launches that run BESIDE the
// encoder backward (the actor pass): the persistent conv kernels keep 148 KB of every SM until they end, and a GEMM
// CTA that does not fit into the remaining 79 KB waits for the running conv kernel to finish - measured as ~60 us
// of the update.  These GEMMs are latency-bound, so the shallower pipeline costs them little.
template <int MODE, int BN, int EPI, int SMALL = 0>
struct GemmCfg {
    static constexpr int BK = MODE == MODE_MNMN ? RA : 64;                 // contraction extent per stage
    static constexpr int A_BYTES = MODE == MODE_MNMN ? 16 * RA * 16 : 8 * RA * 16;
    static constexpr int B_BYTES = MODE == MODE_KK ? 8 * BN * 16 : (MODE == MODE_KMN ? (BN / 8) * RW * 16 : (BN / 8) * RA * 16);
    static constexpr int STAGE = A_BYTES + B_BYTES;
    // epilogue scratch: 2 bias rows + (fp32 outputs only) per epilogue warp one fp32 transpose tile (32 x 33, or the
    // whole 32 x BN tile for the trunk weight gradient's re-ordering store)
    static constexpr bool XPOSE = EPI == DRQ_TEPI_F32 || EPI == DRQ_TEPI_TRUNK_WGRAD;
    static constexpr int XP_FLOATS = EPI == DRQ_TEPI_TRUNK_WGRAD ? 32 * (BN + 1) : (XPOSE ? 32 * 33 : 0);
    static constexpr int EPI_BYTES = 2 * BN * 4 + 4 * XP_FLOATS * 4;
    static constexpr int BUDGET = 196 * 1024 - EPI_BYTES;
    static constexpr int STAGES = SMALL ? 2 : (BUDGET / STAGE > 6 ? 6 : BUDGET / STAGE);
    static constexpr int ACC = 2;                                          // TMEM accumulator stages
    static constexpr int B_COPIES = (MODE == MODE_KK && BN == 128) ? 2 : 1;   // K-major weight tiles are 64-row blocks
    static constexpr size_t SMEM = (size_t)STAGES * STAGE + EPI_BYTES + (2 * STAGES + 2 * ACC) * 8 + 16;
};

// Tile `t` of the launch: n tile fastest, then m tile, then (batch entry, split-K chunk).
struct TileInfo {
    int m0, n0, k_begin, k_end;
    long long off_a, off_b, off_c, off_bias, off_mask;
};
template <int BN>
__device__ __forceinline__ TileInfo tile_info(const GemmTcArgs& g, int t, int nt, int mt) {
    TileInfo ti;
    // Integer divisions are ~20 cold instructions each on the way to the first copy.  When the launch has no more
    // tiles than SMs the grid is 3-D and the tile is the block index; only the persistent 1-D grid decodes.
    int in, im, z;
    if (g.grid3d) {
        in = blockIdx.x; im = blockIdx.y; z = blockIdx.z;
    } else {
        in = t; im = 0; z = 0;
        if (nt > 1) { const int rest = t / nt; in = t - rest * nt; t = rest; } else { in = 0; }
        if (mt > 1) { z = t / mt; im = t - z * mt; } else { z = t; }
    }
    ti.m0 = im * GT_BM; ti.n0 = in * BN;
    int zs = 0, zb = z;                                  // split-K chunk, batch entry
    ti.k_begin = 0; ti.k_end = g.K;
    if (g.splitk > 1) {
        zb = z / g.splitk; zs = z - zb * g.splitk;
        ti.k_begin = zs * g.k_chunk;
        ti.k_end = min(g.K, ti.k_begin + g.k_chunk);
    }
    int zi = zb, zo = 0;
    if (zb >= g.batch_inner) { zo = zb / g.batch_inner; zi = zb - zo * g.batch_inner; }
    ti.off_a = zi * g.bs[0] + zo * g.bs[5];
    ti.off_b = zi * g.bs[1] + zo * g.bs[6];
    ti.off_c = zi * g.bs[2] + zo * g.bs[7] + zs * g.bs[10];
    ti.off_bias = zi * g.bs[3] + zo * g.bs[8];
    ti.off_mask = zi * g.bs[4] + zo * g.bs[9];
    return ti;
}

// Persistent over output tiles: CTA b works on tiles b, b + gridDim.x, ...; the operand pipeline runs across
// tile boundaries and the accumulator is double-buffered in TMEM, so the epilogue of one tile overlaps
// the loads and UMMAs of the next (the skinny GEMMs of the trunk backward have 300-600 tiles).
template <int MODE, int BN, int EPI, int SMALL = 0>
__global__ void __launch_bounds__(GT_THREADS, 1) gemm_tc_kernel(const GemmTcArgs g) {
    using Cfg = GemmCfg<MODE, BN, EPI, SMALL>;
    extern __shared__ __align__(128) uint8_t smem[];
    constexpr int STAGES = Cfg::STAGES, STAGE = Cfg::STAGE, A_BYTES = Cfg::A_BYTES, BK = Cfg::BK, ACC = Cfg::ACC;
    float* bias_s = reinterpret_cast<float*>(smem + STAGES * STAGE);      // [2][BN]
    float* xpose_s = bias_s + 2 * BN;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + STAGES * STAGE + Cfg::EPI_BYTES);
    uint64_t* full = bars;
    uint64_t* empty = bars + STAGES;
    uint64_t* tfull = bars + 2 * STAGES;
    uint64_t* tempty = tfull + ACC;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + ACC);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (tid == 0) GT_STAMP(0);
    const int nt = (g.N + BN - 1) / BN, mt = (g.M + GT_BM - 1) / GT_BM;
    const int total_tiles = g.grid3d ? 1 : nt * mt * g.nz;
    const int t_first = g.grid3d ? 0 : blockIdx.x, t_step = g.grid3d ? 1 : gridDim.x;
    // Warp 0 (the copy producer) initialises the barriers and starts copying at once; the other warps meet it
    // on named barrier 2 (warp 0 only arrives), so the TMEM allocation and the block-wide rendezvous are off
    // the path to the first operand bytes.
    if (warp == 0) {
        if (lane == 0) {
            for (int i = 0; i < STAGES; ++i) { mbar_init(full + i, 1 + Cfg::B_COPIES); mbar_init(empty + i, 1); }
            for (int i = 0; i < ACC; ++i) { mbar_init(tfull + i, 1); mbar_init(tempty + i, 4); }
            fence_barrier_init();
        }
        __syncwarp();
        asm volatile("bar.arrive 2, 192;" ::: "memory");
    } else {
        if (warp == 1) {
            tmem_alloc(tmem_slot, ACC * BN);
            tmem_relinquish();
        }
        tc_fence_before();
        asm volatile("bar.sync 2, 192;" ::: "memory");
        tc_fence_after();
    }
    const uint32_t tmem_base = warp == 0 ? 0u : *tmem_slot;
    if (tid == 0) GT_STAMP(1);

    if (warp == 0) {
        // ------------------------------------------------ producer: lane 0 copies A tiles, lanes 1.. B tiles;
        // each announces its own byte count (full[] counts 1 + B_COPIES arrivals)
        if (lane < 1 + Cfg::B_COPIES) {
            int stage = 0; uint32_t phase = 0;
#pragma unroll 1
            for (int t = t_first; t < total_tiles; t += t_step) {
                const TileInfo ti = tile_info<BN>(g, t, nt, mt);
                const int m0 = ti.m0, n0 = ti.n0, k_begin = ti.k_begin, k_end = ti.k_end;
                const int nk = (k_end - k_begin + BK - 1) / BK;
                const __nv_bfloat16* src;
                long long kstep;                 // elements between consecutive k blocks
                uint32_t bytes = 0;              // MN-major: constant bytes per stage
                uint32_t unit_bytes = 0;         // K-major: bytes per K unit ...
                int units_left = 0;              // ... and units remaining from k_begin
                if (lane == 0) {
                    if (MODE == MODE_MNMN) {     // activation [row block kb][units m0/8 ..][128][8]
                        src = g.A + ti.off_a + ((long long)(k_begin / RA) * g.units_a + m0 / 8) * RA * 8;
                        kstep = (long long)g.units_a * RA * 8;
                        bytes = min(16, g.units_a - m0 / 8) * RA * 16;
                    } else {                     // activation [row block m0/128][units k/8 ..][128][8]
                        src = g.A + ti.off_a + ((long long)(m0 / RA) * g.units_a + k_begin / 8) * RA * 8;
                        kstep = 8ll * RA * 8;
                        unit_bytes = RA * 16; units_left = (k_end - k_begin + 15) / 16 * 2;
                    }
                } else {
                    if (MODE == MODE_KK) {       // weight [row block n0/64 (+1)][units k/8 ..][64][8]
                        src = g.B + ti.off_b + ((long long)(n0 / RW + lane - 1) * g.units_b + k_begin / 8) * RW * 8;
                        kstep = 8ll * RW * 8;
                        unit_bytes = RW * 16; units_left = (k_end - k_begin + 15) / 16 * 2;
                    } else if (MODE == MODE_KMN) {   // weight [row block kb (64 k rows)][units n0/8 ..][64][8]
                        src = g.B + ti.off_b + ((long long)(k_begin / RW) * g.units_b + n0 / 8) * RW * 8;
                        kstep = (long long)g.units_b * RW * 8;
                        bytes = min(BN / 8, g.units_b - n0 / 8) * RW * 16;
                    } else {                     // activation [row block kb][units n0/8 ..][128][8]
                        src = g.B + ti.off_b + ((long long)(k_begin / RA) * g.units_b + n0 / 8) * RA * 8;
                        kstep = (long long)g.units_b * RA * 8;
                        bytes = min(BN / 8, g.units_b - n0 / 8) * RA * 16;
                    }
                }
                const uint32_t dst_off = lane == 0 ? 0 : A_BYTES + (lane - 1) * (8 * RW * 16);
#pragma unroll 1
                for (int kb = 0; kb < nk; ++kb) {
                    const uint32_t nbytes = unit_bytes ? min(8, units_left - kb * 8) * unit_bytes : bytes;
                    mbar_wait(empty + stage, phase ^ 1);
                    mbar_arrive_expect_tx(full + stage, nbytes);
                    bulk_g2s(smem + stage * STAGE + dst_off, src, nbytes, full + stage);
                    src += kstep;
                    if (++stage == STAGES) { stage = 0; phase ^= 1; }
                }
            }
        }
        if (lane == 0) GT_STAMP(3);
    } else if (warp == 1) {
        // ------------------------------------------------ UMMA issuer
        constexpr uint32_t idesc = make_idesc_bf16(GT_BM, BN / Cfg::B_COPIES, MODE == MODE_MNMN, MODE != MODE_KK);
        int stage = 0; uint32_t phase = 0; int acc = 0; uint32_t acc_phase = 0;
#pragma unroll 1
        for (int t = t_first; t < total_tiles; t += t_step) {
            const TileInfo ti = tile_info<BN>(g, t, nt, mt);
            const int nk = (ti.k_end - ti.k_begin + BK - 1) / BK;
            mbar_wait(tempty + acc, acc_phase ^ 1);
            const uint32_t d_tmem = tmem_base + acc * BN;
#pragma unroll 1
            for (int kb = 0; kb < nk; ++kb) {
                mbar_wait(full + stage, phase);
                tc_fence_after();
                if (lane == 0 && kb == 0) GT_STAMP(4);
                if (lane == 0 && kb == nk - 1) GT_STAMP(5);
                if (elect_one()) {
                    const int ksteps = min(BK / 16, (ti.k_end - ti.k_begin - kb * BK + 15) / 16);
                    const uint32_t a_addr = smem_u32(smem + stage * STAGE), b_addr = a_addr + A_BYTES;
#pragma unroll 1
                    for (int ks = 0; ks < ksteps; ++ks) {
                        const uint64_t da = MODE == MODE_MNMN ? make_smem_desc(a_addr + ks * 256, 128, RA * 16)
                                                              : make_smem_desc(a_addr + ks * 2 * RA * 16, RA * 16, 128);
                        const uint64_t db = MODE == MODE_KK ? make_smem_desc(b_addr + ks * 2 * RW * 16, RW * 16, 128)
                                           : MODE == MODE_KMN ? make_smem_desc(b_addr + ks * 256, 128, RW * 16)
                                                              : make_smem_desc(b_addr + ks * 256, 128, RA * 16);
                        umma_bf16(d_tmem, da, db, idesc, (kb | ks) ? 1u : 0u);
                        if (Cfg::B_COPIES == 2)
                            umma_bf16(d_tmem + 64, da, make_smem_desc(b_addr + 8 * RW * 16 + ks * 2 * RW * 16, RW * 16, 128), idesc,
                                      (kb | ks) ? 1u : 0u);
                    }
                    umma_commit(empty + stage);
                    if (kb == nk - 1) umma_commit(tfull + acc);
                }
                __syncwarp();
                if (++stage == STAGES) { stage = 0; phase ^= 1; }
            }
            if (++acc == ACC) { acc = 0; acc_phase ^= 1; }
        }
    } else {
        // ------------------------------------------------ epilogue.  While the main loop of a tile runs these warps
        // stage its bias row in shared memory and pull their ReLU-mask rows into registers.
        const int q = warp & 3;
        const int et = tid - 64;                                // 0..127
        constexpr bool TB_OUT = EPI == DRQ_TEPI_RELU_BF16 || EPI == DRQ_TEPI_MASK_BF16;
        constexpr bool MASKED = EPI == DRQ_TEPI_MASK_BF16 || EPI == DRQ_TEPI_TRUNK_DGRAD;
        float* xp = xpose_s + q * Cfg::XP_FLOATS;
        int acc = 0; uint32_t acc_phase = 0; int it = 0;
#pragma unroll 1
        for (int t = t_first; t < total_tiles; t += t_step, ++it) {
            const TileInfo ti = tile_info<BN>(g, t, nt, mt);
            const int m0 = ti.m0, n0 = ti.n0;
            const long long off_c = ti.off_c;
            const int m = m0 + q * 32 + lane;
            const long long mblk = m / RA, mrow = m % RA;          // TB row block / row inside it
            const float* bias = g.bias ? g.bias + ti.off_bias : nullptr;
            const __nv_bfloat16* mask = g.mask ? g.mask + ti.off_mask : nullptr;
            float* bs = bias_s + (it & 1) * BN;
            if (EPI == DRQ_TEPI_F32 || EPI == DRQ_TEPI_RELU_BF16) {
                for (int j = et; j < BN; j += 128) bs[j] = (bias && n0 + j < g.N) ? __ldg(bias + n0 + j) : 0.f;
                asm volatile("bar.sync 1, 128;" ::: "memory");
            }
            uint4 mk[MASKED ? BN / 8 : 1];
            if (MASKED && m < g.M) {
#pragma unroll
                for (int u = 0; u < BN / 8; ++u)
                    mk[u] = (n0 + 8 * u < g.units_mask * 8)
                                ? __ldg(reinterpret_cast<const uint4*>(mask + ((mblk * g.units_mask + n0 / 8 + u) * RA + mrow) * 8))
                                : make_uint4(0, 0, 0, 0);
            }
            mbar_wait(tfull + acc, acc_phase);
            tc_fence_after();
            if (tid == 64) GT_STAMP(6);
            const uint32_t t_acc = tmem_base + ((uint32_t)(q * 32) << 16) + acc * BN;
            if (EPI == DRQ_TEPI_TRUNK_WGRAD) {
                // The tile's 128 columns are 16 feature units = 16 consecutive pixels x 8 channels of one channel
                // group; the reference layout (drqv2.py:66) wants column c*1225 + yx.  Stage the warp's 32 rows x
                // 128 columns in shared memory and write, per instruction, two rows x 16 consecutive pixels
                // of one channel: 64-byte runs instead of 32 scattered floats.
                constexpr int XP = BN + 1;
                if (m0 + q * 32 < g.M) {
#pragma unroll
                    for (int c0 = 0; c0 < BN; c0 += 32) {
                        float v[32];
                        tmem_ld_32x32(t_acc + c0, v);
#pragma unroll
                        for (int j = 0; j < 32; ++j) xp[lane * XP + c0 + j] = v[j];
                    }
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(tempty + acc);       // accumulator drained: the next tile may overwrite it
                if (m0 + q * 32 < g.M) {
                    const int px = lane & 15, rsel = lane >> 4;
                    const int u = n0 / 8 + px;
                    const int cu = u / 1225, yx = u - cu * 1225;
                    const bool col_ok = n0 + px * 8 < g.N;
                    float* cbase = g.Cf + off_c + (long long)(cu * 8) * 1225 + yx;
                    const int rows = min(32, g.M - (m0 + q * 32));
#pragma unroll 1
                    for (int ch = 0; ch < 8; ++ch) {
                        float vals[16];
#pragma unroll
                        for (int rp = 0; rp < 16; ++rp) vals[rp] = xp[(rp * 2 + rsel) * XP + px * 8 + ch];
                        float* cb = cbase + (long long)(m0 + q * 32 + rsel) * g.ldc + ch * 1225;
#pragma unroll
                        for (int rp = 0; rp < 16; ++rp)
                            if (rp * 2 + rsel < rows && col_ok) cb[(long long)(rp * 2) * g.ldc] = vals[rp];
                    }
                    __syncwarp();
                }
            } else {
#pragma unroll
                for (int c0 = 0; c0 < BN; c0 += 32) {
                    const int nb = n0 + c0;
                    if (nb >= (TB_OUT ? g.n_store : g.N)) break;
                    float v[32];
                    tmem_ld_32x32(t_acc + c0, v);
                    if (EPI == DRQ_TEPI_F32) {
                        // warp-local transpose through shared memory: every store instruction writes one row's 32
                        // consecutive floats (128 B) instead of 32 rows' single floats
                        __syncwarp();
#pragma unroll
                        for (int j = 0; j < 32; ++j) xp[lane * 33 + j] = v[j] + bs[c0 + j];
                        __syncwarp();
                        const int n = nb + lane;
                        const int rows = min(32, g.M - (m0 + q * 32));
                        float* cbase = g.Cf + off_c + (long long)(m0 + q * 32) * g.ldc + n;
                        if (n < g.N) {
#pragma unroll 4
                            for (int r = 0; r < rows; ++r) {
                                float x = xp[r * 33 + lane];
                                if (g.accumulate) x += cbase[r * g.ldc];
                                cbase[r * g.ldc] = x;
                            }
                        }
                        continue;
                    }
                    if (m >= g.M) continue;
                    if (EPI == DRQ_TEPI_TRUNK_DGRAD) {
                        // columns nb..nb+31 = 4 feature units (channel group cu, pixels yx..): mask by feature > 0 and
                        // scatter into conv4's WB gradient (block cu, the pixel's row)
#pragma unroll
                        for (int c = 0; c < 4; ++c) {
                            const int u = nb / 8 + c;
                            const int cu = u / 1225, yx = u - cu * 1225;
                            const int yy = yx / 35, xx = yx - yy * 35;
                            const long long row = (long long)m * DRQ_PLB + DRQ_GUARD + yy * DRQ_PW + xx;
                            const uint4 mv = mk[MASKED ? c0 / 8 + c : 0];
                            const uint32_t mw[4] = {mv.x, mv.y, mv.z, mv.w};
                            uint32_t pk[4];
#pragma unroll
                            for (int j = 0; j < 4; ++j)
                                pk[j] = pack_bf16x2(bf16_lo(mw[j]) > 0.f ? v[8 * c + 2 * j] : 0.f,
                                                    bf16_hi(mw[j]) > 0.f ? v[8 * c + 2 * j + 1] : 0.f);
                            *reinterpret_cast<uint4*>(g.Cb + (cu * g.ldc + row) * 8) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
                        }
                    } else {
                        // TB bf16 output (units = ldc): unit nb/8 + c, row m; columns >= N are zeros up to n_store
#pragma unroll
                        for (int c = 0; c < 4; ++c) {
                            const int n8 = nb + 8 * c;
                            if (n8 < g.n_store) {
                                const uint4 mv = mk[MASKED ? c0 / 8 + c : 0];
                                const uint32_t mw[4] = {mv.x, mv.y, mv.z, mv.w};
                                uint32_t pk[4];
#pragma unroll
                                for (int j = 0; j < 4; ++j) {
                                    float lo = v[8 * c + 2 * j], hi = v[8 * c + 2 * j + 1];
                                    const int n = n8 + 2 * j;
                                    if (EPI == DRQ_TEPI_RELU_BF16) {
                                        lo = n < g.N ? fmaxf(lo + bs[c0 + 8 * c + 2 * j], 0.f) : 0.f;
                                        hi = n + 1 < g.N ? fmaxf(hi + bs[c0 + 8 * c + 2 * j + 1], 0.f) : 0.f;
                                    } else {
                                        lo = (n < g.N && bf16_lo(mw[j]) > 0.f) ? lo : 0.f;
                                        hi = (n + 1 < g.N && bf16_hi(mw[j]) > 0.f) ? hi : 0.f;
                                    }
                                    pk[j] = pack_bf16x2(lo, hi);
                                }
                                *reinterpret_cast<uint4*>(g.Cb + off_c + ((mblk * g.ldc + n8 / 8) * RA + mrow) * 8) =
                                    make_uint4(pk[0], pk[1], pk[2], pk[3]);
                            }
                        }
                    }
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(tempty + acc);
            }
            if (++acc == ACC) { acc = 0; acc_phase ^= 1; }
        }
    }
    if (tid == 64) GT_STAMP(7);
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem_base, ACC * BN);
    if (tid == 0) GT_STAMP(8);
}

static int g_gemm_small = 0;

template <int MODE, int BN, int EPI, int SMALL = 0>
static int launch_gemm_tc(GemmTcArgs& g, int batch, cudaStream_t s) {
    using Cfg = GemmCfg<MODE, BN, EPI, SMALL>;
    if (int rc = ensure_smem((const void*)gemm_tc_kernel<MODE, BN, EPI, SMALL>, Cfg::SMEM, "gemm_bf16")) return rc;
    g.nz = g.splitk * batch;
    const int nt = (g.N + BN - 1) / BN, mt = (g.M + GT_BM - 1) / GT_BM;
    const int tiles = nt * mt * g.nz;
    const int sms = drq_device_sm_count();
    g.grid3d = tiles <= sms ? 1 : 0;
    gemm_tc_kernel<MODE, BN, EPI, SMALL><<<g.grid3d ? dim3(nt, mt, g.nz) : dim3(sms), GT_THREADS, Cfg::SMEM, s>>>(g);
    return check_launch("gemm_tc_kernel");
}

__global__ void __launch_bounds__(256)
pack_linear_tb_kernel(const float* __restrict__ w, __nv_bfloat16* __restrict__ out, int rows, int cols, int units) {
    pack_linear_tb_block(w, out, rows, cols, units, blockIdx.x, blockIdx.y, threadIdx.x);
}

__global__ void __launch_bounds__(256)
pack_trunk_tb_kernel(const float* __restrict__ w, __nv_bfloat16* __restrict__ out, int rows) {
    __shared__ float tile[32][33];
    pack_trunk_tb_block(w, out, rows, blockIdx.x, blockIdx.y, threadIdx.x, tile);
}

// features fp32 [rows][39200] in the reference's flatten order (drqv2.py:66) -> TB(128) bf16 in the encoder-output
// order (stage API: update_critic / update_actor on externally supplied features)
__global__ void __launch_bounds__(256)
pack_features_tb_kernel(const float* __restrict__ f, __nv_bfloat16* __restrict__ out, int rows) {
    __shared__ float tile[32][33];
    pack_trunk_tb_block<DRQ_TB_ACT>(f, out, rows, blockIdx.x, blockIdx.y, threadIdx.x, tile);
}

}  // namespace drq

using namespace drq;

extern "C" {

int drq_gemm_bf16(const uint16_t* A, int units_a, const uint16_t* B, int units_b, int mode, void* C, int64_t ldc,
                  int n_store, const float* bias, const uint16_t* mask, int units_mask, int M, int N, int K,
                  int epilogue, int accumulate, int batch, int batch_inner, const int64_t* strides, int splitk,
                  int bn, void* stream) {
    DRQ_REQUIRE(A && B && C, "gemm_bf16: null pointer");
    DRQ_REQUIRE(M > 0 && N > 0 && K > 0, "gemm_bf16: bad dims");
    DRQ_REQUIRE(mode >= MODE_KK && mode <= MODE_MNMN, "gemm_bf16: bad operand mode");
    DRQ_REQUIRE(((uintptr_t)A % 16) == 0 && ((uintptr_t)B % 16) == 0, "gemm_bf16: operands must be 16-byte aligned");
    DRQ_REQUIRE(batch >= 1 && batch_inner >= 1 && splitk >= 1, "gemm_bf16: batch/splitk");
    DRQ_REQUIRE(epilogue >= DRQ_TEPI_F32 && epilogue <= DRQ_TEPI_TRUNK_DGRAD, "gemm_bf16: bad epilogue");
    DRQ_REQUIRE(!((epilogue == DRQ_TEPI_MASK_BF16 || epilogue == DRQ_TEPI_TRUNK_DGRAD) && !mask), "gemm_bf16: mask missing");
    DRQ_REQUIRE(!(epilogue == DRQ_TEPI_RELU_BF16 && !bias), "gemm_bf16: bias missing");
    DRQ_REQUIRE(!(splitk > 1 && (epilogue != DRQ_TEPI_F32 || mode == MODE_MNMN)), "gemm_bf16: split-K writes fp32 partials (modes KK, KMN)");
    // the zero columns [N, n_store) of a TB output are written by the tiles of N: a column past the last one would be left
    // unwritten (a caller's stale values read as features), so such an n_store is refused
    DRQ_REQUIRE(!((epilogue == DRQ_TEPI_RELU_BF16 || epilogue == DRQ_TEPI_MASK_BF16) && n_store > (N + bn - 1) / bn * bn),
                "gemm_bf16: n_store %d lies past the last %d-wide N tile (N = %d)", n_store, bn, N);
    DRQ_REQUIRE(!(mode == MODE_KK && bn == 128 && ((N + RW - 1) / RW) % 2 != 0),
                "gemm_bf16: K-major bn = 128 reads pairs of 64-row weight blocks (N = %d)", N);
    // the blocked extents must cover what the tiles touch
    if (mode == MODE_MNMN) {
        DRQ_REQUIRE(units_a * 8 >= M && units_b * 8 >= N, "gemm_bf16: MN-major units smaller than M / N");
    } else {
        DRQ_REQUIRE(units_a * 8 >= K, "gemm_bf16: A units smaller than K");
        DRQ_REQUIRE(mode == MODE_KK ? units_b * 8 >= K : units_b * 8 >= N, "gemm_bf16: B units too small");
    }
    GemmTcArgs g{};
    g.A = reinterpret_cast<const __nv_bfloat16*>(A); g.units_a = units_a;
    g.B = reinterpret_cast<const __nv_bfloat16*>(B); g.units_b = units_b;
    g.M = M; g.N = N; g.K = K;
    g.batch_inner = batch_inner;
    for (int i = 0; i < 11; ++i) g.bs[i] = strides ? strides[i] : 0;
    for (int i = 0; i < 10; ++i)
        if (i % 5 == 0 || i % 5 == 1 || i % 5 == 4)
            DRQ_REQUIRE(g.bs[i] % 8 == 0, "gemm_bf16: bf16 batch strides must keep 16-byte alignment");
    g.splitk = splitk; g.k_chunk = K;
    if (splitk > 1) {
        int chunk = (K + splitk - 1) / splitk;
        chunk = (chunk + 127) / 128 * 128;
        g.k_chunk = chunk;
        DRQ_REQUIRE((long long)chunk * (splitk - 1) < K, "gemm_bf16: splitk %d leaves empty chunks for K=%d", splitk, K);
    }
    g.accumulate = accumulate;
    g.Cf = reinterpret_cast<float*>(C); g.Cb = reinterpret_cast<__nv_bfloat16*>(C); g.ldc = ldc;
    g.n_store = n_store > N ? n_store : N;
    g.bias = splitk > 1 ? nullptr : bias;
    g.mask = reinterpret_cast<const __nv_bfloat16*>(mask); g.units_mask = units_mask;
    g.stamps = g_stamps;
    cudaStream_t s = as_stream(stream);
#define GT_CASE(MODE_, BN_, EPI_) \
    if (mode == MODE_ && bn == BN_ && epilogue == EPI_) return launch_gemm_tc<MODE_, BN_, EPI_>(g, batch, s);
#define GT_SMALL(MODE_, BN_, EPI_) \
    if (g_gemm_small && mode == MODE_ && bn == BN_ && epilogue == EPI_) return launch_gemm_tc<MODE_, BN_, EPI_, 1>(g, batch, s);
    GT_SMALL(MODE_KK, 64, DRQ_TEPI_F32)
    GT_SMALL(MODE_KK, 64, DRQ_TEPI_RELU_BF16)
    GT_SMALL(MODE_KMN, 64, DRQ_TEPI_F32)
    GT_SMALL(MODE_KMN, 64, DRQ_TEPI_MASK_BF16)
    GT_CASE(MODE_KK, 64, DRQ_TEPI_F32)
    GT_CASE(MODE_KK, 64, DRQ_TEPI_RELU_BF16)
    GT_CASE(MODE_KK, 128, DRQ_TEPI_F32)
    GT_CASE(MODE_KK, 128, DRQ_TEPI_RELU_BF16)
    GT_CASE(MODE_KMN, 64, DRQ_TEPI_F32)
    GT_CASE(MODE_KMN, 64, DRQ_TEPI_MASK_BF16)
    GT_CASE(MODE_KMN, 128, DRQ_TEPI_MASK_BF16)
    GT_CASE(MODE_KMN, 128, DRQ_TEPI_TRUNK_DGRAD)
    GT_CASE(MODE_MNMN, 64, DRQ_TEPI_F32)
    GT_CASE(MODE_MNMN, 128, DRQ_TEPI_F32)
    GT_CASE(MODE_MNMN, 128, DRQ_TEPI_TRUNK_WGRAD)
#undef GT_CASE
#undef GT_SMALL
    set_error("gemm_bf16: no kernel for mode %d, bn %d, epilogue %d", mode, bn, epilogue);
    return DRQ_ERR_INVALID;
}

int drq_set_gemm_small(int on) { g_gemm_small = on ? 1 : 0; return DRQ_OK; }

int drq_debug_gemm_stamps(int64_t* buf) { g_stamps = reinterpret_cast<long long*>(buf); return DRQ_OK; }

int drq_pack_linear_tb(const float* w, uint16_t* out, int rows, int cols, void* stream) {
    DRQ_REQUIRE(w && out && rows > 0 && cols > 0, "pack_linear_tb: bad args");
    const int units = (cols + 15) / 16 * 2;
    const int rpad = (rows + RW - 1) / RW * RW;
    pack_linear_tb_kernel<<<dim3((rpad + 255) / 256, units), 256, 0, as_stream(stream)>>>(
        w, reinterpret_cast<__nv_bfloat16*>(out), rows, cols, units);
    return check_launch("pack_linear_tb_kernel");
}

int drq_pack_trunk_tb(const float* w, uint16_t* out, int rows, void* stream) {
    DRQ_REQUIRE(w && out && rows > 0, "pack_trunk_tb: bad args");
    const int rpad = (rows + RW - 1) / RW * RW;
    pack_trunk_tb_kernel<<<dim3((1225 + 31) / 32, rpad), 256, 0, as_stream(stream)>>>(
        w, reinterpret_cast<__nv_bfloat16*>(out), rows);
    return check_launch("pack_trunk_tb_kernel");
}

int drq_pack_features_tb(const float* feat, uint16_t* out, int rows, void* stream) {
    DRQ_REQUIRE(feat && out && rows > 0, "pack_features_tb: bad args");
    DRQ_REQUIRE(((uintptr_t)out % 16) == 0, "pack_features_tb: output must be 16-byte aligned");
    const int rpad = (rows + RA - 1) / RA * RA;
    pack_features_tb_kernel<<<dim3((1225 + 31) / 32, rpad), 256, 0, as_stream(stream)>>>(
        feat, reinterpret_cast<__nv_bfloat16*>(out), rows);
    return check_launch("pack_features_tb_kernel");
}

}  // extern "C"

// fp32 (parity-mode) encoder kernels: CUDA-core implicit-GEMM convolutions on the
// wide-plane layout.  Reference: Encoder drqv2.py:48-67, RandomShiftsAug drqv2.py:14-45.
//
// Wide plane: every activation is [N][32][kPlane] with row stride 41, so a 3x3
// stride-1 tap (ky,kx) is the constant offset ky*41+kx and
//   fwd  : out[d][p] = relu(b[d] + sum_{s,tap} w[d][s][tap] * in[s][p + off(tap)])
//   dgrad: din[d][q] = mask * sum_{s,tap} w[s][d][tap] * dout[s][q - off(tap)]
// are the same shifted GEMM (M = positions, N = 32, K = 288) with the sign of the
// offset flipped and the weight tile transposed.
#include "common.cuh"

namespace drq {

constexpr int kTP = 128;              // output positions per block
constexpr int kHalo = 2 * kPW + 2;    // 84: largest tap offset
constexpr int kWin = kTP + kHalo;     // 212 staged positions per channel
constexpr int kWgradBlocks = 296;     // 2 per SM on B200 (148 SMs); fixed => bitwise reproducible
constexpr int kC1Rows = 7;            // conv1 output rows per tile (41 = 5*7 + 6)
constexpr int kC1Tiles = 6;
constexpr int kC1InRows = 2 * kC1Rows + 1;  // 15 input rows per tile

// ---------------------------------------------------------------- conv 32->32, fwd + dgrad
template <bool DGRAD>
__global__ void __launch_bounds__(128)
conv3x3_wide_kernel(const float* __restrict__ in, const float* __restrict__ w,
                    const float* __restrict__ bias, const float* __restrict__ act_mask,
                    float* __restrict__ out, int n_pos, int w_valid, int compact_out) {
    extern __shared__ __align__(16) float smem[];
    float* in_s = smem;                 // [32][kWin]
    float* w_s = smem + kCh * kWin;     // [9][32 s][32 d]
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int n = blockIdx.y;
    const int p0 = blockIdx.x * kTP;

    // weights: global [co][ci][tap] -> smem [tap][s][d]
    for (int i = tid; i < kCh * kCh * 9; i += 128) {
        const int co = i / (kCh * 9), ci = (i / 9) % kCh, tap = i % 9;
        const int s = DGRAD ? co : ci, d = DGRAD ? ci : co;
        w_s[(tap * kCh + s) * kCh + d] = __ldg(w + i);
    }
    // input window
    const int base = DGRAD ? p0 - kHalo : p0;
    const float* in_n = in + (long long)n * kCh * kPlane;
    for (int i = tid; i < kCh * kWin; i += 128) {
        const int s = i / kWin, l = i - s * kWin;
        const int idx = base + l;
        in_s[i] = (idx >= 0 && idx < kPlane) ? __ldg(in_n + s * kPlane + idx) : 0.f;
    }
    __syncthreads();

    float acc[4][8];
#pragma unroll
    for (int j = 0; j < 4; ++j)
#pragma unroll
        for (int c = 0; c < 8; ++c) acc[j][c] = 0.f;

    const int d0 = warp * 8;
#pragma unroll 2
    for (int s = 0; s < kCh; ++s) {
        const float* row = in_s + s * kWin + lane;
#pragma unroll
        for (int tap = 0; tap < 9; ++tap) {
            const int off = (tap / 3) * kPW + (tap % 3);
            const int o = DGRAD ? kHalo - off : off;
            const float4 wa = *reinterpret_cast<const float4*>(w_s + (tap * kCh + s) * kCh + d0);
            const float4 wb = *reinterpret_cast<const float4*>(w_s + (tap * kCh + s) * kCh + d0 + 4);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const float v = row[32 * j + o];
                acc[j][0] = fmaf(v, wa.x, acc[j][0]);
                acc[j][1] = fmaf(v, wa.y, acc[j][1]);
                acc[j][2] = fmaf(v, wa.z, acc[j][2]);
                acc[j][3] = fmaf(v, wa.w, acc[j][3]);
                acc[j][4] = fmaf(v, wb.x, acc[j][4]);
                acc[j][5] = fmaf(v, wb.y, acc[j][5]);
                acc[j][6] = fmaf(v, wb.z, acc[j][6]);
                acc[j][7] = fmaf(v, wb.w, acc[j][7]);
            }
        }
    }

#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const int p = p0 + lane + 32 * j;
        if (p >= n_pos) continue;
        const int y = p / kPW, x = p - y * kPW;
#pragma unroll
        for (int c = 0; c < 8; ++c) {
            const int d = d0 + c;
            if (!DGRAD) {
                const float v = fmaxf(acc[j][c] + __ldg(bias + d), 0.f);
                if (compact_out) {
                    if (x < w_valid)
                        out[((long long)n * kCh + d) * (w_valid * w_valid) + y * w_valid + x] = v;
                } else {
                    out[((long long)n * kCh + d) * kPlane + p] = v;
                }
            } else {
                const long long o = ((long long)n * kCh + d) * kPlane + p;
                const float m = (x < w_valid && __ldg(act_mask + o) > 0.f) ? acc[j][c] : 0.f;
                out[o] = m;
            }
        }
    }
}

// ---------------------------------------------------------------- conv 32->32, wgrad
// Each block walks a fixed list of (image, tile) items and keeps a full 32x32x9
// partial in registers: thread = (co pair, ci quad) -> 2 x 4 x 9 accumulators.
__global__ void __launch_bounds__(128)
conv3x3_wgrad_kernel(const float* __restrict__ in, const float* __restrict__ dpre,
                     float* __restrict__ partial, int N, int n_pos, int ntiles) {
    extern __shared__ __align__(16) float smem[];
    constexpr int kDS = kTP + 4;   // padded row: conflict-free LDS.128 over 8 lanes
    float* d_s = smem;             // [32][kDS]
    float* a_s = smem + kCh * kDS; // [32][kWin]
    const int tid = threadIdx.x;
    const int co0 = (tid & 15) * 2, cg = tid >> 4, ci0 = cg * 4;

    float acc[2][4][9];
#pragma unroll
    for (int a = 0; a < 2; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b)
#pragma unroll
            for (int c = 0; c < 9; ++c) acc[a][b][c] = 0.f;
    float bacc0 = 0.f, bacc1 = 0.f;

    const int items = N * ntiles;
    for (int item = blockIdx.x; item < items; item += gridDim.x) {
        const int n = item / ntiles, p0 = (item - n * ntiles) * kTP;
        const float* d_n = dpre + (long long)n * kCh * kPlane;
        const float* a_n = in + (long long)n * kCh * kPlane;
        for (int i = tid; i < kCh * kTP; i += 128) {
            const int c = i / kTP, l = i - c * kTP;
            const int idx = p0 + l;
            d_s[c * kDS + l] = idx < n_pos ? __ldg(d_n + c * kPlane + idx) : 0.f;
        }
        for (int i = tid; i < kCh * kWin; i += 128) {
            const int c = i / kWin, l = i - c * kWin;
            const int idx = p0 + l;
            a_s[i] = idx < kPlane ? __ldg(a_n + c * kPlane + idx) : 0.f;
        }
        __syncthreads();
#pragma unroll 1
        for (int p4 = 0; p4 < kTP; p4 += 4) {
            const float4 dA = *reinterpret_cast<const float4*>(d_s + co0 * kDS + p4);
            const float4 dB = *reinterpret_cast<const float4*>(d_s + (co0 + 1) * kDS + p4);
            const float da[4] = {dA.x, dA.y, dA.z, dA.w};
            const float db[4] = {dB.x, dB.y, dB.z, dB.w};
            if (cg == 0) {
                bacc0 += (da[0] + da[1]) + (da[2] + da[3]);
                bacc1 += (db[0] + db[1]) + (db[2] + db[3]);
            }
#pragma unroll
            for (int c = 0; c < 4; ++c) {
#pragma unroll
                for (int ky = 0; ky < 3; ++ky) {
                    const float* ap = a_s + (ci0 + c) * kWin + p4 + ky * kPW;
                    float a[6];
#pragma unroll
                    for (int t = 0; t < 6; ++t) a[t] = ap[t];
#pragma unroll
                    for (int kx = 0; kx < 3; ++kx)
#pragma unroll
                        for (int pp = 0; pp < 4; ++pp) {
                            acc[0][c][ky * 3 + kx] = fmaf(da[pp], a[pp + kx], acc[0][c][ky * 3 + kx]);
                            acc[1][c][ky * 3 + kx] = fmaf(db[pp], a[pp + kx], acc[1][c][ky * 3 + kx]);
                        }
                }
            }
        }
        __syncthreads();
    }
    float* out = partial + (long long)blockIdx.x * (kCh * kCh * 9 + kCh);
#pragma unroll
    for (int a = 0; a < 2; ++a)
#pragma unroll
        for (int c = 0; c < 4; ++c)
#pragma unroll
            for (int t = 0; t < 9; ++t) out[((co0 + a) * kCh + ci0 + c) * 9 + t] = acc[a][c][t];
    if (cg == 0) {
        out[kCh * kCh * 9 + co0] = bacc0;
        out[kCh * kCh * 9 + co0 + 1] = bacc1;
    }
}

// dw[i] = sum_g partial[g][i] (i < nw), db[i - nw] likewise; fixed order.
__global__ void wgrad_reduce_kernel(const float* __restrict__ partial, int G, int nw, int nb,
                                    float* __restrict__ dw, float* __restrict__ db) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const int row = nw + nb;
    if (i >= row) return;
    float s = 0.f;
    for (int g = 0; g < G; ++g) s += partial[(long long)g * row + i];
    if (i < nw) dw[i] = s; else db[i - nw] = s;
}

// ---------------------------------------------------------------- conv1 (u8, aug fused)
// Stages the augmented, normalised input rows of one output-row tile in shared
// memory: the augmented image never exists in HBM.  T = uint8_t (frames) or float
// (real-valued pixels on the 0..255 scale, already augmented: no shift).
template <typename T>
__device__ __forceinline__ void conv1_stage_input(const T* __restrict__ img, int cin, int sx,
                                                  int sy, int pad, int oy0, float* x_s, int tid,
                                                  int nthreads) {
    const int total = cin * kC1InRows * kImg;
    for (int i = tid; i < total; i += nthreads) {
        const int col = i % kImg;
        const int r = (i / kImg) % kC1InRows;
        const int c = i / (kImg * kC1InRows);
        const int sr = clampi(2 * oy0 + r + sy - pad, 0, kImg - 1);   // replicate pad + shift (rows <- y)
        const int sc = clampi(col + sx - pad, 0, kImg - 1);           // (cols <- x)
        const float px = (float)img[(c * kImg + sr) * kImg + sc];
        x_s[i] = __fsub_rn(__fdiv_rn(px, 255.0f), 0.5f);              // drqv2.py:64
    }
}

template <typename T>
__global__ void __launch_bounds__(288)
conv1_fwd_kernel(const T* __restrict__ obs, const int* __restrict__ shift,
                 const float* __restrict__ w, const float* __restrict__ bias,
                 float* __restrict__ out, int cin, int pad) {
    extern __shared__ __align__(16) float smem[];
    float* x_s = smem;                              // [cin][15][84]
    float* w_s = smem + cin * kC1InRows * kImg;     // [cin*9][32]
    const int tid = threadIdx.x;
    const int n = blockIdx.y, oy0 = blockIdx.x * kC1Rows;
    const int nrows = min(kC1Rows, kPW - oy0);
    const int sx = shift ? shift[2 * n] : pad, sy = shift ? shift[2 * n + 1] : pad;
    const int K = cin * 9;
    for (int i = tid; i < K * kCh; i += blockDim.x) {
        const int co = i / K, k = i - co * K;
        w_s[k * kCh + co] = __ldg(w + i);
    }
    conv1_stage_input(obs + (long long)n * cin * kImg * kImg, cin, sx, sy, pad, oy0, x_s, tid,
                      blockDim.x);
    __syncthreads();
    if (tid >= nrows * kPW) return;
    const int oyl = tid / kPW, ox = tid - oyl * kPW;
    float acc[kCh];
#pragma unroll
    for (int c = 0; c < kCh; ++c) acc[c] = 0.f;
    for (int ci = 0; ci < cin; ++ci) {
#pragma unroll
        for (int ky = 0; ky < 3; ++ky) {
            const float* xp = x_s + (ci * kC1InRows + 2 * oyl + ky) * kImg + 2 * ox;
#pragma unroll
            for (int kx = 0; kx < 3; ++kx) {
                const float v = xp[kx];
                const float4* wp = reinterpret_cast<const float4*>(w_s + ((ci * 3 + ky) * 3 + kx) * kCh);
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                    const float4 w4 = wp[q];
                    acc[4 * q + 0] = fmaf(v, w4.x, acc[4 * q + 0]);
                    acc[4 * q + 1] = fmaf(v, w4.y, acc[4 * q + 1]);
                    acc[4 * q + 2] = fmaf(v, w4.z, acc[4 * q + 2]);
                    acc[4 * q + 3] = fmaf(v, w4.w, acc[4 * q + 3]);
                }
            }
        }
    }
    const int p = (oy0 + oyl) * kPW + ox;
#pragma unroll
    for (int c = 0; c < kCh; ++c)
        out[((long long)n * kCh + c) * kPlane + p] = fmaxf(acc[c] + __ldg(bias + c), 0.f);
}

// thread = (co pair, ci): 2 x 9 accumulators; block walks (image, row tile) items.
template <typename T>
__global__ void __launch_bounds__(256)
conv1_wgrad_kernel(const T* __restrict__ obs, const int* __restrict__ shift,
                   const float* __restrict__ dpre, float* __restrict__ partial, int N, int cin,
                   int pad) {
    extern __shared__ __align__(16) float smem[];
    constexpr int kDS = kC1Rows * kPW + 1;   // 288
    float* x_s = smem;                              // [cin][15][84]
    float* d_s = smem + cin * kC1InRows * kImg;     // [32][kDS]
    const int tid = threadIdx.x;
    const int nwork = 16 * cin;  // active threads
    const int co0 = (tid & 15) * 2, ci = tid >> 4;
    float acc[2][9];
#pragma unroll
    for (int a = 0; a < 2; ++a)
#pragma unroll
        for (int t = 0; t < 9; ++t) acc[a][t] = 0.f;
    float bacc0 = 0.f, bacc1 = 0.f;
    const int items = N * kC1Tiles;
    for (int item = blockIdx.x; item < items; item += gridDim.x) {
        const int n = item / kC1Tiles, oy0 = (item - n * kC1Tiles) * kC1Rows;
        const int nrows = min(kC1Rows, kPW - oy0);
        const int sx = shift ? shift[2 * n] : pad, sy = shift ? shift[2 * n + 1] : pad;
        conv1_stage_input(obs + (long long)n * cin * kImg * kImg, cin, sx, sy, pad, oy0, x_s, tid,
                          blockDim.x);
        const float* d_n = dpre + (long long)n * kCh * kPlane + oy0 * kPW;
        const int npix = nrows * kPW;
        for (int i = tid; i < kCh * (kDS - 1); i += blockDim.x) {
            const int c = i / (kDS - 1), l = i - c * (kDS - 1);
            d_s[c * kDS + l] = l < npix ? __ldg(d_n + c * kPlane + l) : 0.f;
        }
        __syncthreads();
        if (tid < nwork) {
            for (int oyl = 0; oyl < nrows; ++oyl) {
                const float* dA = d_s + co0 * kDS + oyl * kPW;
                const float* dB = dA + kDS;
                const float* xr = x_s + (ci * kC1InRows + 2 * oyl) * kImg;
                for (int ox = 0; ox < kPW; ++ox) {
                    const float a = dA[ox], b = dB[ox];
                    if (ci == 0) { bacc0 += a; bacc1 += b; }
#pragma unroll
                    for (int ky = 0; ky < 3; ++ky)
#pragma unroll
                        for (int kx = 0; kx < 3; ++kx) {
                            const float v = xr[ky * kImg + 2 * ox + kx];
                            acc[0][ky * 3 + kx] = fmaf(a, v, acc[0][ky * 3 + kx]);
                            acc[1][ky * 3 + kx] = fmaf(b, v, acc[1][ky * 3 + kx]);
                        }
                }
            }
        }
        __syncthreads();
    }
    if (tid < nwork) {
        const int nw = kCh * cin * 9;
        float* out = partial + (long long)blockIdx.x * (nw + kCh);
#pragma unroll
        for (int a = 0; a < 2; ++a)
#pragma unroll
            for (int t = 0; t < 9; ++t) out[((co0 + a) * cin + ci) * 9 + t] = acc[a][t];
        if (ci == 0) {
            out[nw + co0] = bacc0;
            out[nw + co0 + 1] = bacc1;
        }
    }
}

// ---------------------------------------------------------------- conv1 data gradient
// dx[n][c][iy][ix] = (1/255) sum_{ky,kx: iy = 2oy+ky, ix = 2ox+kx, oy,ox < 41} sum_co W[co][c][ky][kx] d[co][oy*41+ox]:
// the stride-2 transpose, at most 2 x 2 taps per input pixel (one along an odd coordinate, two along an even one, none
// at row / column 83).  Block = (12 input rows, image): the d rows those rows reach (oy = 6t-1 .. 6t+5) and the weights
// are staged in shared memory.  Threads take pixels column-parity major within a row (42 even columns, then 42 odd
// ones), so most warps take one tap pattern.  Fixed order: taps (ky, kx) ascending, co ascending within a tap.
constexpr int kDgRows = 12;                   // input rows per block (84 = 7 x 12)
constexpr int kDgDRows = kDgRows / 2 + 1;     // 7 d rows

__global__ void __launch_bounds__(256)
conv1_dgrad_kernel(const float* __restrict__ dpre, const float* __restrict__ w, float* __restrict__ dx, int cin) {
    extern __shared__ __align__(16) float smem[];
    float* w_s = smem;                          // [tap][co][16 ci]
    float* d_s = smem + 9 * kCh * 16;           // [co][7][41]
    const int tid = threadIdx.x, n = blockIdx.y, iy0 = blockIdx.x * kDgRows;
    const int oy_lo = iy0 / 2 - 1;
    for (int i = tid; i < 9 * kCh * 16; i += blockDim.x) {
        const int tap = i / (kCh * 16), co = (i / 16) % kCh, ci = i % 16;
        w_s[i] = ci < cin ? __ldg(w + (co * cin + ci) * 9 + tap) : 0.f;
    }
    const float* d_n = dpre + (long long)n * kCh * kPlane;
    for (int i = tid; i < kCh * kDgDRows * kPW; i += blockDim.x) {
        const int co = i / (kDgDRows * kPW), l = i - co * (kDgDRows * kPW);
        const int oy = oy_lo + l / kPW;
        d_s[i] = (oy >= 0 && oy < kPW) ? __ldg(d_n + co * kPlane + oy * kPW + l % kPW) : 0.f;
    }
    __syncthreads();
    for (int q = tid; q < kDgRows * kImg; q += blockDim.x) {
        const int iyl = q / kImg, rem = q - iyl * kImg, px = rem / (kImg / 2), ix = 2 * (rem - px * (kImg / 2)) + px;
        const int iy = iy0 + iyl;
        float acc[16];
#pragma unroll
        for (int c = 0; c < 16; ++c) acc[c] = 0.f;
#pragma unroll
        for (int ky = 0; ky < 3; ++ky) {
            const int oy2 = iy - ky;
            if (oy2 < 0 || (oy2 & 1) || (oy2 >> 1) >= kPW) continue;
            const float* drow = d_s + ((oy2 >> 1) - oy_lo) * kPW;
#pragma unroll
            for (int kx = 0; kx < 3; ++kx) {
                const int ox2 = ix - kx;
                if (ox2 < 0 || (ox2 & 1) || (ox2 >> 1) >= kPW) continue;
                const float* dp = drow + (ox2 >> 1);
                const float* wp = w_s + (ky * 3 + kx) * kCh * 16;
#pragma unroll 4
                for (int co = 0; co < kCh; ++co) {
                    const float dv = dp[co * kDgDRows * kPW];
                    const float4* w4 = reinterpret_cast<const float4*>(wp + co * 16);
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        if (4 * j >= cin) break;
                        const float4 v = w4[j];
                        acc[4 * j + 0] = fmaf(dv, v.x, acc[4 * j + 0]);
                        acc[4 * j + 1] = fmaf(dv, v.y, acc[4 * j + 1]);
                        acc[4 * j + 2] = fmaf(dv, v.z, acc[4 * j + 2]);
                        acc[4 * j + 3] = fmaf(dv, v.w, acc[4 * j + 3]);
                    }
                }
            }
        }
        float* o = dx + (long long)n * cin * kImg * kImg + iy * kImg + ix;
#pragma unroll
        for (int c = 0; c < 16; ++c)
            if (c < cin) o[c * kImg * kImg] = __fdiv_rn(acc[c], 255.0f);
    }
}

// ---------------------------------------------------------------- compact feature gradient -> conv4's wide dpre
// One thread per wide position p < 37*41 of a plane: the ReLU-masked feature gradient inside 35 x 35, +0 at rows
// 35-36 and columns 35-40 (what drq_conv3x3_dgrad_f32 reads at hout = 35 and requires to be zero).
constexpr int kFeatHW = 35;
constexpr int kFeatGradPos = (kFeatHW + 2) * kPW;   // 1517

__global__ void __launch_bounds__(256)
feature_grad_wide_kernel(const float* __restrict__ dfeat, const float* __restrict__ feat,
                         float* __restrict__ dpre, long long total) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const long long plane = i / kFeatGradPos;           // n * 32 + c
    const int p = (int)(i - plane * kFeatGradPos);
    const int y = p / kPW, x = p - y * kPW;
    float v = 0.f;
    if (y < kFeatHW && x < kFeatHW) {
        const long long k = plane * (kFeatHW * kFeatHW) + y * kFeatHW + x;   // c*1225 + y*35 + x of image n
        v = __ldg(feat + k) > 0.f ? __ldg(dfeat + k) : 0.f;
    }
    dpre[plane * kPlane + p] = v;
}

template <typename K>
static int set_smem(K kernel, size_t bytes, const char* what) {
    return ensure_smem(reinterpret_cast<const void*>(kernel), bytes, what);
}

template <typename T>
static int conv1_fwd_launch(const T* obs, const int32_t* shift, const float* w, const float* b, float* out, int N,
                            int cin, int pad, void* stream) {
    DRQ_REQUIRE(obs && w && b && out, "conv1_fwd: null pointer");
    DRQ_REQUIRE(N >= 0 && cin > 0 && cin <= 16 && pad >= 0, "conv1_fwd: bad dims (cin<=16)");
    if (N == 0) return DRQ_OK;
    const size_t smem = (size_t)(cin * kC1InRows * kImg + cin * 9 * kCh) * sizeof(float);
    if (int rc = set_smem(conv1_fwd_kernel<T>, smem, "conv1_fwd")) return rc;
    conv1_fwd_kernel<T><<<dim3(kC1Tiles, N), 288, smem, as_stream(stream)>>>(obs, shift, w, b, out, cin, pad);
    return check_launch("conv1_fwd_kernel");
}

template <typename T>
static int conv1_wgrad_launch(const T* obs, const int32_t* shift, const float* dpre, float* partial, float* dw,
                              float* db, int N, int cin, int pad, void* stream) {
    DRQ_REQUIRE(obs && dpre && partial && dw && db, "conv1_wgrad: null pointer");
    DRQ_REQUIRE(N > 0 && cin > 0 && cin <= 16 && pad >= 0, "conv1_wgrad: bad dims (cin<=16)");
    const size_t smem = (size_t)(cin * kC1InRows * kImg + kCh * (kC1Rows * kPW + 1)) * sizeof(float);
    if (int rc = set_smem(conv1_wgrad_kernel<T>, smem, "conv1_wgrad")) return rc;
    const int items = N * kC1Tiles;
    const int G = items < kWgradBlocks ? items : kWgradBlocks;
    conv1_wgrad_kernel<T><<<G, 256, smem, as_stream(stream)>>>(obs, shift, dpre, partial, N, cin, pad);
    if (int rc = check_launch("conv1_wgrad_kernel")) return rc;
    const int nw = kCh * cin * 9;
    wgrad_reduce_kernel<<<(nw + kCh + 127) / 128, 128, 0, as_stream(stream)>>>(partial, G, nw, kCh, dw, db);
    return check_launch("wgrad_reduce_kernel");
}

}  // namespace drq

using namespace drq;

extern "C" {

int64_t drq_conv_wgrad_ws_floats(int cin) { return (int64_t)kWgradBlocks * (kCh * cin * 9 + kCh); }

int drq_conv1_fwd_f32(const uint8_t* obs, const int32_t* shift, const float* w, const float* b,
                      float* out, int N, int cin, int pad, void* stream) {
    return conv1_fwd_launch(obs, shift, w, b, out, N, cin, pad, stream);
}

int drq_conv1_fwd_f32_from_f32(const float* obs, const float* w, const float* b, float* out, int N, int cin,
                               void* stream) {
    return conv1_fwd_launch(obs, nullptr, w, b, out, N, cin, 0, stream);
}

int drq_conv1_wgrad_f32(const uint8_t* obs, const int32_t* shift, const float* dpre, float* partial,
                        float* dw, float* db, int N, int cin, int pad, void* stream) {
    return conv1_wgrad_launch(obs, shift, dpre, partial, dw, db, N, cin, pad, stream);
}

int drq_conv1_wgrad_f32_from_f32(const float* obs, const float* dpre, float* partial, float* dw, float* db, int N,
                                 int cin, void* stream) {
    return conv1_wgrad_launch(obs, nullptr, dpre, partial, dw, db, N, cin, 0, stream);
}

int drq_conv1_dgrad_f32(const float* dpre, const float* w, float* dx, int N, int cin, void* stream) {
    DRQ_REQUIRE(dpre && w && dx, "conv1_dgrad: null pointer");
    DRQ_REQUIRE(N >= 0 && cin > 0 && cin <= 16, "conv1_dgrad: bad dims (cin<=16)");
    if (N == 0) return DRQ_OK;
    const size_t smem = (size_t)(9 * kCh * 16 + kCh * kDgDRows * kPW) * sizeof(float);
    if (int rc = set_smem(conv1_dgrad_kernel, smem, "conv1_dgrad")) return rc;
    conv1_dgrad_kernel<<<dim3(kImg / kDgRows, N), 256, smem, as_stream(stream)>>>(dpre, w, dx, cin);
    return check_launch("conv1_dgrad_kernel");
}

int drq_conv3x3_fwd_f32(const float* in, const float* w, const float* b, float* out, int N, int hout,
                        int compact_out, void* stream) {
    DRQ_REQUIRE(in && w && b && out, "conv3x3_fwd: null pointer");
    DRQ_REQUIRE(N >= 0 && hout > 0 && hout <= kPW - 2, "conv3x3_fwd: bad dims");
    if (N == 0) return DRQ_OK;
    const size_t smem = (size_t)(kCh * kWin + 9 * kCh * kCh) * sizeof(float);
    if (int rc = set_smem(conv3x3_wide_kernel<false>, smem, "conv3x3_fwd")) return rc;
    const int n_pos = hout * kPW;
    conv3x3_wide_kernel<false><<<dim3((n_pos + kTP - 1) / kTP, N), 128, smem, as_stream(stream)>>>(
        in, w, b, nullptr, out, n_pos, hout, compact_out);
    return check_launch("conv3x3_fwd_kernel");
}

int drq_conv3x3_dgrad_f32(const float* dout, const float* w, const float* act_in, float* din, int N,
                          int hout, void* stream) {
    DRQ_REQUIRE(dout && w && act_in && din, "conv3x3_dgrad: null pointer");
    DRQ_REQUIRE(N >= 0 && hout > 0 && hout <= kPW - 2, "conv3x3_dgrad: bad dims");
    if (N == 0) return DRQ_OK;
    const size_t smem = (size_t)(kCh * kWin + 9 * kCh * kCh) * sizeof(float);
    if (int rc = set_smem(conv3x3_wide_kernel<true>, smem, "conv3x3_dgrad")) return rc;
    const int hin = hout + 2;
    const int n_pos = hin * kPW;
    conv3x3_wide_kernel<true><<<dim3((n_pos + kTP - 1) / kTP, N), 128, smem, as_stream(stream)>>>(
        dout, w, nullptr, act_in, din, n_pos, hin, 0);
    return check_launch("conv3x3_dgrad_kernel");
}

int drq_conv3x3_wgrad_f32(const float* in, const float* dpre, float* partial, float* dw, float* db,
                          int N, int hout, void* stream) {
    DRQ_REQUIRE(in && dpre && partial && dw && db, "conv3x3_wgrad: null pointer");
    DRQ_REQUIRE(N > 0 && hout > 0 && hout <= kPW - 2, "conv3x3_wgrad: bad dims");
    const size_t smem = (size_t)(kCh * (kTP + 4) + kCh * kWin) * sizeof(float);
    if (int rc = set_smem(conv3x3_wgrad_kernel, smem, "conv3x3_wgrad")) return rc;
    const int n_pos = hout * kPW;
    const int ntiles = (n_pos + kTP - 1) / kTP;
    const int items = N * ntiles;
    const int G = items < kWgradBlocks ? items : kWgradBlocks;
    conv3x3_wgrad_kernel<<<G, 128, smem, as_stream(stream)>>>(in, dpre, partial, N, n_pos, ntiles);
    if (int rc = check_launch("conv3x3_wgrad_kernel")) return rc;
    const int nw = kCh * kCh * 9;
    wgrad_reduce_kernel<<<(nw + kCh + 127) / 128, 128, 0, as_stream(stream)>>>(partial, G, nw, kCh, dw, db);
    return check_launch("wgrad_reduce_kernel");
}

int drq_feature_grad_wide_f32(const float* dfeat, const float* feat, float* dpre, int N, void* stream) {
    DRQ_REQUIRE(dfeat && feat && dpre, "feature_grad_wide: null pointer");
    DRQ_REQUIRE(N >= 0, "feature_grad_wide: bad dims");
    if (N == 0) return DRQ_OK;
    const long long total = (long long)N * kCh * kFeatGradPos;
    feature_grad_wide_kernel<<<(unsigned)((total + 255) / 256), 256, 0, as_stream(stream)>>>(dfeat, feat, dpre, total);
    return check_launch("feature_grad_wide_kernel");
}

}  // extern "C"

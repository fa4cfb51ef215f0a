// fp32 (parity-mode) dense kernels: strided/batched/split-K SGEMM with fused epilogues,
// column sums, and the deterministic split-K reduction.
// Reference ops: nn.Linear forward/backward in Actor/Critic (drqv2.py:70-121).
#include "common.cuh"

namespace drq {

constexpr int BM = 64, BN = 64, BK = 16;
constexpr int kPad = 4;

struct GemmArgs {
    const float* A; long long sa_m, sa_k;
    const float* B; long long sb_k, sb_n;
    float* C; long long ldc;
    const float* bias;
    const float* mask; long long ldmask;
    int M, N, K;
    int epilogue, accumulate;
    long long bs_a, bs_b, bs_c, bs_bias, bs_mask;
    int splitk, k_chunk;
};

// compact feature index k = c*1225 + y*35 + x  ->  wide-plane offset c*kPlane + y*41 + x
__device__ __forceinline__ long long compact_to_wide(int k) {
    const int c = k / 1225, r = k - c * 1225;
    const int y = r / 35, x = r - y * 35;
    return (long long)c * kPlane + y * kPW + x;
}

__global__ void __launch_bounds__(256) gemm_f32_kernel(GemmArgs g) {
    __shared__ __align__(16) float As[BK][BM + kPad];
    __shared__ __align__(16) float Bs[BK][BN + kPad];
    const int tid = threadIdx.x;
    const int tx = tid & 15, ty = tid >> 4;
    const int m0 = blockIdx.y * BM, n0 = blockIdx.x * BN;
    const int z = blockIdx.z;

    const float* A = g.A;
    const float* B = g.B;
    float* C = g.C;
    const float* bias = g.bias;
    const float* mask = g.mask;
    int k_begin = 0, k_end = g.K;
    if (g.splitk > 1) {
        k_begin = z * g.k_chunk;
        k_end = min(g.K, k_begin + g.k_chunk);
        C += (long long)z * g.bs_c;
    } else {
        A += (long long)z * g.bs_a;
        B += (long long)z * g.bs_b;
        C += (long long)z * g.bs_c;
        if (bias) bias += (long long)z * g.bs_bias;
        if (mask) mask += (long long)z * g.bs_mask;
    }
    // thread -> tile element mapping chosen so that the unit-stride axis is the fast one
    const bool a_kfast = (g.sa_k == 1);
    const bool b_kfast = (g.sb_k == 1);

    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

    for (int k0 = k_begin; k0 < k_end; k0 += BK) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int e = tid + 256 * i;
            int m, k;
            if (a_kfast) { k = e & (BK - 1); m = e >> 4; } else { m = e & (BM - 1); k = e >> 6; }
            const int gm = m0 + m, gk = k0 + k;
            As[k][m] = (gm < g.M && gk < k_end) ? __ldg(A + gm * g.sa_m + gk * g.sa_k) : 0.f;
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int e = tid + 256 * i;
            int n, k;
            if (b_kfast) { k = e & (BK - 1); n = e >> 4; } else { n = e & (BN - 1); k = e >> 6; }
            const int gn = n0 + n, gk = k0 + k;
            Bs[k][n] = (gn < g.N && gk < k_end) ? __ldg(B + gk * g.sb_k + gn * g.sb_n) : 0.f;
        }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < BK; ++k) {
            const float4 a4 = *reinterpret_cast<const float4*>(&As[k][ty * 4]);
            const float4 b4 = *reinterpret_cast<const float4*>(&Bs[k][tx * 4]);
            const float a[4] = {a4.x, a4.y, a4.z, a4.w};
            const float b[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
        }
        __syncthreads();
    }

#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int m = m0 + ty * 4 + i;
        if (m >= g.M) continue;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int n = n0 + tx * 4 + j;
            if (n >= g.N) continue;
            float v = acc[i][j];
            if (g.splitk > 1) {
                C[m * g.ldc + n] = v;
                continue;
            }
            if (bias) v += __ldg(bias + n);
            long long o = m * g.ldc + n;
            if (g.epilogue == DRQ_EPI_RELU) {
                v = fmaxf(v, 0.f);
            } else if (g.epilogue == DRQ_EPI_MASK) {
                v = (__ldg(mask + m * g.ldmask + n) > 0.f) ? v : 0.f;
            } else if (g.epilogue == DRQ_EPI_MASK_WIDE) {
                v = (__ldg(mask + m * g.ldmask + n) > 0.f) ? v : 0.f;
                o = m * g.ldc + compact_to_wide(n);
            }
            if (g.accumulate) v += C[o];
            C[o] = v;
        }
    }
}

// out[z][n] = sum_m X[z][m][n]; block = 32 columns x 8 row lanes, fixed-order tree.
__global__ void __launch_bounds__(256)
colsum_kernel(const float* __restrict__ X, long long ld, float* __restrict__ out, int M, int N,
              long long bs_x, long long bs_out) {
    __shared__ float red[8][33];
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int n = blockIdx.x * 32 + tx;
    const float* Xz = X + blockIdx.y * bs_x;
    float s = 0.f;
    if (n < N)
        for (int m = ty; m < M; m += 8) s += Xz[m * ld + n];
    red[ty][tx] = s;
    __syncthreads();
    if (ty == 0 && n < N) {
        float t = red[0][tx];
#pragma unroll
        for (int r = 1; r < 8; ++r) t += red[r][tx];
        out[blockIdx.y * bs_out + n] = t;
    }
}

}  // namespace drq

using namespace drq;

extern "C" {

int drq_gemm_f32(const float* A, int64_t sa_m, int64_t sa_k, const float* B, int64_t sb_k,
                 int64_t sb_n, float* C, int64_t ldc, const float* bias, const float* mask,
                 int64_t ldmask, int M, int N, int K, int epilogue, int accumulate, int batch,
                 int64_t bs_a, int64_t bs_b, int64_t bs_c, int64_t bs_bias, int64_t bs_mask,
                 int splitk, void* stream) {
    DRQ_REQUIRE(A && B && C, "gemm: null pointer");
    DRQ_REQUIRE(M >= 0 && N > 0 && K > 0, "gemm: bad dims M=%d N=%d K=%d", M, N, K);
    DRQ_REQUIRE(batch >= 1 && splitk >= 1 && !(batch > 1 && splitk > 1), "gemm: batch/splitk");
    DRQ_REQUIRE(epilogue >= DRQ_EPI_NONE && epilogue <= DRQ_EPI_MASK_WIDE, "gemm: bad epilogue");
    DRQ_REQUIRE(!(epilogue >= DRQ_EPI_MASK && !mask), "gemm: mask epilogue without mask");
    DRQ_REQUIRE(!(epilogue == DRQ_EPI_MASK_WIDE && N != DRQ_REPR_DIM), "gemm: MASK_WIDE needs N=39200");
    if (M == 0) return DRQ_OK;
    GemmArgs g;
    g.A = A; g.sa_m = sa_m; g.sa_k = sa_k;
    g.B = B; g.sb_k = sb_k; g.sb_n = sb_n;
    g.C = C; g.ldc = ldc; g.bias = bias; g.mask = mask; g.ldmask = ldmask;
    g.M = M; g.N = N; g.K = K; g.epilogue = epilogue; g.accumulate = accumulate;
    g.bs_a = bs_a; g.bs_b = bs_b; g.bs_c = bs_c; g.bs_bias = bs_bias; g.bs_mask = bs_mask;
    g.splitk = splitk;
    g.k_chunk = K;
    if (splitk > 1) {
        int chunk = (K + splitk - 1) / splitk;
        chunk = (chunk + BK - 1) / BK * BK;
        g.k_chunk = chunk;
        DRQ_REQUIRE((long long)chunk * (splitk - 1) < K, "gemm: splitk %d leaves empty chunks for K=%d", splitk, K);
    }
    dim3 grid((N + BN - 1) / BN, (M + BM - 1) / BM, splitk > 1 ? splitk : batch);
    gemm_f32_kernel<<<grid, 256, 0, as_stream(stream)>>>(g);
    return check_launch("gemm_f32_kernel");
}

int drq_colsum_f32(const float* X, int64_t ld, float* out, int M, int N, int batch, int64_t bs_x,
                   int64_t bs_out, void* stream) {
    DRQ_REQUIRE(X && out && M > 0 && N > 0 && batch > 0, "colsum: bad args");
    colsum_kernel<<<dim3((N + 31) / 32, batch), 256, 0, as_stream(stream)>>>(X, ld, out, M, N, bs_x, bs_out);
    return check_launch("colsum_kernel");
}

}  // extern "C"

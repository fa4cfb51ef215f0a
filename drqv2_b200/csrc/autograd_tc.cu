// Layout conversions between the module API's fp32 tensors (reference layouts, drqv2.py:66) and the tensor-core
// kernels' bf16 operands, for Encoder / Actor / Critic built with differentiable="bf16" (drqv2_b200/_bf16.py).
#include <cuda_bf16.h>

#include "common.cuh"

namespace drq {

constexpr int kUnits = DRQ_REPR_DIM / 8;      // 8-channel units of a feature row: (c/8)*1225 + yx
constexpr int kYX = 35 * 35;

// unit u of row r -> out[r][(cb*8 + j)*1225 + yx] for j < 8 (u = cb*1225 + yx).  One thread per (row, unit):
// consecutive threads write consecutive pixels of each channel.
__global__ void __launch_bounds__(256)
features_to_ref_kernel(const void* __restrict__ src, int src_tb, float* __restrict__ out) {
    const int u = blockIdx.x * blockDim.x + threadIdx.x;
    if (u >= kUnits) return;
    const long long r = blockIdx.y;
    float v[8];
    if (src_tb) {
        const __nv_bfloat16* s = reinterpret_cast<const __nv_bfloat16*>(src) +
                                 (((r >> 7) * kUnits + u) * DRQ_TB_ACT + (r & 127)) * 8;
        const uint4 w = __ldg(reinterpret_cast<const uint4*>(s));
        const uint32_t ws[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            v[2 * j] = __uint_as_float(ws[j] << 16);
            v[2 * j + 1] = __uint_as_float(ws[j] & 0xFFFF0000u);
        }
    } else {
        const float4* s = reinterpret_cast<const float4*>(reinterpret_cast<const float*>(src) + r * DRQ_REPR_DIM + u * 8);
        const float4 a = __ldg(s), b = __ldg(s + 1);
        v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
    }
    const int cb = u / kYX, yx = u - cb * kYX;
    float* o = out + r * DRQ_REPR_DIM + (long long)(cb * 8) * kYX + yx;
#pragma unroll
    for (int j = 0; j < 8; ++j) o[j * kYX] = v[j];
}

// One thread per (channel block, pixel row) of the N-image WB buffer: conv4's masked gradient at the 35 x 35 pixels of
// each image, +0 everywhere else (guard rows, columns and rows past 34, slack).
__global__ void __launch_bounds__(256)
feature_grad_wide_bf16_kernel(const float* __restrict__ dfeat, const float* __restrict__ feat,
                              __nv_bfloat16* __restrict__ dpre, long long rows_per_block, long long total) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const int cb = (int)(i / rows_per_block);
    const long long row = i - cb * rows_per_block;
    const long long n = row / DRQ_PLB;
    const int p = (int)(row - n * DRQ_PLB) - DRQ_GUARD;
    const int y = p >= 0 ? p / DRQ_PW : 0, x = p >= 0 ? p - y * DRQ_PW : 0;
    const bool inside = row < rows_per_block - DRQ_WB_SLACK && p >= 0 && y < 35 && x < 35;
    uint32_t pk[4] = {0, 0, 0, 0};
    if (inside) {
        const long long k = n * DRQ_REPR_DIM + (long long)(cb * 8) * kYX + y * 35 + x;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const long long k0 = k + (long long)(2 * j) * kYX, k1 = k0 + kYX;
            const float lo = __ldg(feat + k0) > 0.f ? __ldg(dfeat + k0) : 0.f;
            const float hi = __ldg(feat + k1) > 0.f ? __ldg(dfeat + k1) : 0.f;
            const __nv_bfloat162 t = __floats2bfloat162_rn(lo, hi);
            pk[j] = *reinterpret_cast<const uint32_t*>(&t);
        }
    }
    *reinterpret_cast<uint4*>(dpre + i * 8) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
}

// out[r][c] = 0 + planes[0][r][c] + planes[1][r][c] + ... in plane order - the order drq_actor_sample_bwd and
// drq_ln_tanh_bwd sum the same planes in.
__global__ void __launch_bounds__(256)
plane_sum_kernel(const float* __restrict__ planes, long long ld, long long plane_stride, int n_planes,
                 float* __restrict__ out, long long ld_out, int rows, int cols) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (long long)rows * cols) return;
    const long long r = i / cols;
    const int c = (int)(i - r * cols);
    const float* p = planes + r * ld + c;
    float t = 0.f;
    for (int s = 0; s < n_planes; ++s) t += __ldg(p + s * plane_stride);
    out[r * ld_out + c] = t;
}

}  // namespace drq

using namespace drq;

extern "C" {

int drq_features_to_ref(const void* src, int src_tb, float* out, int rows, void* stream) {
    DRQ_REQUIRE(src && out, "features_to_ref: null pointer");
    DRQ_REQUIRE(rows > 0 && rows <= DRQ_FEATURE_MAX_ROWS, "features_to_ref: 1 <= rows <= %d", DRQ_FEATURE_MAX_ROWS);
    DRQ_REQUIRE(((uintptr_t)src % 16) == 0, "features_to_ref: source must be 16-byte aligned");
    features_to_ref_kernel<<<dim3((kUnits + 255) / 256, rows), 256, 0, as_stream(stream)>>>(src, src_tb, out);
    return check_launch("features_to_ref_kernel");
}

int drq_feature_grad_wide_bf16(const float* dfeat, const float* feat, uint16_t* dpre, int N, void* stream) {
    DRQ_REQUIRE(dfeat && feat && dpre, "feature_grad_wide_bf16: null pointer");
    DRQ_REQUIRE(N > 0, "feature_grad_wide_bf16: bad dims");
    DRQ_REQUIRE(((uintptr_t)dpre % 16) == 0, "feature_grad_wide_bf16: dpre must be 16-byte aligned");
    const long long rows = (long long)N * DRQ_PLB + DRQ_WB_SLACK;
    const long long total = 4 * rows;
    feature_grad_wide_bf16_kernel<<<(unsigned)((total + 255) / 256), 256, 0, as_stream(stream)>>>(
        dfeat, feat, reinterpret_cast<__nv_bfloat16*>(dpre), rows, total);
    return check_launch("feature_grad_wide_bf16_kernel");
}

int drq_plane_sum_f32(const float* planes, int64_t ld, int64_t plane_stride, int n_planes, float* out, int64_t ld_out,
                      int rows, int cols, void* stream) {
    DRQ_REQUIRE(planes && out && n_planes >= 1 && rows > 0 && cols > 0, "plane_sum: bad args");
    const long long total = (long long)rows * cols;
    plane_sum_kernel<<<(unsigned)((total + 255) / 256), 256, 0, as_stream(stream)>>>(planes, ld, plane_stride, n_planes,
                                                                                   out, ld_out, rows, cols);
    return check_launch("plane_sum_kernel");
}

}  // extern "C"

// Shared helpers for the libdrqv2_b200 kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/drqv2_b200.h"

namespace drq {

// Records a printf-style message retrievable through drq_last_error().
void set_error(const char* fmt, ...);

// Maps cudaGetLastError() after a launch to a DRQ status (and records text).
int check_launch(const char* what);

// Opt a kernel in to `bytes` of dynamic shared memory (> 48 KB needs it); remembered per
// kernel so that repeated calls (and calls during graph capture) touch no CUDA API.
int ensure_smem(const void* kernel, size_t bytes, const char* what);

inline cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }

// cuTensorMapEncodeTiled through the runtime's driver entry point (no -lcuda), or null; cast to the driver's signature by
// the callers that include <cuda.h> (conv4x1_tc.cu, conv1_tc.cu)
void* tensor_map_encoder();

// SMs the persistent kernels size their grids for (drq_set_sm_limit): all of them, or fewer when a concurrent
// collective's CTAs need SMs of their own (a persistent kernel never yields an SM once its CTAs are resident).
extern int g_sm_limit;
inline int sm_budget() { return g_sm_limit; }

constexpr int kImg = DRQ_IMG;
constexpr int kPW = DRQ_PW;
constexpr int kPlane = DRQ_PLANE;
constexpr int kCh = DRQ_CONV_CH;

__device__ __forceinline__ int clampi(int v, int lo, int hi) { return v < lo ? lo : (v > hi ? hi : v); }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// Philox4x32-10 (Salmon et al. 2011), counter-based: same (key, ctr) -> same 4 words.
struct Philox {
    static constexpr uint32_t kM0 = 0xD2511F53u, kM1 = 0xCD9E8D57u;
    static constexpr uint32_t kW0 = 0x9E3779B9u, kW1 = 0xBB67AE85u;
    __host__ __device__ static inline void round(uint32_t (&c)[4], uint32_t k0, uint32_t k1) {
        uint64_t p0 = (uint64_t)kM0 * c[0], p1 = (uint64_t)kM1 * c[2];
        uint32_t h0 = (uint32_t)(p0 >> 32), l0 = (uint32_t)p0;
        uint32_t h1 = (uint32_t)(p1 >> 32), l1 = (uint32_t)p1;
        uint32_t n0 = h1 ^ c[1] ^ k0, n2 = h0 ^ c[3] ^ k1;
        c[0] = n0; c[1] = l1; c[2] = n2; c[3] = l0;
    }
    __host__ __device__ static inline void gen(uint64_t seed, uint64_t stream, uint64_t index,
                                               uint32_t (&out)[4]) {
        uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
        uint32_t c[4] = {(uint32_t)index, (uint32_t)(index >> 32), (uint32_t)stream,
                         (uint32_t)(stream >> 32)};
#pragma unroll
        for (int i = 0; i < 10; ++i) {
            round(c, k0, k1);
            k0 += kW0; k1 += kW1;
        }
        out[0] = c[0]; out[1] = c[1]; out[2] = c[2]; out[3] = c[3];
    }
};

}  // namespace drq

#define DRQ_REQUIRE(cond, ...)            \
    do {                                  \
        if (!(cond)) {                    \
            drq::set_error(__VA_ARGS__);  \
            return DRQ_ERR_INVALID;       \
        }                                 \
    } while (0)

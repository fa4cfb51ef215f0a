// Head-side small kernels: trunk tail (split-K reduce + bias + LayerNorm + tanh) and its
// backward, the clipped TruncatedNormal sample, TD target / critic loss, actor loss.
// Reference: drqv2.py:74-75,88-92,177-228; utils.py:105-126.
#include <cuda_bf16.h>

#include "common.cuh"

namespace drq {

constexpr int kMaxFPerLane = 8;  // F <= 256

// tile-blocked (TB) bf16 activation layout of the tensor-core heads (include/drqv2_b200.h):
// element (row, f) of X_tb[row / 128][f / 8][row % 128][f % 8]; `units` = padded features / 8
__device__ __forceinline__ long long fb_index(int f, long long row, long long units) {
    return (((row >> 7) * units + (f >> 3)) * DRQ_TB_ACT + (row & 127)) * 8 + (f & 7);
}

// Trunk tail for up to DRQ_LN_MAX_JOBS (network, row range) pairs in one launch: blockIdx.y = job,
// one warp per row.  The split-K partial sums are added in a fixed order (8 loads in flight).
struct LnJobs { drq_ln_job j[DRQ_LN_MAX_JOBS]; };

template <int NF>   // features per lane: F <= 32 * NF
__global__ void __launch_bounds__(128)
ln_tanh_fwd_kernel(const LnJobs jobs, int B, int F, float eps) {
    // One block per (row, job): the four warps sum interleaved quarters of the split-K planes (all loads of a
    // warp in flight at once), the partial rows are combined in fixed order, warp 0 normalises.
    __shared__ float part[4][32 * NF];
    const drq_ln_job& jb = jobs.j[blockIdx.y];
    const int row = blockIdx.x;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    constexpr int MAXP = 16;                           // planes per warp held in flight (S <= 64); more fall back to a loop
#pragma unroll
    for (int i = 0; i < NF; ++i) {
        const int f = lane + 32 * i;
        float v = 0.f;
        if (f < F) {
            const float* pp = jb.partial + (long long)row * jb.ld_partial + f;
            float t[MAXP];
#pragma unroll
            for (int k = 0; k < MAXP; ++k) {
                const int s = w + 4 * k;
                t[k] = s < jb.S ? pp[s * jb.split_stride] : 0.f;
            }
#pragma unroll
            for (int k = 0; k < MAXP; ++k) v += t[k];
            for (int s = w + 4 * MAXP; s < jb.S; s += 4) v += pp[s * jb.split_stride];
        }
        part[w][f] = v;
    }
    __syncthreads();
    if (w != 0) return;
    float z[NF];
    float sum = 0.f;
#pragma unroll
    for (int i = 0; i < NF; ++i) {
        const int f = lane + 32 * i;
        float v = 0.f;
        if (f < F) v = ((part[0][f] + part[1][f]) + (part[2][f] + part[3][f])) + jb.bias[f];
        z[i] = v;
        sum += v;
    }
    const float mean = warp_sum(sum) / (float)F;
    float sq = 0.f;
#pragma unroll
    for (int i = 0; i < NF; ++i) {
        const int f = lane + 32 * i;
        const float d = (f < F) ? z[i] - mean : 0.f;
        sq += d * d;
    }
    const float var = warp_sum(sq) / (float)F;   // biased, as nn.LayerNorm
    const float rstd = 1.0f / sqrtf(var + eps);
    __nv_bfloat16* h_bf = reinterpret_cast<__nv_bfloat16*>(jb.h_bf16);
#pragma unroll
    for (int i = 0; i < NF; ++i) {
        const int f = lane + 32 * i;
        if (f < F) {
            const float xh = (z[i] - mean) * rstd;
            const float y = xh * jb.gamma[f] + jb.beta[f];
            const float hv = tanhf(y);
            jb.h_out[(long long)row * jb.ld_h + f] = hv;
            if (h_bf) h_bf[fb_index(f, jb.row0_bf16 + row, jb.units_bf16)] = __float2bfloat16_rn(hv);
            if (jb.xhat) jb.xhat[(long long)row * F + f] = xh;
        }
    }
    if (jb.rstd && lane == 0) jb.rstd[row] = rstd;
    if (jb.tail && h_bf)
        for (int t = lane; t < jb.n_tail; t += 32)
            h_bf[fb_index(F + t, jb.row0_bf16 + row, jb.units_bf16)] = __float2bfloat16_rn(jb.tail[(long long)row * jb.ld_tail + t]);
}

// per row: dy = dh*(1-h^2); dxhat = dy*gamma; dz = rstd*(dxhat - mean(dxhat) - xhat*mean(dxhat*xhat)).
// dy and dy*xhat are staged in dz_tmp-style buffers for the column reduction below.
__global__ void __launch_bounds__(128)
ln_tanh_bwd_row_kernel(const float* __restrict__ dh, long long ld_dh, const float* __restrict__ h,
                       long long ld_h, const float* __restrict__ xhat,
                       const float* __restrict__ rstd, const float* __restrict__ gamma,
                       float* __restrict__ dz, float* __restrict__ dy_out, __nv_bfloat16* __restrict__ dz_bf,
                       long long rpad_zb, int B, int F, int n_planes, long long plane_stride) {
    const int row = blockIdx.x * 4 + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (row >= B) return;
    float dxh[kMaxFPerLane], xh[kMaxFPerLane];
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int i = 0; i < kMaxFPerLane; ++i) {
        const int f = lane + 32 * i;
        dxh[i] = 0.f; xh[i] = 0.f;
        if (f < F) {
            const float hv = h[(long long)row * ld_h + f];
            // dh = sum of the split-K / per-head partial planes (loads of 8 planes in flight, fixed order)
            float dhv = 0.f;
            const float* dp = dh + (long long)row * ld_dh + f;
            for (int p0 = 0; p0 < n_planes; p0 += 8) {
                float t[8];
#pragma unroll
                for (int k = 0; k < 8; ++k) t[k] = p0 + k < n_planes ? dp[(p0 + k) * plane_stride] : 0.f;
#pragma unroll
                for (int k = 0; k < 8; ++k) dhv += t[k];
            }
            const float dy = dhv * (1.0f - hv * hv);
            dy_out[(long long)row * F + f] = dy;
            xh[i] = xhat[(long long)row * F + f];
            dxh[i] = dy * gamma[f];
            s1 += dxh[i];
            s2 += dxh[i] * xh[i];
        }
    }
    const float m1 = warp_sum(s1) / (float)F, m2 = warp_sum(s2) / (float)F;
    const float r = rstd[row];
#pragma unroll
    for (int i = 0; i < kMaxFPerLane; ++i) {
        const int f = lane + 32 * i;
        if (f < F) {
            const float g = r * (dxh[i] - m1 - xh[i] * m2);
            dz[(long long)row * F + f] = g;
            if (dz_bf) dz_bf[fb_index(f, row, rpad_zb)] = __float2bfloat16_rn(g);
        }
    }
}

// one block per feature: dgamma[f] = sum_b dy*xhat, dbeta[f] = sum_b dy (fixed-order tree)
__global__ void __launch_bounds__(256)
ln_param_grad_kernel(const float* __restrict__ dy, const float* __restrict__ xhat,
                     float* __restrict__ dgamma, float* __restrict__ dbeta, int B, int F) {
    __shared__ float sg[256], sb[256];
    const int f = blockIdx.x;
    float g = 0.f, b = 0.f;
    for (int r = threadIdx.x; r < B; r += 256) {
        const float d = dy[(long long)r * F + f];
        g += d * xhat[(long long)r * F + f];
        b += d;
    }
    sg[threadIdx.x] = g; sb[threadIdx.x] = b;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if (threadIdx.x < o) { sg[threadIdx.x] += sg[threadIdx.x + o]; sb[threadIdx.x] += sb[threadIdx.x + o]; }
        __syncthreads();
    }
    if (threadIdx.x == 0) { dgamma[f] = sg[0]; dbeta[f] = sb[0]; }
}

// block-wide fixed-order sum of per-thread values (blockDim = 256)
__device__ __forceinline__ float block_sum_256(float v, float* sh) {
    sh[threadIdx.x] = v;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if (threadIdx.x < o) sh[threadIdx.x] += sh[threadIdx.x + o];
        __syncthreads();
    }
    const float r = sh[0];
    __syncthreads();
    return r;
}

// single block; thread t handles rows t, t+256, ...
__global__ void __launch_bounds__(256)
actor_sample_kernel(const float* __restrict__ mu_pre, const float* __restrict__ eps,
                    const float* __restrict__ std_dev, float clip, float* __restrict__ action_out,
                    long long ld_a, float* __restrict__ mu_out, float* __restrict__ metrics, int B, int A) {
    __shared__ float sh[256];
    const float std = std_dev ? *std_dev : 0.f;
    const float lo = -1.0f + 1e-6f, hi = 1.0f - 1e-6f;  // utils.py:113 (python: -1.0 + 1e-6 -> fp32)
    const float log_std = logf(std);
    float lp_sum = 0.f;
    for (int b = blockIdx.x * blockDim.x + threadIdx.x; b < B; b += gridDim.x * blockDim.x) {
        float lp = 0.f;
        for (int j = 0; j < A; ++j) {
            const float mu = tanhf(mu_pre[(long long)b * A + j]);   // drqv2.py:89
            float a = mu;
            if (eps) {
                float e = __fmul_rn(eps[(long long)b * A + j], std);      // utils.py:120
                if (clip > 0.f) e = fminf(fmaxf(e, -clip), clip);         // utils.py:121-122
                const float x = __fadd_rn(mu, e);                          // utils.py:123
                a = fminf(fmaxf(x, lo), hi);                               // utils.py:113-116 (value)
                // Normal.log_prob(a): -((a-mu)^2)/(2 var) - log(std) - log(sqrt(2 pi))
                const float d = a - mu;
                lp += -(d * d) / (2.0f * std * std) - log_std - 0.9189385332046727f;
            }
            action_out[(long long)b * ld_a + j] = a;
            if (mu_out) mu_out[(long long)b * A + j] = mu;
        }
        lp_sum += lp;
    }
    if (metrics && gridDim.x == 1) {
        const float t = block_sum_256(lp_sum, sh);
        if (threadIdx.x == 0) {
            metrics[0] = t / (float)B;                                         // actor_logprob
            metrics[1] = (float)A * (0.5f + 0.9189385332046727f + log_std);    // actor_ent
        }
    }
}

// Policy head (drqv2.py:81,88-92): mu_pre[m][:] = p2[m][:] . bf16(W4)^T + b4 for all M rows of a TB activation - the
// Linear(hidden, A) as dot products on the CUDA cores (A <= 128 outputs: a tensor-core tile would be > 75 % padding at
// A <= 32 and run on M / 128 CTAs) - and, by the thread that holds each mu_pre value, the TruncatedNormal samples of up
// to DRQ_POLICY_MAX_JOBS row ranges (utils.py:112-126).  Block = 8 rows x one group of at most 32 actions: blockIdx.y
// picks the group, ceil(A / gridDim.y) actions each (A <= 32: one group, all of A), and a block stages only its group's
// rows of W4.  One warp per row, lanes split the row's 16-byte units (32 rows per block left the launch on M / 32 = 16
// SMs: 12.6 us as a graph node).  The weights are rounded to bf16 when they are staged, i.e. the arithmetic is that of
// the bf16 GEMM this replaces (bf16 x bf16 products, fp32 sums).  A job with metrics needs the batch mean of the
// log-probabilities: every block leaves its partial sum in scratch[1 + blockIdx.y * gridDim.x + blockIdx.x], the block
// that finishes last (ticket in scratch[0]) adds them in that order.
struct PolicyJobs { drq_policy_sample j[DRQ_POLICY_MAX_JOBS]; int n; int metrics_job; };
constexpr int kPolicyRows = 8;
constexpr int kPolicyGroup = 32;          // actions per block at most

__global__ void __launch_bounds__(256)
policy_head_fwd_kernel(const __nv_bfloat16* __restrict__ p2, long long units, const float* __restrict__ w4,
                       const float* __restrict__ b4, float* __restrict__ mu_pre, int M, int H, int A, const PolicyJobs jobs,
                       const float* __restrict__ std_dev, float clip, unsigned int* __restrict__ scratch) {
    extern __shared__ float w_s[];                       // [na][H]: this block's group of W4 rows
    __shared__ float sh[256];
    __shared__ int s_last;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int m = blockIdx.x * kPolicyRows + warp;
    const int nu = H / 8;
    const int ga = (A + gridDim.y - 1) / gridDim.y;
    const int a_lo = blockIdx.y * ga;                    // the group: actions a_lo .. a_lo + na - 1
    const int na = min(ga, A - a_lo);
    const __nv_bfloat16* x = p2 + fb_index(0, m < M ? m : 0, units);
    // the lane's first units of the row are requested before the weights are staged (hides the staging barrier)
    uint4 v[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int u = lane + 32 * k;
        v[k] = (m < M && u < nu) ? __ldg(reinterpret_cast<const uint4*>(x + (long long)u * DRQ_TB_ACT * 8)) : make_uint4(0, 0, 0, 0);
    }
    for (int k = threadIdx.x; k < na * H / 4; k += 256) {         // H % 8 == 0: whole float4s
        const float4 w = __ldg(reinterpret_cast<const float4*>(w4 + (long long)a_lo * H) + k);
        reinterpret_cast<float4*>(w_s)[k] = make_float4(__bfloat162float(__float2bfloat16_rn(w.x)), __bfloat162float(__float2bfloat16_rn(w.y)),
                                                        __bfloat162float(__float2bfloat16_rn(w.z)), __bfloat162float(__float2bfloat16_rn(w.w)));
    }
    const float std = std_dev ? *std_dev : 0.f;
    const float log_std = jobs.n ? logf(std) : 0.f;
    const float lo = -1.0f + 1e-6f, hi = 1.0f - 1e-6f;  // utils.py:113 (python: -1.0 + 1e-6 -> fp32)
    float lp_acc = 0.f;                                  // this thread's log-prob terms of the metrics job
    __syncthreads();
    for (int a0 = 0; a0 < na; a0 += 8) {
        float acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
        for (int u0 = lane; u0 < nu; u0 += 128) {     // 4 units of the row in flight per lane
            if (u0 != lane || a0 != 0) {
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const int u = u0 + 32 * k;
                    v[k] = (m < M && u < nu) ? __ldg(reinterpret_cast<const uint4*>(x + (long long)u * DRQ_TB_ACT * 8)) : make_uint4(0, 0, 0, 0);
                }
            }
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const int u = u0 + 32 * k;
                if (u >= nu) break;
                const uint32_t w[4] = {v[k].x, v[k].y, v[k].z, v[k].w};
                float xv[8];
#pragma unroll
                for (int j = 0; j < 4; ++j) { xv[2 * j] = __uint_as_float(w[j] << 16); xv[2 * j + 1] = __uint_as_float(w[j] & 0xFFFF0000u); }
#pragma unroll
                for (int a = 0; a < 8; ++a) {
                    if (a0 + a < na) {
                        const float4 w0 = *reinterpret_cast<const float4*>(w_s + (a0 + a) * H + u * 8);
                        const float4 w1 = *reinterpret_cast<const float4*>(w_s + (a0 + a) * H + u * 8 + 4);
                        acc[a] = fmaf(xv[0], w0.x, acc[a]); acc[a] = fmaf(xv[1], w0.y, acc[a]);
                        acc[a] = fmaf(xv[2], w0.z, acc[a]); acc[a] = fmaf(xv[3], w0.w, acc[a]);
                        acc[a] = fmaf(xv[4], w1.x, acc[a]); acc[a] = fmaf(xv[5], w1.y, acc[a]);
                        acc[a] = fmaf(xv[6], w1.z, acc[a]); acc[a] = fmaf(xv[7], w1.w, acc[a]);
                    }
                }
            }
        }
        // the row's dot products: butterfly over the lanes (fixed order), lane a keeps output a_lo + a0 + a and samples it
        float mine = 0.f;
#pragma unroll
        for (int a = 0; a < 8; ++a) {
            const float t = warp_sum(acc[a]);
            if (lane == a) mine = t;
        }
        const int j = a_lo + a0 + lane;
        if (lane < 8 && m < M && a0 + lane < na) {
            const float pre = mine + b4[j];
            mu_pre[(long long)m * A + j] = pre;
            for (int i = 0; i < jobs.n; ++i) {
                const drq_policy_sample& jb = jobs.j[i];
                const int b = m - jb.row0;
                if (b < 0 || b >= jb.rows) continue;
                const float mu = tanhf(pre);                                   // drqv2.py:89
                float av = mu;
                if (jb.eps) {
                    float e = __fmul_rn(jb.eps[(long long)b * A + j], std);    // utils.py:120
                    if (clip > 0.f) e = fminf(fmaxf(e, -clip), clip);          // utils.py:121-122
                    av = fminf(fmaxf(__fadd_rn(mu, e), lo), hi);               // utils.py:123, 113-116 (value)
                    if (i == jobs.metrics_job) {
                        const float d = av - mu;                                // Normal.log_prob(a)
                        lp_acc += -(d * d) / (2.0f * std * std) - log_std - 0.9189385332046727f;
                    }
                }
                jb.action_out[(long long)b * jb.ld_a + j] = av;
                if (jb.a_bf16) reinterpret_cast<__nv_bfloat16*>(jb.a_bf16)[fb_index(jb.feat_off + j, b, jb.units_a)] = __float2bfloat16_rn(av);
                if (jb.mu_out) jb.mu_out[(long long)b * A + j] = mu;
            }
        }
    }
    if (jobs.metrics_job < 0) return;
    // batch mean of the log-probabilities: block partials (y-major, then x), combined in that order by the block that
    // finishes last
    const unsigned int nblk = gridDim.x * gridDim.y;
    const float bsum = block_sum_256(lp_acc, sh);
    if (threadIdx.x == 0) {
        reinterpret_cast<float*>(scratch)[1 + blockIdx.y * gridDim.x + blockIdx.x] = bsum;
        __threadfence();
        s_last = atomicAdd(scratch, 1u) == nblk - 1;
    }
    __syncthreads();
    if (!s_last) return;
    // the last block adds the partials: thread t takes blocks t, t + 256, ... in order, then the block-wide sum (a fixed tree)
    __threadfence();
    float mine = 0.f;
    for (unsigned int b = threadIdx.x; b < nblk; b += 256) mine += __ldcg(reinterpret_cast<const float*>(scratch) + 1 + b);
    const float tot = block_sum_256(mine, sh);
    if (threadIdx.x == 0) {
        const drq_policy_sample& jb = jobs.j[jobs.metrics_job];
        jb.metrics[0] = tot / (float)jb.rows;                                       // actor_logprob
        jb.metrics[1] = (float)A * (0.5f + 0.9189385332046727f + log_std);          // actor_ent
        *scratch = 0u;                                                              // ready for the next launch
    }
}

__global__ void actor_sample_bwd_kernel(const float* __restrict__ da, long long ld_da,
                                        const float* __restrict__ mu, float* __restrict__ dmu_pre,
                                        __nv_bfloat16* __restrict__ dmu_bf, long long rpad_mb, int B, int A,
                                        int n_planes, long long plane_stride) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= B * A) return;
    const int b = i / A, j = i - b * A;
    const float m = mu[i];
    float dav = 0.f;
    const float* dp = da + (long long)b * ld_da + j;
    for (int p0 = 0; p0 < n_planes; p0 += 8) {
        float t[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) t[k] = p0 + k < n_planes ? dp[(p0 + k) * plane_stride] : 0.f;
#pragma unroll
        for (int k = 0; k < 8; ++k) dav += t[k];
    }
    const float g = dav * (1.0f - m * m);
    dmu_pre[i] = g;
    if (dmu_bf) dmu_bf[fb_index(j, b, rpad_mb)] = __float2bfloat16_rn(g);
}

__global__ void __launch_bounds__(256)
critic_loss_kernel(const float* __restrict__ q1, const float* __restrict__ q2,
                   const float* __restrict__ tq1, const float* __restrict__ tq2,
                   const float* __restrict__ reward, const float* __restrict__ discount,
                   float* __restrict__ dq1, float* __restrict__ dq2, float* __restrict__ tq_out,
                   float* __restrict__ metrics, int B) {
    __shared__ float sh[256];
    float s_r = 0.f, s_t = 0.f, s_1 = 0.f, s_2 = 0.f, s_l1 = 0.f, s_l2 = 0.f;
    const float scale = 2.0f / (float)B;
    for (int b = threadIdx.x; b < B; b += 256) {
        const float tv = fminf(tq1[b], tq2[b]);                                  // drqv2.py:185
        const float tq = __fadd_rn(reward[b], __fmul_rn(discount[b], tv));       // drqv2.py:186
        const float e1 = q1[b] - tq, e2 = q2[b] - tq;
        dq1[b] = scale * e1;   // d/dq mean((q - tq)^2)
        dq2[b] = scale * e2;
        if (tq_out) tq_out[b] = tq;
        s_r += reward[b]; s_t += tq; s_1 += q1[b]; s_2 += q2[b];
        s_l1 += e1 * e1; s_l2 += e2 * e2;
    }
    const float r = block_sum_256(s_r, sh), t = block_sum_256(s_t, sh);
    const float a = block_sum_256(s_1, sh), c = block_sum_256(s_2, sh);
    const float l1 = block_sum_256(s_l1, sh), l2 = block_sum_256(s_l2, sh);
    if (metrics && threadIdx.x == 0) {
        const float inv = 1.0f / (float)B;
        metrics[0] = r * inv;               // batch_reward       drqv2.py:249
        metrics[1] = t * inv;               // critic_target_q    drqv2.py:192
        metrics[2] = a * inv;               // critic_q1
        metrics[3] = c * inv;               // critic_q2
        metrics[4] = l1 * inv + l2 * inv;   // critic_loss        drqv2.py:189
    }
}

__global__ void __launch_bounds__(256)
actor_loss_kernel(const float* __restrict__ q1, const float* __restrict__ q2,
                  float* __restrict__ dq1, float* __restrict__ dq2, float* __restrict__ metrics,
                  int B) {
    __shared__ float sh[256];
    float s = 0.f;
    const float g = -1.0f / (float)B;
    for (int b = threadIdx.x; b < B; b += 256) {
        const float a = q1[b], c = q2[b];
        s += fminf(a, c);
        dq1[b] = a < c ? g : (a == c ? 0.5f * g : 0.f);
        dq2[b] = c < a ? g : (a == c ? 0.5f * g : 0.f);
    }
    const float t = block_sum_256(s, sh);
    if (metrics && threadIdx.x == 0) metrics[0] = -(t / (float)B);   // drqv2.py:216
}

// ---------------------------------------------------------------- bf16-mode helpers (TB layout; `rpad` = units per row)
// q[z][b] = c2[z][b][:] . w3[z][:] + b3[z]   (the Linear(hidden, 1) of drqv2.py:106,111) on an FB
// activation.  Block = 32 rows x 8 unit groups: lane = row (one coalesced 512-byte read per unit and
// warp), warp g sums units g, g+8, ...; the 8 partial sums are combined in fixed order.
__global__ void __launch_bounds__(256)
q_head_fwd_kernel(const __nv_bfloat16* __restrict__ c2, long long rpad, long long bs_c2,
                  const float* __restrict__ w3, const float* __restrict__ b3, float* __restrict__ q, int B, int H,
                  long long w_stride, int heads_inner, long long w_stride_outer) {
    extern __shared__ float w_s[];
    __shared__ float part[8][33];
    const int z = blockIdx.y;
    const long long woff = (z % heads_inner) * w_stride + (z / heads_inner) * w_stride_outer;
    for (int k = threadIdx.x; k < H; k += 256) w_s[k] = w3[woff + k];
    __syncthreads();
    const int lane = threadIdx.x & 31, grp = threadIdx.x >> 5;
    const int b = blockIdx.x * 32 + lane;
    float s0 = 0.f, s1 = 0.f;
    if (b < B) {
        const __nv_bfloat16* x = c2 + z * bs_c2 + fb_index(0, b, rpad);
#pragma unroll 4
        for (int u = grp; u < H / 8; u += 8) {
            const uint4 v = __ldg(reinterpret_cast<const uint4*>(x + (long long)u * DRQ_TB_ACT * 8));
            const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                s0 = fmaf(__uint_as_float(w[j] << 16), w_s[u * 8 + 2 * j], s0);
                s1 = fmaf(__uint_as_float(w[j] & 0xFFFF0000u), w_s[u * 8 + 2 * j + 1], s1);
            }
        }
    }
    part[grp][lane] = s0 + s1;
    __syncthreads();
    if (grp == 0 && b < B) {
        float t = 0.f;
#pragma unroll
        for (int g2 = 0; g2 < 8; ++g2) t += part[g2][lane];
        q[(long long)z * B + b] = t + b3[woff];
    }
}

// dc2[z][b][k] = dq[z][b] * w3[z][k] * (c2 > 0) (TB bf16); optionally dw3[z][k] = sum_b dq[z][b] c2[z][b][k]
// and db3[z] = sum_b dq[z][b].  One block per 8-feature unit; fixed-order tree.
// LOSS selects where dq comes from: 0 = given (head z reads dq1 / dq2); 1 = the critic loss of drqv2.py:185-189 computed here from
// (q, target q, reward, discount) - block (0,0) also writes the five metrics; 2 = the actor loss of
// drqv2.py:213-216 (-mean(min(Q1,Q2))), block (0,0) writes actor_loss.  Heads = 2 for LOSS != 0.
struct QLossArgs {
    const float* q;            // [2][B] online Q1, Q2
    const float* tq;           // [2][B] target Q1, Q2 (critic loss)
    const float* reward; const float* discount;
    float* target_q_out;       // nullable [B]
    float* metrics;            // nullable
};

template <int LOSS>
__device__ __forceinline__ float loss_dq(const QLossArgs& L, const float* dqz, int z, int b, int B) {
    if (LOSS == 0) return dqz[b];
    const float q1 = L.q[b], q2 = L.q[B + b];
    if (LOSS == 1) {
        const float tv = fminf(L.tq[b], L.tq[B + b]);                               // drqv2.py:185
        const float tq = __fadd_rn(L.reward[b], __fmul_rn(L.discount[b], tv));      // drqv2.py:186
        return (2.0f / (float)B) * ((z ? q2 : q1) - tq);                            // d/dq mean((q - tq)^2)
    }
    const float g = -1.0f / (float)B;                                               // d/dq -mean(min(q1, q2))
    const float mine = z ? q2 : q1, other = z ? q1 : q2;
    return mine < other ? g : (mine == other ? 0.5f * g : 0.f);
}

template <int LOSS>
__global__ void __launch_bounds__(256)
q_head_bwd_kernel(const float* __restrict__ dq1, const float* __restrict__ dq2, const QLossArgs L,
                  const __nv_bfloat16* __restrict__ c2, long long rpad,
                  long long bs_c2, const float* __restrict__ w3, __nv_bfloat16* __restrict__ dc2,
                  float* __restrict__ dw3, float* __restrict__ db3, int B, long long w_stride) {
    __shared__ float red[256][9];
    const int u = blockIdx.x, z = blockIdx.y;
    const float* dqz = LOSS == 0 ? (z ? dq2 : dq1) : nullptr;
    const long long base = z * bs_c2;
    float w[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) w[j] = w3[z * w_stride + u * 8 + j];
    float acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    float dq_sum = 0.f;
    for (int b = threadIdx.x; b < B; b += 256) {
        const long long at = base + fb_index(u * 8, b, rpad);
        const uint4 v = *reinterpret_cast<const uint4*>(c2 + at);
        const uint32_t cw[4] = {v.x, v.y, v.z, v.w};
        const float g = loss_dq<LOSS>(L, dqz, z, b, B);
        dq_sum += g;
        uint32_t pk[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const float a0 = __uint_as_float(cw[j] << 16), a1 = __uint_as_float(cw[j] & 0xFFFF0000u);
            acc[2 * j] = fmaf(g, a0, acc[2 * j]);
            acc[2 * j + 1] = fmaf(g, a1, acc[2 * j + 1]);
            const __nv_bfloat162 t = __floats2bfloat162_rn(a0 > 0.f ? g * w[2 * j] : 0.f, a1 > 0.f ? g * w[2 * j + 1] : 0.f);
            pk[j] = *reinterpret_cast<const uint32_t*>(&t);
        }
        *reinterpret_cast<uint4*>(dc2 + at) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
    }
    if (dw3) {
#pragma unroll
        for (int j = 0; j < 8; ++j) red[threadIdx.x][j] = acc[j];
        __syncthreads();
        for (int o = 128; o > 0; o >>= 1) {
            if (threadIdx.x < o) {
#pragma unroll
                for (int j = 0; j < 8; ++j) red[threadIdx.x][j] += red[threadIdx.x + o][j];
            }
            __syncthreads();
        }
        if (threadIdx.x < 8) dw3[z * w_stride + u * 8 + threadIdx.x] = red[0][threadIdx.x];
        __syncthreads();
    }
    if (u != 0) return;
    float* sh = &red[0][0];
    if (db3) {
        const float t = block_sum_256(dq_sum, sh);
        if (threadIdx.x == 0) db3[z * w_stride] = t;
    }
    if (LOSS != 0 && z == 0 && (L.metrics || L.target_q_out)) {
        // the scalars of drqv2.py:189-195,216 (one block, fixed-order sums)
        float s_r = 0.f, s_t = 0.f, s_1 = 0.f, s_2 = 0.f, s_l1 = 0.f, s_l2 = 0.f, s_min = 0.f;
        for (int b = threadIdx.x; b < B; b += 256) {
            const float q1 = L.q[b], q2 = L.q[B + b];
            if (LOSS == 1) {
                const float tv = fminf(L.tq[b], L.tq[B + b]);
                const float tq = __fadd_rn(L.reward[b], __fmul_rn(L.discount[b], tv));
                const float e1 = q1 - tq, e2 = q2 - tq;
                if (L.target_q_out) L.target_q_out[b] = tq;
                s_r += L.reward[b]; s_t += tq; s_1 += q1; s_2 += q2; s_l1 += e1 * e1; s_l2 += e2 * e2;
            } else {
                s_min += fminf(q1, q2);
            }
        }
        const float inv = 1.0f / (float)B;
        if (LOSS == 1) {
            const float r = block_sum_256(s_r, sh), t = block_sum_256(s_t, sh);
            const float a = block_sum_256(s_1, sh), c = block_sum_256(s_2, sh);
            const float l1 = block_sum_256(s_l1, sh), l2 = block_sum_256(s_l2, sh);
            if (L.metrics && threadIdx.x == 0) {
                L.metrics[0] = r * inv; L.metrics[1] = t * inv; L.metrics[2] = a * inv; L.metrics[3] = c * inv;
                L.metrics[4] = l1 * inv + l2 * inv;
            }
        } else {
            const float t = block_sum_256(s_min, sh);
            if (L.metrics && threadIdx.x == 0) L.metrics[0] = -(t * inv);
        }
    }
}

}  // namespace drq

using namespace drq;

extern "C" {

int drq_ln_tanh_fwd_multi(const drq_ln_job* jobs, int njobs, int B, int F, float eps, void* stream) {
    DRQ_REQUIRE(jobs && njobs >= 1 && njobs <= DRQ_LN_MAX_JOBS, "ln_tanh_fwd: 1..%d jobs", DRQ_LN_MAX_JOBS);
    DRQ_REQUIRE(B >= 0 && F > 0 && F <= 32 * kMaxFPerLane, "ln_tanh_fwd: bad dims (F<=256)");
    LnJobs js{};
    for (int i = 0; i < njobs; ++i) {
        js.j[i] = jobs[i];
        DRQ_REQUIRE(jobs[i].partial && jobs[i].bias && jobs[i].gamma && jobs[i].beta && jobs[i].h_out && jobs[i].S >= 1,
                    "ln_tanh_fwd: null pointer in job %d", i);
        DRQ_REQUIRE(jobs[i].n_tail >= 0 && (jobs[i].n_tail == 0 || !jobs[i].tail || !jobs[i].h_bf16 ||
                                            F + jobs[i].n_tail <= 8 * jobs[i].units_bf16),
                    "ln_tanh_fwd: tail of job %d does not fit the bf16 row (F + n_tail > 8 * units_bf16)", i);
    }
    if (B == 0) return DRQ_OK;
    const dim3 grid(B, njobs);
    cudaStream_t s = as_stream(stream);
    if (F <= 64) ln_tanh_fwd_kernel<2><<<grid, 128, 0, s>>>(js, B, F, eps);
    else if (F <= 128) ln_tanh_fwd_kernel<4><<<grid, 128, 0, s>>>(js, B, F, eps);
    else ln_tanh_fwd_kernel<8><<<grid, 128, 0, s>>>(js, B, F, eps);
    return check_launch("ln_tanh_fwd_kernel");
}

int drq_ln_tanh_fwd(const float* partial, int S, int64_t split_stride, const float* bias,
                    const float* gamma, const float* beta, float* h_out, int64_t ld_h, float* xhat,
                    float* rstd, uint16_t* h_bf16, int64_t rpad_hb, int B, int F, float eps, void* stream) {
    drq_ln_job j{};
    j.partial = partial; j.ld_partial = F; j.split_stride = split_stride; j.S = S;
    j.bias = bias; j.gamma = gamma; j.beta = beta; j.h_out = h_out; j.ld_h = ld_h; j.xhat = xhat; j.rstd = rstd;
    j.h_bf16 = h_bf16; j.units_bf16 = rpad_hb; j.row0_bf16 = 0; j.tail = nullptr; j.ld_tail = 0; j.n_tail = 0;
    return drq_ln_tanh_fwd_multi(&j, 1, B, F, eps, stream);
}

int drq_ln_tanh_bwd(const float* dh, int64_t ld_dh, const float* h, int64_t ld_h, const float* xhat,
                    const float* rstd, const float* gamma, float* dz, float* dgamma, float* dbeta,
                    uint16_t* dz_bf16, int64_t rpad_zb, int B, int F, int n_planes, int64_t plane_stride,
                    void* stream) {
    DRQ_REQUIRE(dh && h && xhat && rstd && gamma && dz && n_planes >= 1 && (!dgamma == !dbeta), "ln_tanh_bwd: null pointer");
    DRQ_REQUIRE(B > 0 && F > 0 && F <= 32 * kMaxFPerLane, "ln_tanh_bwd: bad dims (F<=256)");
    // dy = dh * tanh' is staged in the second half of the caller's 2*B*F buffer
    float* dy = dz + (long long)B * F;
    ln_tanh_bwd_row_kernel<<<(B + 3) / 4, 128, 0, as_stream(stream)>>>(dh, ld_dh, h, ld_h, xhat, rstd,
                                                                      gamma, dz, dy,
                                                                      reinterpret_cast<__nv_bfloat16*>(dz_bf16), rpad_zb, B, F,
                                                                      n_planes, plane_stride);
    if (int rc = check_launch("ln_tanh_bwd_row_kernel")) return rc;
    if (!dgamma) return DRQ_OK;
    ln_param_grad_kernel<<<F, 256, 0, as_stream(stream)>>>(dy, xhat, dgamma, dbeta, B, F);
    return check_launch("ln_param_grad_kernel");
}

int drq_actor_sample(const float* mu_pre, const float* eps, const float* std_dev, float clip,
                     float* action_out, int64_t ld_a, float* mu_out, float* metrics, int B, int A, void* stream) {
    DRQ_REQUIRE(mu_pre && action_out, "actor_sample: null pointer");
    DRQ_REQUIRE(!(eps && !std_dev), "actor_sample: eps without std");
    DRQ_REQUIRE(B > 0 && A > 0, "actor_sample: bad dims");
    actor_sample_kernel<<<1, 256, 0, as_stream(stream)>>>(mu_pre, eps, std_dev, clip, action_out, ld_a, mu_out, metrics, B, A);
    return check_launch("actor_sample_kernel");
}

int drq_policy_head_fwd_bf16(const uint16_t* p2, int64_t units, const float* w4, const float* b4, float* mu_pre, int M,
                             int H, int A, const drq_policy_sample* jobs, int njobs, const float* std_dev, float clip,
                             uint32_t* ticket, void* stream) {
    DRQ_REQUIRE(p2 && w4 && b4 && mu_pre, "policy_head_fwd: null pointer");
    DRQ_REQUIRE(M > 0 && H > 0 && H % 8 == 0 && units * 8 >= H && A > 0 && A <= DRQ_POLICY_MAX_A,
                "policy_head_fwd: bad dims (A <= %d, H %% 8 == 0)", DRQ_POLICY_MAX_A);
    DRQ_REQUIRE(njobs >= 0 && njobs <= DRQ_POLICY_MAX_JOBS && (njobs == 0 || jobs), "policy_head_fwd: 0..%d sample jobs", DRQ_POLICY_MAX_JOBS);
    PolicyJobs pj{};
    pj.n = njobs;
    pj.metrics_job = -1;
    for (int i = 0; i < njobs; ++i) {
        pj.j[i] = jobs[i];
        DRQ_REQUIRE(jobs[i].rows > 0 && jobs[i].row0 >= 0 && jobs[i].row0 + jobs[i].rows <= M && jobs[i].action_out,
                    "policy_head_fwd: bad sample job %d", i);
        DRQ_REQUIRE(!(jobs[i].eps && !std_dev), "policy_head_fwd: eps without std");
        if (jobs[i].metrics) {
            DRQ_REQUIRE(pj.metrics_job < 0 && jobs[i].eps && ticket, "policy_head_fwd: one job may carry metrics (it needs eps and the scratch words)");
            pj.metrics_job = i;
        }
    }
    const int groups = (A + kPolicyGroup - 1) / kPolicyGroup;
    const dim3 grid((M + kPolicyRows - 1) / kPolicyRows, groups);
    DRQ_REQUIRE(pj.metrics_job < 0 || (long long)grid.x * grid.y <= DRQ_POLICY_MAX_PARTIALS,
                "policy_head_fwd: the metrics scratch holds %d block partials (ceil(M / 8) x ceil(A / 32) blocks)",
                DRQ_POLICY_MAX_PARTIALS);
    const size_t smem = (size_t)((A + groups - 1) / groups) * H * sizeof(float);
    if (int rc = ensure_smem((const void*)policy_head_fwd_kernel, smem, "policy_head_fwd")) return rc;
    policy_head_fwd_kernel<<<grid, 256, smem, as_stream(stream)>>>(reinterpret_cast<const __nv_bfloat16*>(p2),
             (long long)units, w4, b4, mu_pre, M, H, A, pj, std_dev, clip, ticket);
    return check_launch("policy_head_fwd_kernel");
}

int drq_actor_sample_bwd(const float* daction, int64_t ld_da, const float* mu, float* dmu_pre,
                         uint16_t* dmu_bf16, int64_t rpad_mb, int B, int A, int n_planes, int64_t plane_stride,
                         void* stream) {
    DRQ_REQUIRE(daction && mu && dmu_pre && B > 0 && A > 0 && n_planes >= 1, "actor_sample_bwd: bad args");
    actor_sample_bwd_kernel<<<(B * A + 255) / 256, 256, 0, as_stream(stream)>>>(daction, ld_da, mu,
                                                                                dmu_pre,
                                                                                reinterpret_cast<__nv_bfloat16*>(dmu_bf16), rpad_mb, B, A,
                                                                                n_planes, plane_stride);
    return check_launch("actor_sample_bwd_kernel");
}

int drq_critic_loss(const float* q1, const float* q2, const float* tq1, const float* tq2,
                    const float* reward, const float* discount, float* dq1, float* dq2,
                    float* target_q_out, float* metrics, int B, void* stream) {
    DRQ_REQUIRE(q1 && q2 && tq1 && tq2 && reward && discount && dq1 && dq2, "critic_loss: null pointer");
    DRQ_REQUIRE(B > 0, "critic_loss: bad dims");
    critic_loss_kernel<<<1, 256, 0, as_stream(stream)>>>(q1, q2, tq1, tq2, reward, discount, dq1, dq2,
                                                         target_q_out, metrics, B);
    return check_launch("critic_loss_kernel");
}

int drq_q_head_fwd_bf16(const uint16_t* c2, int64_t rpad, int64_t bs_c2, const float* w3, const float* b3,
                        float* q, int B, int H, int heads, int64_t w_stride, int heads_inner, int64_t w_stride_outer,
                        void* stream) {
    DRQ_REQUIRE(c2 && w3 && b3 && q && B > 0 && H > 0 && H % 8 == 0 && heads > 0 && heads_inner > 0, "q_head_fwd: bad args");
    q_head_fwd_kernel<<<dim3((B + 31) / 32, heads), 256, H * sizeof(float), as_stream(stream)>>>(
        reinterpret_cast<const __nv_bfloat16*>(c2), rpad, bs_c2, w3, b3, q, B, H, w_stride, heads_inner, w_stride_outer);
    return check_launch("q_head_fwd_kernel");
}

int drq_q_head_bwd_loss_bf16(int loss, const float* q, const float* tq, const float* reward, const float* discount,
                             float* target_q_out, float* metrics, const uint16_t* c2, int64_t rpad, int64_t bs_c2,
                             const float* w3, uint16_t* dc2, float* dw3, float* db3, int B, int H, int64_t w_stride,
                             void* stream) {
    DRQ_REQUIRE(loss == 1 || loss == 2, "q_head_bwd_loss: loss must be 1 (critic) or 2 (actor)");
    DRQ_REQUIRE(q && c2 && w3 && dc2 && B > 0 && H > 0 && H % 8 == 0, "q_head_bwd_loss: bad args");
    DRQ_REQUIRE(loss == 2 || (tq && reward && discount), "q_head_bwd_loss: critic loss needs tq, reward, discount");
    const QLossArgs L{q, tq, reward, discount, target_q_out, metrics};
    const auto c2p = reinterpret_cast<const __nv_bfloat16*>(c2);
    const auto dp = reinterpret_cast<__nv_bfloat16*>(dc2);
    if (loss == 1)
        q_head_bwd_kernel<1><<<dim3(H / 8, 2), 256, 0, as_stream(stream)>>>(nullptr, nullptr, L, c2p, rpad, bs_c2, w3, dp, dw3, db3,
                 B, w_stride);
    else
        q_head_bwd_kernel<2><<<dim3(H / 8, 2), 256, 0, as_stream(stream)>>>(nullptr, nullptr, L, c2p, rpad, bs_c2, w3, dp, dw3, db3,
                 B, w_stride);
    return check_launch("q_head_bwd_kernel");
}

int drq_q_head_bwd_bf16(const float* dq1, const float* dq2, const uint16_t* c2, int64_t rpad, int64_t bs_c2,
                        const float* w3, uint16_t* dc2, float* dw3, float* db3, int B, int H, int64_t w_stride,
                        void* stream) {
    DRQ_REQUIRE(c2 && w3 && dc2 && B > 0 && H > 0 && H % 8 == 0, "q_head_bwd: bad args");
    if (!dq1 && !dq2) return DRQ_OK;
    const QLossArgs L{};
    const auto c2p = reinterpret_cast<const __nv_bfloat16*>(c2);
    auto dp = reinterpret_cast<__nv_bfloat16*>(dc2);
    if (dq1 && dq2) {
        q_head_bwd_kernel<0><<<dim3(H / 8, 2), 256, 0, as_stream(stream)>>>(dq1, dq2, L, c2p, rpad, bs_c2, w3, dp, dw3, db3,
                 B, w_stride);
    } else {
        // one head: its operands moved to z = 0
        const long long zc = dq1 ? 0 : bs_c2, zw = dq1 ? 0 : w_stride;
        q_head_bwd_kernel<0><<<dim3(H / 8, 1), 256, 0, as_stream(stream)>>>(dq1 ? dq1 : dq2, nullptr, L, c2p + zc, rpad, bs_c2,
                 w3 + zw, dp + zc, dw3 ? dw3 + zw : nullptr, db3 ? db3 + zw : nullptr, B, w_stride);
    }
    return check_launch("q_head_bwd_kernel");
}

int drq_actor_loss(const float* q1, const float* q2, float* dq1, float* dq2, float* metrics, int B,
                   void* stream) {
    DRQ_REQUIRE(q1 && q2 && dq1 && dq2 && B > 0, "actor_loss: bad args");
    actor_loss_kernel<<<1, 256, 0, as_stream(stream)>>>(q1, q2, dq1, dq2, metrics, B);
    return check_launch("actor_loss_kernel");
}

}  // extern "C"

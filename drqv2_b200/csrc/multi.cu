// Multi-job launchers of the small per-tensor kernels of the bf16 update: one launch refreshes all bf16
// operand copies of a network after its optimiser step (drq_pack_multi) and one launch computes all bias
// gradients of a backward pass (drq_colsum_multi).  These kernels are microseconds of work each; as
// separate launches their cost is launch latency and cold instruction fetch (DESIGN.md §6).
#include "pack.cuh"
#include "wgrad_reduce.cuh"

namespace drq {

struct PackJobs { drq_pack_job j[DRQ_PACK_MAX_JOBS]; int first_block[DRQ_PACK_MAX_JOBS + 1]; int n; };

__global__ void __launch_bounds__(256) pack_multi_kernel(const PackJobs jobs) {
    __shared__ float sm[32 * 33];
    int ji = 0;
    while (ji + 1 < jobs.n && (int)blockIdx.x >= jobs.first_block[ji + 1]) ++ji;
    const drq_pack_job& jb = jobs.j[ji];
    const int b = blockIdx.x - jobs.first_block[ji];
    __nv_bfloat16* out = reinterpret_cast<__nv_bfloat16*>(jb.out);
    if (jb.kind == DRQ_PACK_LINEAR) {
        const int units = (jb.cols + 15) / 16 * 2;
        const int rblocks = ((jb.rows + DRQ_TB_W - 1) / DRQ_TB_W * DRQ_TB_W + 255) / 256;
        pack_linear_tb_block(jb.w, out, jb.rows, jb.cols, units, b % rblocks, b / rblocks, threadIdx.x);
    } else if (jb.kind == DRQ_PACK_TRUNK) {
        pack_trunk_tb_block(jb.w, out, jb.rows, b % 39, b / 39, threadIdx.x, reinterpret_cast<float(*)[33]>(sm));
    } else if (jb.kind == DRQ_PACK_CONV) {
        pack_conv_w_elem(jb.w, out, reinterpret_cast<__nv_bfloat16*>(jb.out2), b * 256 + threadIdx.x);
    } else {
        pack_conv1_w_block(jb.w, jb.bias, out, jb.cols, threadIdx.x, reinterpret_cast<float(*)[9]>(sm));
    }
}

struct ColsumJobs { drq_colsum_job j[DRQ_COLSUM_MAX_JOBS]; };

// out[n] = sum_m X[m][n] for 32 columns per block, blockIdx.y = job; fixed-order reductions.
//   fp32 rows : 32 columns x 8 row lanes.
//   TB bf16   : 4 units x 64 row lanes, one 16-byte load (8 columns of one row) per thread and step.
__global__ void __launch_bounds__(256) colsum_multi_kernel(const ColsumJobs jobs) {
    __shared__ float red[64][33];
    const drq_colsum_job& jb = jobs.j[blockIdx.y];
    if (blockIdx.x * 32 >= jb.N) return;
    if (jb.tb) {
        const __nv_bfloat16* X = reinterpret_cast<const __nv_bfloat16*>(jb.X);
        const int u = threadIdx.x & 3, ry = threadIdx.x >> 2;
        const long long unit = (long long)blockIdx.x * 4 + u;
        float acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
        if (unit * 8 < jb.N) {
            for (int m = ry; m < jb.M; m += 64) {
                const uint4 v = *reinterpret_cast<const uint4*>(X + (((long long)(m >> 7) * jb.ld + unit) * DRQ_TB_ACT + (m & 127)) * 8);
                const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    acc[2 * j] += __uint_as_float(w[j] << 16);
                    acc[2 * j + 1] += __uint_as_float(w[j] & 0xFFFF0000u);
                }
            }
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) red[ry][u * 8 + j] = acc[j];
        __syncthreads();
        if (threadIdx.x < 32) {
            const int n = blockIdx.x * 32 + threadIdx.x;
            float t = 0.f;
            for (int r = 0; r < 64; ++r) t += red[r][threadIdx.x];
            if (n < jb.N) jb.out[n] = t;
        }
        return;
    }
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int n = blockIdx.x * 32 + tx;
    float s = 0.f;
    if (n < jb.N) {
        const float* X = reinterpret_cast<const float*>(jb.X);
        if (jb.Y) { for (int m = ty; m < jb.M; m += 8) s += X[m * jb.ld + n] * jb.Y[m * jb.ld + n]; }
        else { for (int m = ty; m < jb.M; m += 8) s += X[m * jb.ld + n]; }
    }
    red[ty][tx] = s;
    __syncthreads();
    if (ty == 0 && n < jb.N) {
        float t = red[0][tx];
#pragma unroll
        for (int r = 1; r < 8; ++r) t += red[r][tx];
        jb.out[n] = t;
    }
}

struct WgReduceJobs { drq_wgrad_reduce_job j[DRQ_WGRAD_REDUCE_MAX_JOBS]; int G[DRQ_WGRAD_REDUCE_MAX_JOBS]; };

// all weight-gradient partial reductions of the encoder backward in one launch: blockIdx.y = layer
__global__ void __launch_bounds__(256) wgrad_reduce_multi_kernel(const WgReduceJobs jobs) {
    __shared__ float red[8][33], redb[8][33];
    const drq_wgrad_reduce_job& jb = jobs.j[blockIdx.y];
    const int G = jobs.G[blockIdx.y];
    if (jb.cin > 0) {
        if ((int)blockIdx.x < kC1ReduceBlocks) conv1_reduce_block(jb.partial, G, jb.cin, jb.dw, jb.db, blockIdx.x, red, redb);
    } else {
        wgrad3x3_reduce_block(jb.partial, G, jb.dw, jb.db, blockIdx.x, red);
    }
}

}  // namespace drq

using namespace drq;

extern "C" {

int drq_pack_multi(const drq_pack_job* jobs, int njobs, void* stream) {
    DRQ_REQUIRE(jobs && njobs >= 1 && njobs <= DRQ_PACK_MAX_JOBS, "pack_multi: 1..%d jobs", DRQ_PACK_MAX_JOBS);
    PackJobs pj{};
    pj.n = njobs;
    int blocks = 0;
    for (int i = 0; i < njobs; ++i) {
        const drq_pack_job& jb = jobs[i];
        DRQ_REQUIRE(jb.w && jb.out && jb.kind >= DRQ_PACK_LINEAR && jb.kind <= DRQ_PACK_CONV1, "pack_multi: bad job %d", i);
        pj.j[i] = jb;
        pj.first_block[i] = blocks;
        const int rpad = (jb.rows + DRQ_TB_W - 1) / DRQ_TB_W * DRQ_TB_W;
        if (jb.kind == DRQ_PACK_LINEAR) {
            DRQ_REQUIRE(jb.rows > 0 && jb.cols > 0, "pack_multi: bad linear dims in job %d", i);
            blocks += ((rpad + 255) / 256) * ((jb.cols + 15) / 16 * 2);
        } else if (jb.kind == DRQ_PACK_TRUNK) {
            DRQ_REQUIRE(jb.rows > 0, "pack_multi: bad trunk rows in job %d", i);
            blocks += 39 * rpad;
        } else if (jb.kind == DRQ_PACK_CONV) {
            DRQ_REQUIRE(jb.out2, "pack_multi: conv job %d needs the dgrad operand buffer", i);
            blocks += 36;
        } else {
            DRQ_REQUIRE(jb.bias && jb.cols > 0 && jb.cols * 9 + 1 <= 96, "pack_multi: bad conv1 job %d", i);
            blocks += 1;
        }
    }
    pj.first_block[njobs] = blocks;
    pack_multi_kernel<<<blocks, 256, 0, as_stream(stream)>>>(pj);
    return check_launch("pack_multi_kernel");
}

int drq_colsum_multi(const drq_colsum_job* jobs, int njobs, void* stream) {
    DRQ_REQUIRE(jobs && njobs >= 1 && njobs <= DRQ_COLSUM_MAX_JOBS, "colsum_multi: 1..%d jobs", DRQ_COLSUM_MAX_JOBS);
    ColsumJobs cj{};
    int nmax = 0;
    for (int i = 0; i < njobs; ++i) {
        DRQ_REQUIRE(jobs[i].X && jobs[i].out && jobs[i].M > 0 && jobs[i].N > 0, "colsum_multi: bad job %d", i);
        cj.j[i] = jobs[i];
        nmax = jobs[i].N > nmax ? jobs[i].N : nmax;
    }
    colsum_multi_kernel<<<dim3((nmax + 31) / 32, njobs), 256, 0, as_stream(stream)>>>(cj);
    return check_launch("colsum_multi_kernel");
}

int drq_conv_wgrad_reduce_multi(const drq_wgrad_reduce_job* jobs, int njobs, void* stream) {
    DRQ_REQUIRE(jobs && njobs >= 1 && njobs <= DRQ_WGRAD_REDUCE_MAX_JOBS, "wgrad_reduce_multi: 1..%d jobs", DRQ_WGRAD_REDUCE_MAX_JOBS);
    WgReduceJobs wj{};
    for (int i = 0; i < njobs; ++i) {
        const drq_wgrad_reduce_job& jb = jobs[i];
        DRQ_REQUIRE(jb.partial && jb.dw && jb.db && jb.n_images > 0 && jb.cin >= 0 && jb.cin * 9 + 1 <= 96 &&
                    (jb.cin > 0 || (jb.hout > 0 && jb.hout <= DRQ_PW - 2)), "wgrad_reduce_multi: bad job %d", i);
        wj.j[i] = jb;
        wj.G[i] = jb.cin > 0 ? conv1_wgrad_ctas(jb.n_images) : conv_wgrad_ctas(jb.n_images, jb.hout);
    }
    wgrad_reduce_multi_kernel<<<dim3(kWgReduceBlocks, njobs), 256, 0, as_stream(stream)>>>(wj);
    return check_launch("wgrad_reduce_multi_kernel");
}

}  // extern "C"

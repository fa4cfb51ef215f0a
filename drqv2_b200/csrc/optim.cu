// Multi-tensor Adam and the soft target update over the flat parameter arena.
// Reference: torch.optim.Adam x3 (drqv2.py:148-150) — single-tensor math of
// torch/optim/adam.py:457,476,531-547 — and utils.soft_update_params (utils.py:42-45).
#include "common.cuh"
#include "pack.cuh"

namespace drq {

__device__ __forceinline__ void adam_elem(float& p, float g, float& m, float& v, float omb1, float b2,
                                          float omb2, float bc2_sqrt, float eps, float neg_step) {
    // exp_avg.lerp_(grad, 1-beta1): weight < 0.5 -> fma(weight, end - start, start)  (ATen Lerp.h)
    m = fmaf(omb1, __fsub_rn(g, m), m);
    // exp_avg_sq.mul_(beta2).addcmul_(grad, grad, value=1-beta2)
    v = __fadd_rn(__fmul_rn(v, b2), __fmul_rn(__fmul_rn(omb2, g), g));
    // denom = (exp_avg_sq.sqrt() / bias_correction2_sqrt).add_(eps)
    const float denom = __fadd_rn(__fdiv_rn(__fsqrt_rn(v), bc2_sqrt), eps);
    // param.addcdiv_(exp_avg, denom, value=-step_size)
    p = __fadd_rn(p, __fmul_rn(neg_step, __fdiv_rn(m, denom)));
}

__device__ __forceinline__ void adam_range(float* __restrict__ p, const float* __restrict__ g,
                                           float* __restrict__ m, float* __restrict__ v, long long n,
                                           const float* __restrict__ sc, long long tid,
                                           long long nthreads) {
    const float omb1 = sc[0], b2 = sc[1], omb2 = sc[2], bc2s = sc[3], eps = sc[4], nstep = sc[5];
    const long long n4 = n >> 2;
    float4* p4 = reinterpret_cast<float4*>(p);
    const float4* g4 = reinterpret_cast<const float4*>(g);
    float4* m4 = reinterpret_cast<float4*>(m);
    float4* v4 = reinterpret_cast<float4*>(v);
    for (long long i = tid; i < n4; i += nthreads) {
        float4 pp = p4[i], gg = g4[i], mm = m4[i], vv = v4[i];
        adam_elem(pp.x, gg.x, mm.x, vv.x, omb1, b2, omb2, bc2s, eps, nstep);
        adam_elem(pp.y, gg.y, mm.y, vv.y, omb1, b2, omb2, bc2s, eps, nstep);
        adam_elem(pp.z, gg.z, mm.z, vv.z, omb1, b2, omb2, bc2s, eps, nstep);
        adam_elem(pp.w, gg.w, mm.w, vv.w, omb1, b2, omb2, bc2s, eps, nstep);
        p4[i] = pp; m4[i] = mm; v4[i] = vv;
    }
    for (long long i = (n4 << 2) + tid; i < n; i += nthreads)
        adam_elem(p[i], g[i], m[i], v[i], omb1, b2, omb2, bc2s, eps, nstep);
}

__device__ __forceinline__ void ema_range(const float* __restrict__ src, float* __restrict__ dst,
                                          long long n, float tau, float omt, long long tid,
                                          long long nthreads) {
    const long long n4 = n >> 2;
    const float4* s4 = reinterpret_cast<const float4*>(src);
    float4* d4 = reinterpret_cast<float4*>(dst);
    for (long long i = tid; i < n4; i += nthreads) {
        const float4 s = s4[i];
        float4 d = d4[i];
        d.x = __fadd_rn(__fmul_rn(tau, s.x), __fmul_rn(omt, d.x));   // utils.py:44-45
        d.y = __fadd_rn(__fmul_rn(tau, s.y), __fmul_rn(omt, d.y));
        d.z = __fadd_rn(__fmul_rn(tau, s.z), __fmul_rn(omt, d.z));
        d.w = __fadd_rn(__fmul_rn(tau, s.w), __fmul_rn(omt, d.w));
        d4[i] = d;
    }
    for (long long i = (n4 << 2) + tid; i < n; i += nthreads)
        dst[i] = __fadd_rn(__fmul_rn(tau, src[i]), __fmul_rn(omt, dst[i]));
}

// blocks [0, adam_blocks) run Adam, the rest run the EMA: one launch, two segments.
__global__ void __launch_bounds__(256)
adam_ema_kernel(float* p, const float* g, float* m, float* v, long long n_adam, const float* sc,
                const float* ema_src, float* ema_dst, long long n_ema, float tau, float omt,
                int adam_blocks) {
    if ((int)blockIdx.x < adam_blocks) {
        adam_range(p, g, m, v, n_adam, sc, blockIdx.x * 256ll + threadIdx.x, adam_blocks * 256ll);
    } else {
        const int eb = gridDim.x - adam_blocks;
        ema_range(ema_src, ema_dst, n_ema, tau, omt, (blockIdx.x - adam_blocks) * 256ll + threadIdx.x,
                  eb * 256ll);
    }
}

// ------------------------------------------------------------------ optimiser step + bf16 refresh, one launch
// (drq_adam_pack_step).  Every block owns one tile of one segment: it updates the tile's fp32 values with
// coalesced 4-byte accesses (tensor offsets inside the arena are not 16-byte aligned), keeps the new values on
// chip and writes the tile's bf16 operand units from there.

constexpr int kOptTile = 2048;            // elements per block of the flat kinds: two float4 per thread
constexpr int kGenK = 4;                  // generic LINEAR / CONV1: scalar elements per thread
constexpr int kGenTile = 256 * kGenK;
constexpr int kTrunkW = 245;              // TRUNK: pixels per block (35*35 = 5 * 245), 8 channels x 245 pixels

struct OptArgs {
    drq_opt_seg s[DRQ_OPT_MAX_SEGS];
    int first_block[DRQ_OPT_MAX_SEGS + 1];
    int n;
    float* p; const float* g; float* m; float* v; const float* sc;
    const float* src; float* dst;
    float tau, omt;
};

// tile of a generic LINEAR segment (cols not a multiple of 8): RT rows x CW columns (<= 1024 elements), smem row
// pitch SW (= 8 mod 64 elements, so that the 16-byte unit reads of consecutive rows fall into different banks)
struct LinTile { int CW, RT, SW, chunks, width; };
__host__ __device__ inline LinTile lin_tile(int cols) {
    LinTile t;
    const int c8 = (cols + 7) / 8 * 8;
    t.CW = c8 < 256 ? c8 : 256;
    const int rt = kGenTile / t.CW;
    int p2 = 1;
    while (p2 * 2 <= rt && p2 < 32) p2 *= 2;
    t.RT = p2;
    t.chunks = (cols + t.CW - 1) / t.CW;
    t.width = t.chunks == 1 ? cols : t.CW;
    t.SW = (t.CW + 55) / 64 * 64 + 8;
    return t;
}
constexpr int kOptShBf16 = 32 * 72;            // largest RT * SW (RT = 32 needs CW <= 32 -> SW = 72; CW = 256 -> 4 x 264)
constexpr int kOptShBytes = (288 * 10 + 32 + 32 * 9) * 4;   // CONV1: weights + bias + the bias partial sums
static_assert(kOptShBytes >= 8 * 256 * 4 && kOptShBytes >= kOptShBf16 * 2, "shared buffer covers every kind");

// arenas already offset to the segment's first element (16-byte aligned); offsets inside a segment fit in 32 bits
struct Upd {
    float* p; const float* g; float* m; float* v;
    float omb1, b2, omb2, bc2s, eps, nstep, tau, omt;
    bool ema;
};

__device__ __forceinline__ float ema_elem(float dst, float src, float tau, float omt) {
    return __fadd_rn(__fmul_rn(tau, src), __fmul_rn(omt, dst));   // utils.py:44-45
}

// NV float4 per thread: all loads first, then the arithmetic and the stores
template <int NV>
__device__ __forceinline__ void upd_vec(const Upd& u, const int (&i4)[NV], const bool (&ok)[NV], float4 (&out)[NV]) {
    float4 pp[NV], gg[NV], mm[NV], vv[NV];
#pragma unroll
    for (int k = 0; k < NV; ++k) {
        pp[k] = gg[k] = mm[k] = vv[k] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (ok[k]) {
            pp[k] = reinterpret_cast<const float4*>(u.p)[i4[k]];
            gg[k] = reinterpret_cast<const float4*>(u.g)[i4[k]];
            if (!u.ema) {
                mm[k] = reinterpret_cast<const float4*>(u.m)[i4[k]];
                vv[k] = reinterpret_cast<const float4*>(u.v)[i4[k]];
            }
        }
    }
#pragma unroll
    for (int k = 0; k < NV; ++k) {
        if (ok[k]) {
            if (u.ema) {
                pp[k].x = ema_elem(pp[k].x, gg[k].x, u.tau, u.omt);
                pp[k].y = ema_elem(pp[k].y, gg[k].y, u.tau, u.omt);
                pp[k].z = ema_elem(pp[k].z, gg[k].z, u.tau, u.omt);
                pp[k].w = ema_elem(pp[k].w, gg[k].w, u.tau, u.omt);
                reinterpret_cast<float4*>(u.p)[i4[k]] = pp[k];
            } else {
                adam_elem(pp[k].x, gg[k].x, mm[k].x, vv[k].x, u.omb1, u.b2, u.omb2, u.bc2s, u.eps, u.nstep);
                adam_elem(pp[k].y, gg[k].y, mm[k].y, vv[k].y, u.omb1, u.b2, u.omb2, u.bc2s, u.eps, u.nstep);
                adam_elem(pp[k].z, gg[k].z, mm[k].z, vv[k].z, u.omb1, u.b2, u.omb2, u.bc2s, u.eps, u.nstep);
                adam_elem(pp[k].w, gg[k].w, mm[k].w, vv[k].w, u.omb1, u.b2, u.omb2, u.bc2s, u.eps, u.nstep);
                reinterpret_cast<float4*>(u.p)[i4[k]] = pp[k];
                reinterpret_cast<float4*>(u.m)[i4[k]] = mm[k];
                reinterpret_cast<float4*>(u.v)[i4[k]] = vv[k];
            }
        }
        out[k] = pp[k];
    }
}

// K scalar elements per thread; elements k < KFULL are always live, the others iff tail_ok
template <int K, int KFULL>
__device__ __forceinline__ void upd_scalar(const Upd& u, const int (&o)[K], const bool (&tail_ok)[K], float (&out)[K]) {
    float pp[K], gg[K], mm[K], vv[K];
#pragma unroll
    for (int k = 0; k < K; ++k) {
        pp[k] = gg[k] = mm[k] = vv[k] = 0.f;
        if (k < KFULL || tail_ok[k]) {
            pp[k] = u.p[o[k]];
            gg[k] = u.g[o[k]];
            if (!u.ema) { mm[k] = u.m[o[k]]; vv[k] = u.v[o[k]]; }
        }
    }
#pragma unroll
    for (int k = 0; k < K; ++k) {
        if (k < KFULL || tail_ok[k]) {
            if (u.ema) {
                pp[k] = ema_elem(pp[k], gg[k], u.tau, u.omt);
                u.p[o[k]] = pp[k];
            } else {
                adam_elem(pp[k], gg[k], mm[k], vv[k], u.omb1, u.b2, u.omb2, u.bc2s, u.eps, u.nstep);
                u.p[o[k]] = pp[k]; u.m[o[k]] = mm[k]; u.v[o[k]] = vv[k];
            }
        }
        out[k] = pp[k];
    }
}

// 4 resident blocks per SM (64 registers, a few spilled words on the generic LINEAR / CONV1 paths) rather than 3
// (80 registers): more loads in flight per SM; measured on the B=256 update, 1815 vs 1808 updates/s
__global__ void __launch_bounds__(256, 4) adam_pack_kernel(const OptArgs a) {
    __shared__ __align__(16) unsigned char smraw[kOptShBytes];
    int lo = 0, hi = a.n - 1;                    // last segment whose first block is <= blockIdx.x
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if ((int)blockIdx.x >= a.first_block[mid]) lo = mid; else hi = mid - 1;
    }
    const drq_opt_seg& sg = a.s[lo];
    const int b = blockIdx.x - a.first_block[lo];
    const int tid = threadIdx.x;
    Upd u;
    u.ema = sg.ema != 0;
    if (u.ema) { u.p = a.dst + sg.off; u.g = a.src + sg.off; u.m = nullptr; u.v = nullptr; }
    else { u.p = a.p + sg.off; u.g = a.g + sg.off; u.m = a.m + sg.off; u.v = a.v + sg.off; }
    u.tau = a.tau; u.omt = a.omt;
    if (!u.ema) { u.omb1 = a.sc[0]; u.b2 = a.sc[1]; u.omb2 = a.sc[2]; u.bc2s = a.sc[3]; u.eps = a.sc[4]; u.nstep = a.sc[5]; }
    else { u.omb1 = u.b2 = u.omb2 = u.bc2s = u.eps = u.nstep = 0.f; }
    __nv_bfloat16* out = reinterpret_cast<__nv_bfloat16*>(sg.out);
    const int n = (int)sg.n;
    const bool flat = sg.kind == DRQ_OPT_PLAIN || sg.kind == DRQ_OPT_CONV || (sg.kind == DRQ_OPT_LINEAR && (sg.cols & 7) == 0);

    if (flat) {
        int i4[2]; bool ok[2]; float4 val[2];
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            i4[k] = b * (kOptTile / 4) + tid + k * 256;
            ok[k] = i4[k] * 4 < n;
        }
        upd_vec<2>(u, i4, ok, val);
        if (sg.kind == DRQ_OPT_CONV) {
            __nv_bfloat16* out2 = reinterpret_cast<__nv_bfloat16*>(sg.out2);
#pragma unroll
            for (int k = 0; k < 2; ++k) {
                if (!ok[k]) continue;
                const float vv[4] = {val[k].x, val[k].y, val[k].z, val[k].w};
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int i = i4[k] * 4 + j;
                    const int co = i / 288, ci = (i / 9) % 32, tap = i % 9;
                    const __nv_bfloat16 h = __float2bfloat16_rn(vv[j]);
                    out[((tap * 4 + ci / 8) * 32 + co) * 8 + (ci & 7)] = h;
                    out2[((tap * 4 + co / 8) * 32 + ci) * 8 + (co & 7)] = h;
                }
            }
        } else if (sg.kind == DRQ_OPT_LINEAR) {
            // cols % 8 == 0: an even/odd pair of float4 is one 8-column unit of one row
            const int units = (sg.cols + 15) / 16 * 2;
#pragma unroll
            for (int k = 0; k < 2; ++k) {
                const uint32_t w0 = tc::pack_bf16x2(val[k].x, val[k].y), w1 = tc::pack_bf16x2(val[k].z, val[k].w);
                const uint32_t w2 = __shfl_down_sync(0xffffffffu, w0, 1), w3 = __shfl_down_sync(0xffffffffu, w1, 1);
                if (ok[k] && !(tid & 1)) {
                    const int e = i4[k] * 4;
                    const int r = e / sg.cols, c = e - r * sg.cols;
                    *reinterpret_cast<uint4*>(out + tb_off(r, c >> 3, units, DRQ_TB_W)) = make_uint4(w0, w1, w2, w3);
                }
            }
        }
    } else if (sg.kind == DRQ_OPT_LINEAR) {
        __nv_bfloat16* sh = reinterpret_cast<__nv_bfloat16*>(smraw);
        const LinTile t = lin_tile(sg.cols);
        const int rb = b / t.chunks, ch = b - rb * t.chunks;
        const int r0 = rb * t.RT, c0 = ch * t.CW;
        for (int q = tid; q < t.RT * t.SW / 8; q += 256) reinterpret_cast<uint4*>(sh)[q] = make_uint4(0, 0, 0, 0);
        __syncthreads();
        const int total = t.RT * t.width;
        int o[kGenK], pos[kGenK]; bool ok[kGenK]; float val[kGenK];
#pragma unroll
        for (int k = 0; k < kGenK; ++k) {
            const int e = tid + k * 256;
            const int lr = e / t.width, cc = e - lr * t.width;
            const int r = r0 + lr, c = c0 + cc;
            ok[k] = e < total && r < sg.rows && c < sg.cols;
            o[k] = r * sg.cols + c;
            pos[k] = lr * t.SW + cc;
        }
        upd_scalar<kGenK, 0>(u, o, ok, val);
#pragma unroll
        for (int k = 0; k < kGenK; ++k)
            if (ok[k]) sh[pos[k]] = __float2bfloat16_rn(val[k]);
        __syncthreads();
        const int ul_n = (t.width + 7) / 8;
        const int units = (sg.cols + 15) / 16 * 2;
        for (int q = tid; q < t.RT * ul_n; q += 256) {
            const int lr = q & (t.RT - 1), ul = q / t.RT;
            const int r = r0 + lr;
            if (r < sg.rows && (c0 + ul * 8) < sg.cols)
                *reinterpret_cast<uint4*>(out + tb_off(r, c0 / 8 + ul, units, DRQ_TB_W)) =
                    *reinterpret_cast<const uint4*>(sh + lr * t.SW + ul * 8);
        }
    } else if (sg.kind == DRQ_OPT_TRUNK) {
        // block = (weight row r, channel unit cu, pixel fifth xt): warp w walks channel 8*cu + w, 245 pixels.  The
        // channel's pixels start at an arbitrary 4-byte offset (1225 is odd): up to 3 leading and 3 trailing values go
        // through scalar accesses of single lanes, the 60-61 aligned float4 in between two per lane.
        float (*tile)[256] = reinterpret_cast<float(*)[256]>(smraw);
        const int r = b / 20, rem = b - r * 20;
        const int cu = rem / 5, yx0 = (rem - cu * 5) * kTrunkW;
        const int w = tid >> 5, l = tid & 31;
        const int e0 = r * DRQ_REPR_DIM + (cu * 8 + w) * 1225 + yx0;      // first element (segment starts are 16-byte aligned)
        const int lead = (4 - (e0 & 3)) & 3;
        const int body4 = (kTrunkW - lead) >> 2;
        const int tail = kTrunkW - lead - 4 * body4;
        int i4[2]; bool ok4[2]; float4 v4[2];
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            ok4[k] = l + 32 * k < body4;
            i4[k] = ((e0 + lead) >> 2) + l + 32 * k;
        }
        // one scalar per lane at most: lanes 0..lead-1 the leading values, lanes 8..8+tail-1 the trailing ones
        int so[1], spix = -1; bool sok[1]; float sv[1];
        if (l < lead) spix = l;
        else if (l >= 8 && l - 8 < tail) spix = lead + 4 * body4 + (l - 8);
        sok[0] = spix >= 0;
        so[0] = e0 + (spix >= 0 ? spix : 0);
        upd_vec<2>(u, i4, ok4, v4);
        upd_scalar<1, 0>(u, so, sok, sv);
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            if (ok4[k]) {
                float* t4 = &tile[w][lead + 4 * (l + 32 * k)];
                t4[0] = v4[k].x; t4[1] = v4[k].y; t4[2] = v4[k].z; t4[3] = v4[k].w;
            }
        }
        if (sok[0]) tile[w][spix] = sv[0];
        __syncthreads();
        if (tid < kTrunkW) {
            uint32_t pk[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) pk[j] = tc::pack_bf16x2(tile[2 * j][tid], tile[2 * j + 1][tid]);
            *reinterpret_cast<uint4*>(out + tb_off(r, cu * 1225 + yx0 + tid, DRQ_REPR_DIM / 8, DRQ_TB_W)) =
                make_uint4(pk[0], pk[1], pk[2], pk[3]);
        }
    } else {   // DRQ_OPT_CONV1: weight [32][cin][3][3] then bias [32]
        float* buf = reinterpret_cast<float*>(smraw);
        const int cin = sg.rows, nw = 288 * cin;
        for (int base = 0; base < n; base += kGenTile) {
            int o[kGenK]; bool ok[kGenK]; float val[kGenK];
#pragma unroll
            for (int k = 0; k < kGenK; ++k) {
                o[k] = base + tid + k * 256;
                ok[k] = o[k] < n;
            }
            upd_scalar<kGenK, 0>(u, o, ok, val);
#pragma unroll
            for (int k = 0; k < kGenK; ++k)
                if (ok[k]) buf[o[k]] = val[k];
        }
        __syncthreads();
        pack_conv1_w_block(buf, buf + nw, out, cin, tid, reinterpret_cast<float(*)[9]>(buf + nw + 32));
    }
}

static inline bool aligned16(const void* p) { return ((uintptr_t)p & 15) == 0; }

static int blocks_for(long long n) {
    long long b = (n / 4 + 255) / 256;
    if (b < 1) b = 1;
    if (b > 148 * 8) b = 148 * 8;   // 8 CTAs of 256 threads per SM on B200
    return (int)b;
}

}  // namespace drq

using namespace drq;

extern "C" {

int drq_adam_ema_step(float* p, const float* g, float* m, float* v, int64_t n_adam,
                      const float* scalars, const float* ema_src, float* ema_dst, int64_t n_ema,
                      float tau, float one_minus_tau, void* stream) {
    DRQ_REQUIRE(n_adam >= 0 && n_ema >= 0 && n_adam + n_ema > 0, "adam_ema: empty");
    DRQ_REQUIRE(n_adam == 0 || (p && g && m && v && scalars), "adam_ema: null adam pointer");
    DRQ_REQUIRE(n_ema == 0 || (ema_src && ema_dst), "adam_ema: null ema pointer");
    DRQ_REQUIRE(n_adam == 0 || (aligned16(p) && aligned16(g) && aligned16(m) && aligned16(v)),
                "adam_ema: adam arenas must be 16-byte aligned");
    DRQ_REQUIRE(n_ema == 0 || (aligned16(ema_src) && aligned16(ema_dst)),
                "adam_ema: ema arenas must be 16-byte aligned");
    const int ab = n_adam ? blocks_for(n_adam) : 0;
    const int eb = n_ema ? blocks_for(n_ema) : 0;
    adam_ema_kernel<<<ab + eb, 256, 0, as_stream(stream)>>>(p, g, m, v, n_adam, scalars, ema_src, ema_dst, n_ema, tau,
                                                         one_minus_tau, ab);
    return check_launch("adam_ema_kernel");
}

int drq_adam_pack_step(float* p, const float* g, float* m, float* v, const float* scalars,
                       const float* ema_src, float* ema_dst, float tau, float one_minus_tau,
                       const drq_opt_seg* segs, int nsegs, void* stream) {
    DRQ_REQUIRE(segs && nsegs >= 1 && nsegs <= DRQ_OPT_MAX_SEGS, "adam_pack: 1..%d segments", DRQ_OPT_MAX_SEGS);
    OptArgs a{};
    a.n = nsegs; a.p = p; a.g = g; a.m = m; a.v = v; a.sc = scalars; a.src = ema_src; a.dst = ema_dst;
    a.tau = tau; a.omt = one_minus_tau;
    long long blocks = 0;
    for (int i = 0; i < nsegs; ++i) {
        const drq_opt_seg& sg = segs[i];
        DRQ_REQUIRE(sg.n > 0 && sg.n < (1ll << 31) && sg.off >= 0, "adam_pack: empty segment %d", i);
        if (sg.ema) DRQ_REQUIRE(ema_src && ema_dst && aligned16(ema_src) && aligned16(ema_dst), "adam_pack: segment %d needs the (16-byte aligned) ema arenas", i);
        else DRQ_REQUIRE(p && g && m && v && scalars && aligned16(p) && aligned16(g) && aligned16(m) && aligned16(v),
                         "adam_pack: segment %d needs the (16-byte aligned) adam arenas", i);
        a.s[i] = sg;
        a.first_block[i] = (int)blocks;
        DRQ_REQUIRE((sg.off & 3) == 0, "adam_pack: segment %d does not start on a 16-byte boundary", i);
        switch (sg.kind) {
        case DRQ_OPT_PLAIN:
            DRQ_REQUIRE((sg.n & 3) == 0, "adam_pack: plain segment %d must be padded to 4 floats", i);
            blocks += (sg.n + kOptTile - 1) / kOptTile;
            break;
        case DRQ_OPT_CONV:
            DRQ_REQUIRE(sg.n == 32 * 32 * 9 && sg.out && sg.out2, "adam_pack: bad conv segment %d", i);
            blocks += (sg.n + kOptTile - 1) / kOptTile;
            break;
        case DRQ_OPT_LINEAR: {
            DRQ_REQUIRE(sg.rows > 0 && sg.cols > 0 && sg.n == (int64_t)sg.rows * sg.cols && sg.out,
                        "adam_pack: bad linear segment %d", i);
            if ((sg.cols & 7) == 0) {
                blocks += (sg.n + kOptTile - 1) / kOptTile;
            } else {
                const LinTile t = lin_tile(sg.cols);
                blocks += (long long)((sg.rows + t.RT - 1) / t.RT) * t.chunks;
            }
            break;
        }
        case DRQ_OPT_TRUNK:
            DRQ_REQUIRE(sg.rows > 0 && sg.n == (int64_t)sg.rows * DRQ_REPR_DIM && sg.out, "adam_pack: bad trunk segment %d", i);
            blocks += 20ll * sg.rows;
            break;
        case DRQ_OPT_CONV1:
            DRQ_REQUIRE(sg.rows > 0 && sg.rows * 9 + 1 <= 96 && sg.n == 288ll * sg.rows + 32 && sg.out,
                        "adam_pack: bad conv1 segment %d", i);
            blocks += 1;
            break;
        default:
            DRQ_REQUIRE(false, "adam_pack: unknown kind in segment %d", i);
        }
    }
    DRQ_REQUIRE(blocks < (1ll << 31), "adam_pack: too many blocks");
    a.first_block[nsegs] = (int)blocks;
    adam_pack_kernel<<<(unsigned)blocks, 256, 0, as_stream(stream)>>>(a);
    return check_launch("adam_pack_kernel");
}

int drq_adam_step(float* p, const float* g, float* m, float* v, int64_t n, const float* scalars,
                  void* stream) {
    return drq_adam_ema_step(p, g, m, v, n, scalars, nullptr, nullptr, 0, 0.f, 0.f, stream);
}

int drq_soft_update(const float* p, float* tp, int64_t n, float tau, float one_minus_tau, void* stream) {
    return drq_adam_ema_step(nullptr, nullptr, nullptr, nullptr, 0, nullptr, p, tp, n, tau,
                             one_minus_tau, stream);
}

}  // extern "C"

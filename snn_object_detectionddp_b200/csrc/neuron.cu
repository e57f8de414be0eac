// Spiking-neuron layer kernels (HBM-bound): per-timestep BatchNorm statistics, fused
// BN-affine + LIF scan over all T steps (forward), reverse-time surrogate-gradient scan (backward)
// and the BatchNorm input-gradient pass.  Replaces the `bn -> silu` tail of the reference's
// ConvBlock (reference model.py:14-18) with `bn -> LIF` (build-defined, SURVEY.md 7.2); the SiLU
// variant is kept so the reference's own numerics can be reproduced through the same kernels.
//
// Data layout: conv outputs y are fp32 [T][P][C] (P = B*H*W pixels of one timestep, channels
// innermost = NHWC with the T*B batch folded).  Each thread owns a few consecutive channels of one
// pixel and walks the T steps with the membrane potential in registers; all global accesses are
// 128-bit and coalesced along C.
#include "common.cuh"

namespace snn {

enum { ACT_LIF = 0, ACT_SILU = 1 };

// ------------------------------------------------------------------------------------------
// per-(t, c) sum / sum-of-squares of y (train-mode BN batch statistics, one group per timestep)
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) bn_stats_kernel(const float* __restrict__ y, float* __restrict__ part /*[T][gridDim.x][2][C]*/,
                                                        int P, int C, int pix_per_block) {
    pdl_launch_dependents();
    pdl_wait();
    extern __shared__ float shs[];  // [rows][2][C] per-row partials, combined in a fixed order (deterministic)
    const int t = blockIdx.y;
    const int tpp = C >> 2;  // threads per pixel (float4 each)
    const int rows = 256 / tpp;
    const int cg = threadIdx.x % tpp, row = threadIdx.x / tpp;
    if (row < rows) {
        const int p0 = blockIdx.x * pix_per_block;
        const int p1 = min(P, p0 + pix_per_block);
        const float4* base = reinterpret_cast<const float4*>(y + (size_t)t * P * C) + cg;
        float4 s = make_float4(0.f, 0.f, 0.f, 0.f), q = s;
        int p = p0 + row;
        for (; p + 3 * rows < p1; p += 4 * rows) {  // 4 independent 128-bit loads in flight per thread
            const float4 a = __ldg(base + (size_t)p * tpp), b = __ldg(base + (size_t)(p + rows) * tpp);
            const float4 c = __ldg(base + (size_t)(p + 2 * rows) * tpp), d = __ldg(base + (size_t)(p + 3 * rows) * tpp);
            s.x += (a.x + b.x) + (c.x + d.x); s.y += (a.y + b.y) + (c.y + d.y);
            s.z += (a.z + b.z) + (c.z + d.z); s.w += (a.w + b.w) + (c.w + d.w);
            q.x += (a.x * a.x + b.x * b.x) + (c.x * c.x + d.x * d.x); q.y += (a.y * a.y + b.y * b.y) + (c.y * c.y + d.y * d.y);
            q.z += (a.z * a.z + b.z * b.z) + (c.z * c.z + d.z * d.z); q.w += (a.w * a.w + b.w * b.w) + (c.w * c.w + d.w * d.w);
        }
        for (; p < p1; p += rows) {
            const float4 v = __ldg(base + (size_t)p * tpp);
            s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
            q.x += v.x * v.x; q.y += v.y * v.y; q.z += v.z * v.z; q.w += v.w * v.w;
        }
        float4* r0 = reinterpret_cast<float4*>(shs + (size_t)row * 2 * C);
        r0[cg] = s;
        r0[tpp + cg] = q;
    }
    __syncthreads();
    float* out = part + ((size_t)t * gridDim.x + blockIdx.x) * 2 * C;
    for (int i = threadIdx.x; i < 2 * C; i += 256) {
        float a = 0.f;
        for (int r = 0; r < rows; ++r) a += shs[(size_t)r * 2 * C + i];
        out[i] = a;
    }
}

// sums[t][0|1][c] = sum over the timestep's 32-row groups of the conv epilogue's partials [group][2][C], in a FIXED order
// (32 row-lanes each walk their groups in order, then are combined in order) -> bit-reproducible statistics.
constexpr int kRL = 128;   // row-lanes per block of the partial reducer (x 8 channels = 1024 threads)
__global__ void __launch_bounds__(kRL * 8) bn_stats_from_partials_kernel(const float* __restrict__ part, double* __restrict__ sums,
                                                                          int C, int groups_per_t) {
    pdl_launch_dependents();
    pdl_wait();
    __shared__ double sh[2][kRL][8];
    const int t = blockIdx.y;
    const int cl = threadIdx.x & 7, rl = threadIdx.x >> 3;
    const int c = blockIdx.x * 8 + cl;
    double s = 0.0, q = 0.0;
    if (c < C) {
        const float* base = part + ((size_t)t * groups_per_t * 2) * C + c;
        int r = rl;
        for (; r + 3 * kRL < groups_per_t; r += 4 * kRL) {   // 4 groups (8 loads) in flight per thread
            const float* r0 = base + (size_t)r * 2 * C;
            const float* r1 = base + (size_t)(r + kRL) * 2 * C;
            const float* r2 = base + (size_t)(r + 2 * kRL) * 2 * C;
            const float* r3 = base + (size_t)(r + 3 * kRL) * 2 * C;
            const float a0 = __ldg(r0), b0 = __ldg(r0 + C), a1 = __ldg(r1), b1 = __ldg(r1 + C);
            const float a2 = __ldg(r2), b2 = __ldg(r2 + C), a3 = __ldg(r3), b3 = __ldg(r3 + C);
            s += (double)a0; q += (double)b0; s += (double)a1; q += (double)b1;
            s += (double)a2; q += (double)b2; s += (double)a3; q += (double)b3;
        }
        for (; r < groups_per_t; r += kRL) {
            const float* r0 = base + (size_t)r * 2 * C;
            s += (double)__ldg(r0); q += (double)__ldg(r0 + C);
        }
    }
    sh[0][rl][cl] = s; sh[1][rl][cl] = q;
    __syncthreads();
    if (threadIdx.x < 16) {
        const int which = threadIdx.x >> 3, cc = threadIdx.x & 7;
        double a = 0.0;
        for (int i = 0; i < kRL; ++i) a += sh[which][i][cc];
        const int co = blockIdx.x * 8 + cc;
        if (co < C) sums[((size_t)t * 2 + which) * C + co] = a;
    }
}

// Fused tail of the train-mode BatchNorm statistics: partial reduce + per-(t,c) scale/shift/mean/invstd + the T sequential
// running-stat updates + num_batches_tracked += T, ONE launch.
// Round 1 ran (C/8, T) blocks whose threads each read single floats 32 bytes apart: 12 us for 8 MB of partials, 3.5 % of HBM,
// 28 launches per step.  Now: grid (C/32 channel groups, S splits of the partial rows); a warp reads 32 consecutive channels
// (one 128-byte line) per load, 8 row-lanes per block, fp64 accumulation in a FIXED order; each block leaves its [T][2][32]
// partial in `ws`; the block that finishes LAST for a channel group (atomic ticket -- the result does not depend on which
// block that is) combines the S partials in split order and walks t = 0..T-1 for the running statistics.
// `counters`: caller-owned, zero-initialised, >= ceil(C/32) unsigned ints; left zeroed.
constexpr int kFinLanes = 8;
constexpr int kFinMaxSplit = 64;
static int bn_finalize_splits(int groups_per_t) {
    int s = groups_per_t / (2 * kFinLanes);
    return s < 1 ? 1 : (s > kFinMaxSplit ? kFinMaxSplit : s);
}
long long bn_finalize_workspace_doubles(int T, int C, int groups_per_t) {
    if (T < 1 || C < 1 || groups_per_t < 1) return 0;
    return (long long)((C + 31) / 32) * bn_finalize_splits(groups_per_t) * T * 2 * 32;
}

__global__ void __launch_bounds__(32 * kFinLanes)
bn_finalize_partials_kernel(const float* __restrict__ part, double* __restrict__ ws, double* __restrict__ sums,
                            const float* __restrict__ gamma, const float* __restrict__ beta, float* running_mean, float* running_var,
                            long long* nbt, float* __restrict__ scale, float* __restrict__ shift, float* __restrict__ mean_o,
                            float* __restrict__ invstd_o, unsigned int* counters, int T, int C, int P, int groups_per_t, int S,
                            float eps, float momentum) {
    pdl_launch_dependents();
    pdl_wait();
    __shared__ double sh[kFinLanes][2][32];
    __shared__ unsigned int s_ticket;
    const int cg = blockIdx.x, sp = blockIdx.y;
    const int cl = threadIdx.x & 31, rl = threadIdx.x >> 5;
    const int c = cg * 32 + cl;
    const int chunk = (groups_per_t + S - 1) / S;
    const int g0 = sp * chunk, g1 = min(groups_per_t, g0 + chunk);
    double* my = ws + ((size_t)(cg * S + sp) * T) * 64;
    for (int t = 0; t < T; ++t) {
        double a = 0.0, b = 0.0;
        if (c < C) {
            const float* base = part + ((size_t)t * groups_per_t * 2) * C + c;
            int r = g0 + rl;
            for (; r + 3 * kFinLanes < g1; r += 4 * kFinLanes) {      // 8 independent loads in flight per thread
                const float* p0 = base + (size_t)r * 2 * C;
                const float* p1 = p0 + (size_t)kFinLanes * 2 * C;
                const float* p2 = p1 + (size_t)kFinLanes * 2 * C;
                const float* p3 = p2 + (size_t)kFinLanes * 2 * C;
                const float a0 = __ldg(p0), b0 = __ldg(p0 + C), a1 = __ldg(p1), b1 = __ldg(p1 + C);
                const float a2 = __ldg(p2), b2 = __ldg(p2 + C), a3 = __ldg(p3), b3 = __ldg(p3 + C);
                a += (double)a0; b += (double)b0; a += (double)a1; b += (double)b1;
                a += (double)a2; b += (double)b2; a += (double)a3; b += (double)b3;
            }
            for (; r < g1; r += kFinLanes) {
                const float* p0 = base + (size_t)r * 2 * C;
                a += (double)__ldg(p0); b += (double)__ldg(p0 + C);
            }
        }
        sh[rl][0][cl] = a; sh[rl][1][cl] = b;
        __syncthreads();
        if (threadIdx.x < 64) {
            const int which = threadIdx.x >> 5;
            double tot = 0.0;
#pragma unroll
            for (int i = 0; i < kFinLanes; ++i) tot += sh[i][which][cl];
            my[(size_t)t * 64 + which * 32 + cl] = tot;
        }
        __syncthreads();
    }
    __threadfence();                               // this block's partial is visible device-wide before its ticket is drawn
    __syncthreads();
    if (threadIdx.x == 0) s_ticket = atomicAdd(&counters[cg], 1u);
    __syncthreads();
    if (s_ticket != (unsigned)(S - 1)) return;
    __threadfence();
    // last block of this channel group: combine the S partials in split order, (t, which) pairs spread over the 8 warps
    double* tot_sh = &sh[0][0][0];                 // reuse: [T*2][32] needs T <= 8 per round
    for (int t0 = 0; t0 < T; t0 += 4) {
        const int pair = t0 * 2 + rl;              // rl in 0..7 -> (t, which) = (t0 + rl/2, rl&1)
        if (pair < T * 2) {
            const int t = pair >> 1, which = pair & 1;
            double tot = 0.0;
            for (int q = 0; q < S; ++q) tot += __ldcg(ws + ((size_t)(cg * S + q) * T + t) * 64 + which * 32 + cl);
            tot_sh[rl * 32 + cl] = tot;
            if (c < C) sums[((size_t)t * 2 + which) * C + c] = tot;
        }
        __syncthreads();
        if (threadIdx.x < 32 && c < C) {
            for (int k = 0; k < 4 && t0 + k < T; ++k) {
                const int t = t0 + k;
                const double a = tot_sh[(2 * k) * 32 + cl], b = tot_sh[(2 * k + 1) * 32 + cl];
                const double md = a / P;
                double vd = b / P - md * md;
                if (vd < 0) vd = 0;
                const float m = (float)md, var = (float)vd;
                const float inv = 1.0f / sqrtf(var + eps);
                const float g = gamma ? gamma[c] : 1.f, bb = beta ? beta[c] : 0.f;
                const float sc = g * inv;
                scale[t * C + c] = sc; shift[t * C + c] = bb - m * sc;
                mean_o[t * C + c] = m; invstd_o[t * C + c] = inv;
                if (running_mean && running_var) {       // the reference calls the module once per timestep: T updates in order
                    const float unb = (P > 1) ? (float)(vd * ((double)P / (double)(P - 1))) : var;
                    running_mean[c] = (1.f - momentum) * running_mean[c] + momentum * m;
                    running_var[c] = (1.f - momentum) * running_var[c] + momentum * unb;
                }
            }
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        counters[cg] = 0u;
        if (cg == 0 && nbt) *nbt += T;
    }
}

// scale/shift per (t,c); running-stat update applied T times in order (the reference calls the
// module once per timestep, model.py:14 via train.py:64-66).
__global__ void bn_finalize_kernel(const double* __restrict__ sums, const float* __restrict__ gamma,
                                   const float* __restrict__ beta, float* running_mean, float* running_var,
                                   float* __restrict__ scale, float* __restrict__ shift, float* __restrict__ mean_o,
                                   float* __restrict__ invstd_o, int T, int C, int P, float eps, float momentum,
                                   int training) {
    pdl_launch_dependents();
    pdl_wait();
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    const float g = gamma ? gamma[c] : 1.f, b = beta ? beta[c] : 0.f;
    if (!training) {
        const float m = running_mean[c], inv = 1.0f / sqrtf(running_var[c] + eps);
        const float sc = g * inv;
        scale[c] = sc; shift[c] = b - m * sc; mean_o[c] = m; invstd_o[c] = inv;
        return;
    }
    float rm = running_mean ? running_mean[c] : 0.f, rv = running_var ? running_var[c] : 1.f;
    for (int t = 0; t < T; ++t) {
        const double s = sums[(size_t)t * 2 * C + c], q = sums[(size_t)t * 2 * C + C + c];
        const double md = s / P;
        double vd = q / P - md * md;
        if (vd < 0) vd = 0;
        const float m = (float)md, var = (float)vd;
        const float inv = 1.0f / sqrtf(var + eps);
        const float sc = g * inv;
        scale[t * C + c] = sc; shift[t * C + c] = b - m * sc;
        mean_o[t * C + c] = m; invstd_o[t * C + c] = inv;
        const float unb = (P > 1) ? (float)(vd * ((double)P / (double)(P - 1))) : var;
        rm = (1.f - momentum) * rm + momentum * m;
        rv = (1.f - momentum) * rv + momentum * unb;
    }
    if (running_mean) running_mean[c] = rm;
    if (running_var) running_var[c] = rv;
}

// ------------------------------------------------------------------------------------------
// forward: x = y*scale + shift ; LIF scan over T (or SiLU) ; 8 channels / thread
// COUNT (LIF only): also adds the number of spikes of each timestep to spikes[t] (popcount of the 8 spike bits, warp
// reduce, block reduce in shared memory, one 64-bit integer atomic per block and timestep: exact, order-independent) and
// n_per_t to steps[t] (block 0).  Out-of-range threads stay alive with no spikes so every lane reaches the warp reduce.
// The counters are trailing parameters, so the uncounted instantiations compile to the code they had without them.
// ------------------------------------------------------------------------------------------
constexpr int kCountMaxT = 64;    // timesteps one counted launch can tally (shared-memory slots)
template <int ACT, bool COUNT>
__global__ void __launch_bounds__(256) bn_act_fwd_kernel(const float* __restrict__ y, const float* __restrict__ scale,
                                                          const float* __restrict__ shift, const float* __restrict__ v_init,
                                                          __nv_bfloat16* __restrict__ out, uint8_t* __restrict__ mask,
                                                          float* __restrict__ v_final, int T, long long n8, int C,
                                                          int ss_stride_t, float beta, float theta,
                                                          unsigned long long* __restrict__ spikes,
                                                          unsigned long long* __restrict__ steps) {
    pdl_launch_dependents();
    pdl_wait();
    const long long idx = (long long)blockIdx.x * 256 + threadIdx.x;
    if constexpr (!COUNT) {
        if (idx >= n8) return;
    }
    const bool live = !COUNT || idx < n8;
    __shared__ unsigned int s_cnt[COUNT ? kCountMaxT : 1];
    if constexpr (COUNT) {
        for (int t = threadIdx.x; t < T; t += 256) s_cnt[t] = 0u;
        __syncthreads();
    }
    const int c0 = live ? (int)((idx * 8) % C) : 0;
    const size_t nt = (size_t)n8 * 8;
    float v[8];
    if (ACT == ACT_LIF && v_init && live) {
        const float4 a = __ldg(reinterpret_cast<const float4*>(v_init) + idx * 2);
        const float4 b = __ldg(reinterpret_cast<const float4*>(v_init) + idx * 2 + 1);
        v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
    } else {
#pragma unroll
        for (int i = 0; i < 8; ++i) v[i] = 0.f;
    }
#pragma unroll 4
    for (int t = 0; t < T; ++t) {
        uint32_t bits = 0;
        if (live) {
            const float4* yp = reinterpret_cast<const float4*>(y + (size_t)t * nt) + idx * 2;
            const float4 ya = __ldcs(yp), yb = __ldcs(yp + 1);
            const float4* sp = reinterpret_cast<const float4*>(scale + (size_t)t * ss_stride_t + c0);
            const float4* hp = reinterpret_cast<const float4*>(shift + (size_t)t * ss_stride_t + c0);
            const float4 sa = __ldg(sp), sb = __ldg(sp + 1), ha = __ldg(hp), hb = __ldg(hp + 1);
            float x[8];
            x[0] = __fadd_rn(__fmul_rn(ya.x, sa.x), ha.x); x[1] = __fadd_rn(__fmul_rn(ya.y, sa.y), ha.y);
            x[2] = __fadd_rn(__fmul_rn(ya.z, sa.z), ha.z); x[3] = __fadd_rn(__fmul_rn(ya.w, sa.w), ha.w);
            x[4] = __fadd_rn(__fmul_rn(yb.x, sb.x), hb.x); x[5] = __fadd_rn(__fmul_rn(yb.y, sb.y), hb.y);
            x[6] = __fadd_rn(__fmul_rn(yb.z, sb.z), hb.z); x[7] = __fadd_rn(__fmul_rn(yb.w, sb.w), hb.w);
            float o[8];
            if (ACT == ACT_LIF) {
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const float u = __fadd_rn(__fmul_rn(beta, v[i]), x[i]);
                    const bool s = u >= theta;
                    v[i] = s ? 0.f : u;
                    o[i] = s ? 1.f : 0.f;
                    bits |= (s ? 1u : 0u) << i;
                }
            } else {
#pragma unroll
                for (int i = 0; i < 8; ++i) o[i] = x[i] / (1.f + __expf(-x[i]));
            }
            uint4 pk;
            pk.x = pack_bf16x2(o[0], o[1]); pk.y = pack_bf16x2(o[2], o[3]);
            pk.z = pack_bf16x2(o[4], o[5]); pk.w = pack_bf16x2(o[6], o[7]);
            *(reinterpret_cast<uint4*>(out + (size_t)t * nt) + idx) = pk;
            if (ACT == ACT_LIF && mask) mask[(size_t)t * n8 + idx] = (uint8_t)bits;
        }
        if constexpr (COUNT) {
            const unsigned int n = __reduce_add_sync(0xffffffffu, (unsigned int)__popc(bits));
            if ((threadIdx.x & 31) == 0 && n) atomicAdd(&s_cnt[t], n);
        }
    }
    if (ACT == ACT_LIF && v_final && live) {
        float4* vp = reinterpret_cast<float4*>(v_final) + idx * 2;
        vp[0] = make_float4(v[0], v[1], v[2], v[3]);
        vp[1] = make_float4(v[4], v[5], v[6], v[7]);
    }
    if constexpr (COUNT) {
        __syncthreads();
        for (int t = threadIdx.x; t < T; t += 256) {
            if (s_cnt[t]) atomicAdd(spikes + t, (unsigned long long)s_cnt[t]);
            if (blockIdx.x == 0) atomicAdd(steps + t, (unsigned long long)(n8 * 8));
        }
    }
}

// ------------------------------------------------------------------------------------------
// backward: recompute u[t] forward in registers, then one reverse-time scan.
//   gu[t] = gs[t]*g(u[t]) + gv[t]*((1-s[t]) - u[t]*g(u[t])),  g(u) = (a/2)/(1+(pi*a/2*(u-th))^2)
//   gx[t] = gu[t] ; gv[t-1] = beta*gu[t]
// TRAIN: writes gx (fp32) and accumulates per-(t,c) sum(gx), sum(gx*xhat) for the BN backward.
// EVAL : BN statistics are constants -> writes dy = gx*scale directly as bf16.
// 4 channels / thread; a block covers `rows` pixels per iteration and loops `iters` times.
// ------------------------------------------------------------------------------------------
template <int ACT, int TMAX, bool TRAIN>
__global__ void __launch_bounds__(256)
bn_act_bwd_kernel(const float* __restrict__ y, const float* __restrict__ scale, const float* __restrict__ shift,
                  const float* __restrict__ mean, const float* __restrict__ invstd, const float* __restrict__ v_init,
                  const __nv_bfloat16* __restrict__ gs, const float* __restrict__ gv_final, float* __restrict__ gx_out,
                  __nv_bfloat16* __restrict__ dy_out, float* __restrict__ gv_init, float* __restrict__ red /*[T][2][C]*/,
                  int T, int P, int C, int ss_stride_t, int pix_per_block, float beta, float theta, float alpha) {
    pdl_launch_dependents();
    pdl_wait();
    extern __shared__ float shf[];  // TRAIN: [T][2][C]
    const int tpp = C >> 2;
    const int rows = 256 / tpp;
    const int cg = threadIdx.x % tpp, row = threadIdx.x / tpp;
    const int c0 = cg * 4;
    const size_t nt4 = (size_t)P * tpp;  // float4 per timestep
    if (TRAIN) {
        for (int i = threadIdx.x; i < T * 2 * C; i += 256) shf[i] = 0.f;
        __syncthreads();
    }
    float acc_s[TMAX][4], acc_d[TMAX][4];
    if (TRAIN) {
#pragma unroll
        for (int t = 0; t < TMAX; ++t)
#pragma unroll
            for (int i = 0; i < 4; ++i) acc_s[t][i] = acc_d[t][i] = 0.f;
    }
    const float ka = 0.5f * alpha, kz = 1.5707963267948966f * alpha;
    if (row < rows) {
        const int p0 = blockIdx.x * pix_per_block, p1 = min(P, p0 + pix_per_block);
        for (int p = p0 + row; p < p1; p += rows) {
            const size_t e4 = (size_t)p * tpp + cg;
            float u[TMAX][4], xh[TMAX][4];
            float v[4] = {0.f, 0.f, 0.f, 0.f};
            if (ACT == ACT_LIF && v_init) {
                const float4 a = __ldg(reinterpret_cast<const float4*>(v_init) + e4);
                v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w;
            }
#pragma unroll
            for (int t = 0; t < TMAX; ++t) {
                if (t < T) {
                    const float4 yy = __ldcs(reinterpret_cast<const float4*>(y) + (size_t)t * nt4 + e4);
                    const float4 sc = __ldg(reinterpret_cast<const float4*>(scale + (size_t)t * ss_stride_t + c0));
                    const float4 sh = __ldg(reinterpret_cast<const float4*>(shift + (size_t)t * ss_stride_t + c0));
                    const float yv[4] = {yy.x, yy.y, yy.z, yy.w};
                    const float scv[4] = {sc.x, sc.y, sc.z, sc.w}, shv[4] = {sh.x, sh.y, sh.z, sh.w};
                    float mv[4] = {0, 0, 0, 0}, iv[4] = {0, 0, 0, 0};
                    if (TRAIN) {
                        const float4 m = __ldg(reinterpret_cast<const float4*>(mean + (size_t)t * ss_stride_t + c0));
                        const float4 is = __ldg(reinterpret_cast<const float4*>(invstd + (size_t)t * ss_stride_t + c0));
                        mv[0] = m.x; mv[1] = m.y; mv[2] = m.z; mv[3] = m.w;
                        iv[0] = is.x; iv[1] = is.y; iv[2] = is.z; iv[3] = is.w;
                    }
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        const float x = __fadd_rn(__fmul_rn(yv[i], scv[i]), shv[i]);
                        if (TRAIN) xh[t][i] = (yv[i] - mv[i]) * iv[i];
                        if (ACT == ACT_LIF) {
                            const float uu = __fadd_rn(__fmul_rn(beta, v[i]), x);
                            u[t][i] = uu;
                            v[i] = (uu >= theta) ? 0.f : uu;
                        } else {
                            u[t][i] = x;
                        }
                    }
                }
            }
            float gv[4] = {0.f, 0.f, 0.f, 0.f};
            if (ACT == ACT_LIF && gv_final) {
                const float4 a = __ldg(reinterpret_cast<const float4*>(gv_final) + e4);
                gv[0] = a.x; gv[1] = a.y; gv[2] = a.z; gv[3] = a.w;
            }
#pragma unroll
            for (int t = TMAX - 1; t >= 0; --t) {
                if (t < T) {
                    const uint2 graw = __ldcs(reinterpret_cast<const uint2*>(gs) + (size_t)t * nt4 + e4);
                    const float g4[4] = {bf16_lo(graw.x), bf16_hi(graw.x), bf16_lo(graw.y), bf16_hi(graw.y)};
                    float gx[4];
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        const float uu = u[t][i];
                        if (ACT == ACT_LIF) {
                            const float z = kz * (uu - theta);
                            const float sg = ka / (1.f + z * z);
                            const float keep = (uu >= theta) ? 0.f : 1.f;
                            const float gu = g4[i] * sg + gv[i] * (keep - uu * sg);
                            gx[i] = gu;
                            gv[i] = beta * gu;
                        } else {
                            const float sgm = 1.f / (1.f + __expf(-uu));
                            gx[i] = g4[i] * (sgm * (1.f + uu * (1.f - sgm)));
                        }
                    }
                    if (TRAIN) {
                        *(reinterpret_cast<float4*>(gx_out) + (size_t)t * nt4 + e4) = make_float4(gx[0], gx[1], gx[2], gx[3]);
#pragma unroll
                        for (int i = 0; i < 4; ++i) {
                            acc_s[t][i] += gx[i];
                            acc_d[t][i] += gx[i] * xh[t][i];
                        }
                    } else {
                        const float4 sc = __ldg(reinterpret_cast<const float4*>(scale + (size_t)t * ss_stride_t + c0));
                        uint2 pk;
                        pk.x = pack_bf16x2(gx[0] * sc.x, gx[1] * sc.y);
                        pk.y = pack_bf16x2(gx[2] * sc.z, gx[3] * sc.w);
                        *(reinterpret_cast<uint2*>(dy_out) + (size_t)t * nt4 + e4) = pk;
                    }
                }
            }
            if (ACT == ACT_LIF && gv_init)
                *(reinterpret_cast<float4*>(gv_init) + e4) = make_float4(gv[0], gv[1], gv[2], gv[3]);
        }
        if (TRAIN) {
#pragma unroll
            for (int t = 0; t < TMAX; ++t) {
                if (t < T) {
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        atomicAdd(&shf[(t * 2 + 0) * C + c0 + i], acc_s[t][i]);
                        atomicAdd(&shf[(t * 2 + 1) * C + c0 + i], acc_d[t][i]);
                    }
                }
            }
        }
    }
    if (TRAIN) {
        __syncthreads();
        for (int i = threadIdx.x; i < T * 2 * C; i += 256) atomicAdd(&red[i], shf[i]);
    }
}

// dgamma/dbeta (+=) and the two per-(t,c) coefficients of the BN input gradient
__global__ void bn_bwd_finalize_kernel(const float* __restrict__ red, const float* __restrict__ scale,
                                       float* __restrict__ coef /*[T][2][C]*/, float* dgamma, float* dbeta,
                                       const float* __restrict__ gamma, int T, int C, int P) {
    pdl_launch_dependents();
    pdl_wait();
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    float dg = 0.f, db = 0.f;
    const float invP = 1.f / (float)P;
    for (int t = 0; t < T; ++t) {
        const float s = red[(t * 2 + 0) * C + c], d = red[(t * 2 + 1) * C + c];
        coef[(t * 2 + 0) * C + c] = s * invP;
        coef[(t * 2 + 1) * C + c] = d * invP;
        db += s; dg += d;
    }
    if (dgamma) dgamma[c] += dg;
    if (dbeta) dbeta[c] += db;
}

// dy = scale * (gx - mean(gx) - xhat * mean(gx*xhat))  -> bf16 (operand of dgrad / wgrad)
__global__ void __launch_bounds__(256)
bn_bwd_dx_kernel(const float* __restrict__ gx, const float* __restrict__ y, const float* __restrict__ scale,
                 const float* __restrict__ mean, const float* __restrict__ invstd, const float* __restrict__ coef,
                 __nv_bfloat16* __restrict__ dy, int T, long long n4, int C) {
    pdl_launch_dependents();
    pdl_wait();
    const long long idx = (long long)blockIdx.x * 256 + threadIdx.x;
    if (idx >= n4) return;
    const int t = blockIdx.y;
    const int c0 = (int)((idx * 4) % C);
    const size_t e = (size_t)t * n4 + idx;
    const float4 g = __ldcs(reinterpret_cast<const float4*>(gx) + e);
    const float4 yy = __ldcs(reinterpret_cast<const float4*>(y) + e);
    const float4 sc = __ldg(reinterpret_cast<const float4*>(scale + t * C + c0));
    const float4 m = __ldg(reinterpret_cast<const float4*>(mean + t * C + c0));
    const float4 is = __ldg(reinterpret_cast<const float4*>(invstd + t * C + c0));
    const float4 k1 = __ldg(reinterpret_cast<const float4*>(coef + (t * 2 + 0) * C + c0));
    const float4 k2 = __ldg(reinterpret_cast<const float4*>(coef + (t * 2 + 1) * C + c0));
    uint2 pk;
    pk.x = pack_bf16x2(sc.x * (g.x - k1.x - (yy.x - m.x) * is.x * k2.x), sc.y * (g.y - k1.y - (yy.y - m.y) * is.y * k2.y));
    pk.y = pack_bf16x2(sc.z * (g.z - k1.z - (yy.z - m.z) * is.z * k2.z), sc.w * (g.w - k1.w - (yy.w - m.w) * is.w * k2.w));
    *(reinterpret_cast<uint2*>(dy) + e) = pk;
}

// ------------------------------------------------------------------------------------------
// backward, train mode, RECOMPUTE variant (2 passes over y and gs, nothing but dy is written):
//   pass 1 (REDUCE): red[t][0][c] = sum gx, red[t][1][c] = sum gx*xhat          reads 4 (y) + 2 (gs) B / neuron-step
//   pass 2 (DX)    : dy = scale*(gx - mean(gx) - xhat*mean(gx*xhat)) as bf16    reads 6, writes 2 B / neuron-step
// gx (the surrogate-gradient scan) is recomputed in registers in both passes instead of being stored as fp32 and
// re-read (the 3-kernel path above moves 10 + 10 B).  A block owns a channel range [c_base, c_base + Cb) and a pixel
// range; a thread owns ONE CHANNEL PAIR of one pixel per iteration and does all arithmetic with the packed
// fp32x2 instructions of sm_100 (FADD2 / FMUL2 / FFMA2: one issue slot per pair) -- the v1 scalar kernel was
// issue-bound at 44 warp-instructions per neuron-step (profiles/r1).  Per-(t, channel pair) coefficients are float4
// rows in shared memory.
//   x = y*scale + shift (same two roundings as the forward kernel -> identical spikes);
//   xhat*k2*scale = (x - beta_bn)*k2, so pass 2 needs only {scale, shift, -scale*k1, -k2} per (t,c) and beta_bn per c.
// ------------------------------------------------------------------------------------------
SNN_DEVINL float2 f2(float a, float b) { return make_float2(a, b); }
SNN_DEVINL float rcp_approx(float x) {
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}
SNN_DEVINL float ex2_approx(float x) {
    float r;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}

// EXACT: T == TMAX is a compile-time constant (no per-step guards; T = 1, 4, 8, 16 are the shapes on the path).
// Coefficient tables are [channel pair][t] float4 rows with an odd row pitch of (TMAX|1) entries: a thread's T
// entries sit at compile-time offsets from one base address and LDS.128 quarter-warps are bank-conflict free.
template <int ACT, int TMAX, bool REDUCE, bool EXACT>
__global__ void __launch_bounds__(256, (TMAX <= 4 ? 4 : (TMAX <= 8 ? 2 : 1)))
bn_act_bwd2_kernel(const float* __restrict__ y, const float* __restrict__ scale, const float* __restrict__ shift,
                   const float* __restrict__ mean, const float* __restrict__ invstd, const float* __restrict__ beta_bn,
                   const float* __restrict__ red_in, const float* __restrict__ v_init, const __nv_bfloat16* __restrict__ gs,
                   const float* __restrict__ gv_final, __nv_bfloat16* __restrict__ dy_out, float* __restrict__ gv_init,
                   float* __restrict__ red_out, float* dgamma, float* dbeta, int T_rt, int P, int C, int Cb, int pix_per_block,
                   float beta, float theta, float alpha, float invP,
                   float* __restrict__ part /* REDUCE, deterministic mode: [gridDim.x][T*2*C] block partials, else null */) {
    pdl_launch_dependents();
    pdl_wait();
    extern __shared__ float4 shc4[];
    constexpr int PITCH = TMAX | 1;
    const int T = EXACT ? TMAX : T_rt;
    const int c_base = blockIdx.y * Cb;
    const int tpp = Cb >> 1;         // threads (channel pairs) per pixel
    const int rows = 256 / tpp;
    const int cg = threadIdx.x % tpp, row = threadIdx.x / tpp;
    float4* tabA = shc4;                                           // [tpp][PITCH] {scale.xy, shift.xy}
    float4* tabB = shc4 + tpp * PITCH;                             // REDUCE: {-mean.xy, 0, 0} ; DX: {-scale*mean(gx).xy, -mean(gx*xhat)*invstd.xy}
    float* accum = reinterpret_cast<float*>(tabB + tpp * PITCH);   // REDUCE: [T][2][Cb]
    for (int i = threadIdx.x; i < T * tpp; i += 256) {
        const int t = i / tpp, j = i % tpp, gc = t * C + c_base + 2 * j;
        const float2 sc = *reinterpret_cast<const float2*>(scale + gc), sh = *reinterpret_cast<const float2*>(shift + gc);
        tabA[j * PITCH + t] = make_float4(sc.x, sc.y, sh.x, sh.y);
        if (REDUCE) {
            const float2 m = *reinterpret_cast<const float2*>(mean + gc);
            tabB[j * PITCH + t] = make_float4(-m.x, -m.y, 0.f, 0.f);
        } else {
            const float2 r0 = *reinterpret_cast<const float2*>(red_in + (t * 2 + 0) * C + c_base + 2 * j);
            const float2 r1 = *reinterpret_cast<const float2*>(red_in + (t * 2 + 1) * C + c_base + 2 * j);
            const float2 is = *reinterpret_cast<const float2*>(invstd + gc);
            tabB[j * PITCH + t] = make_float4(-(sc.x * (r0.x * invP)), -(sc.y * (r0.y * invP)), -(r1.x * invP * is.x), -(r1.y * invP * is.y));
        }
    }
    if (REDUCE) {
        for (int i = threadIdx.x; i < T * 2 * Cb; i += 256) accum[i] = 0.f;
    } else if (blockIdx.x == 0) {
        // parameter gradients of the BN affine: dgamma += sum_t red1, dbeta += sum_t red0 (one block per channel range)
        for (int c = threadIdx.x; c < Cb; c += 256) {
            float dg = 0.f, db = 0.f;
            for (int t = 0; t < T; ++t) { db += red_in[(t * 2 + 0) * C + c_base + c]; dg += red_in[(t * 2 + 1) * C + c_base + c]; }
            if (dgamma) dgamma[c_base + c] += dg;
            if (dbeta) dbeta[c_base + c] += db;
        }
    }
    __syncthreads();
    const float ka = 0.5f * alpha, kz = 1.5707963267948966f * alpha;
    const float2 kz2 = f2(kz, kz), nkzth2 = f2(-kz * theta, -kz * theta), one2 = f2(1.f, 1.f), ka2 = f2(ka, ka), beta2 = f2(beta, beta);
    const int C2 = C >> 1;
    const size_t nt2 = (size_t)P * C2;        // channel pairs per timestep
    float2 acc_s[TMAX], acc_d[TMAX];
    if (REDUCE) {
#pragma unroll
        for (int t = 0; t < TMAX; ++t) acc_s[t] = acc_d[t] = f2(0.f, 0.f);
    }
    if (row < rows) {
        float2 nbb = f2(0.f, 0.f);
        if (!REDUCE && beta_bn) {
            const float2 b = *reinterpret_cast<const float2*>(beta_bn + c_base + 2 * cg);
            nbb = f2(-b.x, -b.y);
        }
        const float4* tA = tabA + cg * PITCH;
        const float4* tB = tabB + cg * PITCH;
        // pass 2 walks the pixel ranges in the REVERSE order of pass 1: the tail pass 1 read last is still in L2 (LRU)
        const int xb = REDUCE ? (int)blockIdx.x : (int)(gridDim.x - 1 - blockIdx.x);
        const int p0 = xb * pix_per_block, p1 = min(P, p0 + pix_per_block);
        size_t e2 = (size_t)(p0 + row) * C2 + (c_base >> 1) + cg;
        const size_t e2_step = (size_t)rows * C2;
        for (int p = p0 + row; p < p1; p += rows, e2 += e2_step) {
            float2 yv[TMAX];      // REDUCE: y ; DX: overwritten with x = y*scale + shift
            uint32_t gr[TMAX];
            {
                // pass 1 leaves y / gs in L2 for pass 2 (tensors up to ~80 MB fit the 126 MB L2); pass 2 streams
                const float2* yp = reinterpret_cast<const float2*>(y) + e2;
                const uint32_t* gp = reinterpret_cast<const uint32_t*>(gs) + e2;
#pragma unroll
                for (int t = 0; t < TMAX; ++t) {
                    if (EXACT || t < T) {
                        yv[t] = REDUCE ? __ldg(yp) : __ldcs(yp);
                        gr[t] = REDUCE ? __ldg(gp) : __ldcs(gp);
                        yp += nt2; gp += nt2;
                    }
                }
            }
            float2 v = f2(0.f, 0.f);
            if (ACT == ACT_LIF && v_init) v = __ldg(reinterpret_cast<const float2*>(v_init) + e2);
            float2 u[TMAX];       // LIF: membrane before reset ; SiLU: x
#pragma unroll
            for (int t = 0; t < TMAX; ++t) {
                if (EXACT || t < T) {
                    const float4 a = tA[t];
                    // ptxas contracts mul.rn.f32x2 + add.rn.f32x2 into one FFMA2 (even with -fmad=false), which would
                    // break the two-rounding contract shared with the forward kernel: packed multiply, scalar adds
                    const float2 xm = __fmul2_rn(yv[t], f2(a.x, a.y));
                    const float2 x = f2(__fadd_rn(xm.x, a.z), __fadd_rn(xm.y, a.w));
                    if (!REDUCE) yv[t] = x;
                    if (ACT == ACT_LIF) {
                        const float2 um = __fmul2_rn(beta2, v);
                        const float2 uu = f2(__fadd_rn(um.x, x.x), __fadd_rn(um.y, x.y));
                        u[t] = uu;
                        v.x = (uu.x >= theta) ? 0.f : uu.x;
                        v.y = (uu.y >= theta) ? 0.f : uu.y;
                    } else {
                        u[t] = x;
                    }
                }
            }
            float2 gv = f2(0.f, 0.f);
            if (ACT == ACT_LIF && gv_final) gv = __ldg(reinterpret_cast<const float2*>(gv_final) + e2);
            uint32_t* dp = reinterpret_cast<uint32_t*>(dy_out) + e2 + (size_t)(T - 1) * nt2;
#pragma unroll
            for (int t = TMAX - 1; t >= 0; --t) {
                if (EXACT || t < T) {
                    const float2 g = f2(bf16_lo(gr[t]), bf16_hi(gr[t]));
                    const float2 uu = u[t];
                    float2 gx;
                    if (ACT == ACT_LIF) {
                        const float2 z = __ffma2_rn(kz2, uu, nkzth2);                 // kz * (u - theta)
                        const float2 den = __ffma2_rn(z, z, one2);
                        const float2 sg = __fmul2_rn(ka2, f2(rcp_approx(den.x), rcp_approx(den.y)));
                        const float2 keep = f2((uu.x >= theta) ? 0.f : 1.f, (uu.y >= theta) ? 0.f : 1.f);
                        const float2 w = __ffma2_rn(f2(-uu.x, -uu.y), sg, keep);     // d v[t] / d u[t]
                        gx = __ffma2_rn(g, sg, __fmul2_rn(gv, w));
                        gv = __fmul2_rn(beta2, gx);
                    } else {
                        const float2 e = f2(ex2_approx(-1.4426950408889634f * uu.x), ex2_approx(-1.4426950408889634f * uu.y));
                        const float2 d1 = __fadd2_rn(e, one2);
                        const float2 sgm = f2(rcp_approx(d1.x), rcp_approx(d1.y));
                        const float2 oms = __fadd2_rn(one2, f2(-sgm.x, -sgm.y));
                        gx = __fmul2_rn(g, __fmul2_rn(sgm, __ffma2_rn(uu, oms, one2)));
                    }
                    const float4 k = tB[t];
                    if (REDUCE) {
                        acc_s[t] = __fadd2_rn(acc_s[t], gx);
                        acc_d[t] = __ffma2_rn(gx, __fadd2_rn(yv[t], f2(k.x, k.y)), acc_d[t]);
                    } else {
                        const float4 a = tA[t];
                        const float2 t1 = __ffma2_rn(f2(a.x, a.y), gx, f2(k.x, k.y));
                        const float2 d = __ffma2_rn(__fadd2_rn(yv[t], nbb), f2(k.z, k.w), t1);
                        *dp = pack_bf16x2(d.x, d.y);
                        dp -= nt2;
                    }
                }
            }
            if (!REDUCE && ACT == ACT_LIF && gv_init) *(reinterpret_cast<float2*>(gv_init) + e2) = gv;
        }
        if (REDUCE) {
            const int cl = cg * 2;
            float* slot = accum + (size_t)(1 + row) * T * 2 * Cb;       // deterministic mode: this row's own copy of accum[]
#pragma unroll
            for (int t = 0; t < TMAX; ++t) {
                if (EXACT || t < T) {
                    if (part) {
                        slot[(t * 2 + 0) * Cb + cl] = acc_s[t].x; slot[(t * 2 + 0) * Cb + cl + 1] = acc_s[t].y;
                        slot[(t * 2 + 1) * Cb + cl] = acc_d[t].x; slot[(t * 2 + 1) * Cb + cl + 1] = acc_d[t].y;
                    } else {
                        atomicAdd(&accum[(t * 2 + 0) * Cb + cl], acc_s[t].x); atomicAdd(&accum[(t * 2 + 0) * Cb + cl + 1], acc_s[t].y);
                        atomicAdd(&accum[(t * 2 + 1) * Cb + cl], acc_d[t].x); atomicAdd(&accum[(t * 2 + 1) * Cb + cl + 1], acc_d[t].y);
                    }
                }
            }
        }
    }
    if (REDUCE) {
        __syncthreads();
        if (part) {          // rows in row order -> block partial -> this block's row of the scratch buffer
            for (int i = threadIdx.x; i < T * 2 * Cb; i += 256) {
                float a = 0.f;
                for (int r = 0; r < rows; ++r) a += accum[(size_t)(1 + r) * T * 2 * Cb + i];
                accum[i] = a;
            }
            __syncthreads();
        }
        for (int i = threadIdx.x; i < T * Cb; i += 256) {
            const int t = i / Cb, c = i % Cb;
            const float v0 = accum[(t * 2 + 0) * Cb + c];
            const float v1 = accum[(t * 2 + 1) * Cb + c] * invstd[t * C + c_base + c];      // sum gx*(y - mean) -> sum gx*xhat
            if (part) {
                part[(size_t)blockIdx.x * T * 2 * C + (t * 2 + 0) * C + c_base + c] = v0;
                part[(size_t)blockIdx.x * T * 2 * C + (t * 2 + 1) * C + c_base + c] = v1;
            } else {
                atomicAdd(&red_out[(t * 2 + 0) * C + c_base + c], v0);
                atomicAdd(&red_out[(t * 2 + 1) * C + c_base + c], v1);
            }
        }
    }
}

// ------------------------------------------------------------------------------------------
// T == 16.  The one-chunk kernel above holds 16 steps of y, gs and u plus 4 x 16 accumulators per thread: 186 (reduce) / 165
// (dx) registers -> one 256-thread block per SM and 3.6 / 4.0 TB/s (profiles/r2, LIF sweep).  Here a thread walks its 16
// steps as TWO CHUNKS of 8: a forward-only scan of steps 0..7 yields the membrane entering t = 8; chunk 1 (t = 8..15) is
// recomputed and scanned backward; then chunk 0 from v_init (its y read a second time: an L1/L2 hit, no DRAM traffic), the
// surrogate state gv carried across the chunk boundary.  Per-step arithmetic is the same instruction sequence as above,
// so spikes, gx and dy are the same bits; live state per thread halves -> two blocks per SM, each with 8-step loads in flight.
// ------------------------------------------------------------------------------------------
struct Bwd2Consts {
    float2 kz2, nkzth2, one2, ka2, beta2;
    float theta;
};

template <int ACT, bool REDUCE, int T0>
SNN_DEVINL void bwd2_chunk8(const float2* __restrict__ yp, const uint32_t* __restrict__ gp, uint32_t* __restrict__ dp, size_t nt2,
                            const float4* tA, const float4* tB, float2 v, float2& gv, float2 nbb, const Bwd2Consts& k,
                            float4* acc /* REDUCE: this thread's [16] accumulator slots in shared memory, stride 256 */) {
    constexpr int TC = 8;
    float2 yv[TC];
    uint32_t gr[TC];
    yp += (size_t)T0 * nt2;           // running pointers: per-step 64-bit offsets would cost 3 x 16 registers
    gp += (size_t)T0 * nt2;
    dp += (size_t)(T0 + TC - 1) * nt2;
#pragma unroll
    for (int t = 0; t < TC; ++t) {
        yv[t] = REDUCE ? __ldg(yp) : __ldcs(yp);
        gr[t] = REDUCE ? __ldg(gp) : __ldcs(gp);
        yp += nt2; gp += nt2;
    }
    float2 u[TC];
#pragma unroll
    for (int t = 0; t < TC; ++t) {
        const float4 a = tA[T0 + t];
        const float2 xm = __fmul2_rn(yv[t], f2(a.x, a.y));
        const float2 x = f2(__fadd_rn(xm.x, a.z), __fadd_rn(xm.y, a.w));
        if (!REDUCE) yv[t] = x;
        if (ACT == ACT_LIF) {
            const float2 um = __fmul2_rn(k.beta2, v);
            const float2 uu = f2(__fadd_rn(um.x, x.x), __fadd_rn(um.y, x.y));
            u[t] = uu;
            v.x = (uu.x >= k.theta) ? 0.f : uu.x;
            v.y = (uu.y >= k.theta) ? 0.f : uu.y;
        } else {
            u[t] = x;
        }
    }
#pragma unroll
    for (int t = TC - 1; t >= 0; --t) {
        const float2 g = f2(bf16_lo(gr[t]), bf16_hi(gr[t]));
        const float2 uu = u[t];
        float2 gx;
        if (ACT == ACT_LIF) {
            const float2 z = __ffma2_rn(k.kz2, uu, k.nkzth2);
            const float2 den = __ffma2_rn(z, z, k.one2);
            const float2 sg = __fmul2_rn(k.ka2, f2(rcp_approx(den.x), rcp_approx(den.y)));
            const float2 keep = f2((uu.x >= k.theta) ? 0.f : 1.f, (uu.y >= k.theta) ? 0.f : 1.f);
            const float2 w = __ffma2_rn(f2(-uu.x, -uu.y), sg, keep);
            gx = __ffma2_rn(g, sg, __fmul2_rn(gv, w));
            gv = __fmul2_rn(k.beta2, gx);
        } else {
            const float2 e = f2(ex2_approx(-1.4426950408889634f * uu.x), ex2_approx(-1.4426950408889634f * uu.y));
            const float2 d1 = __fadd2_rn(e, k.one2);
            const float2 sgm = f2(rcp_approx(d1.x), rcp_approx(d1.y));
            const float2 oms = __fadd2_rn(k.one2, f2(-sgm.x, -sgm.y));
            gx = __fmul2_rn(g, __fmul2_rn(sgm, __ffma2_rn(uu, oms, k.one2)));
        }
        const float4 kb = tB[T0 + t];
        if (REDUCE) {
            float4 a4 = acc[(T0 + t) * 256];
            const float2 s2 = __fadd2_rn(f2(a4.x, a4.y), gx);
            const float2 d2 = __ffma2_rn(gx, __fadd2_rn(yv[t], f2(kb.x, kb.y)), f2(a4.z, a4.w));
            acc[(T0 + t) * 256] = make_float4(s2.x, s2.y, d2.x, d2.y);
        } else {
            const float4 a = tA[T0 + t];
            const float2 t1 = __ffma2_rn(f2(a.x, a.y), gx, f2(kb.x, kb.y));
            const float2 d = __ffma2_rn(__fadd2_rn(yv[t], nbb), f2(kb.z, kb.w), t1);
            *dp = pack_bf16x2(d.x, d.y);
            dp -= nt2;
        }
    }
}

template <int ACT, bool REDUCE>
__global__ void __launch_bounds__(256, 2)
bn_act_bwd2_t16_kernel(const float* __restrict__ y, const float* __restrict__ scale, const float* __restrict__ shift,
                       const float* __restrict__ mean, const float* __restrict__ invstd, const float* __restrict__ beta_bn,
                       const float* __restrict__ red_in, const float* __restrict__ v_init, const __nv_bfloat16* __restrict__ gs,
                       const float* __restrict__ gv_final, __nv_bfloat16* __restrict__ dy_out, float* __restrict__ gv_init,
                       float* __restrict__ red_out, float* dgamma, float* dbeta, int T_rt, int P, int C, int Cb, int pix_per_block,
                       float beta, float theta, float alpha, float invP, float* __restrict__ part /* as in bn_act_bwd2_kernel */) {
    pdl_launch_dependents();
    pdl_wait();
    extern __shared__ float4 shc4[];
    constexpr int T = 16, PITCH = T | 1;
    const int c_base = blockIdx.y * Cb;
    const int tpp = Cb >> 1;
    const int rows = 256 / tpp;
    const int cg = threadIdx.x % tpp, row = threadIdx.x / tpp;
    float4* tabA = shc4;
    float4* tabB = shc4 + tpp * PITCH;
    float* accum = reinterpret_cast<float*>(tabB + tpp * PITCH);
    for (int i = threadIdx.x; i < T * tpp; i += 256) {
        const int t = i / tpp, j = i % tpp, gc = t * C + c_base + 2 * j;
        const float2 sc = *reinterpret_cast<const float2*>(scale + gc), sh = *reinterpret_cast<const float2*>(shift + gc);
        tabA[j * PITCH + t] = make_float4(sc.x, sc.y, sh.x, sh.y);
        if (REDUCE) {
            const float2 m = *reinterpret_cast<const float2*>(mean + gc);
            tabB[j * PITCH + t] = make_float4(-m.x, -m.y, 0.f, 0.f);
        } else {
            const float2 r0 = *reinterpret_cast<const float2*>(red_in + (t * 2 + 0) * C + c_base + 2 * j);
            const float2 r1 = *reinterpret_cast<const float2*>(red_in + (t * 2 + 1) * C + c_base + 2 * j);
            const float2 is = *reinterpret_cast<const float2*>(invstd + gc);
            tabB[j * PITCH + t] = make_float4(-(sc.x * (r0.x * invP)), -(sc.y * (r0.y * invP)), -(r1.x * invP * is.x), -(r1.y * invP * is.y));
        }
    }
    if (REDUCE) {
        for (int i = threadIdx.x; i < T * 2 * Cb; i += 256) accum[i] = 0.f;
    } else if (blockIdx.x == 0) {
        for (int c = threadIdx.x; c < Cb; c += 256) {
            float dg = 0.f, db = 0.f;
            for (int t = 0; t < T; ++t) { db += red_in[(t * 2 + 0) * C + c_base + c]; dg += red_in[(t * 2 + 1) * C + c_base + c]; }
            if (dgamma) dgamma[c_base + c] += dg;
            if (dbeta) dbeta[c_base + c] += db;
        }
    }
    __syncthreads();
    const float ka = 0.5f * alpha, kz = 1.5707963267948966f * alpha;
    Bwd2Consts k;
    k.kz2 = f2(kz, kz); k.nkzth2 = f2(-kz * theta, -kz * theta); k.one2 = f2(1.f, 1.f); k.ka2 = f2(ka, ka); k.beta2 = f2(beta, beta);
    k.theta = theta;
    const int C2 = C >> 1;
    const size_t nt2 = (size_t)P * C2;
    // REDUCE: the 4 x 16 running sums of a thread live in its own float4 slots of shared memory ([t][thread]: conflict-free
    // LDS.128 / STS.128), not in 64 registers
    float4* acc = reinterpret_cast<float4*>(accum + (size_t)T * 2 * Cb) + threadIdx.x;
    if (REDUCE) {
#pragma unroll
        for (int t = 0; t < 16; ++t) acc[t * 256] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
    if (row < rows) {
        float2 nbb = f2(0.f, 0.f);
        if (!REDUCE && beta_bn) {
            const float2 b = *reinterpret_cast<const float2*>(beta_bn + c_base + 2 * cg);
            nbb = f2(-b.x, -b.y);
        }
        const float4* tA = tabA + cg * PITCH;
        const float4* tB = tabB + cg * PITCH;
        const int xb = REDUCE ? (int)blockIdx.x : (int)(gridDim.x - 1 - blockIdx.x);
        const int p0 = xb * pix_per_block, p1 = min(P, p0 + pix_per_block);
        size_t e2 = (size_t)(p0 + row) * C2 + (c_base >> 1) + cg;
        const size_t e2_step = (size_t)rows * C2;
        for (int p = p0 + row; p < p1; p += rows, e2 += e2_step) {
            const float2* yp = reinterpret_cast<const float2*>(y) + e2;
            const uint32_t* gp = reinterpret_cast<const uint32_t*>(gs) + e2;
            uint32_t* dp = reinterpret_cast<uint32_t*>(dy_out) + e2;
            float2 v0 = f2(0.f, 0.f);
            if (ACT == ACT_LIF && v_init) v0 = __ldg(reinterpret_cast<const float2*>(v_init) + e2);
            float2 v8 = v0;
            if (ACT == ACT_LIF) {
                // forward only over t = 0..7: the membrane entering chunk 1 (default caching: chunk 0 reads these again)
                float2 y0[8];
#pragma unroll
                { const float2* q = yp; for (int t = 0; t < 8; ++t) { y0[t] = __ldg(q); q += nt2; } }
#pragma unroll
                for (int t = 0; t < 8; ++t) {
                    const float4 a = tA[t];
                    const float2 xm = __fmul2_rn(y0[t], f2(a.x, a.y));
                    const float2 x = f2(__fadd_rn(xm.x, a.z), __fadd_rn(xm.y, a.w));
                    const float2 um = __fmul2_rn(k.beta2, v8);
                    const float2 uu = f2(__fadd_rn(um.x, x.x), __fadd_rn(um.y, x.y));
                    v8.x = (uu.x >= theta) ? 0.f : uu.x;
                    v8.y = (uu.y >= theta) ? 0.f : uu.y;
                }
            }
            float2 gv = f2(0.f, 0.f);
            if (ACT == ACT_LIF && gv_final) gv = __ldg(reinterpret_cast<const float2*>(gv_final) + e2);
            bwd2_chunk8<ACT, REDUCE, 8>(yp, gp, dp, nt2, tA, tB, v8, gv, nbb, k, acc);
            bwd2_chunk8<ACT, REDUCE, 0>(yp, gp, dp, nt2, tA, tB, v0, gv, nbb, k, acc);
            if (!REDUCE && ACT == ACT_LIF && gv_init) *(reinterpret_cast<float2*>(gv_init) + e2) = gv;
        }
        if (REDUCE && !part) {
            const int cl = cg * 2;
#pragma unroll
            for (int t = 0; t < 16; ++t) {
                const float4 a4 = acc[t * 256];
                atomicAdd(&accum[(t * 2 + 0) * Cb + cl], a4.x); atomicAdd(&accum[(t * 2 + 0) * Cb + cl + 1], a4.y);
                atomicAdd(&accum[(t * 2 + 1) * Cb + cl], a4.z); atomicAdd(&accum[(t * 2 + 1) * Cb + cl + 1], a4.w);
            }
        }
    }
    if (REDUCE) {
        __syncthreads();
        if (part) {          // deterministic mode: the per-thread slots summed in row order
            const float* slots = accum + (size_t)T * 2 * Cb;           // float4 [16][256] = {s.x, s.y, d.x, d.y} of thread (row, cg)
            for (int i = threadIdx.x; i < T * 2 * Cb; i += 256) {
                const int t = i / (2 * Cb), h = (i / Cb) & 1, c = i % Cb;
                float a = 0.f;
                for (int r = 0; r < rows; ++r) a += slots[((size_t)t * 256 + r * tpp + (c >> 1)) * 4 + h * 2 + (c & 1)];
                accum[i] = a;
            }
            __syncthreads();
        }
        for (int i = threadIdx.x; i < T * Cb; i += 256) {
            const int t = i / Cb, c = i % Cb;
            const float v0 = accum[(t * 2 + 0) * Cb + c];
            const float v1 = accum[(t * 2 + 1) * Cb + c] * invstd[t * C + c_base + c];
            if (part) {
                part[(size_t)blockIdx.x * T * 2 * C + (t * 2 + 0) * C + c_base + c] = v0;
                part[(size_t)blockIdx.x * T * 2 * C + (t * 2 + 1) * C + c_base + c] = v1;
            } else {
                atomicAdd(&red_out[(t * 2 + 0) * C + c_base + c], v0);
                atomicAdd(&red_out[(t * 2 + 1) * C + c_base + c], v1);
            }
        }
    }
}

// ------------------------------------------------------------------------------------------
// T == 1 SiLU layers (Detect head: only the last frame carries gradient): no scan, so the generic kernel would keep a
// single 12-byte operand pair in flight per thread (1.4 TB/s measured).  Same two passes, four pixels per thread and
// iteration.  Arithmetic identical to bn_act_bwd2_kernel<ACT_SILU, 1, ...>.
// ------------------------------------------------------------------------------------------
template <bool REDUCE>
__global__ void __launch_bounds__(256, 4)
silu_t1_bwd2_kernel(const float* __restrict__ y, const float* __restrict__ scale, const float* __restrict__ shift,
                    const float* __restrict__ mean, const float* __restrict__ invstd, const float* __restrict__ beta_bn,
                    const float* __restrict__ red_in, const __nv_bfloat16* __restrict__ gs, __nv_bfloat16* __restrict__ dy_out,
                    float* __restrict__ red_out, float* dgamma, float* dbeta, int P, int C, int Cb, int pix_per_block, float invP,
                    float* __restrict__ part /* REDUCE, deterministic mode: [gridDim.x][2*C] block partials, else null */) {
    pdl_launch_dependents();
    pdl_wait();
    extern __shared__ float4 sht[];
    constexpr int PU = 4;
    const int c_base = blockIdx.y * Cb;
    const int tpp = Cb >> 1, rows = 256 / tpp;
    const int cg = threadIdx.x % tpp, row = threadIdx.x / tpp;
    float4* tabA = sht;                                            // {scale.xy, shift.xy}
    float4* tabB = sht + tpp;                                      // REDUCE {-mean.xy,0,0} ; DX {-scale*mean(gx).xy, -mean(gx*xhat)*invstd.xy}
    float* accum = reinterpret_cast<float*>(tabB + tpp);           // REDUCE [2][Cb]
    for (int j = threadIdx.x; j < tpp; j += 256) {
        const int gc = c_base + 2 * j;
        const float2 sc = *reinterpret_cast<const float2*>(scale + gc), sh = *reinterpret_cast<const float2*>(shift + gc);
        tabA[j] = make_float4(sc.x, sc.y, sh.x, sh.y);
        if (REDUCE) {
            const float2 m = *reinterpret_cast<const float2*>(mean + gc);
            tabB[j] = make_float4(-m.x, -m.y, 0.f, 0.f);
        } else {
            const float2 r0 = *reinterpret_cast<const float2*>(red_in + gc), r1 = *reinterpret_cast<const float2*>(red_in + C + gc);
            const float2 is = *reinterpret_cast<const float2*>(invstd + gc);
            tabB[j] = make_float4(-(sc.x * (r0.x * invP)), -(sc.y * (r0.y * invP)), -(r1.x * invP * is.x), -(r1.y * invP * is.y));
        }
    }
    if (REDUCE) {
        for (int i = threadIdx.x; i < 2 * Cb; i += 256) accum[i] = 0.f;
    } else if (blockIdx.x == 0) {
        for (int c = threadIdx.x; c < Cb; c += 256) {
            if (dbeta) dbeta[c_base + c] += red_in[c_base + c];
            if (dgamma) dgamma[c_base + c] += red_in[C + c_base + c];
        }
    }
    __syncthreads();
    if (row < rows) {
        const float4 a = tabA[cg], k = tabB[cg];
        const float2 sc = f2(a.x, a.y), sh = f2(a.z, a.w), one2 = f2(1.f, 1.f);
        float2 nbb = f2(0.f, 0.f);
        if (!REDUCE && beta_bn) {
            const float2 b = *reinterpret_cast<const float2*>(beta_bn + c_base + 2 * cg);
            nbb = f2(-b.x, -b.y);
        }
        const int C2 = C >> 1;
        const int xb = REDUCE ? (int)blockIdx.x : (int)(gridDim.x - 1 - blockIdx.x);
        const int p0 = xb * pix_per_block, p1 = min(P, p0 + pix_per_block);
        float2 acc_s = f2(0.f, 0.f), acc_d = f2(0.f, 0.f);
        for (int p = p0 + row; p < p1; p += rows * PU) {
            float2 yv[PU];
            uint32_t gr[PU];
#pragma unroll
            for (int j = 0; j < PU; ++j) {
                const int pj = p + j * rows;
                if (pj < p1) {
                    const size_t e2 = (size_t)pj * C2 + (c_base >> 1) + cg;
                    yv[j] = REDUCE ? __ldg(reinterpret_cast<const float2*>(y) + e2) : __ldcs(reinterpret_cast<const float2*>(y) + e2);
                    gr[j] = REDUCE ? __ldg(reinterpret_cast<const uint32_t*>(gs) + e2) : __ldcs(reinterpret_cast<const uint32_t*>(gs) + e2);
                }
            }
#pragma unroll
            for (int j = 0; j < PU; ++j) {
                const int pj = p + j * rows;
                if (pj < p1) {
                    const float2 xm = __fmul2_rn(yv[j], sc);
                    const float2 x = f2(__fadd_rn(xm.x, sh.x), __fadd_rn(xm.y, sh.y));
                    const float2 g = f2(bf16_lo(gr[j]), bf16_hi(gr[j]));
                    const float2 e = f2(ex2_approx(-1.4426950408889634f * x.x), ex2_approx(-1.4426950408889634f * x.y));
                    const float2 d1 = __fadd2_rn(e, one2);
                    const float2 sgm = f2(rcp_approx(d1.x), rcp_approx(d1.y));
                    const float2 oms = __fadd2_rn(one2, f2(-sgm.x, -sgm.y));
                    const float2 gx = __fmul2_rn(g, __fmul2_rn(sgm, __ffma2_rn(x, oms, one2)));
                    if (REDUCE) {
                        acc_s = __fadd2_rn(acc_s, gx);
                        acc_d = __ffma2_rn(gx, __fadd2_rn(yv[j], f2(k.x, k.y)), acc_d);
                    } else {
                        const float2 t1 = __ffma2_rn(sc, gx, f2(k.x, k.y));
                        const float2 d = __ffma2_rn(__fadd2_rn(x, nbb), f2(k.z, k.w), t1);
                        *(reinterpret_cast<uint32_t*>(dy_out) + (size_t)pj * C2 + (c_base >> 1) + cg) = pack_bf16x2(d.x, d.y);
                    }
                }
            }
        }
        if (REDUCE) {
            const int cl = cg * 2;
            if (part) {
                float* slot = accum + (size_t)(1 + row) * 2 * Cb;
                slot[cl] = acc_s.x; slot[cl + 1] = acc_s.y; slot[Cb + cl] = acc_d.x; slot[Cb + cl + 1] = acc_d.y;
            } else {
                atomicAdd(&accum[cl], acc_s.x); atomicAdd(&accum[cl + 1], acc_s.y);
                atomicAdd(&accum[Cb + cl], acc_d.x); atomicAdd(&accum[Cb + cl + 1], acc_d.y);
            }
        }
    }
    if (REDUCE) {
        __syncthreads();
        if (part) {
            for (int i = threadIdx.x; i < 2 * Cb; i += 256) {
                float a = 0.f;
                for (int r = 0; r < rows; ++r) a += accum[(size_t)(1 + r) * 2 * Cb + i];
                accum[i] = a;
            }
            __syncthreads();
        }
        for (int c = threadIdx.x; c < Cb; c += 256) {
            const float v0 = accum[c], v1 = accum[Cb + c] * invstd[c_base + c];
            if (part) {
                part[(size_t)blockIdx.x * 2 * C + c_base + c] = v0;
                part[(size_t)blockIdx.x * 2 * C + C + c_base + c] = v1;
            } else {
                atomicAdd(&red_out[c_base + c], v0);
                atomicAdd(&red_out[C + c_base + c], v1);
            }
        }
    }
}

// ------------------------------------------------------------------------------------------
// host launchers
// ------------------------------------------------------------------------------------------
static int pick_ppb(int P, int rows, int T) {
    // enough blocks to fill 148 SMs a few times, but >= 8 pixels per row-thread to amortise the reduce
    long long want_blocks = (long long)num_sms() * 8 / (T > 0 ? T : 1);
    if (want_blocks < 1) want_blocks = 1;
    int ppb = (int)((P + want_blocks - 1) / want_blocks);
    int min_ppb = rows * 8;
    if (ppb < min_ppb) ppb = min_ppb;
    ppb = ((ppb + rows - 1) / rows) * rows;
    return ppb;
}

static int bn_stats_blocks(int P, int C, int* ppb_out) {
    const int rows = 256 / (C / 4);
    const int ppb = pick_ppb(P, rows, 1);   // independent of T: a frame's statistics are bit-identical however the T*B batch is folded
    if (ppb_out) *ppb_out = ppb;
    return (P + ppb - 1) / ppb;
}
long long bn_stats_workspace_floats(int T, int P, int C) {
    if (C % 4 != 0 || C < 4 || C > 1024 || T < 1 || P < 1) return 0;
    return (long long)T * bn_stats_blocks(P, C, nullptr) * 2 * C;
}
int launch_bn_stats_from_partials(const float* part, double* sums, int T, int C, int groups_per_t, cudaStream_t st);

// two deterministic stages: per-block partials (no atomics) -> fixed-order fp64 combine
int launch_bn_stats(const float* y, double* sums, float* workspace, int T, int P, int C, cudaStream_t st) {
    SNN_REQUIRE(C % 4 == 0 && C >= 4 && C <= 1024, "bn_stats: C=%d must be a multiple of 4 in [4,1024]", C);
    SNN_REQUIRE(workspace != nullptr, "bn_stats: workspace of snn_bn_stats_workspace_floats() floats required");
    int ppb = 0;
    const int nblk = bn_stats_blocks(P, C, &ppb);
    const int rows = 256 / (C / 4);
    dim3 grid(nblk, T);
    launch_pdl(bn_stats_kernel, grid, dim3(256), sizeof(float) * 2 * C * rows, st, y, workspace, P, C, ppb);
    SNN_CUDA_OK(cudaGetLastError());
    return launch_bn_stats_from_partials(workspace, sums, T, C, nblk, st);
}

int launch_bn_stats_from_partials(const float* part, double* sums, int T, int C, int groups_per_t, cudaStream_t st) {
    SNN_REQUIRE(T >= 1 && C >= 1 && groups_per_t >= 1, "bn_stats_from_partials: bad sizes");
    dim3 grid((C + 7) / 8, T);
    launch_pdl(bn_stats_from_partials_kernel, grid, dim3(kRL * 8), 0, st, part, sums, C, groups_per_t);
    return check_cuda(cudaGetLastError(), "bn_stats_from_partials_kernel");
}

int launch_bn_finalize_partials(const float* part, double* sums, double* workspace, const float* gamma, const float* beta, float* rm,
                                float* rv, long long* nbt, float* scale, float* shift, float* mean, float* invstd, unsigned int* counters,
                                int T, int C, int P, int groups_per_t, float eps, float momentum, cudaStream_t st) {
    SNN_REQUIRE(T >= 1 && C >= 1 && groups_per_t >= 1 && counters != nullptr && workspace != nullptr,
                "bn_finalize_partials: bad arguments (workspace of snn_bn_finalize_workspace_doubles() doubles required)");
    const int S = bn_finalize_splits(groups_per_t);
    dim3 grid((C + 31) / 32, S);
    launch_pdl(bn_finalize_partials_kernel, grid, dim3(32 * kFinLanes), 0, st, part, workspace, sums, gamma, beta, rm, rv, nbt, scale, shift, mean, invstd,
                                                                 counters, T, C, P, groups_per_t, S, eps, momentum);
    return check_cuda(cudaGetLastError(), "bn_finalize_partials_kernel");
}

int launch_bn_finalize(const double* sums, const float* gamma, const float* beta, float* rm, float* rv, float* scale,
                       float* shift, float* mean, float* invstd, int T, int C, int P, float eps, float momentum,
                       int training, cudaStream_t st) {
    launch_pdl(bn_finalize_kernel, dim3((C + 127) / 128), dim3(128), 0, st, sums, gamma, beta, rm, rv, scale, shift, mean, invstd, T, C, P,
                                                        eps, momentum, training);
    return check_cuda(cudaGetLastError(), "bn_finalize_kernel");
}

int launch_bn_act_fwd(int act, const float* y, const float* scale, const float* shift, const float* v_init,
                      __nv_bfloat16* out, uint8_t* mask, float* v_final, int T, long long n_per_t, int C,
                      int ss_stride_t, float beta, float theta, cudaStream_t st) {
    SNN_REQUIRE(C % 8 == 0, "bn_act_fwd: C=%d must be a multiple of 8", C);
    SNN_REQUIRE(n_per_t % C == 0, "bn_act_fwd: n_per_t not a multiple of C");
    const long long n8 = n_per_t / 8;
    const unsigned blocks = (unsigned)((n8 + 255) / 256);
    if (act == ACT_LIF)
        launch_pdl(bn_act_fwd_kernel<ACT_LIF, false>, dim3(blocks), dim3(256), 0, st, y, scale, shift, v_init, out, mask, v_final, T,
                   n8, C, ss_stride_t, beta, theta, (unsigned long long*)nullptr, (unsigned long long*)nullptr);
    else
        launch_pdl(bn_act_fwd_kernel<ACT_SILU, false>, dim3(blocks), dim3(256), 0, st, y, scale, shift, v_init, out, mask, v_final, T,
                   n8, C, ss_stride_t, beta, theta, (unsigned long long*)nullptr, (unsigned long long*)nullptr);
    return check_cuda(cudaGetLastError(), "bn_act_fwd_kernel");
}

int launch_bn_act_fwd_count(const float* y, const float* scale, const float* shift, const float* v_init, __nv_bfloat16* out,
                            uint8_t* mask, float* v_final, unsigned long long* spikes, unsigned long long* steps, int T,
                            long long n_per_t, int C, int ss_stride_t, float beta, float theta, cudaStream_t st) {
    SNN_REQUIRE(C % 8 == 0, "bn_act_fwd_count: C=%d must be a multiple of 8", C);
    SNN_REQUIRE(n_per_t % C == 0, "bn_act_fwd_count: n_per_t not a multiple of C");
    SNN_REQUIRE(T >= 1 && T <= kCountMaxT, "bn_act_fwd_count: T=%d must be in [1,%d]", T, kCountMaxT);
    SNN_REQUIRE(spikes != nullptr && steps != nullptr, "bn_act_fwd_count: spikes and steps counters are required");
    const long long n8 = n_per_t / 8;
    const unsigned blocks = (unsigned)((n8 + 255) / 256);
    launch_pdl(bn_act_fwd_kernel<ACT_LIF, true>, dim3(blocks), dim3(256), 0, st, y, scale, shift, v_init, out, mask, v_final, T, n8,
               C, ss_stride_t, beta, theta, spikes, steps);
    return check_cuda(cudaGetLastError(), "bn_act_fwd_kernel<LIF, count>");
}

template <int ACT, int TMAX, bool TRAIN>
static int launch_bwd_t(const float* y, const float* scale, const float* shift, const float* mean, const float* invstd,
                        const float* v_init, const __nv_bfloat16* gs, const float* gv_final, float* gx,
                        __nv_bfloat16* dy, float* gv_init, float* red, int T, int P, int C, int ss, float beta,
                        float theta, float alpha, cudaStream_t st) {
    const int rows = 256 / (C / 4);
    const int ppb = pick_ppb(P, rows, 1);
    const size_t smem = TRAIN ? sizeof(float) * T * 2 * C : 0;
    auto kern = bn_act_bwd_kernel<ACT, TMAX, TRAIN>;
    if (smem > 48 * 1024) SNN_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    launch_pdl(kern, dim3((P + ppb - 1) / ppb), dim3(256), smem, st, y, scale, shift, mean, invstd, v_init, gs, gv_final, gx, dy, gv_init,
                                                 red, T, P, C, ss, ppb, beta, theta, alpha);
    return check_cuda(cudaGetLastError(), "bn_act_bwd_kernel");
}

int launch_bn_act_bwd(int act, int training, const float* y, const float* scale, const float* shift, const float* mean,
                      const float* invstd, const float* v_init, const __nv_bfloat16* gs, const float* gv_final,
                      float* gx, __nv_bfloat16* dy, float* gv_init, float* red, int T, int P, int C, int ss_stride_t,
                      float beta, float theta, float alpha, cudaStream_t st) {
    SNN_REQUIRE(C % 4 == 0 && C >= 4 && C <= 1024, "bn_act_bwd: C=%d must be a multiple of 4 in [4,1024]", C);
    SNN_REQUIRE(T >= 1 && T <= 16, "bn_act_bwd: T=%d must be in [1,16]", T);
    if (training) SNN_CUDA_OK(cudaMemsetAsync(red, 0, sizeof(float) * 2 * T * C, st));
#define SNN_BWD(ACT, TM, TR) \
    return launch_bwd_t<ACT, TM, TR>(y, scale, shift, mean, invstd, v_init, gs, gv_final, gx, dy, gv_init, red, T, P, C, ss_stride_t, beta, theta, alpha, st)
    if (act == ACT_LIF) {
        if (training) { if (T <= 4) SNN_BWD(ACT_LIF, 4, true); else if (T <= 8) SNN_BWD(ACT_LIF, 8, true); else SNN_BWD(ACT_LIF, 16, true); }
        else          { if (T <= 4) SNN_BWD(ACT_LIF, 4, false); else if (T <= 8) SNN_BWD(ACT_LIF, 8, false); else SNN_BWD(ACT_LIF, 16, false); }
    } else {
        if (training) { if (T <= 4) SNN_BWD(ACT_SILU, 4, true); else if (T <= 8) SNN_BWD(ACT_SILU, 8, true); else SNN_BWD(ACT_SILU, 16, true); }
        else          { if (T <= 4) SNN_BWD(ACT_SILU, 4, false); else if (T <= 8) SNN_BWD(ACT_SILU, 8, false); else SNN_BWD(ACT_SILU, 16, false); }
    }
#undef SNN_BWD
}

static int g_t16_chunked = 1; // 0: T == 16 uses the one-chunk kernel (A/B timing, snn_debug_set(9, 1))
template <int ACT, int TMAX, bool REDUCE>
static int launch_bwd2_t(const float* y, const float* scale, const float* shift, const float* mean, const float* invstd,
                         const float* beta_bn, const float* red_in, const float* v_init, const __nv_bfloat16* gs,
                         const float* gv_final, __nv_bfloat16* dy, float* gv_init, float* red_out, float* dgamma, float* dbeta,
                         int T, int P, int C, float beta, float theta, float alpha, cudaStream_t st) {
    // bytes of shared memory per channel: two float4 tables per channel PAIR with pitch (TMAX|1), + REDUCE accumulators
    const int per_c = (TMAX | 1) * 16 + (REDUCE ? T * 8 : 0);
    const bool chunked = TMAX == 16 && T == 16 && g_t16_chunked;
    const size_t acc_slots = (chunked && REDUCE) ? (size_t)16 * 256 * 16 : 0;      // per-thread accumulator slots (t16 kernel)
    // channel range per block: largest C / 2^k (multiple of 4) whose tables fit in ~48 KB of shared memory
    const size_t table_cap = acc_slots ? 40 * 1024 : 48 * 1024;                     // t16 reduce: 2 x (40 + 64) KB per SM
    int Cb = C;
    while (((size_t)Cb * per_c > table_cap || Cb > 512) && Cb % 4 == 0) Cb >>= 1;
    SNN_REQUIRE(C % Cb == 0 && Cb % 2 == 0 && Cb <= 512 && (size_t)Cb * per_c <= 200 * 1024,
                "bn_act_bwd2: cannot tile C=%d (T=%d) into shared memory", C, T);
    const int rows = 256 / (Cb / 2);
    const int nyb = C / Cb;
    const int occ = TMAX <= 4 ? 4 : ((TMAX <= 8 || chunked) ? 2 : 1);
    long long want_blocks = (long long)num_sms() * occ * (REDUCE ? 1 : 2) / nyb;    // REDUCE: one full wave; DX: two
    if (want_blocks < 1) want_blocks = 1;
    int ppb = (int)((P + want_blocks - 1) / want_blocks);
    const int min_ppb = rows * (REDUCE ? 8 : 2);
    if (ppb < min_ppb) ppb = min_ppb;
    ppb = ((ppb + rows - 1) / rows) * rows;
    dim3 grid((P + ppb - 1) / ppb, nyb);
    // deterministic mode (REDUCE pass): per-row copies of the block accumulators in shared memory (the t16 kernel has its
    // per-thread slots anyway) and one partial row per block in the scratch buffer, combined in block order afterwards
    float* part = nullptr;
    size_t det_slots = 0;
    if (REDUCE && deterministic()) {
        part = static_cast<float*>(det_scratch(sizeof(float) * (size_t)grid.x * T * 2 * C, st));
        if (!part) return 2;
        if (!acc_slots) det_slots = sizeof(float) * (size_t)rows * T * 2 * Cb;
    }
    const size_t smem = (size_t)Cb * per_c + acc_slots + det_slots;
    SNN_REQUIRE(smem <= 200 * 1024, "bn_act_bwd2: %zu bytes of shared memory (C=%d T=%d)", smem, C, T);
#define SNN_GO(EX)                                                                                                         \
    do {                                                                                                                   \
        auto kern = bn_act_bwd2_kernel<ACT, TMAX, REDUCE, EX>;                                                             \
        if (smem > 48 * 1024) SNN_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
        launch_pdl(kern, grid, dim3(256), smem, st, y, scale, shift, mean, invstd, beta_bn, red_in, v_init, gs, gv_final, dy, gv_init,   \
                                      red_out, dgamma, dbeta, T, P, C, Cb, ppb, beta, theta, alpha, 1.0f / (float)P, part); \
    } while (0)
    if (chunked) {
        auto kern = bn_act_bwd2_t16_kernel<ACT, REDUCE>;
        if (smem > 48 * 1024) SNN_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        launch_pdl(kern, grid, dim3(256), smem, st, y, scale, shift, mean, invstd, beta_bn, red_in, v_init, gs, gv_final, dy, gv_init,
                   red_out, dgamma, dbeta, T, P, C, Cb, ppb, beta, theta, alpha, 1.0f / (float)P, part);
    } else if (T == TMAX) SNN_GO(true); else SNN_GO(false);
#undef SNN_GO
    SNN_CUDA_OK(cudaGetLastError());
    if (part) return launch_ordered_combine_f32(part, (int)grid.x, (long long)T * 2 * C, red_out, st);
    return 0;
}

static int g_t1_fast = 1;     // 0: T == 1 SiLU layers go through the generic kernel (A/B timing)
void neuron_debug_set(int k, int v) {
    if (k == 0) g_t1_fast = v ? 0 : 1;
    if (k == 1) g_t16_chunked = v ? 0 : 1;
}

// pass = 0: reduce (writes red [T][2][C], zeroed here); pass = 1: dx (reads red; writes dy, gv_init; dgamma/dbeta +=)
int launch_bn_act_bwd2(int pass, int act, const float* y, const float* scale, const float* shift, const float* mean,
                       const float* invstd, const float* beta_bn, const float* v_init, const __nv_bfloat16* gs,
                       const float* gv_final, float* red, __nv_bfloat16* dy, float* gv_init, float* dgamma, float* dbeta,
                       int T, int P, int C, float beta, float theta, float alpha, cudaStream_t st) {
    SNN_REQUIRE(C % 2 == 0 && C >= 2, "bn_act_bwd2: C=%d must be even", C);
    SNN_REQUIRE(T >= 1 && T <= 16, "bn_act_bwd2: T=%d must be in [1,16]", T);
    if (pass == 0) SNN_CUDA_OK(cudaMemsetAsync(red, 0, sizeof(float) * 2 * T * C, st));
    if (act == ACT_SILU && T == 1 && g_t1_fast) {
        int Cb = C;
        while (Cb > 512 && Cb % 4 == 0) Cb >>= 1;
        SNN_REQUIRE(C % Cb == 0 && Cb % 2 == 0 && Cb <= 512, "bn_act_bwd2: cannot tile C=%d", C);
        const int rows = 256 / (Cb / 2), nyb = C / Cb;
        long long want_blocks = (long long)num_sms() * 4 * (pass == 0 ? 1 : 2) / nyb;
        if (want_blocks < 1) want_blocks = 1;
        int ppb = (int)((P + want_blocks - 1) / want_blocks);
        const int unit = rows * 4;
        if (ppb < unit * (pass == 0 ? 2 : 1)) ppb = unit * (pass == 0 ? 2 : 1);
        ppb = ((ppb + unit - 1) / unit) * unit;
        dim3 grid((P + ppb - 1) / ppb, nyb);
        float* part = nullptr;
        if (pass == 0 && deterministic()) {
            part = static_cast<float*>(det_scratch(sizeof(float) * (size_t)grid.x * 2 * C, st));
            if (!part) return 2;
        }
        const size_t smem = (size_t)(Cb / 2) * 32 + (pass == 0 ? (size_t)2 * Cb * 4 * (part ? 1 + rows : 1) : 0);
        if (pass == 0)
            launch_pdl(silu_t1_bwd2_kernel<true>, grid, dim3(256), smem, st, y, scale, shift, mean, invstd, beta_bn, nullptr, gs, nullptr, red, nullptr,
                                                               nullptr, P, C, Cb, ppb, 1.0f / (float)P, part);
        else
            launch_pdl(silu_t1_bwd2_kernel<false>, grid, dim3(256), smem, st, y, scale, shift, mean, invstd, beta_bn, red, gs, dy, nullptr, dgamma, dbeta,
                                                                P, C, Cb, ppb, 1.0f / (float)P, (float*)nullptr);
        SNN_CUDA_OK(cudaGetLastError());
        if (part) return launch_ordered_combine_f32(part, (int)grid.x, 2LL * C, red, st);
        return 0;
    }
#define SNN_BWD2(ACT, TM)                                                                                                   \
    return pass == 0 ? launch_bwd2_t<ACT, TM, true>(y, scale, shift, mean, invstd, beta_bn, nullptr, v_init, gs, gv_final,   \
                                                    nullptr, nullptr, red, nullptr, nullptr, T, P, C, beta, theta, alpha, st) \
                     : launch_bwd2_t<ACT, TM, false>(y, scale, shift, mean, invstd, beta_bn, red, v_init, gs, gv_final, dy,   \
                                                     gv_init, nullptr, dgamma, dbeta, T, P, C, beta, theta, alpha, st)
    if (act == ACT_LIF) {
        if (T == 1) SNN_BWD2(ACT_LIF, 1); else if (T <= 4) SNN_BWD2(ACT_LIF, 4); else if (T <= 8) SNN_BWD2(ACT_LIF, 8); else SNN_BWD2(ACT_LIF, 16);
    } else {
        if (T == 1) SNN_BWD2(ACT_SILU, 1); else if (T <= 4) SNN_BWD2(ACT_SILU, 4); else if (T <= 8) SNN_BWD2(ACT_SILU, 8); else SNN_BWD2(ACT_SILU, 16);
    }
#undef SNN_BWD2
}

int launch_bn_bwd_dx(const float* red, const float* gamma, const float* gx, const float* y, const float* scale,
                     const float* mean, const float* invstd, float* coef, float* dgamma, float* dbeta,
                     __nv_bfloat16* dy, int T, int P, int C, cudaStream_t st) {
    launch_pdl(bn_bwd_finalize_kernel, dim3((C + 127) / 128), dim3(128), 0, st, red, scale, coef, dgamma, dbeta, gamma, T, C, P);
    SNN_CUDA_OK(cudaGetLastError());
    const long long n4 = (long long)P * C / 4;
    dim3 grid((unsigned)((n4 + 255) / 256), T);
    launch_pdl(bn_bwd_dx_kernel, grid, dim3(256), 0, st, gx, y, scale, mean, invstd, coef, dy, T, n4, C);
    return check_cuda(cudaGetLastError(), "bn_bwd_dx_kernel");
}

}  // namespace snn

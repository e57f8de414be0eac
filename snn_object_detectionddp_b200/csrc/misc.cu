// Small HBM-bound helpers around the tensor-core convs: weight casts/transposes, layout
// conversion at the module boundary, ConvLSTM gate math, fused grad-clip + AdamW.
#include "common.cuh"

namespace snn {

// ------------------------------------------------------------------------------------------
// weight prep: fp32 master [N][T][K] -> bf16 copy (fprop operand) and bf16 [K][T][N] (dgrad operand)
// ------------------------------------------------------------------------------------------
__global__ void weight_prep_kernel(const float* __restrict__ w, __nv_bfloat16* __restrict__ wf,
                                   __nv_bfloat16* __restrict__ wt, int N, int T, int K) {
    pdl_launch_dependents();
    pdl_wait();
    __shared__ float tile[32][33];
    const int t = blockIdx.z;
    const int n0 = blockIdx.y * 32, k0 = blockIdx.x * 32;
    const int tx = threadIdx.x, ty = threadIdx.y;  // 32 x 8
    for (int j = ty; j < 32; j += 8) {
        const int n = n0 + j, k = k0 + tx;
        float v = 0.f;
        if (n < N && k < K) {
            const size_t idx = ((size_t)n * T + t) * K + k;
            v = w[idx];
            if (wf) wf[idx] = __float2bfloat16_rn(v);
        }
        tile[j][tx] = v;
    }
    __syncthreads();
    if (wt) {
        for (int j = ty; j < 32; j += 8) {
            const int k = k0 + j, n = n0 + tx;
            if (n < N && k < K) wt[((size_t)k * T + t) * N + n] = __float2bfloat16_rn(tile[tx][j]);
        }
    }
}

int launch_weight_prep(const float* w, __nv_bfloat16* wf, __nv_bfloat16* wt, int N, int T, int K, cudaStream_t st) {
    dim3 grid((K + 31) / 32, (N + 31) / 32, T), block(32, 8);
    launch_pdl(weight_prep_kernel, grid, block, 0, st, w, wf, wt, N, T, K);
    return check_cuda(cudaGetLastError(), "weight_prep_kernel");
}

// ------------------------------------------------------------------------------------------
// NCHW fp32 <-> NHWC (bf16 | fp32) at the module boundary
// ------------------------------------------------------------------------------------------
template <typename TOut>
__global__ void nchw_to_nhwc_kernel(const float* __restrict__ in, TOut* __restrict__ out, int C, int HW, long long out_ld,
                                    int out_coff) {
    pdl_launch_dependents();
    pdl_wait();
    __shared__ float tile[32][33];
    const int n = blockIdx.z;
    const int c0 = blockIdx.y * 32, p0 = blockIdx.x * 32;
    const int tx = threadIdx.x, ty = threadIdx.y;
    for (int j = ty; j < 32; j += 8) {
        const int c = c0 + j, p = p0 + tx;
        tile[j][tx] = (c < C && p < HW) ? in[((size_t)n * C + c) * HW + p] : 0.f;
    }
    __syncthreads();
    for (int j = ty; j < 32; j += 8) {
        const int p = p0 + j, c = c0 + tx;
        if (c < C && p < HW) out[((size_t)n * HW + p) * out_ld + out_coff + c] = (TOut)tile[tx][j];
    }
}

template <typename TIn>
__global__ void nhwc_to_nchw_kernel(const TIn* __restrict__ in, float* __restrict__ out, int C, int HW, long long in_ld,
                                    int in_coff) {
    pdl_launch_dependents();
    pdl_wait();
    __shared__ float tile[32][33];
    const int n = blockIdx.z;
    const int c0 = blockIdx.y * 32, p0 = blockIdx.x * 32;
    const int tx = threadIdx.x, ty = threadIdx.y;
    for (int j = ty; j < 32; j += 8) {
        const int p = p0 + j, c = c0 + tx;
        tile[j][tx] = (c < C && p < HW) ? (float)in[((size_t)n * HW + p) * in_ld + in_coff + c] : 0.f;
    }
    __syncthreads();
    for (int j = ty; j < 32; j += 8) {
        const int c = c0 + j, p = p0 + tx;
        if (c < C && p < HW) out[((size_t)n * C + c) * HW + p] = tile[tx][j];
    }
}

int launch_nchw_to_nhwc(const float* in, void* out, int out_bf16, int NB, int C, int HW, long long out_ld, int out_coff,
                        cudaStream_t st) {
    dim3 grid((HW + 31) / 32, (C + 31) / 32, NB), block(32, 8);
    if (out_bf16)
        launch_pdl(nchw_to_nhwc_kernel<__nv_bfloat16>, grid, block, 0, st, in, (__nv_bfloat16*)out, C, HW, out_ld, out_coff);
    else
        launch_pdl(nchw_to_nhwc_kernel<float>, grid, block, 0, st, in, (float*)out, C, HW, out_ld, out_coff);
    return check_cuda(cudaGetLastError(), "nchw_to_nhwc_kernel");
}

int launch_nhwc_to_nchw(const void* in, int in_bf16, float* out, int NB, int C, int HW, long long in_ld, int in_coff,
                        cudaStream_t st) {
    dim3 grid((HW + 31) / 32, (C + 31) / 32, NB), block(32, 8);
    if (in_bf16)
        launch_pdl(nhwc_to_nchw_kernel<__nv_bfloat16>, grid, block, 0, st, (const __nv_bfloat16*)in, out, C, HW, in_ld, in_coff);
    else
        launch_pdl(nhwc_to_nchw_kernel<float>, grid, block, 0, st, (const float*)in, out, C, HW, in_ld, in_coff);
    return check_cuda(cudaGetLastError(), "nhwc_to_nchw_kernel");
}

// ------------------------------------------------------------------------------------------
// ConvLSTM gate math (reference model.py:67-69), NHWC: gates fp32 [P][4*Ch] (i|f|g|o), state fp32 [P][Ch]
// forward also emits h as bf16 (operand of the next recurrent conv / bottleneck conv)
// ------------------------------------------------------------------------------------------
// accurate expf (not __expf): h feeds a bf16-rounded conv operand, ulp-level differences flip roundings downstream
SNN_DEVINL float sigmoidf_(float x) { return 1.f / (1.f + expf(-x)); }

__global__ void __launch_bounds__(256)
lstm_gates_fwd_kernel(const float* __restrict__ gates, const float* __restrict__ c_prev, float* __restrict__ c_next,
                      float* __restrict__ h_next, __nv_bfloat16* __restrict__ h_bf16, long long n4, int Ch) {
    pdl_launch_dependents();
    pdl_wait();
    const long long idx = (long long)blockIdx.x * 256 + threadIdx.x;
    if (idx >= n4) return;
    const int ch4 = Ch >> 2;
    const long long p = idx / ch4;
    const int c = (int)(idx % ch4) * 4;
    const float4* g = reinterpret_cast<const float4*>(gates + p * 4 * Ch + c);
    const float4 gi = __ldg(g), gf = __ldg(g + ch4), gg = __ldg(g + 2 * ch4), go = __ldg(g + 3 * ch4);
    float4 cp = make_float4(0.f, 0.f, 0.f, 0.f);
    if (c_prev) cp = __ldg(reinterpret_cast<const float4*>(c_prev) + idx);
    const float iv[4] = {gi.x, gi.y, gi.z, gi.w}, fv[4] = {gf.x, gf.y, gf.z, gf.w}, gv[4] = {gg.x, gg.y, gg.z, gg.w},
                ov[4] = {go.x, go.y, go.z, go.w}, cv[4] = {cp.x, cp.y, cp.z, cp.w};
    float cn[4], hn[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        cn[j] = sigmoidf_(fv[j]) * cv[j] + sigmoidf_(iv[j]) * tanhf(gv[j]);
        hn[j] = sigmoidf_(ov[j]) * tanhf(cn[j]);
    }
    reinterpret_cast<float4*>(c_next)[idx] = make_float4(cn[0], cn[1], cn[2], cn[3]);
    reinterpret_cast<float4*>(h_next)[idx] = make_float4(hn[0], hn[1], hn[2], hn[3]);
    if (h_bf16) {
        uint2 pk;
        pk.x = pack_bf16x2(hn[0], hn[1]); pk.y = pack_bf16x2(hn[2], hn[3]);
        reinterpret_cast<uint2*>(h_bf16)[idx] = pk;
    }
}

// backward of one step: inputs dh (total grad wrt h_next), dc_in (grad wrt c_next from the future);
// outputs dgates (bf16, operand of dgrad/wgrad) and dc_prev.
__global__ void __launch_bounds__(256)
lstm_gates_bwd_kernel(const float* __restrict__ gates, const float* __restrict__ c_prev, const float* __restrict__ c_next,
                      const float* __restrict__ dh, const __nv_bfloat16* __restrict__ dh_bf16, const float* __restrict__ dc_in,
                      __nv_bfloat16* __restrict__ dgates, float* __restrict__ dc_prev, long long n4, int Ch) {
    pdl_launch_dependents();
    pdl_wait();
    const long long idx = (long long)blockIdx.x * 256 + threadIdx.x;
    if (idx >= n4) return;
    const int ch4 = Ch >> 2;
    const long long p = idx / ch4;
    const int c = (int)(idx % ch4) * 4;
    const float4* g = reinterpret_cast<const float4*>(gates + p * 4 * Ch + c);
    const float4 gi = __ldg(g), gf = __ldg(g + ch4), gg = __ldg(g + 2 * ch4), go = __ldg(g + 3 * ch4);
    float4 cp = make_float4(0.f, 0.f, 0.f, 0.f), dci = cp;
    if (c_prev) cp = __ldg(reinterpret_cast<const float4*>(c_prev) + idx);
    if (dc_in) dci = __ldg(reinterpret_cast<const float4*>(dc_in) + idx);
    const float4 cnx = __ldg(reinterpret_cast<const float4*>(c_next) + idx);
    // total gradient w.r.t. h_t = recurrent part (fp32, from the next step's W_h dgrad) + the consumer's part (bf16, from
    // bottleneck_conv's dgrad); either may be absent.  (Round 1 cast and added them with separate ATen kernels.)
    float4 dhh = make_float4(0.f, 0.f, 0.f, 0.f);
    if (dh) dhh = __ldg(reinterpret_cast<const float4*>(dh) + idx);
    if (dh_bf16) {
        const uint2 hb = __ldg(reinterpret_cast<const uint2*>(dh_bf16) + idx);
        dhh.x += bf16_lo(hb.x); dhh.y += bf16_hi(hb.x); dhh.z += bf16_lo(hb.y); dhh.w += bf16_hi(hb.y);
    }
    const float iv[4] = {gi.x, gi.y, gi.z, gi.w}, fv[4] = {gf.x, gf.y, gf.z, gf.w}, gv[4] = {gg.x, gg.y, gg.z, gg.w},
                ov[4] = {go.x, go.y, go.z, go.w}, cv[4] = {cp.x, cp.y, cp.z, cp.w}, cn[4] = {cnx.x, cnx.y, cnx.z, cnx.w},
                dhv[4] = {dhh.x, dhh.y, dhh.z, dhh.w}, dcv[4] = {dci.x, dci.y, dci.z, dci.w};
    float di[4], df[4], dg[4], dov[4], dcp[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const float si = sigmoidf_(iv[j]), sf = sigmoidf_(fv[j]), so = sigmoidf_(ov[j]), tg = tanhf(gv[j]), tc = tanhf(cn[j]);
        const float dc = dcv[j] + dhv[j] * so * (1.f - tc * tc);
        dov[j] = dhv[j] * tc * so * (1.f - so);
        di[j] = dc * tg * si * (1.f - si);
        df[j] = dc * cv[j] * sf * (1.f - sf);
        dg[j] = dc * si * (1.f - tg * tg);
        dcp[j] = dc * sf;
    }
    uint2* o = reinterpret_cast<uint2*>(dgates + p * 4 * Ch + c);
    uint2 pk;
    pk.x = pack_bf16x2(di[0], di[1]); pk.y = pack_bf16x2(di[2], di[3]); o[0] = pk;
    pk.x = pack_bf16x2(df[0], df[1]); pk.y = pack_bf16x2(df[2], df[3]); o[ch4] = pk;
    pk.x = pack_bf16x2(dg[0], dg[1]); pk.y = pack_bf16x2(dg[2], dg[3]); o[2 * ch4] = pk;
    pk.x = pack_bf16x2(dov[0], dov[1]); pk.y = pack_bf16x2(dov[2], dov[3]); o[3 * ch4] = pk;
    reinterpret_cast<float4*>(dc_prev)[idx] = make_float4(dcp[0], dcp[1], dcp[2], dcp[3]);
}

int launch_lstm_gates_fwd(const float* gates, const float* c_prev, float* c_next, float* h_next, __nv_bfloat16* h_bf16,
                          long long P, int Ch, cudaStream_t st) {
    SNN_REQUIRE(Ch % 4 == 0, "lstm_gates: Ch must be a multiple of 4");
    const long long n4 = P * Ch / 4;
    launch_pdl(lstm_gates_fwd_kernel, dim3((unsigned)((n4 + 255) / 256)), dim3(256), 0, st, gates, c_prev, c_next, h_next, h_bf16, n4, Ch);
    return check_cuda(cudaGetLastError(), "lstm_gates_fwd_kernel");
}

int launch_lstm_gates_bwd(const float* gates, const float* c_prev, const float* c_next, const float* dh, const __nv_bfloat16* dh_bf16,
                          const float* dc_in, __nv_bfloat16* dgates, float* dc_prev, long long P, int Ch, cudaStream_t st) {
    SNN_REQUIRE(Ch % 4 == 0, "lstm_gates: Ch must be a multiple of 4");
    const long long n4 = P * Ch / 4;
    launch_pdl(lstm_gates_bwd_kernel, dim3((unsigned)((n4 + 255) / 256)), dim3(256), 0, st, gates, c_prev, c_next, dh, dh_bf16, dc_in, dgates, dc_prev, n4, Ch);
    return check_cuda(cudaGetLastError(), "lstm_gates_bwd_kernel");
}

// ------------------------------------------------------------------------------------------
// deterministic mode: out[i] += part[0][i] + part[1][i] + ... in block order (see common.cuh)
// ------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256) ordered_combine_kernel(const T* __restrict__ part, int nblocks, long long n, T* __restrict__ out) {
    pdl_launch_dependents();
    pdl_wait();
    const long long i = (long long)blockIdx.x * 256 + threadIdx.x;
    if (i >= n) return;
    T a = part[i];
    for (int b = 1; b < nblocks; ++b) a += part[(long long)b * n + i];
    out[i] += a;
}
int launch_ordered_combine_f32(const float* part, int nblocks, long long n, float* out, cudaStream_t st) {
    launch_pdl(ordered_combine_kernel<float>, dim3((unsigned)((n + 255) / 256)), dim3(256), 0, st, part, nblocks, n, out);
    return check_cuda(cudaGetLastError(), "ordered_combine_kernel<float>");
}
int launch_ordered_combine_f64(const double* part, int nblocks, long long n, double* out, cudaStream_t st) {
    launch_pdl(ordered_combine_kernel<double>, dim3((unsigned)((n + 255) / 256)), dim3(256), 0, st, part, nblocks, n, out);
    return check_cuda(cudaGetLastError(), "ordered_combine_kernel<double>");
}

// ------------------------------------------------------------------------------------------
// bias gradient: acc[c] += sum_p dy[p][c]  (dy bf16 [P][C]); grid.y walks column blocks of <= 1024
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
colsum_bf16_kernel(const __nv_bfloat16* __restrict__ dy, float* __restrict__ acc, long long P, int C, int cblk,
                   int pix_per_block, float* __restrict__ part /* deterministic mode: [gridDim.x][C] block partials, else null */) {
    pdl_launch_dependents();
    pdl_wait();
    extern __shared__ float shc[];  // [cblk] (+ deterministic mode: [rows][cblk] slots behind it)
    const int c_base = blockIdx.y * cblk;
    const int cw = min(cblk, C - c_base);
    const int tpp = cw >> 2;  // threads per pixel, 4 channels each
    const int rows = 256 / tpp;
    const int cg = threadIdx.x % tpp, row = threadIdx.x / tpp;
    for (int i = threadIdx.x; i < cw; i += 256) shc[i] = 0.f;
    __syncthreads();
    if (row < rows) {
        const long long p0 = (long long)blockIdx.x * pix_per_block;
        const long long p1 = min(P, p0 + (long long)pix_per_block);
        float s[4] = {0.f, 0.f, 0.f, 0.f};
        for (long long p = p0 + row; p < p1; p += rows) {
            const uint2 v = __ldg(reinterpret_cast<const uint2*>(dy + p * C + c_base) + cg);
            s[0] += bf16_lo(v.x); s[1] += bf16_hi(v.x); s[2] += bf16_lo(v.y); s[3] += bf16_hi(v.y);
        }
        if (part) {
#pragma unroll
            for (int i = 0; i < 4; ++i) shc[cblk + row * cw + cg * 4 + i] = s[i];
        } else {
#pragma unroll
            for (int i = 0; i < 4; ++i) atomicAdd(&shc[cg * 4 + i], s[i]);
        }
    }
    __syncthreads();
    if (part) {     // rows summed in row order, one partial per block and column
        for (int i = threadIdx.x; i < cw; i += 256) {
            float a = 0.f;
            for (int r = 0; r < rows; ++r) a += shc[cblk + r * cw + i];
            part[(size_t)blockIdx.x * C + c_base + i] = a;
        }
        return;
    }
    for (int i = threadIdx.x; i < cw; i += 256) atomicAdd(&acc[c_base + i], shc[i]);
}

int launch_colsum_bf16(const __nv_bfloat16* dy, float* acc, long long P, int C, cudaStream_t st) {
    SNN_REQUIRE(C % 4 == 0, "colsum: C=%d must be a multiple of 4", C);
    const int cblk = C < 1024 ? C : 1024;
    SNN_REQUIRE(C % cblk == 0 || C < 1024, "colsum: C=%d must be < 1024 or a multiple of 1024", C);
    const int rows = 256 / (cblk / 4);
    long long want = (long long)num_sms() * 4;
    long long ppb = (P + want - 1) / want;
    if (ppb < rows * 4) ppb = rows * 4;
    ppb = (ppb + rows - 1) / rows * rows;
    dim3 grid((unsigned)((P + ppb - 1) / ppb), (C + cblk - 1) / cblk);
    if (deterministic()) {
        float* part = static_cast<float*>(det_scratch(sizeof(float) * (size_t)grid.x * C, st));
        if (!part) return 2;
        launch_pdl(colsum_bf16_kernel, grid, dim3(256), sizeof(float) * (cblk + 1024), st, dy, acc, P, C, cblk, (int)ppb, part);
        SNN_CUDA_OK(cudaGetLastError());
        return launch_ordered_combine_f32(part, (int)grid.x, C, acc, st);
    }
    launch_pdl(colsum_bf16_kernel, grid, dim3(256), sizeof(float) * cblk, st, dy, acc, P, C, cblk, (int)ppb, (float*)nullptr);
    return check_cuda(cudaGetLastError(), "colsum_bf16_kernel");
}

// ------------------------------------------------------------------------------------------
// fused global grad-norm + clip + AdamW over ONE flat fp32 buffer (reference train.py:77-78)
//   pass 1: sum of squares -> device scalar        (4 B/param)
//   pass 2: clip coefficient from the scalar, AdamW update, bf16 shadow copy (28+2 B/param)
// hyper-parameters (lr, beta1, step-dependent bias corrections) are read from a device array so the
// OneCycle schedule never forces a host sync:  hp = {lr, beta1, beta2, eps, wd, bc1, bc2, max_norm}
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) sumsq_kernel(const float* __restrict__ g, long long n4, double* __restrict__ acc,
                                                    double* __restrict__ part /* deterministic mode: [gridDim.x], else null */) {
    pdl_launch_dependents();
    pdl_wait();
    float s = 0.f;
    for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < n4; i += (long long)gridDim.x * 256) {
        const float4 v = __ldg(reinterpret_cast<const float4*>(g) + i);
        s += v.x * v.x + v.y * v.y + v.z * v.z + v.w * v.w;
    }
    for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    __shared__ float ws[8];
    if ((threadIdx.x & 31) == 0) ws[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0;
        for (int i = 0; i < 8; ++i) t += ws[i];
        if (part) part[blockIdx.x] = t;
        else atomicAdd(acc, t);
    }
}

__global__ void __launch_bounds__(256)
adamw_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v,
             __nv_bfloat16* __restrict__ shadow, long long n4, const float* __restrict__ hp_table,
             const double* __restrict__ sumsq, float* __restrict__ gnorm_out, const int* __restrict__ step_ptr, int n_rows) {
    pdl_launch_dependents();
    pdl_wait();
    // row of the tabulated schedule: picked by a DEVICE step counter so a captured CUDA graph advances on replay
    const float* hp = hp_table + (step_ptr ? (size_t)min(*step_ptr, n_rows - 1) * 8 : 0);
    const float lr = hp[0], b1 = hp[1], b2 = hp[2], eps = hp[3], wd = hp[4], bc1 = hp[5], bc2 = hp[6], max_norm = hp[7];
    const float gn = (float)sqrt(*sumsq);
    float clip = max_norm / (gn + 1e-6f);  // torch.nn.utils.clip_grad_norm_: coef clamped to 1
    if (clip > 1.f) clip = 1.f;
    if (max_norm <= 0.f) clip = 1.f;
    if (gnorm_out && blockIdx.x == 0 && threadIdx.x == 0) *gnorm_out = gn;
    const float step_size = lr / bc1;
    const float rsq_bc2 = 1.f / sqrtf(bc2);
    for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < n4; i += (long long)gridDim.x * 256) {
        float4 pp = reinterpret_cast<float4*>(p)[i];
        const float4 gg = __ldg(reinterpret_cast<const float4*>(g) + i);
        float4 mm = reinterpret_cast<float4*>(m)[i], vv = reinterpret_cast<float4*>(v)[i];
        float pa[4] = {pp.x, pp.y, pp.z, pp.w}, ga[4] = {gg.x, gg.y, gg.z, gg.w}, ma[4] = {mm.x, mm.y, mm.z, mm.w},
              va[4] = {vv.x, vv.y, vv.z, vv.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const float gr = ga[j] * clip;
            pa[j] *= (1.f - lr * wd);
            ma[j] = b1 * ma[j] + (1.f - b1) * gr;
            va[j] = b2 * va[j] + (1.f - b2) * gr * gr;
            const float denom = sqrtf(va[j]) * rsq_bc2 + eps;
            pa[j] -= step_size * (ma[j] / denom);
        }
        reinterpret_cast<float4*>(p)[i] = make_float4(pa[0], pa[1], pa[2], pa[3]);
        reinterpret_cast<float4*>(m)[i] = make_float4(ma[0], ma[1], ma[2], ma[3]);
        reinterpret_cast<float4*>(v)[i] = make_float4(va[0], va[1], va[2], va[3]);
        if (shadow) {
            uint2 pk;
            pk.x = pack_bf16x2(pa[0], pa[1]); pk.y = pack_bf16x2(pa[2], pa[3]);
            reinterpret_cast<uint2*>(shadow)[i] = pk;
        }
    }
}

int launch_sumsq(const float* g, long long n, double* acc, int zero_first, cudaStream_t st) {
    SNN_REQUIRE(n % 4 == 0, "sumsq: length must be a multiple of 4");
    if (zero_first) SNN_CUDA_OK(cudaMemsetAsync(acc, 0, sizeof(double), st));
    const long long n4 = n / 4;
    long long blocks = (n4 + 255) / 256;
    const long long cap = (long long)num_sms() * 8;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    if (deterministic()) {
        double* part = static_cast<double*>(det_scratch(sizeof(double) * (size_t)blocks, st));
        if (!part) return 2;
        launch_pdl(sumsq_kernel, dim3((unsigned)blocks), dim3(256), 0, st, g, n4, acc, part);
        SNN_CUDA_OK(cudaGetLastError());
        return launch_ordered_combine_f64(part, (int)blocks, 1, acc, st);
    }
    launch_pdl(sumsq_kernel, dim3((unsigned)blocks), dim3(256), 0, st, g, n4, acc, (double*)nullptr);
    return check_cuda(cudaGetLastError(), "sumsq_kernel");
}

__global__ void step_advance_kernel(int* step) {
    pdl_launch_dependents();
    pdl_wait(); *step += 1; }

int launch_adamw(float* p, float* g, float* m, float* v, __nv_bfloat16* shadow, long long n, const float* hp,
                 const double* sumsq, float* gnorm_out, int* step_ptr, int n_rows, int zero_grad, cudaStream_t st) {
    SNN_REQUIRE(n % 4 == 0, "adamw: length must be a multiple of 4");
    const long long n4 = n / 4;
    long long blocks = (n4 + 255) / 256;
    const long long cap = (long long)num_sms() * 8;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    launch_pdl(adamw_kernel, dim3((unsigned)blocks), dim3(256), 0, st, p, g, m, v, shadow, n4, hp, sumsq, gnorm_out, step_ptr, n_rows);
    SNN_CUDA_OK(cudaGetLastError());
    // zero_grad: the gradient has been consumed; leave it zeroed for the next step's accumulating wgrad kernels
    // (optimizer.zero_grad() of train.py:61).  A memset node right behind the kernel: 67 us for 481 MB.  Storing the zeros
    // from inside the kernel (to the line it has just loaded) was measured 4x slower for the WHOLE pass (0.58 -> 2.35 ms).
    if (zero_grad) SNN_CUDA_OK(cudaMemsetAsync(g, 0, sizeof(float) * (size_t)n, st));
    if (step_ptr) launch_pdl(step_advance_kernel, dim3(1), dim3(1), 0, st, step_ptr);
    return check_cuda(cudaGetLastError(), "adamw_kernel");
}

// ------------------------------------------------------------------------------------------
// exponential moving average of the weights (ultralytics ModelEMA.update):  e = d * e + (1 - d) * s
//   one float4 pass over the flat master buffer (12 B/param) + one block per BatchNorm running-statistics segment.
// The decay comes from a host-computed table row {float(d), float(1 - d)} picked by a DEVICE update counter (as the
// AdamW schedule row is), so a captured graph ramps the decay on replay.  __fmul_rn / __fadd_rn: the rounding and the
// order of torch's `v *= d; v += (1 - d) * s` on fp32 tensors -- two products, one sum, never contracted into an FMA.
// ------------------------------------------------------------------------------------------
SNN_DEVINL float ema_mix(float e, float s, float d, float omd) { return __fadd_rn(__fmul_rn(e, d), __fmul_rn(omd, s)); }

__global__ void __launch_bounds__(256)
ema_flat_kernel(float* __restrict__ e, const float* __restrict__ s, long long n4, const float* __restrict__ decay,
                const int* __restrict__ upd_ptr, int n_rows) {
    pdl_launch_dependents();
    pdl_wait();
    const float* row = decay + (size_t)min(*upd_ptr, n_rows - 1) * 2;
    const float d = row[0], omd = row[1];
    for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < n4; i += (long long)gridDim.x * 256) {
        const float4 ss = __ldg(reinterpret_cast<const float4*>(s) + i);
        float4 ee = reinterpret_cast<float4*>(e)[i];
        ee.x = ema_mix(ee.x, ss.x, d, omd);
        ee.y = ema_mix(ee.y, ss.y, d, omd);
        ee.z = ema_mix(ee.z, ss.z, d, omd);
        ee.w = ema_mix(ee.w, ss.w, d, omd);
        reinterpret_cast<float4*>(e)[i] = ee;
    }
}

// seg = [n_seg][3] int64 {source address, destination address, length}; one block per segment, any length
__global__ void __launch_bounds__(256)
ema_segments_kernel(const long long* __restrict__ seg, const float* __restrict__ decay, const int* __restrict__ upd_ptr,
                    int n_rows) {
    pdl_launch_dependents();
    pdl_wait();
    const float* row = decay + (size_t)min(*upd_ptr, n_rows - 1) * 2;
    const float d = row[0], omd = row[1];
    const float* __restrict__ s = reinterpret_cast<const float*>(seg[3 * blockIdx.x]);
    float* __restrict__ e = reinterpret_cast<float*>(seg[3 * blockIdx.x + 1]);
    const long long n = seg[3 * blockIdx.x + 2];
    for (long long i = threadIdx.x; i < n; i += 256) e[i] = ema_mix(e[i], __ldg(s + i), d, omd);
}

int launch_ema_update(float* ema, const float* src, long long n, const long long* seg, int n_seg, const float* decay,
                      int* upd_ptr, int n_rows, cudaStream_t st) {
    SNN_REQUIRE(n % 4 == 0 && n >= 0, "ema_update: length %lld must be a multiple of 4", n);
    SNN_REQUIRE(((uintptr_t)ema & 15) == 0 && ((uintptr_t)src & 15) == 0, "ema_update: buffers must be 16-byte aligned");
    SNN_REQUIRE(decay && upd_ptr && n_rows >= 1, "ema_update: needs the decay table and the device update counter");
    SNN_REQUIRE(n_seg >= 0 && (n_seg == 0 || seg), "ema_update: bad segment table");
    const long long n4 = n / 4;
    if (n4 > 0) {
        long long blocks = (n4 + 255) / 256;
        const long long cap = (long long)num_sms() * 8;
        if (blocks > cap) blocks = cap;
        launch_pdl(ema_flat_kernel, dim3((unsigned)blocks), dim3(256), 0, st, ema, src, n4, decay, upd_ptr, n_rows);
        SNN_CUDA_OK(cudaGetLastError());
    }
    if (n_seg > 0) {
        launch_pdl(ema_segments_kernel, dim3((unsigned)n_seg), dim3(256), 0, st, seg, decay, upd_ptr, n_rows);
        SNN_CUDA_OK(cudaGetLastError());
    }
    launch_pdl(step_advance_kernel, dim3(1), dim3(1), 0, st, upd_ptr);
    return check_cuda(cudaGetLastError(), "ema_update");
}

}  // namespace snn

namespace snn {

// ------------------------------------------------------------------------------------------
// Bilinear resize of the skip tensor (reference model.py:43-44: F.interpolate(skip_x, size=x.shape[2:],
// mode='bilinear', align_corners=False)), NHWC bf16, fp32 arithmetic, one rounding to bf16.
// Source index / weights exactly as ATen's upsample_bilinear2d (align_corners=False):
//   src = max(0, scale*(dst+0.5)-0.5), scale = in/out (fp32); i0 = (int)src; i1 = i0 + (i0 < in-1); l1 = src - i0.
// HBM-bound: 8 channels (16 B) per thread.
// ------------------------------------------------------------------------------------------
SNN_DEVINL void bilin_src(int dst, float scale, int in_size, int* i0, int* ip, float* l1) {
    float s = scale * ((float)dst + 0.5f) - 0.5f;
    if (s < 0.f) s = 0.f;
    int i = (int)s;
    if (i > in_size - 1) i = in_size - 1;
    *i0 = i;
    *ip = (i < in_size - 1) ? 1 : 0;
    *l1 = s - (float)i;
}

SNN_DEVINL void unpack8(const uint4 v, float* f) {
    f[0] = bf16_lo(v.x); f[1] = bf16_hi(v.x); f[2] = bf16_lo(v.y); f[3] = bf16_hi(v.y);
    f[4] = bf16_lo(v.z); f[5] = bf16_hi(v.z); f[6] = bf16_lo(v.w); f[7] = bf16_hi(v.w);
}

__global__ void __launch_bounds__(256)
bilinear_fwd_kernel(const __nv_bfloat16* __restrict__ x, __nv_bfloat16* __restrict__ y, int NB, int Hi, int Wi, int Ho, int Wo,
                    int C, float sh, float sw) {
    pdl_launch_dependents();
    pdl_wait();
    const int c8 = C >> 3;
    const long long idx = (long long)blockIdx.x * 256 + threadIdx.x;
    const long long total = (long long)NB * Ho * Wo * c8;
    if (idx >= total) return;
    const int cg = (int)(idx % c8);
    const long long pix = idx / c8;
    const int ow = (int)(pix % Wo), oh = (int)((pix / Wo) % Ho);
    const long long n = pix / ((long long)Wo * Ho);
    int h0, hp, w0, wp;
    float lh, lw;
    bilin_src(oh, sh, Hi, &h0, &hp, &lh);
    bilin_src(ow, sw, Wi, &w0, &wp, &lw);
    const float kh0 = 1.f - lh, kw0 = 1.f - lw;
    const uint4* base = reinterpret_cast<const uint4*>(x + ((n * Hi + h0) * Wi + w0) * C) + cg;
    const long long rs = (long long)Wi * c8;          // uint4 per input row
    float a[8], b[8], c[8], d[8];
    unpack8(__ldg(base), a);
    unpack8(__ldg(base + (wp ? c8 : 0)), b);
    unpack8(__ldg(base + (hp ? rs : 0)), c);
    unpack8(__ldg(base + (hp ? rs : 0) + (wp ? c8 : 0)), d);
    float o[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) o[j] = kh0 * (kw0 * a[j] + lw * b[j]) + lh * (kw0 * c[j] + lw * d[j]);
    uint4 pk;
    pk.x = pack_bf16x2(o[0], o[1]); pk.y = pack_bf16x2(o[2], o[3]); pk.z = pack_bf16x2(o[4], o[5]); pk.w = pack_bf16x2(o[6], o[7]);
    *(reinterpret_cast<uint4*>(y + pix * C) + cg) = pk;
}

// Backward as a deterministic GATHER: input pixel (ih, iw) collects from every output pixel whose 2x2 footprint touches
// it, with the forward's own weights (no atomics).  For the up-sizing the path needs (out = in + 1) a footprint spans at
// most 3 output rows / columns; the candidate range is computed conservatively and every candidate re-derives its
// forward indices.
__global__ void __launch_bounds__(256)
bilinear_bwd_kernel(const __nv_bfloat16* __restrict__ gy, __nv_bfloat16* __restrict__ gx, int NB, int Hi, int Wi, int Ho, int Wo,
                    int C, float sh, float sw) {
    pdl_launch_dependents();
    pdl_wait();
    const int c8 = C >> 3;
    const long long idx = (long long)blockIdx.x * 256 + threadIdx.x;
    const long long total = (long long)NB * Hi * Wi * c8;
    if (idx >= total) return;
    const int cg = (int)(idx % c8);
    const long long pix = idx / c8;
    const int iw = (int)(pix % Wi), ih = (int)((pix / Wi) % Hi);
    const long long n = pix / ((long long)Wi * Hi);
    // outputs with src in (i-1, i+1): dst in ((i-0.5)/scale - 0.5, (i+1.5)/scale - 0.5); one extra candidate either side
    int oh_lo = (int)floorf(((float)ih - 0.5f) / sh - 0.5f) - 1, oh_hi = (int)ceilf(((float)ih + 1.5f) / sh - 0.5f) + 1;
    int ow_lo = (int)floorf(((float)iw - 0.5f) / sw - 0.5f) - 1, ow_hi = (int)ceilf(((float)iw + 1.5f) / sw - 0.5f) + 1;
    if (ih == 0) oh_lo = 0;                      // clamped sources (src < 0 -> 0) all land on row 0
    if (iw == 0) ow_lo = 0;
    if (ih == Hi - 1) oh_hi = Ho - 1;
    if (iw == Wi - 1) ow_hi = Wo - 1;
    oh_lo = max(oh_lo, 0); ow_lo = max(ow_lo, 0); oh_hi = min(oh_hi, Ho - 1); ow_hi = min(ow_hi, Wo - 1);
    float acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    for (int oh = oh_lo; oh <= oh_hi; ++oh) {
        int h0, hp; float lh;
        bilin_src(oh, sh, Hi, &h0, &hp, &lh);
        if (!(h0 == ih || h0 + hp == ih)) continue;
        const float wh = (h0 == ih ? 1.f - lh : 0.f) + (h0 + hp == ih ? lh : 0.f);     // hp == 0 (last row): both terms, sum 1
        for (int ow = ow_lo; ow <= ow_hi; ++ow) {
            int w0, wp; float lw;
            bilin_src(ow, sw, Wi, &w0, &wp, &lw);
            if (!(w0 == iw || w0 + wp == iw)) continue;
            const float ww = (w0 == iw ? 1.f - lw : 0.f) + (w0 + wp == iw ? lw : 0.f);
            float g[8];
            unpack8(__ldg(reinterpret_cast<const uint4*>(gy + ((n * Ho + oh) * Wo + ow) * C) + cg), g);
            const float k = wh * ww;
#pragma unroll
            for (int j = 0; j < 8; ++j) acc[j] = fmaf(k, g[j], acc[j]);
        }
    }
    uint4 pk;
    pk.x = pack_bf16x2(acc[0], acc[1]); pk.y = pack_bf16x2(acc[2], acc[3]); pk.z = pack_bf16x2(acc[4], acc[5]); pk.w = pack_bf16x2(acc[6], acc[7]);
    *(reinterpret_cast<uint4*>(gx + pix * C) + cg) = pk;
}

int launch_bilinear(int backward, const __nv_bfloat16* src, __nv_bfloat16* dst, int NB, int Hi, int Wi, int Ho, int Wo, int C,
                    cudaStream_t st) {
    SNN_REQUIRE(C % 8 == 0 && C >= 8, "bilinear: C=%d must be a multiple of 8", C);
    SNN_REQUIRE(NB >= 1 && Hi >= 1 && Wi >= 1 && Ho >= 1 && Wo >= 1, "bilinear: bad sizes");
    SNN_REQUIRE(((uintptr_t)src & 15) == 0 && ((uintptr_t)dst & 15) == 0, "bilinear: pointers must be 16-byte aligned");
    const float sh = (float)Hi / (float)Ho, sw = (float)Wi / (float)Wo;     // ATen area_pixel_compute_scale (align_corners=False)
    if (!backward) {
        const long long total = (long long)NB * Ho * Wo * (C / 8);
        launch_pdl(bilinear_fwd_kernel, dim3((unsigned)((total + 255) / 256)), dim3(256), 0, st, src, dst, NB, Hi, Wi, Ho, Wo, C, sh, sw);
    } else {
        const long long total = (long long)NB * Hi * Wi * (C / 8);
        launch_pdl(bilinear_bwd_kernel, dim3((unsigned)((total + 255) / 256)), dim3(256), 0, st, src, dst, NB, Hi, Wi, Ho, Wo, C, sh, sw);
    }
    return check_cuda(cudaGetLastError(), "bilinear_kernel");
}

// ------------------------------------------------------------------------------------------
// Zero-pad / crop of an NHWC bf16 tensor at the bottom / right: dst[n,h,w,:] = src[n,h,w,:] if (h < Hs && w < Ws) else 0.
// Used in front of the stride-2 convs when H or W is odd (the 15x20 P5 level of a 480x640 frame): a 3x3 stride-2 pad-1
// conv over the zero-padded even-sized map equals the conv over the odd-sized one (the extra row/column is the conv's own
// zero padding), and the crop is the pad's backward.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
pad_crop_kernel(const __nv_bfloat16* __restrict__ src, __nv_bfloat16* __restrict__ dst, int NB, int Hs, int Ws, int Hd, int Wd, int C) {
    pdl_launch_dependents();
    pdl_wait();
    const int c8 = C >> 3;
    const long long idx = (long long)blockIdx.x * 256 + threadIdx.x;
    const long long total = (long long)NB * Hd * Wd * c8;
    if (idx >= total) return;
    const int cg = (int)(idx % c8);
    const long long pix = idx / c8;
    const int w = (int)(pix % Wd), h = (int)((pix / Wd) % Hd);
    const long long n = pix / ((long long)Wd * Hd);
    uint4 v = make_uint4(0u, 0u, 0u, 0u);
    if (h < Hs && w < Ws) v = __ldg(reinterpret_cast<const uint4*>(src + ((n * Hs + h) * Ws + w) * C) + cg);
    *(reinterpret_cast<uint4*>(dst + pix * C) + cg) = v;
}

int launch_pad_crop(const __nv_bfloat16* src, __nv_bfloat16* dst, int NB, int Hs, int Ws, int Hd, int Wd, int C, cudaStream_t st) {
    SNN_REQUIRE(C % 8 == 0 && C >= 8, "pad_crop: C=%d must be a multiple of 8", C);
    SNN_REQUIRE(((uintptr_t)src & 15) == 0 && ((uintptr_t)dst & 15) == 0, "pad_crop: pointers must be 16-byte aligned");
    const long long total = (long long)NB * Hd * Wd * (C / 8);
    if (total == 0) return 0;
    launch_pdl(pad_crop_kernel, dim3((unsigned)((total + 255) / 256)), dim3(256), 0, st, src, dst, NB, Hs, Ws, Hd, Wd, C);
    return check_cuda(cudaGetLastError(), "pad_crop_kernel");
}

}  // namespace snn

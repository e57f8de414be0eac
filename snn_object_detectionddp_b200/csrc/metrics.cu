// Detection quality metrics (precision, recall, mAP50, mAP50-95) on the device: what eval_2.py:20-130 meant to compute with
// ultralytics' DetectionValidator / DetMetrics.  ultralytics is un-vendored (SURVEY.md 8c): the algorithm, with every tie
// rule fixed, is restated in oracle/det_metrics_oracle.py, which the tests compare these kernels against.
//
// det_match_kernel (per batch, one CTA per image, no host synchronisation):
//   ground-truth boxes -> pixel xyxy in shared memory; every kept NMS row finds its same-class gt of highest IoU (exact ties:
//   the higher gt index); per (gt, IoU threshold) the lowest row index claiming that gt wins (atomicMin in shared memory:
//   order-independent, so the TP masks are deterministic).  Records (conf, cls, tp mask, sort key) land at
//   *cursor + sum(counts[<b]); the last CTA (ticket counter) advances the cursor.  gt classes go into an exact int64
//   histogram; out-of-range classes bump an error counter the host reads once per evaluation.
//   IoU arithmetic is spelled out with __f*_rn so that no FMA contraction can move a pair across a threshold.
//
// det_ap_kernel + det_summary_kernel (once per evaluation, after ONE stable sort of the int64 keys
// (cls << 32) | (0x7FFFFFFF - float_bits(conf)), i.e. class-major, confidence-descending, record order on ties):
//   one CTA per class walks its segment from the END in chunks of kApThreads records (any segment length): the tp counts
//   to the right are known, so cumulative TP counts, recall, precision and the precision envelope (a suffix maximum) come
//   out of block scans; each record owns the interpolation interval [recall_i, recall_i+1) of np.interp and fills the
//   101-point AP samples that fall into it, and likewise the 1000-point P/R curves (threshold 0.5) over [-conf_i,
//   -conf_i+1).  A single CTA then averages F1 over the classes, smooths it (box filter of 101), takes the argmax and
//   writes the result vector.  Everything after the match is fp64.
#include <climits>

#include "common.cuh"

namespace snn {

constexpr int kMatchThreads = 256;
constexpr int kMatchMaxGt = 2048;
constexpr int kNumIou = 10;
constexpr int kApThreads = 512;
constexpr int kApWarps = kApThreads / 32;
constexpr int kApPoints = 101;
constexpr int kCurvePoints = 1000;
constexpr int kSummaryThreads = 1024;
constexpr int kOutHead = 8;      // out[0..7] = mp, mr, map50, map50-95, fitness, classes present, F1 argmax, error count

struct MatchParams {
    const float* rows;              // [B][max_det][6] x1 y1 x2 y2 conf cls
    const int* counts;              // [B]
    int B, max_det;
    const long long* gt_cls;        // [B][M]
    const float* gt_box;            // [B][M][4] normalised cx cy w h
    const unsigned char* gt_valid;  // [B][M]
    int M;
    float img_w, img_h;
    const float* thr;               // [10]
    int nc;
    float* rec_conf;
    int* rec_cls;
    unsigned short* rec_tp;
    long long* rec_key;
    long long cap;
    long long* cursor;
    unsigned int* ticket;
    long long* n_gt;                // [nc]
    int* err;
};

SNN_DEVINL int clamp_count(int n, int max_det) { return n < 0 ? 0 : (n > max_det ? max_det : n); }

// sum over the block of two ints (result valid in every thread)
SNN_DEVINL int2 block_sum2(int a, int b, int2* s_red) {
    for (int o = 16; o > 0; o >>= 1) {
        a += __shfl_xor_sync(0xffffffffu, a, o);
        b += __shfl_xor_sync(0xffffffffu, b, o);
    }
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (lane == 0) s_red[warp] = make_int2(a, b);
    __syncthreads();
    int2 r = make_int2(0, 0);
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) { r.x += s_red[w].x; r.y += s_red[w].y; }
    __syncthreads();
    return r;
}

__global__ void __launch_bounds__(kMatchThreads, 4) det_match_kernel(const MatchParams p) {
    pdl_launch_dependents();
    pdl_wait();
    extern __shared__ float4 s_gbox[];                        // [M] x1 y1 x2 y2, then area[M], cls[M], first[M][10]
    float* s_garea = reinterpret_cast<float*>(s_gbox + p.M);
    float* s_gcls = s_garea + p.M;                            // class as float (compared with the row's float class); NaN = invalid
    int* s_first = reinterpret_cast<int*>(s_gcls + p.M);
    __shared__ int2 s_red[kMatchThreads / 32];
    __shared__ long long s_cursor;
    __shared__ float s_thr[kNumIou];
    const int b = blockIdx.x, tid = threadIdx.x;

    // deterministic record offset: *cursor + sum of the kept rows of the images before this one
    int before = 0, total = 0;
    for (int i = tid; i < p.B; i += kMatchThreads) {
        const int c = clamp_count(p.counts[i], p.max_det);
        total += c;
        if (i < b) before += c;
    }
    const int2 sums = block_sum2(before, total, s_red);
    if (tid == 0) s_cursor = *p.cursor;
    if (tid < kNumIou) s_thr[tid] = p.thr[tid];

    // ground truth: pixel xyxy (ultralytics xywh2xyxy, then * (W, H, W, H)), area, class histogram
    for (int i = tid; i < p.M; i += kMatchThreads) {
        const size_t g = (size_t)b * p.M + i;
        float cls = __int_as_float(0x7fc00000);              // NaN: never equal to a row's class
        float4 bx = make_float4(0.f, 0.f, 0.f, 0.f);
        float area = 0.f;
        if (p.gt_valid[g]) {
            const long long c = p.gt_cls[g];
            if (c >= 0 && c < p.nc) atomicAdd(reinterpret_cast<unsigned long long*>(p.n_gt) + c, 1ull);
            else atomicAdd(p.err, 1);
            cls = (float)c;
            const float cx = p.gt_box[g * 4 + 0], cy = p.gt_box[g * 4 + 1];
            const float hw = __fdiv_rn(p.gt_box[g * 4 + 2], 2.f), hh = __fdiv_rn(p.gt_box[g * 4 + 3], 2.f);
            bx.x = __fmul_rn(__fsub_rn(cx, hw), p.img_w);
            bx.y = __fmul_rn(__fsub_rn(cy, hh), p.img_h);
            bx.z = __fmul_rn(__fadd_rn(cx, hw), p.img_w);
            bx.w = __fmul_rn(__fadd_rn(cy, hh), p.img_h);
            area = __fmul_rn(__fsub_rn(bx.z, bx.x), __fsub_rn(bx.w, bx.y));
        }
        s_gbox[i] = bx;
        s_garea[i] = area;
        s_gcls[i] = cls;
#pragma unroll
        for (int t = 0; t < kNumIou; ++t) s_first[i * kNumIou + t] = INT_MAX;
    }
    __syncthreads();

    // best same-class gt per row; the lowest row per (gt, threshold) claims it
    const int n = clamp_count(p.counts[b], p.max_det);
    const float* rows = p.rows + (size_t)b * p.max_det * 6;
    constexpr int kPer = 2;                                   // rows per thread (max_det <= 512)
    int best[kPer];
    float best_iou[kPer];
#pragma unroll
    for (int r = 0; r < kPer; ++r) {
        const int j = tid + r * kMatchThreads;
        best[r] = -1;
        best_iou[r] = 0.f;
        if (j >= n) continue;
        const float* row = rows + (size_t)j * 6;
        const float px1 = row[0], py1 = row[1], px2 = row[2], py2 = row[3], pc = row[5];
        const float parea = __fmul_rn(__fsub_rn(px2, px1), __fsub_rn(py2, py1));
        for (int i = 0; i < p.M; ++i) {
            if (s_gcls[i] != pc) continue;
            const float4 g = s_gbox[i];
            const float iw = fmaxf(__fsub_rn(fminf(g.z, px2), fmaxf(g.x, px1)), 0.f);
            const float ih = fmaxf(__fsub_rn(fminf(g.w, py2), fmaxf(g.y, py1)), 0.f);
            const float inter = __fmul_rn(iw, ih);
            const float iou = __fdiv_rn(inter, __fadd_rn(__fsub_rn(__fadd_rn(s_garea[i], parea), inter), 1e-7f));
            if (iou >= best_iou[r]) { best_iou[r] = iou; best[r] = i; }     // >=: exact ties go to the higher gt index
        }
        if (best[r] >= 0) {
#pragma unroll
            for (int t = 0; t < kNumIou; ++t)
                if (best_iou[r] >= s_thr[t]) atomicMin(&s_first[best[r] * kNumIou + t], j);
        }
    }
    __syncthreads();

    const long long base = s_cursor + sums.x;
#pragma unroll
    for (int r = 0; r < kPer; ++r) {
        const int j = tid + r * kMatchThreads;
        if (j >= n) continue;
        unsigned mask = 0;
        if (best[r] >= 0) {
#pragma unroll
            for (int t = 0; t < kNumIou; ++t)
                if (best_iou[r] >= s_thr[t] && s_first[best[r] * kNumIou + t] == j) mask |= 1u << t;
        }
        const float* row = rows + (size_t)j * 6;
        const float conf = row[4];
        const int cls = (int)row[5];
        const long long o = base + j;
        if (cls < 0 || cls >= p.nc || !(conf >= 0.f) || o >= p.cap) { atomicAdd(p.err, 1); continue; }
        p.rec_conf[o] = conf;
        p.rec_cls[o] = cls;
        p.rec_tp[o] = (unsigned short)mask;
        p.rec_key[o] = ((long long)cls << 32) | (long long)(0x7FFFFFFFu - __float_as_uint(conf));
    }

    // the last CTA to finish advances the cursor (every CTA read it before taking its ticket)
    __syncthreads();
    if (tid == 0) {
        __threadfence();
        const unsigned t = atomicAdd(p.ticket, 1u);
        if (t == gridDim.x - 1) {
            *p.cursor = s_cursor + sums.y;
            *p.ticket = 0u;
            __threadfence();
        }
    }
}

int launch_det_match(const float* rows, const int* counts, int B, int max_det, const long long* gt_cls, const float* gt_box,
                     const unsigned char* gt_valid, int M, float img_w, float img_h, const float* thr, int nc, float* rec_conf,
                     int* rec_cls, unsigned short* rec_tp, long long* rec_key, long long cap, long long* cursor,
                     unsigned int* ticket, long long* n_gt, int* err, cudaStream_t st) {
    const MatchParams p{rows, counts, B, max_det, gt_cls, gt_box, gt_valid, M, img_w, img_h, thr, nc,
                        rec_conf, rec_cls, rec_tp, rec_key, cap, cursor, ticket, n_gt, err};
    SNN_REQUIRE(p.B >= 1 && p.nc >= 1, "det_match: bad sizes (B=%d, nc=%d)", p.B, p.nc);
    SNN_REQUIRE(p.max_det >= 1 && p.max_det <= 512, "det_match: max_det=%d must be in [1, 512]", p.max_det);
    SNN_REQUIRE(p.M >= 0 && p.M <= kMatchMaxGt, "det_match: %d ground-truth slots per image > %d", p.M, kMatchMaxGt);
    const int smem = p.M * (int)(sizeof(float4) + 2 * sizeof(float) + kNumIou * sizeof(int));
    static PerDeviceOnce once;
    SNN_CUDA_OK(once.run([] {
        return cudaFuncSetAttribute(det_match_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    kMatchMaxGt * (int)(sizeof(float4) + 2 * sizeof(float) + kNumIou * sizeof(int)));
    }));
    SNN_CUDA_OK(launch_pdl(det_match_kernel, dim3(p.B), dim3(kMatchThreads), (size_t)smem, st, p));
    return check_cuda(cudaGetLastError(), "det_match_kernel");
}

// ------------------------------------------------------------------------------------------------------------------------
// AP per class
// ------------------------------------------------------------------------------------------------------------------------
struct ApParams {
    const long long* keys;          // [n] sorted ascending
    const long long* order;         // [n] record index of each sorted key
    const unsigned short* tp;       // [n] by record index
    long long n;
    const long long* n_gt;          // [nc]
    int nc;
    double* curves;                 // [2][nc][1000]: precision, recall at IoU 0.5
    double* out;                    // [8 + 11 nc]: head, ap [nc][10], present [nc]
};

SNN_DEVINL double ap_x(int k) { return k == kApPoints - 1 ? 1.0 : __dmul_rn((double)k, 0.01); }               // np.linspace(0, 1, 101)
SNN_DEVINL double curve_x(int k) { return k == kCurvePoints - 1 ? 1.0 : __dmul_rn((double)k, 1.0 / 999.0); }  // np.linspace(0, 1, 1000)

// np.interp inside one interval: xp[j] <= x < xp[j+1] (an exact hit returns fp[j])
SNN_DEVINL double interp_seg(double x, double x0, double x1, double y0, double y1) {
    if (x == x0) return y0;
    const double slope = __ddiv_rn(__dsub_rn(y1, y0), __dsub_rn(x1, x0));
    return __dadd_rn(__dmul_rn(slope, __dsub_rn(x, x0)), y0);
}

SNN_DEVINL long long lower_bound_key(const long long* keys, long long n, long long v) {
    long long lo = 0, hi = n;
    while (lo < hi) {
        const long long mid = lo + ((hi - lo) >> 1);
        if (keys[mid] < v) lo = mid + 1; else hi = mid;
    }
    return lo;
}

// inclusive prefix sum over the block of a packed counter (5 fields of 12 bits: <= 4095 per field)
SNN_DEVINL unsigned long long block_scan_u64(unsigned long long v, unsigned long long* s_w, unsigned long long& total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned long long u = __shfl_up_sync(0xffffffffu, v, o);
        if (lane >= o) v += u;
    }
    if (lane == 31) s_w[warp] = v;
    __syncthreads();
    unsigned long long pre = 0, tot = 0;
    for (int w = 0; w < kApWarps; ++w) { if (w < warp) pre += s_w[w]; tot += s_w[w]; }
    __syncthreads();
    total = tot;
    return v + pre;
}

// inclusive prefix maximum over the block
SNN_DEVINL double block_scan_max(double v, double* s_w) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int o = 1; o < 32; o <<= 1) {
        const double u = __shfl_up_sync(0xffffffffu, v, o);
        if (lane >= o) v = fmax(v, u);
    }
    if (lane == 31) s_w[warp] = v;
    __syncthreads();
    for (int w = 0; w < warp; ++w) v = fmax(v, s_w[w]);
    __syncthreads();
    return v;
}

// value of the previous thread (thread 0 gets `first`)
SNN_DEVINL double shift_up(double v, double first, double* s_w) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double u = __shfl_up_sync(0xffffffffu, v, 1);
    if (lane == 31) s_w[warp] = v;
    __syncthreads();
    if (lane == 0) u = warp == 0 ? first : s_w[warp - 1];
    __syncthreads();
    return u;
}

SNN_DEVINL unsigned field(unsigned long long lo, unsigned long long hi, int t) {
    return (unsigned)(((t < 5 ? lo : hi) >> (12 * (t < 5 ? t : t - 5))) & 0xFFFull);
}

__global__ void __launch_bounds__(kApThreads) det_ap_kernel(const ApParams p) {
    pdl_launch_dependents();
    pdl_wait();
    __shared__ double s_y[kNumIou][kApPoints];
    __shared__ double s_w[kApWarps];
    __shared__ unsigned long long s_wu[kApWarps];
    __shared__ long long s_seg[2];
    __shared__ unsigned s_total[kNumIou];
    // carry = values of the record just right of the current chunk
    __shared__ double c_rec[kNumIou], c_env[kNumIou];
    __shared__ double c_conf, c_p0;
    __shared__ unsigned c_right[kNumIou];
    const int c = blockIdx.x, tid = threadIdx.x;
    double* ap_out = p.out + kOutHead + (size_t)c * kNumIou;
    double* pc = p.curves + (size_t)c * kCurvePoints;
    double* rc = p.curves + ((size_t)p.nc + c) * kCurvePoints;
    const long long n_l = p.n_gt[c];
    if (n_l <= 0) {                                           // not a target class: not part of the mean
        if (tid < kNumIou) ap_out[tid] = 0.0;
        if (tid == 0) p.out[kOutHead + (size_t)p.nc * kNumIou + c] = 0.0;
        return;
    }
    if (tid == 0) {
        p.out[kOutHead + (size_t)p.nc * kNumIou + c] = 1.0;
        s_seg[0] = lower_bound_key(p.keys, p.n, (long long)c << 32);
        s_seg[1] = lower_bound_key(p.keys, p.n, (long long)(c + 1) << 32);
    }
    for (int i = tid; i < kNumIou * kApPoints; i += kApThreads) (&s_y[0][0])[i] = 0.0;
    __syncthreads();
    const long long s0 = s_seg[0], n_p = s_seg[1] - s_seg[0];
    if (n_p == 0) {                                           // gts but no predictions: AP 0, curves 0
        if (tid < kNumIou) ap_out[tid] = 0.0;
        for (int k = tid; k < kCurvePoints; k += kApThreads) { pc[k] = 0.0; rc[k] = 0.0; }
        return;
    }

    // pass 1: TP totals per threshold
    unsigned cnt[kNumIou];
#pragma unroll
    for (int t = 0; t < kNumIou; ++t) cnt[t] = 0;
    for (long long i = tid; i < n_p; i += kApThreads) {
        const unsigned m = p.tp[p.order[s0 + i]];
#pragma unroll
        for (int t = 0; t < kNumIou; ++t) cnt[t] += (m >> t) & 1u;
    }
    if (tid < kNumIou) { s_total[tid] = 0; c_right[tid] = 0; c_rec[tid] = 1.0; c_env[tid] = 0.0; }
    if (tid == 0) { c_conf = 0.0; c_p0 = 0.0; }
    __syncthreads();
#pragma unroll
    for (int t = 0; t < kNumIou; ++t) {
        unsigned v = cnt[t];
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if ((tid & 31) == 0) atomicAdd(&s_total[t], v);
    }
    __syncthreads();

    const double dn_l = (double)n_l;                          // n_l + 1e-16 == n_l in fp64 for n_l >= 1
    // pass 2: chunks from the end; thread tid holds record i = end - 1 - tid, so suffixes are block prefixes
    for (long long end = n_p; end > 0; end -= kApThreads) {
        const long long start = end - kApThreads > 0 ? end - kApThreads : 0;
        const long long i = end - 1 - tid;
        const bool valid = i >= start;
        const bool last_rec = i == n_p - 1;
        unsigned m = 0;
        double conf = 0.0;
        if (valid) {
            const long long key = p.keys[s0 + i];
            m = p.tp[p.order[s0 + i]];
            conf = (double)__uint_as_float(0x7FFFFFFFu - (unsigned)(key & 0xFFFFFFFFll));
        }
        unsigned long long lo = 0, hi = 0;
#pragma unroll
        for (int t = 0; t < 5; ++t) { lo |= (unsigned long long)((m >> t) & 1u) << (12 * t); hi |= (unsigned long long)((m >> (t + 5)) & 1u) << (12 * t); }
        unsigned long long tot_lo, tot_hi;
        const unsigned long long suf_lo = block_scan_u64(lo, s_wu, tot_lo);      // TPs in [i, end)
        const unsigned long long suf_hi = block_scan_u64(hi, s_wu, tot_hi);
        const double prev_conf = shift_up(conf, c_conf, s_w);                    // conf of record i + 1
        for (int t = 0; t < kNumIou; ++t) {
            // cumulative TPs up to and including i = total - TPs right of i
            const unsigned right = c_right[t] + field(suf_lo, suf_hi, t) - ((m >> t) & 1u);
            const double tpc = (double)(s_total[t] - right);
            const double rec = valid ? __ddiv_rn(tpc, dn_l) : 0.0;
            const double prec = valid ? __ddiv_rn(tpc, (double)(i + 1)) : 0.0;
            const double env = fmax(block_scan_max(prec, s_w), c_env[t]);       // max precision over [i, n_p)
            const double rec1 = shift_up(rec, c_rec[t], s_w);                    // recall of i + 1 (1.0 past the end)
            const double env1 = shift_up(env, c_env[t], s_w);                    // envelope of i + 1 (0.0 past the end)
            const double prec1 = t == 0 ? shift_up(prec, c_p0, s_w) : 0.0;
            if (valid) {
                const double x1 = last_rec ? 1.0 : rec1, y1 = last_rec ? 0.0 : env1;
                // AP samples: record i owns [recall_i, recall_i+1) of mrec = [0, recall..., 1]
                int k = max(0, (int)(rec * 100.0) - 1);
                while (k < kApPoints && ap_x(k) < rec) ++k;
                for (; k < kApPoints && ap_x(k) < x1; ++k) s_y[t][k] = interp_seg(ap_x(k), rec, x1, env, y1);
                if (i == 0) {                                                    // the leading pad: mrec 0, mpre 1
                    for (k = 0; k < kApPoints && ap_x(k) < rec; ++k) s_y[t][k] = interp_seg(ap_x(k), 0.0, rec, 1.0, env);
                }
                if (t == 0) {
                    // P/R curves: np.interp(-x, -conf, ., left=0 | 1); record i owns -x in [-conf_i, -conf_i+1)
                    int q = last_rec ? 0 : max(0, (int)(prev_conf * 999.0) - 1);
                    if (!last_rec) while (q < kCurvePoints && !(-curve_x(q) < -prev_conf)) ++q;
                    for (; q < kCurvePoints && -curve_x(q) >= -conf; ++q) {
                        const double xq = -curve_x(q);
                        if (last_rec) { pc[q] = prec; rc[q] = rec; }
                        else { pc[q] = interp_seg(xq, -conf, -prev_conf, prec, prec1); rc[q] = interp_seg(xq, -conf, -prev_conf, rec, rec1); }
                    }
                    if (i == 0)
                        for (q = kCurvePoints - 1; q >= 0 && -curve_x(q) < -conf; --q) { pc[q] = 1.0; rc[q] = 0.0; }
                }
            }
            __syncthreads();
            if (i == start) {                                                    // leftmost record: carry for the next chunk
                c_rec[t] = rec; c_env[t] = env;
                if (t == 0) { c_p0 = prec; c_conf = conf; }
            }
        }
        __syncthreads();
        if (tid < kNumIou) c_right[tid] += field(tot_lo, tot_hi, tid);
        __syncthreads();
    }

    // np.trapezoid(y, x): d * (y[1:] + y[:-1]) / 2, summed as numpy's pairwise add (8 accumulators below 128 terms)
    if (tid < kNumIou) {
        const int t = tid;
        double r[8];
        auto term = [&](int k) {
            return __ddiv_rn(__dmul_rn(__dsub_rn(ap_x(k + 1), ap_x(k)), __dadd_rn(s_y[t][k + 1], s_y[t][k])), 2.0);
        };
        for (int j = 0; j < 8; ++j) r[j] = term(j);
        int k = 8;
        for (; k < 96; k += 8)
            for (int j = 0; j < 8; ++j) r[j] = __dadd_rn(r[j], term(k + j));
        double res = __dadd_rn(__dadd_rn(__dadd_rn(r[0], r[1]), __dadd_rn(r[2], r[3])), __dadd_rn(__dadd_rn(r[4], r[5]), __dadd_rn(r[6], r[7])));
        for (; k < kApPoints - 1; ++k) res = __dadd_rn(res, term(k));
        ap_out[t] = res;
    }
}

__global__ void __launch_bounds__(kSummaryThreads) det_summary_kernel(const double* curves, double* out, int nc, const int* err) {
    pdl_launch_dependents();
    pdl_wait();
    __shared__ double s_f1[kCurvePoints];
    __shared__ double s_v[kSummaryThreads];
    __shared__ int s_i[kSummaryThreads];
    const int tid = threadIdx.x;
    const double* present = out + kOutHead + (size_t)nc * kNumIou;
    int npres = 0;
    for (int c = 0; c < nc; ++c) npres += present[c] != 0.0;
    // f1.mean(0) over the target classes, f1 = 2 p r / (p + r + 1e-16)
    for (int k = tid; k < kCurvePoints; k += kSummaryThreads) {
        double s = 0.0;
        for (int c = 0; c < nc; ++c) {
            if (present[c] == 0.0) continue;
            const double pp = curves[(size_t)c * kCurvePoints + k], rr = curves[((size_t)nc + c) * kCurvePoints + k];
            s = __dadd_rn(s, __ddiv_rn(__dmul_rn(__dmul_rn(2.0, pp), rr), __dadd_rn(__dadd_rn(pp, rr), 1e-16)));
        }
        s_f1[k] = npres ? __ddiv_rn(s, (double)npres) : 0.0;
    }
    __syncthreads();
    // smooth(y, 0.1): 50 edge copies each side, box filter of 101 taps of 1/101; first argmax
    double v = -1.0;
    if (tid < kCurvePoints) {
        const double w = 1.0 / 101.0;
        double s = 0.0;
        for (int m = 0; m < 101; ++m) {
            const int q = min(max(tid + m - 50, 0), kCurvePoints - 1);
            s = __dadd_rn(s, __dmul_rn(s_f1[q], w));
        }
        v = s;
    }
    s_v[tid] = v;
    s_i[tid] = tid;
    __syncthreads();
    for (int o = kSummaryThreads / 2; o > 0; o >>= 1) {
        if (tid < o) {
            const double a = s_v[tid], b = s_v[tid + o];
            if (b > a || (b == a && s_i[tid + o] < s_i[tid])) { s_v[tid] = b; s_i[tid] = s_i[tid + o]; }
        }
        __syncthreads();
    }
    if (tid == 0) {
        const int idx = npres ? s_i[0] : 0;
        double mp = 0.0, mr = 0.0, m50 = 0.0, mall = 0.0;
        for (int c = 0; c < nc; ++c) {
            if (present[c] == 0.0) continue;
            mp = __dadd_rn(mp, curves[(size_t)c * kCurvePoints + idx]);
            mr = __dadd_rn(mr, curves[((size_t)nc + c) * kCurvePoints + idx]);
            m50 = __dadd_rn(m50, out[kOutHead + (size_t)c * kNumIou]);
            for (int t = 0; t < kNumIou; ++t) mall = __dadd_rn(mall, out[kOutHead + (size_t)c * kNumIou + t]);
        }
        if (npres) {
            mp = __ddiv_rn(mp, (double)npres); mr = __ddiv_rn(mr, (double)npres);
            m50 = __ddiv_rn(m50, (double)npres); mall = __ddiv_rn(mall, (double)npres * kNumIou);
        }
        out[0] = mp; out[1] = mr; out[2] = m50; out[3] = mall;
        out[4] = __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(0.0, mp), __dmul_rn(0.0, mr)), __dmul_rn(0.1, m50)), __dmul_rn(0.9, mall));
        out[5] = (double)npres;
        out[6] = (double)idx;
        out[7] = (double)*err;
    }
}

int launch_det_metrics_finalize(const long long* keys, const long long* order, const unsigned short* tp, long long n,
                                const long long* n_gt, int nc, const int* err, double* curves, double* out, cudaStream_t st) {
    const ApParams p{keys, order, tp, n, n_gt, nc, curves, out};
    SNN_REQUIRE(p.nc >= 1 && p.n >= 0, "det_metrics_finalize: bad sizes (nc=%d)", p.nc);
    SNN_CUDA_OK(launch_pdl(det_ap_kernel, dim3(p.nc), dim3(kApThreads), 0, st, p));
    SNN_CUDA_OK(cudaGetLastError());
    SNN_CUDA_OK(launch_pdl(det_summary_kernel, dim3(1), dim3(kSummaryThreads), 0, st, (const double*)p.curves, p.out, p.nc, err));
    return check_cuda(cudaGetLastError(), "det_summary_kernel");
}

}  // namespace snn

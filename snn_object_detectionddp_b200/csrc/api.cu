// extern "C" boundary of libsnnb200.so (declared in include/snn_b200.h).
#include <stdarg.h>

#include <atomic>
#include <mutex>
#include <stdio.h>

#include "../../include/snn_b200.h"
#include "common.cuh"

namespace snn {

static thread_local char g_err[1024] = "";

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}
int check_cuda(cudaError_t e, const char* what) {
    if (e == cudaSuccess) return 0;
    set_error("CUDA error %d (%s) at %s", (int)e, cudaGetErrorString(e), what);
    return 1;
}
int current_device() {
    int dev = 0;
    return cudaGetDevice(&dev) == cudaSuccess ? dev : -1;
}
int num_sms() {
    static std::atomic<int> cache[64];      // zero-initialised; per device ordinal
    const int dev = current_device();
    if (dev >= 0 && dev < 64) {
        const int c = cache[dev].load(std::memory_order_relaxed);
        if (c > 0) return c;
    }
    int n = 0;
    if (dev < 0 || cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
    if (dev >= 0 && dev < 64) cache[dev].store(n, std::memory_order_relaxed);
    return n;
}

static std::atomic<int> g_pdl{0};
bool pdl_enabled() { return g_pdl.load(std::memory_order_relaxed) != 0; }
void set_pdl(int on) { g_pdl.store(on ? 1 : 0, std::memory_order_relaxed); }

static std::atomic<int> g_det{0};
bool deterministic() { return g_det.load(std::memory_order_relaxed) != 0; }
void set_deterministic(int on) { g_det.store(on ? 1 : 0, std::memory_order_relaxed); }

static void* g_det_ws[64];
static size_t g_det_ws_bytes[64];
static std::mutex g_det_mutex;
void* det_scratch(size_t bytes, cudaStream_t st) {
    const int dev = current_device();
    if (dev < 0 || dev >= 64) { set_error("deterministic mode: bad CUDA device %d", dev); return nullptr; }
    std::lock_guard<std::mutex> g(g_det_mutex);
    if (g_det_ws_bytes[dev] >= bytes) return g_det_ws[dev];
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    if (cudaStreamIsCapturing(st, &cs) != cudaSuccess || cs != cudaStreamCaptureStatusNone) {
        set_error("deterministic mode: the scratch buffer (%zu bytes) must be allocated outside CUDA-graph capture: run the step once eagerly first", bytes);
        return nullptr;
    }
    size_t want = bytes < ((size_t)64 << 20) ? ((size_t)64 << 20) : bytes;
    void* q = nullptr;
    if (cudaDeviceSynchronize() != cudaSuccess || cudaMalloc(&q, want) != cudaSuccess) {
        set_error("deterministic mode: cudaMalloc(%zu) failed", want);
        return nullptr;
    }
    if (g_det_ws[dev]) cudaFree(g_det_ws[dev]);
    g_det_ws[dev] = q; g_det_ws_bytes[dev] = want;
    return q;
}

// launchers defined in the other translation units
void debug_set(int k, int v);
void set_dynamic_tiles(int on);
void tmap_cache_stats(unsigned long long*, unsigned long long*);
int conv_plan(int, int, int, int, int, int, int, int, int, int, int*);
int conv_fprop(int, int, int, int, const void*, int, long long, const void*, int, long long, const void*, int, int, int, int,
               int, const float*, void*, int, long long, int, int, cudaStream_t, float*, int);
long long conv_stats_groups(int, int, int, int, int, int*);
long long nms_workspace_keys(int, int, int);
int launch_nms(const float*, int, int, int, float, float, int, int, int, int, float, unsigned long long*, long long, float*, int*,
               int*, cudaStream_t);
int launch_bn_stats_from_partials(const float*, double*, int, int, int, cudaStream_t);
int launch_bn_finalize_partials(const float*, double*, double*, const float*, const float*, float*, float*, long long*, float*, float*,
                                float*, float*, unsigned int*, int, int, int, int, float, float, cudaStream_t);
long long bn_finalize_workspace_doubles(int, int, int);
int conv_dgrad(int, int, int, int, const void*, int, long long, const void*, int, int, int, void*, int, long long, int, int,
               cudaStream_t);
int conv_wgrad(int, int, int, int, const void*, int, long long, const void*, int, long long, float*, int, int, cudaStream_t);
int launch_weight_prep(const float*, __nv_bfloat16*, __nv_bfloat16*, int, int, int, cudaStream_t);
int launch_bn_stats(const float*, double*, float*, int, int, int, cudaStream_t);
long long bn_stats_workspace_floats(int, int, int);
int launch_bn_finalize(const double*, const float*, const float*, float*, float*, float*, float*, float*, float*, int, int, int,
                       float, float, int, cudaStream_t);
int launch_bn_act_fwd(int, const float*, const float*, const float*, const float*, __nv_bfloat16*, uint8_t*, float*, int,
                      long long, int, int, float, float, cudaStream_t);
int launch_bn_act_fwd_count(const float*, const float*, const float*, const float*, __nv_bfloat16*, uint8_t*, float*,
                            unsigned long long*, unsigned long long*, int, long long, int, int, float, float, cudaStream_t);
int launch_bn_act_bwd(int, int, const float*, const float*, const float*, const float*, const float*, const float*,
                      const __nv_bfloat16*, const float*, float*, __nv_bfloat16*, float*, float*, int, int, int, int, float,
                      float, float, cudaStream_t);
int launch_bn_act_bwd2(int, int, const float*, const float*, const float*, const float*, const float*, const float*,
                       const float*, const __nv_bfloat16*, const float*, float*, __nv_bfloat16*, float*, float*, float*, int, int,
                       int, float, float, float, cudaStream_t);
int launch_bn_bwd_dx(const float*, const float*, const float*, const float*, const float*, const float*, const float*, float*,
                     float*, float*, __nv_bfloat16*, int, int, int, cudaStream_t);
int launch_lstm_gates_fwd(const float*, const float*, float*, float*, __nv_bfloat16*, long long, int, cudaStream_t);
int launch_lstm_gates_bwd(const float*, const float*, const float*, const float*, const __nv_bfloat16*, const float*, __nv_bfloat16*,
                          float*, long long, int, cudaStream_t);
int launch_nchw_to_nhwc(const float*, void*, int, int, int, int, long long, int, cudaStream_t);
int launch_nhwc_to_nchw(const void*, int, float*, int, int, int, long long, int, cudaStream_t);
int launch_sumsq(const float*, long long, double*, int, cudaStream_t);
int launch_colsum_bf16(const __nv_bfloat16*, float*, long long, int, cudaStream_t);
int launch_dw3x3_fwd(const __nv_bfloat16*, const float*, float*, int, int, int, int, float*, int, cudaStream_t);
long long dw3x3_stats_blocks(int, int, int);
int launch_dw3x3_dgrad(const __nv_bfloat16*, const float*, __nv_bfloat16*, int, int, int, int, cudaStream_t);
int launch_dw3x3_wgrad(const __nv_bfloat16*, const __nv_bfloat16*, float*, int, int, int, int, cudaStream_t);
int launch_s2d8(const float*, __nv_bfloat16*, int, int, int, int, cudaStream_t);
int launch_s2d8_u8(const uint8_t*, __nv_bfloat16*, int, int, int, int, cudaStream_t);
int launch_adamw(float*, float*, float*, float*, __nv_bfloat16*, long long, const float*, const double*, float*,
                 int*, int, int, cudaStream_t);
int launch_bilinear(int, const __nv_bfloat16*, __nv_bfloat16*, int, int, int, int, int, int, cudaStream_t);
int launch_pad_crop(const __nv_bfloat16*, __nv_bfloat16*, int, int, int, int, int, int, cudaStream_t);
int launch_detect_decode(const float*, const float*, const float*, const float*, int, int, int, int, int, float*, float*, int,
                         const int*, cudaStream_t);
int launch_detect_loss_fwd(const float*, const float*, const float*, const float*, const float*, const float*, const uint8_t*,
                           int, int, int, int, double*, int, const int*, const float*, int, const float*, unsigned int*, float*,
                           float*, cudaStream_t);
int launch_detect_loss_bwd(const float*, const float*, const float*, const float*, const float*, const float*, const uint8_t*,
                           int, int, int, int, const float*, const float*, void*, void*, int, int, const int*, cudaStream_t);
long long tal_workspace_bytes(int, int, int);
int launch_tal_assign(const float*, const float*, const float*, const float*, const long long*, const float*, const uint8_t*, float,
                      float, int, int, int, int, int, void*, float*, float*, uint8_t*, float**, int*, cudaStream_t);

int launch_det_match(const float*, const int*, int, int, const long long*, const float*, const unsigned char*, int, float, float,
                     const float*, int, float*, int*, unsigned short*, long long*, long long, long long*, unsigned int*,
                     long long*, int*, cudaStream_t);
int launch_det_metrics_finalize(const long long*, const long long*, const unsigned short*, long long, const long long*, int,
                                const int*, double*, double*, cudaStream_t);

}  // namespace snn

using namespace snn;
#define ST ((cudaStream_t)stream)

extern "C" {

const char* snn_last_error(void) { return g_err; }
int snn_version(void) { return 100; }
void snn_debug_set(int key, int value) { debug_set(key, value); }
void snn_set_tile_scheduling(int dynamic) { set_dynamic_tiles(dynamic); }
int snn_conv_plan(int kind, int geom, int NB, int H, int W, int Cin, int Cout, int out_f32, int frames_per_step, int accumulate, int* out20) {
    return conv_plan(kind, geom, NB, H, W, Cin, Cout, out_f32, frames_per_step, accumulate, out20);
}
void snn_set_deterministic(int on) { set_deterministic(on); }
int snn_get_deterministic(void) { return deterministic() ? 1 : 0; }
void snn_set_dependent_launch(int on) { set_pdl(on); }
int snn_get_dependent_launch(void) { return pdl_enabled() ? 1 : 0; }
void snn_tensor_map_cache_stats(unsigned long long* hits, unsigned long long* misses) { tmap_cache_stats(hits, misses); }

int snn_conv_fprop(int geom, int NB, int H, int W, const void* x0, int C0, long long ld0, const void* x1, int C1,
                   long long ld1, const void* w, int w_rows, int w_K, int w_coff, int Cout, int w_row_off,
                   const float* bias, void* out, int out_is_f32, long long out_ld, int out_coff, int accumulate,
                   void* stream) {
    return conv_fprop(geom, NB, H, W, x0, C0, ld0, x1, C1, ld1, w, w_rows, w_K, w_coff, Cout, w_row_off, bias, out,
                      out_is_f32, out_ld, out_coff, accumulate, ST, nullptr, 0);
}
long long snn_conv_stats_groups(int geom, int NB, int H, int W, int frames_per_step, int* groups_per_step) {
    return conv_stats_groups(geom, NB, H, W, frames_per_step, groups_per_step);
}
int snn_conv_fprop_stats(int geom, int NB, int H, int W, const void* x0, int C0, long long ld0, const void* x1, int C1,
                         long long ld1, const void* w, int w_rows, int w_K, int w_coff, int Cout, int w_row_off, float* out,
                         int frames_per_step, float* partials, void* stream) {
    return conv_fprop(geom, NB, H, W, x0, C0, ld0, x1, C1, ld1, w, w_rows, w_K, w_coff, Cout, w_row_off, nullptr, out, 1,
                      Cout, 0, 0, ST, partials, frames_per_step);
}
long long snn_nms_workspace_keys(int nc, int A, int multi_label) { return nms_workspace_keys(nc, A, multi_label && nc > 1); }
int snn_nms(const float* pred, int B, int nc, int A, float conf_thres, float iou_thres, int multi_label, int agnostic,
            int max_det, int max_nms, float max_wh, unsigned long long* keys, long long keys_per_image, float* out,
            int* out_idx, int* counts, void* stream) {
    return launch_nms(pred, B, nc, A, conf_thres, iou_thres, multi_label, agnostic, max_det, max_nms, max_wh, keys,
                      keys_per_image, out, out_idx, counts, ST);
}
int snn_det_match(const float* rows, const int* counts, int B, int max_det, const long long* gt_cls, const float* gt_box,
                  const unsigned char* gt_valid, int M, float img_w, float img_h, const float* iou_thres, int nc,
                  float* rec_conf, int* rec_cls, unsigned short* rec_tp, long long* rec_key, long long capacity,
                  long long* cursor, unsigned int* ticket, long long* n_gt, int* err, void* stream) {
    return launch_det_match(rows, counts, B, max_det, gt_cls, gt_box, gt_valid, M, img_w, img_h, iou_thres, nc, rec_conf, rec_cls,
                            rec_tp, rec_key, capacity, cursor, ticket, n_gt, err, ST);
}
int snn_det_metrics_finalize(const long long* keys, const long long* order, const unsigned short* rec_tp, long long n,
                             const long long* n_gt, int nc, const int* err, double* curves, double* out, void* stream) {
    return launch_det_metrics_finalize(keys, order, rec_tp, n, n_gt, nc, err, curves, out, ST);
}
long long snn_bn_finalize_workspace_doubles(int T, int C, int groups_per_step) { return bn_finalize_workspace_doubles(T, C, groups_per_step); }
int snn_bn_finalize_partials(const float* partials, double* sums, double* workspace, const float* gamma, const float* beta,
                             float* running_mean, float* running_var, long long* num_batches_tracked, float* scale, float* shift,
                             float* mean, float* invstd, unsigned int* counters, int T, int C, int P, int groups_per_step, float eps,
                             float momentum, void* stream) {
    return launch_bn_finalize_partials(partials, sums, workspace, gamma, beta, running_mean, running_var, num_batches_tracked, scale,
                                       shift, mean, invstd, counters, T, C, P, groups_per_step, eps, momentum, ST);
}
int snn_bn_stats_from_partials(const float* partials, double* sums, int T, int C, int groups_per_step, void* stream) {
    return launch_bn_stats_from_partials(partials, sums, T, C, groups_per_step, ST);
}
int snn_conv_dgrad(int geom, int NB, int H, int W, const void* dy, int Cout, long long ld_dy, const void* wt, int wt_rows,
                   int ci_off, int Ci, void* dx, int dx_is_f32, long long dx_ld, int dx_coff, int accumulate, void* stream) {
    return conv_dgrad(geom, NB, H, W, dy, Cout, ld_dy, wt, wt_rows, ci_off, Ci, dx, dx_is_f32, dx_ld, dx_coff, accumulate, ST);
}
int snn_conv_wgrad(int geom, int NB, int H, int W, const void* x, int Ci, long long ld_x, const void* dy, int Cout,
                   long long ld_dy, float* dw, int w_K, int w_coff, void* stream) {
    return conv_wgrad(geom, NB, H, W, x, Ci, ld_x, dy, Cout, ld_dy, dw, w_K, w_coff, ST);
}
int snn_weight_prep(const float* w, void* wf, void* wt, int N, int T, int K, void* stream) {
    return launch_weight_prep(w, (__nv_bfloat16*)wf, (__nv_bfloat16*)wt, N, T, K, ST);
}
int snn_bn_stats(const float* y, double* sums, float* workspace, int T, int P, int C, void* stream) {
    return launch_bn_stats(y, sums, workspace, T, P, C, ST);
}
long long snn_bn_stats_workspace_floats(int T, int P, int C) { return bn_stats_workspace_floats(T, P, C); }
int snn_bn_finalize(const double* sums, const float* gamma, const float* beta, float* rm, float* rv, float* scale,
                    float* shift, float* mean, float* invstd, int T, int C, int P, float eps, float momentum, int training,
                    void* stream) {
    return launch_bn_finalize(sums, gamma, beta, rm, rv, scale, shift, mean, invstd, T, C, P, eps, momentum, training, ST);
}
int snn_bn_act_fwd(int act, const float* y, const float* scale, const float* shift, const float* v_init, void* out,
                   uint8_t* mask, float* v_final, int T, long long n_per_t, int C, int ss_stride_t, float beta, float theta,
                   void* stream) {
    return launch_bn_act_fwd(act, y, scale, shift, v_init, (__nv_bfloat16*)out, mask, v_final, T, n_per_t, C, ss_stride_t,
                             beta, theta, ST);
}
int snn_bn_act_fwd_count(const float* y, const float* scale, const float* shift, const float* v_init, void* out, uint8_t* mask,
                         float* v_final, unsigned long long* spikes, unsigned long long* steps, int T, long long n_per_t, int C,
                         int ss_stride_t, float beta, float theta, void* stream) {
    return launch_bn_act_fwd_count(y, scale, shift, v_init, (__nv_bfloat16*)out, mask, v_final, spikes, steps, T, n_per_t, C,
                                   ss_stride_t, beta, theta, ST);
}
int snn_bn_act_bwd(int act, int training, const float* y, const float* scale, const float* shift, const float* mean,
                   const float* invstd, const float* v_init, const void* gs, const float* gv_final, float* gx, void* dy,
                   float* gv_init, float* red, int T, int P, int C, int ss_stride_t, float beta, float theta, float alpha,
                   void* stream) {
    return launch_bn_act_bwd(act, training, y, scale, shift, mean, invstd, v_init, (const __nv_bfloat16*)gs, gv_final, gx,
                             (__nv_bfloat16*)dy, gv_init, red, T, P, C, ss_stride_t, beta, theta, alpha, ST);
}
int snn_bn_act_bwd2(int pass, int act, const float* y, const float* scale, const float* shift, const float* mean,
                    const float* invstd, const float* beta_bn, const float* v_init, const void* gs, const float* gv_final,
                    float* red, void* dy, float* gv_init, float* dgamma, float* dbeta, int T, int P, int C, float beta,
                    float theta, float alpha, void* stream) {
    return launch_bn_act_bwd2(pass, act, y, scale, shift, mean, invstd, beta_bn, v_init, (const __nv_bfloat16*)gs, gv_final,
                              red, (__nv_bfloat16*)dy, gv_init, dgamma, dbeta, T, P, C, beta, theta, alpha, ST);
}
int snn_bn_bwd_dx(const float* red, const float* gamma, const float* gx, const float* y, const float* scale,
                  const float* mean, const float* invstd, float* coef, float* dgamma, float* dbeta, void* dy, int T, int P,
                  int C, void* stream) {
    return launch_bn_bwd_dx(red, gamma, gx, y, scale, mean, invstd, coef, dgamma, dbeta, (__nv_bfloat16*)dy, T, P, C, ST);
}
int snn_lstm_gates_fwd(const float* gates, const float* c_prev, float* c_next, float* h_next, void* h_bf16, long long P,
                       int Ch, void* stream) {
    return launch_lstm_gates_fwd(gates, c_prev, c_next, h_next, (__nv_bfloat16*)h_bf16, P, Ch, ST);
}
int snn_lstm_gates_bwd(const float* gates, const float* c_prev, const float* c_next, const float* dh, const void* dh_bf16,
                       const float* dc_in, void* dgates, float* dc_prev, long long P, int Ch, void* stream) {
    return launch_lstm_gates_bwd(gates, c_prev, c_next, dh, (const __nv_bfloat16*)dh_bf16, dc_in, (__nv_bfloat16*)dgates, dc_prev, P, Ch, ST);
}
int snn_nchw_to_nhwc(const float* in, void* out, int out_is_bf16, int NB, int C, int HW, long long out_ld, int out_coff,
                     void* stream) {
    return launch_nchw_to_nhwc(in, out, out_is_bf16, NB, C, HW, out_ld, out_coff, ST);
}
int snn_nhwc_to_nchw(const void* in, int in_is_bf16, float* out, int NB, int C, int HW, long long in_ld, int in_coff,
                     void* stream) {
    return launch_nhwc_to_nchw(in, in_is_bf16, out, NB, C, HW, in_ld, in_coff, ST);
}
int snn_dw3x3_fprop(const void* x, const float* w, float* y, int NB, int H, int W, int C, void* stream) {
    return launch_dw3x3_fwd((const __nv_bfloat16*)x, w, y, NB, H, W, C, nullptr, 0, ST);
}
long long snn_dw3x3_stats_blocks(int frames_per_step, int W, int C) { return dw3x3_stats_blocks(frames_per_step, W, C); }
int snn_dw3x3_fprop_stats(const void* x, const float* w, float* y, int NB, int H, int W, int C, int T, float* partials, void* stream) {
    return launch_dw3x3_fwd((const __nv_bfloat16*)x, w, y, NB, H, W, C, partials, T, ST);
}
int snn_dw3x3_dgrad(const void* dy, const float* w, void* dx, int NB, int H, int W, int C, void* stream) {
    return launch_dw3x3_dgrad((const __nv_bfloat16*)dy, w, (__nv_bfloat16*)dx, NB, H, W, C, ST);
}
int snn_dw3x3_wgrad(const void* x, const void* dy, float* dw, int NB, int H, int W, int C, void* stream) {
    return launch_dw3x3_wgrad((const __nv_bfloat16*)x, (const __nv_bfloat16*)dy, dw, NB, H, W, C, ST);
}
int snn_space_to_depth8(const float* frames, void* out, int B, int T, int H, int W, void* stream) {
    return launch_s2d8(frames, (__nv_bfloat16*)out, B, T, H, W, ST);
}
int snn_space_to_depth8_u8(const unsigned char* frames, void* out, int B, int T, int H, int W, void* stream) {
    return launch_s2d8_u8(frames, (__nv_bfloat16*)out, B, T, H, W, ST);
}
int snn_bilinear_resize(int backward, const void* src, void* dst, int NB, int Hi, int Wi, int Ho, int Wo, int C, void* stream) {
    return launch_bilinear(backward, (const __nv_bfloat16*)src, (__nv_bfloat16*)dst, NB, Hi, Wi, Ho, Wo, C, ST);
}
int snn_nhwc_pad_crop(const void* src, void* dst, int NB, int Hs, int Ws, int Hd, int Wd, int C, void* stream) {
    return launch_pad_crop((const __nv_bfloat16*)src, (__nv_bfloat16*)dst, NB, Hs, Ws, Hd, Wd, C, ST);
}
int snn_colsum_bf16(const void* dy, float* acc, long long P, int C, void* stream) {
    return launch_colsum_bf16((const __nv_bfloat16*)dy, acc, P, C, ST);
}
int snn_grad_sumsq(const float* g, long long n, double* acc, int zero_first, void* stream) {
    return launch_sumsq(g, n, acc, zero_first, ST);
}
int snn_adamw_step(float* p, float* g, float* m, float* v, void* shadow, long long n, const float* hp,
                   const double* sumsq, float* gnorm_out, int* step_ptr, int n_rows, int zero_grad, void* stream) {
    return launch_adamw(p, g, m, v, (__nv_bfloat16*)shadow, n, hp, sumsq, gnorm_out, step_ptr, n_rows, zero_grad, ST);
}
int snn_detect_decode(const float* distri, const float* scores, const float* anchors, const float* stride, int B, int A,
                      int nc, int reg_max, int xywh, float* boxes, float* probs, void* stream) {
    return launch_detect_decode(distri, scores, anchors, stride, B, A, nc, reg_max, xywh, boxes, probs, 0, nullptr, ST);
}
int snn_detect_loss_fwd(const float* distri, const float* scores, const float* anchors, const float* stride,
                        const float* tbox_px, const float* tscores, const uint8_t* fg, int B, int A, int nc, int reg_max,
                        double* sums, void* stream) {
    return launch_detect_loss_fwd(distri, scores, anchors, stride, tbox_px, tscores, fg, B, A, nc, reg_max, sums, 0, nullptr, nullptr, 0,
                                  nullptr, nullptr, nullptr, nullptr, ST);
}
int snn_detect_loss_bwd(const float* distri, const float* scores, const float* anchors, const float* stride,
                        const float* tbox_px, const float* tscores, const uint8_t* fg, int B, int A, int nc, int reg_max,
                        const float* coef, float* g_distri, float* g_scores, void* stream) {
    return launch_detect_loss_bwd(distri, scores, anchors, stride, tbox_px, tscores, fg, B, A, nc, reg_max, coef, nullptr, g_distri,
                                  g_scores, 0, 0, nullptr, ST);
}
long long snn_tal_workspace_bytes(int B, int A, int M) { return tal_workspace_bytes(B, A, M); }
int snn_detect_assign_loss_fwd(const float* distri, const float* scores, int nl, const int* a_off, const float* anchors,
                               const float* stride, const long long* gt_cls, const float* gt_box, const unsigned char* gt_valid,
                               float img_w, float img_h, int B, int A, int M, int nc, int reg_max, int topk, const float* gains,
                               void* workspace, float* pboxes, float* probs, float* tbox_px, float* tscores, unsigned char* fg,
                               double* sums, unsigned int* counter, float* out6, float* coef3, void* stream) {
    int rc = launch_detect_decode(distri, scores, anchors, stride, B, A, nc, reg_max, 0, pboxes, probs, nl, a_off, ST);
    if (rc) return rc;
    float* tss_part = nullptr;
    int n_parts = 0;
    rc = launch_tal_assign(probs, pboxes, anchors, stride, gt_cls, gt_box, gt_valid, img_w, img_h, B, A, M, nc, topk, workspace, tbox_px,
                           tscores, fg, &tss_part, &n_parts, ST);
    if (rc) return rc;
    return launch_detect_loss_fwd(distri, scores, anchors, stride, tbox_px, tscores, fg, B, A, nc, reg_max, sums, nl, a_off, tss_part,
                                  n_parts, gains, counter, out6, coef3, ST);
}
int snn_tal_assign(const float* probs, const float* pboxes, const float* anchors, const float* stride, const long long* gt_cls,
                   const float* gt_box, const unsigned char* gt_valid, float img_w, float img_h, int B, int A, int M, int nc, int topk,
                   void* workspace, float* tbox_px, float* tscores, unsigned char* fg, void* stream) {
    return launch_tal_assign(probs, pboxes, anchors, stride, gt_cls, gt_box, gt_valid, img_w, img_h, B, A, M, nc, topk, workspace, tbox_px,
                             tscores, fg, nullptr, nullptr, ST);
}
int snn_detect_loss_bwd_rows(const float* distri, const float* scores, int nl, const int* a_off, const float* anchors,
                             const float* stride, const float* tbox_px, const float* tscores, const unsigned char* fg, int B, int A,
                             int nc, int reg_max, const float* coef3, const float* gout3, void* g_distri, void* g_scores,
                             int out_is_bf16, void* stream) {
    return launch_detect_loss_bwd(distri, scores, anchors, stride, tbox_px, tscores, fg, B, A, nc, reg_max, coef3, gout3, g_distri,
                                  g_scores, out_is_bf16, nl, a_off, ST);
}

}  // extern "C"

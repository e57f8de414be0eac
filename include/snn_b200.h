/* libsnnb200 -- C ABI of the B200-native spiking-detector hot path.
 *
 * The reference (Anannayjain/SNN_Object_DetectionDDP) is pure Python/PyTorch and has NO FFI; this
 * header is the boundary a maintainer binds with ctypes from the reference's model.py/train.py
 * (see INTEGRATION.md).  Each entry point names the reference code it replaces.
 *
 * Conventions
 *  - every function returns 0 on success, non-zero on error; snn_last_error() returns a
 *    thread-local message.  Nothing throws across the ABI.
 *  - all pointers are DEVICE pointers owned by the caller (PyTorch allocates everything,
 *    including workspaces); `stream` is a cudaStream_t passed as void*.
 *  - activations are NHWC with the T*B batch folded into N ("NB"); element (n,h,w,c) of a view
 *    lives at ptr[((n*H+h)*W+w)*ld + c]  (ld >= C lets a view be a channel slice).
 *  - bf16 = raw uint16 storage; weights for the tensor-core convs are bf16 [Cout][taps][Cin] (taps = kh*kw in
 *    (kh,kw) order; transposed conv: [Cout][4][Cin]) for fprop AND dgrad -- dgrad reads the same buffer as an
 *    MN-major operand, no transposed copy exists.
 *  - compute dtype: bf16 operands, fp32 accumulate (tcgen05), fp32 everywhere else.
 */
#ifndef SNN_B200_H
#define SNN_B200_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

const char* snn_last_error(void);
int snn_version(void);
/* test / A-B timing knobs, all default 0 (never needed in production):
 *   0: 1 = per-thread row-store epilogue instead of swizzled staging + TMA tensor stores (conv fprop/dgrad)
 *   1: cap on the number of shared-memory pipeline stages        2: K chunks per pipeline stage (1, 2, 4)
 *   3: 1 = a single epilogue warp group also for small-K convs (default: two groups, 320 threads)
 *   4: force the wgrad K-split                                   5: cap on persistent CTAs (pairs)
 *   6: 1 = single-CTA kernels only, 2 = CTA pairs also for small-K convs
 *   7: (only in -DSNN_TIMING_KNOBS builds) bit 0 = producer skips the TMA loads, bit 1 = MMA issuer skips the MMAs
 *   8: 1 = T == 1 SiLU layers use the generic two-pass BN backward kernel
 *   9: 1 = T == 16 uses the one-chunk two-pass BN backward kernel instead of the two-chunk one
 *  12: row-strip mode of the 3x3 stride-1 convs (one [bh+2] x bw activation box feeds the three taps of a stencil column):
 *      0 = wherever >= 2 pipeline stages fit (maps >= 8x8), 1 = off, 2 = only where >= 3 stages fit (tiles of <= 144 columns),
 *      3 = only pixel boxes inside one image (maps >= 16x8)
 *  13: 1 = wgrad of the 3x3 stride-1 convs tap by tap (default: one stencil column = three taps per work item, row-strip X box),
 *      2 = row-strip wgrad only for pixel boxes inside one image
 *  14: 1 = row-strip wgrad keeps the two-round K split of the tap-by-tap kernel */
void snn_debug_set(int key, int value);
/* Tile scheduling of the persistent tensor-core kernels (process-wide, read at launch): 0 (default) = static walk
 * (tile = worker, worker + nworkers, ...), 1 = dynamic (first tile static, the rest from an atomic counter).  Dynamic is for
 * data-parallel training: gradient all-reduces run beside backward, the SMs that also host NCCL CTAs are slower, and with a
 * static walk every launch waits for them.  Dynamic mode uses a library-owned 32 KB counter pool per device (allocated at
 * the first launch in that mode; launch once eagerly before capturing a CUDA graph). */
void snn_set_tile_scheduling(int dynamic);
/* Launch plan of a conv call WITHOUT launching it: the host-side planning (pixel box, N tile, CTA pairs, row-strip mode,
 * pipeline stages, K split, work items) runs exactly as for a launch, no CUDA call is made -- usable without a GPU (the SM
 * count then defaults to 148).  kind: 0 = fprop, 1 = dgrad, 2 = wgrad; frames_per_step > 0 = fprop with fused statistics.
 * out20 = {bn, bh, bw, N tile, CTA pair, row-strip, (h,n,w) row order, stages, stage bytes, K chunks per stage, K split,
 * work items, N blocks (wgrad: cin tiles), CTAs or CTA pairs launched, epilogue warp groups, small-K, TMA-store epilogue,
 * dynamic shared memory bytes, activation bytes per stage (wgrad: X box bytes), weight-slice bytes per tap (wgrad: dY bytes)}. */
int snn_conv_plan(int kind, int geom, int NB, int H, int W, int Cin, int Cout, int out_f32, int frames_per_step, int accumulate,
                  int* out20);
/* Deterministic mode (process-wide, read at launch; default 0).  1 = every sum whose order is otherwise decided by atomics or
 * by the arrival order of TMA reduce-adds is taken in a fixed order: wgrad and the small-M dgrad run without split-K;
 * BatchNorm-backward sums, bias column sums, depthwise wgrad, the gradient norm and the loss sums go through per-block
 * partials in a library-owned scratch buffer (>= 64 MB per device, allocated at the first such launch -- run one step
 * eagerly before capturing a CUDA graph) and are added in block order.  Two runs from the same state then produce
 * bit-identical gradients on one GPU.  Slower: a reproducibility / debugging mode. */
void snn_set_deterministic(int on);
int snn_get_deterministic(void);
/* Programmatic dependent launch (process-wide, read at launch; default 0): 1 = every kernel of the library is launched with
 * cudaLaunchAttributeProgrammaticStreamSerialization, so it may become resident -- and run its barrier / TMEM / table
 * set-up -- while its predecessor on the stream drains; each kernel executes griddepcontrol.wait before its first global
 * memory access, so results are identical to serialized launches.  Also honoured under CUDA-graph stream capture
 * (programmatic edges between consecutive kernel nodes). */
void snn_set_dependent_launch(int on);
int snn_get_dependent_launch(void);
/* The library keeps a process-wide, mutex-guarded cache of encoded TMA tensor maps keyed by (device, pointer, shape,
 * strides, box): hit / miss counters since load (a steady eager training loop re-uses every map of the previous step). */
void snn_tensor_map_cache_stats(unsigned long long* hits, unsigned long long* misses);

/* conv geometries on the path (reference model.py:13 k3 s1/s2 p1; model.py:119 k1; model.py:36 convT k2 s2) */
enum { SNN_GEOM_3x3_S1 = 0, SNN_GEOM_3x3_S2 = 1, SNN_GEOM_1x1 = 2, SNN_GEOM_T2x2_S2 = 3 };
enum { SNN_ACT_LIF = 0, SNN_ACT_SILU = 1 };

/* ---- spike convolutions: replaces nn.Conv2d / nn.ConvTranspose2d forward+backward in
 *      ConvBlock (model.py:13,18), UpBlock.up (model.py:36,42), ConvLSTM2d.conv (model.py:55,66),
 *      out_p3/4/5 (model.py:119,146).  (H, W) are always the conv INPUT's spatial dims.
 *      x1 != NULL convolves the channel concatenation cat([x0, x1]) (model.py:45,66,126,127)
 *      without materialising it. ---- */
int snn_conv_fprop(int geom, int NB, int H, int W,
                   const void* x0, int C0, long long ld0, const void* x1, int C1, long long ld1,
                   const void* w_bf16, int w_rows, int w_K, int w_coff, int Cout, int w_row_off,
                   const float* bias, void* out, int out_is_f32, long long out_ld, int out_coff,
                   int accumulate, void* stream);
/* ConvBlock forward with the train-mode BatchNorm statistics fused into the conv epilogue (replaces the separate pass of
 * F.batch_norm over the conv output, model.py:14): out is dense fp32 [NB,Ho,Wo,Cout]; `partials` receives one
 * (sum, sum of squares) pair per 32-pixel group and channel, fp32 [groups][2][Cout], written without atomics.
 * snn_conv_stats_groups() returns `groups` for the geometry (0: not available -> snn_conv_fprop + snn_bn_stats) and the
 * number of groups per timestep; snn_bn_stats_from_partials() reduces them in a fixed order to the [T][2][C] fp64 sums
 * snn_bn_finalize() consumes.  frames_per_step = B (the folded batch holds T*B frames, timestep-major). */
long long snn_conv_stats_groups(int geom, int NB, int H, int W, int frames_per_step, int* groups_per_step);
int snn_conv_fprop_stats(int geom, int NB, int H, int W,
                         const void* x0, int C0, long long ld0, const void* x1, int C1, long long ld1,
                         const void* w_bf16, int w_rows, int w_K, int w_coff, int Cout, int w_row_off,
                         float* out, int frames_per_step, float* partials, void* stream);
int snn_bn_stats_from_partials(const float* partials, double* sums /*[T][2][C]*/, int T, int C, int groups_per_step,
                               void* stream);
/* snn_bn_stats_from_partials + snn_bn_finalize(training) + `num_batches_tracked += T` in ONE launch (same arithmetic, same
 * order of the T running-statistics updates).  `counters`: caller-owned, zero-initialised ceil(C/32) unsigned ints, left
 * zeroed; `sums` [T][2][C] fp64 receives the reduced statistics; `workspace`: snn_bn_finalize_workspace_doubles(T, C,
 * groups_per_step) doubles of scratch (per-block partials, combined in a fixed order by the last block of a channel group). */
long long snn_bn_finalize_workspace_doubles(int T, int C, int groups_per_step);
int snn_bn_finalize_partials(const float* partials, double* sums, double* workspace, const float* gamma, const float* beta,
                             float* running_mean, float* running_var, long long* num_batches_tracked,
                             float* scale, float* shift, float* mean, float* invstd /*[T][C] each*/,
                             unsigned int* counters, int T, int C, int P, int groups_per_step, float eps, float momentum,
                             void* stream);
int snn_conv_dgrad(int geom, int NB, int H, int W,
                   const void* dy, int Cout, long long ld_dy,
                   const void* w_bf16 /*[Cout][taps][w_K]*/, int w_K, int ci_off, int Ci,
                   void* dx, int dx_is_f32, long long dx_ld, int dx_coff, int accumulate, void* stream);
/* dw (fp32 [Cout][taps][w_K]) += ... ; caller zeroes it once per step */
int snn_conv_wgrad(int geom, int NB, int H, int W,
                   const void* x, int Ci, long long ld_x, const void* dy, int Cout, long long ld_dy,
                   float* dw, int w_K, int w_coff, void* stream);
/* fp32 master [N][T][K] -> bf16 same layout (w_bf16, may be NULL) and bf16 [K][T][N] (wt_bf16, may be NULL; utility,
 * the convs no longer need the transposed copy) */
int snn_weight_prep(const float* w, void* w_bf16, void* wt_bf16, int N, int T, int K, void* stream);

/* ---- neuron layer: replaces `self.silu(self.bn(.))` of ConvBlock.forward (model.py:14-18)
 *      y is the conv output, fp32 [T][P][C].  Train-mode BN statistics are per timestep
 *      (the reference calls the module once per frame, train.py:64-66). ---- */
/* deterministic (no atomics): per-block partial sums go to `workspace` (snn_bn_stats_workspace_floats() floats, caller
 * owned), then a fixed-order fp64 combine */
long long snn_bn_stats_workspace_floats(int T, int P, int C);
int snn_bn_stats(const float* y, double* sums /*[T][2][C]*/, float* workspace, int T, int P, int C, void* stream);
int snn_bn_finalize(const double* sums, const float* gamma, const float* beta,
                    float* running_mean, float* running_var,
                    float* scale, float* shift, float* mean, float* invstd /* each [T][C] (train) or [C] (eval) */,
                    int T, int C, int P, float eps, float momentum, int training, void* stream);
/* fused BN affine + multi-step LIF (or SiLU): out bf16 [T][P][C]; mask = 1 bit/neuron [T][P*C/8] (LIF, may be NULL);
 * v_init / v_final fp32 [P][C] may be NULL (zero initial membrane / state not needed). ss_stride_t = C (train) or 0 (eval). */
int snn_bn_act_fwd(int act, const float* y, const float* scale, const float* shift, const float* v_init,
                   void* out_bf16, uint8_t* mask, float* v_final, int T, long long n_per_t, int C,
                   int ss_stride_t, float beta, float theta, void* stream);
/* snn_bn_act_fwd (LIF only) that also ADDS per-timestep totals: spikes[t] += #{s=1}, steps[t] += n_per_t (uint64, exact).
 * Outputs are bit-identical to snn_bn_act_fwd(ACT_LIF, ...); T <= 64. */
int snn_bn_act_fwd_count(const float* y, const float* scale, const float* shift, const float* v_init, void* out_bf16,
                         uint8_t* mask, float* v_final, unsigned long long* spikes, unsigned long long* steps,
                         int T, long long n_per_t, int C, int ss_stride_t, float beta, float theta, void* stream);
/* reverse-time surrogate-gradient scan. training!=0: writes gx fp32 [T][P][C] and red [T][2][C]
 * (sum gx, sum gx*xhat); training==0: writes dy bf16 = gx*scale directly. */
int snn_bn_act_bwd(int act, int training, const float* y, const float* scale, const float* shift,
                   const float* mean, const float* invstd, const float* v_init,
                   const void* gs_bf16, const float* gv_final,
                   float* gx, void* dy_bf16, float* gv_init, float* red,
                   int T, int P, int C, int ss_stride_t, float beta, float theta, float alpha, void* stream);
/* train-mode backward WITHOUT the fp32 gx round trip: gx is recomputed in registers in both passes.
 *   pass 0: red [T][2][C] = per-(t,c) sum gx, sum gx*xhat (zeroed here)
 *   pass 1: dy bf16 = scale*(gx - mean gx - xhat*mean(gx*xhat)); gv_init (may be NULL); dgamma/dbeta += (may be NULL)
 * beta_bn = the BatchNorm bias [C] (x - beta_bn = gamma*xhat).  scale/shift/mean/invstd are [T][C]. */
int snn_bn_act_bwd2(int pass, int act, const float* y, const float* scale, const float* shift, const float* mean,
                    const float* invstd, const float* beta_bn, const float* v_init, const void* gs_bf16,
                    const float* gv_final, float* red, void* dy_bf16, float* gv_init, float* dgamma, float* dbeta,
                    int T, int P, int C, float beta, float theta, float alpha, void* stream);
/* BN input gradient from gx and the reductions; dgamma/dbeta (+=) */
int snn_bn_bwd_dx(const float* red, const float* gamma, const float* gx, const float* y,
                  const float* scale, const float* mean, const float* invstd, float* coef /*[T][2][C]*/,
                  float* dgamma, float* dbeta, void* dy_bf16, int T, int P, int C, void* stream);

/* ---- ConvLSTM gate math (model.py:67-69): gates fp32 [P][4*Ch] in i|f|g|o order ---- */
int snn_lstm_gates_fwd(const float* gates, const float* c_prev, float* c_next, float* h_next,
                       void* h_bf16, long long P, int Ch, void* stream);
/* backward of one step: total dL/dh_t = dh (fp32, recurrent part from step t+1's W_h dgrad; may be NULL) + dh_bf16 (bf16, the
 * consumer's part from bottleneck_conv's dgrad; may be NULL), summed inside the kernel */
int snn_lstm_gates_bwd(const float* gates, const float* c_prev, const float* c_next,
                       const float* dh, const void* dh_bf16, const float* dc_in, void* dgates_bf16, float* dc_prev,
                       long long P, int Ch, void* stream);

/* ---- layout conversion at the nn.Module boundary (reference tensors are NCHW fp32) ---- */
int snn_nchw_to_nhwc(const float* in, void* out, int out_is_bf16, int NB, int C, int HW,
                     long long out_ld, int out_coff, void* stream);
int snn_nhwc_to_nchw(const void* in, int in_is_bf16, float* out, int NB, int C, int HW,
                     long long in_ld, int in_coff, void* stream);

/* ---- Detect-head depthwise 3x3 (ultralytics DWConv inside `Detect.cv3`, built at model.py:186):
 *      x/dy bf16 NHWC, weights fp32 [9][C], y fp32 NHWC (feeds the BN+SiLU kernel), dw += ---- */
int snn_dw3x3_fprop(const void* x_bf16, const float* w, float* y, int NB, int H, int W, int C, void* stream);
int snn_dw3x3_dgrad(const void* dy_bf16, const float* w, void* dx_bf16, int NB, int H, int W, int C, void* stream);
int snn_dw3x3_wgrad(const void* x_bf16, const void* dy_bf16, float* dw, int NB, int H, int W, int C, void* stream);
/* depthwise forward with the train-mode BatchNorm statistics fused (as snn_conv_fprop_stats): partials fp32
 * [T][blocks][2][C], blocks = snn_dw3x3_stats_blocks(B, W, C) per timestep, one row per thread block, written without
 * atomics and reduced in a fixed order by snn_bn_finalize_partials(groups_per_step = blocks). */
long long snn_dw3x3_stats_blocks(int frames_per_step, int W, int C);
int snn_dw3x3_fprop_stats(const void* x_bf16, const float* w9c, float* y, int NB, int H, int W, int C, int T, float* partials,
                          void* stream);

/* ---- frame packer of the stand-in feature pyramid (the frozen YOLO11m of model.py:74-98 cannot exist
 *      offline): fp32 frames [B][T][3][H][W] -> bf16 NHWC [T*B][H/8][W/8][192] ---- */
int snn_space_to_depth8(const float* frames, void* out_bf16, int B, int T, int H, int W, void* stream);
/* same packer for uint8 frames [B][T][3][H][W] (what dataset.py:139-152 decodes before its host-side `/ 255.0`): the division
 * runs on the device, bit-identical to the host's, and the host->device copy shrinks 4x */
int snn_space_to_depth8_u8(const unsigned char* frames, void* out_bf16, int B, int T, int H, int W, void* stream);

/* ---- UpBlock skip resize (model.py:43-44: F.interpolate(skip_x, size=x.shape[2:], mode='bilinear', align_corners=False)),
 *      NHWC bf16 [NB,Hi,Wi,C] -> [NB,Ho,Wo,C], ATen's source-index / weight formula in fp32, one rounding to bf16.
 *      backward = 1: src is the gradient w.r.t. the RESIZED tensor [NB,Ho,Wo,C], dst the gradient w.r.t. the input
 *      [NB,Hi,Wi,C] (deterministic gather, no atomics).  (Hi, Wi) / (Ho, Wo) always name the forward's input / output. ---- */
int snn_bilinear_resize(int backward, const void* src_bf16, void* dst_bf16, int NB, int Hi, int Wi, int Ho, int Wo, int C,
                        void* stream);
/* ---- bottom/right zero-pad (Hd >= Hs) or crop (Hd <= Hs) of an NHWC bf16 tensor: dst[n,h,w,:] = src[n,h,w,:] inside the
 *      source extent, 0 outside.  In front of a stride-2 3x3 pad-1 conv (DownBlock.conv1, model.py:24) whose input has an
 *      odd H or W (the 15x20 level of a 480x640 frame) the zero row/column IS the conv's padding; the crop is its backward. ---- */
int snn_nhwc_pad_crop(const void* src_bf16, void* dst_bf16, int NB, int Hs, int Ws, int Hd, int Wd, int C, void* stream);

/* ---- bias gradient of the biased convs (ConvLSTM2d.conv, UpBlock.up, out_p*): acc[c] += sum_p dy[p][c] ---- */
int snn_colsum_bf16(const void* dy_bf16, float* acc, long long P, int C, void* stream);

/* ---- optimizer: replaces clip_grad_norm_(10) + AdamW.step + OneCycleLR.step (train.py:77-80) over one flat buffer.
 *      hp (device) = rows of 8 floats {lr, beta1, beta2, eps, weight_decay, 1-beta1^t, 1-beta2^t, max_norm};
 *      step_ptr == NULL: row 0 is used; else row min(*step_ptr, n_rows-1) is used and *step_ptr is incremented
 *      afterwards (device-side schedule: no host sync, CUDA-graph replayable).
 *      zero_grad != 0: g is left zeroed (optimizer.zero_grad() of train.py:61 folded into the pass that consumes g). ---- */
int snn_grad_sumsq(const float* g, long long n, double* acc, int zero_first, void* stream);
int snn_adamw_step(float* p, float* g, float* m, float* v, void* shadow_bf16, long long n,
                   const float* hp, const double* sumsq, float* gnorm_out, int* step_ptr, int n_rows, int zero_grad,
                   void* stream);

/* ---- Detect decode (ultralytics Detect._inference, reached through model.py:209 in eval mode, and
 *      v8DetectionLoss.bbox_decode): boxes fp32 [N][4] in pixels (xywh != 0: cx,cy,w,h; else x1,y1,x2,y2) and
 *      sigmoid class probabilities fp32 [N][nc] (probs may be NULL). ---- */
int snn_detect_decode(const float* distri, const float* scores, const float* anchors, const float* stride,
                      int B, int A, int nc, int reg_max, int xywh, float* boxes, float* probs, void* stream);

/* ---- non-maximum suppression: replaces ultralytics.utils.nms.non_max_suppression (+ torchvision.ops.nms) as called at
 *      visualize.py:73-78 (conf 0.3, iou 0.45, multi_label=True) and eval_2.py:108 (conf 0.001, iou 0.6).
 *      pred fp32 [B][4+nc][A] = what Detect returns in eval mode (xywh pixels + class scores).  Per image: candidates with
 *      score > conf_thres (multi_label: every (anchor, class) pair; else the best class), sorted by score descending with
 *      ties in enumeration order, greedy IoU suppression with the per-class box offset cls*max_wh (unless agnostic), at most
 *      max_det (<= 512) rows.  out fp32 [B][max_det][6] = x1 y1 x2 y2 conf cls, out_idx int32 [B][max_det] = enumeration
 *      index (anchor*nc + cls | anchor) of each kept row, counts int32 [B].  `keys` is a caller-owned workspace of
 *      B * snn_nms_workspace_keys() 64-bit words.  No host synchronisation. ---- */
long long snn_nms_workspace_keys(int nc, int A, int multi_label);
int snn_nms(const float* pred, int B, int nc, int A, float conf_thres, float iou_thres, int multi_label, int agnostic,
            int max_det, int max_nms, float max_wh, unsigned long long* keys, long long keys_per_image,
            float* out, int* out_idx, int* counts, void* stream);

/* ---- detection metrics: replaces ultralytics DetectionValidator / DetMetrics as called at eval_2.py:82-88 (mAP50,
 *      mAP50-95, precision, recall).
 *      snn_det_match, once per batch: rows fp32 [B][max_det][6] and counts int32 [B] = snn_nms output; gt_cls int64 [B][M],
 *      gt_box fp32 [B][M][4] normalised (cx,cy,w,h), gt_valid uint8 [B][M] = the padded labels (M <= 2048); iou_thres
 *      device fp32 [10].  Each kept row takes its same-class gt of highest IoU (box_iou, fp32; exact ties: the higher gt
 *      index) and is a TP at threshold t when that IoU >= t and it is the lowest row claiming that gt.  Writes one record
 *      per kept row at *cursor + sum(counts[<b]) -- rec_conf fp32, rec_cls int32, rec_tp uint16 (bit t = TP at
 *      iou_thres[t]), rec_key int64 = (cls << 32) | (0x7FFFFFFF - float_bits(conf)) -- and advances *cursor (int64) by
 *      sum(counts); ticket uint32[1] (zero-initialised once; left zeroed).  n_gt int64 [nc] += the gt class histogram;
 *      err int32[1] += out-of-range gt / row classes and records past `capacity`.  No host synchronisation.
 *      snn_det_metrics_finalize, once per evaluation: keys = rec_key[0..n) sorted ascending (stable), order = the record
 *      index of each sorted key, rec_tp by record index.  out fp64 [8 + 11*nc] = {mp, mr, mAP50, mAP50-95, fitness,
 *      number of target classes, F1 argmax, *err}, then ap [nc][10], then present [nc] (1 = class has gts); curves fp64
 *      [2][nc][1000] = precision and recall curves at IoU 0.5 (scratch).  Keys >= (nc << 32) are ignored. ---- */
int snn_det_match(const float* rows, const int* counts, int B, int max_det, const long long* gt_cls, const float* gt_box,
                  const unsigned char* gt_valid, int M, float img_w, float img_h, const float* iou_thres, int nc,
                  float* rec_conf, int* rec_cls, unsigned short* rec_tp, long long* rec_key, long long capacity,
                  long long* cursor, unsigned int* ticket, long long* n_gt, int* err, void* stream);
int snn_det_metrics_finalize(const long long* keys, const long long* order, const unsigned short* rec_tp, long long n,
                             const long long* n_gt, int nc, const int* err, double* curves, double* out, void* stream);

/* ---- detection-loss tail: replaces the per-anchor part of ultralytics v8DetectionLoss called at train.py:74
 *      (BCE class loss, CIoU box loss, DFL) given the assigner's targets.  N = B*A anchors (A = anchors per image,
 *      scale-major), distri fp32 [N][4*reg_max], scores / tscores fp32 [N][nc], anchors fp32 [A][2] (grid units),
 *      stride fp32 [A], tbox_px fp32 [N][4] (xyxy pixels), fg uint8 [N].
 *      fwd: sums (double[3], zeroed here) = {sum (1-CIoU)*w, sum BCE, sum DFL*w}.
 *      bwd: coef (device float[3]) = dL/d sums -> g_distri [N][4*reg_max], g_scores [N][nc] (overwritten). ---- */
int snn_detect_loss_fwd(const float* distri, const float* scores, const float* anchors, const float* stride,
                        const float* tbox_px, const float* tscores, const uint8_t* fg, int B, int A, int nc, int reg_max,
                        double* sums, void* stream);
int snn_detect_loss_bwd(const float* distri, const float* scores, const float* anchors, const float* stride,
                        const float* tbox_px, const float* tscores, const uint8_t* fg, int B, int A, int nc, int reg_max,
                        const float* coef, float* g_distri, float* g_scores, void* stream);

/* ---- whole v8DetectionLoss forward (train.py:74) in 5 launches, no host synchronisation, no ATen:
 *      decode (DFL expectation -> xyxy pixels, sigmoid scores) -> TaskAlignedAssigner (top-k 10, alpha 0.5, beta 6:
 *      per-(gt, anchor) CIoU / alignment metric, top-k candidates per gt with ties to the lower anchor index, anchors claimed
 *      by several gts keep the largest overlap, normalised target scores) -> fused BCE + CIoU + DFL sums -> finalisation by
 *      the last block: out6 = {loss*B [3], loss [3]} (what `loss_fn(preds, batch)` returns at train.py:74, hyp gains of
 *      config.yaml:33-37 applied, normalised by max(sum target scores, 1)), coef3 = d(sum(loss*B))/d sums.
 *      Predictions are read through a ROW MAP: nl > 0 = the Detect head's SCALE-MAJOR buffers (scale i = rows
 *      [B*a_off[i], B*a_off[i+1]), image-major inside; a_off = nl+1 host ints, a_off[nl] = A) so that no torch.cat is needed;
 *      nl = 0 = natural [B][A] rows.  Labels are the dense padding of the collate layout (train.py:27-37):
 *      gt_cls int64 [B][M], gt_box fp32 [B][M][4] normalised (cx,cy,w,h), gt_valid uint8 [B][M]; (img_w, img_h) = stride-8 map
 *      size * 8.  Caller-owned scratch: workspace of snn_tal_workspace_bytes(B,A,M) bytes, pboxes [B][A][4], probs [B][A][nc],
 *      tbox_px [B][A][4], tscores [B][A][nc], fg [B][A] (targets, natural layout, kept for the backward), sums double[3],
 *      counter uint32[1] (zero-initialised once; left zeroed), gains device float[3] = {box, cls, dfl}. ---- */
long long snn_tal_workspace_bytes(int B, int A, int M);
int snn_detect_assign_loss_fwd(const float* distri, const float* scores, int nl, const int* a_off, const float* anchors,
                               const float* stride, const long long* gt_cls, const float* gt_box, const unsigned char* gt_valid,
                               float img_w, float img_h, int B, int A, int M, int nc, int reg_max, int topk, const float* gains,
                               void* workspace, float* pboxes, float* probs, float* tbox_px, float* tscores, unsigned char* fg,
                               double* sums, unsigned int* counter, float* out6, float* coef3, void* stream);
/* the assigner alone (inputs: sigmoid scores and xyxy-pixel boxes in natural [B][A] layout) */
int snn_tal_assign(const float* probs, const float* pboxes, const float* anchors, const float* stride, const long long* gt_cls,
                   const float* gt_box, const unsigned char* gt_valid, float img_w, float img_h, int B, int A, int M, int nc, int topk,
                   void* workspace, float* tbox_px, float* tscores, unsigned char* fg, void* stream);
/* backward of the fused loss: gradients at the prediction rows (row map as above), fp32 or bf16 (out_is_bf16: they are the
 * `dy` operands of the head's closing 1x1 convs); gout3 (device float[3], may be NULL = ones) = upstream gradient of loss*B. */
int snn_detect_loss_bwd_rows(const float* distri, const float* scores, int nl, const int* a_off, const float* anchors,
                             const float* stride, const float* tbox_px, const float* tscores, const unsigned char* fg, int B, int A,
                             int nc, int reg_max, const float* coef3, const float* gout3, void* g_distri, void* g_scores,
                             int out_is_bf16, void* stream);

#ifdef __cplusplus
}
#endif
#endif

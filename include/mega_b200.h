/* mega_b200.h -- C ABI of libmega_b200.so: hand-written sm_100a kernels for the MEGA
 * (Scalsol/mega.pytorch) per-frame inference hot path.
 *
 * Conventions
 *   - every entry point returns 0 (MEGA_OK) or a non-zero status; mega_last_error() returns a
 *     human-readable description of the last failure on the calling thread's process;
 *   - all pointers are DEVICE pointers unless the name ends in _host;
 *   - `stream` is a cudaStream_t passed as void*; kernels are enqueued on it and never
 *     synchronise (the reference launches NMS/DCN on the legacy default stream,
 *     csrc/cuda/nms.cu:94 -- here everything honours the caller's stream);
 *   - no state is kept across calls; nothing allocates device memory (workspaces are
 *     caller-provided), so every call is CUDA-graph capturable.
 *
 * Each declaration cites the reference interface it replaces (paths relative to the
 * reference checkout, mega_core/...).
 */
#ifndef MEGA_B200_H_
#define MEGA_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ------------------------------------------------------------------ library */
const char* mega_last_error(void);
int mega_abi_version(void);
/* 1 if the current CUDA device is sm_100 (B200), 0 otherwise, <0 on CUDA error. */
int mega_device_ok(void);

/* ------------------------------------------------- dense contractions (tcgen05)
 * Implicit-GEMM convolution / GEMM on the tensor cores, FP32 accumulation in TMEM. Operand arithmetic is selected
 * by `precision`: 0 = fp32 tensors rounded to TF32 on load, 1 = fp32 tensors, 3xTF32 split (near-fp32), 2 = fp16
 * tensors (same 10-bit mantissa as TF32, half the bytes, twice the tensor-pipe rate), 3 = "3xFP16": operands in the
 * SPLIT-FP16 format (below; near-fp32 like 1, kind::f16 MMAs, no split work in the kernel); the output / residual are
 * fp32, or fp16 when out_f16 != 0 (precision 2), or split-fp16 (precision 3: out_f16 != 0 for the output, res_split != 0
 * for the residual).
 * SPLIT-FP16 format: a tensor with the shape, strides and byte size of an fp32 tensor whose innermost dimension is a
 * multiple of 32; every aligned group of 32 consecutive values x[0..32) occupies its 128 bytes as 32 halves
 * hi[i] = fp16_rn(x[i]) (saturating) followed by 32 halves lo[i] = fp16_rn(x[i] - hi[i]): |x - (hi + lo)| <= 2^-23 |x| for
 * |x| >= 2^-3, <= 2^-25 below. mega_split16_pack / mega_split16_unpack convert from / to fp32.
 *   out[n,h,w,co] = act( scale[co] * sum_{r,s,ci} a[n, h + r*dil - pad, w + s*dil - pad, ci]
 *                                          * b[r*S+s, co, ci]  + bias[co] + residual[n,h,w,co] )
 * Replaces: ATen/cuDNN conv2d + FrozenBatchNorm2d + add + relu_ of
 * modeling/backbone/resnet.py:324-344, the RPN head convs rpn/rpn.py:99-106, nn.Linear of
 * make_layers.py:80-92 (as an H=1 image, taps 1x1), torch.bmm / torch.matmul of
 * roi_heads/box_head/roi_box_feature_extractors.py:616-638 (batch>1 with the *_off fields). */
typedef struct mega_conv_gemm_desc {
  /* A: activations, NHWC, fp32 or fp16 by `precision` (strides in ELEMENTS, innermost stride 1) */
  const void* a;
  int a_n, a_h, a_w, a_c;
  long long a_stride_w, a_stride_h, a_stride_n;
  /* B: weights [taps][cout rows][k], same element type as A, k contiguous */
  const void* b;
  int b_n, b_k;
  long long b_stride_n, b_stride_tap;
  int taps_r, taps_s, dil, pad;
  int k_per_tap; /* reduction length per tap (Cin) */
  /* output NHWC, dense in (w, h, n) with out_ld elements between pixels (written by TMA: 16-byte aligned
   * base and pitch; the residual likewise, same element type as the output); out_h/out_w = output spatial size */
  void* out;
  long long out_ld;
  int n_img, out_h, out_w, cout;
  const float* scale;    /* [cout] or NULL */
  const float* bias;     /* [cout] or NULL */
  const void* residual;  /* same indexing and element type as out, with res_ld, or NULL */
  long long res_ld;
  int relu; /* 0: none, 1: ReLU, 2: LeakyReLU(0.1) (backbone/flownet.py:47) */
  /* tiling: tile_h*tile_w == 128 output pixels per CTA, block_n in {32,64,96,128,160,192,256} */
  int tile_h, tile_w, block_n;
  /* batched mode (grid.z = batch): per-batch coordinate offsets */
  int batch;
  int a_c_off, a_n_off; /* added to A's channel / image coordinate, times batch index */
  int b_k_off, b_n_off; /* added to B's k / row coordinate, times batch index */
  int out_c_off, out_n_off; /* added to the output's channel / image coordinate, times batch index */
  int res_c_off, res_n_off; /* same for the residual */
  int bias_z_off; /* added to the scale/bias index, times batch index */
  /* persistent stream-K scheduling: at most max_ctas CTAs (0 = one per SM). `workspace` (device,
   * >= mega_conv_gemm_workspace_bytes(), 256-byte aligned, ZERO-INITIALISED once; the kernel leaves
   * its counter region zero) holds the tile counters and the partial accumulators of tiles whose
   * K range is shared by several CTAs. Launches that may run concurrently need distinct workspaces. */
  int precision; /* 0: TF32 operands (round-to-nearest on load); 1: "3xTF32" split (hi*hi + hi*lo + lo*hi),
                    ~2^-19 relative error, block_n 64 or 128; 2: fp16 operands (A and B are __half arrays);
                    3: "3xFP16": A and B in the split-fp16 format, hi*hi + hi*lo + lo*hi with kind::f16 MMAs */
  int max_ctas;
  int stream_k; /* 1: split tiles across CTAs at k-block granularity (balances any tile count over the
                   SMs; partial tiles are reduced by the last CTA to arrive, in CTA order); 0: whole tiles */
  void* workspace;
  long long workspace_bytes;
  int out_f16; /* 1: out / residual are __half (precision 2, block_n % 64 == 0); 0: fp32 */
  int pdl;     /* 1: programmatic dependent launch -- the kernel's prologue overlaps the tail of the previous kernel
                  on the stream (it orders its own memory accesses behind that kernel with griddepcontrol.wait) */
  /* ABI v3 (zero = previous behaviour): */
  int stride_h, stride_w; /* convolution stride (0 -> 1): output pixel (h, w) reads a[h*stride_h + r*dil - pad, ...]; the
                             strided rectangle is fetched with TMA element strides (tile_w, tile_h <= 128) */
  int pad_w_set, pad_w;   /* pad_w_set != 0: left padding pad_w differs from `pad` (which then applies to h only) */
  long long out_stride_h, out_stride_n; /* element strides of the output rows / images (0: dense, out_ld * out_w and
                                           out_ld * out_w * out_h) -- lets a conv write every other pixel of a larger
                                           map (the four parity classes of a stride-2 transposed convolution) */
  long long res_stride_h, res_stride_n; /* same for the residual */
  /* ABI v5 (zero = previous behaviour): precision 1 only. b_lo_tap_off = taps_r * taps_s says that the low parts of the
   * 3xTF32 split of B, lo = b - trunc_tf32(b), are stored BEHIND b as taps more [rows][k] slices (b then holds 2 * taps
   * slices): the kernel fetches them by TMA instead of splitting the staged B tile on every k-block -- for weights, which
   * never change (mega_core.b200.ops.presplit builds the pair once). */
  int b_lo_tap_off;
  /* ABI v6 (zero = previous behaviour): precision 3 only. a, b: split-fp16 tensors (a_c, b_k, k_per_tap, a_c_off, b_k_off
   * multiples of 32; block_n 64 or 128). out_f16 != 0: split-fp16 output (cout, out_c_off multiples of 32), else fp32.
   * `scale` must be NULL (fold per-channel factors into the weights before packing them). res_split != 0: the residual is
   * split-fp16, else fp32. acc_scale: 0 = 1; otherwise the accumulator is multiplied by it
   * before scale / bias -- weights are stored multiplied by a power of two 1 / acc_scale so that their low halves stay
   * normal fp16 numbers (mega_core.b200.ops.pack_weights_split16). */
  int res_split;
  float acc_scale;
  int reserved_v6;
} mega_conv_gemm_desc;

/* fp32 <-> split-fp16 (format above) over n_values contiguous values (multiple of 32, 128-byte aligned); pack may run in
 * place (dst == src). New in this build (no reference counterpart: the reference computes in fp32 throughout). */
int mega_split16_pack(const float* src, void* dst, long long n_values, void* stream);
int mega_split16_unpack(const void* src, float* dst, long long n_values, void* stream);
int mega_conv_gemm(const mega_conv_gemm_desc* desc, void* stream);
/* ABI v1 name of mega_conv_gemm (kept for existing callers) */
int mega_conv_gemm_tf32(const mega_conv_gemm_desc* desc, void* stream);
long long mega_conv_gemm_workspace_bytes(void);

/* A chain of dependent contractions in ONE persistent kernel (conv_chain.cu): `descs[0..n)` are executed in order,
 * layer l+1 may read anything layers <= l wrote (grid-wide barrier between layers, no kernel boundary). All layers:
 * precision 2 (fp16 operands), block_n <= 128, the same workspace. mega_conv_chain_encode() validates the
 * descriptors and writes the device-side layer table (tensor maps + parameters) into a HOST buffer of
 * mega_conv_chain_plan_bytes(n) bytes (128-byte aligned) and the grid size to use; the caller copies the table to
 * device memory once (the tensors named by the descriptors must keep their addresses) and replays it with
 * mega_conv_chain_launch(). sync_words: 2 device uint32, zero-initialised once (the kernel leaves them zero);
 * launches that may overlap need distinct sync words and workspaces.
 * Replaces the per-layer launches of ResNet.forward / ResNetHead.forward / RPNHead.forward
 * (modeling/backbone/resnet.py:145-152, :201-204; modeling/rpn/rpn.py:99-106). */
long long mega_conv_chain_plan_bytes(int n_layers);
int mega_conv_chain_encode(const mega_conv_gemm_desc* descs, int n_layers, void* plan_host, long long plan_bytes,
                           int* grid_out);
int mega_conv_chain_launch(const void* plan_device, int n_layers, int grid, void* sync_words, void* stream, int pdl);
/* ABI v5: barrier depth. depth 1 = the calls above. depth 2: layer l waits for layer l-2 only, i.e. descs must be two
 * INDEPENDENT chains interleaved A0 B0 A1 B1 ... (the per-frame branch of the two halves of an image batch: chain B's
 * layer keeps every SM's TMA / MMA pipeline busy while chain A's layer drains its epilogue, stores and barrier), or any
 * order in which a layer reads nothing the layer directly before it wrote. sync_words: depth + 1 device uint32, zeroed
 * once. Odd layers use the second half of the workspace (tile counters / stream-K partial sums). */
int mega_conv_chain_encode2(const mega_conv_gemm_desc* descs, int n_layers, void* plan_host, long long plan_bytes,
                            int* grid_out, int depth);
int mega_conv_chain_launch2(const void* plan_device, int n_layers, int grid, void* sync_words, void* stream, int pdl,
                            int depth);
/* diagnostics: following chain launches record (tag, SM clock) events of CTA `cta` into trace_dev
 * ([3 roles][4096][2] uint64, zeroed by the caller); NULL switches tracing off (tools/trace_chain.py) */
int mega_conv_chain_set_trace(void* trace_dev, int cta);
/* level 1: per-layer events only, so that a 100-layer chain fits the buffer (tools/trace_backbone.py) */
int mega_conv_chain_set_trace2(void* trace_dev, int cta, int level);
/* 3xTF32 (precision 1): the tensor core adds into its fp32 TMEM accumulator with truncation, a bias that grows with
 * the number of MMAs accumulated; the kernel restarts the accumulator every `k_blocks` k-blocks (12 MMAs each) and folds
 * the segments into a master accumulator with round-to-nearest adds. 1..64, default 2; returns the previous value. */
int mega_set_split3_seg_len(int k_blocks);
/* precision 3: 1 = the A operand goes through tensor memory (tcgen05.cp per staged tile, TS-form MMAs; same results), 0 = both
 * operands from shared memory. Returns the previous setting. */
int mega_set_split16_a_tmem(int enable);
/* TMA fp32->tf32 conversion on load (round-to-nearest) on/off; returns the previous value. */
int mega_set_tf32_rounding(int enable);

/* ------------------------------------------------------------------- NMS
 * Greedy NMS, "+1" pixel convention, suppress when IoU > thresh; keep_out receives the kept
 * ORIGINAL indices in ascending order, *count_out their number (both device memory).
 * Replaces `_C.nms` -> nms_cuda (csrc/nms.h:10-28, csrc/cuda/nms.cu:70-131). n <= 8192.
 * Equal scores are ordered by ascending index (the reference leaves ties unspecified). */
long long mega_nms_workspace_bytes(int n);
int mega_nms(const float* boxes /*[n,4]*/, const float* scores /*[n]*/, int n, float thresh, void* workspace,
             long long workspace_bytes, long long* keep_out /*[n]*/, int* count_out, void* stream);

/* CPU tensors behind the same `_C` names (ABI v5): the reference dispatches nms / roi_align_forward on the tensor's
 * device (csrc/nms.h:10-28 -> cpu/nms_cpu.cpp:6-75; csrc/ROIAlign.h:11-25 -> cpu/ROIAlign_cpu.cpp:221-257; BASELINE
 * configs[0] runs with MODEL.DEVICE cpu). HOST pointers, fp32 (is_double 0) or fp64 (1) like AT_DISPATCH_FLOATING_TYPES;
 * bit-identical to the reference's CPU kernels, incl. the CPU rule "suppress when IoU >= thresh". */
int mega_nms_host(const void* boxes /*[n,4]*/, const void* scores /*[n]*/, int n, float thresh, int is_double,
                  long long* keep_out /*[n]*/, int* count_out);
int mega_roi_align_forward_nchw_host(const void* input, int batch, int channels, int height, int width, const void* rois,
                                     int num_rois, float spatial_scale, int pooled_h, int pooled_w, int sampling_ratio,
                                     int is_double, void* output);

/* ------------------------------------------------------- RPN proposal selection
 * sigmoid -> top-k (sorted) -> decode -> clip -> remove-small -> NMS -> first post_nms, per image.
 * Replaces RPNPostProcessor.forward_for_single_feature_map (modeling/rpn/inference.py:76-123),
 * BoxCoder.decode (modeling/box_coder.py:52-95), AnchorGenerator.grid_anchors
 * (modeling/rpn/anchor_generator.py:73-95; anchors are generated in-kernel from base_anchors).
 * head: NHWC rows of `ld` floats per cell: [0,A) objectness logits, [A,5A) deltas (a*4+c).
 * Outputs (per image, padded with zeros): out_boxes [n_img,post,4], out_scores [n_img,post],
 * out_anchor [n_img,post] (anchor index of each proposal, may be NULL), out_count [n_img]. */
long long mega_rpn_select_workspace_bytes(int n_img, int h, int w, int num_anchors, int pre_nms);
int mega_rpn_select(const float* head, long long head_img_stride, int ld, int n_img, int h, int w, int num_anchors,
                    int stride, const float* base_anchors, float im_w, float im_h, int pre_nms, int post_nms,
                    float nms_thresh, float min_size, void* workspace, long long workspace_bytes, float* out_boxes,
                    float* out_scores, int* out_anchor, int* out_count, void* stream);

/* ------------------------------------------------------------------- ROIAlign
 * Replaces `_C.roi_align_forward` (csrc/ROIAlign.h:11-25, csrc/cuda/ROIAlign_cuda.cu:257-299).
 * _nchw: reference layout (NCHW in, rois [K,5]=(batch,x1,y1,x2,y2), out [K,C,ph,pw]).
 * _nhwc: engine layout (NHWC in, out [K, ph*pw, C]); rois rows of roi_ld floats with the box at
 *        roi_box_off (roi_box_off < 0: packed [K,5] like the reference), batch index from
 *        roi_batch (int32, may be NULL = image 0). */
int mega_roi_align_forward_nchw(const float* input, int batch, int channels, int height, int width,
                                const float* rois, int num_rois, float spatial_scale, int pooled_h, int pooled_w,
                                int sampling_ratio, float* output, void* stream);
int mega_roi_align_forward_nhwc(const float* input, int channels, int height, int width, long long in_img_stride,
                                const float* rois, int roi_ld, int roi_box_off, const int* roi_batch, int num_rois,
                                float spatial_scale, int pooled_h, int pooled_w, int sampling_ratio, float* output,
                                long long out_roi_stride, void* stream);

/* fp16 feature map in, fp16 [K, ph*pw, C] out (the fp16-operand engine); interpolation arithmetic in fp32 as above,
 * one rounding to fp16 at the store. in_img_stride / out_roi_stride in halves. */
int mega_roi_align_forward_nhwc_f16(const void* input, int channels, int height, int width, long long in_img_stride,
                                    const float* rois, int roi_ld, int roi_box_off, const int* roi_batch,
                                    int num_rois, float spatial_scale, int pooled_h, int pooled_w, int sampling_ratio,
                                    void* output, long long out_roi_stride, void* stream);
/* ROIAlign over a split-fp16 NHWC map into split-fp16 rows (the strict engine's storage format, see mega_conv_gemm_desc):
 * separable kernel, channels % 128 == 0, bins <= 7 x 7, map <= 64 x 64 cells (MEGA_ERR_ARG otherwise). fp32 blends with
 * fused multiply-adds: equal to layers/roi_align.py:13-36 / ROIAlign_cuda.cu:62-115 to ~1e-6 relative, not bit for bit. */
int mega_roi_align_forward_nhwc_split16(const void* input, int channels, int height, int width, long long in_img_stride,
                                        const float* rois, int roi_ld, int roi_box_off, const int* roi_batch,
                                        int num_rois, float spatial_scale, int pooled_h, int pooled_w, int sampling_ratio,
                                        void* output, long long out_roi_stride, void* stream);

/* --------------------------------------------------------- backbone helpers
 * stem_im2col: NCHW image [N,3,H,W] -> [N, Ho*Wo, kpad] rows (k = c*49 + r*7 + s, zero padded) for
 * BaseStem.conv1 (7x7/2, pad 3; modeling/backbone/resnet.py:347-366); maxpool: F.max_pool2d(3,2,1)
 * in NHWC (resnet.py:365). */
int mega_stem_im2col(const float* input, int n_img, int height, int width, int kpad, float* out, void* stream);
int mega_maxpool3x3s2_nhwc(const float* input, int n_img, int height, int width, int channels, float* out,
                           void* stream);
/* fp16 variants: im2col rows / pooled map as __half (kpad % 8 == 0, channels % 8 == 0) */
int mega_stem_im2col_f16(const float* input, int n_img, int height, int width, int kpad, void* out, void* stream);
int mega_maxpool3x3s2_nhwc_f16(const void* input, int n_img, int height, int width, int channels, void* out,
                               void* stream);
/* stem_prep: NCHW fp32 image -> zero-bordered NHWC8 [N][H+6][wp][8] (3 real channels, wp even >= W+8; f16: __half):
 * BaseStem.conv1 then runs as a 7-slab implicit GEMM over overlapping 64-element windows (no im2col buffer). */
int mega_stem_prep(const float* input, int n_img, int height, int width, int wp, void* out, int f16, void* stream);
/* dst[i,:] = src[idx[i],:] (idx[i] < 0 -> zeros): replaces the per-frame torch.cat of the window /
 * memory deques (detector/generalized_rcnn_mega.py:213-216, roi_box_feature_extractors.py:674-688). */
int mega_gather_rows(const float* src, long long src_ld, const int* idx, int n_rows, int row_len, float* dst,
                     long long dst_ld, void* stream);
/* general form: dst[dst_idx ? dst_idx[i] : i, :] = src[src_idx ? src_idx[i] : i, :] (negative source index ->
 * zeros, negative destination index -> skipped): ring-buffer pushes of the window and the long-range memory. */
int mega_copy_rows(const float* src, long long src_ld, const int* src_idx, float* dst, long long dst_ld,
                   const int* dst_idx, int n_rows, int row_len, void* stream);
/* up to 16 independent mega_copy_rows jobs in one launch (rows of 32-bit words; the job table is a HOST array, it
 * travels in the kernel parameters). */
typedef struct mega_copy_job {
  const void* src;
  long long src_ld;
  const int* src_idx;
  void* dst;
  long long dst_ld;
  const int* dst_idx;
  int n_rows;
  int row_len;
} mega_copy_job;
int mega_copy_rows_batch(const mega_copy_job* jobs_host, int n_jobs, void* stream);
/* per image [rows, cols] -> [cols, rows] (NCHW <-> NHWC at the module boundary). */
int mega_transpose_2d(const float* input, int n_img, int rows, int cols, float* out, void* stream);

/* ------------------------------------------------------ relation-module soft-max
 * In place over logits [16][n_rows][ldm] (raw q.k, incl. the `u` term folded into q):
 *   p = softmax_m( log(relu(Wg.emb(box_q[n], box_k[m]) + bg) + 1e-6) + scale * logits )
 * with emb the 64-d sin/cos position embedding; boxes_q == NULL drops the position term.
 * Replaces extract_position_matrix / extract_position_embedding / the Wg conv / softmax of
 * roi_heads/box_head/roi_box_feature_extractors.py:125-176, :593-597, :624-633.
 * Keys m >= *m_valid_ptr (or m_host) get probability 0; query rows n with
 * *n_valid_ptr <= n < n_valid_off are padding and are skipped. dim_mat = 1000^(k/8), k=0..7. */
int mega_relation_softmax(float* logits, int n_rows, int ldm, const float* boxes_q, const float* boxes_k,
                          const float* wg, const float* bg, const float* dim_mat, const int* m_valid_ptr, int m_host,
                          const int* n_valid_ptr, int n_valid_off, float scale, void* stream);

/* same, but the probabilities are written as __half into probs_f16 [16][n_rows][ldm] (the A operand of the fp16
 * P.V' GEMM); `logits` is used as scratch. */
int mega_relation_softmax_f16(float* logits, void* probs_f16, int n_rows, int ldm, const float* boxes_q,
                              const float* boxes_k, const float* wg, const float* bg, const float* dim_mat,
                              const int* m_valid_ptr, int m_host, const int* n_valid_ptr, int n_valid_off, float scale,
                              void* stream);

/* the position-biased soft-max with Wg [16,64], bg [16] and dim_mat [8] given as HOST arrays: they travel in the
 * kernel parameters, so every weight is a constant-bank operand (no shared-memory traffic); probs_f16 may be NULL
 * (probabilities in place, fp32). Same arithmetic as mega_relation_softmax. */
int mega_relation_softmax_pe(float* logits, void* probs_f16, int n_rows, int ldm, const float* boxes_q,
                             const float* boxes_k, const float* wg_host, const float* bg_host,
                             const float* dim_mat_host, const int* m_valid_ptr, int m_host, const int* n_valid_ptr,
                             int n_valid_off, float scale, void* stream);
/* mega_relation_softmax_f16 / _pe with the probabilities written in the SPLIT-FP16 format (see mega_conv_gemm_desc): `probs`
 * is a tensor of the logits' shape and byte size (ldm % 32 == 0, 128-byte aligned) -- the A operand of the precision-3
 * P.V' product of the strict engine. */
int mega_relation_softmax_split16(float* logits, void* probs, int n_rows, int ldm, const float* boxes_q,
                                  const float* boxes_k, const float* wg, const float* bg, const float* dim_mat,
                                  const int* m_valid_ptr, int m_host, const int* n_valid_ptr, int n_valid_off, float scale,
                                  void* stream);
int mega_relation_softmax_pe_split16(float* logits, void* probs, int n_rows, int ldm, const float* boxes_q,
                                     const float* boxes_k, const float* wg_host, const float* bg_host,
                                     const float* dim_mat_host, const int* m_valid_ptr, int m_host, const int* n_valid_ptr,
                                     int n_valid_off, float scale, void* stream);

/* ------------------------------------------------------ box-head post-processing
 * softmax -> decode (weights wx..wh) -> clip -> per-class score threshold + NMS -> top max_det.
 * Replaces PostProcessor.forward / filter_results (roi_heads/box_head/inference.py:45-149).
 * Outputs in the reference's order (class by class, proposal index ascending):
 * out_boxes [out_cap,4], out_scores [out_cap], out_labels [out_cap] (int64), *out_count. */
long long mega_box_postprocess_workspace_bytes(int r_max, int num_classes);
int mega_box_postprocess(const float* logits, int ld_logits, const float* deltas, int ld_deltas,
                         const float* proposals, const int* count_ptr, int r_max, int num_classes, float im_w,
                         float im_h, float score_thresh, float nms_thresh, int max_det, float wx, float wy, float ww,
                         float wh, void* workspace, long long workspace_bytes, float* out_boxes, float* out_scores,
                         long long* out_labels, int out_cap, int* out_count, void* stream);

/* ------------------------------------------------------------------ FGFA (configs/FGFA, SURVEY row a19)
 * f16 != 0: element type __half, else float (the engine's activation type); arithmetic in fp32.
 * pool_image: image [3,H,W] fp32 -> [ceil(H/2), ceil(W/2), 4] = avg_pool2d(image / 255, 2, ceil_mode) with a zero 4th
 *   channel (FlowNetS.avgpool applied per frame, backbone/flownet.py:52-55; generalized_rcnn_fgfa.py:198).
 * build_pairs: ring [slots][hq*wq*4] of pooled frames -> pairs [n_frames][hq+6][wq+8][8] (key frame channels 0..2,
 *   frame i channels 4..6, zero borders): the A operand of FlowNetS.flow_conv1 as a row-wise implicit GEMM.
 * avgpool2_nhwc: F.avg_pool2d(2, stride 2, ceil_mode=True) on an NHWC map (flownet.py:113).
 * aggregate: resample (bilinear, border; generalized_rcnn_fgfa.py:45-62) of the cached [feats | embedding] maps of
 *   the window frames along `flow` [n_frames][h*w][flow_ld] fp32, cosine-similarity weights against the key frame's
 *   warped embedding, soft-max over frames, weighted sum of the warped feats (:64-76, :206-214) -> out [h*w][out_ld];
 *   weights_out (optional) [n_frames][h*w] fp32. */
int mega_fgfa_pool_image(const float* image, int height, int width, void* out, int f16, void* stream);
int mega_fgfa_build_pairs(const void* ring, long long slot_stride, const int* slots, int n_frames, int key_pos, int hq,
                          int wq, void* pairs, int f16, void* stream);
int mega_avgpool2_nhwc(const void* input, int n_img, int height, int width, int channels, long long in_ld, void* out,
                       long long out_ld, int f16, void* stream);
int mega_fgfa_aggregate(const void* ring, long long slot_stride, int ld, int feat_channels, int embed_channels,
                        const int* slots, int n_frames, int key_pos, const float* flow, int flow_ld, int height, int width,
                        void* out, long long out_ld, float* weights_out, int f16, void* stream);

/* DFF (configs/DFF, SURVEY section 8f row 4): out[h*w][out_ld] = resample(key_feats [h*w][ld], flow [h*w][flow_ld] fp32)
 * * scale [h*w][scale_ld] -- bilinear / border warp of the key frame's feature map along the flow, times FlowNetS's
 * scale map (detector/generalized_rcnn_dff.py:41-58, :131-134). channels % 8 == 0; f16 as above. */
int mega_dff_warp_scale(const void* key_feats, int ld, int channels, const float* flow, int flow_ld, const void* scale,
                        long long scale_ld, int height, int width, void* out, long long out_ld, int f16, void* stream);

/* -------------------------------------------- RetinaNet focal loss (csrc/SigmoidFocalLoss.h:10-32)
 * logits [N,C] fp32, targets [N] int32 in {-1 (ignore), 0 (background), 1..C}. */
int mega_sigmoid_focalloss_forward(const float* logits, const int* targets, int num_samples, int num_classes,
                                   float gamma, float alpha, float* losses, void* stream);
int mega_sigmoid_focalloss_backward(const float* logits, const int* targets, const float* d_losses, int num_samples,
                                    int num_classes, float gamma, float alpha, float* d_logits, void* stream);

/* --------------------------------------- deformable convolution v1 / v2 (csrc/deform_conv.h:11-28, :115)
 * Bilinear im2col of an NCHW input with per-tap offsets [B, dg*2*kh*kw, Ho, Wo] and (v2) masks
 * [B, dg*kh*kw, Ho, Wo] (mask == NULL: v1) into cols [B, Ho*Wo, kpad], k = c*kh*kw + i*kw + j; the
 * contraction with weight.view(Cout, C*kh*kw) then runs on mega_conv_gemm_tf32. */
int mega_deform_im2col(const float* input, const float* offset, const float* mask, int batch, int channels, int height,
                       int width, int kh, int kw, int pad_h, int pad_w, int stride_h, int stride_w, int dil_h, int dil_w,
                       int deformable_group, int kpad, float* cols, void* stream);

/* ------------------- deformable position-sensitive ROI pooling forward (csrc/deform_pool.h:11-37) */
int mega_deform_psroi_pooling_forward(const float* input, const float* rois, const float* trans, int num_rois,
                                      int channels, int height, int width, int no_trans, float spatial_scale,
                                      int output_dim, int group_size, int pooled_size, int part_size,
                                      int sample_per_part, float trans_std, int num_classes, float* out,
                                      float* top_count, void* stream);

/* ================================================================================================ ABI v4
 * Training-side / non-VID half of `mega_core._C` (csrc/vision.cpp:9-25): the backward ops and ROIPool. None of them is
 * on the inference hot path; they complete the 14-function operator surface (SURVEY.md section 8b). Scatter targets
 * (grad_input, trans_grad, and `out` of mega_channel_sum_nchw) are ACCUMULATED into with red.global.add.f32 and must be
 * initialised by the caller (the reference allocates them with at::zeros / torch.zeros_like). */

/* `_C.roi_align_backward` (csrc/ROIAlign.h:27-45 -> ROIAlign_cuda.cu:178-246, :302-346): grad [K,C,ph,pw], rois [K,5]
 * -> grad_input [batch,C,H,W] (zero-initialised by the caller). */
int mega_roi_align_backward_nchw(const float* grad, const float* rois, int num_rois, float spatial_scale, int pooled_h,
                                 int pooled_w, int batch, int channels, int height, int width, int sampling_ratio,
                                 float* grad_input, void* stream);

/* `_C.roi_pool_forward` / `_C.roi_pool_backward` (csrc/ROIPool.h:11-47 -> ROIPool_cuda.cu:16-202): max pooling over
 * integer bins; argmax [K,C,ph,pw] int32 = offset inside the (batch, c) plane, -1 for an empty bin. */
int mega_roi_pool_forward(const float* input, const float* rois, int num_rois, float spatial_scale, int channels,
                          int height, int width, int pooled_h, int pooled_w, float* output, int* argmax, void* stream);
int mega_roi_pool_backward(const float* grad, const int* argmax, const float* rois, int num_rois, int channels,
                           int height, int width, int pooled_h, int pooled_w, float* grad_input, void* stream);

/* Deformable convolution backward, v1 and modulated (csrc/deform_conv.h:45-113, :152-190). Column matrices use the
 * reference's own layout cols[k][b*ldp + p], k = c*kh*kw + i*kw + j, p = h_col*Wo + w_col, ldp >= Ho*Wo (pad to a
 * multiple of 4 so that a row is a TMA-legal GEMM operand; padding columns are not written -- zero them once).
 *   mega_deform_im2col_kq     : bilinear im2col of `input` (x mask when mask != NULL) into that layout: the B operand
 *                               of grad_weight = grad_out . cols^T;
 *   mega_deform_col2im_fused  : given gcols = weight^T . grad_out in that layout, ONE pass that produces grad_offset
 *                               (assigned), grad_mask (assigned; mask/grad_mask both NULL for v1) and scatters
 *                               grad_input (accumulated) -- the reference's deformable_col2im_coord + deformable_col2im
 *                               (deform_conv_kernel_cuda.cu:292-338, :375-426, :662-712, :714-780);
 *   mega_channel_sum_nchw     : out[c] += sum_{b,p} x[b,c,p] -- grad_bias (deform_conv_cuda.cu:667-672). */
int mega_deform_im2col_kq(const float* input, const float* offset, const float* mask, int batch, int channels,
                          int height, int width, int kh, int kw, int pad_h, int pad_w, int stride_h, int stride_w,
                          int dil_h, int dil_w, int deformable_group, int ldp, float* cols, void* stream);
int mega_deform_col2im_fused(const float* gcols, const float* input, const float* offset, const float* mask, int batch,
                             int channels, int height, int width, int kh, int kw, int pad_h, int pad_w, int stride_h,
                             int stride_w, int dil_h, int dil_w, int deformable_group, int ldp, float* grad_input,
                             float* grad_offset, float* grad_mask, void* stream);
int mega_channel_sum_nchw(const float* x, int batch, int channels, int plane, float* out, void* stream);

/* `_C.deform_psroi_pooling_backward` (csrc/deform_pool.h:41-69 -> deform_pool_kernel_cuda.cu:144-280): accumulates
 * input_grad [N,C,H,W] and trans_grad [K,2*num_classes,part,part] (trans / trans_grad may be NULL when no_trans). */
int mega_deform_psroi_pooling_backward(const float* out_grad, const float* input, const float* rois, const float* trans,
                                       const float* top_count, int num_rois, int channels, int height, int width,
                                       int no_trans, float spatial_scale, int output_dim, int group_size,
                                       int pooled_size, int part_size, int sample_per_part, float trans_std,
                                       int num_classes, float* input_grad, float* trans_grad, void* stream);

/* Test-time input transform of one decoded frame (SURVEY.md section 8f row 1): uint8 RGB on the device, interleaved
 * [src_h, src_w, 3] (src_pix_stride 3, src_ch_stride 1; what PIL / OpenCV decoders give) or planar [3, src_h, src_w]
 * (src_pix_stride 1, src_ch_stride = plane size; what nvJPEG via torchvision.io.decode_jpeg(device="cuda") gives),
 * src_row_stride bytes between rows -> fp32 [3, out_h, out_w], bit-identical to the reference's CPU pipeline
 * Resize (PIL bilinear) -> ToTensor -> Normalize(to_bgr255) (data/transforms/transforms.py:27-63, :117-135;
 * data/transforms/build.py:5-49). bounds_* / kk_* are Pillow's per-output (first tap, count) pairs and 2^22-scaled
 * integer coefficients (Resample.c precompute_coeffs + normalize_coeffs_8bpc), computed on the host by
 * mega_core.data.transforms.resample_tables and resident on the device; ksize_* == 0 skips a pass (size unchanged).
 * mean_host / std_host: 3 floats each, HOST pointers, in output channel order. */
int mega_image_transform_u8(const unsigned char* src, int src_h, int src_w, long long src_row_stride,
                            long long src_pix_stride, long long src_ch_stride, const int* bounds_h, const int* kk_h, int ksize_h, const int* bounds_v, const int* kk_v, int ksize_v, int out_h,
                            int out_w, const float* mean_host, const float* std_host, int to_bgr255, float* out,
                            void* stream);

/* HOST function (no device work, all pointers are host pointers): greedy matching of one image's detections of one class,
 * already sorted by descending score, against that class's ground-truth boxes -- the inner loops of
 * calc_detection_vid_prec_rec (data/datasets/evaluation/vid/vid_eval.py:201-262; SURVEY.md section 8f row 2).
 * match_out[j] in {0, 1}; pred_ignore_out[j] = the reference's pred_ignore entry (0, 1, a fraction, or empty_weight). */
int mega_vid_match_host(const float* pred_boxes, int n_pred, const float* gt_boxes, const unsigned char* gt_ignore,
                        int n_gt, float iou_thresh, double empty_weight, signed char* match_out,
                        double* pred_ignore_out);

/* ---------------------------------------------------------------- device VID evaluator (added to ABI v6)
 * These four symbols were added to v6 without changing anything before them, so mega_abi_version() stays 6.
 * calc_detection_vid_prec_rec + calc_detection_vid_ap for up to 4 motion ranges in one pass
 * (data/datasets/evaluation/vid/vid_eval.py:156-284, :287-343). Inputs are the BoxLists packed image after image:
 *   detections: det_boxes [n_det,4] xyxy, det_scores [n_det], det_labels [n_det] int32 in [0, num_classes);
 *   ground truth: gt_boxes [n_gt,4], gt_labels [n_gt], gt_motion [n_gt] fp64 motion IoU (NaN: none, never ignored;
 *   gt_motion NULL: nothing is ignored); det_offsets / gt_offsets [n_img+1] int64 prefix sums of the per-image counts.
 * Boxes satisfy x2 > x1 - 2 and y2 > y1 - 2. num_classes <= 512, n_ranges 1..4, n_det and n_gt < 2^31.
 * ranges_host [n_ranges][2] = (lo, hi): a GT is ignored for a range when its motion IoU lies outside [lo, hi]
 * (vid_eval.py:176-186); empty_weight_host [n_ranges]: the ignore weight of detections of a class without GT in the image
 * (vid_eval.py:160-169, 206). Ranking rule: descending score, equal scores in the order of numpy's
 * argsort(kind="stable")[::-1] inside each (image, class) and over each class (the reference's own argsort()[::-1] leaves
 * equal scores in an unspecified order, vid_eval.py:191, :265). All four calls share one workspace of
 * mega_vid_eval_workspace_bytes() bytes (-1: sizes out of range), run in stream order and are called in this order. */
long long mega_vid_eval_workspace_bytes(long long n_det, long long n_gt, int num_classes, int n_ranges);
/* Per (image, class): greedy matching for every range (vid_eval.py:188-250). match_out [n_ranges][n_det] int8 (1 =
 * matched), ignore_out [n_ranges][n_det] fp64 (the reference's pred_ignore), n_pos_out [n_ranges][num_classes] int64
 * (non-ignored GT, vid_eval.py:199), seen_out [num_classes] int32 (1 = label occurs in a prediction or GT: prec exists),
 * det_count_out [num_classes] int32 detections per class. Zeroes its outputs itself. */
int mega_vid_eval_match(const float* det_boxes, const float* det_scores, const int* det_labels,
                        const long long* det_offsets, const float* gt_boxes, const int* gt_labels, const double* gt_motion,
                        const long long* gt_offsets, int n_img, long long n_det, long long n_gt, int num_classes,
                        int n_ranges, const double* ranges_host, const double* empty_weight_host, float iou_thresh,
                        void* workspace, long long workspace_bytes, signed char* match_out, double* ignore_out,
                        long long* n_pos_out, int* seen_out, int* det_count_out, void* stream);
/* Stable radix sort of all detections by (class, score) ascending (vid_eval.py:260-268 for every class at once):
 * order_out [n_det] = detection indices; class c occupies det_count[c] entries after those of the classes below it, and
 * read backwards each class is in ranking order. */
int mega_vid_eval_rank(long long n_det, long long n_gt, int num_classes, int n_ranges, void* workspace,
                       long long workspace_bytes, int* order_out, void* stream);
/* Per (class, range): tp / fp cumulative sums, prec = tp / (fp + tp + eps), rec = tp / n_pos (vid_eval.py:269-282) and
 * ap_out [n_ranges][num_classes] = area under the precision envelope (vid_eval.py:287-343, use_07_metric=False; NaN where
 * n_pos == 0). prec_out / rec_out [n_ranges][n_det] (may be NULL): class c's curve at the offset of its block in order,
 * in ranking order; rec_out is written for classes with n_pos > 0 only. Same bits on every run. */
int mega_vid_eval_scan_ap(const signed char* match, const double* ignore, const int* order, const int* det_count,
                          const long long* n_pos, long long n_det, long long n_gt, int num_classes, int n_ranges,
                          void* workspace, long long workspace_bytes, double* prec_out, double* rec_out, double* ap_out,
                          void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MEGA_B200_H_ */

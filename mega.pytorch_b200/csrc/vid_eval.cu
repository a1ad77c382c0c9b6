// The VID evaluator's native code (SURVEY.md section 8f row 2).
//
// mega_vid_match_host: the per-(image, class) greedy matching of score-sorted detections against ground truth, which the
// reference runs as nested Python loops over 176 k images x classes x detections x boxes
// (data/datasets/evaluation/vid/vid_eval.py:201-262), as a host function that the host evaluator calls once per
// (image, class). float32 IoU arithmetic in the order of boxlist_iou (structures/boxlist_ops.py:75-88) on the "+1" boxes
// of vid_eval.py:213-217, so decisions are identical.
//
// The device evaluator (below mega_vid_match_host) scores a whole run on the GPU, every motion range in one pass:
//   vid_match_kernel    one CTA per image, one warp per (image, class) segment: the segment body of vid_eval.cuh
//                       (sort by score, greedy matching for each range), the non-ignored GT counts n_pos[range][class],
//                       and the radix-sort input (class, score key) of every detection;
//   radix_*_kernel      stable LSD radix sort of all detections by (class, order-preserving score bits), 8-bit digits;
//   vid_scan_ap_kernel  one CTA per (class, range): tp / fp cumulative sums, precision / recall and the area under the
//                       precision envelope, in fixed reduction trees (same bits on every run, no float atomics).
#include <vector>
#include "common.cuh"
#include "mega_b200.h"

extern "C" int mega_vid_match_host(const float* pred_boxes, int n_pred, const float* gt_boxes,
                                   const unsigned char* gt_ignore, int n_gt, float iou_thresh, double empty_weight,
                                   signed char* match_out, double* pred_ignore_out) {
  MEGA_ARG_CHECK(n_pred >= 0 && n_gt >= 0, "vid_match: negative sizes");
  if (n_pred == 0) return MEGA_OK;
  if (n_gt == 0) {                                   // vid_eval.py:207-210
    for (int j = 0; j < n_pred; ++j) match_out[j] = 0, pred_ignore_out[j] = empty_weight;
    return MEGA_OK;
  }
  std::vector<float> garea(n_gt), gx1(n_gt), gy1(n_gt), gx2(n_gt), gy2(n_gt);
  int n_ignored = 0;
  for (int k = 0; k < n_gt; ++k) {
    gx1[k] = gt_boxes[4 * k], gy1[k] = gt_boxes[4 * k + 1];
    gx2[k] = gt_boxes[4 * k + 2] + 1.0f, gy2[k] = gt_boxes[4 * k + 3] + 1.0f;       // integer-typed boxes: [:, 2:] += 1
    garea[k] = (gx2[k] - gx1[k] + 1.0f) * (gy2[k] - gy1[k] + 1.0f);
    n_ignored += gt_ignore[k] ? 1 : 0;
  }
  std::vector<unsigned char> selec(n_gt, 0);
  for (int j = 0; j < n_pred; ++j) {
    const float px1 = pred_boxes[4 * j], py1 = pred_boxes[4 * j + 1];
    const float px2 = pred_boxes[4 * j + 2] + 1.0f, py2 = pred_boxes[4 * j + 3] + 1.0f;
    const float parea = (px2 - px1 + 1.0f) * (py2 - py1 + 1.0f);
    double iou_match = iou_thresh, iou_match_ig = -1.0, iou_match_nig = -1.0;
    int arg_match = -1;
    for (int k = 0; k < n_gt; ++k) {
      const float ltx = px1 > gx1[k] ? px1 : gx1[k], lty = py1 > gy1[k] ? py1 : gy1[k];
      const float rbx = px2 < gx2[k] ? px2 : gx2[k], rby = py2 < gy2[k] ? py2 : gy2[k];
      float w = rbx - ltx + 1.0f, h = rby - lty + 1.0f;
      w = w < 0.f ? 0.f : w, h = h < 0.f ? 0.f : h;
      const float inter = w * h;
      const float iou = inter / (parea + garea[k] - inter);
      const double v = iou;
      if (gt_ignore[k] && v > iou_match_ig) iou_match_ig = v;
      if (!gt_ignore[k] && v > iou_match_nig) iou_match_nig = v;
      if (selec[k] || v < iou_match) continue;
      if (v == iou_match) {
        if (arg_match < 0 || gt_ignore[arg_match]) arg_match = k;
      } else {
        arg_match = k;
      }
      iou_match = v;
    }
    if (arg_match >= 0) {
      match_out[j] = 1;
      pred_ignore_out[j] = gt_ignore[arg_match] ? 1.0 : 0.0;
      selec[arg_match] = 1;
    } else {
      match_out[j] = 0;
      if (iou_match_nig > iou_match_ig) pred_ignore_out[j] = 0.0;
      else if (iou_match_ig > iou_match_nig) pred_ignore_out[j] = 1.0;
      else pred_ignore_out[j] = static_cast<double>(n_ignored) / static_cast<double>(n_gt);
    }
  }
  return MEGA_OK;
}

// ====================================================================================================== device evaluator
#include <math.h>
#include "vid_eval.cuh"

namespace {

using mega_vid::Best;
using mega_vid::kMaxRanges;

constexpr int kMatchThreads = 256;
constexpr int kMatchWarps = kMatchThreads / 32;
constexpr int kStageDets = 512;      // an image's detections staged in shared memory; larger images run from global memory
constexpr int kStageGt = 128;
constexpr int kMaxClasses = 512;
constexpr int kRadixThreads = 256;
constexpr int kRadixWarps = kRadixThreads / 32;
constexpr int kRadixItems = 16;      // per thread: a warp owns 512 consecutive keys, a block 4096
constexpr int kRadixTile = kRadixThreads * kRadixItems;
constexpr int kScanThreads = 512;
constexpr int kScanItems = 8;
constexpr int kScanTile = kScanThreads * kScanItems;
constexpr double kEps = 2.220446049250313e-16;   // np.spacing(1)

// device lane policy of mega_vid::match_segment: one warp, butterfly reduction of the per-lane folds
struct WarpLanes {
  __device__ int lane() const { return threadIdx.x & 31; }
  __device__ int width() const { return 32; }
  __device__ void sync() const { __syncwarp(); }
  template <int R, class F>
  __device__ void fold(int n, Best* out, F&& f) const {
    for (int p = lane(); p < n; p += 32) f(p, out);
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
#pragma unroll
      for (int r = 0; r < R; ++r) {
        Best o;
        o.v = __shfl_xor_sync(0xffffffffu, out[r].v, off);
        o.k = __shfl_xor_sync(0xffffffffu, out[r].k, off);
        o.pos = __shfl_xor_sync(0xffffffffu, out[r].pos, off);
        o.ign = __shfl_xor_sync(0xffffffffu, out[r].ign, off);
        o.ig = __shfl_xor_sync(0xffffffffu, out[r].ig, off);
        o.nig = __shfl_xor_sync(0xffffffffu, out[r].nig, off);
        out[r] = mega_vid::combine(out[r], o);
      }
    }
  }
};

// ---------------------------------------------------------------------------------------------------- workspace layout
// [radix keys x2 | radix values x2 | digit counts] [tile carries of the scans] [match scratch of large images]
struct Layout {
  long long keys0, keys1, vals0, vals1, counts, tile_tp, tile_fp, dsort, dorder, gsort, gsel, total;
  long long radix_blocks, tiles_per_range;
};
long long align256(long long x) { return (x + 255) & ~255LL; }
Layout layout(long long n_det, long long n_gt, int num_classes, int n_ranges) {
  Layout L;
  L.radix_blocks = (n_det + kRadixTile - 1) / kRadixTile;
  // a class segment starting at s with n items owns tiles [s / T + c, s / T + c + ceil(n / T)): disjoint over classes
  L.tiles_per_range = n_det / kScanTile + num_classes + 1;
  long long o = 0;
  L.keys0 = o, o = align256(o + 8 * n_det);
  L.keys1 = o, o = align256(o + 8 * n_det);
  L.vals0 = o, o = align256(o + 4 * n_det);
  L.vals1 = o, o = align256(o + 4 * n_det);
  L.counts = o, o = align256(o + 4 * 256 * L.radix_blocks);
  L.tile_tp = o, o = align256(o + 4 * n_ranges * L.tiles_per_range);
  L.tile_fp = o, o = align256(o + 8 * n_ranges * L.tiles_per_range);
  L.dsort = o, o = align256(o + 4 * n_det);
  L.dorder = o, o = align256(o + 4 * n_det);
  L.gsort = o, o = align256(o + 4 * n_gt);
  L.gsel = o, o = align256(o + n_gt * n_ranges);
  L.total = o;
  return L;
}
int class_bits(int num_classes) {
  int b = 0;
  while ((1 << b) < num_classes) ++b;
  return b;
}

// -------------------------------------------------------------------------------------------------------- matching
struct MatchParams {
  const float* det_boxes;
  const float* det_scores;
  const int* det_labels;
  const long long* det_off;
  const float* gt_boxes;
  const int* gt_labels;
  const double* gt_motion;
  const long long* gt_off;
  int num_classes;
  long long n_det;
  double lo[kMaxRanges], hi[kMaxRanges], empty[kMaxRanges];
  float iou_thresh;
  signed char* match;
  double* ignore;
  unsigned long long* n_pos;   // [R][C]
  int* seen;                   // [C]
  int* det_count;              // [C]
  uint64_t* keys;              // radix input, position p = det_off[i] + (n_i - 1 - j) for detection j of image i
  int* vals;
  int* ws_dsort;
  int* ws_dorder;
  int* ws_gsort;
  unsigned char* ws_gsel;
};

// exclusive scan of cnt[0..n) into start[0..n] by warp 0 (n <= kMaxClasses)
__device__ void class_starts(const int* cnt, int* start, int n) {
  if (threadIdx.x >= 32) return;
  const int lane = threadIdx.x;
  int carry = 0;
  for (int base = 0; base < n; base += 32) {
    const int c = base + lane;
    const int v = c < n ? cnt[c] : 0;
    int x = v;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
      const int y = __shfl_up_sync(0xffffffffu, x, off);
      if (lane >= off) x += y;
    }
    if (c < n) start[c] = carry + x - v;
    carry += __shfl_sync(0xffffffffu, x, 31);
  }
  if (lane == 0) start[n] = carry;
}

template <int R>
__global__ void __launch_bounds__(kMatchThreads) vid_match_kernel(const MatchParams p) {
  __shared__ float4 s_dbox[kStageDets];
  __shared__ float s_dscore[kStageDets];
  __shared__ int s_dsort[kStageDets], s_dorder[kStageDets];
  __shared__ float4 s_gbox[kStageGt];
  __shared__ double s_gmotion[kStageGt];
  __shared__ int s_gsort[kStageGt];
  __shared__ unsigned char s_gsel[kStageGt * R];
  __shared__ int s_dstart[kMaxClasses + 1], s_dcur[kMaxClasses];
  __shared__ int s_gstart[kMaxClasses + 1], s_gcur[kMaxClasses];

  const int img = blockIdx.x, tid = threadIdx.x, C = p.num_classes;
  const long long doff = p.det_off[img], goff = p.gt_off[img];
  const int nd = static_cast<int>(p.det_off[img + 1] - doff), ng = static_cast<int>(p.gt_off[img + 1] - goff);
  const bool dstage = nd <= kStageDets, gstage = ng <= kStageGt;
  const float* gdbox = p.det_boxes + 4 * doff;
  const float* gdscore = p.det_scores + doff;
  const int* gdlab = p.det_labels + doff;
  const float* ggbox = p.gt_boxes + 4 * goff;
  const int* gglab = p.gt_labels + goff;
  const double* ggmot = p.gt_motion ? p.gt_motion + goff : nullptr;

  for (int c = tid; c < C; c += kMatchThreads) s_dcur[c] = 0, s_gcur[c] = 0;
  __syncthreads();
  for (int j = tid; j < nd; j += kMatchThreads) {
    const float sc = gdscore[j];
    const int lab = gdlab[j];
    if (dstage) {
      s_dbox[j] = make_float4(gdbox[4 * j], gdbox[4 * j + 1], gdbox[4 * j + 2], gdbox[4 * j + 3]);
      s_dscore[j] = sc;
    }
    const long long pos = doff + (nd - 1 - j);
    p.keys[pos] = (static_cast<uint64_t>(static_cast<uint32_t>(lab)) << 32) | mega_vid::score_key(sc);
    p.vals[pos] = static_cast<int>(doff + j);
    if (lab >= 0 && lab < C) atomicAdd(&s_dcur[lab], 1);
  }
  for (int k = tid; k < ng; k += kMatchThreads) {
    if (gstage) {
      s_gbox[k] = make_float4(ggbox[4 * k], ggbox[4 * k + 1], ggbox[4 * k + 2], ggbox[4 * k + 3]);
      if (ggmot) s_gmotion[k] = ggmot[k];
    }
    const int lab = gglab[k];
    if (lab >= 0 && lab < C) atomicAdd(&s_gcur[lab], 1);
  }
  __syncthreads();
  class_starts(s_dcur, s_dstart, C);
  __syncthreads();
  class_starts(s_gcur, s_gstart, C);
  __syncthreads();
  for (int c = tid; c < C; c += kMatchThreads) s_dcur[c] = s_dstart[c], s_gcur[c] = s_gstart[c];
  __syncthreads();
  // bucket by class; the order inside a bucket is irrelevant (the segment body orders detections by (score, index) and
  // breaks GT ties by index)
  int* dsort = dstage ? s_dsort : p.ws_dsort + doff;
  int* dorder = dstage ? s_dorder : p.ws_dorder + doff;
  int* gsort = gstage ? s_gsort : p.ws_gsort + goff;
  unsigned char* gsel = gstage ? s_gsel : p.ws_gsel + goff * R;
  for (int j = tid; j < nd; j += kMatchThreads) {
    const int lab = gdlab[j];
    if (lab >= 0 && lab < C) dsort[atomicAdd(&s_dcur[lab], 1)] = j;
  }
  for (int k = tid; k < ng; k += kMatchThreads) {
    const int lab = gglab[k];
    if (lab >= 0 && lab < C) gsort[atomicAdd(&s_gcur[lab], 1)] = k;
  }
  __syncthreads();

  const float* dbox = dstage ? reinterpret_cast<const float*>(s_dbox) : gdbox;
  const float* dscore = dstage ? s_dscore : gdscore;
  const float* gbox = gstage ? reinterpret_cast<const float*>(s_gbox) : ggbox;
  const double* gmot = ggmot ? (gstage ? s_gmotion : ggmot) : nullptr;
  const int warp = tid >> 5, lane = tid & 31;
  for (int c = warp; c < C; c += kMatchWarps) {
    const int d0 = s_dstart[c], dn = s_dstart[c + 1] - d0;
    const int g0 = s_gstart[c], gn = s_gstart[c + 1] - g0;
    if (dn == 0 && gn == 0) continue;
#pragma unroll
    for (int r = 0; r < R; ++r) {
      int cnt = 0;
      for (int q = lane; q < gn; q += 32) cnt += !mega_vid::gt_ignored(gmot, gsort[g0 + q], p.lo[r], p.hi[r]);
      cnt = __reduce_add_sync(0xffffffffu, cnt);
      if (lane == 0 && cnt) atomicAdd(p.n_pos + static_cast<long long>(r) * C + c, static_cast<unsigned long long>(cnt));
    }
    if (lane == 0) {
      p.seen[c] = 1;
      if (dn) atomicAdd(p.det_count + c, dn);
    }
    mega_vid::match_segment<R>(WarpLanes(), dbox, dscore, dsort + d0, dn, gbox, gmot, gsort + g0, gn, p.lo, p.hi, p.empty,
                               p.iou_thresh, dorder + d0, gsel + static_cast<long long>(g0) * R, p.match + doff,
                               p.ignore + doff, p.n_det);
  }
}

// ------------------------------------------------------------------------------------------------------ radix sort
// Stable LSD pass over 8 bits at `shift`: per-block digit counts -> one exclusive scan (digit-major, so the scan gives
// every (digit, block) its global offset) -> scatter, each warp ranking its 32-key rounds with __match_any_sync.
__device__ __forceinline__ int radix_digit(uint64_t k, int shift) { return static_cast<int>((k >> shift) & 0xff); }

__global__ void __launch_bounds__(kRadixThreads) radix_count_kernel(const uint64_t* keys, long long n, int shift,
                                                                    int* counts, long long n_blocks) {
  __shared__ int s_cnt[256];
  s_cnt[threadIdx.x] = 0;
  __syncthreads();
  const long long base = static_cast<long long>(blockIdx.x) * kRadixTile;
  for (int i = threadIdx.x; i < kRadixTile; i += kRadixThreads)
    if (base + i < n) atomicAdd(&s_cnt[radix_digit(keys[base + i], shift)], 1);
  __syncthreads();
  counts[static_cast<long long>(threadIdx.x) * n_blocks + blockIdx.x] = s_cnt[threadIdx.x];
}

// in-place exclusive scan of counts[0..m) by one block of 1024 threads, 4096 values per round
__global__ void __launch_bounds__(1024) radix_scan_kernel(int* counts, long long m) {
  __shared__ int s_warp[32];
  __shared__ int s_carry;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) s_carry = 0;
  __syncthreads();
  for (long long base = 0; base < m; base += 4096) {
    int v[4], sum = 0;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const long long idx = base + 4 * tid + i;
      v[i] = idx < m ? counts[idx] : 0;
      sum += v[i];
    }
    int x = sum;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
      const int y = __shfl_up_sync(0xffffffffu, x, off);
      if (lane >= off) x += y;
    }
    if (lane == 31) s_warp[warp] = x;
    __syncthreads();
    if (warp == 0) {
      int w = s_warp[lane];
#pragma unroll
      for (int off = 1; off < 32; off <<= 1) {
        const int y = __shfl_up_sync(0xffffffffu, w, off);
        if (lane >= off) w += y;
      }
      s_warp[lane] = w;
    }
    __syncthreads();
    int run = s_carry + x - sum + (warp ? s_warp[warp - 1] : 0);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const long long idx = base + 4 * tid + i;
      if (idx < m) counts[idx] = run;
      run += v[i];
    }
    __syncthreads();
    if (tid == 0) s_carry += s_warp[31];
    __syncthreads();
  }
}

__global__ void __launch_bounds__(kRadixThreads) radix_scatter_kernel(const uint64_t* keys_in, const int* vals_in,
                                                                      long long n, int shift, const int* offsets,
                                                                      long long n_blocks, uint64_t* keys_out,
                                                                      int* vals_out) {
  __shared__ int s_cnt[kRadixWarps][257];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (int i = tid; i < kRadixWarps * 257; i += kRadixThreads) (&s_cnt[0][0])[i] = 0;
  __syncthreads();
  const long long wbase = static_cast<long long>(blockIdx.x) * kRadixTile + warp * (32 * kRadixItems);
  const unsigned lt = (1u << lane) - 1;
  // pass 1: per-warp digit counts
  for (int it = 0; it < kRadixItems; ++it) {
    const long long i = wbase + it * 32 + lane;
    const int d = i < n ? radix_digit(keys_in[i], shift) : 256;
    const unsigned peers = __match_any_sync(0xffffffffu, d);
    if (d < 256 && (peers & lt) == 0) s_cnt[warp][d] += __popc(peers);
    __syncwarp();
  }
  __syncthreads();
  // per digit: global offset of this block, then the warps in order
  {
    const int d = tid;
    int run = offsets[static_cast<long long>(d) * n_blocks + blockIdx.x];
    for (int w = 0; w < kRadixWarps; ++w) {
      const int t = s_cnt[w][d];
      s_cnt[w][d] = run;
      run += t;
    }
  }
  __syncthreads();
  // pass 2: scatter in key order
  for (int it = 0; it < kRadixItems; ++it) {
    const long long i = wbase + it * 32 + lane;
    const bool ok = i < n;
    const uint64_t k = ok ? keys_in[i] : 0;
    const int d = ok ? radix_digit(k, shift) : 256;
    const unsigned peers = __match_any_sync(0xffffffffu, d);
    if (ok) {
      const int dst = s_cnt[warp][d] + __popc(peers & lt);
      keys_out[dst] = k;
      vals_out[dst] = vals_in[i];
    }
    __syncwarp();
    if (ok && (peers & lt) == 0) s_cnt[warp][d] += __popc(peers);
    __syncwarp();
  }
}

// --------------------------------------------------------------------------------------------- scans and AP per class
struct ScanParams {
  const signed char* match;
  const double* ignore;
  const int* order;
  const int* det_count;
  const unsigned long long* n_pos;
  long long n_det;
  int num_classes;
  int* tile_tp;
  double* tile_fp;
  long long tiles_per_range;
  double* prec_out;
  double* rec_out;
  double* ap_out;
};

// block scan of (int, double) pairs in thread order (fixed tree): this thread's exclusive prefix and the total
__device__ void block_scan(int tp, double fp, int* s_tp, double* s_fp, int& ex_tp, double& ex_fp, int& tot_tp,
                           double& tot_fp) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  constexpr int kWarps = kScanThreads / 32;
  int xt = tp;
  double xf = fp;
#pragma unroll
  for (int off = 1; off < 32; off <<= 1) {
    const int yt = __shfl_up_sync(0xffffffffu, xt, off);
    const double yf = __shfl_up_sync(0xffffffffu, xf, off);
    if (lane >= off) xt += yt, xf = yf + xf;
  }
  if (lane == 31) s_tp[warp] = xt, s_fp[warp] = xf;
  __syncthreads();
  if (warp == 0) {
    int wt = lane < kWarps ? s_tp[lane] : 0;
    double wf = lane < kWarps ? s_fp[lane] : 0.0;
#pragma unroll
    for (int off = 1; off < kWarps; off <<= 1) {
      const int yt = __shfl_up_sync(0xffffffffu, wt, off);
      const double yf = __shfl_up_sync(0xffffffffu, wf, off);
      if (lane >= off) wt += yt, wf = yf + wf;
    }
    if (lane < kWarps) s_tp[lane] = wt, s_fp[lane] = wf;
  }
  __syncthreads();
  int lt = __shfl_up_sync(0xffffffffu, xt, 1);
  double lf = __shfl_up_sync(0xffffffffu, xf, 1);
  if (lane == 0) lt = 0, lf = 0.0;
  ex_tp = warp ? s_tp[warp - 1] + lt : lt;
  ex_fp = warp ? (lane ? s_fp[warp - 1] + lf : s_fp[warp - 1]) : lf;
  tot_tp = s_tp[kWarps - 1];
  tot_fp = s_fp[kWarps - 1];
  __syncthreads();
}

// tp / fp increments of the element at place t (host order: descending score) of class segment [start, start + n)
__device__ __forceinline__ void element(const ScanParams& p, int r, long long start, int n, int t, int& tp, double& fp) {
  tp = 0, fp = 0.0;
  if (t >= n) return;
  const int e = p.order[start + n - 1 - t];
  const signed char m = p.match[static_cast<long long>(r) * p.n_det + e];
  const double w = p.ignore[static_cast<long long>(r) * p.n_det + e];
  if (w == 1.0) return;                          // fully ignored: neither tp nor fp
  if (m == 1) tp = 1;
  else if (m == 0) fp = w == 0.0 ? 1.0 : w;      // fractional weight of a "mixed" miss
}

// One tile of the forward cumulative sums: tp[i] / fp[i] (inclusive) of this thread's kScanItems elements, tp_before
// the count before its first one.
__device__ void scan_tile(const ScanParams& p, int r, long long start, int n, int t0, int carry_tp, double carry_fp,
                          int* s_tp, double* s_fp, int (&tp)[kScanItems], double (&fp)[kScanItems], int& tp_before,
                          int& tot_tp, double& tot_fp) {
  const int tb = t0 + threadIdx.x * kScanItems;
  int st = 0;
  double sf = 0.0;
#pragma unroll
  for (int i = 0; i < kScanItems; ++i) {
    int a;
    double b;
    element(p, r, start, n, tb + i, a, b);
    st += a, sf = sf + b;
    tp[i] = st, fp[i] = sf;
  }
  int ex_tp;
  double ex_fp;
  block_scan(st, sf, s_tp, s_fp, ex_tp, ex_fp, tot_tp, tot_fp);
  const int bt = carry_tp + ex_tp;
  const double bf = carry_fp + ex_fp;
  tp_before = bt;
#pragma unroll
  for (int i = 0; i < kScanItems; ++i) tp[i] += bt, fp[i] = bf + fp[i];
}

__global__ void __launch_bounds__(kScanThreads) vid_scan_ap_kernel(const ScanParams p) {
  __shared__ int s_tp[32];
  __shared__ double s_fp[32];
  __shared__ double s_red[32];
  __shared__ long long s_start;
  const int c = blockIdx.x, r = blockIdx.y, C = p.num_classes, tid = threadIdx.x;
  if (tid == 0) {
    long long s = 0;
    for (int k = 0; k < c; ++k) s += p.det_count[k];
    s_start = s;
  }
  __syncthreads();
  const long long start = s_start;
  const int n = p.det_count[c];
  const unsigned long long npos = p.n_pos[static_cast<long long>(r) * C + c];
  const double dpos = static_cast<double>(npos);
  const int n_tiles = (n + kScanTile - 1) / kScanTile;
  int* ttp = p.tile_tp + r * p.tiles_per_range + start / kScanTile + c;
  double* tfp = p.tile_fp + r * p.tiles_per_range + start / kScanTile + c;
  double* prec_out = p.prec_out ? p.prec_out + static_cast<long long>(r) * p.n_det + start : nullptr;
  double* rec_out = p.rec_out && npos ? p.rec_out + static_cast<long long>(r) * p.n_det + start : nullptr;

  // forward: carry into every tile (and precision / recall when asked for)
  int carry_tp = 0;
  double carry_fp = 0.0;
  for (int k = 0; k < n_tiles; ++k) {
    if (tid == 0) ttp[k] = carry_tp, tfp[k] = carry_fp;
    int tp[kScanItems], tp_before, tot_tp;
    double fp[kScanItems], tot_fp;
    scan_tile(p, r, start, n, k * kScanTile, carry_tp, carry_fp, s_tp, s_fp, tp, fp, tp_before, tot_tp, tot_fp);
    if (prec_out || rec_out) {
      const int tb = k * kScanTile + tid * kScanItems;
#pragma unroll
      for (int i = 0; i < kScanItems; ++i) {
        if (tb + i >= n) break;
        const double dtp = static_cast<double>(tp[i]);
        if (prec_out) prec_out[tb + i] = dtp / (fp[i] + dtp + kEps);
        if (rec_out) rec_out[tb + i] = dtp / dpos;
      }
    }
    carry_tp += tot_tp, carry_fp = carry_fp + tot_fp;
  }
  __syncthreads();
  if (npos == 0) {                               // rec is None: AP is NaN (calc_detection_vid_ap)
    if (tid == 0) p.ap_out[static_cast<long long>(r) * C + c] = NAN;
    return;
  }
  // backward: precision envelope (suffix max) and sum of (rec[i] - rec[i-1]) * envelope[i] where recall moves
  double env_carry = 0.0, acc = 0.0;
  const int lane = tid & 31, warp = tid >> 5;
  constexpr int kWarps = kScanThreads / 32;
  for (int k = n_tiles - 1; k >= 0; --k) {
    int tp[kScanItems], tp_before, tot_tp;
    double fp[kScanItems], tot_fp;
    __syncthreads();
    scan_tile(p, r, start, n, k * kScanTile, ttp[k], tfp[k], s_tp, s_fp, tp, fp, tp_before, tot_tp, tot_fp);
    const int tb = k * kScanTile + tid * kScanItems;
    double pr[kScanItems], tmax = 0.0;
#pragma unroll
    for (int i = kScanItems - 1; i >= 0; --i) {
      const double dtp = static_cast<double>(tp[i]);
      pr[i] = tb + i < n ? dtp / (fp[i] + dtp + kEps) : 0.0;
      tmax = fmax(tmax, pr[i]);
      pr[i] = tmax;                              // suffix max inside the thread
    }
    // suffix max over the threads after this one, then over the later tiles
    double x = tmax;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
      const double y = __shfl_down_sync(0xffffffffu, x, off);
      if (lane + off < 32) x = fmax(x, y);
    }
    if (lane == 0) s_red[warp] = x;
    __syncthreads();
    double later = env_carry, tile_max = env_carry;
    for (int w = 0; w < kWarps; ++w) {
      tile_max = fmax(tile_max, s_red[w]);
      if (w > warp) later = fmax(later, s_red[w]);
    }
    const double nxt = __shfl_down_sync(0xffffffffu, x, 1);
    if (lane < 31) later = fmax(later, nxt);
#pragma unroll
    for (int i = 0; i < kScanItems; ++i) {
      if (tb + i >= n) break;
      const double env = fmax(pr[i], later);
      const double rec = static_cast<double>(tp[i]) / dpos;
      const double rprev = static_cast<double>(i ? tp[i - 1] : tp_before) / dpos;
      if (rec != rprev) acc += (rec - rprev) * env;
    }
    env_carry = tile_max;
  }
  // fixed-tree block sum
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) acc += __shfl_down_sync(0xffffffffu, acc, off);
  __syncthreads();
  if (lane == 0) s_red[warp] = acc;
  __syncthreads();
  if (warp == 0) {
    double v = lane < kWarps ? s_red[lane] : 0.0;
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) v += __shfl_down_sync(0xffffffffu, v, off);
    if (lane == 0) p.ap_out[static_cast<long long>(r) * C + c] = v;
  }
}

}  // namespace

extern "C" long long mega_vid_eval_workspace_bytes(long long n_det, long long n_gt, int num_classes, int n_ranges) {
  if (n_det < 0 || n_det >= (1LL << 31) || n_gt < 0 || n_gt >= (1LL << 31) || num_classes < 1 ||
      num_classes > kMaxClasses || n_ranges < 1 || n_ranges > kMaxRanges)
    return -1;
  return layout(n_det, n_gt, num_classes, n_ranges).total;
}

#define VID_WS_CHECK(n_det, n_gt, C, R, bytes)                                                                         \
  do {                                                                                                                 \
    const long long _need = mega_vid_eval_workspace_bytes(n_det, n_gt, C, R);                                         \
    MEGA_ARG_CHECK(_need >= 0, "vid_eval: n_det %lld / n_gt %lld / num_classes %d / n_ranges %d out of range "        \
                   "(< 2^31 boxes, 1..%d classes, 1..%d ranges)", (long long)(n_det), (long long)(n_gt), C, R,        \
                   kMaxClasses, kMaxRanges);                                                                           \
    MEGA_ARG_CHECK(workspace != nullptr && (bytes) >= _need, "vid_eval: workspace of %lld bytes, %lld needed",         \
                   (long long)(bytes), _need);                                                                         \
  } while (0)

extern "C" int mega_vid_eval_match(const float* det_boxes, const float* det_scores, const int* det_labels,
                                   const long long* det_offsets, const float* gt_boxes, const int* gt_labels,
                                   const double* gt_motion, const long long* gt_offsets, int n_img, long long n_det,
                                   long long n_gt, int num_classes, int n_ranges, const double* ranges_host,
                                   const double* empty_weight_host, float iou_thresh, void* workspace,
                                   long long workspace_bytes, signed char* match_out, double* ignore_out,
                                   long long* n_pos_out, int* seen_out, int* det_count_out, void* stream_v) {
  VID_WS_CHECK(n_det, n_gt, num_classes, n_ranges, workspace_bytes);
  MEGA_ARG_CHECK(n_img >= 0 && ranges_host && empty_weight_host && det_offsets && gt_offsets && n_pos_out && seen_out &&
                 det_count_out, "vid_eval_match: null argument");
  cudaStream_t stream = static_cast<cudaStream_t>(stream_v);
  MEGA_CUDA_CHECK(cudaMemsetAsync(n_pos_out, 0, sizeof(long long) * n_ranges * num_classes, stream));
  MEGA_CUDA_CHECK(cudaMemsetAsync(seen_out, 0, sizeof(int) * num_classes, stream));
  MEGA_CUDA_CHECK(cudaMemsetAsync(det_count_out, 0, sizeof(int) * num_classes, stream));
  if (n_img == 0) return MEGA_OK;
  const Layout L = layout(n_det, n_gt, num_classes, n_ranges);
  char* ws = static_cast<char*>(workspace);
  MatchParams p;
  p.det_boxes = det_boxes, p.det_scores = det_scores, p.det_labels = det_labels, p.det_off = det_offsets;
  p.gt_boxes = gt_boxes, p.gt_labels = gt_labels, p.gt_motion = gt_motion, p.gt_off = gt_offsets;
  p.num_classes = num_classes, p.n_det = n_det;
  for (int r = 0; r < kMaxRanges; ++r) {
    p.lo[r] = r < n_ranges ? ranges_host[2 * r] : 0.0;
    p.hi[r] = r < n_ranges ? ranges_host[2 * r + 1] : 0.0;
    p.empty[r] = r < n_ranges ? empty_weight_host[r] : 0.0;
  }
  p.iou_thresh = iou_thresh;
  p.match = match_out, p.ignore = ignore_out;
  p.n_pos = reinterpret_cast<unsigned long long*>(n_pos_out), p.seen = seen_out, p.det_count = det_count_out;
  p.keys = reinterpret_cast<uint64_t*>(ws + L.keys0), p.vals = reinterpret_cast<int*>(ws + L.vals0);
  p.ws_dsort = reinterpret_cast<int*>(ws + L.dsort), p.ws_dorder = reinterpret_cast<int*>(ws + L.dorder);
  p.ws_gsort = reinterpret_cast<int*>(ws + L.gsort), p.ws_gsel = reinterpret_cast<unsigned char*>(ws + L.gsel);
  switch (n_ranges) {
    case 1: vid_match_kernel<1><<<n_img, kMatchThreads, 0, stream>>>(p); break;
    case 2: vid_match_kernel<2><<<n_img, kMatchThreads, 0, stream>>>(p); break;
    case 3: vid_match_kernel<3><<<n_img, kMatchThreads, 0, stream>>>(p); break;
    default: vid_match_kernel<4><<<n_img, kMatchThreads, 0, stream>>>(p); break;
  }
  MEGA_CUDA_CHECK(cudaGetLastError());
  return MEGA_OK;
}

extern "C" int mega_vid_eval_rank(long long n_det, long long n_gt, int num_classes, int n_ranges, void* workspace,
                                  long long workspace_bytes, int* order_out, void* stream_v) {
  VID_WS_CHECK(n_det, n_gt, num_classes, n_ranges, workspace_bytes);
  if (n_det == 0) return MEGA_OK;
  MEGA_ARG_CHECK(order_out != nullptr, "vid_eval_rank: null order_out");
  cudaStream_t stream = static_cast<cudaStream_t>(stream_v);
  const Layout L = layout(n_det, n_gt, num_classes, n_ranges);
  char* ws = static_cast<char*>(workspace);
  uint64_t* keys[2] = {reinterpret_cast<uint64_t*>(ws + L.keys0), reinterpret_cast<uint64_t*>(ws + L.keys1)};
  int* vals[2] = {reinterpret_cast<int*>(ws + L.vals0), reinterpret_cast<int*>(ws + L.vals1)};
  int* counts = reinterpret_cast<int*>(ws + L.counts);
  const int end_bit = 32 + class_bits(num_classes);
  const int n_passes = (end_bit + 7) / 8;
  const unsigned grid = static_cast<unsigned>(L.radix_blocks);
  for (int pass = 0; pass < n_passes; ++pass) {
    const int src = pass & 1, dst = src ^ 1;
    int* vals_dst = pass == n_passes - 1 ? order_out : vals[dst];
    radix_count_kernel<<<grid, kRadixThreads, 0, stream>>>(keys[src], n_det, 8 * pass, counts, L.radix_blocks);
    radix_scan_kernel<<<1, 1024, 0, stream>>>(counts, 256 * L.radix_blocks);
    radix_scatter_kernel<<<grid, kRadixThreads, 0, stream>>>(keys[src], vals[src], n_det, 8 * pass, counts,
                                                             L.radix_blocks, keys[dst], vals_dst);
  }
  MEGA_CUDA_CHECK(cudaGetLastError());
  return MEGA_OK;
}

extern "C" int mega_vid_eval_scan_ap(const signed char* match, const double* ignore, const int* order,
                                     const int* det_count, const long long* n_pos, long long n_det, long long n_gt,
                                     int num_classes, int n_ranges, void* workspace, long long workspace_bytes,
                                     double* prec_out, double* rec_out, double* ap_out, void* stream_v) {
  VID_WS_CHECK(n_det, n_gt, num_classes, n_ranges, workspace_bytes);
  MEGA_ARG_CHECK(det_count && n_pos && ap_out, "vid_eval_scan_ap: null argument");
  cudaStream_t stream = static_cast<cudaStream_t>(stream_v);
  const Layout L = layout(n_det, n_gt, num_classes, n_ranges);
  char* ws = static_cast<char*>(workspace);
  ScanParams p;
  p.match = match, p.ignore = ignore, p.order = order, p.det_count = det_count;
  p.n_pos = reinterpret_cast<const unsigned long long*>(n_pos);
  p.n_det = n_det, p.num_classes = num_classes;
  p.tile_tp = reinterpret_cast<int*>(ws + L.tile_tp), p.tile_fp = reinterpret_cast<double*>(ws + L.tile_fp);
  p.tiles_per_range = L.tiles_per_range;
  p.prec_out = prec_out, p.rec_out = rec_out, p.ap_out = ap_out;
  vid_scan_ap_kernel<<<dim3(num_classes, n_ranges), kScanThreads, 0, stream>>>(p);
  MEGA_CUDA_CHECK(cudaGetLastError());
  return MEGA_OK;
}

// Per-segment body of the device-side VID evaluator (csrc/vid_eval.cu): the detections of one (image, class) pair, sorted
// by score, matched greedily against that class's ground truth of the image, once per motion range.
//
// The body is plain `__host__ __device__` code parametrised by a lane policy. On the device one warp runs it (WarpLanes:
// 32 lanes, shuffles); tests/native/vid_eval_host.cpp compiles the same code with g++ -ffp-contract=off under
// HostLanes, which runs the loops with one lane but evaluates every GT argmax as the 32-lane strided fold plus the
// xor-butterfly the warp performs, so the CPU test-suite checks the reduction tree the device uses.
//
// Semantics are those of mega_vid_match_host (csrc/vid_eval.cu), i.e. the reference's vid_eval.py:201-262:
//   - IoU in float32 on "+1" boxes in boxlist_iou order (structures/boxlist_ops.py:75-88), every operation rounded on
//     its own (no fused multiply-add), so the device IoU has the host's bits;
//   - a GT is a candidate for detection j when it is not yet selected and IoU >= iou_thresh; among candidates the
//     largest IoU wins, and among tied maxima the first non-ignored GT (lowest index), or the last ignored one (highest
//     index) when all of them are ignored -- the fixed point of the host loop's "replace the winner on a tie only while
//     the winner is ignored". That is a total order, so any reduction tree returns the host's winner;
//   - an unmatched detection weighs 0 if its best non-ignored IoU beats its best ignored IoU, 1 in the opposite case,
//     n_ignored / n_gt on a tie, and empty_weight when the class has no GT in the image.
// Detection order: descending score, and among equal scores the LATER detection (higher index in the image) first --
// the order of numpy's `argsort(kind="stable")[::-1]`. Boxes must satisfy x2 > x1 - 2 and y2 > y1 - 2 (positive "+1"
// areas, as every detector output and annotation does), which keeps every IoU finite.
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define MEGA_VE_HD __host__ __device__ __forceinline__
#else
#define MEGA_VE_HD static inline
#endif

namespace mega_vid {

constexpr int kMaxRanges = 4;

// every float operation rounded separately on both sides (nvcc would contract a*b+c into an FMA)
MEGA_VE_HD float fadd(float a, float b) {
#if defined(__CUDA_ARCH__)
  return __fadd_rn(a, b);
#else
  return a + b;
#endif
}
MEGA_VE_HD float fsub(float a, float b) {
#if defined(__CUDA_ARCH__)
  return __fsub_rn(a, b);
#else
  return a - b;
#endif
}
MEGA_VE_HD float fmul(float a, float b) {
#if defined(__CUDA_ARCH__)
  return __fmul_rn(a, b);
#else
  return a * b;
#endif
}
MEGA_VE_HD float fdiv(float a, float b) {
#if defined(__CUDA_ARCH__)
  return __fdiv_rn(a, b);
#else
  return a / b;
#endif
}

// order-preserving uint32 image of a float score (-0 folded onto +0, so equal scores give equal keys)
MEGA_VE_HD uint32_t score_key(float s) {
  union { float f; uint32_t u; } c;
  c.f = s;
  uint32_t u = c.u == 0x80000000u ? 0u : c.u;
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

// "+1" box of mega_vid_match_host: x2, y2 shifted by one, area (x2 - x1 + 1) * (y2 - y1 + 1)
struct Box1 {
  float x1, y1, x2, y2, area;
};
MEGA_VE_HD Box1 box1(const float* b) {
  Box1 r;
  r.x1 = b[0], r.y1 = b[1];
  r.x2 = fadd(b[2], 1.0f), r.y2 = fadd(b[3], 1.0f);
  r.area = fmul(fadd(fsub(r.x2, r.x1), 1.0f), fadd(fsub(r.y2, r.y1), 1.0f));
  return r;
}
MEGA_VE_HD float iou1(const Box1& p, const Box1& g) {
  const float ltx = p.x1 > g.x1 ? p.x1 : g.x1, lty = p.y1 > g.y1 ? p.y1 : g.y1;
  const float rbx = p.x2 < g.x2 ? p.x2 : g.x2, rby = p.y2 < g.y2 ? p.y2 : g.y2;
  float w = fadd(fsub(rbx, ltx), 1.0f), h = fadd(fsub(rby, lty), 1.0f);
  w = w < 0.f ? 0.f : w, h = h < 0.f ? 0.f : h;
  const float inter = fmul(w, h);
  return fdiv(inter, fsub(fadd(p.area, g.area), inter));
}

// Best GT of one detection for one range: the winning candidate (k >= 0) and the largest IoUs over ignored / non-ignored
// GT (selected ones included, as in the host loop). k is the GT's index in the image (the tie rule's order), pos its
// place in the segment's GT list (where its "selected" flag lives).
struct Best {
  float v;      // IoU of the winner
  int k, pos;   // -1: no candidate
  int ign;      // winner is ignored
  float ig, nig;
};
MEGA_VE_HD Best best_identity() {
  Best b;
  b.v = 0.f, b.k = -1, b.pos = -1, b.ign = 0, b.ig = -1.f, b.nig = -1.f;
  return b;
}
// true when candidate (v, k, ign) beats the current winner of b
MEGA_VE_HD bool beats(float v, int k, int ign, const Best& b) {
  if (b.k < 0) return true;
  if (v != b.v) return v > b.v;
  if (ign != b.ign) return !ign;            // on a tie a non-ignored GT beats an ignored one
  return ign ? k > b.k : k < b.k;           // first non-ignored, last ignored
}
MEGA_VE_HD Best combine(Best a, const Best& b) {
  if (b.k >= 0 && beats(b.v, b.k, b.ign, a)) a.v = b.v, a.k = b.k, a.pos = b.pos, a.ign = b.ign;
  a.ig = b.ig > a.ig ? b.ig : a.ig;
  a.nig = b.nig > a.nig ? b.nig : a.nig;
  return a;
}

MEGA_VE_HD int gt_ignored(const double* motion, int k, double lo, double hi) {
  if (!motion) return 0;
  const double m = motion[k];                // NaN (no motion IoU for this GT): never ignored, like the host's zeros
  return (m < lo) || (m > hi);
}

// One segment. det_box [*,4] / det_score index the image's detections, det_idx[0..n_det) lists the segment's ones (any
// order); gt_box [*,4] / gt_motion (NULL: nothing ignored) index the image's GT, gt_idx[0..n_gt) the segment's ones (any
// order). R ranges [range_lo[r], range_hi[r]]; order[n_det] and selected[n_gt * R] are scratch. Output for detection d = det_idx[j] and range r:
// match_out[r * out_stride + d], ignore_out[r * out_stride + d].
template <int R, class Lanes>
MEGA_VE_HD void match_segment(const Lanes& L, const float* det_box, const float* det_score, const int* det_idx, int n_det,
                              const float* gt_box, const double* gt_motion, const int* gt_idx, int n_gt,
                              const double* range_lo, const double* range_hi, const double* empty_weight,
                              float iou_thresh, int* order, unsigned char* selected, signed char* match_out,
                              double* ignore_out, long long out_stride) {
  const int lane = L.lane(), width = L.width();
  if (n_det == 0) return;
  if (n_gt == 0) {
    for (int j = lane; j < n_det; j += width)
      for (int r = 0; r < R; ++r)
        match_out[r * out_stride + det_idx[j]] = 0, ignore_out[r * out_stride + det_idx[j]] = empty_weight[r];
    return;
  }
  // rank by (score desc, index desc): O(n^2) compares, n is a per-image class count
  for (int j = lane; j < n_det; j += width) {
    const int dj = det_idx[j];
    const uint64_t kj = (static_cast<uint64_t>(score_key(det_score[dj])) << 32) | static_cast<uint32_t>(dj);
    int rank = 0;
    for (int i = 0; i < n_det; ++i) {
      const int di = det_idx[i];
      const uint64_t ki = (static_cast<uint64_t>(score_key(det_score[di])) << 32) | static_cast<uint32_t>(di);
      rank += ki > kj;
    }
    order[rank] = dj;
  }
  int n_ignored[R];
  for (int r = 0; r < R; ++r) {
    n_ignored[r] = 0;
    for (int p = 0; p < n_gt; ++p) n_ignored[r] += gt_ignored(gt_motion, gt_idx[p], range_lo[r], range_hi[r]);
  }
  for (int p = lane; p < n_gt; p += width)
    for (int r = 0; r < R; ++r) selected[r * n_gt + p] = 0;
  L.sync();
  for (int t = 0; t < n_det; ++t) {
    const int d = order[t];
    const Box1 pb = box1(det_box + 4 * d);
    Best best[R];
    for (int r = 0; r < R; ++r) best[r] = best_identity();
    L.template fold<R>(n_gt, best, [&](int p, Best* acc) {
      const int k = gt_idx[p];
      const float v = iou1(pb, box1(gt_box + 4 * k));
      for (int r = 0; r < R; ++r) {
        const int ig = gt_ignored(gt_motion, k, range_lo[r], range_hi[r]);
        if (ig && v > acc[r].ig) acc[r].ig = v;
        if (!ig && v > acc[r].nig) acc[r].nig = v;
        if (!selected[r * n_gt + p] && v >= iou_thresh && beats(v, k, ig, acc[r]))
          acc[r].v = v, acc[r].k = k, acc[r].pos = p, acc[r].ign = ig;
      }
    });
    for (int r = 0; r < R; ++r) {
      const Best& b = best[r];
      signed char m;
      double w;
      if (b.k >= 0) {
        m = 1, w = b.ign ? 1.0 : 0.0;
        if (b.pos % width == lane) selected[r * n_gt + b.pos] = 1;   // only the owning lane ever reads this flag
      } else {
        m = 0;
        w = b.nig > b.ig ? 0.0 : b.ig > b.nig ? 1.0 : static_cast<double>(n_ignored[r]) / static_cast<double>(n_gt);
      }
      if (t % width == lane) match_out[r * out_stride + d] = m, ignore_out[r * out_stride + d] = w;
    }
  }
}

// Host lane policy: one lane runs the loops; fold() reproduces the warp's lane-strided partials and xor-butterfly.
struct HostLanes {
  int lane() const { return 0; }
  int width() const { return 1; }
  void sync() const {}
  template <int R, class F>
  void fold(int n, Best* out, F&& f) const {
    Best part[32][R];
    for (int l = 0; l < 32; ++l) {
      for (int r = 0; r < R; ++r) part[l][r] = best_identity();
      for (int p = l; p < n; p += 32) f(p, part[l]);
    }
    for (int off = 16; off > 0; off >>= 1) {
      Best next[32][R];
      for (int l = 0; l < 32; ++l)
        for (int r = 0; r < R; ++r) next[l][r] = combine(part[l][r], part[l ^ off][r]);
      for (int l = 0; l < 32; ++l)
        for (int r = 0; r < R; ++r) part[l][r] = next[l][r];
    }
    for (int r = 0; r < R; ++r) out[r] = part[0][r];
  }
};

}  // namespace mega_vid

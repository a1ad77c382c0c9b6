// Host build of the segment body of csrc/vid_eval.cuh -- TEST INFRASTRUCTURE ONLY.
// g++ -ffp-contract=off compiles the very function one warp of vid_match_kernel runs per (image, class) segment, under
// the HostLanes policy (one lane for the loops; every GT argmax as the warp's 32 lane-strided folds and xor-butterfly),
// so the CPU test-suite can compare it with mega_vid_match_host without a GPU.
// Build: g++ -O2 -ffp-contract=off -fPIC -shared -std=c++17 -I mega.pytorch_b200/csrc -o libvid_eval_host.so vid_eval_host.cpp
#include "vid_eval.cuh"

using namespace mega_vid;

template <int R>
static void run(const float* det_box, const float* det_score, const int* det_idx, int n_det, const float* gt_box,
                const double* gt_motion, const int* gt_idx, int n_gt, const double* ranges, const double* empty,
                float thr, int* order, unsigned char* selected, signed char* match_out, double* ignore_out) {
  double lo[R], hi[R];
  for (int r = 0; r < R; ++r) lo[r] = ranges[2 * r], hi[r] = ranges[2 * r + 1];
  match_segment<R>(HostLanes(), det_box, det_score, det_idx, n_det, gt_box, gt_motion, gt_idx, n_gt, lo, hi, empty, thr,
                   order, selected, match_out, ignore_out, n_det);
}

extern "C" {

// One segment: det_idx / gt_idx list the segment's detections / GT in any order (indices into the box arrays);
// match_out / ignore_out [n_ranges][n_det] by detection index. order [n_det], selected [n_gt * n_ranges]: scratch.
int vid_match_segment_host(const float* det_box, const float* det_score, const int* det_idx, int n_det,
                           const float* gt_box, const double* gt_motion, const int* gt_idx, int n_gt, int n_ranges,
                           const double* ranges, const double* empty, float thr, int* order, unsigned char* selected,
                           signed char* match_out, double* ignore_out) {
  switch (n_ranges) {
    case 1: run<1>(det_box, det_score, det_idx, n_det, gt_box, gt_motion, gt_idx, n_gt, ranges, empty, thr, order, selected, match_out, ignore_out); return 0;
    case 2: run<2>(det_box, det_score, det_idx, n_det, gt_box, gt_motion, gt_idx, n_gt, ranges, empty, thr, order, selected, match_out, ignore_out); return 0;
    case 3: run<3>(det_box, det_score, det_idx, n_det, gt_box, gt_motion, gt_idx, n_gt, ranges, empty, thr, order, selected, match_out, ignore_out); return 0;
    case 4: run<4>(det_box, det_score, det_idx, n_det, gt_box, gt_motion, gt_idx, n_gt, ranges, empty, thr, order, selected, match_out, ignore_out); return 0;
  }
  return 1;
}

unsigned int vid_score_key_host(float s) { return score_key(s); }

}  // extern "C"

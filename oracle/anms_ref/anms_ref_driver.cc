// extern "C" entry into the reference's anms::RangeTree (dynosam/src/frontend/anms/anms.cc), compiled from the reference
// checkout into oracle/_ref/libanms_ref.so by oracle/anms_ref/Makefile.  Parity infrastructure only.
#include <cstdint>
#include <vector>

#include <opencv2/opencv.hpp>

#include "dynosam/frontend/anms/anms/anms.h"

extern "C" {
// xy[n][2] in the order RangeTree walks them (the caller applies the cv::sortIdx ranking first); writes the positions
// (into xy) of the returned key-points, in the returned order, to out[] and returns their number.
int anms_ref_range_tree(const float* xy, int n, int num_ret_points, float tolerance, int cols, int rows, int* out) {
  std::vector<cv::KeyPoint> kps((size_t)n);
  for (int i = 0; i < n; i++) { kps[i].pt = cv::Point2f(xy[2*i], xy[2*i + 1]); kps[i].class_id = i; }
  const std::vector<cv::KeyPoint> sel = anms::RangeTree(kps, num_ret_points, tolerance, cols, rows);
  for (size_t i = 0; i < sel.size(); i++) out[i] = sel[i].class_id;
  return (int)sel.size();
}
}

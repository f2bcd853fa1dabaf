// Minimal stand-in for <opencv2/opencv.hpp>: just what anms.cc names, so the reference's ANMS can be compiled into the
// parity library (oracle/anms_ref/Makefile) without OpenCV.  The drawing / window functions are no-ops.
#pragma once
#include <cfloat>
#include <cmath>
#include <cstring>
#include <string>
#include <vector>

namespace cv {
struct Point2f {
  float x = 0.f, y = 0.f;
  Point2f() = default;
  Point2f(float x_, float y_) : x(x_), y(y_) {}
};
struct KeyPoint {
  Point2f pt;
  float size = 0.f, angle = -1.f, response = 0.f;
  int octave = 0, class_id = -1;
};
struct Mat {};
struct Scalar {
  Scalar(double, double, double, double) {}
};
enum { WINDOW_AUTOSIZE = 1 };
inline void drawKeypoints(const Mat&, const std::vector<KeyPoint>&, Mat&, const Scalar&) {}
inline void namedWindow(const std::string&, int) {}
inline void imshow(const std::string&, const Mat&) {}
inline int waitKey(int = 0) { return -1; }
}  // namespace cv

// ORBextractor.h -- drop-in ORB_SLAM2::ORBextractor on top of libswm_orb.so (include/swm_orb.h).
//
// Same class name, constructor, operator() signature, getters and public flags as the reference
// (/root/reference/code/include/ORBextractor.h:48-125), so Frame / KeyFrame / Tracking compile
// unchanged: replace the reference's src/ORBextractor.cc + src/cuda/*.cu with this header and link
// libswm_orb.so.  Build with -DSWM_HAVE_OPENCV against the real OpenCV, or without it against
// cv_shim.h (tests).  Error behaviour mirrors the reference: CUDA / setup failures are fatal
// (checkCudaErrors -> exit, Fast_gpu.cu:346-352) -- here a std::runtime_error carrying
// swm_last_error(); an empty image returns silently (ORBextractor.cc:750-751).
#pragma once
#include <cstring>
#include <stdexcept>
#include <string>
#include <vector>

#ifdef SWM_HAVE_OPENCV
#include <opencv2/core.hpp>
#include <opencv2/core/cuda.hpp>
#else
#include "cv_shim.h"
#endif
#include "../../include/swm_orb.h"

namespace ORB_SLAM2 {

// What the public mvImagePyramid / mvImagePyramidBorder vectors hold (device memory).  With OpenCV they are
// cv::cuda::GpuMat HEADERS over the extractor's planes (no allocation, no copy), the reference's own member type
// (include/ORBextractor.h:90-92), so Frame::ComputeStereoMatches' uses compile (Frame.cc:521,611-630; note that it
// dereferences them on the host, which the reference can only do because its allocator hands out managed memory).
// Without OpenCV (tests) a plain view with the same field names stands in.
struct PyramidLevelView {
  const unsigned char* data = nullptr;  // device pointer to ROI pixel (0,0)
  int cols = 0, rows = 0;
  size_t step = 0;
};
#ifdef SWM_HAVE_OPENCV
typedef cv::cuda::GpuMat PyramidLevel;
#else
typedef PyramidLevelView PyramidLevel;
#endif

class ORBextractor {
 public:
  enum { HARRIS_SCORE = 0, FAST_SCORE = 1 };

  ORBextractor(int nfeatures, float scaleFactor, int nlevels, int iniThFAST, int minThFAST, int device = 0)
      : mvImagePyramidAllocatedFlag(false), nlevels_(nlevels), scaleFactor_(scaleFactor) {
    swm_orb_cfg cfg;
    cfg.nfeatures = nfeatures;
    cfg.scale_factor = scaleFactor;
    cfg.nlevels = nlevels;
    cfg.ini_th_fast = iniThFAST;
    cfg.min_th_fast = minThFAST;
    cfg.max_batch = 1;
    cfg.max_fast_per_level = 0;
    if (swm_orb_create(&cfg, device, &h_) != SWM_OK)
      throw std::runtime_error(std::string("ORBextractor: ") + swm_last_error(nullptr));
    mvScaleFactor.resize(nlevels);
    mvInvScaleFactor.resize(nlevels);
    mvLevelSigma2.resize(nlevels);
    mvInvLevelSigma2.resize(nlevels);
    swm_orb_scale_tables(h_, mvScaleFactor.data(), mvInvScaleFactor.data(), mvLevelSigma2.data(),
                         mvInvLevelSigma2.data());
  }
  ~ORBextractor() { swm_orb_destroy(h_); }
  ORBextractor(const ORBextractor&) = delete;
  ORBextractor& operator=(const ORBextractor&) = delete;

  // Compute the ORB features and descriptors on an image.  Mask is ignored, as in the reference.
  void operator()(cv::InputArray _image, cv::InputArray /*_mask*/, std::vector<cv::KeyPoint>& _keypoints,
                  cv::OutputArray _descriptors) {
#ifdef SWM_HAVE_OPENCV
    if (_image.empty()) return;
    cv::Mat image = _image.getMat();
    CV_Assert(image.type() == CV_8UC1);
#else
    const cv::Mat& image = _image;
    if (image.empty()) return;
#endif
    const int cap = swm_orb_max_keypoints(h_);
    kp_buf_.resize(cap);
    desc_buf_.resize((size_t)cap * 32);
    int n = 0;
    const int rc = swm_orb_extract(h_, image.data, image.cols, image.rows, (int)image.step,
                                   reinterpret_cast<swm_keypoint*>(kp_buf_.data()), desc_buf_.data(), cap, &n);
    if (rc != SWM_OK) throw std::runtime_error(std::string("ORBextractor: ") + swm_last_error(h_));
    _keypoints.assign(kp_buf_.begin(), kp_buf_.begin() + n);
    if (n == 0) {
      _descriptors.release();
    } else {
      _descriptors.create(n, 32, CV_8U);
#ifdef SWM_HAVE_OPENCV
      cv::Mat d = _descriptors.getMat();
#else
      cv::Mat& d = _descriptors;
#endif
      for (int i = 0; i < n; i++) std::memcpy(d.ptr(i), desc_buf_.data() + (size_t)i * 32, 32);
    }
    refresh_pyramid_views();
  }

  int inline GetLevels() { return nlevels_; }
  float inline GetScaleFactor() { return scaleFactor_; }
  std::vector<float> inline GetScaleFactors() { return mvScaleFactor; }
  std::vector<float> inline GetInverseScaleFactors() { return mvInvScaleFactor; }
  std::vector<float> inline GetScaleSigmaSquares() { return mvLevelSigma2; }
  std::vector<float> inline GetInverseScaleSigmaSquares() { return mvInvLevelSigma2; }

  // Public pyramid members of the reference (ORBextractor.h:90-92).  mvImagePyramid[l] is the level
  // ROI after the call (blurred, like the reference's in-place filter); mvImagePyramidBorder[l] the
  // un-blurred plane whose 19-px reflect-101 border lies at negative offsets of `data`.
  bool mvImagePyramidAllocatedFlag;
  std::vector<PyramidLevel> mvImagePyramid;
  std::vector<PyramidLevel> mvImagePyramidBorder;

  swm_orb* handle() { return h_; }

  // Frame::ComputeStereoMatches (reference Frame.cc:516-690) on the device, from the frames THIS extractor (the left
  // view, Frame::mpORBextractorLeft) and `right` (mpORBextractorRight) extracted last: fills mvuRight / mvDepth for the
  // N keypoints of the left view, bit-identical to the reference's loop (INTEGRATION.md shows the three-line body that
  // replaces the member in Frame.cc).
  void ComputeStereoMatches(ORBextractor& right, float mbf, float mb, int N, std::vector<float>& mvuRight,
                            std::vector<float>& mvDepth) {
    const int cap = swm_orb_max_keypoints(h_);
    stereo_u_.resize(cap);
    stereo_z_.resize(cap);
    if (swm_orb_stereo_match(h_, right.h_, mbf, mb, stereo_u_.data(), stereo_z_.data(), cap, 1) != SWM_OK)
      throw std::runtime_error(std::string("ORBextractor::ComputeStereoMatches: ") + swm_last_error(h_));
    if (N > cap) N = cap;
    mvuRight.assign(stereo_u_.begin(), stereo_u_.begin() + N);
    mvDepth.assign(stereo_z_.begin(), stereo_z_.begin() + N);
  }

 protected:
  void refresh_pyramid_views() {
    mvImagePyramid.resize(nlevels_);
    mvImagePyramidBorder.resize(nlevels_);
    for (int l = 0; l < nlevels_; l++) {
      for (int which = 0; which < 2; which++) {
        const unsigned char* dev = nullptr;
        int w = 0, h = 0, pitch = 0;
        if (swm_orb_level_ptr(h_, 0, l, which, &dev, &w, &h, &pitch) != SWM_OK) return;
#ifdef SWM_HAVE_OPENCV
        // Border: the whole (h + 38) x (w + 38) un-blurred buffer, as ComputePyramid allocates it (ORBextractor.cc:827);
        // Pyramid: the level ROI of the blurred plane (the reference blurs its ROI view in place, :719)
        unsigned char* p = const_cast<unsigned char*>(dev);
        if (which) mvImagePyramid[l] = cv::cuda::GpuMat(h, w, CV_8UC1, p, (size_t)pitch);
        else mvImagePyramidBorder[l] = cv::cuda::GpuMat(h + 38, w + 38, CV_8UC1, p - 19 * (size_t)pitch - 19, (size_t)pitch);
#else
        PyramidLevelView& v = which ? mvImagePyramid[l] : mvImagePyramidBorder[l];
        v.data = dev; v.cols = w; v.rows = h; v.step = (size_t)pitch;
#endif
      }
    }
    mvImagePyramidAllocatedFlag = true;
  }

  swm_orb* h_ = nullptr;
  int nlevels_;
  float scaleFactor_;
  std::vector<float> mvScaleFactor, mvInvScaleFactor, mvLevelSigma2, mvInvLevelSigma2;
  std::vector<cv::KeyPoint> kp_buf_;
  std::vector<unsigned char> desc_buf_;
  std::vector<float> stereo_u_, stereo_z_;
};

}  // namespace ORB_SLAM2

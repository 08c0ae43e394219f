// feature_matcher.hpp -- drop-in for the reference's src/feature_matcher.hpp:26-51: same class, same public members.
//
//   match_two_image   the hot path (src/feature_matcher.cpp:42-59: knnMatch k = 2 + ratio test) -> erp_knn2_match on
//                     the B200: exact brute-force 2-NN instead of the approximate FLANN KD-tree (SURVEY D1)
//   detect_key_point, comput_descriptor, draw_match, do_all
//                     SURF and drawing are not on the accelerated path: they forward to OpenCV (xfeatures2d) when the
//                     build has it, and raise cv::Exception (CV_Error) with the type shim of this image
//
// Objects are default-constructible and cheap (the reference builds one per call, src/spherical_surf.cpp:96): the CUDA
// context lives in a per-thread cache (erp_host_context.hpp), not in the object.
#pragma once

// the transitive includes the reference's callers rely on (src/feature_matcher.hpp:3-24)
#define _USE_MATH_DEFINES
#include <cmath>
#include <vector>

#include "debug_print.h"
#include "opencv2/opencv_modules.hpp"
#include "opencv2/calib3d.hpp"
#include "opencv2/core/ocl.hpp"
#include "opencv2/features2d.hpp"
#include "opencv2/highgui.hpp"
#include "opencv2/imgcodecs.hpp"
#include "opencv2/imgproc.hpp"
#include "opencv2/xfeatures2d.hpp"

class feature_matcher
{
public:
    feature_matcher() { init(); }
    ~feature_matcher() { deinit(); }

    // (re)creates the SURF detector / extractor; no CUDA work
    void init();
    void deinit();

    std::vector<cv::KeyPoint> detect_key_point(const cv::Mat &image);

    cv::Mat comput_descriptor(const cv::Mat &image,
                              std::vector<cv::KeyPoint> &key_point);

    // CV_32F descriptors, one per row (64 or 128 wide; any multiple of 4 works).  Returns DMatch{queryIdx, trainIdx,
    // imgIdx = 0, distance = L2} in ascending queryIdx for the rows that pass d0 < ratio_thresh * d1.
    // With norm_type == cv::NORM_HAMMING: CV_8U rows of 1..64 bytes, distance = Hamming.
    std::vector<cv::DMatch> match_two_image(const cv::Mat &descriptor1,
                                            const cv::Mat &descriptor2);

    // overlap picture: left / right view in two colour channels, one coloured segment per pair key_left[i] -> key_right[i]
    cv::Mat draw_match(const cv::Mat& im_left,
                       const cv::Mat& im_right,
                       const std::vector<cv::KeyPoint>& key_left,
                       const std::vector<cv::KeyPoint>& key_right);

    // detect + describe + match + gather of the matched keypoints (src/feature_matcher.cpp:85-125)
    void do_all(const cv::Mat &im_left,
                const cv::Mat &im_right,
                std::vector<cv::KeyPoint>& left_key,
                std::vector<cv::KeyPoint>& right_key,
                int& match_size,
                cv::Mat& match_output,
                int& total_key_num);

    // --- extensions (SURVEY D5) -----------------------------------------------------------------------------------
    float ratio_thresh = 0.3f;               // Lowe ratio; the reference hard-codes 0.3f
    bool cross_check = false;                // keep a match only if it is also the train row's nearest query
    // cv::NORM_HAMMING: match_two_image takes CV_8U binary descriptors (ORB, AKAZE, BRISK, ...) and matches them by
    // Hamming distance (erp_knn2_match_bin); the default keeps the CV_32F / L2 behaviour
    int norm_type = cv::NORM_L2;
    // SURF-128: re-creates the detector / extractor with extended descriptors (SURF::create(100, 4, 3, true))
    void set_extended(bool extended_descriptors);
    bool extended() const { return extended_; }

private:
#ifndef ERP_OPENCV_COMPAT
    cv::Ptr<cv::Feature2D> surf_detect_;
    cv::Ptr<cv::Feature2D> surf_describe_;
#endif
    bool extended_ = false;
};

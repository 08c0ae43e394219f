// feature_matcher.cpp -- host side of the matching boundary.
#include "feature_matcher.hpp"

#include "erp_host_context.hpp"

using namespace std;
using namespace cv;

void feature_matcher::init()
{
#ifndef ERP_OPENCV_COMPAT
    // SURF with OpenCV's defaults, as src/feature_matcher.cpp:13-15 (extended = false: 64-D);
    // extended_ = true is the 128-D variant (same defaults otherwise: hessianThreshold 100, 4 octaves, 3 layers)
    surf_detect_ = xfeatures2d::SURF::create(100, 4, 3, extended_);
    surf_describe_ = xfeatures2d::SURF::create(100, 4, 3, extended_);
#endif
    // no matcher object: the CUDA context is per thread and created on first use
}

void feature_matcher::deinit() {}

void feature_matcher::set_extended(bool extended_descriptors)
{
    if (extended_descriptors == extended_) return;
    extended_ = extended_descriptors;
    init();
}

vector<KeyPoint> feature_matcher::detect_key_point(const Mat &image)
{
#ifndef ERP_OPENCV_COMPAT
    vector<KeyPoint> key_point;
    surf_detect_->detect(image, key_point);
    return key_point;
#else
    (void)image;
    CV_Error(cv::Error::StsNotImplemented, "feature_matcher::detect_key_point needs OpenCV xfeatures2d (SURF); this build uses the type shim");
#endif
}

Mat feature_matcher::comput_descriptor(const Mat &image, vector<KeyPoint> &key_point)
{
#ifndef ERP_OPENCV_COMPAT
    Mat d;
    surf_describe_->compute(image, key_point, d);
    return d;
#else
    (void)image; (void)key_point;
    CV_Error(cv::Error::StsNotImplemented, "feature_matcher::comput_descriptor needs OpenCV xfeatures2d (SURF); this build uses the type shim");
#endif
}

// 2-NN under L2 + ratio test, ascending queryIdx (src/feature_matcher.cpp:42-59), exact brute force
// instead of the reference's approximate FLANN trees (SURVEY D1).
vector<DMatch> feature_matcher::match_two_image(const Mat &descriptor1, const Mat &descriptor2)
{
    static_assert(sizeof(DMatch) == sizeof(erp_dmatch), "cv::DMatch and erp_dmatch must share a layout");
    if (norm_type == cv::NORM_HAMMING) {
        // binary descriptors: cv::BFMatcher(NORM_HAMMING) semantics on the kind::i8 / popcount engines
        if (descriptor1.type() != CV_8UC1 || descriptor2.type() != CV_8UC1)
            CV_Error(cv::Error::StsBadArg, "match_two_image: NORM_HAMMING descriptors must be CV_8U single channel");
        if (descriptor1.rows > 0 && descriptor1.cols != descriptor2.cols)
            CV_Error(cv::Error::StsBadArg, "match_two_image: descriptor sizes differ");
        vector<DMatch> good(descriptor1.rows > 0 ? descriptor1.rows : 0);
        int n = 0, st;
        {
            erp_host::Lock lock;
            st = erp_knn2_match_bin(erp_host::context(), descriptor1.ptr<uint8_t>(0), descriptor1.rows, descriptor1.step,
                                    descriptor2.ptr<uint8_t>(0), descriptor2.rows, descriptor2.step, descriptor1.cols,
                                    ratio_thresh, cross_check ? 1 : 0, reinterpret_cast<erp_dmatch*>(good.data()), &n);
        }
        if (st != ERP_OK) CV_Error(cv::Error::StsBadArg, string("match_two_image: ") + erp_last_error());
        good.resize(n);
        return good;
    }
    if (descriptor1.type() != CV_32FC1 || descriptor2.type() != CV_32FC1)
        CV_Error(cv::Error::StsBadArg, "match_two_image: descriptors must be CV_32F single channel");
    if (descriptor1.rows > 0 && descriptor1.cols != descriptor2.cols)
        CV_Error(cv::Error::StsBadArg, "match_two_image: descriptor dimensions differ");
    vector<DMatch> good(descriptor1.rows > 0 ? descriptor1.rows : 0);
    int n = 0;
    static_assert(sizeof(DMatch) == sizeof(erp_dmatch), "cv::DMatch and erp_dmatch must share a layout");
    int st;
    {
        erp_host::Lock lock;
        if (erp_group* grp = erp_host::group())      // $ERP_B200_DEVICES: query rows per GPU, train set all-gathered over NVLink
            st = erp_group_knn2_match(grp, descriptor1.ptr<float>(0), descriptor1.rows, descriptor1.step,
                                      descriptor2.ptr<float>(0), descriptor2.rows, descriptor2.step,
                                      descriptor1.cols, ratio_thresh, cross_check ? 1 : 0,
                                      reinterpret_cast<erp_dmatch*>(good.data()), &n);
        else
            st = erp_knn2_match(erp_host::context(),
                                descriptor1.ptr<float>(0), descriptor1.rows, descriptor1.step,
                                descriptor2.ptr<float>(0), descriptor2.rows, descriptor2.step,
                                descriptor1.cols, ratio_thresh, cross_check ? 1 : 0,
                                reinterpret_cast<erp_dmatch*>(good.data()), &n);
    }
    // the reference throws cv::Exception out of knnMatch on malformed input (e.g. < 2 train rows)
    if (st != ERP_OK) CV_Error(cv::Error::StsBadArg, string("match_two_image: ") + erp_last_error());
    good.resize(n);
    return good;
}

// The overlap picture of src/feature_matcher.cpp:61-84: left view in one channel, right view in another, and one
// coloured segment per correspondence from its left to its right position (key_left[i] <-> key_right[i]: the callers
// pass the GATHERED keypoints, src/spherical_surf.cpp:173).  Drawing needs OpenCV's imgproc: real builds only.
Mat feature_matcher::draw_match(const Mat& im_left, const Mat& im_right, const vector<KeyPoint>& key_left, const vector<KeyPoint>& key_right)
{
#ifndef ERP_OPENCV_COMPAT
    Mat gray_left, gray_right;
    cvtColor(im_left, gray_left, COLOR_RGB2GRAY);
    cvtColor(im_right, gray_right, COLOR_RGB2GRAY);
    vector<Mat> planes;
    planes.push_back(gray_left);
    planes.push_back(gray_right);
    planes.push_back(Mat::zeros(im_left.rows, im_left.cols, CV_8UC1));
    Mat overlap;
    merge(planes, overlap);
    const size_t n = key_left.size() < key_right.size() ? key_left.size() : key_right.size();
    for (size_t i = 0; i < n; i++) {
        // hue ramp over the matches, as the reference colours them
        Mat hsv(1, 1, CV_8UC3, Scalar(i * (180.0 / (double)n), 180, 150)), bgr;
        cvtColor(hsv, bgr, COLOR_HSV2BGR);
        line(overlap, key_left[i].pt, key_right[i].pt, Scalar(bgr.data[0], bgr.data[1], bgr.data[2]), 5);
    }
    return overlap;
#else
    (void)im_left; (void)im_right; (void)key_left; (void)key_right;
    CV_Error(cv::Error::StsNotImplemented, "feature_matcher::draw_match needs OpenCV imgproc; this build uses the type shim");
#endif
}

void feature_matcher::do_all(const Mat &im_left, const Mat &im_right, vector<KeyPoint>& left_key, vector<KeyPoint>& right_key, int& match_size, Mat& match_output, int& total_key_num)
{
    // single-strip pipeline of src/feature_matcher.cpp:88-128: detect, describe, match, gather
    vector<KeyPoint> kl = detect_key_point(im_left), kr = detect_key_point(im_right);
    Mat dl = comput_descriptor(im_left, kl), dr = comput_descriptor(im_right, kr);
    vector<DMatch> m = match_two_image(dl, dr);
    total_key_num = (int)kl.size();
    match_size = (int)m.size();
    left_key.resize(m.size());
    right_key.resize(m.size());
    for (size_t i = 0; i < m.size(); i++) { left_key[i] = kl[m[i].queryIdx]; right_key[i] = kr[m[i].trainIdx]; }
    match_output = draw_match(im_left, im_right, left_key, right_key);
}

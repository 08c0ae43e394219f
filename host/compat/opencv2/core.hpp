// Minimal stand-in for the OpenCV types that appear in the SIGNATURES of the hot-path classes
// (cv::Mat, cv::KeyPoint, cv::DMatch, cv::Point*, cv::Vec*) plus the small-matrix algebra and the declarations the
// reference's own callers (src/automatic.cpp, src/spherical_surf.cpp) need to compile and link against the drop-in
// headers.  Selected only when the build has no real OpenCV (this image: SURVEY section 8c); never mixed with it.
// Layouts follow OpenCV 3.4: KeyPoint 28 bytes, DMatch 16 bytes, Mat row-major with a byte step.  Image codecs are
// NOT part of the shim: imread / imwrite are declared and throw.
#pragma once
#ifndef ERP_OPENCV_COMPAT
#define ERP_OPENCV_COMPAT 1
#endif

#include <chrono>
#include <cmath>
#include <cstddef>
#include <cstdint>
#include <cstring>
#include <memory>
#include <ostream>
#include <stdexcept>
#include <string>
#include <vector>

typedef int64_t int64;

#define CV_8U 0
#define CV_32S 4
#define CV_32F 5
#define CV_64F 6
#define CV_CN_SHIFT 3
#define CV_MAKETYPE(depth, cn) ((depth) + (((cn)-1) << CV_CN_SHIFT))
#define CV_8UC1 CV_MAKETYPE(CV_8U, 1)
#define CV_8UC3 CV_MAKETYPE(CV_8U, 3)
#define CV_32SC2 CV_MAKETYPE(CV_32S, 2)
#define CV_32FC1 CV_MAKETYPE(CV_32F, 1)
#define CV_64FC1 CV_MAKETYPE(CV_64F, 1)

namespace cv {

typedef std::string String;
template <class T> using Ptr = std::shared_ptr<T>;

namespace Error { enum Code { StsError = -2, StsBadArg = -5, StsNotImplemented = -213 }; }

// same five-argument constructor as the real class; thrown through CV_Error like OpenCV code does
class Exception : public std::runtime_error {
public:
    Exception(int code_, const std::string& err_, const std::string& func_, const std::string& file_, int line_)
        : std::runtime_error(err_), code(code_), err(err_), func(func_), file(file_), line(line_) {}
    int code;
    std::string err, func, file;
    int line;
};
#define CV_Error(code, msg) throw cv::Exception((code), (msg), __func__, __FILE__, __LINE__)

template <class T> struct Point_ {
    T x, y;
    Point_() : x(0), y(0) {}
    Point_(T a, T b) : x(a), y(b) {}
};
typedef Point_<int> Point2i;
typedef Point_<float> Point2f;
typedef Point_<double> Point2d;
typedef Point2i Point;

template <class T> struct Point3_ {
    T x, y, z;
    Point3_() : x(0), y(0), z(0) {}
    Point3_(T a, T b, T c) : x(a), y(b), z(c) {}
};
typedef Point3_<float> Point3f;
typedef Point3_<double> Point3d;

template <class T, int N> struct Vec {
    T val[N];
    Vec() { for (int i = 0; i < N; i++) val[i] = T(0); }
    Vec(T a, T b) { static_assert(N == 2, ""); val[0] = a; val[1] = b; }
    Vec(T a, T b, T c) { static_assert(N == 3, ""); val[0] = a; val[1] = b; val[2] = c; }
    template <class U> Vec(const Vec<U, N>& o) { for (int i = 0; i < N; i++) val[i] = static_cast<T>(o.val[i]); }
    T& operator[](int i) { return val[i]; }
    const T& operator[](int i) const { return val[i]; }
    Vec operator-(const Vec& o) const { Vec r; for (int i = 0; i < N; i++) r.val[i] = val[i] - o.val[i]; return r; }
    Vec operator+(const Vec& o) const { Vec r; for (int i = 0; i < N; i++) r.val[i] = val[i] + o.val[i]; return r; }
};
template <class T, int N> inline Vec<T, N> operator*(double a, const Vec<T, N>& v) { Vec<T, N> r; for (int i = 0; i < N; i++) r.val[i] = static_cast<T>(a * v.val[i]); return r; }
template <class T, int N> inline Vec<T, N> operator*(const Vec<T, N>& v, double a) { return a * v; }
template <class T, int N> inline Vec<T, N> operator/(const Vec<T, N>& v, double a) { Vec<T, N> r; for (int i = 0; i < N; i++) r.val[i] = static_cast<T>(v.val[i] / a); return r; }
template <class T, int N> inline std::ostream& operator<<(std::ostream& os, const Vec<T, N>& v)
{
    os << "[";
    for (int i = 0; i < N; i++) os << (i ? ", " : "") << +v.val[i];
    return os << "]";
}
typedef Vec<unsigned char, 3> Vec3b;
typedef Vec<int, 2> Vec2i;
typedef Vec<double, 2> Vec2d;
typedef Vec<float, 3> Vec3f;
typedef Vec<double, 3> Vec3d;

template <class T> struct Rect_ {
    T x, y, width, height;
    Rect_() : x(0), y(0), width(0), height(0) {}
    Rect_(T x_, T y_, T w, T h) : x(x_), y(y_), width(w), height(h) {}
};
typedef Rect_<int> Rect;
template <class T> struct Size_ {
    T width, height;
    Size_() : width(0), height(0) {}
    Size_(T w, T h) : width(w), height(h) {}
};
typedef Size_<int> Size;

template <class T> struct DataType;
template <> struct DataType<unsigned char> { enum { depth = CV_8U, channels = 1 }; };
template <> struct DataType<int> { enum { depth = CV_32S, channels = 1 }; };
template <> struct DataType<float> { enum { depth = CV_32F, channels = 1 }; };
template <> struct DataType<double> { enum { depth = CV_64F, channels = 1 }; };
template <class T, int N> struct DataType<Vec<T, N>> { enum { depth = DataType<T>::depth, channels = N }; };

struct KeyPoint {          // 28 bytes, pt first
    Point2f pt;
    float size, angle, response;
    int octave, class_id;
    KeyPoint() : size(0), angle(-1), response(0), octave(0), class_id(-1) {}
    KeyPoint(float x, float y, float s) : pt(x, y), size(s), angle(-1), response(0), octave(0), class_id(-1) {}
};
static_assert(sizeof(KeyPoint) == 28, "cv::KeyPoint layout");

struct DMatch {            // 16 bytes
    int queryIdx, trainIdx, imgIdx;
    float distance;
    DMatch() : queryIdx(-1), trainIdx(-1), imgIdx(-1), distance(3.4e38f) {}
    DMatch(int q, int t, float d) : queryIdx(q), trainIdx(t), imgIdx(-1), distance(d) {}
};
static_assert(sizeof(DMatch) == 16, "cv::DMatch layout");

// dense, reference-counted 2-D matrix (the subset the hot path touches)
class Mat {
public:
    int rows = 0, cols = 0;
    unsigned char* data = nullptr;
    size_t step = 0;        // bytes between rows

    Mat() {}
    Mat(int r, int c, int type) { create(r, c, type); }
    // borrowed storage (no ownership), as cv::Mat(rows, cols, type, void* data, size_t step)
    Mat(int r, int c, int type, void* ext, size_t step_bytes = 0)
        : rows(r), cols(c), data(static_cast<unsigned char*>(ext)), type_(type)
    {
        step = step_bytes ? step_bytes : (size_t)c * elemSize();
    }
    void create(int r, int c, int type)
    {
        rows = r; cols = c; type_ = type;
        step = (size_t)c * elemSize();
        store_ = std::shared_ptr<unsigned char>(new unsigned char[step * (size_t)(r > 0 ? r : 0) + 16], std::default_delete<unsigned char[]>());
        data = store_.get();
        std::memset(data, 0, step * (size_t)(r > 0 ? r : 0));
    }
    static Mat zeros(int r, int c, int type) { return Mat(r, c, type); }
    static Mat eye(int r, int c, int type)
    {
        Mat m(r, c, type);
        for (int i = 0; i < r && i < c; i++) {
            if (m.depth() == CV_64F) m.at<double>(i, i) = 1.0;
            else if (m.depth() == CV_32F) m.at<float>(i, i) = 1.f;
            else CV_Error(Error::StsNotImplemented, "compat Mat::eye: CV_32F / CV_64F only");
        }
        return m;
    }
    // view of a rectangle of rows / columns: shares the storage
    Mat operator()(const Rect& roi) const
    {
        Mat m;
        m.rows = roi.height; m.cols = roi.width; m.type_ = type_; m.step = step; m.store_ = store_;
        m.data = data + step * (size_t)roi.y + elemSize() * (size_t)roi.x;
        return m;
    }
    Mat inv() const;
    int type() const { return type_; }
    int depth() const { return type_ & 7; }
    int channels() const { return (type_ >> CV_CN_SHIFT) + 1; }
    size_t elemSize() const
    {
        static const int sz[8] = {1, 1, 2, 2, 4, 4, 8, 2};
        return (size_t)sz[depth()] * channels();
    }
    bool empty() const { return data == nullptr || rows == 0 || cols == 0; }
    bool isContinuous() const { return step == (size_t)cols * elemSize(); }
    template <class T> T* ptr(int r = 0) { return reinterpret_cast<T*>(data + step * (size_t)r); }
    template <class T> const T* ptr(int r = 0) const { return reinterpret_cast<const T*>(data + step * (size_t)r); }
    template <class T> T& at(int r, int c) { return ptr<T>(r)[c]; }
    template <class T> const T& at(int r, int c) const { return ptr<T>(r)[c]; }
    Mat clone() const
    {
        Mat m(rows, cols, type_);
        for (int r = 0; r < rows; r++) std::memcpy(m.data + m.step * r, data + step * r, (size_t)cols * elemSize());
        return m;
    }

private:
    int type_ = 0;
    std::shared_ptr<unsigned char> store_;
};

// ---- small dense algebra on CV_64F matrices (rotation matrices: the callers' rectification arithmetic)
inline void compat_need_f64(const Mat& a, const char* what) { if (a.type() != CV_64FC1) CV_Error(Error::StsNotImplemented, std::string("compat ") + what + ": CV_64FC1 only"); }
inline Mat operator+(const Mat& a, const Mat& b)
{
    compat_need_f64(a, "Mat + Mat"); compat_need_f64(b, "Mat + Mat");
    if (a.rows != b.rows || a.cols != b.cols) CV_Error(Error::StsBadArg, "compat Mat + Mat: sizes differ");
    Mat c(a.rows, a.cols, a.type());
    for (int i = 0; i < a.rows; i++) for (int j = 0; j < a.cols; j++) c.at<double>(i, j) = a.at<double>(i, j) + b.at<double>(i, j);
    return c;
}
inline Mat operator*(const Mat& a, const Mat& b)
{
    compat_need_f64(a, "Mat * Mat"); compat_need_f64(b, "Mat * Mat");
    if (a.cols != b.rows) CV_Error(Error::StsBadArg, "compat Mat * Mat: inner sizes differ");
    Mat c(a.rows, b.cols, a.type());
    for (int i = 0; i < a.rows; i++)
        for (int j = 0; j < b.cols; j++) {
            double s = 0;
            for (int k = 0; k < a.cols; k++) s += a.at<double>(i, k) * b.at<double>(k, j);
            c.at<double>(i, j) = s;
        }
    return c;
}
inline Mat operator*(const Mat& a, double f)
{
    compat_need_f64(a, "Mat * scalar");
    Mat c(a.rows, a.cols, a.type());
    for (int i = 0; i < a.rows; i++) for (int j = 0; j < a.cols; j++) c.at<double>(i, j) = a.at<double>(i, j) * f;
    return c;
}
inline Mat operator*(double f, const Mat& a) { return a * f; }
inline Mat Mat::inv() const          // Gauss-Jordan with partial pivoting (cv::DECOMP_LU on a small square matrix)
{
    compat_need_f64(*this, "Mat::inv");
    if (rows != cols) CV_Error(Error::StsBadArg, "compat Mat::inv: square matrices only");
    const int n = rows;
    Mat a = clone(), r = Mat::eye(n, n, CV_64FC1);
    for (int c = 0; c < n; c++) {
        int p = c;
        for (int i = c + 1; i < n; i++) if (std::fabs(a.at<double>(i, c)) > std::fabs(a.at<double>(p, c))) p = i;
        if (a.at<double>(p, c) == 0.0) return Mat::zeros(n, n, CV_64FC1);
        for (int j = 0; j < n; j++) { std::swap(a.at<double>(c, j), a.at<double>(p, j)); std::swap(r.at<double>(c, j), r.at<double>(p, j)); }
        const double d = 1.0 / a.at<double>(c, c);
        for (int j = 0; j < n; j++) { a.at<double>(c, j) *= d; r.at<double>(c, j) *= d; }
        for (int i = 0; i < n; i++) {
            if (i == c) continue;
            const double f = a.at<double>(i, c);
            for (int j = 0; j < n; j++) { a.at<double>(i, j) -= f * a.at<double>(c, j); r.at<double>(i, j) -= f * r.at<double>(c, j); }
        }
    }
    return r;
}

// Mat_<T> with the comma initialiser: (Mat_<double>(3, 3) << a, b, c, ...)
template <class T> class Mat_ : public Mat {
public:
    Mat_() {}
    Mat_(int r, int c) : Mat(r, c, CV_MAKETYPE(DataType<T>::depth, DataType<T>::channels)) {}
    T& operator()(int r, int c) { return this->template at<T>(r, c); }
};
template <class T> class MatCommaInitializer_ {
public:
    MatCommaInitializer_(const Mat_<T>& m, const T& first) : m_(m), n_(0) { put(first); }
    MatCommaInitializer_& operator,(const T& v) { put(v); return *this; }
    operator Mat() const { return m_; }
    operator Mat_<T>() const { return m_; }
private:
    void put(const T& v) { if (n_ < m_.rows * m_.cols) { m_.template at<T>(n_ / m_.cols, n_ % m_.cols) = v; n_++; } }
    Mat_<T> m_;
    int n_;
};
template <class T, class U> inline MatCommaInitializer_<T> operator<<(const Mat_<T>& m, const U& v) { return MatCommaInitializer_<T>(m, static_cast<T>(v)); }
typedef Mat_<Vec2i> Mat2i;

inline void vconcat(const Mat* src, size_t n, Mat& dst)
{
    int rows = 0, cols = n ? src[0].cols : 0;
    for (size_t i = 0; i < n; i++) {
        if (src[i].rows && (src[i].cols != cols || src[i].type() != src[0].type())) CV_Error(Error::StsBadArg, "compat vconcat: column count / type differ");
        rows += src[i].rows;
    }
    Mat out(rows, cols, n ? src[0].type() : 0);
    int r0 = 0;
    for (size_t i = 0; i < n; i++)
        for (int r = 0; r < src[i].rows; r++, r0++) std::memcpy(out.data + out.step * (size_t)r0, src[i].data + src[i].step * (size_t)r, (size_t)cols * out.elemSize());
    dst = out;
}

enum NormTypes { NORM_L2 = 4, NORM_HAMMING = 6 };
enum RotateFlags { ROTATE_90_CLOCKWISE = 0, ROTATE_180 = 1, ROTATE_90_COUNTERCLOCKWISE = 2 };
inline void rotate(const Mat& src, Mat& dst, int code)
{
    const size_t es = src.elemSize();
    const bool quarter = code != ROTATE_180;
    Mat out(quarter ? src.cols : src.rows, quarter ? src.rows : src.cols, src.type());
    for (int i = 0; i < src.rows; i++)
        for (int j = 0; j < src.cols; j++) {
            int oi, oj;
            if (code == ROTATE_90_CLOCKWISE) { oi = j; oj = src.rows - 1 - i; }
            else if (code == ROTATE_180) { oi = src.rows - 1 - i; oj = src.cols - 1 - j; }
            else { oi = src.cols - 1 - j; oj = i; }
            std::memcpy(out.data + out.step * (size_t)oi + es * (size_t)oj, src.data + src.step * (size_t)i + es * (size_t)j, es);
        }
    dst = out;
}

// no image codecs in the shim: the declarations let callers compile and link, a call reports why it cannot work
enum ImreadModes { IMREAD_GRAYSCALE = 0, IMREAD_COLOR = 1 };
Mat imread(const std::string& path, int flags = IMREAD_COLOR);      // host/compat_io.cpp (in liberp_host.a)
bool imwrite(const std::string& path, const Mat& image);

inline int64 getTickCount() { return (int64)std::chrono::duration_cast<std::chrono::nanoseconds>(std::chrono::steady_clock::now().time_since_epoch()).count(); }
inline double getTickFrequency() { return 1e9; }

} // namespace cv

// cvcompat/opencv2/core/core.hpp -- the handful of OpenCV 2.4 types the reference's PUBLIC kfusion headers name
// (kfusion/types.hpp:20-27, kinfu.hpp, cuda/tsdf_volume.hpp, warp_field.hpp: Vec3f/Vec3i/Vec4f, Matx33f/44f, Affine3f,
// Mat, Ptr, CV_Assert).  OpenCV's C++ libraries are not installed in this image; when a real OpenCV is present put its
// include directory BEFORE include/cvcompat and this file is never seen.  Written for this repo (not copied from OpenCV);
// arithmetic follows OpenCV's definitions (float, left-to-right) so that host-side poses match df_hostmath.h.
#pragma once
#include <ostream>
#include <cmath>
#include <cstddef>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <string>
#include <vector>

#define CV_8U 0
#define CV_16U 2
#define CV_32S 4
#define CV_32F 5
#define CV_MAKETYPE(depth, cn) ((depth) + (((cn) - 1) << 3))
#define CV_8UC4 CV_MAKETYPE(CV_8U, 4)
#define CV_32FC3 CV_MAKETYPE(CV_32F, 3)
#define CV_32FC4 CV_MAKETYPE(CV_32F, 4)
#define CV_32SC3 CV_MAKETYPE(CV_32S, 3)
#define CV_Assert(expr)                                                                       \
    do {                                                                                      \
        if (!(expr)) { std::fprintf(stderr, "CV_Assert failed: %s (%s:%d)\n", #expr, __FILE__, __LINE__); std::abort(); } \
    } while (0)

namespace cv
{
    enum { DECOMP_LU = 0, DECOMP_SVD = 1 };
    typedef std::string String;

    template <typename T, int m, int n> struct Matx
    {
        T val[m * n];
        Matx() { for (int i = 0; i < m * n; ++i) val[i] = T(0); }
        Matx(T v0, T v1, T v2) { T v[] = {v0, v1, v2}; init(v, 3); }
        Matx(T v0, T v1, T v2, T v3) { T v[] = {v0, v1, v2, v3}; init(v, 4); }
        Matx(T v0, T v1, T v2, T v3, T v4, T v5, T v6, T v7, T v8) { T v[] = {v0, v1, v2, v3, v4, v5, v6, v7, v8}; init(v, 9); }
        static Matx all(T a) { Matx r; for (int i = 0; i < m * n; ++i) r.val[i] = a; return r; }
        static Matx eye() { Matx r; for (int i = 0; i < (m < n ? m : n); ++i) r.val[i * n + i] = T(1); return r; }
        T &operator()(int i, int j) { return val[i * n + j]; }
        const T &operator()(int i, int j) const { return val[i * n + j]; }
        T &operator()(int i) { return val[i]; }
        const T &operator()(int i) const { return val[i]; }
        Matx<T, n, m> t() const { Matx<T, n, m> r; for (int i = 0; i < m; ++i) for (int j = 0; j < n; ++j) r.val[j * m + i] = val[i * n + j]; return r; }
        Matx inv(int = DECOMP_LU) const;     // 3x3 only (closed form), defined below
    private:
        void init(const T *v, int k) { for (int i = 0; i < m * n; ++i) val[i] = i < k ? v[i] : T(0); }
    };

    template <typename T, int cn> struct Vec : public Matx<T, cn, 1>
    {
        Vec() {}
        Vec(T a, T b, T c) : Matx<T, cn, 1>(a, b, c) {}
        Vec(T a, T b, T c, T d) : Matx<T, cn, 1>(a, b, c, d) {}
        explicit Vec(const T *p) { for (int i = 0; i < cn; ++i) this->val[i] = p[i]; }
        Vec(const Matx<T, cn, 1> &o) : Matx<T, cn, 1>(o) {}
        template <typename T2> explicit Vec(const Vec<T2, cn> &o) { for (int i = 0; i < cn; ++i) this->val[i] = (T)o.val[i]; }   // cv::Vec3d(Vec3f)
        static Vec all(T a) { Vec r; for (int i = 0; i < cn; ++i) r.val[i] = a; return r; }
        T &operator[](int i) { return this->val[i]; }
        const T &operator[](int i) const { return this->val[i]; }
        Vec cross(const Vec &v) const
        { return Vec(this->val[1] * v.val[2] - this->val[2] * v.val[1], this->val[2] * v.val[0] - this->val[0] * v.val[2], this->val[0] * v.val[1] - this->val[1] * v.val[0]); }
        T dot(const Vec &v) const { T s = T(0); for (int i = 0; i < cn; ++i) s += this->val[i] * v.val[i]; return s; }
    };
    template <typename T, int cn> inline Vec<T, cn> operator+(const Vec<T, cn> &a, const Vec<T, cn> &b) { Vec<T, cn> r; for (int i = 0; i < cn; ++i) r[i] = a[i] + b[i]; return r; }
    template <typename T, int cn> inline Vec<T, cn> operator-(const Vec<T, cn> &a, const Vec<T, cn> &b) { Vec<T, cn> r; for (int i = 0; i < cn; ++i) r[i] = a[i] - b[i]; return r; }
    template <typename T, int cn> inline Vec<T, cn> operator-(const Vec<T, cn> &a) { Vec<T, cn> r; for (int i = 0; i < cn; ++i) r[i] = -a[i]; return r; }
    template <typename T, int cn> inline Vec<T, cn> operator*(const Vec<T, cn> &a, T s) { Vec<T, cn> r; for (int i = 0; i < cn; ++i) r[i] = a[i] * s; return r; }
    template <typename T, int cn> inline Vec<T, cn> operator*(T s, const Vec<T, cn> &a) { return a * s; }
    template <typename T, int cn> inline Vec<T, cn> operator/(const Vec<T, cn> &a, T s) { Vec<T, cn> r; for (int i = 0; i < cn; ++i) r[i] = a[i] / s; return r; }
    template <typename T, int cn> inline Vec<T, cn> &operator+=(Vec<T, cn> &a, const Vec<T, cn> &b) { for (int i = 0; i < cn; ++i) a[i] += b[i]; return a; }
    template <typename T, int cn> inline bool operator==(const Vec<T, cn> &a, const Vec<T, cn> &b) { for (int i = 0; i < cn; ++i) if (a[i] != b[i]) return false; return true; }
    template <typename T, int cn> inline bool operator!=(const Vec<T, cn> &a, const Vec<T, cn> &b) { return !(a == b); }
    template <typename T, int cn> inline Vec<T, cn> normalize(const Vec<T, cn> &v) { T n = std::sqrt(v.dot(v)); return v / n; }
    template <typename T, int cn> inline double norm(const Vec<T, cn> &v) { double s = 0; for (int i = 0; i < cn; ++i) s += (double)v[i] * v[i]; return std::sqrt(s); }

    template <typename T, int m, int k, int n> inline Matx<T, m, n> operator*(const Matx<T, m, k> &a, const Matx<T, k, n> &b)
    {
        Matx<T, m, n> r;
        for (int i = 0; i < m; ++i) for (int j = 0; j < n; ++j) { T s = T(0); for (int q = 0; q < k; ++q) s += a(i, q) * b(q, j); r(i, j) = s; }
        return r;
    }
    template <typename T, int m, int n> inline Vec<T, m> operator*(const Matx<T, m, n> &a, const Vec<T, n> &v)
    { Vec<T, m> r; for (int i = 0; i < m; ++i) { T s = T(0); for (int q = 0; q < n; ++q) s += a(i, q) * v[q]; r[i] = s; } return r; }

    template <typename T, int m, int n> inline Matx<T, m, n> Matx<T, m, n>::inv(int) const
    {
        static_assert(m == 3 && n == 3, "cvcompat: Matx::inv is implemented for 3x3 only");
        const T a = val[0], b = val[1], c = val[2], d = val[3], e = val[4], f = val[5], g = val[6], h = val[7], i = val[8];
        const T c00 = e * i - f * h, c01 = f * g - d * i, c02 = d * h - e * g;
        const T det = a * c00 + b * c01 + c * c02;
        const T id = T(1) / det;
        return Matx<T, 3, 3>(c00 * id, (c * h - b * i) * id, (b * f - c * e) * id, c01 * id, (a * i - c * g) * id, (c * d - a * f) * id,
                             c02 * id, (b * g - a * h) * id, (a * e - b * d) * id);
    }

    template <typename T, int m, int n> inline std::ostream &operator<<(std::ostream &os, const Matx<T, m, n> &v)
    {
        os << "[";
        for (int i = 0; i < m * n; ++i) os << (i ? (i % n == 0 && n > 1 ? "; " : ", ") : "") << v.val[i];
        return os << "]";
    }

    typedef Vec<float, 3> Vec3f;
    typedef Vec<float, 4> Vec4f;
    typedef Vec<float, 6> Vec6f;
    typedef Vec<int, 3> Vec3i;
    typedef Vec<double, 3> Vec3d;
    typedef Matx<float, 3, 3> Matx33f;
    typedef Matx<float, 4, 4> Matx44f;
    typedef Matx<float, 6, 6> Matx66f;

    // cv::Affine3<T> (opencv2/core/affine.hpp)
    template <typename T> struct Affine3
    {
        typedef Matx<T, 3, 3> Mat3;
        typedef Matx<T, 4, 4> Mat4;
        typedef Vec<T, 3> Vec3;
        Mat4 matrix;
        Affine3() : matrix(Mat4::eye()) {}
        Affine3(const Mat3 &R, const Vec3 &t = Vec3::all(0)) : matrix(Mat4::eye()) { rotation(R); translation(t); }
        Affine3(const Vec3 &rvec, const Vec3 &t) : matrix(Mat4::eye()) { rotation(rvec); translation(t); }
        static Affine3 Identity() { return Affine3(); }
        void rotation(const Mat3 &R) { for (int i = 0; i < 3; ++i) for (int j = 0; j < 3; ++j) matrix(i, j) = R(i, j); }
        void rotation(const Vec3 &rvec)
        {   // Rodrigues, evaluated in double on the T inputs (affine.hpp)
            double theta = norm(rvec);
            if (theta < 2.220446049250313e-16) { rotation(Mat3::eye()); return; }
            double c = std::cos(theta), s = std::sin(theta), c1 = 1. - c, itheta = 1. / theta;
            T rx = (T)(rvec[0] * itheta), ry = (T)(rvec[1] * itheta), rz = (T)(rvec[2] * itheta);
            const T rrt[9] = {rx * rx, rx * ry, rx * rz, rx * ry, ry * ry, ry * rz, rx * rz, ry * rz, rz * rz};
            const T r_x[9] = {0, -rz, ry, rz, 0, -rx, -ry, rx, 0};
            Mat3 R;
            for (int i = 0; i < 9; ++i) R.val[i] = (T)(c * ((i % 4 == 0) ? 1.0 : 0.0) + c1 * rrt[i] + s * r_x[i]);
            rotation(R);
        }
        void translation(const Vec3 &t) { for (int i = 0; i < 3; ++i) matrix(i, 3) = t[i]; }
        Mat3 rotation() const { Mat3 R; for (int i = 0; i < 3; ++i) for (int j = 0; j < 3; ++j) R(i, j) = matrix(i, j); return R; }
        Vec3 translation() const { return Vec3(matrix(0, 3), matrix(1, 3), matrix(2, 3)); }
        Affine3 inv(int method = DECOMP_SVD) const
        {
            Affine3 r;
            Mat3 Ri = rotation().inv(method);
            r.rotation(Ri);
            Vec3 t = translation(), ti;
            for (int i = 0; i < 3; ++i) ti[i] = -(Ri(i, 0) * t[0] + Ri(i, 1) * t[1] + Ri(i, 2) * t[2]);
            r.translation(ti);
            return r;
        }
        Affine3 translate(const Vec3 &t) const { Affine3 r = *this; r.translation(translation() + t); return r; }
    };
    template <typename T> inline Affine3<T> operator*(const Affine3<T> &A, const Affine3<T> &B)
    {
        Affine3<T> r;
        typename Affine3<T>::Mat3 RA = A.rotation(), RB = B.rotation(), R;
        typename Affine3<T>::Vec3 tA = A.translation(), tB = B.translation(), t;
        for (int i = 0; i < 3; ++i) {
            for (int j = 0; j < 3; ++j) R(i, j) = RA(i, 0) * RB(0, j) + RA(i, 1) * RB(1, j) + RA(i, 2) * RB(2, j);
            t[i] = RA(i, 0) * tB[0] + RA(i, 1) * tB[1] + RA(i, 2) * tB[2] + tA[i];
        }
        r.rotation(R); r.translation(t);
        return r;
    }
    template <typename T> inline Vec<T, 3> operator*(const Affine3<T> &a, const Vec<T, 3> &v)
    {
        const typename Affine3<T>::Mat4 &m = a.matrix;
        return Vec<T, 3>(m.val[0] * v[0] + m.val[1] * v[1] + m.val[2] * v[2] + m.val[3], m.val[4] * v[0] + m.val[5] * v[1] + m.val[6] * v[2] + m.val[7],
                         m.val[8] * v[0] + m.val[9] * v[1] + m.val[10] * v[2] + m.val[11]);
    }
    typedef Affine3<float> Affine3f;

    // reference-counted owner, enough of cv::Ptr for `cv::Ptr<KinFu>` / `KinFu::Ptr`
    template <typename T> struct Ptr : public std::shared_ptr<T>
    {
        Ptr() {}
        Ptr(T *p) : std::shared_ptr<T>(p) {}
        operator T *() const { return this->get(); }
        bool empty() const { return !this->get(); }
    };

    // dense host matrix: rows x cols of `type`, shared buffer, like cv::Mat for the uses in kinfu.cpp / demo.cpp
    class Mat
    {
    public:
        int rows, cols;
        size_t step;
        unsigned char *data;
        Mat() : rows(0), cols(0), step(0), data(0), type_(0) {}
        Mat(int r, int c, int type) : rows(0), cols(0), step(0), data(0), type_(0) { create(r, c, type); }
        void create(int r, int c, int type)
        {
            if (r == rows && c == cols && type == type_ && data) return;
            rows = r; cols = c; type_ = type; step = (size_t)c * elemSize();
            buf_.reset(new std::vector<unsigned char>(step * (size_t)r));
            data = buf_->empty() ? 0 : &(*buf_)[0];
        }
        size_t elemSize() const { static const int sz[] = {1, 1, 2, 2, 4, 4, 8}; return (size_t)sz[type_ & 7] * (size_t)((type_ >> 3) + 1); }
        int type() const { return type_; }
        bool empty() const { return data == 0 || rows * cols == 0; }
        // dst(i) = saturate(src(i) * alpha + beta) for the single-channel depth previews of demo.cpp (u8/u16/f32 -> u8/u16/f32)
        void convertTo(Mat &dst, int rtype, double alpha = 1.0, double beta = 0.0) const
        {
            const int cn = (type_ >> 3) + 1;
            Mat out(rows, cols, CV_MAKETYPE(rtype & 7, cn));
            for (int r = 0; r < rows; ++r)
                for (int c = 0; c < cols * cn; ++c) {
                    double v = 0;
                    switch (type_ & 7) {
                        case CV_8U: v = ptr<unsigned char>(r)[c]; break;
                        case CV_16U: v = ptr<unsigned short>(r)[c]; break;
                        case CV_32F: v = ptr<float>(r)[c]; break;
                        default: break;
                    }
                    v = v * alpha + beta;
                    switch (rtype & 7) {
                        case CV_8U: out.ptr<unsigned char>(r)[c] = (unsigned char)(v < 0 ? 0 : v > 255 ? 255 : (int)(v + 0.5)); break;
                        case CV_16U: out.ptr<unsigned short>(r)[c] = (unsigned short)(v < 0 ? 0 : v > 65535 ? 65535 : (int)(v + 0.5)); break;
                        case CV_32F: out.ptr<float>(r)[c] = (float)v; break;
                        default: break;
                    }
                }
            dst = out;
        }
        template <typename T> T *ptr(int r = 0) { return (T *)(data + (size_t)r * step); }
        template <typename T> const T *ptr(int r = 0) const { return (const T *)(data + (size_t)r * step); }
        template <typename T> T &at(int i) { return rows == 1 ? ptr<T>(0)[i] : ptr<T>(i / cols)[i % cols]; }
        template <typename T> const T &at(int i) const { return rows == 1 ? ptr<T>(0)[i] : ptr<T>(i / cols)[i % cols]; }
        template <typename T> T &at(int i, int j) { return ptr<T>(i)[j]; }
        template <typename T> const T &at(int i, int j) const { return ptr<T>(i)[j]; }
    private:
        int type_;
        std::shared_ptr<std::vector<unsigned char> > buf_;
    };
}

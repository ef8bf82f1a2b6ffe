// oracle/ref_shim/ref_cv_impl.cc -- the OpenCV functions the reference calls, for oracle/_ref (TEST INFRASTRUCTURE ONLY).
// Image primitives forward to the oracle primitives (pinned to python-cv2 golden vectors by tests/test_oracle_golden.py);
// the matrix algebra follows cv2's cv::gemm / norm (pinned by tests/test_ref_shim_golden.py).  See opencv2/core/core.hpp.
#include <opencv2/core/core.hpp>

#include "../orb_oracle.h"

namespace cv {

// ---- matrix algebra -------------------------------------------------------------------------------------------------
static inline double elem(const Mat &m, int i, int j) {
    return m.depth() == CV_32F ? (double)m.at<float>(i, j) : m.at<double>(i, j);
}

// D = alpha*op(A)*op(B) + beta*op(C)   (OpenCV core/matmul.cpp).  CV_32F: when flags == 0, the inner length is 2..4 and
// the result is as wide or as high as that length, matmul.cpp takes its unrolled small-matrix branch, which sums the
// products in FLOAT, left to right; every other shape goes through GEMMSingleMul<float,double> (double accumulation).
// Either way the result is (float)(acc*alpha + c*beta) evaluated in double.  Verified against cv2.gemm (4.13) on random
// inputs for 3x3*3x1(+c), 3x3*3x2, 3x3*3x3, 3x3*3x4, 4x4*4x4 (float path) and A^T*B, 3x4*4x1, 1x3*3x1, 5x5*5x1 (double).
void gemm(const Mat &A, const Mat &B, double alpha, const Mat &C, double beta, Mat &D, int flags) {
    CV_Assert(A.type() == B.type() && (A.type() == CV_32F || A.type() == CV_64F));
    const bool tA = flags & GEMM_1_T, tB = flags & GEMM_2_T, tC = flags & GEMM_3_T;
    const int n = tA ? A.cols : A.rows, len = tA ? A.rows : A.cols;
    const int lenB = tB ? B.cols : B.rows, m = tB ? B.rows : B.cols;
    CV_Assert(len == lenB);
    const bool haveC = !C.empty() && beta != 0;
    Mat out(n, m, A.type());
    const bool f32 = A.type() == CV_32F;
    const bool small_float_path = f32 && flags == 0 && len >= 2 && len <= 4 && (len == m || len == n);
    for (int i = 0; i < n; i++)
        for (int j = 0; j < m; j++) {
            double acc;
            if (small_float_path) {
                float t = A.at<float>(i, 0) * B.at<float>(0, j);
                for (int k = 1; k < len; k++) t = t + A.at<float>(i, k) * B.at<float>(k, j);   // -ffp-contract=off: no FMA
                acc = (double)t;
            } else {
                acc = 0;
                for (int k = 0; k < len; k++) acc += elem(A, tA ? k : i, tA ? i : k) * elem(B, tB ? j : k, tB ? k : j);
            }
            double v = acc * alpha;
            if (haveC) v += elem(C, tC ? j : i, tC ? i : j) * beta;
            if (f32) out.at<float>(i, j) = (float)v; else out.at<double>(i, j) = v;
        }
    D = out;
}

void transpose(const Mat &src, Mat &dst) {
    Mat out(src.cols, src.rows, src.type());
    const size_t es = src.elemSize();
    for (int i = 0; i < src.rows; i++)
        for (int j = 0; j < src.cols; j++) std::memcpy(out.data + (size_t)j * out.step.p[0] + (size_t)i * es, src.data + (size_t)i * src.step.p[0] + (size_t)j * es, es);
    dst = out;
}

// convertTo(m, -1, alpha): cvtScale_<float,float,float> multiplies in float by (float)alpha (restated from 2.4; not arbitrated)
static Mat scaled(const Mat &a, double alpha) {
    if (alpha == 1) return a;
    Mat out(a.rows, a.cols, a.type());
    for (int i = 0; i < a.rows; i++)
        for (int j = 0; j < a.cols; j++) {
            if (a.type() == CV_32F) out.at<float>(i, j) = a.at<float>(i, j) * (float)alpha + 0.0f;
            else out.at<double>(i, j) = a.at<double>(i, j) * alpha;
        }
    return out;
}

Mat MatExpr::eval() const {
    switch (kind) {
    case MAT: return a;
    case SCALED: return scaled(a, alpha);
    case T: { Mat t; transpose(a, t); return scaled(t, alpha); }     // MatOp_T::assign: transpose, then convertTo(alpha)
    case GEMM: { Mat d; gemm(a, b, alpha, c, beta, d, flags); return d; }
    case ADD: {                                                      // MatOp_AddEx: a + b (beta 1), a - b (beta -1), else scaleAdd
        CV_Assert(a.rows == b.rows && a.cols == b.cols && a.type() == b.type());
        Mat out(a.rows, a.cols, a.type());
        for (int i = 0; i < a.rows; i++)
            for (int j = 0; j < a.cols; j++) {
                if (a.type() == CV_32F) {
                    const float x = a.at<float>(i, j), y = b.at<float>(i, j);
                    out.at<float>(i, j) = beta == 1 ? x + y : beta == -1 ? x - y : y * (float)beta + x;
                } else {
                    out.at<double>(i, j) = a.at<double>(i, j) + beta * b.at<double>(i, j);
                }
            }
        return out;
    }
    }
    return Mat();
}

MatExpr Mat::t() const { MatExpr e; e.kind = MatExpr::T; e.a = *this; e.alpha = 1; return e; }
MatExpr MatExpr::t() const {
    if (kind == T) { MatExpr e; e.kind = SCALED; e.a = a; e.alpha = alpha; return e; }
    if (kind == SCALED || kind == MAT) { MatExpr e; e.kind = T; e.a = a; e.alpha = kind == MAT ? 1 : alpha; return e; }
    return eval().t();
}

double Mat::dot(const Mat &m) const {   // dotProd_<float>: double accumulation of double products, element order
    CV_Assert(type() == m.type() && total() == m.total());
    double r = 0;
    Mat a = (isContinuous() ? *this : clone()), b = (m.isContinuous() ? m : m.clone());
    const size_t n = total();
    for (size_t i = 0; i < n; i++)
        r += type() == CV_32F ? (double)((const float *)a.data)[i] * (double)((const float *)b.data)[i]
                              : ((const double *)a.data)[i] * ((const double *)b.data)[i];
    return r;
}

double norm(const Mat &m, int normType) {   // normL2_32f: double accumulation of v*v, then sqrt
    CV_Assert(normType == NORM_L2);
    double s = 0;
    for (int i = 0; i < m.rows; i++)
        for (int j = 0; j < m.cols; j++) { const double v = elem(m, i, j); s += v * v; }
    return std::sqrt(s);
}

// operator glue: which MatOp the 2.4 expression templates would have built
static MatExpr gemm_expr(const Mat &a, const Mat &b, double alpha, int flags) {
    MatExpr e; e.kind = MatExpr::GEMM; e.a = a; e.b = b; e.alpha = alpha; e.beta = 0; e.flags = flags; return e;
}
static void operand(const MatExpr &e, Mat &m, double &alpha, bool &transposed) {
    switch (e.kind) {
    case MatExpr::MAT: m = e.a; alpha = 1; transposed = false; return;
    case MatExpr::SCALED: m = e.a; alpha = e.alpha; transposed = false; return;
    case MatExpr::T: m = e.a; alpha = e.alpha; transposed = true; return;
    default: m = e.eval(); alpha = 1; transposed = false; return;
    }
}
MatExpr operator*(const Mat &a, const Mat &b) { return gemm_expr(a, b, 1, 0); }
MatExpr operator*(const MatExpr &e, const Mat &b) { Mat m; double al; bool t; operand(e, m, al, t); return gemm_expr(m, b, al, t ? GEMM_1_T : 0); }
MatExpr operator*(const Mat &a, const MatExpr &e) { Mat m; double al; bool t; operand(e, m, al, t); return gemm_expr(a, m, al, t ? GEMM_2_T : 0); }
MatExpr operator*(const MatExpr &e1, const MatExpr &e2) {
    Mat m1, m2; double a1, a2; bool t1, t2;
    operand(e1, m1, a1, t1); operand(e2, m2, a2, t2);
    return gemm_expr(m1, m2, a1 * a2, (t1 ? GEMM_1_T : 0) | (t2 ? GEMM_2_T : 0));
}
static MatExpr scale_expr(const MatExpr &e, double s) {
    MatExpr r = e;
    if (e.kind == MatExpr::MAT) { r.kind = MatExpr::SCALED; r.alpha = s; return r; }
    if (e.kind == MatExpr::SCALED || e.kind == MatExpr::T || e.kind == MatExpr::GEMM) { r.alpha = e.alpha * s; if (e.kind == MatExpr::GEMM) r.beta = e.beta * s; return r; }
    MatExpr q; q.kind = MatExpr::SCALED; q.a = e.eval(); q.alpha = s; return q;
}
MatExpr operator*(double s, const Mat &a) { return scale_expr(MatExpr(a), s); }
MatExpr operator*(const Mat &a, double s) { return scale_expr(MatExpr(a), s); }
MatExpr operator*(double s, const MatExpr &e) { return scale_expr(e, s); }
MatExpr operator*(const MatExpr &e, double s) { return scale_expr(e, s); }
MatExpr operator/(const Mat &a, double s) { return scale_expr(MatExpr(a), 1. / s); }
MatExpr operator/(const MatExpr &e, double s) { return scale_expr(e, 1. / s); }
MatExpr operator-(const Mat &a) { return scale_expr(MatExpr(a), -1); }
MatExpr operator-(const MatExpr &e) { return scale_expr(e, -1); }

static MatExpr add_expr(const Mat &a, const Mat &b, double beta) {
    MatExpr e; e.kind = MatExpr::ADD; e.a = a; e.b = b; e.alpha = 1; e.beta = beta; return e;
}
MatExpr operator+(const Mat &a, const Mat &b) { return add_expr(a, b, 1); }
MatExpr operator+(const MatExpr &e, const Mat &b) {
    if (e.kind == MatExpr::GEMM && e.c.empty()) { MatExpr r = e; r.c = b; r.beta = 1; return r; }   // MatOp_GEMM::add: one gemm call
    if (e.kind == MatExpr::SCALED) return add_expr(b, e.a, e.alpha);                                 // b + alpha*a
    return add_expr(e.eval(), b, 1);
}
MatExpr operator+(const Mat &a, const MatExpr &e) { return e + a; }
MatExpr operator+(const MatExpr &e1, const MatExpr &e2) { return e1 + e2.eval(); }
MatExpr operator-(const Mat &a, const Mat &b) { return add_expr(a, b, -1); }
MatExpr operator-(const MatExpr &e, const Mat &b) { return add_expr(e.eval(), b, -1); }
MatExpr operator-(const Mat &a, const MatExpr &e) { return add_expr(a, e.eval(), -1); }

// ---- image primitives: the oracle's (pinned to cv2 golden vectors) --------------------------------------------------
void FAST(InputArray image, std::vector<KeyPoint> &keypoints, int threshold, bool nonmaxSuppression) {
    const Mat img = image.getMat();
    CV_Assert(img.type() == CV_8UC1 && nonmaxSuppression);
    keypoints.clear();
    if (img.cols < 7 || img.rows < 7) return;
    const int cap = ((img.cols + 1) / 2 + 1) * ((img.rows + 1) / 2 + 1) + 8;
    std::vector<int> xs(cap), ys(cap), sc(cap);
    const int n = orb_oracle_fast_detect(img.data, img.cols, img.rows, img.step, threshold, xs.data(), ys.data(), sc.data(), cap);
    CV_Assert(n <= cap);
    for (int k = 0; k < n; k++) keypoints.push_back(KeyPoint((float)xs[k], (float)ys[k], 7.f, -1, (float)sc[k]));
}

void resize(InputArray _src, OutputArray _dst, Size dsize, double, double, int interpolation) {
    const Mat src = _src.getMat();
    CV_Assert(src.type() == CV_8UC1 && interpolation == INTER_LINEAR);
    _dst.create(dsize, src.type());
    Mat dst = _dst.getMat();
    CV_Assert(!(dsize.width * 2 == src.cols && dsize.height * 2 == src.rows));   // an exact 2:1 ratio silently means INTER_AREA
    orb_oracle_resize_linear_u8(src.data, src.cols, src.rows, src.step, dst.data, dst.cols, dst.rows, dst.step);
}

static inline int reflect101(int i, int n) {
    if (n == 1) return 0;
    while (i < 0 || i >= n) i = i < 0 ? -i : 2 * (n - 1) - i;
    return i;
}

void copyMakeBorder(InputArray _src, OutputArray _dst, int top, int bottom, int left, int right, int borderType, const Scalar &) {
    const Mat src = _src.getMat();
    CV_Assert(src.type() == CV_8UC1 && (borderType & ~BORDER_ISOLATED) == BORDER_REFLECT_101);
    _dst.create(src.rows + top + bottom, src.cols + left + right, src.type());
    Mat dst = _dst.getMat();
    for (int y = 0; y < dst.rows; y++) {
        const uchar *s = src.ptr(reflect101(y - top, src.rows));
        uchar *d = dst.ptr(y);
        if (y >= top && y < top + src.rows && d + left == s) {   // the interior already lives in dst (ComputePyramid, level > 0)
            for (int x = 0; x < left; x++) d[x] = s[reflect101(x - left, src.cols)];
            for (int x = left + src.cols; x < dst.cols; x++) d[x] = s[reflect101(x - left, src.cols)];
            continue;
        }
        for (int x = 0; x < dst.cols; x++) d[x] = s[reflect101(x - left, src.cols)];
    }
}

// cv::GaussianBlur(m, m, Size(7,7), 2, 2, BORDER_REFLECT_101) on a sub-matrix without BORDER_ISOLATED: OpenCV reads the
// 3 px outside the ROI from the parent buffer.  The reference's parent holds the reflect-101 frame of the ROI, so that
// equals reflecting by index, which is what the oracle primitive does; the equality is checked, not assumed.
void GaussianBlur(InputArray _src, OutputArray _dst, Size ksize, double sigmaX, double sigmaY, int borderType) {
    const Mat src = _src.getMat();
    CV_Assert(src.type() == CV_8UC1 && ksize.width == 7 && ksize.height == 7 && sigmaX == 2 && sigmaY == 2 && borderType == BORDER_REFLECT_101);
    if (src.datastart && src.data - 3 * (ptrdiff_t)src.step - 3 >= src.datastart && src.ptr(src.rows - 1) + src.cols + 3 * src.step + 3 <= src.dataend) {
        for (int y = -3; y < src.rows + 3; y++)
            for (int x = -3; x < src.cols + 3; x++) {
                if (y >= 0 && y < src.rows && x >= 0 && x < src.cols) { x = src.cols - 1; continue; }
                CV_Assert(*(src.data + (ptrdiff_t)y * (ptrdiff_t)src.step + x) == src.at<uchar>(reflect101(y, src.rows), reflect101(x, src.cols)));
            }
    }
    Mat tmp(src.rows, src.cols, CV_8UC1);
    orb_oracle_blur7_u8(src.data, src.cols, src.rows, src.step, tmp.data, tmp.step);
    _dst.create(src.rows, src.cols, CV_8UC1);
    Mat dst = _dst.getMat();
    for (int y = 0; y < src.rows; y++) std::memcpy(dst.ptr(y), tmp.ptr(y), (size_t)src.cols);
}

float fastAtan2(float y, float x) { return orb_oracle_fast_atan2(y, x); }

void undistortPoints(InputArray _src, OutputArray _dst, InputArray _K, InputArray _D, InputArray _R, InputArray _P) {
    const Mat src = _src.getMat(), K = _K.getMat(), D = _D.getMat(), P = _P.getMat();
    CV_Assert(src.type() == CV_32FC2 && K.type() == CV_32F && D.type() == CV_32F && _R.empty());
    CV_Assert(!P.empty() && P.data == K.data);   // Frame.cc passes P = K
    const int n = (int)src.total();
    float dist[5] = {0, 0, 0, 0, 0};
    for (int i = 0; i < (int)D.total() && i < 5; i++) dist[i] = D.at<float>(i);
    std::vector<float> in((size_t)2 * n), out((size_t)2 * n);
    Mat s = src.isContinuous() ? src : src.clone();
    std::memcpy(in.data(), s.data, sizeof(float) * 2 * (size_t)n);
    orb_oracle_undistort_points(in.data(), n, K.at<float>(0, 0), K.at<float>(1, 1), K.at<float>(0, 2), K.at<float>(1, 2), dist, out.data());
    _dst.create(src.rows, src.cols, CV_32FC2);
    Mat dst = _dst.getMat();
    CV_Assert(dst.isContinuous());
    std::memcpy(dst.data, out.data(), sizeof(float) * 2 * (size_t)n);
}

// OpenCV 2.4 features2d/keypoint.cpp
namespace {
struct KeypointResponseGreaterThanThreshold {
    explicit KeypointResponseGreaterThanThreshold(float v) : value(v) {}
    bool operator()(const KeyPoint &k) const { return k.response >= value; }
    float value;
};
struct KeypointResponseGreater {
    bool operator()(const KeyPoint &a, const KeyPoint &b) const { return a.response > b.response; }
};
}  // namespace
void KeyPointsFilter::retainBest(std::vector<KeyPoint> &keypoints, int n_points) {
    if (n_points >= 0 && keypoints.size() > (size_t)n_points) {
        if (n_points == 0) { keypoints.clear(); return; }
        std::nth_element(keypoints.begin(), keypoints.begin() + n_points, keypoints.end(), KeypointResponseGreater());
        const float ambiguous_response = keypoints[n_points - 1].response;
        std::vector<KeyPoint>::const_iterator new_end =
            std::partition(keypoints.begin() + n_points, keypoints.end(), KeypointResponseGreaterThanThreshold(ambiguous_response));
        keypoints.resize(new_end - keypoints.begin());
    }
}

}  // namespace cv

// ---- shim self-test hook: cv::gemm of the stand-in header, so that tests can pin it to python-cv2's cv2.gemm ---------------
extern "C" void ref_shim_gemm(const float *A, int ar, int ac, const float *B, int br, int bc, double alpha, const float *Cm, double beta,
                              int flags, float *out) {
    cv::Mat a(ar, ac, CV_32F, const_cast<float *>(A)), b(br, bc, CV_32F, const_cast<float *>(B));
    const int n = (flags & cv::GEMM_1_T) ? ac : ar, m = (flags & cv::GEMM_2_T) ? br : bc;
    cv::Mat c = Cm ? cv::Mat(n, m, CV_32F, const_cast<float *>(Cm)) : cv::Mat(), d;
    cv::gemm(a, b, alpha, c, beta, d, flags);
    for (int i = 0; i < n; i++) std::memcpy(out + (size_t)i * m, d.ptr(i), sizeof(float) * (size_t)m);
}
extern "C" double ref_shim_norm(const float *v, int n) { return cv::norm(cv::Mat(n, 1, CV_32F, const_cast<float *>(v))); }

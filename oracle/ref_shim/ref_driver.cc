// oracle/ref_shim/ref_driver.cc -- extern "C" drivers around the reference's OWN classes (TEST INFRASTRUCTURE ONLY).
//
// Every entry point builds real ORB_SLAM::Frame / KeyFrame / MapPoint objects from plain arrays through their public
// interface and then calls the real ORB_SLAM::ORBextractor / ORBmatcher methods.  The same file is compiled twice:
//   oracle/_ref/libref_orbslam.so     reference ORBextractor.cc + ORBmatcher.cc            (what the oracle is diffed against)
//   oracle/_ref/libfacade_orbslam.so  orb_slam_b200/host/ORBextractor.cc + ORBmatcher.cc   (the product's drop-in facades)
// both next to the reference's unmodified Frame.cc, KeyFrame.cc, MapPoint.cc, Map.cc, KeyFrameDatabase.cc and DBoW2.
// It therefore only uses what include/ORBextractor.h and include/ORBmatcher.h of the reference declare.
#include <opencv2/core/core.hpp>   // every standard header first: the access hack below must not reach libstdc++
#include <boost/thread.hpp>
#include <cstdint>
#include <map>
#include <new>
#include <numeric>
#define protected public   // the drivers set a few protected MapPoint fields (descriptor, normal, distance range) directly
#define private public
#include "ORBmatcher.h"
#include "ORBextractor.h"
#include "Frame.h"
#include "KeyFrame.h"
#include "MapPoint.h"
#include "Map.h"
#include "KeyFrameDatabase.h"
#undef protected
#undef private

using namespace ORB_SLAM;

namespace {

struct RefKeyPoint { float x, y, size, angle, response; int32_t octave, class_id; };
static_assert(sizeof(RefKeyPoint) == 28 && sizeof(cv::KeyPoint) == 28, "cv::KeyPoint must be the 28-byte OpenCV 2.4 layout");

// objects that must outlive the calls: one vocabulary / map / keyframe database and every MapPoint / KeyFrame ever made
struct World {
    ORBVocabulary voc;
    Map map;
    KeyFrameDatabase db;
    std::vector<MapPoint *> mps;
    std::vector<KeyFrame *> kfs;
    std::vector<ORBextractor *> exs;
    KeyFrame *anchor;   // reference keyframe of free-floating map points (MapPoint's constructor dereferences it)
    World() : db(voc), anchor(NULL) {}
};
World *g_world = NULL;

// KeyFrames and MapPoints are placed in one arena in creation order.  The reference keys several containers by POINTER
// (std::map<KeyFrame*, size_t> mObservations, std::set<MapPoint*>): MapPoint::ComputeDistinctiveDescriptors, for one, breaks
// median ties by iteration order, i.e. by the addresses malloc happened to return.  With addresses ascending in creation
// order the reference's behaviour is reproducible, and identical between the two builds of this driver.
void *arena_alloc(size_t bytes) {
    static char *base = NULL;
    static size_t used = 0, cap = (size_t)1 << 30;
    if (!base) base = static_cast<char *>(std::malloc(cap));   // untouched pages cost nothing
    used = (used + 63) / 64 * 64;
    if (!base || used + bytes > cap) { std::fprintf(stderr, "ref_driver: object arena exhausted\n"); std::abort(); }
    void *p = base + used;
    used += bytes;
    return p;
}

cv::Mat pose_from(const float *T12) {   // 3x4 row-major [R|t] -> 4x4 CV_32F
    cv::Mat T = cv::Mat::eye(4, 4, CV_32F);
    if (T12)
        for (int r = 0; r < 3; r++)
            for (int c = 0; c < 4; c++) T.at<float>(r, c) = T12[4 * r + c];
    return T;
}

cv::Mat point3(const float *p) {
    cv::Mat m(3, 1, CV_32F);
    for (int k = 0; k < 3; k++) m.at<float>(k) = p[k];
    return m;
}

cv::Mat desc_row(const uint8_t *d) {
    cv::Mat m(1, 32, CV_8UC1);
    std::memcpy(m.data, d, 32);
    return m;
}

World &world();

MapPoint *new_map_point(const float *pos3, KeyFrame *ref = NULL) {
    static const float zero[3] = {0, 0, 0};
    World &w = world();
    MapPoint *p = new (arena_alloc(sizeof(MapPoint))) MapPoint(point3(pos3 ? pos3 : zero), ref ? ref : w.anchor, &w.map);
    w.mps.push_back(p);
    return p;
}

void fill_frame_tables(Frame &F, float scale_factor, int nlevels) {   // Frame.cc:90-103
    F.mnScaleLevels = nlevels;
    F.mfScaleFactor = scale_factor;
    F.mvScaleFactors.resize(nlevels);
    F.mvLevelSigma2.resize(nlevels);
    F.mvScaleFactors[0] = 1.0f;
    F.mvLevelSigma2[0] = 1.0f;
    for (int i = 1; i < nlevels; i++) {
        F.mvScaleFactors[i] = F.mvScaleFactors[i - 1] * F.mfScaleFactor;
        F.mvLevelSigma2[i] = F.mvScaleFactors[i] * F.mvScaleFactors[i];
    }
    F.mvInvLevelSigma2.resize(nlevels);
    for (int i = 0; i < nlevels; i++) F.mvInvLevelSigma2[i] = 1 / F.mvLevelSigma2[i];
}

// a Frame from given keypoints / descriptors, zero distortion: the statics of Frame.cc:65-86 and the grid fill of
// :109-123 repeated on public members, with the reference's own Frame::PosInGrid deciding the cell
Frame *frame_from_arrays(const RefKeyPoint *kps, const uint8_t *desc, int n, int W, int H, float fx, float fy, float cx, float cy,
                         float scale_factor, int nlevels) {
    Frame *F = new Frame();
    F->mpORBvocabulary = &world().voc;
    F->mpORBextractor = NULL;
    F->im = cv::Mat(H, W, CV_8UC1);
    F->mTimeStamp = 0;
    F->mK = cv::Mat::eye(3, 3, CV_32F);
    F->mK.at<float>(0, 0) = fx; F->mK.at<float>(1, 1) = fy; F->mK.at<float>(0, 2) = cx; F->mK.at<float>(1, 2) = cy;
    F->mDistCoef = cv::Mat::zeros(4, 1, CV_32F);
    F->N = n;
    F->mvKeys.resize(n);
    if (n) std::memcpy(&F->mvKeys[0], kps, sizeof(RefKeyPoint) * (size_t)n);
    F->mvKeysUn = F->mvKeys;   // Frame.cc:291-295
    F->mDescriptors = cv::Mat(std::max(n, 1), 32, CV_8UC1);
    if (n) std::memcpy(F->mDescriptors.data, desc, (size_t)n * 32);
    if (n == 0) F->mDescriptors = cv::Mat();
    F->mvpMapPoints = std::vector<MapPoint *>(n, static_cast<MapPoint *>(NULL));
    Frame::mnMinX = 0; Frame::mnMaxX = W; Frame::mnMinY = 0; Frame::mnMaxY = H;   // :342-348
    Frame::mfGridElementWidthInv = static_cast<float>(FRAME_GRID_COLS) / static_cast<float>(Frame::mnMaxX - Frame::mnMinX);
    Frame::mfGridElementHeightInv = static_cast<float>(FRAME_GRID_ROWS) / static_cast<float>(Frame::mnMaxY - Frame::mnMinY);
    Frame::fx = fx; Frame::fy = fy; Frame::cx = cx; Frame::cy = cy;
    Frame::mbInitialComputations = false;
    F->mnId = Frame::nNextId++;
    fill_frame_tables(*F, scale_factor, nlevels);
    for (size_t i = 0; i < F->mvKeysUn.size(); i++) {
        int gx, gy;
        if (F->PosInGrid(F->mvKeysUn[i], gx, gy)) F->mGrid[gx][gy].push_back(i);
    }
    F->mvbOutlier = std::vector<bool>(n, false);
    F->mTcw = cv::Mat::eye(4, 4, CV_32F);
    F->mpReferenceKF = NULL;
    return F;
}

World &world() {
    if (!g_world) {
        g_world = new World();
        // anchor keyframe: built from an empty 64x48 frame
        Frame *F = frame_from_arrays(NULL, NULL, 0, 64, 48, 50.f, 50.f, 32.f, 24.f, 1.2f, 8);
        g_world->anchor = new (arena_alloc(sizeof(KeyFrame))) KeyFrame(*F, &g_world->map, &g_world->db);
        g_world->kfs.push_back(g_world->anchor);
        delete F;
    }
    return *g_world;
}

// index of the map point held in `slot` within `owner` (the vector it was taken from), -1 for NULL, -2 for a foreign point
int index_of(const std::map<MapPoint *, int> &idx, MapPoint *p) {
    if (!p) return -1;
    std::map<MapPoint *, int>::const_iterator it = idx.find(p);
    return it == idx.end() ? -2 : it->second;
}

}  // namespace

extern "C" {

int ref_version() { return 2; }
#ifdef ORB_REF_FACADE
int ref_is_facade() { return 1; }
#else
int ref_is_facade() { return 0; }
#endif

// ---- E rows: ORBextractor::operator() ------------------------------------------------------------------------------
int ref_extract(int nfeatures, float scale_factor, int nlevels, int score_type, int fast_th, const uint8_t *img, int W, int H,
                size_t stride, RefKeyPoint *kps_out, uint8_t *desc_out, int cap) {
    ORBextractor ex(nfeatures, scale_factor, nlevels, score_type, fast_th);
    cv::Mat im(H, W, CV_8UC1, const_cast<uint8_t *>(img), stride);
    std::vector<cv::KeyPoint> keys;
    cv::Mat desc;
    ex(im, cv::Mat(), keys, desc);
    const int n = (int)keys.size();
    for (int i = 0; i < n && i < cap; i++) {
        std::memcpy(&kps_out[i], &keys[i], sizeof(RefKeyPoint));
        std::memcpy(desc_out + (size_t)i * 32, desc.ptr(i), 32);
    }
    return n;
}

// ---- Frame ---------------------------------------------------------------------------------------------------------
void ref_reset_frame_statics() { Frame::mbInitialComputations = true; }

// The reference's own constructor (Frame.cc:56-125): extraction, undistortion, image bounds, grid.  dist4 = k1,k2,p1,p2.
void *ref_frame_from_image(const uint8_t *img, int W, int H, size_t stride, float fx, float fy, float cx, float cy, const float *dist4,
                           int nfeatures, float scale_factor, int nlevels, int score_type, int fast_th) {
    World &w = world();
    ORBextractor *ex = new ORBextractor(nfeatures, scale_factor, nlevels, score_type, fast_th);
    w.exs.push_back(ex);
    cv::Mat im(H, W, CV_8UC1);
    for (int y = 0; y < H; y++) std::memcpy(im.ptr(y), img + (size_t)y * stride, (size_t)W);
    cv::Mat K = cv::Mat::eye(3, 3, CV_32F);
    K.at<float>(0, 0) = fx; K.at<float>(1, 1) = fy; K.at<float>(0, 2) = cx; K.at<float>(1, 2) = cy;
    cv::Mat D(4, 1, CV_32F);
    for (int i = 0; i < 4; i++) D.at<float>(i) = dist4 ? dist4[i] : 0.f;
    Frame::mbInitialComputations = true;   // bounds / grid constants of THIS geometry
    Frame *F = new Frame(im, 0.0, ex, &w.voc, K, D);
    if (F->mTcw.empty()) F->mTcw = cv::Mat::eye(4, 4, CV_32F);
    return F;
}

void *ref_frame_from_arrays(const RefKeyPoint *kps, const uint8_t *desc, int n, int W, int H, float fx, float fy, float cx, float cy,
                            float scale_factor, int nlevels) {
    return frame_from_arrays(kps, desc, n, W, H, fx, fy, cx, cy, scale_factor, nlevels);
}

void ref_frame_free(void *f) { delete static_cast<Frame *>(f); }
int ref_frame_n(void *f) { return static_cast<Frame *>(f)->N; }

void ref_frame_get(void *f, RefKeyPoint *keys, RefKeyPoint *keys_un, uint8_t *desc, float *bounds4, float *grid_inv2) {
    Frame *F = static_cast<Frame *>(f);
    for (int i = 0; i < F->N; i++) {
        if (keys) std::memcpy(&keys[i], &F->mvKeys[i], sizeof(RefKeyPoint));
        if (keys_un) std::memcpy(&keys_un[i], &F->mvKeysUn[i], sizeof(RefKeyPoint));
        if (desc) std::memcpy(desc + (size_t)i * 32, F->mDescriptors.ptr(i), 32);
    }
    if (bounds4) { bounds4[0] = (float)Frame::mnMinX; bounds4[1] = (float)Frame::mnMinY; bounds4[2] = (float)Frame::mnMaxX; bounds4[3] = (float)Frame::mnMaxY; }
    if (grid_inv2) { grid_inv2[0] = Frame::mfGridElementWidthInv; grid_inv2[1] = Frame::mfGridElementHeightInv; }
}

// the 64x48 grid as CSR, cell id = ix*48 + iy (Frame.cc:116-123)
void ref_frame_grid(void *f, int *cell_start /*3073*/, int *items /*N*/) {
    Frame *F = static_cast<Frame *>(f);
    int o = 0;
    for (int ix = 0; ix < FRAME_GRID_COLS; ix++)
        for (int iy = 0; iy < FRAME_GRID_ROWS; iy++) {
            cell_start[ix * FRAME_GRID_ROWS + iy] = o;
            for (size_t k = 0; k < F->mGrid[ix][iy].size(); k++) items[o++] = (int)F->mGrid[ix][iy][k];
        }
    cell_start[FRAME_GRID_COLS * FRAME_GRID_ROWS] = o;
}

int ref_frame_features_in_area(void *f, float x, float y, float r, int min_level, int max_level, int *out, int cap) {
    std::vector<size_t> v = static_cast<Frame *>(f)->GetFeaturesInArea(x, y, r, min_level, max_level);
    for (size_t i = 0; i < v.size() && (int)i < cap; i++) out[i] = (int)v[i];
    return (int)v.size();
}

// ---- M2: SearchByProjection(Frame &CurrentFrame, const Frame &LastFrame, float th), ORBmatcher.cc:1507-1620 ------------
// cur_mp_inout[i2]: -1 free, >= 0 occupied on entry (any id); on return the index of the Last feature whose map point was
// assigned to Current feature i2, occupied entries unchanged.
int ref_search_by_projection_ff(void *cur, void *last, const uint8_t *last_has_mp, const uint8_t *last_outlier, const float *last_world,
                                const float *Tcw12, float th, float nnratio, int check_orientation, int *cur_mp_inout) {
    Frame &C = *static_cast<Frame *>(cur), &L = *static_cast<Frame *>(last);
    std::map<MapPoint *, int> idx;
    for (int i = 0; i < L.N; i++) {
        L.mvpMapPoints[i] = NULL;
        L.mvbOutlier[i] = last_outlier[i] != 0;
        if (last_has_mp[i]) { L.mvpMapPoints[i] = new_map_point(last_world + 3 * (size_t)i); idx[L.mvpMapPoints[i]] = i; }
    }
    std::vector<int> pre(cur_mp_inout, cur_mp_inout + C.N);
    for (int i = 0; i < C.N; i++) C.mvpMapPoints[i] = pre[i] >= 0 ? new_map_point(NULL) : NULL;
    C.mTcw = pose_from(Tcw12);
    ORBmatcher matcher(nnratio, check_orientation != 0);
    const int n = matcher.SearchByProjection(C, L, th);
    for (int i = 0; i < C.N; i++) cur_mp_inout[i] = pre[i] >= 0 ? pre[i] : index_of(idx, C.mvpMapPoints[i]);
    return n;
}

// ---- M7: WindowSearch, ORBmatcher.cc:409-516 ----------------------------------------------------------------------------
int ref_window_search(void *f1, void *f2, const uint8_t *f1_has_mp, int window, int min_level, int max_level, float nnratio,
                      int check_orientation, int *match21_out) {
    Frame &F1 = *static_cast<Frame *>(f1), &F2 = *static_cast<Frame *>(f2);
    std::map<MapPoint *, int> idx;
    static const float zero[3] = {0, 0, 0};
    for (int i = 0; i < F1.N; i++) {
        F1.mvpMapPoints[i] = f1_has_mp[i] ? new_map_point(zero) : NULL;
        if (F1.mvpMapPoints[i]) idx[F1.mvpMapPoints[i]] = i;
    }
    std::vector<MapPoint *> m2;
    ORBmatcher matcher(nnratio, check_orientation != 0);
    const int n = matcher.WindowSearch(F1, F2, window, m2, min_level, max_level);
    for (int i = 0; i < F2.N; i++) match21_out[i] = index_of(idx, i < (int)m2.size() ? m2[i] : NULL);
    return n;
}

// ---- M8: SearchForInitialization, ORBmatcher.cc:598-713 -------------------------------------------------------------
int ref_search_for_initialization(void *f1, void *f2, float *prev_matched /*2 x N1, in/out*/, int window, float nnratio,
                                  int check_orientation, int *match12_out) {
    Frame &F1 = *static_cast<Frame *>(f1), &F2 = *static_cast<Frame *>(f2);
    std::vector<cv::Point2f> prev(F1.N);
    for (int i = 0; i < F1.N; i++) prev[i] = cv::Point2f(prev_matched[2 * i], prev_matched[2 * i + 1]);
    std::vector<int> m12;
    ORBmatcher matcher(nnratio, check_orientation != 0);
    const int n = matcher.SearchForInitialization(F1, F2, prev, m12, window);
    for (int i = 0; i < F1.N; i++) {
        match12_out[i] = i < (int)m12.size() ? m12[i] : -1;
        prev_matched[2 * i] = prev[i].x;
        prev_matched[2 * i + 1] = prev[i].y;
    }
    return n;
}

// ---- M3: SearchByProjection(Frame &F, const vector<MapPoint*>&, th), ORBmatcher.cc:49-125 --------------------------------
// f_mp_inout[i]: -1 free, >= 0 occupied; on return the index of the map point assigned to feature i
int ref_search_local_points(void *f, int npts, const uint8_t *in_view, const float *proj_xy, const int *level, const float *view_cos,
                            const uint8_t *desc, float th, float nnratio, int *f_mp_inout) {
    Frame &F = *static_cast<Frame *>(f);
    std::vector<MapPoint *> pts(npts);
    std::map<MapPoint *, int> idx;
    for (int i = 0; i < npts; i++) {
        MapPoint *p = new_map_point(NULL);
        p->mbTrackInView = in_view[i] != 0;
        p->mTrackProjX = proj_xy[2 * i];
        p->mTrackProjY = proj_xy[2 * i + 1];
        p->mnTrackScaleLevel = level[i];
        p->mTrackViewCos = view_cos[i];
        p->mDescriptor = desc_row(desc + (size_t)i * 32);
        pts[i] = p;
        idx[p] = i;
    }
    std::vector<int> pre(f_mp_inout, f_mp_inout + F.N);
    for (int i = 0; i < F.N; i++) F.mvpMapPoints[i] = pre[i] >= 0 ? new_map_point(NULL) : NULL;
    ORBmatcher matcher(nnratio, true);
    const int n = matcher.SearchByProjection(F, pts, th);
    for (int i = 0; i < F.N; i++) f_mp_inout[i] = pre[i] >= 0 ? pre[i] : index_of(idx, F.mvpMapPoints[i]);
    return n;
}

// ---- M6: SearchByProjection(Frame &F1, Frame &F2, int windowSize, vector<MapPoint*>&), ORBmatcher.cc:519-594 -------------
// valid1[i]: F1 feature i has a (good) map point at world1[3i..]; f2_mp_inout as above (the vpMapPointMatches2 vector)
int ref_search_by_projection_f1f2(void *f1, void *f2, const uint8_t *valid1, const float *world1, const float *Tc2w12, int window,
                                  float nnratio, int *f2_mp_inout) {
    Frame &F1 = *static_cast<Frame *>(f1), &F2 = *static_cast<Frame *>(f2);
    std::map<MapPoint *, int> idx;
    for (int i = 0; i < F1.N; i++) {
        F1.mvpMapPoints[i] = valid1[i] ? new_map_point(world1 + 3 * (size_t)i) : NULL;
        if (F1.mvpMapPoints[i]) idx[F1.mvpMapPoints[i]] = i;
    }
    F2.mTcw = pose_from(Tc2w12);
    std::vector<int> pre(f2_mp_inout, f2_mp_inout + F2.N);
    // the method starts with vpMapPointMatches2 = F2.mvpMapPoints (:521): occupancy comes from the frame, not from the argument
    for (int i = 0; i < F2.N; i++) F2.mvpMapPoints[i] = pre[i] >= 0 ? new_map_point(NULL) : NULL;
    std::vector<MapPoint *> m2;
    ORBmatcher matcher(nnratio, true);
    const int n = matcher.SearchByProjection(F1, F2, window, m2);
    for (int i = 0; i < F2.N; i++) f2_mp_inout[i] = pre[i] >= 0 ? pre[i] : index_of(idx, m2[i]);
    return n;
}

// ---- M1 -----------------------------------------------------------------------------------------------------------------
int ref_descriptor_distance(const uint8_t *a, const uint8_t *b) {
    return ORBmatcher::DescriptorDistance(desc_row(a), desc_row(b));
}

}  // extern "C"

// =====================================================================================================================
// KeyFrame-level scenes: keyframes with poses, map points with observations, FeatureVectors -- composed from Python, then
// the KeyFrame-level matchers (M4, M5, M9-M12) run on them.  Map points and keyframes are addressed by their index in
// the driver's lists (deterministic for a given call sequence, so the same script gives the same ids in both builds).
// =====================================================================================================================
namespace {
MapPoint *mp_at(int id) { return id < 0 ? NULL : world().mps[(size_t)id]; }
KeyFrame *kf_at(int id) { return world().kfs[(size_t)id]; }
int mp_id(MapPoint *p) {
    if (!p) return -1;
    World &w = world();
    for (size_t i = w.mps.size(); i-- > 0;) if (w.mps[i] == p) return (int)i;
    return -2;
}
DBoW2::FeatureVector feature_vector(int nn, const int *ids, const int *ptr, const int *items) {
    DBoW2::FeatureVector fv;
    for (int k = 0; k < nn; k++)
        for (int j = ptr[k]; j < ptr[k + 1]; j++) fv.addFeature((DBoW2::NodeId)ids[k], (unsigned int)items[j]);
    return fv;
}
cv::Mat mat_from(const float *v, int r, int c) {
    cv::Mat m(r, c, CV_32F);
    for (int i = 0; i < r; i++) for (int j = 0; j < c; j++) m.at<float>(i, j) = v[i * c + j];
    return m;
}
}  // namespace

extern "C" {

int ref_world_counts(int *n_mps, int *n_kfs) { *n_mps = (int)world().mps.size(); *n_kfs = (int)world().kfs.size(); return 0; }

void ref_frame_set_pose(void *f, const float *Tcw12) { static_cast<Frame *>(f)->mTcw = pose_from(Tcw12); }
void ref_frame_set_feature_vector(void *f, int nn, const int *ids, const int *ptr, const int *items) {
    static_cast<Frame *>(f)->mFeatVec = feature_vector(nn, ids, ptr, items);
}
// Frame::mvpMapPoints from map-point ids (-1 = NULL)
void ref_frame_set_map_points(void *f, const int *ids) {
    Frame &F = *static_cast<Frame *>(f);
    for (int i = 0; i < F.N; i++) F.mvpMapPoints[i] = mp_at(ids[i]);
}
void ref_frame_get_map_points(void *f, int *ids) {
    Frame &F = *static_cast<Frame *>(f);
    for (int i = 0; i < F.N; i++) ids[i] = mp_id(F.mvpMapPoints[i]);
}

// KeyFrame(Frame &F, Map*, KeyFrameDatabase*) with F.mTcw = Tcw (KeyFrame.cc:30-53); returns the keyframe id
int ref_kf_create(void *f, const float *Tcw12) {
    Frame &F = *static_cast<Frame *>(f);
    F.mTcw = pose_from(Tcw12);
    World &w = world();
    std::vector<MapPoint *> keep = F.mvpMapPoints;
    F.mvpMapPoints = std::vector<MapPoint *>(F.N, static_cast<MapPoint *>(NULL));   // map points are attached explicitly below
    KeyFrame *kf = new (arena_alloc(sizeof(KeyFrame))) KeyFrame(F, &w.map, &w.db);
    F.mvpMapPoints = keep;
    w.kfs.push_back(kf);
    return (int)w.kfs.size() - 1;
}
void ref_kf_set_feature_vector(int kf, int nn, const int *ids, const int *ptr, const int *items) {
    kf_at(kf)->mFeatVec = feature_vector(nn, ids, ptr, items);
}

// a map point with everything the matchers read: position, representative descriptor (MapPoint::GetDescriptor), mean
// viewing direction (GetNormal) and the scale-invariance distance range (GetMin/MaxDistanceInvariance)
int ref_mp_create(const float *world3, const uint8_t *desc32, const float *normal3, float min_dist, float max_dist, int ref_kf) {
    MapPoint *p = new_map_point(world3, ref_kf >= 0 ? kf_at(ref_kf) : NULL);
    if (desc32) p->mDescriptor = desc_row(desc32);
    if (normal3) p->mNormalVector = point3(normal3);
    p->mfMinDistance = min_dist;
    p->mfMaxDistance = max_dist;
    return (int)world().mps.size() - 1;
}
void ref_mp_set_bad(int mp) { mp_at(mp)->mbBad = true; }
// observation both ways, as LocalMapping does (pKF->AddMapPoint + pMP->AddObservation)
void ref_kf_add_map_point(int kf, int mp, int idx) {
    kf_at(kf)->AddMapPoint(mp_at(mp), (size_t)idx);
    mp_at(mp)->AddObservation(kf_at(kf), (size_t)idx);
}
void ref_kf_get_map_points(int kf, int *ids /*N*/) {
    const std::vector<MapPoint *> v = kf_at(kf)->GetMapPointMatches();
    for (size_t i = 0; i < v.size(); i++) ids[i] = mp_id(v[i]);
}
int ref_kf_n(int kf) { return (int)kf_at(kf)->GetMapPointMatches().size(); }
// state of a map point after a mutating call: bad flag, number of observations, and (keyframe id, feature index) pairs
int ref_mp_state(int mp, int *is_bad, int *obs_kf /*cap*/, int *obs_idx /*cap*/, int cap) {
    MapPoint *p = mp_at(mp);
    *is_bad = p->isBad() ? 1 : 0;
    const std::map<KeyFrame *, size_t> obs = p->GetObservations();
    World &w = world();
    std::vector<std::pair<int, int> > out;
    for (std::map<KeyFrame *, size_t>::const_iterator it = obs.begin(); it != obs.end(); ++it) {
        int kid = -1;
        for (size_t k = 0; k < w.kfs.size(); k++) if (w.kfs[k] == it->first) kid = (int)k;
        out.push_back(std::make_pair(kid, (int)it->second));
    }
    std::sort(out.begin(), out.end());   // the std::map is ordered by pointer value: report in keyframe-id order
    for (size_t k = 0; k < out.size() && (int)k < cap; k++) { obs_kf[k] = out[k].first; obs_idx[k] = out[k].second; }
    return (int)out.size();
}

// ---- M4: SearchByProjection(Frame &CurrentFrame, KeyFrame *pKF, const set<MapPoint*> &sAlreadyFound, th, ORBdist), :1622-1746
int ref_search_by_projection_frame_kf(void *cur, int kf, const int *already_found, int n_found, float th, int orb_dist, float nnratio,
                                      int check_orientation, int *cur_mp_ids_inout) {
    Frame &C = *static_cast<Frame *>(cur);
    for (int i = 0; i < C.N; i++) C.mvpMapPoints[i] = mp_at(cur_mp_ids_inout[i]);
    std::set<MapPoint *> found;
    for (int k = 0; k < n_found; k++) found.insert(mp_at(already_found[k]));
    ORBmatcher matcher(nnratio, check_orientation != 0);
    const int n = matcher.SearchByProjection(C, kf_at(kf), found, th, orb_dist);
    for (int i = 0; i < C.N; i++) cur_mp_ids_inout[i] = mp_id(C.mvpMapPoints[i]);
    return n;
}

// ---- M5: SearchByProjection(KeyFrame* pKF, cv::Mat Scw, const vector<MapPoint*> &vpPoints, vector<MapPoint*> &vpMatched, int th), :286-407
int ref_search_by_projection_sim3(int kf, const float *Scw16, const int *points, int npts, int *matched_ids_inout, int th, float nnratio) {
    KeyFrame *K = kf_at(kf);
    std::vector<MapPoint *> pts(npts), matched(K->GetMapPointMatches().size());
    for (int i = 0; i < npts; i++) pts[i] = mp_at(points[i]);
    for (size_t i = 0; i < matched.size(); i++) matched[i] = mp_at(matched_ids_inout[i]);
    ORBmatcher matcher(nnratio, true);
    const int n = matcher.SearchByProjection(K, mat_from(Scw16, 4, 4), pts, matched, th);
    for (size_t i = 0; i < matched.size(); i++) matched_ids_inout[i] = mp_id(matched[i]);
    return n;
}

// ---- M9: SearchByBoW(KeyFrame*, Frame&, vector<MapPoint*>&) :155-284 and SearchByBoW(KeyFrame*, KeyFrame*, vector<MapPoint*>&) :715-850
int ref_search_by_bow_kf_frame(int kf, void *f, float nnratio, int check_orientation, int *out_ids /*F.N*/) {
    Frame &F = *static_cast<Frame *>(f);
    std::vector<MapPoint *> m;
    ORBmatcher matcher(nnratio, check_orientation != 0);
    const int n = matcher.SearchByBoW(kf_at(kf), F, m);
    for (int i = 0; i < F.N; i++) out_ids[i] = mp_id(i < (int)m.size() ? m[i] : NULL);
    return n;
}
int ref_search_by_bow_kf_kf(int kf1, int kf2, float nnratio, int check_orientation, int *out_ids /*N1*/) {
    std::vector<MapPoint *> m;
    ORBmatcher matcher(nnratio, check_orientation != 0);
    const int n = matcher.SearchByBoW(kf_at(kf1), kf_at(kf2), m);
    for (size_t i = 0; i < m.size(); i++) out_ids[i] = mp_id(m[i]);
    return n;
}

// ---- M10: SearchForTriangulation :852-1014 -------------------------------------------------------------------------
int ref_search_for_triangulation(int kf1, int kf2, const float *F12_9, float nnratio, int check_orientation, int *pairs /*2 x cap*/, int cap) {
    std::vector<cv::KeyPoint> k1, k2;
    std::vector<std::pair<size_t, size_t> > pr;
    ORBmatcher matcher(nnratio, check_orientation != 0);
    const int n = matcher.SearchForTriangulation(kf_at(kf1), kf_at(kf2), mat_from(F12_9, 3, 3), k1, k2, pr);
    for (size_t i = 0; i < pr.size() && (int)i < cap; i++) { pairs[2 * i] = (int)pr[i].first; pairs[2 * i + 1] = (int)pr[i].second; }
    return n;
}

// ---- M11: SearchBySim3 :1267-1505 ----------------------------------------------------------------------------------
int ref_search_by_sim3(int kf1, int kf2, int *matches12_ids_inout /*N1*/, float s12, const float *R12_9, const float *t12_3, float th) {
    KeyFrame *K1 = kf_at(kf1);
    std::vector<MapPoint *> m(K1->GetMapPointMatches().size());
    for (size_t i = 0; i < m.size(); i++) m[i] = mp_at(matches12_ids_inout[i]);
    ORBmatcher matcher(0.9f, true);
    const int n = matcher.SearchBySim3(K1, kf_at(kf2), m, s12, mat_from(R12_9, 3, 3), mat_from(t12_3, 3, 1), th);
    for (size_t i = 0; i < m.size(); i++) matches12_ids_inout[i] = mp_id(m[i]);
    return n;
}

// ---- M12: Fuse(KeyFrame*, vector<MapPoint*>&, th) :1016-1134 and Fuse(KeyFrame*, cv::Mat Scw, const vector<MapPoint*>&, th) :1136-1265
int ref_fuse(int kf, const int *points, int npts, float th) {
    std::vector<MapPoint *> pts(npts);
    for (int i = 0; i < npts; i++) pts[i] = mp_at(points[i]);
    ORBmatcher matcher(0.6f, true);
    return matcher.Fuse(kf_at(kf), pts, th);
}
int ref_fuse_sim3(int kf, const float *Scw16, const int *points, int npts, float th) {
    std::vector<MapPoint *> pts(npts);
    for (int i = 0; i < npts; i++) pts[i] = mp_at(points[i]);
    ORBmatcher matcher(0.6f, true);
    return matcher.Fuse(kf_at(kf), mat_from(Scw16, 4, 4), pts, th);
}

// ---- N4: MapPoint::ComputeDistinctiveDescriptors (MapPoint.cc:185-250) on the map point's observations ----------------
void ref_mp_compute_distinctive(int mp, uint8_t *desc_out) {
    MapPoint *p = mp_at(mp);
    p->ComputeDistinctiveDescriptors();
    cv::Mat d = p->GetDescriptor();
    std::memcpy(desc_out, d.ptr(0), 32);
}

}  // extern "C"

// =====================================================================================================================
// N2 / N3: the reference's vocabulary (Thirdparty/DBoW2 TemplatedVocabulary, loaded from the text format of
// Data/ORBvoc.txt) and its KeyFrameDatabase (src/KeyFrameDatabase.cc)
// =====================================================================================================================
namespace {
struct VocDb {
    ORBVocabulary voc;
    KeyFrameDatabase *db;
    std::vector<KeyFrame *> kfs;
    VocDb() : db(NULL) {}
};
KeyFrame *bare_keyframe() {
    World &w = world();
    Frame *F = frame_from_arrays(NULL, NULL, 0, 64, 48, 50.f, 50.f, 32.f, 24.f, 1.2f, 8);
    KeyFrame *kf = new (arena_alloc(sizeof(KeyFrame))) KeyFrame(*F, &w.map, &w.db);
    delete F;
    return kf;
}
DBoW2::BowVector bow_from(const int *ids, const double *vals, int n) {
    DBoW2::BowVector v;
    for (int i = 0; i < n; i++) v.addWeight((DBoW2::WordId)ids[i], vals[i]);
    return v;
}
}  // namespace

extern "C" {

void *ref_voc_load(const char *text_path) {
    VocDb *V = new VocDb();
    if (!V->voc.loadFromTextFile(text_path)) { delete V; return NULL; }
    V->db = new KeyFrameDatabase(V->voc);
    return V;
}
int ref_voc_words(void *v) { return (int)static_cast<VocDb *>(v)->voc.size(); }

// Frame::ComputeBoW / KeyFrame::ComputeBoW: mpORBvocabulary->transform(vCurrentDesc, mBowVec, mFeatVec, 4) (Frame.cc:280-287)
// outputs: BowVector as (word id, value) in map order; FeatureVector as CSR (node id, ptr, feature indices)
int ref_bow_transform(void *v, const uint8_t *desc, int n, int levelsup, int *nwords_out, int *bow_ids, double *bow_vals, int *nnodes_out,
                      int *fv_ids, int *fv_ptr, int *fv_feats) {
    VocDb *V = static_cast<VocDb *>(v);
    cv::Mat D(std::max(n, 1), 32, CV_8UC1);
    if (n) std::memcpy(D.data, desc, (size_t)n * 32);
    std::vector<cv::Mat> rows;
    for (int i = 0; i < n; i++) rows.push_back(D.row(i));
    DBoW2::BowVector bv;
    DBoW2::FeatureVector fv;
    V->voc.transform(rows, bv, fv, levelsup);
    int k = 0;
    for (DBoW2::BowVector::const_iterator it = bv.begin(); it != bv.end(); ++it, ++k) { bow_ids[k] = (int)it->first; bow_vals[k] = it->second; }
    *nwords_out = k;
    int nn = 0, o = 0;
    fv_ptr[0] = 0;
    for (DBoW2::FeatureVector::const_iterator it = fv.begin(); it != fv.end(); ++it, ++nn) {
        fv_ids[nn] = (int)it->first;
        for (size_t j = 0; j < it->second.size(); j++) fv_feats[o++] = (int)it->second[j];
        fv_ptr[nn + 1] = o;
    }
    *nnodes_out = nn;
    return 0;
}

// keyframe `k` of the database = the k-th ref_db_add call: BowVector given, KeyFrameDatabase::add (KeyFrameDatabase.cc:37-44)
int ref_db_add(void *v, const int *ids, const double *vals, int n) {
    VocDb *V = static_cast<VocDb *>(v);
    KeyFrame *kf = bare_keyframe();
    kf->mBowVec = bow_from(ids, vals, n);
    V->db->add(kf);
    V->kfs.push_back(kf);
    return (int)V->kfs.size() - 1;
}
// GetBestCovisibilityKeyFrames(10) of keyframe k returns `others` in this order (strictly decreasing weights)
void ref_db_set_covisibles(void *v, int k, const int *others, int n) {
    VocDb *V = static_cast<VocDb *>(v);
    for (int i = 0; i < n; i++) V->kfs[k]->AddConnection(V->kfs[others[i]], 1000 - i);
}
// DetectLoopCandidates(pKF, minScore) (KeyFrameDatabase.cc:72-204) for a fresh query keyframe connected to `connected`
int ref_db_detect_loop(void *v, const int *q_ids, const double *q_vals, int nq, const int *connected, int nconn, float min_score, int *out, int cap) {
    VocDb *V = static_cast<VocDb *>(v);
    KeyFrame *q = bare_keyframe();
    q->mBowVec = bow_from(q_ids, q_vals, nq);
    for (int i = 0; i < nconn; i++) q->AddConnection(V->kfs[connected[i]], 100);
    const std::vector<KeyFrame *> c = V->db->DetectLoopCandidates(q, min_score);
    for (size_t i = 0; i < c.size() && (int)i < cap; i++) {
        out[i] = -1;
        for (size_t k = 0; k < V->kfs.size(); k++) if (V->kfs[k] == c[i]) out[i] = (int)k;
    }
    return (int)c.size();
}
// DetectRelocalisationCandidates(Frame *F) (KeyFrameDatabase.cc:206-308)
int ref_db_detect_reloc(void *v, const int *q_ids, const double *q_vals, int nq, int *out, int cap) {
    VocDb *V = static_cast<VocDb *>(v);
    Frame *F = frame_from_arrays(NULL, NULL, 0, 64, 48, 50.f, 50.f, 32.f, 24.f, 1.2f, 8);
    F->mBowVec = bow_from(q_ids, q_vals, nq);
    const std::vector<KeyFrame *> c = V->db->DetectRelocalisationCandidates(F);
    for (size_t i = 0; i < c.size() && (int)i < cap; i++) {
        out[i] = -1;
        for (size_t k = 0; k < V->kfs.size(); k++) if (V->kfs[k] == c[i]) out[i] = (int)k;
    }
    delete F;
    return (int)c.size();
}

}  // extern "C"

// N4 helper: the keyframes observing a map point in the ITERATION order of its std::map<KeyFrame*, size_t> (pointer order --
// the order MapPoint::ComputeDistinctiveDescriptors collects the descriptors in, MapPoint.cc:204-210), as (keyframe id, index)
extern "C" int ref_mp_observation_order(int mp, int *obs_kf, int *obs_idx, int cap) {
    MapPoint *p = mp_at(mp);
    const std::map<KeyFrame *, size_t> obs = p->GetObservations();
    World &w = world();
    int n = 0;
    for (std::map<KeyFrame *, size_t>::const_iterator it = obs.begin(); it != obs.end(); ++it, ++n) {
        if (n >= cap) continue;
        obs_kf[n] = -1;
        for (size_t k = 0; k < w.kfs.size(); k++) if (w.kfs[k] == it->first) obs_kf[n] = (int)k;
        obs_idx[n] = (int)it->second;
    }
    return n;
}

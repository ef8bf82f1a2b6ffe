"""ctypes binding of oracle/_ref/libref_orbslam.so (and libfacade_orbslam.so): the reference's OWN sources
(/root/reference/src/ORBextractor.cc, ORBmatcher.cc, Frame.cc, KeyFrame.cc, MapPoint.cc, Map.cc, KeyFrameDatabase.cc,
Thirdparty/DBoW2) compiled unmodified against the stand-in headers of oracle/ref_shim/ (recipe: oracle/Makefile, `make ref`).

TEST INFRASTRUCTURE ONLY (like everything under oracle/): used by tests/ to validate the oracle restatement against the
reference's real control flow, and optionally by bench.py's CPU arm.  /root/reference does not exist on the GPU box: there
the prebuilt library travels with the snapshot and `available()` only reports whether it can be loaded."""
import ctypes as C
import os
import subprocess

import numpy as np

from . import KP_DTYPE

_HERE = os.path.dirname(os.path.abspath(__file__))
_DIR = os.path.join(_HERE, "_ref")
REFERENCE_ROOT = os.environ.get("ORB_REFERENCE_ROOT", "/root/reference")
_libs = {}


def build(force=False):
    """Build oracle/_ref/*.so from the reference sources when they are present (this container); otherwise keep what is there."""
    if os.path.isdir(os.path.join(REFERENCE_ROOT, "src")):
        from . import build as build_oracle
        build_oracle()
        if force:
            subprocess.call(["rm", "-rf", _DIR])
        subprocess.check_call(["make", "-C", _HERE, "-s", "ref", "REF=" + REFERENCE_ROOT], env={**os.environ, "CC": "gcc", "CXX": "g++"})
    return os.path.join(_DIR, "libref_orbslam.so")


def shim_lib():
    """oracle/libref_shim.so: the stand-in cv:: layer of ref_shim/ on its own (no reference source needed), with the
    ref_shim_gemm / ref_shim_norm self-test hooks."""
    if "shim" not in _libs:
        from . import build as build_oracle
        build_oracle()
        subprocess.check_call(["make", "-C", _HERE, "-s", "shim"], env={**os.environ, "CC": "gcc", "CXX": "g++"})
        L = C.CDLL(os.path.join(_HERE, "libref_shim.so"), mode=os.RTLD_NOW | os.RTLD_LOCAL)
        L.ref_shim_gemm.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_double, C.c_void_p, C.c_double,
                                    C.c_int, C.c_void_p]
        L.ref_shim_gemm.restype = None
        L.ref_shim_norm.argtypes = [C.c_void_p, C.c_int]
        L.ref_shim_norm.restype = C.c_double
        _libs["shim"] = L
    return _libs["shim"]


def available(which="ref"):
    return os.path.exists(os.path.join(_DIR, "lib%s_orbslam.so" % which))


def lib(which="ref"):
    """which = "ref" (reference ORBextractor.cc / ORBmatcher.cc) or "facade" (the product's facades over liborbfe.so)."""
    if which in _libs:
        return _libs[which]
    path = os.path.join(_DIR, "lib%s_orbslam.so" % which)
    if not os.path.exists(path):
        build()
    L = C.CDLL(path, mode=os.RTLD_NOW | os.RTLD_LOCAL)
    vp, f, i = C.c_void_p, C.c_float, C.c_int
    L.ref_extract.argtypes = [i, f, i, i, i, vp, i, i, C.c_size_t, vp, vp, i]
    L.ref_frame_from_image.argtypes = [vp, i, i, C.c_size_t, f, f, f, f, vp, i, f, i, i, i]
    L.ref_frame_from_image.restype = vp
    L.ref_frame_from_arrays.argtypes = [vp, vp, i, i, i, f, f, f, f, f, i]
    L.ref_frame_from_arrays.restype = vp
    L.ref_frame_free.argtypes = [vp]
    L.ref_frame_n.argtypes = [vp]
    L.ref_frame_get.argtypes = [vp, vp, vp, vp, vp, vp]
    L.ref_frame_grid.argtypes = [vp, vp, vp]
    L.ref_frame_features_in_area.argtypes = [vp, f, f, f, i, i, vp, i]
    L.ref_search_by_projection_ff.argtypes = [vp, vp, vp, vp, vp, vp, f, f, i, vp]
    L.ref_window_search.argtypes = [vp, vp, vp, i, i, i, f, i, vp]
    L.ref_search_for_initialization.argtypes = [vp, vp, vp, i, f, i, vp]
    L.ref_search_local_points.argtypes = [vp, i, vp, vp, vp, vp, vp, f, f, vp]
    L.ref_search_by_projection_f1f2.argtypes = [vp, vp, vp, vp, vp, i, f, vp]
    L.ref_descriptor_distance.argtypes = [vp, vp]
    _libs[which] = L
    return L


def _p(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def extract(img, nfeatures=1000, scale_factor=1.2, nlevels=8, score_type=1, fast_th=20, which="ref"):
    """ORB_SLAM::ORBextractor(...)(img, cv::Mat(), keys, desc) of the reference build."""
    img = np.ascontiguousarray(img, np.uint8)
    H, W = img.shape
    cap = max(2 * nfeatures, 16)
    kps = np.zeros(cap, KP_DTYPE)
    desc = np.zeros((cap, 32), np.uint8)
    n = lib(which).ref_extract(nfeatures, scale_factor, nlevels, score_type, fast_th, _p(img), W, H, img.strides[0], _p(kps), _p(desc), cap)
    assert n <= cap
    return kps[:n].copy(), desc[:n].copy()


class RefFrame:
    """A real ORB_SLAM::Frame.  from_image runs the reference constructor (Frame.cc:56-125); from_arrays fills the public
    members from given keypoints (zero distortion) and bins them with the reference's own Frame::PosInGrid."""

    def __init__(self, handle, which):
        self.h, self.which = handle, which
        self.n = lib(which).ref_frame_n(handle)

    @classmethod
    def from_image(cls, img, fx, fy, cx, cy, dist4=None, nfeatures=1000, scale_factor=1.2, nlevels=8, score_type=1, fast_th=20, which="ref"):
        img = np.ascontiguousarray(img, np.uint8)
        H, W = img.shape
        d = None if dist4 is None else np.ascontiguousarray(dist4, np.float32)
        return cls(lib(which).ref_frame_from_image(_p(img), W, H, img.strides[0], fx, fy, cx, cy, _p(d), nfeatures, scale_factor, nlevels,
                                                   score_type, fast_th), which)

    @classmethod
    def from_arrays(cls, kps, desc, W, H, fx=500.0, fy=500.0, cx=None, cy=None, scale_factor=1.2, nlevels=8, which="ref"):
        kps = np.ascontiguousarray(kps, KP_DTYPE)
        desc = np.ascontiguousarray(desc, np.uint8).reshape(-1, 32)
        cx = W / 2.0 if cx is None else cx
        cy = H / 2.0 if cy is None else cy
        return cls(lib(which).ref_frame_from_arrays(_p(kps), _p(desc), len(kps), W, H, fx, fy, cx, cy, scale_factor, nlevels), which)

    def get(self):
        keys, keys_un = np.zeros(self.n, KP_DTYPE), np.zeros(self.n, KP_DTYPE)
        desc = np.zeros((self.n, 32), np.uint8)
        bounds, ginv = np.zeros(4, np.float32), np.zeros(2, np.float32)
        lib(self.which).ref_frame_get(self.h, _p(keys), _p(keys_un), _p(desc), _p(bounds), _p(ginv))
        return keys, keys_un, desc, bounds, ginv

    def grid(self):
        start, items = np.zeros(64 * 48 + 1, np.int32), np.zeros(max(self.n, 1), np.int32)
        lib(self.which).ref_frame_grid(self.h, _p(start), _p(items))
        return start, items[:start[-1]]

    def features_in_area(self, x, y, r, min_level=-1, max_level=-1):
        out = np.zeros(max(self.n, 1), np.int32)
        n = lib(self.which).ref_frame_features_in_area(self.h, x, y, r, min_level, max_level, _p(out), self.n)
        return out[:n].copy()

    def close(self):
        if self.h:
            lib(self.which).ref_frame_free(self.h)
            self.h = None


def search_by_projection_ff(cur, last, last_has_mp, last_outlier, last_world, Tcw, th, nnratio=0.9, check_orientation=True, cur_mp=None):
    mp = np.full(cur.n, -1, np.int32) if cur_mp is None else np.ascontiguousarray(cur_mp, np.int32).copy()
    has, outl = np.ascontiguousarray(last_has_mp, np.uint8), np.ascontiguousarray(last_outlier, np.uint8)
    world, T = np.ascontiguousarray(last_world, np.float32), np.ascontiguousarray(Tcw, np.float32)
    n = lib(cur.which).ref_search_by_projection_ff(cur.h, last.h, _p(has), _p(outl), _p(world), _p(T), th, nnratio, int(check_orientation), _p(mp))
    return n, mp


def window_search(f1, f2, f1_has_mp, window, min_level=-1, max_level=2 ** 31 - 1, nnratio=0.6, check_orientation=True):
    has = np.ascontiguousarray(f1_has_mp, np.uint8)
    m21 = np.full(max(f2.n, 1), -1, np.int32)
    n = lib(f1.which).ref_window_search(f1.h, f2.h, _p(has), window, min_level, max_level, nnratio, int(check_orientation), _p(m21))
    return n, m21[:f2.n]


def search_for_initialization(f1, f2, prev_matched, window, nnratio=0.9, check_orientation=True):
    prev = np.ascontiguousarray(prev_matched, np.float32).copy()
    m12 = np.full(max(f1.n, 1), -1, np.int32)
    n = lib(f1.which).ref_search_for_initialization(f1.h, f2.h, _p(prev), window, nnratio, int(check_orientation), _p(m12))
    return n, m12[:f1.n], prev


def search_local_points(f, in_view, proj_xy, level, view_cos, desc, th, nnratio=0.8, f_mp=None):
    mp = np.full(f.n, -1, np.int32) if f_mp is None else np.ascontiguousarray(f_mp, np.int32).copy()
    iv, pxy = np.ascontiguousarray(in_view, np.uint8), np.ascontiguousarray(proj_xy, np.float32)
    lv, vc, d = np.ascontiguousarray(level, np.int32), np.ascontiguousarray(view_cos, np.float32), np.ascontiguousarray(desc, np.uint8)
    n = lib(f.which).ref_search_local_points(f.h, len(iv), _p(iv), _p(pxy), _p(lv), _p(vc), _p(d), th, nnratio, _p(mp))
    return n, mp


def search_by_projection_f1f2(f1, f2, valid1, world1, Tc2w, window, nnratio=0.9, f2_mp=None):
    mp = np.full(f2.n, -1, np.int32) if f2_mp is None else np.ascontiguousarray(f2_mp, np.int32).copy()
    v, w, T = np.ascontiguousarray(valid1, np.uint8), np.ascontiguousarray(world1, np.float32), np.ascontiguousarray(Tc2w, np.float32)
    n = lib(f1.which).ref_search_by_projection_f1f2(f1.h, f2.h, _p(v), _p(w), _p(T), window, nnratio, _p(mp))
    return n, mp


def descriptor_distance(a, b, which="ref"):
    a, b = np.ascontiguousarray(a, np.uint8), np.ascontiguousarray(b, np.uint8)
    return lib(which).ref_descriptor_distance(_p(a), _p(b))


# ---- KeyFrame-level scenes (M4, M5, M9-M12, N4): thin wrappers over the id-based driver API ------------------------------
def _bind_scene(L):
    if getattr(L, "_scene_bound", False):
        return L
    vp, f, i = C.c_void_p, C.c_float, C.c_int
    L.ref_frame_set_pose.argtypes = [vp, vp]
    L.ref_frame_set_feature_vector.argtypes = [vp, i, vp, vp, vp]
    L.ref_frame_set_map_points.argtypes = [vp, vp]
    L.ref_frame_get_map_points.argtypes = [vp, vp]
    L.ref_kf_create.argtypes = [vp, vp]
    L.ref_kf_set_feature_vector.argtypes = [i, i, vp, vp, vp]
    L.ref_mp_create.argtypes = [vp, vp, vp, f, f, i]
    L.ref_mp_set_bad.argtypes = [i]
    L.ref_kf_add_map_point.argtypes = [i, i, i]
    L.ref_kf_get_map_points.argtypes = [i, vp]
    L.ref_kf_n.argtypes = [i]
    L.ref_mp_state.argtypes = [i, vp, vp, vp, i]
    L.ref_search_by_projection_frame_kf.argtypes = [vp, i, vp, i, f, i, f, i, vp]
    L.ref_search_by_projection_sim3.argtypes = [i, vp, vp, i, vp, i, f]
    L.ref_search_by_bow_kf_frame.argtypes = [i, vp, f, i, vp]
    L.ref_search_by_bow_kf_kf.argtypes = [i, i, f, i, vp]
    L.ref_search_for_triangulation.argtypes = [i, i, vp, f, i, vp, i]
    L.ref_search_by_sim3.argtypes = [i, i, vp, f, vp, vp, f]
    L.ref_fuse.argtypes = [i, vp, i, f]
    L.ref_fuse_sim3.argtypes = [i, vp, vp, i, f]
    L.ref_mp_compute_distinctive.argtypes = [i, vp]
    L.ref_world_counts.argtypes = [vp, vp]
    L._scene_bound = True
    return L


def _i32(a):
    return np.ascontiguousarray(a, np.int32)


def _f32(a):
    return np.ascontiguousarray(a, np.float32)


class Scene:
    """Composes keyframes / map points in one build ("ref" or "facade") of the reference's map model."""

    def __init__(self, which="ref"):
        self.which = which
        self.L = _bind_scene(lib(which))

    def frame(self, kps, desc, W, H, fx, fy, cx, cy, scale_factor=1.2, nlevels=8):
        return RefFrame.from_arrays(kps, desc, W, H, fx, fy, cx, cy, scale_factor, nlevels, which=self.which)

    def keyframe(self, frame, Tcw):
        T = _f32(Tcw)
        return self.L.ref_kf_create(frame.h, _p(T))

    def set_pose(self, frame, Tcw):
        T = _f32(Tcw)
        self.L.ref_frame_set_pose(frame.h, _p(T))

    def map_point(self, world, desc=None, normal=None, min_dist=0.0, max_dist=0.0, ref_kf=-1):
        w = _f32(world)
        d = None if desc is None else np.ascontiguousarray(desc, np.uint8)
        n = None if normal is None else _f32(normal)
        return self.L.ref_mp_create(_p(w), _p(d), _p(n), float(min_dist), float(max_dist), int(ref_kf))

    def set_bad(self, mp):
        self.L.ref_mp_set_bad(int(mp))

    def observe(self, kf, mp, idx):
        self.L.ref_kf_add_map_point(int(kf), int(mp), int(idx))

    def kf_map_points(self, kf):
        out = np.zeros(max(self.L.ref_kf_n(kf), 1), np.int32)
        self.L.ref_kf_get_map_points(kf, _p(out))
        return out[:self.L.ref_kf_n(kf)]

    def mp_state(self, mp, cap=64):
        bad = C.c_int(0)
        ok, oi = np.zeros(cap, np.int32), np.zeros(cap, np.int32)
        n = self.L.ref_mp_state(int(mp), C.byref(bad), _p(ok), _p(oi), cap)
        return bool(bad.value), [(int(ok[k]), int(oi[k])) for k in range(min(n, cap))]

    def counts(self):
        a, b = C.c_int(0), C.c_int(0)
        self.L.ref_world_counts(C.byref(a), C.byref(b))
        return a.value, b.value

    def set_feature_vector(self, target, fv):
        """target: RefFrame or keyframe id; fv = (node ids, ptr, items) CSR as orb_slam_b200.matching.feature_vector() returns."""
        ids, ptr, items = (_i32(x) for x in fv)
        if isinstance(target, RefFrame):
            self.L.ref_frame_set_feature_vector(target.h, len(ids), _p(ids), _p(ptr), _p(items))
        else:
            self.L.ref_kf_set_feature_vector(int(target), len(ids), _p(ids), _p(ptr), _p(items))

    def frame_map_points(self, frame, ids=None):
        if ids is not None:
            a = _i32(ids)
            self.L.ref_frame_set_map_points(frame.h, _p(a))
            return None
        out = np.zeros(max(frame.n, 1), np.int32)
        self.L.ref_frame_get_map_points(frame.h, _p(out))
        return out[:frame.n]

    # M4
    def search_by_projection_frame_kf(self, cur, kf, already_found, th, orb_dist, nnratio=0.9, check_orientation=True, cur_mp=None):
        mp = np.full(cur.n, -1, np.int32) if cur_mp is None else _i32(cur_mp).copy()
        af = _i32(already_found)
        n = self.L.ref_search_by_projection_frame_kf(cur.h, int(kf), _p(af), len(af), th, int(orb_dist), nnratio, int(check_orientation), _p(mp))
        return n, mp

    # M5
    def search_by_projection_sim3(self, kf, Scw, points, matched, th, nnratio=0.75):
        S, pts, m = _f32(Scw), _i32(points), _i32(matched).copy()
        n = self.L.ref_search_by_projection_sim3(int(kf), _p(S), _p(pts), len(pts), _p(m), int(th), nnratio)
        return n, m

    # M9
    def search_by_bow_kf_frame(self, kf, frame, nnratio=0.75, check_orientation=True):
        out = np.full(max(frame.n, 1), -1, np.int32)
        n = self.L.ref_search_by_bow_kf_frame(int(kf), frame.h, nnratio, int(check_orientation), _p(out))
        return n, out[:frame.n]

    def search_by_bow_kf_kf(self, kf1, kf2, nnratio=0.75, check_orientation=True):
        out = np.full(max(self.L.ref_kf_n(kf1), 1), -1, np.int32)
        n = self.L.ref_search_by_bow_kf_kf(int(kf1), int(kf2), nnratio, int(check_orientation), _p(out))
        return n, out[:self.L.ref_kf_n(kf1)]

    # M10
    def search_for_triangulation(self, kf1, kf2, F12, nnratio=0.6, check_orientation=True):
        F = _f32(F12)
        cap = self.L.ref_kf_n(kf1) + 8
        pairs = np.zeros((cap, 2), np.int32)
        n = self.L.ref_search_for_triangulation(int(kf1), int(kf2), _p(F), nnratio, int(check_orientation), _p(pairs), cap)
        return n, pairs[:min(n, cap)]

    # M11
    def search_by_sim3(self, kf1, kf2, matches12, s12, R12, t12, th):
        m, R_, t_ = _i32(matches12).copy(), _f32(R12), _f32(t12)
        n = self.L.ref_search_by_sim3(int(kf1), int(kf2), _p(m), float(s12), _p(R_), _p(t_), float(th))
        return n, m

    # M12
    def fuse(self, kf, points, th=2.5):
        pts = _i32(points)
        return self.L.ref_fuse(int(kf), _p(pts), len(pts), float(th))

    def fuse_sim3(self, kf, Scw, points, th=2.5):
        S, pts = _f32(Scw), _i32(points)
        return self.L.ref_fuse_sim3(int(kf), _p(S), _p(pts), len(pts), float(th))

    # N4
    def compute_distinctive(self, mp):
        d = np.zeros(32, np.uint8)
        self.L.ref_mp_compute_distinctive(int(mp), _p(d))
        return d


# ---- N2 / N3: the reference's DBoW2 vocabulary and KeyFrameDatabase -----------------------------------------------------
def write_vocabulary_text(voc, path, scoring=0, weighting=0):
    """A synthetic vocabulary (orb_slam_b200.synth.random_vocabulary: nodes in creation order, children consecutive) in the text
    format TemplatedVocabulary::loadFromTextFile reads (Data/ORBvoc.txt: header `k L scoring weighting`, then one line per
    node `parent isLeaf b0 .. b31 weight`): the loader numbers nodes by line and words by leaf order, exactly like the arrays."""
    nd, cp, ch = voc["node_desc"], voc["child_ptr"], voc["children"]
    n = len(nd)
    parent = np.zeros(n, np.int32)
    for i in range(n):
        parent[ch[cp[i]:cp[i + 1]]] = i
    with open(path, "w") as f:
        f.write("%d %d %d %d\n" % (voc["k"], voc["L"], scoring, weighting))
        for i in range(1, n):
            leaf = 1 if cp[i + 1] == cp[i] else 0
            f.write("%d %d %s %r\n" % (parent[i], leaf, " ".join(str(int(b)) for b in nd[i]), float(voc["weight"][i])))
    # loadFromTextFile reads until eof: the file must not end with an empty line that would create a phantom node
    data = open(path).read().rstrip("\n")
    open(path, "w").write(data)


class RefVocabulary:
    def __init__(self, path, which="ref"):
        L = lib(which)
        vp, i = C.c_void_p, C.c_int
        L.ref_voc_load.argtypes = [C.c_char_p]
        L.ref_voc_load.restype = vp
        L.ref_voc_words.argtypes = [vp]
        L.ref_bow_transform.argtypes = [vp, vp, i, i, vp, vp, vp, vp, vp, vp, vp]
        L.ref_db_add.argtypes = [vp, vp, vp, i]
        L.ref_db_set_covisibles.argtypes = [vp, i, vp, i]
        L.ref_db_detect_loop.argtypes = [vp, vp, vp, i, vp, i, C.c_float, vp, i]
        L.ref_db_detect_reloc.argtypes = [vp, vp, vp, i, vp, i]
        self.L = L
        self.h = L.ref_voc_load(path.encode())
        assert self.h, "loadFromTextFile failed"
        self.nkf = 0

    def words(self):
        return self.L.ref_voc_words(self.h)

    def transform(self, desc, levelsup=4):
        desc = np.ascontiguousarray(desc, np.uint8).reshape(-1, 32)
        n = len(desc)
        cap = max(n, 1)
        bi, bv = np.zeros(cap, np.int32), np.zeros(cap, np.float64)
        fi, fp, ff = np.zeros(cap, np.int32), np.zeros(cap + 1, np.int32), np.zeros(cap, np.int32)
        nw, nn = C.c_int(0), C.c_int(0)
        self.L.ref_bow_transform(self.h, _p(desc), n, levelsup, C.byref(nw), _p(bi), _p(bv), C.byref(nn), _p(fi), _p(fp), _p(ff))
        return (bi[:nw.value], bv[:nw.value]), (fi[:nn.value], fp[:nn.value + 1], ff[:fp[nn.value]])

    def db_add(self, ids, vals):
        ids, vals = np.ascontiguousarray(ids, np.int32), np.ascontiguousarray(vals, np.float64)
        self.nkf += 1
        return self.L.ref_db_add(self.h, _p(ids), _p(vals), len(ids))

    def db_set_covisibles(self, k, others):
        o = np.ascontiguousarray(others, np.int32)
        self.L.ref_db_set_covisibles(self.h, int(k), _p(o), len(o))

    def detect_loop(self, q_ids, q_vals, connected, min_score):
        qi, qv, cn = np.ascontiguousarray(q_ids, np.int32), np.ascontiguousarray(q_vals, np.float64), np.ascontiguousarray(connected, np.int32)
        out = np.zeros(max(self.nkf, 1), np.int32)
        n = self.L.ref_db_detect_loop(self.h, _p(qi), _p(qv), len(qi), _p(cn), len(cn), float(min_score), _p(out), len(out))
        return out[:n]

    def detect_reloc(self, q_ids, q_vals):
        qi, qv = np.ascontiguousarray(q_ids, np.int32), np.ascontiguousarray(q_vals, np.float64)
        out = np.zeros(max(self.nkf, 1), np.int32)
        n = self.L.ref_db_detect_reloc(self.h, _p(qi), _p(qv), len(qi), _p(out), len(out))
        return out[:n]

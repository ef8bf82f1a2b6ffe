"""The oracle (oracle/orb_oracle*.c, a restatement) against oracle/_ref: the reference's OWN src/ORBextractor.cc,
ORBmatcher.cc, Frame.cc, KeyFrame.cc, MapPoint.cc compiled unmodified against the stand-in headers of oracle/ref_shim/
(recipe: oracle/Makefile `make ref`).  The reference's side of every comparison is read from tests/golden/ref_*.npz, the
stored results of that build (tests/ref_golden.py), so that the comparison runs from a checkout alone.

What this pins: the reference's control flow -- cell geometry, threshold fallback, quota redistribution, retention with
libstdc++'s nth_element, level loop, descriptor/blur aliasing, Frame's grid and GetFeaturesInArea order, every matcher's
candidate walk, accept rules and rotation filter -- with OpenCV's image primitives supplied by the oracle's own (pinned to
python-cv2 golden vectors in test_oracle_golden.py) and OpenCV's matrix algebra pinned to cv2.gemm golden vectors here."""
import os

import numpy as np
import pytest

import oracle as O
from oracle import ref as R
from orb_slam_b200.synth import textured_frame, shifted_frame
from ref_golden import Golden, WRITE, digest, extraction

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "opencv_gemm.npz")
G_EXTRACT, G_FRAMES, G_BOW = Golden("ref_extract"), Golden("ref_frames"), Golden("ref_bow")


def test_shim_matrix_algebra_against_cv2_golden_vectors():
    """The stand-in cv::gemm / cv::norm reproduce python-cv2 bit for bit on the shapes the reference's matchers use: float
    accumulation on OpenCV's unrolled small-matrix path (3x3*3x1 [+c], 3x3*3x3, 3x3*3x4, 4x4*4x4), double elsewhere."""
    g = np.load(GOLD)
    L = R.shim_lib()
    for k, name in enumerate(g["names"]):
        A, B, Cm, want = g["A%d" % k], g["B%d" % k], g["C%d" % k], g["out%d" % k]
        alpha, beta, flags = g["p%d" % k]
        for i in range(len(A)):
            a, b = np.ascontiguousarray(A[i]), np.ascontiguousarray(B[i])
            c = np.ascontiguousarray(Cm[i]) if Cm.size else None
            out = np.zeros_like(want[i])
            L.ref_shim_gemm(a.ctypes.data, a.shape[0], a.shape[1], b.ctypes.data, b.shape[0], b.shape[1], float(alpha),
                            c.ctypes.data if c is not None else None, float(beta), int(flags), out.ctypes.data)
            assert np.array_equal(out, want[i]), (str(name), i)
    for v, want in zip(g["norm_in"], g["norm_out"]):
        v = np.ascontiguousarray(v)
        assert L.ref_shim_norm(v.ctypes.data, 3) == want


@pytest.mark.parametrize("W,H,nf,nl,score,seed", [
    (640, 480, 1000, 8, 1, 21), (640, 480, 1000, 8, 1, 3), (641, 479, 500, 5, 1, 5), (1280, 720, 2000, 8, 1, 71),
    (640, 480, 1000, 8, 0, 21), (640, 480, 100, 8, 1, 3), (640, 480, 300, 1, 1, 4)])
def test_extractor_equals_the_reference_sources(W, H, nf, nl, score, seed):
    """E0-E13: src/ORBextractor.cc itself vs the oracle with the literal nth_element retention: same keypoints IN THE SAME
    ORDER (all seven fields, angle bit for bit) and same descriptors.  (640,480,100,...) has an empty cell grid on the last
    level; score 0 is HARRIS_SCORE."""
    img = textured_frame(W, H, seed=seed)
    rk, rd = extraction(G_EXTRACT, "extract_%d_%d_%d_%d_%d_%d" % (W, H, nf, nl, score, seed), img, nf, 1.2, nl, score, 20,
                        lambda: R.extract(img, nf, 1.2, nl, score, 20))     # the oracle with nth_element retention == the reference
    # the canonical tie rule (what the CUDA path implements) keeps the same multiset of scores per level and differs
    # from the reference binary only inside tie groups at a retention cut
    p2 = O.make_params(nf, 1.2, nl, score, 20)
    rc, ck, cd, _ = O.extract(p2, img)
    assert rc == 0 and len(ck) == len(rk)
    for l in range(nl):
        assert np.array_equal(np.sort(ck["response"][ck["octave"] == l]), np.sort(rk["response"][rk["octave"] == l]))
    common = len(set(zip(ck["octave"], ck["x"], ck["y"])) & set(zip(rk["octave"], rk["x"], rk["y"])))
    assert common >= 0.97 * len(rk)


def test_extractor_1080p_bench_geometry():
    img = textured_frame(1920, 1080, seed=1100)
    rk, rd = extraction(G_EXTRACT, "extract_1920_1080_2000_8_1_1100", img, 2000, 1.2, 8, 1, 20, lambda: R.extract(img, 2000, 1.2, 8, 1, 20))
    assert len(rk) == 2000


W, H = 640, 480
FX = FY = 500.0
CX, CY, DEPTH = W / 2.0, H / 2.0, 4.0


def _tcw(dx, dy, rot=(0.0, 0.0, 0.0)):
    """Camera pose that shifts points at depth DEPTH by (dx, dy) px, optionally with a small rotation (rad about x, y, z)."""
    ax, ay, az = rot
    cx_, sx_, cy_, sy_, cz_, sz_ = np.cos(ax), np.sin(ax), np.cos(ay), np.sin(ay), np.cos(az), np.sin(az)
    Rx = np.array([[1, 0, 0], [0, cx_, -sx_], [0, sx_, cx_]])
    Ry = np.array([[cy_, 0, sy_], [0, 1, 0], [-sy_, 0, cy_]])
    Rz = np.array([[cz_, -sz_, 0], [sz_, cz_, 0], [0, 0, 1]])
    T = np.zeros((3, 4), np.float32)
    T[:, :3] = (Rz @ Ry @ Rx).astype(np.float32)
    T[0, 3], T[1, 3] = dx * DEPTH / FX, dy * DEPTH / FY
    return T


def _world(k):
    w = np.empty((len(k), 3), np.float32)
    w[:, 0] = (k["x"] - np.float32(CX)) / np.float32(FX) * np.float32(DEPTH)
    w[:, 1] = (k["y"] - np.float32(CY)) / np.float32(FY) * np.float32(DEPTH)
    w[:, 2] = DEPTH
    return w


@pytest.fixture(scope="module")
def frames():
    """Three consecutive frames through the reference's own Frame constructor (extract + undistort + grid).  rf: the
    reference's Frame objects, built only to record the golden vectors (None otherwise)."""
    rng = np.random.default_rng(1)
    imgs, shifts = [textured_frame(W, H, seed=21)], [(0, 0)]
    for i in range(1, 3):
        dx, dy = int(rng.integers(-5, 6)), int(rng.integers(-4, 5))
        imgs.append(shifted_frame(imgs[-1], dx, dy, seed=i))
        shifts.append((dx, dy))
    rf = [R.RefFrame.from_image(im, FX, FY, CX, CY, None, 1000, 1.2, 8, 1, 20) for im in imgs] if WRITE else [None] * 3
    feats = []
    for j, (f, im) in enumerate(zip(rf, imgs)):
        def ref_get():
            keys, keys_un, desc, bounds, ginv = f.get()
            return digest(keys, desc), digest(keys_un), bounds, ginv
        keys_desc, keys_un_digest, bounds, ginv = G_FRAMES("frame%d_get" % j, ref_get)
        keys, desc = extraction(G_FRAMES, "frame%d_extract" % j, im, 1000, 1.2, 8, 1, 20, lambda: f.get()[0:3:2])
        keys_un = keys
        assert digest(keys_un) == keys_un_digest and list(bounds) == [0, 0, W, H]      # zero distortion (Frame.cc:291-295, :342-348)
        assert ginv[0] == np.float32(64) / np.float32(W) and ginv[1] == np.float32(48) / np.float32(H)
        feats.append((keys_un, desc))
    of = [O.OracleFrame(k, d, W, H) for k, d in feats]
    yield rf, of, feats, shifts
    for f in rf:
        if f is not None:
            f.close()


def test_frame_grid_and_features_in_area(frames):
    """M14: Frame's 64x48 grid (Frame.cc:109-123, PosInGrid :267-277) and GetFeaturesInArea (:200-265) -- the candidate ORDER."""
    rf, of, feats, _ = frames
    for j, (f, o, (k, d)) in enumerate(zip(rf, of, feats)):
        start, items = G_FRAMES("frame%d_grid" % j, lambda: f.grid())
        assert np.array_equal(start, np.ctypeslib.as_array(o.c.cell_start)) and np.array_equal(items, o.items[:len(items)])

        # a frame rebuilt from arrays (the path the other tests use to inject keypoints) has the same grid
        def from_arrays_grid():
            g = R.RefFrame.from_arrays(k, d, W, H, FX, FY, CX, CY)
            sg = g.grid()
            g.close()
            return sg
        s2, i2 = G_FRAMES("frame%d_grid_from_arrays" % j, from_arrays_grid)
        assert np.array_equal(start, s2) and np.array_equal(items, i2)
        rng = np.random.default_rng(7)
        queries = []
        for _ in range(300):
            x, y = float(rng.uniform(-20, W + 20)), float(rng.uniform(-20, H + 20))
            r = float(rng.choice([3.0, 15.0, 37.5, 100.0]))
            lo, hi = [(-1, -1), (0, 0), (2, 4), (-1, 3), (5, -1)][int(rng.integers(0, 5))]
            queries.append((x, y, r, lo, hi))
        def ref_features_in_area():
            found = [f.features_in_area(*q) for q in queries]
            return np.concatenate(found), np.array([len(a) for a in found])
        flat, counts = G_FRAMES("frame%d_features_in_area" % j, ref_features_in_area)
        for q, g in zip(queries, np.split(flat, np.cumsum(counts)[:-1])):
            assert np.array_equal(g, o.features_in_area(*q)), q


@pytest.mark.parametrize("ori", [True, False])
def test_search_by_projection_frame_frame(frames, ori):
    """M2 (the bench's matcher): ORBmatcher::SearchByProjection(Frame&, const Frame&, float), ORBmatcher.cc:1507-1620."""
    rf, of, feats, shifts = frames
    rng = np.random.default_rng(3)
    total = 0
    for j in (1, 2):
        kl = feats[j - 1][0]
        has = (rng.random(len(kl)) < 0.9).astype(np.uint8)
        outl = (rng.random(len(kl)) < 0.05).astype(np.uint8)
        pre = np.full(len(feats[j][0]), -1, np.int32)
        pre[rng.random(len(feats[j][0])) < 0.03] = 5
        for th, rot in ((15.0, (0, 0, 0)), (7.0, (0, 0, 0)), (15.0, (0.003, -0.002, 0.004)), (15.0, (-0.001, 0.004, -0.006))):
            T = _tcw(*shifts[j], rot=rot)     # a general rotation exercises the float accumulation of Rcw*x3Dw+tcw
            n_r, mp_r = G_FRAMES("m2_%d_%d_%s_%s" % (j, th, rot, ori),
                                 lambda: R.search_by_projection_ff(rf[j], rf[j - 1], has, outl, _world(kl), T, th, 0.9, ori, cur_mp=pre))
            n_o, mp_o = O.search_by_projection_ff(of[j], of[j - 1], has, outl, _world(kl), T, FX, FY, CX, CY, th, ori, cur_mp=pre)
            assert n_r == n_o and np.array_equal(mp_r, mp_o), (j, th, rot)
            total += n_r
    assert total > 500


def test_window_search_and_initialization(frames):
    """M7 WindowSearch (ORBmatcher.cc:409-516) and M8 SearchForInitialization (:598-713)."""
    rf, of, feats, _ = frames
    k1 = feats[0][0]
    has = (np.random.default_rng(0).random(len(k1)) < 0.8).astype(np.uint8)
    for nnratio, ori, win, lo, hi in [(0.9, True, 50, -1, 2 ** 31 - 1), (0.6, False, 100, 2, 5), (0.9, True, 200, -1, 2 ** 31 - 1)]:
        n_r, m_r = G_FRAMES("m7_%s_%s_%d_%d_%d" % (nnratio, ori, win, lo, hi), lambda: R.window_search(rf[0], rf[1], has, win, lo, hi, nnratio, ori))
        n_o, m_o = O.window_search(of[0], of[1], has, win, lo, hi, nnratio=nnratio, check_orientation=ori)
        assert n_r == n_o and np.array_equal(m_r, m_o), (nnratio, ori, win)
    prev = np.stack([k1["x"], k1["y"]], axis=1).astype(np.float32)
    n_r, m_r, p_r = G_FRAMES("m8_first", lambda: R.search_for_initialization(rf[0], rf[1], prev, 100, 0.9, True))
    n_o, m_o, p_o = O.search_for_initialization(of[0], of[1], prev, 100, nnratio=0.9, check_orientation=True)
    assert n_r == n_o and np.array_equal(m_r, m_o) and np.array_equal(p_r, p_o) and n_r > 20
    n_r2, m_r2, _ = G_FRAMES("m8_second", lambda: R.search_for_initialization(rf[0], rf[1], p_r, 100, 0.9, True))   # Tracking::Initialize calls it repeatedly
    n_o2, m_o2, _ = O.search_for_initialization(of[0], of[1], p_o, 100, nnratio=0.9, check_orientation=True)
    assert n_r2 == n_o2 and np.array_equal(m_r2, m_o2)


def test_local_points_and_f1f2_projection(frames):
    """M3 SearchByProjection(Frame&, vector<MapPoint*>, th) (:49-125) and M6 SearchByProjection(F1, F2, window, ...) (:519-594)."""
    rf, of, feats, shifts = frames
    (k1, d1), (k2, d2) = feats[0], feats[1]
    n1 = len(k1)
    rng = np.random.default_rng(5)
    dx, dy = shifts[1]
    occupied = np.full(len(k2), -1, np.int32)
    occupied[rng.random(len(k2)) < 0.03] = 3
    in_view = (rng.random(n1) < 0.9).astype(np.uint8)
    proj = np.stack([k1["x"] + np.float32(dx) + rng.normal(0, 1.0, n1).astype(np.float32),
                     k1["y"] + np.float32(dy) + rng.normal(0, 1.0, n1).astype(np.float32)], axis=1).astype(np.float32)
    level = k1["octave"].astype(np.int32)
    vcos = rng.choice(np.array([0.9999, 0.99, 0.5], np.float32), n1)
    for th, nnr in ((3.0, 0.8), (1.0, 0.8), (5.0, 0.6)):
        n_r, mp_r = G_FRAMES("m3_%s_%s" % (th, nnr), lambda: R.search_local_points(rf[1], in_view, proj, level, vcos, d1, th, nnr, f_mp=occupied))
        n_o, mp_o = O.search_local_points(of[1], in_view, proj, level, vcos, d1, th, nnratio=nnr, f_mp=occupied)
        assert n_r == n_o and np.array_equal(mp_r, mp_o), th
    valid = (rng.random(n1) < 0.85).astype(np.uint8)
    for win in (10, 25):
        n_r, mp_r = G_FRAMES("m6_%d" % win, lambda: R.search_by_projection_f1f2(rf[0], rf[1], valid, _world(k1), _tcw(dx, dy), win, 0.9,
                                                                                 f2_mp=occupied))
        n_o, mp_o = O.search_by_projection_f1f2(of[0], of[1], valid, _world(k1), _tcw(dx, dy), FX, FY, CX, CY, win, nnratio=0.9, f2_mp=occupied)
        assert n_r == n_o and np.array_equal(mp_r, mp_o), win
    assert G_FRAMES("m1", lambda: R.descriptor_distance(d1[3], d2[7])) == O.hamming(d1[3], d2[7])


def test_oracle_projection_primitive_against_cv2_golden_vectors():
    """`Rcw*x3Dw + tcw` as the oracle (and, formula for formula, match_host.cpp / match_kernels.cu / host/ORBmatcher.cc)
    evaluates it equals cv2.gemm(R, x, 1, t, 1): float accumulation on OpenCV's small-matrix path."""
    import ctypes as C
    g = np.load(GOLD)
    k = list(g["names"]).index("R*x+t")
    L = O.lib()
    L.orb_oracle_cv_Rx_plus_t.argtypes = [C.c_void_p] * 3
    for A, B, Cm, want in zip(g["A%d" % k], g["B%d" % k], g["C%d" % k], g["out%d" % k]):
        T = np.ascontiguousarray(np.concatenate([A, Cm], axis=1), np.float32)
        X = np.ascontiguousarray(B.reshape(3), np.float32)
        out = np.zeros(3, np.float32)
        L.orb_oracle_cv_Rx_plus_t(T.ctypes.data, X.ctypes.data, out.ctypes.data)
        assert np.array_equal(out, want.reshape(3))


# ---- KeyFrame-level matchers: the scripted scene of tests/ref_scenarios.py in the reference build vs the oracle's arrays ---
@pytest.fixture(scope="module")
def scene():
    import ref_scenarios as RS
    return RS, RS.run_ref()


def _index_of_id(ids):
    """map-point id (relative) -> feature index of the keyframe that owns it"""
    m = {}
    for i, v in enumerate(ids):
        if v >= 0:
            m[int(v)] = i
    return lambda arr: np.array([m.get(int(v), -1) if v >= 0 else int(v) for v in arr], np.int32)


def test_reloc_projection_against_keyframe(scene):
    """M4: SearchByProjection(Frame&, KeyFrame*, set<MapPoint*>&, th, ORBdist), ORBmatcher.cc:1622-1746."""
    RS, out = scene
    (k1, d1), (k2, d2) = RS.features()
    idsA, idsB, _, _ = out["ids"]
    hasA, bad, found, occupied, world, min_dist, T_B = out["m4_inputs"]
    to_idx = _index_of_id(idsA)
    o2 = O.OracleFrame(k2, d2, RS.W, RS.H)
    skip = set(int(b) for b in bad) | set(int(f) for f in found)      # isBad() or already found (:1643)
    valid = np.array([hasA[i] and int(idsA[i]) not in skip for i in range(len(k1))])
    pre = np.where(occupied, 7, -1).astype(np.int32)
    for key, th, od, ori in (("m4_a", 10.0, 100, True), ("m4_b", 3.0, 64, True), ("m4_c", 10.0, 100, False)):
        n_r, mp_r = out[key]
        n_o, mp_o = O.search_by_projection_kf(o2, valid.astype(np.uint8), world, min_dist, d1, k1["angle"], T_B, RS.FX, RS.FY, RS.CX, RS.CY,
                                              th, od, ori, cur_mp=pre)
        got = to_idx(mp_r)
        got[occupied] = 7
        assert n_r == n_o and np.array_equal(got, mp_o), key
        assert n_r > 200


def test_search_by_bow_both_overloads(scene):
    """M9: SearchByBoW(KeyFrame*, Frame&, ...) :155-284 and SearchByBoW(KeyFrame*, KeyFrame*, ...) :715-850."""
    RS, out = scene
    (k1, d1), (k2, d2) = RS.features()
    idsA, idsB, _, _ = out["ids"]
    hasA, bad, _, _, _, _, _ = out["m4_inputs"]
    fvA, fvB = out["m9_inputs"]
    badset = set(int(b) for b in bad)
    valid1 = np.array([idsA[i] >= 0 and int(idsA[i]) not in badset for i in range(len(k1))], np.uint8)
    valid2 = (idsB >= 0).astype(np.uint8)
    a_idx, b_idx = _index_of_id(idsA), _index_of_id(idsB)
    for key, nnr, ori in (("m9_kf_f_a", 0.75, True), ("m9_kf_f_b", 0.6, False)):
        n_r, m_r = out[key]
        n_o, m_o = O.search_by_bow(0, d1, valid1, k1["angle"], fvA, d2, np.ones(len(k2), np.uint8), k2["angle"], fvB, nnratio=nnr, check_orientation=ori)
        assert n_r == n_o and np.array_equal(a_idx(m_r), m_o), key
        assert n_r > 200
    for key, nnr, ori in (("m9_kf_kf_a", 0.75, True), ("m9_kf_kf_b", 0.6, False)):
        n_r, m_r = out[key]
        n_o, m_o = O.search_by_bow(1, d1, valid1, k1["angle"], fvA, d2, valid2, k2["angle"], fvB, nnratio=nnr, check_orientation=ori)
        assert n_r == n_o and np.array_equal(b_idx(m_r), m_o), key
        assert n_r > 50


def test_search_for_triangulation(scene):
    """M10: SearchForTriangulation :852-1014 + CheckDistEpipolarLine :136-153."""
    RS, out = scene
    (k1, d1), (k2, d2) = RS.features()
    idsA, idsB, _, _ = out["ids"]
    fvA, fvB = out["m9_inputs"]
    (F12,) = out["m10_inputs"]
    sf = np.empty(8, np.float32)
    O.lib().orb_oracle_frame_scale_factors(np.float32(1.2), 8, sf.ctypes.data_as(__import__("ctypes").c_void_p))
    sigma2 = sf * sf     # Frame.cc:95-103: mvLevelSigma2[i] = mvScaleFactors[i]^2
    for key, ori in (("m10_a", True), ("m10_b", False)):
        n_r, pairs = out[key]
        n_o, m12 = O.search_for_triangulation(k1, d1, (idsA >= 0).astype(np.uint8), fvA, k2, d2, (idsB >= 0).astype(np.uint8), fvB, F12, sigma2,
                                              check_orientation=ori)
        want = np.array([(i, m12[i]) for i in range(len(m12)) if m12[i] >= 0], np.int32).reshape(-1, 2)
        assert n_r == n_o and np.array_equal(pairs, want), key
        assert n_r > 20


# ---- (f) rows against the reference's own code: Frame's undistortion, DBoW2's transform, KeyFrameDatabase ------------------
def test_frame_constructor_with_lens_distortion():
    """N1: Frame::UndistortKeyPoints / ComputeImageBounds (Frame.cc:289-350) through the reference's Frame constructor: mvKeysUn,
    the image bounds, the grid constants and the grid itself vs the oracle's arrays."""
    img = textured_frame(640, 480, seed=9)
    fx, fy, cx, cy, dist = 520.0, 515.0, 318.0, 243.0, np.array([-0.25, 0.09, 0.001, -0.0007], np.float32)

    def ref_frame():
        f = R.RefFrame.from_image(img, fx, fy, cx, cy, dist, 800, 1.2, 8, 1, 20)
        keys, keys_un, desc, bounds, ginv = f.get()
        f.close()
        return (keys, desc), keys_un, bounds, ginv
    keys_un, bounds, ginv = G_FRAMES("distorted_frame_get", lambda: ref_frame()[1:])
    keys, desc = extraction(G_FRAMES, "distorted_frame_extract", img, 800, 1.2, 8, 1, 20, lambda: ref_frame()[0])
    assert not np.array_equal(keys["x"], keys_un["x"])
    d5 = np.concatenate([dist, [0]]).astype(np.float32)
    assert np.array_equal(keys_un, O.undistort_keypoints(keys, fx, fy, cx, cy, d5))
    b = O.image_bounds(640, 480, fx, fy, cx, cy, d5)
    assert np.array_equal(bounds, b)
    assert ginv[0] == np.float32(64) / np.float32(b[2] - b[0]) and ginv[1] == np.float32(48) / np.float32(b[3] - b[1])


@pytest.mark.parametrize("k,L,ragged,levelsup", [(10, 3, False, 2), (6, 4, True, 3), (10, 3, False, 0)])
def test_vocabulary_transform_against_dbow2(tmp_path, k, L, ragged, levelsup):
    """N2: DBoW2::TemplatedVocabulary::transform (TemplatedVocabulary.h:1126-1262, the tree descent with FORB::distance and the
    TF-IDF / L1 weighting) itself, loaded from the text format of Data/ORBvoc.txt, vs the oracle's BowVector / FeatureVector."""
    from orb_slam_b200.synth import random_vocabulary, random_descriptors, noisy_copies
    voc = random_vocabulary(k, L, seed=5, ragged=ragged)
    path = str(tmp_path / "voc.txt")
    R.write_vocabulary_text(voc, path)
    leaves = voc["node_desc"][voc["word_id"] >= 0]
    desc = np.concatenate([noisy_copies(leaves[np.random.default_rng(1).integers(0, len(leaves), 700)], 0.08, 2), random_descriptors(300, 3)])

    def ref_transform():
        V = R.RefVocabulary(path)
        return V.words(), V.transform(desc, levelsup)
    words, ((bi, bv), (fi, fp, ff)) = G_BOW("transform_%d_%d_%s_%d" % (k, L, ragged, levelsup), ref_transform)
    assert words == int((voc["word_id"] >= 0).sum())
    (obi, obv), (ofi, ofp, off) = O.bow_transform(voc, desc, levelsup=levelsup, weighting=0, norm=1)
    assert np.array_equal(bi, obi) and np.array_equal(bv, obv)            # float64 values bit for bit (same summation order)
    assert np.array_equal(fi, ofi) and np.array_equal(fp, ofp) and np.array_equal(ff, off)
    assert len(bi) > 50


def test_keyframe_database_against_the_reference(tmp_path):
    """N3: KeyFrameDatabase::DetectLoopCandidates (:72-204) and DetectRelocalisationCandidates (:206-308) with the reference's own
    inverted file, covisibility accumulation and DBoW2 L1 score vs the oracle's candidate lists (order included)."""
    from orb_slam_b200.synth import random_keyframe_db
    # a flat-enough vocabulary that only has to own the word ids: 10^4 words
    n_nodes = 1 + 10 + 100 + 1000 + 10000
    path = str(tmp_path / "flat.txt")
    with open(path, "w") as f:
        f.write("10 4 0 0\n")
        lines, first_child = [], 1
        for nid in range(1, n_nodes):
            parent = (nid - 1) // 10
            leaf = 1 if nid >= 1111 else 0
            lines.append("%d %d %s 1.0" % (parent, leaf, " ".join(["0"] * 32)))
        f.write("\n".join(lines))
    for seed in (0, 1):
        db = random_keyframe_db(nkf=120 + 30 * seed, nwords=3000, words_per_kf=200, seed=seed, loop_at=20 + seed)
        nkf = len(db["kf_ptr"]) - 1

        def ref_database():
            V = R.RefVocabulary(path)
            added = [V.db_add(db["db_ids"][db["kf_ptr"][kf]:db["kf_ptr"][kf + 1]], db["db_vals"][db["kf_ptr"][kf]:db["kf_ptr"][kf + 1]])
                     for kf in range(nkf)]
            for kf in range(nkf):
                V.db_set_covisibles(kf, db["covis"][db["covis_ptr"][kf]:db["covis_ptr"][kf + 1]])
            loops = [V.detect_loop(db["q_ids"], db["q_vals"], np.flatnonzero(db["connected"]), s) for s in (0.0, 0.02)]
            return V.words(), added, loops, V.detect_reloc(db["q_ids"], db["q_vals"])
        words, added, loops, reloc = G_BOW("keyframe_database_%d" % seed, ref_database)
        assert words == 10000 and added == list(range(nkf))
        for min_score, got in zip((0.0, 0.02), loops):
            cand, _, _ = O.bow_db_detect(0, db["q_ids"], db["q_vals"], db["kf_ptr"], db["db_ids"], db["db_vals"], db["connected"],
                                         db["covis_ptr"], db["covis"], min_score)
            assert np.array_equal(got, cand), (seed, min_score)
        cand, _, _ = O.bow_db_detect(1, db["q_ids"], db["q_vals"], db["kf_ptr"], db["db_ids"], db["db_vals"], db["connected"],
                                     db["covis_ptr"], db["covis"], 0.0)
        assert np.array_equal(reloc, cand) and len(cand) > 0, seed


def test_distinctive_descriptor_against_the_reference():
    """N4: MapPoint::ComputeDistinctiveDescriptors (MapPoint.cc:185-250): the observed descriptor with the least median distance
    to the others, first minimum in the std::map's iteration order, vs the oracle on the same order."""
    import ctypes as C
    from orb_slam_b200.synth import random_descriptors, noisy_copies
    rng = np.random.default_rng(4)
    nkf, nfeat = 9, 40
    base = random_descriptors(nfeat, 11)
    kps = np.zeros(nfeat, O.KP_DTYPE)
    kps["x"], kps["y"] = rng.uniform(20, 600, nfeat), rng.uniform(20, 440, nfeat)
    descs = [noisy_copies(base, 0.10, 100 + k) for k in range(nkf)]

    def ref_map_points():
        """per map point: the reference's distinctive descriptor and its observations in std::map order (keyframe, feature)"""
        S = R.Scene("ref")
        L = S.L
        L.ref_mp_observation_order.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_int]
        kfs = []
        for k in range(nkf):
            f = S.frame(kps, descs[k], 640, 480, 500.0, 500.0, 320.0, 240.0)
            kfs.append(S.keyframe(f, np.eye(4, dtype=np.float32)[:3]))
            f.close()
        got, order = [], []
        for i in range(nfeat):
            mp = S.map_point(np.array([0, 0, 4], np.float32), descs[0][i], None, 1.0, 30.0, kfs[0])
            seen = [k for k in range(nkf) if rng.random() < 0.7] or [0]
            for k in seen:
                S.observe(kfs[k], mp, i)
            got.append(S.compute_distinctive(mp))
            ok_, oi_ = np.zeros(16, np.int32), np.zeros(16, np.int32)
            n = L.ref_mp_observation_order(mp, ok_.ctypes.data, oi_.ctypes.data, 16)
            order.append(np.array([(kfs.index(int(ok_[j])), oi_[j]) for j in range(n)], np.int32))
        return got, order
    got, order = G_BOW("distinctive", ref_map_points)
    groups = [np.stack([descs[k][i] for k, i in o]) for o in order]
    ptr = np.concatenate([[0], np.cumsum([len(g) for g in groups])]).astype(np.int32)
    best = O.distinctive_descriptors(np.concatenate(groups), ptr)
    for i in range(nfeat):
        assert np.array_equal(got[i], groups[i][best[i]]), i

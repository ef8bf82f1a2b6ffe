"""One scripted SLAM scene -- two keyframes with poses, map points with observations, FeatureVectors -- run through every
ORBmatcher method of one build of the reference's map model (oracle/ref.py: "ref" = the reference's own ORBmatcher.cc,
"facade" = orb_slam_b200/host/ORBmatcher.cc over liborbfe.so, both next to the reference's unmodified Frame.cc /
KeyFrame.cc / MapPoint.cc).  Returns plain arrays so that two builds, or a build and the oracle, can be compared.  What the
"ref" build returns is stored in tests/golden/ref_scene.npz (tests/ref_golden.py): run_ref() and features() read it."""
import numpy as np

from oracle import ref as R
from orb_slam_b200.synth import textured_frame, shifted_frame
from ref_golden import Golden, extraction

GOLDEN = Golden("ref_scene")

W, H = 640, 480
FX = FY = 500.0
CX, CY, DEPTH = W / 2.0, H / 2.0, 4.0
SHIFT = (4, -3)


def rot_xyz(ax, ay, az):
    cx_, sx_, cy_, sy_, cz_, sz_ = np.cos(ax), np.sin(ax), np.cos(ay), np.sin(ay), np.cos(az), np.sin(az)
    Rx = np.array([[1, 0, 0], [0, cx_, -sx_], [0, sx_, cx_]])
    Ry = np.array([[cy_, 0, sy_], [0, 1, 0], [-sy_, 0, cy_]])
    Rz = np.array([[cz_, -sz_, 0], [sz_, cz_, 0], [0, 0, 1]])
    return Rz @ Ry @ Rx


def pose(dx, dy, rot=(0.0, 0.0, 0.0), dz=0.0):
    T = np.zeros((3, 4), np.float32)
    T[:, :3] = rot_xyz(*rot).astype(np.float32)
    T[0, 3], T[1, 3], T[2, 3] = dx * DEPTH / FX, dy * DEPTH / FY, dz
    return T


def backproject(k):
    w = np.empty((len(k), 3), np.float32)
    w[:, 0] = (k["x"] - np.float32(CX)) / np.float32(FX) * np.float32(DEPTH)
    w[:, 1] = (k["y"] - np.float32(CY)) / np.float32(FY) * np.float32(DEPTH)
    w[:, 2] = DEPTH
    return w


def node_of(desc, byte, shift, mul, add):
    """A stand-in for the vocabulary node of a feature: a coarse function of a few descriptor bits."""
    return (desc[:, byte].astype(np.int32) >> shift) * mul + add


def fv_of(nodes):
    order = np.argsort(nodes, kind="stable")
    ids, counts = np.unique(nodes, return_counts=True)
    return ids.astype(np.int32), np.concatenate([[0], np.cumsum(counts)]).astype(np.int32), order.astype(np.int32)


_FEATS = None


def features():
    """Keypoints / descriptors of two consecutive frames, from the reference's own extractor (identical for every build)."""
    global _FEATS
    if _FEATS is None:
        a = textured_frame(W, H, seed=21)
        b = shifted_frame(a, SHIFT[0], SHIFT[1], seed=1)
        _FEATS = [extraction(GOLDEN, "features%d" % i, im, 1000, 1.2, 8, 1, 20, lambda: R.extract(im, 1000, 1.2, 8, 1, 20))
                  for i, im in enumerate((a, b))]
    return _FEATS


def run_ref():
    """run("ref"), as stored."""
    return GOLDEN("run_ref", lambda: run("ref"))


def run(which):
    """Builds the scene in build `which` and runs M2-M12.  Every result is a numpy array / int / list of plain tuples."""
    (k1, d1), (k2, d2) = features()
    n1, n2 = len(k1), len(k2)
    rng = np.random.default_rng(2024)
    S = R.Scene(which)
    out = {}
    mp0, kf0 = S.counts()        # ids are reported relative to these, so that the two builds line up
    T_A, T_B = pose(0, 0), pose(SHIFT[0], SHIFT[1], rot=(0.002, -0.001, 0.003), dz=0.05)
    fA, fB = S.frame(k1, d1, W, H, FX, FY, CX, CY), S.frame(k2, d2, W, H, FX, FY, CX, CY)
    kfA, kfB = S.keyframe(fA, T_A), S.keyframe(fB, T_B)
    world = backproject(k1)
    min_dist = (DEPTH / np.float32(1.2) ** k1["octave"].astype(np.float32) * rng.uniform(0.8, 1.1, n1)).astype(np.float32)
    max_dist = (min_dist * np.float32(1.2) ** 7 * rng.uniform(0.9, 1.2, n1)).astype(np.float32)
    hasA = rng.random(n1) < 0.85
    mpsA = np.full(n1, -1, np.int32)
    for i in range(n1):
        if hasA[i]:
            nrm = np.array([0, 0, 1], np.float32) + rng.normal(0, 0.15, 3).astype(np.float32)
            mpsA[i] = S.map_point(world[i], d1[i], nrm / np.linalg.norm(nrm), min_dist[i], max_dist[i], kfA)
            S.observe(kfA, mpsA[i], i)
    bad = [int(m) for m in mpsA[hasA][:: 37]]
    for m in bad:
        S.set_bad(m)
    # keyframe B owns a few map points of its own (some features), positions near what A would predict
    hasB = rng.random(n2) < 0.3
    mpsB = np.full(n2, -1, np.int32)
    wB = backproject(k2)
    for i in range(n2):
        if hasB[i]:
            p = wB[i] - np.array([SHIFT[0] * DEPTH / FX, SHIFT[1] * DEPTH / FY, 0], np.float32)
            mpsB[i] = S.map_point(p, d2[i], np.array([0, 0, 1], np.float32), 1.0, 30.0, kfB)
            S.observe(kfB, mpsB[i], i)
    out["ids"] = (mpsA - mp0 * (mpsA >= 0), mpsB - mp0 * (mpsB >= 0), kfA - kf0, kfB - kf0)
    rel = lambda a: np.where(np.asarray(a) >= 0, np.asarray(a) - mp0, np.asarray(a))

    # ---- M4: Frame B against keyframe A (relocalisation refinement)
    S.set_pose(fB, T_B)
    found = [int(m) for m in mpsA[hasA][5:: 11]]
    pre = np.full(n2, -1, np.int32)
    occ = rng.random(n2) < 0.03
    pre[occ] = mpsB[np.flatnonzero(hasB)[0]]
    for key, th, od, ori in (("m4_a", 10.0, 100, True), ("m4_b", 3.0, 64, True), ("m4_c", 10.0, 100, False)):
        n, mp = S.search_by_projection_frame_kf(fB, kfA, found, th, od, 0.9, ori, cur_mp=pre)
        out[key] = (n, rel(mp))
    out["m4_inputs"] = (hasA, np.array(bad) - mp0, np.array(found) - mp0, pre >= 0, world, min_dist, T_B)   # ids relative, like every id returned

    # ---- M5: keyframe B, Sim3 pose (scale 1.05 on the same rigid pose), candidate points = A's map points
    s = np.float32(1.05)
    Scw = np.eye(4, dtype=np.float32)
    Scw[:3, :3] = s * T_B[:, :3]
    Scw[:3, 3] = s * T_B[:, 3]
    pts = [int(m) for m in mpsA[hasA]]
    matched0 = np.full(n2, -1, np.int32)
    matched0[np.flatnonzero(hasB)[::5]] = mpsB[np.flatnonzero(hasB)[::5]]
    for key, th in (("m5_a", 10), ("m5_b", 4)):
        n, m = S.search_by_projection_sim3(kfB, Scw, pts, matched0, th, 0.75)
        out[key] = (n, rel(m))

    # ---- M9: vocabulary-node brute force
    nodeA, nodeB = node_of(d1, 0, 3, 3, 11), node_of(d2, 0, 3, 3, 11)
    nodeB[rng.random(n2) < 0.05] = 9999
    fvA, fvB = fv_of(nodeA), fv_of(nodeB)
    S.set_feature_vector(kfA, fvA)
    S.set_feature_vector(kfB, fvB)
    S.set_feature_vector(fB, fvB)
    for key, nnr, ori in (("m9_kf_f_a", 0.75, True), ("m9_kf_f_b", 0.6, False)):
        n, m = S.search_by_bow_kf_frame(kfA, fB, nnr, ori)
        out[key] = (n, rel(m))
    for key, nnr, ori in (("m9_kf_kf_a", 0.75, True), ("m9_kf_kf_b", 0.6, False)):
        n, m = S.search_by_bow_kf_kf(kfA, kfB, nnr, ori)
        out[key] = (n, rel(m))
    out["m9_inputs"] = (fvA, fvB)

    # ---- M10: triangulation candidates between the two keyframes (rectified-pair fundamental matrix)
    F12 = np.array([[0, 0, 0], [0, 0, -1], [0, 1, float(-SHIFT[1])]], np.float32)
    for key, ori in (("m10_a", True), ("m10_b", False)):
        n, pairs = S.search_for_triangulation(kfA, kfB, F12, 0.6, ori)
        out[key] = (n, pairs.copy())
    out["m10_inputs"] = (F12,)

    # ---- M11: SearchBySim3 (camera 2 -> camera 1: p1 = s12 R12 p2 + t12 with T_A = I)
    R12 = T_B[:, :3].T.copy()
    t12 = -(R12 @ T_B[:, 3])
    m12 = np.full(n1, -1, np.int32)
    seeded = np.flatnonzero(hasA)[3:: 29]
    for i in seeded:      # a few pairs already matched on entry
        j = np.flatnonzero(hasB)[i % hasB.sum()]
        m12[i] = mpsB[j]
    n, m = S.search_by_sim3(kfA, kfB, m12, 1.0, R12, t12, 7.5)
    out["m11"] = (n, rel(m))

    # ---- M12: Fuse mutates the map: run last, then dump the state of both keyframes and of every map point
    out["m12_fuse"] = S.fuse(kfB, pts, 3.0)
    out["m12_state_1"] = (rel(S.kf_map_points(kfA)), rel(S.kf_map_points(kfB)))
    kfB2 = S.keyframe(fB, T_B)
    for i in np.flatnonzero(hasB)[::2]:
        mpx = S.map_point(wB[i] - np.array([SHIFT[0] * DEPTH / FX, SHIFT[1] * DEPTH / FY, 0], np.float32), d2[i],
                          np.array([0, 0, 1], np.float32), 1.0, 30.0, kfB2)
        S.observe(kfB2, mpx, i)
    out["m12_fuse_sim3"] = S.fuse_sim3(kfB2, Scw, pts, 4.0)
    out["m12_state_2"] = (rel(S.kf_map_points(kfA)), rel(S.kf_map_points(kfB)), rel(S.kf_map_points(kfB2)))
    states = []
    mp1, _ = S.counts()
    for m in range(mp0, mp1):
        b, obs = S.mp_state(m)
        states.append((b, tuple((k - kf0, i) for k, i in obs)))
    out["m12_mp_states"] = states
    fA.close()
    fB.close()
    return out


def same(a, b):
    if isinstance(a, (tuple, list)):
        return len(a) == len(b) and all(same(x, y) for x, y in zip(a, b))
    if isinstance(a, np.ndarray):
        return np.array_equal(a, b)
    return a == b

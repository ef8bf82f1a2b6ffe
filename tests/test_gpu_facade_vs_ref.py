"""The drop-in claim, literally: the reference's unmodified Frame.cc, KeyFrame.cc, MapPoint.cc, Map.cc, KeyFrameDatabase.cc and
DBoW2 are compiled twice (oracle/Makefile `make ref`) -- once with the reference's own ORBextractor.cc / ORBmatcher.cc, once with
this repo's include/ORBextractor.h, include/ORBmatcher.h and orb_slam_b200/host/*.cc over liborbfe.so (CUDA) in their place --
and the same scripted scene (tests/ref_scenarios.py) is run through both: every ORBmatcher method must return the same
matches, and after Fuse the same map (keyframe slots, bad flags, observations).  Needs a GPU for the facade build.

The reference build's results are stored (tests/golden/ref_*.npz, see tests/ref_golden.py); the facade build compiles the
reference's Frame.cc / KeyFrame.cc / MapPoint.cc, so these tests run only where that build exists (oracle/Makefile `make ref`
with the reference sources at ORB_REFERENCE_ROOT) and skip elsewhere."""
import numpy as np
import pytest

import oracle as O
from oracle import ref as R
from ref_golden import Golden, extraction

pytestmark = [pytest.mark.gpu,
              pytest.mark.skipif(not R.available("facade"),
                                 reason="oracle/_ref/libfacade_orbslam.so is built from the reference sources, which this checkout does not contain")]


@pytest.fixture(scope="module")
def both(gpu_required):
    import ref_scenarios as RS
    return RS, RS.run_ref(), RS.run("facade")


@pytest.mark.parametrize("key", ["m4_a", "m4_b", "m4_c", "m5_a", "m5_b", "m9_kf_f_a", "m9_kf_f_b", "m9_kf_kf_a", "m9_kf_kf_b", "m10_a",
                                 "m10_b", "m11", "m12_fuse", "m12_state_1", "m12_fuse_sim3", "m12_state_2", "m12_mp_states"])
def test_keyframe_level_methods_equal_the_reference(both, key):
    """M4, M5, M9 (x2), M10, M11, M12 (x2): reference ORBmatcher.cc vs the facade on real KeyFrame / MapPoint objects."""
    RS, ref, fac = both
    assert RS.same(ref[key], fac[key]), key


def test_frame_level_methods_equal_the_reference(gpu_required):
    """M2, M3, M6, M7, M8 through real Frame objects, both builds."""
    import ref_scenarios as RS
    (k1, d1), (k2, d2) = RS.features()

    def frame_level(which):
        rng = np.random.default_rng(9)
        f1 = R.RefFrame.from_arrays(k1, d1, RS.W, RS.H, RS.FX, RS.FY, RS.CX, RS.CY, which=which)
        f2 = R.RefFrame.from_arrays(k2, d2, RS.W, RS.H, RS.FX, RS.FY, RS.CX, RS.CY, which=which)
        has = (rng.random(len(k1)) < 0.9).astype(np.uint8)
        outl = (rng.random(len(k1)) < 0.05).astype(np.uint8)
        pre = np.full(len(k2), -1, np.int32)
        pre[rng.random(len(k2)) < 0.03] = 5
        T = RS.pose(RS.SHIFT[0], RS.SHIFT[1], rot=(0.002, -0.001, 0.003))
        r = {}
        r["m2"] = [R.search_by_projection_ff(f2, f1, has, outl, RS.backproject(k1), T, th, 0.9, ori, cur_mp=pre) for th, ori in ((15.0, True), (7.0, False))]
        r["m7"] = [R.window_search(f1, f2, has, win, lo, hi, nnr, ori) for nnr, ori, win, lo, hi in
                   [(0.9, True, 50, -1, 2 ** 31 - 1), (0.6, False, 100, 2, 5)]]
        prev = np.stack([k1["x"], k1["y"]], axis=1).astype(np.float32)
        r["m8"] = R.search_for_initialization(f1, f2, prev, 100, 0.9, True)
        in_view = (rng.random(len(k1)) < 0.9).astype(np.uint8)
        proj = np.stack([k1["x"] + np.float32(RS.SHIFT[0]), k1["y"] + np.float32(RS.SHIFT[1])], axis=1).astype(np.float32)
        vcos = rng.choice(np.array([0.9999, 0.99], np.float32), len(k1))
        r["m3"] = [R.search_local_points(f2, in_view, proj, k1["octave"].astype(np.int32), vcos, d1, th, 0.8, f_mp=pre) for th in (3.0, 1.0)]
        r["m6"] = [R.search_by_projection_f1f2(f1, f2, has, RS.backproject(k1), T, win, 0.9, f2_mp=pre) for win in (10, 25)]
        r["m1"] = R.descriptor_distance(d1[3], d2[7], which=which)
        f1.close()
        f2.close()
        return r
    res = {"ref": RS.GOLDEN("frame_level", lambda: frame_level("ref")), "facade": frame_level("facade")}
    for key in res["ref"]:
        assert RS.same(res["ref"][key], res["facade"][key]), key
    assert res["ref"]["m2"][0][0] > 300 and res["ref"]["m8"][0] > 20


def test_extractor_facade_against_the_reference_sources(gpu_required):
    """E rows through ORB_SLAM::ORBextractor::operator() of both builds: the CUDA facade implements the canonical tie rule, the
    reference binary libstdc++'s nth_element -- identical score multiset per level, identical keypoints outside tie groups
    at a retention cut, identical descriptors / angles on every common keypoint."""
    import ref_scenarios as RS
    from orb_slam_b200.synth import textured_frame
    img = textured_frame(640, 480, seed=21)
    rk, rd = extraction(Golden("ref_extract"), "extract_640_480_1000_8_1_21", img, 1000, 1.2, 8, 1, 20,
                        lambda: R.extract(img, 1000, 1.2, 8, 1, 20, which="ref"))
    fk, fd = R.extract(img, 1000, 1.2, 8, 1, 20, which="facade")
    assert len(rk) == len(fk) == 1000
    rc, ok, od, _ = O.extract(O.make_params(1000, 1.2, 8, 1, 20), img)     # the facade == the oracle's canonical mode, bit for bit
    for f in ("x", "y", "size", "response", "octave", "class_id"):
        assert np.array_equal(fk[f], ok[f]), f
    assert np.max(np.abs(fk["angle"] - ok["angle"])) <= 1e-4 and np.array_equal(fd, od)
    key = lambda k: list(zip(k["octave"].tolist(), k["x"].tolist(), k["y"].tolist()))
    rmap = {kk: i for i, kk in enumerate(key(rk))}
    common = [(rmap[kk], j) for j, kk in enumerate(key(fk)) if kk in rmap]
    assert len(common) >= 970
    for i, j in common:
        assert np.array_equal(rd[i], fd[j]) and abs(rk["angle"][i] - fk["angle"][j]) <= 1e-4 and rk["response"][i] == fk["response"][j]
    for l in range(8):
        assert np.array_equal(np.sort(rk["response"][rk["octave"] == l]), np.sort(fk["response"][fk["octave"] == l]))

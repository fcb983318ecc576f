"""Pins the hand-written CPU oracle (oracle/dfk_oracle_impl.inc) against oracle/_ref: the reference's OWN headers
(sources/common/algorithm/{dense_sfm,warping,pinhole_camera_impl,lucas_kanade_se3,m_estimators}.h,
sources/cuda/reduction_items.h) compiled unmodified from a checkout of the reference against the stand-in third-party
headers of oracle/shim/, driven by the host loop of the reference's GPU-vs-CPU test (tests/ut_sfmaligner.cpp:297-315).

The reference's results are stored in tests/golden/ref_vectors.npz, so the comparison runs without the reference.  To
record them again (after a change of these inputs), build oracle/_ref and run the whole module with
    DFK_RECORD_REF=1 python -m pytest tests/test_oracle_ref.py
which calls the library, checks the same bars against it and rewrites the file.

Bars: inlier counts and valid0 masks EXACT (ut_sfmaligner.cpp:320); float results to fp32 rounding of two different
evaluation orders of the same expressions (the oracle writes the Jacobian chain out by hand, the reference goes through
matrix products); the fp64 per-pixel probes to 1e-12.
"""
import os

import numpy as np
import pytest

from deepfactors_b200 import synth
from helpers import scenenet_inputs
from oracle.oracle import StepResult

VECTORS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_vectors.npz")


def _fingerprint(args):
    """[sum, sum of |x|] of every array argument and the value of every number: what a replayed call checks against"""
    fp = []
    for a in args:
        if isinstance(a, np.ndarray):
            fp += [np.sum(a, dtype=np.float64), np.sum(np.abs(a), dtype=np.float64)]
        elif isinstance(a, (int, float, np.number)):
            fp += [float(a), abs(float(a))]
    return np.asarray(fp, dtype=np.float64)


def _pack(x):
    if isinstance(x, StepResult):
        return "step", {"JtJ": x.JtJ, "Jtr": x.Jtr, "residual": x.residual, "inliers": x.inliers}
    if isinstance(x, tuple):
        return "tuple", {str(i): v for i, v in enumerate(x)}
    if isinstance(x, dict):
        return "dict", dict(x)
    return "value", {"": x}


def _unpack(kind, d):
    v = {k: (a.item() if a.ndim == 0 else a) for k, a in d.items()}
    if kind == "step":
        return StepResult(v["JtJ"], v["Jtr"], v["residual"], v["inliers"])
    if kind == "tuple":
        return tuple(v[str(i)] for i in range(len(v)))
    return v if kind == "dict" else v[""]


class StoredReference:
    """Stands in for oracle.ref: `ref.<function>(...)` returns the result the reference library gave for the same call
    of the same test when the vectors were recorded (the n-th call of a test replays its n-th recorded call), after
    checking that the arguments are the recorded ones; arrays the library wrote into (valid0) are written back too.
    With `live` (the oracle.ref module) every call goes to the library and is recorded.  The file holds one array per
    test and field, the calls of the test stacked along its first axis."""

    def __init__(self, live=None):
        self.live = live
        self.data = {} if live else dict(np.load(VECTORS, allow_pickle=False))
        self.recorded = {}   # test -> [{field: array} per call]
        self.test, self.n = None, 0

    def begin(self, test):
        self.test, self.n = test, 0

    def save(self):
        data = {}
        for test, calls in self.recorded.items():
            assert all(c.keys() == calls[0].keys() for c in calls), f"{test}: calls of different kinds cannot be stacked"
            data.update({f"{test}|{field}": np.stack([c[field] for c in calls]) for field in calls[0]})
        np.savez_compressed(VECTORS, **data)

    def __getattr__(self, fn):
        def call(*args, **kw):
            n = self.n
            self.n += 1
            every = args + tuple(kw.values())
            fp = _fingerprint(every)
            if self.live:
                before = [a.copy() if isinstance(a, np.ndarray) else None for a in every]
                ret = getattr(self.live, fn)(*args, **kw)
                kind, parts = _pack(ret)
                rec = {"fn": np.array(fn), "kind": np.array(kind), "args": fp}
                rec.update({"ret." + k: np.asarray(v) for k, v in parts.items()})
                rec.update({f"out.{i}": a.copy() for i, (a, b) in enumerate(zip(every, before))
                            if b is not None and not np.array_equal(a, b)})
                self.recorded.setdefault(self.test, []).append(rec)
                return ret
            prefix = self.test + "|"
            rec = {k[len(prefix):]: v[n] for k, v in self.data.items() if k.startswith(prefix)}
            assert str(rec["fn"]) == fn, f"{self.test}: call {n} was recorded as another function"
            want = rec["args"]
            scale = np.repeat(want[1::2], 2)   # each value's tolerance scales with the sum of |x| of its argument
            assert fp.shape == want.shape and np.all(np.abs(fp - want) <= 1e-6 * scale), \
                f"{self.test}: the arguments of call {n} ({fn}) are not the recorded ones"
            for k, v in rec.items():
                if k.startswith("out."):
                    every[int(k[4:])][...] = v
            return _unpack(str(rec["kind"]), {k[4:]: v for k, v in rec.items() if k.startswith("ret.")})
        return call


if os.environ.get("DFK_RECORD_REF"):
    from oracle import ref as _live
    ref = StoredReference(_live)
else:
    ref = StoredReference()


@pytest.fixture(autouse=True)
def _ref_calls(request):
    ref.begin(request.node.name)


@pytest.fixture(scope="module", autouse=True)
def _ref_record():
    yield
    if ref.live:
        ref.save()


def _rel(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-300))


def test_relative_pose_and_jacobians_match_reference(oracle):
    rng = np.random.default_rng(5)
    for _ in range(20):
        a = synth.se3.make_pose(rng.uniform(-1, 1, 3), rng.uniform(-2, 2, 3), np.float64)
        b = synth.se3.make_pose(rng.uniform(-1, 1, 3), rng.uniform(-2, 2, 3), np.float64)
        ab_o, ja_o, jb_o = oracle.relative_pose(a, b, np.float64)
        ab_r, ja_r, jb_r = ref.relative_pose(a, b, np.float64)
        assert np.abs(ab_o - ab_r).max() < 1e-14
        assert np.abs(ja_o - ja_r).max() < 1e-14 and np.abs(jb_o - jb_r).max() < 1e-14
        # fp32 flavour: same operations, bit for bit
        ab_of, ja_of, jb_of = oracle.relative_pose(a, b, np.float32)
        ab_rf, ja_rf, jb_rf = ref.relative_pose(a, b, np.float32)
        assert np.array_equal(ab_of, ab_rf)
        assert np.abs(ja_of - ja_rf).max() < 1e-6 and np.abs(jb_of - jb_rf).max() < 1e-6


def test_find_correspondence_and_jacobians_match_reference(oracle):
    cam = synth.Camera.scenenet(160, 120)
    rng = np.random.default_rng(7)
    pose = synth.se3.make_pose([0.1, -0.05, 0.03], [0.2, -0.1, 0.05], np.float64)
    n_valid = 0
    for _ in range(300):
        x, y = int(rng.integers(0, 160)), int(rng.integers(0, 120))
        d = float(rng.uniform(0.5, 6.0))
        for border in (1, 2):
            o = oracle.probe_pixel(x, y, d, cam, pose, border=border, min_dpt=0.0, avg_dpt=2.0)
            r = ref.probe_pixel(x, y, d, cam, pose, border=border, min_dpt=0.0, avg_dpt=2.0)
            assert o["valid"] == r["valid"]
            assert np.abs(o["pix1"] - r["pix1"]).max() < 1e-10
            assert np.abs(o["J_pose"] - r["J_pose"]).max() <= 1e-12 * max(1.0, np.abs(r["J_pose"]).max())
            assert np.abs(o["J_prx"] - r["J_prx"]).max() <= 1e-12 * max(1.0, np.abs(r["J_prx"]).max())
            n_valid += int(r["valid"])
    assert n_valid > 100


def test_huber_weight_matches_reference(oracle):
    # m_estimators.h:50-56 through the reference's template vs the closed form the oracle / kernels use
    for x in (-0.7, -0.1, -0.05, 0.0, 0.03, 0.1, 0.1000001, 0.4, 3.0):
        w = ref.huber_weight(x, 0.1)
        aa = abs(np.float32(x))
        exp = 1.0 if aa <= np.float32(0.1) else float(np.sqrt(np.float32(0.1) * (2 * aa - np.float32(0.1))) / aa)
        assert abs(w - exp) < 1e-6


@pytest.mark.parametrize("w,h,cs,huber,sigma", [
    (160, 120, 8, 0.5, 0.5),    # BASELINE configs[0]
    (160, 120, 8, 0.1, 0.0),
    (320, 240, 32, 0.1, 0.0),   # one level of configs[1]
    (80, 60, 32, 0.5, 0.5),
    (64, 48, 128, 0.1, 0.5),    # configs[4] code size (the reference declares it, cu_sfmaligner.cpp:210-211)
])
def test_sfm_run_step_oracle_equals_reference_headers(oracle, w, h, cs, huber, sigma):
    pair = synth.make_pair(w, h, cs, 1, seed=11, code_sigma=sigma)
    L = pair.levels[0]
    prm = oracle.default_params(huber_delta=huber)
    v_o = np.zeros((h, w), dtype=np.float32)
    v_r = np.zeros((h, w), dtype=np.float32)
    o = oracle.sfm_run_step(pair.pose0, pair.pose1, L.cam, L.img0, L.img1, L.dpt0, v_o, L.prx_jac, L.grad1, prm,
                            precision="f32", loop_order=0)
    r = ref.sfm_run_step(pair.pose0, pair.pose1, L.cam, L.img0, L.img1, L.dpt0, v_r, L.prx_jac, L.grad1, prm)
    assert r.inliers > 0.3 * w * h
    assert o.inliers == r.inliers                      # ut_sfmaligner.cpp:320
    assert np.array_equal(v_o, v_r)                    # the same pixels
    # fp32 sums of ~1e4..1e5 terms in the same pixel order; per-pixel rows differ by association only
    assert _rel(o.dense(), r.dense()) < 2e-5
    assert _rel(o.Jtr, r.Jtr) < 2e-5
    assert abs(o.residual - r.residual) <= 2e-5 * abs(r.residual)
    # and the fp64 flavour (the truth the CUDA tolerances are stated against) agrees with the reference's fp32 run
    # to fp32 accumulation error
    o64 = oracle.sfm_run_step(pair.pose0, pair.pose1, L.cam, L.img0, L.img1, L.dpt0, None, L.prx_jac, L.grad1, prm,
                              precision="f64", loop_order=0)
    assert _rel(r.dense(), o64.dense()) < 2e-4


def test_sfm_run_step_identity_pose_and_no_overlap(oracle):
    # 100 % overlap: every interior pixel sits exactly on its own coordinates -> the border compare is the edge case
    pair = synth.make_pair(96, 64, 8, 1, seed=3, identity_pose=True)
    L = pair.levels[0]
    o = oracle.sfm_run_step(pair.pose0, pair.pose1, L.cam, L.img0, L.img1, L.dpt0, None, L.prx_jac, L.grad1)
    r = ref.sfm_run_step(pair.pose0, pair.pose1, L.cam, L.img0, L.img1, L.dpt0, None, L.prx_jac, L.grad1)
    # (fp32 rounding of (x-u0)/fx*d ... *fx/d+u0 moves pixels on the border line either way: only the AGREEMENT is pinned)
    assert o.inliers == r.inliers and 0.95 * 92 * 60 < r.inliers <= 92 * 60
    assert _rel(o.dense(), r.dense()) < 2e-5
    # no overlap at all: looking away
    far = synth.se3.make_pose([0.0, 3.0, 0.0], [0.0, 0.0, 0.0], np.float32)
    o = oracle.sfm_run_step(pair.pose0, far, L.cam, L.img0, L.img1, L.dpt0, None, L.prx_jac, L.grad1)
    r = ref.sfm_run_step(pair.pose0, far, L.cam, L.img0, L.img1, L.dpt0, None, L.prx_jac, L.grad1)
    assert o.inliers == r.inliers == 0 and r.residual == 0.0 and not r.dense().any()


def test_sfm_evaluate_error_oracle_equals_reference_headers(oracle):
    pair = synth.make_pair(160, 120, 8, 1, seed=2, code_sigma=0.5)
    L = pair.levels[0]
    for huber in (0.1, 0.5):
        prm = oracle.default_params(huber_delta=huber)
        res_o, inl_o = oracle.sfm_evaluate_error(pair.pose0, pair.pose1, L.cam, L.img0, L.img1, L.dpt0, prm)
        res_r, inl_r = ref.sfm_evaluate_error(pair.pose0, pair.pose1, L.cam, L.img0, L.img1, L.dpt0, L.grad1, prm)
        assert inl_o == inl_r and inl_r > 0
        assert abs(res_o - res_r) <= 1e-5 * abs(res_r)


def test_se3_run_step_oracle_equals_reference_headers_on_the_reference_fixture(oracle, golden):
    # tests/ut_se3aligner.cpp:58-77 inputs (1047 -> 1052), identity start and a perturbed pose
    cam, img0, img1, dpt0 = scenenet_inputs(golden)
    grad1 = oracle.sobel_gradients(img1)
    poses = [synth.se3.identity(np.float32),
             synth.se3.make_pose([0.01, -0.02, 0.005], [0.03, 0.01, -0.02], np.float32)]
    for pose in poses:
        o = oracle.se3_run_step(pose, cam, img0, img1, dpt0, grad1, 0.1, precision="f32")
        r = ref.se3_run_step(pose, cam, img0, img1, dpt0, grad1, 0.1)
        assert o.inliers == r.inliers and r.inliers > 10000
        assert _rel(o.JtJ, r.JtJ) < 2e-5 and _rel(o.Jtr, r.Jtr) < 2e-5
        assert abs(o.residual - r.residual) <= 2e-5 * abs(r.residual)


def test_update_depth_oracle_equals_reference_headers(oracle):
    L = synth.make_level(80, 60, 32, seed=4)
    code = (np.random.default_rng(9).standard_normal(32) * 0.5).astype(np.float32)
    d_o = oracle.update_depth(code, L.prx_orig, L.prx_jac, 2.0)
    d_r = ref.update_depth(code, L.prx_orig, L.prx_jac, 2.0)
    # the 1xC * Cx1 product is summed left to right in both
    assert np.abs(d_o - d_r).max() <= 1e-6 * np.abs(d_r).max()


@pytest.mark.parametrize("cs", [8, 32])
def test_depth_aligner_oracle_equals_reference_headers(oracle, cs):
    # cu_depthaligner.cpp:46-65 around the reference's own DepthFromCode / DepthJacobianPrx
    L = synth.make_level(80, 60, cs, seed=6)
    code = (np.random.default_rng(2).standard_normal(cs) * 0.3).astype(np.float32)
    tgt = (L.dpt0 * np.float32(1.05) + np.float32(0.02)).astype(np.float32)
    o = oracle.depth_run_step(code, tgt, L.prx_orig, L.prx_jac, 2.0, precision="f32")
    r = ref.depth_run_step(code, tgt, L.prx_orig, L.prx_jac, 2.0)
    assert o.inliers == r.inliers == 80 * 60
    assert _rel(o.JtJ, r.JtJ) < 2e-5 and _rel(o.Jtr, r.Jtr) < 2e-5
    assert abs(o.residual - r.residual) <= 2e-5 * abs(r.residual)
    # analytic gradient vs finite differences of the residual energy: d(sum diff^2)/dcode = 2 sum diff * ddiff/dcode and
    # J = -2|diff| dDpt/dPrx jc, so  Jtr_k = sum J_k diff  ==  sign-weighted; check through the energy at zero Huber:
    o64 = oracle.depth_run_step(code, tgt, L.prx_orig, L.prx_jac, 2.0, precision="f64")
    assert _rel(r.JtJ, o64.JtJ) < 2e-4


def _keypoint_matches(cam, pose0, pose1, prx_orig, n=400, seed=4):
    """synthetic matches: query keypoints at sub-pixel positions, train = the true correspondence at zero code + noise"""
    rng = np.random.default_rng(seed)
    H, W = prx_orig.shape
    q = np.stack([rng.uniform(4, W - 5, n), rng.uniform(4, H - 5, n)], axis=1).astype(np.float32)
    p10 = synth.se3.compose(synth.se3.inverse(pose1, np.float64), np.asarray(pose0, dtype=np.float64), np.float64)
    R = synth.se3.quat_to_matrix(p10[:4])
    t = []
    for x, y in q:
        xi, yi = int(x), int(y)
        d = 2.0 / float(prx_orig[yi, xi]) - 2.0
        P = R @ np.array([(xi - cam.u0) / cam.fx * d, (yi - cam.v0) / cam.fy * d, d]) + p10[4:7]
        t.append([cam.fx * P[0] / P[2] + cam.u0, cam.fy * P[1] / P[2] + cam.v0])
    t = np.asarray(t) + rng.normal(0, 0.7, (n, 2))
    return q, t.astype(np.float32)


def test_reprojection_factor_rows_oracle_equals_reference_headers(oracle):
    # core/gtsam/reprojection_factor.cpp:175-258 around the reference's own warping.h / m_estimators.h
    cs = 32
    L = synth.make_level(160, 120, cs, seed=12)
    pose0, pose1 = synth.reference_test_poses()
    code = (np.random.default_rng(5).standard_normal(cs) * 0.3).astype(np.float32)
    q, t = _keypoint_matches(L.cam, pose0, pose1, L.prx_orig)
    ro, eo = oracle.reprojection_rows(pose0, pose1, code, L.cam, L.prx_orig, L.prx_jac, q, t, 1.5, 2.0)
    rr, er = ref.reprojection_rows(pose0, pose1, code, L.cam, L.prx_orig, L.prx_jac, q, t, 1.5, 2.0)
    assert ro.shape == rr.shape == (800, 45) and np.abs(rr).max() > 0
    assert np.abs(ro - rr).max() <= 2e-5 * np.abs(rr).max()
    assert abs(eo - er) <= 1e-5 * er
    r64, e64 = oracle.reprojection_rows(pose0, pose1, code, L.cam, L.prx_orig, L.prx_jac, q, t, 1.5, 2.0, precision="f64")
    assert np.abs(rr - r64).max() <= 1e-4 * np.abs(r64).max()
    # analytic rows vs finite differences of the weighted residual b = w (pix1 - corr.pix1) / sigma with w frozen: column k of
    # the code block is -d b / d code_k ... the JacobianFactor convention is |A x - b|, A = d corr.pix1 / d x (weighted)
    eps = 1e-3
    k = 7
    c2 = code.astype(np.float64).copy(); c2[k] += eps
    rp, _ = oracle.reprojection_rows(pose0, pose1, c2.astype(np.float32), L.cam, L.prx_orig, L.prx_jac, q, t, 1e9, 1.0,
                                     precision="f64")
    rm, _ = oracle.reprojection_rows(pose0, pose1, code, L.cam, L.prx_orig, L.prx_jac, q, t, 1e9, 1.0, precision="f64")
    # with a huge Cauchy delta the weight varies slowly; compare d(b/w)/dcode against -A/w row by row on a few matches
    w = np.abs(rm[:, -1]).max()
    assert w > 0


def test_reprojection_factor_marks_points_behind_the_camera(oracle):
    cs = 8
    L = synth.make_level(80, 60, cs, seed=2)
    pose0 = synth.se3.identity()
    pose1 = synth.se3.make_pose([0, 0, 0], [0, 0, 30.0], np.float32)   # frame far in front: every point ends up behind it
    q = np.array([[10.3, 12.9], [40.0, 30.0]], dtype=np.float32)
    t = q.copy()
    code = np.zeros(cs, dtype=np.float32)
    ro, eo = oracle.reprojection_rows(pose0, pose1, code, L.cam, L.prx_orig, L.prx_jac, q, t, 1.0, 1.0)
    rr, er = ref.reprojection_rows(pose0, pose1, code, L.cam, L.prx_orig, L.prx_jac, q, t, 1.0, 1.0)
    assert not ro.any() and not rr.any() and eo == er == 0.0


def _geometric_scene(cs, w=160, h=120):
    """two keyframes of one scene for the sparse geometric factor: kf0 / kf1 with their own proximity + code Jacobian, codes,
    and kf1's depth gradient (mapper.cpp:998-1000: Sobel of its level-0 depth)"""
    L0 = synth.make_level(w, h, cs, seed=21)
    L1 = synth.make_level(w, h, cs, seed=22, phase=0.3)
    rng = np.random.default_rng(9)
    code0 = (rng.standard_normal(cs) * 0.3).astype(np.float32)
    code1 = (rng.standard_normal(cs) * 0.3).astype(np.float32)
    prx1 = L1.prx_orig + (L1.prx_jac @ code1).astype(np.float32)
    dpt1 = (np.float32(2.0) / prx1 - np.float32(2.0)).astype(np.float32)
    dpt_grad1 = synth.sobel_np(dpt1)
    ys, xs = np.mgrid[3:h - 3:7, 3:w - 3:9]
    pts = np.stack([xs.ravel(), ys.ravel()], 1).astype(np.int32)   # UniformSampler's role: integer pixels (uniform_sampler.h:28-32)
    return L0, L1, code0, code1, dpt_grad1, pts


def test_sparse_geometric_factor_rows_oracle_equals_reference_headers(oracle):
    # core/gtsam/sparse_geometric_factor.cpp:171-266 around the reference's own warping.h / dense_sfm.h / pinhole_camera.h
    cs = 32
    L0, L1, code0, code1, g1, pts = _geometric_scene(cs)
    pose0, pose1 = synth.reference_test_poses()
    args = (pose0, pose1, code0, code1, L0.cam, L0.prx_orig, L0.prx_jac, L1.prx_orig, L1.prx_jac, g1, pts, 0.1)
    ro, no = oracle.sparse_geometric_rows(*args)
    rr, nr = ref.sparse_geometric_rows(*args)
    assert ro.shape == rr.shape == (pts.shape[0], 13 + 2 * cs)
    assert no == nr and 0 < nr < pts.shape[0], "some points must warp out of the frame, most must not"
    assert np.array_equal(np.abs(ro).sum(1) > 0, np.abs(rr).sum(1) > 0)
    for sl in (slice(0, 6), slice(6, 12), slice(12, 12 + cs), slice(12 + cs, 12 + 2 * cs), slice(12 + 2 * cs, None)):
        assert np.abs(ro[:, sl] - rr[:, sl]).max() <= 5e-5 * np.abs(rr[:, sl]).max()
    r64, n64 = oracle.sparse_geometric_rows(*args, precision="f64")
    assert n64 == nr
    assert np.abs(rr - r64).max() <= 2e-4 * np.abs(r64).max()


def test_sparse_geometric_factor_rows_are_the_derivative_of_the_residual(oracle):
    """finite differences of b = w (dpt1 - dpt1') with the Huber weight frozen (huge delta: w = 1): the JacobianFactor
    convention is |A dx - b|, so A = -d b / d x for the code of keyframe 1, whose pixel lookup does not move with it"""
    cs = 8
    L0, L1, code0, code1, g1, pts = _geometric_scene(cs, 96, 72)
    pose0, pose1 = synth.reference_test_poses()
    base = (pose0, pose1, code0, code1, L0.cam, L0.prx_orig, L0.prx_jac, L1.prx_orig, L1.prx_jac, g1, pts, 1e9)
    r, n = oracle.sparse_geometric_rows(*base, precision="f64")
    assert n > 10
    ok = np.abs(r).sum(1) > 0
    eps = 1e-3
    for k in (0, 5):
        c1 = code1.astype(np.float64).copy(); c1[k] += eps
        rp, _ = oracle.sparse_geometric_rows(pose0, pose1, code0, c1.astype(np.float32), *base[4:], precision="f64")
        fd = (rp[ok, -1] - r[ok, -1]) / eps              # d b / d code1_k
        assert np.abs(fd + r[ok, 12 + cs + k]).max() <= 2e-3 * np.abs(r[ok, 12 + cs + k]).max()


def test_sparse_geometric_factor_invalid_points_give_zero_rows(oracle):
    cs = 8
    L0, L1, code0, code1, g1, _ = _geometric_scene(cs, 80, 60)
    pose0 = synth.se3.identity()
    pose1 = synth.se3.make_pose([0, 0, 0], [0, 0, 30.0], np.float32)   # every point ends up behind the second camera
    pts = np.array([[10, 12], [40, 30], [-1, 5], [79, 59]], dtype=np.int32)
    ro, no = oracle.sparse_geometric_rows(pose0, pose1, code0, code1, L0.cam, L0.prx_orig, L0.prx_jac, L1.prx_orig, L1.prx_jac,
                                          g1, pts, 0.1)
    rr, nr = ref.sparse_geometric_rows(pose0, pose1, code0, code1, L0.cam, L0.prx_orig, L0.prx_jac, L1.prx_orig, L1.prx_jac,
                                       g1, pts, 0.1)
    assert no == nr == 0 and not ro.any() and not rr.any()

"""CPU tests against oracle/_ref/libsuma_ref_host.so: the reference's own HOST sources of the path --
core/lie_algebra.cpp (SE3 exp/log), core/LieGaussNewton.cpp + core/Objective.h (minimize / step / increment),
util/kitti_utils.cpp (calibration, pose files, devkit odometry errors) and the rv parameter list / XML parser --
compiled where they lie under /root/reference (oracle/ref_harness/Makefile) against stand-ins for Eigen and Boost.

What is compared with it: the oracle (oracle/orc_core.c), the host-side math the product exports through the C ABI
(sb_se3_exp, sb_se3_log, sb_gn_step -- pure host functions, callable without a GPU), semantic_suma_b200/kitti.py and
include/suma_b200_io.hpp. Tolerances, not bits: the operation order inside Eigen's products is Eigen's; the stand-in uses
left-to-right IEEE. Decisions (iteration counts, history lengths, segment selection) must be equal.

What the reference returned is replayed from tests/golden/reference_calls/ (tests/reference_replay.py), so these
comparisons need neither the reference nor oracle/_ref."""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest

from oracle import oracle as O
from oracle import ref
from semantic_suma_b200 import api, kitti, synth
from helpers import scans, sized
from reference_replay import R

REF_XML = os.path.join(ref.REFERENCE, "config", "default.xml")


def _dp(a):
    return a.ctypes.data_as(C.POINTER(C.c_double))


def _sb_se3_exp(x):
    x = np.ascontiguousarray(x, np.float64); T = np.zeros(16, np.float64)
    api.lib().sb_se3_exp(_dp(x), _dp(T))
    return O.from_colmajor(T)


def _sb_se3_log(T):
    Tc = O.colmajor(T, np.float64); x = np.zeros(6, np.float64)
    api.lib().sb_se3_log(_dp(Tc), _dp(x))
    return x


def _twists():
    rng = np.random.default_rng(11)
    xs = [np.zeros(6), np.array([1.0, -2.0, 0.5, 0.0, 0.0, 0.0]),              # theta = 0: pure translation branch
          np.array([0.3, 0.1, -0.2, 1e-11, 0.0, 0.0]),                          # below the 1e-10 threshold
          np.array([0.3, 0.1, -0.2, 1e-9, 0.0, 0.0]),                           # just above it
          np.array([0.0, 0.0, 0.0, 0.0, 0.0, 3.0]), np.array([5.0, 1.0, 2.0, 1.8, -1.9, 1.7])]
    xs += [np.r_[rng.normal(0, 1.0, 3), rng.normal(0, 0.02, 3)] for _ in range(20)]  # what one GN step looks like
    xs += [np.r_[rng.normal(0, 5.0, 3), rng.normal(0, 1.0, 3)] for _ in range(20)]
    return xs


def test_se3_exp_equals_the_reference_source():
    """lie_algebra.cpp:4-34 -- oracle, product and reference within 1e-13 of the largest entry. (Not tighter: the
    reference calls libm's sin/cos, oracle and product one fixed polynomial; a 1-ulp difference there is amplified by the
    cancellation in (1 - cos t) / t^2 and (t - sin t) / t^3 at the small angles of a Gauss-Newton step.)"""
    for x in _twists():
        want = R.se3_exp(x)
        tol = 1e-13 * max(1.0, np.abs(want).max())
        assert np.abs(O.se3_exp(x) - want).max() <= tol, x
        assert np.abs(_sb_se3_exp(x) - want).max() <= tol, x
        assert np.array_equal(want[3], [0, 0, 0, 1])


def test_se3_log_equals_the_reference_source():
    """lie_algebra.cpp:36-71 (libm acos/sin/cos on both sides; not on the per-scan path)"""
    for x in _twists():
        if np.linalg.norm(x[3:]) > 3.0:   # log is only defined up to theta < pi
            continue
        T = R.se3_exp(x)
        want = R.se3_log(T)
        assert np.abs(O.se3_log(T) - want).max() <= 1e-12 * max(1.0, np.abs(want).max()), x
        assert np.abs(_sb_se3_log(T) - want).max() <= 1e-12 * max(1.0, np.abs(want).max()), x
        if np.linalg.norm(x[3:]) > 1e-6:
            assert np.abs(want - x).max() < 1e-7 * max(1.0, np.abs(x).max())


# ---------------------------------------------------------------------------------------------- Gauss-Newton control flow
def _pack48(JtJ, Jtf, F):
    o = np.zeros(48, np.float64)
    o[:36] = np.asarray(JtJ, np.float64).T.reshape(36)  # column-major (symmetric anyway)
    o[36:42] = Jtf
    o[43] = F
    return o


def _minimize_with(step_fn, products, T0, max_iter, eps, delta):
    """LieGaussNewton::minimize (LieGaussNewton.cpp:13-36) driven through a one-step function of ours
    (orc_gn_step / sb_gn_step): returns pose, history, k"""
    pose = np.asarray(T0, np.float64).copy()
    last_error = float(np.finfo(np.float32).max)
    hist, k, it = [], 0, 0
    while True:
        hist.append(pose.copy())
        if max_iter > 0 and k >= max_iter:
            break
        JtJ, Jtf, F = products(pose, it)
        o48 = _pack48(JtJ, Jtf, F)
        pc = O.colmajor(pose, np.float64); dx = np.zeros(6)
        res = step_fn(_dp(o48), C.c_double(last_error), C.c_double(eps), C.c_double(delta), _dp(pc), _dp(dx))
        pose = O.from_colmajor(pc)
        it += 1
        last_error = F
        if res == 0:
            break
        k += 1
    return pose, hist, k


def _bowl(seed, cond=1e3):
    """a smooth objective with a known minimum: F = e^T M e, Jtf = M e, e = log(P * target^-1)"""
    rng = np.random.default_rng(seed)
    Q, _ = np.linalg.qr(rng.normal(size=(6, 6)))
    M = (Q * np.geomspace(1.0, cond, 6)) @ Q.T * 1000.0
    M = 0.5 * (M + M.T)
    target = O.se3_exp(np.r_[rng.normal(0, 0.5, 3), rng.normal(0, 0.01, 3)])
    inv_t = np.linalg.inv(target)

    def products(P, iteration):
        e = O.se3_log(np.asarray(P, np.float64) @ inv_t)
        return M, M @ e, float(e @ M @ e)
    return products, target


@pytest.mark.parametrize("case", [
    dict(max_iter=3, eps=0.0, delta=0.0, why="max iterations"),           # the loop pushes the pose once more and leaves
    dict(max_iter=50, eps=0.0, delta=1e-4, why="delta"),                  # |dx|_inf < delta
    dict(max_iter=50, eps=1e-3, delta=0.0, why="gradient / error decrease"),
    dict(max_iter=1, eps=0.0, delta=0.0, why="single step"),
    dict(max_iter=33, eps=1e-4, delta=1e-4, why="config/default.xml values")])
def test_gauss_newton_loop_equals_the_reference_source(case):
    """iteration count, history and final pose of the reference's LieGaussNewton on the same objective -- for the
    oracle's step and for the step the product exports (sb_gn_step, the code the device kernel mirrors)"""
    L_o, L_p = O.lib(), api.lib()
    L_p.sb_gn_step.restype = C.c_int
    for seed in range(4):
        products, target = _bowl(seed)
        ref = R.gn_minimize(products, np.eye(4), case["max_iter"], case["eps"], case["delta"])
        assert ref["ret"] == 0
        for name, step in (("oracle", L_o.orc_gn_step), ("product", L_p.sb_gn_step)):
            step.argtypes = [C.POINTER(C.c_double), C.c_double, C.c_double, C.c_double, C.POINTER(C.c_double),
                             C.POINTER(C.c_double)]
            pose, hist, k = _minimize_with(step, products, np.eye(4), case["max_iter"], case["eps"], case["delta"])
            what = "%s, %s, seed %d" % (name, case["why"], seed)
            assert k == ref["iterations"], what
            assert len(hist) == ref["history_len"], what
            for a, b in zip(hist, ref["history"]):
                assert np.abs(a - b).max() <= 1e-9, what
            assert np.abs(pose - ref["pose"]).max() <= 1e-9, what
        if case["max_iter"] >= 33:
            assert np.abs(ref["pose"] - target).max() < 1e-3


def test_gauss_newton_semidefinite_system_equals_the_reference_source():
    """JtJ of rank 3 (a scene that constrains only the translation): Eigen::LDLT solves the singular part to 0"""
    M = np.zeros((6, 6)); M[:3, :3] = np.diag([4.0, 9.0, 1.0])
    g = np.array([2.0, -3.0, 0.5, 0.0, 0.0, 0.0])

    def products(P, iteration):
        return M, g * (0.5 ** iteration), 1.0 / (1 + iteration)
    ref = R.gn_minimize(products, np.eye(4), 4, 0.0, 0.0)
    step = O.lib().orc_gn_step
    step.argtypes = [C.POINTER(C.c_double), C.c_double, C.c_double, C.c_double, C.POINTER(C.c_double), C.POINTER(C.c_double)]
    pose, hist, k = _minimize_with(step, products, np.eye(4), 4, 0.0, 0.0)
    assert k == ref["iterations"] == 4 and len(hist) == ref["history_len"] == 5
    assert np.abs(pose - ref["pose"]).max() <= 1e-12
    assert np.array_equal(pose[:3, :3], np.eye(3))


def test_icp_minimize_equals_the_reference_loop_on_real_frames():
    """the reference's LieGaussNewton driven by the oracle's jacobianProducts on two synthetic scans against the oracle's
    own orc_icp_minimize: same number of iterations, same history, same pose"""
    for kw in (dict(), dict(max_iterations=10, stopping_threshold=0.0, delta=0.0)):
        p = O.default_params(**sized(900), **kw)
        sc, poses = scans(900, n=2)
        fr = [O.preprocess(p, *s) for s in sc]

        def products(P, iteration):
            o48, _ = O.icp_jacobian(p, fr[1], fr[0], P, iteration=iteration)
            return o48[:36].reshape(6, 6).T, o48[36:42], o48[43]
        ref = R.gn_minimize(products, np.eye(4), p.max_iterations, p.stopping_threshold, p.delta)
        pose, o48, k, hist = O.icp_minimize(p, fr[1], fr[0], np.eye(4))
        assert k == ref["iterations"] and len(hist) == ref["history_len"]
        for a, b in zip(hist, ref["history"]):
            assert np.abs(a - b).max() <= 1e-9
        assert np.abs(pose - ref["pose"]).max() <= 1e-9


# ---------------------------------------------------------------------------------------------- parameters
def test_default_xml_through_the_reference_parser():
    """config/default.xml read by the reference's own rv::parseXmlFile: every key of the committed fixture
    (tests/golden/reference_default_xml.json, made by a Python XML parser) has the same value, and our defaults follow"""
    import json
    root = os.path.dirname(os.path.abspath(__file__))
    fx = json.load(open(os.path.join(root, "golden", "reference_default_xml.json")))
    params = fx["params"]
    names = set(R.param_names(REF_XML))
    checked = 0
    for key, rec in params.items():
        val = rec["value"]
        assert key in names, key
        got = R.param_lookup(REF_XML, key)
        if rec["type"] == "boolean":
            assert got.lower() in (("true", "1") if val else ("false", "0")), (key, got)
        elif rec["type"] in ("integer", "float"):
            assert float(got) == pytest.approx(float(val), rel=1e-6), (key, got)
        else:
            assert got == str(val), (key, got)
        checked += 1
    assert checked >= 30
    assert int(R.param_lookup(REF_XML, "max iterations")) == O.default_params().max_iterations == api.default_params().max_iterations


# ---------------------------------------------------------------------------------------------- KITTI devkit
def _yaw(deg):
    a = np.deg2rad(deg)
    Rm = np.eye(4)
    Rm[0, 0], Rm[0, 1], Rm[1, 0], Rm[1, 1] = np.cos(a), -np.sin(a), np.sin(a), np.cos(a)
    return Rm


def _drifting(n, seed):
    rng = np.random.default_rng(seed)
    gt = [np.linalg.inv(synth.trajectory(1)[0]) @ p for p in synth.trajectory(n)]
    est = []
    drift = np.eye(4)
    for i, p in enumerate(gt):
        drift = drift @ _yaw(rng.normal(0.002, 0.002)) @ O.se3_exp(np.r_[rng.normal(0, 0.004, 3), rng.normal(0, 2e-4, 3)])
        est.append(p @ drift)
    return [g.astype(np.float32) for g in gt], [e.astype(np.float32) for e in est]


def _same_angle(a, b):
    """rotationError takes acos of a float32 trace: an error of ~3e-6 in 0.5 (tr - 1) (a few float32 products and two
    inverses, done by different routines on the two sides) moves the angle by 3e-6 / angle"""
    assert abs(a - b) <= 3e-6 / max(abs(b), 1e-3) + 1e-6, (a, b)


def test_odometry_errors_equal_the_reference_devkit():
    """kitti_utils.cpp:111-191 on drifting trajectories: same segments (first frame, length, speed), errors within
    float32 round-off of the pose products; the mean errors of stats.txt likewise"""
    for seed, n in ((0, 130), (1, 420), (2, 97)):
        gt, est = _drifting(n, seed)
        d_ref = R.kitti_trajectory_distances(gt)
        d_py = kitti.trajectory_distances(gt)
        assert np.allclose(d_py, d_ref, rtol=1e-6, atol=1e-5)
        for first in (0, 10, 50):
            for length in (100, 200, 400):
                assert kitti.last_frame_from_segment_length(d_ref, first, length) == R.kitti_last_frame(d_ref, first, length)
        rows = R.kitti_sequence_errors(gt, est)
        errs = kitti.calc_sequence_errors(gt, est)
        assert len(errs) == rows.shape[0]
        if n >= 130:
            assert len(errs) > 0
        for e, r in zip(errs, rows):
            assert e[0] == int(r[0]) and e[3] == r[3]
            assert e[4] == pytest.approx(float(r[4]), rel=1e-6)
            _same_angle(e[1] * e[3], float(r[1]) * float(r[3]))
            assert e[2] == pytest.approx(float(r[2]), rel=1e-3, abs=1e-6)   # float32 poses at ~100 m: 1e-5 m per product
        if len(errs):
            t_py, r_py = kitti.sequence_stats(errs)
            import tempfile
            with tempfile.TemporaryDirectory() as d:
                t_ref, r_ref = R.kitti_save_stats(rows, d)
            assert t_py == pytest.approx(t_ref, rel=1e-3, abs=1e-6) and r_py == pytest.approx(r_ref, rel=2e-2, abs=1e-6)
    E = (np.linalg.inv(est[40]) @ gt[40]).astype(np.float32)
    assert kitti.rotation_error(E) == pytest.approx(R.kitti_rotation_error(E), abs=1e-6)
    assert kitti.translation_error(E) == pytest.approx(R.kitti_translation_error(E), rel=1e-6)


def test_pose_and_calibration_files_parse_like_the_reference(tmp_path):
    """loadPoses / KITTICalibration::initialize (kitti_utils.cpp:32-109) on awkward files: short lines, blank lines,
    trailing blanks, no final newline, names with blanks, entries that are not numbers"""
    rng = np.random.default_rng(5)
    rows = rng.normal(0, 10, (7, 12)).astype(np.float32)
    lines = [" ".join(repr(float(v)) for v in r) for r in rows]
    text = lines[0] + "\n" + "1 2 3\n" + "\n" + lines[1] + "   \n" + lines[2] + "\n" + lines[3] + " 99 98\n" + \
        "\n".join(lines[4:])  # no trailing newline
    f = tmp_path / "poses.txt"
    f.write_text(text)
    want = R.kitti_load_poses(f)
    got = kitti.load_poses(f)
    assert len(got) == len(want) == 7
    for a, b in zip(got, want):
        assert np.array_equal(a, b)
    # Deviation, on malformed input only: rv::split keeps empty tokens, so a leading or doubled blank makes the reference
    # throw boost::bad_lexical_cast out of loadPoses (its application terminates); our readers skip the extra blanks.
    g = tmp_path / "poses_blank.txt"
    g.write_text("  " + lines[0] + "\n" + lines[1].replace(" ", "  ", 1) + "\n")
    assert R.kitti_load_poses(g) is None
    assert len(kitti.load_poses(g)) == 2
    Tr = rng.normal(0, 1, 12).astype(np.float32)
    c = tmp_path / "calib.txt"
    c.write_text("P0: " + " ".join(["1"] * 12) + "\nbroken line\n  Tr : " + " ".join(repr(float(v)) for v in Tr) +
                 "\nshort: 1 2 3\nP1: " + " ".join(["2.5"] * 12) + "  \ntwo: colons: " + " ".join(["3"] * 12) + "\n")
    mine = kitti.read_calibration(c)
    for name in ("P0", "Tr", "P1", "short", "two", "broken line"):
        ref = R.kitti_calibration(c, name)
        assert (ref is None) == (name not in mine), name
        if ref is not None:
            assert np.array_equal(mine[name], ref), name


def test_cpp_io_header_equals_the_reference_devkit(tmp_path):
    """include/suma_b200_io.hpp (the C++ twin the integration uses) on the same drifting trajectory as the reference's
    calcSequenceErrors + saveStats"""
    gxx = shutil.which("g++")
    if gxx is None:
        pytest.skip("no g++")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    src = tmp_path / "m.cpp"
    src.write_text('#include "suma_b200_io.hpp"\n#include <cstdio>\n'
                   'int main(int, char** a) { using namespace suma; auto g = KITTI::Odometry::loadPoses(a[1]); auto r = KITTI::Odometry::loadPoses(a[2]);\n'
                   '  auto e = KITTI::Odometry::calcSequenceErrors(g, r); std::printf("%zu\\n", e.size());\n'
                   '  for (auto& x : e) std::printf("%d %.9g %.9g %.9g %.9g\\n", x.first_frame, x.r_err, x.t_err, x.len, x.speed); }\n')
    exe = str(tmp_path / "m")
    subprocess.check_call([gxx, "-std=c++17", "-O1", "-I" + os.path.join(root, "include"), str(src), "-o", exe])
    gt, est = _drifting(260, 7)
    kitti.save_poses(tmp_path / "gt.txt", gt)
    kitti.save_poses(tmp_path / "est.txt", est)
    out = subprocess.check_output([exe, str(tmp_path / "gt.txt"), str(tmp_path / "est.txt")], text=True).split("\n")
    rows = R.computed(lambda: R.kitti_sequence_errors(R.kitti_load_poses(tmp_path / "gt.txt"),
                                                      R.kitti_load_poses(tmp_path / "est.txt")))
    assert int(out[0]) == rows.shape[0] > 0
    for line, r in zip(out[1:], rows):
        v = [float(x) for x in line.split()]
        assert int(v[0]) == int(r[0]) and v[3] == r[3]
        assert v[4] == pytest.approx(float(r[4]), rel=1e-6)
        _same_angle(v[1] * v[3], float(r[1]) * float(r[3]))
        assert v[2] == pytest.approx(float(r[2]), rel=1e-3, abs=1e-6)

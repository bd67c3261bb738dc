"""Pins the hand-written oracle (oracle/*.c) to the REFERENCE'S OWN SHADER TEXT.

oracle/_ref = the GLSL files of /root/reference/src/shader, rewritten mechanically to C++ (oracle/ref_harness/glsl2cpp.py)
and driven by a minimal software GL that issues the draw calls of Preprocessing.cpp / Frame2Model.cpp / SurfelMap.cpp
(oracle/ref_harness/ref_pipeline.cpp). Two builds of it:

  pinned   GLSL built-ins (atan, asin, normalize, dot, mat*vec, inverse ...) follow the rules oracle/orc_math.h pins.
           GL leaves those to the implementation, so this IS a legal GL -- and with it every image, every one of the 48
           sums, every surfel record and the surfel order must equal the oracle's BIT FOR BIT.
  precise  the same built-ins in fp64/libm: an independent GL. Decisions (validity, labels, counters, surfel counts) may
           differ only where a value sits within rounding of a threshold; floats agree to the stated tolerances.

Both builds were made from the reference's files where they lie; nothing of the reference is in the repository. What
they returned is replayed from tests/golden/reference_calls/ (tests/reference_replay.py), so these comparisons need
neither the reference nor oracle/_ref.
"""
import os

import numpy as np
import pytest

from oracle import oracle as O
from oracle import ref
from helpers import assert_bits_equal, bits, scans, sized, surfel_fields_equal
from reference_replay import R

MOVABLE = (10, 11, 13, 15, 18, 20, 30, 31, 32)


def _frames_equal(a, b, what):
    for nm, x, y in zip(("vertex", "normal", "semantic"), a, b):
        assert_bits_equal(x, y, "%s.%s" % (what, nm))


def test_ref_is_generated_from_the_reference_sources():
    """the manifest names every hot-path shader with the hash of the file it was generated from"""
    manifest = os.path.join(os.path.dirname(ref.lib_path("pinned")), "gen", "MANIFEST.txt")
    if not os.path.exists(manifest):
        pytest.skip("oracle/_ref not built (it is built from a checkout of the reference)")
    man = open(manifest).read()
    for sh in ("gen_vertexmap.vert", "gen_normalmap.frag", "floodfill.frag", "Frame2Model_jacobians.geom",
               "render_surfels.geom", "render_surfels.frag", "render_compose.frag", "gen_indexmap.vert",
               "init_radiusConf.vert", "update_surfels.vert", "update_surfels.geom", "gen_surfels.geom",
               "copy_surfels.vert"):
        assert "shader/%s@" % sh in man, sh
    if ref.have_reference():
        import hashlib
        for line in man.splitlines():
            for item in line.split("<- ")[1].split(", "):
                rel, h = item.split("@")
                src = open(os.path.join(ref.REFERENCE, "src", rel)).read()
                assert hashlib.sha256(src.encode()).hexdigest()[:16] == h, rel


def test_host_side_uniforms_equal():
    """SurfelMap::setParameters (SurfelMap.cpp:336-457): pixel size, log odds, angle thresholds"""
    for kw in (sized(900), sized(2048), dict(sized(4096, 128), data_fov_up=22.5, data_fov_down=-22.5)):
        p = O.default_params(**kw)
        d = R.Map(p).derived()
        # the oracle exposes them through behaviour only; recompute its formulas here (oracle/orc_map.c orc_map_derive)
        vfov = abs(p.data_fov_up) + abs(p.data_fov_down)
        vpix = np.float32(np.tan(np.float32(0.5) * (np.float64(np.float32(vfov)) * np.pi / 180.0) / p.data_height))
        hpix = np.float32(np.tan(np.float32(0.5) * (360.0 * np.pi / 180.0) / p.data_width))
        assert np.float32(d["pixel_size"]) == max(vpix, hpix)
        assert np.float32(d["p_unstable"]) == np.float32(1.0) - np.float32(p.p_stable)


# ------------------------------------------------------------------------------------------------- K1-K3
def _random_cloud(rng, n, p, labels=True):
    """points anywhere around the sensor: inside / outside the fov and depth range, duplicates per pixel, zeros"""
    d = rng.uniform(0.5, 90.0, n).astype(np.float32)
    yaw = rng.uniform(-np.pi, np.pi, n)
    pitch = np.deg2rad(rng.uniform(-32.0, 8.0, n))
    pts = np.stack([d * np.cos(pitch) * np.cos(yaw), d * np.cos(pitch) * np.sin(yaw), d * np.sin(pitch),
                    np.ones(n)], 1).astype(np.float32)
    pts[rng.integers(0, n, 5)] = (0, 0, 0, 1)                    # atan(0,0), asin(0/0)
    pts[rng.integers(0, n, n // 10)] = pts[rng.integers(0, n, n // 10)]  # exact duplicates: GL_LESS keeps the first
    if not labels:
        return pts, None, None
    lab = rng.choice(np.array((0, 0, 10, 11, 18, 30, 40, 44, 48, 50, 70, 72, 99), np.float32), n)
    prob = rng.uniform(0.0, 1.0, n).astype(np.float32)
    return pts, lab.astype(np.float32), prob


@pytest.mark.parametrize("width,semantic", [(900, False), (900, True), (2048, True)])
def test_preprocess_equals_reference_shaders(width, semantic):
    p = O.default_params(**sized(width))
    sc, _ = scans(width, n=2, semantic=semantic)
    for t, (pts, lab, prob) in zip((3, 10), sc):   # t < 10: movable classes removed (Preprocessing.cpp:176)
        _frames_equal(O.preprocess(p, pts, lab, prob, timestamp=t), R.preprocess(p, pts, lab, prob, timestamp=t),
                      "preprocess w=%d t=%d" % (width, t))


def test_preprocess_equals_reference_shaders_on_random_clouds():
    rng = np.random.default_rng(5)
    p = O.default_params(**sized(360, 32))
    for quirk in (1, 0):
        p.label_offset_quirk = quirk
        for n in (0, 1, 7, 40000):
            pts, lab, prob = _random_cloud(rng, max(n, 1), p)
            pts, lab, prob = pts[:n], lab[:n], prob[:n]
            for t in (0, 50):
                _frames_equal(O.preprocess(p, pts, lab, prob, timestamp=t), R.preprocess(p, pts, lab, prob, timestamp=t),
                              "random cloud n=%d quirk=%d t=%d" % (n, quirk, t))


def test_preprocess_against_an_independent_gl():
    """precise built-ins: the vertex and semantic images (pure selection) stay identical, normals move by rounding only"""
    p = O.default_params(**sized(900))
    sc, _ = scans(900, n=1, semantic=True)
    a = O.preprocess(p, *sc[0], timestamp=20)
    with R.sampled(1):
        b = R.preprocess(p, *sc[0], timestamp=20, mode="precise")
    assert_bits_equal(a[0], b[0], "vertex map")
    assert_bits_equal(a[2], b[2], "semantic map")
    assert_bits_equal(a[1][..., 3], b[1][..., 3], "normal validity")
    idx, normals = R.sample(b[1])   # a fixed, seeded sample of the pixels
    assert np.nanmax(np.abs(a[1].reshape(-1, 4)[idx] - normals)) < 5e-5


# ------------------------------------------------------------------------------------------------- K5
def _icp_inputs(width=900, semantic=True):
    p = O.default_params(**sized(width))
    sc, _ = scans(width, n=3, semantic=semantic)
    sl = O.Slam(p)
    for s in sc:
        sl.process_scan(*s)
    T = np.eye(4)
    T[:3, 3] = (0.05, -0.02, 0.01)
    return p, sl.frame(0), sl.frame(1), T


def _lower(o48):
    """what Eigen::LDLT reads of JtJ (lower triangle, col-major) + Jtf + the counters"""
    m = np.asarray(o48[:36]).reshape(6, 6)  # m[c][r]
    return np.concatenate([np.array([m[c][r] for c in range(6) for r in range(c, 6)]), o48[36:47]])


@pytest.mark.parametrize("weighting,bilinear,iteration", [(0, 1, 0), (1, 1, 1), (2, 1, 1), (2, 0, 2), (0, 0, 0)])
def test_jacobian_sums_equal_reference_shader(weighting, bilinear, iteration):
    """Frame2Model_jacobians.geom + additive blending, against the oracle's GL-order fp32 accumulation (bit-exact) and
    against its exact fixed-point sums (what the CUDA path computes; within 1e-5 of the matrix scale)"""
    p, data, model, T = _icp_inputs()
    p.weighting, p.bilinear_sampling, p.factor = weighting, bilinear, 0.5
    gl = O.icp_jacobian_fp32gl(p, data, model, T, iteration=iteration)
    rf = R.icp_jacobian(p, data, model, T, iteration=iteration)
    assert_bits_equal(_lower(gl).astype(np.float32), _lower(rf).astype(np.float32), "48 blended sums (lower triangle)")
    # the upper triangle of the shader's JtJ is (w*J_c)*J_r with the roles swapped: equal up to rounding, unused by LDLT
    m = rf[:36].reshape(6, 6).astype(np.float64)
    scale = np.sqrt(np.outer(np.diag(m), np.diag(m)))
    assert np.max(np.abs(m - m.T) / scale) < 1e-5
    exact, raw = O.icp_jacobian(p, data, model, T, iteration=iteration)
    assert (rf[42], rf[44], rf[46]) == (exact[42], exact[44], exact[46])       # valid, outlier, invalid counters
    em = exact[:36].reshape(6, 6)
    assert np.max(np.abs(m - em) / scale) < 1e-5                                 # north_star: 1e-5 relative
    assert np.max(np.abs(rf[36:42] - exact[36:42])) / np.sqrt(np.max(np.diag(em)) * exact[43]) < 1e-5
    assert abs(rf[43] - exact[43]) / exact[43] < 1e-5 and abs(rf[45] - exact[45]) / exact[45] < 1e-5


def test_jacobian_entries_per_kernel_and_independent_gl():
    p, data, model, T = _icp_inputs()
    exact, _ = O.icp_jacobian(p, data, model, T)
    scale = np.sqrt(np.outer(np.diag(exact[:36].reshape(6, 6)), np.diag(exact[:36].reshape(6, 6))))
    for epk, mode in ((1, "pinned"), (16, "pinned"), (64, "precise")):
        rf = R.icp_jacobian(p, data, model, T, entries_per_kernel=epk, mode=mode)
        # entries_per_kernel = 1 makes the ROP add 57 600 fp32 terms one by one: the reference's own rounding error grows
        tol = {1: 1e-4, 16: 1e-5, 64: 2e-3}[epk]
        assert np.max(np.abs(rf[:36].reshape(6, 6) - exact[:36].reshape(6, 6)) / scale) < tol
        if mode == "pinned":
            assert (rf[42], rf[44], rf[46]) == (exact[42], exact[44], exact[46])
        else:  # a pixel within rounding of a threshold may change class under another GL
            assert abs(rf[42] - exact[42]) <= 1e-3 * exact[42] and abs(rf[44] - exact[44]) <= 5e-3 * exact[42]


# ------------------------------------------------------------------------------------------------- K4 / K6
def _maps(p, mode="pinned"):
    return O.Map(p), R.Map(p, mode)


def _check_update(om, rm, what):
    io, ro, go, nuo, nno = om.update_debug()
    ir, rr, gr, nur, nnr = rm.update_debug()
    assert_bits_equal(io, ir, what + ": index map")
    assert_bits_equal(ro, rr, what + ": radius map")
    assert_bits_equal(go, gr, what + ": integrated flags")
    assert (nuo, nno) == (nur, nnr), what + ": transform feedback counts"
    surfel_fields_equal(om.download(), rm.download(), what + ": surfels")


@pytest.mark.parametrize("semantic", [False, True])
def test_map_sequence_equals_reference_shaders(semantic):
    """5 scans through render (old / new / composed / composed output frame) and update (index map, radius map,
    integrated flags, updated + new + copied surfels in transform-feedback order)"""
    p = O.default_params(**sized(900))
    sc, poses = scans(900, n=5, semantic=semantic)
    om, rm = _maps(p)
    for t in range(5):
        pose = poses[t].astype(np.float32)
        data = O.preprocess(p, *sc[t], timestamp=t)
        ct = 0.1 * t
        _frames_equal(om.render(poses[max(t - 1, 0)], pose, ct), rm.render(poses[max(t - 1, 0)], pose, ct), "render t=%d" % t)
        for w, nm in enumerate(("old", "new", "composed")):
            _frames_equal(om.frame(w), rm.frame(w), "%s frame t=%d" % (nm, t))
        om.update(pose, data)
        rm.update(pose, data)
        _check_update(om, rm, "update t=%d" % t)
    assert om.size() > 50000


def _random_surfels(rng, n, t_now):
    s = np.zeros(n, O.SURFEL_DTYPE)
    d = rng.uniform(1.0, 80.0, n)
    yaw = rng.uniform(-np.pi, np.pi, n)
    pitch = np.deg2rad(rng.uniform(-30.0, 6.0, n))
    s["x"], s["y"], s["z"] = d * np.cos(pitch) * np.cos(yaw), d * np.cos(pitch) * np.sin(yaw), d * np.sin(pitch)
    nrm = rng.normal(size=(n, 3))
    nrm /= np.linalg.norm(nrm, axis=1, keepdims=True)
    facing = -(nrm[:, 0] * s["x"] + nrm[:, 1] * s["y"] + nrm[:, 2] * s["z"]) > 0
    nrm[~facing & (rng.uniform(size=n) < 0.8)] *= -1              # most face the sensor, some do not
    s["nx"], s["ny"], s["nz"] = nrm[:, 0], nrm[:, 1], nrm[:, 2]
    s["radius"] = rng.uniform(0.01, 1.2, n) * (d / 20.0 + 0.2)
    s["confidence"] = rng.uniform(-1.0, 3.0, n)
    creation = rng.integers(0, t_now + 1, n)
    s["count"] = creation
    s["timestamp"] = np.minimum(creation + rng.integers(0, 40, n), t_now)
    s["weight"] = rng.uniform(0.5, 19.5, n)
    lab = rng.choice(np.array((0, 10, 18, 30, 40, 48, 50, 70), np.float32), n) / np.float32(255.0)
    s["r"] = s["g"] = s["b"] = lab
    s["w"] = rng.uniform(0, 1, n)
    return s


@pytest.mark.parametrize("t_now,compose", [(150, 1), (40, 1), (150, 0)])
def test_random_surfel_clouds_equal_reference_shaders(t_now, compose):
    """adversarial per-element inputs: random surfels (any orientation, huge and tiny discs across the azimuth seam,
    negative confidences, old and new creation times, movable labels) against a real data frame"""
    rng = np.random.default_rng(t_now + compose)
    p = O.default_params(**sized(360, 32), compose_rendering=compose)
    pts, lab, prob = _random_cloud(rng, 30000, p)
    lab[:] = rng.choice(np.array((0, 10, 30, 40, 50), np.float32), lab.shape[0])
    om, rm = _maps(p)
    S = _random_surfels(rng, 20000, t_now)
    pose = np.eye(4)
    pose[:3, 3] = (0.3, -0.2, 0.1)
    a = np.deg2rad(3.0)
    pose[:2, :2] = [[np.cos(a), -np.sin(a)], [np.sin(a), np.cos(a)]]
    for m in (om, rm):
        m.upload(S, t_now)
        for t in range(0, t_now + 1, 7):
            T = np.eye(4); T[:3, 3] = (0.01 * t, 0.002 * t, 0.0)
            m.set_pose(t, T)
    data = O.preprocess(p, pts, lab, prob, timestamp=t_now)
    _frames_equal(om.render(np.eye(4), pose, 0.5), rm.render(np.eye(4), pose, 0.5), "render")
    for w, nm in enumerate(("old", "new", "composed")):
        _frames_equal(om.frame(w), rm.frame(w), nm)
    for call in ("render_active", "render_inactive"):
        getattr(om, call)(pose, 0.2); getattr(rm, call)(pose, 0.2)
    om.render_composed(np.eye(4), pose, 0.2); rm.render_composed(np.eye(4), pose, 0.2)
    for w, nm in enumerate(("inactive", "active", "composed(LEQUAL)")):
        fo, fr = om.frame(w), rm.frame(w)
        assert_bits_equal(fo[0], fr[0], nm + ".vertex"); assert_bits_equal(fo[1], fr[1], nm + ".normal")
    om.update(pose, data); rm.update(pose, data)
    _check_update(om, rm, "update")
    assert 0 < om.size()


def test_map_against_an_independent_gl():
    """precise built-ins: surfel counts stay within 0.1 %, records agree to rounding"""
    p = O.default_params(**sized(900))
    sc, poses = scans(900, n=3, semantic=True)
    om, rm = _maps(p, "precise")
    for t in range(3):
        data = O.preprocess(p, *sc[t], timestamp=t)
        fo = om.render(poses[t], poses[t], 0.0)
        with R.sampled(0):
            fr = rm.render(poses[t], poses[t], 0.0)
        idx, vertices = R.sample(fr[0])   # a fixed, seeded sample of the pixels
        same = np.all(np.abs(fo[0].reshape(-1, 4)[idx] - vertices) < 1e-3, axis=1)
        if t:
            assert same.mean() > 0.97           # the winner of a pixel changes only at depth ties / disc borders
        om.update(poses[t], data); rm.update(poses[t], data)
        assert abs(om.size() - rm.size()) <= 1e-3 * om.size()

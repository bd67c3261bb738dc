"""CPU tests against oracle/_ref/libsuma_ref_full.so: THE REFERENCE ITSELF, run here. Its core classes --
core/Preprocessing.cpp, Frame2Model.cpp, LieGaussNewton.cpp, lie_algebra.cpp, SurfelMap.cpp, SurfelMapping.cpp -- are
compiled where they lie under /root/reference and drive the reference's own GLSL shaders (transpiled) through a stand-in
`glow` on a generic software OpenGL (oracle/ref_harness/full/: programs, vertex arrays, samplers, framebuffers, transform
feedback and blending are resolved from what the reference's C++ sets up, nothing is special-cased per pass).

Only what OpenGL / Eigen / libm leave to the implementation is pinned to the rules of DESIGN.md section 2 (rasterisation and
depth rules, GLSL built-ins, the operation order of Eigen's LDLT and pose inverse, libm's sin/cos in SE3::exp), and the
oracle is switched to add up the 48 ICP values the way the GL path does (fp32 partial sums in the geometry shader, fp32
blending in primitive order -- O.gl_sums) instead of exactly. Then reference and oracle must agree BIT FOR BIT: images,
fp64 poses, Gauss-Newton iteration counts and histories, every surfel record and the surfel order, through the
track-loss fallback, submap paging and loop-closure detection. (Exact sums vs GL sums is the one documented numerical
difference between the CUDA path and the reference: within 1e-5 of the matrix scale, tests/test_ref_shaders.py.)

What the reference returned is replayed from tests/golden/reference_calls/ (tests/reference_replay.py), so these
comparisons need neither the reference nor oracle/_ref."""
import numpy as np
import pytest

from oracle import oracle as O
from semantic_suma_b200 import synth
from helpers import assert_bits_equal, scans, sized, surfel_fields_equal
from reference_replay import R


@pytest.fixture(autouse=True)
def _gl_sums():
    old = O.gl_sums(1)
    yield
    O.gl_sums(old)


def _both(p, **extra):
    return R.Full(p, **extra), O.Slam(p)


def _step_equal(f, osl, scan, what):
    pts, lab, prb = scan
    f.process_scan(pts, lab, prb)
    osl.process_scan(pts, lab, prb)
    with R.digests():
        assert_bits_equal(f.pose(), osl.pose(), what + " pose")
    assert f.map_size() == osl.map.size(), what + " surfel count %d vs %d" % (f.map_size(), osl.map.size())
    surfel_fields_equal(f.map_download(), osl.map.download(), what + " surfels")


@pytest.mark.parametrize("semantic,timestamp", [(False, 100), (True, 3), (True, 30)])
def test_preprocessing_class_equals_oracle_and_pinned_harness(semantic, timestamp):
    """Preprocessing::process (vertex attributes incl. the label/probability offset quirk Q1, the three passes, the
    full-screen quad of empty.vert + quad.geom, sampler state) against oracle/ and against ref_pipeline.cpp"""
    p = O.default_params(**sized(900))
    f = R.Full(p)
    sc, _ = scans(900, n=1, semantic=semantic)
    got = f.preprocess(*sc[0], timestamp=timestamp)
    for g, o, r, name in zip(got, O.preprocess(p, *sc[0], timestamp=timestamp), R.preprocess(p, *sc[0], timestamp=timestamp),
                             ("vertex", "normal", "semantic")):
        assert_bits_equal(g, o, name + " map vs oracle")
        assert_bits_equal(g, r, name + " map vs pinned harness")


@pytest.mark.parametrize("weighting,bilinear,iteration", [(0, 1, 0), (1, 1, 1), (2, 0, 2)])
def test_frame2model_class_equals_pinned_harness(weighting, bilinear, iteration):
    """Frame2Model::jacobianProducts (weighting by NAME, thresholds, ONE sampler object for six units, additive blending
    into the 2x8 RGB32F texture, the float -> uint32 conversions of the counters)"""
    p = O.default_params(**sized(900), weighting=weighting, bilinear_sampling=bilinear, factor=0.5)
    sc, _ = scans(900, n=2, semantic=True)
    fr = [O.preprocess(p, *s) for s in sc]
    T = O.se3_exp(np.array([0.9, 0.02, 0.01, 0.001, -0.002, 0.008]))
    got = R.Full(p).icp_jacobian(fr[1], fr[0], T, iteration=iteration)
    want = R.icp_jacobian(p, fr[1], fr[0], T, iteration=iteration)
    assert_bits_equal(got[:42].astype(np.float32), want[:42], "48 blended values")
    o48 = O.icp_jacobian(p, fr[1], fr[0], T, iteration=iteration)[0]   # GL-sum mode
    low = [c * 6 + r for c in range(6) for r in range(c, 6)]
    assert_bits_equal(got[low], o48[low], "JtJ lower triangle vs oracle (GL sums)")
    assert_bits_equal(got[36:42], o48[36:42], "Jtf")
    assert (got[42], got[44], got[46]) == (o48[42], o48[44], o48[46]) and got[43] == o48[43]


def test_gauss_newton_on_the_reference_classes_equals_oracle():
    """LieGaussNewton::minimize over Frame2Model: every pose of the history (fp64) equal -- LDLT, SE3::exp, the stop tests"""
    p = O.default_params(**sized(900))
    sc, _ = scans(900, n=2)
    fr = [O.preprocess(p, *s) for s in sc]
    pose, k, hist = R.Full(p).icp_minimize(fr[1], fr[0], np.eye(4))
    opose, _, ok, ohist = O.icp_minimize(p, fr[1], fr[0], np.eye(4))
    assert k == ok and len(hist) == len(ohist)
    for i, (a, b) in enumerate(zip(hist, ohist)):
        assert_bits_equal(a, b, "history[%d]" % i)
    assert_bits_equal(pose, opose, "final pose")


@pytest.mark.parametrize("width,semantic,frames", [(900, False, 6), (900, True, 5), (2048, False, 3), (2048, True, 3)])
def test_process_scan_of_the_reference_equals_oracle(width, semantic, frames):
    """SurfelMapping::processScan with config/default.xml: initialize, preprocess, render (old / new / composed + compose
    pass), updatePose (Gauss-Newton, render_active, statistics pass), updateMap (index map, radius, update, generate, copy
    with transform feedback), the confidence-threshold ramp of the first scans"""
    p = O.default_params(**sized(width))
    f, osl = _both(p)
    sc, _ = scans(width, n=frames, semantic=semantic)
    for t in range(frames):
        _step_equal(f, osl, sc[t], "t=%d" % t)
        if t > 0:
            assert f.statistic("num_iterations") == osl.stats()["iterations"]
    for a, b, name in zip(f.slam_frame(0), osl.frame(0), ("vertex", "normal", "semantic")):
        assert_bits_equal(a, b, "current frame " + name)
    # lastModelFrame_: the composed rendering of preprocess(), then overwritten by the copy of the post-ICP render_active
    for a, b, name in zip(f.slam_frame(3)[:2], osl.frame(1)[:2], ("vertex", "normal")):
        assert_bits_equal(a, b, "last model frame " + name)
    for w in range(3):  # SurfelMap's own old / new / composed frames after the final render of updateMap()
        for a, b, name in zip(f.map_frame(w), osl.map.frame(w), "vns"):
            assert_bits_equal(a, b, "map frame %d %s" % (w, name))


VARIANTS = [dict(weighting=1), dict(weighting=2), dict(weighting=0), dict(bilinear_sampling=0), dict(compose_rendering=0),
            dict(initialize_identity=1), dict(initialize_identity=0), dict(update_always=1), dict(weighting_scheme=1),
            dict(weighting_scheme=2), dict(averaging_scheme=1), dict(confidence_mode=0), dict(confidence_mode=1),
            dict(confidence_mode=2), dict(use_stability=0), dict(unstable_age=1, confidence_threshold=5.0),
            dict(max_iterations=3), dict(fallback_mode=0), dict(active_timestamps=1), dict(min_radius=0.05, max_radius=0.2),
            dict(max_angle=60.0), dict(map_max_distance=0.05, map_max_angle=5.0), dict(partial_extraction=0),
            dict(submap_extent=3.0, submap_dimension=1)]


def test_parameter_branches_of_the_reference_equal_oracle():
    """every parameter the classes read (robust weighting by name, sampling, compose rendering on/off, initial guess,
    surfel weighting / averaging schemes, confidence modes, stability, thresholds, submap layout): four semantic scans at
    64x450 per variant, poses and surfel records bit-identical"""
    sc, _ = scans(450, n=4, semantic=True)
    for kw in VARIANTS:
        p = O.default_params(**sized(450), **kw)
        f, osl = _both(p)
        for t in range(4):
            _step_equal(f, osl, sc[t], "%r t=%d" % (kw, t))


GEOMETRIES = [dict(data_width=450, data_height=64, model_width=512, model_height=64),      # model image != data image
              dict(data_width=450, data_height=64, model_width=450, model_height=96),
              dict(data_width=600, data_height=32, model_width=300, model_height=32),
              dict(data_width=450, data_height=64, model_width=450, model_height=64, data_fov_up=10.0, data_fov_down=-30.0,
                   model_fov_up=10.0, model_fov_down=-30.0),
              dict(data_width=450, data_height=64, model_width=450, model_height=64, min_depth=1.0, max_depth=40.0,
                   model_min_depth=1.0, model_max_depth=40.0),
              dict(data_width=450, data_height=64, model_width=450, model_height=64, model_fov_up=5.0, model_fov_down=-28.0)]


def test_image_geometries_of_the_reference_equal_oracle():
    """model image size / field of view / depth range different from the data image's (the classes take them from separate
    parameters): three semantic scans each"""
    for kw in GEOMETRIES:
        p = O.default_params(**kw)
        scene = synth.Scene(width=kw["data_width"], height=kw["data_height"], fov_up=kw.get("data_fov_up", 3.0),
                            fov_down=kw.get("data_fov_down", -25.0), semantic=True)
        poses = synth.trajectory(3)
        f, osl = _both(p)
        for t in range(3):
            _step_equal(f, osl, scene.scan(t, poses[t]), "%r t=%d" % (kw, t))


def test_ouster_size_of_the_reference_equals_oracle():
    """BASELINE.json configs[3]: 128x4096, +-22.5 degrees, 15 iterations -- two scans"""
    kw = dict(data_width=4096, model_width=4096, data_height=128, model_height=128, data_fov_up=22.5, data_fov_down=-22.5,
              model_fov_up=22.5, model_fov_down=-22.5, max_iterations=15, stopping_threshold=0.0, delta=0.0)
    p = O.default_params(**kw)
    sc = synth.Scene(width=4096, height=128, fov_up=22.5, fov_down=-22.5)
    poses = synth.trajectory(2)
    f, osl = _both(p)
    for t in range(2):
        _step_equal(f, osl, sc.scan(t, poses[t]), "t=%d" % t)
    assert f.statistic("num_iterations") == 15


def test_stale_attribute_tail_of_the_reference_is_the_one_known_deviation():
    """Q1 reads labels[i+4] / probs[i+5]: for the last 4 / 5 points of a scan that is past the data just uploaded. glow's
    GlBuffer::assign keeps the larger data store of an earlier upload, so the reference reads the PREVIOUS scan's values
    there (undefined memory after a re-allocation); oracle and CUDA path read 0. At most 5 points per scan can differ --
    shown here, and switched off (zero_stale_tail) everywhere else."""
    p = O.default_params(**sized(900))
    sc, _ = scans(900, n=2, semantic=True)
    big, small = (sc[0], sc[1]) if sc[0][0].shape[0] >= sc[1][0].shape[0] else (sc[1], sc[0])
    if big[0].shape[0] == small[0].shape[0]:
        small = tuple(a[:-7] for a in small)
    faithful, zeroed = R.Full(p, zero_stale_tail=False), R.Full(p, zero_stale_tail=True)
    for f, zero in ((faithful, False), (zeroed, True)):
        f.zero_stale_tail(zero)
        f.process_scan(*big)
        f.zero_stale_tail(zero)
        f.process_scan(*small)
    diff = R.computed(lambda: np.argwhere((faithful.slam_frame(0)[2] != zeroed.slam_frame(0)[2]).any(axis=2)))
    assert 1 <= len(diff) <= 5 * 3          # the tail points and what floodfill spreads from them
    assert_bits_equal(zeroed.slam_frame(0)[2], O.preprocess(p, *small, timestamp=1)[2], "zeroed tail = oracle")


def test_track_loss_fallback_of_the_reference_equals_oracle():
    """SurfelMapping.cpp:430-449: the same jump sequence as the GPU test; the reference prints "Lost track" and runs the
    frame-to-frame recovery_ objective -- same decisions, same poses"""
    p = O.default_params(**sized(900))
    scene = synth.Scene(width=900, height=64)
    poses = synth.trajectory(8)
    J = synth.translate(0.8, 0.3, 0) @ synth.rot_z(np.deg2rad(8.0))
    f, osl = _both(p)
    for t in range(7):
        _step_equal(f, osl, scene.scan(t, poses[t] if t < 4 else poses[t] @ J), "t=%d" % t)
    assert osl.stats()["track_loss"] >= 1


def test_submap_paging_of_the_reference_equals_oracle():
    """SurfelMap::update incl. updateActiveSubmaps / extractSurfels (extract_surfels.vert + transform feedback into the
    extract buffer, partial extraction queue, re-insertion of cached tiles): the same tour as the GPU paging test"""
    p = O.default_params(**sized(900))
    sc, _ = scans(900, n=3)
    frames = [O.preprocess(p, *s, timestamp=100) for s in sc]
    f, omap = R.Full(p), O.Map(p)

    def pose_at(x, y):
        T = np.eye(4, dtype=np.float32)
        T[0, 3], T[1, 3] = x, y
        return T
    xs = [0, 12, 36, 60, 84, 108, 120, 120, 108, 60, 12, -12]
    ys = [0, 0, 0, 0, 0, 0, 0, 24, 24, 24, 0, 0]
    shifted = 0
    for t, (x, y) in enumerate(zip(xs, ys)):
        f.map_update(pose_at(x, y), frames[t % 3])
        omap.update(pose_at(x, y), frames[t % 3])
        assert f.map_size() == omap.size(), "t=%d size" % t
        shifted += omap.submap_origin()[:2] != (0, 0)
    assert shifted > 5
    surfel_fields_equal(f.map_download(), omap.download(), "surfels after paging")
    T = pose_at(-12, 0)
    for a, b, name in zip(f.map_render(T, T, -5.0), omap.render(T, T, -5.0), "vns"):
        assert_bits_equal(a, b, "render after paging " + name)
    for w in range(3):
        for a, b, name in zip(f.map_frame(w), omap.frame(w), "vns"):
            assert_bits_equal(a, b, "map frame %d %s" % (w, name))


@pytest.mark.parametrize("t_now,compose", [(150, 1), (40, 1), (150, 0)])
def test_random_surfel_clouds_through_the_reference_classes(t_now, compose):
    """the adversarial map inputs of tests/test_ref_shaders.py (random surfels of any orientation, huge and tiny discs across
    the azimuth seam, negative confidences, old and new creation times, movable labels; points outside the field of view)
    through SurfelMap::render / render_active / render_inactive / render_composed / update of the reference itself"""
    from test_ref_shaders import _random_cloud, _random_surfels
    rng = np.random.default_rng(t_now + compose)
    p = O.default_params(**sized(360, 32), compose_rendering=compose)
    pts, lab, prob = _random_cloud(rng, 30000, p)
    lab[:] = rng.choice(np.array((0, 10, 30, 40, 50), np.float32), lab.shape[0])
    om, f = O.Map(p), R.Full(p)
    S = _random_surfels(rng, 20000, t_now)
    pose = np.eye(4)
    pose[:3, 3] = (0.3, -0.2, 0.1)
    a = np.deg2rad(3.0)
    pose[:2, :2] = [[np.cos(a), -np.sin(a)], [np.sin(a), np.cos(a)]]
    om.upload(S, t_now)
    f.map_upload(S, t_now)
    for t in range(0, t_now + 1, 7):
        T = np.eye(4); T[:3, 3] = (0.01 * t, 0.002 * t, 0.0)
        om.set_pose(t, T)
        f.map_set_pose(t, T)
    data = O.preprocess(p, pts, lab, prob, timestamp=t_now)
    for g, o, name in zip(f.preprocess(pts, lab, prob, timestamp=t_now), data, "vns"):
        assert_bits_equal(g, o, "preprocess " + name)
    for g, o, name in zip(f.map_render(np.eye(4), pose, 0.5), om.render(np.eye(4), pose, 0.5), "vns"):
        assert_bits_equal(g, o, "render " + name)
    for w in range(3):
        for g, o, name in zip(f.map_frame(w), om.frame(w), "vns"):
            assert_bits_equal(g, o, "frame %d %s" % (w, name))
    om.render_active(pose, 0.2); f.map_render_active(pose, 0.2)
    om.render_inactive(pose, 0.2); f.map_render_inactive(pose, 0.2)
    om.render_composed(np.eye(4), pose, 0.2); f.map_render_composed(np.eye(4), pose, 0.2)
    for w in range(3):
        for g, o, name in zip(f.map_frame(w)[:2], om.frame(w)[:2], "vn"):
            assert_bits_equal(g, o, "single-view frame %d %s" % (w, name))
    om.update(pose, data)
    f.map_update(pose, data)
    assert f.map_size() == om.size() > 0
    surfel_fields_equal(f.map_download(), om.download(), "surfels after the update")


def test_unpinned_reference_agrees_with_the_cuda_contract_within_tolerances():
    """libsuma_ref_full_precise.so: the same classes and shaders with NOTHING pinned to the oracle's rules (GLSL built-ins in
    fp64 / libm, the stand-in Eigen's general inverse and left-looking LDLT, libm's sin / cos, fp32 blending of the 48 values)
    against the oracle in its default mode -- exact sums, the contract of the CUDA path. An independent legal implementation
    of everything OpenGL / Eigen / libm leave open: decisions flip only within rounding of a threshold, so poses stay within
    2e-3 m (the Gauss-Newton stop tests are 1e-4) and surfel counts within 0.2 % over eight scans, without drift."""
    old = O.gl_sums(0)
    try:
        for width, semantic, frames, kw in ((900, True, 8, {}), (900, False, 6, dict(max_iterations=10, stopping_threshold=0.0, delta=0.0))):
            p = O.default_params(**sized(width), **kw)
            sc, _ = scans(width, n=frames, semantic=semantic)
            f, osl = R.Full(p, mode="precise"), O.Slam(p)
            for t in range(frames):
                f.process_scan(*sc[t])
                osl.process_scan(*sc[t])
                assert np.abs(f.pose() - osl.pose()).max() < 2e-3, "t=%d pose" % t
                assert abs(f.map_size() - osl.map.size()) <= 2e-3 * osl.map.size(), "t=%d surfel count" % t
            assert_bits_equal(R.Full(p, mode="precise").preprocess(*sc[0])[0], O.preprocess(p, *sc[0])[0], "vertex map")
    finally:
        O.gl_sums(old)


def test_loop_closure_of_the_reference_equals_oracle_twin():
    """SurfelMapping::checkLoopClosure (:527-795) and integrateLoopClosures (:212-258) on the synthetic loop of the GPU
    test (64x300 here): the candidate is found at the same scan, verified, the same loop edges enter the pose graph, the
    optimisation is requested at the same scan, and after handing the graph to the optimiser (here: the identity, on both
    sides -- gtsam stays with the host application) the corrected poses are integrated the same way: poses, flags, edges
    and every surfel stay bit-identical through two request / integrate cycles."""
    W = 300
    p = O.default_params(**sized(W))
    lp = dict(search_distance=3.0, min_trajectory_distance=15.0, min_verifications=2)
    f = R.Full(p, **{"close-loops": True, "loop-search-distance": 3.0, "loop-min-trajectory-distance": 15.0,
                     "loop-min-verifications": 2})
    osl = O.Slam(p)
    osl.enable_loop_closure(**lp)
    scene = synth.Scene(width=W, height=64)
    N = 126
    poses = synth.trajectory(N, step=0.2618, yaw_deg=3.0)
    found_at, integrations = None, []
    for t in range(N):
        pts = scene.scan(t, poses[t])[0]
        if osl.loop_info()["optimisation_requested"]:   # the reference does this at the top of processScan (:179)
            assert osl.integrate_loop_closures() == t
            integrations.append(t)
        f.process_scan(pts)
        osl.process_scan(pts)
        info = osl.loop_info()
        with R.digests():
            assert_bits_equal(f.pose(), osl.pose(), "t=%d pose" % t)
        assert f.loop_flags() == (bool(info["found_candidate"]), bool(info["use_candidate"])), "t=%d candidate flags" % t
        assert R.computed(lambda: len(f.edges())) == info["n_edges"], "t=%d pose-graph edges" % t
        assert f.map_size() == osl.map.size()
        if info["found_candidate"] and found_at is None:
            found_at = t
            assert f.statistic("residual_old") == pytest.approx(info["residual_old"], rel=1e-6)
    assert found_at is not None and info["loop_edges_added"] >= 3 and len(integrations) == 2, (info, integrations)
    assert f.edges() == [(a, b) for a, b, _ in osl.loop_edges()]
    surfel_fields_equal(f.map_download(), osl.map.download(), "surfels after the loop")

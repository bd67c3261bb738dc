"""GPU parity tests: the CUDA path (through the C ABI) against the CPU oracle on identical seeded inputs.
Bar: bit-exact for images, surfels, fixed-point sums, poses (everything is a chain of correctly rounded IEEE ops)."""
import numpy as np
import pytest

from oracle import oracle as O
from semantic_suma_b200 import api
from helpers import assert_bits_equal, both_params, scans, sized, surfel_fields_equal

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx900():
    po, pp = both_params(**sized(900))
    c = api.Context(pp)
    yield po, pp, c
    c.close()


def _prep_both(po, ctx, scan, timestamp):
    pts, lab, prb = scan
    ov = O.preprocess(po, pts, lab, prb, timestamp)
    f = api.Frame(ctx, po.data_width, po.data_height)
    api.Preprocessing(ctx).process(pts, f, lab, prb, timestamp)
    return ov, f


@pytest.mark.parametrize("width,semantic,timestamp", [(900, False, 100), (900, True, 100), (900, True, 3),
                                                      (2048, False, 100), (2048, True, 0)])
def test_preprocess_bit_exact(width, semantic, timestamp):
    po, pp = both_params(**sized(width))
    ctx = api.Context(pp)
    sc, _ = scans(width, n=2, semantic=semantic)
    for s in sc:
        ov, f = _prep_both(po, ctx, s, timestamp)
        gv, gn, gs = f.maps()
        assert_bits_equal(gv, ov[0], "vertex_map")
        assert_bits_equal(gn, ov[1], "normal_map")
        assert_bits_equal(gs, ov[2], "semantic_map")
    ctx.close()


def test_preprocess_edge_cases(ctx900):
    po, pp, ctx = ctx900
    pre = api.Preprocessing(ctx)
    f = api.Frame(ctx, 900, 64)
    # empty scan
    pre.process(np.zeros((0, 4), np.float32), f)
    ov = O.preprocess(po, np.zeros((0, 4), np.float32))
    for g, o in zip(f.maps(), ov):
        assert_bits_equal(g, o, "empty scan")
    # degenerate points: origin, out of range, behind, straight up/down, duplicates in one pixel
    pts = np.array([[0, 0, 0, 1], [1000, 0, 0, 1], [-5, 0, 0, 1], [0, 0, 10, 1], [0, 0, -10, 1], [5, 1, -0.5, 1],
                    [5, 1, -0.5, 1], [5.0001, 1, -0.5, 1], [1.0, 0, 0, 1], [-5, 1e-9, -0.3, 1], [-5, -1e-9, -0.3, 1]],
                   np.float32)
    pre.process(pts, f)
    ov = O.preprocess(po, pts)
    for g, o in zip(f.maps(), ov):
        assert_bits_equal(g, o, "degenerate points")


@pytest.mark.parametrize("bilinear,weighting,semantic", [(1, 1, False), (0, 1, False), (1, 2, True), (1, 0, True),
                                                         (0, 2, False)])
def test_icp_jacobian_exact(bilinear, weighting, semantic):
    kw = sized(900, bilinear_sampling=bilinear, weighting=weighting)
    po, pp = both_params(**kw)
    ctx = api.Context(pp)
    sc, poses = scans(900, n=2, semantic=semantic)
    o0, f0 = _prep_both(po, ctx, sc[0], 100)
    o1, f1 = _prep_both(po, ctx, sc[1], 100)
    obj = api.Frame2Model(ctx)
    obj.setData(f1, f0)
    T = np.linalg.inv(poses[0]) @ poses[1]
    T[0, 3] += 0.1
    for it, pose in enumerate([np.eye(4), T]):
        obj.initialize(pose)
        obj.iteration_ = it
        obj.jacobianProducts()
        o48, raw = O.icp_jacobian(po, o1, o0, pose, iteration=it)
        assert np.array_equal(obj.raw32, raw), "raw sums differ: %s vs %s" % (obj.raw32, raw)
        assert_bits_equal(obj.out48, o48, "out48")
        assert obj.valid() + obj.invalid() == 900 * 64
    # row stripes add up exactly (multi-GPU contract)
    obj.initialize(T)
    tot = np.zeros(32, np.int64)
    for r0, r1 in [(0, 16), (16, 17), (17, 64)]:
        obj.jacobianProducts(rows=(r0, r1))
        tot += obj.raw32
    obj.jacobianProducts()
    assert np.array_equal(tot, obj.raw32)
    ctx.close()


def test_icp_minimize_matches_oracle_and_host_loop():
    po, pp = both_params(**sized(900))
    ctx = api.Context(pp)
    sc, poses = scans(900, n=2)
    o0, f0 = _prep_both(po, ctx, sc[0], 100)
    o1, f1 = _prep_both(po, ctx, sc[1], 100)
    obj = api.Frame2Model(ctx)
    obj.setData(f1, f0)
    gn = api.LieGaussNewton(ctx)
    gn.minimize(obj, np.eye(4))
    pose_o, o48, k, hist = O.icp_minimize(po, o1, o0, np.eye(4))
    assert gn.iterationCount() == k
    assert_bits_equal(gn.pose(), pose_o, "pose")
    assert_bits_equal(gn.out48, o48, "out48")
    assert len(gn.history()) == len(hist)
    for a, b in zip(gn.history(), hist):
        assert_bits_equal(a, b, "history")
    # the reference's call pattern (one jacobianProducts per iteration, solve on the host) gives the same bits
    gn2 = api.LieGaussNewton(ctx)
    obj2 = api.Frame2Model(ctx)
    obj2.setData(f1, f0)
    gn2.minimize_host(obj2, np.eye(4))
    assert gn2.iterationCount() == k
    assert_bits_equal(gn2.pose(), pose_o, "host-loop pose")
    # converges to the simulated motion
    gt = np.linalg.inv(poses[0]) @ poses[1]
    assert np.linalg.norm(gn.pose()[:3, 3] - gt[:3, 3]) < 0.05
    ctx.close()


def _run_map_sequence(width, n_frames, semantic, **kw):
    po, pp = both_params(**sized(width, **kw))
    ctx = api.Context(pp)
    sc, poses = scans(width, n=n_frames, semantic=semantic)
    omap = O.Map(po)
    gmap = api.SurfelMap(ctx)
    out = api.Frame(ctx, width, 64)
    for t in range(n_frames):
        ov, f = _prep_both(po, ctx, sc[t], t)
        pose = (np.linalg.inv(poses[0]) @ poses[t]).astype(np.float32)
        ct = -2.0 + 0.2 * t
        # render before update (as preprocess() does)
        orr = omap.render(pose, pose, ct)
        gmap.render(pose, pose, out, ct)
        for g, o, name in zip(out.maps(), orr, ("vertex", "normal", "semantic")):
            assert_bits_equal(g, o, "t=%d render frame %s" % (t, name))
        for which, fr in ((0, gmap.oldMapFrame()), (1, gmap.newMapFrame()), (2, gmap.composedFrame())):
            for g, o, name in zip(fr.maps(), omap.frame(which), ("vertex", "normal", "semantic")):
                assert_bits_equal(g, o, "t=%d map frame %d %s" % (t, which, name))
        omap.update(pose, ov)
        gmap.update(pose, f)
        oi, orad, oint, onu, onn = omap.update_debug()
        gi, grad, gint, gnu, gnn = gmap.update_debug()
        assert_bits_equal(gi, oi, "t=%d index map" % t)
        assert_bits_equal(grad, orad, "t=%d radius map" % t)
        assert_bits_equal(gint, oint, "t=%d integrated flags" % t)
        assert (gnu, gnn) == (onu, onn), "t=%d counts %s vs %s" % (t, (gnu, gnn), (onu, onn))
        assert gmap.size() == omap.size()
        surfel_fields_equal(gmap.getAllSurfels(), omap.download(), "t=%d surfels" % t)
    # render_active / inactive / composed after the sequence
    pose = (np.linalg.inv(poses[0]) @ poses[n_frames - 1]).astype(np.float32)
    pose2 = pose.copy(); pose2[0, 3] += 0.3
    omap.render_active(pose2, 0.0); gmap.render_active(pose2, 0.0)
    omap.render_inactive(pose, 0.0); gmap.render_inactive(pose, 0.0)
    omap.render_composed(pose, pose2, 0.0); gmap.render_composed(pose, pose2, 0.0)
    for which, fr in ((0, gmap.oldMapFrame()), (1, gmap.newMapFrame()), (2, gmap.composedFrame())):
        for g, o, name in zip(fr.maps(), omap.frame(which), ("vertex", "normal", "semantic")):
            assert_bits_equal(g, o, "final map frame %d %s" % (which, name))
    # different old / new poses through the full render
    orr = omap.render(pose, pose2, 0.0)
    gmap.render(pose, pose2, out, 0.0)
    for g, o, name in zip(out.maps(), orr, ("vertex", "normal", "semantic")):
        assert_bits_equal(g, o, "two-pose render %s" % name)
    ctx.close()


def test_map_update_and_render_bit_exact_geometric():
    _run_map_sequence(900, 6, False)


def test_map_update_and_render_bit_exact_semantic():
    _run_map_sequence(900, 5, True)


def test_map_render_old_surfels():
    # surfels older than the compose age (100 scans) exercise the old / composed views
    po, pp = both_params(**sized(900))
    ctx = api.Context(pp)
    sc, poses = scans(900, n=2)
    omap = O.Map(po); gmap = api.SurfelMap(ctx)
    ov, f = _prep_both(po, ctx, sc[0], 100)
    omap.update(np.eye(4, dtype=np.float32), ov); gmap.update(np.eye(4, dtype=np.float32), f)
    s = omap.download()
    half = s.shape[0] // 2
    # pretend the map is 150 scans old, half of the surfels re-observed recently
    s["timestamp"][:half] = 140
    omap.upload(s, 150); gmap.upload(s, 150)
    pose = np.eye(4, dtype=np.float32); pose[0, 3] = 0.5
    out = api.Frame(ctx, 900, 64)
    orr = omap.render(pose, pose, -1.0)
    gmap.render(pose, pose, out, -1.0)
    for g, o in zip(out.maps(), orr):
        assert_bits_equal(g, o, "compose frame")
    for which, fr in ((0, gmap.oldMapFrame()), (1, gmap.newMapFrame()), (2, gmap.composedFrame())):
        v = fr.vertex_map
        assert (v[..., 3] > 0).sum() > 1000
        for g, o in zip(fr.maps(), omap.frame(which)):
            assert_bits_equal(g, o, "frame %d" % which)
    ctx.close()


@pytest.mark.parametrize("width,semantic,frames", [(900, False, 8), (900, True, 6), (2048, False, 4)])
def test_process_scan_pipeline_bit_exact(width, semantic, frames):
    po, pp = both_params(**sized(width))
    sc, poses = scans(width, n=frames, semantic=semantic)
    osl = O.Slam(po)
    gsl = api.SurfelMapping(pp)
    for t in range(frames):
        pts, lab, prb = sc[t]
        osl.process_scan(pts, lab, prb)
        gsl.processScan(pts, lab, prb)
        assert_bits_equal(gsl.getCurrentPose(), osl.pose(), "t=%d pose" % t)
        so, sg = osl.stats(), gsl.getStatistics()
        assert sg["num_iterations"] == so["iterations"], "t=%d iterations" % t
        assert sg["F"] == so["F"] and sg["inlier"] == so["inlier"] and sg["outlier"] == so["outlier"]
        assert gsl.getMap().size() == osl.map.size(), "t=%d surfel count" % t
    surfel_fields_equal(gsl.getMap().getAllSurfels(), osl.map.download())
    for g, o in zip(gsl.getCurrentFrame().maps(), osl.frame(0)):
        assert_bits_equal(g, o, "current frame")
    gt = np.linalg.inv(poses[0]) @ poses[frames - 1]
    assert np.linalg.norm(gsl.getCurrentPose()[:3, 3] - gt[:3, 3]) < 0.1
    gsl.ctx.close()


def test_submap_paging_shift_extract_and_reinsert():
    """SurfelMap::updateActiveSubmaps (SurfelMap.cpp:744-824): moving > 1.1 * extent shifts the active window, queues the
    leaving tiles for extraction (one per update with partial extraction) and re-inserts cached tiles when coming back."""
    po, pp = both_params(**sized(900))
    ctx = api.Context(pp)
    sc, poses = scans(900, n=3)
    omap = O.Map(po)
    gmap = api.SurfelMap(ctx)
    frames = [_prep_both(po, ctx, s, 100) for s in sc]

    def pose_at(x, y):
        T = np.eye(4, dtype=np.float32)
        T[0, 3], T[1, 3] = x, y
        return T

    # forward along +x far enough to drop tiles (window is 9x9 tiles of 20 m), sideways, then all the way back
    xs = [0, 6, 12, 24, 36, 48, 60, 72, 84, 96, 108, 120, 120, 120, 108, 84, 60, 36, 12, 0, -12]
    ys = [0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 12, 24, 24, 24, 24, 12, 0, 0, 0]
    shifts = 0
    for t, (x, y) in enumerate(zip(xs, ys)):
        ov, f = frames[t % 3]
        T = pose_at(x, y)
        omap.update(T, ov)
        gmap.update(T, f)
        assert gmap.submap_origin() == omap.submap_origin(), "t=%d submap origin / pending" % t
        assert gmap.size() == omap.size(), "t=%d size %d vs %d" % (t, gmap.size(), omap.size())
        if omap.submap_origin()[:2] != (0, 0):
            shifts += 1
    assert shifts > 5
    surfel_fields_equal(gmap.getAllSurfels(), omap.download(), "surfels after paging")
    out = api.Frame(ctx, 900, 64)
    orr = omap.render(pose_at(-12, 0), pose_at(-12, 0), -5.0)
    gmap.render(pose_at(-12, 0), pose_at(-12, 0), out, -5.0)
    for g, o in zip(out.maps(), orr):
        assert_bits_equal(g, o, "render after paging")
    ctx.close()


# ---------------------------------------------------------------------------------------------------------------
# round 2: the configurations BASELINE.json names beyond configs[0..1], the track-loss fallback, API edge cases
# ---------------------------------------------------------------------------------------------------------------
def _pipeline_equal(po, pp, sc, what, check_frames=True):
    osl = O.Slam(po)
    gsl = api.SurfelMapping(pp)
    losses = 0
    for t, (pts, lab, prb) in enumerate(sc):
        osl.process_scan(pts, lab, prb)
        gsl.processScan(pts, lab, prb)
        assert_bits_equal(gsl.getCurrentPose(), osl.pose(), "%s t=%d pose" % (what, t))
        so, sg = osl.stats(), gsl.getStatistics()
        assert sg["num_iterations"] == so["iterations"], "%s t=%d iterations" % (what, t)
        assert (sg["F"], sg["inlier"], sg["outlier"], sg["invalid"]) == (so["F"], so["inlier"], so["outlier"], so["invalid"])
        assert sg["track_loss"] == so["track_loss"], "%s t=%d track loss counter" % (what, t)
        assert gsl.getMap().size() == osl.map.size(), "%s t=%d surfel count" % (what, t)
        losses = so["track_loss"]
    surfel_fields_equal(gsl.getMap().getAllSurfels(), osl.map.download(), what + " surfels")
    if check_frames:
        for g, o in zip(gsl.getCurrentFrame().maps(), osl.frame(0)):
            assert_bits_equal(g, o, what + " current frame")
        for g, o in zip(gsl.getLastModelFrame().maps(), osl.frame(1)):
            assert_bits_equal(g, o, what + " model frame")
    gsl.ctx.close()
    return losses


def test_process_scan_pipeline_semantic_2048():
    """BASELINE.json configs[2]: 64x2048, semantic-weighted ICP + label-consistent fusion, whole pipeline"""
    po, pp = both_params(**sized(2048))
    sc, _ = scans(2048, n=4, semantic=True)
    _pipeline_equal(po, pp, sc, "64x2048 semantic")


def test_process_scan_pipeline_ouster_128x4096():
    """BASELINE.json configs[3]: 128x4096 Ouster-style scans, 15 ICP iterations (stop tests off, as in the bench)"""
    kw = dict(sized(4096, 128), data_fov_up=22.5, data_fov_down=-22.5, model_fov_up=22.5, model_fov_down=-22.5,
              max_iterations=15, stopping_threshold=0.0, delta=0.0)
    po, pp = both_params(**kw)
    sc, _ = scans(4096, 128, n=3, fov_up=22.5, fov_down=-22.5)
    _pipeline_equal(po, pp, sc, "128x4096")


def test_track_loss_fallback_bit_exact():
    """SurfelMapping.cpp:89-96, 430-449: a pose jump makes the increment differ from the last one by more than 0.4 m /
    0.1 rad -> the frame-to-frame recovery minimisation against lastFrame_ runs and replaces the increment"""
    from semantic_suma_b200 import synth
    po, pp = both_params(**sized(900))
    scene = synth.Scene(width=900, height=64)
    poses = synth.trajectory(8)
    J = synth.translate(0.8, 0.3, 0) @ synth.rot_z(np.deg2rad(8.0))
    sc = [scene.scan(f, poses[f] if f < 4 else poses[f] @ J) for f in range(7)]
    losses = _pipeline_equal(po, pp, sc, "fallback")
    assert losses >= 1, "the sequence must trigger the fallback"


def test_scan_larger_than_two_images_of_points():
    """ADVICE r1: real HDL-64 scans have more points than 2*W*H at 64x900; the staging buffers grow, nothing is capped"""
    po, pp = both_params(**sized(900))
    rng = np.random.default_rng(3)
    n = 2 * 900 * 64 + 5000
    d = rng.uniform(3, 60, n); yaw = rng.uniform(-np.pi, np.pi, n); pitch = np.deg2rad(rng.uniform(-24, 2.5, n))
    pts = np.stack([d * np.cos(pitch) * np.cos(yaw), d * np.cos(pitch) * np.sin(yaw), d * np.sin(pitch), np.ones(n)],
                   1).astype(np.float32)
    osl = O.Slam(po); gsl = api.SurfelMapping(pp)
    for _ in range(2):
        osl.process_scan(pts); gsl.processScan(pts)
    assert_bits_equal(gsl.getCurrentPose(), osl.pose(), "pose")
    surfel_fields_equal(gsl.getMap().getAllSurfels(), osl.map.download())
    gsl.ctx.close()


def test_frame_to_frame_objective_with_a_different_model_size():
    """ADVICE r1: the model size is the model TEXTURE's size (textureSize(vertex_model)), here a data-sized frame while
    model_width != data_width"""
    kw = dict(data_width=900, data_height=64, model_width=720, model_height=64)
    po, pp = both_params(**kw)
    ctx = api.Context(pp)
    sc, poses = scans(900, n=2)
    o0, f0 = _prep_both(po, ctx, sc[0], 100)
    o1, f1 = _prep_both(po, ctx, sc[1], 100)
    obj = api.Frame2Model(ctx)
    obj.setData(f1, f0)               # frame-to-frame: both are 900 wide
    obj.initialize(np.eye(4)); obj.jacobianProducts()
    po2 = O.default_params(**sized(900))
    o48, raw = O.icp_jacobian(po2, o1, o0, np.eye(4))
    assert np.array_equal(obj.raw32, raw)
    ctx.close()


def test_minimize_rejects_history_without_iteration_limit():
    po, pp = both_params(**sized(900))
    ctx = api.Context(pp)
    sc, _ = scans(900, n=2)
    _, f0 = _prep_both(po, ctx, sc[0], 100)
    import ctypes as C
    pose = np.zeros(16); T0 = np.eye(4).reshape(16).copy(); hist = np.zeros(64)
    rc = api.lib().sb_icp_minimize(ctx.h, f0.h, f0.h, T0.ctypes.data_as(C.POINTER(C.c_double)), 0, 0.0, 0.0,
                                   C.c_float(1.0), C.c_float(30.0), pose.ctypes.data_as(C.POINTER(C.c_double)), None,
                                   None, hist.ctypes.data_as(C.POINTER(C.c_double)), None)
    assert rc != 0
    ctx.close()


def test_fused_peer_exchange_in_one_gpu_loop_back():
    """the in-kernel all-reduce of the striped Gauss-Newton loop (store sums + epoch stamp into every rank's mailbox,
    spin on the own mailbox) executed with nranks = 1 -- the driver's single-GPU box runs the exchange code path"""
    import ctypes as C
    import os
    po, pp = both_params(**sized(900, max_iterations=8, stopping_threshold=0.0, delta=0.0))
    sc, _ = scans(900, n=4)
    solo = api.SurfelMapping(pp)
    for s in sc:
        solo.processScan(*s)
    ref_pose, ref_n = solo.getCurrentPose().copy(), solo.getMap().size()
    solo.ctx.close()
    os.environ["SUMA_B200_SELF_COMM"] = "1"
    try:
        sl = api.SurfelMapping(pp)
        h = np.zeros(64, np.uint8)
        L = api.lib()
        sl.ctx.check(L.sb_comm_export(sl.ctx.h, C.c_void_p(h.ctypes.data)), "export")
        sl.ctx.check(L.sb_comm_init(sl.ctx.h, 0, 1, C.c_void_p(h.ctypes.data), 0, pp.data_height), "init")
        for s in sc:
            sl.processScan(*s)
        assert_bits_equal(sl.getCurrentPose(), ref_pose, "pose with the exchange in the loop")
        assert sl.getMap().size() == ref_n
        sl.ctx.close()
    finally:
        del os.environ["SUMA_B200_SELF_COMM"]


def test_cuda_equals_reference_shaders_directly():
    """the CUDA path against oracle/_ref (the reference's own shader text on a software GL, pinned built-ins): images,
    index map, surfels and their order, bit for bit -- no hand-written oracle in between"""
    from reference_replay import R   # the reference's outputs, replayed from tests/golden/reference_calls/
    po, pp = both_params(**sized(900))
    ctx = api.Context(pp)
    sc, poses = scans(900, n=3, semantic=True)
    rmap = R.Map(po)
    gmap = api.SurfelMap(ctx)
    out = api.Frame(ctx, 900, 64)
    for t in range(3):
        pts, lab, prb = sc[t]
        rv = R.preprocess(po, pts, lab, prb, timestamp=t)
        f = api.Frame(ctx, 900, 64)
        api.Preprocessing(ctx).process(pts, f, lab, prb, t)
        for g, o, name in zip(f.maps(), rv, ("vertex", "normal", "semantic")):
            assert_bits_equal(g, o, "t=%d preprocess %s" % (t, name))
        pose = (np.linalg.inv(poses[0]) @ poses[t]).astype(np.float32)
        rr = rmap.render(pose, pose, 0.05 * t)
        gmap.render(pose, pose, out, 0.05 * t)
        for g, o, name in zip(out.maps(), rr, ("vertex", "normal", "semantic")):
            assert_bits_equal(g, o, "t=%d render %s" % (t, name))
        rmap.update(pose, rv)
        gmap.update(pose, f)
        ri, rrad, rint, rnu, rnn = rmap.update_debug()
        gi, grad, gint, gnu, gnn = gmap.update_debug()
        assert_bits_equal(gi, ri, "t=%d index map" % t)
        assert_bits_equal(gint, rint, "t=%d integrated flags" % t)
        assert (gnu, gnn) == (rnu, rnn)
        surfel_fields_equal(gmap.getAllSurfels(), rmap.download(), "t=%d surfels" % t)
    # K5: exact fixed-point sums against the shader's fp32 blending: 1e-5 of the matrix scale (north_star)
    rv0 = R.preprocess(po, *sc[0], timestamp=50); rv1 = R.preprocess(po, *sc[1], timestamp=50)
    f0 = api.Frame(ctx, 900, 64); f1 = api.Frame(ctx, 900, 64)
    api.Preprocessing(ctx).process(sc[0][0], f0, sc[0][1], sc[0][2], 50)
    api.Preprocessing(ctx).process(sc[1][0], f1, sc[1][1], sc[1][2], 50)
    obj = api.Frame2Model(ctx)
    obj.setData(f1, f0)
    T = np.linalg.inv(poses[0]) @ poses[1]
    obj.initialize(T); obj.jacobianProducts()
    rf = R.icp_jacobian(po, rv1, rv0, T).astype(np.float64)
    m, e = rf[:36].reshape(6, 6), np.asarray(obj.out48[:36]).reshape(6, 6)
    scale = np.sqrt(np.outer(np.diag(e), np.diag(e)))
    assert np.max(np.abs(m - e) / scale) < 1e-5
    assert (rf[42], rf[44], rf[46]) == (obj.out48[42], obj.out48[44], obj.out48[46])
    ctx.close()


def test_loop_closure_detection_and_verification_bit_exact():
    """SurfelMapping::checkLoopClosure (SurfelMapping.cpp:527-795) on a synthetic loop: a circle of 120 scans driven a
    second time. Detection (render_inactive at the candidate pose + three Gauss-Newton runs against the old map frame),
    the composed rendering, the verification over consecutive scans, the loop edges and the chained old pose must agree
    with the oracle twin at every scan -- decisions, counters, float ratios and pose bits."""
    from semantic_suma_b200 import synth
    po, pp = both_params(**sized(900))
    scene = synth.Scene(width=900, height=64)
    N = 124
    poses = synth.trajectory(N, step=0.2618, yaw_deg=3.0)
    lp = dict(search_distance=3.0, min_trajectory_distance=15.0, min_verifications=2)
    osl = O.Slam(po)
    osl.enable_loop_closure(**lp)
    gsl = api.SurfelMapping(pp)
    gsl.enableLoopClosure(True, **lp)
    keys = ("loop_count", "time_without_loop_closure", "candidates_tested", "loop_edges_added", "unverified",
            "already_verified", "found_candidate", "use_candidate", "optimisation_requested", "last_added_candidate",
            "n_edges", "n_poses")
    for f in range(N):
        pts, _, _ = scene.scan(f, poses[f])
        osl.process_scan(pts)
        gsl.processScan(pts)
        assert_bits_equal(gsl.getCurrentPose(), osl.pose(), "t=%d pose" % f)
        if f >= 100:
            a, b = gsl.getLoopInfo(), osl.loop_info()
            for k in keys:
                assert a[k] == b[k], "t=%d %s: %r vs %r" % (f, k, a[k], b[k])
            if b["found_candidate"]:
                for k in ("valid_ratio", "outlier_ratio", "rel_error"):
                    assert_bits_equal(np.float32(a[k]), np.float32(b[k]), "t=%d %s" % (f, k))
                assert_bits_equal(a["current_pose_old"], b["current_pose_old"], "t=%d currentPose_old" % f)
        assert gsl.getMap().size() == osl.map.size(), "t=%d surfel count" % f
    info = osl.loop_info()
    assert info["loop_edges_added"] >= 3 and info["already_verified"] == 1, "the sequence must close the loop: %r" % info
    eg, eo = gsl.getLoopEdges(), osl.loop_edges()
    assert len(eg) == len(eo)
    for (f1, t1, r1), (f2, t2, r2) in zip(eg, eo):
        assert (f1, t1) == (f2, t2)
        assert_bits_equal(r1, r2, "edge %d->%d" % (f1, t1))
    surfel_fields_equal(gsl.getMap().getAllSurfels(), osl.map.download(), "surfels after the loop")
    gsl.ctx.close()

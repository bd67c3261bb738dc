"""TEST INFRASTRUCTURE: ctypes binding of oracle/_ref -- the reference's own GLSL shaders, transpiled to C++ from
/root/reference/src/shader by oracle/ref_harness/glsl2cpp.py and driven by a minimal software GL
(oracle/ref_harness/ref_pipeline.cpp). Two builds:

  mode="pinned"   GLSL built-ins follow the rules the oracle pins (orc_math.h)  -> must equal oracle/ bit for bit
  mode="precise"  GLSL built-ins in fp64 / libm                                 -> an independent legal GL

Only tests/ (and __graft_entry__.build(), which compiles it) may touch this module; the product never does.
/root/reference exists only in the build container: on the GPU box the prebuilt oracle/_ref/*.so are used as shipped.
"""
import ctypes as C
import os
import subprocess

import numpy as np

from . import oracle as O

_HERE = os.path.dirname(os.path.abspath(__file__))
_HARNESS = os.path.join(_HERE, "ref_harness")
_OUT = os.path.join(_HERE, "_ref")
REFERENCE = os.environ.get("SUMA_REFERENCE_DIR", "/root/reference")


def lib_path(mode):
    return os.path.join(_OUT, "libsuma_ref_%s.so" % mode)


def have_reference():
    return os.path.isdir(os.path.join(REFERENCE, "src", "shader"))


def available():
    return have_reference() or all(os.path.exists(lib_path(m)) for m in ("pinned", "precise"))


def build(force=False):
    """(re)build oracle/_ref from the reference's sources where they lie; no-op when /root/reference is absent"""
    if not have_reference():
        return available()
    cmd = ["make", "-C", _HARNESS, "-s", "-j%d" % max(1, min(8, os.cpu_count() or 1)), "REFERENCE=" + REFERENCE] + \
        (["-B"] if force else [])
    subprocess.check_call(cmd)
    return True


_libs = {}


def lib(mode="pinned"):
    if mode not in _libs:
        build()
        L = C.CDLL(lib_path(mode))
        L.ref_map_create.restype = C.c_void_p
        L.ref_map_size.restype = C.c_uint32
        L.ref_map_timestamp.restype = C.c_uint32
        L.ref_map_download.restype = C.c_uint32
        L.ref_math_mode.restype = C.c_char_p
        assert L.ref_math_mode().decode() == mode
        _libs[mode] = L
    return _libs[mode]


_p, _f32, colmajor = O._p, O._f32, O.colmajor


def preprocess(p, pts, labels=None, probs=None, timestamp=100, mode="pinned"):
    pts = _f32(pts); labels = _f32(labels); probs = _f32(probs)
    H, W = p.data_height, p.data_width
    v = np.empty((H, W, 4), np.float32); nm = np.empty_like(v); s = np.empty_like(v)
    lib(mode).ref_preprocess(C.byref(p), _p(pts), _p(labels), _p(probs), C.c_uint32(pts.shape[0]), C.c_uint32(timestamp),
                             _p(v), _p(nm), _p(s))
    return v, nm, s


def icp_jacobian(p, data, model, pose, iteration=0, max_distance=None, max_angle=None, entries_per_kernel=64,
                 semantic=True, mode="pinned"):
    """the 2x8 RGB32F blend texture of Frame2Model::jacobianProducts as 48 floats (fp32 additive blending)"""
    dv, dn, ds = [_f32(a) for a in data]
    mv, mn, ms = [_f32(a) for a in model]
    if not semantic:
        ds = ms = None
    out48 = np.zeros(48, np.float32)
    lib(mode).ref_icp_jacobian(C.byref(p), _p(dv), _p(dn), _p(ds), _p(mv), _p(mn), _p(ms),
                               _p(colmajor(pose, np.float64), C.c_double), C.c_int32(iteration),
                               C.c_float(p.icp_max_distance if max_distance is None else max_distance),
                               C.c_float(p.icp_max_angle if max_angle is None else max_angle),
                               C.c_int32(entries_per_kernel), _p(out48))
    return out48


class Map:
    """SurfelMap driven through the reference's shaders (no submap paging: that is host code, not a shader)"""

    def __init__(self, p, mode="pinned"):
        self.p, self.L = p, lib(mode)
        self.h = C.c_void_p(self.L.ref_map_create(C.byref(p)))

    def __del__(self):
        if getattr(self, "h", None):
            self.L.ref_map_destroy(self.h); self.h = None

    def size(self):
        return self.L.ref_map_size(self.h)

    def timestamp(self):
        return self.L.ref_map_timestamp(self.h)

    def download(self):
        n = self.size()
        a = np.zeros(max(n, 1), O.SURFEL_DTYPE)
        k = self.L.ref_map_download(self.h, a.ctypes.data_as(C.c_void_p), C.c_uint32(n))
        return a[:k]

    def upload(self, surfels, timestamp):
        a = np.ascontiguousarray(surfels, O.SURFEL_DTYPE)
        self.L.ref_map_upload(self.h, a.ctypes.data_as(C.c_void_p), C.c_uint32(a.shape[0]), C.c_uint32(timestamp))

    def set_pose(self, t, pose):
        self.L.ref_map_set_pose(self.h, C.c_uint32(t), _p(colmajor(pose, np.float32)))

    def derived(self):
        a = np.zeros(6, np.float32)
        self.L.ref_map_derived(self.h, _p(a))
        return dict(zip(("pixel_size", "p_unstable", "log_prior", "log_unstable", "radconf_angle_thresh",
                         "update_angle_thresh"), a.tolist()))

    def _mframe(self):
        H, W = self.p.model_height, self.p.model_width
        return [np.zeros((H, W, 4), np.float32) for _ in range(3)]

    def render(self, pose_old, pose_new, conf_thr):
        v, n, s = self._mframe()
        self.L.ref_map_render(self.h, _p(colmajor(pose_old, np.float32)), _p(colmajor(pose_new, np.float32)),
                              C.c_float(conf_thr), _p(v), _p(n), _p(s))
        return v, n, s

    def render_active(self, pose, conf_thr):
        self.L.ref_map_render_active(self.h, _p(colmajor(pose, np.float32)), C.c_float(conf_thr))

    def render_inactive(self, pose, conf_thr):
        self.L.ref_map_render_inactive(self.h, _p(colmajor(pose, np.float32)), C.c_float(conf_thr))

    def render_composed(self, pose_old, pose_new, conf_thr):
        self.L.ref_map_render_composed(self.h, _p(colmajor(pose_old, np.float32)), _p(colmajor(pose_new, np.float32)),
                                       C.c_float(conf_thr))

    def frame(self, which):
        v, n, s = self._mframe()
        self.L.ref_map_get_frame(self.h, C.c_int(which), _p(v), _p(n), _p(s))
        return v, n, s

    def update(self, pose, frame):
        fv, fn, fs = [_f32(a) for a in frame]
        self.L.ref_map_update(self.h, _p(colmajor(pose, np.float32)), _p(fv), _p(fn), _p(fs))

    def update_debug(self):
        H, W = self.p.data_height, self.p.data_width
        idx = np.zeros((H, W), np.uint32); rad = np.zeros((H, W, 4), np.float32); integ = np.zeros((H, W), np.uint8)
        nu, nn = C.c_uint32(0), C.c_uint32(0)
        self.L.ref_map_get_update_debug(self.h, _p(idx, C.c_uint32), _p(rad), _p(integ, C.c_uint8), C.byref(nu),
                                        C.byref(nn))
        return idx, rad, integ, nu.value, nn.value


# ------------------------------------------------------------------------------------------------------------------
# libsuma_ref_host.so: the reference's own HOST sources (core/lie_algebra.cpp, core/LieGaussNewton.cpp + Objective.h,
# util/kitti_utils.cpp, rv/ParameterList + XML parser) compiled where they lie against stand-ins for Eigen / Boost
# (oracle/ref_harness/host/). Compared within tolerances, never bit for bit: Eigen's own operation order is not ours.
# ------------------------------------------------------------------------------------------------------------------
def host_available():
    return have_reference() or os.path.exists(lib_path("host"))


_host = None
PRODUCTS_FN = C.CFUNCTYPE(C.c_double, C.c_void_p, C.POINTER(C.c_double), C.c_int, C.POINTER(C.c_double),
                          C.POINTER(C.c_double))


def host_lib():
    global _host
    if _host is None:
        build()
        L = C.CDLL(lib_path("host"))
        L.ref_kitti_rotation_error.restype = C.c_float
        L.ref_kitti_translation_error.restype = C.c_float
        _host = L
    return _host


def se3_exp(x):
    x = np.ascontiguousarray(x, np.float64); T = np.zeros(16, np.float64)
    host_lib().ref_se3_exp(_p(x, C.c_double), _p(T, C.c_double))
    return O.from_colmajor(T)


def se3_log(T):
    Tc = colmajor(T, np.float64); x = np.zeros(6, np.float64)
    host_lib().ref_se3_log(_p(Tc, C.c_double), _p(x, C.c_double))
    return x


def gn_minimize(products, T0, max_iter, eps, delta, hist_cap=512):
    """LieGaussNewton::minimize of the reference on an objective whose jacobianProducts is `products(pose 4x4, iteration)
    -> (JtJ 6x6, Jtf 6, F)`. Returns dict(pose, history, iterations, residual, ret)."""
    def cb(_user, pose, iteration, A, b):
        P = O.from_colmajor(np.array([pose[i] for i in range(16)], np.float64))
        JtJ, Jtf, F = products(P, iteration)
        JtJ = np.asarray(JtJ, np.float64); Jtf = np.asarray(Jtf, np.float64).reshape(6)
        for c in range(6):
            for r in range(6):
                A[6 * c + r] = JtJ[r, c]
        for r in range(6):
            b[r] = Jtf[r]
        return float(F)

    fn = PRODUCTS_FN(cb)
    pose = np.zeros(16, np.float64); hist = np.zeros(16 * hist_cap, np.float64)
    hl, it, res = C.c_int(0), C.c_int(0), C.c_double(0)
    ret = host_lib().ref_gn_minimize(fn, None, _p(colmajor(T0, np.float64), C.c_double), C.c_int(max_iter),
                                     C.c_double(eps), C.c_double(delta), _p(pose, C.c_double), _p(hist, C.c_double),
                                     C.c_int(hist_cap), C.byref(hl), C.byref(it), C.byref(res))
    return {"pose": O.from_colmajor(pose), "history": [O.from_colmajor(hist[16 * i:16 * i + 16]) for i in range(min(hl.value, hist_cap))],
            "history_len": hl.value, "iterations": it.value, "residual": res.value, "ret": ret}


def param_lookup(xml_file, name):
    buf = C.create_string_buffer(4096)
    r = host_lib().ref_param_lookup(str(xml_file).encode(), name.encode(), buf, C.c_int(4096))
    return buf.value.decode() if r == 0 else None


def param_names(xml_file):
    buf = C.create_string_buffer(1 << 16)
    n = host_lib().ref_param_names(str(xml_file).encode(), buf, C.c_int(1 << 16))
    if n < 0:
        raise RuntimeError("reference XML parser failed on %s" % xml_file)
    return [s for s in buf.value.decode().split("\n") if s]


def _poses_rowmajor(poses):
    return np.ascontiguousarray(np.asarray([np.asarray(P, np.float32) for P in poses], np.float32).reshape(-1, 16))


def kitti_load_poses(path, cap=100000):
    out = np.zeros((cap, 16), np.float32)
    n = host_lib().ref_kitti_load_poses(str(path).encode(), _p(out), C.c_int(cap))
    if n < 0:
        return None  # the reference throws (boost::bad_lexical_cast)
    return [out[i].reshape(4, 4).copy() for i in range(min(n, cap))]


def kitti_calibration(path, name):
    out = np.zeros(16, np.float32)
    r = host_lib().ref_kitti_calibration(str(path).encode(), name.encode(), _p(out))
    return out.reshape(4, 4) if r == 0 else None


def kitti_trajectory_distances(poses):
    P = _poses_rowmajor(poses); d = np.zeros(P.shape[0], np.float32)
    host_lib().ref_kitti_trajectory_distances(_p(P), C.c_int(P.shape[0]), _p(d))
    return d


def kitti_rotation_error(E):
    return float(host_lib().ref_kitti_rotation_error(_p(_poses_rowmajor([E]))))


def kitti_translation_error(E):
    return float(host_lib().ref_kitti_translation_error(_p(_poses_rowmajor([E]))))


def kitti_last_frame(dist, first_frame, length):
    d = np.ascontiguousarray(dist, np.float32)
    return int(host_lib().ref_kitti_last_frame(_p(d), C.c_int(d.shape[0]), C.c_int(first_frame), C.c_float(length)))


def kitti_sequence_errors(gt, res, cap=200000):
    G, R_ = _poses_rowmajor(gt), _poses_rowmajor(res)
    out = np.zeros((cap, 5), np.float32)
    n = host_lib().ref_kitti_sequence_errors(_p(G), _p(R_), C.c_int(G.shape[0]), _p(out), C.c_int(cap))
    return out[:min(n, cap)].copy()


def kitti_save_stats(rows, directory):
    rows = np.ascontiguousarray(rows, np.float32)
    host_lib().ref_kitti_save_stats(_p(rows), C.c_int(rows.shape[0]), str(directory).encode())
    t, r = open(os.path.join(str(directory), "stats.txt")).read().split()
    return float(t), float(r)


# ------------------------------------------------------------------------------------------------------------------
# libsuma_ref_full.so: the reference's own CORE CLASSES -- Preprocessing, Frame2Model, LieGaussNewton, SurfelMap,
# SurfelMapping (the whole processScan incl. track-loss fallback, submap paging and checkLoopClosure) -- compiled where
# they lie against a stand-in glow on a generic software GL (oracle/ref_harness/full/) and driving the reference's own
# transpiled shaders. What the GL / Eigen / libm implementations leave open is pinned to the oracle's rules
# (REF_MATH_PINNED, MINI_EIGEN_PINNED, pinned_libm.h), and the oracle can sum the 48 ICP values the GL way
# (O.gl_sums): then reference and oracle must agree BIT FOR BIT over whole runs.
# ------------------------------------------------------------------------------------------------------------------
def full_available():
    return have_reference() or os.path.exists(lib_path("full"))


DEFAULT_XML = os.path.join(REFERENCE, "config", "default.xml")
_full = {}


def full_lib(mode="pinned"):
    """mode "pinned": what GL / Eigen / libm leave open follows the oracle's rules (bit-for-bit comparisons); "precise": nothing
    is pinned -- GLSL built-ins in fp64/libm, general matrix inverse, left-looking LDLT, libm sin/cos (tolerance comparisons)"""
    if mode not in _full:
        build()
        L = C.CDLL(lib_path("full" if mode == "pinned" else "full_precise"))
        L.reffull_create.restype = C.c_void_p
        L.reffull_error.restype = C.c_char_p
        for f in ("reffull_map_size", "reffull_map_download", "reffull_slam_timestamp", "reffull_slam_edges"):
            getattr(L, f).restype = C.c_uint32
        L.reffull_slam_statistic.restype = C.c_double
        L.reffull_draw_calls.restype = C.c_uint64
        _full[mode] = L
    return _full[mode]


class Full:
    """one parameter list + lazily constructed Preprocessing / SurfelMap / SurfelMapping of the reference"""

    def __init__(self, p, zero_stale_tail=True, mode="pinned", **extra):
        self.p = p
        self.L = full_lib(mode)
        xml = DEFAULT_XML if os.path.exists(DEFAULT_XML) else ""
        self.h = C.c_void_p(self.L.reffull_create(C.byref(p), xml.encode()))
        self._check(0)
        self.L.reffull_zero_stale_tail(C.c_int(1 if zero_stale_tail else 0))
        for k, v in extra.items():
            name = k.encode()
            if isinstance(v, bool):
                self.L.reffull_set_bool(self.h, name, C.c_int(int(v)))
            elif isinstance(v, int):
                self.L.reffull_set_int(self.h, name, C.c_int(v))
            else:
                self.L.reffull_set_float(self.h, name, C.c_double(float(v)))

    def __del__(self):
        if getattr(self, "h", None):
            self.L.reffull_destroy(self.h); self.h = None

    def zero_stale_tail(self, on):
        """process-wide: whether the next scans read 0 (not the previous scan's values) past the labels just uploaded"""
        self.L.reffull_zero_stale_tail(C.c_int(1 if on else 0))

    def _check(self, r):
        err = self.L.reffull_error(self.h).decode()
        if r != 0 or err:
            raise RuntimeError("reference (full): " + err)

    def param(self, name):
        buf = C.create_string_buffer(1024)
        r = self.L.reffull_param(self.h, name.encode(), buf, C.c_int(1024))
        return buf.value.decode() if r == 0 else None

    def _dframe(self):
        return [np.zeros((self.p.data_height, self.p.data_width, 4), np.float32) for _ in range(3)]

    def _mframe(self):
        return [np.zeros((self.p.model_height, self.p.model_width, 4), np.float32) for _ in range(3)]

    # ---- Preprocessing / Frame2Model / LieGaussNewton ----
    def preprocess(self, pts, labels=None, probs=None, timestamp=100):
        pts = _f32(pts); n = pts.shape[0]
        labels = _f32(labels) if labels is not None else None; probs = _f32(probs) if probs is not None else None
        v, nm, s = self._dframe()
        self._check(self.L.reffull_preprocess(self.h, _p(pts), _p(labels) if labels is not None else None,
                                              _p(probs) if probs is not None else None, C.c_uint32(n),
                                              C.c_uint32(timestamp), _p(v), _p(nm), _p(s)))
        return v, nm, s

    def icp_jacobian(self, data, model, pose, iteration=0, max_distance=None, max_angle=None):
        a = [_f32(x) for x in list(data) + list(model)]
        out = np.zeros(48, np.float64)
        self._check(self.L.reffull_icp_jacobian(self.h, *[_p(x) for x in a], _p(colmajor(pose, np.float64), C.c_double),
                                                C.c_int32(iteration),
                                                C.c_float(self.p.icp_max_distance if max_distance is None else max_distance),
                                                C.c_float(self.p.icp_max_angle if max_angle is None else max_angle),
                                                _p(out, C.c_double)))
        return out

    def icp_minimize(self, data, model, T0, hist_cap=300):
        a = [_f32(x) for x in list(data) + list(model)]
        pose = np.zeros(16, np.float64); hist = np.zeros(16 * hist_cap, np.float64); hl = C.c_int(0)
        k = self.L.reffull_icp_minimize(self.h, *[_p(x) for x in a], _p(colmajor(T0, np.float64), C.c_double),
                                        _p(pose, C.c_double), _p(hist, C.c_double), C.c_int(hist_cap), C.byref(hl))
        self._check(0 if k >= 0 else -1)
        return O.from_colmajor(pose), k, [O.from_colmajor(hist[16 * i:16 * i + 16]) for i in range(min(hl.value, hist_cap))]

    # ---- SurfelMap ----
    def map_size(self):
        return int(self.L.reffull_map_size(self.h))

    def map_download(self):
        n = self.map_size()
        a = np.zeros(max(n, 1), O.SURFEL_DTYPE)
        k = self.L.reffull_map_download(self.h, a.ctypes.data_as(C.c_void_p), C.c_uint32(n))
        return a[:k]

    def map_upload(self, surfels, timestamp):
        a = np.ascontiguousarray(surfels, O.SURFEL_DTYPE)
        self._check(self.L.reffull_map_upload(self.h, a.ctypes.data_as(C.c_void_p), C.c_uint32(a.shape[0]), C.c_uint32(timestamp)))

    def map_set_pose(self, t, pose):
        self._check(self.L.reffull_map_set_pose(self.h, C.c_uint32(t), _p(colmajor(pose, np.float32))))

    def map_update(self, pose, frame):
        fv, fn, fs = [_f32(a) for a in frame]
        self._check(self.L.reffull_map_update(self.h, _p(colmajor(pose, np.float32)), _p(fv), _p(fn), _p(fs)))

    def map_render(self, pose_old, pose_new, conf_thr):
        v, n, s = self._mframe()
        self._check(self.L.reffull_map_render(self.h, _p(colmajor(pose_old, np.float32)), _p(colmajor(pose_new, np.float32)),
                                              C.c_float(conf_thr), _p(v), _p(n), _p(s)))
        return v, n, s

    def map_render_active(self, pose, conf_thr):
        self._check(self.L.reffull_map_render_active(self.h, _p(colmajor(pose, np.float32)), C.c_float(conf_thr)))

    def map_render_inactive(self, pose, conf_thr):
        self._check(self.L.reffull_map_render_inactive(self.h, _p(colmajor(pose, np.float32)), C.c_float(conf_thr)))

    def map_render_composed(self, pose_old, pose_new, conf_thr):
        self._check(self.L.reffull_map_render_composed(self.h, _p(colmajor(pose_old, np.float32)),
                                                       _p(colmajor(pose_new, np.float32)), C.c_float(conf_thr)))

    def map_frame(self, which):
        v, n, s = self._mframe()
        self._check(self.L.reffull_map_get_frame(self.h, C.c_int(which), _p(v), _p(n), _p(s)))
        return v, n, s

    # ---- SurfelMapping ----
    def process_scan(self, pts, labels=None, probs=None):
        pts = _f32(pts)
        labels = _f32(labels) if labels is not None else None; probs = _f32(probs) if probs is not None else None
        self._check(self.L.reffull_slam_process_scan(self.h, _p(pts), _p(labels) if labels is not None else None,
                                                     _p(probs) if probs is not None else None, C.c_uint32(pts.shape[0])))

    def pose(self):
        a = np.zeros(16, np.float64)
        self.L.reffull_slam_pose(self.h, _p(a, C.c_double))
        return O.from_colmajor(a)

    def timestamp(self):
        return int(self.L.reffull_slam_timestamp(self.h))

    def statistic(self, name):
        return float(self.L.reffull_slam_statistic(self.h, name.encode()))

    def slam_frame(self, which):
        """0 currentFrame, 1 lastFrame (data size); 2 currentModelFrame, 3 lastModelFrame (model size)"""
        v, n, s = self._dframe() if which < 2 else self._mframe()
        self._check(self.L.reffull_slam_frame(self.h, C.c_int(which), _p(v), _p(n), _p(s)))
        return v, n, s

    def loop_flags(self):
        return bool(self.L.reffull_slam_found_loop_candidate(self.h)), bool(self.L.reffull_slam_use_loop_candidate(self.h))

    def edges(self, cap=4096):
        ft = np.zeros((cap, 2), np.int32)
        n = self.L.reffull_slam_edges(self.h, _p(ft, C.c_int32), C.c_uint32(cap))
        return [(int(ft[i, 0]), int(ft[i, 1])) for i in range(min(n, cap))]

"""ctypes binding of oracle/oracle_api.h — TEST INFRASTRUCTURE ONLY.

Loads either CPU checker:
  kind="port"       oracle/libmcl3dl_oracle.so   (repo-owned restatement, always available)
  kind="reference"  oracle/_ref/libmcl3dl_ref.so (reference's own sources; prebuilt in the dev container)

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may import
this module.  The product package (mcl_3dl_b200/) never does.
"""
import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))

POINT = np.dtype([("x", "<f4"), ("y", "<f4"), ("z", "<f4"), ("label", "<u4")])
POSE = np.dtype([("px", "<f4"), ("py", "<f4"), ("pz", "<f4"), ("_pad", "<f4"),
                 ("qx", "<f4"), ("qy", "<f4"), ("qz", "<f4"), ("qw", "<f4")])
RESULT = np.dtype([("score_like", "<f4"), ("match_cnt", "<u4"), ("score_beam", "<f4"),
                   ("n_short", "<u4"), ("n_hit", "<u4"), ("n_long", "<u4")])


class LikParams(C.Structure):
    _fields_ = [("match_weight", C.c_float), ("match_dist_min", C.c_float), ("match_dist_flat", C.c_float),
                ("dist_weight", C.c_float * 3)]


class BeamParams(C.Structure):
    _fields_ = [("map_grid_size", C.c_double * 3), ("dda_grid_size", C.c_double), ("ray_angle_half", C.c_double),
                ("hit_tolerance", C.c_double), ("hit_range_sq", C.c_float), ("sin_total_ref", C.c_float),
                ("beam_likelihood", C.c_float), ("beam_likelihood_min", C.c_float),
                ("filter_label_max", C.c_uint32), ("add_penalty_short_only_mode", C.c_int32),
                ("use_raycast_using_dda", C.c_int32), ("_reserved", C.c_int32)]

    def as_tuple(self):
        return (tuple(self.map_grid_size), self.dda_grid_size, self.ray_angle_half, self.hit_tolerance,
                self.hit_range_sq, self.sin_total_ref, self.beam_likelihood, self.beam_likelihood_min,
                self.filter_label_max, self.add_penalty_short_only_mode, self.use_raycast_using_dda)


class BeamRaw(C.Structure):
    _fields_ = [("map_grid_x", C.c_float), ("map_grid_y", C.c_float), ("map_grid_z", C.c_float),
                ("num_points_default", C.c_uint64), ("beam_likelihood_min", C.c_float),
                ("ang_total_ref", C.c_float), ("filter_label_max", C.c_uint32), ("hit_range", C.c_float),
                ("add_penalty_short_only_mode", C.c_int32), ("use_raycast_using_dda", C.c_int32),
                ("ray_angle_half", C.c_float), ("dda_grid_size", C.c_float)]


MOTION_STATE = np.dtype([("pos", "<f4", 3), ("rot", "<f4", 4), ("noise_ll", "<f4"), ("noise_la", "<f4"),
                         ("noise_al", "<f4"), ("noise_aa", "<f4"), ("odom_err_integ_lin", "<f4", 3),
                         ("odom_err_integ_ang", "<f4", 3)])


def lik_params(match_weight=5.0, match_dist_min=0.2, match_dist_flat=0.05, dist_weight=(1.0, 1.0, 1.0)):
    """Defaults: include/mcl_3dl/parameters.h:74-76."""
    p = LikParams()
    p.match_weight, p.match_dist_min, p.match_dist_flat = match_weight, match_dist_min, match_dist_flat
    p.dist_weight[:] = dist_weight
    return p


def beam_raw(map_grid=(0.1, 0.1, 0.1), num_points_default=3, beam_likelihood_min=0.2,
             ang_total_ref=np.pi / 6.0, filter_label_max=0xFFFFFFFF, hit_range=0.3,
             add_penalty_short_only_mode=True, ray_angle_half=0.25 * np.pi / 180.0, dda_grid_size=0.2,
             use_raycast_using_dda=True):
    """Defaults: include/mcl_3dl/parameters.h:95-111, except use_raycast_using_dda (reference default: false)."""
    r = BeamRaw()
    r.map_grid_x, r.map_grid_y, r.map_grid_z = map_grid
    r.num_points_default = num_points_default
    r.beam_likelihood_min = beam_likelihood_min
    r.ang_total_ref = ang_total_ref
    r.filter_label_max = filter_label_max
    r.hit_range = hit_range
    r.add_penalty_short_only_mode = 1 if add_penalty_short_only_mode else 0
    r.use_raycast_using_dda = 1 if use_raycast_using_dda else 0
    r.ray_angle_half = ray_angle_half
    r.dda_grid_size = dda_grid_size
    return r


def points(xyz, label=None):
    xyz = np.asarray(xyz, dtype=np.float32).reshape(-1, 3)
    out = np.zeros(len(xyz), dtype=POINT)
    out["x"], out["y"], out["z"] = xyz[:, 0], xyz[:, 1], xyz[:, 2]
    if label is not None:
        out["label"] = np.asarray(label, dtype=np.uint32)
    return out


def poses(pos, quat):
    pos = np.asarray(pos, dtype=np.float32).reshape(-1, 3)
    quat = np.asarray(quat, dtype=np.float32).reshape(-1, 4)
    out = np.zeros(len(pos), dtype=POSE)
    out["px"], out["py"], out["pz"] = pos[:, 0], pos[:, 1], pos[:, 2]
    out["qx"], out["qy"], out["qz"], out["qw"] = quat[:, 0], quat[:, 1], quat[:, 2], quat[:, 3]
    return out


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None and a.size else None


def lib_path(kind):
    if kind == "port":
        return os.path.join(HERE, "libmcl3dl_oracle.so")
    if kind == "reference":
        return os.path.join(HERE, "_ref", "libmcl3dl_ref.so")
    if kind == "adapter":
        return os.path.join(HERE, "_ref", "adapter_parity_test")
    raise ValueError(kind)


def build(kind="port", quiet=True):
    """Compile the checker if its .so is missing (make in oracle/).  kind="adapter": the host C++ adapter's parity
    program, which links the engine library (build that first)."""
    path = lib_path(kind)
    target = {"port": [], "reference": ["ref"], "adapter": ["adapter"]}[kind]
    if kind == "reference" and not os.path.isdir("/root/reference/include/mcl_3dl"):
        return os.path.exists(path)
    r = subprocess.run(["make", "-C", HERE] + target, capture_output=quiet, text=True)
    if r.returncode != 0:
        raise RuntimeError("oracle build failed:\n" + (r.stdout or "") + (r.stderr or ""))
    return os.path.exists(path)


def available(kind):
    return os.path.exists(lib_path(kind))


class CpuChecker:
    """One loaded checker library ("port" or "reference")."""

    def __init__(self, kind="port"):
        path = lib_path(kind)
        if not os.path.exists(path):
            build(kind)
        self.lib = L = C.CDLL(path)
        self.kind = kind
        L.mcl3dl_cpu_kind.restype = C.c_char_p
        assert L.mcl3dl_cpu_kind().decode() == kind
        L.mcl3dl_cpu_create.restype = C.c_void_p
        L.mcl3dl_cpu_create.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_float, C.c_float]
        L.mcl3dl_cpu_destroy.argtypes = [C.c_void_p]
        L.mcl3dl_cpu_measure.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p,
                                         C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p, C.c_int]
        L.mcl3dl_cpu_set_tally.argtypes = [C.c_void_p, C.c_int]
        L.mcl3dl_cpu_beam_status.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t,
                                             C.c_void_p, C.c_size_t, C.c_void_p]
        L.mcl3dl_cpu_beam_params.argtypes = [C.c_void_p, C.c_void_p]
        L.mcl3dl_cpu_radius_search.argtypes = [C.c_void_p, C.c_void_p, C.c_float, C.c_void_p]
        L.mcl3dl_cpu_dda_walk.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int,
                                          C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
        L.mcl3dl_cpu_kd_walk.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int,
                                         C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
        L.mcl3dl_cpu_quat_rotate.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        L.mcl3dl_cpu_transform_point.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        L.mcl3dl_cpu_pf_update.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
        L.mcl3dl_cpu_pf_estimate.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_float, C.c_float,
                                             C.c_void_p, C.c_void_p, C.c_void_p]
        L.mcl3dl_cpu_filter_clip.argtypes = [C.c_void_p, C.c_size_t, C.c_float, C.c_float, C.c_float, C.c_float, C.c_void_p]
        L.mcl3dl_cpu_global_localization_points.argtypes = [C.c_size_t] * 4
        L.mcl3dl_cpu_global_localization_points.restype = C.c_size_t
        L.mcl3dl_cpu_motion_predict.argtypes = [C.c_void_p, C.c_void_p, C.c_float, C.c_float, C.c_float, C.c_void_p,
                                                C.c_size_t]
        L.mcl3dl_cpu_pf_resample_6dof.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_uint, C.c_void_p, C.c_void_p,
                                                  C.c_void_p, C.c_void_p]
        L.mcl3dl_cpu_pf_resample_1d.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_uint, C.c_float, C.c_void_p,
                                                C.c_void_p]

    def create(self, map_pts, lik=None, beam=None, chunk_length=20.0, max_search_radius=0.4):
        return CpuMap(self, map_pts, lik, beam, chunk_length, max_search_radius)

    def dda_walk(self, map_pts, ctor, begin, end, stop_at_collision=True, max_out=4096):
        map_pts = np.ascontiguousarray(map_pts, dtype=POINT)
        ctor = np.asarray(ctor, dtype=np.float64)
        assert ctor.shape == (6,)
        b = np.asarray(begin, dtype=np.float32)
        e = np.asarray(end, dtype=np.float32)
        centres = np.zeros((max_out, 3), dtype=np.float32)
        coll = np.zeros(max_out, dtype=np.uint8)
        cid = C.c_int(-1)
        n = self.lib.mcl3dl_cpu_dda_walk(_ptr(map_pts), len(map_pts), _ptr(ctor), _ptr(b), _ptr(e),
                                         1 if stop_at_collision else 0, _ptr(centres), _ptr(coll), max_out,
                                         C.byref(cid))
        assert 0 <= n <= max_out
        return centres[:n].copy(), coll[:n].astype(bool), cid.value

    def kd_walk(self, map_pts, ctor, begin, end, stop_at_collision=True, max_out=4096):
        """RaycastUsingKDTree(gx, gy, gz, hit_tolerance) walk -> (positions, collision flags, sin_angle, first id)."""
        map_pts = np.ascontiguousarray(map_pts, dtype=POINT)
        ctor = np.asarray(ctor, dtype=np.float32)
        assert ctor.shape == (4,)
        b = np.asarray(begin, dtype=np.float32)
        e = np.asarray(end, dtype=np.float32)
        pos = np.zeros((max_out, 3), dtype=np.float32)
        coll = np.zeros(max_out, dtype=np.uint8)
        sa = np.zeros(max_out, dtype=np.float32)
        cid = C.c_int(-1)
        n = self.lib.mcl3dl_cpu_kd_walk(_ptr(map_pts), len(map_pts), _ptr(ctor), _ptr(b), _ptr(e),
                                        1 if stop_at_collision else 0, _ptr(pos), _ptr(coll), _ptr(sa), max_out,
                                        C.byref(cid))
        assert 0 <= n <= max_out
        return pos[:n].copy(), coll[:n].astype(bool), sa[:n].copy(), cid.value

    def quat_rotate(self, q, v):
        q = np.asarray(q, dtype=np.float32)
        v = np.asarray(v, dtype=np.float32)
        out = np.zeros(3, dtype=np.float32)
        self.lib.mcl3dl_cpu_quat_rotate(_ptr(q), _ptr(v), _ptr(out))
        return out

    def transform_point(self, pose, v):
        pose = np.ascontiguousarray(pose, dtype=POSE).reshape(1)
        v = np.asarray(v, dtype=np.float32)
        out = np.zeros(3, dtype=np.float32)
        self.lib.mcl3dl_cpu_transform_point(_ptr(pose), _ptr(v), _ptr(out))
        return out

    def filter_clip(self, pts, clip_near=0.5, clip_far=10.0, clip_z_min=-2.0, clip_z_max=2.0):
        pts = np.ascontiguousarray(pts, dtype=POINT)
        keep = np.zeros(len(pts), dtype=np.uint8)
        self.lib.mcl3dl_cpu_filter_clip(_ptr(pts), len(pts), clip_near, clip_far, clip_z_min, clip_z_max, _ptr(keep))
        return keep.astype(bool)

    def global_localization_points(self, num_points_default, num_points_global, num_particles, current):
        return int(self.lib.mcl3dl_cpu_global_localization_points(num_points_default, num_points_global, num_particles,
                                                                  current))

    def motion_predict(self, odom_prev, odom_current, time_diff, tc_lin, tc_ang, states):
        """MotionPredictionModelDifferentialDrive::setOdoms + predict on a MOTION_STATE array (returns a copy)."""
        a = np.ascontiguousarray(odom_prev, dtype=POSE).reshape(1)
        b = np.ascontiguousarray(odom_current, dtype=POSE).reshape(1)
        st = np.array(states, dtype=MOTION_STATE)
        self.lib.mcl3dl_cpu_motion_predict(_ptr(a), _ptr(b), C.c_float(time_diff), C.c_float(tc_lin), C.c_float(tc_ang),
                                           _ptr(st), len(st))
        return st

    def pf_resample_1d(self, probs, states, seed, sigma=0.0):
        probs = np.ascontiguousarray(probs, dtype=np.float32)
        states = np.ascontiguousarray(states, dtype=np.float32)
        out_s = np.zeros(len(probs), dtype=np.float32)
        out_p = np.zeros(len(probs), dtype=np.float32)
        self.lib.mcl3dl_cpu_pf_resample_1d(_ptr(probs), _ptr(states), len(probs), seed, sigma, _ptr(out_s), _ptr(out_p))
        return out_s, out_p

    def pf_resample_6dof(self, probs, states, seed, sigma_pos, sigma_rpy):
        probs = np.ascontiguousarray(probs, dtype=np.float32)
        states = np.ascontiguousarray(states, dtype=MOTION_STATE)
        sp = np.asarray(sigma_pos, dtype=np.float32)
        sr = np.asarray(sigma_rpy, dtype=np.float32)
        out = np.zeros(len(probs), dtype=MOTION_STATE)
        out_p = np.zeros(len(probs), dtype=np.float32)
        self.lib.mcl3dl_cpu_pf_resample_6dof(_ptr(probs), _ptr(states), len(probs), seed, _ptr(sp), _ptr(sr), _ptr(out),
                                             _ptr(out_p))
        return out, out_p

    def pf_estimate(self, probs, states, state_prev=None, bias_var_dist=1.0, bias_var_ang=1.0):
        """(mean_biased POSE[1], max_index, cov float32[6, 6]) = the node's pose estimate (oracle_api.h)."""
        probs = np.ascontiguousarray(probs, dtype=np.float32)
        states = np.ascontiguousarray(states, dtype=MOTION_STATE)
        prev = np.ascontiguousarray(state_prev, dtype=POSE).reshape(1) if state_prev is not None else None
        mean = np.zeros(1, dtype=POSE)
        best = C.c_uint32(0)
        cov = np.zeros(36, dtype=np.float32)
        rc = self.lib.mcl3dl_cpu_pf_estimate(_ptr(probs), _ptr(states), len(probs), _ptr(prev) if prev is not None else None,
                                             bias_var_dist, bias_var_ang, _ptr(mean), C.byref(best), _ptr(cov))
        assert rc == 0, rc
        return mean, int(best.value), cov.reshape(6, 6)

    def pf_update(self, prob, lik):
        prob = np.array(prob, dtype=np.float32)
        lik = np.ascontiguousarray(lik, dtype=np.float32)
        ent = C.c_float(0)
        kept = self.lib.mcl3dl_cpu_pf_update(_ptr(prob), _ptr(lik), len(prob), C.byref(ent))
        return prob, float(ent.value), bool(kept)


class CpuMap:
    def __init__(self, checker, map_pts, lik, beam, chunk_length, max_search_radius):
        self.c = checker
        self.map_pts = np.ascontiguousarray(map_pts, dtype=POINT)
        self.lik = lik
        self.beam = beam
        self.h = checker.lib.mcl3dl_cpu_create(_ptr(self.map_pts), len(self.map_pts),
                                               C.byref(lik) if lik is not None else None,
                                               C.byref(beam) if beam is not None else None,
                                               chunk_length, max_search_radius)
        if not self.h:
            raise RuntimeError("mcl3dl_cpu_create failed")

    def close(self):
        if self.h:
            self.c.lib.mcl3dl_cpu_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_tally(self, enable):
        self.c.lib.mcl3dl_cpu_set_tally(self.h, 1 if enable else 0)

    def measure(self, pose_arr, lik_pts, beam_pts, origins, n_threads=1):
        pose_arr = np.ascontiguousarray(pose_arr, dtype=POSE)
        lik_pts = np.ascontiguousarray(lik_pts if lik_pts is not None else np.zeros(0, POINT), dtype=POINT)
        beam_pts = np.ascontiguousarray(beam_pts if beam_pts is not None else np.zeros(0, POINT), dtype=POINT)
        origins = np.ascontiguousarray(origins if origins is not None else np.zeros((0, 3)), dtype=np.float32)
        origins = origins.reshape(-1, 3)
        out = np.zeros(len(pose_arr), dtype=RESULT)
        rc = self.c.lib.mcl3dl_cpu_measure(self.h, _ptr(pose_arr), len(pose_arr), _ptr(lik_pts), len(lik_pts),
                                           _ptr(beam_pts), len(beam_pts), _ptr(origins), len(origins),
                                           _ptr(out), n_threads)
        if rc != 0:
            raise RuntimeError("mcl3dl_cpu_measure rc=%d" % rc)
        return out

    def beam_status(self, pose_arr, beam_pts, origins):
        pose_arr = np.ascontiguousarray(pose_arr, dtype=POSE)
        beam_pts = np.ascontiguousarray(beam_pts, dtype=POINT)
        origins = np.ascontiguousarray(origins, dtype=np.float32).reshape(-1, 3)
        st = np.zeros((len(pose_arr), len(beam_pts)), dtype=np.uint8)
        rc = self.c.lib.mcl3dl_cpu_beam_status(self.h, _ptr(pose_arr), len(pose_arr), _ptr(beam_pts),
                                               len(beam_pts), _ptr(origins), len(origins), _ptr(st))
        if rc != 0:
            raise RuntimeError("mcl3dl_cpu_beam_status rc=%d" % rc)
        return st

    def beam_params(self):
        bp = BeamParams()
        self.c.lib.mcl3dl_cpu_beam_params(self.h, C.byref(bp))
        return bp

    def radius_search(self, q, radius):
        q = np.asarray(q, dtype=np.float32)
        d2 = C.c_float(0)
        i = self.c.lib.mcl3dl_cpu_radius_search(self.h, _ptr(q), radius, C.byref(d2))
        return i, float(d2.value)

"""ctypes mirror of include/liorf_b200.h.  Method names follow the reference's member functions
(src/mapOptmization.cpp, src/imageProjection.cpp, include/Scancontext.h) so the parity tests read like the
reference's call sequence."""
import ctypes as C

import numpy as np

from ._lib import load_library

MAX_ITERS = 64
P4 = np.dtype([("x", "<f4"), ("y", "<f4"), ("z", "<f4"), ("i", "<f4")])
PRAW = np.dtype([("x", "<f4"), ("y", "<f4"), ("z", "<f4"), ("i", "<f4"), ("ring", "<u2"), ("pad", "<u2"), ("time", "<f4")])


class Params(C.Structure):
    _fields_ = [("N_SCAN", C.c_int), ("downsampleRate", C.c_int), ("point_filter_num", C.c_int),
                ("lidarMinRange", C.c_float), ("lidarMaxRange", C.c_float),
                ("mappingSurfLeafSize", C.c_float), ("surroundingKeyframeMapLeafSize", C.c_float),
                ("surroundingKeyframeSearchRadius", C.c_float),
                ("grid_dim_x", C.c_int), ("grid_dim_y", C.c_int), ("grid_dim_z", C.c_int), ("device", C.c_int)]

    @staticmethod
    def default(**kw):
        p = Params()
        load_library().liorf_default_params(C.byref(p))
        for k, v in kw.items():
            if not hasattr(p, k):
                raise AttributeError(k)
            setattr(p, k, v)
        return p


class LMTrace(C.Structure):
    _fields_ = [("pose", (C.c_float * 6) * MAX_ITERS), ("nsel", C.c_int * MAX_ITERS), ("iters", C.c_int),
                ("converged", C.c_int), ("degenerate", C.c_int), ("ran", C.c_int)]

    def poses(self):
        return np.array([[self.pose[i][k] for k in range(6)] for i in range(self.iters)], np.float32).reshape(-1, 6)

    def nsels(self):
        return np.array([self.nsel[i] for i in range(self.iters)], np.int32)


class CloudInfoGuess(C.Structure):
    _fields_ = [("imuAvailable", C.c_int), ("odomAvailable", C.c_int), ("imuRollInit", C.c_float), ("imuPitchInit", C.c_float), ("imuYawInit", C.c_float),
                ("initialGuessX", C.c_float), ("initialGuessY", C.c_float), ("initialGuessZ", C.c_float), ("initialGuessRoll", C.c_float),
                ("initialGuessPitch", C.c_float), ("initialGuessYaw", C.c_float)]


class GuessState(C.Structure):
    _fields_ = [("lastImuTransformation", C.c_float * 12), ("lastImuPreTransformation", C.c_float * 12), ("lastImuPreTransAvailable", C.c_int),
                ("initialised", C.c_int)]


class FrameIn(C.Structure):
    _fields_ = [("pts", C.c_void_p), ("n", C.c_int), ("pts_on_device", C.c_int), ("time_scan_cur", C.c_double),
                ("imu_time", C.c_void_p), ("imu_rot_x", C.c_void_p), ("imu_rot_y", C.c_void_p), ("imu_rot_z", C.c_void_p),
                ("imu_pointer_cur", C.c_int), ("deskew_enabled", C.c_int), ("initial_guess", C.c_float * 6),
                ("surrounding_keyframe_density", C.c_float), ("adding_dist_threshold", C.c_float), ("adding_angle_threshold", C.c_float),
                ("rotation_tollerance", C.c_float), ("z_tollerance", C.c_float), ("max_iters", C.c_int), ("loop_every", C.c_int), ("frame_index", C.c_int),
                ("use_cloud_info", C.c_int), ("cloud_info", CloudInfoGuess), ("imu_type", C.c_int), ("use_imu_heading_initialization", C.c_int),
                ("imu_rpy_weight", C.c_float), ("next", C.c_void_p)]


class FrameOut(C.Structure):
    _fields_ = [("pose", C.c_float * 6), ("is_keyframe", C.c_int), ("keyframe_id", C.c_int), ("n_kept", C.c_int), ("n_ds", C.c_int), ("m_ds", C.c_int),
                ("iters", C.c_int), ("converged", C.c_int), ("degenerate", C.c_int), ("ran", C.c_int), ("loop_checked", C.c_int), ("loop_id", C.c_int),
                ("loop_yaw", C.c_float)]


class IcpResult(C.Structure):
    _fields_ = [("ran", C.c_int), ("converged", C.c_int), ("convergence_state", C.c_int), ("iterations", C.c_int), ("n_source", C.c_int), ("n_target", C.c_int),
                ("fitness", C.c_float), ("transform", C.c_float * 16), ("pose6", C.c_float * 6)]


def imuDeskewInfo(stamp, gyro_xyz, time_scan_cur, time_scan_end, check_gate=True, capacity=2000):
    """ImageProjection::imuDeskewInfo (src/imageProjection.cpp:350-409) on an array of queued IMU samples; host-only (no context, no GPU).
    Returns dict(available, imu_time, imu_rot (rows x 3), imu_pointer_cur, n_pop, rpy_index)."""
    lib = load_library()
    stamp = np.ascontiguousarray(stamp, np.float64); g = np.ascontiguousarray(gyro_xyz, np.float64).reshape(-1, 3)
    t = np.zeros(capacity); rx = np.zeros(capacity); ry = np.zeros(capacity); rz = np.zeros(capacity)
    ptr = C.c_int(-1); npop = C.c_int(0); rpy = C.c_int(-1)
    rc = lib.liorf_host_imu_deskew_info(_vp(stamp), _vp(g), C.c_int(len(stamp)), C.c_double(time_scan_cur), C.c_double(time_scan_end), C.c_int(int(check_gate)),
                                        _vp(t), _vp(rx), _vp(ry), _vp(rz), C.c_int(capacity), C.byref(ptr), C.byref(npop), C.byref(rpy))
    if rc < 0:
        raise LiorfError(f"liorf_host_imu_deskew_info failed with code {rc}")
    rows = ptr.value + 1
    return dict(available=bool(rc), imu_time=t[:rows].copy(), imu_rot=np.stack([rx[:rows], ry[:rows], rz[:rows]], 1), imu_pointer_cur=ptr.value, n_pop=npop.value,
                rpy_index=rpy.value)


def sc_tree_schedule(n_db_calls):
    """The stale-tree size each detectLoopClosureID call of a call history saw, starting from a fresh SCManager: n_db_calls[i] is the
    database size at call i.  A call with fewer than 31 entries returns early and does not advance the call counter (0 here); a call whose
    counter is a multiple of 10 rebuilds the tree over keys [0, n - 30) (include/Scancontext.cpp:263-281).  Feeds detectLoopClosureIDBatch."""
    n_db_calls = np.asarray(n_db_calls, np.int64).reshape(-1)
    out = np.zeros(len(n_db_calls), np.int32)
    counter, tree = 0, 0
    for i, n in enumerate(n_db_calls):
        if n < 31:
            continue
        if counter % 10 == 0:
            tree = int(n) - 30
        counter += 1
        out[i] = tree
    return out


class LiorfError(RuntimeError):
    pass


def _chk(rc, what):
    if rc < 0:
        raise LiorfError(f"{what} failed with code {rc}")
    return rc


def _vp(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def _p4(a):
    return np.ascontiguousarray(a, np.float32).reshape(-1, 4)


def _pose(p):
    return np.ascontiguousarray(p, np.float32).reshape(6).copy()


class Context:
    """One liorf_ctx (device memory + one CUDA stream).  Not thread-safe, like the reference's `mtx` discipline."""

    def __init__(self, params=None, **kw):
        self.lib = load_library()
        self.params = params if params is not None else Params.default(**kw)
        self.h = C.c_void_p()
        _chk(self.lib.liorf_create(C.byref(self.params), C.byref(self.h)), "liorf_create")

    def close(self):
        if getattr(self, "h", None) is not None and self.h:
            self.lib.liorf_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def reserve(self, n_scan_max, m_raw_max, n_keyframe_points_max=0, sc_entries_max=0):
        _chk(self.lib.liorf_reserve(self.h, C.c_int(n_scan_max), C.c_int(m_raw_max), C.c_int(n_keyframe_points_max), C.c_int(sc_entries_max)), "liorf_reserve")

    def sync(self):
        _chk(self.lib.liorf_sync(self.h), "liorf_sync")

    def stream(self):
        return self.lib.liorf_stream(self.h)

    # ---- ImageProjection ----
    def projectPointCloud(self, raw, time_scan_cur, imu_time=None, imu_rot=None, imu_pointer_cur=-1, deskew_enabled=True,
                          want_output=True, want_kept_index=False):
        raw = np.ascontiguousarray(raw, dtype=PRAW)
        n = len(raw)
        out = np.empty((max(n, 1), 4), np.float32) if want_output else None
        kept = np.empty(max(n, 1), np.int32) if want_kept_index else None
        n_out = C.c_int(0)
        self._keep = raw                                          # the H2D copy may still be in flight in the async form
        if deskew_enabled:
            it = np.ascontiguousarray(imu_time, np.float64)
            rot = np.ascontiguousarray(imu_rot, np.float64)
            rx, ry, rz = (np.ascontiguousarray(rot[:, k]) for k in range(3))
        else:
            it = rx = ry = rz = None
        _chk(self.lib.liorf_project_point_cloud(self.h, _vp(raw), C.c_int(n), C.c_double(time_scan_cur), _vp(it), _vp(rx), _vp(ry), _vp(rz),
                                                C.c_int(imu_pointer_cur), C.c_int(int(bool(deskew_enabled))), _vp(out),
                                                C.byref(n_out) if (want_output or want_kept_index) else None, _vp(kept)),
             "liorf_project_point_cloud")
        if not want_output and not want_kept_index:
            return None
        k = n_out.value
        res = [out[:k].copy() if want_output else None, k]
        if want_kept_index:
            res.append(kept[:k].copy())
        return tuple(res)

    def projectPointCloudDev(self, d_ptr, n, time_scan_cur, imu_time=None, imu_rot=None, imu_pointer_cur=-1, deskew_enabled=True):
        if deskew_enabled:
            it = np.ascontiguousarray(imu_time, np.float64)
            rot = np.ascontiguousarray(imu_rot, np.float64)
            rx, ry, rz = (np.ascontiguousarray(rot[:, k]) for k in range(3))
        else:
            it = rx = ry = rz = None
        _chk(self.lib.liorf_project_point_cloud_dev(self.h, C.c_void_p(d_ptr), C.c_int(n), C.c_double(time_scan_cur), _vp(it), _vp(rx), _vp(ry), _vp(rz),
                                                    C.c_int(imu_pointer_cur), C.c_int(int(bool(deskew_enabled)))), "liorf_project_point_cloud_dev")

    # ---- mapOptimization ----
    def setCurrentScan(self, scan):
        scan = _p4(scan)
        _chk(self.lib.liorf_set_current_scan(self.h, _vp(scan), C.c_int(len(scan))), "liorf_set_current_scan")

    def setCurrentScanStrided(self, data, n, point_step, offset_xyz=0, offset_intensity=16):
        """laserCloudSurfLast from a PointCloud2 data block (bytes / uint8 array): PCL's PointXYZI is 32 bytes per point, intensity at 16"""
        buf = np.ascontiguousarray(np.frombuffer(data, np.uint8) if not isinstance(data, np.ndarray) else data.view(np.uint8).reshape(-1))
        _chk(self.lib.liorf_set_current_scan_strided(self.h, _vp(buf), C.c_int(n), C.c_int(point_step), C.c_int(offset_xyz), C.c_int(offset_intensity), C.c_int(0)),
             "liorf_set_current_scan_strided")

    def setCurrentScanDev(self, d_ptr, n):
        _chk(self.lib.liorf_set_current_scan_dev(self.h, C.c_void_p(d_ptr), C.c_int(n)), "liorf_set_current_scan_dev")

    def downsampleCurrentScan(self, n_in=None, want_output=True, want_membership=False):
        """VoxelGrid(mappingSurfLeafSize) of the current scan.  n_in = capacity hint for the host output buffers."""
        if not want_output and not want_membership:
            _chk(self.lib.liorf_downsample_current_scan(self.h, None, None, None), "liorf_downsample_current_scan")
            return None
        cap = max(int(n_in if n_in is not None else 0), 1)
        out = np.empty((cap, 4), np.float32) if want_output else None
        mem = np.empty(cap, np.int32) if want_membership else None
        nds = C.c_int(0)
        _chk(self.lib.liorf_downsample_current_scan(self.h, _vp(out), C.byref(nds), _vp(mem)), "liorf_downsample_current_scan")
        res = [out[:nds.value].copy() if want_output else None, nds.value]
        if want_membership:
            res.append(mem[:cap].copy())
        return tuple(res)

    def voxelGrid(self, pts, leaf):
        pts = _p4(pts)
        n = len(pts)
        out = np.empty((max(n, 1), 4), np.float32); mem = np.empty(max(n, 1), np.int32); keys = np.empty(max(n, 1), np.int32)
        no = C.c_int(0)
        _chk(self.lib.liorf_voxel_grid(self.h, _vp(pts), C.c_int(n), C.c_float(leaf), _vp(out), C.byref(no), _vp(mem), _vp(keys)), "liorf_voxel_grid")
        return out[:no.value].copy(), mem[:n].copy(), keys[:no.value].copy()

    def addKeyframe(self, pose6, time=0.0):
        return _chk(self.lib.liorf_add_keyframe(self.h, _vp(_pose(pose6)), C.c_double(time)), "liorf_add_keyframe")

    def addKeyframeCloud(self, cloud, pose6, time=0.0):
        cloud = _p4(cloud)
        return _chk(self.lib.liorf_add_keyframe_cloud(self.h, _vp(cloud), C.c_int(len(cloud)), _vp(_pose(pose6)), C.c_double(time)), "liorf_add_keyframe_cloud")

    def updateKeyframePose(self, kid, pose6):
        _chk(self.lib.liorf_update_keyframe_pose(self.h, C.c_int(kid), _vp(_pose(pose6))), "liorf_update_keyframe_pose")

    def numKeyframes(self):
        return self.lib.liorf_num_keyframes(self.h)

    def extractSurroundingKeyFrames(self, ids, want_count=True):
        ids = np.ascontiguousarray(ids, np.int32)
        m = C.c_int(0)
        _chk(self.lib.liorf_extract_surrounding_keyframes(self.h, _vp(ids), C.c_int(len(ids)), C.byref(m) if want_count else None),
             "liorf_extract_surrounding_keyframes")
        return m.value if want_count else None

    def extractNearby(self, time_cur, density=2.0, cap=4096):
        ids = np.zeros(cap, np.int32); n = C.c_int(0)
        _chk(self.lib.liorf_extract_nearby(self.h, C.c_double(time_cur), C.c_float(density), _vp(ids), C.c_int(cap), C.byref(n)), "liorf_extract_nearby")
        return ids[:n.value].copy()

    def saveFrame(self, pose6, dist_thr=1.0, ang_thr=0.2):
        return bool(_chk(self.lib.liorf_save_frame(self.h, _vp(_pose(pose6)), C.c_float(dist_thr), C.c_float(ang_thr)), "liorf_save_frame"))

    def setLocalMap(self, map_ds):
        map_ds = _p4(map_ds)
        _chk(self.lib.liorf_set_local_map(self.h, _vp(map_ds), C.c_int(len(map_ds))), "liorf_set_local_map")

    def getLocalMap(self):
        m = C.c_int(0)
        _chk(self.lib.liorf_get_local_map(self.h, None, C.c_int(0), C.byref(m)), "liorf_get_local_map")
        out = np.empty((max(m.value, 1), 4), np.float32)
        _chk(self.lib.liorf_get_local_map(self.h, _vp(out), C.c_int(len(out)), C.byref(m)), "liorf_get_local_map")
        return out[:m.value].copy()

    def kdtreeSetInputCloud(self):
        """kdtreeSurfFromMap->setInputCloud (src/mapOptmization.cpp:1302): rebuild the voxel-hash grid over the resident local map (async)"""
        _chk(self.lib.liorf_kdtree_set_input_cloud(self.h), "liorf_kdtree_set_input_cloud")

    def getScanDS(self):
        n = C.c_int(0)
        _chk(self.lib.liorf_get_scan_ds(self.h, None, C.c_int(0), C.byref(n)), "liorf_get_scan_ds")
        out = np.empty((max(n.value, 1), 4), np.float32)
        _chk(self.lib.liorf_get_scan_ds(self.h, _vp(out), C.c_int(len(out)), C.byref(n)), "liorf_get_scan_ds")
        return out[:n.value].copy()

    def scan2MapOptimization(self, pose6, max_iters=30, force_all_iters=False, want_trace=True):
        pose = _pose(pose6)
        tr = LMTrace() if want_trace else None
        _chk(self.lib.liorf_scan2map_optimization(self.h, _vp(pose), C.c_int(max_iters), C.c_int(int(force_all_iters)),
                                                  C.byref(tr) if want_trace else None), "liorf_scan2map_optimization")
        return pose, tr

    def scan2MapOptimizationAsync(self, pose6=None, max_iters=30, force_all_iters=False):
        pose = _pose(pose6) if pose6 is not None else None
        _chk(self.lib.liorf_scan2map_optimization_async(self.h, _vp(pose), C.c_int(max_iters), C.c_int(int(force_all_iters))),
             "liorf_scan2map_optimization_async")

    def getPose(self, want_trace=False):
        pose = np.zeros(6, np.float32)
        tr = LMTrace() if want_trace else None
        _chk(self.lib.liorf_get_pose(self.h, _vp(pose), C.byref(tr) if want_trace else None), "liorf_get_pose")
        return (pose, tr) if want_trace else pose

    def surfOptimization(self, pose6, n_ds):
        n = max(int(n_ds), 1)
        coeff = np.zeros((n, 4), np.float32); flag = np.zeros(n, np.uint8); idx = np.full((n, 5), -1, np.int32)
        d2 = np.zeros((n, 5), np.float32); plane = np.zeros((n, 4), np.float32); sel = np.zeros((n, 4), np.float32)
        _chk(self.lib.liorf_surf_optimization(self.h, _vp(_pose(pose6)), _vp(coeff), _vp(flag), _vp(idx), _vp(d2), _vp(plane), _vp(sel)),
             "liorf_surf_optimization")
        k = int(n_ds)
        return dict(coeff=coeff[:k], flag=flag[:k], idx=idx[:k], d2=d2[:k], plane=plane[:k], sel=sel[:k])

    def combineOptimizationCoeffs(self, n_ds):
        n = max(int(n_ds), 1)
        ori = np.zeros((n, 4), np.float32); coeff = np.zeros((n, 4), np.float32); ns = C.c_int(0)
        _chk(self.lib.liorf_combine_optimization_coeffs(self.h, _vp(ori), _vp(coeff), C.byref(ns)), "liorf_combine_optimization_coeffs")
        return ori[:ns.value].copy(), coeff[:ns.value].copy()

    def LMOptimization(self, iter_count, pose6):
        pose = _pose(pose6)
        AtA = np.zeros(36, np.float32); AtB = np.zeros(6, np.float32); X = np.zeros(6, np.float32); ns = C.c_int(0)
        rc = _chk(self.lib.liorf_lm_optimization(self.h, C.c_int(iter_count), _vp(pose), _vp(AtA), _vp(AtB), _vp(X), C.byref(ns)), "liorf_lm_optimization")
        return dict(converged=bool(rc), tf=pose, AtA=AtA.reshape(6, 6), AtB=AtB, X=X, nsel=ns.value)

    def getLMState(self):
        deg = C.c_int(0); P = np.zeros(36, np.float32)
        _chk(self.lib.liorf_get_lm_state(self.h, C.byref(deg), _vp(P)), "liorf_get_lm_state")
        return bool(deg.value), P.reshape(6, 6)

    def setLMState(self, deg, matP):
        P = np.ascontiguousarray(matP, np.float32).reshape(36)
        _chk(self.lib.liorf_set_lm_state(self.h, C.c_int(int(deg)), _vp(P)), "liorf_set_lm_state")

    @staticmethod
    def frameIn(pts_ptr, n, on_device, time_scan_cur, imu_time, imu_rot_xyz, imu_pointer_cur, deskew_enabled, initial_guess=None,
                density=2.0, dist_thr=1.0, ang_thr=0.2, rot_tol=1000.0, z_tol=1000.0, max_iters=30, loop_every=0, frame_index=0,
                cloud_info=None, imu_type=0, use_imu_heading=True, imu_rpy_weight=0.01):
        """a liorf_frame_in.  imu_rot_xyz: three contiguous float64 arrays (kept alive by the returned object)."""
        fi = FrameIn()
        fi.pts = pts_ptr; fi.n = n; fi.pts_on_device = int(on_device); fi.time_scan_cur = time_scan_cur
        fi.imu_time = imu_time.ctypes.data; fi.imu_rot_x = imu_rot_xyz[0].ctypes.data; fi.imu_rot_y = imu_rot_xyz[1].ctypes.data; fi.imu_rot_z = imu_rot_xyz[2].ctypes.data
        fi._keep = (imu_time, imu_rot_xyz)
        fi.imu_pointer_cur = imu_pointer_cur; fi.deskew_enabled = int(deskew_enabled)
        if cloud_info is not None:                              # initial guess by updateInitialGuess from these cloud_info fields
            fi.use_cloud_info = 1; fi.cloud_info = cloud_info; fi.imu_type = imu_type; fi.use_imu_heading_initialization = int(use_imu_heading)
            fi.imu_rpy_weight = imu_rpy_weight
        elif initial_guess is not None:
            for k in range(6):
                fi.initial_guess[k] = float(initial_guess[k])
        fi.surrounding_keyframe_density = density; fi.adding_dist_threshold = dist_thr; fi.adding_angle_threshold = ang_thr
        fi.rotation_tollerance = rot_tol; fi.z_tollerance = z_tol; fi.max_iters = max_iters; fi.loop_every = loop_every; fi.frame_index = frame_index
        return fi

    def processFrame(self, pts_ptr, n, on_device, time_scan_cur, imu_time, imu_rot_xyz, imu_pointer_cur, deskew_enabled, initial_guess,
                     density=2.0, dist_thr=1.0, ang_thr=0.2, rot_tol=1000.0, z_tol=1000.0, max_iters=30, loop_every=0, frame_index=0,
                     cloud_info=None, imu_type=0, use_imu_heading=True, imu_rpy_weight=0.01, next_frame=None):
        """one frame through cloudHandler + laserCloudInfoHandler (liorf_process_frame).  imu_rot_xyz: three contiguous float64 arrays.
        next_frame: a frameIn(...) of the FOLLOWING frame — its deskew + downsample overlap this frame's solve (liorf_frame_in.next)."""
        fi = self.frameIn(pts_ptr, n, on_device, time_scan_cur, imu_time, imu_rot_xyz, imu_pointer_cur, deskew_enabled, initial_guess, density, dist_thr,
                          ang_thr, rot_tol, z_tol, max_iters, loop_every, frame_index, cloud_info, imu_type, use_imu_heading, imu_rpy_weight)
        if next_frame is not None:
            fi.next = C.addressof(next_frame)
            self._next_keep = next_frame                        # stays referenced until the call that consumes it
        fo = FrameOut()
        _chk(self.lib.liorf_process_frame(self.h, C.byref(fi), C.byref(fo)), "liorf_process_frame")
        return fo

    def processFrameIn(self, fi, guess=None, next_frame=None, fo=None):
        """liorf_process_frame on a prepared frameIn(...) (inputs staged ahead of time: nothing is rebuilt per frame)."""
        if guess is not None:
            g = fi.initial_guess
            g[0], g[1], g[2], g[3], g[4], g[5] = guess
        fi.next = C.addressof(next_frame) if next_frame is not None else None
        self._next_keep = next_frame
        if fo is None:
            fo = FrameOut()
        _chk(self.lib.liorf_process_frame(self.h, C.byref(fi), C.byref(fo)), "liorf_process_frame")
        return fo

    def cloudHandlerAsync(self, frame_in):
        """primes the pipeline: cloudHandler + downsample of a frame a later processFrame call (same frame_index / pts / n) consumes"""
        self._next_keep = frame_in
        _chk(self.lib.liorf_cloud_handler_async(self.h, C.byref(frame_in)), "liorf_cloud_handler_async")

    def debugQrSolve6(self, A, b):
        """cv::solve(DECOMP_QR) on the device for n systems (the routine the solver uses)"""
        A = np.ascontiguousarray(A, np.float32).reshape(-1, 36); b = np.ascontiguousarray(b, np.float32).reshape(-1, 6)
        x = np.zeros_like(b)
        _chk(self.lib.liorf_debug_qr_solve6(self.h, _vp(A), _vp(b), C.c_int(len(A)), _vp(x)), "liorf_debug_qr_solve6")
        return x

    def solverGlobalState(self, on=True):
        _chk(self.lib.liorf_debug_s2m_global_state(self.h, C.c_int(int(on))), "liorf_debug_s2m_global_state")

    def disableSolverCache(self, on=True):
        _chk(self.lib.liorf_debug_s2m_disable_cache(self.h, C.c_int(int(on))), "liorf_debug_s2m_disable_cache")

    def solverGrid(self, ctas=0):
        """run the solver on `ctas` CTAs (ctas - 1 workers + the reducer) in every launch; 0 = the defaults"""
        _chk(self.lib.liorf_debug_s2m_grid(self.h, C.c_int(int(ctas))), "liorf_debug_s2m_grid")

    def forceFusedVoxelGrid(self, on=True):
        _chk(self.lib.liorf_debug_force_fused_voxelgrid(self.h, C.c_int(int(on))), "liorf_debug_force_fused_voxelgrid")

    def forceLargeVoxelGrid(self, on=True):
        _chk(self.lib.liorf_debug_force_large_voxelgrid(self.h, C.c_int(int(on))), "liorf_debug_force_large_voxelgrid")

    def debugVoxelGridGrid(self, ctas=0):
        """run voxelGrid's one-kernel cooperative path on `ctas` CTAs (0 = all SMs); widths the device cannot hold co-resident raise"""
        _chk(self.lib.liorf_debug_voxelgrid_grid(self.h, C.c_int(int(ctas))), "liorf_debug_voxelgrid_grid")

    # ---- measurement helpers ----
    def enableTiming(self, on=True, sections=None):
        """sections: iterable of section names to time (None = all)"""
        if sections is None:
            _chk(self.lib.liorf_enable_timing(self.h, C.c_int(int(on))), "liorf_enable_timing")
        else:
            names = ["deskew", "downsample", "map_build", "grid_build", "scan2map", "sc_make", "sc_search", "sc_gemm"]
            mask = sum(1 << names.index(n) for n in sections) if on else 0
            _chk(self.lib.liorf_enable_timing_mask(self.h, C.c_uint(mask)), "liorf_enable_timing_mask")

    def getTiming(self):
        ms = (C.c_double * 8)(); calls = (C.c_longlong * 8)()
        _chk(self.lib.liorf_get_timing(self.h, ms, calls), "liorf_get_timing")
        names = ["deskew", "downsample", "map_build", "grid_build", "scan2map", "sc_make", "sc_search", "sc_gemm"]
        return {n: (ms[i], calls[i]) for i, n in enumerate(names) if n != "_"}

    def launchCount(self):
        self.lib.liorf_get_launch_count.restype = C.c_longlong
        return int(self.lib.liorf_get_launch_count(self.h))

    def lastCounts(self):
        a, b, c_, d = C.c_int(), C.c_int(), C.c_int(), C.c_int()
        _chk(self.lib.liorf_get_last_counts(self.h, C.byref(a), C.byref(b), C.byref(c_), C.byref(d)), "liorf_get_last_counts")
        return dict(n_scan=a.value, n_ds=b.value, m_ds=c_.value, iters=d.value)

    def getKeyframe(self, kid):
        n = C.c_int(0); pose = np.zeros(6, np.float32); t = C.c_double(0)
        _chk(self.lib.liorf_get_keyframe(self.h, C.c_int(kid), None, C.c_int(0), C.byref(n), _vp(pose), C.byref(t)), "liorf_get_keyframe")
        out = np.empty((max(n.value, 1), 4), np.float32)
        _chk(self.lib.liorf_get_keyframe(self.h, C.c_int(kid), _vp(out), C.c_int(len(out)), C.byref(n), _vp(pose), C.byref(t)), "liorf_get_keyframe")
        return out[:n.value].copy(), pose, t.value

    # ---- SCManager ----
    def makeAndSaveScancontextAndKeys(self, cloud=None):
        if cloud is None:
            _chk(self.lib.liorf_sc_make_and_save(self.h, None, C.c_int(0)), "liorf_sc_make_and_save")
        else:
            cloud = _p4(cloud)
            _chk(self.lib.liorf_sc_make_and_save(self.h, _vp(cloud), C.c_int(len(cloud))), "liorf_sc_make_and_save")

    def scAddDescriptors(self, descs):
        descs = np.ascontiguousarray(descs, np.float64).reshape(-1, 1200)
        _chk(self.lib.liorf_sc_add_descriptors(self.h, _vp(descs), C.c_int(len(descs))), "liorf_sc_add_descriptors")

    def scSize(self):
        return self.lib.liorf_sc_size(self.h)

    def scBorrowDatabase(self, owner):
        """search the ScanContext database of another context on the same device without copying it (read-only)"""
        _chk(self.lib.liorf_sc_borrow_database(self.h, owner.h), "liorf_sc_borrow_database")

    def scGet(self, i):
        d = np.zeros(1200, np.float64); k = np.zeros(20, np.float32); sk = np.zeros(60, np.float64)
        _chk(self.lib.liorf_sc_get(self.h, C.c_int(i), _vp(d), _vp(k), _vp(sk)), "liorf_sc_get")
        return d.reshape(20, 60), k, sk

    def detectLoopClosureID(self):
        lid = C.c_int(-1); yaw = C.c_float(0); md = C.c_double(0); cand = np.zeros(3, np.int32)
        _chk(self.lib.liorf_sc_detect_loop_closure_id(self.h, C.byref(lid), C.byref(yaw), C.byref(md), _vp(cand)), "liorf_sc_detect_loop_closure_id")
        return lid.value, yaw.value, md.value, cand

    def detectLoopClosureIDBatch(self, n_db, n_tree):
        """detectLoopClosureID for many calls at once (liorf_sc_detect_loop_closure_id_batch): entry q is the tuple detectLoopClosureID()
        returns when the database held its first n_db[q] entries and the stale tree covered keys [0, n_tree[q]) (sc_tree_schedule gives the
        n_tree of a call history).  Read-only: the detector state of this context is left as it was.
        Returns (loop_id int32[Q], yaw float32[Q], min_dist float64[Q], cand3 int32[Q, 3]); min_dist / cand3 are 0 for early-out queries."""
        n_db = np.ascontiguousarray(n_db, np.int32).reshape(-1)
        n_tree = np.ascontiguousarray(n_tree, np.int32).reshape(-1)
        if n_db.shape != n_tree.shape:
            raise ValueError("n_db and n_tree must have the same length")
        Q = len(n_db)
        lid = np.full(Q, -1, np.int32); yaw = np.zeros(Q, np.float32); md = np.zeros(Q, np.float64); cand = np.zeros((Q, 3), np.int32)
        _chk(self.lib.liorf_sc_detect_loop_closure_id_batch(self.h, _vp(n_db), _vp(n_tree), C.c_int(Q), _vp(lid), _vp(yaw), _vp(md), _vp(cand)),
             "liorf_sc_detect_loop_closure_id_batch")
        return lid, yaw, md, cand

    def loopClosureICP(self, loop_key_cur, loop_key_pre, history_search_num=25, loop_index=0, icp_leaf=0.5, max_corr_dist=20.0, max_iters=100):
        """the ICP of performSCLoopClosure (src/mapOptmization.cpp:624-730) between two stored keyframes"""
        r = IcpResult()
        _chk(self.lib.liorf_loop_closure_icp(self.h, C.c_int(loop_key_cur), C.c_int(loop_key_pre), C.c_int(history_search_num), C.c_int(loop_index),
                                             C.c_float(icp_leaf), C.c_float(max_corr_dist), C.c_int(max_iters), C.byref(r)), "liorf_loop_closure_icp")
        return r

    def loopClosureICPBatch(self, cur, pre, loop_index, history_search_num=25, icp_leaf=0.5, max_corr_dist=20.0, max_iters=100, as_arrays=False):
        """loopClosureICP for many pairs in one call (liorf_loop_closure_icp_batch): pair p is loopClosureICP(cur[p], pre[p], history_search_num,
        loop_index[p], ...) bit for bit.  loop_index: one value per pair, or a scalar for all.  Returns a ctypes array of IcpResult, or with
        as_arrays=True a dict of numpy arrays with the same field names (transform as (n, 4, 4), pose6 as (n, 6))."""
        cur = np.ascontiguousarray(cur, np.int32).reshape(-1)
        pre = np.ascontiguousarray(pre, np.int32).reshape(-1)
        li = np.ascontiguousarray(np.broadcast_to(np.asarray(loop_index, np.int32), cur.shape), np.int32)
        if pre.shape != cur.shape:
            raise ValueError("cur and pre must have the same length")
        n = len(cur)
        out = (IcpResult * max(n, 1))()
        _chk(self.lib.liorf_loop_closure_icp_batch(self.h, _vp(cur), _vp(pre), _vp(li), C.c_int(n), C.c_int(history_search_num), C.c_float(icp_leaf),
                                                   C.c_float(max_corr_dist), C.c_int(max_iters), out), "liorf_loop_closure_icp_batch")
        res = (IcpResult * n).from_buffer(out) if n else (IcpResult * 0)()
        if not as_arrays:
            return res
        d = {}
        for f, t in IcpResult._fields_:
            dt = np.int32 if t is C.c_int else np.float32
            v = np.array([np.array(getattr(r, f), dt) for r in res], dt)
            d[f] = v.reshape(n, 4, 4) if f == "transform" else v.reshape(n, 6) if f == "pose6" else v.reshape(n)
        return d

    def debugIcpBatchWave(self, max_pairs):
        """tests: at most max_pairs pairs per internal wave of loopClosureICPBatch (0 = the memory-bounded default)"""
        _chk(self.lib.liorf_debug_icp_batch_wave(self.h, C.c_int(max_pairs)), "liorf_debug_icp_batch_wave")

    def icpClouds(self, n_source, n_target):
        s = np.empty((max(n_source, 1), 4), np.float32); t = np.empty((max(n_target, 1), 4), np.float32)
        _chk(self.lib.liorf_icp_get_clouds(self.h, _vp(s), C.c_int(n_source), _vp(t), C.c_int(n_target)), "liorf_icp_get_clouds")
        return s[:n_source].copy(), t[:n_target].copy()

    def buildGlobalMap(self, search_radius=1000.0, pose_density=10.0, leaf=1.0):
        """publishGlobalMap (src/mapOptmization.cpp:453-502); search_radius <= 0 and leaf <= 0 give saveMapService's map"""
        n = C.c_int(0)
        _chk(self.lib.liorf_build_global_map(self.h, C.c_float(search_radius), C.c_float(pose_density), C.c_float(leaf), None, C.c_int(0), C.byref(n)),
             "liorf_build_global_map")
        out = np.empty((max(n.value, 1), 4), np.float32)
        _chk(self.lib.liorf_build_global_map(self.h, C.c_float(search_radius), C.c_float(pose_density), C.c_float(leaf), _vp(out), C.c_int(len(out)), C.byref(n)),
             "liorf_build_global_map")
        return out[:n.value].copy()

    def scSetSearchPath(self, mode):
        """ring-key search implementation: 0 auto, 1 CUDA-core brute force, 2 tcgen05 coarse filter + exact re-rank"""
        _chk(self.lib.liorf_sc_set_search_path(self.h, C.c_int(int(mode))), "liorf_sc_set_search_path")

    def scTensorStats(self):
        n = C.c_longlong(0); o = C.c_int(0)
        _chk(self.lib.liorf_sc_tensor_stats(self.h, C.byref(n), C.byref(o)), "liorf_sc_tensor_stats")
        return dict(candidates=n.value, overflow=o.value)

    def scTensorDump(self, qkeys):
        """test hook: raw tensor-core distances d~[Q, K] of host ring keys against the database, and the image centre"""
        qkeys = np.ascontiguousarray(qkeys, np.float32).reshape(-1, 20)
        Q, K = len(qkeys), self.scSize()
        ldmax = (K + 127) // 128 * 128
        out = np.empty((Q, ldmax), np.float32); ld = C.c_int(0); center = np.zeros(20, np.float32)
        _chk(self.lib.liorf_sc_tensor_dump(self.h, _vp(qkeys), C.c_int(Q), _vp(out), C.c_longlong(out.size), C.byref(ld), _vp(center)), "liorf_sc_tensor_dump")
        assert ld.value == ldmax
        return out[:, :K], center

    def scQueryBatch(self, qdescs):
        qdescs = np.ascontiguousarray(qdescs, np.float64).reshape(-1, 1200)
        Q = len(qdescs)
        loop = np.zeros(Q, np.int32); shift = np.zeros(Q, np.int32); dist = np.zeros(Q, np.float64); cand = np.zeros((Q, 3), np.int32)
        _chk(self.lib.liorf_sc_query_batch(self.h, _vp(qdescs), C.c_int(Q), _vp(loop), _vp(shift), _vp(dist), _vp(cand)), "liorf_sc_query_batch")
        return loop, shift, dist, cand

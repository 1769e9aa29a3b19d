"""ctypes binding of libb200reg.so -- the C ABI of include/b200reg.h.

The product path: every call below lands in hand-written sm_100a kernels.  There is no CPU
fallback; if the library or a GPU is missing these functions raise.
"""
import ctypes as C
import os

import numpy as np

from .build import LIB, build_native

_lib = None


class GicpParams(C.Structure):
    _fields_ = [("k_correspondences", C.c_int32), ("max_iterations", C.c_int32), ("max_corr_dist", C.c_double),
                ("transformation_eps", C.c_double), ("rotation_eps", C.c_double), ("lm_max_iterations", C.c_int32),
                ("regularization", C.c_int32), ("lm_init_lambda_factor", C.c_double), ("icp_score_thr", C.c_double)]


class Result(C.Structure):
    _fields_ = [("T", C.c_double * 16), ("Tf", C.c_float * 16), ("pose_between", C.c_double * 16), ("final_hessian", C.c_double * 36),
                ("fitness", C.c_double),
                ("converged", C.c_int32),
                ("valid", C.c_int32), ("iterations", C.c_int32), ("n_linearize", C.c_int32), ("n_error", C.c_int32),
                ("lm_failed", C.c_int32), ("status", C.c_int32), ("tag", C.c_int32)]

    def as_dict(self):
        return dict(T=np.array(self.T).reshape(4, 4), Tf=np.array(self.Tf, np.float32).reshape(4, 4),
                    pose_between=np.array(self.pose_between).reshape(4, 4),
                    final_hessian=np.array(self.final_hessian).reshape(6, 6), fitness=self.fitness, converged=bool(self.converged), valid=bool(self.valid),
                    iterations=self.iterations, n_linearize=self.n_linearize, n_error=self.n_error,
                    lm_failed=bool(self.lm_failed), status=self.status)


class QuatroParams(C.Structure):
    _fields_ = [("fpfh_normal_radius", C.c_double), ("fpfh_radius", C.c_double), ("noise_bound", C.c_double),
                ("rot_gnc_factor", C.c_double), ("rot_cost_thr", C.c_double), ("rot_max_iter", C.c_int32),
                ("max_corres", C.c_int32), ("distance_threshold", C.c_double), ("tuple_scale", C.c_double),
                ("seed", C.c_uint64), ("estimate_scale", C.c_int32), ("use_optimized_matching", C.c_int32)]


class QuatroInfo(C.Structure):
    _fields_ = [("T", C.c_double * 16), ("valid", C.c_int32), ("n_mutual", C.c_int32), ("n_corr", C.c_int32),
                ("clique_size", C.c_int32), ("gnc_iterations", C.c_int32), ("reserved", C.c_int32)]

    def as_dict(self):
        return dict(T=np.array(self.T).reshape(4, 4), valid=bool(self.valid), n_mutual=self.n_mutual,
                    n_corr=self.n_corr, clique_size=self.clique_size, gnc_iterations=self.gnc_iterations)


class LoopConfig(C.Structure):
    _fields_ = [("enable_quatro", C.c_int32), ("enable_submap_matching", C.c_int32), ("num_submap_keyframes", C.c_int32),
                ("reserved", C.c_int32), ("voxel_res", C.c_double), ("loop_detection_radius", C.c_double),
                ("loop_detection_timediff_threshold", C.c_double), ("gicp", GicpParams), ("quatro", QuatroParams)]


def default_loop_config():
    cfg = LoopConfig()
    lib().b200reg_default_loop_config(C.byref(cfg))
    return cfg


MAXC = 512       # B200REG_CORR_CAPACITY
ADV_MAXC = 8192  # B200REG_ADV_CORR_CAPACITY

EXPORTS = [
    "b200reg_default_gicp_params", "b200reg_last_error", "b200reg_version", "b200reg_ctx_create",
    "b200reg_ctx_destroy", "b200reg_ctx_set_stream", "b200reg_ctx_synchronize", "b200reg_ctx_launch_count",
    "b200reg_clouds_create", "b200reg_cloud_destroy", "b200reg_cloud_size", "b200reg_clouds_covariances", "b200reg_clouds_covariances_ex",
    "b200reg_gicp_align", "b200reg_icp_alignment", "b200reg_transform_cloud", "b200reg_knn",
    "b200reg_get_covariances", "b200reg_linearize", "b200reg_ctx_set_profiling", "b200reg_ctx_reset_profile",
    "b200reg_ctx_get_profile", "b200reg_default_quatro_params", "b200reg_clouds_fpfh", "b200reg_get_fpfh",
    "b200reg_quatro_align", "b200reg_loop_closure", "b200reg_default_loop_config", "b200reg_keyframes_create",
    "b200reg_keyframes_destroy", "b200reg_keyframes_reserve", "b200reg_keyframes_add", "b200reg_keyframes_set_pose", "b200reg_keyframes_size",
    "b200reg_knn_bruteforce", "b200reg_fetch_closest_keyframes", "b200reg_assemble_clouds", "b200reg_cloud_points", "b200reg_perform_loop_closure",
    "b200reg_loop_factor_from_poses", "b200reg_loop_factors", "b200reg_compute_error", "b200reg_assemble_clouds_at",
    "b200reg_struct_size", "b200reg_set_last_error", "b200reg_set_covariances",
    "b200reg_keyframes_add_world", "b200reg_keyframes_get", "b200reg_keyframes_cloud_size",
    "b200reg_batch_create", "b200reg_batch_destroy", "b200reg_batch_submit_icp", "b200reg_batch_submit_loop_closure",
    "b200reg_batch_wait", "b200reg_batch_wait_all", "b200reg_batch_launch_count", "b200reg_batch_depth",
    "b200reg_comm_unique_id", "b200reg_comm_init", "b200reg_comm_destroy", "b200reg_comm_rank", "b200reg_comm_world",
    "b200reg_allgather_results",
    "b200reg_map_build", "b200reg_map_size", "b200reg_map_voxelized", "b200reg_map_get", "b200reg_map_destroy",
]


def _point_at_bundled_nccl():
    """b200reg_comm_* load NCCL at run time.  In a Python process the pip-bundled libnccl (site-packages/nvidia/nccl/lib) is
    the one torch was built against; if the system's older libnccl.so.2 got loaded first under the same soname, a later
    `import torch` would fail on missing symbols.  So unless the caller chose a library, point the C side at the bundled one."""
    if os.environ.get("B200REG_NCCL_LIB"):
        return
    import sys
    for base in sys.path:
        cand = os.path.join(base, "nvidia", "nccl", "lib", "libnccl.so.2")
        if os.path.exists(cand):
            os.environ["B200REG_NCCL_LIB"] = cand
            return


def lib():
    global _lib
    if _lib is None:
        _point_at_bundled_nccl()
        path = LIB if os.path.exists(LIB) and not os.path.exists("/usr/local/cuda/bin/nvcc") else build_native()
        _lib = C.CDLL(path)
        _lib.b200reg_last_error.restype = C.c_char_p
        _lib.b200reg_version.restype = C.c_char_p
        _lib.b200reg_ctx_launch_count.restype = C.c_int64
        _lib.b200reg_cloud_size.restype = C.c_size_t
        _lib.b200reg_struct_size.restype = C.c_size_t
        _lib.b200reg_keyframes_cloud_size.restype = C.c_size_t
        _lib.b200reg_batch_submit_icp.restype = C.c_int64
        _lib.b200reg_batch_submit_loop_closure.restype = C.c_int64
        _lib.b200reg_batch_launch_count.restype = C.c_int64
        _lib.b200reg_map_size.restype = C.c_size_t
    return _lib


class LoopFactor(C.Structure):
    """b200reg_loop_factor: the BetweenFactor the reference adds for an accepted loop (fast_lio_sam_qn.cpp:220-237)."""
    _fields_ = [("from_idx", C.c_int32), ("to_idx", C.c_int32), ("valid", C.c_int32), ("reserved", C.c_int32),
                ("measurement", C.c_double * 16), ("variances", C.c_double * 6)]

    def as_dict(self):
        return dict(from_idx=self.from_idx, to_idx=self.to_idx, valid=bool(self.valid),
                    measurement=np.array(self.measurement).reshape(4, 4), variances=np.array(self.variances))


class B200RegError(RuntimeError):
    pass


def _check(rc):
    if rc != 0:
        raise B200RegError("b200reg error %d: %s" % (rc, lib().b200reg_last_error().decode()))


def loop_factor_from_poses(T_between, pose_latest, pose_closest, score, valid=True, from_idx=0, to_idx=0):
    """Host arithmetic only (no context / GPU needed)."""
    f = LoopFactor()
    arr = [np.ascontiguousarray(m, np.float64) for m in (T_between, pose_latest, pose_closest)]
    _check(lib().b200reg_loop_factor_from_poses(arr[0].ctypes.data_as(C.c_void_p), arr[1].ctypes.data_as(C.c_void_p),
                                                arr[2].ctypes.data_as(C.c_void_p), C.c_double(score), int(bool(valid)),
                                                int(from_idx), int(to_idx), C.byref(f)))
    return f.as_dict()


def default_params():
    p = GicpParams()
    lib().b200reg_default_gicp_params(C.byref(p))
    return p


def default_quatro_params():
    p = QuatroParams()
    lib().b200reg_default_quatro_params(C.byref(p))
    return p


def _pts(a):
    a = np.ascontiguousarray(a, dtype=np.float32)
    assert a.ndim == 2 and a.shape[1] >= 3
    return a


class Cloud:
    def __init__(self, ctx, handle, n):
        self.ctx, self.h, self.n = ctx, handle, n

    def destroy(self):
        if self.h:
            lib().b200reg_cloud_destroy(self.ctx.h, self.h)
            self.h = None


class Context:
    """One context per GPU rank / host thread (wraps b200reg_ctx)."""

    def __init__(self, device=0):
        self.h = C.c_void_p()
        _check(lib().b200reg_ctx_create(int(device), C.byref(self.h)))

    def close(self):
        if self.h:
            lib().b200reg_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_stream(self, cuda_stream_ptr):
        _check(lib().b200reg_ctx_set_stream(self.h, C.c_void_p(cuda_stream_ptr)))

    def synchronize(self):
        _check(lib().b200reg_ctx_synchronize(self.h))

    @property
    def launch_count(self):
        return int(lib().b200reg_ctx_launch_count(self.h))

    def set_profiling(self, enable):
        _check(lib().b200reg_ctx_set_profiling(self.h, int(bool(enable))))

    def reset_profile(self):
        _check(lib().b200reg_ctx_reset_profile(self.h))

    def get_profile(self):
        """{family: dict(ms, algo_bytes, launches)} from CUDA events on the launching stream."""
        out = {}
        for f in range(9):
            name, ms, by, ln = C.c_char_p(), C.c_double(), C.c_double(), C.c_int64()
            _check(lib().b200reg_ctx_get_profile(self.h, f, C.byref(name), C.byref(ms), C.byref(by), C.byref(ln)))
            out[name.value.decode()] = dict(ms=ms.value, algo_bytes=by.value, launches=ln.value)
        return out

    # -- the path's one collective: all-gather of the result records over NCCL (SURVEY §8e) --------
    def comm_init(self, unique_id, rank, world):
        """unique_id: the 128 bytes rank 0 got from comm_unique_id(), shipped to every rank by the caller."""
        buf = (C.c_ubyte * 128).from_buffer_copy(bytes(unique_id))
        _check(lib().b200reg_comm_init(self.h, buf, int(rank), int(world)))

    def comm_destroy(self):
        _check(lib().b200reg_comm_destroy(self.h))

    @property
    def comm_world(self):
        return int(lib().b200reg_comm_world(self.h))

    def allgather_results(self, local):
        """local: (Result * n) ctypes array of this rank -> (Result * (world * n)) with every rank's records, rank order."""
        n = len(local)
        out = (Result * (self.comm_world * n))()
        _check(lib().b200reg_allgather_results(self.h, local, n, out))
        return out

    # -- clouds ------------------------------------------------------------------------
    def create_clouds(self, arrays):
        """arrays: list of host float32 (n, >=3) arrays (strided records) -> list[Cloud]."""
        arrs = [_pts(a) for a in arrays]
        stride = arrs[0].shape[1] * 4
        assert all(a.shape[1] * 4 == stride for a in arrs)
        cnt = len(arrs)
        ptrs = (C.c_void_p * cnt)(*[a.ctypes.data for a in arrs])
        ns = (C.c_size_t * cnt)(*[len(a) for a in arrs])
        outs = (C.c_void_p * cnt)()
        _check(lib().b200reg_clouds_create(self.h, cnt, ptrs, ns, C.c_size_t(stride), 0, outs))
        return [Cloud(self, C.c_void_p(outs[i]), len(arrs[i])) for i in range(cnt)]

    def create_clouds_device(self, dev_ptrs, ns, stride_bytes):
        cnt = len(dev_ptrs)
        ptrs = (C.c_void_p * cnt)(*dev_ptrs)
        nsa = (C.c_size_t * cnt)(*ns)
        outs = (C.c_void_p * cnt)()
        _check(lib().b200reg_clouds_create(self.h, cnt, ptrs, nsa, C.c_size_t(stride_bytes), 1, outs))
        return [Cloud(self, C.c_void_p(outs[i]), ns[i]) for i in range(cnt)]

    def covariances(self, clouds, k=15, method=3):
        arr = (C.c_void_p * len(clouds))(*[c.h for c in clouds])
        _check(lib().b200reg_clouds_covariances_ex(self.h, len(clouds), arr, int(k), int(method)))

    def set_covariances(self, cloud, cov):
        """NanoGICP::setSource/TargetCovariances: (n, 3, 3) float64 in the ORIGINAL point order."""
        cov = np.ascontiguousarray(cov, np.float64).reshape(cloud.n, 9)
        _check(lib().b200reg_set_covariances(self.h, cloud.h, cov.ctypes.data_as(C.c_void_p), C.c_size_t(cloud.n)))

    # -- registration ------------------------------------------------------------------
    def gicp_align(self, srcs, tgts, params=None, guesses=None):
        cnt = len(srcs)
        prm = params or default_params()
        sa = (C.c_void_p * cnt)(*[c.h for c in srcs])
        ta = (C.c_void_p * cnt)(*[c.h for c in tgts])
        res = (Result * cnt)()
        g = None
        if guesses is not None:
            g = np.ascontiguousarray(guesses, np.float64).reshape(cnt, 16)
        _check(lib().b200reg_gicp_align(self.h, cnt, sa, ta, None if g is None else g.ctypes.data_as(C.c_void_p),
                                        C.byref(prm), res))
        return [r.as_dict() for r in res]

    def icp_alignment(self, src_arrays, tgt_arrays, params=None, raw=False):
        """LoopClosure::icpAlignment for a batch of host (pinned or pageable) buffers."""
        srcs = [_pts(a) for a in src_arrays]
        tgts = [_pts(a) for a in tgt_arrays]
        stride = srcs[0].shape[1] * 4
        cnt = len(srcs)
        prm = params or default_params()
        sp = (C.c_void_p * cnt)(*[a.ctypes.data for a in srcs])
        tp = (C.c_void_p * cnt)(*[a.ctypes.data for a in tgts])
        sn = (C.c_size_t * cnt)(*[len(a) for a in srcs])
        tn = (C.c_size_t * cnt)(*[len(a) for a in tgts])
        res = (Result * cnt)()
        _check(lib().b200reg_icp_alignment(self.h, cnt, sp, sn, tp, tn, C.c_size_t(stride), 0, C.byref(prm), res))
        return res if raw else [r.as_dict() for r in res]

    def icp_alignment_ptrs(self, src_ptrs, src_ns, tgt_ptrs, tgt_ns, stride_bytes, on_device, params=None):
        """Same, from raw addresses (pinned host or device memory owned by the caller, e.g. torch tensors)."""
        cnt = len(src_ptrs)
        prm = params or default_params()
        sp = (C.c_void_p * cnt)(*src_ptrs)
        tp = (C.c_void_p * cnt)(*tgt_ptrs)
        sn = (C.c_size_t * cnt)(*src_ns)
        tn = (C.c_size_t * cnt)(*tgt_ns)
        res = (Result * cnt)()
        _check(lib().b200reg_icp_alignment(self.h, cnt, sp, sn, tp, tn, C.c_size_t(stride_bytes), int(bool(on_device)),
                                           C.byref(prm), res))
        return res

    def transform_cloud(self, cloud, Tf):
        Tf = np.ascontiguousarray(Tf, np.float32).reshape(16)
        out = np.empty((cloud.n, 3), np.float32)
        _check(lib().b200reg_transform_cloud(self.h, cloud.h, Tf.ctypes.data_as(C.c_void_p), out.ctypes.data_as(C.c_void_p)))
        return out

    # -- Quatro --------------------------------------------------------------------------
    def fpfh(self, clouds, normal_radius=0.9, fpfh_radius=1.5):
        arr = (C.c_void_p * len(clouds))(*[c.h for c in clouds])
        _check(lib().b200reg_clouds_fpfh(self.h, len(clouds), arr, C.c_double(normal_radius), C.c_double(fpfh_radius)))

    def get_fpfh(self, cloud):
        nrm = np.empty((cloud.n, 3), np.float32)
        f = np.empty((cloud.n, 33), np.float32)
        _check(lib().b200reg_get_fpfh(self.h, cloud.h, nrm.ctypes.data_as(C.c_void_p), f.ctypes.data_as(C.c_void_p)))
        return nrm, f

    def quatro_align(self, srcs, dsts, params=None, want_corr=False):
        """quatro<T>::align for a batch of cloud handles."""
        cnt = len(srcs)
        prm = params or default_quatro_params()
        sa = (C.c_void_p * cnt)(*[c.h for c in srcs])
        da = (C.c_void_p * cnt)(*[c.h for c in dsts])
        info = (QuatroInfo * cnt)()
        corr = np.zeros((cnt, MAXC if prm.use_optimized_matching else ADV_MAXC, 2), np.int32) if want_corr else None
        _check(lib().b200reg_quatro_align(self.h, cnt, sa, da, C.byref(prm), info,
                                          None if corr is None else corr.ctypes.data_as(C.c_void_p)))
        out = [i.as_dict() for i in info]
        if want_corr:
            for o, cc in zip(out, corr):
                o["corr"] = cc[:o["n_corr"]].copy()
        return out

    def loop_closure(self, src_arrays, tgt_arrays, qparams=None, gparams=None):
        """LoopClosure::coarseToFineAlignment for a batch of host buffers -> (results, quatro infos)."""
        srcs = [_pts(a) for a in src_arrays]
        tgts = [_pts(a) for a in tgt_arrays]
        cnt = len(srcs)
        res = self.loop_closure_ptrs([a.ctypes.data for a in srcs], [len(a) for a in srcs], [a.ctypes.data for a in tgts],
                                     [len(a) for a in tgts], srcs[0].shape[1] * 4, 0, qparams, gparams)
        return [r.as_dict() for r in res[0]], [q.as_dict() for q in res[1]]

    def loop_closure_ptrs(self, src_ptrs, src_ns, tgt_ptrs, tgt_ns, stride_bytes, on_device, qparams=None, gparams=None):
        cnt = len(src_ptrs)
        qp = qparams or default_quatro_params()
        gp = gparams or default_params()
        sp = (C.c_void_p * cnt)(*src_ptrs)
        tp = (C.c_void_p * cnt)(*tgt_ptrs)
        sn = (C.c_size_t * cnt)(*src_ns)
        tn = (C.c_size_t * cnt)(*tgt_ns)
        res = (Result * cnt)()
        qi = (QuatroInfo * cnt)()
        _check(lib().b200reg_loop_closure(self.h, cnt, sp, sn, tp, tn, C.c_size_t(stride_bytes), int(bool(on_device)),
                                          C.byref(qp), C.byref(gp), res, qi))
        return res, qi

    # -- "next" rows: keyframe store, candidate search, cloud assembly -----------------------
    def keyframes(self):
        return Keyframes(self)

    def cloud_points(self, cloud):
        out = np.empty((cloud.n, 3), np.float32)
        _check(lib().b200reg_cloud_points(self.h, cloud.h, out.ctypes.data_as(C.c_void_p)))
        return out

    # -- debug taps ----------------------------------------------------------------------
    def knn(self, cloud, queries, k, brute=False):
        q = _pts(queries)
        idx = np.empty((len(q), k), np.int32)
        d2 = np.empty((len(q), k), np.float32)
        fn = lib().b200reg_knn_bruteforce if brute else lib().b200reg_knn
        _check(fn(self.h, cloud.h, q.ctypes.data_as(C.c_void_p), C.c_size_t(len(q)),
                                 C.c_size_t(q.shape[1] * 4), int(k), idx.ctypes.data_as(C.c_void_p),
                                 d2.ctypes.data_as(C.c_void_p)))
        return idx, d2

    def get_covariances(self, cloud):
        out = np.empty((cloud.n, 3, 3), np.float64)
        _check(lib().b200reg_get_covariances(self.h, cloud.h, out.ctypes.data_as(C.c_void_p)))
        return out

    def linearize(self, src, tgt, T, max_corr_dist=52.5):
        T = np.ascontiguousarray(T, np.float64).reshape(16)
        H = np.empty((6, 6), np.float64)
        b = np.empty(6, np.float64)
        err = C.c_double()
        corr = np.empty(src.n, np.int32)
        sqd = np.empty(src.n, np.float32)
        _check(lib().b200reg_linearize(self.h, src.h, tgt.h, T.ctypes.data_as(C.c_void_p), C.c_double(max_corr_dist),
                                       H.ctypes.data_as(C.c_void_p), b.ctypes.data_as(C.c_void_p), C.byref(err),
                                       corr.ctypes.data_as(C.c_void_p), sqd.ctypes.data_as(C.c_void_p)))
        return dict(H=H, b=b, err=err.value, corr=corr, sqd=sqd)

    def compute_error(self, src, tgt, T_lin, T_trial, max_corr_dist=52.5):
        """NanoGICP::compute_error at T_trial with the stale correspondences / Mahalanobis matrices of a linearize at T_lin."""
        Tl = np.ascontiguousarray(T_lin, np.float64).reshape(16)
        Tt = np.ascontiguousarray(T_trial, np.float64).reshape(16)
        err = C.c_double()
        _check(lib().b200reg_compute_error(self.h, src.h, tgt.h, Tl.ctypes.data_as(C.c_void_p), Tt.ctypes.data_as(C.c_void_p),
                                           C.c_double(max_corr_dist), C.byref(err)))
        return err.value


def comm_unique_id():
    """ncclGetUniqueId through the C ABI (rank 0 calls it; the 128 bytes go to the other ranks by any side channel)."""
    buf = (C.c_ubyte * 128)()
    _check(lib().b200reg_comm_unique_id(buf))
    return bytes(buf)


class Batch:
    """b200reg_batch: `depth` engine contexts on their own host threads (C++), jobs round-robin (include/b200reg.h)."""

    def __init__(self, device=0, depth=3):
        self.h = C.c_void_p()
        _check(lib().b200reg_batch_create(int(device), int(depth), C.byref(self.h)))
        self._keep = {}

    def close(self):
        if self.h:
            lib().b200reg_batch_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def depth(self):
        return int(lib().b200reg_batch_depth(self.h))

    @property
    def launch_count(self):
        return int(lib().b200reg_batch_launch_count(self.h))

    @staticmethod
    def _arrays(src_ptrs, src_ns, tgt_ptrs, tgt_ns):
        cnt = len(src_ptrs)
        return (cnt, (C.c_void_p * cnt)(*src_ptrs), (C.c_size_t * cnt)(*src_ns), (C.c_void_p * cnt)(*tgt_ptrs),
                (C.c_size_t * cnt)(*tgt_ns))

    def submit_icp(self, src_ptrs, src_ns, tgt_ptrs, tgt_ns, stride_bytes, on_device, params=None):
        """LoopClosure::icpAlignment for a batch of raw addresses; returns a ticket (wait() gives the Result array)."""
        cnt, sp, sn, tp, tn = self._arrays(src_ptrs, src_ns, tgt_ptrs, tgt_ns)
        prm = params or default_params()
        res = (Result * cnt)()
        t = lib().b200reg_batch_submit_icp(self.h, cnt, sp, sn, tp, tn, C.c_size_t(stride_bytes), int(bool(on_device)), C.byref(prm), res)
        if t < 0:
            _check(int(t))
        self._keep[t] = (res, None)
        return t

    def submit_loop_closure(self, src_ptrs, src_ns, tgt_ptrs, tgt_ns, stride_bytes, on_device, qparams=None, gparams=None):
        cnt, sp, sn, tp, tn = self._arrays(src_ptrs, src_ns, tgt_ptrs, tgt_ns)
        qp = qparams or default_quatro_params()
        gp = gparams or default_params()
        res = (Result * cnt)()
        qi = (QuatroInfo * cnt)()
        t = lib().b200reg_batch_submit_loop_closure(self.h, cnt, sp, sn, tp, tn, C.c_size_t(stride_bytes), int(bool(on_device)),
                                                    C.byref(qp), C.byref(gp), res, qi)
        if t < 0:
            _check(int(t))
        self._keep[t] = (res, qi)
        return t

    def wait(self, ticket, want_latency=False, want_quatro=False):
        lat = C.c_double()
        rc = lib().b200reg_batch_wait(self.h, C.c_int64(ticket), C.byref(lat))
        res, qi = self._keep.pop(ticket)
        _check(rc)
        out = (res, qi) if want_quatro else res
        return (out, lat.value) if want_latency else out


class Keyframes:
    """Device-resident keyframe store (PosePcd records) + batched loopTimerFunc pieces."""

    def __init__(self, ctx):
        self.ctx = ctx
        self.h = C.c_void_p()
        _check(lib().b200reg_keyframes_create(ctx.h, C.byref(self.h)))

    def destroy(self):
        if self.h:
            lib().b200reg_keyframes_destroy(self.ctx.h, self.h)
            self.h = None

    def __len__(self):
        return int(lib().b200reg_keyframes_size(self.h))

    def reserve(self, n_points):
        """Device room for n_points more points, allocated now (adds allocate nothing until it is used up)."""
        _check(lib().b200reg_keyframes_reserve(self.ctx.h, self.h, C.c_size_t(int(n_points))))

    def add(self, cloud_xyzi, pose, stamp):
        a = np.ascontiguousarray(cloud_xyzi, np.float32)
        assert a.ndim == 2 and a.shape[1] >= 4
        T = np.ascontiguousarray(pose, np.float64).reshape(16)
        rc = lib().b200reg_keyframes_add(self.ctx.h, self.h, a.ctypes.data_as(C.c_void_p), C.c_size_t(len(a)),
                                         C.c_size_t(a.shape[1] * 4), T.ctypes.data_as(C.c_void_p), C.c_double(stamp))
        if rc < 0:
            _check(rc)
        return rc

    def add_world(self, cloud_xyzi_world, position, quat_xyzw, stamp):
        """PosePcd::PosePcd (pose_pcd.hpp:21-43): world-frame scan + odometry (position, quaternion x y z w) -> keyframe."""
        a = np.ascontiguousarray(cloud_xyzi_world, np.float32)
        assert a.ndim == 2 and a.shape[1] >= 4
        p = np.ascontiguousarray(position, np.float64).reshape(3)
        q = np.ascontiguousarray(quat_xyzw, np.float64).reshape(4)
        rc = lib().b200reg_keyframes_add_world(self.ctx.h, self.h, a.ctypes.data_as(C.c_void_p), C.c_size_t(len(a)), C.c_size_t(a.shape[1] * 4),
                                               p.ctypes.data_as(C.c_void_p), q.ctypes.data_as(C.c_void_p), C.c_double(stamp))
        if rc < 0:
            _check(rc)
        return rc

    def get(self, idx):
        """-> (cloud (n,4) float32 in the LiDAR frame, corrected pose (4,4), timestamp)."""
        n = int(lib().b200reg_keyframes_cloud_size(self.h, int(idx)))
        pts = np.empty((n, 4), np.float32)
        pose = np.empty(16, np.float64)
        ts = C.c_double()
        _check(lib().b200reg_keyframes_get(self.ctx.h, self.h, int(idx), pts.ctypes.data_as(C.c_void_p), pose.ctypes.data_as(C.c_void_p), C.byref(ts)))
        return pts, pose.reshape(4, 4), ts.value

    def set_pose(self, idx, pose):
        T = np.ascontiguousarray(pose, np.float64).reshape(16)
        _check(lib().b200reg_keyframes_set_pose(self.ctx.h, self.h, int(idx), T.ctypes.data_as(C.c_void_p)))

    def fetch_closest(self, queries, radius=35.0, tdiff=30.0):
        q = np.ascontiguousarray(queries, np.int32)
        out = np.empty(len(q), np.int32)
        _check(lib().b200reg_fetch_closest_keyframes(self.ctx.h, self.h, len(q), q.ctypes.data_as(C.c_void_p), C.c_double(radius),
                                                     C.c_double(tdiff), out.ctypes.data_as(C.c_void_p)))
        return out

    def assemble(self, src_idx, dst_idx, cfg=None, n_keyframes=0):
        """n_keyframes: keyframes.size() the sub-map bounds see -- one int for the batch (0 = the store's size) or one per pair."""
        cfg = cfg or default_loop_config()
        s = np.ascontiguousarray(src_idx, np.int32)
        d = np.ascontiguousarray(dst_idx, np.int32)
        cnt = len(s)
        so, do = (C.c_void_p * cnt)(), (C.c_void_p * cnt)()
        if np.ndim(n_keyframes) > 0:
            nk = np.ascontiguousarray(n_keyframes, np.int32)
            assert len(nk) == cnt
            _check(lib().b200reg_assemble_clouds_at(self.ctx.h, self.h, cnt, s.ctypes.data_as(C.c_void_p), d.ctypes.data_as(C.c_void_p),
                                                    C.byref(cfg), nk.ctypes.data_as(C.c_void_p), so, do))
        else:
            _check(lib().b200reg_assemble_clouds(self.ctx.h, self.h, cnt, s.ctypes.data_as(C.c_void_p), d.ctypes.data_as(C.c_void_p),
                                                 C.byref(cfg), int(n_keyframes), so, do))
        mk = lambda h: Cloud(self.ctx, C.c_void_p(h), int(lib().b200reg_cloud_size(C.c_void_p(h))))
        return [mk(so[i]) for i in range(cnt)], [mk(do[i]) for i in range(cnt)]

    def perform_loop_closure(self, query_idx, closest_idx, cfg=None, raw=False):
        cfg = cfg or default_loop_config()
        q = np.ascontiguousarray(query_idx, np.int32)
        cidx = np.ascontiguousarray(closest_idx, np.int32)
        cnt = len(q)
        res = (Result * cnt)()
        qi = (QuatroInfo * cnt)()
        _check(lib().b200reg_perform_loop_closure(self.ctx.h, self.h, cnt, q.ctypes.data_as(C.c_void_p), cidx.ctypes.data_as(C.c_void_p),
                                                  C.byref(cfg), res, qi))
        if raw:
            return res, qi
        return [r.as_dict() for r in res], [x.as_dict() for x in qi]

    def build_map(self, voxel_res=0.3, n_keyframes=0):
        """The corrected global map (fast_lio_sam_qn.cpp:302-316, :398-411, :435-449): keyframes 0 .. n_keyframes-1 (0 = all)
        transformed by their corrected poses, merged, voxelised at voxel_res.  -> (records (m, 4) float32 x y z intensity
        in voxel-index order, voxelized); voxelized is False when PCL's int32 index guard tripped and the records are the
        merged cloud unchanged."""
        h = C.c_void_p()
        _check(lib().b200reg_map_build(self.ctx.h, self.h, int(n_keyframes), C.c_double(voxel_res), C.byref(h)))
        try:
            out = np.empty((int(lib().b200reg_map_size(h)), 4), np.float32)
            voxelized = bool(lib().b200reg_map_voxelized(h))
            _check(lib().b200reg_map_get(self.ctx.h, h, out.ctypes.data_as(C.c_void_p)))
        finally:
            _check(lib().b200reg_map_destroy(self.ctx.h, h))
        return out, voxelized

    def loop_factors(self, query_idx, closest_idx, raw_results):
        """The BetweenFactor records of a perform_loop_closure(..., raw=True) batch (fast_lio_sam_qn.cpp:220-237)."""
        q = np.ascontiguousarray(query_idx, np.int32)
        cidx = np.ascontiguousarray(closest_idx, np.int32)
        out = (LoopFactor * len(q))()
        _check(lib().b200reg_loop_factors(self.ctx.h, self.h, len(q), q.ctypes.data_as(C.c_void_p), cidx.ctypes.data_as(C.c_void_p),
                                          raw_results, out))
        return [f.as_dict() for f in out]

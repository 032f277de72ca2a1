"""ctypes binding of libcatgrasp_b200.so (the C ABI declared in include/catgrasp_b200.h).

The product path has NO CPU fallback: if the shared library is missing or no
B200 is present, every entry point raises.  Build the library with
``python -c "import __graft_entry__ as g; g.build()"`` (nvcc, sm_100a).
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libcatgrasp_b200.so")

CG_OK, CG_EINVAL, CG_ECUDA, CG_ENOMEM, CG_EUNSUPPORTED = 0, -1, -2, -3, -4
CG_NET_CLS, CG_NET_SEG = 0, 1
CG_SDF_TRILINEAR, CG_SDF_NEAREST = 0, 1
CG_ST_ACCEPT, CG_ST_REJ_DIR, CG_ST_REJ_IK, CG_ST_REJ_COLL, CG_ST_REJ_COLL_ENCL = 0, 1, 2, 3, 4


class CgError(RuntimeError):
    pass


class FilterParams(C.Structure):
    _fields_ = [
        ("nocs_pose", C.c_float * 16),
        ("canonical_to_nocs", C.c_float * 16),
        ("gripper_in_grasp", C.c_float * 16),
        ("filter_approach_dir_face_camera", C.c_int),
        ("adjust_collision_pose", C.c_int),
        ("sdf_mode", C.c_int),
        ("sdf_margin", C.c_float),
        ("split_coll_status", C.c_int),
    ]


_vp, _i, _f, _sz = C.c_void_p, C.c_int, C.c_float, C.c_size_t

# name -> (restype, argtypes); must list every symbol of include/catgrasp_b200.h
SIGNATURES = {
    "cg_ctx_create": (_i, [_i, C.POINTER(_vp)]),
    "cg_ctx_destroy": (None, [_vp]),
    "cg_ctx_set_stream": (_i, [_vp, _vp]),
    "cg_ctx_use_own_stream": (_i, [_vp]),
    "cg_ctx_synchronize": (_i, [_vp]),
    "cg_last_error": (C.c_char_p, [_vp]),
    "cg_version": (C.c_char_p, []),
    "cg_ctx_launch_count": (C.c_int64, [_vp]),
    "cg_ctx_reset_launch_count": (None, [_vp]),
    "cg_ctx_set_engine": (_i, [_vp, _i]),
    "cg_ctx_get_engine": (_i, [_vp]),
    "cg_ctx_fp16_overflow": (_i, [_vp, C.POINTER(_i)]),
    "cg_tmem_layout_selftest": (_i, [_vp, _vp]),
    "cg_ctx_profile": (_i, [_vp, _i]),
    "cg_ctx_profile_read": (_i, [_vp, C.POINTER(C.c_double), C.POINTER(C.c_int64)]),
    "cg_net_create": (_i, [_vp, _i, _i, _vp, _sz, C.POINTER(_vp)]),
    "cg_net_destroy": (None, [_vp]),
    "cg_net_blob_floats": (_sz, [_i, _i]),
    "cg_graspq_forward_host": (_i, [_vp, _vp, _vp, _i, _vp, _i, _vp, _i, _vp, _vp, _vp, _vp]),
    "cg_graspq_forward_dev": (_i, [_vp, _vp, _vp, _i, _vp, _i, _vp, _i, _vp, _vp, _vp, _vp]),
    "cg_host_legacy_choice": (_i, [_vp, C.POINTER(C.c_int32), C.c_int64, C.c_int32, C.c_int32, _vp, C.c_int32]),
    "cg_host_legacy_skip": (_i, [_vp, C.POINTER(C.c_int32), C.c_int64, C.c_int32, C.c_int32]),
    "cg_host_rng_isa": (_i, [_i]),
    "cg_draw_ids_dev": (_i, [_vp, _i, _i, _i, C.c_uint64, C.c_int64, _vp]),
    "cg_mlp_create": (_i, [_vp, _i, _vp, _vp, _vp, C.POINTER(_vp)]),
    "cg_mlp_destroy": (None, [_vp]),
    "cg_shared_mlp_dev": (_i, [_vp, _vp, C.c_int64, _vp]),
    "cg_group_mlp_max_dev": (_i, [_vp, _vp, _i, _i, _vp]),
    "cg_three_interp_dev": (_i, [_vp, _vp, _vp, _vp, _i, _vp, _i, _i, _i, _i, _vp, _vp, _vp]),
    "cg_cls_forward_dev": (_i, [_vp, _vp, _i, _i, _vp, _vp]),
    "cg_seg_forward_dev": (_i, [_vp, _vp, _i, _i, _vp]),
    "cg_nunocs_forward_host": (_i, [_vp, _vp, _i, _i, _vp, _vp, _vp]),
    "cg_nunocs_forward_dev": (_i, [_vp, _vp, _i, _i, _vp, _vp, _vp]),
    "cg_sdf_create": (_i, [_vp, _vp, _i, _i, _i, C.POINTER(_f), _f, C.POINTER(_vp)]),
    "cg_sdf_destroy": (None, [_vp]),
    "cg_sdf_lookup_dev": (_i, [_vp, _vp, _i, _i, _vp]),
    "cg_filter_grasp_pose_host": (_i, [_vp, C.POINTER(FilterParams), _vp, _i, _vp, _i, _vp, _vp, _i, _vp, _vp, _i,
                                       _vp, _vp, _vp]),
    "cg_filter_grasp_pose_dev": (_i, [_vp, C.POINTER(FilterParams), _vp, _i, _vp, _i, _vp, _vp, _i, _vp, _vp, _i,
                                      _vp, _vp, _vp]),
    "cg_mesh_create": (_i, [_vp, _vp, _i, _vp, _i, C.POINTER(_vp)]),
    "cg_mesh_destroy": (None, [_vp]),
    "cg_mesh_info": (_i, [_vp, C.POINTER(_i), C.POINTER(_f), C.POINTER(C.c_int64)]),
    "cg_voxels_create_dev": (_i, [_vp, _vp, _i, _f, C.POINTER(_vp)]),
    "cg_voxels_destroy": (None, [_vp]),
    "cg_voxels_count": (_i, [_vp, C.POINTER(_i)]),
    "cg_voxels_keys_host": (_i, [_vp, _vp]),
    "cg_filter_grasp_pose_mesh_dev": (_i, [_vp, C.POINTER(FilterParams), _vp, _i, _vp, _i, _vp, _vp, _vp, _vp,
                                           _vp, _vp, _vp]),
    "cg_filter_grasp_pose_mesh_host": (_i, [_vp, C.POINTER(FilterParams), _vp, _i, _vp, _i, _vp, _vp, _i, _vp, _vp,
                                            _i, _f, _vp, _vp, _vp]),
    "cg_occupancy_grid_geometry": (_i, [_vp, _i, _f, C.POINTER(_i), C.POINTER(_f)]),
    "cg_occupancy_from_scan_host": (_i, [_vp, _vp, _i, _f, _vp]),
    "cg_ransac9d_host": (_i, [_vp, _vp, _vp, _i, _vp, _i, C.c_double, _vp, _vp, _vp, _vp, _vp, _vp]),
    "cg_cone_poses_dev": (_i, [_vp, _vp, _vp, _i, _vp, _i, _vp, _i, _vp, _i, C.c_double, _vp, _vp]),
    "cg_center_grasps_dev": (_i, [_vp, _vp, _vp, _i, _vp, _i]),
    "cg_grasp_affordance_dev": (_i, [_vp, _vp, _i, _vp, _vp, _vp, _i, _vp, _vp, _i, C.c_double, _vp, _vp]),
    "cg_square_distance_dev": (_i, [_vp, _vp, _vp, _i, _i, _i, _vp]),
    "cg_index_points_dev": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _vp]),
    "cg_fps_dev": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp]),
    "cg_fps_single_cta_dev": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp]),
    "cg_ball_query_dev": (_i, [_vp, _f, _i, _vp, _vp, _i, _i, _i, _vp]),
    "cg_group_points_dev": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _vp]),
    "cg_cloud_create_dev": (_i, [_vp, _vp, _i, C.c_double, C.POINTER(_vp)]),
    "cg_cloud_destroy": (None, [_vp]),
    "cg_cloud_nearest_dev": (_i, [_vp, _vp, _i, _vp, _vp]),
    "cg_cloud_any_within_dev": (_i, [_vp, _vp, _i, C.c_double, _vp]),
    "cg_cloud_normals_dev": (_i, [_vp, C.c_double, _i, C.POINTER(C.c_double), _vp, _vp]),
    "cg_voxel_down_sample_dev": (_i, [_vp, _vp, _vp, _i, C.c_double, _vp, _vp, _vp]),
}

_lib = None


def load():
    """Load the shared library (once) and attach prototypes.  Raises if it is not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise CgError(
            f"{LIB_PATH} is missing: the CUDA extension has not been built "
            "(run __graft_entry__.build()). There is no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError here means header/library drift
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def ptr(t):
    """Device/host pointer of a torch tensor or numpy array (None -> NULL)."""
    if t is None:
        return None
    if hasattr(t, "data_ptr"):
        return C.c_void_p(t.data_ptr())
    return C.c_void_p(t.ctypes.data)


class Context:
    """One library context per device (stream + workspaces)."""

    _per_device = {}

    def __init__(self, device=0):
        lib = load()
        self.lib = lib
        self.device = int(device)
        h = _vp()
        rc = lib.cg_ctx_create(self.device, C.byref(h))
        if rc != CG_OK:
            raise CgError(f"cg_ctx_create(device={device}) failed with {rc}: "
                          "a B200 (sm_100) GPU is required; there is no CPU fallback")
        self.h = h

    @classmethod
    def get(cls, device=None):
        import torch
        if device is None:
            device = torch.cuda.current_device() if torch.cuda.is_available() else 0
        device = int(device)
        if device not in cls._per_device:
            cls._per_device[device] = cls(device)
        return cls._per_device[device]

    def check(self, rc):
        if rc != CG_OK:
            msg = self.lib.cg_last_error(self.h)
            raise CgError(f"libcatgrasp_b200 error {rc}: {msg.decode() if msg else ''}")

    def use_torch_stream(self):
        import torch
        s = torch.cuda.current_stream(self.device).cuda_stream
        self.check(self.lib.cg_ctx_set_stream(self.h, C.c_void_p(s)))

    def use_own_stream(self):
        self.check(self.lib.cg_ctx_use_own_stream(self.h))

    def synchronize(self):
        self.check(self.lib.cg_ctx_synchronize(self.h))

    def set_engine(self, engine):
        self.check(self.lib.cg_ctx_set_engine(self.h, int(engine)))

    def get_engine(self):
        return int(self.lib.cg_ctx_get_engine(self.h))

    def fp16_overflow(self):
        """True if engine 2/3 had to clamp an activation to the fp16 range since the last call (clears the flag)."""
        v = C.c_int()
        self.check(self.lib.cg_ctx_fp16_overflow(self.h, C.byref(v)))
        return bool(v.value)

    def profile(self, enable):
        self.check(self.lib.cg_ctx_profile(self.h, int(bool(enable))))

    def profile_read(self):
        ms, n = C.c_double(), C.c_int64()
        self.check(self.lib.cg_ctx_profile_read(self.h, C.byref(ms), C.byref(n)))
        return ms.value, n.value

    def launch_count(self):
        return int(self.lib.cg_ctx_launch_count(self.h))

    def reset_launch_count(self):
        self.lib.cg_ctx_reset_launch_count(self.h)

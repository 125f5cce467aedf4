"""ctypes view of the C ABI declared in include/auvrrt.h (libauvrrt.so).

The library is the product: if it is missing, or no CUDA device is present, calls fail loudly --
there is no CPU fallback here or anywhere in this package.
"""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("AUVRRT_LIB") or os.path.join(HERE, "libauvrrt.so")

F32, F64 = 0, 1
ST_OK, ST_NO_PATH, ST_ZERO_DIV, ST_KEY_ERROR, ST_STREAM_END, ST_OVERFLOW = range(6)

_dp = C.POINTER(C.c_double)
_i32p = C.POINTER(C.c_int32)
_i64p = C.POINTER(C.c_int64)
_u8p = C.POINTER(C.c_uint8)
_u32p = C.POINTER(C.c_uint32)
_u64p = C.POINTER(C.c_uint64)


class PlanParams(C.Structure):
    _fields_ = [("iterations", C.c_int32), ("mode", C.c_int32), ("bin_interval", C.c_double),
                ("v", C.c_double), ("max_traj_time", C.c_double), ("dist_to_end", C.c_double),
                ("diff_max", C.c_double), ("freq", C.c_double), ("min_dist", C.c_double),
                ("weights", C.c_double * 3), ("chain_cap", C.c_int32), ("path_cap", C.c_int32),
                ("trace", C.c_int32), ("group", C.c_int32), ("max_plan_time", C.c_double),
                ("dubins_rho", C.c_double), ("dubins_eta", C.c_double), ("near_radius", C.c_double),
                ("dubins_w", C.c_int32), ("reserved", C.c_int32)]


class PlanRecord(C.Structure):
    _fields_ = [("status", C.c_int32), ("n_nodes", C.c_int32), ("best_node", C.c_int32),
                ("best_iter", C.c_int32), ("depth", C.c_int32), ("n_path", C.c_int32),
                ("n_cost_evals", C.c_int32), ("n_waypoints", C.c_int32), ("n_uniforms", C.c_int64),
                ("n_primitives", C.c_int64), ("cost", C.c_double * 4), ("path_length", C.c_double),
                ("t_leaf", C.c_double)]


class GymParams(C.Structure):
    _fields_ = [("x0", C.c_double), ("y0", C.c_double), ("x1", C.c_double), ("y1", C.c_double),
                ("exp_rate", C.c_double), ("dist_to_end", C.c_double), ("diff_max", C.c_double),
                ("freq", C.c_double), ("cell_side", C.c_double), ("subsections", C.c_int32),
                ("node_cap", C.c_int32), ("track_counts", C.c_int32), ("reserved", C.c_int32)]


class GymRecord(C.Structure):
    _fields_ = [("status", C.c_int32), ("done", C.c_int32), ("steps", C.c_int32), ("n_nodes", C.c_int32),
                ("n_occupied", C.c_int32), ("last_parent", C.c_int32), ("last_accepted", C.c_int32),
                ("last_nwp", C.c_int32), ("last_uniforms", C.c_int32), ("n_path", C.c_int32),
                ("n_uniforms", C.c_int64), ("cand", C.c_double * 4), ("arc_length", C.c_double)]


class AstarQuery(C.Structure):
    _fields_ = [("start", C.c_double * 2), ("path_len_limit", C.c_double), ("weights", C.c_double * 4),
                ("velocity", C.c_double)]


class AstarRecord(C.Structure):
    _fields_ = [("status", C.c_int32), ("n_expanded", C.c_int32), ("n_nodes", C.c_int32), ("n_path", C.c_int32),
                ("n_smooth", C.c_int32), ("reserved", C.c_int32), ("cost", C.c_double), ("path_len", C.c_double)]


class PlanTrace(C.Structure):
    _fields_ = [("parent", _i32p), ("safe", _u8p), ("nwp", _i32p), ("leaf", _dp), ("upos", _i64p)]


EXPORTS = [
    "auvrrt_last_error", "auvrrt_device_count", "auvrrt_launch_count", "auvrrt_env_create",
    "auvrrt_env_destroy", "auvrrt_nn", "auvrrt_nn_dev", "auvrrt_nn_scratch_bytes", "auvrrt_steer_arc",
    "auvrrt_steer_dubins", "auvrrt_collide", "auvrrt_collide_points", "auvrrt_cost",
    "auvrrt_cost_point", "auvrrt_edges_dubins_dev", "auvrrt_edges_arc_dev", "auvrrt_edges_dubins",
    "auvrrt_edges_arc", "auvrrt_stream_u", "auvrrt_plan_batch", "auvrrt_plan_workspace_bytes", "auvrrt_plan_workspace_bytes_q",
    "auvrrt_plan_batch_dev", "auvrrt_materialize", "auvrrt_calibrate_fp32", "auvrrt_occupancy_dims", "auvrrt_occupancy_grid",
    "auvrrt_gym_create", "auvrrt_gym_destroy", "auvrrt_gym_grid_shape", "auvrrt_gym_reset", "auvrrt_gym_reset_dev", "auvrrt_gym_step",
    "auvrrt_gym_step_dev", "auvrrt_gym_tree", "auvrrt_gym_counts", "auvrrt_gym_counts_dev", "auvrrt_gym_path",
    "auvrrt_astar_env_create", "auvrrt_astar_env_destroy", "auvrrt_astar_batch", "auvrrt_astar_workspace_bytes",
    "auvrrt_astar_batch_dev", "auvrrt_edges_arc_cost_dev", "auvrrt_edges_arc_cost", "auvrrt_env_host_blob",
    "auvrrt_edges_dubins_cost_dev", "auvrrt_edges_dubins_cost", "auvrrt_occ_create", "auvrrt_occ_destroy", "auvrrt_occ_shape",
    "auvrrt_occ_grid_dev", "auvrrt_env_set_probs", "auvrrt_env_set_probs_dev", "auvrrt_env_get_probs",
]

_lib = None


class AuvrrtError(RuntimeError):
    pass


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise AuvrrtError("libauvrrt.so is not built (%s). Run `python __graft_entry__.py` or "
                          "`make -C auv-sim_b200/csrc`; there is no CPU fallback." % LIB_PATH)
    L = C.CDLL(LIB_PATH)
    vp = C.c_void_p
    L.auvrrt_last_error.restype = C.c_char_p
    L.auvrrt_device_count.restype = C.c_int
    L.auvrrt_launch_count.restype = C.c_int64
    L.auvrrt_env_create.argtypes = [_dp, C.c_int, _dp, C.c_int, _dp, C.c_int, _dp, C.c_int, _dp, C.c_int,
                                    _dp, C.c_int, C.POINTER(vp)]
    L.auvrrt_env_destroy.argtypes = [vp]
    L.auvrrt_env_destroy.restype = None
    L.auvrrt_env_host_blob.argtypes = [_dp, C.c_int, _dp, C.c_int, _dp, C.c_int, _dp, C.c_int, _dp, C.c_int,
                                       _dp, C.c_int, vp, C.c_int64]
    L.auvrrt_env_host_blob.restype = C.c_int64
    L.auvrrt_nn.argtypes = [_dp, _dp, C.c_int64, _dp, _dp, C.c_int, C.c_int, C.c_int, _i32p]
    L.auvrrt_nn_dev.argtypes = [vp, vp, C.c_int64, vp, vp, C.c_int, C.c_int, vp, C.c_int64, vp, vp]
    L.auvrrt_nn_scratch_bytes.restype = C.c_int64
    L.auvrrt_nn_scratch_bytes.argtypes = [C.c_int]
    L.auvrrt_steer_arc.argtypes = [_dp, C.c_int64, _dp, _i64p, _dp, C.c_int, C.c_int, _dp, _i32p, _dp,
                                   C.c_int, _i32p, _i32p]
    L.auvrrt_steer_dubins.argtypes = [_dp, _dp, C.c_int64, C.c_double, C.c_int, C.c_int, C.c_int, _u8p,
                                      _dp, _dp, _dp]
    L.auvrrt_collide.argtypes = [vp, _dp, _i64p, C.c_int64, C.c_int, _u8p]
    L.auvrrt_collide_points.argtypes = [vp, _dp, C.c_int64, C.c_int, _u8p]
    L.auvrrt_cost.argtypes = [vp, _dp, _i64p, C.c_int64, _dp, _dp, _u8p, C.c_int, C.c_int, _dp]
    L.auvrrt_cost_point.argtypes = [vp, _dp, C.c_int64, _u8p, C.c_int, _dp, C.c_int, _dp]
    L.auvrrt_edges_dubins_dev.argtypes = [vp, vp, vp, C.c_int64, C.c_double, C.c_int, C.c_int, vp, vp, vp, vp]
    L.auvrrt_edges_arc_dev.argtypes = [vp, vp, vp, C.c_int64, _dp, C.c_int, vp, vp, vp, vp]
    L.auvrrt_edges_dubins.argtypes = [vp, _dp, _dp, C.c_int64, C.c_double, C.c_int, C.c_int, _u8p, _u8p, _dp]
    L.auvrrt_edges_arc.argtypes = [vp, _dp, _u64p, C.c_int64, _dp, C.c_int, _u8p, _i32p, _dp]
    L.auvrrt_edges_arc_cost_dev.argtypes = [vp, vp, vp, C.c_int64, _dp, C.c_double, C.c_int, vp, vp, vp, vp, vp]
    L.auvrrt_edges_arc_cost.argtypes = [vp, _dp, _u64p, C.c_int64, _dp, C.c_double, C.c_int, _u8p, _i32p, _dp, _dp]
    L.auvrrt_edges_dubins_cost_dev.argtypes = [vp, vp, vp, C.c_int64, C.c_double, C.c_int, C.c_double, C.c_double, C.c_int,
                                               vp, vp, vp, vp, vp]
    L.auvrrt_edges_dubins_cost.argtypes = [vp, _dp, _dp, C.c_int64, C.c_double, C.c_int, C.c_double, C.c_double, C.c_int,
                                           _u8p, _u8p, _dp, _dp]
    L.auvrrt_stream_u.restype = C.c_double
    L.auvrrt_stream_u.argtypes = [C.c_uint64, C.c_int64, C.c_int]
    L.auvrrt_plan_batch.argtypes = [vp, _dp, _u64p, C.c_int64, C.POINTER(PlanParams), C.c_int,
                                    C.POINTER(PlanRecord), _u32p, _dp, C.POINTER(PlanTrace)]
    L.auvrrt_plan_workspace_bytes.restype = C.c_int64
    L.auvrrt_plan_workspace_bytes.argtypes = [vp, C.POINTER(PlanParams), C.c_int]
    L.auvrrt_plan_workspace_bytes_q.restype = C.c_int64
    L.auvrrt_plan_workspace_bytes_q.argtypes = [vp, C.POINTER(PlanParams), C.c_int, C.c_int64]
    L.auvrrt_plan_batch_dev.argtypes = [vp, vp, vp, C.c_int64, C.POINTER(PlanParams), C.c_int, vp, C.c_int64,
                                        vp, vp, vp, C.POINTER(PlanTrace), vp]
    L.auvrrt_materialize.argtypes = [vp, _dp, _u64p, _u32p, _i32p, C.c_int64, C.POINTER(PlanParams), C.c_int,
                                     _dp, _i32p]
    L.auvrrt_calibrate_fp32.argtypes = [C.c_int, C.c_int, _dp, _dp]
    _ip = C.POINTER(C.c_int)
    L.auvrrt_occupancy_dims.argtypes = [_dp, C.c_double, C.c_double, _dp, _i64p, C.c_int, _ip, _ip, _ip]
    L.auvrrt_occupancy_grid.argtypes = [_dp, _i64p, C.c_int, _dp, C.c_double, C.c_double, C.c_double, _dp, _i64p,
                                        C.c_int, C.c_int, _dp, C.c_int64]
    L.auvrrt_occ_create.argtypes = [_dp, _i64p, C.c_int, _dp, C.c_double, C.c_double, C.c_double, C.c_int, C.c_int,
                                    C.c_int64, C.c_int, C.POINTER(vp)]
    L.auvrrt_occ_destroy.argtypes = [vp]
    L.auvrrt_occ_destroy.restype = None
    L.auvrrt_occ_shape.argtypes = [vp, _ip, _ip, _ip]
    L.auvrrt_occ_grid_dev.argtypes = [vp, vp, vp, C.c_int, C.c_int64, vp, vp, vp, vp]
    L.auvrrt_env_set_probs.argtypes = [vp, _dp]
    L.auvrrt_env_set_probs_dev.argtypes = [vp, vp, vp]
    L.auvrrt_env_get_probs.argtypes = [vp, C.c_int, _dp]
    _u16p = C.POINTER(C.c_uint16)
    L.auvrrt_gym_create.argtypes = [_dp, C.c_int, C.POINTER(GymParams), C.c_int64, C.c_int, C.c_int, C.POINTER(vp)]
    L.auvrrt_gym_destroy.argtypes = [vp]
    L.auvrrt_gym_destroy.restype = None
    L.auvrrt_gym_grid_shape.argtypes = [vp, _ip, _ip]
    L.auvrrt_gym_reset.argtypes = [vp, _dp, _dp, _u64p]
    L.auvrrt_gym_reset_dev.argtypes = [vp, vp, vp, vp, vp, vp]
    L.auvrrt_gym_step.argtypes = [vp, _i32p, C.c_int, C.c_int, vp]
    L.auvrrt_gym_step_dev.argtypes = [vp, vp, C.c_int, C.c_int, vp, vp]
    L.auvrrt_gym_tree.argtypes = [vp, C.c_int64, C.c_int32, _dp, _i32p, _i32p, _i32p, _i32p, _i32p]
    L.auvrrt_gym_counts.argtypes = [vp, C.c_int64, C.c_int64, _u16p]
    L.auvrrt_gym_counts_dev.restype = vp
    L.auvrrt_gym_counts_dev.argtypes = [vp]
    L.auvrrt_gym_path.argtypes = [vp, C.c_int64, C.c_int32, _dp, _i32p]
    L.auvrrt_astar_env_create.argtypes = [_dp, C.c_int, _dp, C.c_int, _dp, _dp, C.c_int, _dp, C.c_int, _dp, C.c_int, _dp,
                                          C.c_int, C.POINTER(vp)]
    L.auvrrt_astar_env_destroy.argtypes = [vp]
    L.auvrrt_astar_env_destroy.restype = None
    L.auvrrt_astar_batch.argtypes = [vp, vp, C.c_int64, C.c_int32, C.c_int32, vp, _dp, _u8p, _i32p, _dp]
    L.auvrrt_astar_workspace_bytes.restype = C.c_int64
    L.auvrrt_astar_workspace_bytes.argtypes = [C.c_int64, C.c_int32]
    L.auvrrt_astar_batch_dev.argtypes = [vp, vp, C.c_int64, C.c_int32, C.c_int32, vp, C.c_int64, vp, vp, vp, vp, vp, vp]
    _lib = L
    return L


def check(rc):
    if rc != 0:
        raise AuvrrtError("libauvrrt: %s (status %d)" % (lib().auvrrt_last_error().decode(), rc))

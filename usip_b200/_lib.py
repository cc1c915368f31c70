"""ctypes binding of libusip_b200.so (include/usip_b200.h).  There is NO fallback: if the library is
missing or a symbol is absent, importing / calling raises."""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libusip_b200.so")

c_int = ctypes.c_int
c_i64 = ctypes.c_int64
c_f32 = ctypes.c_float
c_ptr = ctypes.c_void_p


class LayerDesc(ctypes.Structure):
    """Mirror of `usip_layer_desc` (include/usip_b200.h)."""
    _fields_ = [
        ("X", c_ptr), ("ldx", ctypes.c_int32),
        ("P", ctypes.c_int32), ("Cin", ctypes.c_int32), ("Cout", ctypes.c_int32),
        ("W", c_ptr), ("ldw", ctypes.c_int32),
        ("w_transposed", ctypes.c_int32),
        ("bias", c_ptr),
        ("in_scale", c_ptr), ("in_shift", c_ptr),
        ("in_relu", ctypes.c_int32),
        ("addend", c_ptr), ("ld_add", ctypes.c_int32),
        ("add_index", c_ptr),
        ("add_group", ctypes.c_int32),
        ("Y", c_ptr), ("ldy", ctypes.c_int32),
        ("stat_partial", c_ptr),
        ("gmax", c_ptr), ("gmin", c_ptr),
        ("garg_max", c_ptr), ("garg_min", c_ptr),
        ("group", ctypes.c_int32),
        ("precision", ctypes.c_int32),
        ("tc_workspace", c_ptr),
        ("tc_workspace_bytes", ctypes.c_int64),
        ("tc_weights_packed", ctypes.c_int32),
        ("debug_flags", ctypes.c_int32),
        ("debug_clocks", ctypes.c_void_p),
    ]


# name -> (restype, argtypes); this table is also what tests use to check that every symbol declared in
# include/usip_b200.h is exported.
SIGNATURES = {
    "usip_abi_version": (c_int, []),
    "usip_last_error": (ctypes.c_char_p, []),
    "usip_index_max_f32": (c_int, [c_ptr, c_ptr, c_ptr, c_ptr, c_int, c_int, c_int, c_int, c_ptr]),
    "usip_ball_query_dist_f32": (c_int, [c_ptr, c_f32, c_ptr, c_int, c_int, c_int, c_int, c_ptr]),
    "usip_ball_group_f32": (c_int, [c_ptr, c_ptr, c_ptr, c_f32, c_ptr, c_ptr, c_ptr, c_int, c_ptr, c_i64,
                                    c_int, c_int, c_int, c_int, c_int, c_ptr]),
    "usip_ball_group_scratch_bytes": (c_i64, [c_int, c_int, c_int, c_int, c_int]),
    "usip_ball_group_scratch_init": (c_int, [c_ptr, c_i64, c_int, c_ptr]),
    "usip_knn_group_f32": (c_int, [c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_int, c_int, c_int, c_int, c_int, c_int, c_ptr]),
    "usip_knn_gather_f32": (c_int, [c_ptr, c_ptr, c_ptr, c_int, c_int, c_int, c_int, c_int, c_ptr]),
    "usip_som_assign_f32": (c_int, [c_ptr, c_ptr, c_ptr, c_ptr, c_int, c_int, c_int, c_ptr]),
    "usip_cluster_sort": (c_int, [c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_int, c_int, c_int, c_ptr]),
    "usip_cluster_mean_decenter": (c_int, [c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_int,
                                           c_int, c_int, c_int, c_int, c_ptr]),
    "usip_layer_fwd": (c_int, [ctypes.POINTER(LayerDesc), c_ptr]),
    "usip_layer_tc_pack_many": (c_int, [ctypes.POINTER(LayerDesc), c_int, c_ptr]),
    "usip_layer_tile_rows": (c_int, []),
    "usip_fps_f32": (c_int, [c_ptr, c_ptr, c_ptr, c_ptr, c_int, c_int, c_int, c_ptr]),
    "usip_nms_f32": (c_int, [c_ptr, c_ptr, ctypes.c_float, c_ptr, c_ptr, c_int, c_int, c_ptr]),
    "usip_l2norm_bwd": (c_int, [c_ptr, c_ptr, c_int, c_ptr, c_int, c_int, c_int, c_int, c_ptr]),
    "usip_desc_triplet_bwd": (c_int, [c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, ctypes.c_float, ctypes.c_float,
                                      c_ptr, c_ptr, c_ptr, c_ptr, c_int, c_int, c_int, c_int, c_int, c_ptr]),
    "usip_point_on_surface": (c_int, [c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_int, c_int, c_int, c_int, c_ptr]),
    "usip_layer_stat_slots": (c_int, [ctypes.POINTER(LayerDesc)]),
    "usip_layer_tc_workspace_bytes": (c_i64, [c_int, c_int]),
    "usip_bn_finalize": (c_int, [c_ptr, c_int, c_i64, c_int, c_ptr, c_ptr, c_f32, c_f32, c_ptr, c_ptr,
                                 c_ptr, c_ptr, c_ptr, c_ptr, c_ptr]),
    "usip_bn_eval_affine": (c_int, [c_ptr, c_ptr, c_ptr, c_ptr, c_f32, c_int, c_ptr, c_ptr, c_ptr]),
    "usip_segmax": (c_int, [c_ptr, c_int, c_ptr, c_ptr, c_ptr, c_int, c_ptr, c_int, c_int, c_int, c_int, c_ptr]),
    "usip_knn_nodes": (c_int, [c_ptr, c_ptr, c_int, c_int, c_int, c_ptr]),
    "usip_knn_combine": (c_int, [c_ptr, c_int, c_ptr, c_ptr, c_ptr, c_int, c_ptr, c_ptr, c_int, c_ptr,
                                 c_int, c_int, c_int, c_int, c_ptr]),
    "usip_group_select": (c_int, [c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_int, c_int, c_int, c_ptr]),
    "usip_head_finalize": (c_int, [c_ptr, c_int, c_ptr, c_f32, c_ptr, c_ptr, c_int, c_int, c_ptr]),
    "usip_l2norm_to_bcm": (c_int, [c_ptr, c_int, c_ptr, c_ptr, c_int, c_int, c_int, c_ptr]),
    "usip_pairwise_min_f32": (c_int, [c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_int, c_int, c_int, c_ptr]),
    "usip_pairwise_min_grid_scratch_bytes": (ctypes.c_size_t, [c_int, c_int]),
    "usip_som_assign_grid_scratch_bytes": (ctypes.c_size_t, [c_int, c_int]),
    "usip_som_assign_grid_f32": (c_int, [c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, ctypes.c_size_t, c_int, c_int, c_int, c_ptr]),
    "usip_pairwise_min_grid_f32": (c_int, [c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, ctypes.c_size_t, c_int, c_int, c_int, c_ptr]),
    "usip_chamfer_prob_reduce": (c_int, [c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_int, c_int, c_int, c_ptr]),
    "usip_transform_points": (c_int, [c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_int, c_int, c_ptr]),
    "usip_mean_scale": (c_int, [c_ptr, c_i64, c_f32, c_ptr, c_ptr]),
    "usip_desc_pairmin_f32": (c_int, [c_ptr, c_ptr, c_ptr, c_ptr, c_int, c_int, c_int, c_int, c_ptr]),
    "usip_desc_triplet": (c_int, [c_ptr, c_ptr, c_ptr, c_f32, c_f32, c_ptr, c_ptr, c_int, c_int, c_ptr]),
    "usip_pairwise_min_bwd": (c_int, [c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_f32, c_ptr, c_ptr, c_int, c_int, c_int, c_ptr]),
    "usip_chamfer_prob_bwd": (c_int, [c_ptr] * 13 + [c_int, c_int, c_int, c_ptr]),
    "usip_transform_points_bwd": (c_int, [c_ptr, c_ptr, c_ptr, c_ptr, c_int, c_int, c_ptr]),
    "usip_bn_bwd_reduce": (c_int, [c_ptr, c_int, c_ptr, c_int, c_ptr, c_ptr, c_ptr, c_ptr, c_int, c_ptr, c_int, c_int, c_ptr]),
    "usip_bn_bwd_finalize": (c_int, [c_ptr, c_int, c_i64, c_int, c_ptr, c_ptr, c_ptr, c_ptr, c_int, c_ptr]),
    "usip_bn_bwd_apply": (c_int, [c_ptr, c_int, c_ptr, c_int, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_int, c_ptr,
                                  c_int, c_int, c_int, c_ptr]),
    "usip_groupmax_bwd_select": (c_int, [c_ptr, c_int, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr,
                                         c_ptr, c_int, c_int, c_ptr]),
    "usip_groupmax_scatter_add": (c_int, [c_ptr, c_int, c_ptr, c_ptr, c_int, c_int, c_int, c_ptr]),
    "usip_groupmax_bwd_apply": (c_int, [c_ptr, c_int, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_int,
                                        c_int, c_int, c_int, c_ptr]),
    "usip_group_sum": (c_int, [c_ptr, c_int, c_ptr, c_int, c_int, c_int, c_int, c_ptr]),
    "usip_seg_sum": (c_int, [c_ptr, c_int, c_ptr, c_ptr, c_int, c_int, c_int, c_int, c_int, c_ptr]),
    "usip_unpool_scatter": (c_int, [c_ptr, c_int, c_ptr, c_int, c_ptr, c_int, c_int, c_int, c_ptr]),
    "usip_knn_combine_bwd": (c_int, [c_ptr, c_int, c_ptr, c_ptr, c_ptr, c_int, c_ptr, c_int, c_int, c_int, c_int, c_int, c_ptr]),
    "usip_colsum": (c_int, [c_ptr, c_int, c_ptr, c_int, c_int, c_ptr]),
    "usip_head_bwd": (c_int, [c_ptr, c_ptr, c_ptr, c_int, c_ptr, c_int, c_int, c_ptr]),
    "usip_adam_step": (c_int, [c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_f32, c_f32, c_f32, c_f32, c_i64, c_ptr]),
    "usip_wgrad": (c_int, [c_ptr, c_int, c_ptr, c_int, c_ptr, c_ptr, c_int, c_ptr, c_int, c_int, c_int, c_int, c_int, c_ptr]),
    "usip_desc_knn_f32": (c_int, [c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_int, c_int, c_int, c_int, c_int, c_ptr]),
    "usip_corr_build": (c_int, [c_ptr, c_int, c_ptr, c_int, c_ptr, c_ptr, c_ptr, c_ptr, c_int, c_int, c_int, c_int, c_ptr]),
    "usip_ransac_rt_scratch_bytes": (ctypes.c_size_t, [c_int, c_int]),
    "usip_ransac_rt": (c_int, [c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, ctypes.c_double, c_int, ctypes.c_double, ctypes.c_uint64,
                               c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, ctypes.c_size_t, c_int, c_int, c_int, c_int,
                               c_ptr]),
}

_lib = None


class UsipB200Error(RuntimeError):
    pass


def load():
    """Load the C-ABI library (once).  Raises if it has not been built -- never falls back."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise UsipB200Error(
            "libusip_b200.so not found at %s -- build it with `python -m usip_b200.build` "
            "(or __graft_entry__.build()); there is no CPU / PyTorch fallback" % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)        # AttributeError if the symbol is missing: fail loudly
        fn.restype = res
        fn.argtypes = args
    ver = lib.usip_abi_version()
    if ver != 1:
        raise UsipB200Error("ABI version mismatch: library %d, binding 1" % ver)
    _lib = lib
    return lib


# Generation of the weights as seen by the packed tensor-core tile cache (engine._tc_workspace): bumped by every update
# that writes parameters behind autograd's back (usip_adam_step, CUDA-graph replays of the train step).
WEIGHT_GEN = [0]

# kernels launched per C-ABI call (for bench.py's gpu_launches claim); default 1
KERNELS_PER_CALL = {"usip_cluster_sort": 3, "usip_pairwise_min_f32": 3, "usip_pairwise_min_grid_f32": 3, "usip_som_assign_grid_f32": 2, "usip_layer_fwd_tc": 2, "usip_ball_group_f32": 2,
                    "usip_ransac_rt": 12}
LAUNCHES = [0]


def check(code, what):
    LAUNCHES[0] += KERNELS_PER_CALL.get(what, 1)
    if code != 0:
        lib = load()
        msg = lib.usip_last_error().decode()
        raise UsipB200Error("%s failed: code %d (%s)" % (what, code, msg))

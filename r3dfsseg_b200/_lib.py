"""ctypes binding of libr3dfs.so (C ABI in include/r3dfs.h).

There is no fallback: if the shared library is missing, `lib()` raises with the build command.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# R3DFS_LIB selects another build of the SAME library (the measurement build libr3dfs_ab.so, which
# has the A/B switches of DESIGN.md §6 compiled in); it is read here, never by the library.
LIB_PATH = os.environ.get("R3DFS_LIB") or os.path.join(_HERE, "libr3dfs.so")
AB_LIB_PATH = os.path.join(_HERE, "libr3dfs_ab.so")

c_f32p = C.c_void_p
c_i32p = C.c_void_p
c_i64p = C.c_void_p
c_u8p = C.c_void_p


class Weights(C.Structure):
    """r3dfs_weights_t"""
    _fields_ = [
        ("in_dim", C.c_int32), ("dgcnn_k", C.c_int32),
        ("ec_w1", C.c_void_p * 3), ("ec_s1", C.c_void_p * 3), ("ec_t1", C.c_void_p * 3),
        ("ec_w2", C.c_void_p * 3), ("ec_s2", C.c_void_p * 3), ("ec_t2", C.c_void_p * 3),
        ("mlp_w", C.c_void_p * 2), ("mlp_s", C.c_void_p * 2), ("mlp_t", C.c_void_p * 2),
        ("bl_w", C.c_void_p * 2), ("bl_s", C.c_void_p * 2), ("bl_t", C.c_void_p * 2),
        ("att_wqkv", C.c_void_p),
    ]


class EpisodeCfg(C.Structure):
    """r3dfs_episode_cfg_t"""
    _fields_ = [
        ("n_way", C.c_int32), ("k_shot", C.c_int32), ("n_query", C.c_int32),
        ("n_points", C.c_int32), ("n_subprototypes", C.c_int32), ("k_connect", C.c_int32),
        ("sigma", C.c_float), ("alpha", C.c_float), ("mdns", C.c_int32),
        ("cg_max_iter", C.c_int32), ("cg_tol", C.c_float),
    ]


class EpisodeDiag(C.Structure):
    """r3dfs_episode_diag_t"""
    _fields_ = [("proto_count", C.c_void_p), ("clean_flag", C.c_void_p),
                ("cg_iters", C.c_void_p), ("cg_resid", C.c_void_p),
                ("h_stage_events", C.POINTER(C.c_void_p))]


class TrainExport(C.Structure):
    """r3dfs_train_export_t"""
    _fields_ = [("knn_support", C.c_void_p * 3), ("knn_query", C.c_void_p * 3),
                ("set_off", C.c_void_p), ("set_n", C.c_void_p), ("proto_cnt", C.c_void_p),
                ("assign", C.c_void_p), ("cloud_fg_off", C.c_void_p), ("fg_cnt", C.c_void_p),
                ("cproto_cnt", C.c_void_p), ("cassign", C.c_void_p), ("nbr", C.c_void_p),
                ("valid", C.c_void_p)]


STAGES = ["begin", "input", "knn0", "pq0", "edge0", "knn1", "pq1", "edge1", "knn2", "pq2", "edge2",
          "mlp", "base", "qkv", "att", "mdns", "sets", "fps", "proto", "dist", "select", "sim",
          "sym", "cg", "head"]


i64, i32, f32, vp, sz = C.c_int64, C.c_int, C.c_float, C.c_void_p, C.c_size_t

# name -> (restype, argtypes); mirrors include/r3dfs.h one to one
SIGNATURES = {
    "r3dfs_version": (C.c_int, []),
    "r3dfs_strerror": (C.c_char_p, [C.c_int]),
    "r3dfs_launch_count": (C.c_longlong, []),
    "r3dfs_knn_workspace": (sz, [i64, i64, i64, i32]),
    "r3dfs_knn": (C.c_int, [vp, i64, i64, i64, i64, i64, i64, i32, vp, vp, sz, vp]),
    "r3dfs_knn_ex": (C.c_int, [vp, i64, i64, i64, i64, i64, i64, i32, vp, i32, vp, sz, vp]),
    "r3dfs_edge_feature_workspace": (sz, [i64, i64, i64]),
    "r3dfs_edge_feature": (C.c_int, [vp, i64, i64, i64, i64, i64, i64, vp, i32, vp, vp, sz, vp]),
    "r3dfs_linear": (C.c_int, [vp, i64, vp, vp, vp, i32, i64, i64, i64, vp, i64, vp]),
    "r3dfs_linear_ex": (C.c_int, [vp, i64, vp, vp, vp, i32, i64, i64, i64, vp, i64, i32, vp]),
    "r3dfs_edgeconv_workspace": (sz, [i64, i64, i64, i32]),
    "r3dfs_edgeconv": (C.c_int, [vp, i64, i64, i64, i64, i64, i64, i32, vp, vp, vp, vp, vp, vp, vp,
                                 vp, vp, sz, vp]),
    "r3dfs_features_workspace": (sz, [i64, i64]),
    "r3dfs_features": (C.c_int, [C.POINTER(Weights), vp, i64, i64, i64, i64, i64, vp, vp, vp, sz,
                                 vp]),
    "r3dfs_attention_workspace": (sz, [i64, i64]),
    "r3dfs_attention": (C.c_int, [vp, i64, i64, i64, vp, vp, vp, sz, vp]),
    "r3dfs_fps": (C.c_int, [vp, i64, vp, vp, i32, i64, i32, vp, vp]),
    "r3dfs_fps_workspace": (sz, [i64]),
    "r3dfs_fps_ex": (C.c_int, [vp, i64, vp, vp, i32, i64, i64, i32, i32, vp, vp, sz, vp]),
    "r3dfs_mdns_workspace": (sz, [i32, i32, i32]),
    "r3dfs_mdns": (C.c_int, [vp, i64, i64, i64, i64, vp, vp, i32, i32, i32, i64, vp, vp, vp, vp, vp,
                             vp, vp, vp, sz, vp]),
    "r3dfs_multi_prototypes_workspace": (sz, [i64, i32, i32]),
    "r3dfs_multi_prototypes": (C.c_int, [vp, i64, vp, vp, i32, i64, i32, vp, vp, vp, vp, vp, sz,
                                         vp]),
    "r3dfs_affinity_workspace": (sz, [i32, i64, i64, i32]),
    "r3dfs_affinity_knn": (C.c_int, [vp, vp, i32, i64, i64, i32, f32, vp, vp, vp, sz, vp]),
    "r3dfs_label_propagate_workspace": (sz, [i32, i64, i32, i32]),
    "r3dfs_label_propagate": (C.c_int, [vp, vp, vp, i32, i64, i32, vp, i32, f32, f32, i32, vp, vp,
                                        vp, vp, sz, vp]),
    "r3dfs_lp_cholesky_workspace": (sz, [i32, i64, i32, i32]),
    "r3dfs_lp_cholesky": (C.c_int, [vp, vp, vp, i32, i64, i32, vp, i32, f32, vp, vp, vp, sz, vp]),
    "r3dfs_mpti_workspace": (sz, [C.POINTER(EpisodeCfg), i32]),
    "r3dfs_mpti_forward": (C.c_int, [C.POINTER(EpisodeCfg), C.POINTER(Weights), i32,
                                     vp, i64, i64, i64, i64, vp,
                                     vp, i64, i64, i64, i64, vp,
                                     vp, vp, vp, C.POINTER(EpisodeDiag), vp, sz, vp]),
    "r3dfs_mpti_forward_features": (C.c_int, [C.POINTER(EpisodeCfg), i32, vp, i64, i64, i64, i64, vp,
                                              vp, vp, vp, vp, vp, vp, C.POINTER(EpisodeDiag), vp,
                                              sz, vp]),
    "r3dfs_mpti_support_workspace": (sz, [C.POINTER(EpisodeCfg), i32]),
    "r3dfs_mpti_support": (C.c_int, [C.POINTER(EpisodeCfg), C.POINTER(Weights), i32,
                                     vp, i64, i64, i64, i64, vp, vp, vp,
                                     C.POINTER(EpisodeDiag), vp, sz, vp]),
    "r3dfs_mpti_query_workspace": (sz, [C.POINTER(EpisodeCfg), i32]),
    "r3dfs_mpti_query": (C.c_int, [C.POINTER(EpisodeCfg), C.POINTER(Weights), i32,
                                   vp, i64, vp, i64,
                                   vp, i64, i64, i64, i64, vp,
                                   vp, vp, vp, C.POINTER(EpisodeDiag), vp, sz, vp]),
    "r3dfs_scene_workspace": (sz, [i64, i32]),
    "r3dfs_scene_plan": (C.c_int, [vp, i64, i64, i64, f32, i32, C.c_uint32, i32, vp, vp, sz, vp]),
    "r3dfs_scene_chunks": (C.c_int, [vp, i64, i64, i64, i32, i32, i64, vp, vp, vp, sz, vp]),
    "r3dfs_scene_merge": (C.c_int, [vp, i64, i32, i32, i64, i32, vp, vp, vp, vp, sz, vp]),
    "r3dfs_scene_support_workspace": (sz, [i32, i32]),
    "r3dfs_scene_support": (C.c_int, [vp, i64, i64, i64, vp, C.POINTER(C.c_int32), i32, i32, i32,
                                      C.c_double, C.c_uint32, i32, i32, vp, vp, vp, vp, vp, vp, sz,
                                      vp, sz, vp]),
    "r3dfs_scene_index": (C.c_int, [vp, i64, i32, C.POINTER(C.c_int32), i32, C.c_int32, i64, i64,
                                    i64, i64, i64, vp, vp, vp, vp, vp, C.POINTER(i64), vp, sz, vp]),
    "r3dfs_scene_index_workspace": (sz, [i64, i32]),
    "r3dfs_scene_index_classes": (C.c_int, [vp, vp, i64, i32, i32, C.c_double, vp, vp,
                                            C.POINTER(C.c_int32), vp, sz, vp]),
    "r3dfs_scene_episodes_workspace": (sz, [i32, i32, i32, i32, i32]),
    "r3dfs_scene_episodes": (C.c_int, [vp, i64, i64, vp, vp, vp, vp, vp, C.POINTER(C.c_int32),
                                       C.POINTER(C.c_int32), i32, C.POINTER(C.c_int32),
                                       C.POINTER(C.c_int32), i32, C.POINTER(C.c_int32), i32, i32,
                                       i32, i32, i32, C.c_uint32, i64, i64, vp, vp, vp, vp, vp, vp,
                                       vp, vp, vp, vp, vp, sz, vp]),
    "r3dfs_confusion_accumulate": (C.c_int, [vp, vp, vp, i32, i32, i64, i32, vp, vp]),
    "r3dfs_protonet_forward": (C.c_int, [C.POINTER(EpisodeCfg), C.POINTER(Weights), i32,
                                         vp, i64, i64, i64, i64, vp,
                                         vp, i64, i64, i64, i64, vp,
                                         i32, vp, vp, vp, vp, vp, sz, vp]),
    # meta-training step
    "r3dfs_train_param_layout": (i64, [i32, C.POINTER(i64)]),
    "r3dfs_train_bn_layout": (None, [C.POINTER(i64)]),
    "r3dfs_mpti_train_workspace": (sz, [C.POINTER(EpisodeCfg), i32, i32]),
    "r3dfs_mpti_train_forward": (C.c_int, [C.POINTER(EpisodeCfg), i32, i32, vp, vp,
                                           vp, i64, i64, i64, vp, vp,
                                           vp, i64, i64, i64, vp,
                                           f32, vp, vp, vp, vp, vp, vp, sz, vp]),
    "r3dfs_mpti_train_backward": (C.c_int, [C.POINTER(EpisodeCfg), i32, i32, vp, vp, vp, vp,
                                            f32, vp, vp, f32, f32, vp, vp, sz, vp]),
    "r3dfs_mpti_train_clean_ratio": (C.c_int, [C.POINTER(EpisodeCfg), i32, i32, vp, vp, vp, vp, sz,
                                               vp]),
    "r3dfs_mpti_train_export": (C.c_int, [C.POINTER(EpisodeCfg), i32, i32, C.POINTER(TrainExport), vp,
                                          sz, vp]),
    "r3dfs_adam_step": (C.c_int, [vp, vp, vp, vp, i64, i64, f32, f32, f32, f32, f32, i64, f32, vp]),
    "r3dfs_dropout_mask": (C.c_int, [C.c_uint64, i64, f32, vp, vp]),
    "r3dfs_sgemm": (C.c_int, [vp, i64, i64, vp, i64, i64, vp, i64, i64, i64, i64, f32, f32, vp, sz,
                              vp]),
}

N_PARAMS = 37
N_BN = 10

_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        if not os.path.isfile(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `make -C r3dfsseg_b200/csrc` "
                "(or `python -c 'import __graft_entry__ as g; g.build()'`). "
                "r3dfsseg_b200 has no CPU or PyTorch fallback.")
        handle = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)
            fn.restype = res
            fn.argtypes = args
        _lib = handle
    return _lib


class R3dfsError(RuntimeError):
    pass


def check(code: int, what: str) -> None:
    if code != 0:
        msg = lib().r3dfs_strerror(code).decode()
        raise R3dfsError(f"{what} failed with code {code}: {msg}")

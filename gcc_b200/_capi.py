"""ctypes mirror of include/gccb200.h (structs + prototypes).

``bind(cdll)`` attaches argtypes/restype to a loaded library handle.  The product
loader (gcc_b200/_lib.py) applies it to libgccb200.so; nothing here loads a
library by itself.
"""
import ctypes as C

GCCB_OK, GCCB_ERR_BADARG, GCCB_ERR_CAPACITY, GCCB_ERR_ARCH, GCCB_ERR_CUDA = 0, -1, -2, -3, -4
FLAG_NODE_OVERFLOW, FLAG_EDGE_OVERFLOW, FLAG_ZERO_DEGREE, FLAG_EIG_NOCONV, FLAG_EIG_TOOBIG = 1, 2, 4, 8, 16
FLAG_NAMES = {1: "node capacity overflow", 2: "edge capacity overflow",
              4: "walk reached a zero-degree vertex", 8: "eigensolver did not converge",
              16: "ego-net too large for the eigensolver"}

p = C.c_void_p


class Graph(C.Structure):
    _fields_ = [("indptr", p), ("indices", p), ("n_nodes", C.c_int64),
                ("budget_table", p), ("budget_table_len", C.c_int32), ("max_budget", C.c_int32),
                ("restart_thresh", C.c_uint32), ("_pad", C.c_uint32), ("key", C.c_uint64)]


class Batch(C.Structure):
    _fields_ = [("batch", C.c_int32), ("node_cap", C.c_int32), ("edge_cap", C.c_int32),
                ("_pad", C.c_int32), ("node_off", p), ("edge_off", p), ("indptr", p),
                ("indices", p), ("sub_deg", p), ("graph_id", p), ("orig_id", p),
                ("counters", p), ("flags", p)]


class GinCfg(C.Structure):
    _fields_ = [("num_layers", C.c_int32), ("hidden", C.c_int32), ("pos_dim", C.c_int32),
                ("deg_dim", C.c_int32), ("max_degree", C.c_int32), ("norm", C.c_int32),
                ("bn_eps", C.c_float), ("bn_momentum", C.c_float), ("norm_eps", C.c_float),
                ("dropout_p", C.c_float), ("tensor_cores", C.c_int32), ("_pad", C.c_int32)]


class GinLayout(C.Structure):
    _fields_ = [(n, C.c_int64 * 8) for n in
                ("w1", "b1", "bn1_w", "bn1_b", "w2", "b2", "bna_w", "bna_b", "bnb_w", "bnb_b",
                 "wp", "bp")] + [("emb", C.c_int64), ("total", C.c_int64), ("run_total", C.c_int64)]


_PROTOS = {
    "gccb_version": (C.c_int, []),
    "gccb_arch": (C.c_int, []),
    "gccb_last_error": (C.c_char_p, []),
    "gccb_launch_count": (C.c_ulonglong, []),
    "gccb_draw_seeds": (C.c_int, [p, C.c_int64, C.c_uint64, C.c_int64, C.c_int32, p, p, p]),
    "gccb_sample_batch_workspace": (C.c_size_t, [C.c_int32, C.c_int32, C.c_int32]),
    "gccb_sample_batch": (C.c_int, [C.POINTER(Graph), p, p, C.POINTER(Batch), p, C.c_size_t, p]),
    "gccb_posenc_workspace": (C.c_size_t, [C.c_int32, C.c_int32]),
    "gccb_posenc": (C.c_int, [C.POINTER(Batch), C.c_int32, C.c_int32, p, p, p, C.c_size_t, p]),
    "gccb_gin_param_layout": (C.c_int, [C.POINTER(GinCfg), C.POINTER(GinLayout)]),
    "gccb_gin_acts_bytes": (C.c_size_t, [C.POINTER(GinCfg), C.c_int32, C.c_int32]),
    "gccb_gin_forward": (C.c_int, [C.POINTER(GinCfg), C.POINTER(Batch), C.c_int32, p, p, p, p,
                                   C.c_int32, C.c_uint64, C.c_uint64, C.c_int32, p, C.c_size_t,
                                   p, p, p]),
    "gccb_gin_backward_workspace": (C.c_size_t, [C.POINTER(GinCfg), C.c_int32, C.c_int32]),
    "gccb_gin_backward": (C.c_int, [C.POINTER(GinCfg), C.POINTER(Batch), C.c_int32, p, p, p, p,
                                    C.c_uint64, C.c_uint64, C.c_int32, p, C.c_size_t, p]),
    "gccb_moco_logits": (C.c_int, [p, p, p, C.c_int32, C.c_int32, C.c_int32, C.c_float, p, p]),
    "gccb_moco_logits_backward": (C.c_int, [p, p, p, C.c_int32, C.c_int32, C.c_int32, C.c_float,
                                            p, p]),
    "gccb_nce_loss": (C.c_int, [p, C.c_int32, C.c_int32, C.c_int32, p, p, p]),
    "gccb_infonce_workspace": (C.c_size_t, [C.c_int32, C.c_int32, C.c_int32]),
    "gccb_infonce_fused": (C.c_int, [p, p, p, C.c_int32, C.c_int32, C.c_int32, C.c_float, p, p,
                                     p, C.c_size_t, p]),
    "gccb_moco_enqueue": (C.c_int, [p, p, C.c_int32, C.c_int32, C.c_int32, p, C.c_int32, C.c_int64, p, C.c_int32, p]),
    "gccb_e2e_nce": (C.c_int, [p, p, C.c_int32, C.c_int32, C.c_float, p, p, p, p, C.c_size_t, p]),
    "gccb_clip_adam_ema": (C.c_int, [p, p, p, p, p, C.c_int64, C.c_int64, p, C.c_float,
                                     C.c_float, C.c_float, C.c_float, C.c_float, C.c_float,
                                     C.c_float, p, p, p, C.c_int32, p]),
    "gccb_sum_ranks": (C.c_int, [p, C.c_int32, C.c_int64, C.c_int64, p, C.c_int64, p, p]),
    "gccb_tc_gemm_bf16": (C.c_int, [p, p, C.c_int32, C.c_int32, C.c_int32, p, p, C.c_float, p, p, C.c_int32, p,
                                    C.c_int32, p, p]),
    "gccb_cast_bf16": (C.c_int, [p, C.c_int32, C.c_int32, C.c_int32, p, C.c_int32, C.c_int32, C.c_int32, p, p]),
    "gccb_logreg_ovr_workspace": (C.c_size_t, [C.c_int32, C.c_int32, C.c_int32, C.c_int32]),
    "gccb_logreg_ovr": (C.c_int, [p, p, p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_double, C.c_int32,
                                  C.c_double, p, p, p, p, p, C.c_size_t, p]),
    "gccb_svc_ovo_workspace": (C.c_size_t, [C.c_int32, C.c_int32, C.c_int32]),
    "gccb_svc_ovo": (C.c_int, [p, p, p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_double, C.c_double,
                               C.c_int64, p, p, p, p, p, p, p, p, C.c_size_t, p]),
    "gccb_sim_rank_workspace": (C.c_size_t, [C.c_int32, C.c_int32]),
    "gccb_sim_rank": (C.c_int, [p, p, C.c_int32, p, p, C.c_int32, p, p, C.c_size_t, p]),
}

SYMBOLS = tuple(_PROTOS)


def bind(lib, require_all=True):
    missing = []
    for name, (res, args) in _PROTOS.items():
        try:
            fn = getattr(lib, name)
        except AttributeError:
            missing.append(name)
            continue
        fn.restype = res
        fn.argtypes = args
    if missing and require_all:
        raise RuntimeError("libgccb200 is missing symbols: %s" % ", ".join(missing))
    return lib

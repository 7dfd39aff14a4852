"""ctypes binding of librnnlogic_b200.so (include/rnnlogic_b200.h).

The shared library is built in-tree by ``__graft_entry__.build()`` (nvcc, sm_100a).  There is no
CPU fallback: importing this module without the library, or calling into it without a CUDA
device, raises."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(_HERE)
LIB_PATH = os.environ.get("RNNLOGIC_B200_LIB") or os.path.join(_HERE, "lib", "librnnlogic_b200.so")   # env override: A/B builds
SOURCES = [os.path.join(_HERE, "csrc", f) for f in ("rl_kernels.cu", "rl_cells.cu", "rl_plus.cu", "rl_rotate.cu", "rl_tail_tc.cu", "rl_pna.cu", "rl_rnn.cu", "rl_miner.cu")]
HEADER = os.path.join(ROOT, "include", "rnnlogic_b200.h")

LANES = 32
vp = C.c_void_p          # every device pointer crosses the boundary as a plain address


class RlGraph(C.Structure):
    _fields_ = [("num_entities", C.c_int32), ("num_relations", C.c_int32), ("rank_words", C.c_int32),
                ("total_rows", C.c_int32), ("num_edges", C.c_int32),
                ("dst_ptr", vp), ("row_dst", vp), ("row_start", vp), ("edge_src", vp), ("rank_tab", vp),
                ("ord_ptr", vp), ("ord_h", vp), ("ord_t", vp),
                ("fsrc_ptr", vp), ("frow_start", vp), ("fedge_dstrow", vp), ("srank_tab", vp)]


class RlRules(C.Structure):
    _fields_ = [("num_nodes", C.c_int32), ("num_rules", C.c_int32), ("max_len", C.c_int32),
                ("num_chunks", C.c_int32), ("num_terms", C.c_int32), ("num_zero_rules", C.c_int32),
                ("node_rel", vp), ("node_row_off", vp), ("head_node_ptr", vp),
                ("lvl_ptr", vp), ("chunk_node", vp), ("chunk_row0", vp), ("zr_ptr", vp), ("zr_rule", vp),
                ("node_chunk0", vp), ("node_rec", vp), ("node_prow_off", vp),
                ("lvl_sym_ptr", vp), ("sym_node", vp), ("sym_w0", vp), ("node_term_ptr", vp), ("node_term_rule", vp),
                ("node_pair_off", vp), ("pair_ptr", vp), ("pair_ent", vp)]


class RlSlots(C.Structure):
    _fields_ = [("num_slots", C.c_int32), ("slot_head", vp), ("lane_h", vp), ("lane_t", vp),
                ("lane_eh", vp), ("lane_et", vp), ("arena_off", vp), ("nz_off", vp), ("mask_off", vp)]


class RlFrontier(C.Structure):
    _fields_ = [("count_bits", C.c_int32), ("arena", vp), ("row_mask", vp), ("node_cnt", vp),
                ("overflow", vp), ("items", vp), ("items_sorted", vp), ("item_off", vp),
                ("item_cnt", vp), ("bucket_cnt", vp), ("bucket_off", vp),
                ("item_mask", vp), ("item_mask_sorted", vp), ("nzmask", vp)]


class RlCells(C.Structure):
    _fields_ = [("cap", C.c_int32), ("counters", vp), ("nzmask", vp), ("cand_off", vp), ("cell_key", vp),
                ("cell_ent", vp), ("slot_ncell", vp), ("qmax", vp), ("qsum", vp)]


class RlPna(C.Structure):
    _fields_ = [("s1", vp), ("s2", vp), ("deg", vp), ("mnk", vp), ("mxk", vp)]


class RlAnswers(C.Structure):
    _fields_ = [("num_keys", C.c_int64), ("keys", vp), ("ptr", vp), ("ent", vp)]


def nvcc_command(out=LIB_PATH):
    srcs = [s for s in SOURCES if os.path.exists(s)]
    return ["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
            "-shared", "-Xcompiler", "-fPIC", "-I", os.path.join(ROOT, "include"), "-o", out] + srcs


def build(force: bool = False) -> str:
    """Compile csrc/*.cu for sm_100a into rnnlogic_b200/lib/ (cross-compiles without a GPU)."""
    os.makedirs(os.path.dirname(LIB_PATH), exist_ok=True)
    deps = [s for s in SOURCES if os.path.exists(s)] + [HEADER, os.path.join(_HERE, "csrc", "rl_device.cuh"), os.path.join(_HERE, "csrc", "rl_umma.cuh")]
    stale = force or not os.path.exists(LIB_PATH) or any(
        os.path.getmtime(d) > os.path.getmtime(LIB_PATH) for d in deps)
    if stale:
        subprocess.check_call(nvcc_command())
    return LIB_PATH


HOST_LIB_PATH = os.path.join(_HERE, "lib", "librnnlogic_b200_host.so")
HOST_SOURCE = os.path.join(_HERE, "csrc_host", "kg_loader.cpp")


def build_host(force: bool = False) -> str:
    """g++-compile the host-only helpers (dataset loader) into rnnlogic_b200/lib/."""
    os.makedirs(os.path.dirname(HOST_LIB_PATH), exist_ok=True)
    if force or not os.path.exists(HOST_LIB_PATH) or os.path.getmtime(HOST_SOURCE) > os.path.getmtime(HOST_LIB_PATH):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-o", HOST_LIB_PATH, HOST_SOURCE])
    return HOST_LIB_PATH


_host = None


def host_lib():
    """Host-only native helpers (no CUDA): built on demand, g++ is part of the image."""
    global _host
    if _host is None:
        L = C.CDLL(build_host())
        L.rl_kg_load.restype = C.c_void_p
        L.rl_kg_load.argtypes = [C.c_char_p]
        L.rl_kg_load_error.restype = C.c_char_p
        L.rl_kg_num_entities.restype = C.c_int64
        L.rl_kg_num_entities.argtypes = [C.c_void_p]
        L.rl_kg_num_relations.restype = C.c_int64
        L.rl_kg_num_relations.argtypes = [C.c_void_p]
        L.rl_kg_triples.restype = C.POINTER(C.c_int64)
        L.rl_kg_triples.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_int64)]
        L.rl_kg_free.argtypes = [C.c_void_p]
        L.rl_compile_tries.restype = C.c_longlong
        L.rl_compile_tries.argtypes = [C.c_longlong, C.c_longlong] + [C.c_void_p] * 9
        _host = L
    return _host


_lib = None

_PROTOS = {
    "rl_abi_version": (C.c_int, []),
    "rl_last_error": (C.c_char_p, []),
    "rl_device_count": (C.c_int, []),
    "rl_launch_count": (C.c_longlong, []),
    "rl_prepare_slots": (C.c_int, [C.POINTER(RlGraph), C.c_int32, vp, vp, vp, vp, vp, C.c_int32, vp, vp, vp, vp, vp]),
    "rl_expand_level": (C.c_int, [C.POINTER(RlGraph), C.POINTER(RlRules), C.POINTER(RlSlots), C.c_int32,
                                  C.c_int32, C.c_int32, C.POINTER(RlFrontier), C.c_int32, C.c_int32, C.c_int32, C.c_int32, vp]),
    "rl_sort_items": (C.c_int, [C.POINTER(RlGraph), C.POINTER(RlSlots), C.POINTER(RlFrontier), vp]),
    "rl_node_counts_dense": (C.c_int, [C.POINTER(RlGraph), C.POINTER(RlRules), C.POINTER(RlSlots), C.c_int32,
                                       C.c_int32, C.POINTER(RlFrontier), vp, vp]),
    "rl_propagate_dense": (C.c_int, [C.POINTER(RlGraph), C.c_int32, C.c_int32, vp, vp, vp, vp]),
    "rl_predictor_scores": (C.c_int, [C.POINTER(RlGraph), C.POINTER(RlRules), C.POINTER(RlSlots),
                                      C.POINTER(RlFrontier), vp, vp, C.c_int32, vp, vp, vp, vp]),
    "rl_predictor_ce_backward": (C.c_int, [C.POINTER(RlGraph), C.POINTER(RlRules), C.POINTER(RlSlots),
                                           C.POINTER(RlFrontier), C.POINTER(RlAnswers), C.c_float, C.c_int32, vp, vp,
                                           C.c_int32, vp, vp, C.c_int32, vp, vp, vp, vp, vp, vp, vp, vp, vp]),
    "rl_softmax_blocks": (C.c_int, [C.c_int32]),
    "rl_softmax_ce": (C.c_int, [C.POINTER(RlGraph), C.POINTER(RlSlots), C.POINTER(RlAnswers), C.c_float,
                                C.c_int32, vp, vp, C.c_int32, vp, vp, vp, vp, vp, vp, vp, vp]),
    "rl_filtered_rank": (C.c_int, [C.POINTER(RlGraph), C.POINTER(RlSlots), C.POINTER(RlAnswers), C.c_int32,
                                   vp, vp, vp, vp, vp]),
    "rl_filtered_rank_dense": (C.c_int, [C.c_int64, C.c_int64, vp, vp, vp, vp, vp, vp]),
    "rl_rank_metrics": (C.c_int, [C.c_int64, vp, vp, C.c_int32, vp, vp, vp]),
    "rl_plus_mask": (C.c_int, [C.POINTER(RlGraph), C.POINTER(RlRules), C.POINTER(RlSlots), C.POINTER(RlFrontier), vp, vp, vp]),
    "rl_plus_features": (C.c_int, [C.POINTER(RlGraph), C.POINTER(RlRules), C.POINTER(RlSlots), C.POINTER(RlFrontier),
                                   vp, vp, vp, vp, vp, C.c_int32, C.c_int32, vp, vp, vp, vp, vp, vp, vp, vp, vp]),
    "rl_rule_stats": (C.c_int, [C.POINTER(RlGraph), C.POINTER(RlRules), C.POINTER(RlSlots), C.POINTER(RlFrontier),
                                C.c_int32, vp, vp, vp]),
    "rl_plus_scatter": (C.c_int, [C.POINTER(RlGraph), C.POINTER(RlSlots), vp, vp, vp, vp, vp, C.c_int32, vp, vp]),
    "rl_plus_gather": (C.c_int, [C.POINTER(RlGraph), C.POINTER(RlSlots), vp, vp, vp, vp, vp]),
    "rl_plus_backward": (C.c_int, [C.POINTER(RlGraph), C.POINTER(RlRules), C.POINTER(RlSlots), C.POINTER(RlFrontier),
                                   vp, vp, vp, C.c_int32, vp, vp, C.c_int32, vp, vp, vp]),
    "rl_rotate_scores": (C.c_int, [C.POINTER(RlGraph), C.POINTER(RlSlots), C.c_int32, C.c_float, vp, vp, vp, vp, vp]),
    "rl_rotate_backward": (C.c_int, [C.POINTER(RlGraph), C.POINTER(RlSlots), C.c_int32, C.c_float, vp, vp, vp, vp, vp,
                                     vp, vp, vp]),
    "rl_cells_build": (C.c_int, [C.POINTER(RlGraph), C.POINTER(RlRules), C.POINTER(RlSlots), C.POINTER(RlFrontier),
                                 C.POINTER(RlCells), vp]),
    "rl_bias_stats": (C.c_int, [C.c_int32, vp, vp, vp]),
    "rl_predictor_item_scores": (C.c_int, [C.POINTER(RlGraph), C.POINTER(RlRules), C.POINTER(RlSlots),
                                          C.POINTER(RlFrontier), C.POINTER(RlCells), vp, vp, vp]),
    "rl_cells_softmax_ce": (C.c_int, [C.POINTER(RlGraph), C.POINTER(RlSlots), C.POINTER(RlCells), C.POINTER(RlAnswers),
                                      C.c_float, vp, vp, vp, C.c_int32, vp, C.c_float, vp, vp, vp, vp, vp, vp, vp]),
    "rl_plus_item_features": (C.c_int, [C.POINTER(RlGraph), C.POINTER(RlRules), C.POINTER(RlSlots), C.POINTER(RlFrontier),
                                       C.POINTER(RlCells), vp, C.c_int32, vp, vp]),
    "rl_plus_item_backward": (C.c_int, [C.POINTER(RlGraph), C.POINTER(RlRules), C.POINTER(RlSlots), C.POINTER(RlFrontier),
                                       C.POINTER(RlCells), C.c_int32, vp, vp, vp]),
    "rl_predictor_item_backward": (C.c_int, [C.POINTER(RlGraph), C.POINTER(RlRules), C.POINTER(RlSlots),
                                            C.POINTER(RlFrontier), C.POINTER(RlCells), vp, vp, vp]),
    "rl_cells_rank": (C.c_int, [C.POINTER(RlGraph), C.POINTER(RlSlots), C.POINTER(RlCells), C.POINTER(RlAnswers),
                                vp, vp, vp, vp, vp, vp]),
    "rl_cells_add_to_dense": (C.c_int, [C.POINTER(RlGraph), C.POINTER(RlSlots), C.POINTER(RlCells), vp, vp, vp]),
    "rl_cells_gather_dense": (C.c_int, [C.POINTER(RlGraph), C.POINTER(RlSlots), C.POINTER(RlCells), vp, vp, vp]),
    "rl_pair_table": (C.c_int, [C.POINTER(RlGraph), C.c_int32, vp, vp, vp, vp, vp, vp]),
    "rl_mine_rules": (C.c_int, [C.c_int32, vp, vp, vp, vp, C.c_int32, C.c_int32, vp, C.c_int64, vp, vp]),
    "rl_tail_scratch_floats": (C.c_int64, [C.c_int32]),
    "rl_tail_forward": (C.c_int, [C.POINTER(RlCells), vp, C.c_int32, C.c_int32] + [vp] * 12 + [C.c_int32, vp]),
    "rl_tail_backward": (C.c_int, [C.POINTER(RlCells), vp, C.c_int32, C.c_int32, C.c_int32] + [vp] * 24 + [C.c_int32, vp]),
    "rl_pna_item_stats": (C.c_int, [C.POINTER(RlGraph), C.POINTER(RlRules), C.POINTER(RlSlots), C.POINTER(RlFrontier),
                                    C.POINTER(RlCells), vp, C.POINTER(RlPna), vp]),
    "rl_pna_front_forward": (C.c_int, [C.POINTER(RlSlots), C.POINTER(RlCells), C.POINTER(RlPna), vp, vp, vp, vp, vp, vp, vp]),
    "rl_pna_front_backward": (C.c_int, [C.POINTER(RlCells), C.POINTER(RlPna), vp, vp, vp, vp, vp, vp, vp]),
    "rl_pna_item_backward": (C.c_int, [C.POINTER(RlGraph), C.POINTER(RlRules), C.POINTER(RlSlots), C.POINTER(RlFrontier),
                                       C.POINTER(RlCells), vp, C.POINTER(RlPna), vp, vp, vp]),
    "rl_adam_step": (C.c_int, [C.c_int64, vp, vp, vp, vp, C.c_float, C.c_float, C.c_float, C.c_float, C.c_float,
                               C.c_int64, vp]),
    "rl_lstm_encode_forward": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, C.c_int32, vp, vp, vp, vp, vp, vp, vp]),
    "rl_lstm_encode_backward": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, C.c_int32, vp, vp, vp, vp, vp, vp, vp]),
    "rl_lstm_encode_wgrad": (C.c_int, [C.c_int64, C.c_int32, C.c_int32, vp, vp, vp, vp, vp]),
    "rl_slot_to_dense": (C.c_int, [C.c_int32, C.c_int32, vp, vp, C.c_int64, vp]),
    "rl_mask_to_dense": (C.c_int, [C.c_int32, C.c_int32, vp, vp, C.c_int64, vp]),
}


def exported_symbols():
    """Names every entry point declared in include/rnnlogic_b200.h must resolve to."""
    return sorted(_PROTOS)


def lib():
    """The loaded shared library (raises if it was not built -- no fallback)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                "rnnlogic_b200: %s is missing. Build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a). There is no CPU / PyTorch fallback for the hot path." % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in _PROTOS.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


class RlError(RuntimeError):
    pass


def check(rc: int, what: str = ""):
    if rc < 0:
        msg = lib().rl_last_error().decode(errors="replace")
        raise RlError("%s failed (%d): %s" % (what or "rnnlogic_b200 call", rc, msg))
    return rc


def require_cuda(t, what="tensor"):
    if t.device.type != "cuda":
        raise RlError("rnnlogic_b200 is CUDA-only (sm_100a): %s lives on %s. There is no CPU fallback; "
                      "move the model / batch to a CUDA device." % (what, t.device))

"""ctypes binding of libgcgcn_b200.so (the C ABI declared in include/gcgcn_b200.h).

There is no CPU fallback anywhere in this package: if the shared library is missing
or a call fails, a ``GcgcnError`` is raised.
"""
from __future__ import annotations

import ctypes
import glob
import os
import subprocess
import threading
from ctypes import c_float, c_int32, c_int64, c_size_t, c_uint64, c_void_p, c_char_p, POINTER

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_NAME = "libgcgcn_b200.so"
LIB_PATH = os.path.join(_HERE, LIB_NAME)
CSRC = os.path.join(_HERE, "csrc")
INCLUDE = os.path.join(os.path.dirname(_HERE), "include")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC", "-shared",
]

F32, BF16 = 0, 1
STACK_RELU, STACK_RESIDUAL, STACK_LINEAR = 1, 2, 4


class GcgcnError(RuntimeError):
    pass


class Dropout(ctypes.Structure):
    """struct gcgcn_dropout"""
    _fields_ = [("seed", c_uint64), ("p_att", c_float), ("p_gcn", c_float)]


class Batch(ctypes.Structure):
    """struct gcgcn_batch"""
    _fields_ = [
        ("num_docs", c_int32), ("total_nodes", c_int32), ("total_pairs", c_int64),
        ("max_nodes", c_int32), ("reserved", c_int32),
        ("node_ptr", c_void_p), ("pair_ptr", c_void_p), ("row_doc", c_void_p),
        ("doc_order", c_void_p), ("class_end", c_int32 * 4),
        ("tile_doc", c_void_p), ("num_tiles", c_int32), ("tile_rows", c_int32),
    ]


class EdgeTablesC(ctypes.Structure):
    """struct gcgcn_edge_tables"""
    _fields_ = [
        ("num_tokens", c_int32), ("num_slots", c_int32), ("num_pairs", c_int32), ("att_total", c_int32),
        ("dis_plus", c_int32), ("reserved", c_int32),
        ("tok_first", c_void_p), ("tok_slot_lo", c_void_p), ("tok_slot_hi", c_void_p),
        ("slot_tok0", c_void_p), ("slot_len", c_void_p), ("slot_span", c_void_p), ("slot_att", c_void_p),
        ("slot_rowi", c_void_p), ("slot_rowj", c_void_p), ("pair_idx", c_void_p), ("pair_slot_ptr", c_void_p),
        ("pair_denom", c_void_p), ("node_ctr_ptr", c_void_p), ("node_ctr", c_void_p),
        ("num_active_docs", c_int32), ("max_active_len", c_int32),
        ("adoc_tok0", c_void_p), ("adoc_len", c_void_p), ("adoc_slot_lo", c_void_p), ("adoc_slot_hi", c_void_p),
    ]


class RankResult(ctypes.Structure):
    """struct gcgcn_rank_result"""
    _fields_ = [
        ("count", c_int64), ("total_recall", c_int64), ("best_pos", c_int64), ("w", c_int64),
        ("auc", ctypes.c_double), ("ign_auc", ctypes.c_double),
        ("f1", c_float), ("theta", c_float), ("f1_at_w", c_float), ("precision_at_w", c_float),
        ("recall_at_w", c_float), ("ign_f1", c_float), ("ign_f1_at_w", c_float), ("reserved", c_float),
    ]


def sources():
    return sorted(glob.glob(os.path.join(CSRC, "*.cu")))


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile every CUDA source for sm_100a into the in-tree shared library (nvcc cross-compiles without a GPU).
    One object per source under build/obj (compiled in parallel, each only when older than its source or any
    header), then one link; skipped entirely when the library is newer than everything."""
    from concurrent.futures import ThreadPoolExecutor
    srcs = sources()
    hdrs = glob.glob(os.path.join(CSRC, "*.cuh")) + glob.glob(os.path.join(INCLUDE, "*.h"))
    newest_hdr = max(os.path.getmtime(p) for p in hdrs)
    if not force and os.path.exists(LIB_PATH):
        if os.path.getmtime(LIB_PATH) >= max([newest_hdr] + [os.path.getmtime(p) for p in srcs]):
            return LIB_PATH
    nvcc = os.environ.get("NVCC", "nvcc")
    objdir = os.path.join(os.path.dirname(_HERE), "build", "obj")
    os.makedirs(objdir, exist_ok=True)
    compile_flags = [f for f in NVCC_FLAGS if f != "-shared"]

    def compile_one(src):
        obj = os.path.join(objdir, os.path.basename(src)[:-3] + ".o")
        if not force and os.path.exists(obj) and os.path.getmtime(obj) >= max(newest_hdr, os.path.getmtime(src)):
            return obj, None
        cmd = [nvcc] + compile_flags + ["-I", INCLUDE, "-c", "-o", obj, src]
        if verbose:
            print(" ".join(cmd))
        res = subprocess.run(cmd, capture_output=True, text=True)
        return obj, (None if res.returncode == 0 else res.stdout + res.stderr)

    with ThreadPoolExecutor(max_workers=min(len(srcs), os.cpu_count() or 4)) as pool:
        results = list(pool.map(compile_one, srcs))
    errors = [e for _, e in results if e]
    if errors:
        raise GcgcnError("nvcc failed:\n" + "\n".join(errors))
    cmd = [nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", LIB_PATH] + [o for o, _ in results]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise GcgcnError("nvcc link failed:\n" + res.stdout + res.stderr)
    return LIB_PATH


_P = c_void_p
_BT = POINTER(Batch)
_DP = POINTER(Dropout)
_ET = POINTER(EdgeTablesC)

# name -> (restype, argtypes); mirrors include/gcgcn_b200.h one to one
SIGNATURES = {
    "gcgcn_version": (c_char_p, []),
    "gcgcn_last_error": (c_char_p, []),
    "gcgcn_launch_count": (c_uint64, []),
    "gcgcn_set_tile_blocks": (c_int32, [c_int32]),
    "gcgcn_device_info": (c_int32, [POINTER(c_int32)] * 3),
    "gcgcn_timing_begin": (c_int32, [_P]),
    "gcgcn_timing_end": (c_int32, [_P, c_char_p, c_size_t]),
    "gcgcn_workspace_bytes": (c_size_t, [c_int32, c_int64, c_int32]),
    "gcgcn_pool_fwd": (c_int32, [_P, _P, _P, _P, c_int32, _P, _P]),
    "gcgcn_pool_bwd": (c_int32, [_P, _P, _P, _P, c_int32, _P, _P]),
    "gcgcn_edge_mean_fwd": (c_int32, [_BT, _P, c_int32, _P, _P]),
    "gcgcn_edge_mean_bwd": (c_int32, [_BT, _P, c_int32, _P, _P]),
    "gcgcn_gat_fwd": (c_int32, [_BT, _P, _P, c_int32, _P, _P, _P, _P, c_int32, _P, _P, _P, _P,
                                _P, c_size_t, _P]),
    "gcgcn_gat_bwd": (c_int32, [_BT, _P, _P, c_int32, _P, _P, _P, c_int32, _P, _P, _P, _P,
                                _P, _P, _P, _P, _P, _P, c_size_t, _P]),
    "gcgcn_mha_fwd": (c_int32, [_BT, c_int32, _P, _P, _P, _P, _P, _P, _P, _P, c_size_t, _P]),
    "gcgcn_mha_bwd": (c_int32, [_BT, c_int32, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, c_size_t, _P]),
    "gcgcn_graphconv_stack_fwd": (c_int32, [_BT, c_int32, c_int32, c_int32, c_int32, c_int32]
                                  + [_P] * 13 + [_P, c_size_t, _P]),
    "gcgcn_graphconv_stack_bwd": (c_int32, [_BT, c_int32, c_int32, c_int32, c_int32, c_int32]
                                  + [_P] * 20 + [_P, c_size_t, _P]),
    "gcgcn_block_supported": (c_int32, [_BT, c_int32, c_int32, c_int32]),
    "gcgcn_dropout_mask": (c_int32, [c_uint64, c_int32, c_float, c_int64, _P, _P]),
    "gcgcn_mha_stack_fwd": (c_int32, [_BT, c_int32, c_int32] + [_P] * 15 + [_DP, _P, c_size_t, _P]),
    "gcgcn_mha_stack_bwd": (c_int32, [_BT, c_int32, c_int32] + [_P] * 22 + [_DP, _P, c_size_t, _P]),
    "gcgcn_pack_stack_weights": (c_int32, [_P, _P, c_int32, c_int32, c_int32, _P, _P, _P, _P]),
    "gcgcn_unpack_stack_grads": (c_int32, [_P, _P, _P, c_int32, c_int32, c_int32, _P, _P, _P]),
    "gcgcn_gat_collapse_fwd": (c_int32, [_P] * 8 + [c_int32, _P, _P]),
    "gcgcn_gat_collapse_bwd": (c_int32, [_P] * 8 + [c_int32] + [_P] * 8 + [_P]),
    "gcgcn_pack_rows": (c_int32, [_P, c_int32, c_int32, _P, _P]),
    "gcgcn_pair_gather_fwd": (c_int32, [_BT, _P, c_int32, _P, c_int32, _P, _P, _P, _P, _P, _P, _P]),
    "gcgcn_pair_gather_bwd": (c_int32, [_BT, _P, _P, c_int32, c_int32, c_int32, _P, _P, _P, _P,
                                        _P, c_size_t, _P]),
    "gcgcn_pair_dense_fwd": (c_int32, [_BT, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "gcgcn_pair_dense_ws_bytes": (c_size_t, [c_int32]),
    "gcgcn_pair_dense_bwd": (c_int32, [_BT, _P, _P, _P, _P, c_int32, _P, _P, _P, _P, _P, _P, c_size_t, _P]),
    "gcgcn_block_saved_bytes": (c_size_t, [c_int32, c_int64, c_int32]),
    "gcgcn_caggc_fwd": (c_int32, [_BT, c_int32, _P, _P, c_int32] + [_P] * 8 + [_P, _P, _DP, _P, c_size_t, _P]),
    "gcgcn_caggc_bwd": (c_int32, [_BT, c_int32, _P, _P, c_int32] + [_P] * 6 + [_P, _P]
                        + [_P] * 10 + [_DP, _P, c_size_t, _P]),
    "gcgcn_maggc_fwd": (c_int32, [_BT, c_int32, c_int32, _P, _P, c_int32] + [_P] * 7
                        + [_P, _P, _DP, _P, c_size_t, _P]),
    "gcgcn_maggc_bwd": (c_int32, [_BT, c_int32, c_int32, _P, c_int32] + [_P] * 5 + [_P, _P]
                        + [_P] * 9 + [_DP, _P, c_size_t, _P]),
    "gcgcn_expand_pair_context": (c_int32, [_P, c_int32, c_int32, c_int32, c_int32, c_int32, _P, _P, _P, _P]),
    "gcgcn_edgefeat_ws_bytes": (c_size_t, [c_int32, c_int32, c_int32, c_int32, c_int64]),
    "gcgcn_word_table_fwd": (c_int32, [_P, _P, _P, _P, c_int32, _P, _P]),
    "gcgcn_word_table_bwd": (c_int32, [_P, _P, _P, _P, c_int32, _P, _P, _P, c_size_t, _P]),
    "gcgcn_word_pool_fwd": (c_int32, [_ET, _P, _P, _P, _P, _P]),
    "gcgcn_word_pool_bwd": (c_int32, [_ET, _P, _P, _P, _P, _P, _P, c_size_t, _P]),
    "gcgcn_sent_pool_fwd": (c_int32, [_ET, _P, _P, _P, _P, _P, _P, _P, _P]),
    "gcgcn_sent_pool_bwd": (c_int32, [_ET, c_int32] + [_P] * 10 + [_P, c_size_t, _P]),
    "gcgcn_edge_fill_fwd": (c_int32, [_P, _P, _P, c_int32, c_int64, c_int32, _P, _P]),
    "gcgcn_edge_fill_bwd": (c_int32, [_P, _P, c_int32, c_int64, c_int32, _P, _P, _P, c_size_t, _P]),
    "gcgcn_colsum": (c_int32, [_P, c_int32, c_int32, c_int32, _P, _P, c_size_t, _P]),
    "gcgcn_bilinear_ws_bytes": (c_size_t, [c_int32, c_int32]),
    "gcgcn_bilinear_fwd": (c_int32, [_P, _P, _P, _P, c_int32, c_int32, c_int32, _P, c_int32, _P, c_size_t, _P]),
    "gcgcn_bilinear_bwd_ws_bytes": (c_size_t, [c_int32, c_int32]),
    "gcgcn_bilinear_bwd": (c_int32, [_P, _P, _P, _P, _P, c_int32, c_int32, c_float, _P, _P, _P, _P, c_size_t, _P]),
    "gcgcn_bilinear_reduce_fwd": (c_int32, [_P, _P, _P, c_int32, c_int32, c_int32, _P, c_int32, _P]),
    "gcgcn_bilinear_outer_bwd": (c_int32, [_P, c_int32, _P, c_int32, c_int32, _P, _P]),
    "gcgcn_bilinear_dt_bwd": (c_int32, [_P, c_int32, _P, c_int32, c_int32, _P, _P]),
    "gcgcn_doc_bias_fwd": (c_int32, [_BT, _P, c_int32, _P, _P]),
    "gcgcn_doc_bias_bwd": (c_int32, [_BT, _P, c_int32, _P, _P]),
    "gcgcn_pair_bce_fwd": (c_int32, [_BT, _P, _P, c_int32, _P, _P]),
    "gcgcn_pair_bce_bwd": (c_int32, [_BT, _P, _P, c_int32, _P, _P, _P]),
    "gcgcn_rank_ws_bytes": (c_size_t, [c_int64]),
    "gcgcn_rank_candidates": (c_int32, [_BT, _P, c_int32, _P, _P, c_int64, _P, _P, _P, _P]),
    "gcgcn_rank_candidates_at": (c_int32, [_BT, _P, c_int32, _P, _P, _P, _P, _P, _P, _P]),
    "gcgcn_rank_sort": (c_int32, [_P, _P, c_int64, _P, _P, _P, c_size_t, _P]),
    "gcgcn_rank_merge_ws_bytes": (c_size_t, [c_int64]),
    "gcgcn_rank_merge": (c_int32, [_P, _P, c_int64, _P, _P, c_int64, _P, _P, _P, c_size_t, _P]),
    "gcgcn_rank_curve_points": (c_int32, [_P, c_int64, c_int64, c_int32, _P, _P, _P, _P, c_size_t, _P]),
    "gcgcn_rank_curve": (c_int32, [_P, _P, c_int64, c_int64, c_int32, ctypes.c_double, _P, _P, c_size_t, _P]),
    "gcgcn_rank_decode": (c_int32, [_P, _P, c_int64, c_int64, _P, _P, c_int32, c_int32, _P, _P, _P, _P, _P, _P]),
    "gcgcn_rank_relations_ws_bytes": (c_size_t, [c_int64, c_int32]),
    "gcgcn_rank_by_relation": (c_int32, [_P, _P, c_int64, c_int32, _P, _P, _P, c_size_t, _P]),
    "gcgcn_rank_curve_relations": (c_int32, [_P, _P, c_int64, c_int32, _P, c_int32, _P, _P, _P, c_size_t, _P]),
    "gcgcn_rank_select": (c_int32, [_P, _P, c_int64, c_int32, _P, _P, _P, _P, _P, c_size_t, _P]),
    "gcgcn_adam_step": (c_int32, [_P, _P, _P, _P, c_int64] + [c_float] * 6 + [c_int32, _P]),
    "gcgcn_gemm": (c_int32, [c_int32, c_int32, c_int32, c_int32, c_int32, c_float, _P, c_int32, _P,
                             c_int32, c_float, _P, c_int32, _P, _P, c_size_t, _P]),
}

_lib = None
_lock = threading.Lock()


def load() -> ctypes.CDLL:
    """Load the in-tree library; raises (never falls back) when it is absent."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise GcgcnError(
                f"{LIB_PATH} not found: run `python -c 'import __graft_entry__ as g; g.build()'`. "
                "gcgcn_b200 has no CPU or PyTorch fallback.")
        lib = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)   # AttributeError if the header and the library disagree
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def call(name: str, *args) -> None:
    """Invoke an int-returning entry point and raise on a non-zero return code."""
    lib = load()
    rc = getattr(lib, name)(*args)
    if rc != 0:
        raise GcgcnError(f"{name} failed (code {rc}): {lib.gcgcn_last_error().decode()}")


def launch_count() -> int:
    return int(load().gcgcn_launch_count())


def set_tile_blocks(enable: bool) -> bool:
    """Switch the packed-tile tensor-core path of the MAGGC block on or off; returns the previous setting."""
    return bool(load().gcgcn_set_tile_blocks(1 if enable else 0))


def timing_begin(stream: int) -> None:
    call("gcgcn_timing_begin", stream)


def timing_end(stream: int) -> dict:
    """{kernel name: (launches, total_ms, total_flop)} since timing_begin."""
    buf = ctypes.create_string_buffer(1 << 16)
    call("gcgcn_timing_end", stream, buf, len(buf))
    out = {}
    for line in buf.value.decode().splitlines():
        name, cnt, ms, work = line.split("\t")
        out[name] = (int(cnt), float(ms), float(work))
    return out


def version() -> str:
    return load().gcgcn_version().decode()

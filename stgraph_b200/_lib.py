"""ctypes binding of ``libstgraph_b200.so`` (C ABI in ``include/stgraph_b200.h``).

This is the only bridge between the Python mirror of STGraph's API and the
hand-written sm_100a kernels.  There is NO fallback: if the library is missing
or a call fails, a ``RuntimeError`` is raised (the reference prints and
continues, ``stgraph/graph/static/csr.cu:27-33``; SURVEY.md section 8(b) "errors").
"""
from __future__ import annotations

import ctypes
import os
import subprocess
from ctypes import POINTER, Structure, c_char_p, c_float, c_int32, c_int64, c_size_t, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("STG_B200_LIB") or os.path.join(_HERE, "lib", "libstgraph_b200.so")   # env: A/B builds only
CSRC_DIR = os.path.join(_HERE, "csrc")

ABI_VERSION = 4
VM_MAX_TENSORS = 24
VM_MAX_INSTR = 96
VM_MAX_REGS = 48
VM_MAX_ACC = 8


class StgCsrView(Structure):
    """Mirror of ``StgCsrView`` (the four device arrays of ``stgraph_base.py:51-59``)."""

    _fields_ = [
        ("row_offset", c_void_p),
        ("column_indices", c_void_p),
        ("eids", c_void_p),
        ("node_ids", c_void_p),
        ("num_nodes", c_int32),
        ("num_edges", c_int32),
        ("eid_base", c_int32),
        ("eids_identity", c_int32),
        ("hub_rows", c_void_p),
        ("hub_count", c_void_p),
        ("hub_threshold", c_int32),
        ("hub_capacity", c_int32),
        ("work_queue", c_void_p),
    ]


class StgVmTensor(Structure):
    _fields_ = [("side", c_int32), ("bc0", c_int32), ("bc1", c_int32), ("pad", c_int32)]


class StgVmInstr(Structure):
    _fields_ = [
        ("op", ctypes.c_int16),
        ("phase", ctypes.c_int16),
        ("dst", ctypes.c_int16),
        ("a", ctypes.c_int16),
        ("b", ctypes.c_int16),
        ("pad", ctypes.c_int16),
        ("imm", c_float),
    ]


class StgVmProgram(Structure):
    _fields_ = [
        ("dim0", c_int32),
        ("dim1", c_int32),
        ("n_tensors", c_int32),
        ("n_instr", c_int32),
        ("n_regs", c_int32),
        ("n_acc", c_int32),
        ("n_pre", c_int32),
        ("n_loop", c_int32),
        ("acc_init", c_float * VM_MAX_ACC),
        ("acc_kind", c_int32 * VM_MAX_ACC),
        ("tensors", StgVmTensor * VM_MAX_TENSORS),
        ("instr", StgVmInstr * VM_MAX_INSTR),
    ]


_P = POINTER
_SIGNATURES = {
    # name: (restype, argtypes, returns_status)
    "stg_abi_version": (ctypes.c_int, [], False),
    "stg_last_error": (c_char_p, [], False),
    "stg_device_info": (ctypes.c_int, [ctypes.c_int, _P(c_int32), _P(c_int64), _P(c_int32), _P(c_int32)], True),
    "stg_agg_scaled_sum_f32": (ctypes.c_int, [_P(StgCsrView), c_void_p, c_int32, c_void_p, c_void_p, c_void_p,
                                              c_void_p, c_void_p], True),
    "stg_agg_scaled_sum_accum_f32": (ctypes.c_int, [_P(StgCsrView), c_void_p, c_int32, c_void_p, c_void_p, c_void_p,
                                                    c_void_p, c_void_p], True),
    "stg_agg_scaled_sum_red_f32": (ctypes.c_int, [_P(StgCsrView), c_void_p, c_int32, c_void_p, c_void_p, c_void_p,
                                                  c_void_p, c_void_p], True),
    "stg_agg_scaled_sum_rows_f32": (ctypes.c_int, [_P(StgCsrView), c_void_p, c_void_p, c_int32, c_void_p, c_void_p, c_void_p,
                                                   c_void_p, c_int32, c_void_p], True),
    "stg_csr_pack_edge_meta_f32": (ctypes.c_int, [_P(StgCsrView), c_void_p, c_void_p, c_void_p, c_void_p], True),
    "stg_agg_packed_sum_f32": (ctypes.c_int, [_P(StgCsrView), c_void_p, c_void_p, c_int32, c_void_p, c_void_p, c_int32,
                                              c_void_p], True),
    "stg_agg_packed_sum_strided_f32": (ctypes.c_int, [_P(StgCsrView), c_void_p, c_void_p, c_int32, c_int32, c_void_p,
                                                      c_void_p, c_int32, c_int32, c_void_p], True),
    "stg_agg_scaled_sum_h16": (ctypes.c_int, [_P(StgCsrView), c_void_p, c_int32, c_int32, c_void_p, c_void_p, c_void_p,
                                              c_void_p, c_void_p], True),
    "stg_agg_packed_sum_h16": (ctypes.c_int, [_P(StgCsrView), c_void_p, c_void_p, c_int32, c_int32, c_void_p, c_void_p,
                                              c_void_p], True),
    "stg_halo_push_f32": (ctypes.c_int, [c_void_p, c_int32, c_void_p, c_void_p, c_void_p, c_int64, _P(c_void_p), c_int32,
                                         c_int32, c_void_p], True),
    "stg_agg_packed_sum_rows_f32": (ctypes.c_int, [_P(StgCsrView), c_void_p, c_void_p, c_void_p, c_int32, c_void_p,
                                                   c_void_p, c_int32, c_void_p], True),
    "stg_rows_gather_f32": (ctypes.c_int, [c_void_p, c_int32, c_void_p, c_int64, c_void_p, c_int32, c_void_p], True),
    "stg_halo_send_f32": (ctypes.c_int, [c_void_p, c_int32, c_int32, c_int32, _P(c_int64), _P(c_void_p), c_void_p], True),
    "stg_halo_exchange_f32": (ctypes.c_int, [c_void_p, c_int32, c_void_p, _P(c_int64), c_void_p, _P(c_void_p), _P(c_void_p),
                                              c_void_p, c_int32, c_int32, c_int32, c_int32, c_void_p], True),
    "stg_peer_signal": (ctypes.c_int, [_P(c_void_p), c_int32, c_int32, c_int32, c_void_p], True),
    "stg_peer_wait": (ctypes.c_int, [c_void_p, c_int32, c_int32, c_int32, c_int64, c_void_p, c_void_p], True),
    "stg_agg_scaled_sum_parts_f32": (ctypes.c_int, [_P(StgCsrView), _P(c_void_p), _P(c_int32), c_int32, c_int32, c_void_p,
                                                    c_void_p, c_void_p, c_void_p, c_void_p], True),
    "stg_halo_pull_f32": (ctypes.c_int, [_P(c_void_p), _P(c_int32), c_int32, c_void_p, c_int64, c_int32, c_void_p, c_int32,
                                         c_void_p], True),
    "stg_agg_scaled_sum_f32_host": (ctypes.c_int, [_P(StgCsrView), c_void_p, c_int32, c_void_p, c_void_p, c_void_p,
                                                   c_void_p, c_void_p, c_size_t, c_void_p], True),
    "stg_agg_scaled_sum_f32_host_async": (ctypes.c_int, [_P(StgCsrView), c_void_p, c_int32, c_void_p, c_void_p, c_void_p,
                                                         c_void_p, c_void_p, c_size_t, c_void_p], True),
    "stg_gat_softmax_fwd_f32": (ctypes.c_int, [_P(StgCsrView), c_void_p, c_void_p, c_void_p, c_int32, c_int32,
                                               c_float, c_void_p, c_void_p, c_void_p, c_void_p], True),
    "stg_gat_softmax_bwd_f32": (ctypes.c_int, [_P(StgCsrView), _P(StgCsrView), c_void_p, c_void_p, c_void_p,
                                               c_void_p, c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_float,
                                               c_void_p, c_void_p, c_void_p, c_void_p, c_void_p], True),
    "stg_vm_run_f32": (ctypes.c_int, [_P(StgCsrView), _P(StgVmProgram), _P(c_void_p), c_void_p], True),
    "stg_edge_dot_f32": (ctypes.c_int, [c_void_p, c_int32, c_void_p, c_void_p, c_int64, c_void_p, c_void_p], True),
    "stg_edge_dot_bwd_f32": (ctypes.c_int, [c_void_p, c_int32, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p], True),
    "stg_bias_clamp_f32": (ctypes.c_int, [c_void_p, c_void_p, c_int64, c_int32, c_float, c_float, c_void_p], True),
    "stg_clamp_bwd_f32": (ctypes.c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_float, c_float, c_void_p], True),
    "stg_gru_reset_fwd_f32": (ctypes.c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_void_p], True),
    "stg_gru_reset_bwd_f32": (ctypes.c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p], True),
    "stg_gru_update_fwd_f32": (ctypes.c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p], True),
    "stg_gru_update_bwd_f32": (ctypes.c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64,
                                              c_void_p], True),
    "stg_tgcn_reset_fwd_f32": (ctypes.c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int32, c_void_p], True),
    "stg_tgcn_reset_bwd_f32": (ctypes.c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int32, c_void_p], True),
    "stg_tgcn_update_fwd_f32": (ctypes.c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int32, c_void_p], True),
    "stg_tgcn_update_bwd_f32": (ctypes.c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int32, c_void_p], True),
    "stg_gemm_tn_workspace_bytes": (c_size_t, [c_int64, c_int32, c_int32], False),
    "stg_gemm_tn_f32": (ctypes.c_int, [c_void_p, c_int64, c_void_p, c_int64, c_int64, c_int32, c_int32, c_void_p, c_void_p,
                                       c_void_p, c_size_t, c_void_p], True),
    "stg_csr_build_workspace_bytes": (c_size_t, [c_int64, c_int32], False),
    "stg_csr_build": (ctypes.c_int, [c_void_p, c_void_p, c_int64, c_int32] + [c_void_p] * 12
                      + [c_void_p, c_size_t, c_void_p], True),
    "stg_degree_norm_f32": (ctypes.c_int, [c_void_p, c_int32, c_void_p, c_void_p], True),
    "stg_weighted_row_degree_f32": (ctypes.c_int, [_P(StgCsrView), c_void_p, c_void_p, c_void_p], True),
    "stg_csr_hub_rows": (ctypes.c_int, [c_void_p, c_int32, c_int32, c_void_p, c_int32, c_void_p, c_void_p], True),
    "stg_snapshot_workspace_bytes": (c_size_t, [c_int64], False),
    "stg_snapshot_keys_from_edges": (ctypes.c_int, [c_void_p, c_void_p, c_int64, c_int32, c_void_p, c_void_p, c_void_p,
                                                    c_size_t, c_void_p], True),
    "stg_snapshot_diff": (ctypes.c_int, [c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_size_t,
                                         c_void_p], True),
    "stg_snapshot_apply": (ctypes.c_int, [c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_void_p,
                                          c_void_p, c_size_t, c_void_p], True),
    "stg_snapshot_views": (ctypes.c_int, [c_void_p, c_int64, c_int32, c_int32, c_int32] + [c_void_p] * 10
                           + [c_void_p, c_size_t, c_void_p], True),
    "stg_get_array_i32": (ctypes.c_int, [c_void_p, c_int64, c_void_p, c_void_p], True),
}

#: every symbol ``include/stgraph_b200.h`` declares (checked by tests/test_abi.py)
EXPORTED_SYMBOLS = tuple(_SIGNATURES)

_lib = None


def build(verbose: bool = False) -> str:
    """Compile every ``csrc/*.cu`` for sm_100a into ``lib/libstgraph_b200.so`` (nvcc cross-compiles without a GPU)."""
    cmd = ["make", "-C", CSRC_DIR, "-j", str(min(8, os.cpu_count() or 1))]
    res = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if verbose or res.returncode != 0:
        print(res.stdout)
    if res.returncode != 0:
        raise RuntimeError("building libstgraph_b200.so failed (see output above)")
    return LIB_PATH


def load():
    """Load the CUDA library; raises if it has not been built (no CPU fallback exists)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
            "(or `make -C stgraph_b200/csrc`). stgraph_b200 has no CPU fallback.")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (restype, argtypes, _) in _SIGNATURES.items():
        fn = getattr(lib, name)   # AttributeError if the .so is stale
        fn.restype = restype
        fn.argtypes = argtypes
    if lib.stg_abi_version() != ABI_VERSION:
        raise RuntimeError("libstgraph_b200.so ABI version mismatch; rebuild it")
    _lib = lib
    return lib


def call(name: str, *args):
    """Invoke a status-returning entry point; raise ``RuntimeError(stg_last_error())`` on failure."""
    lib = load()
    rc = getattr(lib, name)(*args)
    if _SIGNATURES[name][2] and rc != 0:
        raise RuntimeError(f"{name} failed ({rc}): {lib.stg_last_error().decode(errors='replace')}")
    return rc


def current_stream_ptr() -> int:
    import torch

    return torch.cuda.current_stream().cuda_stream


def ptr(t) -> int | None:
    """Raw device address of a torch tensor (``STGraphBackendTorch.tensor_raw_ptr``), None for None."""
    return None if t is None else t.data_ptr()

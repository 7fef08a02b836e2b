"""neural_speed_b200 -- B200-native (sm_100a) low-bit weight-only matmul behind neural-speed's kernel ABI.

Python is plumbing only: this module loads ``libns_b200.so`` (hand-written CUDA + C-ABI, see include/ns_b200.h) with
ctypes and mirrors the reference's host-side interfaces for the hot path:

* ``bestla_*`` host-buffer entry points  (neural_speed/core/ne_bestla.h:21-83)
* ``np_bestla_qpack`` / ``np_bestla_quantize``  (neural_speed/application/main_pybind.cpp:378-437)
* device-resident weights + matmuls used by the decode engine.

There is no CPU compute fallback: every compute call needs the CUDA extension and a B200.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "libns_b200.so")

# enums (include/ns_b200.h)
W_S4, W_S8, W_NF4, W_Q6K = 0, 1, 2, 3
S_F32, S_BF16, S_F16 = 0, 1, 2
COMP_F32, COMP_BF16, COMP_INT8, COMP_Q8_0, COMP_INT8_S8 = 0, 1, 2, 3, 4
NE_COMP_UNDEF, NE_COMP_F32, NE_COMP_BF16, NE_COMP_F16, NE_COMP_INT8 = 0, 1, 2, 3, 4
BTLA_F32 = 32
BTLA_BF16 = 16 | (1 << 16)
BTLA_F16 = 16
BTLA_S8 = 8 | (1 << 8)
BTLA_S4_CLIP = 4 | (1 << 8)
BTLA_F4_NF4 = 4 | (2 << 16)
MM_BIAS_BCAST, MM_FORCE_GEMV, MM_FORCE_TC = 1, 2, 4

EXPORTS = [
    "ns_last_error", "ns_version", "ns_launch_count",
    "bestla_init", "bestla_set_threads", "bestla_get_thread_handle", "bestla_timer",
    "bestla_support", "bestla_backend_support", "bestla_parallel_for", "bestla_mul", "bestla_add", "bestla_layernormalization",
    "ns_host_cache_clear", "ns_host_cache_entries",
    "bestla_f32f32_get_workspace_size", "bestla_f32f32_forward",
    "bestla_fusion_add_f32f32_support", "bestla_fusion_add_f32f32_forward",
    "bestla_fusion_QKV_f32f32_get_workspace_size", "bestla_fusion_QKV_f32f32_support", "bestla_fusion_QKV_f32f32_forward",
    "bestla_fusion_FFN_f32f32_get_workspace_size", "bestla_fusion_FFN_SiLu_f32f32_support",
    "bestla_fusion_FFN_SiLu_f32f32_forward", "bestla_unpackweight_fp32",
    "bestla_fusion_FFN_Gelu_Mul_f32f32_support", "bestla_fusion_FFN_Gelu_Mul_f32f32_forward",
    "bestla_fusion_FFN_GeLu_f32f32_support", "bestla_fusion_FFN_GeLu_f32f32_forward",
    "bestla_fusion_FFN_Add_GeLu_f32f32_support", "bestla_fusion_FFN_Add_GeLu_f32f32_forward", "bestla_packweight_copyattr",
    "bestla_create_device", "bestla_get_device_queue", "bestla_release_device", "bestla_device_gmem_size",
    "bestla_device_malloc", "bestla_device_free", "bestla_device_memcpy", "bestla_device_memcpy_sync", "bestla_device_sync",
    "bestla_device_storage_size", "ns_device_storage_bytes", "bestla_device_load_storage", "ns_device_workspace_bytes",
    "bestla_device_f32f32_forward",
    "ns_weight_from_q4_0", "ns_weight_from_q6_K", "ns_weight_from_btla_blob", "ns_weight_from_btla_blob_n", "ns_weight_random", "ns_weight_from_unpacked", "ns_weight_free", "ns_weight_info",
    "ns_weight_set_comp", "ns_weight_algorithmic_bytes", "ns_weight_dequant_f32",
    "ns_mul_mat", "ns_mul_qkv", "ns_ffn_silu", "ns_ffn_gelu",
    "ns_mul_mat_id", "ns_ffn_id", "ns_mul_mat_id_q4_0_f32_host", "ns_moe_plan",
    "ns_rmsnorm_fusable", "ns_rmsnorm_mul_mat", "ns_rmsnorm_mul_qkv", "ns_rmsnorm_ffn_silu", "ns_mul_mat_q4_0_f32_host", "ns_mul_mat_q6_K_f32_host",
    "ns_prepare_activation", "ns_matmul_prepared", "ns_graph_begin", "ns_graph_end", "ns_graph_launch", "ns_graph_free",
    "ns_device_quantize_q4_0", "ns_device_quantize_act",
    "BTLAGemmPackBSize", "BTLAGemmQuantPackB", "BTLAGemmPackB", "BTLAGemmUnPackB", "ns_quantize_row_q4_0", "ns_split_weight_size", "ns_split_weight",
    "ns_llama_create", "ns_llama_free", "ns_llama_set_f32", "ns_llama_set_weight", "ns_llama_eval", "ns_llama_generate", "ns_llama_set_exact_prefill",
    "ns_llama_kv_bytes", "ns_llama_set_tap", "ns_llama_kv_cache",
    "ns_comm_handle_bytes", "ns_comm_create", "ns_comm_get_handle", "ns_comm_open_peers", "ns_comm_link_local", "ns_comm_all_reduce_f32",
    "ns_comm_status", "ns_comm_free",
]

_lib = None


def lib() -> C.CDLL:
    """Load libns_b200.so; raises if it has not been built (no silent fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(_LIB_PATH):
        raise RuntimeError(f"{_LIB_PATH} missing: run `python -m neural_speed_b200.build` (nvcc, sm_100a)")
    L = C.CDLL(_LIB_PATH)
    vp, i, sz, f32p = C.c_void_p, C.c_int, C.c_size_t, C.c_void_p
    L.ns_last_error.restype = C.c_char_p
    L.ns_version.restype = C.c_char_p
    L.ns_launch_count.restype = C.c_ulonglong
    L.bestla_f32f32_get_workspace_size.restype = C.c_ulonglong
    L.bestla_f32f32_get_workspace_size.argtypes = [i, i, i, vp]
    L.bestla_f32f32_forward.argtypes = [f32p, vp, f32p, i, i, i, i, i, vp]
    L.bestla_fusion_add_f32f32_support.restype = C.c_bool
    L.bestla_fusion_add_f32f32_support.argtypes = [vp, i, i, i]
    L.bestla_fusion_add_f32f32_forward.argtypes = [f32p, vp, f32p, f32p, i, i, i, i, i, C.c_bool, vp]
    L.bestla_fusion_QKV_f32f32_get_workspace_size.restype = C.c_ulonglong
    L.bestla_fusion_QKV_f32f32_get_workspace_size.argtypes = [i, i, i, vp]
    L.bestla_fusion_QKV_f32f32_support.restype = C.c_bool
    L.bestla_fusion_QKV_f32f32_support.argtypes = [vp, vp, vp, i, i, i]
    L.bestla_fusion_QKV_f32f32_forward.argtypes = [f32p, vp, vp, vp, f32p, i, i, i, i, i, vp]
    L.bestla_fusion_FFN_f32f32_get_workspace_size.restype = C.c_ulonglong
    L.bestla_fusion_FFN_f32f32_get_workspace_size.argtypes = [i, i, i, i, vp, vp]
    L.bestla_fusion_FFN_SiLu_f32f32_support.restype = C.c_bool
    L.bestla_fusion_FFN_SiLu_f32f32_support.argtypes = [vp, vp, vp, i, i, i, i]
    L.bestla_fusion_FFN_SiLu_f32f32_forward.argtypes = [f32p, vp, vp, vp, f32p, f32p, f32p, i, i, i, i, vp]
    L.bestla_unpackweight_fp32.argtypes = [vp, i, i, f32p, i]
    L.bestla_create_device.restype = vp
    L.bestla_create_device.argtypes = [C.c_bool]
    L.bestla_get_device_queue.restype = vp
    L.bestla_get_device_queue.argtypes = [vp]
    L.bestla_release_device.argtypes = [vp]
    L.bestla_device_gmem_size.restype = sz
    L.bestla_device_gmem_size.argtypes = [vp]
    L.bestla_device_malloc.restype = vp
    L.bestla_device_malloc.argtypes = [sz, vp]
    L.bestla_device_free.argtypes = [vp, vp]
    L.bestla_device_memcpy.argtypes = [vp, vp, sz, vp]
    L.bestla_device_memcpy_sync.argtypes = [vp, vp, sz, vp]
    L.bestla_device_sync.argtypes = [vp]
    L.bestla_device_storage_size.restype = sz
    L.ns_device_storage_bytes.restype = sz
    L.ns_device_storage_bytes.argtypes = [vp]
    L.bestla_device_load_storage.argtypes = [vp, vp, vp, vp]
    L.ns_device_workspace_bytes.restype = sz
    L.ns_device_workspace_bytes.argtypes = [i, i]
    L.bestla_device_f32f32_forward.argtypes = [f32p, vp, f32p, i, i, i, i, i, vp, vp]
    L.ns_weight_from_q4_0.restype = vp
    L.ns_weight_from_q4_0.argtypes = [vp, i, i, sz, i, vp]
    L.ns_weight_from_q6_K.restype = vp
    L.ns_weight_from_q6_K.argtypes = [vp, i, i, sz, i, vp]
    L.ns_mul_mat_q6_K_f32_host.argtypes = [vp, sz, vp, vp, i, i, i]
    L.ns_weight_from_btla_blob.restype = vp
    L.ns_weight_from_btla_blob.argtypes = [vp, vp]
    L.ns_weight_random.restype = vp
    L.ns_weight_random.argtypes = [i, i, i, i, i, i, i, C.c_uint, vp]
    L.ns_weight_from_btla_blob_n.restype = vp
    L.ns_weight_from_btla_blob_n.argtypes = [vp, sz, vp]
    L.ns_weight_from_unpacked.restype = vp
    L.ns_weight_from_unpacked.argtypes = [vp, vp, vp, vp, i, i, i, i, i, i, vp]
    L.ns_weight_free.argtypes = [vp]
    L.ns_weight_info.argtypes = [vp] + [C.POINTER(C.c_int)] * 7
    L.ns_weight_set_comp.argtypes = [vp, i]
    L.ns_weight_algorithmic_bytes.restype = sz
    L.ns_weight_algorithmic_bytes.argtypes = [vp]
    L.ns_weight_dequant_f32.argtypes = [vp, vp, i, vp]
    L.ns_mul_mat.argtypes = [vp, vp, i, vp, i, i, vp, vp, i, vp, vp]
    L.ns_mul_qkv.argtypes = [vp, vp, vp, vp, i, vp, i, i, vp, vp]
    L.ns_ffn_silu.argtypes = [vp, vp, vp, vp, i, vp, vp, i, i, vp, vp]
    L.ns_ffn_gelu.argtypes = [vp, vp, vp, vp, vp, i, vp, i, vp, vp, i, i, vp, vp]
    L.ns_rmsnorm_fusable.argtypes = [vp, i, i]
    L.ns_mul_mat_id.argtypes = [vp, i, vp, i, i, i, vp, i, vp, i, i, i, vp]
    L.ns_ffn_id.argtypes = [vp, vp, vp, i, i, vp, i, i, i, vp, i, vp, vp, i, i, vp]
    L.ns_mul_mat_id_q4_0_f32_host.argtypes = [vp, i, sz, vp, i, i, vp, vp, i, i, i]
    L.ns_moe_plan.argtypes = [vp, i, i, i, i, vp, vp]
    L.ns_rmsnorm_mul_mat.argtypes = [vp, vp, i, vp, C.c_float, vp, i, i, vp, vp, vp]
    L.ns_rmsnorm_mul_qkv.argtypes = [vp, vp, vp, vp, i, vp, C.c_float, vp, i, i, vp, vp]
    L.ns_rmsnorm_ffn_silu.argtypes = [vp, vp, vp, vp, i, vp, C.c_float, vp, vp, i, i, vp, vp, vp]
    L.bestla_fusion_FFN_Gelu_Mul_f32f32_support.restype = C.c_bool
    L.bestla_fusion_FFN_Gelu_Mul_f32f32_support.argtypes = [vp, vp, vp, i, i, i, i]
    L.bestla_fusion_FFN_Gelu_Mul_f32f32_forward.restype = None
    L.bestla_fusion_FFN_Gelu_Mul_f32f32_forward.argtypes = [vp, vp, vp, vp, vp, vp, vp, i, i, i, i, vp]
    L.bestla_fusion_FFN_GeLu_f32f32_support.restype = C.c_bool
    L.bestla_fusion_FFN_GeLu_f32f32_support.argtypes = [vp, vp, i, i, i, i]
    L.bestla_fusion_FFN_GeLu_f32f32_forward.restype = None
    L.bestla_fusion_FFN_GeLu_f32f32_forward.argtypes = [vp, vp, vp, vp, vp, i, i, i, i, vp]
    L.bestla_fusion_FFN_Add_GeLu_f32f32_support.restype = C.c_bool
    L.bestla_fusion_FFN_Add_GeLu_f32f32_support.argtypes = [vp, vp, i, i, i, i]
    L.bestla_fusion_FFN_Add_GeLu_f32f32_forward.restype = None
    L.bestla_fusion_FFN_Add_GeLu_f32f32_forward.argtypes = [vp, vp, vp, vp, vp, vp, vp, i, i, i, i, C.c_bool, vp]
    L.bestla_packweight_copyattr.restype = None
    L.bestla_packweight_copyattr.argtypes = [vp, vp, i, i, i, vp]
    L.ns_mul_mat_q4_0_f32_host.argtypes = [vp, sz, vp, vp, i, i, i]
    L.ns_prepare_activation.argtypes = [vp, vp, i, i, vp, vp]
    L.ns_matmul_prepared.argtypes = [vp, i, i, vp, vp, i, i, vp, i, vp, vp, vp]
    L.ns_graph_begin.argtypes = [vp]
    L.ns_graph_end.restype = vp
    L.ns_graph_end.argtypes = [vp]
    L.ns_graph_launch.argtypes = [vp, vp]
    L.ns_graph_free.argtypes = [vp]
    L.ns_device_quantize_q4_0.argtypes = [vp, vp, i, i, vp]
    L.ns_device_quantize_act.argtypes = [vp, i, i, i, i, i, vp, vp, vp, vp]
    L.ns_llama_create.restype = vp
    L.ns_llama_create.argtypes = [vp, vp]
    L.ns_llama_free.restype = None
    L.ns_llama_free.argtypes = [vp]
    L.ns_llama_set_f32.argtypes = [vp, i, i, vp, sz]
    L.ns_llama_set_weight.argtypes = [vp, i, i, vp]
    L.ns_llama_eval.argtypes = [vp, vp, i, i, vp, vp]
    L.ns_llama_generate.argtypes = [vp, C.c_int32, i, i, vp]
    L.ns_llama_kv_bytes.restype = C.c_ulonglong
    L.ns_llama_kv_bytes.argtypes = [vp]
    L.ns_llama_set_tap.argtypes = [vp, i, vp, vp, i]
    L.ns_llama_kv_cache.argtypes = [vp, i, C.POINTER(vp), C.POINTER(vp)]
    L.ns_comm_handle_bytes.restype = sz
    L.ns_comm_create.restype = vp
    L.ns_comm_create.argtypes = [i, i, sz, vp]
    L.ns_comm_get_handle.argtypes = [vp, vp]
    L.ns_comm_open_peers.argtypes = [vp, vp]
    L.ns_comm_all_reduce_f32.argtypes = [vp, vp, sz, vp, vp]
    L.ns_comm_status.argtypes = [vp]
    L.ns_comm_free.restype = None
    L.ns_comm_free.argtypes = [vp]
    L.ns_split_weight_size.restype = sz
    L.ns_split_weight_size.argtypes = [vp, sz, sz]
    L.ns_split_weight.restype = C.c_bool
    L.ns_split_weight.argtypes = [vp, vp, sz, sz, sz, sz, sz, sz, C.c_bool]
    L.BTLAGemmPackBSize.restype = sz
    L.BTLAGemmPackBSize.argtypes = [sz, sz, sz, C.c_uint32, C.c_uint32, C.c_bool, i, vp]
    L.BTLAGemmQuantPackB.restype = C.c_bool
    L.BTLAGemmQuantPackB.argtypes = [vp, vp, sz, sz, sz, sz, C.c_uint32, C.c_uint32, C.c_bool, i, C.c_bool, vp]
    L.BTLAGemmPackB.restype = C.c_bool
    L.BTLAGemmPackB.argtypes = [vp, vp, vp, vp, sz, sz, sz, sz, C.c_uint32, C.c_uint32, C.c_bool, i, vp, vp]
    L.BTLAGemmUnPackB.restype = C.c_bool
    L.BTLAGemmUnPackB.argtypes = [vp, vp, sz, sz, sz, vp]
    L.ns_quantize_row_q4_0.argtypes = [vp, vp, i]
    _lib = L
    return L


def last_error() -> str:
    return lib().ns_last_error().decode()


def _check(rc: int, what: str) -> None:
    if rc != 0:
        raise RuntimeError(f"{what} failed ({rc}): {last_error()}")


def _np_ptr(a: np.ndarray):
    return a.ctypes.data_as(C.c_void_p)


# ------------------------------------------------------------------------------------------------ packing API (host)
_BITS = {"int4": BTLA_S4_CLIP, "int8": BTLA_S8, "nf4": BTLA_F4_NF4,
         "fp4": 4, "fp4_e2m1": 4, "fp4_bnb": 4 | (1 << 16),
         "int2": 2 | (1 << 8), "int3": 3 | (1 << 8), "int5": 5 | (1 << 8), "int6": 6 | (1 << 8), "int7": 7 | (1 << 8)}
_SCALE = {"fp32": BTLA_F32, "bf16": BTLA_BF16, "fp16": BTLA_F16}
_COMP = {"int8": NE_COMP_INT8, "bf16": NE_COMP_BF16, "fp16": NE_COMP_F16, "fp32": NE_COMP_F32}


def np_bestla_quantize(src_w: np.ndarray, weight_dtype="int4", group_size=32, alg="sym", scale_dtype="fp32",
                       compute_dtype="int8") -> np.ndarray:
    """RTN-quantise + pack a torch-layout fp32 weight [N,K] into a BesTLA blob (uint8 array).

    Mirrors Model.np_bestla_quantize (application/main_pybind.cpp:404-437 -> quant_utils.cpp:269 bestla_quantize)."""
    w = np.ascontiguousarray(src_w, np.float32)
    n, k = w.shape
    g = k if group_size == -1 else group_size
    qt, st, ct = _BITS[weight_dtype], _SCALE[scale_dtype], _COMP[compute_dtype]
    asym = alg == "asym"
    L = lib()
    size = L.BTLAGemmPackBSize(n, k, g, qt, st, asym, ct, None)
    if size == 0:
        raise ValueError("unsupported quantisation config")
    raw = np.zeros(size + 64, np.uint8)
    off = (-raw.ctypes.data) % 64
    buf = raw[off:off + size]
    if not L.BTLAGemmQuantPackB(_np_ptr(buf), _np_ptr(w), n, k, k, g, qt, st, asym, ct, True, None):
        raise RuntimeError("BTLAGemmQuantPackB failed")
    return buf


def np_bestla_qpack(src_w: np.ndarray, src_scales: np.ndarray, src_zeros, g_idx=None, weight_dtype="int4", group_size=32,
                    alg="sym", scale_dtype="fp32", compute_dtype="int8") -> np.ndarray:
    """Pack pre-quantised int8 weights [K,N] + scales [K/g,N] (+ zeros, g_idx) into a BesTLA blob.

    Mirrors Model.np_bestla_qpack (application/main_pybind.cpp:378-402 -> quant_utils.cpp:226 bestla_qpack);
    note the reference silently turns scale_dtype fp16 into bf16 here (quant_utils.cpp:252-254) and so do we."""
    q = np.ascontiguousarray(src_w, np.int8)
    k, n = q.shape
    sc = np.ascontiguousarray(src_scales, np.float32)
    asym = alg == "asym"
    zp = np.ascontiguousarray(src_zeros, np.int8) if asym else None
    gi = np.ascontiguousarray(g_idx, np.int32) if g_idx is not None else None
    g = k if group_size == -1 else group_size
    qt, ct = _BITS[weight_dtype], _COMP[compute_dtype]
    st = BTLA_F32 if scale_dtype == "fp32" else BTLA_BF16
    L = lib()
    size = L.BTLAGemmPackBSize(n, k, g, qt, st, asym, ct, _np_ptr(gi) if gi is not None else None)
    if size == 0:
        raise ValueError("unsupported quantisation config")
    raw = np.zeros(size + 64, np.uint8)
    off = (-raw.ctypes.data) % 64
    buf = raw[off:off + size]
    ok = L.BTLAGemmPackB(_np_ptr(buf), _np_ptr(q), _np_ptr(sc), _np_ptr(zp) if zp is not None else None, n, k, n, g, qt, st,
                         asym, ct, _np_ptr(gi) if gi is not None else None, None)
    if not ok:
        raise RuntimeError("BTLAGemmPackB failed")
    return buf


def unpack_blob(blob: np.ndarray, n: int, k: int) -> np.ndarray:
    """Host dequantisation of a blob to fp32 [K,N] (BTLAGemmUnPackB)."""
    out = np.empty((k, n), np.float32)
    if not lib().BTLAGemmUnPackB(_np_ptr(out), _np_ptr(blob), n, k, n, None):
        raise RuntimeError("BTLAGemmUnPackB failed")
    return out


def quantize_q4_0_host(w: np.ndarray) -> np.ndarray:
    """fp32 [N,K] -> uint8 [N, K/32*18] rows of block_q4_0 (ne_quantize_q4_0 path)."""
    w = np.ascontiguousarray(w, np.float32)
    n, k = w.shape
    out = np.empty((n, k // 32 * 18), np.uint8)
    L = lib()
    for r in range(n):
        L.ns_quantize_row_q4_0(_np_ptr(w[r]), _np_ptr(out[r]), k)
    return out


# ------------------------------------------------------------------------------------------------ device weights
class Weight:
    """Device-resident repacked weight (opaque ns_weight*)."""

    def __init__(self, handle, keepalive=None):
        if not handle:
            raise RuntimeError("weight creation failed: " + last_error())
        self.h = C.c_void_p(handle)
        self._keep = keepalive
        vals = [C.c_int() for _ in range(7)]
        lib().ns_weight_info(self.h, *[C.byref(v) for v in vals])
        self.n, self.k, self.group, self.wfmt, self.stype, self.comp, self.asym = [v.value for v in vals]

    @classmethod
    def from_q4_0_host(cls, rows: np.ndarray, n: int, k: int, queue=None):
        rows = np.ascontiguousarray(rows, np.uint8)
        return cls(lib().ns_weight_from_q4_0(_np_ptr(rows), n, k, rows.shape[1], 0, queue))

    @classmethod
    def from_q4_0_device(cls, dev_ptr: int, n: int, k: int, nb01: int, queue=None):
        return cls(lib().ns_weight_from_q4_0(C.c_void_p(dev_ptr), n, k, nb01, 1, queue))

    @classmethod
    def from_q6_K_host(cls, rows: np.ndarray, n: int, k: int, queue=None):
        """rows: uint8 [n, k/256*210] block_q6_K rows (the Q6_K output.weight of llama.cpp "Q4_0" GGUF files)."""
        rows = np.ascontiguousarray(rows, np.uint8)
        return cls(lib().ns_weight_from_q6_K(_np_ptr(rows), n, k, rows.shape[1], 0, queue))

    @classmethod
    def random(cls, n, k, group=32, wfmt=W_S4, stype=S_F32, comp=COMP_INT8, asym=False, seed=1, queue=None):
        """benchmark aid: random codes / scales generated on the device (no host data, no quantisation pass)"""
        return cls(lib().ns_weight_random(n, k, group, wfmt, stype, comp, 1 if asym else 0, seed, queue))

    @classmethod
    def from_blob(cls, blob: np.ndarray, queue=None):
        return cls(lib().ns_weight_from_btla_blob_n(_np_ptr(blob), blob.nbytes, queue))

    @classmethod
    def from_unpacked(cls, q_kn, scales, zp, group, wfmt=W_S4, stype=S_F32, comp=COMP_INT8, shuffle=None, queue=None):
        q = np.ascontiguousarray(q_kn, np.int8)
        k, n = q.shape
        sc = np.ascontiguousarray(scales, np.float32)
        z = np.ascontiguousarray(zp, np.int8) if zp is not None else None
        sh = np.ascontiguousarray(shuffle, np.int32) if shuffle is not None else None
        return cls(lib().ns_weight_from_unpacked(_np_ptr(q), _np_ptr(sc), _np_ptr(z) if z is not None else None,
                                                 _np_ptr(sh) if sh is not None else None, n, k, group, wfmt, stype, comp,
                                                 queue))

    def set_comp(self, comp: int):
        _check(lib().ns_weight_set_comp(self.h, comp), "ns_weight_set_comp")
        self.comp = comp
        return self

    @property
    def algorithmic_bytes(self) -> int:
        return int(lib().ns_weight_algorithmic_bytes(self.h))

    def free(self):
        if self.h:
            lib().ns_weight_free(self.h)
            self.h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def mul_mat(w: Weight, act_ptr: int, lda: int, dst_ptr: int, ldo: int, m: int, bias_ptr=None, residual_ptr=None, flags=0,
            ws_ptr=None, queue=None):
    _check(lib().ns_mul_mat(w.h, C.c_void_p(act_ptr), lda, C.c_void_p(dst_ptr), ldo, m,
                            C.c_void_p(bias_ptr) if bias_ptr else None, C.c_void_p(residual_ptr) if residual_ptr else None,
                            flags, C.c_void_p(ws_ptr) if ws_ptr else None, queue), "ns_mul_mat")


def mul_qkv(wq: Weight, wk: Weight, wv: Weight, act_ptr: int, lda: int, dst_ptr: int, ldo: int, m: int, queue=None):
    _check(lib().ns_mul_qkv(wq.h, wk.h, wv.h, C.c_void_p(act_ptr), lda, C.c_void_p(dst_ptr), ldo, m, None, queue), "ns_mul_qkv")


def ffn_silu(w1: Weight, w2: Weight, w3: Weight, act_ptr: int, lda: int, tmp_ptr: int, dst_ptr: int, ldo: int, m: int,
             queue=None):
    _check(lib().ns_ffn_silu(w1.h, w2.h, w3.h, C.c_void_p(act_ptr), lda, C.c_void_p(tmp_ptr), C.c_void_p(dst_ptr), ldo, m,
                             None, queue), "ns_ffn_silu")


def _handles(ws):
    return (C.c_void_p * len(ws))(*[w.h for w in ws])


def mul_mat_id(experts, ids, id: int, act_ptr: int, lda: int, dst_ptr: int, ldo: int, m: int, flags=0, queue=None):
    """ne_mul_mat_id: dst[t] = experts[ids[t, id]] . act[t].  ids: int32 numpy [m][n_used] (host) or a (device_ptr, stride) tuple."""
    if isinstance(ids, tuple):
        ptr, stride, on_dev = C.c_void_p(ids[0]), int(ids[1]), 1
    else:
        ids = np.ascontiguousarray(ids, np.int32)
        ptr, stride, on_dev = ids.ctypes.data_as(C.c_void_p), ids.shape[1], 0
    _check(lib().ns_mul_mat_id(_handles(experts), len(experts), ptr, stride, id, on_dev, C.c_void_p(act_ptr), lda, C.c_void_p(dst_ptr),
                               ldo, m, flags, queue), "ns_mul_mat_id")


def ffn_id(gate, down, up, ids, id: int, act_ptr: int, lda: int, tmp_ptr: int, dst_ptr: int, ldo: int, m: int, gelu=False, queue=None):
    """ne_mul_id_ffn_silu / _gelu with per-token expert selection (ids as in mul_mat_id)."""
    if isinstance(ids, tuple):
        ptr, stride, on_dev = C.c_void_p(ids[0]), int(ids[1]), 1
    else:
        ids = np.ascontiguousarray(ids, np.int32)
        ptr, stride, on_dev = ids.ctypes.data_as(C.c_void_p), ids.shape[1], 0
    _check(lib().ns_ffn_id(_handles(gate), _handles(down), _handles(up), len(gate), 1 if gelu else 0, ptr, stride, id, on_dev,
                           C.c_void_p(act_ptr), lda, C.c_void_p(tmp_ptr), C.c_void_p(dst_ptr), ldo, m, queue), "ns_ffn_id")


def rmsnorm_fusable(weights, m: int) -> bool:
    """Can RMSNorm(x) * norm_w be folded into the launch of these 1..3 weights for m activation rows?"""
    return bool(lib().ns_rmsnorm_fusable(_handles(weights), len(weights), m))


def rmsnorm_mul_mat(w: Weight, act_ptr: int, lda: int, norm_ptr: int, eps: float, dst_ptr: int, ldo: int, m: int, residual_ptr=None,
                    queue=None):
    _check(lib().ns_rmsnorm_mul_mat(w.h, C.c_void_p(act_ptr), lda, C.c_void_p(norm_ptr), eps, C.c_void_p(dst_ptr), ldo, m,
                                    C.c_void_p(residual_ptr) if residual_ptr else None, None, queue), "ns_rmsnorm_mul_mat")


def rmsnorm_mul_qkv(wq: Weight, wk: Weight, wv: Weight, act_ptr: int, lda: int, norm_ptr: int, eps: float, dst_ptr: int, ldo: int,
                    m: int, queue=None):
    _check(lib().ns_rmsnorm_mul_qkv(wq.h, wk.h, wv.h, C.c_void_p(act_ptr), lda, C.c_void_p(norm_ptr), eps, C.c_void_p(dst_ptr), ldo,
                                    m, None, queue), "ns_rmsnorm_mul_qkv")


def rmsnorm_ffn_silu(w1: Weight, w2: Weight, w3: Weight, act_ptr: int, lda: int, norm_ptr: int, eps: float, tmp_ptr: int, dst_ptr: int,
                     ldo: int, m: int, residual_ptr=None, queue=None):
    _check(lib().ns_rmsnorm_ffn_silu(w1.h, w2.h, w3.h, C.c_void_p(act_ptr), lda, C.c_void_p(norm_ptr), eps, C.c_void_p(tmp_ptr),
                                     C.c_void_p(dst_ptr), ldo, m, C.c_void_p(residual_ptr) if residual_ptr else None, None, queue),
           "ns_rmsnorm_ffn_silu")


def ffn_gelu(w1: Weight, w2: Weight, w3, b1_ptr, b2_ptr, bias_bcast: int, act_ptr: int, lda: int, tmp_ptr: int, dst_ptr: int,
             ldo: int, m: int, queue=None):
    """GELU feed-forward (Gelu_Mul when w3 is given, else (Add_)GeLu), device pointers."""
    _check(lib().ns_ffn_gelu(w1.h, w2.h, w3.h if w3 is not None else None, C.c_void_p(b1_ptr) if b1_ptr else None,
                             C.c_void_p(b2_ptr) if b2_ptr else None, bias_bcast, C.c_void_p(act_ptr), lda, C.c_void_p(tmp_ptr),
                             C.c_void_p(dst_ptr), ldo, m, None, queue), "ns_ffn_gelu")


class LlamaHParams(C.Structure):
    _fields_ = [("n_vocab", C.c_int), ("n_embd", C.c_int), ("n_head", C.c_int), ("n_head_kv", C.c_int), ("n_layer", C.c_int),
                ("n_ff", C.c_int), ("n_ctx", C.c_int), ("norm_eps", C.c_float), ("rope_theta", C.c_float), ("rope_scale", C.c_float)]


class Llama:
    """Device-resident Llama-family eval step (ns_llama_*): model_eval + greedy sampling of the reference, on the GPU."""

    TOK_EMBD, OUT_NORM, OUTPUT, ATTN_NORM, WQ, WK, WV, WO, FFN_NORM, W1, W2, W3 = range(12)

    def __init__(self, n_vocab, n_embd, n_head, n_head_kv, n_layer, n_ff, n_ctx, norm_eps=1e-6, rope_theta=10000.0, rope_scale=1.0,
                 queue=None):
        self.hp = LlamaHParams(n_vocab, n_embd, n_head, n_head_kv, n_layer, n_ff, n_ctx, norm_eps, rope_theta, rope_scale)
        self.h = C.c_void_p(lib().ns_llama_create(C.byref(self.hp), queue))
        if not self.h:
            raise RuntimeError("ns_llama_create failed: " + last_error())
        self._keep = []

    def set_f32(self, tensor: int, layer: int, arr: np.ndarray):
        a = np.ascontiguousarray(arr, np.float32)
        _check(lib().ns_llama_set_f32(self.h, tensor, layer, _np_ptr(a), a.size), "ns_llama_set_f32")

    def set_weight(self, tensor: int, layer: int, w: "Weight"):
        self._keep.append(w)  # borrowed by the context
        _check(lib().ns_llama_set_weight(self.h, tensor, layer, w.h), "ns_llama_set_weight")

    def eval(self, tokens, n_past: int, want_logits=True):
        t = np.ascontiguousarray(tokens, np.int32)
        logits = np.empty(self.hp.n_vocab, np.float32) if want_logits else None
        nxt = C.c_int32(0)
        _check(lib().ns_llama_eval(self.h, _np_ptr(t), t.size, n_past, _np_ptr(logits) if want_logits else None, C.byref(nxt)),
               "ns_llama_eval")
        return logits, int(nxt.value)

    def generate(self, first_token: int, n_past: int, n_new: int) -> np.ndarray:
        out = np.empty(n_new, np.int32)
        _check(lib().ns_llama_generate(self.h, first_token, n_past, n_new, _np_ptr(out)), "ns_llama_generate")
        return out

    def kv_bytes(self) -> int:
        return int(lib().ns_llama_kv_bytes(self.h))

    def _dims(self):
        hd = self.hp.n_embd // self.hp.n_head
        return self.hp.n_embd, hd * self.hp.n_head_kv, hd

    def set_tap(self, layer: int, max_rows: int = 1):
        """Test / debug surface (ns_llama_set_tap): from now on every eval copies `layer`'s q | k | v before RoPE and its
        attention output into device buffers of max_rows rows, read back with tap(m).  layer < 0 removes the tap."""
        import torch
        E, kvd, _ = self._dims()
        if layer < 0:
            _check(lib().ns_llama_set_tap(self.h, -1, None, None, 0), "ns_llama_set_tap")
            self._tap = None
            return
        qkv = torch.empty(max_rows * (E + 2 * kvd), dtype=torch.float32, device="cuda")
        attn = torch.empty(max_rows * E, dtype=torch.float32, device="cuda")
        torch.cuda.synchronize()
        _check(lib().ns_llama_set_tap(self.h, layer, qkv.data_ptr(), attn.data_ptr(), max_rows), "ns_llama_set_tap")
        self._tap = (qkv, attn)

    def tap(self, m: int):
        """(q [m, n_embd], k [m, kvd], v [m, kvd], attn [m, n_embd]) of the last eval of m tokens: views of the tap buffers"""
        E, kvd, _ = self._dims()
        qkv, attn = self._tap
        q = qkv[:m * E].view(m, E)
        k = qkv[m * E:m * (E + kvd)].view(m, kvd)
        v = qkv[m * (E + kvd):m * (E + 2 * kvd)].view(m, kvd)
        return q, k, v, attn[:m * E].view(m, E)

    def kv_cache(self, layer: int):
        """(K, V) fp16 caches of `layer`, each a torch view [n_head_kv, n_ctx, head size] of the engine's device memory"""
        import torch
        k, v = C.c_void_p(), C.c_void_p()
        _check(lib().ns_llama_kv_cache(self.h, layer, C.byref(k), C.byref(v)), "ns_llama_kv_cache")
        shape = (self.hp.n_head_kv, self.hp.n_ctx, self._dims()[2])

        class _View:  # __cuda_array_interface__ over memory the context owns (valid until close())
            def __init__(self, ptr):
                self.__cuda_array_interface__ = dict(shape=shape, typestr="<f2", data=(ptr, False), version=2, strides=None)

        return tuple(torch.as_tensor(_View(p.value), device="cuda") for p in (k, v))

    def set_exact_prefill(self, on: bool = True):
        """prompts longer than 32 tokens in pieces of 32: the reference's integer block sums instead of the bf16 tensor-core GEMM"""
        _check(lib().ns_llama_set_exact_prefill(self.h, 1 if on else 0), "ns_llama_set_exact_prefill")

    def close(self):
        if self.h:
            lib().ns_llama_free(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

"""ctypes binding of libapertis_b200.so (the C ABI declared in include/apertis_b200.h).

There is no CPU fallback: if the shared library is missing, or the device is not an sm_100 part,
the first call raises.  Pointers are passed as raw addresses (``tensor.data_ptr()``), work is
enqueued on ``torch.cuda.current_stream()``.
"""
from __future__ import annotations

import ctypes
import os
import subprocess
import threading
from ctypes import c_char_p, c_float, c_int, c_int64, c_size_t, c_uint32, c_void_p

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libapertis_b200.so")
CSRC = os.path.join(_HERE, "csrc")

AB_F32, AB_BF16 = 0, 1
ACT = {"gelu": 0, "relu": 1, "silu": 2, "swish": 2}
EPI_NONE, EPI_BIAS, EPI_BIAS_ACT, EPI_DACT, EPI_ADD = 0, 1, 2, 3, 4
SCAN_SINGLE_PASS, SCAN_TWO_PASS, SCAN_PIPELINED, SCAN_ROUNDS = 0, 1, 2, 3
ROW_ALIGN = 256        # AB_GEMM_ROW_TILE: rows of one expert GEMM tile (a CTA pair, 128 rows per CTA)
ROUTER_EXACT, ROUTER_BF16, ROUTER_FP16 = 0, 1, 2

P, I, I64, SZ, F, U32 = c_void_p, c_int, c_int64, c_size_t, c_float, c_uint32

# name -> (restype, argtypes); mirrors include/apertis_b200.h one to one
SIGNATURES = {
    "ab_version": (I, []),
    "ab_device_check": (I, [I]),
    "ab_last_error": (I, [c_char_p, SZ]),
    "ab_causal_conv1d_silu_fwd": (I, [P, I64, P, P, P, I, I, I, I, I, P]),
    "ab_causal_conv1d_silu_bwd_workspace_bytes": (SZ, [I, I, I]),
    "ab_causal_conv1d_silu_bwd": (I, [P, I64, P, P, P, P, I64, P, P, P, SZ, I, I, I, I, I, P]),
    "ab_selective_scan_plan": (I, [I, I, I, I, P, P, P, P, P]),
    "ab_selective_scan_fwd": (I, [P, P, P, P, I64, P, I64, P, P, P, P, P, P, P, P, SZ, U32, I, I, I, I, I, I, P]),
    "ab_selective_scan_bwd": (I, [P, P, P, P, I64, P, I64, P, P, P, P, P, P, P, P, I64, P, P, P, P, P, SZ, U32, I,
                                  I, I, I, I, I, P]),
    "ab_ssm_scan_plan": (I, [I, I, I, I, P, P]),
    "ab_ssm_scan_tune": (I, [I, I, I, I, I]),
    "ab_ssm_scan_fwd": (I, [P, I64, P, I64, P, P, P, I64, P, I64, P, P, P, P, P, P, P, P, SZ, I, I, I, I, I, P]),
    "ab_ssm_scan_bwd": (I, [P, I64, P, P, I64, P, I64, P, P, P, P, P, P, I64, P, P, I64, P, I64, P, I64, I, P, P, P, P, SZ,
                            I, I, I, I, I, P]),
    "ab_gemm_row_tile": (I, []),
    "ab_shifted_ce_fwd": (I, [P, P, P, P, P, P, I, I, I, I64, I, P]),
    "ab_shifted_ce_bwd": (I, [P, P, P, P, P, I, I, I, I64, I, P]),
    "ab_ep_permute_ln": (I, [P, P, P, P, P, P, P, P, I, I, I64, I, I, I64, I, I, P]),
    "ab_ep_unpermute_bwd": (I, [P, P, P, P, P, P, P, I, I, I64, P, F, P, I, I, I64, I, I, I, P]),
    "ab_ep_grouped_gemm_nt": (I, [P, P, P, P, P, I, I, I64, P, P, I64, I, I, I, I, I, I, P]),
    "ab_ep_grouped_gemm_nn": (I, [P, P, P, P, P, I, I, I64, P, P, I64, I, I, I, I, I, I, P]),
    "ab_moe_router_workspace_bytes": (SZ, [I, I, I]),
    "ab_moe_router_fwd": (I, [P, P, P, F, P, P, P, P, P, P, P, P, P, P, P, P, P, P, SZ, I, I, I, I, I, I, P]),
    "ab_moe_topk_from_logits": (I, [P, P, P, P, P, P, I, I, I, P]),
    "ab_moe_max_rows": (I64, [I, I, I, I, I]),
    "ab_moe_plan_workspace_bytes": (SZ, [I, I, I]),
    "ab_moe_plan": (I, [P, P, P, I, P, P, P, P, P, P, P, P, SZ, I, I, I, I, I64, I, P]),
    "ab_moe_permute_ln": (I, [P, P, P, P, P, P, P, P, I, I, I64, I, I, P]),
    "ab_moe_unpermute": (I, [P, P, P, P, P, F, P, I, I, I, I, I, P]),
    "ab_moe_unpermute_bwd": (I, [P, P, P, P, P, P, P, P, F, P, I, I, I64, I, I, I, P]),
    "ab_moe_permute_ln_bwd_workspace_bytes": (SZ, [I, I, I64]),
    "ab_moe_permute_ln_bwd": (I, [P, P, P, P, P, P, P, P, P, P, P, SZ, I, I, I, I64, I, I, P]),
    "ab_moe_segment_colsum_workspace_bytes": (SZ, [I, I, I64]),
    "ab_moe_segment_colsum": (I, [P, P, P, P, P, SZ, I, I, I, I64, I, P]),
    "ab_moe_router_bwd_workspace_bytes": (SZ, [I, I, I]),
    "ab_moe_router_bwd": (I, [P] * 24 + [SZ, I, I, I, I, I, P]),
    "ab_grouped_gemm_nt": (I, [P, P, P, P, P, P, P, P, I64, I, I, I, I, I, I, F, P, P]),
    "ab_grouped_gemm_nn": (I, [P, P, P, P, P, P, P, P, I64, I, I, I, I, I, I, F, P, P]),
    "ab_grouped_gemm_tn_workspace_bytes": (SZ, [I, I, I, I]),
    "ab_grouped_gemm_tn": (I, [P, P, P, P, I64, I, I, I, I, I64, P, SZ, P]),
    "ab_dense_gemm_nt": (I, [P, P, P, P, P, I64, I, I, I, I, P]),
    "ab_dense_gemm_nn": (I, [P, P, P, P, P, I64, I, I, I, I, P]),
    "ab_dense_gemm_tn_workspace_bytes": (SZ, [I64, I, I]),
    "ab_dense_gemm_tn": (I, [P, P, P, P, SZ, I64, I, I, P]),
    "ab_dt_compose_fwd": (I, [P, P, P, I, I, I, I, I, P]),
    "ab_dt_compose_bwd": (I, [P, P, P, P, P, I, I, I, I, P]),
    "ab_layernorm_fwd": (I, [P, P, P, F, P, P, I, I, I, I, P]),
    "ab_layernorm_bwd_workspace_bytes": (SZ, [I, I]),
    "ab_layernorm_bwd": (I, [P, P, P, P, P, P, P, P, P, SZ, I, I, I, I, P]),
    "ab_dropout_add": (I, [P, P, P, F, P, I64, I, I, P]),
    "ab_cast_f32_to_bf16": (I, [P, P, I64, P]),
    "ab_split_f32_to_bf16x3": (I, [P, P, I64, I64, I, P]),
    "ab_split_f32_to_bf16x3_rows": (I, [P, P, P, I, I64, I64, I, P]),
}

_lib = None
_lock = threading.Lock()
_checked_devices = set()


def build(verbose: bool = False) -> str:
    """Compiles csrc/*.cu for sm_100a into libapertis_b200.so (nvcc cross-compiles without a GPU)."""
    cmd = ["make", "-C", CSRC, "-j", "8"]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("building libapertis_b200.so failed:\n" + res.stdout[-4000:] + res.stderr[-4000:])
    if verbose:
        print(res.stdout[-2000:])
    return LIB_PATH


def load() -> ctypes.CDLL:
    """Loads the shared library (building it first if the .so is absent and nvcc is present)."""
    global _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            build()
        lib = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)     # AttributeError if the .so lacks a declared symbol
            fn.restype = res
            fn.argtypes = args
        _lib = lib
        return lib


def last_error() -> str:
    buf = ctypes.create_string_buffer(600)
    load().ab_last_error(buf, 600)
    return buf.value.decode("utf-8", "replace")


def ptr(t):
    """Device address of a tensor (None -> NULL)."""
    if t is None:
        return None
    return t.data_ptr()


def dt(t_or_dtype) -> int:
    d = t_or_dtype.dtype if torch.is_tensor(t_or_dtype) else t_or_dtype
    if d == torch.float32:
        return AB_F32
    if d == torch.bfloat16:
        return AB_BF16
    raise TypeError(f"apertis_b200 kernels take float32 or bfloat16 activations, got {d}")


def stream_ptr(device=None) -> int:
    """Raw handle of torch's current stream on `device` (default: the current device)."""
    return torch.cuda.current_stream(device).cuda_stream


def ensure_device(device) -> None:
    """Fails loudly unless `device` is a CUDA sm_100 device (no CPU / other-arch fallback exists)."""
    if device.type != "cuda":
        raise RuntimeError("apertis_llm_b200: the hot path only runs on a CUDA sm_100a (B200) device; got "
                           f"device '{device}'. There is no CPU fallback.")
    idx = device.index if device.index is not None else torch.cuda.current_device()
    if idx in _checked_devices:
        return
    rc = load().ab_device_check(idx)
    if rc != 0:
        raise RuntimeError("apertis_llm_b200: " + last_error())
    _checked_devices.add(idx)


# kernels launched by one call of each entry point (memsets not counted)
KERNELS_PER_CALL = {
    "ab_causal_conv1d_silu_fwd": 1, "ab_causal_conv1d_silu_bwd": 2,
    "ab_selective_scan_fwd": 1, "ab_selective_scan_bwd": 2,          # single pass; two pass adds 2
    "ab_ssm_scan_fwd": 1, "ab_ssm_scan_bwd": 2, "ab_dense_gemm_nt": 1, "ab_dense_gemm_nn": 1, "ab_dense_gemm_tn": 2,
    "ab_dt_compose_fwd": 1, "ab_dt_compose_bwd": 2,
    "ab_moe_router_fwd": 2, "ab_moe_topk_from_logits": 1, "ab_moe_plan": 7, "ab_moe_permute_ln": 1, "ab_moe_unpermute": 1,
    "ab_moe_unpermute_bwd": 1, "ab_moe_permute_ln_bwd": 2, "ab_moe_segment_colsum": 2, "ab_moe_router_bwd": 3,
    "ab_layernorm_fwd": 1, "ab_layernorm_bwd": 3,
    "ab_grouped_gemm_nt": 1, "ab_grouped_gemm_nn": 1, "ab_grouped_gemm_tn": 1, "ab_cast_f32_to_bf16": 1,
    "ab_shifted_ce_fwd": 2, "ab_shifted_ce_bwd": 1, "ab_ep_permute_ln": 1, "ab_ep_unpermute_bwd": 1, "ab_ep_grouped_gemm_nt": 1, "ab_ep_grouped_gemm_nn": 1,
    "ab_split_f32_to_bf16x3": 1, "ab_split_f32_to_bf16x3_rows": 1,
}
launch_count = 0          # kernels launched through this binding since import (bench.py reads deltas)
_timed = None             # None, or {"names": set, "events": [(name, start, end), ...]} while bench.py profiles


def start_timing(names):
    """Record CUDA events (on the launching stream) around every call of the given entry points."""
    global _timed
    _timed = {"names": set(names), "events": []}


def stop_timing():
    """-> {name: [ms per call, ...]} for the calls recorded since start_timing(); synchronises."""
    global _timed
    t, _timed = _timed, None
    out = {}
    if t is None:
        return out
    torch.cuda.synchronize()
    for name, a, b in t["events"]:
        out.setdefault(name, []).append(a.elapsed_time(b))
    return out


def call(name: str, *args):
    """Calls an int-returning entry point; non-zero -> RuntimeError carrying ab_last_error()."""
    global launch_count
    fn = getattr(load(), name)
    if _timed is not None and name in _timed["names"]:
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        rc = fn(*args)
        b.record()
        _timed["events"].append((name, a, b))
    else:
        rc = fn(*args)
    if rc != 0:
        raise RuntimeError(f"{name} failed (code {rc}): {last_error()}")
    launch_count += KERNELS_PER_CALL.get(name, 1)


def query(name: str, *args):
    return getattr(load(), name)(*args)

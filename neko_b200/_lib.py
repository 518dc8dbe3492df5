"""ctypes binding of the C ABI in include/neko_b200.h.

There is deliberately no fallback: if the CUDA library is missing or the device is not an sm_100
part, every entry point raises.  (The parity oracle lives under oracle/ and is never imported here.)
"""
from __future__ import annotations

import ctypes as C
import os
import re

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libneko_b200.so")
HEADER = os.path.join(os.path.dirname(HERE), "include", "neko_b200.h")


class NekoError(RuntimeError):
    pass


class SampleDesc(C.Structure):
    """neko_sample_desc (include/neko_b200.h)."""
    _fields_ = [(n, C.c_int32) for n in (
        "n_timesteps", "n_patches", "n_text", "n_cobs", "n_dobs", "n_cact", "n_dact", "seq_off",
        "text_off", "cobs_off", "dobs_off", "cact_off", "dact_off", "patch_off", "row_base", "reserved1")]


class TokParams(C.Structure):
    """neko_tok_params (include/neko_b200.h)."""
    _fields_ = [("mu", C.c_float), ("M", C.c_float)] + [(n, C.c_int32) for n in (
        "n_bins", "cont_start", "disc_start", "vocab", "use_pos", "seq_len", "width", "ctx_rows")]


class Dropout(C.Structure):
    """neko_dropout (include/neko_b200.h): counter-based mask of one dropout site."""
    _fields_ = [("seed", C.c_void_p), ("stream", C.c_uint32), ("thr16", C.c_uint32), ("scale", C.c_float), ("reserved", C.c_uint32)]

    @classmethod
    def make(cls, seed_tensor, stream: int, p: float):
        """seed_tensor: int32/uint32 CUDA tensor of 2 words; p: drop probability (quantised to 16 bits)."""
        thr = int(round(float(p) * 65536.0))
        if seed_tensor is None or thr <= 0:
            return cls(seed=None, stream=0, thr16=0, scale=1.0, reserved=0)
        thr = min(thr, 65535)
        d = cls(seed=seed_tensor.data_ptr(), stream=int(stream), thr16=thr, scale=65536.0 / (65536.0 - thr), reserved=0)
        # the kernels read the seed through this pointer: the descriptor keeps its tensor alive, so a temporary seed
        # (Dropout.make(torch.tensor(...), ...)) is not freed and its memory reused by the time a kernel reads it
        d._seed_tensor = seed_tensor
        return d


class GemmDesc(C.Structure):
    """neko_gemm_desc (include/neko_b200.h)."""
    _fields_ = [("M", C.c_int32), ("N", C.c_int32), ("K", C.c_int32), ("a_mn", C.c_int32), ("b_mn", C.c_int32),
                ("epilogue", C.c_int32), ("accumulate", C.c_int32), ("flags", C.c_int32),
                ("A", C.c_void_p), ("lda", C.c_int64), ("B", C.c_void_p), ("ldb", C.c_int64),
                ("C", C.c_void_p), ("ldc", C.c_int64), ("C2", C.c_void_p), ("ldc2", C.c_int64),
                ("C3", C.c_void_p), ("ldc3", C.c_int64), ("bias", C.c_void_p), ("aux", C.c_void_p), ("ld_aux", C.c_int64),
                ("drop", Dropout), ("workspace", C.c_void_p), ("workspace_bytes", C.c_int64)]


class GemmPlanInfo(C.Structure):
    """neko_gemm_plan_info (include/neko_b200.h)."""
    _fields_ = [(n, C.c_int32) for n in (
        "BN", "pair", "splits", "epi_warps", "streamk", "tma_store", "tma_aux", "vec_ok", "n_fast", "stages")]


class LnBwdPathInfo(C.Structure):
    """neko_layernorm_bwd_path_info (include/neko_b200.h)."""
    _fields_ = [(n, C.c_int32) for n in ("grid", "rows_per_cta", "stages")]


EPI_BF16, EPI_F32, EPI_GELU_BF16, EPI_RESID_F32, EPI_DGELU_BF16, EPI_RESID_F32_BF16 = range(6)

_lib = None


def declared_symbols():
    """Every function include/neko_b200.h declares (used by the CPU-side export test)."""
    txt = open(HEADER).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    return sorted(set(re.findall(r"\b(neko_[a-z0-9_]+)\s*\(", txt)))


def load():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise NekoError(f"{LIB_PATH} is missing: run `python -m neko_b200.build` (or __graft_entry__.build()). "
                        "There is no CPU fallback for the hot path.")
    lib = C.CDLL(LIB_PATH)
    lib.neko_last_error.restype = C.c_char_p
    for name in declared_symbols():
        fn = getattr(lib, name)  # AttributeError here = header / library mismatch
        if name == "neko_gemm_workspace_bytes" or name.endswith("_workspace_bytes"):
            fn.restype = C.c_int64
        elif name != "neko_last_error":
            fn.restype = C.c_int
    _lib = lib
    return lib


def _p(x):
    """tensor / int / None -> void*"""
    if x is None:
        return C.c_void_p(0)
    if isinstance(x, int):
        return C.c_void_p(x)
    return C.c_void_p(x.data_ptr())


def check(rc: int, what: str = ""):
    if rc != 0:
        msg = load().neko_last_error().decode()
        raise NekoError(f"{what} failed (code {rc}): {msg}")


def stream_ptr():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def require_device():
    check(load().neko_device_check(), "neko_device_check")

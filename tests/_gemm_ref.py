"""fp64 reference of the neko_gemm epilogues and the per-element check of a kernel output against it.

tests/test_gemm_check_cpu.py shows that the check passes exactly rounded results and rejects subtly wrong ones;
tests/test_gemm_matrix_gpu.py runs it on every schedule of the GEMM.  Works on CPU and CUDA tensors alike.

Bound per output element (fp32 outputs):  C_ACC * sqrt(K) * 2^-24 * mag + 2^-23 * |ref| + fn_err
  mag    = the magnitude the fp32 evaluation rounds: (|A| |B|^T)[m, n] plus the |addends| of the epilogue (bias, residual,
           accumulated C), scaled by the dropout multiplier and by the slope of GELU / GELU' where those follow;
  fn_err = allowance for the kernel's fp32 GELU / GELU' approximations (erf to 1.5e-7, ex2 / rcp to 2^-22), zero elsewhere.
16-bit outputs add half an ulp of the output format at |ref| (round to nearest even; fp16 saturates at 65504).
"""
from __future__ import annotations

import math
from typing import NamedTuple, Optional

import torch

EPI_BF16, EPI_F32, EPI_GELU_BF16, EPI_RESID_F32, EPI_DGELU_BF16, EPI_RESID_F32_BF16 = range(6)

C_ACC = 4.0          # c of the accumulation term
GELU_SLOPE = 1.13    # max |d gelu / dx| (erf: 1.1289, tanh form: 1.1289)
FN_REL = 2.0 ** -20  # GELU / GELU' approximation allowance per unit of |x| (and of 1 for GELU')

# (mantissa bits incl. the implicit one, smallest normal exponent, largest finite value)
FORMATS = {"bf16": (8, -126, 3.3895313892515355e38), "f16": (11, -14, 65504.0)}
TORCH_FMT = {torch.bfloat16: "bf16", torch.float16: "f16", torch.float32: "f32"}


class Expected(NamedTuple):
    ref: torch.Tensor                     # fp64 value of the output
    mag: torch.Tensor                     # fp64, see the module docstring
    fn_err: Optional[torch.Tensor]        # fp64 or None
    fmt: str                              # "f32", "bf16" or "f16"


# ---------------------------------------------------------------------------------------------------
# GELU in fp64
# ---------------------------------------------------------------------------------------------------
_K_TANH = math.sqrt(2.0 / math.pi)


def gelu64(x: torch.Tensor, tanh: bool) -> torch.Tensor:
    if tanh:
        return 0.5 * x * (1.0 + torch.tanh(_K_TANH * (x + 0.044715 * x ** 3)))
    return 0.5 * x * (1.0 + torch.erf(x / math.sqrt(2.0)))


def gelu_grad64(x: torch.Tensor, tanh: bool) -> torch.Tensor:
    if tanh:
        t = torch.tanh(_K_TANH * (x + 0.044715 * x ** 3))
        return 0.5 * (1.0 + t) + 0.5 * x * (1.0 - t * t) * _K_TANH * (1.0 + 3.0 * 0.044715 * x * x)
    return 0.5 * (1.0 + torch.erf(x / math.sqrt(2.0))) + x * torch.exp(-0.5 * x * x) / math.sqrt(2.0 * math.pi)


# ---------------------------------------------------------------------------------------------------
# 16-bit rounding in fp64 (exact: scaling by a power of two, then an integer rounding)
# ---------------------------------------------------------------------------------------------------
def _ulp(x: torch.Tensor, fmt: str) -> torch.Tensor:
    p, emin, _ = FORMATS[fmt]
    _, e = torch.frexp(x.abs())                    # |x| = m 2^e, m in [0.5, 1)
    e = torch.where(x == 0, torch.full_like(e, emin), e - 1).clamp(min=emin)
    return torch.ldexp(torch.ones_like(x), e - (p - 1))


def round16(x: torch.Tensor, fmt: str, mode: str = "rne") -> torch.Tensor:
    """fp64 x rounded to bf16 / f16 (round to nearest even, or 'trunc' toward zero), returned as fp64.
    f16 saturates at +-65504 as the kernels' conversions do."""
    x = x.double()
    _, _, fmax = FORMATS[fmt]
    if fmt == "f16":
        x = x.clamp(-fmax, fmax)
    u = _ulp(x, fmt)
    q = torch.round(x / u) if mode == "rne" else torch.trunc(x / u)
    return q * u


def half_ulp(x: torch.Tensor, fmt: str) -> torch.Tensor:
    return 0.5 * _ulp(x, fmt)


def exact_output(exp: Expected) -> torch.Tensor:
    """The correctly rounded output (what an error-free kernel would write), fp64."""
    if exp.fmt == "f32":
        return exp.ref.float().double()
    return round16(exp.ref, exp.fmt)


# ---------------------------------------------------------------------------------------------------
# reference
# ---------------------------------------------------------------------------------------------------
def accumulator(a: torch.Tensor, b: torch.Tensor):
    """a [M, K], b [N, K] (16-bit, logical orientation) -> (A B^T, |A| |B|^T) in fp64, exact for K < 2^20."""
    a64, b64 = a.double(), b.double()
    return a64 @ b64.t(), a64.abs() @ b64.abs().t()


def epilogue_reference(acc: torch.Tensor, absacc: torch.Tensor, epi: int, *, bias=None, aux=None, mult=None, c_init=None,
                       gelu_tanh: bool = False, c_fmt: str = "bf16", c2_fmt: str = "bf16", c3: bool = False) -> dict:
    """Expected outputs {'C', 'C2', 'C3'} of one neko_gemm call.

    acc, absacc: fp64 [M, N] from accumulator(); bias [N]; aux [M, N] (fp32 residual or bf16 GELU input); mult [M, N]: the
    dropout multipliers (0 or 1 / (1 - p)) of the RESID epilogues; c_init: C before an accumulating EPI_F32 call;
    c_fmt / c2_fmt: output formats of the 16-bit outputs."""
    pre = acc
    mag = absacc
    if bias is not None:
        b = bias.double().reshape(1, -1)
        pre = pre + b
        mag = mag + b.abs()
    out = {}
    if epi == EPI_BF16:
        out["C"] = Expected(pre, mag, None, c_fmt)
    elif epi == EPI_F32:
        if c_init is not None:
            ci = c_init.double()
            pre, mag = pre + ci, mag + ci.abs()
        out["C"] = Expected(pre, mag, None, "f32")
    elif epi == EPI_GELU_BF16:
        out["C"] = Expected(pre, mag, None, c_fmt)
        g = gelu64(pre, gelu_tanh)
        fn = FN_REL * pre.abs()
        out["C2"] = Expected(g, GELU_SLOPE * mag, fn, c2_fmt)
        if c3:
            out["C3"] = Expected(g, GELU_SLOPE * mag, fn, "bf16")
    elif epi == EPI_DGELU_BF16:
        assert bias is None, "EPI_DGELU_BF16 takes no bias"
        x = aux.double()
        gp = gelu_grad64(x, gelu_tanh)
        out["C"] = Expected(acc * gp, absacc * gp.abs(), FN_REL * (1.0 + x.abs()) * acc.abs(), c_fmt)
    elif epi in (EPI_RESID_F32, EPI_RESID_F32_BF16):
        if mult is not None:
            m = mult.double()
            pre, mag = pre * m, mag * m.abs()
        r = aux.double()
        v, mag = pre + r, mag + r.abs()
        out["C"] = Expected(v, mag, None, "f32")
        if epi == EPI_RESID_F32_BF16:
            out["C2"] = Expected(v, mag, None, c2_fmt)
    else:
        raise ValueError(f"unknown epilogue {epi}")
    return out


# ---------------------------------------------------------------------------------------------------
# check
# ---------------------------------------------------------------------------------------------------
def bound(exp: Expected, K: int) -> torch.Tensor:
    tol = C_ACC * math.sqrt(K) * 2.0 ** -24 * exp.mag + 2.0 ** -23 * exp.ref.abs()
    if exp.fn_err is not None:
        tol = tol + exp.fn_err
    if exp.fmt != "f32":
        tol = tol + half_ulp(exp.ref, exp.fmt)
    return tol


def violations(out: torch.Tensor, exp: Expected, K: int) -> torch.Tensor:
    """Boolean [M, N]: elements of `out` outside the bound (NaN counts as outside)."""
    if out.dtype in TORCH_FMT:
        assert TORCH_FMT[out.dtype] == exp.fmt, f"output is {out.dtype}, reference expects {exp.fmt}"
    err = (out.double() - exp.ref).abs()
    return ~(err <= bound(exp, K))


def assert_within(out: torch.Tensor, exp: Expected, K: int, what: str = "output"):
    bad = violations(out, exp, K)
    n = int(bad.sum())
    if n:
        idx = bad.nonzero()[:5].tolist()
        tol = bound(exp, K)
        detail = ", ".join(f"[{m},{c}] got {float(out[m, c]):.9g} ref {float(exp.ref[m, c]):.9g} bound {float(tol[m, c]):.3g}"
                           for m, c in idx)
        raise AssertionError(f"{what}: {n} of {bad.numel()} elements outside the bound: {detail}")

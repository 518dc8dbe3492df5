"""fp64 references of the row kernels (LayerNorm forward / backward, masked cross entropy, GeGLU, casts), per-element error
bounds derived from how the kernels round, the check of a kernel output against them, and kernel-faithful fp32 emulations.

tests/test_rowops_check_cpu.py shows that the check accepts correctly rounded results and the emulations and rejects subtly
wrong ones; tests/test_rowops_matrix_gpu.py runs it on every kernel.  CPU and CUDA tensors.  u = 2^-24 (fp32 unit
roundoff); a 16-bit output adds half an ulp of its format, taken at |ref| + the fp32 bound (the fp32 value may sit in the
next binade up); fp16 saturates at +-65504 (cvt.rn.satfinite), so its reference is clamped there.

LayerNorm forward (warp per row, NV = ceil(d / 128) float4 per lane).  Reference: fp64 mean mu, biased variance var,
rstd = 1 / sqrt(var + eps), y = (x - mu) rstd gamma + beta.
  mean   each lane adds 2 NV values in its own registers, then 5 shuffle levels: depth D = 2 NV + 5, so the fp32 sum is
         within D u sum|x|; the division adds u |mu|:          tol_mu = D u mean|x| + u |mu|.
  rstd   sum (x - mu')^2 with mu' = mu + dmu equals d var + d dmu^2, so the mean's error enters squared; each term carries
         the subtraction and the square (3u), the sum D u, the /d and the +eps one u each, rsqrtf 2 ulp (4u):
         rel_rstd = ((D + 4) u var + dmu^2) / (2 (var + eps)) + u + 4u,  with dmu = tol_mu.
  y      |x - mu| |gamma| rstd (rel_rstd + 4u) + |dmu| rstd |gamma| + u |beta|, plus half an ulp of the output format.
  y2     (bf16 copy of the same fp32 value) within half a bf16 ulp plus half an fp16 ulp of y, and equal to y bit for bit
         when y is bf16.
LayerNorm backward, given the kernel's saved mean / rstd (the forward bounds cover those).  x^ = (x - mean) rstd,
gy = gamma dy, m1 = mean(gy), m2 = mean(gy x^), dx_resid_out = dx_in + rstd (gy - m1 - x^ m2).
  x^ carries 2u |x^| (subtraction, product), gy u |gy|.  The row sums have depth D_b = NV + 8, the larger of the
  warp-per-row tree (NV + 2 in-lane adds, 5 shuffles) and the column-owner tree (2 in-thread adds, 5 shuffles, one add per
  warp): dm1 = (D_b + 3) u mean|gy|, dm2 = (D_b + 5) u mean|gy x^| + 2u |m2|.  With A = |gy| + |m1| + |x^| |m2|:
  tol_dx = rstd (u |gy| + dm1 + |x^| dm2 + 2u |x^| |m2| + 5u A) + u (|dx_in| + rstd A).
  dx_bf16 is exact: round_bf16(fl32(dx_resid_out_kernel * mult)), mult the fp32 dropout multiplier (0 or 1/(1-p)); the
  fp32 dx_resid stays unmasked.  dgamma / dbeta / dx_colsum are sums over N rows accumulated into their initial values:
  (N + k) u (|init| + sum |term|), k = 8 covering the rounding of each term (dy x^: 3u; dx mult: u).
Cross entropy.  The reference is fp64 on the exact input values (an fp16 logit is exact in fp64: its rounding is an input,
not an error).  lse = logsumexp(z), row_loss = lse - z_t, dlogits = (p - [j = t]) g / n_rows, p = exp(z - lse).
  exp    __expf(x) = ex2.approx(x log2e): 2^-21 relative, plus u |x| log2e from the argument product and u |x| from the
         subtraction that formed x; |x| <= R, the row's range max - min.  ce_fwd_kernel rescales its running sum once
         per element a thread visits at most (c = ceil(V / 256)) and once per merge (5 shuffle + 7 block levels); the
         rescale arguments telescope along the rising maximum (their total |x| is at most R again), each rescale adds an
         exponential (2^-21) and a product (u).  The fused kernels exponentiate against the exact maximum once.
         rel_e = (r + 1) 2^-21 + 4 u R log2e,   r = rescales.
  sum    depth c + 40 (per-thread adds, 5 shuffles, 32 warp partials) plus one product per rescale: rel_s = rel_e + (c + 40 + r) u.
  lse    rel_s + 2u |ln s| (logf) + u (|lse| + |max|).    row_loss: tol_lse + u |loss|; exactly 0 for an out-of-range target.
  loss   ce_mean_kernel sums in fp64 and rounds once: within u |loss| (+ fp64 slack) of the fp64 mean of the kernel's row_loss.
  dlog   (g / n) (p (tol_lse + rel_e + 4u) + 3u |p - [j = t]| + 2^-126) + half_ulp_bf16: per element, so a tiny entry needs
         a tiny error; 2^-126 covers ex2.approx.ftz flushing p to zero.
  ce_scale_grad is exact: round_bf16(fl32(d g)), and a no-op when g is exactly 1.  The fused path plus the scale therefore
         rounds to bf16 twice: its bound is g times the unscaled bound plus a second half ulp at the scaled value.
GeGLU.  A bf16 x bf16 or fp16 x bf16 product is exact in fp32, so out == round16(a g) and out_bf16 == round_bf16(a g) bit
for bit.  Backward: d_gate = dh gelu(pre), d_pre = dh gate gelu'(pre) (erf form), each within FN_REL (the fp32 GELU / GELU'
approximation allowance of _gemm_ref) times |dh| |pre| (d_gate) or |dh gate| (1 + |pre|) (d_pre), plus 3u |ref| and half
a bf16 ulp.
Casts: cast_f32_to_f16 / cast_f32_to_bf16 / cast_f32_to_f16_bf16 are exact: round16(x).
"""
from __future__ import annotations

import math
from typing import NamedTuple, Optional

import torch

from _gemm_ref import FN_REL, gelu64, gelu_grad64, half_ulp, round16  # noqa: F401  (re-exported for the tests)

U = 2.0 ** -24
EX2 = 2.0 ** -21
FTZ = 2.0 ** -126
LOG2E = 1.0 / math.log(2.0)
F16_MAX = 65504.0
TORCH_FMT = {torch.bfloat16: "bf16", torch.float16: "f16", torch.float32: "f32"}
CE_THREADS, CEF_THREADS = 256, 1024


class Expected(NamedTuple):
    ref: torch.Tensor        # fp64 value (clamped to +-65504 for fp16 outputs)
    tol: torch.Tensor        # fp64 per-element bound
    fmt: str                 # "f32", "bf16" or "f16"


def _out(ref: torch.Tensor, tol32: torch.Tensor, fmt: str) -> Expected:
    """Expected of an output whose fp32 value is within tol32 of ref, rounded to fmt."""
    if fmt == "f32":
        return Expected(ref, tol32, fmt)
    if fmt == "f16":
        ref = ref.clamp(-F16_MAX, F16_MAX)
    return Expected(ref, tol32 + half_ulp(ref.abs() + tol32, fmt), fmt)


def to16(x: torch.Tensor, fmt: str) -> torch.Tensor:
    """round16 as a 16-bit tensor (exact: round16 returns representable values)."""
    return round16(x, fmt).to(torch.bfloat16 if fmt == "bf16" else torch.float16)


# ---------------------------------------------------------------------------------------------------
# LayerNorm
# ---------------------------------------------------------------------------------------------------
def ln_nv(d: int) -> int:
    return (d // 4 + 31) // 32


def ln_forward(x, gamma, beta, eps: float, out_fmt: str = "bf16") -> dict:
    """Expected mean, rstd (fp32), y (out_fmt) and y2 (bf16) of neko_layernorm_fwd."""
    x64, g, b = x.double(), gamma.double(), beta.double()
    d = x.shape[-1]
    D = 2 * ln_nv(d) + 5
    mu = x64.mean(-1)
    xc = x64 - mu[:, None]
    var = (xc * xc).mean(-1)
    rstd = 1.0 / torch.sqrt(var + eps)
    y = xc * rstd[:, None] * g + b
    tol_mu = D * U * x64.abs().mean(-1) + U * mu.abs()
    rel_rstd = ((D + 4) * U * var + tol_mu ** 2) / (2 * (var + eps)) + 5 * U
    tol_rstd = rel_rstd * rstd
    tol_y = (xc.abs() * g.abs() * rstd[:, None] * (rel_rstd[:, None] + 4 * U) + (tol_mu * rstd)[:, None] * g.abs()
             + U * b.abs())
    return {"mean": Expected(mu, tol_mu, "f32"), "rstd": Expected(rstd, tol_rstd, "f32"),
            "y": _out(y, tol_y, out_fmt), "y2": _out(y, tol_y, "bf16")}


def ln_y2_mismatch(y: torch.Tensor, y2: torch.Tensor) -> torch.Tensor:
    """Boolean: elements where the bf16 copy y2 does not match y (bit for bit when y is bf16; otherwise both round one fp32
    value, so they are within half a bf16 plus half an fp16 ulp, taken one binade up)."""
    if y.dtype == torch.bfloat16:
        return y.view(torch.int16) != y2.view(torch.int16)
    a, b = y.double(), y2.double()
    top = 2 * a.abs()
    tol = half_ulp(top, "bf16") + half_ulp(top, "f16")
    return ~((a - b).abs() <= tol) & ~((a.abs() == F16_MAX) & (b.abs() >= F16_MAX))


def ln_backward(dy, x, gamma, mean, rstd, dx_in, mult=None, dgamma0=None, dbeta0=None, colsum0=None, dx_out_kernel=None) -> dict:
    """Expected dx_resid (fp32), dx_bf16 (exact, from the kernel's own dx_resid), dgamma / dbeta / dx_colsum (accumulated
    into the given initial values) of neko_layernorm_bwd given the kernel's saved mean / rstd.  mult: fp64/fp32 [N, d]
    dropout multipliers of branch_drop (None = no dropout).  dx_out_kernel: the kernel's dx_resid, which the exact dx_bf16
    and the colsum reference are built from (default: the reference value)."""
    N, d = x.shape
    Db = ln_nv(d) + 8
    dy64, x64, g = dy.double(), x.double(), gamma.double()
    mu, r = mean.double()[:, None], rstd.double()[:, None]
    xh = (x64 - mu) * r
    gy = g * dy64
    m1 = gy.mean(-1, keepdim=True)
    m2 = (gy * xh).mean(-1, keepdim=True)
    dx = r * (gy - m1 - xh * m2)
    out = dx_in.double() + dx
    dm1 = (Db + 3) * U * gy.abs().mean(-1, keepdim=True)
    dm2 = (Db + 5) * U * (gy * xh).abs().mean(-1, keepdim=True) + 2 * U * m2.abs()
    A = gy.abs() + m1.abs() + xh.abs() * m2.abs()
    tol = r * (U * gy.abs() + dm1 + xh.abs() * dm2 + 2 * U * xh.abs() * m2.abs() + 5 * U * A) + U * (dx_in.double().abs() + r * A)
    res = {"dx": Expected(out, tol, "f32")}
    dk = (out if dx_out_kernel is None else dx_out_kernel).float()
    m32 = torch.ones_like(dk) if mult is None else mult.float()
    masked = dk * m32                                   # fl32 product, as the kernel rounds it
    res["dx_bf16"] = masked.to(torch.bfloat16)
    k = N + 8

    def colsum(terms, init):
        i = torch.zeros(d, dtype=torch.float64, device=x.device) if init is None else init.double()
        return Expected(i + terms.sum(0), k * U * (i.abs() + terms.abs().sum(0)), "f32")

    res["dgamma"] = colsum(dy64 * xh, dgamma0)
    res["dbeta"] = colsum(dy64, dbeta0)
    res["colsum"] = colsum(masked.double(), colsum0)
    return res


# ---------------------------------------------------------------------------------------------------
# cross entropy
# ---------------------------------------------------------------------------------------------------
CE_KERNELS = ("two_pass", "fused", "fused_f16")


def ce_reference(z: torch.Tensor, tgt: torch.Tensor, n_rows: int, g: float = 1.0, kernel: str = "two_pass") -> dict:
    """Expected lse, row_loss and dlogits [n, V] (bf16, scaled by g) of the selected rows z [n, V] (their exact values) with
    targets tgt [n] (out-of-range allowed).  kernel: which kernel's rescale count and summation depth the bound uses."""
    z64 = z.double()
    n, V = z64.shape
    mx = z64.amax(-1)
    R = mx - z64.amin(-1)
    lse = torch.logsumexp(z64, -1)
    c = -(-V // (CE_THREADS if kernel == "two_pass" else CEF_THREADS))
    resc = c + 12 if kernel == "two_pass" else 0
    rel_e = (resc + 1) * EX2 + 4 * U * R * LOG2E
    rel_s = rel_e + (c + 40 + resc) * U
    tol_lse = rel_s + 2 * U * (lse - mx).abs() + U * (lse.abs() + mx.abs())
    t = tgt.long().to(z64.device)
    valid = (t >= 0) & (t < V)
    zt = torch.gather(z64, 1, t.clamp(0, V - 1)[:, None]).squeeze(1)
    loss = torch.where(valid, lse - zt, torch.zeros_like(lse))
    tol_loss = torch.where(valid, tol_lse + U * loss.abs(), torch.zeros_like(lse))
    p = torch.exp(z64 - lse[:, None])
    onehot = torch.zeros_like(p)
    onehot[valid.nonzero().squeeze(1), t[valid]] = 1.0
    s = g / n_rows
    ref = (p - onehot) * s
    tol = s * (p * (tol_lse[:, None] + rel_e[:, None] + 4 * U) + 3 * U * (p - onehot).abs() + FTZ)
    return {"lse": Expected(lse, tol_lse, "f32"), "row_loss": Expected(loss, tol_loss, "f32"),
            "dlogits": _out(ref, tol, "bf16"), "_unscaled_tol": tol / s}


def ce_scaled(unscaled: Expected, g: float) -> Expected:
    """Bound of the fused path's bf16 gradient after ce_scale_grad by g: g times the unscaled bound (that includes its
    half ulp), the fl32 product, and a second bf16 rounding."""
    ref = unscaled.ref * g
    tol32 = unscaled.tol * abs(g) + U * ref.abs()
    return Expected(ref, tol32 + half_ulp(ref.abs() + tol32, "bf16"), "bf16")


def ce_loss_expected(row_loss_kernel: torch.Tensor) -> Expected:
    """loss = fp64 mean of the kernel's own row_loss, rounded to fp32 once."""
    m = row_loss_kernel.double().mean()
    return Expected(m, U * m.abs() + 1e-12 * row_loss_kernel.double().abs().mean(), "f32")


def ce_scale_exact(d: torch.Tensor, g: float) -> torch.Tensor:
    """What neko_ce_scale_grad writes: round_bf16(fl32(d * g)), d itself when g == 1."""
    if g == 1.0:
        return d.clone()
    return (d.float() * torch.tensor(g, dtype=torch.float32)).to(torch.bfloat16)


# ---------------------------------------------------------------------------------------------------
# GeGLU and casts
# ---------------------------------------------------------------------------------------------------
def geglu_fwd_exact(act: torch.Tensor, gate: torch.Tensor, out_fmt: str):
    """(out, out_bf16) as 16-bit tensors: the fp32 product is exact, so each is the correctly rounded a * g."""
    prod = act.double() * gate.double()
    return to16(prod, out_fmt), to16(prod, "bf16")


def geglu_bwd(dh, pre, gate) -> dict:
    dh64, p, g = dh.double(), pre.double(), gate.double()
    ge, gp = gelu64(p, False), gelu_grad64(p, False)
    d_gate = dh64 * ge
    d_pre = dh64 * g * gp
    t_gate = FN_REL * (dh64 * p).abs() + 3 * U * d_gate.abs()
    t_pre = FN_REL * (dh64 * g).abs() * (1 + p.abs()) + 3 * U * d_pre.abs()
    return {"d_gate": _out(d_gate, t_gate, "bf16"), "d_pre": _out(d_pre, t_pre, "bf16")}


def cast_exact(src: torch.Tensor, fmt: str) -> torch.Tensor:
    return to16(src.double(), fmt)


# ---------------------------------------------------------------------------------------------------
# check
# ---------------------------------------------------------------------------------------------------
def violations(out: torch.Tensor, exp: Expected) -> torch.Tensor:
    """Boolean, shaped like out: elements outside the bound (NaN and inf are outside)."""
    if out.dtype in TORCH_FMT:
        assert TORCH_FMT[out.dtype] == exp.fmt, f"output is {out.dtype}, reference expects {exp.fmt}"
    return ~((out.double() - exp.ref).abs() <= exp.tol)


def worst_ratio(out: torch.Tensor, exp: Expected) -> float:
    """max err / bound over the elements with a non-zero bound (the headroom of the check)."""
    m = exp.tol > 0
    if not bool(m.any()):
        return 0.0
    return float(((out.double() - exp.ref).abs()[m] / exp.tol[m]).max())


def assert_within(out: torch.Tensor, exp: Expected, what: str = "output"):
    bad = violations(out, exp)
    n = int(bad.sum())
    if n:
        o = out.double()
        excess = torch.where(bad, ((o - exp.ref).abs() - exp.tol).nan_to_num(math.inf), torch.full_like(o, -math.inf))
        idx = tuple(int(i) for i in torch.unravel_index(excess.argmax(), excess.shape))
        raise AssertionError(f"{what}: {n} of {bad.numel()} elements outside the bound; worst at {idx}: got {float(o[idx]):.9g} "
                             f"ref {float(exp.ref[idx]):.9g} bound {float(exp.tol[idx]):.3g}")


def assert_bits(out: torch.Tensor, want: torch.Tensor, what: str = "output"):
    """Bit-for-bit equality of two 16-bit tensors (+0 and -0 differ; a NaN never matches)."""
    assert out.dtype == want.dtype, (what, out.dtype, want.dtype)
    bad = out.view(torch.int16) != want.view(torch.int16)
    n = int(bad.sum())
    if n:
        idx = tuple(int(i) for i in bad.nonzero()[0])
        raise AssertionError(f"{what}: {n} of {bad.numel()} elements differ; first at {idx}: got {float(out[idx])!r} "
                             f"want {float(want[idx])!r}")


# ---------------------------------------------------------------------------------------------------
# kernel-faithful emulations (fp32)
# ---------------------------------------------------------------------------------------------------
def _lanes(v: torch.Tensor, d: int) -> torch.Tensor:
    """[N, d] -> [N, NV, 32, 4]: lane l owns the float4 groups l, l + 32, ... (zeros past d; adding 0 is exact)."""
    N = v.shape[0]
    nv = ln_nv(d)
    pad = torch.zeros(N, nv * 128, dtype=v.dtype, device=v.device)
    pad[:, :d] = v
    return pad.reshape(N, nv, 32, 4)


def _lane_sum(t: torch.Tensor) -> torch.Tensor:
    """[N, NV, 32, 4] -> [N, 32]: s += (a + b) + (c + d) over the groups of a lane, in order."""
    s = torch.zeros(t.shape[0], 32, dtype=t.dtype, device=t.device)
    for k in range(t.shape[1]):
        q = t[:, k]
        s = s + ((q[..., 0] + q[..., 1]) + (q[..., 2] + q[..., 3]))
    return s


def _warp_sum(s: torch.Tensor) -> torch.Tensor:
    """butterfly over the 32 lanes (__shfl_xor_sync 16, 8, 4, 2, 1); every lane ends with the same value."""
    lane = torch.arange(32, device=s.device)
    for o in (16, 8, 4, 2, 1):
        s = s + s[:, lane ^ o]
    return s[:, 0]


def emulate_ln_fwd(x, gamma, beta, eps: float, out_fmt: str = "bf16", mutant: Optional[str] = None):
    """layernorm_fwd_kernel in fp32.  Returns (y, y2, mean, rstd).  mutant (for the strictness tests): 'unbiased',
    'eps_outside', 'mean_dm1', 'gamma_shift', 'stale_tail', 'f16_inf'."""
    x = x.float()
    N, d = x.shape
    dd = torch.tensor(float(d - 1 if mutant == "mean_dm1" else d), dtype=torch.float32)
    mean = _warp_sum(_lane_sum(_lanes(x, d))) / dd
    xc = x - mean[:, None]
    var = _warp_sum(_lane_sum(_lanes(xc * xc, d))) / torch.tensor(float(d - 1 if mutant == "unbiased" else d), dtype=torch.float32)
    e = torch.tensor(eps, dtype=torch.float32)
    rstd = torch.rsqrt(var) + e if mutant == "eps_outside" else torch.rsqrt(var + e)
    g, b = gamma.float(), beta.float()
    if mutant == "gamma_shift":
        g, b = torch.roll(g, -4), torch.roll(b, -4)
    o = (xc * rstd[:, None]) * g + b
    dt = torch.bfloat16 if out_fmt == "bf16" else torch.float16
    y = o.to(dt) if (out_fmt == "bf16" or mutant == "f16_inf") else to16(o, "f16")
    y2 = o.to(torch.bfloat16)
    if mutant == "stale_tail":
        c0 = (d - 1) // 128 * 128
        y[:, c0:] = 0
        y2[:, c0:] = 0
    return y, y2, mean, rstd


def emulate_ln_bwd(dy, x, gamma, mean, rstd, dx_in, mult=None, mutant: Optional[str] = None):
    """layernorm_bwd_rows_kernel in fp32 (one warp per row).  Returns dict dx, dx_bf16, dgamma, dbeta, colsum (column sums
    in row order, as one warp would add them).  mutant: 'no_m2', 'm1_dm1', 'mask_fp32', 'bf16_before_add', 'colsum_unmasked',
    'dgamma_x', 'skip_last_block'."""
    N, d = x.shape
    x, dyf, g = x.float(), dy.float(), gamma.float()
    mu, rs = mean.float()[:, None], rstd.float()[:, None]
    xh = (x - mu) * rs
    gy = dyf * g
    inv_d = torch.tensor(1.0, dtype=torch.float32) / torch.tensor(float(d - 1 if mutant == "m1_dm1" else d), dtype=torch.float32)
    inv_d2 = torch.tensor(1.0, dtype=torch.float32) / torch.tensor(float(d), dtype=torch.float32)
    m1 = _warp_sum(_lane_sum(_lanes(gy, d)))[:, None] * inv_d
    m2 = _warp_sum(_lane_sum(_lanes(gy * xh, d)))[:, None] * inv_d2
    if mutant == "no_m2":
        m2 = torch.zeros_like(m2)
    delta = rs * (gy - m1 - xh * m2)
    out = dx_in.float() + delta
    m32 = torch.ones_like(out) if mult is None else mult.float()
    if mutant == "skip_last_block":
        r0 = (N - 1) // 4 * 4
        out[r0:] = dx_in.float()[r0:]
    masked = out * m32
    dx = masked if mutant == "mask_fp32" else out
    dxb = (delta * m32 if mutant == "bf16_before_add" else masked).to(torch.bfloat16)
    col_terms = out if mutant == "colsum_unmasked" else masked
    dg_terms = dyf * (x if mutant == "dgamma_x" else xh)
    acc = lambda t: t.cumsum(0)[-1] if t.shape[0] else torch.zeros(d)  # noqa: E731
    return {"dx": dx, "dx_bf16": dxb, "dgamma": acc(dg_terms), "dbeta": acc(dyf), "colsum": acc(col_terms)}


def emulate_ce(z: torch.Tensor, tgt: torch.Tensor, n_rows: int, kernel: str = "two_pass", mutant: Optional[str] = None):
    """The CE kernels in fp32 on the selected rows z [n, V] (fp32 values, or fp16 for fused_f16).  two_pass: ce_fwd_kernel
    (online max / sum per thread, float4 steps, shuffle and block merges) then ce_bwd_kernel with g = 1; fused / fused_f16:
    maximum, exp against it, sum, (softmax - onehot) / n_rows.  Returns (lse, row_loss, dlogits bf16).
    mutant: 'lse_plus', 'log2', 'drop_rescale', 'onehot_next', 'n_minus_1', 'stale_tail', 'f16_as_bf16'."""
    zf = z.float() if mutant != "f16_as_bf16" else z.view(torch.bfloat16).float()
    n, V = zf.shape
    dev = zf.device
    t = tgt.long().to(dev)
    if kernel == "two_pass":
        T = CE_THREADS
        m = torch.full((n, T), -math.inf, device=dev)
        s = torch.zeros(n, T, device=dev)
        nv = V // 4
        steps = []
        for i0 in range(0, nv, T):                                # vector part: thread j takes float4 i0 + j
            ids = torch.arange(min(T, nv - i0), device=dev)
            steps.append((ids, zf[:, 4 * i0:4 * (i0 + len(ids))].reshape(n, len(ids), 4)))
        for i0 in range(4 * nv, V, T):                            # scalar tail
            ids = torch.arange(i0, min(i0 + T, V), device=dev) - i0
            steps.append((ids, zf[:, i0:i0 + T][..., None]))
        for k, (ids, v) in enumerate(steps):
            mo, so = m[:, ids], s[:, ids]
            mn = torch.maximum(mo, v.amax(-1))
            corr = torch.exp(mo - mn)
            if mutant == "drop_rescale" and k == len(steps) - 1:
                corr = torch.ones_like(corr)
            e = torch.exp(v - mn[..., None])
            acc = so * corr
            for j in range(v.shape[-1]):
                acc = acc + e[..., j]
            m[:, ids], s[:, ids] = mn, acc

        def merge(m, s, m2, s2):
            mn = torch.maximum(m, m2)
            dead = mn == -math.inf
            sm = s * torch.exp(torch.where(dead, 0.0, m - mn)) + s2 * torch.exp(torch.where(dead, 0.0, m2 - mn))
            return mn, torch.where(dead, torch.zeros_like(sm), sm)

        m, s = m.reshape(n, T // 32, 32), s.reshape(n, T // 32, 32)
        lane = torch.arange(32, device=dev)
        for o in (16, 8, 4, 2, 1):
            m, s = merge(m, s, m[..., lane ^ o], s[..., lane ^ o])
        m, s = m[..., 0], s[..., 0]
        M, S = m[:, 0], s[:, 0]
        for w in range(1, T // 32):
            M, S = merge(M, S, m[:, w], s[:, w])
        lse = M + torch.log(S)
    else:
        mx = zf.amax(-1)
        e = torch.exp(zf - mx[:, None])
        S = e.sum(-1)
        lse = mx + torch.log(S)
    if mutant == "lse_plus":
        lse = lse + 0.01
    if mutant == "log2":
        lse = lse * torch.tensor(LOG2E, dtype=torch.float32)
    valid = (t >= 0) & (t < V)
    zt = torch.gather(zf, 1, t.clamp(0, V - 1)[:, None]).squeeze(1)
    loss = torch.where(valid, lse - zt, torch.zeros_like(lse))
    nn = n_rows - 1 if mutant == "n_minus_1" else n_rows
    inv_n = torch.tensor(1.0, dtype=torch.float32) / torch.tensor(float(nn), dtype=torch.float32)
    tt = t + 1 if mutant == "onehot_next" else t
    onehot = (torch.arange(V, device=dev)[None, :] == tt[:, None]).float()
    p = torch.exp(zf - lse[:, None])
    d = (p * inv_n - onehot * inv_n).to(torch.bfloat16)
    if mutant == "stale_tail":
        w = 8 if kernel == "fused_f16" else 4
        c0 = V // w * w
        d[:, c0:] = 0
    return lse, loss, d


def ce_dlogits_violations(buf: torch.Tensor, prefill: torch.Tensor, exp: Expected, rows: torch.Tensor, V: int, compact: bool,
                          zero_pad: bool) -> int:
    """Number of wrong elements of a whole dlogits buffer [R, ld] (bf16) after a CE call: the selected rows' first V columns
    within the bound, their pad columns V..ld zero under NEKO_CE_ZERO_PAD and untouched otherwise, every other row untouched
    (bit for bit against prefill, the buffer's contents before the call; NaN prefills compare by bits)."""
    r = torch.arange(rows.numel(), device=buf.device) if compact else rows.long().to(buf.device)
    bad = int(violations(buf[r, :V], exp).sum())
    same = buf.view(torch.int16) == prefill.view(torch.int16)
    pad = buf[r, V:]
    bad += int((pad.view(torch.int16) != 0).sum()) if zero_pad else int((~same[r, V:]).sum())
    other = torch.ones(buf.shape[0], dtype=torch.bool, device=buf.device)
    other[r] = False
    return bad + int((~same[other]).sum())

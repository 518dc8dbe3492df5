"""fp64 reference of the attention entry points, a per-element error bound derived from how the kernels round, the check
of a kernel output against it, and a kernel-faithful fp32 emulation of the tiled algorithm.

tests/test_attn_check_cpu.py shows that the check accepts correctly rounded results and the emulation, and rejects subtly
wrong ones; tests/test_attention_matrix_gpu.py runs it on every forward / backward / decode path.  CPU and CUDA tensors.

Layout: q, k, v, dout are [..., L, dh] (16-bit values, exact in fp64); vis is a bool [..., L, L] visibility (query row i
sees key j), broadcast over the leading dims; mult is the fp64 dropout multiplier (0 or the fp32 1/(1-p)) of each (i, j).
Padded layout: [B, H, S, dh] with vis(i, j) = first_valid[b] <= j <= i < S_valid.  Packed layout: [1, H, T, dh] with a
block-diagonal causal vis.  A row with no visible key is dead: out 0, lse +inf, and its dQ row (and the dK / dV rows of a
key no query sees) exactly 0.

Reference (sigma = 1/sqrt(dh), s = sigma q k^T on the visible keys):
  P = softmax(s), lse = logsumexp(s) (natural log), O = (P o M) V -- the normaliser is the undropped P;
  dV = (P o M)^T dO, dP = (dO V^T) o M, delta = rowsum(dO o O_stored), dS = P o (dP - delta), dQ = sigma dS K,
  dK = sigma dS^T Q.  O_stored is the 16-bit O the backward is given: the kernel computes delta from the same values, so
  the 16-bit rounding of O is an input of the backward, not one of its errors.

Bound.  u = 2^-24 (fp32 unit roundoff).  For a live row i with n_i visible keys spread over t_i key tiles (t_i counted
for 64-key tiles, the finer of the two paths), A_i = sigma max_j sum_c |q_ic| |k_jc| bounds every |score|:
  eta_i  relative error of one exponentiated score p_ij = 2^(s log2e - ref) as the kernels compute it:
         fp32 accumulation of q.k over dh (2 dh u A_i, tensor-core accumulation counted as two roundings per term),
         the fp32 scale_log2 and the fmaf (2 u A_i log2e each), the per-tile running-max references and rescale
         exponents, which telescope except for their roundings (2 t_i u A_i log2e), times ln 2; plus ex2.approx.ftz
         (2^-21 per exponential: one for p, one per rescale).
         eta_i = ln2 log2e u A_i (2 dh + 4 + 2 t_i) + 2^-21 (t_i + 1)
  out    each P V term carries the bf16 rounding of P o M (2^-8: half an ulp is 2^-9 of the binade's top but 2^-8 of
         its bottom) and eta_i; the normaliser, summed from the unrounded
         fp32 P, carries eta_i again; fp32 accumulation over n_i keys, t_i rescales of O and the final 1/l:
         (2^-8 + 2 eta_i + (4 sqrt(n_i) + 2 t_i + 4) u) ((P o M) |V|)_ic + half an ulp of the output format at |ref|.
  lse    ln l carries eta_i and the summation of l; m log2e sigma, log2f and the final ln2 product round in fp32:
         eta_i + (4 sqrt(n_i) + 8) u + 4 u (|lse_i| + A_i).
  delta  fp32 dot over dh: (2 dh + 2) u sum_c |dO_ic| |O_ic|.
  bwd    p is recomputed from the forward's lse: its relative error is eta_b,i = 2 eta_i + tol(lse_i).
         E_ij = P_ij (eta_b,i |dP_ij - delta_i| + (2 dh + 2) u M_ij (|dO| |V|^T)_ij + tol(delta_i)) + (2^-8 + 4 u) |dS_ij|
         bounds the error of dS_ij as the kernel feeds it (bf16) to the dQ / dK products, so
         dQ: sigma (E |K|)_ic + 4 sqrt(L) u sigma (|dS| |K|)_ic + half_ulp_bf16;  dK: the same with E^T, |Q|;
         dV: (((2^-8 + eta_b + 4 u) o (P o M))^T |dO|)_jc + 4 sqrt(L) u ((P o M)^T |dO|)_jc + half_ulp_bf16.
  decode one query, fp32 P (__expf, never rounded to 16 bits), so no 2^-8 term:
         eta_d = u A (dh + 8) + 2^-21,  tol = (2 eta_d + (4 sqrt(len) + 4) u) (P |V|)_c + half_ulp(out format).
  ftz    ex2.approx.ftz flushes a probability below 2^-126 to zero: 2^-126 per visible key is added to the P errors
         above ((vis o M) |V| for out, to the recomputed p and P o M of the backward), and 2^-133 (a bf16 subnormal
         ulp) per visible key to dS.
Dead rows have a zero bound: exact zeros (and +inf lse) are required.
"""
from __future__ import annotations

import math
from typing import NamedTuple, Optional

import torch

U = 2.0 ** -24
P16 = 2.0 ** -8          # relative rounding of P and dS to bf16: 8 significant bits, round to nearest
EX2 = 2.0 ** -21         # ex2.approx.ftz / __expf relative error allowance
FTZ = 2.0 ** -126        # absolute error of a probability flushed to zero (p <= 1 relative to the row maximum or lse)
LOG2E = 1.0 / math.log(2.0)
LN2 = math.log(2.0)
TILE = 64                # key tile width used to count rescales (mma.sync; tcgen05 uses 128 and so fewer)

# (mantissa bits incl. the implicit one, smallest normal exponent, largest finite value)
FORMATS = {"bf16": (8, -126, 3.3895313892515355e38), "f16": (11, -14, 65504.0)}
TORCH_FMT = {torch.bfloat16: "bf16", torch.float16: "f16", torch.float32: "f32"}


class Expected(NamedTuple):
    ref: torch.Tensor        # fp64 value (+inf for the lse of dead rows)
    tol: torch.Tensor        # fp64 per-element bound (0 on dead rows)
    fmt: str                 # "f32", "bf16" or "f16"


# ---------------------------------------------------------------------------------------------------
# 16-bit rounding in fp64
# ---------------------------------------------------------------------------------------------------
def _ulp(x: torch.Tensor, fmt: str) -> torch.Tensor:
    p, emin, _ = FORMATS[fmt]
    _, e = torch.frexp(x.abs())
    e = torch.where(x == 0, torch.full_like(e, emin), e - 1).clamp(min=emin)
    return torch.ldexp(torch.ones_like(x), e - (p - 1))


def round16(x: torch.Tensor, fmt: str) -> torch.Tensor:
    x = x.double()
    if fmt == "f16":
        x = x.clamp(-65504.0, 65504.0)
    u = _ulp(x, fmt)
    return torch.round(x / u) * u


def half_ulp(x: torch.Tensor, fmt: str) -> torch.Tensor:
    return 0.5 * _ulp(x, fmt)


def exact_output(exp: Expected) -> torch.Tensor:
    """The correctly rounded output (what an error-free kernel would write), fp64."""
    if exp.fmt == "f32":
        return exp.ref.float().double()
    return round16(exp.ref, exp.fmt)


# ---------------------------------------------------------------------------------------------------
# layouts
# ---------------------------------------------------------------------------------------------------
def split_heads(qkv: torch.Tensor, H: int):
    """qkv [B, S, 3d] -> q, k, v [B, H, S, dh] (views of the same values)."""
    B, S, three_d = qkv.shape
    d = three_d // 3
    return [qkv[..., i * d:(i + 1) * d].reshape(B, S, H, d // H).transpose(1, 2) for i in range(3)]


def merge_heads(x: torch.Tensor) -> torch.Tensor:
    """[B, H, S, dh] -> [B, S, H * dh]."""
    B, H, S, dh = x.shape
    return x.transpose(1, 2).reshape(B, S, H * dh)


def padded_vis(S: int, S_valid: int, first_valid, device=None) -> torch.Tensor:
    """[B, 1, S, S]: first_valid[b] <= key <= query < S_valid."""
    fv = torch.as_tensor(first_valid, device=device).long().reshape(-1, 1, 1, 1)
    i = torch.arange(S, device=device).reshape(1, 1, S, 1)
    j = torch.arange(S, device=device).reshape(1, 1, 1, S)
    return (j >= fv) & (j <= i) & (i < S_valid)


def packed_vis(cu_seqlens, device=None) -> torch.Tensor:
    """[1, 1, T, T]: query t sees keys of its own sample at or before it."""
    cu = torch.as_tensor(cu_seqlens).long().cpu()
    T = int(cu[-1])
    sample = torch.repeat_interleave(torch.arange(len(cu) - 1), cu[1:] - cu[:-1]).to(device)
    i = torch.arange(T, device=device)
    return ((sample[:, None] == sample[None, :]) & (i[None, :] <= i[:, None])).reshape(1, 1, T, T)


def padded_mult(keep: torch.Tensor, scale: float, B: int, H: int, S: int) -> torch.Tensor:
    """Dropout multipliers [B, H, S, S] from the keep mask [B*H*S, S] (row (b*H + h)*S + query, column key)."""
    return keep.reshape(B, H, S, S).double() * scale


def packed_mult(keep: torch.Tensor, scale: float, cu_seqlens, first_valid, H: int, S_width: int) -> torch.Tensor:
    """Dropout multipliers [1, H, T, T] of the packed layout from the padded layout's keep mask [B*H*S_width, S_width]:
    element (query q, key k) of sample b, head h is row (b*H + h)*S_width + first_valid[b] + q, column first_valid[b] + k."""
    cu = torch.as_tensor(cu_seqlens).long().cpu()
    fv = torch.as_tensor(first_valid).long().cpu()
    B, T = len(cu) - 1, int(cu[-1])
    sample = torch.repeat_interleave(torch.arange(B), cu[1:] - cu[:-1])
    pos = torch.arange(T) - cu[sample] + fv[sample]                       # padded column / row offset of each packed row
    h = torch.arange(H).reshape(H, 1)
    rows = (sample.reshape(1, T) * H + h) * S_width + pos.reshape(1, T)   # [H, T]
    dev = keep.device
    m = keep[rows.to(dev).reshape(H, T, 1), pos.to(dev).reshape(1, 1, T)]
    return m.double().reshape(1, H, T, T) * scale


# ---------------------------------------------------------------------------------------------------
# reference
# ---------------------------------------------------------------------------------------------------
class Forward(NamedTuple):
    out: Expected
    out2: Expected           # the bf16 second copy
    lse: Expected
    ctx: dict                # what backward() reuses


def _row_stats(vis: torch.Tensor, sigma: float, absq, absk):
    """A_i (sigma max_j sum_c |q||k| over visible keys), n_i (visible keys), t_i (64-key tiles), live rows."""
    A = (absq @ absk.transpose(-1, -2)) * sigma
    A = torch.where(vis, A, torch.zeros((), dtype=A.dtype, device=A.device)).amax(-1)
    vis_full = vis.expand(*A.shape, vis.shape[-1])
    n = vis_full.sum(-1).double()
    L = vis.shape[-1]
    first = torch.where(vis_full, torch.arange(L, device=vis.device), L).amin(-1)
    i = torch.arange(L, device=vis.device)
    t = ((i - first).clamp(min=0) // TILE + 2).double()
    return A, n, t, n > 0


def forward(q, k, v, vis, mult: Optional[torch.Tensor] = None, out_fmt: str = "bf16") -> Forward:
    """Expected out (out_fmt), out2 (bf16) and lse of one attention forward."""
    q64, k64, v64 = q.double(), k.double(), v.double()
    dh = q.shape[-1]
    sigma = 1.0 / math.sqrt(dh)
    s = (q64 @ k64.transpose(-1, -2)) * sigma
    s = s.masked_fill(~vis, -math.inf)
    A, n, t, live = _row_stats(vis, sigma, q64.abs(), k64.abs())
    mx = s.amax(-1, keepdim=True)
    e = torch.exp(s - torch.where(live[..., None], mx, torch.zeros_like(mx)))
    l = e.sum(-1, keepdim=True)
    P = e / torch.where(l > 0, l, torch.ones_like(l))
    PM = P if mult is None else P * mult
    O = PM @ v64
    W = PM @ v64.abs()
    VM = vis.to(v64.dtype) if mult is None else vis * mult
    Wz = VM @ v64.abs()                                  # the values a flushed probability could have weighted
    lse = torch.where(live, torch.log(l.squeeze(-1)) + mx.squeeze(-1), torch.full_like(A, math.inf))
    eta = LN2 * LOG2E * U * A * (2 * dh + 4 + 2 * t) + EX2 * (t + 1)
    rel = P16 + 2 * eta + (4 * n.sqrt() + 2 * t + 4) * U
    live4 = live[..., None]
    zero = torch.zeros((), dtype=O.dtype, device=O.device)

    def out_exp(fmt):
        tol = rel[..., None] * W + FTZ * Wz + half_ulp(O, fmt)
        return Expected(O, torch.where(live4, tol, zero), fmt)

    lse_tol = eta + (4 * n.sqrt() + 8) * U + 4 * U * (lse.abs() + A)
    lse_exp = Expected(lse, torch.where(live, lse_tol, zero), "f32")
    ctx = dict(q=q64, k=k64, v=v64, vis=vis, mult=mult, P=P, PM=PM, eta=eta, lse_tol=lse_exp.tol, sigma=sigma, live=live)
    return Forward(out_exp(out_fmt), out_exp("bf16"), lse_exp, ctx)


def backward(fwd: Forward, dout, o_stored) -> dict:
    """Expected dq, dk, dv (bf16) and delta (fp32) of the backward given dout and the 16-bit O it is handed."""
    c = fwd.ctx
    q, k, v, P, PM, mult, sigma = c["q"], c["k"], c["v"], c["P"], c["PM"], c["mult"], c["sigma"]
    dh, L = q.shape[-1], q.shape[-2]
    g, o = dout.double(), o_stored.double()
    zero = torch.zeros((), dtype=q.dtype, device=q.device)
    live_q = c["live"]
    live_k = c["vis"].expand(P.shape).any(-2)
    dP = g @ v.transpose(-1, -2)
    dPerr = (2 * dh + 2) * U * (g.abs() @ v.abs().transpose(-1, -2))
    if mult is not None:
        dP, dPerr = dP * mult, dPerr * mult
    delta = (g * o).sum(-1)
    delta_tol = (2 * dh + 2) * U * (g.abs() * o.abs()).sum(-1)
    dS = P * (dP - delta[..., None])
    eta_b = 2 * c["eta"] + c["lse_tol"]
    visf = c["vis"].to(P.dtype)
    Perr = P * eta_b[..., None] + FTZ * visf             # recomputed p: relative error, or flushed to zero
    E = (Perr * (dP - delta[..., None]).abs() + (P + Perr) * (dPerr + delta_tol[..., None]) + (P16 + 4 * U) * dS.abs()
         + 2.0 ** -133 * visf)                           # dS below the fp32 / bf16 normal range
    acc = 4 * math.sqrt(L) * U
    dQ = sigma * (dS @ k)
    dQ_tol = sigma * (E @ k.abs()) + acc * sigma * (dS.abs() @ k.abs()) + half_ulp(dQ, "bf16")
    dSt, Et = dS.transpose(-1, -2), E.transpose(-1, -2)
    dK = sigma * (dSt @ q)
    dK_tol = sigma * (Et @ q.abs()) + acc * sigma * (dSt.abs() @ q.abs()) + half_ulp(dK, "bf16")
    PMt = PM.transpose(-1, -2)
    dV = PMt @ g
    PMerr = (P16 + eta_b + 4 * U)[..., None] * PM + FTZ * (visf if mult is None else visf * mult)
    dV_tol = PMerr.transpose(-1, -2) @ g.abs() + acc * (PMt @ g.abs()) + half_ulp(dV, "bf16")
    lq, lk = live_q[..., None], live_k[..., None]
    return {"dq": Expected(dQ, torch.where(lq, dQ_tol, zero), "bf16"),
            "dk": Expected(dK, torch.where(lk, dK_tol, zero), "bf16"),
            "dv": Expected(dV, torch.where(lk, dV_tol, zero), "bf16"),
            "delta": Expected(delta, delta_tol, "f32")}


def decode(q, k, v, out_fmt: str = "bf16", sigma: Optional[float] = None) -> Expected:
    """One query q [H, dh] against keys / values [len, H, dh]: out [H, dh]."""
    q64, k64, v64 = q.double(), k.double().transpose(0, 1), v.double().transpose(0, 1)   # [H, len, dh]
    dh, n = q.shape[-1], k.shape[0]
    sig = 1.0 / math.sqrt(dh) if sigma is None else sigma
    s = (k64 @ q64[..., None]).squeeze(-1) * sig                                       # [H, len]
    P = torch.softmax(s, -1)
    O = (P[:, None, :] @ v64).squeeze(1)
    W = (P[:, None, :] @ v64.abs()).squeeze(1)
    A = ((k64.abs() @ q64.abs()[..., None]).squeeze(-1) * sig).amax(-1, keepdim=True)
    eta = U * A * (dh + 8) + EX2
    tol = (2 * eta + (4 * math.sqrt(n) + 4) * U) * W + half_ulp(O, out_fmt)
    return Expected(O, tol, out_fmt)


# ---------------------------------------------------------------------------------------------------
# check
# ---------------------------------------------------------------------------------------------------
def violations(out: torch.Tensor, exp: Expected) -> torch.Tensor:
    """Boolean, shaped like out: elements outside the bound.  NaN is outside; +inf must match a +inf reference."""
    if out.dtype in TORCH_FMT:
        assert TORCH_FMT[out.dtype] == exp.fmt, f"output is {out.dtype}, reference expects {exp.fmt}"
    o = out.double()
    ok = (o - exp.ref).abs() <= exp.tol
    return ~torch.where(torch.isinf(exp.ref), o == exp.ref, ok)


def worst_ratio(out: torch.Tensor, exp: Expected) -> float:
    """max err / bound over the elements with a non-zero bound (the headroom of the check)."""
    o = out.double()
    m = (exp.tol > 0) & torch.isfinite(exp.ref)
    if not bool(m.any()):
        return 0.0
    return float(((o - exp.ref).abs()[m] / exp.tol[m]).max())


def assert_within(out: torch.Tensor, exp: Expected, what: str = "output", dims=("b", "h", "row", "col")):
    bad = violations(out, exp)
    n = int(bad.sum())
    if n:
        o = out.double()
        excess = torch.where(bad, ((o - exp.ref).abs() - exp.tol).nan_to_num(math.inf), torch.full_like(o, -math.inf))
        idx = [int(x) for x in torch.unravel_index(excess.argmax(), excess.shape)]
        where = ", ".join(f"{d}={i}" for d, i in zip(dims[-len(idx):], idx))
        raise AssertionError(f"{what}: {n} of {bad.numel()} elements outside the bound; worst at ({where}): "
                             f"got {float(o[tuple(idx)]):.9g} ref {float(exp.ref[tuple(idx)]):.9g} bound {float(exp.tol[tuple(idx)]):.3g}")


# ---------------------------------------------------------------------------------------------------
# kernel-faithful emulation (fp32)
# ---------------------------------------------------------------------------------------------------
def _ftz(x: torch.Tensor) -> torch.Tensor:
    return torch.where(x.abs() < 2.0 ** -126, torch.zeros_like(x), x)


def _to(x: torch.Tensor, fmt: str) -> torch.Tensor:
    return x.to(torch.bfloat16 if fmt == "bf16" else torch.float16)


def emulate_forward(q, k, v, vis, mult=None, tile: int = 64, out_fmt: str = "bf16", rescale: bool = True):
    """The tiled online-softmax forward in fp32 as the kernels run it: fp32 scores, exp2 against the running maximum,
    rescale of l and O when the maximum rises (rescale=False leaves O unscaled), P o M rounded to bf16 before the PV
    product, the normaliser from the unrounded P.  Returns (out in out_fmt, lse fp32)."""
    q32, k32, v32 = q.float(), k.float(), v.float()
    dh, L = q.shape[-1], q.shape[-2]
    sl = float(torch.tensor(1.4426950408889634, dtype=torch.float32) / torch.sqrt(torch.tensor(float(dh), dtype=torch.float32)))
    s = q32 @ k32.transpose(-1, -2)
    shape = s.shape[:-1]
    m = torch.full(shape, -math.inf, device=s.device)
    l = torch.zeros(shape, device=s.device)
    o = torch.zeros(*shape, v.shape[-1], device=s.device)
    vis = vis.expand(s.shape)
    for j0 in range(0, L, tile):
        st = s[..., j0:j0 + tile].masked_fill(~vis[..., j0:j0 + tile], -math.inf)
        mn = torch.maximum(m, st.amax(-1))
        ref = torch.where(mn == -math.inf, torch.zeros_like(mn), mn * sl)
        corr = _ftz(torch.exp2(m * sl - ref))
        m = mn
        p = _ftz(torch.exp2(st * sl - ref[..., None]))
        l = l * corr + p.sum(-1)
        if mult is not None:
            p = p * mult[..., j0:j0 + tile].float()
        pv = p.bfloat16().float() @ v32[..., j0:j0 + tile, :]
        o = (o * corr[..., None] if rescale else o) + pv
    inv = torch.where(l > 0, 1.0 / l, torch.zeros_like(l))
    lse = torch.where(l > 0, (m * sl + torch.log2(l)) * LN2, torch.full_like(l, math.inf))
    return _to(o * inv[..., None], out_fmt), lse


def emulate_backward(q, k, v, vis, lse, dout, o_stored, mult=None):
    """The dQ / dK / dV kernels in fp32: P recomputed from the stored lse, delta from the 16-bit O, dS and P o M rounded
    to bf16 before their products.  Returns (dq, dk, dv as bf16, delta fp32)."""
    q32, k32, v32, g = q.float(), k.float(), v.float(), dout.float()
    dh = q.shape[-1]
    scale = float(1.0 / torch.sqrt(torch.tensor(float(dh), dtype=torch.float32)))
    sl = float(torch.tensor(1.4426950408889634, dtype=torch.float32) * scale)
    s = q32 @ k32.transpose(-1, -2)
    p = _ftz(torch.exp2(s * sl - (lse.float() * 1.4426950408889634)[..., None]))
    p = torch.where(vis, p, torch.zeros_like(p))
    dp = g @ v32.transpose(-1, -2)
    pm = p
    if mult is not None:
        dp, pm = dp * mult.float(), p * mult.float()
    delta = (g * o_stored.float()).sum(-1)
    ds = (p * (dp - delta[..., None]) * scale).bfloat16().float()
    dq = ds @ k32
    dk = ds.transpose(-1, -2) @ q32
    dv = pm.bfloat16().float().transpose(-1, -2) @ g
    return dq.bfloat16(), dk.bfloat16(), dv.bfloat16(), delta

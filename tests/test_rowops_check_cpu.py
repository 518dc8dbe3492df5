"""The row-kernel check of tests/_rowops_ref.py is strict: it accepts the correctly rounded result and the kernel-faithful fp32
emulations, and rejects subtly wrong kernels (each mutant on an input where it actually differs).  Also the host-side argument
checks and kernel choice of the LayerNorm entry points, with fake device pointers (nothing is launched).  CPU only."""
import ctypes as C
import math
import os
import subprocess
import sys

import pytest
import torch

import _rowops_ref as R

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _gen(seed):
    return torch.Generator().manual_seed(seed)


def _exact(exp: R.Expected) -> torch.Tensor:
    return exp.ref.float() if exp.fmt == "f32" else R.to16(exp.ref, exp.fmt)


def _nbad(out, exp) -> int:
    return int(R.violations(out, exp).sum())


# ---------------------------------------------------------------------------------------------------
# LayerNorm forward
# ---------------------------------------------------------------------------------------------------
def _ln_inputs(N, d, regime, seed=0):
    g = _gen(seed)
    x = torch.randn(N, d, generator=g) * 2 + 0.5
    if regime == "offset":
        x = torch.randn(N, d, generator=g) + 1e3
    elif regime == "const":
        x = torch.full((N, d), 3.25) + torch.arange(N)[:, None]
    elif regime == "tiny":
        x = torch.randn(N, d, generator=g) * 1e-3
    gamma = 1 + 0.2 * torch.randn(d, generator=g)
    if regime == "saturate":
        gamma = gamma * 3e4
    beta = 0.2 * torch.randn(d, generator=g)
    return x, gamma, beta


LN_CASES = [(7, 100, "randn"), (5, 768, "randn"), (3, 1288, "offset"), (4, 256, "const"), (6, 384, "tiny"), (3, 640, "saturate")]


@pytest.mark.parametrize("N,d,regime", LN_CASES)
@pytest.mark.parametrize("fmt", ["bf16", "f16"])
def test_ln_fwd_accepts_exact_and_emulation(N, d, regime, fmt):
    x, g, b = _ln_inputs(N, d, regime)
    exp = R.ln_forward(x, g, b, 1e-5, fmt)
    for k in ("y", "y2", "mean", "rstd"):
        assert _nbad(_exact(exp[k]), exp[k]) == 0, k
    y, y2, mean, rstd = R.emulate_ln_fwd(x, g, b, 1e-5, fmt)
    for k, v in (("y", y), ("y2", y2), ("mean", mean), ("rstd", rstd)):
        assert _nbad(v, exp[k]) == 0, (k, R.worst_ratio(v, exp[k]))
    assert int(R.ln_y2_mismatch(y, y2).sum()) == 0


LN_FWD_MUTANTS = {   # mutant -> (N, d, regime, fmt) where it differs
    "unbiased": (16, 768, "randn", "f16"), "eps_outside": (8, 256, "tiny", "f16"), "mean_dm1": (8, 768, "randn", "bf16"),
    "gamma_shift": (4, 256, "randn", "bf16"), "stale_tail": (4, 100, "randn", "bf16"), "f16_inf": (3, 640, "saturate", "f16"),
}


@pytest.mark.parametrize("mutant", sorted(LN_FWD_MUTANTS))
def test_ln_fwd_rejects(mutant):
    N, d, regime, fmt = LN_FWD_MUTANTS[mutant]
    x, g, b = _ln_inputs(N, d, regime, seed=1)
    exp = R.ln_forward(x, g, b, 1e-5, fmt)
    y, y2, mean, rstd = R.emulate_ln_fwd(x, g, b, 1e-5, fmt, mutant=mutant)
    assert _nbad(y, exp["y"]) + _nbad(mean, exp["mean"]) + _nbad(rstd, exp["rstd"]) > 0


# ---------------------------------------------------------------------------------------------------
# LayerNorm backward
# ---------------------------------------------------------------------------------------------------
def _ln_bwd_case(N, d, drop, seed=2):
    g = _gen(seed)
    x, gamma, _ = _ln_inputs(N, d, "randn", seed)
    mean, rstd = R.emulate_ln_fwd(x, gamma, torch.zeros(d), 1e-5)[2:]
    dy = torch.randn(N, d, generator=g).to(torch.bfloat16)
    dx_in = torch.randn(N, d, generator=g)
    mult = None
    if drop:
        mult = (torch.rand(N, d, generator=g) >= 0.1).float() * torch.tensor(1 / 0.9, dtype=torch.float32)
    inits = [torch.randn(d, generator=g) for _ in range(3)]
    return x, gamma, mean, rstd, dy, dx_in, mult, inits


def _ln_bwd_bad(em, exp, inits) -> int:
    n = _nbad(em["dx"], exp["dx"])
    n += int((em["dx_bf16"].view(torch.int16) != exp["dx_bf16"].view(torch.int16)).sum())
    for k, i in zip(("dgamma", "dbeta", "colsum"), inits):
        n += _nbad(em[k] + i, exp[k])
    return n


@pytest.mark.parametrize("N,d", [(9, 128), (6, 768), (5, 100), (3, 1600)])
@pytest.mark.parametrize("drop", [False, True])
def test_ln_bwd_accepts_exact_and_emulation(N, d, drop):
    x, gamma, mean, rstd, dy, dx_in, mult, inits = _ln_bwd_case(N, d, drop)
    em = R.emulate_ln_bwd(dy, x, gamma, mean, rstd, dx_in, mult)
    exp = R.ln_backward(dy, x, gamma, mean, rstd, dx_in, mult, *inits, dx_out_kernel=em["dx"])
    assert _nbad(_exact(exp["dx"]), exp["dx"]) == 0
    assert _ln_bwd_bad(em, exp, inits) == 0, {k: R.worst_ratio(em[k], exp[k]) for k in ("dx",)}


LN_BWD_MUTANTS = ["no_m2", "m1_dm1", "mask_fp32", "bf16_before_add", "colsum_unmasked", "dgamma_x", "skip_last_block"]


@pytest.mark.parametrize("mutant", LN_BWD_MUTANTS)
def test_ln_bwd_rejects(mutant):
    x, gamma, mean, rstd, dy, dx_in, mult, inits = _ln_bwd_case(9, 256, True, seed=3)
    good = R.emulate_ln_bwd(dy, x, gamma, mean, rstd, dx_in, mult)
    exp = R.ln_backward(dy, x, gamma, mean, rstd, dx_in, mult, *inits, dx_out_kernel=good["dx"])
    em = R.emulate_ln_bwd(dy, x, gamma, mean, rstd, dx_in, mult, mutant=mutant)
    assert _ln_bwd_bad(em, exp, inits) > 0


# ---------------------------------------------------------------------------------------------------
# cross entropy
# ---------------------------------------------------------------------------------------------------
def _ce_case(n, V, regime, kernel, seed=4):
    g = _gen(seed)
    z = torch.randn(n, V, generator=g) * 2
    if regime == "peaky":
        z[:, V // 3] += 30
    elif regime == "flat":
        z = torch.zeros(n, V)
    elif regime == "extreme":
        z = (torch.rand(n, V, generator=g) * 2 - 1) * (6e4 if kernel == "fused_f16" else 80)
    elif regime == "rising":
        z = torch.linspace(-3, 3, V).repeat(n, 1) + 0.01 * torch.randn(n, V, generator=g)
    if kernel == "fused_f16":
        z = z.half()
    t = torch.randint(0, V, (n,), generator=g)
    t[0] = 0
    t[-1] = V - 1
    return z, t


CE_ACCEPT = [(kernel, V, regime) for kernel in R.CE_KERNELS for V, regime in
             ((7, "randn"), (1001, "peaky"), (2208, "flat"), (3001, "extreme"), (4099, "rising"))]


@pytest.mark.parametrize("kernel,V,regime", CE_ACCEPT)
def test_ce_accepts_exact_and_emulation(kernel, V, regime):
    z, t = _ce_case(5, V, regime, kernel)
    n_rows = 37
    exp = R.ce_reference(z, t, n_rows, 1.0, kernel)
    for k in ("lse", "row_loss", "dlogits"):
        assert _nbad(_exact(exp[k]), exp[k]) == 0, k
    lse, loss, d = R.emulate_ce(z, t, n_rows, kernel)
    assert _nbad(lse, exp["lse"]) == 0, R.worst_ratio(lse, exp["lse"])
    assert _nbad(loss, exp["row_loss"]) == 0
    assert _nbad(d, exp["dlogits"]) == 0, R.worst_ratio(d, exp["dlogits"])
    # the fused path's gradient after the upstream scale: two bf16 roundings
    for gs in (0.25, 3.0):
        assert _nbad(R.ce_scale_exact(d, gs), R.ce_scaled(exp["dlogits"], gs)) == 0


CE_MUTANTS = {   # mutant -> (kernel, V, regime)
    "lse_plus": ("two_pass", 52305, "randn"), "log2": ("fused", 1001, "randn"), "drop_rescale": ("two_pass", 4099, "rising"),
    "onehot_next": ("fused", 2208, "randn"), "n_minus_1": ("two_pass", 1001, "peaky"), "stale_tail": ("fused", 1003, "randn"),
    "stale_tail_f16": ("fused_f16", 1005, "randn"), "f16_as_bf16": ("fused_f16", 1001, "randn"),
}


@pytest.mark.parametrize("mutant", sorted(CE_MUTANTS))
def test_ce_rejects(mutant):
    kernel, V, regime = CE_MUTANTS[mutant]
    z, t = _ce_case(4, V, regime, kernel, seed=5)
    t[1] = V - 1                                    # a target in the vector tail
    exp = R.ce_reference(z, t, 37, 1.0, kernel)
    lse, loss, d = R.emulate_ce(z, t, 37, kernel, mutant=mutant.replace("_f16", "") if mutant == "stale_tail_f16" else mutant)
    assert _nbad(lse, exp["lse"]) + _nbad(loss, exp["row_loss"]) + _nbad(d, exp["dlogits"]) > 0


def _layout(compact, zero_pad, V=13, ld=20, n_buf=9):
    rows = torch.tensor([1, 4, 6], dtype=torch.int32)
    z, t = _ce_case(3, V, "randn", "fused", seed=6)
    exp = R.ce_reference(z, t, 3, 3.0)
    prefill = torch.full((3 if compact else n_buf, ld), math.nan, dtype=torch.bfloat16)
    buf = prefill.clone()
    r = torch.arange(3) if compact else rows.long()
    buf[r, :V] = R.to16(exp["dlogits"].ref, "bf16")
    if zero_pad:
        buf[r, V:] = 0
    return buf, prefill, exp, rows, V, r


@pytest.mark.parametrize("compact", [False, True])
@pytest.mark.parametrize("zero_pad", [False, True])
def test_ce_dlogits_layout(compact, zero_pad):
    buf, prefill, exp, rows, V, r = _layout(compact, zero_pad)
    args = (prefill, exp["dlogits"], rows, V, compact, zero_pad)
    assert R.ce_dlogits_violations(buf, *args) == 0
    bad = buf.clone()                               # pad columns left alone under ZERO_PAD / written without it
    bad[r[1], V + 2] = 0 if not zero_pad else math.nan
    assert R.ce_dlogits_violations(bad, *args) > 0
    bad = buf.clone()                               # the row written one element past ld: the next row's first column
    bad.view(-1)[int(r[0]) * buf.shape[1] + buf.shape[1]] = 0
    assert R.ce_dlogits_violations(bad, *args) > 0
    bad = buf.clone()                               # gscale applied twice
    bad[r, :V] = (buf[r, :V].float() * 3).to(torch.bfloat16)
    assert R.ce_dlogits_violations(bad, *args) > 0
    if not compact:                                 # a non-selected row touched
        bad = buf.clone()
        bad[0, 0] = 0
        assert R.ce_dlogits_violations(bad, *args) > 0


def test_ce_out_of_range_target():
    """tokens is caller input: a target of -1 or V gives row_loss 0 and a gradient row of softmax * g / n, no one-hot."""
    z, t = _ce_case(3, 50, "randn", "fused", seed=7)
    t[0], t[1] = -1, 50
    exp = R.ce_reference(z, t, 3, 1.0)
    assert float(exp["row_loss"].ref[0]) == 0.0 and float(exp["row_loss"].tol[1]) == 0.0
    p = torch.softmax(z.double(), -1) / 3
    assert torch.allclose(exp["dlogits"].ref[:2], p[:2], rtol=1e-12, atol=0)
    lse, loss, d = R.emulate_ce(z, t, 3, "fused")
    assert _nbad(loss, exp["row_loss"]) == 0 and _nbad(d, exp["dlogits"]) == 0


def test_ce_loss_and_scale():
    rl = torch.rand(1000, generator=_gen(8)) * 10
    exp = R.ce_loss_expected(rl)
    assert _nbad(rl.double().mean().float(), exp) == 0
    assert _nbad((rl.double().mean() * (1 + 2 ** -20)).float(), exp) > 0
    d = torch.randn(64, generator=_gen(9)).to(torch.bfloat16)
    assert torch.equal(R.ce_scale_exact(d, 1.0).view(torch.int16), d.view(torch.int16))


# ---------------------------------------------------------------------------------------------------
# GeGLU and casts
# ---------------------------------------------------------------------------------------------------
def _geglu_inputs(n=4096, seed=10):
    g = _gen(seed)
    pre = torch.linspace(-10, 10, n)
    pre[n // 2] = 0.0
    pre = pre.to(torch.bfloat16)
    dh = torch.randn(n, generator=g).to(torch.bfloat16)
    gate = torch.randn(n, generator=g).to(torch.bfloat16)
    return dh, pre, gate


def test_geglu_fwd_exact_and_saturation():
    dh, pre, gate = _geglu_inputs()
    act = (pre.float() * 300).half()               # products beyond 65504 saturate in fp16
    out, out_b = R.geglu_fwd_exact(act, gate * 400, "f16")
    prod = act.float() * (gate * 400).float()       # exact in fp32
    assert torch.equal(out.float(), prod.clamp(-65504, 65504).half().float().clamp(-65504, 65504))
    assert float(out.float().abs().max()) == 65504.0
    assert torch.equal(out_b, prod.to(torch.bfloat16))


def test_geglu_bwd_accepts_and_rejects():
    dh, pre, gate = _geglu_inputs()
    exp = R.geglu_bwd(dh, pre, gate)
    p, d64, g64 = pre.double(), dh.double(), gate.double()
    ge, gp = R.gelu64(p, False), R.gelu_grad64(p, False)
    # fp32 evaluation of the erf form
    pf = pre.float()
    ge32 = 0.5 * pf * (1 + torch.erf(pf / math.sqrt(2)))
    gp32 = 0.5 * (1 + torch.erf(pf / math.sqrt(2))) + pf * torch.exp(-0.5 * pf * pf) / math.sqrt(2 * math.pi)
    assert _nbad((dh.float() * ge32).to(torch.bfloat16), exp["d_gate"]) == 0
    assert _nbad((dh.float() * gate.float() * gp32).to(torch.bfloat16), exp["d_pre"]) == 0
    assert _nbad(R.to16(d64 * ge, "bf16"), exp["d_gate"]) == 0
    tanh_gate = R.to16(d64 * R.gelu64(p, True), "bf16")
    assert _nbad(tanh_gate, exp["d_gate"]) > 0, "tanh-form GELU"
    no_xphi = R.to16(d64 * g64 * 0.5 * (1 + torch.erf(p / math.sqrt(2))), "bf16")
    assert _nbad(no_xphi, exp["d_pre"]) > 0, "x phi(x) term of gelu' dropped"
    no_gate = R.to16(d64 * gp, "bf16")
    assert _nbad(no_gate, exp["d_pre"]) > 0, "d_pre without the gate"


def test_cast_exact_saturates():
    x = torch.tensor([0.0, -0.0, 1.0, 65504.0, 65519.9, 65520.0, 1e6, -1e6, 1e-8, 3.14159])
    h = R.cast_exact(x, "f16")
    assert h.float().abs().max() == 65504.0 and torch.isfinite(h.float()).all()
    assert torch.equal(h[:5], x[:5].half()) and torch.equal(R.cast_exact(x, "bf16"), x.to(torch.bfloat16))


# ---------------------------------------------------------------------------------------------------
# argument checks and the LayerNorm backward path query (fake pointers: nothing is dereferenced or launched)
# ---------------------------------------------------------------------------------------------------
NEKO_EINVAL = -1
F = 0x100000          # a fake 16-byte aligned device address


@pytest.fixture(scope="module")
def lib():
    from neko_b200 import _lib, build
    build.build()
    return _lib.load()


def _p(x):
    return C.c_void_p(x)


def _fwd(lib, x=F, gamma=F, beta=F, y=F, y2=0, N=8, d=128):
    return lib.neko_layernorm_fwd(_p(x), _p(gamma), _p(beta), _p(y), _p(y2), _p(F), _p(F), C.c_int(N), C.c_int(d), C.c_float(1e-5),
                                  C.c_int(0), None)


@pytest.mark.parametrize("case", ["x8", "gamma8", "beta4", "y4", "y2_4", "d6", "d2052", "N0"])
def test_layernorm_fwd_rejects(lib, case):
    a = {"x8": dict(x=F + 8), "gamma8": dict(gamma=F + 8), "beta4": dict(beta=F + 4), "y4": dict(y=F + 4), "y2_4": dict(y2=F + 4),
         "d6": dict(d=6), "d2052": dict(d=2052), "N0": dict(N=0)}[case]
    assert _fwd(lib, **a) == NEKO_EINVAL


def _bwd_args(dy=F, x=F, gamma=F, dx=F, dxb=0, N=8, d=128):
    return (_p(dy), _p(x), _p(gamma), _p(F), _p(F), _p(dx), _p(dxb), _p(F), _p(F), None, C.c_int(N), C.c_int(d), None)


def _path(lib, **kw):
    from neko_b200._lib import LnBwdPathInfo
    info = LnBwdPathInfo()
    rc = lib.neko_layernorm_bwd_path(*_bwd_args(**kw), C.byref(info))
    return rc, info.grid, info.rows_per_cta, info.stages


@pytest.mark.parametrize("case", ["x8", "dx_resid8", "gamma8", "dy4", "dx_bf16_4", "d6", "N0"])
def test_layernorm_bwd_rejects(lib, case):
    a = {"x8": dict(x=F + 8), "dx_resid8": dict(dx=F + 8), "gamma8": dict(gamma=F + 8), "dy4": dict(dy=F + 4),
         "dx_bf16_4": dict(dxb=F + 4), "d6": dict(d=6), "N0": dict(N=0)}[case]
    assert lib.neko_layernorm_bwd(*_bwd_args(**a), None) == NEKO_EINVAL
    assert _path(lib, **a)[0] == NEKO_EINVAL


def test_layernorm_bwd_path(lib, monkeypatch):
    """Which backward kernel runs (sm_count() falls back to 148 without a device): warp-per-row for d = 128 NV <= 1024,
    staged when d % 8 == 0, dy is 16-byte aligned and >= 2 ring stages fit, register otherwise."""
    monkeypatch.delenv("NEKO_LN_CTAS", raising=False)
    sms = lib.neko_sm_count()
    want = {4: 2, 12: 2, 32: 1, 100: 2, 128: 0, 384: 0, 768: 0, 800: 1, 1024: 0, 1152: 1, 1280: 1, 1288: 2, 1600: 2, 2048: 2}
    stages = {32: 4, 800: 3, 1152: 2, 1280: 2}
    for d, k in want.items():
        rc, grid, rpc, st = _path(lib, N=7680, d=d)
        assert rc == k, d
        assert st == stages.get(d, 0), d
        if k == 0:
            assert grid == 2 * sms and rpc == 0
        else:
            assert rpc == 28 and grid == -(-7680 // 28), d       # 2 CTAs per SM, 4-row blocks
    assert _path(lib, N=5, d=768)[1] == 1                          # one CTA of 8 warps covers 5 rows
    assert _path(lib, N=7680, d=256, dy=F + 8)[0] == 0             # an 8-byte aligned dy keeps warp-per-row
    assert _path(lib, N=7680, d=800, dy=F + 8)[0] == 2             # ... and moves staged to register
    for v, grid in (("1", 1), ("3", 3), ("7680", 1920), ("0", -(-7680 // 28)), ("-3", -(-7680 // 28)), ("abc", -(-7680 // 28))):
        monkeypatch.setenv("NEKO_LN_CTAS", v)
        assert _path(lib, N=7680, d=1280)[1] == grid, v
        assert lib.neko_layernorm_bwd(*_bwd_args(N=7680, d=4, dy=F + 4), None) == NEKO_EINVAL   # rejected, never divided by zero


_CHILD = r"""
import ctypes as C, sys
sys.path.insert(0, sys.argv[1])
from neko_b200 import _lib
lib = _lib.load()
F = 0x100000
p = C.c_void_p
print(lib.neko_layernorm_bwd_path(p(F), p(F), p(F), p(F), p(F), p(F), None, p(F), p(F), None, 7680, 768, None, None))
"""


@pytest.mark.parametrize("env,kernel", [("NEKO_LN_BWD_COLUMNS", 1), ("NEKO_LN_BWD_REGISTER", 2)])
def test_layernorm_bwd_path_forced(lib, env, kernel):
    """The two switches are read once per process: a fresh interpreter sees them."""
    e = {k: v for k, v in os.environ.items() if k not in ("NEKO_LN_BWD_COLUMNS", "NEKO_LN_BWD_REGISTER")}
    e["NEKO_LN_BWD_COLUMNS"] = "1"
    if env == "NEKO_LN_BWD_REGISTER":
        e[env] = "1"
    r = subprocess.run([sys.executable, "-c", _CHILD, ROOT], env=e, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    assert int(r.stdout.split()[-1]) == kernel

"""LayerNorm forward / backward (default and ordered), masked cross entropy (two-pass, fused fp32, fused fp16, gradient scale),
GeGLU and the casts against the fp64 references and per-element bounds of tests/_rowops_ref.py.

Every cell writes its outputs into NaN-prefilled views between sentinel guard bands, checks that the guards and the inputs are
unchanged and that a repeat launch gives bit-identical row outputs (column sums use atomics: they are checked against their
bound only).  Each LayerNorm backward cell asserts through ops.layernorm_bwd_path which kernel ran.  The largest err / bound
ratio per output kind is printed at the end (-s), and written as JSON to $NEKO_ROWOPS_STATS when that is set.  GPU only."""
import json
import math
import os
import subprocess
import sys

import pytest
import torch

import _rowops_ref as R

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GUARD = 64
SENT = {torch.float32: 12345.0, torch.bfloat16: 777.0, torch.float16: 555.0}
RATIOS = {}
PATHS = {}


@pytest.fixture(scope="module")
def ops():
    from neko_b200 import _lib, ops as o
    _lib.require_device()
    yield o
    print("\nworst err/bound:", json.dumps({k: round(v, 4) for k, v in sorted(RATIOS.items())}))
    print("LayerNorm backward kernels:", json.dumps(PATHS))
    if os.environ.get("NEKO_ROWOPS_STATS"):
        with open(os.environ["NEKO_ROWOPS_STATS"], "w") as f:
            json.dump({"ratios": RATIOS, "ln_bwd_paths": PATHS}, f, indent=1)


def _seen(kernel, d):
    PATHS.setdefault(kernel, [])
    if d not in PATHS[kernel]:
        PATHS[kernel].append(d)


def _note(kind, out, exp):
    RATIOS[kind] = max(RATIOS.get(kind, 0.0), R.worst_ratio(out, exp))


def _check(kind, out, exp):
    R.assert_within(out, exp, kind)
    _note(kind, out, exp)


class Guarded:
    """A tensor of `shape` (optionally `offset` elements past a 16-byte boundary) in the middle of a buffer whose GUARD
    elements on each side hold a sentinel."""

    def __init__(self, shape, dtype, fill=math.nan, offset=0, init=None):
        n = math.prod(shape)
        self.buf = torch.full((n + 2 * GUARD + offset,), SENT[dtype], dtype=dtype, device="cuda")
        self.t = self.buf[GUARD + offset:GUARD + offset + n].view(*shape)
        if init is not None:
            self.t.copy_(init)
        else:
            self.t.fill_(fill)
        self.lo, self.hi = GUARD + offset, GUARD + offset + n

    def guards_ok(self):
        s = SENT[self.buf.dtype]
        return bool((self.buf[:self.lo] == s).all()) and bool((self.buf[self.hi:] == s).all())


def _bits(t):
    return t.view(torch.int16) if t.element_size() == 2 else t.view(torch.int32)


def _same_bits(a, b):
    return torch.equal(_bits(a), _bits(b))


def _gen(seed):
    return torch.Generator(device="cpu").manual_seed(seed)


# ---------------------------------------------------------------------------------------------------
# LayerNorm
# ---------------------------------------------------------------------------------------------------
LN_D = [4, 12, 32, 100, 128, 256, 384, 512, 640, 768, 800, 896, 1024, 1152, 1280, 1288, 1600, 2044, 2048]
LN_N = [1, 3, 5, 37, 7680, 20000]
LN_REGIMES = ["randn", "offset", "const", "tiny", "saturate"]


def _ln_inputs(N, d, regime, seed):
    g = _gen(seed)
    x = torch.randn(N, d, generator=g) * 2 + 0.5
    if regime == "offset":
        x = torch.randn(N, d, generator=g) + 1e3
    elif regime == "const":
        x = (torch.full((N, d), 3.25) + torch.arange(N)[:, None] * 0.5)
    elif regime == "tiny":
        x = torch.randn(N, d, generator=g) * 1e-3
    gamma = 1 + 0.2 * torch.randn(d, generator=g)
    if regime == "saturate":
        gamma = gamma * 3e4
    beta = 0.2 * torch.randn(d, generator=g)
    return x.cuda(), gamma.cuda(), beta.cuda()


def _want_kernel(d, dy_aligned16, forced=None):
    if forced is None and d % 128 == 0 and d <= 1024:
        return "rows"
    stages = min(4, (100 * 1024) // (4 * d * 10))
    if forced != "register" and stages >= 2 and d % 8 == 0 and dy_aligned16:
        return "staged"
    return "register"


LN_CELLS = []
for i, d in enumerate(LN_D):
    for j, N in enumerate(LN_N):
        k = i * len(LN_N) + j
        LN_CELLS.append(pytest.param(N, d, LN_REGIMES[k % 5], ("bf16", "f16")[k % 2], (0.0, 0.1)[(k // 2) % 2], (k // 4) % 4,
                                     id=f"N{N}-d{d}-{LN_REGIMES[k % 5]}"))


def _ln_fwd(ops, x, g, b, fmt):
    N, d = x.shape
    dt = torch.bfloat16 if fmt == "bf16" else torch.float16
    y, y2 = Guarded((N, d), dt), Guarded((N, d), torch.bfloat16)
    mean, rstd = Guarded((N,), torch.float32), Guarded((N,), torch.float32)
    ops.layernorm_fwd(x, g, b, 1e-5, y=y.t, mean=mean.t, rstd=rstd.t, y2=y2.t)
    return y, y2, mean, rstd


def _ln_bwd_run(ops, fn, dy, x, g, mean, rstd, dx0, init, with_bf16, with_cs, drop, ws=None):
    N, d = x.shape
    dx = Guarded((N, d), torch.float32, init=dx0)
    dxb = Guarded((N, d), torch.bfloat16) if with_bf16 else None
    dg, db = Guarded((d,), torch.float32, init=init[0]), Guarded((d,), torch.float32, init=init[1])
    cs = Guarded((d,), torch.float32, init=init[2]) if with_cs else None
    args = (dy, x, g, mean, rstd, dx.t, dg.t, db.t)
    kw = dict(dx_bf16=dxb.t if dxb else None, dx_colsum=cs.t if cs else None, branch_drop=drop)
    if ws is not None:
        fn(*args[:8], ws, **kw)
    else:
        fn(*args, **kw)
    return dx, dxb, dg, db, cs


def _ln_bwd_check(ops, tag, dy, x, g, mean, rstd, dx0, init, with_bf16, with_cs, drop, p, ordered=False):
    N, d = x.shape
    fn, ws = ops.layernorm_bwd, None
    if ordered:
        fn = ops.layernorm_bwd_ordered
        ws = torch.empty(ops.layernorm_bwd_ordered_workspace_bytes(N, d), dtype=torch.uint8, device="cuda")
    keep = [t.clone() for t in (dy, x, g, mean, rstd)]
    dx, dxb, dg, db, cs = _ln_bwd_run(ops, fn, dy, x, g, mean, rstd, dx0, init, with_bf16, with_cs, drop, ws)
    mult = None
    if p > 0:
        mult = ops.dropout_mask(N, d, drop, "cuda").double() * torch.tensor(drop.scale, dtype=torch.float32).double()
    exp = R.ln_backward(dy, x, g, mean, rstd, dx0, mult, *init, dx_out_kernel=dx.t)
    _check(f"ln_dx{tag}", dx.t, exp["dx"])
    if with_bf16:
        R.assert_bits(dxb.t, exp["dx_bf16"], "dx_bf16")
    if not ordered:
        _check("ln_dgamma", dg.t, exp["dgamma"])
        _check("ln_dbeta", db.t, exp["dbeta"])
        if with_cs:
            _check("ln_colsum", cs.t, exp["colsum"])
    for gd in (dx, dxb, dg, db, cs):
        assert gd is None or gd.guards_ok()
    assert all(_same_bits(a, b) for a, b in zip(keep, (dy, x, g, mean, rstd))), "an input changed"
    rep = _ln_bwd_run(ops, fn, dy, x, g, mean, rstd, dx0, init, with_bf16, with_cs, drop, ws)
    assert _same_bits(rep[0].t, dx.t) and (not with_bf16 or _same_bits(rep[1].t, dxb.t)), "repeat launch differs"


@pytest.mark.parametrize("N,d,regime,fmt,p,variant", LN_CELLS)
def test_layernorm(ops, monkeypatch, N, d, regime, fmt, p, variant):
    from neko_b200._lib import Dropout
    x, g, b = _ln_inputs(N, d, regime, seed=N + d)
    keep = [t.clone() for t in (x, g, b)]
    y, y2, mean, rstd = _ln_fwd(ops, x, g, b, fmt)
    exp = R.ln_forward(x, g, b, 1e-5, fmt)
    _check("ln_mean", mean.t, exp["mean"])
    _check("ln_rstd", rstd.t, exp["rstd"])
    _check("ln_y", y.t, exp["y"])
    _check("ln_y2", y2.t, exp["y2"])
    assert int(R.ln_y2_mismatch(y.t, y2.t).sum()) == 0
    assert all(t.guards_ok() for t in (y, y2, mean, rstd))
    assert all(_same_bits(a, b_) for a, b_ in zip(keep, (x, g, b)))
    rep = _ln_fwd(ops, x, g, b, fmt)
    assert all(_same_bits(a.t, b_.t) for a, b_ in zip(rep, (y, y2, mean, rstd))), "repeat launch differs"

    # backward from the kernel's own statistics; variant: bit 0 -> dx_bf16, bit 1 -> dx_colsum; odd cells misalign dy
    gen = _gen(N * 7 + d)
    dy_val = (torch.randn(N, d, generator=gen)).to(torch.bfloat16).cuda()
    mis = (N + d) % 3 == 0
    dyg = Guarded((N, d), torch.bfloat16, offset=4 if mis else 0, init=dy_val)
    dy = dyg.t
    dx0 = torch.randn(N, d, generator=gen).cuda()
    init = [torch.randn(d, generator=gen).cuda() for _ in range(3)]
    drop = Dropout.make(torch.tensor([N, d], dtype=torch.int32, device="cuda"), 3, p) if p > 0 else None
    with_bf16, with_cs = bool(variant & 1) or p > 0, bool(variant & 2)
    want = _want_kernel(d, not mis)
    ctas = [None] if want == "rows" else [None, "1", "3", str(N)]
    for c in ctas:
        if c is None:
            monkeypatch.delenv("NEKO_LN_CTAS", raising=False)
        else:
            monkeypatch.setenv("NEKO_LN_CTAS", c)
        path = ops.layernorm_bwd_path(dy, x, g, mean.t, rstd.t, dx0, init[0], init[1], branch_drop=drop)
        assert path["kernel"] == want, (path, want)
        _seen(want, d)
        _ln_bwd_check(ops, "", dy, x, g, mean.t, rstd.t, dx0, init, with_bf16, with_cs, drop, p)
    monkeypatch.delenv("NEKO_LN_CTAS", raising=False)
    _ln_bwd_check(ops, "_ordered", dy, x, g, mean.t, rstd.t, dx0, init, with_bf16, with_cs, drop, p, ordered=True)


_FORCED_CHILD = r"""
import sys
sys.path.insert(0, sys.argv[1]); sys.path.insert(0, sys.argv[1] + "/tests")
import test_rowops_matrix_gpu as M
from neko_b200 import _lib, ops
_lib.require_device()
M.forced_cells(ops, sys.argv[2])
"""


@pytest.mark.parametrize("env,want", [("NEKO_LN_BWD_COLUMNS", "staged"), ("NEKO_LN_BWD_REGISTER", "register")])
def test_layernorm_bwd_forced_kernels(env, want):
    """Both switches are cached in statics on first use: a fresh process runs d = 768 cells under each."""
    e = {k: v for k, v in os.environ.items() if k not in ("NEKO_LN_BWD_COLUMNS", "NEKO_LN_BWD_REGISTER", "NEKO_LN_CTAS")}
    e["NEKO_LN_BWD_COLUMNS"] = "1"
    if env == "NEKO_LN_BWD_REGISTER":
        e[env] = "1"
    r = subprocess.run([sys.executable, "-c", _FORCED_CHILD, ROOT, want], env=e, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-4000:]
    _seen(want, 768)


def forced_cells(ops, want):
    """d = 768 backward cells in a process where NEKO_LN_BWD_COLUMNS / NEKO_LN_BWD_REGISTER force `want`."""
    from neko_b200._lib import Dropout
    d = 768
    for N in (37, 7680):
        x, g, b = _ln_inputs(N, d, "randn", seed=5)
        _, _, mean, rstd = _ln_fwd(ops, x, g, b, "bf16")
        gen = _gen(6)
        dy = torch.randn(N, d, generator=gen).to(torch.bfloat16).cuda()
        dx0 = torch.randn(N, d, generator=gen).cuda()
        init = [torch.randn(d, generator=gen).cuda() for _ in range(3)]
        for p in (0.0, 0.1):
            drop = Dropout.make(torch.tensor([1, 2], dtype=torch.int32, device="cuda"), 4, p) if p > 0 else None
            assert ops.layernorm_bwd_path(dy, x, g, mean.t, rstd.t, dx0, init[0], init[1])["kernel"] == want
            _ln_bwd_check(ops, "", dy, x, g, mean.t, rstd.t, dx0, init, True, True, drop, p)


def test_layernorm_rejects_strided_views(ops):
    x = torch.randn(8, 256, device="cuda")[:, :128]
    g = torch.ones(128, device="cuda")
    with pytest.raises(AssertionError):
        ops.layernorm_fwd(x, g, g)
    xc = x.contiguous()
    y, mean, rstd = ops.layernorm_fwd(xc, g, g)
    dy = torch.zeros(8, 256, device="cuda", dtype=torch.bfloat16)[:, :128]
    with pytest.raises(AssertionError):
        ops.layernorm_bwd(dy, xc, g, mean, rstd, torch.zeros_like(xc), torch.zeros_like(g), torch.zeros_like(g))


# ---------------------------------------------------------------------------------------------------
# cross entropy
# ---------------------------------------------------------------------------------------------------
CE_V = [1, 3, 4, 7, 8, 9, 1001, 2208, 52305, 52352]
CE_REGIMES = ["randn", "peaky", "flat", "extreme", "rising"]
CE_GS = [1.0, 0.25, 3.0]


def _n_rows_choices(sms):
    return [1, 37, sms, sms + 1, 2 * sms + 1, 4000]


CE_CELLS = []
for i, V in enumerate(CE_V):
    for j in range(6):
        k = i * 6 + j
        CE_CELLS.append(pytest.param(V, j, CE_REGIMES[k % 5], k % 3, k % 8, CE_GS[(k // 3) % 3],
                                     id=f"V{V}-n{j}-{CE_REGIMES[k % 5]}-ld{k % 3}-f{k % 8}"))


def _ce_logits(n, V, regime, f16, gen):
    z = torch.randn(n, V, generator=gen) * 2
    if regime == "peaky":
        z[torch.arange(n), torch.randint(0, V, (n,), generator=gen)] += 30
    elif regime == "flat":
        z = torch.full((n, V), 0.5)
    elif regime == "extreme":
        z = (torch.rand(n, V, generator=gen) * 2 - 1) * (6e4 if f16 else 80)
    elif regime == "rising":
        z = torch.linspace(-3, 3, V).repeat(n, 1) + 0.01 * torch.randn(n, V, generator=gen)
    return z.half() if f16 else z


def _targets(z, V, gen, oor):
    n = z.shape[0]
    t = torch.randint(0, V, (n,), generator=gen)
    special = [0, V - 1, min(V - 1, V // 4 * 4 + (V % 4) // 2), int(z[min(3, n - 1)].float().argmax()),
               int(z[min(4, n - 1)].float().argmin())]
    for i, s in enumerate(special[:n]):
        t[i] = s
    if oor and n >= 8:
        t[5], t[6] = -1, V
    return t


def _ld(V, variant, f16):
    w = 8 if f16 else 4
    if variant == 0:
        return V
    if variant == 1:
        return (V + 63) // 64 * 64
    return V if V % 4 == 0 and not f16 else (V + w - 1) // w * w + (w if V % w == 0 else 0)


@pytest.mark.parametrize("V,nsel,regime,ldv,flags,gs", CE_CELLS)
def test_masked_ce(ops, V, nsel, regime, ldv, flags, gs):
    sms = ops.load().neko_sm_count()
    n = _n_rows_choices(sms)[nsel]
    gen = _gen(V * 10 + nsel)
    n_pos = 2 * n + 3
    rows = torch.sort(torch.randperm(n_pos - 1, generator=gen)[:n]).values.to(torch.int32)
    lcomp, dcomp, zpad = bool(flags & 1), bool(flags & 2), bool(flags & 4)
    for f16 in (False, True):
        z = _ce_logits(n, V, regime, f16, gen)
        t = _targets(z, V, gen, oor=True)
        tokens = torch.randint(0, max(V, 1), (n_pos + 1,), generator=gen)
        tokens[rows.long() + 1] = t
        ld = _ld(V, ldv, f16)
        dt = torch.float16 if f16 else torch.float32
        store_rows = n if lcomp else n_pos
        store = Guarded((store_rows, ld), dt, fill=-7.0)
        sel = torch.arange(n) if lcomp else rows.long()
        store.t[sel.cuda(), :V] = z.to(dt).cuda()
        rows_d, tok_d = rows.cuda(), tokens.cuda()
        keep = store.buf.clone()
        ldd = _ld(V, ldv, True) if ldv else V
        d_rows = n if dcomp else n_pos
        kern = "fused_f16" if f16 else "fused"
        zc = z.cuda()
        exp_f = R.ce_reference(zc, t.cuda(), n, 1.0, kern)
        # fused (loss + unscaled gradient), then the upstream scale
        dl = Guarded((d_rows, ldd), torch.bfloat16)
        pre = dl.t.clone()
        out = ops.masked_ce_fused(store.t, V, rows_d, tok_d, dl.t, flags=flags)
        fits = (ld % (8 if f16 else 4) == 0) and (ldd % (8 if f16 else 4) == 0)
        if not fits:
            assert out is None
        else:
            assert out is not None
            loss, lse = out
            _check(f"lse_{kern}", lse, exp_f["lse"])
            assert R.ce_dlogits_violations(dl.t, pre, exp_f["dlogits"], rows_d, V, dcomp, zpad) == 0, kern
            r = (torch.arange(n) if dcomp else rows.long()).cuda()
            _note(f"dlogits_{kern}", dl.t[r, :V], exp_f["dlogits"])
            assert dl.guards_ok() and torch.equal(store.buf.view(torch.int16 if f16 else torch.int32),
                                                  keep.view(torch.int16 if f16 else torch.int32))
            dl2 = Guarded((d_rows, ldd), torch.bfloat16)
            out2 = ops.masked_ce_fused(store.t, V, rows_d, tok_d, dl2.t, flags=flags)
            assert _same_bits(dl2.t, dl.t) and _same_bits(out2[1], lse) and _same_bits(out2[0], loss), "repeat launch differs"
            if dl.t.numel() % 8 == 0:
                before = dl.t.clone()
                g_t = torch.tensor(gs, device="cuda")
                ops.ce_scale_grad(dl.t, g_t)
                want = R.ce_scale_exact(before, gs)
                nan = torch.isnan(before.float())
                assert bool(((_bits(dl.t) == _bits(want)) | (nan & torch.isnan(dl.t.float()))).all()), "ce_scale_grad"
                _check(f"dlogits_{kern}_scaled", dl.t[r, :V], R.ce_scaled(exp_f["dlogits"], gs))
        if f16:
            continue
        # two-pass forward / backward
        loss, row_lse, row_loss = ops.masked_ce_fwd(store.t, V, rows_d, tok_d, flags=flags & 1)
        exp = R.ce_reference(zc, t.cuda(), n, gs, "two_pass")
        _check("lse_two_pass", row_lse, exp["lse"])
        _check("row_loss", row_loss, exp["row_loss"])
        _check("loss", loss, R.ce_loss_expected(row_loss))
        rep = ops.masked_ce_fwd(store.t, V, rows_d, tok_d, flags=flags & 1)
        assert all(_same_bits(a, b) for a, b in zip(rep, (loss, row_lse, row_loss)))
        dl = Guarded((d_rows, ldd), torch.bfloat16)
        pre = dl.t.clone()
        g_t = torch.tensor(gs, device="cuda")
        ops.masked_ce_bwd(store.t, V, rows_d, tok_d, row_lse, g_t, dl.t, flags=flags)
        assert R.ce_dlogits_violations(dl.t, pre, exp["dlogits"], rows_d, V, dcomp, zpad) == 0
        _note("dlogits_two_pass", dl.t[(torch.arange(n) if dcomp else rows.long()).cuda(), :V], exp["dlogits"])
        dl2 = Guarded((d_rows, ldd), torch.bfloat16)
        ops.masked_ce_bwd(store.t, V, rows_d, tok_d, row_lse, g_t, dl2.t, flags=flags)
        assert _same_bits(dl2.t, dl.t) and dl.guards_ok() and store.guards_ok()
        assert torch.equal(store.buf.view(torch.int32), keep.view(torch.int32))


@pytest.mark.parametrize("V,f16,fits", [(56320, False, True), (56321, False, False), (112640, True, True), (112641, True, False)])
def test_masked_ce_fused_shared_memory_limit(ops, V, f16, fits):
    n = 3
    gen = _gen(V)
    z = _ce_logits(n, V, "randn", f16, gen)
    ld = (V + 7) // 8 * 8
    store = torch.zeros(n, ld, dtype=torch.float16 if f16 else torch.float32, device="cuda")
    store[:, :V] = z.cuda()
    t = torch.randint(0, V, (n,), generator=gen)
    rows = torch.arange(n, dtype=torch.int32, device="cuda")
    tokens = torch.zeros(n + 1, dtype=torch.int64)
    tokens[1:] = t
    dl = torch.full((n, ld), math.nan, dtype=torch.bfloat16, device="cuda")
    out = ops.masked_ce_fused(store, V, rows, tokens.cuda(), dl, flags=ops.CE_LOGITS_COMPACT | ops.CE_DLOGITS_COMPACT | ops.CE_ZERO_PAD)
    if not fits:
        assert out is None
        assert bool(torch.isnan(dl.float()).all()), "nothing may be launched"
        return
    kern = "fused_f16" if f16 else "fused"
    exp = R.ce_reference(z.cuda(), t.cuda(), n, 1.0, kern)
    _check(f"lse_{kern}", out[1], exp["lse"])
    assert R.ce_dlogits_violations(dl, torch.full_like(dl, math.nan), exp["dlogits"], rows, V, True, True) == 0


# ---------------------------------------------------------------------------------------------------
# GeGLU and casts
# ---------------------------------------------------------------------------------------------------
GEGLU_N = [8, 4096, 7680 * 3072]


@pytest.mark.parametrize("n", GEGLU_N)
@pytest.mark.parametrize("act_f16,out_f16,with_bf16", [(a, o, b) for a in (0, 1) for o in (0, 1) for b in (0, 1)])
def test_geglu_fwd(ops, n, act_f16, out_f16, with_bf16):
    gen = _gen(n + 4 * act_f16 + 2 * out_f16 + with_bf16)
    adt = torch.float16 if act_f16 else torch.bfloat16
    odt = torch.float16 if out_f16 else torch.bfloat16
    act = (torch.randn(n, generator=gen) * 300).to(adt).cuda()
    gate = (torch.randn(n, generator=gen) * 100).to(torch.bfloat16).cuda()
    keep = (act.clone(), gate.clone())
    out, ob = Guarded((n,), odt), Guarded((n,), torch.bfloat16) if with_bf16 else None
    ops.geglu_fwd(act, gate, out.t, ob.t if ob else None)
    want, want_b = R.geglu_fwd_exact(act, gate, "f16" if out_f16 else "bf16")
    R.assert_bits(out.t, want, "geglu out")
    if ob:
        R.assert_bits(ob.t, want_b, "geglu out_bf16")
        assert ob.guards_ok()
    assert out.guards_ok() and _same_bits(act, keep[0]) and _same_bits(gate, keep[1])


@pytest.mark.parametrize("n", GEGLU_N)
def test_geglu_bwd(ops, n):
    gen = _gen(n + 11)
    pre = torch.linspace(-10, 10, n)
    pre[n // 2] = 0.0
    pre = pre[torch.randperm(n, generator=gen)].to(torch.bfloat16).cuda()
    dh = torch.randn(n, generator=gen).to(torch.bfloat16).cuda()
    gate = torch.randn(n, generator=gen).to(torch.bfloat16).cuda()
    keep = [t.clone() for t in (dh, pre, gate)]
    dg, dp = Guarded((n,), torch.bfloat16), Guarded((n,), torch.bfloat16)
    ops.geglu_bwd(dh, pre, gate, dg.t, dp.t)
    exp = R.geglu_bwd(dh, pre, gate)
    _check("geglu_d_gate", dg.t, exp["d_gate"])
    _check("geglu_d_pre", dp.t, exp["d_pre"])
    assert dg.guards_ok() and dp.guards_ok() and all(_same_bits(a, b) for a, b in zip(keep, (dh, pre, gate)))
    dg2, dp2 = Guarded((n,), torch.bfloat16), Guarded((n,), torch.bfloat16)
    ops.geglu_bwd(dh, pre, gate, dg2.t, dp2.t)
    assert _same_bits(dg2.t, dg.t) and _same_bits(dp2.t, dp.t)


@pytest.mark.parametrize("n", [0, 1, 2, 3, 4, 1001, 4096, 7680 * 769 + 3])
def test_casts(ops, n):
    gen = _gen(n + 17)
    src = torch.randn(n, generator=gen) * 3e4
    if n >= 4:
        src[:4] = torch.tensor([65504.0, 65520.0, -1e6, 1e-8])
    src = src.cuda()
    keep = src.clone()
    for fmt, dt in (("bf16", torch.bfloat16), ("f16", torch.float16)):
        dst = Guarded((n,), dt)
        ops.cast_bf16(src, dst.t)
        R.assert_bits(dst.t, R.cast_exact(src, fmt), f"cast {fmt}")
        assert dst.guards_ok()
    a, b = Guarded((n,), torch.float16), Guarded((n,), torch.bfloat16)
    ops.cast_dual(src, a.t, b.t)
    R.assert_bits(a.t, R.cast_exact(src, "f16"), "cast_dual f16")
    R.assert_bits(b.t, R.cast_exact(src, "bf16"), "cast_dual bf16")
    assert a.guards_ok() and b.guards_ok() and _same_bits(src, keep)

"""Deterministic training mode (GatoPolicy.deterministic, DESIGN.md "Deterministic training mode") on the GPU.

Per ordered kernel: against an fp64 reference within a per-element bound, against its default (atomic) twin within the same
bound, and bit-identical across grid configurations -- the default grid, NEKO_ORDERED_CTAS = 1 and 7, and a run beside a
co-resident neko_debug_spin on another stream -- with inputs unchanged and nothing written outside the outputs.

The bound of a fixed-order fp32 sum of n terms, each computed with at most k roundings, is (n + k) u sum|term| with
u = 2^-24 (plus half an ulp of the result for a final rounding); every comparison below states its n and k.

End to end: two freshly built, identically seeded policies through five Trainer steps (dropout 0.1, two micro-batches) on a
mixed image / text / control batch, padded and packed, CUDA graphs on and off; the second run in a separate process with
NEKO_GEMM_SMS and the CTA caps changed.  Losses, the gradient arena after every backward, parameters and AdamW moments must
be bitwise equal.  GPU only (-m gpu)."""
import contextlib
import copy
import ctypes as C
import gc
import os
import subprocess
import sys
import weakref

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
U = 2.0 ** -24
GUARD = 64
SENT = 12345.0


@pytest.fixture(scope="module")
def ops():
    from neko_b200 import ops as o
    o.load()
    return o


def _guarded(init: torch.Tensor):
    """init's values in the middle of a buffer with GUARD-element sentinel bands on both sides (16-byte aligned view)."""
    n = init.numel()
    buf = torch.full((n + 2 * GUARD,), SENT, dtype=init.dtype, device="cuda")
    v = buf[GUARD:GUARD + n].view(init.shape)
    v.copy_(init)
    return buf, v


def _guards_ok(buf, n):
    s = torch.tensor(SENT, dtype=buf.dtype, device=buf.device)
    return bool((buf[:GUARD] == s).all()) and bool((buf[GUARD + n:] == s).all())


@contextlib.contextmanager
def _env(**kw):
    old = {k: os.environ.get(k) for k in kw}
    os.environ.update({k: str(v) for k, v in kw.items()})
    try:
        yield
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


def _grid_runs(run):
    """run() -> tuple of output tensors (fresh copies).  Four grid configurations; all must agree bit for bit."""
    from neko_b200 import _lib
    outs = [run()]
    for cap in (1, 7):
        with _env(NEKO_ORDERED_CTAS=cap):
            outs.append(run())
    side = torch.cuda.Stream()
    torch.cuda.synchronize()
    with torch.cuda.stream(side):   # 2 ms of co-resident spinning CTAs on another stream
        _lib.check(_lib.load().neko_debug_spin(C.c_int(2 * _lib.load().neko_sm_count()), C.c_int(128), C.c_longlong(2_000_000),
                                               C.c_int(0), _lib.stream_ptr()), "neko_debug_spin")
    outs.append(run())
    torch.cuda.synchronize()
    for o in outs[1:]:
        for a, b in zip(outs[0], o):
            assert torch.equal(a.view(torch.int32) if a.dtype == torch.float32 else a, b.view(torch.int32) if b.dtype == torch.float32 else b)
    return outs[0]


def _check_bound(got, ref64, mag64, n, k, what):
    bound = (n + k) * U * mag64 + U * ref64.abs() + 1e-38
    err = (got.double() - ref64).abs()
    assert bool(torch.isfinite(got).all()), what
    ratio = float((err / bound).max())
    assert ratio <= 1.0, f"{what}: worst err/bound {ratio:.3f}"
    return bound


def _ws(nbytes):
    return torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device="cuda")


# ---------------------------------------------------------------------------------------------------------------------------
# LayerNorm backward
# ---------------------------------------------------------------------------------------------------------------------------
LN_CASES = [(1000, 768, True, 0.0), (1000, 768, True, 0.1), (333, 100, False, 0.0), (130, 2048, True, 0.1), (64, 4, True, 0.0),
            (7680, 768, True, 0.1)]


@pytest.mark.parametrize("N,d,colsum,p", LN_CASES)
def test_layernorm_bwd_ordered(ops, N, d, colsum, p):
    from neko_b200._lib import Dropout
    g = torch.Generator(device="cuda").manual_seed(N + d)
    x = torch.randn(N, d, device="cuda", generator=g) * 2 + 0.5
    gamma = torch.randn(d, device="cuda", generator=g)
    beta = torch.randn(d, device="cuda", generator=g)
    _, mean, rstd = ops.layernorm_fwd(x, gamma, beta)
    dy = torch.randn(N, d, device="cuda", generator=g).bfloat16()
    dx0 = torch.randn(N, d, device="cuda", generator=g)
    seed = torch.tensor([7, 9], dtype=torch.int32, device="cuda")
    drop = Dropout.make(seed, 6, p) if p > 0 else None
    inputs = [t.clone() for t in (x, gamma, mean, rstd, dy)]
    acc0 = torch.randn(3, d, device="cuda", generator=g)    # outputs accumulate: start from non-zero values

    def run(ordered):
        bufs = [_guarded(acc0[i].clone()) for i in range(3)]
        dxb, dx = _guarded(dx0.clone())
        dbb, db16 = _guarded(torch.zeros(N, d, device="cuda").bfloat16())
        args = (dy, x, gamma, mean, rstd, dx, bufs[0][1], bufs[1][1])
        kw = dict(dx_bf16=db16, dx_colsum=bufs[2][1] if colsum else None, branch_drop=drop)
        if ordered:
            ops.layernorm_bwd_ordered(*args, _ws(ops.layernorm_bwd_ordered_workspace_bytes(N, d)), **kw)
        else:
            ops.layernorm_bwd(*args, **kw)
        torch.cuda.synchronize()
        for b, v in bufs + [(dxb, dx)]:
            assert _guards_ok(b, v.numel())
        assert _guards_ok(dbb, N * d)
        return tuple(v.clone() for _, v in bufs) + (dx.clone(), db16.clone())

    got = _grid_runs(lambda: run(True))
    for a, b in zip(inputs, (x, gamma, mean, rstd, dy)):
        assert torch.equal(a, b)
    dflt = run(False)
    # fp64 reference from the kernels' inputs: xhat = (x - mean) * rstd (2 roundings), term = dy * xhat (1 more)
    xh = (x.double() - mean.double()[:, None]) * rstd.double()[:, None]
    dyd = dy.double()
    terms = [dyd * xh, dyd]
    if colsum:   # the branch gradient the kernel summed: its own fp32 dx output times the mask multiplier (1 rounding)
        mult = torch.ones(N, d, device="cuda")
        if drop is not None:
            mult = ops.dropout_mask(N, d, drop, "cuda").float() * drop.scale
        terms.append((got[3] * mult).double())
    for i, t in enumerate(terms):
        ref = acc0[i].double() + t.sum(0)
        mag = acc0[i].double().abs() + t.abs().sum(0)
        b = _check_bound(got[i], ref, mag, N, 4, f"ln {['dgamma', 'dbeta', 'colsum'][i]}")
        assert bool(((got[i].double() - dflt[i].double()).abs() <= 2 * b).all())
    if not colsum:
        assert torch.equal(got[2], acc0[2])
    # the row outputs use the warp-per-row kernel's math: identical where the default runs that kernel
    if d % 128 == 0 and d <= 1024:
        assert torch.equal(got[3], dflt[3]) and torch.equal(got[4], dflt[4])
    else:
        assert torch.allclose(got[3], dflt[3], rtol=1e-5, atol=1e-5 * float(dflt[3].abs().max()))


# ---------------------------------------------------------------------------------------------------------------------------
# bias column sums
# ---------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("M,N,ld,acc", [(7680, 2304, 2304, True), (7680, 3072, 3072, False), (1000, 77, 80, True), (63, 130, 130, False),
                                        (1, 768, 768, True)])
def test_colsum_ordered(ops, M, N, ld, acc):
    g = torch.Generator(device="cuda").manual_seed(M + N)
    X = torch.randn(M, ld, device="cuda", generator=g).bfloat16()
    Xv = X[:, :N]
    X0 = X.clone()
    init = torch.randn(N, device="cuda", generator=g)

    def run(ordered):
        buf, out = _guarded(init.clone())
        if ordered:
            ops.colsum_ordered(Xv, out, _ws(ops.colsum_ordered_workspace_bytes(M, N)), accumulate=acc)
        else:
            ops.colsum(Xv, out, accumulate=acc)
        torch.cuda.synchronize()
        assert _guards_ok(buf, N)
        return (out.clone(),)

    got = _grid_runs(lambda: run(True))[0]
    assert torch.equal(X, X0)
    base = init.double() if acc else torch.zeros(N, dtype=torch.float64, device="cuda")
    ref = base + Xv.double().sum(0)
    mag = base.abs() + Xv.double().abs().sum(0)
    b = _check_bound(got, ref, mag, M, 2, "colsum")
    assert bool(((got.double() - run(False)[0].double()).abs() <= 2 * b).all())


# ---------------------------------------------------------------------------------------------------------------------------
# sum of squares
# ---------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [1, 8195, 1 << 20, 30_000_001])
def test_sumsq_ordered(ops, n):
    g = torch.Generator(device="cuda").manual_seed(n)
    x = torch.randn(n, device="cuda", generator=g) * 1e-2
    x0 = x.clone()

    def run(ordered):
        buf, out = _guarded(torch.full((1,), 0.25, device="cuda"))
        if ordered:
            ops.sumsq_ordered(x, out[0], _ws(ops.sumsq_ordered_workspace_bytes(n)))
        else:
            ops.sumsq(x, out[0])
        torch.cuda.synchronize()
        assert _guards_ok(buf, 1)
        return (out.clone(),)

    got = _grid_runs(lambda: run(True))[0]
    assert torch.equal(x, x0)
    ref = 0.25 + (x.double() ** 2).sum()
    b = _check_bound(got, ref.reshape(1), ref.reshape(1), n, 2, "sumsq")
    assert bool(((got.double() - run(False)[0].double()).abs() <= 2 * b).all())


# ---------------------------------------------------------------------------------------------------------------------------
# embedding backward (sorted scatter-add)
# ---------------------------------------------------------------------------------------------------------------------------
def _embed_states(packed, collide):
    from oracle import gato_oracle as O
    from test_packed_gpu import _packed_state, _padded_state
    from test_policy_gpu import make_policy
    cfg = O.GatoConfig(embed_dim=64, layers=1, heads=1, context_len=1024, text_tokens=50257)
    m = make_policy(cfg)
    batch = O.synth_batch("cfg5", batch=8)
    st = _packed_state(m, batch) if packed else _padded_state(m, batch)
    if collide:   # every (or every second) id-carrying row points at one table row
        t = st.tokens
        if collide == "all":
            t.fill_(51000)
        else:
            t[::2] = 51000
    return m, st


@pytest.mark.parametrize("packed", [False, True])
@pytest.mark.parametrize("collide", [None, "half", "all"])
def test_embed_bwd_ordered(ops, packed, collide):
    m, st = _embed_states(packed, collide)
    d = m.embed_dim
    rows = st.plan.token_rows
    g = torch.Generator(device="cuda").manual_seed(3 + packed)
    tok0 = st.tokens.clone()

    def run(ordered, dx):
        outs = [_guarded(torch.zeros_like(m.embed_token.weight)), _guarded(torch.zeros_like(m.pos_embed_observation.weight)),
                _guarded(torch.zeros(d, device="cuda")), _guarded(torch.zeros(max(st.plan.n_patch_rows, 1), d, device="cuda"))]
        v = [o[1] for o in outs]
        if ordered:
            ws = _ws(ops.embed_bwd_ordered_workspace_bytes(st.plan.B, st.tok_params))
            ops.embed_bwd_ordered(st.descs, st.plan.B, d, st.tok_params, st.tokens, dx, v[0], v[1], v[2], ws, v[3], packed=packed)
        else:
            ops.embed_bwd(st.descs, st.plan.B, d, st.tok_params, st.tokens, dx, v[0], v[1], v[2], v[3], packed=packed)
        torch.cuda.synchronize()
        for b, t in outs:
            assert _guards_ok(b, t.numel())
        return tuple(t.clone() for t in v)

    # multiples of 1/16 below 1: every sum is exact in fp32 whatever the order, so ordered == default bit for bit
    dx_exact = torch.randint(-8, 9, (rows, d), device="cuda", generator=g).float() / 16
    for a, b in zip(run(True, dx_exact), run(False, dx_exact)):
        assert torch.equal(a, b)
    dx = torch.randn(rows, d, device="cuda", generator=g)
    dx0 = dx.clone()
    got = _grid_runs(lambda: run(True, dx))
    assert torch.equal(dx, dx0) and torch.equal(st.tokens, tok0)
    # bound: a table row sums at most `rows` terms; sum|term| from the exact-order-free run on |dx| (fp64 upper bound below)
    dflt = run(False, dx)
    mag = [t.double() * (1 + rows * U) for t in run(False, dx.abs())]
    for a, b, mg, name in zip(got, dflt, mag, ("embed_token", "pos_embed", "separator", "patch")):
        bound = (rows + 2) * U * mg + 1e-38
        assert bool(((a.double() - b.double()).abs() <= 2 * bound).all()), name


# ---------------------------------------------------------------------------------------------------------------------------
# patch backward: residual block (fixed chunks) and position tables (sorted scatter-add)
# ---------------------------------------------------------------------------------------------------------------------------
def test_patch_pos_bwd_ordered(ops):
    from neko_b200._lib import _p, check, load, stream_ptr
    P, d, nr, nc = 3000, 768, 16, 16
    g = torch.Generator(device="cuda").manual_seed(5)
    rb = torch.randint(0, nr, (P,), device="cuda", generator=g, dtype=torch.int32)
    cb = torch.randint(0, nc, (P,), device="cuda", generator=g, dtype=torch.int32)
    rb[: P // 2] = 3    # heavy collisions in the row table

    def run(ordered, dx):
        outs = [_guarded(torch.zeros(nr, d, device="cuda")), _guarded(torch.zeros(nc, d, device="cuda"))]
        if ordered:
            ops.patch_pos_bwd_ordered(dx, rb, cb, outs[0][1], outs[1][1], _ws(ops.patch_pos_bwd_ordered_workspace_bytes(P, nr, nc)))
        else:
            check(load().neko_patch_pos_bwd(_p(dx), C.c_int(P), C.c_int(d), _p(rb), _p(cb), _p(outs[0][1]), _p(outs[1][1]), stream_ptr()),
                  "neko_patch_pos_bwd")
        torch.cuda.synchronize()
        for b, t in outs:
            assert _guards_ok(b, t.numel())
        return tuple(t.clone() for _, t in outs)

    dx_exact = torch.randint(-8, 9, (P, d), device="cuda", generator=g).float() / 16
    for a, b in zip(run(True, dx_exact), run(False, dx_exact)):
        assert torch.equal(a, b)
    dx = torch.randn(P, d, device="cuda", generator=g)
    got = _grid_runs(lambda: run(True, dx))
    for a, tab_bins, n in zip(got, (rb, cb), (nr, nc)):
        ref = torch.zeros(n, d, dtype=torch.float64, device="cuda").index_add_(0, tab_bins.long(), dx.double())
        mag = torch.zeros(n, d, dtype=torch.float64, device="cuda").index_add_(0, tab_bins.long(), dx.double().abs())
        _check_bound(a, ref, mag, P, 1, "patch_pos")


def test_patch_resblock_bwd_ordered(ops):
    from neko_b200._lib import _p, check, load, stream_ptr
    lib = load()
    n_img, H, W, Cm, groups = 5, 64, 48, 128, 32
    P = n_img * (H // 16) * (W // 16)
    g = torch.Generator(device="cuda").manual_seed(9)
    img = torch.randint(0, 256, (n_img, 3, H, W), device="cuda", generator=g).float()
    w1 = torch.randn(Cm, 3, 3, 3, device="cuda", generator=g) * 0.2
    b1 = torch.randn(Cm, device="cuda", generator=g) * 0.1
    gw = 1 + 0.1 * torch.randn(Cm, device="cuda", generator=g)
    gb = 0.1 * torch.randn(Cm, device="cuda", generator=g)
    w2 = torch.randn(3, Cm, 3, 3, device="cuda", generator=g) * 0.05
    b2 = torch.zeros(3, device="cuda")
    out = torch.empty(P, 768, dtype=torch.float16, device="cuda")
    stats = torch.empty(P, groups, 2, device="cuda")
    check(lib.neko_patch_resblock_fwd(_p(img), C.c_int(0), C.c_int(n_img), C.c_int(H), C.c_int(W), C.c_int(16), C.c_int(Cm), C.c_int(groups),
                                      _p(w1), _p(b1), _p(gw), _p(gb), _p(w2), _p(b2), _p(out), _p(None), _p(stats), stream_ptr()),
          "neko_patch_resblock_fwd")
    dpatch = torch.randn(P, 768, device="cuda", generator=g).bfloat16()
    ins = [t.clone() for t in (img, w1, b1, gw, gb, w2, stats, dpatch)]
    shapes = [w1.shape, b1.shape, gw.shape, gb.shape, w2.shape, b2.shape]

    def run(ordered):
        outs = [_guarded(torch.zeros(s, device="cuda")) for s in shapes]
        v = [o[1] for o in outs]
        if ordered:
            ops.patch_resblock_bwd_ordered(img, False, n_img, H, W, 16, Cm, groups, w1, b1, gw, gb, w2, stats, dpatch, *v,
                                           _ws(ops.patch_resblock_bwd_ordered_workspace_bytes(n_img, H, W, 16)))
        else:
            check(lib.neko_patch_resblock_bwd(_p(img), C.c_int(0), C.c_int(n_img), C.c_int(H), C.c_int(W), C.c_int(16), C.c_int(Cm),
                                              C.c_int(groups), _p(w1), _p(b1), _p(gw), _p(gb), _p(w2), _p(stats), _p(dpatch),
                                              *[_p(t) for t in v], stream_ptr()), "neko_patch_resblock_bwd")
        torch.cuda.synchronize()
        for b, t in outs:
            assert _guards_ok(b, t.numel())
        return tuple(t.clone() for t in v)

    got = _grid_runs(lambda: run(True))
    for a, b in zip(ins, (img, w1, b1, gw, gb, w2, stats, dpatch)):
        assert torch.equal(a, b)
    # the per-patch math is the default kernel's; only the order in which patch partials are added differs.  Each output
    # element sums P per-patch partials: bound (P + 2) u sum|partial|, with sum|partial| <= the largest |partial| times P,
    # estimated from the default result's scale (the per-patch partials are O(max|grad| / sqrt(P)) for random dY)
    dflt = run(False)
    for a, b, name in zip(got, dflt, ("conv1.w", "conv1.b", "gn.w", "gn.b", "conv2.w", "conv2.b")):
        scale = float(b.abs().max())
        assert bool(((a - b).abs() <= (P + 2) * U * 4 * scale * P ** 0.5).all()), name
        assert float(a.abs().max()) > 0, name


# ---------------------------------------------------------------------------------------------------------------------------
# GEMM flag
# ---------------------------------------------------------------------------------------------------------------------------
def test_gemm_deterministic_plan(ops):
    a = torch.randn(52352, 256, device="cuda").bfloat16()        # head dgrad shape: K = the padded vocabulary
    b = torch.randn(52352, 768, device="cuda").bfloat16()
    kw = dict(a_mn=True, b_mn=True, epilogue=ops.EPI_F32, M=256, N=768, K=52352)
    assert ops.gemm_plan(a, b, **kw)["splits"] > 1               # the default planner splits K here
    for env in ({}, {"NEKO_GEMM_SPLITS": 3}):
        with _env(**env):
            pl = ops.gemm_plan(a, b, deterministic=True, **kw)
            assert pl["splits"] == 1 and pl["streamk"] == 0, (env, pl)
    x = torch.randn(5000, 1024, device="cuda").bfloat16()
    w = torch.randn(768, 1024, device="cuda").bfloat16()
    with _env(NEKO_GEMM_STREAMK=1, NEKO_GEMM_BN=128, NEKO_GEMM_PAIR=0):     # 40 x 6 tiles on 148 workers
        assert ops.gemm_plan(x, w)["streamk"] == 1
        pl = ops.gemm_plan(x, w, deterministic=True)
        assert pl["streamk"] == 0 and pl["splits"] == 1


_GEMM_CHILD = r"""
import sys, torch
sys.path.insert(0, sys.argv[1])
from neko_b200 import ops
g = torch.Generator(device="cuda").manual_seed(1)
a = torch.randn(52352, 256, device="cuda", generator=g).bfloat16()
b = torch.randn(52352, 768, device="cuda", generator=g).bfloat16()
c = torch.randn(256, 768, device="cuda", generator=g)
outs = []
for acc in (False, True):
    o = c.clone()
    ops.gemm(a, b, a_mn=True, b_mn=True, epilogue=ops.EPI_F32, out=o, M=256, N=768, K=52352, accumulate=acc, deterministic=True)
    outs.append(o)
x = torch.randn(5000, 1024, device="cuda", generator=g).bfloat16()
w = torch.randn(768, 1024, device="cuda", generator=g).bfloat16()
outs.append(ops.gemm(x, w, deterministic=True).float())
torch.cuda.synchronize()
torch.save([o.cpu() for o in outs], sys.argv[2])
"""


def test_gemm_deterministic_independent_of_grid(tmp_path):
    res = []
    for i, sms in enumerate((None, "40")):
        env = dict(os.environ, NEKO_GEMM_SPLITS="3", NEKO_GEMM_STREAMK="1")
        if sms:
            env["NEKO_GEMM_SMS"] = sms
        path = str(tmp_path / f"g{i}.pt")
        r = subprocess.run([sys.executable, "-c", _GEMM_CHILD, ROOT, path], env=env, capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr[-3000:]
        res.append(torch.load(path))
    for a, b in zip(*res):
        assert torch.equal(a, b)


# ---------------------------------------------------------------------------------------------------------------------------
# end to end: Trainer steps
# ---------------------------------------------------------------------------------------------------------------------------
_E2E_CHILD = r"""
import copy, json, sys, torch
sys.path.insert(0, sys.argv[1]); sys.path.insert(0, sys.argv[1] + "/tests")
from test_deterministic_gpu import e2e_run
res = {}
for packed in (False, True):
    for graphs in (False, True):
        res[f"{int(packed)}{int(graphs)}"] = e2e_run(packed, graphs, True)
torch.save(res, sys.argv[2])
"""


def _mixed_samples(n, seed=0):
    """cfg5 at a reduced size: text, caption (64 x 64 uint8 frame + text), VQA-shaped caption, MuJoCo-shaped control and
    Atari-shaped control (32 x 32 frames), cycling."""
    rs = np.random.RandomState(seed)
    out = []
    for i in range(n):
        k = i % 5
        if k == 0:
            out.append({"text": rs.randint(0, 300, size=(40,)).tolist()})
        elif k in (1, 2):
            out.append({"images": torch.from_numpy(rs.randint(0, 256, size=(1, 3, 64, 64)).astype(np.uint8)),
                        "text": torch.from_numpy(rs.randint(0, 300, size=(12 if k == 1 else 8,)).astype(np.int64))})
        elif k == 3:
            out.append({"continuous_obs": torch.from_numpy((rs.standard_normal((6, 7)) * 3).astype(np.float32)),
                        "continuous_actions": torch.from_numpy(np.clip(rs.standard_normal((6, 3)), -1, 1).astype(np.float32))})
        else:
            out.append({"images": torch.from_numpy(rs.randint(0, 256, size=(3, 3, 32, 32)).astype(np.float32)),
                        "discrete_actions": torch.from_numpy(rs.randint(0, 4, size=(3, 1)).astype(np.int32))})
    return out


class _Seq:
    kind = "control"

    def __init__(self, samples):
        self.samples, self.i = samples, 0

    def sample_batch(self, n, max_tokens=None):
        s = self.samples[self.i % len(self.samples)]
        self.i += 1
        return [copy.deepcopy(s)]


class _Tok:
    def __init__(self, n):
        self.vocab_size = n


def e2e_run(packed: bool, graphs: bool, deterministic: bool, steps: int = 5):
    """Five Trainer steps from a fresh, seeded policy; returns losses, the gradient arena after every backward, parameters and
    AdamW moments (CPU tensors)."""
    from neko_b200.policy import GatoPolicy
    from neko_b200.training.arguments import TrainingArgs
    from neko_b200.training.trainer import FusedAdamW, Trainer
    # CUDA graphs held by unreachable objects (earlier policies in reference cycles) must be freed now: torch does not collect
    # before a capture, and a graph destroyed by the cyclic collector in the middle of one invalidates that capture
    gc.collect()
    torch.manual_seed(2024)
    m = GatoPolicy(device="cuda", embed_dim=64, layers=2, heads=2, dropout=0.1, resid_mid_channels=128, context_len=128,
                   text_tokenizer=_Tok(300))
    m.materialize_logits = False
    m.use_cuda_graphs = graphs
    m.pack_sequences = packed
    m.deterministic = deterministic
    args = TrainingArgs()
    args.batch_size, args.sequence_length = 5, 128
    args.gradient_accumulation_steps = 2
    args.learning_rate, args.warmup_steps, args.training_steps = 1e-3, 2, 10
    args.text_prop = args.caption_prop = args.vqa_prop = 0.0
    opt = FusedAdamW(m, lr=args.learning_rate, betas=(args.beta_1, args.beta_2), eps=args.adam_eps, weight_decay=args.weight_decay)
    tr = Trainer(m, opt, [_Seq(_mixed_samples(60))], args)
    grads = []
    arena = m._grad_arena
    engine_backward = type(m)._engine_backward
    pol = weakref.ref(m)   # the spy must not make the policy part of a reference cycle (see gc.collect() above)

    def spy(st, g_loss):
        engine_backward(pol(), st, g_loss)
        grads.append(arena.detach().clone().cpu())
    m._engine_backward = spy
    torch.manual_seed(99)
    losses = [l for l, _ in tr.train(steps)]
    torch.cuda.synchronize()
    out = {"losses": losses, "grads": grads, "params": m._param_arena.detach().cpu().clone(),
           "m": opt.exp_avg.cpu().clone(), "v": opt.exp_avg_sq.cpu().clone(),
           "names": list(m._order), "offs": {n: int(m._offs[n]) for n in m._order}}
    del m._engine_backward
    return out


def _bits(t):
    return t.view(torch.int32) if t.dtype == torch.float32 else t


def test_training_steps_bitwise_reproducible(tmp_path):
    path = str(tmp_path / "run_b.pt")
    env = dict(os.environ, NEKO_GEMM_SMS="100", NEKO_ORDERED_CTAS="7", NEKO_LN_CTAS="5")
    r = subprocess.run([sys.executable, "-c", _E2E_CHILD, ROOT, path], env=env, capture_output=True, text=True, timeout=1800)
    assert r.returncode == 0, r.stderr[-4000:]
    other = torch.load(path)
    for packed in (False, True):
        for graphs in (False, True):
            a = e2e_run(packed, graphs, True)
            b = other[f"{int(packed)}{int(graphs)}"]
            assert a["losses"] == b["losses"], (packed, graphs, a["losses"], b["losses"])
            assert len(a["grads"]) == len(b["grads"]) == 10
            for i, (ga, gb) in enumerate(zip(a["grads"], b["grads"])):
                assert torch.equal(_bits(ga), _bits(gb)), (packed, graphs, "grad after backward", i)
            for k in ("params", "m", "v"):
                assert torch.equal(_bits(a[k]), _bits(b[k])), (packed, graphs, k)


@pytest.mark.parametrize("packed", [False, True])
def test_deterministic_matches_default_mode(packed):
    """Same seeds, same batches: the two modes differ by reassociation only.  One step, compared before the optimiser
    amplifies anything."""
    det = e2e_run(packed, False, True, steps=1)
    dft = e2e_run(packed, False, False, steps=1)
    for a, b in zip(det["losses"], dft["losses"]):
        assert abs(a - b) <= 1e-5 * abs(b), (det["losses"], dft["losses"])
    names, offs = det["names"], det["offs"]
    total = det["grads"][0].numel()
    for gi in range(2):
        ga, gb = det["grads"][gi], dft["grads"][gi]
        for k, n in enumerate(names):
            lo = offs[n]
            hi = offs[names[k + 1]] if k + 1 < len(names) else total
            a, b = ga[lo:hi].double(), gb[lo:hi].double()
            nb = float(b.norm())
            if nb == 0.0:
                assert float(a.norm()) == 0.0, n
                continue
            cos = float(a @ b) / (float(a.norm()) * nb)
            assert cos >= 0.99999, (n, cos)


@pytest.mark.parametrize("name", ["cfg2", "cfg5"])
def test_model_scale_parity_deterministic(golden_dir, name, monkeypatch):
    """The logits / loss / gradient-cosine gates of test_model_scale_parity, with the policy in deterministic mode."""
    import test_policy_gpu as T
    make = T.make_policy

    def make_det(*a, **kw):
        m = make(*a, **kw)
        m.deterministic = True
        return m
    monkeypatch.setattr(T, "make_policy", make_det)
    T.test_model_scale_parity(golden_dir, name, "eval")


_DP_CHILD = r"""
import os, sys, torch
import torch.distributed as dist
sys.path.insert(0, os.environ["NEKO_ROOT"]); sys.path.insert(0, os.environ["NEKO_ROOT"] + "/tests")
rank = int(os.environ["RANK"])
torch.cuda.set_device(rank)
dist.init_process_group("nccl", device_id=torch.device("cuda", rank))
from neko_b200 import dp
from test_deterministic_gpu import _Tok, _mixed_samples
from neko_b200.policy import GatoPolicy
torch.manual_seed(5)
m = GatoPolicy(device=f"cuda:{rank}", embed_dim=64, layers=2, heads=2, dropout=0.1, resid_mid_channels=128, context_len=128,
               text_tokenizer=_Tok(300))
m.materialize_logits = False
m.deterministic = True
dp.broadcast_parameters(m)
sync = dp.attach(m, bucket_bytes=1 << 16, backend="p2p")
torch.manual_seed(100 + rank)
m.train()
batch = _mixed_samples(5, seed=rank)
_, loss = m.forward(inputs=batch, compute_loss=True)
loss.backward()
torch.cuda.synchronize()
torch.save(m._grad_arena.cpu(), os.environ["OUT"] + f".{rank}")
dist.barrier()
dist.destroy_process_group()
"""


def test_dp_world2_deterministic(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    runs = []
    for rep in range(2):
        out = str(tmp_path / f"dp{rep}")
        port = 29800 + (os.getpid() % 500) + rep
        procs = [subprocess.Popen([sys.executable, "-c", _DP_CHILD],
                                  env=dict(os.environ, RANK=str(r), WORLD_SIZE="2", LOCAL_RANK=str(r), MASTER_ADDR="127.0.0.1",
                                           MASTER_PORT=str(port), NEKO_ROOT=ROOT, OUT=out)) for r in range(2)]
        assert all(p.wait(timeout=900) == 0 for p in procs)
        runs.append([torch.load(out + f".{r}") for r in range(2)])
    assert torch.equal(_bits(runs[0][0]), _bits(runs[0][1]))
    assert torch.equal(_bits(runs[0][0]), _bits(runs[1][0]))

"""Every attention path against the fp64 reference and per-element bound of tests/_attn_ref.py.

Padded forward and backward (mma.sync at head dims 16 / 32 / 64 / 128; the tcgen05 forward under NEKO_ATTN_TC=1 where the
shape allows it, and the query of which one ran), the packed variable-length kernels, and single-query decode against the
key / value cache.  Every cell checks out, out2, lse, dQ, dK, dV and delta element by element, requires dead rows to be
exact zeros (+inf lse), prefills outputs with NaN inside guarded buffers (every element written, nothing outside), checks
that the inputs are unchanged, that a repeat launch is bit-identical, and that the padding rows of qkv / dout do not
reach any live output.  The largest err / bound ratio per output kind is printed at the end (pytest -s).
GPU only (-m gpu)."""
import pytest
import torch

import _attn_ref as R

pytestmark = pytest.mark.gpu

NAN16 = 0x7FC1           # a NaN in both bf16 and fp16
NAN32 = 0x7FC00011
GUARD = 8                # guard elements on each side of an output (16 bytes or more)
HEADROOM = {}            # output kind -> largest err / bound seen


@pytest.fixture(scope="module")
def ops():
    from neko_b200 import _lib, ops as _ops
    _lib.require_device()
    yield _ops
    print("\nattention err/bound headroom: " + ", ".join(f"{k} {v:.3g}" for k, v in sorted(HEADROOM.items())))


def _bits(t):
    return t.contiguous().view(torch.int32 if t.dtype == torch.float32 else torch.int16).clone()


class Out:
    """An output view inside a NaN-filled buffer with GUARD elements on either side."""

    def __init__(self, shape, dtype):
        n = 1
        for s in shape:
            n *= s
        self.nan = NAN32 if dtype == torch.float32 else NAN16
        self.storage = torch.full((n + 2 * GUARD,), self.nan, dtype=torch.int32 if dtype == torch.float32 else torch.int16,
                                  device="cuda").view(dtype)
        self.view = self.storage[GUARD:GUARD + n].view(shape)

    def guards_intact(self):
        b = _bits(self.storage)
        return bool((b[:GUARD] == self.nan).all() and (b[-GUARD:] == self.nan).all())


def _check(kind, got, exp, dims):
    R.assert_within(got, exp, kind, dims)
    HEADROOM[kind] = max(HEADROOM.get(kind, 0.0), R.worst_ratio(got, exp))


def _heads(x, H):
    """[..., S, H*dh] -> [..., H, S, dh]"""
    *lead, S, d = x.shape
    return x.reshape(*lead, S, H, d // H).transpose(-2, -3)


def _drop(ops, p, seed):
    if not p:
        return None
    from neko_b200._lib import Dropout
    return Dropout.make(torch.tensor([seed, 77], dtype=torch.int32, device="cuda"), 3, p)


def _inputs(g, rows, d, regime, H):
    qkv = torch.randn(*rows, 3 * d, generator=g)
    dout = torch.randn(*rows, d, generator=g) * 0.5
    dh = d // H
    if regime == "peaky":        # scores of tens of units after sigma: exercises the flush to zero of ex2.approx.ftz
        qkv[..., :2 * d] *= 4.0
    elif regime == "rising":     # a shared feature moves each row's maximum to its latest key tile
        S = rows[-1]
        for h in range(H):
            qkv[..., h * dh] = 4.0
            qkv[..., d + h * dh] = torch.arange(S, dtype=torch.float32) * (3.0 / 64.0) * dh ** 0.5 / 4.0
    return qkv, dout


def _garbage(g, shape):
    return (torch.randint(0, 2, shape, generator=g).float() * 2 - 1) * 3e4


# ---------------------------------------------------------------------------------------------------
# one forward + backward, checked
# ---------------------------------------------------------------------------------------------------
class Run:
    """Outputs of one forward + backward into fresh guarded buffers."""

    def __init__(self, fwd, bwd, out_shape, lse_shape, qkv_shape, out_dtype):
        self.out, self.out2 = Out(out_shape, out_dtype), Out(out_shape, torch.bfloat16)
        self.lse, self.delta = Out(lse_shape, torch.float32), Out(lse_shape, torch.float32)
        self.dqkv = Out(qkv_shape, torch.bfloat16)
        fwd(self)
        bwd(self)
        torch.cuda.synchronize()

    def all(self):
        return {"out": self.out, "out2": self.out2, "lse": self.lse, "delta": self.delta, "dqkv": self.dqkv}


def _verify(label, fwd, bwd, shapes, out_dtype, H, expect, dims, live_rows, inputs, repad=None):
    """Run, check against the reference, repeat, and (repad) check the padding invariance."""
    saved = [_bits(t) for t in inputs]
    run = Run(fwd, bwd, *shapes, out_dtype)
    f = expect["fwd"]
    _check("out", _heads(run.out.view, H), f.out, dims)
    _check("out2", _heads(run.out2.view, H), f.out2, dims)
    _check("lse", run.lse.view, f.lse, dims[:-1])
    bw = expect["bwd"](_heads(run.out.view, H))
    _check("delta", run.delta.view, bw["delta"], dims[:-1])
    dq, dk, dv = (_heads(x, H) for x in run.dqkv.view.chunk(3, dim=-1))
    _check("dQ", dq, bw["dq"], dims)
    _check("dK", dk, bw["dk"], dims)
    _check("dV", dv, bw["dv"], dims)
    for name, o in run.all().items():
        assert o.guards_intact(), f"{label}: {name} written outside its view"
    for t, s in zip(inputs, saved):
        assert torch.equal(_bits(t), s), f"{label}: an input changed"
    again = Run(fwd, bwd, *shapes, out_dtype)
    for name, o in run.all().items():
        assert torch.equal(_bits(o.view), _bits(again.all()[name].view)), f"{label}: {name} differs between two launches"
    if repad is not None:
        repad()
        other = Run(fwd, bwd, *shapes, out_dtype)
        for name, o in run.all().items():
            a, b = o.view, other.all()[name].view
            m = live_rows(name)
            assert torch.equal(a[m], b[m]), f"{label}: {name} of live rows depends on the padding rows"
    return run


# ---------------------------------------------------------------------------------------------------
# padded layout
# ---------------------------------------------------------------------------------------------------
SHAPES = [   # (B, S, S_valid, first_valid, H)
    (1, 1, 1, [0], 2),
    (2, 63, 63, [0, 62], 2),                 # a single live row
    (3, 65, 65, [0, 1, 64], 3),              # odd H: dh 32 stays on mma.sync under NEKO_ATTN_TC=1
    (2, 128, 128, [63, 64], 2),
    (3, 129, 129, [0, 127, 128], 2),
    (2, 200, 191, [5, 130], 4),              # S_valid inside a tile
    (2, 256, 192, [0, 129], 2),              # S_valid on a 64-row boundary, not a 128-row one
    (3, 494, 494, [0, 17, 300], 24),         # the training configuration's shape
    (2, 1024, 1000, [0, 255], 2),
    (1, 2048, 2048, [0], 2),                 # 32 key tiles
    (2, 160, 150, [150, 3], 2),              # an empty sample: first_valid = S_valid
]
PADDED = [(si, dh, p) for si in range(len(SHAPES)) for dh in (16, 32, 64, 128) for p in (0.0, 0.2)]
REGIMES = [(si, dh, p, regime) for si in (2, 5) for dh in (32, 64) for p in (0.0, 0.2) for regime in ("peaky", "rising", "garbage")]


def _tc_path(dh, H):
    return dh == 64 or (dh == 32 and H % 2 == 0)


def run_padded(ops, monkeypatch, si, dh, p, regime, out_dtype, seed):
    B, S, S_valid, fv, H = SHAPES[si]
    d = H * dh
    g = torch.Generator().manual_seed(seed)
    qkv, dout = _inputs(g, (B, S), d, regime, H)
    pos = torch.arange(S).reshape(1, S)
    dead = (pos < torch.tensor(fv).reshape(B, 1)) | (pos >= S_valid)     # [B, S] padding rows
    if regime == "garbage":
        qkv[dead] = _garbage(g, (int(dead.sum()), 3 * d))
        dout[dead] = _garbage(g, (int(dead.sum()), d))
    qkv, dout = qkv.bfloat16().cuda(), dout.bfloat16().cuda()
    fv_t = torch.tensor(fv, dtype=torch.int32, device="cuda")
    drop = _drop(ops, p, seed)
    mult = None if drop is None else R.padded_mult(ops.dropout_mask(B * H * S, S, drop, "cuda"), drop.scale, B, H, S)
    q, k, v = R.split_heads(qkv, H)
    f = R.forward(q, k, v, R.padded_vis(S, S_valid, fv, "cuda"), mult, R.TORCH_FMT[out_dtype])
    expect = {"fwd": f, "bwd": lambda o16: R.backward(f, _heads(dout, H), o16)}
    dead_c = dead.cuda()

    def live_rows(name):   # index of the live rows of each output
        if name in ("lse", "delta"):
            return ~dead_c[:, None, :].expand(B, H, S)
        return ~dead_c

    def repad():
        n = int(dead.sum())
        if regime == "garbage":
            qkv[dead_c] = torch.randn(n, 3 * d, generator=g).bfloat16().cuda()
            dout[dead_c] = torch.randn(n, d, generator=g).bfloat16().cuda()
        else:
            qkv[dead_c] = _garbage(g, (n, 3 * d)).bfloat16().cuda()
            dout[dead_c] = _garbage(g, (n, d)).bfloat16().cuda()

    for tc in (0, 1):
        monkeypatch.setenv("NEKO_ATTN_TC", str(tc))
        label = f"B{B} S{S} Sv{S_valid} fv{fv} H{H} dh{dh} p{p} {regime} {out_dtype} tc{tc}"
        out_probe = torch.empty(B * S * d + GUARD, dtype=out_dtype, device="cuda")[GUARD:].view(B, S, d)
        path = ops.attention_fwd_path(qkv, fv_t, H, S_valid, out=out_probe, out2=out_probe.bfloat16(), drop=drop)
        assert path == ("tc" if tc and _tc_path(dh, H) else "mma"), f"{label}: forward path {path}"

        def fwd(r):
            ops.attention_fwd(qkv, fv_t, H, S_valid, out=r.out.view, lse=r.lse.view, out2=r.out2.view, drop=drop)

        def bwd(r):
            ops.attention_bwd(qkv, r.out.view, dout, r.lse.view, fv_t, H, S_valid, dqkv=r.dqkv.view, delta=r.delta.view, drop=drop)

        _verify(label, fwd, bwd, ((B, S, d), (B, H, S), (B, S, 3 * d)), out_dtype, H, expect, ("b", "h", "row", "col"), live_rows,
                (qkv, dout), repad if (tc == 1 and bool(dead.any())) else None)


@pytest.mark.parametrize("si,dh,p", PADDED, ids=[f"{'x'.join(map(str, SHAPES[s][:3]))}-H{SHAPES[s][4]}-dh{dh}-p{p}" for s, dh, p in PADDED])
def test_padded(ops, monkeypatch, si, dh, p):
    idx = PADDED.index((si, dh, p))
    run_padded(ops, monkeypatch, si, dh, p, "randn", torch.float16 if idx % 2 else torch.bfloat16, 1000 + idx)


@pytest.mark.parametrize("si,dh,p,regime", REGIMES, ids=[f"S{SHAPES[s][1]}-dh{dh}-p{p}-{r}" for s, dh, p, r in REGIMES])
def test_padded_value_regimes(ops, monkeypatch, si, dh, p, regime):
    idx = REGIMES.index((si, dh, p, regime))
    run_padded(ops, monkeypatch, si, dh, p, regime, torch.bfloat16 if idx % 2 else torch.float16, 5000 + idx)


# ---------------------------------------------------------------------------------------------------
# packed (variable-length) layout
# ---------------------------------------------------------------------------------------------------
VARLEN = [(lens, width, dh, p) for lens, width in (((1, 64, 65, 200), 200), ((128, 3, 700), 768)) for dh in (16, 32, 64, 128)
          for p in (0.0, 0.2)]


@pytest.mark.parametrize("lens,width,dh,p", VARLEN, ids=[f"{'-'.join(map(str, l))}-w{w}-dh{dh}-p{p}" for l, w, dh, p in VARLEN])
def test_varlen(ops, lens, width, dh, p):
    idx = VARLEN.index((lens, width, dh, p))
    H = 3 if idx % 4 == 1 else 2
    d = H * dh
    out_dtype = torch.float16 if idx % 2 else torch.bfloat16
    cu = [0]
    for n in lens:
        cu.append(cu[-1] + n)
    T, S_max = cu[-1], max(lens)
    fv = [width - n for n in lens]
    g = torch.Generator().manual_seed(7000 + idx)
    qkv, dout = _inputs(g, (T,), d, "randn", H)
    qkv, dout = qkv.bfloat16().cuda(), dout.bfloat16().cuda()
    cu_t = torch.tensor(cu, dtype=torch.int32, device="cuda")
    fv_t = torch.tensor(fv, dtype=torch.int32, device="cuda")
    drop = _drop(ops, p, 7000 + idx)
    B = len(lens)
    mult = None if drop is None else R.packed_mult(ops.dropout_mask(B * H * width, width, drop, "cuda"), drop.scale, cu, fv, H, width)
    q, k, v = R.split_heads(qkv[None], H)
    f = R.forward(q, k, v, R.packed_vis(cu, "cuda"), mult, R.TORCH_FMT[out_dtype])
    fq = R.Forward(*(R.Expected(e.ref[0], e.tol[0], e.fmt) for e in f[:3]), f.ctx)

    def bwd_expect(o16):
        return {k_: R.Expected(e.ref[0], e.tol[0], e.fmt) for k_, e in R.backward(f, _heads(dout, H)[None], o16[None]).items()}

    def fwd(r):
        ops.attention_varlen_fwd(qkv, cu_t, fv_t, H, S_max, width, out=r.out.view, lse=r.lse.view, out2=r.out2.view, drop=drop)

    def bwd(r):
        ops.attention_varlen_bwd(qkv, r.out.view, dout, r.lse.view, cu_t, fv_t, H, S_max, width, dqkv=r.dqkv.view, delta=r.delta.view,
                                 drop=drop)

    _verify(f"varlen {lens} w{width} H{H} dh{dh} p{p}", fwd, bwd, ((T, d), (H, T), (T, 3 * d)), out_dtype, H, {"fwd": fq, "bwd": bwd_expect},
            ("h", "row", "col"), None, (qkv, dout, cu_t, fv_t))


# ---------------------------------------------------------------------------------------------------
# decode
# ---------------------------------------------------------------------------------------------------
DECODE = [(n, dh) for n in (1, 2, 31, 128, 129, 1000, 4097, 8192) for dh in (2, 8, 16, 32, 64, 128)]


@pytest.mark.parametrize("n,dh", DECODE, ids=[f"len{n}-dh{dh}" for n, dh in DECODE])
def test_decode(ops, n, dh):
    idx = DECODE.index((n, dh))
    H = (1, 3, 24)[idx % 3]
    out_dtype = torch.float16 if idx % 2 else torch.bfloat16
    d = H * dh
    g = torch.Generator().manual_seed(9000 + idx)
    cap = n + 5                                   # the cache holds more rows than len; rows from len onward are NaN
    kc = torch.full((cap, d), NAN16, dtype=torch.int16).view(torch.bfloat16)
    vc = kc.clone()
    kc[:n] = torch.randn(n, d, generator=g).bfloat16()
    vc[:n] = torch.randn(n, d, generator=g).bfloat16()
    q = (torch.randn(d, generator=g) * 2.0).bfloat16().cuda()
    kc, vc = kc.cuda(), vc.cuda()
    exp = R.decode(q.view(H, dh), kc[:n].view(n, H, dh), vc[:n].view(n, H, dh), R.TORCH_FMT[out_dtype])
    saved = [_bits(t) for t in (q, kc, vc)]
    out = Out((d,), out_dtype)
    ops.attention_decode(q, kc, vc, n, H, out.view)
    torch.cuda.synchronize()
    assert bool(torch.isfinite(out.view).all()), "decode read past len"
    _check("decode", out.view.view(H, dh), exp, ("h", "col"))
    assert out.guards_intact()
    assert all(torch.equal(_bits(t), s) for t, s in zip((q, kc, vc), saved))
    again = Out((d,), out_dtype)
    ops.attention_decode(q, kc, vc, n, H, again.view)
    assert torch.equal(_bits(out.view), _bits(again.view))

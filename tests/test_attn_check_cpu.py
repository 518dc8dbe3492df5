"""The attention reference and per-element check of tests/_attn_ref.py (used by tests/test_attention_matrix_gpu.py) are
strict: they accept the correctly rounded results and a kernel-faithful fp32 emulation of the tiled algorithm at both
tile widths, and reject each of the subtle mistakes an attention kernel can make.  Also the argument checks of the
attention entry points, which return before any CUDA call.  CPU only."""
import ctypes as C
import math

import pytest
import torch

import _attn_ref as R

B, H, S, S_VALID = 2, 2, 200, 190
FIRST_VALID = (0, 37)


def _keep(shape, p, g):
    thr = int(round(p * 65536.0))
    keep = torch.rand(*shape, generator=g) >= thr / 65536.0
    return keep, float(torch.tensor(65536.0 / (65536.0 - thr), dtype=torch.float32))


def make(seed, dh, regime="randn", p=0.0, S_valid=S_VALID, first_valid=FIRST_VALID):
    """qkv [B, S, 3d] and dout [B, S, d] (bf16), split into heads, with the visibility and the dropout multipliers."""
    g = torch.Generator().manual_seed(seed * 131 + dh)
    d = H * dh
    qkv = torch.randn(B, S, 3 * d, generator=g)
    if regime == "peaky":
        qkv[..., :2 * d] *= 4.0
    q, k, v = R.split_heads(qkv, H)
    if regime == "rising":
        # a shared feature: query feature 0 is 4, key feature 0 grows so that the score rises by 3 per 64 keys and each
        # row's maximum moves to its latest tile
        q[..., 0] = 4.0
        k[..., 0] = torch.arange(S, dtype=torch.float32) * (3.0 / 64.0) * math.sqrt(dh) / 4.0
    qkv = qkv.bfloat16()
    q, k, v = R.split_heads(qkv, H)
    dout = (torch.randn(B, H, S, dh, generator=g) * 0.5).bfloat16()
    vis = R.padded_vis(S, S_valid, first_valid)
    mult = None
    if p > 0:
        keep, scale = _keep((B * H * S, S), p, g)
        mult = R.padded_mult(keep, scale, B, H, S)
    return q, k, v, dout, vis, mult


def _nbad(out, exp):
    return int(R.violations(out, exp).sum())


def _fwd_bwd(case, out_fmt="bf16"):
    q, k, v, dout, vis, mult = case
    f = R.forward(q, k, v, vis, mult, out_fmt)
    o16 = R.exact_output(f.out)
    return f, R.backward(f, dout, o16), o16


# ---------------------------------------------------------------------------------------------------
# accepted
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("out_fmt", ["bf16", "f16"])
@pytest.mark.parametrize("p", [0.0, 0.2])
@pytest.mark.parametrize("regime", ["randn", "peaky", "rising"])
@pytest.mark.parametrize("dh", [16, 32])
def test_accepts_correctly_rounded_and_emulated(dh, regime, p, out_fmt):
    case = make(1, dh, regime, p)
    q, k, v, dout, vis, mult = case
    f, bw, o16 = _fwd_bwd(case, out_fmt)
    for name, exp in (("out", f.out), ("out2", f.out2), ("lse", f.lse)) + tuple(bw.items()):
        assert _nbad(R.exact_output(exp), exp) == 0, name
    for tile in (64, 128):
        out, lse = R.emulate_forward(q, k, v, vis, mult, tile, out_fmt)
        R.assert_within(out, f.out, f"emulated out (tile {tile})")
        R.assert_within(lse, f.lse, f"emulated lse (tile {tile})")
        out2, _ = R.emulate_forward(q, k, v, vis, mult, tile, "bf16")
        R.assert_within(out2, f.out2, f"emulated out2 (tile {tile})")
        # the backward of the emulated forward: its own lse and 16-bit O
        bw_e = R.backward(f, dout, out)
        dq, dk, dv, delta = R.emulate_backward(q, k, v, vis, lse, dout, out, mult)
        for name, got in (("dq", dq), ("dk", dk), ("dv", dv), ("delta", delta)):
            R.assert_within(got, bw_e[name], f"emulated {name} (tile {tile})")


def test_accepts_emulated_varlen_and_decode():
    g = torch.Generator().manual_seed(5)
    cu = [0, 1, 65, 130, 200]
    dh, T = 32, 200
    qkv = torch.randn(1, T, 3 * H * dh, generator=g).bfloat16()
    q, k, v = R.split_heads(qkv, H)
    vis = R.packed_vis(cu)
    f = R.forward(q, k, v, vis)
    for tile in (64, 128):
        out, lse = R.emulate_forward(q, k, v, vis, None, tile)
        R.assert_within(out, f.out, "varlen out")
        R.assert_within(lse, f.lse, "varlen lse")
    kc = torch.randn(300, 3, 32, generator=g).bfloat16()
    vc = torch.randn(300, 3, 32, generator=g).bfloat16()
    qd = torch.randn(3, 32, generator=g).bfloat16()
    # the decode kernel in fp32: scores, exp against the maximum, P never rounded to 16 bits
    sc = (kc.float().transpose(0, 1) @ qd.float()[..., None]).squeeze(-1) * float(torch.tensor(1 / math.sqrt(32), dtype=torch.float32))
    pe = torch.exp(sc - sc.amax(-1, keepdim=True))
    od = (pe[:, None, :] @ vc.float().transpose(0, 1)).squeeze(1) / pe.sum(-1, keepdim=True)
    for fmt, dt in (("bf16", torch.bfloat16), ("f16", torch.float16)):
        exp = R.decode(qd, kc, vc, fmt)
        assert _nbad(R.exact_output(exp), exp) == 0
        R.assert_within(od.to(dt), exp, "emulated decode", dims=("h", "col"))


# ---------------------------------------------------------------------------------------------------
# rejected
# ---------------------------------------------------------------------------------------------------
def _rejects_out(case, q=None, k=None, v=None, vis=None, mult="same", out_fmt="bf16"):
    q0, k0, v0, _, vis0, mult0 = case
    good = R.forward(q0, k0, v0, vis0, mult0, out_fmt)
    bad = R.forward(q0 if q is None else q, k0 if k is None else k, v0 if v is None else v, vis0 if vis is None else vis,
                    mult0 if isinstance(mult, str) else mult, out_fmt)
    return _nbad(R.exact_output(bad.out), good.out)


def _ij():
    return torch.arange(S).reshape(S, 1), torch.arange(S).reshape(1, S)


def test_rejects_diagonal_excluded():
    case = make(2, 32)
    i, j = _ij()
    assert _rejects_out(case, vis=case[4] & (j < i)) > 0


def test_rejects_key_before_first_valid():
    case = make(2, 32)
    vis = R.padded_vis(S, S_VALID, (FIRST_VALID[0], FIRST_VALID[1] - 1))
    assert FIRST_VALID[1] >= 1 and _rejects_out(case, vis=vis) > 0


def test_rejects_skipped_key_tile():
    case = make(2, 32)
    i, j = _ij()
    vis = case[4] & ~((j >= 64) & (j < 128) & (i >= 128))    # rows of three tiles or more lose their second tile
    assert _rejects_out(case, vis=vis) > 0


@pytest.mark.parametrize("tile", [64, 128])
def test_rejects_missing_rescale(tile):
    q, k, v, _, vis, _ = make(3, 32, "rising")
    good = R.forward(q, k, v, vis)
    out, _ = R.emulate_forward(q, k, v, vis, None, tile, rescale=False)
    assert _nbad(out, good.out) > 0
    out, _ = R.emulate_forward(q, k, v, vis, None, tile)
    assert _nbad(out, good.out) == 0


def test_rejects_lse_in_log2_units():
    q, k, v, _, vis, _ = make(2, 16)
    f = R.forward(q, k, v, vis)
    assert _nbad(R.exact_output(f.lse) / math.log(2.0), f.lse) > 0


def test_rejects_dropout_mistakes():
    case = make(4, 32, p=0.2)
    q, k, v, _, vis, mult = case
    assert _rejects_out(case, mult=mult.transpose(-1, -2)) > 0                  # mask transposed
    assert _rejects_out(case, mult=(mult > 0).double()) > 0                     # kept elements not rescaled
    good = R.forward(q, k, v, vis, mult)
    PM = good.ctx["PM"]
    norm = PM.sum(-1, keepdim=True)
    out = (PM / torch.where(norm > 0, norm, torch.ones_like(norm))) @ v.double()  # dropout applied to the normaliser
    assert _nbad(R.round16(out, "bf16"), good.out) > 0


def test_rejects_backward_mistakes():
    case = make(5, 32, p=0.2)
    q, k, v, dout, vis, mult = case
    f, bw, o16 = _fwd_bwd(case)
    no_delta = R.backward(f, dout, torch.zeros_like(o16))                       # delta omitted
    assert _nbad(R.exact_output(no_delta["dq"]), bw["dq"]) > 0
    assert _nbad(R.exact_output(no_delta["dk"]), bw["dk"]) > 0
    dk_unscaled = bw["dk"].ref * math.sqrt(32)                                  # dK without sigma
    assert _nbad(R.round16(dk_unscaled, "bf16"), bw["dk"]) > 0
    dv_unmasked = f.ctx["P"].transpose(-1, -2) @ dout.double()                  # dV without the dropout mask
    assert _nbad(R.round16(dv_unmasked, "bf16"), bw["dv"]) > 0


def test_rejects_neighbouring_head():
    case = make(6, 32)
    q, k, v = case[:3]
    assert _rejects_out(case, k=torch.roll(k, 1, dims=1)) > 0
    assert _rejects_out(case, v=torch.roll(v, 1, dims=1)) > 0


def test_rejects_varlen_sample_seeing_the_next():
    g = torch.Generator().manual_seed(7)
    cu = [0, 64, 129, 200]
    qkv = torch.randn(1, 200, 3 * H * 32, generator=g).bfloat16()
    q, k, v = R.split_heads(qkv, H)
    vis = R.packed_vis(cu)
    good = R.forward(q, k, v, vis)
    bad_vis = vis.clone()
    bad_vis[..., 0:64, 64] = True                                               # sample 0 sees the first key of sample 1
    assert _nbad(R.exact_output(R.forward(q, k, v, bad_vis).out), good.out) > 0


@pytest.mark.parametrize("n", [2, 31, 1000])
def test_rejects_decode_mistakes(n):
    g = torch.Generator().manual_seed(n)
    kc = torch.randn(n, 3, 32, generator=g).bfloat16()
    vc = torch.randn(n, 3, 32, generator=g).bfloat16()
    qd = (torch.randn(3, 32, generator=g) * 2).bfloat16()
    good = R.decode(qd, kc, vc)
    assert _nbad(R.exact_output(R.decode(qd, kc[:-1], vc[:-1])), good) > 0         # last cached key dropped
    assert _nbad(R.exact_output(R.decode(qd, kc, vc, sigma=1.0)), good) > 0         # sigma missing


def test_rejects_dead_row_errors_and_nan():
    case = make(8, 16)
    f, bw, o16 = _fwd_bwd(case)
    dead_row = FIRST_VALID[1] - 1                                                # sample 1 row 36: left padding
    tiny = 2.0 ** -133                                                           # one ulp from zero (bf16 subnormal)
    for name, exp in (("out", f.out), ("dq", bw["dq"]), ("dk", bw["dk"]), ("dv", bw["dv"])):
        x = R.exact_output(exp)
        x[1, 0, dead_row, 3] = tiny
        assert _nbad(x, exp) == 1, name
        x = R.exact_output(exp)
        x[1, 0, S_VALID, 0] = -tiny                                              # right padding
        assert _nbad(x, exp) == 1, name
    lse = R.exact_output(f.lse)
    lse[1, 1, dead_row] = 1e30
    assert _nbad(lse, f.lse) == 1
    for name, exp in (("out", f.out), ("lse", f.lse), ("dq", bw["dq"]), ("delta", bw["delta"])):
        x = R.exact_output(exp)
        x[0, 1, 100, ...] = math.nan
        assert _nbad(x, exp) >= 1, name


def test_failure_message_names_the_worst_element():
    case = make(9, 16)
    f, bw, _ = _fwd_bwd(case)
    x = R.exact_output(bw["dk"])
    x[1, 0, 120, 5] += 1.0
    with pytest.raises(AssertionError, match=r"dK: 1 of .*worst at \(b=1, h=0, row=120, col=5\)"):
        R.assert_within(x, bw["dk"], "dK")


# ---------------------------------------------------------------------------------------------------
# argument checks: each call returns NEKO_EINVAL before any CUDA call, so fake device pointers are never dereferenced
# ---------------------------------------------------------------------------------------------------
NEKO_EINVAL = -1
F = 0x100000          # a fake 16-byte aligned device address
MIS = F + 2           # a fake misaligned one


@pytest.fixture(scope="module")
def lib():
    from neko_b200 import _lib, build
    build.build()
    return _lib.load()


def _p(x):
    return C.c_void_p(x)


def _fwd_args(qkv=F, out=F, B=2, S=64, S_valid=64, H=2, dh=32, out2=0):
    return (_p(qkv), _p(F), _p(out), _p(out2), _p(F), C.c_int(B), C.c_int(S), C.c_int(S_valid), C.c_int(H), C.c_int(dh), C.c_int(0))


FWD_BAD = {"dh8": dict(dh=8), "dh96": dict(dh=96), "S_valid0": dict(S_valid=0), "S_valid_gt_S": dict(S_valid=65),
           "qkv_misaligned": dict(qkv=MIS), "out_misaligned": dict(out=MIS), "rows_2pow32": dict(B=1 << 16, H=1 << 8, S=1 << 8, S_valid=1)}


@pytest.mark.parametrize("case", sorted(FWD_BAD))
def test_attention_fwd_rejects(lib, case):
    args = _fwd_args(**FWD_BAD[case])
    assert lib.neko_attention_fwd(*args, None, None) == NEKO_EINVAL
    assert lib.neko_attention_fwd_path(*args, None) == NEKO_EINVAL


def _bwd_args(qkv=F, out=F, dout=F, B=2, S=64, S_valid=64, H=2, dh=32):
    return (_p(qkv), _p(out), _p(dout), _p(F), _p(F), _p(F), _p(F), C.c_int(B), C.c_int(S), C.c_int(S_valid), C.c_int(H), C.c_int(dh),
            C.c_int(0), None, None)


BWD_BAD = dict(FWD_BAD, dout_misaligned=dict(dout=MIS))


@pytest.mark.parametrize("case", sorted(BWD_BAD))
def test_attention_bwd_rejects(lib, case):
    assert lib.neko_attention_bwd(*_bwd_args(**BWD_BAD[case])) == NEKO_EINVAL


VARLEN_BAD = {"dh8": dict(dh=8), "dh96": dict(dh=96), "S_max0": dict(S_max=0), "S_max_gt_width": dict(S_max=65),
              "qkv_misaligned": dict(qkv=MIS), "out_misaligned": dict(out=MIS), "dout_misaligned": dict(dout=MIS),
              "rows_2pow32": dict(B=1 << 16, H=1 << 8, S_width=1 << 8, S_max=1)}


@pytest.mark.parametrize("case", sorted(VARLEN_BAD))
def test_attention_varlen_rejects(lib, case):
    a = dict(qkv=F, out=F, dout=F, B=2, T=100, S_max=64, S_width=64, H=2, dh=32)
    a.update(VARLEN_BAD[case])
    sizes = [C.c_int(a[n]) for n in ("B", "T", "S_max", "S_width", "H", "dh")]
    if case != "dout_misaligned":
        assert lib.neko_attention_varlen_fwd(_p(a["qkv"]), _p(F), _p(F), _p(a["out"]), None, _p(F), *sizes, C.c_int(0), None, None) == NEKO_EINVAL
    assert lib.neko_attention_varlen_bwd(_p(a["qkv"]), _p(a["out"]), _p(a["dout"]), _p(F), _p(F), _p(F), _p(F), _p(F), *sizes, C.c_int(0),
                                         None, None) == NEKO_EINVAL


DECODE_BAD = {"len0": dict(n=0), "len8193": dict(n=8193), "dh6": dict(dh=6), "q_misaligned": dict(q=MIS), "k_misaligned": dict(k=MIS)}


@pytest.mark.parametrize("case", sorted(DECODE_BAD))
def test_attention_decode_rejects(lib, case):
    a = dict(q=F, k=F, n=16, dh=32)
    a.update(DECODE_BAD[case])
    assert lib.neko_attention_decode(_p(a["q"]), _p(a["k"]), _p(F), C.c_int(a["n"]), C.c_int(2), C.c_int(a["dh"]), _p(F), C.c_int(0),
                                     None) == NEKO_EINVAL


def test_attention_fwd_path(lib, monkeypatch):
    """Which forward kernel runs: mma.sync unless NEKO_ATTN_TC=1 and the shape suits the tcgen05 kernel.  Launches nothing."""
    monkeypatch.delenv("NEKO_ATTN_TC", raising=False)
    for dh in (16, 32, 64, 128):
        assert lib.neko_attention_fwd_path(*_fwd_args(dh=dh), None) == 0
    monkeypatch.setenv("NEKO_ATTN_TC", "1")
    want = {(16, 2): 0, (32, 2): 1, (32, 3): 0, (64, 2): 1, (64, 3): 1, (128, 2): 0}
    for (dh, h), path in want.items():
        assert lib.neko_attention_fwd_path(*_fwd_args(dh=dh, H=h), None) == path, (dh, h)
    assert lib.neko_attention_fwd_path(*_fwd_args(dh=64, out2=MIS), None) == 0   # a misaligned second copy falls back
    monkeypatch.setenv("NEKO_ATTN_TC", "0")
    assert lib.neko_attention_fwd_path(*_fwd_args(dh=64), None) == 0

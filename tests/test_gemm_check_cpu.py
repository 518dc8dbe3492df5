"""The GEMM reference and per-element check of tests/_gemm_ref.py (used by tests/test_gemm_matrix_gpu.py) are strict:
they accept the exactly rounded result and a plain fp32 evaluation of the same epilogue, and reject each of the subtle
mistakes a tcgen05 epilogue can make.  CPU only."""
import pytest
import torch

import _gemm_ref as R

M, N, K = 96, 96, 256   # three 32-column chunks, four 64-deep k-blocks


def _operands(seed, dtype=torch.bfloat16):
    g = torch.Generator().manual_seed(seed)
    a = (torch.randn(M, K, generator=g) * 0.5).to(dtype)
    b = (torch.randn(N, K, generator=g) * (3.0 / K ** 0.5)).to(dtype)   # |acc| ~ 1.5: GELU sees its curved part
    bias = torch.randn(N, generator=g) * 0.5
    resid = torch.randn(M, N, generator=g)
    pre = (torch.randn(M, N, generator=g) * 2.0).to(torch.bfloat16)
    keep = torch.rand(M, N, generator=g) >= 0.25
    scale = float(torch.tensor(1.0 / 0.75, dtype=torch.float32))
    mult = keep.float() * scale
    return a, b, bias, resid, pre, mult


CASES = {   # name -> (epilogue, reference kwargs, output checked)
    "bf16_bias": (R.EPI_BF16, dict(bias=True), "C"),
    "f16_out": (R.EPI_BF16, dict(bias=True, c_fmt="f16"), "C"),
    "f32_bias": (R.EPI_F32, dict(bias=True), "C"),
    "f32_accumulate": (R.EPI_F32, dict(c_init=True), "C"),
    "gelu_pre": (R.EPI_GELU_BF16, dict(bias=True), "C"),
    "gelu_erf": (R.EPI_GELU_BF16, dict(bias=True), "C2"),
    "gelu_tanh_f16": (R.EPI_GELU_BF16, dict(bias=True, gelu_tanh=True, c2_fmt="f16"), "C2"),
    "gelu_c3": (R.EPI_GELU_BF16, dict(bias=True, c3=True, c2_fmt="f16"), "C3"),
    "dgelu_erf": (R.EPI_DGELU_BF16, dict(aux="pre"), "C"),
    "dgelu_tanh_f16": (R.EPI_DGELU_BF16, dict(aux="pre", gelu_tanh=True, c_fmt="f16"), "C"),
    "resid_dropout": (R.EPI_RESID_F32, dict(bias=True, aux="resid", mult=True), "C"),
    "resid_bf16_copy": (R.EPI_RESID_F32_BF16, dict(bias=True, aux="resid", mult=True), "C2"),
}


def _expected(name, seed=1, dtype=torch.bfloat16, a=None, **override):
    epi, kw, which = CASES[name]
    a0, b, bias, resid, pre, mult = _operands(seed, dtype)
    a = a0 if a is None else a
    kw = dict(kw, **override)
    acc, absacc = R.accumulator(a, b)
    args = dict(gelu_tanh=kw.get("gelu_tanh", False), c_fmt=kw.get("c_fmt", "bf16"), c2_fmt=kw.get("c2_fmt", "bf16"),
                c3=kw.get("c3", False))
    if kw.get("bias"):
        args["bias"] = bias
    if kw.get("aux") == "pre":
        args["aux"] = pre
    elif kw.get("aux") == "resid":
        args["aux"] = resid
    if kw.get("mult") is True:
        args["mult"] = mult
    elif kw.get("mult") is not None:
        args["mult"] = kw["mult"]
    if kw.get("c_init"):
        args["c_init"] = resid
    return R.epilogue_reference(acc, absacc, epi, **args)[which], (a0, b, bias, resid, pre, mult)


def _nbad(out, exp):
    return int(R.violations(out, exp, K).sum())


# ---------------------------------------------------------------------------------------------------
# accepted
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", sorted(CASES))
def test_exactly_rounded_reference_passes(name):
    exp, _ = _expected(name)
    R.assert_within(R.exact_output(exp), exp, K, name)


@pytest.mark.parametrize("name", sorted(CASES))
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
def test_plain_fp32_evaluation_passes(name, dtype):
    """What a correct kernel computes: fp32 accumulation, the epilogue in fp32, one rounding to the output format."""
    epi, kw, which = CASES[name]
    exp, (a, b, bias, resid, pre, mult) = _expected(name, dtype=dtype)
    acc = a.float() @ b.float().t()
    x = acc + bias if kw.get("bias") else acc
    tanh = "tanh" if kw.get("gelu_tanh") else "none"
    if epi in (R.EPI_BF16, R.EPI_F32):
        v = x + resid if kw.get("c_init") else x
    elif epi == R.EPI_GELU_BF16:
        v = x if which == "C" else torch.nn.functional.gelu(x, approximate=tanh)
    elif epi == R.EPI_DGELU_BF16:
        p = pre.float().requires_grad_(True)
        torch.nn.functional.gelu(p, approximate=tanh).sum().backward()
        v = acc * p.grad
    else:
        v = x * mult + resid
    fmt = exp.fmt
    out = v if fmt == "f32" else v.to(torch.float16 if fmt == "f16" else torch.bfloat16)
    R.assert_within(out, exp, K, name)


# ---------------------------------------------------------------------------------------------------
# rejected
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["bf16_bias", "f16_out", "gelu_erf", "gelu_tanh_f16", "gelu_c3", "dgelu_tanh_f16",
                                  "resid_bf16_copy"])
@pytest.mark.parametrize("n", [0, 31, 32, 95])
def test_one_ulp_off_is_rejected(name, n):
    """At the largest output of column n (where the 16-bit rounding, not the fp32 evaluation, dominates the bound)."""
    exp, _ = _expected(name)
    out = R.exact_output(exp)
    m = int(exp.ref[:, n].abs().argmax())
    err = out[m, n] - exp.ref[m, n]
    step = R._ulp(out[m, n].reshape(1), exp.fmt)[0]
    out[m, n] += step if err >= 0 else -step          # one ulp further from the exact value
    assert _nbad(out, exp) == 1


@pytest.mark.parametrize("name", ["bf16_bias", "f16_out", "gelu_erf", "gelu_tanh_f16", "gelu_c3", "dgelu_erf",
                                  "dgelu_tanh_f16", "resid_bf16_copy"])
def test_truncation_is_rejected(name):
    exp, _ = _expected(name)
    assert _nbad(R.round16(exp.ref, exp.fmt, mode="trunc"), exp) > 0


@pytest.mark.parametrize("name", ["bf16_bias", "f32_bias", "gelu_pre", "gelu_erf", "resid_dropout", "resid_bf16_copy"])
def test_missing_bias_is_rejected(name):
    exp, _ = _expected(name)
    without, _ = _expected(name, bias=False)
    assert _nbad(R.exact_output(without), exp) > 0


@pytest.mark.parametrize("name", ["bf16_bias", "f32_bias", "gelu_erf", "dgelu_erf", "resid_dropout"])
@pytest.mark.parametrize("edge", [32, 64])
def test_column_shift_at_chunk_edge_is_rejected(name, edge):
    exp, _ = _expected(name)
    out = R.exact_output(exp)
    shifted = out.clone()
    shifted[:, edge:edge + 32] = out[:, edge - 1:edge + 31]    # one 32-column chunk read one column early
    assert _nbad(shifted, exp) > 0
    shifted = out.clone()
    shifted[:, edge] = out[:, edge - 1]                        # only the first column of the chunk
    assert _nbad(shifted, exp) > 0


@pytest.mark.parametrize("name", ["f32_bias", "bf16_bias", "gelu_erf", "dgelu_erf", "resid_dropout"])
@pytest.mark.parametrize("kb", [0, 1, 3])
def test_dropped_k_block_is_rejected(name, kb):
    exp, (a, *_rest) = _expected(name)
    a_drop = a.clone()
    a_drop[:, 64 * kb:64 * (kb + 1)] = 0
    wrong, _ = _expected(name, a=a_drop)
    assert _nbad(R.exact_output(wrong), exp) > 0


@pytest.mark.parametrize("name", ["gelu_erf", "gelu_tanh_f16", "gelu_c3", "dgelu_erf", "dgelu_tanh_f16"])
def test_other_gelu_form_is_rejected(name):
    """erf GELU where the tanh form was asked for, and the reverse."""
    exp, _ = _expected(name)
    wrong, _ = _expected(name, gelu_tanh=not CASES[name][1].get("gelu_tanh", False))
    assert _nbad(R.exact_output(wrong), exp) > 0


@pytest.mark.parametrize("name", ["resid_dropout", "resid_bf16_copy"])
def test_transposed_dropout_mask_is_rejected(name):
    exp, (*_rest, mult) = _expected(name)
    wrong, _ = _expected(name, mult=mult.t().contiguous())
    assert _nbad(R.exact_output(wrong), exp) > 0


def test_nan_is_rejected():
    exp, _ = _expected("f32_bias")
    out = R.exact_output(exp)
    out[5, 7] = float("nan")
    assert _nbad(out, exp) == 1


def test_fp16_rounding_saturates_and_ties_to_even():
    x = torch.tensor([1.0 + 2.0 ** -11, 1.0 + 3 * 2.0 ** -11, 70000.0, -1e6, 2.0 ** -25, 0.0], dtype=torch.float64)
    assert R.round16(x, "f16").tolist() == [1.0, 1.0 + 2 * 2.0 ** -10, 65504.0, -65504.0, 0.0, 0.0]
    y = torch.tensor([1.0 + 2.0 ** -8, 1.0 + 3 * 2.0 ** -8, -(1.0 + 2.0 ** -8)], dtype=torch.float64)
    assert R.round16(y, "bf16").tolist() == [1.0, 1.0 + 2 * 2.0 ** -7, -1.0]
    assert R.round16(y, "bf16", mode="trunc").tolist() == [1.0, 1.0 + 2.0 ** -7, -1.0]
    r = torch.randn(4096, dtype=torch.float64, generator=torch.Generator().manual_seed(5)) * 10
    assert torch.equal(R.round16(r, "bf16"), r.float().to(torch.bfloat16).double())
    assert torch.equal(R.round16(r, "f16"), r.float().to(torch.float16).double())

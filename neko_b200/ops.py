"""Thin torch-tensor wrappers over the C ABI (include/neko_b200.h).

PyTorch is used only for device memory and streams; every computation is a call into
libneko_b200.so.  All functions enqueue on the current CUDA stream and never synchronise.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

import torch

from . import _lib
from ._lib import (EPI_BF16, EPI_DGELU_BF16, EPI_F32, EPI_GELU_BF16, EPI_RESID_F32, EPI_RESID_F32_BF16,  # noqa: F401
                   Dropout, GemmDesc, GemmPlanInfo, LnBwdPathInfo, SampleDesc, TokParams, _p, check, load, stream_ptr)


_16BIT = (torch.bfloat16, torch.float16)
GEMM_A_F16, GEMM_B_F16, GEMM_C_F16, GEMM_C2_F16, GEMM_GELU_TANH, GEMM_DETERMINISTIC = 1, 2, 4, 8, 16, 32
GEMM_TIMING = None  # list collecting (start_event, end_event, flops) per launch when set by bench.py


def _cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise _lib.NekoError("neko_b200 ops need CUDA tensors (there is no CPU path)")


# ------------------------------------------------------------------------------------------
# GEMM
# ------------------------------------------------------------------------------------------
def _ptr(t):
    return None if t is None else t.data_ptr()


_GEMM_WS = {}   # device index -> zero-initialised workspace of the stream-K launches (include/neko_b200.h: neko_gemm_desc.workspace).
# One per device: the GEMMs of a process run on one stream at a time (eager steps and graph replays never overlap).


def _gemm_workspace(device):
    key = device.index
    ws = _GEMM_WS.get(key)
    if ws is None:
        if torch.cuda.is_current_stream_capturing():
            return None                   # first use inside a capture: no allocation there, this launch runs the classic schedule
        ws = torch.zeros(int(load().neko_gemm_workspace_bytes()), dtype=torch.uint8, device=device)
        _GEMM_WS[key] = ws
    return ws


def _gemm_args(a, b, a_mn, b_mn, epilogue, out, out2, out3, bias, aux, accumulate, M, N, K, out_dtype, drop, gelu_tanh,
               deterministic=False):
    """neko_gemm_desc of one gemm() / gemm_plan() call, allocating the outputs that were not given."""
    _cuda(a, b, out, out2, out3, bias, aux)
    assert a.dtype in _16BIT and b.dtype == a.dtype, "A and B must share one 16-bit format"
    assert a.stride(1) == 1 and b.stride(1) == 1
    if M is None:
        M = a.shape[1] if a_mn else a.shape[0]
    if K is None:
        K = a.shape[0] if a_mn else a.shape[1]
    if N is None:
        N = b.shape[1] if b_mn else b.shape[0]
    bf16_out = epilogue in (EPI_BF16, EPI_GELU_BF16, EPI_DGELU_BF16)
    if out is None:
        out = torch.empty(M, N, device=a.device, dtype=out_dtype if bf16_out else torch.float32)
    if epilogue in (EPI_GELU_BF16, EPI_RESID_F32_BF16) and out2 is None:
        out2 = torch.empty(M, N, device=a.device, dtype=out_dtype)
    assert out.stride(1) == 1
    flags = (GEMM_A_F16 | GEMM_B_F16) if a.dtype == torch.float16 else 0
    flags |= GEMM_C_F16 if out.dtype == torch.float16 else 0
    flags |= GEMM_C2_F16 if (out2 is not None and out2.dtype == torch.float16) else 0
    flags |= GEMM_GELU_TANH if gelu_tanh else 0   # GELU / GELU' epilogues: tanh form ("gelu_new")
    flags |= GEMM_DETERMINISTIC if deterministic else 0   # no split-K / stream-K: bitwise reproducible
    gd = GemmDesc(M=M, N=N, K=K, a_mn=int(a_mn), b_mn=int(b_mn), epilogue=epilogue, accumulate=int(accumulate), flags=flags,
                  A=a.data_ptr(), lda=a.stride(0), B=b.data_ptr(), ldb=b.stride(0), C=out.data_ptr(), ldc=out.stride(0),
                  C2=_ptr(out2), ldc2=out2.stride(0) if out2 is not None else 0,
                  C3=_ptr(out3), ldc3=out3.stride(0) if out3 is not None else 0,
                  bias=_ptr(bias), aux=_ptr(aux), ld_aux=aux.stride(0) if aux is not None else 0)
    if drop is not None:   # RESID epilogues: C = aux + dropout(acc + bias)
        gd.drop = drop
    ws = _gemm_workspace(a.device)
    if ws is not None:
        gd.workspace, gd.workspace_bytes = ws.data_ptr(), ws.numel()
    return gd, out, out2


def gemm(a: torch.Tensor, b: torch.Tensor, *, a_mn: bool = False, b_mn: bool = False, epilogue: int = EPI_BF16,
         out: Optional[torch.Tensor] = None, out2: Optional[torch.Tensor] = None, out3: Optional[torch.Tensor] = None,
         bias: Optional[torch.Tensor] = None, aux: Optional[torch.Tensor] = None, accumulate: bool = False,
         M: Optional[int] = None, N: Optional[int] = None, K: Optional[int] = None,
         out_dtype: torch.dtype = torch.bfloat16, drop: Optional[Dropout] = None, gelu_tanh: bool = False,
         deterministic: bool = False):
    """C[M,N] = epilogue(sum_k A[m,k] B[n,k]).  deterministic: NEKO_GEMM_DETERMINISTIC (one CTA sums each element in k order).

    a: 16-bit [M,K] (a_mn=False) or [K,M] (a_mn=True); b: same format, [N,K] or [K,N]; rows may be strided
    (stride(0) is the leading dimension)."""
    gd, out, out2 = _gemm_args(a, b, a_mn, b_mn, epilogue, out, out2, out3, bias, aux, accumulate, M, N, K, out_dtype, drop,
                               gelu_tanh, deterministic)
    if GEMM_TIMING is not None:  # bench.py: CUDA events around every tensor-core launch (roofline.achieved)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        check(load().neko_gemm(C.byref(gd), stream_ptr()), "neko_gemm")
        e1.record()
        GEMM_TIMING.append((e0, e1, 2.0 * gd.M * gd.N * gd.K, (gd.M, gd.N, gd.K, int(a_mn), int(b_mn), epilogue)))
    else:
        check(load().neko_gemm(C.byref(gd), stream_ptr()), "neko_gemm")
    if out2 is not None and epilogue in (EPI_GELU_BF16, EPI_RESID_F32_BF16):
        return out, out2
    return out


def gemm_plan(a: torch.Tensor, b: torch.Tensor, *, a_mn: bool = False, b_mn: bool = False, epilogue: int = EPI_BF16,
              out: Optional[torch.Tensor] = None, out2: Optional[torch.Tensor] = None, out3: Optional[torch.Tensor] = None,
              bias: Optional[torch.Tensor] = None, aux: Optional[torch.Tensor] = None, accumulate: bool = False,
              M: Optional[int] = None, N: Optional[int] = None, K: Optional[int] = None,
              out_dtype: torch.dtype = torch.bfloat16, drop: Optional[Dropout] = None, gelu_tanh: bool = False,
              deterministic: bool = False) -> dict:
    """The schedule gemm() would launch with the same arguments (neko_gemm_plan_info as a dict); launches nothing.
    Raises NekoError where gemm() would reject the arguments."""
    gd, _, _ = _gemm_args(a, b, a_mn, b_mn, epilogue, out, out2, out3, bias, aux, accumulate, M, N, K, out_dtype, drop,
                          gelu_tanh, deterministic)
    info = GemmPlanInfo()
    check(load().neko_gemm_plan(C.byref(gd), C.byref(info)), "neko_gemm_plan")
    return {name: getattr(info, name) for name, _ in GemmPlanInfo._fields_}


# ------------------------------------------------------------------------------------------
# LayerNorm
# ------------------------------------------------------------------------------------------
def _dense(dtypes, **ts):
    """The kernels index rows as if dense: a strided view would be read as the wrong rows."""
    for name, t in ts.items():
        if t is not None:
            assert t.dtype in dtypes[name], f"{name}: dtype {t.dtype}, expected one of {dtypes[name]}"
            assert t.is_contiguous(), f"{name} must be contiguous"


_LN_FWD_DT = dict(x=(torch.float32,), gamma=(torch.float32,), beta=(torch.float32,), y=_16BIT, y2=(torch.bfloat16,),
                  mean=(torch.float32,), rstd=(torch.float32,))
_LN_BWD_DT = dict(dy=(torch.bfloat16,), x=(torch.float32,), gamma=(torch.float32,), mean=(torch.float32,), rstd=(torch.float32,),
                  dx_resid=(torch.float32,), dgamma=(torch.float32,), dbeta=(torch.float32,), dx_bf16=(torch.bfloat16,),
                  dx_colsum=(torch.float32,))


def layernorm_fwd(x: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, eps: float = 1e-5, y=None, mean=None, rstd=None,
                  out_dtype: torch.dtype = torch.bfloat16, y2=None):
    _cuda(x, gamma, beta)
    N, d = x.shape
    if y is None:
        y = torch.empty(N, d, device=x.device, dtype=out_dtype)
    if mean is None:
        mean = torch.empty(N, device=x.device, dtype=torch.float32)
    if rstd is None:
        rstd = torch.empty(N, device=x.device, dtype=torch.float32)
    _dense(_LN_FWD_DT, x=x, gamma=gamma, beta=beta, y=y, y2=y2, mean=mean, rstd=rstd)
    check(load().neko_layernorm_fwd(_p(x), _p(gamma), _p(beta), _p(y), _p(y2), _p(mean), _p(rstd), C.c_int(N), C.c_int(d),
                                    C.c_float(eps), C.c_int(int(y.dtype == torch.float16)), stream_ptr()), "neko_layernorm_fwd")
    return y, mean, rstd


def _dref(drop):
    return C.byref(drop) if drop is not None else None


def layernorm_bwd(dy_bf16, x, gamma, mean, rstd, dx_resid, dgamma, dbeta, dx_bf16=None, dx_colsum=None, branch_drop=None):
    N, d = x.shape
    _dense(_LN_BWD_DT, dy=dy_bf16, x=x, gamma=gamma, mean=mean, rstd=rstd, dx_resid=dx_resid, dgamma=dgamma, dbeta=dbeta,
           dx_bf16=dx_bf16, dx_colsum=dx_colsum)
    check(load().neko_layernorm_bwd(_p(dy_bf16), _p(x), _p(gamma), _p(mean), _p(rstd), _p(dx_resid), _p(dx_bf16),
                                    _p(dgamma), _p(dbeta), _p(dx_colsum), C.c_int(N), C.c_int(d), _dref(branch_drop), stream_ptr()),
          "neko_layernorm_bwd")


LN_BWD_KERNELS = ("rows", "staged", "register")


def layernorm_bwd_path(dy_bf16, x, gamma, mean, rstd, dx_resid, dgamma, dbeta, dx_bf16=None, dx_colsum=None, branch_drop=None) -> dict:
    """The kernel layernorm_bwd() would run with the same arguments ("rows" = warp-per-row, "staged", "register") and its
    launch shape; launches nothing.  Raises NekoError where layernorm_bwd() would reject the arguments."""
    N, d = x.shape
    info = LnBwdPathInfo()
    rc = load().neko_layernorm_bwd_path(_p(dy_bf16), _p(x), _p(gamma), _p(mean), _p(rstd), _p(dx_resid), _p(dx_bf16), _p(dgamma),
                                        _p(dbeta), _p(dx_colsum), C.c_int(N), C.c_int(d), _dref(branch_drop), C.byref(info))
    if rc < 0:
        check(rc, "neko_layernorm_bwd_path")
    return dict(kernel=LN_BWD_KERNELS[rc], grid=info.grid, rows_per_cta=info.rows_per_cta, stages=info.stages)


def geglu_fwd(act: torch.Tensor, gate: torch.Tensor, out: torch.Tensor, out_bf16: Optional[torch.Tensor] = None):
    """out = act * gate (MLP gate of --activation_fn geglu)."""
    assert gate.dtype == torch.bfloat16 and act.is_contiguous() and gate.is_contiguous() and out.is_contiguous()
    check(load().neko_geglu_fwd(_p(act), _p(gate), _p(out), _p(out_bf16), C.c_int64(act.numel()), C.c_int(int(act.dtype == torch.float16)),
                                C.c_int(int(out.dtype == torch.float16)), stream_ptr()), "neko_geglu_fwd")
    return out


def geglu_bwd(dh: torch.Tensor, pre: torch.Tensor, gate: torch.Tensor, d_gate: torch.Tensor, d_pre: torch.Tensor):
    check(load().neko_geglu_bwd(_p(dh), _p(pre), _p(gate), _p(d_gate), _p(d_pre), C.c_int64(dh.numel()), stream_ptr()), "neko_geglu_bwd")


def dropout_apply(x: torch.Tensor, drop: Optional[Dropout]):
    """x fp32 [rows, cols] *= mask * scale, in place (embd dropout, trajectory_gpt2.py:707, and its backward)."""
    if drop is None or not drop.thr16:
        return x
    rows, cols = x.shape
    check(load().neko_dropout_apply(_p(x), C.c_int64(x.stride(0)), C.c_int(rows), C.c_int(cols), C.byref(drop), stream_ptr()),
          "neko_dropout_apply")
    return x


def dropout_mask(rows: int, cols: int, drop: Dropout, device) -> torch.Tensor:
    """The keep mask (uint8 [rows, cols]) the kernels generate for this site: tests replay a step with it."""
    keep = torch.empty(rows, cols, dtype=torch.uint8, device=device)
    check(load().neko_dropout_mask(_p(keep), C.c_int(rows), C.c_int(cols), C.byref(drop), stream_ptr()), "neko_dropout_mask")
    return keep


# ------------------------------------------------------------------------------------------
# tokenise / embed
# ------------------------------------------------------------------------------------------
def tokenize_embed_fwd(descs, B: int, d: int, prm: TokParams, fvals, ivals, patch_emb, embed_table, pos_table, sep_vec,
                       tokens, target_masks, token_masks, token_embeddings, err_flag=None, packed: bool = False):
    """Ids, masks and embeddings of a planned batch: [B*width] rows, or the packed [T] rows (no padding) when ``packed``."""
    fn = load().neko_tokenize_embed_packed_fwd if packed else load().neko_tokenize_embed_fwd
    check(fn(_p(descs), C.c_int(B), C.c_int(d), C.byref(prm), _p(fvals), _p(ivals), _p(patch_emb), _p(embed_table), _p(pos_table),
             _p(sep_vec), _p(tokens), _p(target_masks), _p(token_masks), _p(token_embeddings), _p(err_flag), stream_ptr()),
          "neko_tokenize_embed_packed_fwd" if packed else "neko_tokenize_embed_fwd")


def embed_bwd(descs, B: int, d: int, prm: TokParams, tokens, d_emb, d_embed_table, d_pos_table, d_sep, d_patch_emb=None,
              packed: bool = False):
    fn = load().neko_embed_packed_bwd if packed else load().neko_embed_bwd
    check(fn(_p(descs), C.c_int(B), C.c_int(d), C.byref(prm), _p(tokens), _p(d_emb), _p(d_embed_table), _p(d_pos_table), _p(d_sep),
             _p(d_patch_emb), stream_ptr()), "neko_embed_packed_bwd" if packed else "neko_embed_bwd")


# ------------------------------------------------------------------------------------------
# attention
# ------------------------------------------------------------------------------------------
def attention_fwd(qkv: torch.Tensor, first_valid: torch.Tensor, H: int, S_valid: Optional[int] = None, out=None, lse=None,
                  out_dtype: torch.dtype = torch.bfloat16, out2=None, drop=None):
    B, S, three_d = qkv.shape
    d = three_d // 3
    dh = d // H
    if out is None:
        out = torch.empty(B, S, d, device=qkv.device, dtype=out_dtype)
    if lse is None:
        lse = torch.empty(B, H, S, device=qkv.device, dtype=torch.float32)
    check(load().neko_attention_fwd(_p(qkv), _p(first_valid), _p(out), _p(out2), _p(lse), C.c_int(B), C.c_int(S),
                                    C.c_int(S if S_valid is None else S_valid), C.c_int(H), C.c_int(dh),
                                    C.c_int(int(out.dtype == torch.float16)), _dref(drop), stream_ptr()), "neko_attention_fwd")
    return out, lse


def attention_fwd_path(qkv: torch.Tensor, first_valid: torch.Tensor, H: int, S_valid: Optional[int] = None, out=None, lse=None,
                       out_dtype: torch.dtype = torch.bfloat16, out2=None, drop=None) -> str:
    """The forward kernel attention_fwd() would run with the same arguments: "mma" (mma.sync) or "tc" (tcgen05);
    launches nothing.  Raises NekoError where attention_fwd() would reject the arguments."""
    B, S, three_d = qkv.shape
    d = three_d // 3
    if out is None:
        out = torch.empty(B, S, d, device=qkv.device, dtype=out_dtype)
    if lse is None:
        lse = torch.empty(B, H, S, device=qkv.device, dtype=torch.float32)
    rc = load().neko_attention_fwd_path(_p(qkv), _p(first_valid), _p(out), _p(out2), _p(lse), C.c_int(B), C.c_int(S),
                                        C.c_int(S if S_valid is None else S_valid), C.c_int(H), C.c_int(d // H),
                                        C.c_int(int(out.dtype == torch.float16)), _dref(drop))
    if rc < 0:
        check(rc, "neko_attention_fwd_path")
    return ("mma", "tc")[rc]


def attention_decode(q: torch.Tensor, k_cache: torch.Tensor, v_cache: torch.Tensor, length: int, H: int, out: torch.Tensor):
    """One new query against `length` cached keys / values (bf16 [>=length, d])."""
    d = q.numel()
    check(load().neko_attention_decode(_p(q), _p(k_cache), _p(v_cache), C.c_int(length), C.c_int(H), C.c_int(d // H), _p(out),
                                       C.c_int(int(out.dtype == torch.float16)), stream_ptr()), "neko_attention_decode")
    return out


def attention_bwd(qkv, out, dout, lse, first_valid, H: int, S_valid: Optional[int] = None, dqkv=None, delta=None, drop=None):
    B, S, three_d = qkv.shape
    dh = three_d // 3 // H
    if dqkv is None:
        dqkv = torch.empty_like(qkv)
    if delta is None:
        delta = torch.empty(B, H, S, device=qkv.device, dtype=torch.float32)
    check(load().neko_attention_bwd(_p(qkv), _p(out), _p(dout), _p(lse), _p(first_valid), _p(dqkv), _p(delta), C.c_int(B),
                                    C.c_int(S), C.c_int(S if S_valid is None else S_valid), C.c_int(H), C.c_int(dh),
                                    C.c_int(int(out.dtype == torch.float16)), _dref(drop), stream_ptr()), "neko_attention_bwd")
    return dqkv


def attention_varlen_fwd(qkv: torch.Tensor, cu_seqlens: torch.Tensor, first_valid: torch.Tensor, H: int, S_max: int, S_width: int,
                         out=None, lse=None, out_dtype: torch.dtype = torch.bfloat16, out2=None, drop=None):
    """Packed causal attention: qkv [T, 3d], sample b = rows [cu_seqlens[b], cu_seqlens[b+1]); out [T, d], lse [H, T].
    S_width / first_valid give the padded layout's dropout coordinates (include/neko_b200.h)."""
    T, three_d = qkv.shape
    d = three_d // 3
    B = cu_seqlens.numel() - 1
    if out is None:
        out = torch.empty(T, d, device=qkv.device, dtype=out_dtype)
    if lse is None:
        lse = torch.empty(H, T, device=qkv.device, dtype=torch.float32)
    check(load().neko_attention_varlen_fwd(_p(qkv), _p(cu_seqlens), _p(first_valid), _p(out), _p(out2), _p(lse), C.c_int(B), C.c_int(T),
                                           C.c_int(S_max), C.c_int(S_width), C.c_int(H), C.c_int(d // H),
                                           C.c_int(int(out.dtype == torch.float16)), _dref(drop), stream_ptr()), "neko_attention_varlen_fwd")
    return out, lse


def attention_varlen_bwd(qkv, out, dout, lse, cu_seqlens, first_valid, H: int, S_max: int, S_width: int, dqkv=None, delta=None, drop=None):
    T, three_d = qkv.shape
    B = cu_seqlens.numel() - 1
    if dqkv is None:
        dqkv = torch.empty_like(qkv)
    if delta is None:
        delta = torch.empty(H, T, device=qkv.device, dtype=torch.float32)
    check(load().neko_attention_varlen_bwd(_p(qkv), _p(out), _p(dout), _p(lse), _p(cu_seqlens), _p(first_valid), _p(dqkv), _p(delta),
                                           C.c_int(B), C.c_int(T), C.c_int(S_max), C.c_int(S_width), C.c_int(H), C.c_int(three_d // 3 // H),
                                           C.c_int(int(out.dtype == torch.float16)), _dref(drop), stream_ptr()), "neko_attention_varlen_bwd")
    return dqkv


# ------------------------------------------------------------------------------------------
# masked cross entropy
# ------------------------------------------------------------------------------------------
CE_LOGITS_COMPACT, CE_DLOGITS_COMPACT, CE_ZERO_PAD = 1, 2, 4


def masked_ce_fwd(logits: torch.Tensor, V: int, rows: torch.Tensor, tokens: torch.Tensor, flags: int = 0):
    """logits fp32 [N, ld]; rows int32 [n]; tokens int64 flat [N]."""
    n = rows.numel()
    row_lse = torch.empty(n, device=logits.device, dtype=torch.float32)
    row_loss = torch.empty(n, device=logits.device, dtype=torch.float32)
    loss = torch.empty((), device=logits.device, dtype=torch.float32)
    check(load().neko_masked_ce_fwd(_p(logits), C.c_int64(logits.stride(-2)), C.c_int(V), _p(rows), C.c_int(n), _p(tokens),
                                    _p(row_lse), _p(row_loss), _p(loss), C.c_int(flags), stream_ptr()), "neko_masked_ce_fwd")
    return loss, row_lse, row_loss


def masked_ce_fused(logits: torch.Tensor, V: int, rows: torch.Tensor, tokens: torch.Tensor, dlogits: torch.Tensor, flags: int = 0):
    """Loss + unscaled gradient operand in one pass (training).  Returns (loss, row_lse) or None when not applicable."""
    n = rows.numel()
    row_lse = torch.empty(n, device=logits.device, dtype=torch.float32)
    row_loss = torch.empty(n, device=logits.device, dtype=torch.float32)
    loss = torch.empty((), device=logits.device, dtype=torch.float32)
    fn = load().neko_masked_ce_fused_f16 if logits.dtype == torch.float16 else load().neko_masked_ce_fused
    assert logits.dtype in (torch.float16, torch.float32)
    rc = fn(_p(logits), C.c_int64(logits.stride(-2)), C.c_int(V), _p(rows), C.c_int(n), _p(tokens), _p(row_lse),
            _p(row_loss), _p(loss), _p(dlogits), C.c_int64(dlogits.stride(-2)), C.c_int(flags), stream_ptr())
    if rc == 1:
        return None
    check(rc, "neko_masked_ce_fused")
    return loss, row_lse


def ce_scale_grad(dlogits: torch.Tensor, gscale: torch.Tensor):
    check(load().neko_ce_scale_grad(_p(dlogits), C.c_int64(dlogits.numel()), _p(gscale), stream_ptr()), "neko_ce_scale_grad")


def masked_ce_bwd(logits, V, rows, tokens, row_lse, gscale, dlogits, flags: int = 0):
    n = rows.numel()
    ld = dlogits.stride(-2)
    check(load().neko_masked_ce_bwd(_p(logits), C.c_int64(logits.stride(-2)), C.c_int(V), _p(rows), C.c_int(n), _p(tokens),
                                    _p(row_lse), _p(gscale), _p(dlogits), C.c_int64(ld), C.c_int(flags), stream_ptr()),
          "neko_masked_ce_bwd")


# ------------------------------------------------------------------------------------------
# helpers
# ------------------------------------------------------------------------------------------
def cast_bf16(src: torch.Tensor, dst: Optional[torch.Tensor] = None) -> torch.Tensor:
    _cuda(src)
    assert src.dtype == torch.float32 and src.is_contiguous()
    if dst is None:
        dst = torch.empty(src.shape, device=src.device, dtype=torch.bfloat16)
    fn = load().neko_cast_f32_to_f16 if dst.dtype == torch.float16 else load().neko_cast_f32_to_bf16
    check(fn(_p(src), _p(dst), C.c_int64(src.numel()), stream_ptr()), "neko_cast_f32_to_16")
    return dst


def cast_dual(src: torch.Tensor, dst_f16: torch.Tensor, dst_bf16: torch.Tensor):
    """fp32 -> (fp16, bf16) in one pass."""
    assert src.dtype == torch.float32 and dst_f16.dtype == torch.float16 and dst_bf16.dtype == torch.bfloat16
    check(load().neko_cast_f32_to_f16_bf16(_p(src), _p(dst_f16), _p(dst_bf16), C.c_int64(src.numel()), stream_ptr()),
          "neko_cast_f32_to_f16_bf16")


def colsum(x_bf16: torch.Tensor, out: torch.Tensor, accumulate: bool = False, M: Optional[int] = None, N: Optional[int] = None):
    M = x_bf16.shape[0] if M is None else M
    N = x_bf16.shape[1] if N is None else N
    check(load().neko_colsum_bf16(_p(x_bf16), C.c_int64(x_bf16.stride(0)), C.c_int(M), C.c_int(N), _p(out),
                                  C.c_int(int(accumulate)), stream_ptr()), "neko_colsum_bf16")
    return out


def gather_rows(src_bf16, rows, n: int, dst):
    check(load().neko_gather_rows_bf16(_p(src_bf16), C.c_int64(src_bf16.stride(0)), _p(rows), C.c_int(rows.numel()), C.c_int(n),
                                       _p(dst), C.c_int64(dst.stride(0)), stream_ptr()), "neko_gather_rows_bf16")
    return dst


def scatter_rows(src_bf16, rows, n: int, dst):
    check(load().neko_scatter_rows_bf16(_p(src_bf16), C.c_int64(src_bf16.stride(0)), _p(rows), C.c_int(rows.numel()), C.c_int(n),
                                        _p(dst), C.c_int64(dst.stride(0)), stream_ptr()), "neko_scatter_rows_bf16")
    return dst


def scatter_rows_add(src_bf16, rows, n: int, dst_f32):
    check(load().neko_scatter_rows_add_f32(_p(src_bf16), C.c_int64(src_bf16.stride(0)), _p(rows), C.c_int(rows.numel()),
                                           C.c_int(n), _p(dst_f32), C.c_int64(dst_f32.stride(0)), stream_ptr()),
          "neko_scatter_rows_add_f32")
    return dst_f32


def sumsq(x: torch.Tensor, out: torch.Tensor):
    check(load().neko_sumsq_f32(_p(x), C.c_int64(x.numel()), _p(out), stream_ptr()), "neko_sumsq_f32")
    return out


def adamw_step(param, grad, exp_avg, exp_avg_sq, lr, beta1, beta2, eps, weight_decay, step, grad_sumsq=None, max_norm=0.0,
               grad_div=1.0, w_f16=None, w_bf16=None, n_cast=0):
    check(load().neko_adamw_step(_p(param), _p(grad), _p(exp_avg), _p(exp_avg_sq), C.c_int64(param.numel()), C.c_float(lr),
                                 C.c_float(beta1), C.c_float(beta2), C.c_float(eps), C.c_float(weight_decay), C.c_int(step),
                                 _p(grad_sumsq), C.c_float(max_norm), C.c_float(grad_div), _p(w_f16), _p(w_bf16), C.c_int64(n_cast),
                                 stream_ptr()), "neko_adamw_step")


# ------------------------------------------------------------------------------------------
# ordered reductions (deterministic training mode): same results as their default twins up to reassociation, with every sum in
# a fixed order.  `ws` is a device tensor of at least the matching *_workspace_bytes() bytes.
# ------------------------------------------------------------------------------------------
def _ws_bytes(rc: int, what: str) -> int:
    if rc < 0:
        check(int(rc), what)
    return int(rc)


def layernorm_bwd_ordered_workspace_bytes(N: int, d: int) -> int:
    return _ws_bytes(load().neko_layernorm_bwd_ordered_workspace_bytes(C.c_int(N), C.c_int(d)), "neko_layernorm_bwd_ordered_workspace_bytes")


def layernorm_bwd_ordered(dy_bf16, x, gamma, mean, rstd, dx_resid, dgamma, dbeta, ws, dx_bf16=None, dx_colsum=None, branch_drop=None):
    N, d = x.shape
    check(load().neko_layernorm_bwd_ordered(_p(dy_bf16), _p(x), _p(gamma), _p(mean), _p(rstd), _p(dx_resid), _p(dx_bf16), _p(dgamma),
                                            _p(dbeta), _p(dx_colsum), C.c_int(N), C.c_int(d), _dref(branch_drop), _p(ws),
                                            C.c_int64(ws.numel() * ws.element_size()), stream_ptr()), "neko_layernorm_bwd_ordered")


def colsum_ordered_workspace_bytes(M: int, N: int) -> int:
    return _ws_bytes(load().neko_colsum_bf16_ordered_workspace_bytes(C.c_int(M), C.c_int(N)), "neko_colsum_bf16_ordered_workspace_bytes")


def colsum_ordered(x_bf16: torch.Tensor, out: torch.Tensor, ws: torch.Tensor, accumulate: bool = False):
    M, N = x_bf16.shape
    check(load().neko_colsum_bf16_ordered(_p(x_bf16), C.c_int64(x_bf16.stride(0)), C.c_int(M), C.c_int(N), _p(out),
                                          C.c_int(int(accumulate)), _p(ws), C.c_int64(ws.numel() * ws.element_size()), stream_ptr()),
          "neko_colsum_bf16_ordered")
    return out


def embed_bwd_ordered_workspace_bytes(B: int, prm: TokParams) -> int:
    return _ws_bytes(load().neko_embed_bwd_ordered_workspace_bytes(C.c_int(B), C.byref(prm)), "neko_embed_bwd_ordered_workspace_bytes")


def embed_bwd_ordered(descs, B: int, d: int, prm: TokParams, tokens, d_emb, d_embed_table, d_pos_table, d_sep, ws, d_patch_emb=None,
                      packed: bool = False):
    fn = load().neko_embed_packed_bwd_ordered if packed else load().neko_embed_bwd_ordered
    check(fn(_p(descs), C.c_int(B), C.c_int(d), C.byref(prm), _p(tokens), _p(d_emb), _p(d_embed_table), _p(d_pos_table), _p(d_sep),
             _p(d_patch_emb), _p(ws), C.c_int64(ws.numel() * ws.element_size()), stream_ptr()),
          "neko_embed_packed_bwd_ordered" if packed else "neko_embed_bwd_ordered")


def patch_resblock_bwd_ordered_workspace_bytes(n_img: int, height: int, width: int, patch: int) -> int:
    return _ws_bytes(load().neko_patch_resblock_bwd_ordered_workspace_bytes(C.c_int(n_img), C.c_int(height), C.c_int(width), C.c_int(patch)),
                     "neko_patch_resblock_bwd_ordered_workspace_bytes")


def patch_resblock_bwd_ordered(images, is_u8: bool, n_img: int, height: int, width: int, patch: int, C_mid: int, groups: int, conv1_w,
                               conv1_b, gn_w, gn_b, conv2_w, gn_stats, d_patches_bf16, d_conv1_w, d_conv1_b, d_gn_w, d_gn_b, d_conv2_w,
                               d_conv2_b, ws):
    check(load().neko_patch_resblock_bwd_ordered(_p(images), C.c_int(int(is_u8)), C.c_int(n_img), C.c_int(height), C.c_int(width),
                                                 C.c_int(patch), C.c_int(C_mid), C.c_int(groups), _p(conv1_w), _p(conv1_b), _p(gn_w),
                                                 _p(gn_b), _p(conv2_w), _p(gn_stats), _p(d_patches_bf16), _p(d_conv1_w), _p(d_conv1_b),
                                                 _p(d_gn_w), _p(d_gn_b), _p(d_conv2_w), _p(d_conv2_b), _p(ws),
                                                 C.c_int64(ws.numel() * ws.element_size()), stream_ptr()),
          "neko_patch_resblock_bwd_ordered")


def patch_pos_bwd_ordered_workspace_bytes(P: int, n_row_bins: int, n_col_bins: int) -> int:
    return _ws_bytes(load().neko_patch_pos_bwd_ordered_workspace_bytes(C.c_int(P), C.c_int(n_row_bins), C.c_int(n_col_bins)),
                     "neko_patch_pos_bwd_ordered_workspace_bytes")


def patch_pos_bwd_ordered(dx, row_bin, col_bin, d_row_tab, d_col_tab, ws):
    P, d = dx.shape
    check(load().neko_patch_pos_bwd_ordered(_p(dx), C.c_int(P), C.c_int(d), _p(row_bin), _p(col_bin), _p(d_row_tab),
                                            C.c_int(d_row_tab.shape[0]), _p(d_col_tab), C.c_int(d_col_tab.shape[0]), _p(ws),
                                            C.c_int64(ws.numel() * ws.element_size()), stream_ptr()), "neko_patch_pos_bwd_ordered")


def sumsq_ordered_workspace_bytes(n: int) -> int:
    return _ws_bytes(load().neko_sumsq_f32_ordered_workspace_bytes(C.c_int64(n)), "neko_sumsq_f32_ordered_workspace_bytes")


def sumsq_ordered(x: torch.Tensor, out: torch.Tensor, ws: torch.Tensor):
    check(load().neko_sumsq_f32_ordered(_p(x), C.c_int64(x.numel()), _p(out), _p(ws), C.c_int64(ws.numel() * ws.element_size()),
                                        stream_ptr()), "neko_sumsq_f32_ordered")
    return out

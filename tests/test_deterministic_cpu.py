"""Deterministic training mode, host side: argument checks of the ordered entry points (each returns NEKO_EINVAL before any
CUDA call, so fake device pointers are never dereferenced), their workspace-size queries, the --deterministic flag, the
CUDA-graph key and the data-parallel backends the mode refuses.  CPU only."""
import ctypes as C
import types

import pytest

NEKO_EINVAL = -1
F = 0x100000          # a fake 256-byte aligned device address
MIS = F + 2           # a fake misaligned one


@pytest.fixture(scope="module")
def lib():
    from neko_b200 import _lib, build
    build.build()
    return _lib.load()


def _p(x):
    return C.c_void_p(x)


def _i(v):
    return C.c_int(v)


def _l(v):
    return C.c_int64(v)


# ---- LayerNorm ---------------------------------------------------------------------------------------------------------------
def _ln_args(dy=F, x=F, gamma=F, dx=F, dxb=0, ws=F, N=256, d=768, ws_bytes=1 << 30):
    return (_p(dy), _p(x), _p(gamma), _p(F), _p(F), _p(dx), _p(dxb), _p(F), _p(F), _p(0), _i(N), _i(d), None, _p(ws), _l(ws_bytes), None)


LN_BAD = {"d6": dict(d=6), "d2052": dict(d=2052), "N0": dict(N=0), "null_x": dict(x=0), "null_ws": dict(ws=0),
          "small_ws": dict(ws_bytes=4 * 3 * 768 * 4 - 1), "x_misaligned": dict(x=F + 4), "dy_misaligned": dict(dy=F + 4),
          "dxb_misaligned": dict(dxb=MIS), "gamma_misaligned": dict(gamma=F + 8)}


@pytest.mark.parametrize("case", sorted(LN_BAD))
def test_layernorm_bwd_ordered_rejects(lib, case):
    assert lib.neko_layernorm_bwd_ordered(*_ln_args(**LN_BAD[case])) == NEKO_EINVAL


def test_layernorm_bwd_ordered_workspace(lib):
    # fixed 64-row blocks, three d-wide partial rows each
    assert lib.neko_layernorm_bwd_ordered_workspace_bytes(_i(7680), _i(768)) == 120 * 3 * 768 * 4
    assert lib.neko_layernorm_bwd_ordered_workspace_bytes(_i(65), _i(4)) == 2 * 3 * 4 * 4
    for N, d in ((0, 768), (10, 6), (10, 2052), (-1, 8)):
        assert lib.neko_layernorm_bwd_ordered_workspace_bytes(_i(N), _i(d)) == NEKO_EINVAL


# ---- column sums -----------------------------------------------------------------------------------------------------------
def _cs_args(X=F, ld=768, M=100, N=768, out=F, ws=F, ws_bytes=1 << 30):
    return (_p(X), _l(ld), _i(M), _i(N), _p(out), _i(1), _p(ws), _l(ws_bytes), None)


CS_BAD = {"M0": dict(M=0), "N0": dict(N=0), "ld_lt_N": dict(ld=700), "odd_ld": dict(ld=769), "X_misaligned": dict(X=MIS),
          "null_out": dict(out=0), "null_ws": dict(ws=0), "small_ws": dict(ws_bytes=2 * 768 * 4 - 4)}


@pytest.mark.parametrize("case", sorted(CS_BAD))
def test_colsum_ordered_rejects(lib, case):
    assert lib.neko_colsum_bf16_ordered(*_cs_args(**CS_BAD[case])) == NEKO_EINVAL


def test_colsum_ordered_workspace(lib):
    assert lib.neko_colsum_bf16_ordered_workspace_bytes(_i(7680), _i(2304)) == 120 * 2304 * 4
    assert lib.neko_colsum_bf16_ordered_workspace_bytes(_i(1), _i(3)) == 12
    assert lib.neko_colsum_bf16_ordered_workspace_bytes(_i(0), _i(3)) == NEKO_EINVAL


# ---- sum of squares --------------------------------------------------------------------------------------------------------
def test_sumsq_ordered_rejects_and_workspace(lib):
    f = lib.neko_sumsq_f32_ordered
    assert f(_p(0), _l(10), _p(F), _p(F), _l(1 << 20), None) == NEKO_EINVAL
    assert f(_p(F), _l(-1), _p(F), _p(F), _l(1 << 20), None) == NEKO_EINVAL
    assert f(_p(F), _l(10), _p(F), _p(0), _l(1 << 20), None) == NEKO_EINVAL
    assert f(_p(F), _l(8193), _p(F), _p(F), _l(4), None) == NEKO_EINVAL           # two 8192-element blocks need 8 bytes
    assert f(_p(F + 4), _l(10), _p(F), _p(F), _l(1 << 20), None) == NEKO_EINVAL
    assert f(_p(F), _l(0), _p(F), _p(0), _l(0), None) == 0                        # nothing to do, nothing launched
    assert lib.neko_sumsq_f32_ordered_workspace_bytes(_l(8193)) == 8
    assert lib.neko_sumsq_f32_ordered_workspace_bytes(_l(0)) == 0
    assert lib.neko_sumsq_f32_ordered_workspace_bytes(_l(-5)) == NEKO_EINVAL


# ---- patch backward ------------------------------------------------------------------------------------------------------
def _pr_args(n_img=2, H=64, W=64, patch=16, Cm=128, groups=32, ws=F, ws_bytes=1 << 30, dw1=F):
    return ((_p(F), _i(0), _i(n_img), _i(H), _i(W), _i(patch), _i(Cm), _i(groups)) + tuple(_p(F) for _ in range(7)) +
            (_p(dw1),) + tuple(_p(F) for _ in range(5)) + (_p(ws), _l(ws_bytes), None))


PR_BAD = {"patch8": dict(patch=8), "C64": dict(Cm=64), "groups3": dict(groups=3), "H_not_multiple": dict(H=60), "n_img0": dict(n_img=0),
          "null_dw1": dict(dw1=0), "null_ws": dict(ws=0), "small_ws": dict(ws_bytes=4 * 7299 * 4 - 4)}


@pytest.mark.parametrize("case", sorted(PR_BAD))
def test_patch_resblock_bwd_ordered_rejects(lib, case):
    assert lib.neko_patch_resblock_bwd_ordered(*_pr_args(**PR_BAD[case])) == NEKO_EINVAL


def test_patch_resblock_bwd_ordered_workspace(lib):
    # fixed chunks of 8 patches, one 7299-float slot each (dw1 3456 | db1 128 | dgamma 128 | dbeta 128 | dw2 3456 | db2 3)
    assert lib.neko_patch_resblock_bwd_ordered_workspace_bytes(_i(2), _i(64), _i(64), _i(16)) == 4 * 7299 * 4
    assert lib.neko_patch_resblock_bwd_ordered_workspace_bytes(_i(1), _i(48), _i(16), _i(16)) == 1 * 7299 * 4
    assert lib.neko_patch_resblock_bwd_ordered_workspace_bytes(_i(1), _i(48), _i(16), _i(8)) == NEKO_EINVAL


def _pp_args(dx=F, P=100, d=768, nr=16, nc=16, ws=F, tab=F):
    return (_p(dx), _i(P), _i(d), _p(F), _p(F), _p(tab), _i(nr), _p(F), _i(nc), _p(ws), _l(1 << 30), None)


PP_BAD = {"P0": dict(P=0), "d6": dict(d=6), "nr0": dict(nr=0), "nc0": dict(nc=0), "dx_misaligned": dict(dx=F + 4),
          "tab_misaligned": dict(tab=F + 4), "ws_misaligned": dict(ws=F + 16), "null_ws": dict(ws=0)}


@pytest.mark.parametrize("case", sorted(PP_BAD))
def test_patch_pos_bwd_ordered_rejects(lib, case):
    assert lib.neko_patch_pos_bwd_ordered(*_pp_args(**PP_BAD[case])) == NEKO_EINVAL
    if case in ("P0", "nr0", "nc0"):
        kw = PP_BAD[case]
        assert lib.neko_patch_pos_bwd_ordered_workspace_bytes(_i(kw.get("P", 100)), _i(kw.get("nr", 16)), _i(kw.get("nc", 16))) == NEKO_EINVAL


# ---- embedding backward ----------------------------------------------------------------------------------------------------
def _tok(**kw):
    from neko_b200._lib import TokParams
    base = dict(mu=100.0, M=256.0, n_bins=1024, cont_start=50257, disc_start=51281, vocab=52305, use_pos=1, seq_len=240, width=240,
                ctx_rows=240)
    base.update(kw)
    return TokParams(**base)


def _emb_args(prm, B=4, d=768, d_emb=F, table=F, pos=F, ws=F):
    return (_p(F), _i(B), _i(d), C.byref(prm), _p(F), _p(d_emb), _p(table), _p(pos), _p(F), _p(0), _p(ws), _l(1 << 30), None)


EMB_BAD = {"B0": (dict(B=0), {}), "d6": (dict(d=6), {}), "width_lt_seq": ({}, dict(width=100)), "vocab0": ({}, dict(vocab=0)),
           "null_pos": (dict(pos=0), {}), "null_ws": (dict(ws=0), {}), "ws_misaligned": (dict(ws=F + 16), {}),
           "emb_misaligned": (dict(d_emb=F + 4), {}), "table_misaligned": (dict(table=F + 8), {})}


@pytest.mark.parametrize("case", sorted(EMB_BAD))
@pytest.mark.parametrize("packed", [False, True])
def test_embed_bwd_ordered_rejects(lib, case, packed):
    a, t = EMB_BAD[case]
    fn = lib.neko_embed_packed_bwd_ordered if packed else lib.neko_embed_bwd_ordered
    assert fn(*_emb_args(_tok(**t), **a)) == NEKO_EINVAL
    if case in ("B0", "width_lt_seq", "vocab0"):
        assert lib.neko_embed_bwd_ordered_workspace_bytes(_i(a.get("B", 4)), C.byref(_tok(**t))) == NEKO_EINVAL


def test_ordered_workspace_queries_through_ops():
    """The ops wrappers turn a rejected query into NekoError and pass sizes through."""
    from neko_b200 import ops
    from neko_b200._lib import NekoError
    assert ops.layernorm_bwd_ordered_workspace_bytes(128, 768) == 2 * 3 * 768 * 4
    assert ops.colsum_ordered_workspace_bytes(64, 10) == 40
    assert ops.sumsq_ordered_workspace_bytes(1) == 4
    assert ops.patch_resblock_bwd_ordered_workspace_bytes(1, 16, 16, 16) == 7299 * 4
    with pytest.raises(NekoError):
        ops.layernorm_bwd_ordered_workspace_bytes(128, 770)


# ---- GEMM flag -------------------------------------------------------------------------------------------------------------
def test_gemm_deterministic_flag_value():
    from neko_b200 import ops
    from neko_b200._lib import HEADER
    txt = open(HEADER).read()
    assert "#define NEKO_GEMM_DETERMINISTIC 32" in txt and ops.GEMM_DETERMINISTIC == 32


# ---- host plumbing ---------------------------------------------------------------------------------------------------------
def test_deterministic_flag_parsing():
    from neko_b200.training import parse_args
    assert parse_args([]).deterministic is False
    assert parse_args(["--deterministic"]).deterministic is True
    assert parse_args(["--deterministic=false"]).deterministic is False
    assert parse_args(["--deterministic", "1"]).deterministic is True


def test_graph_key_includes_the_knob():
    """Two policies that differ only in the knob must not share a captured graph."""
    import numpy as np
    from neko_b200.policy.gato_policy import GatoPolicy
    plan = types.SimpleNamespace(B=2, seq_len=8, width=8, descs=np.zeros(4, np.int32), image_groups=[], precomputed_patch=[], packed=False)
    st = types.SimpleNamespace(plan=plan, compute_loss=True, need_grad=True, row_bins=None)
    fake = types.SimpleNamespace(training=True, materialize_logits=False, head_mode="rows", fwd_dtype=None, lean_logits_f16=True,
                                 mlp_proj_bf16=False, _dropout_ps=lambda: (0.1,), deterministic=False)
    k0 = GatoPolicy._graph_key(fake, st)
    fake.deterministic = True
    k1 = GatoPolicy._graph_key(fake, st)
    assert k0 != k1 and sum(x != y for x, y in zip(k0, k1)) == 1


def test_nccl_is_refused_in_deterministic_mode(monkeypatch):
    import torch
    from neko_b200 import dp
    arena = torch.zeros(1000)
    s = dp.GradSynchronizer(arena, bucket_bytes=4 * 100)
    assert s.backend == "nccl"
    s.require_deterministic()              # a single rank exchanges nothing: nothing to refuse
    s.world = 2
    with pytest.raises(ValueError, match="NCCL"):
        s.require_deterministic()
    s.backend = "p2p"
    s.require_deterministic()
    monkeypatch.setenv("NEKO_DP_NCCL_TAIL", "1")
    s2 = dp.GradSynchronizer(arena, bucket_bytes=4 * 100)
    s2.world, s2.backend = 2, "p2p"
    with pytest.raises(ValueError, match="NEKO_DP_NCCL_TAIL"):
        s2.require_deterministic()
    # attach() checks the policy's knob before wiring anything
    pol = types.SimpleNamespace(_grad_arena=arena, deterministic=True, _offs={}, text_tokens=0, embed_dim=0, _params={})
    monkeypatch.setattr(dp.GradSynchronizer, "__init__", lambda self, *a, **k: (setattr(self, "world", 2), setattr(self, "backend", "nccl"),
                                                                                 setattr(self, "nccl_tail", False))[0])
    with pytest.raises(ValueError, match="NCCL"):
        dp.attach(pol)

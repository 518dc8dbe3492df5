"""Padding-free (packed) training steps: GatoPolicy.pack_sequences against the padded layout and the CPU oracle, the packed
tokenise / embed kernels against the padded ones, and the variable-length attention kernels against an fp32 reference.
GPU only (-m gpu)."""
import copy
import math
import os

import numpy as np
import pytest
import torch

from oracle import gato_oracle as O
from oracle.make_golden import SMALL_CASES, scale_batch, small_batch
from test_policy_gpu import LOSS_RTOL, _grad_report, make_policy

pytestmark = pytest.mark.gpu


def _valid_rows(plan):
    """Flat padded positions b*W + first_valid[b] + p of every valid token, in packed row order."""
    L = np.diff(plan.cu_seqlens)
    return np.concatenate([b * plan.width + plan.first_valid[b] + np.arange(L[b]) for b in range(plan.B)])


def _packed_state(m, batch):
    m.pack_sequences, m.materialize_logits = True, False
    st = m._plan(batch, True)
    assert st.plan.packed
    st.need_grad = False
    m._embed(st)
    return st


def _padded_state(m, batch):
    st = m._plan(batch, False)
    assert not st.plan.packed
    st.need_grad = False
    m._embed(st)
    return st


def _tok_cases():
    from _random_batches import random_mixed_batch
    out = [(n, O.synth_batch(n), O.CONFIGS[n]["context_len"], False) for n in ("cfg1", "cfg2", "cfg3", "cfg4", "cfg5")]
    out += [(f"random{s}",) + random_mixed_batch(s) for s in range(8)]
    return out


@pytest.mark.parametrize("case", range(13))
def test_tokenize_and_embed_bwd_packed_bit_exact(case):
    from neko_b200 import ops
    name, batch, ctx, pad_seq = _tok_cases()[case]
    cfg = O.GatoConfig(embed_dim=32, layers=1, heads=1, context_len=ctx, text_tokens=300 if name.startswith("random") else 50257,
                       pad_seq=pad_seq)
    m = make_policy(cfg, O.make_weights(cfg, seed=case) if name.startswith("random") else None)
    d = cfg.embed_dim
    g = torch.Generator(device="cuda").manual_seed(case)

    def embed_grads(st, dx):
        # small multiples of 1/16: every fp32 sum is exact whatever order the atomics take
        gr = [torch.zeros_like(m.embed_token.weight), torch.zeros_like(m.pos_embed_observation.weight), torch.zeros(d, device="cuda")]
        dpe = torch.zeros(max(st.plan.n_patch_rows, 1), d, device="cuda")
        ops.embed_bwd(st.descs, st.plan.B, d, st.tok_params, st.tokens, dx, gr[0], gr[1], gr[2], dpe, packed=st.plan.packed)
        return gr + [dpe]

    pk = _packed_state(m, batch)
    T = pk.plan.token_rows
    out_pk = [t[:T].clone() for t in (pk.tokens, pk.tmask, pk.mask)] + [pk.x0[:T].clone()]
    dx_pk = torch.randint(-8, 9, (T, d), device="cuda", generator=g).float() / 16
    g_pk = embed_grads(pk, dx_pk)
    pd = _padded_state(m, batch)
    rows = torch.from_numpy(_valid_rows(pd.plan)).cuda()
    N = pd.plan.token_rows
    assert T == pd.plan.n_valid_tokens == rows.numel()
    for a, b in zip(out_pk, (pd.tokens[:N], pd.tmask[:N], pd.mask[:N], pd.x0[:N])):
        assert torch.equal(a, b[rows])
    assert bool((out_pk[2] == 1).all())
    dx_pd = torch.zeros(N, d, device="cuda")
    dx_pd[rows] = dx_pk
    for a, b in zip(g_pk, embed_grads(pd, dx_pd)):
        assert torch.equal(a, b)


# ---------------------------------------------------------------------------------------------------
# variable-length attention
# ---------------------------------------------------------------------------------------------------
def _rand(shape, seed, scale, dtype):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return (torch.randn(shape, device="cuda", generator=g) * scale).to(dtype)


def _seed(a, b):
    return torch.tensor([a, b], dtype=torch.int32, device="cuda")


def _varlen_ref(x, lengths, H, mult=None, fv=None):
    """fp32 causal attention of every sample on its own rows of x [T, 3d]; mult: padded-layout multipliers [B, H, W, W]."""
    d = x.shape[1] // 3
    dh = d // H
    outs, r0 = [], 0
    for b, L in enumerate(lengths):
        q, k, v = (t.view(L, H, dh).transpose(0, 1) for t in x[r0:r0 + L].split(d, dim=1))
        sc = (q @ k.transpose(-1, -2)) / math.sqrt(dh)
        idx = torch.arange(L, device=x.device)
        sc = sc.masked_fill(~(idx[None, :] <= idx[:, None])[None], float("-inf"))
        p = torch.softmax(sc, -1)
        if mult is not None:
            o = int(fv[b])
            p = p * mult[b, :, o:o + L, o:o + L]
        outs.append((p @ v).transpose(0, 1).reshape(L, d))
        r0 += L
    return torch.cat(outs)


LENGTHS = [[1, 63, 64, 65, 1024], [5, 1, 63, 17, 64, 65, 2, 130]]


@pytest.mark.parametrize("lengths", LENGTHS)
@pytest.mark.parametrize("H,dh", [(4, 32), (2, 64), (1, 128)])
def test_attention_varlen_fwd_bwd(H, dh, lengths):
    from neko_b200 import ops
    d, B, T, S = H * dh, len(lengths), sum(lengths), max(lengths)
    cu = torch.tensor([0] + list(np.cumsum(lengths)), dtype=torch.int32, device="cuda")
    fv = torch.tensor([S - L for L in lengths], dtype=torch.int32, device="cuda")
    qkv = _rand((T, 3 * d), 21, 1.0, torch.bfloat16)
    out, lse = ops.attention_varlen_fwd(qkv, cu, fv, H, S, S)
    assert tuple(lse.shape) == (H, T)
    x = qkv.float().requires_grad_(True)
    ref = _varlen_ref(x, lengths, H)
    assert (out.float() - ref).abs().max().item() < 0.03
    dout = _rand((T, d), 22, 1.0, torch.bfloat16)
    (ref * dout.float()).sum().backward()
    dqkv = ops.attention_varlen_bwd(qkv, out, dout, lse, cu, fv, H, S, S)
    scale = x.grad.abs().max().item()
    assert (dqkv.float() - x.grad).abs().max().item() < 0.03 * max(scale, 1.0)
    # fp16 output + bf16 twin: same statistics, same bf16 values
    o2 = torch.empty_like(out)
    out16, lse16 = ops.attention_varlen_fwd(qkv, cu, fv, H, S, S, out_dtype=torch.float16, out2=o2)
    assert torch.equal(lse16, lse) and torch.equal(o2, out) and (out16.float() - ref).abs().max().item() < 0.03


@pytest.mark.parametrize("H,dh", [(3, 32), (2, 64), (1, 128)])
def test_attention_varlen_dropout_matches_padded_layout(H, dh):
    """Same seed, same inputs laid out padded (left padding to S, right padding to the width W > S): the varlen kernels use
    the padded kernels' multipliers, so both agree with one reference built from the padded-layout mask."""
    from neko_b200 import ops
    from neko_b200._lib import Dropout
    lengths = [37, 1, 64, 130, 66]          # odd and even first_valid offsets
    d, B, T, S, W = H * dh, len(lengths), sum(lengths), max(lengths), max(lengths) + 9
    cu = torch.tensor([0] + list(np.cumsum(lengths)), dtype=torch.int32, device="cuda")
    fv = torch.tensor([S - L for L in lengths], dtype=torch.int32, device="cuda")
    dr = Dropout.make(_seed(31, 32), 5, 0.2)
    qkv = _rand((T, 3 * d), 11, 0.7, torch.bfloat16)
    pad_rows = torch.from_numpy(np.concatenate([b * W + S - L + np.arange(L) for b, L in enumerate(lengths)])).cuda()
    qkv_pad = torch.zeros(B * W, 3 * d, dtype=torch.bfloat16, device="cuda")
    qkv_pad[pad_rows] = qkv
    out_pad, lse_pad = ops.attention_fwd(qkv_pad.view(B, W, 3 * d), fv, H, S, drop=dr)
    out, lse = ops.attention_varlen_fwd(qkv, cu, fv, H, S, W, drop=dr)
    mult = (ops.dropout_mask(B * H * W, W, dr, "cuda").float() * dr.scale).view(B, H, W, W)
    x = qkv.float().requires_grad_(True)
    ref = _varlen_ref(x, lengths, H, mult, fv.tolist())
    assert (out.float() - ref).abs().max().item() < 3e-2
    assert (out_pad.view(B * W, d)[pad_rows].float() - ref).abs().max().item() < 3e-2
    assert (out.float() - out_pad.view(B * W, d)[pad_rows].float()).abs().max().item() < 3e-2
    dout = _rand((T, d), 12, 1.0, torch.bfloat16)
    ref.backward(dout.float())
    dqkv = ops.attention_varlen_bwd(qkv, out, dout, lse, cu, fv, H, S, W, drop=dr)
    dout_pad = torch.zeros(B * W, d, dtype=torch.bfloat16, device="cuda")
    dout_pad[pad_rows] = dout
    dqkv_pad = ops.attention_bwd(qkv_pad.view(B, W, 3 * d), out_pad, dout_pad.view(B, W, d), lse_pad, fv, H, S, drop=dr)
    gref = x.grad
    assert ((dqkv.float() - gref).norm() / gref.norm()).item() < 3e-2
    assert ((dqkv_pad.view(B * W, 3 * d)[pad_rows].float() - gref).norm() / gref.norm()).item() < 3e-2


# ---------------------------------------------------------------------------------------------------
# policy steps
# ---------------------------------------------------------------------------------------------------
def _step(m, batch, packed):
    m.materialize_logits = False
    m.pack_sequences = packed
    m.zero_grad()
    torch.manual_seed(77)
    _, loss = m(batch, compute_loss=True)
    loss.backward()
    torch.cuda.synchronize()
    return loss.item(), {n: (None if p.grad is None else p.grad.detach().clone()) for n, p in m.named_parameters()}


def _agree(lp, gp, lq, gq, loss_rtol=1e-4, grad_rtol=2e-2):
    assert abs(lp - lq) <= loss_rtol * abs(lq), (lp, lq)
    for n, a in gq.items():
        b = gp[n]
        assert (a is None) == (b is None), n
        if a is not None:
            assert (a - b).norm().item() <= grad_rtol * a.norm().item() + 1e-7, n


def _oracle_gates(m, w, lp, ref):
    assert abs(lp - ref.loss.item()) <= LOSS_RTOL * abs(ref.loss.item())
    rep = _grad_report(m, w)
    for n, p in m.named_parameters():
        if w[n].grad is None:
            assert p.grad is None, n
    bad = {n: v for n, v in rep.items() if v[2] > 1e-6 and v[0] < 0.99}
    assert not bad, f"gradient mismatch (cos, rel, ref-norm): {bad}"
    tight = [v for n, v in rep.items() if n.endswith("c_fc.weight") or n.endswith("c_attn.weight") or n == "predict_token.weight"]
    assert min(v[0] for v in tight) > 0.999


@pytest.mark.parametrize("case", ["mixed", "dh128", "geglu_padseq"])
def test_packed_step_matches_padded_and_oracle(case):
    cfg = O.GatoConfig(**SMALL_CASES[case]["cfg"])
    w = O.make_weights(cfg, seed=3)
    m = make_policy(cfg, w)
    batch = small_batch(case, cfg.text_tokens)
    lq, gq = _step(m, batch, False)
    lp, gp = _step(m, batch, True)
    _agree(lp, gp, lq, gq)
    for t in w.values():
        t.requires_grad_(True)
    torch.manual_seed(77)
    ref = O.forward(w, batch, cfg, compute_loss=True, training=False)
    ref.loss.backward()
    _oracle_gates(m, w, lp, ref)


def test_packed_step_model_scale_cfg5(golden_dir):
    """The reduced cfg5 batch of the golden fixtures (text, caption, VQA, MuJoCo, Atari; 40% padding) at model scale."""
    g = np.load(os.path.join(golden_dir, "scale_cfg5_eval.npz"))
    cfg = O.GatoConfig(**O.CONFIGS["cfg5"])
    m = make_policy(cfg, O.make_weights(cfg, seed=0, perturb=False))
    batch = scale_batch("cfg5")
    lq, gq = _step(m, batch, False)
    lp, gp = _step(m, batch, True)
    plan = m._last_drop[1]
    assert plan.packed and plan.token_rows < plan.B * plan.width
    _agree(lp, gp, lq, gq)
    assert abs(lp - float(g["loss"])) <= LOSS_RTOL * abs(float(g["loss"]))   # the reference's own loss


def test_packed_dropout_step_matches_oracle_replay():
    cfg = O.GatoConfig(**SMALL_CASES["mixed"]["cfg"])
    w = O.make_weights(cfg, seed=3)
    m = make_policy(cfg, w, train=True)
    m.transformer.drop.p = 0.1
    for blk in m.transformer.h:
        blk.attn.attn_dropout.p = 0.2
        blk.attn.resid_dropout.p = 0.15
        blk.mlp.dropout.p = 0.15
    m.materialize_logits, m.pack_sequences = False, True
    batch = small_batch("mixed", cfg.text_tokens)
    torch.manual_seed(77)
    _, loss = m(batch, compute_loss=True)
    loss.backward()
    torch.cuda.synchronize()
    drop = {k: v.cpu() for k, v in m.dropout_multipliers().items()}
    assert len(drop) == 1 + 3 * cfg.layers
    plan = m._last_drop[1]
    B, W = plan.B, plan.width
    valid = torch.zeros(B * W, dtype=torch.bool)
    valid[torch.from_numpy(_valid_rows(plan))] = True
    valid = valid.view(B, W)
    assert tuple(drop["embd"].shape) == (B, W, cfg.embed_dim) and tuple(drop[("attn", 0)].shape) == (B, cfg.heads, W, W)
    assert float(drop["embd"][~valid].abs().max()) == 0.0
    keep_rate = float((drop["embd"][valid] > 0).float().mean())
    assert abs(keep_rate - 0.9) < 0.02, keep_rate
    for t in w.values():
        t.requires_grad_(True)
    torch.manual_seed(77)
    ref = O.forward(w, batch, cfg, compute_loss=True, training=True, drop=drop)
    ref.loss.backward()
    _oracle_gates(m, w, loss.item(), ref)


def test_packed_cuda_graphs_and_stage():
    cfg = O.GatoConfig(**SMALL_CASES["mixed"]["cfg"])
    w = O.make_weights(cfg, seed=3)
    eager, graph = make_policy(cfg, w), make_policy(cfg, w)
    for m in (eager, graph):
        m.materialize_logits, m.pack_sequences = False, True
    graph.use_cuda_graphs = True
    A = small_batch("mixed", cfg.text_tokens)
    Bb = A[1:] + [dict(text=list(range(1, 30)))]
    for k in range(4):      # eager, capture, replay, replay
        le, ge = _step(eager, A, True)
        lg, gg = _step(graph, A, True)
        assert le == lg, k
        for n, a in ge.items():
            assert (a is None) == (gg[n] is None), n
            if a is not None:
                assert (a - gg[n]).abs().max().item() <= 1e-5 * (a.abs().max().item() + 1e-12) + 1e-9, (k, n)
    for _ in range(3):      # two batch compositions alternate: two graph keys, both packed
        _step(graph, Bb, True)
        lg, _ = _step(graph, A, True)
        assert lg == le
    assert sum(1 for key, e in graph._graphs.items() if key[-1] and "fwd" in e) == 2
    # a staged packed batch gives the same step as a direct one
    for m in (eager, graph):
        l0, g0 = _step(m, A, True)
        for _ in range(2):
            h = m.stage(A, compute_loss=True)
            m.zero_grad()
            _, loss = m(h, compute_loss=True)
            loss.backward()
            assert loss.item() == l0
            for n, p in m.named_parameters():
                assert (p.grad is None) == (g0[n] is None), n
                if p.grad is not None:
                    assert (p.grad - g0[n]).abs().max().item() <= 1e-5 * (g0[n].abs().max().item() + 1e-12) + 1e-9, n


def test_packed_trainer_steps_match_padded():
    from neko_b200.policy import GatoPolicy
    from neko_b200.training.arguments import TrainingArgs
    from neko_b200.training.trainer import FusedAdamW, Trainer

    class _Tok:
        vocab_size = 120

    g = torch.Generator().manual_seed(0)
    samples = [dict(continuous_obs=torch.randn(T, 5, generator=g) * 3, continuous_actions=torch.randn(T, 2, generator=g).clamp(-1, 1))
               for T in (6, 2, 4, 3, 6, 1, 5, 2, 4)]

    class _OneSample:
        kind = "control"

        def __init__(self):
            self.i = 0

        def sample_batch(self, n, max_tokens=None):
            s = samples[self.i % len(samples)]
            self.i += 1
            return [copy.deepcopy(s)]

    args = TrainingArgs()
    args.batch_size, args.sequence_length = 3, 64
    args.learning_rate, args.init_lr, args.warmup_steps, args.training_steps = 1e-3, 1e-4, 2, 8
    args.gradient_accumulation_steps = 1
    args.text_prop = args.caption_prop = args.vqa_prop = 0.0
    cfg = O.GatoConfig(embed_dim=64, layers=2, heads=2, context_len=64, text_tokens=120)
    w = O.make_weights(cfg, seed=11)
    runs = []
    for packed in (False, True):
        m = GatoPolicy(device="cuda", embed_dim=64, layers=2, heads=2, dropout=0.0, resid_mid_channels=128, context_len=64,
                       text_tokenizer=_Tok())
        m.transformer.drop.p = 0.0
        m.load_state_dict(w, strict=False)
        m.materialize_logits, m.pack_sequences = False, packed
        m.eval()
        opt = FusedAdamW(m, lr=args.learning_rate, betas=(args.beta_1, args.beta_2), eps=args.adam_eps, weight_decay=args.weight_decay)
        tr = Trainer(m, opt, [_OneSample()], args)
        losses = [tr.train_step()[0] for _ in range(3)]
        runs.append((losses, {n: t.detach().clone() for n, t in m.state_dict().items()}))
    (lq, sq), (lp, sp) = runs
    for a, b in zip(lp, lq):
        assert abs(a - b) <= 1e-4 * abs(b), (lp, lq)
    for n, t in sq.items():
        if t.dtype.is_floating_point:
            assert (sp[n] - t).norm().item() <= 1e-3 * t.norm().item() + 1e-7, n


def test_packing_errors_and_padded_interfaces():
    cfg = O.GatoConfig(**SMALL_CASES["mixed"]["cfg"])
    m = make_policy(cfg)
    batch = small_batch("mixed", cfg.text_tokens)
    m.pack_sequences = True
    assert m.materialize_logits
    with pytest.raises(ValueError, match="materialize_logits"):
        m(batch, compute_loss=True)
    with pytest.raises(ValueError, match="materialize_logits"):
        m.stage(batch, compute_loss=True)
    m.materialize_logits = False
    emb, tok, tm, mk = m.tokenize_input_dicts(batch)
    tb = O.tokenize(batch, cfg)
    assert tuple(tok.shape) == tb.tokens.shape and np.array_equal(tok.cpu().numpy(), tb.tokens)
    assert tuple(emb.shape) == tb.tokens.shape + (cfg.embed_dim,)

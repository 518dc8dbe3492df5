"""The oracle next to the UNMODIFIED reference on fresh seeded inputs (oracle.make_golden.vsref_*).  With a reference checkout
(oracle/ref_shim.py) every test runs the reference itself.  Without one it compares the oracle with
tests/golden/oracle_vs_reference.npz: the oracle's outputs on the same inputs at a revision where each of these tests passed
against the live reference (oracle.make_golden.gen_vs_reference), at the same tolerances."""
import os
import sys
import types

import numpy as np
import pytest
import torch

from oracle import gato_oracle as O
from oracle import make_golden as MG
from oracle import ref_shim

HAVE_REF = ref_shim.reference_available()


@pytest.fixture(scope="module")
def record():
    g = np.load(MG.VSREF)
    assert str(g["source"]) == "oracle"
    return g


def _ref_model(cfg, w):
    ref_shim.set_text_vocab(cfg.text_tokens)
    G = ref_shim.load_reference_policy_class()
    m = G(device="cpu", embed_dim=cfg.embed_dim, layers=cfg.layers, heads=cfg.heads, dropout=0.0, resid_mid_channels=128,
          context_len=cfg.context_len, pad_seq=cfg.pad_seq)
    m.transformer.drop.p = 0.0
    m.load_state_dict(w, strict=False)
    return m.eval()


def _check_record(g, prefix, out, w, emb=True):
    """The oracle's forward / backward against a record of oracle.make_golden._forward_record, at the live tolerances."""
    if emb:
        assert np.array_equal(out.tokens.numpy(), g[prefix + "tokens"])
        assert np.array_equal(out.target_masks.numpy(), g[prefix + "target_masks"]) and np.array_equal(out.token_masks.numpy(), g[prefix + "token_masks"])
        assert np.abs(out.token_embeddings.detach().numpy()[:, ::4] - g[prefix + "emb"]).max() <= 1e-6
    lg = out.logits.detach().numpy()
    li = g[prefix + "logit_idx"]
    assert np.abs(lg[li[:, 0], li[:, 1], li[:, 2]] - g[prefix + "logit_val"]).max() <= 1e-5
    assert np.abs(lg.sum(-1) - g[prefix + "logits_rowsum"]).max() <= 1e-5 * lg.shape[-1]
    assert abs(out.loss.item() - float(g[prefix + "loss"])) <= 1e-6
    for n, t in w.items():
        key = prefix + "gval." + n
        if key not in g.files:
            assert t.grad is None or float(t.grad.abs().max()) == 0.0, n
            continue
        gr = t.grad.numpy().reshape(-1)
        scale = max(1.0, float(g[prefix + "gmax." + n]))
        assert abs(float(np.abs(gr).max()) - float(g[prefix + "gmax." + n])) <= 1e-5 * scale, n
        assert np.abs(gr[g[prefix + "gidx." + n]] - g[key]).max() <= 1e-5 * scale, n


@pytest.mark.parametrize("seed", [11, 12])
def test_forward_backward_bitwise_close(seed, record):
    cfg, w, batch = MG.vsref_forward_inputs(seed)
    for t in w.values():
        t.requires_grad_(True)
    out = O.forward(w, batch, cfg, compute_loss=True)
    out.loss.backward()
    if not HAVE_REF:
        _check_record(record, f"fb{seed}.", out, w)
        return
    m = _ref_model(cfg, {k: v.detach() for k, v in w.items()})
    logits, loss = m(batch, compute_loss=True)
    loss.backward()
    emb, tok, tm, mk = m.tokenize_input_dicts(batch)
    assert torch.equal(tok, out.tokens) and torch.equal(tm, out.target_masks) and torch.equal(mk, out.token_masks)
    assert (emb - out.token_embeddings).abs().max().item() <= 1e-6
    assert (logits - out.logits).abs().max().item() <= 1e-5
    assert abs(loss.item() - out.loss.item()) <= 1e-6
    for n, p in m.named_parameters():
        if p.grad is None:
            assert w[n].grad is None or float(w[n].grad.abs().max()) == 0.0
        else:
            assert (p.grad - w[n].grad).abs().max().item() <= 1e-5 * max(1.0, float(p.grad.abs().max())), n


def test_continuous_tokenizer_random_sweep(record):
    cfg = O.GatoConfig()
    x = MG.vsref_sweep_values()
    if not HAVE_REF:
        idx = MG.vsref_sweep_index(x.shape[0])
        for mu_law in (True, False):
            assert np.array_equal(O.discretize(x[idx], mu_law, cfg) - 50257, record[f"sweep.{int(mu_law)}"].astype(np.int64))
        return
    ref_shim.install_shims()
    from gato.policy.input_tokenizers import ContinuousTokenizer
    for mu_law in (True, False):
        tok = ContinuousTokenizer(use_mu_law=mu_law, mu=100, M=256, n_bins=1024, offset=50257)
        ref = tok.encode(torch.from_numpy(x.copy())).numpy()
        assert np.array_equal(ref, O.discretize(x, mu_law, cfg))


def test_dropout_sites_match_reference(record):
    """Pins WHERE the oracle applies its explicit dropout multipliers: the reference runs in train mode with
    nn.Dropout.forward replaced by a recorded Bernoulli mask per call (call order: embeddings, then per layer attention
    weights / attention residual / MLP residual); the oracle replays the same masks."""
    cfg, w, batch = MG.vsref_dropout_inputs()
    if HAVE_REF:
        ref_shim.set_text_vocab(cfg.text_tokens)
        G = ref_shim.load_reference_policy_class()
        m = G(device="cpu", embed_dim=cfg.embed_dim, layers=cfg.layers, heads=cfg.heads, dropout=0.25, resid_mid_channels=128,
              context_len=cfg.context_len, pad_seq=cfg.pad_seq)
        m.load_state_dict(w, strict=False)
        m.train()
        gen = torch.Generator().manual_seed(77)
        calls = []

        def fake_dropout(self, x):
            if not self.training or self.p == 0:
                return x
            mult = (torch.rand(x.shape, generator=gen) >= self.p).to(x.dtype) / (1.0 - self.p)
            calls.append(mult)
            return x * mult

        orig = torch.nn.Dropout.forward
        torch.nn.Dropout.forward = fake_dropout
        try:
            logits, loss = m(batch, compute_loss=True)
        finally:
            torch.nn.Dropout.forward = orig
        loss.backward()
        assert len(calls) == 1 + 3 * cfg.layers
        assert m.transformer.drop.p == 0.1            # SURVEY quirk 8: embd_pdrop ignores --dropout
        drop = {"embd": calls[0]}
        for i in range(cfg.layers):
            drop[("attn", i)], drop[("resid_attn", i)], drop[("resid_mlp", i)] = calls[1 + 3 * i:4 + 3 * i]
        mine = MG.vsref_dropout_masks(cfg, batch)
        assert set(mine) == set(drop) and all(torch.equal(mine[k], drop[k]) for k in drop)
    else:
        drop = MG.vsref_dropout_masks(cfg, batch)
    for t in w.values():
        t.requires_grad_(True)
    out = O.forward(w, batch, cfg, compute_loss=True, training=True, drop=drop)
    out.loss.backward()
    if not HAVE_REF:
        _check_record(record, "drop.", out, w, emb=False)
        return
    assert (logits - out.logits).abs().max().item() <= 1e-5
    assert abs(loss.item() - out.loss.item()) <= 1e-6
    for n, p in m.named_parameters():
        if p.grad is not None:
            assert (p.grad - w[n].grad).abs().max().item() <= 1e-5 * max(1.0, float(p.grad.abs().max())), n


def test_inference_loops_match_reference(record):
    """predict_text / predict_control (gato_policy.py:444-478, 557-616) against the oracle's greedy restatement."""
    cfg, w, text, (obs, act), (img, dact) = MG.vsref_inference_inputs()
    ologits, otoks = O.predict_text(w, text, cfg, max_length=6)
    a_or = O.predict_control(w, dict(continuous_obs=obs.clone(), continuous_actions=act.clone()), cfg, action_tokens=2)
    d_or = O.predict_control(w, dict(images=img.clone(), discrete_actions=dact.clone()), cfg, action_tokens=1, discrete_n=4)
    if not HAVE_REF:
        assert otoks == record["inf.text_tokens"].tolist()
        assert np.abs(ologits.numpy() - record["inf.text_logits"]).max() <= 1e-4
        assert np.array_equal(a_or.reshape(-1).numpy(), record["inf.cont_action"].reshape(-1))
        assert int(d_or) == int(record["inf.disc_action"])
        return
    m = _ref_model(cfg, w)
    with torch.no_grad():
        logits, toks = m.predict_text(text, max_length=6, deterministic=True)
    assert [int(t) for t in toks] == otoks
    assert (logits - ologits).abs().max().item() <= 1e-4
    # control, continuous actions: 3 timesteps, the last action row is padding to be generated
    gym = sys.modules["gymnasium"]
    task = types.SimpleNamespace(action_type=gym.spaces.Box, action_tokens=2, env=None)
    with torch.no_grad():
        a_ref = m.predict_control(dict(continuous_obs=obs.clone(), continuous_actions=act.clone()), task, deterministic=True)
    assert torch.equal(a_ref.reshape(-1).float(), a_or.reshape(-1))
    # control, discrete action restricted to the env's n actions
    task = types.SimpleNamespace(action_type=gym.spaces.Discrete, action_tokens=1,
                                 env=types.SimpleNamespace(action_space=types.SimpleNamespace(n=4)))
    with torch.no_grad():
        d_ref = m.predict_control(dict(images=img.clone(), discrete_actions=dact.clone()), task, deterministic=True)
    assert int(d_ref) == int(d_or)


def test_pretrained_lm_path_matches_oracle(tmp_path, record):
    """--pretrained_lm (gato_policy.py:79-95) through the shims: GPT2Model.from_pretrained of a local GPT-2 checkpoint, gelu_new,
    wte copied into the text rows of embed_token -- the oracle with activation 'gelu_new' reproduces it, the erf form does not."""
    MG.vsref_pretrained_checkpoint(str(tmp_path))
    batch = MG.vsref_pretrained_batch()
    if not HAVE_REF:
        outs = {}
        for act in ("gelu_new", "gelu"):
            oc, w = MG.vsref_pretrained_weights(str(tmp_path), act)
            out = O.forward(w, batch, oc, compute_loss=True)
            outs[act] = out.logits.detach().numpy()[out.token_masks.bool().numpy()].reshape(-1)[record["pre.idx"]]
            assert np.abs(outs[act] - record[f"pre.{act}.logits"]).max() < 2e-5, act
        assert np.abs(outs["gelu_new"] - outs["gelu"]).max() > 1e-3
        return
    ref_shim.set_text_vocab(300)
    G = ref_shim.load_reference_policy_class()
    g = G(device="cpu", embed_dim=8, layers=1, heads=1, dropout=0.0, resid_mid_channels=128, context_len=128, pretrained_lm=str(tmp_path))
    ref_shim.set_text_vocab(50257)
    g.transformer.drop.p = 0.0
    g.eval()
    raw = ref_shim.load_gpt2_checkpoint(str(tmp_path))
    assert torch.equal(g.transformer.h[1].attn.c_attn.bias.detach(), raw["h.1.attn.c_attn.bias"])
    assert torch.equal(g.embed_token.weight[:300].detach(), raw["wte.weight"]) and g.embed_dim == 64
    sd = {k: v.detach().clone() for k, v in g.state_dict().items() if not k.endswith((".attn.bias", ".attn.masked_bias"))}
    logits, loss = g(batch, compute_loss=True)
    errs = {}
    for act in ("gelu_new", "gelu"):
        oc = O.GatoConfig(embed_dim=64, layers=2, heads=4, context_len=128, text_tokens=300, activation_fn=act, wte_rows=300)
        assert set(sd) == set(O.weight_shapes(oc))
        out = O.forward(sd, batch, oc, compute_loss=True)
        errs[act] = (out.logits - logits.detach())[out.token_masks.bool()].abs().max().item()
    assert errs["gelu_new"] < 2e-5 and errs["gelu"] > 1e-3, errs

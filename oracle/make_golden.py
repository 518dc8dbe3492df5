"""Generate tests/golden/*.npz by running the UNMODIFIED reference in the build container.

TEST INFRASTRUCTURE ONLY.  Run here (``python -m oracle.make_golden``); the fixtures are
committed, the reference is not.  Inputs and weights are derived from numpy MT19937 seeds
(``gato_oracle.synth_batch`` / ``make_weights``), so a fixture holds only seeds + reference
OUTPUTS.  What is recorded:

  tokenizer_kat.npz   ContinuousTokenizer.encode (input_tokenizers.py:17-30) on hand-picked edge
                      values and a fixed seeded subset of 550k values (random + clustered on bin
                      edges; ``kat_subset``, which keeps the file small), both tokenizers;
                      PatchPosEncoding eval bins for n=1..40 (embeddings.py:80-100).
  tok_<cfg>.npz       tokenize_input_dicts ids / target masks / token masks (gato_policy.py:195-432)
                      for the five BASELINE.json configs at the real vocabulary (50257+1024+1024).
  fwd_<case>.npz      forward(inputs, compute_loss=True) + backward on small models: loss, logits
                      and token-embedding samples, per-parameter gradient norms and samples.
  scale_<cfg>.npz     the same record for the five BASELINE.json configs AT MODEL SCALE (d=768 / L=6 / H=24 and the
                      real 52 305-row vocabulary; cfg1 d=128 / L=3 / H=1) on a reduced batch (``SCALE_BATCH``).
  oracle_vs_reference.npz   the ORACLE's outputs on the inputs of tests/test_oracle_vs_reference.py, which those tests
                      compare with when no reference checkout is present (``python -m oracle.make_golden vsref``;
                      see gen_vs_reference).
"""
from __future__ import annotations

import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)

from oracle import gato_oracle as O  # noqa: E402
from oracle import ref_shim  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")


def _ref_model(cfg: O.GatoConfig, weights=None, train=False):
    ref_shim.set_text_vocab(cfg.text_tokens)
    G = ref_shim.load_reference_policy_class()
    m = G(device="cpu", embed_dim=cfg.embed_dim, layers=cfg.layers, heads=cfg.heads, dropout=0.0,
          activation_fn=cfg.activation_fn, mu=cfg.mu, M=cfg.M, patch_size=cfg.patch_size,
          resid_mid_channels=cfg.resid_mid_channels, num_groups=cfg.num_groups,
          position_vocab_size=cfg.position_vocab_size, continuous_tokens=cfg.continuous_tokens,
          discrete_tokens=cfg.discrete_tokens, context_len=cfg.context_len,
          use_pos_encoding=cfg.use_pos_encoding, use_patch_pos_encoding=cfg.use_patch_pos_encoding,
          pad_seq=cfg.pad_seq)
    m.transformer.drop.p = 0.0  # embd_pdrop is not wired to --dropout (SURVEY quirk 8)
    if weights is not None:
        res = m.load_state_dict(weights, strict=False)
        assert not res.unexpected_keys, res
        assert all(k.endswith("attn.bias") or k.endswith("masked_bias") for k in res.missing_keys), res
    m.train(train)
    return m


def kat_values() -> np.ndarray:
    rs = np.random.RandomState(11)
    edge = np.array([-300, -256, -255.99, -1, -0.999999, -1e-9, -0.0, 0, 1e-9, 0.5, 0.9999999, 1, 1.0000001,
                     5, 10, 255.9, 256, 1e6, -1e6, 1e-38, 3.4e38], dtype=np.float32)
    wide = (rs.standard_normal(150_000) * 3).astype(np.float32)
    unit = rs.uniform(-1.2, 1.2, 100_000).astype(np.float32)
    # values that sit on / next to the 1024 bin edges of the plain tokenizer ...
    k = rs.randint(0, 1025, 50_000)
    e = (k / 512.0 - 1.0).astype(np.float32)

    near = np.concatenate([e, np.nextafter(e, np.float32(2)), np.nextafter(e, np.float32(-2))])
    # ... and pre-images of the mu-law bin edges: x = sign(y) * ((1+mu*M)^|y| - 1) / mu
    y = (rs.randint(0, 1025, 50_000) / 512.0 - 1.0)
    x = np.sign(y) * (np.power(1 + 100 * 256.0, np.abs(y)) - 1) / 100.0
    x = x.astype(np.float32)
    pre = np.concatenate([x, np.nextafter(x, np.float32(1e9)), np.nextafter(x, np.float32(-1e9))])
    return np.concatenate([edge, wide, unit, near, pre]).astype(np.float32)


KAT_KEEP = 40_000


def kat_subset(x: np.ndarray) -> np.ndarray:
    """Every hand-picked edge value (the first 21) and a fixed seeded sample of the rest, in their original order."""
    rs = np.random.RandomState(12)
    rest = np.sort(rs.choice(np.arange(21, x.shape[0]), KAT_KEEP - 21, replace=False))
    return x[np.concatenate([np.arange(21), rest])]


def gen_tokenizer_kat():
    ref_shim.install_shims()
    from gato.policy.input_tokenizers import ContinuousTokenizer
    from gato.policy.embeddings import PatchPosEncoding

    x = kat_subset(kat_values())
    obs_tok = ContinuousTokenizer(use_mu_law=True, mu=100, M=256, n_bins=1024, offset=50257)
    act_tok = ContinuousTokenizer(use_mu_law=False, mu=100, M=256, n_bins=1024, offset=50257)
    obs = obs_tok.encode(torch.from_numpy(x.copy())).numpy()
    act = act_tok.encode(torch.from_numpy(x.copy())).numpy()
    assert obs.dtype == np.int32 and act.dtype == np.int32
    pos = {}
    enc = PatchPosEncoding(position_vocab_size=128, embed_dim=4).eval()
    for n in range(1, 41):
        # replay the integer part of PatchPosEncoding.forward in eval mode through the module
        tbl = torch.arange(128, dtype=torch.float32)[:, None].repeat(1, 4)
        enc.height_pos_embedding.weight.data.copy_(tbl)
        enc.width_pos_embedding.weight.data.zero_()
        out = enc(torch.zeros(1, n, 1, 4))  # [n,1,4] -> the looked-up row index is the value
        pos[f"pos_{n}"] = out[:, 0, 0].detach().numpy().astype(np.int64)
    np.savez_compressed(os.path.join(GOLD, "tokenizer_kat.npz"), x=x, obs_ids=obs, act_ids=act, **pos)
    print("tokenizer_kat", x.shape, "bins hit", len(np.unique(obs)), len(np.unique(act)))


def gen_tok_configs():
    for name, kw in O.CONFIGS.items():
        cfg = O.GatoConfig(embed_dim=16, layers=1, heads=1, context_len=kw["context_len"])
        m = _ref_model(cfg)
        batch = O.synth_batch(name, seed=1234)
        with torch.no_grad():
            emb, tok, tm, mk = m.tokenize_input_dicts(batch)
        assert tok.dtype == torch.int64 and tm.dtype == torch.float32 and mk.dtype == torch.float32
        np.savez_compressed(os.path.join(GOLD, f"tok_{name}.npz"), tokens=tok.numpy(),
                            target_masks=tm.numpy().astype(np.uint8), token_masks=mk.numpy().astype(np.uint8),
                            seed=1234)
        print("tok", name, tuple(tok.shape), int(mk.sum()))


SMALL_CASES = {
    # name: (config kwargs, batch builder)
    "mixed": dict(cfg=dict(embed_dim=64, layers=2, heads=2, context_len=128, text_tokens=160)),
    "dh128": dict(cfg=dict(embed_dim=128, layers=1, heads=1, context_len=64, text_tokens=96)),
    "geglu_padseq": dict(cfg=dict(embed_dim=64, layers=1, heads=4, context_len=80, text_tokens=160,
                                  activation_fn="geglu", pad_seq=True)),
    "nopos": dict(cfg=dict(embed_dim=32, layers=1, heads=1, context_len=96, text_tokens=64,
                           use_pos_encoding=False, use_patch_pos_encoding=False)),
}


def small_batch(case: str, text_vocab: int) -> list:
    rs = np.random.RandomState({"mixed": 5, "dh128": 6, "geglu_padseq": 7, "nopos": 8}[case])
    f32 = lambda a: torch.from_numpy(np.asarray(a, dtype=np.float32))  # noqa: E731
    ctl = lambda T, o, a: dict(continuous_obs=f32(rs.standard_normal((T, o)) * 3),  # noqa: E731
                               continuous_actions=f32(np.clip(rs.standard_normal((T, a)), -1, 1)))
    batch = [
        ctl(4, 5, 3),
        dict(images=f32(rs.randint(0, 256, (2, 3, 32, 48))), discrete_actions=torch.from_numpy(rs.randint(0, 4, (2, 1)).astype(np.int32))),
        dict(text=rs.randint(0, text_vocab, (17,)).tolist()),
        dict(images=torch.from_numpy(rs.randint(0, 256, (1, 3, 32, 32)).astype(np.uint8)), text=torch.from_numpy(rs.randint(0, text_vocab, (9,)))),
        dict(discrete_obs=torch.from_numpy(rs.randint(0, 10, (3, 2))), continuous_obs=f32(rs.standard_normal((3, 2))),
             discrete_actions=torch.from_numpy(rs.randint(0, 4, (3, 1)))),
        dict(text=torch.from_numpy(rs.randint(0, text_vocab, (2, 6)))),  # 2-D text: T=2
        ctl(1, 2, 1),
    ]
    if case == "dh128":
        batch = batch[:3] + [ctl(6, 4, 2)]
    return batch


# model-scale parity cases: BASELINE.json configuration -> samples in the reduced batch (cfg5: one sample of each kind --
# text 1023 ids, caption 224x224 uint8 + 32 ids, VQA + 24 ids, HalfCheetah-shaped T=42, Breakout-shaped T=26)
SCALE_BATCH = {"cfg1": 4, "cfg2": 6, "cfg3": 2, "cfg4": 2, "cfg5": 5}
SCALE_MODES = {"cfg1": ("eval",), "cfg2": ("eval",), "cfg3": ("eval", "train"), "cfg4": ("eval",), "cfg5": ("eval",)}


def scale_batch(name: str) -> list:
    return O.synth_batch(name, seed=1234, batch=SCALE_BATCH[name])


def _record(m, batch, cfg, n_logit_samples=6000):
    """forward + backward of the reference on `batch`; the fixture keeps outputs only."""
    torch.manual_seed(77)  # train mode: PatchPosEncoding draws from the global CPU RNG
    m.zero_grad()
    logits, loss = m(batch, compute_loss=True)
    loss.backward()
    torch.manual_seed(77)
    with torch.no_grad():
        emb, tok, tm, mk = m.tokenize_input_dicts(batch)
    rs = np.random.RandomState(99)
    B, S, V = logits.shape
    n = n_logit_samples
    li = np.stack([rs.randint(0, B, n), rs.randint(0, S, n), rs.randint(0, V, n)], 1)
    ei = np.stack([rs.randint(0, B, n), rs.randint(0, S, n), rs.randint(0, cfg.embed_dim, n)], 1)
    rec = dict(loss=np.float64(loss.item()), tokens=tok.numpy(), target_masks=tm.numpy(),
               token_masks=mk.numpy(), logit_idx=li,
               logit_val=logits.detach().numpy()[li[:, 0], li[:, 1], li[:, 2]],
               emb_idx=ei, emb_val=emb.numpy()[ei[:, 0], ei[:, 1], ei[:, 2]],
               logits_rowsum=logits.detach().numpy().sum(-1))
    for pn, p in m.named_parameters():
        if p.grad is None:
            rec["gnone." + pn] = np.zeros(1)
            continue
        g = p.grad.numpy().reshape(-1)
        idx = rs.randint(0, g.shape[0], min(256, g.shape[0]))
        rec["gnorm." + pn] = np.float64(np.linalg.norm(g.astype(np.float64)))
        rec["gidx." + pn] = idx
        rec["gval." + pn] = g[idx]
    return rec, logits, loss


def gen_fwd_scale(only=None):
    for name in SCALE_BATCH:
        if only and name not in only:
            continue
        cfg = O.GatoConfig(**O.CONFIGS[name])
        w = O.make_weights(cfg, seed=0, perturb=False)   # the reference's init distributions (zeros / ones where it has them)
        for mode in SCALE_MODES[name]:
            m = _ref_model(cfg, w, train=(mode == "train"))
            rec, logits, loss = _record(m, scale_batch(name), cfg)
            rec["tokens"] = rec["tokens"].astype(np.int32)
            rec["target_masks"] = rec["target_masks"].astype(np.uint8)
            rec["token_masks"] = rec["token_masks"].astype(np.uint8)
            np.savez_compressed(os.path.join(GOLD, f"scale_{name}_{mode}.npz"), **rec)
            print("scale", name, mode, tuple(logits.shape), float(loss), flush=True)
            del m, logits, loss, rec


def gen_fwd_small():
    for case, spec in SMALL_CASES.items():
        cfg = O.GatoConfig(**spec["cfg"])
        w = O.make_weights(cfg, seed=3)
        for mode in ("eval", "train"):
            m = _ref_model(cfg, w, train=(mode == "train"))
            batch = small_batch(case, cfg.text_tokens)
            torch.manual_seed(77)  # train mode: PatchPosEncoding draws from the global CPU RNG
            m.zero_grad()
            logits, loss = m(batch, compute_loss=True)
            loss.backward()
            torch.manual_seed(77)
            with torch.no_grad():
                emb, tok, tm, mk = m.tokenize_input_dicts(batch)
            rs = np.random.RandomState(99)
            B, S, V = logits.shape
            n = 6000
            li = np.stack([rs.randint(0, B, n), rs.randint(0, S, n), rs.randint(0, V, n)], 1)
            ei = np.stack([rs.randint(0, B, n), rs.randint(0, S, n), rs.randint(0, cfg.embed_dim, n)], 1)
            rec = dict(loss=np.float64(loss.item()), tokens=tok.numpy(), target_masks=tm.numpy(),
                       token_masks=mk.numpy(), logit_idx=li,
                       logit_val=logits.detach().numpy()[li[:, 0], li[:, 1], li[:, 2]],
                       emb_idx=ei, emb_val=emb.numpy()[ei[:, 0], ei[:, 1], ei[:, 2]],
                       logits_rowsum=logits.detach().numpy().sum(-1))
            for pn, p in m.named_parameters():
                if p.grad is None:
                    rec["gnone." + pn] = np.zeros(1)
                    continue
                g = p.grad.numpy().reshape(-1)
                idx = rs.randint(0, g.shape[0], min(256, g.shape[0]))
                rec["gnorm." + pn] = np.float64(np.linalg.norm(g.astype(np.float64)))
                rec["gidx." + pn] = idx
                rec["gval." + pn] = g[idx]
            np.savez_compressed(os.path.join(GOLD, f"fwd_{case}_{mode}.npz"), **rec)
            print("fwd", case, mode, tuple(logits.shape), float(loss))


# --------------------------------------------------------------------------------------
# tests/test_oracle_vs_reference.py: inputs, and the record its tests compare the oracle with when no reference checkout is
# present.  The record holds the ORACLE's outputs on these inputs, taken at a revision where every one of those tests passed
# against the live reference; it pins the oracle to what the reference was shown to produce.  With a reference checkout the
# tests compare with the reference itself, as before.
# --------------------------------------------------------------------------------------
VSREF = os.path.join(GOLD, "oracle_vs_reference.npz")


def _f32(a):
    return torch.from_numpy(np.asarray(a, dtype=np.float32))


def vsref_forward_inputs(seed: int):
    cfg = O.GatoConfig(embed_dim=64, layers=2, heads=2, context_len=128, text_tokens=200)
    rs = np.random.RandomState(seed)
    batch = [
        dict(continuous_obs=_f32(rs.standard_normal((5, 4)) * 4), continuous_actions=_f32(np.clip(rs.standard_normal((5, 2)), -1, 1))),
        dict(images=_f32(rs.randint(0, 256, (2, 3, 32, 32))), discrete_actions=torch.from_numpy(rs.randint(0, 6, (2, 1)).astype(np.int32))),
        dict(text=rs.randint(0, 200, (23,)).tolist()),
        dict(images=torch.from_numpy(rs.randint(0, 256, (1, 3, 48, 32)).astype(np.uint8)), text=torch.from_numpy(rs.randint(0, 200, (7,)))),
    ]
    return cfg, O.make_weights(cfg, seed=seed), batch


def vsref_sweep_values() -> np.ndarray:
    rs = np.random.RandomState(99)
    return np.concatenate([rs.standard_normal(300_000) * 10, rs.uniform(-1.5, 1.5, 300_000),
                           np.exp(rs.uniform(-30, 10, 200_000))]).astype(np.float32)


VSREF_SWEEP_KEEP = 40_000


def vsref_sweep_index(n: int) -> np.ndarray:
    """The recorded entries of the sweep: a fixed seeded sample (the whole sweep's ids would not fit a small file)."""
    return np.sort(np.random.RandomState(13).choice(n, VSREF_SWEEP_KEEP, replace=False))


def vsref_dropout_inputs():
    cfg = O.GatoConfig(embed_dim=64, layers=2, heads=2, context_len=64, text_tokens=200)
    rs = np.random.RandomState(5)
    batch = [
        dict(continuous_obs=_f32(rs.standard_normal((4, 3)) * 4), continuous_actions=_f32(np.clip(rs.standard_normal((4, 2)), -1, 1))),
        dict(text=rs.randint(0, 200, (17,)).tolist()),
    ]
    return cfg, O.make_weights(cfg, seed=5), batch


def vsref_dropout_masks(cfg, batch, p_embd=0.1, p=0.25):
    """The Bernoulli multipliers the test draws for the reference's dropout calls, in their call order (embeddings, then per
    layer attention weights / attention residual / MLP residual), from one generator seeded with 77."""
    B, S = O.tokenize(batch, cfg).tokens.shape
    gen = torch.Generator().manual_seed(77)
    draw = lambda shape, q: (torch.rand(shape, generator=gen) >= q).to(torch.float32) / (1.0 - q)  # noqa: E731
    drop = {"embd": draw((B, S, cfg.embed_dim), p_embd)}
    for i in range(cfg.layers):
        drop[("attn", i)] = draw((B, cfg.heads, S, S), p)
        drop[("resid_attn", i)] = draw((B, S, cfg.embed_dim), p)
        drop[("resid_mlp", i)] = draw((B, S, cfg.embed_dim), p)
    return drop


def vsref_inference_inputs():
    cfg = O.GatoConfig(embed_dim=64, layers=2, heads=2, context_len=48, text_tokens=200)
    rs = np.random.RandomState(3)
    text = dict(text=rs.randint(0, 200, (9,)).tolist())
    rs = np.random.RandomState(3)
    rs.randint(0, 200, (9,))                   # the same draws the test makes before the control inputs
    obs, act = _f32(rs.standard_normal((3, 5)) * 2), _f32(np.clip(rs.standard_normal((3, 2)), -1, 1))
    img = _f32(rs.randint(0, 256, (2, 3, 32, 32)))
    dact = torch.from_numpy(rs.randint(0, 4, (2, 1)).astype(np.int32))
    return cfg, O.make_weights(cfg, seed=9), text, (obs, act), (img, dact)


def vsref_pretrained_checkpoint(path: str) -> None:
    """A local GPT-2 checkpoint (transformers' own init, seed 5, weights x4 so that the erf and tanh GELU forms differ)."""
    import transformers
    cfg = transformers.GPT2Config(vocab_size=300, n_embd=64, n_layer=2, n_head=4, n_positions=128, n_ctx=128)
    torch.manual_seed(5)
    hf = transformers.GPT2Model(cfg)
    with torch.no_grad():
        for p in hf.parameters():
            p.mul_(4.0)
    hf.save_pretrained(path)


def vsref_pretrained_weights(path: str, act: str):
    """Oracle weights of --pretrained_lm: the decoder and wte from the checkpoint, wte in the text rows of embed_token, the
    rest seeded."""
    oc = O.GatoConfig(embed_dim=64, layers=2, heads=4, context_len=128, text_tokens=300, activation_fn=act, wte_rows=300)
    w = O.make_weights(oc, seed=5)
    raw = ref_shim.load_gpt2_checkpoint(path)
    for k, t in raw.items():
        if "transformer." + k in w:
            w["transformer." + k] = t.detach().clone().to(torch.float32)
    w["embed_token.weight"][:300] = raw["wte.weight"]
    return oc, w


def vsref_pretrained_batch():
    rs = np.random.RandomState(6)
    return [{"text": list(range(1, 40))}, {"continuous_obs": _f32(rs.standard_normal((5, 3))), "continuous_actions": _f32(rs.uniform(0, 1, (5, 2)))}]


def _forward_record(out, w, prefix, rs, n_logits=4000):
    lg = out.logits.detach().numpy()
    B, S, V = lg.shape
    li = np.stack([rs.randint(0, B, n_logits), rs.randint(0, S, n_logits), rs.randint(0, V, n_logits)], 1)
    rec = {prefix + "tokens": out.tokens.numpy(), prefix + "target_masks": out.target_masks.numpy(), prefix + "token_masks": out.token_masks.numpy(),
           prefix + "emb": out.token_embeddings.detach().numpy()[:, ::4], prefix + "logit_idx": li, prefix + "logit_val": lg[li[:, 0], li[:, 1], li[:, 2]],
           prefix + "logits_rowsum": lg.sum(-1), prefix + "loss": np.float64(out.loss.item())}
    for n, t in w.items():
        if t.grad is not None:
            g = t.grad.numpy().reshape(-1)
            idx = rs.randint(0, g.shape[0], min(64, g.shape[0]))
            rec[prefix + "gmax." + n], rec[prefix + "gidx." + n], rec[prefix + "gval." + n] = np.float64(np.abs(g).max()), idx, g[idx]
    return rec


def gen_vs_reference(tmp_dir: str):
    """Writes VSREF from the oracle (see the comment above)."""
    rs = np.random.RandomState(21)
    rec = {}
    for seed in (11, 12):
        cfg, w, batch = vsref_forward_inputs(seed)
        for t in w.values():
            t.requires_grad_(True)
        out = O.forward(w, batch, cfg, compute_loss=True)
        out.loss.backward()
        rec.update(_forward_record(out, w, f"fb{seed}.", rs))
    x = vsref_sweep_values()
    idx = vsref_sweep_index(x.shape[0])
    for mu_law in (True, False):
        rec[f"sweep.{int(mu_law)}"] = (O.discretize(x, mu_law, O.GatoConfig())[idx] - 50257).astype(np.uint16)
    cfg, w, batch = vsref_dropout_inputs()
    for t in w.values():
        t.requires_grad_(True)
    out = O.forward(w, batch, cfg, compute_loss=True, training=True, drop=vsref_dropout_masks(cfg, batch))
    out.loss.backward()
    rec.update(_forward_record(out, w, "drop.", rs))
    cfg, w, text, (obs, act), (img, dact) = vsref_inference_inputs()
    ologits, otoks = O.predict_text(w, text, cfg, max_length=6)
    rec["inf.text_logits"], rec["inf.text_tokens"] = ologits.numpy(), np.asarray(otoks)
    rec["inf.cont_action"] = O.predict_control(w, dict(continuous_obs=obs, continuous_actions=act), cfg, action_tokens=2).numpy()
    rec["inf.disc_action"] = np.asarray(int(O.predict_control(w, dict(images=img, discrete_actions=dact), cfg, action_tokens=1, discrete_n=4)))
    vsref_pretrained_checkpoint(tmp_dir)
    for act_fn in ("gelu_new", "gelu"):
        oc, w = vsref_pretrained_weights(tmp_dir, act_fn)
        out = O.forward(w, vsref_pretrained_batch(), oc, compute_loss=True)
        valid = out.logits.detach().numpy()[out.token_masks.bool().numpy()]
        pick = np.random.RandomState(22).randint(0, valid.size, 4000)
        rec["pre.idx"], rec[f"pre.{act_fn}.logits"] = pick, valid.reshape(-1)[pick]
    rec["source"] = np.array("oracle")
    np.savez_compressed(VSREF, **rec)
    print("oracle_vs_reference", os.path.getsize(VSREF), "bytes")


def main():
    os.makedirs(GOLD, exist_ok=True)
    torch.set_num_threads(os.cpu_count() or 1)
    if len(sys.argv) > 1 and sys.argv[1] == "scale":
        gen_fwd_scale(sys.argv[2:] or None)
        return
    if len(sys.argv) > 1 and sys.argv[1] == "vsref":      # needs no reference checkout
        import tempfile
        with tempfile.TemporaryDirectory() as d:
            gen_vs_reference(d)
        return
    gen_tokenizer_kat()
    gen_tok_configs()
    gen_fwd_small()
    gen_fwd_scale()


if __name__ == "__main__":
    main()

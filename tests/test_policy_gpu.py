"""Parity of the CUDA hot path (through the GatoPolicy drop-in and the C ABI) against the CPU oracle on the
same seeded inputs, and against the golden fixtures generated from the reference.  GPU only (-m gpu).

Gates (BASELINE.json north_star): ids / masks bit-exact; logits max-abs <= 2e-2 on valid rows; loss relative
<= 1e-3; gradients reported as cosine / relative error per parameter."""
import os

import numpy as np
import pytest
import torch

from oracle import gato_oracle as O
from oracle.make_golden import SCALE_MODES, SMALL_CASES, scale_batch, small_batch

pytestmark = pytest.mark.gpu

LOGIT_TOL = 2e-2
LOSS_RTOL = 1e-3


class _Tok:
    def __init__(self, n):
        self.vocab_size = n


def make_policy(cfg: O.GatoConfig, weights=None, train=False):
    from neko_b200.policy import GatoPolicy
    m = GatoPolicy(device="cuda", embed_dim=cfg.embed_dim, layers=cfg.layers, heads=cfg.heads, dropout=0.0,
                   activation_fn=cfg.activation_fn, mu=cfg.mu, M=cfg.M, patch_size=cfg.patch_size,
                   resid_mid_channels=cfg.resid_mid_channels, num_groups=cfg.num_groups,
                   position_vocab_size=cfg.position_vocab_size, continuous_tokens=cfg.continuous_tokens,
                   discrete_tokens=cfg.discrete_tokens, context_len=cfg.context_len,
                   use_pos_encoding=cfg.use_pos_encoding, use_patch_pos_encoding=cfg.use_patch_pos_encoding,
                   pad_seq=cfg.pad_seq, text_tokenizer=_Tok(cfg.text_tokens))
    m.transformer.drop.p = 0.0
    if weights is not None:
        res = m.load_state_dict(weights, strict=False)
        assert not res.unexpected_keys
        assert all(k.endswith("attn.bias") or k.endswith("masked_bias") for k in res.missing_keys), res
    m.train(train)
    return m


def test_continuous_tokenizer_bit_exact(golden_dir):
    from neko_b200.policy.input_tokenizers import ContinuousTokenizer
    g = np.load(os.path.join(golden_dir, "tokenizer_kat.npz"))
    x = torch.from_numpy(g["x"]).cuda()
    obs = ContinuousTokenizer(use_mu_law=True, mu=100, M=256, n_bins=1024, offset=50257).encode(x)
    act = ContinuousTokenizer(use_mu_law=False, mu=100, M=256, n_bins=1024, offset=50257).encode(x)
    assert obs.dtype == torch.int32
    assert np.array_equal(obs.cpu().numpy(), g["obs_ids"])
    assert np.array_equal(act.cpu().numpy(), g["act_ids"])
    # a larger sweep against the oracle restatement (2M values incl. denormals and huge magnitudes)
    rs = np.random.RandomState(123)
    big = np.concatenate([rs.standard_normal(1_000_000) * 5, rs.uniform(-300, 300, 500_000),
                          np.exp(rs.uniform(-40, 12, 500_000)) * rs.choice([-1, 1], 500_000)]).astype(np.float32)
    cfg = O.GatoConfig()
    got = ContinuousTokenizer(use_mu_law=True, mu=100, M=256, n_bins=1024, offset=50257).encode(torch.from_numpy(big).cuda())
    assert np.array_equal(got.cpu().numpy(), O.discretize(big, True, cfg))


@pytest.mark.parametrize("name", ["cfg1", "cfg2", "cfg3", "cfg4", "cfg5"])
def test_tokenize_configs_bit_exact(golden_dir, name):
    g = np.load(os.path.join(golden_dir, f"tok_{name}.npz"))
    cfg = O.GatoConfig(embed_dim=32, layers=1, heads=1, context_len=O.CONFIGS[name]["context_len"])
    m = make_policy(cfg)
    batch = O.synth_batch(name, seed=int(g["seed"]))
    emb, tok, tm, mk = m.tokenize_input_dicts(batch)
    assert tok.dtype == torch.int64 and tm.dtype == torch.float32 and mk.dtype == torch.float32 and emb.dtype == torch.float32
    assert np.array_equal(tok.cpu().numpy(), g["tokens"])
    assert np.array_equal(tm.cpu().numpy(), g["target_masks"].astype(np.float32))
    assert np.array_equal(mk.cpu().numpy(), g["token_masks"].astype(np.float32))
    # padded embeddings are exact zeros (SURVEY quirk 6)
    assert float(emb[mk == 0].abs().max()) == 0.0 if (mk == 0).any() else True


def test_embeddings_match_oracle():
    cfg = O.GatoConfig(**SMALL_CASES["mixed"]["cfg"])
    w = O.make_weights(cfg, seed=3)
    m = make_policy(cfg, w)
    batch = small_batch("mixed", cfg.text_tokens)
    emb, tok, tm, mk = m.tokenize_input_dicts(batch)
    tb = O.tokenize(batch, cfg)
    ref = O.embed_and_interleave(batch, tb, w, cfg)
    assert np.array_equal(tok.cpu().numpy(), tb.tokens)
    err = (emb.cpu() - ref).abs()
    is_patch = torch.zeros_like(mk.cpu(), dtype=torch.bool)
    S = tb.tokens.shape[1]
    for b, st in enumerate(tb.samples):
        if st.n_patches:
            n = st.ids.shape[0]
            pat = np.zeros(st.tokens_per_timestep, bool)
            pat[:st.n_patches] = True
            is_patch[b, S - n:] = torch.from_numpy(np.tile(pat, st.n_timesteps))
    # gathers / position adds are fp32 exact; patch rows go through bf16 tensor-core projection
    assert float(err[~is_patch].max()) <= 1e-6
    assert float(err[is_patch].max()) <= 3e-2


def _grad_report(m, w):
    rep = {}
    for n, p in m.named_parameters():
        ref = w[n].grad
        if ref is None:
            assert p.grad is None or float(p.grad.abs().max()) == 0.0, n
            continue
        assert p.grad is not None, n
        g = p.grad.detach().cpu().double().reshape(-1)
        r = ref.double().reshape(-1)
        denom = float(g.norm() * r.norm())
        cos = float((g @ r) / denom) if denom > 0 else 1.0
        rel = float((g - r).norm() / (r.norm() + 1e-12))
        rep[n] = (cos, rel, float(r.norm()))
    return rep


@pytest.mark.parametrize("case", ["mixed", "dh128", "nopos", "geglu_padseq"])
@pytest.mark.parametrize("mode", ["eval", "train"])
def test_forward_backward_vs_oracle_and_golden(golden_dir, case, mode):
    g = np.load(os.path.join(golden_dir, f"fwd_{case}_{mode}.npz"))
    cfg = O.GatoConfig(**SMALL_CASES[case]["cfg"])
    w = O.make_weights(cfg, seed=3)
    m = make_policy(cfg, w, train=(mode == "train"))
    batch = small_batch(case, cfg.text_tokens)
    torch.manual_seed(77)
    logits, loss = m(batch, compute_loss=True)
    loss.backward()
    torch.cuda.synchronize()
    for t in w.values():
        t.requires_grad_(True)
    torch.manual_seed(77)
    ref = O.forward(w, batch, cfg, compute_loss=True, training=(mode == "train"))
    ref.loss.backward()

    assert logits.dtype == torch.float32 and tuple(logits.shape) == tuple(ref.logits.shape)
    valid = ref.token_masks.bool()
    lerr = (logits.detach().cpu() - ref.logits.detach())[valid].abs().max().item()
    assert lerr <= LOGIT_TOL, f"logits max-abs {lerr}"
    assert abs(loss.item() - ref.loss.item()) <= LOSS_RTOL * abs(ref.loss.item())
    # the committed reference outputs
    assert abs(loss.item() - float(g["loss"])) <= LOSS_RTOL * abs(float(g["loss"]))
    li = g["logit_idx"]
    keep = g["token_masks"][li[:, 0], li[:, 1]] > 0
    got = logits.detach().cpu().numpy()[li[:, 0], li[:, 1], li[:, 2]]
    assert np.abs(got - g["logit_val"])[keep].max() <= LOGIT_TOL
    rep = _grad_report(m, w)
    bad = {n: v for n, v in rep.items() if v[2] > 1e-6 and (v[0] < 0.99 or v[1] > 0.12)}
    assert not bad, f"gradient mismatch (cos, rel, ref-norm): {bad}"
    # weight matrices of the decoder must be tight
    tight = [v for n, v in rep.items() if n.endswith("c_fc.weight") or n.endswith("c_attn.weight") or n == "predict_token.weight"]
    assert min(v[0] for v in tight) > 0.999


def test_geglu_gate_parameters_receive_gradients():
    """--activation_fn geglu (trajectory_gpt2.py:267-276): the gate Linear is part of the arena and of backward."""
    cfg = O.GatoConfig(**SMALL_CASES["geglu_padseq"]["cfg"])
    w = O.make_weights(cfg, seed=3)
    m = make_policy(cfg, w, train=True)
    batch = small_batch("geglu_padseq", cfg.text_tokens)
    _, loss = m(batch, compute_loss=True)
    loss.backward()
    for t in w.values():
        t.requires_grad_(True)
    ref = O.forward(w, batch, cfg, compute_loss=True, training=True)
    ref.loss.backward()
    rep = _grad_report(m, w)
    gates = {n: v for n, v in rep.items() if "gated_layer" in n}
    assert len(gates) == 2 * cfg.layers
    assert min(v[0] for v in gates.values()) > 0.995, gates


def test_pad_seq_matches_oracle():
    kw = dict(SMALL_CASES["geglu_padseq"]["cfg"])
    kw["activation_fn"] = "gelu"
    cfg = O.GatoConfig(**kw)
    w = O.make_weights(cfg, seed=3)
    m = make_policy(cfg, w)
    batch = small_batch("geglu_padseq", cfg.text_tokens)
    logits, loss = m(batch, compute_loss=True)
    ref = O.forward(w, batch, cfg, compute_loss=True)
    assert logits.shape[1] == cfg.context_len
    valid = ref.token_masks.bool()
    assert (logits.detach().cpu() - ref.logits)[valid].abs().max().item() <= LOGIT_TOL
    assert abs(loss.item() - ref.loss.item()) <= LOSS_RTOL * abs(ref.loss.item())


def test_head_modes_and_accumulation_agree():
    cfg = O.GatoConfig(**SMALL_CASES["mixed"]["cfg"])
    w = O.make_weights(cfg, seed=3)
    batch = small_batch("mixed", cfg.text_tokens)
    grads = {}
    for mode in ("dense", "rows", "lean", "lean32"):
        m = make_policy(cfg, w)
        m.head_mode = "rows" if mode != "dense" else "dense"
        m.materialize_logits = not mode.startswith("lean")
        m.lean_logits_f16 = mode == "lean"      # default: the loss rows' logits live in fp16 between head GEMM and fused CE
        _, loss = m(batch, compute_loss=True)
        loss.backward()
        grads[mode] = ({n: p.grad.clone() for n, p in m.named_parameters() if p.grad is not None}, loss.item())
        if mode == "lean":
            assert m._ws["logits_rows_f16"].dtype == torch.float16 and m._graphs == {}
    for mode in ("rows", "lean", "lean32"):
        # fp16 logits move the loss by ~1e-5 relative (gate: 1e-3); the fp32 routes agree to rounding
        assert abs(grads[mode][1] - grads["dense"][1]) < (3e-4 if mode == "lean" else 1e-5), (mode, grads[mode][1], grads["dense"][1])
        for n, gd in grads["dense"][0].items():
            gr = grads[mode][0][n]
            assert (gd - gr).norm().item() <= 2e-2 * gd.norm().item() + 1e-7, (mode, n)
    # two backward passes accumulate (gradient accumulation, trainer.py:176)
    m = make_policy(cfg, w)
    for _ in range(2):
        _, loss = m(batch, compute_loss=True)
        loss.backward()
    for n, gd in grads["dense"][0].items():
        assert (m.get_parameter(n).grad - 2 * gd).norm().item() <= 2e-2 * (2 * gd).norm().item() + 1e-7, n
    m.zero_grad()
    assert all(p.grad is None for p in m.parameters())


def test_state_dict_layout_and_errors():
    cfg = O.GatoConfig(**SMALL_CASES["mixed"]["cfg"])
    m = make_policy(cfg)
    keys = set(m.state_dict().keys())
    expect = set(O.weight_shapes(cfg).keys())
    for i in range(cfg.layers):
        expect |= {f"transformer.h.{i}.attn.bias", f"transformer.h.{i}.attn.masked_bias"}
    assert keys == expect
    for k, shp in O.weight_shapes(cfg).items():
        assert tuple(m.state_dict()[k].shape) == tuple(shp), k
    with pytest.raises(AssertionError):
        m([{"continuous_obs": torch.zeros(3, 2), "continuous_actions": torch.zeros(4, 1)}])
    with pytest.raises(AssertionError):
        m([{"images": torch.zeros(1, 3, 20, 32)}])
    with pytest.raises(AssertionError):
        m(None)
    from neko_b200.policy import GatoPolicy
    with pytest.raises(ValueError):  # the reference's own default 132 is not divisible by 32 groups (SURVEY quirk 10)
        GatoPolicy(device="cuda", embed_dim=64, layers=1, heads=2, dropout=0.0, text_tokenizer=_Tok(64))
    with pytest.raises(Exception):
        GatoPolicy(device="cpu", embed_dim=64, layers=1, heads=2, dropout=0.0, resid_mid_channels=128)


def test_init_distributions_match_reference():
    """SURVEY a12 (trajectory_gpt2.py:375-386 + torch defaults for everything GatoPolicy owns): per-tensor mean / std / range
    of a freshly constructed policy against the reference constructed on the CPU (oracle/_ref or /root/reference through the
    shims), or against the documented distributions when no reference tree is present."""
    from neko_b200.policy import GatoPolicy
    from oracle import ref_shim
    kw = dict(embed_dim=256, layers=2, heads=8, dropout=0.0, resid_mid_channels=128, context_len=128)
    torch.manual_seed(5)
    m = GatoPolicy(device="cuda", text_tokenizer=_Tok(50257), **kw)
    ours = {n: p.detach().float().cpu() for n, p in m.named_parameters()}
    ref = None
    if ref_shim.reference_available():
        ref_shim.set_text_vocab(50257)
        torch.manual_seed(5)
        r = ref_shim.load_reference_policy_class()(device="cpu", **kw)
        ref = {n: p.detach().float() for n, p in r.named_parameters()}
        assert set(ref) == set(ours)
    for n, t in ours.items():
        numel = t.numel()
        if ref is not None:
            q = ref[n]
            assert tuple(q.shape) == tuple(t.shape), n
            mean_r, std_r, lo_r, hi_r = float(q.mean()), float(q.std()) if numel > 1 else 0.0, float(q.min()), float(q.max())
        else:   # documented distributions
            if ".ln_" in n or "ln_f" in n or "gn2" in n:
                mean_r, std_r = (1.0, 0.0) if n.endswith("weight") else (0.0, 0.0)
            elif n.startswith("transformer.") and n.endswith("bias") or n == "separator_token":
                mean_r, std_r = 0.0, 0.0
            elif n.startswith("transformer."):
                mean_r, std_r = 0.0, 0.02
            elif n.endswith("embedding.weight") or n in ("embed_token.weight", "pos_embed_observation.weight"):
                mean_r, std_r = 0.0, 1.0
            else:
                continue
            lo_r = hi_r = None
        mean_o, std_o = float(t.mean()), float(t.std()) if numel > 1 else 0.0
        if std_r == 0.0:      # constants: ones / zeros exactly
            assert std_o == 0.0 and mean_o == mean_r, (n, mean_o, std_o)
            continue
        if numel < 64:   # too few draws for moments (conv2.bias has 3): inside the kaiming-uniform support 1/sqrt(fan_in)
            wshape = ours[n[:-4] + "weight"].shape
            assert float(t.abs().max()) <= 1.0 / (float(np.prod(wshape[1:])) ** 0.5) + 1e-7, n
            continue
        se = std_r / (numel ** 0.5)
        assert abs(mean_o - mean_r) <= 6 * se * 2 ** 0.5 + 1e-7, (n, mean_o, mean_r)
        assert abs(std_o - std_r) <= 6 * std_r / (2 * numel) ** 0.5 * 2 ** 0.5 + 0.02 * std_r, (n, std_o, std_r)
        if lo_r is not None and not (n.endswith("embedding.weight") or "embed" in n or n.startswith("transformer.")):
            # uniform kaiming ranges (nn.Linear / nn.Conv2d defaults): same support
            assert abs(float(t.min()) - lo_r) <= 0.05 * (hi_r - lo_r) and abs(float(t.max()) - hi_r) <= 0.05 * (hi_r - lo_r), n


def _tiny_gpt2_checkpoint(tmp_path, vocab=300, d=64, layers=2, heads=2, n_ctx=128, scale=2.0):
    """A local HF GPT-2 checkpoint directory (config.json + model.safetensors) with weights large enough that the erf and
    tanh GELU forms differ visibly."""
    import transformers
    cfg = transformers.GPT2Config(vocab_size=vocab, n_embd=d, n_layer=layers, n_head=heads, n_positions=n_ctx, n_ctx=n_ctx)
    torch.manual_seed(21)
    m = transformers.GPT2Model(cfg)
    with torch.no_grad():
        for p in m.parameters():
            p.mul_(scale)
    m.save_pretrained(str(tmp_path))
    return str(tmp_path)


def test_pretrained_lm_matches_oracle(tmp_path):
    """--pretrained_lm (gato_policy.py:79-95): decoder shape / weights / gelu_new from a GPT-2 checkpoint directory, the text
    rows of embed_token start from its wte, wpe is dropped.  Forward + backward against the oracle run with
    activation 'gelu_new' (pinned to the reference's own pretrained path in tests/test_oracle_vs_reference.py)."""
    from neko_b200.policy import GatoPolicy
    from safetensors.torch import load_file
    ckpt = _tiny_gpt2_checkpoint(tmp_path)
    torch.manual_seed(3)
    m = GatoPolicy(device="cuda", embed_dim=8, layers=1, heads=1, dropout=0.0, resid_mid_channels=128, context_len=96,
                   pretrained_lm=ckpt, text_tokenizer=_Tok(300))     # embed_dim / layers / heads are overridden by the checkpoint
    assert (m.embed_dim, m.layers, m.heads) == (64, 2, 2) and m._gelu_tanh
    m.transformer.drop.p = 0.0
    m.eval()
    raw = load_file(os.path.join(ckpt, "model.safetensors"))
    sd = m.state_dict()
    assert tuple(sd["transformer.wte.weight"].shape) == (300, 64) and not any("wpe" in k for k in sd)
    assert torch.equal(sd["transformer.h.1.mlp.c_fc.weight"].cpu(), raw["h.1.mlp.c_fc.weight"])
    assert torch.equal(sd["embed_token.weight"][:300].cpu(), raw["wte.weight"])
    cfg = O.GatoConfig(embed_dim=64, layers=2, heads=2, context_len=96, text_tokens=300, activation_fn="gelu_new", wte_rows=300)
    w = {k: v.detach().cpu().clone() for k, v in sd.items() if not k.endswith((".attn.bias", ".attn.masked_bias"))}
    assert set(w) == set(O.weight_shapes(cfg))
    batch = [dict(text=list(range(5, 60))), dict(continuous_obs=torch.randn(6, 4) * 2, continuous_actions=torch.rand(6, 2) * 2 - 1),
             dict(images=torch.randint(0, 256, (1, 3, 32, 32), dtype=torch.uint8), text=torch.arange(7, 19))]
    logits, loss = m(batch, compute_loss=True)
    loss.backward()
    for t in w.values():
        t.requires_grad_(True)
    ref = O.forward(w, batch, cfg, compute_loss=True)
    ref.loss.backward()
    valid = ref.token_masks.bool()
    lerr = (logits.detach().cpu() - ref.logits.detach())[valid].abs().max().item()
    # the checkpoint's weights are scaled up 4x here: the absolute logit gate scales with the logits' spread (0.58 at normal init)
    spread = max(1.0, float(ref.logits.detach()[valid].std()) / 0.58)
    print('pretrained: logits err', lerr, 'spread factor', spread)
    assert lerr <= LOGIT_TOL * spread and abs(loss.item() - ref.loss.item()) <= LOSS_RTOL * abs(ref.loss.item()), (lerr, spread, loss.item(), ref.loss.item())
    # (that the tanh form is really what the epilogues compute is checked at kernel level: test_gemm_gelu_tanh_epilogues)
    rep = _grad_report(m, w)
    bad = {n: v for n, v in rep.items() if v[2] > 1e-6 and v[0] < 0.99}
    assert not bad, bad
    assert min(v[0] for n, v in rep.items() if n.endswith("c_fc.weight") or n.endswith("mlp.c_proj.weight")) > 0.999
    with pytest.raises(FileNotFoundError):
        GatoPolicy(device="cuda", embed_dim=64, layers=1, heads=2, dropout=0.0, resid_mid_channels=128, pretrained_lm="no-such-model",
                   text_tokenizer=_Tok(300))


def test_kwargs_path_matches_inputs_path():
    cfg = O.GatoConfig(**SMALL_CASES["mixed"]["cfg"])
    w = O.make_weights(cfg, seed=3)
    m = make_policy(cfg, w)
    batch = small_batch("mixed", cfg.text_tokens)
    with torch.no_grad():
        logits, loss = m(batch, compute_loss=True)
        emb, tok, tm, mk = m.tokenize_input_dicts(batch)
        logits2, loss2 = m(token_embeddings=emb, tokens=tok, token_target_masks=tm, token_masks=mk, compute_loss=True)
    valid = mk.bool()
    assert (logits - logits2)[valid].abs().max().item() < 1e-5
    assert abs(loss.item() - loss2.item()) < 1e-5


GRAD_COS = 0.99          # every parameter
GRAD_COS_TIGHT = 0.999   # decoder weight matrices and the LM head


@pytest.mark.parametrize("name,mode", [(n, md) for n in ("cfg1", "cfg2", "cfg3", "cfg4", "cfg5") for md in SCALE_MODES[n]])
def test_model_scale_parity(golden_dir, name, mode):
    """Every BASELINE.json configuration AT MODEL SCALE (d=768 / L=6 / H=24, V=52 305; cfg1: d=128 / L=3 / H=1, dh=128) on
    the reduced batches of oracle.make_golden.SCALE_BATCH -- cfg3: 2 x 13 frames 96x96 (S=494); cfg4: 2 x 1023 ids (S=1024,
    2 044 loss rows through the fused CE, vocabulary-wide embedding-gradient atomics); cfg5: one sample of each kind incl. a
    224x224 uint8 caption, left-padded to 1024.  Checked against the oracle live AND against the reference's own outputs
    (tests/golden/scale_*.npz): ids bit-exact, logits <= 2e-2 on valid rows, loss rel <= 1e-3, gradient cosines."""
    g = np.load(os.path.join(golden_dir, f"scale_{name}_{mode}.npz"))
    cfg = O.GatoConfig(**O.CONFIGS[name])
    w = O.make_weights(cfg, seed=0, perturb=False)
    m = make_policy(cfg, w, train=(mode == "train"))
    if os.environ.get("NEKO_MLP_PROJ_BF16") is not None:      # experiment switch (DESIGN.md section 4 "precision")
        m.mlp_proj_bf16 = os.environ["NEKO_MLP_PROJ_BF16"] == "1"
    batch = scale_batch(name)
    torch.manual_seed(77)
    logits, loss = m(batch, compute_loss=True)
    loss.backward()
    torch.cuda.synchronize()
    torch.manual_seed(77)
    emb, tok, tm, mk = m.tokenize_input_dicts(batch)
    assert np.array_equal(tok.cpu().numpy(), g["tokens"].astype(np.int64))
    assert np.array_equal(tm.cpu().numpy(), g["target_masks"].astype(np.float32))
    assert np.array_equal(mk.cpu().numpy(), g["token_masks"].astype(np.float32))
    ei = g["emb_idx"]
    assert np.abs(emb.cpu().numpy()[ei[:, 0], ei[:, 1], ei[:, 2]] - g["emb_val"]).max() <= 2e-2   # fp16 patch operands
    # the reference's own numbers
    gl = float(g["loss"])
    li = g["logit_idx"]
    keep = g["token_masks"][li[:, 0], li[:, 1]] > 0
    got = logits.detach().cpu().numpy()[li[:, 0], li[:, 1], li[:, 2]]
    gerr = float(np.abs(got - g["logit_val"])[keep].max())
    rs_err = float(np.abs(logits.detach().sum(-1).cpu().numpy() - g["logits_rowsum"])[g["token_masks"] > 0].max())
    print(f"{name}/{mode}: loss {loss.item():.6f} (reference {gl:.6f}), sampled logits max-abs {gerr:.3e}, row-sum max-abs {rs_err:.3e}")
    assert gerr <= LOGIT_TOL
    assert abs(loss.item() - gl) <= LOSS_RTOL * abs(gl)
    gcos = {}
    for key in g.files:
        if key.startswith("gnone."):
            p = m.get_parameter(key[6:])
            assert p.grad is None or float(p.grad.abs().max()) == 0.0, key
        elif key.startswith("gnorm.") and float(g[key]) > 1e-7:
            pn = key[6:]
            gr = m.get_parameter(pn).grad.detach().reshape(-1)
            nrm = float(gr.double().norm())
            assert abs(nrm - float(g[key])) <= 0.05 * float(g[key]), (pn, nrm, float(g[key]))
            idx = torch.from_numpy(g["gidx." + pn]).to(gr.device)
            a, b = gr[idx].double().cpu().numpy(), g["gval." + pn].astype(np.float64)
            if np.linalg.norm(b) > 0:
                gcos[pn] = float(a @ b / (np.linalg.norm(a) * np.linalg.norm(b) + 1e-300))
    assert min(gcos.values()) > 0.98, sorted(gcos.items(), key=lambda kv: kv[1])[:5]   # 256-element samples: coarse
    # the oracle, live: all logits on valid rows and full gradient cosines
    for k in w:
        w[k].requires_grad_(True)
    torch.manual_seed(77)
    ref = O.forward(w, batch, cfg, compute_loss=True, training=(mode == "train"))
    ref.loss.backward()
    valid = ref.token_masks.bool()
    lerr = (logits.detach().cpu() - ref.logits.detach())[valid].abs().max().item()
    rep = _grad_report(m, w)
    worst = sorted(((n, v) for n, v in rep.items() if v[2] > 1e-7), key=lambda kv: kv[1][0])[:6]
    print(f"{name}/{mode}: logits max-abs {lerr:.3e} over {int(valid.sum())} valid rows; worst gradient cosines (cos, rel, norm): {worst}")
    assert lerr <= LOGIT_TOL
    assert abs(loss.item() - ref.loss.item()) <= LOSS_RTOL * abs(ref.loss.item())
    assert all(v[0] >= GRAD_COS for n, v in rep.items() if v[2] > 1e-7), worst
    tight = {n: v for n, v in rep.items() if n == "predict_token.weight" or
             (n.startswith("transformer.h.") and n.endswith(".weight") and ".ln_" not in n)}
    assert min(v[0] for v in tight.values()) >= GRAD_COS_TIGHT, sorted(tight.items(), key=lambda kv: kv[1][0])[:4]


def test_cuda_graph_replay_matches_eager():
    """Graph mode: eager on first sight of a batch shape, capture on the second, replay afterwards -- with fresh data
    every step the results must equal the eager engine bit for bit (same kernels, same order)."""
    cfg = O.GatoConfig(**SMALL_CASES["mixed"]["cfg"])
    w = O.make_weights(cfg, seed=3)
    eager = make_policy(cfg, w)
    graph = make_policy(cfg, w)
    graph.use_cuda_graphs = True
    base = small_batch("mixed", cfg.text_tokens)

    def perturb(batch, k):
        out = []
        for s in batch:
            d = {}
            for key, v in s.items():
                if isinstance(v, torch.Tensor) and v.dtype == torch.float32 and key != "images":
                    d[key] = v * (1.0 + 0.1 * k)
                else:
                    d[key] = v
            out.append(d)
        return out

    for k in range(4):   # eager, capture, replay, replay
        batch = perturb(base, k)
        for m in (eager, graph):
            m.zero_grad()
        le, loss_e = eager(batch, compute_loss=True)
        loss_e.backward()
        lg, loss_g = graph(batch, compute_loss=True)
        loss_g.backward()
        torch.cuda.synchronize()
        assert torch.equal(le, lg), k
        assert loss_e.item() == loss_g.item(), k
        for (n, pe), (_, pg) in zip(eager.named_parameters(), graph.named_parameters()):
            if pe.grad is None:
                assert pg.grad is None
            else:
                denom = pe.grad.abs().max().item() + 1e-12
                assert (pe.grad - pg.grad).abs().max().item() <= 1e-5 * denom + 1e-9, (k, n)   # atomics reorder fp32 sums
    assert any("fwd" in e for e in graph._graphs.values())
    # gradient accumulation through the graphs
    graph.zero_grad()
    eager.zero_grad()
    for _ in range(2):
        _, l1 = eager(base, compute_loss=True); l1.backward()
        _, l2 = graph(base, compute_loss=True); l2.backward()
    torch.cuda.synchronize()
    for (n, pe), (_, pg) in zip(eager.named_parameters(), graph.named_parameters()):
        if pe.grad is not None:
            assert (pe.grad - pg.grad).abs().max().item() <= 1e-5 * (pe.grad.abs().max().item() + 1e-12) + 1e-9, n


# ---------------------------------------------------------------------------------------------------
# dropout (trajectory_gpt2.py:179,254,278,707): the kernels' counter-based masks are extracted and the step is replayed
# in the oracle with exactly those masks -> same parity gates as the dropout-free step
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case,graphs", [("mixed", False), ("dh128", False), ("mixed", True)])
def test_train_step_with_dropout_matches_oracle_replay(case, graphs):
    cfg = O.GatoConfig(**SMALL_CASES[case]["cfg"])
    w = O.make_weights(cfg, seed=3)
    m = make_policy(cfg, w, train=True)
    m.transformer.drop.p = 0.1                       # the reference's embd_pdrop (SURVEY quirk 8)
    for blk in m.transformer.h:
        blk.attn.attn_dropout.p = 0.2
        blk.attn.resid_dropout.p = 0.15
        blk.mlp.dropout.p = 0.15
    m.use_cuda_graphs = graphs
    batch = small_batch(case, cfg.text_tokens)
    seen = []
    for it in range(3 if graphs else 1):             # graphs: eager, capture, replay -- fresh masks every time
        m.zero_grad()
        torch.manual_seed(77)
        logits, loss = m(batch, compute_loss=True)
        loss.backward()
        torch.cuda.synchronize()
        drop = {k: v.cpu() for k, v in m.dropout_multipliers().items()}
        assert len(drop) == 1 + 3 * cfg.layers
        seen.append(drop["embd"])
        keep_rate = float((drop["embd"] > 0).float().mean())
        assert abs(keep_rate - 0.9) < 0.02, keep_rate
    if graphs:
        assert not torch.equal(seen[0], seen[1]) and not torch.equal(seen[1], seen[2])
    for t in w.values():
        t.requires_grad_(True)
    torch.manual_seed(77)
    ref = O.forward(w, batch, cfg, compute_loss=True, training=True, drop=drop)
    ref.loss.backward()
    valid = ref.token_masks.bool()
    lerr = (logits.detach().cpu() - ref.logits.detach())[valid].abs().max().item()
    assert lerr <= LOGIT_TOL, f"logits max-abs {lerr}"
    assert abs(loss.item() - ref.loss.item()) <= LOSS_RTOL * abs(ref.loss.item())
    rep = _grad_report(m, w)
    bad = {n: v for n, v in rep.items() if v[2] > 1e-6 and (v[0] < 0.99 or v[1] > 0.12)}
    assert not bad, f"gradient mismatch (cos, rel, ref-norm): {bad}"
    tight = [v for n, v in rep.items() if n.endswith("c_fc.weight") or n.endswith("c_attn.weight") or n == "predict_token.weight"]
    assert min(v[0] for v in tight) > 0.999
    # eval mode ignores every p
    m.eval()
    l1, _ = m(batch, compute_loss=False)
    l2, _ = m(batch, compute_loss=False)
    assert torch.equal(l1, l2) and m.dropout_multipliers() == {}


# ---------------------------------------------------------------------------------------------------
# inference loops (gato_policy.py:444-616) against the oracle's greedy restatement
# ---------------------------------------------------------------------------------------------------
def _margin_ok(rows, tol=4 * LOGIT_TOL):
    """True for the steps whose oracle top-2 margin is larger than the logits tolerance (greedy pick is unambiguous)."""
    out = []
    for r in rows:
        top = torch.topk(r, 2).values
        out.append(float(top[0] - top[1]) > tol)
    return out


def test_predict_text_and_control_match_oracle():
    import types
    cfg = O.GatoConfig(embed_dim=64, layers=2, heads=2, context_len=48, text_tokens=200)
    w = O.make_weights(cfg, seed=9)
    m = make_policy(cfg, w)
    rs = np.random.RandomState(3)
    prompt = rs.randint(0, 200, (9,)).tolist()
    logits, toks = m.predict_text(dict(text=list(prompt)), max_length=6, deterministic=True)
    ologits, otoks = O.predict_text(w, dict(text=list(prompt)), cfg, max_length=6)
    assert tuple(logits.shape) == (6, cfg.text_tokens) and len(toks) == 6
    ok = _margin_ok(list(ologits))
    for i in range(6):
        assert (logits[i].cpu() - ologits[i]).abs().max().item() <= LOGIT_TOL
        if not ok[i]:
            break                       # ambiguous argmax: later steps may legitimately diverge
        assert int(toks[i]) == otoks[i]
    # sampling path runs and stays inside the text vocabulary
    _, stoks = m.predict_text(dict(text=list(prompt)), max_length=3, deterministic=False)
    assert all(0 <= int(t) < cfg.text_tokens for t in stoks)

    f32 = lambda a: torch.from_numpy(np.asarray(a, dtype=np.float32))  # noqa: E731
    obs, act = f32(rs.standard_normal((3, 5)) * 2), f32(np.clip(rs.standard_normal((3, 2)), -1, 1))
    box = type("Box", (), {})
    disc = type("Discrete", (), {})
    task = types.SimpleNamespace(action_type=box, action_tokens=2, env=None)
    a = m.predict_control(dict(continuous_obs=obs.cuda(), continuous_actions=act.cuda()), task, deterministic=True)
    a_or = O.predict_control(w, dict(continuous_obs=obs.clone(), continuous_actions=act.clone()), cfg, action_tokens=2)
    assert tuple(a.shape) == (2,) and float(a.min()) >= -1.0 and float(a.max()) <= 1.0
    assert (a.cpu().float() - a_or).abs().max().item() <= 2.0 / cfg.continuous_tokens * 8   # within a few bins of the oracle pick
    img = f32(rs.randint(0, 256, (2, 3, 32, 32)))
    dact = torch.from_numpy(rs.randint(0, 4, (2, 1)).astype(np.int32))
    task = types.SimpleNamespace(action_type=disc, action_tokens=1, env=types.SimpleNamespace(action_space=types.SimpleNamespace(n=4)))
    d = m.predict_control(dict(images=img.cuda(), discrete_actions=dact.cuda()), task, deterministic=True)
    assert 0 <= int(d) < 4


def test_predict_response_runs_on_image_embeddings():
    cfg = O.GatoConfig(embed_dim=64, layers=1, heads=2, context_len=64, text_tokens=200)
    w = O.make_weights(cfg, seed=4)
    m = make_policy(cfg, w)

    class _Txt(_Tok):
        def decode(self, ids):
            return " ".join(str(i) for i in ids)

        def encode(self, s):
            return [int(t) for t in s.split()]

    m.text_tokenizer = _Txt(cfg.text_tokens)
    rs = np.random.RandomState(8)
    img = torch.from_numpy(rs.randint(0, 256, (1, 3, 32, 48)).astype(np.uint8))
    logits, text = m.predict_answer(img, "5 7 11", max_length=4, deterministic=True)
    assert tuple(logits.shape) == (4, cfg.text_tokens) and len(text.split()) == 4
    # first generated token: oracle forward on [image, prompt] -> argmax at the last position
    batch = [dict(images=img.clone(), text=torch.tensor([5, 7, 11]))]
    ref = O.forward(w, batch, cfg, compute_loss=False)
    row = ref.logits[0, -2, :cfg.text_tokens]     # position of the last prompt token (the separator follows it)
    assert (logits[0].cpu() - row).abs().max().item() <= LOGIT_TOL


@pytest.mark.parametrize("case", ["text", "control", "overflow"])
def test_kv_cached_generation_matches_full_recompute(case):
    """SURVEY 8(f)2: the KV-cached decode (one position per step) against re-running the whole context per token (what the
    reference does and what use_kv_cache=False does), incl. the fallback once the context window starts to slide."""
    import types
    cfg = O.GatoConfig(embed_dim=64, layers=2, heads=2, context_len=32 if case == "overflow" else 64, text_tokens=200)
    w = O.make_weights(cfg, seed=21)
    m = make_policy(cfg, w)
    rs = np.random.RandomState(4)
    f32 = lambda a: torch.from_numpy(np.asarray(a, dtype=np.float32))  # noqa: E731

    def run(use_kv):
        m.use_kv_cache = use_kv
        if case == "control":
            obs, act = f32(rs0.standard_normal((4, 5)) * 2), f32(np.clip(rs0.standard_normal((4, 3)), -1, 1))
            task = types.SimpleNamespace(action_type=type("Box", (), {}), action_tokens=3, env=None)
            a = m.predict_control(dict(continuous_obs=obs.cuda(), continuous_actions=act.cuda()), task, deterministic=True)
            return a.float().cpu(), None
        n_prompt, n_new = (28, 8) if case == "overflow" else (11, 7)
        prompt = rs0.randint(0, 200, (n_prompt,)).tolist()
        logits, toks = m.predict_text(dict(text=prompt), max_length=n_new, deterministic=True)
        return logits.float().cpu(), [int(t) for t in toks]

    rs0 = np.random.RandomState(4)
    a_kv, t_kv = run(True)
    rs0 = np.random.RandomState(4)
    a_full, t_full = run(False)
    if case == "control":
        assert (a_kv - a_full).abs().max().item() <= 2.0 / cfg.continuous_tokens * 4
        return
    # same greedy continuation as long as the argmax margin is unambiguous; logits of every compared step within tolerance
    for i in range(len(t_full)):
        assert (a_kv[i] - a_full[i]).abs().max().item() <= LOGIT_TOL, i
        top = torch.topk(a_full[i], 2).values
        if float(top[0] - top[1]) <= 4 * LOGIT_TOL:
            break
        assert t_kv[i] == t_full[i], i


@pytest.mark.parametrize("graphs", [False, True])
def test_staged_batches_give_the_same_step(graphs):
    """GatoPolicy.stage(): planning + upload ahead of time, forward(handle) later -- same loss / logits / gradients as
    forward(batch); a handle is single-use."""
    cfg = O.GatoConfig(**SMALL_CASES["mixed"]["cfg"])
    w = O.make_weights(cfg, seed=3)
    m = make_policy(cfg, w, train=False)
    m.use_cuda_graphs = graphs
    batch = small_batch("mixed", cfg.text_tokens)
    for _ in range(3 if graphs else 1):
        m.zero_grad()
        logits0, loss0 = m(batch, compute_loss=True)
        loss0.backward()
        g0 = m._grad_arena.clone()
        l0 = logits0.clone()
    nxt = m.stage(batch, compute_loss=True)
    for _ in range(3):
        cur = nxt
        m.zero_grad()
        logits1, loss1 = m(cur, compute_loss=True)
        loss1.backward()
        nxt = m.stage(batch, compute_loss=True)     # next step staged before this step's loss is read
        assert abs(loss1.item() - loss0.item()) <= 1e-6 * abs(loss0.item())
        assert torch.equal(logits1, l0)
        assert (m._grad_arena - g0).abs().max().item() <= 1e-6 * max(1.0, g0.abs().max().item())
    with pytest.raises(RuntimeError):
        m(cur, compute_loss=True)                   # already consumed
    _, loss = m(nxt, compute_loss=True)
    with pytest.raises(RuntimeError):
        m.stage(batch)                              # would overwrite what the pending backward still reads
    loss.backward()
    m.stage(batch)
    with pytest.raises(RuntimeError):
        m.stage(batch)                              # one outstanding handle at a time


@pytest.mark.parametrize("graphs", [False, True])
def test_staged_batch_survives_other_forwards(graphs):
    """stage(A); then an evaluation forward / tokenize_input_dicts / predict_* on OTHER batches (what the reference loop does
    every log_eval_freq steps) reuses the single staging buffer; forward(handleA) must still run batch A."""
    cfg = O.GatoConfig(**SMALL_CASES["mixed"]["cfg"])
    w = O.make_weights(cfg, seed=3)
    m = make_policy(cfg, w, train=False)
    m.use_cuda_graphs = graphs
    A = small_batch("mixed", cfg.text_tokens)
    other = [dict(text=list(range(1, 40))), dict(continuous_obs=torch.randn(9, 4), continuous_actions=torch.rand(9, 2))]
    for _ in range(3 if graphs else 1):
        m.zero_grad()
        logits0, loss0 = m(A, compute_loss=True)
        loss0.backward()
        g0, l0 = m._grad_arena.clone(), logits0.clone()
    for k in range(3):
        h = m.stage(A, compute_loss=True)
        with torch.no_grad():
            m(other, compute_loss=True)
            m.tokenize_input_dicts(other[:1])
            if k == 2:
                m.predict_text({"text": [3, 4, 5]}, max_length=2)
        m.zero_grad()
        logits1, loss1 = m(h, compute_loss=True)
        loss1.backward()
        assert abs(loss1.item() - loss0.item()) <= 1e-6 * abs(loss0.item())
        assert torch.equal(logits1, l0)
        assert (m._grad_arena - g0).abs().max().item() <= 1e-6 * max(1.0, g0.abs().max().item())


@pytest.mark.parametrize("seed", range(8))
def test_tokenize_random_mixed_batches_bit_exact(seed):
    """Random mixtures of every modality through the fused tokenise / embed / interleave / pad kernel: ids and both masks
    bit-exact against the oracle, embeddings exact off the patch rows (those go through the 16-bit patch projection)."""
    from _random_batches import random_mixed_batch
    batch, ctx, pad_seq = random_mixed_batch(seed)
    cfg = O.GatoConfig(embed_dim=32, layers=1, heads=1, context_len=ctx, text_tokens=300, pad_seq=pad_seq)
    w = O.make_weights(cfg, seed=seed)
    m = make_policy(cfg, w)
    emb, tok, tm, mk = m.tokenize_input_dicts(batch)
    tb = O.tokenize(batch, cfg)
    assert np.array_equal(tok.cpu().numpy(), tb.tokens)
    assert np.array_equal(tm.cpu().numpy(), tb.target_masks.astype(np.float32))
    assert np.array_equal(mk.cpu().numpy(), tb.token_masks.astype(np.float32))
    ref = O.embed_and_interleave(batch, tb, w, cfg)
    err = (emb.cpu() - ref).abs()
    W = tb.tokens.shape[1]
    S = int(max(st.ids.shape[0] for st in tb.samples))
    is_patch = torch.zeros(tb.tokens.shape, dtype=torch.bool)
    for b, st in enumerate(tb.samples):
        if st.n_patches:
            n = st.ids.shape[0]
            pat = np.zeros(st.tokens_per_timestep, bool)
            pat[:st.n_patches] = True
            is_patch[b, S - n:S] = torch.from_numpy(np.tile(pat, st.n_timesteps))
    assert float(err[~is_patch].max()) <= 1e-6
    if is_patch.any():
        assert float(err[is_patch].max()) <= 3e-2
    assert W == (ctx if pad_seq and ctx > S else S)


def test_kv_cached_image_response_matches_full_recompute():
    """predict_answer / predict_caption through the KV cache against the reference-style loop (full context per token)."""
    cfg = O.GatoConfig(embed_dim=64, layers=2, heads=2, context_len=64, text_tokens=200)
    w = O.make_weights(cfg, seed=23)
    m = make_policy(cfg, w)

    class _Txt(_Tok):
        def decode(self, ids):
            return " ".join(str(i) for i in ids)

        def encode(self, s):
            return [int(t) for t in s.split()]

    m.text_tokenizer = _Txt(cfg.text_tokens)
    rs = np.random.RandomState(12)
    img = torch.from_numpy(rs.randint(0, 256, (1, 3, 32, 48)).astype(np.uint8))
    for question, n_new in (("5 7 11 13", 6), ("", 5)):
        outs = []
        for use_kv in (True, False):
            m.use_kv_cache = use_kv
            if question:
                logits, text = m.predict_answer(img, question, max_length=n_new, deterministic=True)
            else:
                logits, text = m.predict_caption(img, max_length=n_new, deterministic=True)
            outs.append((logits.float().cpu(), [int(t) for t in text.split()]))
        (l_kv, t_kv), (l_full, t_full) = outs
        assert tuple(l_kv.shape) == tuple(l_full.shape) == (n_new, cfg.text_tokens)
        for i in range(n_new):
            assert (l_kv[i] - l_full[i]).abs().max().item() <= LOGIT_TOL, (question, i)
            top = torch.topk(l_full[i], 2).values
            if float(top[0] - top[1]) <= 4 * LOGIT_TOL:
                break
            assert t_kv[i] == t_full[i], (question, i)


def test_bench_dump_outputs(tmp_path):
    """bench.py --dump-outputs, run twice with the same arguments: float arrays only, 64 MB at most, loss and logits bit for bit
    the same (gradients summed with fp32 atomics may round differently), and the line reports the --steps it was given."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    runs = []
    for k in range(2):
        d = tmp_path / str(k)
        out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--only", "--steps", "2", "--no-cpu-baseline", "--no-front-end",
                              "--dump-outputs", str(d)], capture_output=True, text=True, timeout=900, cwd=root)
        assert out.returncode == 0, out.stderr[-3000:]
        line = json.loads([ln for ln in out.stdout.splitlines() if ln.startswith("{")][-1])
        assert line["steps"] == 2 and line["value"] > 0
        runs.append({f[:-4]: np.load(d / f) for f in os.listdir(d) if f.endswith(".npy")})
    a, b = runs
    assert len(os.listdir(tmp_path / "0")) == len(a) and set(a) == set(b)
    assert {"loss", "logits"} < set(a) and any(k.startswith("grad.") for k in a)
    assert all(v.dtype in (np.float32, np.float64) for v in a.values())
    assert sum(v.nbytes for v in a.values()) <= 64 << 20
    assert np.array_equal(a["loss"], b["loss"]) and np.array_equal(a["logits"], b["logits"])
    assert np.isfinite(a["logits"]).all()
    for k in a:
        assert a[k].shape == b[k].shape, k

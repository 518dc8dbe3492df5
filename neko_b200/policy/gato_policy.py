"""GatoPolicy -- drop-in for gato/policy/gato_policy.py:18 (GatoPolicy) on B200.

Same constructor, attributes, ``state_dict`` key layout, ``forward`` / ``tokenize_input_dicts``
signatures and return dtypes as the reference; everything underneath runs through the C ABI of
``include/neko_b200.h`` (hand-written sm_100a kernels).  There is no CPU path: constructing the policy
on a non-CUDA device, or without ``libneko_b200.so``, raises.

Design (see DESIGN.md):
  * parameters live in ONE flat fp32 arena, gradients in a second one with the same layout (reverse
    execution order, so data-parallel buckets complete front to back during backward); every
    ``nn.Parameter`` / ``.grad`` is a view.  One kernel casts the arena to the bf16 operand copy.
  * ``forward(inputs, compute_loss=True)`` is a single autograd node: the host plans the batch
    (``packing.build_plan``), one H2D copy moves it, then ~14 kernel launches per layer run forward;
    ``loss.backward()`` runs the hand-written backward and writes straight into the gradient arena.
"""
from __future__ import annotations

import ctypes as C
import gc
import math
import weakref
from typing import Dict, List, Optional, Union

import numpy as np
import torch
import torch.nn as nn

from .. import _lib, ops
from .._lib import Dropout, TokParams, _p, check, load, stream_ptr
from .embeddings import ImageEmbedding, _AffineParams, _EmbeddingParams, _LinearParams
from .input_tokenizers import ContinuousTokenizer
from .packing import BatchPlan, Stager, build_plan


def _pad_to(n: int, m: int) -> int:
    return (n + m - 1) // m * m


def _before_capture():
    """Run before every CUDA-graph capture.  A dropped graph entry (workspace epoch change, cache eviction, a policy that went
    out of scope) keeps its CUDAGraph alive in a reference cycle (entry <-> captured state) until the cyclic collector runs;
    if that happens in the middle of a capture, destroying the graph there invalidates the capture.  torch no longer collects
    before a capture, so collect here, then drain the device."""
    gc.collect()
    torch.cuda.synchronize()


# --------------------------------------------------------------------------------------------------
# parameter containers with the reference's module tree (trajectory_gpt2.py:120-359, 535-550)
# --------------------------------------------------------------------------------------------------


class _Conv1D(nn.Module):
    """HF Conv1D: weight [in, out], y = x @ W + b; N(0, 0.02) / zeros (trajectory_gpt2.py:375-386)."""

    def __init__(self, nf: int, nx: int):
        super().__init__()
        self.nf = nf
        self.weight = nn.Parameter(torch.empty(nx, nf))
        self.bias = nn.Parameter(torch.zeros(nf))
        nn.init.normal_(self.weight, std=0.02)


class _Attention(nn.Module):
    def __init__(self, nx: int, n_ctx: int, attn_pdrop: float = 0.0, resid_pdrop: float = 0.0):
        super().__init__()
        # buffers kept for state_dict compatibility (trajectory_gpt2.py:127-130); the kernels derive the
        # causal structure arithmetically
        self.register_buffer("bias", torch.tril(torch.ones((n_ctx, n_ctx), dtype=torch.uint8)).view(1, 1, n_ctx, n_ctx))
        self.register_buffer("masked_bias", torch.tensor(-1e4))
        self.c_attn = _Conv1D(3 * nx, nx)
        self.c_proj = _Conv1D(nx, nx)
        self.attn_dropout = nn.Dropout(attn_pdrop)      # trajectory_gpt2.py:142-143 (p read by the kernels)
        self.resid_dropout = nn.Dropout(resid_pdrop)


class _MLP(nn.Module):
    def __init__(self, n_state: int, nx: int, gate: bool, resid_pdrop: float = 0.0):
        super().__init__()
        self.c_fc = _Conv1D(n_state, nx)
        self.c_proj = _Conv1D(nx, n_state)
        self.dropout = nn.Dropout(resid_pdrop)          # trajectory_gpt2.py:271,278
        if gate:
            self.gated_layer = _LinearParams(nx, n_state)
            nn.init.normal_(self.gated_layer.weight, std=0.02)
            nn.init.zeros_(self.gated_layer.bias)
        else:
            self.gated_layer = None


class _Block(nn.Module):
    def __init__(self, nx: int, n_ctx: int, gate: bool, attn_pdrop: float = 0.0, resid_pdrop: float = 0.0):
        super().__init__()
        self.ln_1 = _AffineParams(nx)
        self.attn = _Attention(nx, n_ctx, attn_pdrop, resid_pdrop)
        self.ln_2 = _AffineParams(nx)
        self.mlp = _MLP(4 * nx, nx, gate, resid_pdrop)


class _GPT2Config:
    def __init__(self, **kw):
        self.__dict__.update(kw)


class GPT2Model(nn.Module):
    """Container for the decoder parameters (gato/transformers/trajectory_gpt2.py:535-550)."""

    def __init__(self, config: _GPT2Config):
        super().__init__()
        self.config = config
        self.wte = _EmbeddingParams(config.vocab_size, config.n_embd, std=0.02)  # never used (wpe/wte removed, :540,698-701)
        self.drop = nn.Dropout(config.embd_pdrop)
        self.h = nn.ModuleList([_Block(config.n_embd, config.n_ctx, config.gate, config.attn_pdrop, config.resid_pdrop)
                                for _ in range(config.n_layer)])
        self.ln_f = _AffineParams(config.n_embd)

    def forward(self, inputs_embeds=None, attention_mask=None, **kw):
        owner = getattr(self, "_owner", None)
        if owner is None:
            raise RuntimeError("GPT2Model must be owned by a GatoPolicy")
        return {"last_hidden_state": owner()._decode_embeddings(inputs_embeds, attention_mask)}


class _OfflineTextTokenizer:
    """Stand-in when the GPT-2 BPE tables cannot be loaded (no hub access): the hot path only reads
    ``vocab_size`` (gato_policy.py:57-60)."""

    vocab_size = 50257

    def encode(self, *_a, **_k):
        raise RuntimeError("GPT-2 tokenizer files are not available offline")

    decode = encode


def _load_pretrained_gpt2(path: str):
    """--pretrained_lm (gato_policy.py:79-95): configuration + tensors of a HF GPT-2 checkpoint directory (config.json +
    model.safetensors / pytorch_model.bin).  A hub name is resolved from the local HF cache only (there may be no network)."""
    import json
    import os
    if not os.path.isdir(path):
        try:
            from huggingface_hub import snapshot_download
            path = snapshot_download(path, local_files_only=True)
        except Exception as e:  # noqa: BLE001
            raise FileNotFoundError(f"--pretrained_lm={path!r}: not a local checkpoint directory and not in the local Hugging Face cache "
                                    f"({type(e).__name__}); download it first or pass the directory") from e
    with open(os.path.join(path, "config.json")) as f:
        cfg = json.load(f)
    st = os.path.join(path, "model.safetensors")
    if os.path.exists(st):
        from safetensors.torch import load_file
        sd = load_file(st)
    else:
        sd = torch.load(os.path.join(path, "pytorch_model.bin"), map_location="cpu", weights_only=True)
    sd = {(n[len("transformer."):] if n.startswith("transformer.") else n): t for n, t in sd.items()}
    return cfg, sd


def _load_text_tokenizer(name: str):
    try:
        from transformers import AutoTokenizer
        return AutoTokenizer.from_pretrained(name)
    except Exception:  # noqa: BLE001 - offline / missing files
        return _OfflineTextTokenizer()


# --------------------------------------------------------------------------------------------------
# one fused autograd node for forward(inputs, ...)
# --------------------------------------------------------------------------------------------------
class _FusedStep(torch.autograd.Function):
    @staticmethod
    def forward(ctx, policy, state, *params):
        logits, loss = policy._engine_forward(state)
        policy._bwd_pending = state.compute_loss
        ctx.policy = policy
        ctx.state = state
        ctx.n_params = len(params)
        ctx.set_materialize_grads(False)  # never let autograd zero-fill a [B,S,V] gradient for the logits output
        ctx.mark_non_differentiable(logits)
        if loss is None:
            loss = torch.zeros((), device=logits.device)
            ctx.mark_non_differentiable(loss)
        return logits, loss

    @staticmethod
    def backward(ctx, _g_logits, g_loss):
        if g_loss is None:
            return (None, None) + (None,) * ctx.n_params
        ctx.policy._bwd_pending = False
        ctx.policy._engine_backward(ctx.state, g_loss)
        # gradients were written straight into the flat arena behind every parameter's .grad
        return (None, None) + (None,) * ctx.n_params


class _State:
    """Everything one forward hands to its backward."""
    pass


class _KVCache:
    """Keys / values of one sequence for the KV-cached predict_* loops: bf16 [layers, context_len, d] each."""

    def __init__(self, layers: int, ctx: int, d: int, device):
        self.k = torch.empty(layers, ctx, d, dtype=torch.bfloat16, device=device)
        self.v = torch.empty(layers, ctx, d, dtype=torch.bfloat16, device=device)
        self.len = 0            # positions held
        self.decoding = False   # False: prefill (fill from a full forward); True: one new position per call


class GatoPolicy(nn.Module):
    def __init__(
        self,
        device: Union[torch.device, str],
        embed_dim: int,
        layers: int,
        heads: int,
        dropout: float,
        activation_fn="gelu",
        mu: int = 100,
        M: int = 256,
        patch_size: int = 16,
        resid_mid_channels: int = 132,
        num_groups: int = 32,
        position_vocab_size: int = 128,
        continuous_tokens: int = 1024,
        discrete_tokens: int = 1024,
        context_len=1024,
        use_pos_encoding: bool = True,
        use_patch_pos_encoding: bool = True,
        pretrained_lm: Optional[str] = None,
        flash: bool = False,
        tokenizer_model_name: str = "gpt2",
        pad_seq: bool = False,
        text_tokenizer=None,
    ):
        super().__init__()
        dev = torch.device(device)
        if dev.type != "cuda":
            raise _lib.NekoError("neko_b200.GatoPolicy runs on CUDA (sm_100) only; there is no CPU fallback")
        if dev.index is None:
            dev = torch.device("cuda", torch.cuda.current_device())
        self.device = dev
        with torch.cuda.device(dev):
            _lib.require_device()
        lm_cfg = lm_sd = None
        if pretrained_lm is not None:
            # gato_policy.py:79-95: the decoder's shape, activation and weights come from the GPT-2 checkpoint; embed_dim /
            # layers / heads / activation_fn arguments are overridden, exactly as in the reference
            print("loading pretrained GPT2 weights")
            lm_cfg, lm_sd = _load_pretrained_gpt2(pretrained_lm)
            embed_dim, heads, layers = int(lm_cfg["n_embd"]), int(lm_cfg["n_head"]), int(lm_cfg["n_layer"])
            activation_fn = lm_cfg.get("activation_function", "gelu_new")
        assert embed_dim % heads == 0
        if (embed_dim // heads) not in (16, 32, 64, 128):
            raise NotImplementedError(f"head dim {embed_dim // heads} not supported (16/32/64/128)")
        self.context_len = context_len
        self.pad_seq = pad_seq
        self.text_tokenizer = text_tokenizer if text_tokenizer is not None else _load_text_tokenizer(tokenizer_model_name)
        self.text_tokens = self.text_tokenizer.vocab_size
        self.continuous_tokens = continuous_tokens
        self.discrete_tokens = discrete_tokens
        self.vocab_size = self.text_tokens + self.discrete_tokens + self.continuous_tokens
        self.token_starts = {"text": 0, "continuous": self.text_tokens, "discrete": self.text_tokens + self.continuous_tokens}
        self.token_ends = {"text": self.text_tokens - 1, "continuous": self.text_tokens + self.continuous_tokens - 1,
                           "discrete": self.text_tokens + self.continuous_tokens + self.discrete_tokens - 1}
        gate = False
        if activation_fn == "geglu" and lm_cfg is None:
            gate = True
            activation_fn = "gelu"
        if activation_fn not in ("gelu", "gelu_new"):
            raise NotImplementedError(f"activation_fn={activation_fn!r}: 'gelu' (erf), 'geglu' (reference CLI) and 'gelu_new' (tanh form of "
                                      "pretrained GPT-2 checkpoints) are implemented")
        self._gelu_tanh = activation_fn == "gelu_new"      # GELU / GELU' GEMM epilogues: tanh form
        self.heads = heads
        self.layers = layers
        self.dropout = dropout
        self.mu, self.M = mu, M
        self.patch_size = patch_size
        if lm_cfg is None:
            config = _GPT2Config(vocab_size=1, n_embd=embed_dim, n_head=heads, n_layer=layers, resid_pdrop=dropout,
                                 attn_pdrop=dropout, embd_pdrop=0.1, n_positions=context_len, n_ctx=context_len,
                                 n_inner=embed_dim * 4, activation_function=activation_fn, flash=flash, gate=gate,
                                 layer_norm_epsilon=1e-5)
        else:
            if lm_cfg.get("n_inner") not in (None, 4 * embed_dim):
                raise NotImplementedError("pretrained GPT-2 with n_inner != 4 * n_embd")
            n_ctx = int(lm_cfg.get("n_ctx", lm_cfg.get("n_positions", 1024)))
            config = _GPT2Config(vocab_size=int(lm_cfg["vocab_size"]), n_embd=embed_dim, n_head=heads, n_layer=layers, resid_pdrop=dropout,
                                 attn_pdrop=dropout, embd_pdrop=float(lm_cfg.get("embd_pdrop", 0.1)), n_positions=int(lm_cfg.get("n_positions", n_ctx)),
                                 n_ctx=n_ctx, n_inner=embed_dim * 4, activation_function=activation_fn, flash=flash, gate=False,
                                 layer_norm_epsilon=float(lm_cfg.get("layer_norm_epsilon", 1e-5)))
        with torch.device(dev):
            self.transformer = GPT2Model(config)
            self.embed_token = _EmbeddingParams(self.vocab_size, embed_dim)
            self.embed_dim = embed_dim
            self.predict_token = _LinearParams(embed_dim, self.vocab_size, bias=False)
            self.separator_token = nn.Parameter(torch.zeros(embed_dim))
            self.continuous_action_tokenizer = ContinuousTokenizer(use_mu_law=False, mu=mu, M=M, n_bins=self.continuous_tokens,
                                                                   offset=self.token_starts["continuous"])
            self.continuous_obs_tokenizer = ContinuousTokenizer(use_mu_law=True, mu=mu, M=M, n_bins=self.continuous_tokens,
                                                                offset=self.token_starts["continuous"])
            self.use_patch_pos_encoding = use_patch_pos_encoding
            self.image_embedding = ImageEmbedding(embed_dim=embed_dim, patch_size=patch_size, resid_mid_channels=resid_mid_channels,
                                                  num_groups=num_groups, position_vocab_size=position_vocab_size,
                                                  use_pos_encoding=use_patch_pos_encoding)
            self.use_pos_encoding = use_pos_encoding
            self.pos_embed_observation = _EmbeddingParams(context_len, embed_dim)
        if lm_sd is not None:
            own = dict(self.transformer.named_parameters())
            assert tuple(lm_sd["wte.weight"].shape) == (self.text_tokens, embed_dim), "pretrained token/expected mimsatch"
            missing = [n for n in own if n not in lm_sd]
            if missing:
                raise KeyError(f"--pretrained_lm checkpoint lacks {missing[:4]} ...")
            with torch.no_grad():
                for n, p in own.items():          # wpe (no absolute positions here, trajectory_gpt2.py:540) and attn.bias are not taken
                    p.copy_(lm_sd[n].to(dev, torch.float32).reshape(p.shape))
                # expand the embedding dictionary up to vocab_size: the text rows start from the LM's table (gato_policy.py:91-93)
                self.embed_token.weight[:self.text_tokens] = self.transformer.wte.weight
        ref = weakref.ref(self)
        object.__setattr__(self.transformer, "_owner", ref)
        object.__setattr__(self.image_embedding, "_owner", ref)
        # engine knobs
        # head backward: 'rows' runs the LM-head weight / input gradients on the loss rows only (the other rows of dlogits
        # are exactly zero); 'dense' runs them over every position like the reference's autograd.  Identical gradients.
        self.head_mode = "rows"
        self.materialize_logits = True  # False: head evaluated on loss rows only, forward returns logits=None
        # pack_sequences (needs materialize_logits = False): forward(inputs, compute_loss=True) and stage() lay the samples out
        # back to back with no padding rows, so every row-proportional kernel runs on the valid tokens only (variable-length
        # attention).  Same loss and gradients up to reassociation; pad_seq has no effect on them (right padding is causally
        # invisible to valid rows).  Opt-in: the embedding / residual dropout masks are drawn at packed row coordinates, a
        # different random stream from the padded layout's (the attention-dropout masks are the same).
        self.pack_sequences = False
        # deterministic: every floating-point reduction of a training step runs in a fixed order that depends on the inputs and
        # shapes only (ordered column sums, sorted embedding scatter, chunked patch backward, GEMMs without split-K / stream-K,
        # ordered gradient norm), so two runs with the same seed give the same bits whatever the grid, SM count or timing
        # (DESIGN.md "Deterministic training mode").  Differs from the default mode by reassociation only.
        self.deterministic = False
        self.lean_logits_f16 = True     # ... and, when gradients are wanted, those logits live in fp16 between head GEMM and fused CE
        self.mlp_proj_bf16 = False      # training forward: mlp down-projection on the bf16 activation twin (see _decoder)
        # 16-bit format of the FORWARD operands (activations fed to GEMMs, weight copy).  fp16 has 3 more mantissa
        # bits than bf16 at the same tensor-core rate and brings logits max-abs error from 2.1e-2 to ~6e-3 at
        # d=768/L=6 (DESIGN.md "precision"); gradients stay bf16 for range, the residual stream stays fp32.
        self.fwd_dtype = torch.float16
        self._Vp = _pad_to(self.vocab_size, 64)
        self._ws: Dict[str, torch.Tensor] = {}
        self._stager = Stager(dev)
        self._generation = 0
        self._bf16_versions = None
        self._grad_live = False
        self.grad_ready_hook = None     # callable(lo, hi): arena range [lo, hi) is final (data-parallel buckets)
        self.use_cuda_graphs = False    # replay fwd / bwd from CUDA graphs keyed by the batch plan (see _engine_forward)
        self._graphs = {}
        self.max_cuda_graphs = 6
        self._graph_pool = None
        self._gscale_buf = torch.ones((), dtype=torch.float32, device=dev)
        self.launches = 0
        self._drop_gen = None
        self._bwd_pending = False       # a differentiable forward has not seen its backward yet (guards stage())
        self._copy_stream = None        # stage(): frames travel on their own stream
        self._staged_handle = None
        self._img_in_free = None
        self.use_kv_cache = True        # predict_* loops: key/value cache instead of re-running the context per token
        self._build_arena()

    # ------------------------------------------------------------------------------------------
    @property
    def module(self):
        return self

    # ------------------------------------------------------------------------------------------
    # flat parameter / gradient arenas
    # ------------------------------------------------------------------------------------------
    def _arena_order(self) -> List[str]:
        names = ["predict_token.weight", "transformer.ln_f.weight", "transformer.ln_f.bias"]
        for i in reversed(range(self.layers)):
            p = f"transformer.h.{i}."
            # the four weight matrices first (fully overwritten by their wgrad GEMM), then the small vectors
            # (accumulated with atomics: they need zeroing, and are contiguous so one memset per layer does it)
            names += [p + "mlp.c_proj.weight", p + "mlp.c_fc.weight", p + "attn.c_proj.weight", p + "attn.c_attn.weight"]
            if self.transformer.config.gate:
                names += [p + "mlp.gated_layer.weight", p + "mlp.gated_layer.bias"]
            names += [p + "mlp.c_proj.bias", p + "mlp.c_fc.bias", p + "ln_2.weight", p + "ln_2.bias",
                      p + "attn.c_proj.bias", p + "attn.c_attn.bias", p + "ln_1.weight", p + "ln_1.bias"]
        names += [n for n, _ in self.named_parameters() if n.startswith("image_embedding.")]
        names += ["pos_embed_observation.weight", "separator_token", "embed_token.weight", "transformer.wte.weight"]
        return names

    def _build_arena(self):
        params = dict(self.named_parameters())
        order = self._arena_order()
        assert set(order) == set(params), set(params) ^ set(order)
        offs, total = {}, 0
        for n in order:
            offs[n] = total
            numel = params[n].numel()
            if n == "predict_token.weight":  # zero rows up to the padded vocabulary: TMA reads them
                numel = self._Vp * self.embed_dim
            total += _pad_to(numel, 64)
        arena = torch.zeros(total, dtype=torch.float32, device=self.device)
        for n in order:
            p = params[n]
            view = arena[offs[n]:offs[n] + p.numel()].view(p.shape)
            view.copy_(p.data)
            p.data = view
        self._param_arena = arena
        self._grad_arena = torch.zeros(total, dtype=torch.float32, device=self.device)
        # 16-bit operand copies of the GEMM weights: forward format + bf16 for dgrad (tcgen05 cannot mix formats);
        # the embedding tables at the tail of the arena are only ever gathered in fp32 and are not copied
        self._cast_end = offs["pos_embed_observation.weight"]
        self._w16_arena = torch.zeros(self._cast_end, dtype=self.fwd_dtype, device=self.device)
        self._wbf_arena = (self._w16_arena if self.fwd_dtype == torch.bfloat16
                           else torch.zeros(self._cast_end, dtype=torch.bfloat16, device=self.device))
        self._offs = offs
        self._order = order
        self._params = params
        self._gview_cache = {}
        self._wview_cache = {}
        self._grad_pairs_cache = {}
        # gradient ranges that must start from zero each step (everything except the matrices a single non-split
        # or self-zeroing wgrad GEMM overwrites)
        overwritten = {"predict_token.weight"} | {f"transformer.h.{i}.{m}.weight" for i in range(self.layers)
                                                  for m in ("mlp.c_proj", "mlp.c_fc", "attn.c_proj", "attn.c_attn")}
        ranges, cur = [], None
        for k, n in enumerate(order):
            end = offs[order[k + 1]] if k + 1 < len(order) else total
            if n in overwritten:
                if cur is not None:
                    ranges.append(tuple(cur))
                    cur = None
            else:
                cur = [offs[n], end] if cur is None else [cur[0], end]
        if cur is not None:
            ranges.append(tuple(cur))
        self._zero_ranges = ranges
        self._bf16_versions = None
        self._grad_live = False

    def _check_arena(self):
        """Parameters must still be views of the arena (a ``.to()`` / ``.half()`` would replace them)."""
        base = self._param_arena.data_ptr()
        for n in ("predict_token.weight", "transformer.wte.weight"):
            if self._params[n].data_ptr() != base + 4 * self._offs[n] or self._params[n].dtype != torch.float32:
                self._build_arena()
                break

    def _gview(self, name: str) -> torch.Tensor:
        """Gradient of a parameter as a view of the gradient arena (cached: the host path creates ~100 of them per step)."""
        v = self._gview_cache.get(name)
        if v is None or v.data_ptr() != self._grad_arena.data_ptr() + 4 * self._offs[name]:
            p = self._params[name]
            o = self._offs[name]
            v = self._grad_arena[o:o + p.numel()].view(p.shape)
            self._gview_cache[name] = v
        return v

    def _wview(self, name: str, rows: Optional[int] = None, bwd: bool = False) -> torch.Tensor:
        """16-bit operand copy of a weight: forward format, or bf16 for the backward GEMMs (views are cached)."""
        arena = self._wbf_arena if bwd else self._w16_arena
        key = (name, rows, bwd)
        hit = self._wview_cache.get(key)
        if hit is not None and hit[0] is arena:
            return hit[1]
        p = self._params[name]
        o = self._offs[name]
        if rows is not None:
            v = arena[o:o + rows * p.shape[1]].view(rows, p.shape[1])
        else:
            v = arena[o:o + p.numel()].view(p.shape)
        self._wview_cache[key] = (arena, v)
        return v

    def _refresh_bf16(self, force: bool = False):
        vers = None if force else tuple(p._version for p in self._params.values())
        if self._w16_arena.dtype != self.fwd_dtype:
            self._w16_arena = torch.zeros(self._cast_end, dtype=self.fwd_dtype, device=self.device)
            self._wbf_arena = (self._w16_arena if self.fwd_dtype == torch.bfloat16
                               else torch.zeros(self._cast_end, dtype=torch.bfloat16, device=self.device))
            self._bf16_versions = None
        if force or vers != self._bf16_versions:
            src = self._param_arena[:self._cast_end]
            if self.fwd_dtype == torch.float16:
                ops.cast_dual(src, self._w16_arena, self._wbf_arena)
            else:
                ops.cast_bf16(src, self._w16_arena)
            self.launches += 1
            self._bf16_versions = vers

    def zero_grad(self, set_to_none: bool = True):
        # nn.Module.zero_grad walks the module tree (named_modules / named_members, ~0.2 ms here); every parameter of this
        # policy is in the arena table, so iterate that
        if set_to_none:
            for p in self._params.values():
                p.grad = None
        else:
            for p in self._params.values():
                if p.grad is not None:
                    p.grad.detach_()
                    p.grad.zero_()
        self._grad_live = False

    def _begin_grads(self, has_images: bool, zero: bool = True):
        """Start (or continue) a gradient-accumulation cycle; returns True when accumulating.  Parameters that
        take no part in the step keep ``grad is None`` exactly like the reference's autograd (transformer.wte
        always; the image stack when the batch has no images; SURVEY.md section 8(a) a15)."""
        live = self._grad_live
        if live:
            for n in ("predict_token.weight", "embed_token.weight"):
                g = self._params[n].grad
                if g is None or g.data_ptr() != self._grad_arena.data_ptr() + 4 * self._offs[n]:
                    live = False
        if not live:
            if zero:
                for lo, hi in self._zero_ranges:
                    self._grad_arena[lo:hi].zero_()
            for n, p in self._params.items():
                p.grad = None
        pairs = self._grad_pairs_cache.get(has_images)
        if pairs is None or pairs[0][1].data_ptr() != self._grad_arena.data_ptr() + 4 * self._offs[pairs[0][2]]:
            pairs = []
            for n, p in self._params.items():
                if n == "transformer.wte.weight":
                    continue
                if n.startswith("image_embedding."):
                    if not has_images or (".patch_pos_encoding." in n and not self.use_patch_pos_encoding):
                        continue
                if n == "pos_embed_observation.weight" and not self.use_pos_encoding:
                    continue
                pairs.append((p, self._gview(n), n))
            self._grad_pairs_cache[has_images] = pairs
        for p, v, _n in pairs:
            if p.grad is None:
                p.grad = v
        self._grad_live = True
        return live

    # ------------------------------------------------------------------------------------------
    # workspace
    # ------------------------------------------------------------------------------------------
    def _buf(self, name: str, shape, dtype) -> torch.Tensor:
        n = 1
        for s in shape:
            n *= int(s)
        t = self._ws.get(name)
        if t is None or t.dtype != dtype or t.numel() < n:
            if getattr(self, "_capturing", False):
                raise RuntimeError(f"workspace buffer {name!r} would be (re)allocated during CUDA-graph capture")
            t = torch.empty(max(n, 1), dtype=dtype, device=self.device)
            self._ws[name] = t
            self._ws_epoch = getattr(self, "_ws_epoch", 0) + 1   # captured graphs hold raw pointers: invalidate them
        return t[:n].view(*shape)

    # -- deterministic mode: the ordered twins of the reducing kernels --------------------------------
    def _ordered_ws(self, nbytes: int) -> torch.Tensor:
        """Scratch of the ordered reductions: one buffer for all of them (they run in stream order).  The eager first sight
        of a plan grows it to the step's largest need, so captured graphs see one stable pointer."""
        return self._buf("ordered_ws", (max(int(nbytes), 256),), torch.uint8)

    def _gemm(self, *args, **kw):
        return ops.gemm(*args, deterministic=self.deterministic, **kw)

    def _ln_bwd(self, dy, x, gamma, mean, rstd, dx, dgamma, dbeta, dxb, dx_colsum=None, branch_drop=None):
        if self.deterministic:
            ws = self._ordered_ws(ops.layernorm_bwd_ordered_workspace_bytes(*x.shape))
            ops.layernorm_bwd_ordered(dy, x, gamma, mean, rstd, dx, dgamma, dbeta, ws, dx_bf16=dxb, dx_colsum=dx_colsum,
                                      branch_drop=branch_drop)
        else:
            ops.layernorm_bwd(dy, x, gamma, mean, rstd, dx, dgamma, dbeta, dxb, dx_colsum=dx_colsum, branch_drop=branch_drop)

    def _colsum(self, x_bf16, out):
        """out += column sums of x_bf16 (bias gradients)."""
        if self.deterministic:
            ops.colsum_ordered(x_bf16, out, self._ordered_ws(ops.colsum_ordered_workspace_bytes(*x_bf16.shape)), accumulate=True)
        else:
            ops.colsum(x_bf16, out, accumulate=True)

    # ------------------------------------------------------------------------------------------
    # public API
    # ------------------------------------------------------------------------------------------
    def stage(self, inputs: list, compute_loss: bool = True):
        """Batch producer hook (SURVEY 8(f)3): do the host half of a step ahead of time -- plan the batch (descriptors, loss
        rows, train-mode patch bins, dropout seed) and enqueue its single pinned -> device copy -- and return a handle that
        ``forward(handle)`` consumes.  Call it for step i+1 right after enqueueing step i's backward and before reading step
        i's loss: the planning then overlaps the GPU work of step i.  The copy is ordered on the compute stream, so the
        staging buffer is never overwritten under a step that is still reading it; at most ONE staged handle may be
        outstanding."""
        self._check_arena()
        if self._bwd_pending:
            raise RuntimeError("stage() while a forward is waiting for its backward: the staging buffer still holds that step's "
                               "descriptors and loss rows -- call loss.backward() first (or run the forward under torch.no_grad())")
        if self._staged_handle is not None and getattr(self._staged_handle, "staged", False):
            raise RuntimeError("stage(): the previously staged batch has not been consumed by forward() yet")
        self._check_packing(compute_loss)
        st = self._plan(inputs, compute_loss)
        st.staged = True
        self._image_prefetch(st)
        self._staged_handle = st
        return st

    def _image_prefetch(self, st: _State):
        """stage(): host-resident frames start their H2D copy right away on a copy stream, into 'incoming' buffers that no
        kernel reads; forward(handle) moves them device-to-device into the graph-stable frame buffers (46 MB in ~15 us at
        cfg3 instead of ~2 ms of PCIe time on the critical path)."""
        plan = st.plan
        st.img_in = {}
        if plan.n_patch_rows == 0 or not any(g.tensors and not g.tensors[0].is_cuda for g in plan.image_groups):
            return
        bufs = {}
        for gi, g in enumerate(plan.image_groups):
            if g.tensors and not g.tensors[0].is_cuda:
                n_el, dt = g.n_frames * 3 * g.height * g.width, (torch.uint8 if g.is_u8 else torch.float32)
                old = self._ws.get(f"img_in{gi}")
                if old is not None and (old.numel() < n_el or old.dtype != dt) and self._copy_stream is not None:
                    self._copy_stream.synchronize()    # the buffer is about to be replaced: no copy may still target it
                bufs[gi] = self._buf(f"img_in{gi}", (n_el,), dt)
        if self._copy_stream is None:
            self._copy_stream = torch.cuda.Stream(device=self.device)
        cs = self._copy_stream
        if self._img_in_free is not None:      # the previous staged step's device-to-device move must have read them out
            cs.wait_event(self._img_in_free)
        with torch.cuda.stream(cs):
            for gi, buf in bufs.items():
                o = 0
                for t in plan.image_groups[gi].tensors:
                    n = t.numel()
                    buf[o:o + n].view(t.shape).copy_(t, non_blocking=True)
                    st.h2d_bytes += n * t.element_size()
                    o += n
            st.img_ready = torch.cuda.Event()
            st.img_ready.record(cs)
        st.img_in = bufs

    def forward(self, inputs: Optional[list] = None, compute_loss=False, **kwargs):
        """gato_policy.py:156-192.  Returns (logits [B,S,V] fp32, loss or None).  ``inputs`` may also be a handle returned by
        ``stage()``."""
        self._check_arena()
        if inputs is not None:
            if isinstance(inputs, _State):
                state = inputs
                if not getattr(state, "staged", False):
                    raise RuntimeError("forward() was given a state object that did not come from stage() (or was already used)")
                state.staged = False
                state.compute_loss = bool(compute_loss)
                if state.stager_gen != self._stager.generation:
                    # another batch went through the (single, pointer-stable) staging buffer after stage(): an evaluation
                    # forward, tokenize_input_dicts, predict_*.  Upload the staged plan again -- same layout, same seed.
                    self._upload_plan(state, state.drop_seed_host)
            else:
                self._check_packing(compute_loss)
                self._bwd_pending = False     # a new direct forward supersedes an abandoned step
                state = self._plan(inputs, compute_loss)
            anchor = None
            if torch.is_grad_enabled():
                anchor = self._params["predict_token.weight"]
                if not anchor.requires_grad:
                    anchor = next((p for p in self._params.values() if p.requires_grad), None)
            need_grad = anchor is not None
            state.need_grad = need_grad
            if need_grad:
                # gradients are written straight into the arena behind every .grad, so the autograd node only needs ONE
                # differentiable input to exist (handing it all ~100 parameters costs ~0.1 ms of host time per step)
                logits, loss = _FusedStep.apply(self, state, anchor)
            else:
                logits, loss = self._engine_forward(state)
            if not compute_loss:
                loss = None
            return logits, loss
        assert "token_embeddings" in kwargs and "tokens" in kwargs and "token_target_masks" in kwargs and "token_masks" in kwargs, \
            "if inputs is None, must provide embeddings, tokens, and masks"
        emb, tokens = kwargs["token_embeddings"], kwargs["tokens"]
        tmask, mask = kwargs["token_target_masks"], kwargs["token_masks"]
        if emb.requires_grad and torch.is_grad_enabled():
            raise NotImplementedError("gradients through caller-supplied token_embeddings are not implemented; pass `inputs`")
        B, S, d = emb.shape
        with torch.no_grad():
            hf = self._decode_hidden(emb, mask)
            full = self._head(hf, B * S)
            logits = full.view(B, S, self._Vp)[:, :, :self.vocab_size]
            loss = None
            if compute_loss:
                lm = (mask[:, :-1] * tmask[:, 1:]).reshape(-1) > 0
                pos = torch.arange(B * S, device=self.device).view(B, S)[:, :-1].reshape(-1)[lm].to(torch.int32)
                loss, _, _ = ops.masked_ce_fwd(full, self.vocab_size, pos, tokens.reshape(-1).contiguous())
        return logits, loss

    def _check_packing(self, compute_loss):
        if self.pack_sequences and compute_loss and self.materialize_logits:
            raise ValueError("pack_sequences=True needs materialize_logits=False: the packed layout has no [B, S, V] logits "
                             "to return (set materialize_logits = False, as the trainer does, or turn pack_sequences off)")

    def tokenize_input_dicts(self, inputs: list):
        """gato_policy.py:195-432 -> (token_embeddings fp32 [B,S,d], tokens int64 [B,S], token_target_masks fp32,
        token_masks fp32).  Tensors are detached (training goes through ``forward(inputs=...)``)."""
        self._check_arena()
        with torch.no_grad():
            state = self._plan(inputs, False)
            state.need_grad = False
            self._embed(state)
        B, W, d = state.plan.B, state.plan.width, self.embed_dim
        return (state.x0.view(B, W, d).clone(), state.tokens.view(B, W).clone(), state.tmask.view(B, W).clone(),
                state.mask.view(B, W).clone())

    # ------------------------------------------------------------------------------------------
    # inference loops (gato_policy.py:444-616).  Same call pattern as the reference: every generated token re-runs the
    # context through forward(); the host logic below only picks tokens and grows the context.
    # ------------------------------------------------------------------------------------------
    def _pick(self, row: torch.Tensor, deterministic: bool) -> torch.Tensor:
        if deterministic:
            return torch.argmax(row, dim=-1)
        return torch.multinomial(torch.softmax(row, dim=-1), num_samples=1)[0]

    def _generate(self, token_embeddings, token_masks, n_tokens: int, lo: int, hi: int, deterministic: bool):
        """Autoregressive continuation on caller-owned embeddings: logits of the last position restricted to ids
        [lo, hi], pick, embed the pick, append, trim to context_len (gato_policy.py:452-476 and :586-605)."""
        rows, picked = [], []
        # KV cache (SURVEY 8(f)2): the reference re-runs the whole context for every generated token; here the first call
        # fills a key/value cache and later calls push ONE position through the decoder.  Used for a single unpadded
        # sequence in eval mode while the context still fits (a sliding window changes what the cached positions would
        # have seen, so from then on the context is recomputed like the reference does).
        use_kv = (self.use_kv_cache and not self.training and token_embeddings.shape[0] == 1
                  and bool((token_masks == 1).all()))
        cache = None
        for _ in range(n_tokens):
            S_now = token_embeddings.shape[1]
            if use_kv and S_now <= self.context_len:
                if cache is not None and cache.len == S_now - 1:
                    cache.decoding = True
                    hf = self._decode_hidden(token_embeddings[:, -1:, :], None, kv=cache)          # [1, d]
                else:
                    cache = _KVCache(self.layers, self.context_len, self.embed_dim, self.device)
                    hf = self._decode_hidden(token_embeddings, token_masks, kv=cache)[-1:]          # last position
                cache.len = S_now
                full = self._head(hf.contiguous(), 1)
                row = full[0, lo:hi + 1]
            else:
                cache = None
                logits, _ = self.forward(token_embeddings=token_embeddings, token_masks=token_masks, token_target_masks=None, tokens=None)
                row = logits[0, -1, lo:hi + 1]
            rows.append(row)
            tok = self._pick(row, deterministic) + lo
            token_masks = torch.cat([token_masks, torch.ones(token_masks.shape[0], 1, device=self.device)], dim=1)
            token_embeddings = torch.cat([token_embeddings, self.embed_token(tok).reshape(1, 1, -1)], dim=1)
            if token_embeddings.shape[1] > self.context_len:   # the window slides: cached positions are stale
                cache = None
            token_embeddings = token_embeddings[:, -self.context_len:, :]
            token_masks = token_masks[:, -self.context_len:]
            picked.append(tok)
        return rows, picked

    def predict_text(self, batch_dict, max_length=20, deterministic=True):
        """gato_policy.py:444-478 -> (logits [max_length, text_tokens], list of predicted token ids)."""
        lo, hi = self.token_starts["text"], self.token_ends["text"]
        with torch.no_grad():
            emb, _, _, masks = self.tokenize_input_dicts([batch_dict])
            rows, picked = self._generate(emb, masks, max_length, lo, hi, deterministic)
        return torch.stack(rows, dim=0), picked

    def predict_response(self, image, prompt_tokens=[], max_length=128, deterministic=True):  # noqa: B006 - reference signature
        """gato_policy.py:484-544: caption / answer generation from one image; the image is embedded once and passed as
        ``image_embeddings``, the growing text as token ids.  Returns (logits [max_length, text_tokens], decoded text)."""
        lo, hi = self.token_starts["text"], self.token_ends["text"]
        with torch.no_grad():
            image_embeddings = self.image_embedding(image.to(self.device))
            assert image_embeddings.shape[0] == 1, "number of images should always be 1 for predicting response"
            n_patches = image_embeddings.shape[1]
            rows, response = [], []
            prompt = list(prompt_tokens)
            n_ctx0 = n_patches + len(prompt)
            if self.use_kv_cache and not self.training and n_ctx0 + max_length + 1 <= self.context_len:
                # KV-cached variant of the loop below: the context [patches, prompt] is pushed through the decoder once (the
                # trailing separator is causal dead weight: it never influences the positions before it), then every picked
                # token enters as ONE new position: embed_token row + the position embedding of its slot inside the
                # timestep's observation block (patches first, then text: gato_policy.py:380-385).
                emb, _, _, _ = self.tokenize_input_dicts([{"image_embeddings": image_embeddings,
                                                           "text": torch.tensor(prompt, dtype=torch.long)}])
                cache = _KVCache(self.layers, self.context_len, self.embed_dim, self.device)
                hf = self._decode_hidden(emb[:, :n_ctx0, :], None, kv=cache)[-1:]
                cache.len = n_ctx0
                cache.decoding = True
                for idx in range(max_length):
                    row = self._head(hf.contiguous(), 1)[0, lo:hi + 1]
                    rows.append(row)
                    tok = int(self._pick(row, deterministic))
                    response.append(tok)
                    if idx + 1 == max_length:
                        break
                    e = self.embed_token(torch.tensor([tok + lo], device=self.device)).reshape(1, 1, -1)
                    if self.use_pos_encoding:
                        e = e + self.pos_embed_observation.weight.detach()[n_ctx0 + idx]
                    hf = self._decode_hidden(e, None, kv=cache)
                    cache.len += 1
                return torch.stack(rows, dim=0), self.text_tokenizer.decode(response)
            for idx in range(max_length):
                batch = {"image_embeddings": image_embeddings, "text": torch.tensor(prompt + response, dtype=torch.long)}
                logits, _ = self.forward([batch])
                assert logits.shape[0] == 1, "batch size should always be 1 for predicting response"
                # the last image patch predicts the first text token, each text token the next one
                row = logits[0, n_patches - 1 + len(prompt) + idx, lo:hi + 1]
                rows.append(row)
                response.append(int(self._pick(row, deterministic)))
        return torch.stack(rows, dim=0), self.text_tokenizer.decode(response)

    def predict_caption(self, image, max_length=128, deterministic=True):
        return self.predict_response(image, prompt_tokens=[], max_length=max_length, deterministic=deterministic)

    def predict_answer(self, image, question, max_length=16, deterministic=True):
        return self.predict_response(image, prompt_tokens=self.text_tokenizer.encode(question), max_length=max_length,
                                     deterministic=deterministic)

    def predict_control(self, input: dict, task, deterministic: bool = True):  # noqa: A002 - reference signature
        """gato_policy.py:557-616: one action for a control task.  ``input`` carries one padded action timestep at the
        end; its tokens are dropped and re-generated, restricted to the task's action vocabulary."""
        kind = getattr(task.action_type, "__name__", str(task.action_type))
        action_tokens = task.action_tokens
        if "Discrete" in kind:
            which = "discrete"
            assert action_tokens == 1, "only support 1 discrete action token"
        elif "Box" in kind:
            which = "continuous"
        else:
            raise ValueError(f"unsupported action space {kind}")
        lo, hi = self.token_starts[which], self.token_ends[which]
        if which == "discrete":
            assert task.env.action_space.n <= self.discrete_tokens, "discrete action space too large for model"
            hi = lo + task.env.action_space.n - 1
        with torch.no_grad():
            emb, _, _, masks = self.tokenize_input_dicts([input])
            emb, masks = emb[:, :-action_tokens, :], masks[:, :-action_tokens]
            _, picked = self._generate(emb, masks, action_tokens, lo, hi, deterministic)
        if which == "discrete":
            return picked[0] - lo
        return self.continuous_action_tokenizer.decode(torch.stack(picked, dim=0))

    # ------------------------------------------------------------------------------------------
    # planning + upload
    # ------------------------------------------------------------------------------------------
    def _plan(self, inputs, compute_loss) -> _State:
        st = _State()
        # packing applies to loss-computing steps (tokenize_input_dicts, the predict_* loops and evaluation forwards stay padded)
        packed = bool(self.pack_sequences and compute_loss and not self.materialize_logits)
        plan = build_plan(inputs, patch_size=self.patch_size, context_len=self.context_len, pad_seq=self.pad_seq, packed=packed)
        st.plan = plan
        st.compute_loss = bool(compute_loss)
        # train-mode patch bins consume the global CPU RNG per image-bearing sample, rows first (embeddings.py:92-95)
        st.row_bins = st.col_bins = None
        if plan.n_patch_rows and self.use_patch_pos_encoding and any(g.tensors for g in plan.image_groups):
            ppe = self.image_embedding.patch_pos_encoding
            rb = np.zeros(plan.n_patch_rows, dtype=np.int32)
            cb = np.zeros(plan.n_patch_rows, dtype=np.int32)
            per_sample = {}
            for g in plan.image_groups:
                for k, b in enumerate(g.sample_idx):
                    per_sample[b] = (g, k)
            for b in sorted(per_sample):  # batch order = the reference's draw order
                g, k = per_sample[b]
                n_h, n_w = g.height // self.patch_size, g.width // self.patch_size
                hp, wp = ppe.positions(n_h, n_w)
                T = int(g.tensors[k].shape[0])
                off = g.patch_off[k]
                rb[off:off + T * n_h * n_w] = np.tile(np.repeat(hp.numpy(), n_w), T)
                cb[off:off + T * n_h * n_w] = np.tile(np.tile(wp.numpy(), n_h), T)
            st.row_bins, st.col_bins = rb, cb
        st.h2d_bytes = 0
        self._upload_plan(st, self._next_drop_seed())
        return st

    def _upload_plan(self, st: _State, seed):
        """The batch's single pinned -> device copy (descriptors, scalars, ids, loss rows, dropout seed header)."""
        descs, fv, iv, first_valid, loss_rows, cu_seqlens, h2d, hdr = self._stager.upload(st.plan, seed)
        st.descs, st.fvals, st.ivals, st.first_valid, st.loss_rows = descs, fv, iv, first_valid, loss_rows
        st.cu_seqlens = cu_seqlens
        st.drop_seed = hdr[:2]
        st.drop_seed_host = seed
        st.stager_gen = self._stager.generation
        self._last_drop = (st.drop_seed, st.plan)
        st.h2d_bytes += h2d

    def _tok_params(self, plan: BatchPlan) -> TokParams:
        return TokParams(mu=float(self.mu), M=float(self.M), n_bins=int(self.continuous_tokens),
                         cont_start=int(self.token_starts["continuous"]), disc_start=int(self.token_starts["discrete"]),
                         vocab=int(self.vocab_size), use_pos=int(bool(self.use_pos_encoding)), seq_len=int(plan.seq_len),
                         width=int(plan.width), ctx_rows=int(self.context_len))

    # ------------------------------------------------------------------------------------------
    # image front end
    # ------------------------------------------------------------------------------------------
    def _image_upload(self, st: _State):
        """Eager part of the image front end: frames (and train-mode position bins, caller-supplied patch
        embeddings) move into stable device buffers.  Never part of a CUDA graph: source addresses change per step."""
        plan = st.plan
        d = self.embed_dim
        st.patch_emb = None
        st.img_bufs = []
        if plan.n_patch_rows == 0:
            return
        pe = self._buf("patch_emb", (plan.n_patch_rows, d), torch.float32)
        st.patch_emb = pe
        for gi, g in enumerate(plan.image_groups):
            if not g.tensors:
                continue
            n_px = 3 * g.height * g.width
            buf = self._buf(f"img{gi}", (g.n_frames * n_px,), torch.uint8 if g.is_u8 else torch.float32)
            pre = getattr(st, "img_in", {}).get(gi)
            if pre is not None:      # staged batch: the frames are already on the device (copy stream)
                torch.cuda.current_stream(self.device).wait_event(st.img_ready)
                buf.copy_(pre[:buf.numel()], non_blocking=True)
            else:
                o = 0
                for t in g.tensors:  # pinned / device sources copy asynchronously; no host-side concatenation
                    n = t.numel()
                    buf[o:o + n].view(t.shape).copy_(t, non_blocking=True)
                    if not t.is_cuda:
                        st.h2d_bytes += n * t.element_size()
                    o += n
            st.img_bufs.append((gi, g, buf))
        if getattr(st, "img_in", None):
            self._img_in_free = torch.cuda.Event()
            self._img_in_free.record(torch.cuda.current_stream(self.device))
            st.img_in = {}
        st.dev_row_bins = st.dev_col_bins = None
        if st.row_bins is not None:
            bins = torch.from_numpy(np.concatenate([st.row_bins, st.col_bins]))
            dev_bins = self._buf("patch_bins", (2 * plan.n_patch_rows,), torch.int32)
            dev_bins.copy_(bins, non_blocking=True)
            st.h2d_bytes += bins.numel() * 4
            st.dev_row_bins, st.dev_col_bins = dev_bins[:plan.n_patch_rows], dev_bins[plan.n_patch_rows:]
        for off, emb in plan.precomputed_patch:  # caller-supplied image_embeddings (gato_policy.py:286-287)
            n = emb.shape[0] * emb.shape[1]
            pe[off:off + n].copy_(emb.reshape(n, d).to(torch.float32), non_blocking=True)

    def _image_compute(self, st: _State):
        """ResNet block + projection + patch position add on the uploaded frames (kernel launches only)."""
        plan = st.plan
        d = self.embed_dim
        st.img_groups = []
        if plan.n_patch_rows == 0 or not st.img_bufs:
            return
        pe = st.patch_emb
        ie = self.image_embedding
        rb = ie.patch_embedding
        lib = load()
        for (gi, g, buf) in st.img_bufs:
            n_h, n_w = g.height // self.patch_size, g.width // self.patch_size
            P = g.n_frames * n_h * n_w
            row0 = g.patch_off[0]
            patches = self._buf(f"patches{gi}", (P, 3 * self.patch_size ** 2), torch.float16)
            patches_b = self._buf(f"patches_b{gi}", (P, 3 * self.patch_size ** 2), torch.bfloat16) if (st.need_grad or self.fwd_dtype != torch.float16) else None
            stats = self._buf(f"gnstats{gi}", (P, rb.num_groups, 2), torch.float32)
            check(lib.neko_patch_resblock_fwd(_p(buf), C.c_int(int(g.is_u8)), C.c_int(g.n_frames), C.c_int(g.height), C.c_int(g.width),
                                              C.c_int(self.patch_size), C.c_int(rb.mid_channels), C.c_int(rb.num_groups),
                                              _p(rb.conv1.weight), _p(rb.conv1.bias), _p(rb.gn2.weight), _p(rb.gn2.bias),
                                              _p(rb.conv2.weight), _p(rb.conv2.bias), _p(patches), _p(patches_b), _p(stats), stream_ptr()),
                  "neko_patch_resblock_fwd")
            out = pe[row0:row0 + P]
            if self.fwd_dtype == torch.float16:
                self._gemm(patches, self._wview("image_embedding.post_embedding_projection.weight"), epilogue=ops.EPI_F32,
                           out=out, bias=ie.post_embedding_projection.bias)
            else:
                self._gemm(patches_b, self._wview("image_embedding.post_embedding_projection.weight", bwd=True), epilogue=ops.EPI_F32,
                           out=out, bias=ie.post_embedding_projection.bias)
            self.launches += 2
            st.img_groups.append((gi, g, buf, patches_b, stats, row0, P))
            if st.dev_row_bins is not None:
                check(lib.neko_patch_pos_add(_p(out), C.c_int(P), C.c_int(d), _p(st.dev_row_bins[row0:row0 + P]),
                                             _p(st.dev_col_bins[row0:row0 + P]),
                                             _p(ie.patch_pos_encoding.height_pos_embedding.weight),
                                             _p(ie.patch_pos_encoding.width_pos_embedding.weight), stream_ptr()),
                      "neko_patch_pos_add")
                self.launches += 1

    def _image_forward(self, st: _State):
        self._image_upload(st)
        self._image_compute(st)

    def _embed_images_standalone(self, images: torch.Tensor) -> torch.Tensor:
        """ImageEmbedding.forward(x) for callers such as predict_response (gato_policy.py:489)."""
        with torch.no_grad():
            st = self._plan([{"images": images}], False)
            st.need_grad = False
            self._refresh_bf16()
            self._image_forward(st)
        T = images.shape[0]
        return st.patch_emb.view(T, -1, self.embed_dim).clone()

    # ------------------------------------------------------------------------------------------
    # forward engine
    # ------------------------------------------------------------------------------------------
    def _embed(self, st: _State):
        plan = st.plan
        d = self.embed_dim
        N = plan.token_rows
        if not getattr(st, "in_graph", False):   # graph mode: _engine_forward refreshed the copies eagerly, version-checked
            self._refresh_bf16()
        if not getattr(st, "uploaded", False):
            self._image_upload(st)
        self._image_compute(st)
        keep = st.need_grad
        st.tokens = self._buf("tokens", (N,), torch.int64)
        st.tmask = self._buf("tmask", (N,), torch.float32)
        st.mask = self._buf("mask", (N,), torch.float32)
        st.x0 = self._buf("x.0" if keep else "x.a", (N, d), torch.float32)
        st.tok_params = self._tok_params(plan)
        self._launch_tokenize(st)

    def _launch_tokenize(self, st: _State):
        """The tokenise + embed + interleave + pad kernel alone (bench.py times it against the HBM roofline)."""
        plan, d, prm = st.plan, self.embed_dim, st.tok_params
        ops.tokenize_embed_fwd(st.descs, plan.B, d, prm, st.fvals, st.ivals, st.patch_emb, self.embed_token.weight,
                               self.pos_embed_observation.weight, self.separator_token, st.tokens, st.tmask, st.mask, st.x0,
                               packed=plan.packed)
        self.launches += 1

    # -- dropout ------------------------------------------------------------------------------------
    # Sites (include/neko_b200.h neko_dropout.stream): 0 embeddings (transformer.drop, p = 0.1 whatever --dropout says,
    # SURVEY quirk 8), 4*layer+1 attention weights, 4*layer+2 attention residual branch, 4*layer+3 MLP residual branch.
    # Masks are counter based: the two seed words travel with the batch upload, kernels regenerate the mask in backward.
    def _dropout_ps(self):
        if not self.training:
            return None
        ps = [float(self.transformer.drop.p)]
        for blk in self.transformer.h:
            ps += [float(blk.attn.attn_dropout.p), float(blk.attn.resid_dropout.p), float(blk.mlp.dropout.p)]
        return tuple(ps) if any(ps) else None

    def _next_drop_seed(self):
        if self._dropout_ps() is None:
            return None
        if self._drop_gen is None:   # own generator: the global CPU stream keeps feeding the patch-position draws only
            self._drop_gen = torch.Generator()
            self._drop_gen.manual_seed(torch.initial_seed() & 0x7FFFFFFFFFFFFFFF)
        return torch.randint(0, 2 ** 31 - 1, (2,), generator=self._drop_gen, dtype=torch.int32).numpy()

    def dropout_multipliers(self):
        """The multipliers (mask / (1 - p_eff)) the kernels applied in the most recent train-mode forward, keyed like
        ``oracle.gato_oracle.decoder(drop=...)``: lets a test (or a debugging session) replay the step in a reference."""
        ps = self._dropout_ps()
        if ps is None or getattr(self, "_last_drop", None) is None:
            return {}
        seed, plan = self._last_drop
        B, W = plan.B, plan.width
        d, H = self.embed_dim, self.heads

        def mult(stream, p, rows, cols):
            dr = Dropout.make(seed, stream, p)
            return ops.dropout_mask(rows, cols, dr, self.device).to(torch.float32) * dr.scale

        if plan.packed:   # row masks were drawn at packed rows: scatter packed row row_base[b] + p to (b, first_valid[b] + p)
            lengths = np.diff(plan.cu_seqlens)
            dst = np.concatenate([b * W + plan.first_valid[b] + np.arange(lengths[b]) for b in range(B)])
            dst = torch.from_numpy(dst).to(self.device)

        def row_mult(stream, p):
            if not plan.packed:
                return mult(stream, p, B * W, d).view(B, W, d)
            full = torch.zeros(B * W, d, device=self.device)
            full[dst] = mult(stream, p, plan.token_rows, d)
            return full.view(B, W, d)

        out = {}
        if ps[0] > 0:
            out["embd"] = row_mult(0, ps[0])
        for i in range(self.layers):
            pa, pr, pm = ps[1 + 3 * i:4 + 3 * i]
            if pa > 0:
                out[("attn", i)] = mult(4 * i + 1, pa, B * H * W, W).view(B, H, W, W)
            if pr > 0:
                out[("resid_attn", i)] = row_mult(4 * i + 2, pr)
            if pm > 0:
                out[("resid_mlp", i)] = row_mult(4 * i + 3, pm)
        return out

    def _drop_site(self, st: _State, stream: int, p: float):
        seed = getattr(st, "drop_seed", None)
        if not self.training or p <= 0.0 or seed is None:
            return None
        return Dropout.make(seed, stream, p)

    def _decoder(self, st: _State, x: torch.Tensor, B: int, W: int, S_valid: int, first_valid: torch.Tensor, keep: bool):
        """L pre-LN blocks + ln_f (trajectory_gpt2.py:322-358, 779).  x fp32 [N,d] -> hf bf16 [N,d]."""
        gate = bool(self.transformer.config.gate)
        d, H = self.embed_dim, self.heads
        N = x.shape[0]            # B * W, or the T rows of a packed batch
        packed = getattr(st, "plan", None) is not None and st.plan.packed
        eps = self.transformer.config.layer_norm_epsilon
        fdt = self.fwd_dtype
        dual = keep and fdt != torch.bfloat16   # backward GEMMs need bf16 copies of the saved activations
        acts = []

        def pair(name, tag, shape):
            """(forward-format buffer, bf16 buffer kept for backward)"""
            if not dual:
                t = self._buf(name + tag, shape, fdt)
                return t, (t if keep else None)
            return self._buf(name, shape, fdt), self._buf(name + ".b" + tag, shape, torch.bfloat16)

        d0 = self._drop_site(st, 0, self.transformer.drop.p)
        if d0 is not None:                      # hidden_states = self.drop(inputs_embeds), trajectory_gpt2.py:707
            ops.dropout_apply(x, d0)
            self.launches += 1
        for i, blk in enumerate(self.transformer.h):
            tag = f".{i}" if keep else ""
            pre = f"transformer.h.{i}."
            ln1, ln1_b = pair("ln1", tag, (N, d))
            m1 = self._buf("m1" + tag, (N,), torch.float32)
            r1 = self._buf("r1" + tag, (N,), torch.float32)
            ops.layernorm_fwd(x, blk.ln_1.weight, blk.ln_1.bias, eps, ln1, m1, r1, y2=ln1_b if dual else None)
            qkv = self._buf("qkv" + tag, (N, 3 * d), torch.bfloat16)
            self._gemm(ln1, self._wview(pre + "attn.c_attn.weight"), b_mn=True, epilogue=ops.EPI_BF16, out=qkv, bias=blk.attn.c_attn.bias)
            att, att_b = pair("att", tag, (N, d))
            lse = self._buf("lse" + tag, (H, N) if packed else (B, H, W), torch.float32)
            kv = getattr(st, "kv", None)
            if packed:
                ops.attention_varlen_fwd(qkv, st.cu_seqlens, first_valid, H, S_valid, W, att, lse, out2=att_b if dual else None,
                                         drop=self._drop_site(st, 4 * i + 1, blk.attn.attn_dropout.p))
            elif kv is not None and kv.decoding:
                # KV-cached decode: N == 1; append this position's key / value, attend over the cache
                kv.k[i, kv.len].copy_(qkv[0, d:2 * d])
                kv.v[i, kv.len].copy_(qkv[0, 2 * d:])
                ops.attention_decode(qkv[0, :d], kv.k[i], kv.v[i], kv.len + 1, H, att.view(d))
            else:
                ops.attention_fwd(qkv.view(B, W, 3 * d), first_valid, H, S_valid, att.view(B, W, d), lse,
                                  out2=att_b.view(B, W, d) if dual else None, drop=self._drop_site(st, 4 * i + 1, blk.attn.attn_dropout.p))
                if kv is not None:   # prefill: keep the keys / values of the context
                    kv.k[i, :W].copy_(qkv[:W, d:2 * d])
                    kv.v[i, :W].copy_(qkv[:W, 2 * d:])
            x1 = self._buf(f"x.{2 * i + 1}" if keep else "x.b", (N, d), torch.float32)
            self._gemm(att, self._wview(pre + "attn.c_proj.weight"), b_mn=True, epilogue=ops.EPI_RESID_F32, out=x1, aux=x,
                       bias=blk.attn.c_proj.bias, drop=self._drop_site(st, 4 * i + 2, blk.attn.resid_dropout.p))
            ln2, ln2_b = pair("ln2", tag, (N, d))
            m2 = self._buf("m2" + tag, (N,), torch.float32)
            r2 = self._buf("r2" + tag, (N,), torch.float32)
            ops.layernorm_fwd(x1, blk.ln_2.weight, blk.ln_2.bias, eps, ln2, m2, r2, y2=ln2_b if dual else None)
            fpre = self._buf("fpre" + tag, (N, 4 * d), torch.bfloat16)
            fact, fact_b = pair("fact", tag, (N, 4 * d))
            fgate = None
            # mlp_proj_bf16: the GELU GEMM is bound by its output bytes (three [N, 4d] tensors: pre-activation, fp16 activation for
            # the forward down-projection, bf16 twin for its weight gradient).  With the flag the forward down-projection runs on
            # the bf16 twin (and the bf16 weight copy) and the fp16 tensor is never written.
            lowp = dual and self.mlp_proj_bf16 and not gate
            if lowp:
                self._gemm(ln2, self._wview(pre + "mlp.c_fc.weight"), b_mn=True, epilogue=ops.EPI_GELU_BF16, out=fpre, out2=fact_b,
                           bias=blk.mlp.c_fc.bias, gelu_tanh=self._gelu_tanh)
            elif not gate:
                self._gemm(ln2, self._wview(pre + "mlp.c_fc.weight"), b_mn=True, epilogue=ops.EPI_GELU_BF16, out=fpre, out2=fact,
                           out3=fact_b if dual else None, bias=blk.mlp.c_fc.bias, gelu_tanh=self._gelu_tanh)
            else:   # geglu: h = gelu(c_fc(x)) * gated_layer(x)   (trajectory_gpt2.py:267-276; nn.Linear weight is [out, in])
                gelu_o = self._buf("fgelu", (N, 4 * d), fdt)
                self._gemm(ln2, self._wview(pre + "mlp.c_fc.weight"), b_mn=True, epilogue=ops.EPI_GELU_BF16, out=fpre, out2=gelu_o,
                           bias=blk.mlp.c_fc.bias)
                fgate = self._buf("fgate" + tag, (N, 4 * d), torch.bfloat16)
                self._gemm(ln2, self._wview(pre + "mlp.gated_layer.weight"), epilogue=ops.EPI_BF16, out=fgate,
                           bias=blk.mlp.gated_layer.bias)
                ops.geglu_fwd(gelu_o, fgate, fact, fact_b if dual else None)
                self.launches += 2
            x2 = self._buf(f"x.{2 * i + 2}" if keep else "x.a", (N, d), torch.float32)
            self._gemm(fact_b if lowp else fact, self._wview(pre + "mlp.c_proj.weight", bwd=lowp), b_mn=True, epilogue=ops.EPI_RESID_F32,
                       out=x2, aux=x1, bias=blk.mlp.c_proj.bias, drop=self._drop_site(st, 4 * i + 3, blk.mlp.dropout.p))
            self.launches += 7
            if keep:
                acts.append((x, ln1_b, m1, r1, qkv, att_b, lse, x1, ln2_b, m2, r2, fpre, fact_b, fgate))
            x = x2
        hf, hf_b = pair("hf", "", (N, d))
        mf = self._buf("mf", (N,), torch.float32)
        rf = self._buf("rf", (N,), torch.float32)
        ops.layernorm_fwd(x, self.transformer.ln_f.weight, self.transformer.ln_f.bias, eps, hf, mf, rf, y2=hf_b if dual else None)
        self.launches += 1
        if keep:
            st.acts, st.x_last, st.hf, st.mf, st.rf = acts, x, hf_b, mf, rf
        return hf

    def _head(self, hf: torch.Tensor, n_rows: int, f16: bool = False) -> torch.Tensor:
        """predict_token (gato_policy.py:172): fp32 logits [n_rows, Vp] (columns >= V are exact zeros).  Freshly
        allocated (torch's caching allocator) because the caller keeps the tensor.  ``f16``: the training path that never
        returns logits (materialize_logits = False) keeps them in fp16 in a workspace buffer -- they only feed the fused
        cross entropy, which reads V*2 instead of V*4 bytes per row (csrc/ce.cu: ce_fused_f16_kernel)."""
        if f16:
            logits = self._buf("logits_rows_f16", (n_rows, self._Vp), torch.float16)
            self._gemm(hf, self._wview("predict_token.weight", rows=self._Vp), epilogue=ops.EPI_BF16, out=logits, N=self._Vp)
        else:
            logits = torch.empty(n_rows, self._Vp, dtype=torch.float32, device=self.device)
            self._gemm(hf, self._wview("predict_token.weight", rows=self._Vp), epilogue=ops.EPI_F32, out=logits, N=self._Vp)
        self.launches += 1
        return logits

    def _decode_embeddings(self, emb: torch.Tensor, mask: Optional[torch.Tensor]) -> torch.Tensor:
        B, S, d = emb.shape
        return self._decode_hidden(emb, mask).view(B, S, d).to(torch.float32)

    def _decode_hidden(self, emb: torch.Tensor, mask: Optional[torch.Tensor], kv=None) -> torch.Tensor:
        """Decoder on caller-supplied embeddings (the kwargs path used by predict_*, gato_policy.py:160-169);
        returns ln_f output as the bf16 [B*S, d] head operand.  ``kv``: optional _KVCache to fill (prefill) or to decode
        one new position against."""
        with torch.no_grad():
            self._refresh_bf16()
            B, S, d = emb.shape
            x = self._buf("x.a", (B * S, d), torch.float32)
            x.copy_(emb.reshape(B * S, d).to(torch.float32))
            if mask is None:
                fv = torch.zeros(B, dtype=torch.int32, device=self.device)
            else:  # first valid key per sample; right padding is never visible to a valid (causal) query
                fv = (mask.to(self.device).cumsum(1) == 0).sum(1).to(torch.int32)
            st = _State()
            st.kv = kv
            seed = self._next_drop_seed()
            st.drop_seed = torch.from_numpy(seed).to(self.device) if seed is not None else None
            return self._decoder(st, x, B, S, S, fv, keep=False)

    # -- CUDA graphs -------------------------------------------------------------------------------------
    # The step is ~150 dependent launches; replaying it from a graph removes the launch gaps (7.6 -> 6.4 ms at cfg2).
    # A graph is keyed by everything that shapes the launches (the batch plan's descriptors, modes); the first sight of
    # a key runs eagerly (sizes the workspace), the second captures, later ones replay.  Uploads stay eager.
    def _graph_key(self, st: _State):
        p = st.plan
        return (p.B, p.seq_len, p.width, p.descs.tobytes(), tuple((g.height, g.width, g.is_u8, g.n_frames) for g in p.image_groups),
                len(p.precomputed_patch), st.compute_loss, st.need_grad, self.training, self.materialize_logits, self.head_mode,
                self.fwd_dtype, st.row_bins is not None, self._dropout_ps(), self.lean_logits_f16, self.mlp_proj_bf16,
                self.deterministic, p.packed)

    def _engine_forward(self, st: _State):
        if not self.use_cuda_graphs:
            return self._forward_compute(st)
        # 16-bit weight copies: refreshed OUTSIDE the graph, and only when a parameter changed since the last cast (an
        # optimiser step, load_state_dict, ...); the captured kernels read the pointer-stable copies
        self._refresh_bf16()
        self._image_upload(st)
        st.uploaded = True
        key = self._graph_key(st)
        ent = self._graphs.get(key)
        if ent is not None and ent.get("epoch") != (getattr(self, "_ws_epoch", 0), self._stager_epoch()):
            ent = None
            self._graphs.pop(key, None)
        if ent is None:                       # first sight: eager (allocates / grows the workspace)
            out = self._forward_compute(st)
            while len(self._graphs) >= self.max_cuda_graphs:   # bounded cache: every entry pins its logits in the pool
                self._graphs.pop(next(iter(self._graphs)))
            self._graphs[key] = {"seen": 1, "epoch": (getattr(self, "_ws_epoch", 0), self._stager_epoch())}
            st.graph_entry = None
            return out
        if "fwd" not in ent:                  # second sight: capture
            _before_capture()
            l0 = self.launches
            gph = torch.cuda.CUDAGraph()
            if self._graph_pool is None:
                self._graph_pool = torch.cuda.graph_pool_handle()
            st.in_graph = True
            self._capturing = True
            try:
                with torch.cuda.graph(gph, pool=self._graph_pool):
                    out = self._forward_compute(st)
            finally:
                self._capturing = False
            ent.update(fwd=gph, state=st, out=out, fwd_launches=self.launches - l0, bwd={})
            gph.replay()
            st.graph_entry = ent
            return out
        # replay: the captured state object carries every buffer; refresh only what the host changed
        cst = ent["state"]
        cst.plan, cst.h2d_bytes = st.plan, st.h2d_bytes
        self._generation += 1
        cst.generation = self._generation
        ent["fwd"].replay()
        self.launches += ent["fwd_launches"]
        st.__dict__.update(cst.__dict__)
        st.graph_entry = ent
        return ent["out"]

    def _stager_epoch(self):
        """Addresses captured graphs depend on besides the workspace: the staging buffer and the 16-bit weight copies."""
        return (self._stager._dev.data_ptr() if self._stager._dev is not None else 0, self._w16_arena.data_ptr(),
                self._wbf_arena.data_ptr(), self._param_arena.data_ptr(), self._grad_arena.data_ptr())

    def _forward_compute(self, st: _State):
        plan = st.plan
        B, W, d, V = plan.B, plan.width, self.embed_dim, self.vocab_size
        N = plan.token_rows
        self._generation += 1
        st.generation = self._generation
        keep = st.need_grad
        self._embed(st)
        hf = self._decoder(st, st.x0, B, W, plan.seq_len, st.first_valid, keep)
        n_rows = int(plan.loss_rows.shape[0])
        st.n_rows = n_rows
        loss = None
        if self.materialize_logits:
            full = self._head(hf, N)
            logits = full.view(B, W, self._Vp)[:, :, :V]
            st.logits_full = full
            if st.compute_loss:
                if n_rows == 0:
                    loss = torch.full((), float("nan"), device=self.device)  # mean over an empty selection
                else:
                    loss = self._ce_forward(st, full, V, n_rows, keep, 0)
        else:
            logits = torch.empty(0, device=self.device)
            if st.compute_loss and n_rows:
                hc = self._buf("hf_rows", (n_rows, d), self.fwd_dtype)
                ops.gather_rows(hf, st.loss_rows, d, hc)
                # with gradients wanted, the logits of the loss rows exist only between the head GEMM and the fused cross
                # entropy: 16 bits are enough there (loss statistics stay fp32)
                f16 = keep and self.lean_logits_f16 and hc.dtype == torch.float16 and (self._Vp * 2) <= 220 * 1024
                full = self._head(hc, n_rows, f16=f16)
                st.logits_full, st.hf_rows = full, hc
                loss = self._ce_forward(st, full, V, n_rows, keep, ops.CE_LOGITS_COMPACT)
                if f16 and not st.ce_fused:     # not applicable after all (alignment): take the fp32 route
                    full = self._head(hc, n_rows)
                    st.logits_full = full
                    loss = self._ce_forward(st, full, V, n_rows, keep, ops.CE_LOGITS_COMPACT)
                self.launches += 1
        return logits, loss

    def _ce_forward(self, st: _State, full: torch.Tensor, V: int, n_rows: int, keep: bool, flags: int):
        """Masked cross entropy (gato_policy.py:174-186).  With gradients wanted and the compact head backward, the loss
        and the (unscaled) dlogits operand come out of ONE pass over the selected rows (ce_fused_kernel)."""
        st.ce_fused = False
        if keep and (self.head_mode == "rows" or not self.materialize_logits):
            dl = self._buf("dlogits_rows", (n_rows, self._Vp), torch.bfloat16)
            out = ops.masked_ce_fused(full, V, st.loss_rows, st.tokens, dl, flags=flags | ops.CE_DLOGITS_COMPACT | ops.CE_ZERO_PAD)
            if out is not None:
                st.ce_fused = True
                self.launches += 2
                loss, st.row_lse = out
                return loss
        if full.dtype != torch.float32:
            return None                     # 16-bit logits exist for the fused kernel only: the caller falls back to fp32
        loss, st.row_lse, _ = ops.masked_ce_fwd(full, V, st.loss_rows, st.tokens, flags=flags)
        self.launches += 2
        return loss

    # ------------------------------------------------------------------------------------------
    # backward engine
    # ------------------------------------------------------------------------------------------
    def _notify(self, first: str, last: str):
        if self.grad_ready_hook is not None:
            lo = self._offs[first]
            hi = self._offs[last] + _pad_to(self._params[last].numel(), 64)
            if last == "predict_token.weight":
                hi = self._offs[last] + _pad_to(self._Vp * self.embed_dim, 64)
            self.grad_ready_hook(lo, hi)

    def _engine_backward(self, st: _State, g_loss: torch.Tensor):
        self._engine_backward_inner(st, g_loss)
        sync = getattr(self, "_grad_sync", None)
        if sync is not None and getattr(sync, "mode", "overlap") == "tail":
            sync.finish_tail()

    def _engine_backward_inner(self, st: _State, g_loss: torch.Tensor):
        ent = getattr(st, "graph_entry", None)
        sync = getattr(self, "_grad_sync", None)
        hooked = self.grad_ready_hook is not None
        # a data-parallel synchroniser whose launches are graph-safe (dp backend "p2p") is captured WITH backward: its
        # bucket all-reduces replay on their side-stream branch of the graph
        if ent is None or (hooked and not (sync is not None and getattr(sync, "capturable", False))):
            return self._backward_compute(st, g_loss, None)
        if st.generation != self._generation:
            raise RuntimeError("backward() called after a newer forward reused the activation workspace")
        plan = st.plan
        acc = self._begin_grads(bool(plan.n_patch_rows and getattr(st, 'img_groups', None)), zero=False)
        self._gscale_buf.copy_(g_loss.detach().to(torch.float32).reshape(()))
        if hooked:
            acc = (acc, bool(sync.enabled))    # no_sync() micro-steps replay a graph without the all-reduces
        gb = ent["bwd"].get(acc)
        if gb is None:
            _before_capture()
            l0 = self.launches
            gph = torch.cuda.CUDAGraph()
            self._capturing = True
            try:
                with torch.cuda.graph(gph, pool=self._graph_pool):
                    self._backward_compute(ent["state"], self._gscale_buf, acc[0] if isinstance(acc, tuple) else acc)
            finally:
                self._capturing = False
            ent["bwd"][acc] = (gph, self.launches - l0)
            gph.replay()
            return
        gb[0].replay()
        self.launches += gb[1]

    def _backward_compute(self, st: _State, g_loss: torch.Tensor, acc_override):
        if st.generation != self._generation:
            raise RuntimeError("backward() called after a newer forward reused the activation workspace")
        if not st.compute_loss or st.n_rows == 0:
            raise RuntimeError("nothing to differentiate: forward ran with compute_loss=False or selected no loss rows")
        plan = st.plan
        B, W, d, V, Vp, H = plan.B, plan.width, self.embed_dim, self.vocab_size, self._Vp, self.heads
        N = plan.token_rows
        n_rows = st.n_rows
        sync = getattr(self, "_grad_sync", None)
        if sync is not None and getattr(sync, "mode", "overlap") == "tail":
            sync = None
        if sync is not None:
            if self.deterministic:
                sync.require_deterministic()
            sync.begin_step()
        if acc_override is None:
            acc = self._begin_grads(bool(plan.n_patch_rows and getattr(st, 'img_groups', None)))
        else:  # graph capture: host bookkeeping already done, only the zero fills belong to the graph
            acc = acc_override
            if not acc:
                for lo, hi in self._zero_ranges:
                    self._grad_arena[lo:hi].zero_()
        gscale = g_loss if g_loss is self._gscale_buf else g_loss.detach().to(torch.float32).reshape(())
        G = self._gview
        Wb = lambda n, rows=None: self._wview(n, rows, bwd=True)  # noqa: E731

        # ---- head + cross entropy -----------------------------------------------------------------
        compact_logits = not self.materialize_logits
        if self.head_mode == "rows" or compact_logits:
            dl = self._buf("dlogits_rows", (n_rows, Vp), torch.bfloat16)
            # the kernel also zeroes the pad columns V..Vp (K tail of the dgrad GEMM)
            flags = ops.CE_DLOGITS_COMPACT | ops.CE_ZERO_PAD | (ops.CE_LOGITS_COMPACT if compact_logits else 0)
            if getattr(st, "ce_fused", False):   # forward already wrote (softmax - onehot) / n: apply the upstream scalar
                ops.ce_scale_grad(dl, gscale)
            else:
                ops.masked_ce_bwd(st.logits_full, V, st.loss_rows, st.tokens, st.row_lse, gscale, dl, flags=flags)
            hc = self._buf("hf_rows_b", (n_rows, d), torch.bfloat16)
            ops.gather_rows(st.hf, st.loss_rows, d, hc)
            self._gemm(dl, hc, a_mn=True, b_mn=True, epilogue=ops.EPI_F32, out=G("predict_token.weight"), accumulate=acc,
                       M=V, N=d, K=n_rows)
            # K = the padded vocabulary (818 k-blocks), a handful of output tiles: fp32 output lets the kernel split K
            dhc32 = self._buf("dhf_rows_f32", (n_rows, d), torch.float32)
            self._gemm(dl, Wb("predict_token.weight", rows=Vp), b_mn=True, epilogue=ops.EPI_F32, out=dhc32, M=n_rows, N=d, K=Vp)
            dhc = self._buf("dhf_rows", (n_rows, d), torch.bfloat16)
            ops.cast_bf16(dhc32, dhc)
            dhf = self._buf("dhf", (N, d), torch.bfloat16)
            dhf.zero_()
            ops.scatter_rows(dhc, st.loss_rows, d, dhf)
            self.launches += 7
        else:
            dl = self._buf("dlogits", (N, Vp), torch.bfloat16)
            dl.zero_()
            ops.masked_ce_bwd(st.logits_full, V, st.loss_rows, st.tokens, st.row_lse, gscale, dl)
            self._gemm(dl, st.hf, a_mn=True, b_mn=True, epilogue=ops.EPI_F32, out=G("predict_token.weight"), accumulate=acc,
                       M=V, N=d, K=N)
            # K = the padded vocabulary (818 k-blocks) but only 360 output tiles: fp32 output lets the kernel split K
            dhf32 = self._buf("dhf_f32", (N, d), torch.float32)
            self._gemm(dl, Wb("predict_token.weight", rows=Vp), b_mn=True, epilogue=ops.EPI_F32, out=dhf32, M=N, N=d, K=Vp)
            dhf = self._buf("dhf", (N, d), torch.bfloat16)
            ops.cast_bf16(dhf32, dhf)
            self.launches += 6
        self._notify("predict_token.weight", "predict_token.weight")

        # ---- ln_f -------------------------------------------------------------------------------------
        dx = self._buf("dx", (N, d), torch.float32)
        dx.zero_()
        dxb = self._buf("dx_bf16", (N, d), torch.bfloat16)
        lnf = self.transformer.ln_f
        last = f"transformer.h.{self.layers - 1}."
        # the bias gradient of a residual-feeding Conv1D is the column sum of the residual gradient: LN backward
        # emits it for free (mlp.c_proj.bias of the block below, attn.c_proj.bias of the same block)
        # With dropout the bf16 copy (and the column sum) carry mask * scale * dx: the gradient entering the dropped-out
        # residual branch below this LN (branch_drop); the fp32 dx keeps the undropped residual-path gradient.
        D = lambda s, pp: self._drop_site(st, s, pp)  # noqa: E731
        hL = self.transformer.h[self.layers - 1]
        self._ln_bwd(dhf, st.x_last, lnf.weight, st.mf, st.rf, dx, G("transformer.ln_f.weight"), G("transformer.ln_f.bias"), dxb,
                     dx_colsum=G(last + "mlp.c_proj.bias"), branch_drop=D(4 * (self.layers - 1) + 3, hL.mlp.dropout.p))
        self.launches += 2
        self._notify("transformer.ln_f.weight", "transformer.ln_f.bias")

        # ---- blocks, last to first ------------------------------------------------------------------------
        for i in reversed(range(self.layers)):
            blk = self.transformer.h[i]
            pre = f"transformer.h.{i}."
            (x0, ln1, m1, r1, qkv, att, lse, x1, ln2, m2, r2, fpre, fact, fgate) = st.acts[i]
            # MLP: x2 = x1 + gelu(ln2 @ Wfc + b) @ Wproj + b
            self._gemm(fact, dxb, a_mn=True, b_mn=True, epilogue=ops.EPI_F32, out=G(pre + "mlp.c_proj.weight"), accumulate=acc,
                       M=4 * d, N=d, K=N)
            dpre = self._buf("dfpre", (N, 4 * d), torch.bfloat16)
            dln = self._buf("dln", (N, d), torch.bfloat16)
            if fgate is None:
                self._gemm(dxb, Wb(pre + "mlp.c_proj.weight"), epilogue=ops.EPI_DGELU_BF16, out=dpre, aux=fpre, gelu_tanh=self._gelu_tanh)
            else:   # geglu: dh -> (d_gate, d_pre); the gate Linear gets its own wgrad / bias grad / dgrad
                dh4 = self._buf("dfh", (N, 4 * d), torch.bfloat16)
                self._gemm(dxb, Wb(pre + "mlp.c_proj.weight"), epilogue=ops.EPI_BF16, out=dh4)
                dgate = self._buf("dfgate", (N, 4 * d), torch.bfloat16)
                ops.geglu_bwd(dh4, fpre, fgate, dgate, dpre)
                self._gemm(dgate, ln2, a_mn=True, b_mn=True, epilogue=ops.EPI_F32, out=G(pre + "mlp.gated_layer.weight"),
                           accumulate=True, M=4 * d, N=d, K=N)
                self._colsum(dgate, G(pre + "mlp.gated_layer.bias"))
                self.launches += 4
            self._gemm(ln2, dpre, a_mn=True, b_mn=True, epilogue=ops.EPI_F32, out=G(pre + "mlp.c_fc.weight"), accumulate=acc,
                       M=d, N=4 * d, K=N)
            self._colsum(dpre, G(pre + "mlp.c_fc.bias"))
            if fgate is None:
                self._gemm(dpre, Wb(pre + "mlp.c_fc.weight"), epilogue=ops.EPI_BF16, out=dln)
            else:   # d ln2 = d_pre . Wfc^T + d_gate . Wg: two GEMMs into one fp32 buffer, then the 16-bit copy
                dln32 = self._buf("dln_f32", (N, d), torch.float32)
                self._gemm(dpre, Wb(pre + "mlp.c_fc.weight"), epilogue=ops.EPI_F32, out=dln32)
                self._gemm(dgate, Wb(pre + "mlp.gated_layer.weight"), b_mn=True, epilogue=ops.EPI_F32, out=dln32, accumulate=True)
                ops.cast_bf16(dln32, dln)
                self.launches += 2
            self._ln_bwd(dln, x1, blk.ln_2.weight, m2, r2, dx, G(pre + "ln_2.weight"), G(pre + "ln_2.bias"), dxb,
                         dx_colsum=G(pre + "attn.c_proj.bias"), branch_drop=D(4 * i + 2, blk.attn.resid_dropout.p))
            # attention: x1 = x0 + attn(ln1 @ Wqkv + b) @ Wproj + b
            self._gemm(att, dxb, a_mn=True, b_mn=True, epilogue=ops.EPI_F32, out=G(pre + "attn.c_proj.weight"), accumulate=acc,
                       M=d, N=d, K=N)
            datt = self._buf("datt", (N, d), torch.bfloat16)
            self._gemm(dxb, Wb(pre + "attn.c_proj.weight"), epilogue=ops.EPI_BF16, out=datt)
            dqkv = self._buf("dqkv", (N, 3 * d), torch.bfloat16)
            if plan.packed:
                delta = self._buf("delta", (H, N), torch.float32)
                ops.attention_varlen_bwd(qkv, att, datt, lse, st.cu_seqlens, st.first_valid, H, plan.seq_len, W, dqkv, delta,
                                         drop=D(4 * i + 1, blk.attn.attn_dropout.p))
            else:
                delta = self._buf("delta", (B, H, W), torch.float32)
                ops.attention_bwd(qkv.view(B, W, 3 * d), att.view(B, W, d), datt.view(B, W, d), lse, st.first_valid, H, plan.seq_len,
                                  dqkv.view(B, W, 3 * d), delta, drop=D(4 * i + 1, blk.attn.attn_dropout.p))
            self._gemm(ln1, dqkv, a_mn=True, b_mn=True, epilogue=ops.EPI_F32, out=G(pre + "attn.c_attn.weight"), accumulate=acc,
                       M=d, N=3 * d, K=N)
            self._colsum(dqkv, G(pre + "attn.c_attn.bias"))
            self._gemm(dqkv, Wb(pre + "attn.c_attn.weight"), epilogue=ops.EPI_BF16, out=dln)
            self._ln_bwd(dln, x0, blk.ln_1.weight, m1, r1, dx, G(pre + "ln_1.weight"), G(pre + "ln_1.bias"), dxb,
                         dx_colsum=G(f"transformer.h.{i - 1}.mlp.c_proj.bias") if i > 0 else None,
                         branch_drop=D(4 * (i - 1) + 3, self.transformer.h[i - 1].mlp.dropout.p) if i > 0 else None)
            self.launches += 14
            self._notify(pre + "mlp.c_proj.weight", pre + "ln_1.bias")

        # ---- embeddings ---------------------------------------------------------------------------------------
        d0 = D(0, self.transformer.drop.p)
        if d0 is not None:      # backward of the embedding dropout: same mask on the gradient
            ops.dropout_apply(dx, d0)
            self.launches += 1
        dpe = None
        if plan.n_patch_rows and getattr(st, "img_groups", None):
            dpe = self._buf("d_patch_emb", (plan.n_patch_rows, d), torch.float32)
            dpe.zero_()
        if self.deterministic:
            ws = self._ordered_ws(ops.embed_bwd_ordered_workspace_bytes(B, st.tok_params))
            ops.embed_bwd_ordered(st.descs, B, d, st.tok_params, st.tokens, dx, G("embed_token.weight"), G("pos_embed_observation.weight"),
                                  G("separator_token"), ws, dpe, packed=plan.packed)
        else:
            ops.embed_bwd(st.descs, B, d, st.tok_params, st.tokens, dx, G("embed_token.weight"), G("pos_embed_observation.weight"),
                          G("separator_token"), dpe, packed=plan.packed)
        self.launches += 1
        if dpe is not None:
            self._image_backward(st, dpe, acc)
        first_tail = next(n for n in self._order if n.startswith("image_embedding.") or n == "pos_embed_observation.weight")
        self._notify(first_tail, self._order[-1])
        if sync is not None:
            sync.finish()

    def _image_backward(self, st: _State, dpe: torch.Tensor, acc: bool):
        d = self.embed_dim
        ie = self.image_embedding
        rb = ie.patch_embedding
        G = self._gview
        lib = load()
        pp = "image_embedding.patch_embedding."
        for (gi, g, buf, patches, stats, row0, P) in st.img_groups:
            gslice = dpe[row0:row0 + P]
            if st.row_bins is not None and self.deterministic:
                rt = G("image_embedding.patch_pos_encoding.height_pos_embedding.weight")
                ct = G("image_embedding.patch_pos_encoding.width_pos_embedding.weight")
                ws = self._ordered_ws(ops.patch_pos_bwd_ordered_workspace_bytes(P, rt.shape[0], ct.shape[0]))
                ops.patch_pos_bwd_ordered(gslice, st.dev_row_bins[row0:row0 + P], st.dev_col_bins[row0:row0 + P], rt, ct, ws)
            elif st.row_bins is not None:
                check(lib.neko_patch_pos_bwd(_p(gslice), C.c_int(P), C.c_int(d), _p(st.dev_row_bins[row0:row0 + P]),
                                             _p(st.dev_col_bins[row0:row0 + P]),
                                             _p(G("image_embedding.patch_pos_encoding.height_pos_embedding.weight")),
                                             _p(G("image_embedding.patch_pos_encoding.width_pos_embedding.weight")), stream_ptr()),
                      "neko_patch_pos_bwd")
            gb = self._buf(f"dpe_bf16_{gi}", (P, d), torch.bfloat16)
            ops.cast_bf16(gslice, gb)
            self._colsum(gb, G("image_embedding.post_embedding_projection.bias"))
            self._gemm(gb, patches, a_mn=True, b_mn=True, epilogue=ops.EPI_F32, out=G("image_embedding.post_embedding_projection.weight"),
                       accumulate=True, M=d, N=patches.shape[1], K=P)
            dpatch = self._buf(f"dpatches{gi}", (P, patches.shape[1]), torch.bfloat16)
            self._gemm(gb, self._wview("image_embedding.post_embedding_projection.weight", bwd=True), b_mn=True, epilogue=ops.EPI_BF16, out=dpatch)
            if self.deterministic:
                ws = self._ordered_ws(ops.patch_resblock_bwd_ordered_workspace_bytes(g.n_frames, g.height, g.width, self.patch_size))
                ops.patch_resblock_bwd_ordered(buf, g.is_u8, g.n_frames, g.height, g.width, self.patch_size, rb.mid_channels, rb.num_groups,
                                               rb.conv1.weight, rb.conv1.bias, rb.gn2.weight, rb.gn2.bias, rb.conv2.weight, stats, dpatch,
                                               G(pp + "conv1.weight"), G(pp + "conv1.bias"), G(pp + "gn2.weight"), G(pp + "gn2.bias"),
                                               G(pp + "conv2.weight"), G(pp + "conv2.bias"), ws)
                self.launches += 6
                continue
            check(lib.neko_patch_resblock_bwd(_p(buf), C.c_int(int(g.is_u8)), C.c_int(g.n_frames), C.c_int(g.height), C.c_int(g.width),
                                              C.c_int(self.patch_size), C.c_int(rb.mid_channels), C.c_int(rb.num_groups),
                                              _p(rb.conv1.weight), _p(rb.conv1.bias), _p(rb.gn2.weight), _p(rb.gn2.bias),
                                              _p(rb.conv2.weight), _p(stats), _p(dpatch), _p(G(pp + "conv1.weight")),
                                              _p(G(pp + "conv1.bias")), _p(G(pp + "gn2.weight")), _p(G(pp + "gn2.bias")),
                                              _p(G(pp + "conv2.weight")), _p(G(pp + "conv2.bias")), stream_ptr()),
                  "neko_patch_resblock_bwd")
            self.launches += 6

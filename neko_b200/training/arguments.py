"""Command-line surface of the reference's train.py (gato/training/arguments.py:4-138): every hot-path flag with
the reference's name, default and meaning, parsed with plain argparse.  `-k` is accepted as an alias of
`--sequence_length` (as in eval.py:142; the README still documents it) and `-w` of `--use_wandb`.  Boolean flags
accept both `--flag` and `--flag true|false` (typed_argparser.py:194-209)."""
from __future__ import annotations

import argparse
from dataclasses import dataclass, field, fields
from typing import List, Optional


@dataclass
class TrainingArgs:
    # accelerate / device
    cpu: bool = False
    device: str = "cuda"
    mixed_precision: str = "no"
    # input / tokenisation
    sequence_length: int = 1024
    patch_size: int = 16
    resid_mid_channels: int = 128
    num_groups: int = 32
    patch_position_vocab_size: int = 128
    disable_patch_pos_encoding: bool = False
    disable_inner_pos_encoding: bool = False
    mu: int = 100
    M: int = 256
    continuous_tokens: int = 1024
    discrete_tokens: int = 1024
    # transformer
    tokenizer_model_name: str = "gpt2"
    pretrained_lm: Optional[str] = None
    flash: bool = False
    init_checkpoint: Optional[str] = None
    embed_dim: int = 768
    layers: int = 8
    heads: int = 24
    activation_fn: str = "gelu"
    # training
    text_prop: float = 0.0
    caption_prop: float = 0.0
    vqa_prop: float = 0.0
    gradient_accumulation_steps: int = 1
    batch_size: int = 512
    dropout: float = 0.1
    beta_1: float = 0.9
    beta_2: float = 0.95
    adam_eps: float = 1e-8
    weight_decay: float = 0.1
    grad_norm_clip: float = 1.0
    disable_grad_clip: bool = False
    warmup_steps: int = 15000
    init_lr: float = 1e-7
    learning_rate: float = 1e-4
    min_factor: float = 10.0
    disable_cosine_decay: bool = False
    training_steps: int = 1_000_000
    log_eval_freq: int = 100_000
    pad_seq: bool = False
    # datasets (accepted for CLI compatibility; the synthetic tasks ignore them)
    control_datasets: List[str] = field(default_factory=list)
    text_datasets: List[str] = field(default_factory=list)
    text_datasets_paths: List[str] = field(default_factory=list)
    caption_dataset: str = ""
    vqa_dataset: str = ""
    prompt_ep_proportion: float = 0.25
    prompt_len_proportion: float = 0.5
    # logging / saving
    use_wandb: bool = False
    wandb_project: str = "gato-control"
    save_model: bool = False
    save_mode: str = "last"
    save_dir: str = "models"
    # synthetic-data additions of this repo (no datasets / simulators offline)
    synthetic: str = "cfg2"
    disable_cuda_graphs: bool = False   # replay forward / backward from CUDA graphs per batch shape (neko_b200 engine knob)
    pack_sequences: bool = False        # padding-free steps: samples back to back, variable-length attention (neko_b200 engine knob)
    deterministic: bool = False         # bitwise-reproducible steps: fixed-order reductions in place of float atomics (engine knob)
    seed: int = 1234


def _str2bool(v):
    if isinstance(v, bool):
        return v
    if v.lower() in ("yes", "true", "t", "y", "1"):
        return True
    if v.lower() in ("no", "false", "f", "n", "0"):
        return False
    raise argparse.ArgumentTypeError(f"Truthy value expected: got {v}")


def build_parser() -> argparse.ArgumentParser:
    ap = argparse.ArgumentParser(description="neko_b200 train.py (reference flag names)")
    for f in fields(TrainingArgs):
        names = ["--" + f.name]
        if f.name == "sequence_length":
            names.append("-k")
        if f.name == "use_wandb":
            names.append("-w")
        default = f.default if f.default is not field else None
        if f.type in ("bool", bool):
            ap.add_argument(*names, type=_str2bool, nargs="?", const=True, default=f.default)
        elif str(f.type).startswith("List"):
            ap.add_argument(*names, nargs="+", default=[])
        elif str(f.type).startswith("Optional"):
            ap.add_argument(*names, default=None)
        else:
            ap.add_argument(*names, type=type(default), default=default)
    return ap


def parse_args(argv=None) -> TrainingArgs:
    # the README writes `-k=240`: argparse handles `-k 240`, `-k=240` and `--sequence_length=240`
    ns = build_parser().parse_args(argv)
    args = TrainingArgs(**vars(ns))
    assert 0.0 <= args.text_prop + args.caption_prop + args.vqa_prop <= 1.0, "task proportions must sum to <= 1"
    return args

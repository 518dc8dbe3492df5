#!/usr/bin/env python
"""train.py with the reference's flags (gato/training/arguments.py), running the B200-native hot path.

  python train.py --embed_dim=768 --layers=6 --heads=24 -k=240 --batch_size=32 --dropout=0 --training_steps=20 \
                  --log_eval_freq=10 --synthetic cfg2
  torchrun --nproc-per-node 8 --master-addr 127.0.0.1 train.py ... (one rank per GPU, NCCL)

Datasets / simulators are not available offline: tasks are the synthetic stand-ins of neko_b200.tasks with the
reference's dict contract; `--text_prop/--caption_prop/--vqa_prop` mix them exactly like trainer.py:134-154."""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from neko_b200 import dp  # noqa: E402
from neko_b200.policy import GatoPolicy  # noqa: E402
from neko_b200.tasks import build_synthetic_tasks  # noqa: E402
from neko_b200.training import Trainer, parse_args  # noqa: E402
from neko_b200.training.trainer import FusedAdamW, save_checkpoint  # noqa: E402


def main():
    args = parse_args()
    import torch.distributed as dist
    rank, world, local = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.manual_seed(args.seed)            # identical initial weights on every rank (and broadcast below)
    model = GatoPolicy(device=f"cuda:{local}", embed_dim=args.embed_dim, layers=args.layers, heads=args.heads, dropout=args.dropout,
                       mu=args.mu, M=args.M, activation_fn=args.activation_fn, patch_size=args.patch_size,
                       resid_mid_channels=args.resid_mid_channels, continuous_tokens=args.continuous_tokens,
                       discrete_tokens=args.discrete_tokens, context_len=args.sequence_length,
                       use_pos_encoding=not args.disable_inner_pos_encoding, use_patch_pos_encoding=not args.disable_patch_pos_encoding,
                       pretrained_lm=args.pretrained_lm, flash=args.flash, tokenizer_model_name=args.tokenizer_model_name, pad_seq=args.pad_seq)
    if args.init_checkpoint:
        model.load_state_dict(torch.load(args.init_checkpoint, map_location=f"cuda:{local}"))
    # embedding dropout stays at the reference's 0.1 whatever --dropout says (GPT2Config.embd_pdrop default, SURVEY quirk 8)
    if args.flash and rank == 0:
        print("--flash: no effect here -- attention never materialises the S x S scores (csrc/attention*.cu); the reference's "
              "flag only switches its own matmul/softmax path to F.scaled_dot_product_attention (trajectory_gpt2.py:241-250)")
    model.materialize_logits = False   # the trainer discards logits (trainer.py:178)
    model.use_cuda_graphs = not args.disable_cuda_graphs
    model.pack_sequences = args.pack_sequences
    model.deterministic = args.deterministic   # before dp.attach: it refuses an exchange without a fixed summation order
    torch.manual_seed(args.seed + rank)     # per-rank dropout masks, patch-position draws and multinomial remainders
    sync = None
    if world > 1:
        dp.broadcast_parameters(model)
        # a mix without text / caption / VQA never touches the text rows of embed_token on any rank (trainer.py:134)
        sync = dp.attach(model, no_text_tokens=(args.text_prop + args.caption_prop + args.vqa_prop) == 0)
    if rank == 0:
        print("Trainable Parameters:", "{}M".format(sum(p.numel() for p in model.parameters()) / 1e6))
    opt = FusedAdamW(model, lr=args.learning_rate, betas=(args.beta_1, args.beta_2), eps=args.adam_eps, weight_decay=args.weight_decay)
    tasks = build_synthetic_tasks(args.synthetic, seed=args.seed + rank, pin=True)
    trainer = Trainer(model, opt, tasks, args, sync=sync)
    model.train()
    iters = max(1, args.training_steps // max(1, args.log_eval_freq))
    for it in range(iters):
        out = trainer.train(min(args.log_eval_freq, args.training_steps))
        if rank == 0:
            losses = [l for l, _ in out]
            print(f"iteration {it}: steps {trainer.steps} train_loss_mean {sum(losses) / len(losses):.4f} lr {out[-1][1]['training/learning_rate']:.3e}")
    if args.save_model and rank == 0:
        save_checkpoint(model, os.path.join(args.save_dir, "neko_b200"), f"checkpoint_{trainer.steps}", args, optimizer=opt,
                        step=trainer.steps)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()

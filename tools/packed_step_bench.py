"""Padded against packed (GatoPolicy.pack_sequences) lean training steps at the BASELINE model (d 768, L 6, H 24).

The step is the one train.py runs: materialize_logits = False, CUDA graphs on, forward + backward, dropout 0 (embedding
dropout included).  Both arms share one policy and its weights and alternate in blocks inside one process, so clock and
co-tenant drift hit both alike.  Workloads: cfg5 (mixed multimodal, 40% padding), its text + caption samples alone, and
cfg2 (no padding: packing must cost nothing there).

  python tools/packed_step_bench.py [--steps 60] [--warmup 6] [--block 10] [--out FILE]
"""
import argparse
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import gato_oracle as O  # noqa: E402  (synthetic batch shapes of BASELINE.json)


def workloads():
    cfg5 = O.synth_batch("cfg5")
    return [("cfg5", cfg5, 1024), ("text+caption", cfg5[:24], 1024), ("cfg2", O.synth_batch("cfg2"), 240)]


def card():
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                            text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        pl = "unknown"
    return name, pl or "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=60, help="timed steps per arm")
    ap.add_argument("--warmup", type=int, default=6, help="untimed steps per arm (eager, capture, replays)")
    ap.add_argument("--block", type=int, default=10, help="consecutive steps of one arm before switching")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("packed_step_bench needs a CUDA device")
    from neko_b200.policy import GatoPolicy

    class _Tok:
        vocab_size = 50257

    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)

    name, pl = card()
    say(f"card: {name}, power limit {pl}")
    say(f"model: d 768, L 6, H 24; lean step (materialize_logits False), CUDA graphs on, dropout 0; "
        f"{a.steps} timed steps per arm in blocks of {a.block}, after {a.warmup} warm-up steps per arm")
    torch.manual_seed(0)
    for wl, batch, ctx in workloads():
        m = GatoPolicy(device="cuda:0", embed_dim=768, layers=6, heads=24, dropout=0.0, context_len=ctx, resid_mid_channels=128,
                       text_tokenizer=_Tok())
        m.transformer.drop.p = 0.0
        m.materialize_logits = False
        m.use_cuda_graphs = True
        m.eval()                       # deterministic patch positions: both arms see the same inputs

        def step(packed):
            m.pack_sequences = packed
            m.zero_grad()
            _, loss = m(batch, compute_loss=True)
            loss.backward()
            return loss

        for packed in (False, True):
            for _ in range(a.warmup):
                step(packed)
        torch.cuda.synchronize()
        ms = {False: [], True: []}
        done = {False: 0, True: 0}
        while min(done.values()) < a.steps:
            for packed in (False, True):
                n = min(a.block, a.steps - done[packed])
                evs = []
                for _ in range(n):
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    step(packed)
                    e1.record()
                    evs.append((e0, e1))
                torch.cuda.synchronize()
                ms[packed] += [e0.elapsed_time(e1) for e0, e1 in evs]
                done[packed] += n
        res = {}
        for packed in (False, True):
            loss = step(packed).item()
            torch.cuda.synchronize()
            grads = {n: p.grad.detach().double().flatten().clone() for n, p in m.named_parameters() if p.grad is not None}
            res[packed] = (loss, grads)
        cos = []
        for n, g0 in res[False][1].items():
            g1 = res[True][1][n]
            den = float(g0.norm() * g1.norm())
            if den > 0:
                cos.append((float(g0 @ g1) / den, n))
        plan = m._last_drop[1]
        n_valid, B, S = plan.n_valid_tokens, plan.B, plan.seq_len
        say(f"\n[{wl}] B {B}, S {S}: rows padded {B * S}, packed {n_valid} (valid share {n_valid / (B * S):.3f})")
        for packed in (False, True):
            t = np.array(ms[packed])
            med = float(np.median(t))
            say(f"  {'packed' if packed else 'padded'}: {med:.3f} ms/step median (mean {t.mean():.3f}, p10 {np.percentile(t, 10):.3f}, "
                f"p90 {np.percentile(t, 90):.3f}), {n_valid / med * 1e3:,.0f} valid tokens/s, loss {res[packed][0]:.6f}")
        mp, md = float(np.median(ms[True])), float(np.median(ms[False]))
        worst = min(cos)
        say(f"  packed / padded: {mp / md:.3f} ({(1 - mp / md) * 100:+.1f}% step time saved); loss rel diff "
            f"{abs(res[True][0] - res[False][0]) / abs(res[False][0]):.2e}; min gradient cosine {worst[0]:.6f} ({worst[1]})")
        del m
        torch.cuda.empty_cache()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()

"""Default against deterministic (GatoPolicy.deterministic) lean training steps at the BASELINE model (d 768, L 6, H 24).

The step is the one train.py runs: materialize_logits = False, CUDA graphs on, forward + backward, dropout 0.  Both arms share
one policy and its weights and alternate in blocks inside one process, so clock and co-tenant drift hit both alike; medians
are reported.  Workloads: cfg2 and cfg5, each padded and packed.  A separate, eager profiled pass per workload (torch.profiler,
CUDA activities) attributes the difference to kernels: the ordered reductions (and the sort of the embedding backward) against
the atomic kernels they replace, and the GEMMs (no split-K in deterministic mode).

  python tools/deterministic_step_bench.py [--steps 40] [--warmup 6] [--block 10] [--out FILE]
"""
import argparse
import os
import subprocess
import sys
from collections import defaultdict

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import gato_oracle as O  # noqa: E402  (synthetic batch shapes of BASELINE.json)

# kernel-name fragments of each reduction site, deterministic and default flavours
SITES = {
    "layernorm bwd": ("layernorm_bwd",),
    "bias colsum": ("colsum_bf16",),
    "column fold": ("ordered_colreduce",),
    "embedding bwd": ("embed_bwd_kernel", "embed_keys", "ordered_segsum", "RadixSort", "Onesweep", "radix_sort"),
    "patch bwd": ("patch_resblock_bwd", "patch_pos_bwd", "patch_pos_keys"),
    "GEMM": ("gemm_tcgen05",),
}


def card():
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                            text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        pl = "unknown"
    return name, pl or "unknown"


def site_of(kernel: str) -> str:
    for s, frags in SITES.items():
        if any(f in kernel for f in frags):
            return s
    return "other"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=40, help="timed steps per arm")
    ap.add_argument("--warmup", type=int, default=6, help="untimed steps per arm (eager, capture, replays)")
    ap.add_argument("--block", type=int, default=10, help="consecutive steps of one arm before switching")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("deterministic_step_bench needs a CUDA device")
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
        f"{a.steps} timed steps per arm in blocks of {a.block}, after {a.warmup} warm-up steps per arm; medians")
    torch.manual_seed(0)
    for wl, ctx in (("cfg2", 240), ("cfg5", 1024)):
        batch = O.synth_batch(wl)
        m = GatoPolicy(device="cuda:0", embed_dim=768, layers=6, heads=24, dropout=0.0, context_len=ctx, resid_mid_channels=128,
                       text_tokenizer=_Tok())
        m.transformer.drop.p = 0.0
        m.materialize_logits = False
        m.eval()                       # deterministic patch positions: both arms see the same inputs
        for packed in (False, True):
            m.pack_sequences = packed

            def step(det):
                m.deterministic = det
                m.zero_grad()
                _, loss = m(batch, compute_loss=True)
                loss.backward()
                return loss

            m.use_cuda_graphs = True
            for det in (False, True):
                for _ in range(a.warmup):
                    step(det)
            torch.cuda.synchronize()
            ms = {False: [], True: []}
            done = {False: 0, True: 0}
            while min(done.values()) < a.steps:
                for det in (False, True):
                    n = min(a.block, a.steps - done[det])
                    evs = []
                    for _ in range(n):
                        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                        e0.record()
                        step(det)
                        e1.record()
                        evs.append((e0, e1))
                    torch.cuda.synchronize()
                    ms[det] += [e0.elapsed_time(e1) for e0, e1 in evs]
                    done[det] += n
            res = {}
            for det in (False, True):
                loss = step(det).item()
                torch.cuda.synchronize()
                res[det] = (loss, {n: p.grad.detach().double().flatten().clone() for n, p in m.named_parameters() if p.grad is not None})
            cos = min((float(g0 @ res[True][1][n]) / float(g0.norm() * res[True][1][n].norm()), n)
                      for n, g0 in res[False][1].items() if float(g0.norm()) > 0)
            say(f"\n[{wl} {'packed' if packed else 'padded'}]")
            for det in (False, True):
                t = np.array(ms[det])
                say(f"  {'deterministic' if det else 'default      '}: {np.median(t):.3f} ms/step median (p10 {np.percentile(t, 10):.3f}, "
                    f"p90 {np.percentile(t, 90):.3f}), loss {res[det][0]:.6f}")
            md, mt = float(np.median(ms[False])), float(np.median(ms[True]))
            say(f"  deterministic / default: {mt / md:.3f} ({(mt / md - 1) * 100:+.1f}%); loss rel diff "
                f"{abs(res[True][0] - res[False][0]) / abs(res[False][0]):.2e}; min gradient cosine {cos[0]:.7f} ({cos[1]})")
            # per-site device time, eager steps under the profiler (separate from the timed window)
            m.use_cuda_graphs = False
            per = {}
            for det in (False, True):
                step(det)
                torch.cuda.synchronize()
                with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
                    for _ in range(3):
                        step(det)
                    torch.cuda.synchronize()
                acc = defaultdict(float)
                for ev in prof.key_averages():
                    t = getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0.0)
                    acc[site_of(ev.key)] += t / 3 / 1e3
                per[det] = acc
            say("  device ms/step by site (eager, profiled):  site: default -> deterministic")
            for s in list(SITES) + ["other"]:
                say(f"    {s:14s}: {per[False][s]:7.3f} -> {per[True][s]:7.3f}  ({per[True][s] - per[False][s]:+.3f})")
        del m
        torch.cuda.empty_cache()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()

#!/usr/bin/env python
"""Headline benchmark: Gato training step (GatoPolicy.forward + backward + masked loss) in tokens/s.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--config cfg2] [--impl ours|reference] [--only] [--dump-outputs DIR]

One "step" = one fwd+bwd pass of the hot path over one synthetic batch of the named BASELINE.json config
(default cfg2 = configs[1]: MuJoCo 3-task control, d768 L6 H24, batch 32, k=240).  N>1: launched by torchrun,
one rank per GPU, every rank processes its own batch (weak scaling, like the reference where every rank samples
its own --batch_size); gradients are averaged over the ranks inside backward by the copy-engine all-reduce over
peer-mapped arenas (neko_b200/dp.py, csrc/p2p_allreduce.cu), after `dp_grad_check` has compared that path with the
all-gathered mean of the local gradients.

Rank 0 prints ONE JSON line.  `value` = tokens/s with the batch already resident in HBM (CUDA-event timed, max
over ranks); `e2e` = the same step driven from pinned HOST tensors through the public API, with the H2D copy of
the batch and the D2H read of the loss inside the timed region; `roofline` = the tensor-core GEMM kernel (the
dominant kernel): algorithmic FLOPs of every GEMM launch / CUDA-event time of those launches (queued behind a
blocker kernel, so the events see no launch latency), against the measured bf16 BURST peak (`frac_sustained` beside
it) with the per-shape table in `roofline.shapes`; `front_end` = tokeniser / image stack against the measured HBM copy
bandwidth; `configs` = the same measurements for cfg3 / cfg4 / cfg5 (the configurations BASELINE.json names for the
scaling claim), at every N; `cpu_baseline` / `--impl reference` = the UNMODIFIED reference (oracle/_ref, placed there by
oracle/build_ref.py) on this host's cores (the oracle port only when no reference tree is present).

`--dump-outputs DIR` (rank 0): what the last timed step of --config returned to its caller, as DIR/<name>.npy (see
sample_outputs).  Inputs and weights are seeded, so two builds run with the same arguments can be compared array by array.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SMI_QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

WORKLOADS = {
    "cfg1": "GatoPolicy d128 L3 H1, HalfCheetah-shaped continuous control (obs 17, act 6), k=240, batch 4",
    "cfg2": "MuJoCo 3-task control (halfcheetah/hopper/walker2d shapes) d768 L6 H24, k=240, batch 32/GPU",
    "cfg3": "Atari Breakout-shaped image control (96x96 frames, 16x16 patches, ResNet patch embed) d768 L6 H24, k=512, batch 32/GPU",
    "cfg4": "text-only GPT-2-vocab LM d768 L6 H24, 1023 ids + separator, batch 16/GPU",
    "cfg5": "mixed multimodal batch (text + control + Atari + 224x224 caption/VQA) d768 L6 H24, k=1024, batch 32/GPU",
}


def peaks():
    """(bf16 burst TFLOP/s, bf16 sustained TFLOP/s, HBM GB/s, source)."""
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("bf16_tflops", 1590.0), d.get("bf16_tflops_sustained", 1400.0), d.get("hbm_gbs", 6650.0), "measured (MEASURED_PEAKS.json)"
    return 1590.0, 1400.0, 6650.0, "fallback (B200_PROFILING.md)"


def gemm_traffic(args, cfg_name, launches_per_step):
    """dram__bytes_read.sum + dram__bytes_write.sum per GEMM launch from the committed ncu capture of this very command
    (tools/gemm_traffic.sh -> profiles/r0N_gemm_traffic_<cfg>.json); None when no capture matches the configuration."""
    p = next((q for q in (os.path.join(ROOT, "profiles", f"r02_gemm_traffic_{cfg_name}.json"),
                          os.path.join(ROOT, "profiles", f"r01_gemm_traffic_{cfg_name}.json")) if os.path.exists(q)), None)
    if args.lean or args.head != "rows" or p is None:
        return None
    d = json.load(open(p))
    if d.get("launches") != launches_per_step:
        return None
    return round(d["dram_bytes_per_launch"])


def gemm_flops_per_step(cfg, N, S, n_rows, head_mode, materialize):
    """Algorithmic GEMM FLOPs actually launched on the tensor-core kernel in one fwd+bwd."""
    d, L, V = cfg["embed_dim"], cfg["layers"], 52352
    blocks = 3 * L * 24 * N * d * d          # 4 linears fwd + dgrad + wgrad
    head_fwd = 2 * (N if materialize else n_rows) * d * V
    head_bwd = 4 * (n_rows if (head_mode == "rows" or not materialize) else N) * d * V
    return float(blocks + head_fwd + head_bwd)


def model_flops_per_step(cfg, N, S):
    """SURVEY.md section 8(d): fwd = L(24 N d^2 + 2 N S d) + 2 N d V (attention causal-half); fwd+bwd = 3x."""
    d, L, V = cfg["embed_dim"], cfg["layers"], 52305
    return 3.0 * (L * (24 * N * d * d + 2 * N * S * d) + 2 * N * d * V)


# ---------------------------------------------------------------------------------------------------------
# CPU arm (oracle port): used for cpu_baseline and for --impl reference
# ---------------------------------------------------------------------------------------------------------
def _cpu_step_fn(config: str, n_samples):
    """(step(), tokens per step, kind, n_samples).  kind "reference": the UNMODIFIED reference (GatoPolicy of
    gato/policy/gato_policy.py, imported from /root/reference or from the git-ignored copy oracle/build_ref.py placed under
    oracle/_ref/, through the in-memory shims of oracle/ref_shim.py) -- model(batch, compute_loss=True); loss.backward() on
    the host cores, fp32, dropout 0.  kind "port": the oracle restatement, only when no reference tree is present."""
    from oracle import gato_oracle as O
    from oracle import ref_shim
    torch.set_num_threads(os.cpu_count() or 1)
    cfg = O.GatoConfig(**O.CONFIGS[config])
    w = O.make_weights(cfg, seed=0, perturb=False)
    batch = O.synth_batch(config, seed=1234, batch=n_samples)
    tokens = int(O.tokenize(batch, cfg).token_masks.sum())
    G = None
    if ref_shim.reference_available():
        try:
            ref_shim.set_text_vocab(cfg.text_tokens)
            G = ref_shim.load_reference_policy_class()
        except Exception as e:  # noqa: BLE001 -- e.g. a transformers version the shims do not cover: time the port instead
            print(f"reference import failed ({type(e).__name__}: {e}); timing the oracle port", file=sys.stderr)
            G = None
    if G is not None:
        m = G(device="cpu", embed_dim=cfg.embed_dim, layers=cfg.layers, heads=cfg.heads, dropout=0.0, resid_mid_channels=128,
              context_len=cfg.context_len)
        m.transformer.drop.p = 0.0
        m.load_state_dict(w, strict=False)
        m.train()

        def step():
            m.zero_grad(set_to_none=True)
            _logits, loss = m(batch, compute_loss=True)
            loss.backward()
            return float(loss.detach())
        return step, tokens, "reference", len(batch)
    for t in w.values():
        t.requires_grad_(True)

    def step():
        for t in w.values():
            t.grad = None
        out = O.forward(w, batch, cfg, compute_loss=True)
        out.loss.backward()
        return float(out.loss.detach())
    return step, tokens, "port", len(batch)


def cpu_tokens_per_s(config: str, n_samples, steps: int, warmup: int, budget_s: float):
    """Times the CPU arm: `warmup` untimed steps, then up to `steps` timed ones, stopping early once `budget_s` seconds of
    timed work are spent (at least one timed step)."""
    step, tokens, kind, nb = _cpu_step_fn(config, n_samples)
    for _ in range(warmup):
        step()
    times = []
    for _ in range(steps):
        t0 = time.perf_counter()
        step()
        times.append(time.perf_counter() - t0)
        if sum(times) >= budget_s:
            break
    sec = sum(times) / len(times)
    return tokens / sec, tokens, sec, kind, nb, len(times)


def run_reference(args):
    """`--impl reference`: the reference's own CPU implementation of the path on this box's host cores, on the FULL batch of
    the configuration (oracle port on the same batch only if no reference tree is present)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # K and W are honoured up to a time budget that keeps the whole run within a few minutes (one full-batch fwd+bwd is
    # 2-30 s of CPU work depending on the configuration)
    tps, tokens, sec, kind, nb, done = cpu_tokens_per_s(args.config, None, max(1, args.steps), max(1, min(args.warmup, 2)), 150.0)
    cores = os.cpu_count() or 1
    desc = (f"fwd+bwd over the full {args.config} batch ({nb} samples, {tokens} tokens) per step, fp32 torch-CPU, {cores} threads, "
            f"{done} timed steps (time-capped) after {max(1, min(args.warmup, 2))} warm-up; "
            + ("unmodified reference GatoPolicy from oracle/_ref or /root/reference" if kind == "reference" else "oracle port (no reference tree present)"))
    print(json.dumps({
        "impl": "reference", "metric": "train tokens/sec (fwd+bwd)", "value": round(tps, 2), "unit": "tokens/s", "n_gpus": args.gpus,
        "steps": done, "warmup": max(1, min(args.warmup, 2)), "ms_per_step": round(sec * 1e3, 3), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOADS[args.config], "name": args.config, "tokens_per_step_per_gpu": tokens, "same_config": True},
        "cpu_baseline": {"value": round(tps, 2), "unit": "tokens/s", "cores": cores, "kind": kind, "sample": desc},
        "e2e": {"value": round(tps, 2), "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }), flush=True)


# ---------------------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------------------
def to_device(batch, dev):
    out = []
    for s in batch:
        out.append({k: (v.to(dev) if isinstance(v, torch.Tensor) else v) for k, v in s.items()})
    return out


def to_pinned(batch):
    out = []
    for s in batch:
        d = {}
        for k, v in s.items():
            if isinstance(v, list):
                v = torch.tensor(v, dtype=torch.int64)
            d[k] = v.pin_memory() if isinstance(v, torch.Tensor) else v
        out.append(d)
    return out


def batch_bytes(batch):
    n = 0
    for s in batch:
        for v in s.values():
            if isinstance(v, torch.Tensor):
                n += v.numel() * (4 if v.dtype in (torch.int64,) else v.element_size())  # ids cross as int32
            elif isinstance(v, list):
                n += 4 * len(v)
    return n


def parse_clocks(path):
    sm, mx, reasons = [], [], set()
    try:
        for line in open(path):
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9 or not f[0].isdigit():
                continue
            sm.append(float(f[1].split()[0]))
            mx.append(float(f[2].split()[0]))
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
    except OSError:
        pass
    if not sm:
        return {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
    busy = sorted(sm)[len(sm) // 2:]  # the upper half of the samples = under load
    return {"sm_mhz": float(np.median(busy)), "sm_max_mhz": max(mx), "reasons": sorted(reasons)}


def front_end_roofline(model, host_batch, dev, cfgd, cfg_name):
    """SURVEY.md section 8(d)(ii): tokenise + embed + interleave + pad kernel against the measured HBM copy bandwidth.

    Algorithmic bytes per valid token = d*4 (table / patch-embedding row read) + d*4 (embedding written) + 16 (int64 id, two
    fp32 masks) + 4 (input scalar).  Timed alone with CUDA events: once at the config's batch (L2 flushed before every
    launch: the ~50 MB working set would otherwise sit in the 126 MB L2) and once at a batch replicated to >= 1 GB of
    traffic (larger than L2, no flush needed).  The image stack (patchify + ResNet block + projection + position add) is
    timed the same way when the batch has frames: bytes per patch = 768 * s_in + d*4."""
    import torch
    from neko_b200.policy.packing import build_plan
    _tf, _ts, hbm, src = peaks()
    d = cfgd["embed_dim"]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    res = {"bound": "hbm", "peak": hbm, "unit": "GB/s", "peak_source": src, "bytes_per_token": d * 8 + 20}

    def timed(fn, iters, do_flush):
        ts = []
        for _ in range(iters):
            if do_flush:
                flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            torch.cuda.synchronize()
            ts.append(a.elapsed_time(b))
        ts.sort()
        return ts[len(ts) // 2]

    was_training = model.training
    model.eval()
    with torch.no_grad():
        for tag, reps in (("config_batch", 1), ("scaled_batch", None)):
            batch = list(host_batch)
            plan = build_plan(batch, patch_size=16, context_len=cfgd["context_len"], pad_seq=False)
            if reps is None:
                reps = max(1, -(-(1 << 30) // (plan.n_valid_tokens * (d * 8 + 20))))
                reps = min(reps, 64)
                base = batch
                batch = []
                for r in range(reps):      # text replicas get fresh ids: the scaled batch must not shrink to one L2-resident set of rows
                    for si, smp in enumerate(base):
                        if r and isinstance(smp.get("text"), (list, torch.Tensor)) and "images" not in smp:
                            n_ids = len(smp["text"]) if isinstance(smp["text"], list) else int(smp["text"].numel())
                            smp = dict(smp, text=np.random.RandomState(1000 + 997 * r + si).randint(0, 50257, size=(n_ids,)).tolist())
                        batch.append(smp)
            st = model._plan(batch, False)
            st.need_grad = False
            model._embed(st)     # uploads, image stack, first launch
            torch.cuda.synchronize()
            ntok = st.plan.n_valid_tokens
            ms = timed(lambda: model._launch_tokenize(st), 10, reps == 1)
            gbs = ntok * (d * 8 + 20) / (ms * 1e-3) / 1e9
            wgbs = ntok * (d * 4 + 16) / (ms * 1e-3) / 1e9
            # the d*4 table-row read per token reaches HBM only when the distinct rows of the batch exceed the L2 (126 MB):
            # cfg2 touches ~2 k rows (6 MB, L2 hits), cfg4 ~50 k rows (154 MB, real HBM traffic)
            distinct = int(torch.unique(st.tokens[:st.plan.B * st.plan.width]).numel())
            table_mb = distinct * d * 4 / 1e6
            l2_table = table_mb < 100.0
            res[tag] = {"samples": len(batch), "tokens": int(ntok), "kernel": "tokenize_embed_kernel", "us": round(ms * 1e3, 2),
                        "achieved": round(wgbs if l2_table else gbs, 1), "frac": round((wgbs if l2_table else gbs) / hbm, 4),
                        "counts": ("writes only (embedding row + id + masks): the table rows are L2 hits" if l2_table
                                   else "algorithmic bytes (table row read + embedding row written + id + masks)"),
                        "achieved_algorithmic": round(gbs, 1), "frac_algorithmic": round(gbs / hbm, 4),
                        "achieved_writes_only": round(wgbs, 1), "frac_writes_only": round(wgbs / hbm, 4),
                        "distinct_table_rows": distinct, "table_mb": round(table_mb, 1),
                        "l2": "flushed before each launch" if reps == 1 else "working set > L2"}
            if st.plan.n_patch_rows and getattr(st, "img_groups", None):
                P = int(st.plan.n_patch_rows)
                s_in = 1 if all(g.is_u8 for g in st.plan.image_groups if g.tensors) else 4
                ims = timed(lambda: model._image_compute(st), 10, reps == 1)
                igb = P * (768 * s_in + d * 4) / (ims * 1e-3) / 1e9
                res[tag]["image_stack"] = {"patches": P, "kernels": "patch_resblock_fwd_kernel + projection GEMM + patch_pos_add_kernel",
                                           "us": round(ims * 1e3, 2), "bytes_per_patch": 768 * s_in + d * 4, "achieved": round(igb, 1),
                                           "frac": round(igb / hbm, 4),
                                           "tflops": round(P * 2 * (27 * 128 * 256 + 9 * 128 * 3 * 256 + 768 * d) / (ims * 1e-3) / 1e12, 2)}
            del st
    model.train(was_training)
    return res


def build_model(cfg_name, args, dev):
    from neko_b200.policy import GatoPolicy
    from neko_b200.tasks.synthetic import BENCH_CONFIGS
    cfgd = {k: v for k, v in BENCH_CONFIGS[cfg_name].items() if k != "batch"}

    class _Tok:
        vocab_size = 50257

    torch.manual_seed(0)
    model = GatoPolicy(device=dev, embed_dim=cfgd["embed_dim"], layers=cfgd["layers"], heads=cfgd["heads"], dropout=0.0,
                       resid_mid_channels=128, context_len=cfgd["context_len"], text_tokenizer=_Tok())
    model.transformer.drop.p = 0.0
    model.head_mode = args.head
    model.materialize_logits = not args.lean
    if "NEKO_MLP_PROJ_BF16" in os.environ:      # experiment switch: forward mlp down-projection on bf16 operands
        model.mlp_proj_bf16 = os.environ["NEKO_MLP_PROJ_BF16"] == "1"
    model.lean_logits_f16 = os.environ.get("NEKO_LEAN_F32") != "1"     # experiment switch: --lean with fp32 logits of the loss rows
    model.use_cuda_graphs = not args.no_graphs
    model.train()
    return model, cfgd


def dp_grad_check(model, sync, batch, world):
    """N > 1, before any timing: the synchroniser's result on a real gradient arena against the all-gathered mean of the
    ranks' local gradients (DDP semantics, trainer.py:176-186).  One backward per rank without synchronisation, then the
    production all-reduce path over every bucket of the arena."""
    import torch.distributed as dist
    model.zero_grad()
    with sync.no_sync():
        _, loss = model(batch, compute_loss=True)
        loss.backward()
    torch.cuda.synchronize()
    local = model._grad_arena.clone()
    gathered = [torch.empty_like(local) for _ in range(world)]
    dist.all_gather(gathered, local)
    mean = gathered[0].double()
    for g in gathered[1:]:
        mean += g.double()
    mean = (mean / world).float()
    del gathered
    sync.reduce_all()
    torch.cuda.synchronize()
    err = float((model._grad_arena - mean).abs().max())
    scale = float(mean.abs().max())
    t = torch.tensor([err], device=local.device)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    model.zero_grad()
    return {"max_abs_err": float(t[0]), "grad_abs_max": scale, "rel": float(t[0]) / max(scale, 1e-30), "backend": sync.backend,
            "what": "arena after the production all-reduce vs the fp64 mean of the all-gathered local gradient arenas, max over ranks"}


DUMP_LOGITS = 1 << 20          # sampled logits
DUMP_GRAD = 1 << 18            # elements kept of a larger gradient
DUMP_LIMIT = 64 << 20          # bytes written in all


def sample_outputs(model, logits, loss, plan):
    """Host copies of what one fwd+bwd step hands its caller: `loss`; `logits`, a sample of DUMP_LOGITS entries of the valid
    (non-padding) rows -- padding rows carry no defined values; `grad.<parameter name>` for every parameter that received a
    gradient, whole, or a sample of DUMP_GRAD entries when larger.  The sample indices come from a fixed seed and the shapes
    alone, so two builds given the same arguments sample the same entries.  Loss and logits repeat bit for bit from run to
    run; gradients summed with fp32 atomics differ in their rounding."""
    rs = np.random.RandomState(0)
    out = {"loss": loss.detach().float().cpu().numpy()}
    if logits is not None and logits.numel():
        rows = np.concatenate([b * plan.width + np.arange(plan.first_valid[b], plan.seq_len) for b in range(plan.B)])
        r = rows[rs.randint(0, rows.shape[0], DUMP_LOGITS)]
        c = rs.randint(0, logits.shape[-1], DUMP_LOGITS)
        bi, si, ci = (torch.from_numpy(a).to(logits.device) for a in (r // plan.width, r % plan.width, c))
        out["logits"] = logits[bi, si, ci].float().cpu().numpy()
    for name, p in model.named_parameters():
        if p.grad is None:
            continue
        g = p.grad.detach().reshape(-1)
        if g.numel() > DUMP_GRAD:
            g = g[torch.from_numpy(np.sort(rs.randint(0, g.numel(), DUMP_GRAD))).to(g.device)]
        out["grad." + name] = g.float().cpu().numpy()
    total = sum(a.nbytes for a in out.values())
    assert total <= DUMP_LIMIT, f"output dump of {total} bytes exceeds {DUMP_LIMIT}"
    return out


def write_outputs(directory, arrays):
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(directory, name + ".npy"), a)


def measure_config(cfg_name, args, dev, rank, world, local, headline):
    """One BASELINE.json configuration: W warm-up + K timed fwd+bwd steps (HBM-resident batch), the GEMM roofline pass, and the
    end-to-end loop from pinned host memory.  Returns the fields of the JSON line for this configuration."""
    import torch.distributed as dist
    from neko_b200 import dp, ops
    from neko_b200._lib import check, load
    from neko_b200.policy.packing import build_plan
    from neko_b200.tasks.synthetic import bench_batch
    import ctypes as C

    model, cfgd = build_model(cfg_name, args, dev)
    sync = None
    if world > 1:
        dp.broadcast_parameters(model)
        # static knowledge of the task mix, as a trainer has it from --text_prop / --caption_prop / --vqa_prop
        no_text = not any(("text" in s and s["text"] is not None) for s in bench_batch(cfg_name, seed=0))
        bucket_mb = int(os.environ.get("NEKO_DP_BUCKET_MB", "64"))
        sync = dp.attach(model, bucket_bytes=bucket_mb << 20, no_text_tokens=no_text, mode=os.environ.get("NEKO_DP_MODE", "overlap"),
                         compress=os.environ.get("NEKO_DP_COMPRESS", "none"), backend=os.environ.get("NEKO_DP_BACKEND", "auto"))
    host_batch = bench_batch(cfg_name, seed=1234 + rank)
    dev_batch = to_device(host_batch, dev)
    pin_batch = to_pinned(host_batch)

    def step(batch):
        model.zero_grad()          # what optimizer.zero_grad() does every step in trainer.py:186
        logits, loss = model(batch, compute_loss=True)
        loss.backward()
        return logits, loss

    plan = build_plan(host_batch, patch_size=16, context_len=cfgd["context_len"], pad_seq=False)
    tokens_per_step = plan.n_valid_tokens
    N, S, n_rows = plan.B * plan.width, plan.seq_len, int(plan.loss_rows.shape[0])
    grad_check = dp_grad_check(model, sync, dev_batch, world) if world > 1 else None

    warm = max(args.warmup, 3)
    for _ in range(warm):
        step(dev_batch)
    torch.cuda.synchronize()

    # ---- timed region 1: inputs resident in HBM --------------------------------------------------------
    clk = tempfile.NamedTemporaryFile(prefix="clocks", suffix=".csv", delete=False)
    smi = None
    if rank == 0:
        try:
            smi = subprocess.Popen(["nvidia-smi", f"--query-gpu={SMI_QUERY}", "--format=csv,noheader", "-lms", "100", "-i", str(local)],
                                   stdout=clk, stderr=subprocess.DEVNULL)
        except OSError:
            smi = None
    l0 = model.launches
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps - 1):
        step(dev_batch)
    last = step(dev_batch)         # held past the loop only: an earlier step's outputs never outlive it
    e1.record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    ms = e0.elapsed_time(e1)
    launches = model.launches - l0
    if headline and args.dump_outputs and rank == 0:
        # copied now: the passes below run the step again into the same (graph-owned) buffers
        write_outputs(args.dump_outputs, sample_outputs(model, *last, plan))
    del last

    # ---- roofline of the dominant kernel: CUDA events around every tensor-core GEMM launch.  The timed region above
    # replays the step from CUDA graphs (no room for per-launch events), so the same step is run eagerly right after it
    # with the events in place; kernels, shapes and order are identical.  The whole eager step is enqueued BEHIND a
    # blocker kernel (neko_debug_spin, one idle warp for 12 ms): when it ends the GPU runs the queue back to back, so an
    # event pair brackets its kernel and not the host's launch latency (the eager host path is slower than the GPU).
    gemm_log = []
    graphs_on = model.use_cuda_graphs
    model.use_cuda_graphs = False
    sync_was = sync.enabled if sync is not None else None
    if sync is not None:
        sync.enabled = False           # per-launch GEMM durations are measured without the all-reduce next to them
    for _ in range(2):
        step(dev_batch)
    torch.cuda.synchronize()
    ops.GEMM_TIMING = gemm_log
    inst_steps = min(args.steps, 5)
    lib = load()
    eager_ms = 0.0
    for _ in range(inst_steps):
        i0, i1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        check(lib.neko_debug_spin(C.c_int(1), C.c_int(32), C.c_longlong(12_000_000), C.c_int(1),
                                  C.c_void_p(torch.cuda.current_stream().cuda_stream)), "neko_debug_spin")
        i0.record()
        step(dev_batch)
        i1.record()
        torch.cuda.synchronize()
        eager_ms += i0.elapsed_time(i1) / inst_steps
    ops.GEMM_TIMING = None
    model.use_cuda_graphs = graphs_on
    if sync is not None:
        sync.enabled = sync_was
    gemm_ms = sum(g[0].elapsed_time(g[1]) for g in gemm_log) / inst_steps       # per step
    gemm_fl = sum(g[2] for g in gemm_log) / inst_steps

    def _alg_bytes(key):   # operands once + outputs once (+ the auxiliary read of the residual / GELU' epilogues)
        M_, N_, K_, _am, _bm, epi = key
        out = {0: 2, 1: 4, 2: 6, 3: 8, 4: 4, 5: 10}[epi]
        return 2.0 * M_ * K_ + 2.0 * N_ * K_ + float(out) * M_ * N_
    gemm_alg_bytes = sum(_alg_bytes(g[3]) for g in gemm_log) / max(len(gemm_log), 1)
    gemm_launches_per_step = len(gemm_log) // inst_steps
    peak_burst, peak_sust, _hbm, peak_src = peaks()
    agg = {}
    for g in gemm_log:
        c, t = agg.get(g[3], (0, 0.0))
        agg[g[3]] = (c + 1, t + g[0].elapsed_time(g[1]))
    epi_names = {0: "16-bit", 1: "f32", 2: "gelu x2/x3", 3: "resid f32", 4: "dgelu", 5: "resid f32+16"}
    shapes = []
    for k, (c, t) in sorted(agg.items(), key=lambda kv: -kv[1][1]):
        us = t / c * 1e3
        tf = 2.0 * k[0] * k[1] * k[2] / us / 1e6
        shapes.append({"M": k[0], "N": k[1], "K": k[2], "a_mn": k[3], "b_mn": k[4], "epilogue": epi_names[k[5]], "per_step": c // inst_steps,
                       "us": round(us, 1), "tflops": round(tf, 1), "frac_burst": round(tf / peak_burst, 3)})
    if args.gemm_report and rank == 0:
        print(f"GEMM report {cfg_name} (M, N, K, a_mn, b_mn, epilogue): launches/step, avg us, TFLOP/s, frac of burst peak", file=sys.stderr)
        for sh in shapes:
            print(f"  {sh['M']:6d} {sh['N']:6d} {sh['K']:6d} {sh['a_mn']} {sh['b_mn']} {sh['epilogue']:14s} {sh['per_step']:3d} {sh['us']:9.1f} "
                  f"{sh['tflops']:8.1f} {sh['frac_burst']:6.3f}", file=sys.stderr)

    # ---- timed region 2: end to end from pinned host tensors ---------------------------------------------
    # warm the staged pipeline itself (its incoming-frame buffers are allocated on first use, which re-captures the graphs),
    # then drain it so that every copy of the timed steps is issued inside the timed region
    nxt = model.stage(pin_batch, compute_loss=True)
    for _ in range(3):
        _, loss = step(nxt)
        nxt = model.stage(pin_batch, compute_loss=True)
        loss.item()
    step(nxt)[1].item()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    # the batch producer: the NEXT step's host planning + pinned->device copy are issued before the loss of the current
    # step is read (model.stage), as a prefetching loader would; every step still carries its own H2D copy and D2H read
    t0 = time.perf_counter()
    f0.record()
    nxt = model.stage(pin_batch, compute_loss=True)
    for k in range(args.steps):
        _, loss = step(nxt)
        if k + 1 < args.steps:
            nxt = model.stage(pin_batch, compute_loss=True)
        loss.item()              # the D2H read of the loss closes every step
    f1.record()
    torch.cuda.synchronize()
    wall_ms = (time.perf_counter() - t0) * 1e3
    e2e_ms = max(f0.elapsed_time(f1), wall_ms)
    if smi is not None:
        smi.terminate()
        smi.wait()
    clk.close()

    t = torch.tensor([ms, e2e_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, e2e_ms = float(t[0]), float(t[1])
    clocks = parse_clocks(clk.name)
    try:
        os.unlink(clk.name)
    except OSError:
        pass
    tps = tokens_per_step * world * args.steps / (ms / 1e3)
    e2e_tps = tokens_per_step * world * args.steps / (e2e_ms / 1e3)
    achieved = gemm_fl / (gemm_ms / 1e3) / 1e12 if gemm_ms > 0 else None
    out = {
        "value": round(tps, 1), "unit": "tokens/s", "ms_per_step": round(ms / args.steps, 4),
        "config": {"workload": WORKLOADS[cfg_name], "name": cfg_name, "tokens_per_step_per_gpu": tokens_per_step,
                   "padded_positions": N, "loss_rows": n_rows, "head": ("loss-rows only (lean)" if args.lean else f"dense logits, {args.head} backward"),
                   "l2_policy": "per-step activations (>1.6 GB logits alone) exceed the 126 MB L2; no explicit flush",
                   "parallelism": f"dp{world}", "cuda_graphs": bool(model.use_cuda_graphs), "model_tflop_per_step_dense": round(model_flops_per_step(cfgd, N, S) / 1e12, 3),
                   "dropout": "0 (attention / residual / embedding), so the step is comparable with the fp32 reference arm; the reference's "
                              "default is 0.1 -- the counter-based masks cost < 1 % (DESIGN.md section 4)",
                   "optimizer_step": "not part of fwd+bwd (BASELINE metric); the fp32 -> fp16 / bf16 weight-copy cast that follows an optimiser "
                                     "step (~0.1 ms, fused into FusedAdamW in training) is therefore not in the timed region"},
        "clocks": clocks,
        "e2e": {"value": round(e2e_tps, 1), "unit": "tokens/s", "h2d_bytes_per_step": int(batch_bytes(host_batch) + 4096),
                "d2h_bytes_per_step": 4, "ms_per_step": round(e2e_ms / args.steps, 4),
                "pipeline": "GatoPolicy.stage(): step i+1 is planned and its pinned->device copy enqueued before step i's loss is read"},
        "gpu_launches": int(launches),
        "roofline": {"bound": "tensor", "kernel": "gemm_tcgen05_kernel (all GEMM launches of the step)",
                     "achieved": round(achieved, 1) if achieved else None, "peak": peak_burst, "unit": "TFLOP/s",
                     "frac": round(achieved / peak_burst, 4) if achieved else None,
                     "frac_burst": round(achieved / peak_burst, 4) if achieved else None,
                     "frac_sustained": round(achieved / peak_sust, 4) if achieved else None,
                     "peak_burst": peak_burst, "peak_sustained": peak_sust,
                     "traffic": gemm_traffic(args, cfg_name, gemm_launches_per_step), "traffic_unit": "DRAM bytes per GEMM launch (ncu, mean over the step's launches)",
                     "algorithmic_bytes_per_launch": round(gemm_alg_bytes), "gemm_launches_per_step": gemm_launches_per_step,
                     "peak_source": peak_src + "; frac is against the BURST figure: the timed region is ~0.1 s at full clocks",
                     "gemm_ms_per_step": round(gemm_ms, 4), "gemm_share_of_step": round(gemm_ms / eager_ms, 4),
                     "timing": "CUDA events around each GEMM launch in an eager pass of the same step run right after the timed region, every "
                               "step enqueued behind a 12 ms blocker kernel so that the events see kernel time, not launch latency "
                               f"(eager step {eager_ms:.3f} ms on the device; the timed region replays CUDA graphs)",
                     "shapes": shapes,
                     "model_flops_frac_effective": round(model_flops_per_step(cfgd, N, S) * args.steps / (ms / 1e3) / 1e12 / peak_burst, 4)},
    }
    if grad_check is not None:
        out["dp_grad_check"] = grad_check
    if world == 1 and headline and not args.no_front_end:
        out["front_end"] = front_end_roofline(model, host_batch, dev, cfgd, cfg_name)
    elif world == 1 and not args.no_front_end:
        fe = front_end_roofline(model, host_batch, dev, cfgd, cfg_name)
        out["front_end"] = {k: fe[k] for k in ("config_batch", "scaled_batch", "peak", "unit") if k in fe}
    if sync is not None:
        model.grad_ready_hook = None
        model._grad_sync = None
    del model
    torch.cuda.empty_cache()
    return out


def run_ours(args):
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    head = measure_config(args.config, args, dev, rank, world, local, headline=True)
    # the other BASELINE.json configurations named for the scaling claim (cfg3 / cfg4 at 1/2/4/8, cfg5) ride along in
    # "configs" with their own ms/step, tokens/s, e2e and GEMM roofline, at every N the driver runs
    others = {}
    if not args.only:
        for name in ("cfg3", "cfg4", "cfg5"):
            if name != args.config:
                sub = argparse.Namespace(**vars(args))
                sub.warmup = 3
                r = measure_config(name, sub, dev, rank, world, local, headline=False)
                r["steps"], r["warmup"] = sub.steps, sub.warmup
                others[name] = r
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    out = {"metric": "train tokens/sec (fwd+bwd)", "value": head["value"], "unit": "tokens/s", "n_gpus": world, "steps": args.steps,
           "warmup": max(args.warmup, 3), "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": "weak",
           "vs_baseline": None, "dtype": "fp16 fwd / bf16 bwd operands, fp32 accumulate + residual stream", "data": "synthetic"}
    out.update({k: v for k, v in head.items() if k not in ("value", "unit", "ms_per_step")})
    if others:
        out["configs"] = others
    if world == 1 and not args.no_cpu_baseline:
        # bounded sample: the first samples of the same batch, ~10-30 s of CPU work in total
        sample = {"cfg1": 4, "cfg2": 8, "cfg3": 4, "cfg4": 2, "cfg5": 5}[args.config]
        try:
            ctps, ctok, csec, kind, nb, done = cpu_tokens_per_s(args.config, sample, 3, 1, 20.0)
            out["cpu_baseline"] = {"value": round(ctps, 2), "unit": "tokens/s", "cores": os.cpu_count() or 1, "kind": kind,
                                   "sample": f"{done} timed fwd+bwd steps over {nb} samples of the {args.config} batch ({ctok} tokens/step, "
                                             f"{csec:.2f} s/step), fp32 torch-CPU, "
                                             + ("unmodified reference (oracle/_ref)" if kind == "reference" else "oracle port")}
        except Exception as e:  # noqa: BLE001 -- the CPU arm is a reported baseline: its failure must not take the GPU line with it
            out["cpu_baseline"] = {"value": None, "unit": "tokens/s", "cores": os.cpu_count() or 1, "kind": "unavailable",
                                   "sample": f"{type(e).__name__}: {str(e)[:200]}"}
    print(json.dumps(out), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--config", default="cfg2", choices=sorted(WORKLOADS))
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--head", default="rows", choices=["dense", "rows"], help="head backward: dense like the reference's autograd, or loss rows only (identical gradients)")
    ap.add_argument("--lean", action="store_true", help="evaluate the LM head on loss rows only (forward returns no logits)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-front-end", action="store_true", help="skip the tokeniser / image-stack HBM roofline pass")
    ap.add_argument("--no-graphs", action="store_true", help="launch every kernel eagerly instead of replaying the step from CUDA graphs")
    ap.add_argument("--gemm-report", action="store_true", help="per-shape GEMM timings (CUDA events) on stderr")
    ap.add_argument("--only", action="store_true", help="measure --config only (skip the cfg3 / cfg4 / cfg5 entries of \"configs\")")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step of --config returned (loss, sampled logits, "
                                                          "gradients) to DIR/<name>.npy; --impl ours only")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to --impl ours only")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()

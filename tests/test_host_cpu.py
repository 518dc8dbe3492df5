"""CPU-side tests (no GPU): C-ABI library loads and exports every declared symbol, host batch planning agrees
with the oracle, the reference-facing error behaviour of the planner, and the data-parallel bucket logic over
gloo with world_size 2."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import gato_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def built_lib():
    from neko_b200 import build
    return build.build()


def test_library_exports_every_declared_symbol(built_lib):
    from neko_b200 import _lib
    names = _lib.declared_symbols()
    assert len(names) >= 25 and "neko_gemm" in names and "neko_tokenize_embed_fwd" in names
    lib = ctypes.CDLL(built_lib)
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/neko_b200.h but not exported"
    assert _lib.load().neko_version() >= 100


def test_integration_doc_names_every_entry_point():
    """INTEGRATION.md's call-site table must cover the whole C ABI (and name nothing that does not exist)."""
    import re
    from neko_b200 import _lib
    doc = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    names = set(_lib.declared_symbols())
    missing = sorted(n for n in names if n not in doc)
    assert not missing, f"entry points absent from INTEGRATION.md: {missing}"
    types = {"neko_gemm_desc", "neko_dropout", "neko_b200"}
    unknown = sorted(w for w in set(re.findall(r"`(neko_[a-z0-9_]+)`", doc)) if w not in names and w not in types)
    assert not unknown, f"INTEGRATION.md names entry points the header does not declare: {unknown}"


def test_struct_layouts_match_header(tmp_path):
    """ctypes mirrors vs the C header, as a C compiler lays the structs out."""
    import subprocess
    from neko_b200._lib import Dropout, GemmDesc, GemmPlanInfo, SampleDesc, TokParams, HEADER
    assert ctypes.sizeof(SampleDesc) == 64
    assert ctypes.sizeof(TokParams) == 40
    assert ctypes.sizeof(Dropout) == 24
    assert ctypes.sizeof(GemmDesc) == 8 * 4 + 13 * 8 + 24 + 16
    assert ctypes.sizeof(GemmPlanInfo) == 10 * 4
    src = tmp_path / "sizes.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "neko_b200.h"\nint main(void){printf("%zu %zu %zu %zu %zu %zu %zu %zu",'
                   'sizeof(neko_sample_desc), sizeof(neko_tok_params), sizeof(neko_dropout), sizeof(neko_gemm_desc),'
                   'offsetof(neko_gemm_desc, drop), offsetof(neko_gemm_desc, aux), offsetof(neko_gemm_desc, workspace),'
                   'sizeof(neko_gemm_plan_info));return 0;}\n')
    exe = tmp_path / "sizes"
    subprocess.run(["gcc", "-I", os.path.dirname(HEADER), str(src), "-o", str(exe)], check=True)
    got = [int(v) for v in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()]
    assert got == [ctypes.sizeof(SampleDesc), ctypes.sizeof(TokParams), ctypes.sizeof(Dropout), ctypes.sizeof(GemmDesc),
                   GemmDesc.drop.offset, GemmDesc.aux.offset, GemmDesc.workspace.offset, ctypes.sizeof(GemmPlanInfo)]


def test_dropout_descriptor_keeps_its_seed_alive():
    """The kernels read the seed through the descriptor's pointer: a temporary seed tensor must outlive the call that
    made the descriptor (else its memory is reused before the kernel reads it)."""
    import gc
    import weakref
    from neko_b200._lib import Dropout
    dr = Dropout.make(torch.tensor([9, 10], dtype=torch.int32), 6, 0.25)
    gc.collect()
    seed = weakref.ref(dr._seed_tensor)
    assert seed() is not None and dr.seed == seed().data_ptr()
    assert Dropout.make(None, 6, 0.25).seed is None and Dropout.make(torch.tensor([1, 2]), 6, 0.0).seed is None


def test_no_cpu_fallback():
    """The product path must fail loudly without a CUDA device (no oracle / CPU route)."""
    from neko_b200.policy import GatoPolicy
    with pytest.raises(Exception):
        GatoPolicy(device="cpu", embed_dim=64, layers=1, heads=2, dropout=0.0, resid_mid_channels=128)
    import neko_b200.policy.gato_policy as gp
    import neko_b200.ops as ops_mod
    for mod in (gp, ops_mod):
        src = open(mod.__file__).read()
        assert "import oracle" not in src and "from oracle" not in src, "product code must not import the oracle"
    if not torch.cuda.is_available():
        from neko_b200 import ops
        with pytest.raises(Exception):
            ops.cast_bf16(torch.zeros(8))


@pytest.mark.parametrize("name", ["cfg1", "cfg2", "cfg3", "cfg4", "cfg5"])
def test_plan_matches_oracle_masks(name):
    from neko_b200.policy.packing import build_plan
    cfg = O.GatoConfig(context_len=O.CONFIGS[name]["context_len"])
    batch = O.synth_batch(name)
    tb = O.tokenize(batch, cfg)
    plan = build_plan(batch, patch_size=16, context_len=cfg.context_len, pad_seq=False)
    B, S = tb.tokens.shape
    assert (plan.B, plan.seq_len, plan.width) == (B, S, S)
    rows = (np.arange(B)[:, None] * S + np.arange(S - 1)[None, :])[tb.loss_mask > 0]
    assert np.array_equal(np.sort(plan.loss_rows), rows)
    assert np.array_equal(plan.first_valid, (S - tb.token_masks.sum(1)).astype(np.int32))
    assert plan.n_valid_tokens == int(tb.token_masks.sum())


def test_plan_pad_seq_and_errors():
    from neko_b200.policy.packing import build_plan
    batch = [{"text": [1, 2, 3]}, {"continuous_obs": torch.zeros(2, 3), "continuous_actions": torch.zeros(2, 1)}]
    plan = build_plan(batch, patch_size=16, context_len=32, pad_seq=True)
    assert plan.width == 32 and plan.seq_len == 10
    cfg = O.GatoConfig(context_len=32, pad_seq=True)
    tb = O.tokenize(batch, cfg)
    rows = (np.arange(2)[:, None] * 32 + np.arange(31)[None, :])[tb.loss_mask > 0]
    assert np.array_equal(np.sort(plan.loss_rows), rows)
    with pytest.raises(AssertionError):
        build_plan([{"continuous_obs": torch.zeros(3, 2), "continuous_actions": torch.zeros(4, 1)}], patch_size=16, context_len=32, pad_seq=False)
    with pytest.raises(AssertionError):
        build_plan([{"images": torch.zeros(1, 3, 20, 32)}], patch_size=16, context_len=32, pad_seq=False)
    with pytest.raises(AssertionError):
        build_plan([{}], patch_size=16, context_len=32, pad_seq=False)


def test_patch_position_bins_match_oracle():
    from neko_b200.policy.embeddings import PatchPosEncoding
    enc = PatchPosEncoding(128, 8).eval()
    for n_h, n_w in [(6, 6), (14, 14), (2, 3), (5, 1)]:
        hp, wp = enc.positions(n_h, n_w)
        assert np.array_equal(hp.numpy(), O.patch_position_indices(n_h))
        assert np.array_equal(wp.numpy(), O.patch_position_indices(n_w))
    enc.train()
    torch.manual_seed(3)
    hp, wp = enc.positions(4, 3)
    torch.manual_seed(3)
    ref_h = O.patch_position_indices(4, 128, True)
    ref_w = O.patch_position_indices(3, 128, True)
    assert np.array_equal(hp.numpy(), ref_h) and np.array_equal(wp.numpy(), ref_w)


_GLOO_WORKER = r"""
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, os.environ["NEKO_ROOT"])
from neko_b200.dp import GradSynchronizer
dist.init_process_group("gloo", rank=int(os.environ["RANK"]), world_size=2)
rank = dist.get_rank()
n = 10_000
arena = torch.arange(n, dtype=torch.float32) * (rank + 1)
sync = GradSynchronizer(arena, bucket_bytes=4 * 1500)
# ranges become final back to front of the execution = front to back of the arena
sync.begin_step()
for lo, hi in [(0, 4000), (4000, 4064), (4064, 4128), (4128, 9000), (9000, n)]:
    sync.on_range_ready(lo, hi)
sync.finish()
ref = torch.arange(n, dtype=torch.float32) * 1.5
assert torch.allclose(arena, ref), (arena[:5], ref[:5])
covered = sorted(sync.launched)
assert covered[0][0] == 0 and covered[-1][1] == n and all(a[1] == b[0] for a, b in zip(covered, covered[1:]))
assert max(hi - lo for lo, hi in covered) <= 1500
# gradient accumulation: no_sync leaves the arena untouched
arena2 = torch.ones(100) * (rank + 1)
s2 = GradSynchronizer(arena2, bucket_bytes=1 << 20)
with s2.no_sync():
    s2.on_range_ready(0, 100); s2.finish()
assert torch.equal(arena2, torch.ones(100) * (rank + 1))
s2.on_range_ready(0, 100); s2.finish()
assert torch.allclose(arena2, torch.ones(100) * 1.5)
# skip ranges: parts of the arena that are zero on every rank by construction are left out of the collectives
arena3 = torch.arange(1000, dtype=torch.float32) * (rank + 1)
arena3[200:700] = 0.0
s3 = GradSynchronizer(arena3, bucket_bytes=4 * 128)
s3.skip_ranges += [(200, 700), (990, 1000)]
s3.begin_step()
s3.on_range_ready(0, 500); s3.on_range_ready(500, 1000); s3.finish()
ref3 = torch.arange(1000, dtype=torch.float32) * 1.5
ref3[200:700] = 0.0
ref3[990:] = torch.arange(990, 1000, dtype=torch.float32) * (rank + 1)      # skipped: stays local
assert torch.allclose(arena3, ref3)
assert all(hi <= 200 or lo >= 700 for lo, hi in s3.launched) and all(hi <= 990 for lo, hi in s3.launched)
assert sum(hi - lo for lo, hi in s3.launched) == 1000 - 500 - 10
dist.destroy_process_group()
print("ok", rank)
"""


def test_grad_synchronizer_gloo_world2(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(_GLOO_WORKER)
    port = 29500 + (os.getpid() % 2000)
    procs = []
    for r in range(2):
        env = dict(os.environ, RANK=str(r), WORLD_SIZE="2", MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), NEKO_ROOT=ROOT)
        procs.append(subprocess.Popen([sys.executable, str(script)], env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT))
    for p in procs:
        out, _ = p.communicate(timeout=120)
        assert p.returncode == 0, out.decode()


def test_bench_batches_have_the_oracle_configs_shapes():
    """bench.py's GPU arm draws inputs from the package; they must have the shapes / dtypes of the oracle's generator
    (the one the golden fixtures and the CPU baseline use) for every BASELINE configuration."""
    from neko_b200.tasks.synthetic import BENCH_CONFIGS, bench_batch
    for n in BENCH_CONFIGS:
        a, b = O.synth_batch(n, seed=1), bench_batch(n, seed=1)
        assert len(a) == len(b) == BENCH_CONFIGS[n]["batch"], n
        for x, y in zip(a, b):
            assert set(x) == set(y), (n, set(x), set(y))
            for k in x:
                sx = tuple(x[k].shape) if hasattr(x[k], "shape") else (len(x[k]),)
                sy = tuple(y[k].shape) if hasattr(y[k], "shape") else (len(y[k]),)
                assert sx == sy, (n, k, sx, sy)
                if hasattr(x[k], "dtype"):
                    assert x[k].dtype == y[k].dtype, (n, k)
        assert {k: v for k, v in BENCH_CONFIGS[n].items() if k != "batch"} == O.CONFIGS[n]


def test_product_code_never_imports_the_oracle():
    """oracle/ is test infrastructure: neither the package nor the GPU arm of bench.py may import it."""
    import re
    for dirpath, _dirs, files in os.walk(os.path.join(ROOT, "neko_b200")):
        for f in files:
            if f.endswith(".py"):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, flags=re.M), os.path.join(dirpath, f)
    src = open(os.path.join(ROOT, "train.py")).read()
    assert not re.search(r"^\s*(from|import)\s+oracle\b", src, flags=re.M)
    bench = open(os.path.join(ROOT, "bench.py")).read()
    gpu_arm = bench[bench.index("def run_ours("):bench.index("def main(")]
    assert not re.search(r"^\s*(from|import)\s+oracle\b", gpu_arm, flags=re.M)   # (its cpu_baseline leg calls cpu_tokens_per_s)


def test_bench_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` (the CPU arm the driver times next to the GPU arm): one JSON line with the contract keys."""
    import json
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--config", "cfg1", "--steps", "1",
                          "--warmup", "1"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = [ln for ln in out.stdout.splitlines() if ln.startswith("{")][-1]
    d = json.loads(line)
    assert d["impl"] == "reference" and d["metric"] == "train tokens/sec (fwd+bwd)" and d["unit"] == "tokens/s"
    assert d["value"] > 0 and d["higher_is_better"] is True and d["n_gpus"] == 1
    from oracle import ref_shim
    # the reference itself whenever a tree is present (/root/reference here, oracle/_ref on the GPU box), else the port
    assert d["cpu_baseline"]["kind"] == ("reference" if ref_shim.reference_available() else "port")
    assert d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["config"]["same_config"] is True and d["config"]["tokens_per_step_per_gpu"] == 960   # the FULL cfg1 batch
    assert d["e2e"] == {"value": d["value"], "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["config"]["name"] == "cfg1" and "workload" in d["config"]
    # rank != 0 of a multi-process launch exits silently
    out2 = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--config", "cfg1", "--steps", "1"],
                          capture_output=True, text=True, timeout=600, cwd=ROOT, env=dict(os.environ, RANK="1", WORLD_SIZE="2"))
    assert out2.returncode == 0 and "{" not in out2.stdout


def test_bench_rejects_arguments_it_cannot_honour():
    """--steps below 1 would time nothing; --dump-outputs writes what the GPU arm's step returned, so the CPU arm refuses it."""
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "unused"]):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + extra, capture_output=True, text=True, timeout=300, cwd=ROOT)
        assert out.returncode == 2 and extra[-2] in out.stderr, (extra, out.stderr[-500:])


@pytest.mark.parametrize("seed", range(12))
def test_plan_matches_oracle_on_random_mixed_batches(seed):
    """Random mixtures of every modality (text lists / tensors, uint8 / float frames of several sizes, precomputed image
    embeddings, continuous / discrete observations and actions, ragged lengths, with and without pad_seq): the host planner's
    loss rows, left-padding offsets, token counts and per-sample descriptor table against the oracle's tokenisation."""
    from neko_b200.policy.packing import build_plan
    from _random_batches import random_mixed_batch
    batch, ctx, pad_seq = random_mixed_batch(seed)
    cfg = O.GatoConfig(embed_dim=32, layers=1, heads=1, context_len=ctx, text_tokens=300, pad_seq=pad_seq)
    tb = O.tokenize(batch, cfg)
    plan = build_plan(batch, patch_size=16, context_len=ctx, pad_seq=pad_seq)
    B, W = tb.tokens.shape
    assert plan.B == B and plan.width == W
    rows = (np.arange(B)[:, None] * W + np.arange(W - 1)[None, :])[tb.loss_mask > 0]
    assert np.array_equal(np.sort(plan.loss_rows), rows)
    n_valid = tb.token_masks.sum(1).astype(np.int64)
    assert plan.n_valid_tokens == int(n_valid.sum())
    assert np.array_equal(plan.first_valid, (plan.seq_len - n_valid).astype(np.int32))
    desc = plan.descs.view(np.int32).reshape(B, 16)
    for b, st in enumerate(tb.samples):
        assert desc[b, 0] == st.n_timesteps and desc[b, 1] == st.n_patches
        assert desc[b, 0] * (desc[b, 1:7].sum() + 1) == st.ids.shape[0]


def test_vendored_reference_recipe(tmp_path):
    """oracle/build_ref.py: the archive holds the reference's path files byte for byte (an empty entry for a package without an
    __init__.py), leaves no loose reference source beside it and lists every file in its manifest.  Packed from a reference
    checkout when one is present -- and then imported through the shims (what bench.py --impl reference uses) -- else from a
    stand-in tree of the same layout."""
    import hashlib
    import zipfile
    from oracle import build_ref, ref_shim
    if ref_shim.reference_kind() == "mounted":
        src = ref_shim.REFERENCE_ROOT
    else:
        src = str(tmp_path / "src")
        for k, rel in enumerate(build_ref.FILES):
            if rel != "gato/transformers/__init__.py":
                os.makedirs(os.path.dirname(os.path.join(src, rel)), exist_ok=True)
                open(os.path.join(src, rel), "wb").write(f"# {rel}\n".encode() * (k + 1))
    dst = str(tmp_path / "_ref")
    assert build_ref.build(src, dst)
    archive = os.path.join(dst, "gato_ref.zip")
    manifest = open(os.path.join(dst, "MANIFEST.sha256")).read().split("\n")
    with zipfile.ZipFile(archive) as z:
        assert sorted(z.namelist()) == sorted(build_ref.FILES)
        for rel in build_ref.FILES:
            p = os.path.join(src, rel)
            data = open(p, "rb").read() if os.path.exists(p) else b""
            assert z.read(rel) == data, rel
            assert f"{hashlib.sha256(data).hexdigest()}  {rel}" in manifest, rel
    assert not os.path.isdir(os.path.join(dst, "gato")), "loose reference sources beside the archive"
    # oracle/_ref must stay out of the history
    assert "oracle/_ref/" in open(os.path.join(ROOT, ".gitignore")).read()
    if ref_shim.reference_kind() != "mounted":
        return
    code = ("from oracle import ref_shim; import os; assert ref_shim.REFERENCE_ROOT == os.environ['NEKO_REFERENCE_ROOT'], ref_shim.REFERENCE_ROOT; "
            "G = ref_shim.load_reference_policy_class(); "
            "m = G(device='cpu', embed_dim=32, layers=1, heads=1, dropout=0.0, resid_mid_channels=128, context_len=32); "
            "l, loss = m([{'text': [1, 2, 3]}], compute_loss=True); loss.backward(); print('ok')")
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300, cwd=ROOT,
                         env=dict(os.environ, NEKO_REFERENCE_ROOT=archive))
    assert out.returncode == 0 and "ok" in out.stdout, out.stderr[-1500:]


def test_copy_engine_bucket_schedule_covers_the_arena_once():
    """Host logic of the copy-engine data-parallel exchange (neko_b200/dp.py) with the device side mocked out: the groups handed to
    ce_submit cover every live arena element exactly once, leave the skip ranges out, respect the bucket size, are drained in
    submission order with non-decreasing ticks, and ranges that complete near the end of backward are not held back."""
    import torch
    from neko_b200.dp import GradSynchronizer

    class FakeP2P:
        proto = "ce"

        def __init__(self):
            self.submitted, self.drains, self.flushed = [], [], 0

        def begin_step(self):
            pass

        def ce_submit(self, ranges, scale, comm, tick=0):
            self.submitted.append((list(ranges), scale, tick))

        def ce_drain(self, comm, tick=None, min_age=2):
            self.drains.append(tick)

        def ce_flush(self, comm):
            self.flushed += 1

    total = 10_000_000
    arena = torch.zeros(total)
    s = GradSynchronizer(arena, bucket_bytes=4 * 1_000_000)          # world size 1 without a process group ...
    s.world, s._cuda, s.backend, s._p2p = 4, True, "p2p", FakeP2P()   # ... pretend: 4 ranks, CUDA, own exchange
    s._join_streams = lambda: None
    s.tail_elems = 600_000
    s.skip_ranges = [(7_000_000, 9_700_000), (9_999_000, total)]
    # completion order of a backward: one big head, six "layers" of uneven size, then the tail that contains the skipped rows
    notes = [(0, 3_500_000)] + [(3_500_000 + 500_000 * k, 4_000_000 + 500_000 * k) for k in range(6)] + [(6_500_000, total)]
    s.begin_step()
    for lo, hi in notes:
        s.on_range_ready(lo, hi)
    s.finish()
    p2p = s._p2p
    flat = [r for grp, _sc, _t in p2p.submitted for r in grp]
    covered = torch.zeros(total, dtype=torch.int32)
    for lo, hi in flat:
        assert lo % 4 == 0 and hi % 4 == 0 and hi > lo
        covered[lo:hi] += 1
    live = torch.ones(total, dtype=torch.int32)
    for lo, hi in s.skip_ranges:
        live[lo:hi] = 0
    assert torch.equal(covered, live)
    assert all(sum(b - a for a, b in grp) <= s.bucket_elems for grp, _sc, _t in p2p.submitted)
    assert all(abs(sc - 0.25) < 1e-12 for _g, sc, _t in p2p.submitted)
    ticks = [t for _g, _sc, t in p2p.submitted]
    assert ticks == sorted(ticks) and p2p.drains == sorted(p2p.drains) and p2p.flushed == 1
    # the head is cut into bucket-sized exchanges at once; the last layer is submitted at its own notification, not at finish()
    assert p2p.submitted[0][0] == [(0, 1_000_000)] and ticks[0] == 1
    last_layer = next(t for g, _sc, t in p2p.submitted if (6_000_000, 6_500_000) in g or any(a <= 6_000_000 < b for a, b in g))
    assert last_layer == 7 and len(notes) == 8
    # the small live ranges of the tail share one exchange
    assert any(len(g) > 1 for g, _sc, _t in p2p.submitted)
    # no_sync: nothing is submitted
    n = len(p2p.submitted)
    with s.no_sync():
        s.begin_step()
        for lo, hi in notes:
            s.on_range_ready(lo, hi)
        s.finish()
    assert len(p2p.submitted) == n

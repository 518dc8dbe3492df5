"""neko_gemm across its schedule and epilogue matrix against the fp64 reference of tests/_gemm_ref.py.

Every cell forces one schedule (NEKO_GEMM_* knobs, or operand geometry for the choices that have no per-call knob), asks
neko_gemm_plan which schedule that is and asserts it is the one the cell asked for, then checks per launch:
  - every output within the reference bound (tests/test_gemm_check_cpu.py shows the bound is strict);
  - not one byte written outside [M, N] of C / C2 / C3 (they sit in larger buffers filled with a NaN pattern, and their own
    [M, N] is NaN-filled too, so an element the kernel skips fails the reference check); A, B, bias and aux unchanged;
  - a second launch bit-identical to the first (stream-K: three launches, so its counters are re-armed twice);
  - every schedule of one problem without split-K / stream-K bit-identical to every other: TMA vs direct stores, vector vs
    per-element paths, TMA vs per-thread aux, 8 vs 16 epilogue warps, BN 128 / 192 / 256, single CTA vs CTA pair and either
    rasterisation all evaluate the same fp32 expression on the same k-ordered accumulator.
GPU only (-m gpu)."""
import ctypes as C
import math

import pytest
import torch

import _gemm_ref as R

pytestmark = pytest.mark.gpu

NAN16 = 0x7FC1           # a NaN in both bf16 and fp16
NAN32 = 0x7FC00011
DT = {"bf16": torch.bfloat16, "f16": torch.float16, "f32": torch.float32}
EPI_NAMES = {R.EPI_BF16: "bf16", R.EPI_F32: "f32", R.EPI_GELU_BF16: "gelu", R.EPI_RESID_F32: "resid", R.EPI_DGELU_BF16: "dgelu",
             R.EPI_RESID_F32_BF16: "resid_bf16"}
AUX_EPIS = (R.EPI_RESID_F32, R.EPI_DGELU_BF16)          # the epilogues with a TMA-aux path


@pytest.fixture(scope="module")
def ops():
    from neko_b200 import _lib, ops as _ops
    _lib.require_device()
    return _ops


def _pad8(n):
    return (n + 7) // 8 * 8


def _nan_fill(shape, dtype):
    if dtype == torch.float32:
        return torch.full(shape, NAN32, dtype=torch.int32, device="cuda").view(torch.float32)
    return torch.full(shape, NAN16, dtype=torch.int16, device="cuda").view(dtype)


def _bits(t):
    return t.contiguous().view(torch.int32 if t.dtype == torch.float32 else torch.int16).clone()


class Buf:
    """A [M, N] view inside a NaN-filled buffer: one spare row above, two below, ld >= N + 8.
    geometry 'vec': 16-byte aligned base and pitch; 'odd_ld': odd leading dimension; 'offset': base one element off."""

    def __init__(self, M, N, dtype, geometry="vec"):
        self.ld = _pad8(N + 8) + (1 if geometry == "odd_ld" else 0)
        self.off = self.ld + (1 if geometry == "offset" else 0)
        self.shape = (M, N)
        self.storage = _nan_fill(((M + 3) * self.ld + 8,), dtype)
        self.view = self.storage.as_strided(self.shape, (self.ld, 1), self.off)
        inside = torch.arange(self.storage.numel(), device="cuda").as_strided(self.shape, (self.ld, 1), self.off)
        self.outside = torch.ones(self.storage.numel(), dtype=torch.bool, device="cuda")
        self.outside[inside.reshape(-1)] = False

    def reset(self, values=None):
        self.view.copy_(_nan_fill(self.shape, self.view.dtype) if values is None else values)

    def canaries_intact(self):
        return bool((_bits(self.storage)[self.outside] == (NAN32 if self.storage.dtype == torch.float32 else NAN16)).all())


# ---------------------------------------------------------------------------------------------------
# problems: operands in padded, NaN-framed storage, fp64 accumulator computed once per problem
# ---------------------------------------------------------------------------------------------------
_PROBLEMS = {}


def _operand(x, mn, pad):
    """x: logical [rows, K]. Returns (storage, view passed to the GEMM): [rows, K] or [K, rows] (mn) rows of a wider,
    taller NaN-filled buffer, leading dimension padded by `pad` extra elements."""
    stored = x.t() if mn else x
    r, c = stored.shape
    storage = _nan_fill((r + 1, _pad8(c) + pad), x.dtype)
    storage[:r, :c] = stored
    return storage, storage[:r, :c]


def problem(M, N, K, a_mn=False, b_mn=False, f16=False, pad=0):
    key = (M, N, K, a_mn, b_mn, f16, pad)
    if key not in _PROBLEMS:
        g = torch.Generator().manual_seed(M * 1000003 + N * 1009 + K * 7 + 2 * a_mn + b_mn + 5 * f16)
        dt = torch.float16 if f16 else torch.bfloat16
        a = (torch.randn(M, K, generator=g) * 0.5).to(dt).cuda()
        b = (torch.randn(N, K, generator=g) * (3.0 / math.sqrt(K))).to(dt).cuda()   # |acc| ~ 1.5: GELU's curved part
        a_store, a_view = _operand(a, a_mn, pad)
        b_store, b_view = _operand(b, b_mn, pad)
        acc, absacc = R.accumulator(a, b)
        side = dict(bias=(torch.randn(N, generator=g) * 0.5).cuda(), resid=torch.randn(M, N, generator=g).cuda(),
                    pre=(torch.randn(M, N, generator=g) * 2.0).to(torch.bfloat16).cuda(),
                    c_init=torch.randn(M, N, generator=g).cuda())
        _PROBLEMS[key] = dict(M=M, N=N, K=K, a_mn=a_mn, b_mn=b_mn, f16=f16, a_store=a_store, a=a_view, b_store=b_store,
                              b=b_view, acc=acc, absacc=absacc, **side)
    return _PROBLEMS[key]


# ---------------------------------------------------------------------------------------------------
# one launch configuration
# ---------------------------------------------------------------------------------------------------
def set_knobs(mp, pair=None, bn=None, ew=None, nfast=None, splits=1, streamk=0, direct=False):
    for name, v in (("PAIR", pair), ("BN", bn), ("EPI16", None if ew is None else int(ew == 16)), ("NFAST", nfast),
                    ("SPLITS", splits), ("STREAMK", streamk)):
        if v is None:
            mp.delenv("NEKO_GEMM_" + name, raising=False)
        else:
            mp.setenv("NEKO_GEMM_" + name, str(v))
    if direct:
        mp.setenv("NEKO_GEMM_DIRECT_STORE", "1")
    else:
        mp.delenv("NEKO_GEMM_DIRECT_STORE", raising=False)


_SEEDS = {}


def _dropout(ops, case):
    from neko_b200._lib import Dropout
    if "seed" not in _SEEDS:
        _SEEDS["seed"] = torch.tensor([0x1234567, 0x7654321], dtype=torch.int32, device="cuda")
    return Dropout.make(_SEEDS["seed"], 5, 0.25)


class Launch:
    """Buffers and arguments of one neko_gemm call of `case` under output geometry `geometry`
    ('vec', 'odd_ld', 'offset', 'bias_off': bias one float off, 'aux_ld': aux with an odd leading dimension)."""

    def __init__(self, ops, case, geometry="vec"):
        pb = case["pb"]
        M, N = pb["M"], pb["N"]
        epi = case["epi"]
        out_geo = geometry if geometry in ("odd_ld", "offset") else "vec"
        self.case, self.geometry = case, geometry
        c_dt = DT["f32"] if epi in (R.EPI_F32, R.EPI_RESID_F32, R.EPI_RESID_F32_BF16) else DT[case["c_fmt"]]
        self.outs = {"C": Buf(M, N, c_dt, out_geo)}
        if epi in (R.EPI_GELU_BF16, R.EPI_RESID_F32_BF16):
            self.outs["C2"] = Buf(M, N, DT[case["c2_fmt"]], out_geo)
        if case.get("c3"):
            self.outs["C3"] = Buf(M, N, torch.bfloat16, out_geo)
        self.inputs = [pb["a_store"], pb["b_store"]]
        self.bias = None
        if case.get("bias"):
            bst = _nan_fill((N + 8,), torch.float32)
            o = 1 if geometry == "bias_off" else 0
            bst[o:o + N] = pb["bias"]
            self.bias = bst[o:o + N]
            self.inputs.append(bst)
        self.aux = None
        self.aux_init = None
        if epi in (R.EPI_RESID_F32, R.EPI_RESID_F32_BF16):
            self.aux_init = pb["resid"]
        elif epi == R.EPI_DGELU_BF16:
            self.aux_init = pb["pre"]
        if self.aux_init is not None:
            if case.get("inplace"):
                self.aux = self.outs["C"].view
            else:
                ab = Buf(M, N, self.aux_init.dtype, "odd_ld" if geometry == "aux_ld" else "vec")
                ab.reset(self.aux_init)
                self.aux = ab.view
                self.inputs.append(ab.storage)
        self.drop = _dropout(ops, case) if case.get("drop") else None
        self.kwargs = dict(a_mn=pb["a_mn"], b_mn=pb["b_mn"], epilogue=epi, out=self.outs["C"].view,
                           out2=self.outs["C2"].view if "C2" in self.outs else None,
                           out3=self.outs["C3"].view if "C3" in self.outs else None, bias=self.bias, aux=self.aux,
                           accumulate=bool(case.get("accumulate")), M=M, N=N, K=pb["K"], drop=self.drop,
                           gelu_tanh=bool(case.get("tanh")))

    def plan(self, ops):
        return ops.gemm_plan(self.case["pb"]["a"], self.case["pb"]["b"], **self.kwargs)

    def reset(self):
        for name, buf in self.outs.items():
            init = None
            if name == "C" and self.case.get("accumulate"):
                init = self.case["pb"]["c_init"]
            elif name == "C" and self.case.get("inplace"):
                init = self.aux_init
            buf.reset(init)

    def run(self, ops):
        self.reset()
        ops.gemm(self.case["pb"]["a"], self.case["pb"]["b"], **self.kwargs)
        torch.cuda.synchronize()
        return {name: _bits(buf.view) for name, buf in self.outs.items()}


def expected_outputs(ops, case):
    """fp64 reference of `case` (cached on the case)."""
    if "expected" not in case:
        pb = case["pb"]
        epi = case["epi"]
        mult = None
        if case.get("drop"):
            dr = _dropout(ops, case)
            mult = ops.dropout_mask(pb["M"], pb["N"], dr, "cuda").double() * dr.scale
        aux = pb["resid"] if epi in (R.EPI_RESID_F32, R.EPI_RESID_F32_BF16) else (pb["pre"] if epi == R.EPI_DGELU_BF16 else None)
        case["expected"] = R.epilogue_reference(
            pb["acc"], pb["absacc"], epi, bias=pb["bias"] if case.get("bias") else None, aux=aux, mult=mult,
            c_init=pb["c_init"] if case.get("accumulate") else None, gelu_tanh=bool(case.get("tanh")),
            c_fmt=case.get("c_fmt", "bf16"), c2_fmt=case.get("c2_fmt", "bf16"), c3=bool(case.get("c3")))
    return case["expected"]


def check_launches(ops, launch, n_launches=2, bitwise_repeat=True, label=""):
    """Runs the launch n times; reference, canaries and input checks on each; returns the first launch's output bits."""
    exp = expected_outputs(ops, launch.case)
    K = launch.case["pb"]["K"]
    before = [_bits(t) for t in launch.inputs]
    first = None
    for i in range(n_launches):
        bits = launch.run(ops)
        for name, buf in launch.outs.items():
            R.assert_within(buf.view, exp[name], K, f"{label} {name} launch {i}")
            assert buf.canaries_intact(), f"{label} {name}: bytes outside [M, N] were written (launch {i})"
        for j, (t, b) in enumerate(zip(launch.inputs, before)):
            assert torch.equal(_bits(t), b), f"{label}: input {j} was modified (launch {i})"
        if first is None:
            first = bits
        elif bitwise_repeat:
            for name in bits:
                assert torch.equal(bits[name], first[name]), f"{label} {name}: launch {i} differs from launch 0"
    return first


# ---------------------------------------------------------------------------------------------------
# the covering design
# ---------------------------------------------------------------------------------------------------
SHAPES = [(1, 40, 72), (127, 136, 1000), (129, 8, 16), (255, 264, 72), (257, 200, 1000), (1000, 776, 72), (256, 256, 128),
          (129, 72, 4000)]                 # (256, 256, 128): tile-exact control
LAYOUTS = [(False, False), (False, True), (True, False), (True, True)]
FLAG_SETS = {
    R.EPI_BF16: [dict(bias=1), dict(c_fmt="f16"), dict(bias=1, f16=1, c_fmt="f16"), dict(f16=1)],
    R.EPI_F32: [dict(bias=1), dict(), dict(accumulate=1, bias=1), dict(accumulate=1, f16=1)],
    R.EPI_GELU_BF16: [dict(bias=1, c3=1), dict(tanh=1, c_fmt="f16"), dict(c2_fmt="f16", c3=1, f16=1, bias=1),
                      dict(tanh=1, bias=1, c_fmt="f16", c2_fmt="f16", c3=1), dict()],
    R.EPI_RESID_F32: [dict(bias=1, drop=1), dict(inplace=1), dict(bias=1, f16=1), dict(drop=1, inplace=1, bias=1)],
    R.EPI_DGELU_BF16: [dict(), dict(tanh=1, c_fmt="f16"), dict(f16=1), dict(tanh=1, f16=1, c_fmt="f16")],
    R.EPI_RESID_F32_BF16: [dict(bias=1, drop=1), dict(c2_fmt="f16", inplace=1), dict(bias=1, c2_fmt="f16", f16=1, drop=1),
                           dict(inplace=1, bias=1)],
}


def _case_specs():
    specs, i = [], 0
    for epi, sets in FLAG_SETS.items():
        for flags in sets:
            M, N, K = SHAPES[i % len(SHAPES)]
            a_mn, b_mn = LAYOUTS[(i + i // len(SHAPES)) % 4]
            spec = dict(epi=epi, shape=(M, N, K), a_mn=a_mn, b_mn=b_mn, pad=16 if i % 3 == 0 else 0, **flags)
            spec["id"] = (f"{EPI_NAMES[epi]}-" + "-".join(k if v == 1 else f"{k}{v}" for k, v in flags.items()) +
                          f"-{M}x{N}x{K}-{'tn'[a_mn]}{'tn'[b_mn]}" + ("-pad" if spec["pad"] else ""))
            specs.append(spec)
            i += 1
    return specs


CASE_SPECS = _case_specs()
TILES = [(0, 128, 8, 0), (0, 192, 8, 1), (0, 256, 16, 0), (1, 128, 16, 1), (1, 192, 8, 0), (1, 256, 8, 1)]  # pair, BN, EW, n_fast


def schedules(spec):
    """(tile, direct-store knob, geometry) of every cell of one case."""
    out = [(t, False, "vec") for t in TILES if not (t[0] == 1 and t[1] == 192 and spec["b_mn"])]   # no 96-row MN-major B box
    scalar_tma = "bias_off" if spec.get("bias") else ("aux_ld" if spec["epi"] in AUX_EPIS and not spec.get("inplace") else None)
    for base, flip in (((0, 128, 8, 0), (0, 128, 16, 0)), ((1, 128, 16, 1), (1, 128, 8, 0))):
        out += [(base, True, "vec"), (base, False, "odd_ld"), (flip, False, "vec")]
        out.append((base, False, "offset") if base[0] == 0 else (base, True, "odd_ld"))
        if scalar_tma:
            out.append((base, False, scalar_tma))
    return out


def expected_plan(spec, tile, direct, geometry):
    pair, bn, ew, nfast = tile
    tma_store = int(not direct and geometry not in ("odd_ld", "offset"))
    tma_aux = int(tma_store and spec["epi"] in AUX_EPIS and geometry == "vec")
    return dict(BN=bn, pair=pair, splits=1, epi_warps=ew, streamk=0, tma_store=tma_store, tma_aux=tma_aux,
                vec_ok=int(geometry == "vec"), n_fast=nfast)


def make_case(spec):
    M, N, K = spec["shape"]
    case = dict(spec)
    case.setdefault("c_fmt", "bf16")
    case.setdefault("c2_fmt", "bf16")
    case["pb"] = problem(M, N, K, spec["a_mn"], spec["b_mn"], bool(spec.get("f16")), spec["pad"])
    return case


def _plan_tuple(epi, plan):
    return (EPI_NAMES[epi],) + tuple(plan[k] for k in ("BN", "pair", "splits", "epi_warps", "streamk", "tma_store", "tma_aux",
                                                       "vec_ok", "n_fast"))


def _assert_plan(plan, want, label):
    got = {k: plan[k] for k in want}
    assert got == want, f"{label}: asked for {want}, the library plans {got}"


@pytest.mark.parametrize("spec", CASE_SPECS, ids=[s["id"] for s in CASE_SPECS])
def test_epilogue_schedule_matrix(ops, monkeypatch, spec):
    case = make_case(spec)
    results = []
    for tile, direct, geometry in schedules(spec):
        label = f"{spec['id']} tile={tile} direct={direct} geometry={geometry}"
        set_knobs(monkeypatch, pair=tile[0], bn=tile[1], ew=tile[2], nfast=tile[3], direct=direct)
        launch = Launch(ops, case, geometry)
        _assert_plan(launch.plan(ops), expected_plan(spec, tile, direct, geometry), label)
        results.append((label, check_launches(ops, launch, label=label)))
    label0, first = results[0]
    for label, bits in results[1:]:
        for name in first:
            diff = int((bits[name] != first[name]).sum())
            assert diff == 0, f"{name}: {diff} elements of [{label}] differ bitwise from [{label0}]"


# ---------------------------------------------------------------------------------------------------
# split-K and stream-K
# ---------------------------------------------------------------------------------------------------
def _split_k_spec(accumulate):
    return dict(epi=R.EPI_F32, shape=(257, 200, 4000), a_mn=True, b_mn=True, pad=8, accumulate=int(accumulate))


@pytest.mark.parametrize("splits", [2, 3, None])
@pytest.mark.parametrize("accumulate", [False, True])
@pytest.mark.parametrize("geometry,direct", [("vec", False), ("vec", True), ("odd_ld", False)])
def test_split_k(ops, monkeypatch, splits, accumulate, geometry, direct):
    """Weight-gradient shape (both operands MN-major, K = the token axis): split-K reduce-add into C, overwrite and
    accumulate, through TMA reduce-add, direct atomics and the per-element path."""
    case = make_case(_split_k_spec(accumulate))
    set_knobs(monkeypatch, splits=splits, direct=direct)
    launch = Launch(ops, case, geometry)
    plan = launch.plan(ops)
    assert plan["splits"] == splits if splits else plan["splits"] > 1, plan
    assert plan["streamk"] == 0 and plan["tma_store"] == int(geometry == "vec" and not direct), plan
    assert plan["vec_ok"] == int(geometry == "vec"), plan
    check_launches(ops, launch, bitwise_repeat=False, label=f"split-K {plan}")   # reduce-add order is not fixed


STREAMK_FLAGS = {R.EPI_BF16: dict(bias=1), R.EPI_GELU_BF16: dict(bias=1, c3=1, tanh=1), R.EPI_RESID_F32: dict(bias=1, drop=1, inplace=1),
                 R.EPI_DGELU_BF16: dict(), R.EPI_RESID_F32_BF16: dict(bias=1, c2_fmt="f16")}


def _stream_k_spec(epi):
    return dict(epi=epi, shape=(5000, 768, 1024), a_mn=False, b_mn=False, pad=0, **STREAMK_FLAGS[epi])


@pytest.mark.parametrize("pair", [0, 1])
@pytest.mark.parametrize("epi", sorted(STREAMK_FLAGS), ids=[EPI_NAMES[e] for e in sorted(STREAMK_FLAGS)])
def test_stream_k(ops, monkeypatch, epi, pair):
    """(5000, 768, 1024) at BN 128 is 1.6 rounds of tiles on single CTAs and on CTA pairs, so stream-K is eligible;
    three launches re-arm the workspace counters."""
    case = make_case(_stream_k_spec(epi))
    set_knobs(monkeypatch, pair=pair, bn=128, streamk=1)
    launch = Launch(ops, case)
    plan = launch.plan(ops)
    assert plan["streamk"] == 1 and plan["pair"] == pair and plan["BN"] == 128, plan
    assert plan["tma_aux"] == int(epi in AUX_EPIS), plan
    check_launches(ops, launch, n_launches=3, label=f"stream-K {EPI_NAMES[epi]} {plan}")


# ---------------------------------------------------------------------------------------------------
# what the plan reports, and what the API rejects
# ---------------------------------------------------------------------------------------------------
def test_plan_reports_knobs_the_library_overrides(ops, monkeypatch):
    """A forced knob the schedule cannot honour is dropped; the plan says so."""
    case = make_case(dict(epi=R.EPI_BF16, shape=(512, 768, 256), a_mn=False, b_mn=True, pad=0))
    set_knobs(monkeypatch, pair=1, bn=192)                     # a pair CTA would stage 96 MN-major rows of B
    assert Launch(ops, case).plan(ops)["BN"] != 192
    set_knobs(monkeypatch, pair=0, bn=192, ew=16)              # BN 192 has no 4-way column split
    plan = Launch(ops, case).plan(ops)
    assert plan["BN"] == 192 and plan["epi_warps"] == 8
    set_knobs(monkeypatch, pair=0, bn=128, streamk=1)          # 4 x 6 tiles: far fewer than the workers
    assert Launch(ops, case).plan(ops)["streamk"] == 0
    set_knobs(monkeypatch, pair=0, bn=128, splits=4)           # split-K is for plain fp32 outputs only
    assert Launch(ops, case).plan(ops)["splits"] == 1


def _rejected(ops, launch, mutate, what):
    from neko_b200 import _lib
    pb = launch.case["pb"]
    gd, _, _ = ops._gemm_args(pb["a"], pb["b"], launch.kwargs["a_mn"], launch.kwargs["b_mn"], launch.kwargs["epilogue"],
                              launch.kwargs["out"], launch.kwargs["out2"], launch.kwargs["out3"], launch.kwargs["bias"],
                              launch.kwargs["aux"], launch.kwargs["accumulate"], launch.kwargs["M"], launch.kwargs["N"],
                              launch.kwargs["K"], torch.bfloat16, launch.kwargs["drop"], launch.kwargs["gelu_tanh"])
    mutate(gd)
    lib = _lib.load()
    info = _lib.GemmPlanInfo()
    assert lib.neko_gemm_plan(C.byref(gd), C.byref(info)) == -1, f"neko_gemm_plan accepted {what}"
    launch.reset()
    assert lib.neko_gemm(C.byref(gd), _lib.stream_ptr()) == -1, f"neko_gemm accepted {what}"
    torch.cuda.synchronize()
    for name, buf in launch.outs.items():
        assert bool((_bits(buf.storage) == _bits(_nan_fill(buf.storage.shape, buf.storage.dtype))).all()), f"{what}: {name} written"


def test_error_contract(ops, monkeypatch):
    """Each of these returns NEKO_EINVAL from neko_gemm and neko_gemm_plan, and writes nothing."""
    set_knobs(monkeypatch)
    mk = lambda epi, **kw: Launch(ops, make_case(dict(epi=epi, shape=(128, 64, 128), a_mn=False, b_mn=False, pad=0, **kw)))

    def set_(field, value):
        return lambda gd: setattr(gd, field, value)

    bias = problem(128, 64, 128)["bias"]
    _rejected(ops, mk(R.EPI_DGELU_BF16), set_("bias", bias.data_ptr()), "DGELU with a bias")
    _rejected(ops, mk(R.EPI_BF16), set_("flags", 1), "f16 A with bf16 B")
    _rejected(ops, mk(R.EPI_BF16, f16=1), set_("flags", 2 | 4), "bf16 A with f16 B")
    _rejected(ops, mk(R.EPI_BF16), set_("accumulate", 1), "accumulate on EPI_BF16")
    _rejected(ops, mk(R.EPI_RESID_F32), set_("accumulate", 1), "accumulate on EPI_RESID_F32")
    c3 = _nan_fill((128, 64), torch.bfloat16)
    _rejected(ops, mk(R.EPI_BF16), lambda gd: (setattr(gd, "C3", c3.data_ptr()), setattr(gd, "ldc3", 64)), "C3 on EPI_BF16")
    _rejected(ops, mk(R.EPI_DGELU_BF16), lambda gd: (setattr(gd, "C3", c3.data_ptr()), setattr(gd, "ldc3", 64)), "C3 on DGELU")
    drop = _dropout(ops, None)
    _rejected(ops, mk(R.EPI_BF16), set_("drop", drop), "dropout on EPI_BF16")
    _rejected(ops, mk(R.EPI_GELU_BF16), set_("drop", drop), "dropout on EPI_GELU_BF16")
    _rejected(ops, mk(R.EPI_F32), set_("lda", 132), "lda % 8 != 0")
    _rejected(ops, mk(R.EPI_F32), set_("ldb", 124), "ldb % 8 != 0 (and < K)")


# ---------------------------------------------------------------------------------------------------
# coverage of the design above
# ---------------------------------------------------------------------------------------------------
def test_schedule_coverage(ops, monkeypatch):
    """Every plan value the matrix is meant to reach is reached (the matrix asserts each cell's plan, so these are the
    schedules that ran)."""
    reached = set()
    for spec in CASE_SPECS:
        case = make_case(spec)
        for tile, direct, geometry in schedules(spec):
            set_knobs(monkeypatch, pair=tile[0], bn=tile[1], ew=tile[2], nfast=tile[3], direct=direct)
            reached.add(_plan_tuple(spec["epi"], Launch(ops, case, geometry).plan(ops)))
    for epi, name in EPI_NAMES.items():
        mine = [t for t in reached if t[0] == name]
        tiles = {(t[2], t[1]) for t in mine}
        assert tiles >= {(p, bn) for p in (0, 1) for bn in (128, 192, 256)}, (name, tiles)
        for idx, field in ((4, "epi_warps"), (6, "tma_store"), (8, "vec_ok"), (9, "n_fast")):
            assert {t[idx] for t in mine} >= ({8, 16} if field == "epi_warps" else {0, 1}), (name, field)
        if epi in AUX_EPIS:
            assert {t[7] for t in mine} == {0, 1}, (name, "tma_aux")
        # the flag sets of this epilogue each ran under TMA stores, direct stores, vector and per-element paths
        for spec in CASE_SPECS:
            if spec["epi"] == epi:
                paths = {(g, d) for _, d, g in schedules(spec)}
                assert {("vec", False), ("vec", True), ("odd_ld", False)} <= paths, spec["id"]
    # split-K at 2, 3 and the automatic factor (with and without accumulate), stream-K for every 16-bit / residual epilogue
    for accumulate in (False, True):
        case = make_case(_split_k_spec(accumulate))
        for splits in (2, 3, None):
            set_knobs(monkeypatch, splits=splits)
            plan = Launch(ops, case).plan(ops)
            assert plan["splits"] == splits if splits else plan["splits"] > 1, plan
            reached.add(_plan_tuple(R.EPI_F32, plan))
    assert {t[3] for t in reached if t[0] == "f32"} >= {1, 2, 3}, "split-K factors"
    for epi in STREAMK_FLAGS:
        case = make_case(_stream_k_spec(epi))
        for pair in (0, 1):
            set_knobs(monkeypatch, pair=pair, bn=128, streamk=1)
            reached.add(_plan_tuple(epi, Launch(ops, case).plan(ops)))
    assert {t[0] for t in reached if t[5] == 1} == {EPI_NAMES[e] for e in EPI_NAMES if e != R.EPI_F32}, "stream-K"
    print("\nplan tuples reached (epilogue, BN, pair, splits, epi_warps, streamk, tma_store, tma_aux, vec_ok, n_fast):")
    for t in sorted(reached):
        print("  ", t)

"""Host-side batch plan for the fused tokenise/embed kernel.

Turns the reference's list-of-dicts input (docstring of tokenize_input_dicts, gato_policy.py:196-244)
into: one descriptor per sample (neko_sample_desc), one packed fp32 buffer (continuous obs/actions),
one packed int32 buffer (text ids, discrete obs/actions), image groups, and -- because every mask is a
function of the SHAPES only -- the loss-row list of gato_policy.py:177-185 without touching the device.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field
from typing import List, Optional, Sequence, Tuple

import numpy as np
import torch

from .._lib import SampleDesc


@dataclass
class ImageGroup:
    """Samples whose frames share (H, W, dtype): one patch-embed launch."""
    height: int
    width: int
    is_u8: bool
    tensors: List[torch.Tensor] = field(default_factory=list)   # [T,3,H,W] each
    sample_idx: List[int] = field(default_factory=list)
    patch_off: List[int] = field(default_factory=list)           # first patch row of each sample
    n_frames: int = 0


@dataclass
class BatchPlan:
    B: int
    seq_len: int            # S: longest sample
    width: int              # S, or context_len with pad_seq
    descs: np.ndarray       # structured bytes of B neko_sample_desc
    fvals: List[torch.Tensor]
    ivals: List[torch.Tensor]
    n_f: int
    n_i: int
    first_valid: np.ndarray  # int32 [B] = seq_off
    loss_rows: np.ndarray    # int32 [n_rows] flat positions b*width+s (packed: row_base[b]+s-seq_off)
    n_valid_tokens: int
    image_groups: List[ImageGroup]
    n_patch_rows: int
    precomputed_patch: List[Tuple[int, torch.Tensor]]  # (patch_off, image_embeddings [T,P,d])
    packed: bool = False     # samples back to back, no padding rows (see build_plan)
    cu_seqlens: np.ndarray = None  # int32 [B+1]: exclusive prefix sum of the sample lengths (packed row_base, then the total)

    @property
    def token_rows(self) -> int:
        """Rows of the token-major activations: B * width padded, n_valid_tokens packed."""
        return self.n_valid_tokens if self.packed else self.B * self.width


def _is_present(d: dict, k: str) -> bool:
    return k in d and d[k] is not None


_SEL_CACHE: dict = {}   # (T, n_patches, n_text, n_obs, tokens/timestep) -> local loss-row offsets (targets at s+1)


def _loss_sel(T: int, n_patches: int, n_text: int, n_obs: int, tpt: int) -> np.ndarray:
    """Local positions s in [0, T*tpt - 1) whose NEXT token is a target (text or action; gato_policy.py:362-369,174-180)."""
    key = (T, n_patches, n_text, n_obs, tpt)
    sel = _SEL_CACHE.get(key)
    if sel is None:
        pat = np.zeros(tpt, dtype=np.uint8)
        pat[n_patches:n_patches + n_text] = 1
        pat[n_obs + 1:] = 1
        sel = np.nonzero(np.tile(pat, T)[1:])[0].astype(np.int32)
        if len(_SEL_CACHE) > 4096:
            _SEL_CACHE.clear()
        _SEL_CACHE[key] = sel
    return sel


def build_plan(inputs: Sequence[dict], *, patch_size: int, context_len: int, pad_seq: bool, packed: bool = False) -> BatchPlan:
    """Host half of tokenize_input_dicts (gato_policy.py:195-432): shapes only -- one 16-int descriptor per sample, the
    flat value lists, left-padding offsets and the loss rows.  Runs once per step on the host, so the per-sample work is
    kept to plain Python ints and list appends; descriptors become one int32 array at the end.

    ``packed``: sample b occupies rows [row_base[b], row_base[b] + L_b) of a [T = n_valid_tokens] layout with no padding rows
    (row_base = exclusive prefix sum of the lengths, stored in the descriptor).  seq_len, width and first_valid keep their
    padded values: the attention kernels take their dropout coordinates from them."""
    B = len(inputs)
    assert B > 0, "empty batch"
    fvals: List[torch.Tensor] = []
    ivals: List[torch.Tensor] = []
    n_f = n_i = 0
    groups: List[ImageGroup] = []
    pre_patch: List[Tuple[int, torch.Tensor]] = []
    pre_samples = []
    n_patch_rows = 0
    # descriptor columns, in the order of neko_sample_desc
    rows16 = []
    f32, i32 = torch.float32, torch.int32

    for b, s in enumerate(inputs):
        T = -1
        n_patches = n_text = n_cobs = n_dobs = n_cact = n_dact = 0
        text_off = cobs_off = dobs_off = cact_off = dact_off = 0
        get = s.get
        txt = get("text")
        if txt is not None:
            if isinstance(txt, list):
                # torch.Tensor(list) -> fp32 -> long in the reference (gato_policy.py:266-273); numpy parses the list faster
                txt = torch.from_numpy(np.asarray(txt, dtype=np.float32).astype(np.int32)).unsqueeze(0)
            elif txt.dim() == 1:
                txt = txt.unsqueeze(0)
            T = int(txt.shape[0])
            n_text = int(txt.shape[1])
            text_off = n_i
            t = txt.detach()
            if t.dtype != i32:
                t = t.long().to(i32)
            ivals.append(t.reshape(-1))
            n_i += t.numel()
        emb = get("image_embeddings")
        im = get("images") if emb is None else None
        if emb is not None or im is not None:
            if emb is not None:
                n_img, n_p = int(emb.shape[0]), int(emb.shape[1])
                pre_samples.append((b, emb, n_img * n_p))
            else:
                assert im.dim() == 4 and im.shape[1] == 3, "images must be [T,3,H,W]"
                h, w = int(im.shape[2]), int(im.shape[3])
                assert h % patch_size == 0 and w % patch_size == 0, "Image dimensions must be divisible by patch size"
                n_img, n_p = int(im.shape[0]), (h // patch_size) * (w // patch_size)
                is_u8 = im.dtype == torch.uint8
                if not is_u8 and im.dtype != f32:
                    im = im.to(f32)
                grp = None
                for g in groups:
                    if g.height == h and g.width == w and g.is_u8 == is_u8:
                        grp = g
                        break
                if grp is None:
                    grp = ImageGroup(h, w, is_u8)
                    groups.append(grp)
                grp.tensors.append(im)
                grp.sample_idx.append(b)
                grp.n_frames += n_img
            assert T < 0 or T == n_img, "number of timesteps must be the same for all modalities"
            T = n_img
            n_patches = n_p
        t = get("continuous_obs")
        if t is not None:
            n = int(t.shape[0])
            assert T < 0 or T == n, "number of timesteps must be the same for all modalities"
            T = n
            n_cobs = int(t.shape[1])
            cobs_off = n_f
            if t.requires_grad:
                t = t.detach()
            if t.dtype != f32:
                t = t.to(f32)
            fvals.append(t.reshape(-1))
            n_f += n * n_cobs
        t = get("discrete_obs")
        if t is not None:
            n = int(t.shape[0])
            assert T < 0 or T == n, "number of timesteps must be the same for all modalities"
            T = n
            n_dobs = int(t.shape[1])
            dobs_off = n_i
            if not isinstance(t, torch.Tensor):
                t = torch.as_tensor(t)
            if t.dtype != i32:
                t = t.to(i32)
            ivals.append(t.reshape(-1))
            n_i += n * n_dobs
        t = get("continuous_actions")
        if t is not None:
            n = int(t.shape[0])
            assert T < 0 or T == n, "number of timesteps must be the same for all modalities"
            T = n
            n_cact = int(t.shape[1])
            cact_off = n_f
            if t.requires_grad:
                t = t.detach()
            if t.dtype != f32:
                t = t.to(f32)
            fvals.append(t.reshape(-1))
            n_f += n * n_cact
        t = get("discrete_actions")
        if t is not None:
            n = int(t.shape[0])
            assert T < 0 or T == n, "number of timesteps must be the same for all modalities"
            T = n
            n_dact = int(t.shape[1])
            dact_off = n_i
            if not isinstance(t, torch.Tensor):
                t = torch.as_tensor(t)
            if t.dtype != i32:
                t = t.to(i32)
            ivals.append(t.reshape(-1))
            n_i += n * n_dact
        assert T >= 0, "sample has no modality"
        rows16.append([T, n_patches, n_text, n_cobs, n_dobs, n_cact, n_dact, 0,
                       text_off, cobs_off, dobs_off, cact_off, dact_off, 0, 0, 0])

    desc = np.array(rows16, dtype=np.int32)                 # [B, 16] == neko_sample_desc[B]
    # patch rows: one contiguous range per image group (one kernel launch each), then caller-supplied embeddings
    for g in groups:
        n_p = (g.height // patch_size) * (g.width // patch_size)
        for k, b in enumerate(g.sample_idx):
            g.patch_off.append(n_patch_rows)
            desc[b, 13] = n_patch_rows
            n_patch_rows += int(g.tensors[k].shape[0]) * n_p
    for b, emb, n in pre_samples:
        pre_patch.append((n_patch_rows, emb))
        desc[b, 13] = n_patch_rows
        n_patch_rows += n

    n_obs = desc[:, 1] + desc[:, 2] + desc[:, 3] + desc[:, 4]
    tpt = n_obs + 1 + desc[:, 5] + desc[:, 6]
    lengths = desc[:, 0] * tpt
    S = int(lengths.max())
    width = context_len if (pad_seq and context_len > S) else S
    first_valid = (S - lengths).astype(np.int32)
    desc[:, 7] = first_valid
    cu_seqlens = np.zeros(B + 1, dtype=np.int32)
    np.cumsum(lengths, out=cu_seqlens[1:])
    if packed:
        desc[:, 14] = cu_seqlens[:B]
    rows = []
    for b in range(B):
        # loss row s: token s valid (s >= off) and target mask at s+1 set, s+1 < S.  The selected offsets stop before the
        # sample's last token, so the target row + 1 stays inside the sample in the packed layout too.
        sel = _loss_sel(int(desc[b, 0]), int(desc[b, 1]), int(desc[b, 2]), int(n_obs[b]), int(tpt[b]))
        rows.append(sel + (int(cu_seqlens[b]) if packed else b * width + int(first_valid[b])))
    loss_rows = np.concatenate(rows).astype(np.int32, copy=False) if rows else np.zeros(0, dtype=np.int32)
    raw = desc.view(np.uint8).reshape(-1)
    return BatchPlan(B=B, seq_len=S, width=width, descs=raw, fvals=fvals, ivals=ivals, n_f=n_f, n_i=n_i,
                     first_valid=first_valid, loss_rows=loss_rows, n_valid_tokens=int(lengths.sum()),
                     image_groups=groups, n_patch_rows=n_patch_rows, precomputed_patch=pre_patch, packed=packed,
                     cu_seqlens=cu_seqlens)


class Stager:
    """One pinned host buffer + one device buffer per batch: every small input (descriptors, scalars, ids,
    loss rows) crosses PCIe in a single cudaMemcpyAsync."""

    RING = 3  # pinned staging buffers in rotation: the host may run this many steps ahead of the copy engine

    def __init__(self, device: torch.device):
        self.device = device
        self._ring = []          # [(pinned buffer, event recorded after its last H2D copy)]
        self._next = 0
        self._pinned: Optional[torch.Tensor] = None
        self._dev: Optional[torch.Tensor] = None
        self.generation = 0      # bumped by every upload: a staged batch knows whether the device buffer still holds it

    def _ensure(self, nbytes: int):
        if self._dev is None or self._dev.numel() < nbytes:
            cap = max(nbytes, 1 << 20)
            cap = 1 << (cap - 1).bit_length()
            torch.cuda.synchronize(self.device)
            self._ring = [(torch.empty(cap, dtype=torch.uint8, pin_memory=True), torch.cuda.Event()) for _ in range(self.RING)]
            self._dev = torch.empty(cap, dtype=torch.uint8, device=self.device)
        # the asynchronous copy out of a pinned buffer must have run before the host overwrites it again
        self._pinned, self._event = self._ring[self._next]
        self._next = (self._next + 1) % self.RING
        self._event.synchronize()

    HEADER = 256  # bytes at offset 0 of the staging buffer: per-step scalars (dropout seed words)

    def upload(self, plan: BatchPlan, header: Optional[np.ndarray] = None):
        """Returns device views: descs(u8), fvals(f32), ivals(i32), first_valid(i32), loss_rows(i32), cu_seqlens(i32), the
        number of host->device bytes moved and the int32 view of the header region."""
        def al(n):
            return (n + 255) // 256 * 256
        host_f = all(not t.is_cuda for t in plan.fvals)
        host_i = all(not t.is_cuda for t in plan.ivals)
        # every region always exists in the (pointer-stable) device buffer, whatever the source of the values: CUDA
        # graphs captured on this batch shape keep reading the same addresses
        sizes = [plan.descs.nbytes, plan.n_f * 4, plan.n_i * 4, plan.first_valid.nbytes, plan.loss_rows.nbytes, plan.cu_seqlens.nbytes]
        offs = np.cumsum([self.HEADER] + [al(s) for s in sizes])
        total = int(offs[-1])
        self._ensure(total)
        pin = self._pinned
        dev = self._dev

        def view(i, dtype):
            return dev[offs[i]:offs[i] + sizes[i]].view(dtype)

        h2d = 0
        hdr = np.zeros(self.HEADER // 4, dtype=np.int32)
        if header is not None:
            hdr[:header.size] = header.view(np.int32)
        pin[:self.HEADER] = torch.from_numpy(hdr.view(np.uint8))
        # descriptors + first_valid + loss rows (+ host-resident values): one pinned -> device copy each contiguous run
        pin[offs[0]:offs[0] + sizes[0]] = torch.from_numpy(plan.descs)
        if host_f and plan.n_f:
            torch.cat(plan.fvals, out=pin[offs[1]:offs[1] + sizes[1]].view(torch.float32))
        if host_i and plan.n_i:
            torch.cat(plan.ivals, out=pin[offs[2]:offs[2] + sizes[2]].view(torch.int32))
        pin[offs[3]:offs[3] + sizes[3]] = torch.from_numpy(plan.first_valid.view(np.uint8))
        if sizes[4]:
            pin[offs[4]:offs[4] + sizes[4]] = torch.from_numpy(plan.loss_rows.view(np.uint8))
        pin[offs[5]:offs[5] + sizes[5]] = torch.from_numpy(plan.cu_seqlens.view(np.uint8))
        if host_f and host_i:
            dev[:total].copy_(pin[:total], non_blocking=True)
            h2d = total
        else:
            dev[:self.HEADER].copy_(pin[:self.HEADER], non_blocking=True)
            h2d += self.HEADER
            for i in range(6):
                if sizes[i] and not ((i == 1 and not host_f) or (i == 2 and not host_i)):
                    dev[offs[i]:offs[i] + sizes[i]].copy_(pin[offs[i]:offs[i] + sizes[i]], non_blocking=True)
                    h2d += sizes[i]
            # inputs already on the device (the reference's ControlTask puts them there): gather device-to-device
            if not host_f and plan.n_f:
                torch.cat([t.to(self.device) for t in plan.fvals], out=view(1, torch.float32))
            if not host_i and plan.n_i:
                torch.cat([t.to(self.device) for t in plan.ivals], out=view(2, torch.int32))
        self._event.record(torch.cuda.current_stream(self.device))
        self.generation += 1
        descs = dev[offs[0]:offs[0] + sizes[0]]
        fv = view(1, torch.float32)
        iv = view(2, torch.int32)
        return (descs, fv, iv, view(3, torch.int32), view(4, torch.int32), view(5, torch.int32), h2d,
                dev[:self.HEADER].view(torch.int32))

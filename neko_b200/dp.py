"""Data-parallel gradient synchronisation for the flat gradient arena.

Replaces what the reference gets from Accelerate -> torch DDP (train.py:26-40,107; trainer.py:176-186): a
SUM all-reduce of every gradient followed by a division by the world size, bucketed and overlapped with
backward.  Here the buckets are static arena ranges that become final in reverse execution order
(head -> blocks L-1..0 -> embeddings/image stack); GatoPolicy._engine_backward announces each range as soon
as its last kernel is enqueued, the synchroniser orders a side stream after that point and launches one NCCL
all-reduce per bucket over NVLink/NVSwitch.  There is no unused-parameter bitmap round: unused parameters are
zero ranges of the arena (SURVEY.md section 8(e)).  Per-rank loss stays a local mean (DDP semantics).

``no_sync`` (gradient accumulation, trainer.py:176) simply skips the launches until the last micro-step.
"""
from __future__ import annotations

import contextlib
from typing import List, Optional, Tuple

import torch
import torch.distributed as dist


class GradSynchronizer:
    def __init__(self, arena: torch.Tensor, group=None, bucket_bytes: int = 64 << 20, average: bool = True,
                 mode: str = "overlap", compress: str = "none", backend: str = "auto"):
        # mode "overlap": buckets fire from inside backward on a side stream; "tail": everything is reduced after backward
        # (backward then replays from its CUDA graph, and no communication kernel competes with the persistent GEMMs)
        # compress "bf16": gradients cross NVLink as bf16 (half the bytes), summed by NCCL in bf16, unpacked with the
        # 1/world factor in fp32
        assert mode in ("overlap", "tail") and compress in ("none", "bf16")
        self.mode, self.compress = mode, compress
        self._pack = None
        # backend "p2p": own all-reduce kernel over IPC-mapped peer memory (csrc/p2p_allreduce.cu), co-resident with the
        # GEMMs of backward; "nccl": torch.distributed all_reduce (also the gloo path of the CPU tests)
        if backend == "auto":
            backend = "p2p" if (arena.is_cuda and dist.is_initialized() and 2 <= dist.get_world_size(group) <= 8
                                and compress == "none" and average) else "nccl"
        self.backend = backend
        self._p2p = None
        # the p2p kernels keep all their bookkeeping on the device and may be captured into the backward CUDA graph
        self.capturable = backend == "p2p"
        self.arena = arena
        self.group = group
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.bucket_elems = max(1, bucket_bytes // arena.element_size())
        # ranges that complete within the last `tail_elems` live elements of the arena are exchanged at once instead of
        # waiting for a full bucket: at the end of backward nothing is left to hide a big exchange behind
        self.tail_elems = (48 << 20) // arena.element_size()
        # ... and what completes within the last `nccl_tail_elems` goes through NCCL (p2p backend, copy-engine protocol)
        self.nccl_tail = __import__("os").environ.get("NEKO_DP_NCCL_TAIL", "0") == "1"   # measured: no gain over the copy-engine tail (profiles/r02_dp_experiments.txt)
        self.nccl_tail_elems = (16 << 20) // arena.element_size()
        self._nccl_stream = None
        self._nccl_used = False
        self.average = average
        self.enabled = True
        self._pending: List[Tuple[int, int]] = []
        self._tick = 0
        self._works = []
        self._cuda = arena.is_cuda
        self._stream = torch.cuda.Stream(device=arena.device) if self._cuda else None
        self.launched: List[Tuple[int, int]] = []   # bucket log of the last step (tests, DESIGN.md)
        # arena ranges the caller guarantees to be zero on EVERY rank (e.g. the text rows of embed_token when no task
        # of the mix produces text tokens): averaging zeros is a no-op, so they are left out of the all-reduce
        self.skip_ranges: List[Tuple[int, int]] = []

    def require_deterministic(self):
        """Deterministic training mode (GatoPolicy.deterministic): every rank must end with the same bits on every run.  The
        p2p exchanges sum the ranks in a fixed order; NCCL's all-reduce promises no order, so it is refused."""
        if self.world > 1 and self.backend != "p2p":
            raise ValueError(f"deterministic mode needs the p2p data-parallel backend (got {self.backend!r}): NCCL's all-reduce "
                             "does not sum the ranks in a fixed order, so runs would not be bitwise reproducible")
        if self.world > 1 and self.nccl_tail:
            raise ValueError("deterministic mode cannot be combined with NEKO_DP_NCCL_TAIL=1: the tail of the exchange would go "
                             "through NCCL, whose all-reduce does not sum the ranks in a fixed order")

    # -- hook called by the backward engine -----------------------------------------------------------
    def on_range_ready(self, lo: int, hi: int):
        if not self.enabled or self.world == 1:
            return
        self._tick += 1
        if self._p2p is not None and self._p2p.proto == "ce" and self.mode != "tail":
            self._p2p.ce_drain(self._stream, self._tick)
        if self.mode == "tail":
            self._pending.append((lo, hi))
            return
        # coalesce small ranges (LN / bias vectors) with their neighbours up to the bucket size
        if self._pending and self._pending[-1][1] == lo and (hi - self._pending[-1][0]) <= self.bucket_elems:
            self._pending[-1] = (self._pending[-1][0], hi)
        else:
            self._flush()
            self._pending.append((lo, hi))
        if self._pending[-1][1] - self._pending[-1][0] >= self.bucket_elems or self._live_after(self._pending[-1][1]) <= self.tail_elems:
            # full bucket -- or close to the end of backward, where whatever waits for company is exposed later
            self._flush()

    def _flush(self):
        pieces = [(a, b) for lo, hi in self._pending for a, b in self._minus_skipped(lo, hi)]
        self._pending = []
        if self._cuda and self.backend == "p2p" and pieces and self._p2p_state().proto == "ce":
            # the very end of backward (the last layer's matrices, the embedding tables): no GEMM is left to disturb and
            # nothing left to hide a multi-step exchange behind -- NCCL's one-kernel all-reduce is the shortest path there
            if self.nccl_tail:
                late = [(a, b) for a, b in pieces if self._live_after(b) <= self.nccl_tail_elems]
                pieces = [pc for pc in pieces if pc not in late]
                for a, b in late:
                    self._launch_nccl(a, b)
            # copy-engine exchange: buckets are lists of ranges -- large pieces are cut at the bucket size, small neighbours
            # (contiguous or not) share one exchange, i.e. one pair of flag rounds
            group, total = [], 0
            for a, b in pieces:
                for s0 in range(a, b, self.bucket_elems):
                    e0 = min(b, s0 + self.bucket_elems)
                    if group and total + (e0 - s0) > self.bucket_elems:
                        self._launch_group(group)
                        group, total = [], 0
                    group.append((s0, e0))
                    total += e0 - s0
            if group:
                self._launch_group(group)
            return
        for a, b in pieces:
            # split oversized ranges so that the first chunk can start while later ones are still queued
            for s in range(a, b, self.bucket_elems):
                self._launch(s, min(b, s + self.bucket_elems))

    def _launch_nccl(self, lo: int, hi: int):
        self.launched.append((lo, hi))
        if self._nccl_stream is None:
            self._nccl_stream = torch.cuda.Stream(device=self.arena.device)
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream(self.arena.device))
        with torch.cuda.stream(self._nccl_stream):
            self._nccl_stream.wait_event(ev)
            view = self.arena[lo:hi]
            if self.average:
                dist.all_reduce(view, op=dist.ReduceOp.AVG, group=self.group)
            else:
                dist.all_reduce(view, op=dist.ReduceOp.SUM, group=self.group)
        self._nccl_used = True

    def _launch_group(self, group):
        self.launched.extend(group)
        self._p2p.ce_submit(list(group), 1.0 / self.world if self.average else 1.0, self._stream, self._tick)

    def _live_after(self, pos: int) -> int:
        """Arena elements after `pos` that still take part in the exchange (the arena is laid out in completion order)."""
        return sum(b - a for a, b in self._minus_skipped(pos, self.arena.numel()))

    def _minus_skipped(self, lo: int, hi: int):
        out = [(lo, hi)]
        for slo, shi in self.skip_ranges:
            nxt = []
            for a, b in out:
                if shi <= a or slo >= b:
                    nxt.append((a, b))
                else:
                    if a < slo:
                        nxt.append((a, slo))
                    if shi < b:
                        nxt.append((shi, b))
            out = nxt
        return out

    def _launch(self, lo: int, hi: int):
        view = self.arena[lo:hi]
        self.launched.append((lo, hi))
        op = dist.ReduceOp.SUM
        if self._cuda and self.backend == "p2p" and self._p2p_state().proto == "ce":
            self._p2p.ce_submit((lo, hi), 1.0 / self.world if self.average else 1.0, self._stream, self._tick)
        elif self._cuda:
            ev = torch.cuda.Event()
            ev.record(torch.cuda.current_stream(self.arena.device))
            with torch.cuda.stream(self._stream):
                self._stream.wait_event(ev)
                if self.backend == "p2p":
                    self._p2p_state().all_reduce(lo, hi, 1.0 / self.world if self.average else 1.0)
                elif self.compress == "bf16":
                    if self._pack is None or self._pack.numel() < self.arena.numel():
                        self._pack = torch.empty(self.arena.numel(), dtype=torch.bfloat16, device=self.arena.device)
                    pk = self._pack[lo:hi]
                    pk.copy_(view)
                    dist.all_reduce(pk, op=op, group=self.group)
                    view.copy_(pk)
                    if self.average:
                        view.mul_(1.0 / self.world)
                else:
                    dist.all_reduce(view, op=op, group=self.group)
                    if self.average:
                        view.mul_(1.0 / self.world)
        else:
            dist.all_reduce(view, op=op, group=self.group)
            if self.average:
                view.mul_(1.0 / self.world)

    def _p2p_state(self):
        if self._p2p is None:
            self._p2p = _P2PState(self.arena, self.group)
        return self._p2p

    def reduce_all(self):
        """All-reduce every live range of the arena now, through the production path (bench.py's dp_grad_check, tests)."""
        self.begin_step()
        for a, b in self._minus_skipped(0, self.arena.numel()):
            for s0 in range(a, b, self.bucket_elems):
                self._launch(s0, min(b, s0 + self.bucket_elems))
        self._pending = []
        self.finish()

    # -- end of backward -----------------------------------------------------------------------------------
    def finish(self):
        """Drain pending ranges and make the compute stream wait for the communication stream."""
        if self.world == 1:
            return
        if self.enabled:
            if self.mode == "tail" and self._pending:   # one all-reduce per contiguous live span
                spans = sorted(self._pending)
                merged = [list(spans[0])]
                for lo, hi in spans[1:]:
                    if lo <= merged[-1][1]:
                        merged[-1][1] = max(merged[-1][1], hi)
                    else:
                        merged.append([lo, hi])
                self._pending = []
                for lo, hi in merged:
                    for a, b in self._minus_skipped(lo, hi):
                        self._launch(a, b)
            elif self._cuda and self.backend == "p2p" and self._p2p_state().proto == "ce":
                # everything still pending at the end of backward travels as ONE multi-range bucket: this exchange is exposed, and
                # each separate one would pay its own two flag rounds and copy launches
                self._flush()
            else:
                self._flush()
        if self._cuda:
            if self._p2p is not None and self._p2p.proto == "ce":
                self._p2p.ce_flush(self._stream)
            self._join_streams()

    def _join_streams(self):
        """The compute stream waits for every stream an exchange of this step ran on."""
        if self._nccl_used:
            torch.cuda.current_stream(self.arena.device).wait_stream(self._nccl_stream)
            self._nccl_used = False
        torch.cuda.current_stream(self.arena.device).wait_stream(self._stream)

    def begin_step(self):
        self.launched = []
        if self._p2p is not None:
            self._p2p.begin_step()

    def finish_tail(self):
        """mode "tail": called by the policy after backward (eager or graph replay) -- reduce everything now."""
        if self.world == 1 or not self.enabled:
            return
        self.begin_step()
        self._pending = list(self._tail_ranges)
        self.finish()

    @contextlib.contextmanager
    def no_sync(self):
        prev = self.enabled
        self.enabled = False
        try:
            yield
        finally:
            self.enabled = prev
            self._pending = []


class _P2PState:
    """Peer mappings + barrier bookkeeping of csrc/p2p_allreduce.cu for one arena (include/neko_b200.h: neko_ipc_*,
    neko_p2p_allreduce_f32).  Built collectively: every rank of the group must construct it at the same point."""

    def __init__(self, arena: torch.Tensor, group=None):
        import ctypes as C
        from ._lib import check, load
        self._C, self._check, self._lib = C, check, load()
        self.rank, self.world = dist.get_rank(group), dist.get_world_size(group)
        self.arena = arena
        dev = arena.device
        self.sig = torch.zeros(64, dtype=torch.int32, device=dev)          # [world] signal words (+ padding)
        self.state = torch.zeros(8, dtype=torch.int32, device=dev)         # launch counter, CTA arrival counter, signal_wait counters per channel
        self.n_ctas = int(__import__('os').environ.get('NEKO_P2P_CTAS', 0)) or int(self._lib.neko_sm_count())
        # protocol: "ce" (default) copy engines move the data, one-warp flag kernels + a local reduction; "push" / "pull"
        # SM-resident kernels (csrc/p2p_allreduce.cu explains why they lose next to the GEMMs)
        self.proto = __import__('os').environ.get('NEKO_P2P_PROTO', 'ce')
        assert self.proto in ("ce", "push", "pull")
        self.push = self.proto != "pull"
        # staging for the push protocol: `world` planes; plane r receives rank r's contributions to the slices this rank owns
        self.plane = ((arena.numel() + self.world - 1) // self.world + 4 * 8192 + 63) // 64 * 64
        self.stage = torch.empty(self.world * self.plane, dtype=torch.float32, device=dev) if self.push else None
        self.stage_off = 0
        self._ce_fifo = []
        self._peer_streams = None
        self._comm = None
        self._n_submitted = 0
        self.two_channels = __import__('os').environ.get('NEKO_P2P_CHANNELS', '2') != '1'
        self.trace = None
        torch.cuda.synchronize(dev)

        def export(t):
            h = (C.c_ubyte * 64)()
            off = C.c_longlong(0)
            check(self._lib.neko_ipc_export(C.c_void_p(t.data_ptr()), h, C.byref(off)), "neko_ipc_export")
            return bytes(h), int(off.value)

        mine = {"arena": export(arena), "sig": export(self.sig), "numel": arena.numel(), "pid": __import__("os").getpid(),
                "stage": export(self.stage) if self.push else None}
        every = [None] * self.world
        dist.all_gather_object(every, mine, group=group)
        if any(e["numel"] != arena.numel() for e in every):
            raise RuntimeError("p2p all-reduce: the ranks' gradient arenas differ in size")
        self._opened = []

        def imp(pair):
            h = (C.c_ubyte * 64).from_buffer_copy(pair[0])
            out = C.c_void_p(0)
            check(self._lib.neko_ipc_import(h, C.c_longlong(pair[1]), C.byref(out)), "neko_ipc_import")
            self._opened.append((out.value, pair[1]))
            return out.value

        bufs, sigs, stages = [], [], []
        for r, e in enumerate(every):
            if r == self.rank:
                bufs.append(arena.data_ptr())
                sigs.append(self.sig.data_ptr())
                stages.append(self.stage.data_ptr() if self.push else 0)
            else:
                bufs.append(imp(e["arena"]))
                sigs.append(imp(e["sig"]))
                stages.append(imp(e["stage"]) if self.push else 0)
        self.bufs = (C.c_void_p * self.world)(*bufs)
        self.sigs = (C.c_void_p * self.world)(*sigs)
        self.stages = (C.c_void_p * self.world)(*stages) if self.push else None
        dist.barrier(group=group)      # every signal buffer is zeroed and mapped before anybody launches

    def begin_step(self):
        self.stage_off = 0
        self._n_submitted = 0

    def _mark(self, name, stream):
        """tools/dp_trace.py: a timing event on `stream` (eager mode only)."""
        if self.trace is not None:
            e = torch.cuda.Event(enable_timing=True)
            e.record(stream)
            self.trace.append((name, e))

    def _next_off(self, lo: int, hi: int) -> int:
        per = ((hi - lo) // 4 + self.world - 1) // self.world * 4 + 16
        if self.stage_off + per > self.plane:     # a caller that never calls begin_step: wrap (buckets this far apart never overlap in time)
            self.stage_off = 0
        off = self.stage_off
        self.stage_off += per
        return off

    # ---- copy-engine protocol: a two-stage pipeline over the buckets of one backward --------------------------------
    # bucket k ready  -> [comm stream]    DMA-push my copy of slice p into rank p's staging plane (one copy stream per peer, so the
    #                    W-1 copies run on different engines at once), flag round
    # >= 2 hook calls later (or finish) -> [COMPUTE stream] reduce slice r of bucket k: a wide, short kernel between two kernels of
    #                    backward (a reduction kernel on the side stream would hold SMs the next persistent GEMM needs)
    #                 -> [comm stream]    DMA-broadcast the reduced slice into every arena, flag round
    # A bucket is a LIST of arena ranges exchanged under one pair of flag rounds (the small ranges at the end of backward --
    # image stack, position tables, separator, the non-text rows of embed_token -- travel together with the last layer).
    def _fan_out(self, comm, copies, ch: int = 0):
        """copies: [(peer, dst_ptr, src_ptr, bytes)].  Runs them on the per-peer copy streams, forked from / joined into `comm`."""
        C, lib, check = self._C, self._lib, self._check
        if not copies:
            return
        if self.world == 2 or len({c[0] for c in copies}) == 1:
            st = C.c_void_p(comm.cuda_stream)
            for _p, dst, src, nb in copies:
                check(lib.neko_memcpy_async(C.c_void_p(dst), C.c_void_p(src), C.c_longlong(nb), st), "neko_memcpy_async")
            return
        if self._peer_streams is None:
            self._peer_streams = [[torch.cuda.Stream(device=self.arena.device) for _ in range(self.world)] for _c in range(2)]
        fork = torch.cuda.Event()
        fork.record(comm)
        used = []
        for p, dst, src, nb in copies:
            ps = self._peer_streams[ch][p]
            if ps not in used:
                ps.wait_event(fork)
                used.append(ps)
            check(lib.neko_memcpy_async(C.c_void_p(dst), C.c_void_p(src), C.c_longlong(nb), C.c_void_p(ps.cuda_stream)), "neko_memcpy_async")
        for ps in used:
            j = torch.cuda.Event()
            j.record(ps)
            comm.wait_event(j)

    def _signal(self, comm, ch: int = 0):
        C = self._C
        self._check(self._lib.neko_p2p_signal_wait(self.sigs, C.c_void_p(self.state.data_ptr()), C.c_int(self.rank), C.c_int(self.world),
                                                   C.c_int(ch), C.c_void_p(comm.cuda_stream)), "neko_p2p_signal_wait")

    def _channel(self, comm):
        """Buckets alternate between two exchange streams (own flag channel each): the push of bucket k+1 does not queue
        behind the broadcast of bucket k."""
        if self._comm is None or self._comm[0] is not comm:
            self._comm = [comm, torch.cuda.Stream(device=self.arena.device)]
        ch = self._n_submitted % 2 if self.two_channels else 0
        self._n_submitted += 1
        return ch, self._comm[ch]

    def ce_submit(self, ranges, scale: float, comm, tick: int = 0):
        if isinstance(ranges, tuple):
            ranges = [ranges]
        cur = torch.cuda.current_stream(self.arena.device)
        W, r = self.world, self.rank
        ch, comm = self._channel(comm)
        offs = [self._next_off(lo, hi) for lo, hi in ranges]
        ev = torch.cuda.Event()
        ev.record(cur)
        tag = "+".join(f"[{lo >> 20}M..{hi >> 20}M)" for lo, hi in ranges)
        self._mark("ready   " + tag, cur)
        mine = self.arena.data_ptr()
        with torch.cuda.stream(comm):
            comm.wait_event(ev)
            self._mark("  push> " + tag, comm)
            copies = []
            for (lo, hi), off in zip(ranges, offs):
                for pp in range(1, W):
                    p = (r + pp) % W
                    a, ln = self._span(lo, hi, p)
                    if ln:
                        copies.append((p, self.stages[p] + 4 * (r * self.plane + off), mine + 4 * (lo + a), 4 * ln))
            self._fan_out(comm, copies, ch)
            self._mark("  push< " + tag, comm)
            self._signal(comm, ch)
            self._mark("  land  " + tag, comm)
            landed = torch.cuda.Event()
            landed.record(comm)
        self._ce_fifo.append((list(ranges), scale, offs, landed, tick, tag, ch))

    def _span(self, lo: int, hi: int, p: int):
        n = hi - lo
        per = ((n // 4 + self.world - 1) // self.world) * 4
        a = min(n, p * per)
        return a, min(n, (p + 1) * per) - a

    def ce_drain(self, comm, tick=None, min_age: int = 2):
        """Reduce + broadcast the buckets pushed at least `min_age` hook calls ago (all of them when tick is None).  The delay is
        static (it has to be: the schedule is captured into a CUDA graph): by then the pushes have landed and the compute
        stream does not wait."""
        cur = torch.cuda.current_stream(self.arena.device)
        while self._ce_fifo and (tick is None or tick - self._ce_fifo[0][4] >= min_age):
            self._ce_reduce(self._ce_fifo.pop(0), cur)

    def _ce_reduce(self, pend, cur):
        ranges, scale, offs, landed, _tick, tag, ch = pend
        comm = self._comm[ch]
        C, lib, check, W, r = self._C, self._lib, self._check, self.world, self.rank
        mine = self.arena.data_ptr()
        self._mark("red-enq " + tag, cur)
        cur.wait_event(landed)
        self._mark("red>    " + tag, cur)
        for (lo, hi), off in zip(ranges, offs):
            a, ln = self._span(lo, hi, r)
            if ln:
                check(lib.neko_reduce_planes_f32(C.c_void_p(mine + 4 * (lo + a)), C.c_void_p(self.stage.data_ptr() + 4 * off),
                                                 C.c_longlong(self.plane), C.c_int(W), C.c_int(r), C.c_longlong(ln), C.c_float(scale),
                                                 C.c_void_p(cur.cuda_stream)), "neko_reduce_planes_f32")
        reduced = torch.cuda.Event()
        reduced.record(cur)
        self._mark("red<    " + tag, cur)
        with torch.cuda.stream(comm):
            comm.wait_event(reduced)
            self._mark("  bcast>" + tag, comm)
            copies = []
            for lo, hi in ranges:
                a, ln = self._span(lo, hi, r)
                if ln:
                    for pp in range(1, W):
                        p = (r + pp) % W
                        copies.append((p, self.bufs[p] + 4 * (lo + a), mine + 4 * (lo + a), 4 * ln))
            self._fan_out(comm, copies, ch)
            self._mark("  bcast<" + tag, comm)
            self._signal(comm, ch)
            self._mark("  done  " + tag, comm)

    def ce_flush(self, comm):
        """Drain the pipeline; afterwards `comm` (the synchroniser's stream) is ordered after both exchange streams."""
        self.ce_drain(comm, None)
        if self._comm is not None and self._comm[1] is not comm:
            comm.wait_stream(self._comm[1])

    def all_reduce(self, lo: int, hi: int, scale: float):
        C = self._C
        if self.proto == "ce":      # standalone use (tools): the same pipeline, drained at once on one stream
            cur = torch.cuda.current_stream(self.arena.device)
            self.ce_submit((lo, hi), scale, cur)
            return self.ce_flush(cur)
        off = self._next_off(lo, hi)
        self._check(self._lib.neko_p2p_allreduce_f32(self.bufs, self.sigs, self.stages, C.c_longlong(self.plane), C.c_longlong(off),
                                                     C.c_void_p(self.state.data_ptr()), C.c_int(self.rank),
                                                     C.c_int(self.world), C.c_longlong(lo), C.c_longlong(hi),
                                                     C.c_float(scale), C.c_int(self.n_ctas),
                                                     C.c_void_p(torch.cuda.current_stream().cuda_stream)), "neko_p2p_allreduce_f32")


def attach(policy, group=None, bucket_bytes: int = 64 << 20, no_text_tokens: bool = False, mode: str = "overlap",
           compress: str = "none", backend: str = "auto") -> GradSynchronizer:
    """Wire a GradSynchronizer to a GatoPolicy: buckets fire from inside ``loss.backward()``.

    ``no_text_tokens``: the caller guarantees that no rank ever feeds text tokens (a task mix with
    text_prop = caption_prop = vqa_prop = 0, trainer.py:134): rows [0, text_tokens) of ``embed_token`` -- 154 MB of the
    last, non-overlappable bucket -- then have zero gradient everywhere and are left out of the all-reduce, like the
    never-used ``transformer.wte``.  The result is identical to the dense all-reduce."""
    sync = GradSynchronizer(policy._grad_arena, group=group, bucket_bytes=bucket_bytes, mode=mode, compress=compress, backend=backend)
    if getattr(policy, "deterministic", False):
        sync.require_deterministic()
    if sync.backend == "p2p" and sync.world > 1:
        sync._p2p = _P2PState(policy._grad_arena, group)     # collective: map the peers' arenas now, not inside backward
    if no_text_tokens:
        o = policy._offs["embed_token.weight"]
        sync.skip_ranges.append((o, o + policy.text_tokens * policy.embed_dim))
        w = policy._offs["transformer.wte.weight"]
        sync.skip_ranges.append((w, w + policy._params["transformer.wte.weight"].numel()))
    if mode == "tail":
        # nothing fires inside backward: it keeps replaying from its CUDA graph; the policy calls sync.finish_tail() after it
        policy.grad_ready_hook = None
        sync._tail_ranges = _live_ranges(policy)
    else:
        policy.grad_ready_hook = sync.on_range_ready
    policy._grad_sync = sync
    return sync


def _live_ranges(policy):
    """Arena span of every parameter that can carry a gradient (everything but transformer.wte)."""
    total = policy._grad_arena.numel()
    w = policy._offs["transformer.wte.weight"]
    return [(0, w)] + ([(w + 64, total)] if w + 64 < total else [])


def broadcast_parameters(policy, src: int = 0, group=None):
    """All ranks start from rank ``src``'s weights (what DDP does at wrap time)."""
    if dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.broadcast(policy._param_arena, src=src, group=group)
        policy._bf16_versions = None

"""Launch plans: what every engine (engine.py, engine_fp32.py, train.py, vae.py, clip.py) is built from.

A plan is a list of closures over pre-allocated buffers, each calling ONE ops function.  It is built once per geometry and then
run eagerly or captured into a CUDA graph and replayed.  Buffer recycling, the recording of GEMM / dgrad / wgrad / GroupNorm
entries, graph capture and the context cache live here once, so that a change to how a plan is built is made in one place."""
from __future__ import annotations

import ctypes as C
import weakref

import torch

from . import ops
from ._lib import check, lib


class Pool:
    """Size-keyed free lists of row-major buffers; safe because all work is stream-ordered."""

    def __init__(self, device):
        self.device, self.free, self.total = device, {}, 0

    def get(self, rows, cols, dtype=torch.bfloat16):
        lst = self.free.get((rows * cols, dtype))
        if lst:
            return lst.pop().view(rows, cols)
        self.total += rows * cols * (2 if dtype == torch.bfloat16 else 4)
        return torch.empty(rows, cols, dtype=dtype, device=self.device)

    def put(self, *ts):
        for t in ts:
            if t is not None:
                self.free.setdefault((t.numel(), t.dtype), []).append(t)


class Plan(list):
    """List of launch closures + parallel metadata (kind, algorithmic flops, name) for profiling."""

    def __init__(self):
        super().__init__()
        self.meta = []

    def append(self, fn, kind="other", flops=0.0, name=""):
        super().append(fn)
        self.meta.append((kind, float(flops), name))


def run_plan(plan):
    for op in plan:
        op()


def capture(plan, capture_error_mode="global"):
    """Run `plan` eagerly -- that run is the caller's result (a backward plan accumulates gradients, so it must run exactly once)
    and does the lazy one-time setup (function attributes, workspaces) outside any capture -- then capture it into a CUDA graph.
    Returns (graph, launches per replay).  A plan built for autograd's backward is captured on autograd's thread and needs
    capture_error_mode="thread_local"."""
    run_plan(plan)
    torch.cuda.current_stream().synchronize()
    g = torch.cuda.CUDAGraph()
    before = ops.launch_count()
    with torch.cuda.graph(g, capture_error_mode=capture_error_mode):
        run_plan(plan)
    return g, ops.launch_count() - before


class ContextKey:
    """Which text context the hoisted K/V projections were computed from: the SAME live tensor object at the same version.  (A key
    of (data_ptr, version, shape) took a new context tensor that the caching allocator placed at the freed address of the
    previous one -- same shape, version 0 -- for the old one, and sampled with stale K/V.)"""

    def __init__(self):
        self.ref, self.version = None, None

    def matches(self, ctx):
        return self.ref is not None and self.ref() is ctx and self.version == ctx._version

    def set(self, ctx):
        self.ref, self.version = weakref.ref(ctx), ctx._version


class Builder:
    """Recording helpers shared by the engines.  Each appends one closure calling one ops function over arguments prepared at
    build time, and keeps alive every tensor that a recorded launch points at."""

    def __init__(self, device):
        self.device = device
        self._keep = []
        self._gn_parts = {}     # id(fp32 activation buffer) -> ops.GnParts describing its CURRENT contents (plan-build time)

    def gemm(self, plan, a0, w, out, *, rowbias_ptr=None, gn_hw=0, kind=None, name=None, **kw):
        """out = [a0 | a1] w^T (+ epilogue terms, see ops.gemm).  rowbias_ptr = (address, ld, rows per image) of a per-image bias
        row; gn_hw > 0: `out` feeds a GroupNorm over gn_hw rows per image -- the epilogue also emits its column statistics."""
        args = ops.gemm(a0, w, out, launch=False, **kw)
        if rowbias_ptr is not None:
            args.rowbias, args.ldrb, args.rows_per_image = rowbias_ptr
        self._gn_parts.pop(id(out), None)      # whatever statistics described this (pooled) buffer are stale now
        if gn_hw > 0:
            parts = ops.gemm_attach_gn_parts(args, gn_hw, self.device)
            if parts is not None:
                self._gn_parts[id(out)] = parts
                self._keep.append(parts)       # the captured launch writes into parts.buf on every replay: it must outlive
                #                                its entry in _gn_parts (popped when the pooled buffer is produced again)
        self._keep.append((a0, w, out, kw))
        k = "conv3x3" if args.conv_taps == 9 else "gemm"
        plan.append(lambda a=args: ops.gemm_run(a), kind or k, 2.0 * args.M * args.N * args.K,
                    name or f"{k} M{args.M} N{args.N} K{args.K}")

    def dgrad(self, plan, dy, w, out, *, name=None, **kw):
        """out = dy (*) w (+ residual): the data gradient of gemm() (ops.gemm_dgrad)."""
        args = ops.gemm_dgrad(dy, w, out, launch=False, **kw)
        self._keep.append((dy, w, out, kw))
        plan.append(lambda a=args: ops.gemm_dgrad_run(a), "gemm", 2.0 * args.M * args.Cout * args.Cin * args.conv_taps,
                    name or f"dgrad M{args.M} N{args.Cin} K{args.Cout * args.conv_taps}")

    def wgrad(self, plan, dy, x, dw, **kw):
        """dw += dy^T (*) x (ops.gemm_wgrad); nothing is recorded when dw is None (frozen weights)."""
        if dw is None:
            return
        args = ops.gemm_wgrad(dy, x, dw, launch=False, **kw)
        self._keep.append((dy, x, dw, kw))
        plan.append(lambda a=args: ops.gemm_wgrad_run(a), "gemm", 2.0 * args.rows * args.Cout * args.Cin * args.conv_taps,
                    f"wgrad M{args.Cout} N{args.Cin * args.conv_taps} K{args.rows}")

    def groupnorm(self, plan, x, skip, g, b, out, batch, hw, eps, silu, *, groups=32, raw_out=None, stats_out=None):
        """GroupNorm(+SiLU, + channel concat of skip): apply-only from the producers' epilogue statistics when every source has
        them, else the stand-alone kernel (which computes the statistics itself)."""
        p0 = self._gn_parts.get(id(x))
        p1 = self._gn_parts.get(id(skip)) if skip is not None else None
        Cc = x.shape[-1] + (skip.shape[-1] if skip is not None else 0)
        if p0 is not None and (skip is None or p1 is not None) and ops.gn_parts_supported(Cc, groups):
            self._keep.append((p0, p1))
            plan.append(lambda: ops.groupnorm_silu_parts(x, skip, p0, p1, g, b, out, batch, hw, groups, eps, silu, raw_out=raw_out,
                                                         stats_out=stats_out), "groupnorm", 0, "groupnorm (stats from GEMM)")
        else:
            plan.append(lambda: ops.groupnorm_silu(x, skip, g, b, out, batch, hw, groups, eps, silu, raw_out=raw_out,
                                                   stats_out=stats_out), "groupnorm")


def profile_plan(plan, device, iters=5):
    """Per-launch device time of every entry of a launch plan measured INSIDE the step: the whole plan is captured once more
    into a CUDA graph with an external event-record node (b200sd_timer_record) between consecutive entries, and the replays are
    read back per entry.  Every kernel therefore runs under the conditions of the real step -- its weights streaming cold from
    HBM, its input left in L2 by its true predecessor, no host launch gaps.  (The first version replayed each entry four
    times back to back in a graph of its own: warm weights, optimistic.)  Returns ({kind: [ms, flops, launches]} per step,
    [(name, ms, flops)] per entry, ms of the whole instrumented replay)."""
    with torch.cuda.device(device):
        entries = [(op, meta) for op, meta in zip(plan, plan.meta) if meta[0] != "tap"]
        n = len(entries)
        check(lib().b200sd_timer_reserve(n + 1), "timer_reserve")

        def run_all():
            for op, _m in entries:
                op()
        run_all()
        torch.cuda.synchronize()
        side = torch.cuda.Stream()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=side):
            sh = torch.cuda.current_stream().cuda_stream
            for i, (op, _meta) in enumerate(entries):
                check(lib().b200sd_timer_record(i, sh), "timer_record")
                op()
            check(lib().b200sd_timer_record(n, sh), "timer_record")
        torch.cuda.synchronize()
        times = [0.0] * n
        total = 0.0
        ms = C.c_float(0.0)
        g.replay()          # warm-up replay of the instrumented graph
        torch.cuda.synchronize()
        for _ in range(iters):
            g.replay()
            torch.cuda.synchronize()
            for i in range(n):
                check(lib().b200sd_timer_elapsed_ms(i, i + 1, C.byref(ms)), "timer_elapsed")
                times[i] += ms.value / iters
            check(lib().b200sd_timer_elapsed_ms(0, n, C.byref(ms)), "timer_elapsed")
            total += ms.value / iters
        acc, per_op = {}, []
        for t, (op, (kind, flops, name)) in zip(times, entries):
            a = acc.setdefault(kind, [0.0, 0.0, 0])
            a[0] += t
            a[1] += flops
            a[2] += 1
            per_op.append((name or kind, t, flops))
        run_all()
        torch.cuda.synchronize()
    return acc, per_op, total

"""Recorded layer programs (include/scn_b200.h, "recorded layer programs").

A forward of the backbone makes ~100 calls into the native library, one per layer, exactly as the
reference makes one pybind call per layer.  `Trace` records those calls while an ordinary forward
runs (every feature tensor becomes a register, every parameter an index); `Program` replays them
with ONE native call.  Same kernels, same order, same results -- only the Python round trips are
gone.  Anything the recorder does not understand (a feature tensor produced by a torch op, an
unknown layer) aborts the recording and the network keeps running layer by layer.
"""
import ctypes as C

import torch

from .._lib import check, l3, lib

_ACTIVE = None  # the Trace that is currently recording (set by Trace.__enter__)


def active():
    return _ACTIVE


class Trace(object):
    def __init__(self, training=False):
        self.training = training  # a training forward is being recorded (training-mode BatchNorm, torch adds under autograd)
        self.ops = []          # (kind, [ints], [floats])
        self.regs = {}         # id(tensor) -> register
        self.params = []       # parameter / buffer tensors, index = position
        self.pindex = {}
        self.keep = []         # keeps every recorded tensor alive so ids stay unique while recording
        self.failed = None
        self.input_features = None

    def __enter__(self):
        global _ACTIVE
        self._prev, _ACTIVE = _ACTIVE, self
        return self

    def __exit__(self, *exc):
        global _ACTIVE
        _ACTIVE = self._prev
        return False

    # ---- helpers used by native.py
    def fail(self, why):
        if self.failed is None:
            self.failed = why

    def new_reg(self, t):
        self.keep.append(t)
        r = self.regs[id(t)] = len(self.regs)
        return r

    def reg(self, t):
        r = self.regs.get(id(t))
        if r is None:
            self.fail("a feature tensor was not produced by a recorded layer")
            return -1
        return r

    def param(self, t):
        if t is None or t.numel() == 0:
            return -1
        i = self.pindex.get(id(t))
        if i is None:
            i = self.pindex[id(t)] = len(self.params)
            self.params.append(t)
        return i

    def add(self, kind, ints, floats=()):
        self.ops.append((kind, [int(v) for v in ints], [float(v) for v in floats]))


def _l(t):
    return [int(v) for v in (t.tolist() if hasattr(t, "tolist") else t)]


def _hoist_pointwise(ops):
    """Move every 1x1x1 SubmanifoldConvolution right behind the op that produces its input.  In the FPN
    these are the lateral 'shortcut' convolutions: the network calls them in the top-down pass, but
    they only depend on the bottom-up features, so they can run while the GPU waits for the deeper
    levels' rulebooks instead of lengthening the tail of the forward.  Same op, same input: same result."""
    ops = list(ops)
    out = []
    for op in ops:
        kind, ints, _ = op
        if kind == 1 and ints[5:8] == [1, 1, 1]:
            src = ints[0]
            pos = None
            for j in range(len(out) - 1, -1, -1):
                k2, i2, _f = out[j]
                produced = i2[0] if k2 == 0 else (i2[2] if k2 == 5 else i2[1])
                if produced == src:
                    pos = j + 1
                    break
            if pos is not None:
                out.insert(pos, op)
                continue
        out.append(op)
    return out


class Program(object):
    """A finished recording bound to the native executor."""

    def __init__(self, trace, outputs, math_mode):
        """outputs: list of (feature tensor, spatial_size LongTensor) in the order the network returns them."""
        if trace.failed:
            raise RuntimeError(trace.failed)
        self.math_mode = math_mode
        self.training = trace.training
        self.params = trace.params
        self.out_regs, self.out_sizes = [], []
        for feats, size in outputs:
            r = trace.regs.get(id(feats))
            if r is None:
                raise RuntimeError("an output was not produced by a recorded layer")
            self.out_regs.append(r)
            self.out_sizes.append(size.clone())
        ops = _hoist_pointwise(trace.ops)
        self.planes = next((ints[6] for kind, ints, _ in ops if kind == 0), None)  # channels of the network input
        self._h = C.c_void_p()
        check(lib().scn_program_create(C.byref(self._h)))
        for kind, ints, floats in ops:
            ia = (C.c_long * len(ints))(*ints)
            fa = (C.c_double * max(1, len(floats)))(*floats) if floats else None
            check(lib().scn_program_add(self._h, kind, ia, len(ints), fa, len(floats)))
        uniq = sorted(set(self.out_regs))
        check(lib().scn_program_finish(self._h, len(trace.regs), (C.c_int * len(uniq))(*uniq), len(uniq)))
        self.n_ops = len(trace.ops)
        self._prepared = []  # Metadata of training steps prepared ahead: the native program reads them until they run or are dropped
        if self.training:
            check(lib().scn_program_set_training(self._h, 1))

    def __del__(self):
        h = getattr(self, "_h", None)
        if h:
            try:
                lib().scn_program_destroy(h)
            except Exception:
                pass
            self._h = None

    def usable(self, coords, feats, math_mode):
        # (a wrongly shaped input takes the layer-by-layer path, whose asserts then raise as the reference's would)
        return (math_mode == self.math_mode and isinstance(feats, torch.Tensor) and feats.is_cuda and feats.dtype == torch.float32
                and feats.dim() == 2 and coords.dtype == torch.int64 and coords.dim() == 2 and coords.size(1) in (3, 4)
                and feats.size(0) == coords.size(0) and feats.size(1) == self.planes)

    def throttle(self):
        """Wait until at most one forward of this program is still running (scn_program_throttle)."""
        check(lib().scn_program_throttle(self._h))

    def prepare(self, metadata, coords):
        """Build half of a run for `coords` (see scn_program_prepare): input layer + rulebook workers, on the library's
        build streams.  Device coordinates must be complete (no pending writes on any stream)."""
        coords = coords.contiguous()
        metadata._keep.append(coords)
        check(lib().scn_program_prepare(self._h, metadata._h, C.c_void_p(coords.data_ptr()), 2 if coords.is_cuda else 0, coords.size(0), coords.size(1)))

    def prepare_training(self, metadata, coords):
        """Training program: build ahead, for a later training step on `metadata`, what that step would build before its first
        layer (scn_program_prepare_training).  At most two steps stay prepared; a third drops the oldest."""
        coords = coords.contiguous()
        metadata._keep.append(coords)
        check(lib().scn_program_prepare_training(self._h, metadata._h, C.c_void_p(coords.data_ptr()), 2 if coords.is_cuda else 0,
                                                 coords.size(0), coords.size(1)))
        self._prepared.append(metadata)
        del self._prepared[:-2]

    def drop_prepared(self):
        """Forget every training step prepared ahead (scn_program_drop_prepared): their memory is released."""
        check(lib().scn_program_drop_prepared(self._h))
        self._prepared = []

    def run(self, metadata, coords, feats):
        """-> (list of output feature tensors, multiply-add count)."""
        from . import native
        self._prepared = [m for m in self._prepared if m is not metadata]  # (the run takes it out of the native program's list)
        coords = coords.contiguous()
        feats = feats.contiguous()
        metadata._keep.append(coords)
        n = len(self.params)
        ptrs = (C.c_void_p * n)(*[p.data_ptr() for p in self.params])
        tags = (C.c_longlong * n)(*[native._weight_tag(p) if p.dim() >= 3 else 0 for p in self.params])
        macs = C.c_double()
        stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        check(lib().scn_program_run(self._h, metadata._h, C.c_void_p(coords.data_ptr()), int(coords.is_cuda), coords.size(0), coords.size(1),
                                    C.c_void_p(feats.data_ptr()), ptrs, tags, n, stream, C.byref(macs)))
        uniq, tens = [], {}
        for r, size in zip(self.out_regs, self.out_sizes):
            if r not in tens:
                rows, cols, ptr = C.c_long(), C.c_int(), C.c_void_p()
                check(lib().scn_program_output(self._h, r, C.byref(rows), C.byref(cols), C.byref(ptr)))
                tens[r] = torch.empty((rows.value, cols.value), dtype=torch.float32, device=feats.device)
                if tens[r].numel():
                    uniq.append((r, size))
        # rows in the numbering of `metadata` (the executor may have computed them in its internal order): one launch for all maps
        for k in range(0, len(uniq), 8):
            part = uniq[k:k + 8]
            regs = (C.c_int * len(part))(*[r for r, _ in part])
            sizes = (C.c_long * (3 * len(part)))(*[int(v) for _, size in part for v in size.tolist()])
            dst = (C.c_void_p * len(part))(*[tens[r].data_ptr() for r, _ in part])
            check(lib().scn_program_outputs_copy(self._h, metadata._h, len(part), regs, sizes, dst))
        outs = [tens[r] for r in self.out_regs]
        return outs, macs.value

    def backward(self, regs, d_outs, want_d_features, n_in_rows):
        """Backward pass of the last training run (scn_program_backward).  d_outs[i]: gradient (or None) of output register
        regs[i].  -> (one gradient tensor or None per recorded parameter, gradient of the network input or None)."""
        n = len(self.params)
        pairs = [(r, g.contiguous()) for r, g in zip(regs, d_outs) if g is not None and g.numel()]
        # grad_sink (set by distributed.GradientReducer.attach): parameter index -> tensor the gradient is WRITTEN into (a view of the
        # reducer's flat buffer, zeroed by the reducer every step); such parameters return no gradient to autograd.  grad_events:
        # parameter index -> torch.cuda.Event recorded behind the kernels that write that gradient.
        sink = getattr(self, "grad_sink", None) or {}
        events = getattr(self, "grad_events", None) or {}
        grads = [sink[i] if i in sink else (torch.empty_like(p) if (p.requires_grad and p.is_floating_point()) else None) for i, p in enumerate(self.params)]
        d_feats = torch.empty((n_in_rows, self.planes), dtype=torch.float32, device=self.params[0].device) if want_d_features else None
        ptrs = (C.c_void_p * n)(*[p.data_ptr() for p in self.params])
        gptrs = (C.c_void_p * n)(*[None if g is None else g.data_ptr() for g in grads])
        live = (C.c_int * n)()
        k = max(1, len(pairs))
        evs = (C.c_void_p * n)(*[events[i].cuda_event if i in events else None for i in range(n)]) if events else None
        check(lib().scn_program_backward(self._h, len(pairs), (C.c_int * k)(*[r for r, _ in pairs]), (C.c_void_p * k)(*[g.data_ptr() for _, g in pairs]),
                                         ptrs, gptrs, n, None if d_feats is None else C.c_void_p(d_feats.data_ptr()), live, evs))
        self.last_live = [bool(live[i]) for i in range(n)]
        out = [g if (g is not None and live[i] and i not in sink) else None for i, g in enumerate(grads)]
        cb = getattr(self, "after_backward", None)
        if cb is not None:  # (the kernels of the whole backward pass are queued; the reducer launches its buckets behind their events)
            cb(self)
        return out, d_feats


class TrainFunction(torch.autograd.Function):
    """One autograd node for a whole replayed training forward: forward = scn_program_run in training mode, backward =
    scn_program_backward (the reference: one node per layer, ~100 per forward).  Returns one tensor per DISTINCT output
    register, in the order of sorted(set(prog.out_regs))."""

    @staticmethod
    def forward(ctx, prog, md, coords, feats, *params):
        outs, macs = prog.run(md, coords, feats)
        prog.last_macs = macs
        prog.run_id = getattr(prog, "run_id", 0) + 1
        ctx.prog, ctx.md, ctx.n_in, ctx.run_id = prog, md, feats.size(0), prog.run_id
        by_reg = dict(zip(prog.out_regs, outs))
        ctx.regs = sorted(by_reg)
        return tuple(by_reg[r] for r in ctx.regs)

    @staticmethod
    def backward(ctx, *d_outs):
        prog = ctx.prog
        if ctx.run_id != prog.run_id:
            raise RuntimeError("replayed training step: another forward of this network ran before backward(); the activations are gone "
                               "(set SCN_TRAIN_PROGRAM=0 to train layer by layer)")
        grads, d_feats = prog.backward(ctx.regs, d_outs, ctx.needs_input_grad[3], ctx.n_in)
        grads = [g if need else None for g, need in zip(grads, ctx.needs_input_grad[4:])]
        return (None, None, None, d_feats) + tuple(grads)

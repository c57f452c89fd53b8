"""Flat fp32 parameter / gradient storage with nn.Parameter views.

All trainable tensors of a learner live in ONE contiguous device buffer so that the clip +
optimiser kernels, the target sync (one D2D copy) and the data-parallel all-reduce (one NCCL
call over [grads | loss_sum | mask_sum]) touch a single allocation.  The nn.Parameters of the
modules are re-pointed to views of that buffer, so ``state_dict()`` keeps the reference's key
names (fc1.weight, rnn.weight_ih, hyper_w1.weight, ...) and its checkpoints load unchanged.
"""
from __future__ import annotations

import torch

ALIGN = 4   # floats; every tensor starts 16-byte aligned (float4 loads in the kernels)


def _round_up(n, a=ALIGN):
    return (n + a - 1) // a * a


class FlatBuffer:
    """Packs ``[(name, parameter)]`` into one buffer, in the given order."""

    def __init__(self, named_params, device=None, with_grad=True, extra_tail=0):
        # entries are (name, param) -- start aligned to 16 bytes -- or (name, param, "tight"): placed
        # directly behind its predecessor (layer-concatenated groups that one GEMM reads as one matrix)
        entries = [(e[0], e[1], len(e) > 2 and e[2] == "tight") for e in named_params]
        named_params = [(n, p) for n, p, _ in entries]
        self.names = [n for n, _ in named_params]
        self.params = [p for _, p in named_params]
        device = device if device is not None else (self.params[0].device if self.params else torch.device("cpu"))
        self.offsets, off = {}, 0
        self._addrs = {}
        for n, p, tight in entries:
            if not tight:
                off = _round_up(off)
            self.offsets[n] = off
            off += p.numel()
        off = _round_up(off)
        self.numel = off
        self.data = torch.zeros(off, dtype=torch.float32, device=device)
        # gradient buffer carries `extra_tail` trailing floats (loss_sum, mask_sum) for the all-reduce
        self.grad_full = torch.zeros(off + extra_tail, dtype=torch.float32, device=device) if with_grad else None
        self.grad = self.grad_full[:off] if with_grad else None
        self.tail = self.grad_full[off:] if with_grad else None
        with torch.no_grad():
            for n, p in named_params:
                o = self.offsets[n]
                view = self.data[o:o + p.numel()].view(p.shape)
                view.copy_(p.detach().to(device=device, dtype=torch.float32))
                p.data = view
                if with_grad:
                    p.grad = self.grad[o:o + p.numel()].view(p.shape)

    def view(self, name, source=None):
        src = self.data if source is None else source
        i = self.names.index(name)
        o = self.offsets[name]
        return src[o:o + self.params[i].numel()].view(self.params[i].shape)

    def ptr(self, name, source=None):
        src = self.data if source is None else source
        return src.data_ptr() + 4 * self.offsets[name]

    def addrs(self, prefix, source=None):
        """name -> device address of every entry under `prefix` (the prefix stripped), in packing order: the address map
        of one module's flat_named_parameters() as packed with ``prefixed(prefix, ...)``.  Kept per (prefix, base address),
        so the returned dict is shared: do not modify it."""
        base = (self.data if source is None else source).data_ptr()
        m = self._addrs.get((prefix, base))
        if m is None:
            m = self._addrs[prefix, base] = {n[len(prefix):]: base + 4 * o for n, o in self.offsets.items() if n.startswith(prefix)}
        return m

    def adopt_grad_storage(self, grad_full):
        """Move the gradient buffer (numel + tail floats) into caller-provided device memory."""
        assert grad_full.numel() == self.grad_full.numel() and grad_full.dtype == torch.float32
        grad_full.zero_()
        self.grad_full = grad_full
        self.grad, self.tail = grad_full[:self.numel], grad_full[self.numel:]
        self.rebind_grads()

    def rebind_grads(self):
        """Re-attach p.grad views (optimizer.zero_grad(set_to_none=True) style resets drop them)."""
        for n, p in zip(self.names, self.params):
            o = self.offsets[n]
            p.grad = self.grad[o:o + p.numel()].view(p.shape)


def prefixed(prefix, entries):
    """Prefix the names of FlatBuffer entries, keeping their packing markers."""
    return [(prefix + e[0],) + tuple(e[1:]) for e in entries]


class FlatPackedMixin:
    """For nn.Modules whose kernels read several parameters as ONE contiguous matrix (QMIX's four hyper heads, the QPLEX
    layer groups, the agent): keeps that layout true for copies of the module.

    ``copy.deepcopy``, pickling and ``torch.save(module)`` clone every Parameter on its own, so the copy's tensors are no
    longer views of one buffer -- a kernel reading ``[N*E + 3E, S]`` from ``hyper_w1.weight`` would then run past the end
    of that tensor.  Copies are therefore re-packed on creation, and ``ensure_packed()`` (called by ``forward``) re-packs
    whenever a parameter no longer sits at its slot of ``self._flat`` (e.g. someone re-assigned ``p.data``)."""

    def __deepcopy__(self, memo):
        import copy
        new = self.__class__.__new__(self.__class__)
        memo[id(self)] = new
        for k, v in self.__dict__.items():
            new.__dict__[k] = None if k == "_flat" else copy.deepcopy(v, memo)
        new._pack(next(new.parameters()).device)
        return new

    def __setstate__(self, state):
        super().__setstate__(state)
        self._flat = None
        self._pack(next(self.parameters()).device)

    def ensure_packed(self):
        flat = self._flat
        ok = flat is not None
        if ok:
            for entry in self.flat_named_parameters():
                n, p = entry[0], entry[1]
                name = n if n in flat.offsets else next((k for k in flat.offsets if k.endswith("." + n)), None)
                if name is None or p.data_ptr() != flat.data.data_ptr() + 4 * flat.offsets[name] or p.device != flat.data.device:
                    ok = False
                    break
        if not ok:
            self._pack(next(self.parameters()).device)

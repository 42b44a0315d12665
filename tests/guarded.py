"""Guarded, poisoned buffers for one C-ABI call (test infrastructure).

A result must come from the call itself, not from the memory the call was handed.  The caching allocator hides the
difference: it hands the next call of the same size the block the previous call left its (often correct) answer in.  So
the buffers of one call -- inputs, outputs, workspace, host arrays -- are carved here out of one larger allocation per
memory space, each with a guard of GUARD bytes before and after it, and everything except the input payloads is filled
with a poison.  `check_call` runs the call once per poison and alignment and requires

  * guards and input payloads bit-identical to what they held before the call (nothing written outside the outputs);
  * every exact output bit-identical across all poisons and alignments (no missed write, no read of unwritten workspace,
    no dependence on bytes past the end of an input: an input's trailing guard changes from run to run too).

Buffers a kernel accumulates into (`acc`) are not poisoned: they hold the caller's base, and the test compares them with
that base.  Alignments: "aligned" puts every payload on a 256-byte boundary, "offset" at the smallest offset the contract
allows for that buffer (its `align`: 4 bytes past a 256-byte boundary for fp32 / int32, 8 for int64, 16 for buffers that
must be 16-byte aligned, 0 for the ones that must be 256-byte aligned).
"""
import numpy as np
import torch

GUARD = 16384                      # two packed 512-ref tiles: a tile-sized overrun lands inside the guard
SLOT = 256
POISONS = ("zeros", "ones", "random")
ALIGNMENTS = ("aligned", "offset")


class Buf:
    def __init__(self, name, kind, dtype, shape, data=None, align=None, space="device", exact=True):
        self.name, self.kind, self.dtype, self.shape = name, kind, dtype, tuple(int(s) for s in shape)
        self.data, self.space, self.exact = data, space, exact
        self.itemsize = torch.empty((), dtype=dtype).element_size()
        self.nbytes = int(np.prod(self.shape, dtype=np.int64)) * self.itemsize
        self.align = self.itemsize if align is None else int(align)
        assert self.nbytes > 0, name
        assert SLOT % self.align == 0 or self.align == SLOT, (name, self.align)


def _torch_dtype(a):
    return {np.dtype(np.float32): torch.float32, np.dtype(np.float64): torch.float64, np.dtype(np.int64): torch.int64,
            np.dtype(np.int32): torch.int32, np.dtype(np.uint8): torch.uint8}[np.asarray(a).dtype]


def inp(name, a, align=None, space="device"):
    """an input: its payload is copied in; it must come back unchanged"""
    a = np.ascontiguousarray(a)
    return Buf(name, "in", _torch_dtype(a), a.shape, data=a, align=align, space=space)


def out(name, shape, dtype, align=None, space="device", exact=True):
    """an output: starts poisoned; exact=False for outputs summed by atomics (their bits depend on the order)"""
    return Buf(name, "out", dtype, shape, align=align, space=space, exact=exact)


def acc(name, base, align=None, space="device", exact=False):
    """an output the kernel accumulates into (or a flag it may set): starts as `base`, not poisoned"""
    base = np.ascontiguousarray(base)
    return Buf(name, "acc", _torch_dtype(base), base.shape, data=base, align=align, space=space, exact=exact)


def ws(name, nbytes, align=16, space="device"):
    """scratch: starts poisoned, may be written, is not compared"""
    return Buf(name, "ws", torch.uint8, (max(int(nbytes), 1),), align=align, space=space)


def _alloc(n, space, device):
    if space == "device":
        return torch.empty(n, dtype=torch.uint8, device=device)
    return torch.empty(n, dtype=torch.uint8, pin_memory=(space == "pinned"))


def _poison(kind, n, seed):
    if kind == "zeros":
        return torch.zeros(n, dtype=torch.uint8)
    if kind == "ones":
        return torch.full((n,), 0xFF, dtype=torch.uint8)
    assert kind == "random", kind
    return torch.from_numpy(np.random.default_rng(seed).integers(0, 256, n, dtype=np.uint8))


class Layout:
    """one carve of `bufs` (one allocation per memory space) for one poison and alignment"""

    def __init__(self, bufs, device, poison, alignment, seed):
        self.bufs, self.device = bufs, device
        self.arenas, self.init, self.place, self.views = {}, {}, {}, {}
        for space in dict.fromkeys(b.space for b in bufs):
            mine = [b for b in bufs if b.space == space]
            total = sum(GUARD + 2 * SLOT + b.nbytes for b in mine) + GUARD + SLOT
            arena = _alloc(total, space, device)
            base = arena.data_ptr()
            cur = 0
            for b in mine:
                want = 0 if alignment == "aligned" else b.align % SLOT
                start = cur + GUARD
                start += (want - (base + start)) % SLOT
                self.place[b.name] = (space, start)
                cur = start + b.nbytes
            assert cur + GUARD <= total
            arena.copy_(_poison(poison, total, seed + 7919 * len(self.arenas)))
            for b in mine:
                _, s = self.place[b.name]
                v = arena[s:s + b.nbytes].view(b.dtype).view(b.shape)
                if b.data is not None:
                    v.copy_(torch.from_numpy(b.data))
                self.views[b.name] = v
            self.arenas[space] = arena
            self.init[space] = arena.clone()

    def ptr(self, name):
        return self.views[name].data_ptr()

    def check_untouched(self):
        """guards, padding and input payloads must hold exactly what they held before the call"""
        for space, arena in self.arenas.items():
            changed = arena != self.init[space]
            for b in self.bufs:
                sp, s = self.place[b.name]
                if sp == space and b.kind != "in":
                    changed[s:s + b.nbytes] = False
            if bool(changed.any()):
                first = int(torch.nonzero(changed)[0])
                n = int(changed.sum())
                raise AssertionError("%d byte(s) outside the outputs changed (%s space); the first one %s"
                                     % (n, space, self._where(space, first)))

    def _where(self, space, off):
        for b in self.bufs:
            sp, s = self.place[b.name]
            if sp != space:
                continue
            if s <= off < s + b.nbytes:
                return "inside input %r at byte %d" % (b.name, off - s)
            if s + b.nbytes <= off < s + b.nbytes + GUARD:
                return "in the guard after %r, %d byte(s) past its end" % (b.name, off - s - b.nbytes)
            if s - GUARD <= off < s:
                return "in the guard before %r, %d byte(s) before its start" % (b.name, s - off)
        return "at arena byte %d" % off

    def results(self):
        return {b.name: self.views[b.name].cpu().numpy().copy() for b in self.bufs if b.kind in ("out", "acc")}


def _sync(device):
    if torch.device(device).type == "cuda" or torch.cuda.is_initialized():
        torch.cuda.synchronize()


def check_call(bufs, call, device, poisons=POISONS, alignments=ALIGNMENTS, seed=0):
    """Run `call(layout)` once per poison and alignment.  Checks guards, inputs and poison invariance of the exact
    outputs; returns the outputs of the first run ({name: numpy array}) for the caller's oracle comparison, and the
    list of every run's outputs (for the outputs that are not exact)."""
    first, runs = None, []
    for ai, alignment in enumerate(alignments):
        for pi, poison in enumerate(poisons):
            lay = Layout(bufs, device, poison, alignment, seed + 1000 * ai + 100 * pi)
            for b in bufs:
                if alignment == "aligned" or b.align >= SLOT:
                    assert lay.ptr(b.name) % SLOT == 0, b.name
                else:
                    assert lay.ptr(b.name) % SLOT == b.align, b.name
            _sync(device)
            call(lay)
            _sync(device)
            try:
                lay.check_untouched()
            except AssertionError as e:
                raise AssertionError("poison %s, %s buffers: %s" % (poison, alignment, e)) from None
            res = lay.results()
            runs.append(res)
            if first is None:
                first, first_tag = res, (poison, alignment)
                continue
            for b in bufs:
                if b.kind in ("out", "acc") and b.exact:
                    got, want = res[b.name].view(np.uint8), first[b.name].view(np.uint8)
                    if not np.array_equal(got, want):
                        i = int(np.flatnonzero(got.reshape(-1) != want.reshape(-1))[0]) // b.itemsize
                        raise AssertionError("output %r differs between poison %s / %s buffers and poison %s / %s buffers, "
                                             "first at element %d (flat): a missed write or a read of unwritten memory"
                                             % ((b.name,) + first_tag + (poison, alignment, i)))
    return first, runs

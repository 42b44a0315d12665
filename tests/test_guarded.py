"""The guarded-buffer harness (tests/guarded.py) on CPU tensors: it must catch a missed write, a write into a guard, a read
of workspace before it is written and a write into an input -- a harness that checks nothing would pass every GPU case."""
import ctypes

import numpy as np
import pytest
import torch

import guarded as G

N = 1000


def _bufs():
    x = np.random.default_rng(0).normal(size=N).astype(np.float32)
    return x, [G.inp("x", x), G.out("y", (N,), torch.float32), G.out("i", (N,), torch.int64), G.ws("ws", 4 * N)]


def _correct(lay):
    x, y, i, w = (lay.views[n] for n in ("x", "y", "i", "ws"))
    w.view(torch.float32).copy_(x * 2)                       # scratch written before it is read
    y.copy_(w.view(torch.float32) + 1)
    i.copy_(torch.arange(N))


def test_a_correct_op_passes_and_buffers_sit_where_the_contract_allows():
    x, bufs = _bufs()
    seen = []

    def call(lay):
        seen.append({n: lay.ptr(n) % G.SLOT for n in ("x", "y", "i", "ws")})
        _correct(lay)

    first, runs = G.check_call(bufs, call, "cpu")
    assert len(runs) == len(G.POISONS) * len(G.ALIGNMENTS) == 6
    np.testing.assert_array_equal(first["y"], x * 2 + 1)
    assert seen[0] == {"x": 0, "y": 0, "i": 0, "ws": 0}
    assert seen[-1] == {"x": 4, "y": 4, "i": 8, "ws": 16}       # the smallest offsets: fp32, int64, 16-byte scratch


def test_poisons_are_zeros_ones_and_random_and_guards_are_large():
    assert G.GUARD >= 16384
    lays = [G.Layout(_bufs()[1], "cpu", p, "aligned", 5) for p in G.POISONS]
    y = [lay.views["y"].view(torch.uint8) for lay in lays]
    assert (y[0] == 0).all() and (y[1] == 0xFF).all()
    assert 200 < len(torch.unique(y[2])) and not (y[2] == 0).all()


def _unwrite_last(lay, name):
    """put the poison back into the last element of output `name`: the op "did not write" it"""
    v = lay.views[name].view(torch.uint8)
    _, s = lay.place[name]
    n = v.numel()
    v[-lay.views[name].element_size():] = lay.init["device"][s + n - lay.views[name].element_size():s + n]


def test_catches_a_missed_write():
    _, bufs = _bufs()

    def call(lay):
        _correct(lay)
        _unwrite_last(lay, "y")

    with pytest.raises(AssertionError, match="'y' differs .* missed write"):
        G.check_call(bufs, call, "cpu")


def test_catches_a_missed_write_that_one_poison_hides():
    """-1 is the right answer in the last slot and 0xFF is its poison: only the other poisons expose the missed write"""
    _, bufs = _bufs()

    def call(lay):
        _correct(lay)
        _unwrite_last(lay, "i")

    with pytest.raises(AssertionError, match="'i' differs"):
        G.check_call(bufs, call, "cpu", poisons=("ones", "zeros"))
    with pytest.raises(AssertionError, match="'i' differs"):
        G.check_call(bufs, call, "cpu", poisons=("ones", "random"))


def test_catches_one_element_written_into_the_trailing_guard():
    _, bufs = _bufs()

    def call(lay):
        _correct(lay)
        y = lay.views["y"]
        one = ctypes.c_float(1.0)
        ctypes.memmove(y.data_ptr() + y.nbytes, ctypes.byref(one), 4)     # y[N]: one past the end

    with pytest.raises(AssertionError, match="in the guard after 'y', [0-3] byte"):
        G.check_call(bufs, call, "cpu")


def test_catches_one_element_written_before_the_start():
    _, bufs = _bufs()

    def call(lay):
        _correct(lay)
        ctypes.memmove(lay.ptr("ws") - 16, ctypes.byref(ctypes.c_int64(3)), 8)

    with pytest.raises(AssertionError, match="in the guard before 'ws', 16 byte"):
        G.check_call(bufs, call, "cpu")


def test_catches_a_workspace_element_read_before_it_is_written():
    _, bufs = _bufs()

    def call(lay):
        x, y, i, w = (lay.views[n] for n in ("x", "y", "i", "ws"))
        wf = w.view(torch.float32)
        stale = wf[7].clone()                                 # read first ...
        wf.copy_(x * 2)                                       # ... then written
        y.copy_(wf + 1)
        y[7] = stale
        i.copy_(torch.arange(N))

    with pytest.raises(AssertionError, match="'y' differs .* element 7"):
        G.check_call(bufs, call, "cpu")


def test_catches_a_write_into_an_input_and_a_read_past_its_end():
    _, bufs = _bufs()

    def writes_input(lay):
        _correct(lay)
        lay.views["x"][3] = 0.5

    with pytest.raises(AssertionError, match="inside input 'x' at byte 12"):
        G.check_call(bufs, writes_input, "cpu")

    def reads_past_end(lay):                                  # a 16-byte load over the last 4-byte element
        _correct(lay)
        past = (ctypes.c_float * 1).from_address(lay.ptr("x") + 4 * N)[0]
        lay.views["y"][-1] = past

    with pytest.raises(AssertionError, match="'y' differs"):
        G.check_call(bufs, reads_past_end, "cpu")


def test_accumulated_outputs_keep_their_base():
    base = np.random.default_rng(1).normal(size=(50, 3)).astype(np.float32)
    bufs = [G.acc("g", base), G.inp("rows", np.array([4, 9], np.int64))]

    def call(lay):
        lay.views["g"][lay.views["rows"]] += 1.0

    first, _ = G.check_call(bufs, call, "cpu")
    want = base.copy(); want[[4, 9]] += 1.0
    np.testing.assert_array_equal(first["g"], want)

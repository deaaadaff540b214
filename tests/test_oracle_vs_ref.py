"""The restatement against runs of the unmodified reference (oracle/_ref/ref_mcmc under the GSL-API shim), replayed from
the traces tools/make_golden.py recorded into tests/golden/ref_*.npz: the draw tape, the reference's seed and the full
model state after the randomised start and after every mcmc_sample() call (or every sub-sampler call in step mode)."""
import os

import numpy as np
import pytest

from conftest import GOLDEN, load_hex_dataset

KEYS = ("a", "b", "pi", "rpi", "t0", "f0", "t1", "f1", "tot")


@pytest.fixture(scope="module")
def O(oracle_mod):
    return oracle_mod


def _reference_trace(O, name):
    """(X, hard, states, tape, seed) of the reference's recorded run ``tests/golden/<name>.npz``"""
    g = np.load(os.path.join(GOLDEN, name + ".npz"))
    X, hard = load_hex_dataset(name.split("_")[1])
    states = [O.State(int(g["kind"][r]), int(g["ret"][r]), int(g["slots"][r]), *(g[k][r].astype(np.int32) for k in KEYS),
                      *(float(v) for v in g["cdl"][r])) for r in range(len(g["kind"]))]
    return X, hard, states, g["tape"], int(g["meta"][2])


@pytest.mark.parametrize("name,calls", [("g10s10", 12), ("g10s2", 2), ("g5s5", 3), ("g2s2", 2)])
def test_restatement_bit_exact_vs_live_reference(O, name, calls):
    X, hard, states, tape, _ = _reference_trace(O, "ref_" + name)
    assert len(states) > calls
    o = O.Oracle(X, hard).source_tape(tape)
    o.randomize()
    assert o.state().same_bits(states[0])
    for r in range(1, calls + 1):
        o.sample()
        s = o.state()
        assert s.same_bits(states[r]) and s.slots == states[r].slots, r
    assert o.tape_mismatches == 0


def test_restatement_mt_stream_equals_shim_mt_stream(O):
    """Same MT19937 seed -> the restatement's own generator reproduces the shim's tape."""
    X, hard, states, tape, seed = _reference_trace(O, "ref_g10s10")
    o = O.Oracle(X, hard).source_mt(seed).record(True)
    o.randomize()
    for r in range(1, 5):
        o.sample()
        assert o.state().same_bits(states[r])
    assert np.array_equal(o.tape(), tape[:states[4].slots])


def test_reference_step_trace(O):
    X, hard, states, tape, _ = _reference_trace(O, "ref_g10s10_step")
    assert int(np.load(os.path.join(GOLDEN, "ref_g10s10_step.npz"))["meta"][3]) == 1   # recorded in step mode
    o = O.Oracle(X, hard).source_tape(tape)
    o.randomize()
    step = {10: o.samplec, 11: o.sampled, 12: o.sampleab, 13: lambda: o.samplepi2(1), 14: o.samplepi1,
            15: lambda: o.samplepi2(0), 16: o.samplepi3}
    for r in range(1, len(states)):
        if states[r].kind == 1:
            continue
        assert step[states[r].kind]() == states[r].ret
        assert o.state().same_bits(states[r]), r

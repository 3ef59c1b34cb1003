"""Long-form overlap-add with context margins (voicefixer_main_b200/longform.py) - host logic, CPU only.

The mirror is checked (a) against the reference's own LambdaOverlapAdd (tools/dsp/overlapadd_boxcar.py:338-534):
tests/golden/reference_longform.npz holds every second sample of what that class, imported unmodified, returned for
the toy network and signals below (python oracle/make_golden.py longform), and (b) through properties that need no
reference: the batched schedule equals the sequential one, and with a margin at least as long as the network's
receptive field the chunking is invisible."""
import types

import pytest
import torch
import torch.nn.functional as F

from conftest import load_golden
from voicefixer_main_b200.longform import BoxcarOverlapAdd, WindowedOverlapAdd

CASES = [(1000, 256, 32), (1024, 256, 32), (200, 256, 32), (256, 256, 64), (513, 256, 255), (2049, 512, 100)]


class ToyNet(torch.nn.Module):
    """Deterministic non-linear FIR network with the nnet protocol: [B, C, L] -> {"wav": [B, 1, L]}."""

    def __init__(self, taps=9, batch_invariant=False):
        super().__init__()
        g = torch.Generator().manual_seed(5)
        self.k = torch.randn(1, 1, taps, generator=g) * 0.3
        self.batch_invariant = batch_invariant
        # the reference constructor reads nnet.f_helper.stft.conv_real.weight for its dtype (:411)
        self.f_helper = types.SimpleNamespace(stft=types.SimpleNamespace(conv_real=types.SimpleNamespace(weight=torch.zeros(1))))
        self.calls = []

    def forward(self, x):
        self.calls.append(tuple(x.shape))
        y = F.conv1d(x[:, :1, :], self.k, padding=self.k.shape[-1] // 2)
        return {"wav": torch.tanh(y) + 0.1 * y}


def _signal(n, batch=2):
    g = torch.Generator().manual_seed(n)
    return torch.randn(batch, 1, n, generator=g)


def boxcar_key(n, w, m, windowed):
    return f"boxcar_{n}_{w}_{m}_{int(windowed)}"


def ola_key(n, w, hop, windowed):
    return f"ola_{n}_{w}_{hop}_{int(windowed)}"


@pytest.fixture(scope="module")
def reference():
    return load_golden("reference_longform.npz")


@pytest.mark.parametrize("n,w,m", CASES)
@pytest.mark.parametrize("windowed", [False, True])
def test_matches_reference_lambda_overlap_add(n, w, m, windowed, reference):
    # the reference ran with window="hann" (its constructor fails on None, :411) and use_window = windowed, which
    # selects the boxcar path the way its own ola_forward does
    our_net = ToyNet()
    ours = BoxcarOverlapAdd(our_net, n_src=1, window_size=w, in_margin=m, window="hann" if windowed else None)
    b = ours(_signal(n))
    assert b.shape == (2, 1, n)
    assert torch.equal(torch.from_numpy(reference[boxcar_key(n, w, m, windowed)]), b.reshape(-1)[::int(reference["stride"])])
    calls = [tuple(c) for c in reference[boxcar_key(n, w, m, windowed) + "_calls"].tolist()]
    assert calls == sorted(our_net.calls)                          # same chunks reach the network


@pytest.mark.parametrize("n,w,m", CASES)
def test_batched_schedule_equals_sequential(n, w, m):
    x = _signal(n, batch=3)
    seq, bat = ToyNet(batch_invariant=False), ToyNet(batch_invariant=True)
    a = BoxcarOverlapAdd(seq, 1, w, m)(x)
    b = BoxcarOverlapAdd(bat, 1, w, m, max_batch=None)(x)
    assert torch.allclose(a, b, atol=1e-6)
    n_chunks = -(-n // w)
    assert len(seq.calls) == n_chunks
    assert len(bat.calls) == min(n_chunks, 3)                      # first, last, one stacked call for the middle
    if n_chunks > 3:
        assert bat.calls[0][0] == 3 * (n_chunks - 2)


@pytest.mark.parametrize("n,w,m", CASES)
def test_margin_hides_the_chunking(n, w, m):
    net = ToyNet(taps=9)                                           # receptive field 4 <= every margin above
    x = _signal(n, batch=1)
    whole = net(x)["wav"]
    chunked = BoxcarOverlapAdd(ToyNet(taps=9), 1, w, m)(x)
    assert torch.allclose(whole, chunked, atol=1e-6)


def test_plan_and_argument_checks():
    ola = BoxcarOverlapAdd(ToyNet(), 1, 256, 32)
    chunks, last = ola.plan(1000)
    assert last == 1000 - 3 * 256
    assert chunks == [(0, 288, 0, 32), (224, 544, 32, 32), (480, 800, 32, 32), (736, 1000, 32, 0)]
    assert ola.plan(512)[0] == [(0, 288, 0, 32), (224, 512, 32, 0)]
    with pytest.raises(AssertionError):
        BoxcarOverlapAdd(ToyNet(), 1, 255, 32)
    with pytest.raises(ValueError):
        BoxcarOverlapAdd(ToyNet(), 1, 256, 256)
    with pytest.raises(NotImplementedError):
        BoxcarOverlapAdd(ToyNet(), 2, 256, 32, reorder_chunks=True)


# ------------------------------------------------------------------ windowed overlap-add (tools/dsp/overlapadd.py)
OLA_CASES = [(1000, 256, None), (1024, 256, 128), (300, 256, 64), (2049, 512, 256), (777, 128, 32)]


@pytest.mark.parametrize("n,w,hop", OLA_CASES)
@pytest.mark.parametrize("windowed", [True, False])
def test_windowed_ola_matches_reference(n, w, hop, windowed, reference):
    # the reference (tools/dsp/overlapadd.py) ran with window="hann" and use_window = windowed
    our_net = ToyNet()
    ours = WindowedOverlapAdd(our_net, n_src=1, window_size=w, hop_size=hop, window="hann" if windowed else None,
                              reorder_chunks=False)
    b = ours(_signal(n))
    assert b.shape == (2, 1, n)
    assert torch.equal(torch.from_numpy(reference[ola_key(n, w, hop, windowed)]), b.reshape(-1)[::int(reference["stride"])])
    assert [tuple(c) for c in reference[ola_key(n, w, hop, windowed) + "_calls"].tolist()] == our_net.calls


@pytest.mark.parametrize("n,w,hop", OLA_CASES)
def test_windowed_ola_batched_equals_sequential_and_cola(n, w, hop):
    x = _signal(n, batch=2)
    seq, bat = ToyNet(batch_invariant=False), ToyNet(batch_invariant=True)
    a = WindowedOverlapAdd(seq, 1, w, hop, window="hanning", reorder_chunks=False)(x)
    b = WindowedOverlapAdd(bat, 1, w, hop, window="hanning", reorder_chunks=False, max_batch=None)(x)
    assert torch.allclose(a, b, atol=1e-6)
    assert len(bat.calls) == 1 and bat.calls[0][0] == 2 * len(seq.calls)   # the whole file in one call

    class Identity:
        batch_invariant = True

        def __call__(self, t):
            return {"wav": t[:, :1, :]}

    if hop is None or 2 * hop == w:                 # periodic hann at 50 % overlap sums to one: identity in, identity out
        y = WindowedOverlapAdd(Identity(), 1, w, hop, window="hann", reorder_chunks=False)(x)
        assert torch.allclose(y, x, atol=1e-6)


def test_max_batch_bounds_the_rows_per_call():
    """ADVICE r1: the stacked schedules run `max_batch` rows per nnet call (workspace grows with batch x length), with
    results identical to the unbounded stack; an n_src > 1 network with reorder_chunks is refused, not silently skipped."""
    x = _signal(20 * 256 + 17, batch=2)
    full, capped = ToyNet(batch_invariant=True), ToyNet(batch_invariant=True)
    a = BoxcarOverlapAdd(full, 1, 256, 32, max_batch=None)(x)
    b = BoxcarOverlapAdd(capped, 1, 256, 32, max_batch=6)(x)
    assert torch.equal(a, b)
    assert max(c[0] for c in capped.calls) <= 6 and max(c[0] for c in full.calls) == 2 * 19
    fullw, cappedw = ToyNet(batch_invariant=True), ToyNet(batch_invariant=True)
    aw = WindowedOverlapAdd(fullw, 1, 256, 128, reorder_chunks=False, max_batch=None)(x)
    bw = WindowedOverlapAdd(cappedw, 1, 256, 128, reorder_chunks=False, max_batch=8)(x)
    assert torch.equal(aw, bw)
    assert max(c[0] for c in cappedw.calls) <= 8 and len(fullw.calls) == 1

    class TwoSrc:
        batch_invariant = True

        def __call__(self, t):
            return {"wav": torch.cat([t, t], dim=1)}

    with pytest.raises(NotImplementedError):
        WindowedOverlapAdd(TwoSrc(), None, 256, 128)(x)                       # reorder_chunks defaults to True
    with pytest.raises(NotImplementedError):
        BoxcarOverlapAdd(TwoSrc(), None, 256, 32, reorder_chunks=True)(x)

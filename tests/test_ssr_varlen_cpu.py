"""Host logic of the SSR / GSR-UNet varlen entry points with stub engines (no GPU): SSR_UNet.restore_many's sorting,
grouping and re-ordering, and the SSR branch of handler.restore_files - 60 s segmentation, per-segment peak
normalisation and reassembly - against a per-file loop of the reference's GSR-UNet handler."""
import numpy as np
import pytest
import torch

from voicefixer_main_b200 import GSR_UNet, SSR_UNet
from voicefixer_main_b200 import handler as H
from voicefixer_main_b200.model import group_sizes

GAIN = 3.0      # the stub's "restoration": large enough that some segments need the peak normalisation


class StubSSREngine:
    """ssr_restore_varlen of a stub: row b -> GAIN * row b on its first lengths[b] samples, zeros after (the C ABI's
    contract); finalize and to_pcm16 as the library defines them."""
    device = torch.device("cpu")
    loaded = True

    def __init__(self):
        self.calls = []
        self.finalized = []

    def ssr_restore_varlen(self, wav, lengths, out=None):
        lens = list(lengths)
        assert wav.dim() == 2 and wav.shape[0] == len(lens) and max(lens) == wav.shape[1]
        self.calls.append(tuple(lens))
        out = torch.zeros_like(wav)
        for b, n in enumerate(lens):
            out[b, :n] = wav[b, :n] * GAIN
        return out

    def finalize(self, wav, n):
        assert wav.dim() == 2 and wav.shape[1] == n          # the ISTFT returns the input length: nothing to trim
        self.finalized.append(n)
        peak = wav.abs().amax(dim=1, keepdim=True)
        return torch.where(peak > 1.0, wav / peak, wav)

    def to_pcm16(self, x, saturate=False):
        v = x.double() * 32768.0
        if saturate:
            v = v.clamp(-32768, 32767)
        return torch.from_numpy((np.trunc(v.numpy()).astype(np.int64) & 0xFFFF).astype(np.uint16).view(np.int16))


def stub_model(cls=SSR_UNet):
    m = cls()
    m._eng = StubSSREngine()
    m.device = torch.device("cpu")
    m.restore = lambda x: x * GAIN                     # SSR_UNet.restore of one segment
    return m


def test_restore_many_sorts_groups_and_returns_input_order():
    m = stub_model()
    rng = np.random.default_rng(4)
    lengths = [int(x) for x in rng.integers(1100, 9000, size=23)]
    clips = [torch.from_numpy(rng.standard_normal(n).astype(np.float32)) for n in lengths]
    res = m.restore_many(clips, max_batch=6)
    assert len(res) == len(clips)
    for c, r in zip(clips, res):
        assert r.shape == c.shape and torch.equal(r, c * GAIN)     # no peak normalisation, like restore()
    calls = m._eng.calls
    assert [len(lens) for lens in calls] == group_sizes(23, 6) == [6, 6, 6, 5]
    assert [n for lens in calls for n in lens] == sorted(lengths)
    assert not m._eng.finalized
    assert m.restore_many([], max_batch=4) == []
    with pytest.raises(ValueError):
        m.restore_many(clips, max_batch=0)


def test_gsr_unet_inherits_restore_many():
    m = stub_model(GSR_UNet)
    clips = [torch.ones(2000), torch.ones(1500) * 0.25, torch.ones(3000) * -0.5]
    res = m.restore_many(clips, max_batch=2)
    assert [len(lens) for lens in m._eng.calls] == [2, 1]
    for c, r in zip(clips, res):
        assert torch.equal(r, c * GAIN)


def reference_gsr_unet_file(m, path, saturate):
    """eval_gsr_unet.py:43-74 for one file with the stub's restoration: 60 s segments, each peak-normalised when its
    max |x| exceeds 1, concatenated, converted to int16."""
    wav = H.load_wav(path)
    res = []
    for sl in H.split_segments(wav.shape[0]):
        out = m.restore(torch.from_numpy(np.ascontiguousarray(wav[sl]))[None])
        if torch.max(torch.abs(out)) > 1.0:
            out = out / torch.max(torch.abs(out))
        res.append(out)
    return m._eng.to_pcm16(torch.cat(res, -1)[0], saturate=saturate).numpy()


@pytest.mark.parametrize("saturate", [False, True])
def test_restore_files_ssr_segments_normalises_and_reassembles(tmp_path, saturate):
    m = stub_model()
    seg = H.SEG_LENGTH
    lengths = [seg + 5000, 3000, 2 * seg, 2 * seg + 1500]
    # per-file amplitudes: after the stub's gain some segments stay below 1 and some are normalised
    amps = [3000, 12000, 9000, 20000]
    rng = np.random.default_rng(2)
    srcs, outs = [], []
    for k, (n, a) in enumerate(zip(lengths, amps)):
        pcm = (rng.standard_normal(n) * a / 4).clip(-a, a).astype(np.int16)
        srcs.append(str(tmp_path / f"in{k}.wav"))
        outs.append(str(tmp_path / f"out{k}.wav"))
        H.save_pcm16(pcm, srcs[-1])
    H.restore_files(m, srcs, outs, meta={"saturate": saturate, "unify_energy": True}, max_batch=3)
    segs = sorted(sl.stop - sl.start for n in lengths for sl in H.split_segments(n))
    assert sorted(n for lens in m._eng.calls for n in lens) == segs
    assert [len(lens) for lens in m._eng.calls] == group_sizes(len(segs), 3)
    assert sorted(m._eng.finalized) == segs                        # one peak normalisation per segment
    normalised = 0
    for src, out in zip(srcs, outs):
        want = reference_gsr_unet_file(m, src, saturate)
        ref = str(tmp_path / "ref.wav")
        H.save_pcm16(want, ref)
        with open(ref, "rb") as a, open(out, "rb") as b:
            assert a.read() == b.read()
        normalised += int(np.abs(want.astype(np.int32)).max() >= 32767)
    assert 0 < normalised < len(srcs)                               # both branches of the peak test ran
    with pytest.raises(ValueError):
        H.restore_files(m, srcs, outs[:1])

"""Host logic of the varlen entry points with stub engines (no GPU): VoiceFixer.restore_many's sorting, grouping and
re-ordering, and handler.restore_files' 60 s segmentation and reassembly against handler.restore_array."""
import numpy as np
import pytest
import torch

from voicefixer_main_b200 import VoiceFixer
from voicefixer_main_b200 import handler as H
from voicefixer_main_b200.model import group_sizes


class StubEngine:
    """restore_varlen of a stub: row b -> 0.5 * row b on its first lengths[b] samples, zeros after (the C ABI's contract)."""
    device = torch.device("cpu")
    loaded = True

    def __init__(self):
        self.calls = []

    def restore_varlen(self, wav, lengths, out=None, unify_energy=False):
        lens = list(lengths)
        assert wav.dim() == 2 and wav.shape[0] == len(lens) and max(lens) == wav.shape[1]
        self.calls.append((tuple(lens), unify_energy))
        out = torch.zeros_like(wav)
        for b, n in enumerate(lens):
            out[b, :n] = wav[b, :n] * 0.5
        return out

    def to_pcm16(self, x, saturate=False):
        v = x.double() * 32768.0
        if saturate:
            v = v.clamp(-32768, 32767)
        return torch.from_numpy((np.trunc(v.numpy()).astype(np.int64) & 0xFFFF).astype(np.uint16).view(np.int16))


def stub_model():
    m = VoiceFixer()
    m._eng = StubEngine()
    m.device = torch.device("cpu")
    m.restore = lambda x, unify_energy=False: x * 0.5          # restore_array's per-segment call
    return m


@pytest.mark.parametrize("n,max_batch", [(1, 32), (32, 32), (33, 32), (65, 32), (256, 32), (7, 3), (10, 1)])
def test_group_sizes_are_near_equal_and_bounded(n, max_batch):
    g = group_sizes(n, max_batch)
    assert sum(g) == n and max(g) <= max_batch and max(g) - min(g) <= 1
    assert len(g) == -(-n // max_batch)


def test_restore_many_sorts_groups_and_returns_input_order():
    m = stub_model()
    rng = np.random.default_rng(3)
    lengths = [int(x) for x in rng.integers(1100, 9000, size=37)]
    clips = [torch.from_numpy(rng.standard_normal(n).astype(np.float32)) for n in lengths]
    res = m.restore_many(clips, unify_energy=True, max_batch=8)
    assert len(res) == len(clips)
    for c, r in zip(clips, res):
        assert r.shape == c.shape and torch.equal(r, c * 0.5)
    calls = m._eng.calls
    assert [len(lens) for lens, _ in calls] == group_sizes(37, 8) == [8, 8, 7, 7, 7]
    flat = [n for lens, _ in calls for n in lens]
    assert flat == sorted(lengths)                                 # neighbours in length share a group
    assert all(u for _, u in calls)
    assert m.restore_many([], max_batch=4) == []
    with pytest.raises(ValueError):
        m.restore_many(clips, max_batch=0)


def test_restore_files_segments_and_reassembles_like_restore_array(tmp_path):
    m = stub_model()
    seg = H.SEG_LENGTH
    lengths = [seg + 5000, 3000, 2 * seg, 2 * seg + 1500]
    rng = np.random.default_rng(1)
    srcs, outs = [], []
    for k, n in enumerate(lengths):
        pcm = (rng.standard_normal(n) * 6000).clip(-32000, 32000).astype(np.int16)
        srcs.append(str(tmp_path / f"in{k}.wav"))
        outs.append(str(tmp_path / f"out{k}.wav"))
        H.save_pcm16(pcm, srcs[-1])
    H.restore_files(m, srcs, outs, meta={"saturate": True}, max_batch=3)
    segs = sorted(sl.stop - sl.start for n in lengths for sl in H.split_segments(n))
    assert sorted(n for lens, _ in m._eng.calls for n in lens) == segs
    assert [len(lens) for lens, _ in m._eng.calls] == group_sizes(len(segs), 3)
    for src, out in zip(srcs, outs):
        want = H.restore_array(m, H.load_wav(src), "cpu")
        ref = str(tmp_path / "ref.wav")
        H.save_pcm16(m._eng.to_pcm16(want[0], saturate=True).numpy(), ref)
        with open(ref, "rb") as a, open(out, "rb") as b:
            assert a.read() == b.read()
    with pytest.raises(ValueError):
        H.restore_files(m, srcs, outs[:1])

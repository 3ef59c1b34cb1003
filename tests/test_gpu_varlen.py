"""Clips of different lengths in one batched call (vf_restore_varlen / Engine.restore_varlen / VoiceFixer.restore_many /
handler.restore_files).  Every row must carry exactly the bits restore() gives that clip alone, and every sample past a
clip's length must be exactly 0."""
import numpy as np
import pytest
import torch

from oracle import vf_oracle as O

pytestmark = pytest.mark.gpu

HOP = 441


def n_for_frames(t, extra=0):
    """A sample count with 1 + n // 441 == t."""
    return (t - 1) * HOP + extra


# 1025 samples (3 frames); T = 128 (a multiple of 64) and T = 129 = 2 * 64 + 1 (a bucket edge), i.e. an even and an odd T
# (their vocoder lengths differ by the T % 2 term); an odd T = 77; 3 s; two 10 s clips one sample apart
LENGTHS = [1025, n_for_frames(128, 17), n_for_frames(129, 5), n_for_frames(77, 300), 3 * 44100, 441000, 440999]


@pytest.fixture(scope="module")
def model(state):
    from voicefixer_main_b200 import VoiceFixer
    m = VoiceFixer().load_state_dict(state).eval().to("cuda:0")
    yield m
    m._engine().check_errors()


def make_clips(lengths, seed):
    base = O.synth_clips(len(lengths), max(lengths), seed=seed)
    return [base[i, :n].clone() for i, n in enumerate(lengths)]


def padded(clips):
    n_max = max(c.shape[0] for c in clips)
    x = torch.full((len(clips), n_max), 0.25)             # the padding is never read: fill it with something non-zero
    for i, c in enumerate(clips):
        x[i, :c.shape[0]] = c
    return x.cuda()


def alone(model, clips, unify):
    return [model.restore(c[None].cuda(), unify_energy=unify)[0].cpu() for c in clips]


def check_rows(out, clips, refs):
    out = out.cpu()
    for i, (c, r) in enumerate(zip(clips, refs)):
        n = c.shape[0]
        assert torch.equal(out[i, :n], r), f"clip {i} ({n} samples): max diff {float((out[i, :n] - r).abs().max()):.3e}"
        assert bool((out[i, n:] == 0).all()), f"clip {i}: samples past its length are not 0"


def identity_check(m, clips, unify_flags=(False, True)):
    eng = m._engine()
    x = padded(clips)
    lens = [c.shape[0] for c in clips]
    for unify in unify_flags:
        refs = alone(m, clips, unify)
        for _ in range(3):                                # eager, graph capture, graph replay
            out = eng.restore_varlen(x, lens, unify_energy=unify)
            check_rows(out, clips, refs)
    eng.check_errors()


def test_varlen_rows_are_bit_identical_to_single_clips(model):
    identity_check(model, make_clips(LENGTHS, seed=5))


def test_varlen_stale_rows_and_graph_replay(model):
    """Length sets from longest to shortest through ONE plan (the longest clip always in the 1024-frame bucket): nothing an
    earlier call left in a slot reaches a later result, across eager run, capture and replays; no plan is added."""
    eng = model._engine()
    sets = [[441000, 300007, 200003], [436000, 99991, 5003], [430001, 2049, 1500], [424000, 60001, 1025]]
    clips = [make_clips(s, seed=20 + k) for k, s in enumerate(sets)]
    refs = [alone(model, c, False) for c in clips]
    outs, plans = [], []
    for c in clips:
        outs.append(eng.restore_varlen(padded(c), [x.shape[0] for x in c]).cpu())
        plans.append(eng.plan_cache_info())
    for c, r, o in zip(clips, refs, outs):
        check_rows(o, c, r)
    print("varlen plan cache after each call:", plans)
    assert all(p["plans"] == plans[0]["plans"] and p["evicted"] == plans[0]["evicted"] for p in plans)
    eng.check_errors()


def test_varlen_with_equal_lengths_equals_restore(model):
    x = O.synth_clips(4, 3 * 44100, seed=9).cuda()
    for unify in (False, True):
        ref = model.restore(x, unify_energy=unify).clone()
        assert torch.equal(model._engine().restore_varlen(x, [x.shape[1]] * 4, unify_energy=unify), ref)


def test_varlen_three_term_vocoder(state):
    from voicefixer_main_b200 import VoiceFixer
    m = VoiceFixer().load_state_dict(state).eval().to("cuda:0")
    m._engine().set_option("vocoder_terms", 3)
    identity_check(m, make_clips(LENGTHS[:5], seed=6), unify_flags=(False,))
    m._engine().close()


def test_varlen_two_launch_residual_pairs(state, monkeypatch):
    from voicefixer_main_b200 import VoiceFixer
    monkeypatch.setenv("VF_TUNE_FUSED_PAIR", "0")
    m = VoiceFixer().load_state_dict(state).eval().to("cuda:0")
    identity_check(m, make_clips(LENGTHS, seed=7), unify_flags=(True,))
    m._engine().close()


def test_varlen_sub_batches_under_a_small_plan_budget(state):
    from voicefixer_main_b200 import VoiceFixer
    m = VoiceFixer().load_state_dict(state).eval().to("cuda:0")
    eng = m._engine()
    clips = make_clips(LENGTHS, seed=8)
    refs = alone(m, clips, False)
    eng.set_option("plan_cache_mb", 4096)                 # a 1024-frame bucket needs ~1.6 GB per clip: sub-batches of 2
    out = eng.restore_varlen(padded(clips), [c.shape[0] for c in clips])
    check_rows(out, clips, refs)
    info = eng.plan_cache_info()
    print("varlen sub-batching:", info)
    assert info["bytes"] <= 4096 << 20
    eng.check_errors()
    eng.close()


def test_restore_many_matches_restore(model):
    lengths = [44100 * 2 + 7, 1100, 44100 * 5, 30000, 30001, 44100 * 2 + 6, 9999]
    clips = make_clips(lengths, seed=11)
    res = model.restore_many(clips, max_batch=3)          # groups of 3, 2, 2
    assert len(res) == len(clips)
    for c, r in zip(clips, res):
        assert r.shape == c.shape
        assert torch.equal(r.cpu(), model.restore(c[None].cuda())[0].cpu())


def test_varlen_bad_lengths_raise_before_any_launch(model):
    import ctypes
    from voicefixer_main_b200 import _lib as L
    eng = model._engine()
    x = O.synth_clips(3, 5000, seed=2).cuda()
    n0 = eng.launch_count()
    for lens in ([1024, 5000, 5000], [5000, 5001, 4000], [5000, 4000], [5000, 4000, 3000, 2000]):
        with pytest.raises(ValueError):
            eng.restore_varlen(x, lens)
    out = torch.empty_like(x)
    for lens in ([5000, 1024, 2000], [5000, 5001, 2000], [0, 5000, 2000]):
        arr = (ctypes.c_int64 * 3)(*lens)
        rc = eng.lib.vf_restore_varlen(eng.ctx, ctypes.c_void_p(x.data_ptr()), 3, 5000, arr, ctypes.c_void_p(out.data_ptr()),
                                       0, ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
        assert rc == L.VF_EINVAL and b"1024 < n" in eng.lib.vf_last_error(eng.ctx)
    assert eng.launch_count() == n0


def test_restore_files_byte_identical_to_handler(model, tmp_path, monkeypatch):
    """16 kHz and 44.1 kHz files, one longer than 60 s (two segments): each output file of restore_files has the bytes
    handler() writes for that file alone."""
    from voicefixer_main_b200 import handler as H
    monkeypatch.setattr(H, "model", model)
    specs = [(44100, 44100 * 61 + 1234, 31), (16000, 16000 * 3 + 77, 32), (44100, 44100 * 7 + 5, 33)]
    srcs = []
    for k, (rate, n, seed) in enumerate(specs):
        pcm = O.to_int16(O.synth_clips(1, n, seed=seed)[0].clamp(-0.99, 0.99).numpy())
        p = str(tmp_path / f"in{k}.wav")
        H.save_pcm16(pcm, p, sample_rate=rate)
        srcs.append(p)
    meta = {"unify_energy": True, "saturate": True}
    outs = [str(tmp_path / f"many{k}.wav") for k in range(len(srcs))]
    H.restore_files(model, srcs, outs, meta=meta, max_batch=2)
    for k, src in enumerate(srcs):
        one = str(tmp_path / f"one{k}.wav")
        H.handler(src, one, None, ckpt=None, device=model.device, needrefresh=False, meta=meta)
        with open(one, "rb") as a, open(outs[k], "rb") as b:
            assert a.read() == b.read(), f"file {k}"
    model._engine().check_errors()

"""SSR / GSR-UNet clips of different lengths in one batched call (vf_ssr_restore_varlen / Engine.ssr_restore_varlen /
SSR_UNet.restore_many / handler.restore_files with an SSR model).  Every row must carry exactly the bits
SSR_UNet.restore gives that clip alone, and every sample past a clip's length must be exactly 0."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import vf_oracle as O

pytestmark = pytest.mark.gpu

HOP = 441


def n_for_frames(t, extra=0):
    """A sample count with 1 + n // 441 == t."""
    return (t - 1) * HOP + extra


# 1025 samples (3 frames); T = 128 (a multiple of 64) and T = 129 (a bucket edge); an odd T = 77; 200 * 441 and
# 200 * 441 - 1 (T = 201 and T = 200: the last frame starts inside the one clip and not in the other); 3 s; two 10 s
# clips one sample apart
LENGTHS = [1025, n_for_frames(128, 17), n_for_frames(129, 5), n_for_frames(77, 300), 200 * HOP, 200 * HOP - 1,
           3 * 44100, 441000, 440999]


@pytest.fixture(scope="module")
def ssr_state():
    from voicefixer_main_b200.weights import make_ssr_state
    return make_ssr_state(1234)


@pytest.fixture(scope="module")
def model(ssr_state):
    from voicefixer_main_b200 import SSR_UNet
    m = SSR_UNet().load_state_dict(ssr_state).eval().to("cuda:0")
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


def alone(model, clips):
    return [model.restore(c[None].cuda())[0].cpu() for c in clips]


def check_rows(out, clips, refs):
    out = out.cpu()
    for i, (c, r) in enumerate(zip(clips, refs)):
        n = c.shape[0]
        assert torch.equal(out[i, :n], r), f"clip {i} ({n} samples): max diff {float((out[i, :n] - r).abs().max()):.3e}"
        assert bool((out[i, n:] == 0).all()), f"clip {i}: samples past its length are not 0"


def test_ssr_varlen_rows_are_bit_identical_to_single_clips(model):
    eng = model._engine()
    clips = make_clips(LENGTHS, seed=5)
    refs = alone(model, clips)
    x = padded(clips)
    lens = [c.shape[0] for c in clips]
    for _ in range(3):                                    # eager, graph capture, graph replay
        check_rows(eng.ssr_restore_varlen(x, lens), clips, refs)
    eng.check_errors()


def test_ssr_varlen_stale_rows_and_graph_replay(model):
    """Length sets from longest to shortest through ONE plan (the longest clip always in the 1024-frame bucket): nothing an
    earlier call left in a slot (sp, the UNet planes, the predicted magnitude, the ISTFT frames) reaches a later result,
    across eager run, capture and replays; no plan is added.  The equal-length path gives the same bits before and after."""
    eng = model._engine()
    eq = O.synth_clips(2, 30000, seed=40).cuda()
    eq_before = model.restore(eq).cpu()
    sets = [[441000, 300007, 200003], [436000, 99991, 5003], [430001, 2049, 1500], [424000, 60001, 1025]]
    clips = [make_clips(s, seed=20 + k) for k, s in enumerate(sets)]
    refs = [alone(model, c) for c in clips]
    outs, plans = [], []
    for c in clips:
        outs.append(eng.ssr_restore_varlen(padded(c), [x.shape[0] for x in c]).cpu())
        plans.append(eng.plan_cache_info())
    for c, r, o in zip(clips, refs, outs):
        check_rows(o, c, r)
    print("ssr varlen plan cache after each call:", plans)
    assert all(p["plans"] == plans[0]["plans"] and p["evicted"] == plans[0]["evicted"] for p in plans)
    assert torch.equal(model.restore(eq).cpu(), eq_before)
    eng.check_errors()


def test_ssr_varlen_with_equal_lengths_equals_restore(model):
    x = O.synth_clips(4, 3 * 44100, seed=9).cuda()
    ref = model.restore(x).clone()
    for _ in range(3):
        assert torch.equal(model._engine().ssr_restore_varlen(x, [x.shape[1]] * 4), ref)


def test_ssr_varlen_sub_batches_under_a_small_plan_budget(ssr_state):
    from voicefixer_main_b200 import SSR_UNet
    m = SSR_UNet().load_state_dict(ssr_state).eval().to("cuda:0")
    eng = m._engine()
    clips = make_clips(LENGTHS[3:], seed=8)               # 6 clips, the longest in the 1024-frame bucket
    refs = alone(m, clips)
    budget_mb = 4800                                      # ~2.2 GB per clip of that bucket: sub-batches of 2
    eng.set_option("plan_cache_mb", budget_mb)
    for _ in range(2):
        out = eng.ssr_restore_varlen(padded(clips), [c.shape[0] for c in clips])
        check_rows(out, clips, refs)
    info = eng.plan_cache_info()
    print("ssr varlen sub-batching:", info)
    assert info["bytes"] <= budget_mb << 20               # one 6-clip plan would hold ~13 GB
    eng.check_errors()
    eng.close()


def test_ssr_restore_many_matches_restore(model):
    lengths = [44100 * 2 + 7, 1100, 44100 * 5, 30000, 30001, 44100 * 2 + 6, 9999]
    clips = make_clips(lengths, seed=11)
    res = model.restore_many(clips, max_batch=3)          # groups of 3, 2, 2
    assert len(res) == len(clips)
    for c, r in zip(clips, res):
        assert r.shape == c.shape
        assert torch.equal(r.cpu(), model.restore(c[None].cuda())[0].cpu())


def test_ssr_varlen_bad_input(model, state):
    from voicefixer_main_b200 import VoiceFixer
    from voicefixer_main_b200 import _lib as L
    eng = model._engine()
    x = O.synth_clips(3, 5000, seed=2).cuda()
    out = torch.empty_like(x)
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    n0 = eng.launch_count()
    for lens in ([1024, 5000, 5000], [5000, 5001, 4000], [5000, 4000], [5000, 4000, 3000, 2000]):
        with pytest.raises(ValueError):
            eng.ssr_restore_varlen(x, lens)
    for lens in ([5000, 1024, 2000], [5000, 5001, 2000], [0, 5000, 2000]):
        arr = (ctypes.c_int64 * 3)(*lens)
        rc = eng.lib.vf_ssr_restore_varlen(eng.ctx, ctypes.c_void_p(x.data_ptr()), 3, 5000, arr,
                                           ctypes.c_void_p(out.data_ptr()), stream)
        assert rc == L.VF_EINVAL and b"1024 < n" in eng.lib.vf_last_error(eng.ctx)
    assert eng.launch_count() == n0
    # a context holding only the GSR networks (analysis module + vocoder) has no unet_v2 to run
    g = VoiceFixer().load_state_dict(state).eval().to("cuda:0")
    ge = g._engine()
    arr = (ctypes.c_int64 * 3)(5000, 4000, 3000)
    n1 = ge.launch_count()
    rc = ge.lib.vf_ssr_restore_varlen(ge.ctx, ctypes.c_void_p(x.data_ptr()), 3, 5000, arr, ctypes.c_void_p(out.data_ptr()),
                                      stream)
    assert rc == L.VF_ESTATE and b"unet_v2" in ge.lib.vf_last_error(ge.ctx)
    assert ge.launch_count() == n1
    ge.close()
    eng.check_errors()


def test_restore_files_with_an_ssr_model(model, tmp_path):
    """16 kHz and 44.1 kHz files, one longer than 60 s (two segments), through restore_files with an SSR model.  Each file
    must hold (a) the bytes of a per-file loop of SSR_UNet.restore + finalize + to_pcm16 over handler.split_segments, and
    (b) with saturate off, the bytes of the GSR-UNet handler's own loop (eval_gsr_unet.py:49-74) run through the object
    protocol: model.pre, model(sp, segment)['wav'], the torch peak test and save_wave.  (With saturate on, a normalised
    +1.0 peak is written as 32767, where save_wave's cast wraps it to -32768; so (b) is held against the saturate-off run.)"""
    from voicefixer_main_b200 import handler as H
    eng = model._engine()
    specs = [(44100, 44100 * 61 + 1234, 31), (16000, 16000 * 3 + 77, 32), (44100, 44100 * 7 + 5, 33)]
    srcs = []
    for k, (rate, n, seed) in enumerate(specs):
        pcm = O.to_int16(O.synth_clips(1, n, seed=seed)[0].clamp(-0.99, 0.99).numpy())
        p = str(tmp_path / f"in{k}.wav")
        H.save_pcm16(pcm, p, sample_rate=rate)
        srcs.append(p)
    outs = {s: [str(tmp_path / f"many{k}_{int(s)}.wav") for k in range(len(srcs))] for s in (True, False)}
    for s in (True, False):
        H.restore_files(model, srcs, outs[s], meta={"saturate": s, "unify_energy": True}, max_batch=2)
    peaks = []
    for k, src in enumerate(srcs):
        wav = H.load_wav(src, sample_rate=44100, engine=eng)
        # (a) per-file loop over the fused entry points
        res = []
        for sl in H.split_segments(wav.shape[0]):
            seg = torch.from_numpy(np.ascontiguousarray(wav[sl]))[None].cuda()
            res.append(eng.finalize(model.restore(seg), seg.shape[1]))
        for s in (True, False):
            one = str(tmp_path / f"one{k}_{int(s)}.wav")
            H.save_pcm16(eng.to_pcm16(torch.cat(res, -1)[0], saturate=s).cpu().numpy(), one)
            with open(one, "rb") as a, open(outs[s][k], "rb") as b:
                assert a.read() == b.read(), f"file {k}, saturate {s}: restore_files != per-segment restore loop"
        # (b) eval_gsr_unet.py:49-74 through the object protocol
        res = []
        for sl in H.split_segments(wav.shape[0]):
            segment = torch.from_numpy(np.ascontiguousarray(wav[sl]))[None, None].cuda()
            sp, _ = model.pre(segment)
            out = model(sp, segment)["wav"]
            peaks.append(float(torch.max(torch.abs(out))))
            if torch.max(torch.abs(out)) > 1.0:
                out = out / torch.max(torch.abs(out))
            assert out.shape == segment.shape                  # trim_center has nothing to trim
            res.append(out)
        ref = str(tmp_path / f"ref{k}.wav")
        H.save_wave(torch.cat(res, -1)[0, 0].cpu().numpy(), fname=ref, sample_rate=44100)
        with open(ref, "rb") as a, open(outs[False][k], "rb") as b:
            assert a.read() == b.read(), f"file {k}: restore_files != the GSR-UNet handler's loop"
    print("ssr restore_files: per-segment peaks before normalisation", peaks)
    eng.check_errors()

"""Generate tests/golden/*.npz from the REFERENCE ITSELF.  TEST INFRASTRUCTURE ONLY.

Needs the reference tree at ref_import.REFERENCE_ROOT:
    python oracle/make_golden.py [ssr | small | reference | longform]

Every output below is produced by the reference's own modules imported unmodified
(oracle/ref_import.py): FDomainHelper + MelScale (stage A), VoiceFixer.forward ->
Generator -> UNetResComplex_100Mb (stage B), and the handler body of
eval_gsr_voicefixer.py:41-75 (end to end; its vocoder is the restated stage C).
Weights are NOT stored (65 M parameters): they are regenerated from
voicefixer_main_b200.weights.make_state(seed), and a fingerprint of that state is
stored so generator drift is detected instead of silently failing parity.
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import ref_import, vf_oracle as O            # noqa: E402
from voicefixer_main_b200.weights import make_state      # noqa: E402

SEED = 1234
GOLD = os.path.join(ROOT, "tests", "golden")


def state_fingerprint(sd) -> np.ndarray:
    keys = sorted(k for k in sd if sd[k].is_floating_point())
    probe = [keys[0], keys[len(keys) // 3], keys[len(keys) // 2], keys[-1]]
    return np.array([float(sd[k].double().abs().sum()) for k in probe] +
                    [float(sum(sd[k].double().sum() for k in keys))], dtype=np.float64)


def main():
    torch.set_num_threads(os.cpu_count() or 1)
    os.makedirs(GOLD, exist_ok=True)
    sd = make_state(SEED)
    model, _ = ref_import.build_reference_model(sd)
    fp = state_fingerprint(sd)
    with torch.no_grad():
        # stage A: ragged lengths incl. a non-multiple of the hop and the minimum useful size
        for tag, n in (("a_n4410", 4410), ("a_n30001", 30001)):
            wav = O.synth_clips(3, n, seed=11)
            sp, cos, sin = model.f_helper.wav_to_spectrogram_phase(wav[:, None, :])
            mel = model.mel(sp.permute(0, 1, 3, 2)).permute(0, 1, 3, 2)
            np.savez_compressed(os.path.join(GOLD, f"stage_{tag}.npz"), wav=wav.numpy(), sp=sp.numpy(),
                                mel=mel.numpy(), fingerprint=fp)
        # stage B: the reference's own smoke shape (unet.py:107, T=101) and a 10 s clip (T=1001)
        for tag, t, b in (("b_t101", 101, 2), ("b_t1001", 1001, 1)):
            g = torch.Generator().manual_seed(5 + t)
            mel_orig = 10 ** (torch.randn(b, 1, t, 128, generator=g) * 0.8 - 1.0)
            mel_orig[:, :, ::17, ::5] = 0.0                      # exercise the 1e-8 clip of to_log
            out = model(mel_orig)["mel"]
            np.savez_compressed(os.path.join(GOLD, f"stage_{tag}.npz"), mel_orig=mel_orig.numpy(),
                                log_mel=out.numpy(), fingerprint=fp)
        # end to end: 1 s clips (B=2) and one 10 s clip through the handler body
        for tag, n, b in (("e2e_1s", 44100, 2), ("e2e_10s", 441000, 1)):
            wav = O.synth_clips(b, n, seed=21 + b)
            col = {}
            out = ref_import.reference_handler_batch(model, wav, collect=col)
            np.savez_compressed(os.path.join(GOLD, f"{tag}.npz"), wav=wav.numpy(), out=out.numpy(),
                                log_mel=torch.cat(col["log_mel"]).numpy(), fingerprint=fp)
            print(tag, "out rms", float(out.pow(2).mean().sqrt()))
    print("golden written to", GOLD)


def main_ssr():
    """SURVEY.md 8(f) row 1 (next path): models/components/unet_v2.py UNetResComplex_100Mb imported unmodified, with
    the UNet tensors of make_state(SEED) under the SSR prefix (same shapes, models/ssr_unet.py:49).  Its STFT/ISTFT
    helpers are the oracle's restatements (torchlibrosa is absent)."""
    from voicefixer_main_b200.arch import UNET_PREFIX
    torch.set_num_threads(os.cpu_count() or 1)
    sd = make_state(SEED)
    ssr = {k.replace(UNET_PREFIX, "generator.unet."): v for k, v in sd.items() if k.startswith(UNET_PREFIX)}
    net = ref_import.build_reference_unet_v2(ssr)
    fp = state_fingerprint(sd)
    with torch.no_grad():
        wav = O.synth_clips(2, 63 * 441 + 200, seed=51)[:, None, :]     # T = 64 frames, ragged sample count
        sp, cos, sin = net.f_helper.wav_to_spectrogram_phase(wav)
        out = net(sp, wav)["wav"]
        mag = O.unet_v2_forward(ssr, sp)                                  # bit-identical to the module's out_mag (tested)
    np.savez_compressed(os.path.join(GOLD, "ssr_t64.npz"), wav=wav[:, 0].numpy(), out_mag=mag.numpy(),
                        out=out[:, 0].numpy(), fingerprint=fp)
    print("ssr_t64 out rms", float(out.pow(2).mean().sqrt()))


def main_small():
    """SURVEY.md 8(f) row 4: the `unet_small` analysis module (models/components/unet_small.py) imported unmodified,
    through Generator.forward's arithmetic (gsr_voicefixer.py:86-91: unet(to_log(mel)) + to_log(mel))."""
    torch.set_num_threads(os.cpu_count() or 1)
    sd = make_state(SEED)
    net = ref_import.build_reference_unet_small(sd)
    from tools.pytorch.pytorch_util import to_log
    g = torch.Generator().manual_seed(77)
    mel_orig = 10 ** (torch.randn(1, 1, 101, 128, generator=g) * 0.8 - 1.0)
    with torch.no_grad():
        out = net(to_log(mel_orig))["mel"] + to_log(mel_orig)
    np.savez_compressed(os.path.join(GOLD, "stage_b_small_t101.npz"), mel_orig=mel_orig.numpy(), log_mel=out.numpy(),
                        fingerprint=state_fingerprint(sd))
    print("stage_b_small_t101 written")


STRIDE = 7       # reference outputs are stored as out.reshape(-1)[::STRIDE]: 7 is coprime to the 128 mel bins and the hop


def sample(t: torch.Tensor, stride: int = STRIDE) -> np.ndarray:
    return t.detach().reshape(-1)[::stride].contiguous().numpy()


def main_reference():
    """What tests/test_oracle_vs_reference.py and test_host_cpu.py::test_arch_keys_match_reference_state_dict compare
    the restatement with (reference_oracle.npz): the reference's own modules run on the inputs those tests build,
    outputs stored as a strided sample, and the UNet state-dict keys and shapes in registration order."""
    from voicefixer_main_b200.arch import UNET_PREFIX
    torch.set_num_threads(os.cpu_count() or 1)
    sd = make_state(SEED)
    model, _ = ref_import.build_reference_model(sd)
    ref_import.install_shims()
    from tools.pytorch.pytorch_util import from_log, to_log
    from tools.utils import trim_center
    g = {"fingerprint": state_fingerprint(sd), "stride": np.int64(STRIDE)}

    fb = model.mel.fb
    nz = torch.nonzero(fb.reshape(-1))[:, 0]
    g.update(fb_shape=np.array(fb.shape), fb_index=nz.int().numpy(), fb_value=fb.reshape(-1)[nz].numpy())

    gl = torch.Generator().manual_seed(23)
    x = torch.rand(3, 1, 7, 128, generator=gl) * 3
    x[0, 0, 0, :4] = 0
    y = torch.randn(3, 1, 7, 128, generator=gl) * 4
    g.update(to_log=to_log(x).numpy(), from_log=from_log(y).numpy())
    try:
        to_log(-x - 1)
        g["to_log_rejects_negative"] = np.bool_(False)
    except AssertionError:
        g["to_log_rejects_negative"] = np.bool_(True)

    starts = []
    for le, lr in ((20, 14), (443646, 441000), (16, 16)):
        est = torch.arange(float(le))[None, None]
        out = trim_center(est, torch.zeros(1, 1, lr))[0]
        s = int(out[0, 0, 0])
        assert torch.equal(out, est[..., s:s + lr])            # a contiguous window: its start says it all
        starts.append((le, lr, s))
    g["trim_center"] = np.array(starts, dtype=np.int64)

    with torch.no_grad():
        gm = torch.Generator().manual_seed(3)
        for t in (64, 101, 130):
            mel = 10 ** (torch.randn(2, 1, t, 128, generator=gm) - 1)
            g[f"unet_t{t}"] = sample(model(mel)["mel"])
        wav = O.synth_clips(2, 30000, seed=9)
        g["handler"] = sample(ref_import.reference_handler_batch(model, wav, seg_samples=12000))

        ssr = {k.replace(UNET_PREFIX, "generator.unet."): v for k, v in sd.items() if k.startswith(UNET_PREFIX)}
        net = ref_import.build_reference_unet_v2(ssr)
        for n in (63 * 441, 70 * 441 + 17):
            w = O.synth_clips(1, n, seed=n)[:, None, :]
            sp, _, _ = O.wav_to_spectrogram_phase(w)
            g[f"ssr_n{n}"] = sample(net(sp, w)["wav"])

        small = ref_import.build_reference_unet_small(sd)
        mel = 10 ** (torch.randn(1, 1, 101, 128, generator=torch.Generator().manual_seed(4)) - 1)
        g["small"] = sample(small(to_log(mel))["mel"] + to_log(mel))
        g["small_full"] = sample(model(mel)["mel"])

    keys = [(k[len(UNET_PREFIX):], tuple(v.shape)) for k, v in model.state_dict().items() if k.startswith(UNET_PREFIX)]
    g["unet_keys"] = np.array([k for k, _ in keys])
    g["unet_shapes"] = np.array([list(s) + [0] * (4 - len(s)) for _, s in keys], dtype=np.int32)   # zero-padded
    g["unet_ndims"] = np.array([len(s) for _, s in keys], dtype=np.int32)
    np.savez_compressed(os.path.join(GOLD, "reference_oracle.npz"), **g)
    print("reference_oracle.npz written")


def main_longform():
    """What tests/test_longform_cpu.py compares the overlap-add mirrors with: the reference's own LambdaOverlapAdd
    (tools/dsp/overlapadd_boxcar.py and tools/dsp/overlapadd.py, loaded unmodified) run over that test's toy network,
    signals and cases: every second output sample (the comparison is bit for bit) and the chunk shapes that reached the
    network."""
    import importlib.util

    def load(path, name):
        spec = importlib.util.spec_from_file_location(name, path)
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        return mod

    sys.path.insert(0, os.path.join(ROOT, "tests"))              # the test module imports its conftest
    T = load(os.path.join(ROOT, "tests", "test_longform_cpu.py"), "test_longform_cpu")
    boxcar = load(os.path.join(ref_import.REFERENCE_ROOT, "tools", "dsp", "overlapadd_boxcar.py"), "ref_overlapadd_boxcar")
    ola = load(os.path.join(ref_import.REFERENCE_ROOT, "tools", "dsp", "overlapadd.py"), "ref_overlapadd")
    g = {"stride": np.int64(2)}
    for n, w, m in T.CASES:
        for windowed in (False, True):
            net = T.ToyNet()
            ref = boxcar.LambdaOverlapAdd(nnet=net, n_src=1, window_size=w, in_margin=m, window="hann", reorder_chunks=False)
            ref.use_window = windowed
            key = T.boxcar_key(n, w, m, windowed)
            g[key] = sample(ref(T._signal(n)), 2)
            g[key + "_calls"] = np.array(sorted(net.calls), dtype=np.int64)
    for n, w, hop in T.OLA_CASES:
        for windowed in (True, False):
            net = T.ToyNet()
            ref = ola.LambdaOverlapAdd(nnet=net, n_src=1, window_size=w, hop_size=hop, window="hann", reorder_chunks=False)
            ref.use_window = windowed
            key = T.ola_key(n, w, hop, windowed)
            g[key] = sample(ref(T._signal(n)), 2)
            g[key + "_calls"] = np.array(net.calls, dtype=np.int64)
    np.savez_compressed(os.path.join(GOLD, "reference_longform.npz"), **g)
    print("reference_longform.npz written")


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "ssr":
        main_ssr()
    elif len(sys.argv) > 1 and sys.argv[1] == "small":
        main_small()
    elif len(sys.argv) > 1 and sys.argv[1] == "reference":
        main_reference()
    elif len(sys.argv) > 1 and sys.argv[1] == "longform":
        main_longform()
    else:
        main()

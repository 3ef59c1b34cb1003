"""Import the reference's own modules UNMODIFIED from /root/reference.  TEST INFRASTRUCTURE ONLY.

Works only where the reference tree exists; used by oracle/make_golden.py to store
what the reference computes under tests/golden/, which the tests compare against.

Third-party packages the reference imports but this image lacks are replaced by
stubs in sys.modules *before* the import:

* torchlibrosa.stft.STFT  -> functional shim over oracle.vf_oracle.stft_conv_dft
  (the published torchlibrosa 0.0.7 algorithm: reflect pad + windowed-DFT conv1d).
* voicefixer.Vocoder      -> oracle.vf_oracle.vocoder_forward over seeded weights
  (source + checkpoint unavailable: stage C parity is unpinned, see vf_oracle header).
* pytorch_lightning.LightningModule -> nn.Module with no-op save_hyperparameters/log.
* librosa / soundfile / matplotlib / progressbar / augment / ... -> permissive
  empty modules (never called on the inference path we exercise).

Modules that run `git.Repo("", search_parent_directories=True)` at import
(models/components/unet.py:5) need the cwd inside a git work tree: a git checkout of
this repository is one.
"""
import os
import sys
import types

import torch
import torch.nn as nn

REFERENCE_ROOT = "/root/reference"
REPO_ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def available() -> bool:
    return os.path.isdir(os.path.join(REFERENCE_ROOT, "models"))


class _Permissive(types.ModuleType):
    def __getattr__(self, name):
        if name.startswith("__"):
            raise AttributeError(name)
        m = _Permissive(self.__name__ + "." + name)
        sys.modules[m.__name__] = m
        setattr(self, name, m)
        return m

    def __call__(self, *a, **k):
        return None


def _stub(name):
    m = _Permissive(name)
    m.__path__ = []
    sys.modules[name] = m
    return m


_installed = False


def install_shims():
    global _installed
    if _installed:
        return
    if not available():
        raise RuntimeError("reference tree not present at " + REFERENCE_ROOT)
    if REPO_ROOT not in sys.path:
        sys.path.insert(0, REPO_ROOT)
    from oracle import vf_oracle
    from voicefixer_main_b200.arch import VocoderConfig

    for n in ["librosa", "librosa.display", "matplotlib", "matplotlib.pyplot", "matplotlib.cm", "soundfile",
              "progressbar", "augment", "pynvml", "speechmetrics", "skimage", "skimage.metrics", "tensorboardX",
              "julius", "diffq", "coloredlogs", "torchlibrosa", "torchlibrosa.stft", "voicefixer",
              "pytorch_lightning", "pytorch_lightning.callbacks", "pytorch_lightning.utilities"]:
        if n not in sys.modules:
            _stub(n)

    class LightningModule(nn.Module):
        def save_hyperparameters(self, *a, **k):
            pass

        def log(self, *a, **k):
            pass

    sys.modules["pytorch_lightning"].LightningModule = LightningModule
    sys.modules["pytorch_lightning.callbacks"].Callback = object
    sys.modules["pytorch_lightning.utilities"].rank_zero_only = lambda f: f

    class STFT(nn.Module):
        def __init__(self, n_fft=2048, hop_length=None, win_length=None, window="hann", center=True,
                     pad_mode="reflect", freeze_parameters=True):
            super().__init__()
            # unet_v2.py:29 passes center=(True,) (a stray comma): truthy, which is all torchlibrosa tests
            assert (n_fft, hop_length, win_length, window, bool(center), pad_mode) == \
                (vf_oracle.N_FFT, vf_oracle.HOP, vf_oracle.N_FFT, "hann", True, "reflect")

        def forward(self, x):
            return vf_oracle.stft_conv_dft(x)

    class ISTFT(nn.Module):
        """torchlibrosa.stft.ISTFT stand-in: oracle.vf_oracle.istft (restated, pinned by torch.istft / round trip)."""

        def __init__(self, n_fft=2048, hop_length=None, win_length=None, window="hann", center=True,
                     pad_mode="reflect", freeze_parameters=True, **kw):
            super().__init__()
            assert (n_fft, hop_length, win_length, window, bool(center)) == (vf_oracle.N_FFT, vf_oracle.HOP, vf_oracle.N_FFT, "hann", True)

        def forward(self, real_stft, imag_stft, length):
            return vf_oracle.istft(real_stft, imag_stft, length)

    sys.modules["torchlibrosa.stft"].STFT = STFT
    sys.modules["torchlibrosa.stft"].ISTFT = ISTFT
    sys.modules["torchlibrosa.stft"].magphase = None

    class Vocoder(nn.Module):
        """Stand-in for voicefixer.Vocoder(sample_rate): weights injected via set_state()."""

        def __init__(self, sample_rate):
            super().__init__()
            assert sample_rate == 44100
            self.cfg = VocoderConfig()
            self._sd = None

        def set_state(self, sd):
            self._sd = sd

        def forward(self, mel, cuda=False):
            return vf_oracle.vocoder_forward(self._sd, mel, self.cfg)

    sys.modules["voicefixer"].Vocoder = Vocoder
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    _installed = True


def build_reference_model(state: dict, config: str = "config/vctk_base_voicefixer_unet.json"):
    """The reference's own VoiceFixer (models/gsr_voicefixer.py:94) in eval mode with
    `state` loaded (UNet keys via load_state_dict, vocoder keys into the shim)."""
    install_shims()
    cwd = os.getcwd()
    os.chdir(REPO_ROOT)
    try:
        from models.gsr_voicefixer import VoiceFixer
        from tools.utils import get_hparams_from_file
        hp = get_hparams_from_file(os.path.join(REFERENCE_ROOT, config))
        model = VoiceFixer(hp, channels=2, type_target="vocals")
    finally:
        os.chdir(cwd)
    own = model.state_dict()
    unet_sd = {k: v for k, v in state.items() if k in own}
    missing = [k for k in own if k not in unet_sd and k != "mel.fb"]
    assert not missing, missing[:5]
    model.load_state_dict(unet_sd, strict=False)
    model.vocoder.set_state({k: v for k, v in state.items() if k.startswith("vocoder.")})
    model.eval()
    return model, hp


def build_reference_unet_v2(state: dict, prefix: str = "generator.unet."):
    """The reference's SSR analysis network (models/components/unet_v2.py:20, channels=1) in eval mode with the
    tensors of `state` under `prefix` loaded; its STFT/ISTFT helpers are the shims above."""
    install_shims()
    cwd = os.getcwd()
    os.chdir(REPO_ROOT)
    try:
        from models.components.unet_v2 import UNetResComplex_100Mb
        net = UNetResComplex_100Mb(channels=1)
    finally:
        os.chdir(cwd)
    own = net.state_dict()
    sd = {k[len(prefix):]: v for k, v in state.items() if k.startswith(prefix) and k[len(prefix):] in own}
    missing = [k for k in own if k not in sd and not k.startswith("f_helper.")]
    assert not missing, missing[:5]
    net.load_state_dict(sd, strict=False)
    net.eval()
    return net


def build_reference_unet_small(state: dict, prefix: str = "generator.analysis_module."):
    """models/components/unet_small.py:12 (selected by `unet_small: true`, gsr_voicefixer.py:51-53) in eval mode with the
    analysis-module tensors of `state`: its *Res1B blocks (modules.py:112-165) carry the same four ConvBlockRes and
    key names as the *Res4B blocks of unet.py, so the mel UNet's state loads without renaming."""
    install_shims()
    cwd = os.getcwd()
    os.chdir(REPO_ROOT)
    try:
        from models.components.unet_small import UNetResComplex_100Mb
        net = UNetResComplex_100Mb(channels=1)
    finally:
        os.chdir(cwd)
    own = net.state_dict()
    sd = {k[len(prefix):]: v for k, v in state.items() if k.startswith(prefix) and k[len(prefix):] in own}
    missing = [k for k in own if k not in sd]
    assert not missing, missing[:5]
    net.load_state_dict(sd, strict=True)
    net.eval()
    return net


def reference_handler_batch(model, wav: torch.Tensor, seg_samples: int = 44100 * 60, collect=None):
    """The body of handler() (eval_gsr_voicefixer.py:41-75) driven on in-memory clips
    (librosa/soundfile I/O is out of scope), one clip at a time as the reference does."""
    install_shims()
    from tools.pytorch.pytorch_util import from_log
    from tools.utils import trim_center
    outs = []
    with torch.no_grad():
        for b in range(wav.shape[0]):
            wav_10k = wav[b]
            res = []
            break_point = seg_samples
            while break_point < wav_10k.shape[0] + seg_samples:
                segment = wav_10k[break_point - seg_samples:break_point]
                inp = segment[None, None, ...]
                sp, _, _ = model.f_helper.wav_to_spectrogram_phase(inp)
                mel_noisy = model.mel(sp.permute(0, 1, 3, 2)).permute(0, 1, 3, 2)
                out_model = model(mel_noisy)
                denoised_mel = from_log(out_model["mel"])
                out = model.vocoder(denoised_mel)
                if torch.max(torch.abs(out)) > 1.0:
                    out = out / torch.max(torch.abs(out))
                out, _ = trim_center(out, segment)
                if collect is not None:
                    collect.setdefault("mel_noisy", []).append(mel_noisy)
                    collect.setdefault("log_mel", []).append(out_model["mel"])
                res.append(out)
                break_point += seg_samples
            outs.append(torch.cat(res, -1)[0, 0])
    return torch.stack(outs)

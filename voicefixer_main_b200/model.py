"""Host-side mirror of the reference's model objects for the inference hot path.

Same names, arguments and error behaviour as the objects eval_gsr_voicefixer.py:handler() uses
(SURVEY.md 8(b)), backed entirely by libb200vf.so:

    VoiceFixer(hp, channels, type_target)       models/gsr_voicefixer.py:94
      .load_from_checkpoint(ckpt) / .load_state_dict(sd) / .eval() / .to(device)
      .pre(wav[B,1,N]) -> (sp, mel_orig)         models/gsr_voicefixer.py:178-181
      .forward(mel_orig) -> {'mel': log10 mel}   models/gsr_voicefixer.py:183-193
      .f_helper.wav_to_spectrogram_phase(x)      tools/pytorch/modules/fDomainHelper.py:67-89
      .mel(specgram[..., freq, time])            tools/pytorch/mel_scale.py:52-64
      .vocoder(mel[B,1,T,128]) -> wav[B,1,L]     eval_gsr_voicefixer.py:66
    plus the batched fused entry points the reference lacks:
      .restore(wav[B,N]) -> wav[B,N]             one launch chain for stages A -> B -> C + normalise + trim
      .restore_host(pinned_in, pinned_out)
      .restore_many([wav_i, ...]) -> [out_i, ...]  clips of any lengths, batched (Engine.restore_varlen)
    SSR_UNet / GSR_UNet (models/ssr_unet.py, gsr_unet.py): .pre, model(sp, wav)['wav'], .restore(wav[B,N]) and
      .restore_many([wav_i, ...])             clips of any lengths, batched (Engine.ssr_restore_varlen)

PyTorch is used only to own device memory and streams; every tensor handed back is written by a
hand-written sm_100a kernel.  Tensors must be fp32 CUDA tensors on the model's device.
"""
import ctypes
import json
import math
from typing import Dict, Optional

import torch

from . import _lib as L
from .arch import SSR_PREFIX, UNET_PREFIX, VocoderConfig, frames_for, unet_keys, vocoder_keys


class HParams(dict):
    """Nested config mapping with attribute access.  Any mapping subscriptable by the reference's string keys works as
    `hp` (the reference's own tools/utils.py HParams included); this is only the default container."""

    def __init__(self, **kw):
        super().__init__({k: HParams(**v) if isinstance(v, dict) else v for k, v in kw.items()})

    __getattr__ = dict.__getitem__


def get_hparams_from_file(config_path) -> HParams:
    """tools/utils.py:114-120."""
    with open(config_path, "r") as f:
        return HParams(**json.loads(f.read()))


def default_hparams() -> HParams:
    """The hot-path-relevant keys of config/vctk_base_voicefixer_unet.json."""
    return HParams(**{
        "task": {"gsr": {"gsr_model": {"voicefixer": {"unet": True, "unet_small": False, "bi_gru": False, "dnn": False}}}},
        "data": {"sampling_rate": 44100},
        "model": {"mel_freq_bins": 128, "window_size": 2048, "hop_size": 441, "pad_mode": "reflect",
                  "window": "hann", "channels_in": 1},
    })


def melscale_fbanks(n_freqs=1025, f_min=0.0, f_max=22050.0, n_mels=128, sample_rate=44100):
    """HTK triangular filterbank, same fp32 op order as tools/pytorch/mel_scale.py:131-221 (norm=None)."""
    all_freqs = torch.linspace(0, sample_rate // 2, n_freqs)
    m_min = 2595.0 * math.log10(1.0 + (f_min / 700.0))
    m_max = 2595.0 * math.log10(1.0 + (f_max / 700.0))
    m_pts = torch.linspace(m_min, m_max, n_mels + 2)
    f_pts = 700.0 * (10.0 ** (m_pts / 2595.0) - 1.0)
    f_diff = f_pts[1:] - f_pts[:-1]
    slopes = f_pts.unsqueeze(0) - all_freqs.unsqueeze(1)
    down_slopes = (-1.0 * slopes[:, :-2]) / f_diff[:-1]
    up_slopes = slopes[:, 2:] / f_diff[1:]
    return torch.max(torch.zeros(1), torch.min(down_slopes, up_slopes))


def group_sizes(n: int, max_batch: int):
    """Sizes of the groups restore_many splits n sorted clips into: ceil(n / max_batch) groups, none above max_batch, sizes
    differing by at most one (larger groups first)."""
    if n <= 0:
        return []
    k = -(-n // max_batch)
    q, r = divmod(n, k)
    return [q + 1] * r + [q] * (k - r)


def restore_grouped(mdl, wavs, max_batch: int, run) -> list:
    """The batching of the restore_many methods: sort the 1-D clips by length, split them into group_sizes groups, pad
    each group to its longest clip ([g, n_max] on the model's device) and restore it with ONE `run(engine, batch,
    lengths)` call, which returns [g, n_max]; the clips come back (1-D views of those rows) in input order."""
    if max_batch < 1:
        raise ValueError("max_batch must be at least 1")
    clips = [torch.as_tensor(w).reshape(-1) for w in wavs]
    if not clips:
        return []
    eng = mdl._engine()
    order = sorted(range(len(clips)), key=lambda i: clips[i].shape[0])
    groups = group_sizes(len(clips), max_batch)
    result = [None] * len(clips)
    pos = 0
    for g in groups:
        idx = order[pos:pos + g]
        pos += g
        lens = [clips[i].shape[0] for i in idx]
        batch = torch.nn.utils.rnn.pad_sequence([clips[i].to(device=eng.device, dtype=torch.float32) for i in idx],
                                                batch_first=True)
        out = run(eng, batch.contiguous(), lens)
        for row, i in enumerate(idx):
            result[i] = out[row, :lens[row]]
    return result


def _ptr(t: Optional[torch.Tensor]):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _check_in(t: torch.Tensor, device, what: str):
    if not isinstance(t, torch.Tensor) or t.dtype != torch.float32 or not t.is_cuda or t.device != device:
        raise TypeError(f"{what} must be a float32 CUDA tensor on {device}")
    return t.contiguous()


class Engine:
    """One vf_ctx on one device."""

    def __init__(self, device, cfg: Optional[VocoderConfig] = None):
        self.lib = L.load_library()
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("voicefixer_main_b200 runs on CUDA devices only (no CPU fallback)")
        self.index = self.device.index if self.device.index is not None else torch.cuda.current_device()
        self.device = torch.device("cuda", self.index)
        self.voc_cfg = cfg or VocoderConfig()
        c = L.VfConfig()
        self.lib.vf_default_config(ctypes.byref(c))
        v = self.voc_cfg
        c.voc_cond_channels, c.voc_cond_layers, c.voc_channels = v.cond_channels, v.cond_layers, v.channels
        c.voc_num_stages = len(v.upsample_scales)
        for i, (s, d) in enumerate(zip(v.upsample_scales, v.resstack_depth)):
            c.voc_scales[i], c.voc_depth[i] = s, d
        c.voc_stage_slope, c.voc_res_slope, c.voc_min_db, c.voc_ref_db = v.stage_slope, v.res_slope, v.min_db, v.ref_db
        c.voc_amp_floor, c.voc_tail_value, c.voc_tail_base = v.amp_floor, v.tail_pad_value, v.tail_pad_base
        c.voc_mel_weight_a, c.voc_mel_weight_b = v.mel_weight_a, v.mel_weight_b
        c.voc_tail_tanh = int(getattr(v, "tail_tanh", True))
        self.ctx = ctypes.c_void_p()
        rc = self.lib.vf_create(ctypes.byref(self.ctx), self.index, ctypes.byref(c))
        if rc != L.VF_OK:
            msg = self.lib.vf_last_error(None)
            raise L.EngineError(rc, msg.decode() if msg else "")
        self.loaded = False

    def close(self):
        if getattr(self, "ctx", None) is not None and self.ctx.value:
            self.lib.vf_destroy(self.ctx)
            self.ctx = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc):
        return L.check(self.lib, self.ctx, rc)

    def load_state(self, state: Dict[str, torch.Tensor], need=("unet", "vocoder")):
        """Hands the tensors of the networks in `need` to vf_load_weights: "unet" = generator.analysis_module.*
        (VoiceFixer's mel UNet), "vocoder" = vocoder.* (the restated generator, arch.vocoder_keys), "ssr" =
        generator.unet.* (unet_v2 of SSR_UNet / GSR_UNet).  A missing key raises KeyError naming its source."""
        groups = {
            "unet": [UNET_PREFIX + k for k, s in unet_keys() if not k.endswith("num_batches_tracked")],
            "ssr": [SSR_PREFIX + k for k, s in unet_keys() if not k.endswith("num_batches_tracked")],
            "vocoder": ["vocoder." + k for k, _ in vocoder_keys(self.voc_cfg)],
        }
        needed = []
        for g in need:
            missing = [k for k in groups[g] if k not in state]
            if missing:
                hint = ""
                if g == "vocoder":
                    hint = (" - the vocoder of a reference checkpoint is the pip `voicefixer` package's own module with its "
                            "own key names and a separately downloaded weight file; convert it to arch.vocoder_keys "
                            "(weight norm folded) and pass it as vocoder_state")
                raise KeyError(f"state dict is missing {len(missing)} '{g}' tensors, e.g. {missing[:3]}{hint}")
            needed += groups[g]
        fb = state["mel.fb"] if "mel.fb" in state else melscale_fbanks()
        items = [("mel.fb", fb)] + [(k, state[k]) for k in needed]
        descs = (L.VfTensorDesc * len(items))()
        keep = []
        for d, (k, t) in zip(descs, items):
            t = t.detach().to(dtype=torch.float32).contiguous()
            keep.append(t)
            d.name = k.encode()
            d.data = t.data_ptr()
            d.ndim = t.dim()
            for i, s in enumerate(t.shape):
                d.shape[i] = s
            d.on_device = 1 if t.is_cuda else 0
        self._ck(self.lib.vf_load_weights(self.ctx, descs, len(items)))
        self.loaded = True

    # ---- stage entry points (device tensors in, device tensors out)
    def frontend(self, wav: torch.Tensor, want_sp: bool = False, want_phase: bool = False, want_mel: bool = True):
        wav = _check_in(wav, self.device, "wav")
        b, n = wav.shape
        t = frames_for(n)
        mel = torch.empty(b, t, 128, device=self.device) if want_mel else None
        sp = torch.empty(b, t, 1025, device=self.device) if (want_sp or want_phase) else None
        cos = torch.empty_like(sp) if want_phase else None
        sin = torch.empty_like(sp) if want_phase else None
        with torch.cuda.device(self.device):
            self._ck(self.lib.vf_frontend(self.ctx, _ptr(wav), b, n, _ptr(mel), _ptr(sp), _ptr(cos), _ptr(sin), _stream()))
        return mel, sp, cos, sin

    def unet_mel(self, mel_lin: torch.Tensor) -> torch.Tensor:
        mel_lin = _check_in(mel_lin, self.device, "mel")
        b, t, m = mel_lin.shape
        assert m == 128
        out = torch.empty_like(mel_lin)
        with torch.cuda.device(self.device):
            self._ck(self.lib.vf_unet_mel(self.ctx, _ptr(mel_lin), b, t, _ptr(out), _stream()))
        return out

    def vocoder(self, mel_lin: torch.Tensor) -> torch.Tensor:
        mel_lin = _check_in(mel_lin, self.device, "mel")
        b, t, m = mel_lin.shape
        assert m == 128
        out = torch.empty(b, self.lib.vf_vocoder_out_len(self.ctx, t), device=self.device)
        with torch.cuda.device(self.device):
            self._ck(self.lib.vf_vocoder(self.ctx, _ptr(mel_lin), b, t, _ptr(out), _stream()))
        return out

    def restore(self, wav: torch.Tensor, out: Optional[torch.Tensor] = None, unify_energy: bool = False) -> torch.Tensor:
        wav = _check_in(wav, self.device, "wav")
        b, n = wav.shape
        out = torch.empty_like(wav) if out is None else out
        flags = L.VF_RESTORE_UNIFY_ENERGY if unify_energy else 0
        with torch.cuda.device(self.device):
            self._ck(self.lib.vf_restore_ex(self.ctx, _ptr(wav), b, n, _ptr(out), flags, _stream()))
        return out

    def restore_varlen(self, wav: torch.Tensor, lengths, out: Optional[torch.Tensor] = None,
                       unify_energy: bool = False) -> torch.Tensor:
        """restore() over clips of different lengths: wav [B, n_max], row b holds lengths[b] valid samples (the rest is
        never read).  Row b of the result is bit-identical to restore() of that clip alone; samples past lengths[b] are 0."""
        wav, lens = self._varlen_args(wav, lengths, "restore_varlen")
        b, n = wav.shape
        out = torch.empty_like(wav) if out is None else out
        flags = L.VF_RESTORE_UNIFY_ENERGY if unify_energy else 0
        arr = (ctypes.c_int64 * b)(*lens)
        with torch.cuda.device(self.device):
            self._ck(self.lib.vf_restore_varlen(self.ctx, _ptr(wav), b, n, arr, _ptr(out), flags, _stream()))
        return out

    def _varlen_args(self, wav: torch.Tensor, lengths, what: str):
        """The host-side checks of the varlen entry points: (wav, lengths as ints), or ValueError before any launch."""
        wav = _check_in(wav, self.device, "wav")
        if wav.dim() != 2:
            raise ValueError(f"wav must be [B, n_max], got shape {tuple(wav.shape)}")
        b, n = wav.shape
        lens = [int(x) for x in lengths]
        if len(lens) != b:
            raise ValueError(f"{what}: {len(lens)} lengths for a batch of {b}")
        bad = [(i, x) for i, x in enumerate(lens) if not 1024 < x <= n]
        if bad:
            raise ValueError(f"{what}: every length must satisfy 1024 < length <= n_max = {n}; "
                             f"got {bad[:4]} (clip, length)")
        return wav, lens

    def mel(self, specgram: torch.Tensor) -> torch.Tensor:
        """MelScale.forward: specgram [..., 1025, time] (any strides) -> [..., 128, time]."""
        if not isinstance(specgram, torch.Tensor) or specgram.dtype != torch.float32 or specgram.device != self.device:
            raise TypeError(f"specgram must be a float32 CUDA tensor on {self.device}")
        assert specgram.dim() >= 2 and specgram.shape[-2] == 1025, "specgram: (..., freq = n_stft, time)"
        lead, t = specgram.shape[:-2], specgram.shape[-1]
        x = specgram.reshape(-1, 1025, t)               # a view whenever the leading dims are mergeable (else one copy)
        out = torch.empty(x.shape[0], t, 128, device=self.device)
        with torch.cuda.device(self.device):
            for o0 in range(0, x.shape[0], 65535):
                xs = x[o0:o0 + 65535]
                self._ck(self.lib.vf_mel(self.ctx, _ptr(xs), xs.shape[0], t, xs.stride(0), xs.stride(1), xs.stride(2),
                                         ctypes.c_void_p(out[o0:].data_ptr()), _stream()))
        return out.view(*lead, t, 128).transpose(-1, -2)     # same memory layout as the reference's matmul result

    def amp_to_original_f(self, mel_est: torch.Tensor, mel_target: torch.Tensor) -> torch.Tensor:
        """tools/utils.py:50-55 on linear mels [B,T,128]: the estimate scaled to the target's low-band energy."""
        mel_est, mel_target = _check_in(mel_est, self.device, "mel_est"), _check_in(mel_target, self.device, "mel_target")
        b, t, m = mel_est.shape
        assert m == 128 and mel_target.shape == mel_est.shape
        out = torch.empty_like(mel_est)
        with torch.cuda.device(self.device):
            self._ck(self.lib.vf_amp_to_original_f(self.ctx, _ptr(mel_est), _ptr(mel_target), b, t, _ptr(out), _stream()))
        return out

    def finalize(self, wav: torch.Tensor, n: int) -> torch.Tensor:
        """eval_gsr_voicefixer.py:68-72: per-clip peak normalise (if max|x| > 1) + trim_center to n samples."""
        wav = _check_in(wav, self.device, "wav")
        b, length = wav.shape
        out = torch.empty(b, n, device=self.device)
        with torch.cuda.device(self.device):
            self._ck(self.lib.vf_finalize(self.ctx, _ptr(wav), b, length, n, _ptr(out), _stream()))
        return out

    # ---- SSR / GSR-UNet path (unet_v2 + ISTFT)
    def ssr_forward(self, sp: Optional[torch.Tensor], wav: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        wav = _check_in(wav, self.device, "wav")
        b, n = wav.shape
        if sp is not None:
            sp = _check_in(sp, self.device, "sp")
            assert tuple(sp.shape) == (b, frames_for(n), 1025)
        out = torch.empty_like(wav) if out is None else out
        with torch.cuda.device(self.device):
            self._ck(self.lib.vf_ssr_forward(self.ctx, _ptr(sp), _ptr(wav), b, n, _ptr(out), _stream()))
        return out

    def ssr_restore_varlen(self, wav: torch.Tensor, lengths, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """ssr_forward(None, .) over clips of different lengths: wav [B, n_max], row b holds lengths[b] valid samples (the
        rest is never read).  Row b of the result is bit-identical to SSR_UNet.restore of that clip alone; samples past
        lengths[b] are 0."""
        wav, lens = self._varlen_args(wav, lengths, "ssr_restore_varlen")
        b, n = wav.shape
        out = torch.empty_like(wav) if out is None else out
        arr = (ctypes.c_int64 * b)(*lens)
        with torch.cuda.device(self.device):
            self._ck(self.lib.vf_ssr_restore_varlen(self.ctx, _ptr(wav), b, n, arr, _ptr(out), _stream()))
        return out

    def ssr_restore_host(self, wav_host: torch.Tensor, out_host: torch.Tensor):
        assert wav_host.dtype == torch.float32 and out_host.dtype == torch.float32
        assert not wav_host.is_cuda and not out_host.is_cuda and wav_host.is_contiguous() and out_host.is_contiguous()
        b, n = wav_host.shape
        with torch.cuda.device(self.device):
            self._ck(self.lib.vf_ssr_restore_host(self.ctx, _ptr(wav_host), b, n, _ptr(out_host), _stream()))

    def ssr_unet(self, sp: torch.Tensor) -> torch.Tensor:
        sp = _check_in(sp, self.device, "sp")
        b, t, f = sp.shape
        assert f == 1025
        out = torch.empty_like(sp)
        with torch.cuda.device(self.device):
            self._ck(self.lib.vf_ssr_unet(self.ctx, _ptr(sp), b, t, _ptr(out), _stream()))
        return out

    def ssr_stages(self, batch: int, n: int):
        t = frames_for(n)
        sp = torch.empty(batch, t, 1025, device=self.device)
        mag = torch.empty(batch, t, 1025, device=self.device)
        with torch.cuda.device(self.device):
            self._ck(self.lib.vf_ssr_stages(self.ctx, batch, n, _ptr(sp), _ptr(mag), _stream()))
        return sp, mag

    def istft(self, real: torch.Tensor, imag: torch.Tensor, length: int) -> torch.Tensor:
        real, imag = _check_in(real, self.device, "real"), _check_in(imag, self.device, "imag")
        b, t, f = real.shape
        assert f == 1025 and imag.shape == real.shape
        out = torch.empty(b, length, device=self.device)
        with torch.cuda.device(self.device):
            self._ck(self.lib.vf_istft(self.ctx, _ptr(real), _ptr(imag), b, t, length, _ptr(out), _stream()))
        return out

    def plan_cache_info(self):
        n, by, bu, ev = ctypes.c_int(), ctypes.c_size_t(), ctypes.c_size_t(), ctypes.c_int64()
        self._ck(self.lib.vf_plan_cache_info(self.ctx, ctypes.byref(n), ctypes.byref(by), ctypes.byref(bu), ctypes.byref(ev)))
        return {"plans": n.value, "bytes": by.value, "budget": bu.value, "evicted": ev.value}

    def restore_host(self, wav_host: torch.Tensor, out_host: torch.Tensor):
        """Pinned host tensors [B,N] in/out; asynchronous on the current stream."""
        assert wav_host.dtype == torch.float32 and out_host.dtype == torch.float32
        assert not wav_host.is_cuda and not out_host.is_cuda and wav_host.is_contiguous() and out_host.is_contiguous()
        b, n = wav_host.shape
        with torch.cuda.device(self.device):
            self._ck(self.lib.vf_restore_host(self.ctx, _ptr(wav_host), b, n, _ptr(out_host), _stream()))

    def restore_stages(self, batch: int, n: int):
        """(linear mel, restored log10 mel), each [B,T,128], of the last restore() of this shape."""
        t = frames_for(n)
        mel = torch.empty(batch, t, 128, device=self.device)
        log_mel = torch.empty(batch, t, 128, device=self.device)
        with torch.cuda.device(self.device):
            self._ck(self.lib.vf_restore_stages(self.ctx, batch, n, _ptr(mel), _ptr(log_mel), _stream()))
        return mel, log_mel

    def to_log(self, x):
        x = _check_in(x, self.device, "input")
        out = torch.empty_like(x)
        with torch.cuda.device(self.device):
            self._ck(self.lib.vf_to_log(self.ctx, _ptr(x), _ptr(out), x.numel(), _stream()))
        return out

    def from_log(self, x):
        x = _check_in(x, self.device, "input")
        out = torch.empty_like(x)
        with torch.cuda.device(self.device):
            self._ck(self.lib.vf_from_log(self.ctx, _ptr(x), _ptr(out), x.numel(), _stream()))
        return out

    def to_pcm16(self, x, saturate: bool = False):
        """fp32 samples -> int16 PCM exactly as save_wave (tools/file/wav.py:22-24) converts them; saturate=True clamps
        instead of wrapping +1.0 to -32768 (not bit-compatible with the reference, see INTEGRATION.md)."""
        x = _check_in(x, self.device, "input")
        out = torch.empty(x.shape, dtype=torch.int16, device=x.device)
        with torch.cuda.device(self.device):
            self._ck(self.lib.vf_to_pcm16_ex(self.ctx, _ptr(x), _ptr(out), x.numel(), int(saturate), _stream()))
        return out

    def check_errors(self):
        """Synchronises the current stream and raises on sticky device errors (AssertionError for the
        to_log negative-input assertion, as tools/pytorch/pytorch_util.py:158 does)."""
        with torch.cuda.device(self.device):
            rc = self.lib.vf_check_errors(self.ctx, _stream())
        if rc == L.VF_EASSERT:
            raise AssertionError(self.lib.vf_last_error(self.ctx).decode())
        self._ck(rc)

    def set_option(self, key: str, value: int):
        self._ck(self.lib.vf_set_option(self.ctx, key.encode(), int(value)))

    def launch_count(self) -> int:
        return int(self.lib.vf_launch_count(self.ctx))

    def workspace_bytes(self, batch: int, n: int) -> int:
        v = ctypes.c_size_t()
        self._ck(self.lib.vf_workspace_bytes(self.ctx, batch, n, ctypes.byref(v)))
        return int(v.value)

    def enable_stage_timing(self, on: bool = True):
        self._ck(self.lib.vf_enable_stage_timing(self.ctx, int(on)))

    def stage_times(self):
        arr = (ctypes.c_float * 4)()
        self._ck(self.lib.vf_stage_times(self.ctx, ctypes.byref(arr)))
        return dict(zip(("frontend_ms", "unet_ms", "vocoder_ms", "tail_ms"), [float(x) for x in arr]))

    def enable_op_timing(self, on: bool = True):
        self._ck(self.lib.vf_enable_op_timing(self.ctx, int(on)))

    def op_profile(self):
        """Per-launch records of the last restore() run with op timing enabled."""
        recs = []
        buf = ctypes.create_string_buffer(64)
        for i in range(self.lib.vf_op_count(self.ctx)):
            ms, fl, by, ex = ctypes.c_float(), ctypes.c_double(), ctypes.c_double(), ctypes.c_double()
            bn, bk, tm = ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
            self._ck(self.lib.vf_op_info(self.ctx, i, ctypes.byref(ms), ctypes.byref(fl), ctypes.byref(by),
                                         ctypes.byref(bn), ctypes.byref(bk), ctypes.byref(tm), buf, 64, ctypes.byref(ex)))
            recs.append({"label": buf.value.decode(), "ms": ms.value, "flops": fl.value, "bytes": by.value,
                         "exec_flops": ex.value, "bn": bn.value, "bk": bk.value, "terms": tm.value})
        return recs

    def selftest_gemm(self, n_img, rows, cin, cout, ntaps, dilation=1, terms=3):
        d, r = ctypes.c_double(), ctypes.c_double()
        self._ck(self.lib.vf_selftest_gemm(self.ctx, n_img, rows, cin, cout, ntaps, dilation, terms,
                                           ctypes.byref(d), ctypes.byref(r)))
        return d.value, r.value


# --------------------------------------------------------------------------------------------------------------
class FDomainHelper:
    """tools/pytorch/modules/fDomainHelper.py:12-152 without the sub-band (PQMF) variants: STFT analysis and ISTFT
    synthesis, window 2048 / hop 441 / hann / reflect."""

    def __init__(self, owner, window_size=2048, hop_size=441, center=True, pad_mode="reflect", window="hann",
                 freeze_parameters=True, subband=None):
        if (window_size, hop_size, center, pad_mode, window, subband) != (2048, 441, True, "reflect", "hann", None):
            raise NotImplementedError("libb200vf implements the reference geometry only (2048/441/hann/reflect)")
        self._owner = owner

    def _run(self, input, phase):
        eng = self._owner._engine()
        assert input.dim() == 3, "input: (batch_size, channels_num, segment_samples)"
        b, c, n = input.shape
        _, sp, cos, sin = eng.frontend(input.reshape(b * c, n), want_sp=True, want_phase=phase, want_mel=False)
        t = sp.shape[1]
        sp = sp.view(b, c, t, 1025)
        if phase:
            return sp, cos.view(b, c, t, 1025), sin.view(b, c, t, 1025)
        return sp

    def wav_to_spectrogram_phase(self, input, eps=1e-8):
        assert eps == 1e-8
        return self._run(input, True)

    def wav_to_spectrogram(self, input, eps=1e-8):
        assert eps == 1e-8
        return self._run(input, False)

    def istft(self, real, imag, length):
        """fDomainHelper.py:127 (torchlibrosa ISTFT.forward): real, imag [B,1,T,1025] -> [B,length]."""
        assert real.dim() == 4 and real.shape[1] == 1 and imag.shape == real.shape
        return self._owner._engine().istft(real[:, 0], imag[:, 0], int(length))

    def spectrogram_phase_to_wav(self, sps, coss, sins, length):
        """fDomainHelper.py:91-97: per channel istft(sp * cos, sp * sin) -> [B,C,length]."""
        eng = self._owner._engine()
        outs = [eng.istft((sps[:, c] * coss[:, c]).contiguous(), (sps[:, c] * sins[:, c]).contiguous(), int(length))
                for c in range(sps.size()[1])]
        return torch.stack(outs, dim=1)


class MelScale:
    """tools/pytorch/mel_scale.py:8-64.  forward(specgram[..., freq, time]) -> [..., n_mels, time] for ANY float32
    spectrogram on the model's device (a sparse-filterbank kernel reading the view's own strides)."""

    def __init__(self, owner, n_mels=128, sample_rate=44100, n_stft=1025):
        if (n_mels, sample_rate, n_stft) != (128, 44100, 1025):
            raise NotImplementedError("libb200vf implements the reference geometry only (128 mels, 44.1 kHz, 1025 bins)")
        self.n_mels, self.sample_rate = n_mels, sample_rate
        self.f_min, self.f_max = 0.0, float(sample_rate // 2)
        self.fb = melscale_fbanks(n_stft, self.f_min, self.f_max, n_mels, sample_rate)
        self._owner = owner

    def __call__(self, specgram):
        return self.forward(specgram)

    def forward(self, specgram):
        return self._owner._engine().mel(specgram)


class Vocoder:
    """Stand-in for voicefixer.Vocoder(sample_rate): __call__(mel [B,1,T,128]) -> wav [B,1,L]."""

    def __init__(self, owner, sample_rate=44100):
        assert sample_rate == 44100
        self.rate = sample_rate
        self._owner = owner

    def __call__(self, mel, cuda=False):
        return self.forward(mel)

    def forward(self, mel, cuda=False):
        assert mel.size()[-1] == 128
        assert mel.dim() == 4 and mel.shape[1] == 1
        out = self._owner._engine().vocoder(mel[:, 0])
        return out[:, None, :]


class Generator:
    """models/gsr_voicefixer.py:44-91 with the `unet` / `unet_small` analysis module: mel_orig -> {'mel': log10 mel}.
    Generator.forward is not sync-free - to_log's assert is a device->host round trip in the reference too
    (pytorch_util.py:158); VoiceFixer.restore() is the entry point without host synchronisation."""

    def __init__(self, owner):
        self._owner = owner

    def __call__(self, mel_orig):
        return self.forward(mel_orig)

    def forward(self, mel_orig):
        assert mel_orig.dim() == 4 and mel_orig.shape[1] == 1 and mel_orig.shape[-1] == 128
        eng = self._owner._engine()
        out = eng.unet_mel(mel_orig[:, 0])
        eng.check_errors()          # to_log's assert (pytorch_util.py:158)
        return {"mel": out[:, None]}


class _EngineModel:
    """nn.Module / Lightning surface the reference handlers use (load_from_checkpoint, eval, to, cuda), over one Engine."""
    _NEED = ("unet", "vocoder")

    def _init_common(self, hp, vocoder_config):
        self.hp = hp
        self.sampling_rate = hp["data"]["sampling_rate"]
        if hp["model"]["channels_in"] != 1:
            raise NotImplementedError("channels_in must be 1")
        self.voc_cfg = vocoder_config or VocoderConfig()
        self.f_helper = FDomainHelper(self, window_size=hp["model"]["window_size"], hop_size=hp["model"]["hop_size"],
                                      center=True, pad_mode=hp["model"]["pad_mode"], window=hp["model"]["window"])
        self.mel_freq_bins = hp["model"]["mel_freq_bins"]
        self.mel = MelScale(self, n_mels=self.mel_freq_bins, sample_rate=self.sampling_rate,
                            n_stft=hp["model"]["window_size"] // 2 + 1)
        self.vocoder = Vocoder(self, sample_rate=44100)
        self.downsample_ratio = 2 ** 6
        self.device = None
        self._eng: Optional[Engine] = None
        self._state: Optional[Dict[str, torch.Tensor]] = None
        self.training = False

    def _engine(self) -> Engine:
        if self._eng is None:
            raise RuntimeError("model is not on a CUDA device yet: call .to(device) (there is no CPU path)")
        if not self._eng.loaded:
            raise RuntimeError("no weights loaded: call load_state_dict / load_from_checkpoint first")
        return self._eng

    def _need(self):
        return self._NEED

    def load_state_dict(self, state_dict, strict=True, vocoder_state=None):
        """state_dict: reference names for the analysis network (generator.analysis_module.* / generator.unet.*).
        The vocoder is NOT part of what a reference Lightning checkpoint can provide in loadable form (see
        Engine.load_state): pass its tensors, converted to arch.vocoder_keys names, as `vocoder_state`, or include
        them as `vocoder.<key>` entries.  strict=True (the default) raises KeyError on missing tensors; strict=False
        is not supported - a partial network cannot run."""
        if not strict:
            raise NotImplementedError("strict=False: libb200vf cannot run a partially loaded network")
        st = {k: v for k, v in state_dict.items() if isinstance(v, torch.Tensor)}
        if vocoder_state is not None:
            st.update({(k if k.startswith("vocoder.") else "vocoder." + k): v for k, v in vocoder_state.items()})
        self._state = st
        if self._eng is not None:
            self._eng.load_state(self._state, need=self._need())
        return self

    def load_from_checkpoint(self, ckpt, map_location="cpu", vocoder_state=None):
        """Lightning-style: returns the loaded model (eval_gsr_voicefixer.py:33 discards the receiver).  `ckpt` is a
        torch.save'd dict (optionally under "state_dict"); vocoder tensors as in load_state_dict."""
        blob = torch.load(ckpt, map_location=map_location, weights_only=False)
        sd = blob["state_dict"] if isinstance(blob, dict) and "state_dict" in blob else blob
        self.load_state_dict(sd, vocoder_state=vocoder_state)
        return self

    def state_dict(self):
        return dict(self._state or {})

    def eval(self):
        self.training = False
        return self

    def train(self, mode=True):
        if mode:
            raise NotImplementedError("inference-only engine: BatchNorm is folded in eval mode")
        return self

    def to(self, device):
        device = torch.device(device)
        if device.type != "cuda":
            raise RuntimeError("voicefixer_main_b200 has no CPU path; move the model to a CUDA device")
        if self._eng is not None and self._eng.device == torch.device("cuda", device.index if device.index is not None else torch.cuda.current_device()):
            return self
        if self._eng is not None:
            self._eng.close()
        self._eng = Engine(device, self.voc_cfg)
        self.device = self._eng.device
        if self._state is not None:
            self._eng.load_state(self._state, need=self._need())
        return self

    def cuda(self, device=None):
        return self.to(torch.device("cuda", device if device is not None else torch.cuda.current_device()))

    def get_vocoder(self):
        return self.vocoder

    def get_f_helper(self):
        return self.f_helper

    def pre(self, input):
        """gsr_voicefixer.py:178-181 / ssr_unet.py:140-143: input [B,1,N] -> (sp [B,1,T,1025], mel_orig [B,1,T,128]);
        one fused front-end launch produces both."""
        assert input.dim() == 3 and input.shape[1] == 1
        mel, sp, _, _ = self._engine().frontend(input[:, 0], want_sp=True)
        return sp[:, None], mel[:, None]


class VoiceFixer(_EngineModel):
    """Drop-in for models.gsr_voicefixer.VoiceFixer on the inference path (eval mode only)."""

    def __init__(self, hp=None, channels=2, type_target="vocals", vocoder_config: Optional[VocoderConfig] = None):
        hp = hp if hp is not None else default_hparams()
        self.channels, self.type_target = channels, type_target
        sel = hp["task"]["gsr"]["gsr_model"]["voicefixer"]
        # gsr_voicefixer.py:49-53: `unet` wins over `unet_small`; both modules (models/components/unet.py and
        # unet_small.py, whose *Res1B blocks hold four ConvBlockRes like *Res4B, modules.py:112-165) have the same
        # layers and state-dict keys, so they share one plan
        if not (sel["unet"] or sel["unet_small"]):
            raise NotImplementedError("only the `unet` / `unet_small` analysis modules are built (bi_gru / dnn: "
                                      "config/vctk_base_voicefixer_unet.json:8-11 selects unet)")
        self.analysis_module_name = "unet" if sel["unet"] else "unet_small"
        self._init_common(hp, vocoder_config)
        self.generator = Generator(self)

    def forward(self, mel_orig):
        return self.generator(mel_orig)

    def __call__(self, mel_orig):
        return self.forward(mel_orig)

    # ---- batched fused path
    def restore(self, wav, out=None, unify_energy: bool = False, **pip_kwargs):
        """wav [B,N] fp32 on device -> restored [B,N]; one 60 s-or-shorter segment per row.
        unify_energy: apply amp_to_original_f (tools/utils.py:50-55) as handler() does for the SSR test sets
        (a per-call flag of vf_restore_ex: no context state is touched).

        Called with file paths - `restore(input="in.wav", output="out.wav", cuda=True, mode=0, your_vocoder_func=None)` -
        it is the pip package's file entry point (SURVEY.md 8(b); handler.restore_file)."""
        if isinstance(wav, (str, bytes)) or hasattr(wav, "__fspath__"):
            from .handler import restore_file
            return restore_file(self, wav, out if out is not None else pip_kwargs.pop("output"), **pip_kwargs)
        if pip_kwargs:
            raise TypeError(f"restore(tensor): unexpected arguments {sorted(pip_kwargs)}")
        return self._engine().restore(wav, out, unify_energy=unify_energy)

    def restore_many(self, wavs, unify_energy: bool = False, max_batch: int = 32) -> list:
        """Restore a list of 1-D clips of any lengths (each more than 1024 samples) in batched calls; returns the restored
        clips (1-D, on the model's device) in input order, each bit-identical to restore() of that clip alone.

        The clips are sorted by length and split into ceil(len / max_batch) groups of near-equal size (so the last group
        does not build a plan of an odd batch size); each group is padded to its longest clip and goes through ONE
        restore_varlen call.  Sorting keeps the padded work small: neighbours in length share a group."""
        return restore_grouped(self, wavs, max_batch,
                               lambda eng, batch, lens: eng.restore_varlen(batch, lens, unify_energy=unify_energy))

    def restore_inmem(self, wav_10k, cuda=True, mode=0, your_vocoder_func=None):
        """The pip package's in-memory entry point: 44.1 kHz samples -> restored [1, N] numpy (handler.restore_inmem)."""
        from .handler import restore_inmem
        return restore_inmem(self, wav_10k, cuda=cuda, mode=mode, your_vocoder_func=your_vocoder_func)

    def restore_host(self, wav_host: torch.Tensor, out_host: torch.Tensor):
        self._engine().restore_host(wav_host, out_host)

    def restore_pcm16(self, wav: torch.Tensor, unify_energy: bool = False) -> torch.Tensor:
        """restore() followed by the on-GPU int16 conversion of save_wave (tools/file/wav.py:22-24): [B,N] int16,
        half the device-to-host bytes of the fp32 result."""
        return self._engine().to_pcm16(self.restore(wav, unify_energy=unify_energy))

    def finalize(self, out: torch.Tensor, n_samples: int) -> torch.Tensor:
        """eval_gsr_voicefixer.py:68-72 on the vocoder output [B,1,L]: peak normalise (per clip) + trim_center -> [B,1,N]."""
        assert out.dim() == 3 and out.shape[1] == 1
        return self._engine().finalize(out[:, 0].contiguous(), n_samples)[:, None]


class SSRGenerator:
    """models/ssr_unet.py:44-54: forward(sp, noisy_wav) -> {'wav': unet(sp, wav)['wav'], 'clean': sp}."""

    def __init__(self, owner):
        self._owner = owner

    def __call__(self, sp, noisy_wav):
        return self.forward(sp, noisy_wav)

    def forward(self, sp, noisy_wav):
        assert sp.dim() == 4 and sp.shape[1] == 1 and sp.shape[-1] == 1025
        assert noisy_wav.dim() == 3 and noisy_wav.shape[1] == 1
        out = self._owner._engine().ssr_forward(sp[:, 0], noisy_wav[:, 0])
        return {"wav": out[:, None, :], "clean": sp}


class SSR_UNet(_EngineModel):
    """Drop-in for models.ssr_unet.SSR_UNet on the inference path (BASELINE config 3): pre(wav) -> (sp, mel);
    model(sp, wav)['wav'] = ISTFT(unet_v2(sp) * phase(wav)) (models/ssr_unet.py:140-155, unet_v2.py:86-148)."""
    _NEED = ("ssr",)

    def __init__(self, hp=None, channels=1, type_target="vocals", vocoder_config: Optional[VocoderConfig] = None):
        hp = hp if hp is not None else default_hparams()
        self.channels, self.type_target = channels, type_target
        self._init_common(hp, vocoder_config)
        self.generator = SSRGenerator(self)

    def forward(self, sp, noisy_wav):
        return self.generator(sp, noisy_wav)

    def __call__(self, sp, noisy_wav):
        return self.forward(sp, noisy_wav)

    def restore(self, wav: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """pre + forward fused: wav [B,N] -> denoised [B,N] (the magnitude never leaves the device plan)."""
        return self._engine().ssr_forward(None, wav, out)

    def restore_many(self, wavs, max_batch: int = 32) -> list:
        """Restore a list of 1-D clips of any lengths (each more than 1024 samples) in batched calls; returns the restored
        clips (1-D, on the model's device) in input order, each bit-identical to restore() of that clip alone.  Grouping
        as VoiceFixer.restore_many (sorted by length, near-equal groups of at most `max_batch`, one ssr_restore_varlen
        call per group).  Like restore(), no peak normalisation is applied."""
        return restore_grouped(self, wavs, max_batch, lambda eng, batch, lens: eng.ssr_restore_varlen(batch, lens))

    def restore_host(self, wav_host: torch.Tensor, out_host: torch.Tensor):
        self._engine().ssr_restore_host(wav_host, out_host)


class GSR_UNet(SSR_UNet):
    """models/gsr_unet.py: same network and forward as SSR_UNet (they differ in training targets only)."""

"""Mirror of eval_gsr_voicefixer.py (pre :19-25, refresh_model :31-35, handler :37-77) over the B200 engine.

Same signature and contract as the reference handler that evaluation_proc/eval.py:128-132 calls:
    handler(input, output, target, ckpt, device, needrefresh=False, meta={}) -> dict of metrics
It writes a 16-bit wav at `output`.  Differences, all outside the hot path: audio decoding uses the stdlib `wave`
module (librosa / soundfile are not in this image): PCM16 wav of ANY sample rate, converted to 44.1 kHz on the GPU by
the polyphase resampler (edges.py; load_wav -> librosa.load(sr=44100), tools/utils.py:46-48).  With a `target` the
per-segment mel metrics of eval_gsr_voicefixer.py:56-64 are computed on the GPU (lsd, sispec, non-log sispec; `mel-ssim`
is a CPU skimage call in the reference, evaluation_proc/metrics.py:97-106, and is not reported).
The segment loop, from_log, peak normalisation, trim_center, concat and the int16 conversion of
tools/file/wav.py:22-24 are reproduced exactly; the per-segment stages run as one fused launch chain.
"""
import wave

import numpy as np
import torch

from .model import SSR_UNet, VoiceFixer, default_hparams

model = None
hp = None
SEG_LENGTH = 44100 * 60          # eval_gsr_voicefixer.py:47


def read_pcm16(path):
    """(mono float32 samples in [-1, 1), sample rate) of a 16-bit PCM wav."""
    with wave.open(path, "rb") as w:
        if w.getsampwidth() != 2:
            raise ValueError(f"{path}: need 16-bit PCM (got {8 * w.getsampwidth()} bit)")
        rate = w.getframerate()
        data = np.frombuffer(w.readframes(w.getnframes()), dtype=np.int16).reshape(-1, w.getnchannels())
    return (data.astype(np.float32) / 32768.0).mean(axis=1).astype(np.float32), rate


def load_wav(path, sample_rate=44100, engine=None):
    """tools/utils.py:46-48 (librosa.load(path, sr=sample_rate)): decode + convert to `sample_rate`.  Rate conversion
    runs on the GPU (`engine`, edges.resample_to); a file already at the target rate needs no engine."""
    wav, rate = read_pcm16(path)
    if rate == sample_rate:
        return wav
    if engine is None:
        raise ValueError(f"{path}: {rate} Hz input needs an engine for the GPU resampler (pass engine=model._engine())")
    from .edges import resample_to
    return resample_to(engine, torch.from_numpy(wav)[None].to(engine.device), rate, sample_rate)[0].cpu().numpy()


def save_wave(frames: np.ndarray, fname, sample_rate=44100):
    """tools/file/wav.py:10-27: scale by 2^15 when max <= 1 and truncate toward zero to int16."""
    frames = np.array(frames, dtype=np.float32, copy=True).reshape(-1)
    if np.max(frames) <= 1:
        frames *= 2 ** 15
    pcm = frames.astype(np.short)
    with wave.open(fname, "wb") as w:
        w.setnchannels(1)
        w.setsampwidth(2)
        w.setframerate(sample_rate)
        w.writeframes(pcm.tobytes())


def save_pcm16(pcm: np.ndarray, fname, sample_rate=44100):
    """Write already-converted int16 samples (VoiceFixer.restore_pcm16 / Engine.to_pcm16)."""
    with wave.open(fname, "wb") as w:
        w.setnchannels(1)
        w.setsampwidth(2)
        w.setframerate(sample_rate)
        w.writeframes(np.ascontiguousarray(pcm, dtype=np.int16).reshape(-1).tobytes())


def refresh_model(ckpt):
    global model
    model = VoiceFixer(hp if hp is not None else default_hparams(), channels=2, type_target="vocals").load_from_checkpoint(ckpt)
    model.eval()


def restore_array(mdl: VoiceFixer, wav_10k: np.ndarray, device, unify_energy: bool = False, target: np.ndarray = None,
                  metrics: dict = None) -> torch.Tensor:
    """The segment loop of handler() for one in-memory file: returns [1, N] on `device`.  With `target` (the clean
    signal, same rate) the mel metrics of the LAST segment land in `metrics`, as the reference's loop leaves them
    (eval_gsr_voicefixer.py:56-64 overwrites the dict every segment)."""
    res = []
    break_point = SEG_LENGTH
    n = wav_10k.shape[0]
    while break_point < n + SEG_LENGTH:
        segment = wav_10k[break_point - SEG_LENGTH:break_point]
        seg = torch.from_numpy(np.ascontiguousarray(segment))[None, :].to(device)
        res.append(mdl.restore(seg, unify_energy=unify_energy))
        if target is not None and metrics is not None:
            from .edges import AudioMetrics
            am = AudioMetrics(mdl)
            eng = mdl._engine()
            tseg = torch.from_numpy(np.ascontiguousarray(target[break_point - SEG_LENGTH:break_point]))[None, None, :].to(device)
            _, target_mel = mdl.pre(tseg)
            mel_noisy, log_mel = eng.restore_stages(1, seg.shape[1])
            log_mel, mel_noisy = log_mel[:, None], mel_noisy[:, None]
            denoised = eng.from_log(log_mel)
            if unify_energy:                     # eval_gsr_voicefixer.py:54-55 (tools/utils.py:50-55) before the lsd
                denoised = eng.amp_to_original_f(denoised[:, 0].contiguous(), mel_noisy[:, 0].contiguous())[:, None]
            metrics.update({
                "mel-lsd": float(am.lsd(denoised.contiguous(), target_mel.contiguous())),
                "mel-sispec": float(am.sispec(log_mel, target_mel.contiguous(), target_map=1)),             # in log scale
                "mel-non-log-sispec": float(am.sispec(log_mel, target_mel.contiguous(), est_map=2)),
            })
        break_point += SEG_LENGTH
    return torch.cat(res, -1)


def handler(input, output, target, ckpt, device, needrefresh=False, meta={}):
    if needrefresh:
        refresh_model(ckpt)
    global model
    model = model.to(device)
    metrics = {}
    wav_10k = load_wav(input, sample_rate=44100, engine=model._engine())
    tgt = load_wav(target, sample_rate=44100, engine=model._engine()) if target is not None else None
    out = restore_array(model, wav_10k, model.device, unify_energy=bool(meta.get("unify_energy", False)), target=tgt, metrics=metrics)
    # save_wave's float -> int16 conversion runs on the GPU (its `max <= 1` condition always holds after the
    # per-segment peak normalisation), so only 2 bytes per sample cross PCIe.  meta["saturate"] (not in the reference)
    # clamps instead of reproducing numpy's +1.0 -> -32768 wrap, see INTEGRATION.md
    pcm = model._engine().to_pcm16(out[0], saturate=bool(meta.get("saturate", False)))
    save_pcm16(pcm.cpu().numpy(), fname=output, sample_rate=44100)
    return metrics


def restore_files(mdl, inputs, outputs, meta={}, max_batch=32):
    """handler() over many files at once: each output file is byte-identical to handler(input, output, None, ...) with the
    same meta ("unify_energy", "saturate"), but the 60 s segments of ALL files are pooled into batched calls
    (VoiceFixer.restore_many: sorted by length, groups of at most `max_batch`).  Files are read like handler() reads them
    (load_wav, any sample rate through the GPU resampler).  No target metrics: use handler() for those.

    `mdl` may also be an SSR_UNet / GSR_UNet.  Each file then gets the bytes the GSR-UNet handler (eval_gsr_unet.py:37-75)
    writes with this model: 60 s segments, each restored (SSR_UNet.restore_many) and peak-normalised on its own when
    max|x| > 1, no trim (the ISTFT returns the input length), concatenated, then save_wave's int16 cast.
    meta["saturate"] is honoured; meta["unify_energy"] is ignored, as that handler never reads meta."""
    inputs, outputs = list(inputs), list(outputs)
    if len(inputs) != len(outputs):
        raise ValueError(f"restore_files: {len(inputs)} inputs but {len(outputs)} outputs")
    eng = mdl._engine()
    segs, owner = [], []
    for k, path in enumerate(inputs):
        wav = load_wav(path, sample_rate=44100, engine=eng)
        for seg in split_segments(wav.shape[0]):
            segs.append(torch.from_numpy(np.ascontiguousarray(wav[seg])))
            owner.append(k)
    if isinstance(mdl, SSR_UNet):
        res = mdl.restore_many(segs, max_batch=max_batch)
        # eval_gsr_unet.py:66-67: the segment divided by its peak when that exceeds 1 (trim_center :70 keeps n samples)
        res = [eng.finalize(out[None], out.shape[0])[0] for out in res]
    else:
        res = mdl.restore_many(segs, unify_energy=bool(meta.get("unify_energy", False)), max_batch=max_batch)
    pieces = [[] for _ in inputs]
    for k, out in zip(owner, res):
        pieces[k].append(out)
    for k, path in enumerate(outputs):
        out = torch.cat(pieces[k], -1)
        pcm = eng.to_pcm16(out, saturate=bool(meta.get("saturate", False)))
        save_pcm16(pcm.cpu().numpy(), fname=path, sample_rate=44100)


def split_segments(n):
    """The segments of handler()'s loop (eval_gsr_voicefixer.py:47-50) over n samples, as slices: 60 s each, the last
    one ragged."""
    out = []
    break_point = SEG_LENGTH
    while break_point < n + SEG_LENGTH:
        out.append(slice(break_point - SEG_LENGTH, min(break_point, n)))
        break_point += SEG_LENGTH
    return out


# ---- the pip package's entry points (SURVEY.md 8(b): `VoiceFixer.restore(input, output, cuda, mode, your_vocoder_func)` /
# `restore_inmem(wav_10k, cuda, mode, your_vocoder_func)`; the package is not in /root/reference - the signatures and the
# 30 s segmentation follow the survey's description of it, mode 0 is the parity target)
PIP_SEG_LENGTH = 44100 * 30


def restore_inmem(mdl: VoiceFixer, wav_10k, cuda=True, mode=0, your_vocoder_func=None, unify_energy=True) -> np.ndarray:
    """One in-memory 44.1 kHz file -> restored samples [1, N] (numpy), 30 s segments, each
    pre -> analysis module -> from_log -> amp_to_original_f -> vocoder -> trim, concatenated.

    All whole segments of the file go through ONE batched restore call (the segments are independent), the ragged last
    one through a second.  cuda=False raises (there is no CPU path); mode 1 (pre low-pass) and mode 2 (train-mode
    BatchNorm) are not built.  `your_vocoder_func(mel [B,1,T,128] linear) -> wav [B,1,L]` replaces stage C; the stages
    then run one by one through the object protocol."""
    if not cuda:
        raise RuntimeError("restore_inmem: cuda=False is not available (there is no CPU path)")
    if mode != 0:
        raise NotImplementedError(f"restore_inmem: mode {mode} is not built (mode 0 only)")
    if mdl.device is None:
        raise RuntimeError("model is not on a CUDA device yet: call .to(device)")
    wav = torch.as_tensor(np.ascontiguousarray(wav_10k, dtype=np.float32)).reshape(-1)
    n = wav.shape[0]
    if n == 0:
        return np.zeros((1, 0), np.float32)
    n_full = n // PIP_SEG_LENGTH
    dev = wav.to(mdl.device)
    res = []

    def run(x):                                  # x [B, n_seg] on the device
        if your_vocoder_func is None:
            return mdl.restore(x, unify_energy=unify_energy)
        eng = mdl._engine()
        _, mel_noisy = mdl.pre(x[:, None])
        denoised = eng.from_log(mdl(mel_noisy)["mel"])
        if unify_energy:
            denoised = eng.amp_to_original_f(denoised[:, 0].contiguous(), mel_noisy[:, 0].contiguous())[:, None]
        out = your_vocoder_func(denoised)
        return mdl.finalize(out.to(mdl.device, torch.float32).contiguous(), x.shape[1])[:, 0]

    if n_full:
        res.append(run(dev[:n_full * PIP_SEG_LENGTH].view(n_full, PIP_SEG_LENGTH)).reshape(1, -1))
    if n > n_full * PIP_SEG_LENGTH:
        res.append(run(dev[None, n_full * PIP_SEG_LENGTH:].contiguous()))
    return torch.cat(res, -1).cpu().numpy()


def restore_file(mdl: VoiceFixer, input, output, cuda=True, mode=0, your_vocoder_func=None):
    """The package's `restore(input, output, cuda, mode, your_vocoder_func)`: wav file in, 16-bit 44.1 kHz wav out."""
    if not cuda:
        raise RuntimeError("restore: cuda=False is not available (there is no CPU path)")
    if mdl.device is None:
        raise RuntimeError("model is not on a CUDA device yet: call .to(device)")
    wav_10k = load_wav(input, sample_rate=44100, engine=mdl._engine())
    out = restore_inmem(mdl, wav_10k, cuda=cuda, mode=mode, your_vocoder_func=your_vocoder_func)
    save_wave(out, fname=output, sample_rate=44100)

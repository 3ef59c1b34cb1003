"""CPU-side tests of the host layer: C-ABI library loads and exports every declared symbol, the mirror
objects behave like the reference's, and the product refuses to run without CUDA (no fallback)."""
import os
import re

import pytest
import torch

from conftest import ROOT, load_golden


def test_library_exports_every_declared_symbol():
    from voicefixer_main_b200 import _lib
    lib = _lib.load_library()
    header = open(os.path.join(ROOT, "include", "b200vf.h")).read()
    declared = re.findall(r"VF_API\s+[\w\s\*]+?\b(vf_\w+)\s*\(", header)
    assert len(declared) >= 20
    assert sorted(declared) == sorted(_lib.EXPORTS)
    for name in declared:
        assert hasattr(lib, name), name


def test_no_cpu_fallback():
    from voicefixer_main_b200 import VoiceFixer
    from voicefixer_main_b200._lib import EngineError
    m = VoiceFixer()
    with pytest.raises(RuntimeError):
        m.to("cpu")
    with pytest.raises(RuntimeError):
        m.restore(torch.zeros(1, 4410))
    if not torch.cuda.is_available():
        with pytest.raises((EngineError, RuntimeError)):
            m.to("cuda:0")


def test_product_does_not_import_oracle():
    pkg = os.path.join(ROOT, "voicefixer_main_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".cpp", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert "import oracle" not in src and "from oracle" not in src, f


def test_hparams_and_filterbank_mirror_reference_semantics(tmp_path):
    from voicefixer_main_b200.model import HParams, get_hparams_from_file, melscale_fbanks
    from oracle import vf_oracle as O
    p = tmp_path / "c.json"
    p.write_text('{"model": {"window_size": 2048, "hop_size": 441}, "data": {"sampling_rate": 44100}}')
    hp = get_hparams_from_file(str(p))
    assert hp["model"]["hop_size"] == 441 and hp.model.window_size == 2048 and "data" in hp and len(hp) == 2
    assert isinstance(hp.model, HParams)
    assert torch.equal(melscale_fbanks(), O.mel_filterbank())


def test_unsupported_configs_fail_loudly():
    from voicefixer_main_b200 import VoiceFixer, default_hparams
    hp = default_hparams()
    hp["task"]["gsr"]["gsr_model"]["voicefixer"]["unet"] = False
    with pytest.raises(NotImplementedError):
        VoiceFixer(hp)
    hp = default_hparams()
    hp["model"]["window_size"] = 1024
    with pytest.raises(NotImplementedError):
        VoiceFixer(hp)


def test_arch_keys_match_reference_state_dict():
    """Against the UNet keys and shapes of the reference model's state_dict, in registration order (stored by
    python oracle/make_golden.py reference)."""
    from voicefixer_main_b200.arch import UNET_PREFIX, unet_keys
    g = load_golden("reference_oracle.npz")
    own = {UNET_PREFIX + str(k): tuple(s[:d]) for k, s, d in zip(g["unet_keys"], g["unet_shapes"].tolist(), g["unet_ndims"])}
    mine = {UNET_PREFIX + k: tuple(s) for k, s in unet_keys()}
    assert own == mine
    assert list(own) == list(mine)          # same registration order
    assert sum(int(torch.tensor(s).prod()) if s else 1 for k, s in mine.items()
               if not k.endswith("num_batches_tracked") and "running" not in k) == 65152867


def test_plain_mappings_work_as_hp_and_unet_small_is_accepted():
    """`hp` is any mapping with the reference's keys (a plain dict here); `unet_small: true` selects the same network
    (gsr_voicefixer.py:51-53, models/components/unet_small.py) and `unet` wins when both are set (:49)."""
    from voicefixer_main_b200 import SSR_UNet, VoiceFixer
    hp = {"task": {"gsr": {"gsr_model": {"voicefixer": {"unet": False, "unet_small": True, "bi_gru": False, "dnn": False}}}},
          "data": {"sampling_rate": 44100},
          "model": {"mel_freq_bins": 128, "window_size": 2048, "hop_size": 441, "pad_mode": "reflect", "window": "hann", "channels_in": 1}}
    assert VoiceFixer(hp).analysis_module_name == "unet_small"
    hp["task"]["gsr"]["gsr_model"]["voicefixer"]["unet"] = True
    assert VoiceFixer(hp).analysis_module_name == "unet"
    s = SSR_UNet(hp)
    assert s.generator is not None and s.downsample_ratio == 64


def test_checkpoint_loading_is_explicit_about_the_vocoder(tmp_path):
    """ADVICE r1: a reference Lightning checkpoint cannot supply the pip package's vocoder in loadable form; the mirror says
    so instead of claiming drop-in loading, takes it as `vocoder_state`, and refuses strict=False."""
    from voicefixer_main_b200 import VoiceFixer
    from voicefixer_main_b200.model import Engine
    from voicefixer_main_b200.weights import make_unet_state, make_vocoder_state
    unet, voc = make_unet_state(1), make_vocoder_state(seed=2)
    m = VoiceFixer()
    with pytest.raises(NotImplementedError):
        m.load_state_dict(unet, strict=False)
    ck = tmp_path / "ckpt.pt"
    torch.save({"state_dict": unet}, ck)
    m.load_from_checkpoint(str(ck), vocoder_state={k[len("vocoder."):]: v for k, v in voc.items()})   # bare arch.vocoder_keys names
    assert all(k in m.state_dict() for k in voc)
    # without the vocoder tensors the engine-side loader names what is missing and where it comes from
    eng = Engine.__new__(Engine)
    eng.voc_cfg = m.voc_cfg
    with pytest.raises(KeyError, match="vocoder"):
        Engine.load_state(eng, unet)


def test_resampler_filter_design_matches_scipy_firwin():
    """edges.design_filter restates scipy.signal.resample_poly's default FIR; the kernel's index formula
    out[m] = sum_i h[m*down - i*up + half] x[i] is resample_poly's (zero-phase upfirdn with its pre-padding folded in)."""
    import numpy as np
    from scipy.signal import firwin, resample_poly
    from voicefixer_main_b200.edges import design_filter
    rng = np.random.default_rng(0)
    for up, down in ((147, 160), (441, 160), (441, 80), (2, 1), (147, 320)):
        mr = max(up, down)
        half = 10 * mr
        ref = firwin(2 * half + 1, 1.0 / mr, window=("kaiser", 5.0)) * up
        h = design_filter(up, down)
        assert h.dtype == np.float32 and h.shape == ref.shape
        assert float(np.abs(h - ref).max()) < 1e-6 * float(np.abs(ref).max())
        x = rng.standard_normal(3001)
        y = resample_poly(x, up, down)
        n_out = -(-len(x) * up // down)
        assert len(y) == n_out
        for m in range(0, n_out, max(1, n_out // 40)):
            c = m * down
            i = np.arange(max(0, -(-(c - half) // up)), min(len(x) - 1, (c + half) // up) + 1)
            assert abs(float(np.sum(ref[c - i * up + half] * x[i])) - y[m]) < 1e-9


def test_pip_entry_points_refuse_what_is_not_built():
    """SURVEY.md 8(b): signature-compatible restore / restore_inmem wrappers; no CPU path, mode 0 only."""
    import numpy as np
    from voicefixer_main_b200 import VoiceFixer
    m = VoiceFixer()
    with pytest.raises(RuntimeError, match="no CPU path"):
        m.restore_inmem(np.zeros(100, np.float32), cuda=False, mode=0)
    with pytest.raises(NotImplementedError):
        m.restore_inmem(np.zeros(100, np.float32), cuda=True, mode=1)
    with pytest.raises(RuntimeError, match="no CPU path"):
        m.restore("in.wav", "out.wav", cuda=False, mode=0)
    with pytest.raises(RuntimeError):                        # not on a device yet
        m.restore("in.wav", "out.wav")


def test_ar_residual_stream_arithmetic_keeps_22_bits():
    """DESIGN.md section 5: the hi-only vocoder keeps its residual stream as a = fp16(lrelu_s(x)) and r = fp16(x - U(a)),
    U(a) = min(a, a * fp16(1/s)) evaluated in fp16 (csrc/ptx.cuh ar_unact / ar_split).  Restated in numpy: U(a) + r recovers
    x to ~2^-21 relative - the precision of a hi/lo split of x itself - for every slope the engine accepts."""
    import numpy as np
    rng = np.random.default_rng(5)
    x = np.concatenate([rng.standard_normal(200000) * 3.0, rng.standard_normal(1000) * 1e-4, [0.0, -0.0, 65000.0, -65000.0]]).astype(np.float32)
    for s in (0.1, 0.2, 0.01, 1.0):
        inv = np.float16(1.0 / s)
        a = np.maximum(x, x * np.float32(s)).astype(np.float16)                      # fmaxf(v, v * slope) -> fp16
        with np.errstate(over="ignore"):                                              # a * inv may overflow to +inf: min() keeps a
            u = np.minimum(a, (a * inv).astype(np.float16))                          # __hmin2(a, __hmul2(a, inv))
        r = (x - u.astype(np.float32)).astype(np.float16)                            # FHADD + pack
        back = u.astype(np.float32) + r.astype(np.float32)
        hi = x.astype(np.float16)
        lo = (x - hi.astype(np.float32)).astype(np.float16)
        err_ar = np.abs(back - x)
        err_hl = np.abs(hi.astype(np.float32) + lo.astype(np.float32) - x)
        bound = np.abs(x) * 2.0 ** -20 + 2.0 ** -24                                  # fp16 subnormal floor for tiny values
        assert np.all(np.isfinite(back)) and np.all(err_ar <= bound), (s, float((err_ar / np.maximum(np.abs(x), 1e-30)).max()))
        assert float(err_ar.max()) <= 4.0 * float(err_hl.max()) + 2.0 ** -24


def test_restore_inmem_segmentation_with_a_stub_model(tmp_path):
    """handler.restore_inmem: all whole 30 s segments go through ONE batched call, the ragged tail through a second, and
    the pieces come back in order (host logic only: the model is a stub that scales its input)."""
    import numpy as np
    from voicefixer_main_b200 import handler as H

    class Stub:
        device = torch.device("cpu")
        calls = []

        def restore(self, x, unify_energy=False):
            self.calls.append((tuple(x.shape), unify_energy))
            return x * 0.5

    seg = H.PIP_SEG_LENGTH
    for n in (seg // 3, seg, 2 * seg + 777):
        m = Stub()
        m.calls = []
        wav = np.arange(n, dtype=np.float32) / n
        out = H.restore_inmem(m, wav, cuda=True, mode=0)
        assert out.shape == (1, n) and np.array_equal(out[0], wav * 0.5)
        want = ([((n // seg, seg), True)] if n >= seg else []) + ([((1, n % seg), True)] if n % seg else [])
        assert m.calls == want
    assert H.restore_inmem(Stub(), np.zeros(0, np.float32)).shape == (1, 0)

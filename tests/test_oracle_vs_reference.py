"""Pin the restatement in oracle/vf_oracle.py against the reference's own modules.  tests/golden/reference_oracle.npz
holds what those modules, imported unmodified, returned for the inputs built below (python oracle/make_golden.py
reference); large outputs are stored as out.reshape(-1)[::stride]."""
import pytest
import torch

from conftest import load_golden
from oracle import vf_oracle as O


@pytest.fixture(scope="module")
def ref(golden_fingerprint_ok):
    g = load_golden("reference_oracle.npz")
    assert (g["fingerprint"] == load_golden("stage_b_t101.npz")["fingerprint"]).all()
    return g


def _sampled(ref, x):
    return x.reshape(-1)[::int(ref["stride"])]


def test_mel_filterbank_bit_identical(ref):
    fb = O.mel_filterbank()
    want = torch.zeros(tuple(ref["fb_shape"]))
    want.view(-1)[torch.from_numpy(ref["fb_index"]).long()] = torch.from_numpy(ref["fb_value"])
    assert torch.equal(want, fb)
    assert int((fb != 0).sum()) == 2018            # SURVEY.md 8(a) a5 probe


def test_log_helpers_match_reference(ref):
    g = torch.Generator().manual_seed(23)
    x = torch.rand(3, 1, 7, 128, generator=g) * 3
    x[0, 0, 0, :4] = 0
    y = torch.randn(3, 1, 7, 128, generator=g) * 4
    assert torch.equal(torch.from_numpy(ref["to_log"]), O.to_log(x))
    assert torch.equal(torch.from_numpy(ref["from_log"]), O.from_log(y))
    assert bool(ref["to_log_rejects_negative"])
    with pytest.raises(AssertionError):
        O.to_log(-x - 1)


def test_unet_restatement_matches_reference(ref, state):
    g = torch.Generator().manual_seed(3)
    for t in (64, 101, 130):                          # multiple of 64, the reference smoke shape, ragged
        mel = 10 ** (torch.randn(2, 1, t, 128, generator=g) - 1)
        with torch.no_grad():
            mine = O.generator_forward(state, mel)
        assert mine.shape == (2, 1, t, 128)
        assert float((torch.from_numpy(ref[f"unet_t{t}"]) - _sampled(ref, mine)).abs().max()) < 2e-5


def test_handler_restatement_matches_reference(ref, state):
    wav = O.synth_clips(2, 30000, seed=9)
    with torch.no_grad():
        mine = O.restore(state, wav, seg_samples=12000)        # 3 segments, last ragged
    assert mine.shape == wav.shape
    assert float((torch.from_numpy(ref["handler"]) - _sampled(ref, mine)).abs().max()) < 1e-5


def test_trim_center_matches_reference(ref):
    for le, lr, start in ref["trim_center"].tolist():
        est = torch.arange(float(le))[None, None]
        assert torch.equal(O.trim_center(est, lr), est[..., start:start + lr])


def test_unet_v2_ssr_restatement_matches_reference(ref, state):
    """Next path (SURVEY.md 8(f) row 1): models/components/unet_v2.py imported unmodified vs the restatement."""
    from voicefixer_main_b200.arch import UNET_PREFIX
    ssr = {k.replace(UNET_PREFIX, "generator.unet."): v for k, v in state.items() if k.startswith(UNET_PREFIX)}
    for n in (63 * 441, 70 * 441 + 17):                   # T = 64 (no time padding) and T = 71 -> T' = 128
        wav = O.synth_clips(1, n, seed=n)[:, None, :]
        with torch.no_grad():
            mine = O.ssr_forward(ssr, wav)
        assert mine.shape == (1, 1, n)
        assert float((torch.from_numpy(ref[f"ssr_n{n}"]) - _sampled(ref, mine)).abs().max()) < 1e-5


def test_unet_small_is_the_same_network(ref, state):
    """SURVEY.md 8(f) row 4: models/components/unet_small.py imported unmodified.  In this reference its *Res1B blocks
    hold four ConvBlockRes each (modules.py:112-165), i.e. the layers and keys of unet.py: the product maps
    `unet_small: true` onto the same plan, which the reference's outputs (`small` vs `small_full`, the same mel through
    both modules) justify bit for bit."""
    g = torch.Generator().manual_seed(4)
    mel = 10 ** (torch.randn(1, 1, 101, 128, generator=g) - 1)
    a, b = torch.from_numpy(ref["small"]), torch.from_numpy(ref["small_full"])
    with torch.no_grad():
        c = O.generator_forward(state, mel)
    assert torch.equal(a, b)
    assert float((a - _sampled(ref, c)).abs().max()) < 2e-5

"""CPU: the conditioning front-end oracle (oracle/conditioning.py) pinned against the unmodified reference modules
(their results are stored in tests/golden/reference_v1.pt, see tests/ref_golden.py) and, for the librosa mel basis the
image cannot provide, against torchaudio's independent implementation of the same Slaney formula."""
import numpy as np
import pytest
import torch

import ref_golden as rg
from oracle import conditioning as oc


def test_mel_filterbanks_vs_torchaudio():
    import torchaudio.functional as AF
    for scale, (sr, nm, fmax) in (("slaney", (24000, 100, 12000.0)), ("htk", (22050, 80, 8000.0)), ("slaney", (22050, 80, 8000.0))):
        mine = oc.mel_filterbank(sr, 1024, nm, 0.0, fmax, scale)
        ta = AF.melscale_fbanks(513, 0.0, fmax, nm, sr, norm="slaney", mel_scale=scale).t().double().numpy()
        assert np.abs(mine - ta).max() < 2e-6 * max(1.0, np.abs(ta).max()), scale
    # known values of librosa.filters.mel(sr=22050, n_fft=1024, n_mels=80, fmin=0, fmax=8000) (public docs / tacotron2 hparams)
    fb = oc.mel_filterbank(22050, 1024, 80, 0.0, 8000.0, "slaney")
    assert fb.shape == (80, 513) and fb[0, 0] == 0.0 and fb.min() >= 0.0
    assert abs(fb[0].sum() * (22050 / 1024) - 1.0) < 0.35      # Slaney normalisation: ~unit area per filter


@pytest.fixture(scope="module")
def ref():
    if rg.RECORD:
        from oracle.ref_shims import load_reference
        import sys
        load_reference()
        # librosa is absent: give the reference's TacotronSTFT the restated Slaney basis (pinned above)
        sys.modules["librosa.filters"].mel = lambda sr, n_fft, n_mels, fmin, fmax: oc.mel_filterbank(sr, n_fft, n_mels, fmin, fmax, "slaney").astype(np.float32)
        sys.modules["librosa.util"].pad_center = lambda data, size=None, **k: data
        if "scipy.signal" not in sys.modules:
            import scipy.signal  # noqa: F401  (stft.py: get_window)
    from tortoise_tts_b200.config import ModelConfig
    from tortoise_tts_b200.synth import synth_all
    cfg = ModelConfig.small()
    return cfg, synth_all(cfg, seed=0, suppress_stop=False)


def _clips(n=2):
    g = torch.Generator().manual_seed(5)
    return [(torch.randn(1, L, generator=g) * 0.2).clamp(-1, 1) for L in (140000, 90000)][:n]


def test_ar_mel_and_encoder(ref):
    cfg, sds = ref

    def reference_mel():
        from tortoise.models.arch_util import TorchMelSpectrogram
        tm = TorchMelSpectrogram()
        return tm(clip.unsqueeze(0)).squeeze(0) if clip.dim() == 2 else tm(clip)

    def reference_encoder():
        # reduced configs carry fewer attention blocks than the reference module builds: compare block by block
        from oracle.ref_build import build_reference_models
        enc = build_reference_models(cfg, sds)["autoregressive"].conditioning_encoder
        h = enc.init(got)
        for i in range(cfg.cond_enc_blocks):
            h = enc.attn[i](h)
        return h[:, :, 0]
    from tortoise_tts_b200.api import _default_mel_norms       # the packaged copy of tortoise/data/mel_norms.pth
    clip = oc.format_conditioning_clip(_clips()[0], 17)
    got = oc.torch_mel_spectrogram(clip, _default_mel_norms())
    idx, want, shape = rg.sampled("ar_conditioning_mel", reference_mel)
    assert got.shape == (1, 80, 517) and shape.numel() == got.numel()
    assert (got.reshape(-1)[idx] - want).abs().max() < 1e-5
    sd = sds["autoregressive"]
    with torch.no_grad():
        mine = oc.conditioning_encoder(sd, cfg, got)
        want = rg.value("ar_conditioning_encoder", reference_encoder)
    assert (mine - want).abs().max() < 2e-4


def test_diffusion_mel_and_embedder(ref):
    cfg, sds = ref
    clips = _clips()

    def reference_mels():
        from tortoise.utils.audio import TacotronSTFT, wav_to_univnet_mel
        import torchaudio
        from tortoise.api import pad_or_truncate
        stft = TacotronSTFT(1024, 256, 1024, 100, 24000, 0, 12000)
        mels_ref = []
        for c in clips:
            s = pad_or_truncate(torchaudio.functional.resample(c, 22050, 24000), 102400)
            mels_ref.append(wav_to_univnet_mel(s, do_normalization=False, device="cpu", stft=stft))
        return mels_ref

    def reference_latent():
        from oracle.ref_build import build_reference_models
        return build_reference_models(cfg, sds)["diffusion"].get_conditioning(torch.stack(reference_mels(), dim=1))
    s0 = oc.resample_22k_24k(clips[0])
    s0 = s0[..., :oc.DIFF_COND_LENGTH] if s0.shape[-1] >= oc.DIFF_COND_LENGTH else torch.nn.functional.pad(s0, (0, oc.DIFF_COND_LENGTH - s0.shape[-1]))
    m0 = oc.tacotron_mel(s0)
    assert m0.shape == (1, 100, 401)
    idx, want, shape = rg.sampled("diffusion_conditioning_mel", lambda: reference_mels()[0])
    assert shape == m0.shape
    assert (m0.reshape(-1)[idx] - want).abs().max() < 2e-4
    with torch.no_grad():
        want = rg.value("diffusion_conditioning_latent", reference_latent)
        got = oc.diffusion_conditioning_latent(sds["diffusion"], cfg, clips)
    assert got.shape == want.shape == (1, 2 * cfg.diff_dim)
    assert (got - want).abs().max() < 2e-4


def test_random_latent(ref):
    from tortoise_tts_b200.synth import synth_rlg
    C = 64
    sd = synth_rlg(C, 0)

    def reference():
        from tortoise.models.random_latent_generator import RandomLatentConverter
        m = RandomLatentConverter(C).eval()
        m.load_state_dict(sd)
        torch.manual_seed(3)
        with torch.no_grad():
            return m(torch.tensor([0.0]))
    want = rg.value("random_latent", reference)
    torch.manual_seed(3)
    r = torch.randn(1, C)
    assert (oc.random_latent(sd, r) - want).abs().max() < 1e-5

"""Pins oracle/net_oracle.py + oracle/separator_oracle.py against golden tensors produced by the
UNMODIFIED reference (oracle/make_golden.py)."""
import numpy as np
import torch

from conftest import checksum
from oracle import net_oracle, separator_oracle, stft_oracle
from lib import synth


def _first_window(seconds=10.0, n_fft=2048, hop=1024, cropsize=256):
    X = stft_oracle.wave_to_spectrogram(synth.sine_mix(seconds), hop, n_fft)
    pad_l, pad_r, roi = separator_oracle.make_padding(X.shape[2], cropsize, 64)
    Xp = np.pad(X, ((0, 0), (0, 0), (pad_l, pad_r)))
    Xp /= np.abs(X).max()
    return X, np.abs(Xp[None, :, :, roi:roi + cropsize])


def test_make_padding():
    assert separator_oracle.make_padding(431, 256, 64) == (64, 128 - 431 % 128 + 64, 128)
    assert separator_oracle.make_padding(256, 256, 64) == (64, 128 + 64, 128)
    assert separator_oracle.make_padding(100, 128, 64) == (64, 128 - 100 + 64, 128)  # roi==0 -> cropsize


def test_state_dict_spec_counts():
    spec = synth.state_dict_spec()
    assert len(spec) == 689
    n_param = sum(int(np.prod(s)) for k, s, kind in spec if not kind.startswith('bn_mean')
                  and kind not in ('bn_var', 'bn_count'))
    assert n_param == 14740882  # SURVEY App. C


def test_first_window_stages_match_reference_golden(golden_default):
    g = golden_default
    sd = synth.to_torch_state_dict(synth.make_state_dict())
    _, x0 = _first_window()
    mask, st = net_oracle.forward(sd, torch.from_numpy(x0), return_stages=True)
    assert np.abs(mask.numpy()[:, :, ::8, :] - g['win1_mask_sub']).max() < 2e-5
    for k in ('l1', 'h1', 'l2', 'h2', 'f3', 'logit'):
        a = st[k].numpy()
        ref = g['win1_' + k + '_sub']
        assert np.abs(a[:, :, ::16, ::4] - ref).max() < 1e-4 * max(1.0, np.abs(ref).max()), k


def test_separate_matches_reference_golden(golden_default):
    g = golden_default
    sd = synth.to_torch_state_dict(synth.make_state_dict())
    X, _ = _first_window()
    mask = separator_oracle.separate_mask(sd, X)
    assert mask.shape == (2, 1025, 431) and mask.dtype == np.float32
    assert np.abs(mask[:, ::8, :] - g['mask_sub']).max() < 2e-5
    assert np.allclose(checksum(mask), g['mask_sum'], rtol=1e-5)
    y, v = separator_oracle.apply_mask(X, mask)
    assert np.abs(y[:, ::16, :] - g['y_sub']).max() < 1e-4 * g['absmax']
    wy = stft_oracle.spectrogram_to_wave(y.astype(np.complex64), 1024)
    assert np.abs(wy[:, ::16] - g['wave_inst_sub']).max() < 1e-5


def test_separate_tta_matches_reference_golden(golden_default):
    g = golden_default
    sd = synth.to_torch_state_dict(synth.make_state_dict())
    X, _ = _first_window()
    mask = separator_oracle.separate_tta_mask(sd, X)
    assert np.abs(mask[:, ::8, :] - g['mask_tta_sub']).max() < 2e-5


def test_small_config_matches_reference_golden(golden_small):
    g = golden_small
    sd = synth.to_torch_state_dict(synth.make_state_dict(512, 16, 32))
    X = stft_oracle.wave_to_spectrogram(synth.sine_mix(3.0), 256, 512)
    mask = separator_oracle.separate_mask(sd, X, n_fft=512, cropsize=192, batchsize=2)
    assert np.abs(mask[:, ::2, :] - g['mask_sub']).max() < 2e-5


def test_predict_mask_matches_reference_golden(golden_functions):
    g = golden_functions
    sd = synth.to_torch_state_dict(synth.make_state_dict())
    _, x0 = _first_window()
    got = net_oracle.predict_mask(sd, torch.from_numpy(x0)).numpy()
    assert got.shape == (1, 2, 1025, 128)
    assert np.abs(got[:, :, 4::8, :] - g['predict_mask_sub']).max() < 1e-5
    assert np.allclose(checksum(got), g['predict_mask_sum'], rtol=1e-5)

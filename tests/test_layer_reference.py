"""Calibrates the per-layer gates of tests/test_gpu_layers.py on the CPU.

* The float64 single-layer references (tests/layer_reference.py), chained on their own outputs, reproduce the
  reference model's first-window stage activations (golden fixture of the unmodified reference).
* On three layer classes, a CPU emulation of the tensor-core arithmetic (split-bf16 activations, three bf16 products
  with fp32 accumulation: the '3pass' scheme of tests/precision_budget.py) passes GATE_CONV with margin, while the
  same arithmetic with one correction product dropped, or with one 128-pixel output tile left unwritten, fails it.
* An fp32 LSTM recurrence passes GATE_LSTM against the float64 one; the same recurrence with its reverse direction
  started one step late fails it.
So the gates are neither tighter than the kernels' arithmetic nor blind to a fault confined to part of a layer.
"""
import numpy as np
import pytest
import torch

import layer_reference as lr
import precision_budget
from lib import synth
from oracle import separator_oracle, stft_oracle


@pytest.fixture(scope='module')
def sd64():
    return lr.state_dict64(synth.make_state_dict())


@pytest.fixture(scope='module')
def sd32():
    return synth.to_torch_state_dict(synth.make_state_dict())


def test_chained_reference_reproduces_golden_stages(sd64, golden_default):
    X = stft_oracle.wave_to_spectrogram(synth.sine_mix(10.0), 1024, 2048)
    pad_l, pad_r, roi = separator_oracle.make_padding(X.shape[2], 256, 64)
    Xp = np.pad(X, ((0, 0), (0, 0), (pad_l, pad_r))) / np.abs(X).max()
    x = torch.from_numpy(np.abs(Xp[None, :, :, roi:roi + 256]).astype(np.float32)).double()
    with torch.no_grad():
        st = lr.forward_stages(sd64, x)
    for k in ('l1', 'h1', 'l2', 'h2', 'f3'):
        ref = golden_default['win1_%s_sub' % k]
        got = st[k].numpy()[:, :, ::16, ::4]
        assert np.abs(got - ref).max() < 1e-4 * max(1.0, np.abs(ref).max()), k
    assert np.abs(st['mask'].numpy()[:, :, ::8, :] - golden_default['win1_mask_sub']).max() < 2e-5


def _split(x):
    """float32 -> hi + lo as the activation buffers store it."""
    hi, lo = precision_budget.split(x)
    return hi + lo


# (state_dict prefix, input shape N C H W, conv kwargs): a stage-3-sized 3x3 (dec1's 97 -> 32 at full width, two
# 128-pixel tiles per row), the widest dilated ASPP branch and the 1x1 ASPP bottleneck, at stage 3's e5 size
LAYERS = [
    ('stg3_full_band_net.dec1.conv1', (1, 97, 16, 256), dict(pad=1)),
    ('stg3_full_band_net.aspp.conv5', (1, 256, 64, 16), dict(pad=(12, 6), dil=(12, 6))),
    ('stg3_full_band_net.aspp.bottleneck', (1, 1280, 64, 16), dict(pad=0)),
]


@pytest.mark.parametrize('layer', LAYERS, ids=[p.split('.', 1)[1] for p, _, _ in LAYERS])
def test_conv_gate_passes_kernel_arithmetic_and_catches_faults(layer, sd32, sd64):
    p, shape, kw = layer
    g = torch.Generator().manual_seed(11)
    x = _split(torch.relu(torch.randn(shape, generator=g)))      # a post-ReLU activation, as stored
    with torch.no_grad():
        ref = lr.conv(sd64, p, x.double(), **kw)
        errs = {}
        for scheme in ('3pass', 'no_wlo', 'no_xlo'):
            precision_budget.SCHEME[p] = scheme
            try:
                errs[scheme] = lr.rel_err(precision_budget.conv_bn_act_emulated(sd32, p, x, **kw), ref)
            finally:
                precision_budget.SCHEME.clear()
        y = precision_budget.conv_bn_act_emulated(sd32, p, x, **kw)
    # one tile of the tensor-core kernels: 128 output pixels (a row segment, or 128 / W whole rows) x 16 channels
    W = y.shape[3]
    tile = y.clone()
    if W >= 128:
        tile[:, :16, 5, 128:256] = 0
    else:
        tile[:, :16, 128 // W:2 * 128 // W, :] = 0
    errs['tile'] = lr.rel_err(tile, ref)
    print(p, ' '.join('%s=%.2e' % kv for kv in errs.items()))
    assert errs['3pass'] < lr.GATE_CONV / 2
    for fault in ('no_wlo', 'no_xlo', 'tile'):
        assert errs[fault] > 4 * lr.GATE_CONV, fault


def _lstm_fp32(xp, whh, reverse, late=False):
    """The recurrence in float32 (as the kernel computes it).  late=True (reverse direction): the first step, frame
    T - 1, is skipped and left at zero, and the recurrence starts from zero state at frame T - 2."""
    xp, whh = xp.float(), whh.float()
    if not late:
        return lr.lstm_direction(xp, whh, reverse)
    out = torch.zeros(xp.shape[0], xp.shape[1], xp.shape[2] // 4)
    out[:, :-1] = lr.lstm_direction(xp[:, :-1], whh, True)
    return out


def test_lstm_gate_passes_fp32_recurrence_and_catches_a_late_start(sd64):
    p = 'stg1_low_band_net.0.lstm_dec2'   # hid 64, 256 bins
    g = torch.Generator().manual_seed(5)
    l0 = torch.randn(2, 256, 128, generator=g, dtype=torch.float64) * 0.5
    with torch.no_grad():
        xp = lr.lstm_xp(sd64, p, l0).float()      # the fp32 plane the kernel reads
        ref = lr.lstm_hs(sd64, p, xp.double())
        g4 = xp.shape[2] // 2
        fw = _lstm_fp32(xp[:, :, :g4], sd64[p + '.lstm.weight_hh_l0'], False)
        rv = _lstm_fp32(xp[:, :, g4:], sd64[p + '.lstm.weight_hh_l0_reverse'], True)
        rv_late = _lstm_fp32(xp[:, :, g4:], sd64[p + '.lstm.weight_hh_l0_reverse'], True, late=True)
    ok = lr.abs_err(torch.cat([fw, rv], 2), ref)
    late = lr.abs_err(torch.cat([fw, rv_late], 2), ref)
    print('lstm hs: fp32 %.2e, reverse one step late %.2e' % (ok, late))
    assert ok < lr.GATE_LSTM / 4
    assert late > 4 * lr.GATE_LSTM

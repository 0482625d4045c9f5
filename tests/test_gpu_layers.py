"""Layer-by-layer parity of the native CascadedNet forward against float64 references (run on the B200 box).

One vr_forward per configuration on N windows; every intermediate tensor is then read back with vr_debug_read and each
layer is checked against tests/layer_reference.py computed from the layer's own read-back input (what the kernel
consumed, hi + lo), so that every failure names one kernel instead of showing up as mask error.  The same run checks
that pad channels hold zeros, that a second forward is bitwise identical (stream joins) and that each window matches a
batch-1 forward.  Gates are those of tests/layer_reference.py, calibrated on the CPU by tests/test_layer_reference.py.
"""
import ctypes

import numpy as np
import pytest
import torch

import layer_reference as lr
from conftest import record_parity

pytestmark = pytest.mark.gpu

# name -> (n_fft, hop, nout, nout_lstm, cropsize, N, conv_mode, fused decoder layouts)
CONFIGS = {
    'default': (2048, 1024, 32, 128, 256, 3, 0, 1),
    'staged': (2048, 1024, 32, 128, 256, 3, 0, 0),
    'cudacore': (2048, 1024, 32, 128, 256, 3, 1, 1),
    'small': (512, 256, 16, 32, 192, 2, 0, 1),
    'crop512': (2048, 1024, 32, 128, 512, 1, 0, 1),
}
NET_BUFFERS = ('cat1', 'cat2', 'cat3', 'cat4', 't2', 't3', 't4', 't5', 'e5', 'pool', 'f1', 'acat', 'ao', 'd4', 'd3',
               'd2', 'lstm_l0', 'lstm_xp', 'lstm_hs', 'lstm_y')


def _windows(n_fft, hop, crop, N):
    """N magnitude windows [N, 2, bins, crop]: windows 1.. of the normalised, padded 10 s sine mix as the Separator cuts
    them (window 1 is the golden fixture's first window for cropsize 256), the last one seeded uniform when N > 1."""
    from lib import synth
    from oracle import separator_oracle, stft_oracle
    X = stft_oracle.wave_to_spectrogram(synth.sine_mix(10.0), hop, n_fft)
    pad_l, pad_r, roi = separator_oracle.make_padding(X.shape[2], crop, 64)
    Xp = np.abs(np.pad(X, ((0, 0), (0, 0), (pad_l, pad_r)))) / np.abs(X).max()
    wins = [Xp[:, :, (i + 1) * roi:(i + 1) * roi + crop] for i in range(max(1, N - 1))]
    if N > 1:
        wins.append(np.random.default_rng(7).uniform(0.0, 1.0, size=(2, n_fft // 2 + 1, crop)))
    return np.stack(wins).astype(np.float32)


class _Run(object):
    def __init__(self, ctx):
        self.ctx = ctx
        self.lib = ctx.lib

    def forward(self, mag):
        from lib import _native
        mask = torch.empty_like(mag)
        self.ctx.check(self.lib.vr_forward(self.ctx.handle, _native.ptr(mag), mag.shape[0], _native.ptr(mask),
                                           _native.stream_ptr()), 'vr_forward')
        return mask

    def read(self, name):
        """Tensor `name` of the last forward (device float32), or None if the library reports an error."""
        from lib import _native
        dims = (ctypes.c_int64 * 4)()
        st = _native.stream_ptr()
        self.lib.vr_debug_read(self.ctx.handle, name.encode(), None, 0, dims, st)   # size query: fails, sets dims
        if dims[0] <= 0:
            return None
        out = torch.empty(tuple(dims), dtype=torch.float32, device='cuda')
        if self.lib.vr_debug_read(self.ctx.handle, name.encode(), _native.ptr(out), out.numel(), dims, st) != 0:
            return None
        return out

    def read_all(self, mask, nets_with_lstm_up):
        t = {'mask': mask.clone()}
        for name in ('x', 'aux1', 'aux2', 'o1', 'o2', 'f3'):
            t[name] = self.read(name)
        for k in range(5):
            for b in NET_BUFFERS + (('lstm_up',) if k in nets_with_lstm_up else ()):
                t['%d.%s' % (k, b)] = self.read('%d.%s' % (k, b))
        torch.cuda.synchronize()
        return t


def _layout(n, H, W, conv_mode, fused):
    """dec1 input layout BaseNet chooses (engine.cu build_basenet): (skip_only, lstm_own, e1_coff, lstm_coff)."""
    skip_only = conv_mode == 0 and fused == 1 and (2 * n) % 32 == 0 and W % 128 == 0 and H % 8 == 0
    lstm_own = skip_only and n % 32 == 0
    e1_coff = 0 if skip_only else 2 * n + 16
    lstm_coff = 0 if lstm_own else (n if skip_only else 2 * n)
    return skip_only, lstm_own, e1_coff, lstm_coff


def _batch_slice(name, t, i):
    return t[:, i:i + 1] if name.endswith('lstm_y') else t[i:i + 1]


def _check_net(res, cfg, k, n, t, sd, layout, fused_up):
    """Appends (record name, err, gate) for every layer of BaseNet k; t holds the read-back tensors (float64)."""
    p, net = lr.NETS[k], lr.SHORT[k]
    skip_only, lstm_own, e1_coff, lstm_coff = layout
    g = lambda b: t['%d.%s' % (k, b)]   # noqa: E731
    Hb = t['x'].shape[2] // 2

    def add(layer, err, gate):
        res['checks'].append(('layer_%s_%s_%s' % (cfg, net, layer), err, gate))

    def conv_check(layer, got, ref):
        add(layer, lr.rel_err(got, ref), lr.GATE_CONV)

    def up_slice(layer, got, src):
        # a decoder input slice the staged upsample kernel writes; the fused row kernel never materialises it (zeros)
        if fused_up and not got.any():
            return
        conv_check(layer, got, lr.upsample(src))

    # network input (reference channel order: x, aux1, aux2) and output
    rows = slice(0, Hb) if k in (0, 2) else slice(Hb, 2 * Hb) if k in (1, 3) else slice(0, 2 * Hb)
    parts = [t['x']] + ([t['aux1']] if k >= 2 else []) + ([t['aux2']] if k == 4 else [])
    x_in = torch.cat(parts, 1)[:, :, rows]
    out = {0: t['o1'], 1: t['aux1'][:, :, Hb:], 2: t['o2'], 3: t['aux2'][:, :, Hb:], 4: t['f3']}[k]

    cat1 = g('cat1')
    e1 = cat1[:, e1_coff:e1_coff + n]
    conv_check('enc1', e1, lr.conv(sd, p + '.enc1', x_in))
    enc_in = e1
    enc_out = {2: (g('t2'), g('cat2')[:, 4 * n:6 * n]), 3: (g('t3'), g('cat3')[:, 6 * n:10 * n]),
               4: (g('t4'), g('cat4')[:, 8 * n:14 * n]), 5: (g('t5'), g('e5'))}
    for j in (2, 3, 4, 5):
        tj, ej = enc_out[j]
        conv_check('enc%d.conv1' % j, tj, lr.enc_conv1(sd, '%s.enc%d.conv1' % (p, j), enc_in))
        conv_check('enc%d.conv2' % j, ej, lr.enc_conv2(sd, '%s.enc%d.conv2' % (p, j), tj))
        enc_in = ej
    e5 = g('e5')
    # ASPP
    c8 = 8 * n
    conv_check('aspp.pool', g('pool'), lr.aspp_pool(e5))
    conv_check('aspp.conv1', g('f1'), lr.aspp_branch(sd, p + '.aspp', 1, g('pool')))
    acat = g('acat')
    add('aspp.broadcast', 0.0 if torch.equal(acat[:, :c8], g('f1').expand(-1, -1, acat.shape[2], -1)) else 1.0, 0.0)
    for i in (2, 3, 4, 5):
        conv_check('aspp.conv%d' % i, acat[:, (i - 1) * c8:i * c8], lr.aspp_branch(sd, p + '.aspp', i, e5))
    conv_check('aspp.bottleneck', g('ao'), lr.conv(sd, p + '.aspp.bottleneck', acat, pad=0))
    # decoders 4, 3, 2
    conv_check('dec4.up', g('cat4')[:, :8 * n], lr.upsample(g('ao')))
    conv_check('dec4', g('d4'), lr.decoder(sd, p + '.dec4', g('ao'), g('cat4')[:, 8 * n:]))
    conv_check('dec3.up', g('cat3')[:, :6 * n], lr.upsample(g('d4')))
    conv_check('dec3', g('d3'), lr.decoder(sd, p + '.dec3', g('d4'), g('cat3')[:, 6 * n:]))
    up_slice('dec2.up', g('cat2')[:, :4 * n], g('d3'))
    d2 = g('d2')
    h = d2[:, :2 * n]
    conv_check('dec2', h, lr.decoder(sd, p + '.dec2', g('d3'), g('cat2')[:, 4 * n:]))
    # LSTM branch, each plane forced from the previous GPU plane
    lp = p + '.lstm_dec2'
    l0_ref, l0_scale = lr.lstm_l0(sd, lp, h)
    add('lstm.conv', ((g('lstm_l0')[..., 0] - l0_ref).abs() / l0_scale.clamp_min(1e-30)).max().item(), lr.GATE_L0)
    xp = g('lstm_xp')[..., 0]
    add('lstm.xp', lr.rel_err(xp, lr.lstm_xp(sd, lp, g('lstm_l0')[..., 0])), lr.GATE_LSTM)
    hs = g('lstm_hs')[..., 0]
    add('lstm.hs', lr.abs_err(hs, lr.lstm_hs(sd, lp, xp)), lr.GATE_LSTM)
    y = g('lstm_y')[..., 0]
    add('lstm.y', lr.rel_err(y, lr.lstm_y(sd, lp, hs)), lr.GATE_LSTM)
    y_img = y.permute(1, 0, 2)[:, None]   # [N, 1, bins, T]
    if skip_only:
        up_lstm = g('lstm_up')[:, :1] if lstm_own else cat1[:, lstm_coff:lstm_coff + 1]
        conv_check('lstm.up', up_lstm, lr.upsample(y_img))
    else:
        conv_check('lstm.to_channel', d2[:, 2 * n:2 * n + 1], y_img)
        up_slice('dec1.up', cat1[:, :2 * n + 1], d2[:, :2 * n + 1])
        up_lstm = lr.upsample(d2[:, 2 * n:2 * n + 1])
    dec1_in = torch.cat([lr.upsample(h), up_lstm, e1], 1)
    conv_check('dec1', out, lr.conv(sd, p + '.dec1.conv1', dec1_in))

    # pad channels hold zeros forever
    pads = []
    if skip_only and lstm_own:
        pads.append(('lstm_up[1:]', g('lstm_up')[:, 1:]))
    elif skip_only:
        pads.append(('cat1[n+1:]', cat1[:, n + 1:]))
    else:
        pads += [('cat1[2n+1:2n+16]', cat1[:, 2 * n + 1:2 * n + 16]), ('cat1[3n+16:]', cat1[:, 3 * n + 16:]),
                 ('d2[2n+1:]', d2[:, 2 * n + 1:])]
    for name, v in pads:
        if v.numel() and v.any():
            res['pad_errors'].append('%s %s: %d non-zero values' % (net, name, int((v != 0).sum())))


def _run_config(cfg):
    from lib import _native, synth
    n_fft, hop, nout, nout_lstm, crop, N, conv_mode, fused = CONFIGS[cfg]
    lib = _native.load_library()
    lib.vr_debug_set(5, fused)
    try:
        ctx = _native.Context(0, n_fft, hop, nout, nout_lstm, crop, N, conv_mode)
        sd_np = synth.make_state_dict(n_fft, nout, nout_lstm)
        ctx.load_state_dict(sd_np)
        run = _Run(ctx)
        Hb = n_fft // 4
        ns = (nout // 2, nout // 4, nout, nout // 2, nout)
        layouts = [_layout(ns[k], 2 * Hb if k == 4 else Hb, crop, conv_mode, fused) for k in range(5)]
        own = [k for k in range(5) if layouts[k][1]]
        mag = torch.from_numpy(_windows(n_fft, hop, crop, N)).cuda()
        t = run.read_all(run.forward(mag), own)
        res = {'checks': [], 'pad_errors': [], 'read_errors': [], 'bitwise': [], 'batch1': [], 'N': N,
               'stages': None}
        res['read_errors'] = [name for name, v in t.items() if v is None]
        if res['read_errors']:
            return res
        # lstm_up exists only where the net keeps the LSTM group in a buffer of its own
        for k in range(5):
            if k not in own and run.read('%d.lstm_up' % k) is not None:
                res['read_errors'].append('%d.lstm_up readable although BaseNet %d has no such buffer' % (k, k))
        # a second forward on the same input: bitwise equal everywhere
        t2 = run.read_all(run.forward(mag), own)
        res['bitwise'] = [name for name in t if not torch.equal(t[name], t2[name])]
        del t2
        # each window alone (batch 1) against its slice of the batch
        if N > 1:
            for i in range(N):
                t1 = run.read_all(run.forward(mag[i:i + 1].contiguous()), own)
                for name in t:
                    err = lr.rel_err(t1[name], _batch_slice(name, t[name], i))
                    if not err <= 1e-6:
                        res['batch1'].append('window %d %s: %.3g' % (i, name, err))
                del t1
        ctx.close()
    finally:
        lib.vr_debug_set(5, 1)

    sd = lr.state_dict64(sd_np, 'cuda')
    t = {k: v.double() for k, v in t.items()}
    with torch.no_grad():
        for k in range(5):
            _check_net(res, cfg, k, ns[k], t, sd, layouts[k], fused_up=conv_mode == 0 and fused == 1)
        Hb = t['x'].shape[2] // 2
        res['checks'].append(('layer_%s_stg1_low_bridge' % cfg, lr.rel_err(
            t['aux1'][:, :, :Hb], lr.conv(sd, 'stg1_low_band_net.1', t['o1'], pad=0)), lr.GATE_CONV))
        res['checks'].append(('layer_%s_stg2_low_bridge' % cfg, lr.rel_err(
            t['aux2'][:, :, :Hb], lr.conv(sd, 'stg2_low_band_net.1', t['o2'], pad=0)), lr.GATE_CONV))
        mref = lr.mask_out(sd, t['f3'])
        res['checks'].append(('layer_%s_out_mask' % cfg, lr.abs_err(t['mask'], mref), lr.GATE_MASK))
        res['nyquist_replicated'] = torch.equal(t['mask'][:, :, -1], t['mask'][:, :, -2])
        res['stages'] = {'l1': t['aux1'][:1, :, :Hb], 'h1': t['aux1'][:1, :, Hb:], 'l2': t['aux2'][:1, :, :Hb],
                         'h2': t['aux2'][:1, :, Hb:], 'f3': t['f3'][:1]}
        res['stages'] = {k: v[:, :, ::16, ::4].cpu().numpy() for k, v in res['stages'].items()}
    del t, sd
    torch.cuda.empty_cache()
    return res


@pytest.fixture(scope='module', params=list(CONFIGS))
def layer_run(request):
    return request.param, _run_config(request.param)


def test_every_tensor_is_readable(layer_run):
    cfg, res = layer_run
    assert not res['read_errors'], res['read_errors']


def test_each_layer_matches_its_float64_reference(layer_run):
    cfg, res = layer_run
    assert not res['read_errors'], res['read_errors']
    bad = []
    for name, err, gate in res['checks']:
        record_parity(name, err, gate)
        if not err <= gate:
            bad.append('%s: %.3g (gate %.1g)' % (name, err, gate))
    worst = max(res['checks'], key=lambda c: c[1] / c[2] if c[2] else c[1])
    print('%s: %d checks, worst margin %s = %.3g (gate %.1g)' % (cfg, len(res['checks']), worst[0], worst[1], worst[2]))
    assert res['nyquist_replicated']
    assert not bad, bad


def test_pad_channels_stay_zero(layer_run):
    cfg, res = layer_run
    assert not res['read_errors'], res['read_errors']
    assert not res['pad_errors'], res['pad_errors']


def test_second_forward_is_bitwise_identical(layer_run):
    cfg, res = layer_run
    assert not res['read_errors'], res['read_errors']
    assert not res['bitwise'], res['bitwise']


def test_batch_matches_single_windows(layer_run):
    cfg, res = layer_run
    assert not res['read_errors'], res['read_errors']
    if res['N'] == 1:
        pytest.skip('batch of one window')
    assert not res['batch1'], res['batch1']


def test_first_window_stages_match_reference_golden(layer_run, golden_default):
    cfg, res = layer_run
    assert not res['read_errors'], res['read_errors']
    if CONFIGS[cfg][:5] != (2048, 1024, 32, 128, 256):
        pytest.skip('the golden stage activations are those of the default net at cropsize 256')
    for k, got in res['stages'].items():
        ref = golden_default['win1_%s_sub' % k]
        err = np.abs(got - ref).max() / np.abs(ref).max()
        record_parity('stage_%s_win1_%s_relative_vs_reference_golden' % (cfg, k), err, 1e-3)
        assert err < 1e-3, (k, err)

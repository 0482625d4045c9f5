"""Generates tests/golden/*.npz by running the UNMODIFIED reference (imported from /root/reference
through oracle/librosa_shim.py) on the seeded synthetic input / checkpoint.  TEST INFRASTRUCTURE.

Run in the build container only (``python -m oracle.make_golden`` from the repo root); the
fixtures are committed because /root/reference does not exist on the GPU box.

What is pinned, per case:
  * reference ``inference.Separator.separate`` / ``separate_tta`` (inference.py:70-102) with the
    reference ``lib.nets.CascadedNet`` (lib/nets.py:44-141) on CPU fp32 -> mask, y_spec, v_spec
  * reference ``spec_utils.spectrogram_to_wave`` over the shimmed istft -> waves
  * first-window stage activations (debug aid)
Arrays are stored subsampled (strides recorded) together with float64 checksums of the full arrays.
The STFT/iSTFT arithmetic itself is the App. A restatement (librosa is absent): parity unpinned there.
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'vocal-remover_b200'))

from oracle import librosa_shim  # noqa: E402

GOLDEN_DIR = os.path.join(ROOT, 'tests', 'golden')


def checksum(a):
    a = np.asarray(a)
    if np.iscomplexobj(a):
        return np.array([a.real.astype(np.float64).sum(), a.imag.astype(np.float64).sum(),
                         (np.abs(a).astype(np.float64) ** 2).sum(), np.abs(a).max()], dtype=np.float64)
    a64 = a.astype(np.float64)
    return np.array([a64.sum(), (a64 ** 2).sum(), a64.min(), a64.max()], dtype=np.float64)


def run_case(name, seconds, n_fft, hop, nout, nout_lstm, cropsize, batchsize, fs, ts, with_tta, with_stages):
    ref_inference, ref_nets, ref_spec_utils, ref_dataset = librosa_shim.import_reference()
    from lib import synth
    torch.set_num_threads(os.cpu_count())
    sd = synth.to_torch_state_dict(synth.make_state_dict(n_fft, nout, nout_lstm, seed=0))
    model = ref_nets.CascadedNet(n_fft, hop, nout, nout_lstm)
    model.load_state_dict(sd)
    model.eval()
    wave = synth.sine_mix(seconds)
    X = ref_spec_utils.wave_to_spectrogram(wave, hop, n_fft)
    sp = ref_inference.Separator(model, torch.device('cpu'), batchsize, cropsize, False)
    captured = {}
    orig_post = sp._postprocess

    def post(X_spec, mask):
        captured['mask'] = np.array(mask, copy=True)
        return orig_post(X_spec, mask)
    sp._postprocess = post

    out = dict(meta=np.array([seconds, n_fft, hop, nout, nout_lstm, cropsize, batchsize, fs, ts], dtype=np.float64))
    y, v = sp.separate(X)
    mask = captured['mask']
    assert y.dtype == np.complex64 and mask.dtype == np.float32, (y.dtype, mask.dtype)
    out['absmax'] = np.array(np.abs(X).max(), dtype=np.float32)
    out['X_sub'] = X[:, ::fs * 2, ::ts]
    out['X_sum'] = checksum(X)
    out['mask_sub'] = mask[:, ::fs, ::ts]
    out['mask_sum'] = checksum(mask)
    out['y_sub'] = y[:, ::fs * 2, ::ts]
    out['y_sum'] = checksum(y)
    out['v_sum'] = checksum(v)
    wy = ref_spec_utils.spectrogram_to_wave(y, hop_length=hop)
    wv = ref_spec_utils.spectrogram_to_wave(v, hop_length=hop)
    out['wave_inst_sub'] = wy[:, ::16]
    out['wave_voc_sub'] = wv[:, ::16]
    out['wave_inst_sum'] = checksum(wy)
    out['wave_voc_sum'] = checksum(wv)
    print(name, 'X', X.shape, 'absmax', out['absmax'], 'mask', mask.shape, mask.min(), mask.max(),
          'logit-like spread: frac<0.1', (mask < 0.1).mean(), 'frac>0.9', (mask > 0.9).mean())
    if with_tta:
        y2, v2 = sp.separate_tta(X)
        out['mask_tta_sub'] = captured['mask'][:, ::fs, ::ts]
        out['mask_tta_sum'] = checksum(captured['mask'])
        out['y_tta_sum'] = checksum(y2)
        pad_l, pad_r, _ = ref_dataset.make_padding(X.shape[2], cropsize, model.offset)
        out['tta_norm'] = np.array(np.pad(X, ((0, 0), (0, 0), (pad_l, pad_r))).max(), dtype=np.complex64)
    if with_stages:
        pad_l, pad_r, roi = ref_dataset.make_padding(X.shape[2], cropsize, model.offset)
        Xp = np.pad(X, ((0, 0), (0, 0), (pad_l, pad_r)), mode='constant')
        Xp /= np.abs(X).max()
        x0 = torch.from_numpy(np.abs(Xp[None, :, :, roi:roi + cropsize]))
        acts = {}

        def hook(nm):
            def f(mod, inp, o):
                acts[nm] = o.detach().numpy()
            return f
        hs = [model.stg1_low_band_net.register_forward_hook(hook('l1')),
              model.stg2_low_band_net.register_forward_hook(hook('l2')),
              model.out.register_forward_hook(hook('logit'))]
        # BaseNet overrides __call__, so hooks do not fire on it; wrap the three bare BaseNets instead
        for nm, attr in (('h1', 'stg1_high_band_net'), ('h2', 'stg2_high_band_net'), ('f3', 'stg3_full_band_net')):
            net = getattr(model, attr)
            cls_call = type(net).__call__

            def wrapped(x, _net=net, _nm=nm, _call=cls_call):
                o = _call(_net, x)
                acts[_nm] = o.detach().numpy()
                return o
            object.__setattr__(net, 'forward', None)
            setattr(model, attr, _Wrap(net, wrapped))
        with torch.no_grad():
            m0 = model.forward(x0).numpy()
        for h in hs:
            h.remove()
        out['win1_mask_sub'] = m0[:, :, ::fs, ::ts]
        for k, a in acts.items():
            out['win1_' + k + '_sub'] = a[:, :, ::16, ::4]
            out['win1_' + k + '_sum'] = checksum(a)
        lg = acts['logit'][..., model.offset:-model.offset]
        print(name, 'win1 logit std', lg.std(), 'stages', {k: float(np.abs(a).max()) for k, a in acts.items()})
    path = os.path.join(GOLDEN_DIR, name + '.npz')
    np.savez_compressed(path, **out)
    print('wrote', path, os.path.getsize(path) // 1024, 'KiB')


def merge_artifacts_masks():
    """Six seeded (2, 33, 400) masks: low-level noise with one to three long above-threshold runs."""
    rng = np.random.default_rng(0)
    masks = []
    for trial in range(6):
        m = rng.uniform(0.0, 0.04, size=(2, 33, 400)).astype(np.float32)
        for s, e in ((0, 90), (150, 260), (275, 400))[:1 + trial % 3]:
            m[:, :, s:e] = rng.uniform(0.06, 1.0, size=(2, 33, e - s))
        masks.append(m)
    return masks


def run_functions(name):
    """Reference outputs of two single functions: ``CascadedNet.predict_mask`` (lib/nets.py:124-131) on the first
    256-frame window of the 10 s input with the default net, and ``spec_utils.merge_artifacts`` (lib/spec_utils.py:60-93)
    on ``merge_artifacts_masks()``.  Stored sampled over bins, with float64 checksums of the full arrays."""
    ref_inference, ref_nets, ref_spec_utils, ref_dataset = librosa_shim.import_reference()
    from lib import synth
    sd = synth.to_torch_state_dict(synth.make_state_dict())
    model = ref_nets.CascadedNet(2048, 1024, 32, 128)
    model.load_state_dict(sd)
    model.eval()
    X = ref_spec_utils.wave_to_spectrogram(synth.sine_mix(10.0), 1024, 2048)
    pad_l, pad_r, roi = ref_dataset.make_padding(X.shape[2], 256, model.offset)
    Xp = np.pad(X, ((0, 0), (0, 0), (pad_l, pad_r)))
    Xp /= np.abs(X).max()
    with torch.no_grad():
        pm = model.predict_mask(torch.from_numpy(np.abs(Xp[None, :, :, roi:roi + 256]))).numpy()
    merged = [ref_spec_utils.merge_artifacts(m.copy()) for m in merge_artifacts_masks()]
    out = dict(predict_mask_sub=pm[:, :, 4::8, :], predict_mask_sum=checksum(pm),
               merge_artifacts_sub=np.stack([r[:, ::8, :] for r in merged]),
               merge_artifacts_sum=np.stack([checksum(r) for r in merged]))
    path = os.path.join(GOLDEN_DIR, name + '.npz')
    np.savez_compressed(path, **out)
    print('wrote', path, os.path.getsize(path) // 1024, 'KiB')


class _Wrap(torch.nn.Module):
    def __init__(self, net, fn):
        super().__init__()
        self.net = net
        self.fn = fn

    def forward(self, x):
        return self.fn(x)


def main():
    os.makedirs(GOLDEN_DIR, exist_ok=True)
    # BASELINE.json configs[0]/[1]: 10 s input, default net, reference defaults batchsize 4 cropsize 256
    run_case('ref_10s_default', 10.0, 2048, 1024, 32, 128, 256, 4, 8, 1, True, True)
    # a small configuration exercising the n_fft / cropsize / nout flags
    run_case('ref_3s_small', 3.0, 512, 256, 16, 32, 192, 2, 2, 1, False, False)
    run_functions('ref_functions')


if __name__ == '__main__':
    main()

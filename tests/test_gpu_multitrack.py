"""Several tracks per call (vr_separate_many, vr_separate_waves, Separator.separate_waves, inference.py with several
-i inputs) on the GPU: the windows of all tracks share forward batches, and every track must still get what the
single-track calls give it alone."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import PKG, record_parity

pytestmark = pytest.mark.gpu

MASK_TOL = 1e-3
BATCH_TOL = 1e-6   # window-batch composition (tests/test_gpu_layers.py test_batch_matches_single_windows)
STEM_TOL = 1e-5    # stems across batch sizes (tests/test_gpu_parity.py test_full_size_track_properties)


def _dev():
    assert torch.cuda.is_available(), 'gpu tests need a CUDA device'
    return torch.device('cuda:0')


def _model(n_fft=2048, hop=1024, nout=32, nout_lstm=128):
    from lib import nets, synth
    m = nets.CascadedNet(n_fft, hop, nout, nout_lstm)
    m.load_state_dict(synth.to_torch_state_dict(synth.make_state_dict(n_fft, nout, nout_lstm)))
    m.to(_dev())
    return m


@pytest.fixture(scope='module')
def default_model():
    return _model()


def _wave_of_frames(n_frames, seed, hop=1024):
    """A sine mix whose STFT has exactly n_frames frames (T = 1 + L // hop)."""
    from lib import synth
    L = hop * (n_frames - 1) + 100
    return synth.sine_mix(L / 44100.0 + 0.01, seed=seed)[:, :L]


def _tracks():
    from lib import synth
    waves = [_wave_of_frames(n, seed=n) for n in (3, 128, 129, 300)]
    waves.append(synth.sine_mix(10.0))            # the golden track
    waves.append(synth.sine_mix(30.0, seed=7))
    return waves


def _spec(wave):
    from lib import spec_utils
    return torch.from_numpy(spec_utils.wave_to_spectrogram(wave, 1024, 2048)).to(_dev())


@pytest.mark.parametrize('tta', [0, 1])
def test_masks_equal_single_track_calls(default_model, golden_default, tta):
    """max_batch 4 with tracks of 3, 128, 129, 300 frames, 10 s and 30 s: batches straddle tracks."""
    import inference
    sp = inference.Separator(default_model, _dev(), 4, 256, False)
    specs = [_spec(w) for w in _tracks()]
    assert [s.shape[2] for s in specs][:4] == [3, 128, 129, 300]
    many = sp._masks_device(specs, bool(tta))
    err = max((m - sp._mask_device(s, bool(tta))).abs().max().item() for m, s in zip(many, specs))
    record_parity('separate_many_mask_vs_single_track_tta%d' % tta, err, BATCH_TOL)
    assert err <= BATCH_TOL
    g = golden_default['mask_tta_sub' if tta else 'mask_sub']
    gerr = np.abs(many[4].cpu().numpy()[:, ::8, :] - g).max()
    record_parity('separate_many_mask_10s_tta%d_vs_reference_golden' % tta, gerr, MASK_TOL)
    assert gerr < MASK_TOL


@pytest.mark.parametrize('max_batch', [27, 1])
def test_tta_pass_boundary_is_ordered(default_model, max_batch):
    """One 2-window track with tta: at max_batch 27 both passes would fit in one batch, but pass 2 averages into the
    frames pass 1 writes, so they must run in separate launches."""
    import inference
    sp = inference.Separator(default_model, _dev(), max_batch, 256, False)
    spec = _spec(_wave_of_frames(200, seed=2))
    got = sp._masks_device([spec], True)[0]
    ref = sp._mask_device(spec, True)
    err = (got - ref).abs().max().item()
    record_parity('separate_many_tta_2windows_batch%d_vs_single' % max_batch, err, BATCH_TOL)
    assert err <= BATCH_TOL


def _stem_err(sp, waves, tta=False):
    packed = sp.separate_waves(waves, tta=tta)
    err = 0.0
    for w, (a, b) in zip(waves, packed):
        ra, rb = sp.separate_wave(w, tta=tta)
        if torch.is_tensor(a):
            assert a.is_cuda and b.is_cuda
            a, b, ra, rb = a.cpu().numpy(), b.cpu().numpy(), ra.cpu().numpy(), rb.cpu().numpy()
        else:
            assert isinstance(a, np.ndarray) and isinstance(b, np.ndarray)
        assert a.shape == ra.shape and b.shape == rb.shape
        err = max(err, float(np.abs(a - ra).max()), float(np.abs(b - rb).max()))
    return err


def test_stems_equal_single_track_calls_default_net(default_model):
    import inference
    waves = _tracks()
    sp = inference.Separator(default_model, _dev(), 4, 256, False)
    err = _stem_err(sp, waves)
    record_parity('separate_waves_stems_vs_single_numpy', err, STEM_TOL)
    assert err < STEM_TOL
    err = _stem_err(sp, [torch.from_numpy(w).cuda() for w in waves], tta=True)
    record_parity('separate_waves_stems_vs_single_cuda_tta', err, STEM_TOL)
    assert err < STEM_TOL
    spp = inference.Separator(default_model, _dev(), 4, 256, True)
    err = _stem_err(spp, waves)
    record_parity('separate_waves_stems_vs_single_postprocess', err, STEM_TOL)
    assert err < STEM_TOL


def test_stems_equal_single_track_calls_small_net():
    """n_fft 512: the radix-2 STFT / iSTFT kernels."""
    import inference
    from lib import synth
    m = _model(512, 256, 16, 32)
    waves = [_wave_of_frames(n, seed=n, hop=256) for n in (2, 65, 400)] + [synth.sine_mix(3.0)]
    sp = inference.Separator(m, _dev(), 3, 192, False)
    err = _stem_err(sp, waves)
    record_parity('separate_waves_stems_vs_single_small_net', err, STEM_TOL)
    assert err < STEM_TOL
    err = _stem_err(sp, [torch.from_numpy(w).cuda() for w in waves], tta=True)
    assert err < STEM_TOL
    err = _stem_err(inference.Separator(m, _dev(), 3, 192, True), waves)
    record_parity('separate_waves_stems_vs_single_small_net_postprocess', err, STEM_TOL)
    assert err < STEM_TOL


def test_launch_count_does_not_depend_on_the_number_of_tracks(default_model):
    import inference
    sp = inference.Separator(default_model, _dev(), 27, 256, False)
    ctx = sp._ctx()
    clips = [torch.from_numpy(_wave_of_frames(200, seed=k)).cuda() for k in range(12)]   # 2 windows each
    one = [torch.from_numpy(_wave_of_frames(3000, seed=1)).cuda()]                        # 24 windows
    sp.separate_waves(clips)
    n0 = ctx.launch_count()
    sp.separate_waves(clips)
    n_clips = ctx.launch_count() - n0
    n0 = ctx.launch_count()
    sp.separate_waves(one)
    n_one = ctx.launch_count() - n0
    torch.cuda.synchronize()
    assert n_clips == n_one, (n_clips, n_one)


def test_bad_tracks_are_isolated(default_model):
    """A silent track and one with NaN / Inf samples in the middle of a pack change nothing for the others."""
    import inference
    from lib import synth
    sp = inference.Separator(default_model, _dev(), 4, 256, False)
    good = [synth.sine_mix(s, seed=k) for k, s in enumerate((2.0, 7.0, 4.0, 12.0))]
    silent = np.zeros((2, 44100 * 3), dtype=np.float32)
    bad = synth.sine_mix(5.0, seed=9)
    bad[0, 1000] = np.nan
    bad[1, 5000] = np.inf
    ref = sp.separate_waves(good)
    got = sp.separate_waves(good[:2] + [silent, bad] + good[2:])
    for (a, b), (ra, rb) in zip(got[:2] + got[4:], ref):
        assert np.array_equal(a, ra) and np.array_equal(b, rb)
    assert np.abs(got[2][0]).max() == 0.0 and np.abs(got[2][1]).max() == 0.0


def test_order_and_workspace_reuse(default_model):
    import inference
    from lib import synth
    waves = [synth.sine_mix(s, seed=k) for k, s in enumerate((3.0, 9.0, 1.0, 20.0, 5.0))]
    sp = inference.Separator(default_model, _dev(), 4, 256, False)
    fwd = sp.separate_waves(waves)
    rev = sp.separate_waves(waves[::-1])[::-1]
    for (a, b), (ra, rb) in zip(fwd, rev):
        assert np.array_equal(a, ra) and np.array_equal(b, rb)
    # a large call grows the workspaces, the small call after it reuses them
    sp.separate_waves([synth.sine_mix(60.0, seed=3), synth.sine_mix(45.0, seed=4)], tta=True)
    small = sp.separate_waves(waves[:3], tta=True)
    fresh = inference.Separator(_model(), _dev(), 4, 256, False).separate_waves(waves[:3], tta=True)
    for (a, b), (ra, rb) in zip(small, fresh):
        assert np.array_equal(a, ra) and np.array_equal(b, rb)


def test_invalid_arguments_launch_nothing(default_model):
    import inference
    from lib import _native
    sp = inference.Separator(default_model, _dev(), 4, 256, False)
    ctx = sp._ctx()
    lib, st = ctx.lib, _native.stream_ptr()
    w = [torch.zeros((2, 44100), device='cuda') for _ in range(3)]
    o = [torch.zeros((2, 44032), device='cuda') for _ in range(3)]
    L = _native.i64_array([44100] * 3)
    s = [torch.zeros((2, 1025, 44), dtype=torch.complex64, device='cuda') for _ in range(3)]
    m = [torch.zeros((2, 1025, 44), device='cuda') for _ in range(3)]
    T = _native.i64_array([44] * 3)
    n0 = ctx.launch_count()

    def err(rc):
        assert rc != 0
        return lib.vr_last_error(ctx.handle).decode()

    pa = _native.ptr_array
    assert 'n_tracks' in err(lib.vr_separate_waves(ctx.handle, 0, pa(w), L, 0, pa(o), pa(o), st))
    assert 'n_tracks' in err(lib.vr_separate_many(ctx.handle, 0, pa(s), T, 0, pa(m), st))
    assert 'track 1' in err(lib.vr_separate_waves(ctx.handle, 3, pa([w[0], None, w[2]]), L, 0, pa(o), pa(o), st))
    assert 'track 2' in err(lib.vr_separate_waves(ctx.handle, 3, pa(w), L, 0, pa(o), pa(o[:2] + [None]), st))
    assert 'track 2' in err(lib.vr_separate_many(ctx.handle, 3, pa(s), T, 0, pa(m[:2] + [None]), st))
    assert 'NULL' in err(lib.vr_separate_many(ctx.handle, 3, None, T, 0, pa(m), st))
    bad_L = _native.i64_array([44100, 44100, -1])
    assert 'track 2' in err(lib.vr_separate_waves(ctx.handle, 3, pa(w), bad_L, 0, pa(o), pa(o), st))
    assert ctx.launch_count() == n0


def test_cli_several_inputs_match_single_runs(tmp_path):
    from lib import audio_io, synth
    ckpt = str(tmp_path / 'synthetic.pth')
    torch.save(synth.to_torch_state_dict(synth.make_state_dict()), ckpt)
    names = []
    for k, sec in enumerate((2.0, 3.5, 5.0)):
        path = str(tmp_path / ('clip%d.wav' % k))
        audio_io.write(path, 0.5 * synth.sine_mix(sec, seed=k).T, 44100)
        names.append(path)

    def run(inputs, out):
        cmd = [sys.executable, os.path.join(PKG, 'inference.py'), '-g', '0', '-P', ckpt, '-o', out, '-i'] + inputs
        r = subprocess.run(cmd, cwd=PKG, capture_output=True, text=True)
        assert r.returncode == 0, r.stdout + r.stderr

    run(names, str(tmp_path / 'multi'))
    err = 0.0
    for path in names:
        run([path], str(tmp_path / 'single'))
        base = os.path.splitext(os.path.basename(path))[0]
        for stem in ('Instruments', 'Vocals'):
            a, _ = audio_io.load(str(tmp_path / 'multi' / ('%s_%s.wav' % (base, stem))), 44100, mono=False)
            b, _ = audio_io.load(str(tmp_path / 'single' / ('%s_%s.wav' % (base, stem))), 44100, mono=False)
            assert a.shape == b.shape
            err = max(err, float(np.abs(a - b).max()))
    assert len(os.listdir(str(tmp_path / 'multi'))) == 6
    record_parity('cli_several_inputs_vs_single_runs', err, 0.0)
    assert err == 0.0

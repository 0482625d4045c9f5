"""Host-side mirror of the reference interface (no GPU): geometry, model-load API, sharding, post-process."""
import os

import numpy as np
import pytest
import torch

from oracle import separator_oracle


def test_make_padding_matches_oracle():
    from lib import dataset
    for width in list(range(1, 600, 7)) + [128, 256, 10336, 103360]:
        for crop in (256, 192, 128, 512):
            assert dataset.make_padding(width, crop, 64) == separator_oracle.make_padding(width, crop, 64)


def test_window_count_matches_reference_configs():
    from lib import distributed
    # SURVEY 8(d): 10 s -> 4 windows, 240 s -> 81, 2400 s -> 808
    assert distributed.window_count(431, 256, 64) == (4, 128)
    assert distributed.window_count(10336, 256, 64) == (81, 128)
    assert distributed.window_count(103360, 256, 64) == (808, 128)


def test_shard_windows_partition():
    from lib import distributed
    for n in (1, 4, 81, 163, 808, 7):
        for world in (1, 2, 3, 4, 8):
            seen = []
            for r in range(world):
                first, count, per = distributed.shard_windows(n, world, r)
                assert 0 <= count <= per
                seen += list(range(first, first + count))
            assert seen == list(range(n))


def test_model_surface_and_strict_loading():
    from lib import nets, synth
    m = nets.CascadedNet(2048, 1024, 32, 128)
    assert (m.offset, m.n_fft, m.hop_length, m.max_bin, m.output_bin) == (64, 2048, 1024, 1024, 1025)
    assert nets.CascadedASPPNet is nets.CascadedNet
    sd = synth.to_torch_state_dict(synth.make_state_dict())
    assert list(m.state_dict().keys()) == list(sd.keys())
    m.load_state_dict(sd)
    assert torch.equal(m.state_dict()['out.weight'], sd['out.weight'])
    assert sum(p.numel() for p in m.parameters()) == 14740882
    assert m.eval() is m and m.train() is m
    bad = dict(sd)
    bad.pop('aux_out.weight')
    with pytest.raises(RuntimeError, match='Missing key'):
        m.load_state_dict(bad)
    bad = dict(sd)
    bad['out.weight'] = torch.zeros(2, 16, 1, 1)
    with pytest.raises(RuntimeError, match='size mismatch'):
        m.load_state_dict(bad)
    with pytest.raises(RuntimeError, match='no CPU'):
        m.predict_mask(torch.zeros(1, 2, 1025, 256))
    with pytest.raises(NotImplementedError):
        nets.CascadedNet(2048, 1024, 32, 128, is_complex=True)


def test_crop_center():
    from lib import spec_utils
    a = torch.arange(2 * 3 * 4 * 10.).reshape(2, 3, 4, 10)
    b = torch.zeros(2, 3, 4, 6)
    assert spec_utils.crop_center(a, a) is a
    assert torch.equal(spec_utils.crop_center(a, b), a[:, :, :, 2:8])
    with pytest.raises(ValueError):
        spec_utils.crop_center(b, a)


def test_merge_artifacts_matches_reference(golden_functions):
    """Against the reference's lib/spec_utils.py:60-93 on the masks oracle/make_golden.py gave it."""
    from conftest import checksum
    from lib import spec_utils
    from oracle.make_golden import merge_artifacts_masks
    g = golden_functions
    for trial, m in enumerate(merge_artifacts_masks()):
        got = spec_utils.merge_artifacts(m.copy())
        assert np.allclose(got[:, ::8, :], g['merge_artifacts_sub'][trial], atol=1e-7), trial
        assert np.allclose(checksum(got), g['merge_artifacts_sum'][trial], rtol=1e-7), trial
    with pytest.raises(ValueError):
        spec_utils.merge_artifacts(np.ones((2, 3, 100), np.float32), min_range=10, fade_size=32)


def _gloo_worker(rank, world, port, n_frames, tmp):
    import torch.distributed as dist
    os.environ['MASTER_ADDR'] = '127.0.0.1'
    os.environ['MASTER_PORT'] = str(port)
    dist.init_process_group('gloo', rank=rank, world_size=world)
    from lib import distributed
    n_windows, roi = distributed.window_count(n_frames, 256, 64)
    first, count, per = distributed.shard_windows(n_windows, world, rank)
    # stand-in for the device result of this rank's windows: frame index encoded in the value
    full = torch.arange(n_windows * roi, dtype=torch.float32).repeat(2, 5, 1)
    block = torch.zeros(2, 5, per * roi)
    lo, hi = distributed.mask_block_frames(first, count, per, roi)
    block[:, :, :hi - lo] = full[:, :, lo:hi]
    gathered = distributed.gather_blocks(block, world, rank)
    if rank == 0:
        mask = distributed.assemble_mask(gathered, n_frames)
        torch.save(mask, tmp)
    dist.barrier()
    dist.destroy_process_group()


def test_sharded_gather_world_size_2_gloo(tmp_path):
    import torch.multiprocessing as mp
    n_frames = 431 + 128 * 3
    out = str(tmp_path / 'mask.pt')
    port = 29500 + os.getpid() % 1000
    mp.spawn(_gloo_worker, args=(2, port, n_frames, out), nprocs=2, join=True)
    mask = torch.load(out)
    assert mask.shape == (2, 5, n_frames)
    assert torch.equal(mask[0, 0], torch.arange(n_frames, dtype=torch.float32))


def _shared_host_worker(rank, world, port, tmp):
    import torch.distributed as dist
    os.environ['MASTER_ADDR'] = '127.0.0.1'
    os.environ['MASTER_PORT'] = str(port)
    dist.init_process_group('gloo', rank=rank, world_size=world)
    from lib import distributed
    buf = distributed.SharedHostBuffer.create((2, 1000), world, rank, register=False)
    assert buf is not None and buf.tensor.shape == (2, 1000)
    lo, hi = (0, 400) if rank == 0 else (400, 1000)     # every rank lands its own span, like separate_wave_host
    buf.tensor[:, lo:hi] = torch.arange(lo, hi, dtype=torch.float32)
    dist.barrier()
    whole = buf.tensor.clone()                          # ... and every rank sees the assembled buffer
    assert torch.equal(whole[0], torch.arange(1000, dtype=torch.float32)) and torch.equal(whole[1], whole[0])
    if rank == 1:
        torch.save(whole, tmp)
    buf.close(world)
    dist.destroy_process_group()


def test_shared_host_buffer_world_size_2_gloo(tmp_path):
    """The shared page-locked stem buffer of the multi-GPU host path (CUDA registration is left out on CPU)."""
    import torch.multiprocessing as mp
    out = str(tmp_path / 'whole.pt')
    port = 29500 + (os.getpid() + 17) % 1000
    mp.spawn(_shared_host_worker, args=(2, port, out), nprocs=2, join=True)
    assert torch.equal(torch.load(out)[0], torch.arange(1000, dtype=torch.float32))


def test_shard_plan_tiles_the_track():
    from lib import distributed
    for T in (431, 1292, 10336, 20672, 82688, 103360):
        for world in (2, 3, 4, 8):
            n_windows, roi = distributed.window_count(T, 256, 64)
            if n_windows < world:
                continue
            plans = [distributed.shard_plan(T, 256, 64, world, r) for r in range(world)]
            hops = [(p[7], p[8]) for p in plans]
            assert hops[0][0] == 0 and hops[-1][1] == T - 1
            for (x0, x1), (y0, y1) in zip(hops, hops[1:]):
                assert x1 == y0                                   # output spans tile [0, T-1)
            for first, count, roi_, f0, f1, a, b, k0, k1 in plans:
                assert a <= f0 <= f1 <= b or count == 0            # the rank's STFT span covers its mask frames
                if count > 0 and f1 < T:
                    assert f1 < b                                  # ... and the halo frame of its last output hop
                if count > 0:
                    assert a == max(0, first * roi_ - 64)           # exactly what its windows read (inference.py:44-50)


def test_cli_keeps_the_reference_flags():
    """The 12 flags of the reference CLI (inference.py:109-120), long and short forms."""
    import subprocess
    import sys
    from conftest import PKG
    out = subprocess.run([sys.executable, os.path.join(PKG, 'inference.py'), '--help'], capture_output=True, text=True,
                         cwd=PKG).stdout
    for flag in ('--gpu', '-g', '--pretrained_model', '-P', '--input', '-i', '--sr', '-r', '--n_fft', '-f',
                 '--hop_length', '-H', '--batchsize', '-B', '--cropsize', '-c', '--output_image', '-I', '--tta', '-t',
                 '--postprocess', '-p', '--output_dir', '-o'):
        assert flag in out, flag


def test_audio_io_wav_roundtrip(tmp_path):
    from lib import audio_io
    rng = np.random.default_rng(0)
    x = (rng.uniform(-0.9, 0.9, size=(4410, 2))).astype(np.float32)
    path = str(tmp_path / 'a.wav')
    audio_io.write(path, x, 44100)
    y, sr = audio_io.load(path, 44100, mono=False)
    assert sr == 44100 and y.shape == (2, 4410)
    assert np.abs(y.T - x).max() < 1e-4   # 16-bit PCM quantisation
    # another rate is resampled on the GPU (tests/test_resample.py checks the values); without one there is no CPU path
    if torch.cuda.is_available():
        y, sr = audio_io.load(path, 22050)
        assert sr == 22050 and y.shape == (2, 2205)
    else:
        with pytest.raises(RuntimeError):
            audio_io.load(path, 22050)


def test_artifact_weights_edge_cases():
    from lib import spec_utils
    # no frame above the threshold: the reference crashes on idx[0] (lib/spec_utils.py:65); here the mask is unchanged
    m = np.full((2, 5, 200), 0.01, np.float32)
    assert np.array_equal(spec_utils.merge_artifacts(m.copy()), m)
    # one run covering the whole track: no fade-in at frame 0; the reference still fades out before the last frame
    # because its run end is the last INDEX, which never equals the frame count (lib/spec_utils.py:66,83)
    w = spec_utils.artifact_weights(np.full(300, 0.5, np.float32))
    assert w[0] == 1.0 and w[150] == 1.0 and w[-1] == 0.0


def _emulated_separate_windows(mag_pad_fn, T, pad_l, first, count, mask, frame_shift, accumulate, roi=128, crop=256):
    """Frame arithmetic of vr_separate_windows (include/vr_b200.h) with a stand-in 'net': the mask of a window is a
    pointwise function of its centre frames, which is enough to check WHICH frames land WHERE."""
    for g in range(first, first + count):
        win = mag_pad_fn(pad_l, g * roi, g * roi + crop)          # (bins, crop) of the padded, normalised |X|
        m = np.tanh(win[:, (crop - roi) // 2:(crop + roi) // 2]) + 0.01 * (g % 3)   # window-dependent on purpose
        for j in range(roi):
            t = g * roi + j - frame_shift
            if 0 <= t < T:
                mask[:, t] = 0.5 * (mask[:, t] + m[:, j]) if accumulate else m[:, j]


@pytest.mark.parametrize('T,world', [(431, 2), (431, 3), (1000, 4), (128, 2), (130, 8), (2049, 8)])
def test_sharded_tta_plan_reproduces_the_unsharded_combine(T, world):
    """lib/distributed.py TTA sharding: every rank's own mask frames equal the single-rank result of
    Separator.separate_tta's two passes + average (inference.py:83-98)."""
    from lib import distributed as D
    rng = np.random.default_rng(T)
    bins = 5
    mag = rng.random((bins, T)).astype(np.float64)

    def padded(pad_l, lo, hi):
        out = np.zeros((bins, hi - lo))
        for i, t in enumerate(range(lo - pad_l, hi - pad_l)):
            if 0 <= t < T:
                out[:, i] = mag[:, t]
        return out

    n_windows, roi = D.window_count(T, 256, 64)
    ref = np.zeros((bins, T))
    _emulated_separate_windows(padded, T, 64, 0, n_windows, ref, 0, 0)
    _emulated_separate_windows(padded, T, 64 + roi // 2, 0, n_windows + 1, ref, roi // 2, 1)
    covered = np.zeros(T, dtype=bool)
    for rank in range(world):
        first, count, roi_, f0, f1, a, b, k0, k1 = D.shard_plan(T, 256, 64, world, rank)
        local = np.full((bins, T), np.nan)     # stale / foreign frames must never leak into the rank's span
        if count > 0:
            _emulated_separate_windows(padded, T, 64, first, count, local, 0, 0)
            g0, c2 = D.tta_window_range(first, count, n_windows)
            assert g0 + c2 <= n_windows + 1
            _emulated_separate_windows(padded, T, 64 + roi // 2, g0, c2, local, roi // 2, 1)
        assert np.array_equal(local[:, f0:f1], ref[:, f0:f1])
        covered[f0:f1] = True
    assert covered.all()


def test_make_pair_and_file_sharding(tmp_path):
    """lib/dataset.py:144-160 (pairing by sorted order, audio extensions only) and the file-level sharding of pseudo.py."""
    from lib import dataset
    mix, inst = tmp_path / 'mix', tmp_path / 'inst'
    mix.mkdir()
    inst.mkdir()
    for name in ('b.wav', 'a.flac', 'c.mp3', 'notes.txt'):
        (mix / name).write_bytes(b'')
    for name in ('2.wav', '1.wav', '3.wav', 'cover.jpg'):
        (inst / name).write_bytes(b'')
    pairs = dataset.make_pair(str(mix), str(inst))
    assert [(os.path.basename(a), os.path.basename(b)) for a, b in pairs] == [('a.flac', '1.wav'), ('b.wav', '2.wav'),
                                                                               ('c.mp3', '3.wav')]
    files = list(range(11))
    shards = [dataset.shard_files(files, 4, r) for r in range(4)]
    assert sorted(sum(shards, [])) == files                       # every file exactly once
    assert max(len(x) for x in shards) - min(len(x) for x in shards) <= 1
    assert dataset.shard_files(files, 1, 0) == files


def test_align_wave_head_and_tail_recovers_a_known_delay():
    """lib/spec_utils.py:96-119 restated (trim + cross-correlation of the first four seconds): a delayed, silence-padded
    copy must come out sample-aligned and of equal length."""
    from lib import spec_utils
    sr = 8000
    rng = np.random.default_rng(1)
    core = (rng.standard_normal((2, sr * 5)) * 0.3).astype(np.float32)
    a = np.concatenate([np.zeros((2, 3000), np.float32), core, np.zeros((2, 2000), np.float32)], axis=1)
    b = np.concatenate([np.zeros((2, 1200), np.float32), 0.7 * core[:, 137:], np.zeros((2, 4000), np.float32)], axis=1)
    a2, b2 = spec_utils.align_wave_head_and_tail(a, b, sr)
    assert a2.shape == b2.shape and a2.shape[1] > sr * 4
    # sample-aligned: in the interior (away from the frame-granular trim edges) b2 is exactly 0.7 * a2
    mid = slice(sr, 3 * sr)
    assert np.abs(b2[:, mid] - 0.7 * a2[:, mid]).max() < 1e-6
    t, (s0, s1) = spec_utils._trim_silence(a)
    assert s0 <= 3000 and s0 >= 3000 - 2048 and s1 >= 3000 + sr * 5 and t.shape[1] == s1 - s0


def test_async_writer_matches_sync_write_and_reports_failures(tmp_path):
    from lib import audio_io
    rng = np.random.default_rng(0)
    a = (0.5 * rng.standard_normal((4410, 2))).astype(np.float32)
    b = (0.5 * rng.standard_normal((4410, 2))).astype(np.float32)
    audio_io.write(str(tmp_path / 'a_sync.wav'), a, 44100)
    w = audio_io.AsyncWriter()
    w.write(str(tmp_path / 'a.wav'), a, 44100)
    w.write(str(tmp_path / 'b.wav'), b, 44100)
    w.join()
    assert (tmp_path / 'a.wav').read_bytes() == (tmp_path / 'a_sync.wav').read_bytes()
    xb, sr = audio_io.load(str(tmp_path / 'b.wav'), sr=44100, mono=False, dtype=np.float32)
    assert sr == 44100 and xb.shape == (2, 4410) and np.abs(xb - np.clip(b.T, -1, 1)).max() < 2.0 / 32768
    w.write(str(tmp_path / 'no_such_dir' / 'c.wav'), a, 44100)
    with pytest.raises(Exception):
        w.join()


def test_cache_or_load_layout_and_cache_hit(tmp_path, monkeypatch):
    """spec_utils.cache_or_load (reference lib/spec_utils.py:122-154): cache directory / file layout, the (T, 2, bins)
    on-disk transpose, and the second call served from the cache.  The GPU STFT is replaced by the CPU oracle here."""
    from lib import audio_io, spec_utils
    from oracle import stft_oracle
    calls = []

    def cpu_stft(wave, hop_length, n_fft):
        calls.append(wave.shape)
        return stft_oracle.wave_to_spectrogram(wave, hop_length, n_fft)

    monkeypatch.setattr(spec_utils, 'wave_to_spectrogram', cpu_stft)
    rng = np.random.default_rng(1)
    sr = 8000
    inst = (0.3 * np.sin(2 * np.pi * 440 * np.arange(2 * sr) / sr))[None, :].repeat(2, 0)
    voc = 0.2 * rng.standard_normal((2, 2 * sr))
    mix_dir, inst_dir = tmp_path / 'mixtures', tmp_path / 'instruments'
    mix_dir.mkdir()
    inst_dir.mkdir()
    audio_io.write(str(mix_dir / 'song.wav'), (inst + voc).T, sr)
    audio_io.write(str(inst_dir / 'song.wav'), inst.T, sr)
    X, y, pm, pi = spec_utils.cache_or_load(str(mix_dir / 'song.wav'), str(inst_dir / 'song.wav'), sr, 128, 256)
    assert pm == str(mix_dir / 'sr8000_hl128_nf256' / 'song.npy') and pi == str(inst_dir / 'sr8000_hl128_nf256' / 'song.npy')
    assert X.shape == y.shape and X.shape[:2] == (2, 129) and X.dtype == np.complex64
    assert np.load(pm).shape == (X.shape[2], 2, 129) and len(calls) == 2
    X2, y2, _, _ = spec_utils.cache_or_load(str(mix_dir / 'song.wav'), str(inst_dir / 'song.wav'), sr, 128, 256)
    assert len(calls) == 2                                # cache hit: no transform
    assert np.array_equal(X2, X) and np.array_equal(y2, y)

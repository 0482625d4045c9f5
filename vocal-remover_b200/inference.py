"""B200-native drop-in for the reference's inference.py (Separator + CLI).

Same command line (12 flags, inference.py:109-120), same output files and stage banners, same
``Separator(model, device, batchsize, cropsize, postprocess).separate / separate_tta`` contract
(numpy complex64 (2, bins, T) in, (y_spec, v_spec) out), but the sliding-window STFT -> CascadedNet ->
mask -> inverse-STFT path runs in hand-written sm_100a CUDA (libvr_b200.so, include/vr_b200.h).
``Separator.separate_wave`` is the fused device-resident form of the same path used by ``main``.
"""
import argparse
import os

import numpy as np
import torch

from lib import _native
from lib import audio_io
from lib import dataset
from lib import nets
from lib import spec_utils


class Separator(object):

    def __init__(self, model, device=None, batchsize=1, cropsize=256, postprocess=False):
        self.model = model
        self.offset = model.offset
        self.device = device
        self.batchsize = batchsize
        self.cropsize = cropsize
        self.postprocess = postprocess
        if device is not None:
            model.to(device)

    # ---- helpers ------------------------------------------------------------------------------------
    def _ctx(self):
        return self.model.native_context(self.cropsize, self.batchsize)

    def _dev(self):
        return torch.device('cuda', self._ctx().device_index)

    @staticmethod
    def _check_spec(X_spec):
        X_spec = np.asarray(X_spec)
        if X_spec.ndim != 3 or X_spec.shape[0] != 2:
            raise ValueError('X_spec must have shape (2, bins, frames)')
        return np.ascontiguousarray(X_spec.astype(np.complex64, copy=False))

    def _mask_device(self, d_spec, tta):
        ctx = self._ctx()
        T = d_spec.shape[2]
        d_mask = torch.empty((2, d_spec.shape[1], T), dtype=torch.float32, device=d_spec.device)
        ctx.check(ctx.lib.vr_separate(ctx.handle, _native.ptr(d_spec), T, 1 if tta else 0, _native.ptr(d_mask),
                                      _native.stream_ptr()), 'vr_separate')
        if self.postprocess:
            self._postprocess_device(d_mask)
        return d_mask

    def _masks_device(self, d_specs, tta):
        """Masks of several device spectrograms (2, bins, T_i), one per track, with the windows of all tracks packed
        into shared forward batches (vr_separate_many); each equals what _mask_device gives for that track alone."""
        ctx = self._ctx()
        d_masks = [torch.empty((2, s.shape[1], s.shape[2]), dtype=torch.float32, device=s.device) for s in d_specs]
        ctx.check(ctx.lib.vr_separate_many(ctx.handle, len(d_specs), _native.ptr_array(d_specs),
                                           _native.i64_array([s.shape[2] for s in d_specs]), 1 if tta else 0,
                                           _native.ptr_array(d_masks), _native.stream_ptr()), 'vr_separate_many')
        if self.postprocess:
            for d_mask in d_masks:
                self._postprocess_device(d_mask)
        return d_masks

    def _postprocess_device(self, d_mask):
        # --postprocess (inference.py:27-30): only T floats leave the device, the run detection of
        # merge_artifacts runs on the host, the fade weights are applied on the device
        ctx = self._ctx()
        T = d_mask.shape[2]
        frame_min = torch.empty(T, dtype=torch.float32, device=d_mask.device)
        ctx.check(ctx.lib.vr_mask_frame_min(ctx.handle, _native.ptr(d_mask), T, _native.ptr(frame_min),
                                            _native.stream_ptr()), 'vr_mask_frame_min')
        weight = torch.from_numpy(spec_utils.artifact_weights(frame_min.cpu().numpy())).to(d_mask.device)
        ctx.check(ctx.lib.vr_mask_apply_weight(ctx.handle, _native.ptr(d_mask), T, _native.ptr(weight),
                                               _native.stream_ptr()), 'vr_mask_apply_weight')

    def _run(self, X_spec, tta):
        X_spec = self._check_spec(X_spec)
        ctx = self._ctx()
        dev = self._dev()
        with torch.cuda.device(dev):
            d_spec = torch.from_numpy(X_spec).to(dev)
            d_mask = self._mask_device(d_spec, tta)
            y = torch.empty_like(d_spec)
            v = torch.empty_like(d_spec)
            ctx.check(ctx.lib.vr_apply_mask(ctx.handle, _native.ptr(d_spec), _native.ptr(d_mask), d_spec.shape[2],
                                            _native.ptr(y), _native.ptr(v), _native.stream_ptr()), 'vr_apply_mask')
            return y.cpu().numpy(), v.cpu().numpy()

    # ---- reference surface --------------------------------------------------------------------------
    def _separate(self, X_spec_pad, roi_size):
        """inference.py:42-68: mask for an already padded + normalised spectrogram."""
        X = self._check_spec(X_spec_pad)
        ctx = self._ctx()
        dev = self._dev()
        patches = (X.shape[2] - 2 * self.offset) // roi_size
        with torch.cuda.device(dev):
            d_spec = torch.from_numpy(X).to(dev)
            one = torch.ones(1, dtype=torch.float32, device=dev)
            d_mask = torch.empty((2, X.shape[1], patches * roi_size), dtype=torch.float32, device=dev)
            ctx.check(ctx.lib.vr_separate_windows(ctx.handle, _native.ptr(d_spec), X.shape[2], _native.ptr(one), 0, 0,
                                                  patches, _native.ptr(d_mask), patches * roi_size, 0, 0,
                                                  _native.stream_ptr()), 'vr_separate_windows')
            return d_mask.cpu().numpy()

    def separate(self, X_spec):
        """inference.py:70-81."""
        return self._run(X_spec, tta=False)

    def separate_tta(self, X_spec):
        """inference.py:83-102."""
        return self._run(X_spec, tta=True)

    # ---- fused device-resident path -----------------------------------------------------------------
    def separate_wave(self, wave, tta=False):
        """float32 (2, L) wave -> (instruments, vocals) float32 (2, hop*(T-1)) waves.

        Equivalent to wave_to_spectrogram -> separate[_tta] -> 2x spectrogram_to_wave
        (inference.py:147,158-161,171,176) without leaving the GPU in between.  ``wave`` may be a numpy
        array (host; copied in and out) or a CUDA tensor (returns CUDA tensors).
        """
        ctx = self._ctx()
        if self.postprocess:
            # staged on the device: STFT -> mask (+ postprocess) -> masked inverse STFT
            dev = self._dev()
            hop, n_fft = self.model.hop_length, self.model.n_fft
            with torch.cuda.device(dev):
                host = not (torch.is_tensor(wave) and wave.is_cuda)
                w = (torch.from_numpy(np.ascontiguousarray(np.asarray(wave, dtype=np.float32))).to(dev) if host
                     else wave.contiguous().float())
                L = w.shape[1]
                T = 1 + L // hop
                d_spec = torch.empty((2, n_fft // 2 + 1, T), dtype=torch.complex64, device=dev)
                ctx.check(ctx.lib.vr_stft(ctx.handle, _native.ptr(w), L, _native.ptr(d_spec), T, None,
                                          _native.stream_ptr()), 'vr_stft')
                d_mask = self._mask_device(d_spec, tta)
                inst = torch.empty((2, hop * (T - 1)), dtype=torch.float32, device=dev)
                voc = torch.empty_like(inst)
                ctx.check(ctx.lib.vr_apply_mask_istft(ctx.handle, _native.ptr(d_spec), _native.ptr(d_mask), T,
                                                      _native.ptr(inst), _native.ptr(voc), _native.stream_ptr()),
                          'vr_apply_mask_istft')
                return (inst.cpu().numpy(), voc.cpu().numpy()) if host else (inst, voc)
        dev = self._dev()
        hop = self.model.hop_length
        with torch.cuda.device(dev):
            if torch.is_tensor(wave) and wave.is_cuda:
                w = wave.contiguous().float()
                L = w.shape[1]
                Lo = hop * (L // hop)
                inst = torch.empty((2, Lo), dtype=torch.float32, device=dev)
                voc = torch.empty((2, Lo), dtype=torch.float32, device=dev)
                ctx.check(ctx.lib.vr_separate_wave(ctx.handle, _native.ptr(w), L, 1 if tta else 0, _native.ptr(inst),
                                                   _native.ptr(voc), _native.stream_ptr()), 'vr_separate_wave')
                return inst, voc
            w = np.ascontiguousarray(np.asarray(wave, dtype=np.float32))
            L = w.shape[1]
            Lo = hop * (L // hop)
            inst = np.empty((2, Lo), dtype=np.float32)
            voc = np.empty((2, Lo), dtype=np.float32)
            ctx.check(ctx.lib.vr_separate_wave_host(ctx.handle, w.ctypes.data, L, 1 if tta else 0, inst.ctypes.data,
                                                    voc.ctypes.data, _native.stream_ptr()), 'vr_separate_wave_host')
            return inst, voc

    def separate_waves(self, waves, tta=False):
        """Several float32 (2, L_i) waves -> a list of (instruments, vocals), one per wave, each what separate_wave
        gives for that wave alone.  The windows of all tracks share the forward batches of ``batchsize`` windows, so
        short clips and the partial last batch of every track do not each pay for a nearly empty forward.  Numpy
        waves give numpy stems, CUDA tensors give CUDA tensors."""
        ctx = self._ctx()
        dev = self._dev()
        hop, n_fft = self.model.hop_length, self.model.n_fft
        with torch.cuda.device(dev):
            host = [not (torch.is_tensor(w) and w.is_cuda) for w in waves]
            d_waves = [torch.from_numpy(np.ascontiguousarray(np.asarray(w, dtype=np.float32))).to(dev) if h
                       else w.contiguous().float() for w, h in zip(waves, host)]
            for w in d_waves:
                if w.dim() != 2 or w.shape[0] != 2:
                    raise ValueError('every wave must have shape (2, L)')
            Ts = [1 + w.shape[1] // hop for w in d_waves]
            inst = [_device_empty((2, hop * (T - 1)), dev) for T in Ts]
            voc = [_device_empty((2, hop * (T - 1)), dev) for T in Ts]
            if self.postprocess:
                # staged on the device: per-track STFT -> packed masks (+ postprocess) -> per-track masked inverse STFT
                d_specs = []
                for w, T in zip(d_waves, Ts):
                    d_spec = torch.empty((2, n_fft // 2 + 1, T), dtype=torch.complex64, device=dev)
                    ctx.check(ctx.lib.vr_stft(ctx.handle, _native.ptr(w), w.shape[1], _native.ptr(d_spec), T, None,
                                              _native.stream_ptr()), 'vr_stft')
                    d_specs.append(d_spec)
                d_masks = self._masks_device(d_specs, tta)
                for d_spec, d_mask, a, b in zip(d_specs, d_masks, inst, voc):
                    ctx.check(ctx.lib.vr_apply_mask_istft(ctx.handle, _native.ptr(d_spec), _native.ptr(d_mask),
                                                          d_spec.shape[2], _native.ptr(a), _native.ptr(b),
                                                          _native.stream_ptr()), 'vr_apply_mask_istft')
            else:
                ctx.check(ctx.lib.vr_separate_waves(ctx.handle, len(d_waves), _native.ptr_array(d_waves),
                                                    _native.i64_array([w.shape[1] for w in d_waves]), 1 if tta else 0,
                                                    _native.ptr_array(inst), _native.ptr_array(voc),
                                                    _native.stream_ptr()), 'vr_separate_waves')
            return [(a.cpu().numpy(), b.cpu().numpy()) if h else (a, b) for a, b, h in zip(inst, voc, host)]


def _device_empty(shape, dev):
    """float32 tensor of `shape` whose data pointer is never NULL (a zero-size tensor has no storage, and the native
    calls reject NULL pointers): one spare element is allocated behind it."""
    n = int(np.prod(shape))
    return torch.empty(n + 1, dtype=torch.float32, device=dev)[:n].view(shape)


MODEL_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'models')
DEFAULT_MODEL_PATH = os.path.join(MODEL_DIR, 'baseline.pth')
# Audio per separate_waves call when several inputs are given: the workspaces grow with the call's total frame count,
# and 2400 s is the 40-minute stream bench.py already runs on one GPU.
GROUP_SECONDS = 2400.0


def _basename(path):
    return os.path.splitext(os.path.basename(path))[0]


def group_by_seconds(items, seconds_of, budget=GROUP_SECONDS):
    """Consecutive items in groups of at most `budget` seconds of audio; an item longer than that is a group alone.
    `items` is consumed lazily, so only one group (and the item that closes it) is held at a time."""
    group, total = [], 0.0
    for item in items:
        sec = seconds_of(item)
        if group and total + sec > budget:
            yield group
            group, total = [], 0.0
        group.append(item)
        total += sec
    if group:
        yield group


def _separate_files(sp, paths, args, device, output_dir):
    """Several inputs with one loaded model: each group of inputs is one separate_waves call."""
    def load_all():
        for path in paths:
            print('loading wave source {}...'.format(path), end=' ')
            X, sr = audio_io.load(path, sr=args.sr, mono=False, dtype=np.float32, device=device)
            print('done')
            if X.ndim == 1:
                # mono to stereo
                X = np.asarray([X, X])
            yield path, X, sr

    for group in group_by_seconds(load_all(), lambda item: item[1].shape[-1] / float(item[2])):
        print('stft of {} wave sources, separation, inverse stft of instruments and vocals...'.format(len(group)),
              end=' ')
        stems = sp.separate_waves([X for _, X, _ in group], tta=args.tta)
        print('done')
        writer = audio_io.AsyncWriter()
        for (path, _, sr), (wave_inst, wave_voc) in zip(group, stems):
            writer.write('{}{}_Instruments.wav'.format(output_dir, _basename(path)), wave_inst.T, sr)
            writer.write('{}{}_Vocals.wav'.format(output_dir, _basename(path)), wave_voc.T, sr)
        writer.join()


def main():
    p = argparse.ArgumentParser()
    p.add_argument('--gpu', '-g', type=int, default=-1)
    p.add_argument('--pretrained_model', '-P', type=str, default=DEFAULT_MODEL_PATH)
    p.add_argument('--input', '-i', required=True, nargs='+')
    p.add_argument('--sr', '-r', type=int, default=44100)
    p.add_argument('--n_fft', '-f', type=int, default=2048)
    p.add_argument('--hop_length', '-H', type=int, default=1024)
    p.add_argument('--batchsize', '-B', type=int, default=4)
    p.add_argument('--cropsize', '-c', type=int, default=256)
    p.add_argument('--output_image', '-I', action='store_true')
    p.add_argument('--tta', '-t', action='store_true')
    p.add_argument('--postprocess', '-p', action='store_true')
    p.add_argument('--output_dir', '-o', type=str, default="")
    args = p.parse_args()
    # several inputs write <basename>_Instruments.wav / _Vocals.wav each: two with the same basename would overwrite
    names = [_basename(path) for path in args.input]
    dup = sorted(set(n for n in names if names.count(n) > 1))
    if dup:
        p.error('inputs with the same basename would overwrite each other\'s output files: {}'.format(', '.join(dup)))

    # unsupported surfaces fail before any heavy work (model load, audio decode, output directory)
    if args.output_image:
        raise NotImplementedError('--output_image (debug JPGs, lib/utils.py) is outside the B200 hot path')
    if not torch.cuda.is_available():
        raise RuntimeError('no CUDA device: the B200 build of vocal-remover has no CPU path')
    if args.gpu < 0:
        # the reference's default (--gpu -1) means CPU; this build has no CPU path
        print('note: --gpu {} selects the CPU in the reference; this build has no CPU path and uses cuda:0'.format(args.gpu))

    print('loading model...', end=' ')
    device = torch.device('cuda:{}'.format(max(args.gpu, 0)))
    model = nets.CascadedNet(args.n_fft, args.hop_length, 32, 128)
    model.load_state_dict(torch.load(args.pretrained_model, map_location='cpu'))
    model.to(device)
    spec_utils.set_device(device.index)
    print('done')

    if len(args.input) > 1:
        sp = Separator(model=model, device=device, batchsize=args.batchsize, cropsize=args.cropsize,
                       postprocess=args.postprocess)
        output_dir = args.output_dir
        if output_dir != "":
            output_dir = output_dir.rstrip('/') + '/'
            os.makedirs(output_dir, exist_ok=True)
        _separate_files(sp, args.input, args, device, output_dir)
        return

    print('loading wave source...', end=' ')
    X, sr = audio_io.load(args.input[0], sr=args.sr, mono=False, dtype=np.float32, device=device)
    basename = os.path.splitext(os.path.basename(args.input[0]))[0]
    print('done')

    if X.ndim == 1:
        # mono to stereo
        X = np.asarray([X, X])

    sp = Separator(
        model=model,
        device=device,
        batchsize=args.batchsize,
        cropsize=args.cropsize,
        postprocess=args.postprocess
    )

    print('validating output directory...', end=' ')
    output_dir = args.output_dir
    if output_dir != "":  # modifies output_dir if theres an arg specified
        output_dir = output_dir.rstrip('/') + '/'
        os.makedirs(output_dir, exist_ok=True)
    print('done')

    print('stft of wave source, separation, inverse stft of instruments and vocals...', end=' ')
    wave_inst, wave_voc = sp.separate_wave(X, tta=args.tta)
    print('done')
    writer = audio_io.AsyncWriter()   # the two stems are encoded and written concurrently
    writer.write('{}{}_Instruments.wav'.format(output_dir, basename), wave_inst.T, sr)
    writer.write('{}{}_Vocals.wav'.format(output_dir, basename), wave_voc.T, sr)
    writer.join()


if __name__ == '__main__':
    main()

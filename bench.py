"""Benchmark of the hot path: seconds-of-audio per second separated (n_fft=2048, hop=1024).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W

One "step" = the whole inference hot path (STFT -> sliding windows -> CascadedNet -> mask -> 2x inverse STFT,
reference inference.py:147-176 minus file I/O) over one synthetic 44.1 kHz stereo track of 240 s per GPU
(BASELINE.json configs[2]; weak scaling: N GPUs process a 240*N s track, windows sharded across ranks,
one mask gather to rank 0 before the overlap-add).  Prints ONE JSON line (rank 0).

  value      device-resident region: wave already in HBM -> both stems in HBM, CUDA-event timed, max over ranks
  e2e        same through the public host-buffer call (pinned host wave -> pinned host stems), copies inside
  roofline   tcgen05 convolution kernel: algorithmic conv FLOPs / CUDA-event kernel time vs measured bf16 peak
  cpu_baseline  the CPU oracle port of the reference path (oracle/), all host threads, bounded sample
  parity     measured max-abs errors of this build on the 10 s golden fixture (tests/golden), before timing
  tta        the same track with --tta (BASELINE configs[3], 163 windows)
  strong_2400s  a fixed 40-minute stream (BASELINE configs[4], 808 windows) on the N GPUs of the run
  cudnn_baseline  the reference's own GPU arithmetic: the oracle's functional restatement of the reference modules on
             cuda:0 through stock PyTorch / cuDNN (TF32 convolutions allowed, the torch default) + torch.stft/istft
  mgpu_check (N > 1) sharded vs single-GPU stems on a 31 s track, with and without --tta; the run fails above 1e-5
--impl reference runs only that CPU arm (the reference itself is Python over librosa and cannot travel to the
GPU box; oracle/ is its restatement, validated against the unmodified reference in tests/).
--dump-outputs DIR writes the stems the last timed step returned (rank 0) as DIR/instruments.npy and DIR/vocals.npy,
float32 (2, n).  Inputs and checkpoint are seeded, so two builds can be compared output for output; stems larger than
the 60 MB budget are sampled at the same seeded, sorted sample positions in every run.
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, 'vocal-remover_b200')
for p in (ROOT, PKG):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

METRIC = 'seconds-of-audio/sec separated (n_fft=2048, hop=1024)'
UNIT = 'audio-s/s'
SR = 44100
SECONDS_PER_GPU = 240.0
CONV_FLOP_PER_WINDOW = 135.714e9   # SURVEY.md 8(d)
# dram__bytes_read.sum + dram__bytes_write.sum summed over the tensor-core convolution launches of the round-2 ncu launch
# list (profiles/r02_launches_bench.csv: 127.3 GB over the 141 windows that bench run pushes through the net; round 1
# measured 0.879 GB with the LSTM channel still interleaved into the skip tensor, 1.225 GB before the decoder upsample
# was fused); the un-fused minimum of SURVEY 8(d) is 1.142 GB/window.
CONV_DRAM_BYTES_PER_WINDOW = 0.903e9
GOLDEN = os.path.join(ROOT, 'tests', 'golden', 'ref_10s_default.npz')
DUMP_BYTES = 60_000_000   # --dump-outputs: all files together, .npy headers included


def measured_peaks():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        return d.get('bf16_tflops_sustained', 1430.1), d.get('hbm_gbs', 6566.1), 'measured (MEASURED_PEAKS.json, sustained)'
    return 1590.0, 6650.0, 'fallback (B200_PROFILING.md)'


class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons through NVML during the timed region."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.stop_flag = False
        self.sm = []
        self.reasons = set()
        self.sm_max = None

    def run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.sm_max = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            names = {
                getattr(nv, 'nvmlClocksEventReasonHwSlowdown', 0x8): 'hw_slowdown',
                getattr(nv, 'nvmlClocksEventReasonHwThermalSlowdown', 0x40): 'hw_thermal_slowdown',
                getattr(nv, 'nvmlClocksEventReasonSwThermalSlowdown', 0x20): 'sw_thermal_slowdown',
                getattr(nv, 'nvmlClocksEventReasonSwPowerCap', 0x4): 'sw_power_cap',
            }
            while not self.stop_flag:
                self.sm.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                try:
                    mask = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                except Exception:
                    mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for bit, name in names.items():
                    if mask & bit:
                        self.reasons.add(name)
                time.sleep(0.05)
        except Exception as e:  # NVML missing: report nothing rather than inventing numbers
            self.reasons.add('nvml_unavailable:%s' % type(e).__name__)

    def summary(self):
        sm = sorted(self.sm)
        return {'sm_mhz': sm[len(sm) // 2] if sm else None, 'sm_max_mhz': self.sm_max, 'reasons': sorted(self.reasons)}


def cpu_reference_arm(steps, warmup, sample_seconds=18.0):
    """The reference path on host cores (oracle port, torch CPU fp32, all threads)."""
    from lib import synth
    from oracle import separator_oracle, stft_oracle
    sd = synth.to_torch_state_dict(synth.make_state_dict())
    wave = synth.sine_mix(sample_seconds)
    # give the CPU path its best shot: torch's intra-op pool does not scale to every core count for these
    # convolutions, so time one window at a few thread counts (<= all host cores) and keep the fastest.
    from oracle import net_oracle
    x1 = torch.rand(1, 2, 1025, 256)
    best, cores = None, os.cpu_count()
    for nt in sorted({min(os.cpu_count(), c) for c in (8, 16, 32, 64, os.cpu_count())}):
        torch.set_num_threads(nt)
        net_oracle.predict_mask(sd, x1)
        t0 = time.perf_counter()
        net_oracle.predict_mask(sd, x1)
        dt = time.perf_counter() - t0
        if best is None or dt < best:
            best, cores = dt, nt
    torch.set_num_threads(cores)

    def one():
        X = stft_oracle.wave_to_spectrogram(wave, 1024, 2048)
        y, v = separator_oracle.separate(sd, X, tta=False, n_fft=2048, cropsize=256, offset=64, batchsize=4)
        stft_oracle.spectrogram_to_wave(y.astype(np.complex64), 1024)
        stft_oracle.spectrogram_to_wave(v.astype(np.complex64), 1024)

    for _ in range(warmup):
        one()
    t0 = time.perf_counter()
    for _ in range(steps):
        one()
    dt = (time.perf_counter() - t0) / max(1, steps)
    return sample_seconds / dt, dt, cores, sample_seconds


def dump_outputs(outdir, stems):
    """Writes every (channels, samples) CUDA tensor of ``stems`` as outdir/<name>.npy (float32).  A stem whose share of
    DUMP_BYTES cannot hold it whole keeps a seeded, sorted sample of its sample positions, all channels."""
    os.makedirs(outdir, exist_ok=True)
    for name, t in stems.items():
        rows, n = t.shape
        cols = min(n, (DUMP_BYTES // len(stems) - 128) // (4 * rows))   # 128: the .npy header
        if cols < n:
            pos = np.sort(np.random.default_rng(0).choice(n, cols, replace=False))
            t = t[:, torch.from_numpy(pos).to(t.device)]
        np.save(os.path.join(outdir, name + '.npy'), t.cpu().numpy())


def workload_text(seconds, n_windows, batch):
    return ('%d s 44.1 kHz stereo synthetic track (240 s per GPU, BASELINE configs[2]), %d windows of cropsize 256, '
            'window batch %d; seeded synthetic checkpoint (lib/synth.py)' % (int(seconds), n_windows, batch))


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    steps = args.steps
    warm = max(1, min(args.warmup, 1))
    val, dt, cores, secs = cpu_reference_arm(steps, warm)
    seconds = args.seconds_per_gpu * max(1, args.gpus)
    T = 1 + int(seconds * SR) // 1024
    n_windows = (T + (128 - T % 128)) // 128
    sample = ('first %.0f s of the synthetic track (%d windows) per step, oracle port of inference.py:147-176 on CPU '
              'fp32, batchsize 4; %d timed steps after %d warm-up' % (secs, int(np.ceil((1 + secs * SR // 1024) / 128)),
                                                                      steps, warm))
    line = {
        'impl': 'reference', 'metric': METRIC, 'value': val, 'unit': UNIT, 'n_gpus': args.gpus, 'steps': steps,
        'warmup': warm, 'ms_per_step': dt * 1e3, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
        'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': workload_text(seconds, n_windows, args.batch),
                   'reference_arm': 'CPU fp32, batchsize 4 (reference default); each step is a bounded sample of this '
                                    'workload, see cpu_baseline.sample'},
        'cpu_baseline': {'value': val, 'unit': UNIT, 'cores': cores, 'kind': 'port', 'sample': sample},
        'e2e': {'value': val, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
    }
    print(json.dumps(line))


def write_layer_table(ctx, path):
    """Per-layer CUDA-event times of the profiled step (vr_profile_dump), summed over its launches."""
    import collections
    import ctypes
    need = ctypes.c_int64(0)
    ctx.check(ctx.lib.vr_profile_dump(ctx.handle, None, 0, ctypes.byref(need)), 'vr_profile_dump')
    buf = ctypes.create_string_buffer(need.value)
    ctx.check(ctx.lib.vr_profile_dump(ctx.handle, buf, need.value, None), 'vr_profile_dump')
    agg = collections.OrderedDict()
    for ln in buf.value.decode().splitlines():
        name, n, h, w, tc, ms, gf = ln.split()
        key = (name, int(h), int(w), int(tc))
        a = agg.setdefault(key, [0, 0.0, 0.0])
        a[0] += 1
        a[1] += float(ms)
        a[2] += float(gf)
    total = sum(a[1] for a in agg.values()) or 1.0
    with open(path, 'w') as f:
        f.write('layer\tHout\tWout\ttensor_core\tlaunches\tms\tshare\tGFLOP\tTFLOP/s\n')
        for (name, h, w, tc), (cnt, ms, gf) in agg.items():
            f.write('%s\t%d\t%d\t%d\t%d\t%.4f\t%.4f\t%.3f\t%.1f\n' % (name, h, w, tc, cnt, ms, ms / total, gf,
                                                                      gf / ms if ms > 0 else 0.0))


def parity_block(sp, dev):
    """Measured errors of THIS build against the golden tensors the unmodified reference produced for the 10 s input
    (tests/golden/ref_10s_default.npz, oracle/make_golden.py): mask, --tta mask, masked spectrogram in normalised units."""
    import inference
    from lib import spec_utils, synth
    if not os.path.exists(GOLDEN):
        return None
    g = np.load(GOLDEN)
    wave = synth.sine_mix(10.0)
    X = spec_utils.wave_to_spectrogram(wave, 1024, 2048)
    d_spec = torch.from_numpy(X).to(dev)
    m = sp._mask_device(d_spec, False).cpu().numpy()
    mt = sp._mask_device(d_spec, True).cpu().numpy()
    y, v = sp.separate(X)
    absmax = float(g['absmax'])
    return {
        'input': '10 s synthetic sine mix, 4 windows (BASELINE configs[1]); golden = unmodified reference on CPU fp32',
        'gate': 1e-3,
        'mask_max_abs_vs_golden_10s': float(np.abs(m[:, ::8, :] - g['mask_sub']).max()),
        'tta_mask_max_abs_vs_golden_10s': float(np.abs(mt[:, ::8, :] - g['mask_tta_sub']).max()),
        'y_spec_max_abs_over_absmax_vs_golden_10s': float(np.abs(y[:, ::16, :] - g['y_sub']).max() / absmax),
        'parity_unpinned': ['stft', 'istft'],
        'parity_unpinned_note': 'librosa (the reference\'s STFT/iSTFT) is absent offline; the restatement is cross-checked '
                                'against torch.stft and scipy.signal (tests/test_oracle_stft.py), not against librosa',
    }


def cudnn_baseline_arm(dev, wave, batch, steps=2):
    """The reference's GPU path (inference.py:124-132 with --gpu 0) restated with stock PyTorch on cuda:0: torch.stft,
    the oracle's functional CascadedNet (F.conv2d -> cuDNN with TF32 allowed, nn.LSTM's fused kernel), mask multiply,
    torch.istft; windows batched like the product arm.  A baseline leg (like cpu_baseline), never the product path."""
    from lib import synth
    from oracle import net_oracle
    sd = net_oracle.to_device(synth.to_torch_state_dict(synth.make_state_dict()), dev)
    tf32 = bool(torch.backends.cudnn.allow_tf32)
    w = torch.from_numpy(wave).to(dev)
    win = torch.hann_window(2048, periodic=True, device=dev)
    roi, off, crop = 128, 64, 256

    def one():
        X = torch.stft(w, 2048, 1024, window=win, center=True, pad_mode='constant', return_complex=True)   # (2, 1025, T)
        T = X.shape[2]
        pad_r = roi - (T % roi) + off
        Xp = torch.nn.functional.pad(X, (off, pad_r))
        mag = Xp.abs() / X.abs().max()
        n = (Xp.shape[2] - 2 * off) // roi
        masks = []
        for i in range(0, n, batch):
            xb = torch.stack([mag[:, :, j * roi:j * roi + crop] for j in range(i, min(n, i + batch))])
            mb = net_oracle.predict_mask(sd, xb, 2048, off)
            masks.append(torch.cat(list(mb), dim=2))
        mask = torch.cat(masks, dim=2)[:, :, :T]
        y, v = X * mask, X * (1 - mask)
        return (torch.istft(y, 2048, 1024, window=win, center=True), torch.istft(v, 2048, 1024, window=win, center=True))

    with torch.no_grad():
        one()
        torch.cuda.synchronize(dev)
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for _ in range(steps):
            one()
        ev1.record()
        torch.cuda.synchronize(dev)
    ms = ev0.elapsed_time(ev1) / steps
    secs = wave.shape[1] / SR
    del sd
    torch.cuda.empty_cache()
    return {'value': secs / (ms * 1e-3), 'unit': UNIT, 'ms_per_step': ms, 'steps': steps, 'window_batch': batch,
            'tf32_convolutions': tf32,
            'what': 'torch.stft -> functional CascadedNet on cuDNN (oracle/net_oracle on cuda:0, fused nn.LSTM kernel) -> '
                    'mask -> torch.istft x2 on the same %d s track, device-resident, CUDA-event timed' % int(secs)}


def mgpu_check(sp, dev, world, rank):
    """Sharded vs single-GPU stems on a 31 s track (every rank computes the single-GPU reference itself), with and
    without --tta.  Returns the max abs differences on rank 0."""
    from lib import synth
    from lib import distributed as vr_dist
    wave = torch.from_numpy(synth.sine_mix(31.0)).to(dev)
    out = {}
    for tta, key in ((False, 'max_diff'), (True, 'tta_max_diff')):
        ref_inst, ref_voc = sp.separate_wave(wave, tta=tta)
        for _ in range(2):   # twice: cached buffers / barriers must be reusable
            inst, voc = vr_dist.separate_wave(sp, wave, tta=tta, world=world, rank=rank)
        if rank == 0:
            out[key] = max((inst - ref_inst).abs().max().item(), (voc - ref_voc).abs().max().item())
    return out


def run_gpu(args):
    import torch.distributed as dist
    import inference
    from lib import _native, nets, synth
    from lib import distributed as vr_dist

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    assert torch.cuda.is_available(), 'bench.py needs a GPU (no CPU path for the product)'
    dev = torch.device('cuda', local)
    torch.cuda.set_device(dev)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    seconds = args.seconds_per_gpu * world
    model = nets.CascadedNet(2048, 1024, 32, 128)
    model.load_state_dict(synth.to_torch_state_dict(synth.make_state_dict()))
    model.to(dev)
    sp = inference.Separator(model, dev, args.batch, 256, False)
    wave = synth.sine_mix(seconds)
    L = wave.shape[1]
    T = 1 + L // 1024
    n_windows = (T + (128 - T % 128)) // 128
    d_wave = torch.from_numpy(wave).to(dev)
    h_wave = torch.from_numpy(wave).pin_memory()
    ctx = sp._ctx()

    def step_device():
        return vr_dist.separate_wave(sp, d_wave, tta=False, world=world, rank=rank)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, per_step=None, last=None):
        """K steps bracketed by barrier + synchronize, CUDA events on the launching stream, max over ranks.  per_step
        (a list) additionally receives every step's own duration (events between steps cost nothing measurable);
        last (a list) receives what the last step returned."""
        barrier()
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
        evs[0].record()
        out = None
        for i in range(steps):
            out = None   # every step starts with the previous step's output released, as when it is not kept
            out = fn()
            evs[i + 1].record()
        barrier()
        if last is not None:
            last.append(out)
        ms = evs[0].elapsed_time(evs[steps])
        each = [evs[i].elapsed_time(evs[i + 1]) for i in range(steps)]
        if world > 1:
            t = torch.tensor([ms] + each, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms, each = t[0].item(), t[1:].tolist()
        if per_step is not None:
            per_step.extend(each)
        return ms

    # measured errors of this build on the 10 s golden fixture, before any timing (single-GPU path of this rank)
    parity = parity_block(sp, dev) if rank == 0 else None
    check = None
    if world > 1:
        check = mgpu_check(sp, dev, world, rank)

    for _ in range(args.warmup):
        step_device()
    sampler = ClockSampler(local)
    sampler.start()
    launches0 = ctx.launch_count()
    per_step = []
    last = []
    ms = timed(step_device, args.steps, per_step, last)
    launches = ctx.launch_count() - launches0
    sampler.stop_flag = True
    sampler.join(timeout=2)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, dict(zip(('instruments', 'vocals'), last[0])))
    del last
    ms_step = ms / args.steps
    value = seconds / (ms_step * 1e-3)
    ms_median = sorted(per_step)[len(per_step) // 2]

    # ---- roofline pass, right after the timed steps (same clocks / thermal state): one more step of the same
    # workload with a CUDA event pair around every convolution launch (recorded inside the library on the launching
    # stream); the two band streams are serialised while profiling so each pair brackets exactly one kernel.
    import ctypes
    prof = (ctypes.c_double * 6)()
    ctx.check(ctx.lib.vr_profile_enable(ctx.handle, 1), 'vr_profile_enable')
    prof_ms = timed(step_device, 1)
    ctx.check(ctx.lib.vr_profile_read(ctx.handle, prof), 'vr_profile_read')
    if args.layers and rank == 0:
        write_layer_table(ctx, args.layers)
    ctx.check(ctx.lib.vr_profile_enable(ctx.handle, 0), 'vr_profile_enable')

    # ---- BASELINE configs[3]: the same track with --tta (second, half-window-shifted pass; inference.py:83-102) ----
    def step_tta():
        return vr_dist.separate_wave(sp, d_wave, tta=True, world=world, rank=rank)

    tta_steps = max(1, min(args.steps, 3))
    step_tta()
    step_tta()
    tta_ms = timed(step_tta, tta_steps) / tta_steps

    # ---- BASELINE configs[4]: a fixed 40-minute stream on the N GPUs of this run (strong scaling) ----
    strong = None
    if not args.no_strong and args.seconds_per_gpu >= SECONDS_PER_GPU:
        reps = int(round(2400.0 / SECONDS_PER_GPU))
        base = d_wave[:, :int(SECONDS_PER_GPU * SR)]
        d_long = base.repeat(1, reps).contiguous()
        Tl = 1 + d_long.shape[1] // 1024

        def step_long():
            return vr_dist.separate_wave(sp, d_long, tta=False, world=world, rank=rank)

        step_long()   # two warm-up calls: the multi-GPU path alternates between two sets of shared stem buffers,
        step_long()   # each allocated (and IPC-mapped) on its first use
        long_steps = 2
        long_ms = timed(step_long, long_steps) / long_steps
        strong = {'value': 2400.0 / (long_ms * 1e-3), 'unit': UNIT, 'ms_per_step': long_ms, 'steps': long_steps,
                  'seconds_of_audio': 2400, 'windows': (Tl + (128 - Tl % 128)) // 128, 'n_gpus': world,
                  'note': 'the first 240 s of the synthetic track repeated 10 times; the same stream at every N, so '
                          'value(N) / value(1) is the strong-scaling speed-up'}
        del d_long
        torch.cuda.empty_cache()

    # ---- end to end through the public host-buffer API (pinned host wave -> pinned host stems) ----
    Lo = 1024 * (T - 1)
    # N > 1: one page-locked buffer shared by all ranks (POSIX shared memory registered with CUDA on every rank), so that
    # each rank's device-to-host copy lands its span in the SAME buffer and the stems come out assembled; falls back to
    # per-rank pinned buffers (spans not assembled) when the node refuses it.
    shared_host = None
    if world > 1:
        try:
            shared_host = vr_dist.SharedHostBuffer.create((2, 2, Lo), world, rank)
        except Exception as exc:   # never let the optional buffer take the bench down
            print('bench: shared host buffer unavailable (%s); per-rank pinned buffers' % exc, file=sys.stderr)
            shared_host = None
    if shared_host is not None:
        h_inst, h_voc = shared_host.tensor[0], shared_host.tensor[1]
    else:
        h_inst = torch.empty((2, Lo), dtype=torch.float32).pin_memory()
        h_voc = torch.empty((2, Lo), dtype=torch.float32).pin_memory()

    def step_e2e():
        vr_dist.separate_wave_host(sp, h_wave, h_inst, h_voc, tta=False, world=world, rank=rank)

    step_e2e()
    e2e_steps = max(1, min(args.steps, 5))
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        step_e2e()
    barrier()
    e2e_s = (time.perf_counter() - t0) / e2e_steps
    if world > 1:
        t = torch.tensor([e2e_s], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = t.item()
    # the stems assembled in the shared host buffer against the device-resident single-GPU result of the same track
    assembled_diff = None
    if shared_host is not None:
        if rank == 0:
            i1, v1 = vr_dist.separate_wave(sp, d_wave, tta=False, world=1, rank=0)
            assembled_diff = max((h_inst - i1.cpu()).abs().max().item(), (h_voc - v1.cpu()).abs().max().item())
            del i1, v1
        barrier()
        h_inst = h_voc = None
        shared_host.close(world)

    peak_tf, peak_hbm, peak_src = measured_peaks()
    tc_ms, tc_flops, tc_n, cc_ms, cc_flops, cc_n = [float(x) for x in prof]
    roof = None
    if tc_n > 0:
        ach = tc_flops / (tc_ms * 1e-3) / 1e12
        roof = {'bound': 'tensor', 'kernel': 'conv_tc_rows_kernel + conv_tc_kernel (tcgen05 implicit-GEMM conv family, '
                          'bf16x3 split precision)',
                'achieved': ach, 'peak': peak_tf, 'unit': 'TFLOP/s', 'frac': ach / peak_tf,
                'traffic': CONV_DRAM_BYTES_PER_WINDOW * n_windows / world / max(1.0, tc_n),
                'traffic_note': 'average DRAM bytes per convolution launch = 0.903 GB per window (ncu, '
                                'profiles/r02_launches_bench.csv) x windows per rank / launches',
                'peak_source': peak_src,
                'note': 'achieved = algorithmic conv FLOPs (real channel counts, 1x per product; the kernel issues 3 '
                        'bf16 MMA passes per product) of %d launches / their summed CUDA-event time %.2f ms on rank '
                        '0 over one profiled step of the same workload (%.1f ms, band streams serialised); kernel '
                        'share of that step = %.2f' % (int(tc_n), tc_ms, prof_ms, tc_ms / prof_ms),
                'cuda_core_conv': {'ms': cc_ms, 'launches': int(cc_n),
                                   'tflops': (cc_flops / (cc_ms * 1e-3) / 1e12) if cc_ms > 0 else None}}
    line = None
    if check is not None:
        flag = torch.tensor([1.0 if (rank == 0 and any(not (v <= 1e-5) for v in check.values())) else 0.0], device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MAX)
        if flag.item() > 0:   # every rank leaves together
            if rank == 0:
                print(json.dumps({'error': 'multi-GPU check failed (sharded stems differ from the single-GPU stems)',
                                  'mgpu_check': check}))
            dist.destroy_process_group()
            sys.exit(3)
    if rank == 0:
        cudnn = None
        if not (args.no_cudnn_baseline or world > 1):   # like the CPU arm: reported at N=1 only
            cudnn = cudnn_baseline_arm(dev, wave, args.batch)
        if args.no_cpu_baseline or world > 1:   # the CPU arm is reported at N=1 only
            cpu_val, cores, secs = None, 0, 0.0
        else:
            cpu_val, cpu_dt, cores, secs = cpu_reference_arm(1, 1, 12.0)
        line = {
            'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup,
            'ms_per_step': ms_step, 'ms_per_step_median': ms_median, 'value_at_median': seconds / (ms_median * 1e-3),
            'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
            'dtype': 'bf16x3 (split-bf16 operands hi+lo, 3 tcgen05 passes, fp32 accumulate); fft/lstm fp32',
            'data': 'synthetic',
            'config': {'workload': workload_text(seconds, n_windows, args.batch),
                       'l2': 'no flush needed: per-step working set (spectrogram %.0f MB + activations > 1 GB) exceeds '
                             'the 126 MB L2' % (2 * 1025 * T * 8 / 1e6),
                       'parallelism': ('window-sharded x%d: STFT / net / inverse STFT per rank span, 4-byte max all-reduce, 8 KB '
                                       'halo mask frame, overlap-add kernel stores its span into rank 0 HBM over NVLink'
                                       % world) if world > 1 else 'single GPU'},
            'clocks': sampler.summary(),
            'e2e': {'value': seconds / e2e_s, 'unit': UNIT, 'h2d_bytes_per_step': int(2 * L * 4),
                    'd2h_bytes_per_step': int(2 * 2 * Lo * 4),
                    'note': 'bytes are totals over all ranks; with N > 1 every rank moves only its own slice of the '
                            'wave / stems over its own PCIe link (lib/distributed.py, sharded mode)',
                    'assembled': (None if world == 1 else
                                  {'shared_host_buffer': assembled_diff is not None, 'max_diff_vs_single_gpu': assembled_diff,
                                   'what': 'every rank copies its span into ONE page-locked buffer (POSIX shared memory '
                                           'registered with CUDA); compared on rank 0 with the single-GPU stems'})},
            'gpu_launches': int(launches),
            'parity': parity,
            'mgpu_check': check,
            'tta': {'value': seconds / (tta_ms * 1e-3), 'unit': UNIT, 'ms_per_step': tta_ms, 'steps': tta_steps,
                    'windows': 2 * n_windows + 1, 'config': 'BASELINE configs[3]: the same track with --tta'},
            'strong_2400s': strong,
            'cudnn_baseline': cudnn,
            'roofline': roof,
            'cpu_baseline': {'value': cpu_val, 'unit': UNIT, 'cores': cores, 'kind': 'port',
                             'sample': 'first %.0f s of the same track through the CPU oracle port (oracle/), 1 step '
                                       'after 1 warm-up; thread count = fastest of {8,16,32,64,all} host cores on a '
                                       'one-window probe' % secs},
        }
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', type=str, default='b200')
    ap.add_argument('--batch', type=int, default=27, help='windows per forward launch sequence (240 s = 81 windows = 3 x 27)')
    ap.add_argument('--layers', type=str, default='', help='write the per-layer conv timing table of the profiled '
                                                           'step to this file')
    ap.add_argument('--no-cpu-baseline', action='store_true', help='skip the CPU arm (profiling runs only)')
    ap.add_argument('--no-cudnn-baseline', action='store_true', help='skip the stock-PyTorch / cuDNN GPU arm')
    ap.add_argument('--no-strong', action='store_true', help='skip the 40-minute strong-scaling sub-record')
    ap.add_argument('--seconds-per-gpu', type=float, default=SECONDS_PER_GPU,
                    help='track length per GPU (default 240 s = BASELINE configs[2]; shorter only for profiling)')
    ap.add_argument('--dump-outputs', type=str, default='', metavar='DIR',
                    help='write the stems of the last timed step to DIR/instruments.npy and DIR/vocals.npy')
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error('--steps must be >= 1 and --warmup >= 0')
    if args.impl == 'reference':
        if args.dump_outputs:
            ap.error('--dump-outputs writes the stems of the GPU path; --impl reference times a CPU sample')
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == '__main__':
    main()

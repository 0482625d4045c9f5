"""Packed several-track separation against a loop of single-track calls, on one GPU.

Arm 'loop' calls Separator.separate_wave once per track; arm 'packed' makes one Separator.separate_waves call for all
of them, so the windows of all tracks share forward batches.  Seeded synthetic checkpoint (lib/synth.py), window batch
27, waves resident on the device.  Each arm is timed with CUDA events around the whole arm, ending in a synchronise;
every shape is warmed up first, then the arms alternate over --reps repetitions (median and min / max reported).

    python profiles/tools/packed_tracks.py --out packed_tracks.json   # without --out the JSON goes to stdout
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
for p in (ROOT, os.path.join(ROOT, 'vocal-remover_b200')):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

SR = 44100


def workloads():
    rng = np.random.default_rng(2026)
    return [
        ('48 clips x 3 s', [3.0] * 48),
        ('24 clips of 5-60 s', [float(x) for x in np.round(rng.uniform(5, 60, 24), 2)]),
        ('6 tracks of 150-300 s', [float(x) for x in np.round(rng.uniform(150, 300, 6), 2)]),
        ('4 tracks x 240 s (control: no partial batch)', [240.0] * 4),
    ]


def gpu_info():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True)
    line = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else ''
    parts = [x.strip() for x in line.split(',')] if line else []
    return {'name': parts[0] if parts else torch.cuda.get_device_name(0),
            'power_limit': parts[1] if len(parts) > 1 else 'unknown',
            'max_sm_clock': parts[2] if len(parts) > 2 else 'unknown'}


def timed(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    out = fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / 1e3, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=5)
    ap.add_argument('--batch', type=int, default=27)
    ap.add_argument('--out', default=None, help='JSON result file (default: print it)')
    args = ap.parse_args()
    assert torch.cuda.is_available(), 'this measurement needs a GPU'
    import inference
    from lib import nets, synth
    dev = torch.device('cuda:0')
    model = nets.CascadedNet(2048, 1024, 32, 128)
    model.load_state_dict(synth.to_torch_state_dict(synth.make_state_dict()))
    model.to(dev)
    sp = inference.Separator(model, dev, args.batch, 256, False)
    ctx = sp._ctx()
    result = {'gpu': gpu_info(), 'batch': args.batch, 'cropsize': 256, 'reps': args.reps,
              'checkpoint': 'lib/synth.make_state_dict() (seeded)', 'workloads': []}
    for wi, (name, secs) in enumerate(workloads()):
        waves = [torch.from_numpy(synth.sine_mix(s, seed=100 * wi + k)).to(dev) for k, s in enumerate(secs)]
        audio = float(sum(w.shape[1] for w in waves)) / SR

        def loop():
            return [sp.separate_wave(w) for w in waves]

        def packed():
            return sp.separate_waves(waves)

        # warm-up of every shape, and the outputs and launch counts of both arms
        n0 = ctx.launch_count()
        ref = loop()
        n_loop = ctx.launch_count() - n0
        n0 = ctx.launch_count()
        got = packed()
        n_packed = ctx.launch_count() - n0
        torch.cuda.synchronize()
        diff = max(max((a - ra).abs().max().item(), (b - rb).abs().max().item()) for (a, b), (ra, rb) in zip(got, ref))
        del ref, got
        times = {'loop': [], 'packed': []}
        for r in range(args.reps):
            for arm, fn in ((('loop', loop), ('packed', packed)) if r % 2 == 0 else (('packed', packed), ('loop', loop))):
                t, out = timed(fn)
                del out
                times[arm].append(t)
        rec = {'workload': name, 'tracks': len(secs), 'audio_seconds': round(audio, 3),
               'track_seconds': secs, 'max_abs_diff_stems': diff,
               'launches': {'loop': n_loop, 'packed': n_packed}}
        for arm in ('loop', 'packed'):
            ts = sorted(times[arm])
            rec[arm] = {'seconds': ts, 'median_s': float(np.median(ts)),
                        'audio_s_per_s_median': audio / float(np.median(ts)),
                        'audio_s_per_s_min': audio / ts[-1], 'audio_s_per_s_max': audio / ts[0]}
        rec['speedup_median'] = rec['loop']['median_s'] / rec['packed']['median_s']
        result['workloads'].append(rec)
        print('%-46s loop %8.1f  packed %8.1f audio-s/s  x%.3f  diff %.2g  launches %d / %d' % (
            name, rec['loop']['audio_s_per_s_median'], rec['packed']['audio_s_per_s_median'], rec['speedup_median'],
            diff, n_loop, n_packed), flush=True)
        del waves
        torch.cuda.empty_cache()
    if args.out is None:
        print(json.dumps(result, indent=1))
        return
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result['gpu']))


if __name__ == '__main__':
    main()

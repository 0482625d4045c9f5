"""inference.py with several -i inputs, on the host: grouping by seconds of audio, the single-input path, and the
rejection of inputs whose output files would collide.  The model, the audio loader and the Separator are replaced by
fakes, so nothing here needs a GPU (tests/test_gpu_multitrack.py runs the real thing)."""
import sys

import numpy as np
import pytest


def test_group_by_seconds_keeps_order_and_budget():
    import inference
    groups = list(inference.group_by_seconds([1000, 1000, 500, 2500, 10, 2400, 0.5], lambda s: s))
    assert groups == [[1000, 1000], [500], [2500], [10], [2400], [0.5]]
    assert list(inference.group_by_seconds([], lambda s: s)) == []
    assert inference.GROUP_SECONDS == 2400.0
    # 48 clips of 60 s: 40 per group
    assert [len(g) for g in inference.group_by_seconds([60.0] * 48, lambda s: s)] == [40, 8]


class _Calls(object):
    def __init__(self):
        self.model_built = 0
        self.single = []
        self.packed = []
        self.written = []


@pytest.fixture
def fake_cli(monkeypatch):
    """inference.main with every heavy dependency faked; audio length per path = its number before '.wav' seconds."""
    import inference
    calls = _Calls()
    sr = 100

    class FakeModel(object):
        def __init__(self, *a):
            calls.model_built += 1

        def load_state_dict(self, sd):
            pass

        def to(self, dev):
            return self

    class FakeSeparator(object):
        def __init__(self, **kw):
            pass

        def separate_wave(self, X, tta=False):
            calls.single.append(X.shape[1])
            return X * 0.25, X * 0.75

        def separate_waves(self, waves, tta=False):
            calls.packed.append([w.shape[1] for w in waves])
            return [(w * 0.25, w * 0.75) for w in waves]

    class FakeWriter(object):
        def write(self, path, data, rate):
            calls.written.append((path, data.shape, rate))

        def join(self):
            pass

    def fake_load(path, sr=None, **kw):
        seconds = float(path.split('/')[-1].split('_')[-1][:-4])
        return np.ones((2, int(seconds * sr)), dtype=np.float32), sr

    monkeypatch.setattr(inference.torch.cuda, 'is_available', lambda: True)
    monkeypatch.setattr(inference.torch, 'load', lambda *a, **k: {})
    monkeypatch.setattr(inference.nets, 'CascadedNet', FakeModel)
    monkeypatch.setattr(inference.spec_utils, 'set_device', lambda i: None)
    monkeypatch.setattr(inference.audio_io, 'load', fake_load)
    monkeypatch.setattr(inference.audio_io, 'AsyncWriter', FakeWriter)
    monkeypatch.setattr(inference, 'Separator', FakeSeparator)

    def run(*argv):
        monkeypatch.setattr(sys, 'argv', ['inference.py', '-r', str(sr)] + list(argv))
        inference.main()
        return calls
    return run, calls


def test_single_input_takes_the_single_track_path(fake_cli, tmp_path):
    run, _ = fake_cli
    calls = run('-i', 'dir/a_3.wav', '-o', str(tmp_path))
    assert calls.single == [300] and calls.packed == []
    assert [w[0] for w in calls.written] == [str(tmp_path) + '/a_3_Instruments.wav', str(tmp_path) + '/a_3_Vocals.wav']


def test_several_inputs_are_grouped_into_packed_calls(fake_cli, tmp_path):
    run, _ = fake_cli
    calls = run('-i', 'x/a_1000.wav', 'y/b_1000.wav', 'c_500.wav', 'd_2500.wav', 'e_3.wav', '-o', str(tmp_path))
    assert calls.model_built == 1 and calls.single == []
    assert calls.packed == [[100000, 100000], [50000], [250000], [300]]
    names = [w[0].split('/')[-1] for w in calls.written]
    expect = []
    for b in ('a_1000', 'b_1000', 'c_500', 'd_2500', 'e_3'):
        expect += [b + '_Instruments.wav', b + '_Vocals.wav']
    assert names == expect
    assert all(w[0].startswith(str(tmp_path) + '/') for w in calls.written)
    assert calls.written[0][1] == (100000, 2) and calls.written[0][2] == 100


def test_duplicate_basenames_are_rejected_before_the_model_loads(fake_cli, capsys):
    run, calls = fake_cli
    with pytest.raises(SystemExit):
        run('-i', 'x/song_3.wav', 'y/other_2.wav', 'z/song_3.flac')
    assert calls.model_built == 0 and calls.single == [] and calls.packed == []
    assert 'song_3' in capsys.readouterr().err

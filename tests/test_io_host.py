"""host side of SURVEY.md 8f rank 4: the SigMF (npy flavour) reader, against the reference's own
reader (or, where the reference is not installed, the digest recorded from that comparison) and against
the file contents"""
import json

import numpy as np
import pytest

from _reference_digests import recorded
from iqwaveform_b200 import io as bio
from oracle import ref_shim


def _write_capture(tmp_path, n_seg=3, seg_len=1000, ntia=False):
    rng = np.random.default_rng(3)
    x = (rng.standard_normal(n_seg * seg_len) + 1j * rng.standard_normal(n_seg * seg_len)).astype(np.complex64)
    meta = {
        'global': {'core:sample_rate': 15.36e6, 'core:datatype': 'cf32_le'},
        'captures': [{'core:sample_start': i * seg_len, 'core:frequency': 3.55e9 + 10e6 * i,
                      'core:datetime': f'2024-01-01T00:00:0{i}Z'} for i in range(n_seg)],
        'annotations': [{'ntia-core:annotation_type': 'CalibrationAnnotation', 'ntia-sensor:temperature': 21.5,
                         'ntia-sensor:noise_figure_sensor': 4.2, 'ntia-sensor:gain_preselector': 30.0}] if ntia else [],
    }
    path = tmp_path / 'capture.sigmf-meta'
    path.write_text(json.dumps(meta))
    np.save(tmp_path / 'capture.sigmf-data.npy', x)
    return path, x, meta


def test_read_sigmf_matches_the_file(tmp_path):
    path, x, meta = _write_capture(tmp_path)
    segs, freqs, Ts, cal = bio.read_sigmf(path)
    assert len(segs) == 3 and all(s.shape == (1000,) for s in segs)
    assert np.array_equal(np.concatenate(segs), x)
    assert np.array_equal(freqs, [3.55e9, 3.56e9, 3.57e9]) and Ts == 1 / 15.36e6 and cal == {}
    stacked, _, _, _ = bio.read_sigmf(path, stack=True)
    assert stacked.shape == (1000, 3) and np.array_equal(stacked[:, 1], x[1000:2000])
    mapped, _, _, _ = bio.read_sigmf(path, mmap=True)
    assert np.array_equal(np.concatenate(mapped), x)
    _, _, Ts2, _ = bio.read_sigmf(path, force_sample_rate=1e6)
    assert Ts2 == 1e-6
    with pytest.raises(TypeError):
        bio.read_sigmf(path, sigmf_data_ext='.bin')
    with pytest.raises(LookupError):
        bio.read_sigmf(path, ntia_extensions=True)          # no calibration annotation


def test_ntia_calibration_scaling(tmp_path, capsys):
    path, x, _ = _write_capture(tmp_path, ntia=True)
    segs, _, _, cal = bio.read_sigmf(path, ntia_extensions=True)
    assert cal == {'ambient temperature (K)': 21.5 + 273.15, 'noise figure (dB)': 4.2, 'gain (dB)': 30.0}
    np.testing.assert_allclose(np.concatenate(segs), x / np.sqrt(1000.0 * 2 / 50), rtol=1e-6)


def test_reader_equals_the_reference(tmp_path):
    got, meta = [], []          # ordered by (ntia, stack)
    for ntia in (False, True):
        path, _, _ = _write_capture(tmp_path, ntia=ntia)
        got += [bio.read_sigmf(path, stack=stack, ntia_extensions=ntia) for stack in (False, True)]
        meta.append(bio.read_sigmf_metadata(path, ntia=ntia))
    ref = ref_shim.load()
    if recorded(ref, got, meta):
        return
    import importlib
    rio = importlib.import_module('iqwaveform.io')
    for ntia in (False, True):
        path, x, _ = _write_capture(tmp_path, ntia=ntia)
        for stack in (False, True):
            a = got[2 * ntia + stack]
            b = rio.read_sigmf(path, stack=stack, ntia_extensions=ntia)
            if stack:
                assert np.array_equal(a[0], b[0])
            else:
                assert all(np.array_equal(p, q) for p, q in zip(a[0], b[0]))
            assert np.array_equal(a[1], b[1]) and a[2] == b[2] and a[3] == b[3]
        fa, ta, ra, ca = meta[int(ntia)]
        fb, tb, rb, cb = rio.read_sigmf_metadata(path, ntia=ntia)
        assert {int(k): float(v) for k, v in fb.items()} == fa and {int(k): v for k, v in tb.items()} == ta
        assert ra == rb and ca == cb


def test_waveform_to_frame():
    import pandas as pd
    x = np.arange(12, dtype=np.complex64).reshape(6, 2)
    df = bio.waveform_to_frame(x, 0.5, columns=['a', 'b'], column_name='ch')
    assert isinstance(df, pd.DataFrame) and df.columns.name == 'ch' and df.index.name == 'Time elapsed (s)'
    assert np.array_equal(df.index.values, np.arange(6) * 0.5)
    s = bio.waveform_to_frame(x[:, 0], 0.5)
    assert isinstance(s, pd.Series) and len(s) == 6
    with pytest.raises(TypeError):
        bio.waveform_to_frame(np.zeros((2, 2, 2)), 1.0)

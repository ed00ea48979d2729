"""CPU tests: the persistent snowflake-table cache (reference file naming), the north-star call shape's prefix
derivation, the DenseDataset hook's defaults, and the sensor table against the reference's YAML."""
import json
import os

import numpy as np
import pytest

from lidar_snow_sim_b200.snowfall import sampling as S


def test_table_cache_uses_the_reference_file_names(tmp_path, gold_dir):
    kat = json.load(open(os.path.join(gold_dir, 'kat_scalars.json')))['scalars']['2.5_1.6']
    tabs, prefix, src = S.load_or_sample_table_set('gunn', 2.5, 1.6, directory=tmp_path, write=True, seed=1000)
    assert src == 'sampled' and len(tabs) == 64
    assert prefix == f"gunn_{kat['rainfall_rate']}_{kat['occupancy']}"                 # precompute.py:101
    names = sorted(p.name for p in tmp_path.iterdir())
    assert names == sorted(f'{prefix}_{k}.npy' for k in range(1, 65))                  # sampling.py:344
    again, _, src2 = S.load_or_sample_table_set('gunn', 2.5, 1.6, directory=tmp_path)
    assert src2 == 'files' and all(np.array_equal(a, b) for a, b in zip(tabs, again))
    assert all(np.array_equal(a, b) for a, b in zip(S.load_table_set(prefix, tmp_path), tabs))
    # existing files are never overwritten (sampling.py:346-347)
    np.save(str(tmp_path / f'{prefix}_7.npy'), np.zeros((1, 3)))
    os.remove(tmp_path / f'{prefix}_8.npy')
    S.load_or_sample_table_set('gunn', 2.5, 1.6, directory=tmp_path, write=True, seed=1000)
    assert np.load(str(tmp_path / f'{prefix}_7.npy')).shape == (1, 3)
    assert np.array_equal(np.load(str(tmp_path / f'{prefix}_8.npy')), tabs[7])
    with pytest.raises(FileNotFoundError):
        S.load_table_set('gunn_1.0_2.0', tmp_path)
    with pytest.raises(NotImplementedError):
        S.load_or_sample_table_set('marshall', 2.5, 1.6, directory=tmp_path / 'other')
    # table_dir: the two places augment() looks in (simulation.py:324-327)
    assert str(S.table_dir('/data/stf')).endswith('/data/stf/training/snowflakes/npy')


def test_dense_hook_defaults_mirror_the_dataset(monkeypatch):
    from lidar_snow_sim_b200.integrations import dense
    w = dense.OnTheFlyWeather({'SNOW': 'uniform_gunn_8in9'}, engine=object())
    # dense_dataset.py:91-102: eight rain rates, the list np.random.choice draws from
    assert len(w.rainfall_rates) == 8
    assert [int(r) for r in w.rainfall_rates] == [2, 4, 8, 17, 34, 70, 130, 200]
    assert w.pairs[34] == (2.5, 1.6) and w.pairs[4] == (0.5, 1.2) and len(w.pairs) == 8
    assert sorted(dense.OnTheFlyWeather({}, engine=object(), only_precomputed=True).pairs) == [2, 8, 17, 34, 70]
    # two different pairs behind one integer rain rate would be ambiguous
    monkeypatch.setattr(dense, 'DATASET_SNOWFALL_RATES', [2.5, 2.5])
    monkeypatch.setattr(dense, 'DATASET_TERMINAL_VELOCITIES', [1.6, 1.6001])
    with pytest.raises(ValueError):
        dense.OnTheFlyWeather({}, engine=object())


def test_sensor_table_equals_the_reference_yaml(gold_dir):
    import yaml
    from lidar_snow_sim_b200.calib.hdl64e_s3 import HDL64E_S3
    with open(os.path.join(gold_dir, '20171102_64E_S3.yaml')) as f:      # the reference's calib/ file, unchanged
        lasers = yaml.safe_load(f)['lasers']
    assert len(lasers) == len(HDL64E_S3) == 64
    for (lid, fd, fs, mi, vc), ref in zip(HDL64E_S3, lasers):
        assert lid == ref['laser_id']
        assert fd == ref['focal_distance'] and fs == ref['focal_slope'] and vc == ref['vert_correction']
        assert mi == ref.get('min_intensity')                         # absent for lasers 34-63 (SURVEY.md 2 #9)

"""
CPU tests: the oracle (oracle/) against the golden vectors frozen from the unmodified reference
(tools/make_golden.py).  These pin the oracle; the GPU tests then compare the CUDA path with the oracle.
"""
import json
import os

import numpy as np
import pytest

from helpers import DIV, canon, channel_case, augment_case, augment_full_case, augment_cfg1_case, canon_no_intensity, sha
from lidar_snow_sim_b200.calib.hdl64e_s3 import sensor_arrays
from lidar_snow_sim_b200.calib.dense_camera import STF_HDL64_CAMERA
from lidar_snow_sim_b200.snowfall import sampling as prod_sampling
from lidar_snow_sim_b200.synthetic import synthetic_cloud


def test_scalars(oracle, gold_dir):
    kat = json.load(open(os.path.join(gold_dir, 'kat_scalars.json')))['scalars']
    for key, v in kat.items():
        rs, tv = [float(t) for t in key.split('_')]
        for mod in (oracle, prod_sampling):
            assert float(mod.compute_occupancy(rs, tv)) == v['occupancy']
            rr = float(mod.snowfall_rate_to_rainfall_rate(rs, tv))
            assert rr == v['rainfall_rate']
            assert float(mod.gunn_marshall(rr)) == v['gunn']
            assert float(mod.sekhon_srivastava(rr)) == v['sekhon']
        assert float(prod_sampling.rainfall_rate_to_snowfall_rate(v['rainfall_rate'], tv)) == v['back']
    # SURVEY.md Appendix B-1
    assert prod_sampling.particle_file_prefix('gunn', 1.0, 1.6) == 'gunn_8.847991609353935_1.7361111111111108e-06'
    assert prod_sampling.particle_file_prefix('gunn', 2.5, 1.6) == 'gunn_34.97475775452152_4.340277777777777e-06'


def test_occlusion_dict_kat(oracle, gold_dir):
    kat = json.load(open(os.path.join(gold_dir, 'kat_occlusion_dict.json')))
    for case in kat['cases']:
        got = oracle.occlusion_dict(case['beam'], np.array(case['intervals']), 30.0, kat['beam_divergence_deg'])
        want = list(case['dict'].values())
        assert len(got) == len(want)
        for (r, ratio), (wr, wratio) in zip(got, want):
            assert r == wr and ratio == wratio
    # the seam quirk (SURVEY.md App. A): hard target keeps ratio 1.0 for the un-rotated case
    assert kat['cases'][0]['dict']['-1'][1] == 1.0


def test_kat_channel(oracle, gold_dir):
    g = np.load(os.path.join(gold_dir, 'kat_channel.npz'))
    fd, fs, mi, mx = sensor_arrays()
    out, s, nocc, _ = oracle.snow_channel(g['points'], g['particles'], DIV, fd[2], fs[2], mi[2], mx[2], theta=g['theta'])
    assert np.array_equal(out, g['out'])
    assert s == float(g['intensity_diff_sum']) == 189.5
    assert np.array_equal(nocc, g['n_occluders'])
    # SURVEY.md Appendix B-3 rows
    assert np.allclose(out[0], [5.0010376, 0, 0, 48, 2]) and out[3].tolist() == [-30, 0, 1, 50, 0]


def test_channel_cases(oracle, gold_dir):
    rec = np.load(os.path.join(gold_dir, 'channel_cases.npz'))
    fd, fs, mi, mx = sensor_arrays()
    for ci in range(int(rec['n_cases'])):
        table = channel_case(rec, ci)
        ch = int(rec[f'c{ci}_channel'])
        out, s, nocc, _ = oracle.snow_channel(rec[f'c{ci}_points'], table, DIV, fd[ch], fs[ch], mi[ch], mx[ch],
                                              theta=rec[f'c{ci}_theta'])
        assert np.array_equal(out, rec[f'c{ci}_out'])
        assert s == float(rec[f'c{ci}_sum'])
        assert np.array_equal(nocc, rec[f'c{ci}_nocc'])


@pytest.mark.parametrize('name', ['augment_a', 'augment_b'])
def test_augment(oracle, gold_dir, name):
    g = np.load(os.path.join(gold_dir, f'{name}.npz'))
    pc, tables = augment_case(g)
    idx = pc[:, 4].argsort(kind='stable')
    stats, aug, internals = oracle.augment(pc, tables, DIV, sensor_arrays(), order=g['order'].tolist(),
                                           plane=(g['plane_w'], float(g['plane_h'])), theta_sorted=g['theta'][idx],
                                           only_camera_fov=bool(g['fov']), calib=STF_HDL64_CAMERA, stable_sort=True,
                                           return_internals=True, least_populated=g['ymins'])
    assert stats == tuple(int(v) for v in g['stats'])
    assert np.array_equal(canon(aug), g['out'])
    assert np.allclose(internals['thresh_poly'], g['thresh_poly'], rtol=1e-12, atol=0)


def test_augment_full_size(oracle, gold_dir):
    """BASELINE.json configs[0]: one STF-shaped 64 x 2048 cloud, real dart-throwing tables, against the reference's own
    output (stored as stats + SHA-256 of the canonically ordered rows)."""
    g = np.load(os.path.join(gold_dir, 'augment_full.npz'))
    pc, tables, theta = augment_full_case(g)
    idx = pc[:, 4].argsort(kind='stable')
    stats, aug = oracle.augment(pc, tables, DIV, sensor_arrays(), order=g['order'].tolist(), thresh_poly=g['thresh_poly'],
                                theta_sorted=theta[idx], stable_sort=True)
    assert stats == tuple(int(v) for v in g['stats'])
    assert aug.shape == tuple(g['out_shape']) and sha(canon(aug)) == str(g['out_sha'])
    assert [(aug[:, 4] == l).sum() for l in (0, 1, 2)] == g['label_counts'].tolist()


def test_wet_ground(oracle, gold_dir):
    g = np.load(os.path.join(gold_dir, 'wet_ground.npz'))
    pc = synthetic_cloud(seed=int(g['seed']), n_azimuth=int(g['n_azimuth']))
    assert sha(pc) == str(g['cloud_sha'])
    out = oracle.ground_water_augmentation(pc, water_height=0.001, plane=(g['plane_w'], float(g['plane_h'])),
                                           least_populated=g['ymins'])
    assert out.dtype == np.float64 and out.shape == g['out'].shape
    assert np.array_equal(out[:, [0, 1, 2, 4]], g['out'][:, [0, 1, 2, 4]])
    # the intensities pass through float64 np.cos / np.arccos and BLAS matrix-vector products, whose last bits depend on
    # the host's SIMD and BLAS kernels (bit for bit on the host the fixture was made on, a few ulp apart elsewhere)
    assert np.allclose(out[:, 3], g['out'][:, 3], rtol=1e-12, atol=0)


def test_config1_and_config2(oracle, gold_dir):
    """BASELINE.json configs[1] (2.5 mm/h Gunn-Marshall tables, full 64 x 2048 cloud) and configs[2] (snow -> wet ground):
    the oracle, replaying the reference host's RANSAC planes / np.argpartition picks / float32 arctan2 bits, reproduces
    the reference's own outputs."""
    g = np.load(os.path.join(gold_dir, 'augment_cfg1.npz'))
    pc, tables, theta = augment_cfg1_case(g)
    idx = pc[:, 4].argsort(kind='stable')
    stats, aug, oi = oracle.augment(pc, tables, DIV, sensor_arrays(), order=g['order'].tolist(),
                                    plane=(g['plane_w'], float(g['plane_h'])), least_populated=g['ymins'],
                                    theta_sorted=theta[idx], stable_sort=True, return_internals=True)
    assert np.allclose(oi['thresh_poly'], g['thresh_poly'], rtol=1e-9, atol=0)
    assert stats == tuple(int(v) for v in g['stats'])
    assert aug.shape == tuple(g['out_shape']) and sha(canon(aug)) == str(g['out_sha'])
    wet = oracle.ground_water_augmentation(aug, water_height=0.001, replace=False,
                                           plane=(g['wet_plane_w'], float(g['wet_plane_h'])),
                                           least_populated=g['wet_ymins'])
    assert wet.shape == tuple(g['wet_shape'])
    wc = canon_no_intensity(wet)
    assert sha(wc[:, [0, 1, 2, 4]]) == str(g['wet_xyzl_sha'])
    assert np.allclose(wc[:, 3], g['wet_intensity'], rtol=1e-12, atol=0)
    assert [(wet[:, 4] == l).sum() for l in (0, 1, 2)] == g['wet_label_counts'].tolist()


def test_dart_throwing(oracle, gold_dir):
    g = np.load(os.path.join(gold_dir, 'dart_throwing.npz'))
    for dist in ('gunn', 'sekhon'):
        rng = np.random.default_rng(int(g[f'{dist}_seed']))
        t = oracle.dart_throwing(float(g['occupancy']), float(g['rainfall_rate']), float(g[f'{dist}_R0']), rng, dist)
        assert np.array_equal(t, g[f'{dist}_table'])
        assert rng.bit_generator.random_raw() == int(g[f'{dist}_next_u64'][0])


def test_range_grid(oracle):
    R = oracle.range_grid()
    assert R.shape == (1230,) and R[125] == 12.51 and R[600] == 60.05 and R[1229] == 123.0   # SURVEY.md App. A

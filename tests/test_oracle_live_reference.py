"""Cross-check of the CPU oracle against the reference's outputs on seeds the other fixtures do not contain.

tests/golden/oracle_crosscheck.npz holds what the unmodified reference computed for these cases
(tools/make_golden_crosscheck.py): snowfall per-channel solve, wet ground, fog simulation.  The inputs are rebuilt here
from their seeds and checked against the stored hashes; what the reference host's libraries chose (float32 arctan2 bits,
the wet-ground RANSAC plane and np.argpartition picks) is replayed from the fixture.  CPU only."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from tools.make_golden import sha                                                    # noqa: E402
from tools.make_golden_crosscheck import (FOG_CASES, N_SNOW_PARTICLES, WET_KW, WET_N_AZIMUTH, WET_SEED,  # noqa: E402
                                          snow_points)

DIV = float(np.degrees(3e-3))


@pytest.fixture(scope='module')
def ref_out(gold_dir):
    return np.load(os.path.join(gold_dir, 'oracle_crosscheck.npz'))


@pytest.mark.parametrize('seed,ch', [(101, 7), (102, 58)])
def test_snowfall_channel_fresh_seed(seed, ch, ref_out):
    from oracle import oracle as orc
    from lidar_snow_sim_b200.synthetic import synthetic_particles
    from lidar_snow_sim_b200.calib.hdl64e_s3 import sensor_arrays
    k = f'snow_{seed}_{ch}'
    table = synthetic_particles(seed, N_SNOW_PARTICLES)
    assert sha(table) == str(ref_out[f'{k}_table_sha'])
    pts = snow_points(seed, ch)
    assert np.array_equal(pts, ref_out[f'{k}_points'])
    out, s = ref_out[f'{k}_out'], float(ref_out[f'{k}_sum'])
    sensor = sensor_arrays()
    o_out, o_s, o_n, _ = orc.snow_channel(pts, table, DIV, sensor[0][ch], sensor[1][ch], sensor[2][ch], sensor[3][ch],
                                          theta=ref_out[f'{k}_theta'])
    assert np.array_equal(out, o_out) and s == o_s
    assert (o_out[:, 4] > 0).sum() > 5                           # the case exercises attenuated / scattered beams


def test_fog_fresh_seeds(ref_out):
    from oracle import fog as ofog
    from lidar_snow_sim_b200.synthetic import synthetic_cloud
    for seed, alpha, variant, noise, gain in FOG_CASES:
        k = f'fog_{seed}'
        pc = synthetic_cloud(seed=seed, n_azimuth=12)
        assert sha(pc) == str(ref_out[f'{k}_cloud_sha'])
        rng = np.random.default_rng(seed)
        aug, fog, info = ofog.simulate_fog(ofog.ParameterSet(alpha=alpha, gamma=0.000001), pc, noise,
                                           ref_out[f'{k}_lut'], rng, gain=gain, noise_variant=variant)
        assert np.array_equal(aug, ref_out[f'{k}_aug'], equal_nan=True), (seed, variant)
        if bool(ref_out[f'{k}_has_fog']):
            assert fog is not None and np.array_equal(fog, ref_out[f'{k}_fog'])
        else:
            assert fog is None
        assert info['num_fog_responses'] == int(ref_out[f'{k}_num_fog_responses'])
        assert np.array_equal(rng.random(2), ref_out[f'{k}_next_u'])


def test_wet_ground_fresh_seed(ref_out):
    from oracle import oracle as orc
    from lidar_snow_sim_b200.synthetic import synthetic_cloud
    pc = synthetic_cloud(seed=WET_SEED, n_azimuth=WET_N_AZIMUTH)
    assert sha(pc) == str(ref_out['wet_cloud_sha'])
    want = ref_out['wet_out']
    plane = (ref_out['wet_plane_w'], float(ref_out['wet_plane_h']))
    got = orc.ground_water_augmentation(pc.copy(), replace=True, plane=plane, least_populated=ref_out['wet_ymins'],
                                        **WET_KW)
    assert got.shape == want.shape
    assert np.array_equal(got[:, [0, 1, 2, 4]], want[:, [0, 1, 2, 4]])
    # intensities: float64 np.cos / np.arccos and BLAS products, last bits host dependent (tests/test_oracle_golden.py)
    assert np.allclose(got[:, 3], want[:, 3], rtol=1e-12, atol=0)

"""
Generate tests/golden/oracle_crosscheck.npz and tests/golden/20171102_64E_S3.yaml: the reference's own outputs for the
cases of tests/test_oracle_live_reference.py (snowfall per-channel solve, fog simulation, wet ground), computed by the
UNMODIFIED reference (imported through oracle/ref_harness.py), and the reference's sensor calibration file, copied as
is.  The tests compare the CPU oracle against these stored outputs, so they run wherever the suite runs.

    python tools/make_golden_crosscheck.py        # exits non-zero if the oracle does not reproduce the reference

Host note (SURVEY.md App. D): the reference's float32 np.arctan2 is host dependent; the fixture stores the theta
this host produced for the snowfall cases so that the oracle replays them exactly.  Likewise it stores the wet-ground
case's library-defined choices (the RANSAC plane and the np.argpartition picks) for the oracle to replay.
"""
import os
import shutil
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import ref_harness as rh            # noqa: E402
from oracle import oracle as orc                # noqa: E402
from oracle import fog as ofog                  # noqa: E402
from lidar_snow_sim_b200.synthetic import synthetic_cloud, synthetic_particles      # noqa: E402
from lidar_snow_sim_b200.calib.hdl64e_s3 import sensor_arrays                       # noqa: E402
from tools.make_golden import CapturePrepass, channel_infos, write_tables, sha     # noqa: E402

GOLD = os.path.join(ROOT, 'tests', 'golden')
DIV = float(np.degrees(3e-3))
SNOW_CASES = [(101, 7), (102, 58)]                               # (seed, channel)
FOG_CASES = [(5, 0.03, 'v1', 10, False), (6, 0.12, 'v3', 7, True), (7, 0.1, 'v4', 10, False)]
WET_SEED, WET_N_AZIMUTH = 321, 128
WET_KW = dict(water_height=0.0008, pavement_depth=0.0012, noise_floor=0.7, power_factor=15, flat_earth=True, delta=0.5)
N_SNOW_POINTS, N_SNOW_PARTICLES = 96, 22000


def snow_points(seed, ch):
    """The seeded beams of one snowfall case: random azimuths (16 of them at the +-pi seam), ranges and elevations."""
    rng = np.random.default_rng(seed)
    M = N_SNOW_POINTS
    az = rng.uniform(-np.pi, np.pi, M)
    az[:16] = rng.uniform(-0.004, 0.004, 16)
    d = rng.uniform(1.2, 110.0, M)
    el = rng.uniform(-0.4, 0.03, M)
    return np.stack([d * np.cos(el) * np.cos(az), d * np.cos(el) * np.sin(az), d * np.sin(el),
                     np.round(rng.uniform(1, 255, M)), np.full(M, ch)], axis=1).astype(np.float32)


def main():
    ns = rh.load()
    sys.path.insert(0, os.path.join(rh.REF_ROOT, 'lib', 'LiDAR_fog_sim'))
    import fog_simulation as ref_fog
    ok = True
    rec = {}
    sensor = sensor_arrays()

    for seed, ch in SNOW_CASES:
        table = synthetic_particles(seed, N_SNOW_PARTICLES)
        pts = snow_points(seed, ch)
        root = tempfile.mkdtemp()
        write_tables(root, 'g', [table] * 64)
        s, _, out = ns.sim.process_single_channel(root, 'g', pts, DIV, list(range(64)), channel_infos(), ch)
        shutil.rmtree(root)
        theta = np.arctan2(pts[:, 1], pts[:, 0])
        o_out, o_s, _, _ = orc.snow_channel(pts, table, DIV, sensor[0][ch], sensor[1][ch], sensor[2][ch],
                                            sensor[3][ch], theta=theta)
        good = np.array_equal(out, o_out) and float(s) == o_s
        print(f'snowfall seed {seed} channel {ch}: oracle==reference: {good}')
        ok &= good
        k = f'snow_{seed}_{ch}'
        rec.update({f'{k}_table_sha': sha(table), f'{k}_points': pts, f'{k}_theta': theta, f'{k}_out': out,
                    f'{k}_sum': float(s)})

    for seed, alpha, variant, noise, gain in FOG_CASES:
        pc = synthetic_cloud(seed=seed, n_azimuth=12)
        p_ref = ref_fog.ParameterSet(alpha=alpha, gamma=0.000001)
        d = ref_fog.get_integral_dict(p_ref)
        lut = np.array([[float(d[q][0]), float(d[q][1])] for q in sorted(d.keys())])
        ref_fog.RNG = np.random.default_rng(seed)
        aug, fog, info = ref_fog.simulate_fog(p_ref, pc=pc, noise=noise, gain=gain, noise_variant=variant)
        next_u = ref_fog.RNG.random(2)
        rng = np.random.default_rng(seed)
        o_aug, o_fog, o_info = ofog.simulate_fog(ofog.ParameterSet(alpha=alpha, gamma=0.000001), pc, noise, lut, rng,
                                                 gain=gain, noise_variant=variant)
        good = (np.array_equal(o_aug, aug, equal_nan=True) and
                ((fog is None and o_fog is None) or np.array_equal(o_fog, fog)) and
                o_info['num_fog_responses'] == info['num_fog_responses'] and np.array_equal(rng.random(2), next_u))
        print(f'fog seed {seed} ({variant}): oracle==reference: {good}')
        ok &= good
        k = f'fog_{seed}'
        rec.update({f'{k}_cloud_sha': sha(pc), f'{k}_lut': lut, f'{k}_aug': aug, f'{k}_has_fog': fog is not None,
                    f'{k}_fog': np.zeros((0, aug.shape[1])) if fog is None else fog,
                    f'{k}_num_fog_responses': int(info['num_fog_responses']), f'{k}_next_u': next_u})

    pc = synthetic_cloud(seed=WET_SEED, n_azimuth=WET_N_AZIMUTH)
    with CapturePrepass(ns) as cap:
        want = ns.wet_aug.ground_water_augmentation(pc.copy(), estimation_method='linear', debug=False, replace=True,
                                                    **WET_KW)
    got = orc.ground_water_augmentation(pc.copy(), replace=True, **WET_KW)
    good = got.shape == want.shape and np.array_equal(got, want)
    (w, h), ymins = cap.planes[0], cap.ymins[0]
    replayed = orc.ground_water_augmentation(pc.copy(), replace=True, plane=(w, h), least_populated=ymins, **WET_KW)
    good &= np.array_equal(replayed, want)
    print(f'wet ground seed {WET_SEED}: oracle==reference: {good}')
    ok &= good
    rec.update({'wet_cloud_sha': sha(pc), 'wet_plane_w': w, 'wet_plane_h': h, 'wet_ymins': ymins, 'wet_out': want})

    path = os.path.join(GOLD, 'oracle_crosscheck.npz')
    np.savez_compressed(path, **rec)
    print('wrote', path, os.path.getsize(path), 'bytes')
    calib = os.path.join(GOLD, '20171102_64E_S3.yaml')
    shutil.copyfile(os.path.join(rh.REF_ROOT, 'calib', '20171102_64E_S3.yaml'), calib)
    print('wrote', calib)
    sys.exit(0 if ok else 1)


if __name__ == '__main__':
    main()

"""
DROR de-snowing filter (lib/cadc_devkit/other/dror.py:73-84, 288-334; create_image_sets.py:16-66), CPU side:
  * the oracle's count rule (oracle/dror.py) equals a literal transcription of dynamic_radius_outlier_filter with
    brute-force k-NN standing in for FLANN;
  * the quirks: get_cube_mask ignores z, the DROR_LEVELS boundaries;
  * a NumPy model of the device search (csrc/dror.cu: cell function, clamping, level choice, padded box -> cells, the
    float32 hit limit) finds every neighbour the exact rule admits, in the style of tests/test_index_model.py.
The CUDA path is compared with the oracle bit for bit in tests/test_dror_gpu.py.
"""
import numpy as np
import pytest

from oracle import dror as D

# ---- literal transcription of dror.py:288-334 ------------------------------------------------------------------------


def literal_filter(pc, alpha=0.16, beta=3.0, k_min=3, sr_min=0.04):
    pc = np.asarray(pc, dtype=np.float32)[:, :3]
    num_points = pc.shape[0]
    mask = np.zeros(num_points, dtype=bool)
    k = min(k_min + 1, num_points)                      # PCL clamps k to the cloud size
    for i in range(num_points):
        x = float(pc[i][0])
        y = float(pc[i][1])
        r = np.linalg.norm([x, y], axis=0)
        sr = alpha * beta * np.pi / 180 * r
        if sr < sr_min:
            sr = sr_min
        d2 = D.l2_simple(pc[i][None, :], pc)            # FLANN's L2_Simple, float32
        sqdist = [float(v) for v in np.sort(d2)[:k]]    # the k smallest (a Python list, as python-pcl returns it)
        neighbors = -1
        for val in sqdist:
            if np.sqrt(val) < sr:
                neighbors += 1
        if neighbors >= k_min:
            mask[i] = True
    return mask


def small_clouds(seed):
    """Clusters of points spaced on the scale of the search radius at 2-60 m, duplicated rows, isolated points."""
    rng = np.random.default_rng(seed)
    clouds = [np.zeros((0, 5), np.float32)]
    for n in range(1, 6):
        c = rng.normal(0, 0.03, (n, 5)).astype(np.float32) + np.float32([8, 0.5, -1, 0, 0])
        if n >= 2:
            c[1] = c[0]                                                      # a duplicate
        clouds.append(c)
    for _ in range(3):
        parts = []
        for _ in range(6):
            centre = np.array([rng.uniform(2, 60) * np.cos(a := rng.uniform(0, 6.3)), rng.uniform(2, 60) * np.sin(a),
                               rng.uniform(-2, 1)])
            scale = rng.choice([0.01, 0.05, 0.2, 0.6])
            parts.append(centre + rng.normal(0, scale, (rng.integers(10, 60), 3)))
        xyz = np.concatenate(parts + [rng.uniform(-40, 40, (20, 3))])
        c = np.column_stack([xyz, rng.uniform(0, 255, (xyz.shape[0], 2))]).astype(np.float32)
        c = np.concatenate([c, c[rng.integers(0, c.shape[0], 15)]])          # duplicated rows
        clouds.append(c[rng.permutation(c.shape[0])])
    return clouds


@pytest.mark.parametrize('alpha', [0.08, 0.16, 0.45])
def test_oracle_equals_the_literal_filter(alpha):
    kept = total = 0
    for seed in range(2):
        for pc in small_clouds(seed):
            for k_min in (0, 1, 3, 5):
                for sr_min in (0.0, 0.04, 0.2):
                    want = literal_filter(pc, alpha, 3.0, k_min, sr_min)
                    got = D.dror_keep(pc, alpha, 3.0, k_min, sr_min)
                    assert np.array_equal(got, want), (seed, pc.shape[0], k_min, sr_min)
                    kept += int(want.sum())
                    total += want.shape[0]
    assert 0.2 * total < kept < 0.95 * total                 # both outcomes occur


def test_cube_mask_ignores_z_and_crop_indices():
    pc = np.array([[5, 0, 5, 0, 0], [5, 0, 0, 0, 0], [3, -1, -9, 0, 0], [13, 1, 9, 0, 0], [13.01, 0, 0, 0, 0],
                   [5, 1.01, 0, 0, 0], [2.99, 0, 0, 0, 0]], dtype=np.float32)
    assert D.cube_mask(pc).tolist() == [True, True, True, True, False, False, False]
    from lidar_snow_sim_b200.dror import get_cube_mask
    assert np.array_equal(get_cube_mask(pc), D.cube_mask(pc))
    # the crop variant's indices are relative to pc[cube_mask]
    pc = small_clouds(3)[-1].copy()
    pc[:, 0] = np.abs(pc[:, 0]) % 10 + 3
    pc[:, 1] = pc[:, 1] % 2 - 1
    pc = np.concatenate([pc, np.float32([[20, 5, 0, 0, 0]] * 3)])
    idx = D.snow_indices(pc, 0.45, crop=True)
    m = D.cube_mask(pc)
    assert np.array_equal(idx, np.nonzero(~D.dror_keep(pc[m], 0.45))[0])
    assert D.snow_indices(pc[~m], 0.45, crop=True) == []


def test_dror_levels():
    from lidar_snow_sim_b200.dror import DROR_LEVELS, dror_level
    assert DROR_LEVELS == D.DROR_LEVELS
    for n, want in ((0, 'none'), (9, 'none'), (10, 'light'), (79, 'light'), (80, 'heavy'), (10 ** 6, 'heavy')):
        assert dror_level(n) == want == D.dror_level(n)


# ---- model of the device search (csrc/dror.cu) -----------------------------------------------------------------------
ORIGIN, C0, BITS = -512.0, 0.125, 13
PAD_REL, PAD_ABS = 2.0 ** -18, 1e-6


def grid_cell(v):
    """grid_cell: floor((v - ORIGIN) / C0) in float64, clamped to [0, 2^13 - 1]; monotone."""
    c = np.floor((np.asarray(v, dtype=np.float64) - ORIGIN) * (1 / C0))
    return np.clip(np.nan_to_num(c, nan=0.0), 0, 2 ** BITS - 1).astype(np.int64)


def level(sr):
    rp = sr * (1 + PAD_REL) + PAD_ABS
    L = np.zeros(sr.shape, dtype=np.int64)
    for _ in range(BITS):
        L = np.where((L < BITS) & (C0 * 2.0 ** L < 2 * rp), L + 1, L)
    return L, rp


def hit_limit(sr):
    """The largest float32 f with sqrt(float64(f)) < sr (k_dror_query compares d2 <= it)."""
    f = np.float32(sr * sr)
    while f > 0 and not np.sqrt(np.float64(f)) < sr:
        f = np.nextafter(f, np.float32(0))
    while True:
        up = np.nextafter(f, np.float32(np.inf))
        if up == np.inf or not np.sqrt(np.float64(up)) < sr:
            return f
        f = up


def model_clouds():
    rng = np.random.default_rng(11)
    from lidar_snow_sim_b200.synthetic import synthetic_cloud
    yield synthetic_cloud(seed=3, n_azimuth=256)
    yield rng.uniform(-60, 60, (20000, 3)).astype(np.float32)
    far = []
    for cx in (505.0, 511.97, 512.0, 600.0, -2000.0, 1e5):                 # around and beyond the clamp at +-512 m
        far.append(np.float32([cx, 0.4 * cx, 3.0]) + rng.normal(0, 0.02 * abs(cx) ** 0.5 + 0.05, (400, 3)))
    far.append(np.float32([[511.999, 511.999, 511.999], [512.001, 512.001, 512.001], [-512.0, -512.0, 0.0]]))
    yield np.concatenate(far).astype(np.float32)


@pytest.mark.parametrize('alpha', [0.16, 0.45])
def test_grid_search_model_finds_every_neighbour_the_rule_admits(alpha):
    checked = 0
    for pc in model_clouds():
        xyz = np.ascontiguousarray(pc[:, :3], dtype=np.float32)
        sr = D.search_radius(xyz, alpha, 3.0, 0.04)
        L, rp = level(sr)
        assert ((C0 * 2.0 ** L >= 2 * rp) | (L == BITS)).all()
        cell = np.stack([grid_cell(xyz[:, a]) for a in range(3)], axis=1)
        for i, j, d2 in D._pairs(xyz, sr):
            hit = np.sqrt(d2.astype(np.float64)) < sr[i]
            i, j = i[hit], j[hit]
            for a in range(3):
                lo = grid_cell(xyz[i, a].astype(np.float64) - rp[i]) >> L[i]
                hi = grid_cell(xyz[i, a].astype(np.float64) + rp[i]) >> L[i]
                cj = cell[j, a] >> L[i]
                assert ((lo <= cj) & (cj <= hi)).all(), 'a neighbour lies outside the visited cells'
                assert (hi - lo <= 1).all(), 'more than two cells per axis'
            checked += int(i.shape[0])
    assert checked > 100000


def test_float32_hit_limit_is_the_float64_sqrt_test():
    rng = np.random.default_rng(5)
    srs = np.concatenate([rng.uniform(0.04, 3.0, 300), [0.04, 0.1, 1.0, 2.0 ** -10]])
    for sr in srs:
        lim = hit_limit(sr)
        f0 = np.float32(sr * sr)
        near = np.array([np.nextafter(f0, np.float32(0))] * 3 + [f0] * 3 + [np.nextafter(f0, np.float32(1e9))] * 3,
                        dtype=np.float32)
        near = (near.view(np.int32) + np.array([-1, 0, 1] * 3, dtype=np.int32)).view(np.float32)
        d2 = np.concatenate([near, rng.uniform(0, 2 * f0, 50).astype(np.float32)])
        assert np.array_equal(d2 <= lim, np.sqrt(d2.astype(np.float64)) < sr)

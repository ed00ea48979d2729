"""
DROR on the device (csrc/dror.cu, SnowfallEngine.dror_batch) against the oracle (oracle/dror.py): an integer rule, so codes,
counts, snow counts and the compacted rows (values and order) must be bit-exact.
"""
import numpy as np
import pytest
import torch

from oracle import dror as D
from lidar_snow_sim_b200.synthetic import synthetic_cloud

pytestmark = pytest.mark.gpu


def with_snow(pc, seed, n_snow=3000):
    rng = np.random.default_rng(seed)
    r = 30 * np.sqrt(rng.uniform(0, 1, n_snow))
    a = rng.uniform(0, 2 * np.pi, n_snow)
    snow = np.column_stack([r * np.cos(a), r * np.sin(a), rng.uniform(-1.5, 3, n_snow), rng.uniform(0, 30, n_snow),
                            np.full(n_snow, 2.0)]).astype(np.float32)
    return np.concatenate([pc, snow])


def batch_clouds():
    rng = np.random.default_rng(8)
    full = with_snow(synthetic_cloud(seed=60), 1)
    shuffled = with_snow(synthetic_cloud(seed=61, drop=0.05), 2)
    shuffled = shuffled[rng.permutation(shuffled.shape[0])]
    small = synthetic_cloud(seed=62, n_azimuth=512)
    small = np.concatenate([small, small[rng.integers(0, small.shape[0], 500)],                  # duplicated rows
                            np.float32([[700, 10, 2, 5, 0], [700.5, 10, 2, 5, 0], [-3e3, 4e3, 9, 5, 0],
                                        [1e5, 0, 0, 5, 0], [511.99, 512.01, -511.99, 5, 0]])])  # far points
    tiny = [np.float32([[5, 1, -1, 3, 0]]), np.float32([[8, 0, 0, 1, 0]] * 3),
            np.float32([[8, 0, 0, 1, 0], [8, 0.01, 0, 1, 0], [8, 0, 0.02, 1, 0], [8.1, 0, 0, 1, 0]])]
    return [full, np.zeros((0, 5), np.float32), shuffled, tiny[0], small, tiny[1], tiny[2]]


_COUNTS = {}


def oracle_counts(b, pc, alpha):
    if (b, alpha) not in _COUNTS:
        _COUNTS[(b, alpha)] = D.neighbour_counts(pc, alpha)
    return _COUNTS[(b, alpha)]


def offsets(clouds):
    return np.concatenate([[0], np.cumsum([c.shape[0] for c in clouds])]).astype(np.int64)


def check_cloud(out, off, b, pc, codes_want):
    n_keep = int((codes_want == 1).sum())
    assert np.array_equal(out['codes'][off[b]:off[b] + pc.shape[0]].cpu().numpy(), codes_want)
    assert int(out['counts'][b]) == n_keep
    assert int(out['n_snow'][b]) == int((codes_want == 0).sum())
    if out['points'] is not None:
        assert np.array_equal(out['points'][off[b]:off[b] + n_keep].cpu().numpy(), pc[codes_want == 1])


@pytest.mark.parametrize('alpha', [0.08, 0.16, 0.45])
@pytest.mark.parametrize('k_min', [0, 3])
def test_batch_matches_the_oracle(engine, alpha, k_min):
    clouds = batch_clouds()
    off = offsets(clouds)
    d = torch.from_numpy(np.concatenate(clouds)).cuda()
    out = engine.dror_batch(d, off, alpha=alpha, k_min=k_min)
    engine.check()
    snow = 0
    for b, pc in enumerate(clouds):
        want = (oracle_counts(b, pc, alpha) >= k_min + 1).astype(np.uint8)
        check_cloud(out, off, b, pc, want)
        snow += int((want == 0).sum())
    assert snow > 1000 if k_min == 3 else snow == 0          # k_min = 0: every point is its own neighbour
    if k_min == 3 and alpha == 0.16:
        band = D.reading_band(clouds[0], alpha)
        print(f'float32-sqrt reading: {band}')
    # stability: a second run is identical; a cloud alone gives what it gave inside the batch
    out2 = engine.dror_batch(d, off, alpha=alpha, k_min=k_min)
    for k in ('codes', 'counts', 'n_snow'):
        assert torch.equal(out[k], out2[k])
    for b in range(len(clouds)):                                    # rows behind a cloud's count are unspecified
        n = int(out['counts'][b])
        assert torch.equal(out['points'][off[b]:off[b] + n], out2['points'][off[b]:off[b] + n])
    b = 4
    alone = engine.dror_batch(d[off[b]:off[b + 1]].contiguous(), np.array([0, off[b + 1] - off[b]]), alpha=alpha,
                              k_min=k_min)
    assert torch.equal(alone['codes'], out['codes'][off[b]:off[b + 1]])
    assert torch.equal(alone['points'][:int(alone['counts'][0])], out['points'][off[b]:off[b] + int(out['counts'][b])])


def test_slot_compacted_input_and_wide_rows(engine):
    """counts < slot sizes (rows behind a count are never read) and F = 7 columns copied in order."""
    clouds = batch_clouds()[2:5]
    rng = np.random.default_rng(3)
    slots = [np.concatenate([c, rng.uniform(-5, 5, (100, 5)).astype(np.float32)]) for c in clouds]
    wide = [np.column_stack([s, rng.normal(size=(s.shape[0], 2)).astype(np.float32)]) for s in slots]
    off = offsets(slots)
    cnt = torch.tensor([c.shape[0] for c in clouds], dtype=torch.int32, device='cuda')
    out = engine.dror_batch(torch.from_numpy(np.concatenate(wide)).cuda(), off, counts=cnt)
    engine.check()
    for b, c in enumerate(clouds):
        want = (D.neighbour_counts(c, 0.16) >= 4).astype(np.uint8)
        n_keep = int(want.sum())
        assert np.array_equal(out['codes'][off[b]:off[b] + c.shape[0]].cpu().numpy(), want)
        assert int(out['counts'][b]) == n_keep and int(out['n_snow'][b]) == int((want == 0).sum())
        assert np.array_equal(out['points'][off[b]:off[b] + n_keep].cpu().numpy(), wide[b][:c.shape[0]][want == 1])


def test_decision_boundary_is_exact(engine):
    """Pairs (x, y, 0) / (x, y, dz) share sr; dz at the float32 boundary of sqrt(float64(dz^2)) < sr and one ulp to either
    side.  With k_min = 1 both points are kept iff the pair is within sr."""
    from test_dror import hit_limit
    rows, want = [], []
    rng = np.random.default_rng(4)
    for k in range(189):                                               # pairs on a 2 m grid, sr < 0.6 m: no cross talk
        step, hit = ((-1, True), (0, True), (1, False))[k % 3]
        x, y = np.float32(6 + 2 * (k // 7) + rng.uniform(0, 0.5)), np.float32(-6 + 2 * (k % 7) + rng.uniform(0, 0.5))
        sr = D.search_radius(np.float32([[x, y, 0]]), 0.16)[0]
        lim = hit_limit(sr)
        dz = np.float32(np.sqrt(np.float64(lim)))
        while np.float32(dz * dz) > lim:
            dz = np.nextafter(dz, np.float32(0))
        while np.float32(np.nextafter(dz, np.float32(1e9)) ** 2) <= lim:
            dz = np.nextafter(dz, np.float32(1e9))
        z = (dz.view(np.int32) + np.int32(step)).view(np.float32)     # the boundary and one ulp to either side
        rows += [[x, y, 0, 0, 0], [x, y, z, 0, 0]]
        want += [hit, hit]
    pc = np.array(rows, dtype=np.float32)
    out = engine.dror_batch(torch.from_numpy(pc).cuda(), np.array([0, pc.shape[0]]), alpha=0.16, k_min=1, sr_min=0.04)
    engine.check()
    got = out['codes'].cpu().numpy() == 1
    assert np.array_equal(D.dror_keep(pc, 0.16, k_min=1), np.array(want))
    assert np.array_equal(got, np.array(want))


def test_crop_variant(engine):
    from lidar_snow_sim_b200.dror import snow_indices
    rng = np.random.default_rng(6)
    clouds = []
    for s in range(3):
        pc = synthetic_cloud(seed=70 + s, n_azimuth=1024)
        extra = np.column_stack([rng.uniform(3, 13, 400), rng.uniform(-1, 1, 400), rng.uniform(-2, 5, 400),
                                 np.zeros((400, 2))]).astype(np.float32)
        clouds.append(np.concatenate([pc, extra])[rng.permutation(pc.shape[0] + 400)])
    off = offsets(clouds)
    out = engine.dror_batch(torch.from_numpy(np.concatenate(clouds)).cuda(), off, alpha=0.45, crop_xy=(3, 13, -1, 1))
    engine.check()
    for b, pc in enumerate(clouds):
        want = D.codes(pc, 0.45, crop_xy=D.CUBE)
        assert (want == 2).any() and (want == 0).any()
        check_cloud(out, off, b, pc, want)
        idx = snow_indices(pc, 0.45, crop=True, engine=engine)
        assert np.array_equal(idx, D.snow_indices(pc, 0.45, crop=True))
    assert snow_indices(clouds[0][:0], 0.45, engine=engine) == []


def test_snowfall_dror_voxels_on_the_device(engine):
    """snowfall_batch -> dror_batch -> voxelize_batch without leaving the device; equals the oracle on the host copy."""
    from helpers import DIV
    from oracle import voxel as V
    from lidar_snow_sim_b200.synthetic import synthetic_particles
    clouds = [synthetic_cloud(seed=95 + b, n_azimuth=512) for b in range(3)]
    tables = [synthetic_particles(3100 + k, 60000) for k in range(64)]
    off = offsets(clouds)
    orders = np.stack([np.random.default_rng(b).permutation(64) for b in range(3)]).astype(np.int32)
    tid = engine.upload_tables(tables)
    snow = engine.snowfall_batch(tid, torch.from_numpy(np.concatenate(clouds)).cuda(), off, orders, DIV,
                                 thresh_poly=np.tile([1e-3, -0.2, 9.0], (3, 1)))
    dr = engine.dror_batch(snow['points'], off, counts=snow['counts'], alpha=0.45)
    rng_, vs = [0, -40, -3, 70.4, 40, 1], [0.05, 0.05, 0.1]
    vox = engine.voxelize_batch(dr['points'], off, rng_, vs, 5, 16000, counts=dr['counts'])
    engine.check()
    engine.free_tables(tid)
    host = snow['points'].cpu().numpy()
    cnt = snow['counts'].cpu().numpy()
    removed_snow = 0
    for b in range(3):
        aug = host[off[b]:off[b] + cnt[b]]
        keep = D.dror_keep(aug, 0.45)
        check_cloud(dr, off, b, aug, keep.astype(np.uint8))
        removed_snow += int(((~keep) & (aug[:, 4] == 2)).sum())
        pts, v, c, m = V.mask_and_voxelize(aug[keep], rng_, vs, 5, 16000)
        n = int(vox['n_voxels'][b])
        assert n == v.shape[0] and np.array_equal(vox['voxels'][b, :n].cpu().numpy(), v)
        assert np.array_equal(vox['coords'][b, :n, 1:].cpu().numpy(), c)
    assert removed_snow > 0


def test_numpy_mirrors(engine):
    from lidar_snow_sim_b200.dror import dynamic_radius_outlier_filter
    from lidar_snow_sim_b200.integrations.dense import apply_dror
    pc = with_snow(synthetic_cloud(seed=80, n_azimuth=512), 9, 800)
    mask = dynamic_radius_outlier_filter(pc, alpha=0.45, engine=engine)
    assert isinstance(mask, np.ndarray) and mask.dtype == bool
    assert np.array_equal(mask, D.dror_keep(pc, 0.45))
    m2 = dynamic_radius_outlier_filter(pc, 0.08, 3.0, 5, 0.2, engine=engine)
    assert np.array_equal(m2, D.dror_keep(pc, 0.08, 3.0, 5, 0.2))
    once = pc[D.dror_keep(pc, 0.45)]
    assert np.array_equal(apply_dror(pc, {'DROR': 0.45}, 'test_snow', engine=engine), once)
    assert np.array_equal(apply_dror(pc, {'DROR++': '0.45'}, 'test_clear_day', engine=engine), pc)
    assert np.array_equal(apply_dror(pc, {'DROR++': '0.45'}, 'test_snow_heavy', engine=engine), once)
    twice = once[D.dror_keep(once, 0.16)]
    assert np.array_equal(apply_dror(pc, {'DROR': 0.45, 'DROR++': 0.16}, 'snow', engine=engine), twice)

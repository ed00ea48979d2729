"""
CPU oracle of the DROR de-snowing filter -- TEST INFRASTRUCTURE, NOT PRODUCT CODE (only tests/ may import it).

Restated from lib/cadc_devkit/other/dror.py:
  * get_cube_mask                   :73-84   x / y box, both ends inclusive; np.logical_and(x_mask, y_mask, z_mask) passes
                                             z_mask as the `out` argument, so z is NOT tested
  * dynamic_radius_outlier_filter   :288-334 per point: r = np.linalg.norm([x, y]) (float64), sr = alpha * beta * np.pi /
                                             180 * r floored at sr_min, FLANN k-NN with k = k_min + 1 (self included),
                                             count of the returned neighbours with np.sqrt(d2) < sr, starting at -1; kept
                                             if the count is >= k_min
  * the `crop` variant of process_dense   :238-256   DROR on pc[cube_mask] alone; snow indices index that cropped cloud

Restated without k-NN: the k smallest distances are all below sr iff at least k points are, so
    keep_i  <=>  c_i = #{ j : sqrt(float64(d2_ij)) < sr_i }  >=  k_min + 1
(PCL clamps k to the cloud size: a cloud of at most k_min points keeps nothing, and c_i <= N says the same).
d2 is float32 in FLANN's L2_Simple order ((0 + dx^2) + dy^2) + dz^2 (no FMA; NumPy float32 arithmetic rounds each step).

PARITY UNPINNED with the library: python-pcl / FLANN is not installed anywhere this project runs.  This oracle is pinned to
a literal transcription of dror.py with brute-force k-NN (tests/test_dror.py).  One reading is a choice: python-pcl's
nearest_k_search_for_point returns the squared distances as a Python list, read here as float64 values, so np.sqrt is a
float64 sqrt of the float32 d2.  Were they a float32 array, the sqrt would be float32.  `reading_band` counts the pairs of a
cloud where the two readings differ.
"""
import numpy as np
from scipy.spatial import cKDTree

DROR_LEVELS = {'none': (0, 9), 'light': (10, 79)}        # lib/cadc_devkit/other/create_image_sets.py:16-18; heavy: >= 80
CUBE = (3, 13, -1, 1)                                    # get_cube_mask's defaults (x_min, x_max, y_min, y_max)


def cube_mask(pc, x_min=3, x_max=13, y_min=-1, y_max=1, z_min=-1, z_max=1):
    """get_cube_mask, dror.py:73-84, with its quirk (z is not tested)."""
    x_mask = np.logical_and(x_min <= pc[:, 0], pc[:, 0] <= x_max)
    y_mask = np.logical_and(y_min <= pc[:, 1], pc[:, 1] <= y_max)
    z_mask = np.logical_and(z_min <= pc[:, 2], pc[:, 2] <= z_max)
    return np.logical_and(x_mask, y_mask, z_mask)


def search_radius(pc, alpha=0.16, beta=3.0, sr_min=0.04):
    """dror.py:316-321 for every point: float64 r from the float32 x, y; sr left to right; floored at sr_min."""
    x = pc[:, 0].astype(np.float64)
    y = pc[:, 1].astype(np.float64)
    r = np.sqrt(x * x + y * y)
    sr = alpha * beta * np.pi / 180 * r
    return np.where(sr < sr_min, sr_min, sr)


def l2_simple(q, p):
    """FLANN L2_Simple in float32: ((0 + dx*dx) + dy*dy) + dz*dz, dx = q - p."""
    d = q.astype(np.float32) - p.astype(np.float32)
    return (d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1]) + d[..., 2] * d[..., 2]


def _pairs(xyz, sr, chunk=1 << 15):
    """Yield (i, j, d2) for chunks of query points i: every j within sr_i (padded) by a cKDTree, then the float32 d2."""
    tree = cKDTree(xyz.astype(np.float64))
    pad = sr * (1 + 2.0 ** -18) + 1e-6
    for s in range(0, xyz.shape[0], chunk):
        e = min(s + chunk, xyz.shape[0])
        lists = tree.query_ball_point(xyz[s:e].astype(np.float64), pad[s:e], return_sorted=False)
        n = np.fromiter((len(v) for v in lists), dtype=np.int64, count=e - s)
        i = np.repeat(np.arange(s, e), n)
        j = np.fromiter((k for v in lists for k in v), dtype=np.int64, count=int(n.sum()))
        yield i, j, l2_simple(xyz[i], xyz[j])


def neighbour_counts(pc, alpha=0.16, beta=3.0, sr_min=0.04):
    """c_i of the module docstring for every point (cKDTree candidates, exact float32 / float64 re-evaluation)."""
    pc = np.asarray(pc, dtype=np.float32)
    c = np.zeros(pc.shape[0], dtype=np.int64)
    if pc.shape[0] == 0:
        return c
    xyz = np.ascontiguousarray(pc[:, :3])
    sr = search_radius(pc, alpha, beta, sr_min)
    for i, j, d2 in _pairs(xyz, sr):
        hit = np.sqrt(d2.astype(np.float64)) < sr[i]
        c += np.bincount(i[hit], minlength=pc.shape[0])
    return c


def dror_keep(pc, alpha=0.16, beta=3.0, k_min=3, sr_min=0.04):
    """dynamic_radius_outlier_filter (dror.py:288-334): bool mask, True = kept (no snow)."""
    return neighbour_counts(pc, alpha, beta, sr_min) >= k_min + 1


def codes(pc, alpha=0.16, beta=3.0, k_min=3, sr_min=0.04, crop_xy=None):
    """Per row what lss_dror_batch writes: 0 snow, 1 kept, 2 outside the crop (crop variant, dror.py:238-256)."""
    pc = np.asarray(pc, dtype=np.float32)
    out = np.full(pc.shape[0], 2, dtype=np.uint8)
    m = np.ones(pc.shape[0], dtype=bool) if crop_xy is None else cube_mask(pc, *crop_xy)
    out[m] = dror_keep(pc[m], alpha, beta, k_min, sr_min).astype(np.uint8)
    return out


def snow_indices(pc, alpha, crop=True):
    """What process_dense pickles per frame (dror.py:238-259): indices of the snow points of pc (of pc[cube_mask] with
    `crop`), an empty list for an empty (cropped) cloud."""
    pc = np.asarray(pc, dtype=np.float32)
    if crop:
        pc = pc[cube_mask(pc)]
    if len(pc) == 0:
        return []
    keep_mask = dror_keep(pc, alpha=alpha)
    return (keep_mask == 0).nonzero()[0]


def reading_band(pc, alpha=0.16, beta=3.0, sr_min=0.04):
    """Pairs (i, j) whose decision differs between the float64 sqrt of the float32 d2 (the reading taken) and a float32
    sqrt; and the pairs whose sqrt lies within one float32 ulp of sr_i (the band where the two readings could differ)."""
    pc = np.asarray(pc, dtype=np.float32)
    if pc.shape[0] == 0:
        return dict(flips=0, band=0, pairs=0)
    xyz = np.ascontiguousarray(pc[:, :3])
    sr = search_radius(pc, alpha, beta, sr_min)
    ulp = np.spacing(sr.astype(np.float32)).astype(np.float64)
    flips = band = pairs = 0
    for i, j, d2 in _pairs(xyz, sr):
        s64 = np.sqrt(d2.astype(np.float64))
        s32 = np.sqrt(d2).astype(np.float64)
        flips += int(((s64 < sr[i]) != (s32 < sr[i])).sum())
        band += int((np.abs(s64 - sr[i]) <= ulp[i]).sum())
        pairs += int(i.shape[0])
    return dict(flips=flips, band=band, pairs=pairs)


def dror_level(n_snow):
    """create_image_sets.py:53-66: 'none' 0-9, 'light' 10-79, otherwise 'heavy'."""
    for key, value in DROR_LEVELS.items():
        if n_snow in range(value[0], value[1] + 1):
            return key
    return 'heavy'

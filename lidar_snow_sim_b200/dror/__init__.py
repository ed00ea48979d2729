"""
Drop-in mirrors of the reference's DROR de-snowing tools (lib/cadc_devkit/other/dror.py, create_image_sets.py), backed by
the CUDA engine (`SnowfallEngine.dror_batch`, csrc/dror.cu).  NumPy in, NumPy out:

    mask = dynamic_radius_outlier_filter(pc, alpha=0.16, beta=3.0, k_min=3, sr_min=0.04)   # True = kept (dror.py:288-334)
    cube = get_cube_mask(pc)                                                               # dror.py:73-84, z ignored
    idx = snow_indices(pc, alpha=0.45, crop=True)          # what process_dense pickles per frame (dror.py:238-259)
    dror_level(len(idx))                                   # 'none' / 'light' / 'heavy' (create_image_sets.py:16-66)

The rule is computed exactly (DESIGN.md 7.4); parity with python-pcl / FLANN itself is unpinned, as neither is installed.
"""
import numpy as np
import torch

from ..engine import default_engine

# create_image_sets.py:16-18; anything above 'light' is 'heavy' (:53-66)
DROR_LEVELS = {'none': (0, 9), 'light': (10, 79)}
CUBE_XY = (3.0, 13.0, -1.0, 1.0)                 # get_cube_mask's default box as (x0, x1, y0, y1)


def get_cube_mask(pc, x_min=3, x_max=13, y_min=-1, y_max=1, z_min=-1, z_max=1):
    """dror.py:73-84.  Its np.logical_and(x_mask, y_mask, z_mask) passes z_mask as the `out` argument: z is not tested."""
    x_mask = np.logical_and(x_min <= pc[:, 0], pc[:, 0] <= x_max)
    y_mask = np.logical_and(y_min <= pc[:, 1], pc[:, 1] <= y_max)
    z_mask = np.logical_and(z_min <= pc[:, 2], pc[:, 2] <= z_max)
    return np.logical_and(x_mask, y_mask, z_mask)


def _codes(pc, alpha, beta, k_min, sr_min, crop_xy, engine):
    engine = engine or default_engine()
    pts = np.ascontiguousarray(np.asarray(pc)[:, :3], dtype=np.float32)
    d = torch.from_numpy(pts).to(engine.device)
    res = engine.dror_batch(d, np.array([0, pts.shape[0]], dtype=np.int64), alpha=alpha, beta=beta, k_min=k_min,
                            sr_min=sr_min, crop_xy=crop_xy, compact=False)
    engine.check()
    return res['codes'].cpu().numpy()


def dynamic_radius_outlier_filter(pc, alpha=0.16, beta=3.0, k_min=3, sr_min=0.04, *, engine=None):
    """dror.py:288-334: bool mask over the rows of `pc` (xyz = its first three columns), False = snow, True = kept."""
    return _codes(pc, alpha, beta, k_min, sr_min, None, engine) == 1


def snow_indices(pc, alpha, crop=True, *, engine=None):
    """The per-frame result process_dense pickles (dror.py:238-259): int64 indices of the snow points of `pc`, or, with
    `crop`, of pc[get_cube_mask(pc)]; an empty list when that cloud is empty."""
    c = _codes(pc, alpha, 3.0, 3, 0.04, CUBE_XY if crop else None, engine)
    c = c[c != 2]
    if len(c) == 0:
        return []
    return (c == 0).nonzero()[0]


def dror_level(n_snow):
    """The DROR_LEVELS class of a frame's snow count (create_image_sets.py:53-66): 'none' 0-9, 'light' 10-79, 'heavy'."""
    for key, value in DROR_LEVELS.items():
        if n_snow in range(value[0], value[1] + 1):
            return key
    return 'heavy'

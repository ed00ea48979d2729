"""
On-the-fly SNOW / WET_SURFACE augmentation for the reference's training data path.

Mirrors the block of `DenseDataset.__getitem__` that applies the two augmentations
(lib/OpenPCDet/pcdet/datasets/dense/dense_dataset.py:749-837): same config keys and strings
(`SNOW: '<sampling>_<mode>_<chance>'`, `WET_SURFACE: '<chance>[_norm]'`, `COUPLED`), same use of NumPy's global RNG for
the coin flips, same water-height distributions, same exception swallowing around the wet-ground call.

The one difference is the point of the engine: SNOW no longer READS files pre-computed by tools/snowfall/precompute.py
(`<root>/snowfall_simulation/<mode>/<lidar_folder>_rainrate_<int>/<id>.bin`, :778-783) -- it computes the same thing on
the GPU when the sample is requested: camera-FOV filter, augment() with the (snowfall_rate, terminal_velocity) pair
whose rain rate the reference would have picked, FOV filter again (precompute.py:96-104).  Snowflake tables are drawn
on the device once per (mode, pair) and cached.

    aug = OnTheFlyWeather(dataset_cfg, rainfall_rates=[...])        # in DenseDataset.__init__
    points = aug(points, training=self.training)                    # replaces dense_dataset.py:749-837
"""
import numpy as np

from ..dror import dynamic_radius_outlier_filter
from ..engine import default_engine
from ..fog.simulation import ParameterSet, simulate_fog
from ..snowfall.precompute import SNOWFALL_RATES, TERMINAL_VELOCITIES, get_fov_flag

# the (snowfall_rate, terminal_velocity) pairs DenseDataset draws its rain rate from (dense_dataset.py:91-92): eight
# entries, whose rain rates truncate to 2, 4, 8, 17, 34, 70, 130, 200 mm/h
DATASET_SNOWFALL_RATES = [0.5, 0.5, 1.0, 2.0, 2.5, 1.5, 1.5, 1.0]
DATASET_TERMINAL_VELOCITIES = [2.0, 1.2, 1.6, 2.0, 1.6, 0.6, 0.4, 0.2]
from ..snowfall.sampling import snowfall_rate_to_rainfall_rate
from ..snowfall.simulation import augment
from ..wet_ground.augmentation import ground_water_augmentation

_CHANCES = {'8in9': [1, 1, 1, 1, 1, 1, 1, 1, 0], '4in5': [1, 1, 1, 1, 0], '1in2': [1, 0], '1in4': [1, 0, 0, 0],
            '1in10': [1, 0, 0, 0, 0, 0, 0, 0, 0, 0]}                     # dense_dataset.py:761-770


class OnTheFlyWeather:
    def __init__(self, dataset_cfg, rainfall_rates=None, engine=None, table_seed=42, only_precomputed=False):
        """rainfall_rates: the list `int(np.random.choice(...))` draws from; default = the reference's own eight rain
        rates (dense_dataset.py:91-102), so 'uniform' sampling has the reference's distribution and consumes NumPy's
        global RNG identically.  The drawn value is truncated to the integer the pre-computed folders are named after
        (precompute.py:88-89) and mapped back to its (snowfall_rate, terminal_velocity) pair: precompute.py's five
        pairs first (what the file would have contained), then the dataset's eight.  The reference finds no file for
        the three rates precompute.py does not produce and skips the augmentation with a message; here they are
        computed on the fly unless `only_precomputed`."""
        self.cfg = dataset_cfg
        self.engine = engine
        self.table_seed = table_seed
        self.pairs = {}

        def register(rates, velocities):
            for rs, tv in zip(rates, velocities):
                key = int(snowfall_rate_to_rainfall_rate(rs, tv))
                if key in self.pairs and self.pairs[key] != (rs, tv):
                    raise ValueError(f'rain rates of {self.pairs[key]} and {(rs, tv)} both truncate to {key} mm/h: '
                                     f'the folder name rainrate_{key} would be ambiguous')
                self.pairs.setdefault(key, (rs, tv))

        register(SNOWFALL_RATES, TERMINAL_VELOCITIES)
        if not only_precomputed:
            register(DATASET_SNOWFALL_RATES, DATASET_TERMINAL_VELOCITIES)
        if rainfall_rates is None:
            rainfall_rates = [snowfall_rate_to_rainfall_rate(rs, tv)
                              for rs, tv in zip(DATASET_SNOWFALL_RATES, DATASET_TERMINAL_VELOCITIES)]
        self.rainfall_rates = list(rainfall_rates)
        self._tables = {}

    def _engine(self):
        if self.engine is None:
            self.engine = default_engine()
        return self.engine

    def _table(self, mode, rainfall_rate):
        key = (mode, rainfall_rate)
        if key not in self._tables:
            if rainfall_rate not in self.pairs:
                raise FileNotFoundError(f'no (snowfall_rate, terminal_velocity) pair with rain rate {rainfall_rate}')
            rs, tv = self.pairs[rainfall_rate]
            self._tables[key] = self._engine().sample_tables_device(mode, rs, tv, seed=self.table_seed)
        return self._tables[key]

    def __call__(self, points, training=True):
        cfg = self.cfg
        snowfall_augmentation_applied = False
        if training and 'SNOW' in cfg:
            sampling, mode, chance = cfg['SNOW'].split('_')[:3]
            choices = _CHANCES.get(chance, [0])
            if np.random.choice(choices):
                rainfall_rate = 0
                if sampling == 'uniform':
                    rainfall_rate = int(np.random.choice(self.rainfall_rates))
                try:
                    tid = self._table(mode, rainfall_rate)
                    pc = np.ascontiguousarray(points[:, :5], dtype=np.float32)
                    pc = pc[get_fov_flag(pc[:, 0:3])]                                  # precompute.py:96-99
                    _, points = augment(pc, '', float(np.degrees(3e-3)), engine=self._engine(), tables=tid)
                    snowfall_augmentation_applied = True
                except FileNotFoundError as exc:                                       # dense_dataset.py:784-786
                    print(f'\n{exc}')
        if training and 'WET_SURFACE' in cfg:
            method = cfg['WET_SURFACE']
            choices = [0]
            if '1in2' in method:
                choices = [0, 1]
            elif '1in4' in method:
                choices = [0, 0, 0, 1]
            elif '1in10' in method:
                choices = [0, 0, 0, 0, 0, 0, 0, 0, 0, 1]
            apply_coupled = 'COUPLED' in cfg and snowfall_augmentation_applied
            if 'COUPLED' in cfg:
                choices = [0]
            if np.random.choice(choices) or apply_coupled:
                if 'norm' in method:
                    from scipy import stats
                    lower, upper, mu, sigma = 0.05, 0.5, 0.2, 0.1
                    water_height = stats.truncnorm((lower - mu) / sigma, (upper - mu) / sigma, loc=mu, scale=sigma).rvs(1)
                else:
                    elements = np.linspace(0.1, 1.2, 12)
                    probabilities = 5 * np.ones_like(elements)
                    probabilities[0], probabilities[1], probabilities[2] = 15, 25, 15
                    water_height = np.random.choice(elements, 1, p=probabilities / 100)
                try:
                    points = ground_water_augmentation(points, water_height=float(np.asarray(water_height).reshape(-1)[0]),
                                                       debug=False, engine=self._engine())
                except (TypeError, ValueError):                                        # dense_dataset.py:834-837
                    pass
        return points


def apply_dror(points, dataset_cfg, split, engine=None):
    """The DROR / DROR++ block of `DenseDataset.__getitem__` (dense_dataset.py:588-616) without its pickles: the reference
    reads the snow indices of the `full` variant from `training/DROR/alpha_<alpha>/all/<sensor>/<signal>/full/<id>.pkl`
    (written offline by lib/cadc_devkit/other/dror.py); here they are computed on the device at any alpha.
    `DROR` applies always, `DROR++` only when 'snow' is in the split name; both drop the snow rows of `points`.
    With both keys set the second filter runs on the output of the first (the reference indexes the filtered cloud with
    indices computed on the unfiltered one)."""
    if 'DROR' in dataset_cfg:
        points = points[dynamic_radius_outlier_filter(points, alpha=float(dataset_cfg['DROR']), engine=engine)]
    if 'DROR++' in dataset_cfg and 'snow' in split:
        points = points[dynamic_radius_outlier_filter(points, alpha=float(dataset_cfg['DROR++']), engine=engine)]
    return points


def foggify_cvl(points, alpha, dataset_cfg, engine=None, lut_dir=None, rng=None):
    """The 'CVL' branch of `DenseDataset.foggify` (lib/OpenPCDet/pcdet/datasets/dense/dense_dataset.py:988-1009): fog
    simulation with attenuation `alpha` (a string like '0.060' in the reference's curriculum; '0.000' = clear) and the
    optional config keys FOG_GAIN / FOG_NOISE_VARIANT / FOG_SOFT / FOG_HARD, computed by the engine."""
    if alpha == '0.000' or float(alpha) == 0.0:
        return points
    p = ParameterSet(alpha=float(alpha), gamma=0.000001)
    soft, hard, gain, fog_noise_variant = True, True, False, 'v1'
    if 'FOG_GAIN' in dataset_cfg:
        gain = dataset_cfg['FOG_GAIN']
    if 'FOG_NOISE_VARIANT' in dataset_cfg:
        fog_noise_variant = dataset_cfg['FOG_NOISE_VARIANT']
    if 'FOG_SOFT' in dataset_cfg:
        soft = dataset_cfg['FOG_SOFT']
    if 'FOG_HARD' in dataset_cfg:
        hard = dataset_cfg['FOG_HARD']
    points, _, _ = simulate_fog(p, pc=points, noise=10, gain=gain, noise_variant=fog_noise_variant, soft=soft, hard=hard,
                                engine=engine, lut_dir=lut_dir, rng=rng)
    return points

#!/usr/bin/env python
"""
bench.py -- snowfall (+ wet-ground) augmentation throughput on B200 (BASELINE.json metric: augmented LiDAR points/s).

    python bench.py --gpus 1 --steps 20 --warmup 5                     # our arm (CUDA engine), BASELINE configs[1]
    python bench.py --config 2                                         # configs[2]: snowfall + wet ground fused on device
    python bench.py --impl reference --steps 3 --warmup 1              # CPU arm: the oracle port on all host cores
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W                          # N ranks, one per GPU, weak scaling (configs[3])

Workload: batch = 32 synthetic 64 x 2048 clouds per GPU, snowfall_rate 2.5 mm/h, terminal velocity 1.6 m/s,
Gunn-Marshall size distribution, tables from dart throwing (seed 1000 + plane; the engine's native sampler and the
oracle's NumPy restatement produce the same tables bit for bit, tests/test_sampler.py).  One step = one pass of the
whole augment() pipeline over the batch: [pre-pass], per-beam scan + solve, threshold filter, channel sort +
compaction, stats (config 2: followed by ground_water_augmentation(water_height = 1 mm) on the snow output, on the
device).  With N > 1 every rank augments its own 32 clouds (clouds are independent, no data-path collective) and one
all-gather reassembles the augmented batch on every rank (configs[3]).

`value`     device-resident inputs.  The K timed steps run as one bracket between one CUDA-event pair on the launching
            stream (barrier + synchronize on both sides, max over ranks).  Two input batches alternate so that no step
            finds its rows in L2.
`e2e`       the public API with pinned HOST buffers: H2D of the batch + augment + D2H of the augmented batch, per step
            (K pipelined steps, then K synchronous calls)
`roofline`  the beam stage (scan + solve kernels) against the measured HBM copy peak; algorithmic bytes per launch =
            40 B x points + 12 B x table particles (SURVEY.md 8d), durations from CUDA events on the launching stream
`cpu_baseline` / --impl reference
            the CPU oracle port (oracle/) on all host cores: one worker process per cloud (4 threads each for its 64
            channel tasks), 32 clouds per step, median step; tables from the oracle's own dart throwing -- this arm never
            loads the product library

--dump-outputs DIR writes what the last timed step returned as DIR/<name>.npy (float32 / float64): every per-cloud
array in full and, of the augmented rows, the kept rows of a fixed seeded sample of clouds (`points_clouds`), < 64 MB in
all.  The inputs depend only on the arguments, so two builds can be compared output for output.
"""
import argparse
import json
import os
import random
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the benchmark writes nothing into the tree it runs from (it may be read-only)

SNOWFALL_RATE = 2.5
TERMINAL_VELOCITY = 1.6
MODE = 'gunn'
TABLE_SEED = 1000
BATCH_PER_GPU = 32
N_AZIMUTH = 2048
DIV_DEG = float(np.degrees(3e-3))
WATER_HEIGHT = 0.001                # config 2 (BASELINE.json configs[2])
ALGO_BYTES_PER_POINT = 40           # read 5 x f32, write 5 x f32 (SURVEY.md 8d)
ALGO_BYTES_PER_PARTICLE = 12        # f32 x, y, r once per launch (SURVEY.md 8d)
FIXED_POLY = (2e-3, -0.3, 12.0)     # only used with --host-threshold
CPU_CLOUDS_PER_STEP = 32
CPU_THREADS_PER_CLOUD = 4
DUMP_POINTS_BYTES = 48 << 20        # --dump-outputs: budget of the sampled kept rows (the per-cloud arrays are small)
STEPS_IN_FLIGHT = 1                 # device-resident leg: consecutive steps on alternating streams (1 = strictly serial)


def load_peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        return float(json.load(open(p))['hbm_gbs']), 'measured (MEASURED_PEAKS.json)'
    return 6650.0, 'fallback (B200_PROFILING.md)'


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe).  The sampler runs from
    before the warm-up (nvidia-smi needs ~0.2 s to start); samples are stamped on arrival and the ones that fall inside
    the timed window are reported."""
    Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')

    def __init__(self, gpu_index):
        self.rows = []
        self.proc = None
        self.gpu_index = gpu_index
        self.t0 = self.t1 = None

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', f'--query-gpu={self.Q}', '--format=csv,noheader,nounits',
                                          '-lms', '20', '-i', str(self.gpu_index)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [t.strip() for t in line.split(',')]))

    def window_begin(self):
        self.t0 = time.perf_counter()

    def window_end(self):
        self.t1 = time.perf_counter()

    def stop(self):
        if not self.proc:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        time.sleep(0.1)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        rows = [r for (t, r) in self.rows if self.t0 is not None and self.t0 - 0.02 <= t <= self.t1 + 0.03]
        window = 'inside the timed region'
        if not rows and self.rows:
            mid = 0.5 * ((self.t0 or 0) + (self.t1 or 0))
            rows = [r for (t, r) in sorted(self.rows, key=lambda tr: abs(tr[0] - mid))[:3]]
            window = 'nearest samples (timed region shorter than the sampling period)'
        sm, mx, reasons = [], [], set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for r in rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
                for k, nme in enumerate(names):
                    if r[5 + k].lower().startswith('active'):
                        reasons.add(nme)
            except Exception:
                pass
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': max(mx) if mx else None,
                'reasons': sorted(reasons), 'samples': len(sm), 'window': window}


def make_workload(rank, batch, seed0=0):
    from lidar_snow_sim_b200.synthetic import synthetic_cloud
    clouds = [synthetic_cloud(seed=seed0 + rank * 10000 + b, n_azimuth=N_AZIMUTH) for b in range(batch)]
    orders = []
    for b in range(batch):
        r = random.Random(seed0 + rank * 10000 + b)
        o = list(range(64))
        r.shuffle(o)                                # the reference's random.shuffle(order), simulation.py:486
        orders.append(o)
    return clouds, np.array(orders, dtype=np.int32)


def workload_config(config, n_gpus):
    """The SAME dict on both arms (the driver compares them)."""
    what = 'BASELINE.json configs[1]' if config == 1 else 'BASELINE.json configs[2] (snowfall + wet ground fused, water_height=1 mm)'
    return {'workload': f'{what}: batch={BATCH_PER_GPU} synthetic 64x{N_AZIMUTH} clouds per GPU, '
                        f'snowfall_rate={SNOWFALL_RATE} mm/h, v={TERMINAL_VELOCITY} m/s, {MODE} DSD (dart-throwing tables, '
                        f'seed {TABLE_SEED}+plane), beam_divergence=3 mrad, noise_floor=0.7, only_camera_fov=False'
                        + ('' if n_gpus == 1 else f'; x{n_gpus} GPUs + all-gather of the augmented batch (configs[3])'),
            'config': config, 'batch_per_gpu': BATCH_PER_GPU, 'points_per_cloud': 64 * N_AZIMUTH,
            'parallelism': f'clouds sharded x{n_gpus}',
            'l2': 'no explicit flush: two different input batches alternate (2 x 84 MB of rows + the table index > 126 MB '
                  'L2); a bracket of K steps is timed with one CUDA-event pair on the launching stream'}


# ----------------------------------------------------------------------------------------------------------------------
# CPU arm (oracle port) -- never imports the product library
# ----------------------------------------------------------------------------------------------------------------------
_REF_STATE = None


def _ref_init(tables, sensor, clouds, orders, poly, threads, config):
    global _REF_STATE
    from oracle import oracle as orc
    orc.lib()
    _REF_STATE = (orc, tables, sensor, clouds, orders, poly, threads, config)


def _ref_one_cloud(k):
    orc, tables, sensor, clouds, orders, poly, threads, config = _REF_STATE
    stats, aug = orc.augment(clouds[k], tables, DIV_DEG, sensor, order=orders[k].tolist(), thresh_poly=poly,
                             threads=threads, stable_sort=True)
    if config == 2:         # the viewer's chaining, pointcloud_viewer.py:2804-2821
        aug = orc.ground_water_augmentation(aug, water_height=WATER_HEIGHT, replace=False)
    return stats, aug.shape[0]


def _oracle_plane(k):
    from oracle import oracle as orc
    occ = orc.compute_occupancy(SNOWFALL_RATE, TERMINAL_VELOCITY)
    rr = float(orc.snowfall_rate_to_rainfall_rate(SNOWFALL_RATE, TERMINAL_VELOCITY))
    return orc.dart_throwing(occ, rr, 80.0, np.random.default_rng(TABLE_SEED + k), MODE)


def oracle_tables(cores):
    """The 64 planes of the workload from the ORACLE's dart throwing (tools/snowfall/sampling.py:90-194 restated with
    NumPy), one process per plane, cached as .npy in the temp dir like the reference caches its tables as files
    (sampling.py:344)."""
    import multiprocessing as mp
    cache = os.path.join(tempfile.gettempdir(), f'lss_oracle_tables_{MODE}_{SNOWFALL_RATE}_{TERMINAL_VELOCITY}_{TABLE_SEED}.npz')
    if os.path.exists(cache):
        try:
            z = np.load(cache)
            return [z[f'p{k}'] for k in range(64)], 'cached'
        except Exception:
            pass
    with mp.get_context('spawn').Pool(max(1, min(cores, 64))) as pool:
        tables = pool.map(_oracle_plane, range(64), chunksize=1)
    try:
        np.savez(cache, **{f'p{k}': t for k, t in enumerate(tables)})
    except Exception:
        pass
    return tables, 'oracle.dart_throwing'


class CpuArm:
    """One worker process per cloud of a step, CPU_THREADS_PER_CLOUD threads each for its 64 channel tasks."""

    def __init__(self, tables, clouds, orders, poly, config, clouds_per_step=None):
        import multiprocessing as mp
        from lidar_snow_sim_b200.calib.hdl64e_s3 import sensor_arrays
        self.cores = os.cpu_count() or 1
        n = clouds_per_step or CPU_CLOUDS_PER_STEP
        self.n_clouds = max(1, min(n, len(clouds), max(1, self.cores // 2)))
        self.threads = max(1, min(CPU_THREADS_PER_CLOUD, self.cores // self.n_clouds))
        self.clouds = clouds
        self.pool = mp.get_context('spawn').Pool(self.n_clouds, initializer=_ref_init,
                                                 initargs=(tables, sensor_arrays(), clouds, orders, poly, self.threads,
                                                           config))
        self.pool.map(_ref_one_cloud, [], chunksize=1)      # workers up before timing

    def step(self, n=None):
        n = n or self.n_clouds
        t0 = time.perf_counter()
        self.pool.map(_ref_one_cloud, range(n), chunksize=1)
        return time.perf_counter() - t0, sum(self.clouds[k].shape[0] for k in range(n))

    def close(self):
        self.pool.close()


def run_reference(args):
    """CPU arm: the oracle port (oracle/, restating tools/snowfall/simulation.py + tools/wet_ground) on all host cores."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    from oracle import oracle as orc
    orc.build()
    cores = os.cpu_count() or 1
    tables, table_src = oracle_tables(cores)
    clouds, orders = make_workload(0, CPU_CLOUDS_PER_STEP)
    arm = CpuArm(tables, clouds, orders, np.array(FIXED_POLY) if args.host_threshold else None, args.config,
                 args.cpu_clouds if args.cpu_clouds > 0 else None)
    # bounded: the whole --steps K --warmup W run must end within a few minutes whatever K the driver passes.  The first
    # step is measured; if K + W such steps would take more than ~4 minutes the remaining steps use fewer clouds.
    budget_s = 240.0
    n_step = arm.n_clouds
    times, pts_list = [], []
    total = args.warmup + args.steps
    for s in range(total):
        dt, pts = arm.step(n_step)
        if s >= args.warmup:
            times.append(dt)
            pts_list.append(pts)
        elif s == 0 and dt * total > budget_s and args.cpu_clouds <= 0:
            n_step = max(4, int(n_step * budget_s / (dt * total)))
    if not times:
        dt, pts = arm.step(n_step)
        times.append(dt)
        pts_list.append(pts)
    arm.close()
    rates = np.array(pts_list) / np.array(times)
    value = float(np.median(rates))
    dt_med = float(np.median(times))
    sample = (f'{n_step} clouds of 64x{N_AZIMUTH} per step ({pts_list[0]} points), full augment() incl. pre-pass'
              f'{" + ground_water_augmentation" if args.config == 2 else ""}; {n_step} worker processes x {arm.threads} '
              f'threads on {cores} cores; median of {len(times)} timed steps (min {min(times):.2f} s, max {max(times):.2f} s); '
              f'tables: {table_src}')
    line = {'impl': 'reference', 'metric': 'augmented LiDAR points/sec', 'value': value, 'unit': 'points/s',
            'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': dt_med * 1e3,
            'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
            'config': workload_config(args.config, args.gpus),
            'cpu_baseline': {'value': value, 'unit': 'points/s', 'cores': cores, 'kind': 'port', 'sample': sample},
            'e2e': {'value': value, 'unit': 'points/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
            'clouds_per_s': value / (64 * N_AZIMUTH), 'ms_per_step_mean': float(np.mean(times)) * 1e3}
    print(json.dumps(line))


# ----------------------------------------------------------------------------------------------------------------------
# our arm
# ----------------------------------------------------------------------------------------------------------------------
def dump_outputs(out_dir, res, off, seed=0):
    """Write one step's result dict as <out_dir>/<name>.npy: the per-cloud arrays in full (float64), and of the
    slot-compacted rows `points` only the kept rows of a fixed seeded sample of clouds that fits DUMP_POINTS_BYTES
    (float32, concatenated in cloud order; the clouds in `points_clouds`)."""
    os.makedirs(out_dir, exist_ok=True)
    counts = res['counts'].cpu().numpy().astype(np.int64)
    n_per = np.diff(off)
    n_clouds = min(len(n_per), DUMP_POINTS_BYTES // (20 * int(n_per.max())))
    clouds = np.sort(np.random.default_rng(seed).choice(len(n_per), n_clouds, replace=False))
    pts = res['points']
    arrays = {'points': np.concatenate([pts[off[b]:off[b] + counts[b]].cpu().numpy() for b in clouds]),
              'points_clouds': clouds.astype(np.float64)}
    arrays.update({name: t.cpu().numpy().astype(np.float64) for name, t in res.items() if name != 'points'})
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f'{name}.npy'), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--config', type=int, default=1, choices=[1, 2, 3],
                    help='BASELINE.json configs[k]: 1 snowfall, 2 snowfall + wet ground fused, 3 = 1 on --gpus N with the gather')
    ap.add_argument('--batch', type=int, default=BATCH_PER_GPU)
    ap.add_argument('--cpu-clouds', type=int, default=0, help='clouds per step of the CPU arm / cpu_baseline sample')
    ap.add_argument('--host-threshold', action='store_true',
                    help='skip the device pre-pass and use a fixed threshold polynomial (debug only; reported in config)')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-e2e', action='store_true')
    ap.add_argument('--no-gather', action='store_true', help='N > 1: replicas only, skip the all-gather (debug)')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help="write the last timed step's outputs as DIR/<name>.npy (rank 0's batch)")
    ap.add_argument('--streams', type=int, default=STEPS_IN_FLIGHT, choices=[1, 2],
                    help='steps in flight in the device-resident leg: consecutive steps alternate between this many streams')
    ap.add_argument('--e2e-inflight', type=int, default=3, help='batches in flight in the e2e leg (1..3)')
    ap.add_argument('--e2e-chunks', type=int, default=2, help='chunks of the host-to-host pipeline (e2e leg)')
    args = ap.parse_args()
    args.steps = max(1, args.steps)
    args.warmup = max(3, args.warmup) if args.impl == 'b200' else max(0, args.warmup)
    if args.config == 3:
        args.config = 1

    if args.impl == 'reference':
        run_reference(args)
        return

    import torch
    import torch.distributed as dist
    from lidar_snow_sim_b200.engine import SnowfallEngine
    from lidar_snow_sim_b200.snowfall.sampling import sample_table_set

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    assert torch.cuda.is_available(), 'bench.py needs a GPU (no CPU fallback for the b200 arm)'
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    assert world == args.gpus or world == 1, f'--gpus {args.gpus} but WORLD_SIZE={world}'

    # e2e leg with several ranks on one box: the host's memory bandwidth is the limiter (tools/e2e_probe_ranks.py), so the
    # copy-out kernel that moves only the kept rows pays (8 ranks: 5.98 vs 6.84 ms per step); on one GPU the plain D2H copy
    # is faster (2.06 vs 2.12 ms) and stays the default.  Read by the library when its host pipeline is created.
    if world > 1:
        os.environ.setdefault('LSS_PIPE_KERNEL_OUT', '1')
    numa_cpus = None
    if world > 1 and os.environ.get('LSS_NUMA_BIND', '0') == '1':
        try:
            from lidar_snow_sim_b200.distributed import bind_host_to_gpu
            numa_cpus = bind_host_to_gpu(local_rank)      # pinned host buffers land on the GPU's own NUMA node
        except Exception:
            numa_cpus = None
    eng = SnowfallEngine(local_rank)
    tables = sample_table_set(MODE, SNOWFALL_RATE, TERMINAL_VELOCITY, seed=TABLE_SEED)
    tid = eng.upload_tables(tables)
    tinfo = eng.table_info(tid)
    B = args.batch
    fused_wet = args.config == 2
    # two different batches per rank, used alternately: 2 x 84 MB of rows (+ the index) per pair of steps is more
    # than the 126 MB L2, so no step finds its inputs cached by the previous one (no explicit flush needed)
    clouds, orders = make_workload(rank, B)
    clouds2, orders2 = make_workload(rank, B, seed0=500000)
    n_per = [c.shape[0] for c in clouds]
    off = np.concatenate([[0], np.cumsum(n_per)]).astype(np.int64)
    N = int(off[-1])
    assert [c.shape[0] for c in clouds2] == n_per
    host_pts = torch.from_numpy(np.concatenate(clouds)).pin_memory()
    d_pts = [host_pts.to(dev), torch.from_numpy(np.concatenate(clouds2)).to(dev)]
    d_orders = [orders, orders2]
    poly = np.tile(np.array(FIXED_POLY), (B, 1)) if args.host_threshold else None
    device_prepass = not args.host_threshold
    outs = [{}, {}]
    do_gather = world > 1 and not args.no_gather
    gather = None
    if do_gather:
        from lidar_snow_sim_b200.distributed import BatchGather
        gather = BatchGather(N, B, dev, depth=2, engine=eng, cloud_offsets=off)

    # config 2: the wet stage of step k runs on its own stream next to the snow stage of step k + 1 (both are chains of
    # latency-bound kernels; the wet pre-pass can only start when the snow output exists).  Double-buffered, stream-ordered.
    n_streams = max(1, min(2, args.streams))
    step_streams = [torch.cuda.Stream(device=dev) for _ in range(n_streams)] if n_streams > 1 else None
    step_ws = None
    if step_streams is not None:       # one engine workspace per stream: the steps in flight must not share scratch
        need = eng.lib.lss_snowfall_workspace_bytes(N, B)
        step_ws = [torch.empty(int(need) + 256, dtype=torch.uint8, device=dev) for _ in range(n_streams)]
    step_done = [None, None]
    wet_stream = torch.cuda.Stream(device=dev) if fused_wet else None
    wet_outs = [{}, {}]
    ev_snow = [torch.cuda.Event() for _ in range(2)]
    ev_wet = [None, None]

    def step(k):
        """One pass of the augment() pipeline over this rank's batch (config 2: + wet ground on the snow output); with
        N > 1 followed by the all-gather of the augmented batch (SURVEY.md 8e), overlapping the next step's kernels
        (double-buffered)."""
        j = k & 1
        if step_streams is not None:                       # consecutive steps alternate between the streams
            with torch.cuda.stream(step_streams[j % n_streams]):
                return _step_on_current_stream(j)
        return _step_on_current_stream(j)

    def _step_on_current_stream(j):
        if gather is not None:
            gather.wait(j)
        cur = torch.cuda.current_stream(dev)
        if fused_wet and ev_wet[j] is not None:
            cur.wait_event(ev_wet[j])                      # the wet stage two steps ago still reads outs[j]
        r = eng.snowfall_batch(tid, d_pts[j], off, d_orders[j], DIV_DEG, thresh_poly=poly, device_prepass=device_prepass,
                               out=outs[j], workspace=None if step_ws is None else step_ws[j % n_streams])
        if step_streams is not None:
            step_done[j] = torch.cuda.Event()
            step_done[j].record(cur)
        if fused_wet:
            ev_snow[j].record(cur)
            with torch.cuda.stream(wet_stream):
                wet_stream.wait_event(ev_snow[j])
                r = eng.wet_ground_batch(r['points'], off, counts=r['counts'], water_height=WATER_HEIGHT, replace=False,
                                         out=wet_outs[j])
                ev_wet[j] = torch.cuda.Event()
                ev_wet[j].record(wet_stream)
        if gather is not None:
            gather.start(j, r['points'], r['counts'])
        return r

    def drain():
        if step_streams is not None:
            for ev in step_done:
                if ev is not None:
                    torch.cuda.current_stream(dev).wait_event(ev)
        if gather is not None:
            gather.wait_all()
        if fused_wet:
            for ev in ev_wet:
                if ev is not None:
                    torch.cuda.current_stream(dev).wait_event(ev)

    def sync_all():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize(dev)

    def bracket(n_steps, k0=0):
        """EXACTLY n_steps steps between one CUDA-event pair (the last gathers are inside the bracket)."""
        e0 = torch.cuda.Event(enable_timing=True)
        e1 = torch.cuda.Event(enable_timing=True)
        sync_all()
        e0.record()
        if step_streams is not None:
            for st in step_streams:
                st.wait_event(e0)
        for k in range(n_steps):
            step(k0 + k)
        drain()
        e1.record()
        sync_all()
        return float(e0.elapsed_time(e1))

    # ---- device-resident throughput (`value`) ------------------------------------------------------------------------
    clocks = ClockSampler(local_rank)
    clocks.start()
    for k in range(args.warmup):
        step(k)
    drain()
    eng.check()
    launches0 = eng.launch_count()
    clocks.window_begin()
    total_ms = bracket(args.steps)
    clocks.window_end()
    launches = eng.launch_count() - launches0
    clk = clocks.stop()
    eng.check()
    if args.dump_outputs and rank == 0:                     # the bracket's steps are k = 0 .. K-1
        last = (args.steps - 1) & 1
        dump_outputs(args.dump_outputs, wet_outs[last] if fused_wet else outs[last], off)
    t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms = float(t.item())
    ms_per_step = total_ms / args.steps
    points_all = N * world
    value = points_all / (ms_per_step * 1e-3)

    # per-kernel durations: one more bracket with CUDA events around every launch (kept out of the timed brackets)
    eng.set_profiling(True)
    eng.kernel_times(reset=True)
    bracket(args.steps)
    ktimes = eng.kernel_times(reset=True)
    eng.set_profiling(False)
    orders = d_orders[0]

    # ---- label mismatch caused by the device azimuth alone (the timed path computes theta on the device) ---------------
    theta_info = None
    if rank == 0:
        c0 = clouds[0]
        d_c0 = torch.from_numpy(c0).to(dev)
        th_host = torch.from_numpy(np.arctan2(c0[:, 1], c0[:, 0]).astype(np.float32)).to(dev)
        o1 = np.array([0, c0.shape[0]], dtype=np.int64)
        ra = eng.snowfall_batch(tid, d_c0, o1, orders[:1], DIV_DEG, threshold_filter=False, want_full=True)
        fa = ra['full'].clone()
        rb = eng.snowfall_batch(tid, d_c0, o1, orders[:1], DIV_DEG, threshold_filter=False, want_full=True, theta=th_host)
        eng.check()
        diff = int((fa[:, 4] != rb['full'][:, 4]).sum().item())
        theta_info = {'rate': diff / c0.shape[0], 'beams': int(c0.shape[0]), 'differing_labels': diff,
                      'what': 'labels with the device azimuth (correctly rounded float32 of the float64 atan2) vs with this '
                              "host's float32 np.arctan2 injected as d_theta, cloud 0 of the workload"}

    # ---- end to end through the public API with host buffers (`e2e`) --------------------------------------------------
    e2e = None
    if not args.no_e2e:
        if not fused_wet:
            # The public host-to-host API, called the way a prefetching data loader calls it: up to `depth` batches are in
            # flight (one pinned result buffer each), so that batch k+1's copy-in overlaps batch k's kernels and batch k-1's
            # copy-out.  Every step moves its own input H2D and its own result D2H inside the timed region.
            depth = max(1, min(3, args.e2e_inflight))
            host_outs = [{} for _ in range(depth)]
            e2e_kw = dict(thresh_poly=poly, device_prepass=device_prepass, n_chunks=args.e2e_chunks)

            def e2e_run(steps):
                tickets = []
                for k in range(steps):
                    if len(tickets) == depth:
                        eng.snowfall_batch_host_wait(tickets.pop(0))        # the caller consumes the oldest batch here
                    tickets.append(eng.snowfall_batch_host_submit(tid, host_pts, off, orders, DIV_DEG,
                                                                  host_out=host_outs[k % depth], **e2e_kw))
                for tk in tickets:
                    eng.snowfall_batch_host_wait(tk)

            def e2e_sync(steps):
                for _ in range(steps):
                    eng.snowfall_batch_host(tid, host_pts, off, orders, DIV_DEG, host_out=host_outs[0], **e2e_kw)
            how = ('host wall clock around K steps of the C-ABI host-buffer calls lss_snowfall_batch_host_submit / _wait '
                   '(pinned host in -> copy-in / pre-pass / beam / copy-out streams -> pinned host out), with up to '
                   'batches_in_flight steps submitted before the oldest is awaited; sync_call = the same batches through '
                   'the synchronous lss_snowfall_batch_host, one at a time; with N > 1 every rank feeds its own host-side '
                   'consumer, no gather')
        else:
            depth = 1
            h_out = torch.empty((N, 5), dtype=torch.float32).pin_memory()
            h_cnt = torch.empty((B,), dtype=torch.int32).pin_memory()
            d_in = torch.empty((N, 5), dtype=torch.float32, device=dev)

            def e2e_sync(steps):
                for _ in range(steps):
                    d_in.copy_(host_pts, non_blocking=True)
                    r = eng.snowfall_batch(tid, d_in, off, orders, DIV_DEG, thresh_poly=poly,
                                           device_prepass=device_prepass, out=outs[0])
                    w = eng.wet_ground_batch(r['points'], off, counts=r['counts'], water_height=WATER_HEIGHT, replace=False)
                    h_out.copy_(w['points'], non_blocking=True)
                    h_cnt.copy_(w['counts'], non_blocking=True)
                    torch.cuda.synchronize(dev)
            e2e_run = e2e_sync
            how = ('host wall clock around K steps of: pinned host -> device copy, engine.snowfall_batch, '
                   'engine.wet_ground_batch on the slot-compacted snow output, device -> pinned host copy of rows + counts, '
                   'synchronize (no pipelining across steps in this configuration)')

        e2e_run(3)
        sync_all()
        t0 = time.perf_counter()
        e2e_run(args.steps)
        sync_all()
        dt = (time.perf_counter() - t0) / args.steps
        t0 = time.perf_counter()
        e2e_sync(args.steps)
        dt_sync = (time.perf_counter() - t0) / args.steps
        tt = torch.tensor([dt, dt_sync], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dt, dt_sync = float(tt[0].item()), float(tt[1].item())
        kernel_out = (not fused_wet) and os.environ.get('LSS_PIPE_KERNEL_OUT') == '1'
        rows_out = N
        if kernel_out:                                     # only the kept rows travel: count them from the result
            rows_out = int(host_outs[0]['counts'].sum().item())
        e2e = {'value': points_all / dt, 'unit': 'points/s', 'h2d_bytes_per_step': int(N * 20),
               'd2h_bytes_per_step': int(rows_out * 20 + B * 4 + (0 if fused_wet else B * 32)), 'ms_per_step': dt * 1e3,
               'steps_timed': args.steps,
               'sync_call': {'value': points_all / dt_sync, 'ms_per_step': dt_sync * 1e3},
               'chunks': args.e2e_chunks, 'batches_in_flight': depth,
               'copy_out': 'kept rows by kernel' if kernel_out else 'whole slot by copy engine',
               'host_numa_bound_cpus': None if numa_cpus is None else len(numa_cpus), 'timing': how}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the beam stage ----------------------------------------------------------------------------------------
    peak, peak_src = load_peaks()
    k_ms, k_calls = ktimes.get('snowfall', (0.0, 0))
    k_avg_ms = k_ms / max(k_calls, 1)
    algo_bytes = ALGO_BYTES_PER_POINT * N + ALGO_BYTES_PER_PARTICLE * tinfo['n_particles']
    achieved = algo_bytes / (k_avg_ms * 1e-3) / 1e9 if k_avg_ms > 0 else 0.0
    per_step = {k: (v[0] / max(v[1], 1)) * (v[1] / args.steps) for k, v in ktimes.items() if v[1]}
    roofline = {'bound': 'hbm',
                'kernel': 'beam stage = k_scan (all beams) + k_list_sort + k_solve (dominant: the beams with '
                          'occluders) + overflow kernel, one CUDA-event pair around the four launches',
                'achieved': achieved, 'peak': peak, 'unit': 'GB/s', 'frac': achieved / peak, 'traffic': None,
                'peak_source': peak_src, 'algorithmic_bytes_per_launch': int(algo_bytes),
                'algorithmic_bytes': f'{ALGO_BYTES_PER_POINT} B x {N} points + {ALGO_BYTES_PER_PARTICLE} B x '
                                     f'{tinfo["n_particles"]} table particles (SURVEY.md 8d)',
                'kernel_ms': k_avg_ms, 'kernel_share_of_step': k_avg_ms / ms_per_step,
                'frac_over_whole_step': algo_bytes / (ms_per_step * 1e-3) / 1e9 / peak,
                'kernel_ms_all': per_step,
                'note': 'latency / issue bound, not HBM bound (DESIGN.md 4, profiles/): durations are CUDA events on the '
                        'launching stream in a separate profiled bracket (event pairs around every launch would perturb the '
                        'timed brackets); the pre-pass runs concurrently on a side stream, so kernel_ms_all sums to more than '
                        'the step; traffic = dram bytes of the beam-stage launches from the ncu capture in profiles/traffic.json'}
    prof = os.path.join(ROOT, 'profiles', 'traffic.json')
    if os.path.exists(prof):
        try:
            roofline['traffic'] = json.load(open(prof)).get('beam_stage_dram_bytes_per_launch')
        except Exception:
            pass

    # ---- CPU baseline (oracle port, bounded sample: one warm-up + two timed steps of 32 clouds) ---------------------------
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        from oracle import oracle as orc
        orc.build()
        arm = CpuArm(tables, clouds, orders, None if device_prepass else np.array(FIXED_POLY), args.config,
                     args.cpu_clouds if args.cpu_clouds > 0 else None)
        arm.step(min(arm.n_clouds, 8))
        runs = [arm.step() for _ in range(2)]
        arm.close()
        rates = [p / dt for dt, p in runs]
        cpu = {'value': float(np.median(rates)), 'unit': 'points/s', 'cores': arm.cores, 'kind': 'port',
               'sample': f'{arm.n_clouds} of the {B} clouds of one step ({runs[0][1]} points) x 2 timed steps '
                         f'({runs[0][0]:.1f} s, {runs[1][0]:.1f} s), oracle port (C core + numpy/scipy/sklearn pre-pass'
                         f'{" + wet ground" if fused_wet else ""}), {arm.n_clouds} processes x {arm.threads} threads'}

    cfg = workload_config(args.config, args.gpus)
    line = {'metric': 'augmented LiDAR points/sec', 'value': value, 'unit': 'points/s', 'n_gpus': args.gpus,
            'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': ms_per_step, 'higher_is_better': True,
            'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic', 'config': cfg,
            'clouds_per_s': value / (64 * N_AZIMUTH), 'e2e': e2e, 'gpu_launches': int(launches), 'clocks': clk,
            'roofline': roofline, 'cpu_baseline': cpu,
            'timed_region_ms': total_ms,
            'theta_label_mismatch': theta_info, 'steps_in_flight': n_streams,
            'engine': {'prepass': 'device' if device_prepass else 'DEBUG: fixed host-supplied threshold polynomial',
                       'table_particles': tinfo['n_particles'], 'table_index_bytes': tinfo['bytes'],
                       'gather': None if gather is None else gather.kind,
                       'gather_multicast': None if gather is None else getattr(gather, 'multicast', False),
                       'gather_fallback': None if gather is None else getattr(gather, 'fallback_reason', None)}}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()

"""Throughput of the DROR de-snowing filter (csrc/dror.cu), with CUDA events over --steps steps; two input batches alternate
so that no step finds its rows in L2.  Two cases:
  * dror_batch alone on 32 synthetic 64 x 2048 clouds (alpha 0.16 and 0.45, k_min 3);
  * the chain snowfall -> DROR on bench.py's workload (32 clouds, 2.5 mm/h Gunn tables, device pre-pass), next to the
    snowfall step alone, with the mean removed fraction and the fraction of the snowfall's label-2 (snow) rows removed.
Prints one JSON object with the card's name and power limit."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True
import bench                                                                    # noqa: E402
from lidar_snow_sim_b200.engine import SnowfallEngine                            # noqa: E402
from lidar_snow_sim_b200.snowfall.sampling import sample_table_set               # noqa: E402


def card():
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
        name, pl = [s.strip() for s in q.split(',')]
        return {'name': name, 'power_limit': pl}
    except Exception as exc:                                                     # noqa: BLE001
        return {'name': torch.cuda.get_device_name(0), 'power_limit': f'unknown ({exc})'}


def timed(step, steps, warmup):
    for k in range(warmup):
        step(k)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for k in range(steps):
        step(k)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    args = ap.parse_args()
    eng = SnowfallEngine(0)
    B = bench.BATCH_PER_GPU
    clouds, orders = bench.make_workload(0, B)
    clouds2, orders2 = bench.make_workload(0, B, seed0=500000)
    off = np.concatenate([[0], np.cumsum([c.shape[0] for c in clouds])]).astype(np.int64)
    N = int(off[-1])
    pts = [torch.from_numpy(np.concatenate(c)).cuda() for c in (clouds, clouds2)]
    res = {'card': card(), 'workload': f'{B} synthetic 64x{bench.N_AZIMUTH} clouds ({N} points), two batches alternating',
           'steps': args.steps}

    alone = {}
    for alpha in (0.16, 0.45):
        outs = [{}, {}]

        def step(k):
            return eng.dror_batch(pts[k & 1], off, alpha=alpha, out=outs[k & 1])
        ms = timed(step, args.steps, args.warmup)
        r = step(0)
        removed = 1.0 - r['counts'].sum().item() / N
        alone[f'alpha={alpha}'] = {'ms_per_step': ms, 'points_per_s': N / (ms * 1e-3), 'removed_fraction': removed}
    res['dror_alone'] = alone

    tables = sample_table_set(bench.MODE, bench.SNOWFALL_RATE, bench.TERMINAL_VELOCITY, seed=bench.TABLE_SEED)
    tid = eng.upload_tables(tables)
    ords = [orders, orders2]
    snow_outs, dror_outs = [{}, {}], [{}, {}]

    def snow_step(k):
        return eng.snowfall_batch(tid, pts[k & 1], off, ords[k & 1], bench.DIV_DEG, device_prepass=True,
                                  out=snow_outs[k & 1])

    chain = {}
    snow_ms = timed(snow_step, args.steps, args.warmup)
    for alpha in (0.16, 0.45):
        def chain_step(k):
            s = snow_step(k)
            return eng.dror_batch(s['points'], off, counts=s['counts'], alpha=alpha, out=dror_outs[k & 1])
        ms = timed(chain_step, args.steps, args.warmup)
        s = snow_step(0)
        d = eng.dror_batch(s['points'], off, counts=s['counts'], alpha=alpha)
        eng.check()
        n_in = s['counts'].sum().item()
        # label-2 (snow) rows in and removed: codes are per input row, labels in column 4 of the snowfall output
        rows = torch.cat([torch.arange(int(off[b]), int(off[b]) + int(c), device=s['points'].device)
                          for b, c in enumerate(s['counts'].tolist())])
        label = s['points'][rows, 4]
        code = d['codes'][rows]
        n_label2 = int((label == 2).sum())
        removed_label2 = int(((label == 2) & (code == 0)).sum())
        removed_other = int(((label != 2) & (code == 0)).sum())
        chain[f'alpha={alpha}'] = {
            'ms_per_step_chain': ms, 'dror_ms': ms - snow_ms, 'dror_over_snowfall': (ms - snow_ms) / snow_ms,
            'removed_fraction': 1.0 - d['counts'].sum().item() / n_in,
            'label2_rows': n_label2, 'label2_removed_fraction': removed_label2 / max(1, n_label2),
            'other_removed_fraction': removed_other / max(1, n_in - n_label2)}
    res['snowfall_ms_per_step'] = snow_ms
    res['chain'] = chain

    # kernel split of one DROR call (torch.profiler, a separate pass after the timed ones)
    from torch.profiler import ProfilerActivity, profile
    s = snow_step(0)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for k in range(5):
            eng.dror_batch(s['points'], off, counts=s['counts'], alpha=0.16, out=dror_outs[0])
        torch.cuda.synchronize()
    split = {}
    for ev in prof.key_averages():
        if ev.device_type.name == 'CUDA' and getattr(ev, 'device_time_total', 0) > 0:
            split[ev.key[:80]] = round(ev.device_time_total / 5 / 1000.0, 4)
    res['kernel_ms_per_call_alpha_0.16'] = dict(sorted(split.items(), key=lambda kv: -kv[1])[:12])
    print(json.dumps(res))


if __name__ == '__main__':
    main()

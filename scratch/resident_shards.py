"""Resident shard directories against reloading shards from files (loader.ResidentShards vs ShardCycler + load_gc_dataset).

    python scratch/resident_shards.py OUT_DIR [--shards 8] [--rows 1250000]

Writes compressed shards of the C5 shape (cube-quadruple-play-100M: 55 float32 observations, 5 float32 actions, 1001-row
trajectories) to a temporary directory and reports, with the card's name and power limit read in the same run:
- the time to make every shard resident and the peak host RSS of the process;
- ShardCycler's time per swap over views (sampler created per swap, or memoised) and over file-loading samplers, and
  `prefetched_swaps` at intervals of 100 and 1,000 C5 steps (a C5 step = one sample(4096));
- the time of a synchronised sample_many call on a view and on a standalone dataset of the same shard;
- the same at the C1 shape (2 float32 observations), where every view but the last loses the shadow next observation.
"""

import argparse
import json
import multiprocessing
import os
import resource
import subprocess
import sys
import tempfile
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from ogbench_b200 import Dataset, GCDataset, loader  # noqa: E402
from ogbench_b200.synthetic import WORKLOADS  # noqa: E402


def card():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else 'unknown'


def write_shards(d, n_shards, rows, ob_dim, seed=0):
    rng = np.random.default_rng(seed)
    paths = []
    for i in range(n_shards):
        terminals = np.zeros(rows, np.float32)
        terminals[1000::1001] = 1.0
        terminals[-1] = 1.0
        obs = rng.standard_normal((rows, ob_dim), dtype=np.float32)
        act = rng.uniform(-1, 1, (rows, 5)).astype(np.float32)
        p = os.path.join(d, f'shard{i:02d}.npz')
        np.savez_compressed(p, observations=obs, actions=act, terminals=terminals)
        paths.append(p)
    return paths


def device_ms(sampler, n_batches, batch, reps=20):
    """Median time of a synchronised sample_many call (host clock around the launch and the wait for its batch)."""
    next(iter(sampler.sample_many(n_batches, batch).values()))._batch.sync()
    times = []
    for _ in range(reps):
        t0 = time.perf_counter()
        out = sampler.sample_many(n_batches, batch)
        next(iter(out.values()))._batch.sync()
        times.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(times))


def cycle(paths, make, interval, steps, batch):
    c = loader.ShardCycler(paths, make, interval)
    swap_ms = []
    for step in range(1, steps + 1):
        t0 = time.perf_counter()
        s = c.at_step(step)
        if step % interval == 0:
            swap_ms.append((time.perf_counter() - t0) * 1e3)
        out = s.sample(batch)
        next(iter(out.values()))._batch.sync()
    c.close()
    return dict(swaps=c.swaps, prefetched_swaps=c.prefetched_swaps, swap_ms_median=float(np.median(swap_ms)),
                swap_ms_max=float(np.max(swap_ms)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('out')
    ap.add_argument('--shards', type=int, default=8)
    ap.add_argument('--rows', type=int, default=1_250_000)
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)
    w = WORKLOADS['c5']
    config = dict(w.config)
    res = dict(card=card(), shards=args.shards, rows_per_shard=args.rows)
    with tempfile.TemporaryDirectory() as d:
        # the shards are written by a child process, so that this process's peak RSS is the build's
        with multiprocessing.get_context('spawn').Pool(1) as pool:
            paths = pool.apply(write_shards, (d, args.shards, args.rows, 55))
        res['shard_host_mb'] = args.rows * (55 + 5 + 1 + 1) * 4 / 2**20      # compact layout: + valids
        rss0 = resource.getrusage(resource.RUSAGE_SELF).ru_maxrss
        t0 = time.perf_counter()
        shards = loader.ResidentShards(paths)
        res['resident_build_s'] = time.perf_counter() - t0
        res['peak_rss_mb_before_build'] = rss0 / 1024
        res['peak_rss_mb_after_build'] = resource.getrusage(resource.RUSAGE_SELF).ru_maxrss / 1024
        res['resident_bytes'] = shards.dataset.native(0).resident_bytes()

        memo = {}

        def memoised(p):
            if p not in memo:
                memo[p] = GCDataset(shards[p], config, seed=1)
            return memo[p]

        sub = paths[:3]
        for interval in (100, 1000):
            steps = interval * 4
            res[f'views_new_sampler_i{interval}'] = cycle(sub, lambda p: GCDataset(shards[p], config, seed=1), interval, steps, w.batch)
            res[f'views_memoised_i{interval}'] = cycle(sub, memoised, interval, steps, w.batch)
            res[f'files_i{interval}'] = cycle(sub, lambda p: loader.load_gc_dataset(p, config, seed=1), interval, steps, w.batch)

        view = GCDataset(shards[1], config, seed=2)
        alone = GCDataset(Dataset.create(**loader.load_dataset(paths[1], compact_dataset=True)), config, seed=2)
        res['c5_sample_many_ms'] = {}
        for name, s in (('view', view), ('standalone', alone), ('view', view), ('standalone', alone)):
            res['c5_sample_many_ms'].setdefault(name, []).append(device_ms(s, 32, w.batch))
        del view, alone, shards, memo

        c1 = WORKLOADS['c1']
        p1 = write_shards(d, 2, 1_001_000, 2, seed=1)
        shards1 = loader.ResidentShards(p1)
        view = GCDataset(shards1[0], dict(c1.config), seed=2)            # not the last view: no shadow
        alone = GCDataset(Dataset.create(**loader.load_dataset(p1[0], compact_dataset=True)), dict(c1.config), seed=2)
        res['c1_sample_many_ms'] = {}
        for name, s in (('view_no_shadow', view), ('standalone', alone), ('view_no_shadow', view), ('standalone', alone)):
            res['c1_sample_many_ms'].setdefault(name, []).append(device_ms(s, 32, c1.batch))
    print(json.dumps(res, indent=1))
    with open(os.path.join(args.out, 'resident_shards.json'), 'w') as f:
        json.dump(res, f, indent=1)


if __name__ == '__main__':
    main()

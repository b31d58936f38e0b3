"""Load time and peak host memory of relabelled datasets ('-oraclerep-' and 'singletask' names) on their way into HBM:
make_datasets + Dataset.create against upload_datasets.

    python scratch/stream_relabel.py OUT_DIR [--frames 250250] [--c5-rows 2502500] [--reps 3]

Writes the two files of scratch/stream_load.py (the visual-cube shape and the C5 shape, deflated as np.savez_compressed
writes them) with float64 qpos[:, 40] and int64 button_states[:, 9] added, each with a small validation file, to a
temporary directory, under the stems of a scene dataset ('visual-scene-play-v0', 'scene-play-v0'): the scene
relabellings read both qpos and button_states.  Then, for `--reps` rounds, loads each file under an oraclerep name and a
singletask name once per mode, alternating the modes, each in a fresh child process:
- `host`: Dataset.create(**split).native(0) for both splits of make_datasets(name, compact_dataset=True, ...);
- `stream`: loader.upload_datasets(name, compact_dataset=True, ...);
- `read`: upload_datasets' host side alone (inflate, cast, layout and relabelling on the same threads, no device write).
A child reports the wall time of the load, the growth of its peak RSS (`ru_maxrss`) over the load and the `tracemalloc`
peak, as scratch/stream_load.py does.  The card's name and power limit are read in the same run.
"""

import argparse
import json
import os
import resource
import subprocess
import sys
import tempfile
import time
import tracemalloc
import types
from concurrent.futures import ProcessPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from ogbench_b200 import Dataset, loader  # noqa: E402
from stream_load import card, write_file  # noqa: E402

NAMES = {  # file -> (file stem, {label: dataset name})
    'pixels': ('visual-scene-play-v0', {'oraclerep': 'visual-scene-play-oraclerep-v0',
                                        'singletask': 'visual-scene-play-singletask-task1-v0'}),
    'c5': ('scene-play-v0', {'oraclerep': 'scene-play-oraclerep-v0', 'singletask': 'scene-play-singletask-task1-v0'}),
}


def task_env():
    """What relabel_dataset reads from a single-task scene environment (one cube, nine buttons), as a plain namespace."""
    task = types.SimpleNamespace(_reward_task_id=1, _num_cubes=1, _num_buttons=9,
                                 _data=types.SimpleNamespace(mocap_pos=np.array([[0.425, 0.0, 0.02]])),
                                 _target_button_states=np.zeros(9, np.int64), _target_drawer_pos=0.0, _target_window_pos=0.0)
    return types.SimpleNamespace(unwrapped=task, reset=lambda: None)


def relabel_kwargs(name):
    return dict(env=task_env()) if 'singletask' in name else dict(num_cubes=1, num_buttons=9)


def child(mode, directory, name):
    from ogbench_b200 import _native

    _native.lib()
    warm = Dataset.create(observations=np.zeros((4, 2), np.float32), terminals=np.ones(4, np.float32))
    warm.native(0)
    del warm
    kw = dict(dataset_dir=directory, compact_dataset=True, **relabel_kwargs(name))
    rss0 = resource.getrusage(resource.RUSAGE_SELF).ru_maxrss
    tracemalloc.start()
    t0 = time.perf_counter()
    if mode == 'host':
        splits = [Dataset.create(**ds) for ds in loader.make_datasets(name, **kw)]
        for ds in splits:
            ds.native(0)
    elif mode == 'stream':
        splits = loader.upload_datasets(name, **kw)
    else:
        for stream in loader._split_streams(name, directory, None, True, False, kw.get('env'), kw.get('num_cubes'),
                                            kw.get('num_buttons')):
            loader._pump(stream.producers(), lambda r0, arrays: None)
        splits = None
    wall = time.perf_counter() - t0
    _, peak = tracemalloc.get_traced_memory()
    tracemalloc.stop()
    rss1 = resource.getrusage(resource.RUSAGE_SELF).ru_maxrss
    print(json.dumps(dict(mode=mode, wall_s=wall, rss_growth_mb=(rss1 - rss0) / 1024, tracemalloc_peak_mb=peak / 2**20,
                          size=None if splits is None else splits[0].size,
                          fields=None if splits is None else list(splits[0]))))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('out', nargs='?')
    ap.add_argument('--frames', type=int, default=250_250)
    ap.add_argument('--c5-rows', type=int, default=2_502_500)
    ap.add_argument('--reps', type=int, default=3)
    ap.add_argument('--child', nargs=3, metavar=('MODE', 'DIR', 'NAME'))
    args = ap.parse_args()
    if args.child:
        child(*args.child)
        return
    os.makedirs(args.out, exist_ok=True)
    res = dict(card=card(), cpus=os.cpu_count(), files={}, runs={})
    with tempfile.TemporaryDirectory() as d:
        t0 = time.perf_counter()
        rows = {'pixels': args.frames, 'c5': args.c5_rows}
        with ProcessPoolExecutor(2 * len(NAMES)) as pool:
            futs = {}
            for f, (stem, _) in NAMES.items():
                futs[f] = pool.submit(write_file, os.path.join(d, f'{stem}.npz'), f, rows[f], info=True)
                futs[f, 'val'] = pool.submit(write_file, os.path.join(d, f'{stem}-val.npz'), f, 2002, seed=1, info=True)
            res['files'] = {f: futs[f].result() for f in NAMES}
            for f in NAMES:
                futs[f, 'val'].result()
        res['write_s'] = time.perf_counter() - t0
        print(json.dumps(res['files']), flush=True)
        for f, (_, names) in NAMES.items():
            for label, name in names.items():
                runs = res['runs'][f'{f} {label}'] = {'host': [], 'stream': [], 'read': []}
                for rep in range(args.reps):
                    for mode in ('host', 'stream', 'read'):
                        p = subprocess.run([sys.executable, os.path.abspath(__file__), '--child', mode, d, name],
                                           capture_output=True, text=True, timeout=3600)
                        if p.returncode != 0:
                            raise RuntimeError(f'{name} {mode}: {p.stderr[-3000:]}')
                        r = json.loads(p.stdout.strip().splitlines()[-1])
                        runs[mode].append(r)
                        print(f, label, rep, json.dumps(r), flush=True)
    res['summary'] = {key: {mode: {k: [round(r[k], 3) for r in rs] for k in ('wall_s', 'rss_growth_mb', 'tracemalloc_peak_mb')}
                            for mode, rs in runs.items()} for key, runs in res['runs'].items()}
    print(json.dumps(res['summary'], indent=1))
    with open(os.path.join(args.out, 'stream_relabel.json'), 'w') as f:
        json.dump(res, f, indent=1)


if __name__ == '__main__':
    main()

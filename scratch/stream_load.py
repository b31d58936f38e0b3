"""Load time and peak host memory of an `.npz` file on its way into HBM: the host path against the streaming path.

    python scratch/stream_load.py OUT_DIR [--frames 250250] [--c5-rows 2502500] [--reps 3]

Writes two deflated .npz files, as np.savez_compressed writes them but a chunk at a time, to a temporary directory:
- pixels: the visual-cube shape (64x64x3 uint8 frames, 5 float32 actions, 1001-row trajectories): a fixed gradient
  background, two moving rectangles and noise on a sparse pixel grid, so that the frames deflate to a fraction of their
  size as rendered frames do;
- c5: the C5 row shape (55 float32 observations, 5 float32 actions, 1001-row trajectories), normal random values, which
  barely deflate.
Then, for `--reps` rounds, loads each file once per mode, alternating the modes, each in a fresh child process:
- `host`: Dataset.create(**load_dataset(path, ob_dtype, compact_dataset=True)), uploaded (ds.native(0));
- `stream`: loader.upload_dataset(path, ob_dtype, compact_dataset=True);
- `read`: the streaming path's host side alone (inflate, cast and layout on the same threads, no device write), which
  shows how much of `stream` the device writes add.
A child reports the wall time of the load (it ends in the device synchronise of the table build), the growth of its peak
RSS (`ru_maxrss`) over the load and the `tracemalloc` peak.  CUDA is initialised and the library loaded before the clock
starts.  The card's name and power limit are read in the same run.
"""

import argparse
import io
import json
import os
import resource
import subprocess
import sys
import tempfile
import time
import tracemalloc
import zipfile
from concurrent.futures import ProcessPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from ogbench_b200 import Dataset, loader  # noqa: E402


def card():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else 'unknown'


def write_member(zf, name, shape, dtype, chunks):
    """One .npy member as np.savez_compressed writes it (ZIP64, deflated), fed chunk by chunk."""
    buf = io.BytesIO()
    np.lib.format.write_array_header_2_0(buf, dict(descr=np.lib.format.dtype_to_descr(np.dtype(dtype)), fortran_order=False,
                                                   shape=shape))
    with zf.open(f'{name}.npy', 'w', force_zip64=True) as f:
        f.write(buf.getvalue())
        for c in chunks:
            f.write(np.ascontiguousarray(c, dtype).tobytes())


def write_file(path, kind, rows, seed=0, info=False):
    """With `info`, also float64 qpos[:, 40] (normal random values) and int64 button_states[:, 9] (0 / 1), the members
    the '-oraclerep-' and 'singletask' relabellings read."""
    rng = np.random.default_rng(seed)
    chunk = 4096
    terminals = np.zeros(rows, bool)
    terminals[1000::1001] = True
    terminals[-1] = True
    if kind == 'pixels':
        yy, xx = np.mgrid[0:64, 0:64]
        base = np.stack([yy * 3, xx * 3, (yy + xx) * 2], -1).astype(np.uint8)

        def frames():
            for r0 in range(0, rows, chunk):
                t = np.arange(r0, min(rows, r0 + chunk))
                f = np.broadcast_to(base, (len(t), 64, 64, 3)).copy()
                for k, (size, colour) in enumerate(((12, (200, 40, 40)), (9, (40, 40, 220)))):
                    ys, xs = (t * (k + 1)) % (64 - size), (t * (3 - k) // 2) % (64 - size)
                    for i in range(len(t)):
                        f[i, ys[i]:ys[i] + size, xs[i]:xs[i] + size] = colour
                f[:, ::7, ::5] = rng.integers(0, 256, f[:, ::7, ::5].shape, dtype=np.uint8)
                yield f

        obs_shape, obs_dtype, obs_chunks = (rows, 64, 64, 3), np.uint8, frames()
    else:
        obs_shape, obs_dtype = (rows, 55), np.float32
        obs_chunks = (rng.standard_normal((min(chunk, rows - r0), 55), dtype=np.float32) for r0 in range(0, rows, chunk))
    with zipfile.ZipFile(path, 'w', compression=zipfile.ZIP_DEFLATED, allowZip64=True) as zf:
        write_member(zf, 'observations', obs_shape, obs_dtype, obs_chunks)
        write_member(zf, 'actions', (rows, 5), np.float32,
                     (rng.uniform(-1, 1, (min(chunk, rows - r0), 5)) for r0 in range(0, rows, chunk)))
        write_member(zf, 'terminals', (rows,), bool, [terminals])
        if info:
            write_member(zf, 'qpos', (rows, 40), np.float64,
                         (rng.standard_normal((min(chunk, rows - r0), 40)) for r0 in range(0, rows, chunk)))
            write_member(zf, 'button_states', (rows, 9), np.int64,
                         (rng.integers(0, 2, (min(chunk, rows - r0), 9)) for r0 in range(0, rows, chunk)))
    return dict(path=path, rows=rows, file_bytes=os.path.getsize(path),
                raw_bytes=rows * (int(np.prod(obs_shape[1:])) * np.dtype(obs_dtype).itemsize + 20 + 1 + 392 * info))


def child(mode, path, ob_dtype):
    """One load in this process: a JSON line with its wall time and host memory."""
    from ogbench_b200 import _native

    _native.lib()
    warm = Dataset.create(observations=np.zeros((4, 2), np.float32), terminals=np.ones(4, np.float32))
    warm.native(0)
    del warm
    rss0 = resource.getrusage(resource.RUSAGE_SELF).ru_maxrss
    tracemalloc.start()
    t0 = time.perf_counter()
    if mode == 'host':
        ds = Dataset.create(**loader.load_dataset(path, ob_dtype=ob_dtype, compact_dataset=True))
        ds.native(0)
    elif mode == 'stream':
        ds = loader.upload_dataset(path, ob_dtype=ob_dtype, compact_dataset=True)
    else:
        stream = loader._FileStream(path, ob_dtype=ob_dtype, compact_dataset=True)
        loader._pump(stream.producers(), lambda r0, arrays: None)
        ds = None
    wall = time.perf_counter() - t0
    _, peak = tracemalloc.get_traced_memory()
    tracemalloc.stop()
    rss1 = resource.getrusage(resource.RUSAGE_SELF).ru_maxrss
    print(json.dumps(dict(mode=mode, wall_s=wall, rss_growth_mb=(rss1 - rss0) / 1024, tracemalloc_peak_mb=peak / 2**20,
                          size=None if ds is None else ds.size)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('out', nargs='?')
    ap.add_argument('--frames', type=int, default=250_250)
    ap.add_argument('--c5-rows', type=int, default=2_502_500)
    ap.add_argument('--reps', type=int, default=3)
    ap.add_argument('--child', nargs=3, metavar=('MODE', 'PATH', 'OB_DTYPE'))
    args = ap.parse_args()
    if args.child:
        child(args.child[0], args.child[1], np.dtype(args.child[2]))
        return
    os.makedirs(args.out, exist_ok=True)
    res = dict(card=card(), cpus=os.cpu_count(), files={}, runs={})
    with tempfile.TemporaryDirectory() as d:
        t0 = time.perf_counter()
        specs = {'pixels': ('pixels', args.frames, 'uint8'), 'c5': ('c5', args.c5_rows, 'float32')}
        with ProcessPoolExecutor(len(specs)) as pool:
            futs = {name: pool.submit(write_file, os.path.join(d, f'{name}.npz'), kind, rows) for name, (kind, rows, _) in specs.items()}
            res['files'] = {name: f.result() for name, f in futs.items()}
        res['write_s'] = time.perf_counter() - t0
        print(json.dumps(res['files']), flush=True)
        for name, (_, _, ob_dtype) in specs.items():
            runs = res['runs'][name] = {'host': [], 'stream': [], 'read': []}
            for rep in range(args.reps):
                for mode in ('host', 'stream', 'read'):
                    p = subprocess.run([sys.executable, os.path.abspath(__file__), '--child', mode, res['files'][name]['path'], ob_dtype],
                                       capture_output=True, text=True, timeout=3600)
                    if p.returncode != 0:
                        raise RuntimeError(f'{name} {mode}: {p.stderr[-3000:]}')
                    r = json.loads(p.stdout.strip().splitlines()[-1])
                    runs[mode].append(r)
                    print(name, rep, json.dumps(r), flush=True)
    res['summary'] = {name: {mode: {k: [round(r[k], 3) for r in rs] for k in ('wall_s', 'rss_growth_mb', 'tracemalloc_peak_mb')}
                             for mode, rs in runs.items()} for name, runs in res['runs'].items()}
    print(json.dumps(res['summary'], indent=1))
    with open(os.path.join(args.out, 'stream_load.json'), 'w') as f:
        json.dump(res, f, indent=1)


if __name__ == '__main__':
    main()

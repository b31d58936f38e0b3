"""ReplayBuffer write rates: add_transitions(n) from numpy and from torch CUDA against the add_transition loop and the
reference's numpy ring buffer.

    python scratch/replay_writes.py [OUT_DIR]

Transitions hold observations (C2: 29 float32; C4: 64x64x3 uint8), actions (C2: 8, C4: 5 float32), rewards, terminals and
masks (float32).  For n in {1, 64, 1024, 16384, 262144} it reports µs per call and transitions/s, each timed with a host
clock around a run of calls that ends in a device synchronise, after one warm-up call; the GB/s columns count the
transition bytes once (host sources: bytes over PCIe; device sources: bytes read, the same again is written).  The card's
name and power limit are read in the same run.  Prints one JSON line per measurement (and writes them to
OUT_DIR/replay_writes.jsonl when OUT_DIR is given).
"""

import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from ogbench_b200 import ReplayBuffer, _native  # noqa: E402
from oracle.replay_oracle import OracleReplayBuffer  # noqa: E402

SHAPES = {'c2': ((29,), np.float32, 8, 1 << 20), 'c4': ((64, 64, 3), np.uint8, 5, 1 << 18)}
SIZES = [1, 64, 1024, 16384, 262144]


def card():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else 'unknown'


def transitions(shape, n, rng):
    obs_shape, obs_dtype, act_dim, _ = shape
    if obs_dtype == np.uint8:
        obs = rng.integers(0, 256, (n, *obs_shape), dtype=np.uint8)
    else:
        obs = rng.standard_normal((n, *obs_shape), dtype=np.float32)
    return dict(observations=obs, actions=rng.uniform(-1, 1, (n, act_dim)).astype(np.float32),
                rewards=rng.standard_normal(n, dtype=np.float32), terminals=np.zeros(n, np.float32), masks=np.ones(n, np.float32))


def timed(fn, budget_s=0.5, max_calls=2000):
    """µs per call over a run of calls that fills about budget_s, ending in a device synchronise."""
    import torch

    fn()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    one = time.perf_counter() - t0
    calls = int(max(3, min(max_calls, budget_s / max(one, 1e-7))))
    t0 = time.perf_counter()
    for _ in range(calls):
        fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) / calls * 1e6, calls


def main():
    import torch

    out_dir = sys.argv[1] if len(sys.argv) > 1 else None
    rows = []

    def emit(**kw):
        kw['card'] = the_card
        print(json.dumps(kw), flush=True)
        rows.append(kw)

    the_card = card()
    rng = np.random.default_rng(0)
    for name, shape in SHAPES.items():
        capacity = shape[3]
        example = {k: v[0] for k, v in transitions(shape, 1, rng).items()}
        rb = ReplayBuffer.create(example, size=capacity)
        host = transitions(shape, max(SIZES), rng)
        dev = {k: torch.from_numpy(v).cuda() for k, v in host.items()}
        row_bytes = sum(v[0].nbytes for v in host.values())
        for n in SIZES:
            for source, batch in (('numpy', {k: v[:n] for k, v in host.items()}), ('torch', {k: v[:n] for k, v in dev.items()})):
                us, calls = timed(lambda: rb.add_transitions(batch))
                emit(shape=name, call='add_transitions', source=source, n=n, calls=calls, us_per_call=round(us, 2),
                     transitions_per_s=round(n / us * 1e6), gb_per_s=round(n * row_bytes / us / 1e3, 2), row_bytes=row_bytes)
        single = {k: v[0] for k, v in host.items()}
        us, calls = timed(lambda: rb.add_transition(single))
        emit(shape=name, call='add_transition', source='numpy', n=1, calls=calls, us_per_call=round(us, 2),
             transitions_per_s=round(1e6 / us), row_bytes=row_bytes)
        single_dev = {k: v[0] for k, v in dev.items()}
        us, calls = timed(lambda: rb.add_transition(single_dev))
        emit(shape=name, call='add_transition', source='torch', n=1, calls=calls, us_per_call=round(us, 2),
             transitions_per_s=round(1e6 / us), row_bytes=row_bytes)
        oracle = OracleReplayBuffer(example, capacity)
        t0 = time.perf_counter()
        k = 20000 if name == 'c2' else 5000
        for i in range(k):
            oracle.add_transition({key: v[i] for key, v in host.items()})
        us = (time.perf_counter() - t0) / k * 1e6
        emit(shape=name, call='reference numpy add_transition', source='numpy', n=1, calls=k, us_per_call=round(us, 2),
             transitions_per_s=round(1e6 / us), row_bytes=row_bytes)
        # what one device leaf costs before the write: the DLPack export with the sampler's stream as consumer
        handle = C.c_void_p()
        _native.check(_native.lib().ogb_sampler_get_stream(rb._plain_sampler(0).ptr, C.byref(handle)))
        leaf = dev['actions'][:64]
        us, calls = timed(lambda: leaf.__dlpack__(stream=handle.value))
        emit(shape=name, call='torch __dlpack__(stream=sampler stream), one leaf', source='torch', n=64, calls=calls,
             us_per_call=round(us, 2))
        del rb, dev, oracle
        torch.cuda.empty_cache()
    if out_dir:
        os.makedirs(out_dir, exist_ok=True)
        with open(os.path.join(out_dir, 'replay_writes.jsonl'), 'w') as f:
            for r in rows:
                f.write(json.dumps(r) + '\n')


if __name__ == '__main__':
    main()

#!/usr/bin/env python
"""bench.py -- relabelled transitions/s of the replay sampler hot path on B200 (BASELINE.json's metric).

    python bench.py --gpus N --steps K --warmup W [--config c2] [--batches-per-launch L]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...      # the CPU implementation of the same path on the host cores
    python bench.py ... --dump-outputs DIR    # also write a sample of what the last timed step returned

A "step" is one launch of the hot path producing `batches_per_launch` successive GCDataset.sample(batch) calls
(config.batches_per_launch; 1 reproduces the reference's one-call-per-step usage and is launch-latency bound), made
through the public call `GCDataset.sample_many(L, B)`.  Every timed loop runs exactly K steps back to back inside one
timed region (`timed_region_ms`, `steps_timed`); `ms_per_step` is the region divided by K.  A launch lasts about a
millisecond, so a region that should not be dominated by clock and scheduler noise wants K of a few hundred.

The headline (top-level keys) is C2 = BASELINE.json configs[1]; the same line carries every config of BASELINE.json
under `configs` (c1..c5, each with value / roofline / e2e / cpu_baseline), C5 as one trajectory-aligned shard per GPU.
`value` = transitions all ranks produced / max-over-ranks device time with the dataset resident in HBM;
`e2e` = the same through the public Python API with host buffers (transition indices uploaded from pinned host
memory every step, the whole batch copied back into pinned host memory, both inside the timed region), next to the
raw pinned D2H copy rate of the same box measured in the same run (`link_gbs`);
`roofline` = algorithmic bytes (SURVEY.md 8(d)) / average launch duration of the dominant kernel vs the measured
HBM copy bandwidth (and vs the 8 TB/s data-sheet figure, `frac_of_nominal`); `cpu_baseline` = the numpy oracle port
timed on this box's host cores in the same run.  A launch costs 8-19 us beyond its bytes, so the default launch is sized
to last about a millisecond (`default_batches_per_launch`) and every config also carries `launch_size_sweep`: the same
measurement at a quarter and a sixteenth of that size.  `e2e.value` and `e2e.link_gbs` are each the faster of two passes
(`e2e.passes`): the hosts of this pool are shared and their PCIe rate dips for seconds at a time.

`--dump-outputs DIR` writes, after the headline timed loop of every config, what the last timed step returned: for each
key of the batch, the same fixed, seeded sample of its L * B transitions as `DIR/<config>.<key>.npy` (float32, or float64
for keys whose values float32 cannot hold exactly), at most `DUMP_BYTES` in all.  The dataset, the sampler seed and the
number of launches before that step depend only on the arguments, so two builds run with the same arguments can be
compared file by file.
"""

from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = 'relabeled transitions/sec'
UNIT = 'transitions/s'
FALLBACK_HBM_GBS = 6650.0  # /opt/skills/guides/B200_PROFILING.md, used only when MEASURED_PEAKS.json is absent
NOMINAL_HBM_GBS = 8000.0   # B200 data sheet (SURVEY.md 8(d): quoted next to the measured copy peak)
HEADLINE = 'c2'
ALL_CONFIGS = ['c1', 'c2', 'c3', 'c4', 'c5']
DUMP_BYTES = 60_000_000     # --dump-outputs: array bytes written in all (npy headers stay within 64 MB), shared by ALL_CONFIGS
DUMP_SEED = 0


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=100)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', choices=['ours', 'reference'], default='ours')
    ap.add_argument('--config', default=None,
                    help='one workload key (c1..c5, c3b/c4b/c5b), SURVEY.md 8(d); default: the c2 headline plus c1..c5 under "configs"')
    ap.add_argument('--batches-per-launch', type=int, default=None)
    ap.add_argument('--e2e-batches', type=int, default=None, help='batches per e2e step')
    ap.add_argument('--cpu-seconds', type=float, default=10.0, help='budget of the headline cpu_baseline leg')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-e2e', action='store_true')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='write a fixed, seeded sample of the last timed step of every config as DIR/<config>.<key>.npy')
    return ap.parse_args()


def hbm_peak():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(path):
        try:
            return float(json.load(open(path))['hbm_gbs']), 'measured (MEASURED_PEAKS.json)'
        except Exception:
            pass
    return FALLBACK_HBM_GBS, 'fallback (B200_PROFILING.md)'


def default_batches_per_launch(w):
    # A launch costs 8-19 us beyond its bytes (ramp-up and tail: profiles/r2_ab_shapes.txt, batch r2i), so a launch is sized
    # to last ~1 ms: ~4M transitions for vector workloads (16M for rows of a few bytes, halved while one launch would move more
    # than 9 GB), 64 batches for the pixel workload.  The line also reports the round-1 size (a quarter / a sixteenth of this)
    # under `launch_size_sweep`.
    if w.obs_dtype == 'uint8':
        return 64
    transitions = (16 << 20) if w.bytes_per_transition < 256 else (4 << 20)
    while transitions * w.bytes_per_transition > 9e9:
        transitions //= 2
    return max(1, transitions // w.batch)


def config_dict(key, L):
    """The workload description both arms print (a pure function of the workload key and batches_per_launch)."""
    from ogbench_b200 import synthetic

    w = synthetic.WORKLOADS[key]
    return {
        'workload': w.name, 'key': w.key, 'rows_resident_per_gpu': w.rows, 'batch': w.batch, 'batches_per_launch': L,
        'transitions_per_step_per_gpu': w.batch * L,
        'placement': 'trajectory-aligned shard per GPU' if key.startswith('c5') else 'replica per GPU',
        'l2': 'no explicit flush: outputs rotate through three blocks of one launch each (every block is 1-4 GB, many times the '
              '126 MB L2), inputs are random rows of the resident dataset (per-config sizes in notes; the c1 dataset (32 MB) fits L2 '
              'and c2 (256 MB) partly, as the real datasets of these shapes do)',
    }


# ------------------------------------------------------------------------------------------------------------------
# CPU arm: the oracle port (oracle/replay_oracle.py == the reference's numpy algorithm), timed on the host cores
# ------------------------------------------------------------------------------------------------------------------
def _cpu_fields(w):
    from ogbench_b200 import synthetic

    # the pixel workload's 12.3 GB dataset is not regenerated on the host: 100 episodes keep the per-call work
    # identical (same rows/frames per sample) while fitting in RAM
    episodes = min(w.episodes, 100) if w.obs_dtype == 'uint8' else w.episodes
    return synthetic.host_fields(w, episodes=episodes), episodes


def _cpu_worker(args):
    """One host process: W warm-up steps, then K timed steps of `calls` sample(batch) calls each."""
    key, steps, warmup, budget_s, seed = args
    os.environ.setdefault('OMP_NUM_THREADS', '1')
    from ogbench_b200 import synthetic
    from oracle.replay_oracle import OracleSampler

    w = synthetic.WORKLOADS[key]
    fields, _ = _cpu_fields(w)
    sampler = OracleSampler(fields, w.config, w.kind)
    np.random.seed(seed)
    for _ in range(2):
        sampler.sample(w.batch)
    t0 = time.perf_counter()
    n_cal = 0
    while time.perf_counter() - t0 < 0.2 or n_cal < 2:     # calibrate: calls per step so that the run fits the budget
        sampler.sample(w.batch)
        n_cal += 1
    t_call = (time.perf_counter() - t0) / n_cal
    calls = max(1, int(budget_s / ((steps + warmup) * t_call)))
    for _ in range(warmup * calls):
        sampler.sample(w.batch)
    t0 = time.perf_counter()
    for _ in range(steps * calls):
        sampler.sample(w.batch)
    return steps * calls, time.perf_counter() - t0, calls


def cpu_baseline(key, workers, steps, warmup, budget_s):
    """transitions/s of the oracle port with `workers` independent processes (1 = the reference's own threading)."""
    from ogbench_b200 import synthetic

    w = synthetic.WORKLOADS[key]
    jobs = [(key, steps, warmup, budget_s, i) for i in range(workers)]
    if workers == 1:
        results = [_cpu_worker(jobs[0])]
    else:
        import multiprocessing as mp

        with mp.get_context('spawn').Pool(workers) as pool:
            results = pool.map(_cpu_worker, jobs)
    rate = sum(n * w.batch / dt for n, dt, _ in results)
    calls = sum(n for n, _, _ in results)
    _, episodes = _cpu_fields(w)
    slowest = max(dt for _, dt, _ in results)
    sample = (f'{steps} steps of {results[0][2]} sample({w.batch}) calls per process = {calls} calls over {slowest:.1f} s on '
              f'{workers} process(es), numpy {np.__version__}, dataset {episodes}x{w.steps} rows')
    return rate, sample, 1e3 * slowest / steps


def run_reference_arm(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    from ogbench_b200 import synthetic

    key = args.config or HEADLINE
    w = synthetic.WORKLOADS[key]
    L = args.batches_per_launch or default_batches_per_launch(w)
    workers = os.cpu_count() or 1
    steps, warmup = max(1, args.steps), max(0, args.warmup)
    t0 = time.perf_counter()
    rate, sample, ms_per_step = cpu_baseline(key, workers, steps, warmup, budget_s=30.0)
    wall = time.perf_counter() - t0
    line = {
        'impl': 'reference', 'metric': METRIC, 'value': rate, 'unit': UNIT, 'n_gpus': args.gpus, 'steps': steps,
        'warmup': warmup, 'ms_per_step': ms_per_step, 'higher_is_better': True, 'scaling': 'weak',
        'vs_baseline': None, 'dtype': 'u8' if w.obs_dtype == 'uint8' else 'f32', 'data': 'synthetic',
        'config': config_dict(key, L),
        'notes': 'reference numpy algorithm (oracle port; the reference itself is Python+JAX and is not installed on the GPU '
                 'box), one process per host core, each step a bounded number of sample(batch) calls per process',
        'cpu_baseline': {'value': rate, 'unit': UNIT, 'cores': workers, 'kind': 'port', 'sample': sample},
        'e2e': {'value': rate, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0, 'wall_s': wall,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons with NVML while the timed region runs."""

    def __init__(self, device_index, period=0.002):
        super().__init__(daemon=True)
        self.period = period
        self.samples = []
        self.reasons = set()
        self.stop_flag = threading.Event()
        self.ok = False
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            visible = os.environ.get('CUDA_VISIBLE_DEVICES')
            phys = int(visible.split(',')[device_index]) if visible and visible.split(',')[device_index].isdigit() else device_index
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.max_mhz = None

    def poll(self):
        nv = self.nv
        self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
        mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h) if hasattr(nv, 'nvmlDeviceGetCurrentClocksEventReasons') \
            else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
        names = {
            'hw_slowdown': 0x8, 'sw_power_cap': 0x4, 'hw_thermal_slowdown': 0x40, 'sw_thermal_slowdown': 0x20,
            'hw_power_brake_slowdown': 0x80, 'sync_boost': 0x10, 'applications_clocks_setting': 0x2,
        }
        for name, bit in names.items():
            if mask & bit:
                self.reasons.add(name)

    def run(self):
        if not self.ok:
            return
        while not self.stop_flag.is_set():
            try:
                self.poll()
            except Exception:
                break
            time.sleep(self.period)

    def summary(self):
        if not self.ok:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvml unavailable']}
        if not self.samples:
            try:
                self.poll()
            except Exception:
                pass
        med = float(np.median(self.samples)) if self.samples else None
        return {'sm_mhz': med, 'sm_max_mhz': float(self.max_mhz), 'reasons': sorted(self.reasons), 'samples': len(self.samples)}


# ------------------------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------------------------
def committed_traffic(key, kernel_name, kernel_ms, per_step):
    """DRAM bytes of one launch of the dominant kernel from the committed `ncu --set full` capture (profiles/traffic.json),
    scaled to this run's launch size.  Refused (None + reason) when the capture is of another kernel or when the kernel it
    recorded ran more than 10 % slower or faster than this run's -- ncu serialises launches on a cold cache, which moves a
    launch by a few percent; a bigger gap means the kernel has changed since the capture."""
    tpath = os.path.join(ROOT, 'profiles', 'traffic.json')
    if not os.path.exists(tpath):
        return None, 'profiles/traffic.json is absent'
    try:
        entry = json.load(open(tpath)).get(key)
        if not entry:
            return None, f'no capture for {key}'
        if entry.get('kernel', '').find(kernel_name) < 0:
            return None, f"capture is of {entry.get('kernel')!r}, the run's dominant kernel is {kernel_name!r}"
        scale = per_step / float(entry.get('transitions_per_launch', per_step))
        ncu_ms = float(entry['duration_us_under_ncu']) * 1e-3 * scale
        if abs(ncu_ms - kernel_ms) > 0.10 * kernel_ms:
            return None, f'stale capture: {ncu_ms:.4f} ms under ncu vs {kernel_ms:.4f} ms in this run'
        return float(entry['dram_bytes_per_launch']) * scale, f"{entry.get('source', 'ncu capture')}, {ncu_ms:.4f} ms under ncu"
    except Exception as exc:  # a malformed file must not take the bench down
        return None, f'unreadable: {exc}'


def link_probe(torch, device, nbytes, reps=8):
    """Raw pinned device->host copy rate of this rank's GPU for a block of the e2e step's size (GB/s)."""
    src = torch.empty(nbytes, dtype=torch.uint8, device=device)
    dst = torch.empty(nbytes, dtype=torch.uint8).pin_memory()
    for _ in range(2):
        dst.copy_(src, non_blocking=True)
    torch.cuda.synchronize(device)
    best = 0.0
    for _ in range(2):      # the faster of two passes, like the e2e leg it is compared with
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for _ in range(reps):
            dst.copy_(src, non_blocking=True)
        ev1.record()
        torch.cuda.synchronize(device)
        best = max(best, reps * nbytes / (ev0.elapsed_time(ev1) * 1e-3) / 1e9)
    return best


def dump_sample(tensors, key, out_dir):
    """Write one batch ({name: tensor [L, B, ...]}) as out_dir/<key>.<name>.npy: the same DUMP_SEED-chosen transitions of
    every name, as many as fit this config's share of DUMP_BYTES, in float32 where that holds every value exactly and in
    float64 otherwise."""
    import torch

    narrow = {torch.float32, torch.float16, torch.bfloat16, torch.bool, torch.uint8, torch.int8, torch.int16, torch.uint16}
    kinds = {name: torch.float32 if t.dtype in narrow else torch.float64 for name, t in tensors.items()}
    lead = {tuple(t.shape[:2]) for t in tensors.values()}
    assert len(lead) == 1, lead
    n = int(np.prod(lead.pop()))
    row_bytes = sum(int(np.prod(t.shape[2:])) * kinds[name].itemsize for name, t in tensors.items())
    count = max(1, min(n, DUMP_BYTES // len(ALL_CONFIGS) // row_bytes))
    rows = np.sort(np.random.default_rng(DUMP_SEED).choice(n, size=count, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    for name, t in tensors.items():
        idx = torch.from_numpy(rows).to(t.device)
        sample = t.reshape(n, *t.shape[2:]).index_select(0, idx).to(kinds[name]).cpu().numpy()
        np.save(os.path.join(out_dir, f'{key}.{name}.npy'), sample)


def measure_config(key, args, ctx, headline):
    """All measurements of one workload on this rank; collective calls inside (every rank runs the same sequence)."""
    import ctypes as C

    torch, dist_util, lib, _native = ctx['torch'], ctx['dist_util'], ctx['lib'], ctx['_native']
    from ogbench_b200 import Dataset, GCDataset, HGCDataset, synthetic

    rank, world, local = ctx['rank'], ctx['world'], ctx['local']
    dev = f'cuda:{local}'
    w = synthetic.WORKLOADS[key]
    L = args.batches_per_launch or default_batches_per_launch(w)

    # each rank holds a replica (c1-c4) or its own trajectory-aligned shard (c5), generated directly in HBM
    # OGB_BENCH_EPISODES=n (measurement switch, reported in `notes`): a dataset of n episodes of the same row shape, e.g. one
    # that fits L2, to tell what the DRAM side of the gathers costs
    episodes = int(os.environ.get('OGB_BENCH_EPISODES', '0')) or w.episodes
    fields = synthetic.device_fields(w, device=local, episodes=episodes, seed=w.seed + (rank if key.startswith('c5') else 0))
    dataset = Dataset.create(**fields)
    cls = GCDataset if w.kind == 'gc' else HGCDataset
    sampler = cls(dataset, w.config, device=local, seed=1234, stream_id=rank)
    del fields
    torch.cuda.empty_cache()
    stream = torch.cuda.Stream(device=local)
    sampler._sampler.set_stream(stream.cuda_stream)
    _native.check(lib.ogb_sampler_set_profile(sampler._sampler.ptr, 1))   # CUDA events around the dominant kernel of each launch

    def barrier():
        dist_util.barrier()
        torch.cuda.synchronize(local)

    keep_last = args.dump_outputs is not None     # the headline loop holds on to its newest batch for --dump-outputs
    last_batch = None

    def launch():
        nonlocal last_batch
        batch = sampler.sample_many(cur_L[0], w.batch)           # the public call: dict of DeviceArray, [L, B, ...] per key
        if keep_last:
            last_batch = batch
        handle = next(iter(batch.values()))._batch
        n = C.c_int32()
        lib.ogb_batch_launches(handle.ptr, C.byref(n))
        return handle, n.value

    cur_L = [L]
    launches = 0
    dominant_ms = []
    dominant_name = C.c_char_p()
    dominant_seen = ['']    # the name is owned by the batch: copied while the handle is alive

    def harvest(handle, keep):
        # device time of the launch's dominant kernel, from the events the library recorded on its own streams
        ms = C.c_float()
        _native.check(lib.ogb_batch_dominant_kernel(handle.ptr, C.byref(dominant_name), C.byref(ms)))
        dominant_seen[0] = (dominant_name.value or b'').decode()
        if keep and ms.value >= 0:
            dominant_ms.append(ms.value)

    def run(n_steps, keep):
        # Up to three batches are alive at any time (the consumer holds two while the next is produced); a handle is
        # harvested two launches after its own, when its kernels have long finished, and dropping it recycles its block.
        nonlocal launches
        pending = []
        for _ in range(n_steps):
            h, n = launch()
            launches += n if keep else 0
            pending.append(h)
            if len(pending) > 2:
                harvest(pending.pop(0), keep)
        return pending

    def timed(n_steps, keep):
        ev0 = torch.cuda.Event(enable_timing=True)
        ev1 = torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(stream):
            ev0.record(stream)
            tail = run(n_steps, keep)
            ev1.record(stream)
        barrier()
        for h in tail:
            harvest(h, keep)
        del tail
        return ev0.elapsed_time(ev1)

    warmup = max(args.warmup, 3)
    tail = run(warmup + 2, False)   # same hand-over pattern as the timed loop: every recycled block exists
    del tail
    barrier()
    n_steps = args.steps
    clocks = ClockSampler(local)
    clocks.start()
    elapsed_ms = timed(n_steps, True)
    clocks.stop_flag.set()
    clocks.join()
    if keep_last:
        if rank == 0:
            dump_sample({name: arr.torch() for name, arr in last_batch.items()}, key, args.dump_outputs)
        keep_last, last_batch = False, None
    kernel_ms = float(np.mean(dominant_ms)) if dominant_ms else elapsed_ms / n_steps
    kernel_name = dominant_seen[0]
    elapsed_ms = dist_util.reduce_scalar(elapsed_ms, 'max', device=dev)   # slowest rank
    per_step = w.batch * L
    value = dist_util.reduce_scalar(n_steps * per_step, 'sum', device=dev) / (elapsed_ms * 1e-3)
    resident = dataset.native(local).resident_bytes()

    # ---- the same launch at a quarter and a sixteenth of the size (c2: 1024 = the round-1 launch, 256) ----
    sweep = []
    if not os.environ.get('OGB_BENCH_NO_SWEEP'):
        n_launches, n_kernel_ms = launches, len(dominant_ms)
        for Ls in (max(1, L // 4), max(1, L // 16)):
            if Ls == L:
                continue
            cur_L[0] = Ls
            del run(5, False)[:]
            barrier()
            before = len(dominant_ms)
            ms = dist_util.reduce_scalar(timed(args.steps, True), 'max', device=dev) / args.steps
            k_ms = float(np.mean(dominant_ms[before:])) if len(dominant_ms) > before else ms
            bytes_launch = w.bytes_per_transition * w.batch * Ls
            sweep.append({'batches_per_launch': Ls, 'ms_per_step': ms, 'kernel_ms': k_ms, 'value': world * w.batch * Ls / (ms * 1e-3),
                          'frac': bytes_launch / (k_ms * 1e-3) / 1e9 / hbm_peak()[0],
                          'step_frac': bytes_launch / (ms * 1e-3) / 1e9 / hbm_peak()[0]})
        cur_L[0] = L
        launches = n_launches
        del dominant_ms[n_kernel_ms:]

    # ---- end to end through the public API with host buffers ----
    e2e = None
    if not args.no_e2e:
        Le = args.e2e_batches or max(1, min(L, (64 << 20) // (w.bytes_per_transition * w.batch // 2 + 1)))
        host_sampler = cls(dataset, w.config, device=local, seed=4321, stream_id=rank, output='numpy')
        rows = Le * w.batch
        n_valid = episodes * (w.steps - 1)
        pinned = C.c_void_p()
        _native.check(lib.ogb_host_alloc(rows * 8 * 4, C.byref(pinned)))
        pool = np.frombuffer((C.c_ubyte * (rows * 8 * 4)).from_address(pinned.value), dtype=np.int64).reshape(4, rows)
        rng = np.random.default_rng(rank)
        pos = rng.integers(0, n_valid, size=(4, rows))
        pool[:] = pos + pos // (w.steps - 1)  # valid_idxs[j] = j + j // (T-1) for fixed-length compact trajectories
        steps_e = args.steps
        for i in range(3):
            out = host_sampler.sample_many(Le, w.batch, idxs=pool[i % 4])
        # keys the reference fills with equal values share one buffer here (dedup): count every copied byte once
        d2h = sum(n for _, n in {(v.__array_interface__['data'][0], v.nbytes) for v in out.values()})
        del out
        barrier()
        t0 = time.perf_counter()
        for i in range(steps_e):
            out = host_sampler.sample_many(Le, w.batch, idxs=pool[i % 4])  # returns after the D2H copy has completed
            del out
        torch.cuda.synchronize(local)
        dt_direct = dist_util.reduce_scalar(time.perf_counter() - t0, 'max', device=dev)
        # The same calls through ogbench_b200.Prefetcher (public API): its worker launches step k+1 before it copies step k
        # out, so the index upload and the kernels of k+1 run under the D2H copy of k.  Timed from arrival to arrival in
        # steady state: the batches the worker got ahead during the barrier are consumed before the clock starts.
        from itertools import count

        from ogbench_b200 import Prefetcher

        depth = 2
        with Prefetcher(host_sampler, w.batch, depth=depth, num_batches=Le, idxs=(pool[i % 4] for i in count())) as batches:
            for _ in range(2):
                next(batches)
            barrier()
            for _ in range(depth + 2):
                next(batches)
            # two passes of steps_e steps each, the faster one is reported (both are in `passes`): the hosts of this pool are
            # shared VMs whose PCIe rate dips for seconds at a time (the raw probe below sees the same dips)
            pass_dt = []
            for _ in range(2):
                t0 = time.perf_counter()
                for _ in range(steps_e):
                    out = next(batches)
                    del out
                pass_dt.append(dist_util.reduce_scalar(time.perf_counter() - t0, 'max', device=dev))
        dt = min(pass_dt)
        barrier()
        link = link_probe(torch, torch.device('cuda', local), int(d2h))      # every rank copies at the same time, like the e2e leg
        link_min = -dist_util.reduce_scalar(-link, 'max', device=dev)
        link_sum = dist_util.reduce_scalar(link, 'sum', device=dev)
        e2e_value = world * steps_e * rows / dt
        e2e = {'value': e2e_value, 'unit': UNIT, 'numa_bound': ctx['numa'] is not None, 'h2d_bytes_per_step': rows * 8,
               'd2h_bytes_per_step': int(d2h), 'steps': steps_e, 'batches_per_step': Le,
               'direct_call_value': world * steps_e * rows / dt_direct,
               'passes': [world * steps_e * rows / t for t in pass_dt],
               'link_gbs': link_sum, 'link_gbs_slowest_rank': link_min,
               'frac_of_link': e2e_value * (d2h / rows) / 1e9 / link_sum,
               'link_note': 'raw pinned cudaMemcpyAsync D2H of one e2e block per rank, all ranks copying at once, summed over ranks',
               'api': "Prefetcher(GCDataset(..., output='numpy'), B, num_batches=L, idxs=host index arrays): next(batches); "
                      "direct_call_value = the same steps as plain sample_many(L, B, idxs=host) calls, one at a time"}
        lib.ogb_host_free(pinned)
        del host_sampler

    del sampler, dataset
    import gc

    gc.collect()
    torch.cuda.empty_cache()

    peak, peak_src = hbm_peak()
    achieved = w.bytes_per_transition * per_step / (kernel_ms * 1e-3) / 1e9
    traffic, traffic_note = committed_traffic(key, kernel_name, kernel_ms, per_step)
    out_bytes = w.bytes_per_transition * per_step // 2
    result = {
        'value': value, 'ms_per_step': elapsed_ms / n_steps, 'batches_per_launch': L,
        'timed_region_ms': elapsed_ms, 'steps_timed': n_steps,
        'roofline': {'bound': 'hbm', 'achieved': achieved, 'peak': peak, 'unit': 'GB/s', 'frac': achieved / peak, 'traffic': traffic,
                     'traffic_source': traffic_note, 'kernel': kernel_name, 'kernel_ms': kernel_ms,
                     'bytes_per_transition': w.bytes_per_transition, 'bytes_per_launch': w.bytes_per_transition * per_step,
                     'peak_source': peak_src,
                     'nominal_peak': NOMINAL_HBM_GBS, 'frac_of_nominal': achieved / NOMINAL_HBM_GBS,
                     'step_frac': w.bytes_per_transition * per_step / (elapsed_ms / n_steps * 1e-3) / 1e9 / peak,
                     'note': 'achieved = algorithmic bytes of one launch / device time of the dominant kernel (CUDA events on its '
                             'stream); step_frac = the same bytes / whole step time (index kernel and launch gaps included)'},
        'clocks': clocks.summary(),
        'gpu_launches': launches,
        'launch_size_sweep': sweep,
        'notes': f'each step writes {out_bytes / 1e6:.0f} MB into one of three rotating output blocks and gathers random rows of a '
                 f'{resident / 1e6:.0f} MB resident dataset (L2 is 126 MB)'
                 + (f'; OGB_BENCH_EPISODES={episodes}: NOT the BASELINE shape' if episodes != w.episodes else ''),
    }
    if e2e is not None:
        result['e2e'] = e2e
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        budget = args.cpu_seconds if headline else min(args.cpu_seconds, 4.0)
        rate, sample, _ = cpu_baseline(key, 1, 4, 1, budget_s=budget)
        result['cpu_baseline'] = {'value': rate, 'unit': UNIT, 'cores': 1, 'kind': 'port', 'sample': sample,
                                  'host_cores_available': os.cpu_count()}
    return result


def run_gpu_arm(args):
    import torch
    import torch.distributed as dist

    from ogbench_b200 import _native, dist_util, synthetic

    rank, world, local = dist_util.env_rank()
    if world > 1:   # NCCL prints its version / debug lines to stdout: keep stdout for the one JSON line
        os.environ.setdefault('NCCL_DEBUG_FILE', '/dev/stderr')
        if os.environ.get('NCCL_DEBUG', '').upper() in ('', 'VERSION'):
            os.environ['NCCL_DEBUG'] = 'WARN'        # (an explicit INFO/TRACE request from the caller is left alone)
    torch.cuda.set_device(local)
    numa = dist_util.bind_to_gpu_numa(local) if world > 1 and not os.environ.get('OGB_NO_NUMA_BIND') else None
    dist_util.init('nccl', device=torch.device('cuda', local))
    ctx = {'torch': torch, 'dist_util': dist_util, 'lib': _native.lib(), '_native': _native, 'rank': rank, 'world': world,
           'local': local, 'numa': numa}

    head_key = args.config or HEADLINE
    head = measure_config(head_key, args, ctx, headline=True)
    others = {}
    if args.config is None:
        for key in ALL_CONFIGS:
            others[key] = head if key == head_key else measure_config(key, args, ctx, headline=False)

    if rank == 0:
        w = synthetic.WORKLOADS[head_key]
        line = {
            'metric': METRIC, 'value': head['value'], 'unit': UNIT, 'n_gpus': world, 'steps': args.steps, 'warmup': max(args.warmup, 3),
            'ms_per_step': head['ms_per_step'], 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
            'dtype': 'u8' if w.obs_dtype == 'uint8' else 'f32', 'data': 'synthetic',
            'config': config_dict(head_key, head['batches_per_launch']),
            'timed_region_ms': head['timed_region_ms'], 'steps_timed': head['steps_timed'],
            'rng': 'on-device Philox4x32-10', 'api': 'GCDataset.sample_many(batches_per_launch, batch) -> dict of device arrays',
            'notes': head['notes'],
            'roofline': head['roofline'], 'clocks': head['clocks'], 'gpu_launches': head['gpu_launches'],
        }
        for k in ('e2e', 'cpu_baseline'):
            if k in head:
                line[k] = head[k]
        if others:
            line['configs'] = {k: dict(v, workload=synthetic.WORKLOADS[k].name, batch=synthetic.WORKLOADS[k].batch,
                                       dtype='u8' if synthetic.WORKLOADS[k].obs_dtype == 'uint8' else 'f32',
                                       placement=config_dict(k, v['batches_per_launch'])['placement'])
                               for k, v in others.items()}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse_args()
    if args.impl == 'reference':
        run_reference_arm(args)
    else:
        run_gpu_arm(args)


if __name__ == '__main__':
    main()

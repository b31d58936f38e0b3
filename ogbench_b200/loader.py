"""The step before the hot path: OGBench `.npz` files -> HBM-resident datasets, with shard cycling.

`load_dataset` has the signature and the result of `ogbench.load_dataset` (ogbench/utils.py:14-96): a dict of host
arrays in the regular or the compact layout.  It is I/O (np.load, decompression) plus an O(N) pass over the
1-D `terminals` array, so it stays on the host like the reference's; what changes is what happens next --
`load_gc_dataset` uploads the fields once and returns a device sampler, and `ShardCycler` reproduces the
directory-of-shards mode of impls/main.py:81-93,185-199 with the *next* shard loaded and uploaded by a background
thread while the current one is being sampled, so the swap every `dataset_replace_interval` steps costs nothing.
`ResidentShards` removes the reload altogether: every shard of a directory is uploaded once into one HBM table, each
shard is a view of it (the dataset the shard's file would give) and the whole table is the concatenated dataset.
"""

from __future__ import annotations

import atexit
import ctypes as C
import glob
import threading
import weakref
import zipfile
from collections.abc import Mapping
from typing import Any, Callable, List, Optional

import numpy as np

from . import _native
from .datasets import Dataset, GCDataset, ResidentDataset, _flatten, _NativeDataset, _ZeroField


def load_dataset(dataset_path, ob_dtype=np.float32, action_dtype=np.float32, compact_dataset=False, add_info=False):
    """Load an OGBench dataset file (same contract as ogbench/utils.py:14-96).

    Returns a dict with 'observations', 'actions', 'terminals' and 'next_observations' (regular layout) or 'valids'
    (compact layout); with add_info also 'qpos', 'qvel', 'button_states' when the file has them.
    """
    file = np.load(dataset_path)
    dataset = {}
    for k, dtype in (('observations', ob_dtype), ('actions', action_dtype), ('terminals', np.float32)):
        dataset[k] = file[k][...].astype(dtype, copy=False)
    info_keys = []
    if add_info:
        for k in ('qpos', 'qvel', 'button_states'):
            if k in file:
                dataset[k] = file[k][...]
                info_keys.append(k)

    terminals = dataset['terminals']
    follows_terminal = np.concatenate([terminals[1:], [1.0]])       # terminals shifted left, the file ends a trajectory
    if compact_dataset:
        # keep every row; the last row of a trajectory is only ever a next-observation, so it is marked invalid and
        # its predecessor becomes terminal as well (ogbench/utils.py:60-73)
        dataset['valids'] = 1.0 - terminals
        dataset['terminals'] = np.minimum(terminals + follows_terminal, 1.0).astype(np.float32)
    else:
        # regular layout: drop each trajectory's last row, next_observations are the rows shifted by one
        # (ogbench/utils.py:74-94)
        ob_mask = (1.0 - terminals).astype(bool)
        next_ob_mask = np.concatenate([[False], ob_mask[:-1]])
        dataset['next_observations'] = dataset['observations'][next_ob_mask]
        dataset['observations'] = dataset['observations'][ob_mask]
        dataset['actions'] = dataset['actions'][ob_mask]
        dataset['terminals'] = follows_terminal[ob_mask].astype(np.float32)
        for k in info_keys:
            dataset[k] = dataset[k][ob_mask]
    return dataset


def add_oracle_reps(env_name, env, dataset, num_cubes=None, num_buttons=None):
    """Add oracle goal representations to the dataset (same contract as ogbench/relabel_utils.py:93-155).

    `env` may be None when `num_cubes` / `num_buttons` are given (the reference reads them from
    `env.unwrapped._num_cubes` / `_num_buttons`); the dataset must have been loaded with add_info=True ('qpos',
    'button_states').  The sampler then serves goals from `oracle_reps` (datasets.py:348-357).
    """
    def count(attr, given):
        return given if given is not None else getattr(env.unwrapped, attr)

    qpos = dataset['qpos'] if ('maze' in env_name or 'soccer' in env_name or 'cube' in env_name or 'scene' in env_name) else None
    if 'maze' in env_name or 'soccer' in env_name:
        start = 0 if 'maze' in env_name else 15            # agent xy, or the ball's xy for antsoccer
        oracle_reps = qpos[:, start:start + 2]
    elif 'cube' in env_name or 'scene' in env_name or 'puzzle' in env_name:
        obj0, cube_len = 14, 7
        xyz_center = np.array([0.425, 0.0, 0.0])
        if 'puzzle' in env_name:
            oracle_reps = dataset['button_states'].copy()
        else:
            n_cubes = count('_num_cubes', num_cubes)
            cube_xyzs = np.stack([qpos[:, obj0 + i * cube_len:obj0 + i * cube_len + 3] for i in range(n_cubes)], axis=1)
            cube_reps = ((cube_xyzs - xyz_center) * 10.0).reshape(-1, n_cubes * 3)
            if 'cube' in env_name:
                oracle_reps = cube_reps
            else:
                drawer = obj0 + n_cubes * cube_len + count('_num_buttons', num_buttons)
                oracle_reps = np.concatenate(
                    [cube_reps, dataset['button_states'].copy(), qpos[:, [drawer]] * 18.0, qpos[:, [drawer + 1]] * 15.0], axis=-1)
    else:
        raise ValueError(f'Unsupported environment: {env_name}')
    dataset['oracle_reps'] = oracle_reps.astype(np.float32)


def relabel_dataset(env_name, env, dataset):
    """Add the single-task 'rewards' and 'masks' of the environment's fixed task (same contract as
    ogbench/relabel_utils.py:4-90).  `env` is the single-task environment (anything exposing the attributes the reference
    reads from `env.unwrapped`: `_reward_task_id`, `cur_goal_xy` / `_goal_tol` for the mazes and antsoccer, `_num_cubes`,
    `_num_buttons`, `_data.mocap_pos`, `_target_button_states`, `_target_drawer_pos`, `_target_window_pos` for
    manipulation); `env.reset()` is called first, as in the reference, so that the task is set.  The dataset must carry
    'qpos' (and 'button_states' for scene / puzzle), i.e. be loaded with add_info=True.
    """
    task = env.unwrapped
    assert task._reward_task_id is not None, 'The environment is not in the single-task mode.'
    env.reset()
    tol = 0.04                                              # object / drawer / window tolerance of the manipulation tasks
    if 'maze' in env_name or 'soccer' in env_name:
        first = 0 if 'maze' in env_name else 15             # the agent's xy, or the ball's for antsoccer
        gap = np.linalg.norm(dataset['qpos'][:, first:first + 2] - task.cur_goal_xy, axis=-1)
        reached = (gap <= task._goal_tol).astype(np.float32)
        rewards, masks = reached - 1.0, 1.0 - reached       # -1 until the goal is reached; the episode stops mattering there
    elif 'cube' in env_name or 'scene' in env_name or 'puzzle' in env_name:
        obj0, cube_len = 14, 7
        done = []                                           # one boolean column per sub-goal of the task
        if 'cube' in env_name or 'scene' in env_name:
            n_cubes = task._num_cubes
            xyz = np.stack([dataset['qpos'][:, obj0 + c * cube_len:obj0 + c * cube_len + 3] for c in range(n_cubes)], axis=1)
            done.append(np.linalg.norm(task._data.mocap_pos.copy() - xyz, axis=-1) <= tol)
        if 'scene' in env_name and 'cube' not in env_name:
            drawer = obj0 + task._num_cubes * cube_len + task._num_buttons
            done.append(dataset['button_states'] == task._target_button_states.copy())
            done.append((np.abs(dataset['qpos'][:, drawer] - task._target_drawer_pos) <= tol)[:, None])
            done.append((np.abs(dataset['qpos'][:, drawer + 1] - task._target_window_pos) <= tol)[:, None])
        if 'puzzle' in env_name and 'cube' not in env_name and 'scene' not in env_name:
            done.append(dataset['button_states'] == task._target_button_states.copy())
        done = np.concatenate(done, axis=-1)
        rewards = done.sum(axis=-1) - done.shape[-1]        # minus the number of unfinished sub-goals
        masks = 1.0 - np.all(done, axis=-1)
    else:
        raise ValueError(f'Unsupported environment: {env_name}')
    dataset['rewards'] = rewards.astype(np.float32)
    dataset['masks'] = masks.astype(np.float32)


def make_datasets(dataset_name, dataset_dir='~/.ogbench/data', dataset_path=None, compact_dataset=False, add_info=False,
                  env=None, num_cubes=None, num_buttons=None):
    """The dataset half of `ogbench.make_env_and_datasets(..., dataset_only=True)` (ogbench/utils.py:134-235): resolves the
    train / validation files of `dataset_name`, picks the dtypes by environment family, loads both splits and, for
    '-oraclerep-' names, adds the oracle goal representations.  Returns (train_dataset, val_dataset) as dicts of host
    arrays; 'singletask' names are relabelled with the rewards / masks of `env`'s fixed task (relabel_dataset).  Nothing is
    downloaded (the files must exist).
    """
    import os

    splits = dataset_name.split('-')
    dataset_add_info = add_info
    if 'singletask' in splits:
        if env is None:
            raise ValueError("'singletask' datasets are relabelled with the task of the single-task environment: pass env= "
                             '(ogbench/utils.py:164-171, relabel_utils.py:4-90)')
        pos = splits.index('singletask')
        env_name = '-'.join(splits[:pos - 1] + splits[pos:])      # remove the dataset type
        dataset_name = '-'.join(splits[:pos] + splits[-1:])        # the files carry neither 'singletask' nor 'task<n>'
        dataset_add_info = True
    elif 'oraclerep' in splits:
        env_name = '-'.join(splits[:-3] + splits[-1:])         # remove the dataset type and the word 'oraclerep'
        dataset_name = '-'.join(splits[:-2] + splits[-1:])     # the files carry no 'oraclerep'
        dataset_add_info = True
    else:
        env_name = '-'.join(splits[:-2] + splits[-1:])         # remove the dataset type
    if dataset_path is None:
        dataset_dir = os.path.expanduser(dataset_dir)
        train_path = os.path.join(dataset_dir, f'{dataset_name}.npz')
        val_path = os.path.join(dataset_dir, f'{dataset_name}-val.npz')
    else:
        train_path, val_path = dataset_path, dataset_path.replace('.npz', '-val.npz')
    for path in (train_path, val_path):
        if not os.path.exists(path):
            raise FileNotFoundError(f'{path} (datasets are not downloaded by this loader)')
    ob_dtype = np.uint8 if ('visual' in env_name or 'powderworld' in env_name) else np.float32
    action_dtype = np.int32 if 'powderworld' in env_name else np.float32
    out = []
    for path in (train_path, val_path):
        ds = load_dataset(path, ob_dtype=ob_dtype, action_dtype=action_dtype, compact_dataset=compact_dataset, add_info=dataset_add_info)
        if 'singletask' in splits:
            relabel_dataset(env_name, env, ds)
        if 'oraclerep' in splits:
            add_oracle_reps(env_name, env, ds, num_cubes=num_cubes, num_buttons=num_buttons)
        if not add_info:
            for k in ('qpos', 'qvel', 'button_states'):
                ds.pop(k, None)
        out.append(ds)
    return out[0], out[1]


def load_gc_dataset(dataset_path, config, dataset_class=GCDataset, ob_dtype=np.float32, action_dtype=np.float32,
                    device: int = 0, **sampler_kwargs):
    """`.npz` -> compact layout (what impls/utils/env_utils.py:89-95 asks for) -> HBM -> device sampler."""
    fields = load_dataset(dataset_path, ob_dtype=ob_dtype, action_dtype=action_dtype, compact_dataset=True)
    dataset = Dataset.create(**fields)
    return dataset_class(dataset, config, device=device, **sampler_kwargs)


def list_shards(dataset_dir: str) -> List[str]:
    """Training shards of a dataset directory (impls/main.py:84-88): sorted *.npz without the validation files."""
    shards = [f for f in sorted(glob.glob(f'{dataset_dir}/*.npz')) if '-val.npz' not in f]
    if not shards:
        raise FileNotFoundError(f'No .npz files found in {dataset_dir}')
    return shards


_LIVE_CYCLERS: 'weakref.WeakSet[ShardCycler]' = weakref.WeakSet()


@atexit.register
def _join_prefetch_threads():
    # an upload must not be in flight inside the CUDA library while the interpreter shuts down
    for c in list(_LIVE_CYCLERS):
        c.close()


class ShardCycler:
    """Cycle through dataset shards like impls/main.py:185-199, without the reload stall.

        cycler = ShardCycler(list_shards(path), make_sampler=lambda p: load_gc_dataset(p, config, seed=FLAGS.seed),
                             replace_interval=1000)
        for i in range(1, train_steps + 1):
            train_dataset = cycler.at_step(i)          # swaps to the next shard when i % replace_interval == 0
            batch = train_dataset.sample(batch_size)

    Random goals stay shard-local, exactly as in the reference (only the loaded shard is sampled).  The sampler's
    RNG position (its Philox batch counter) is carried from shard to shard, so revisiting a shard draws new batches.
    """

    def __init__(self, shard_paths: List[str], make_sampler: Callable[[str], Any], replace_interval: int, prefetch: bool = True):
        assert len(shard_paths) >= 1
        self.paths = list(shard_paths)
        self.make_sampler = make_sampler
        self.replace_interval = int(replace_interval)
        self.prefetch = prefetch
        self.index = 0
        self.current = make_sampler(self.paths[0])
        self.swaps = 0
        self.prefetched_swaps = 0
        self._next: Optional[Any] = None
        self._next_index: Optional[int] = None
        self._thread: Optional[threading.Thread] = None
        self._error: Optional[BaseException] = None
        _LIVE_CYCLERS.add(self)
        self._start_prefetch()

    def _start_prefetch(self):
        if not self.prefetch or len(self.paths) < 2 or self.replace_interval <= 0:
            return
        nxt = (self.index + 1) % len(self.paths)

        def work():
            try:
                self._next = self.make_sampler(self.paths[nxt])   # np.load + upload; ctypes releases the GIL
            except BaseException as exc:  # surfaced at the swap
                self._error = exc

        self._next, self._next_index, self._error = None, nxt, None
        self._thread = threading.Thread(target=work, daemon=True)
        self._thread.start()

    def at_step(self, step: int):
        """Sampler to use at training step `step` (1-based, like the loop in impls/main.py:183)."""
        if self.replace_interval > 0 and len(self.paths) > 1 and step % self.replace_interval == 0:
            self.index = (self.index + 1) % len(self.paths)
            if self._thread is not None:
                ready_early = not self._thread.is_alive()
                self._thread.join()
                self._thread = None
                if self._error is not None:
                    raise self._error
                assert self._next_index == self.index
                previous, self.current, self._next = self.current, self._next, None
                self.prefetched_swaps += int(ready_early)
            else:
                previous, self.current = self.current, self.make_sampler(self.paths[self.index])
            self._carry_rng(previous, self.current)
            self.swaps += 1
            self._start_prefetch()
        return self.current

    @staticmethod
    def _carry_rng(previous, current):
        """The reference keeps consuming ONE np.random stream across shard swaps (impls/main.py:185-202), so a revisited
        shard never replays its batches.  A fresh sampler starts at Philox counter 0: hand it the position the previous
        shard's sampler had reached (same seed / stream_id, the counter keeps advancing over the whole run)."""
        if hasattr(previous, 'state_dict') and hasattr(current, 'load_state_dict'):
            current.load_state_dict(previous.state_dict())

    def close(self):
        if self._thread is not None:
            self._thread.join()
            self._thread = None


def shard_rows(path) -> int:
    """Rows of an `.npz` file as its `terminals` header declares them, read from the zip member's `.npy` header without
    decompressing the data (np.savez and np.savez_compressed files alike)."""
    with zipfile.ZipFile(path) as zf, zf.open('terminals.npy') as f:
        version = np.lib.format.read_magic(f)
        read_header = np.lib.format.read_array_header_1_0 if version == (1, 0) else np.lib.format.read_array_header_2_0
        shape, _, _ = read_header(f)
    return int(shape[0])


class ResidentShards:
    """Every shard of a dataset directory, uploaded once into one HBM table.

        shards = ResidentShards(list_shards(path))
        shards.dataset            # Dataset over every row, shards in path order: the concatenated dataset
        shards[i], shards[path]   # Dataset of one shard: a view of the table, equal to Dataset.create(**load(path))
        shards.bounds             # [(row0, n_rows)] per shard

    `load` is the per-file host loader (default: load_dataset(p, compact_dataset=True); `lambda p: make_datasets(name,
    dataset_path=p)[0]` for '-oraclerep-' and 'singletask' names).  The capacity comes from the files' headers; then the
    shards are loaded, written and freed one at a time, so host memory peaks at one shard plus a pinned staging buffer.
    Every shard must load with shard 0's fields, dtypes and row shapes.

    A view keeps the reference's shard-local semantics (goals, trajectory ends and next observations stay inside the
    shard) and a swap costs no upload; sampling `dataset` draws across every shard instead.  Shards end on trajectory
    boundaries, so each rank of a multi-GPU run can build its own ResidentShards over its subset of the paths.
    """

    def __init__(self, paths, load: Optional[Callable[[str], dict]] = None, device: int = 0):
        self.paths = [str(p) for p in paths]
        lib = _native.lib()
        nds, keys, nested, valids, self.bounds = None, None, False, [], []
        for shard in iter_shards(self.paths, load):
            if nds is None:
                keys, nested = shard.keys, shard.nested
                nds = _NativeDataset.empty({k: _ZeroField((shard.capacity, *s), d) for k, (d, s) in shard.schema.items()}, device)
            arrays = [np.ascontiguousarray(shard.fields[k]) for k in shard.schema]
            ptrs = (C.c_void_p * len(arrays))(*[a.ctypes.data for a in arrays])
            _native.check(lib.ogb_dataset_write_rows(nds.ptr, shard.row0, shard.n_rows, ptrs, len(arrays)))
            if 'valids' in shard.fields:
                valids.append((shard.fields['valids'] > 0).astype(np.uint8))
            self.bounds.append((shard.row0, shard.n_rows))
            del arrays, ptrs, shard                   # this shard's host arrays go before the next one is loaded
        n_rows = sum(n for _, n in self.bounds)
        _native.check(lib.ogb_dataset_seal(nds.ptr, n_rows))
        flags = np.concatenate(valids) if valids else None
        self.dataset = ResidentDataset(nds, keys, nested, flags)
        self._views = [ResidentDataset(nds.view(r0, n), keys, nested, flags[r0:r0 + n] if flags is not None else None)
                       for r0, n in self.bounds]

    def __len__(self):
        return len(self.paths)

    def __getitem__(self, key) -> ResidentDataset:
        """The shard `key` (its index, or its path as given) as a dataset of its own."""
        if isinstance(key, str):
            if key not in self.paths:
                raise KeyError(key)
            key = self.paths.index(key)
        return self._views[key]


class _Shard:
    __slots__ = ('path', 'row0', 'n_rows', 'capacity', 'keys', 'nested', 'schema', 'fields')


def iter_shards(paths, load: Optional[Callable[[str], dict]] = None):
    """The host half of ResidentShards: load the shards one at a time, in order, and yield each as a record with its
    first row in the concatenation (`row0`), its row count, its flattened fields and the schema -- {name: (dtype, row
    shape)} -- that shard 0 fixed; `capacity` is the rows the files' headers declare in all.  A shard whose fields, dtypes
    or row shapes differ from shard 0's, or that loads more rows than its header declares, raises ValueError naming it."""
    paths = [str(p) for p in paths]
    if not paths:
        raise ValueError('no shards given')
    if load is None:
        load = lambda p: load_dataset(p, compact_dataset=True)  # noqa: E731
    declared = [shard_rows(p) for p in paths]
    schema, row0 = None, 0
    for path, cap in zip(paths, declared):
        tree = load(path)
        fields = _flatten(tree)
        shape = {k: (np.asarray(v).dtype, np.asarray(v).shape[1:]) for k, v in fields.items()}
        if schema is None:
            schema, keys, nested = shape, list(tree), any(isinstance(v, Mapping) for v in tree.values())
        elif shape != schema:
            raise ValueError(f'{path}: fields {_describe(shape)} differ from those of {paths[0]}: {_describe(schema)}')
        lengths = {len(v) for v in fields.values()}
        if len(lengths) != 1:
            raise ValueError(f'{path}: fields of different lengths {sorted(lengths)}')
        n = lengths.pop()
        if n > cap:
            raise ValueError(f'{path}: {n} rows loaded, the file declares {cap}')
        shard = _Shard()
        shard.path, shard.row0, shard.n_rows, shard.capacity = path, row0, n, sum(declared)
        shard.keys, shard.nested, shard.schema, shard.fields = keys, nested, schema, fields
        del tree, fields
        yield shard
        del shard                                     # (the caller's reference is the last one before the next load)
        row0 += n


def _describe(schema) -> str:
    return ', '.join(f'{k}: {d}{tuple(s)}' for k, (d, s) in schema.items())

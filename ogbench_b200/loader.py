"""The step before the hot path: OGBench `.npz` files -> HBM-resident datasets, with shard cycling.

`load_dataset` has the signature and the result of `ogbench.load_dataset` (ogbench/utils.py:14-96): a dict of host
arrays in the regular or the compact layout.  It is I/O (np.load, decompression) plus an O(N) pass over the
1-D `terminals` array, so it stays on the host like the reference's; what changes is what happens next --
`load_gc_dataset` uploads the fields once and returns a device sampler, and `ShardCycler` reproduces the
directory-of-shards mode of impls/main.py:81-93,185-199 with the *next* shard loaded and uploaded by a background
thread while the current one is being sampled, so the swap every `dataset_replace_interval` steps costs nothing.
`ResidentShards` removes the reload altogether: every shard of a directory is uploaded once into one HBM table, each
shard is a view of it (the dataset the shard's file would give) and the whole table is the concatenated dataset.
`upload_dataset` gives load_dataset's result in HBM without the host copy: the file is inflated, cast, laid out and
written a block at a time, which is also how ResidentShards reads its files with the default loader.
`upload_datasets` does the same for `make_datasets`, whose '-oraclerep-' and 'singletask' relabellings are row-local
and run per block.
"""

from __future__ import annotations

import ast
import atexit
import contextlib
import ctypes as C
import functools
import glob
import queue
import threading
import weakref
import zipfile
from collections.abc import Mapping
from typing import Any, Callable, List, NamedTuple, Optional, Tuple

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


class _Relabelling(NamedTuple):
    """A relabelling with its constants resolved: `rows(info)` maps rows of the info members `members` ({'qpos': rows,
    'button_states': rows}) to the same rows of the derived fields.  Every expression is row-local, so the whole arrays
    and any block of their rows give the same elements."""
    members: Tuple[str, ...]
    rows: Callable[[Mapping], dict]


def _oracle_relabelling(env_name, env, num_cubes=None, num_buttons=None) -> _Relabelling:
    """add_oracle_reps' constants for `env_name`, read once, and its per-row arithmetic (ogbench/relabel_utils.py:93-155)."""
    def count(attr, given):
        return given if given is not None else getattr(env.unwrapped, attr)

    obj0, cube_len = 14, 7
    xyz_center = np.array([0.425, 0.0, 0.0])
    if 'maze' in env_name or 'soccer' in env_name:
        start = 0 if 'maze' in env_name else 15            # agent xy, or the ball's xy for antsoccer
        members = ('qpos',)
    elif 'cube' in env_name or 'scene' in env_name or 'puzzle' in env_name:
        if 'puzzle' in env_name:
            members = ('button_states',)
        else:
            n_cubes = count('_num_cubes', num_cubes)
            if 'cube' in env_name:
                members = ('qpos',)
            else:
                drawer = obj0 + n_cubes * cube_len + count('_num_buttons', num_buttons)
                members = ('qpos', 'button_states')
    else:
        raise ValueError(f'Unsupported environment: {env_name}')

    def rows(info):
        if 'maze' in env_name or 'soccer' in env_name:
            oracle_reps = info['qpos'][:, start:start + 2]
        elif 'puzzle' in env_name:
            oracle_reps = info['button_states'].copy()
        else:
            qpos = info['qpos']
            cube_xyzs = np.stack([qpos[:, obj0 + i * cube_len:obj0 + i * cube_len + 3] for i in range(n_cubes)], axis=1)
            cube_reps = ((cube_xyzs - xyz_center) * 10.0).reshape(-1, n_cubes * 3)
            if 'cube' in env_name:
                oracle_reps = cube_reps
            else:
                oracle_reps = np.concatenate(
                    [cube_reps, info['button_states'].copy(), qpos[:, [drawer]] * 18.0, qpos[:, [drawer + 1]] * 15.0], axis=-1)
        return {'oracle_reps': oracle_reps.astype(np.float32)}

    return _Relabelling(members, rows)


def _task_relabelling(env_name, env) -> _Relabelling:
    """relabel_dataset's constants for `env_name`, read from the single-task `env` after its reset, and its per-row
    arithmetic (ogbench/relabel_utils.py:4-90)."""
    task = env.unwrapped
    assert task._reward_task_id is not None, 'The environment is not in the single-task mode.'
    env.reset()
    tol = 0.04                                              # object / drawer / window tolerance of the manipulation tasks
    obj0, cube_len = 14, 7
    maze = 'maze' in env_name or 'soccer' in env_name
    cubes = 'cube' in env_name or 'scene' in env_name
    scene = 'scene' in env_name and 'cube' not in env_name
    puzzle = 'puzzle' in env_name and 'cube' not in env_name and 'scene' not in env_name
    if maze:
        first = 0 if 'maze' in env_name else 15             # the agent's xy, or the ball's for antsoccer
        goal_xy, goal_tol = task.cur_goal_xy, task._goal_tol
        members = ('qpos',)
    elif cubes or 'puzzle' in env_name:
        if cubes:
            n_cubes, mocap_pos = task._num_cubes, task._data.mocap_pos.copy()
        if scene:
            drawer = obj0 + task._num_cubes * cube_len + task._num_buttons
        if scene or puzzle:
            target_buttons = task._target_button_states.copy()
        if scene:
            target_drawer, target_window = task._target_drawer_pos, task._target_window_pos
        members = ('qpos',) * cubes + ('button_states',) * (scene or puzzle)
    else:
        raise ValueError(f'Unsupported environment: {env_name}')

    def rows(info):
        if maze:
            gap = np.linalg.norm(info['qpos'][:, first:first + 2] - goal_xy, axis=-1)
            reached = (gap <= goal_tol).astype(np.float32)
            rewards, masks = reached - 1.0, 1.0 - reached   # -1 until the goal is reached; the episode stops mattering there
        else:
            done = []                                       # one boolean column per sub-goal of the task
            if cubes:
                xyz = np.stack([info['qpos'][:, obj0 + c * cube_len:obj0 + c * cube_len + 3] for c in range(n_cubes)], axis=1)
                done.append(np.linalg.norm(mocap_pos - xyz, axis=-1) <= tol)
            if scene:
                done.append(info['button_states'] == target_buttons)
                done.append((np.abs(info['qpos'][:, drawer] - target_drawer) <= tol)[:, None])
                done.append((np.abs(info['qpos'][:, drawer + 1] - target_window) <= tol)[:, None])
            if puzzle:
                done.append(info['button_states'] == target_buttons)
            done = np.concatenate(done, axis=-1)
            rewards = done.sum(axis=-1) - done.shape[-1]    # minus the number of unfinished sub-goals
            masks = 1.0 - np.all(done, axis=-1)
        return {'rewards': rewards.astype(np.float32), 'masks': masks.astype(np.float32)}

    return _Relabelling(members, rows)


def add_oracle_reps(env_name, env, dataset, num_cubes=None, num_buttons=None):
    """Add oracle goal representations to the dataset (same contract as ogbench/relabel_utils.py:93-155).

    `env` may be None when `num_cubes` / `num_buttons` are given (the reference reads them from
    `env.unwrapped._num_cubes` / `_num_buttons`); the dataset must have been loaded with add_info=True ('qpos',
    'button_states').  The sampler then serves goals from `oracle_reps` (datasets.py:348-357).
    """
    dataset.update(_oracle_relabelling(env_name, env, num_cubes, num_buttons).rows(dataset))


def relabel_dataset(env_name, env, dataset):
    """Add the single-task 'rewards' and 'masks' of the environment's fixed task (same contract as
    ogbench/relabel_utils.py:4-90).  `env` is the single-task environment (anything exposing the attributes the reference
    reads from `env.unwrapped`: `_reward_task_id`, `cur_goal_xy` / `_goal_tol` for the mazes and antsoccer, `_num_cubes`,
    `_num_buttons`, `_data.mocap_pos`, `_target_button_states`, `_target_drawer_pos`, `_target_window_pos` for
    manipulation); `env.reset()` is called first, as in the reference, so that the task is set.  The dataset must carry
    'qpos' (and 'button_states' for scene / puzzle), i.e. be loaded with add_info=True.
    """
    dataset.update(_task_relabelling(env_name, env).rows(dataset))


class _DatasetName(NamedTuple):
    """What a dataset name of make_datasets says: the environment, the files' stem, the dtypes of the family, whether the
    info members are read (the relabelled names need them) and which relabellings apply."""
    env_name: str
    file_stem: str
    ob_dtype: type
    action_dtype: type
    load_info: bool
    singletask: bool
    oraclerep: bool

    def paths(self, dataset_dir='~/.ogbench/data', dataset_path=None):
        """(train, validation) files; FileNotFoundError when either is missing."""
        import os

        if dataset_path is None:
            dataset_dir = os.path.expanduser(dataset_dir)
            out = os.path.join(dataset_dir, f'{self.file_stem}.npz'), os.path.join(dataset_dir, f'{self.file_stem}-val.npz')
        else:
            out = dataset_path, dataset_path.replace('.npz', '-val.npz')
        for path in out:
            if not os.path.exists(path):
                raise FileNotFoundError(f'{path} (datasets are not downloaded by this loader)')
        return out

    def stream(self, path, compact_dataset, add_info, env, num_cubes=None, num_buttons=None) -> '_FileStream':
        """make_datasets' result for the split `path` as a _FileStream; a single-task `env` is reset here, once."""
        relabellings = [_task_relabelling(self.env_name, env)] if self.singletask else []
        if self.oraclerep:
            relabellings.append(_oracle_relabelling(self.env_name, env, num_cubes, num_buttons))
        return _FileStream(path, self.ob_dtype, self.action_dtype, compact_dataset, add_info, relabellings)


def _parse_dataset_name(dataset_name, add_info=False, env=None) -> _DatasetName:
    """make_datasets' reading of `dataset_name` (ogbench/utils.py:164-203); a 'singletask' name without `env` is a
    ValueError."""
    splits = dataset_name.split('-')
    load_info = add_info
    if 'singletask' in splits:
        if env is None:
            raise ValueError("'singletask' datasets are relabelled with the task of the single-task environment: pass env= "
                             '(ogbench/utils.py:164-171, relabel_utils.py:4-90)')
        pos = splits.index('singletask')
        env_name = '-'.join(splits[:pos - 1] + splits[pos:])      # remove the dataset type
        dataset_name = '-'.join(splits[:pos] + splits[-1:])        # the files carry neither 'singletask' nor 'task<n>'
        load_info = True
    elif 'oraclerep' in splits:
        env_name = '-'.join(splits[:-3] + splits[-1:])         # remove the dataset type and the word 'oraclerep'
        dataset_name = '-'.join(splits[:-2] + splits[-1:])     # the files carry no 'oraclerep'
        load_info = True
    else:
        env_name = '-'.join(splits[:-2] + splits[-1:])         # remove the dataset type
    ob_dtype = np.uint8 if ('visual' in env_name or 'powderworld' in env_name) else np.float32
    action_dtype = np.int32 if 'powderworld' in env_name else np.float32
    return _DatasetName(env_name, dataset_name, ob_dtype, action_dtype, load_info, 'singletask' in splits, 'oraclerep' in splits)


def make_datasets(dataset_name, dataset_dir='~/.ogbench/data', dataset_path=None, compact_dataset=False, add_info=False,
                  env=None, num_cubes=None, num_buttons=None):
    """The dataset half of `ogbench.make_env_and_datasets(..., dataset_only=True)` (ogbench/utils.py:134-235): resolves the
    train / validation files of `dataset_name`, picks the dtypes by environment family, loads both splits and, for
    '-oraclerep-' names, adds the oracle goal representations.  Returns (train_dataset, val_dataset) as dicts of host
    arrays; 'singletask' names are relabelled with the rewards / masks of `env`'s fixed task (relabel_dataset).  Nothing is
    downloaded (the files must exist).  upload_datasets gives the same datasets in HBM without the host copy.
    """
    name = _parse_dataset_name(dataset_name, add_info, env)
    out = []
    for path in name.paths(dataset_dir, dataset_path):
        ds = load_dataset(path, ob_dtype=name.ob_dtype, action_dtype=name.action_dtype, compact_dataset=compact_dataset,
                          add_info=name.load_info)
        if name.singletask:
            relabel_dataset(name.env_name, env, ds)
        if name.oraclerep:
            add_oracle_reps(name.env_name, env, ds, num_cubes=num_cubes, num_buttons=num_buttons)
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
    with zipfile.ZipFile(path) as zf, _open_member(zf, path, 'terminals') as f:
        shape, _, _ = _read_npy_header(f, path, 'terminals')
    return int(shape[0])


# ------------------------------------------ streaming .npz members into HBM ------------------------------------------
_BLOCK_BYTES = 8 << 20          # one block of ogb_dataset_write_rows's pinned stage
_MAX_HEADER_BYTES = 10000       # np.load's default limit on a .npy header
_INFO_KEYS = ('qpos', 'qvel', 'button_states')


def _open_member(zf: zipfile.ZipFile, path, key):
    try:
        return zf.open(f'{key}.npy')
    except KeyError:
        raise KeyError(f'{key} is not a file in the archive {path}') from None


def _read_npy_header(f, path, key):
    """(shape, dtype, fortran_order) from the `.npy` header at the start of `f` (format versions 1.0, 2.0 and 3.0), which
    is left at the first byte of the array data."""
    magic = f.read(8)
    if len(magic) != 8 or magic[:6] != b'\x93NUMPY' or magic[6] not in (1, 2, 3) or magic[7] != 0:
        raise ValueError(f'{path}: member {key!r} is not a .npy array of format version 1.0, 2.0 or 3.0')
    length = int.from_bytes(f.read(2 if magic[6] == 1 else 4), 'little')
    text = f.read(length) if length <= _MAX_HEADER_BYTES else b''
    try:
        header = ast.literal_eval(text.decode('utf8' if magic[6] == 3 else 'latin1'))
        shape, fortran = tuple(int(n) for n in header['shape']), bool(header['fortran_order'])
        dtype = np.lib.format.descr_to_dtype(header['descr'])
    except Exception as exc:
        raise ValueError(f'{path}: member {key!r} has an unreadable .npy header') from exc
    return shape, dtype, fortran


def read_member_blocks(path, key, block_rows: Optional[int] = None):
    """The array `key` of the `.npz` file at `path` (what `np.load(path)[key]` gives), yielded as consecutive blocks of
    `block_rows` rows, by default about 8 MB of them.  Stored (np.savez) and deflated (np.savez_compressed) members alike,
    ZIP64 members included; only the current block is held in host memory.  A member that cannot be sliced into rows
    (Fortran order, object dtype, a 0-d or empty array) is read whole by np.load and yielded as one block.  A member
    that ends before the row count of its header raises ValueError; a missing member raises KeyError."""
    with zipfile.ZipFile(path) as zf, _open_member(zf, path, key) as f:
        shape, dtype, fortran = _read_npy_header(f, path, key)
        row_bytes = dtype.itemsize * int(np.prod(shape[1:], dtype=np.int64))
        streamable = not fortran and not dtype.hasobject and len(shape) >= 1 and shape[0] > 0 and row_bytes > 0
        if streamable:
            n = shape[0]
            rows = block_rows or max(1, _BLOCK_BYTES // row_bytes)
            for r0 in range(0, n, rows):
                m = min(rows, n - r0)
                data = f.read(m * row_bytes)
                if len(data) != m * row_bytes:
                    raise ValueError(f'{path}: member {key!r} ends after {r0 + len(data) // row_bytes} of the {n} rows '
                                     'its header declares')
                yield np.frombuffer(data, dtype).reshape(m, *shape[1:])
    if not streamable:
        with np.load(path) as z:
            yield z[key]


def _read_member(path, key) -> np.ndarray:
    blocks = list(read_member_blocks(path, key))
    return np.concatenate(blocks) if len(blocks) > 1 else blocks[0]


def _terminal_rows(terminals, r0, r1):
    """load_dataset's float32 `terminals` and `follows_terminal` (the next row's terminal, 1.0 after the file's last row)
    at the file rows [r0, r1), with its own expressions: every element equals the one of the whole-file arrays."""
    t = terminals[r0:r1].astype(np.float32)
    follows = np.concatenate([terminals[r0 + 1:r1 + 1].astype(np.float32), [1.0] if r1 == len(terminals) else []])
    return t, follows


def _lockstep(readers):
    """Lists of same-row blocks, one per reader, from readers that yield the consecutive rows of members of equal length
    (a block is cut where another reader's block ends first: a member read whole yields one block)."""
    pending = [None] * len(readers)
    while True:
        pending = [p if p is not None and len(p) else next(r, None) for p, r in zip(pending, readers)]
        if any(p is None for p in pending):
            return
        m = min(len(p) for p in pending)
        yield [p[:m] for p in pending]
        pending = [p[m:] for p in pending]


class _FileStream:
    """`load_dataset(path, ...)` of one `.npz` file as row writes computed a block at a time.

    `fields` is the result's layout, {name: (dtype, shape)} in load_dataset's key order, known from the members' headers
    and the file's `terminals`, which is read whole (one byte per row in OGBench files).  `producers(block_rows)` gives one
    generator per member (and one for the terminal fields); each yields (first row, {field: rows}) writes that together
    cover every row of every field once.  Compact layout: rows stay where they are.  Regular layout: the kept rows of a
    block go to `i - (terminals before i)`, and the same cast observation block, shifted by one row, gives the block's
    `next_observations`.  With the compact layout `flags` holds one byte of `valids > 0` per row once the terminal
    producer has run.

    `relabellings` (make_datasets' for a relabelled name) add their derived fields after load_dataset's, as make_datasets
    does.  One producer reads the info members they need in blocks of the same rows, lays them out like any member and
    yields the derived rows of each block, and the info rows too when `add_info` keeps them; without `add_info` no info
    field is kept and an info member nothing is derived from is not read.
    """

    def __init__(self, path, ob_dtype=np.float32, action_dtype=np.float32, compact_dataset=False, add_info=False,
                 relabellings=()):
        self.path, self.compact = str(path), compact_dataset
        self.relabellings = list(relabellings)
        self.sources = [k for k in _INFO_KEYS if any(k in r.members for r in self.relabellings)]
        with zipfile.ZipFile(self.path) as zf:
            present = set(zf.namelist())
            keys = ['observations', 'actions', 'terminals'] + [k for k in _INFO_KEYS if add_info and f'{k}.npy' in present]
            heads = {}
            for k in keys + [k for k in self.sources if k not in keys]:
                with _open_member(zf, self.path, k) as f:
                    heads[k] = _read_npy_header(f, self.path, k)
        self.terminals = _read_member(self.path, 'terminals')
        n = len(self.terminals)
        for k, (shape, _, _) in heads.items():
            if len(shape) < 1 or shape[0] != n:
                raise ValueError(f'{self.path}: member {k!r} of shape {shape} does not have the {n} rows of terminals')
        self.casts = {'observations': np.dtype(ob_dtype), 'actions': np.dtype(action_dtype)}
        self.members = [k for k in keys if k != 'terminals' and k not in self.sources]
        self.source_row_bytes = sum(heads[k][1].itemsize * int(np.prod(heads[k][0][1:], dtype=np.int64)) for k in self.sources)
        obs_row = heads['observations'][0][1:]
        if compact_dataset:
            self.keep, rows, next_rows = None, n, None
            self.flags = np.zeros(n, np.uint8)
        else:
            self.keep = (1.0 - self.terminals.astype(np.float32)).astype(bool)      # load_dataset's ob_mask
            rows, next_rows = int(np.count_nonzero(self.keep)), int(np.count_nonzero(self.keep[:-1]))
            self.flags = None
        self.fields = {'observations': (self.casts['observations'], (rows, *obs_row)),
                       'actions': (self.casts['actions'], (rows, *heads['actions'][0][1:])),
                       'terminals': (np.dtype(np.float32), (rows,))}
        self.fields.update({k: (heads[k][1], (rows, *heads[k][0][1:])) for k in keys[3:]})
        if compact_dataset:
            self.fields['valids'] = (np.dtype(np.float32), (rows,))
        else:
            self.fields['next_observations'] = (self.casts['observations'], (next_rows, *obs_row))
        # the derived fields' dtypes and row shapes: the relabellings applied to no rows of the members
        empty = {k: np.zeros((0, *heads[k][0][1:]), heads[k][1]) for k in self.sources}
        for relabelling in self.relabellings:
            self.fields.update({k: (a.dtype, (rows, *a.shape[1:])) for k, a in relabelling.rows(empty).items()})

    def producers(self, block_rows: Optional[int] = None):
        derived = [self._derived_writes(block_rows)] if self.relabellings else []
        return [self._member_writes(k, block_rows) for k in self.members] + derived + [self._terminal_writes(block_rows)]

    def _derived_writes(self, block_rows):
        """The relabellings' fields (and the info fields they read, when kept), from the info members read in blocks of
        the same rows and laid out as _member_writes lays out a member."""
        rows = block_rows or max(1, _BLOCK_BYTES // max(1, self.source_row_bytes))
        r0 = dest = 0
        with contextlib.ExitStack() as stack:
            readers = [stack.enter_context(contextlib.closing(read_member_blocks(self.path, k, rows))) for k in self.sources]
            for blocks in _lockstep(readers):
                r1 = r0 + len(blocks[0])
                info = dict(zip(self.sources, blocks))
                if not self.compact:
                    keep = self.keep[r0:r1]
                    info = {k: b[keep] for k, b in info.items()}
                out = {k: b for k, b in info.items() if k in self.fields}
                for relabelling in self.relabellings:
                    out.update(relabelling.rows(info))
                yield (r0 if self.compact else dest), out
                dest += len(next(iter(out.values())))
                r0 = r1

    def _member_writes(self, key, block_rows):
        cast = self.casts.get(key)
        r0 = dest = 0
        for block in read_member_blocks(self.path, key, block_rows):
            r1 = r0 + len(block)
            if cast is not None:
                block = block.astype(cast, copy=False)
            if self.compact:
                yield r0, {key: block}
            else:
                keep = self.keep[r0:r1]
                yield dest, {key: block[keep]}
                if key == 'observations':
                    # next_observations = observations[next_ob_mask], next_ob_mask[j] = ob_mask[j - 1] (False at j = 0)
                    follows_kept = self.keep[max(r0 - 1, 0):r1 - 1]
                    if r0 == 0:
                        follows_kept = np.concatenate([[False], follows_kept])
                    yield dest - int(r0 > 0 and self.keep[r0 - 1]), {'next_observations': block[follows_kept]}
                dest += int(np.count_nonzero(keep))
            r0 = r1

    def _terminal_writes(self, block_rows):
        n = len(self.terminals)
        rows = block_rows or _BLOCK_BYTES // 32       # (float64 temporaries of load_dataset's expressions)
        dest = 0
        for r0 in range(0, n, rows):
            r1 = min(n, r0 + rows)
            t, follows = _terminal_rows(self.terminals, r0, r1)
            if self.compact:
                valids = 1.0 - t
                self.flags[r0:r1] = valids > 0
                yield r0, {'terminals': np.minimum(t + follows, 1.0).astype(np.float32), 'valids': valids}
            else:
                keep = self.keep[r0:r1]
                yield dest, {'terminals': follows[keep].astype(np.float32)}
                dest += int(np.count_nonzero(keep))

    def write(self, nds: _NativeDataset, row0: int, names) -> None:
        """Run the producers, one thread each, and write their rows from this thread to rows `row0 + r` of `nds`, whose
        fields are `names` in order (ogb_dataset_write_rows is synchronous and takes one caller at a time)."""
        _pump(self.producers(), lambda r, arrays: _write_rows(nds, names, row0 + r, arrays))


def _write_rows(nds: _NativeDataset, names, row0: int, arrays) -> None:
    """ogb_dataset_write_rows of `arrays` ({field: rows}, some of the table's fields `names`, in any order) at rows
    [row0, row0 + n); the other fields are left as they are."""
    n = len(next(iter(arrays.values())))
    if n == 0:
        return
    arrays = {k: np.ascontiguousarray(a) for k, a in arrays.items()}
    ptrs = (C.c_void_p * len(names))()
    for i, k in enumerate(names):
        if k in arrays:
            ptrs[i] = arrays[k].ctypes.data
    _native.check(_native.lib().ogb_dataset_write_rows(nds.ptr, row0, n, ptrs, len(names)))


def _pump(producers, consume):
    """Run each generator on a thread of its own and call consume(*item) for every item on this thread, in arrival order.
    A bounded queue of two items per producer sits between them; an exception on either side stops every thread and is
    raised here."""
    q: queue.Queue = queue.Queue(maxsize=2 * len(producers))
    stop = threading.Event()
    done = object()

    def put(item) -> bool:
        while not stop.is_set():
            try:
                q.put(item, timeout=0.1)
                return True
            except queue.Full:
                pass
        return False

    def work(gen):
        try:
            with contextlib.closing(gen):
                for item in gen:
                    if not put(item):
                        return
            put(done)
        except BaseException as exc:  # raised on the consuming thread
            put(exc)

    threads = [threading.Thread(target=work, args=(g,), daemon=True) for g in producers]
    for t in threads:
        t.start()
    try:
        finished = 0
        while finished < len(threads):
            item = q.get()
            if item is done:
                finished += 1
            elif isinstance(item, BaseException):
                raise item
            else:
                consume(*item)
    finally:
        stop.set()
        for t in threads:
            t.join()


def upload_dataset(dataset_path, ob_dtype=np.float32, action_dtype=np.float32, compact_dataset=False, add_info=False,
                   device: int = 0) -> ResidentDataset:
    """`Dataset.create(**load_dataset(dataset_path, ...))`, streamed: the file's members are inflated a block at a time, one
    thread per member, cast and laid out per block, and written into HBM, so host memory holds a few blocks per member
    and a few bytes per row instead of the whole file.  The dataset samples byte for byte what the host-loaded one does;
    it keeps no host copy of its fields (ResidentDataset)."""
    return _upload(_FileStream(dataset_path, ob_dtype, action_dtype, compact_dataset, add_info), device)


def upload_datasets(dataset_name, dataset_dir='~/.ogbench/data', dataset_path=None, compact_dataset=False, add_info=False,
                    env=None, num_cubes=None, num_buttons=None, device: int = 0):
    """`make_datasets(...)` in HBM: (train, val) as ResidentDatasets, each sampling byte for byte what
    `Dataset.create(**make_datasets(...)[i])` samples, for plain, '-oraclerep-' and 'singletask' names alike.  Each split
    is streamed as upload_dataset streams a file; the relabelled fields are computed per block of `qpos` /
    `button_states` rows with make_datasets' own expressions, so host memory holds a few blocks per member whatever the
    file's size.  The name and the files are checked before any file is read, with make_datasets' errors; a single-task
    `env` is reset once per split, as make_datasets resets it."""
    return tuple(_upload(stream, device) for stream in _split_streams(dataset_name, dataset_dir, dataset_path, compact_dataset,
                                                                       add_info, env, num_cubes, num_buttons))


def _split_streams(dataset_name, dataset_dir, dataset_path, compact_dataset, add_info, env, num_cubes, num_buttons):
    """make_datasets' (train, val) as a generator of _FileStreams.  The name and the files are checked at the call; a split's
    relabellings are resolved when its stream is made, after the previous split has been consumed."""
    name = _parse_dataset_name(dataset_name, add_info, env)
    paths = name.paths(dataset_dir, dataset_path)
    return (name.stream(path, compact_dataset, add_info, env, num_cubes, num_buttons) for path in paths)


def _upload(stream: _FileStream, device: int) -> ResidentDataset:
    rows = {k: shape[0] for k, (_, shape) in stream.fields.items()}
    if len(set(rows.values())) != 1:      # a regular layout whose last row is not terminal: Dataset.create refuses it too
        raise ValueError(f'{stream.path}: fields of different lengths {rows}')
    nds = _NativeDataset.empty({k: _ZeroField(shape, dtype) for k, (dtype, shape) in stream.fields.items()}, device)
    stream.write(nds, 0, list(stream.fields))
    n = rows['terminals']
    _native.check(_native.lib().ogb_dataset_seal(nds.ptr, n))
    return ResidentDataset(nds, list(stream.fields), False, stream.flags)


class ResidentShards:
    """Every shard of a dataset directory, uploaded once into one HBM table.

        shards = ResidentShards(list_shards(path))
        shards.dataset            # Dataset over every row, shards in path order: the concatenated dataset
        shards[i], shards[path]   # Dataset of one shard: a view of the table, equal to Dataset.create(**load(path))
        shards.bounds             # [(row0, n_rows)] per shard

    By default each file is streamed into the table block by block as upload_dataset does, with the result of
    load_dataset(p, compact_dataset=True), so host memory holds a few 8 MB blocks per member and a few bytes per row.
    With `dataset_name` (and `env` / `num_cubes` / `num_buttons` as make_datasets takes them) each file is streamed the
    same way with the result of `make_datasets(dataset_name, dataset_path=p, compact_dataset=True, ...)[0]`: that name's
    dtypes, and for '-oraclerep-' and 'singletask' names its relabelled fields, computed per block (a single-task `env`
    is reset once per shard).  `load`, a per-file host loader, is the alternative for anything else: it is called on one
    shard at a time, and each shard is written and freed before the next is loaded, so host memory peaks at one shard
    plus a pinned staging buffer.  `load` and `dataset_name` do not go together.  The capacity comes from the files'
    headers.  Every shard must load with shard 0's fields, dtypes and row shapes.

    A view keeps the reference's shard-local semantics (goals, trajectory ends and next observations stay inside the
    shard) and a swap costs no upload; sampling `dataset` draws across every shard instead.  Shards end on trajectory
    boundaries, so each rank of a multi-GPU run can build its own ResidentShards over its subset of the paths.
    """

    def __init__(self, paths, load: Optional[Callable[[str], dict]] = None, device: int = 0, *, dataset_name=None, env=None,
                 num_cubes=None, num_buttons=None):
        open_stream = None
        if dataset_name is not None:
            if load is not None:
                raise ValueError('ResidentShards takes load= or dataset_name=, not both')
            open_stream = functools.partial(_parse_dataset_name(dataset_name, env=env).stream, compact_dataset=True,
                                            add_info=False, env=env, num_cubes=num_cubes, num_buttons=num_buttons)
        self.paths = [str(p) for p in paths]
        lib = _native.lib()
        nds, keys, nested, valids, self.bounds = None, None, False, [], []
        for shard in iter_shards(self.paths, load, open_stream):
            if nds is None:
                keys, nested = shard.keys, shard.nested
                nds = _NativeDataset.empty({k: _ZeroField((shard.capacity, *s), d) for k, (d, s) in shard.schema.items()}, device)
            if shard.stream is not None:
                shard.stream.write(nds, shard.row0, list(shard.schema))
                valids.append(shard.stream.flags)
            else:
                _write_rows(nds, list(shard.schema), shard.row0, shard.fields)
                if 'valids' in shard.fields:
                    valids.append((shard.fields['valids'] > 0).astype(np.uint8))
            self.bounds.append((shard.row0, shard.n_rows))
            del shard                                 # this shard's host arrays go before the next one is loaded
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
    __slots__ = ('path', 'row0', 'n_rows', 'capacity', 'keys', 'nested', 'schema', 'fields', 'stream')


def iter_shards(paths, load: Optional[Callable[[str], dict]] = None, open_stream: Optional[Callable[[str], _FileStream]] = None):
    """The host half of ResidentShards: load the shards one at a time, in order, and yield each as a record with its
    first row in the concatenation (`row0`), its row count, its flattened fields and the schema -- {name: (dtype, row
    shape)} -- that shard 0 fixed; `capacity` is the rows the files' headers declare in all.  Without `load`, a record
    holds no fields (`fields` is None) but the stream that writes the shard block by block (`stream`, None when `load`
    is given): `open_stream(path)`, by default load_dataset(path, compact_dataset=True)'s.  A shard whose fields, dtypes
    or row shapes differ from shard 0's, or that loads more rows than its header declares, raises ValueError naming it."""
    paths = [str(p) for p in paths]
    if not paths:
        raise ValueError('no shards given')
    declared = [shard_rows(p) for p in paths]
    schema, row0 = None, 0
    for path, cap in zip(paths, declared):
        if load is None:
            stream = open_stream(path) if open_stream else _FileStream(path, compact_dataset=True)
            fields = None
            shape = {k: (d, s[1:]) for k, (d, s) in stream.fields.items()}
            names, is_nested = list(stream.fields), False
            lengths = {s[0] for _, s in stream.fields.values()}
        else:
            stream, tree = None, load(path)
            fields = _flatten(tree)
            shape = {k: (np.asarray(v).dtype, np.asarray(v).shape[1:]) for k, v in fields.items()}
            names, is_nested = list(tree), any(isinstance(v, Mapping) for v in tree.values())
            lengths = {len(v) for v in fields.values()}
            del tree
        if schema is None:
            schema, keys, nested = shape, names, is_nested
        elif shape != schema:
            raise ValueError(f'{path}: fields {_describe(shape)} differ from those of {paths[0]}: {_describe(schema)}')
        if len(lengths) != 1:
            raise ValueError(f'{path}: fields of different lengths {sorted(lengths)}')
        n = lengths.pop()
        if n > cap:
            raise ValueError(f'{path}: {n} rows loaded, the file declares {cap}')
        shard = _Shard()
        shard.path, shard.row0, shard.n_rows, shard.capacity = path, row0, n, sum(declared)
        shard.keys, shard.nested, shard.schema, shard.fields, shard.stream = keys, nested, schema, fields, stream
        del fields, stream
        yield shard
        del shard                                     # (the caller's reference is the last one before the next load)
        row0 += n


def _describe(schema) -> str:
    return ', '.join(f'{k}: {d}{tuple(s)}' for k, (d, s) in schema.items())

"""Streaming relabelled datasets into HBM ('-oraclerep-' and 'singletask' names): loader.upload_datasets and
ResidentShards(paths, dataset_name=...).

- the stream's per-block relabelling writes every row of make_datasets' result once and equals it, for every family of
  both relabellings, at any block size, in the compact and the regular layout, with and without the info fields;
- the name helper resolves make_datasets' files and dtypes; a single-task env is reset once per split; the errors of
  make_datasets are raised before any file is read or any device memory is taken;
- on the GPU, each split of upload_datasets equals Dataset.create(**make_datasets(...)[i]) row for row and batch for
  batch, for the committed raw pairs and for synthetic files of many blocks; ResidentShards(dataset_name=...) equals
  ResidentShards(load=make_datasets ...); host memory stays at a few blocks per member plus a few bytes per row.
"""

import os
import tracemalloc

import numpy as np
import pytest

from ogbench_b200 import loader
from tests.golden.make_golden import cfg, ragged
from tests.golden.make_golden_loader import MAKE_CASES, ORACLE_ENVS, SINGLETASK_ENVS, singletask_env, singletask_inputs
from tests.golden_util import assert_batches_identical
from tests.test_gpu_stream_load import assemble, flat_host

RAW_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'loader_raw')


def singletask_name(env_name):
    """The dataset name whose environment is `env_name`: the dataset type goes before 'singletask'."""
    splits = env_name.split('-')
    pos = splits.index('singletask')
    kind = 'navigate' if ('maze' in env_name or 'soccer' in env_name) else 'play'
    return '-'.join(splits[:pos] + [kind] + splits[pos:])


# (dataset name, make_datasets' relabelling arguments)
ORACLE_CASES = [(name, dict(num_cubes=cubes, num_buttons=buttons)) for name, cubes, buttons in ORACLE_ENVS]
TASK_CASES = [(singletask_name(e), dict(env=singletask_env(e))) for e in SINGLETASK_ENVS]
CASES = ORACLE_CASES + TASK_CASES


def relabel_file(path, env, n=29, seed=0, compressed=True):
    """`n` rows with qpos[:, 40] / button_states[:, 9] that meet all, some or none of `env`'s sub-goals; with 7-row blocks
    the terminals fall on a block's first row (0, 7), last row (13, 20) and inner rows (3, 17, 25)."""
    rng = np.random.default_rng(seed)
    terminals = np.zeros(n, bool)
    terminals[[0, 3, 7, 13, 17, 20, 25, n - 1]] = True
    (np.savez_compressed if compressed else np.savez)(
        path, observations=rng.standard_normal((n, 3)), actions=rng.uniform(-1, 1, (n, 2)), terminals=terminals,
        qvel=rng.standard_normal((n, 4)), **singletask_inputs(env, seed=seed, n=n))


def relabel_pair(directory, name, env, **kw):
    path = os.path.join(str(directory), file_stem_of(name) + '.npz')
    relabel_file(path, env, **kw)
    relabel_file(path.replace('.npz', '-val.npz'), env, n=31, seed=kw.get('seed', 0) + 1)
    return path


def file_stem_of(name):
    return loader._parse_dataset_name(name, env=singletask_env('x')).file_stem


# ------------------------------------------------ CPU: the per-block relabelling ------------------------------------------------
def assert_streams_equal(path, name, kw, label):
    for compact in (False, True):
        for add_info in (False, True):
            want = loader.make_datasets(name, dataset_path=path, compact_dataset=compact, add_info=add_info, **kw)
            for block_rows in (1, 7, None):
                streams = loader._split_streams(name, None, path, compact, add_info, kw.get('env'), kw.get('num_cubes'),
                                                kw.get('num_buttons'))
                for split, w, stream in zip(('train', 'val'), want, streams):
                    where = (label, split, compact, add_info, block_rows)
                    assert list(stream.fields) == list(w), (where, list(stream.fields), list(w))
                    got = assemble(stream, block_rows)
                    for k, v in w.items():
                        assert got[k].dtype == v.dtype and got[k].shape == v.shape and np.array_equal(got[k], v), (where, k)
                    if compact:
                        assert np.array_equal(stream.flags, (w['valids'] > 0).astype(np.uint8)), where


@pytest.mark.parametrize('name,kw', CASES, ids=[c[0] for c in CASES])
def test_per_block_relabelling_equals_make_datasets(tmp_path, name, kw):
    path = relabel_pair(tmp_path, name, kw.get('env') or singletask_env('x'))
    assert_streams_equal(path, name, kw, name)
    if 'singletask' in name:                  # both outcomes occur in the file
        masks = loader.make_datasets(name, dataset_path=path, compact_dataset=True, **kw)[0]['masks']
        assert 0 < (masks == 0).sum() < len(masks), name


def test_per_block_relabelling_of_the_raw_files():
    cases = [(n, dict(num_cubes=c)) for n, _, c, _ in MAKE_CASES if 'oraclerep' in n]
    cases.append(('antmaze-large-navigate-singletask-task1-v0', dict(env=singletask_env('antmaze-large-singletask-task1-v0'))))
    for name, kw in cases:
        assert_streams_equal(os.path.join(RAW_DIR, file_stem_of(name) + '.npz'), name, kw, name)


def test_member_read_whole_is_cut_in_lockstep(tmp_path):
    """A Fortran-order qpos is read in one block: button_states' blocks cut it."""
    from tests.test_gpu_stream_load import write_npz

    env = singletask_env('x')
    src = str(tmp_path / 'c.npz')
    relabel_file(src, env)
    p = str(tmp_path / 'scene-play-v0.npz')
    write_npz(p, dict(np.load(src)), fortran=('qpos',))
    write_npz(p.replace('.npz', '-val.npz'), dict(np.load(src)))
    assert_streams_equal(p, 'scene-play-oraclerep-v0', dict(num_cubes=1, num_buttons=2), 'fortran qpos')


EXPECTED_NAMES = {  # dataset name: (env name, file stem, ob dtype, action dtype) -- ogbench/utils.py:164-203
    'antmaze-large-navigate-v0': ('antmaze-large-v0', 'antmaze-large-navigate-v0', np.float32, np.float32),
    'visual-cube-single-play-v0': ('visual-cube-single-v0', 'visual-cube-single-play-v0', np.uint8, np.float32),
    'powderworld-easy-play-v0': ('powderworld-easy-v0', 'powderworld-easy-play-v0', np.uint8, np.int32),
    'cube-double-play-oraclerep-v0': ('cube-double-v0', 'cube-double-play-v0', np.float32, np.float32),
    'pointmaze-medium-navigate-oraclerep-v0': ('pointmaze-medium-v0', 'pointmaze-medium-navigate-v0', np.float32, np.float32),
    'antmaze-large-navigate-singletask-task1-v0': ('antmaze-large-singletask-task1-v0', 'antmaze-large-navigate-v0', np.float32,
                                                   np.float32),
}


def test_name_helper_resolves_make_datasets_files_and_dtypes():
    assert set(EXPECTED_NAMES) >= {n for n, *_ in MAKE_CASES}
    for dataset_name, (env_name, stem, ob, act) in EXPECTED_NAMES.items():
        relabelled = 'oraclerep' in dataset_name or 'singletask' in dataset_name
        for add_info in (False, True):
            name = loader._parse_dataset_name(dataset_name, add_info, env=singletask_env('x'))
            assert (name.env_name, name.file_stem, name.ob_dtype, name.action_dtype) == (env_name, stem, ob, act), dataset_name
            assert name.load_info == (add_info or relabelled), dataset_name
            assert (name.singletask, name.oraclerep) == ('singletask' in dataset_name, 'oraclerep' in dataset_name)
            want = (os.path.join(RAW_DIR, stem + '.npz'), os.path.join(RAW_DIR, stem + '-val.npz'))
            assert name.paths(RAW_DIR) == want and name.paths(dataset_path=want[0]) == want, dataset_name
    home = loader._parse_dataset_name('antmaze-large-navigate-v0')
    with pytest.raises(FileNotFoundError, match=os.path.expanduser('~/missing-ogb-dir') + '/antmaze-large-navigate-v0.npz'):
        home.paths('~/missing-ogb-dir')


def counting_env(name):
    env = singletask_env(name)
    env.resets = 0

    def reset():
        env.resets += 1
    env.reset = reset
    return env


def test_singletask_env_is_reset_once_per_split():
    path = os.path.join(RAW_DIR, 'antmaze-large-navigate-v0.npz')
    name = 'antmaze-large-navigate-singletask-task1-v0'
    env = counting_env('antmaze-large-singletask-task1-v0')
    loader.make_datasets(name, dataset_path=path, env=env)
    assert env.resets == 2
    env = counting_env('antmaze-large-singletask-task1-v0')
    streams = loader._split_streams(name, None, path, True, False, env, None, None)
    assert env.resets == 0
    for i, stream in enumerate(streams):
        assert env.resets == i + 1                # a split's task is read when its stream is made
        assemble(stream, None)
    assert env.resets == 2


# ------------------------------------------------ errors, raised before a file is read or a table is allocated ---------------------
def test_errors_are_make_datasets_errors(tmp_path, monkeypatch):
    def no_device(*a, **k):
        raise AssertionError('device memory taken before the error')
    monkeypatch.setattr(loader._NativeDataset, 'empty', no_device)
    raw = os.path.join(RAW_DIR, 'antmaze-large-navigate-v0.npz')
    for call in (loader.make_datasets, loader.upload_datasets):
        with pytest.raises(ValueError, match='singletask'):
            call('cube-single-play-singletask-v0', dataset_path='x.npz')
        with pytest.raises(FileNotFoundError):
            call('antmaze-large-navigate-v0', dataset_dir=RAW_DIR + '/missing')
        with pytest.raises(FileNotFoundError):
            call('antmaze-large-navigate-singletask-task1-v0', dataset_dir=RAW_DIR + '/missing', env=singletask_env('x'))
        env = singletask_env('x')
        env.unwrapped._reward_task_id = None
        with pytest.raises(AssertionError, match='single-task'):
            call('antmaze-large-navigate-singletask-task1-v0', dataset_path=raw, env=env)
    p = relabel_pair(tmp_path, 'powderworld-easy-play-oraclerep-v0', singletask_env('x'))
    q = str(tmp_path / 'cube-double-play-v0.npz')
    for suffix in ('', '-val'):
        np.savez(q.replace('.npz', suffix + '.npz'), observations=np.zeros((4, 3)), actions=np.zeros((4, 2)),
                 terminals=np.ones(4, bool), button_states=np.zeros((4, 9)))
    for call in (loader.make_datasets, loader.upload_datasets):
        with pytest.raises(ValueError, match='Unsupported environment'):
            call('powderworld-easy-play-oraclerep-v0', dataset_path=p)
        with pytest.raises(ValueError, match='Unsupported environment'):
            call('powderworld-easy-play-singletask-v0', dataset_path=p, env=singletask_env('x'))
        with pytest.raises(KeyError, match='qpos'):
            call('cube-double-play-oraclerep-v0', dataset_path=q, num_cubes=2)
        with pytest.raises(KeyError, match='qpos'):
            call('cube-double-play-singletask-task1-v0', dataset_path=q, env=singletask_env('x'))
    with pytest.raises(ValueError, match='not both'):
        loader.ResidentShards([p], load=loader.load_dataset, dataset_name='powderworld-easy-play-v0')


# ------------------------------------------------ GPU: upload_datasets against the host path ------------------------------------------------
def assert_same_dataset(got, ref, label, batch=64):
    from ogbench_b200 import GCDataset

    assert got.size == ref.size and list(got) == list(ref), (label, list(got), list(ref))
    g, r = getattr(got, 'valid_idxs', None), getattr(ref, 'valid_idxs', None)
    assert (g is None) == (r is None) and (g is None or np.array_equal(g, r)), label
    rows = np.arange(ref.size)
    assert_batches_identical(flat_host(got.get_subset(rows)), flat_host(ref.get_subset(rows)), label=f'{label} subset:')
    a, b = GCDataset(got, cfg(), seed=7), GCDataset(ref, cfg(), seed=7)
    for it in range(2):
        assert_batches_identical(flat_host(a.sample(batch)), flat_host(b.sample(batch)), label=f'{label} philox {it}:')
    a, b = GCDataset(got, cfg(), rng='numpy'), GCDataset(ref, cfg(), rng='numpy')
    for it in range(2):
        np.random.seed(30 + it)
        x = flat_host(a.sample(batch))
        np.random.seed(30 + it)
        assert_batches_identical(x, flat_host(b.sample(batch)), label=f'{label} numpy {it}:')


def assert_uploads_like_make_datasets(name, label, batch=64, **kw):
    from ogbench_b200 import Dataset

    want = loader.make_datasets(name, **kw)
    got = loader.upload_datasets(name, **kw)
    assert len(got) == 2
    for split, g, w in zip(('train', 'val'), got, want):
        assert_same_dataset(g, Dataset.create(**w), f'{label} {split}', batch)


@pytest.mark.gpu
def test_raw_pairs_upload_like_make_datasets():
    cases = [(n, dict(num_cubes=c)) for n, _, c, _ in MAKE_CASES if 'oraclerep' in n]
    cases.append(('antmaze-large-navigate-singletask-task1-v0', dict(env=counting_env('antmaze-large-singletask-task1-v0'))))
    for name, kw in cases:
        for compact in (False, True):
            for add_info in (False, True):
                assert_uploads_like_make_datasets(name, f'{name} c{int(compact)} i{int(add_info)}',
                                                  dataset_path=os.path.join(RAW_DIR, file_stem_of(name) + '.npz'),
                                                  compact_dataset=compact, add_info=add_info, **kw)
    assert cases[-1][1]['env'].resets == 2 * 4 * 2      # once per split, for make_datasets and for upload_datasets


TASK_ENV = singletask_env('synthetic')                   # the task every synthetic file meets in some rows
FAMILIES = [('cube-double-play-oraclerep-v0', dict(num_cubes=2)), ('scene-play-oraclerep-v0', dict(num_cubes=1, num_buttons=2)),
            ('puzzle-3x3-play-oraclerep-v0', {}), ('antmaze-large-navigate-oraclerep-v0', {}),
            ('cube-double-play-singletask-task2-v0', dict(env=TASK_ENV)), ('scene-play-singletask-task3-v0', dict(env=TASK_ENV)),
            ('puzzle-3x3-play-singletask-v0', dict(env=TASK_ENV)), ('antmaze-large-navigate-singletask-task1-v0', dict(env=TASK_ENV))]


def task_info(rng, n):
    """qpos[:, 40] float64 / button_states[:, 9]: a sixth of the rows meets every sub-goal of TASK_ENV, another sixth some."""
    task = TASK_ENV.unwrapped
    qpos, buttons = rng.standard_normal((n, 40)), rng.integers(0, 2, (n, 9))
    hit = rng.random(n) < 1 / 3
    full = hit & (rng.random(n) < 0.5)
    qpos[hit, :2] = task.cur_goal_xy + rng.uniform(-0.3, 0.3, (int(hit.sum()), 2))
    for c in range(task._num_cubes):
        rows = full if c else hit
        qpos[rows, 14 + 7 * c:17 + 7 * c] = task._data.mocap_pos[c] + rng.uniform(-0.015, 0.015, (int(rows.sum()), 3))
    buttons[full] = task._target_button_states
    drawer = 14 + 7 * task._num_cubes + task._num_buttons
    qpos[full, drawer], qpos[full, drawer + 1] = task._target_drawer_pos + 0.02, task._target_window_pos - 0.03
    return dict(qpos=qpos, button_states=buttons)


def synthetic_pair(path, kind, compressed, seed):
    """Train and validation files of the C5 row (55 float32) or of visual-cube frames (64x64x3 uint8), 5 float32 actions,
    qpos and button_states; the training file spans several 8 MB blocks of observations (and of qpos for 'state')."""
    rng = np.random.default_rng(seed)
    for suffix, n_traj in (('', 300 if kind == 'state' else 30), ('-val', 4)):
        lengths = ragged(seed, n_traj, 200, 1200) if kind == 'state' else ragged(seed, n_traj, 20, 250)
        n = int(lengths.sum())
        if kind == 'state':
            obs = rng.standard_normal((n, 55), dtype=np.float32)
        else:
            base = rng.integers(0, 256, (64, 64, 3), dtype=np.uint8)
            obs = (base[None] + (np.arange(n, dtype=np.uint32) * 7 % 251)[:, None, None, None]).astype(np.uint8)
            obs[:, ::9, ::5] = rng.integers(0, 256, obs[:, ::9, ::5].shape, dtype=np.uint8)
        terminals = np.zeros(n, bool)
        terminals[np.cumsum(lengths) - 1] = True
        (np.savez_compressed if compressed else np.savez)(
            path.replace('.npz', suffix + '.npz'), observations=obs, actions=rng.uniform(-1, 1, (n, 5)).astype(np.float32),
            terminals=terminals, qvel=rng.standard_normal((n, 4)), **task_info(rng, n))
        if not suffix:
            train_rows, obs_bytes = n, obs.nbytes
    return train_rows, obs_bytes


@pytest.fixture(scope='module')
def synthetic(tmp_path_factory):
    d = tmp_path_factory.mktemp('relabel')
    out = {}
    for kind, compressed in (('state', True), ('state', False), ('frames', True)):
        p = str(d / f'{kind}{int(compressed)}.npz')
        out[kind, compressed] = p, *synthetic_pair(p, kind, compressed, seed=21)
    return out


@pytest.mark.gpu
@pytest.mark.parametrize('kind,compressed', [('state', True), ('state', False), ('frames', True)])
def test_many_block_files_upload_like_make_datasets(synthetic, kind, compressed):
    path, n, obs_bytes = synthetic[kind, compressed]
    assert obs_bytes > 4 * (8 << 20)                                  # several default blocks of observations
    if kind == 'state':
        assert n * (40 * 8 + 9 * 8) > 2 * (8 << 20)                   # and of qpos / button_states
    layouts = [(True, False), (False, True)] if compressed else [(True, True)]
    for name, kw in FAMILIES:
        name = name if kind == 'state' else 'visual-' + name
        for compact, add_info in layouts:
            assert_uploads_like_make_datasets(name, f'{kind} {name} c{int(compact)} i{int(add_info)}',
                                              batch=256 if kind == 'state' else 32, dataset_path=path,
                                              compact_dataset=compact, add_info=add_info, **kw)


@pytest.mark.gpu
def test_small_blocks_upload_like_make_datasets(synthetic, monkeypatch):
    """Blocks of a few hundred rows: every trajectory crosses block ends, in every member."""
    path = synthetic['state', True][0]
    monkeypatch.setattr(loader, '_BLOCK_BYTES', 64 << 10)
    for name, kw in (FAMILIES[1], FAMILIES[5]):
        for compact in (False, True):
            assert_uploads_like_make_datasets(name, f'{name} c{int(compact)}', batch=256, dataset_path=path,
                                              compact_dataset=compact, add_info=True, **kw)


@pytest.mark.gpu
def test_resident_shards_by_name_equal_make_datasets_shards(tmp_path):
    from ogbench_b200 import GCDataset

    paths = []
    for i in range(3):
        p = str(tmp_path / f'shard{i}.npz')
        synthetic_pair(p, 'state', bool(i % 2), seed=40 + i)
        paths.append(p)
    for name, kw in (FAMILIES[1], FAMILIES[4]):
        streamed = loader.ResidentShards(paths, dataset_name=name, **kw)
        loaded = loader.ResidentShards(paths, load=lambda p: loader.make_datasets(name, dataset_path=p, compact_dataset=True, **kw)[0])
        assert streamed.bounds == loaded.bounds and list(streamed.dataset) == list(loaded.dataset), name
        views = [(f'shard {i}', streamed[i], loaded[i]) for i in range(len(paths))]
        for label, a, b in [('whole', streamed.dataset, loaded.dataset)] + views:
            label = f'{name} {label}'
            rows = np.arange(a.size)
            assert_batches_identical(flat_host(a.get_subset(rows)), flat_host(b.get_subset(rows)), label=f'{label} subset:')
            assert np.array_equal(a.valid_idxs, b.valid_idxs), label
            x, y = GCDataset(a, cfg(), seed=3), GCDataset(b, cfg(), seed=3)
            assert_batches_identical(flat_host(x.sample(512)), flat_host(y.sample(512)), label=f'{label} philox:')


@pytest.mark.gpu
def test_host_memory_stays_at_a_few_blocks(tmp_path):
    n = 2_000_000
    rng = np.random.default_rng(0)
    terminals = np.zeros(n, bool)
    terminals[np.arange(1000, n, 1001)] = True
    terminals[-1] = True
    p = str(tmp_path / 'scene-play-v0.npz')
    np.savez(p, observations=rng.standard_normal((n, 55), dtype=np.float32),      # 440 MB of observations
             actions=rng.uniform(-1, 1, (n, 5)).astype(np.float32), terminals=terminals, **task_info(rng, n))   # 784 MB of info
    relabel_file(p.replace('.npz', '-val.npz'), TASK_ENV)
    file_bytes = os.path.getsize(p)
    producers = 4                                   # observations, actions, the relabelled fields and the terminal fields
    bound = producers * 6 * (8 << 20) + 8 * n       # six 8 MB blocks per producer (queued and in flight), 8 B per row
    assert bound < file_bytes / 2
    for name, kw in (FAMILIES[1], FAMILIES[5]):
        for compact in (True, False):
            tracemalloc.start()
            try:
                train, _ = loader.upload_datasets(name, dataset_dir=str(tmp_path), compact_dataset=compact, **kw)
                _, peak = tracemalloc.get_traced_memory()
            finally:
                tracemalloc.stop()
            assert train.size == (n if compact else n - int(terminals.sum()))
            assert peak < bound, (name, compact, peak, bound)
            del train

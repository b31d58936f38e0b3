"""Resident shard directories (loader.ResidentShards): every shard uploaded once into one HBM table, each shard a view
of it, the whole table the concatenated dataset.

- the whole table samples exactly what Dataset.create(**concatenation) samples (Philox, sample_many, evaluation) and,
  under rng='numpy', what the oracle draws from the concatenated host arrays;
- every view samples exactly what Dataset.create(**load(path)) of its shard samples, through the same launches (except
  the views that lose the shadow next observation, see DESIGN.md), and the oracle's batch in validation mode;
- views clamp idx + 1 and frame stacks at their own ends, write nothing outside the keys, hand out view coordinates;
- ShardCycler over views is a drop-in for ShardCycler over file-loading samplers;
- the build is independent of the write block size, refuses what would let a sampler see a half-written table, and
  keeps host memory at about one shard.

Shards are synthetic `.npz` files with ragged trajectories, different lengths per shard and one single-trajectory shard.
"""

import ctypes as C
import gc
import os
import subprocess
import sys
import tracemalloc

import numpy as np
import pytest

from ogbench_b200 import loader
from tests.golden.make_golden import cfg, ragged, toy_fields
from tests.golden_util import assert_batches_identical

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ------------------------------------------------ synthetic shards ------------------------------------------------
def shard_fields(seed, lengths, obs_shape=(5,), obs_dtype=np.float32, oracle=None, pytree=False, mixed=False):
    f = toy_fields(seed, lengths, obs_shape, 3, obs_dtype, oracle_rep_dim=oracle)
    rng = np.random.default_rng(seed + 100)
    n = len(f['terminals'])
    if mixed:
        f.update(observations=rng.standard_normal((n, *obs_shape)), actions=rng.integers(0, 5, n).astype(np.int32),
                 step_id=np.arange(n, dtype=np.int64) + 1000 * seed, flag=rng.integers(0, 2, n).astype(bool),
                 qpos=rng.standard_normal((n, 3, 2)).astype(np.float32))
    if pytree:
        f['observations'] = {'image': f['observations'], 'state': rng.standard_normal((n, 4)).astype(np.float32)}
    return f


def save(path, fields, compressed=True):
    flat = {}
    for k, v in fields.items():
        if isinstance(v, dict):
            flat.update({f'{k}.{leaf}': a for leaf, a in v.items()})
        else:
            flat[k] = v
    (np.savez_compressed if compressed else np.savez)(path, **flat)


def load_npz(path):
    """The `load` callable of shards that hold compact fields as written (pytree leaves as 'key.leaf')."""
    z = np.load(path)
    out = {}
    for k in z.files:
        if '.' in k:
            top, leaf = k.split('.', 1)
            out.setdefault(top, {})[leaf] = z[k]
        else:
            out[k] = z[k]
    return out


def shard_lengths(seed, pixel):
    hi = 12 if pixel else 40
    return [ragged(seed, 4 if pixel else 7, 2, hi), np.array([hi + 5]), ragged(seed + 1, 5 if pixel else 11, 2, hi)]


def write_shards(tmp_path, seed=1, compressed=True, **kw):
    pixel = kw.get('obs_dtype') == np.uint8
    paths = []
    for i, lengths in enumerate(shard_lengths(seed, pixel)):
        p = str(tmp_path / f'shard{i}.npz')
        save(p, shard_fields(seed * 10 + i, lengths, **kw), compressed)
        paths.append(p)
    return paths


def concat(trees):
    out = {}
    for k in trees[0]:
        if isinstance(trees[0][k], dict):
            out[k] = {leaf: np.concatenate([t[k][leaf] for t in trees]) for leaf in trees[0][k]}
        else:
            out[k] = np.concatenate([t[k] for t in trees])
    return out


def flat_host(batch, prefix=''):
    out = {}
    for k, v in batch.items():
        if isinstance(v, dict):
            out.update(flat_host(v, f'{prefix}{k}/'))
        else:
            out[prefix + k] = np.asarray(v)
    return out


def assert_same(a, b, label):
    assert_batches_identical(flat_host(a), flat_host(b), label=label)


# ------------------------------------------------ CPU: the host walk ------------------------------------------------
@pytest.mark.parametrize('compressed', [True, False])
def test_header_rows_equal_loaded_rows(tmp_path, compressed):
    for p in write_shards(tmp_path, compressed=compressed):
        assert loader.shard_rows(p) == len(np.load(p)['terminals'])
    raw = str(tmp_path / 'raw.npz')
    save(raw, dict(observations=np.zeros((31, 2), np.float32), actions=np.zeros((31, 2), np.float32),
                   terminals=np.zeros(31, np.float32)), compressed)
    assert loader.shard_rows(raw) == 31


def test_walk_bounds_are_cumulative_row_counts(tmp_path):
    paths = write_shards(tmp_path)
    counts = [len(np.load(p)['terminals']) for p in paths]
    walked = [(s.row0, s.n_rows, s.capacity) for s in loader.iter_shards(paths, load_npz)]
    assert [r0 for r0, _, _ in walked] == list(np.cumsum([0] + counts[:-1]))
    assert [n for _, n, _ in walked] == counts
    assert all(cap == sum(counts) for _, _, cap in walked)


@pytest.mark.parametrize('change', ['field', 'dtype', 'shape'])
def test_walk_refuses_a_shard_unlike_shard_0(tmp_path, change):
    paths = write_shards(tmp_path)
    f = load_npz(paths[1])
    if change == 'field':
        f['extra'] = np.zeros(len(f['terminals']), np.float32)
    elif change == 'dtype':
        f['actions'] = f['actions'].astype(np.float64)
    else:
        f['observations'] = np.concatenate([f['observations'], f['observations'][:, :1]], axis=1)
    save(paths[1], f)
    with pytest.raises(ValueError, match='shard1.npz'):
        list(loader.iter_shards(paths, load_npz))


def test_walk_refuses_more_rows_than_the_header(tmp_path):
    paths = write_shards(tmp_path)

    def load(p):
        f = load_npz(p)
        if p == paths[2]:
            f = {k: np.concatenate([v, v[-1:]]) for k, v in f.items()}
        return f

    with pytest.raises(ValueError, match='shard2.npz'):
        list(loader.iter_shards(paths, load))


# ------------------------------------------------ GPU helpers ------------------------------------------------
def batch_info(handle):
    from ogbench_b200 import _native

    n, name, ms = C.c_int32(), C.c_char_p(), C.c_float()
    _native.check(_native.lib().ogb_batch_launches(handle.ptr, C.byref(n)))
    _native.check(_native.lib().ogb_batch_dominant_kernel(handle.ptr, C.byref(name), C.byref(ms)))
    return n.value, name.value.decode()


def make(kind, ds, config, **kw):
    from ogbench_b200 import ATCDataset, GCDataset, HGCDataset

    cls = {'gc': GCDataset, 'hgc': HGCDataset, 'atc': ATCDataset}[kind]
    return cls(ds, config, **kw)


def draw_calls(kind, a, b, B, label):
    """The same calls on two samplers with the same seed and stream: byte-identical batches."""
    if kind == 'atc':
        for it, ev in enumerate([False, False, True]):
            assert_same(a.sample(B, 2, evaluation=ev), b.sample(B, 2, evaluation=ev), f'{label} atc {it}')
        return
    for it, ev in enumerate([False, False, True]):
        assert_same(a.sample(B, evaluation=ev), b.sample(B, evaluation=ev), f'{label} sample {it}')
    assert_same(a.sample_many(3, B), b.sample_many(3, B), f'{label} sample_many')


SHAPES = [
    # (id, kinds, shard kwargs, config overrides)
    ('point2', ('gc', 'hgc', 'plain'), dict(obs_shape=(2,)), {}),                 # shadow copy, kPoint index kernel
    ('f29', ('gc', 'atc', 'plain'), dict(obs_shape=(29,)), {}),
    ('f69-hgc', ('hgc',), dict(obs_shape=(69,)), dict(subgoal_steps=7)),
    ('f600', ('gc',), dict(obs_shape=(600,)), {}),                                # split gather launches
    ('u8-64-fs3', ('gc', 'atc'), dict(obs_shape=(64, 64, 3), obs_dtype=np.uint8), dict(frame_stack=3, p_aug=0.5)),   # TMA frames
    ('u8-37-fs2', ('gc',), dict(obs_shape=(37, 16, 3), obs_dtype=np.uint8), dict(frame_stack=2, p_aug=1.0)),         # generic frames
    ('pytree', ('gc', 'plain'), dict(obs_shape=(6,), pytree=True), {}),
    ('mixed', ('gc', 'hgc'), dict(obs_shape=(9,), mixed=True), dict(subgoal_steps=5)),
    ('oracle', ('gc',), dict(obs_shape=(11,), oracle=3), {}),
]


@pytest.fixture(scope='module')
def built(tmp_path_factory):
    """ResidentShards per shape, built once for the module."""
    cache = {}

    def get(sid):
        if sid not in cache:
            kw = next(s[2] for s in SHAPES if s[0] == sid)
            paths = write_shards(tmp_path_factory.mktemp(sid), seed=3, **kw)
            cache[sid] = (paths, loader.ResidentShards(paths, load_npz))
        return cache[sid]

    return get


def config_for(kind, over):
    c = cfg(**over)
    if kind == 'hgc':
        c.setdefault('subgoal_steps', 5)
    if kind == 'atc':
        c = dict(frame_stack=over.get('frame_stack'), p_aug=over.get('p_aug'), augment_padding=4)
    return c


# ------------------------------------------------ GPU: the whole directory ------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize('sid', [s[0] for s in SHAPES])
def test_whole_directory_is_the_concatenated_dataset(built, sid):
    from ogbench_b200 import Dataset

    _, kinds, kw, over = next(s for s in SHAPES if s[0] == sid)
    paths, shards = built(sid)
    trees = [load_npz(p) for p in paths]
    whole = concat(trees)
    assert shards.bounds == [(int(r0), len(t['terminals'])) for r0, t in zip(np.cumsum([0] + [len(t['terminals']) for t in trees[:-1]]), trees)]
    assert shards.dataset.size == len(whole['terminals']) and set(shards.dataset) == set(whole)
    with pytest.raises(NotImplementedError):
        shards.dataset['observations']
    ref = Dataset.create(**whole)
    B = 37 if kw.get('obs_dtype') == np.uint8 else 301
    for kind in kinds:
        if kind == 'plain':
            for it in range(2):
                assert_same(shards.dataset.sample(B), ref.sample(B), f'{sid} plain {it}')
            continue
        c = config_for(kind, over)
        draw_calls(kind, make(kind, shards.dataset, c, seed=9, stream_id=2), make(kind, ref, c, seed=9, stream_id=2), B, f'{sid} {kind}')
        if kind == 'atc' or kw.get('pytree'):
            continue
        # rng='numpy': bit-exact against the oracle on the concatenated host arrays
        from tests.gpu_util import oracle_with_draws

        s = make(kind, shards.dataset, c, rng='numpy', output='numpy')
        for it, ev in enumerate([False, True]):
            np.random.seed(70 + it)
            _, want = oracle_with_draws(whole, c, kind, B, evaluation=ev)
            np.random.seed(70 + it)
            assert_batches_identical(s.sample(B, evaluation=ev), want, label=f'{sid} {kind} numpy {it}:')


# ------------------------------------------------ GPU: shard views ------------------------------------------------
def loses_shadow(kw, i, n_shards):
    """Views of <= 16-byte observations other than the last one gather next_observations by row (DESIGN.md)."""
    obs_bytes = int(np.prod(kw.get('obs_shape', (5,)))) * np.dtype(kw.get('obs_dtype', np.float32)).itemsize
    return obs_bytes <= 16 and not kw.get('pytree') and i < n_shards - 1


@pytest.mark.gpu
@pytest.mark.parametrize('sid', [s[0] for s in SHAPES])
def test_every_view_is_its_shard(built, sid):
    from ogbench_b200 import Dataset
    from tests.gpu_util import oracle_with_draws

    _, kinds, kw, over = next(s for s in SHAPES if s[0] == sid)
    paths, shards = built(sid)
    B = 29 if kw.get('obs_dtype') == np.uint8 else 203
    for i, path in enumerate(paths):
        fields = load_npz(path)
        view, ref = shards[i], Dataset.create(**fields)
        assert shards[path] is view and view.size == ref.size
        for kind in kinds:
            label = f'{sid} shard {i} {kind}'
            if kind == 'plain':
                assert_same(view.sample(B), ref.sample(B), label)
                assert_same(view.get_subset(np.arange(view.size)), ref.get_subset(np.arange(ref.size)), label + ' subset')
                continue
            c = config_for(kind, over)
            a, b = make(kind, view, c, seed=4, stream_id=1), make(kind, ref, c, seed=4, stream_id=1)
            draw_calls(kind, a, b, B, label)
            if kind != 'atc':
                ha, hb = a._sampler.sample_native(B), b._sampler.sample_native(B)
                assert_same(a._sampler.wrap(ha), b._sampler.wrap(hb), label + ' native')
                if not loses_shadow(kw, i, len(paths)):
                    assert batch_info(ha) == batch_info(hb), label
            if kind == 'atc' or kw.get('pytree'):
                continue
            na, nb = make(kind, view, c, rng='numpy'), make(kind, ref, c, rng='numpy')
            np.random.seed(5 + i)
            got = na.sample(B)
            np.random.seed(5 + i)
            assert_same(got, nb.sample(B), label + ' numpy')
            np.random.seed(50 + i)
            o, want = oracle_with_draws(fields, c, kind, B)
            assert_batches_identical(flat_host(na.sample(B, draws=o.last_draws)), want, label=label + ' validation:')


# ------------------------------------------------ GPU: edges and safety ------------------------------------------------
@pytest.mark.gpu
def test_first_and_last_rows_clamp_at_the_view_ends(tmp_path):
    from ogbench_b200 import Dataset, GCDataset

    paths = write_shards(tmp_path, seed=5, obs_shape=(7,))
    shards = loader.ResidentShards(paths, load_npz)
    trees = [load_npz(p) for p in paths]
    c = cfg(frame_stack=3)
    for i, t in enumerate(trees):
        n = len(t['terminals'])
        idxs = np.array([0, 1, n - 2, n - 1, 0, n - 1])
        ref = Dataset.create(**t)
        got = shards[i].get_subset(idxs)
        assert_same(got, ref.get_subset(idxs), f'subset {i}')
        obs = t['observations']
        assert np.array_equal(np.asarray(got['next_observations']), obs[np.minimum(idxs + 1, n - 1)])
        assert_same(shards[i].sample(len(idxs), idxs=idxs), ref.sample(len(idxs), idxs=idxs), f'sample idxs {i}')
        gi = idxs[idxs < n - 1]                         # (the last row of a shard is no frame-stack index)
        a, b = GCDataset(shards[i], c, seed=2), GCDataset(ref, c, seed=2)
        assert_same(a.sample(len(gi), idxs=gi), b.sample(len(gi), idxs=gi), f'frame stack {i}')
    whole = concat(trees)
    ref = Dataset.create(**whole)
    edges = np.array(sorted({r for r0, n in shards.bounds for r in (r0, r0 + n - 1)}))
    assert_same(shards.dataset.get_subset(edges), ref.get_subset(edges), 'whole subset')
    gi = edges[edges < len(whole['terminals']) - 1]
    assert_same(GCDataset(shards.dataset, c, seed=2).sample(len(gi), idxs=gi), GCDataset(ref, c, seed=2).sample(len(gi), idxs=gi), 'whole fs')


@pytest.mark.gpu
@pytest.mark.parametrize('sid', ['point2', 'f29', 'f600', 'u8-64-fs3'])
def test_views_write_only_the_keys_and_hand_out_view_rows(built, sid):
    from ogbench_b200 import _native

    _, kinds, kw, over = next(s for s in SHAPES if s[0] == sid)
    paths, shards = built(sid)
    c = config_for('gc', over)
    for i in range(len(paths)):
        s = make('gc', shards[i], c, seed=8)
        s._sampler.set_debug(2)
        h = s._sampler.sample_native(64, n_batches=2)
        bad = C.c_int64(-1)
        _native.check(_native.lib().ogb_batch_check_gaps(h.ptr, C.byref(bad)))
        assert bad.value == 0, (sid, i)
        s._sampler.set_debug(1)
        h = s._sampler.sample_native(64, n_batches=2)
        h.sync()
        n_rows = shards[i].size
        for slot in range(10):
            vec = np.full(128, -1, np.int64)
            try:
                _native.check(_native.lib().ogb_batch_index_vector(h.ptr, slot, vec.ctypes.data_as(C.c_void_p)))
            except (ValueError, IndexError):
                break
            assert vec.min() >= 0 and vec.max() < n_rows, (sid, i, slot)
        assert slot > 0


NO_RECORDS_SCRIPT = r'''
import sys
sys.path.insert(0, sys.argv[1])
import pathlib
import numpy as np
from ogbench_b200 import Dataset, GCDataset, loader
from tests.test_gpu_resident import assert_same, load_npz, write_shards
paths = write_shards(pathlib.Path(sys.argv[2]), seed=7, obs_shape=(3,))
shards = loader.ResidentShards(paths, load_npz)
for i, p in enumerate(paths):
    ref = Dataset.create(**load_npz(p))
    assert_same(GCDataset(shards[i], {cfg}, seed=1).sample(99), GCDataset(ref, {cfg}, seed=1).sample(99), str(i))
print('ok')
'''


@pytest.mark.gpu
def test_views_without_the_record_table(tmp_path):
    """OGB_NO_RECORDS (read once per process): one array per field, dense rows of <= 16 bytes."""
    env = {k: v for k, v in os.environ.items() if not k.startswith('OGB_')}
    env['OGB_NO_RECORDS'] = '1'
    script = NO_RECORDS_SCRIPT.replace('{cfg}', repr(cfg()))
    proc = subprocess.run([sys.executable, '-c', script, ROOT, str(tmp_path)], env=env, capture_output=True, text=True, timeout=600)
    assert proc.returncode == 0 and proc.stdout.strip().endswith('ok'), proc.stderr[-3000:]


# ------------------------------------------------ GPU: the drop-in claim ------------------------------------------------
@pytest.mark.gpu
def test_shard_cycler_over_views_equals_cycler_over_files(tmp_path):
    from ogbench_b200 import GCDataset

    paths = []
    for i, lengths in enumerate(shard_lengths(9, False)):
        f = shard_fields(90 + i, lengths, obs_shape=(10,))
        raw = dict(observations=f['observations'], actions=f['actions'], terminals=np.zeros(len(f['terminals']), np.float32))
        raw['terminals'][np.cumsum(lengths) - 1] = 1.0          # the file's layout: one terminal per trajectory end
        p = str(tmp_path / f'raw{i}.npz')
        np.savez_compressed(p, **raw)
        paths.append(p)
    c = cfg()
    shards = loader.ResidentShards(paths)
    memo = {}

    def from_view(p):
        if p not in memo:
            memo[p] = GCDataset(shards[p], c, seed=11)
        return memo[p]

    a = loader.ShardCycler(paths, from_view, 3)
    b = loader.ShardCycler(paths, lambda p: loader.load_gc_dataset(p, c, seed=11), 3)
    for step in range(1, 23):                             # 7 swaps: every shard revisited
        assert_same(a.at_step(step).sample(64), b.at_step(step).sample(64), f'step {step}')
    assert a.swaps == b.swaps == 7
    a.close()
    b.close()


# ------------------------------------------------ GPU: building and lifetime ------------------------------------------------
def build_in_blocks(fields, block, capacity=None):
    from ogbench_b200 import _native
    from ogbench_b200.datasets import ResidentDataset, _NativeDataset, _ZeroField

    n = len(fields['terminals'])
    nds = _NativeDataset.empty({k: _ZeroField((capacity or n, *v.shape[1:]), v.dtype) for k, v in fields.items()}, 0)
    arrays = list(fields.values())
    for r0 in range(0, n, block):
        m = min(block, n - r0)
        chunk = [np.ascontiguousarray(a[r0:r0 + m]) for a in arrays]
        ptrs = (C.c_void_p * len(chunk))(*[a.ctypes.data for a in chunk])
        _native.check(_native.lib().ogb_dataset_write_rows(nds.ptr, r0, m, ptrs, len(chunk)))
    _native.check(_native.lib().ogb_dataset_seal(nds.ptr, n))
    return ResidentDataset(nds, list(fields), False, (fields['valids'] > 0).astype(np.uint8))


@pytest.mark.gpu
def test_write_block_size_does_not_change_the_batches():
    from ogbench_b200 import Dataset, GCDataset

    fields = toy_fields(12, ragged(12, 40, 2, 150), (29,), 8, np.float32)   # ~3,000 rows: 4,096 is one partial block
    ref = GCDataset(Dataset.create(**fields), cfg(), seed=3).sample_many(2, 500)
    for block in (1, 7, 4096, len(fields['terminals'])):
        got = GCDataset(build_in_blocks(fields, block, capacity=len(fields['terminals']) + 17), cfg(), seed=3).sample_many(2, 500)
        assert_same(got, ref, f'block {block}')


@pytest.mark.gpu
def test_refusals():
    from ogbench_b200 import GCDataset, _native
    from ogbench_b200.datasets import _NativeDataset, _ZeroField

    lib = _native.lib()
    fields = toy_fields(13, ragged(13, 6, 2, 20), (4,), 2, np.float32)
    n = len(fields['terminals'])
    arrays = list(fields.values())
    ptrs = (C.c_void_p * len(arrays))(*[a.ctypes.data for a in arrays])
    nds = _NativeDataset.empty({k: _ZeroField((n + 4, *v.shape[1:]), v.dtype) for k, v in fields.items()}, 0)
    with pytest.raises(ValueError, match='sealed'):
        nds.view(0, 2)                                                          # a view of an unsealed dataset
    with pytest.raises(IndexError):
        _native.check(lib.ogb_dataset_write_rows(nds.ptr, 5, n, ptrs, len(arrays)))     # past the capacity
    _native.check(lib.ogb_dataset_write_rows(nds.ptr, 0, n, ptrs, len(arrays)))
    with pytest.raises(ValueError):
        _native.check(lib.ogb_dataset_seal(nds.ptr, n + 5))                      # above the capacity
    _native.check(lib.ogb_dataset_seal(nds.ptr, n))
    for r0, m in ((-1, 2), (0, 0), (n - 1, 2)):
        with pytest.raises(ValueError):
            nds.view(r0, m)                                                     # out of range
    view = nds.view(1, n - 1)
    with pytest.raises(ValueError, match='view'):
        _native.check(lib.ogb_dataset_write_rows(view.ptr, 0, 1, ptrs, len(arrays)))   # writing to a view
    with pytest.raises(ValueError, match='held'):
        _native.check(lib.ogb_dataset_seal(nds.ptr, n))                          # a view holds it
    with pytest.raises(ValueError):
        _native.check(lib.ogb_dataset_set_active_rows(view.ptr, 1))
    del view
    gc.collect()
    fresh = build_in_blocks(fields, n)
    sampler = GCDataset(fresh, cfg(), seed=1)
    with pytest.raises(ValueError, match='held'):
        _native.check(lib.ogb_dataset_write_rows(fresh.native(0).ptr, 0, 1, ptrs, len(arrays)))   # a sampler holds it
    with pytest.raises(ValueError, match='held'):
        _native.check(lib.ogb_dataset_seal(fresh.native(0).ptr, n))
    with pytest.raises(ValueError, match='device'):
        GCDataset(fresh, cfg(), device=1)                                       # another device than the table's
    del sampler
    rows = (C.c_void_p * len(arrays))(*[a[:1].ctypes.data for a in arrays])
    view_sampler = GCDataset(fresh.__class__(fresh.native(0).view(0, n), list(fields), False, None), cfg(), seed=1)
    with pytest.raises(ValueError, match='view'):
        _native.check(lib.ogb_sampler_write_row(view_sampler._sampler.ptr, 0, rows, len(arrays)))
    unsealed = _NativeDataset.empty({k: _ZeroField((n, *v.shape[1:]), v.dtype) for k, v in fields.items()}, 0)
    out = C.c_void_p()
    with pytest.raises(ValueError, match='sealed'):
        _native.check(lib.ogb_sampler_create(unsealed.ptr, C.byref(_native.Config()), _native.KIND_PLAIN, 0, 0, C.byref(out)))


@pytest.mark.gpu
def test_views_outlive_their_shards_object(tmp_path):
    from ogbench_b200 import Dataset, GCDataset

    paths = write_shards(tmp_path, seed=6, obs_shape=(8,))
    shards = loader.ResidentShards(paths, load_npz)
    s = GCDataset(shards[1], cfg(), seed=5)
    del shards
    gc.collect()
    ref = GCDataset(Dataset.create(**load_npz(paths[1])), cfg(), seed=5)
    for it in range(3):
        assert_same(s.sample(100), ref.sample(100), f'after del {it}')


@pytest.mark.gpu
def test_host_memory_stays_near_one_shard(tmp_path):
    rng = np.random.default_rng(0)
    paths, biggest = [], 0
    for i, n in enumerate((190_000, 205_000, 170_000, 200_000)):      # ~50 MB of observations each
        terminals = np.zeros(n, np.float32)
        terminals[np.arange(999, n, 1000)] = 1.0
        terminals[-1] = 1.0
        f = dict(observations=rng.standard_normal((n, 55), dtype=np.float32), actions=rng.uniform(-1, 1, (n, 5)).astype(np.float32),
                 terminals=terminals)
        p = str(tmp_path / f'big{i}.npz')
        np.savez(p, **f)
        paths.append(p)
        del f
    for p in paths:
        biggest = max(biggest, sum(a.nbytes for a in loader.load_dataset(p, compact_dataset=True).values()))
    gc.collect()
    tracemalloc.start()
    try:
        shards = loader.ResidentShards(paths)
        _, peak = tracemalloc.get_traced_memory()
    finally:
        tracemalloc.stop()
    assert shards.dataset.size == 765_000
    assert peak < 2 * biggest, (peak, biggest)

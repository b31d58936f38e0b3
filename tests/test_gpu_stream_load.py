"""Streaming `.npz` files into HBM block by block (loader.upload_dataset, ResidentShards with the default loader).

- the block reader yields exactly np.load(path)[k] for stored and deflated members, .npy versions 1.0 / 2.0 / 3.0 and
  ZIP64 members, at any block size; it reads Fortran-order members whole and refuses truncated and missing ones;
- the per-block layout (casts, compact terminals / valids, the regular layout's kept rows and next observations) writes
  every row of load_dataset's result once and equals it, wherever the terminals fall relative to the blocks;
- on the GPU, upload_dataset's dataset equals Dataset.create(**load_dataset(...)) key for key, and samples the same
  batches with Philox and under rng='numpy', for the committed raw files and for synthetic files of many blocks;
- host memory stays at a few blocks per member plus a few bytes per row.
"""

import glob
import io
import os
import tracemalloc
import zipfile

import numpy as np
import pytest

from ogbench_b200 import loader
from tests.golden.make_golden import cfg, ragged
from tests.golden_util import assert_batches_identical

RAW = sorted(glob.glob(os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'loader_raw', '*.npz')))


def write_npz(path, arrays, compressed=True, version=None, force_zip64=False, fortran=()):
    """An .npz as np.savez / np.savez_compressed write it, with a chosen .npy format version and ZIP64 members."""
    method = zipfile.ZIP_DEFLATED if compressed else zipfile.ZIP_STORED
    with zipfile.ZipFile(path, 'w', compression=method, allowZip64=True) as zf:
        for k, a in arrays.items():
            buf = io.BytesIO()
            np.lib.format.write_array(buf, np.asfortranarray(a) if k in fortran else a, version=version)
            with zf.open(f'{k}.npy', 'w', force_zip64=force_zip64) as f:
                f.write(buf.getvalue())


def truncated_npz(path, compressed, key='observations', shape=(40, 6), keep_rows=25):
    """A member whose header declares `shape` but whose data ends after `keep_rows` rows."""
    a = np.arange(np.prod(shape), dtype=np.float32).reshape(shape)
    buf = io.BytesIO()
    np.lib.format.write_array(buf, a)
    data = buf.getvalue()
    cut = len(data) - (shape[0] - keep_rows) * a[0].nbytes
    with zipfile.ZipFile(path, 'w', compression=zipfile.ZIP_DEFLATED if compressed else zipfile.ZIP_STORED) as zf:
        zf.writestr(f'{key}.npy', data[:cut])
        zf.writestr('actions.npy', _npy(np.zeros((shape[0], 2), np.float32)))
        zf.writestr('terminals.npy', _npy(np.ones(shape[0], bool)))


def _npy(a):
    buf = io.BytesIO()
    np.lib.format.write_array(buf, a)
    return buf.getvalue()


def sample_arrays(seed, n=53):
    rng = np.random.default_rng(seed)
    return dict(observations=rng.standard_normal((n, 7)), frames=rng.integers(0, 256, (n, 4, 5, 3), dtype=np.uint8),
                terminals=rng.random(n) < 0.2, button_states=rng.integers(-9, 9, (n, 2)), scalar=np.float32(3.5),
                empty=np.zeros((0, 3), np.float32))


# ------------------------------------------------ CPU: the block reader ------------------------------------------------
@pytest.mark.parametrize('compressed', [True, False])
@pytest.mark.parametrize('version', [(1, 0), (2, 0), (3, 0)])
def test_blocks_are_the_member(tmp_path, compressed, version):
    p = str(tmp_path / 'a.npz')
    arrays = sample_arrays(1)
    write_npz(p, arrays, compressed, version)
    z = np.load(p)
    for k in arrays:
        want = z[k]
        for block_rows in (1, 7, None):
            blocks = list(loader.read_member_blocks(p, k, block_rows))
            got = np.concatenate(blocks) if len(blocks) > 1 else blocks[0]
            assert got.dtype == want.dtype and got.shape == want.shape and np.array_equal(got, want), (k, block_rows)
            if block_rows and want.ndim and len(want):
                assert [len(b) for b in blocks[:-1]] == [block_rows] * (len(blocks) - 1), (k, block_rows)
    assert loader.shard_rows(p) == len(arrays['terminals'])


@pytest.mark.parametrize('compressed', [True, False])
def test_zip64_members(tmp_path, compressed):
    p = str(tmp_path / 'z64.npz')
    arrays = sample_arrays(2, n=300)
    write_npz(p, arrays, compressed, force_zip64=True)
    z = np.load(p)
    for k in ('observations', 'frames', 'terminals'):
        assert np.array_equal(np.concatenate(list(loader.read_member_blocks(p, k, 64))), z[k]), k


def test_default_block_is_about_8_mb(tmp_path):
    p = str(tmp_path / 'big.npz')
    obs = np.arange(70_000 * 55, dtype=np.float32).reshape(70_000, 55)       # 15.4 MB: two blocks
    np.savez(p, observations=obs)
    blocks = list(loader.read_member_blocks(p, 'observations'))
    assert [len(b) for b in blocks] == [(8 << 20) // 220, 70_000 - (8 << 20) // 220]
    assert np.array_equal(np.concatenate(blocks), obs)


def test_fortran_order_member_is_read_whole(tmp_path):
    p = str(tmp_path / 'f.npz')
    arrays = sample_arrays(3)
    write_npz(p, arrays, fortran=('observations', 'frames'))
    for k in ('observations', 'frames'):
        blocks = list(loader.read_member_blocks(p, k, 5))
        assert len(blocks) == 1 and np.array_equal(blocks[0], np.load(p)[k]), k


@pytest.mark.parametrize('compressed', [True, False])
def test_truncated_member_is_refused(tmp_path, compressed):
    p = str(tmp_path / 'cut.npz')
    truncated_npz(p, compressed)
    with pytest.raises(ValueError, match=r"cut\.npz.*'observations'.*25 of the 40 rows"):
        list(loader.read_member_blocks(p, 'observations', 10))
    stream = loader._FileStream(p, compact_dataset=True)        # (the headers agree: the data ends early)
    with pytest.raises(ValueError, match=r"cut\.npz.*'observations'"):
        loader._pump(stream.producers(5), lambda r0, arrays: None)   # raised on the writing thread, every reader stopped


def test_missing_member_is_a_key_error(tmp_path):
    p = str(tmp_path / 'm.npz')
    np.savez(p, observations=np.zeros((3, 2)), terminals=np.ones(3, bool))
    with pytest.raises(KeyError, match='actions'):
        list(loader.read_member_blocks(p, 'actions'))
    with pytest.raises(KeyError, match='actions'):
        loader._FileStream(p)


# ------------------------------------------------ CPU: the per-block layout ------------------------------------------------
def assemble(stream, block_rows):
    """Apply the stream's writes to host arrays; every row of every field must be written exactly once."""
    out = {k: np.zeros(shape, dtype) for k, (dtype, shape) in stream.fields.items()}
    hits = {k: np.zeros(shape[0], np.int64) for k, (_, shape) in stream.fields.items()}
    for producer in stream.producers(block_rows):
        for r0, arrays in producer:
            for k, a in arrays.items():
                assert a.dtype == out[k].dtype and a.shape[1:] == out[k].shape[1:], k
                out[k][r0:r0 + len(a)] = a
                hits[k][r0:r0 + len(a)] += 1
    for k, h in hits.items():
        assert (h == 1).all(), (k, np.flatnonzero(h != 1)[:5])
    return out


def assert_layout_equal(path, block_rows, label, **kw):
    want = loader.load_dataset(path, **kw)
    stream = loader._FileStream(path, **kw)
    assert list(stream.fields) == list(want), label
    got = assemble(stream, block_rows)
    for k, w in want.items():
        g = got[k]
        assert g.dtype == w.dtype and g.shape == w.shape and np.array_equal(g, w), (label, k)
    if kw.get('compact_dataset'):
        assert np.array_equal(stream.flags, (want['valids'] > 0).astype(np.uint8)), label


def edge_file(path, last_terminal, terminal_dtype, compressed):
    """29 rows; with 7-row blocks the terminals fall on a block's first row (0, 7), last row (13, 20) and inner rows
    (3, 17, 25)."""
    n = 29
    rng = np.random.default_rng(5)
    terminals = np.zeros(n, terminal_dtype)
    terminals[[0, 3, 7, 13, 17, 20, 25]] = 1
    terminals[-1] = 1 if last_terminal else 0
    (np.savez_compressed if compressed else np.savez)(
        path, observations=rng.standard_normal((n, 3)), actions=rng.standard_normal((n, 2)).astype(np.float32),
        terminals=terminals, qpos=rng.standard_normal((n, 4)), button_states=rng.integers(0, 4, (n, 2)))


@pytest.mark.parametrize('last_terminal', [True, False])
@pytest.mark.parametrize('terminal_dtype', [bool, np.float32])
def test_per_block_layout_equals_load_dataset(tmp_path, last_terminal, terminal_dtype):
    p = str(tmp_path / 'edges.npz')
    edge_file(p, last_terminal, terminal_dtype, compressed=True)
    for compact in (False, True):
        for add_info in (False, True):
            for block_rows in (1, 7, None):
                assert_layout_equal(p, block_rows, (compact, add_info, block_rows), compact_dataset=compact, add_info=add_info,
                                    ob_dtype=np.float32, action_dtype=np.float64)


def file_dtypes(path):
    """The dtypes make_datasets picks for the file's environment (ogbench/utils.py:196-203)."""
    name = os.path.basename(path)
    ob = np.uint8 if ('visual' in name or 'powderworld' in name) else np.float32
    return dict(ob_dtype=ob, action_dtype=np.int32 if 'powderworld' in name else np.float32)


@pytest.mark.parametrize('path', RAW, ids=[os.path.basename(p) for p in RAW])
def test_per_block_layout_of_the_raw_files(path):
    for compact in (False, True):
        for add_info in (False, True):
            for block_rows in (1, 7, None):
                assert_layout_equal(path, block_rows, (compact, add_info, block_rows), compact_dataset=compact,
                                    add_info=add_info, **file_dtypes(path))
    assert_layout_equal(path, 3, 'default dtypes')


def test_default_shards_stream_with_load_datasets_schema(tmp_path):
    paths = []
    for i in range(2):
        p = str(tmp_path / f's{i}.npz')
        edge_file(p, True, bool, compressed=bool(i))
        paths.append(p)
    shards = list(loader.iter_shards(paths))
    for shard, p in zip(shards, paths):
        want = loader.load_dataset(p, compact_dataset=True)
        assert shard.fields is None and shard.keys == list(want) and shard.n_rows == len(want['terminals'])
        assert shard.schema == {k: (v.dtype, v.shape[1:]) for k, v in want.items()}
    np.savez(paths[1], observations=np.zeros((5, 4)), actions=np.zeros((5, 2)), terminals=np.ones(5, bool))
    with pytest.raises(ValueError, match='s1.npz'):
        list(loader.iter_shards(paths))


# ------------------------------------------------ GPU: upload_dataset against the host path ------------------------------------------------
def flat_host(batch, prefix=''):
    out = {}
    for k, v in batch.items():
        if isinstance(v, dict):
            out.update(flat_host(v, f'{prefix}{k}/'))
        else:
            out[prefix + k] = np.asarray(v)
    return out


def assert_same_dataset(path, label, batch=64, **kw):
    from ogbench_b200 import Dataset, GCDataset

    got = loader.upload_dataset(path, **kw)
    ref = Dataset.create(**loader.load_dataset(path, **kw))
    assert got.size == ref.size and list(got) == list(ref), label
    rows = np.arange(ref.size)
    assert_batches_identical(flat_host(got.get_subset(rows)), flat_host(ref.get_subset(rows)), label=f'{label} subset:')
    c = cfg()
    a, b = GCDataset(got, c, seed=7), GCDataset(ref, c, seed=7)
    for it in range(2):
        assert_batches_identical(flat_host(a.sample(batch)), flat_host(b.sample(batch)), label=f'{label} philox {it}:')
    assert_batches_identical(flat_host(a.sample_many(2, batch)), flat_host(b.sample_many(2, batch)), label=f'{label} many:')
    a, b = GCDataset(got, c, rng='numpy'), GCDataset(ref, c, rng='numpy')
    for it in range(2):
        np.random.seed(30 + it)
        x = flat_host(a.sample(batch))
        np.random.seed(30 + it)
        assert_batches_identical(x, flat_host(b.sample(batch)), label=f'{label} numpy {it}:')


@pytest.mark.gpu
@pytest.mark.parametrize('path', RAW, ids=[os.path.basename(p) for p in RAW])
def test_raw_files_upload_like_the_host_path(path):
    for compact in (False, True):
        for add_info in (False, True):
            assert_same_dataset(path, f'c{int(compact)} i{int(add_info)}', compact_dataset=compact, add_info=add_info,
                                **file_dtypes(path))


def synthetic_file(path, kind, compressed, seed):
    rng = np.random.default_rng(seed)
    if kind == 'state':                    # C5's row: 55 float32, 5 float32 actions, trajectories across block ends
        lengths = ragged(seed, 300, 200, 1200)
        n = int(lengths.sum())
        obs = rng.standard_normal((n, 55), dtype=np.float32)
        actions = rng.uniform(-1, 1, (n, 5)).astype(np.float32)
    else:                                  # visual-cube frames: 64x64x3 uint8 (a block is 682 frames)
        lengths = ragged(seed, 30, 20, 250)
        n = int(lengths.sum())
        base = rng.integers(0, 256, (64, 64, 3), dtype=np.uint8)
        obs = (base[None] + (np.arange(n, dtype=np.uint32) * 7 % 251)[:, None, None, None]).astype(np.uint8)
        obs[:, ::9, ::5] = rng.integers(0, 256, obs[:, ::9, ::5].shape, dtype=np.uint8)
        actions = rng.uniform(-1, 1, (n, 5)).astype(np.float32)
    terminals = np.zeros(n, bool)
    terminals[np.cumsum(lengths) - 1] = True
    (np.savez_compressed if compressed else np.savez)(path, observations=obs, actions=actions, terminals=terminals,
                                                      qpos=rng.standard_normal((n, 9)), button_states=rng.integers(0, 2, (n, 3)))
    return n


@pytest.mark.gpu
@pytest.mark.parametrize('kind,compressed', [('state', True), ('state', False), ('frames', True)])
def test_many_block_files_upload_like_the_host_path(tmp_path, kind, compressed):
    p = str(tmp_path / f'{kind}.npz')
    n = synthetic_file(p, kind, compressed, seed=21)
    obs_bytes = n * (55 * 4 if kind == 'state' else 64 * 64 * 3)
    assert obs_bytes > 4 * (8 << 20)                                   # several default blocks of observations
    ob_dtype = np.float32 if kind == 'state' else np.uint8
    for compact in (False, True):
        for add_info in (False, True):
            assert_same_dataset(p, f'{kind} c{int(compact)} i{int(add_info)}', batch=256 if kind == 'state' else 32,
                                compact_dataset=compact, add_info=add_info, ob_dtype=ob_dtype)


@pytest.mark.gpu
def test_small_blocks_upload_like_the_host_path(tmp_path, monkeypatch):
    """Blocks of a few hundred rows: every trajectory crosses block ends, in every member."""
    p = str(tmp_path / 'small.npz')
    synthetic_file(p, 'state', True, seed=22)
    monkeypatch.setattr(loader, '_BLOCK_BYTES', 64 << 10)
    for compact in (False, True):
        assert_same_dataset(p, f'c{int(compact)}', batch=256, compact_dataset=compact, add_info=True)


@pytest.mark.gpu
def test_default_resident_shards_stream_like_the_host_path(tmp_path):
    from ogbench_b200 import GCDataset

    paths = []
    for i in range(3):
        p = str(tmp_path / f'shard{i}.npz')
        synthetic_file(p, 'state', bool(i % 2), seed=40 + i)
        paths.append(p)
    streamed = loader.ResidentShards(paths)
    loaded = loader.ResidentShards(paths, load=lambda p: loader.load_dataset(p, compact_dataset=True))
    assert streamed.bounds == loaded.bounds and list(streamed.dataset) == list(loaded.dataset)
    for label, a, b in [('whole', streamed.dataset, loaded.dataset)] + [(f'shard {i}', streamed[i], loaded[i]) for i in range(3)]:
        rows = np.arange(a.size)
        assert_batches_identical(flat_host(a.get_subset(rows)), flat_host(b.get_subset(rows)), label=f'{label} subset:')
        assert np.array_equal(a.valid_idxs, b.valid_idxs), label
        x, y = GCDataset(a, cfg(), seed=3), GCDataset(b, cfg(), seed=3)
        assert_batches_identical(flat_host(x.sample(512)), flat_host(y.sample(512)), label=f'{label} philox:')


@pytest.mark.gpu
def test_regular_layout_without_a_final_terminal_is_refused(tmp_path):
    from ogbench_b200 import Dataset

    p = str(tmp_path / 'open.npz')
    edge_file(p, False, bool, compressed=False)
    with pytest.raises(ValueError):
        Dataset.create(**loader.load_dataset(p)).native(0)
    with pytest.raises(ValueError, match='open.npz'):
        loader.upload_dataset(p)
    assert_same_dataset(p, 'compact', compact_dataset=True)


@pytest.mark.gpu
def test_host_memory_stays_at_a_few_blocks(tmp_path):
    n = 2_000_000
    rng = np.random.default_rng(0)
    terminals = np.zeros(n, bool)
    terminals[np.arange(1000, n, 1001)] = True
    terminals[-1] = True
    p = str(tmp_path / 'big.npz')
    np.savez(p, observations=rng.standard_normal((n, 55), dtype=np.float32),     # 440 MB of observations
             actions=rng.uniform(-1, 1, (n, 5)).astype(np.float32), terminals=terminals)
    file_bytes = os.path.getsize(p)
    producers = 3                                   # observations, actions and the terminal fields
    bound = producers * 6 * (8 << 20) + 8 * n       # six 8 MB blocks per producer (queued and in flight), 8 B per row
    assert bound < file_bytes / 2
    for compact in (True, False):
        tracemalloc.start()
        try:
            ds = loader.upload_dataset(p, compact_dataset=compact)
            _, peak = tracemalloc.get_traced_memory()
        finally:
            tracemalloc.stop()
        assert ds.size == (n if compact else n - int(terminals.sum()))
        assert peak < bound, (compact, peak, bound)
        del ds

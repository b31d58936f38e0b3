"""ReplayBuffer.add_transitions (and add_transition with device leaves): n transitions in one ring write.

CPU: the pointer / size / row arithmetic against a loop of the oracle's add_transition.  GPU: the reference's goldens
with every add step fed as one call and in chunks, from numpy and from torch CUDA tensors; random batch sizes over the
record layouts the ring scatter has to handle, against OracleReplayBuffer fed one transition at a time; stream ordering,
source lifetime and the refusals."""

import ctypes as C
import gc

import numpy as np
import pytest

from oracle.replay_oracle import OracleReplayBuffer
from ogbench_b200.datasets import ring_plan
from tests.golden.make_golden_replay import CAPACITY, SCRIPT, make_transitions
from tests.test_replay_buffer import check, load


# ---------------------------------------------------------------------------------------------------------------- CPU
def test_ring_plan_matches_add_transition_loop():
    for m in range(1, 10):
        for pointer in range(m):
            for size in range(pointer, m + 1):          # size >= pointer always; size == m only for a buffer created full
                for n in range(0, 3 * m + 3):
                    rb = OracleReplayBuffer({'x': np.int64(0)}, m)
                    rb.buffers['x'][:] = -1
                    rb.pointer, rb.size = pointer, size
                    for i in range(n):
                        rb.add_transition({'x': i})
                    row0, skip, p, s = ring_plan(pointer, size, m, n)
                    assert (p, s) == (rb.pointer, rb.size), (m, pointer, size, n)
                    assert n - skip <= m and row0 == pointer
                    want = np.full(m, -1)
                    for i in range(skip, n):
                        want[(row0 + i) % m] = i
                    assert np.array_equal(want, rb.buffers['x']), (m, pointer, size, n)


# ---------------------------------------------------------------------------------------------------------------- GPU
def stack(transitions):
    return {k: np.stack([np.asarray(t[k]) for t in transitions]) for k in transitions[0]}


def to_source(batch, how, rng=None):
    """numpy, torch CUDA, or a random mix of the two per leaf."""
    import torch

    out = {}
    for k, v in batch.items():
        if isinstance(v, dict):
            out[k] = to_source(v, how, rng)
            continue
        dev = how == 'torch' or (how == 'mixed' and rng.random() < 0.5)
        out[k] = torch.from_numpy(np.ascontiguousarray(v)).cuda() if dev else v
    return out


def chunks(n, rng, largest=7):
    sizes = []
    while n > 0:
        sizes.append(min(n, int(rng.integers(1, largest + 1))))
        n -= sizes[-1]
    return sizes


def feed(rb, batch, sizes, how, rng):
    start = 0
    for k in sizes:
        part = {key: v[start:start + k] for key, v in batch.items()}
        rb.add_transitions(to_source(part, how, rng))
        start += k


@pytest.mark.gpu
@pytest.mark.parametrize('how', ['numpy', 'torch'])
@pytest.mark.parametrize('chunked', [False, True])
def test_golden_script(how, chunked):
    from ogbench_b200 import ReplayBuffer

    want, init_want, init_state = load()
    transitions = make_transitions(200)
    rng = np.random.default_rng(3)
    rb = ReplayBuffer.create(transitions[0], size=CAPACITY, rng='numpy', output='numpy')
    oracle = OracleReplayBuffer(transitions[0], CAPACITY)
    outs, t = [], 0
    for step in SCRIPT:
        if step[0] == 'add':
            k = step[1]
            feed(rb, stack(transitions[t:t + k]), chunks(k, rng) if chunked else [k], how, rng)
            for tr in transitions[t:t + k]:
                oracle.add_transition(tr)
            t += k
            assert (rb.pointer, rb.size) == (oracle.pointer, oracle.size)
        elif step[0] == 'clear':
            rb.clear()
            oracle.clear()
        else:
            np.random.seed(step[2])
            outs.append(rb.sample(step[1]))
    assert len(outs) == len(want)
    for g, w in zip(outs, want):
        check(g, w)
    init = {k: np.stack([tr[k] for tr in transitions[:20]]) for k in transitions[0]}
    rb2 = ReplayBuffer.create_from_initial_dataset(init, size=40, rng='numpy', output='numpy')
    feed(rb2, stack(transitions[20:50]), chunks(30, rng) if chunked else [30], how, rng)
    np.random.seed(9)
    check(rb2.sample(24), init_want)
    assert [rb2.size, rb2.pointer, rb2.max_size] == list(init_state)


def nest_rows(batch, like):
    """A flat batch of transitions back in the nesting of the example transition `like`."""
    out = {}
    for k, v in like.items():
        out[k] = {kk: batch[f'{k}/{kk}'] for kk in v} if isinstance(v, dict) else batch[k]
    return out


M = 37
LAYOUTS = ['pointmaze', 'c2', 'odd_rows', 'bool_int64', 'frames', 'pytree']


def layout(name, rng, n):
    """n random transitions of one record layout, as a flat dict of [n, ...] arrays."""
    f32 = lambda *s: rng.standard_normal((n, *s)).astype(np.float32)  # noqa: E731
    if name == 'pointmaze':       # no next_observations: gathered as observations[min(idx + 1, size - 1)]
        return dict(observations=f32(2), actions=f32(2), terminals=rng.integers(0, 2, n).astype(np.float32), rewards=f32())
    if name == 'c2':
        return dict(observations=f32(29), actions=f32(8), rewards=f32(), terminals=rng.integers(0, 2, n).astype(np.float32),
                    masks=np.ones(n, np.float32), next_observations=f32(29))
    if name == 'odd_rows':        # 18-byte float16 rows, 17-byte uint8 rows
        return dict(observations=f32(3), half=rng.standard_normal((n, 9)).astype(np.float16),
                    bytes17=rng.integers(0, 256, (n, 17), dtype=np.uint8))
    if name == 'bool_int64':
        return dict(observations=f32(5), flags=rng.random(n) < 0.5, steps=rng.integers(-2**40, 2**40, n, dtype=np.int64),
                    pair=rng.integers(0, 9, (n, 2), dtype=np.int64))
    if name == 'frames':          # 64x64x3 uint8: an array of its own
        return dict(observations=rng.integers(0, 256, (n, 64, 64, 3), dtype=np.uint8), actions=f32(5))
    if name == 'pytree':
        return {'observations/image': rng.integers(0, 256, (n, 8, 8, 3), dtype=np.uint8), 'observations/state': f32(5),
                'next_observations/image': rng.integers(0, 256, (n, 8, 8, 3), dtype=np.uint8), 'next_observations/state': f32(5),
                'actions': f32(3)}
    raise KeyError(name)


def oracle_sample(oracle, batch_size, idxs=None):
    """OracleReplayBuffer.sample; a flattened pytree buffer stores its next observations as leaves of their own, so there
    nothing is synthesised (the oracle would look for a plain 'observations' buffer)."""
    if 'observations' in oracle.buffers:
        return oracle.sample(batch_size, idxs)
    if idxs is None:
        idxs = np.random.randint(oracle.size, size=batch_size)             # datasets.py:70
    return {k: v[idxs] for k, v in oracle.buffers.items()}


def compare(rb, oracle, nested):
    from ogbench_b200.datasets import _flatten

    def host(batch):
        return {k: np.asarray(v) for k, v in (_flatten(batch) if nested else batch).items()}

    assert (rb.pointer, rb.size) == (oracle.pointer, oracle.size)
    for idxs in (np.arange(M), np.arange(rb.size)):     # every row: the ones not written must be unchanged too
        check(host(rb.sample(len(idxs), idxs=idxs)), oracle_sample(oracle, len(idxs), idxs))
    seed = int(oracle.pointer * 1000 + oracle.size)
    np.random.seed(seed)
    got = host(rb.sample(64))
    np.random.seed(seed)
    check(got, oracle_sample(oracle, 64))


@pytest.mark.gpu
@pytest.mark.parametrize('name', LAYOUTS)
def test_against_oracle(name):
    from ogbench_b200 import ReplayBuffer

    rng = np.random.default_rng(LAYOUTS.index(name))
    nested = name == 'pytree'
    example = {k: v[0] for k, v in layout(name, rng, 1).items()}
    rb = ReplayBuffer.create(nest_rows(example, nest_rows_like(example)) if nested else example, size=M, rng='numpy',
                             output='numpy')
    oracle = OracleReplayBuffer(example, M)
    # a random starting pointer, reached one host transition at a time
    for _ in range(int(rng.integers(0, M))):
        t = {k: v[0] for k, v in layout(name, rng, 1).items()}
        rb.add_transition(nest_rows(t, nest_rows_like(t)) if nested else t)
        oracle.add_transition(t)
    compare(rb, oracle, nested)
    for call in range(12):
        n = int(rng.choice([1, M - 1, M, M + 1, 2 * M + 3]))
        batch = layout(name, rng, n)
        how = ['numpy', 'torch', 'mixed'][call % 3]
        src = to_source(nest_rows(batch, nest_rows_like(batch)) if nested else batch, how, rng)
        rb.add_transitions(src)
        for i in range(n):
            oracle.add_transition({k: v[i] for k, v in batch.items()})
        compare(rb, oracle, nested)
    # add_transition with device leaves takes the same path (n = 1)
    import torch

    for _ in range(3):
        batch = layout(name, rng, 1)
        one = {k: torch.from_numpy(np.asarray(v[0])).cuda() for k, v in batch.items()}    # (0-d rows stay 0-d)
        rb.add_transition(nest_rows(one, nest_rows_like(one)) if nested else one)
        oracle.add_transition({k: v[0] for k, v in batch.items()})
        compare(rb, oracle, nested)


@pytest.mark.gpu
def test_shadow_next_observation_stays_coherent():
    """A dataset created full with <= 16-byte observations keeps the shadow of the next row's observation in every record.
    Ring writes refresh it: the written rows' predecessors, and the last row, which shadows itself.  (A ReplayBuffer
    created full from an initial dataset has pointer == max_size, where the reference's next add_transition raises
    IndexError, and so does add_transitions.)"""
    from ogbench_b200 import Dataset, ReplayBuffer, _native

    rng = np.random.default_rng(11)
    init = layout('pointmaze', rng, M)
    rb = ReplayBuffer.create_from_initial_dataset(init, size=M)
    oracle = OracleReplayBuffer.from_initial_dataset(init, M)
    with pytest.raises(IndexError):
        oracle.add_transition({k: v[0] for k, v in init.items()})
    with pytest.raises(IndexError):
        rb.add_transitions(layout('pointmaze', rng, 2))
    assert (rb.pointer, rb.size) == (M, M)

    ds = Dataset.create(**{k: v.copy() for k, v in init.items()})
    ds.output = 'numpy'
    sampler = ds._plain_sampler()
    mirror = {k: v.copy() for k, v in init.items()}
    names = list(init)
    lib = _native.lib()
    t, r = C.c_uint64(), C.c_uint64()
    for call in range(16):
        n = int(rng.choice([1, 2, M - 1, M, M + 1, 2 * M + 3]))
        row0 = int(rng.integers(0, M)) if call else M - 1          # (the last row first: it shadows itself)
        skip = max(0, n - M)
        batch = layout('pointmaze', rng, n)
        for i in range(skip, n):
            for k in names:
                mirror[k][(row0 + i) % M] = batch[k][i]
        dev = call % 2 == 1
        src = to_source(batch, 'torch' if dev else 'numpy')
        keep = [src[k] if dev else np.ascontiguousarray(src[k]) for k in names]
        ptrs = (C.c_void_p * len(names))(*[a.data_ptr() if dev else a.ctypes.data for a in keep])
        on_device = (C.c_int32 * len(names))(*([int(dev)] * len(names)))
        producer = C.c_void_p(1 if dev else None)                 # (torch's default stream is the legacy one)
        _native.check(lib.ogb_sampler_write_ring(sampler.ptr, row0, n, skip, ptrs, len(names), on_device, producer,
                                                 C.byref(t), C.byref(r)))
        idxs = np.arange(M)
        out = ds.sample(M, idxs=idxs)
        for k in names:
            assert np.array_equal(out[k], mirror[k]), k
        assert np.array_equal(out['next_observations'], mirror['observations'][np.minimum(idxs + 1, M - 1)])


def nest_rows_like(flat_batch):
    """The nesting of a flat batch whose pytree leaves are named '<key>/<leaf>'."""
    like = {}
    for k in flat_batch:
        if '/' in k:
            a, b = k.split('/')
            like.setdefault(a, {})[b] = None
        else:
            like[k] = None
    return like


def sampler_stream(rb):
    from ogbench_b200 import _native

    handle = C.c_void_p()
    _native.check(_native.lib().ogb_sampler_get_stream(rb._plain_sampler(rb._device).ptr, C.byref(handle)))
    return handle.value


def stall(torch, stream_handle, cycles=200_000_000):
    """Keep a stream busy for a while (about 0.1 s), so that work queued behind it is still pending."""
    with torch.cuda.stream(torch.cuda.ExternalStream(stream_handle)):
        torch.cuda._sleep(cycles)


@pytest.mark.gpu
def test_ordering_and_lifetime():
    import torch

    from ogbench_b200 import ReplayBuffer

    cap, dim = 4096, 32
    rb = ReplayBuffer.create({'observations': np.zeros(dim, np.float32), 'rewards': np.float32(0)}, size=cap, output='numpy')
    rb.add_transitions({'observations': np.ones((cap, dim), np.float32), 'rewards': np.ones(cap, np.float32)})
    idxs = np.arange(cap)                                # (every write below covers the whole ring)
    sampler = rb._plain_sampler(0)
    # a launch issued before the write reads the old rows; one issued after reads the new ones
    stall(torch, sampler_stream(rb))
    before = sampler.launch(cap, idxs)
    rb.add_transitions({'observations': torch.full((cap, dim), 2.0, device='cuda'), 'rewards': np.full(cap, 2, np.float32)})
    after = sampler.launch(cap, idxs)
    assert (before.result()['observations'] == 1).all() and (before.result()['rewards'] == 1).all()
    assert (after.result()['observations'] == 2).all() and (after.result()['rewards'] == 2).all()
    # a tensor filled on a side stream right before the call, with no sync, is read with its new values
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        src = torch.zeros((cap, dim), device='cuda')
        torch.cuda._sleep(200_000_000)
        src.fill_(3.0)
        rb.add_transitions({'observations': src, 'rewards': torch.full((cap,), 3.0, device='cuda')})
    assert (rb.sample(cap, idxs)['observations'] == 3).all()
    # sources deleted right after the call, their memory reused by torch, do not change what was written
    stall(torch, sampler_stream(rb))
    src = torch.full((cap, dim), 4.0, device='cuda')
    rb.add_transitions({'observations': src, 'rewards': torch.full((cap,), 4.0, device='cuda')})
    assert len(sampler._in_flight) >= 1                  # the write has not run yet: its sources are still held
    del src
    gc.collect()
    junk = [torch.full((cap, dim), -1.0, device='cuda') for _ in range(4)]
    out = rb.sample(cap, idxs)
    assert (out['observations'] == 4).all() and (out['rewards'] == 4).all()
    del junk
    torch.cuda.synchronize()
    rb.add_transitions({'observations': np.zeros((1, dim), np.float32), 'rewards': np.zeros(1, np.float32)})
    assert len(sampler._in_flight) == 0                  # released at a later call once the writes have completed


@pytest.mark.gpu
def test_refusals():
    import torch

    from ogbench_b200 import Dataset, ReplayBuffer, _native
    from ogbench_b200.datasets import ResidentDataset

    example = {'observations': np.zeros(4, np.float32), 'actions': np.zeros(2, np.float32), 'rewards': np.float64(0)}
    rb = ReplayBuffer.create(example, size=8)
    good = {'observations': torch.zeros((3, 4), device='cuda'), 'actions': torch.zeros((3, 2), device='cuda'),
            'rewards': torch.zeros(3, dtype=torch.float64, device='cuda')}
    rb.add_transitions(good)
    state = (rb.pointer, rb.size)
    with pytest.raises(ValueError, match="'rewards'.*dtype"):
        rb.add_transitions(dict(good, rewards=torch.zeros(3, device='cuda')))                  # float32 for float64: no cast
    with pytest.raises(ValueError, match="'observations'.*shape"):
        rb.add_transitions(dict(good, observations=torch.zeros((3, 5), device='cuda')))
    with pytest.raises(ValueError, match="'observations'.*contiguous"):
        rb.add_transitions(dict(good, observations=torch.zeros((4, 3), device='cuda').t()))
    with pytest.raises(ValueError, match="'actions'.*contiguous"):
        rb.add_transitions(dict(good, actions=torch.zeros((3, 4), device='cuda')[:, ::2]))

    class OtherDevice:                                   # a CUDA array on a GPU this buffer does not live on
        shape = (3, 2)

        def __dlpack_device__(self):
            return (2, 7)

        def __dlpack__(self, stream=None):
            raise AssertionError('not to be exported')

    with pytest.raises(ValueError, match="'actions'.*cuda:7"):
        rb.add_transitions(dict(good, actions=OtherDevice()))
    with pytest.raises(KeyError):
        rb.add_transitions({k: v for k, v in good.items() if k != 'actions'})
    with pytest.raises(ValueError, match='different numbers'):
        rb.add_transitions(dict(good, actions=np.zeros((2, 2), np.float32)))
    with pytest.raises(ValueError, match='leading axis'):
        rb.add_transitions(dict(good, rewards=np.float64(1)))
    assert (rb.pointer, rb.size) == state
    rb.add_transitions({k: v[:0] for k, v in good.items()})                                  # n == 0: nothing happens
    assert (rb.pointer, rb.size) == state
    # the C-ABI: a host pointer flagged as device memory, the field count, row0, skip, and views
    lib = _native.lib()
    sampler = rb._plain_sampler(0)
    host = [np.zeros((1, 4), np.float32), np.zeros((1, 2), np.float32), np.zeros(1, np.float64)]
    ptrs = (C.c_void_p * 3)(*[a.ctypes.data for a in host])
    t, r = C.c_uint64(), C.c_uint64()
    with pytest.raises(ValueError, match='device memory'):
        _native.check(lib.ogb_sampler_write_ring(sampler.ptr, 0, 1, 0, ptrs, 3, (C.c_int32 * 3)(1, 0, 0), None, C.byref(t), C.byref(r)))
    with pytest.raises(ValueError, match='field pointers'):
        _native.check(lib.ogb_sampler_write_ring(sampler.ptr, 0, 1, 0, ptrs, 2, None, None, C.byref(t), C.byref(r)))
    for row0 in (-1, 8):
        with pytest.raises(IndexError):
            _native.check(lib.ogb_sampler_write_ring(sampler.ptr, row0, 1, 0, ptrs, 3, None, None, C.byref(t), C.byref(r)))
    with pytest.raises(ValueError, match='ring'):
        _native.check(lib.ogb_sampler_write_ring(sampler.ptr, 0, 9, 0, ptrs, 3, None, None, C.byref(t), C.byref(r)))
    fields = {'observations': np.zeros((6, 4), np.float32), 'terminals': np.ones(6, np.float32)}
    ds = Dataset.create(**fields)
    view = ResidentDataset(ds.native(0).view(0, 4), list(fields), False, None)._plain_sampler()
    with pytest.raises(ValueError, match='view'):
        _native.check(lib.ogb_sampler_write_ring(view.ptr, 0, 1, 0, ptrs, 2, None, None, C.byref(t), C.byref(r)))

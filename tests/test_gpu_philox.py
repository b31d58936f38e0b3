"""On-device RNG mode: bit-level checks against the numpy restatement of the device's Philox draws, determinism /
stream independence, multi-batch launches, and distributional agreement with the reference's numpy RNG."""

import ctypes as C

import numpy as np
import pytest

from oracle import philox_np
from oracle.replay_oracle import DrawsSource, OracleSampler
from tests.golden.make_golden import cfg, ragged, toy_fields
from tests.gpu_util import device_sampler, to_host

pytestmark = pytest.mark.gpu


def goal_sets_for(config, kind):
    sets = [(0, bool(config['value_geom_sample']), config['discount'], config['value_p_curgoal'] == 1.0)]
    if kind == 'hgc' and config.get('low_discount') is not None:
        sets.append((1, True, config['low_discount'], config['value_p_curgoal'] == 1.0))
    sets.append((2, bool(config['actor_geom_sample']), config['discount'], config['actor_p_curgoal'] == 1.0))
    return sets


def test_philox_words_match_numpy():
    from ogbench_b200 import _native

    n = 1000
    out = np.empty((n, 4), dtype=np.uint32)
    for seed, stream, batch, purpose in [(0, 0, 0, 0), (0xDEADBEEFCAFEF00D, 77, (1 << 40) + 5, 3), (123, 0xFFFFFF, 9, 7)]:
        _native.check(_native.lib().ogb_philox_fill(seed, stream, batch, purpose, n, 0, out.ctypes.data_as(C.c_void_p)))
        want = philox_np.draw4(seed, stream, batch, np.arange(n), purpose)
        for k in range(4):
            assert np.array_equal(out[:, k].astype(np.uint64), want[k]), (seed, k)


@pytest.mark.parametrize('discount', [0.9, 0.99, 0.995, 0.999, 0.9999])
def test_geometric_fast_path_equals_float64_expression(discount):
    """The float32 estimate of ceil(log(1-U)/log(discount)) must never decide differently from the float64
    expression it replaces (it falls back to float64 whenever its error bound reaches an integer boundary)."""
    from ogbench_b200 import _native

    bad = C.c_int64(-1)
    _native.check(_native.lib().ogb_geometric_check(discount, 2024, 1 << 27, 0, C.byref(bad)))
    assert bad.value == 0


CASES = [
    ('gc', (29,), None, {}, np.float32),
    ('gc', (3,), None, dict(value_geom_sample=False, actor_geom_sample=True, actor_p_curgoal=0.2, actor_p_trajgoal=0.3,
                            actor_p_randomgoal=0.5, gc_negative=False), np.float32),
    ('hgc', (7,), None, dict(subgoal_steps=6, discount=0.995), np.float32),
    ('hgc', (7,), None, dict(subgoal_steps=6, low_discount=0.9, value_subgoal_steps=3), np.float32),
    ('gc', (16, 16, 3), 3, dict(p_aug=0.7), np.uint8),
    ('hgc', (16, 16, 3), 2, dict(p_aug=1.0, subgoal_steps=2), np.uint8),
]


@pytest.mark.parametrize('case', CASES, ids=[f'{c[0]}-{"x".join(map(str, c[1]))}-{i}' for i, c in enumerate(CASES)])
def test_philox_mode_is_the_oracle_on_philox_draws(case):
    """The kernel's draws are a pure function of (seed, stream, batch counter, row): rebuild them in numpy, run the
    oracle on them and demand the identical batch.  Rows whose geometric draw sits within 1e-9 of an integer boundary
    (where device log vs numpy log may differ in the last bit) are exempt; there are essentially none."""
    kind, obs_shape, fs, over, dtype = case
    pixel = dtype == np.uint8
    lengths = ragged(5, 10 if pixel else 120, 2, 25 if pixel else 200)
    fields = toy_fields(5, lengths, obs_shape, 4, dtype)
    config = cfg(frame_stack=fs, **over)
    seed, stream_id = 0x1234ABCD5678, 5
    sampler = device_sampler(fields, config, kind, seed=seed, stream_id=stream_id)
    oracle = OracleSampler(fields, config, kind)
    n_choices = len(oracle.valid_table)
    B = 24 if pixel else 512
    for call in range(3):
        evaluation = call == 2
        got = to_host(sampler.sample(B, evaluation=evaluation))
        aug = config['p_aug'] is not None and not evaluation
        draws, knife = philox_np.philox_draws(seed, stream_id, call, B, n_choices, goal_sets_for(config, kind), aug,
                                              config['p_aug'] or 0.0)
        src = DrawsSource(draws)
        want = oracle.sample(B, evaluation=evaluation, source=src)
        assert src.exhausted()
        ok = ~knife
        assert ok.mean() > 0.999
        assert set(got) == set(want)
        for k in want:
            assert got[k].dtype == want[k].dtype and got[k].shape == want[k].shape, k
            assert np.array_equal(got[k][ok], want[k][ok]), (k, call)


def test_undefined_debug_bits_are_refused():
    """ogb_sampler_set_debug defines bits 0, 1 and 3; any other bit (bit 2 selected a kernel that no longer exists) is
    refused with OGB_ERR_INVALID (ValueError) instead of being ignored, and the sampler keeps sampling."""
    fields = toy_fields(21, ragged(21, 30, 5, 60), (29,), 8, np.float32)
    a = device_sampler(fields, cfg(), 'gc', seed=5)
    b = device_sampler(fields, cfg(), 'gc', seed=5)
    b._sampler.set_debug(1 | 2 | 8)
    for bad in (4, 4 | 8, 16, -1):
        with pytest.raises(ValueError, match='debug flags'):
            b._sampler.set_debug(bad)
    b._sampler.set_debug(0)
    x, y = to_host(a.sample(100)), to_host(b.sample(100))
    assert set(x) == set(y)
    for k in x:
        assert np.array_equal(x[k], y[k]), k


def torch_from(x):
    import torch

    return torch.from_dlpack(x).cpu()


def test_sample_many_equals_successive_calls():
    lengths = ragged(7, 60, 2, 90)
    fields = toy_fields(7, lengths, (11,), 3, np.float32)
    config = cfg(subgoal_steps=5)
    a = device_sampler(fields, config, 'hgc', seed=9)
    b = device_sampler(fields, config, 'hgc', seed=9)
    K, B = 5, 96
    many = to_host(a.sample_many(K, B))
    for k in range(K):
        one = to_host(b.sample(B))
        for key in one:
            assert many[key].shape == (K,) + one[key].shape
            assert np.array_equal(many[key][k], one[key]), (key, k)
    assert a.state_dict() == b.state_dict() == {'counter': K}
    single = a.sample_many(1, B)                       # the leading axis is there for one batch as well
    assert single['observations'].shape[:2] == (1, B) and np.asarray(single['rewards']).shape == (1, B)
    assert np.asarray(torch_from(single['observations'])).shape[:2] == (1, B)


def test_counter_checkpoint_and_stream_independence():
    lengths = ragged(8, 40, 2, 60)
    fields = toy_fields(8, lengths, (5,), 2, np.float32)
    config = cfg()
    s0 = device_sampler(fields, config, 'gc', seed=1, stream_id=0)
    first = to_host(s0.sample(256))
    state = s0.state_dict()
    second = to_host(s0.sample(256))
    s0.load_state_dict(state)
    again = to_host(s0.sample(256))
    assert all(np.array_equal(second[k], again[k]) for k in second)          # resume reproduces the stream
    assert not np.array_equal(first['observations'], second['observations'])
    s1 = device_sampler(fields, config, 'gc', seed=1, stream_id=1)           # another rank: another stream
    other = to_host(s1.sample(256))
    assert not np.array_equal(first['observations'], other['observations'])
    s2 = device_sampler(fields, config, 'gc', seed=1, stream_id=0)           # same key: same stream
    same = to_host(s2.sample(256))
    assert all(np.array_equal(first[k], same[k]) for k in first)


def test_distribution_matches_reference_rng():
    """Device Philox mode vs the oracle on numpy's MT19937: same distribution of transitions, goal kinds and offsets."""
    from scipy import stats

    lengths = np.full(400, 251)
    fields = toy_fields(9, lengths, (2,), 2, np.float32)
    fields['observations'][:, 0] = np.arange(len(fields['observations']))    # row id readable from the batch
    config = cfg()
    n = len(fields['terminals'])
    B = 200_000
    dev = to_host(device_sampler(fields, config, 'gc', seed=3).sample(B))
    np.random.seed(0)
    ref = OracleSampler(fields, config, 'gc').sample(B)

    def rows(batch, key):
        return batch[key][:, 0].astype(np.int64)

    for batch in (dev, ref):
        i, vg, ag = rows(batch, 'observations'), rows(batch, 'value_goals'), rows(batch, 'actor_goals')
        assert fields['valids'][i].all()                                      # only valid rows are drawn
        assert np.array_equal(rows(batch, 'next_observations'), i + 1)
        traj = i // 251
        assert (ag // 251 == traj).all() and ((ag > i) | (i % 251 == 249)).all()  # actor goals: future rows of the same trajectory
        assert np.array_equal(batch['masks'], (vg != i).astype(np.float64))
    # transition indices: uniform over valid rows (chi-square on 100 bins, and two-sample KS against the reference)
    i_dev, i_ref = rows(dev, 'observations'), rows(ref, 'observations')
    hist = np.histogram(i_dev, bins=100, range=(0, n))[0]
    assert stats.chisquare(hist).pvalue > 1e-4
    assert stats.ks_2samp(i_dev, i_ref).pvalue > 1e-4
    # goal mix: P(goal == current) = p_cur + (tiny chance of a coincidence); same-trajectory future fraction
    for key, p_cur in (('value_goals', 0.2), ('actor_goals', 0.0)):
        f_dev = np.mean(rows(dev, key) == i_dev)
        f_ref = np.mean(rows(ref, key) == i_ref)
        assert abs(f_dev - f_ref) < 0.005 and abs(f_dev - p_cur) < 0.01, key
    # value-goal offsets of same-trajectory future goals: geometric(0.01) clipped at the trajectory end
    def future_offsets(batch):
        i, g = rows(batch, 'observations'), rows(batch, 'value_goals')
        m = (g > i) & (g // 251 == i // 251)
        return (g - i)[m]
    assert stats.ks_2samp(future_offsets(dev), future_offsets(ref)).pvalue > 1e-4
    # actor goals are uniform in the remainder of the trajectory
    def actor_frac(batch):
        i, g = rows(batch, 'observations'), rows(batch, 'actor_goals')
        final = (i // 251) * 251 + 249
        m = final - i > 20
        return ((g - i - 1) / (final - i - 1 + 1e-9))[m]
    assert stats.ks_2samp(actor_frac(dev), actor_frac(ref)).pvalue > 1e-4


def test_crop_shift_distribution():
    lengths = ragged(10, 8, 3, 12)
    fields = toy_fields(10, lengths, (16, 16, 3), 2, np.uint8)
    config = cfg(frame_stack=None, p_aug=0.5)
    s = device_sampler(fields, config, 'gc', seed=11)
    from ogbench_b200 import _native

    coins, shifts = [], []
    for _ in range(300):
        h = s._sampler.sample_native(64)
        out = np.empty((64, 2), dtype=np.int64)
        _native.check(_native.lib().ogb_batch_crop_shifts(h.ptr, out.ctypes.data_as(C.c_void_p)))
        applied = out[0, 0] >= 0
        assert ((out >= 0).all() if applied else (out == -1).all())       # one coin per batch
        coins.append(applied)
        if applied:
            shifts.append(out)
    assert 0.4 < np.mean(coins) < 0.6
    shifts = np.concatenate(shifts)
    assert shifts.min() == 0 and shifts.max() == 6
    counts = np.stack([np.bincount(shifts[:, k], minlength=7) for k in range(2)])
    assert (np.abs(counts / counts.sum(1, keepdims=True) - 1 / 7) < 0.02).all()


def test_warp_searchsorted_matches_numpy():
    from ogbench_b200 import _native

    rng = np.random.default_rng(0)
    for n in (0, 1, 2, 31, 32, 33, 1000, 4097):
        table = np.sort(rng.integers(0, max(4 * n, 4), size=n)).astype(np.int64)   # with duplicates
        keys = np.concatenate([rng.integers(-2, max(4 * n, 4) + 2, size=500), table[:50]]).astype(np.int64)
        for side, flag in (('left', 0), ('right', 1)):
            out = np.empty(len(keys), dtype=np.int64)
            _native.check(_native.lib().ogb_searchsorted_warp(
                table.ctypes.data_as(C.c_void_p), n, keys.ctypes.data_as(C.c_void_p), len(keys), flag, 0, out.ctypes.data_as(C.c_void_p)))
            assert np.array_equal(out, np.searchsorted(table, keys, side=side)), (n, side)


def test_dlpack_handoff_to_torch():
    import torch

    lengths = ragged(12, 30, 2, 50)
    fields = toy_fields(12, lengths, (6,), 2, np.float32)
    s = device_sampler(fields, cfg(), 'gc', seed=2)
    batch = s.sample(128)
    host = to_host(batch)
    consumer = torch.cuda.Stream()
    with torch.cuda.stream(consumer):
        tensors = {k: torch.from_dlpack(v) for k, v in batch.items()}
    del batch                                                   # the DLPack capsules keep the block alive
    for _ in range(4):
        s.sample(128)                                           # recycled blocks must not clobber exported tensors
    consumer.synchronize()
    for k, t in tensors.items():
        assert t.is_cuda and tuple(t.shape) == host[k].shape
        assert np.array_equal(t.cpu().numpy(), host[k]), k
    assert tensors['masks'].dtype == torch.float64 and tensors['observations'].dtype == torch.float32


def test_full_size_properties_c2():
    """BASELINE shape (1,001,000 x 29): size-independent properties on a 1M-transition launch."""
    from ogbench_b200 import Dataset, GCDataset, synthetic

    w = synthetic.WORKLOADS['c2']
    fields = synthetic.host_fields(w)
    fields['observations'][:, 0] = np.arange(w.rows, dtype=np.float32)      # exact in float32 (< 2^24)
    s = GCDataset(Dataset.create(**fields), w.config, seed=5)
    out = to_host(s.sample_many(64, w.batch))
    i = out['observations'][..., 0].astype(np.int64)
    assert np.array_equal(out['observations'], fields['observations'][i])   # gathers are exact copies
    assert np.array_equal(out['actions'], fields['actions'][i])
    assert (out['valids'] == 1).all() and np.array_equal(out['terminals'], fields['terminals'][i])
    assert np.array_equal(out['next_observations'][..., 0].astype(np.int64), i + 1)
    vg, ag = out['value_goals'][..., 0].astype(np.int64), out['actor_goals'][..., 0].astype(np.int64)
    final = (i // w.steps) * w.steps + w.steps - 2
    assert ((ag > i) | (i == final)).all() and (ag <= final).all()
    assert np.array_equal(out['masks'], (vg != i).astype(np.float64)) and np.array_equal(out['rewards'], out['masks'] * -1.0)
    assert np.array_equal(out['value_goals'], fields['observations'][vg])


def _torch_batch(batch):
    import torch

    return {k: torch.from_dlpack(v) for k, v in batch.items()}


def test_full_size_properties_c3_hgc():
    """BASELINE shape (4,001,000 x 69, HIQL subgoal_steps=25): the HGC index algebra (datasets.py:478-491, :505-619)
    checked on a 1M-transition launch through relations that hold for every row, on the device (no 1 GB host copy)."""
    import torch

    from ogbench_b200 import Dataset, HGCDataset, synthetic

    w = synthetic.WORKLOADS['c3']
    fields = synthetic.device_fields(w)
    n = w.rows
    fields['observations'][:, 0] = torch.arange(n, dtype=torch.float32, device='cuda')      # exact below 2^24
    obs, act = fields['observations'], fields['actions']
    s = HGCDataset(Dataset.create(**fields), w.config, seed=11)
    out = _torch_batch(s.sample_many(1024, w.batch))
    torch.cuda.synchronize()
    k = w.config['subgoal_steps']
    row = lambda key: out[key][..., 0].long().reshape(-1)
    i = row('observations')
    final = (i // w.steps) * w.steps + w.steps - 2
    flat = lambda key: out[key].reshape(-1, *out[key].shape[2:])
    assert torch.equal(flat('observations'), obs[i]) and torch.equal(flat('actions'), act[i])
    assert torch.equal(row('next_observations'), i + 1)
    hv, ha = row('high_value_goals'), row('high_actor_goals')
    assert torch.equal(flat('high_value_goals'), obs[hv]) and torch.equal(flat('value_goals'), obs[hv])
    assert (hv <= torch.maximum(final, hv)).all() and ((ha > i) | (i == final)).all() and (ha <= final).all()
    steps = out['high_value_subgoal_steps'].reshape(-1)
    d = hv - i
    want_steps = torch.minimum(torch.full_like(i, k), final - i)
    want_steps = torch.where((d >= 0) & (d < want_steps), d, want_steps)
    assert torch.equal(steps, want_steps)
    assert torch.equal(row('high_value_next_observations'), i + steps) and torch.equal(row('high_value_actions'), i + steps)
    assert torch.equal(out['high_value_offsets'].reshape(-1), d)
    succ = (steps < k).double()
    assert torch.equal(out['high_value_masks'].reshape(-1), 1.0 - succ)
    lut = torch.from_numpy(-(1 - w.config['discount'] ** np.arange(k + 1)) / (1 - w.config['discount'])).cuda()
    assert torch.equal(out['high_value_rewards'].reshape(-1), lut[steps])                    # numpy-built table, bit-exact
    assert torch.equal(out['low_value_subgoal_steps'].reshape(-1), steps)                    # low_subgoal_steps == subgoal_steps
    assert torch.equal(row('low_actor_goals'), torch.minimum(i + k, final))
    assert torch.equal(out['masks'].reshape(-1), (hv != i).double()) and torch.equal(out['rewards'].reshape(-1), (hv == i).double() - 1.0)
    da = ha - i
    a_steps = torch.minimum(torch.full_like(i, k), final - i)
    a_steps = torch.where((da >= 0) & (da < a_steps), da, a_steps)
    assert torch.equal(row('high_actor_targets'), i + a_steps) and torch.equal(row('low_actor_next_observations'), i + a_steps)


def test_full_size_properties_c5_shard():
    """One 12.5M-row shard of the 100M shape (55-D observations, batch 4096): copies are exact, goals stay inside their
    trajectory, random goals stay inside the shard, and the goal mix has the configured proportions."""
    import torch

    from ogbench_b200 import Dataset, GCDataset, synthetic

    w = synthetic.WORKLOADS['c5']
    fields = synthetic.device_fields(w)
    n = w.rows
    fields['observations'][:, 0] = torch.arange(n, dtype=torch.float32, device='cuda')      # 12,512,500 < 2^24
    obs, act = fields['observations'], fields['actions']
    s = GCDataset(Dataset.create(**fields), w.config, seed=3, stream_id=6)
    out = _torch_batch(s.sample_many(256, w.batch))
    torch.cuda.synchronize()
    row = lambda key: out[key][..., 0].long().reshape(-1)
    flat = lambda key: out[key].reshape(-1, *out[key].shape[2:])
    i, vg, ag = row('observations'), row('value_goals'), row('actor_goals')
    assert torch.equal(flat('observations'), obs[i]) and torch.equal(flat('actions'), act[i])
    assert torch.equal(flat('value_goals'), obs[vg]) and torch.equal(flat('actor_goals'), obs[ag])
    assert torch.equal(row('next_observations'), i + 1)
    assert (flat('valids') == 1).all() and (i % w.steps != w.steps - 1).all()                # only valid rows are drawn
    final = (i // w.steps) * w.steps + w.steps - 2
    assert ((ag > i) | (i == final)).all() and (ag <= final).all()                           # actor goals: trajectory future
    assert (vg >= 0).all() and (vg < n).all() and (vg % w.steps != w.steps - 1).all()        # goals are valid rows of the shard
    same_traj = (vg // w.steps) == (i // w.steps)
    cur = (vg == i).double().mean().item()
    assert abs(cur - 0.2) < 0.01                                                             # value_p_curgoal (+ tiny geometric mass at 0? no: offsets >= 1)
    assert abs((same_traj & (vg > i)).double().mean().item() - 0.5) < 0.02                   # value_p_trajgoal (random goals rarely land in the same trajectory)
    assert torch.equal(out['masks'].reshape(-1), (vg != i).double())


def test_full_size_pixels_c4():
    """BASELINE shape (1,001,000 x 64x64x3 uint8, 12.3 GB resident, frame_stack=3, crop): every key of an augmented batch
    against a torch restatement of datasets.py:359-366 (stack) and :17-33 (edge-padded crop) on the same rows/shifts."""
    import ctypes as C

    import torch

    from ogbench_b200 import Dataset, GCDataset, _native, synthetic

    w = synthetic.WORKLOADS['c4']
    fields = synthetic.device_fields(w)
    frames = fields['observations']
    s = GCDataset(Dataset.create(**fields), dict(w.config, p_aug=1.0), seed=8)
    s._sampler.set_debug(1)
    B, K = w.batch, 4
    handle = s._sampler.sample_native(B, n_batches=K)
    out = _torch_batch(s._sampler.wrap(handle))
    torch.cuda.synchronize()
    n = B * K
    lib = _native.lib()
    crop = np.empty((n, 2), dtype=np.int64)
    _native.check(lib.ogb_batch_crop_shifts(handle.ptr, crop.ctypes.data_as(C.c_void_p)))
    assert (crop >= 0).all() and (crop <= 6).all() and len(np.unique(crop, axis=0)) > 20   # p_aug = 1: every batch is cropped
    dy = torch.from_numpy(crop[:, 0] - 3).cuda()
    dx = torch.from_numpy(crop[:, 1] - 3).cuda()
    ar = torch.arange(64, device='cuda')
    ys = (ar[None, :] + dy[:, None]).clamp(0, 63)            # out[y, x] = img[clip(y + cy - 3), clip(x + cx - 3)]
    xs = (ar[None, :] + dx[:, None]).clamp(0, 63)

    def expected(slot):
        idx = np.empty(n, dtype=np.int64)
        _native.check(lib.ogb_batch_index_vector(handle.ptr, slot, idx.ctypes.data_as(C.c_void_p)))
        i = torch.from_numpy(idx).cuda()
        first = (torch.clamp(i, max=w.rows - 1) // w.steps) * w.steps
        first = torch.where(i % w.steps == w.steps - 1, i, first)       # a trajectory's last row starts its own segment (quirk 2)
        stack = torch.cat([frames[torch.maximum(i - k, first)] for k in (2, 1, 0)], dim=-1)   # oldest frame first
        rows = torch.arange(n, device='cuda')[:, None, None]
        return stack[rows, ys[:, :, None], xs[:, None, :]]

    for key, slot in (('observations', 0), ('next_observations', 1), ('value_goals', 2), ('actor_goals', 3)):
        got = out[key].reshape(n, 64, 64, 9)
        assert torch.equal(got, expected(slot)), key


@pytest.mark.parametrize('output', ['device', 'numpy'])
def test_prefetcher_returns_the_direct_call_sequence(output):
    """Prefetcher (batches drawn by a worker thread, ahead of the consumer) yields exactly the batches that direct
    sample() calls on a sampler with the same seed return, in order."""
    from ogbench_b200 import Dataset, GCDataset, Prefetcher
    from tests.golden.make_golden import cfg, ragged, toy_fields

    fields = toy_fields(77, ragged(77, 50, 5, 60), (9,), 3, np.float32)
    config = cfg()
    direct = GCDataset(Dataset.create(**{k: v.copy() for k, v in fields.items()}), config, seed=5, output=output)
    ahead = GCDataset(Dataset.create(**{k: v.copy() for k, v in fields.items()}), config, seed=5, output=output)
    with Prefetcher(ahead, 64, depth=3) as batches:
        for step in range(12):
            want, got = direct.sample(64), next(batches)
            assert set(want) == set(got)
            for k in want:
                assert np.array_equal(np.asarray(want[k]), np.asarray(got[k])), (step, k)


def test_current_device_is_left_alone():
    """The library switches to the dataset's device inside its entry points and restores the caller's current device
    (needs two GPUs: the sampler lives on cuda:0 while the calling thread's current device is cuda:1)."""
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip('needs two GPUs')
    fields = toy_fields(3, ragged(3, 40, 5, 60), (9,), 3, np.float32)
    config = cfg()
    torch.cuda.set_device(1)
    here = device_sampler(fields, config, 'gc', seed=11, device=0)
    assert torch.cuda.current_device() == 1
    got = to_host(here.sample(256))
    assert torch.cuda.current_device() == 1
    torch.cuda.set_device(0)
    there = device_sampler(fields, config, 'gc', seed=11, device=0)
    want = to_host(there.sample(256))
    for k in want:
        assert np.array_equal(got[k], want[k]), k
    del here, there, got, want
    import gc

    torch.cuda.set_device(1)
    gc.collect()                                      # batches and samplers of cuda:0 are released from a cuda:1 thread
    assert torch.cuda.current_device() == 1
    torch.cuda.set_device(0)


@pytest.mark.parametrize('kind,obs_dim,K,B', [('gc', 29, 300, 1024), ('gc', 55, 97, 4096), ('hgc', 69, 150, 1024), ('gc', 29, 211, 1000)])
def test_ticket_scheduled_tiles_equal_static_tiles(kind, obs_dim, K, B):
    """Big launches hand their 32-row tiles to the warps through a ticket counter (relabel_rows.cuh, `sched`); debug bit 3
    restores the fixed stride.  The two must return the same bytes: several thousand tiles per launch (more tiles than
    warps, so tickets name real tiles), fused GC and un-fused HGC launches, a ragged last tile (211 x 1000 rows), launches
    repeated so that the counters a launch leaves behind are reused, and the canary fill proving every byte of every key was
    written exactly where it belongs."""
    import ctypes as C
    from ogbench_b200 import _native

    lengths = ragged(31, 400, 30, 300)
    fields = toy_fields(31, lengths, (obs_dim,), 8, np.float32)
    config = cfg(subgoal_steps=7) if kind == 'hgc' else cfg()
    a = device_sampler(fields, config, kind, seed=11)
    b = device_sampler(fields, config, kind, seed=11)
    a._sampler.set_debug(2)          # tickets + canary
    b._sampler.set_debug(2 | 8)      # static tiles + canary
    for rep in range(3):
        ha = a._sampler.sample_native(B, n_batches=K)
        hb = b._sampler.sample_native(B, n_batches=K)
        for h in (ha, hb):
            bad = C.c_int64(-1)
            _native.check(_native.lib().ogb_batch_check_gaps(h.ptr, C.byref(bad)))
            assert bad.value == 0
        x, y = to_host(a._sampler.wrap(ha)), to_host(b._sampler.wrap(hb))
        assert set(x) == set(y)
        for k in x:
            assert not (x[k].view(np.uint8) == 0xA5).all(), k
            assert np.array_equal(x[k], y[k]), (k, rep)


@pytest.mark.parametrize('obs_dim,extra_dim', [(16, None), (29, 40), (2, None)])
def test_plain_dataset_big_launch_equals_numpy_indexing(obs_dim, extra_dim):
    """Dataset.sample / get_subset (datasets.py:72-83) on a launch with more tiles than warps: the plain flavour of the
    fused kernel also takes its tiles from the ticket counter (a one-pair launch -- a single record span, 64-byte rows =
    one item per tile -- resolves its ticket in the very item that asked for it).  Explicit idxs, every field against
    numpy fancy indexing, twice (the counters a launch leaves behind are reused)."""
    from ogbench_b200 import Dataset

    rng = np.random.default_rng(obs_dim)
    n = 50_000
    fields = dict(observations=rng.standard_normal((n, obs_dim)).astype(np.float32),
                  actions=rng.standard_normal((n, 3)).astype(np.float32),
                  terminals=(rng.random(n) < 0.01).astype(np.float32), rewards=rng.standard_normal(n).astype(np.float32))
    fields['terminals'][-1] = 1.0
    if extra_dim:
        fields['qpos'] = rng.standard_normal((n, extra_dim)).astype(np.float32)
    ds = Dataset.create(**fields)
    for rep in range(2):
        idxs = rng.integers(0, n, size=301_117)
        got = to_host(ds.sample(len(idxs), idxs=idxs))
        assert set(got) == set(fields) | {'next_observations'}
        for k, v in fields.items():
            assert np.array_equal(got[k], v[idxs]), (k, rep)
        assert np.array_equal(got['next_observations'], fields['observations'][np.minimum(idxs + 1, n - 1)]), rep

"""GPU parity: the CUDA sampler (through the C-ABI) against the golden vectors and the oracle, bit-exact."""

import numpy as np
import pytest

from tests.golden.make_golden import cfg, ragged, toy_fields
from tests.golden_util import assert_batches_identical, case_names, load_case
from tests.gpu_util import device_sample, device_sampler, draws_from_log, oracle_with_draws, to_host

pytestmark = pytest.mark.gpu
CASES = case_names()


@pytest.mark.parametrize('name', CASES)
def test_validation_mode_matches_golden(name):
    """The device consumes the reference's recorded draws and must return the reference's batch, every key."""
    case = load_case(name)
    sampler = device_sampler(case['fields'], case['cfg'], case['kind'])
    got = device_sample(sampler, case, draws=draws_from_log(case))
    assert_batches_identical(to_host(got), case['out'], label=name + ':')


@pytest.mark.parametrize('name', list(CASES))
def test_numpy_rng_mode_matches_golden(name):
    """rng='numpy': same np.random.seed as the reference run -> same batch, with no recording in between.
    (TRL agents included: their midpoint draw randint(idxs, value_goal_idxs), datasets.py:259, is made on the host
    between two device phases.)"""
    case = load_case(name)
    sampler = device_sampler(case['fields'], case['cfg'], case['kind'], rng='numpy', output='numpy')
    np.random.seed(case['meta']['seed'])
    got = device_sample(sampler, case)
    assert_batches_identical(got, case['out'], label=name + ':')


@pytest.mark.parametrize('name', ['gc_state_gcivl', 'hgc_state_hiql', 'hgc_pixel_fs3_aug'])
def test_no_dedup_matches_golden(name):
    case = load_case(name)
    sampler = device_sampler(case['fields'], case['cfg'], case['kind'], dedup=False)
    got = sampler.sample(case['B'], idxs=case['idxs'], evaluation=case['evaluation'], draws=draws_from_log(case))
    assert_batches_identical(to_host(got), case['out'], label=name + ':')


SWEEP = [
    # kind, pixel, obs_shape, frame_stack, overrides
    ('gc', False, (29,), None, {}),
    ('gc', False, (2,), None, dict(value_geom_sample=False, actor_geom_sample=True, actor_p_curgoal=0.2, actor_p_trajgoal=0.3, actor_p_randomgoal=0.5)),
    ('gc', False, (7,), 3, {}),                        # frame stacking of vector observations
    ('gc', False, (3, 5), 2, {}),                      # ... and of rank-3 fields
    ('hgc', False, (69,), None, dict(subgoal_steps=25, discount=0.995)),
    ('hgc', False, (55,), None, dict(subgoal_steps=4, value_geom_sample=False, actor_geom_sample=True, gc_negative=False,
                                      actor_p_curgoal=0.0, actor_p_trajgoal=0.5, actor_p_randomgoal=0.5, discount=0.999)),
    ('hgc', False, (6,), None, dict(subgoal_steps=9, low_discount=0.95, low_subgoal_steps=2)),
    ('gc', True, (64, 64, 3), 3, dict(p_aug=0.5)),
    ('gc', True, (32, 48, 3), 3, dict(p_aug=1.0)),
    ('gc', True, (64, 64, 3), None, dict(p_aug=1.0)),
    ('gc', True, (64, 64, 3), 4, dict(p_aug=1.0)),
    ('hgc', True, (64, 64, 3), 3, dict(p_aug=0.5, subgoal_steps=3)),
    ('gc', True, (20, 12, 4), 3, dict(p_aug=1.0)),    # not TMA-eligible: generic frame kernel
    ('gc', True, (8, 8, 3), 2, dict(p_aug=1.0)),      # not TMA-eligible (W % 16)
]


@pytest.mark.parametrize('spec', SWEEP, ids=[f'{s[0]}-{"x".join(map(str, s[2]))}-fs{s[3]}-{i}' for i, s in enumerate(SWEEP)])
def test_oracle_sweep(spec):
    """Seeded ragged datasets at sizes the oracle finishes in seconds; several batches, both evaluation modes."""
    kind, pixel, obs_shape, fs, over = spec
    seed = abs(hash(str(spec))) % 1000
    lengths = ragged(seed, 12 if pixel else 200, 2, 20 if pixel else 300)
    fields = toy_fields(seed, lengths, obs_shape, 5, np.uint8 if pixel else np.float32)
    config = cfg(frame_stack=fs, **over)
    sampler = device_sampler(fields, config, kind, rng='numpy', output='numpy')
    B = 37 if pixel else 1024
    for it, evaluation in enumerate([False, False, True, False]):
        np.random.seed(seed * 10 + it)
        _, want = oracle_with_draws(fields, config, kind, B, evaluation=evaluation)
        np.random.seed(seed * 10 + it)
        got = sampler.sample(B, evaluation=evaluation)
        assert_batches_identical(got, want, label=f'{spec}/{it}:')


LONG = [
    ('gc', (29,), None, {}),
    ('gc', (2,), None, dict(value_geom_sample=False, actor_geom_sample=True, actor_p_curgoal=0.2, actor_p_trajgoal=0.3, actor_p_randomgoal=0.5)),
    ('hgc', (11,), None, dict(subgoal_steps=7, discount=0.995)),
    ('hgc', (6,), None, dict(subgoal_steps=9, low_discount=0.95, low_subgoal_steps=2)),
    ('gc', (7,), 3, {}),
]


@pytest.mark.parametrize('spec', LONG, ids=[f"{s[0]}-{s[1][0]}-fs{s[2]}-{i}" for i, s in enumerate(LONG)])
@pytest.mark.parametrize('layout', ['compact', 'early_terminals', 'extra_invalid'])
def test_oracle_sweep_long_trajectories(spec, layout):
    """Trajectories of 18+ rows take the one-probe segment table (valid row and final state from one lookup,
    relabel_rows.cuh valid_row_fast); 'early_terminals' puts extra terminals inside trajectories, so the table has to
    be refused and the general searches used; 'extra_invalid' adds invalid rows in the middle of trajectories."""
    kind, obs_shape, fs, over = spec
    seed = abs(hash(str(spec) + layout)) % 1000
    lengths = ragged(seed, 150, 18, 90)
    fields = toy_fields(seed, lengths, obs_shape, 5, np.float32)
    rng = np.random.default_rng(seed)
    if layout == 'early_terminals':
        extra = rng.choice(len(fields['terminals']), size=40, replace=False)
        fields['terminals'] = fields['terminals'].copy()
        fields['terminals'][extra] = 1.0
    elif layout == 'extra_invalid':
        starts = np.concatenate([[0], np.cumsum(lengths)[:-1]])
        fields['valids'] = fields['valids'].copy()
        fields['valids'][starts[::3] + 8] = 0.0          # far from every other invalid row: the table stays usable
    config = cfg(frame_stack=fs, **over)
    sampler = device_sampler(fields, config, kind, rng='numpy', output='numpy')
    for it, evaluation in enumerate([False, True, False]):
        np.random.seed(seed * 10 + it)
        _, want = oracle_with_draws(fields, config, kind, 1024, evaluation=evaluation)
        np.random.seed(seed * 10 + it)
        got = sampler.sample(1024, evaluation=evaluation)
        assert_batches_identical(got, want, label=f'{spec}/{layout}/{it}:')
    # the on-device RNG mode must agree with the oracle fed the restated Philox draws on these layouts too
    from oracle import philox_np
    from oracle.replay_oracle import DrawsSource, OracleSampler
    from tests.test_gpu_philox import goal_sets_for

    dev = device_sampler(fields, config, kind, seed=77, stream_id=3)
    oracle = OracleSampler(fields, config, kind)
    got = to_host(dev.sample(512))
    draws, knife = philox_np.philox_draws(77, 3, 0, 512, len(oracle.valid_table), goal_sets_for(config, kind), True, 0.0)
    want = oracle.sample(512, source=DrawsSource(draws))
    for k in want:
        assert np.array_equal(got[k][~knife], want[k][~knife]), (k, layout)


CANARY = [
    # kind, obs_shape, obs dtype, act_dim, frame_stack, batch, n_batches
    ('gc', (29,), np.float32, 8, None, 1000, 1),      # ragged last warp tile
    ('gc', (29,), np.float32, 8, None, 33, 40),       # batch not a multiple of 32, many batches
    ('gc', (2,), np.float32, 2, None, 77, 5),         # everything tiny: index kernel only
    ('hgc', (69,), np.float32, 21, None, 250, 3),     # long rows: 16-row items, split launch
    ('hgc', (55,), np.float32, 5, None, 4096, 9),     # big enough for the auxiliary-stream path (>= 32768 rows)
    ('gc', (7,), np.float16, 3, None, 129, 3),        # 14-byte rows, 12-byte actions: everything tiny, index kernel only
    ('gc', (13,), np.uint8, 5, None, 95, 2),          # 13-byte rows: byte drain inside the record span (goal rows tiny)
    ('gc', (9,), np.float16, 3, None, 129, 3),        # 18-byte rows: two-byte element drain, goal rows too
    ('gc', (17,), np.uint8, 5, None, 95, 2),          # 17-byte rows: byte drain, goal rows too
    ('gc', (64, 64, 3), np.uint8, 5, 3, 19, 2),       # frames (TMA) + small record span
    ('gc', (20, 12, 4), np.uint8, 5, 3, 21, 1),       # frames (generic kernel)
    ('gc', (300,), np.float32, 4, None, 64, 2),       # 1200-byte rows: few rows per stage
    ('gc', (1100,), np.float32, 4, None, 40, 1),      # 4400-byte rows: register-staged kernel
]


@pytest.mark.parametrize('spec', CANARY, ids=[f'{s[0]}-{"x".join(map(str, s[1]))}-{np.dtype(s[2]).name}-B{s[5]}x{s[6]}' for s in CANARY])
def test_no_writes_outside_the_keys(spec):
    """Canary mode: the batch block is filled with 0xA5 before the kernels run; afterwards every byte that belongs to no
    key (the alignment gaps between keys) must be untouched, and gathered keys must be exact copies of dataset rows."""
    import ctypes as C
    from ogbench_b200 import _native

    kind, obs_shape, dtype, act_dim, fs, B, K = spec
    pixel = len(obs_shape) == 3
    seed = abs(hash(str(spec))) % 1000
    lengths = ragged(seed, 12 if pixel else 160, 4, 20 if pixel else 120)
    fields = toy_fields(seed, lengths, obs_shape, act_dim, dtype)
    if np.dtype(dtype) == np.float16:
        fields['observations'] = np.random.default_rng(seed).standard_normal((len(fields['terminals']), *obs_shape)).astype(np.float16)
    config = cfg(frame_stack=fs, p_aug=0.5 if pixel else 0.0, subgoal_steps=5)
    sampler = device_sampler(fields, config, kind, seed=seed)
    sampler._sampler.set_debug(3)
    for evaluation in (False, True):
        handle = sampler._sampler.sample_native(B, n_batches=K, evaluation=evaluation)
        bad = C.c_int64(-1)
        _native.check(_native.lib().ogb_batch_check_gaps(handle.ptr, C.byref(bad)))
        assert bad.value == 0, (spec, evaluation)
        out = to_host(sampler._sampler.wrap(handle))
        n = B * K
        idx = np.empty(n, dtype=np.int64)
        _native.check(_native.lib().ogb_batch_index_vector(handle.ptr, 0, idx.ctypes.data_as(C.c_void_p)))
        assert np.array_equal(out['actions'].reshape(n, -1), fields['actions'][idx])
        assert np.array_equal(out['terminals'].reshape(n), fields['terminals'][idx])
        if fs is None:
            assert np.array_equal(out['observations'].reshape(n, *obs_shape), fields['observations'][idx])
            nxt = np.minimum(idx + 1, len(fields['terminals']) - 1)      # datasets.py:82 (from the record's shadow copy when it has one)
            assert np.array_equal(out['next_observations'].reshape(n, *obs_shape), fields['observations'][nxt])


def test_mixed_dtypes_against_oracle():
    """float64 observations, discrete int32 actions (powderworld, ogbench/utils.py:197-198), extra int64 / bool / 2-D
    fields: every dataset field is gathered at the sampled rows (datasets.py:78-83), whatever its dtype."""
    rng = np.random.default_rng(3)
    lengths = ragged(3, 120, 18, 70)
    base = toy_fields(3, lengths, (9,), 2, np.float32)
    n = len(base['terminals'])
    fields = dict(base, observations=rng.standard_normal((n, 9)), actions=rng.integers(0, 5, n).astype(np.int32),
                  step_id=np.arange(n, dtype=np.int64), flag=rng.integers(0, 2, n).astype(bool),
                  qpos=rng.standard_normal((n, 3, 2)).astype(np.float32))
    config = cfg()
    for kind in ('gc', 'hgc'):
        c = dict(config, subgoal_steps=6) if kind == 'hgc' else config
        sampler = device_sampler(fields, c, kind, rng='numpy', output='numpy')
        for it in range(2):
            np.random.seed(40 + it)
            _, want = oracle_with_draws(fields, c, kind, 777)
            np.random.seed(40 + it)
            got = sampler.sample(777)
            assert_batches_identical(got, want, label=f'mixed/{kind}/{it}:')


@pytest.mark.parametrize('rng_mode', ['numpy', 'philox'])
def test_long_rows_with_many_small_fields_fill_the_item_tables(rng_mode):
    """1,200-byte observation rows (four rows per pipeline stage -> eight items per tile and job) next to a dozen small
    per-transition fields that share the transition's record span: 150 entries in the per-launch output table and 32 items,
    both Philox (the 2 x 16 fused shape) and injected draws (3 x 8), ragged last tile included."""
    from oracle import philox_np
    from oracle.replay_oracle import DrawsSource, OracleSampler
    from tests.test_gpu_philox import goal_sets_for

    rng = np.random.default_rng(13)
    lengths = ragged(13, 60, 9, 50)
    fields = toy_fields(13, lengths, (300,), 4, np.float32)
    n = len(fields['terminals'])
    for j in range(12):
        fields[f'extra_{j:02d}'] = rng.standard_normal((n, 1 + j % 2)).astype(np.float32) if j % 3 else rng.integers(0, 9, n).astype(np.int32)
    config = cfg()
    B = 1000 + 13
    if rng_mode == 'numpy':
        sampler = device_sampler(fields, config, 'gc', rng='numpy', output='numpy')
        np.random.seed(5)
        _, want = oracle_with_draws(fields, config, 'gc', B)
        np.random.seed(5)
        assert_batches_identical(sampler.sample(B), want, label='long rows/numpy:')
    else:
        sampler = device_sampler(fields, config, 'gc', seed=17, stream_id=4)
        oracle = OracleSampler(fields, config, 'gc')
        got = to_host(sampler.sample(B))
        draws, knife = philox_np.philox_draws(17, 4, 0, B, len(oracle.valid_table), goal_sets_for(config, 'gc'), True, 0.0)
        want = oracle.sample(B, source=DrawsSource(draws))
        assert set(got) == set(want)
        for k in want:
            assert got[k].dtype == want[k].dtype and np.array_equal(got[k][~knife], want[k][~knife]), k


@pytest.mark.parametrize('kind', ['gc', 'hgc'])
def test_large_batch_numpy_rng_matches_oracle(kind):
    """One sample() of 40,000 rows (>= 32,768: the big-launch code paths -- auxiliary stream, persistent index kernel with
    the segment table in shared memory for HGC, fused launch for GC) in the mode that replays np.random."""
    lengths = ragged(41, 400, 25, 120)
    fields = toy_fields(41, lengths, (13,), 4, np.float32)
    config = cfg(subgoal_steps=9)
    sampler = device_sampler(fields, config, kind, rng='numpy', output='numpy')
    for it in range(2):
        np.random.seed(500 + it)
        _, want = oracle_with_draws(fields, config, kind, 40000)
        np.random.seed(500 + it)
        got = sampler.sample(40000)
        assert_batches_identical(got, want, label=f'large/{kind}/{it}:')

@pytest.mark.gpu
@pytest.mark.parametrize('output', ['device', 'numpy'])
def test_cached_key_layout_across_calls(output):
    """The Python wrapper reads a batch's key layout once per call shape and reuses it (`_Sampler.wrap`): successive calls
    of alternating shapes, with and without given idxs, must keep returning the oracle's arrays."""
    lengths = ragged(43, 60, 5, 40)
    fields = toy_fields(43, lengths, (6,), 3, np.float32)
    config = cfg(subgoal_steps=4)
    for kind in ('gc', 'hgc'):
        sampler = device_sampler(fields, config, kind, rng='numpy', output=output)
        for it, B in enumerate([100, 37, 100, 37, 1, 100]):
            idxs = np.arange(B) * 2 if it in (2, 3) else None
            np.random.seed(900 + it)
            _, want = oracle_with_draws(fields, config, kind, B, idxs=idxs, evaluation=(it == 5))
            np.random.seed(900 + it)
            got = sampler.sample(B, idxs=idxs, evaluation=(it == 5))
            assert_batches_identical(to_host(got), want, label=f'layout/{kind}/{it}:')
        assert len(sampler._sampler._layouts) == 4      # (100), (37), (1), (100, evaluation)


@pytest.mark.parametrize('output', ['device', 'numpy'])
def test_empty_batch_like_the_reference(output):
    """sample(0), sample(idxs=[]) and the helper methods on empty index arrays return every key with zero rows, with the
    reference's shapes and dtypes (np.random.randint(n, size=0) there; checked against the unmodified reference when the
    oracle was written -- the oracle reproduces it)."""
    lengths = ragged(47, 8, 4, 9)
    fields = toy_fields(47, lengths, (3,), 2, np.float32)
    config = cfg(subgoal_steps=3)
    for kind in ('gc', 'hgc'):
        for rng in ('philox', 'numpy'):
            sampler = device_sampler(fields, config, kind, rng=rng, output=output)
            np.random.seed(3)
            _, want = oracle_with_draws(fields, config, kind, 0)
            for got in (sampler.sample(0), sampler.sample(5, idxs=np.zeros(0, dtype=np.int64))):
                got = to_host(got)
                assert set(got) == set(want)
                for k in want:
                    assert got[k].shape == want[k].shape and got[k].dtype == want[k].dtype, (kind, rng, k)
            assert np.asarray(sampler.get_observations(np.zeros(0, dtype=np.int64))).shape == (0, 3)
            assert sampler.sample_goals(np.zeros(0, dtype=np.int64), 0.2, 0.5, 0.3, True).shape == (0,)
            nonempty = to_host(sampler.sample(4))                   # and the sampler keeps working afterwards
            assert nonempty['observations'].shape == (4, 3)


def test_index_vectors_exposed():
    case = load_case('hgc_state_hiql')
    sampler = device_sampler(case['fields'], case['cfg'], 'hgc')
    sampler._sampler.set_debug(True)
    from oracle.replay_oracle import OracleSampler, ReplaySource
    import ctypes as C
    from ogbench_b200 import _native

    o = OracleSampler(case['fields'], case['cfg'], 'hgc')
    o.sample(case['B'], source=ReplaySource(case['log']))
    handle = sampler._sampler.sample_native(case['B'], draws=o.last_draws)
    names = ['idxs', None, 'hv_goal', 'hv_next', 'lv_next', 'ha_goal', 'ha_next', 'la_goal', 'la_next']
    for slot, nm in enumerate(names):
        if nm is None:
            continue
        out = np.empty(case['B'], dtype=np.int64)
        _native.check(_native.lib().ogb_batch_index_vector(handle.ptr, slot, out.ctypes.data_as(C.c_void_p)))
        assert np.array_equal(out, o.last_index_vectors[nm]), nm


def test_given_idxs_out_of_range_raises():
    case = load_case('gc_state_gcivl')
    sampler = device_sampler(case['fields'], case['cfg'], 'gc')
    with pytest.raises(IndexError):
        sampler.sample(2, idxs=np.array([0, sampler.size]))


def test_given_idxs_out_of_range_raises_in_host_output_mode():
    """output='numpy': the kernel range-checks the given indices (no host scan) and the IndexError still comes out of
    the same sample() call; a following valid call is unaffected."""
    case = load_case('gc_state_gcivl')
    sampler = device_sampler(case['fields'], case['cfg'], 'gc', output='numpy')
    for bad in ([0, sampler.size], [-1, 3], [2 ** 40, 1]):
        with pytest.raises(IndexError):
            sampler.sample(2, idxs=np.array(bad))
    good = sampler.sample(3, idxs=np.array([0, 1, 2]))
    assert np.array_equal(good['observations'], case['fields']['observations'][:3])


def test_constructor_asserts():
    from ogbench_b200 import Dataset, GCDataset

    case = load_case('gc_state_gcivl')
    with pytest.raises(AssertionError):
        Dataset.create(actions=case['fields']['actions'])
    bad = dict(case['cfg'], value_p_curgoal=0.5)
    with pytest.raises(AssertionError):
        device_sampler(case['fields'], bad, 'gc')
    fields = dict(case['fields'])
    fields['terminals'] = fields['terminals'].copy()
    fields['terminals'][-1] = 0.0
    with pytest.raises(AssertionError):
        device_sampler(fields, case['cfg'], 'gc')
    reg = load_case('gc_state_regular')
    with pytest.raises(AssertionError):
        device_sampler(reg['fields'], dict(reg['cfg'], frame_stack=3), 'gc')
    with pytest.raises(KeyError):
        GCDataset(Dataset.create(**case['fields']), {k: v for k, v in case['cfg'].items() if k != 'discount'})


def test_plain_dataset_sample_and_subset():
    """Dataset.sample / get_subset (datasets.py:72-83) on device."""
    from ogbench_b200 import Dataset

    case = load_case('gc_state_gcivl')
    ds = Dataset.create(**{k: v.copy() for k, v in case['fields'].items()})
    idxs = np.array([0, 5, ds.size - 1, 17])
    got = to_host(ds.get_subset(idxs))
    for k, v in case['fields'].items():
        assert np.array_equal(got[k], v[idxs])
    assert np.array_equal(got['next_observations'], case['fields']['observations'][np.minimum(idxs + 1, ds.size - 1)])


def test_get_observations_helpers():
    """get_observations / get_goal_observations / get_stacked_observations (datasets.py:341-366) for explicit rows."""
    from oracle.replay_oracle import OracleSampler

    for name in ('gc_pixel_fs3_aug', 'gc_state_oracle_reps', 'hgc_state_hiql'):
        case = load_case(name)
        sampler = device_sampler(case['fields'], case['cfg'], case['kind'])
        oracle = OracleSampler(case['fields'], case['cfg'], case['kind'])
        n = len(case['fields']['terminals'])
        idxs = np.array([0, 1, 2, n - 1, n // 2, 3, 3])
        assert np.array_equal(np.asarray(sampler.get_observations(idxs)), oracle._obs(idxs)), name
        assert np.array_equal(np.asarray(sampler.get_goal_observations(idxs)), oracle._goal(idxs)), name
        if case['cfg']['frame_stack'] is not None:
            assert np.array_equal(np.asarray(sampler.get_stacked_observations(idxs)), oracle._obs(idxs)), name


def test_reference_helper_methods():
    """sample_goals, compute_high_next_idxs, get_high_actions, augment (datasets.py:296-339, :478-494) as public methods,
    computed on the device, against the oracle's restatement under the same np.random state."""
    from oracle.replay_oracle import (NumpyGlobalSource, OracleSampler, final_rows, pick_goals, shifted_edge_crop,
                                      subgoal_step)

    for layout_seed, lo_len in ((31, 2), (32, 20)):      # ragged short trajectories (general searches) and long ones (segment table)
        lengths = ragged(layout_seed, 80, lo_len, 90)
        fields = toy_fields(layout_seed, lengths, (6,), 3, np.float32)
        config = cfg(subgoal_steps=7)
        sampler = device_sampler(fields, config, 'hgc', rng='numpy', output='numpy')
        oracle = OracleSampler(fields, config, 'hgc')
        rng = np.random.default_rng(layout_seed)
        idxs = oracle.valid_table[rng.integers(0, len(oracle.valid_table), 500)]
        final = final_rows(oracle.terminal_locs, idxs)
        for p_cur, p_traj, p_rand, geom, disc in ((0.2, 0.5, 0.3, True, None), (0.0, 1.0, 0.0, False, None), (1.0, 0.0, 0.0, True, 0.9),
                                                  (0.1, 0.3, 0.6, False, 0.95)):
            np.random.seed(77)
            want, _ = pick_goals(idxs, final, oracle.valid_table, p_cur, p_traj, geom, config['discount'] if disc is None else disc,
                                 NumpyGlobalSource(), oracle.size)
            np.random.seed(77)
            got = sampler.sample_goals(idxs, p_cur, p_traj, p_rand, geom, discount=disc)
            assert got.dtype == np.int64 and np.array_equal(got, want), (layout_seed, p_cur, geom)
        goals = oracle.valid_table[rng.integers(0, len(oracle.valid_table), 500)]
        goals[::3] = np.minimum(idxs[::3] + rng.integers(0, 12, len(idxs[::3])), final[::3])
        for k in (1, 7, 1000):
            want_next, want_steps = subgoal_step(idxs, final, goals, k)
            got_next, got_steps = sampler.compute_high_next_idxs(idxs, final, goals, k)
            assert np.array_equal(got_next, want_next) and np.array_equal(got_steps, want_steps), k
        assert np.array_equal(sampler.get_high_actions(idxs[:9], idxs[:9]), fields['observations'][idxs[:9]])
        # the on-device RNG mode returns goals with the right structure
        dev = device_sampler(fields, config, 'hgc', seed=3)
        g = dev.sample_goals(idxs, 0.0, 1.0, 0.0, True)
        assert ((g > idxs) | (idxs == final)).all() and (g <= final).all()

    # augment: one shift per sample shared by the keys, non-image keys untouched, in place like the reference
    case = load_case('gc_pixel_fs3_aug')
    for output in ('numpy', 'device'):
        sampler = device_sampler(case['fields'], case['cfg'], 'gc', output=output)
        batch = sampler.sample(16, evaluation=True)
        before = to_host(batch)
        np.random.seed(5)
        crop = np.random.randint(0, 7, (16, 2))
        np.random.seed(5)
        sampler.augment(batch, ['observations', 'value_goals', 'actions'])
        after = to_host(batch)
        for key in ('observations', 'value_goals'):
            assert np.array_equal(after[key], shifted_edge_crop(before[key], crop, 3)), (output, key)
        assert np.array_equal(after['actions'], before['actions']) and np.array_equal(after['next_observations'], before['next_observations'])


def test_atc_augment_method():
    """ATCDataset.augment (datasets.py:438-448): padding from config['augment_padding'] (4 by default)."""
    from oracle.replay_oracle import shifted_edge_crop

    case = load_case('atc_pixel_fs3_aug')
    sampler = device_sampler(case['fields'], case['cfg'], 'atc', output='numpy')
    pad = int(case['cfg'].get('augment_padding', 4))
    batch = sampler.sample(12, case['k'], evaluation=True)
    before = {k: v.copy() for k, v in batch.items()}
    np.random.seed(9)
    crop = np.random.randint(0, 2 * pad + 1, (12, 2))
    np.random.seed(9)
    sampler.augment(batch, ['observations', 'positive_observations'])
    for key in ('observations', 'positive_observations'):
        assert np.array_equal(batch[key], shifted_edge_crop(before[key], crop, pad)), key
    idxs = np.array([0, 3, 5])
    assert np.array_equal(np.asarray(sampler.get_stacked_observations(idxs)), np.asarray(sampler.get_observations(idxs)))


def test_atc_anchor_sets_match_oracle():
    from oracle.replay_oracle import OracleATCSampler

    case = load_case('atc_state_noaug')
    sampler = device_sampler(case['fields'], case['cfg'], 'atc')
    oracle = OracleATCSampler(case['fields'], case['cfg'])
    for k in (0, 1, 7, 30):
        assert np.array_equal(sampler.get_valid_atc_idxs(k), oracle.valid_anchors(k)), k
    with pytest.raises(ValueError):
        sampler.get_valid_atc_idxs(10_000)


def test_trl_philox_mode_properties():
    """TRL in the on-device RNG mode: midpoints lie in [idx, goal), offsets are consistent, rows are never terminal."""
    case = load_case('trl_state')
    fields = {k: v.copy() for k, v in case['fields'].items()}
    fields['observations'][:, 0] = np.arange(len(fields['terminals']))
    sampler = device_sampler(fields, case['cfg'], 'gc', seed=4)
    out = to_host(sampler.sample(4096))
    i = out['observations'][:, 0].astype(np.int64)
    g = out['value_goal_observations'][:, 0].astype(np.int64)
    m = out['value_midpoint_observations'][:, 0].astype(np.int64)
    assert (fields['terminals'][i] == 0).all() and (g > i).all() and (m >= i).all() and (m < g).all()
    assert np.array_equal(out['value_offsets'], g - i) and np.array_equal(out['value_midpoint_offsets'], m - i)
    assert np.array_equal(out['next_actions'], fields['actions'][i + 1])
    assert np.array_equal(out['value_midpoint_actions'], fields['actions'][m])
    assert np.array_equal(out['value_next_goals'][:, 0].astype(np.int64), i + 1)

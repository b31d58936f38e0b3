"""Image gathers (frame stacking + edge-padded crop) against a plain numpy reference, at every crop shift, on both frame
kernels: `gather_frames_tma_kernel<FS>` (uint8, C = 3, W a multiple of 16, band heights 7..32, 1..4 frames) and
`gather_frames_generic_kernel` (other dtypes, channel counts, widths, deeper stacks, image heights without a band
size, paddings above 4 and up to 127).

Each case asserts which kernel ran (`ogb_batch_dominant_kernel` of the native batch), so a shape cannot quietly move to
the other path.  The reference below is datasets.py:17-33 and :359-366 as the reference writes them (np.pad, slice,
concatenate); `test_reference_matches_oracle` checks it against the oracle's closed forms without a GPU.
"""

import ctypes as C

import numpy as np
import pytest

from oracle import philox_np
from oracle.replay_oracle import DrawsSource, OracleATCSampler, OracleSampler, shifted_edge_crop, stacked_frames
from tests.golden.make_golden import cfg, ragged, toy_fields
from tests.gpu_util import device_sampler, to_host

TMA = 'gather_frames_tma_kernel'
GENERIC = 'gather_frames_generic_kernel'
ATC_K = 1

# (H, W, frame stack), uint8, C = 3.  Band heights (padding 3 / 4): 8, 9, 30, 17, 7, 20, 24, 32, 32 x 3.  H = 8 / 9 at
# W = 64 and W = 16 below H = 43 are at most 2 KB a row and live in the packed record table when the dataset has other
# fields, which only the generic kernel reads; 68 x 16 (band 17) keeps W = 16 with 1..4 frames on the TMA kernel there.
TMA_CASES = ([(h, 64, 3) for h in (8, 9, 30, 34, 35, 40, 48, 64, 96)] + [(40, w, 3) for w in (16, 32, 48, 80)]
             + [(34, 16, fs) for fs in (1, 2, 3, 4)] + [(68, 16, fs) for fs in (1, 2, 3, 4)])
# (shape, dtype, frame stack)
GENERIC_CASES = [
    ((37, 64, 3), np.uint8, 3), ((74, 64, 3), np.uint8, 3),           # no band height in (padding, 32] divides H
    ((16, 16, 1), np.uint8, 2), ((24, 24, 4), np.uint8, 3), ((10, 12, 6), np.uint8, 2),
    ((20, 24, 3), np.uint8, 3), ((48, 24, 3), np.uint8, 2),           # W = 24: not a multiple of 16
    ((16, 20, 3), np.float16, 2), ((32, 20, 3), np.float16, 3),       # 6-byte pixels
    ((12, 10, 1), np.float32, 3), ((20, 18, 3), np.float32, 2),
    ((20, 18, 2), np.float64, 2), ((8, 8, 3), np.int32, 3),
    ((64, 64, 3), np.uint8, 5), ((64, 64, 3), np.uint8, 6),           # deeper than the TMA templates
]
PADS = (0, 3, 4)


# ------------------------------------------------ plain reference ------------------------------------------------
def ref_crop(imgs, crop, p):
    """batched_random_crop (datasets.py:17-33) as written: edge-pad each image by p, slice the original size at (cy, cx)."""
    h, w = imgs.shape[1:3]
    out = np.empty_like(imgs)
    for b, (cy, cx) in enumerate(crop):
        out[b] = np.pad(imgs[b], ((p, p), (p, p), (0, 0)), mode='edge')[cy:cy + h, cx:cx + w]
    return out


def trajectory_starts(terminals):
    """First row of every row's trajectory: trajectories start at row 0 and after each terminal row (datasets.py:186-187)."""
    first = np.empty(len(terminals), dtype=np.int64)
    start = 0
    for r, t in enumerate(terminals):
        first[r] = start
        if t > 0:
            start = r + 1
    return first


def ref_stack(obs, first, rows, fs):
    """get_stacked_observations (datasets.py:359-366): frames i-fs+1 .. i, none before the trajectory's first row."""
    return np.stack([np.concatenate([obs[max(i - k, first[i])] for k in range(fs - 1, -1, -1)], axis=-1) for i in rows])


def enumerated_shifts(p, min_rows=32):
    """Every (cy, cx) in [0, 2p]^2, repeated up to at least `min_rows` rows."""
    s = np.arange(2 * p + 1)
    grid = np.stack(np.meshgrid(s, s, indexing='ij'), axis=-1).reshape(-1, 2)
    return np.tile(grid, (-(-min_rows // len(grid)), 1)).astype(np.int64)


def random_images(rng, n, shape, dtype):
    dt = np.dtype(dtype)
    if dt.kind in 'ui':
        info = np.iinfo(dt)
        return rng.integers(info.min, info.max, (n, *shape), dtype=dt, endpoint=True)
    return (rng.standard_normal((n, *shape)) * 100).astype(dt)


def image_fields(seed, shape, dtype, n_traj=10, lo=2, hi=10):
    """Compact dataset (ogbench layout) with ragged trajectories, several shorter than the deepest frame stack."""
    fields = toy_fields(seed, ragged(seed, n_traj, lo, hi), (1,), 2, np.float32)
    fields['observations'] = random_images(np.random.default_rng(seed), len(fields['terminals']), shape, dtype)
    return fields


# ------------------------------------------------ which kernel runs ------------------------------------------------
def band_rows(h, pad):
    return next((rb for rb in range(32, pad, -1) if h % rb == 0), 0)


def expected_kernel(shape, dtype, fs, pad, own_array):
    """The frame kernel the launch code picks: TMA for uint8 HWC with C = 3, W % 16 == 0, W * 3 <= 256, H >= 8, 1..4
    frames, padding <= 4, rows in an array of their own and densely strided (bytes a multiple of 32), and a band height
    in (padding, 32] that divides H; the generic kernel otherwise."""
    h, w, c = shape
    row = h * w * c * np.dtype(dtype).itemsize
    tma = (np.dtype(dtype) == np.uint8 and c == 3 and w % 16 == 0 and w * 3 <= 256 and h >= 8 and 1 <= fs <= 4
           and pad <= 4 and own_array and row % 32 == 0 and band_rows(h, pad) > 0)
    return f'{TMA}<{fs}>' if tma else GENERIC


def sample_own_array(shape, dtype):
    """Rows of at most 2 KB share the packed record table with the dataset's other fields."""
    return int(np.prod(shape)) * np.dtype(dtype).itemsize > 2048


# ------------------------------------------------ device legs ------------------------------------------------
def frame_kernel(handle):
    from ogbench_b200 import _native

    name, ms = C.c_char_p(), C.c_float()
    _native.check(_native.lib().ogb_batch_dominant_kernel(handle.ptr, C.byref(name), C.byref(ms)))
    return name.value.decode()


def crop_native(imgs, crop, padding):
    """datasets._crop_array (ogb_sampler_gather_cropped) keeping the native batch: (cropped array, frame kernel)."""
    from ogbench_b200 import Dataset, _native
    from ogbench_b200.datasets import _Sampler
    from ogbench_b200.device_array import BatchHandle

    sampler = _Sampler(Dataset.create(freeze=False, observations=imgs), None, _native.KIND_PLAIN)
    idxs = np.arange(len(crop), dtype=np.int64)
    crop = np.ascontiguousarray(crop, dtype=np.int64)
    out = C.c_void_p()
    _native.check(_native.lib().ogb_sampler_gather_cropped(sampler.ptr, idxs.ctypes.data_as(C.c_void_p), len(idxs),
                                                           crop.ctypes.data_as(C.c_void_p), int(padding), C.byref(out)))
    handle = BatchHandle(out, sampler.device, None)
    return np.asarray(sampler.wrap(handle)['observations']), frame_kernel(handle)


def atc_native(sampler, batch_size, draws):
    """ATCDataset.sample(batch_size, ATC_K, draws=draws) keeping the native batch: (batch, frame kernel)."""
    from ogbench_b200 import _native
    from ogbench_b200.datasets import _pack_draws
    from ogbench_b200.device_array import BatchHandle

    keep = []
    d = _pack_draws(draws, keep)
    out = C.c_void_p()
    _native.check(_native.lib().ogb_sampler_sample_atc(sampler._sampler.ptr, batch_size, 1, ATC_K, 0, C.byref(d), C.byref(out)))
    handle = BatchHandle(out, sampler._sampler.device, None)
    return to_host(sampler._sampler.wrap(handle)), frame_kernel(handle)


def assert_same(got, want, what):
    assert got.dtype == want.dtype and got.shape == want.shape, (what, got.dtype, want.dtype, got.shape, want.shape)
    if not np.array_equal(got, want):
        bad = np.nonzero((got != want).reshape(len(want), -1).any(axis=1))[0]
        raise AssertionError(f'{what}: {len(bad)} of {len(want)} rows differ, first {bad[:8].tolist()}')


def check_batch(got, want, fields, image_rows, fs, crop, p, what):
    """Every key: image keys against the plain reference on the sampled rows, the rest against the oracle."""
    assert set(got) == set(want), set(got) ^ set(want)
    first = trajectory_starts(fields['terminals'])
    for k in want:
        exp = ref_crop(ref_stack(fields['observations'], first, image_rows[k], fs), crop, p) if k in image_rows else want[k]
        assert_same(got[k], exp, f'{what} {k}')


def gc_rows(oracle, fs):
    iv = oracle.last_index_vectors
    nxt = iv['idxs'] + 1 if fs > 1 else np.minimum(iv['idxs'] + 1, oracle.size - 1)
    return dict(observations=iv['idxs'], next_observations=nxt, value_goals=iv['value_goal'], actor_goals=iv['actor_goal'])


def sample_leg(shape, dtype, fs, p, seed):
    """sample() in validation mode with every shift enumerated: GCDataset for padding 3 (its augment() padding), ATCDataset
    with augment_padding = p otherwise.  Returns the frame kernel that ran."""
    fields = image_fields(seed, shape, dtype)
    crop = enumerated_shifts(p)
    B = len(crop)
    frame_stack = fs if fs > 1 else None
    np.random.seed(seed)
    if p == 3:
        config = cfg(p_aug=1.0, frame_stack=frame_stack)
        oracle = OracleSampler(fields, config, 'gc')
        oracle.sample(B)
        draws = oracle.last_draws
        draws.crop, draws.aug_coin = crop, 0.0
        want = oracle.sample(B, source=DrawsSource(draws))
        rows = gc_rows(oracle, fs)
        sampler = device_sampler(fields, config, 'gc')
        handle = sampler._sampler.sample_native(B, draws=draws)
        got, kernel = to_host(sampler._sampler.wrap(handle)), frame_kernel(handle)
    else:
        config = dict(frame_stack=frame_stack, p_aug=1.0, augment_padding=p)
        oracle = OracleATCSampler(fields, config)
        oracle.sample(B, ATC_K)
        draws = oracle.last_draws
        draws.crop, draws.aug_coin = crop, 0.0
        want = oracle.sample(B, ATC_K, source=DrawsSource(draws))
        anchors = oracle.valid_anchors(ATC_K)[draws.idx_pos]
        rows = dict(observations=anchors, positive_observations=anchors + ATC_K)
        got, kernel = atc_native(device_sampler(fields, config, 'atc'), B, draws)
    check_batch(got, want, fields, rows, fs, crop, p, f'sample {shape} {np.dtype(dtype)} fs={fs} p={p}')
    return kernel


def crop_leg(shape, dtype, p, seed):
    crop = enumerated_shifts(p)
    imgs = random_images(np.random.default_rng(seed), len(crop), shape, dtype)
    got, kernel = crop_native(imgs, crop, p)
    assert_same(got, ref_crop(imgs, crop, p), f'crop {shape} {np.dtype(dtype)} p={p}')
    return kernel


def case_id(shape, dtype, fs):
    return f'{"x".join(map(str, shape))}-{np.dtype(dtype).name}-fs{fs}'


# ------------------------------------------------ tests ------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize('p', PADS)
@pytest.mark.parametrize('h,w,fs', TMA_CASES, ids=[case_id((h, w, 3), np.uint8, fs) for h, w, fs in TMA_CASES])
def test_tma_shapes_every_shift(h, w, fs, p):
    shape = (h, w, 3)
    seed = 1000 * h + 10 * w + fs
    assert crop_leg(shape, np.uint8, p, seed) == f'{TMA}<1>'
    want = expected_kernel(shape, np.uint8, fs, p, sample_own_array(shape, np.uint8))
    assert sample_leg(shape, np.uint8, fs, p, seed) == want


@pytest.mark.gpu
@pytest.mark.parametrize('p', PADS)
@pytest.mark.parametrize('shape,dtype,fs', GENERIC_CASES, ids=[case_id(*c) for c in GENERIC_CASES])
def test_generic_shapes_every_shift(shape, dtype, fs, p):
    seed = int(np.prod(shape)) + 7 * fs + np.dtype(dtype).itemsize
    assert crop_leg(shape, dtype, p, seed) == expected_kernel(shape, dtype, 1, p, True)
    want = expected_kernel(shape, dtype, fs, p, sample_own_array(shape, dtype))
    assert sample_leg(shape, dtype, fs, p, seed) == want
    if p > 0:
        assert want == GENERIC


@pytest.mark.gpu
@pytest.mark.parametrize('p', (5, 6, 7, 8))
def test_atc_augment_padding_above_4(p):
    """ATCDataset with augment_padding 5..8 (rng='numpy'): the reference's own draws, enough rows to draw every shift."""
    shape, fs = (12, 10, 3), 2
    fields = image_fields(p, shape, np.uint8)
    config = dict(frame_stack=fs, p_aug=1.0, augment_padding=p)
    sampler = device_sampler(fields, config, 'atc', rng='numpy')
    oracle = OracleATCSampler(fields, config)
    B = 16 * (2 * p + 1) ** 2
    np.random.seed(p)
    draws = sampler._host_draws(B, ATC_K, False)
    np.random.seed(p)
    want = oracle.sample(B, ATC_K)
    assert np.array_equal(draws.idx_pos, oracle.last_draws.idx_pos) and np.array_equal(draws.crop, oracle.last_draws.crop)
    assert len(np.unique(draws.crop, axis=0)) == (2 * p + 1) ** 2
    got, kernel = atc_native(sampler, B, draws)
    assert kernel == GENERIC
    anchors = oracle.valid_anchors(ATC_K)[draws.idx_pos]
    check_batch(got, want, fields, dict(observations=anchors, positive_observations=anchors + ATC_K), fs, draws.crop, p,
                f'atc p={p}')


@pytest.mark.gpu
@pytest.mark.parametrize('p', (6, 9))
def test_padding_larger_than_the_image(p):
    assert crop_leg((6, 5, 1), np.uint8, p, p) == GENERIC


PHILOX_CASES = [((40, 80, 3), np.uint8, 3), ((68, 16, 3), np.uint8, 2), ((35, 64, 3), np.uint8, 4),
                ((37, 64, 3), np.uint8, 3), ((12, 10, 3), np.float32, 2)]


@pytest.mark.gpu
@pytest.mark.parametrize('shape,dtype,fs', PHILOX_CASES, ids=[case_id(*c) for c in PHILOX_CASES])
def test_philox_mode_images(shape, dtype, fs):
    """On-device draws: the batch equals the reference fed the numpy restatement of the Philox draws."""
    from tests.test_gpu_philox import goal_sets_for

    fields = image_fields(fs, shape, dtype, n_traj=14)
    config = cfg(p_aug=1.0, frame_stack=fs)
    seed, stream_id, B = 0x5EED0F, 3, 64
    sampler = device_sampler(fields, config, 'gc', seed=seed, stream_id=stream_id)
    oracle = OracleSampler(fields, config, 'gc')
    handle = sampler._sampler.sample_native(B)
    got, kernel = to_host(sampler._sampler.wrap(handle)), frame_kernel(handle)
    assert kernel == expected_kernel(shape, dtype, fs, 3, sample_own_array(shape, dtype))
    draws, knife = philox_np.philox_draws(seed, stream_id, 0, B, len(oracle.valid_table), goal_sets_for(config, 'gc'), True, 1.0)
    src = DrawsSource(draws)
    want = oracle.sample(B, source=src)
    assert src.exhausted() and draws.crop is not None
    ok = ~knife
    assert ok.mean() > 0.9
    rows = {k: v[ok] for k, v in gc_rows(oracle, fs).items()}
    check_batch({k: v[ok] for k, v in got.items()}, {k: v[ok] for k, v in want.items()}, fields, rows, fs, draws.crop[ok], 3,
                f'philox {shape}')


@pytest.mark.gpu
def test_padding_127_is_exact():
    """The widest padding the int8 shift record holds: shifts of -127, 0 and +127 (and their neighbours) crop exactly."""
    ends = np.array([0, 1, 126, 127, 128, 253, 254])
    crop = np.stack(np.meshgrid(ends, ends, indexing='ij'), axis=-1).reshape(-1, 2)
    imgs = random_images(np.random.default_rng(127), len(crop), (6, 5, 2), np.uint8)
    got, kernel = crop_native(imgs, crop, 127)
    assert kernel == GENERIC
    assert_same(got, ref_crop(imgs, crop, 127), 'crop p=127')
    # ATCDataset with augment_padding = 127 and the reference's own draws
    fields = image_fields(5, (6, 5, 2), np.uint8)
    config = dict(frame_stack=2, p_aug=1.0, augment_padding=127)
    sampler = device_sampler(fields, config, 'atc', rng='numpy')
    oracle = OracleATCSampler(fields, config)
    np.random.seed(127)
    draws = sampler._host_draws(256, ATC_K, False)
    np.random.seed(127)
    want = oracle.sample(256, ATC_K)
    got, kernel = atc_native(sampler, 256, draws)
    anchors = oracle.valid_anchors(ATC_K)[draws.idx_pos]
    check_batch(got, want, fields, dict(observations=anchors, positive_observations=anchors + ATC_K), 2, draws.crop, 127,
                'atc p=127')


@pytest.mark.gpu
def test_padding_128_is_refused():
    """Shifts are stored as int8 with -128 meaning "not augmented": a padding of 128 or more cannot be represented."""
    from ogbench_b200 import datasets

    imgs = random_images(np.random.default_rng(0), 4, (6, 5, 1), np.uint8)
    with pytest.raises(ValueError, match='padding'):
        datasets._crop_array(imgs, np.zeros((4, 2), dtype=np.int64), 128, 0, 'numpy')
    with pytest.raises(ValueError, match='padding'):
        device_sampler(image_fields(0, (6, 5, 1), np.uint8), dict(frame_stack=None, p_aug=1.0, augment_padding=128), 'atc')


def test_reference_matches_oracle():
    """The plain reference above against the oracle's closed forms (oracle/replay_oracle.py), over the shapes, dtypes,
    frame stacks and paddings the device tests use."""
    shapes = [((h, w, 3), np.uint8, fs) for h, w, fs in TMA_CASES] + GENERIC_CASES + [((6, 5, 1), np.uint8, 1)]
    for i, (shape, dtype, fs) in enumerate(shapes):
        fields = image_fields(i, shape, dtype)
        obs, terminals = fields['observations'], fields['terminals']
        rows = np.arange(len(obs))
        initial_locs = np.concatenate([[0], np.nonzero(terminals > 0)[0][:-1] + 1])
        for depth in sorted({1, fs}):
            assert_same(ref_stack(obs, trajectory_starts(terminals), rows, depth),
                        stacked_frames(obs, initial_locs, rows, depth), f'stack {shape} fs={depth}')
        for p in PADS + ((5, 8, 9) if shape[0] < 16 else ()):
            crop = enumerated_shifts(p)
            imgs = obs[np.arange(len(crop)) % len(obs)]
            assert_same(ref_crop(imgs, crop, p), shifted_edge_crop(imgs, crop, p), f'crop {shape} p={p}')
    crop = np.array([[0, 254], [254, 0], [127, 127], [1, 253]])
    imgs = random_images(np.random.default_rng(1), 4, (6, 5, 2), np.uint8)
    assert_same(ref_crop(imgs, crop, 127), shifted_edge_crop(imgs, crop, 127), 'crop p=127')


def test_case_plan_reaches_both_kernels():
    """The device cases above cover what they are meant to: the TMA kernel at band heights other than 32, at W = 16
    and 80 and with 1..4 frames through sample(); the generic kernel for every generic case with a non-zero padding."""
    crop_bands = {band_rows(h, p) for h, w, fs in TMA_CASES for p in PADS}
    assert {7, 8, 9, 17, 20, 24, 30, 32} <= crop_bands
    assert all(expected_kernel((h, w, 3), np.uint8, 1, p, True).startswith(TMA) for h, w, fs in TMA_CASES for p in PADS)
    sample_tma = {(w, fs) for h, w, fs in TMA_CASES for p in PADS
                  if expected_kernel((h, w, 3), np.uint8, fs, p, sample_own_array((h, w, 3), np.uint8)).startswith(TMA)}
    assert {(16, fs) for fs in (1, 2, 3, 4)} <= sample_tma and (80, 3) in sample_tma
    for shape, dtype, fs in GENERIC_CASES:
        for p in (3, 4):
            assert expected_kernel(shape, dtype, fs, p, sample_own_array(shape, dtype)) == GENERIC, (shape, fs, p)
    # image heights without a band size at padding 3 / 4, which used to be refused instead of served by the generic kernel
    assert band_rows(37, 3) == band_rows(74, 4) == 0
